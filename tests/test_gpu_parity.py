"""GPU: the engine behind the reference's call surface (MDM.forward, ClassifierFreeSampleModel.forward,
p_sample_loop / ddim_sample_loop) against
  (1) tests/golden/sampler.npz -- outputs of the UNMODIFIED reference on the same seeded inputs, and
  (2) the CPU oracle (oracle/condmdi_oracle.py) run here on the same inputs,
at the reference's parity gate rtol 1e-3 / atol 1e-4 (fp32), plus size-independent properties at B=64.
Everything goes through the public API, i.e. through the C ABI of libcondmdi_b200.so.
"""
import os

import numpy as np
import pytest
import torch

import condmdi_b200 as C
from oracle import condmdi_oracle as O

pytestmark = pytest.mark.gpu
GATE = dict(rtol=1e-3, atol=1e-4)
B, D, L = 2, 263, 196
DEV = "cuda:0"


@pytest.fixture(scope="module")
def gold(golden_dir):
    return np.load(os.path.join(golden_dir, "sampler.npz"))


@pytest.fixture(scope="module")
def gi():
    return O.golden_inputs()


def _model(text):
    sd = O.random_state_dict(seed=7, text=text)
    m = C.MDM(cond_mode="text" if text else "no_cond", cond_mask_prob=0.1)
    missing, unexpected = m.load_state_dict(sd, strict=False)
    assert not missing and not unexpected
    return m.cuda(), sd


@pytest.fixture(scope="module")
def plain():
    return _model(False)


@pytest.fixture(scope="module")
def texty(gi):
    m, sd = _model(True)
    m.encode_text = lambda texts: gi["cond"].to(DEV)
    return m, sd


def close(a, b, **tol):
    a, b = torch.as_tensor(a).cpu().float(), torch.as_tensor(b).cpu().float()
    ok = torch.allclose(a, b, **tol)
    if not ok:
        err = (a - b).abs()
        print(f"max_abs={err.max():.3e} mean_abs={err.mean():.3e} viol={(err > tol['atol'] + tol['rtol'] * b.abs()).float().mean():.5f}")
    return ok


# ------------------------------------------------------------------------------------------------
# one denoiser evaluation
# ------------------------------------------------------------------------------------------------
def test_forward_no_cond_vs_reference_golden(plain, gi, gold):
    m, sd = plain
    t = torch.tensor(gold["fwd_nocond.t"])
    got = m(gi["x"].to(DEV), t.to(DEV), y={})          # per-sample timesteps [999, 37]
    assert got.shape == (B, D, 1, L) and got.dtype == torch.float32 and got.is_cuda
    assert close(got, gold["fwd_nocond.out"], **GATE)
    assert close(got, O.mdm_forward(sd, gi["x"], t), **GATE)


def test_forward_text_uncond_cfg_vs_reference_golden(texty, gi, gold):
    m, sd = texty
    t = torch.tensor([500, 500])
    x = gi["x"].to(DEV)
    assert close(m(x, t.to(DEV), y={"text": ["a", "b"]}), gold["fwd_text.out"], **GATE)
    assert close(m(x, t.to(DEV), y={"text": ["a", "b"], "uncond": True}), O.mdm_forward(sd, gi["x"], t, gi["cond"], uncond=True), **GATE)
    w = C.ClassifierFreeSampleModel(m)
    y = {"text": ["a", "b"], "text_scale": gi["text_scale"].to(DEV)}
    got = w(x, t.to(DEV), y=y, obs_x0=x, obs_mask=None)   # obs_* are accepted and ignored, like the reference's MDM
    assert "uncond" not in y                              # the caller's y is not mutated (cfg_sampler.py:28)
    assert close(got, gold["fwd_cfg.out"], **GATE)


def test_forward_from_host_tensors_raises(plain, gi):
    m, _ = plain
    with pytest.raises(RuntimeError):
        m(gi["x"], torch.tensor([1, 1]), y={})


# ------------------------------------------------------------------------------------------------
# sampling loops with the shared noise tape
# ------------------------------------------------------------------------------------------------
def test_p_sample_loop_three_steps_vs_reference_golden(plain, gi, gold):
    m, sd = plain
    eng = m.engine_for(torch.device(DEV), max_batch=B)
    diff = C.create_gaussian_diffusion()
    eng.set_schedule(diff.betas, diff.timestep_map)
    tape = gi["tape"].to(DEV)
    res = {}
    for use_graph in (True, False):
        res[use_graph] = eng.sample(B, x_T=tape[0], noise_tape=tape[1:], num_steps=3, want_pred_xstart=True, use_graph=use_graph)
    assert close(res[True]["sample"], gold["ddpm_uncond.sample"], **GATE)
    assert close(res[True]["pred_xstart"], gold["ddpm_uncond.pred_xstart"], **GATE)
    assert torch.equal(res[True]["sample"], res[False]["sample"])  # graph replay == plain launches, bit for bit


def test_full_1000_step_ddpm_loop_vs_reference_golden(plain, golden_dir):
    """configs[1] at B=2, the whole chain: 1000 engine steps against the reference's own CPU run of the same loop on the
    same noise (tests/golden/long_loop.npz) -- error growth over the full length, through the public API and the graph."""
    g = np.load(os.path.join(golden_dir, "long_loop.npz"))
    m, _ = plain
    diff = C.create_gaussian_diffusion()
    diff.noise_tape = O.long_loop_tape().to(DEV)
    out = diff.p_sample_loop(m, (B, D, 1, L), clip_denoised=False, model_kwargs={"y": {}})
    assert close(out, g["sample"], **GATE)


def test_ddim50_full_loop_vs_reference_golden(plain, gi, gold):
    m, sd = plain
    d50 = C.create_gaussian_diffusion(timestep_respacing="ddim50")
    assert d50.num_timesteps == 50
    d50.noise_tape = gi["tape"][torch.arange(51) % 8].to(DEV)
    got = d50.ddim_sample_loop(m, (B, D, 1, L), model_kwargs={"y": {}}, clip_denoised=False, progress=True)
    assert got.shape == (B, D, 1, L) and got.is_cuda
    assert close(got, gold["ddim50.sample"], **GATE)


def test_cfg_imputation_loop_vs_reference_golden(texty, gi, gold):
    m, sd = texty
    w = C.ClassifierFreeSampleModel(m)
    diff = C.create_gaussian_diffusion()
    diff.noise_tape = gi["tape"].to(DEV)
    x_obs, kf = gi["x_obs"].to(DEV), gi["kf_mask"].to(DEV)
    ykw = {"text": ["a", "b"], "text_scale": gi["text_scale"].to(DEV), "mask": gi["y_mask"].to(DEV), "lengths": gi["lengths"],
           "imputate": 1, "stop_imputation_at": 1, "replacement_distribution": "conditional", "inpainted_motion": x_obs,
           "inpainting_mask": kf, "tokens": None, "log_name": "x"}  # unknown keys are tolerated
    got = diff.p_sample_loop(w, (B, D, 1, L), model_kwargs={"y": ykw, "obs_x0": x_obs, "obs_mask": kf}, skip_timesteps=996,
                             init_image=x_obs, clip_denoised=False)
    assert close(got, gold["cfg_impute.sample"], **GATE)
    # generator form: step k=2 is t=1 (>= stop_imputation_at): observed entries are EXACTLY the observations
    outs = list(diff.p_sample_loop_progressive(w, (B, D, 1, L), model_kwargs={"y": ykw}, skip_timesteps=996, init_image=x_obs))
    assert len(outs) == 4
    M = (gi["kf_mask"] * gi["y_mask"].float()).bool()
    assert torch.equal(outs[2]["pred_xstart"].cpu()[M], gi["x_obs"][M])
    assert close(outs[2]["pred_xstart"], gold["cfg_impute.pred_xstart_t1"], **GATE)
    assert not torch.equal(outs[3]["pred_xstart"].cpu()[M], gi["x_obs"][M])  # t=0 < stop_imputation_at: left free
    assert close(outs[3]["sample"], got, rtol=0, atol=0)                      # chunked loop == fused loop, bit for bit
    # dump_steps returns pred_xstart at the requested iterations (gaussian_diffusion.py:1208-1213)
    dump = diff.p_sample_loop(w, (B, D, 1, L), model_kwargs={"y": ykw}, skip_timesteps=996, init_image=x_obs, dump_steps=[0, 2])
    assert len(dump) == 2 and torch.equal(dump[1], outs[2]["pred_xstart"]) and torch.equal(dump[0], outs[0]["pred_xstart"])


def test_reconstruction_guidance_vs_reference_golden(texty, gi, gold):
    """config 4 of BASELINE.json: CFG + imputation + reconstruction guidance (weight 20), first 2 steps (t = 999, 998)"""
    m, sd = texty
    w = C.ClassifierFreeSampleModel(m)
    diff = C.create_gaussian_diffusion()
    diff.noise_tape = gi["tape"].to(DEV)
    x_obs, kf = gi["x_obs"].to(DEV), gi["kf_mask"].to(DEV)
    ykw = {"text": ["a", "b"], "text_scale": gi["text_scale"].to(DEV), "mask": gi["y_mask"].to(DEV), "lengths": gi["lengths"],
           "imputate": 1, "stop_imputation_at": 1, "replacement_distribution": "conditional", "inpainted_motion": x_obs,
           "inpainting_mask": kf, "reconstruction_guidance": True, "reconstruction_weight": 20.0, "gradient_schedule": None,
           "diffusion_steps": 1000, "stop_recguidance_at": 0}
    outs = []
    for k, o in enumerate(diff.p_sample_loop_progressive(w, (B, D, 1, L), model_kwargs={"y": ykw})):
        outs.append(o)
        if k == 1:
            break
    assert close(outs[1]["sample"], gold["recon.sample"], **GATE)
    assert close(outs[1]["pred_xstart"], gold["recon.pred_xstart"], **GATE)
    # and against the oracle's autograd implementation, one more step further
    c = O.Conditioning(cond_emb=gi["cond"], cfg=True, text_scale=gi["text_scale"], y_mask=gi["y_mask"], imputate=True,
                       stop_imputation_at=1, inpainted_motion=gi["x_obs"], inpainting_mask=gi["kf_mask"],
                       reconstruction_guidance=True, reconstruction_weight=20.0)
    ref = O.sample_loop(sd, O.make_tables(""), (B, D, 1, L), c, gi["tape"], "ddpm", max_steps=2, return_all=True)
    assert close(outs[1]["sample"], ref[-1]["sample"], **GATE)


def test_reconstruction_guidance_without_imputation_and_stop_step(texty, gi):
    """guidance only (no imputation), no CFG wrapper, exponential schedule, stop_recguidance_at inside the run"""
    m, sd = texty
    diff = C.create_gaussian_diffusion()
    diff.noise_tape = gi["tape"].to(DEV)
    x_obs, kf = gi["x_obs"].to(DEV), gi["kf_mask"].to(DEV)
    ykw = {"text": ["a", "b"], "mask": gi["y_mask"].to(DEV), "inpainted_motion": x_obs, "inpainting_mask": kf,
           "reconstruction_guidance": True, "reconstruction_weight": 5.0, "gradient_schedule": "exponential",
           "diffusion_steps": 1000, "stop_recguidance_at": 2}
    got = diff.p_sample_loop(m, (B, D, 1, L), model_kwargs={"y": ykw}, skip_timesteps=996, init_image=x_obs)  # t = 3, 2, 1, 0
    c = O.Conditioning(cond_emb=gi["cond"], y_mask=gi["y_mask"], inpainted_motion=gi["x_obs"], inpainting_mask=gi["kf_mask"],
                       reconstruction_guidance=True, reconstruction_weight=5.0, gradient_schedule="exponential",
                       stop_recguidance_at=2)
    ref = O.sample_loop(sd, O.make_tables(""), (B, D, 1, L), c, gi["tape"], "ddpm", skip_timesteps=996, init_image=gi["x_obs"])
    assert close(got, ref, **GATE)


def test_marginal_replacement_is_plain_sampling(texty, gi):
    """gaussian_diffusion.py:437-439: the 'marginal' branch only calls the model."""
    m, sd = texty
    diff = C.create_gaussian_diffusion()
    diff.noise_tape = gi["tape"].to(DEV)
    y0 = {"text": ["a", "b"]}
    y1 = dict(y0, imputate=1, stop_imputation_at=0, replacement_distribution="marginal", inpainted_motion=gi["x_obs"].to(DEV),
              inpainting_mask=gi["kf_mask"].to(DEV), mask=gi["y_mask"].to(DEV))
    a = diff.p_sample_loop(m, (B, D, 1, L), model_kwargs={"y": y0}, skip_timesteps=997)
    b = diff.p_sample_loop(m, (B, D, 1, L), model_kwargs={"y": y1}, skip_timesteps=997)
    assert torch.equal(a, b)


def test_host_buffer_path_equals_device_path(plain, gi):
    m, sd = plain
    eng = m.engine_for(torch.device(DEV), max_batch=B)
    diff = C.create_gaussian_diffusion(timestep_respacing="ddim50")
    eng.set_schedule(diff.betas, diff.timestep_map)
    xT = gi["tape"][0]
    a = eng.sample(B, sampler=C.capi.SAMPLER_DDIM, x_T=xT.to(DEV), seed=11, skip_timesteps=45, want_pred_xstart=True)
    b = eng.sample(B, sampler=C.capi.SAMPLER_DDIM, x_T=xT.pin_memory(), seed=11, skip_timesteps=45, want_pred_xstart=True,
                   host_buffers=True)
    assert not b["sample"].is_cuda
    assert torch.equal(a["sample"].cpu(), b["sample"]) and torch.equal(a["pred_xstart"].cpu(), b["pred_xstart"])


def test_engine_noise_is_seeded_and_shard_independent(plain):
    m, sd = plain
    eng = m.engine_for(torch.device(DEV), max_batch=4)
    diff = C.create_gaussian_diffusion()
    eng.set_schedule(diff.betas, diff.timestep_map)
    full = eng.sample(4, seed=5, num_steps=3)["sample"].clone()
    again = eng.sample(4, seed=5, num_steps=3)["sample"].clone()
    other = eng.sample(4, seed=6, num_steps=3)["sample"].clone()
    lo = eng.sample(2, seed=5, num_steps=3, sample_offset=0)["sample"].clone()
    hi = eng.sample(2, seed=5, num_steps=3, sample_offset=2)["sample"].clone()
    assert torch.equal(full, again) and not torch.equal(full, other)
    assert torch.equal(full[:2], lo) and torch.equal(full[2:], hi)   # rank r of a sharded run reproduces rows [r*B/G, ...)
    assert torch.isfinite(full).all()


def test_torch_seed_reproducibility_through_public_api(plain):
    m, _ = plain
    diff = C.create_gaussian_diffusion(timestep_respacing="ddim50")
    outs = []
    for _ in range(2):
        torch.manual_seed(10)
        outs.append(diff.ddim_sample_loop(m, (B, D, 1, L), model_kwargs={"y": {}}, skip_timesteps=46))
    assert torch.equal(outs[0], outs[1])


@pytest.mark.parametrize("sampler", ["p_sample_loop", "ddim_sample_loop"])
def test_torch_stream_mode_draws_what_the_reference_loop_would(plain, sampler):
    """rng='torch' (the default): after torch.manual_seed(s) the loop consumes exactly the noise the reference's loop
    would draw on this GPU -- randn(*shape) then one randn_like per step (gaussian_diffusion.py:1248, :696, :1407) --
    and leaves torch's generator where the reference would leave it."""
    from condmdi_b200.diffusion import _cuda_rng_state
    m, _ = plain
    shape, skip = (B, D, 1, L), 44
    diff = C.create_gaussian_diffusion(timestep_respacing="ddim50")
    assert diff.rng == "torch"
    n_steps = diff.num_timesteps - skip
    torch.manual_seed(31)
    tape = torch.stack([torch.randn(*shape, device=DEV)] + [torch.randn(*shape, device=DEV) for _ in range(n_steps)])
    state_after = _cuda_rng_state(torch.device(DEV))
    diff.noise_tape = tape
    want = getattr(diff, sampler)(m, shape, model_kwargs={"y": {}}, skip_timesteps=skip)
    diff.noise_tape = None
    torch.manual_seed(31)
    got = getattr(diff, sampler)(m, shape, model_kwargs={"y": {}}, skip_timesteps=skip)
    assert torch.equal(got, want)
    assert _cuda_rng_state(torch.device(DEV)) == state_after
    # the generator form consumes the same stream one step at a time
    torch.manual_seed(31)
    last = None
    for last in getattr(diff, sampler + "_progressive")(m, shape, model_kwargs={"y": {}}, skip_timesteps=skip):
        pass
    assert torch.equal(last["sample"], want)
    # and the engine generator is still selectable
    diff.rng = "engine"
    torch.manual_seed(31)
    other = getattr(diff, sampler)(m, shape, model_kwargs={"y": {}}, skip_timesteps=skip)
    assert torch.isfinite(other).all()
    if sampler == "p_sample_loop":  # DDIM with eta = 0 multiplies the per-step noise by sigma = 0
        assert not torch.equal(other, want)


# ------------------------------------------------------------------------------------------------
# full benchmark size: properties that need no CPU-sized reference
# ------------------------------------------------------------------------------------------------
def test_full_size_batch_independence_and_finiteness(plain, gi):
    """B=64 (the BASELINE shape): rows do not interact, so the first rows of a big batch equal a small batch."""
    m, sd = plain
    g = torch.Generator().manual_seed(3)
    x = torch.randn(64, D, 1, L, generator=g).to(DEV)
    t = torch.full((64,), 123, device=DEV)
    big = m(x, t, y={})
    small = m(x[:3].contiguous(), t[:3], y={})
    assert torch.isfinite(big).all()
    assert close(big[:3], small, rtol=1e-6, atol=1e-6)
    # and the small batch is itself pinned to the oracle
    assert close(small, O.mdm_forward(sd, x[:3].cpu(), t[:3].cpu()), **GATE)


def test_full_size_loop_runs_and_imputes_exactly(texty):
    m, sd = texty
    Bf = 64
    g = torch.Generator().manual_seed(4)
    cond = torch.randn(Bf, 512, generator=g).to(DEV)
    m_enc = m.encode_text
    m.encode_text = lambda texts: cond
    try:
        w = C.ClassifierFreeSampleModel(m)
        x_obs = torch.randn(Bf, D, 1, L, generator=g).to(DEV)
        lengths = torch.randint(20, 197, (Bf,), generator=g)
        kf = C.get_keyframes_mask(x_obs, lengths, "benchmark_sparse", trans_length=5)
        y_mask = (torch.arange(L)[None] < lengths[:, None]).view(Bf, 1, 1, L).to(DEV)
        diff = C.create_gaussian_diffusion()
        y = {"text": [""] * Bf, "text_scale": torch.full((Bf,), 2.5, device=DEV), "mask": y_mask, "imputate": 1,
             "stop_imputation_at": 0, "replacement_distribution": "conditional", "inpainted_motion": x_obs, "inpainting_mask": kf}
        outs = list(diff.p_sample_loop_progressive(w, (Bf, D, 1, L), model_kwargs={"y": y}, skip_timesteps=998))
        M = (kf & y_mask)
        assert torch.equal(outs[-1]["pred_xstart"][M], x_obs[M])  # stop_imputation_at=0: imputed at every step incl. t=0
        # at t=0 the posterior mean coefficient on x_t is 0 and no noise is added: the sample IS pred_xstart there
        assert torch.equal(outs[-1]["sample"][M], x_obs[M])
        assert torch.isfinite(outs[-1]["sample"]).all()
    finally:
        m.encode_text = m_enc


# ------------------------------------------------------------------------------------------------
# objects with the reference's surface: its MDM module tree and the attributes of its SpacedDiffusion
# ------------------------------------------------------------------------------------------------
def test_drop_in_under_reference_objects(gi, gold, golden_dir):
    from standin import StockDiffusion, StockMDM

    ref_model = StockMDM()
    missing, unexpected = ref_model.load_state_dict(O.random_state_dict(seed=7), strict=False)
    assert not missing and not unexpected
    ref_model = ref_model.to(DEV).eval()
    sched = np.load(os.path.join(golden_dir, "schedules.npz"))   # the reference's own respaced ddim50 schedule
    fast = C.accelerate(StockDiffusion(sched["ddim50.betas"], sched["ddim50.timestep_map"]))
    fast.noise_tape = gi["tape"][torch.arange(51) % 8].to(DEV)
    got = fast.ddim_sample_loop(ref_model, (B, D, 1, L), model_kwargs={"y": {}})
    # the reference's ddim_sample_loop on the same weights and noise; its default clip_denoised=True leaves a
    # START_X model's prediction unclipped, so that run is the stored ddim50 fixture
    assert close(got, gold["ddim50.sample"], **GATE)


# ------------------------------------------------------------------------------------------------
# post-processing: sampler output -> joint positions on the GPU (SURVEY 8f-2)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag,abs_3d", [("rel", False), ("abs", True)])
def test_sample_to_joints_vs_reference_golden(golden_dir, tag, abs_3d):
    g = np.load(os.path.join(golden_dir, "postprocess.npz"))
    inp = O.postprocess_inputs()
    got = C.sample_to_joints(inp["sample"].to(DEV), g[f"{tag}.mean"], g[f"{tag}.std"], 22, abs_3d)
    assert got.is_cuda and got.shape == (3, 22, 3, 196)
    assert close(got, g[f"{tag}.joints"], rtol=1e-4, atol=1e-4)
    rag = C.recover_from_ric(inp["ragged"].to(DEV), 22, abs_3d)   # the reference function's own signature, 57 frames
    assert rag.shape == (2, 1, 57, 22, 3)
    assert close(rag, g[f"{tag}.ragged"], rtol=1e-4, atol=1e-4)


def test_sample_to_joints_full_batch_vs_oracle_and_cpu_tensor_raises():
    gen = torch.Generator().manual_seed(9)
    sample = torch.randn(64, D, 1, L, generator=gen)
    mean, std = torch.randn(D, generator=gen) * 0.3, torch.rand(D, generator=gen) * 0.2 + 0.01
    want = O.sample_to_joints(sample, mean, std, 22, False)
    got = C.sample_to_joints(sample.to(DEV), mean, std, 22, False).cpu()
    # prefix sums over 196 frames of O(1) steps: compare against the trajectory's scale (ulp-level sin/cos differences
    # between the CPU and GPU math libraries are integrated along the path)
    assert (got - want).abs().max() <= 2e-5 * want.abs().max() + 1e-5, (got - want).abs().max()
    kit = torch.randn(5, 40, 251, generator=gen)                  # KIT layout: 21 joints, 251 features
    assert close(C.recover_from_ric(kit.to(DEV), 21), O.recover_from_ric(kit, 21), rtol=1e-4, atol=1e-4)
    with pytest.raises(RuntimeError):
        C.recover_from_ric(kit, 21)                                # no CPU fallback
