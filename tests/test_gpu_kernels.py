"""GPU: each production kernel, called through the C ABI, against an fp64 / oracle reference.

Tolerances are written next to each assertion.  The bf16x3 (hi/lo split) mode is the one that must meet the
reference's fp32 parity gate rtol 1e-3 / atol 1e-4; plain bf16 is checked against a bf16-sized bound.
"""
import ctypes

import numpy as np
import pytest
import torch

import condmdi_b200 as C
from oracle import condmdi_oracle as O

pytestmark = pytest.mark.gpu
GATE = dict(rtol=1e-3, atol=1e-4)


def _lib():
    return C.capi.load()


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def run_linear(M, N, K, prec, bn, act=0, bias=True, res=False, seed=0, scale=1.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    A = torch.randn(M, K, device="cuda", generator=g) * scale
    W = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    b = torch.randn(N, device="cuda", generator=g) if bias else None
    r = torch.randn(M, N, device="cuda", generator=g) if res else None
    out = torch.full((M, N), float("nan"), device="cuda")
    C.capi.check(_lib().cmdi_test_linear(_p(A), _p(W), _p(b), _p(r), _p(out), M, N, K, act, prec, bn, None))
    torch.cuda.synchronize()
    ref = A.double() @ W.double().t()
    if bias:
        ref = ref + b.double()
    if res:
        ref = ref + r.double()
    if act == 1:
        ref = torch.nn.functional.gelu(ref)
    return out.double(), ref


@pytest.mark.parametrize("M,N,K,bn", [
    (128, 128, 64, 128), (128, 256, 64, 256), (1, 8, 8, 128), (130, 264, 512, 128), (1000, 1536, 512, 256),
    (12608, 1536, 512, 256), (12544, 512, 263, 128), (12608, 264, 512, 128), (25216, 512, 1024, 128),
    # negative block_n: the CTA-pair kernel (cta_group::2), tile 256 x |block_n|
    (256, 256, 64, -256), (1, 8, 8, -128), (130, 264, 512, -128), (1000, 1536, 512, -256), (12608, 1536, 512, -256),
    (12608, 512, 1024, -128), (256, 192, 64, -128), (1000, 1536, 512, -128), (12608, 1536, 512, -128), (300, 1000, 512, -256),
    (25216, 1536, 512, -256),
])
def test_linear_bf16x3_meets_fp32_gate(M, N, K, bn):
    out, ref = run_linear(M, N, K, 3, bn)
    assert not torch.isnan(out).any()
    assert torch.allclose(out, ref, **GATE)
    assert (out - ref).abs().max() < 1e-4  # typical 3e-5 at |C| ~ 7


@pytest.mark.parametrize("bn", [256, -256, -128])
@pytest.mark.parametrize("act,res", [(1, False), (0, True), (1, True)])
def test_linear_epilogues(act, res, bn):
    out, ref = run_linear(777, 1024, 512, 3, bn, act=act, res=res)
    assert torch.allclose(out, ref, **GATE)


@pytest.mark.parametrize("bn", [-256, -128, 128])
def test_linear_residual_rederived_from_layernorm_input(monkeypatch, bn):
    """default residual path between encoder sublayers: LayerNorm publishes (mean, rstd) per row and writes only the
    bf16 planes; the next epilogue re-derives LayerNorm's fp32 output from its input"""
    monkeypatch.setenv("CMDI_TEST_RES_LN", "1")
    M, N, K = 777, 512, 512
    g = torch.Generator(device="cuda").manual_seed(3)
    A = torch.randn(M, K, device="cuda", generator=g)
    W = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    b = torch.randn(N, device="cuda", generator=g)
    v = torch.randn(M, N, device="cuda", generator=g) * 2 + 0.3
    out = torch.full((M, N), float("nan"), device="cuda")
    C.capi.check(_lib().cmdi_test_linear(_p(A), _p(W), _p(b), _p(v), _p(out), M, N, K, 0, 3, bn, None))
    torch.cuda.synchronize()
    ln = torch.nn.functional.layer_norm(v.double(), (N,), torch.full((N,), 1.5, device="cuda", dtype=torch.float64),
                                        torch.full((N,), -0.25, device="cuda", dtype=torch.float64), 1e-5)
    ref = A.double() @ W.double().t() + b.double() + ln
    assert torch.allclose(out.double(), ref, **GATE)
    assert (out.double() - ref).abs().max() < 1e-4


def test_linear_plain_bf16_is_bf16_accurate():
    out, ref = run_linear(512, 512, 512, 1, 128)
    err = (out - ref).abs().max().item()
    assert 1e-4 < err < 5e-2  # 2^-9 operand rounding over K=512: ~1e-2; far outside the fp32 gate by design


def test_linear_large_magnitudes_and_zero_rows():
    out, ref = run_linear(300, 512, 512, 3, 128, scale=100.0)
    assert torch.allclose(out, ref, rtol=1e-4, atol=1e-2)
    A = torch.zeros(256, 512, device="cuda")
    W = torch.randn(512, 512, device="cuda")
    out = torch.full((256, 512), float("nan"), device="cuda")
    C.capi.check(_lib().cmdi_test_linear(_p(A), _p(W), None, None, _p(out), 256, 512, 512, 0, 3, 128, None))
    torch.cuda.synchronize()
    assert torch.equal(out, torch.zeros_like(out))


def ref_attention(qkv, nseq, S, H):
    x = qkv.double().view(nseq, S, 3, H, 128)
    q, k, v = x[:, :, 0].transpose(1, 2), x[:, :, 1].transpose(1, 2), x[:, :, 2].transpose(1, 2)
    p = torch.softmax(q @ k.transpose(-1, -2) / 128 ** 0.5, dim=-1)
    return (p @ v).transpose(1, 2).reshape(nseq * S, H * 128)


@pytest.mark.parametrize("nseq,S,H", [(1, 197, 1), (3, 197, 4), (2, 100, 4), (2, 1, 4), (2, 128, 2), (2, 129, 2), (1, 207, 4), (64, 197, 4)])
def test_attention_bf16x3_meets_fp32_gate(nseq, S, H):
    g = torch.Generator(device="cuda").manual_seed(S)
    qkv = torch.randn(nseq * S, 3 * H * 128, device="cuda", generator=g)
    out = torch.full((nseq * S, H * 128), float("nan"), device="cuda")
    C.capi.check(_lib().cmdi_test_attention(_p(qkv), _p(out), nseq, S, H, 3, None))
    torch.cuda.synchronize()
    ref = ref_attention(qkv, nseq, S, H)
    assert torch.allclose(out.double(), ref, **GATE)
    assert (out.double() - ref).abs().max() < 5e-5


def test_attention_peaked_softmax():
    """large logits: exercises the max-subtraction path (one key dominates per query)"""
    nseq, S, H = 2, 197, 4
    g = torch.Generator(device="cuda").manual_seed(5)
    qkv = torch.randn(nseq * S, 3 * H * 128, device="cuda", generator=g)
    qkv[:, : 2 * H * 128] *= 6.0
    out = torch.empty(nseq * S, H * 128, device="cuda")
    C.capi.check(_lib().cmdi_test_attention(_p(qkv), _p(out), nseq, S, H, 3, None))
    torch.cuda.synchronize()
    # the split's error grows with the logit magnitude (|q.k| ~ 400 here, 36x the model's): widen atol accordingly
    err = (out.double() - ref_attention(qkv, nseq, S, H)).abs().max().item()
    assert err < 2e-3, err


def test_layernorm():
    g = torch.Generator(device="cuda").manual_seed(1)
    v = torch.randn(1001, 512, device="cuda", generator=g) * 3 + 0.5
    gamma, beta = torch.randn(512, device="cuda", generator=g), torch.randn(512, device="cuda", generator=g)
    out = torch.empty_like(v)
    C.capi.check(_lib().cmdi_test_layernorm(_p(v), _p(gamma), _p(beta), _p(out), 1001, None))
    torch.cuda.synchronize()
    ref = torch.nn.functional.layer_norm(v.double(), (512,), gamma.double(), beta.double(), 1e-5)
    assert torch.allclose(out.double(), ref, rtol=1e-5, atol=1e-5)


def test_layernorm_backward_matches_autograd():
    g = torch.Generator(device="cuda").manual_seed(2)
    v32 = torch.randn(777, 512, device="cuda", generator=g) * 2 + 0.3
    gamma32 = torch.randn(512, device="cuda", generator=g)
    dy32 = torch.randn(777, 512, device="cuda", generator=g)
    v = v32.double().requires_grad_(True)
    y = torch.nn.functional.layer_norm(v, (512,), gamma32.double(), torch.zeros(512, device="cuda", dtype=torch.float64), 1e-5)
    (ref,) = torch.autograd.grad(y, v, dy32.double())
    out = torch.empty(777, 512, device="cuda")
    C.capi.check(_lib().cmdi_test_layernorm_bwd(_p(dy32), _p(v32), _p(gamma32), _p(out), 777, None))
    torch.cuda.synchronize()
    err = (out.double() - ref).abs().max().item()
    assert err < 2e-5, err  # fp32 kernel vs fp64 autograd on identical fp32 inputs (|dV| up to ~4)


@pytest.mark.parametrize("nseq,S,H", [(1, 197, 1), (3, 197, 4), (2, 50, 4), (2, 5, 2), (2, 1, 4), (2, 128, 2), (2, 129, 2),
                                      (1, 207, 4), (64, 197, 4)])
def test_attention_backward_matches_autograd(nseq, S, H):
    g = torch.Generator(device="cuda").manual_seed(S)
    qkv = torch.randn(nseq * S, 3 * H * 128, device="cuda", generator=g)
    dO = torch.randn(nseq * S, H * 128, device="cuda", generator=g)
    x = qkv.double().requires_grad_(True)
    out = ref_attention(x, nseq, S, H)
    (ref,) = torch.autograd.grad(out, x, dO.double())
    got = torch.full_like(qkv, float("nan"))
    C.capi.check(_lib().cmdi_test_attention_bwd(_p(qkv), _p(dO), _p(got), nseq, S, H, None))
    torch.cuda.synchronize()
    # tcgen05 kernel: every product with the bf16 hi/lo split (attention_bwd_tc.cu)
    assert torch.allclose(got.double(), ref, rtol=1e-3, atol=1e-4)
    assert (got.double() - ref).abs().max() < 1e-4


def test_attention_backward_cuda_core_kernel_agrees(monkeypatch):
    """the fp32 CUDA-core kernel (test-only TU attention_bwd_simt_test.cu) stays as the independent implementation of the same math"""
    monkeypatch.setenv("CMDI_TEST_ATTN_BWD_SIMT", "1")
    nseq, S, H = 2, 197, 4
    g = torch.Generator(device="cuda").manual_seed(5)
    qkv = torch.randn(nseq * S, 3 * H * 128, device="cuda", generator=g)
    dO = torch.randn(nseq * S, H * 128, device="cuda", generator=g)
    simt = torch.full_like(qkv, float("nan"))
    C.capi.check(_lib().cmdi_test_attention_bwd(_p(qkv), _p(dO), _p(simt), nseq, S, H, None))
    monkeypatch.delenv("CMDI_TEST_ATTN_BWD_SIMT")
    tc = torch.full_like(qkv, float("nan"))
    C.capi.check(_lib().cmdi_test_attention_bwd(_p(qkv), _p(dO), _p(tc), nseq, S, H, None))
    torch.cuda.synchronize()
    assert (simt - tc).abs().max() < 1e-4


def test_counter_based_normal_generator():
    n = 263 * 196
    a = torch.empty(8, n, device="cuda")
    C.capi.check(_lib().cmdi_test_normal(_p(a), 8, n, 1234, 7, 0, None))
    b = torch.empty(4, n, device="cuda")
    C.capi.check(_lib().cmdi_test_normal(_p(b), 4, n, 1234, 7, 4, None))  # samples 4..7 generated on their own
    c = torch.empty(8, n, device="cuda")
    C.capi.check(_lib().cmdi_test_normal(_p(c), 8, n, 1235, 7, 0, None))
    torch.cuda.synchronize()
    assert torch.equal(a[4:], b)          # keyed by the GLOBAL sample index: independent of sharding
    assert not torch.equal(a, c)
    x = a.double().flatten()
    assert abs(x.mean()) < 5e-3 and abs(x.var() - 1) < 1e-2 and abs((x ** 3).mean()) < 2e-2 and abs((x ** 4).mean() - 3) < 5e-2
    assert torch.isfinite(a).all() and a.abs().max() < 7


@pytest.mark.parametrize("numel", [1000, 4 * 263 * 196, 64 * 263 * 196, 5_000_003])
def test_torch_compatible_normal_stream_is_bit_exact(numel):
    """CMDI_RNG_TORCH: the engine regenerates torch.randn's CUDA stream from (seed, philox offset) -- the noise a
    reference GPU run draws at gaussian_diffusion.py:696 / :1248 / :1407."""
    from condmdi_b200.diffusion import _cuda_rng_state, aten_launch_policy
    dev = torch.device("cuda:0")
    torch.manual_seed(20240917)
    torch.randn(12345, device=dev)  # move the generator off offset 0
    threads, inc = aten_launch_policy(numel, dev)
    for _ in range(2):              # two consecutive draws: the offset bookkeeping matters for the second
        seed, off = _cuda_rng_state(dev)
        ref = torch.randn(numel, device=dev)
        assert _cuda_rng_state(dev) == (seed, off + inc)
        out = torch.empty(numel, device=dev)
        C.capi.check(_lib().cmdi_test_normal_aten(_p(out), numel, seed, off, threads, None))
        torch.cuda.synchronize()
        assert torch.equal(out, ref), f"max |d| = {(out - ref).abs().max().item()}"


# ---------------------------------------------------------------------------------------------------
# the diffusion-step kernel against the oracle's formulas evaluated by torch on the CPU
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def step_engine():
    eng = C.Engine(torch.device("cuda:0"), max_batch=4)
    yield eng
    eng.close()


def _step_inputs(B=3, seed=0):
    g = torch.Generator().manual_seed(seed)
    mk = lambda: torch.randn(B, 263, 1, 196, generator=g)  # noqa: E731
    return dict(out_c=mk(), out_u=mk(), x=mk(), noise=mk(), x_obs=mk(), scale=torch.tensor([2.5, 0.0, -1.0])[:B],
                mask=O.get_keyframes_mask(torch.zeros(B, 263, 1, 196), torch.tensor([196, 120, 57])[:B], "benchmark_sparse", 5))


@pytest.mark.parametrize("respacing,sampler,eta,t", [("", 0, 0.0, 999), ("", 0, 0.0, 1), ("", 0, 0.0, 0), ("ddim50", 1, 0.0, 49),
                                                   ("ddim50", 1, 0.0, 0), ("ddim100", 1, 0.5, 60), ("ddim100", 1, 1.0, 0)])
@pytest.mark.parametrize("cfg,impute", [(False, False), (True, False), (True, True), (False, True)])
def test_diffusion_step_matches_oracle(step_engine, respacing, sampler, eta, t, cfg, impute):
    tab = O.make_tables(respacing)
    step_engine.set_schedule(tab.betas, tab.timestep_map)
    d = _step_inputs()
    B = d["x"].shape[0]
    tt = torch.tensor([t] * B)
    stop_at = 1
    # oracle formulas (p_mean_variance tail + p_sample / ddim_sample) with the model output given
    out = d["out_u"] + (d["scale"].view(-1, 1, 1, 1) * (d["out_c"] - d["out_u"])) if cfg else d["out_c"]
    M = d["mask"]
    if impute and t >= stop_at:
        out = (out * ~M) + (d["x_obs"] * M)
    x0 = out
    if sampler == 0:
        mean = O.extract(tab.posterior_mean_coef1, tt, x0.shape) * x0 + O.extract(tab.posterior_mean_coef2, tt, x0.shape) * d["x"]
        nonzero = (tt != 0).float().view(-1, 1, 1, 1)
        ref = mean + nonzero * torch.exp(0.5 * O.extract(tab.posterior_log_variance_clipped, tt, x0.shape)) * d["noise"]
    else:
        eps = (O.extract(tab.sqrt_recip_alphas_cumprod, tt, x0.shape) * d["x"] - x0) / O.extract(tab.sqrt_recipm1_alphas_cumprod, tt, x0.shape)
        ab, abp = O.extract(tab.alphas_cumprod, tt, x0.shape), O.extract(tab.alphas_cumprod_prev, tt, x0.shape)
        sigma = eta * torch.sqrt((1 - abp) / (1 - ab)) * torch.sqrt(1 - ab / abp)
        nonzero = (tt != 0).float().view(-1, 1, 1, 1)
        ref = x0 * torch.sqrt(abp) + torch.sqrt(1 - abp - sigma ** 2) * eps + nonzero * sigma * d["noise"]
    cu = lambda v: v.cuda().contiguous()  # noqa: E731
    x_next, pred = step_engine.test_step(sampler, eta, t, cu(d["out_c"]), cu(d["out_u"]) if cfg else None, cu(d["scale"]),
                                         cu(d["x"]), cu(d["noise"]), impute, stop_at, cu(d["x_obs"]),
                                         cu(M.to(torch.uint8)))
    torch.cuda.synchronize()
    # same fp32 operation order as the reference; only exp/sqrt may differ in the last ulp between libraries
    assert torch.allclose(x_next.cpu(), ref, rtol=2e-6, atol=2e-6)
    assert torch.equal(pred.cpu(), x0)  # CFG combine + imputation blend are bit-exact
    if impute and t >= stop_at:
        assert torch.equal(pred.cpu()[M], d["x_obs"][M])  # observed entries are exactly the observations
