// The sampling engine behind the C ABI of include/condmdi_b200.h.
//
// One engine per device.  It owns (a) the MDM weights as bf16 hi/lo planes + their TMA descriptors,
// (b) the diffusion tables as fp32 device arrays, (c) every activation buffer of one denoiser pass, sized
// once for 2*max_batch sequences (the CFG cond+uncond pass is one batch-doubled pass), and (d) one captured
// CUDA graph per loop configuration.  A sampling step is 20 kernel launches of this library (plus one memset of the
// chain's dependency counters) and nothing else:
//
//   token_rows -> frame-embed GEMM -> QKV_0 GEMM -> 8 x [attention, chain: out-proj(+residual), FFN1(+GELU),
//                 FFN2(+residual), QKV_{l+1} | output head] -> diffusion_step
//
// with every LayerNorm folded into the GEMMs around it (run_denoiser_chain).  Guided steps and CMDI_CHAIN=0 run the
// unchained pass instead: one launch per linear layer plus the LayerNorm kernels, 60 launches per step.
//
// The step index lives on the device (decremented by diffusion_step), so the same graph is replayed for
// every step of a loop with no host work in between (reference: one Python iteration + ~150 PyTorch ops
// + several H2D table copies per step, gaussian_diffusion.py:1270-1297, :2225, respace.py:129).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/condmdi_b200.h"
#include "kernels.h"

using namespace cmdi;

struct UnetModel;  // engine_unet.inc

namespace {

#define CK(expr)                                                                                    \
  do {                                                                                              \
    cudaError_t _e = (expr);                                                                        \
    if (_e != cudaSuccess) {                                                                        \
      set_last_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__);   \
      return 1;                                                                                     \
    }                                                                                               \
  } while (0)
#define CKI(expr)          \
  do {                     \
    if ((expr) != 0) return 1; \
  } while (0)

constexpr int kDModel = 512;
constexpr int kBnWide = 256;    // QKV, FFN1
constexpr int kBnNarrow = 128;  // N = 512 / 264 outputs: more tiles per wave

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

struct Planes {  // a bf16 hi/lo operand: [rows, ld] row-major, with TMA maps for a given box height
  __nv_bfloat16* hi = nullptr;
  __nv_bfloat16* lo = nullptr;
  int rows = 0, cols = 0, ld = 0;
  CUtensorMap map_hi{}, map_lo{};
  CUtensorMap pair_hi{}, pair_lo{};  // same planes, box height halved: W operand of the CTA-pair kernel
  CUtensorMap st_hi{}, st_lo{};      // same planes as a TMA-store target: box {64, 32}
  CUtensorMap st32_hi{}, st32_lo{};  // ... box {32, 32}, 64-byte swizzle (32-column slices of the chained epilogue)
  CUtensorMap tap_hi{}, tap_lo{};    // A operand of a k-tap convolution: box {64, 136} (the rows of all taps at once)
  bool has_tap = false;
};

struct LayerW {
  Planes wqkv, wo, w1, w2;
  float *bqkv = nullptr, *bo = nullptr, *b1 = nullptr, *b2 = nullptr;
  float *g1 = nullptr, *be1 = nullptr, *g2 = nullptr, *be2 = nullptr;
};

struct LayerWT {  // transposed weight planes for dX = dY W
  Planes wqkvT, woT, w1T, w2T;
};
struct LayerStash {  // forward values the backward pass of one layer needs
  Planes qkv;
  CUtensorMap q_hi{}, q_lo{}, kv_hi{}, kv_lo{}, kh_hi{}, kh_lo{};
  float *v1 = nullptr, *v2 = nullptr, *pre = nullptr;
};

struct FoldedW {  // a linear layer with the LayerNorm in front of it folded in (LinearParams::fold_stats)
  Planes w;            // W * gamma
  float* c = nullptr;  // [N] sum_k W[n,k] gamma[k]
  float* d = nullptr;  // [N] sum_k W[n,k] beta[k] + b[n]
};
struct ChainTables {  // per number of sequences: the phase lists of the chained launches, one list per encoder layer
  ChainPhaseDesc* dev = nullptr;  // [layers][kMaxChainPhases]
  std::vector<int> total_tiles;   // per layer
  int num_phases = 4;
};

struct GraphKey {  // compared with memcmp: no padding bytes
  int B, cfg, sampler, impute, stop_at, tape_mode, has_cond;
  float eta;
  const void* tape;
  int uncond, guided;
  bool operator<(const GraphKey& o) const { return memcmp(this, &o, sizeof(GraphKey)) < 0; }
};

}  // namespace

struct cmdi_engine {
  cmdi_model_cfg cfg{};
  int device = 0, num_sms = 148;
  int nsplit = 3;
  int debug = 0;            // CMDI_DEBUG (bring-up knob)
  bool no_graph = false;    // CMDI_NO_GRAPH=1: plain stream launches even when the caller asks for graph replay
  float2 *ln_stats1 = nullptr, *ln_stats2 = nullptr;  // (mean, rstd) per token row published by norm1 / norm2
  int D = 263, D_pad = 264, L = 196, S = 197, ff = 1024, H = 4, layers = 8, maxB = 0;
  int max_seqs = 0, seq_rows = 0, seq_rows_pad = 0, frame_rows = 0, frame_rows_pad = 0;
  std::vector<void*> allocs;
  // weights
  Planes w_in, w_out;
  float *b_in = nullptr, *b_out = nullptr;
  std::vector<LayerW> lw;
  float *pe = nullptr;  // [5000, 512]
  float *te_w0 = nullptr, *te_b0 = nullptr, *te_w2 = nullptr, *te_b2 = nullptr;
  float *et_w = nullptr, *et_b = nullptr;
  bool weights_loaded = false, temb_valid = false;
  float* temb_table = nullptr;  // [5000, 512] time_embed(pe[t]) for every ORIGINAL timestep t
  Planes pe_p, te_w0_p, te_w2_p, temb_h_p;  // operands of the timestep-embedding table GEMMs
  CUtensorMap temb_st{};
  // schedule
  int T = 0;
  std::vector<double> h_sqrt_acp, h_sqrt_1m_acp;
  std::vector<int> h_tmap;
  float* tables = nullptr;  // 7 x [T]
  int* d_tmap = nullptr;
  StepTables tab{};
  // activations
  float* x_state = nullptr;
  Planes x_state_p;
  float *xseq = nullptr, *x1 = nullptr, *vsum = nullptr, *model_out = nullptr, *pred_x0 = nullptr, *x_obs = nullptr;
  Planes xseq_p, x1_p, qkv_p, attn_p, ffh_p;
  CUtensorMap q_map_hi{}, q_map_lo{}, kv_map_hi{}, kv_map_lo{}, kh_map_hi{}, kh_map_lo{};  // Q {64,128}, K/V {64,208}, K half {64,104}
  CUtensorMap vsum_st{};  // fp32 TMA-store target for the pre-LayerNorm sums
  CUtensorMap xseq_st{};  // fp32 TMA-store target of xseq (backward pass)
  uint8_t* obs_mask = nullptr;
  float *cond_emb = nullptr, *cond_proj = nullptr, *text_scale = nullptr;
  int* step_ctr = nullptr;  // [2]: step index, block-arrival counter
  RngState* rng = nullptr;  // generator state of the running loop (device-resident: step graphs do not depend on it)
  float *ref_a = nullptr, *ref_b = nullptr;  // reference-layout staging [maxB, D, L]
  uint8_t *ref_mask = nullptr, *ymask = nullptr;
  // reconstruction guidance
  std::vector<LayerWT> lwt;
  Planes w_inT, w_outT;
  std::vector<LayerStash> stash;
  bool stash_ready = false;
  float2* attn_stats = nullptr;          // [seq_rows_pad, H] softmax statistics handed from pass 0 to pass 1 of the attention backward
  CUtensorMap do_f_hi{}, do_f_lo{};      // attn_p planes (dO) as 208-row operands
  Planes seed_p;               // dL/d(model output rows), frame-major [2*frame_rows_pad, D_pad]
  float* guide_grad = nullptr; // dL/dz per pass, frame-major [2*frame_rows_pad, D_pad]
  float* guide_coef = nullptr; // [T] w_r[t] * sqrt(alpha_bar_t) / 2
  // forward path with LayerNorm folded into the consuming linear layers and the linear layers of a layer chained into one
  // persistent launch (gemm_chain.cu).  CMDI_CHAIN=0 selects the round-1 path (one launch per layer + LayerNorm kernels),
  // which guided steps (they stash LayerNorm inputs for the backward pass) always use.
  bool use_chain = true;
  int chain_skip = 0;         // CMDI_CHAIN_SKIP=4 / 2: timing decomposition without operand loads / without MMAs (wrong results)
  std::vector<FoldedW> f_qkv, f_w1;
  FoldedW f_out;
  std::vector<float*> beta_bo, beta_b2;         // [layer]: norm2_{l-1}.bias + out_proj_l.bias, norm1_l.bias + linear2_l.bias (chained epilogues)
  std::vector<CUtensorMap> wo_chain, w2_chain;  // [layer][hi, lo]: wo / w2 planes with the chain's W box
  float2 *stats1 = nullptr, *stats2 = nullptr;  // [seq_rows_pad][16] partial row statistics of v1 / v2 (32-column slices)
  int* chain_ctr = nullptr;                     // [layers][3][max_m_pairs] dependency counters, zeroed every pass
  int max_m_pairs = 0;
  long long* chain_dbg = nullptr;               // CMDI_CHAIN_DBG=1: cycle counters of layer 1's chain during cmdi_profile_pass
  std::map<int, ChainTables> chain_tables;
  UnetModel* unet = nullptr;  // MDM_UNET denoiser (cfg.arch == CMDI_ARCH_UNET): engine_unet.inc
  std::map<GraphKey, cudaGraphExec_t> graphs;
  int64_t launches = 0;
};

namespace {

template <class T>
int dev_alloc(cmdi_engine* e, T** out, size_t count) {
  void* p = nullptr;
  const size_t bytes = (count * sizeof(T) + 255) / 256 * 256;
  CK(cudaMalloc(&p, bytes));
  CK(cudaMemset(p, 0, bytes));
  e->allocs.push_back(p);
  *out = reinterpret_cast<T*>(p);
  return 0;
}

int alloc_planes(cmdi_engine* e, Planes* pl, int rows, int cols, int ld, int box_rows) {
  pl->rows = rows; pl->cols = cols; pl->ld = ld;
  CKI(dev_alloc(e, &pl->hi, (size_t)rows * ld));
  CKI(dev_alloc(e, &pl->lo, (size_t)rows * ld));
  CKI(make_tmap_bf16_2d(&pl->map_hi, pl->hi, rows, cols, ld, 64, box_rows));
  CKI(make_tmap_bf16_2d(&pl->map_lo, pl->lo, rows, cols, ld, 64, box_rows));
  CKI(make_tmap_bf16_2d(&pl->pair_hi, pl->hi, rows, cols, ld, 64, box_rows / 2));
  CKI(make_tmap_bf16_2d(&pl->pair_lo, pl->lo, rows, cols, ld, 64, box_rows / 2));
  CKI(make_tmap_bf16_2d(&pl->st_hi, pl->hi, rows, cols, ld, 64, 32));
  CKI(make_tmap_bf16_2d(&pl->st_lo, pl->lo, rows, cols, ld, 64, 32));
  CKI(make_tmap_bf16_2d(&pl->st32_hi, pl->hi, rows, cols, ld, 32, 32));
  CKI(make_tmap_bf16_2d(&pl->st32_lo, pl->lo, rows, cols, ld, 32, 32));
  if (box_rows == 128 && rows >= 136) {
    CKI(make_tmap_bf16_2d(&pl->tap_hi, pl->hi, rows, cols, ld, 64, 136));
    CKI(make_tmap_bf16_2d(&pl->tap_lo, pl->lo, rows, cols, ld, 64, 136));
    pl->has_tap = true;
  }
  return 0;
}

// fp32 source (host or device) -> device fp32 copy of `count` floats
int upload_f32(cmdi_engine* e, float* dst, const cmdi_tensor_desc& t, size_t count, cudaStream_t s) {
  if ((size_t)t.numel != count) {
    set_last_error("tensor %s: expected %zu elements, got %lld", t.name, count, (long long)t.numel);
    return 1;
  }
  CK(cudaMemcpyAsync(dst, t.data, count * 4, t.on_host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, s));
  return 0;
}

// fp32 [rows, cols] source -> bf16 planes (zero padded to pl.ld / pl.rows)
int upload_planes(cmdi_engine* e, Planes& pl, const cmdi_tensor_desc& t, int rows, int cols, float* scratch, cudaStream_t s,
                  Planes* transposed = nullptr) {
  if ((size_t)t.numel != (size_t)rows * cols) {
    set_last_error("tensor %s: expected %d x %d elements, got %lld", t.name, rows, cols, (long long)t.numel);
    return 1;
  }
  const float* src = t.data;
  if (t.on_host) {
    CK(cudaMemcpyAsync(scratch, t.data, (size_t)rows * cols * 4, cudaMemcpyHostToDevice, s));
    src = scratch;
  }
  CK(launch_split_planes(src, rows, cols, cols, pl.hi, pl.lo, pl.ld, s));
  if (transposed) CK(launch_transpose_split(src, rows, cols, transposed->hi, transposed->lo, transposed->ld, s));
  return 0;
}

int run_linear(cmdi_engine* e, const Planes& a, const Planes& w, const LinearParams& p_in, int block_n, cudaStream_t s,
               const Planes* out_planes = nullptr, const CUtensorMap* out_f32 = nullptr);

int ensure_temb(cmdi_engine* e, cudaStream_t s) {
  if (e->temb_valid) return 0;
  // TimestepEmbedder (mdm.py:345-353) for every original timestep: time_embed(pe[t]), once per weight load, as two
  // launches of the pair GEMM (round 1 ran this table on fp32 CUDA cores: 2 x 0.65 ms on every weight load)
  const int n = 5000;
  CK(launch_split_planes(e->pe, n, kDModel, kDModel, e->pe_p.hi, e->pe_p.lo, kDModel, s));
  CK(launch_split_planes(e->te_w0, kDModel, kDModel, kDModel, e->te_w0_p.hi, e->te_w0_p.lo, kDModel, s));
  CK(launch_split_planes(e->te_w2, kDModel, kDModel, kDModel, e->te_w2_p.hi, e->te_w2_p.lo, kDModel, s));
  LinearParams t0{};
  t0.M = n; t0.N = kDModel; t0.K = kDModel; t0.nsplit = 3; t0.nsplit_out = 3; t0.bias = e->te_b0; t0.act = 2;
  t0.out_hi = e->temb_h_p.hi; t0.out_lo = e->temb_h_p.lo; t0.ld_bf = kDModel;
  CKI(run_linear(e, e->pe_p, e->te_w0_p, t0, kBnNarrow, s, &e->temb_h_p));
  LinearParams t2{};
  t2.M = n; t2.N = kDModel; t2.K = kDModel; t2.nsplit = 3; t2.nsplit_out = 3; t2.bias = e->te_b2;
  t2.out_f32 = e->temb_table; t2.ld_f32 = kDModel;
  CKI(run_linear(e, e->temb_h_p, e->te_w2_p, t2, kBnNarrow, s, nullptr, &e->temb_st));
  e->launches += 5;
  e->temb_valid = true;
  return 0;
}

int run_linear(cmdi_engine* e, const Planes& a, const Planes& w, const LinearParams& p_in, int block_n, cudaStream_t s,
               const Planes* out_planes, const CUtensorMap* out_f32) {
  LinearParams p = p_in;
  p.debug = e->debug;
  LinearStoreMaps st;
  if (out_planes) { st.hi = &out_planes->st_hi; st.lo = &out_planes->st_lo; }
  st.f32 = out_f32;
  if (a.has_tap) { st.a_tap_hi = &a.tap_hi; st.a_tap_lo = &a.tap_lo; }
  CK(launch_linear_pair(a.map_hi, a.map_lo, w.pair_hi, w.pair_lo, p, block_n, e->num_sms, s, &st));
  return 0;
}

}  // namespace
#include "engine_unet.inc"
namespace {

bool chain_eligible(const cmdi_engine* e);
int prepare_chain(cmdi_engine* e, int nseq);
int run_denoiser_chain(cmdi_engine* e, int B, bool dup, int n_cond_seqs, bool has_cond, const int* tmap_dev, cudaStream_t s,
                       std::vector<cudaEvent_t>* evs, int reps);

// One denoiser pass over `nseq` sequences whose frame features are in x_state planes (first B sequences;
// with dup the frame embedding is written for sequences [0,B) and [B,2B)).
int run_denoiser(cmdi_engine* e, int B, bool dup, int n_cond_seqs, bool has_cond, const int* tmap_dev, cudaStream_t s,
                 std::vector<cudaEvent_t>* evs = nullptr, int reps = 1, std::vector<LayerStash>* stash = nullptr) {
  if (e->unet) return unet_run(e, e->unet, B, dup, n_cond_seqs, has_cond, tmap_dev, s);
  if (!stash && chain_eligible(e)) return run_denoiser_chain(e, B, dup, n_cond_seqs, has_cond, tmap_dev, s, evs, reps);
  auto mark = [&]() -> int {
    if (!evs) return 0;
    cudaEvent_t ev;
    CK(cudaEventCreate(&ev));
    CK(cudaEventRecord(ev, s));
    evs->push_back(ev);
    return 0;
  };
  CKI(mark());
  const int nseq = dup ? 2 * B : B;
  const int M = nseq * e->S;
  TokenParams tk{};
  tk.temb_table = e->temb_table; tk.step_ptr = e->step_ctr; tk.timestep_map = tmap_dev;
  tk.cond_proj = has_cond ? e->cond_proj : nullptr; tk.uncond_proj = has_cond ? e->et_b : nullptr;
  tk.pe0 = e->pe; tk.num_seqs = nseq; tk.n_cond_seqs = n_cond_seqs; tk.seq_len = e->S;
  tk.x_f32 = e->xseq; tk.x_hi = e->xseq_p.hi; tk.x_lo = e->xseq_p.lo;
  for (int r_ = 0; r_ < reps; ++r_) CK(launch_token_rows(tk, s));
  CKI(mark());

  // LayerNorm writes only the bf16 planes and its row statistics; the sublayer that needs its fp32 output as the
  // residual re-derives it in the epilogue from LayerNorm's input (bit-identical, 26 MB less traffic per LayerNorm)
  LinearParams p{};
  // frame embedding + positional encoding (mdm.py:271, :279-280)
  p.M = B * e->L; p.N = kDModel; p.K = e->D; p.nsplit = e->nsplit; p.bias = e->b_in; p.pos_enc = e->pe;
  p.rowmap = ROWMAP_FRAMES_TO_SEQ; p.frames = e->L; p.dup_row_offset = dup ? B * e->S : 0;
  p.out_f32 = e->xseq; p.ld_f32 = kDModel; p.out_hi = e->xseq_p.hi; p.out_lo = e->xseq_p.lo; p.ld_bf = kDModel;
  p.nsplit_out = e->nsplit;
  for (int r_ = 0; r_ < reps; ++r_) CKI(run_linear(e, e->x_state_p, e->w_in, p, kBnNarrow, s));
  CKI(mark());

  for (int l = 0; l < e->layers; ++l) {
    const LayerW& w = e->lw[l];
    LayerStash* ls = stash ? &(*stash)[l] : nullptr;  // guided steps keep what the backward pass needs, per layer
    Planes& qkv_out = ls ? ls->qkv : e->qkv_p;
    float* v1_out = ls ? ls->v1 : e->vsum;
    float* v2_out = ls ? ls->v2 : e->vsum;
    // QKV projection
    LinearParams q{};
    q.M = M; q.N = 3 * kDModel; q.K = kDModel; q.nsplit = e->nsplit; q.bias = w.bqkv;
    q.out_hi = qkv_out.hi; q.out_lo = qkv_out.lo; q.ld_bf = 3 * kDModel; q.nsplit_out = e->nsplit;
    for (int r_ = 0; r_ < reps; ++r_) CKI(run_linear(e, e->xseq_p, w.wqkv, q, kBnWide, s, &qkv_out));
    CKI(mark());
    // attention core
    AttnParams a{};
    a.num_seqs = nseq; a.seq_len = e->S; a.num_heads = e->H; a.nsplit = e->nsplit; a.nsplit_out = e->nsplit;
    a.out_hi = e->attn_p.hi; a.out_lo = e->attn_p.lo; a.ld_out = kDModel;
    const AttnMaps am = ls ? AttnMaps{&ls->q_hi, &ls->q_lo, &ls->kh_hi, &ls->kh_lo, &ls->kv_hi, &ls->kv_lo, &e->attn_p.st_hi, &e->attn_p.st_lo}
                           : AttnMaps{&e->q_map_hi, &e->q_map_lo, &e->kh_map_hi, &e->kh_map_lo, &e->kv_map_hi, &e->kv_map_lo, &e->attn_p.st_hi, &e->attn_p.st_lo};
    for (int r_ = 0; r_ < reps; ++r_) CK(launch_attention(am, a, s));
    CKI(mark());
    // out-proj + residual, then LayerNorm1
    {
      LinearParams o{};
      o.M = M; o.N = kDModel; o.K = kDModel; o.nsplit = e->nsplit; o.bias = w.bo; o.residual = e->xseq; o.ld_res = kDModel;
      if (l > 0) {
        // residual = norm2 of the previous layer, from its input (in place when that is the shared vsum buffer)
        o.residual = nullptr; o.ln_src = stash ? (*stash)[l - 1].v2 : e->vsum; o.ld_ln = kDModel; o.ln_stats = e->ln_stats2;
        o.ln_gamma = e->lw[l - 1].g2; o.ln_beta = e->lw[l - 1].be2;
      }
      o.out_f32 = v1_out; o.ld_f32 = kDModel; o.nsplit_out = e->nsplit;
      for (int r_ = 0; r_ < reps; ++r_) CKI(run_linear(e, e->attn_p, w.wo, o, kBnNarrow, s, nullptr, ls ? nullptr : &e->vsum_st));
      CKI(mark());
      for (int r_ = 0; r_ < reps; ++r_)
        CK(launch_layernorm512(v1_out, w.g1, w.be1, 1e-5f, M, nullptr, e->x1_p.hi, e->nsplit == 3 ? e->x1_p.lo : nullptr, s, e->ln_stats1));
      CKI(mark());
    }
    // FFN
    LinearParams f1{};
    f1.M = M; f1.N = e->ff; f1.K = kDModel; f1.nsplit = e->nsplit; f1.bias = w.b1; f1.act = 1;
    f1.out_hi = e->ffh_p.hi; f1.out_lo = e->ffh_p.lo; f1.ld_bf = e->ff; f1.nsplit_out = e->nsplit;
    if (ls) { f1.out_f32 = ls->pre; f1.ld_f32 = e->ff; f1.f32_pre = 1; }  // pre-activation for the GELU backward
    for (int r_ = 0; r_ < reps; ++r_) CKI(run_linear(e, e->x1_p, w.w1, f1, kBnWide, s, &e->ffh_p));
    CKI(mark());
    {
      LinearParams f2{};
      f2.M = M; f2.N = kDModel; f2.K = e->ff; f2.nsplit = e->nsplit; f2.bias = w.b2;
      f2.ln_src = v1_out; f2.ld_ln = kDModel; f2.ln_stats = e->ln_stats1; f2.ln_gamma = w.g1; f2.ln_beta = w.be1;
      f2.out_f32 = v2_out; f2.ld_f32 = kDModel; f2.nsplit_out = e->nsplit;
      for (int r_ = 0; r_ < reps; ++r_) CKI(run_linear(e, e->ffh_p, w.w2, f2, kBnNarrow, s, nullptr, ls ? nullptr : &e->vsum_st));
      CKI(mark());
      for (int r_ = 0; r_ < reps; ++r_)
        CK(launch_layernorm512(v2_out, w.g2, w.be2, 1e-5f, M, nullptr, e->xseq_p.hi, e->nsplit == 3 ? e->xseq_p.lo : nullptr, s, e->ln_stats2));
      CKI(mark());
    }
  }
  // output head on tokens 1.. (mdm.py:284 "[1:]", :304-305)
  LinearParams h{};
  h.M = M; h.N = e->D_pad; h.K = kDModel; h.nsplit = e->nsplit; h.bias = e->b_out;
  h.rowmap = ROWMAP_SEQ_TO_FRAMES; h.frames = e->L; h.out_f32 = e->model_out; h.ld_f32 = e->D_pad; h.nsplit_out = e->nsplit;
  for (int r_ = 0; r_ < reps; ++r_) CKI(run_linear(e, e->xseq_p, e->w_out, h, kBnNarrow, s));
  CKI(mark());
  return 0;
}
bool chain_eligible(const cmdi_engine* e) {
  return e->use_chain && e->debug == 0 && e->layers >= 1;
}

// Phase lists for `nseq` sequences: layer l = [out-proj_l, FFN1_l, FFN2_l, QKV_{l+1} | output head].
int get_chain_tables(cmdi_engine* e, int nseq, const ChainTables** out) {
  auto it = e->chain_tables.find(nseq);
  if (it != e->chain_tables.end()) {
    *out = &it->second;
    return 0;
  }
  const int M = nseq * e->S;
  const int m_pairs = (M + 255) / 256;
  std::vector<ChainPhaseDesc> host((size_t)e->layers * kMaxChainPhases);
  ChainTables ct;
  ct.total_tiles.assign(e->layers, 0);
  auto base = [&](ChainPhaseDesc& d, const Planes& a, const CUtensorMap& w_hi, const CUtensorMap& w_lo, int N, int K, int bn) {
    memset(&d, 0, sizeof(d));
    d.a_hi = a.map_hi; d.a_lo = a.map_lo; d.w_hi = w_hi; d.w_lo = w_lo;
    d.o_hi = a.map_hi; d.o_lo = a.map_hi;  // placeholders unless set below
    ChainPhaseInfo& pi = d.info;
    pi.p.M = M; pi.p.N = N; pi.p.K = K; pi.p.nsplit = e->nsplit; pi.p.nsplit_out = e->nsplit; pi.p.rowmap = ROWMAP_IDENTITY;
    pi.p.debug = e->chain_skip;
    pi.block_n = bn; pi.num_m_pairs = m_pairs; pi.num_n_blocks = (N + bn - 1) / bn; pi.num_k_blocks = (K + 63) / 64;
  };
  for (int l = 0; l < e->layers; ++l) {
    const LayerW& w = e->lw[l];
    ChainPhaseDesc* ph = &host[(size_t)l * kMaxChainPhases];
    int* ctr = e->chain_ctr + (size_t)l * 3 * e->max_m_pairs;
    // out-proj + residual -> v1 (planes + partial statistics)
    base(ph[0], e->attn_p, e->wo_chain[2 * l], e->wo_chain[2 * l + 1], kDModel, kDModel, kBnWide);
    {
      LinearParams& p = ph[0].info.p;
      if (l == 0) { p.bias = w.bo; p.residual = e->xseq; p.ld_res = kDModel; }
      else {
        // bias folded into the beta of the re-derived LayerNorm residual: one vector (and 32 shuffles + adds per slice) less
        p.ld_ln = kDModel; p.ln_partials = e->stats2; p.ln_gamma = e->lw[l - 1].g2; p.ln_beta = e->beta_bo[l];
        p.ln_src_hi = e->xseq_p.hi; p.ln_src_lo = e->xseq_p.lo;
      }
      p.out_hi = e->x1_p.hi; p.out_lo = e->x1_p.lo; p.ld_bf = kDModel; p.stats_out = e->stats1;
      ph[0].o_hi = e->x1_p.st32_hi; ph[0].o_lo = e->x1_p.st32_lo;
      ph[0].info.done_ctr = ctr;
    }
    // FFN1 (norm1 folded) + GELU -> hidden planes
    base(ph[1], e->x1_p, e->f_w1[l].w.pair_hi, e->f_w1[l].w.pair_lo, e->ff, kDModel, kBnWide);
    {
      LinearParams& p = ph[1].info.p;
      p.bias = e->f_w1[l].d; p.fold_c = e->f_w1[l].c; p.fold_stats = e->stats1; p.act = 1;
      p.out_hi = e->ffh_p.hi; p.out_lo = e->ffh_p.lo; p.ld_bf = e->ff;
      ph[1].info.pair_epilogue = 1; ph[1].o_hi = e->ffh_p.st_hi; ph[1].o_lo = e->ffh_p.st_lo;
      ph[1].info.wait_ctr = ctr; ph[1].info.wait_target = ph[0].info.num_n_blocks * 2;
      ph[1].info.done_ctr = ctr + e->max_m_pairs;
    }
    // FFN2 + residual LN1(v1) -> v2 (planes + partial statistics)
    base(ph[2], e->ffh_p, e->w2_chain[2 * l], e->w2_chain[2 * l + 1], kDModel, e->ff, kBnWide);
    {
      LinearParams& p = ph[2].info.p;
      p.ld_ln = kDModel; p.ln_partials = e->stats1; p.ln_gamma = w.g1; p.ln_beta = e->beta_b2[l];
      p.ln_src_hi = e->x1_p.hi; p.ln_src_lo = e->x1_p.lo;
      p.out_hi = e->xseq_p.hi; p.out_lo = e->xseq_p.lo; p.ld_bf = kDModel; p.stats_out = e->stats2;
      ph[2].o_hi = e->xseq_p.st32_hi; ph[2].o_lo = e->xseq_p.st32_lo;
      ph[2].info.wait_ctr = ctr + e->max_m_pairs; ph[2].info.wait_target = ph[1].info.num_n_blocks * 2;
      ph[2].info.done_ctr = ctr + 2 * e->max_m_pairs;
    }
    if (l + 1 < e->layers) {
      // next layer's QKV projection (norm2 folded)
      const FoldedW& fq = e->f_qkv[l + 1];
      base(ph[3], e->xseq_p, fq.w.pair_hi, fq.w.pair_lo, 3 * kDModel, kDModel, kBnWide);
      LinearParams& p = ph[3].info.p;
      p.bias = fq.d; p.fold_c = fq.c; p.fold_stats = e->stats2;
      p.out_hi = e->qkv_p.hi; p.out_lo = e->qkv_p.lo; p.ld_bf = 3 * kDModel;
      ph[3].info.pair_epilogue = 1; ph[3].o_hi = e->qkv_p.st_hi; ph[3].o_lo = e->qkv_p.st_lo;
    } else {
      // output head on tokens 1.. (norm2 of the last layer folded), frame-major fp32 rows
      base(ph[3], e->xseq_p, e->f_out.w.pair_hi, e->f_out.w.pair_lo, e->D_pad, kDModel, kBnWide);
      LinearParams& p = ph[3].info.p;
      p.bias = e->f_out.d; p.fold_c = e->f_out.c; p.fold_stats = e->stats2;
      p.rowmap = ROWMAP_SEQ_TO_FRAMES; p.frames = e->L; p.out_f32 = e->model_out; p.ld_f32 = e->D_pad;
    }
    ph[3].info.wait_ctr = ctr + 2 * e->max_m_pairs; ph[3].info.wait_target = ph[2].info.num_n_blocks * 2;
    int tiles = 0;
    for (int i = 0; i < kMaxChainPhases; ++i) {
      ph[i].info.tile_begin = tiles;
      tiles += ph[i].info.num_m_pairs * ph[i].info.num_n_blocks;
      ph[i].info.tile_end = tiles;
    }
    ct.total_tiles[l] = tiles;
  }
  CKI(dev_alloc(e, &ct.dev, host.size()));
  CK(cudaMemcpy(ct.dev, host.data(), host.size() * sizeof(ChainPhaseDesc), cudaMemcpyHostToDevice));
  auto ins = e->chain_tables.emplace(nseq, std::move(ct));
  *out = &ins.first->second;
  return 0;
}

// Build (outside any stream capture: it allocates) the phase lists a pass over `nseq` sequences will use.
int prepare_chain(cmdi_engine* e, int nseq) {
  if (!chain_eligible(e)) return 0;
  const ChainTables* ct = nullptr;
  return get_chain_tables(e, nseq, &ct);
}

// The denoiser pass with LayerNorm folded into the consuming linear layers and each encoder layer's linear layers
// chained into one launch: token rows, frame embedding, QKV_0, then per layer {attention, chain}: 3 + 2 * layers launches.
int run_denoiser_chain(cmdi_engine* e, int B, bool dup, int n_cond_seqs, bool has_cond, const int* tmap_dev, cudaStream_t s,
                       std::vector<cudaEvent_t>* evs, int reps) {
  auto mark = [&]() -> int {
    if (!evs) return 0;
    cudaEvent_t ev;
    CK(cudaEventCreate(&ev));
    CK(cudaEventRecord(ev, s));
    evs->push_back(ev);
    return 0;
  };
  const int nseq = dup ? 2 * B : B;
  const int M = nseq * e->S;
  const ChainTables* ct = nullptr;
  CKI(get_chain_tables(e, nseq, &ct));
  // the dependency counters of all chained launches of this pass start from zero (one memset node per step)
  CK(cudaMemsetAsync(e->chain_ctr, 0, (size_t)e->layers * 3 * e->max_m_pairs * sizeof(int), s));
  CKI(mark());
  TokenParams tk{};
  tk.temb_table = e->temb_table; tk.step_ptr = e->step_ctr; tk.timestep_map = tmap_dev;
  tk.cond_proj = has_cond ? e->cond_proj : nullptr; tk.uncond_proj = has_cond ? e->et_b : nullptr;
  tk.pe0 = e->pe; tk.num_seqs = nseq; tk.n_cond_seqs = n_cond_seqs; tk.seq_len = e->S;
  tk.x_f32 = e->xseq; tk.x_hi = e->xseq_p.hi; tk.x_lo = e->xseq_p.lo;
  for (int r_ = 0; r_ < reps; ++r_) CK(launch_token_rows(tk, s));
  CKI(mark());
  LinearParams p{};
  p.M = B * e->L; p.N = kDModel; p.K = e->D; p.nsplit = e->nsplit; p.bias = e->b_in; p.pos_enc = e->pe;
  p.rowmap = ROWMAP_FRAMES_TO_SEQ; p.frames = e->L; p.dup_row_offset = dup ? B * e->S : 0;
  p.out_f32 = e->xseq; p.ld_f32 = kDModel; p.out_hi = e->xseq_p.hi; p.out_lo = e->xseq_p.lo; p.ld_bf = kDModel;
  p.nsplit_out = e->nsplit;
  for (int r_ = 0; r_ < reps; ++r_) CKI(run_linear(e, e->x_state_p, e->w_in, p, kBnNarrow, s));
  CKI(mark());
  LinearParams q{};
  q.M = M; q.N = 3 * kDModel; q.K = kDModel; q.nsplit = e->nsplit; q.bias = e->lw[0].bqkv;
  q.out_hi = e->qkv_p.hi; q.out_lo = e->qkv_p.lo; q.ld_bf = 3 * kDModel; q.nsplit_out = e->nsplit;
  for (int r_ = 0; r_ < reps; ++r_) CKI(run_linear(e, e->xseq_p, e->lw[0].wqkv, q, kBnWide, s, &e->qkv_p));
  CKI(mark());
  AttnParams a{};
  a.num_seqs = nseq; a.seq_len = e->S; a.num_heads = e->H; a.nsplit = e->nsplit; a.nsplit_out = e->nsplit;
  a.out_hi = e->attn_p.hi; a.out_lo = e->attn_p.lo; a.ld_out = kDModel;
  const AttnMaps am{&e->q_map_hi, &e->q_map_lo, &e->kh_map_hi, &e->kh_map_lo, &e->kv_map_hi, &e->kv_map_lo, &e->attn_p.st_hi, &e->attn_p.st_lo};
  for (int l = 0; l < e->layers; ++l) {
    for (int r_ = 0; r_ < reps; ++r_)
      CK(launch_attention(am, a, s));
    CKI(mark());
    for (int r_ = 0; r_ < reps; ++r_) {
      if (reps > 1)  // profiling repeats one launch back to back: its counters start from zero each time
        CK(cudaMemsetAsync(e->chain_ctr + (size_t)l * 3 * e->max_m_pairs, 0, (size_t)3 * e->max_m_pairs * sizeof(int), s));
      CK(launch_linear_chain(ct->dev + (size_t)l * kMaxChainPhases, kMaxChainPhases, ct->total_tiles[l], e->num_sms, s,
                             (evs && l == 1) ? e->chain_dbg : nullptr));
    }
    CKI(mark());
  }
  return 0;
}

int ensure_stash(cmdi_engine* e) {
  if (e->stash_ready) return 0;
  CK(configure_attention_bwd_tc_kernel());
  e->stash.resize(e->layers);
  int rc = 0;
  rc = rc || dev_alloc(e, &e->attn_stats, (size_t)e->seq_rows_pad * e->H);
  rc = rc || make_tmap_bf16_2d(&e->do_f_hi, e->attn_p.hi, e->seq_rows_pad, kDModel, kDModel, 64, kAttnKeyPad);
  rc = rc || make_tmap_bf16_2d(&e->do_f_lo, e->attn_p.lo, e->seq_rows_pad, kDModel, kDModel, 64, kAttnKeyPad);
  for (auto& ls : e->stash) {
    rc = rc || alloc_planes(e, &ls.qkv, e->seq_rows_pad, 3 * kDModel, 3 * kDModel, 128);
    rc = rc || make_tmap_bf16_2d(&ls.q_hi, ls.qkv.hi, e->seq_rows_pad, 3 * kDModel, 3 * kDModel, 64, 128);
    rc = rc || make_tmap_bf16_2d(&ls.q_lo, ls.qkv.lo, e->seq_rows_pad, 3 * kDModel, 3 * kDModel, 64, 128);
    rc = rc || make_tmap_bf16_2d(&ls.kv_hi, ls.qkv.hi, e->seq_rows_pad, 3 * kDModel, 3 * kDModel, 64, kAttnKeyPad);
    rc = rc || make_tmap_bf16_2d(&ls.kv_lo, ls.qkv.lo, e->seq_rows_pad, 3 * kDModel, 3 * kDModel, 64, kAttnKeyPad);
    rc = rc || make_tmap_bf16_2d(&ls.kh_hi, ls.qkv.hi, e->seq_rows_pad, 3 * kDModel, 3 * kDModel, 64, kAttnKeyPad / 2);
    rc = rc || make_tmap_bf16_2d(&ls.kh_lo, ls.qkv.lo, e->seq_rows_pad, 3 * kDModel, 3 * kDModel, 64, kAttnKeyPad / 2);
    rc = rc || dev_alloc(e, &ls.v1, (size_t)e->seq_rows_pad * kDModel);
    rc = rc || dev_alloc(e, &ls.v2, (size_t)e->seq_rows_pad * kDModel);
    rc = rc || dev_alloc(e, &ls.pre, (size_t)e->seq_rows_pad * e->ff);
  }
  rc = rc || alloc_planes(e, &e->seed_p, 2 * e->frame_rows_pad, e->D_pad, e->D_pad, 128);
  rc = rc || dev_alloc(e, &e->guide_grad, (size_t)2 * e->frame_rows_pad * e->D_pad);
  if (rc) return 1;
  e->stash_ready = true;
  return 0;
}

// Backward pass of the (CFG-wrapped) denoiser w.r.t. its input, seeded with dL/dx0_hat of the reconstruction loss
// (gaussian_diffusion.py:415-416).  Result: guide_grad[nseq * L, D_pad] (cond rows, then uncond rows under CFG).
// Scratch: xseq / x1 (fp32 + planes) carry the running gradients; qkv_p / attn_p / ffh_p the per-layer ones.
constexpr int kBackwardLaunchesPerLayer = 8;  // the attention backward is two launches (dQ pass, dK/dV pass)
int run_backward(cmdi_engine* e, int B, bool cfg, cudaStream_t s) {
  const int nseq = cfg ? 2 * B : B;
  const int M = nseq * e->S, MF = nseq * e->L;
  GuidanceSeedParams gp{};
  gp.B = B; gp.L = e->L; gp.D = e->D; gp.D_pad = e->D_pad; gp.cfg = cfg; gp.model_out = e->model_out;
  gp.text_scale = e->text_scale; gp.x_obs = e->x_obs; gp.obs_mask = e->obs_mask; gp.seed_hi = e->seed_p.hi; gp.seed_lo = e->seed_p.lo;
  CK(launch_guidance_seed(gp, s));
  // output head backward: d(xseq) rows s >= 1; the token rows receive no gradient from the head
  CK(cudaMemsetAsync(e->xseq, 0, (size_t)M * kDModel * 4, s));
  LinearParams h{};
  h.M = MF; h.N = kDModel; h.K = e->D_pad; h.nsplit = e->nsplit; h.rowmap = ROWMAP_FRAMES_TO_SEQ; h.frames = e->L;
  h.out_f32 = e->xseq; h.ld_f32 = kDModel; h.nsplit_out = e->nsplit;
  CKI(run_linear(e, e->seed_p, e->w_outT, h, kBnNarrow, s));
  for (int l = e->layers - 1; l >= 0; --l) {
    const LayerW& w = e->lw[l];
    const LayerWT& wt = e->lwt[l];
    LayerStash& ls = e->stash[l];
    // LayerNorm2 backward: xseq (dY) -> x1 (dV2)
    CK(launch_layernorm512_bwd(e->xseq, ls.v2, w.g2, 1e-5f, M, e->x1, e->x1_p.hi, e->x1_p.lo, s));
    // linear2 backward fused with the GELU backward: dPre = (dV2 W2) * gelu'(pre)
    LinearParams b2{};
    b2.M = M; b2.N = e->ff; b2.K = kDModel; b2.nsplit = e->nsplit; b2.grad_aux = ls.pre; b2.ld_aux = e->ff;
    b2.out_hi = e->ffh_p.hi; b2.out_lo = e->ffh_p.lo; b2.ld_bf = e->ff; b2.nsplit_out = e->nsplit;
    CKI(run_linear(e, e->x1_p, wt.w2T, b2, kBnWide, s, &e->ffh_p));
    // linear1 backward + the skip path: dX1 = dPre W1 + dV2
    LinearParams b1{};
    b1.M = M; b1.N = kDModel; b1.K = e->ff; b1.nsplit = e->nsplit; b1.residual = e->x1; b1.ld_res = kDModel;
    b1.out_f32 = e->xseq; b1.ld_f32 = kDModel; b1.nsplit_out = e->nsplit;
    CKI(run_linear(e, e->ffh_p, wt.w1T, b1, kBnNarrow, s, nullptr, &e->xseq_st));
    // LayerNorm1 backward: xseq (dX1) -> x1 (dV1)
    CK(launch_layernorm512_bwd(e->xseq, ls.v1, w.g1, 1e-5f, M, e->x1, e->x1_p.hi, e->x1_p.lo, s));
    // out-proj backward: dAttn = dV1 Wo
    LinearParams bo{};
    bo.M = M; bo.N = kDModel; bo.K = kDModel; bo.nsplit = e->nsplit;
    bo.out_hi = e->attn_p.hi; bo.out_lo = e->attn_p.lo; bo.ld_bf = kDModel; bo.nsplit_out = e->nsplit;
    CKI(run_linear(e, e->x1_p, wt.woT, bo, kBnNarrow, s, &e->attn_p));
    // attention backward: (Q, K, V, dAttn) -> dQ | dK | dV
    AttnBwdParams ab{};
    ab.num_seqs = nseq; ab.seq_len = e->S; ab.num_heads = e->H; ab.qkv_hi = ls.qkv.hi; ab.qkv_lo = ls.qkv.lo;
    ab.do_hi = e->attn_p.hi; ab.do_lo = e->attn_p.lo; ab.ld_do = kDModel; ab.dqkv_hi = e->qkv_p.hi; ab.dqkv_lo = e->qkv_p.lo;
    ab.ld_dqkv = 3 * kDModel; ab.nsplit = e->nsplit; ab.stats = e->attn_stats;
    AttnBwdTcMaps bm{&ls.q_hi, &ls.q_lo, &ls.kv_hi, &ls.kv_lo, &e->attn_p.map_hi, &e->attn_p.map_lo, &e->do_f_hi, &e->do_f_lo,
                     &e->qkv_p.st_hi, &e->qkv_p.st_lo};
    CK(launch_attention_bwd_tc(bm, ab, s));
    // QKV projection backward + the skip path: dX = dQKV Wqkv + dV1
    LinearParams bq{};
    bq.M = M; bq.N = kDModel; bq.K = 3 * kDModel; bq.nsplit = e->nsplit; bq.residual = e->x1; bq.ld_res = kDModel;
    bq.out_f32 = e->xseq; bq.ld_f32 = kDModel; bq.nsplit_out = e->nsplit;
    if (l == 0) { bq.out_hi = e->xseq_p.hi; bq.out_lo = e->xseq_p.lo; bq.ld_bf = kDModel; }
    CKI(run_linear(e, e->qkv_p, wt.wqkvT, bq, kBnNarrow, s, l == 0 ? &e->xseq_p : nullptr, &e->xseq_st));
  }
  // frame embedding backward: dz rows (frame-major); the token rows of dxseq are dropped
  LinearParams fi{};
  fi.M = M; fi.N = e->D_pad; fi.K = kDModel; fi.nsplit = e->nsplit; fi.rowmap = ROWMAP_SEQ_TO_FRAMES; fi.frames = e->L;
  fi.out_f32 = e->guide_grad; fi.ld_f32 = e->D_pad; fi.nsplit_out = e->nsplit;
  CKI(run_linear(e, e->xseq_p, e->w_inT, fi, kBnNarrow, s));
  return 0;
}
int launches_per_backward(const cmdi_engine* e) {
  return 3 + e->layers * kBackwardLaunchesPerLayer + 1;
}

int launches_per_pass(const cmdi_engine* e, bool guided = false) {
  if (e->unet) return unet_launches_per_pass(e->unet);
  if (!guided && chain_eligible(e)) return 3 + 2 * e->layers;
  return 1 + 1 + e->layers * 7 + 1;
}

int check_ready(cmdi_engine* e, int B, bool need_schedule) {
  if (!e->weights_loaded) {
    set_last_error("weights not loaded (cmdi_load_weights)");
    return 1;
  }
  if (need_schedule && e->T == 0) {
    set_last_error("schedule not set (cmdi_set_schedule)");
    return 1;
  }
  if (B < 1 || B > e->maxB) {
    set_last_error("batch %d outside [1, max_batch=%d]", B, e->maxB);
    return 1;
  }
  return 0;
}

}  // namespace

// ==================================================================================================
// C ABI
// ==================================================================================================
extern "C" int cmdi_engine_create(const cmdi_model_cfg* cfg, int device, cmdi_engine** out) {
  if (!cfg || !out) {
    set_last_error("null argument");
    return 1;
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    set_last_error("no CUDA device: condmdi_b200 has no CPU fallback");
    return 1;
  }
  CK(cudaSetDevice(device));
  cudaDeviceProp prop{};
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    set_last_error("device %d is sm_%d%d; this library contains sm_100a code only (B200)", device, prop.major, prop.minor);
    return 1;
  }
  const bool is_unet = cfg->arch == CMDI_ARCH_UNET;
  if (cfg->arch != CMDI_ARCH_TRANS_ENC && !is_unet) {
    set_last_error("unknown architecture %d", cfg->arch);
    return 1;
  }
  if (cfg->latent_dim != kDModel || cfg->njoints < 8 || cfg->max_batch < 1 ||
      (cfg->precision != CMDI_PRECISION_BF16X3 && cfg->precision != CMDI_PRECISION_BF16) ||
      (!is_unet && (cfg->num_heads * 128 != cfg->latent_dim || cfg->ff_size % 256 != 0 || cfg->nframes + 1 > kAttnKeyPad))) {
    set_last_error("unsupported model configuration (need latent_dim=512, 4 heads of 128, ff %% 256 == 0, nframes <= 207)");
    return 1;
  }
  CK(configure_linear2_kernels());
  CK(configure_attention_kernel());
  CK(configure_linear_chain_kernel());
  cmdi_engine* e = new cmdi_engine();
  if (const char* g = getenv("CMDI_DEBUG")) e->debug = atoi(g);
  if (const char* g = getenv("CMDI_NO_GRAPH")) e->no_graph = atoi(g) != 0;
  if (const char* g = getenv("CMDI_CHAIN")) e->use_chain = atoi(g) != 0;
  if (const char* g = getenv("CMDI_CHAIN_SKIP")) e->chain_skip = atoi(g) & 6;
  e->cfg = *cfg; e->device = device; e->num_sms = prop.multiProcessorCount; e->nsplit = cfg->precision;
  // the chained launches spin on counters other CTA pairs bump: every pair must be resident at once
  if (e->use_chain && linear_chain_max_clusters(e->num_sms) < e->num_sms / 2) e->use_chain = false;
  e->D = cfg->njoints; e->D_pad = round_up(cfg->njoints, 8); e->L = cfg->nframes; e->S = cfg->nframes + 1;
  e->ff = is_unet ? 256 : cfg->ff_size; e->H = cfg->num_heads; e->layers = is_unet ? 0 : cfg->num_layers; e->maxB = cfg->max_batch;
  if (is_unet) e->S = 2;  // the transformer's sequence buffers are not used: keep them tiny
  e->max_seqs = 2 * e->maxB;
  e->seq_rows = e->max_seqs * e->S;
  e->seq_rows_pad = round_up(e->seq_rows, 128) + 256;  // attention K/V boxes of the last sequence read 208 rows
  e->frame_rows = e->maxB * e->L;
  e->frame_rows_pad = round_up(e->frame_rows, 128);
  int rc = 0;
#define A(expr) rc = rc || (expr)
  // weights
  A(alloc_planes(e, &e->w_in, kDModel, e->D_pad, e->D_pad, kBnNarrow));
  A(alloc_planes(e, &e->w_out, round_up(e->D_pad, kBnNarrow), kDModel, kDModel, kBnNarrow));
  A(dev_alloc(e, &e->b_in, kDModel));
  A(dev_alloc(e, &e->b_out, round_up(e->D_pad, kBnNarrow)));
  e->lw.resize(e->layers);
  for (auto& w : e->lw) {
    A(alloc_planes(e, &w.wqkv, 3 * kDModel, kDModel, kDModel, kBnWide));
    A(alloc_planes(e, &w.wo, kDModel, kDModel, kDModel, kBnNarrow));
    A(alloc_planes(e, &w.w1, e->ff, kDModel, kDModel, kBnWide));
    A(alloc_planes(e, &w.w2, kDModel, e->ff, e->ff, kBnNarrow));
    A(dev_alloc(e, &w.bqkv, 3 * kDModel)); A(dev_alloc(e, &w.bo, kDModel));
    A(dev_alloc(e, &w.b1, e->ff)); A(dev_alloc(e, &w.b2, kDModel));
    A(dev_alloc(e, &w.g1, kDModel)); A(dev_alloc(e, &w.be1, kDModel));
    A(dev_alloc(e, &w.g2, kDModel)); A(dev_alloc(e, &w.be2, kDModel));
  }
  e->lwt.resize(e->layers);
  for (auto& t : e->lwt) {
    A(alloc_planes(e, &t.wqkvT, kDModel, 3 * kDModel, 3 * kDModel, kBnNarrow));
    A(alloc_planes(e, &t.woT, kDModel, kDModel, kDModel, kBnNarrow));
    A(alloc_planes(e, &t.w1T, kDModel, e->ff, e->ff, kBnNarrow));
    A(alloc_planes(e, &t.w2T, e->ff, kDModel, kDModel, kBnWide));
  }
  A(alloc_planes(e, &e->w_inT, round_up(e->D_pad, kBnNarrow), kDModel, kDModel, kBnNarrow));
  A(alloc_planes(e, &e->w_outT, kDModel, e->D_pad, e->D_pad, kBnNarrow));
  A(dev_alloc(e, &e->pe, (size_t)5000 * kDModel));
  A(dev_alloc(e, &e->te_w0, (size_t)kDModel * kDModel)); A(dev_alloc(e, &e->te_b0, kDModel));
  A(dev_alloc(e, &e->te_w2, (size_t)kDModel * kDModel)); A(dev_alloc(e, &e->te_b2, kDModel));
  A(dev_alloc(e, &e->et_w, (size_t)kDModel * 512)); A(dev_alloc(e, &e->et_b, kDModel));
  A(dev_alloc(e, &e->temb_table, (size_t)5000 * kDModel));
  A(alloc_planes(e, &e->pe_p, 5120, kDModel, kDModel, 128));
  A(alloc_planes(e, &e->temb_h_p, 5120, kDModel, kDModel, 128));
  A(alloc_planes(e, &e->te_w0_p, kDModel, kDModel, kDModel, kBnNarrow));
  A(alloc_planes(e, &e->te_w2_p, kDModel, kDModel, kDModel, kBnNarrow));
  A(make_tmap_2d(&e->temb_st, e->temb_table, 4, 5000, kDModel, kDModel, 32, 32));
  // activations
  A(dev_alloc(e, &e->x_state, (size_t)e->frame_rows_pad * e->D_pad));
  A(alloc_planes(e, &e->x_state_p, e->frame_rows_pad, e->D_pad, e->D_pad, 128));
  A(dev_alloc(e, &e->xseq, (size_t)e->seq_rows_pad * kDModel));
  A(dev_alloc(e, &e->x1, (size_t)e->seq_rows_pad * kDModel));
  A(dev_alloc(e, &e->vsum, (size_t)e->seq_rows_pad * kDModel));
  A(alloc_planes(e, &e->xseq_p, e->seq_rows_pad, kDModel, kDModel, 128));
  A(alloc_planes(e, &e->x1_p, e->seq_rows_pad, kDModel, kDModel, 128));
  A(alloc_planes(e, &e->qkv_p, e->seq_rows_pad, 3 * kDModel, 3 * kDModel, 128));
  A(alloc_planes(e, &e->attn_p, e->seq_rows_pad, kDModel, kDModel, 128));
  A(alloc_planes(e, &e->ffh_p, e->seq_rows_pad, e->ff, e->ff, 128));
  A(make_tmap_bf16_2d(&e->q_map_hi, e->qkv_p.hi, e->seq_rows_pad, 3 * kDModel, 3 * kDModel, 64, 128));
  A(make_tmap_bf16_2d(&e->q_map_lo, e->qkv_p.lo, e->seq_rows_pad, 3 * kDModel, 3 * kDModel, 64, 128));
  A(make_tmap_bf16_2d(&e->kv_map_hi, e->qkv_p.hi, e->seq_rows_pad, 3 * kDModel, 3 * kDModel, 64, kAttnKeyPad));
  A(make_tmap_bf16_2d(&e->kv_map_lo, e->qkv_p.lo, e->seq_rows_pad, 3 * kDModel, 3 * kDModel, 64, kAttnKeyPad));
  A(make_tmap_bf16_2d(&e->kh_map_hi, e->qkv_p.hi, e->seq_rows_pad, 3 * kDModel, 3 * kDModel, 64, kAttnKeyPad / 2));
  A(make_tmap_bf16_2d(&e->kh_map_lo, e->qkv_p.lo, e->seq_rows_pad, 3 * kDModel, 3 * kDModel, 64, kAttnKeyPad / 2));
  A(make_tmap_2d(&e->vsum_st, e->vsum, 4, e->seq_rows_pad, kDModel, kDModel, 32, 32));
  A(make_tmap_2d(&e->xseq_st, e->xseq, 4, e->seq_rows_pad, kDModel, kDModel, 32, 32));
  A(dev_alloc(e, &e->model_out, (size_t)2 * e->frame_rows_pad * e->D_pad));
  A(dev_alloc(e, &e->pred_x0, (size_t)e->frame_rows_pad * e->D_pad));
  A(dev_alloc(e, &e->x_obs, (size_t)e->frame_rows_pad * e->D_pad));
  A(dev_alloc(e, &e->obs_mask, (size_t)e->frame_rows_pad * e->D_pad));
  A(dev_alloc(e, &e->cond_emb, (size_t)e->maxB * 512));
  A(dev_alloc(e, &e->cond_proj, (size_t)e->maxB * kDModel));
  A(dev_alloc(e, &e->text_scale, e->maxB));
  A(dev_alloc(e, &e->step_ctr, 4));
  A(dev_alloc(e, &e->rng, 1));
  // chained forward path: folded weights, partial row statistics, dependency counters
  e->f_qkv.resize(e->layers);
  e->f_w1.resize(e->layers);
  for (int l = 0; l < e->layers; ++l) {
    if (l > 0) {
      A(alloc_planes(e, &e->f_qkv[l].w, 3 * kDModel, kDModel, kDModel, kBnWide));
      A(dev_alloc(e, &e->f_qkv[l].c, 3 * kDModel)); A(dev_alloc(e, &e->f_qkv[l].d, 3 * kDModel));
    }
    A(alloc_planes(e, &e->f_w1[l].w, e->ff, kDModel, kDModel, kBnWide));
    A(dev_alloc(e, &e->f_w1[l].c, e->ff)); A(dev_alloc(e, &e->f_w1[l].d, e->ff));
  }
  A(alloc_planes(e, &e->f_out.w, round_up(e->D_pad, 256), kDModel, kDModel, kBnWide));
  A(dev_alloc(e, &e->f_out.c, round_up(e->D_pad, 256))); A(dev_alloc(e, &e->f_out.d, round_up(e->D_pad, 256)));
  e->wo_chain.resize(2 * e->layers);
  e->beta_bo.assign(e->layers, nullptr); e->beta_b2.assign(e->layers, nullptr);
  for (int l = 0; l < e->layers; ++l) { A(dev_alloc(e, &e->beta_bo[l], kDModel)); A(dev_alloc(e, &e->beta_b2[l], kDModel)); }
  e->w2_chain.resize(2 * e->layers);
  for (int l = 0; l < e->layers && !rc; ++l) {
    const LayerW& w = e->lw[l];
    A(make_tmap_bf16_2d(&e->wo_chain[2 * l], w.wo.hi, kDModel, kDModel, kDModel, 64, kBnWide / 2));
    A(make_tmap_bf16_2d(&e->wo_chain[2 * l + 1], w.wo.lo, kDModel, kDModel, kDModel, 64, kBnWide / 2));
    A(make_tmap_bf16_2d(&e->w2_chain[2 * l], w.w2.hi, kDModel, e->ff, e->ff, 64, kBnWide / 2));
    A(make_tmap_bf16_2d(&e->w2_chain[2 * l + 1], w.w2.lo, kDModel, e->ff, e->ff, 64, kBnWide / 2));
  }
  A(dev_alloc(e, &e->stats1, (size_t)e->seq_rows_pad * 16));
  A(dev_alloc(e, &e->stats2, (size_t)e->seq_rows_pad * 16));
  e->max_m_pairs = (e->seq_rows_pad + 255) / 256;
  A(dev_alloc(e, &e->chain_ctr, (size_t)e->layers * 3 * e->max_m_pairs));
  if (getenv("CMDI_CHAIN_DBG")) A(dev_alloc(e, &e->chain_dbg, (size_t)e->num_sms * kMaxChainPhases * 16));
  A(dev_alloc(e, &e->ln_stats1, (size_t)e->seq_rows_pad));
  A(dev_alloc(e, &e->ln_stats2, (size_t)e->seq_rows_pad));
  A(dev_alloc(e, &e->ref_a, (size_t)e->maxB * e->D * e->L));
  A(dev_alloc(e, &e->ref_b, (size_t)e->maxB * e->D * e->L));
  A(dev_alloc(e, &e->ref_mask, (size_t)e->maxB * e->D * e->L));
  A(dev_alloc(e, &e->ymask, (size_t)e->maxB * e->L));
#undef A
  if (rc) {
    cmdi_engine_destroy(e);
    return 1;
  }
  if (is_unet) {
    e->unet = new UnetModel();
    if (unet_create(e, e->unet, cfg)) {
      cmdi_engine_destroy(e);
      return 1;
    }
  }
  // default positional-encoding buffer (mdm.py:322-330); overwritten if the state dict carries 'sequence_pos_encoder.pe'
  {
    std::vector<float> pe((size_t)5000 * kDModel);
    for (int pos = 0; pos < 5000; ++pos)
      for (int i = 0; i < kDModel; i += 2) {
        const float div = expf((float)i * (float)(-std::log(10000.0) / kDModel));
        pe[(size_t)pos * kDModel + i] = sinf((float)pos * div);
        pe[(size_t)pos * kDModel + i + 1] = cosf((float)pos * div);
      }
    CK(cudaMemcpy(e->pe, pe.data(), pe.size() * 4, cudaMemcpyHostToDevice));
  }
  *out = e;
  return 0;
}

extern "C" int cmdi_engine_destroy(cmdi_engine* e) {
  if (!e) return 0;
  cudaSetDevice(e->device);
  cudaDeviceSynchronize();
  for (auto& kv : e->graphs) cudaGraphExecDestroy(kv.second);
  delete e->unet;
  for (void* p : e->allocs) cudaFree(p);
  if (e->tables) cudaFree(e->tables);
  if (e->d_tmap) cudaFree(e->d_tmap);
  if (e->guide_coef) cudaFree(e->guide_coef);
  delete e;
  return 0;
}

extern "C" int64_t cmdi_launch_count(const cmdi_engine* e) { return e ? e->launches : 0; }

extern "C" int cmdi_load_weights(cmdi_engine* e, const cmdi_tensor_desc* tensors, int n) {
  if (!e || !tensors) {
    set_last_error("null argument");
    return 1;
  }
  CK(cudaSetDevice(e->device));
  cudaStream_t s = 0;
  // staging for host-resident weight matrices: the largest one of this configuration
  float* scratch = nullptr;
  size_t scratch_elems = (size_t)3 * kDModel * kDModel;
  if ((size_t)e->ff * kDModel > scratch_elems) scratch_elems = (size_t)e->ff * kDModel;
  if ((size_t)kDModel * e->D_pad > scratch_elems) scratch_elems = (size_t)kDModel * e->D_pad;
  CK(cudaMalloc(&scratch, scratch_elems * 4));
  struct ScratchGuard { float* p; ~ScratchGuard() { cudaFree(p); } } scratch_guard{scratch};
  std::map<std::string, const cmdi_tensor_desc*> by_name;
  for (int i = 0; i < n; ++i) by_name[tensors[i].name] = &tensors[i];
  std::string missing;
  auto get = [&](const std::string& k) -> const cmdi_tensor_desc* {
    auto it = by_name.find(k);
    if (it == by_name.end()) {
      missing += k + " ";
      return nullptr;
    }
    return it->second;
  };
  int rc = 0;
#define LOAD_F32(dst, key, count)                         \
  do {                                                    \
    const cmdi_tensor_desc* t_ = get(key);                \
    if (t_) rc = rc || upload_f32(e, dst, *t_, count, s); \
  } while (0)
#define LOAD_PL(pl, key, rows, cols, tr)                                        \
  do {                                                                          \
    const cmdi_tensor_desc* t_ = get(key);                                      \
    if (t_) rc = rc || upload_planes(e, pl, *t_, rows, cols, scratch, s, tr);   \
  } while (0)
  if (!e->unet) {
    LOAD_PL(e->w_in, "input_process.poseEmbedding.weight", kDModel, e->D, &e->w_inT);
    LOAD_F32(e->b_in, "input_process.poseEmbedding.bias", kDModel);
    LOAD_PL(e->w_out, "output_process.poseFinal.weight", e->D, kDModel, &e->w_outT);
    LOAD_F32(e->b_out, "output_process.poseFinal.bias", (size_t)e->D);
  }
  LOAD_F32(e->te_w0, "embed_timestep.time_embed.0.weight", (size_t)kDModel * kDModel);
  LOAD_F32(e->te_b0, "embed_timestep.time_embed.0.bias", kDModel);
  LOAD_F32(e->te_w2, "embed_timestep.time_embed.2.weight", (size_t)kDModel * kDModel);
  LOAD_F32(e->te_b2, "embed_timestep.time_embed.2.bias", kDModel);
  if (e->cfg.has_text) {
    LOAD_F32(e->et_w, "embed_text.weight", (size_t)kDModel * 512);
    LOAD_F32(e->et_b, "embed_text.bias", kDModel);
  }
  if (by_name.count("sequence_pos_encoder.pe")) LOAD_F32(e->pe, "sequence_pos_encoder.pe", (size_t)5000 * kDModel);
  if (e->unet && !rc) rc = unet_load_weights(e, e->unet, by_name, missing, s);
  for (int l = 0; l < e->layers; ++l) {
    LayerW& w = e->lw[l];
    const std::string p = "seqTransEncoder.layers." + std::to_string(l) + ".";
    LOAD_PL(w.wqkv, p + "self_attn.in_proj_weight", 3 * kDModel, kDModel, &e->lwt[l].wqkvT);
    LOAD_F32(w.bqkv, p + "self_attn.in_proj_bias", (size_t)3 * kDModel);
    LOAD_PL(w.wo, p + "self_attn.out_proj.weight", kDModel, kDModel, &e->lwt[l].woT);
    LOAD_F32(w.bo, p + "self_attn.out_proj.bias", kDModel);
    LOAD_PL(w.w1, p + "linear1.weight", e->ff, kDModel, &e->lwt[l].w1T);
    LOAD_F32(w.b1, p + "linear1.bias", (size_t)e->ff);
    LOAD_PL(w.w2, p + "linear2.weight", kDModel, e->ff, &e->lwt[l].w2T);
    LOAD_F32(w.b2, p + "linear2.bias", kDModel);
    LOAD_F32(w.g1, p + "norm1.weight", kDModel);
    LOAD_F32(w.be1, p + "norm1.bias", kDModel);
    LOAD_F32(w.g2, p + "norm2.weight", kDModel);
    LOAD_F32(w.be2, p + "norm2.bias", kDModel);
  }
#undef LOAD_F32
#undef LOAD_PL
  // ---- LayerNorm folded into the layers that consume it (chained forward path): W * gamma planes, c, d ----
  if (missing.empty() && !rc && !e->unet) {
    float* folded = nullptr;
    CK(cudaMalloc(&folded, scratch_elems * 4));
    ScratchGuard folded_guard{folded};
    auto fold = [&](FoldedW& fw, const std::string& key, int rows, int cols, const float* gamma, const float* beta,
                    const float* bias_dev) -> int {
      const cmdi_tensor_desc* t = by_name[key];
      const float* src = t->data;
      if (t->on_host) {
        CK(cudaMemcpyAsync(scratch, t->data, (size_t)rows * cols * 4, cudaMemcpyHostToDevice, s));
        src = scratch;
      }
      CK(launch_fold_ln(src, rows, cols, gamma, beta, bias_dev, folded, fw.c, fw.d, s));
      CK(launch_split_planes(folded, rows, cols, cols, fw.w.hi, fw.w.lo, fw.w.ld, s));
      return 0;
    };
    for (int l = 0; l < e->layers && !rc; ++l) {
      const std::string p = "seqTransEncoder.layers." + std::to_string(l) + ".";
      if (l > 0)
        rc = rc || fold(e->f_qkv[l], p + "self_attn.in_proj_weight", 3 * kDModel, kDModel, e->lw[l - 1].g2, e->lw[l - 1].be2, e->lw[l].bqkv);
      rc = rc || fold(e->f_w1[l], p + "linear1.weight", e->ff, kDModel, e->lw[l].g1, e->lw[l].be1, e->lw[l].b1);
    }
    rc = rc || fold(e->f_out, "output_process.poseFinal.weight", e->D, kDModel, e->lw[e->layers - 1].g2, e->lw[e->layers - 1].be2, e->b_out);
    for (int l = 0; l < e->layers && !rc; ++l) {
      if (l > 0) CK(launch_add_vectors(e->lw[l - 1].be2, e->lw[l].bo, e->beta_bo[l], kDModel, s));
      CK(launch_add_vectors(e->lw[l].be1, e->lw[l].b2, e->beta_b2[l], kDModel, s));
    }
    cudaError_t fe = cudaStreamSynchronize(s);
    if (!rc) CK(fe);
  }
  cudaError_t se = cudaStreamSynchronize(s);
  if (!missing.empty()) {
    set_last_error("state dict is missing: %s", missing.c_str());
    return 1;
  }
  if (rc) return 1;
  CK(se);
  e->weights_loaded = true;
  e->temb_valid = false;
  for (auto& kv : e->graphs) cudaGraphExecDestroy(kv.second);
  e->graphs.clear();
  return 0;
}

extern "C" int cmdi_set_schedule(cmdi_engine* e, const double* betas_in, int T, const int64_t* timestep_map) {
  if (!e || !betas_in || T < 2 || !timestep_map) {
    set_last_error("cmdi_set_schedule: bad arguments");
    return 1;
  }
  CK(cudaSetDevice(e->device));
  // float64 tables exactly as GaussianDiffusion.__init__ builds them (gaussian_diffusion.py:183-217),
  // cast to fp32 at the point _extract_into_tensor does (.float() after the gather, :2225).
  std::vector<double> betas(betas_in, betas_in + T), acp(T), acp_prev(T), post_var(T);
  double run = 1.0;
  for (int i = 0; i < T; ++i) {
    if (!(betas[i] > 0 && betas[i] <= 1)) {
      set_last_error("betas must lie in (0, 1]");
      return 1;
    }
    run *= (1.0 - betas[i]);
    acp[i] = run;
  }
  // np.cumprod is a sequential product in float64: identical rounding to the loop above
  for (int i = 0; i < T; ++i) acp_prev[i] = i == 0 ? 1.0 : acp[i - 1];
  std::vector<float> host((size_t)7 * T);
  e->h_sqrt_acp.assign(T, 0.0);
  e->h_sqrt_1m_acp.assign(T, 0.0);
  for (int i = 0; i < T; ++i) post_var[i] = betas[i] * (1.0 - acp_prev[i]) / (1.0 - acp[i]);
  for (int i = 0; i < T; ++i) {
    const double alpha = 1.0 - betas[i];
    host[0 * T + i] = (float)(betas[i] * std::sqrt(acp_prev[i]) / (1.0 - acp[i]));          // posterior_mean_coef1
    host[1 * T + i] = (float)((1.0 - acp_prev[i]) * std::sqrt(alpha) / (1.0 - acp[i]));     // posterior_mean_coef2
    host[2 * T + i] = (float)std::log(post_var[i == 0 ? 1 : i]);                            // posterior_log_variance_clipped
    host[3 * T + i] = (float)std::sqrt(1.0 / acp[i]);                                       // sqrt_recip_alphas_cumprod
    host[4 * T + i] = (float)std::sqrt(1.0 / acp[i] - 1);                                   // sqrt_recipm1_alphas_cumprod
    host[5 * T + i] = (float)acp[i];
    host[6 * T + i] = (float)acp_prev[i];
    e->h_sqrt_acp[i] = std::sqrt(acp[i]);
    e->h_sqrt_1m_acp[i] = std::sqrt(1.0 - acp[i]);
  }
  if (e->tables) cudaFree(e->tables);
  if (e->d_tmap) cudaFree(e->d_tmap);
  e->tables = nullptr; e->d_tmap = nullptr;
  CK(cudaMalloc(&e->tables, host.size() * 4));
  CK(cudaMemcpy(e->tables, host.data(), host.size() * 4, cudaMemcpyHostToDevice));
  e->h_tmap.resize(T);
  for (int i = 0; i < T; ++i) {
    if (timestep_map[i] < 0 || timestep_map[i] >= 5000) {
      set_last_error("timestep_map[%d]=%lld outside the positional table", i, (long long)timestep_map[i]);
      return 1;
    }
    e->h_tmap[i] = (int)timestep_map[i];
  }
  CK(cudaMalloc(&e->d_tmap, (size_t)T * 4));
  CK(cudaMemcpy(e->d_tmap, e->h_tmap.data(), (size_t)T * 4, cudaMemcpyHostToDevice));
  e->T = T;
  e->tab.post_coef1 = e->tables + 0 * T; e->tab.post_coef2 = e->tables + 1 * T; e->tab.post_logvar = e->tables + 2 * T;
  e->tab.sqrt_recip_acp = e->tables + 3 * T; e->tab.sqrt_recipm1_acp = e->tables + 4 * T;
  e->tab.acp = e->tables + 5 * T; e->tab.acp_prev = e->tables + 6 * T;
  for (auto& kv : e->graphs) cudaGraphExecDestroy(kv.second);
  e->graphs.clear();
  return 0;
}

namespace {

// staging helper: returns a device pointer holding `bytes` of user data (copying when the user pointer is host memory)
const void* stage_in(const void* user, void* dev_scratch, size_t bytes, bool host, cudaStream_t s, int* rc) {
  if (!user) return nullptr;
  if (!host) return user;
  cudaError_t e = cudaMemcpyAsync(dev_scratch, user, bytes, cudaMemcpyHostToDevice, s);
  if (e != cudaSuccess) {
    set_last_error("H2D copy failed: %s", cudaGetErrorString(e));
    *rc = 1;
  }
  return dev_scratch;
}

int prepare_cond(cmdi_engine* e, int B, const float* cond_emb_user, bool host, cudaStream_t s) {
  if (!cond_emb_user) return 0;
  if (!e->cfg.has_text) {
    set_last_error("cond_emb given but the engine was created with has_text = 0");
    return 1;
  }
  CK(cudaMemcpyAsync(e->cond_emb, cond_emb_user, (size_t)B * 512 * 4, host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, s));
  // embed_text(enc_text): once per call instead of once per step and pass (mdm.py:249-250 re-runs it every step)
  CK(launch_small_linear(e->cond_emb, e->et_w, e->et_b, e->cond_proj, B, kDModel, 512, 0, s));
  e->launches += 1;
  return 0;
}

// model_kwargs['obs_x0'] / ['obs_mask'] of a keyframe-conditioned MDM_UNET (mdm_unet.py:765-783): staged frame-major once
// per call; the transformer ignores them (SURVEY 8b note 2)
int stage_keyframe_input(cmdi_engine* e, int B, const float* obs_x0, const uint8_t* obs_mask, bool host, cudaStream_t s) {
  if (!e->unet) return 0;
  if ((obs_x0 == nullptr) != (obs_mask == nullptr)) {
    set_last_error("with spatial conditioning, both obs_x0 and obs_mask must be provided (mdm_unet.py:775)");
    return 1;
  }
  if (e->unet->kf && !obs_x0) {
    set_last_error("a keyframe-conditioned UNet needs obs_x0 and obs_mask");
    return 1;
  }
  e->unet->has_kf = e->unet->kf && obs_x0 != nullptr;
  if (!e->unet->has_kf) return 0;
  int rc = 0;
  const size_t n = (size_t)B * e->D * e->L;
  const float* obs = (const float*)stage_in(obs_x0, e->ref_b, n * 4, host, s, &rc);
  const uint8_t* msk = (const uint8_t*)stage_in(obs_mask, e->ref_mask, n, host, s, &rc);
  if (rc) return 1;
  CK(launch_ref_to_frames(obs, B, e->D, e->L, e->D_pad, e->unet->kf_obs, nullptr, nullptr, s));
  CK(launch_mask_to_frames(msk, nullptr, B, e->D, e->L, e->D_pad, e->unet->kf_mask, s));
  e->launches += 2;
  return 0;
}

}  // namespace

extern "C" int cmdi_model_forward(cmdi_engine* e, const cmdi_forward_args* a, float* out, void* stream_) {
  if (!e || !a || !out || !a->x) {
    set_last_error("null argument");
    return 1;
  }
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream_);
  CK(cudaSetDevice(e->device));
  const int B = a->batch;
  CKI(check_ready(e, B, false));
  if (a->cfg && (!a->cond_emb || !a->text_scale)) {
    set_last_error("cfg forward needs cond_emb and text_scale (cfg_sampler.py:26, :35)");
    return 1;
  }
  if (a->timestep < 0 || a->timestep >= 5000) {
    set_last_error("timestep %d outside the positional table", a->timestep);
    return 1;
  }
  const bool host = a->host_buffers != 0;
  const size_t n = (size_t)B * e->D * e->L;
  CKI(ensure_temb(e, s));
  CKI(prepare_chain(e, a->cfg ? 2 * B : B));
  int rc = 0;
  const float* x = (const float*)stage_in(a->x, e->ref_a, n * 4, host, s, &rc);
  if (rc) return 1;
  CK(launch_ref_to_frames(x, B, e->D, e->L, e->D_pad, e->unet ? e->x_state : nullptr, e->x_state_p.hi, e->x_state_p.lo, s));  // the UNet's input builder reads fp32
  CKI(stage_keyframe_input(e, B, a->obs_x0, a->obs_mask, host, s));
  CKI(prepare_cond(e, B, a->cond_emb, host, s));
  if (a->cfg) CK(cudaMemcpyAsync(e->text_scale, a->text_scale, (size_t)B * 4, host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, s));
  CK(launch_set_int(e->step_ctr, a->timestep, s));
  const bool has_cond = a->cond_emb != nullptr;
  const int n_cond = a->uncond ? 0 : B;  // y['uncond'] under the CFG wrapper makes BOTH passes unconditional (cfg_sampler.py:28-33)
  CKI(run_denoiser(e, B, a->cfg != 0, n_cond, has_cond, /*tmap*/ nullptr, s));
  // combine (cfg) into pred_x0 via the step kernel's pass-through mode, then back to the reference layout
  StepParams sp{};
  sp.tab = e->tab; sp.step_ptr = e->step_ctr; sp.advance = 0; sp.B = B; sp.L = e->L; sp.D = e->D; sp.D_pad = e->D_pad;
  sp.sampler = 2; sp.model_out = e->model_out; sp.cfg = a->cfg != 0; sp.text_scale = e->text_scale; sp.x_t = e->x_state;
  sp.x_next = nullptr; sp.pred_xstart = e->pred_x0;
  CK(launch_diffusion_step(sp, s));
  float* dst = host ? e->ref_b : out;
  CK(launch_frames_to_ref(e->pred_x0, B, e->D, e->L, e->D_pad, dst, s));
  e->launches += launches_per_pass(e) + 4;
  if (host) {
    CK(cudaMemcpyAsync(out, e->ref_b, n * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
  }
  return 0;
}

extern "C" int cmdi_sample(cmdi_engine* e, const cmdi_sample_args* a, float* out, void* stream_) {
  if (!e || !a || !out) {
    set_last_error("null argument");
    return 1;
  }
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream_);
  CK(cudaSetDevice(e->device));
  const int B = a->batch;
  CKI(check_ready(e, B, true));
  if (a->sampler != CMDI_SAMPLER_DDPM && a->sampler != CMDI_SAMPLER_DDIM) {
    set_last_error("unknown sampler %d", a->sampler);
    return 1;
  }
  if (a->cfg && (!a->cond_emb || !a->text_scale)) {
    set_last_error("cfg sampling needs cond_emb and text_scale (cfg_sampler.py:26, :35)");
    return 1;
  }
  if ((a->imputate || a->recon_guidance) && (!a->inpainted_motion || !a->inpainting_mask)) {
    set_last_error("imputate / reconstruction_guidance need inpainted_motion and inpainting_mask (editing_util.py:330, :343)");
    return 1;
  }
  if (a->recon_guidance && e->unet) {
    set_last_error("reconstruction guidance (the denoiser's input-VJP) is implemented for the transformer denoiser only");
    return 1;
  }
  if (a->recon_guidance) {
    if (!a->recon_coef) {
      set_last_error("reconstruction_guidance needs recon_coef");
      return 1;
    }
    CKI(ensure_stash(e));
    if (!e->guide_coef) CK(cudaMalloc(&e->guide_coef, (size_t)5000 * 4));
    CK(cudaMemcpyAsync(e->guide_coef, a->recon_coef, (size_t)e->T * 4, cudaMemcpyHostToDevice, s));
  }
  if (a->skip_timesteps < 0 || a->skip_timesteps >= e->T) {
    set_last_error("skip_timesteps %d outside [0, %d)", a->skip_timesteps, e->T);
    return 1;
  }
  const bool host = a->host_buffers != 0;
  const size_t n = (size_t)B * e->D * e->L;
  const int t0 = e->T - 1 - a->skip_timesteps;
  const int nsteps = (a->num_steps > 0 && a->num_steps < t0 + 1) ? a->num_steps : t0 + 1;
  CKI(ensure_temb(e, s));
  CKI(prepare_chain(e, a->cfg ? 2 * B : B));
  int rc = 0;

  // ---- x_T (gaussian_diffusion.py:1245-1248) ----
  const float* xT = (const float*)stage_in(a->x_T, e->ref_a, n * 4, host, s, &rc);
  if (rc) return 1;
  RngState rng{};
  rng.seed = a->seed; rng.sample_offset = a->sample_offset; rng.mode = a->rng_mode;
  rng.aten_offset = a->aten_offset; rng.aten_increment = a->aten_increment; rng.aten_threads = a->aten_threads;
  if (a->rng_mode == CMDI_RNG_TORCH) {
    if (a->aten_threads == 0 || a->aten_increment == 0 || (a->aten_increment & 3) || (a->aten_offset & 3)) {
      set_last_error("rng_mode=CMDI_RNG_TORCH needs aten_threads > 0 and aten_offset / aten_increment multiples of 4");
      return 1;
    }
  } else if (a->rng_mode != CMDI_RNG_ENGINE) {
    set_last_error("unknown rng_mode %d", a->rng_mode);
    return 1;
  }
  if (!xT) {
    if (a->rng_mode == CMDI_RNG_TORCH) {
      CK(launch_fill_normal_aten(e->ref_a, n, a->seed, a->aten_offset, a->aten_threads, s));
      rng.aten_offset += a->aten_increment;  // the per-step draws follow the x_T draw in the stream
    } else {
      CK(launch_fill_normal_ref(e->ref_a, B, (size_t)e->D * e->L, a->seed, 0ull, a->sample_offset, s));
    }
    xT = e->ref_a;
    e->launches += 1;
  }
  CK(launch_set_rng(e->rng, rng, s));
  e->launches += 1;
  // ---- init_image / skip_timesteps: img = q_sample(init_image, t0, img) (:1252-1260) ----
  if (!a->resume && (a->init_image || a->skip_timesteps)) {
    const float* init = (const float*)stage_in(a->init_image, e->ref_b, n * 4, host, s, &rc);
    if (rc) return 1;
    if (!init) {
      CK(cudaMemsetAsync(e->ref_b, 0, n * 4, s));
      init = e->ref_b;
    }
    CK(launch_axpby(init, xT, (float)e->h_sqrt_acp[t0], (float)e->h_sqrt_1m_acp[t0], e->ref_a, n, s));
    xT = e->ref_a;
    e->launches += 1;
  }
  CK(launch_ref_to_frames(xT, B, e->D, e->L, e->D_pad, e->x_state, e->x_state_p.hi, e->x_state_p.lo, s));
  e->launches += 1;
  // ---- keyframes ----
  if (a->imputate || a->recon_guidance) {
    const float* obs = (const float*)stage_in(a->inpainted_motion, e->ref_b, n * 4, host, s, &rc);
    const uint8_t* msk = (const uint8_t*)stage_in(a->inpainting_mask, e->ref_mask, n, host, s, &rc);
    const uint8_t* ym = (const uint8_t*)stage_in(a->y_mask, e->ymask, (size_t)B * e->L, host, s, &rc);
    if (rc) return 1;
    CK(launch_ref_to_frames(obs, B, e->D, e->L, e->D_pad, e->x_obs, nullptr, nullptr, s));
    CK(launch_mask_to_frames(msk, ym, B, e->D, e->L, e->D_pad, e->obs_mask, s));
    e->launches += 2;
  }
  CKI(stage_keyframe_input(e, B, a->obs_x0, a->obs_mask, host, s));
  // ---- conditioning ----
  CKI(prepare_cond(e, B, a->cond_emb, host, s));
  if (a->cfg) CK(cudaMemcpyAsync(e->text_scale, a->text_scale, (size_t)B * 4, host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, s));
  CK(launch_set_int(e->step_ctr, t0, s));
  CK(launch_set_int(e->step_ctr + 2, t0, s));
  e->launches += 2;

  const float* tape = a->noise_tape;
  if (tape && host) {
    set_last_error("noise_tape must be a device pointer (it is a test aid; stage it once outside the call)");
    return 1;
  }
  const bool has_cond = a->cond_emb != nullptr;
  auto enqueue_step = [&](cudaStream_t st, bool guided) -> int {
    CKI(run_denoiser(e, B, a->cfg != 0, a->uncond ? 0 : B, has_cond, e->d_tmap, st, nullptr, 1,
                     guided ? &e->stash : nullptr));
    if (guided) CKI(run_backward(e, B, a->cfg != 0, st));
    StepParams sp{};
    sp.tab = e->tab; sp.step_ptr = e->step_ctr; sp.advance = 1; sp.B = B; sp.L = e->L; sp.D = e->D; sp.D_pad = e->D_pad;
    sp.sampler = a->sampler; sp.eta = a->eta; sp.model_out = e->model_out; sp.cfg = a->cfg != 0; sp.text_scale = e->text_scale;
    sp.x_t = e->x_state; sp.impute = a->imputate != 0; sp.stop_imputation_at = a->stop_imputation_at;
    sp.x_obs = e->x_obs; sp.obs_mask = e->obs_mask;
    sp.guided = guided; sp.guide_grad = e->guide_grad; sp.guide_coef = e->guide_coef;
    sp.noise_ref = tape; sp.tape_t0 = -1; sp.rng = e->rng;  // first step index: step_ctr[2] (graphs do not depend on it)
    sp.x_next = e->x_state; sp.x_next_hi = e->x_state_p.hi; sp.x_next_lo = e->nsplit == 3 ? e->x_state_p.lo : nullptr;
    sp.pred_xstart = e->pred_x0;
    CK(launch_diffusion_step(sp, st));
    return 0;
  };

  auto get_exec = [&](bool guided, cudaGraphExec_t* out_exec) -> int {
    GraphKey key{};
    memset(&key, 0, sizeof(key));
    key.B = B; key.cfg = a->cfg != 0; key.sampler = a->sampler; key.impute = a->imputate != 0;
    key.stop_at = a->stop_imputation_at; key.tape_mode = tape != nullptr; key.has_cond = has_cond; key.eta = a->eta;
    key.tape = tape; key.uncond = a->uncond != 0;  // no first step index: it lives in device memory
    key.guided = guided;
    auto it = e->graphs.find(key);
    if (it != e->graphs.end()) {
      *out_exec = it->second;
      return 0;
    }
    // capture on a private stream so a caller's legacy/default stream is never put into capture mode
    cudaStream_t cs = nullptr;
    CK(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
    cudaGraph_t graph = nullptr;
    CK(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
    const int erc = enqueue_step(cs, guided);
    cudaError_t ce = cudaStreamEndCapture(cs, &graph);
    cudaStreamDestroy(cs);
    if (erc) return 1;
    CK(ce);
    cudaGraphExec_t ex = nullptr;
    CK(cudaGraphInstantiate(&ex, graph, 0));
    cudaGraphDestroy(graph);
    e->graphs[key] = ex;
    *out_exec = ex;
    return 0;
  };
  if (e->graphs.size() > 16) {  // bounded cache; cleared before this call takes any handle out of it
    for (auto& kv : e->graphs) cudaGraphExecDestroy(kv.second);
    e->graphs.clear();
  }
  // one graph per step (capturing 10 or 50 consecutive steps into one graph was measured: no gain)
  cudaGraphExec_t exec[2] = {nullptr, nullptr};  // [guided]

  int dump_i = 0;
  for (int k = 0; k < nsteps; ++k) {
    // utils/editing_util.py:325-333: guidance is active while t >= stop_recguidance_at (t is uniform over the batch)
    const bool guided = a->recon_guidance && (t0 - k) >= a->stop_recguidance_at;
    // use_graph 1: calls of one or two steps are launched directly unless a step graph of this configuration already
    // exists (capturing and instantiating one costs more than it saves there); use_graph 2 (the *_progressive
    // generators: one native call per step, many calls): always through the step graph
    // (a noise tape -- test aid -- is addressed through a kernel argument: per-step calls with a moving tape pointer
    //  would capture a new graph every step, so they are launched directly)
    bool via_graph = a->use_graph && !e->no_graph && (nsteps >= 3 || (a->use_graph >= 2 && !tape));
    if (a->use_graph && !e->no_graph && !via_graph) {
      GraphKey probe{};
      memset(&probe, 0, sizeof(probe));
      probe.B = B; probe.cfg = a->cfg != 0; probe.sampler = a->sampler; probe.impute = a->imputate != 0;
      probe.stop_at = a->stop_imputation_at; probe.tape_mode = tape != nullptr; probe.has_cond = has_cond; probe.eta = a->eta;
      probe.tape = tape; probe.uncond = a->uncond != 0; probe.guided = guided;
      via_graph = e->graphs.count(probe) != 0;
    }
    if (via_graph) {
      if (!exec[guided]) CKI(get_exec(guided, &exec[guided]));
      CK(cudaGraphLaunch(exec[guided], s));
    } else {
      CKI(enqueue_step(s, guided));
    }
    e->launches += launches_per_pass(e, guided) + 1 + (guided ? launches_per_backward(e) : 0);
    if (a->dump_xstart && dump_i < a->n_dump && a->dump_steps[dump_i] == k) {
      if (host) {
        CK(launch_frames_to_ref(e->pred_x0, B, e->D, e->L, e->D_pad, e->ref_b, s));
        CK(cudaMemcpyAsync(a->dump_xstart + (size_t)dump_i * n, e->ref_b, n * 4, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
      } else {
        CK(launch_frames_to_ref(e->pred_x0, B, e->D, e->L, e->D_pad, a->dump_xstart + (size_t)dump_i * n, s));
      }
      e->launches += 1;
      ++dump_i;
    }
  }
  // ---- results back in the reference layout ----
  if (host) {
    CK(launch_frames_to_ref(e->x_state, B, e->D, e->L, e->D_pad, e->ref_a, s));
    CK(cudaMemcpyAsync(out, e->ref_a, n * 4, cudaMemcpyDeviceToHost, s));
    if (a->pred_xstart_out) {
      CK(launch_frames_to_ref(e->pred_x0, B, e->D, e->L, e->D_pad, e->ref_b, s));
      CK(cudaMemcpyAsync(a->pred_xstart_out, e->ref_b, n * 4, cudaMemcpyDeviceToHost, s));
    }
    CK(cudaStreamSynchronize(s));
  } else {
    CK(launch_frames_to_ref(e->x_state, B, e->D, e->L, e->D_pad, out, s));
    if (a->pred_xstart_out) CK(launch_frames_to_ref(e->pred_x0, B, e->D, e->L, e->D_pad, a->pred_xstart_out, s));
  }
  e->launches += a->pred_xstart_out ? 2 : 1;
  return 0;
}

extern "C" int cmdi_test_step(cmdi_engine* e, int sampler, float eta, int t, int B, const float* model_out_c,
                              const float* model_out_u, const float* text_scale, const float* x_t, const float* noise,
                              int impute, int stop_imputation_at, const float* x_obs, const uint8_t* mask, float* x_next,
                              float* pred_xstart, void* stream_) {
  if (!e) {
    set_last_error("null engine");
    return 1;
  }
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream_);
  CK(cudaSetDevice(e->device));
  if (e->T == 0 || B < 1 || B > e->maxB || t < 0 || t >= e->T) {
    set_last_error("cmdi_test_step: bad state/arguments");
    return 1;
  }
  const size_t fr = (size_t)B * e->L * e->D_pad;
  CK(launch_ref_to_frames(model_out_c, B, e->D, e->L, e->D_pad, e->model_out, nullptr, nullptr, s));
  if (model_out_u) CK(launch_ref_to_frames(model_out_u, B, e->D, e->L, e->D_pad, e->model_out + fr, nullptr, nullptr, s));
  CK(launch_ref_to_frames(x_t, B, e->D, e->L, e->D_pad, e->x_state, nullptr, nullptr, s));
  if (impute) {
    CK(launch_ref_to_frames(x_obs, B, e->D, e->L, e->D_pad, e->x_obs, nullptr, nullptr, s));
    CK(launch_mask_to_frames(mask, nullptr, B, e->D, e->L, e->D_pad, e->obs_mask, s));
  }
  if (model_out_u) CK(cudaMemcpyAsync(e->text_scale, text_scale, (size_t)B * 4, cudaMemcpyDeviceToDevice, s));
  CK(launch_set_int(e->step_ctr, t, s));
  StepParams sp{};
  sp.tab = e->tab; sp.step_ptr = e->step_ctr; sp.advance = 0; sp.B = B; sp.L = e->L; sp.D = e->D; sp.D_pad = e->D_pad;
  sp.sampler = sampler; sp.eta = eta; sp.model_out = e->model_out; sp.cfg = model_out_u != nullptr; sp.text_scale = e->text_scale;
  sp.x_t = e->x_state; sp.impute = impute; sp.stop_imputation_at = stop_imputation_at; sp.x_obs = e->x_obs; sp.obs_mask = e->obs_mask;
  sp.noise_ref = noise; sp.tape_t0 = t; sp.x_next = e->x_state; sp.x_next_hi = e->x_state_p.hi; sp.x_next_lo = e->x_state_p.lo;
  sp.pred_xstart = e->pred_x0;
  CK(launch_diffusion_step(sp, s));
  CK(launch_frames_to_ref(e->x_state, B, e->D, e->L, e->D_pad, x_next, s));
  if (pred_xstart) CK(launch_frames_to_ref(e->pred_x0, B, e->D, e->L, e->D_pad, pred_xstart, s));
  return 0;
}

extern "C" int cmdi_recover_from_ric(const float* data, long long stride_seq, long long stride_frame, long long stride_feat,
                                     const float* mean, const float* std, int num_seqs, int nframes, int nfeats,
                                     int joints_num, int abs_3d, float* out, long long ostride_seq, long long ostride_frame,
                                     long long ostride_joint, long long ostride_coord, void* stream_) {
  if (!data || !out || num_seqs < 0 || nframes < 1 || nframes > 2048 || joints_num < 2 || nfeats < 4 + 3 * (joints_num - 1) ||
      ((mean == nullptr) != (std == nullptr))) {
    set_last_error("cmdi_recover_from_ric: bad arguments (need 1 <= nframes <= 2048, nfeats >= 4 + 3*(joints_num-1), "
                   "mean and std both set or both NULL)");
    return 1;
  }
  CK(launch_recover_from_ric(data, stride_seq, stride_frame, stride_feat, mean, std, num_seqs, nframes, joints_num, abs_3d != 0,
                             out, ostride_seq, ostride_frame, ostride_joint, ostride_coord,
                             reinterpret_cast<cudaStream_t>(stream_)));
  return 0;
}

// Per-kernel device times of one denoiser pass (plain launches with CUDA events between them, on the caller's
// stream; each launch is issued `repeats` times back to back and the mean is reported, which hides the host's
// launch latency behind queued work): ms[i] is the i-th launch of the pass in order
//   token_rows, frame_embed, {qkv, attention, out_proj, ln1, ffn1, ffn2, ln2} x layers, out_head.
extern "C" int cmdi_profile_pass(cmdi_engine* e, int batch, int cfg, int repeats, float* ms, int capacity, int* count, void* stream_) {
  if (!e || !ms || !count) {
    set_last_error("null argument");
    return 1;
  }
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream_);
  CK(cudaSetDevice(e->device));
  CKI(check_ready(e, batch, false));
  if (e->unet) {
    set_last_error("cmdi_profile_pass is implemented for the transformer denoiser");
    return 1;
  }
  CKI(ensure_temb(e, s));
  CK(launch_set_int(e->step_ctr, 500, s));
  std::vector<cudaEvent_t> evs;
  const bool has_cond = cfg != 0 && e->cfg.has_text;
  if (cfg && !has_cond) {
    set_last_error("cfg profiling needs a text model");
    return 1;
  }
  if (repeats < 1) repeats = 1;
  CKI(prepare_chain(e, cfg ? 2 * batch : batch));
  const int rc = run_denoiser(e, batch, cfg != 0, batch, has_cond, nullptr, s, &evs, repeats);
  cudaError_t se = cudaStreamSynchronize(s);
  int n = (int)evs.size() - 1;
  if (rc == 0 && se == cudaSuccess) {
    *count = n;
    for (int i = 0; i < n && i < capacity; ++i) {
      cudaEventElapsedTime(&ms[i], evs[i], evs[i + 1]);
      ms[i] /= (float)repeats;
    }
  }
  for (cudaEvent_t ev : evs) cudaEventDestroy(ev);
  if (rc) return 1;
  CK(se);
  if (e->chain_dbg) {
    std::vector<long long> h((size_t)e->num_sms * kMaxChainPhases * 16);
    CK(cudaMemcpy(h.data(), e->chain_dbg, h.size() * 8, cudaMemcpyDeviceToHost));
    CK(cudaMemset(e->chain_dbg, 0, h.size() * 8));
    const char* names[16] = {"tiles", "tma_dep_wait", "tma_slot_wait", "mma_operand_wait", "mma_acc_wait", "epi0_acc_wait", "epi0_slices", "epi0_publish",
                             "s_rowstats", "s_stage_free", "s_loads+acc", "s_fold_bias_res", "s_stats", "s_f32_store", "s_plane_store", "-"};
    for (int ph = 0; ph < kMaxChainPhases; ++ph) {
      double tiles = 0, acc[16] = {0};
      for (int b = 0; b < e->num_sms; ++b) {
        tiles += (double)h[((size_t)b * kMaxChainPhases + ph) * 16];
        for (int k = 1; k < 16; ++k) acc[k] += (double)h[((size_t)b * kMaxChainPhases + ph) * 16 + k];
      }
      // tiles are counted by both CTAs' TMA threads; the MMA counters exist on leaders only
      fprintf(stderr, "chain dbg phase %d: %.0f tile visits (%d repeats);  cycles per tile:", ph, tiles, repeats);
      for (int k = 1; k < 15; ++k) fprintf(stderr, " %s=%.0f", names[k], acc[k] / (tiles > 0 ? tiles : 1) * ((k == 3 || k == 4) ? 2.0 : 1.0));
      fprintf(stderr, "\n");
    }
  }
  e->launches += (int64_t)launches_per_pass(e) * repeats;
  return 0;
}
