// Kernel-level C-ABI entry points used by the parity tests (declared in include/condmdi_b200.h).
// They stage fp32 inputs into the bf16 hi/lo planes the kernels consume, build the TMA descriptors,
// launch the production kernel and hand back fp32 results.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../include/condmdi_b200.h"
#include "kernels.h"

using namespace cmdi;

namespace {

#define CK(expr)                                                                   \
  do {                                                                             \
    cudaError_t _e = (expr);                                                       \
    if (_e != cudaSuccess) {                                                       \
      set_last_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return 1;                                                                    \
    }                                                                              \
  } while (0)

struct DevBuf {
  void* p = nullptr;
  ~DevBuf() {
    if (p) cudaFree(p);
  }
  cudaError_t alloc(size_t bytes) {
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaSuccess) e = cudaMemset(p, 0, bytes);
    return e;
  }
  template <class T>
  T* as() {
    return reinterpret_cast<T*>(p);
  }
};

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

int num_sms_of_current_device() {
  int dev = 0, n = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
  return n;
}

}  // namespace

extern "C" int cmdi_test_linear(const float* A, const float* W, const float* bias, const float* residual, float* C, int M,
                                int N, int K, int act, int precision, int block_n, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  const int bn_abs = block_n < 0 ? -block_n : block_n;
  const int Kp = round_up(K, 8), Mp = round_up(M, 256), Np = round_up(N, bn_abs);
  DevBuf a_hi, a_lo, w_hi, w_lo;
  CK(a_hi.alloc((size_t)Mp * Kp * 2));
  CK(a_lo.alloc((size_t)Mp * Kp * 2));
  CK(w_hi.alloc((size_t)Np * Kp * 2));
  CK(w_lo.alloc((size_t)Np * Kp * 2));
  CK(launch_split_planes(A, M, K, K, a_hi.as<__nv_bfloat16>(), a_lo.as<__nv_bfloat16>(), Kp, stream));
  CK(launch_split_planes(W, N, K, K, w_hi.as<__nv_bfloat16>(), w_lo.as<__nv_bfloat16>(), Kp, stream));
  const bool pair = true;  // every linear layer runs on the CTA-pair kernel (the sign of block_n is accepted and ignored)
  if (block_n < 0) block_n = -block_n;
  CUtensorMap ma_hi, ma_lo, mw_hi, mw_lo;
  if (make_tmap_bf16_2d(&ma_hi, a_hi.p, Mp, Kp, Kp, 64, 128)) return 1;
  if (make_tmap_bf16_2d(&ma_lo, a_lo.p, Mp, Kp, Kp, 64, 128)) return 1;
  if (make_tmap_bf16_2d(&mw_hi, w_hi.p, Np, Kp, Kp, 64, pair ? block_n / 2 : block_n)) return 1;
  if (make_tmap_bf16_2d(&mw_lo, w_lo.p, Np, Kp, Kp, 64, pair ? block_n / 2 : block_n)) return 1;
  CUtensorMap mc_f32;
  if (make_tmap_2d(&mc_f32, C, 4, M, N, N, 32, 32)) return 1;
  LinearStoreMaps stm;
  stm.f32 = &mc_f32;
  LinearParams p{};
  p.M = M; p.N = N; p.K = K; p.nsplit = precision;
  p.bias = bias; p.residual = residual; p.ld_res = N;
  DevBuf ln_g, ln_b, ln_s;
  if (residual && N == 512 && getenv("CMDI_TEST_RES_LN")) {
    // the residual is LayerNorm(`residual`) (gamma = 1.5, beta = -0.25), re-derived in the epilogue from the
    // statistics the LayerNorm kernel publishes
    std::vector<float> hg(512, 1.5f), hb(512, -0.25f);
    CK(ln_g.alloc(512 * 4)); CK(ln_b.alloc(512 * 4)); CK(ln_s.alloc((size_t)M * sizeof(float2)));
    CK(cudaMemcpyAsync(ln_g.p, hg.data(), 512 * 4, cudaMemcpyHostToDevice, stream));
    CK(cudaMemcpyAsync(ln_b.p, hb.data(), 512 * 4, cudaMemcpyHostToDevice, stream));
    CK(cudaStreamSynchronize(stream));
    CK(launch_layernorm512(residual, ln_g.as<float>(), ln_b.as<float>(), 1e-5f, M, nullptr, nullptr, nullptr, stream, ln_s.as<float2>()));
    p.residual = nullptr; p.ln_src = residual; p.ld_ln = N; p.ln_stats = ln_s.as<float2>();
    p.ln_gamma = ln_g.as<float>(); p.ln_beta = ln_b.as<float>();
  }
  p.act = act; p.rowmap = ROWMAP_IDENTITY;
  p.out_f32 = C; p.ld_f32 = N;
  p.nsplit_out = precision;
  if (pair) {
    CK(configure_linear2_kernels());
    DevBuf dbg, o_hi, o_lo;
    CUtensorMap mo_hi, mo_lo;
    const bool want_dbg = getenv("CMDI_TEST_DBG") != nullptr;
    if (const char* d = getenv("CMDI_DEBUG")) p.debug = atoi(d);
    if (want_dbg) {
      CK(dbg.alloc(148 * 16 * 8));
      p.dbg_cycles = dbg.as<long long>();
      CK(o_hi.alloc((size_t)Mp * Np * 2));
      CK(o_lo.alloc((size_t)Mp * Np * 2));
      if (make_tmap_bf16_2d(&mo_hi, o_hi.p, Mp, Np, Np, 64, 32)) return 1;
      if (make_tmap_bf16_2d(&mo_lo, o_lo.p, Mp, Np, Np, 64, 32)) return 1;
      stm.hi = &mo_hi;
      stm.lo = &mo_lo;
      p.out_hi = o_hi.as<__nv_bfloat16>();  // realistic stores: bf16 planes like the engine's QKV / FFN1
      p.out_lo = o_lo.as<__nv_bfloat16>();
      p.ld_bf = Np;
      if (getenv("CMDI_TEST_NOF32")) p.out_f32 = nullptr;
      CK(launch_linear_pair(ma_hi, ma_lo, mw_hi, mw_lo, p, block_n, num_sms_of_current_device(), stream, &stm));
    }
    CK(launch_linear_pair(ma_hi, ma_lo, mw_hi, mw_lo, p, block_n, num_sms_of_current_device(), stream, &stm));
    if (want_dbg) {
      std::vector<long long> h(148 * 16);
      CK(cudaStreamSynchronize(stream));
      CK(cudaMemcpy(h.data(), dbg.p, h.size() * 8, cudaMemcpyDeviceToHost));
      double acc[16] = {0};
      int n_lead = 0, n_all = 0;
      for (int b = 0; b < 148; ++b) {
        if (h[b * 16 + 4] == 0) continue;
        ++n_all;
        for (int k = 4; k < 8; ++k) acc[k] += (double)h[b * 16 + k];
        if (h[b * 16 + 0]) { ++n_lead; for (int k = 0; k < 3; ++k) acc[k] += (double)h[b * 16 + k]; }
      }
      printf("dbg cycles (mean per CTA): mma total=%.0f wait_tmem_empty=%.0f wait_full=%.0f | epi total=%.0f wait_tmem_full=%.0f work=%.0f arrive=%.0f (leaders %d, ctas %d)\n",
             acc[0] / n_lead, acc[1] / n_lead, acc[2] / n_lead, acc[4] / n_all, acc[5] / n_all, acc[6] / n_all, acc[7] / n_all, n_lead, n_all);
      fflush(stdout);
    }
  }
  CK(cudaStreamSynchronize(stream));  // staging buffers are freed on return
  return 0;
}

extern "C" int cmdi_test_layernorm(const float* v, const float* gamma, const float* beta, float* out, int rows,
                                   void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  CK(launch_layernorm512(v, gamma, beta, 1e-5f, rows, out, nullptr, nullptr, stream));
  return 0;
}

extern "C" int cmdi_test_attention(const float* qkv, float* O, int num_seqs, int S, int H, int precision, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  if (S > kAttnKeyPad) {
    set_last_error("cmdi_test_attention: S=%d exceeds %d", S, kAttnKeyPad);
    return 1;
  }
  const int rows = num_seqs * S;
  const int rows_p = round_up(rows, 128) + 256;  // tiles of the last sequence read past its end
  const int ld = 3 * H * 128, ldo = H * 128;
  DevBuf q_hi, q_lo, o_hi, o_lo;
  CK(q_hi.alloc((size_t)rows_p * ld * 2));
  CK(q_lo.alloc((size_t)rows_p * ld * 2));
  CK(o_hi.alloc((size_t)rows_p * ldo * 2));
  CK(o_lo.alloc((size_t)rows_p * ldo * 2));
  CK(launch_split_planes(qkv, rows, ld, ld, q_hi.as<__nv_bfloat16>(), q_lo.as<__nv_bfloat16>(), ld, stream));
  CUtensorMap mq_hi, mq_lo, mkv_hi, mkv_lo;
  if (make_tmap_bf16_2d(&mq_hi, q_hi.p, rows_p, ld, ld, 64, 128)) return 1;
  if (make_tmap_bf16_2d(&mq_lo, q_lo.p, rows_p, ld, ld, 64, 128)) return 1;
  if (make_tmap_bf16_2d(&mkv_hi, q_hi.p, rows_p, ld, ld, 64, kAttnKeyPad)) return 1;
  if (make_tmap_bf16_2d(&mkv_lo, q_lo.p, rows_p, ld, ld, 64, kAttnKeyPad)) return 1;
  CUtensorMap mkh_hi, mkh_lo;
  if (make_tmap_bf16_2d(&mkh_hi, q_hi.p, rows_p, ld, ld, 64, kAttnKeyPad / 2)) return 1;
  if (make_tmap_bf16_2d(&mkh_lo, q_lo.p, rows_p, ld, ld, 64, kAttnKeyPad / 2)) return 1;
  CUtensorMap mo_hi, mo_lo;
  if (make_tmap_bf16_2d(&mo_hi, o_hi.p, rows_p, ldo, ldo, 64, 32)) return 1;
  if (make_tmap_bf16_2d(&mo_lo, o_lo.p, rows_p, ldo, ldo, 64, 32)) return 1;
  CK(configure_attention_kernel());
  const AttnMaps am{&mq_hi, &mq_lo, &mkh_hi, &mkh_lo, &mkv_hi, &mkv_lo, &mo_hi, &mo_lo};
  AttnParams p{};
  p.num_seqs = num_seqs; p.seq_len = S; p.num_heads = H; p.nsplit = precision; p.nsplit_out = 3;
  p.out_hi = o_hi.as<__nv_bfloat16>(); p.out_lo = o_lo.as<__nv_bfloat16>(); p.ld_out = ldo;
  DevBuf adbg;
  const int nctas = ((S + 127) / 128) * H * num_seqs;
  if (getenv("CMDI_TEST_DBG")) {
    CK(adbg.alloc((size_t)nctas * 16 * 8));
    CK(cudaMemset(adbg.p, 0, (size_t)nctas * 16 * 8));
    p.dbg_cycles = adbg.as<long long>();
    CK(launch_attention(am, p, stream));
  }
  CK(launch_attention(am, p, stream));
  if (p.dbg_cycles) {
    std::vector<long long> h((size_t)nctas * 16);
    CK(cudaStreamSynchronize(stream));
    CK(cudaMemcpy(h.data(), adbg.p, h.size() * 8, cudaMemcpyDeviceToHost));
    double a[16] = {0};
    {
      // per-CTA-pair sums over its items; slot 7 = item count
      double items = 0;
      for (int c = 0; c < nctas; ++c) items += (double)h[(size_t)c * 16 + 7];
      for (int c = 0; c < nctas; ++c) for (int k = 0; k < 12; ++k) a[k] += (double)h[(size_t)c * 16 + k] / items;
      printf("attention dbg cycles (mean per item): MMA thread wait_q=%.0f wait_k=%.0f S-issue=%.0f wait_P=%.0f wait_V=%.0f PV-issue=%.0f wait_PV_retired=%.0f | "
             "softmax warp: wait_S=%.0f softmax=%.0f last_wait_O=%.0f output=%.0f (items %.0f)\n",
             a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[8], a[9], a[10], a[11], items);
      double pro = 0, tot_max = 0, n = 0;
      for (int c = 0; c < nctas; ++c) {
        if (h[(size_t)c * 16 + 7] == 0) continue;
        n += 1;
        pro += (double)h[(size_t)c * 16 + 12];
        if ((double)h[(size_t)c * 16 + 13] > tot_max) tot_max = (double)h[(size_t)c * 16 + 13];
      }
      printf("attention dbg: CTA pairs=%.0f prologue=%.0f cycles, longest pair (MMA thread) %.0f cycles\n", n, pro / n, tot_max);
      fflush(stdout);
      p.dbg_cycles = nullptr;
    }
  }
  // O = hi + lo (fp32) for the test
  {
    std::vector<uint16_t> hh((size_t)rows * ldo), hl((size_t)rows * ldo);
    std::vector<float> ho((size_t)rows * ldo);
    CK(cudaStreamSynchronize(stream));
    CK(cudaMemcpy(hh.data(), o_hi.p, hh.size() * 2, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(hl.data(), o_lo.p, hl.size() * 2, cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < ho.size(); ++i) {
      uint32_t a = (uint32_t)hh[i] << 16, b = (uint32_t)hl[i] << 16;
      float fa, fb;
      memcpy(&fa, &a, 4);
      memcpy(&fb, &b, 4);
      ho[i] = fa + fb;
    }
    CK(cudaMemcpy(O, ho.data(), ho.size() * 4, cudaMemcpyHostToDevice));
  }
  return 0;
}

extern "C" int cmdi_test_normal_aten(float* out, long long numel, unsigned long long seed, unsigned long long offset,
                                     unsigned int threads, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  if (threads == 0 || (offset & 3) || numel < 0) {
    set_last_error("cmdi_test_normal_aten: threads must be > 0 and offset a multiple of 4");
    return 1;
  }
  CK(launch_fill_normal_aten(out, (size_t)numel, seed, offset, threads, stream));
  return 0;
}

extern "C" int cmdi_test_normal(float* out, int B, long long per_sample, unsigned long long seed, unsigned long long stream_id,
                                unsigned long long sample_offset, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  CK(launch_fill_normal_ref(out, B, (size_t)per_sample, seed, stream_id, sample_offset, stream));
  return 0;
}

extern "C" int cmdi_test_layernorm_bwd(const float* dy, const float* v, const float* gamma, float* dv, int rows, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  DevBuf hi;
  CK(hi.alloc((size_t)rows * 512 * 2));
  CK(launch_layernorm512_bwd(dy, v, gamma, 1e-5f, rows, dv, hi.as<__nv_bfloat16>(), nullptr, stream));
  CK(cudaStreamSynchronize(stream));
  return 0;
}

// qkv: fp32 [num_seqs*S, 3*H*128], dO: fp32 [num_seqs*S, H*128] -> dqkv fp32 (hi + lo of the kernel's planes)
extern "C" int cmdi_test_attention_bwd(const float* qkv, const float* dO, float* dqkv, int num_seqs, int S, int H, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  const int rows = num_seqs * S, ld = 3 * H * 128, ldo = H * 128;
  const int rows_p = round_up(rows, 128) + 256;  // tiles of the last sequence read past its end
  DevBuf q_hi, q_lo, d_hi, d_lo, g_hi, g_lo, stats;
  CK(q_hi.alloc((size_t)rows_p * ld * 2)); CK(q_lo.alloc((size_t)rows_p * ld * 2));
  CK(d_hi.alloc((size_t)rows_p * ldo * 2)); CK(d_lo.alloc((size_t)rows_p * ldo * 2));
  CK(g_hi.alloc((size_t)rows_p * ld * 2)); CK(g_lo.alloc((size_t)rows_p * ld * 2));
  CK(stats.alloc((size_t)rows_p * H * sizeof(float2)));
  CK(cudaMemsetAsync(q_hi.p, 0, (size_t)rows_p * ld * 2, stream)); CK(cudaMemsetAsync(q_lo.p, 0, (size_t)rows_p * ld * 2, stream));
  CK(cudaMemsetAsync(d_hi.p, 0, (size_t)rows_p * ldo * 2, stream)); CK(cudaMemsetAsync(d_lo.p, 0, (size_t)rows_p * ldo * 2, stream));
  CK(launch_split_planes(qkv, rows, ld, ld, q_hi.as<__nv_bfloat16>(), q_lo.as<__nv_bfloat16>(), ld, stream));
  CK(launch_split_planes(dO, rows, ldo, ldo, d_hi.as<__nv_bfloat16>(), d_lo.as<__nv_bfloat16>(), ldo, stream));
  AttnBwdParams p{};
  p.num_seqs = num_seqs; p.seq_len = S; p.num_heads = H; p.qkv_hi = q_hi.as<__nv_bfloat16>(); p.qkv_lo = q_lo.as<__nv_bfloat16>();
  p.do_hi = d_hi.as<__nv_bfloat16>(); p.do_lo = d_lo.as<__nv_bfloat16>(); p.ld_do = ldo;
  p.dqkv_hi = g_hi.as<__nv_bfloat16>(); p.dqkv_lo = g_lo.as<__nv_bfloat16>();
  p.ld_dqkv = ld; p.nsplit = 3; p.stats = stats.as<float2>();
  if (!getenv("CMDI_TEST_ATTN_BWD_SIMT")) {
    CUtensorMap qt_hi, qt_lo, qf_hi, qf_lo, dt_hi, dt_lo, df_hi, df_lo, o_hi, o_lo;
    if (make_tmap_bf16_2d(&qt_hi, q_hi.p, rows_p, ld, ld, 64, 128)) return 1;
    if (make_tmap_bf16_2d(&qt_lo, q_lo.p, rows_p, ld, ld, 64, 128)) return 1;
    if (make_tmap_bf16_2d(&qf_hi, q_hi.p, rows_p, ld, ld, 64, kAttnKeyPad)) return 1;
    if (make_tmap_bf16_2d(&qf_lo, q_lo.p, rows_p, ld, ld, 64, kAttnKeyPad)) return 1;
    if (make_tmap_bf16_2d(&dt_hi, d_hi.p, rows_p, ldo, ldo, 64, 128)) return 1;
    if (make_tmap_bf16_2d(&dt_lo, d_lo.p, rows_p, ldo, ldo, 64, 128)) return 1;
    if (make_tmap_bf16_2d(&df_hi, d_hi.p, rows_p, ldo, ldo, 64, kAttnKeyPad)) return 1;
    if (make_tmap_bf16_2d(&df_lo, d_lo.p, rows_p, ldo, ldo, 64, kAttnKeyPad)) return 1;
    if (make_tmap_bf16_2d(&o_hi, g_hi.p, rows_p, ld, ld, 64, 32)) return 1;
    if (make_tmap_bf16_2d(&o_lo, g_lo.p, rows_p, ld, ld, 64, 32)) return 1;
    CK(configure_attention_bwd_tc_kernel());
    AttnBwdTcMaps bm{&qt_hi, &qt_lo, &qf_hi, &qf_lo, &dt_hi, &dt_lo, &df_hi, &df_lo, &o_hi, &o_lo};
    CK(launch_attention_bwd_tc(bm, p, stream));
  } else {
    CK(configure_attention_bwd_kernel());
    CK(launch_attention_bwd(p, stream));
  }
  CK(cudaStreamSynchronize(stream));
  std::vector<uint16_t> hh((size_t)rows * ld), hl((size_t)rows * ld);
  std::vector<float> ho((size_t)rows * ld);
  CK(cudaMemcpy(hh.data(), g_hi.p, hh.size() * 2, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(hl.data(), g_lo.p, hl.size() * 2, cudaMemcpyDeviceToHost));
  for (size_t i = 0; i < ho.size(); ++i) {
    uint32_t a = (uint32_t)hh[i] << 16, b = (uint32_t)hl[i] << 16;
    float fa, fb;
    memcpy(&fa, &a, 4);
    memcpy(&fb, &b, 4);
    ho[i] = fa + fb;
  }
  CK(cudaMemcpy(dqkv, ho.data(), ho.size() * 4, cudaMemcpyHostToDevice));
  return 0;
}
