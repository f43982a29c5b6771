// Host-visible launch interface of the sm_100a kernels (internal to the shared library).
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace cmdi {

// ----------------------------------------------------------------------------------------------
// linear layer: C[M,N] = epilogue(A[M,K] * W[N,K]^T)      (gemm.cu)
// ----------------------------------------------------------------------------------------------
enum RowMap : int {
  ROWMAP_IDENTITY = 0,
  ROWMAP_FRAMES_TO_SEQ = 1,  // A row b*L + l      -> out row b*(L+1) + l + 1   (frame embed, mdm.py:279)
  ROWMAP_SEQ_TO_FRAMES = 2,  // A row b*(L+1) + s  -> out row b*L + s - 1, s=0 dropped (mdm.py:284 "[1:]")
  ROWMAP_HALO_TO_FRAMES = 3, // A row b*row_period + row_lo + l -> out row b*frames + l for l < frames (UNet output, mdm_unet.py:822)
};
constexpr int kMaxTaps = 10;

// Output tensor maps for the TMA-store epilogue (identity row map only): bf16 planes with box {64, 32}, fp32 with
// box {32, 32}; `rows` of each map must equal the number of valid output rows (TMA clips the M tail).
struct LinearStoreMaps {
  const CUtensorMap* hi = nullptr;
  const CUtensorMap* lo = nullptr;
  const CUtensorMap* f32 = nullptr;
  // optional A-operand maps with a {64, 136} box: let a k-tap convolution load the A rows of all taps once (gemm2.cu)
  const CUtensorMap* a_tap_hi = nullptr;
  const CUtensorMap* a_tap_lo = nullptr;
};

struct LinearParams {
  int M;       // valid A rows
  int N;       // valid output columns
  int K;       // reduction extent (any value; tail k-block is zero-filled by TMA)
  int nsplit;  // 1: A_hi*W_hi            (bf16)
               // 3: + A_hi*W_lo + A_lo*W_hi   (bf16x3, ~fp32 accuracy)
  const float* bias;      // [N] or null
  const float* residual;  // fp32 [rows, ld_res], indexed by OUTPUT row; or null
  int ld_res;
  // residual = LayerNorm(ln_src) re-derived in the epilogue from LayerNorm's fp32 INPUT [rows, ld_ln], the per-row
  // (mean, rstd) it published and its gamma / beta: bit-identical to the fp32 tensor LayerNorm would have written,
  // which it then does not have to write.  ln_src may alias out_f32 (each block is read before it is stored).
  const float* ln_src;
  int ld_ln;
  const float2* ln_stats;
  const float* ln_gamma;
  const float* ln_beta;
  // ---- chained launches only (gemm_chain.cu) ----
  // ... or from the partial statistics per row a producer epilogue published (stats_out below) instead of ln_stats
  const float2* ln_partials;
  // ... with LayerNorm's input read back as the bf16 hi + lo planes [rows, ld_ln] the producer wrote for the next GEMM
  // anyway (v = hi + lo to 2^-17 relative: the same quantisation the GEMMs' A operand already has), so that the
  // producer need not store an fp32 copy as well.  The chained epilogue reads LayerNorm's input only this way (not ln_src).
  const __nv_bfloat16* ln_src_hi;
  const __nv_bfloat16* ln_src_lo;
  // LayerNorm folded into THIS linear layer (the A operand is the un-normalised v, the W operand is W * gamma):
  //   LN(v) W^T = rstd * (v (W.gamma)^T - mean * c) + d,   c[n] = sum_k W[n,k] gamma[k],  d[n] = sum_k W[n,k] beta[k] + b[n]
  // fold_stats: [rows][16] float2 slots, the first 4 hold the partial (mean, M2) of the A row's four 128-column quarters;
  // fold_c: [N]; `bias` carries d.
  const float2* fold_stats;
  const float* fold_c;
  // publish the partial statistics of the OUTPUT rows: stats_out[row * 16 + q] = (mean, sum of squared deviations) over
  // the 128 output columns one epilogue warp owns (N must be 512); consumed by ln_partials / fold_stats
  float2* stats_out;
  const float* pos_enc;  // fp32 [L+1, N] table added per output sequence position (ROWMAP_FRAMES_TO_SEQ); or null
  int act;               // 0 none, 1 exact erf GELU, 2 SiLU, 3 Mish (x tanh(softplus(x)), nn.Mish)
  int f32_pre;           // 1: out_f32 receives the value BEFORE the activation (stash for the GELU backward)
  const float* grad_aux; // fp32 [rows, ld_aux] or null: multiply by gelu'(grad_aux[row, col])  (GELU backward)
  int ld_aux;
  int rowmap;            // RowMap
  int frames;            // L for the two sequence row maps
  int dup_row_offset;    // >0: also store every output row at (row + dup_row_offset)  (CFG: cond + uncond copies)
  float* out_f32;        // fp32 [rows, ld_f32] or null
  int ld_f32;
  __nv_bfloat16* out_hi;  // bf16 planes [rows, ld_bf] or null
  __nv_bfloat16* out_lo;  // written only when nsplit_out == 3
  int ld_bf;
  int nsplit_out;  // 1 or 3: whether the consumer of out_hi/out_lo wants the lo plane
  // ---- 1-D convolutions as GEMMs over a channel-last [rows, C] activation (UNet denoiser, gemm2.cu) ----
  // The reduction runs over num_taps blocks of k_per_tap columns; block j reads A at (row + tap_row[j], tap_a_col[j] + k)
  // and W at column tap_w_col[j] + k.  A rows outside the tensor are zero-filled by TMA.  num_taps = 0: a plain linear layer.
  int num_taps, k_per_tap;
  int tap_row[kMaxTaps], tap_a_col[kMaxTaps], tap_w_col[kMaxTaps];
  // rows are valid outputs when row_lo <= row % row_period < row_hi (the others are the zero halo between sequences and
  // are WRITTEN AS ZEROS); row_period = 0: every row < M is valid
  int row_period, row_lo, row_hi;
  // output columns n >= n_split land at column n + n_gap (transposed-convolution even / odd phases into interleaved rows)
  int n_split, n_gap;
  int debug;       // bring-up only (CMDI_DEBUG): 1 = skip global stores, 2 = skip MMA issue, 4 = skip TMA loads
  long long* dbg_cycles;  // bring-up only: per-CTA cycle counters [gridDim.x][16] (see gemm2.cu) or null
  int tma_store;   // set by the launcher when LinearStoreMaps are given: outputs leave through cp.async.bulk.tensor stores
};

// CTA-pair (cta_group::2) version: 256-row tiles shared by two SMs of a cluster. W box is {64, block_n / 2}.   (gemm2.cu)
cudaError_t configure_linear2_kernels();
cudaError_t launch_linear_pair(const CUtensorMap& a_hi, const CUtensorMap& a_lo, const CUtensorMap& w_hi,
                               const CUtensorMap& w_lo, const LinearParams& p, int block_n, int num_sms,
                               cudaStream_t stream, const LinearStoreMaps* st = nullptr);

// A chain of linear layers in ONE persistent launch (gemm_chain.cu): the tiles of all phases form one list walked by
// the 74 CTA pairs; a tile whose A rows are produced by an earlier phase of the same launch waits on a per-row-pair
// counter the producing epilogues bump.  Removes the kernel boundaries and the per-kernel tile quantisation.
constexpr int kMaxChainPhases = 4;
struct ChainPhaseInfo {
  LinearParams p;
  int block_n;                 // 256 (the epilogue distributes the eight 32-column slices of a tile over its warps)
  int num_m_pairs, num_n_blocks, num_k_blocks;
  int tile_begin, tile_end;    // global tile index range of this phase (tile = m_pair * num_n_blocks + n_blk)
  int* wait_ctr;               // [num_m_pairs] or null: A rows of pair m are complete when wait_ctr[m] >= wait_target
  int wait_target;
  int* done_ctr;               // [num_m_pairs] or null: each CTA adds 1 once its half of a tile is in memory
  // 1: planes-only phase (FFN1, QKV) whose epilogue works on 64-column pairs, o_hi / o_lo are {64, 32} boxes with the
  // 128 B swizzle;  0: 32-column slices (residual phases, output head), o_hi / o_lo are {32, 32} boxes with the 64 B swizzle
  int pair_epilogue;
};
struct alignas(128) ChainPhaseDesc {
  CUtensorMap a_hi, a_lo, w_hi, w_lo, o_hi, o_lo;
  ChainPhaseInfo info;
};
cudaError_t configure_linear_chain_kernel();
// phases: device array; returns cudaErrorInvalidConfiguration if `num_sms / 2` clusters cannot be co-resident
cudaError_t launch_linear_chain(const ChainPhaseDesc* phases_dev, int num_phases, int total_tiles, int num_sms,
                                cudaStream_t stream, long long* dbg = nullptr);
int linear_chain_max_clusters(int num_sms);

// ----------------------------------------------------------------------------------------------
// self-attention core: O = softmax(Q K^T / sqrt(dh)) V per (sequence, head)      (attention.cu)
// ----------------------------------------------------------------------------------------------
struct AttnParams {
  int num_seqs;   // sequences (B, or 2B under CFG)
  int seq_len;    // S = L+1 (<= 208)
  int num_heads;  // H, head dim fixed at 128
  int nsplit;     // 1 or 3 (as above, applied to both Q K^T and P V)
  int nsplit_out;
  __nv_bfloat16* out_hi;  // [num_seqs*seq_len (+pad), H*128]
  __nv_bfloat16* out_lo;
  int ld_out;
  long long* dbg_cycles;  // bring-up only: [num_clusters][16] cycle counters or null
};
// qkv maps: bf16 [rows, 3*H*128] row-major planes (hi, lo); box {64, 128} for Q, {64, 208} for V (and K in the backward
// kernel), {64, 104} for K (each CTA of a pair holds half of the keys).
// o maps: the output planes [rows, H*128] as TMA-store targets, box {64, 32}.
struct AttnMaps {
  const CUtensorMap *q_hi, *q_lo, *kh_hi, *kh_lo, *kv_hi, *kv_lo, *o_hi, *o_lo;
};
cudaError_t configure_attention_kernel();
cudaError_t launch_attention(const AttnMaps& maps, const AttnParams& p, cudaStream_t stream);
constexpr int kAttnKeyPad = 208;

// ----------------------------------------------------------------------------------------------
// elementwise / row kernels      (elementwise.cu)
// ----------------------------------------------------------------------------------------------
// y = LayerNorm(v) * gamma + beta over rows of 512; writes fp32 and bf16 planes.
// (stats_out: optional [rows] (mean, rstd) for epilogues that re-derive the output, see LinearParams::ln_src)
cudaError_t launch_layernorm512(const float* v, const float* gamma, const float* beta, float eps, int rows, float* out_f32,
                                __nv_bfloat16* out_hi, __nv_bfloat16* out_lo, cudaStream_t stream, float2* stats_out = nullptr);

// fp32 CUDA-core linear for the tiny per-loop tables: out[r, n] = act(in[r,:] . W[n,:] + b[n])
// act: 0 none, 2 SiLU
cudaError_t launch_small_linear(const float* in, const float* W, const float* bias, float* out, int rows, int N, int K,
                                int act, cudaStream_t stream);

// Conditioning token rows of the sequence buffer (mdm.py:245-251, :279-280):
//   x[seq*S + 0, :] = temb[step_t, :] + (cond_proj[seq % B] if seq < n_cond_seqs else uncond_bias) + pe[0, :]
struct TokenParams {
  const float* temb_table;  // [5000, 512] time_embed(pe[t]) for every ORIGINAL timestep t
  const int* step_ptr;      // device: current sampler step index t
  const int* timestep_map;  // device [T]: sampler step -> original timestep (respace.py:128-133); null = identity
  const float* cond_proj;   // [B, 512] embed_text(cond) (bias included) or null (no_cond)
  const float* uncond_proj; // [512] embed_text(0) = bias, or null
  const float* pe0;         // [512]
  int num_seqs;             // total sequences
  int n_cond_seqs;          // first n use cond_proj[seq], the rest use uncond_proj
  int seq_len;
  float* x_f32;             // [num_seqs*seq_len, 512]
  __nv_bfloat16* x_hi;
  __nv_bfloat16* x_lo;
};
cudaError_t launch_token_rows(const TokenParams& p, cudaStream_t stream);

// Diffusion step (gaussian_diffusion.py:352-534, :656-713, :1358-1416) on frame-major state [B*L, D_pad].
struct StepTables {            // device pointers, each [T] fp32, indexed by sampler step t
  const float* post_coef1;     // posterior_mean_coef1
  const float* post_coef2;     // posterior_mean_coef2
  const float* post_logvar;    // posterior_log_variance_clipped
  const float* sqrt_recip_acp;    // sqrt(1/alphas_cumprod)
  const float* sqrt_recipm1_acp;  // sqrt(1/alphas_cumprod - 1)
  const float* acp;               // alphas_cumprod
  const float* acp_prev;          // alphas_cumprod_prev
};
struct RngState {
  unsigned long long seed;           // Philox key
  unsigned long long sample_offset;  // mode 0: global index of local sample 0 (results independent of sharding)
  unsigned long long aten_offset;    // mode 1: philox offset (in 32-bit outputs, multiple of 4) of the first per-step draw
  unsigned long long aten_increment; // mode 1: offset consumed by one randn_like of B*D*L elements
  unsigned int aten_threads;         // mode 1: grid.x * 256 of ATen's distribution kernel for that numel
  int mode;
};
struct StepParams {
  StepTables tab;
  int* step_ptr;            // device [3]: current step t (decremented by the kernel's last block when advance != 0),
                            // block-arrival counter, first step index of the call
  int advance;
  int B, L, D, D_pad;
  int sampler;              // 0 = ancestral DDPM (p_sample), 1 = DDIM (ddim_sample_with_grad, cond_fn=None),
                            // 2 = no update: only pred_xstart (= guided/imputed model output) is written
  float eta;                // DDIM
  const float* model_out;   // [B*L (x2 when cfg), D_pad] raw denoiser output(s); uncond half at +B*L rows
  int cfg;                  // 1: out = u + s[b]*(c - u)
  const float* text_scale;  // [B]
  const float* x_t;         // [B*L, D_pad]
  // imputation (gaussian_diffusion.py:427-435): applied when impute != 0 and t >= stop_imputation_at
  int impute;
  int stop_imputation_at;
  const float* x_obs;          // [B*L, D_pad] frame-major
  const uint8_t* obs_mask;     // [B*L, D_pad] frame-major, already AND-ed with y.mask
  // reconstruction guidance (gaussian_diffusion.py:418-425): x0_tilde = x0_hat - coef[t] * (grad * ~M)
  int guided;
  const float* guide_grad;     // [B*L (x2 when cfg), D_pad] dL/dz of the cond (and uncond) pass
  const float* guide_coef;     // [T] w_r[t] * sqrt(alpha_bar_t) / 2
  // noise
  const float* noise_ref;      // tape base, reference layout [steps][B, D, 1, L]; slice (tape_t0 - t) is this step's
                               // randn_like draw; null -> in-kernel Philox
  int tape_t0;                 // >= 0: the call's first step index; -1: read it from step_ptr[2]
  // generator state, device-resident so a captured step graph does not depend on it (RngState below).
  // rng_mode 0: engine generator keyed by (seed, t + 1, global sample index, element quad);
  // rng_mode 1: the stream of torch.randn_like on this device (ATen's Philox offsets / thread mapping), draw
  //             number (tape_t0 - t) after `aten_offset`
  const RngState* rng;
  // outputs
  float* x_next;               // [B*L, D_pad]
  __nv_bfloat16* x_next_hi;
  __nv_bfloat16* x_next_lo;
  float* pred_xstart;          // [B*L, D_pad] or null
};
cudaError_t launch_diffusion_step(const StepParams& p, cudaStream_t stream);

// HumanML3D vectors -> joint positions (recover_from_ric), strides in elements; mean/stdv null = already de-normalised
cudaError_t launch_recover_from_ric(const float* data, long long sb, long long sf, long long sc, const float* mean,
                                    const float* stdv, int B, int L, int joints, int abs_3d, float* out, long long ob,
                                    long long of, long long oj, long long oc, cudaStream_t stream);
cudaError_t launch_set_rng(RngState* dst, const RngState& value, cudaStream_t stream);
// out[i] = the i-th element torch.randn(numel, device=cuda) would produce with generator (seed, offset), where
// `threads` is ATen's launch width for that numel (256 * min(SMs * maxThreadsPerSM / 256, ceil(numel / 256)))
cudaError_t launch_fill_normal_aten(float* out, size_t numel, unsigned long long seed, unsigned long long offset,
                                    unsigned int threads, cudaStream_t stream);

// layout converters between the reference layout [B, D, 1, L] and frame-major [B*L, D_pad]
cudaError_t launch_ref_to_frames(const float* ref, int B, int D, int L, int D_pad, float* out_f32, __nv_bfloat16* out_hi,
                                 __nv_bfloat16* out_lo, cudaStream_t stream);
cudaError_t launch_frames_to_ref(const float* frames, int B, int D, int L, int D_pad, float* ref, cudaStream_t stream);
// mask: ref-layout bool bytes [B, D, 1, L] AND y_mask [B, L] (or null) -> frame-major bytes
cudaError_t launch_mask_to_frames(const uint8_t* ref_mask, const uint8_t* y_mask, int B, int D, int L, int D_pad,
                                  uint8_t* out, cudaStream_t stream);
// q_sample (gaussian_diffusion.py:311-328) in reference layout: out = a*x0 + b*noise
cudaError_t launch_axpby(const float* x, const float* y, float a, float b, float* out, size_t n, cudaStream_t stream);
// standard normal fill (Philox4x32-10 + Box-Muller), value at flat index i of sample s depends on (seed, stream_id, s, i) only
cudaError_t launch_fill_normal_ref(float* out, int B, size_t per_sample, unsigned long long seed,
                                   unsigned long long stream_id, unsigned long long sample_offset, cudaStream_t stream);
cudaError_t launch_set_int(int* p, int v, cudaStream_t stream);

// LayerNorm folded into its consumer: Wf = W * gamma (fp32 [N,K]), c[n] = sum_k Wf[n,k], d[n] = sum_k W[n,k] beta[k] + bias[n]
cudaError_t launch_add_vectors(const float* a, const float* b, float* out, int n, cudaStream_t stream);
cudaError_t launch_fold_ln(const float* W, int N, int K, const float* gamma, const float* beta, const float* bias, float* Wf,
                           float* c, float* d, cudaStream_t stream);
// fp32 [rows, cols] -> bf16 planes [rows, ld] (zero padded columns)
cudaError_t launch_split_planes(const float* in, int rows, int cols, int ld_in, __nv_bfloat16* hi, __nv_bfloat16* lo,
                                int ld_out, cudaStream_t stream);

// ----------------------------------------------------------------------------------------------
// MDM_UNET denoiser pieces      (unet_kernels.cu; the convolutions run on the pair GEMM, gemm2.cu)
// ----------------------------------------------------------------------------------------------
struct UnetInputParams {
  int B, L, D, D_pad;          // frame-major sources [B*L, D_pad]
  const float* x_t;
  const float* obs;            // observed keyframes (null: not keyframe-conditioned)
  const uint8_t* obs_mask;
  int copies;                  // 2 under CFG: sequences b and b + B receive the same input
  int row_period, row_lo;      // halo layout of the destination
  int ld;                      // destination row pitch (elements, even)
  __nv_bfloat16* out_hi;
  __nv_bfloat16* out_lo;
};
cudaError_t launch_unet_input(const UnetInputParams& p, cudaStream_t stream);
// emb planes [num_seqs, 512]; TokenParams::seq_len carries B (conditioning row = seq % B), x_f32 is unused
cudaError_t launch_unet_emb(const TokenParams& p, cudaStream_t stream);
struct GroupNormParams {
  int C, groups, L;            // channels, groups, positions per sequence
  int row_period, row_lo;      // halo layout (rows of sequence b: b * row_period + row_lo + l)
  float eps;
  const float* y;              // fp32 [rows, ld_y] convolution output (bias included)
  int ld_y;
  const float* gamma;
  const float* beta;
  const float* ada;            // [num_seqs, ld_ada] fp32: [scale (C) | shift (C)] per sequence, or null
  int ld_ada;
  const float* res_f32;        // residual added AFTER the activation: fp32 [rows, ld_res] ...
  const __nv_bfloat16* res_hi; // ... or bf16 hi/lo planes [rows, ld_res] (x = hi + lo), or none
  const __nv_bfloat16* res_lo;
  int ld_res;
  __nv_bfloat16* out_hi;       // planes [rows, ld_out] (pointer already offset to the first output column)
  __nv_bfloat16* out_lo;
  int ld_out;
};
cudaError_t configure_groupnorm_kernel();
cudaError_t launch_groupnorm_mish(const GroupNormParams& p, int num_seqs, cudaStream_t stream);
// weight re-layouts: Conv1d [Co,Ci,k] -> tap-major planes [Co, k*Cp]; ConvTranspose1d(4,2,1) [Ci,Co,4] -> planes [2Co, 3Ci]
cudaError_t launch_conv_weight_planes(const float* w, int Co, int Ci, int k, int Cp, __nv_bfloat16* hi, __nv_bfloat16* lo, int ld,
                                      cudaStream_t stream);
cudaError_t launch_convt_weight_planes(const float* w, int Ci, int Co, __nv_bfloat16* hi, __nv_bfloat16* lo, int ld, cudaStream_t stream);

// ----------------------------------------------------------------------------------------------
// backward pieces for reconstruction guidance      (backward.cu)
// ----------------------------------------------------------------------------------------------
struct GuidanceSeedParams {
  int B, L, D, D_pad, cfg;
  const float* model_out;    // [B*L (x2 when cfg), D_pad] raw denoiser outputs (uncond half at +B*L rows)
  const float* text_scale;   // [B]
  const float* x_obs;        // [B*L, D_pad]
  const uint8_t* obs_mask;   // [B*L, D_pad]
  __nv_bfloat16* seed_hi;    // [B*L (x2), D_pad] dL/d(model output rows)
  __nv_bfloat16* seed_lo;
};
cudaError_t launch_guidance_seed(const GuidanceSeedParams& p, cudaStream_t stream);
cudaError_t launch_layernorm512_bwd(const float* dy, const float* v, const float* gamma, float eps, int rows, float* dv,
                                    __nv_bfloat16* dv_hi, __nv_bfloat16* dv_lo, cudaStream_t stream);
struct AttnBwdParams {
  int num_seqs, seq_len, num_heads;
  const __nv_bfloat16* qkv_hi;   // stashed forward Q|K|V planes [rows, 3*H*128]
  const __nv_bfloat16* qkv_lo;
  const __nv_bfloat16* do_hi;    // dO planes [rows, H*128]
  const __nv_bfloat16* do_lo;
  int ld_do;
  __nv_bfloat16* dqkv_hi;        // out: dQ|dK|dV planes [rows, 3*H*128]
  __nv_bfloat16* dqkv_lo;
  // tensor-core kernel only
  int ld_dqkv;                   // 3*H*128
  int nsplit;                    // 1 or 3
  float2* stats;                 // [rows, H]: (max*c + log2(sum), delta) per query row, written by pass 0, read by pass 1
};
cudaError_t configure_attention_bwd_kernel();
cudaError_t launch_attention_bwd(const AttnBwdParams& p, cudaStream_t stream);  // fp32 CUDA cores: the independent
                                                                               // implementation the unit tests compare against (attention_bwd_simt_test.cu)
// tcgen05 version (attention_bwd_tc.cu).  Maps over the bf16 planes, box {64, rows}: *_t = 128-row tiles, *_f = 208-row
// operands; out_* = the dqkv planes as TMA-store targets, box {64, 32}.
struct AttnBwdTcMaps {
  const CUtensorMap *qkv_t_hi, *qkv_t_lo, *qkv_f_hi, *qkv_f_lo, *do_t_hi, *do_t_lo, *do_f_hi, *do_f_lo, *out_hi, *out_lo;
};
cudaError_t configure_attention_bwd_tc_kernel();
cudaError_t launch_attention_bwd_tc(const AttnBwdTcMaps& m, const AttnBwdParams& p, cudaStream_t stream);
cudaError_t launch_transpose_split(const float* w, int R, int C, __nv_bfloat16* hi, __nv_bfloat16* lo, int ld_out,
                                   cudaStream_t stream);

// ----------------------------------------------------------------------------------------------
// TMA descriptor creation (tma_host.cu)
// ----------------------------------------------------------------------------------------------
// bf16 row-major [rows, cols] with row pitch ld elements; box {box_cols (=64), box_rows}; 128 B swizzle.
int make_tmap_bf16_2d(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_cols,
                      uint32_t box_rows);
// generic: elem_bytes 2 (bf16) or 4 (fp32); box_cols * elem_bytes must be 128
int make_tmap_2d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t rows, uint64_t cols, uint64_t ld,
                 uint32_t box_cols, uint32_t box_rows);

void set_last_error(const char* fmt, ...);

// Launch helper (cudaLaunchKernelEx so cluster-dimensioned kernels and plain ones share one path).  Programmatic
// dependent launch was built and measured in round 1 (graph replay 3.5 % SLOWER with the programmatic edges) and removed.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                 Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cfg.numAttrs = 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
const char* get_last_error();

}  // namespace cmdi
