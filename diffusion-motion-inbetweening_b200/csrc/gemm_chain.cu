// Several linear layers of an encoder layer in ONE persistent launch of CTA pairs (tcgen05.mma.cta_group::2).
//
// Why.  Launched one by one (gemm2.cu), every linear layer pays (a) its own tile quantisation -- QKV is 300 pair
// tiles on 74 clusters = 4.05 rounds, i.e. 5; the N = 512 layers 2.7 rounds, i.e. 3 -- and (b) a kernel boundary
// whose cost is the tail imbalance of the last round + the prologue + the first TMA round trip, because every one of
// these kernels owns all shared memory and all 512 TMEM columns of its SM and a successor cannot become resident
// early.  Here the tiles of out-proj, FFN1, FFN2 and the NEXT layer's QKV projection (or the output head) form one
// list of 700 tiles (256 x 256 each) walked by the 74 clusters in order; the smem rings, the TMEM double buffer and the
// warp roles simply keep running across phase boundaries.
//
// Dependencies.  Phase p + 1 reads, as its A operand, rows that phase p writes.  Tiles are ordered row-pair-major
// inside a phase; when a CTA's half of a tile is in memory it bumps a per-(phase, row-pair) counter, and the TMA
// producer of a consuming tile spins on that counter (acquire) before it issues the first load of the tile.
// All clusters are co-resident (grid = 2 x 74 <= SM count, checked at start-up with the occupancy API) and walk
// their tiles in increasing global index, and a tile only ever waits for tiles of LOWER index: no deadlock.
//
//   epilogue warp:     TMA stores -> cp.async.bulk.wait_group 0 -> mbarrier.arrive(publish[tile & 3])     (release.cta;
//                      the other lanes' plain stores are ordered before lane 0's arrive by __syncwarp)
//   publisher warp:    mbarrier wait(publish[..]) (acquire.cta) -> fence.proxy.async -> __threadfence -> atomicAdd(counter)
//   consumer TMA lane: ld.acquire.gpu(counter) >= target -> fence.proxy.async -> cp.async.bulk.tensor loads
//   consumer epilogue: ordered after the TMA lane's acquire through full[] -> MMA -> tmem_full[]; its reads of
//                      activations written in this launch use ld.global.cg
//
// Epilogue (see also the measurements at kNumEpiWarps).  Eight warps, two per TMEM lane group.  A tile of a phase with
// a residual (out-proj, FFN2) is cut into eight 32-column slices, four per warp: bias, the residual LayerNorm(v)
// re-derived from v's bf16 planes (coalesced loads transposed through the warp's 4 KB staging tile, the next slice's block
// prefetched into registers), partial row statistics, one store of both bf16 planes through 64-byte-swizzled boxes.  A
// tile of a planes-only phase (FFN1, QKV) is cut into four 64-column pairs, two per warp: folded-LayerNorm scale / shift,
// bias, GELU (branch-free rational erf), hi plane then lo plane through 128-byte-swizzled boxes.  Per-column constants
// are loaded once per tile into registers and handed out by shuffle; the release fence / counter bump lives in a warp of
// its own.  Shared memory: A ring 2 x 32 KB, W ring 3 x 32 KB (separate barriers), 8 x 4 KB staging tiles = 192 KB.
#include "common.cuh"
#include "gemm_epilogue.cuh"
#include "kernels.h"

namespace cmdi {

namespace {

constexpr int kBlockM = 128;  // per CTA; 256 per pair
constexpr int kBlockN = 256;
constexpr int kBlockK = 64;
constexpr int kUmmaK = 16;
// Epilogue warps, ring depths and the L1 left beside the shared memory, measured at B = 64 (same box, A/B/A/B):
//   12 epilogue warps (128 registers), A 3 + W 2 stages        482 steps/s
//   12 warps with 2 KB staging tiles,  A 3 + W 3               504
//    8 warps (168 registers),          A 3 + W 3  (224 KB)     520   <- round-2 mid-point
//    8 warps, 64-column pairs in the planes-only phases, A 3 + W 3 (224 KB)   514-523 (another box)
//    same, A 2 + W 3 (192 KB) or A 2 + W 2 (160 KB)            528-535
//    same, A 2 + W 3 + a second staging tile per warp (224 KB) 514
// The epilogue is issue- and latency-bound, not occupancy-bound (fewer warps with more registers win), and what the
// third A stage buys the producer is less than what its 32 KB cost the epilogue as L1: the per-tile constants, the row
// statistics and the few spilled registers around the barrier waits live there, and at 224 KB of shared memory only
// ~25 KB of L1 remain.  A second staging tile per warp (stores never waiting for the previous store's read) bought
// nothing at equal shared memory.
#ifndef CMDI_CHAIN_STAGES_W
#define CMDI_CHAIN_STAGES_W 3
#endif
constexpr int kNumEpiWarps = 8;  // the slice / pair assignment below is written for two warps per lane group
constexpr int kWarpsPerLaneGroup = kNumEpiWarps / 4;
constexpr int kFirstEpiWarp = 3;
constexpr int kNumThreads = (kFirstEpiWarp + kNumEpiWarps) * 32;
#ifndef CMDI_CHAIN_STAGES_A
#define CMDI_CHAIN_STAGES_A 2
#endif
constexpr int kStagesA = CMDI_CHAIN_STAGES_A, kStagesW = CMDI_CHAIN_STAGES_W;
constexpr int kPlaneBytes = kBlockM * kBlockK * 2;   // one bf16 plane of a 128-row x 64-column operand block = 16 KB
constexpr int kOperandBytes = 2 * kPlaneBytes;       // hi + lo
constexpr int kSlices = kBlockN / 32;                // 32-column slices per tile
constexpr int kAccStride = 256;                      // TMEM columns per accumulator buffer
constexpr uint32_t kTmemCols = 512;
constexpr int kPublishBars = 4;

struct __align__(8) ChainBarriers {
  uint64_t full_a[kStagesA], empty_a[kStagesA];
  uint64_t full_w[kStagesW], empty_w[kStagesW];
  uint64_t tmem_full[2], tmem_empty[2];
  uint64_t publish[kPublishBars];
  uint32_t tmem_base;
  uint32_t pad;
};

constexpr int kSmemBytes = 1024 + (kStagesA + kStagesW) * kOperandBytes + kNumEpiWarps * kEpiStageBytes + (int)sizeof(ChainBarriers) +
                           kMaxChainPhases * (int)sizeof(ChainPhaseInfo);
static_assert(kSmemBytes <= 232448, "shared memory budget");

__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }

// Bounded like mbar_wait: a protocol bug must trap, not hang the GPU.
__device__ __forceinline__ void wait_counter(const int* ctr, int target) {
  if (ld_acquire_gpu(ctr) >= target) return;
  const long long t0 = clock64();
  while (ld_acquire_gpu(ctr) < target) {
    __nanosleep(32);
    if (clock64() - t0 > 4000000000LL) {
      printf("cmdi: chain dependency timeout block=%d counter=%p value=%d target=%d\n", blockIdx.x, ctr, ld_acquire_gpu(ctr), target);
      __trap();
    }
  }
}

// Partial LayerNorm statistics: every epilogue warp Chan-combines the (mean, M2) of its slices of a tile in registers and
// publishes ONE partial per row, so a 512-wide row has kRowPartials = (512 / 256) * kWarpsPerLaneGroup partials of
// 512 / kRowPartials columns each.
static_assert(kSlices % kWarpsPerLaneGroup == 0, "equal column counts per partial");
constexpr int kRowPartials = 2 * kWarpsPerLaneGroup;
constexpr int kPartialStride = 16;  // float2 per row in the statistics arrays (engine.cu allocates 16)

// (mean, rstd) of a 512-wide row from its partial statistics (Chan et al. parallel combination, equal counts; fp32)
__device__ __forceinline__ float2 combine_row_stats(const float2* partials_row) {
  float m[kRowPartials], q = 0.f, s = 0.f;
#pragma unroll
  for (int i = 0; i < kRowPartials / 2; ++i) {
    const uint4 a = ld_global_cg_v4(partials_row + 2 * i);
    m[2 * i] = __uint_as_float(a.x);
    m[2 * i + 1] = __uint_as_float(a.z);
    q += __uint_as_float(a.y) + __uint_as_float(a.w);
  }
#pragma unroll
  for (int i = 0; i < kRowPartials; ++i) s += m[i];
  const float mean = s * (1.0f / kRowPartials);
  float dev = 0.f;
#pragma unroll
  for (int i = 0; i < kRowPartials; ++i) {
    const float d = m[i] - mean;
    dev = fmaf(d, d, dev);
  }
  const float var = (q + (512.0f / kRowPartials) * dev) * (1.0f / 512.0f);
  return make_float2(mean, rsqrtf(var + 1e-5f));  // nn.LayerNorm default eps, as nn.TransformerEncoderLayer uses it
}

// hi and lo planes of a 32-row x 32-column block (thread `lane` holds row `lane` as 16 bf16x2 words per plane) through
// the warp's staging tile as two {64 B x 32 rows} boxes with the 64-byte swizzle (16-byte chunk c of row r sits at
// chunk c ^ ((r >> 1) & 3): conflict-free for a row-per-lane writer), one bulk tensor store each.
__device__ __forceinline__ void store_planes_tma(uint32_t stage, int lane, const uint32_t (&hw)[16], const uint32_t (&lw)[16],
                                                 const CUtensorMap* map_hi, const CUtensorMap* map_lo, bool with_lo, int col, int row) {
  if (lane == 0) tma_store_wait_read();
  __syncwarp();
  const uint32_t sw = (uint32_t)(lane >> 1) & 3u;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    st_shared_v4(stage + lane * 64 + ((c ^ sw) << 4), hw[c * 4], hw[c * 4 + 1], hw[c * 4 + 2], hw[c * 4 + 3]);
    if (with_lo) st_shared_v4(stage + 2048 + lane * 64 + ((c ^ sw) << 4), lw[c * 4], lw[c * 4 + 1], lw[c * 4 + 2], lw[c * 4 + 3]);
  }
  fence_proxy_async_smem();
  __syncwarp();
  if (lane == 0) {
    tma_store_2d(map_hi, stage, col, row);
    if (with_lo) tma_store_2d(map_lo, stage + 2048, col, row);
    tma_store_commit();
  }
}

// erf(x) as a rational function of the clamped argument (numerator degree 13, denominator degree 8 in x; max abs error
// 3.7e-7 over the real line, checked against math.erf in tests/test_host_logic.py): branch-free, 14 FMAs + one division.
// The FFN1 epilogue is issue-bound and CUDA's erff (two polynomial branches + exp) was its largest single item (8 % of
// the chain kernel's samples); |GELU error| <= 6.4e-7 against 2^-17 ~ 7.6e-6 relative of the bf16x3 products around it.
__device__ __forceinline__ float erf_rational(float x) {
  x = fminf(fmaxf(x, -4.0f), 4.0f);
  const float x2 = x * x;
  float p = -2.72614225801306e-10f;
  p = fmaf(p, x2, 2.77068142495902e-08f);
  p = fmaf(p, x2, -2.10102402082508e-06f);
  p = fmaf(p, x2, -5.69250639462346e-05f);
  p = fmaf(p, x2, -7.34990630326855e-04f);
  p = fmaf(p, x2, -2.95459980854025e-03f);
  p = fmaf(p, x2, -1.60960333262415e-02f);
  float q = -1.45660718464996e-05f;
  q = fmaf(q, x2, -2.13374055278905e-04f);
  q = fmaf(q, x2, -1.68282697438203e-03f);
  q = fmaf(q, x2, -7.37332916720468e-03f);
  q = fmaf(q, x2, -1.42647390514189e-02f);
  return __fdividef(x * p, q);
}
__device__ __forceinline__ float gelu_fast(float x) { return 0.5f * x * (1.0f + erf_rational(x * 0.70710678118654752440f)); }

constexpr int kSlicesPerWarp = (kSlices + kWarpsPerLaneGroup - 1) / kWarpsPerLaneGroup;  // of one tile

struct RowStats {   // per-tile cache of what this thread needs for its slices of the tile
  float2 fold, ln;                 // (mean, rstd) of its row: folded LayerNorm of the A operand / LayerNorm of the residual
  // Per-COLUMN constants (bias, folded-LN c, LayerNorm gamma / beta of the residual): lane l holds column l of the warp's
  // k-th slice of the tile, loaded with one coalesced request per vector before the tile's accumulator wait
  // (load_tile_constants) and handed out by shuffle.  History: fetched at the point of use they were ~15 % of this kernel's
  // stall samples (an L2 round trip costs 2-3 us under this load); loaded per tile but one predicated load at a time, 11 %.
  // (Per slice, one slice ahead, in 4 registers instead of 16: slower, 154.6 -> 161.6 us per launch.)
  float bias[kSlicesPerWarp], c[kSlicesPerWarp], g[kSlicesPerWarp], b[kSlicesPerWarp];
  float run_mean, run_m2;          // running statistics of this thread's output row over the warp's slices of the tile
};
__device__ __forceinline__ float pick(const float (&a)[kSlicesPerWarp], int k) {
  float v = a[0];
#pragma unroll
  for (int i = 1; i < kSlicesPerWarp; ++i) v = (k == i) ? a[i] : v;
  return v;
}

// Start of a tile for one epilogue warp: per-column constants of its (up to) four 32-column slices and the statistics of
// its row.  `pairs` (ChainPhaseInfo::pair_epilogue): the warp owns two 64-column pairs (slices 2q, 2q+1 for
// q = warp_in_group, warp_in_group + 2) instead of the alternating slices warp_in_group + 2k.
__device__ __forceinline__ int warp_slice(int k, int warp_in_group, bool pairs) {
  return pairs ? 2 * (warp_in_group + kWarpsPerLaneGroup * (k >> 1)) + (k & 1) : warp_in_group + k * kWarpsPerLaneGroup;
}
// The constants do not depend on anything computed in this launch: they are requested BEFORE the warp waits for the tile's
// accumulator, all loads of a vector in flight together (indices clamped instead of predicated; measured before: one
// predicated load at a time, each followed by the spill of its result, was 11 % of this kernel's stall samples).
__device__ __forceinline__ void load_tile_constants(const LinearParams& p, RowStats& rs, int n_blk, int warp_in_group, bool pairs, int lane) {
  int idx[kSlicesPerWarp];
  bool ok[kSlicesPerWarp];
#pragma unroll
  for (int k = 0; k < kSlicesPerWarp; ++k) {
    const int sl = warp_slice(k, warp_in_group, pairs);
    const int n = n_blk * kBlockN + sl * 32 + lane;
    ok[k] = sl < kSlices && n < p.N;
    idx[k] = ok[k] ? n : 0;
  }
  const bool ln = p.ln_src_hi != nullptr;
  float t[4][kSlicesPerWarp];
#pragma unroll
  for (int k = 0; k < kSlicesPerWarp; ++k) {
    t[0][k] = p.bias ? __ldg(p.bias + idx[k]) : 0.f;
    t[1][k] = p.fold_stats ? __ldg(p.fold_c + idx[k]) : 0.f;
    t[2][k] = ln ? __ldg(p.ln_gamma + idx[k]) : 0.f;
    t[3][k] = ln ? __ldg(p.ln_beta + idx[k]) : 0.f;
  }
#pragma unroll
  for (int k = 0; k < kSlicesPerWarp; ++k) {
    rs.bias[k] = ok[k] ? t[0][k] : 0.f;
    rs.c[k] = ok[k] ? t[1][k] : 0.f;
    rs.g[k] = ok[k] ? t[2][k] : 0.f;
    rs.b[k] = ok[k] ? t[3][k] : 0.f;
  }
}
// ... and, once the accumulator (hence the producer phase's statistics) is there, the statistics of the thread's row
__device__ __forceinline__ void load_row_statistics(const LinearParams& p, RowStats& rs, int row) {
  if (p.fold_stats) rs.fold = combine_row_stats(p.fold_stats + (size_t)row * kPartialStride);
  if (p.ln_partials) rs.ln = combine_row_stats(p.ln_partials + (size_t)row * kPartialStride);
  rs.run_mean = 0.f; rs.run_m2 = 0.f;
}

// A 64-column pair of slices of a phase that writes planes only (FFN1, QKV): one accumulator read, one pass of math over
// 64 values and two {128 B x 32 rows} plane stores -- half the per-slice synchronisation (TMEM load wait, staging-tile
// turn-around, proxy fence) per column of the 32-column path, which needs its registers for the residual instead.
__device__ __forceinline__ void epilogue_pair(const LinearParams& p, const ChainPhaseDesc& pd, uint32_t tmem_acc, int m_blk, int n_blk,
                                              int pair, int k2, int lane_group, int lane, uint32_t stage, const RowStats& rs) {
  const int n0 = n_blk * kBlockN + pair * 64;
  if (n0 >= p.N) return;  // warp-uniform
  const int warp_row0 = m_blk * kBlockM + lane_group * 32;
  uint32_t v[64];
  tmem_ld32(tmem_acc + pair * 64, *reinterpret_cast<uint32_t(*)[32]>(&v[0]));
  tmem_ld32(tmem_acc + pair * 64 + 32, *reinterpret_cast<uint32_t(*)[32]>(&v[32]));
  tmem_ld_wait();
  float f[64];
#pragma unroll
  for (int j = 0; j < 64; ++j) f[j] = __uint_as_float(v[j]);
  if (p.fold_stats) {
    const float nm = -rs.fold.x, c0 = pick(rs.c, 2 * k2), c1 = pick(rs.c, 2 * k2 + 1);
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      f[j] = __fmaf_rn(nm, __shfl_sync(0xffffffffu, c0, j), f[j]) * rs.fold.y;
      f[32 + j] = __fmaf_rn(nm, __shfl_sync(0xffffffffu, c1, j), f[32 + j]) * rs.fold.y;
    }
  }
  if (p.bias) {
    const float b0 = pick(rs.bias, 2 * k2), b1 = pick(rs.bias, 2 * k2 + 1);
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      f[j] += __shfl_sync(0xffffffffu, b0, j);
      f[32 + j] += __shfl_sync(0xffffffffu, b1, j);
    }
  }
  if (p.act == 1) {
#pragma unroll
    for (int j = 0; j < 64; ++j) f[j] = gelu_fast(f[j]);
  }
  // hi plane first, the remainders stay in f (same arithmetic as split_bf16x2, 96 instead of 128 live registers)
  uint32_t w[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * j], f[2 * j + 1]);
    w[j] = *reinterpret_cast<const uint32_t*>(&h);
    f[2 * j] -= __uint_as_float(w[j] << 16);
    f[2 * j + 1] -= __uint_as_float(w[j] & 0xffff0000u);
  }
  store_block_tma(stage, lane, w, &pd.o_hi, n0, warp_row0);
  if (p.nsplit_out == 3) {
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const __nv_bfloat162 l = __floats2bfloat162_rn(f[2 * j], f[2 * j + 1]);
      w[j] = *reinterpret_cast<const uint32_t*>(&l);
    }
    store_block_tma(stage, lane, w, &pd.o_lo, n0, warp_row0);
  }
}

// One 32-column slice of a 128-row accumulator: TMEM -> registers -> [folded LayerNorm] -> bias -> [residual] ->
// [partial statistics] -> row-mapped fp32 rows (output head) or bf16 hi/lo planes.
__device__ __forceinline__ void epilogue_slice(const LinearParams& p, const ChainPhaseDesc& pd, uint32_t tmem_acc, int m_blk, int n_blk,
                                               int slice, int k_in_tile, int lane_group, int lane, uint32_t stage, RowStats& rs, uint4 (&rv)[8],
                                               bool& rv_ready, int next_slice, int warp_in_group, long long* dbg) {
  long long t0 = clock64(), t1;
#define CMDI_T(i) do { if (dbg) { t1 = clock64(); dbg[i] += t1 - t0; t0 = t1; } } while (0)
  const int warp_row0 = m_blk * kBlockM + lane_group * 32;
  const int row = warp_row0 + lane;
  const int n0 = n_blk * kBlockN + slice * 32;
  if (n0 >= p.N) return;  // warp-uniform: columns beyond the layer's width (output head)
  // residual = LayerNorm(v) re-derived from v's bf16 hi / lo planes, or fp32 rows added as they are (layer 0's out-proj)
  const bool res_planes = p.ln_src_hi != nullptr;
  const bool has_res = p.residual || res_planes;
  // the staging tile is about to be rewritten (residual fetch or stores): the bulk store issued from it has been read out
  CMDI_T(8);   // row statistics
  if (lane == 0) tma_store_wait_read();
  __syncwarp();
  CMDI_T(9);   // staging free
  // Residual block of 32 rows x 32 columns, fetched coalesced into rv: fp32 rows (8 x 16 B per thread, 4 complete 128 B
  // row segments per instruction) or the two bf16 planes (4 + 4 x 16 B, 8 complete 64 B segments per instruction).
  // Under this kernel's load an L2 round trip costs ~2 us, so the block of the warp's NEXT slice of the same tile is
  // requested while this one is processed (below); only a tile's first slice pays the latency here.
  auto fetch_residual = [&](int n) {
    if (res_planes) {
#pragma unroll
      for (int it = 0; it < 4; ++it) {
        const long long off = (long long)(warp_row0 + it * 8 + (lane >> 2)) * p.ld_ln + n + (lane & 3) * 8;
        rv[it] = ld_global_cg_v4(p.ln_src_hi + off);
        rv[4 + it] = ld_global_cg_v4(p.ln_src_lo + off);
      }
    } else {
#pragma unroll
      for (int it = 0; it < 8; ++it)
        rv[it] = ld_global_cg_v4(p.residual + (long long)(warp_row0 + it * 4 + (lane >> 3)) * p.ld_res + n + (lane & 7) * 4);
    }
  };
  if (has_res && !rv_ready) fetch_residual(n0);
  rv_ready = false;
  uint32_t v[32];
  tmem_ld32(tmem_acc + slice * 32, v);
  tmem_ld_wait();
  CMDI_T(10);  // residual loads issued + accumulator read
  float f[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
  if (p.fold_stats) {
    // acc = v (W.gamma)^T  ->  rstd * (acc - mean * c[n]);  the bias added next carries W beta + b
    const float nm = -rs.fold.x, ck = pick(rs.c, k_in_tile);
#pragma unroll
    for (int j = 0; j < 32; ++j) f[j] = __fmaf_rn(nm, __shfl_sync(0xffffffffu, ck, j), f[j]) * rs.fold.y;
  }
  if (p.bias) {
    const float bk = pick(rs.bias, k_in_tile);
#pragma unroll
    for (int j = 0; j < 32; ++j) f[j] += __shfl_sync(0xffffffffu, bk, j);
  }
  if (has_res) {
    // transpose through the staging tile: every thread gets its own row
    if (res_planes) {
      // hi block at +0, lo block at +2048, 64 B rows, 16 B chunk c of row r at chunk c ^ ((r >> 1) & 3)
#pragma unroll
      for (int it = 0; it < 4; ++it) {
        const int rr = it * 8 + (lane >> 2);
        const uint32_t a = stage + rr * 64 + ((((uint32_t)lane & 3u) ^ (((uint32_t)rr >> 1) & 3u)) << 4);
        st_shared_v4(a, rv[it].x, rv[it].y, rv[it].z, rv[it].w);
        st_shared_v4(a + 2048, rv[4 + it].x, rv[4 + it].y, rv[4 + it].z, rv[4 + it].w);
      }
    } else {
      const int c = lane & 7;
#pragma unroll
      for (int it = 0; it < 8; ++it) {
        const int rr = it * 4 + (lane >> 3);
        st_shared_v4(stage + rr * 128 + ((c ^ (rr & 7)) << 4), rv[it].x, rv[it].y, rv[it].z, rv[it].w);
      }
    }
    if (next_slice >= 0 && n_blk * kBlockN + next_slice * 32 < p.N) {
      // the registers are free again: request the residual block of this warp's next slice (same tile, same rows)
      fetch_residual(n_blk * kBlockN + next_slice * 32);
      rv_ready = true;
    }
    __syncwarp();
    const float gk = pick(rs.g, k_in_tile), btk = pick(rs.b, k_in_tile);
    if (res_planes) {
      const uint32_t sw = ((uint32_t)lane >> 1) & 3u;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const uint4 uh = ld_shared_v4(stage + lane * 64 + (((uint32_t)c ^ sw) << 4));
        const uint4 ul = ld_shared_v4(stage + 2048 + lane * 64 + (((uint32_t)c ^ sw) << 4));
        const uint32_t hw[4] = {uh.x, uh.y, uh.z, uh.w}, lw[4] = {ul.x, ul.y, ul.z, ul.w};
#pragma unroll
        for (int w = 0; w < 4; ++w) {
          const int j = c * 8 + w * 2;
          const float x0 = __uint_as_float(hw[w] << 16) + __uint_as_float(lw[w] << 16);
          const float x1 = __uint_as_float(hw[w] & 0xffff0000u) + __uint_as_float(lw[w] & 0xffff0000u);
          f[j] += ln_apply(x0, rs.ln.x, rs.ln.y, __shfl_sync(0xffffffffu, gk, j), __shfl_sync(0xffffffffu, btk, j));
          f[j + 1] += ln_apply(x1, rs.ln.x, rs.ln.y, __shfl_sync(0xffffffffu, gk, j + 1), __shfl_sync(0xffffffffu, btk, j + 1));
        }
      }
    } else {
#pragma unroll
      for (int g = 0; g < 8; ++g) {
        const uint4 u = ld_shared_v4(stage + lane * 128 + ((g ^ (lane & 7)) << 4));
        f[g * 4 + 0] += __uint_as_float(u.x); f[g * 4 + 1] += __uint_as_float(u.y);
        f[g * 4 + 2] += __uint_as_float(u.z); f[g * 4 + 3] += __uint_as_float(u.w);
      }
    }
  }
  CMDI_T(11);  // fold + bias + residual
  if (p.stats_out) {
    // LayerNorm statistics of this thread's 32 output values (two-pass in registers), merged into the running pair of
    // the warp's earlier slices of this tile; the warp's last slice of the tile publishes the partial
    float sm = 0.f;
#pragma unroll
    for (int j = 0; j < 32; j += 4) sm += (f[j] + f[j + 1]) + (f[j + 2] + f[j + 3]);
    const float mean32 = sm * (1.0f / 32.0f);
    float q = 0.f;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float a = f[j] - mean32;
      q = fmaf(a, a, q);
    }
    // Chan's update with n_a = 32 k, n_b = 32: n_b / n_ab = 1 / (k + 1), n_a n_b / n_ab = 32 k / (k + 1)
    const float inv = k_in_tile == 0 ? 1.0f : k_in_tile == 1 ? 0.5f : k_in_tile == 2 ? (1.0f / 3.0f) : 0.25f;
    static_assert(kSlicesPerWarp <= 4, "reciprocal table");
    const float delta = mean32 - rs.run_mean;
    rs.run_mean += delta * inv;
    rs.run_m2 += q + delta * delta * (32.0f * (float)k_in_tile * inv);
    if (k_in_tile == kSlicesPerWarp - 1)
      p.stats_out[(size_t)row * kPartialStride + n_blk * kWarpsPerLaneGroup + warp_in_group] = make_float2(rs.run_mean, rs.run_m2);
  }
  CMDI_T(12);  // statistics
  if (p.out_f32) {
    // row-mapped fp32 output (output head: sequence rows -> frame rows, token row dropped): masked coalesced stores
    uint32_t w[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) w[j] = __float_as_uint(f[j]);
    RowSlots rows;
    rows.ok = 0;
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      int pos_unused;
      long long r;
      if (map_row(p, warp_row0 + it * 4 + (lane >> 3), r, pos_unused)) rows.ok |= 1u << it;
      rows.row[it] = (int)r;
    }
    store_block_coalesced(stage, lane, w, reinterpret_cast<char*>(p.out_f32 + n0), rows, (long long)p.ld_f32 * 4, (p.N - n0) / 4, 1, 0);
  }
  CMDI_T(13);  // fp32 store
  if (p.out_hi) {
    uint32_t hw[16], lw[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) split_bf16x2(f[2 * j], f[2 * j + 1], hw[j], lw[j]);
    store_planes_tma(stage, lane, hw, lw, &pd.o_hi, &pd.o_lo, p.nsplit_out == 3, n0, warp_row0);
  }
  CMDI_T(14);  // plane stores
#undef CMDI_T
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kNumThreads, 1)
linear_chain_kernel(const ChainPhaseDesc* __restrict__ phases, const int num_phases, const int total_tiles, long long* dbg) {
  // dbg (bring-up, CMDI_CHAIN_DBG=1): [gridDim.x][kMaxChainPhases][8] cycle counters per CTA and phase:
  //   0 tiles  1 tma: dependency wait  2 tma: slot wait  3 mma: operand wait  4 mma: accumulator wait
  //   5 epilogue warp 0: accumulator wait  6 its slice work  7 its publish wait
  long long* dbg_me = dbg ? dbg + (size_t)blockIdx.x * kMaxChainPhases * 16 : nullptr;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* ring_a = smem;
  uint8_t* ring_w = ring_a + kStagesA * kOperandBytes;
  uint8_t* epi_stage = ring_w + kStagesW * kOperandBytes;  // kNumEpiWarps x 4 KB store-staging tiles
  ChainBarriers* bars = reinterpret_cast<ChainBarriers*>(epi_stage + kNumEpiWarps * kEpiStageBytes);
  ChainPhaseInfo* info = reinterpret_cast<ChainPhaseInfo*>(bars + 1);

  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = cluster_ctarank();
  const bool leader = cta_rank == 0;
  const int cluster_id = blockIdx.x >> 1;
  const int num_clusters = gridDim.x >> 1;
  const int my_tiles = (total_tiles - cluster_id + num_clusters - 1) / num_clusters;

  // phase descriptors (all but the tensor maps) into shared memory: every role reads them per tile
  for (int i = threadIdx.x; i < num_phases * (int)(sizeof(ChainPhaseInfo) / 4); i += kNumThreads) {
    const int ph = i / (int)(sizeof(ChainPhaseInfo) / 4), w = i % (int)(sizeof(ChainPhaseInfo) / 4);
    reinterpret_cast<uint32_t*>(info + ph)[w] = reinterpret_cast<const uint32_t*>(&phases[ph].info)[w];
  }
  if (warp_idx == 0 && lane == 0) {
    for (int ph = 0; ph < num_phases; ++ph) {
      tma_prefetch_desc(&phases[ph].a_hi);
      tma_prefetch_desc(&phases[ph].w_hi);
    }
    for (int s = 0; s < kStagesA; ++s) {
      mbar_init(&bars->full_a[s], 1);
      mbar_init(&bars->empty_a[s], 1);
    }
    for (int s = 0; s < kStagesW; ++s) {
      mbar_init(&bars->full_w[s], 1);
      mbar_init(&bars->empty_w[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&bars->tmem_full[s], 1);
      mbar_init(&bars->tmem_empty[s], 2 * 4 * kSlices);  // every (CTA, lane group, slice) arrives once per tile
    }
    for (int s = 0; s < kPublishBars; ++s) mbar_init(&bars->publish[s], kNumEpiWarps);
    fence_barrier_init();
  }
  if (warp_idx == 2) {
    tmem_alloc_2sm(&bars->tmem_base, kTmemCols);
    tmem_relinquish_2sm();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // barrier inits + TMEM allocation visible to both CTAs
  tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;

  if (warp_idx == 0) {
    // ===================================== TMA producer (both CTAs) =====================================
    if (lane == 0) {
      int sa = 0, sw = 0, ph = 0;
      uint32_t pa = 0, pw = 0;
      for (int seq = 0; seq < my_tiles; ++seq) {
        const int tile = cluster_id + seq * num_clusters;
        while (tile >= info[ph].tile_end) ++ph;
        const ChainPhaseInfo& pi = info[ph];
        const ChainPhaseDesc& pd = phases[ph];
        const int local = tile - pi.tile_begin;
        const int m_pair = local / pi.num_n_blocks;
        const int m_blk = 2 * m_pair + (int)cta_rank;
        const int n_blk = local % pi.num_n_blocks;
        const int nplanes = (pi.p.nsplit == 3) ? 2 : 1;
        const uint32_t tx_bytes = 2u * nplanes * kPlaneBytes;  // both CTAs' loads complete on the leader's barrier
        long long c0 = clock64();
        if (pi.wait_ctr) {
          // the A rows of this row pair are written by an earlier phase of this launch
          wait_counter(pi.wait_ctr + m_pair, pi.wait_target);
          fence_proxy_async_all();
        }
        if (dbg_me) { dbg_me[ph * 16 + 0] += 1; dbg_me[ph * 16 + 1] += clock64() - c0; }
        for (int kb = 0; kb < pi.num_k_blocks; ++kb) {
          c0 = clock64();
          mbar_wait(&bars->empty_w[sw], pw ^ 1);
          if (pi.p.debug & 4) {
            // bring-up decomposition (CMDI_DEBUG=4): no operand loads, only the pipeline bookkeeping
            mbar_wait(&bars->empty_a[sa], pa ^ 1);
            if (leader) { mbar_arrive(&bars->full_w[sw]); mbar_arrive(&bars->full_a[sa]); }
            if (++sa == kStagesA) { sa = 0; pa ^= 1; }
            if (++sw == kStagesW) { sw = 0; pw ^= 1; }
            continue;
          }
          uint8_t* dw = ring_w + (size_t)sw * kOperandBytes;
          if (leader) mbar_arrive_expect_tx(&bars->full_w[sw], tx_bytes);
          tma_load_2d_2sm(dw, &pd.w_hi, &bars->full_w[sw], kb * kBlockK, n_blk * kBlockN + (int)cta_rank * (kBlockN / 2));
          if (nplanes == 2)
            tma_load_2d_2sm(dw + kPlaneBytes, &pd.w_lo, &bars->full_w[sw], kb * kBlockK, n_blk * kBlockN + (int)cta_rank * (kBlockN / 2));
          mbar_wait(&bars->empty_a[sa], pa ^ 1);
          if (dbg_me) dbg_me[ph * 16 + 2] += clock64() - c0;
          uint8_t* da = ring_a + (size_t)sa * kOperandBytes;
          if (leader) mbar_arrive_expect_tx(&bars->full_a[sa], tx_bytes);
          tma_load_2d_2sm(da, &pd.a_hi, &bars->full_a[sa], kb * kBlockK, m_blk * kBlockM);
          if (nplanes == 2) tma_load_2d_2sm(da + kPlaneBytes, &pd.a_lo, &bars->full_a[sa], kb * kBlockK, m_blk * kBlockM);
          if (++sa == kStagesA) { sa = 0; pa ^= 1; }
          if (++sw == kStagesW) { sw = 0; pw ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp_idx == 1) {
    // ====================================== MMA issuer (leader CTA only) ======================================
    if (leader && lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(2 * kBlockM, kBlockN, 0);
      int sa = 0, sw = 0, ph = 0;
      uint32_t pa = 0, pw = 0;
      for (int seq = 0; seq < my_tiles; ++seq) {
        const int tile = cluster_id + seq * num_clusters;
        while (tile >= info[ph].tile_end) ++ph;
        const ChainPhaseInfo& pi = info[ph];
        const bool split = pi.p.nsplit == 3;
        const int acc = seq & 1;
        long long c0 = clock64();
        mbar_wait(&bars->tmem_empty[acc], ((seq >> 1) & 1) ^ 1);
        if (dbg_me) dbg_me[ph * 16 + 4] += clock64() - c0;
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * kAccStride;
        for (int kb = 0; kb < pi.num_k_blocks; ++kb) {
          c0 = clock64();
          mbar_wait(&bars->full_w[sw], pw);
          mbar_wait(&bars->full_a[sa], pa);
          if (dbg_me) dbg_me[ph * 16 + 3] += clock64() - c0;
          tc_fence_after();
          const uint32_t a_addr = smem_u32(ring_a + (size_t)sa * kOperandBytes);
          const uint32_t w_addr = smem_u32(ring_w + (size_t)sw * kOperandBytes);
          const uint64_t da_hi = make_desc_kmajor_sw128(a_addr);
          const uint64_t db_hi = make_desc_kmajor_sw128(w_addr);
          if (pi.p.debug & 2) {
            // bring-up decomposition (CMDI_DEBUG=2): no MMAs, only the pipeline bookkeeping
          } else if (split) {
            const uint64_t da_lo = make_desc_kmajor_sw128(a_addr + kPlaneBytes);
            const uint64_t db_lo = make_desc_kmajor_sw128(w_addr + kPlaneBytes);
#pragma unroll
            for (int k = 0; k < kBlockK / kUmmaK; ++k)
              umma_ss_2sm(d_tmem, desc_advance(da_lo, k * kUmmaK * 2), desc_advance(db_hi, k * kUmmaK * 2), idesc,
                          (kb > 0 || k > 0) ? 1u : 0u);
#pragma unroll
            for (int k = 0; k < kBlockK / kUmmaK; ++k)
              umma_ss_2sm(d_tmem, desc_advance(da_hi, k * kUmmaK * 2), desc_advance(db_lo, k * kUmmaK * 2), idesc, 1u);
#pragma unroll
            for (int k = 0; k < kBlockK / kUmmaK; ++k)
              umma_ss_2sm(d_tmem, desc_advance(da_hi, k * kUmmaK * 2), desc_advance(db_hi, k * kUmmaK * 2), idesc, 1u);
          } else {
#pragma unroll
            for (int k = 0; k < kBlockK / kUmmaK; ++k)
              umma_ss_2sm(d_tmem, desc_advance(da_hi, k * kUmmaK * 2), desc_advance(db_hi, k * kUmmaK * 2), idesc,
                          (kb > 0 || k > 0) ? 1u : 0u);
          }
          umma_commit_2sm(&bars->empty_a[sa], 0x3);  // frees the slots in BOTH CTAs
          umma_commit_2sm(&bars->empty_w[sw], 0x3);
          if (++sa == kStagesA) { sa = 0; pa ^= 1; }
          if (++sw == kStagesW) { sw = 0; pw ^= 1; }
        }
        umma_commit_2sm(&bars->tmem_full[acc], 0x3);  // both CTAs' epilogues may read their half of the tile
      }
    }
    __syncwarp();
  } else if (warp_idx == 2) {
    // ============ publisher: one release fence + counter bump per tile, off the epilogue warps' critical path ============
    if (lane == 0) {
      int ph = 0;
      for (int seq = 0; seq < my_tiles; ++seq) {
        const int tile = cluster_id + seq * num_clusters;
        while (tile >= info[ph].tile_end) ++ph;
        const ChainPhaseInfo& pi = info[ph];
        mbar_wait(&bars->publish[seq & (kPublishBars - 1)], (seq / kPublishBars) & 1);
        if (pi.done_ctr) {
          fence_proxy_async_all();
          __threadfence();
          atomicAdd(pi.done_ctr + (tile - pi.tile_begin) / pi.num_n_blocks, 1);
        }
      }
    }
    __syncwarp();
  } else {
    // ============ epilogue warps: two per TMEM lane group; four 32-column slices or two 64-column pairs per warp and tile ============
    const int ew = warp_idx - kFirstEpiWarp;
    const int lane_group = warp_idx & 3;  // the TMEM lanes a warp may touch: 32 * (warp index % 4)
    const int j3 = ew >> 2;               // index within the lane group
    const uint32_t epi_stage_addr = smem_u32(epi_stage + ew * kEpiStageBytes);
    const uint32_t tmem_lane = tmem_base + ((uint32_t)(lane_group * 32) << 16);
    int ph = 0;
    RowStats rs{};
    // everything this warp stored for tile `seq` is in memory: tell the publisher
    auto publish = [&](int seq) {
      __syncwarp();  // the other lanes' plain stores (row-mapped outputs, partial statistics) before lane 0's release
      if (lane == 0) {
        tma_store_wait_all();
        mbar_arrive(&bars->publish[seq & (kPublishBars - 1)]);
      }
    };
    for (int seq = 0; seq < my_tiles; ++seq) {
      long long c0 = clock64();
      const int tile = cluster_id + seq * num_clusters;
      while (tile >= info[ph].tile_end) ++ph;
      const ChainPhaseInfo& pi = info[ph];
      const int local = tile - pi.tile_begin;
      const int m_blk = 2 * (local / pi.num_n_blocks) + (int)cta_rank;
      const int n_blk = local % pi.num_n_blocks;
      const int acc = seq & 1;
      const bool pairs = pi.pair_epilogue != 0;
      load_tile_constants(pi.p, rs, n_blk, j3, pairs, lane);
      mbar_wait(&bars->tmem_full[acc], (seq >> 1) & 1);
      long long c1 = clock64();
      tc_fence_after();
      load_row_statistics(pi.p, rs, m_blk * kBlockM + lane_group * 32 + lane);
      const uint32_t tmem_acc = tmem_lane + acc * kAccStride;
      long long* dbg_w = (dbg_me && ew == 0 && lane == 0) ? dbg_me + ph * 16 : nullptr;
      if (pairs) {
#pragma unroll 1
        for (int k2 = 0; k2 < kSlicesPerWarp / 2; ++k2) {
          epilogue_pair(pi.p, phases[ph], tmem_acc, m_blk, n_blk, j3 + kWarpsPerLaneGroup * k2, k2, lane_group, lane, epi_stage_addr, rs);
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {  // one arrival per 32-column slice keeps the barrier's count independent of the phase
            mbar_arrive_on_leader(&bars->tmem_empty[acc]);
            mbar_arrive_on_leader(&bars->tmem_empty[acc]);
          }
        }
      } else {
        uint4 rv[8];  // residual block in flight for this warp's next slice (see epilogue_slice)
        bool rv_ready = false;
#pragma unroll 1
        for (int k = 0; k < kSlicesPerWarp; ++k) {
          const int slice = j3 + k * kWarpsPerLaneGroup;
          const int next_slice = k + 1 < kSlicesPerWarp ? slice + kWarpsPerLaneGroup : -1;
          epilogue_slice(pi.p, phases[ph], tmem_acc, m_blk, n_blk, slice, k, lane_group, lane, epi_stage_addr, rs, rv, rv_ready,
                         next_slice, j3, dbg_w);
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_on_leader(&bars->tmem_empty[acc]);
        }
      }
      long long c2 = clock64();
      publish(seq);
      if (dbg_me && ew == 0 && lane == 0) {
        dbg_me[ph * 16 + 5] += c1 - c0; dbg_me[ph * 16 + 6] += c2 - c1; dbg_me[ph * 16 + 7] += clock64() - c2;
      }
    }
    if (lane == 0) tma_store_wait_all();
  }

  tc_fence_before();
  cluster_sync_all();  // nobody touches the pair's TMEM / barriers after this point
  if (warp_idx == 2) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, kTmemCols);
  }
}

}  // namespace

cudaError_t configure_linear_chain_kernel() {
  return cudaFuncSetAttribute(linear_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
}

// how many CTA pairs of this kernel can be resident at once on the current device (they spin on each other's counters:
// the launch must never exceed this)
int linear_chain_max_clusters(int num_sms) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(2 * (num_sms / 2));
  cfg.blockDim = dim3(kNumThreads);
  cfg.dynamicSmemBytes = kSmemBytes;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, linear_chain_kernel, &cfg) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

cudaError_t launch_linear_chain(const ChainPhaseDesc* phases_dev, int num_phases, int total_tiles, int num_sms, cudaStream_t stream,
                                long long* dbg) {
  if (num_phases < 1 || num_phases > kMaxChainPhases || total_tiles < 1) {
    set_last_error("launch_linear_chain: bad phase list (%d phases, %d tiles)", num_phases, total_tiles);
    return cudaErrorInvalidValue;
  }
  static int max_clusters = -1;
  if (max_clusters < 0) max_clusters = linear_chain_max_clusters(num_sms);
  int clusters = num_sms / 2;
  if (clusters > total_tiles) clusters = total_tiles;
  if (clusters > max_clusters) {
    set_last_error("launch_linear_chain: %d co-resident CTA pairs needed, the device offers %d", clusters, max_clusters);
    return cudaErrorInvalidConfiguration;
  }
  return launch_kernel(linear_chain_kernel, dim3(2 * clusters), dim3(kNumThreads), (size_t)kSmemBytes, stream, phases_dev,
                          num_phases, total_tiles, dbg);
}

}  // namespace cmdi
