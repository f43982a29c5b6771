// Self-attention core of nn.MultiheadAttention for the MDM encoder (reference: model/mdm.py:107-114, :284;
// no key-padding mask -- `src_key_padding_mask` is commented out there), head dim 128, S <= 208 keys:
//
//   O[s, :] = softmax_j( Q[s,:] . K[j,:] / sqrt(128) ) V[j, :]
//
// One CTA PAIR (cluster of 2) per (sequence, head): CTA r owns query rows [128 r, 128 r + 128).  Both contractions run
// on tcgen05 tensor cores as cta_group::2 MMAs (M = 256):
//   S = Q K^T   : A = Q tiles (smem, K-major), B = K (smem, K-major, keys split between the CTAs), D = 256 x 208 fp32
//   O = P V     : A = P (bf16, written into TMEM by the softmax warps over S), B = V (smem, MN-major, head-dim columns
//                 split between the CTAs), D = 256 x 128 fp32, double-buffered in TMEM
// Q, K and V are read straight out of the QKV projection's [tokens, 3*H*128] bf16 planes with TMA
// (no head-split or transpose kernels).  With nsplit = 3 every product uses the hi/lo bf16 split
// (X_lo*Y_hi + X_hi*Y_lo + X_hi*Y_hi), P included, so the result is fp32-accurate.
//
// warp 0: TMA producer   warp 1: MMA issuer (leader CTA; + TMEM alloc)
// warps 2..9: softmax + output.  Two threads per query row (TMEM lane group = warp % 4, key half = (warp-2)/4):
//   each keeps its ~104 logits in registers (one TMEM read), the halves exchange row max / row sum through
//   shared memory, P is written back to TMEM, and O leaves as bf16 hi / lo planes through TMA stores.
#include "common.cuh"
#include "gemm_epilogue.cuh"
#include "kernels.h"

namespace cmdi {

namespace {

constexpr int kHeadDim = 128;
constexpr int kQTile = 128;
constexpr int kKeyPad = kAttnKeyPad;            // 208 = 13 * 16
constexpr int kQBlockBytes = kQTile * 128;      // 64 dh-columns of 128 queries
constexpr int kKVBlockBytes = kKeyPad * 128;    // 64 dh-columns of 208 keys  (26 swizzle atoms)
constexpr int kQPlane = 2 * kQBlockBytes;       // 32768
constexpr int kNumSoftmaxWarps = 8;
constexpr int kThreads = 64 + kNumSoftmaxWarps * 32;
// TMEM columns
constexpr uint32_t kColS = 0, kColPHi = 0, kTmemCols = 512;
// key chunks (16 keys each) per half: half 0 -> chunks [0,7), half 1 -> chunks [7,13)
constexpr int kChunks0 = 7, kChunks1 = 6;
// ... of which the first kEarly0 / kEarly1 are handed to the P V product early (see softmax_half).  Cycles per launch at
// 64 x 197 x 4 for (kEarly0, kEarly1): (3,2) 58.3k, (4,3) 57.0k, (5,4) 57.8k, (6,5) 59.4k; without the early hand-over 59.4k.
constexpr int kEarly0 = 4, kEarly1 = 3;

__device__ __forceinline__ void named_barrier_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// logits of this thread's key range -> registers, row max, exchange, probabilities -> TMEM, row sum
// `part_a`: barrier (on the pair's leader) that collects one arrival per softmax warp once the first EARLY chunks of P
// are in tensor memory -- the P V product over those keys starts while the remaining probabilities are computed.
template <int CHUNK0, int NCHUNKS, int EARLY>
__device__ __forceinline__ float softmax_half(uint32_t trow, int S, bool split, float c_scale, float (*red_max)[128], int half,
                                              int row, uint32_t col_plo, uint64_t* part_a, int lane) {
  float s[NCHUNKS * 16];
  {
    // all TMEM reads in flight at once, one wait
    uint32_t v[NCHUNKS][16];
#pragma unroll
    for (int c = 0; c < NCHUNKS; ++c) tmem_ld16(trow + kColS + (CHUNK0 + c) * 16, v[c]);
    tmem_ld_wait();
#pragma unroll
    for (int c = 0; c < NCHUNKS; ++c)
#pragma unroll
      for (int j = 0; j < 16; ++j)
        s[c * 16 + j] = ((CHUNK0 + c) * 16 + j < S) ? __uint_as_float(v[c][j]) : -INFINITY;  // padded keys: exp2 -> 0
  }
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < NCHUNKS * 16; ++i) mx = fmaxf(mx, s[i]);
  red_max[half][row] = mx;
  // every S value is in registers now: after this barrier P may overwrite the S columns
  tc_fence_before();
  named_barrier_sync(1, kNumSoftmaxWarps * 32);
  tc_fence_after();
  mx = fmaxf(red_max[0][row], red_max[1][row]);
  const float mc = mx * c_scale;
  float sum = 0.f;
#pragma unroll
  for (int c = 0; c < NCHUNKS; ++c) {
    uint32_t ph[8], pl[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float p0 = fast_exp2(fmaf(s[c * 16 + j * 2], c_scale, -mc));
      const float p1 = fast_exp2(fmaf(s[c * 16 + j * 2 + 1], c_scale, -mc));
      sum += p0 + p1;
      split_bf16x2(p0, p1, ph[j], pl[j]);
    }
    tmem_st8(trow + kColPHi + (CHUNK0 + c) * 8, ph);
    if (split) tmem_st8(trow + col_plo + (CHUNK0 + c) * 8, pl);
    if (c == EARLY - 1) {
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_on_leader(part_a);
    }
  }
  return sum;
}

// ------------------------------------------------------------------------------------------------
// Shared memory.  K is split by keys and V by head-dim columns between the two CTAs, so a CTA holds Q (64 KB) + half of
// K (52 KB) + half of V (52 KB) + its store staging (32 KB) with NO region shared between operands: Q_{i+1} and K_{i+1}
// are requested as soon as S_i is complete and V_{i+1} as soon as O_i is, all of it behind the softmax / PV / output
// work of item i.  (Round 1's one-CTA-per-query-tile kernel needed 272 KB for the same residency: V_lo overlaid Q, so
// Q_{i+1} could only be requested at o_done_i and its ~2 us L2 round trip sat on every item's critical path; measured
// at 64 x 197 x 4: 44.2 -> 40.2 us per launch on the same box.)
// Per item the tensor pipe needs ~2500 cycles for S and ~2500 for P V (3 bf16 terms each) and the softmax warps ~6000;
// S_{i+1} cannot start before P_i V_i has retired (P overwrites S in place: two S buffers + O exceed the 512 TMEM
// columns), so the loop softmax -> P V -> S -> softmax bounds an item at ~12 000 cycles; the output of item i-1 is
// written under P_i V_i / S_{i+1} from the other O buffer.
// ------------------------------------------------------------------------------------------------
constexpr int kKHalf = kKeyPad / 2;                     // 104 keys per CTA
constexpr int kKHalfBlockBytes = kKHalf * 128;          // 64 dh-columns of 104 keys (13 swizzle atoms)
constexpr int kKHalfPlane = 2 * kKHalfBlockBytes;       // 26624
constexpr int kVHalfPlane = kKVBlockBytes;              // 64 dh-columns of 208 keys: 26624
constexpr int kPOffQHi = 0, kPOffQLo = kQPlane;
constexpr int kPOffKHi = 2 * kQPlane, kPOffKLo = kPOffKHi + kKHalfPlane;
constexpr int kPOffVHi = kPOffKLo + kKHalfPlane, kPOffVLo = kPOffVHi + kVHalfPlane;
constexpr int kPOffStage = kPOffVLo + kVHalfPlane;
constexpr int kPairSmemTiles = kPOffStage + kNumSoftmaxWarps * kEpiStageBytes;  // 204800
// TMEM columns of the pair kernel: P (hi | lo) overwrites S in place, O is double-buffered (the output stores of item i
// run under the PV product of item i+1)
constexpr uint32_t kPColPLo = 104, kPColO = 208, kPColOStride = 128;
static_assert(kPColO + 2 * kPColOStride <= kTmemCols, "tensor memory budget");
static_assert(kKHalfBlockBytes % 1024 == 0 && kVHalfPlane % 1024 == 0, "swizzle-atom alignment of the operand tiles");

struct __align__(8) AttnPairBarriers {
  uint64_t q_full, k_full, v_full;  // on the leader CTA: both CTAs' loads complete there
  uint64_t s_done, o_done;          // in both CTAs (multicast commit)
  uint64_t p_part, p_full;          // on the leader: one arrival per softmax warp of the pair (early chunks / all of P)
  uint32_t tmem_base;
  uint32_t pad;
  float red_max[2][128];
  float red_sum[2][128];
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
attention_pair_kernel(const __grid_constant__ CUtensorMap map_q_hi, const __grid_constant__ CUtensorMap map_q_lo,
                      const __grid_constant__ CUtensorMap map_kh_hi, const __grid_constant__ CUtensorMap map_kh_lo,
                      const __grid_constant__ CUtensorMap map_kv_hi, const __grid_constant__ CUtensorMap map_kv_lo,
                      const __grid_constant__ CUtensorMap map_o_hi, const __grid_constant__ CUtensorMap map_o_lo,
                      const AttnParams p, const int num_items) {
  const long long t_entry = clock64();
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  AttnPairBarriers* bars = reinterpret_cast<AttnPairBarriers*>(smem + kPairSmemTiles);

  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int S = p.seq_len;
  const bool split = (p.nsplit == 3);
  const uint32_t cta_rank = cluster_ctarank();
  const bool leader = cta_rank == 0;
  const int cluster_id = blockIdx.x >> 1;
  const int num_clusters = gridDim.x >> 1;

  if (warp_idx == 0 && lane == 0) {
    tma_prefetch_desc(&map_q_hi);
    tma_prefetch_desc(&map_kh_hi);
    tma_prefetch_desc(&map_kv_hi);
    mbar_init(&bars->q_full, 1);
    mbar_init(&bars->k_full, 1);
    mbar_init(&bars->v_full, 1);
    mbar_init(&bars->s_done, 1);
    mbar_init(&bars->o_done, 1);
    mbar_init(&bars->p_part, 2 * kNumSoftmaxWarps);
    mbar_init(&bars->p_full, 2 * kNumSoftmaxWarps);
    fence_barrier_init();
  }
  if (warp_idx == 1) {
    tmem_alloc_2sm(&bars->tmem_base, kTmemCols);
    tmem_relinquish_2sm();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // barrier inits + TMEM allocation visible to both CTAs
  tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;

  // item -> (sequence, head)
  auto decode = [&](int w, int& seq, int& head) {
    head = w % p.num_heads;
    seq = w / p.num_heads;
  };

  if (warp_idx == 0) {
    // ===================================== TMA producer (both CTAs) =====================================
    if (lane == 0) {
      const uint32_t planes = split ? 2 : 1;
      auto load_q = [&](int w) {   // this CTA's 128 query rows
        int seq, head;
        decode(w, seq, head);
        const int row = seq * S + (int)cta_rank * kQTile, col = head * kHeadDim;
        if (leader) mbar_arrive_expect_tx(&bars->q_full, 2 * planes * kQPlane);
        for (int j = 0; j < 2; ++j) {
          tma_load_2d_2sm(smem + kPOffQHi + j * kQBlockBytes, &map_q_hi, &bars->q_full, col + j * 64, row);
          if (split) tma_load_2d_2sm(smem + kPOffQLo + j * kQBlockBytes, &map_q_lo, &bars->q_full, col + j * 64, row);
        }
      };
      auto load_k = [&](int w) {   // this CTA's 104 keys of K
        int seq, head;
        decode(w, seq, head);
        const int row = seq * S + (int)cta_rank * kKHalf, col = p.num_heads * kHeadDim + head * kHeadDim;
        if (leader) mbar_arrive_expect_tx(&bars->k_full, 2 * planes * kKHalfPlane);
        for (int j = 0; j < 2; ++j) {
          tma_load_2d_2sm(smem + kPOffKHi + j * kKHalfBlockBytes, &map_kh_hi, &bars->k_full, col + j * 64, row);
          if (split) tma_load_2d_2sm(smem + kPOffKLo + j * kKHalfBlockBytes, &map_kh_lo, &bars->k_full, col + j * 64, row);
        }
      };
      auto load_v = [&](int w) {   // this CTA's 64 head-dim columns of V, all keys
        int seq, head;
        decode(w, seq, head);
        const int col = 2 * p.num_heads * kHeadDim + head * kHeadDim + (int)cta_rank * 64;
        if (leader) mbar_arrive_expect_tx(&bars->v_full, 2 * planes * kVHalfPlane);
        tma_load_2d_2sm(smem + kPOffVHi, &map_kv_hi, &bars->v_full, col, seq * S);
        if (split) tma_load_2d_2sm(smem + kPOffVLo, &map_kv_lo, &bars->v_full, col, seq * S);
      };
      int w = cluster_id;
      if (w < num_items) {
        load_q(w);
        load_k(w);
        load_v(w);
      }
      for (uint32_t it = 0; w < num_items; w += num_clusters, ++it) {
        const uint32_t ph = it & 1;
        const int wn = w + num_clusters;
        mbar_wait(&bars->s_done, ph);  // Q_i and K_i consumed (in both CTAs)
        if (wn < num_items) {
          load_q(wn);
          load_k(wn);
        }
        mbar_wait(&bars->o_done, ph);  // V_i consumed
        if (wn < num_items) load_v(wn);
      }
    }
    __syncwarp();
  } else if (warp_idx == 1) {
    // ====================================== MMA issuer (leader CTA only) ======================================
    if (leader && lane == 0) {
      const uint32_t sbase = smem_u32(smem);
      constexpr uint32_t idesc_s = make_idesc_bf16(2 * kQTile, kKeyPad, 0);
      constexpr uint32_t idesc_o = make_idesc_bf16(2 * kQTile, kHeadDim, 1);
      const int nterms = split ? 3 : 1;
      long long acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      auto issue_s = [&](uint32_t ph) {
        long long t0 = clock64(), t1;
        mbar_wait(&bars->q_full, ph);
        t1 = clock64(); acc[0] += t1 - t0; t0 = t1;
        mbar_wait(&bars->k_full, ph);
        t1 = clock64(); acc[1] += t1 - t0; t0 = t1;
        tc_fence_after();
        uint32_t accum = 0;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
#pragma unroll
          for (int term = 0; term < 3; ++term) {
            if (term >= nterms) break;
            const uint32_t qo = (split && term == 0) ? kPOffQLo : kPOffQHi;
            const uint32_t ko = (split && term == 1) ? kPOffKLo : kPOffKHi;
            const uint64_t da = make_desc_kmajor_sw128(sbase + qo + j * kQBlockBytes);
            const uint64_t db = make_desc_kmajor_sw128(sbase + ko + j * kKHalfBlockBytes);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
              umma_ss_2sm(tmem_base + kColS, desc_advance(da, kk * 32), desc_advance(db, kk * 32), idesc_s, accum);
              accum = 1;
            }
          }
        }
        umma_commit_2sm(&bars->s_done, 0x3);
        t1 = clock64(); acc[2] += t1 - t0;
      };
      const long long t_loop = clock64();
      uint32_t it = 0;
      if (cluster_id < num_items) issue_s(0);
      for (int w = cluster_id; w < num_items; w += num_clusters, ++it) {
        const uint32_t ph = it & 1;
        long long t0 = clock64(), t1;
        // ---------------- O = P V ----------------
        // (p_full of this item also implies the softmax warps have finished reading O of item i-2, the previous user of
        // this O buffer: they store item i-1's output after arriving here and item i-2's before)
        mbar_wait(&bars->p_part, ph);
        t1 = clock64(); acc[3] += t1 - t0; t0 = t1;
        mbar_wait(&bars->v_full, ph);
        t1 = clock64(); acc[4] += t1 - t0; t0 = t1;
        tc_fence_after();
        const uint64_t dv_hi = make_desc_mnmajor_sw128(sbase + kPOffVHi, kKVBlockBytes);
        const uint64_t dv_lo = make_desc_mnmajor_sw128(sbase + kPOffVLo, kKVBlockBytes);
        const uint32_t col_o = tmem_base + kPColO + ph * kPColOStride;
        // one bf16 term over the key chunks [c0, c1) of half 0 and [d0, d1) of half 1 (term-major order: alternating the
        // operand planes per chunk measured 70 % slower)
        uint32_t accum = 0;
        auto pv_term = [&](uint32_t p_col, uint64_t dv, int c0, int c1, int d0, int d1) {
#pragma unroll
          for (int c = 0; c < kChunks0; ++c) {
            if (c < c0 || c >= c1) continue;
            umma_ts_2sm(col_o, tmem_base + p_col + c * 8, desc_advance(dv, c * 2048), idesc_o, accum);
            accum = 1;
          }
#pragma unroll
          for (int c = 0; c < kChunks1; ++c) {
            if (c < d0 || c >= d1) continue;
            umma_ts_2sm(col_o, tmem_base + p_col + (kChunks0 + c) * 8, desc_advance(dv, (kChunks0 + c) * 2048), idesc_o, accum);
            accum = 1;
          }
        };
        // keys whose probabilities are already in tensor memory: the first kEarly0 / kEarly1 chunks of the two halves
        if (split) pv_term(kPColPLo, dv_hi, 0, kEarly0, 0, kEarly1);
        pv_term(kColPHi, dv_hi, 0, kEarly0, 0, kEarly1);
        if (split) pv_term(kColPHi, dv_lo, 0, kEarly0, 0, kEarly1);
        t1 = clock64(); acc[5] += t1 - t0; t0 = t1;
        mbar_wait(&bars->p_full, ph);
        t1 = clock64(); acc[3] += t1 - t0; t0 = t1;
        tc_fence_after();
        if (split) pv_term(kPColPLo, dv_hi, kEarly0, kChunks0, kEarly1, kChunks1);
        pv_term(kColPHi, dv_hi, kEarly0, kChunks0, kEarly1, kChunks1);
        if (split) pv_term(kColPHi, dv_lo, kEarly0, kChunks0, kEarly1, kChunks1);
        umma_commit_2sm(&bars->o_done, 0x3);
        t1 = clock64(); acc[5] += t1 - t0; t0 = t1;
        if (w + num_clusters < num_items) {
          // S_{i+1} overwrites the columns P_i is read from: wait until the PV MMAs have retired (the output stores of
          // item i, ~3000 cycles, cover it)
          mbar_wait(&bars->o_done, ph);
          t1 = clock64(); acc[6] += t1 - t0;
          issue_s(ph ^ 1);
        }
        acc[7] += 1;
      }
      if (p.dbg_cycles) {
        for (int i = 0; i < 8; ++i) p.dbg_cycles[(size_t)cluster_id * 16 + i] = acc[i];
        p.dbg_cycles[(size_t)cluster_id * 16 + 12] = t_loop - t_entry;
        p.dbg_cycles[(size_t)cluster_id * 16 + 13] = clock64() - t_entry;
      }
    }
    __syncwarp();
  } else {
    // ---------------- softmax + output: two threads per query row (both CTAs, each its own 128 rows) ----------------
    const int sw = warp_idx - 2;
    const int lane_group = warp_idx & 3;
    const int half = sw >> 2;
    const int row = lane_group * 32 + lane;
    const uint32_t trow = tmem_base + ((uint32_t)(lane_group * 32) << 16);
    const float c_scale = 0.08838834764831845f * 1.4426950408889634f;  // 1/sqrt(128) * log2(e)
    const uint32_t stage = smem_u32(smem + kPOffStage + sw * kEpiStageBytes);
    const long long pitch = (long long)p.ld_out * 2;
    const int group_row0 = (int)cta_rank * kQTile + lane_group * 32;  // first query of this warp's 32 rows
    long long sacc[4] = {0, 0, 0, 0};
    // output of one item: O (TMEM buffer `buf`) * 1 / row sum -> bf16 hi / lo planes
    auto write_output = [&](int w, uint32_t buf, float inv) {
      int seq, head;
      decode(w, seq, head);
      const int row0 = seq * S;
      uint32_t v0[32], v1[32];
      tmem_ld32(trow + kPColO + buf * kPColOStride + half * 64, v0);
      tmem_ld32(trow + kPColO + buf * kPColOStride + half * 64 + 32, v1);
      tmem_ld_wait();
      uint32_t hw[32], lw[32];
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        split_bf16x2(__uint_as_float(v0[2 * j]) * inv, __uint_as_float(v0[2 * j + 1]) * inv, hw[j], lw[j]);
        split_bf16x2(__uint_as_float(v1[2 * j]) * inv, __uint_as_float(v1[2 * j + 1]) * inv, hw[16 + j], lw[16 + j]);
      }
      if (group_row0 + 32 <= S) {
        store_block_tma(stage, lane, hw, &map_o_hi, head * kHeadDim + half * 64, row0 + group_row0);
        if (p.nsplit_out == 3) store_block_tma(stage, lane, lw, &map_o_lo, head * kHeadDim + half * 64, row0 + group_row0);
      } else if (group_row0 < S) {
        RowSlots rows;
        rows.ok = 0;
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          const int qp = group_row0 + r * 4 + (lane >> 3);
          rows.row[r] = (qp < S) ? (row0 + qp) : 0;
          if (qp < S) rows.ok |= 1u << r;
        }
        char* dst_hi = reinterpret_cast<char*>(p.out_hi + head * kHeadDim + half * 64);
        store_block_coalesced(stage, lane, hw, dst_hi, rows, pitch, 8, 1, 0);
        if (p.nsplit_out == 3) {
          char* dst_lo = reinterpret_cast<char*>(p.out_lo + head * kHeadDim + half * 64);
          store_block_coalesced(stage, lane, lw, dst_lo, rows, pitch, 8, 1, 0);
        }
      }
    };
    // Software pipeline: softmax of item i, then -- while the pair's tensor cores run P_i V_i and S_{i+1} -- the output
    // of item i-1 from the other O buffer.  No barrier wait is needed for that output: s_done_i, waited for above, was
    // issued after the MMA thread saw o_done_{i-1}.
    uint32_t it = 0;
    int w_prev = -1;
    float inv_prev = 0.f;
    for (int w = cluster_id; w < num_items; w += num_clusters, ++it) {
      const uint32_t ph = it & 1;
      long long u0 = clock64(), u1;
      mbar_wait(&bars->s_done, ph);
      u1 = clock64(); sacc[0] += u1 - u0; u0 = u1;
      tc_fence_after();
      float sum;
      if (half == 0) {
        sum = softmax_half<0, kChunks0, kEarly0>(trow, S, split, c_scale, bars->red_max, 0, row, kPColPLo, &bars->p_part, lane);
      } else {
        sum = softmax_half<kChunks0, kChunks1, kEarly1>(trow, S, split, c_scale, bars->red_max, 1, row, kPColPLo, &bars->p_part, lane);
      }
      bars->red_sum[half][row] = sum;
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_on_leader(&bars->p_full);
      named_barrier_sync(1, kNumSoftmaxWarps * 32);  // red_sum of both halves visible
      const float inv = 1.0f / (bars->red_sum[0][row] + bars->red_sum[1][row]);
      u1 = clock64(); sacc[1] += u1 - u0; u0 = u1;
      if (w_prev >= 0) write_output(w_prev, ph ^ 1, inv_prev);
      u1 = clock64(); sacc[3] += u1 - u0;
      w_prev = w;
      inv_prev = inv;
    }
    if (w_prev >= 0) {
      const uint32_t last = (it - 1) & 1;
      long long u0 = clock64(), u1;
      mbar_wait(&bars->o_done, last);
      u1 = clock64(); sacc[2] += u1 - u0; u0 = u1;
      tc_fence_after();
      write_output(w_prev, last, inv_prev);
      sacc[3] += clock64() - u0;
    }
    if (p.dbg_cycles && sw == 0 && lane == 0)
      for (int i = 0; i < 4; ++i) p.dbg_cycles[(size_t)cluster_id * 16 + 8 + i] = sacc[i];
    if (lane == 0) tma_store_wait_all();  // bulk stores of the last item complete before the CTA exits
  }

  tc_fence_before();
  cluster_sync_all();  // nobody touches the pair's TMEM / barriers after this point
  if (warp_idx == 1) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, kTmemCols);
  }
}

}  // namespace

cudaError_t configure_attention_kernel() {
  return cudaFuncSetAttribute(attention_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              (int)(1024 + kPairSmemTiles + sizeof(AttnPairBarriers)));
}

cudaError_t launch_attention(const AttnMaps& m, const AttnParams& p, cudaStream_t stream) {
  if (p.seq_len > kKeyPad || p.seq_len < 1 || (p.nsplit != 1 && p.nsplit != 3)) {
    set_last_error("launch_attention: unsupported seq_len=%d nsplit=%d", p.seq_len, p.nsplit);
    return cudaErrorInvalidValue;
  }
  static int num_sms = 0;
  if (num_sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
  }
  const int num_items = p.num_heads * p.num_seqs;
  const int clusters = num_items < num_sms / 2 ? num_items : num_sms / 2;
  const size_t smem = 1024 + kPairSmemTiles + sizeof(AttnPairBarriers);
  return launch_kernel(attention_pair_kernel, dim3(2 * clusters), dim3(kThreads), smem, stream, *m.q_hi, *m.q_lo, *m.kh_hi, *m.kh_lo,
                       *m.kv_hi, *m.kv_lo, *m.o_hi, *m.o_lo, p, num_items);
}

}  // namespace cmdi
