// CTA-pair version of the linear layers: two SMs of a cluster share one 256 x BLOCK_N output tile
// (tcgen05.mma.cta_group::2, M = 256).
//
// Why: with one CTA per tile the operand traffic is 128*64 (A) + BLOCK_N*64 (W) elements per k-block for
// 128 x BLOCK_N x 64 MACs; at B=64 the QKV GEMM then pulls ~460 MB through L2->SM per launch and is bound by
// that (profiles/r01: 15% of tensor peak).  In pair mode each CTA loads its own 128 A rows but only HALF of the
// W tile (the MMA reads the other half from the peer's shared memory), so the same MACs need 1.5x fewer bytes
// from L2, the smem ring is 64 KB/stage (3 stages instead of 2) and W is read from smem once per pair.
//
// Protocol (both CTAs run the same code; rank 0 is the leader):
//   full[s]       lives on the leader: 1 arrival (leader's arrive.expect_tx for BOTH CTAs' bytes) + complete_tx from
//                 the TMA loads of both CTAs (cp.async.bulk.tensor ... cta_group::2 targets the leader's barrier)
//   empty[s]      per CTA, signalled by the leader's tcgen05.commit multicast to both CTAs
//   tmem_full[a]  per CTA, same multicast commit
//   tmem_empty[a] on the leader: epilogue warps of BOTH CTAs arrive on it (remote arrive from the peer)
#include "common.cuh"
#include "gemm_epilogue.cuh"
#include "kernels.h"

namespace cmdi {

namespace {

constexpr int kBlockM = 128;  // per CTA; 256 per pair
constexpr int kBlockK = 64;
constexpr int kUmmaK = 16;
constexpr int kNumEpiWarps = 8;
constexpr int kNumThreads = 64 + kNumEpiWarps * 32;
constexpr int kMaxStages = 8;
constexpr int kSmemLimit = 232448;
constexpr int kABytes = kBlockM * kBlockK * 2;

struct __align__(8) PairBarriers {
  uint64_t full[kMaxStages];
  uint64_t empty[kMaxStages];
  uint64_t full_a[2], empty_a[2];  // TAP_REUSE: the A ring
  uint64_t tmem_full[2];
  uint64_t tmem_empty[2];
  uint32_t tmem_base;
  uint32_t pad;
};

// TAP_REUSE (k-tap convolutions whose taps are consecutive row shifts of the same A columns): the A tile of a channel
// block is loaded ONCE as 128 + (taps - 1) rows (box of kTapRows rows) and every tap's MMAs read it through a descriptor
// whose start address is shifted by `tap` rows (128 B each), against that tap's own W tile: A ring of 2 tiles + W ring of `num_stages` tiles instead of
// `num_stages` (A, W) stages.  For k = 5 that is 33 + 5 x 32 KB of operands per CTA and channel block instead of
// 5 x 64 KB -- the mainloop of these GEMMs sits on the L2->SM operand stream (DESIGN.md 8).
constexpr int kTapRows = 136;                          // 128 + 8: up to 8 further taps (whole swizzle atoms)
constexpr int kATapBytes = kTapRows * kBlockK * 2;     // one plane of an A tile with its tap rows: 17 KB
constexpr int kTapStagesA = 2;

template <int BLOCK_N, bool TAP_REUSE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kNumThreads, 1)
linear2_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
               const __grid_constant__ CUtensorMap map_w_hi, const __grid_constant__ CUtensorMap map_w_lo,
               const __grid_constant__ CUtensorMap map_o_hi, const __grid_constant__ CUtensorMap map_o_lo,
               const __grid_constant__ CUtensorMap map_o_f32,
               const LinearParams p, const int num_stages, const int num_m_pairs, const int num_n_blocks) {
  constexpr int kHalfN = BLOCK_N / 2;               // W rows this CTA loads
  constexpr int kBBytes = kHalfN * kBlockK * 2;
  // double-buffered accumulator: 128 lanes x BLOCK_N fp32 each
  constexpr uint32_t kTmemCols = 2 * BLOCK_N;
  static_assert(BLOCK_N == 128 || BLOCK_N == 256, "BLOCK_N");

  griddep_launch_dependents();
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));

  const int nplanes = (p.nsplit == 3) ? 2 : 1;
  // general: num_stages x {A planes, W planes};  TAP_REUSE: kTapStagesA x {A planes with tap rows}, num_stages x {W planes}
  const uint32_t stage_bytes = TAP_REUSE ? nplanes * kBBytes : nplanes * (kABytes + kBBytes);
  const uint32_t a_tile_bytes = nplanes * kATapBytes;
  uint8_t* ring_a = smem;                                                        // TAP_REUSE only
  uint8_t* ring = TAP_REUSE ? smem + (size_t)kTapStagesA * a_tile_bytes : smem;  // stages (general) / W tiles (TAP_REUSE)
  uint8_t* epi_stage = ring + (size_t)num_stages * stage_bytes;  // kNumEpiWarps x 4 KB store-staging tiles
  PairBarriers* bars = reinterpret_cast<PairBarriers*>(epi_stage + kNumEpiWarps * kEpiStageBytes);

  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = cluster_ctarank();
  const bool leader = cta_rank == 0;
  const int cluster_id = blockIdx.x >> 1;
  const int num_clusters = gridDim.x >> 1;
  const int num_tiles = num_m_pairs * num_n_blocks;
  const int num_k_blocks = (p.K + kBlockK - 1) / kBlockK;
  const int kb_per_tap = p.num_taps > 0 ? p.k_per_tap / kBlockK : num_k_blocks;  // convolution taps: see LinearParams

  if (warp_idx == 0 && lane == 0) {
    tma_prefetch_desc(&map_a_hi);
    tma_prefetch_desc(&map_w_hi);
    for (int s = 0; s < num_stages; ++s) {
      mbar_init(&bars->full[s], 1);
      mbar_init(&bars->empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&bars->tmem_full[s], 1);
      mbar_init(&bars->tmem_empty[s], 2 * kNumEpiWarps);
      mbar_init(&bars->full_a[s], 1);
      mbar_init(&bars->empty_a[s], 1);
    }
    fence_barrier_init();
  }
  if (warp_idx == 1) {
    tmem_alloc_2sm(&bars->tmem_base, kTmemCols);
    tmem_relinquish_2sm();
  }
  tc_fence_before();
  cluster_sync_all();  // barrier inits + TMEM allocation visible to both CTAs
  tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;
  griddep_wait();  // everything above overlapped the previous kernel's tail; global memory is touched from here on

  if (warp_idx == 0) {
    // ===================================== TMA producer (both CTAs) =====================================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      if constexpr (TAP_REUSE) {
        int sa_i = 0;
        uint32_t pa = 0;
        for (int tile = cluster_id; tile < num_tiles; tile += num_clusters) {
          const int m_blk = 2 * (tile / num_n_blocks) + (int)cta_rank;
          const int n_blk = tile % num_n_blocks;
          for (int cb = 0; cb < kb_per_tap; ++cb) {
            // the A rows of all taps of this channel block: rows m_blk * 128 + tap_row[0] .. + 127 + (taps - 1)
            mbar_wait(&bars->empty_a[sa_i], pa ^ 1);
            uint8_t* sa = ring_a + (size_t)sa_i * a_tile_bytes;
            if (leader) mbar_arrive_expect_tx(&bars->full_a[sa_i], 2 * a_tile_bytes);
            tma_load_2d_2sm(sa, &map_a_hi, &bars->full_a[sa_i], p.tap_a_col[0] + cb * kBlockK, m_blk * kBlockM + p.tap_row[0]);
            if (nplanes == 2)
              tma_load_2d_2sm(sa + kATapBytes, &map_a_lo, &bars->full_a[sa_i], p.tap_a_col[0] + cb * kBlockK, m_blk * kBlockM + p.tap_row[0]);
            if (++sa_i == kTapStagesA) { sa_i = 0; pa ^= 1; }
            for (int tap = 0; tap < p.num_taps; ++tap) {
              mbar_wait(&bars->empty[stage], phase ^ 1);
              uint8_t* sb = ring + (size_t)stage * stage_bytes;
              if (leader) mbar_arrive_expect_tx(&bars->full[stage], 2 * stage_bytes);
              const int w_col = p.tap_w_col[tap] + cb * kBlockK;
              tma_load_2d_2sm(sb, &map_w_hi, &bars->full[stage], w_col, n_blk * BLOCK_N + (int)cta_rank * kHalfN);
              if (nplanes == 2)
                tma_load_2d_2sm(sb + kBBytes, &map_w_lo, &bars->full[stage], w_col, n_blk * BLOCK_N + (int)cta_rank * kHalfN);
              if (++stage == num_stages) { stage = 0; phase ^= 1; }
            }
          }
        }
      } else {
      for (int tile = cluster_id; tile < num_tiles; tile += num_clusters) {
        const int m_blk = 2 * (tile / num_n_blocks) + (int)cta_rank;
        const int n_blk = tile % num_n_blocks;
        for (int kb = 0; kb < num_k_blocks; ++kb) {
          mbar_wait(&bars->empty[stage], phase ^ 1);
          uint8_t* sa = smem + (size_t)stage * stage_bytes;
          uint8_t* sb = sa + nplanes * kABytes;
          if (p.debug & 4) {
            if (leader) mbar_arrive(&bars->full[stage]);
            if (++stage == num_stages) { stage = 0; phase ^= 1; }
            continue;
          }
          if (leader) mbar_arrive_expect_tx(&bars->full[stage], 2 * stage_bytes);
          int a_col = kb * kBlockK, w_col = a_col, a_row = m_blk * kBlockM;
          if (p.num_taps > 0) {
            const int tap = kb / kb_per_tap, kc = (kb - tap * kb_per_tap) * kBlockK;
            a_col = p.tap_a_col[tap] + kc; w_col = p.tap_w_col[tap] + kc; a_row += p.tap_row[tap];
          }
          tma_load_2d_2sm(sa, &map_a_hi, &bars->full[stage], a_col, a_row);
          tma_load_2d_2sm(sb, &map_w_hi, &bars->full[stage], w_col, n_blk * BLOCK_N + (int)cta_rank * kHalfN);
          if (nplanes == 2) {
            tma_load_2d_2sm(sa + kABytes, &map_a_lo, &bars->full[stage], a_col, a_row);
            tma_load_2d_2sm(sb + kBBytes, &map_w_lo, &bars->full[stage], w_col, n_blk * BLOCK_N + (int)cta_rank * kHalfN);
          }
          if (++stage == num_stages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
      }
    }
    __syncwarp();
  } else if (warp_idx == 1) {
    // ====================================== MMA issuer (leader CTA only) ======================================
    if (leader && lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(2 * kBlockM, BLOCK_N, 0);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      int sa_i = 0;      // TAP_REUSE: A ring position / parity
      uint32_t pa = 0;
      long long t_wait_empty = 0, t_wait_full = 0, t_begin = clock64();
      for (int tile = cluster_id; tile < num_tiles; tile += num_clusters) {
        long long c0 = clock64();
        mbar_wait(&bars->tmem_empty[acc], acc_phase ^ 1);
        t_wait_empty += clock64() - c0;
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
        if constexpr (TAP_REUSE) {
          uint32_t accum = 0;
          for (int cb = 0; cb < kb_per_tap; ++cb) {
            c0 = clock64();
            mbar_wait(&bars->full_a[sa_i], pa);
            t_wait_full += clock64() - c0;
            const uint32_t sa = smem_u32(ring_a + (size_t)sa_i * a_tile_bytes);
            for (int tap = 0; tap < p.num_taps; ++tap) {
              c0 = clock64();
              mbar_wait(&bars->full[stage], phase);
              t_wait_full += clock64() - c0;
              tc_fence_after();
              const uint32_t sb = smem_u32(ring + (size_t)stage * stage_bytes);
              // A rows shifted by `tap`: start address + tap * 128 B.  The 128-byte swizzle is a function of the absolute
              // shared-memory address (bits 7-9 into bits 4-6) for TMA and MMA alike, so a row-shifted view needs no
              // descriptor base offset (measured: with base offset = tap the results are wrong).
              const uint64_t da_hi = make_desc_kmajor_sw128(sa + tap * 128);
              const uint64_t db_hi = make_desc_kmajor_sw128(sb);
              if (nplanes == 2) {
                const uint64_t da_lo = make_desc_kmajor_sw128(sa + kATapBytes + tap * 128);
                const uint64_t db_lo = make_desc_kmajor_sw128(sb + kBBytes);
#pragma unroll
                for (int k = 0; k < kBlockK / kUmmaK; ++k) {
                  umma_ss_2sm(d_tmem, desc_advance(da_lo, k * kUmmaK * 2), desc_advance(db_hi, k * kUmmaK * 2), idesc, accum);
                  accum = 1;
                }
#pragma unroll
                for (int k = 0; k < kBlockK / kUmmaK; ++k)
                  umma_ss_2sm(d_tmem, desc_advance(da_hi, k * kUmmaK * 2), desc_advance(db_lo, k * kUmmaK * 2), idesc, 1u);
#pragma unroll
                for (int k = 0; k < kBlockK / kUmmaK; ++k)
                  umma_ss_2sm(d_tmem, desc_advance(da_hi, k * kUmmaK * 2), desc_advance(db_hi, k * kUmmaK * 2), idesc, 1u);
              } else {
#pragma unroll
                for (int k = 0; k < kBlockK / kUmmaK; ++k) {
                  umma_ss_2sm(d_tmem, desc_advance(da_hi, k * kUmmaK * 2), desc_advance(db_hi, k * kUmmaK * 2), idesc, accum);
                  accum = 1;
                }
              }
              umma_commit_2sm(&bars->empty[stage], 0x3);
              if (++stage == num_stages) { stage = 0; phase ^= 1; }
            }
            umma_commit_2sm(&bars->empty_a[sa_i], 0x3);  // all taps of this channel block have read the A tile
            if (++sa_i == kTapStagesA) { sa_i = 0; pa ^= 1; }
          }
        } else {
        for (int kb = 0; kb < num_k_blocks; ++kb) {
          c0 = clock64();
          mbar_wait(&bars->full[stage], phase);
          t_wait_full += clock64() - c0;
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + (size_t)stage * stage_bytes);
          const uint32_t sb = sa + nplanes * kABytes;
          const uint64_t da_hi = make_desc_kmajor_sw128(sa);
          const uint64_t db_hi = make_desc_kmajor_sw128(sb);
          if (p.debug & 2) {
            // no MMAs: only the pipeline bookkeeping
          } else if (nplanes == 2) {
            const uint64_t da_lo = make_desc_kmajor_sw128(sa + kABytes);
            const uint64_t db_lo = make_desc_kmajor_sw128(sb + kBBytes);
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
          umma_commit_2sm(&bars->empty[stage], 0x3);  // frees the slot in BOTH CTAs
          if (++stage == num_stages) {
            stage = 0;
            phase ^= 1;
          }
        }
        }
        umma_commit_2sm(&bars->tmem_full[acc], 0x3);  // both CTAs' epilogues may read their half of the tile
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
      if (p.dbg_cycles) {
        long long* d = p.dbg_cycles + (size_t)blockIdx.x * 16;
        d[0] = clock64() - t_begin; d[1] = t_wait_empty; d[2] = t_wait_full;
      }
    }
    __syncwarp();
  } else {
    // ======================================= epilogue (both CTAs, own 128 rows) =======================================
    const int epi = warp_idx - 2;
    const int lane_group = warp_idx & 3;
    const int col_part = epi >> 2;
    const uint32_t epi_stage_addr = smem_u32(epi_stage + epi * kEpiStageBytes);
    const EpiStoreMaps epi_maps{&map_o_hi, &map_o_lo, &map_o_f32};
    int acc = 0;
    uint32_t acc_phase = 0;
    long long t_wait = 0, t_work = 0, t_arrive = 0, t_begin = clock64();
    for (int tile = cluster_id; tile < num_tiles; tile += num_clusters) {
      const int m_blk = 2 * (tile / num_n_blocks) + (int)cta_rank;
      const int n_blk = tile % num_n_blocks;
      long long c0 = clock64();
      mbar_wait(&bars->tmem_full[acc], acc_phase);
      long long c1 = clock64();
      tc_fence_after();
      epilogue_tile<BLOCK_N>(p, epi_maps, tmem_base, (uint32_t)(acc * BLOCK_N), m_blk, n_blk, lane_group, col_part, lane, epi_stage_addr);
      long long c2 = clock64();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_on_leader(&bars->tmem_empty[acc]);
      long long c3 = clock64();
      t_wait += c1 - c0; t_work += c2 - c1; t_arrive += c3 - c2;
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    if (p.dbg_cycles && epi == 0 && lane == 0) {
      long long* d = p.dbg_cycles + (size_t)blockIdx.x * 16;
      d[4] = clock64() - t_begin; d[5] = t_wait; d[6] = t_work; d[7] = t_arrive;
    }
    if (p.tma_store && lane == 0) tma_store_wait_read();
  }

  tc_fence_before();
  cluster_sync_all();  // nobody touches the pair's TMEM / barriers after this point
  if (warp_idx == 1) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, kTmemCols);
  }
}

template <int BLOCK_N>
cudaError_t launch_impl2(const CUtensorMap& a_hi, const CUtensorMap& a_lo, const CUtensorMap& w_hi, const CUtensorMap& w_lo,
                         const LinearParams& p_in, int num_sms, cudaStream_t stream, const LinearStoreMaps* st) {
  LinearParams p = p_in;
  p.tma_store = 0;
  CUtensorMap o_hi = a_hi, o_lo = a_hi, o_f32 = a_hi;  // placeholders when the STG epilogue is used
  if (st && (st->hi || st->f32) && p.rowmap == ROWMAP_IDENTITY && p.dup_row_offset == 0 &&
      (!p.out_hi || (st->hi && (p.nsplit_out != 3 || st->lo))) && (!p.out_f32 || st->f32)) {
    p.tma_store = 1;
    if (st->hi) o_hi = *st->hi;
    if (st->lo) o_lo = *st->lo;
    if (st->f32) o_f32 = *st->f32;
  }
  constexpr int kBBytes = (BLOCK_N / 2) * kBlockK * 2;
  const int nplanes = (p.nsplit == 3) ? 2 : 1;
  const int num_m_pairs = (p.M + 2 * kBlockM - 1) / (2 * kBlockM);
  const int num_n_blocks = (p.N + BLOCK_N - 1) / BLOCK_N;
  const int num_tiles = num_m_pairs * num_n_blocks;
  int clusters = num_sms / 2;
  if (clusters > num_tiles) clusters = num_tiles;
  const int fixed = 1024 + kNumEpiWarps * kEpiStageBytes + (int)sizeof(PairBarriers);
  // convolution whose taps are consecutive row shifts of the same A columns, and an A map with a kTapRows-row box
  bool reuse = st && st->a_tap_hi && (nplanes == 1 || st->a_tap_lo) && p.num_taps >= 2 && p.num_taps <= kTapRows - kBlockM + 1;
  for (int t = 1; reuse && t < p.num_taps; ++t)
    reuse = p.tap_a_col[t] == p.tap_a_col[0] && p.tap_row[t] == p.tap_row[0] + t;
  if (reuse) {
    const int w_bytes = nplanes * kBBytes, a_bytes = kTapStagesA * nplanes * kATapBytes;
    int num_stages = (kSmemLimit - fixed - a_bytes) / w_bytes;
    if (num_stages > 4) num_stages = 4;  // beyond ~200 KB the L1 left for the epilogue costs more than the depth buys
    const size_t smem = (size_t)fixed + a_bytes + (size_t)num_stages * w_bytes;
    return launch_kernel(linear2_kernel<BLOCK_N, true>, dim3(2 * clusters), dim3(kNumThreads), smem, stream, *st->a_tap_hi,
                         nplanes == 2 ? *st->a_tap_lo : *st->a_tap_hi, w_hi, w_lo, o_hi, o_lo, o_f32, p, num_stages, num_m_pairs, num_n_blocks);
  }
  const int stage_bytes = nplanes * (kABytes + kBBytes);
  int num_stages = (kSmemLimit - fixed) / stage_bytes;
  if (num_stages > kMaxStages) num_stages = kMaxStages;
  const size_t smem = (size_t)fixed + (size_t)num_stages * stage_bytes;
  return launch_kernel(linear2_kernel<BLOCK_N, false>, dim3(2 * clusters), dim3(kNumThreads), smem, stream, a_hi, a_lo, w_hi, w_lo,
                       o_hi, o_lo, o_f32, p, num_stages, num_m_pairs, num_n_blocks);
}

}  // namespace

cudaError_t configure_linear2_kernels() {
  cudaError_t e = cudaSuccess;
  auto set = [&](auto kernel) {
    if (e == cudaSuccess) e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit);
  };
  set(linear2_kernel<128, false>); set(linear2_kernel<256, false>);
  set(linear2_kernel<128, true>); set(linear2_kernel<256, true>);
  return e;
}

// Tensor maps: A box {64, 128}; W box {64, block_n / 2}.
cudaError_t launch_linear_pair(const CUtensorMap& a_hi, const CUtensorMap& a_lo, const CUtensorMap& w_hi, const CUtensorMap& w_lo,
                               const LinearParams& p, int block_n, int num_sms, cudaStream_t stream,
                               const LinearStoreMaps* st) {
  if (p.N % 8 != 0 || (p.nsplit != 1 && p.nsplit != 3)) {
    set_last_error("launch_linear_pair: N must be a multiple of 8 and nsplit 1 or 3 (N=%d nsplit=%d)", p.N, p.nsplit);
    return cudaErrorInvalidValue;
  }
  if (block_n == 256) return launch_impl2<256>(a_hi, a_lo, w_hi, w_lo, p, num_sms, stream, st);
  if (block_n == 128) return launch_impl2<128>(a_hi, a_lo, w_hi, w_lo, p, num_sms, stream, st);
  set_last_error("launch_linear_pair: unsupported block_n %d", block_n);
  return cudaErrorInvalidValue;
}

}  // namespace cmdi
