// Epilogue shared by the 1-CTA and 2-CTA linear kernels: one 128 x BLOCK_N accumulator tile, TMEM -> registers ->
// bias / positional encoding / residual / GELU -> fp32 and bf16 hi/lo planes in global memory.
//
// Thread mapping: epilogue warp w owns TMEM lanes 32*(w%4).. (thread = output row) and half of the tile's columns,
// processed 64 columns at a time.  A thread therefore holds a ROW fragment, which is the wrong shape for global
// memory: every 32-row x 128-byte block is transposed through a per-warp 4 KB shared-memory staging tile (16-byte
// chunks XOR-swizzled by row & 7: conflict-free both ways) and moved with fully coalesced 16-byte accesses, 4
// complete 128-byte row segments per instruction.
//
// Latency notes from the r01 cycle-counter probe (profiles/r01c_*): the first version spent ~18k cycles per tile
// here (> the 12k-cycle MMA mainloop it should hide under) because (a) the 16 bias loads of a 64-column chunk sat
// behind per-group bounds branches and were exposed one after the other, and (b) each staged row was load ->
// shuffle -> store serially.  Now: the bias of a warp's columns is ONE coalesced load per tile (broadcast by shuffle),
// the row offsets of the 8 rows a lane stores are precomputed per tile, and staging reads are batched ahead of the
// global stores.
#pragma once

#include "common.cuh"
#include "kernels.h"

namespace cmdi {

constexpr int kEpiBlockM = 128;
constexpr int kEpiStageBytes = 32 * 128;  // per epilogue warp

__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }

// nn.Mish: x * tanh(softplus(x)), softplus with PyTorch's threshold 20
__device__ __forceinline__ float mish_f(float x) { return x * tanhf(x > 20.0f ? x : log1pf(expf(x))); }

// d/dx [0.5 x (1 + erf(x / sqrt 2))]
__device__ __forceinline__ float gelu_erf_grad(float x) {
  return 0.5f * (1.0f + erff(x * 0.70710678118654752440f)) + x * 0.3989422804014327f * __expf(-0.5f * x * x);
}

__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint4 ld_shared_v4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}

// The 8 rows (of the warp's 32) that this lane moves in the coalesced phase: row it*4 + lane/8, chunk lane%8.
struct RowSlots {
  int row[8];        // output row index of slot `it` (0 when invalid)
  uint32_t ok;       // bit it: the row is valid
};

// Store a 32-row x 32-word block (thread `lane` holds row `lane` in w[0..31]).  Slot it's row goes to
// dst_base + rows.row[it] * pitch_bytes; the 16-byte chunk c of a row is written if c < valid_chunks.
__device__ __forceinline__ void store_block_coalesced(uint32_t stage, int lane, const uint32_t (&w)[32], char* dst_base,
                                                      const RowSlots& rows, long long pitch_bytes, int valid_chunks,
                                                      int ncopies, long long dup_bytes) {
  __syncwarp();
#pragma unroll
  for (int j = 0; j < 8; ++j)
    st_shared_v4(stage + lane * 128 + ((j ^ (lane & 7)) << 4), w[j * 4], w[j * 4 + 1], w[j * 4 + 2], w[j * 4 + 3]);
  __syncwarp();
  const int c = lane & 7;
  uint4 v[8];
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    const int rr = it * 4 + (lane >> 3);
    v[it] = ld_shared_v4(stage + rr * 128 + ((c ^ (rr & 7)) << 4));
  }
  if (c < valid_chunks) {
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      if ((rows.ok >> it) & 1u) {
        char* d = dst_base + (long long)rows.row[it] * pitch_bytes + c * 16;
        st_global_v4(d, v[it].x, v[it].y, v[it].z, v[it].w);
        if (ncopies == 2) st_global_v4(d + dup_bytes, v[it].x, v[it].y, v[it].z, v[it].w);
      }
    }
  }
}

// Same block, but handed to the TMA: the staging tile already has the 128-byte-swizzle layout a {128 B x 32 rows} box
// expects, so one elected lane issues a bulk tensor store (rows beyond the map's extent are clipped by the TMA).
__device__ __forceinline__ void store_block_tma(uint32_t stage, int lane, const uint32_t (&w)[32], const CUtensorMap* map,
                                                int col, int row) {
  if (lane == 0) tma_store_wait_read();  // the previous store issued from this staging tile has been read out
  __syncwarp();
#pragma unroll
  for (int j = 0; j < 8; ++j)
    st_shared_v4(stage + lane * 128 + ((j ^ (lane & 7)) << 4), w[j * 4], w[j * 4 + 1], w[j * 4 + 2], w[j * 4 + 3]);
  fence_proxy_async_smem();
  __syncwarp();
  if (lane == 0) {
    tma_store_2d(map, stage, col, row);
    tma_store_commit();
  }
}

// 16-byte load that bypasses L1 (ld.global.cg): activation blocks may have been written by another CTA of the SAME
// launch (chained linear layers, gemm_chain.cu), and L1 is not coherent across SMs
__device__ __forceinline__ uint4 ld_global_cg_v4(const void* p) {
  uint4 v;
  asm volatile("ld.global.cg.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
  return v;
}

// Inverse: fetch a 32-row x 128-byte block with coalesced 16-byte loads and hand every thread its own row.
__device__ __forceinline__ void load_block_coalesced(uint32_t stage, int lane, uint32_t (&w)[32], const char* src_base,
                                                     const RowSlots& rows, long long pitch_bytes, int valid_chunks) {
  const int c = lane & 7;
  uint4 v[8];
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    v[it] = make_uint4(0u, 0u, 0u, 0u);
    if (((rows.ok >> it) & 1u) && c < valid_chunks)
      v[it] = ld_global_cg_v4(src_base + (long long)rows.row[it] * pitch_bytes + c * 16);
  }
  __syncwarp();
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    const int rr = it * 4 + (lane >> 3);
    st_shared_v4(stage + rr * 128 + ((c ^ (rr & 7)) << 4), v[it].x, v[it].y, v[it].z, v[it].w);
  }
  __syncwarp();
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const uint4 u = ld_shared_v4(stage + lane * 128 + ((j ^ (lane & 7)) << 4));
    w[j * 4] = u.x; w[j * 4 + 1] = u.y; w[j * 4 + 2] = u.z; w[j * 4 + 3] = u.w;
  }
}

// output row / validity of A-row `a_row` under the linear's row map
__device__ __forceinline__ bool map_row(const LinearParams& p, int a_row, long long& out_row, int& pos) {
  bool valid = a_row < p.M;
  out_row = a_row;
  pos = 0;
  if (p.rowmap == ROWMAP_FRAMES_TO_SEQ) {
    const int b = a_row / p.frames;
    const int l = a_row - b * p.frames;
    out_row = (long long)b * (p.frames + 1) + l + 1;
    pos = l + 1;
  } else if (p.rowmap == ROWMAP_SEQ_TO_FRAMES) {
    const int S = p.frames + 1;
    const int b = a_row / S;
    const int s = a_row - b * S;
    valid = valid && (s > 0);
    out_row = (long long)b * p.frames + (s - 1);
  }
  else if (p.rowmap == ROWMAP_HALO_TO_FRAMES) {
    const int b = a_row / p.row_period;
    const int l = a_row - b * p.row_period - p.row_lo;
    valid = valid && l >= 0 && l < p.frames;
    out_row = (long long)b * p.frames + l;
  }
  if (!valid) out_row = 0;
  return valid;
}

struct EpiStoreMaps {
  const CUtensorMap* hi;
  const CUtensorMap* lo;
  const CUtensorMap* f32;
};

template <int BLOCK_N>
__device__ __forceinline__ void epilogue_tile(const LinearParams& p, const EpiStoreMaps& maps, uint32_t tmem_base, uint32_t acc_col,
                                              int m_blk, int n_blk, int lane_group, int col_part, int lane, uint32_t stage) {
  constexpr int kBlockM = kEpiBlockM;
  // the two column parts of a tile: halves (whole 64-column chunks per warp)
  constexpr int part_cols = BLOCK_N / 2;
  const int col_start = col_part == 0 ? 0 : part_cols;
  const int warp_row0 = m_blk * kBlockM + lane_group * 32;
  RowSlots rows;
  rows.ok = 0;
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    int pos_unused;
    long long r;
    if (map_row(p, warp_row0 + it * 4 + (lane >> 3), r, pos_unused)) rows.ok |= 1u << it;
    rows.row[it] = (int)r;
  }
  RowSlots pe_rows;  // rows of the positional-encoding table for the same 8 slots (frame embed only)
  pe_rows.ok = rows.ok;
  if (p.pos_enc) {
#pragma unroll
    for (int it = 0; it < 8; ++it) pe_rows.row[it] = (warp_row0 + it * 4 + (lane >> 3)) % p.frames + 1;
  }
  const int ncopies = (p.debug & 1) ? 0 : ((p.dup_row_offset > 0) ? 2 : 1);
  // bias of this warp's column range: one coalesced 16-byte load per lane per tile (lane l: 4 columns from 4l),
  // issued before the accumulator is touched; consumers fetch it by shuffle
  float4 bias4 = make_float4(0.f, 0.f, 0.f, 0.f);
  {
    const int nb = n_blk * BLOCK_N + col_start + lane * 4;
    if (p.bias && lane * 4 < part_cols && nb < p.N) bias4 = __ldg(reinterpret_cast<const float4*>(p.bias + nb));
  }

  // residual re-derived from LayerNorm's input: gamma / beta of this warp's columns like the bias, and the
  // (mean, rstd) of the row this thread owns in the blocks load_block_coalesced hands out (row = warp_row0 + lane)
  float4 lng4 = make_float4(0.f, 0.f, 0.f, 0.f), lnb4 = lng4;
  float2 ln_st = make_float2(0.f, 0.f);
  if (p.ln_src) {
    const int nb = n_blk * BLOCK_N + col_start + lane * 4;
    if (lane * 4 < part_cols && nb < p.N) {
      lng4 = __ldg(reinterpret_cast<const float4*>(p.ln_gamma + nb));
      lnb4 = __ldg(reinterpret_cast<const float4*>(p.ln_beta + nb));
    }
    if (warp_row0 + lane < p.M) ln_st = p.ln_stats[warp_row0 + lane];
  }

#pragma unroll 1
  for (int c64 = 0; c64 < part_cols / 64; ++c64) {
    const int col_in_tile = col_start + c64 * 64;
    const int n0 = n_blk * BLOCK_N + col_in_tile;
    if (p.tma_store) {
      // the staging tile is about to be rewritten by ordinary shared-memory stores (residual fetch): the bulk store
      // issued from it earlier must have finished reading it
      if (lane == 0) tma_store_wait_read();
      __syncwarp();
    }
    uint32_t v0[32], v1[32];
    tmem_ld32(tmem_addr(tmem_base, lane_group * 32, acc_col + col_in_tile), v0);
    tmem_ld32(tmem_addr(tmem_base, lane_group * 32, acc_col + col_in_tile + 32), v1);
    if (n0 >= p.N) {  // warp-uniform: nothing to write for this chunk
      tmem_ld_wait();
      continue;
    }
    tmem_ld_wait();
    float f[64];
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      f[j] = __uint_as_float(v0[j]);
      f[32 + j] = __uint_as_float(v1[j]);
    }
    if (p.bias) {
      // lane (c64*16 + g) holds the bias of columns [n0 + 4g, n0 + 4g + 4)
#pragma unroll
      for (int g = 0; g < 16; ++g) {
        const int src = c64 * 16 + g;
        f[g * 4 + 0] += __shfl_sync(0xffffffffu, bias4.x, src);
        f[g * 4 + 1] += __shfl_sync(0xffffffffu, bias4.y, src);
        f[g * 4 + 2] += __shfl_sync(0xffffffffu, bias4.z, src);
        f[g * 4 + 3] += __shfl_sync(0xffffffffu, bias4.w, src);
      }
    }
    if (p.pos_enc) {
      // + pe[pos]: rows of the positional table, fetched coalesced like the residual
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        uint32_t r[32];
        load_block_coalesced(stage, lane, r, reinterpret_cast<const char*>(p.pos_enc + n0 + h * 32), pe_rows,
                             (long long)p.N * 4, (p.N - n0 - h * 32) / 4);
#pragma unroll
        for (int j = 0; j < 32; ++j) f[h * 32 + j] += __uint_as_float(r[j]);
      }
    }
    if (p.residual) {
      // x + sublayer(x): the fp32 residual rows are fetched coalesced, one 32-column block at a time
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        uint32_t r[32];
        load_block_coalesced(stage, lane, r, reinterpret_cast<const char*>(p.residual + n0 + h * 32), rows,
                             (long long)p.ld_res * 4, (p.N - n0 - h * 32) / 4);
#pragma unroll
        for (int j = 0; j < 32; ++j) f[h * 32 + j] += __uint_as_float(r[j]);
      }
    }
    if (p.ln_src) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        uint32_t r[32];
        load_block_coalesced(stage, lane, r, reinterpret_cast<const char*>(p.ln_src + n0 + h * 32), rows,
                             (long long)p.ld_ln * 4, (p.N - n0 - h * 32) / 4);
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          const int src = c64 * 16 + h * 8 + g;  // lane holding gamma / beta of columns [n0 + h*32 + 4g, +4)
          f[h * 32 + g * 4 + 0] += ln_apply(__uint_as_float(r[g * 4 + 0]), ln_st.x, ln_st.y, __shfl_sync(0xffffffffu, lng4.x, src), __shfl_sync(0xffffffffu, lnb4.x, src));
          f[h * 32 + g * 4 + 1] += ln_apply(__uint_as_float(r[g * 4 + 1]), ln_st.x, ln_st.y, __shfl_sync(0xffffffffu, lng4.y, src), __shfl_sync(0xffffffffu, lnb4.y, src));
          f[h * 32 + g * 4 + 2] += ln_apply(__uint_as_float(r[g * 4 + 2]), ln_st.x, ln_st.y, __shfl_sync(0xffffffffu, lng4.z, src), __shfl_sync(0xffffffffu, lnb4.z, src));
          f[h * 32 + g * 4 + 3] += ln_apply(__uint_as_float(r[g * 4 + 3]), ln_st.x, ln_st.y, __shfl_sync(0xffffffffu, lng4.w, src), __shfl_sync(0xffffffffu, lnb4.w, src));
        }
      }
    }
    if (p.grad_aux) {
      // GELU backward: dPre = dH * gelu'(pre), pre stashed by the forward pass
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        uint32_t r[32];
        load_block_coalesced(stage, lane, r, reinterpret_cast<const char*>(p.grad_aux + n0 + h * 32), rows,
                             (long long)p.ld_aux * 4, (p.N - n0 - h * 32) / 4);
#pragma unroll
        for (int j = 0; j < 32; ++j) f[h * 32 + j] *= gelu_erf_grad(__uint_as_float(r[j]));
      }
    }
    if (ncopies == 0) continue;
    if (p.f32_pre && p.out_f32) {
      // stash the pre-activation value (fp32) before the activation is applied
      const long long dup = (long long)p.dup_row_offset * p.ld_f32 * 4;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        uint32_t w[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) w[j] = __float_as_uint(f[h * 32 + j]);
        const int nb = n0 + h * 32;
        if (p.tma_store) {
          if (nb < p.N) store_block_tma(stage, lane, w, maps.f32, nb, warp_row0);
        } else {
          store_block_coalesced(stage, lane, w, reinterpret_cast<char*>(p.out_f32 + nb), rows, (long long)p.ld_f32 * 4,
                                (p.N - nb) / 4, ncopies, dup);
        }
      }
    }
    if (p.act == 1) {
#pragma unroll
      for (int j = 0; j < 64; ++j) f[j] = gelu_erf(f[j]);
    } else if (p.act == 2) {
#pragma unroll
      for (int j = 0; j < 64; ++j) f[j] = f[j] / (1.0f + expf(-f[j]));  // SiLU (TimestepEmbedder, mdm.py:347)
    } else if (p.act == 3) {
#pragma unroll
      for (int j = 0; j < 64; ++j) f[j] = mish_f(f[j]);
    }
    if (p.row_period && p.rowmap == ROWMAP_IDENTITY) {
      // halo rows between sequences: the value computed there is meaningless, the consumer relies on zeros
      const int rr = (warp_row0 + lane) % p.row_period;
      if (rr < p.row_lo || rr >= p.row_hi) {
#pragma unroll
        for (int j = 0; j < 64; ++j) f[j] = 0.f;
      }
    }
    const int oc = n0 + ((p.n_split > 0 && n0 >= p.n_split) ? p.n_gap : 0);  // output column of this chunk
    if (p.tma_store) {
      // identity row map: the staging tile goes out as one bulk tensor store per 32 x 128 B block
      if (p.out_f32 && !p.f32_pre) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          uint32_t w[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) w[j] = __float_as_uint(f[h * 32 + j]);
          if (n0 + h * 32 < p.N) store_block_tma(stage, lane, w, maps.f32, oc + h * 32, warp_row0);
        }
      }
      if (p.out_hi) {
        uint32_t hw[32], lw[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) split_bf16x2(f[2 * j], f[2 * j + 1], hw[j], lw[j]);
        store_block_tma(stage, lane, hw, maps.hi, oc, warp_row0);
        if (p.nsplit_out == 3) store_block_tma(stage, lane, lw, maps.lo, oc, warp_row0);
      }
      continue;
    }
    if (p.out_f32 && !p.f32_pre) {
      // two 32-column fp32 blocks: 128 B per row each
      const long long dup = (long long)p.dup_row_offset * p.ld_f32 * 4;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        uint32_t w[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) w[j] = __float_as_uint(f[h * 32 + j]);
        const int nb = n0 + h * 32;
        // 16-byte chunks (4 floats) still inside N; may be <= 0 or >= 8
        store_block_coalesced(stage, lane, w, reinterpret_cast<char*>(p.out_f32 + nb), rows, (long long)p.ld_f32 * 4,
                              (p.N - nb) / 4, ncopies, dup);
      }
    }
    if (p.out_hi) {
      // one 64-column bf16 block per plane: 128 B per row
      uint32_t hw[32], lw[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) split_bf16x2(f[2 * j], f[2 * j + 1], hw[j], lw[j]);
      const long long dup = (long long)p.dup_row_offset * p.ld_bf * 2;
      const int chunks = (p.N - n0) / 8;  // 16-byte chunks (8 bf16) still inside N
      store_block_coalesced(stage, lane, hw, reinterpret_cast<char*>(p.out_hi + n0), rows, (long long)p.ld_bf * 2, chunks,
                            ncopies, dup);
      if (p.nsplit_out == 3)
        store_block_coalesced(stage, lane, lw, reinterpret_cast<char*>(p.out_lo + n0), rows, (long long)p.ld_bf * 2,
                              chunks, ncopies, dup);
    }
  }
}

}  // namespace cmdi
