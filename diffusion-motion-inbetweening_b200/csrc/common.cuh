// Device-side primitives for the sm_100a kernels of the CondMDI sampling engine.
//
// Everything here is a thin wrapper over one PTX instruction: mbarrier, TMA
// (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld / st / fences) and the
// shared-memory + instruction descriptors the 5th-gen tensor cores consume.
// Descriptor bit layouts follow the PTX ISA "tcgen05 matrix descriptors" tables.
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda.h>
#include <stdio.h>
#include <stdint.h>

namespace cmdi {

// ----------------------------------------------------------------------------------------------
// small helpers
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

// 2^x on the SFU (ex2.approx.ftz: relative error ~2^-22, exp2(-inf) = 0)
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// bf16 split of an fp32 value: v ~= hi + lo with |v - hi - lo| <= 2^-17 |v|.
__device__ __forceinline__ void split_bf16(float v, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(v);
  lo = __float2bfloat16_rn(v - __bfloat162float(hi));
}

__device__ __forceinline__ uint32_t pack_bf16x2(__nv_bfloat16 a, __nv_bfloat16 b) {
  return (uint32_t)__bfloat16_as_ushort(a) | ((uint32_t)__bfloat16_as_ushort(b) << 16);
}

// Split two fp32 values at once: hi_word / lo_word hold {a (low half), b (high half)} as bf16x2.
// One packed cvt.rn.bf16x2.f32 per plane (half the conversion-pipe work of four scalar converts).
__device__ __forceinline__ void split_bf16x2(float a, float b, uint32_t& hi_word, uint32_t& lo_word) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  hi_word = *reinterpret_cast<const uint32_t*>(&h);
  const float ha = __uint_as_float(hi_word << 16), hb = __uint_as_float(hi_word & 0xffff0000u);
  const __nv_bfloat162 l = __floats2bfloat162_rn(a - ha, b - hb);
  lo_word = *reinterpret_cast<const uint32_t*>(&l);
}

// y = (x - mean) * rstd * gamma + beta with a fixed operation order: the LayerNorm kernel and the epilogues that
// re-derive LayerNorm's output as a residual (from its fp32 input and the row statistics) must agree bit for bit.
__device__ __forceinline__ float ln_apply(float x, float mean, float rstd, float g, float b) {
  return __fmaf_rn(__fmul_rn(__fsub_rn(x, mean), rstd), g, b);
}

// ----------------------------------------------------------------------------------------------
// programmatic dependent launch: a kernel launched with programmaticStreamSerializationAllowed may start while its
// predecessor drains; it must not touch global memory before griddep_wait() (no-op for ordinary launches)
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ----------------------------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// make generic-proxy smem writes visible to the async proxy (TMA / UMMA reads of smem)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must surface as a trapped kernel (an error the host sees),
// never as a hung GPU. ~4e9 cycles is seconds; every legitimate wait here is microseconds.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) {
      printf("cmdi: mbarrier timeout block=(%d,%d) thread=%d bar=%u parity=%u\n", blockIdx.x, blockIdx.y,
             threadIdx.x, smem_u32(bar), parity);
      __trap();
    }
  }
}

// ----------------------------------------------------------------------------------------------
// TMA
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
// 2D tiled load: box lands in smem (swizzled as the map says), completes `bytes` on the mbarrier.
// c0 = coordinate along the contiguous (inner) dimension, c1 = row coordinate.
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int32_t c0,
                                            int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

// L2 prefetch of a box (no shared-memory destination, no completion to wait for)
__device__ __forceinline__ void tma_prefetch_2d(const CUtensorMap* map, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"(reinterpret_cast<uint64_t>(map)), "r"(c0),
               "r"(c1)
               : "memory");
}

// 2D tiled store: the (128B-swizzled) smem box is written to global memory; completion is tracked by bulk async-groups.
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t smem_src_addr, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(map)),
               "r"(smem_src_addr), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all committed bulk stores of this thread have finished READING their shared-memory source
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// ... and have completed their global writes
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ----------------------------------------------------------------------------------------------
// tcgen05: TMEM allocation
// ----------------------------------------------------------------------------------------------
// Whole warp executes. ncols: power of two in [32, 512].
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ----------------------------------------------------------------------------------------------
// tcgen05: descriptors
// ----------------------------------------------------------------------------------------------
// Shared-memory matrix descriptor (64 bit):
//   [0,14)  start address >> 4        [16,30) leading-dim byte offset >> 4
//   [32,46) stride-dim byte offset >> 4   [46,48) version = 1 (sm_100)
//   [49,52) base offset = 0 (tiles are 1024 B aligned)   [61,64) swizzle: 2 = 128 B
//
// K-major operand, 128 B swizzle (tile written by a TMA box of 64 bf16 x rows):
//   row r at byte r*128, 16 B chunks XOR-swizzled by (r & 7); 8-row atoms 1024 B apart -> SBO = 1024.
//   LBO is unused for swizzled K-major layouts (set to 1 like CUTLASS does).
// MN-major operand, 128 B swizzle (TMA box of 64 contiguous MN-elements x K rows):
//   K index k at byte k*128 inside a 64-wide MN group -> SBO = 1024 (8 K-rows),
//   next 64-wide MN group LBO bytes further (= rows_in_box * 128).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;  // version
  d |= (uint64_t)2 << 61;  // SWIZZLE_128B
  return d;
}
__device__ __forceinline__ uint64_t make_desc_kmajor_sw128(uint32_t smem_addr) {
  return make_smem_desc(smem_addr, 16, 1024);
}
__device__ __forceinline__ uint64_t make_desc_mnmajor_sw128(uint32_t smem_addr, uint32_t mn_group_stride_bytes) {
  return make_smem_desc(smem_addr, mn_group_stride_bytes, 1024);
}
// advance a descriptor's start address by `bytes` (must keep the result inside the 14-bit field)
__device__ __forceinline__ uint64_t desc_advance(uint64_t desc, uint32_t bytes) { return desc + (uint64_t)(bytes >> 4); }

// Instruction descriptor for kind::f16 with BF16 operands and FP32 accumulation.
//   [4,6) c_format = 1 (F32)   [7,10) a_format = 1 (BF16)   [10,13) b_format = 1 (BF16)
//   [15] a_major (0 = K)   [16] b_major (0 = K, 1 = MN)   [17,23) N >> 3   [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_idesc_bf16(uint32_t M, uint32_t N, uint32_t b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (b_mn_major << 16) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// ----------------------------------------------------------------------------------------------
// tcgen05: MMA issue / commit (single thread)
// ----------------------------------------------------------------------------------------------
// D[tmem] (+)= A[smem] * B[smem]
__device__ __forceinline__ void umma_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]   (A: lane = row, each 32-bit column holds two consecutive K elements)
__device__ __forceinline__ void umma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrives once all tcgen05 ops previously issued by this thread have completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// ----------------------------------------------------------------------------------------------
// tcgen05: TMEM <-> registers (warp-collective; warp w touches lanes 32*(w%4) .. +31)
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// 32 lanes x 16 consecutive 32-bit columns: thread i gets row (lane base + i), v[j] = column j
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
// 32 lanes x 8 consecutive 32-bit columns
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(v[0]),
               "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}

// 32 lanes x 32 consecutive 32-bit columns
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"
      "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
      "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]),
      "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]),
      "r"(v[31])
      : "memory");
}

// TMEM address = (lane << 16) | column
__device__ __forceinline__ uint32_t tmem_addr(uint32_t base, uint32_t lane, uint32_t col) {
  return base + (lane << 16) + col;
}

// ----------------------------------------------------------------------------------------------
// vector global stores / loads
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void st_global_v4(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.global.v4.b32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void st_global_v4f(float* p, float a, float b, float c, float d) {
  asm volatile("st.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

}  // namespace cmdi

// ==============================================================================================
// CTA-pair (cta_group::2) variants: two SMs of one cluster cooperate on one 256-row MMA tile
// ==============================================================================================
namespace cmdi {

// In the shared::cluster window bit 24 of a CTA-local shared address selects the odd CTA of a pair;
// clearing it addresses the same offset in the even ("leader") CTA.
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA load issued by either CTA of the pair; the transaction bytes are counted on the LEADER CTA's mbarrier
__device__ __forceinline__ void tma_load_2d_2sm(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1)
      : "memory");
}
// arrive on the leader CTA's copy of `bar` (works from both CTAs of the pair)
__device__ __forceinline__ void mbar_arrive_on_leader(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPeerBitMask) : "memory");
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_2sm() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem, 256 rows over both CTAs] (+)= A[smem of both CTAs] * B[smem of both CTAs]; issued by the leader only
__device__ __forceinline__ void umma_ss_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// ... with A read from tensor memory (each CTA's lanes hold its 128 rows of A)
__device__ __forceinline__ void umma_ts_2sm(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on `bar` in every CTA of `cta_mask` once the pair's previously issued MMAs have completed
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(cta_mask)
               : "memory");
}

}  // namespace cmdi
