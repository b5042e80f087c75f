// dahitra_b200 — inline-PTX helpers shared by the tcgen05 kernels (sm_100a): mbarrier, TMA, UMMA descriptors,
// tcgen05.mma / commit / ld / st, TMEM allocation.
#pragma once
#include "common.cuh"
#include <cuda.h>
#include <cstdio>

// conv_tc2.cu: fp32 tiled tensor map through the driver entry point (no -lcuda); strides in bytes for dims 1..rank-1
int dh_encode_tiled_f32(CUtensorMap* out, const void* ptr, int rank, const unsigned long long* dims,
                        const unsigned long long* strides, const unsigned* box, bool swizzle128);
int dh_encode_tiled_f32_sw(CUtensorMap* out, const void* ptr, int rank, const unsigned long long* dims,
                           const unsigned long long* strides, const unsigned* box, int swizzle_bytes);
int dh_encode_tiled_f16_sw(CUtensorMap* out, const void* ptr, int rank, const unsigned long long* dims,     // FP16 elements
                           const unsigned long long* strides, const unsigned* box, int swizzle_bytes);

namespace dhtc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// programmatic dependent launch (no-ops when the launch does not carry the attribute): everything above `pdl_wait` overlaps
// the tail of the previous launch in the stream; its results are visible after it
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// mbarrier wait.  Release builds wait for as long as it takes (no trap, no printf on the hot path).  A debug build
// (-DDH_MBAR_TIMEOUT, `DAHITRA_DEBUG_BUILD=1` for _lib.build) bounds the wait: a pipeline that cannot make progress (bad
// tensor map, lost arrive) then traps after a few seconds instead of hanging, and the launch reports
// cudaErrorLaunchFailure to the caller.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
#ifdef DH_MBAR_TIMEOUT
  uint32_t spins = 0;
#endif
  do {
    // the suspend-time hint (ns) lets the thread sleep inside try_wait instead of burning issue slots in this loop
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(bar), "r"(parity), "r"(10000u) : "memory");
#ifdef DH_MBAR_TIMEOUT
    if (!done && ++spins > (1u << 19)) {
      printf("[mbar timeout] block %d thread %d bar smem+0x%x parity %u\n", blockIdx.x, threadIdx.x, bar, parity);
      __trap();
    }
#endif
  } while (!done);
}
// ---- CTA-pair (cta_group::2) helpers: cluster rank / sync, remote mbarrier arrive, TMA signalling the leader's barrier
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `smem_addr` (a shared::cta address of this CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_local(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_bar) {       // release at cluster scope
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}
// wait on a LOCAL barrier whose arrivals may come from the peer CTA (acquire at cluster scope)
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
  uint32_t done;
#ifdef DH_MBAR_TIMEOUT
  uint32_t spins = 0;
#endif
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(bar), "r"(parity), "r"(10000u) : "memory");
#ifdef DH_MBAR_TIMEOUT
    if (!done && ++spins > (1u << 19)) __trap();
#endif
  } while (!done);
}
// TMA loads issued by either CTA of a pair whose completion bytes are counted on `cluster_bar` (normally the leader's)
__device__ __forceinline__ void tma_load_4d_2sm(uint32_t dst, const CUtensorMap* tm, uint32_t cluster_bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(tm), "r"(cluster_bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst, const CUtensorMap* tm, uint32_t cluster_bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(tm), "r"(cluster_bar), "r"(c0), "r"(c1) : "memory");
}
// nearest TF32-representable value, ties away from zero — what cvt.rna.tf32.f32 returns for finite inputs, in two
// integer instructions (the cvt is emulated with four on sm_100a)
__device__ __forceinline__ float tf32_round(float v) {
  return __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xFFFFE000u);
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
// 1-D bulk copy global -> shared (bytes multiple of 16, both addresses 16-B aligned)
__device__ __forceinline__ void bulk_load_1d(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// generic-proxy smem writes -> visible to the async proxy (TMA / tcgen05.mma operand reads)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major, SWIZZLE_128B operand descriptor: rows of 128 B, 8-row atoms of 1024 B (SBO = 1024), version 1 (sm_100).
// The tile base must be 1024-B aligned; K is advanced by adding (bytes >> 4) to the start-address field.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  return (uint64_t)((smem_addr & 0x3FFFF) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// instruction descriptor, kind::tf32: D = F32 (bit 4), A = B = TF32 (2 at bits 7, 10), both K-major, N>>3 at 17, M>>4 at 24
__host__ __device__ constexpr uint32_t umma_idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// bf16 operands (kind::f16): K-major SWIZZLE_64B tiles with 64-byte rows (32 bf16), 8-row atoms of 512 B, K = 16 per MMA
__device__ __forceinline__ uint64_t umma_desc_sw64(uint32_t smem_addr, uint32_t sbo_bytes) {
  return (uint64_t)((smem_addr & 0x3FFFF) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)4 << 61);
}
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {      // D = F32, A = B = BF16 (1 at bits 7, 10), K-major
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__host__ __device__ constexpr uint32_t umma_idesc_f16(int M, int N) {       // D = F32, A = B = F16 (0 at bits 7, 10), K-major
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// two floats -> packed f16x2, saturating at +-65504 (`lo` lands in the low half), and back
__device__ __forceinline__ uint32_t pack_f16x2_sat(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ float f16_lo(uint32_t p) { float f; asm("{ .reg .b16 l, h; mov.b32 {l, h}, %1; cvt.f32.f16 %0, l; }" : "=f"(f) : "r"(p)); return f; }
__device__ __forceinline__ float f16_hi(uint32_t p) { float f; asm("{ .reg .b16 l, h; mov.b32 {l, h}, %1; cvt.f32.f16 %0, h; }" : "=f"(f) : "r"(p)); return f; }
// two floats -> packed bf16x2 (round to nearest even); `lo` lands in the low half
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// A operand read from tensor memory (lane = row m, column = k; 8 columns per K=8 step), B from shared memory
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// CTA-pair MMA: M = 256 (128 rows from each CTA's A tile at the same smem offset), B = N/2 rows from each CTA; issued by the
// leader CTA only.  The commit arrives on the barrier at the same offset in BOTH CTAs.
__device__ __forceinline__ void umma_tf32_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_bf16_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit_2sm(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t slot_smem_addr, uint32_t ncols) {   // one whole warp in EACH CTA of the pair
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_smem_addr), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t slot_smem_addr, uint32_t ncols) {   // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_smem_addr), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {         // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// warp-wide TMEM -> registers: lane i of the warp reads 32 (or 16) consecutive columns of TMEM lane (base_lane + i)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
        "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]),
        "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]),
        "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// packed fp32 pairs (sm_100: FFMA2 / FADD2 / FMUL2 — two IEEE fp32 operations per issued instruction; the results are the
// same as the scalar instructions', lane by lane)
__device__ __forceinline__ unsigned long long f2_pack(float2 a) { unsigned long long r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a.x), "f"(a.y)); return r; }
__device__ __forceinline__ float2 f2_unpack(unsigned long long r) { float2 d; asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(r)); return d; }
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  unsigned long long d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(f2_pack(a)), "l"(f2_pack(b)), "l"(f2_pack(c))); return f2_unpack(d);
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) { unsigned long long d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(f2_pack(a)), "l"(f2_pack(b))); return f2_unpack(d); }
__device__ __forceinline__ float2 fsub2(float2 a, float2 b) { unsigned long long d; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(f2_pack(a)), "l"(f2_pack(b))); return f2_unpack(d); }
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) { unsigned long long d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(f2_pack(a)), "l"(f2_pack(b))); return f2_unpack(d); }
__device__ __forceinline__ float2 f2_bcast(float s) { return make_float2(s, s); }

// float index of element (row r, column k) inside a K-major SWIZZLE_128B tile of 32-float rows
__host__ __device__ __forceinline__ int sw128_idx(int r, int k) { return r * 32 + ((((k >> 2) ^ (r & 7)) << 2) | (k & 3)); }

}  // namespace dhtc
