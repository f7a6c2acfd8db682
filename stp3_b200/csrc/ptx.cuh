// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld).
#pragma once
#include <cstdint>
#include <cuda.h>  // CUtensorMap (types only; the encode entry point is fetched at run time)

namespace stp3 {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// two fp32 -> packed bf16x2 (round to nearest even): low half = a, high half = b
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}

// 256-bit global accesses (sm_100: LDG.256 / STG.256): one full 32-byte sector per lane and instruction.  32-byte aligned.
__device__ __forceinline__ void ld_global_nc_v8(const void* p, uint32_t (&v)[8]) {
  asm volatile("ld.global.nc.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "l"(p));
}
__device__ __forceinline__ void ld_global_v8(const void* p, uint32_t (&v)[8]) {      // coherent (data written earlier)
  asm volatile("ld.global.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "l"(p)
               : "memory");
}
__device__ __forceinline__ uint4 ld_global_v4(const void* p) {                        // coherent 128-bit load
  uint4 r;
  asm volatile("ld.global.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p) : "memory");
  return r;
}
__device__ __forceinline__ void st_global_v8(void* p, const uint32_t (&v)[8]) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]),
               "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}

__device__ __forceinline__ void st_global_v8f(void* p, const float* v) {             // 8 consecutive floats, 32-byte aligned
  asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]),
               "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
               : "memory");
}

// true in exactly one (elected) lane of a converged warp.  Code guarded by it may use the uniform datapath
// (UTCHMMA / UTMALDG / UTCBAR are uniform instructions): guarding them with `lane == 0` instead makes the compiler
// wrap every one of them in an elect-and-retry loop (~7 SASS instructions per MMA, which throttles N=64 MMAs).
__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .b32 rx;\n\t"
      ".reg .pred px;\n\t"
      "elect.sync rx|px, 0xFFFFFFFF;\n\t"
      "selp.u32 %0, 1, 0, px;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {   // acquire at cluster scope
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAITC_%=:\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONEC_%=;\n\t"
      "bra WAITC_%=;\n\t"
      "DONEC_%=:\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

// ---------------------------------------------------------------- programmatic dependent launch
// launch_dependents: the next kernel of the stream (launched with programmatic stream serialization) may start its
// prologue once every CTA of this grid has passed this point or exited.  wait: blocks until the preceding grid has
// completed and flushed its memory; everything that reads or writes dependent global memory comes after it.  Both
// are no-ops for a kernel launched without the attribute.
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---------------------------------------------------------------- thread-block clusters / CTA pairs
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_expect_tx_cluster(uint32_t cluster_addr, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cluster.b64 _, [%0], %1;" ::"r"(cluster_addr),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                            int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}

// CTA-pair variants: the data lands in the executing CTA's shared memory, the transaction bytes are signalled on an
// mbarrier that may live in the peer CTA (`bar_cluster` is a shared::cluster address, see mapa())
__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* m, uint32_t bar_cluster, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(m), "r"(bar_cluster), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d_pair(void* dst, const CUtensorMap* m, uint32_t bar_cluster, int c0, int c1,
                                                 int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, "
      "%6, %7}], [%2];" ::"r"(smem_u32(dst)),
      "l"(m), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}

// im2col mode (rank-4 (N, H, W, C) tensor map from cuTensorMapEncodeIm2col): pixelsPerColumn consecutive pixels of the
// map's bounding box, starting at (n, h, w) and walking W, then H, then N, each read at (h + off_h, w + off_w);
// pixels outside the tensor are zero-filled.  One pixel = one channelsPerPixel-wide shared-memory row.
__device__ __forceinline__ void tma_load_im2col_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c, int w, int h,
                                                   int n, uint16_t off_w, uint16_t off_h) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
      "[%2], {%7, %8};" ::"r"(smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar)), "r"(c), "r"(w), "r"(h), "r"(n), "h"(off_w), "h"(off_h)
      : "memory");
}
__device__ __forceinline__ void tma_load_im2col_4d_pair(void* dst, const CUtensorMap* m, uint32_t bar_cluster, int c,
                                                        int w, int h, int n, uint16_t off_w, uint16_t off_h) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.im2col.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
      "%4, %5, %6}], [%2], {%7, %8};" ::"r"(smem_u32(dst)),
      "l"(m), "r"(bar_cluster), "r"(c), "r"(w), "r"(h), "r"(n), "h"(off_w), "h"(off_h)
      : "memory");
}

// ---------------------------------------------------------------- tcgen05 / TMEM
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem) {   // one full warp; writes the base address to smem
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {     // same warp that allocated
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
// CTA pair (cta_group::2): warp w of BOTH CTAs executes the alloc / dealloc; the pair gets the same columns in each SM
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* dst_smem) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]^T, bf16 x bf16 -> fp32; issued by ONE thread
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier when all previously issued MMAs of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// CTA pair: D is 256 x N (rows 0..127 in the leader's TMEM, 128..255 in the peer's), A = each CTA's own 128 x K tile,
// B = N/2 x K rows from each CTA (same shared-memory offsets in both).  Issued by ONE thread of the leader CTA.
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on the mbarrier at this shared-memory offset in BOTH CTAs of the pair once the MMAs issued so far completed
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"((uint16_t)3)
      : "memory");
}

// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (lane = TMEM lane of this warp's quarter)
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major operand tile in shared memory, rows of 64 bf16 (128 B) with the 128-byte swizzle TMA writes:
// start address >> 4 | LBO (unused for swizzled K-major, canonical value 1) | SBO = 1024 B between 8-row groups |
// descriptor version 1 (sm_100) | layout type 2 = SWIZZLE_128B
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// kind::f16 instruction descriptor: D=f32, A=B=bf16, both K-major, M x N
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

}  // namespace ptx
}  // namespace stp3
