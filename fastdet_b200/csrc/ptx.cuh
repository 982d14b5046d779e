// ptx.cuh — thin inline-PTX wrappers for the sm_100a features the conv kernels use:
// mbarrier, TMA (tiled + im2col), tcgen05 (alloc / mma / commit / ld) and the fences between
// the generic, async and tensor-core proxies.  Nothing here is generic CUDA; this file only
// compiles for compute_100a.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace fd {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// 16-byte read-only load that does not allocate in L1 (streamed once: residual tiles)
__device__ __forceinline__ uint4 ld_nc_v4(const uint4* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

// 16-byte load that bypasses L1 (data written by other CTAs of the same launch: split-K partial sums)
__device__ __forceinline__ float4 ld_cg_f4(const float* p) {
    float4 r;
    asm volatile("ld.global.cg.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p) : "memory");
    return r;
}
// 32-byte read-only load (one full L2 sector per lane), no L1 allocation
struct U32x8 { uint32_t v[8]; };
__device__ __forceinline__ U32x8 ld_nc_v8(const void* p) {
    U32x8 r;
    asm volatile("ld.global.nc.L1::no_allocate.v8.u32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]), "=r"(r.v[6]), "=r"(r.v[7])
                 : "l"(p));
    return r;
}

// ---------------------------------------------------------------- programmatic dependent launch
// wait: returns once every grid this launch depends on has completed and its writes are visible (no-op for a
// launch without the programmatic-serialisation attribute).  launch_dependents: lets the next kernel in the
// stream start its prologue (barrier init, TMEM allocation, weight prefetch) on SMs as they drain.
__device__ __forceinline__ void grid_dep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void grid_dep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug must surface as a launch failure (trap), never as a hung GPU.
#ifndef FD_MBAR_TIMEOUT_CYCLES
#define FD_MBAR_TIMEOUT_CYCLES 4000000000LL  // ~2 s at 1.9 GHz
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > FD_MBAR_TIMEOUT_CYCLES) __trap();
    }
}

// shared-space stores by 32-bit shared address (a generic pointer into shared memory compiles to generic ST.E)
__device__ __forceinline__ void st_shared_v2(uint32_t addr, uint32_t x, uint32_t y) {
    asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void st_shared_v2_if(uint32_t addr, uint32_t x, uint32_t y, bool pred) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %3, 0;\n\t@q st.shared.v2.b32 [%0], {%1, %2};\n\t}" ::"r"(addr), "r"(x), "r"(y), "r"(static_cast<uint32_t>(pred)) : "memory");
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ void st_shared_v4_if(uint32_t addr, uint32_t x, uint32_t y, uint32_t z, uint32_t w, bool pred) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %5, 0;\n\t@q st.shared.v4.b32 [%0], {%1, %2, %3, %4};\n\t}" ::"r"(addr), "r"(x), "r"(y), "r"(z), "r"(w), "r"(static_cast<uint32_t>(pred)) : "memory");
}

__device__ __forceinline__ uint4 ld_shared_v4(uint32_t addr) {
    uint4 r;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr) : "memory");
    return r;
}

// 16-byte asynchronous copy global -> shared (LDGSTS), L1-allocating; src_bytes = 0 writes zeros (padding)
__device__ __forceinline__ void cp_async_16(uint32_t dst, const void* src, uint32_t src_bytes) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
// arrive on `bar` once every cp.async this thread has issued so far has landed (the arrival is one of the barrier's
// expected count: initialise the barrier with the number of threads that execute this)
__device__ __forceinline__ void cp_async_arrive_noinc(uint64_t* bar) {
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// Variants taking raw shared-space addresses (no generic->shared conversion in single-thread hot loops).
__device__ __forceinline__ bool mbar_try_wait_addr(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait_addr(uint32_t bar, uint32_t parity) {
    if (mbar_try_wait_addr(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait_addr(bar, parity)) {
        if (clock64() - t0 > FD_MBAR_TIMEOUT_CYCLES) __trap();
    }
}
__device__ __forceinline__ void mbar_arrive_expect_tx_addr(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}

// true in exactly one lane of a fully active warp
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}

// ---------------------------------------------------------------- clusters / CTA pairs
// In the shared::cluster window of a CTA pair, bit 24 of a shared address selects the CTA; clearing it addresses
// the same offset in the pair's leader (even) CTA.
static constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on an mbarrier given by a shared::cluster address (own CTA or the pair's leader)
__device__ __forceinline__ void mbar_arrive_cluster_addr(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bar) : "memory");
}

// ---------------------------------------------------------------- TMA
// CTA-pair loads: data lands in the issuing CTA's shared memory, the transaction bytes on `bar`, which may be the
// leader CTA's barrier.
__device__ __forceinline__ void tma2_load_2d_addr(uint32_t dst, uint64_t map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
        "l"(map), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
// CTA-pair load multicast to the CTAs in `cta_mask` (cluster ranks): the box lands at the same shared-memory offset in
// every destination CTA and its bytes are counted on the barrier at `bar`'s offset in each destination's pair leader.
__device__ __forceinline__ void tma2_load_2d_mcast_addr(uint32_t dst, uint64_t map, uint32_t bar, int c0, int c1, uint16_t cta_mask) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster"
        " [%0], [%1, {%4, %5}], [%2], %3;" ::"r"(dst),
        "l"(map), "r"(bar), "h"(cta_mask), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma2_load_im2col_4d_addr(uint32_t dst, uint64_t map, uint32_t bar, int c, int w, int h,
                                                         int n, uint16_t ow, uint16_t oh) {
    asm volatile(
        "cp.async.bulk.tensor.4d.im2col.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6}], [%2], {%7, %8};" ::"r"(dst),
        "l"(map), "r"(bar), "r"(c), "r"(w), "r"(h), "r"(n), "h"(ow), "h"(oh)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d_addr(uint32_t dst, uint64_t map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::
            "r"(dst),
        "l"(map), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_im2col_4d_addr(uint32_t dst, uint64_t map, uint32_t bar, int c, int w, int h,
                                                        int n, uint16_t ow, uint16_t oh) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6}], [%2], {%7, %8};" ::"r"(dst),
        "l"(map), "r"(bar), "r"(c), "r"(w), "r"(h), "r"(n), "h"(ow), "h"(oh)
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2D tiled load: box lands in smem (swizzled as the map says), completes tx bytes on `bar`.
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::
            "r"(smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
// 4D im2col load over an NHWC tensor (dims C,W,H,N): `pixelsPerColumn` output pixels starting at
// base pixel (w,h,n), filter-tap offset (ow,oh), `channelsPerPixel` channels starting at c.
__device__ __forceinline__ void tma_load_im2col_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c, int w,
                                                   int h, int n, uint16_t ow, uint16_t oh) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6}], [%2], {%7, %8};" ::"r"(smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c), "r"(w), "r"(h), "r"(n), "h"(ow), "h"(oh)
        : "memory");
}
// 2D tiled store smem -> global (bulk async group).
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(m)),
                 "r"(smem_u32(src)), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, const void* src, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(m)),
                 "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, const void* src, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(m)),
                 "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ---------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
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

// D[tmem] (+)= A[smem desc] * B[smem desc], bf16 x bf16 -> fp32, one CTA.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Arrive on `bar` once every tcgen05.mma issued so far by this thread has retired.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
// CTA-pair variants (cta_group::2): allocation is issued by the same warp of both CTAs; the MMA is issued by the
// leader and spans both SMs; commit multicasts its arrive to the barrier at the same offset in the masked CTAs.
__device__ __forceinline__ void tmem_alloc2(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
                 "r"(ncols)
                 : "memory");
}
__device__ __forceinline__ void tmem_relinquish2() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma2_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                           uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma2_commit_mcast_addr(uint32_t bar, uint16_t cta_mask) {
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
        "h"(cta_mask)
        : "memory");
}
__device__ __forceinline__ void umma_commit_addr(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// Warp-collective: 32 lanes x 32 consecutive fp32 columns; lane i gets row (lane_base + i).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, "
        "%15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor for a K-major bf16 operand tile whose rows are one swizzle
// span wide (128 B for SWIZZLE_128B, 64 B for SWIZZLE_64B): 8-row groups are `sbo_bytes` apart.
//   bits [0,14)  start address >> 4        bits [16,30) leading byte offset >> 4 (unused here: 1)
//   bits [32,46) stride byte offset >> 4   bits [46,48) version = 1 (sm_100)
//   bits [61,64) layout: 2 = SWIZZLE_128B, 4 = SWIZZLE_64B
__device__ __forceinline__ uint64_t make_kmajor_desc(uint32_t smem_addr, uint32_t sbo_bytes, uint32_t layout_type) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF);
    d |= static_cast<uint64_t>(1) << 16;
    d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(layout_type & 7) << 61;
    return d;
}
// Instruction descriptor: bf16 A/B (K-major both), fp32 accumulate, M = 128, N = n.
__host__ __device__ constexpr uint32_t make_idesc_bf16_f32(int m, int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(n >> 3) << 17) |
           (static_cast<uint32_t>(m >> 4) << 24);
}

}  // namespace ptx
}  // namespace fd
