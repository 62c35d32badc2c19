// lz_tc.cuh -- PTX wrappers for the Blackwell tensor path (tcgen05 / TMEM / TMA / mbarrier / clusters) shared by the
// fused-trunk kernel (lz_trunk.cu) and the per-layer convolution kernels (lz_conv.cu).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>

namespace lzb {
namespace tc {

constexpr uint64_t kWatchdogCycles = 4000000000ull;       // ~2 s: a lost arrival traps instead of hanging the GPU

// ---- PTX wrappers -------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t mapa_rank(uint32_t addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// Relaxed on purpose: this arrive only hands a TMEM accumulator back (ordered by tcgen05.fence::before_thread_sync);
// a .release here is a MEMBAR.GPU that waits for the thread's outstanding global stores (~2,000 cycles per tile).
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_bar) {
    asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    return done;
}
static __device__ __noinline__ void mbar_wait_slow(uint32_t bar, uint32_t parity) {
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if ((uint64_t)(clock64() - t0) > kWatchdogCycles) {
            printf("lz_tc: mbarrier wait timed out (block %d thread %d bar 0x%x parity %u)\n", (int)blockIdx.x,
                   (int)threadIdx.x, bar, parity);
            __trap();
        }
    }
}
// fast path: one try_wait (which itself suspends the thread for a while); the watchdog only starts after it fails
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    if (!mbar_try_wait(bar, parity)) mbar_wait_slow(bar, parity);
}
// One lane of the (converged) warp; the compiler then knows the guarded region runs single-threaded and keeps the
// tcgen05 / TMA operands in uniform registers (a plain `lane == 0` test makes it wrap every UTCHMMA / UTMALDG in a
// divergence "waterfall" loop: ~80 cycles per instruction instead of ~10).
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
constexpr uint64_t kL2Default = 0x1000000000000000ull;   // the default L2 cache-hint descriptor

__device__ __forceinline__ void tma_tile2d_2sm(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "l"(kL2Default)
        : "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (rows of 128 B, 8-row groups 1024 B apart).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// kind::f16 instruction descriptor: D = f32, A = B = bf16, both K-major, N = 128, M = 256 (cta_group::2).
constexpr uint32_t kInstrDesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(128 >> 3) << 17) | ((256u >> 4) << 24);   // N = 128

__device__ __forceinline__ void umma_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(kInstrDesc), "r"(accumulate)
        : "memory");
}
// all MMAs issued so far by this thread -> one arrival on `bar` in every CTA of `mask` when they complete
__device__ __forceinline__ void umma_commit_2sm(uint32_t bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"(mask) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&h);
}


// 4-D tiled load (used for the padded board copies: box = 64 ch x 6 x 7 x 3 boards, zeros outside the tensor)
__device__ __forceinline__ void tma_tile4d_2sm(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c, int w, int h, int n) {
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4, %5, %6}], [%2], %7;"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c), "r"(w), "r"(h), "r"(n), "l"(kL2Default)
        : "memory");
}
// Arrive on a barrier in another CTA of the cluster with the default semantics (release at CTA scope: MEMBAR.ALL.CTA,
// i.e. this warp's shared-memory stores have been performed, then the arrive leaves the SM).  An arrive with
// `.release.cluster` would compile to MEMBAR.ALL.GPU + ERRBAR + CGAERRBAR (~1,000 cycles per use, measured in the trunk
// kernel).  This is the form CUTLASS's ClusterBarrier::arrive(cta_id) uses for every cross-CTA pipeline hand-off.
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_bar) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
          "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]),
          "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]),
          "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

}  // namespace tc
}  // namespace lzb
