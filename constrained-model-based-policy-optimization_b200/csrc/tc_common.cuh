// sm_100a primitives used by the tcgen05 kernels: mbarrier, bulk async copy (TMA engine, UBLKCP),
// tcgen05 alloc / mma / commit / ld, shared-memory matrix descriptors.
//
// Operand layout (both A and B): K-major, 128-byte swizzle.  A "panel" is [rows x 64 elements]
// of a 16-bit type: row r occupies 128 B at  (r/8)*1024 + (r%8)*128 ; inside the row the 16-byte
// chunk c (elements 8c..8c+7) is stored at chunk position c ^ (r%8)  (Swizzle<3,4,3>).  Panels
// are 1024-byte aligned so the swizzle phase equals (r%8).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}

// one lane of a fully converged warp (the same lane every time: tcgen05.commit tracks the MMAs
// issued by the executing thread, so issue and commit must come from one thread)
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}

// ---- mbarrier ------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
// Suspend-time hint of every try_wait (ns): without it a try_wait on an incomplete phase returns after a
// few tens of cycles, and the spin loops of the ~10 waiting warps of a CTA issue as many instructions as
// the warps doing the epilogue arithmetic -- on the same issue ports and the same MIO queues as their
// MUFU / LDS instructions (ncu: 25 M try_wait executions per launch against 0.7 M useful waits).
constexpr uint32_t MBAR_SUSPEND_NS = 20000;
// Bounded spin: a protocol bug must not hang the GPU (a hung box is a lost box).  On timeout the
// kernel traps, which surfaces as a launch failure on the host.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t done = 0;
    // rolled: ptxas unrolls this loop 64x otherwise (2 KB of code per wait site, ~40 KB per kernel)
#pragma unroll 1
    // a try_wait suspends for up to ~9 us (measured: 2^26 spins = 9.6 min): 2^19 spins trap a deadlock
    // after ~4.5 s, three orders of magnitude above any legitimate wait
    for (uint32_t spin = 0; spin < (1u << 18); ++spin) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr), "r"(parity), "r"(MBAR_SUSPEND_NS)
            : "memory");
        if (done) return;
    }
    // No printf here: a device-side call in each of the ~20 inlined wait sites costs the kernel 10 %
    // (caller-saved registers around the call constrain the allocation of the hot loops).  The trap
    // surfaces as a launch failure on the host.
    __trap();
}

// the same on a precomputed shared-window address (the generic -> shared conversion of a pointer costs
// two special-register reads per use in the hot loops)
__device__ __forceinline__ void mbar_arrive_a(uint32_t addr) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(addr) : "memory");
}
__device__ __forceinline__ void mbar_wait_a(uint32_t addr, uint32_t parity) {
    uint32_t done = 0;
#pragma unroll 1
    for (uint32_t spin = 0; spin < (1u << 18); ++spin) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr), "r"(parity), "r"(MBAR_SUSPEND_NS)
            : "memory");
        if (done) return;
    }
    __trap();
}

// ---- async-proxy copy: global -> shared, completion on an mbarrier ------------------------------
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst_smem)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
// the same, MULTICAST to the CTAs of the cluster named by `cta_mask`: the bytes land at the same CTA-relative
// offset in every destination CTA and complete_tx is signalled on the mbarrier at the same offset in each
__device__ __forceinline__ void bulk_g2s_mc(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar, uint16_t cta_mask) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;" ::"r"(
            smem_u32(dst_smem)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar)), "h"(cta_mask)
        : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
// all threads of all CTAs of the cluster
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// generic-proxy writes to smem -> visible to the async proxy (tensor core / TMA reads)
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---- tcgen05 ------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* slot_in_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(slot_in_smem)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, 16-bit operands, fp32 accumulate; issued by ONE thread
__device__ __forceinline__ void mma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on `bar` when every tcgen05 op issued so far by this thread has completed
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                     smem_u32(bar))
                 : "memory");
}
// the same arrive, delivered to the barrier at this CTA-relative offset in every CTA of `cta_mask`
__device__ __forceinline__ void mma_commit_mc(uint64_t* bar, uint16_t cta_mask) {
    asm volatile(
        "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
            smem_u32(bar)),
        "h"(cta_mask)
        : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
          "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
          "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
          "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
          "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
          "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---- descriptors --------------------------------------------------------------------------------
// shared-memory matrix descriptor, K-major, SWIZZLE_128B, 8-row groups 1024 B apart
// (cute::UMMA::SmemDescriptor: start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46), version=1 [46,48),
//  layout_type=2 [61,64))
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t smem_addr) {
    return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) |
           (2ull << 61);
}
// instruction descriptor for kind::f16: fp32 accumulate, A/B both `fmt` (0 = f16, 1 = bf16),
// both K-major, M = 128, N = n  (cute::UMMA::InstrDescriptor)
__host__ __device__ constexpr uint32_t idesc_f16(int fmt, int n) {
    return (1u << 4) | ((uint32_t)fmt << 7) | ((uint32_t)fmt << 10) | ((uint32_t)(n >> 3) << 17) |
           ((uint32_t)(128 >> 4) << 24);
}

// byte offset of 16-byte chunk `c` (elements 8c..8c+7) of row `r` inside a swizzled panel
__host__ __device__ constexpr uint32_t panel_off(int r, int c) {
    return (uint32_t)((r >> 3) * 1024 + (r & 7) * 128 + ((c ^ (r & 7)) << 4));
}

// ---- 16-bit conversion ---------------------------------------------------------------------------
template <int FMT> struct Cvt;
template <> struct Cvt<0> {   // fp16, saturating so a diverged rollout clamps instead of producing inf
    __device__ static uint32_t pack(float a, float b) {
        uint32_t d;
        asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(b), "f"(a));   // d = {hi: b, lo: a}
        return d;
    }
};
template <> struct Cvt<1> {   // bf16
    __device__ static uint32_t pack(float a, float b) {
        __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
        return *reinterpret_cast<uint32_t*>(&h);
    }
};

__device__ __forceinline__ float tanh_approx(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// swish(x) = x*sigmoid(x) = t + t*tanh(t) for a pre-halved argument t = x/2  (one MUFU)
__device__ __forceinline__ float swish_half(float t) { return fmaf(t, tanh_approx(t), t); }

}  // namespace tc
namespace tc {
// D[tmem] (+)= A[tmem] * B[smem]^T : A operand read from tensor memory (lane = row, one 32-bit
// column = two consecutive 16-bit K elements)
__device__ __forceinline__ void mma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                           uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
        "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
}  // namespace tc

namespace tc {
// NT consecutive B tiles ([64 x 64] 16-bit, 8 KB apart) x 4 K-steps of TS-form MMAs into ONE accumulator, issued
// from a single asm statement whose operand addresses are derived by add instructions from the two bases.
// With one C++-level operand per MMA, ptxas materialises every tensor-memory address and descriptor in a
// general register and moves it to a uniform register (IMAD.MOV + R2UR per operand: ~40 per 16 MMAs), which
// made the issuing thread -- not the tensor pipe -- the bound of the layer-1 phase.  Chained adds stay on the
// uniform datapath after one R2UR per base.
#define CMBPO_MMA_TS_STEP(P)                                                             \
    "tcgen05.mma.cta_group::1.kind::f16 [%0], [ta], db, %3, " P ";\n\t"                  \
    "add.u32 ta, ta, 8;\n\tadd.u64 db, db, 2;\n\t"
#define CMBPO_MMA_TS_TILE(P0)                                                            \
    CMBPO_MMA_TS_STEP(P0) CMBPO_MMA_TS_STEP("pt") CMBPO_MMA_TS_STEP("pt") CMBPO_MMA_TS_STEP("pt") \
    "add.u64 db, db, 504;\n\t"
template <int NT>
__device__ __forceinline__ void mma_f16_ts_tiles(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                                 uint32_t accumulate_first) {
    static_assert(NT == 1 || NT == 2 || NT == 4, "tiles per stage");
    if (NT == 4) {
        asm volatile(
            "{\n\t.reg .pred p0, pt;\n\t.reg .b32 ta;\n\t.reg .b64 db;\n\t"
            "setp.ne.b32 p0, %4, 0;\n\tsetp.eq.b32 pt, 0, 0;\n\tmov.b32 ta, %1;\n\tmov.b64 db, %2;\n\t"
            CMBPO_MMA_TS_TILE("p0") CMBPO_MMA_TS_TILE("pt") CMBPO_MMA_TS_TILE("pt") CMBPO_MMA_TS_TILE("pt")
            "}" ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate_first)
            : "memory");
    } else if (NT == 2) {
        asm volatile(
            "{\n\t.reg .pred p0, pt;\n\t.reg .b32 ta;\n\t.reg .b64 db;\n\t"
            "setp.ne.b32 p0, %4, 0;\n\tsetp.eq.b32 pt, 0, 0;\n\tmov.b32 ta, %1;\n\tmov.b64 db, %2;\n\t"
            CMBPO_MMA_TS_TILE("p0") CMBPO_MMA_TS_TILE("pt")
            "}" ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate_first)
            : "memory");
    } else {
        asm volatile(
            "{\n\t.reg .pred p0, pt;\n\t.reg .b32 ta;\n\t.reg .b64 db;\n\t"
            "setp.ne.b32 p0, %4, 0;\n\tsetp.eq.b32 pt, 0, 0;\n\tmov.b32 ta, %1;\n\tmov.b64 db, %2;\n\t"
            CMBPO_MMA_TS_TILE("p0")
            "}" ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate_first)
            : "memory");
    }
}
}  // namespace tc
