// tcgen05 / TMEM / mbarrier / bulk-copy building blocks for sm_100a (inline PTX, no CUTLASS).
// Encodings follow the PTX ISA "tcgen05" chapter; field layouts cross-checked against the CuTe headers
// vendored in the image (cute/arch/mma_sm100_desc.hpp: SmemDescriptor, InstrDescriptor).
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

namespace pnb {
namespace umma {

// ---- shared-memory operand layouts (K-major, 16-bit elements) -------------------------------------------------
// An operand tile is [rows][BK] with BK = 32 elements (64 bytes of K per row).  Two layouts are implemented:
//   LAYOUT_NONE  "interleaved" 8x16B core matrices:  byte(r, k) = (r/8)*SBO + (k/8)*LBO + (r%8)*16 + (k%8)*2
//                with LBO = 128, SBO = 512  -> 64 bytes per row on average, no swizzle, conflict-free 16B stores
//   LAYOUT_SW64  64B rows, 16B chunks XOR-swizzled with bits (r/2)%4 (Swizzle<2,4,3>); 8-row group = 512 B
enum { LAYOUT_NONE = 0, LAYOUT_SW64 = 4, LAYOUT_SW128 = 2 };
constexpr int BK = 32;  // K elements per operand block

template <int LAYOUT>
__host__ __device__ __forceinline__ uint32_t tile_offset_bytes(int r, int k) {  // k in [0, BK) (or [0,64) for SW128)
    if (LAYOUT == LAYOUT_NONE) return (uint32_t)((r >> 3) * 512 + (k >> 3) * 128 + (r & 7) * 16 + (k & 7) * 2);
    if (LAYOUT == LAYOUT_SW64) return (uint32_t)(r * 64 + ((((k >> 3) ^ (r >> 1)) & 3) * 16) + (k & 7) * 2);
    return (uint32_t)(r * 128 + ((((k >> 3) ^ r) & 7) * 16) + (k & 7) * 2);  // SW128: 64 k per row
}

// 64-bit shared-memory matrix descriptor (SmemDescriptor): start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46),
// version=1 [46,48), layout type [61,64).
template <int LAYOUT>
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3fff);
    uint32_t lbo, sbo;
    if (LAYOUT == LAYOUT_NONE) { lbo = 128; sbo = 512; }
    else if (LAYOUT == LAYOUT_SW64) { lbo = 16; sbo = 512; }   // LBO unused for swizzled K-major (encode 1)
    else { lbo = 16; sbo = 1024; }
    d |= (uint64_t)((lbo >> 4) & 0x3fff) << 16;
    d |= (uint64_t)((sbo >> 4) & 0x3fff) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)LAYOUT << 61;
    return d;
}
// byte advance of the start address for the k-th UMMA_K(=16 elements) step inside a block
template <int LAYOUT>
__device__ __forceinline__ uint32_t kstep_advance_bytes(int ks) {
    return LAYOUT == LAYOUT_NONE ? (uint32_t)ks * 256u : (uint32_t)ks * 32u;
}

// 32-bit instruction descriptor, kind::f16, BF16 x BF16 -> F32, both operands K-major.
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N) {
    return (1u << 4)                      // c_format = F32
           | (1u << 7)                    // a_format = BF16
           | (1u << 10)                   // b_format = BF16
           | ((uint32_t)(N >> 3) << 17)   // n_dim
           | ((uint32_t)(M >> 4) << 24);  // m_dim
}

// ---- mbarrier ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)   // NO suspend-time hint: ptxas turns a hint into NANOSLEEP(hint) after a miss
        : "memory");
    return ok != 0;
}
// Probe up to four barriers with independent try_wait instructions (their ~100-cycle latencies overlap instead of
// adding up on the single issuing thread); returns true only if all phases have completed.
__device__ __forceinline__ bool mbar_try_wait4(uint64_t* b0, uint32_t p0, uint64_t* b1, uint32_t p1, uint64_t* b2, uint32_t p2,
                                               uint64_t* b3, uint32_t p3) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred q0, q1, q2, q3;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 q0, [%1], %5;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 q1, [%2], %6;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 q2, [%3], %7;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 q3, [%4], %8;\n\t"
        "and.pred q0, q0, q1;\n\tand.pred q2, q2, q3;\n\tand.pred q0, q0, q2;\n\t"
        "selp.u32 %0, 1, 0, q0;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(b0)), "r"(smem_u32(b1)), "r"(smem_u32(b2)), "r"(smem_u32(b3)), "r"(p0), "r"(p1), "r"(p2), "r"(p3)
        : "memory");
    return ok != 0;
}
// two-barrier form of the probe
__device__ __forceinline__ bool mbar_try_wait2(uint64_t* b0, uint32_t p0, uint64_t* b1, uint32_t p1) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred q0, q1;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 q0, [%1], %3;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 q1, [%2], %4;\n\t"
        "and.pred q0, q0, q1;\n\tselp.u32 %0, 1, 0, q0;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(b0)), "r"(smem_u32(b1)), "r"(p0), "r"(p1)
        : "memory");
    return ok != 0;
}
// Warp-uniformity for the issuing warp: every lane of the issuer executes the same code on the same values, but values that come from
// memory (the TMEM base address, the tile count) or from per-lane barrier probes are not PROVABLY uniform, and ptxas then keeps the MMA
// operands in ordinary registers and moves them to uniform registers for every single UTCHMMA (ELECT + ~8 R2UR.BROADCAST + VOTEU each).
// A constant-lane shuffle / a vote makes them uniform by construction: the descriptors then live in uniform registers.
__device__ __forceinline__ uint32_t uni32(uint32_t x) { return __shfl_sync(0xffffffffu, x, 0); }
__device__ __forceinline__ bool uni(bool b) { return __all_sync(0xffffffffu, b) != 0; }
__device__ __forceinline__ uint64_t globaltimer_ns_fwd() {
    uint64_t t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
// Non-blocking probe (test_wait never suspends the thread; try_wait may, up to a hardware time limit).
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ bool mbar_spin_wait(uint64_t* bar, uint32_t parity, int* err_flag, int code) {   // test_wait spin, 2 s bound
    if (mbar_test_wait(bar, parity)) return true;
    const uint64_t t0 = globaltimer_ns_fwd();
    for (;;) {
        if (mbar_test_wait(bar, parity)) return true;
        if (globaltimer_ns_fwd() - t0 > 2000000000ull) break;
    }
    if (err_flag) atomicCAS(err_flag, 0, code);      // the FIRST time-out is the diagnostic one (the others follow from it)
    return false;
}
__device__ __forceinline__ uint64_t globaltimer_ns() {
    uint64_t t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
// Bounded wait (2 s wall clock): a protocol bug must surface as an error flag, never as a hung GPU.
__device__ __forceinline__ bool mbar_wait(uint64_t* bar, uint32_t parity, int* err_flag, int code) {
    if (mbar_try_wait(bar, parity)) return true;
    const uint64_t t0 = globaltimer_ns();
    for (;;) {
        if (mbar_try_wait(bar, parity)) return true;
        if (globaltimer_ns() - t0 > 2000000000ull) break;
    }
    if (err_flag) atomicCAS(err_flag, 0, code);      // the FIRST time-out is the diagnostic one (the others follow from it)
    return false;
}

// ---- 1-D bulk async copy global -> shared (TMA engine, UBLKCP in SASS), completes on an mbarrier -------------------
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- TMEM ---------------------------------------------------------------------------------------------------------
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result) {  // whole warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "n"(NCOLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
}
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {  // whole warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS));
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem], single thread issues.
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]: A is M x K in TMEM, lane = row, each 32-bit column holds two consecutive K elements.
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
        "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// 32 lanes x 8 consecutive columns <- 8 registers per thread
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t* v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(v[0]), "r"(v[1]),
                 "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// ---- lean issue path: the single issuing thread must spend < ~25 instructions per MMA (128-160 cycles each), so
// descriptors are split into a constant high word and a low word that only needs an integer add per k-step.
//   low word  = (smem_addr >> 4) & 0x3fff | (LBO >> 4) << 16        high word = (SBO >> 4) | 1 << 14 | layout << 29
template <int LAYOUT>
__device__ __forceinline__ uint32_t desc_lo(uint32_t smem_addr) {
    return ((smem_addr >> 4) & 0x3fffu) | ((LAYOUT == LAYOUT_NONE ? 128u : 16u) >> 4) << 16;
}
template <int LAYOUT>
__device__ __forceinline__ constexpr uint32_t desc_hi() {
    return ((LAYOUT == LAYOUT_SW128 ? 1024u : 512u) >> 4) | (1u << 14) | ((uint32_t)LAYOUT << 29);
}
template <int LAYOUT>
__device__ __forceinline__ constexpr uint32_t kstep_adv16() { return LAYOUT == LAYOUT_NONE ? 16u : 2u; }   // in 16-byte units
__device__ __forceinline__ void mma_ss2(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                        uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tmov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\tsetp.ne.b32 p, %6, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}" ::"r"(d_tmem),
        "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void mma_ts2(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_lo, uint32_t b_hi, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 db;\n\tmov.b64 db, {%2, %3};\n\tsetp.ne.b32 p, %5, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n\t}" ::"r"(d_tmem),
        "r"(a_tmem), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Warp-uniform issue path: the WHOLE issuer warp executes these (convergent); one elected lane issues.  With warp-uniform
// operands ptxas keeps the descriptors in uniform registers (no R2UR / no uniformising loop around UTCHMMA).
__device__ __forceinline__ void mma_ss2_w(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, pe;\n\t.reg .b64 da, db;\n\telect.sync _|pe, 0xffffffff;\n\t"
        "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\tsetp.ne.b32 p, %6, 0;\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}" ::"r"(d_tmem),
        "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void mma_ts2_w(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_lo, uint32_t b_hi, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, pe;\n\t.reg .b64 db;\n\telect.sync _|pe, 0xffffffff;\n\t"
        "mov.b64 db, {%2, %3};\n\tsetp.ne.b32 p, %5, 0;\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n\t}" ::"r"(d_tmem),
        "r"(a_tmem), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void mma_commit_w(uint64_t* bar) {
    asm volatile(
        "{\n\t.reg .pred pe;\n\telect.sync _|pe, 0xffffffff;\n\t"
        "@pe tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(smem_u32(bar))
        : "memory");
}
// all previously issued MMAs of this thread -> arrive(1) on the mbarrier when complete
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mma2_commit_local_w(uint64_t* bar) {   // cta_group::2 commit, arrive on the issuing CTA's barrier only
    asm volatile(
        "{\n\t.reg .pred pe;\n\telect.sync _|pe, 0xffffffff;\n\t"
        "@pe tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(smem_u32(bar))
        : "memory");
}
// ---- CTA pair (cluster of 2, tcgen05 cta_group::2) ----------------------------------------------------------------
// One tcgen05.mma.cta_group::2 (issued by the rank-0 CTA) computes D[256 x N]: CTA r owns accumulator rows
// 128r..128r+127 in ITS tensor memory, supplies its own 128 A rows and the B rows N/2*r .. N/2*(r+1)-1 from ITS shared
// memory at the descriptor's offset (same offsets in both CTAs).  Halves the B bytes each SM stages and reads.
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same variable in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_cta(const void* local_smem, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(local_smem)), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    // default semantics (.release.cta), as CUTLASS' ClusterBarrier::arrive(cta_id): an explicit .release.cluster compiles to
    // MEMBAR.ALL.GPU + ERRBAR + CGAERRBAR in front of every arrive (measured: it doubles the epilogue time)
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc2(uint32_t* smem_result) {  // the same warp of BOTH CTAs
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "n"(NCOLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::);
}
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS));
}
__device__ __forceinline__ void mma2_ss2_w(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                           uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, pe;\n\t.reg .b64 da, db;\n\telect.sync _|pe, 0xffffffff;\n\t"
        "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\tsetp.ne.b32 p, %6, 0;\n\t"
        "@pe tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %5, p;\n\t}" ::"r"(d_tmem),
        "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void mma2_ts2_w(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_lo, uint32_t b_hi, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, pe;\n\t.reg .b64 db;\n\telect.sync _|pe, 0xffffffff;\n\t"
        "mov.b64 db, {%2, %3};\n\tsetp.ne.b32 p, %5, 0;\n\t"
        "@pe tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], db, %4, p;\n\t}" ::"r"(d_tmem),
        "r"(a_tmem), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
        : "memory");
}
// all MMAs issued so far by this thread -> arrive(1) on the barrier at this shared-memory offset in every CTA of `mask`
__device__ __forceinline__ void mma2_commit_w(uint64_t* bar, uint16_t mask) {
    asm volatile(
        "{\n\t.reg .pred pe;\n\telect.sync _|pe, 0xffffffff;\n\t"
        "@pe tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n\t}" ::"r"(smem_u32(bar)),
        "h"(mask)
        : "memory");
}
// 32 lanes x 32 consecutive columns (fp32 / b32) -> 32 registers per thread (thread = lane of the warp's quadrant)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* v) {
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
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- fp32 -> (hi, lo) bf16 split: x ~= hi + lo with |x - hi - lo| <= 2^-17 |x| ------------------------------------
__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
    hi = __float2bfloat16_rn(x);
    lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}
// two floats -> packed hi pair / lo pair (element 0 in the low half).  The hi pair is widened back to fp32 with a shift and a mask
// (exact: a bf16 is the upper half of its fp32): F2FP.PACK_AB + SHF/LOP3 + 2 FADD + F2FP.PACK_AB, without the PRMT extract / re-pack
// that __low2float / __high2float compile to.
__device__ __forceinline__ void split_bf16x2(float a, float b, uint32_t& hi, uint32_t& lo) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    const float ra = a - __uint_as_float(hi << 16), rb = b - __uint_as_float(hi & 0xffff0000u);
    const __nv_bfloat162 l = __floats2bfloat162_rn(ra, rb);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}

}  // namespace umma
}  // namespace pnb
