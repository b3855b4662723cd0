// bf16 fused linear layer on the 5th-gen tensor cores (sm_100a):  Y = epi(A @ W + b)
//
//   A  [rows, K]  bf16 row-major (K-major), leading dimension lda, fetched by TMA (SWIZZLE_128B boxes
//                 of 128 rows x 64 columns; columns past K are zero-filled by the TMA unit)
//   Wt [N, K64]   bf16, the layer's kernel transposed (K-major), K padded to a multiple of 64
//   D  [128, BN]  fp32 accumulator in TMEM (BN <= 256 columns), one tcgen05.mma per 16 columns of K
//   Y             written by the epilogue warps straight from TMEM: bias, leaky-relu / query epilogue,
//                 bf16 or fp32 stores, optional split of the output columns over two buffers
//
// One CTA computes one 128 x BN tile.  Warp roles (192 threads): warp 0 = TMA producer (one elected
// lane), warp 1 = TMEM allocator + MMA issuer (one elected lane), warps 2..5 = epilogue (TMEM lane
// quadrant = warp_id % 4).  Two CTAs are resident per SM (2 x 96 KB of shared memory, 2 x 256 TMEM
// columns), so one CTA's epilogue overlaps the other's main loop.
#pragma once
#include <cuda.h>
#include "dsat_common.cuh"

namespace dsat {
namespace tc {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_N = 256;          // TMEM columns per CTA; tiles at the right edge use fewer
constexpr int BLOCK_K = 64;           // 64 bf16 = 128 bytes = one swizzle row
constexpr int STAGES = 2;
constexpr int THREADS = 192;
constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;     // 16 KB
constexpr int B_BYTES = BLOCK_N * BLOCK_K * 2;     // 32 KB
constexpr int SMEM_BYTES = STAGES * (A_BYTES + B_BYTES) + 1024 /*align*/ + 256 /*barriers*/;

enum TcEpilogue : int { TC_LINEAR = 0, TC_LRELU = 1, TC_QUERY = 2 };

struct TcOut {
    void* ptr0; int ld0; int bf16_0;      // columns [0, split)
    void* ptr1; int ld1; int bf16_1;      // columns [split, N) written at column (col - split); may be null
    int split;                            // multiple of 32
};

// ------------------------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tcgen05_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc], bf16 inputs, fp32 accumulate, issued by one thread
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}

// Forms for a warp that runs its issue loop converged (all 32 lanes execute the same control flow, the lane picked
// by elect.sync issues).  Inside an `if (lane == 0)` region the compiler has to wrap every uniform-register
// operand of UTCHMMA / UTCBAR in an ELECT + R2UR.BROADCAST + BRA.U.ANY loop, and that single thread's instruction
// stream was the critical path of the fused MLP kernels (~560 cycles of overhead per four MMAs).
__device__ __forceinline__ void umma_bf16_elect(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p, q;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "elect.sync _|q, 0xffffffff;\n"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// One K block (four 16-wide k-steps of a SWIZZLE_128B atom: the descriptors advance by 2 in the >>4 address field) and
// the commit that frees its ring slot, in a single asm block: one election and far fewer scalar instructions in the
// issuing warp, whose instruction stream competes with two busy epilogue warps for its scheduler.
__device__ __forceinline__ void umma_bf16_kblock_commit_elect(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                              uint32_t accumulate_first, uint64_t* slot_free_bar) {
    asm volatile(
        "{\n"
        ".reg .pred p, q, t;\n"
        ".reg .b64 a1, a2, a3, b1, b2, b3;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "setp.eq.b32 t, 0, 0;\n"
        "add.s64 a1, %1, 2;\n add.s64 a2, %1, 4;\n add.s64 a3, %1, 6;\n"
        "add.s64 b1, %2, 2;\n add.s64 b2, %2, 4;\n add.s64 b3, %2, 6;\n"
        "elect.sync _|q, 0xffffffff;\n"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], a1, b1, %3, t;\n"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], a2, b2, %3, t;\n"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], a3, b3, %3, t;\n"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%5];\n"
        "}\n" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate_first), "r"(smem_u32(slot_free_bar)) : "memory");
}
// ---- CTA-pair forms (cluster of 2, tcgen05 cta_group::2): the leader CTA (cluster rank 0) issues MMAs with M = 256
// that read A and B from both CTAs' shared memory (same offsets) and write each CTA's 128 accumulator rows into its own
// tensor memory.  Barriers the leader's issue warp waits on live in the leader's shared memory and are arrived on
// remotely (mapa + shared::cluster addressing); barriers that producers / epilogues wait on are per CTA and are
// signalled by the leader's multicast commits.
__device__ __forceinline__ uint32_t cluster_rank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t mapa_rank(uint32_t local_smem_addr, uint32_t rank) {   // shared::cluster address in CTA `rank`
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_expect_tx_at(uint32_t cluster_addr, uint32_t bytes) {
    // default semantics (release at CTA scope): the producer thread has written nothing the other CTA reads, the bytes arrive
    // through the TMA; a cluster-scope release here made every expect_tx a cluster-wide fence in the producer's issue loop
    asm volatile("mbarrier.arrive.expect_tx.shared::cluster.b64 _, [%0], %1;" ::"r"(cluster_addr), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive_at(uint32_t cluster_addr) {
    // default semantics (release at CTA scope), as CUTLASS's ClusterBarrier::arrive(cta_id): what the arriving epilogue warps
    // wrote is read by their OWN CTA's tensor core (after fence.proxy.async.shared::cta) or was read from TMEM
    // (tcgen05.fence::before_thread_sync); nothing of it is read by threads of the other CTA
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA load into THIS CTA's shared memory whose completion is signalled on a barrier given by its shared::cluster address
__device__ __forceinline__ void tma_load_2d_cg2(void* smem_dst, const CUtensorMap* map, uint32_t bar_cluster_addr, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(map), "r"(bar_cluster_addr), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void umma_bf16_elect_cg2(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p, q;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "elect.sync _|q, 0xffffffff;\n"
        "@q tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// arrives on the barrier at the same shared-memory offset in BOTH CTAs once all prior MMAs completed
__device__ __forceinline__ void tcgen05_commit_elect_cg2(uint64_t* bar) {
    asm volatile(
        "{\n"
        ".reg .pred q;\n"
        ".reg .b16 m;\n"
        "mov.b16 m, 3;\n"
        "elect.sync _|q, 0xffffffff;\n"
        "@q tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], m;\n"
        "}\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void umma_bf16_kblock_commit_elect_cg2(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                                  uint32_t accumulate_first, uint64_t* slot_free_bar) {
    asm volatile(
        "{\n"
        ".reg .pred p, q, t;\n"
        ".reg .b64 a1, a2, a3, b1, b2, b3;\n"
        ".reg .b16 m;\n"
        "mov.b16 m, 3;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "setp.eq.b32 t, 0, 0;\n"
        "add.s64 a1, %1, 2;\n add.s64 a2, %1, 4;\n add.s64 a3, %1, 6;\n"
        "add.s64 b1, %2, 2;\n add.s64 b2, %2, 4;\n add.s64 b3, %2, 6;\n"
        "elect.sync _|q, 0xffffffff;\n"
        "@q tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
        "@q tcgen05.mma.cta_group::2.kind::f16 [%0], a1, b1, %3, t;\n"
        "@q tcgen05.mma.cta_group::2.kind::f16 [%0], a2, b2, %3, t;\n"
        "@q tcgen05.mma.cta_group::2.kind::f16 [%0], a3, b3, %3, t;\n"
        "@q tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%5], m;\n"
        "}\n" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate_first), "r"(smem_u32(slot_free_bar)) : "memory");
}
// One K block (four k-steps) without a commit: used where several K blocks share one ring slot (the split-precision
// kernels multiply two A planes with the same weight block).
__device__ __forceinline__ void umma_bf16_kblock_elect(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                       uint32_t accumulate_first) {
    asm volatile(
        "{\n"
        ".reg .pred p, q, t;\n"
        ".reg .b64 a1, a2, a3, b1, b2, b3;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "setp.eq.b32 t, 0, 0;\n"
        "add.s64 a1, %1, 2;\n add.s64 a2, %1, 4;\n add.s64 a3, %1, 6;\n"
        "add.s64 b1, %2, 2;\n add.s64 b2, %2, 4;\n add.s64 b3, %2, 6;\n"
        "elect.sync _|q, 0xffffffff;\n"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], a1, b1, %3, t;\n"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], a2, b2, %3, t;\n"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], a3, b3, %3, t;\n"
        "}\n" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate_first) : "memory");
}
__device__ __forceinline__ void umma_bf16_kblock_elect_cg2(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                           uint32_t accumulate_first) {
    asm volatile(
        "{\n"
        ".reg .pred p, q, t;\n"
        ".reg .b64 a1, a2, a3, b1, b2, b3;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "setp.eq.b32 t, 0, 0;\n"
        "add.s64 a1, %1, 2;\n add.s64 a2, %1, 4;\n add.s64 a3, %1, 6;\n"
        "add.s64 b1, %2, 2;\n add.s64 b2, %2, 4;\n add.s64 b3, %2, 6;\n"
        "elect.sync _|q, 0xffffffff;\n"
        "@q tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
        "@q tcgen05.mma.cta_group::2.kind::f16 [%0], a1, b1, %3, t;\n"
        "@q tcgen05.mma.cta_group::2.kind::f16 [%0], a2, b2, %3, t;\n"
        "@q tcgen05.mma.cta_group::2.kind::f16 [%0], a3, b3, %3, t;\n"
        "}\n" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate_first) : "memory");
}
// A operand in TENSOR memory (the tcgen05.mma [a_tmem] form; B from shared memory as above): 16-bit A elements sit two
// per 32-bit column, row r of A in lane r (cta_group::2: each CTA's 128 rows in its own tensor memory, same column).  The
// x3 hidden epilogue stores the hi and lo planes interleaved per 32 K values: columns [32j, 32j+16) hold the hi plane of
// K in [32j, 32j+32), [32j+16, 32j+32) the lo plane.  So k-step k of a plane starts at column 32 (k/2) + 8 (k%2), and
// the four k-steps of a K block of 64 at +0, +8, +32, +40 from the block's column 64 kb.
__device__ __forceinline__ uint32_t tmem_a_kstep(int k) { return (uint32_t)(32 * (k >> 1) + 8 * (k & 1)); }
template <bool PAIR>
__device__ __forceinline__ void umma_bf16_ts_elect(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    if constexpr (PAIR) {
        asm volatile(
            "{\n"
            ".reg .pred p, q;\n"
            "setp.ne.b32 p, %4, 0;\n"
            "elect.sync _|q, 0xffffffff;\n"
            "@q tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n"
            "}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
    } else {
        asm volatile(
            "{\n"
            ".reg .pred p, q;\n"
            "setp.ne.b32 p, %4, 0;\n"
            "elect.sync _|q, 0xffffffff;\n"
            "@q tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
            "}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
    }
}
// one full K block (four k-steps) of the [a_tmem] form, one election
template <bool PAIR>
__device__ __forceinline__ void umma_bf16_ts_kblock_elect(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                                          uint32_t accumulate_first) {
#define DSAT_UMMA_TS_KBLOCK(CG)                                                              \
    "{\n"                                                                                    \
    ".reg .pred p, q, t;\n"                                                                  \
    ".reg .b32 a1, a2, a3;\n"                                                                \
    ".reg .b64 b1, b2, b3;\n"                                                                \
    "setp.ne.b32 p, %4, 0;\n"                                                                \
    "setp.eq.b32 t, 0, 0;\n"                                                                 \
    "add.u32 a1, %1, 8;\n add.u32 a2, %1, 32;\n add.u32 a3, %1, 40;\n"                       \
    "add.s64 b1, %2, 2;\n add.s64 b2, %2, 4;\n add.s64 b3, %2, 6;\n"                         \
    "elect.sync _|q, 0xffffffff;\n"                                                          \
    "@q tcgen05.mma.cta_group::" CG ".kind::f16 [%0], [%1], %2, %3, p;\n"                    \
    "@q tcgen05.mma.cta_group::" CG ".kind::f16 [%0], [a1], b1, %3, t;\n"                    \
    "@q tcgen05.mma.cta_group::" CG ".kind::f16 [%0], [a2], b2, %3, t;\n"                    \
    "@q tcgen05.mma.cta_group::" CG ".kind::f16 [%0], [a3], b3, %3, t;\n"                    \
    "}\n"
    if constexpr (PAIR)
        asm volatile(DSAT_UMMA_TS_KBLOCK("2") ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate_first) : "memory");
    else
        asm volatile(DSAT_UMMA_TS_KBLOCK("1") ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate_first) : "memory");
#undef DSAT_UMMA_TS_KBLOCK
}
__device__ __forceinline__ void tcgen05_commit_elect(uint64_t* bar) {
    asm volatile(
        "{\n"
        ".reg .pred q;\n"
        "elect.sync _|q, 0xffffffff;\n"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n"
        "}\n" ::"r"(smem_u32(bar)) : "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (sm_100 format, version 1):
// start address >> 4, leading byte offset unused (0), stride byte offset = 8 rows * 128 B = 1024 >> 4.
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;            // descriptor version (sm_100)
    d |= (uint64_t)2 << 61;            // SWIZZLE_128B
    return d;
}

// kind::f16 instruction descriptor: D fp32, A and B bf16, both K-major, M x N tile
__device__ __forceinline__ uint32_t make_idesc_bf16(int m, int n) {
    uint32_t d = 0;
    d |= 1u << 4;                      // c_format = F32
    d |= 1u << 7;                      // a_format = BF16
    d |= 1u << 10;                     // b_format = BF16
    d |= (uint32_t)(n >> 3) << 17;     // N / 8
    d |= (uint32_t)(m >> 4) << 24;     // M / 16
    return d;
}

__device__ __forceinline__ void tmem_ld_32cols(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void store_chunk(const TcOut& out, size_t row, int col, const float (&v)[32]) {
    const bool second = out.ptr1 != nullptr && col >= out.split;
    void* base = second ? out.ptr1 : out.ptr0;
    const int ld = second ? out.ld1 : out.ld0;
    const int c = second ? col - out.split : col;
    const int is_bf16 = second ? out.bf16_1 : out.bf16_0;
    if (is_bf16) {
        __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(base) + row * ld + c;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            uint4 pack;
            __nv_bfloat162 p0 = __floats2bfloat162_rn(v[8 * j + 0], v[8 * j + 1]);
            __nv_bfloat162 p1 = __floats2bfloat162_rn(v[8 * j + 2], v[8 * j + 3]);
            __nv_bfloat162 p2 = __floats2bfloat162_rn(v[8 * j + 4], v[8 * j + 5]);
            __nv_bfloat162 p3 = __floats2bfloat162_rn(v[8 * j + 6], v[8 * j + 7]);
            pack.x = *reinterpret_cast<uint32_t*>(&p0); pack.y = *reinterpret_cast<uint32_t*>(&p1);
            pack.z = *reinterpret_cast<uint32_t*>(&p2); pack.w = *reinterpret_cast<uint32_t*>(&p3);
            reinterpret_cast<uint4*>(dst)[j] = pack;
        }
    } else {
        float* dst = reinterpret_cast<float*>(base) + row * ld + c;
#pragma unroll
        for (int j = 0; j < 8; ++j)
            reinterpret_cast<float4*>(dst)[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    }
}

// --------------------------------------------------------------------------------------- kernel
// grid.x = row tiles * n_tiles (N tiles fastest so that CTAs sharing an A tile run back to back)
__global__ void __launch_bounds__(THREADS, 2)
tc_linear_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                 const float* __restrict__ bias, TcOut out, int rows, int K, int N, int n_tiles, int epi, int qmaps,
                 int a_box_rows, int b_box_rows) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* smem_a = smem;                                   // STAGES x 16 KB
    uint8_t* smem_b = smem + STAGES * A_BYTES;                // STAGES x 32 KB
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * (A_BYTES + B_BYTES));
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* tmem_full_bar = empty_bar + STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row0 = (blockIdx.x / n_tiles) * BLOCK_M;
    const int n0 = (blockIdx.x % n_tiles) * BLOCK_N;
    const int bn = min(BLOCK_N, N - n0);                      // multiple of 16
    const int k_blocks = (K + BLOCK_K - 1) / BLOCK_K;

    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        mbar_init(tmem_full_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
    }
    if (warp == 1) {   // TMEM allocation by one full warp; the address lands in shared memory
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(BLOCK_N));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {     // ===== TMA producer =====
            for (int kb = 0; kb < k_blocks; ++kb) {
                const int s = kb % STAGES;
                const uint32_t phase = (kb / STAGES) & 1;
                mbar_wait(&empty_bar[s], phase ^ 1);
                mbar_expect_tx(&full_bar[s], (uint32_t)(a_box_rows + b_box_rows) * (BLOCK_K * 2));
                tma_load_2d(smem_a + s * A_BYTES, &map_a, &full_bar[s], kb * BLOCK_K, row0);
                tma_load_2d(smem_b + s * B_BYTES, &map_b, &full_bar[s], kb * BLOCK_K, n0);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {     // ===== MMA issuer =====
            const uint32_t idesc = make_idesc_bf16(BLOCK_M, bn);
            for (int kb = 0; kb < k_blocks; ++kb) {
                const int s = kb % STAGES;
                const uint32_t phase = (kb / STAGES) & 1;
                mbar_wait(&full_bar[s], phase);
                tcgen05_fence_after();
                const uint64_t da = make_smem_desc_sw128(smem_u32(smem_a + s * A_BYTES));
                const uint64_t db = make_smem_desc_sw128(smem_u32(smem_b + s * B_BYTES));
                const int ksteps = min(BLOCK_K / 16, (K - kb * BLOCK_K + 15) / 16);     // skip the zero-filled tail
                for (int k = 0; k < ksteps; ++k) {
                    // advancing 16 bf16 = 32 bytes along K inside the swizzled row: +2 in the (>>4) address field
                    umma_bf16(tmem_base, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kb | k) != 0);
                }
                tcgen05_commit(&empty_bar[s]);            // frees the stage once these MMAs have read it
            }
            tcgen05_commit(tmem_full_bar);                // accumulator complete
        }
    } else {                 // ===== epilogue warps 2..5 =====
        const int quad = warp & 3;                        // TMEM lane quadrant this warp may access
        const size_t row = (size_t)row0 + quad * 32 + lane;
        mbar_wait(tmem_full_bar, 0);
        tcgen05_fence_after();
        for (int c = 0; c < bn; c += 32) {
            uint32_t raw[32];
            tmem_ld_32cols(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)c, raw);
            if (row < (size_t)rows) {
                float v[32];
                const int col = n0 + c;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    float x = __uint_as_float(raw[j]) + ((col + j < N) ? __ldg(bias + col + j) : 0.f);
                    if (epi == TC_LRELU) x = x > 0.f ? x : 0.2f * x;
                    v[j] = x;
                }
                const int valid = min(32, bn - c);
                if (valid == 32) {
                    store_chunk(out, row, col, v);
                    if (epi == TC_QUERY) {      // softplus(+q), softplus(-q) next to the query
                        float sp[32], sn[32];
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            // softplus(x) = max(x,0) + log(1 + exp(-|x|)); softplus(-x) = softplus(x) - x.
                            // fast intrinsics: the result is rounded to bf16 anyway
                            const float tail = __logf(1.0f + __expf(-fabsf(v[j])));
                            sp[j] = fmaxf(v[j], 0.f) + tail;
                            sn[j] = fmaxf(-v[j], 0.f) + tail;
                        }
                        store_chunk(out, row, col + qmaps, sp);
                        store_chunk(out, row, col + 2 * qmaps, sn);
                    }
                } else {                        // right edge of an N that is not a multiple of 32 (N = 16k)
                    const bool second = out.ptr1 != nullptr && col >= out.split;
                    void* base = second ? out.ptr1 : out.ptr0;
                    const int ld = second ? out.ld1 : out.ld0;
                    const int cc = second ? col - out.split : col;
                    const int is_bf16 = second ? out.bf16_1 : out.bf16_0;
                    for (int j = 0; j < valid; ++j) {
                        if (is_bf16) reinterpret_cast<__nv_bfloat16*>(base)[row * ld + cc + j] = __float2bfloat16_rn(v[j]);
                        else reinterpret_cast<float*>(base)[row * ld + cc + j] = v[j];
                    }
                }
            }
        }
        tcgen05_fence_before();
    }
    __syncthreads();
    if (warp == 1) {
        tcgen05_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(BLOCK_N));
    }
}

// ------------------------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// 2-D bf16 tensor [rows, cols] with row stride ld (elements); box = 64 columns x box_rows rows, SWIZZLE_128B
inline bool make_bf16_map(CUtensorMap* map, const void* base, long long rows, int cols, int ld, int box_rows) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return false;
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
    cuuint32_t box[2] = {(cuuint32_t)BLOCK_K, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

struct TcLinear {
    CUtensorMap map_a, map_b;
    const float* bias;
    TcOut out;
    int rows, K, N, epi, qmaps;
    int a_box_rows, b_box_rows;     // TMA box heights the descriptors were encoded with
};

inline cudaError_t configure_tc_device() {
    static PerDeviceOnce configured;
    if (configured.done()) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(tc_linear_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (e == cudaSuccess) configured.mark();
    return e;
}

inline cudaError_t launch_tc_linear(const TcLinear& op, cudaStream_t stream) {
    if (op.rows <= 0) return cudaSuccess;
    {
        cudaError_t e = configure_tc_device();
        if (e != cudaSuccess) return e;
    }
    const int n_tiles = ceil_div(op.N, BLOCK_N);
    const unsigned grid = (unsigned)(n_tiles * ceil_div(op.rows, BLOCK_M));
    tc_linear_kernel<<<grid, THREADS, SMEM_BYTES, stream>>>(op.map_a, op.map_b, op.bias, op.out, op.rows, op.K, op.N,
                                                             n_tiles, op.epi, op.qmaps, op.a_box_rows, op.b_box_rows);
    return cudaGetLastError();
}

}  // namespace tc
}  // namespace dsat
