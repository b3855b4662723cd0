// Whole-MLP persistent kernel on the 5th-gen tensor cores: the 2 or 3 Dense layers of one QuerySAT MLP
// (reference model/mlp.py:42-50) for tiles of 128 rows, one CTA per SM looping over its tiles.
// Hidden activations never leave the SM: each layer's fp32 accumulator is drained from TMEM by the
// epilogue warps (bias, leaky-relu, bf16) straight into shared memory in the K-major SWIZZLE_128B
// layout that the next layer's tcgen05.mma reads as its A operand.
//
//   shared memory   AH region   : the input tile A [128, K0] (TMA, 16 KB per 64 columns); after layer l
//                                 finished it is overwritten by that layer's hidden activations
//                   weight ring : 2-4 slots; slot = W_l^T[n_half*256 .. +256, kb*64 .. +64] (from L2)
//                   out staging : 4 x 4.5 KB, per-warp transpose so that the output leaves in 64/128-byte rows
//   tensor memory   512 columns; when every layer is at most 256 wide consecutive layers alternate between
//                   the two halves, so the first layer of tile i+1 accumulates while tile i's output drains
//   warps           0 = TMA producer, 1 = MMA issuer (+TMEM alloc), 2..5 = epilogue (lane quadrant = warp%4)
//
//                   input ring  : (a_slots > 0) the 64-column blocks of the input tile stream through their own ring
//                                 instead of resting in AH, so the next tile's input is fetched while this tile's
//                                 later layers and epilogues still run (AH then holds hidden activations only)
//                   ping-pong   : (pp) two tiles are in flight, tile parity s owns accumulator half s and hidden region
//                                 H[s]; the MMA warp issues L1(A) L1(B) L2(A) L2(B) ..., so every epilogue of one tile
//                                 runs under an MMA phase of the other (the final epilogue stages through its own,
//                                 by then dead, H[s])
// mbarriers:  a_full (TMA->MMA, per tile)      ah_free (MMA->TMA, AH may take the next input tile)
//             ring full/empty (TMA<->MMA)       tmem_full[buf] (MMA->epilogue)   tmem_empty[buf] (epilogue->MMA)
//             h_full (epilogue->MMA, hidden activations of a layer are in shared memory)
#pragma once
#include "dsat_gemm_tc.cuh"

namespace dsat {
namespace fm {

using tc::TcOut;

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;
constexpr int MAX_THREADS = 320;
constexpr int MAX_LAYERS = 3;
constexpr int MAX_SLOTS = 8;
constexpr int AH_BLOCK_BYTES = BLOCK_M * BLOCK_K * 2;      // 16 KB: 128 rows x 64 bf16
constexpr int TMEM_COLS = 512;
constexpr int STAGE_ROW = 128 + 16;                        // bytes per staged row (one 32-column fp32 chunk + pad)
constexpr int BAR_BYTES = 512;
constexpr int MAX_A_SLOTS = 8;
constexpr int SMEM_LIMIT = 227 * 1024;

struct FmLayer {
    int K, N;              // multiples of 16; N <= 512
    int epi;               // tc::TC_LINEAR / TC_LRELU / TC_QUERY (query only on the last layer)
    int box_rows;          // TMA box height of this layer's weight map (min(256, N))
    int bias_off;          // offset of this layer's biases in the shared bias array
    const float* bias;
};

// One accumulator-sized piece of work in split mode: columns [n0, n0 + N) of one layer, N <= 256.
struct FmStep {
    short layer, n0, N;
    char hidden;           // the result goes to the hidden region (blocks n0/64 ...), else to global memory
    char wait_next;        // its epilogue overwrites shared memory that the NEXT step's MMAs still read
};
constexpr int MAX_STEPS = 6;

struct FmParams {
    int n_layers;
    FmLayer layer[MAX_LAYERS];
    int rows, n_tiles, a_box_rows, ah_blocks, slots, slot_bytes, two_bufs, qmaps;
    int pair;              // CTA-pair mode (cluster of 2, cta_group::2): host-side flag, the kernel is a separate instantiation
    int pp;                // ping-pong: two tiles in flight (needs a_slots > 0 and two_bufs)
    int stage_in_h;        // the output staging of a tile aliases its (by then dead) hidden region, at byte offset stage_off
    int stage_off;
    int a_slots;           // > 0: layer 0's A operand streams through an input ring of that many 16 KB blocks
    int stage_row;         // bytes per staged output row: 80 when every output is bf16 (64 B + pad), else 144
    int bias_total;        // floats in the shared bias array
    int smem_pad;          // bytes the plan reserved for aligning the dynamic shared memory base to 1024
    int epi_warps;         // 4 or 8 epilogue warps: with 8, two warps share a TMEM lane quadrant and alternate 32-column chunks
    int split;             // split mode (fused_mlp_split_kernel): 512-wide layers run as two 256-column steps, see below;
                           // only the current step's biases are in shared memory (2 x 256 floats, staged per step)
    int n_steps;
    FmStep step[MAX_STEPS];
    TcOut out;
    long long* prof;       // optional [16] cycle counters of CTA 0 (wait/work breakdown), nullptr = off
};

#define DSAT_TIMED_WAIT(acc, call)                 \
    do {                                           \
        if (timing) {                              \
            const long long t0__ = clock64();      \
            call;                                  \
            acc += clock64() - t0__;               \
        } else {                                   \
            call;                                  \
        }                                          \
    } while (0)

// ---- explicit shared-space accesses and split TMEM load / wait (software pipelining of the epilogue)
__device__ __forceinline__ void sts128(uint32_t addr, const uint4& v) {
    // volatile keeps the order relative to the (volatile) fences and barrier operations; no "memory" clobber, so the
    // compiler does not have to re-load every memory-resident value after each store
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w));
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ float4 lds128f(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void tmem_ld_32cols_async(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
// wait for the outstanding tcgen05.ld; the registers are in/out operands so that no use is scheduled above the wait
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                   "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
                   "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
                   "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31]));
}

// 32 columns of this warp's 32 TMEM lanes; tcgen05.wait::st (tmem_st_wait) before anyone is told the data is there
__device__ __forceinline__ void tmem_st_32cols(uint32_t taddr, const uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
          "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
          "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]),
          "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ uint4 pack8_bf16(const float* v) {
    __nv_bfloat162 p0 = __floats2bfloat162_rn(v[0], v[1]), p1 = __floats2bfloat162_rn(v[2], v[3]);
    __nv_bfloat162 p2 = __floats2bfloat162_rn(v[4], v[5]), p3 = __floats2bfloat162_rn(v[6], v[7]);
    uint4 pack;
    pack.x = *reinterpret_cast<uint32_t*>(&p0); pack.y = *reinterpret_cast<uint32_t*>(&p1);
    pack.z = *reinterpret_cast<uint32_t*>(&p2); pack.w = *reinterpret_cast<uint32_t*>(&p3);
    return pack;
}

// bias (+ leaky relu) of one 32-column chunk; the 32 biases come in as eight 16-byte shared loads
__device__ __forceinline__ void bias_act_chunk(const uint32_t (&raw)[32], uint32_t bias_addr, bool lrelu, float (&v)[32]) {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const float4 b = lds128f(bias_addr + 16 * q);
        const float x0 = __uint_as_float(raw[4 * q]) + b.x, x1 = __uint_as_float(raw[4 * q + 1]) + b.y;
        const float x2 = __uint_as_float(raw[4 * q + 2]) + b.z, x3 = __uint_as_float(raw[4 * q + 3]) + b.w;
        v[4 * q] = lrelu ? fmaxf(x0, 0.2f * x0) : x0;
        v[4 * q + 1] = lrelu ? fmaxf(x1, 0.2f * x1) : x1;
        v[4 * q + 2] = lrelu ? fmaxf(x2, 0.2f * x2) : x2;
        v[4 * q + 3] = lrelu ? fmaxf(x3, 0.2f * x3) : x3;
    }
}

// bf16 outputs: round the fp32 accumulator to bf16 pairs first, then bias add and leaky relu on packed pairs
// (HADD2/HMUL2/HMNMX2.BF16): 2.3x fewer instructions per chunk than the fp32 version; the result is stored as
// bf16 either way.  32 bf16 biases = four 16-byte shared loads.
__device__ __forceinline__ void bias_act_chunk_bf16(const uint32_t (&raw)[32], uint32_t bias_f_addr, bool lrelu, uint4 (&out)[4]) {
    // bias add in fp32 (one rounding to bf16, as on the per-layer path), leaky relu on packed bf16 pairs
    const __nv_bfloat162 slope = __floats2bfloat162_rn(0.2f, 0.2f);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const float4 b0 = lds128f(bias_f_addr + 32 * q), b1 = lds128f(bias_f_addr + 32 * q + 16);
        const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
        uint32_t ow[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            __nv_bfloat162 x = __floats2bfloat162_rn(__uint_as_float(raw[8 * q + 2 * i]) + bb[2 * i],
                                                     __uint_as_float(raw[8 * q + 2 * i + 1]) + bb[2 * i + 1]);
            if (lrelu) x = __hmax2(x, __hmul2(x, slope));
            ow[i] = *reinterpret_cast<uint32_t*>(&x);
        }
        out[q] = make_uint4(ow[0], ow[1], ow[2], ow[3]);
    }
}

// packed variant of store_chunk_fast for bf16 outputs
__device__ __forceinline__ void store_chunk_packed(uint32_t stage_addr, int stage_row, int lane, const uint4 (&w)[4], int valid,
                                                   uint8_t* gbase, size_t row_pitch_bytes, size_t row_first,
                                                   int rows_left, int col) {
    const uint32_t mine = stage_addr + lane * stage_row;
#pragma unroll
    for (int q = 0; q < 4; ++q) sts128(mine + 16 * q, w[q]);
    __syncwarp();
    const int valid_pieces = valid / 8;
    uint4 t[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int pidx = lane + 32 * k;
        t[k] = lds128(stage_addr + (pidx >> 2) * stage_row + 16 * (pidx & 3));
    }
    uint8_t* g0 = gbase + row_first * row_pitch_bytes + (size_t)col * 2;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int pidx = lane + 32 * k;
        const int rr = pidx >> 2, piece = pidx & 3;
        if (rr < rows_left && piece < valid_pieces)
            *reinterpret_cast<uint4*>(g0 + (size_t)rr * row_pitch_bytes + 16 * piece) = t[k];
    }
    __syncwarp();
}

// one 32-column chunk of one output row per lane -> global memory through a per-warp transpose buffer (explicit
// shared-space accesses: the generic-pointer version stalled every store on a generic load)
template <bool BF16>
__device__ __forceinline__ void store_chunk_fast(uint32_t stage_addr, int stage_row, int lane, const float (&v)[32], int valid,
                                                 uint8_t* gbase, size_t row_pitch_bytes, size_t row_first,
                                                 int rows_left, int col) {
    const uint32_t mine = stage_addr + lane * stage_row;
    if (BF16) {
#pragma unroll
        for (int q = 0; q < 4; ++q) sts128(mine + 16 * q, pack8_bf16(&v[8 * q]));
    } else {
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            uint4 w;
            w.x = __float_as_uint(v[4 * q]); w.y = __float_as_uint(v[4 * q + 1]);
            w.z = __float_as_uint(v[4 * q + 2]); w.w = __float_as_uint(v[4 * q + 3]);
            sts128(mine + 16 * q, w);
        }
    }
    __syncwarp();
    constexpr int ES = BF16 ? 2 : 4;
    constexpr int PIECES = BF16 ? 4 : 8;
    const int valid_pieces = valid * ES / 16;
    uint4 t[PIECES];
#pragma unroll
    for (int k = 0; k < PIECES; ++k) {
        const int pidx = lane + 32 * k;
        t[k] = lds128(stage_addr + (pidx / PIECES) * stage_row + 16 * (pidx % PIECES));
    }
    uint8_t* g0 = gbase + row_first * row_pitch_bytes + (size_t)col * ES;
#pragma unroll
    for (int k = 0; k < PIECES; ++k) {
        const int pidx = lane + 32 * k;
        const int rr = pidx / PIECES, piece = pidx % PIECES;
        if (rr < rows_left && piece < valid_pieces)
            *reinterpret_cast<uint4*>(g0 + (size_t)rr * row_pitch_bytes + 16 * piece) = t[k];
    }
    __syncwarp();
}

struct EpiCtx {           // loop-invariant scalars of one (tile, layer) epilogue, all in registers
    uint32_t lane_addr, ah_addr, bl_addr, stage_addr;
    int N, epi, cpar, cstep, r, lane, qmaps, stage_row;
    size_t row_first; int rows_left;
    void* ptr0; void* ptr1; int ld0, ld1, bf0, bf1, split;
};

template <bool HIDDEN>
__device__ __forceinline__ void epi_process(const EpiCtx& e, const uint32_t (&raw)[32], int c) {
    const bool lrelu = e.epi == tc::TC_LRELU;
    if (HIDDEN) {
        // K-major SWIZZLE_128B: 16-byte chunk j of row r of block kb sits at kb*16KB + r*128 + ((j ^ (r & 7)) << 4)
        uint4 w[4];
        bias_act_chunk_bf16(raw, e.bl_addr + 4u * (uint32_t)c, lrelu, w);
        const uint32_t blk = e.ah_addr + (uint32_t)(c >> 6) * AH_BLOCK_BYTES + (uint32_t)e.r * 128;
        const int j0 = (c & 63) >> 3;
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (c + 8 * q < e.N) sts128(blk + (uint32_t)(((j0 + q) ^ (e.r & 7)) << 4), w[q]);
        return;
    }
    const bool second = e.ptr1 != nullptr && c >= e.split;
    uint8_t* gbase = reinterpret_cast<uint8_t*>(second ? e.ptr1 : e.ptr0);
    const int is_bf16 = second ? e.bf1 : e.bf0;
    const size_t pitch = (size_t)(second ? e.ld1 : e.ld0) * (is_bf16 ? 2 : 4);
    const int cc = second ? c - e.split : c;
    const int valid = min(32, e.N - c);
    if (is_bf16 && e.epi != tc::TC_QUERY) {
        uint4 w[4];
        bias_act_chunk_bf16(raw, e.bl_addr + 4u * (uint32_t)c, lrelu, w);
        store_chunk_packed(e.stage_addr, e.stage_row, e.lane, w, valid, gbase, pitch, e.row_first, e.rows_left, cc);
        return;
    }
    float v[32];
    bias_act_chunk(raw, e.bl_addr + 4u * (uint32_t)c, lrelu, v);
    if (is_bf16) store_chunk_fast<true>(e.stage_addr, e.stage_row, e.lane, v, valid, gbase, pitch, e.row_first, e.rows_left, cc);
    else store_chunk_fast<false>(e.stage_addr, e.stage_row, e.lane, v, valid, gbase, pitch, e.row_first, e.rows_left, cc);
    if (e.epi == tc::TC_QUERY) {
        float sp[32], sn[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            const float t = __logf(1.0f + __expf(-fabsf(v[i])));
            sp[i] = fmaxf(v[i], 0.f) + t;
            sn[i] = fmaxf(-v[i], 0.f) + t;
        }
        if (is_bf16) {
            store_chunk_fast<true>(e.stage_addr, e.stage_row, e.lane, sp, valid, gbase, pitch, e.row_first, e.rows_left, cc + e.qmaps);
            store_chunk_fast<true>(e.stage_addr, e.stage_row, e.lane, sn, valid, gbase, pitch, e.row_first, e.rows_left, cc + 2 * e.qmaps);
        } else {
            store_chunk_fast<false>(e.stage_addr, e.stage_row, e.lane, sp, valid, gbase, pitch, e.row_first, e.rows_left, cc + e.qmaps);
            store_chunk_fast<false>(e.stage_addr, e.stage_row, e.lane, sn, valid, gbase, pitch, e.row_first, e.rows_left, cc + 2 * e.qmaps);
        }
    }
}

// Drain one accumulator: software pipeline, the tcgen05.ld of the next chunk is in flight while this one is
// processed.  For the last layer the accumulator is handed back (tmem_empty) as soon as this warp's last TMEM
// read has landed; for hidden layers the caller arrives after the shared-memory stores are fenced.
// barrier arrive by shared-memory address: this CTA's barrier, or (PAIR) the leader CTA's through shared::cluster
template <bool PAIR>
__device__ __forceinline__ void arrive_addr(uint32_t addr) {
    if constexpr (PAIR) tc::mbar_arrive_at(addr);
    else asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(addr) : "memory");
}

// One arrival per epilogue WARP (the barriers count warps): every lane has done its own fences, the warp converges, one
// lane signals.  In CTA-pair mode the arrival is a remote (cluster) operation; 256 of them per barrier phase serialised.
template <bool PAIR>
__device__ __forceinline__ void warp_arrive(uint32_t addr, int lane) {
    __syncwarp();
    if (lane == 0) arrive_addr<PAIR>(addr);
}

template <bool HIDDEN, bool PAIR>
__device__ __forceinline__ void epi_drain(const EpiCtx& e, uint32_t tmem_empty_addr) {
    bool released = false;
    if constexpr (!HIDDEN) {
#pragma unroll 1
        for (int c = 32 * e.cpar; c < e.N; c += e.cstep) {
            uint32_t ra[32];
            tmem_ld_32cols_async(e.lane_addr + (uint32_t)c, ra);
            tmem_ld_wait(ra);
            if (!HIDDEN && c + e.cstep >= e.N) {     // last TMEM read of this warp: hand the accumulator back early
                tc::tcgen05_fence_before();
                warp_arrive<PAIR>(tmem_empty_addr, e.lane);
                released = true;
            }
            epi_process<HIDDEN>(e, ra, c);
        }
    } else {
        // hidden layers (the MMA warp waits for these): two register buffers, chunk c + cstep is on its way out of
        // TMEM while chunk c is processed.  (The final epilogue keeps one buffer: its store path needs the registers.)
        int c = 32 * e.cpar;
        if (c < e.N) {
            uint32_t ra[32], rb[32];
            tmem_ld_32cols_async(e.lane_addr + (uint32_t)c, ra);
#pragma unroll 1
            while (true) {
                tmem_ld_wait(ra);
                const int c1 = c + e.cstep;
                if (c1 < e.N) tmem_ld_32cols_async(e.lane_addr + (uint32_t)c1, rb);
                epi_process<HIDDEN>(e, ra, c);
                if (c1 >= e.N) break;
                tmem_ld_wait(rb);
                c = c1 + e.cstep;
                if (c < e.N) tmem_ld_32cols_async(e.lane_addr + (uint32_t)c, ra);
                epi_process<HIDDEN>(e, rb, c1);
                if (c >= e.N) break;
            }
        }
    }
    if (!HIDDEN && !released) { tc::tcgen05_fence_before(); warp_arrive<PAIR>(tmem_empty_addr, e.lane); }
}

template <bool TIMING, bool PAIR>
__global__ void __launch_bounds__(MAX_THREADS, 1)
fused_mlp_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w0, const __grid_constant__ CUtensorMap map_w1,
                 const __grid_constant__ CUtensorMap map_w2, FmParams p) {
    using namespace tc;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    if ((int)(smem - smem_raw) > p.smem_pad) __trap();     // the plan assumed a better aligned base (dyn_smem_pad)
    uint8_t* ah = smem;
    const size_t h_bytes = (size_t)p.ah_blocks * AH_BLOCK_BYTES;          // one AH / hidden region
    uint8_t* a_ring = smem + (p.pp ? 2 : 1) * h_bytes;
    uint8_t* ring = a_ring + (size_t)p.a_slots * AH_BLOCK_BYTES;
    uint8_t* stage_all = ring + (size_t)p.slots * p.slot_bytes;
    uint8_t* tail = stage_all + (p.stage_in_h ? 0 : (size_t)p.epi_warps * 32 * p.stage_row);
    uint64_t* a_full = reinterpret_cast<uint64_t*>(tail);
    uint64_t* ah_free = a_full + 1;
    uint64_t* h_full = a_full + 2;                     // [2]
    uint64_t* tmem_full = a_full + 4;                  // [2]
    uint64_t* tmem_empty = a_full + 6;                 // [2]
    uint64_t* ring_full = a_full + 8;                  // [MAX_SLOTS]
    uint64_t* ring_empty = a_full + 8 + MAX_SLOTS;     // [MAX_SLOTS]
    uint64_t* a_ring_full = a_full + 8 + 2 * MAX_SLOTS;                  // [MAX_A_SLOTS]
    uint64_t* a_ring_empty = a_ring_full + MAX_A_SLOTS;                  // [MAX_A_SLOTS]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(a_ring_empty + MAX_A_SLOTS);
    float* bias_s = reinterpret_cast<float*>(tail + BAR_BYTES);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int epi_threads = 32 * p.epi_warps;
    const CUtensorMap* map_w[MAX_LAYERS] = {&map_w0, &map_w1, &map_w2};
    const bool timing = TIMING && p.prof != nullptr && blockIdx.x == 0;   // TIMING = false strips every counter
    const long long t_kernel0 = timing ? clock64() : 0;
    long long w0 = 0, w1 = 0, w2 = 0, w3 = 0, w4 = 0, w5 = 0, w6 = 0, w7 = 0;

    // PAIR (launched as clusters of 2): rank 0 leads.  "full"-type barriers (waited on by the leader's issue warp) count
    // one arrival per CTA / per epilogue thread of both CTAs; "empty"-type and tmem_full barriers are local and get one
    // arrival from the leader's multicast commit.
    const uint32_t rank = PAIR ? cluster_rank() : 0u;
    const bool leader = rank == 0;
    constexpr int NC = PAIR ? 2 : 1;
    if (threadIdx.x == 0) {
        mbar_init(a_full, NC);
        mbar_init(ah_free, 1);
        for (int b = 0; b < 2; ++b) {
            mbar_init(&h_full[b], NC * p.epi_warps);
            mbar_init(&tmem_full[b], 1);
            mbar_init(&tmem_empty[b], NC * p.epi_warps);
        }
        for (int s = 0; s < MAX_SLOTS; ++s) { mbar_init(&ring_full[s], NC); mbar_init(&ring_empty[s], 1); }
        for (int s = 0; s < MAX_A_SLOTS; ++s) { mbar_init(&a_ring_full[s], NC); mbar_init(&a_ring_empty[s], 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w0) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w1) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w2) : "memory");
    }
    if (warp == 1) {
        if constexpr (PAIR) {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS));
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS));
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
        }
    }
    if (warp >= 2) {
        for (int l = 0; l < p.n_layers; ++l)
            for (int i = threadIdx.x - 64; i < p.layer[l].N; i += epi_threads) {
                bias_s[p.layer[l].bias_off + i] = __ldg(p.layer[l].bias + i);
            }
    }
    tcgen05_fence_before();
    __syncthreads();
    if constexpr (PAIR) cluster_sync_all();              // both CTAs' barriers exist before any remote arrive
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int n_layers = p.n_layers;
    // Every wait, in CTA-pair mode too, acquires at CTA scope: barriers completed by TMA transactions or tcgen05.commit order
    // async-proxy work on both sides, and the peer's epilogue threads arrive on tmem_empty / h_full only for what this CTA's
    // tensor core reads (tc::mbar_arrive_at).  (With a cluster-scope try_wait on every ring slot the pair instantiation
    // spent ~2 k cycles per k-block.)
    // address of the barrier the leader's issue warp waits on (this CTA's own one when not paired)
    auto at_leader = [&](uint64_t* bar) -> uint32_t { return PAIR ? mapa_rank(smem_u32(bar), 0) : smem_u32(bar); };
    // This CTA's tiles are blockIdx.x + j * gridDim.x, j < nt.  All three roles walk the same sequence of
    // (tile, layer) steps: tile by tile, or (pp) in groups of two tiles with the layers interleaved
    // L1(A) L1(B) L2(A) L2(B) ...  For step (j, l) with s = j & 1 inside its group:
    //   pp    : accumulator half s, hidden region s, both used once per layer and group
    //   else  : accumulator half alternates per step when every layer fits 256 columns, one hidden region
    // work units: 128-row tiles of this CTA, or (PAIR) 256-row macro tiles of the pair, of which this CTA owns half
    const int unit0 = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int unit_stride = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    const int n_units = PAIR ? (p.n_tiles + 1) / 2 : p.n_tiles;
    const int nt = unit0 < n_units ? (n_units - unit0 + unit_stride - 1) / unit_stride : 0;
    auto tile_of = [&](int j) { const int u = unit0 + j * unit_stride; return PAIR ? 2 * u + (int)rank : u; };
    const int group = p.pp ? 2 : 1;
    struct Step { int tile, buf, use, hidx, hcnt; };
    auto make_step = [&](int j0, int s, int l) {
        Step st;
        const int j = j0 + s;
        st.tile = tile_of(j);
        if (p.pp) {
            st.buf = s; st.use = (j0 >> 1) * n_layers + l;
            st.hidx = s; st.hcnt = (j0 >> 1) * (n_layers - 1) + (l - 1);
        } else {
            const int g = j * n_layers + l;
            st.buf = p.two_bufs ? (g & 1) : 0; st.use = p.two_bufs ? (g >> 1) : g;
            st.hidx = 0; st.hcnt = j * (n_layers - 1) + (l - 1);
        }
        return st;
    };

    if (warp == 0) {
        if (lane == 0) {   // ================================ TMA producer
            const int k0_blocks = (p.layer[0].K + BLOCK_K - 1) / BLOCK_K;
            int slot = 0; uint32_t phase = 0;
            int aslot = 0; uint32_t aphase = 0;
            auto load_2d = [&](uint8_t* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
                if constexpr (PAIR) tma_load_2d_cg2(dst, map, at_leader(bar), c0, c1); else tma_load_2d(dst, map, bar, c0, c1);
            };
            auto expect = [&](uint64_t* bar, uint32_t bytes) {
                if constexpr (PAIR) mbar_expect_tx_at(at_leader(bar), bytes); else mbar_expect_tx(bar, bytes);
            };
            auto load_a_block = [&](uint8_t* dst, uint64_t* bar, int kb, int tile) {
                load_2d(dst, &map_a, bar, kb * BLOCK_K, tile * BLOCK_M);
            };
            for (int j0 = 0; j0 < nt; j0 += group)
                for (int l = 0; l < n_layers; ++l)
                    for (int s = 0; s < group; ++s) {
                        if (j0 + s >= nt) continue;
                        const int j = j0 + s, tile = tile_of(j);
                        if (l == 0 && p.a_slots == 0) {      // whole input tile into AH
                            if (j > 0) DSAT_TIMED_WAIT(w0, mbar_wait(ah_free, (uint32_t)((j - 1) & 1)));   // tile j-1 no longer reads AH
                            expect(a_full, (uint32_t)(k0_blocks * p.a_box_rows) * (BLOCK_K * 2));
                            for (int kb = 0; kb < k0_blocks; ++kb) load_a_block(ah + (size_t)kb * AH_BLOCK_BYTES, a_full, kb, tile);
                        }
                        const int kbs = (p.layer[l].K + BLOCK_K - 1) / BLOCK_K;
                        const int halves = (p.layer[l].N + 255) / 256;
                        for (int kb = 0; kb < kbs; ++kb) {
                            if (l == 0 && p.a_slots > 0) {     // input block kb of this tile into the input ring
                                DSAT_TIMED_WAIT(w0, mbar_wait(&a_ring_empty[aslot], aphase ^ 1));
                                expect(&a_ring_full[aslot], (uint32_t)p.a_box_rows * (BLOCK_K * 2));
                                load_a_block(a_ring + (size_t)aslot * AH_BLOCK_BYTES, &a_ring_full[aslot], kb, tile);
                                if (++aslot == p.a_slots) { aslot = 0; aphase ^= 1; }
                            }
                            for (int h = 0; h < halves; ++h) {
                                DSAT_TIMED_WAIT(w1, mbar_wait(&ring_empty[slot], phase ^ 1));
                                if constexpr (PAIR) {     // this CTA's half of the weight block: rows [h*256 + rank*bn/2, +bn/2) of W^T
                                    const int bn = min(256, p.layer[l].N - h * 256);
                                    expect(&ring_full[slot], (uint32_t)(bn / 2) * (BLOCK_K * 2));
                                    load_2d(ring + (size_t)slot * p.slot_bytes, map_w[l], &ring_full[slot], kb * BLOCK_K,
                                            h * 256 + (int)rank * (bn / 2));
                                } else {
                                    expect(&ring_full[slot], (uint32_t)p.layer[l].box_rows * (BLOCK_K * 2));
                                    load_2d(ring + (size_t)slot * p.slot_bytes, map_w[l], &ring_full[slot], kb * BLOCK_K, h * 256);
                                }
                                if (++slot == p.slots) { slot = 0; phase ^= 1; }
                            }
                        }
                    }
        }
    } else if (warp == 1) {
        if (leader) {      // ================================ MMA issuer: the whole warp runs the loop converged, one lane issues
            int slot = 0; uint32_t phase = 0;
            int aslot = 0; uint32_t aphase = 0;
            auto commit = [&](uint64_t* bar) {
                if constexpr (PAIR) tcgen05_commit_elect_cg2(bar); else tcgen05_commit_elect(bar);
            };
            for (int j0 = 0; j0 < nt; j0 += group)
                for (int l = 0; l < n_layers; ++l)
                    for (int s = 0; s < group; ++s) {
                        if (j0 + s >= nt) continue;
                        const Step st = make_step(j0, s, l);
                        const int j = j0 + s;
                        DSAT_TIMED_WAIT(w0, mbar_wait(&tmem_empty[st.buf], (uint32_t)((st.use & 1) ^ 1)));   // accumulator drained
                        const bool streamed = l == 0 && p.a_slots > 0;
                        if (l == 0) { if (!streamed) DSAT_TIMED_WAIT(w1, mbar_wait(a_full, (uint32_t)(j & 1))); }
                        else DSAT_TIMED_WAIT(w2, mbar_wait(&h_full[st.hidx], (uint32_t)(st.hcnt & 1)));
                        tcgen05_fence_after();
                        const int K = p.layer[l].K, N = p.layer[l].N;
                        const int kbs = (K + BLOCK_K - 1) / BLOCK_K;
                        const int halves = (N + 255) / 256;
                        const uint32_t acc = tmem_base + (uint32_t)(st.buf * 256);
                        const uint8_t* a_src = ah + (size_t)st.hidx * h_bytes;
                        const long long t_kb0 = timing ? clock64() : 0;
                        for (int kb = 0; kb < kbs; ++kb) {
                            // (no tcgen05 fence after the ring waits: TMA writes and MMA reads are both async-proxy accesses
                            //  ordered by the mbarrier; the fences that matter are the per-step ones above)
                            if (streamed) { DSAT_TIMED_WAIT(w1, mbar_wait(&a_ring_full[aslot], aphase)); }
                            const uint64_t da = make_smem_desc_sw128(smem_u32(streamed ? a_ring + (size_t)aslot * AH_BLOCK_BYTES
                                                                                       : a_src + (size_t)kb * AH_BLOCK_BYTES));
                            const int ksteps = min(BLOCK_K / 16, (K - kb * BLOCK_K + 15) / 16);
                            for (int h = 0; h < halves; ++h) {
                                const int bn = min(256, N - h * 256);
                                const uint32_t idesc = make_idesc_bf16(PAIR ? 2 * BLOCK_M : BLOCK_M, bn);
                                DSAT_TIMED_WAIT(w3, mbar_wait(&ring_full[slot], phase));
                                const uint64_t db = make_smem_desc_sw128(smem_u32(ring + (size_t)slot * p.slot_bytes));
                                const long long t_i0 = timing ? clock64() : 0;
                                const uint32_t acc_h = acc + (uint32_t)(h * 256);
                                if (ksteps == BLOCK_K / 16) {       // full K block: four MMAs and the slot's commit in one go
                                    if constexpr (PAIR) umma_bf16_kblock_commit_elect_cg2(acc_h, da, db, idesc, kb != 0, &ring_empty[slot]);
                                    else umma_bf16_kblock_commit_elect(acc_h, da, db, idesc, kb != 0, &ring_empty[slot]);
                                } else {
                                    for (int k = 0; k < ksteps; ++k) {
                                        if constexpr (PAIR) umma_bf16_elect_cg2(acc_h, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kb | k) != 0);
                                        else umma_bf16_elect(acc_h, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kb | k) != 0);
                                    }
                                    commit(&ring_empty[slot]);
                                }
                                const long long t_i1 = timing ? clock64() : 0;
                                if (timing) { w4 += t_i1 - t_i0; w5 += clock64() - t_i1; }
                                if (++slot == p.slots) { slot = 0; phase ^= 1; }
                            }
                            if (streamed) {
                                commit(&a_ring_empty[aslot]);
                                if (++aslot == p.a_slots) { aslot = 0; aphase ^= 1; }
                            }
                        }
                        const long long t_kb1 = timing ? clock64() : 0;
                        commit(&tmem_full[st.buf]);
                        if (l == n_layers - 1 && p.a_slots == 0) commit(ah_free);
                        if (timing) { w6 += t_kb1 - t_kb0; w7 += clock64() - t_kb1; }
                    }
        }
    } else {               // ================================ epilogue warps (4 or 8)
        const int quad = warp & 3;
        EpiCtx e;
        e.r = quad * 32 + lane;                            // row inside the tile = TMEM lane
        e.lane = lane;
        e.cpar = (warp - 2) >> 2;                          // which 32-column chunks of the quadrant this warp takes
        e.cstep = 32 * (p.epi_warps >> 2);
        e.stage_row = p.stage_row;
        e.qmaps = p.qmaps;
        e.ptr0 = p.out.ptr0; e.ptr1 = p.out.ptr1; e.ld0 = p.out.ld0; e.ld1 = p.out.ld1;
        e.bf0 = p.out.bf16_0; e.bf1 = p.out.bf16_1; e.split = p.out.split;
        const uint32_t bias_addr0 = smem_u32(bias_s);
        const uint32_t stage_off = (uint32_t)(warp - 2) * (32 * p.stage_row);
        for (int j0 = 0; j0 < nt; j0 += group)
            for (int l = 0; l < n_layers; ++l)
                for (int s = 0; s < group; ++s) {
                    if (j0 + s >= nt) continue;
                    const Step st = make_step(j0, s, l);
                    e.row_first = (size_t)st.tile * BLOCK_M + quad * 32;
                    e.rows_left = p.rows - (int)e.row_first;
                    DSAT_CHECK(st.tile >= 0 && st.tile <= p.n_tiles);
                    e.ah_addr = smem_u32(ah + (size_t)st.hidx * h_bytes);
                    e.stage_addr = (p.stage_in_h ? e.ah_addr + (uint32_t)p.stage_off : smem_u32(stage_all)) + stage_off;
                    e.N = p.layer[l].N; e.epi = p.layer[l].epi;
                    e.bl_addr = bias_addr0 + 4u * (uint32_t)p.layer[l].bias_off;
                    e.lane_addr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(st.buf * 256);
                    DSAT_TIMED_WAIT(w0, mbar_wait(&tmem_full[st.buf], (uint32_t)(st.use & 1)));
                    tcgen05_fence_after();
                    const long long t_epi0 = timing ? clock64() : 0;
                    const uint32_t empty_addr = at_leader(&tmem_empty[st.buf]);
                    if (l + 1 < n_layers) {
                        epi_drain<true, PAIR>(e, empty_addr);
                        tcgen05_fence_before();
                        // st.shared -> visible to the MMA (async proxy)
                        // (pair mode too: the hidden activations are the A operand, which each CTA's tensor core reads from its
                        //  OWN shared memory; only B halves cross the pair.  The all-spaces form of the fence made the
                        //  hidden epilogues of the pair instantiation 2.4x slower.)
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        __syncwarp();
                        if (lane == 0) { arrive_addr<PAIR>(empty_addr); arrive_addr<PAIR>(at_leader(&h_full[st.hidx])); }
                        if (timing) w1 += clock64() - t_epi0;
                    } else {
                        epi_drain<false, PAIR>(e, empty_addr);
                        // staging inside the hidden region: no epilogue warp may start writing the next hidden activations
                        // there while another one still reads back its staged output (named barrier of the epilogue warps)
                        if (p.stage_in_h) asm volatile("bar.sync 1, %0;" ::"r"(epi_threads) : "memory");
                        if (timing) w2 += clock64() - t_epi0;
                    }
                }
    }
    if (timing && lane == 0 && (warp == 0 || warp == 1 || warp == 2)) {
        // [0] kernel cycles; producer: [1] ah_free wait [2] ring_empty wait; MMA: [3] tmem_empty wait [4] a_full wait
        // [5] h_full wait [6] ring_full wait; epilogue warp 2: [7] tmem_full wait [8] hidden epilogues [9] final epilogues
        const long long total = clock64() - t_kernel0;
        if (warp == 0) { p.prof[0] = total; p.prof[1] = w0; p.prof[2] = w1; }
        if (warp == 1) { p.prof[3] = w0; p.prof[4] = w1; p.prof[5] = w2; p.prof[6] = w3; p.prof[10] = total; p.prof[12] = w4; p.prof[13] = w5; p.prof[14] = w6; p.prof[15] = w7; }
        if (warp == 2) { p.prof[7] = w0; p.prof[8] = w1; p.prof[9] = w2; p.prof[11] = total; }
    }
    (void)w4; (void)w5; (void)w6; (void)w7;
    tcgen05_fence_before();
    __syncthreads();
    if constexpr (PAIR) cluster_sync_all();              // the leader's MMAs may still read this CTA's shared memory
    if (warp == 1) {
        tcgen05_fence_after();
        if constexpr (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS));
        else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS));
    }
}


// ---- Split mode: an MLP whose hidden layers are 512 wide (the literal MLP: 144 -> 512 -> 512 -> 256) fills all 512
// TMEM columns with one layer, so in fused_mlp_kernel every epilogue runs with the tensor pipe idle -- and draining
// TMEM is slow (about 64 B per cycle and SM: 8 N cycles for a [128, N] fp32 accumulator against N K / 32 for its MMAs).
// Here the work of a tile is a sequence of STEPS of at most 256 columns,
//        L1[0:256) L1[256:512) L2[0:256) L2[256:512) L3
// that alternate between the two accumulator halves (step g uses half g & 1, across tiles too), so the epilogue of one
// step runs under the MMAs of the next one wherever the data allow it:
//   * a layer reading the hidden region waits for blocks 0-3 (h_full[0]) before k-block 0 and for blocks 4-7
//     (h_full[1]) before k-block 4: L2's first half starts while L1's second half is still draining;
//   * the epilogue of a first half overwrites shared memory that the second half's MMAs still read (the input tile,
//     or the previous hidden layer), so it also waits for the NEXT step's tmem_full (FmStep::wait_next);
//   * the last step's output drains while the next tile's first step already accumulates in the other half.
// Input tile resident in AH (blocks 0 ..), one hidden region, weight ring as in fused_mlp_kernel.
template <bool PAIR>
__global__ void __launch_bounds__(MAX_THREADS, 1)
fused_mlp_split_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w0, const __grid_constant__ CUtensorMap map_w1,
                       const __grid_constant__ CUtensorMap map_w2, FmParams p) {
    using namespace tc;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    if ((int)(smem - smem_raw) > p.smem_pad) __trap();
    uint8_t* ah = smem;
    uint8_t* ring = smem + (size_t)p.ah_blocks * AH_BLOCK_BYTES;
    uint8_t* stage_all = ring + (size_t)p.slots * p.slot_bytes;
    uint8_t* tail = stage_all + (p.stage_in_h ? 0 : (size_t)p.epi_warps * 32 * p.stage_row);
    uint64_t* a_full = reinterpret_cast<uint64_t*>(tail);
    uint64_t* ah_free = a_full + 1;
    uint64_t* h_full = a_full + 2;                     // [2]: hidden blocks 0-3 / 4-7 written
    uint64_t* tmem_full = a_full + 4;                  // [2]
    uint64_t* tmem_empty = a_full + 6;                 // [2]
    uint64_t* ring_full = a_full + 8;                  // [MAX_SLOTS]
    uint64_t* ring_empty = a_full + 8 + MAX_SLOTS;     // [MAX_SLOTS]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(a_full + 8 + 2 * MAX_SLOTS + 2 * MAX_A_SLOTS);
    float* bias_s = reinterpret_cast<float*>(tail + BAR_BYTES);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int epi_threads = 32 * p.epi_warps;
    const CUtensorMap* map_w[MAX_LAYERS] = {&map_w0, &map_w1, &map_w2};
    // PAIR (clusters of 2, cta_group::2, as in fused_mlp_kernel): rank 0 leads and issues M = 256 MMAs; each CTA loads its own
    // 128 input rows and HALF of every weight block; "full" barriers live in the leader and count both CTAs, "empty"
    // barriers and tmem_full are local and get the leader's multicast commits.
    const uint32_t rank = PAIR ? cluster_rank() : 0u;
    const bool leader = rank == 0;
    constexpr int NC = PAIR ? 2 : 1;
    auto at_leader = [&](uint64_t* bar) -> uint32_t { return PAIR ? mapa_rank(smem_u32(bar), 0) : smem_u32(bar); };
    if (threadIdx.x == 0) {
        mbar_init(a_full, NC);
        mbar_init(ah_free, 1);
        for (int b = 0; b < 2; ++b) {
            mbar_init(&h_full[b], NC * p.epi_warps);
            mbar_init(&tmem_full[b], 1);
            mbar_init(&tmem_empty[b], NC * p.epi_warps);
        }
        for (int s = 0; s < MAX_SLOTS; ++s) { mbar_init(&ring_full[s], NC); mbar_init(&ring_empty[s], 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w0) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w1) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w2) : "memory");
    }
    if (warp == 1) {
        if constexpr (PAIR) {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS));
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS));
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    if constexpr (PAIR) cluster_sync_all();              // both CTAs' barriers exist before any remote arrive
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int nv = p.n_steps;
    // work units: 128-row tiles of this CTA, or (PAIR) 256-row macro tiles of the pair, of which this CTA owns one half
    const int unit0 = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int unit_stride = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    const int n_units = PAIR ? (p.n_tiles + 1) / 2 : p.n_tiles;
    const int nt = unit0 < n_units ? (n_units - unit0 + unit_stride - 1) / unit_stride : 0;
    auto tile_of = [&](int j) { const int u = unit0 + j * unit_stride; return PAIR ? 2 * u + (int)rank : u; };
    const int n_hidden = p.n_layers - 1;

    if (warp == 0) {
        if (lane == 0) {   // ================================ TMA producer
            const int k0_blocks = (p.layer[0].K + BLOCK_K - 1) / BLOCK_K;
            int slot = 0; uint32_t phase = 0;
            for (int j = 0; j < nt; ++j) {
                const int tile = tile_of(j);
                for (int v = 0; v < nv; ++v) {
                    const FmStep st = p.step[v];
                    if (v == 0) {      // the input tile into AH, once the previous tile's last layer no longer reads it
                        if (j > 0) mbar_wait(ah_free, (uint32_t)((j - 1) & 1));
                        if constexpr (PAIR) mbar_expect_tx_at(at_leader(a_full), (uint32_t)(k0_blocks * p.a_box_rows) * (BLOCK_K * 2));
                        else mbar_expect_tx(a_full, (uint32_t)(k0_blocks * p.a_box_rows) * (BLOCK_K * 2));
                        for (int kb = 0; kb < k0_blocks; ++kb) {
                            if constexpr (PAIR) tma_load_2d_cg2(ah + (size_t)kb * AH_BLOCK_BYTES, &map_a, at_leader(a_full), kb * BLOCK_K, tile * BLOCK_M);
                            else tma_load_2d(ah + (size_t)kb * AH_BLOCK_BYTES, &map_a, a_full, kb * BLOCK_K, tile * BLOCK_M);
                        }
                    }
                    const int kbs = (p.layer[st.layer].K + BLOCK_K - 1) / BLOCK_K;
                    for (int kb = 0; kb < kbs; ++kb) {
                        mbar_wait(&ring_empty[slot], phase ^ 1);
                        if constexpr (PAIR) {      // this CTA's half of the step's weight rows (the maps have half-height boxes)
                            mbar_expect_tx_at(at_leader(&ring_full[slot]), (uint32_t)(st.N / 2) * (BLOCK_K * 2));
                            tma_load_2d_cg2(ring + (size_t)slot * p.slot_bytes, map_w[st.layer], at_leader(&ring_full[slot]), kb * BLOCK_K,
                                            st.n0 + (int)rank * (st.N / 2));
                        } else {
                            mbar_expect_tx(&ring_full[slot], (uint32_t)p.layer[st.layer].box_rows * (BLOCK_K * 2));
                            tma_load_2d(ring + (size_t)slot * p.slot_bytes, map_w[st.layer], &ring_full[slot], kb * BLOCK_K, st.n0);
                        }
                        if (++slot == p.slots) { slot = 0; phase ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 1) {    // ================================ MMA issuer (whole warp converged, one elected lane issues)
        int slot = 0; uint32_t phase = 0;
        auto commit = [&](uint64_t* bar) { if constexpr (PAIR) tcgen05_commit_elect_cg2(bar); else tcgen05_commit_elect(bar); };
        if (leader)
        for (int j = 0; j < nt; ++j)
            for (int v = 0; v < nv; ++v) {
                const FmStep st = p.step[v];
                const int g = j * nv + v, buf = g & 1, use = g >> 1;
                mbar_wait(&tmem_empty[buf], (uint32_t)((use & 1) ^ 1));          // this accumulator half is drained
                if (st.layer == 0) mbar_wait(a_full, (uint32_t)(j & 1));
                tcgen05_fence_after();
                const int K = p.layer[st.layer].K;
                const int kbs = (K + BLOCK_K - 1) / BLOCK_K;
                const uint32_t idesc = make_idesc_bf16(PAIR ? 2 * BLOCK_M : BLOCK_M, st.N);
                const uint32_t acc = tmem_base + (uint32_t)(buf * 256);
                const uint32_t hphase = (uint32_t)((j * n_hidden + (st.layer - 1)) & 1);
                for (int kb = 0; kb < kbs; ++kb) {
                    if (st.layer > 0 && (kb & 3) == 0) {      // the next four hidden blocks are in shared memory
                        mbar_wait(&h_full[kb >> 2], hphase);
                        tcgen05_fence_after();
                    }
                    const uint64_t da = make_smem_desc_sw128(smem_u32(ah + (size_t)kb * AH_BLOCK_BYTES));
                    const int ksteps = min(BLOCK_K / 16, (K - kb * BLOCK_K + 15) / 16);
                    mbar_wait(&ring_full[slot], phase);
                    const uint64_t db = make_smem_desc_sw128(smem_u32(ring + (size_t)slot * p.slot_bytes));
                    if (ksteps == BLOCK_K / 16) {
                        if constexpr (PAIR) umma_bf16_kblock_commit_elect_cg2(acc, da, db, idesc, kb != 0, &ring_empty[slot]);
                        else umma_bf16_kblock_commit_elect(acc, da, db, idesc, kb != 0, &ring_empty[slot]);
                    } else {
                        for (int k = 0; k < ksteps; ++k) {
                            if constexpr (PAIR) umma_bf16_elect_cg2(acc, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kb | k) != 0);
                            else umma_bf16_elect(acc, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kb | k) != 0);
                        }
                        commit(&ring_empty[slot]);
                    }
                    if (++slot == p.slots) { slot = 0; phase ^= 1; }
                }
                commit(&tmem_full[buf]);
                if (v == nv - 1) commit(ah_free);
            }
    } else {               // ================================ epilogue warps
        const int quad = warp & 3;
        EpiCtx e;
        e.r = quad * 32 + lane;
        e.lane = lane;
        e.cpar = (warp - 2) >> 2;
        e.cstep = 32 * (p.epi_warps >> 2);
        e.stage_row = p.stage_row;
        e.qmaps = p.qmaps;
        e.ptr0 = p.out.ptr0; e.ptr1 = p.out.ptr1; e.ld0 = p.out.ld0; e.ld1 = p.out.ld1;
        e.bf0 = p.out.bf16_0; e.bf1 = p.out.bf16_1; e.split = p.out.split;
        const uint32_t stage_off = (uint32_t)(warp - 2) * (32 * p.stage_row);
        e.stage_addr = (p.stage_in_h ? smem_u32(ah) + (uint32_t)p.stage_off : smem_u32(stage_all)) + stage_off;
        // the biases of the step after this one travel from global memory into registers while this step
        // is processed, and into one of two 256-float shared buffers at the start of their step
        const int et = (int)threadIdx.x - 64;
        float bnext[2] = {0.f, 0.f};
        auto fetch_bias = [&](int v) {
            const FmStep s = p.step[v];
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const int i = et + k * epi_threads;
                bnext[k] = i < s.N ? __ldg(p.layer[s.layer].bias + s.n0 + i) : 0.f;
            }
        };
        if (nt > 0) fetch_bias(0);
        for (int j = 0; j < nt; ++j) {
            const int tile = tile_of(j);
            e.row_first = (size_t)tile * BLOCK_M + quad * 32;
            e.rows_left = p.rows - (int)e.row_first;
            for (int v = 0; v < nv; ++v) {
                const FmStep st = p.step[v];
                const int g = j * nv + v, buf = g & 1, use = g >> 1;
                e.N = st.N; e.epi = p.layer[st.layer].epi;
                float* dst = bias_s + (g & 1) * 256;      // last read two steps ago; every warp passed the previous step's barrier since
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    const int i = et + k * epi_threads;
                    if (i < 256) dst[i] = bnext[k];
                }
                fetch_bias(v + 1 < nv ? v + 1 : 0);
                asm volatile("bar.sync 2, %0;" ::"r"(epi_threads) : "memory");
                e.bl_addr = smem_u32(dst);
                e.ah_addr = smem_u32(ah) + (uint32_t)(st.n0 >> 6) * AH_BLOCK_BYTES;
                e.lane_addr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(buf * 256);
                mbar_wait(&tmem_full[buf], (uint32_t)(use & 1));
                if (st.wait_next) mbar_wait(&tmem_full[buf ^ 1], (uint32_t)(((g + 1) >> 1) & 1));
                tcgen05_fence_after();
                const uint32_t empty_addr = at_leader(&tmem_empty[buf]);
                if (st.hidden) {
                    epi_drain<true, PAIR>(e, empty_addr);
                    tcgen05_fence_before();
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) { arrive_addr<PAIR>(empty_addr); arrive_addr<PAIR>(at_leader(&h_full[st.n0 >> 8])); }
                } else {
                    epi_drain<false, PAIR>(e, empty_addr);
                    if (p.stage_in_h) asm volatile("bar.sync 1, %0;" ::"r"(epi_threads) : "memory");
                }
            }
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    if constexpr (PAIR) cluster_sync_all();              // the leader's MMAs may still read this CTA's shared memory
    if (warp == 1) {
        tcgen05_fence_after();
        if constexpr (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS));
        else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS));
    }
}

struct FusedMlp {
    CUtensorMap map_a;
    CUtensorMap map_w[MAX_LAYERS];
    FmParams p;
    int smem_bytes;
    CUtensorMap map_wp[MAX_LAYERS];     // weight maps with half-height boxes (CTA-pair mode: each CTA loads half a block)
    bool stream_input = false;      // request the input ring (FmParams::a_slots), set before plan_fused
    bool pair_mode = false;         // request the CTA-pair instantiation: half-height weight slots (map_wp), clusters of 2
};

// Dynamic shared memory has to start on a 1024-byte boundary (SWIZZLE_128B atoms).  The base is that well aligned in
// practice; a one-off probe checks it so that the plans do not have to give up 1 KB (the clause MLP's ping-pong plan
// fits with a few hundred bytes to spare).  The kernel traps if a base ever needs more than the planned pad.
__global__ void smem_base_probe_kernel(unsigned* out) {
    extern __shared__ __align__(1024) uint8_t probe_raw[];
    *out = tc::smem_u32(probe_raw);
}
inline int dyn_smem_pad() {
    static int pads[64];
    static PerDeviceOnce probed;
    const int dev_id = PerDeviceOnce::current();
    if (dev_id < 0) return 1024;
    int& pad = pads[dev_id];
    if (probed.done()) return pad;
    probed.mark();
    pad = 1024;
    unsigned* dev = nullptr;
    unsigned host = 1;
    if (cudaMalloc(&dev, sizeof(unsigned)) != cudaSuccess) return pad;
    cudaFuncSetAttribute(smem_base_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT);
    smem_base_probe_kernel<<<1, 1, SMEM_LIMIT>>>(dev);
    if (cudaMemcpy(&host, dev, sizeof(unsigned), cudaMemcpyDeviceToHost) == cudaSuccess && (host & 1023u) == 0) pad = 0;
    cudaFree(dev);
    return pad;
}

constexpr int PAIR_A_SLOTS = 4;     // input-ring cap of a CTA pair that streams one tile at a time
// half-height weight slots reserved before the input ring gets the rest (CTA pair + ping-pong): the update MLP measured
// 0.263 / 0.230 / 0.245 ms with 4 / 3 / 2 (input ring 2 / 3 / 4)
constexpr int PAIR_PP_WMIN = 3;

// shared-memory plan; returns false when the MLP does not fit
inline bool plan_fused(FusedMlp& f) {
    FmParams& p = f.p;
    int blocks = (p.layer[0].K + 63) / 64;
    const int pad = dyn_smem_pad();
    p.smem_pad = pad;
    int bias_total = 0, max_box = 0;
    p.two_bufs = 1;
    p.a_slots = 0;
    p.pp = 0;
    p.split = 0;
    p.n_steps = 0;
    p.stage_in_h = 0;
    p.stage_off = 0;
    for (int l = 0; l < p.n_layers; ++l) {
        if (l + 1 < p.n_layers) blocks = max(blocks, (p.layer[l].N + 63) / 64);
        p.layer[l].bias_off = bias_total;
        bias_total += (p.layer[l].N + 31) / 32 * 32;
        max_box = max(max_box, p.layer[l].box_rows);
        if (p.layer[l].N > 256) p.two_bufs = 0;
    }
    p.ah_blocks = blocks;
    p.bias_total = bias_total;
    // CTA pair: needs equal weight halves per MMA (N <= 256, or a multiple of 256) and at least one full macro tile
    bool pair = f.pair_mode && p.rows > BLOCK_M;
    for (int l = 0; l < p.n_layers; ++l) {
        const int N = p.layer[l].N;
        if (N % 16 || (N > 256 && N % 256)) pair = false;
    }
    p.pair = pair ? 1 : 0;
    p.slot_bytes = ((pair ? max_box / 2 : max_box) * BLOCK_K * 2 + 1023) / 1024 * 1024;
    p.n_tiles = ceil_div(p.rows, BLOCK_M);
    {
        const FmLayer& last = p.layer[p.n_layers - 1];
        const bool all_bf16 = p.out.bf16_0 && (p.out.ptr1 == nullptr || p.out.bf16_1) && last.epi != tc::TC_QUERY;
        p.stage_row = all_bf16 ? 80 : STAGE_ROW;
    }
    p.a_slots = 0;
    p.epi_warps = 4;
    if (f.stream_input && p.n_layers > 1) {
        // streamed input: AH keeps hidden activations only; the input gets its own ring (as deep as fits next to two
        // weight slots and eight epilogue warps, at most two tiles' worth)
        int h_blocks = 1;
        for (int l = 0; l + 1 < p.n_layers; ++l) h_blocks = max(h_blocks, (p.layer[l].N + 63) / 64);
        const int k0_blocks = (p.layer[0].K + 63) / 64;
        if (p.two_bufs) {
            // two tiles in flight: two hidden regions; a tile's output staging aliases its own hidden region when it fits
            for (int ew : {8, 4}) {
                const int h_bytes = h_blocks * AH_BLOCK_BYTES, stage_bytes = ew * 32 * p.stage_row;
                const int in_h = stage_bytes <= h_bytes;
                const int fixed = pad + 2 * h_bytes + (in_h ? 0 : stage_bytes) + BAR_BYTES + bias_total * 4;
                // weight slots to reserve before the input ring gets the rest: four half-height ones in pair mode
                int w_min = p.pair ? PAIR_PP_WMIN : 2;
                if (SMEM_LIMIT - fixed - w_min * p.slot_bytes < 2 * AH_BLOCK_BYTES) w_min = 2;
                int a_slots = (SMEM_LIMIT - fixed - w_min * p.slot_bytes) / AH_BLOCK_BYTES;
                if (a_slots > 2 * k0_blocks) a_slots = 2 * k0_blocks;
                if (a_slots > MAX_A_SLOTS) a_slots = MAX_A_SLOTS;
                if (SMEM_LIMIT - fixed - w_min * p.slot_bytes < 0 || a_slots < 2) continue;
                p.pp = 1; p.stage_in_h = in_h; p.a_slots = a_slots; p.epi_warps = ew; p.ah_blocks = h_blocks;
                const int base = fixed + a_slots * AH_BLOCK_BYTES;
                for (int slots = MAX_SLOTS; slots >= 2; --slots)
                    if (base + slots * p.slot_bytes <= SMEM_LIMIT) { p.slots = slots; f.smem_bytes = base + slots * p.slot_bytes; break; }
                return true;
            }
        }
        for (int ew : {8, 4}) {
            // one tile at a time: the final epilogue can still stage through the (dead) hidden region; three weight slots
            // are reserved before the input ring takes the rest
            const int stage_bytes = ew * 32 * p.stage_row;
            const int in_h = stage_bytes <= h_blocks * AH_BLOCK_BYTES;
            int w_min = 3;
            int fixed = pad + h_blocks * AH_BLOCK_BYTES + w_min * p.slot_bytes + (in_h ? 0 : stage_bytes) + BAR_BYTES + bias_total * 4;
            if (SMEM_LIMIT - fixed < 2 * AH_BLOCK_BYTES) { fixed -= p.slot_bytes; w_min = 2; }
            int a_slots = (SMEM_LIMIT - fixed) / AH_BLOCK_BYTES;
            if (a_slots > 2 * k0_blocks) a_slots = 2 * k0_blocks;
            if (a_slots > MAX_A_SLOTS) a_slots = MAX_A_SLOTS;
            // CTA pair: weight slots are half-height (as large as an input block) and the in-order producer never runs the
            // input ring further ahead than the weight ring lets it: the weight ring gets the larger share
            if (p.pair && a_slots > PAIR_A_SLOTS) a_slots = PAIR_A_SLOTS;
            fixed -= (w_min - 2) * p.slot_bytes;          // `fixed` below counts two weight slots
            if (a_slots >= 2 && a_slots >= (k0_blocks + 1) / 2) {
                p.a_slots = a_slots;
                p.epi_warps = ew;
                p.ah_blocks = h_blocks;
                p.stage_in_h = in_h;
                p.stage_off = 0;
                const int base = fixed - 2 * p.slot_bytes + a_slots * AH_BLOCK_BYTES;
                for (int slots = MAX_SLOTS; slots >= 2; --slots)
                    if (base + slots * p.slot_bytes <= SMEM_LIMIT) { p.slots = slots; f.smem_bytes = base + slots * p.slot_bytes; break; }
                return true;
            }
        }
    }
    // Resident-input mode.  The final epilogue may stage through the part of AH above the input blocks: the hidden
    // activations there are dead once the last layer's MMAs have completed, the next tile's input only overwrites the
    // first k0 blocks, and the next hidden epilogue comes after this one in the same warps' program order.
    const int k0_blocks_res = (p.layer[0].K + 63) / 64;
    // split mode: every hidden layer exactly 512 wide (two accumulator halves, two h_full halves), output <= 256
    bool split = p.n_layers >= 2 && p.layer[p.n_layers - 1].N <= 256 && p.rows > 0;
    for (int l = 0; l + 1 < p.n_layers; ++l) split = split && p.layer[l].N == 512;
    const int bias_bytes = split ? 2 * 256 * 4 : bias_total * 4;
    for (int ew : {8, 4}) {     // prefer 8 epilogue warps when two ring slots still fit
        const int stage_bytes = ew * 32 * p.stage_row;
        const int in_h = p.n_layers > 1 && (blocks - k0_blocks_res) * AH_BLOCK_BYTES >= stage_bytes;
        if (pad + blocks * AH_BLOCK_BYTES + 2 * p.slot_bytes + (in_h ? 0 : stage_bytes) + BAR_BYTES + bias_bytes <= SMEM_LIMIT) {
            p.epi_warps = ew;
            p.stage_in_h = in_h;
            p.stage_off = in_h ? k0_blocks_res * AH_BLOCK_BYTES : 0;
            break;
        }
    }
    for (int slots = MAX_SLOTS; slots >= 2; --slots) {
        const int total = pad + blocks * AH_BLOCK_BYTES + slots * p.slot_bytes + (p.stage_in_h ? 0 : p.epi_warps * 32 * p.stage_row) + BAR_BYTES + bias_bytes;
        if (total <= SMEM_LIMIT) {
            p.slots = slots;
            f.smem_bytes = total;
            if (split) {
                int n = 0;
                for (int l = 0; l < p.n_layers; ++l) {
                    const bool hidden = l + 1 < p.n_layers;
                    for (int n0 = 0; n0 < p.layer[l].N; n0 += 256) {
                        FmStep& st = p.step[n++];
                        st.layer = (short)l; st.n0 = (short)n0; st.N = (short)min(256, p.layer[l].N - n0);
                        st.hidden = hidden ? 1 : 0;
                        st.wait_next = hidden && n0 + 256 < p.layer[l].N ? 1 : 0;
                    }
                }
                p.n_steps = n;
                p.split = 1;
            }
            return true;
        }
    }
    return false;
}

inline cudaError_t configure_fused_device() {
    static PerDeviceOnce configured;        // MaxDynamicSharedMemorySize is a per-device function attribute
    if (configured.done()) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(fused_mlp_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(fused_mlp_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(fused_mlp_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(fused_mlp_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(fused_mlp_split_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(fused_mlp_split_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT);
    if (e == cudaSuccess) configured.mark();
    return e;
}

inline cudaError_t launch_fused(const FusedMlp& f, int sm_count, cudaStream_t stream) {
    if (f.p.rows <= 0) return cudaSuccess;
    {
        cudaError_t e = configure_fused_device();
        if (e != cudaSuccess) return e;
    }
    const unsigned threads = 64 + 32 * f.p.epi_warps;
    const int last = f.p.n_layers > 2 ? 2 : 1;
    if (f.p.pair) {     // clusters of two CTAs, one 256-row macro tile per pair and pass; weight maps with half-height boxes
        const int n_macro = (f.p.n_tiles + 1) / 2;
        const int pairs = n_macro < sm_count / 2 ? n_macro : sm_count / 2;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(2 * pairs); cfg.blockDim = dim3(threads); cfg.dynamicSmemBytes = (size_t)f.smem_bytes; cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        if (f.p.split) return cudaLaunchKernelEx(&cfg, fused_mlp_split_kernel<true>, f.map_a, f.map_wp[0], f.map_wp[1], f.map_wp[last], f.p);
        if (f.p.prof) return cudaLaunchKernelEx(&cfg, fused_mlp_kernel<true, true>, f.map_a, f.map_wp[0], f.map_wp[1], f.map_wp[last], f.p);
        return cudaLaunchKernelEx(&cfg, fused_mlp_kernel<false, true>, f.map_a, f.map_wp[0], f.map_wp[1], f.map_wp[last], f.p);
    }
    const unsigned grid = (unsigned)(f.p.n_tiles < sm_count ? f.p.n_tiles : sm_count);
    if (f.p.split) {    // (no instrumented build of the split kernel: dsat_profile_fused reads zeros for it)
        fused_mlp_split_kernel<false><<<grid, threads, f.smem_bytes, stream>>>(f.map_a, f.map_w[0], f.map_w[1], f.map_w[last], f.p);
        return cudaGetLastError();
    }
    if (f.p.prof)   // instrumented build of the same kernel (dsat_profile_fused)
        fused_mlp_kernel<true, false><<<grid, threads, f.smem_bytes, stream>>>(f.map_a, f.map_w[0], f.map_w[1], f.map_w[last], f.p);
    else
        fused_mlp_kernel<false, false><<<grid, threads, f.smem_bytes, stream>>>(f.map_a, f.map_w[0], f.map_w[1], f.map_w[last], f.p);
    return cudaGetLastError();
}

}  // namespace fm
}  // namespace dsat
