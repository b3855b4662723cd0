// fp32-accurate whole-MLP kernel on the 5th-gen tensor cores ("x3": three bf16 split products per fp32 product).
//
// The reference computes every Dense layer in fp32 (model/mlp.py:24,39; call sites model/query_sat.py:240,252,261,
// 278,283).  bf16 operands alone give 2^-9 relative error per product; here every fp32 value v is carried as two
// bf16 planes  hi = bf16(v), lo = bf16(v - hi)  (v = hi + lo up to 2^-17 |v|) and a product of activations x and
// weights w is accumulated in the SAME fp32 TMEM accumulator as
//         x_hi * w_hi  +  x_lo * w_hi  +  x_hi * w_lo                       (dropped: x_lo * w_lo ~ 2^-18 |x||w|)
// i.e. three kind::f16 tcgen05.mma passes over every K block.  Errors are ~1e-5 relative to |x||w| per product,
// against 4e-3 for plain bf16 and 6e-8 for fp32 FMA chains.
//
// Layout and pipeline (one persistent CTA per SM, or a CTA pair with cta_group::2 when PAIR):
//   global  A operand   : two bf16 planes [rows, lda] (hi, lo), written by the producing kernels (gathers, PairNorm,
//                         noise) in that form; fetched by TMA as SWIZZLE_128B blocks of 128 rows x 64 columns
//           weights     : per layer a stacked K-major array [2 N, K64] (rows [0,N) = hi, [N,2N) = lo)
//   shared  input ring  : 16 KB blocks; a K block of the input occupies two consecutive slots (hi, lo)
//           weight ring : slots of N x 64 (PAIR: N/2 x 64) bf16; per K block first W_hi (multiplies A_hi and A_lo), then W_lo
//   tensor  memory      : two accumulators of <= 256 columns; consecutive (tile, layer) steps alternate between them,
//                         so the final epilogue of a tile drains while the next tile's first layer accumulates
//           hidden      : the activations between layers never leave tensor memory: the epilogue warps read a hidden
//                         accumulator, add bias + leaky relu, split, and store the hi/lo planes back into the columns they
//                         read (tc::tmem_a_kstep has the layout); the next layer's MMAs take them as A operand from there
//                         and accumulate into the other half
//   warps               : 0 = TMA producer, 1 = MMA issuer (+ TMEM alloc), 2.. = 4 or 8 epilogue warps
// A single wide layer (N > 256, the 512-wide layers of lit_query) runs as `n_groups` column groups of 256: the work
// unit is (tile, group) and its output goes to global memory as fp32 rows or as hi/lo planes for the next launch.
#pragma once
#include "dsat_mlp_fused.cuh"

namespace dsat {
namespace x3 {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;
constexpr int BLK_BYTES = BLOCK_M * BLOCK_K * 2;     // 16 KB
constexpr int MAX_LAYERS = 3;
constexpr int MAX_RING = 12;                          // a whole tile of the clause MLP's input: 6 K blocks x 2 planes
constexpr int TMEM_COLS = 512;
constexpr int STAGE_ROW = 128 + 16;
// barrier block: 4 rings of mbarriers, tmem_full[2], tmem_empty[2], h_full[2], the TMEM address; then the early-exit bits
constexpr int SKIP_UNITS = 1024;                      // units per CTA up to which early-exit skipping is evaluated
constexpr int SKIP_OFF = 512;
constexpr int BAR_BYTES = SKIP_OFF + SKIP_UNITS / 8;
static_assert((4 * MAX_RING + 6) * 8 + 4 <= SKIP_OFF, "x3 barriers overlap the early-exit bits");
constexpr int SMEM_LIMIT = 227 * 1024;

enum OutMode : int { OUT_F32 = 0, OUT_SPLIT = 1 };

struct X3Layer {
    int K, N;              // multiples of 16; N <= 256 (the group width for a grouped single layer)
    int epi;               // tc::TC_LINEAR / TC_LRELU / TC_QUERY (query only on the last layer)
    int w_lo_row;          // row of the lo plane in the stacked weight array (= the layer's total N)
    int bias_off;          // offset of this layer's biases in the shared bias array
    int n_total;           // total output columns of the layer (> N only for a grouped single layer)
    const float* bias;
};

struct X3Params {
    int n_layers;
    X3Layer layer[MAX_LAYERS];
    int rows, n_tiles, n_groups, a_box_rows;
    int a_slots, w_slots, w_slot_bytes;
    int epi_warps, smem_pad, bias_total, qmaps, pair;
    int out_mode;          // OUT_F32: out0 = fp32 [rows, ld_out]; OUT_SPLIT: out0 / out1 = bf16 hi / lo planes [rows, ld_out]
    void* out0; void* out1; int ld_out;
    long long* prof;       // optional [9] cycle counters of CTA 0's issue warp and first epilogue warp (nullptr = off)
    // early exit (reference model/query_sat.py:330-338): rows of chain c belong to early-exit group c / chains_per_group;
    // a work unit all of whose rows belong to finished groups is skipped by every warp role (nullptr = never skip)
    const int* done; int rows_per_chain, chains_per_group;
};

// v -> (hi, lo) bf16 pairs of two neighbouring values (dsat_common.cuh)
__device__ __forceinline__ void split2(float v0, float v1, uint32_t& hi, uint32_t& lo) { split_bf16x2(v0, v1, hi, lo); }

struct Epi {
    uint32_t lane_addr, bl_addr, stage_addr;
    int N, epi, cpar, cstep, lane, qmaps, col0;
    size_t row_first; int rows_left;
    void* out0; void* out1; int ld_out, out_mode;
};

// hidden layer: bias + leaky relu in fp32, split, and both planes back into the 32 accumulator columns just read
// (hi of K in [c, c+32) at columns [c, c+16), lo at [c+16, c+32), two bf16 per column, the lower K in the low half):
// the A operand of the next layer's MMAs (tc::tmem_a_kstep).  Columns past N hold values of unused accumulator columns
// and are never read as A: the next layer's K steps stop at its K <= N.
__device__ __forceinline__ void epi_hidden(const Epi& e, const uint32_t (&raw)[32], int c) {
    float v[32];
    fm::bias_act_chunk(raw, e.bl_addr + 4u * (uint32_t)c, e.epi == tc::TC_LRELU, v);
    uint32_t w[32];
#pragma unroll
    for (int i = 0; i < 16; ++i) split2(v[2 * i], v[2 * i + 1], w[i], w[16 + i]);
    fm::tmem_st_32cols(e.lane_addr + (uint32_t)c, w);
}

__device__ __forceinline__ void epi_final(const Epi& e, const uint32_t (&raw)[32], int c) {
    float v[32];
    fm::bias_act_chunk(raw, e.bl_addr + 4u * (uint32_t)c, e.epi == tc::TC_LRELU, v);
    const int valid = min(32, e.N - c);
    const int col = e.col0 + c;
    if (e.out_mode == OUT_SPLIT) {
        uint4 hi[4], lo[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            split2(v[8 * q], v[8 * q + 1], hi[q].x, lo[q].x);
            split2(v[8 * q + 2], v[8 * q + 3], hi[q].y, lo[q].y);
            split2(v[8 * q + 4], v[8 * q + 5], hi[q].z, lo[q].z);
            split2(v[8 * q + 6], v[8 * q + 7], hi[q].w, lo[q].w);
        }
        const size_t pitch = (size_t)e.ld_out * 2;
        fm::store_chunk_packed(e.stage_addr, STAGE_ROW, e.lane, hi, valid, reinterpret_cast<uint8_t*>(e.out0), pitch, e.row_first, e.rows_left, col);
        fm::store_chunk_packed(e.stage_addr, STAGE_ROW, e.lane, lo, valid, reinterpret_cast<uint8_t*>(e.out1), pitch, e.row_first, e.rows_left, col);
        return;
    }
    uint8_t* gbase = reinterpret_cast<uint8_t*>(e.out0);
    const size_t pitch = (size_t)e.ld_out * 4;
    fm::store_chunk_fast<false>(e.stage_addr, STAGE_ROW, e.lane, v, valid, gbase, pitch, e.row_first, e.rows_left, col);
    if (e.epi == tc::TC_QUERY) {      // softplus(+q), softplus(-q) next to the query (reference loss/sat.py:132-133), full precision
        float sp[32], sn[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            // softplus(+-v) = max(+-v, 0) + log(1 + exp(-|v|)) with the fast exponential and logarithm: the query epilogue was
            // the kernel's bottleneck (log1pf + expf: ~40 instructions per element; the issue warp waited 40 % of its time for
            // the epilogue warps).  1 + e is exact to 6e-8 absolute, which is all that exp(-sum softplus) downstream can see.
            const float t = __logf(1.0f + __expf(-fabsf(v[i])));
            sp[i] = fmaxf(v[i], 0.f) + t;
            sn[i] = fmaxf(-v[i], 0.f) + t;
        }
        fm::store_chunk_fast<false>(e.stage_addr, STAGE_ROW, e.lane, sp, valid, gbase, pitch, e.row_first, e.rows_left, col + e.qmaps);
        fm::store_chunk_fast<false>(e.stage_addr, STAGE_ROW, e.lane, sn, valid, gbase, pitch, e.row_first, e.rows_left, col + 2 * e.qmaps);
    }
}

template <bool PAIR>
__global__ void __launch_bounds__(64 + 32 * 8, 1)      // producer + issuer + at most 8 epilogue warps
x3_mlp_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
              const __grid_constant__ CUtensorMap map_w0, const __grid_constant__ CUtensorMap map_w1,
              const __grid_constant__ CUtensorMap map_w2, X3Params p) {
    using namespace tc;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    if ((int)(smem - smem_raw) > p.smem_pad) __trap();
    uint8_t* a_ring = smem;
    uint8_t* w_ring = a_ring + (size_t)p.a_slots * BLK_BYTES;
    uint8_t* stage_all = w_ring + (size_t)p.w_slots * p.w_slot_bytes;
    uint8_t* tail = stage_all + (size_t)p.epi_warps * 32 * STAGE_ROW;
    uint64_t* a_full = reinterpret_cast<uint64_t*>(tail);          // [MAX_RING]
    uint64_t* a_empty = a_full + MAX_RING;
    uint64_t* w_full = a_empty + MAX_RING;
    uint64_t* w_empty = w_full + MAX_RING;
    uint64_t* tmem_full = w_empty + MAX_RING;                       // [2]
    uint64_t* tmem_empty = tmem_full + 2;                           // [2]
    uint64_t* h_full = tmem_empty + 2;                              // [2]: hidden columns [0, 128), [128, 256)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(h_full + 2);
    float* bias_s = reinterpret_cast<float*>(tail + BAR_BYTES);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int epi_threads = 32 * p.epi_warps;
    const CUtensorMap* map_w[MAX_LAYERS] = {&map_w0, &map_w1, &map_w2};
    const CUtensorMap* map_a[2] = {&map_a_hi, &map_a_lo};
    const uint32_t rank = PAIR ? cluster_rank() : 0u;
    const bool leader = rank == 0;
    constexpr int NC = PAIR ? 2 : 1;
    const bool timing = p.prof != nullptr && blockIdx.x == 0;

    if (threadIdx.x == 0) {
        for (int s = 0; s < MAX_RING; ++s) {
            mbar_init(&a_full[s], NC); mbar_init(&a_empty[s], 1);
            mbar_init(&w_full[s], NC); mbar_init(&w_empty[s], 1);
        }
        for (int b = 0; b < 2; ++b) { mbar_init(&tmem_full[b], 1); mbar_init(&tmem_empty[b], NC * p.epi_warps); }
        for (int h = 0; h < 2; ++h) mbar_init(&h_full[h], NC * p.epi_warps);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a_hi) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a_lo) : "memory");
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
    if (warp >= 2 && warp < 2 + p.epi_warps) {
        for (int l = 0; l < p.n_layers; ++l)
            for (int i = threadIdx.x - 64; i < p.layer[l].n_total; i += epi_threads) bias_s[p.layer[l].bias_off + i] = __ldg(p.layer[l].bias + i);
    }
    tcgen05_fence_before();
    __syncthreads();
    if constexpr (PAIR) cluster_sync_all();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int L = p.n_layers, G = p.n_groups;
    auto at_leader = [&](uint64_t* bar) -> uint32_t { return PAIR ? mapa_rank(smem_u32(bar), 0) : smem_u32(bar); };
    // work units: (tile, group) for a CTA, (256-row macro tile, group) for a pair
    const int unit0 = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int unit_stride = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    const int n_units = (PAIR ? (p.n_tiles + 1) / 2 : p.n_tiles) * G;
    const int nt = unit0 < n_units ? (n_units - unit0 + unit_stride - 1) / unit_stride : 0;
    auto tile_of = [&](int j) { const int u = (unit0 + j * unit_stride) / G; return PAIR ? 2 * u + (int)rank : u; };
    auto group_of = [&](int j) { return (unit0 + j * unit_stride) % G; };
    // Units all of whose rows belong to finished early-exit groups are skipped.  Every role must take the same decision (the
    // rings and the accumulator parities count PROCESSED units), and nobody should wait for an L2 round trip per unit on its
    // issue path: the flags of this CTA's units are evaluated once, by all threads, into shared memory (`done` is written by
    // an earlier kernel and constant during this one).  More than SKIP_UNITS units per CTA: no skipping in this launch.
    uint32_t* skip_bits = reinterpret_cast<uint32_t*>(tail + SKIP_OFF);
    const bool skipping = p.done != nullptr && nt <= SKIP_UNITS;
    if (skipping) {
        for (int base = 32 * warp; base < nt; base += (int)blockDim.x) {      // one unit per thread, one 32-bit word per warp pass
            const int j = base + lane;
            bool all = false;
            if (j < nt) {
                const int u = (unit0 + j * unit_stride) / G;
                const int r0 = (PAIR ? 2 * u : u) * BLOCK_M;
                int r1 = r0 + (PAIR ? 2 * BLOCK_M : BLOCK_M);
                r1 = (r1 < p.rows ? r1 : p.rows) - 1;
                const int g0 = (r0 / p.rows_per_chain) / p.chains_per_group, g1 = (r1 / p.rows_per_chain) / p.chains_per_group;
                all = true;
                for (int g = g0; g <= g1 && all; ++g) all = __ldg(p.done + g) != 0;
            }
            const uint32_t bits = __ballot_sync(0xffffffffu, all);
            if (lane == 0) skip_bits[base >> 5] = bits;
        }
        __syncthreads();
    }
    auto unit_done = [&](int j) -> bool { return skipping && ((skip_bits[j >> 5] >> (j & 31)) & 1u) != 0; };

    if (warp == 0) {
        if (lane == 0) {   // ================================ TMA producer
            int as = 0, ws = 0; uint32_t aph = 0, wph = 0;
            for (int j = 0; j < nt; ++j) {
                if (unit_done(j)) continue;
                const int tile = tile_of(j), grp = group_of(j);
                for (int l = 0; l < L; ++l) {
                    const X3Layer& ly = p.layer[l];
                    const int kbs = (ly.K + BLOCK_K - 1) / BLOCK_K;
                    const int wrows = PAIR ? ly.N / 2 : ly.N;
                    for (int kb = 0; kb < kbs; ++kb) {
                        if (l == 0) {
                            for (int pl = 0; pl < 2; ++pl) {
                                mbar_wait(&a_empty[as], aph ^ 1);
                                uint8_t* dst = a_ring + (size_t)as * BLK_BYTES;
                                if constexpr (PAIR) {
                                    mbar_expect_tx_at(at_leader(&a_full[as]), (uint32_t)p.a_box_rows * (BLOCK_K * 2));
                                    tma_load_2d_cg2(dst, map_a[pl], at_leader(&a_full[as]), kb * BLOCK_K, tile * BLOCK_M);
                                } else {
                                    mbar_expect_tx(&a_full[as], (uint32_t)p.a_box_rows * (BLOCK_K * 2));
                                    tma_load_2d(dst, map_a[pl], &a_full[as], kb * BLOCK_K, tile * BLOCK_M);
                                }
                                if (++as == p.a_slots) { as = 0; aph ^= 1; }
                            }
                        }
                        for (int pl = 0; pl < 2; ++pl) {
                            mbar_wait(&w_empty[ws], wph ^ 1);
                            uint8_t* dst = w_ring + (size_t)ws * p.w_slot_bytes;
                            const int row = pl * ly.w_lo_row + grp * 256 + (int)rank * wrows;
                            if constexpr (PAIR) {
                                mbar_expect_tx_at(at_leader(&w_full[ws]), (uint32_t)wrows * (BLOCK_K * 2));
                                tma_load_2d_cg2(dst, map_w[l], at_leader(&w_full[ws]), kb * BLOCK_K, row);
                            } else {
                                mbar_expect_tx(&w_full[ws], (uint32_t)wrows * (BLOCK_K * 2));
                                tma_load_2d(dst, map_w[l], &w_full[ws], kb * BLOCK_K, row);
                            }
                            if (++ws == p.w_slots) { ws = 0; wph ^= 1; }
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (leader) {      // ================================ MMA issuer: whole warp converged, one elected lane issues
            int as = 0, ws = 0; uint32_t aph = 0, wph = 0;
            long long t_wait_acc = 0, t_wait_h = 0, t_wait_a = 0, t_wait_w = 0, t_wait_read = 0;
            const long long t_begin = timing ? clock64() : 0;
            auto commit = [&](uint64_t* bar) { if constexpr (PAIR) tcgen05_commit_elect_cg2(bar); else tcgen05_commit_elect(bar); };
            // hidden layers: A (hi or lo plane) from tensor memory at column ta
            auto kblock_ts = [&](uint32_t acc, uint32_t ta, uint64_t db, uint32_t idesc, uint32_t accum, int ksteps, uint64_t* free_bar) {
                if (ksteps == BLOCK_K / 16) {
                    umma_bf16_ts_kblock_elect<PAIR>(acc, ta, db, idesc, accum);
                } else {
                    for (int k = 0; k < ksteps; ++k)
                        umma_bf16_ts_elect<PAIR>(acc, ta + tmem_a_kstep(k), db + (uint64_t)(2 * k), idesc, (accum | (uint32_t)k) != 0);
                }
                if (free_bar) commit(free_bar);
            };
            auto kblock = [&](uint32_t acc, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accum, int ksteps, uint64_t* free_bar) {
                if (ksteps == BLOCK_K / 16) {
                    if (free_bar) {
                        if constexpr (PAIR) umma_bf16_kblock_commit_elect_cg2(acc, da, db, idesc, accum, free_bar);
                        else umma_bf16_kblock_commit_elect(acc, da, db, idesc, accum, free_bar);
                    } else {
                        if constexpr (PAIR) umma_bf16_kblock_elect_cg2(acc, da, db, idesc, accum);
                        else umma_bf16_kblock_elect(acc, da, db, idesc, accum);
                    }
                } else {
                    for (int k = 0; k < ksteps; ++k) {
                        if constexpr (PAIR) umma_bf16_elect_cg2(acc, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (accum | (uint32_t)k) != 0);
                        else umma_bf16_elect(acc, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (accum | (uint32_t)k) != 0);
                    }
                    if (free_bar) commit(free_bar);
                }
            };
#define X3_WAIT(acc_t, call) do { if (timing) { const long long t0__ = clock64(); call; acc_t += clock64() - t0__; } else { call; } } while (0)
            int jp = 0;         // processed units
            for (int j = 0; j < nt; ++j) {
                if (unit_done(j)) continue;
                for (int l = 0; l < L; ++l) {
                    const int g = jp * L + l, buf = g & 1, use = g >> 1;
                    X3_WAIT(t_wait_acc, mbar_wait(&tmem_empty[buf], (uint32_t)((use & 1) ^ 1)));
                    // Step g - 1 of a hidden layer read its A operand from this half.  The PTX ISA orders tcgen05.mma pairs
                    // only on the same accumulator, so the MMAs writing here wait until those reads have completed (the
                    // commit on tmem_full of step g - 1; the issuer made the next commit to that barrier itself, so the
                    // phase cannot have moved on).
                    if (g > 0 && (l > 0 ? l - 1 : L - 1) > 0)
                        X3_WAIT(t_wait_read, mbar_wait(&tmem_full[buf ^ 1], (uint32_t)(((g - 1) >> 1) & 1)));
                    const uint32_t h_par = (uint32_t)((jp * (L - 1) + (l - 1)) & 1);
                    tcgen05_fence_after();
                    const int K = p.layer[l].K, N = p.layer[l].N;
                    const int kbs = (K + BLOCK_K - 1) / BLOCK_K;
                    const uint32_t idesc = make_idesc_bf16(PAIR ? 2 * BLOCK_M : BLOCK_M, N);
                    const uint32_t acc = tmem_base + (uint32_t)(buf * 256);
                    const uint32_t hid = tmem_base + (uint32_t)((buf ^ 1) * 256);      // layer l - 1's activations
                    for (int kb = 0; kb < kbs; ++kb) {
                        const int ksteps = min(BLOCK_K / 16, (K - kb * BLOCK_K + 15) / 16);
                        if (l == 0) {
                            const int as_hi = as;
                            const uint32_t ph_hi = aph;
                            if (++as == p.a_slots) { as = 0; aph ^= 1; }
                            const int as_lo = as;
                            const uint32_t ph_lo = aph;
                            if (++as == p.a_slots) { as = 0; aph ^= 1; }
                            X3_WAIT(t_wait_a, mbar_wait(&a_full[as_hi], ph_hi));
                            X3_WAIT(t_wait_a, mbar_wait(&a_full[as_lo], ph_lo));
                            const uint64_t da_hi = make_smem_desc_sw128(smem_u32(a_ring + (size_t)as_hi * BLK_BYTES));
                            const uint64_t da_lo = make_smem_desc_sw128(smem_u32(a_ring + (size_t)as_lo * BLK_BYTES));
                            X3_WAIT(t_wait_w, mbar_wait(&w_full[ws], wph));
                            uint64_t db = make_smem_desc_sw128(smem_u32(w_ring + (size_t)ws * p.w_slot_bytes));
                            kblock(acc, da_hi, db, idesc, kb != 0, ksteps, nullptr);        // x_hi * w_hi
                            kblock(acc, da_lo, db, idesc, 1u, ksteps, &w_empty[ws]);        // x_lo * w_hi
                            if (++ws == p.w_slots) { ws = 0; wph ^= 1; }
                            X3_WAIT(t_wait_w, mbar_wait(&w_full[ws], wph));
                            db = make_smem_desc_sw128(smem_u32(w_ring + (size_t)ws * p.w_slot_bytes));
                            kblock(acc, da_hi, db, idesc, 1u, ksteps, &w_empty[ws]);        // x_hi * w_lo
                            if (++ws == p.w_slots) { ws = 0; wph ^= 1; }
                            commit(&a_empty[as_hi]); commit(&a_empty[as_lo]);
                        } else {
                            const uint32_t ta_hi = hid + (uint32_t)(kb * BLOCK_K), ta_lo = ta_hi + 16;
                            if ((kb & 1) == 0 && kb < 4) {      // K blocks 0-1 / 2-3: the epilogue releases 128 columns at a time
                                X3_WAIT(t_wait_h, mbar_wait(&h_full[kb >> 1], h_par));
                                tcgen05_fence_after();
                            }
                            X3_WAIT(t_wait_w, mbar_wait(&w_full[ws], wph));
                            uint64_t db = make_smem_desc_sw128(smem_u32(w_ring + (size_t)ws * p.w_slot_bytes));
                            kblock_ts(acc, ta_hi, db, idesc, kb != 0, ksteps, nullptr);     // x_hi * w_hi
                            kblock_ts(acc, ta_lo, db, idesc, 1u, ksteps, &w_empty[ws]);     // x_lo * w_hi
                            if (++ws == p.w_slots) { ws = 0; wph ^= 1; }
                            X3_WAIT(t_wait_w, mbar_wait(&w_full[ws], wph));
                            db = make_smem_desc_sw128(smem_u32(w_ring + (size_t)ws * p.w_slot_bytes));
                            kblock_ts(acc, ta_hi, db, idesc, 1u, ksteps, &w_empty[ws]);     // x_hi * w_lo
                            if (++ws == p.w_slots) { ws = 0; wph ^= 1; }
                        }
                    }
                    commit(&tmem_full[buf]);
                }
                ++jp;
            }
#undef X3_WAIT
            if (timing && lane == 0) {
                p.prof[0] = clock64() - t_begin; p.prof[1] = t_wait_acc; p.prof[2] = t_wait_h; p.prof[3] = t_wait_a; p.prof[4] = t_wait_w;
                p.prof[8] = t_wait_read;
            }
        }
    } else if (warp < 2 + p.epi_warps) {               // ================================ epilogue warps
        const int quad = warp & 3;
        Epi e;
        e.lane = lane;
        e.cpar = (warp - 2) >> 2;
        e.cstep = 32 * (p.epi_warps >> 2);
        e.qmaps = p.qmaps;
        e.out0 = p.out0; e.out1 = p.out1; e.ld_out = p.ld_out; e.out_mode = p.out_mode;
        const uint32_t bias_addr0 = smem_u32(bias_s);
        e.stage_addr = smem_u32(stage_all) + (uint32_t)(warp - 2) * (32 * STAGE_ROW);
        long long t_wait_full = 0, t_hidden = 0, t_final = 0;
        int jp = -1;
        for (int j = 0; j < nt; ++j) {
            if (unit_done(j)) continue;
            ++jp;
            const int tile = tile_of(j), grp = group_of(j);
            DSAT_CHECK(tile >= 0 && (tile < p.n_tiles || (PAIR && tile == p.n_tiles)) && grp >= 0 && grp < G);
            e.row_first = (size_t)tile * BLOCK_M + quad * 32;
            e.rows_left = p.rows - (int)e.row_first;
            e.col0 = grp * 256;
            for (int l = 0; l < L; ++l) {
                const int g = jp * L + l, buf = g & 1, use = g >> 1;
                e.N = p.layer[l].N; e.epi = p.layer[l].epi;
                e.bl_addr = bias_addr0 + 4u * (uint32_t)(p.layer[l].bias_off + grp * 256);
                e.lane_addr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(buf * 256);
                const long long t0 = timing ? clock64() : 0;
                mbar_wait(&tmem_full[buf], (uint32_t)(use & 1));
                tcgen05_fence_after();
                const long long t1 = timing ? clock64() : 0;
                const uint32_t empty_addr = at_leader(&tmem_empty[buf]);
                if (l + 1 < L) {
                    // The planes are in tensor memory before the issuer hears of them, 128 columns at a time (h_full[0] once
                    // this warp's chunks below column 128 are stored: the next layer's K blocks 0-1 start while the epilogue
                    // works on the rest).  The accumulator half stays in use (as A) until the next layer's MMAs completed:
                    // the arrival on tmem_empty only keeps its phases counting steps, the issuer orders the half's next
                    // accumulation after those MMAs itself.
                    bool low_done = false;
                    auto release = [&](int h) {
                        fm::tmem_st_wait();
                        tcgen05_fence_before();
                        __syncwarp();
                        if (lane == 0) {
                            if (h == 1) fm::arrive_addr<PAIR>(empty_addr);
                            fm::arrive_addr<PAIR>(at_leader(&h_full[h]));
                        }
                    };
                    // two register buffers: chunk c + cstep is on its way out of TMEM while chunk c is processed
                    int c = 32 * e.cpar;
                    if (c < e.N) {
                        uint32_t ra[32], rb[32];
                        fm::tmem_ld_32cols_async(e.lane_addr + (uint32_t)c, ra);
#pragma unroll 1
                        while (true) {
                            fm::tmem_ld_wait(ra);
                            const int c1 = c + e.cstep;
                            if (c1 < e.N) fm::tmem_ld_32cols_async(e.lane_addr + (uint32_t)c1, rb);
                            epi_hidden(e, ra, c);
                            if (!low_done && c1 >= 128) { release(0); low_done = true; }
                            if (c1 >= e.N) break;
                            fm::tmem_ld_wait(rb);
                            c = c1 + e.cstep;
                            if (c < e.N) fm::tmem_ld_32cols_async(e.lane_addr + (uint32_t)c, ra);
                            epi_hidden(e, rb, c1);
                            if (!low_done && c >= 128) { release(0); low_done = true; }
                            if (c >= e.N) break;
                        }
                    }
                    if (!low_done) release(0);
                    release(1);
                    if (timing) t_hidden += clock64() - t1;
                } else {
                    bool released = false;
#pragma unroll 1
                    for (int c = 32 * e.cpar; c < e.N; c += e.cstep) {
                        uint32_t ra[32];
                        fm::tmem_ld_32cols_async(e.lane_addr + (uint32_t)c, ra);
                        fm::tmem_ld_wait(ra);
                        if (c + e.cstep >= e.N) {       // last TMEM read of this warp: hand the accumulator back early
                            tcgen05_fence_before();
                            fm::warp_arrive<PAIR>(empty_addr, lane);
                            released = true;
                        }
                        epi_final(e, ra, c);
                    }
                    if (!released) { tcgen05_fence_before(); fm::warp_arrive<PAIR>(empty_addr, lane); }
                    if (timing) t_final += clock64() - t1;
                }
                if (timing) t_wait_full += t1 - t0;
            }
        }
        if (timing && warp == 2 && lane == 0) { p.prof[5] = t_wait_full; p.prof[6] = t_hidden; p.prof[7] = t_final; }
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

// ------------------------------------------------------------------------------------ host side
struct X3Mlp {
    CUtensorMap map_a_hi, map_a_lo;
    CUtensorMap map_w[MAX_LAYERS];
    X3Params p;
    int smem_bytes = 0;
    bool pair_mode = false;     // request the CTA-pair instantiation
    bool ready = false;
};

// shared-memory plan; returns false when the MLP does not fit
inline bool plan_x3(X3Mlp& f) {
    X3Params& p = f.p;
    const int pad = fm::dyn_smem_pad();
    p.smem_pad = pad;
    int bias_total = 0, max_n = 0;
    bool pair = f.pair_mode && p.rows > BLOCK_M;
    for (int l = 0; l < p.n_layers; ++l) {
        X3Layer& ly = p.layer[l];
        if (ly.N > 256 || ly.N % 16 || ly.K % 16) return false;
        if (l > 0 && ly.K > p.layer[l - 1].N) return false;     // a hidden layer's A: the columns layer l - 1 wrote
        ly.bias_off = bias_total;
        bias_total += (ly.n_total + 31) / 32 * 32;
        max_n = max(max_n, ly.N);
    }
    if (p.n_groups > 1 && p.n_layers != 1) return false;
    p.pair = pair ? 1 : 0;
    p.bias_total = bias_total;
    p.n_tiles = ceil_div(p.rows, BLOCK_M);
    p.w_slot_bytes = ((pair ? max_n / 2 : max_n) * BLOCK_K * 2 + 1023) / 1024 * 1024;
    for (int ew : {8, 4}) {
        const int fixed = pad + ew * 32 * STAGE_ROW + BAR_BYTES + bias_total * 4;
        int avail = SMEM_LIMIT - fixed;
        int a = 2, w = 2;
        if (avail < a * BLK_BYTES + w * p.w_slot_bytes) continue;
        avail -= a * BLK_BYTES + w * p.w_slot_bytes;
        // grow the rings in turn, the input ring first (the input comes from HBM, the weights from L2)
        while (true) {
            bool grew = false;
            if (a <= w && a < MAX_RING && avail >= BLK_BYTES) { ++a; avail -= BLK_BYTES; grew = true; }
            else if (w < MAX_RING && avail >= p.w_slot_bytes) { ++w; avail -= p.w_slot_bytes; grew = true; }
            else if (a < MAX_RING && avail >= BLK_BYTES) { ++a; avail -= BLK_BYTES; grew = true; }
            if (!grew) break;
        }
        p.a_slots = a; p.w_slots = w; p.epi_warps = ew;
        f.smem_bytes = fixed + a * BLK_BYTES + w * p.w_slot_bytes;
        f.ready = true;
        return true;
    }
    return false;
}

inline cudaError_t configure_x3_device(int) {
    static PerDeviceOnce configured;                // MaxDynamicSharedMemorySize is a per-device function attribute
    if (configured.done()) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(x3_mlp_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(x3_mlp_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT);
    if (e == cudaSuccess) configured.mark();
    return e;
}

inline cudaError_t launch_x3(const X3Mlp& f, int device, int sm_count, cudaStream_t stream) {
    if (f.p.rows <= 0) return cudaSuccess;
    cudaError_t e = configure_x3_device(device);
    if (e != cudaSuccess) return e;
    const unsigned threads = 64 + 32 * f.p.epi_warps;
    if (f.p.pair) {
        const int n_units = (f.p.n_tiles + 1) / 2 * f.p.n_groups;
        const int pairs = n_units < sm_count / 2 ? n_units : sm_count / 2;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(2 * pairs); cfg.blockDim = dim3(threads); cfg.dynamicSmemBytes = (size_t)f.smem_bytes; cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        return cudaLaunchKernelEx(&cfg, x3_mlp_kernel<true>, f.map_a_hi, f.map_a_lo, f.map_w[0], f.map_w[1], f.map_w[2], f.p);
    }
    const int n_units = f.p.n_tiles * f.p.n_groups;
    const unsigned grid = (unsigned)(n_units < sm_count ? n_units : sm_count);
    x3_mlp_kernel<false><<<grid, threads, f.smem_bytes, stream>>>(f.map_a_hi, f.map_a_lo, f.map_w[0], f.map_w[1], f.map_w[2], f.p);
    return cudaGetLastError();
}

}  // namespace x3
}  // namespace dsat
