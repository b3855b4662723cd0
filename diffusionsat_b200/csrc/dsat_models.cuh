// Every model of a formula over n <= 63 variables, by brute force over all 2^n assignments (dsat_enumerate_models): the
// exact model set the uniformity statistics compare the sampler's histogram against (the reference counts models with
// unigen/approxmc, utils/AllSolutions.py:44-68).
//
// An assignment is the integer of the reference encoding (x1 = bit 0, utils/VariableAssignment.py:63-69).  Its low six
// bits, the values of variables 1..6, are the 64 lanes of one 64-bit word; the rest, H = assignment >> 6, is one thread's
// work item.  The host compiles every clause once per call into
//   pos_hi / neg_hi  its positive / negative literals on variables 7..n as bits of H (variable v = bit v-7),
//   lane_sat         the lanes in which one of its literals on variables 1..6 is true,
// so for a given H the clause holds in all 64 lanes when (H & pos_hi) | (~H & neg_hi) != 0 and in lane_sat otherwise.
// `ok`, the lanes that satisfy every clause so far, is ANDed down clause by clause until it is 0.
//
// Ascending output without a sort: a count pass writes each block's number of models, a single-CTA scan turns them into
// offsets, and an emit pass recomputes `ok` and writes the set lanes of every H in order.  Block b covers the contiguous H
// range [h0 + b*H_PER_BLOCK, +H_PER_BLOCK) and thread t of step k takes H = base + k*THREADS + t, so blocks, steps and
// threads are all ascending in H.  The host enumerates at most 2^CHUNK_LOG2 assignments per launch.
#pragma once
#include "dsat_common.cuh"

namespace dsat {
namespace models {

constexpr int THREADS = 256;
constexpr int STEPS = 8;                                         // H values per thread
constexpr long long H_PER_BLOCK = (long long)THREADS * STEPS;
constexpr int TILE = 1024;                                       // clauses staged in shared memory at a time
constexpr int CHUNK_LOG2 = 36;                                   // assignments per launch: a few ms to tens of ms each
constexpr int SCAN_THREADS = 1024, SCAN_ITEMS = 4;

struct Clause { unsigned long long pos_hi, neg_hi, lane_sat; };

// lanes of the STEPS values H = h + k*THREADS (those below h_end) that satisfy every clause.  Called by every thread of
// the block (the clause tiles are staged with __syncthreads).
__device__ __forceinline__ void eval_models(const Clause* __restrict__ clauses, int m, unsigned long long lane_mask,
                                           unsigned long long h, unsigned long long h_end, unsigned long long (&ok)[STEPS]) {
    __shared__ unsigned long long s_pos[TILE], s_neg[TILE], s_lane[TILE];
#pragma unroll
    for (int k = 0; k < STEPS; ++k) ok[k] = h + (unsigned long long)k * THREADS < h_end ? lane_mask : 0ull;
    for (int base = 0; base < m; base += TILE) {
        const int cnt = min(TILE, m - base);
        __syncthreads();                                         // the previous tile has been read by every thread
        for (int j = threadIdx.x; j < cnt; j += THREADS) {
            const Clause c = clauses[base + j];
            s_pos[j] = c.pos_hi; s_neg[j] = c.neg_hi; s_lane[j] = c.lane_sat;
        }
        __syncthreads();
        bool alive = false;
#pragma unroll
        for (int k = 0; k < STEPS; ++k) {
            const unsigned long long H = h + (unsigned long long)k * THREADS;
            unsigned long long o = ok[k];
            for (int j = 0; j < cnt && o; ++j)
                if (!((H & s_pos[j]) | (~H & s_neg[j]))) o &= s_lane[j];
            ok[k] = o;
            alive |= o != 0;
        }
        if (!__syncthreads_or(alive)) break;                     // no lane of the block is left
    }
}

// exclusive prefix sum over the block's threads (in thread order) and the block's total
__device__ __forceinline__ unsigned block_exclusive_scan(unsigned v, unsigned* total) {
    __shared__ unsigned warp_tot[THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const unsigned t = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += t; }
    if (lane == 31) warp_tot[warp] = x;
    __syncthreads();
    unsigned before = 0, sum = 0;
#pragma unroll
    for (int w = 0; w < THREADS / 32; ++w) {
        before += w < warp ? warp_tot[w] : 0u;
        sum += warp_tot[w];
    }
    __syncthreads();                                             // warp_tot may be written again by the next call
    *total = sum;
    return before + x - v;
}

// block_models[b] = number of models in block b's H range (at most 64 * H_PER_BLOCK = 2^17)
__global__ void __launch_bounds__(THREADS) count_kernel(const Clause* __restrict__ clauses, int m, unsigned long long lane_mask,
                                                        unsigned long long h0, unsigned long long h_end,
                                                        unsigned* __restrict__ block_models) {
    unsigned long long ok[STEPS];
    eval_models(clauses, m, lane_mask, h0 + blockIdx.x * (unsigned long long)H_PER_BLOCK + threadIdx.x, h_end, ok);
    unsigned n = 0;
#pragma unroll
    for (int k = 0; k < STEPS; ++k) n += __popcll(ok[k]);
    unsigned total;
    block_exclusive_scan(n, &total);
    if (threadIdx.x == 0) block_models[blockIdx.x] = total;
}

// offsets[b] = models of blocks [0, b); *total = models of all n blocks (one CTA, SCAN_ITEMS consecutive blocks per thread)
__global__ void __launch_bounds__(SCAN_THREADS) scan_kernel(const unsigned* __restrict__ block_models, int n,
                                                            unsigned long long* __restrict__ offsets,
                                                            unsigned long long* __restrict__ total) {
    __shared__ unsigned long long warp_tot[SCAN_THREADS / 32];
    __shared__ unsigned long long carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int base = 0; base < n; base += SCAN_THREADS * SCAN_ITEMS) {
        const int i0 = base + threadIdx.x * SCAN_ITEMS;
        unsigned v[SCAN_ITEMS];
        unsigned long long mine = 0;
#pragma unroll
        for (int q = 0; q < SCAN_ITEMS; ++q) { v[q] = i0 + q < n ? block_models[i0 + q] : 0u; mine += v[q]; }
        unsigned long long x = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned long long t = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += t; }
        if (lane == 31) warp_tot[warp] = x;
        __syncthreads();
        if (warp == 0) {
            unsigned long long w = warp_tot[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const unsigned long long t = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += t; }
            warp_tot[lane] = w;
        }
        __syncthreads();
        unsigned long long at = carry + (warp ? warp_tot[warp - 1] : 0ull) + x - mine;
#pragma unroll
        for (int q = 0; q < SCAN_ITEMS; ++q) {
            if (i0 + q < n) offsets[i0 + q] = at;
            at += v[q];
        }
        __syncthreads();
        if (threadIdx.x == 0) carry += warp_tot[31];
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry;
}

// the models of block b's H range, ascending, at out[offsets[b]...]; only indices below `limit` are written
__global__ void __launch_bounds__(THREADS) emit_kernel(const Clause* __restrict__ clauses, int m, unsigned long long lane_mask,
                                                       unsigned long long h0, unsigned long long h_end,
                                                       const unsigned long long* __restrict__ offsets, unsigned long long limit,
                                                       unsigned long long* __restrict__ out) {
    unsigned long long ok[STEPS];
    const unsigned long long h = h0 + blockIdx.x * (unsigned long long)H_PER_BLOCK + threadIdx.x;
    eval_models(clauses, m, lane_mask, h, h_end, ok);
    unsigned long long pos = offsets[blockIdx.x];
#pragma unroll
    for (int k = 0; k < STEPS; ++k) {
        unsigned total;
        unsigned long long at = pos + block_exclusive_scan(__popcll(ok[k]), &total);
        const unsigned long long high = (h + (unsigned long long)k * THREADS) << 6;
        for (unsigned long long o = ok[k]; o && at < limit; o &= o - 1) out[at++] = high | (unsigned long long)(__ffsll((long long)o) - 1);
        pos += total;
    }
}

}  // namespace models
}  // namespace dsat
