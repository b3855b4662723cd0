// Device-side histogram of the sampled assignments: sort / unique / count of the packed satisfying assignments of one
// launch (reference satuniformity/DiffusionSampler.py:283-307 builds {solution_as_int: count} one sample at a time in
// Python; utils/VariableAssignment.py:63-69 is the int encoding the packed words already carry).
//
// The chains of a launch are few (<= 2^17) and a key is 1..4 64-bit words, so the sort is a plain bitonic network over
// chain INDICES in global memory (the keys themselves never move); unsatisfied chains and chains beyond the caller's limit
// sort last.  Heads of equal-key runs are flagged, a single-CTA scan numbers them, and one pass writes each run's key and
// its length.  Output order = ascending numeric value of the assignment (most significant word compared first).
//
// Segmented form (several formulas in one launch, dsat_hist_reduce_segments): `seg` maps each chain index to its segment,
// -1 for a chain that does not count.  It is monotone in the index, so ordering by (segment, key, index) keeps the
// segments apart and in order; a run starts where the segment or the key changes, and emit records each run's segment.
#pragma once
#include "dsat_common.cuh"

namespace dsat {
namespace hist {

__device__ __forceinline__ int key_cmp(const unsigned long long* __restrict__ packed, int words, int a, int b) {
    for (int w = words - 1; w >= 0; --w) {
        const unsigned long long ka = packed[(size_t)a * words + w], kb = packed[(size_t)b * words + w];
        if (ka != kb) return ka < kb ? -1 : 1;
    }
    return 0;
}

// total order on slots: live chain indices by (segment, key, index), dead slots (-1) last
__device__ __forceinline__ bool slot_less(const unsigned long long* __restrict__ packed, int words, int a, int b,
                                          const int* __restrict__ seg) {
    if (a < 0) return false;
    if (b < 0) return true;
    if (seg) {
        const int sa = __ldg(seg + a), sb = __ldg(seg + b);
        if (sa != sb) return sa < sb;
    }
    const int c = key_cmp(packed, words, a, b);
    return c < 0 || (c == 0 && a < b);
}

__global__ void init_kernel(int n_pad, int limit, const unsigned char* __restrict__ is_sat, int* __restrict__ idx,
                            const int* __restrict__ seg) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_pad) idx[i] = (i < limit && is_sat[i] && (!seg || __ldg(seg + i) >= 0)) ? i : -1;
}

// one compare-exchange layer of the bitonic network: partner = i ^ j, direction from bit k of i
__global__ void bitonic_kernel(int* __restrict__ idx, int n_pad, int j, int k, const unsigned long long* __restrict__ packed, int words,
                               const int* __restrict__ seg) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int p = i ^ j;
    if (i >= n_pad || p <= i) return;
    const int a = idx[i], b = idx[p];
    const bool up = (i & k) == 0;
    if (slot_less(packed, words, b, a, seg) == up) { idx[i] = b; idx[p] = a; }
}

// the whole network for n_pad <= 2048 in one CTA's shared memory
__global__ void __launch_bounds__(1024) bitonic_small_kernel(int* __restrict__ idx, int n_pad, const unsigned long long* __restrict__ packed, int words,
                                                             const int* __restrict__ seg) {
    __shared__ int s[2048];
    for (int i = threadIdx.x; i < n_pad; i += blockDim.x) s[i] = idx[i];
    __syncthreads();
    for (int k = 2; k <= n_pad; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n_pad; i += blockDim.x) {
                const int p = i ^ j;
                if (p > i) {
                    const int a = s[i], b = s[p];
                    const bool up = (i & k) == 0;
                    if (slot_less(packed, words, b, a, seg) == up) { s[i] = b; s[p] = a; }
                }
            }
            __syncthreads();
        }
    for (int i = threadIdx.x; i < n_pad; i += blockDim.x) idx[i] = s[i];
}

// flag[i] = 1 where a run of equal keys starts; then an inclusive scan in place (single CTA), totals[0] = number of runs,
// totals[1] = number of live slots
__global__ void __launch_bounds__(1024) heads_scan_kernel(const int* __restrict__ idx, int n_pad, const unsigned long long* __restrict__ packed,
                                                           int words, int* __restrict__ run_id, int* __restrict__ totals,
                                                           const int* __restrict__ seg) {
    __shared__ int warp_tot[32];
    __shared__ int carry, live_tot;
    if (threadIdx.x == 0) { carry = 0; live_tot = 0; }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int live_mine = 0;
    for (int base = 0; base < n_pad; base += blockDim.x) {
        const int i = base + threadIdx.x;
        int flag = 0;
        if (i < n_pad) {
            const int a = idx[i];
            if (a >= 0) {
                ++live_mine;
                const int prev = i == 0 ? -1 : idx[i - 1];
                flag = (prev < 0) ? 1 : (key_cmp(packed, words, prev, a) != 0 || (seg && __ldg(seg + prev) != __ldg(seg + a)));
            }
        }
        int v = flag;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += t; }
        if (lane == 31) warp_tot[warp] = v;
        __syncthreads();
        if (warp == 0) {
            int w = warp_tot[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += t; }
            warp_tot[lane] = w;
        }
        __syncthreads();
        const int before = carry + (warp ? warp_tot[warp - 1] : 0);
        if (i < n_pad) run_id[i] = before + v;        // 1-based id of the run slot i belongs to (valid where idx[i] >= 0)
        __syncthreads();
        if (threadIdx.x == 0) carry += warp_tot[31];
        __syncthreads();
    }
    atomicAdd(&live_tot, live_mine);
    __syncthreads();
    if (threadIdx.x == 0) { totals[0] = carry; totals[1] = live_tot; }
}

__global__ void emit_kernel(const int* __restrict__ idx, const int* __restrict__ run_id, int n_pad, const unsigned long long* __restrict__ packed,
                            int words, unsigned long long* __restrict__ keys_out, unsigned long long* __restrict__ counts_out,
                            const int* __restrict__ seg, int* __restrict__ run_seg) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pad) return;
    const int a = idx[i];
    if (a < 0) return;
    const int u = run_id[i] - 1;
    if (i == 0 || run_id[i - 1] != run_id[i]) {
        for (int w = 0; w < words; ++w) keys_out[(size_t)u * words + w] = packed[(size_t)a * words + w];
        if (seg) run_seg[u] = __ldg(seg + a);
    }
    atomicAdd(&counts_out[u], 1ull);
}

inline int next_pow2(int x) { int p = 1; while (p < x) p <<= 1; return p; }

// Enqueue the whole reduction on `stream`.  Scratch: idx, run_id [n_pad] int; keys_out [n, words]; counts_out [n]; totals [2].
// seg (optional, [n]): segment of each chain index (monotone, -1 = not counted); run_seg [n] then receives each run's segment.
inline cudaError_t enqueue(cudaStream_t stream, int n, int limit, int words, const unsigned long long* packed, const unsigned char* is_sat,
                           int* idx, int* run_id, unsigned long long* keys_out, unsigned long long* counts_out, int* totals, long long* launches,
                           const int* seg = nullptr, int* run_seg = nullptr) {
    const int n_pad = next_pow2(n < 2 ? 2 : n);
    const int threads = 256, blocks = (n_pad + threads - 1) / threads;
    init_kernel<<<blocks, threads, 0, stream>>>(n_pad, limit < n ? limit : n, is_sat, idx, seg);
    ++*launches;
    if (n_pad <= 2048) {
        bitonic_small_kernel<<<1, 1024, 0, stream>>>(idx, n_pad, packed, words, seg);
        ++*launches;
    } else {
        for (int k = 2; k <= n_pad; k <<= 1)
            for (int j = k >> 1; j > 0; j >>= 1) {
                bitonic_kernel<<<blocks, threads, 0, stream>>>(idx, n_pad, j, k, packed, words, seg);
                ++*launches;
            }
    }
    cudaError_t e = cudaMemsetAsync(counts_out, 0, (size_t)n * sizeof(unsigned long long), stream);
    if (e != cudaSuccess) return e;
    heads_scan_kernel<<<1, 1024, 0, stream>>>(idx, n_pad, packed, words, run_id, totals, seg);
    emit_kernel<<<blocks, threads, 0, stream>>>(idx, run_id, n_pad, packed, words, keys_out, counts_out, seg, run_seg);
    *launches += 2;
    return cudaGetLastError();
}

}  // namespace hist
}  // namespace dsat
