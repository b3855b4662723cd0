// PairNorm + residual/carry, the logit-map head with the per-graph SAT check, the batch early-exit
// bookkeeping, and the per-denoising-step kernels (randomized rounding, posterior, first-SAT latch,
// bit packing).  All of them treat a graph (= one chain of one formula) as the unit of work: graph
// `gid` is formula `gid % n_graphs` of chain `gid / n_graphs`, its nodes are contiguous rows.
#pragma once
#include "dsat_common.cuh"
#include "dsat_message.cuh"

namespace dsat {

template <int V>
__device__ __forceinline__ int lane_col(int lane, int i) {
    if constexpr (V == 2) return lane * 2 + i;
    else return (i >> 2) * 128 + lane * 4 + (i & 3);
}

// ------------------------------------------------------------------------------------ PairNorm
// reference layers/normalization.py:43-71 with graph_norm = membership/count (model/query_sat.py:206-211):
//   x -= sum_{nodes of the graph} x * (1/count)      per feature
//   x *= rsqrt(mean_f(x^2) + 1e-6)                   per node
// fused with the caller's  new = x*0.25 + 0.1*old  (model/query_sat.py:265-266, 279-280) and with the
// end-of-round  s = s*0.2 + s*0.8  (:347-348).  PRE (optional) receives the state before that carry:
// it is what variables_output reads (:283).  TS / TX = storage type of the input and of the state
// (float on the fp32 path, bf16 on the tensor-core path; the arithmetic is fp32 either way).
constexpr int PN_WARPS = 8;
#ifndef PN_BF16_CTAS
#define PN_BF16_CTAS 4     // resident CTAs per SM of pairnorm_bf16_kernel (64 registers); 3: -6 %, 5 spills: -40 %
#endif
constexpr int PN_UNROLL = 4;      // rows in flight per warp (memory-level parallelism)

template <int V, typename TS, typename TX>
__global__ void __launch_bounds__(PN_WARPS * 32)
pairnorm_kernel(const int* __restrict__ seg, int n_graphs_unit, int rows_per_chain, int total_graphs,
                const TS* __restrict__ SRC, int ld_src, int src_off,
                TX* __restrict__ STATE, int ld_state,
                TX* __restrict__ PRE, int ld_pre,
                // split-plane state (fp32-accurate tensor-core path): hi planes + distance to the lo planes, instead of STATE / PRE
                __nv_bfloat16* STATE_HI = nullptr, size_t state_plane = 0,
                __nv_bfloat16* __restrict__ PRE_HI = nullptr, size_t pre_plane = 0,
                SkipInfo skip = SkipInfo{nullptr, 1}) {
    constexpr int F = 32 * V;
    __shared__ float red[PN_WARPS][F];
    __shared__ float mean_s[F];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int gid = blockIdx.x; gid < total_graphs; gid += gridDim.x) {
        const int chain = gid / n_graphs_unit, lg = gid % n_graphs_unit;
        if (chain_done(skip, chain)) continue;
        const size_t base = (size_t)chain * rows_per_chain;
        const size_t r0 = base + __ldg(seg + lg), r1 = base + __ldg(seg + lg + 1);
        const float wgt = 1.0f / (float)(r1 - r0);
        LaneVec<V> sum;
#pragma unroll
        for (int i = 0; i < V; ++i) sum.v[i] = 0.f;
        {
            size_t r = r0 + warp;
            for (; r + (PN_UNROLL - 1) * PN_WARPS < r1; r += PN_UNROLL * PN_WARPS) {
                LaneVec<V> x[PN_UNROLL];
#pragma unroll
                for (int u = 0; u < PN_UNROLL; ++u)
                    x[u] = lane_load_t<V, TS>(SRC + (r + u * PN_WARPS) * ld_src + src_off, lane);
#pragma unroll
                for (int u = 0; u < PN_UNROLL; ++u)
#pragma unroll
                    for (int i = 0; i < V; ++i) sum.v[i] += x[u].v[i] * wgt;
            }
            for (; r < r1; r += PN_WARPS) {
                LaneVec<V> x = lane_load_t<V, TS>(SRC + r * ld_src + src_off, lane);
#pragma unroll
                for (int i = 0; i < V; ++i) sum.v[i] += x.v[i] * wgt;
            }
        }
#pragma unroll
        for (int i = 0; i < V; ++i) red[warp][lane_col<V>(lane, i)] = sum.v[i];
        __syncthreads();
        for (int col = tid; col < F; col += PN_WARPS * 32) {
            float s = 0.f;
#pragma unroll
            for (int w = 0; w < PN_WARPS; ++w) s += red[w][col];
            mean_s[col] = s;
        }
        __syncthreads();
        LaneVec<V> mean;
#pragma unroll
        for (int i = 0; i < V; ++i) mean.v[i] = mean_s[lane_col<V>(lane, i)];
        auto finish_row = [&](size_t r, LaneVec<V> x, const LaneVec<V>& old) {
            float ss = 0.f;
#pragma unroll
            for (int i = 0; i < V; ++i) { x.v[i] -= mean.v[i]; ss += x.v[i] * x.v[i]; }
            ss = warp_sum(ss);
            const float inv = rsqrtf(ss / (float)F + 1.0e-6f);
            LaneVec<V> nw, carried;
#pragma unroll
            for (int i = 0; i < V; ++i) {
                nw.v[i] = __fadd_rn(__fmul_rn(x.v[i] * inv, 0.25f), __fmul_rn(0.1f, old.v[i]));
                carried.v[i] = __fadd_rn(__fmul_rn(nw.v[i], 0.2f), __fmul_rn(nw.v[i], 0.8f));
            }
            if (STATE_HI) {
                if (PRE_HI) lane_store_split<V>(PRE_HI + r * ld_pre, pre_plane, lane, nw);
                lane_store_split<V>(STATE_HI + r * ld_state, state_plane, lane, carried);
                return;
            }
            if (PRE) lane_store_t<V, TX>(PRE + r * ld_pre, lane, nw);
            lane_store_t<V, TX>(STATE + r * ld_state, lane, carried);
        };
        auto load_old = [&](size_t r) {
            return STATE_HI ? lane_load_split_rw<V>(STATE_HI + r * ld_state, state_plane, lane)
                            : lane_load_rw_t<V, TX>(STATE + r * ld_state, lane);
        };
        {
            size_t r = r0 + warp;
            for (; r + (PN_UNROLL - 1) * PN_WARPS < r1; r += PN_UNROLL * PN_WARPS) {
                LaneVec<V> x[PN_UNROLL], old[PN_UNROLL];
#pragma unroll
                for (int u = 0; u < PN_UNROLL; ++u) {
                    x[u] = lane_load_t<V, TS>(SRC + (r + u * PN_WARPS) * ld_src + src_off, lane);
                    old[u] = load_old(r + u * PN_WARPS);
                }
#pragma unroll
                for (int u = 0; u < PN_UNROLL; ++u) finish_row(r + u * PN_WARPS, x[u], old[u]);
            }
            for (; r < r1; r += PN_WARPS) {
                LaneVec<V> x = lane_load_t<V, TS>(SRC + r * ld_src + src_off, lane);
                LaneVec<V> old = load_old(r);
                finish_row(r, x, old);
            }
        }
        __syncthreads();
    }
}

// The same operation for graphs whose rows fit in shared memory (fp32-accurate tensor-core path: fp32 input, hi/lo-plane
// state).  pairnorm_kernel reads its input twice and relies on L2 for the second pass, with only a few 512-byte rows in
// flight per warp; here a CTA pulls the whole graph in with asynchronous copies (every byte of the graph in flight at
// once, each read from HBM exactly once), takes the column means out of shared memory, and the second pass needs global
// memory only for the old state and the stores.  blockDim.x = any multiple of 32 up to 1024.
template <int V>
__global__ void __launch_bounds__(1024)
pairnorm_smem_kernel(const int* __restrict__ seg, int n_graphs_unit, int rows_per_chain, int total_graphs,
                     const float* __restrict__ SRC, int ld_src, int src_off,
                     __nv_bfloat16* STATE_HI, size_t state_plane, int ld_state,
                     __nv_bfloat16* __restrict__ PRE_HI, size_t pre_plane, int ld_pre, SkipInfo skip = SkipInfo{nullptr, 1}) {
    constexpr int F = 32 * V;
    constexpr int PPR = F / 4;                         // 16-byte pieces per row
    extern __shared__ __align__(16) uint8_t pn_smem[];
    float* mean_s = reinterpret_cast<float*>(pn_smem);             // [F]
    float* part = mean_s + F;                                       // [groups][F]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const int groups = blockDim.x / F > 0 ? blockDim.x / F : 1;     // thread groups that sum interleaved rows of one column
    float* rows = part + groups * F;                                // [graph rows][F]
    for (int gid = blockIdx.x; gid < total_graphs; gid += gridDim.x) {
        const int chain = gid / n_graphs_unit, lg = gid % n_graphs_unit;
        if (chain_done(skip, chain)) continue;
        const size_t base = (size_t)chain * rows_per_chain;
        const size_t r0 = base + __ldg(seg + lg);
        const int nrows = __ldg(seg + lg + 1) - __ldg(seg + lg);
        const float wgt = 1.0f / (float)nrows;
        DSAT_CHECK(nrows > 0 && r0 + nrows <= (size_t)(chain + 1) * rows_per_chain);
        for (int i = tid; i < nrows * PPR; i += blockDim.x) {
            const int r = i / PPR, k = i % PPR;
            cp_async16(rows + (size_t)r * F + 4 * k, SRC + (r0 + r) * ld_src + src_off + 4 * k);
        }
        cp_async_wait_all();
        __syncthreads();
        if (tid < groups * F) {                                     // column sums: thread = (row group, column)
            const int col = tid % F, grp = tid / F;
            float s = 0.f;
            for (int r = grp; r < nrows; r += groups) s += rows[(size_t)r * F + col] * wgt;
            part[grp * F + col] = s;
        }
        __syncthreads();
        if (tid < F) {
            float s = 0.f;
            for (int k = 0; k < groups; ++k) s += part[k * F + tid];
            mean_s[tid] = s;
        }
        __syncthreads();
        LaneVec<V> mean;
#pragma unroll
        for (int i = 0; i < V; ++i) mean.v[i] = mean_s[lane_col<V>(lane, i)];
        auto finish_row = [&](int r, const LaneVec<V>& old) {
            LaneVec<V> x = lane_load_rw<V>(rows + (size_t)r * F, lane);
            float ss = 0.f;
#pragma unroll
            for (int i = 0; i < V; ++i) { x.v[i] -= mean.v[i]; ss += x.v[i] * x.v[i]; }
            ss = warp_sum(ss);
            const float inv = rsqrtf(ss / (float)F + 1.0e-6f);
            LaneVec<V> nw, carried;
#pragma unroll
            for (int i = 0; i < V; ++i) {
                nw.v[i] = __fadd_rn(__fmul_rn(x.v[i] * inv, 0.25f), __fmul_rn(0.1f, old.v[i]));
                carried.v[i] = __fadd_rn(__fmul_rn(nw.v[i], 0.2f), __fmul_rn(nw.v[i], 0.8f));
            }
            if (PRE_HI) lane_store_split<V>(PRE_HI + (r0 + r) * ld_pre, pre_plane, lane, nw);
            lane_store_split<V>(STATE_HI + (r0 + r) * ld_state, state_plane, lane, carried);
        };
        int r = warp;
        for (; r + (PN_UNROLL - 1) * nwarps < nrows; r += PN_UNROLL * nwarps) {
            LaneVec<V> old[PN_UNROLL];
#pragma unroll
            for (int u = 0; u < PN_UNROLL; ++u) old[u] = lane_load_split_rw<V>(STATE_HI + (r0 + r + u * nwarps) * ld_state, state_plane, lane);
#pragma unroll
            for (int u = 0; u < PN_UNROLL; ++u) finish_row(r + u * nwarps, old[u]);
        }
        for (; r < nrows; r += nwarps) finish_row(r, lane_load_split_rw<V>(STATE_HI + (r0 + r) * ld_state, state_plane, lane));
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------- head
// KL(Bernoulli(pa) || Bernoulli(pb)), probabilities as parameters (TFP's registered Bernoulli KL,
// external): pa*(log pa - log pb) + (1-pa)*(log1p(-pa) - log1p(-pb)), 0*inf := 0.
__device__ __forceinline__ float bernoulli_kl(float pa, float pb) {
    const float qa = 1.0f - pa;
    const float t1 = pa == 0.f ? 0.f : pa * (logf(pa) - logf(pb));
    const float t2 = qa == 0.f ? 0.f : qa * (log1pf(-pa) - log1pf(-pb));
    return t1 + t2;
}

// bf16 storage on both sides (tensor-core path): a lane moves 16 bytes = 8 features, so a row takes F/8 lanes and a
// warp load covers 32/(F/8) rows: half as many memory instructions per byte as the generic kernel's 8-byte lanes, and
// PN_UNROLL row groups in flight give twice the bytes in flight per warp.  Same arithmetic (fp32), different summation
// order than the generic kernel.
template <int F>
__global__ void __launch_bounds__(PN_WARPS * 32, PN_BF16_CTAS)
pairnorm_bf16_kernel(const int* __restrict__ seg, int n_graphs_unit, int rows_per_chain, int total_graphs,
                     const __nv_bfloat16* __restrict__ SRC, int ld_src, int src_off,
                     __nv_bfloat16* __restrict__ STATE, int ld_state,
                     __nv_bfloat16* __restrict__ PRE, int ld_pre, SkipInfo skip = SkipInfo{nullptr, 1}) {
    constexpr int LPR = F / 8, RPW = 32 / LPR, GROUP = PN_WARPS * RPW;     // rows covered by one load of the whole CTA
    __shared__ float red[PN_WARPS][F];
    __shared__ float mean_s[F];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int sub = lane / LPR, li = lane % LPR;
    for (int gid = blockIdx.x; gid < total_graphs; gid += gridDim.x) {
        const int chain = gid / n_graphs_unit, lg = gid % n_graphs_unit;
        if (chain_done(skip, chain)) continue;
        const size_t base = (size_t)chain * rows_per_chain;
        const size_t r0 = base + __ldg(seg + lg), r1 = base + __ldg(seg + lg + 1);
        const float wgt = 1.0f / (float)(r1 - r0);
        float sum[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) sum[i] = 0.f;
        // (loop bounds are warp-uniform: the row of a lane is rb + sub, guarded by rr < r1)
        for (size_t rb = r0 + warp * RPW; rb < r1; rb += (size_t)PN_UNROLL * GROUP) {
            const size_t r = rb + sub;
            uint4 x[PN_UNROLL];
#pragma unroll
            for (int u = 0; u < PN_UNROLL; ++u) {
                const size_t rr = r + (size_t)u * GROUP;
                x[u] = make_uint4(0u, 0u, 0u, 0u);
                if (rr < r1) x[u] = __ldg(reinterpret_cast<const uint4*>(SRC + rr * ld_src + src_off) + li);
            }
#pragma unroll
            for (int u = 0; u < PN_UNROLL; ++u) {
                float v[8];
                unpack8(x[u], v);
#pragma unroll
                for (int i = 0; i < 8; ++i) sum[i] += v[i] * wgt;
            }
        }
#pragma unroll
        for (int off = LPR; off < 32; off <<= 1)
#pragma unroll
            for (int i = 0; i < 8; ++i) sum[i] += __shfl_xor_sync(0xffffffffu, sum[i], off);
        if (sub == 0) {
#pragma unroll
            for (int i = 0; i < 8; ++i) red[warp][li * 8 + i] = sum[i];
        }
        __syncthreads();
        for (int col = tid; col < F; col += PN_WARPS * 32) {
            float s = 0.f;
#pragma unroll
            for (int w = 0; w < PN_WARPS; ++w) s += red[w][col];
            mean_s[col] = s;
        }
        __syncthreads();
        float mean[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) mean[i] = mean_s[li * 8 + i];
        for (size_t rb = r0 + warp * RPW; rb < r1; rb += (size_t)PN_UNROLL * GROUP) {
            const size_t r = rb + sub;
            uint4 x[PN_UNROLL], old[PN_UNROLL];
#pragma unroll
            for (int u = 0; u < PN_UNROLL; ++u) {
                const size_t rr = r + (size_t)u * GROUP;
                x[u] = make_uint4(0u, 0u, 0u, 0u); old[u] = x[u];
                if (rr < r1) {
                    x[u] = __ldg(reinterpret_cast<const uint4*>(SRC + rr * ld_src + src_off) + li);
                    old[u] = reinterpret_cast<const uint4*>(STATE + rr * ld_state)[li];
                }
            }
#pragma unroll
            for (int u = 0; u < PN_UNROLL; ++u) {
                const size_t rr = r + (size_t)u * GROUP;
                float v[8], o[8], nw[8], carried[8];
                unpack8(x[u], v);
                unpack8(old[u], o);
                float ss = 0.f;
#pragma unroll
                for (int i = 0; i < 8; ++i) { v[i] -= mean[i]; ss += v[i] * v[i]; }
#pragma unroll
                for (int off = LPR / 2; off > 0; off >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, off);
                const float inv = rsqrtf(ss / (float)F + 1.0e-6f);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    nw[i] = __fadd_rn(__fmul_rn(v[i] * inv, 0.25f), __fmul_rn(0.1f, o[i]));
                    carried[i] = __fadd_rn(__fmul_rn(nw[i], 0.2f), __fmul_rn(nw[i], 0.8f));
                }
                if (rr < r1) {
                    if (PRE) reinterpret_cast<uint4*>(PRE + rr * ld_pre)[li] = pack8(nw);
                    reinterpret_cast<uint4*>(STATE + rr * ld_state)[li] = pack8(carried);
                }
            }
        }
        __syncthreads();
    }
}


__device__ __forceinline__ int graph_clauses_unsat(const UnitGraphDev& g, int lg, size_t rowbase,
                                                   const unsigned char* bits, int tid, int nthreads) {
    int unsat = 0;
    const int c0 = __ldg(g.clause_seg + lg), c1 = __ldg(g.clause_seg + lg + 1);
    for (int j = c0 + tid; j < c1; j += nthreads) {
        const int e0 = __ldg(g.cl_rowptr + j), e1 = __ldg(g.cl_rowptr + j + 1);
        int sat = 0;
        for (int e = e0; e < e1; ++e) {
            const int code = __ldg(g.cl_lit + e);
            sat |= ((int)bits[rowbase + (code >> 1)] != (code & 1));   // literal true: bit 1 for +v, bit 0 for -v
        }
        unsat |= !sat;
    }
    return unsat;
}

// Scalars of one denoising step, resident on the device: a captured CUDA graph of one step is replayed for every step of a
// run, so whatever changes from step to step is read through (table, cursor) instead of being baked into the launch.
// The host fills the table with exactly the values it would otherwise pass by value.
struct StepParams {
    float noise_scale;                   // 1 - t/N                                  (DiffusionSampler.py:106)
    float t, ts, norm_plus;              // train_loss scalars                       (model/query_sat.py:41-53)
    float t1, one_minus_alpha;           // posterior scalars                        (DiffusionSampler.py:30-33)
    unsigned int step;                   // denoising step index (Philox counter, latch step)
    int pad_;
    unsigned long long seed, element_offset;
};
__global__ void step_advance_kernel(int* cursor) { *cursor += 1; }

// Logit-map selection (reference model/query_sat.py:289-292,317-320,328-329 with train_loss :40-53)
// and is_batch_sat's per-clause test (utils/sat.py:118-124), one CTA per graph.  Graphs whose
// early-exit group already finished are skipped: their OUT keeps the logits of the round that broke.
__global__ void __launch_bounds__(128)
head_kernel(UnitGraphDev g, int total_graphs, int group_graphs,
            const float* __restrict__ LOGITS, int ld_logits, const int* __restrict__ labels,
            float t, float ts, float norm_plus,
            const int* __restrict__ done, float* __restrict__ OUT, unsigned char* BITS,
            int* __restrict__ graph_sat, float* __restrict__ graph_loss, int* __restrict__ graph_map,
            const StepParams* __restrict__ sp_tab = nullptr, const int* __restrict__ sp_cur = nullptr,
            const int* __restrict__ graph_group = nullptr) {     // early-exit group of each graph (variable groups), or null
    __shared__ float red[4][DSAT_LOGIT_MAPS];
    __shared__ int best_s;
    if (sp_tab) { const StepParams sp = sp_tab[*sp_cur]; t = sp.t; ts = sp.ts; norm_plus = sp.norm_plus; }
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int gid = blockIdx.x;
    if (gid >= total_graphs) return;
    if (done[graph_group ? __ldg(graph_group + gid) : gid / group_graphs]) return;
    const int chain = gid / g.n_graphs, lg = gid % g.n_graphs;
    const int v0 = __ldg(g.var_seg + lg), v1 = __ldg(g.var_seg + lg + 1);
    const size_t rowbase = (size_t)chain * g.n;
    const float wgt = 1.0f / (float)(v1 - v0);

    float part[DSAT_LOGIT_MAPS];
#pragma unroll
    for (int k = 0; k < DSAT_LOGIT_MAPS; ++k) part[k] = 0.f;
    for (int v = v0 + tid; v < v1; v += 128) {
        const size_t row = rowbase + v;
        const float y = (float)__ldg(labels + row);
        const float pa = y * (1.0f - ts) + ts / 2.0f;
        const float4 za = __ldg(reinterpret_cast<const float4*>(LOGITS + row * ld_logits));
        const float4 zb = __ldg(reinterpret_cast<const float4*>(LOGITS + row * ld_logits + 4));
        const float z[8] = {za.x, za.y, za.z, za.w, zb.x, zb.y, zb.z, zb.w};
#pragma unroll
        for (int k = 0; k < DSAT_LOGIT_MAPS; ++k) {
            const float pb = sigmoid_f(z[k]) * (1.0f - t) + t / 2.0f;
            part[k] += (bernoulli_kl(pa, pb) / norm_plus) * wgt;
        }
    }
#pragma unroll
    for (int k = 0; k < DSAT_LOGIT_MAPS; ++k) {
        const float s = warp_sum(part[k]);
        if (lane == 0) red[warp][k] = s;
    }
    __syncthreads();
    if (tid == 0) {
        float tot[DSAT_LOGIT_MAPS];
        int best = 0;
#pragma unroll
        for (int k = 0; k < DSAT_LOGIT_MAPS; ++k) {
            tot[k] = (red[0][k] + red[1][k]) + (red[2][k] + red[3][k]);
            if (tot[k] < tot[best]) best = k;           // ties keep the lowest index (tf.argmin)
        }
        // sum(sort_desc(loss) * [1,4,9,...,64]); the caller divides by 204 (model/query_sat.py:311-313)
        for (int a = 1; a < DSAT_LOGIT_MAPS; ++a) {
            float key = tot[a]; int b = a - 1;
            while (b >= 0 && tot[b] < key) { tot[b + 1] = tot[b]; --b; }
            tot[b + 1] = key;
        }
        float acc = 0.f;
        for (int k = 0; k < DSAT_LOGIT_MAPS; ++k) acc += tot[k] * (float)((k + 1) * (k + 1));
        graph_loss[gid] = acc;
        graph_map[gid] = best;
        best_s = best;
    }
    __syncthreads();
    const int best = best_s;
    for (int v = v0 + tid; v < v1; v += 128) {
        const size_t row = rowbase + v;
        const float z = __ldg(LOGITS + row * ld_logits + best);
        OUT[row] = z;
        BITS[row] = (unsigned char)sigmoid_bit(z);
    }
    __syncthreads();
    const int unsat = __syncthreads_or(graph_clauses_unsat(g, lg, rowbase, BITS, tid, 128));
    if (tid == 0) graph_sat[gid] = !unsat;
}

// Batch-global early exit (reference model/query_sat.py:330-338): a group (= one reference batch of
// graphs) stops at the first round in which every one of its graphs is satisfied.  Also accumulates
// the scalar loss of :311-315,323.  Groups are runs of group_graphs graphs, or [group_seg[i], group_seg[i+1])
// when variable groups are bound (reference batches of several formulas in one launch, dsat_set_batches).
__global__ void group_finalize_kernel(int n_groups, int group_graphs, int total_graphs, int round,
                                      const int* __restrict__ graph_sat, const float* __restrict__ graph_loss,
                                      int* done, int* steps_taken, float* loss_sum, int* rounds_run,
                                      const int* __restrict__ group_seg = nullptr) {
    const int grp = blockIdx.x * blockDim.x + threadIdx.x;
    if (grp >= n_groups || done[grp]) return;
    const int g0 = group_seg ? __ldg(group_seg + grp) : grp * group_graphs;
    const int g1 = group_seg ? __ldg(group_seg + grp + 1) : min(g0 + group_graphs, total_graphs);
    int all = 1;
    float ls = 0.f;
    for (int gi = g0; gi < g1; ++gi) { all &= graph_sat[gi]; ls += graph_loss[gi]; }
    loss_sum[grp] += ls / 204.0f;
    rounds_run[grp] += 1;
    steps_taken[grp] = round;
    if (all) done[grp] = 1;
}

// ------------------------------------------------------------------------------ per-step kernels
struct NoiseSource {
    unsigned long long seed;
    unsigned long long element_offset;   // global index of local row 0 (global_chain0 * n_unit)
    unsigned int step;
    // per-graph noise bases (dsat_set_batches): row r draws element graph_elem0[row_graph[r]] + r, where graph_elem0 holds
    // each graph's base minus its first row (mod 2^64); null = element_offset + r
    const int* row_graph = nullptr;
    const unsigned long long* graph_elem0 = nullptr;
};

__device__ __forceinline__ unsigned long long noise_element(const NoiseSource& ns, long long r) {
    return ns.row_graph ? __ldg(ns.graph_elem0 + __ldg(ns.row_graph + r)) + (unsigned long long)r
                        : ns.element_offset + (unsigned long long)r;
}

// Model-call start: aux columns [normal4 | noisy2 | noise_scale | 0 0 | pad], state = ones, labels.
// If `uniforms_or_null`/X are given this is also the randomized rounding of the denoising step
// (reference model/query_sat.py:55-60, DiffusionSampler.py:107-109): r = floor(x0 + U), x = [r, 1-r].
__global__ void step_begin_kernel(long long n_rows, float noise_scale, float2* X,
                                  const float* __restrict__ noisy_in,      // [n_rows,2] explicit noisy_num or null
                                  const float* __restrict__ uniforms_in,   // [n_rows] or null -> Philox
                                  const int* __restrict__ labels_in,       // [n_rows] or null -> Philox
                                  int* __restrict__ labels,
                                  float* __restrict__ VROW, int ld, int aux_off, __nv_bfloat16* __restrict__ VROW_B,
                                  NoiseSource ns, size_t lo_plane = 0,     // lo_plane > 0: VROW_B is a hi plane with its lo plane that far on
                                  const StepParams* __restrict__ sp_tab = nullptr, const int* __restrict__ sp_cur = nullptr,
                                  int gumbel = 0) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    if (sp_tab) {
        const StepParams sp = sp_tab[*sp_cur];
        noise_scale = sp.noise_scale; ns.seed = sp.seed; ns.element_offset = sp.element_offset; ns.step = sp.step;
    }
    float a, b;
    if (noisy_in) {
        a = noisy_in[2 * r]; b = noisy_in[2 * r + 1];
    } else {
        if (gumbel && !uniforms_in) {
            // Gumbel-argmax over the two classes (the sampler the reference sketches in model/query_sat.py:15-28, hard instead
            // of soft): class k wins with probability x_k / (x_0 + x_1) -- the same distribution as floor(x_0 + U), but not
            // the same sample under the same uniform, so this mode is validated statistically only
            const Philox4 p = noise_draw(ns.seed, noise_element(ns, r), ns.step, 0, STREAM_UNIFORM);
            const float g0 = -logf(-logf(u32_to_unit_float(p.x) + 1e-20f) + 1e-20f);
            const float g1 = -logf(-logf(u32_to_unit_float(p.y) + 1e-20f) + 1e-20f);
            const float2 x = X[r];
            a = (logf(fmaxf(x.x, 1e-20f)) + g0 >= logf(fmaxf(x.y, 1e-20f)) + g1) ? 1.0f : 0.0f;
        } else {
            const float u = uniforms_in ? uniforms_in[r]
                                        : u32_to_unit_float(noise_draw(ns.seed, noise_element(ns, r), ns.step, 0, STREAM_UNIFORM).x);
            a = floorf(X[r].x + u);
        }
        b = 1.0f - a;
    }
    if (X) X[r] = make_float2(a, b);
    if (VROW) {
        float* aux = VROW + (size_t)r * ld + aux_off;
        reinterpret_cast<float4*>(aux)[1] = make_float4(a, b, noise_scale, 0.f);
        reinterpret_cast<float4*>(aux)[2] = make_float4(0.f, 0.f, 0.f, 0.f);
        reinterpret_cast<float4*>(aux)[3] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    if (VROW_B && lo_plane) {   // split planes: a, b are 0/1 (exact in bf16), the noise scale is split
        __nv_bfloat16* auxh = VROW_B + (size_t)r * ld + aux_off;
        __nv_bfloat16* auxl = auxh + lo_plane;
        uint32_t ab_hi, ab_lo, ns_hi, ns_lo;
        split_bf16x2(a, b, ab_hi, ab_lo);
        split_bf16x2(noise_scale, 0.f, ns_hi, ns_lo);
        reinterpret_cast<uint32_t*>(auxh)[2] = ab_hi; reinterpret_cast<uint32_t*>(auxl)[2] = ab_lo;
        reinterpret_cast<uint32_t*>(auxh)[3] = ns_hi; reinterpret_cast<uint32_t*>(auxl)[3] = ns_lo;
#pragma unroll
        for (int i = 4; i < 8; ++i) { reinterpret_cast<uint32_t*>(auxh)[i] = 0u; reinterpret_cast<uint32_t*>(auxl)[i] = 0u; }
    } else if (VROW_B) {   // columns 4..15 of the bf16 aux block (0..3 are the per-round normals)
        __nv_bfloat16* auxb = VROW_B + (size_t)r * ld + aux_off;
        __nv_bfloat162 z = __floats2bfloat162_rn(0.f, 0.f);
        reinterpret_cast<__nv_bfloat162*>(auxb)[2] = __floats2bfloat162_rn(a, b);
        reinterpret_cast<__nv_bfloat162*>(auxb)[3] = __floats2bfloat162_rn(noise_scale, 0.f);
#pragma unroll
        for (int i = 4; i < 8; ++i) reinterpret_cast<__nv_bfloat162*>(auxb)[i] = z;
    }
    labels[r] = labels_in ? labels_in[r]
                          : (int)(noise_draw(ns.seed, noise_element(ns, r), ns.step, 0, STREAM_LABEL).x & 1u);
}

// Fresh N(0,1)[.,4] every round (reference model/query_sat.py:239).
__global__ void round_noise_kernel(long long n_rows, const float* __restrict__ normals_in /*[n_rows,4] or null*/,
                                   float* __restrict__ VROW, int ld, int aux_off, __nv_bfloat16* __restrict__ VROW_B,
                                   NoiseSource ns, unsigned int round, size_t lo_plane = 0,
                                   const StepParams* __restrict__ sp_tab = nullptr, const int* __restrict__ sp_cur = nullptr,
                                   SkipInfo skip = SkipInfo{nullptr, 1}, int rows_per_chain = 1) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    if (chain_done(skip, (int)(r / rows_per_chain))) return;
    if (sp_tab) {
        const StepParams sp = sp_tab[*sp_cur];
        ns.seed = sp.seed; ns.element_offset = sp.element_offset; ns.step = sp.step;
    }
    float4 nrm;
    if (normals_in) {
        nrm = __ldg(reinterpret_cast<const float4*>(normals_in) + r);
    } else {
        Philox4 p = noise_draw(ns.seed, noise_element(ns, r), ns.step, round, STREAM_NORMAL);
        box_muller(p.x, p.y, nrm.x, nrm.y);
        box_muller(p.z, p.w, nrm.z, nrm.w);
    }
    if (VROW) reinterpret_cast<float4*>(VROW + (size_t)r * ld + aux_off)[0] = nrm;
    if (VROW_B && lo_plane) {
        uint2 hi, lo;
        split_bf16x2(nrm.x, nrm.y, hi.x, lo.x);
        split_bf16x2(nrm.z, nrm.w, hi.y, lo.y);
        __nv_bfloat16* auxh = VROW_B + (size_t)r * ld + aux_off;
        *reinterpret_cast<uint2*>(auxh) = hi;
        *reinterpret_cast<uint2*>(auxh + lo_plane) = lo;
    } else if (VROW_B) {
        __nv_bfloat162* auxb = reinterpret_cast<__nv_bfloat162*>(VROW_B + (size_t)r * ld + aux_off);
        auxb[0] = __floats2bfloat162_rn(nrm.x, nrm.y);
        auxb[1] = __floats2bfloat162_rn(nrm.z, nrm.w);
    }
}

__global__ void fill_cols_bf16_kernel(__nv_bfloat16* __restrict__ dst, int ld, long long rows, int cols8, float value) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * cols8) return;
    const long long r = i / cols8; const int c = (int)(i % cols8);
    __nv_bfloat162 v = __floats2bfloat162_rn(value, value);
    uint4 pack;
    pack.x = pack.y = pack.z = pack.w = *reinterpret_cast<uint32_t*>(&v);
    reinterpret_cast<uint4*>(dst + (size_t)r * ld)[c] = pack;
}

__global__ void fill_cols_kernel(float* __restrict__ dst, int ld, long long rows, int cols4, float value) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * cols4) return;
    const long long r = i / cols4; const int c = (int)(i % cols4);
    reinterpret_cast<float4*>(dst + (size_t)r * ld)[c] = make_float4(value, value, value, value);
}

// End of a denoising step, one CTA per graph: p = sigmoid(prediction); posterior
// q(x_{t-1} | x_t, x0_hat) (reference DiffusionSampler.py:29-37,127-129, written exactly as there:
// x_hat uses t1); xx = round(p); first-SAT latch (:154-170).
struct PosteriorScalars { float t1, one_minus_alpha; };

__global__ void __launch_bounds__(128)
step_end_kernel(UnitGraphDev g, int total_graphs, const float* __restrict__ OUT, float2* X,
                PosteriorScalars ps, int step, unsigned char* LAST, unsigned char* LATCH,
                int* __restrict__ latch_step, int* __restrict__ sat_now,
                const StepParams* __restrict__ sp_tab = nullptr, const int* __restrict__ sp_cur = nullptr) {
    const int tid = threadIdx.x;
    const int gid = blockIdx.x;
    if (gid >= total_graphs) return;
    if (sp_tab) {
        const StepParams sp = sp_tab[*sp_cur];
        ps.t1 = sp.t1; ps.one_minus_alpha = sp.one_minus_alpha; step = (int)sp.step;
    }
    const int chain = gid / g.n_graphs, lg = gid % g.n_graphs;
    const int v0 = __ldg(g.var_seg + lg), v1 = __ldg(g.var_seg + lg + 1);
    const size_t rowbase = (size_t)chain * g.n;
    const float t1 = ps.t1, oma = ps.one_minus_alpha;
    for (int v = v0 + tid; v < v1; v += 128) {
        const size_t row = rowbase + v;
        const float p = sigmoid_f(OUT[row]);
        const float2 x = X[row];
        const float h0 = (1.0f - p) * (1.0f - t1) + t1 / 2.0f;      // distribution_at_time(x0, t1)
        const float h1 = p * (1.0f - t1) + t1 / 2.0f;
        const float u0 = (x.x * (1.0f - oma) + oma / 2.0f) * h0;     // distribution_at_time(x, 1-alpha_t) * x_new
        const float u1 = (x.y * (1.0f - oma) + oma / 2.0f) * h1;
        const float s = (u0 + u1) + 1.0e-8f;
        X[row] = make_float2(u0 / s, u1 / s);
        LAST[row] = (unsigned char)(p > 0.5f ? 1 : 0);
    }
    __syncthreads();
    const int unsat = __syncthreads_or(graph_clauses_unsat(g, lg, rowbase, LAST, tid, 128));
    if (tid == 0) sat_now[gid] = !unsat;
    if (!unsat && latch_step[gid] < 0) {
        for (int v = v0 + tid; v < v1; v += 128) LATCH[rowbase + v] = LAST[rowbase + v];
        __syncthreads();
        if (tid == 0) latch_step[gid] = step;
    }
}

// Final assignment of a graph = latched bits if any, else the last step's (reference :182-185);
// packed little-endian into 64-bit words, x1 = bit 0 (utils/VariableAssignment.py:63-69).
__global__ void __launch_bounds__(128)
pack_assignments_kernel(UnitGraphDev g, int total_graphs, int words_per_graph,
                        const unsigned char* LAST, const unsigned char* LATCH, const int* __restrict__ latch_step,
                        unsigned long long* __restrict__ packed, unsigned char* __restrict__ is_sat,
                        unsigned char* FINAL) {
    const int tid = threadIdx.x;
    const int gid = blockIdx.x;
    if (gid >= total_graphs) return;
    const int chain = gid / g.n_graphs, lg = gid % g.n_graphs;
    const int v0 = __ldg(g.var_seg + lg), v1 = __ldg(g.var_seg + lg + 1);
    const size_t rowbase = (size_t)chain * g.n;
    const unsigned char* src = latch_step[gid] >= 0 ? LATCH : LAST;
    for (int v = v0 + tid; v < v1; v += 128) FINAL[rowbase + v] = src[rowbase + v];
    for (int w = tid; w < words_per_graph; w += 128) {
        unsigned long long word = 0ull;
        const int b0 = v0 + w * 64;
        for (int i = 0; i < 64 && b0 + i < v1; ++i)
            word |= (unsigned long long)(src[rowbase + b0 + i] & 1) << i;
        packed[(size_t)gid * words_per_graph + w] = word;
    }
    __syncthreads();
    const int unsat = __syncthreads_or(graph_clauses_unsat(g, lg, rowbase, FINAL, tid, 128));
    if (tid == 0) is_sat[gid] = (unsigned char)(!unsat);
}

}  // namespace dsat
