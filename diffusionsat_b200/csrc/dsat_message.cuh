// Message passing over the clause-literal graph: segment-sum SpMM kernels that share ONE adjacency
// (the unit graph's CSR/CSC) across all chains.  Rows of chain c live at offset c*rows_per_chain, so
// the index arrays are read once per warp and stay in L1/L2 for every chain.
//
// One warp produces one output row; lane l owns the columns described in dsat_common.cuh (float4 per
// lane at width 128).  Gathered rows are 512-byte contiguous (width 128, fp32): one fully coalesced
// request per edge, and the edge loop is unrolled so that several requests are in flight per warp.
//
//   clause_gather  : reference model/query_sat.py:241 (loss/sat.py:132-135) and :255-256
//   literal_gather : reference model/query_sat.py:245-246 (closed form of the GradientTape) and :269-273
//   spmm_*         : the same segment-sum cores on caller buffers (roofline sweeps, SURVEY.md section 8d)
#pragma once
#include "dsat_common.cuh"

namespace dsat {

struct UnitGraphDev {
    int n, m, nnz, n_graphs;            // unit sizes
    const int* cl_rowptr;               // [m+1]
    const int* cl_lit;                  // [nnz] literal codes 2*var+sign
    const int* lit_rowptr;              // [2n+1]
    const int* lit_clause;              // [nnz]
    const int* var_seg;                 // [n_graphs+1]
    const int* clause_seg;              // [n_graphs+1]
    const float* deg_w;                 // [2n]  rsqrt(max(deg(lit),1))
    const float* vdeg_w;                // [n]   rsqrt(max(deg(+v)+deg(-v),1))   (the reference's factor 4 is carried by cl4)
    const float* rev_w;                 // [m]   rsqrt(max(|clause|,1))
    const int* var_order;               // [n]   variables by descending degree (rows of one warp pass get similar lengths)
    // 16-bit copies of the adjacency for the shared-memory gathers (null when a count does not fit 16 bits):
    //   cl_idx16  = [cl_rowptr (m+1) | cl_lit (nnz)],  lit_idx16 = [lit_rowptr (2n+1) | lit_clause (nnz) | var_order (n)]
    // each section starts on a 16-byte boundary; *_vecs = length in 16-byte units
    const unsigned short* cl_idx16;
    const unsigned short* lit_idx16;
    int cl_idx16_vecs, lit_idx16_vecs;
    int cl_col_off, lit_col_off, lit_ord_off;      // section starts, in elements
};

constexpr int GATHER_WARPS = 8;

// Position of a warp in the flattened (chain, row) space of a grid-stride kernel.  The stride is split into
// (chains, rows) once, so a step costs two adds and a compare instead of a 64-bit division per row (which made
// the short-row kernels issue-bound: ~60 % issue-slot use for four memory operations per row).
struct RowCursor {
    int c, pos;           // chain, row position inside the chain
    int step_c, step_pos; // the grid stride, decomposed
};
__device__ __forceinline__ RowCursor row_cursor(long long first, long long stride, int rows) {
    RowCursor k;
    k.c = (int)(first / rows);
    k.pos = (int)(first - (long long)k.c * rows);
    k.step_c = (int)(stride / rows);
    k.step_pos = (int)(stride - (long long)k.step_c * rows);
    return k;
}
__device__ __forceinline__ void row_cursor_step(RowCursor& k, int rows) {
    k.c += k.step_c;
    k.pos += k.step_pos;
    if (k.pos >= rows) { k.pos -= rows; ++k.c; }
}

// ------------------------------------------------------------------------------ clause side
// For clause j of chain c:
//   cmsg[j] = rev_w[j] * sum_{lit in j} LIT[var(lit)][sign(lit)*Q : +Q]
//   cl4[j]  = 4 * exp(-sum_{lit in j} SP[var(lit)][sign(lit)*Q : +Q])        SP = softplus(+-query)
// LIT rows have leading dimension ld_lit (2Q used), SP rows ld_sp with the pair starting at column sp_off.
// Output goes to OUT[(c*m + j)*ld_out + out_off : +2Q] = [cmsg | cl4].
template <int V, typename T>
__global__ void __launch_bounds__(GATHER_WARPS * 32)
clause_gather_kernel(UnitGraphDev g, int chains,
                     const T* __restrict__ LIT, int ld_lit,
                     const T* __restrict__ SP, int ld_sp, int sp_off,
                     T* __restrict__ OUT, int ld_out, int out_off,
                     __nv_bfloat16* __restrict__ OUT_HI = nullptr, size_t out_plane = 0,    // split-plane output instead of OUT
                     SkipInfo skip = SkipInfo{nullptr, 1}) {
    constexpr int Q = 32 * V;
    const int lane = threadIdx.x & 31;
    RowCursor cur = row_cursor((long long)blockIdx.x * GATHER_WARPS + (threadIdx.x >> 5),
                               (long long)gridDim.x * GATHER_WARPS, g.m);
    for (; cur.c < chains; row_cursor_step(cur, g.m)) {
        const int c = cur.c, j = cur.pos;
        if (chain_done(skip, c)) continue;
        const int e0 = __ldg(g.cl_rowptr + j), e1 = __ldg(g.cl_rowptr + j + 1);
        DSAT_CHECK(j >= 0 && j < g.m && 0 <= e0 && e0 <= e1 && e1 <= g.nnz);
        const size_t vbase = (size_t)c * g.n;
        LaneVec<V> acc_l, acc_s;
#pragma unroll
        for (int i = 0; i < V; ++i) { acc_l.v[i] = 0.f; acc_s.v[i] = 0.f; }
        int e = e0;
        for (; e + 3 <= e1; e += 3) {   // 3-SAT fast path: three edges in flight
            int c0 = __ldg(g.cl_lit + e), c1 = __ldg(g.cl_lit + e + 1), c2 = __ldg(g.cl_lit + e + 2);
            DSAT_CHECK((unsigned)c0 < 2u * g.n && (unsigned)c1 < 2u * g.n && (unsigned)c2 < 2u * g.n);
            const size_t r0 = vbase + (c0 >> 1), r1 = vbase + (c1 >> 1), r2 = vbase + (c2 >> 1);
            LaneVec<V> l0 = lane_load_t<V, T>(LIT + r0 * ld_lit + (c0 & 1) * Q, lane);
            LaneVec<V> l1 = lane_load_t<V, T>(LIT + r1 * ld_lit + (c1 & 1) * Q, lane);
            LaneVec<V> l2 = lane_load_t<V, T>(LIT + r2 * ld_lit + (c2 & 1) * Q, lane);
            LaneVec<V> s0 = lane_load_t<V, T>(SP + r0 * ld_sp + sp_off + (c0 & 1) * Q, lane);
            LaneVec<V> s1 = lane_load_t<V, T>(SP + r1 * ld_sp + sp_off + (c1 & 1) * Q, lane);
            LaneVec<V> s2 = lane_load_t<V, T>(SP + r2 * ld_sp + sp_off + (c2 & 1) * Q, lane);
#pragma unroll
            for (int i = 0; i < V; ++i) {
                acc_l.v[i] = ((acc_l.v[i] + l0.v[i]) + l1.v[i]) + l2.v[i];
                acc_s.v[i] = ((acc_s.v[i] + s0.v[i]) + s1.v[i]) + s2.v[i];
            }
        }
        for (; e < e1; ++e) {
            int c0 = __ldg(g.cl_lit + e);
            DSAT_CHECK((unsigned)c0 < 2u * g.n);
            const size_t r0 = vbase + (c0 >> 1);
            LaneVec<V> l0 = lane_load_t<V, T>(LIT + r0 * ld_lit + (c0 & 1) * Q, lane);
            LaneVec<V> s0 = lane_load_t<V, T>(SP + r0 * ld_sp + sp_off + (c0 & 1) * Q, lane);
#pragma unroll
            for (int i = 0; i < V; ++i) { acc_l.v[i] += l0.v[i]; acc_s.v[i] += s0.v[i]; }
        }
        const float rw = __ldg(g.rev_w + j);
#pragma unroll
        for (int i = 0; i < V; ++i) {
            acc_l.v[i] *= rw;
            acc_s.v[i] = 4.0f * expf(-acc_s.v[i]);
        }
        if (OUT_HI) {
            __nv_bfloat16* dsth = OUT_HI + ((size_t)c * g.m + j) * ld_out + out_off;
            lane_store_split<V>(dsth, out_plane, lane, acc_l);
            lane_store_split<V>(dsth + Q, out_plane, lane, acc_s);
            continue;
        }
        T* dst = OUT + ((size_t)c * g.m + j) * ld_out + out_off;
        lane_store_t<V, T>(dst, lane, acc_l);
        lane_store_t<V, T>(dst + Q, lane, acc_s);
    }
}

// ----------------------------------------------------------------------------- literal side
// For variable v of chain c (pos = literal code 2v, neg = 2v+1):
//   S4+- = sum_{clauses j containing +-v} cl4[j]            (cl4 = 4*clauses_loss)
//   g[v] = (-sigma(q)*S4+ + sigma(-q)*S4-) * vdeg_w[v]      == variables_grad of reference :245-246
//   vloss+-[v] = deg_w[+-v] * sum_{j containing +-v} MSG[j] == variables_loss_pos/neg of reference :269-273
// CL4 rows: ld_cl, column cl_off; MSG rows: ld_msg, column 0; QRY rows: ld_q (query in columns [0,Q)).
// Output OUT[(c*n+v)*ld_out + out_off : +3Q] = [g | vloss+ | vloss-].
template <int V, typename T>
__global__ void __launch_bounds__(GATHER_WARPS * 32)
literal_gather_kernel(UnitGraphDev g, int chains,
                      const T* __restrict__ CL4, int ld_cl, int cl_off,
                      const T* __restrict__ MSG, int ld_msg,
                      const T* __restrict__ QRY, int ld_q,
                      T* __restrict__ OUT, int ld_out, int out_off,
                      __nv_bfloat16* __restrict__ OUT_HI = nullptr, size_t out_plane = 0,    // split-plane output instead of OUT
                      const __nv_bfloat16* __restrict__ CL4_HI = nullptr, size_t cl_plane = 0,    // split-plane CL4 instead of CL4
                      SkipInfo skip = SkipInfo{nullptr, 1}) {
    constexpr int Q = 32 * V;
    const int lane = threadIdx.x & 31;
    RowCursor cur = row_cursor((long long)blockIdx.x * GATHER_WARPS + (threadIdx.x >> 5),
                               (long long)gridDim.x * GATHER_WARPS, g.n);
    for (; cur.c < chains; row_cursor_step(cur, g.n)) {
        const int c = cur.c, v = cur.pos;
        if (chain_done(skip, c)) continue;
        const size_t cbase = (size_t)c * g.m;
        LaneVec<V> s4[2], ms[2];
#pragma unroll
        for (int sgn = 0; sgn < 2; ++sgn) {
#pragma unroll
            for (int i = 0; i < V; ++i) { s4[sgn].v[i] = 0.f; ms[sgn].v[i] = 0.f; }
            const int code = 2 * v + sgn;
            const int e0 = __ldg(g.lit_rowptr + code), e1 = __ldg(g.lit_rowptr + code + 1);
            DSAT_CHECK(code < 2 * g.n && 0 <= e0 && e0 <= e1 && e1 <= g.nnz);
            int e = e0;
            for (; e + 2 <= e1; e += 2) {
                DSAT_CHECK((unsigned)__ldg(g.lit_clause + e) < (unsigned)g.m && (unsigned)__ldg(g.lit_clause + e + 1) < (unsigned)g.m);
                const size_t j0 = cbase + __ldg(g.lit_clause + e), j1 = cbase + __ldg(g.lit_clause + e + 1);
                LaneVec<V> a0 = CL4_HI ? lane_load_split_rw<V>(CL4_HI + j0 * ld_cl + cl_off, cl_plane, lane)
                                       : lane_load_t<V, T>(CL4 + j0 * ld_cl + cl_off, lane);
                LaneVec<V> a1 = CL4_HI ? lane_load_split_rw<V>(CL4_HI + j1 * ld_cl + cl_off, cl_plane, lane)
                                       : lane_load_t<V, T>(CL4 + j1 * ld_cl + cl_off, lane);
                LaneVec<V> b0 = lane_load_t<V, T>(MSG + j0 * ld_msg, lane);
                LaneVec<V> b1 = lane_load_t<V, T>(MSG + j1 * ld_msg, lane);
#pragma unroll
                for (int i = 0; i < V; ++i) {
                    s4[sgn].v[i] = (s4[sgn].v[i] + a0.v[i]) + a1.v[i];
                    ms[sgn].v[i] = (ms[sgn].v[i] + b0.v[i]) + b1.v[i];
                }
            }
            for (; e < e1; ++e) {
                const size_t j0 = cbase + __ldg(g.lit_clause + e);
                LaneVec<V> a0 = CL4_HI ? lane_load_split_rw<V>(CL4_HI + j0 * ld_cl + cl_off, cl_plane, lane)
                                       : lane_load_t<V, T>(CL4 + j0 * ld_cl + cl_off, lane);
                LaneVec<V> b0 = lane_load_t<V, T>(MSG + j0 * ld_msg, lane);
#pragma unroll
                for (int i = 0; i < V; ++i) { s4[sgn].v[i] += a0.v[i]; ms[sgn].v[i] += b0.v[i]; }
            }
        }
        const size_t row = (size_t)c * g.n + v;
        LaneVec<V> q = lane_load_t<V, T>(QRY + row * ld_q, lane);
        const float vw = __ldg(g.vdeg_w + v);
        const float dwp = __ldg(g.deg_w + 2 * v), dwn = __ldg(g.deg_w + 2 * v + 1);
        LaneVec<V> grad;
#pragma unroll
        for (int i = 0; i < V; ++i) {
            const float sg = sigmoid_f(q.v[i]), sgn_ = sigmoid_f(-q.v[i]);
            grad.v[i] = (-sg * s4[0].v[i] + sgn_ * s4[1].v[i]) * vw;
            ms[0].v[i] *= dwp;
            ms[1].v[i] *= dwn;
        }
        if (OUT_HI) {
            __nv_bfloat16* dsth = OUT_HI + row * ld_out + out_off;
            lane_store_split<V>(dsth, out_plane, lane, grad);
            lane_store_split<V>(dsth + Q, out_plane, lane, ms[0]);
            lane_store_split<V>(dsth + 2 * Q, out_plane, lane, ms[1]);
            continue;
        }
        T* dst = OUT + row * ld_out + out_off;
        lane_store_t<V, T>(dst, lane, grad);
        lane_store_t<V, T>(dst + Q, lane, ms[0]);
        lane_store_t<V, T>(dst + 2 * Q, lane, ms[1]);
    }
}

// Grid of a grid-stride gather kernel: exactly one resident wave (occupancy x SM count).  More blocks than fit at
// once would make every later wave sweep all chains again (block b strides over the whole row range), so each
// chain's gathered table would be fetched from HBM once per wave instead of once (measured 2.7x DRAM reads).
template <typename Kernel>
inline int gather_grid(Kernel kernel, long long total_rows, int rows_per_block, int sm_count) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, GATHER_WARPS * 32, 0) != cudaSuccess || per_sm < 1)
        per_sm = 1;
    long long blocks = (total_rows + rows_per_block - 1) / rows_per_block;
    const long long cap = (long long)sm_count * per_sm;
    if (blocks > cap) blocks = cap;
    return (int)(blocks < 1 ? 1 : blocks);
}

}  // namespace dsat

// ===================================================================== shared-memory staged variants
// For small formulas the gathered tables of one chain fit in shared memory: a CTA copies the chain's
// rows in once with coalesced 16-byte loads (each row read from L2/HBM exactly once) and every edge
// then reads shared memory instead of L2.  blockIdx.x = chain, blockIdx.y = feature slice of width W
// (the features are independent, so a slice is a complete sub-problem).  bf16 storage, fp32 sums.
// Work split inside a warp: LPR = W/8 lanes share one output row (16 bytes = 8 features per lane), so a
// warp produces 32/LPR rows per pass: the index loads and address arithmetic are amortised over 8
// features instead of 4.
namespace dsat {

struct Acc8 { float v[8]; };

__device__ __forceinline__ void acc8_zero(Acc8& a) {
#pragma unroll
    for (int i = 0; i < 8; ++i) a.v[i] = 0.f;
}
// fp32 accumulator += one bf16 half of a packed pair, in ONE instruction: sm_100a's mixed-precision add
// (PTX add.rn.f32.bf16, SASS FHADD.BF16 with an .H0/.H1 operand selector) widens the bf16 operand exactly and rounds the
// fp32 sum once -- bit-identical to widening by shift/mask and an FADD, at half the instructions.  The gathers are
// issue-bound (ncu: 73-88 % issue-slot use), and unpack + add was all of their inner loop.
__device__ __forceinline__ float add_bf16_lo(float acc, uint32_t pair) {
    float d;
    asm("add.rn.f32.bf16 %0, %1, %2;" : "=f"(d) : "h"((unsigned short)(pair & 0xffffu)), "f"(acc));
    return d;
}
__device__ __forceinline__ float add_bf16_hi(float acc, uint32_t pair) {
    float d;
    asm("add.rn.f32.bf16 %0, %1, %2;" : "=f"(d) : "h"((unsigned short)(pair >> 16)), "f"(acc));
    return d;
}
// add 8 bf16 (one uint4) to 8 fp32 accumulators
__device__ __forceinline__ void acc8_add(Acc8& a, const uint4& w) {
    const uint32_t u[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        a.v[2 * i] = add_bf16_lo(a.v[2 * i], u[i]);
        a.v[2 * i + 1] = add_bf16_hi(a.v[2 * i + 1], u[i]);
    }
}
__device__ __forceinline__ void unpack8(const uint4& w, float (&f)[8]) {
    const uint32_t u[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        f[2 * i] = __uint_as_float(u[i] << 16);
        f[2 * i + 1] = __uint_as_float(u[i] & 0xffff0000u);
    }
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
    uint4 w;
    __nv_bfloat162 p0 = __floats2bfloat162_rn(f[0], f[1]), p1 = __floats2bfloat162_rn(f[2], f[3]);
    __nv_bfloat162 p2 = __floats2bfloat162_rn(f[4], f[5]), p3 = __floats2bfloat162_rn(f[6], f[7]);
    w.x = *reinterpret_cast<uint32_t*>(&p0); w.y = *reinterpret_cast<uint32_t*>(&p1);
    w.z = *reinterpret_cast<uint32_t*>(&p2); w.w = *reinterpret_cast<uint32_t*>(&p3);
    return w;
}

// streamed 16-byte load that does not allocate in L1: with ~220 KB of the SM carved out as shared memory only a few
// KB of L1 remain, and they should keep the adjacency (read by every CTA) rather than rows that are used once
__device__ __forceinline__ uint4 ldg_stream(const uint4* p) {
    uint4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}

// asynchronous 16-byte global -> shared copy (LDGSTS, L2 only): no register round trip, so a thread can have all of
// its pieces in flight at once instead of eight
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
    asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
}

template <typename T>
__device__ __forceinline__ void stage_rows_async(T* __restrict__ dst, const T* __restrict__ src, int rows, int ld_src,
                                                 int width, int tid, int nthreads) {
    const int vec_per_row = width * (int)sizeof(T) / 16;
    const int total = rows * vec_per_row;
    for (int i = tid; i < total; i += nthreads) {
        const int r = i / vec_per_row, k = i % vec_per_row;
        cp_async16(reinterpret_cast<uint4*>(dst + (size_t)r * width) + k, reinterpret_cast<const uint4*>(src + (size_t)r * ld_src) + k);
    }
}

template <typename T>
__device__ __forceinline__ void stage_rows(T* __restrict__ dst, const T* __restrict__ src, int rows, int ld_src,
                                           int width, int tid, int nthreads) {
    const int vec_per_row = width * (int)sizeof(T) / 16;
    const int total = rows * vec_per_row;
    constexpr int U = 8;                                    // independent 16-byte loads in flight per thread
    for (int i0 = tid; i0 < total; i0 += U * nthreads) {
        uint4 a[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = i0 + u * nthreads;
            if (i < total) a[u] = ldg_stream(reinterpret_cast<const uint4*>(src + (size_t)(i / vec_per_row) * ld_src) + i % vec_per_row);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = i0 + u * nthreads;
            if (i < total) reinterpret_cast<uint4*>(dst + (size_t)(i / vec_per_row) * width)[i % vec_per_row] = a[u];
        }
    }
}

// clause side: tables LIT[2n][W] and SP[2n][W] of the chain's slice (row = literal code 2*var+sign)
template <int W, bool SI>
__global__ void __launch_bounds__(512, 3)     // 40 registers: three CTAs per SM measured best (4 spills, 2 leaves latency exposed)
clause_gather_smem_kernel(UnitGraphDev g, int Q,
                          const __nv_bfloat16* __restrict__ LIT, int ld_lit,
                          const __nv_bfloat16* __restrict__ SP, int ld_sp, int sp_off,
                          __nv_bfloat16* __restrict__ OUT, int ld_out, int out_off, SkipInfo skip = SkipInfo{nullptr, 1}) {
    if (chain_done(skip, (int)blockIdx.x)) return;     // the whole CTA works on one chain
    using T = __nv_bfloat16;
    constexpr int LPR = W / 8, RPW = 32 / LPR;
    extern __shared__ __align__(16) uint8_t gsm[];
    T* t_lit = reinterpret_cast<T*>(gsm);
    T* t_sp = t_lit + (size_t)2 * g.n * W;
    // SI: the adjacency is staged too (16-bit).  Read from global it costs an L2 round trip per entry, because the
    // shared-memory carve-out leaves almost no L1, and that chain of dependent loads dominated the gather phase.
    const unsigned short* s_idx = reinterpret_cast<const unsigned short*>(t_sp + (size_t)2 * g.n * W);
    const int chain = blockIdx.x, slice = blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const int sub = lane / LPR, li = lane % LPR;
    const size_t vbase = (size_t)chain * g.n;
    {   // stage both tables with asynchronous copies (all pieces of a thread in flight at once)
        const int total = 2 * g.n * LPR;                    // (variable, sign, 16-byte piece)
        for (int i = tid; i < total; i += blockDim.x) {
            const int code = i / LPR, k = i % LPR, v = code >> 1, sgn = code & 1;
            cp_async16(reinterpret_cast<uint4*>(t_lit + (size_t)code * W) + k,
                       reinterpret_cast<const uint4*>(LIT + (vbase + v) * ld_lit + sgn * Q + slice * W) + k);
            cp_async16(reinterpret_cast<uint4*>(t_sp + (size_t)code * W) + k,
                       reinterpret_cast<const uint4*>(SP + (vbase + v) * ld_sp + sp_off + sgn * Q + slice * W) + k);
        }
    }
    if constexpr (SI) {
        uint4* d = reinterpret_cast<uint4*>(const_cast<unsigned short*>(s_idx));
        for (int i = tid; i < g.cl_idx16_vecs; i += blockDim.x) d[i] = __ldg(reinterpret_cast<const uint4*>(g.cl_idx16) + i);
    }
    cp_async_wait_all();
    __syncthreads();
    for (int j0 = warp * RPW; j0 < g.m; j0 += nwarps * RPW) {
        const int j = j0 + sub;
        const bool live = j < g.m;
        int e0 = 0, e1 = 0;
        if (live) {
            if constexpr (SI) { e0 = s_idx[j]; e1 = s_idx[j + 1]; }
            else { e0 = __ldg(g.cl_rowptr + j); e1 = __ldg(g.cl_rowptr + j + 1); }
        }
        Acc8 al, as;
        acc8_zero(al); acc8_zero(as);
        int e = e0;
        for (; e + 3 <= e1; e += 3) {      // 3-SAT: all six table reads of a clause in flight before the first add
            const int c0 = SI ? (int)s_idx[g.cl_col_off + e] : __ldg(g.cl_lit + e);
            const int c1 = SI ? (int)s_idx[g.cl_col_off + e + 1] : __ldg(g.cl_lit + e + 1);
            const int c2 = SI ? (int)s_idx[g.cl_col_off + e + 2] : __ldg(g.cl_lit + e + 2);
            DSAT_CHECK((unsigned)c0 < 2u * g.n && (unsigned)c1 < 2u * g.n && (unsigned)c2 < 2u * g.n && e + 3 <= g.nnz);
            const uint4 l0 = reinterpret_cast<const uint4*>(t_lit + (size_t)c0 * W)[li];
            const uint4 p0 = reinterpret_cast<const uint4*>(t_sp + (size_t)c0 * W)[li];
            const uint4 l1 = reinterpret_cast<const uint4*>(t_lit + (size_t)c1 * W)[li];
            const uint4 p1 = reinterpret_cast<const uint4*>(t_sp + (size_t)c1 * W)[li];
            const uint4 l2 = reinterpret_cast<const uint4*>(t_lit + (size_t)c2 * W)[li];
            const uint4 p2 = reinterpret_cast<const uint4*>(t_sp + (size_t)c2 * W)[li];
            acc8_add(al, l0); acc8_add(as, p0);
            acc8_add(al, l1); acc8_add(as, p1);
            acc8_add(al, l2); acc8_add(as, p2);
        }
        for (; e < e1; ++e) {
            const int code = SI ? (int)s_idx[g.cl_col_off + e] : __ldg(g.cl_lit + e);
            acc8_add(al, reinterpret_cast<const uint4*>(t_lit + (size_t)code * W)[li]);
            acc8_add(as, reinterpret_cast<const uint4*>(t_sp + (size_t)code * W)[li]);
        }
        if (live) {
            const float rw = __ldg(g.rev_w + j);
            float ol[8], os[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) { ol[i] = al.v[i] * rw; os[i] = 4.0f * __expf(-as.v[i]); }
            T* dst = OUT + ((size_t)chain * g.m + j) * ld_out + out_off + slice * W;
            reinterpret_cast<uint4*>(dst)[li] = pack8(ol);
            reinterpret_cast<uint4*>(dst + Q)[li] = pack8(os);
        }
    }
}

// literal side: tables CL4[m][W] and MSG[m][W] of the chain's slice
template <int W, bool SI>
__global__ void __launch_bounds__(1024)
literal_gather_smem_kernel(UnitGraphDev g, int Q,
                           const __nv_bfloat16* __restrict__ CL4, int ld_cl, int cl_off,
                           const __nv_bfloat16* __restrict__ MSG, int ld_msg,
                           const __nv_bfloat16* __restrict__ QRY, int ld_q,
                           __nv_bfloat16* __restrict__ OUT, int ld_out, int out_off, SkipInfo skip = SkipInfo{nullptr, 1}) {
    if (chain_done(skip, (int)blockIdx.x)) return;     // the whole CTA works on one chain
    using T = __nv_bfloat16;
    constexpr int LPR = W / 8, RPW = 32 / LPR;
    extern __shared__ __align__(16) uint8_t gsm[];
    T* t_cl = reinterpret_cast<T*>(gsm);
    T* t_ms = t_cl + (size_t)g.m * W;
    const unsigned short* s_idx = reinterpret_cast<const unsigned short*>(t_ms + (size_t)g.m * W);   // see clause side
    const int chain = blockIdx.x, slice = blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const int sub = lane / LPR, li = lane % LPR;
    const size_t cbase = (size_t)chain * g.m;
    if (ld_cl == W && ld_msg == W) {   // dense [m, W] tables (Q == W): constant row pitch
        stage_rows_async<T>(t_cl, CL4 + cbase * W + cl_off, g.m, W, W, tid, blockDim.x);
        stage_rows_async<T>(t_ms, MSG + cbase * W, g.m, W, W, tid, blockDim.x);
    } else {
        stage_rows_async<T>(t_cl, CL4 + cbase * ld_cl + cl_off + slice * W, g.m, ld_cl, W, tid, blockDim.x);
        stage_rows_async<T>(t_ms, MSG + cbase * ld_msg + slice * W, g.m, ld_msg, W, tid, blockDim.x);
    }
    if constexpr (SI) {
        uint4* d = reinterpret_cast<uint4*>(const_cast<unsigned short*>(s_idx));
        for (int i = tid; i < g.lit_idx16_vecs; i += blockDim.x) d[i] = __ldg(reinterpret_cast<const uint4*>(g.lit_idx16) + i);
    }
    cp_async_wait_all();
    __syncthreads();
    // variables are taken in order of descending degree: the RPW rows of a pass then have similar entry counts (a
    // pass runs for its longest row), and the heaviest passes are dealt first
    for (int v0 = warp * RPW; v0 < g.n; v0 += nwarps * RPW) {
        const bool live = v0 + sub < g.n;
        int v = 0;
        if (live) v = SI ? (int)s_idx[g.lit_ord_off + v0 + sub] : __ldg(g.var_order + v0 + sub);
        // the epilogue's global operands are requested first: their L2 latency hides under the entry loops
        const size_t row = (size_t)chain * g.n + v;
        T* dst = OUT + row * ld_out + out_off + slice * W;
        uint4 qraw = make_uint4(0u, 0u, 0u, 0u);
        float vw = 0.f, dw[2] = {0.f, 0.f};
        if (live) {
            qraw = __ldg(reinterpret_cast<const uint4*>(QRY + row * ld_q + slice * W) + li);
            vw = __ldg(g.vdeg_w + v);
            dw[0] = __ldg(g.deg_w + 2 * v); dw[1] = __ldg(g.deg_w + 2 * v + 1);
        }
        Acc8 s4[2];
#pragma unroll
        for (int sgn = 0; sgn < 2; ++sgn) {
            Acc8 ms;
            acc8_zero(s4[sgn]); acc8_zero(ms);
            const int code = 2 * v + sgn;
            int e0 = 0, e1 = 0;
            if (live) {
                if constexpr (SI) { e0 = s_idx[code]; e1 = s_idx[code + 1]; }
                else { e0 = __ldg(g.lit_rowptr + code); e1 = __ldg(g.lit_rowptr + code + 1); }
            }
            auto col = [&](int e) { return SI ? (int)s_idx[g.lit_col_off + e] : __ldg(g.lit_clause + e); };
            int e = e0;
            for (; e + 3 <= e1; e += 3) {      // three entries = six table reads in flight
                const int j0 = col(e), j1 = col(e + 1), j2 = col(e + 2);
                DSAT_CHECK((unsigned)j0 < (unsigned)g.m && (unsigned)j1 < (unsigned)g.m && (unsigned)j2 < (unsigned)g.m && e + 3 <= g.nnz);
                const uint4 a0 = reinterpret_cast<const uint4*>(t_cl + (size_t)j0 * W)[li];
                const uint4 b0 = reinterpret_cast<const uint4*>(t_ms + (size_t)j0 * W)[li];
                const uint4 a1 = reinterpret_cast<const uint4*>(t_cl + (size_t)j1 * W)[li];
                const uint4 b1 = reinterpret_cast<const uint4*>(t_ms + (size_t)j1 * W)[li];
                const uint4 a2 = reinterpret_cast<const uint4*>(t_cl + (size_t)j2 * W)[li];
                const uint4 b2 = reinterpret_cast<const uint4*>(t_ms + (size_t)j2 * W)[li];
                acc8_add(s4[sgn], a0); acc8_add(ms, b0);
                acc8_add(s4[sgn], a1); acc8_add(ms, b1);
                acc8_add(s4[sgn], a2); acc8_add(ms, b2);
            }
            for (; e < e1; ++e) {
                const int j = col(e);
                acc8_add(s4[sgn], reinterpret_cast<const uint4*>(t_cl + (size_t)j * W)[li]);
                acc8_add(ms, reinterpret_cast<const uint4*>(t_ms + (size_t)j * W)[li]);
            }
            if (live) {                        // this polarity's message sum leaves right away (fewer live accumulators)
                float lo[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) lo[i] = ms.v[i] * dw[sgn];
                reinterpret_cast<uint4*>(dst + (1 + sgn) * Q)[li] = pack8(lo);
            }
        }
        if (live) {
            float q[8], grad[8];
            unpack8(qraw, q);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float sg = 1.0f / (1.0f + __expf(-q[i]));
                grad[i] = (-sg * s4[0].v[i] + (1.0f - sg) * s4[1].v[i]) * vw;
            }
            reinterpret_cast<uint4*>(dst)[li] = pack8(grad);
        }
    }
}

// ------------------------------------------------------------------ fp32 tables (fp32-accurate tensor-core path)
// The same shared-memory design with fp32 tables: the gathered operands of that path are the fp32 outputs of the x3 MLP
// kernels (LIT, softplus pair, clause messages) and the 4*clauses_loss columns of the clause rows' hi/lo planes; the
// outputs go straight into the hi/lo planes the next MLP reads as its A operand.  A lane owns 4 features (16 bytes);
// sums run in edge order from zero, so they are bit-identical to clause_gather_kernel / literal_gather_kernel.
struct Acc4 { float v[4]; };
__device__ __forceinline__ void acc4_add(Acc4& a, const float4& w) { a.v[0] += w.x; a.v[1] += w.y; a.v[2] += w.z; a.v[3] += w.w; }
__device__ __forceinline__ void store_split4(__nv_bfloat16* dst_hi, size_t plane, int li, const float (&f)[4]) {
    uint2 hi, lo;
    split_bf16x2(f[0], f[1], hi.x, lo.x);
    split_bf16x2(f[2], f[3], hi.y, lo.y);
    reinterpret_cast<uint2*>(dst_hi)[li] = hi;
    reinterpret_cast<uint2*>(dst_hi + plane)[li] = lo;
}

// Role 0 of the literal side with the hi / lo planes of 4*clauses_loss kept as TWO bf16 tables (the same bytes as one fp32
// table): both are staged with cp.async -- converting to fp32 while staging went through registers in two dependent batches
// and left the role-0 CTAs latency-bound -- and every edge adds hi and lo with the one-instruction widening add (acc += hi;
// acc += lo).  A lane owns 8 features.
template <int W, bool SI>
__device__ __forceinline__ void literal_grad_from_planes(const UnitGraphDev& g, int Q, const __nv_bfloat16* __restrict__ CL4_HI,
                                                         size_t cl_plane, int ld_cl, int cl_off, const float* __restrict__ QRY, int ld_q,
                                                         __nv_bfloat16* __restrict__ OUT_HI, size_t out_plane, int ld_out, int out_off,
                                                         uint8_t* gsm, int chain, int slice) {
    using T = __nv_bfloat16;
    constexpr int LPR = W / 8, RPW = 32 / LPR;
    T* t_hi = reinterpret_cast<T*>(gsm);
    T* t_lo = t_hi + (size_t)g.m * W;
    const unsigned short* s_idx = reinterpret_cast<const unsigned short*>(t_lo + (size_t)g.m * W);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const int sub = lane / LPR, li = lane % LPR;
    const size_t cbase = (size_t)chain * g.m;
    const T* src = CL4_HI + cbase * ld_cl + cl_off + slice * W;
    stage_rows_async<T>(t_hi, src, g.m, ld_cl, W, tid, blockDim.x);
    stage_rows_async<T>(t_lo, src + cl_plane, g.m, ld_cl, W, tid, blockDim.x);
    if constexpr (SI) {
        uint4* d = reinterpret_cast<uint4*>(const_cast<unsigned short*>(s_idx));
        for (int i = tid; i < g.lit_idx16_vecs; i += blockDim.x) d[i] = __ldg(reinterpret_cast<const uint4*>(g.lit_idx16) + i);
    }
    cp_async_wait_all();
    __syncthreads();
    for (int v0 = warp * RPW; v0 < g.n; v0 += nwarps * RPW) {
        const bool live = v0 + sub < g.n;
        int v = 0;
        if (live) v = SI ? (int)s_idx[g.lit_ord_off + v0 + sub] : __ldg(g.var_order + v0 + sub);
        const size_t row = (size_t)chain * g.n + v;
        float4 q0 = make_float4(0.f, 0.f, 0.f, 0.f), q1 = q0;
        float vw = 0.f;
        if (live) {
            const float4* qp = reinterpret_cast<const float4*>(QRY + row * ld_q + slice * W) + 2 * li;
            q0 = __ldg(qp); q1 = __ldg(qp + 1);
            vw = __ldg(g.vdeg_w + v);
        }
        Acc8 s4[2];
#pragma unroll
        for (int sgn = 0; sgn < 2; ++sgn) {
            acc8_zero(s4[sgn]);
            const int code = 2 * v + sgn;
            int e0 = 0, e1 = 0;
            if (live) {
                if constexpr (SI) { e0 = s_idx[code]; e1 = s_idx[code + 1]; }
                else { e0 = __ldg(g.lit_rowptr + code); e1 = __ldg(g.lit_rowptr + code + 1); }
            }
            auto col = [&](int e) { return SI ? (int)s_idx[g.lit_col_off + e] : __ldg(g.lit_clause + e); };
            int e = e0;
            for (; e + 3 <= e1; e += 3) {
                const int j0 = col(e), j1 = col(e + 1), j2 = col(e + 2);
                DSAT_CHECK((unsigned)j0 < (unsigned)g.m && (unsigned)j1 < (unsigned)g.m && (unsigned)j2 < (unsigned)g.m);
                const uint4 a0 = reinterpret_cast<const uint4*>(t_hi + (size_t)j0 * W)[li];
                const uint4 b0 = reinterpret_cast<const uint4*>(t_lo + (size_t)j0 * W)[li];
                const uint4 a1 = reinterpret_cast<const uint4*>(t_hi + (size_t)j1 * W)[li];
                const uint4 b1 = reinterpret_cast<const uint4*>(t_lo + (size_t)j1 * W)[li];
                const uint4 a2 = reinterpret_cast<const uint4*>(t_hi + (size_t)j2 * W)[li];
                const uint4 b2 = reinterpret_cast<const uint4*>(t_lo + (size_t)j2 * W)[li];
                acc8_add(s4[sgn], a0); acc8_add(s4[sgn], b0);
                acc8_add(s4[sgn], a1); acc8_add(s4[sgn], b1);
                acc8_add(s4[sgn], a2); acc8_add(s4[sgn], b2);
            }
            for (; e < e1; ++e) {
                const int j = col(e);
                acc8_add(s4[sgn], reinterpret_cast<const uint4*>(t_hi + (size_t)j * W)[li]);
                acc8_add(s4[sgn], reinterpret_cast<const uint4*>(t_lo + (size_t)j * W)[li]);
            }
        }
        if (!live) continue;
        const float qv[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
        float grad[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float sg = sigmoid_f(qv[i]), sgn_ = sigmoid_f(-qv[i]);
            grad[i] = (-sg * s4[0].v[i] + sgn_ * s4[1].v[i]) * vw;
        }
        __nv_bfloat16* dst = OUT_HI + row * ld_out + out_off + slice * W;
        uint4 hi, lo;
        split_bf16x2(grad[0], grad[1], hi.x, lo.x); split_bf16x2(grad[2], grad[3], hi.y, lo.y);
        split_bf16x2(grad[4], grad[5], hi.z, lo.z); split_bf16x2(grad[6], grad[7], hi.w, lo.w);
        reinterpret_cast<uint4*>(dst)[li] = hi;
        reinterpret_cast<uint4*>(dst + out_plane)[li] = lo;
    }
}

// One table per CTA: blockIdx.y = slice * 2 + role.  The two sums of the literal side are independent, so a CTA stages only
// ONE of the two tables and can afford a slice twice as wide: the adjacency walk (index loads, address arithmetic) is
// amortised over twice the features -- these kernels are issue-bound, not bandwidth-bound.
//   role 0: tables 4*clauses_loss (hi / lo) -> variables_grad (literal_grad_from_planes)
//   role 1: table messages -> loss_pos | loss_neg
template <int W, bool SI>
__global__ void __launch_bounds__(512, 2)
literal_gather_smem_f32_kernel(UnitGraphDev g, int Q,
                               const __nv_bfloat16* __restrict__ CL4_HI, size_t cl_plane, int ld_cl, int cl_off,
                               const float* __restrict__ MSG, int ld_msg,
                               const float* __restrict__ QRY, int ld_q,
                               __nv_bfloat16* __restrict__ OUT_HI, size_t out_plane, int ld_out, int out_off, SkipInfo skip = SkipInfo{nullptr, 1}) {
    if (chain_done(skip, (int)blockIdx.x)) return;     // the whole CTA works on one chain
    constexpr int LPR = W / 4, RPW = 32 / LPR;
    extern __shared__ __align__(16) uint8_t gsm[];
    const int chain = blockIdx.x, slice = blockIdx.y >> 1;
    if ((blockIdx.y & 1) == 0) {
        literal_grad_from_planes<W, SI>(g, Q, CL4_HI, cl_plane, ld_cl, cl_off, QRY, ld_q, OUT_HI, out_plane, ld_out, out_off, gsm, chain, slice);
        return;
    }
    float* tab = reinterpret_cast<float*>(gsm);
    const unsigned short* s_idx = reinterpret_cast<const unsigned short*>(tab + (size_t)g.m * W);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const int sub = lane / LPR, li = lane % LPR;
    const size_t cbase = (size_t)chain * g.m;
    stage_rows_async<float>(tab, MSG + cbase * ld_msg + slice * W, g.m, ld_msg, W, tid, blockDim.x);
    if constexpr (SI) {
        uint4* d = reinterpret_cast<uint4*>(const_cast<unsigned short*>(s_idx));
        for (int i = tid; i < g.lit_idx16_vecs; i += blockDim.x) d[i] = __ldg(reinterpret_cast<const uint4*>(g.lit_idx16) + i);
    }
    cp_async_wait_all();
    __syncthreads();
    for (int v0 = warp * RPW; v0 < g.n; v0 += nwarps * RPW) {
        const bool live = v0 + sub < g.n;
        int v = 0;
        if (live) v = SI ? (int)s_idx[g.lit_ord_off + v0 + sub] : __ldg(g.var_order + v0 + sub);
        const size_t row = (size_t)chain * g.n + v;
        __nv_bfloat16* dst = OUT_HI + row * ld_out + out_off + slice * W;
        float dw[2] = {0.f, 0.f};
        if (live) { dw[0] = __ldg(g.deg_w + 2 * v); dw[1] = __ldg(g.deg_w + 2 * v + 1); }
        Acc4 sum[2];
#pragma unroll
        for (int sgn = 0; sgn < 2; ++sgn) {
            Acc4 acc = {{0.f, 0.f, 0.f, 0.f}};
            const int code = 2 * v + sgn;
            int e0 = 0, e1 = 0;
            if (live) {
                if constexpr (SI) { e0 = s_idx[code]; e1 = s_idx[code + 1]; }
                else { e0 = __ldg(g.lit_rowptr + code); e1 = __ldg(g.lit_rowptr + code + 1); }
            }
            auto col = [&](int e) { return SI ? (int)s_idx[g.lit_col_off + e] : __ldg(g.lit_clause + e); };
            int e = e0;
            for (; e + 4 <= e1; e += 4) {
                const int j0 = col(e), j1 = col(e + 1), j2 = col(e + 2), j3 = col(e + 3);
                DSAT_CHECK((unsigned)j0 < (unsigned)g.m && (unsigned)j1 < (unsigned)g.m && (unsigned)j2 < (unsigned)g.m &&
                           (unsigned)j3 < (unsigned)g.m && e + 4 <= g.nnz);
                const float4 a0 = reinterpret_cast<const float4*>(tab + (size_t)j0 * W)[li];
                const float4 a1 = reinterpret_cast<const float4*>(tab + (size_t)j1 * W)[li];
                const float4 a2 = reinterpret_cast<const float4*>(tab + (size_t)j2 * W)[li];
                const float4 a3 = reinterpret_cast<const float4*>(tab + (size_t)j3 * W)[li];
                acc4_add(acc, a0); acc4_add(acc, a1); acc4_add(acc, a2); acc4_add(acc, a3);
            }
            for (; e < e1; ++e) acc4_add(acc, reinterpret_cast<const float4*>(tab + (size_t)col(e) * W)[li]);
            sum[sgn] = acc;
        }
        if (!live) continue;
#pragma unroll
        for (int sgn = 0; sgn < 2; ++sgn) {
            float o[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) o[i] = sum[sgn].v[i] * dw[sgn];
            store_split4(dst + (1 + sgn) * Q, out_plane, li, o);
        }
    }
}

// clause side, both tables in one CTA (slice W): measured faster than one table per CTA at cfg2 (0.52 vs 0.61 ms per round):
// with a row per warp pass the single-table walk is latency-bound on its index -> table-row chain
template <int W, bool SI>
__global__ void __launch_bounds__(512, 3)
clause_gather_smem_f32x2_kernel(UnitGraphDev g, int Q,
                                const float* __restrict__ LIT, int ld_lit,
                                const float* __restrict__ SP, int ld_sp, int sp_off,
                                __nv_bfloat16* __restrict__ OUT_HI, size_t out_plane, int ld_out, int out_off, SkipInfo skip = SkipInfo{nullptr, 1}) {
    if (chain_done(skip, (int)blockIdx.x)) return;     // the whole CTA works on one chain
    constexpr int LPR = W / 4, RPW = 32 / LPR;
    extern __shared__ __align__(16) uint8_t gsm[];
    float* t_lit = reinterpret_cast<float*>(gsm);
    float* t_sp = t_lit + (size_t)2 * g.n * W;
    const unsigned short* s_idx = reinterpret_cast<const unsigned short*>(t_sp + (size_t)2 * g.n * W);
    const int chain = blockIdx.x, slice = blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const int sub = lane / LPR, li = lane % LPR;
    const size_t vbase = (size_t)chain * g.n;
    {
        const int total = 2 * g.n * LPR;                    // (variable, sign, 16-byte piece)
        for (int i = tid; i < total; i += blockDim.x) {
            const int code = i / LPR, k = i % LPR, v = code >> 1, sgn = code & 1;
            cp_async16(reinterpret_cast<uint4*>(t_lit + (size_t)code * W) + k,
                       reinterpret_cast<const uint4*>(LIT + (vbase + v) * ld_lit + sgn * Q + slice * W) + k);
            cp_async16(reinterpret_cast<uint4*>(t_sp + (size_t)code * W) + k,
                       reinterpret_cast<const uint4*>(SP + (vbase + v) * ld_sp + sp_off + sgn * Q + slice * W) + k);
        }
    }
    if constexpr (SI) {
        uint4* d = reinterpret_cast<uint4*>(const_cast<unsigned short*>(s_idx));
        for (int i = tid; i < g.cl_idx16_vecs; i += blockDim.x) d[i] = __ldg(reinterpret_cast<const uint4*>(g.cl_idx16) + i);
    }
    cp_async_wait_all();
    __syncthreads();
    for (int j0 = warp * RPW; j0 < g.m; j0 += nwarps * RPW) {
        const int j = j0 + sub;
        const bool live = j < g.m;
        int e0 = 0, e1 = 0;
        if (live) {
            if constexpr (SI) { e0 = s_idx[j]; e1 = s_idx[j + 1]; }
            else { e0 = __ldg(g.cl_rowptr + j); e1 = __ldg(g.cl_rowptr + j + 1); }
        }
        Acc4 al = {{0.f, 0.f, 0.f, 0.f}}, as = {{0.f, 0.f, 0.f, 0.f}};
        int e = e0;
        for (; e + 3 <= e1; e += 3) {
            const int c0 = SI ? (int)s_idx[g.cl_col_off + e] : __ldg(g.cl_lit + e);
            const int c1 = SI ? (int)s_idx[g.cl_col_off + e + 1] : __ldg(g.cl_lit + e + 1);
            const int c2 = SI ? (int)s_idx[g.cl_col_off + e + 2] : __ldg(g.cl_lit + e + 2);
            DSAT_CHECK((unsigned)c0 < 2u * g.n && (unsigned)c1 < 2u * g.n && (unsigned)c2 < 2u * g.n && e + 3 <= g.nnz);
            const float4 l0 = reinterpret_cast<const float4*>(t_lit + (size_t)c0 * W)[li];
            const float4 p0 = reinterpret_cast<const float4*>(t_sp + (size_t)c0 * W)[li];
            const float4 l1 = reinterpret_cast<const float4*>(t_lit + (size_t)c1 * W)[li];
            const float4 p1 = reinterpret_cast<const float4*>(t_sp + (size_t)c1 * W)[li];
            const float4 l2 = reinterpret_cast<const float4*>(t_lit + (size_t)c2 * W)[li];
            const float4 p2 = reinterpret_cast<const float4*>(t_sp + (size_t)c2 * W)[li];
            acc4_add(al, l0); acc4_add(as, p0);
            acc4_add(al, l1); acc4_add(as, p1);
            acc4_add(al, l2); acc4_add(as, p2);
        }
        for (; e < e1; ++e) {
            const int code = SI ? (int)s_idx[g.cl_col_off + e] : __ldg(g.cl_lit + e);
            acc4_add(al, reinterpret_cast<const float4*>(t_lit + (size_t)code * W)[li]);
            acc4_add(as, reinterpret_cast<const float4*>(t_sp + (size_t)code * W)[li]);
        }
        if (live) {
            const float rw = __ldg(g.rev_w + j);
            float ol[4], os[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) { ol[i] = al.v[i] * rw; os[i] = 4.0f * expf(-as.v[i]); }
            __nv_bfloat16* dst = OUT_HI + ((size_t)chain * g.m + j) * ld_out + out_off + slice * W;
            store_split4(dst, out_plane, li, ol);
            store_split4(dst + Q, out_plane, li, os);
        }
    }
}

}  // namespace dsat
