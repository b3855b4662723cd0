// libdsat.so: context, buffers, launch orchestration and the C ABI of include/dsat.h.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/dsat.h"
#include "../../include/dsat_debug.h"
#include "dsat_common.cuh"
#include "dsat_gemm_simt.cuh"
#include "dsat_message.cuh"
#include "dsat_spmm.cuh"
#include "dsat_graph_host.cuh"
#include "dsat_norm_head.cuh"
#include "dsat_hist.cuh"
#include "dsat_gemm_tc.cuh"
#include "dsat_mlp_fused.cuh"
#include "dsat_mlp_x3.cuh"

using namespace dsat;

// Synchronous copy that is also ordered against the context's NON-BLOCKING stream: a pageable
// host-to-device cudaMemcpy may return while its DMA is still in flight, and work queued afterwards on a
// non-blocking stream is not ordered behind it.
static cudaError_t dsat_memcpy_sync(void* dst, const void* src, size_t bytes, cudaMemcpyKind kind) {
    cudaError_t e = cudaMemcpy(dst, src, bytes, kind);
    if (e == cudaSuccess && kind == cudaMemcpyHostToDevice) e = cudaDeviceSynchronize();
    return e;
}

namespace {

template <typename T>
struct DevBuf {
    T* p = nullptr;
    size_t count = 0;       // elements in use
    size_t cap = 0;         // elements allocated
    // (Re)size.  An allocation that is large enough is kept: cudaFree / cudaMalloc of multi-gigabyte buffers cost ~0.1 s per
    // re-bound graph once the context had seen a few shapes (mixed-formula batches change shape with every batch).
    cudaError_t alloc(size_t n) {
        if (p && n <= cap) { count = n; return cudaSuccess; }
        release();
        if (n == 0) return cudaSuccess;
        cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&p), n * sizeof(T));
        if (e == cudaSuccess) { count = n; cap = n; }
        else p = nullptr;
        return e;
    }
    void drop() { count = 0; }      // contents invalid, memory kept for the next alloc
    void release() {
        if (p) cudaFree(p);
        p = nullptr; count = 0; cap = 0;
    }
    cudaError_t upload(const T* host, size_t n, cudaStream_t s) {
        return cudaMemcpyAsync(p, host, n * sizeof(T), cudaMemcpyHostToDevice, s);
    }
};

struct PackedLayer {          // one launched linear op
    DevBuf<float> w, b;
    DevBuf<__nv_bfloat16> w_bf16;   // [N, K] K-major copy for the tensor-core path
    int K = 0, N = 0;
};

enum OpId { OP_V1 = 0, OP_Q2, OP_L2, OP_L3, OP_C1, OP_C2, OP_U1, OP_U2, OP_U3, OP_O1, OP_O2, OP_COUNT };

}  // namespace

constexpr int SPMM_DW_CLAUSE = 2;        // int4 per clause-side row descriptor: four entries cover every clause of k<=4-SAT
struct dsat_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::string err;
    long long launches = 0;
    int precision = DSAT_F32_TC;        // default: fp32-accurate Dense layers on the tensor cores
    // per-class CUDA-event marks (dsat_profile_rounds)
    struct ProfMark { cudaEvent_t ev; int cls; };
    std::vector<ProfMark> prof;
    size_t prof_used = 0;
    bool profiling = false;

    // model
    bool has_model = false;
    int F = 0, Q = 0, HQ = 0, HL = 0, HC = 0, HU = 0, HO = 0;
    PackedLayer ops[OP_COUNT];

    // graph
    bool has_graph = false;
    int n = 0, m = 0, nnz = 0, n_graphs = 0, chains = 0, group_graphs = 0, n_groups = 0, total_graphs = 0;
    int words = 0;
    int max_graph_vars = 0, max_graph_clauses = 0;      // largest formula of the unit (shared-memory PairNorm)
    // variable early-exit groups and per-graph noise bases (dsat_set_batches); cleared by dsat_set_graph
    bool has_batches = false, has_noise_base = false;
    DevBuf<int> batch_seg, graph_group;  // [n_groups+1] group bounds, [total_graphs] group of each graph
    DevBuf<int> row_graph;               // [Nt] graph of each variable row
    DevBuf<unsigned long long> graph_elem0;   // [total_graphs] noise base of the graph minus its first row (mod 2^64)
    long long Nt = 0, Mt = 0;
    DevBuf<int> cl_rowptr, cl_lit, lit_rowptr, lit_clause, var_seg, clause_seg;
    DevBuf<float> deg_w, vdeg_w, rev_w;
    DevBuf<int> var_order;               // variables by descending degree (literal-side gather)
    DevBuf<unsigned short> cl_idx16, lit_idx16;   // 16-bit adjacency blocks for the shared-memory gathers (dsat_message.cuh)
    int cl_idx16_vecs = 0, lit_idx16_vecs = 0, cl_col_off = 0, lit_col_off = 0, lit_ord_off = 0;
    DevBuf<int> cl_desc, lit_desc, lit_desc4;   // standalone segment sums: row descriptors in processing order (dsat_spmm.cuh);
                                                // the literal side keeps a 2-int4 and a 4-int4 form (chosen per shape)
    std::vector<int32_t> h_cl_rowptr, h_cl_lit, h_lit_rowptr, h_lit_clause;     // host copy of the bound graph (ensure_spmm_desc)
    std::vector<float> h_deg_w, h_rev_w;
    bool spmm_desc_ready = false;

    // activations
    bool has_buffers = false;
    DevBuf<float> VROW, CROW, H1, H2, QS, LIT, CH, COUT, U1, U2, UOUT, SPRE, O1, LOGITS, OUT;
    DevBuf<float2> X;
    DevBuf<int> labels, done, steps_taken, rounds_run, graph_sat, graph_map, latch_step, sat_now;
    DevBuf<float> loss_sum, graph_loss;
    DevBuf<unsigned char> BITS, LAST, LATCH, FINAL, is_sat, sat_any;
    DevBuf<unsigned long long> packed;
    // histogram reduction scratch (dsat_hist.cuh)
    DevBuf<int> hist_idx, hist_run, hist_totals, hist_seg, hist_run_seg;
    DevBuf<unsigned long long> hist_keys, hist_counts;
    // injected noise staging
    DevBuf<float> inj_normals, inj_uniforms, inj_noisy;
    DevBuf<int> inj_labels;
    // bf16 activations of the tensor-core path (A operands are fetched by TMA from these)
    DevBuf<__nv_bfloat16> VROWb, CROWb, H1b, H2b, QSb, LITb, CHb, COUTb, U1b, U2b, UOUTb, SPREb, O1b;
    CUtensorMap map_a[OP_COUNT];        // A operand of each linear op
    CUtensorMap map_b[OP_COUNT];        // transposed bf16 weights
    int a_box_rows[OP_COUNT] = {0}, b_box_rows[OP_COUNT] = {0};
    bool has_tc_buffers = false;
    // whole-MLP kernels (dsat_mlp_fused.cuh): query, literal, clause, update, output
    fm::FusedMlp fused[5];
    bool fused_ready = false;
    // fp32-accurate tensor-core path (dsat_mlp_x3.cuh): MLP inputs live as hi/lo bf16 planes [2][rows][ld]
    DevBuf<__nv_bfloat16> VROWp, CROWp, SPREp, H1p, H2p;
    DevBuf<__nv_bfloat16> wx[12];       // stacked hi/lo K-major weights [2N, K64] per reference layer
    int wx_k64[12] = {0}, wx_n[12] = {0};
    x3::X3Mlp x3[7];                    // query, lit layer 1, lit layer 2, lit layer 3, clause, update, output
    bool has_x3_buffers = false;
    bool x3_ready = false;
    bool has_simt_buffers = false;
    float last_noise_scale = 0.f;
    int sampling = DSAT_SAMPLE_INVERSE_CDF;
    // one captured denoising step (dsat_sample_enqueue without injected noise): replayed once per step, the step's scalars
    // come from step_tab[*step_cur] on the device
    DevBuf<StepParams> step_tab;
    DevBuf<int> step_cur;
    std::vector<StepParams> step_tab_host;
    cudaGraphExec_t step_graph = nullptr;
    long long generation = 0, step_graph_generation = -1;   // bumped whenever a pointer or plan baked into the graph changes
    int step_graph_rounds = -1, step_graph_precision = -1, step_launches = 0;

    int ldv() const { return F + DSAT_AUX_PAD + 3 * Q; }
    int ldc() const { return F + 2 * Q; }
    int ldh1() const { return HQ + HL; }
};

#ifdef DSAT_ASSERT
static int* g_assert_host = nullptr;     // host view of g_dsat_assert_slot (mapped memory: readable after a trap)
static std::string assert_note() {
    return g_assert_host && g_assert_host[0] ? " [DSAT_ASSERT failed at line " + std::to_string(g_assert_host[0]) + " of a kernel header]" : "";
}
#else
static std::string assert_note() { return ""; }
#endif

#define CK_CUDA(ctx, expr)                                                              \
    do {                                                                                \
        cudaError_t e__ = (expr);                                                       \
        if (e__ != cudaSuccess) {                                                       \
            (ctx)->err = std::string(#expr) + ": " + cudaGetErrorString(e__) + assert_note(); \
            return DSAT_ERR_CUDA;                                                       \
        }                                                                               \
    } while (0)

#define CK_ARG(ctx, cond, msg)                                                          \
    do {                                                                                \
        if (!(cond)) { (ctx)->err = (msg); return DSAT_ERR_ARG; }                       \
    } while (0)

#define LAUNCHED(ctx)                                                                   \
    do {                                                                                \
        (ctx)->launches++;                                                              \
        CK_CUDA(ctx, cudaGetLastError());                                               \
    } while (0)

namespace {

// Opt every kernel that uses more than 48 KB of dynamic shared memory in, once per device (the attribute is per device),
// at context creation: nothing on the launch path calls cudaFuncSetAttribute, so launches can be captured into a graph.
cudaError_t configure_kernels_for_device() {
    static PerDeviceOnce configured;
    if (configured.done()) return cudaSuccess;
    cudaError_t e = cudaSuccess;
    auto opt_in = [&](auto kernel) {
        if (e == cudaSuccess) e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    };
    opt_in(clause_gather_smem_kernel<128, true>); opt_in(clause_gather_smem_kernel<128, false>);
    opt_in(clause_gather_smem_kernel<64, true>); opt_in(clause_gather_smem_kernel<64, false>);
    opt_in(clause_gather_smem_kernel<32, true>); opt_in(clause_gather_smem_kernel<32, false>);
    opt_in(literal_gather_smem_kernel<128, true>); opt_in(literal_gather_smem_kernel<128, false>);
    opt_in(literal_gather_smem_kernel<64, true>); opt_in(literal_gather_smem_kernel<64, false>);
    opt_in(literal_gather_smem_kernel<32, true>); opt_in(literal_gather_smem_kernel<32, false>);
    opt_in(clause_gather_smem_f32x2_kernel<128, true>); opt_in(clause_gather_smem_f32x2_kernel<128, false>);
    opt_in(clause_gather_smem_f32x2_kernel<64, true>); opt_in(clause_gather_smem_f32x2_kernel<64, false>);
    opt_in(clause_gather_smem_f32x2_kernel<32, true>); opt_in(clause_gather_smem_f32x2_kernel<32, false>);
    opt_in(literal_gather_smem_f32_kernel<128, true>); opt_in(literal_gather_smem_f32_kernel<128, false>);
    opt_in(literal_gather_smem_f32_kernel<64, true>); opt_in(literal_gather_smem_f32_kernel<64, false>);
    opt_in(literal_gather_smem_f32_kernel<32, true>); opt_in(literal_gather_smem_f32_kernel<32, false>);
    opt_in(pairnorm_smem_kernel<2>); opt_in(pairnorm_smem_kernel<4>); opt_in(pairnorm_smem_kernel<8>);
    if (e == cudaSuccess) e = fm::configure_fused_device();
    if (e == cudaSuccess) e = x3::configure_x3_device(0);
    if (e == cudaSuccess) e = tc::configure_tc_device();
    if (e == cudaSuccess) configured.mark();
    return e;
}

UnitGraphDev graph_view(const dsat_ctx* c) {
    UnitGraphDev g;
    g.n = c->n; g.m = c->m; g.nnz = c->nnz; g.n_graphs = c->n_graphs;
    g.cl_rowptr = c->cl_rowptr.p; g.cl_lit = c->cl_lit.p;
    g.lit_rowptr = c->lit_rowptr.p; g.lit_clause = c->lit_clause.p;
    g.var_seg = c->var_seg.p; g.clause_seg = c->clause_seg.p;
    g.deg_w = c->deg_w.p; g.vdeg_w = c->vdeg_w.p; g.rev_w = c->rev_w.p;
    g.var_order = c->var_order.p;
    g.cl_idx16 = c->cl_idx16_vecs ? c->cl_idx16.p : nullptr;
    g.lit_idx16 = c->lit_idx16_vecs ? c->lit_idx16.p : nullptr;
    g.cl_idx16_vecs = c->cl_idx16_vecs; g.lit_idx16_vecs = c->lit_idx16_vecs;
    g.cl_col_off = c->cl_col_off; g.lit_col_off = c->lit_col_off; g.lit_ord_off = c->lit_ord_off;
    return g;
}

// rows of finished early-exit groups are skipped when the groups consist of whole chains.
// Variable groups (dsat_set_batches) are not runs of whole chains: nothing is skipped, which changes no result.
SkipInfo skip_info(const dsat_ctx* c) {
    if (c->has_batches || c->n_graphs <= 0 || c->group_graphs % c->n_graphs != 0) return SkipInfo{nullptr, 1};
    return SkipInfo{c->done.p, c->group_graphs / c->n_graphs};
}

// Philox element of local row 0 = chain_offset * n, or the per-graph bases bound by dsat_set_batches
NoiseSource noise_source(const dsat_ctx* c, uint64_t seed, uint64_t element_offset, unsigned step) {
    NoiseSource ns{seed, element_offset, step};
    if (c->has_noise_base) { ns.row_graph = c->row_graph.p; ns.graph_elem0 = c->graph_elem0.p; }
    return ns;
}

// buffers every precision uses: the fp32 outputs of the MLPs, the diffusion state and the per-graph bookkeeping
int ensure_common_buffers(dsat_ctx* c) {
    if (c->has_buffers) return DSAT_OK;
    if (!c->has_model || !c->has_graph) { c->err = "set the model and the graph first"; return DSAT_ERR_STATE; }
    const size_t Nt = (size_t)c->Nt, Mt = (size_t)c->Mt;
    CK_CUDA(c, c->QS.alloc(Nt * 3 * c->Q));
    CK_CUDA(c, c->LIT.alloc(Nt * 2 * c->Q));
    CK_CUDA(c, c->COUT.alloc(Mt * (c->Q + c->F)));
    CK_CUDA(c, c->UOUT.alloc(Nt * c->F));
    CK_CUDA(c, c->LOGITS.alloc(Nt * DSAT_LOGIT_PAD));
    CK_CUDA(c, c->OUT.alloc(Nt));
    CK_CUDA(c, c->X.alloc(Nt + 1));
    CK_CUDA(c, c->labels.alloc(Nt));
    CK_CUDA(c, c->BITS.alloc(Nt));
    CK_CUDA(c, c->LAST.alloc(Nt));
    CK_CUDA(c, c->LATCH.alloc(Nt));
    CK_CUDA(c, c->FINAL.alloc(Nt));
    const size_t G = (size_t)c->total_graphs, NG = (size_t)c->n_groups;
    CK_CUDA(c, c->done.alloc(NG));
    CK_CUDA(c, c->steps_taken.alloc(NG));
    CK_CUDA(c, c->rounds_run.alloc(NG));
    CK_CUDA(c, c->loss_sum.alloc(NG));
    CK_CUDA(c, c->graph_sat.alloc(G));
    CK_CUDA(c, c->graph_map.alloc(G));
    CK_CUDA(c, c->graph_loss.alloc(G));
    CK_CUDA(c, c->latch_step.alloc(G));
    CK_CUDA(c, c->sat_now.alloc(G));
    CK_CUDA(c, c->is_sat.alloc(G));
    CK_CUDA(c, c->sat_any.alloc(G));
    CK_CUDA(c, c->packed.alloc(G * c->words));
    CK_CUDA(c, cudaMemsetAsync(c->OUT.p, 0, c->OUT.count * sizeof(float), c->stream));
    c->has_buffers = true;
    return DSAT_OK;
}

// + the fp32 row buffers and hidden activations of the CUDA-core path
int ensure_buffers(dsat_ctx* c) {
    int rc = ensure_common_buffers(c);
    if (rc) return rc;
    if (c->has_simt_buffers) return DSAT_OK;
    const size_t Nt = (size_t)c->Nt, Mt = (size_t)c->Mt;
    CK_CUDA(c, c->VROW.alloc(Nt * c->ldv()));
    CK_CUDA(c, c->CROW.alloc(Mt * c->ldc()));
    CK_CUDA(c, c->H1.alloc(Nt * c->ldh1()));
    CK_CUDA(c, c->H2.alloc(Nt * c->HL));
    CK_CUDA(c, c->CH.alloc(Mt * c->HC));
    CK_CUDA(c, c->U1.alloc(Nt * c->HU));
    CK_CUDA(c, c->U2.alloc(Nt * c->HU));
    CK_CUDA(c, c->SPRE.alloc(Nt * c->F));
    CK_CUDA(c, c->O1.alloc(Nt * c->HO));
    // padded columns must be zero forever: clear everything once
    CK_CUDA(c, cudaMemsetAsync(c->VROW.p, 0, c->VROW.count * sizeof(float), c->stream));
    CK_CUDA(c, cudaMemsetAsync(c->CROW.p, 0, c->CROW.count * sizeof(float), c->stream));
    c->has_simt_buffers = true;
    return DSAT_OK;
}

static int pick_slice_width(size_t table_rows, int Q, size_t* bytes_out, int budget_kb, int elt_bytes = 2);

// bf16 activation buffers + the TMA descriptors of every A operand (they depend on the row counts)
int ensure_tc_buffers(dsat_ctx* c) {
    if (c->has_tc_buffers) return DSAT_OK;
    int rc = ensure_common_buffers(c);
    if (rc) return rc;
    const size_t Nt = (size_t)c->Nt, Mt = (size_t)c->Mt;
    const int F = c->F, Q = c->Q;
    CK_CUDA(c, c->VROWb.alloc(Nt * c->ldv()));
    CK_CUDA(c, c->CROWb.alloc(Mt * c->ldc()));
    CK_CUDA(c, c->H1b.alloc(Nt * c->ldh1()));
    CK_CUDA(c, c->H2b.alloc(Nt * c->HL));
    CK_CUDA(c, c->QSb.alloc(Nt * 3 * Q));
    CK_CUDA(c, c->LITb.alloc(Nt * 2 * Q));
    CK_CUDA(c, c->CHb.alloc(Mt * c->HC));
    CK_CUDA(c, c->COUTb.alloc(Mt * (Q + F)));
    CK_CUDA(c, c->UOUTb.alloc(Nt * F));
    CK_CUDA(c, c->U1b.alloc(Nt * c->HU));
    CK_CUDA(c, c->U2b.alloc(Nt * c->HU));
    CK_CUDA(c, c->SPREb.alloc(Nt * F));
    CK_CUDA(c, c->O1b.alloc(Nt * c->HO));
    CK_CUDA(c, cudaMemsetAsync(c->VROWb.p, 0, c->VROWb.count * 2, c->stream));
    CK_CUDA(c, cudaMemsetAsync(c->CROWb.p, 0, c->CROWb.count * 2, c->stream));
    struct Src { const void* p; long long rows; int k; int ld; };
    const Src srcs[OP_COUNT] = {
        {c->VROWb.p, c->Nt, F + DSAT_AUX_PAD, c->ldv()},        // OP_V1
        {c->H1b.p, c->Nt, c->HQ, c->ldh1()},                    // OP_Q2
        {c->H1b.p + c->HQ, c->Nt, c->HL, c->ldh1()},            // OP_L2
        {c->H2b.p, c->Nt, c->HL, c->HL},                        // OP_L3
        {c->CROWb.p, c->Mt, F + 2 * Q, c->ldc()},               // OP_C1
        {c->CHb.p, c->Mt, c->HC, c->HC},                        // OP_C2
        {c->VROWb.p, c->Nt, F + DSAT_AUX_PAD + 3 * Q, c->ldv()},// OP_U1
        {c->U1b.p, c->Nt, c->HU, c->HU},                        // OP_U2
        {c->U2b.p, c->Nt, c->HU, c->HU},                        // OP_U3
        {c->SPREb.p, c->Nt, F, F},                              // OP_O1
        {c->O1b.p, c->Nt, c->HO, c->HO},                        // OP_O2
    };
    for (int op = 0; op < OP_COUNT; ++op) {
        if (srcs[op].k != c->ops[op].K) { c->err = "internal: A operand width mismatch"; return DSAT_ERR_STATE; }
        c->a_box_rows[op] = (int)(srcs[op].rows < tc::BLOCK_M ? srcs[op].rows : tc::BLOCK_M);
        if (!tc::make_bf16_map(&c->map_a[op], srcs[op].p, srcs[op].rows, srcs[op].k, srcs[op].ld, c->a_box_rows[op])) {
            c->err = "cuTensorMapEncodeTiled failed for an activation operand";
            return DSAT_ERR_CUDA;
        }
    }
    {   // whole-MLP kernels: one launch per MLP, hidden activations stay in shared memory
        enum { FQ = 0, FL, FC, FU, FO };
        const int k64_v1 = (c->ops[OP_V1].K + 63) / 64 * 64;
        struct L { int op; int n; const __nv_bfloat16* w; const float* b; int epi; };
        auto build = [&](int which, int a_op, std::initializer_list<L> layers, tc::TcOut out) -> bool {
            fm::FusedMlp& f = c->fused[which];
            f.map_a = c->map_a[a_op];
            f.p.n_layers = (int)layers.size();
            f.p.rows = (int)(a_op == OP_C1 ? c->Mt : c->Nt);
            f.p.a_box_rows = c->a_box_rows[a_op];
            f.p.qmaps = Q;
            f.p.prof = nullptr;
            f.p.out = out;
            int i = 0;
            for (const L& l : layers) {
                const int K = c->ops[l.op].K, K64 = (K + 63) / 64 * 64;
                f.p.layer[i].K = K; f.p.layer[i].N = l.n; f.p.layer[i].epi = l.epi; f.p.layer[i].bias = l.b;
                f.p.layer[i].box_rows = l.n < 256 ? l.n : 256;
                if (!tc::make_bf16_map(&f.map_w[i], l.w, l.n, K64, K64, f.p.layer[i].box_rows)) return false;
                if (!tc::make_bf16_map(&f.map_wp[i], l.w, l.n, K64, K64, f.p.layer[i].box_rows / 2)) return false;
                ++i;
            }
            // input ring for all but the literal MLP, which keeps its input resident (split mode where every hidden layer is
            // 512 wide); two tiles in flight wherever they fit
            f.stream_input = which != FL;
            // CTA pair (cta_group::2) for the literal (split mode), clause and update MLPs: measured 4 %, 7 % and 9 % faster there,
            // 2-5 % slower for the small query and output MLPs; the clause pair with two tiles in flight (half-height weight
            // slots: three of them next to three input slots) measured 4 % faster than with one
            f.pair_mode = which == FL || which == FC || which == FU;
            if (!fm::plan_fused(f)) return false;
            if (getenv("DSAT_PLAN_LOG"))
                fprintf(stderr, "[dsat] fused mlp %d: smem %d B (pad %d), hidden blocks %d x%d, input ring %d, weight ring %d x %d B, "
                        "epilogue warps %d, ping-pong %d, staging in hidden %d, cta pair %d, split %d (%d steps)\n", which, f.smem_bytes, f.p.smem_pad, f.p.ah_blocks,
                        f.p.pp ? 2 : 1, f.p.a_slots, f.p.slots, f.p.slot_bytes, f.p.epi_warps, f.p.pp, f.p.stage_in_h, f.p.pair, f.p.split, f.p.n_steps);
            return true;
        };
        auto W = [&](int op) { return (const __nv_bfloat16*)c->ops[op].w_bf16.p; };
        auto B = [&](int op) { return (const float*)c->ops[op].b.p; };
        tc::TcOut o;
        bool ok = true;
        o = {c->QSb.p, 3 * Q, 1, nullptr, 0, 0, 0};
        ok = ok && build(FQ, OP_V1, {{OP_V1, c->HQ, W(OP_V1), B(OP_V1), tc::TC_LRELU},
                                     {OP_Q2, Q, W(OP_Q2), B(OP_Q2), tc::TC_QUERY}}, o);
        o = {c->LITb.p, 2 * Q, 1, nullptr, 0, 0, 0};
        ok = ok && build(FL, OP_V1, {{OP_V1, c->HL, W(OP_V1) + (size_t)c->HQ * k64_v1, B(OP_V1) + c->HQ, tc::TC_LRELU},
                                     {OP_L2, c->HL, W(OP_L2), B(OP_L2), tc::TC_LRELU},
                                     {OP_L3, 2 * Q, W(OP_L3), B(OP_L3), tc::TC_LINEAR}}, o);
        o = {c->COUTb.p, Q + F, 1, nullptr, 0, 0, 0};
        ok = ok && build(FC, OP_C1, {{OP_C1, c->HC, W(OP_C1), B(OP_C1), tc::TC_LRELU},
                                     {OP_C2, Q + F, W(OP_C2), B(OP_C2), tc::TC_LINEAR}}, o);
        o = {c->UOUTb.p, F, 1, nullptr, 0, 0, 0};
        ok = ok && build(FU, OP_U1, {{OP_U1, c->HU, W(OP_U1), B(OP_U1), tc::TC_LRELU},
                                     {OP_U2, c->HU, W(OP_U2), B(OP_U2), tc::TC_LRELU},
                                     {OP_U3, F, W(OP_U3), B(OP_U3), tc::TC_LINEAR}}, o);
        o = {c->LOGITS.p, DSAT_LOGIT_PAD, 0, nullptr, 0, 0, 0};
        ok = ok && build(FO, OP_O1, {{OP_O1, c->HO, W(OP_O1), B(OP_O1), tc::TC_LRELU},
                                     {OP_O2, DSAT_LOGIT_PAD, W(OP_O2), B(OP_O2), tc::TC_LINEAR}}, o);
        c->fused_ready = ok;
    }
    c->has_tc_buffers = true;
    return DSAT_OK;
}

// bf16 transposed ([N, K64], K-major) copies of the packed fp32 weights and their TMA descriptors
int tc_pack_weights(dsat_ctx* c) {
    for (int op = 0; op < OP_COUNT; ++op) {
        const int K = c->ops[op].K, N = c->ops[op].N;
        const int K64 = (K + 63) / 64 * 64;
        std::vector<float> w((size_t)K * N);
        CK_CUDA(c, dsat_memcpy_sync(w.data(), c->ops[op].w.p, w.size() * sizeof(float), cudaMemcpyDeviceToHost));
        std::vector<__nv_bfloat16> wt((size_t)N * K64, __float2bfloat16(0.f));
        for (int k = 0; k < K; ++k)
            for (int n = 0; n < N; ++n) wt[(size_t)n * K64 + k] = __float2bfloat16(w[(size_t)k * N + n]);
        CK_CUDA(c, c->ops[op].w_bf16.alloc(wt.size()));
        CK_CUDA(c, dsat_memcpy_sync(c->ops[op].w_bf16.p, wt.data(), wt.size() * 2, cudaMemcpyHostToDevice));
        c->b_box_rows[op] = N < tc::BLOCK_N ? N : tc::BLOCK_N;
        if (!tc::make_bf16_map(&c->map_b[op], c->ops[op].w_bf16.p, N, K64, K64, c->b_box_rows[op])) {
            c->err = "cuTensorMapEncodeTiled failed for a weight operand (no CUDA driver?)";
            return DSAT_ERR_CUDA;
        }
    }
    return DSAT_OK;
}

// Invalidate every activation buffer (shape or model changed).  The memory stays with the context and is reused by the next
// ensure_*_buffers when it is large enough; dsat_destroy frees it (free_buffers).
void release_buffers(dsat_ctx* c) {
    c->generation++;        // every pointer a captured step holds may change
    c->VROW.drop(); c->CROW.drop(); c->H1.drop(); c->H2.drop(); c->QS.drop(); c->LIT.drop();
    c->CH.drop(); c->COUT.drop(); c->U1.drop(); c->U2.drop(); c->UOUT.drop(); c->SPRE.drop();
    c->O1.drop(); c->LOGITS.drop(); c->OUT.drop(); c->X.drop(); c->labels.drop();
    c->BITS.drop(); c->LAST.drop(); c->LATCH.drop(); c->FINAL.drop();
    c->done.drop(); c->steps_taken.drop(); c->rounds_run.drop(); c->loss_sum.drop();
    c->graph_sat.drop(); c->graph_map.drop(); c->graph_loss.drop(); c->latch_step.drop();
    c->sat_now.drop(); c->is_sat.drop(); c->sat_any.drop(); c->packed.drop();
    c->inj_normals.drop(); c->inj_uniforms.drop(); c->inj_noisy.drop(); c->inj_labels.drop();
    c->hist_idx.drop(); c->hist_run.drop(); c->hist_totals.drop(); c->hist_keys.drop(); c->hist_counts.drop();
    c->VROWb.drop(); c->CROWb.drop(); c->H1b.drop(); c->H2b.drop(); c->QSb.drop(); c->LITb.drop();
    c->CHb.drop(); c->COUTb.drop(); c->UOUTb.drop(); c->U1b.drop(); c->U2b.drop(); c->SPREb.drop();
    c->O1b.drop();
    c->has_tc_buffers = false;
    c->VROWp.drop(); c->CROWp.drop(); c->SPREp.drop(); c->H1p.drop(); c->H2p.drop();
    c->has_x3_buffers = false;
    c->has_buffers = false;
    c->has_simt_buffers = false;
}

void free_buffers(dsat_ctx* c) {
    c->VROW.release(); c->CROW.release(); c->H1.release(); c->H2.release(); c->QS.release(); c->LIT.release();
    c->CH.release(); c->COUT.release(); c->U1.release(); c->U2.release(); c->UOUT.release(); c->SPRE.release();
    c->O1.release(); c->LOGITS.release(); c->OUT.release(); c->X.release(); c->labels.release();
    c->BITS.release(); c->LAST.release(); c->LATCH.release(); c->FINAL.release();
    c->done.release(); c->steps_taken.release(); c->rounds_run.release(); c->loss_sum.release();
    c->graph_sat.release(); c->graph_map.release(); c->graph_loss.release(); c->latch_step.release();
    c->sat_now.release(); c->is_sat.release(); c->sat_any.release(); c->packed.release();
    c->inj_normals.release(); c->inj_uniforms.release(); c->inj_noisy.release(); c->inj_labels.release();
    c->hist_idx.release(); c->hist_run.release(); c->hist_totals.release(); c->hist_keys.release(); c->hist_counts.release();
    c->hist_seg.release(); c->hist_run_seg.release();
    c->VROWb.release(); c->CROWb.release(); c->H1b.release(); c->H2b.release(); c->QSb.release(); c->LITb.release();
    c->CHb.release(); c->COUTb.release(); c->UOUTb.release(); c->U1b.release(); c->U2b.release(); c->SPREb.release();
    c->O1b.release();
    c->has_tc_buffers = false;
    c->VROWp.release(); c->CROWp.release(); c->SPREp.release(); c->H1p.release(); c->H2p.release();
    c->has_x3_buffers = false;
    c->has_buffers = false;
    c->has_simt_buffers = false;
}

// ---------------------------------------------------------------------------- launch helpers
enum ProfClass { PROF_CLAUSE_GATHER = OP_COUNT, PROF_LITERAL_GATHER, PROF_NORM_CLAUSE, PROF_NORM_VAR, PROF_HEAD,
                 PROF_NOISE, PROF_END, PROF_CLASSES = PROF_END };

// an event before every launch group: the interval up to the next mark belongs to `cls`
void prof_mark(dsat_ctx* c, int cls) {
    if (!c->profiling) return;
    if (c->prof_used == c->prof.size()) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        c->prof.push_back({e, cls});
    }
    c->prof[c->prof_used].cls = cls;
    cudaEventRecord(c->prof[c->prof_used].ev, c->stream);
    c->prof_used++;
}

// ------------------------------------------------------------------ fp32-accurate tensor-core path (x3)
// Stacked hi/lo K-major copies [2N, K64] of the twelve reference layers, cut out of the packed fp32 operators.
int x3_pack_weights(dsat_ctx* c) {
    struct Cut { int op, col0, n; };
    const Cut cuts[12] = {
        {OP_V1, 0, c->HQ}, {OP_Q2, 0, c->Q}, {OP_V1, c->HQ, c->HL}, {OP_L2, 0, c->HL}, {OP_L3, 0, 2 * c->Q},
        {OP_C1, 0, c->HC}, {OP_C2, 0, c->Q + c->F}, {OP_U1, 0, c->HU}, {OP_U2, 0, c->HU}, {OP_U3, 0, c->F},
        {OP_O1, 0, c->HO}, {OP_O2, 0, DSAT_LOGIT_PAD}};
    for (int i = 0; i < 12; ++i) {
        const int op = cuts[i].op, K = c->ops[op].K, Nop = c->ops[op].N, n = cuts[i].n;
        const int K64 = (K + 63) / 64 * 64;
        std::vector<float> w((size_t)K * Nop);
        CK_CUDA(c, dsat_memcpy_sync(w.data(), c->ops[op].w.p, w.size() * sizeof(float), cudaMemcpyDeviceToHost));
        std::vector<__nv_bfloat16> wt((size_t)2 * n * K64, __float2bfloat16(0.f));
        for (int k = 0; k < K; ++k)
            for (int j = 0; j < n; ++j) {
                const float v = w[(size_t)k * Nop + cuts[i].col0 + j];
                const __nv_bfloat16 hi = __float2bfloat16(v);
                wt[(size_t)j * K64 + k] = hi;
                wt[(size_t)(n + j) * K64 + k] = __float2bfloat16(v - __bfloat162float(hi));
            }
        CK_CUDA(c, c->wx[i].alloc(wt.size()));
        CK_CUDA(c, dsat_memcpy_sync(c->wx[i].p, wt.data(), wt.size() * 2, cudaMemcpyHostToDevice));
        c->wx_k64[i] = K64; c->wx_n[i] = n;
    }
    return DSAT_OK;
}

// the seven x3 launches, slots of dsat_ctx::x3
enum { XQ = 0, XL1, XL2, XL3, XC, XU, XO };

int ensure_x3_buffers(dsat_ctx* c) {
    if (c->has_x3_buffers) return DSAT_OK;
    int rc = ensure_common_buffers(c);
    if (rc) return rc;
    const size_t Nt = (size_t)c->Nt, Mt = (size_t)c->Mt;
    const int F = c->F, Q = c->Q;
    CK_CUDA(c, c->VROWp.alloc(2 * Nt * c->ldv()));
    CK_CUDA(c, c->CROWp.alloc(2 * Mt * c->ldc()));
    CK_CUDA(c, c->SPREp.alloc(2 * Nt * F));
    CK_CUDA(c, c->H1p.alloc(2 * Nt * c->HL));
    CK_CUDA(c, c->H2p.alloc(2 * Nt * c->HL));
    CK_CUDA(c, cudaMemsetAsync(c->VROWp.p, 0, c->VROWp.count * 2, c->stream));
    CK_CUDA(c, cudaMemsetAsync(c->CROWp.p, 0, c->CROWp.count * 2, c->stream));
    struct L { int wi; int op; int bias_off; int epi; };        // wi = index into wx[] (reference layer order)
    auto build = [&](int which, const __nv_bfloat16* a_hi, size_t a_plane, long long rows, int k, int lda,
                     std::initializer_list<L> layers, int n_groups, int out_mode, void* out0, void* out1, int ld_out) -> bool {
        x3::X3Mlp& f = c->x3[which];
        f.ready = false;
        x3::X3Params& p = f.p;
        p.n_layers = (int)layers.size();
        p.rows = (int)rows;
        p.n_groups = n_groups;
        p.a_box_rows = (int)(rows < x3::BLOCK_M ? rows : x3::BLOCK_M);
        p.qmaps = Q;
        p.prof = nullptr;
        p.out_mode = out_mode; p.out0 = out0; p.out1 = out1; p.ld_out = ld_out;
        {
            const SkipInfo sk = skip_info(c);
            p.done = sk.done; p.chains_per_group = sk.chains_per_group;
            p.rows_per_chain = rows == c->Mt ? c->m : c->n;
        }
        f.pair_mode = which != XQ && which != XO;       // CTA pair for all but the query and output MLPs
        if (!tc::make_bf16_map(&f.map_a_hi, a_hi, rows, k, lda, p.a_box_rows)) return false;
        if (!tc::make_bf16_map(&f.map_a_lo, a_hi + a_plane, rows, k, lda, p.a_box_rows)) return false;
        int i = 0;
        for (const L& l : layers) {
            x3::X3Layer& ly = p.layer[i];
            const int n_total = c->wx_n[l.wi];
            ly.K = c->ops[l.op].K; ly.N = n_groups > 1 ? 256 : n_total; ly.n_total = n_total;
            ly.epi = l.epi; ly.w_lo_row = n_total; ly.bias = c->ops[l.op].b.p + l.bias_off;
            if (n_groups > 1 && n_total != 256 * n_groups) return false;
            ++i;
        }
        if (!x3::plan_x3(f)) return false;
        i = 0;
        for (const L& l : layers) {     // weight boxes: the layer's N rows, or half of them per CTA of a pair
            const int box = f.p.pair ? p.layer[i].N / 2 : p.layer[i].N;
            if (!tc::make_bf16_map(&f.map_w[i], c->wx[l.wi].p, 2 * c->wx_n[l.wi], c->wx_k64[l.wi], c->wx_k64[l.wi], box)) return false;
            ++i;
        }
        for (; i < x3::MAX_LAYERS; ++i) f.map_w[i] = f.map_w[0];
        if (getenv("DSAT_PLAN_LOG"))
            fprintf(stderr, "[dsat] x3 mlp %d: smem %d B, input ring %d, weight ring %d x %d B, epilogue warps %d, cta pair %d, groups %d\n",
                    which, f.smem_bytes, p.a_slots, p.w_slots, p.w_slot_bytes, p.epi_warps, p.pair, p.n_groups);
        return true;
    };
    const size_t vplane = Nt * c->ldv(), cplane = Mt * c->ldc(), splane = Nt * F, hplane = Nt * c->HL;
    bool ok = true;
    ok = ok && build(XQ, c->VROWp.p, vplane, c->Nt, F + DSAT_AUX_PAD, c->ldv(),
                     {{0, OP_V1, 0, tc::TC_LRELU}, {1, OP_Q2, 0, tc::TC_QUERY}}, 1, x3::OUT_F32, c->QS.p, nullptr, 3 * Q);
    const int lgroups = c->HL > 256 ? c->HL / 256 : 1;
    ok = ok && (c->HL <= 256 || c->HL % 256 == 0);
    ok = ok && build(XL1, c->VROWp.p, vplane, c->Nt, F + DSAT_AUX_PAD, c->ldv(),
                     {{2, OP_V1, c->HQ, tc::TC_LRELU}}, lgroups, x3::OUT_SPLIT, c->H1p.p, c->H1p.p + hplane, c->HL);
    ok = ok && build(XL2, c->H1p.p, hplane, c->Nt, c->HL, c->HL,
                     {{3, OP_L2, 0, tc::TC_LRELU}}, lgroups, x3::OUT_SPLIT, c->H2p.p, c->H2p.p + hplane, c->HL);
    const int l3groups = 2 * Q > 256 ? 2 * Q / 256 : 1;
    ok = ok && build(XL3, c->H2p.p, hplane, c->Nt, c->HL, c->HL,
                     {{4, OP_L3, 0, tc::TC_LINEAR}}, l3groups, x3::OUT_F32, c->LIT.p, nullptr, 2 * Q);
    if (Q + F <= 256 && c->HC <= 256)
        ok = ok && build(XC, c->CROWp.p, cplane, c->Mt, F + 2 * Q, c->ldc(),
                         {{5, OP_C1, 0, tc::TC_LRELU}, {6, OP_C2, 0, tc::TC_LINEAR}}, 1, x3::OUT_F32, c->COUT.p, nullptr, Q + F);
    else ok = false;
    if (c->HU <= 256)
        ok = ok && build(XU, c->VROWp.p, vplane, c->Nt, F + DSAT_AUX_PAD + 3 * Q, c->ldv(),
                         {{7, OP_U1, 0, tc::TC_LRELU}, {8, OP_U2, 0, tc::TC_LRELU}, {9, OP_U3, 0, tc::TC_LINEAR}}, 1, x3::OUT_F32,
                         c->UOUT.p, nullptr, F);
    else ok = false;
    ok = ok && build(XO, c->SPREp.p, splane, c->Nt, F, F,
                     {{10, OP_O1, 0, tc::TC_LRELU}, {11, OP_O2, 0, tc::TC_LINEAR}}, 1, x3::OUT_F32, c->LOGITS.p, nullptr, DSAT_LOGIT_PAD);
    c->x3_ready = ok;
    if (!ok) { c->err = "the fp32-accurate tensor-core path supports feature_maps = query_maps <= 128 (hidden widths <= 256 or 512)"; return DSAT_ERR_UNSUPPORTED; }
    c->has_x3_buffers = true;
    return DSAT_OK;
}

int run_x3(dsat_ctx* c, int which, int prof_class) {
    prof_mark(c, prof_class);
    CK_CUDA(c, x3::launch_x3(c->x3[which], c->device, c->sm_count, c->stream));
    c->launches++;
    return DSAT_OK;
}

int run_linear(dsat_ctx* c, int op, const float* A, int lda, float* Y, int ldy, long long rows, int epi) {
    prof_mark(c, op);
    LinearOp l;
    l.A = A; l.lda = lda; l.W = c->ops[op].w.p; l.ldw = c->ops[op].N; l.bias = c->ops[op].b.p;
    l.Y = Y; l.ldy = ldy; l.rows = (int)rows; l.K = c->ops[op].K; l.N = c->ops[op].N; l.epi = epi; l.qmaps = c->Q;
    CK_CUDA(c, launch_sgemm(l, c->stream));
    c->launches++;
    return DSAT_OK;
}

template <typename KernelLauncher>
int dispatch_width(dsat_ctx* c, int width, KernelLauncher&& fn) {
    switch (width) {
        case 64: fn(std::integral_constant<int, 2>()); break;
        case 128: fn(std::integral_constant<int, 4>()); break;
        case 256: fn(std::integral_constant<int, 8>()); break;
        default: c->err = "feature width must be 64, 128 or 256"; return DSAT_ERR_UNSUPPORTED;
    }
    return DSAT_OK;
}

struct LossScalars { float t, ts, norm_plus; };


// host-side fp32 scalars of train_loss (reference model/query_sat.py:41-42,48-53)
float kl_host(float pa, float pb) {
    float qa = 1.0f - pa;
    float t1 = pa == 0.f ? 0.f : pa * (logf(pa) - logf(pb));
    float t2 = qa == 0.f ? 0.f : qa * (log1pf(-pa) - log1pf(-pb));
    return t1 + t2;
}
LossScalars loss_scalars(float noise_scale) {
    LossScalars s;
    s.t = powf(noise_scale, 0.5f);
    s.ts = fminf(s.t + 0.01f, 1.0f);
    float pa = 0.0f * (1.0f - s.ts) + s.ts / 2.0f;      // distribution_at_time(0, ts)
    float pb = 0.0f * (1.0f - 1.0f) + 1.0f / 2.0f;      // distribution_at_time(0, 1)
    s.norm_plus = kl_host(pa, pb) + 1e-4f;
    return s;
}

static inline bool use_tc(const dsat_ctx* c) { return c->precision == DSAT_BF16 || c->precision == DSAT_BF16_UNFUSED; }
static inline bool use_x3(const dsat_ctx* c) { return c->precision == DSAT_F32_TC; }
// the variable rows in the active precision: fp32 on the CUDA cores, bf16 (hi plane) on the tensor-core paths
static inline float* vrow_f(dsat_ctx* c) { return c->precision == DSAT_F32 ? c->VROW.p : nullptr; }
static inline __nv_bfloat16* vrow_b(dsat_ctx* c) { return use_tc(c) ? c->VROWb.p : use_x3(c) ? c->VROWp.p : nullptr; }
static inline __nv_bfloat16* crow_b(dsat_ctx* c) { return use_tc(c) ? c->CROWb.p : use_x3(c) ? c->CROWp.p : nullptr; }

// buffers of the active precision
int ensure_active_buffers(dsat_ctx* c) {
    if (use_tc(c)) return ensure_tc_buffers(c);
    if (use_x3(c)) return ensure_x3_buffers(c);
    return ensure_buffers(c);
}

int begin_call(dsat_ctx* c, float noise_scale, const float* noisy_dev, const float* uniforms_dev,
               const int* labels_dev, bool use_x, NoiseSource ns, const StepParams* sp_tab = nullptr, const int* sp_cur = nullptr) {
    const long long Nt = c->Nt;
    const int threads = 256;
    const bool x3p = use_x3(c);
    const size_t vplane = x3p ? (size_t)Nt * c->ldv() : 0, cplane = x3p ? (size_t)c->Mt * c->ldc() : 0;
    c->last_noise_scale = noise_scale;
    step_begin_kernel<<<(unsigned)((Nt + threads - 1) / threads), threads, 0, c->stream>>>(
        Nt, noise_scale, use_x ? c->X.p : nullptr, noisy_dev, uniforms_dev, labels_dev, c->labels.p,
        vrow_f(c), c->ldv(), c->F, vrow_b(c), ns, vplane, sp_tab, sp_cur, c->sampling == DSAT_SAMPLE_GUMBEL ? 1 : 0);
    LAUNCHED(c);
    {   // variables_state = ones, clauses_state = ones (reference model/query_sat.py:141,148)
        long long tot;
        if (vrow_f(c)) {
            tot = Nt * (c->F / 4);
            fill_cols_kernel<<<(unsigned)((tot + threads - 1) / threads), threads, 0, c->stream>>>(
                c->VROW.p, c->ldv(), Nt, c->F / 4, 1.0f);
            LAUNCHED(c);
            tot = c->Mt * (c->F / 4);
            fill_cols_kernel<<<(unsigned)((tot + threads - 1) / threads), threads, 0, c->stream>>>(
                c->CROW.p, c->ldc(), c->Mt, c->F / 4, 1.0f);
            LAUNCHED(c);
        } else {
            tot = Nt * (c->F / 8);
            fill_cols_bf16_kernel<<<(unsigned)((tot + threads - 1) / threads), threads, 0, c->stream>>>(
                vrow_b(c), c->ldv(), Nt, c->F / 8, 1.0f);
            LAUNCHED(c);
            if (x3p) {      // lo plane of a state of ones
                fill_cols_bf16_kernel<<<(unsigned)((tot + threads - 1) / threads), threads, 0, c->stream>>>(
                    vrow_b(c) + vplane, c->ldv(), Nt, c->F / 8, 0.0f);
                LAUNCHED(c);
            }
            tot = c->Mt * (c->F / 8);
            fill_cols_bf16_kernel<<<(unsigned)((tot + threads - 1) / threads), threads, 0, c->stream>>>(
                crow_b(c), c->ldc(), c->Mt, c->F / 8, 1.0f);
            LAUNCHED(c);
            if (x3p) {
                fill_cols_bf16_kernel<<<(unsigned)((tot + threads - 1) / threads), threads, 0, c->stream>>>(
                    crow_b(c) + cplane, c->ldc(), c->Mt, c->F / 8, 0.0f);
                LAUNCHED(c);
            }
        }
    }
    CK_CUDA(c, cudaMemsetAsync(c->done.p, 0, c->done.count * sizeof(int), c->stream));
    CK_CUDA(c, cudaMemsetAsync(c->steps_taken.p, 0xff, c->steps_taken.count * sizeof(int), c->stream));
    CK_CUDA(c, cudaMemsetAsync(c->rounds_run.p, 0, c->rounds_run.count * sizeof(int), c->stream));
    CK_CUDA(c, cudaMemsetAsync(c->loss_sum.p, 0, c->loss_sum.count * sizeof(float), c->stream));
    return DSAT_OK;
}

// one tensor-core linear op; out0/out1 describe where the output columns go
int run_linear_tc(dsat_ctx* c, int op, long long rows, int epi, void* p0, int ld0, bool bf0,
                  void* p1 = nullptr, int ld1 = 0, bool bf1 = false, int split = 0) {
    prof_mark(c, op);
    tc::TcLinear l;
    l.map_a = c->map_a[op]; l.map_b = c->map_b[op]; l.bias = c->ops[op].b.p;
    l.out.ptr0 = p0; l.out.ld0 = ld0; l.out.bf16_0 = bf0 ? 1 : 0;
    l.out.ptr1 = p1; l.out.ld1 = ld1; l.out.bf16_1 = bf1 ? 1 : 0; l.out.split = split;
    l.rows = (int)rows; l.K = c->ops[op].K; l.N = c->ops[op].N; l.epi = epi; l.qmaps = c->Q;
    l.a_box_rows = c->a_box_rows[op]; l.b_box_rows = c->b_box_rows[op];
    CK_CUDA(c, tc::launch_tc_linear(l, c->stream));
    c->launches++;
    return DSAT_OK;
}

int run_fused(dsat_ctx* c, int which, int prof_class) {
    prof_mark(c, prof_class);
    CK_CUDA(c, fm::launch_fused(c->fused[which], c->sm_count, c->stream));
    c->launches++;
    return DSAT_OK;
}

// Shared-memory staged gathers (small formulas): pick the widest feature slice whose two tables fit;
// returns false when they do not fit (the L2-gather kernels run instead).
static int pick_slice_width(size_t table_rows, int Q, size_t* bytes_out, int budget_kb, int elt_bytes) {
    // budget_kb: shared memory per CTA we aim for (smaller slices -> more co-resident CTAs, so one CTA's staging
    // overlaps the others' compute)
    const int widths[3] = {128, 64, 32};
    for (int pass = 0; pass < 2; ++pass)
        for (int w : widths) {
            if (w > Q || Q % w) continue;
            const size_t bytes = 2 * table_rows * (size_t)w * (size_t)elt_bytes;
            if (bytes <= (size_t)(pass == 0 ? budget_kb : 220) * 1024u) { *bytes_out = bytes; return w; }
        }
    return 0;
}

// staging the 16-bit adjacency next to the tables is worth it only if it does not cost a resident CTA
static bool idx_fits(size_t table_bytes, int idx_vecs) {
    if (idx_vecs <= 0) return false;
    const size_t sm_bytes = 227 * 1024, reserved = 1024, with_idx = table_bytes + (size_t)idx_vecs * 16;
    if (with_idx + reserved > sm_bytes) return false;
    return sm_bytes / (with_idx + reserved) == sm_bytes / (table_bytes + reserved);
}


bool launch_clause_gather_smem(dsat_ctx* c, const UnitGraphDev& g) {
    if (c->n_graphs != 1) return false;
    size_t bytes = 0;
    const int w = pick_slice_width((size_t)2 * c->n, c->Q, &bytes, 56);    // measured best at cfg2: 4 CTAs per SM
    if (!w) return false;
    dim3 grid((unsigned)c->chains, (unsigned)(c->Q / w));
    const int Q = c->Q;
    const bool si = idx_fits(bytes, g.cl_idx16_vecs);
    const size_t smem = bytes + (si ? (size_t)g.cl_idx16_vecs * 16 : 0);
    auto launch = [&](auto kernel) -> bool {
        kernel<<<grid, 512, smem, c->stream>>>(g, Q, c->LITb.p, 2 * Q, c->QSb.p, 3 * Q, Q, c->CROWb.p, c->ldc(), c->F, skip_info(c));
        return true;
    };
    if (w == 128) return si ? launch(clause_gather_smem_kernel<128, true>) : launch(clause_gather_smem_kernel<128, false>);
    if (w == 64) return si ? launch(clause_gather_smem_kernel<64, true>) : launch(clause_gather_smem_kernel<64, false>);
    return si ? launch(clause_gather_smem_kernel<32, true>) : launch(clause_gather_smem_kernel<32, false>);
}

bool launch_literal_gather_smem(dsat_ctx* c, const UnitGraphDev& g) {
    if (c->n_graphs != 1) return false;
    size_t bytes = 0;
    const int w = pick_slice_width((size_t)c->m, c->Q, &bytes, 112);
    if (!w) return false;
    dim3 grid((unsigned)c->chains, (unsigned)(c->Q / w));
    const int Q = c->Q, F = c->F;
    const bool si = idx_fits(bytes, g.lit_idx16_vecs);
    const size_t smem = bytes + (si ? (size_t)g.lit_idx16_vecs * 16 : 0);
    auto launch = [&](auto kernel) -> bool {
        kernel<<<grid, 512, smem, c->stream>>>(g, Q, c->CROWb.p, c->ldc(), F + Q, c->COUTb.p, Q + F, c->QSb.p, 3 * Q, c->VROWb.p,
                                               c->ldv(), F + DSAT_AUX_PAD, skip_info(c));
        return true;
    };
    if (w == 128) return si ? launch(literal_gather_smem_kernel<128, true>) : launch(literal_gather_smem_kernel<128, false>);
    if (w == 64) return si ? launch(literal_gather_smem_kernel<64, true>) : launch(literal_gather_smem_kernel<64, false>);
    return si ? launch(literal_gather_smem_kernel<32, true>) : launch(literal_gather_smem_kernel<32, false>);
}

// fp32 tables (fp32-accurate tensor-core path): outputs go to the hi/lo planes
bool launch_clause_gather_smem_f32(dsat_ctx* c, const UnitGraphDev& g) {
    if (c->n_graphs != 1) return false;
    size_t bytes = 0;
    const int w = pick_slice_width((size_t)2 * c->n, c->Q, &bytes, 110, 4);       // both fp32 tables per CTA
    // one CTA per SM cannot overlap its staging with another CTA's gather: measured slower than the L2 gather (uf250)
    if (!w || bytes > 112 * 1024) return false;
    dim3 grid((unsigned)c->chains, (unsigned)(c->Q / w));
    const int Q = c->Q;
    const bool si = idx_fits(bytes, g.cl_idx16_vecs);
    const size_t smem = bytes + (si ? (size_t)g.cl_idx16_vecs * 16 : 0);
    const size_t cplane = (size_t)c->Mt * c->ldc();
    auto launch = [&](auto kernel) -> bool {
        kernel<<<grid, 512, smem, c->stream>>>(g, Q, c->LIT.p, 2 * Q, c->QS.p, 3 * Q, Q, c->CROWp.p, cplane, c->ldc(), c->F, skip_info(c));
        return true;
    };
    if (w == 128) return si ? launch(clause_gather_smem_f32x2_kernel<128, true>) : launch(clause_gather_smem_f32x2_kernel<128, false>);
    if (w == 64) return si ? launch(clause_gather_smem_f32x2_kernel<64, true>) : launch(clause_gather_smem_f32x2_kernel<64, false>);
    return si ? launch(clause_gather_smem_f32x2_kernel<32, true>) : launch(clause_gather_smem_f32x2_kernel<32, false>);
}

bool launch_literal_gather_smem_f32(dsat_ctx* c, const UnitGraphDev& g) {
    if (c->n_graphs != 1) return false;
    size_t bytes = 0;
    const int w = pick_slice_width((size_t)c->m, c->Q, &bytes, 112, 2);             // one fp32 table per CTA
    if (!w || bytes > 112 * 1024) return false;     // (as on the clause side: uf250's 1065 clause rows ran 1.39 ms against 1.09 ms)
    dim3 grid((unsigned)c->chains, (unsigned)(2 * (c->Q / w)));
    const int Q = c->Q, F = c->F;
    const bool si = idx_fits(bytes, g.lit_idx16_vecs);
    const size_t smem = bytes + (si ? (size_t)g.lit_idx16_vecs * 16 : 0);
    const size_t cplane = (size_t)c->Mt * c->ldc(), vplane = (size_t)c->Nt * c->ldv();
    auto launch = [&](auto kernel) -> bool {
        kernel<<<grid, 512, smem, c->stream>>>(g, Q, c->CROWp.p, cplane, c->ldc(), F + Q, c->COUT.p, Q + F, c->QS.p, 3 * Q,
                                                c->VROWp.p, vplane, c->ldv(), F + DSAT_AUX_PAD, skip_info(c));
        return true;
    };
    if (w == 128) return si ? launch(literal_gather_smem_f32_kernel<128, true>) : launch(literal_gather_smem_f32_kernel<128, false>);
    if (w == 64) return si ? launch(literal_gather_smem_f32_kernel<64, true>) : launch(literal_gather_smem_f32_kernel<64, false>);
    return si ? launch(literal_gather_smem_f32_kernel<32, true>) : launch(literal_gather_smem_f32_kernel<32, false>);
}

// PairNorm with the graph resident in shared memory (split-plane path); false when a graph does not fit
template <int V>
bool launch_pairnorm_smem(dsat_ctx* c, const int* seg, int rows_per_chain, int max_graph_rows, const float* src, int ld_src, int src_off,
                          __nv_bfloat16* state_hi, size_t state_plane, int ld_state, __nv_bfloat16* pre_hi, size_t pre_plane, int ld_pre) {
    constexpr int F = 32 * V;
    // small graphs: several CTAs of 256 threads per SM; large ones: one CTA of 1024 threads
    const size_t row_bytes = (size_t)max_graph_rows * F * 4;
    const int threads = row_bytes > 100 * 1024 ? 1024 : row_bytes > 48 * 1024 ? 512 : 256;
    const int groups = threads / F > 0 ? threads / F : 1;
    const size_t smem = (size_t)(F + groups * F) * 4 + row_bytes;
    if (smem > 227 * 1024) return false;
    int per_sm = (int)((228 * 1024) / (smem + 1024));
    const int by_threads = 2048 / threads;
    if (per_sm > by_threads) per_sm = by_threads;
    if (per_sm < 1) per_sm = 1;
    int grid = c->sm_count * per_sm;
    if (grid > c->total_graphs) grid = c->total_graphs;
    pairnorm_smem_kernel<V><<<grid, threads, smem, c->stream>>>(seg, c->n_graphs, rows_per_chain, c->total_graphs, src, ld_src, src_off,
                                                                state_hi, state_plane, ld_state, pre_hi, pre_plane, ld_pre, skip_info(c));
    return true;
}

// One MLP in the active precision: 0 variables_query (VROW -> QS), 1 lit_query (VROW -> LIT), 2 clause_update
// (CROW -> COUT), 3 update_gate (VROW -> UOUT), 4 variables_output (SPRE -> LOGITS).  On the per-layer paths the query and
// literal MLPs share their first layer (OP_V1, both halves in one launch): `v1_done` says it has already run.
// Each launch is profiled under the last linear op it runs.
int run_mlp(dsat_ctx* c, int which, bool v1_done = false) {
    const long long Nt = c->Nt, Mt = c->Mt;
    const int F = c->F, Q = c->Q, ldh1 = c->ldh1();
    int rc = DSAT_OK;
    if (use_x3(c)) {
        switch (which) {
            case 0: return run_x3(c, XQ, OP_Q2);
            case 1: if ((rc = run_x3(c, XL1, OP_V1)) || (rc = run_x3(c, XL2, OP_L2))) return rc;
                    return run_x3(c, XL3, OP_L3);
            case 2: return run_x3(c, XC, OP_C2);
            case 3: return run_x3(c, XU, OP_U3);
            default: return run_x3(c, XO, OP_O2);
        }
    }
    if (c->precision == DSAT_BF16 && c->fused_ready) {
        static const int cls[5] = {OP_Q2, OP_L3, OP_C2, OP_U3, OP_O2};
        return run_fused(c, which, cls[which]);
    }
    if (use_tc(c)) {
        if (which <= 1 && !v1_done && (rc = run_linear_tc(c, OP_V1, Nt, tc::TC_LRELU, c->H1b.p, ldh1, true))) return rc;
        switch (which) {
            case 0: return run_linear_tc(c, OP_Q2, Nt, tc::TC_QUERY, c->QSb.p, 3 * Q, true);
            case 1: if ((rc = run_linear_tc(c, OP_L2, Nt, tc::TC_LRELU, c->H2b.p, c->HL, true))) return rc;
                    return run_linear_tc(c, OP_L3, Nt, tc::TC_LINEAR, c->LITb.p, 2 * Q, true);
            case 2: if ((rc = run_linear_tc(c, OP_C1, Mt, tc::TC_LRELU, c->CHb.p, c->HC, true))) return rc;
                    return run_linear_tc(c, OP_C2, Mt, tc::TC_LINEAR, c->COUTb.p, Q + F, true);
            case 3: if ((rc = run_linear_tc(c, OP_U1, Nt, tc::TC_LRELU, c->U1b.p, c->HU, true)) ||
                        (rc = run_linear_tc(c, OP_U2, Nt, tc::TC_LRELU, c->U2b.p, c->HU, true))) return rc;
                    return run_linear_tc(c, OP_U3, Nt, tc::TC_LINEAR, c->UOUTb.p, F, true);
            default: if ((rc = run_linear_tc(c, OP_O1, Nt, tc::TC_LRELU, c->O1b.p, c->HO, true))) return rc;
                     return run_linear_tc(c, OP_O2, Nt, tc::TC_LINEAR, c->LOGITS.p, DSAT_LOGIT_PAD, false);
        }
    }
    const int ldv = c->ldv(), ldc = c->ldc();
    if (which <= 1 && !v1_done && (rc = run_linear(c, OP_V1, c->VROW.p, ldv, c->H1.p, ldh1, Nt, EPI_LRELU))) return rc;
    switch (which) {
        case 0: return run_linear(c, OP_Q2, c->H1.p, ldh1, c->QS.p, 3 * Q, Nt, EPI_QUERY);
        case 1: if ((rc = run_linear(c, OP_L2, c->H1.p + c->HQ, ldh1, c->H2.p, c->HL, Nt, EPI_LRELU))) return rc;
                return run_linear(c, OP_L3, c->H2.p, c->HL, c->LIT.p, 2 * Q, Nt, EPI_LINEAR);
        case 2: if ((rc = run_linear(c, OP_C1, c->CROW.p, ldc, c->CH.p, c->HC, Mt, EPI_LRELU))) return rc;
                return run_linear(c, OP_C2, c->CH.p, c->HC, c->COUT.p, Q + F, Mt, EPI_LINEAR);
        case 3: if ((rc = run_linear(c, OP_U1, c->VROW.p, ldv, c->U1.p, c->HU, Nt, EPI_LRELU)) ||
                    (rc = run_linear(c, OP_U2, c->U1.p, c->HU, c->U2.p, c->HU, Nt, EPI_LRELU))) return rc;
                return run_linear(c, OP_U3, c->U2.p, c->HU, c->UOUT.p, F, Nt, EPI_LINEAR);
        default: if ((rc = run_linear(c, OP_O1, c->SPRE.p, F, c->O1.p, c->HO, Nt, EPI_LRELU))) return rc;
                 return run_linear(c, OP_O2, c->O1.p, c->HO, c->LOGITS.p, DSAT_LOGIT_PAD, Nt, EPI_LINEAR);
    }
}

// One message-passing round (reference model/query_sat.py:225-348).
int run_round(dsat_ctx* c, int round, const float* normals_dev, NoiseSource ns, LossScalars ls,
              const StepParams* sp_tab = nullptr, const int* sp_cur = nullptr) {
    const long long Nt = c->Nt, Mt = c->Mt;
    const int F = c->F, Q = c->Q, ldv = c->ldv(), ldc = c->ldc();
    const UnitGraphDev g = graph_view(c);
    const bool tcp = use_tc(c);
    const bool x3p = use_x3(c);
    const size_t vplane = x3p ? (size_t)Nt * ldv : 0, cplane = x3p ? (size_t)Mt * ldc : 0;
    const SkipInfo skip = skip_info(c);
    int rc;
    {
        const int threads = 256;
        prof_mark(c, PROF_NOISE);
        round_noise_kernel<<<(unsigned)((Nt + threads - 1) / threads), threads, 0, c->stream>>>(
            Nt, normals_dev, vrow_f(c), ldv, F, vrow_b(c), ns, (unsigned)round, vplane, sp_tab, sp_cur, skip, c->n);
        LAUNCHED(c);
    }
    // variables_query (+ softplus pair) (:240);  lit_query (:252), which shares the first layer on the per-layer paths
    if ((rc = run_mlp(c, 0)) || (rc = run_mlp(c, 1, true))) return rc;
    // clause side gather: clause_messages and 4*clauses_loss                    (:241, :248, :255-256)
    prof_mark(c, PROF_CLAUSE_GATHER);
    rc = dispatch_width(c, Q, [&](auto v) {
        constexpr int V = decltype(v)::value;
        const int grid = tcp ? gather_grid(clause_gather_kernel<V, __nv_bfloat16>, Mt, GATHER_WARPS, c->sm_count)
                             : gather_grid(clause_gather_kernel<V, float>, Mt, GATHER_WARPS, c->sm_count);
        if (x3p) {
            if (!launch_clause_gather_smem_f32(c, g))
                clause_gather_kernel<V, float><<<grid, GATHER_WARPS * 32, 0, c->stream>>>(
                    g, c->chains, c->LIT.p, 2 * Q, c->QS.p, 3 * Q, Q, nullptr, ldc, F, crow_b(c), cplane, skip);
        } else if (!tcp)
            clause_gather_kernel<V, float><<<grid, GATHER_WARPS * 32, 0, c->stream>>>(
                g, c->chains, c->LIT.p, 2 * Q, c->QS.p, 3 * Q, Q, c->CROW.p, ldc, F, nullptr, 0, skip);
        else if (!launch_clause_gather_smem(c, g))
            clause_gather_kernel<V, __nv_bfloat16><<<grid, GATHER_WARPS * 32, 0, c->stream>>>(
                g, c->chains, c->LITb.p, 2 * Q, c->QSb.p, 3 * Q, Q, c->CROWb.p, ldc, F, nullptr, 0, skip);
    });
    if (rc) return rc;
    LAUNCHED(c);
    // clause_update MLP                                                          (:258-261)
    if ((rc = run_mlp(c, 2))) return rc;
    // literal side gather                                                        (:245-246, :269-273)
    prof_mark(c, PROF_LITERAL_GATHER);
    rc = dispatch_width(c, Q, [&](auto v) {
        constexpr int V = decltype(v)::value;
        const int grid = tcp ? gather_grid(literal_gather_kernel<V, __nv_bfloat16>, Nt, GATHER_WARPS, c->sm_count)
                             : gather_grid(literal_gather_kernel<V, float>, Nt, GATHER_WARPS, c->sm_count);
        if (x3p) {  // 4*clauses_loss is read back as hi + lo from the clause rows' planes
            if (!launch_literal_gather_smem_f32(c, g))
                literal_gather_kernel<V, float><<<grid, GATHER_WARPS * 32, 0, c->stream>>>(
                    g, c->chains, nullptr, ldc, F + Q, c->COUT.p, Q + F, c->QS.p, 3 * Q, nullptr, ldv, F + DSAT_AUX_PAD,
                    vrow_b(c), vplane, crow_b(c), cplane, skip);
        } else if (!tcp)
            literal_gather_kernel<V, float><<<grid, GATHER_WARPS * 32, 0, c->stream>>>(
                g, c->chains, c->CROW.p, ldc, F + Q, c->COUT.p, Q + F, c->QS.p, 3 * Q, c->VROW.p, ldv, F + DSAT_AUX_PAD,
                nullptr, 0, nullptr, 0, skip);
        else if (!launch_literal_gather_smem(c, g))
            literal_gather_kernel<V, __nv_bfloat16><<<grid, GATHER_WARPS * 32, 0, c->stream>>>(
                g, c->chains, c->CROWb.p, ldc, F + Q, c->COUTb.p, Q + F, c->QSb.p, 3 * Q, c->VROWb.p, ldv, F + DSAT_AUX_PAD,
                nullptr, 0, nullptr, 0, skip);
    });
    if (rc) return rc;
    LAUNCHED(c);
    // clause PairNorm + residual + carry                                        (:263-266, :348)
    prof_mark(c, PROF_NORM_CLAUSE);
    rc = dispatch_width(c, F, [&](auto v) {
        constexpr int V = decltype(v)::value;
        const int grid = c->total_graphs < c->sm_count * 8 ? c->total_graphs : c->sm_count * 8;
        if (x3p) {
            if (!launch_pairnorm_smem<V>(c, c->clause_seg.p, c->m, c->max_graph_clauses, c->COUT.p, Q + F, Q, crow_b(c), cplane, ldc,
                                         nullptr, 0, 0))
                pairnorm_kernel<V, float, float><<<grid, PN_WARPS * 32, 0, c->stream>>>(
                    c->clause_seg.p, c->n_graphs, c->m, c->total_graphs, c->COUT.p, Q + F, Q, nullptr, ldc, nullptr, 0,
                    crow_b(c), cplane, nullptr, 0, skip);
        } else if (!tcp)
            pairnorm_kernel<V, float, float><<<grid, PN_WARPS * 32, 0, c->stream>>>(
                c->clause_seg.p, c->n_graphs, c->m, c->total_graphs, c->COUT.p, Q + F, Q, c->CROW.p, ldc, nullptr, 0,
                nullptr, 0, nullptr, 0, skip);
        else
            pairnorm_bf16_kernel<32 * V><<<grid, PN_WARPS * 32, 0, c->stream>>>(
                c->clause_seg.p, c->n_graphs, c->m, c->total_graphs, c->COUTb.p, Q + F, Q, c->CROWb.p, ldc, nullptr, 0, skip);
    });
    if (rc) return rc;
    LAUNCHED(c);
    // update_gate MLP                                                            (:277-278)
    if ((rc = run_mlp(c, 3))) return rc;
    // variables PairNorm + residual + carry                                     (:279-280, :347)
    prof_mark(c, PROF_NORM_VAR);
    rc = dispatch_width(c, F, [&](auto v) {
        constexpr int V = decltype(v)::value;
        int grid = c->total_graphs < c->sm_count * 8 ? c->total_graphs : c->sm_count * 8;
        if (x3p) {
            if (!launch_pairnorm_smem<V>(c, c->var_seg.p, c->n, c->max_graph_vars, c->UOUT.p, F, 0, vrow_b(c), vplane, ldv,
                                         c->SPREp.p, (size_t)Nt * F, F))
                pairnorm_kernel<V, float, float><<<grid, PN_WARPS * 32, 0, c->stream>>>(
                    c->var_seg.p, c->n_graphs, c->n, c->total_graphs, c->UOUT.p, F, 0, nullptr, ldv, nullptr, F,
                    vrow_b(c), vplane, c->SPREp.p, (size_t)Nt * F, skip);
        } else if (!tcp)
            pairnorm_kernel<V, float, float><<<grid, PN_WARPS * 32, 0, c->stream>>>(
                c->var_seg.p, c->n_graphs, c->n, c->total_graphs, c->UOUT.p, F, 0, c->VROW.p, ldv, c->SPRE.p, F,
                nullptr, 0, nullptr, 0, skip);
        else
            pairnorm_bf16_kernel<32 * V><<<grid, PN_WARPS * 32, 0, c->stream>>>(
                c->var_seg.p, c->n_graphs, c->n, c->total_graphs, c->UOUTb.p, F, 0, c->VROWb.p, ldv, c->SPREb.p, F, skip);
    });
    if (rc) return rc;
    LAUNCHED(c);
    // variables_output MLP                                                       (:283)
    if ((rc = run_mlp(c, 4))) return rc;
    // logit map selection, SAT check, early exit                                 (:289-338)
    prof_mark(c, PROF_HEAD);
    head_kernel<<<c->total_graphs, 128, 0, c->stream>>>(g, c->total_graphs, c->group_graphs, c->LOGITS.p,
                                                         DSAT_LOGIT_PAD, c->labels.p, ls.t, ls.ts, ls.norm_plus,
                                                         c->done.p, c->OUT.p, c->BITS.p, c->graph_sat.p,
                                                         c->graph_loss.p, c->graph_map.p, sp_tab, sp_cur,
                                                         c->has_batches ? c->graph_group.p : nullptr);
    LAUNCHED(c);
    group_finalize_kernel<<<(c->n_groups + 127) / 128, 128, 0, c->stream>>>(
        c->n_groups, c->group_graphs, c->total_graphs, round, c->graph_sat.p, c->graph_loss.p, c->done.p,
        c->steps_taken.p, c->loss_sum.p, c->rounds_run.p, c->has_batches ? c->batch_seg.p : nullptr);
    LAUNCHED(c);
    prof_mark(c, PROF_END);
    return DSAT_OK;
}

int pack_weights(dsat_ctx* c, const float* const* kernels, const float* const* biases, const int* in_dims,
                 const int* out_dims) {
    // reference layer order: query0 query1 lit0 lit1 lit2 clause0 clause1 upd0 upd1 upd2 out0 out1
    const int F = c->F, Q = c->Q, A = DSAT_AUX_PAD;
    const int hq = out_dims[0], hl = out_dims[2], hc = out_dims[5], hu = out_dims[7], ho = out_dims[10];
    c->HQ = pad16(hq); c->HL = pad16(hl); c->HC = pad16(hc); c->HU = pad16(hu); c->HO = pad16(ho);

    auto upload = [&](int op, int K, int N, const std::vector<float>& w, const std::vector<float>& b) -> int {
        c->ops[op].K = K; c->ops[op].N = N;
        CK_CUDA(c, c->ops[op].w.alloc((size_t)K * N));
        CK_CUDA(c, c->ops[op].b.alloc((size_t)N));
        CK_CUDA(c, dsat_memcpy_sync(c->ops[op].w.p, w.data(), w.size() * sizeof(float), cudaMemcpyHostToDevice));
        CK_CUDA(c, dsat_memcpy_sync(c->ops[op].b.p, b.data(), b.size() * sizeof(float), cudaMemcpyHostToDevice));
        return DSAT_OK;
    };
    // copy a [rows, cols] block of a reference kernel (leading dim src_ld) into a packed matrix
    auto blit = [](std::vector<float>& dst, int dst_ld, int dst_r, int dst_c, const float* src, int src_ld,
                   int src_r, int rows, int cols) {
        for (int r = 0; r < rows; ++r)
            memcpy(&dst[(size_t)(dst_r + r) * dst_ld + dst_c], src + (size_t)(src_r + r) * src_ld, cols * sizeof(float));
    };
    auto plain = [&](int op, int layer, int Kp, int Np) -> int {
        std::vector<float> w((size_t)Kp * Np, 0.f), b(Np, 0.f);
        blit(w, Np, 0, 0, kernels[layer], out_dims[layer], 0, in_dims[layer], out_dims[layer]);
        memcpy(b.data(), biases[layer], out_dims[layer] * sizeof(float));
        return upload(op, Kp, Np, w, b);
    };
    int rc;
    {   // OP_V1: rows [variables F | aux 9 (+7 zero)], cols [query hidden | lit hidden]
        const int K = F + A, N = c->HQ + c->HL;
        std::vector<float> w((size_t)K * N, 0.f), b(N, 0.f);
        blit(w, N, 0, 0, kernels[0], hq, 0, F + 9, hq);
        blit(w, N, 0, c->HQ, kernels[2], hl, 0, F + 9, hl);
        memcpy(b.data(), biases[0], hq * sizeof(float));
        memcpy(b.data() + c->HQ, biases[2], hl * sizeof(float));
        if ((rc = upload(OP_V1, K, N, w, b))) return rc;
    }
    if ((rc = plain(OP_Q2, 1, c->HQ, Q))) return rc;
    if ((rc = plain(OP_L2, 3, c->HL, c->HL))) return rc;
    if ((rc = plain(OP_L3, 4, c->HL, 2 * Q))) return rc;
    if ((rc = plain(OP_C1, 5, F + 2 * Q, c->HC))) return rc;
    if ((rc = plain(OP_C2, 6, c->HC, Q + F))) return rc;
    {   // OP_U1: reference rows [grad Q | variables F | aux 9 | loss_pos Q | loss_neg Q]
        //        packed rows    [variables F | aux 16 | grad Q | loss_pos Q | loss_neg Q]
        const int K = F + A + 3 * Q, N = c->HU;
        std::vector<float> w((size_t)K * N, 0.f), b(N, 0.f);
        blit(w, N, 0, 0, kernels[7], hu, Q, F + 9, hu);
        blit(w, N, F + A, 0, kernels[7], hu, 0, Q, hu);
        blit(w, N, F + A + Q, 0, kernels[7], hu, Q + F + 9, 2 * Q, hu);
        memcpy(b.data(), biases[7], hu * sizeof(float));
        if ((rc = upload(OP_U1, K, N, w, b))) return rc;
    }
    if ((rc = plain(OP_U2, 8, c->HU, c->HU))) return rc;
    if ((rc = plain(OP_U3, 9, c->HU, F))) return rc;
    if ((rc = plain(OP_O1, 10, F, c->HO))) return rc;
    if ((rc = plain(OP_O2, 11, c->HO, DSAT_LOGIT_PAD))) return rc;
    return DSAT_OK;
}

}  // namespace

// =================================================================================== C ABI
static void drop_step_graph(dsat_ctx* c) {
    if (c->step_graph) cudaGraphExecDestroy(c->step_graph);
    c->step_graph = nullptr;
    c->step_graph_generation = -1;
}

extern "C" {

int dsat_version(void) { return 2; }

int dsat_build_info(void) {
    int flags = 1;      // the tcgen05 paths are always compiled in
#ifdef DSAT_ASSERT
    flags |= 2;
#endif
    return flags;
}

int dsat_create(int device, dsat_ctx** out) {
    if (!out) return DSAT_ERR_ARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) return DSAT_ERR_CUDA;
    dsat_ctx* c = new dsat_ctx();
    c->device = device;
    if (cudaSetDevice(device) != cudaSuccess) { delete c; return DSAT_ERR_CUDA; }
    cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (configure_kernels_for_device() != cudaSuccess) { delete c; return DSAT_ERR_CUDA; }
#ifdef DSAT_ASSERT
    if (!g_assert_host && cudaHostAlloc(reinterpret_cast<void**>(&g_assert_host), 2 * sizeof(int), cudaHostAllocMapped) == cudaSuccess) {
        g_assert_host[0] = g_assert_host[1] = 0;
        int* dev_view = nullptr;
        if (cudaHostGetDevicePointer(reinterpret_cast<void**>(&dev_view), g_assert_host, 0) == cudaSuccess)
            cudaMemcpyToSymbol(g_dsat_assert_slot, &dev_view, sizeof(dev_view));
    }
#endif
    if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return DSAT_ERR_CUDA; }
    c->stream = c->own_stream;
    cudaEventCreate(&c->ev0);
    cudaEventCreate(&c->ev1);
    *out = c;
    return DSAT_OK;
}

void dsat_destroy(dsat_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    drop_step_graph(c);
    c->step_tab.release(); c->step_cur.release();
    free_buffers(c);
    for (auto& op : c->ops) {
        op.w.release(); op.b.release();
        op.w_bf16.release();
    }
    for (auto& w : c->wx) w.release();
    c->cl_rowptr.release(); c->cl_lit.release(); c->lit_rowptr.release(); c->lit_clause.release();
    c->batch_seg.release(); c->graph_group.release(); c->row_graph.release(); c->graph_elem0.release();
    c->var_seg.release(); c->clause_seg.release(); c->deg_w.release(); c->vdeg_w.release(); c->rev_w.release(); c->var_order.release();
    c->cl_idx16.release(); c->lit_idx16.release(); c->cl_idx16_vecs = c->lit_idx16_vecs = 0;
    c->cl_desc.release(); c->lit_desc.release(); c->lit_desc4.release();
    for (auto& pm : c->prof) cudaEventDestroy(pm.ev);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;
}

const char* dsat_last_error(const dsat_ctx* c) { return c ? c->err.c_str() : "null context"; }

int dsat_set_stream(dsat_ctx* c, void* s) {
    if (!c) return DSAT_ERR_ARG;
    c->generation++;
    c->stream = s ? reinterpret_cast<cudaStream_t>(s) : c->own_stream;
    return DSAT_OK;
}

int dsat_synchronize(dsat_ctx* c) {
    if (!c) return DSAT_ERR_ARG;
    CK_CUDA(c, cudaSetDevice(c->device));
    CK_CUDA(c, cudaStreamSynchronize(c->stream));
    return DSAT_OK;
}

int dsat_timer_begin(dsat_ctx* c) {
    if (!c) return DSAT_ERR_ARG;
    CK_CUDA(c, cudaSetDevice(c->device));
    CK_CUDA(c, cudaEventRecord(c->ev0, c->stream));
    return DSAT_OK;
}

int dsat_timer_end(dsat_ctx* c, float* ms) {
    if (!c || !ms) return DSAT_ERR_ARG;
    CK_CUDA(c, cudaEventRecord(c->ev1, c->stream));
    CK_CUDA(c, cudaEventSynchronize(c->ev1));
    CK_CUDA(c, cudaEventElapsedTime(ms, c->ev0, c->ev1));
    return DSAT_OK;
}

long long dsat_launch_count(const dsat_ctx* c) { return c ? c->launches : 0; }

// widths the x3 kernels tile: every layer at most 256 wide, or a single layer that is a multiple of 256
static bool x3_supported(const dsat_ctx* c) {
    auto wide_ok = [](int n) { return n <= 256 || n % 256 == 0; };
    return c->HQ <= 256 && c->HC <= 256 && c->HU <= 256 && c->HO <= 256 && c->Q + c->F <= 256 && wide_ok(c->HL) && wide_ok(2 * c->Q);
}

int dsat_get_precision(const dsat_ctx* c) { return c ? c->precision : DSAT_ERR_ARG; }

int dsat_set_precision(dsat_ctx* c, int dtype) {
    if (!c) return DSAT_ERR_ARG;
    if (dtype == DSAT_F32 || dtype == DSAT_BF16 || dtype == DSAT_BF16_UNFUSED) { c->precision = dtype; return DSAT_OK; }
    if (dtype == DSAT_F32_TC) {
        if (c->has_model && !x3_supported(c)) {
            c->err = "DSAT_F32_TC needs layer widths of at most 256 (feature_maps, query_maps <= 128); use DSAT_F32";
            return DSAT_ERR_UNSUPPORTED;
        }
        c->precision = dtype;
        return DSAT_OK;
    }
    c->err = "unknown precision";
    return DSAT_ERR_UNSUPPORTED;
}

int dsat_set_sampling(dsat_ctx* c, int mode) {
    if (!c) return DSAT_ERR_ARG;
    CK_ARG(c, mode == DSAT_SAMPLE_INVERSE_CDF || mode == DSAT_SAMPLE_GUMBEL, "dsat_set_sampling: unknown mode");
    if (mode != c->sampling) c->generation++;        // baked into the captured step
    c->sampling = mode;
    return DSAT_OK;
}

int dsat_set_model(dsat_ctx* c, int n_layers, const float* const* kernels, const float* const* biases,
                   const int* in_dims, const int* out_dims) {
    if (!c) return DSAT_ERR_ARG;
    CK_ARG(c, n_layers == 12 && kernels && biases && in_dims && out_dims, "dsat_set_model: expected 12 layers");
    CK_CUDA(c, cudaSetDevice(c->device));
    const int F = in_dims[10], Q = out_dims[1];
    CK_ARG(c, (F == 64 || F == 128 || F == 256) && (Q == 64 || Q == 128 || Q == 256),
           "feature_maps and query_maps must be 64, 128 or 256");
    const int v1 = F + 9;
    bool ok = in_dims[0] == v1 && in_dims[1] == out_dims[0] && in_dims[2] == v1 && in_dims[3] == out_dims[2] &&
              in_dims[4] == out_dims[3] && out_dims[4] == 2 * Q && in_dims[5] == F + 2 * Q &&
              in_dims[6] == out_dims[5] && out_dims[6] == F + Q && in_dims[7] == Q + v1 + 2 * Q &&
              in_dims[8] == out_dims[7] && in_dims[9] == out_dims[8] && out_dims[9] == F &&
              in_dims[11] == out_dims[10] && out_dims[11] == DSAT_LOGIT_MAPS;
    CK_ARG(c, ok, "dsat_set_model: layer dimensions do not form the QuerySAT MLPs");
    CK_CUDA(c, cudaStreamSynchronize(c->stream));
    if (c->has_buffers && (c->F != F || c->Q != Q)) release_buffers(c);
    c->generation++;        // weight buffers are re-allocated
    // the whole-MLP plans hold the weight pointers and their TMA descriptors: rebuild them with the next launch
    c->has_tc_buffers = false; c->has_x3_buffers = false; c->fused_ready = false; c->x3_ready = false;
    c->F = F; c->Q = Q;
    int rc = pack_weights(c, kernels, biases, in_dims, out_dims);
    if (rc) return rc;
    if ((rc = tc_pack_weights(c))) return rc;
    if ((rc = x3_pack_weights(c))) return rc;
    // widths the split-precision kernels do not tile run their Dense layers on the CUDA cores instead (same fp32 results)
    if (c->precision == DSAT_F32_TC && !x3_supported(c)) c->precision = DSAT_F32;
    c->has_model = true;
    return DSAT_OK;
}

int dsat_set_graph(dsat_ctx* c, int n_vars, int n_clauses, int nnz, const int32_t* cl_rowptr, const int32_t* cl_lit,
                   const int32_t* lit_rowptr, const int32_t* lit_clause, int n_graphs, const int32_t* var_seg,
                   const int32_t* clause_seg, int n_chains, int group_graphs) {
    if (!c) return DSAT_ERR_ARG;
    // everything is validated before the context is touched: a rejected call leaves the previous graph bound
    CK_ARG(c, n_vars > 0 && n_clauses > 0 && nnz >= 0 && n_graphs > 0 && n_chains > 0,
           "dsat_set_graph: bad sizes (a formula needs at least one variable and one clause)");
    CK_ARG(c, cl_rowptr && lit_rowptr && var_seg && clause_seg && (nnz == 0 || (cl_lit && lit_clause)),
           "dsat_set_graph: null index array");
    CK_ARG(c, cl_rowptr[0] == 0 && cl_rowptr[n_clauses] == nnz && lit_rowptr[0] == 0 && lit_rowptr[2 * n_vars] == nnz,
           "dsat_set_graph: row pointers do not cover nnz");
    for (int j = 0; j < n_clauses; ++j)
        CK_ARG(c, cl_rowptr[j + 1] >= cl_rowptr[j], "dsat_set_graph: clause row pointers are not monotone");
    for (int l = 0; l < 2 * n_vars; ++l)
        CK_ARG(c, lit_rowptr[l + 1] >= lit_rowptr[l], "dsat_set_graph: literal row pointers are not monotone");
    CK_ARG(c, var_seg[0] == 0 && var_seg[n_graphs] == n_vars && clause_seg[0] == 0 && clause_seg[n_graphs] == n_clauses,
           "dsat_set_graph: graph segments do not cover the unit");
    {   // the CSR (clause -> literal codes) and the CSC (literal code -> clauses) must describe the same multiset of edges
        std::vector<int> deg(2 * (size_t)n_vars, 0);
        for (int e = 0; e < nnz; ++e) {
            CK_ARG(c, cl_lit[e] >= 0 && cl_lit[e] < 2 * n_vars, "dsat_set_graph: literal code out of range");
            CK_ARG(c, lit_clause[e] >= 0 && lit_clause[e] < n_clauses, "dsat_set_graph: clause id out of range");
            deg[cl_lit[e]]++;
        }
        for (int l = 0; l < 2 * n_vars; ++l)
            CK_ARG(c, deg[l] == lit_rowptr[l + 1] - lit_rowptr[l], "dsat_set_graph: CSR and CSC disagree on a literal's degree");
    }
    int max_graph_vars = 0, max_graph_clauses = 0;
    for (int g = 0; g < n_graphs; ++g) {
        CK_ARG(c, var_seg[g + 1] > var_seg[g] && clause_seg[g + 1] >= clause_seg[g], "dsat_set_graph: empty or unordered graph segment");
        if (var_seg[g + 1] - var_seg[g] > max_graph_vars) max_graph_vars = var_seg[g + 1] - var_seg[g];
        if (clause_seg[g + 1] - clause_seg[g] > max_graph_clauses) max_graph_clauses = clause_seg[g + 1] - clause_seg[g];
    }
    CK_ARG(c, (long long)n_chains * n_vars < (1ll << 31) - 256 && (long long)n_chains * n_clauses < (1ll << 31) - 256,
           "dsat_set_graph: too many rows for one context; use fewer chains per context");
    CK_CUDA(c, cudaSetDevice(c->device));
    CK_CUDA(c, cudaStreamSynchronize(c->stream));
    // same shape as before (the usual case: the same formula re-bound, or another formula of the same size):
    // keep the activation buffers and their TMA descriptors, only the index arrays are replaced
    const int total_graphs_new = n_graphs * n_chains;
    const int group_new = group_graphs > 0 ? group_graphs : total_graphs_new;
    const bool same_shape = c->has_graph && c->n == n_vars && c->m == n_clauses && c->n_graphs == n_graphs &&
                            c->chains == n_chains && c->words == ceil_div(max_graph_vars, 64) &&
                            c->group_graphs == group_new && !c->has_batches;
    if (!same_shape) release_buffers(c);
    c->generation++;        // the index arrays are re-allocated
    c->has_graph = false;               // set again at the end: an upload that fails half way leaves no graph bound
    c->has_batches = c->has_noise_base = false;
    c->n = n_vars; c->m = n_clauses; c->nnz = nnz; c->n_graphs = n_graphs; c->chains = n_chains;
    c->total_graphs = n_graphs * n_chains;
    c->group_graphs = group_graphs > 0 ? group_graphs : c->total_graphs;
    c->n_groups = ceil_div(c->total_graphs, c->group_graphs);
    c->Nt = (long long)n_chains * n_vars;
    c->Mt = (long long)n_chains * n_clauses;
    c->words = ceil_div(max_graph_vars, 64);
    c->max_graph_vars = max_graph_vars; c->max_graph_clauses = max_graph_clauses;

    std::vector<float> deg_w(2 * n_vars), vdeg_w(n_vars), rev_w(n_clauses > 0 ? n_clauses : 1);
    for (int l = 0; l < 2 * n_vars; ++l) {
        float d = (float)(lit_rowptr[l + 1] - lit_rowptr[l]);
        deg_w[l] = 1.0f / sqrtf(fmaxf(d, 1.0f));
    }
    for (int v = 0; v < n_vars; ++v) {
        float d = (float)(lit_rowptr[2 * v + 2] - lit_rowptr[2 * v]);
        vdeg_w[v] = 1.0f / sqrtf(fmaxf(d, 1.0f));
    }
    for (int j = 0; j < n_clauses; ++j) {
        float d = (float)(cl_rowptr[j + 1] - cl_rowptr[j]);
        rev_w[j] = 1.0f / sqrtf(fmaxf(d, 1.0f));
    }
    auto up_i = [&](DevBuf<int>& b, const int32_t* h, size_t cnt) -> cudaError_t {
        cudaError_t e = b.alloc(cnt > 0 ? cnt : 1);
        if (e != cudaSuccess || cnt == 0) return e;
        return dsat_memcpy_sync(b.p, h, cnt * sizeof(int), cudaMemcpyHostToDevice);
    };
    auto up_f = [&](DevBuf<float>& b, const std::vector<float>& h) -> cudaError_t {
        cudaError_t e = b.alloc(h.size());
        if (e != cudaSuccess) return e;
        return dsat_memcpy_sync(b.p, h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice);
    };
    CK_CUDA(c, up_i(c->cl_rowptr, cl_rowptr, n_clauses + 1));
    CK_CUDA(c, up_i(c->cl_lit, cl_lit, nnz));
    CK_CUDA(c, up_i(c->lit_rowptr, lit_rowptr, 2 * n_vars + 1));
    CK_CUDA(c, up_i(c->lit_clause, lit_clause, nnz));
    CK_CUDA(c, up_i(c->var_seg, var_seg, n_graphs + 1));
    CK_CUDA(c, up_i(c->clause_seg, clause_seg, n_graphs + 1));
    CK_CUDA(c, up_f(c->deg_w, deg_w));
    CK_CUDA(c, up_f(c->vdeg_w, vdeg_w));
    {
        std::vector<int> vord(n_vars > 0 ? n_vars : 1, 0);
        for (int v = 0; v < n_vars; ++v) vord[v] = v;
        std::stable_sort(vord.begin(), vord.begin() + n_vars, [&](int a, int b) {
            return lit_rowptr[2 * a + 2] - lit_rowptr[2 * a] > lit_rowptr[2 * b + 2] - lit_rowptr[2 * b];
        });
        CK_CUDA(c, up_i(c->var_order, vord.data(), (size_t)n_vars));
        // 16-bit adjacency blocks (sections padded to 16 bytes)
        c->cl_idx16_vecs = c->lit_idx16_vecs = 0;
        if (nnz < 65536 && 2 * n_vars < 65536 && n_clauses < 65536 && n_vars > 0 && n_clauses > 0) {
            auto pad8 = [](size_t x) { return (x + 7) / 8 * 8; };
            std::vector<unsigned short> blk;
            auto put = [&](const int* src, size_t cnt) {
                const size_t at = blk.size();
                blk.resize(at + pad8(cnt), 0);
                for (size_t i = 0; i < cnt; ++i) blk[at + i] = (unsigned short)src[i];
                return (int)at;
            };
            auto upload = [&](DevBuf<unsigned short>& dst) -> cudaError_t {
                cudaError_t e = dst.alloc(blk.size());
                if (e != cudaSuccess) return e;
                return dsat_memcpy_sync(dst.p, blk.data(), blk.size() * sizeof(unsigned short), cudaMemcpyHostToDevice);
            };
            put(cl_rowptr, (size_t)n_clauses + 1);
            c->cl_col_off = put(cl_lit, (size_t)nnz);
            CK_CUDA(c, upload(c->cl_idx16));
            c->cl_idx16_vecs = (int)(blk.size() / 8);
            blk.clear();
            put(lit_rowptr, (size_t)2 * n_vars + 1);
            c->lit_col_off = put(lit_clause, (size_t)nnz);
            c->lit_ord_off = put(vord.data(), (size_t)n_vars);
            CK_CUDA(c, upload(c->lit_idx16));
            c->lit_idx16_vecs = (int)(blk.size() / 8);
        }
    }
    CK_CUDA(c, up_f(c->rev_w, rev_w));
    // host copy for the row descriptors of the standalone segment sums, which are built by the first dsat_spmm call on this
    // graph (ensure_spmm_desc): the model path never pays for them
    c->h_cl_rowptr.assign(cl_rowptr, cl_rowptr + n_clauses + 1);
    c->h_cl_lit.assign(cl_lit, cl_lit + nnz);
    c->h_lit_rowptr.assign(lit_rowptr, lit_rowptr + 2 * n_vars + 1);
    c->h_lit_clause.assign(lit_clause, lit_clause + nnz);
    c->h_deg_w = deg_w;
    c->h_rev_w = rev_w;
    c->spmm_desc_ready = false;
    c->has_graph = true;
    return DSAT_OK;
}

int dsat_words_per_graph(const dsat_ctx* c) { return c ? c->words : 0; }

int dsat_set_batches(dsat_ctx* c, int n_groups, const int32_t* group_seg, const uint64_t* noise_base) {
    if (!c) return DSAT_ERR_ARG;
    CK_ARG(c, c->has_graph, "dsat_set_batches: bind a graph first");
    const int G = c->total_graphs;
    CK_ARG(c, n_groups > 0 && n_groups <= G && group_seg, "dsat_set_batches: bad group count or null group_seg");
    CK_ARG(c, group_seg[0] == 0 && group_seg[n_groups] == G, "dsat_set_batches: groups do not cover the graphs of the context");
    for (int i = 0; i < n_groups; ++i)
        CK_ARG(c, group_seg[i + 1] > group_seg[i], "dsat_set_batches: empty or unordered group");
    // host copies of the unit's graph segments: row range of every graph
    std::vector<int> var_seg(c->n_graphs + 1);
    CK_CUDA(c, cudaSetDevice(c->device));
    CK_CUDA(c, cudaStreamSynchronize(c->stream));
    CK_CUDA(c, dsat_memcpy_sync(var_seg.data(), c->var_seg.p, var_seg.size() * sizeof(int), cudaMemcpyDeviceToHost));
    auto row0 = [&](int gi) { return (uint64_t)(gi / c->n_graphs) * (uint64_t)c->n + (uint64_t)var_seg[gi % c->n_graphs]; };
    if (noise_base)
        for (int gi = 0; gi < G; ++gi) {
            const uint64_t vars = (uint64_t)(var_seg[gi % c->n_graphs + 1] - var_seg[gi % c->n_graphs]);
            CK_ARG(c, noise_base[gi] <= UINT64_MAX - vars, "dsat_set_batches: a graph's Philox elements would wrap around 2^64");
        }
    std::vector<int> group_of(G);
    for (int i = 0; i < n_groups; ++i)
        for (int gi = group_seg[i]; gi < group_seg[i + 1]; ++gi) group_of[gi] = i;
    // everything validated: commit (every table a captured step reads may move, so the step is captured again)
    c->generation++;
    c->has_batches = c->has_noise_base = false;
    CK_CUDA(c, c->batch_seg.alloc(n_groups + 1));
    CK_CUDA(c, dsat_memcpy_sync(c->batch_seg.p, group_seg, (n_groups + 1) * sizeof(int), cudaMemcpyHostToDevice));
    CK_CUDA(c, c->graph_group.alloc(G));
    CK_CUDA(c, dsat_memcpy_sync(c->graph_group.p, group_of.data(), G * sizeof(int), cudaMemcpyHostToDevice));
    if (noise_base) {
        std::vector<int> rg((size_t)c->Nt);
        std::vector<unsigned long long> e0(G);
        for (int gi = 0; gi < G; ++gi) {
            const uint64_t r0 = row0(gi), r1 = r0 + (uint64_t)(var_seg[gi % c->n_graphs + 1] - var_seg[gi % c->n_graphs]);
            for (uint64_t r = r0; r < r1; ++r) rg[r] = gi;
            e0[gi] = noise_base[gi] - r0;           // element of row r = e0 + r (mod 2^64)
        }
        CK_CUDA(c, c->row_graph.alloc(rg.size()));
        CK_CUDA(c, dsat_memcpy_sync(c->row_graph.p, rg.data(), rg.size() * sizeof(int), cudaMemcpyHostToDevice));
        CK_CUDA(c, c->graph_elem0.alloc(G));
        CK_CUDA(c, dsat_memcpy_sync(c->graph_elem0.p, e0.data(), G * sizeof(unsigned long long), cudaMemcpyHostToDevice));
    }
    // per-group bookkeeping is sized by the group count
    c->n_groups = n_groups;
    if (c->has_buffers) {
        CK_CUDA(c, c->done.alloc(n_groups));
        CK_CUDA(c, c->steps_taken.alloc(n_groups));
        CK_CUDA(c, c->rounds_run.alloc(n_groups));
        CK_CUDA(c, c->loss_sum.alloc(n_groups));
    }
    c->has_batches = true;
    c->has_noise_base = noise_base != nullptr;
    return DSAT_OK;
}

// ---------------------------------------------------------------------------------- graph build (host)
int dsat_graph_build(int n_vars, int n_clauses, long long nnz, const int32_t* lens, const int32_t* flat, int32_t* cl_rowptr,
                     int32_t* cl_lit, int32_t* lit_rowptr, int32_t* lit_clause, int32_t* bad_clause) {
    if (bad_clause) *bad_clause = -1;
    if (n_vars < 0 || n_clauses < 0 || nnz < 0 || nnz >= (1ll << 31) || !cl_rowptr || !lit_rowptr ||
        (n_clauses > 0 && !lens) || (nnz > 0 && (!flat || !cl_lit || !lit_clause)))
        return DSAT_ERR_ARG;
    long long total = 0;
    for (int j = 0; j < n_clauses; ++j) {
        if (lens[j] < 0) return DSAT_ERR_ARG;
        total += lens[j];
    }
    if (total != nnz) return DSAT_ERR_ARG;
    const long long rc = dsat::graph_build_host(n_vars, n_clauses, lens, flat, cl_rowptr, cl_lit, lit_rowptr, lit_clause);
    if (rc < 0) {
        if (bad_clause) *bad_clause = (int32_t)(-rc - 1);
        return DSAT_ERR_ARG;
    }
    return DSAT_OK;
}

// ----------------------------------------------------------------------------------- model call
int dsat_model_call(dsat_ctx* c, float noise_scale, const float* noisy_num, const int32_t* labels,
                    const float* normals, int rounds, uint64_t seed, uint64_t chain_offset, float* prediction_out,
                    int32_t* steps_taken, float* loss) {
    if (!c) return DSAT_ERR_ARG;
    CK_ARG(c, noisy_num && prediction_out && rounds >= 0, "dsat_model_call: null buffer or negative rounds");
    CK_ARG(c, !c->has_noise_base || chain_offset == 0, "dsat_model_call: chain_offset must be 0 while noise bases are bound");
    CK_CUDA(c, cudaSetDevice(c->device));
    int rc = ensure_active_buffers(c);
    if (rc) return rc;
    const size_t Nt = (size_t)c->Nt;
    CK_CUDA(c, c->inj_noisy.alloc(Nt * 2));
    CK_CUDA(c, c->inj_noisy.upload(noisy_num, Nt * 2, c->stream));
    if (labels) {
        CK_CUDA(c, c->inj_labels.alloc(Nt));
        CK_CUDA(c, c->inj_labels.upload(labels, Nt, c->stream));
    }
    if (normals && rounds > 0) {
        CK_CUDA(c, c->inj_normals.alloc(Nt * 4 * rounds));
        CK_CUDA(c, c->inj_normals.upload(normals, Nt * 4 * rounds, c->stream));
    }
    const NoiseSource ns = noise_source(c, seed, chain_offset * (uint64_t)c->n, 0u);
    if ((rc = begin_call(c, noise_scale, c->inj_noisy.p, nullptr, labels ? c->inj_labels.p : nullptr, false, ns))) return rc;
    const LossScalars ls = loss_scalars(noise_scale);
    for (int r = 0; r < rounds; ++r)
        if ((rc = run_round(c, r, normals ? c->inj_normals.p + (size_t)r * Nt * 4 : nullptr, ns, ls))) return rc;
    CK_CUDA(c, cudaMemcpyAsync(prediction_out, c->OUT.p, Nt * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    std::vector<float> lsum(c->n_groups);
    std::vector<int> rrun(c->n_groups);
    if (steps_taken)
        CK_CUDA(c, cudaMemcpyAsync(steps_taken, c->steps_taken.p, c->n_groups * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CK_CUDA(c, cudaMemcpyAsync(lsum.data(), c->loss_sum.p, c->n_groups * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    CK_CUDA(c, cudaMemcpyAsync(rrun.data(), c->rounds_run.p, c->n_groups * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CK_CUDA(c, cudaStreamSynchronize(c->stream));
    if (loss)
        for (int g = 0; g < c->n_groups; ++g) loss[g] = rrun[g] > 0 ? lsum[g] / (float)rrun[g] : 0.f;
    return DSAT_OK;
}

// --------------------------------------------------------------------------------------- sampler
// scalars of denoising step t of n_steps, computed on the host exactly as the by-value launch path does
static StepParams step_params(int t, int n_steps, uint64_t seed, uint64_t element_offset) {
    StepParams sp;
    const double ns_d = 1.0 - (double)t / (double)n_steps;       // Python float (DiffusionSampler.py:106)
    sp.noise_scale = (float)ns_d;
    const LossScalars ls = loss_scalars(sp.noise_scale);
    sp.t = ls.t; sp.ts = ls.ts; sp.norm_plus = ls.norm_plus;
    // posterior scalars (reference DiffusionSampler.py:30-33): pow in fp32, max() in Python floats
    const float t1 = powf(sp.noise_scale, 0.5f);
    const double t_prev = ns_d - 1.0 / (double)n_steps;
    const float t2 = powf((float)(t_prev > 0.0 ? t_prev : 0.0), 0.5f);
    const float alpha = (1.0f - t1) / (1.0f - t2);
    sp.t1 = t1;
    sp.one_minus_alpha = 1.0f - alpha;
    sp.step = (unsigned)t; sp.pad_ = 0;
    sp.seed = seed; sp.element_offset = element_offset;
    return sp;
}

// launches of one denoising step; with sp_tab the step's scalars are read on the device (graph capture)
static int enqueue_step(dsat_ctx* c, const StepParams& sp, int n_rounds, const float* uniforms_dev, const int* labels_dev,
                        const float* normals_dev, const StepParams* sp_tab, const int* sp_cur) {
    const UnitGraphDev g = graph_view(c);
    const NoiseSource ns = noise_source(c, sp.seed, sp.element_offset, sp.step);
    int rc = begin_call(c, sp.noise_scale, nullptr, uniforms_dev, labels_dev, true, ns, sp_tab, sp_cur);
    if (rc) return rc;
    LossScalars ls; ls.t = sp.t; ls.ts = sp.ts; ls.norm_plus = sp.norm_plus;
    for (int r = 0; r < n_rounds; ++r) {
        const float* nrm = normals_dev ? normals_dev + (size_t)r * c->Nt * 4 : nullptr;
        if ((rc = run_round(c, r, nrm, ns, ls, sp_tab, sp_cur))) return rc;
    }
    PosteriorScalars ps;
    ps.t1 = sp.t1; ps.one_minus_alpha = sp.one_minus_alpha;
    step_end_kernel<<<c->total_graphs, 128, 0, c->stream>>>(g, c->total_graphs, c->OUT.p, c->X.p, ps, (int)sp.step,
                                                             c->LAST.p, c->LATCH.p, c->latch_step.p, c->sat_now.p, sp_tab, sp_cur);
    LAUNCHED(c);
    if (sp_tab) {
        step_advance_kernel<<<1, 1, 0, c->stream>>>(const_cast<int*>(sp_cur));
        LAUNCHED(c);
    }
    return DSAT_OK;
}

static int sample_enqueue_impl(dsat_ctx* c, int n_steps, int n_rounds, uint64_t seed, uint64_t chain_offset,
                               const float* uniforms_dev, const int* labels_dev, const float* normals_dev) {
    int rc = ensure_active_buffers(c);
    if (rc) return rc;
    const long long Nt = c->Nt;
    const UnitGraphDev g = graph_view(c);
    {   // x = 0.5 (reference DiffusionSampler.py:86)
        const long long rows4 = (2 * Nt + 3) / 4;      // X is allocated with one spare float2
        fill_cols_kernel<<<(unsigned)((rows4 + 255) / 256), 256, 0, c->stream>>>(
            reinterpret_cast<float*>(c->X.p), 4, rows4, 1, 0.5f);
        LAUNCHED(c);
    }
    CK_CUDA(c, cudaMemsetAsync(c->latch_step.p, 0xff, c->latch_step.count * sizeof(int), c->stream));
    CK_CUDA(c, cudaMemsetAsync(c->sat_any.p, 0, c->sat_any.count, c->stream));
    const uint64_t element_offset = chain_offset * (uint64_t)c->n;
    const bool injected = uniforms_dev || labels_dev || normals_dev;
    if (!injected && !c->profiling) {
        // One denoising step is captured once and replayed n_steps times: the ~12 launches per round are issued by the
        // graph executor back to back instead of one cudaLaunchKernel each (small formulas are launch-bound: 12.5 k launches
        // per run).  Everything that differs between steps lives in step_tab[*step_cur].
        c->step_tab_host.resize(n_steps);
        for (int t = 0; t < n_steps; ++t) c->step_tab_host[t] = step_params(t, n_steps, seed, element_offset);
        if (c->step_tab.count < (size_t)n_steps) { CK_CUDA(c, c->step_tab.alloc(n_steps)); c->generation++; }
        if (!c->step_cur.p) { CK_CUDA(c, c->step_cur.alloc(1)); c->generation++; }
        CK_CUDA(c, cudaMemcpyAsync(c->step_tab.p, c->step_tab_host.data(), n_steps * sizeof(StepParams), cudaMemcpyHostToDevice, c->stream));
        CK_CUDA(c, cudaMemsetAsync(c->step_cur.p, 0, sizeof(int), c->stream));
        if (!c->step_graph || c->step_graph_generation != c->generation || c->step_graph_rounds != n_rounds ||
            c->step_graph_precision != c->precision) {
            drop_step_graph(c);
            cudaGraph_t graph = nullptr;
            CK_CUDA(c, cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
            const long long launches_before = c->launches;
            rc = enqueue_step(c, c->step_tab_host[0], n_rounds, nullptr, nullptr, nullptr, c->step_tab.p, c->step_cur.p);
            const cudaError_t ce = cudaStreamEndCapture(c->stream, &graph);
            c->step_launches = (int)(c->launches - launches_before);
            c->launches = launches_before;
            if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
            CK_CUDA(c, ce);
            const cudaError_t ie = cudaGraphInstantiate(&c->step_graph, graph, 0);
            cudaGraphDestroy(graph);
            CK_CUDA(c, ie);
            c->step_graph_generation = c->generation;
            c->step_graph_rounds = n_rounds;
            c->step_graph_precision = c->precision;
        }
        for (int t = 0; t < n_steps; ++t) {
            CK_CUDA(c, cudaGraphLaunch(c->step_graph, c->stream));
            c->launches += c->step_launches;
        }
    } else {
        for (int t = 0; t < n_steps; ++t) {
            const StepParams sp = step_params(t, n_steps, seed, element_offset);
            if ((rc = enqueue_step(c, sp, n_rounds, uniforms_dev ? uniforms_dev + (size_t)t * Nt : nullptr,
                                   labels_dev ? labels_dev + (size_t)t * Nt : nullptr,
                                   normals_dev ? normals_dev + (size_t)t * n_rounds * Nt * 4 : nullptr, nullptr, nullptr)))
                return rc;
        }
    }
    pack_assignments_kernel<<<c->total_graphs, 128, 0, c->stream>>>(g, c->total_graphs, c->words, c->LAST.p, c->LATCH.p,
                                                                     c->latch_step.p, c->packed.p, c->is_sat.p, c->FINAL.p);
    LAUNCHED(c);
    return DSAT_OK;
}

int dsat_sample_enqueue(dsat_ctx* c, int n_steps, int n_rounds, uint64_t seed, uint64_t chain_offset) {
    if (!c) return DSAT_ERR_ARG;
    CK_ARG(c, n_steps > 0 && n_rounds >= 0, "dsat_sample: bad step or round count");
    CK_ARG(c, !c->has_noise_base || chain_offset == 0, "dsat_sample: chain_offset must be 0 while noise bases are bound");
    CK_CUDA(c, cudaSetDevice(c->device));
    return sample_enqueue_impl(c, n_steps, n_rounds, seed, chain_offset, nullptr, nullptr, nullptr);
}

int dsat_sample_fetch(dsat_ctx* c, uint64_t* packed, uint8_t* is_sat, int32_t* latch_step, uint8_t* sat_any_step) {
    if (!c) return DSAT_ERR_ARG;
    CK_ARG(c, c->has_buffers, "dsat_sample_fetch: nothing was sampled");
    CK_CUDA(c, cudaSetDevice(c->device));
    const size_t G = (size_t)c->total_graphs;
    if (packed)
        CK_CUDA(c, cudaMemcpyAsync(packed, c->packed.p, G * c->words * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
    if (is_sat) CK_CUDA(c, cudaMemcpyAsync(is_sat, c->is_sat.p, G, cudaMemcpyDeviceToHost, c->stream));
    if (latch_step)
        CK_CUDA(c, cudaMemcpyAsync(latch_step, c->latch_step.p, G * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CK_CUDA(c, cudaStreamSynchronize(c->stream));
    if (sat_any_step) {
        // cum_accuracy of diffusion(): a graph counts once any step's rounded prediction satisfied it,
        // which is exactly "latched" (reference DiffusionSampler.py:119-130,154-170)
        std::vector<int> ls(G);
        CK_CUDA(c, dsat_memcpy_sync(ls.data(), c->latch_step.p, G * sizeof(int), cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < G; ++i) sat_any_step[i] = ls[i] >= 0;
    }
    return DSAT_OK;
}

int dsat_sample(dsat_ctx* c, int n_steps, int n_rounds, uint64_t seed, uint64_t chain_offset, const float* uniforms,
                const int32_t* labels, const float* normals, uint64_t* packed, uint8_t* is_sat, int32_t* latch_step,
                uint8_t* sat_any_step) {
    if (!c) return DSAT_ERR_ARG;
    CK_ARG(c, n_steps > 0 && n_rounds >= 0, "dsat_sample: bad step or round count");
    CK_ARG(c, !c->has_noise_base || chain_offset == 0, "dsat_sample: chain_offset must be 0 while noise bases are bound");
    CK_CUDA(c, cudaSetDevice(c->device));
    int rc = ensure_active_buffers(c);
    if (rc) return rc;
    const size_t Nt = (size_t)c->Nt;
    if (uniforms) {
        CK_CUDA(c, c->inj_uniforms.alloc(Nt * n_steps));
        CK_CUDA(c, c->inj_uniforms.upload(uniforms, Nt * n_steps, c->stream));
    }
    if (labels) {
        CK_CUDA(c, c->inj_labels.alloc(Nt * n_steps));
        CK_CUDA(c, c->inj_labels.upload(labels, Nt * n_steps, c->stream));
    }
    if (normals && n_rounds > 0) {
        CK_CUDA(c, c->inj_normals.alloc(Nt * 4 * n_rounds * n_steps));
        CK_CUDA(c, c->inj_normals.upload(normals, Nt * 4 * n_rounds * n_steps, c->stream));
    }
    rc = sample_enqueue_impl(c, n_steps, n_rounds, seed, chain_offset, uniforms ? c->inj_uniforms.p : nullptr,
                             labels ? c->inj_labels.p : nullptr, (normals && n_rounds > 0) ? c->inj_normals.p : nullptr);
    if (rc) return rc;
    return dsat_sample_fetch(c, packed, is_sat, latch_step, sat_any_step);
}

// ------------------------------------------------------------------------------------- histogram
int dsat_hist_reduce(dsat_ctx* c, int chain_limit, uint64_t* keys_out, int64_t* counts_out, int capacity, int32_t* n_unique,
                     int32_t* n_sat) {
    if (!c) return DSAT_ERR_ARG;
    CK_ARG(c, c->has_buffers, "dsat_hist_reduce: nothing was sampled");
    CK_ARG(c, n_unique && capacity >= 0 && (capacity == 0 || (keys_out && counts_out)), "dsat_hist_reduce: null output");
    CK_CUDA(c, cudaSetDevice(c->device));
    const int G = c->total_graphs, words = c->words;
    const int limit = chain_limit > 0 && chain_limit < G ? chain_limit : G;
    const int n_pad = hist::next_pow2(G < 2 ? 2 : G);
    if (c->hist_idx.count < (size_t)n_pad) {
        CK_CUDA(c, c->hist_idx.alloc(n_pad));
        CK_CUDA(c, c->hist_run.alloc(n_pad));
        CK_CUDA(c, c->hist_totals.alloc(2));
        CK_CUDA(c, c->hist_keys.alloc((size_t)G * words));
        CK_CUDA(c, c->hist_counts.alloc(G));
    }
    CK_CUDA(c, hist::enqueue(c->stream, G, limit, words, c->packed.p, c->is_sat.p, c->hist_idx.p, c->hist_run.p, c->hist_keys.p,
                             c->hist_counts.p, c->hist_totals.p, &c->launches));
    int totals[2] = {0, 0};
    CK_CUDA(c, cudaMemcpyAsync(totals, c->hist_totals.p, sizeof(totals), cudaMemcpyDeviceToHost, c->stream));
    CK_CUDA(c, cudaStreamSynchronize(c->stream));
    *n_unique = totals[0];
    if (n_sat) *n_sat = totals[1];
    const int k = totals[0] < capacity ? totals[0] : capacity;
    if (k > 0) {
        CK_CUDA(c, cudaMemcpyAsync(keys_out, c->hist_keys.p, (size_t)k * words * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
        CK_CUDA(c, cudaMemcpyAsync(counts_out, c->hist_counts.p, (size_t)k * sizeof(int64_t), cudaMemcpyDeviceToHost, c->stream));
        CK_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    CK_ARG(c, totals[0] <= capacity, "dsat_hist_reduce: capacity too small (n_unique holds the required size)");
    return DSAT_OK;
}

int dsat_hist_reduce_segments(dsat_ctx* c, int n_segments, const int32_t* graph_seg, const int32_t* limit, uint64_t* keys_out,
                              int64_t* counts_out, int capacity, int32_t* seg_runs, int32_t* n_sat) {
    if (!c) return DSAT_ERR_ARG;
    CK_ARG(c, c->has_buffers, "dsat_hist_reduce_segments: nothing was sampled");
    const int G = c->total_graphs, words = c->words;
    CK_ARG(c, n_segments > 0 && graph_seg && limit && seg_runs, "dsat_hist_reduce_segments: bad segment count or null array");
    CK_ARG(c, capacity >= 0 && (capacity == 0 || (keys_out && counts_out)), "dsat_hist_reduce_segments: null output");
    CK_ARG(c, graph_seg[0] >= 0 && graph_seg[n_segments] <= G, "dsat_hist_reduce_segments: segments outside the context's graphs");
    for (int s = 0; s < n_segments; ++s) {
        CK_ARG(c, graph_seg[s + 1] >= graph_seg[s], "dsat_hist_reduce_segments: unordered segments");
        CK_ARG(c, limit[s] >= 0, "dsat_hist_reduce_segments: negative limit");
    }
    CK_CUDA(c, cudaSetDevice(c->device));
    std::vector<int> seg(G, -1);            // segment of each counted chain index (monotone), -1 outside every limit
    for (int s = 0; s < n_segments; ++s) {
        const int end = graph_seg[s] + std::min(limit[s], graph_seg[s + 1] - graph_seg[s]);
        for (int gi = graph_seg[s]; gi < end; ++gi) seg[gi] = s;
    }
    const int n_pad = hist::next_pow2(G < 2 ? 2 : G);
    CK_CUDA(c, c->hist_idx.alloc(n_pad));
    CK_CUDA(c, c->hist_run.alloc(n_pad));
    CK_CUDA(c, c->hist_totals.alloc(2));
    CK_CUDA(c, c->hist_keys.alloc((size_t)G * words));
    CK_CUDA(c, c->hist_counts.alloc(G));
    CK_CUDA(c, c->hist_seg.alloc(G));
    CK_CUDA(c, c->hist_run_seg.alloc(G));
    CK_CUDA(c, cudaMemcpyAsync(c->hist_seg.p, seg.data(), G * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    CK_CUDA(c, hist::enqueue(c->stream, G, G, words, c->packed.p, c->is_sat.p, c->hist_idx.p, c->hist_run.p, c->hist_keys.p,
                             c->hist_counts.p, c->hist_totals.p, &c->launches, c->hist_seg.p, c->hist_run_seg.p));
    int totals[2] = {0, 0};
    CK_CUDA(c, cudaMemcpyAsync(totals, c->hist_totals.p, sizeof(totals), cudaMemcpyDeviceToHost, c->stream));
    CK_CUDA(c, cudaStreamSynchronize(c->stream));      // (also keeps `seg` alive until its upload has run)
    const int K = totals[0];
    std::vector<int> run_seg(K);
    if (K > 0) CK_CUDA(c, dsat_memcpy_sync(run_seg.data(), c->hist_run_seg.p, K * sizeof(int), cudaMemcpyDeviceToHost));
    for (int s = 0, u = 0; s <= n_segments; ++s) {      // runs come segment by segment
        while (u < K && run_seg[u] < s) ++u;
        seg_runs[s] = u;
    }
    if (n_sat) *n_sat = totals[1];
    const int k = K < capacity ? K : capacity;
    if (k > 0) {
        CK_CUDA(c, cudaMemcpyAsync(keys_out, c->hist_keys.p, (size_t)k * words * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
        CK_CUDA(c, cudaMemcpyAsync(counts_out, c->hist_counts.p, (size_t)k * sizeof(int64_t), cudaMemcpyDeviceToHost, c->stream));
        CK_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    CK_ARG(c, K <= capacity, "dsat_hist_reduce_segments: capacity too small (seg_runs[n_segments] holds the required size)");
    return DSAT_OK;
}

// ------------------------------------------------------------------------------------------ SpMM
// The spmm_rows_kernel instantiation of each (direction, dtype, row bytes), measured on the n = 10000 sweep
// (profiles/r2_spmm_variants.txt).  Clause side: registers for the gathers (no spills) and, for fp32 rows of >= 512 bytes,
// the prefetched descriptor; bf16 rows of >= 256 bytes run with half the lanes per row (twice the gathers in flight per
// warp).  Literal side: the twelve-entry descriptor (desc4) for rows of <= 256 bytes, the plain 32-register kernel for
// 512-byte fp32 rows, half the lanes for 512-byte bf16 rows.
using SpmmKernel = void (*)(const int4*, const int*, int, int, int, const void*, void*);
struct SpmmPlan { SpmmKernel kernel; bool desc4; bool half_lanes; };
static SpmmPlan spmm_plan(int direction, bool bf16, int row_bytes) {
    if (direction == 0) {
        if (bf16) {
            if (row_bytes == 128) return {spmm_rows_kernel<128, true, 6>, false, false};
            if (row_bytes == 256) return {spmm_rows_kernel<256, true, 4, false, 2, 8>, false, true};
            return {spmm_rows_kernel<512, true, 4, false, 2, 16>, false, true};
        }
        if (row_bytes == 256) return {spmm_rows_kernel<256, false, 8>, false, false};
        if (row_bytes == 512) return {spmm_rows_kernel<512, false, 5, true>, false, false};
        return {spmm_rows_kernel<1024, false, 4, true>, false, false};
    }
    if (bf16) {
        if (row_bytes == 128) return {spmm_rows_kernel<128, true, 5, false, 4>, true, false};
        if (row_bytes == 256) return {spmm_rows_kernel<256, true, 5, false, 4>, true, false};
        return {spmm_rows_kernel<512, true, 4, false, 2, 16>, false, true};
    }
    if (row_bytes == 256) return {spmm_rows_kernel<256, false, 6, false, 4>, true, false};
    if (row_bytes == 512) return {spmm_rows_kernel<512, false, 8>, false, false};
    return {spmm_rows_kernel<1024, false, 5>, false, false};
}

// Row descriptors of the standalone segment sums (dsat_spmm.cuh), built on first use after dsat_set_graph.
// Processing order: rows of equal length are grouped (the rows sharing a warp pass then run the same number of steps), and
// inside a length rows that share their first gathered row become neighbours, so the warps of one CTA hit L1; a row's
// {index, length, scale, first entry} and its first 4 * (dw - 1) gathered rows are packed into dw int4.
static int ensure_spmm_desc(dsat_ctx* c) {
    if (c->spmm_desc_ready) return DSAT_OK;
    auto pack = [&](int rows, const int* rowptr, const int* col, const std::vector<float>& scale, int none, int dw,
                    DevBuf<int>& dst) -> cudaError_t {
        std::vector<int> ord(rows > 0 ? rows : 1, 0), key(rows > 0 ? rows : 1, 0);
        for (int j = 0; j < rows; ++j) {
            ord[j] = j;
            int mn = none;
            for (int e = rowptr[j]; e < rowptr[j + 1]; ++e) mn = col[e] < mn ? col[e] : mn;
            key[j] = mn;
        }
        std::stable_sort(ord.begin(), ord.begin() + rows, [&](int a, int b) {
            const int la = rowptr[a + 1] - rowptr[a], lb = rowptr[b + 1] - rowptr[b];
            return la != lb ? la > lb : key[a] < key[b];
        });
        const size_t w = 4 * (size_t)dw;
        std::vector<int> desc(w * (size_t)(rows > 0 ? rows : 1), 0);
        for (int p = 0; p < rows; ++p) {
            const int j = ord[p], len = rowptr[j + 1] - rowptr[j];
            int bits;
            memcpy(&bits, &scale[j], sizeof(int));
            int* d = &desc[w * (size_t)p];
            d[0] = j; d[1] = len; d[2] = bits; d[3] = rowptr[j];
            for (int k = 0; k < 4 * (dw - 1); ++k) d[4 + k] = k < len ? col[rowptr[j] + k] : -1;
        }
        cudaError_t e = dst.alloc(desc.size());
        if (e != cudaSuccess) return e;
        return dsat_memcpy_sync(dst.p, desc.data(), desc.size() * sizeof(int), cudaMemcpyHostToDevice);
    };
    const int* no_col = nullptr;
    const int* cl_col = c->h_cl_lit.empty() ? no_col : c->h_cl_lit.data();
    const int* lit_col = c->h_lit_clause.empty() ? no_col : c->h_lit_clause.data();
    CK_CUDA(c, pack(c->m, c->h_cl_rowptr.data(), cl_col, c->h_rev_w, 2 * c->n, SPMM_DW_CLAUSE, c->cl_desc));
    CK_CUDA(c, pack(2 * c->n, c->h_lit_rowptr.data(), lit_col, c->h_deg_w, c->m, 2, c->lit_desc));
    CK_CUDA(c, pack(2 * c->n, c->h_lit_rowptr.data(), lit_col, c->h_deg_w, c->m, 4, c->lit_desc4));
    c->spmm_desc_ready = true;
    return DSAT_OK;
}

int dsat_spmm(dsat_ctx* c, int direction, const void* x_dev, void* y_dev, int feat, int dtype, int chains) {
    if (!c) return DSAT_ERR_ARG;
    CK_ARG(c, c->has_graph, "dsat_spmm: graph not set");
    CK_ARG(c, x_dev && y_dev && chains > 0 && (direction == 0 || direction == 1), "dsat_spmm: bad argument");
    CK_ARG(c, dtype == DSAT_F32 || dtype == DSAT_BF16, "dsat_spmm: dtype must be f32 or bf16");
    CK_CUDA(c, cudaSetDevice(c->device));
    if (int rc_desc = ensure_spmm_desc(c)) return rc_desc;
    const int* colidx = direction == 0 ? c->cl_lit.p : c->lit_clause.p;
    const int rows_out = direction == 0 ? c->m : 2 * c->n;
    const int rows_in = direction == 0 ? 2 * c->n : c->m;
    int rc = DSAT_OK;
    const int row_bytes = feat * (dtype == DSAT_BF16 ? 2 : 4);
    if (feat != 64 && feat != 128 && feat != 256) {
        c->err = "feature width must be 64, 128 or 256";
        rc = DSAT_ERR_UNSUPPORTED;
    } else {
        const SpmmPlan plan = spmm_plan(direction, dtype == DSAT_BF16, row_bytes);
        const int4* rowdesc = reinterpret_cast<const int4*>(direction == 0 ? c->cl_desc.p : plan.desc4 ? c->lit_desc4.p : c->lit_desc.p);
        const int rows_per_block = GATHER_WARPS * (row_bytes >= 512 ? 1 : 512 / row_bytes) * (plan.half_lanes ? 2 : 1);
        const int grid = gather_grid(plan.kernel, (long long)chains * rows_out, rows_per_block, c->sm_count);
        plan.kernel<<<grid, GATHER_WARPS * 32, 0, c->stream>>>(rowdesc, colidx, rows_out, rows_in, chains, x_dev, y_dev);
    }
    if (rc) return rc;
    LAUNCHED(c);
    return DSAT_OK;
}

// --------------------------------------------------------------------------------------- profile
// Cycle breakdown of CTA 0 of one whole-MLP kernel (0 query, 1 literal, 2 clause, 3 update, 4 output): 16 counters,
// see dsat_mlp_fused.cuh.  The activations must have been produced by a previous round.
int dsat_profile_fused(dsat_ctx* c, int which, long long* counters16) {
    if (!c || !counters16 || which < 0 || which > 6) return DSAT_ERR_ARG;
    CK_CUDA(c, cudaSetDevice(c->device));
    if (use_x3(c)) {    // the seven x3 launches (query, lit 1, lit 2, lit 3, clause, update, output): 9 counters, see dsat_mlp_x3.cuh
        int rc = ensure_x3_buffers(c);
        if (rc) return rc;
        DevBuf<long long> d;
        CK_CUDA(c, d.alloc(16));
        CK_CUDA(c, cudaMemsetAsync(d.p, 0, 16 * sizeof(long long), c->stream));
        x3::X3Mlp f = c->x3[which];
        f.p.prof = d.p;
        cudaError_t e = x3::launch_x3(f, c->device, c->sm_count, c->stream);
        c->launches++;
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e == cudaSuccess) e = dsat_memcpy_sync(counters16, d.p, 16 * sizeof(long long), cudaMemcpyDeviceToHost);
        d.release();
        CK_CUDA(c, e);
        return DSAT_OK;
    }
    if (which > 4) return DSAT_ERR_ARG;
    int rc = ensure_tc_buffers(c);
    if (rc) return rc;
    CK_ARG(c, c->fused_ready, "fused kernels unavailable");
    DevBuf<long long> d;
    CK_CUDA(c, d.alloc(16));
    CK_CUDA(c, cudaMemsetAsync(d.p, 0, 16 * sizeof(long long), c->stream));
    fm::FusedMlp f = c->fused[which];
    f.p.prof = d.p;
    cudaError_t e = fm::launch_fused(f, c->sm_count, c->stream);
    c->launches++;
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e == cudaSuccess) e = dsat_memcpy_sync(counters16, d.p, 16 * sizeof(long long), cudaMemcpyDeviceToHost);
    d.release();
    CK_CUDA(c, e);
    return DSAT_OK;
}

int dsat_profile_classes(void) { return PROF_CLASSES; }

int dsat_profile_rounds(dsat_ctx* c, int rounds, uint64_t seed, float* class_ms, int32_t* class_launches) {
    if (!c || !class_ms) return DSAT_ERR_ARG;
    CK_ARG(c, rounds > 0, "dsat_profile_rounds: rounds must be positive");
    CK_CUDA(c, cudaSetDevice(c->device));
    int rc = ensure_active_buffers(c);
    if (rc) return rc;
    {   // x = 0.5 so that step_begin can round it
        const long long rows4 = (2 * c->Nt + 3) / 4;
        fill_cols_kernel<<<(unsigned)((rows4 + 255) / 256), 256, 0, c->stream>>>(reinterpret_cast<float*>(c->X.p), 4, rows4, 1, 0.5f);
        LAUNCHED(c);
    }
    NoiseSource ns{seed, 0ull, 0u};
    if ((rc = begin_call(c, 0.5f, nullptr, nullptr, nullptr, true, ns))) return rc;
    const LossScalars ls = loss_scalars(0.5f);
    c->prof_used = 0;
    c->profiling = true;
    for (int r = 0; r < rounds && rc == 0; ++r) rc = run_round(c, r, nullptr, ns, ls);
    c->profiling = false;
    if (rc) return rc;
    CK_CUDA(c, cudaStreamSynchronize(c->stream));
    for (int k = 0; k < PROF_CLASSES; ++k) { class_ms[k] = 0.f; if (class_launches) class_launches[k] = 0; }
    for (size_t i = 0; i + 1 < c->prof_used; ++i) {
        const int cls = c->prof[i].cls;
        if (cls < 0 || cls >= PROF_CLASSES) continue;
        float ms = 0.f;
        CK_CUDA(c, cudaEventElapsedTime(&ms, c->prof[i].ev, c->prof[i + 1].ev));
        class_ms[cls] += ms;
        if (class_launches) class_launches[cls] += 1;
    }
    return DSAT_OK;
}

// ----------------------------------------------------------------------------------------- debug
// Where a debug buffer lives in the active precision.  Its rows and ld are the same in every precision; the storage is
// fp32, bf16, or hi/lo bf16 planes (the lo plane rows*ld elements after the hi plane at p), or none for a buffer the
// precision does not hold (hidden activations that stay on-chip).
enum DebugStore { STORE_NONE, STORE_F32, STORE_BF16, STORE_PLANES };
struct DebugLoc { DebugStore store; void* p; };
struct DebugBuf { long long rows; int ld; DebugLoc at; };

static int debug_buffer(dsat_ctx* c, int id, DebugBuf* d) {
    const long long Nt = c->Nt, Mt = c->Mt;
    auto f32 = [](void* p) { return DebugLoc{STORE_F32, p}; };
    auto b16 = [](void* p) { return DebugLoc{STORE_BF16, p}; };
    auto planes = [](void* p) { return DebugLoc{STORE_PLANES, p}; };
    const DebugLoc none{STORE_NONE, nullptr};
    struct Row { long long rows; int ld; DebugLoc simt, bf16, x3; };     // DSAT_F32, DSAT_BF16(_UNFUSED), DSAT_F32_TC
    Row r;
    switch (id) {
        case DSAT_BUF_VROW: r = {Nt, c->ldv(), f32(c->VROW.p), b16(c->VROWb.p), planes(c->VROWp.p)}; break;
        case DSAT_BUF_CROW: r = {Mt, c->ldc(), f32(c->CROW.p), b16(c->CROWb.p), planes(c->CROWp.p)}; break;
        case DSAT_BUF_H1: r = {Nt, c->ldh1(), f32(c->H1.p), none, none}; break;
        case DSAT_BUF_H2: r = {Nt, c->HL, f32(c->H2.p), none, planes(c->H2p.p)}; break;
        case DSAT_BUF_QS: r = {Nt, 3 * c->Q, f32(c->QS.p), b16(c->QSb.p), f32(c->QS.p)}; break;
        case DSAT_BUF_LIT: r = {Nt, 2 * c->Q, f32(c->LIT.p), b16(c->LITb.p), f32(c->LIT.p)}; break;
        case DSAT_BUF_CH: r = {Mt, c->HC, f32(c->CH.p), none, none}; break;
        case DSAT_BUF_COUT: r = {Mt, c->Q + c->F, f32(c->COUT.p), b16(c->COUTb.p), f32(c->COUT.p)}; break;
        case DSAT_BUF_U1: r = {Nt, c->HU, f32(c->U1.p), none, none}; break;
        case DSAT_BUF_U2: r = {Nt, c->HU, f32(c->U2.p), none, none}; break;
        case DSAT_BUF_UOUT: r = {Nt, c->F, f32(c->UOUT.p), b16(c->UOUTb.p), f32(c->UOUT.p)}; break;
        case DSAT_BUF_SPRE: r = {Nt, c->F, f32(c->SPRE.p), b16(c->SPREb.p), planes(c->SPREp.p)}; break;
        case DSAT_BUF_O1: r = {Nt, c->HO, f32(c->O1.p), none, none}; break;
        case DSAT_BUF_LOGITS: r = {Nt, DSAT_LOGIT_PAD, f32(c->LOGITS.p), f32(c->LOGITS.p), f32(c->LOGITS.p)}; break;
        case DSAT_BUF_OUT: r = {Nt, 1, f32(c->OUT.p), f32(c->OUT.p), f32(c->OUT.p)}; break;
        case DSAT_BUF_X: r = {Nt, 2, f32(c->X.p), f32(c->X.p), f32(c->X.p)}; break;
        default: c->err = "unknown buffer id"; return DSAT_ERR_ARG;
    }
    *d = {r.rows, r.ld, use_x3(c) ? r.x3 : use_tc(c) ? r.bf16 : r.simt};
    return DSAT_OK;
}

// dsat_debug_read / dsat_debug_write: the buffers of the active precision, and where buffer `id` lives there
static int debug_access(dsat_ctx* c, int id, long long count, DebugBuf* d) {
    CK_CUDA(c, cudaSetDevice(c->device));
    int rc = ensure_active_buffers(c);
    if (rc || (rc = debug_buffer(c, id, d))) return rc;
    if (d->at.store == STORE_NONE) { c->err = "the active precision does not hold this buffer (it stays on-chip)"; return DSAT_ERR_UNSUPPORTED; }
    CK_ARG(c, count == d->rows * d->ld, "dsat_debug_read / dsat_debug_write: count must be rows*ld");
    CK_CUDA(c, cudaStreamSynchronize(c->stream));
    return DSAT_OK;
}

int dsat_debug_dims(const dsat_ctx* cc, int buffer, long long* rows, int* ld) {
    dsat_ctx* c = const_cast<dsat_ctx*>(cc);
    if (!c || !rows || !ld) return DSAT_ERR_ARG;
    CK_ARG(c, c->has_model && c->has_graph, "set the model and the graph first");
    DebugBuf d;
    if (int rc = debug_buffer(c, buffer, &d)) return rc;
    *rows = d.rows; *ld = d.ld;
    return DSAT_OK;
}

int dsat_debug_read(dsat_ctx* c, int buffer, float* host_out, long long count) {
    if (!c || !host_out) return DSAT_ERR_ARG;
    DebugBuf d;
    if (int rc = debug_access(c, buffer, count, &d)) return rc;
    if (d.at.store == STORE_F32) {
        CK_CUDA(c, dsat_memcpy_sync(host_out, d.at.p, (size_t)count * sizeof(float), cudaMemcpyDeviceToHost));
        return DSAT_OK;
    }
    const bool split = d.at.store == STORE_PLANES;
    std::vector<__nv_bfloat16> tmp((size_t)count * (split ? 2 : 1));
    CK_CUDA(c, dsat_memcpy_sync(tmp.data(), d.at.p, tmp.size() * 2, cudaMemcpyDeviceToHost));
    for (long long i = 0; i < count; ++i)
        host_out[i] = split ? __bfloat162float(tmp[i]) + __bfloat162float(tmp[count + i]) : __bfloat162float(tmp[i]);
    return DSAT_OK;
}

int dsat_debug_write(dsat_ctx* c, int buffer, const float* host_in, long long count) {
    if (!c || !host_in) return DSAT_ERR_ARG;
    DebugBuf d;
    if (int rc = debug_access(c, buffer, count, &d)) return rc;
    if (d.at.store == STORE_F32) {
        CK_CUDA(c, dsat_memcpy_sync(d.at.p, host_in, (size_t)count * sizeof(float), cudaMemcpyHostToDevice));
        return DSAT_OK;
    }
    const bool split = d.at.store == STORE_PLANES;
    std::vector<__nv_bfloat16> tmp((size_t)count * (split ? 2 : 1));
    for (long long i = 0; i < count; ++i) {     // round to nearest, as the kernels' __float2bfloat16_rn
        const __nv_bfloat16 hi = __float2bfloat16(host_in[i]);
        tmp[i] = hi;
        if (split) tmp[count + i] = __float2bfloat16(host_in[i] - __bfloat162float(hi));
    }
    CK_CUDA(c, dsat_memcpy_sync(d.at.p, tmp.data(), tmp.size() * 2, cudaMemcpyHostToDevice));
    return DSAT_OK;
}

// Stand-alone run of the tensor-core linear kernel on host data (parity test of the tcgen05 path):
// out = epi(bf16(A) @ bf16(W) + bias), out is [rows, N] fp32 (for the query epilogue [rows, 3N]).
int dsat_tc_linear_test(dsat_ctx* c, int rows, int K, int N, const float* a_host, const float* w_host,
                        const float* bias_host, int epi, int out_bf16, float* out_host) {
    if (!c || !a_host || !w_host || !bias_host || !out_host) return DSAT_ERR_ARG;
    CK_ARG(c, rows > 0 && K > 0 && N > 0 && K % 16 == 0 && N % 16 == 0, "dsat_tc_linear_test: K and N must be multiples of 16");
    CK_ARG(c, epi != tc::TC_QUERY || N % 32 == 0, "query epilogue needs N % 32 == 0");
    CK_CUDA(c, cudaSetDevice(c->device));
    const int K64 = (K + 63) / 64 * 64;
    const int out_cols = epi == tc::TC_QUERY ? 3 * N : N;
    std::vector<__nv_bfloat16> a((size_t)rows * K), wt((size_t)N * K64, __float2bfloat16(0.f));
    for (size_t i = 0; i < a.size(); ++i) a[i] = __float2bfloat16(a_host[i]);
    for (int k = 0; k < K; ++k)
        for (int n = 0; n < N; ++n) wt[(size_t)n * K64 + k] = __float2bfloat16(w_host[(size_t)k * N + n]);
    DevBuf<__nv_bfloat16> da, dw, dout_b;
    DevBuf<float> db, dout_f;
    CK_CUDA(c, da.alloc(a.size()));
    CK_CUDA(c, dw.alloc(wt.size()));
    CK_CUDA(c, db.alloc(N));
    CK_CUDA(c, dout_b.alloc((size_t)rows * out_cols));
    CK_CUDA(c, dout_f.alloc((size_t)rows * out_cols));
    CK_CUDA(c, dsat_memcpy_sync(da.p, a.data(), a.size() * 2, cudaMemcpyHostToDevice));
    CK_CUDA(c, dsat_memcpy_sync(dw.p, wt.data(), wt.size() * 2, cudaMemcpyHostToDevice));
    CK_CUDA(c, dsat_memcpy_sync(db.p, bias_host, N * sizeof(float), cudaMemcpyHostToDevice));
    tc::TcLinear l;
    l.a_box_rows = rows < tc::BLOCK_M ? rows : tc::BLOCK_M;
    l.b_box_rows = N < tc::BLOCK_N ? N : tc::BLOCK_N;
    if (!tc::make_bf16_map(&l.map_a, da.p, rows, K, K, l.a_box_rows) || !tc::make_bf16_map(&l.map_b, dw.p, N, K64, K64, l.b_box_rows)) {
        c->err = "cuTensorMapEncodeTiled failed";
        da.release(); dw.release(); db.release(); dout_b.release(); dout_f.release();
        return DSAT_ERR_CUDA;
    }
    l.bias = db.p;
    l.out.ptr0 = out_bf16 ? (void*)dout_b.p : (void*)dout_f.p; l.out.ld0 = out_cols; l.out.bf16_0 = out_bf16 ? 1 : 0;
    l.out.ptr1 = nullptr; l.out.ld1 = 0; l.out.bf16_1 = 0; l.out.split = 0;
    l.rows = rows; l.K = K; l.N = N; l.epi = epi; l.qmaps = N;
    cudaError_t e = tc::launch_tc_linear(l, c->stream);
    c->launches++;
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e == cudaSuccess) {
        if (out_bf16) {
            std::vector<__nv_bfloat16> ob((size_t)rows * out_cols);
            e = dsat_memcpy_sync(ob.data(), dout_b.p, ob.size() * 2, cudaMemcpyDeviceToHost);
            for (size_t i = 0; i < ob.size(); ++i) out_host[i] = __bfloat162float(ob[i]);
        } else {
            e = dsat_memcpy_sync(out_host, dout_f.p, (size_t)rows * out_cols * sizeof(float), cudaMemcpyDeviceToHost);
        }
    }
    da.release(); dw.release(); db.release(); dout_b.release(); dout_f.release();
    CK_CUDA(c, e);
    return DSAT_OK;
}

// Randomized rounding of the CURRENT diffusion state X alone (dsat_debug_write of DSAT_BUF_X first): X <- one-hot sample
// drawn with the context's sampling mode and the Philox stream (seed, step).
int dsat_debug_rounding(dsat_ctx* c, uint64_t seed, int step) {
    if (!c) return DSAT_ERR_ARG;
    CK_CUDA(c, cudaSetDevice(c->device));
    int rc = ensure_active_buffers(c);
    if (rc) return rc;
    NoiseSource ns{seed, 0ull, (unsigned)step};
    if ((rc = begin_call(c, 0.5f, nullptr, nullptr, nullptr, true, ns))) return rc;
    CK_CUDA(c, cudaStreamSynchronize(c->stream));
    return DSAT_OK;
}

int dsat_debug_begin(dsat_ctx* c, float noise_scale, const float* noisy_num, const int32_t* labels) {
    if (!c || !noisy_num) return DSAT_ERR_ARG;
    CK_CUDA(c, cudaSetDevice(c->device));
    int rc = ensure_active_buffers(c);
    if (rc) return rc;
    const size_t Nt = (size_t)c->Nt;
    CK_CUDA(c, c->inj_noisy.alloc(Nt * 2));
    CK_CUDA(c, c->inj_noisy.upload(noisy_num, Nt * 2, c->stream));
    if (labels) {
        CK_CUDA(c, c->inj_labels.alloc(Nt));
        CK_CUDA(c, c->inj_labels.upload(labels, Nt, c->stream));
    }
    NoiseSource ns{0ull, 0ull, 0u};
    if ((rc = begin_call(c, noise_scale, c->inj_noisy.p, nullptr, labels ? c->inj_labels.p : nullptr, false, ns))) return rc;
    CK_CUDA(c, cudaStreamSynchronize(c->stream));
    return DSAT_OK;
}

int dsat_debug_round(dsat_ctx* c, int round, const float* normals) {
    if (!c) return DSAT_ERR_ARG;
    CK_CUDA(c, cudaSetDevice(c->device));
    int rc = ensure_active_buffers(c);
    if (rc) return rc;
    const size_t Nt = (size_t)c->Nt;
    if (normals) {
        CK_CUDA(c, c->inj_normals.alloc(Nt * 4));
        CK_CUDA(c, c->inj_normals.upload(normals, Nt * 4, c->stream));
    }
    CK_CUDA(c, cudaStreamSynchronize(c->stream));
    const float noise_scale = c->last_noise_scale;      // set by dsat_debug_begin
    NoiseSource ns{0ull, 0ull, 0u};
    rc = run_round(c, round, normals ? c->inj_normals.p : nullptr, ns, loss_scalars(noise_scale));
    if (rc) return rc;
    CK_CUDA(c, cudaStreamSynchronize(c->stream));
    return DSAT_OK;
}

// One MLP alone in the active precision, on whatever its input buffer holds (written with dsat_debug_write):
// 0 variables_query (VROW -> QS), 1 lit_query (VROW -> LIT), 2 clause_update (CROW -> COUT), 3 update_gate (VROW -> UOUT),
// 4 variables_output (SPRE -> LOGITS).
int dsat_debug_mlp(dsat_ctx* c, int which) {
    if (!c || which < 0 || which > 4) return DSAT_ERR_ARG;
    CK_CUDA(c, cudaSetDevice(c->device));
    int rc = ensure_active_buffers(c);
    if (rc || (rc = run_mlp(c, which))) return rc;
    CK_CUDA(c, cudaStreamSynchronize(c->stream));
    return DSAT_OK;
}

int dsat_debug_groups(dsat_ctx* c, int32_t* done, int32_t* steps_taken, float* loss_sum, int32_t* graph_sat,
                      int32_t* graph_map) {
    if (!c) return DSAT_ERR_ARG;
    CK_ARG(c, c->has_buffers, "no buffers yet");
    CK_CUDA(c, cudaSetDevice(c->device));
    CK_CUDA(c, cudaStreamSynchronize(c->stream));
    if (done) CK_CUDA(c, dsat_memcpy_sync(done, c->done.p, c->n_groups * sizeof(int), cudaMemcpyDeviceToHost));
    if (steps_taken) CK_CUDA(c, dsat_memcpy_sync(steps_taken, c->steps_taken.p, c->n_groups * sizeof(int), cudaMemcpyDeviceToHost));
    if (loss_sum) CK_CUDA(c, dsat_memcpy_sync(loss_sum, c->loss_sum.p, c->n_groups * sizeof(float), cudaMemcpyDeviceToHost));
    if (graph_sat) CK_CUDA(c, dsat_memcpy_sync(graph_sat, c->graph_sat.p, c->total_graphs * sizeof(int), cudaMemcpyDeviceToHost));
    if (graph_map) CK_CUDA(c, dsat_memcpy_sync(graph_map, c->graph_map.p, c->total_graphs * sizeof(int), cudaMemcpyDeviceToHost));
    return DSAT_OK;
}

}  // extern "C"
