/*
 * dsat.h -- C ABI of the B200-native DiffusionSAT sampling hot path (libdsat.so).
 *
 * The reference (LUMII-Syslab/DiffusionSAT) has no FFI of its own: its boundary for this path is the
 * Python API  DiffusionSampler(model_path, dimacs).samples(n)  and  QuerySAT.diffusion_step(...).
 * Each entry point below names the reference code it replaces (file:line into the reference tree).
 * The Python mirror of that API (diffusionsat_b200/) binds these symbols with ctypes; INTEGRATION.md
 * shows the stub a maintainer of the reference would add.
 *
 * Conventions: plain pointers and sizes only; every call returns 0 or a negative dsat_status and
 * leaves a message for dsat_last_error(); no exceptions cross the ABI; "host" buffers are caller
 * owned and copied, "dev" buffers are device pointers of the context's device; one context per GPU,
 * not thread-safe; all work is issued on the context's stream; there is no CPU fallback.
 * Profiling, parity and debug hooks (not part of the product surface) live in dsat_debug.h.
 *
 * Row order of every per-variable array is the reference's batch order: variable v of graph g of
 * chain c sits at  c*n_vars + v  with n_vars the unit's variable total (data/dimac.py:239-241,
 * data/SatSpecifics.py:22-35); graphs are numbered  c*n_graphs + g.
 */
#ifndef DSAT_H_
#define DSAT_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dsat_ctx dsat_ctx;

enum dsat_status {
    DSAT_OK = 0,
    DSAT_ERR_ARG = -1,      /* bad argument / call order */
    DSAT_ERR_CUDA = -2,     /* CUDA runtime error, see dsat_last_error */
    DSAT_ERR_STATE = -3,    /* model or graph not set */
    DSAT_ERR_UNSUPPORTED = -4
};

/* Arithmetic of the twelve Dense layers (everything else is fp32 in every mode):
 *   DSAT_F32          fp32 FMA on the CUDA cores (bit-level cross-check of the tensor-core paths)
 *   DSAT_F32_TC       fp32-accurate on the tcgen05 tensor cores: every operand is carried as two bf16 planes (hi, lo) and
 *                     every product is three bf16 MMAs into one fp32 accumulator (~1e-5 relative); the default of the
 *                     Python drop-in classes; matches the reference's fp32 Dense layers within the 1e-3 tolerance
 *   DSAT_BF16         plain bf16 operands and bf16 activation storage, one tcgen05 kernel per MLP (stated separately)
 *   DSAT_BF16_UNFUSED the same with one tcgen05 kernel per Dense layer */
enum dsat_dtype { DSAT_F32 = 0, DSAT_BF16 = 1, DSAT_BF16_UNFUSED = 2, DSAT_F32_TC = 3 };

int dsat_version(void);

/* Lifetime.  One context per GPU.  Replaces the implicit TF runtime/device placement of
 * satuniformity/DiffusionSampler.py:197-213. */
int dsat_create(int device, dsat_ctx** out);
void dsat_destroy(dsat_ctx* ctx);
const char* dsat_last_error(const dsat_ctx* ctx);

/* Use a caller stream (cudaStream_t passed as void*) for all work; NULL restores the own stream. */
int dsat_set_stream(dsat_ctx* ctx, void* cuda_stream);
int dsat_synchronize(dsat_ctx* ctx);
/* CUDA-event timing on the context's stream (bench.py): begin records, end records+syncs, ms out. */
int dsat_timer_begin(dsat_ctx* ctx);
int dsat_timer_end(dsat_ctx* ctx, float* elapsed_ms);
/* kernels launched by this context since creation (bench.py "gpu_launches") */
long long dsat_launch_count(const dsat_ctx* ctx);

/* Weights of the twelve Dense layers in the order variables_query/0,1  lit_query/0,1,2
 * clause_update/0,1  update_gate/0,1,2  variables_output/0,1; kernels[i] is row-major [in,out] fp32,
 * biases[i] is [out].  Replaces the checkpoint restore of DiffusionSampler.py:215-227 and the layer
 * construction of model/query_sat.py:117-122 (model/mlp.py:23-24,39). */
int dsat_set_model(dsat_ctx* ctx, int n_layers, const float* const* kernels, const float* const* biases,
                   const int* in_dims, const int* out_dims);

/* How the denoising step rounds x to a one-hot sample: DSAT_SAMPLE_INVERSE_CDF = floor(x0 + U), the reference's live code
 * (model/query_sat.py:55-60) and the mode every bit-exact parity statement refers to; DSAT_SAMPLE_GUMBEL = Gumbel-argmax
 * (the sampler sketched in model/query_sat.py:15-28), same distribution, validated statistically. */
enum dsat_sampling { DSAT_SAMPLE_INVERSE_CDF = 0, DSAT_SAMPLE_GUMBEL = 1 };
int dsat_set_sampling(dsat_ctx* ctx, int mode);

/* dtype of the MLP path, see enum dsat_dtype */
int dsat_set_precision(dsat_ctx* ctx, int dtype);
/* The active dtype.  A new context starts in DSAT_F32_TC; dsat_set_model switches it to DSAT_F32 (CUDA cores, the same
 * fp32 results) for layer widths the split-precision kernels do not tile (feature_maps or query_maps = 256). */
int dsat_get_precision(const dsat_ctx* ctx);

/* Unit graph shared by all chains.  cl_lit holds literal codes 2*var+sign (var 0-based in the unit);
 * lit_rowptr is indexed by literal code.  var_seg/clause_seg [n_graphs+1] delimit the formulas of a
 * disjoint union.  group_graphs = graphs per early-exit batch (reference: all graphs of one TF batch,
 * model/query_sat.py:330-338); 0 means "all graphs of this context".
 * Replaces data/dimac.py:14-18,213-260 + data/SatSpecifics.py:21-69 (adjacency construction) and the
 * degree weights of model/query_sat.py:193-197.
 * Every argument is validated before the context is touched (sizes, monotone row pointers, index ranges, CSR and CSC
 * describing the same edges): a rejected call leaves the previously bound graph in place.  Binding a graph of another
 * shape re-plans the kernels but re-uses the context's device allocations when they are large enough; a context keeps
 * its largest allocations until dsat_destroy. */
int dsat_set_graph(dsat_ctx* ctx, int n_vars, int n_clauses, int nnz,
                   const int32_t* cl_rowptr, const int32_t* cl_lit,
                   const int32_t* lit_rowptr, const int32_t* lit_clause,
                   int n_graphs, const int32_t* var_seg, const int32_t* clause_seg,
                   int n_chains, int group_graphs);

/* Reference batches of several formulas in one launch (a disjoint union bound by dsat_set_graph).
 * Early-exit group i = graphs [group_seg[i], group_seg[i+1]) of the context's n_chains*n_graphs graphs (replaces
 * group_graphs); if noise_base is not NULL, the Philox element of variable v (0-based inside its graph) of graph gi is
 * noise_base[gi] + v, and dsat_sample / dsat_sample_enqueue / dsat_model_call then require chain_offset == 0.
 * Validated before anything changes; cleared by the next dsat_set_graph.
 * With noise_base[gi] = (c0 + j) * n_k for copy j of a formula of n_k variables, a copy draws exactly the noise of chain
 * c0 + j of that formula bound alone, so its samples do not depend on which formulas share the launch.  The steps_taken /
 * loss outputs of dsat_model_call have one entry per bound group.  Finished groups are not skipped (their results are
 * the same either way). */
int dsat_set_batches(dsat_ctx* ctx, int n_groups, const int32_t* group_seg, const uint64_t* noise_base);

/* Host-only helper (no context, no device): the index arrays dsat_set_graph takes, from the signed 1-based literals of all
 * clauses laid end to end (lens[j] literals for clause j, sum = nnz; a disjoint union passes its formulas already shifted by
 * their variable offsets, data/dimac.py:165-170,239-241).  cl_rowptr [n_clauses+1], cl_lit [nnz] (codes 2*var+sign, inside a
 * clause in the order of the reference's literal rows: positives by variable, then negatives; repeated literals kept),
 * lit_rowptr [2*n_vars+1], lit_clause [nnz] (ascending, repeats kept).  Replaces data/dimac.py:14-18 (compute_adj_indices)
 * + data/SatSpecifics.py:21-69 (create_adj_matrices) for callers that build many graphs per second (mixed-formula batches);
 * diffusionsat_b200/graph.py holds the same construction in numpy and the tests compare the two.
 * A literal of magnitude 0 or > n_vars returns DSAT_ERR_ARG with *bad_clause = its clause (else -1; may be NULL). */
int dsat_graph_build(int n_vars, int n_clauses, long long nnz, const int32_t* lens, const int32_t* flat,
                     int32_t* cl_rowptr, int32_t* cl_lit, int32_t* lit_rowptr, int32_t* lit_clause, int32_t* bad_clause);

/* One model call = QuerySAT.diffusion_step / call(training=False)  (model/query_sat.py:133-184,
 * 186-373, 467-481).  Host buffers: noisy_num [N,2]; labels [N] int32 or NULL (drawn from Philox,
 * the reference draws them with tf.random at :145); normals [rounds,N,4] or NULL (Philox; reference
 * tf.random.normal at :239); prediction_out [N] logits; steps_taken/loss [n_groups] (may be NULL). */
int dsat_model_call(dsat_ctx* ctx, float noise_scale, const float* noisy_num, const int32_t* labels,
                    const float* normals, int rounds, uint64_t seed, uint64_t chain_offset,
                    float* prediction_out, int32_t* steps_taken, float* loss);

/* Whole reverse-diffusion run for all chains of the context = diffusion() + the per-graph
 * int-encoding / SAT check of samples()  (satuniformity/DiffusionSampler.py:78-191, 283-303;
 * utils/VariableAssignment.py:63-90).  Optional injected noise (host): uniforms [steps,N],
 * labels [steps,N] int32, normals [steps,rounds,N,4]; NULL = Philox keyed by (seed, global chain).
 * Outputs (host): packed [n_total_graphs, words] little-endian 64-bit words, x1 = bit 0;
 * is_sat [n_total_graphs]; latch_step [n_total_graphs] (-1 = never satisfied);
 * sat_any_step [n_total_graphs] (cum_accuracy flags of diffusion(), may be NULL). */
int dsat_sample(dsat_ctx* ctx, int n_steps, int n_rounds, uint64_t seed, uint64_t chain_offset,
                const float* uniforms, const int32_t* labels, const float* normals,
                uint64_t* packed, uint8_t* is_sat, int32_t* latch_step, uint8_t* sat_any_step);
/* The same run split for resident benchmarking: enqueue only (no host copies, no sync), then fetch. */
int dsat_sample_enqueue(dsat_ctx* ctx, int n_steps, int n_rounds, uint64_t seed, uint64_t chain_offset);
int dsat_sample_fetch(dsat_ctx* ctx, uint64_t* packed, uint8_t* is_sat, int32_t* latch_step,
                      uint8_t* sat_any_step);
int dsat_words_per_graph(const dsat_ctx* ctx);

/* Stand-alone segment-sum SpMM on device buffers (message-passing roofline sweeps):
 * direction 0: clause <- literal   Y[c,j,:] = rev_w[j]  * sum_{lit in j} X[c,lit,:]   X [chains,2n,feat]
 * direction 1: literal <- clause   Y[c,l,:] = deg_w[l] * sum_{j contains l} X[c,j,:]  X [chains,m,feat]
 * (tf.sparse.sparse_dense_matmul call sites model/query_sat.py:255,269).  feat in {64,128,256}.
 * The first call after dsat_set_graph builds the row descriptors of the bound graph on the host and uploads them
 * (a few ms at n = 10000); the model path never pays for them.  Sums run in entry order with fp32 accumulation. */
int dsat_spmm(dsat_ctx* ctx, int direction, const void* x_dev, void* y_dev, int feat, int dtype, int chains);

/* Histogram of the last dsat_sample / dsat_sample_enqueue run, reduced on the device: sort, unique and count of the
 * packed SATISFYING assignments of chains [0, chain_limit) (chain_limit <= 0: all chains of the context).
 * keys_out [capacity, words] (word 0 = variables 1..64, as in `packed`), ascending by the integer they encode;
 * counts_out [capacity]; *n_unique = number of distinct assignments, *n_sat = satisfied chains counted (may be NULL).
 * Returns DSAT_ERR_ARG with *n_unique set when capacity is too small.  Replaces the per-sample dict update of
 * satuniformity/DiffusionSampler.py:283-307 (int encoding utils/VariableAssignment.py:63-69); the cross-GPU merge of
 * these tables is diffusionsat_b200/dist.py (NCCL all-gather of keys + reduce of counts). */
int dsat_hist_reduce(dsat_ctx* ctx, int chain_limit, uint64_t* keys_out, int64_t* counts_out, int capacity,
                     int32_t* n_unique, int32_t* n_sat);

/* dsat_hist_reduce per formula: segment s = graphs [graph_seg[s], graph_seg[s+1]), of which the first limit[s]
 * count.  Keys ascend within a segment, segments in order; seg_runs[n_segments+1] = offsets of each segment's runs.
 * Segments are ordered and lie inside the context's graphs; graphs outside every segment do not count.  keys_out has
 * dsat_words_per_graph words per key (a formula with fewer variables has zero high words); *n_sat = satisfied graphs
 * counted over all segments (may be NULL).  Returns DSAT_ERR_ARG with seg_runs[n_segments] = the required capacity
 * when capacity is too small. */
int dsat_hist_reduce_segments(dsat_ctx* ctx, int n_segments, const int32_t* graph_seg, const int32_t* limit,
                              uint64_t* keys_out, int64_t* counts_out, int capacity, int32_t* seg_runs, int32_t* n_sat);

#ifdef __cplusplus
}
#endif
#endif /* DSAT_H_ */
