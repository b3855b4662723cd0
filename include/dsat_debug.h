/*
 * dsat_debug.h -- profiling, parity and debug hooks of libdsat.so.
 *
 * These entry points exist for bench.py (per-class device time), the parity tests (run one round, one MLP or one
 * linear op alone; read and write activation buffers) and kernel tuning.  They are exported by the same library but
 * are NOT part of the drop-in surface (include/dsat.h); they may change with the kernels.
 */
#ifndef DSAT_DEBUG_H_
#define DSAT_DEBUG_H_

#include "dsat.h"

#ifdef __cplusplus
extern "C" {
#endif

/* debug/parity access to the activation buffers of one round (dsat_debug_read / dsat_debug_write) */
enum dsat_buffer {
    DSAT_BUF_VROW = 0,    /* [N, F+16+3Q]  variables | aux16 | variables_grad | loss_pos | loss_neg */
    DSAT_BUF_CROW = 1,    /* [M, F+2Q]     clause_state | clause_messages | 4*clauses_loss          */
    DSAT_BUF_H1 = 2,      /* [N, Hq+4Q]    hidden of variables_query | first hidden of lit_query     */
    DSAT_BUF_H2 = 3,      /* [N, 4Q]       second hidden of lit_query                                 */
    DSAT_BUF_QS = 4,      /* [N, 3Q]       query | softplus(query) | softplus(-query)                 */
    DSAT_BUF_LIT = 5,     /* [N, 2Q]       lit_query output (positive | negative literal features)    */
    DSAT_BUF_CH = 6,      /* [M, Hc]       hidden of clause_update                                    */
    DSAT_BUF_COUT = 7,    /* [M, Q+F]      clause_update output (message to literals | new value)     */
    DSAT_BUF_U1 = 8,      /* [N, Hu] */
    DSAT_BUF_U2 = 9,      /* [N, Hu] */
    DSAT_BUF_UOUT = 10,   /* [N, F]        update_gate output before PairNorm                          */
    DSAT_BUF_SPRE = 11,   /* [N, F]        variables after PairNorm+residual, before the 0.2/0.8 carry  */
    DSAT_BUF_O1 = 12,     /* [N, Ho] */
    DSAT_BUF_LOGITS = 13, /* [N, 16]       8 logit maps + padding                                       */
    DSAT_BUF_OUT = 14,    /* [N]           selected logit per variable (out_logits)                     */
    DSAT_BUF_X = 15,      /* [N, 2]        diffusion state x                                            */
    DSAT_BUF_COUNT = 16
};

/* Per-kernel-class device time of `rounds` message-passing rounds, measured with CUDA events on the
 * context's stream (bench.py roofline).  Classes 0..10 are the eleven linear ops in launch order
 * (v1->hidden, query out, lit 2, lit 3, clause 1, clause 2, update 1, 2, 3, output 1, 2), then
 * clause gather, literal gather, clause PairNorm, variable PairNorm, head, noise.
 * class_ms / class_launches have dsat_profile_classes() entries. */
int dsat_profile_classes(void);
/* clock64 wait/work breakdown of CTA 0 of one whole-MLP kernel (0 query .. 4 output); 16 counters */
int dsat_profile_fused(dsat_ctx* ctx, int which, long long* counters16);
int dsat_profile_rounds(dsat_ctx* ctx, int rounds, uint64_t seed, float* class_ms, int32_t* class_launches);

/* Stand-alone run of the tcgen05 linear kernel on host data (parity of the tensor-core MLP path,
 * model/mlp.py:42-50): out = epi(bf16(a) @ bf16(w) + bias); a [rows,K], w [K,N], out [rows,N] fp32
 * ([rows,3N] for epi 2 = query epilogue with the softplus pair); epi 0 linear, 1 leaky-relu 0.2. */
int dsat_tc_linear_test(dsat_ctx* ctx, int rows, int K, int N, const float* a_host, const float* w_host,
                        const float* bias_host, int epi, int out_bf16, float* out_host);

/* Build flags of the loaded library: bit 0 = tcgen05 paths compiled in (always 1), bit 1 = -DDSAT_ASSERT debug build
 * (bounds checks). */
int dsat_build_info(void);

/* Randomized rounding alone: X (DSAT_BUF_X, written with dsat_debug_write) <- one-hot sample drawn with the context's
 * sampling mode from the Philox stream (seed, step). */
int dsat_debug_rounding(dsat_ctx* ctx, uint64_t seed, int step);

/* Parity hooks: run the pieces of one model call separately and read/write activation buffers.  dsat_debug_read /
 * dsat_debug_write convert between the caller's fp32 and the buffer's storage in the active precision (fp32, bf16, or
 * hi + lo bf16 planes); a buffer the precision does not hold (hidden activations that stay on-chip) returns
 * DSAT_ERR_UNSUPPORTED.  dsat_debug_dims answers for every buffer. */
int dsat_debug_begin(dsat_ctx* ctx, float noise_scale, const float* noisy_num, const int32_t* labels);
int dsat_debug_round(dsat_ctx* ctx, int round, const float* normals /* [N,4] host */);
int dsat_debug_dims(const dsat_ctx* ctx, int buffer, long long* rows, int* ld);
int dsat_debug_read(dsat_ctx* ctx, int buffer, float* host_out, long long count);
int dsat_debug_write(dsat_ctx* ctx, int buffer, const float* host_in, long long count);
int dsat_debug_groups(dsat_ctx* ctx, int32_t* done, int32_t* steps_taken, float* loss_sum,
                      int32_t* graph_sat, int32_t* graph_map);
/* One MLP alone in the active precision on the current contents of its input buffer (model/query_sat.py:117-122):
 * which = 0 variables_query (VROW -> QS), 1 lit_query (VROW -> LIT), 2 clause_update (CROW -> COUT),
 * 3 update_gate (VROW -> UOUT), 4 variables_output (SPRE -> LOGITS). */
int dsat_debug_mlp(dsat_ctx* ctx, int which);

#ifdef __cplusplus
}
#endif
#endif /* DSAT_DEBUG_H_ */
