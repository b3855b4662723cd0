"""CPU ORACLE for the DiffusionSAT sampling hot path  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl
reference`` legs may import this module. The product path (``diffusionsat_b200``) never does and
fails loudly when its CUDA library is missing.

What it is: a torch-CPU restatement (fp32 to mirror the reference's TF CPU run, fp64 as "truth")
of the reference's algorithm for the path, written against the reference's own batch layout — one
disjoint-union graph with ``N`` variables and ``M`` clauses in total, positive literal rows
``[0,N)``, negative rows ``[N,2N)`` — so that every function below can be read next to the
reference lines it follows:

=============================  ==========================================================
function here                   reference file:line
=============================  ==========================================================
``mlp``                         ``model/mlp.py:23-24,39,42-50``
``pair_norm``                   ``layers/normalization.py:43-71``, graph-norm matrices
                                ``model/query_sat.py:206-211``
``degree_weights``              ``model/query_sat.py:193-197``
``softplus_loss_adj``           ``loss/sat.py:125-137``
``train_loss``                  ``model/query_sat.py:40-53`` (+ TFP Bernoulli KL, external)
``distribution_at_time``        ``model/query_sat.py:66-68``
``is_batch_sat``                ``utils/sat.py:118-124``
``model_loop``                  ``model/query_sat.py:186-373``
``model_call``                  ``model/query_sat.py:133-184`` / ``diffusion_step`` ``:467-481``
``randomized_rounding``         ``model/query_sat.py:55-60``
``reverse_distribution_step_theoretic``  ``satuniformity/DiffusionSampler.py:29-37``
``graph_sat_flags``             ``metrics/sat_metrics.py:60-85``
``diffusion``                   ``satuniformity/DiffusionSampler.py:78-191``
``samples``                     ``satuniformity/DiffusionSampler.py:229-311``
=============================  ==========================================================

PARITY STATUS: the arithmetic of the path lives in TensorFlow 2.4 / TFP 0.12 (``requirements.txt:2-4``),
which cannot be imported in this container, and the reference ships no tests or golden vectors for
it (SURVEY.md section 4). The pure-Python parts (DIMACS parsing, literal indexing, int encoding,
SAT check, chi-square) ARE pinned against the reference modules themselves
(``tests/golden/make_golden.py``). The model arithmetic is additionally pinned by executing the
reference's own ``model/query_sat.py`` / ``DiffusionSampler.py`` source over a torch-backed stand-in
for the TensorFlow ops it calls (``oracle/tf_shim``; fixtures in ``tests/golden/``): that pins the
control flow, tensor plumbing and op order of the reference, while the semantics of each TF op remain
"as documented", i.e. *parity unpinned at the TF-kernel level*.

All randomness is injected: ``normals`` [rounds, N, 4] (``tf.random.normal`` at ``:239``), ``labels`` [N]
(``:145``) and ``uniforms`` [steps, N] (``:57``).
"""

from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch
import torch.nn.functional as F_

T_POWER = 0.5          # reference model/query_sat.py:13
LOGIT_MAPS = 8         # reference model/query_sat.py:99
LEAKY_ALPHA = 0.2      # tf.nn.leaky_relu default (external)
PAIRNORM_EPS = 1e-6    # reference layers/normalization.py:29


# --------------------------------------------------------------------------------------- graph
@dataclass
class OracleGraph:
    """The reference's batch: COO of ``adj_matrix`` [2N, M] in its storage order plus graph ids."""

    lit_row: torch.Tensor      # int64 [E]  literal row (positives [0,N), negatives [N,2N))
    clause: torch.Tensor       # int64 [E]
    n_vars: int                # N (batch total)
    n_clauses: int             # M (batch total)
    var_graph: torch.Tensor    # int64 [N] graph id of each variable
    clause_graph: torch.Tensor # int64 [M]
    n_graphs: int
    clauses_per_graph: list    # python clause lists per graph, local 1-based variables
    vars_per_graph: list       # python ints

    @staticmethod
    def from_formulas(formulas) -> "OracleGraph":
        """``formulas`` = [(n_vars, clauses), ...]; union built as reference ``data/dimac.py:213-260``
        + ``data/SatSpecifics.py:21-69``."""
        pos, neg, var_graph, clause_graph = [], [], [], []
        off, cidx = 0, 0
        for g, (n, clauses) in enumerate(formulas):
            for clause in clauses:
                for lit in clause:
                    if lit > 0:
                        pos.append((lit - 1 + off, cidx))
                    elif lit < 0:
                        neg.append((-lit - 1 + off, cidx))
                clause_graph.append(g)
                cidx += 1
            var_graph += [g] * n
            off += n
        n_total = off
        pairs = pos + [(r + n_total, c) for r, c in neg]
        idx = torch.tensor(pairs, dtype=torch.int64).reshape(-1, 2)
        return OracleGraph(
            lit_row=idx[:, 0].contiguous(), clause=idx[:, 1].contiguous(),
            n_vars=n_total, n_clauses=cidx,
            var_graph=torch.tensor(var_graph, dtype=torch.int64),
            clause_graph=torch.tensor(clause_graph, dtype=torch.int64),
            n_graphs=len(formulas),
            clauses_per_graph=[[list(c) for c in cl] for _, cl in formulas],
            vars_per_graph=[int(n) for n, _ in formulas],
        )

    @staticmethod
    def copies(n_vars, clauses, chains) -> "OracleGraph":
        """``chains`` identical copies of one formula (reference ``data/diffusion_sat_instances.py:91-94``)."""
        return OracleGraph.from_formulas([(n_vars, clauses)] * chains)

    # sparse x dense products with the adjacency, values all 1.0, duplicates counted -------------
    def lit_from_clause(self, x_clause: torch.Tensor) -> torch.Tensor:
        """``tf.sparse.sparse_dense_matmul(adj_matrix, x)``: [M,K] -> [2N,K]."""
        out = torch.zeros(2 * self.n_vars, x_clause.shape[1], dtype=x_clause.dtype)
        return out.index_add_(0, self.lit_row, x_clause[self.clause])

    def clause_from_lit(self, x_lit: torch.Tensor) -> torch.Tensor:
        """``tf.sparse.sparse_dense_matmul(tf.sparse.transpose(adj_matrix), x)``: [2N,K] -> [M,K]."""
        out = torch.zeros(self.n_clauses, x_lit.shape[1], dtype=x_lit.dtype)
        return out.index_add_(0, self.clause, x_lit[self.lit_row])


# ------------------------------------------------------------------------------------- weights
def weights_to_torch(weights, dtype=torch.float32):
    """``QuerySATWeights`` -> {mlp_name: [(W,b),...]} of torch tensors."""
    out = {}
    for name in ("variables_query", "lit_query", "clause_update", "update_gate", "variables_output"):
        out[name] = [(torch.from_numpy(np.asarray(w)).to(dtype), torch.from_numpy(np.asarray(b)).to(dtype))
                     for w, b in weights.mlp(name)]
    return out


# ------------------------------------------------------------------------------- building blocks
def mlp(x, layers):
    """Dense(leaky_relu 0.2) x (L-1) then linear Dense; y = x @ W + b."""
    for w, b in layers[:-1]:
        x = F_.leaky_relu(x @ w + b, LEAKY_ALPHA)
    w, b = layers[-1]
    return x @ w + b


def graph_norm_weights(graph_ids, n_graphs, dtype):
    """Row weights of ``graph / reduce_sum(graph, -1)``: 1/count of the node's graph."""
    counts = torch.bincount(graph_ids, minlength=n_graphs).to(dtype)
    return (1.0 / counts)[graph_ids]


def pair_norm(x, graph_ids, n_graphs, eps=PAIRNORM_EPS):
    w = graph_norm_weights(graph_ids, n_graphs, x.dtype)
    mean = torch.zeros(n_graphs, x.shape[1], dtype=x.dtype).index_add_(0, graph_ids, x * w[:, None])
    x = x - mean[graph_ids]
    variance = torch.mean(torch.square(x), dim=1, keepdim=True)
    return x * torch.rsqrt(variance + eps)


def softplus_loss_adj(query, graph: OracleGraph):
    literals = F_.softplus(torch.cat([query, -query], dim=0))
    return torch.exp(-graph.clause_from_lit(literals))


def distribution_at_time(x, time_increment):
    return x * (1 - time_increment) + time_increment / 2


def _bernoulli_kl(pa, pb):
    """KL(Bernoulli(pa) || Bernoulli(pb)) with probabilities as parameters; TFP 0.12's registered
    Bernoulli/Bernoulli KL computes pa*(log pa - log pb) + (1-pa)*(log1p(-pa) - log1p(-pb))
    with 0*inf := 0 (external; restated from the published formula)."""
    t1 = torch.where(pa == 0, torch.zeros_like(pa), pa * (torch.log(pa) - torch.log(pb)))
    qa = 1 - pa
    t2 = torch.where(qa == 0, torch.zeros_like(pa), qa * (torch.log1p(-pa) - torch.log1p(-pb)))
    return t1 + t2


def train_loss(labels, logits, noise_scale, label_smoothing=0.01):
    """labels, logits: [N, maps]; noise_scale: 0-dim tensor of the working dtype."""
    t = torch.pow(noise_scale, T_POWER)
    ts = torch.minimum(t + label_smoothing, torch.ones_like(t))
    labels_at_t = distribution_at_time(labels, ts)
    probs_at_t = distribution_at_time(torch.sigmoid(logits), t)
    loss = _bernoulli_kl(labels_at_t, probs_at_t)
    norm = _bernoulli_kl(distribution_at_time(torch.zeros_like(t), ts),
                         distribution_at_time(torch.zeros_like(t), torch.ones_like(t)))
    return loss / (norm + 1e-4)


def degree_weights(graph: OracleGraph, dtype):
    """``model/query_sat.py:193-197``: literal degrees [2N,1], clause sizes [M,1], ``degree_weight`` [2N,1],
    ``var_degree_weight`` [N,1] and ``rev_degree_weight`` [M,1]."""
    n, m = graph.n_vars, graph.n_clauses
    ones_e = torch.ones(graph.lit_row.shape[0], dtype=dtype)
    lit_degree = torch.zeros(2 * n, dtype=dtype).index_add_(0, graph.lit_row, ones_e)[:, None]
    rev_lit_degree = torch.zeros(m, dtype=dtype).index_add_(0, graph.clause, ones_e)[:, None]
    degree_weight = torch.rsqrt(torch.clamp(lit_degree, min=1))
    var_degree_weight = 4 * torch.rsqrt(torch.clamp(lit_degree[:n] + lit_degree[n:], min=1))
    rev_degree_weight = torch.rsqrt(torch.clamp(rev_lit_degree, min=1))
    return lit_degree, rev_lit_degree, degree_weight, var_degree_weight, rev_degree_weight


def is_batch_sat(out_logits, graph: OracleGraph):
    variables = torch.round(torch.sigmoid(out_logits))          # half-to-even, as tf.round
    literals = torch.cat([variables, 1 - variables], dim=0)
    clauses_sat = torch.clamp(graph.clause_from_lit(literals), 0, 1)
    return clauses_sat.min() if clauses_sat.numel() else torch.tensor(1.0, dtype=out_logits.dtype)


def query_gradient_analytic(query, clauses_loss, graph: OracleGraph):
    """d(sum clauses_loss)/d(query), closed form of the inner GradientTape (``:227-245``):
    d/dq exp(-S) with S = sum softplus(+-q) gives -sigma(q)*S+ + sigma(-q)*S- where
    S+- = (adj_matrix @ clauses_loss) on the positive / negative literal row of the variable."""
    s = graph.lit_from_clause(clauses_loss)
    n = graph.n_vars
    return -torch.sigmoid(query) * s[:n] + torch.sigmoid(-query) * s[n:]


# ------------------------------------------------------------------------------------ the model
def model_loop(graph: OracleGraph, w, noise_scale, noisy_num, labels, normals, rounds,
               dtype=torch.float32, trace=None, teacher=None, use_autograd=False):
    """Reference ``QuerySAT.loop`` for ``training=False``, ``supervised=True``, ``denoised_num=None``.

    ``trace``: optional list that receives one dict of intermediates per executed round.
    ``teacher``: optional list of per-round dicts with ``variables`` / ``clause_state`` to start each
    round from (teacher forcing for parity tests).
    Returns ``(out_logits [N], steps_taken, unsupervised_loss, last_logits [N,8], best_map [N])``.
    """
    n, m, g_cnt = graph.n_vars, graph.n_clauses, graph.n_graphs
    f = w["variables_output"][0][0].shape[0]
    q = w["variables_query"][-1][0].shape[1]
    ns = torch.as_tensor(noise_scale, dtype=dtype)

    _, _, degree_weight, var_degree_weight, rev_degree_weight = degree_weights(graph, dtype)

    var_w = graph_norm_weights(graph.var_graph, g_cnt, dtype)

    noisy_labels = torch.cat([noisy_num.to(dtype), torch.zeros(n, 1, dtype=dtype) + ns,
                              torch.zeros(n, 2, dtype=dtype)], dim=-1)          # :214-219
    variables = torch.ones(n, f, dtype=dtype)                                    # call() :148
    clause_state = torch.ones(m, f, dtype=dtype)                                 # call() :141
    last_logits = torch.zeros(n, LOGIT_MAPS, dtype=dtype)
    best_map = torch.zeros(n, dtype=torch.int64)
    labels_f = labels.to(dtype)[:, None].expand(n, LOGIT_MAPS)
    costs = torch.square(torch.arange(1, LOGIT_MAPS + 1, dtype=dtype))
    step_losses = []
    step = -1

    for step in range(rounds):
        if teacher is not None:
            variables = teacher[step]["variables"].to(dtype)
            clause_state = teacher[step]["clause_state"].to(dtype)
        v1 = torch.cat([variables, normals[step].to(dtype), noisy_labels], dim=-1)      # :239
        if use_autograd:
            v1q = v1.detach()
            qw = [(a.detach(), b.detach()) for a, b in w["variables_query"]]
            query = mlp(v1q, qw).requires_grad_(True)
            clauses_loss = softplus_loss_adj(query, graph)
            (grad,) = torch.autograd.grad(clauses_loss.sum(), query)
            query, clauses_loss = query.detach(), clauses_loss.detach()
        else:
            query = mlp(v1, w["variables_query"])                                        # :240
            clauses_loss = softplus_loss_adj(query, graph)                               # :241
            grad = query_gradient_analytic(query, clauses_loss, graph)                   # :245
        variables_grad = grad * var_degree_weight                                        # :246
        clauses_loss4 = clauses_loss * 4                                                 # :248

        var_msg = mlp(v1, w["lit_query"])                                                # :252
        literals = torch.cat([var_msg[:, :q], var_msg[:, q:]], dim=0)                    # :253-254
        clause_messages = graph.clause_from_lit(literals) * rev_degree_weight            # :255-256
        clause_unit = torch.cat([clause_state, clause_messages, clauses_loss4], dim=-1)  # :258
        clause_data = mlp(clause_unit, w["clause_update"])                               # :261

        variables_loss_all = clause_data[:, :q]                                          # :263
        new_clause_value = pair_norm(clause_data[:, q:], graph.clause_graph, g_cnt) * 0.25   # :264-265
        clause_state = new_clause_value + 0.1 * clause_state                             # :266

        variables_loss = graph.lit_from_clause(variables_loss_all) * degree_weight       # :269-270
        loss_pos, loss_neg = variables_loss[:n], variables_loss[n:]                      # :273

        unit = torch.cat([variables_grad, v1, loss_pos, loss_neg], dim=-1)               # :277
        new_variables = pair_norm(mlp(unit, w["update_gate"]), graph.var_graph, g_cnt) * 0.25  # :278-279
        variables = new_variables + 0.1 * variables                                      # :280

        logits = mlp(variables, w["variables_output"])                                   # :283
        per_var_loss = train_loss(labels_f, logits, ns)                                  # :289-291
        per_graph_loss = torch.zeros(g_cnt, LOGIT_MAPS, dtype=dtype).index_add_(
            0, graph.var_graph, per_var_loss * var_w[:, None])                           # :292
        sorted_desc = torch.sort(per_graph_loss, dim=-1, descending=True).values
        logit_loss = (sorted_desc * costs).sum() / costs.sum()                           # :311-315
        best_graph_map = torch.argmin(per_graph_loss, dim=-1)                            # :317 (ties -> first)
        best_map = best_graph_map[graph.var_graph]                                       # :318-320
        step_losses.append(logit_loss)                                                   # :323
        out_logits = torch.gather(logits, 1, best_map[:, None])                          # :328-329
        is_sat = is_batch_sat(out_logits, graph)                                         # :330

        if trace is not None:
            trace.append(dict(v1=v1, query=query, clauses_loss=clauses_loss, variables_grad=variables_grad,
                              var_msg=var_msg, clause_messages=clause_messages, clause_data=clause_data,
                              clause_state=clause_state, variables_loss=variables_loss,
                              update_out=None, variables=variables, logits=logits,
                              per_graph_loss=per_graph_loss, best_graph_map=best_graph_map,
                              out_logits=out_logits[:, 0], is_sat=float(is_sat), logit_loss=float(logit_loss)))
        last_logits = logits
        if float(is_sat) == 1.0:                                                         # :331-338
            break
        variables = variables * 0.2 + variables * 0.8                                    # :347
        clause_state = clause_state * 0.2 + clause_state * 0.8                           # :348

    unsupervised_loss = torch.stack(step_losses).mean() if step_losses else torch.zeros((), dtype=dtype)
    out_logits = torch.gather(last_logits, 1, best_map[:, None])[:, 0]                   # :371-372
    return out_logits, step, unsupervised_loss, last_logits, best_map


def model_call(graph, w, noise_scale, noisy_num, labels, normals, rounds=32, dtype=torch.float32, **kw):
    """``QuerySAT.diffusion_step`` -> ``{"steps_taken", "loss", "prediction"}`` (``:467-481``)."""
    out_logits, step, loss, _, _ = model_loop(graph, w, noise_scale, noisy_num, labels, normals, rounds,
                                              dtype=dtype, **kw)
    return {"steps_taken": step, "loss": loss, "prediction": out_logits}


# ------------------------------------------------------------------------------- diffusion steps
def randomized_rounding(x, uniform):
    """``floor(x[:,0:1] + U)`` -> ``[r, 1-r]``; column 0 = "variable is False"."""
    rounded = torch.floor(x[:, 0:1] + uniform.reshape(-1, 1).to(x.dtype))
    return torch.cat([rounded, 1 - rounded], dim=-1)


def reverse_distribution_step_theoretic(x, x0, t, t_increment):
    """``t`` and ``t_increment`` are Python floats as in the reference (``max`` in Python,
    ``pow`` in the tensor dtype)."""
    dtype = x.dtype
    t1 = torch.pow(torch.tensor(t, dtype=dtype), T_POWER)
    t2 = torch.pow(torch.tensor(max(0.0, t - t_increment), dtype=dtype), T_POWER)
    x_new = distribution_at_time(x0, t1)
    alpha_t = (1 - t1) / (1 - t2)
    x_unnormed = distribution_at_time(x, 1 - alpha_t) * x_new
    return x_unnormed / (x_unnormed.sum(dim=-1, keepdim=True) + 1e-8)


def graph_sat_flags(bits, graph: OracleGraph):
    """Per-graph "all clauses satisfied" of 0/1 assignments [N] (``metrics/sat_metrics.py:74-83``)."""
    lits = torch.cat([bits, 1 - bits]).to(torch.int64)
    per_clause = torch.zeros(graph.n_clauses, dtype=torch.int64).index_add_(0, graph.clause, lits[graph.lit_row])
    sat = torch.clamp(per_clause, 0, 1)
    per_graph = torch.zeros(graph.n_graphs, dtype=torch.int64).index_add_(0, graph.clause_graph, sat)
    total = torch.bincount(graph.clause_graph, minlength=graph.n_graphs)
    return per_graph == total


def _satisfiable_py(bits, clauses):
    """``VariableAssignment.satisfiable`` (``utils/VariableAssignment.py:79-90``) on a bool list."""
    for clause in clauses:
        ok = False
        for lit in clause:
            if (lit > 0) == bits[abs(lit) - 1]:
                ok = True
                break
        if not ok:
            return False
    return True


def diffusion(n_steps, graph: OracleGraph, w, uniforms, labels, normals, rounds=32, dtype=torch.float32,
              trace=None):
    """Reference ``diffusion()``.

    ``uniforms`` [n_steps, N], ``labels`` [n_steps, N] int, ``normals`` [n_steps, rounds, N, 4].
    Returns ``(mean cum_accuracy, predictions [N] of 0/1 floats, latch_step [N] ints)``.
    """
    n = graph.n_vars
    x = torch.zeros(n, 2, dtype=dtype) + 0.5                                             # :86
    fixed_step = [-1] * n
    fixed_val = [0.0] * n
    cum_accuracy = np.zeros(graph.n_graphs)
    predictions = None
    for t in range(n_steps):
        noise_scale = 1 - t / n_steps                                                    # :106
        x_noisy = randomized_rounding(x, uniforms[t])                                    # :107
        x = x_noisy                                                                      # :108-109
        out = model_call(graph, w, noise_scale, x_noisy, labels[t], normals[t], rounds, dtype=dtype)
        predictions = torch.sigmoid(out["prediction"])                                   # :61-62
        total_accuracy = graph_sat_flags(torch.round(predictions), graph)                # :119-124
        x = reverse_distribution_step_theoretic(
            x, torch.stack([1 - predictions, predictions], dim=1), noise_scale, 1 / n_steps)  # :127-129
        cum_accuracy = np.maximum(cum_accuracy, total_accuracy.numpy())                  # :130
        xx = torch.round(predictions)                                                    # :154
        shift = 0
        for cur_clauses, cur_n in zip(graph.clauses_per_graph, graph.vars_per_graph):    # :157-170
            if fixed_step[shift] >= 0:
                shift += cur_n
                continue
            vals = xx[shift:shift + cur_n]
            if _satisfiable_py([bool(b) for b in vals], cur_clauses):
                fixed_val[shift:shift + cur_n] = [float(v) for v in vals]
                fixed_step[shift:shift + cur_n] = [t] * cur_n
            shift += cur_n
        if trace is not None:
            trace.append(dict(x_noisy=x_noisy, prediction_logits=out["prediction"], predictions=predictions,
                              x=x, steps_taken=out["steps_taken"], loss=out["loss"]))
    final = torch.round(predictions).numpy().copy()                                      # :182
    for i in range(n):
        if fixed_step[i] >= 0:
            final[i] = fixed_val[i]                                                      # :183-185
    return float(np.mean(cum_accuracy)), final, np.asarray(fixed_step)


def encode_assignment(bits) -> int:
    """``VariableAssignment.__int__`` (``utils/VariableAssignment.py:63-69``)."""
    value = 0
    for pos, bit in enumerate(bits):
        if int(bit) == 1:
            value |= 1 << pos
    return value


def samples(n_samples, n_vars, clauses, w, noise_fn, chains_per_batch, n_steps=32, rounds=32,
            dtype=torch.float32, max_batches=None):
    """Reference ``DiffusionSampler.samples``: ``noise_fn(batch_index)`` returns
    ``(uniforms, labels, normals)`` for one batch of ``chains_per_batch`` chains."""
    hist, total, sat_total, needed = {}, 0, 0, n_samples
    graph = OracleGraph.copies(n_vars, clauses, chains_per_batch)
    key_len = max(abs(l) for c in clauses for l in c)        # VariableAssignment(clauses=...) :34-36
    batch = 0
    while needed > 0:
        if max_batches is not None and batch >= max_batches:
            break
        if total > 0 and sat_total / total < 0.005:                                      # :261-263
            break
        uniforms, labels, normals = noise_fn(batch)
        _, predictions, _ = diffusion(n_steps, graph, w, uniforms, labels, normals, rounds, dtype)
        batch += 1
        for i in range(chains_per_batch):                                                # :283-307
            bits = predictions[i * n_vars:(i + 1) * n_vars]
            if len(bits) > key_len:
                raise IndexError("list assignment index out of range")   # as assign_all_from_bit_list would
            padded = [int(b) == 1 for b in bits] + [False] * (key_len - len(bits))
            total += 1
            if _satisfiable_py(padded, clauses):
                sat_total += 1
                key = encode_assignment(padded)
                hist[key] = hist.get(key, 0) + 1
                needed -= 1
                if needed == 0:
                    break
    return hist
