"""One round on the default path (DSAT_F32_TC), stage by stage, against fp64 restatements of each operation.

Every case binds a graph, writes random per-row state (rows of different magnitude) into VROW[:, :F] and CROW[:, :F],
reads it back (a write onto the hi/lo planes rounds it), runs one round with injected normals and reads every buffer the
round leaves.  Each stage is then restated in fp64 (the oracle's building blocks: ``OracleGraph.clause_from_lit`` /
``lit_from_clause``, ``degree_weights``, ``query_gradient_analytic``, ``pair_norm``, ``train_loss``) on the buffers the
device itself fed that stage, so errors do not carry from one stage to the next, and compared element-wise.

Bounds (u = 2^-24, the fp32 unit roundoff; first-order error analysis of the kernels' fp32 operations; CUDA's expf,
rsqrtf are within 2 ulp = 4u relative, logf and log1pf within 1 ulp = 2u; the host's weights 1/sqrtf(d) within 2u):

* hi/lo planes: a value v stored as hi = bf16(v), lo = bf16(v - hi) reads back within 2^-16 |v| (two roundings to 8
  significant bits), so every plane output adds PLANE * |value| with PLANE = 2^-16.
* noise: VROW[:, F:F+9] = [normals | noisy | noise_scale | 0 0]; split onto the planes, so within PLANE * |value|.
* sums: a k-term fp32 sum in any association is within k u sum|terms| of the exact one.  Clause messages
  rev_w * sum LIT and literal losses deg_w * sum COUT: (k + 3) u w sum|terms| (the sum, the weight's 2u, the product).
* 4 exp(-S): S within k u S, expf within 4u, so within ((1 + 4u) exp(k u S) - 1) of the value.
* gradient (-sigma(q) S+ + sigma(-q) S-) vw: the terms cancel, so the bound is relative to
  A = sigma(q) S+ + sigma(-q) S-: S+- sum 2k hi and lo plane entries (2k u), sigmoid_f is within 6u (expf 4u, the add and
  the division u each), the two products, the difference and the weight add 5u: (2 kmax + 11) u vw A.
* PairNorm (per graph mean over n rows, then per row x / sqrt(mean_f(x^2) + 1e-6)): the fp32 column mean is within
  dmu = (n + 18) u mean|x| (products by the rounded 1/n, and a summation tree at most n + 16 additions deep: the
  thread groups of the shared-memory kernel or the warps of the generic one).  With Delta = max over the row's columns
  of dmu and sigma the row's exact standard deviation, the normalized value y is off by at most
  (dmu + |y| Delta) / (sigma - Delta), plus (F/2 + 9) u |y| for the subtraction, the sum of squares (F terms; halved by
  the square root), rsqrtf and the product.  new = 0.25 y + 0.1 old adds u (0.1 |old| + |new|); the carry
  new * 0.2 + new * 0.8 adds 3u |carried| (the fp32 constants 0.1, 0.2, 0.8 are restated as the kernels use them).
* head: per-variable KL(pa || pb) with pa = y(1 - ts) + ts/2, pb = sigmoid(z)(1 - t) + t/2 (t = 0.5 exactly; the fp32
  ts is within u of fp64's).  pa is within 2u, qa = 1 - pa within 3u, pb within 8u pb; through the logarithms, the
  differences, the products and the sum this gives
  e_kl = u (14 + 8 pb/(1 - pb) + 8 (|log pa| + |log pb| + |log1p(-pa)| + |log1p(-pb)|) + 3 (|t1| + |t2|)).
  The normalizer carries e_kl(ts/2, 1/2)/norm + 2u relative; the division, the 1/n weight and its product 3u; the graph
  sum n u.  Graph maps are compared where every other map's loss is above the best one's by more than both bounds;
  OUT must equal the selected logit bit for bit; graph_sat is exact (bits of OUT with |OUT| > 2^-20, where
  sigmoid_f(z) > 0.5 is z > 0); the group loss sum adds the sort (1-Lipschitz), the 8-term weighted sum (7u), the group sum
  and the division by 204.

Plan coverage: no device hook reports the chosen kernels, so the host rules of dsat_api.cu that pick them
(``pick_slice_width``, ``idx_fits``, the 112 KB cutoffs, the ``n_graphs != 1`` rule, ``launch_pairnorm_smem``'s thread
and fit rule) are restated here and ``test_cases_reach_every_plan`` (CPU) checks that CASES reach every cell of the plan
table for F = Q = 128 and F = Q = 64.  Unreachable by construction: slice width 128 when Q = 64 (the width must divide
Q).  The L2 gathers' row cursor steps inside a chain in ``big``: its 43000 clause and 10000 variable rows per chain exceed
the grid's warps (at most 2048 threads per SM = 8 blocks of 8 warps on 148 SMs = 9472 warps).
"""
import numpy as np
import pytest
import torch

from diffusionsat_b200 import _lib, graph as G, synth
from oracle import querysat_oracle as O
from tests import helpers as H

U = 2.0 ** -24
PLANE = 2.0 ** -16
AUX = 16
NOISE_SCALE = 0.25                      # t = sqrt(0.25) = 0.5 exactly in fp32 and fp64
C01, C02, C08 = (float(np.float32(c)) for c in (0.1, 0.2, 0.8))
KB = 1024


# ----------------------------------------------------------------------------------- plan rules (dsat_api.cu)
def pick_slice_width(table_rows, Q, budget_kb, elt_bytes):
    for budget in (budget_kb, 220):
        for w in (128, 64, 32):
            if w > Q or Q % w:
                continue
            b = 2 * table_rows * w * elt_bytes
            if b <= budget * KB:
                return w, b
    return 0, 0


def idx_fits(table_bytes, idx_vecs):
    if idx_vecs <= 0:
        return False
    sm, reserved, with_idx = 227 * KB, 1024, table_bytes + idx_vecs * 16
    if with_idx + reserved > sm:
        return False
    return sm // (with_idx + reserved) == sm // (table_bytes + reserved)


def idx16_vecs(n, m, nnz):
    """16-byte lengths of the 16-bit adjacency blocks dsat_set_graph stages (0 when an index does not fit 16 bits)."""
    if not (nnz < 65536 and 2 * n < 65536 and m < 65536):
        return 0, 0
    pad8 = lambda x: (x + 7) // 8 * 8
    return (pad8(m + 1) + pad8(nnz)) // 8, (pad8(2 * n + 1) + pad8(nnz) + pad8(n)) // 8


def gather_plans(n, m, nnz, n_graphs, Q):
    """(clause gather, literal gather): ("smem", W, SI) or ("L2",)."""
    cl_vecs, lit_vecs = idx16_vecs(n, m, nnz)
    plans = []
    for rows, budget, elt, vecs in ((2 * n, 110, 4, cl_vecs), (m, 112, 2, lit_vecs)):
        w, b = pick_slice_width(rows, Q, budget, elt)
        plans.append(("L2",) if n_graphs != 1 or not w or b > 112 * KB else ("smem", w, idx_fits(b, vecs)))
    return tuple(plans)


def pairnorm_plan(max_graph_rows, F):
    """launch_pairnorm_smem: ("smem", threads) or ("generic",) when the largest graph does not fit."""
    row_bytes = max_graph_rows * F * 4
    threads = 1024 if row_bytes > 100 * KB else 512 if row_bytes > 48 * KB else 256
    groups = max(threads // F, 1)
    return ("smem", threads) if (F + groups * F) * 4 + row_bytes <= 227 * KB else ("generic",)


def plan_of(formulas, F, Q):
    n = sum(f[0] for f in formulas)
    m = sum(len(f[1]) for f in formulas)
    nnz = sum(len(c) for f in formulas for c in f[1])
    cg, lg = gather_plans(n, m, nnz, len(formulas), Q)
    return {"clause_gather": cg, "literal_gather": lg,
            "pairnorm_clause": pairnorm_plan(max(len(f[1]) for f in formulas), F),
            "pairnorm_var": pairnorm_plan(max(f[0] for f in formulas), F)}


def plan_cells(F, Q):
    widths = [w for w in (128, 64, 32) if w <= Q and Q % w == 0]
    cells = set()
    for stage in ("clause_gather", "literal_gather"):
        cells |= {(stage, ("smem", w, si)) for w in widths for si in (True, False)} | {(stage, ("L2",))}
    for stage in ("pairnorm_clause", "pairnorm_var"):
        cells |= {(stage, ("smem", t)) for t in (256, 512, 1024)} | {(stage, ("generic",))}
    return cells


# ------------------------------------------------------------------------------------------------- cases
def odd_formula(n, m, seed):
    """Clause lengths 1..8 (every remainder of the edge unrolls), repeated literals, an empty clause, variable n in no
    clause, variable 1 in 45 clauses."""
    rng = np.random.default_rng(seed)
    clauses = []
    for j in range(m - 1):
        k = int(rng.integers(1, 9))
        vs = rng.integers(1, n, size=k)                 # variables 1..n-1: variable n keeps degree 0
        c = [int(v) if rng.random() < 0.5 else -int(v) for v in vs]
        if j % 7 == 0:
            c.append(c[0])                              # a repeated literal
        if j < 45:
            c.append(1 if j % 2 else -1)
        clauses.append(c)
    clauses.insert(m // 2, [])
    return n, clauses


def _3sat(n, m, seed=0, k=3):
    return synth.random_3sat(n, m, seed=seed, k=k)


def _ksat(n, m, seed=0):
    return synth.random_ksat_mixed(n, m, seed=seed)


# name -> (formulas builder, chains, F, Q, options); the comment is the plan at F = Q = 128 (clause / literal gather)
CASES = {
    "w128_w128": (lambda: [_3sat(30, 128, 1)], 5, 128, 128, {}),
    "odd_w128": (lambda: [odd_formula(40, 100, 2)], 3, 128, 128, {}),
    "w128_w64": (lambda: [_ksat(50, 300, 3)], 7, 128, 128, {}),
    "w64_w64": (lambda: [_3sat(100, 428, 4)], 13, 128, 128, {}),
    "odd_w32_w32": (lambda: [odd_formula(150, 640, 5)], 3, 128, 128, {}),
    "uf250": (lambda: [_3sat(250, 1065, 250)], 3, 128, 128, {}),
    "n500": (lambda: [_3sat(500, 2129, 6)], 2, 128, 128, {}),
    # idx_fits false: the staged adjacency would cost a resident CTA
    "noidx_c128": (lambda: [_ksat(22, 44, 7)], 5, 128, 128, {}),
    "noidx_c64": (lambda: [_ksat(71, 426, 8)], 3, 128, 128, {}),
    "noidx_l64": (lambda: [_3sat(40, 296, 9)], 5, 128, 128, {}),
    "noidx_c32_l128": (lambda: [_ksat(111, 222, 10)], 3, 128, 128, {}),
    "noidx_l32": (lambda: [_ksat(93, 558, 11)], 3, 128, 128, {}),
    "big": (lambda: [_3sat(10000, 43000, 5)], 2, 128, 128, {}),
    "union_small": (lambda: [_3sat(30, 128, 12), (1, [[1]]), _ksat(12, 40, 13), odd_formula(20, 50, 14)], 3, 128, 128, {}),
    "union_generic": (lambda: [_3sat(500, 2129, 15), (1, [[-1]]), _ksat(20, 60, 16)], 2, 128, 128, {}),
    "f128_q64": (lambda: [_ksat(50, 300, 17)], 5, 128, 64, {}),
    "f64_q128": (lambda: [_ksat(50, 300, 18)], 5, 64, 128, {}),
    "bias_w64": (lambda: [_3sat(100, 428, 19)], 4, 128, 128, {"bias": 30.0}),
    "bias_uf250": (lambda: [_3sat(250, 1065, 20)], 2, 128, 128, {"bias": 30.0}),
    # F = Q = 64
    "q64_w64": (lambda: [_3sat(100, 428, 21)], 7, 64, 64, {}),
    "q64_odd_w32": (lambda: [odd_formula(150, 640, 22)], 3, 64, 64, {}),
    "q64_uf250": (lambda: [_3sat(250, 1065, 23)], 3, 64, 64, {}),
    "q64_n500": (lambda: [_3sat(500, 2129, 24)], 2, 64, 64, {}),
    "q64_n1000": (lambda: [_3sat(1000, 4258, 25)], 2, 64, 64, {}),
    "q64_c512": (lambda: [_3sat(60, 256, 26)], 5, 64, 64, {}),
    "q64_noidx_c64": (lambda: [_3sat(21, 89, 27)], 5, 64, 64, {}),
    "q64_noidx_l64": (lambda: [_3sat(20, 40, 28)], 5, 64, 64, {}),
    "q64_noidx_c32": (lambda: [_3sat(111, 222, 29)], 3, 64, 64, {}),
    "q64_noidx_l32": (lambda: [_ksat(93, 558, 30)], 3, 64, 64, {}),
}

# group_graphs = 1 on formulas most assignments satisfy: some chains finish in round 0 and are skipped in round 1
SKIP_CASES = {
    "skip_smem": (lambda: [(3, [[1, 2, 3]])], 48, 128, 128, {}),
    "skip_l2": (lambda: [_3sat(250, 1065, 31, k=10)], 16, 128, 128, {}),
}


# ------------------------------------------------------------------------------------------ device side
def bind(ctx, spec, seed, group):
    build, chains, F, Q, opts = spec
    formulas = build()
    wts = H.make_weights(F, Q, seed=40 + seed, bias_scale=0.1)
    if opts.get("bias"):            # large offsets on the PairNorm inputs: the last layers of clause_update (columns Q:)
        rng = np.random.default_rng(seed)                               # and of update_gate
        k, b = wts.layers["clause_update/1"]
        b = b.copy(); b[Q:] += opts["bias"] * rng.choice([-1.0, 1.0], F).astype(np.float32)
        wts.layers["clause_update/1"] = (k, b)
        k, b = wts.layers["update_gate/2"]
        wts.layers["update_gate/2"] = (k, b + opts["bias"] * rng.choice([-1.0, 1.0], F).astype(np.float32))
    ctx.set_model(wts)
    ctx.set_precision(_lib.F32_TC)
    ctx.set_graph(G.build_union_graph(formulas), chains=chains, group_graphs=group)
    assert ctx.get_precision() == _lib.F32_TC
    return formulas, chains, F, Q


def write_state(ctx, rng, F):
    """Random state of different magnitude per row into VROW[:, :F] and CROW[:, :F]; returns what the device holds."""
    state = {}
    for name in ("VROW", "CROW"):
        buf = ctx.debug_read(name)
        x = rng.standard_normal((buf.shape[0], F)) * rng.uniform(0.05, 4.0, (buf.shape[0], 1))
        buf[:, :F] = x.astype(np.float32)
        ctx.debug_write(name, buf)
        state[name] = ctx.debug_read(name)[:, :F].astype(np.float64)
    return state


def run_round(ctx, rng, round_index, n_rows):
    normals = rng.standard_normal((n_rows, 4)).astype(np.float32)
    ctx.debug_round(round_index, normals)
    bufs = {k: ctx.debug_read(k) for k in ("VROW", "CROW", "QS", "LIT", "COUT", "UOUT", "SPRE", "LOGITS", "OUT")}
    bufs["normals"] = normals
    bufs["groups"] = ctx.debug_groups()
    return bufs


# ------------------------------------------------------------------------------------------ checks
def within(name, got, want, bound, rows=None):
    got = np.asarray(got, dtype=np.float64)
    want = np.broadcast_to(np.asarray(want, dtype=np.float64), got.shape)
    bound = np.broadcast_to(np.asarray(bound, dtype=np.float64), got.shape)
    if rows is not None:
        got, want, bound = got[rows], want[rows], bound[rows]
    err = np.abs(got - want)
    bad = ~(err <= bound)
    if bad.any():
        i = np.unravel_index(np.argmax(np.where(bad, err / np.maximum(bound, 1e-300), 0)), bad.shape)
        raise AssertionError("%s: %d of %d elements outside the bound; at %r got %.9g want %.9g (error %.3g, bound %.3g)" % (
            name, int(bad.sum()), bad.size, tuple(int(j) for j in i), got[i], want[i], err[i], bound[i]))


def t64(x):
    return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64))


def plane_bound(err, want):
    return err + PLANE * (np.abs(want) + err)


def check_noise(b, noisy, F, rows):
    want = np.concatenate([b["normals"], noisy, np.full((len(noisy), 1), NOISE_SCALE), np.zeros((len(noisy), 2))], axis=1)
    within("noise columns", b["VROW"][:, F:F + 9], want, PLANE * np.abs(want), rows)


def check_clause_gather(b, og, F, Q, rows):
    _, k, _, _, rev_w = (t.numpy() for t in O.degree_weights(og, torch.float64))
    lit, qs = t64(b["LIT"]), t64(b["QS"])
    literals = torch.cat([lit[:, :Q], lit[:, Q:]], dim=0)
    want = og.clause_from_lit(literals).numpy() * rev_w
    err = rev_w * (k + 3) * U * og.clause_from_lit(literals.abs()).numpy()
    within("clause messages", b["CROW"][:, F:F + Q], want, plane_bound(err, want), rows)
    s = og.clause_from_lit(torch.cat([qs[:, Q:2 * Q], qs[:, 2 * Q:]], dim=0)).numpy()
    want = 4.0 * np.exp(-s)
    err = want * ((1 + 4 * U) * np.exp(k * U * np.abs(s)) - 1)
    within("4*clauses_loss", b["CROW"][:, F + Q:], want, plane_bound(err, want), rows)


def check_literal_gather(b, og, F, Q, rows):
    deg, _, deg_w, vdeg_w, _ = (t.numpy() for t in O.degree_weights(og, torch.float64))
    n = og.n_vars
    cl4, q = b["CROW"][:, F + Q:].astype(np.float64), b["QS"][:, :Q].astype(np.float64)
    want = (O.query_gradient_analytic(t64(q), t64(cl4 / 4), og) * t64(vdeg_w)).numpy()
    s = og.lit_from_clause(t64(np.abs(cl4))).numpy()
    sig = 1 / (1 + np.exp(-q))
    a = sig * s[:n] + (1 - sig) * s[n:]
    err = vdeg_w / 4 * (2 * np.maximum(deg[:n], deg[n:]) + 11) * U * a
    col = F + AUX
    within("variables_grad", b["VROW"][:, col:col + Q], want, plane_bound(err, want), rows)
    msg = t64(b["COUT"][:, :Q])
    want = og.lit_from_clause(msg).numpy() * deg_w
    err = deg_w * (deg + 3) * U * og.lit_from_clause(msg.abs()).numpy()
    bound = plane_bound(err, want)
    within("loss_pos", b["VROW"][:, col + Q:col + 2 * Q], want[:n], bound[:n], rows)
    within("loss_neg", b["VROW"][:, col + 2 * Q:col + 3 * Q], want[n:], bound[n:], rows)


def pairnorm_want(x, old, graph_ids, n_graphs):
    """fp64 PairNorm + residual + carry of the device's input rows and their bounds: (new, bound, carried, bound)."""
    F = x.shape[1]
    gid = graph_ids
    y = O.pair_norm(t64(x), gid, n_graphs).numpy()
    w = O.graph_norm_weights(gid, n_graphs, torch.float64)
    cnt = torch.bincount(gid, minlength=n_graphs).numpy().astype(np.float64)
    mean_abs = torch.zeros(n_graphs, F, dtype=torch.float64).index_add_(0, gid, t64(np.abs(x)) * w[:, None]).numpy()
    mean = torch.zeros(n_graphs, F, dtype=torch.float64).index_add_(0, gid, t64(x) * w[:, None]).numpy()
    g = gid.numpy()
    dmu = ((cnt + 18) * U)[:, None] * mean_abs
    dmu_r = dmu[g]
    delta = dmu_r.max(axis=1, keepdims=True)
    d = x - mean[g]
    sigma = np.sqrt(np.mean(d * d, axis=1, keepdims=True) + O.PAIRNORM_EPS)
    assert (delta < sigma).all(), "the mean's error bound reaches a row's standard deviation"
    dy = (dmu_r + np.abs(y) * delta) / (sigma - delta) + (F / 2 + 9) * U * np.abs(y)
    new = 0.25 * y + C01 * old
    dnew = 0.25 * dy + U * (C01 * np.abs(old) + np.abs(new))
    carried = new * C02 + new * C08
    dcar = dnew * (C02 + C08) + 3 * U * np.abs(carried)
    return new, plane_bound(dnew, new), carried, plane_bound(dcar, carried)


def check_pairnorms(b, before, og, F, Q, rows_v, rows_c):
    _, _, carried, bound = pairnorm_want(b["COUT"][:, Q:].astype(np.float64), before["CROW"], og.clause_graph, og.n_graphs)
    within("clause PairNorm (carried state)", b["CROW"][:, :F], carried, bound, rows_c)
    new, nbound, carried, bound = pairnorm_want(b["UOUT"].astype(np.float64), before["VROW"], og.var_graph, og.n_graphs)
    within("variable PairNorm (SPRE)", b["SPRE"], new, nbound, rows_v)
    within("variable PairNorm (carried state)", b["VROW"][:, :F], carried, bound, rows_v)


def kl_error(pa, pb):
    la, lb, l1a, l1b = np.log(pa), np.log(pb), np.log1p(-pa), np.log1p(-pb)
    t1, t2 = pa * (la - lb), (1 - pa) * (l1a - l1b)
    return t1 + t2, U * (14 + 8 * pb / (1 - pb) + 8 * (np.abs(la) + np.abs(lb) + np.abs(l1a) + np.abs(l1b))
                         + 3 * (np.abs(t1) + np.abs(t2)))


def check_head(b, og, unit, chains, labels, graphs, groups_before=None, loss_before=None):
    """`graphs`: bool per graph, which graphs the round computed."""
    z = b["LOGITS"][:, :8].astype(np.float64)
    lab = labels.astype(np.float64)[:, None]
    per_var = O.train_loss(t64(np.repeat(lab, 8, axis=1)), t64(z), torch.tensor(NOISE_SCALE, dtype=torch.float64)).numpy()
    t = np.sqrt(NOISE_SCALE)
    ts = min(t + 0.01, 1.0)
    kl, e_kl = kl_error(lab * (1 - ts) + ts / 2, (1 / (1 + np.exp(-z))) * (1 - t) + t / 2)
    norm, e_norm = kl_error(np.float64(ts / 2), np.float64(0.5))
    norm += 1e-4
    e_v = (e_kl + (3 * U + e_norm / norm + 2 * U) * np.abs(kl)) / norm
    G_ = og.n_graphs
    w = O.graph_norm_weights(og.var_graph, G_, torch.float64)
    cnt = torch.bincount(og.var_graph, minlength=G_).numpy().astype(np.float64)
    gsum = lambda v: torch.zeros(G_, 8, dtype=torch.float64).index_add_(0, og.var_graph, t64(v) * w[:, None]).numpy()
    pgl = gsum(per_var)
    e_g = gsum(e_v) + cnt[:, None] * U * gsum(np.abs(kl) / norm)
    best = np.argmin(pgl, axis=1)
    pb_, eb = pgl[np.arange(G_), best][:, None], e_g[np.arange(G_), best][:, None]
    others = np.arange(8)[None, :] != best[:, None]
    clear = np.all(~others | (pgl - pb_ > e_g + eb), axis=1) & graphs
    got = b["groups"]
    assert clear.sum() >= 0.5 * graphs.sum(), "only %d of %d graphs have a clear best logit map" % (clear.sum(), graphs.sum())
    np.testing.assert_array_equal(got["graph_map"][clear], best[clear], err_msg="graph_map")
    # OUT is the selected map's logit, bit for bit
    gmap_v = got["graph_map"][og.var_graph.numpy()]
    vrows = graphs[og.var_graph.numpy()]
    sel = b["LOGITS"][np.arange(len(gmap_v)), gmap_v]
    np.testing.assert_array_equal(b["OUT"][vrows, 0].view(np.uint32), sel[vrows].view(np.uint32), err_msg="OUT")
    # graph_sat: clauses of each graph under the bits of OUT
    out = b["OUT"][:, 0]
    bits = out > 0
    n, m = unit.n_vars, unit.n_clauses
    codes = unit.cl_lit.astype(np.int64)
    cl_of_edge = np.repeat(np.arange(m), np.diff(unit.cl_rowptr))
    sat = np.zeros(G_, dtype=bool)
    for c in range(chains):
        true_lit = bits[c * n + (codes >> 1)] != (codes & 1).astype(bool)
        per_clause = np.bincount(cl_of_edge, weights=true_lit, minlength=m) > 0
        for lg in range(unit.n_graphs):
            sat[c * unit.n_graphs + lg] = per_clause[unit.clause_seg[lg]:unit.clause_seg[lg + 1]].all()
    clear_bits = np.array([(np.abs(out[og.var_graph.numpy() == gi]) > 2.0 ** -20).all() for gi in range(G_)])
    check = graphs & clear_bits
    assert check.sum() >= 0.9 * graphs.sum()
    np.testing.assert_array_equal(got["graph_sat"][check], sat[check], err_msg="graph_sat")
    # loss sum of each group: sum over its graphs of sum(sort_desc(loss) * (k+1)^2) / 204
    costs = (np.arange(1, 9) ** 2).astype(np.float64)
    srt = -np.sort(-pgl, axis=1)
    gl = (srt * costs).sum(axis=1) / 204
    egl = e_g.max(axis=1) + 7 * U * (np.abs(srt) * costs).sum(axis=1) / 204
    per_group = len(got["loss_sum"])
    gg = G_ // per_group
    want = gl.reshape(per_group, gg).sum(axis=1)
    err = egl.reshape(per_group, gg).sum(axis=1) + (gg + 1) * U * np.abs(gl).reshape(per_group, gg).sum(axis=1)
    live = graphs.reshape(per_group, gg).all(axis=1)
    if loss_before is not None:
        want = want + loss_before
        err = err + U * np.abs(want)
    within("group loss sum", got["loss_sum"][live], want[live], err[live])


def oracle_graph(formulas, chains):
    return O.OracleGraph.from_formulas([(n, [list(c) for c in cl]) for n, cl in formulas] * chains)


def check_round(b, before, og, unit, chains, F, Q, noisy, labels, live_chains, loss_before=None):
    n, m = unit.n_vars, unit.n_clauses
    rows_v = np.repeat(live_chains, n)
    rows_c = np.repeat(live_chains, m)
    check_noise(b, noisy, F, rows_v)
    check_clause_gather(b, og, F, Q, rows_c)
    check_literal_gather(b, og, F, Q, rows_v)
    check_pairnorms(b, before, og, F, Q, rows_v, rows_c)
    check_head(b, og, unit, chains, labels, np.repeat(live_chains, unit.n_graphs), loss_before=loss_before)


def start(ctx, spec, seed, group=0):
    formulas, chains, F, Q = bind(ctx, spec, seed, group)
    unit = ctx.graph
    rng = np.random.default_rng(100 + seed)
    n_rows = unit.n_vars * chains
    noisy = np.zeros((n_rows, 2), dtype=np.float32)
    noisy[np.arange(n_rows), rng.integers(0, 2, n_rows)] = 1.0
    labels = rng.integers(0, 2, n_rows).astype(np.int32)
    ctx.debug_begin(NOISE_SCALE, noisy, labels)
    before = write_state(ctx, rng, F)
    return formulas, chains, F, Q, unit, rng, noisy, labels, before


# ------------------------------------------------------------------------------------------------- tests
def test_cases_reach_every_plan():
    for fq in (128, 64):
        reached = set()
        for build, _, F, Q, _ in list(CASES.values()) + list(SKIP_CASES.values()):
            if F == fq and Q == fq:
                reached |= set(plan_of(build(), F, Q).items())
        missing = plan_cells(fq, fq) - reached
        assert not missing, "F = Q = %d: no case reaches %s" % (fq, sorted(missing))


def test_plan_rules_pin_the_documented_shapes():
    """The shapes the kernels' comments and the README quote land where they say."""
    assert plan_of([(30, [[1, 2, 3]] * 128)], 128, 128)["clause_gather"][:2] == ("smem", 128)
    assert plan_of([(100, [[1, 2, 3]] * 428)], 128, 128)["literal_gather"][:2] == ("smem", 64)
    uf250 = plan_of([(250, [[1, 2, 3]] * 1065)], 128, 128)
    assert uf250 == {"clause_gather": ("L2",), "literal_gather": ("L2",), "pairnorm_clause": ("generic",),
                     "pairnorm_var": ("smem", 1024)}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_round_stages(ctx, case):
    formulas, chains, F, Q, unit, rng, noisy, labels, before = start(ctx, CASES[case], list(CASES).index(case))
    b = run_round(ctx, rng, 0, unit.n_vars * chains)
    og = oracle_graph(formulas, chains)
    check_round(b, before, og, unit, chains, F, Q, noisy, labels, np.ones(chains, dtype=bool))


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(SKIP_CASES))
def test_finished_groups_are_skipped(ctx, case):
    """Round 0 finishes some one-chain groups; in round 1 their rows and OUT stay bit-identical and the live chains
    still pass every stage check."""
    formulas, chains, F, Q, unit, rng, noisy, labels, before = start(ctx, SKIP_CASES[case], 50 + list(SKIP_CASES).index(case), group=1)
    og = oracle_graph(formulas, chains)
    n_rows = unit.n_vars * chains
    b0 = run_round(ctx, rng, 0, n_rows)
    check_round(b0, before, og, unit, chains, F, Q, noisy, labels, np.ones(chains, dtype=bool))
    done = b0["groups"]["done"].astype(bool)
    assert 0 < done.sum() < chains, "round 0 finished %d of %d chains: nothing to skip or nothing live" % (done.sum(), chains)
    before1 = {"VROW": b0["VROW"][:, :F].astype(np.float64), "CROW": b0["CROW"][:, :F].astype(np.float64)}
    b1 = run_round(ctx, rng, 1, n_rows)
    for name, rows in (("VROW", unit.n_vars), ("CROW", unit.n_clauses), ("SPRE", unit.n_vars), ("OUT", unit.n_vars)):
        fin = np.repeat(done, rows)
        np.testing.assert_array_equal(b1[name][fin].view(np.uint32), b0[name][fin].view(np.uint32),
                                      err_msg="%s rows of finished chains changed" % name)
    np.testing.assert_array_equal(b1["groups"]["loss_sum"][done], b0["groups"]["loss_sum"][done])
    check_round(b1, before1, og, unit, chains, F, Q, noisy, labels, ~done, loss_before=b0["groups"]["loss_sum"])
