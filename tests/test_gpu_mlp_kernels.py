"""Every whole-MLP kernel on its own (dsat_debug_mlp: input rows + packed weights -> output) against an fp64
restatement of reference model/mlp.py:42-50 (Dense = x @ kernel + bias, hidden activation leaky_relu 0.2), element-wise.

* fp32-accurate tensor-core path (DSAT_F32_TC, the default) and the CUDA-core fp32 path: |got - want| <= 2e-4 |want| +
  1e-4 rms(want row) per element (the reference's own fp32 arithmetic sits at ~1e-6 of the row's magnitude, the
  split-bf16 products at ~1e-5; the absolute term is per ROW because the rows are scaled differently).
* bf16 path: the fp64 chain rounds to bf16 exactly where the kernel does (operands, hidden activations after the bias add,
  leaky relu on bf16 values, outputs); 2e-3 |want| + 2e-3 rms for at least 99 % of the elements (half a bf16 ulp), and
  one bf16 ulp (8e-3) for every element: an accumulator within rounding distance of a bf16 tie may round the other way.

Shapes (SHAPES), each of which selects other kernel plans:
* bench: n = 100, m = 428 (the bench formula's shape) with 700 chains: 547 variable tiles and 2341 clause tiles, so every
  persistent CTA (or CTA pair) loops over several tiles, rings wrap, and the last tile is partial;
* one_tile: n = 20 with one chain, at most 128 rows per MLP: the single-CTA instantiations (split, x3 and whole-MLP);
* f128_q64: feature_maps 128, query_maps 64: the literal MLP through the resident-input fused_mlp_kernel (hidden 256);
* lit_hidden_384 (bf16 only; the fp32-accurate kernels tile hidden widths of at most 256 or multiples of 256): hidden
  layers wider than 256 columns without split mode.
The reference values are computed for rows drawn from the first, middle and last tiles and a random subset."""
import numpy as np
import pytest

from diffusionsat_b200 import _lib, graph as G, synth
from tests import helpers as H

pytestmark = pytest.mark.gpu

SHAPES = {   # name -> (variables, chains, feature_maps, query_maps, literal hidden width (None = 4 query_maps))
    "bench": (100, 700, 128, 128, None),
    "one_tile": (20, 1, 128, 128, None),
    "f128_q64": (100, 70, 128, 64, None),
    "lit_hidden_384": (100, 70, 128, 128, 384),
}
FP32_SHAPES = ("bench", "one_tile", "f128_q64")


def mlps(F, Q):
    """name -> (input buffer, output buffer, output columns)"""
    return {"variables_query": ("VROW", "QS", 3 * Q), "lit_query": ("VROW", "LIT", 2 * Q),
            "clause_update": ("CROW", "COUT", Q + F), "update_gate": ("VROW", "UOUT", F),
            "variables_output": ("SPRE", "LOGITS", 8)}


def sample_rows(rows, rng):
    picks = [np.arange(0, min(rows, 160)), np.arange(max(rows // 2 - 100, 0), min(rows // 2 + 100, rows)),
             np.arange(max(rows - 200, 0), rows), rng.integers(0, rows, 400)]
    return np.unique(np.concatenate(picks))


def lrelu(x):
    return np.maximum(x, 0.2 * x)


def softplus64(x):
    return np.maximum(x, 0.0) + np.log1p(np.exp(-np.abs(x)))


def reference_fp64(name, x, wts):
    """fp64 chain of one MLP on the reference's column order; x is in the kernels' packed row layout."""
    F, Q = wts.feature_maps, wts.query_maps
    layers = wts.mlp(name)
    if name in ("variables_query", "lit_query"):
        h = x[:, :F + 9]
    elif name == "update_gate":      # packed [variables F | aux16 | grad Q | loss+ Q | loss- Q] -> reference [grad | v1 | loss+ | loss-]
        h = np.concatenate([x[:, F + 16:F + 16 + Q], x[:, :F + 9], x[:, F + 16 + Q:]], axis=1)
    else:
        h = x
    h = h.astype(np.float64)
    for i, (w, b) in enumerate(layers):
        h = h @ w.astype(np.float64) + b.astype(np.float64)
        if i + 1 < len(layers):
            h = lrelu(h)
    if name == "variables_query":
        h = np.concatenate([h, softplus64(h), softplus64(-h)], axis=1)
    return h


def reference_bf16_chain(name, x, wts):
    """The same chain with bf16 rounding at the kernel's rounding points (dsat_mlp_fused.cuh)."""
    r = H.bf16_round
    F, Q = wts.feature_maps, wts.query_maps
    layers = wts.mlp(name)
    if name in ("variables_query", "lit_query"):
        h = x[:, :F + 9]
    elif name == "update_gate":
        h = np.concatenate([x[:, F + 16:F + 16 + Q], x[:, :F + 9], x[:, F + 16 + Q:]], axis=1)
    else:
        h = x
    h = r(h).astype(np.float64)
    for i, (w, b) in enumerate(layers):
        acc = h @ r(w).astype(np.float64) + b.astype(np.float64)
        if i + 1 < len(layers):
            hb = r(acc).astype(np.float64)                     # bias add in fp32, one rounding to bf16
            h = np.maximum(hb, r(hb * float(r(np.float32(0.2))))).astype(np.float64)    # leaky relu on bf16 values
        else:
            h = acc
    if name == "variables_query":
        h = np.concatenate([h, softplus64(h), softplus64(-h)], axis=1)
    if name != "variables_output":                             # logits stay fp32, every other output is stored as bf16
        h = r(h).astype(np.float64)
    return h


def run_case(ctx, precision, shape, seed=0):
    n_vars, chains, F, Q, lit_hidden = SHAPES[shape]
    _, clauses = synth.random_3sat(n_vars, seed=3)
    if shape == "one_tile":
        assert len(clauses) <= 128
    wts = H.make_weights(F, Q, seed=31 + seed, bias_scale=0.1, lit_hidden=lit_hidden)
    ctx.set_model(wts)
    ctx.set_precision(precision)
    ctx.set_graph(G.build_unit_graph(n_vars, clauses), chains=chains, group_graphs=0)
    rng = np.random.default_rng(seed)
    checked = {}
    for name, (src, dst, out_cols) in mlps(F, Q).items():
        rows, ld = ctx.debug_dims(src)
        x = rng.standard_normal((rows, ld)).astype(np.float32)
        if src == "VROW":
            x[:, F + 9:F + 16] = 0.0                           # aux padding columns are zero by construction
        x *= rng.uniform(0.2, 2.0, size=(rows, 1)).astype(np.float32)      # rows of different magnitude
        ctx.debug_write(src, x)
        ctx.debug_mlp(name)
        got = ctx.debug_read(dst)[:, :out_cols].astype(np.float64)
        pick = sample_rows(rows, rng)
        checked[name] = (got[pick], x[pick], wts)
    return checked


@pytest.mark.parametrize("precision", ["fp32", "fp32_simt"])
def test_fp32_mlp_kernels_elementwise(ctx, precision):
    for shape in FP32_SHAPES:
        for name, (got, x, wts) in run_case(ctx, _lib.PRECISIONS[precision], shape).items():
            want = reference_fp64(name, x, wts)
            rms = float(np.sqrt(np.mean(want ** 2)))
            bound = 2e-4 * np.abs(want) + 1e-4 * np.sqrt(np.mean(want ** 2, axis=1, keepdims=True))
            bad = np.abs(got - want) > bound
            assert not bad.any(), "%s (%s, %s): %d of %d elements off, worst %.3e at value %.3e (rms %.3e)" % (
                name, precision, shape, int(bad.sum()), bad.size, float(np.abs(got - want).max()),
                float(want[np.unravel_index(np.argmax(np.abs(got - want)), want.shape)]), rms)


def test_bf16_mlp_kernels_elementwise(ctx):
    for shape in SHAPES:
        for name, (got, x, wts) in run_case(ctx, _lib.BF16, shape).items():
            want = reference_bf16_chain(name, x, wts)
            rms = float(np.sqrt(np.mean(want ** 2)))
            err = np.abs(got - want)
            tight = err <= 2e-3 * np.abs(want) + 2e-3 * rms
            loose = err <= 8e-3 * np.abs(want) + 8e-3 * rms
            assert tight.mean() >= 0.99, "%s (%s): only %.4f of the elements within half a bf16 ulp" % (name, shape, tight.mean())
            assert loose.all(), "%s (%s): %d elements beyond one bf16 ulp, worst %.3e (rms %.3e)" % (
                name, shape, int((~loose).sum()), float(err.max()), rms)

