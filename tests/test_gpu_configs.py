"""GPU parity on the other BASELINE.json configurations (they are parity cases, not bench lines):
configs[2] uf250-shaped 3-SAT (n=250, m=1065; tables too large for the shared-memory gathers, so the
L2-gather kernels run), configs[3] a training-shaped batch of mixed k-SAT formulas as ONE disjoint-union
graph through the QuerySAT API (general graph mode: per-graph segments, reference-layout COO input),
configs[4] the n=10000 graph for the segment-sum kernels at widths 64/128/256."""
import numpy as np
import pytest
import torch

from diffusionsat_b200 import _lib, graph as G, synth
from oracle import querysat_oracle as O
from tests import helpers as H

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("precision,tol", [(_lib.F32_TC, 1e-3), (_lib.F32, 1e-3), (_lib.BF16, 8e-2)])
def test_uf250_shape_model_call(ctx, precision, tol):
    n_vars, m, chains, rounds = 250, 1065, 3, 4
    _, clauses = synth.random_3sat(n_vars, m, seed=250)
    wts = H.make_weights(seed=13)
    ctx.set_model(wts)
    ctx.set_precision(precision)
    ctx.set_graph(G.build_unit_graph(n_vars, clauses), chains=chains, group_graphs=0)
    n_rows = n_vars * chains
    noise = H.noise_for(n_rows, rounds, 31)
    noisy = O.randomized_rounding(torch.full((n_rows, 2), 0.5), torch.from_numpy(noise["uniform"])).numpy()
    graph, out, trace = H.oracle_trace(n_vars, clauses, chains, wts, 0.5, noisy, noise, rounds)
    ctx.debug_begin(0.5, noisy, noise["labels"])
    for r in range(rounds):
        ctx.debug_round(r, noise["normals"][r])
    assert H.rel_err(ctx.debug_read("LOGITS")[:, :8], trace[-1]["logits"].numpy()) < tol
    assert H.rel_err(ctx.debug_read("SPRE"), trace[-1]["variables"].numpy()) < tol


def test_mixed_ksat_union_batch_through_querysat_api(ctx):
    from diffusionsat_b200.query_sat import QuerySAT
    rng = np.random.default_rng(3)
    formulas = []
    for s in range(9):
        n = int(rng.integers(3, 40))
        formulas.append(synth.random_ksat_mixed(n, int(rng.integers(n, 4 * n)), seed=100 + s))
    union = G.build_union_graph(formulas)
    assert G.sat_node_count(union.n_vars, union.n_clauses) <= G.MAX_NODES_PER_BATCH
    coo, shape = union.reference_coo(1)
    vg = np.repeat(np.arange(len(formulas)), [n for n, _ in formulas])
    cg = np.repeat(np.arange(len(formulas)), [len(c) for _, c in formulas])
    wts = H.make_weights(seed=17)
    rounds = 5
    model = QuerySAT(optimizer=None, test_rounds=rounds, weights=wts, context=ctx)
    n_rows = union.n_vars
    noise = H.noise_for(n_rows, rounds, 8)
    noisy = O.randomized_rounding(torch.full((n_rows, 2), 0.5), torch.from_numpy(noise["uniform"])).numpy()
    res = model.diffusion_step((coo, shape), cg, vg, None, 0.3, noisy, labels=noise["labels"], normals=noise["normals"])
    og = O.OracleGraph.from_formulas(formulas)
    trace = []
    want = O.model_loop(og, O.weights_to_torch(wts), 0.3, torch.from_numpy(noisy),
                        torch.from_numpy(noise["labels"].astype(np.int64)), torch.from_numpy(noise["normals"]), rounds,
                        trace=trace)
    assert res["steps_taken"] == want[1]
    gmap = ctx.debug_groups()["graph_map"]
    same = np.repeat(gmap == trace[-1]["best_graph_map"].numpy(), [n for n, _ in formulas])
    assert same.mean() > 0.6
    assert H.rel_err(res["prediction"][same], want[0].numpy()[same]) < 1e-3
    assert abs(float(res["loss"]) - float(want[2])) < 1e-3 * max(1.0, abs(float(want[2])))
    # predict_step draws its own noise: shape and finiteness only
    out = model.predict_step((coo, shape), cg, vg, None)
    assert out["prediction"].shape == (n_rows,) and np.isfinite(out["prediction"]).all()
    # prediction_tries > 1 (reference model/query_sat.py:429-445): a graph keeps the logits of the first try that
    # satisfied it and zeros otherwise, so every non-zero block must satisfy its formula
    from diffusionsat_b200.query_sat import is_graph_sat
    model.prediction_tries = 3
    out3 = model.predict_step((coo, shape), cg, vg, None)
    model.prediction_tries = 1
    flags = is_graph_sat(out3["prediction"], coo, shape, cg, len(formulas))
    for gi in range(len(formulas)):
        block = out3["prediction"][vg == gi]
        assert (block != 0).any() == bool(flags[gi]) or not (block != 0).any()
        if (block != 0).any():
            assert flags[gi] == 1.0
    # plot_step: labels = solutions (ragged), explicit noise level
    sols = [np.zeros(n, dtype=np.int32) for n, _ in formulas]
    outp = model.plot_step((coo, shape), cg, vg, sols, 0.5)
    assert outp["prediction"].shape == (n_rows,) and np.isfinite(outp["prediction"]).all()


@pytest.mark.parametrize("feat", [64, 128, 256])
def test_n10000_segment_sums_roundtrip_properties(ctx, feat):
    """Full-size graph of configs[4]: linearity and a checksum instead of an element-wise oracle."""
    n, m, chains = 10000, 43000, 2
    _, clauses = synth.random_3sat(n, m, seed=5)
    unit = G.build_unit_graph(n, clauses)
    ctx.set_model(H.make_weights(seed=1))
    ctx.set_graph(unit, chains=1, group_graphs=0)
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(1)
    x1 = torch.randn(chains, 2 * n, feat, generator=g).to(dev)
    x2 = torch.randn(chains, 2 * n, feat, generator=g).to(dev)
    y1, y2, y12 = (torch.empty(chains, m, feat, device=dev) for _ in range(3))
    x12 = 2 * x1 - x2
    torch.cuda.synchronize()
    ctx.spmm(0, x1.data_ptr(), y1.data_ptr(), feat, 0, chains)
    ctx.spmm(0, x2.data_ptr(), y2.data_ptr(), feat, 0, chains)
    ctx.spmm(0, x12.data_ptr(), y12.data_ptr(), feat, 0, chains)
    ctx.synchronize()
    assert torch.allclose(y12, 2 * y1 - y2, rtol=1e-4, atol=1e-4)                 # linearity
    # checksum: sum over clauses of sqrt(|c|)*Y equals sum over literals of deg(lit)*X
    deg = torch.from_numpy(unit.lit_degree().astype(np.float32)).to(dev)
    lhs = (y1 * np.sqrt(3.0)).sum(dim=1)
    rhs = (x1 * deg[None, :, None]).sum(dim=1)
    assert torch.allclose(lhs, rhs, rtol=2e-3, atol=2e-2)
    # the other direction on ones: every literal row sums its clause count
    ones = torch.ones(chains, m, feat, device=dev)
    z = torch.empty(chains, 2 * n, feat, device=dev)
    ctx.spmm(1, ones.data_ptr(), z.data_ptr(), feat, 0, chains)
    ctx.synchronize()
    want = torch.sqrt(torch.clamp(deg, min=1)) * (deg > 0)                        # deg * rsqrt(max(deg,1))
    assert torch.allclose(z[0, :, 0], want, rtol=1e-5, atol=1e-6)
