"""GPU tests of the tensor-core (tcgen05, bf16) MLP path.

Stated tolerance of the bf16 path: one linear op against an fp64 product of the SAME bf16-rounded
operands within 2e-3 relative (fp32 accumulation); one teacher-forced round's logits within 5e-2
relative of the fp32 oracle; free-running 32-round logits are reported, not asserted tightly."""
import numpy as np
import pytest
import torch

from diffusionsat_b200 import _lib, graph as G, synth
from oracle import querysat_oracle as O
from tests import helpers as H

pytestmark = pytest.mark.gpu


def bf16_round(x):
    return torch.from_numpy(np.asarray(x, dtype=np.float32)).to(torch.bfloat16).to(torch.float64).numpy()


@pytest.mark.parametrize("rows,k,n,epi", [
    (300, 64, 32, 0), (128, 144, 672, 1), (1000, 528, 240, 1), (257, 160, 128, 2), (77, 128, 16, 0),
    (513, 512, 512, 1), (4096, 384, 208, 1), (130, 208, 256, 0), (64, 240, 128, 0)])
def test_tc_linear_matches_reference_product(ctx, rows, k, n, epi):
    rng = np.random.default_rng(rows + k + n)
    a = rng.standard_normal((rows, k)).astype(np.float32)
    w = (rng.standard_normal((k, n)) / np.sqrt(k)).astype(np.float32)
    b = rng.standard_normal(n).astype(np.float32) * 0.1
    want = bf16_round(a) @ bf16_round(w) + b.astype(np.float64)
    if epi == 1:
        want = np.where(want > 0, want, 0.2 * want)
    got = ctx.tc_linear_test(a, w, b, epi=epi, out_bf16=False)
    scale = np.abs(want).max()
    assert np.abs(got[:, :n] - want).max() / scale < 2e-3
    if epi == 2:
        assert np.abs(got[:, n:2 * n] - np.logaddexp(0, want)).max() < 2e-3 * max(scale, 1)
        assert np.abs(got[:, 2 * n:] - np.logaddexp(0, -want)).max() < 2e-3 * max(scale, 1)
    got_b = ctx.tc_linear_test(a, w, b, epi=epi, out_bf16=True)
    assert np.abs(got_b[:, :n] - want).max() / scale < 1e-2


def test_bf16_round_against_fp32_oracle(ctx):
    n_vars, chains, seed = 30, 5, 0
    _, clauses = synth.random_3sat(n_vars, seed=seed)
    wts = H.make_weights(seed=11)
    ctx.set_model(wts)
    ctx.set_precision(_lib.BF16)
    ctx.set_graph(G.build_unit_graph(n_vars, clauses), chains=chains, group_graphs=0)
    n_rows, rounds = n_vars * chains, 3
    noise = H.noise_for(n_rows, rounds, seed)
    noisy = O.randomized_rounding(torch.full((n_rows, 2), 0.5), torch.from_numpy(noise["uniform"])).numpy()
    graph, _, trace = H.oracle_trace(n_vars, clauses, chains, wts, 0.625, noisy, noise, rounds)
    ctx.debug_begin(0.625, noisy, noise["labels"])
    F = 128
    for r in range(rounds):
        if r > 0:
            prev = trace[r - 1]
            carry = lambda x: (x * np.float32(0.2) + x * np.float32(0.8)).astype(np.float32)
            vrow = ctx.debug_read("VROW"); vrow[:, :F] = carry(prev["variables"].numpy()); ctx.debug_write("VROW", vrow)
            crow = ctx.debug_read("CROW"); crow[:, :F] = carry(prev["clause_state"].numpy()); ctx.debug_write("CROW", crow)
        ctx.debug_round(r, noise["normals"][r])
        tr = trace[r]
        assert H.rel_err(ctx.debug_read("SPRE"), tr["variables"].numpy()) < 5e-2
        assert H.rel_err(ctx.debug_read("LOGITS")[:, :8], tr["logits"].numpy()) < 5e-2
        crow = ctx.debug_read("CROW")
        assert H.rel_err(crow[:, :F], (tr["clause_state"].numpy() * np.float32(0.2) + tr["clause_state"].numpy() * np.float32(0.8))) < 5e-2


def test_bf16_sampler_runs_and_is_deterministic(ctx):
    n_vars, clauses = 5, [[-1, 2], [1, -2], [-3, 4, 5]]
    ctx.set_model(H.make_weights(seed=2))
    ctx.set_precision(_lib.BF16)
    ctx.set_graph(G.build_unit_graph(n_vars, clauses), chains=64, group_graphs=8)
    a = ctx.sample(6, 4, seed=5)
    b = ctx.sample(6, 4, seed=5)
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)
    models = set(synth.enumerate_solutions(n_vars, clauses))
    from diffusionsat_b200.sampler import unpack_assignments
    vals = unpack_assignments(a[0], n_vars)
    for v, s in zip(vals, a[1]):
        assert (v in models) == bool(s)          # the SAT flag is exact integer work in both precisions


FUSED_SHAPES = {   # id -> (variables, chains, feature_maps, query_maps, literal hidden width (None = 4 query_maps))
    "7": (100, 7, 128, 128, None),
    "600": (100, 600, 128, 128, None),
    "one_tile": (20, 1, 128, 128, None),
    "f128_q64": (100, 60, 128, 64, None),
    "lit_hidden_384": (100, 60, 128, 128, 384),
}


@pytest.mark.parametrize("shape", list(FUSED_SHAPES))
def test_fused_mlp_kernels_match_per_layer_kernels(ctx, shape):
    """One kernel per MLP (hidden activations in shared memory) against one kernel per Dense layer:
    same bf16 rounding points, same accumulation order -> logits agree to fp32 round-off.
    7 chains: at most one 128-row tile per CTA; 600 chains: 3-4 variable tiles and 13-14 clause tiles per CTA, i.e.
    the persistent loop, the input ring wrap-around and the ping-pong pairing with odd and even tile counts.
    one_tile (at most 128 rows per MLP): the single-CTA instantiations; f128_q64: the literal MLP with its input resident in
    fused_mlp_kernel; lit_hidden_384: hidden layers wider than 256 columns without split mode."""
    n_vars, chains, F, Q, lit_hidden = FUSED_SHAPES[shape]
    rounds = 3
    _, clauses = synth.random_3sat(n_vars, seed=4)
    wts = H.make_weights(F, Q, seed=9, lit_hidden=lit_hidden)
    n_rows = n_vars * chains
    noise = H.noise_for(n_rows, rounds, 3)
    noisy = O.randomized_rounding(torch.full((n_rows, 2), 0.5), torch.from_numpy(noise["uniform"])).numpy()
    ctx.set_model(wts)
    ctx.set_graph(G.build_unit_graph(n_vars, clauses), chains=chains, group_graphs=0)
    out = {}
    for name, code in (("fused", _lib.BF16), ("per_layer", 2), ("fp32", _lib.F32)):
        ctx.set_precision(code)
        ctx.debug_begin(0.5, noisy, noise["labels"])
        for r in range(rounds):
            ctx.debug_round(r, noise["normals"][r])
        out[name] = (ctx.debug_read("LOGITS").copy(), ctx.debug_read("SPRE").copy(), ctx.debug_read("CROW")[:, :F].copy())
    for a, b in zip(out["fused"], out["per_layer"]):
        # two bf16 realisations (leaky relu on packed bf16 pairs vs fp32); same bound as against the oracle.  The
        # maximum over thousands of rows sits further out in the tail of the rounding noise, so the large cases bound
        # the maximum at 1e-1 and the rms error at 2e-2: a misplaced or stale tile would be an O(1) error
        assert H.rel_err(a, b) < (5e-2 if n_rows < 1000 else 1e-1)
        scale = max(float(np.sqrt(np.mean(b.astype(np.float64) ** 2))), 1e-12)
        err2 = ((a.astype(np.float64) - b) ** 2).mean(axis=1)
        assert float(np.sqrt(err2.mean())) / scale < 3.5e-2             # typical: 2e-2 after three rounds
        pad = (-len(err2)) % 128
        tiles = np.sqrt(np.pad(err2, (0, pad)).reshape(-1, 128).mean(axis=1)) / scale
        assert tiles.max() < 1e-1                                         # every 128-row tile on its own
    # and against the fp32 parity path (SIMT GEMMs, general gather kernels, generic PairNorm): independent kernels all
    # the way, so this also covers the shared-memory gathers and the bf16 PairNorm at a size with many chains per SM
    for a, b in zip(out["fused"], out["fp32"]):
        scale = max(float(np.sqrt(np.mean(b.astype(np.float64) ** 2))), 1e-12)
        err2 = ((a.astype(np.float64) - b) ** 2).mean(axis=1)
        assert float(np.sqrt(err2.mean())) / scale < 5e-2
        pad = (-len(err2)) % 128
        assert (np.sqrt(np.pad(err2, (0, pad)).reshape(-1, 128).mean(axis=1)) / scale).max() < 1.5e-1
