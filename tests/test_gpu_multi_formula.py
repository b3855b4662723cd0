"""Several formulas sampled in one launch (MultiDiffusionSampler, dsat_set_batches, dsat_hist_reduce_segments).

* contract: ``MultiDiffusionSampler(...).samples(n)[k]`` equals the per-file ``DiffusionSampler(...).samples(n)`` dict for
  formulas of one shared-memory-PairNorm class, with the trained fixture weights, on both fp32-accurate paths;
* oracle: groups of a union run with per-graph noise bases reproduce, bit for bit, the run of that group alone (on the
  device, and on the CPU oracle with the noise regenerated from the groups' noise bases);
* the segmented histogram against numpy per segment; argument validation; formulas of different PairNorm classes."""
import os

import numpy as np
import pytest
import torch

from diffusionsat_b200 import _lib, dist as D, graph as G, philox, synth
from diffusionsat_b200 import sampler as S
from diffusionsat_b200.sampler import DiffusionSampler, MultiDiffusionSampler
from diffusionsat_b200.variable_assignment import VariableAssignment
from diffusionsat_b200.weights import load_weights
from oracle import querysat_oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIXTURE = os.path.join(ROOT, "tests", "golden", "trained_small.npz")
MAX_NODES = 500             # reference batches of 2-3 copies at n = 24..30: early exit on small groups


def _files(tmp_path, sizes, seed0=0):
    out, formulas = [], []
    for i, n in enumerate(sizes):
        n_vars, clauses, _ = synth.planted_3sat(n, seed=seed0 + i)
        p = tmp_path / ("f%d_n%d.cnf" % (i, n))
        p.write_text(synth.dimacs_text(n_vars, clauses))
        out.append(str(p))
        formulas.append((n_vars, clauses))
    return out, formulas


def _satisfies(clauses, key, n):
    bits = [(key >> v) & 1 for v in range(n)]
    return all(any((bits[abs(l) - 1] == 1) == (l > 0) for l in c) for c in clauses)


def _pairnorm_threads(rows, feature_maps=128):
    """Thread count launch_pairnorm_smem picks for the largest graph (dsat_api.cu): what fixes its reduction order."""
    b = rows * feature_maps * 4
    return 1024 if b > 100 * 1024 else 512 if b > 48 * 1024 else 256


@pytest.mark.parametrize("precision", ["fp32", "fp32_simt"])
def test_multi_sampler_equals_per_file_samplers(ctx, tmp_path, monkeypatch, precision):
    files, formulas = _files(tmp_path, [24, 30, 26, 28, 25, 27])
    assert len({_pairnorm_threads(len(c)) for _, c in formulas}) == 1
    assert len({_pairnorm_threads(n) for n, _ in formulas}) == 1
    # a small row budget: launches hold a few formulas each, so formulas wait and launches differ from the solo ones
    monkeypatch.setattr(S, "ROWS_CAP", 60_000)
    kw = dict(seed=21, chain_offset=5, max_nodes_per_batch=MAX_NODES, precision=precision)
    ms = MultiDiffusionSampler(FIXTURE, files, context=ctx, **kw)
    assert {f.batch_chains for f in ms.formulas} <= {1, 2, 3}
    launches0 = ctx.launch_count()
    got = ms.samples(64)
    stats = ms.last_stats
    print("multi: %d kernel launches; per formula %r" % (ctx.launch_count() - launches0, stats))
    for k, f in enumerate(files):
        solo = DiffusionSampler(FIXTURE, f, context=ctx, **kw)
        want = solo.samples(64)
        assert got[k] == want, "formula %d: %d of %d keys differ" % (k, len(set(got[k].items()) ^ set(want.items())), len(want))
        assert stats[k]["total"] == solo.last_stats["total"] and stats[k]["sat"] == solo.last_stats["sat"]


def test_multi_sampler_bf16_is_valid(ctx, tmp_path):
    files, formulas = _files(tmp_path, [24, 30, 26, 28, 25, 27])
    kw = dict(seed=21, chain_offset=5, max_nodes_per_batch=MAX_NODES, precision="bf16")
    ms = MultiDiffusionSampler(FIXTURE, files, context=ctx, **kw)
    got = ms.samples(64)
    equal = 0
    for k, (n, clauses) in enumerate(formulas):
        st = ms.last_stats[k]          # a formula may abort under the reference's 0.5 % rule, as its own sampler would
        assert sum(got[k].values()) == st["sat"] and (st["sat"] == 64 or st["stopped_on_rate"])
        assert all(_satisfies(clauses, key, n) for key in got[k])
        equal += got[k] == DiffusionSampler(FIXTURE, files[k], context=ctx, **kw).samples(64)
    print("bf16: %d of %d formulas equal to their per-file sampler; %r" % (equal, len(files), ms.last_stats))
    assert any(st["sat"] == 64 for st in ms.last_stats)


def _bits_of(packed_rows, n):
    out = np.zeros((packed_rows.shape[0], n), dtype=np.uint8)
    for v in range(n):
        out[:, v] = (packed_rows[:, v // 64] >> np.uint64(v % 64)) & np.uint64(1)
    return out


def test_union_groups_match_their_solo_runs_and_the_oracle(ctx, tmp_path):
    _, formulas = _files(tmp_path, [24, 30, 27], seed0=40)
    wts = load_weights(FIXTURE)
    ctx.set_model(wts)
    ctx.set_precision("fp32")
    batches = [G.chains_per_reference_batch(n, len(c), MAX_NODES) for n, c in formulas]
    copies = [2 * batches[0], 3 * batches[1], 2 * batches[2]]
    first = [3, 100, 9]                      # global chain id of each formula's copy 0
    flat = [G.flatten_formula(n, c) for n, c in formulas]
    unit = G.build_union_graph([flat[k] for k in range(3) for _ in range(copies[k])])
    group_seg, base, where = [0], [], []
    for k, (n, _) in enumerate(formulas):
        for j in range(0, copies[k], batches[k]):
            where.append((k, group_seg[-1], j))
            group_seg.append(group_seg[-1] + batches[k])
        base += [(first[k] + j) * n for j in range(copies[k])]
    seed = 31
    ctx.set_graph(unit, chains=1)
    ctx.set_batches(group_seg, np.array(base, dtype=np.uint64))
    packed, is_sat, latch, _ = ctx.sample(32, 32, seed=seed)
    for gi in (0, len(where) // 2, len(where) - 1):           # first, middle and last group: three different formulas
        k, g0, j0 = where[gi]
        n, clauses = formulas[k]
        b = batches[k]
        rows = slice(g0, g0 + b)
        # the same group alone on the device
        ctx.set_graph(G.build_unit_graph(n, clauses), chains=b, group_graphs=b)
        p1, s1, l1, _ = ctx.sample(32, 32, seed=seed, chain_offset=first[k] + j0)
        np.testing.assert_array_equal(packed[rows, :p1.shape[1]], p1)
        np.testing.assert_array_equal(is_sat[rows], s1)
        np.testing.assert_array_equal(latch[rows], l1)
        # and on the oracle, with the noise regenerated from the group's noise bases
        elems = np.concatenate([np.arange(base[g0 + i], base[g0 + i] + n, dtype=np.uint64) for i in range(b)])
        uniforms = np.stack([philox.uniforms(seed, elems, t) for t in range(32)])
        labels = np.stack([philox.labels(seed, elems, t) for t in range(32)])
        normals = np.stack([np.stack([philox.normals(seed, elems, t, r) for r in range(32)]) for t in range(32)])
        _, final, latch_o = O.diffusion(32, O.OracleGraph.copies(n, clauses, b), O.weights_to_torch(wts),
                                        torch.from_numpy(uniforms), torch.from_numpy(labels.astype(np.int64)),
                                        torch.from_numpy(normals), 32)
        want_bits = np.asarray(final).reshape(b, n).astype(np.uint8)
        got_bits = _bits_of(packed[rows], n)
        exact = int((got_bits == want_bits).all(axis=1).sum())
        print("group %d (formula %d, %d copies): %d bit-exact against the oracle" % (gi, k, b, exact))
        assert exact == b
        np.testing.assert_array_equal(latch[rows], np.asarray(latch_o).reshape(b, n)[:, 0])
        want_sat = [VariableAssignment(n_vars=n, clauses=clauses) for _ in range(b)]
        for i, a in enumerate(want_sat):
            a.assign_all([bool(x) for x in want_bits[i]])
            assert bool(is_sat[g0 + i]) == a.satisfiable()
        ctx.set_graph(unit, chains=1)
        ctx.set_batches(group_seg, np.array(base, dtype=np.uint64))


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_skipping_finished_groups_changes_nothing(ctx, precision):
    """Whole-chain groups bound with group_graphs skip the rows of finished groups; the same groups bound through
    dsat_set_batches (no noise bases) compute every row.  Both runs give the same bits."""
    n_vars, clauses, _ = synth.planted_3sat(24, seed=5)
    chains, group, steps, rounds = 96, 3, 16, 32
    unit = G.build_unit_graph(n_vars, clauses)
    ctx.set_model(load_weights(FIXTURE))
    ctx.set_precision(precision)
    runs = []
    for skip in (True, False):
        ctx.set_graph(unit, chains=chains, group_graphs=group)
        if not skip:
            ctx.set_batches(np.arange(0, chains + 1, group))
        runs.append(ctx.sample(steps, rounds, seed=13) + (ctx.debug_groups()["steps_taken"],))
    assert (runs[0][-1] < rounds - 1).any(), "no group finished early: nothing was skipped"
    for name, a, b in zip(("packed", "is_sat", "latch_step", "sat_any", "steps_taken"), *runs):
        np.testing.assert_array_equal(a, b, err_msg=name)


def test_segmented_histogram_equals_numpy(ctx):
    ctx.set_model(load_weights(FIXTURE))
    ctx.set_precision("bf16")
    sizes, copies = [14, 70, 20, 14], [300, 40, 0, 260]          # keys of 1 and 2 words; an empty segment
    flat = [G.flatten_formula(*synth.planted_3sat(n, int(4 * n) if n < 60 else 250, seed=3 + i)[:2])
            for i, n in enumerate(sizes)]
    unit = G.build_union_graph([flat[k] for k in range(len(sizes)) for _ in range(copies[k])])
    ctx.set_graph(unit, chains=1, group_graphs=20)
    packed, is_sat, _, _ = ctx.sample(8, 6, seed=5)
    seg = np.concatenate([[0], np.cumsum(copies)]).astype(np.int32)
    for limits in ([300, 40, 0, 260], [77, 9, 5, 1000]):
        tables, n_sat = ctx.hist_reduce_segments(seg, limits)
        total = 0
        for s in range(len(sizes)):
            lo, hi = seg[s], seg[s + 1]
            sat = is_sat[lo:hi].copy()
            sat[min(limits[s], hi - lo):] = 0
            want_k, want_c = D.local_histogram(packed[lo:hi], sat)
            np.testing.assert_array_equal(tables[s][0], want_k)
            np.testing.assert_array_equal(tables[s][1], want_c)
            total += int(sat.sum())
        assert n_sat == total and total > 0
        assert len(tables[0][1]) >= 2 and len(tables[2][1]) == 0
    # capacity too small: an error, and seg_runs[n_segments] holds the size needed
    lib = ctx._lib
    lim = np.array(limits, dtype=np.int32)
    keys = np.empty((1, packed.shape[1]), dtype=np.uint64)
    counts = np.empty(1, dtype=np.int64)
    runs = np.zeros(len(sizes) + 1, dtype=np.int32)
    import ctypes as C
    rc = lib.dsat_hist_reduce_segments(ctx._h, len(sizes), seg.ctypes.data_as(C.POINTER(C.c_int32)),
                                       lim.ctypes.data_as(C.POINTER(C.c_int32)), keys.ctypes.data_as(C.POINTER(C.c_uint64)),
                                       counts.ctypes.data_as(C.POINTER(C.c_int64)), 1, runs.ctypes.data_as(C.POINTER(C.c_int32)),
                                       None)
    assert rc == -1                                             # DSAT_ERR_ARG
    assert runs[-1] == sum(len(t[1]) for t in tables) > 1


def test_bad_batches_are_rejected_and_leave_the_binding(ctx):
    ctx.set_model(load_weights(FIXTURE))
    ctx.set_precision("bf16")
    n, clauses, _ = synth.planted_3sat(20, seed=8)
    unit = G.build_union_graph([G.flatten_formula(n, clauses)] * 6)
    ctx.set_graph(unit, chains=1)
    base = np.arange(6, dtype=np.uint64) * np.uint64(n) + np.uint64(40 * n)
    ctx.set_batches([0, 2, 4, 6], base)
    ref = ctx.sample(4, 4, seed=2)
    for bad_seg in ([0, 2, 2, 6], [0, 4, 2, 6], [0, 2, 4], [1, 2, 4, 6], [0, 2, 4, 7]):
        with pytest.raises(_lib.DsatError):
            ctx.set_batches(bad_seg, base)
    with pytest.raises(_lib.DsatError):                         # elements of the last graph would wrap around 2^64
        ctx.set_batches([0, 2, 4, 6], np.concatenate([base[:5], [np.uint64(2 ** 64 - 5)]]))
    with pytest.raises(_lib.DsatError):                         # bound noise bases replace chain_offset
        ctx.sample(4, 4, seed=2, chain_offset=1)
    again = ctx.sample(4, 4, seed=2)
    for a, b in zip(ref, again):
        np.testing.assert_array_equal(a, b)
    # the bases are what the noise depends on: the same graphs as chains 40.. of the formula bound alone
    ctx.set_graph(G.build_unit_graph(n, clauses), chains=6, group_graphs=2)
    solo = ctx.sample(4, 4, seed=2, chain_offset=40)
    for a, b in zip(ref, solo):
        np.testing.assert_array_equal(a, b)


def test_mixed_pairnorm_classes_are_valid(ctx, tmp_path):
    files, formulas = _files(tmp_path, [20, 100], seed0=60)
    assert _pairnorm_threads(len(formulas[0][1])) != _pairnorm_threads(len(formulas[1][1]))
    ms = MultiDiffusionSampler(FIXTURE, files, context=ctx, seed=3, precision="fp32")
    got = ms.samples([32, 8])
    for k, (n, clauses) in enumerate(formulas):
        st = ms.last_stats[k]
        assert sum(got[k].values()) == st["sat"]
        assert st["sat"] == [32, 8][k] or st["stopped_on_rate"]
        assert all(_satisfies(clauses, key, n) for key in got[k])
    assert ms.last_stats[0]["sat"] == 32
