"""Exact model enumeration on the GPU (dsat_enumerate_models, uniformity.enumerate_models / count_models): equal, element
for element and in order, to synth.enumerate_solutions (the numpy specification) up to n = 22, and above that to a
recursive enumerator written here (split on a variable, simplify, unit-propagate), which shares nothing with the brute
force.  Replaces the reference's unigen/approxmc counting (utils/AllSolutions.py:44-68)."""
import ctypes as C
import os

import numpy as np
import pytest

from diffusionsat_b200 import synth, uniformity

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIXTURE = os.path.join(ROOT, "tests", "golden", "trained_small.npz")


def models_by_search(n_vars, clauses):
    """Every model (ints, x1 = bit 0), ascending, by DPLL-style search; variables left unassigned at a leaf are free."""
    norm = []
    for c in clauses:
        lits = set(c)
        if any(-l in lits for l in lits):
            continue                                    # x or not x holds everywhere
        if not lits:
            return []                                   # an empty clause holds nowhere
        norm.append(sorted(lits))
    out = []

    def assign(cls, lit):
        kept = []
        for c in cls:
            if lit in c:
                continue
            if -lit in c:
                c = [l for l in c if l != -lit]
                if not c:
                    return None
            kept.append(c)
        return kept

    def search(cls, fixed):
        while True:
            unit = next((c[0] for c in cls if len(c) == 1), None)
            if unit is None:
                break
            fixed = {**fixed, abs(unit): unit > 0}
            cls = assign(cls, unit)
            if cls is None:
                return
        if not cls:
            free = [v for v in range(1, n_vars + 1) if v not in fixed]
            base = sum(1 << (v - 1) for v, val in fixed.items() if val)
            for bits in range(1 << len(free)):
                out.append(base | sum(1 << (v - 1) for i, v in enumerate(free) if (bits >> i) & 1))
            return
        var = abs(min(cls, key=len)[0])
        for lit in (var, -var):
            rest = assign(cls, lit)
            if rest is not None:
                search(rest, {**fixed, var: lit > 0})

    search(norm, {})
    return sorted(out)


def _edge_cases():
    return [
        ("empty clause", 4, [[1, 2], [], [-3]]),
        ("only an empty clause", 3, [[]]),
        ("repeated literals", 8, [[1, 1, -2], [3, 3, 3], [-7, -7, 8, -7], [2, 2]]),
        ("tautologies", 9, [[1, -1], [4, 2, -4], [8, -8, 9], [-9, 3], [-3, 7]]),
        ("unit clauses", 10, [[3], [-7], [10], [1, 2, -9], [-1, 5]]),
        ("variable in no clause", 9, [[1, -2], [2, 3], [-4, 9], [-1, -3, 9]]),
        ("no clauses", 7, []),
        ("n=1 x1", 1, [[1]]),
        ("n=1 not x1", 1, [[-1]]),
        ("n=1 contradiction", 1, [[1], [-1]]),
        ("n=1 tautology", 1, [[1, -1]]),
        ("n=1 free", 1, []),
    ]


def _random_cases():
    cases = []
    for seed in range(3):
        for n in (8, 14, 22) if seed == 0 else (8, 14):
            cases.append(("random_3sat n=%d seed %d" % (n, seed), *synth.random_3sat(n, seed=seed)))
            cases.append(("planted_3sat n=%d seed %d" % (n, seed), *synth.planted_3sat(n, seed=seed)[:2]))
            cases.append(("random_ksat_mixed n=%d seed %d" % (n, seed), *synth.random_ksat_mixed(n, 2 * n, seed=seed)))
    for n in (5, 6, 7):                                 # around the 64-lane word (variables 1..6)
        for seed in range(4):
            cases.append(("random_ksat_mixed n=%d seed %d" % (n, seed), *synth.random_ksat_mixed(n, n, seed=seed)))
            cases.append(("random_3sat n=%d seed %d" % (n, seed), *synth.random_3sat(n, 2 * n, seed=seed)))
    cases.append(("few clauses n=20", *synth.random_3sat(20, 12, seed=5)))       # more models than Context's first capacity
    return cases


# ------------------------------------------------------------------------------------------------------------ CPU tier
def test_search_enumerator_equals_the_numpy_specification():
    """The independent check used above n = 24 agrees with synth.enumerate_solutions where both run."""
    for name, n, clauses in _edge_cases() + [c for c in _random_cases() if c[1] <= 14]:
        assert models_by_search(n, clauses) == synth.enumerate_solutions(n, clauses), name
    assert len(models_by_search(5, [[-1, 2], [1, -2], [-3, 4, 5]])) == 14


def test_more_than_63_variables_is_refused_before_any_context():
    _, clauses = synth.random_3sat(64, 100, seed=0)
    with pytest.raises(ValueError):
        uniformity.enumerate_models(64, clauses)
    with pytest.raises(ValueError):
        uniformity.count_models(64, clauses)
    with pytest.raises(ValueError):
        uniformity.enumerate_models(0, [])


# ------------------------------------------------------------------------------------------------------------ GPU tier
@pytest.mark.gpu
def test_equal_to_enumerate_solutions_element_for_element(ctx):
    for name, n, clauses in _edge_cases() + _random_cases():
        want = synth.enumerate_solutions(n, clauses)
        got = uniformity.enumerate_models(n, clauses, context=ctx)
        assert got.dtype == np.uint64, name
        assert got.tolist() == want, "%s: %d models, want %d" % (name, len(got), len(want))
        assert uniformity.count_models(n, clauses, context=ctx) == len(want), name


@pytest.mark.gpu
def test_reference_known_answer(ctx):
    """utils/test_AllSolutions.py: [[-1, 2], [1, -2], [-3, 4, 5]] over 5 variables has 14 models."""
    assert uniformity.count_models(5, [[-1, 2], [1, -2], [-3, 4, 5]], context=ctx) == 14
    assert len(uniformity.enumerate_models(5, [[-1, 2], [1, -2], [-3, 4, 5]], context=ctx)) == 14


@pytest.mark.gpu
@pytest.mark.parametrize("n,m,seed", [(30, 133, 0), (36, None, 1), (40, None, 2), (44, None, 3)])
def test_above_the_numpy_limit_equal_to_the_search(ctx, n, m, seed):
    """2^40 and 2^44 assignments take 16 and 256 launches of 2^36 each (dsat_models.cuh: CHUNK_LOG2)."""
    _, clauses, hidden = synth.planted_3sat(n, m, seed=seed)
    want = models_by_search(n, clauses)
    launches = ctx.launch_count()
    got = uniformity.enumerate_models(n, clauses, context=ctx)
    if n >= 40:
        assert ctx.launch_count() - launches >= 2 * 2 ** (n - 36)        # count + scan per chunk at least
    assert got.tolist() == want
    assert sum(int(b) << i for i, b in enumerate(hidden)) in set(want)      # the planted assignment is a model
    assert uniformity.count_models(n, clauses, context=ctx) == len(want)


@pytest.mark.gpu
def test_count_only_capacity_and_argument_checks(ctx):
    lib = ctx._lib
    n, clauses = synth.random_3sat(18, 40, seed=4)
    want = synth.enumerate_solutions(n, clauses)
    assert len(want) > 10
    lens = np.array([len(c) for c in clauses], dtype=np.int32)
    flat = np.array([l for c in clauses for l in c], dtype=np.int32)
    ip = C.POINTER(C.c_int32)

    def call(n_vars=n, lens=lens, flat=flat, out=None, capacity=0, nnz=None):
        count = C.c_longlong(-7)
        rc = lib.dsat_enumerate_models(ctx._h, n_vars, len(lens), int(flat.size if nnz is None else nnz),
                                       lens.ctypes.data_as(ip), flat.ctypes.data_as(ip),
                                       None if out is None else out.ctypes.data_as(C.POINTER(C.c_uint64)), capacity,
                                       C.byref(count))
        return rc, count.value

    assert call() == (0, len(want))                                         # count only
    out = np.zeros(len(want), dtype=np.uint64)
    assert call(out=out, capacity=len(want)) == (0, len(want))
    assert out.tolist() == want
    small = np.zeros(len(want) - 3, dtype=np.uint64)
    assert call(out=small, capacity=small.size) == (-1, len(want))          # DSAT_ERR_ARG with the required size
    assert small.tolist() == want[:small.size]                              # the models that fit are written
    assert call(out=None, capacity=5)[0] == -1                              # null output with a capacity
    assert call(out=out, capacity=-1)[0] == -1
    assert call(n_vars=64)[0] == -1
    assert call(n_vars=0)[0] == -1
    assert call(nnz=flat.size - 1)[0] == -1                                 # lens do not sum to nnz
    bad = flat.copy()
    bad[5] = 0
    assert call(flat=bad)[0] == -1
    bad[5] = 19                                                             # beyond n_vars
    assert call(flat=bad)[0] == -1
    bad[5] = -19
    assert call(flat=bad)[0] == -1
    assert call(out=out, capacity=len(want)) == (0, len(want))              # the context is still usable


@pytest.mark.gpu
def test_enumeration_leaves_the_context_state_untouched(ctx):
    from diffusionsat_b200 import graph as G
    from diffusionsat_b200.weights import load_weights
    n, clauses, _ = synth.planted_3sat(20, 80, seed=6)
    ctx.set_model(load_weights(FIXTURE))
    ctx.set_graph(G.build_unit_graph(n, clauses), chains=64, group_graphs=16)
    precision = ctx.get_precision()
    before = ctx.sample(32, 32, seed=11)
    models = uniformity.enumerate_models(n, clauses, context=ctx)
    uniformity.enumerate_models(40, synth.planted_3sat(40, seed=2)[1], context=ctx)     # several chunks
    assert ctx.get_precision() == precision
    after = ctx.sample(32, 32, seed=11)
    for a, b in zip(before, after):
        np.testing.assert_array_equal(a, b)
    packed, is_sat = after[0], after[1].astype(bool)
    assert is_sat.any()
    assert set((packed[is_sat, 0] & np.uint64((1 << n) - 1)).tolist()) <= set(models.tolist())


@pytest.mark.gpu
def test_sampler_draws_only_models(ctx, tmp_path):
    """DiffusionSampler with the trained fixture on the bench's trained_weights formula (n = 30): every key is a model."""
    from diffusionsat_b200.sampler import DiffusionSampler
    n, clauses, _ = synth.planted_3sat(30, 133, seed=0)
    cnf = tmp_path / "planted30.cnf"
    cnf.write_text(synth.dimacs_text(n, clauses))
    hist = DiffusionSampler(FIXTURE, str(cnf), context=ctx).samples(200)
    models = set(uniformity.enumerate_models(n, clauses, context=ctx).tolist())
    assert sum(hist.values()) == 200
    assert set(hist) <= models
