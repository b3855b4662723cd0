"""Model enumeration by ordered search on the GPU (dsat_enumerate_models_search, uniformity.enumerate_models_by_search /
count_models_by_search): element for element and in order the brute force's list up to n = 44, and above 63 variables
the list of models_by_search (the CPU enumerator of test_gpu_model_enumeration.py, which shares nothing with either)."""
import ctypes as C
import os
import random

import numpy as np
import pytest

from diffusionsat_b200 import synth, uniformity
from diffusionsat_b200.dist import keys_to_ints
from tests.test_gpu_model_enumeration import _edge_cases, _random_cases, models_by_search

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIXTURE = os.path.join(ROOT, "tests", "golden", "trained_small.npz")
DSAT_ERR_ARG, DSAT_ERR_UNSUPPORTED = -1, -4


def _as_ints(keys, n):
    assert keys.dtype == np.uint64 and keys.ndim == 2 and keys.shape[1] == (n + 63) // 64
    return keys_to_ints(keys, n)


def _boundary_formula(n, seed):
    """Free and forced variables on both sides of every word boundary below n, a few open clauses among them, a
    tautology, repeated literals and (for n > 64) a variable above bit 63 that appears in no clause."""
    rng = random.Random(seed)
    near = sorted({v for b in (1, 63, 64, 65, 127, 128, 129, n - 1, n) for v in (b - 1, b, b + 1) if 1 <= v <= n})
    free = {near[1], near[-2]} | ({65} if n >= 65 else set())          # in no clause
    branch = [v for v in near if v not in free]
    clauses = []
    for _ in range(len(branch)):
        vs = rng.sample(branch, min(len(branch), rng.choice((2, 3))))
        clauses.append([v if rng.random() < 0.5 else -v for v in vs])
    for v in range(1, n + 1):
        if v not in free and v not in near:
            clauses.append([v] if rng.random() < 0.5 else [-v, -v])      # forced; repeated literal
    clauses.append([branch[0], -branch[0], branch[-1]])                  # a tautology
    clauses.append([branch[1], branch[1], -branch[2], branch[1]])        # repeated literals in an open clause
    return n, clauses


def _chunked_formula():
    """n = 70: the 15 variables 56..70 each decide the value of one low variable (h = not l), every other variable is
    forced.  The frontier doubles on every level without a conflict or a leaf until it holds 2^15 nodes, more than one
    search launch takes, and every node below it is one model: 32768 models."""
    clauses = []
    for i, h in enumerate(range(56, 71)):
        clauses += [[h, i + 1], [-h, -(i + 1)]]
    clauses += [[v] if v % 2 else [-v] for v in range(16, 56)]
    return 70, clauses


# ------------------------------------------------------------------------------------------------------------ CPU tier
def test_out_of_range_is_refused_before_any_context():
    for n in (0, 1025, -3):
        with pytest.raises(ValueError):
            uniformity.enumerate_models_by_search(n, [[1]])
        with pytest.raises(ValueError):
            uniformity.count_models_by_search(n, [[1]])


def test_hand_made_formulas_are_small_and_straddle_the_words():
    for n in (64, 65, 127, 128, 129, 1024):
        _, clauses = _boundary_formula(n, seed=n)
        used = {abs(l) for c in clauses for l in c}
        if n > 64:
            assert 65 not in used
        want = models_by_search(n, clauses)
        assert 0 < len(want) < 20000, (n, len(want))
    n, clauses = _chunked_formula()
    assert len(models_by_search(n, clauses)) == 2 ** 15


# ------------------------------------------------------------------------------------------------------------ GPU tier
@pytest.mark.gpu
def test_equal_to_the_brute_force_element_for_element(ctx):
    for name, n, clauses in _edge_cases() + _random_cases():
        want = uniformity.enumerate_models(n, clauses, context=ctx).tolist()
        got = uniformity.enumerate_models_by_search(n, clauses, context=ctx)
        assert _as_ints(got, n) == want, "%s: %d models, want %d" % (name, len(got), len(want))
        assert uniformity.count_models_by_search(n, clauses, context=ctx) == len(want), name


@pytest.mark.gpu
@pytest.mark.parametrize("n,m,seed", [(30, 133, 0), (36, None, 1), (40, None, 2), (44, None, 3)])
def test_equal_to_the_brute_force_on_planted_formulas(ctx, n, m, seed):
    _, clauses, hidden = synth.planted_3sat(n, m, seed=seed)
    want = uniformity.enumerate_models(n, clauses, context=ctx).tolist()
    assert _as_ints(uniformity.enumerate_models_by_search(n, clauses, context=ctx), n) == want
    assert uniformity.count_models_by_search(n, clauses, context=ctx) == len(want)
    assert sum(int(b) << i for i, b in enumerate(hidden)) in set(want)


BEYOND_63 = [("random_3sat(64, seed=2)", lambda: synth.random_3sat(64, seed=2)),
             ("random_3sat(80, seed=1)", lambda: synth.random_3sat(80, seed=1)),
             ("random_3sat(80, seed=2)", lambda: synth.random_3sat(80, seed=2)),
             ("random_3sat(100, seed=1)", lambda: synth.random_3sat(100, seed=1)),
             ("bench formula random_3sat(100, seed=0)", lambda: synth.random_3sat(100, seed=0)),
             ("unsatisfiable random_3sat(64, seed=1)", lambda: synth.random_3sat(64, seed=1)),
             ("unsatisfiable random_3sat(100, seed=3)", lambda: synth.random_3sat(100, seed=3))]


@pytest.mark.gpu
@pytest.mark.parametrize("name,make", BEYOND_63, ids=[b[0] for b in BEYOND_63])
def test_beyond_63_variables_equal_to_the_cpu_search(ctx, name, make):
    n, clauses = make()
    want = models_by_search(n, clauses)
    assert _as_ints(uniformity.enumerate_models_by_search(n, clauses, context=ctx), n) == want
    assert uniformity.count_models_by_search(n, clauses, context=ctx) == len(want)
    if "unsatisfiable" in name:
        assert want == []


@pytest.mark.gpu
def test_planted_64_holds_its_planted_assignment(ctx):
    n, clauses, hidden = synth.planted_3sat(64, seed=0)
    want = models_by_search(n, clauses)
    got = _as_ints(uniformity.enumerate_models_by_search(n, clauses, context=ctx), n)
    assert got == want
    assert sum(int(b) << i for i, b in enumerate(hidden)) in set(got)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [64, 65, 127, 128, 129, 1024])
def test_hand_made_formulas_across_word_boundaries(ctx, n):
    _, clauses = _boundary_formula(n, seed=n)
    want = models_by_search(n, clauses)
    assert _as_ints(uniformity.enumerate_models_by_search(n, clauses, context=ctx), n) == want
    assert uniformity.count_models_by_search(n, clauses, context=ctx) == len(want)
    with_empty = clauses + [[]]
    assert uniformity.enumerate_models_by_search(n, with_empty, context=ctx).shape == (0, (n + 63) // 64)
    assert uniformity.count_models_by_search(n, with_empty, context=ctx) == 0


@pytest.mark.gpu
def test_bench_formula_has_1272_models(ctx):
    n, clauses = synth.random_3sat(100, seed=0)
    assert uniformity.count_models_by_search(n, clauses, context=ctx) == 1272


def _raw_call(ctx, n_vars, clauses, out=None, capacity=0, nnz=None, lens=None, flat=None):
    lens = np.array([len(c) for c in clauses], dtype=np.int32) if lens is None else lens
    flat = np.array([l for c in clauses for l in c], dtype=np.int32) if flat is None else flat
    ip = C.POINTER(C.c_int32)
    count = C.c_longlong(-7)
    rc = ctx._lib.dsat_enumerate_models_search(ctx._h, n_vars, len(lens), int(flat.size if nnz is None else nnz),
                                               lens.ctypes.data_as(ip), flat.ctypes.data_as(ip),
                                               None if out is None else out.ctypes.data_as(C.POINTER(C.c_uint64)),
                                               capacity, C.byref(count))
    return rc, count.value


@pytest.mark.gpu
def test_counts_up_to_2_63_minus_1_and_overflow_refused(ctx):
    assert uniformity.count_models_by_search(64, [[1], [2]], context=ctx) == 2 ** 62
    assert uniformity.count_models_by_search(1024, [[v] for v in range(3, 965)], context=ctx) == 2 ** 62
    assert _raw_call(ctx, 63, []) == (DSAT_ERR_UNSUPPORTED, -1)              # 2^63
    assert _raw_call(ctx, 64, []) == (DSAT_ERR_UNSUPPORTED, -1)              # 64 free variables
    assert _raw_call(ctx, 65, [[1]]) == (DSAT_ERR_UNSUPPORTED, -1)
    # an open clause below variables that no clause holds: counted without branching on them, so these return at once
    assert uniformity.count_models_by_search(63, [[1, 2]], context=ctx) == 3 * 2 ** 61
    assert _raw_call(ctx, 66, [[1, 2]]) == (DSAT_ERR_UNSUPPORTED, -1)       # 3 * 2^64
    _, bench = synth.random_3sat(100, seed=0)
    assert _raw_call(ctx, 1024, bench) == (DSAT_ERR_UNSUPPORTED, -1)        # 1272 * 2^924
    assert uniformity.count_models_by_search(150, bench, context=ctx) == 1272 << 50
    assert uniformity.count_models_by_search(100, bench, context=ctx) == 1272     # the context is still usable


@pytest.mark.gpu
def test_variables_in_no_clause_above_the_formula(ctx):
    """A DIMACS header that declares more variables than the clauses use: the models of the used ones times every value
    of the unused ones, in order."""
    _, clauses = synth.random_3sat(80, seed=2)
    want = models_by_search(84, clauses)
    assert len(want) == 3473 * 16
    assert _as_ints(uniformity.enumerate_models_by_search(84, clauses, context=ctx), 84) == want
    assert uniformity.count_models_by_search(84, clauses, context=ctx) == len(want)


@pytest.mark.gpu
def test_variables_in_no_clause_between_used_ones(ctx):
    """Variables 41..44 in no clause, below used ones: writing the models out branches on them in order, and the
    subtrees without a model below them (random_3sat(80) at the threshold has many) are searched once, not 2^4 times."""
    _, clauses = synth.random_3sat(80, seed=1)
    shifted = [[l if abs(l) <= 40 else l + (4 if l > 0 else -4) for l in c] for c in clauses]
    want = models_by_search(84, shifted)
    assert len(want) == 9184 * 16
    assert _as_ints(uniformity.enumerate_models_by_search(84, shifted, context=ctx), 84) == want
    assert uniformity.count_models_by_search(84, shifted, context=ctx) == len(want)
    assert _raw_call(ctx, 1000, shifted) == (DSAT_ERR_UNSUPPORTED, -1)


@pytest.mark.gpu
def test_count_only_capacity_and_argument_checks(ctx):
    n, clauses = synth.random_3sat(80, seed=2)
    want = models_by_search(n, clauses)
    assert len(want) > 10
    lens = np.array([len(c) for c in clauses], dtype=np.int32)
    flat = np.array([l for c in clauses for l in c], dtype=np.int32)

    def call(n_vars=n, flat=flat, **kw):
        return _raw_call(ctx, n_vars, clauses, lens=lens, flat=flat, **kw)

    assert call() == (0, len(want))                                         # count only
    out = np.zeros((len(want), 2), dtype=np.uint64)
    assert call(out=out, capacity=len(want)) == (0, len(want))
    assert keys_to_ints(out, n) == want
    small = np.zeros((len(want) - 3, 2), dtype=np.uint64)
    assert call(out=small, capacity=len(small)) == (DSAT_ERR_ARG, len(want))    # with the required size
    assert keys_to_ints(small, n) == want[:len(small)]                          # the models that fit are written
    assert call(out=None, capacity=5)[0] == DSAT_ERR_ARG                        # null output with a capacity
    assert call(out=out, capacity=-1)[0] == DSAT_ERR_ARG
    for bad_n in (0, 1025):
        assert call(n_vars=bad_n)[0] == DSAT_ERR_ARG
    assert call(nnz=flat.size - 1)[0] == DSAT_ERR_ARG                           # lens do not sum to nnz
    bad = flat.copy()
    for lit in (0, 81, -81):
        bad[5] = lit
        assert call(flat=bad)[0] == DSAT_ERR_ARG
    out[:] = 0
    assert call(out=out, capacity=len(want)) == (0, len(want))                  # the context is still usable
    assert keys_to_ints(out, n) == want


@pytest.mark.gpu
def test_search_over_several_launches(ctx):
    """2^15 frontier nodes: the search takes more than one launch (dsat_model_search.cuh: CHUNK_NODES = 2^14), and the
    models of the later launch follow those of the first."""
    n, clauses = _chunked_formula()
    want = models_by_search(n, clauses)
    launches = ctx.launch_count()
    assert uniformity.count_models_by_search(n, clauses, context=ctx) == len(want)
    assert ctx.launch_count() - launches >= 3 * 15 + 2 * 2          # 15 levels of 3 launches, 2 chunks of count + scan
    assert _as_ints(uniformity.enumerate_models_by_search(n, clauses, context=ctx), n) == want


@pytest.mark.gpu
def test_search_leaves_the_context_state_untouched(ctx):
    from diffusionsat_b200 import graph as G
    from diffusionsat_b200.weights import load_weights
    n, clauses, _ = synth.planted_3sat(20, 80, seed=6)
    ctx.set_model(load_weights(FIXTURE))
    ctx.set_graph(G.build_unit_graph(n, clauses), chains=64, group_graphs=16)
    precision = ctx.get_precision()
    before = ctx.sample(32, 32, seed=11)
    models = uniformity.enumerate_models_by_search(n, clauses, context=ctx)
    uniformity.enumerate_models_by_search(*_chunked_formula(), context=ctx)        # several launches
    uniformity.count_models_by_search(100, synth.random_3sat(100, seed=0)[1], context=ctx)
    assert ctx.get_precision() == precision
    after = ctx.sample(32, 32, seed=11)
    for a, b in zip(before, after):
        np.testing.assert_array_equal(a, b)
    packed, is_sat = after[0], after[1].astype(bool)
    assert is_sat.any()
    assert set(keys_to_ints(packed[is_sat], n)) <= set(_as_ints(models, n))


# planted_3sat(72, 280, seed=1): 257 004 models.  The fixture was trained on n <= 30 and satisfies 2 of the 256 chains
# below (seed 3, fp32 on a B200); the run is deterministic, so the assertion that some chain is satisfied holds.
SAMPLER_FORMULA = (72, 280, 1)


@pytest.mark.gpu
def test_sampler_keys_beyond_64_variables_are_models(ctx):
    from diffusionsat_b200 import graph as G
    from diffusionsat_b200.weights import load_weights
    n, m, seed = SAMPLER_FORMULA
    _, clauses, _ = synth.planted_3sat(n, m, seed=seed)
    ctx.set_model(load_weights(FIXTURE))
    ctx.set_graph(G.build_unit_graph(n, clauses), chains=256, group_graphs=256)
    packed, is_sat = ctx.sample(64, 32, seed=3)[:2]
    is_sat = is_sat.astype(bool)
    assert packed.shape[1] == 2
    assert is_sat.sum() >= 1, "no chain satisfied the formula"
    models = set(_as_ints(uniformity.enumerate_models_by_search(n, clauses, context=ctx), n))
    assert set(keys_to_ints(packed[is_sat], n)) <= models
