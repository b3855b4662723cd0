"""Uniformity statistics of a sample histogram (host side, scipy) and the exact model set they compare against.

Mirror of reference ``utils/chi_square.py:7-36`` (``chi_square_likelihood``) and of the comparison made in
``diffusion_metrics.py:111,130-147`` (histogram against the ideal ``k`` samples per solution).  The model set comes from
:func:`enumerate_models` (GPU brute force, ``dsat_enumerate_models``), which replaces the reference's unigen/approxmc
counting (``utils/AllSolutions.py:44-68``).
"""

from __future__ import annotations

from scipy import stats

MAX_ENUMERATION_VARS = 63


def _models_call(n_vars, clauses, count_only, context, device):
    if not 1 <= int(n_vars) <= MAX_ENUMERATION_VARS:
        raise ValueError("exact model enumeration takes 1..%d variables, got %d" % (MAX_ENUMERATION_VARS, n_vars))
    from . import _lib
    ctx = context if context is not None else _lib.Context(device)
    try:
        return ctx.enumerate_models(int(n_vars), [list(c) for c in clauses], count_only=count_only)
    finally:
        if context is None:
            ctx.close()


def enumerate_models(n_vars: int, clauses, *, context=None, device: int = 0):
    """Every model of a formula over ``n_vars <= 63`` variables as ``uint64`` integers in the reference encoding (x1 = bit
    0), ascending; the same list as ``synth.enumerate_solutions`` for any size the GPU can go through (2^n assignments).
    ``context``: a ``_lib.Context`` to run on (its model, graph and sampling state are left as they are); otherwise a
    context on ``device`` is created for the call."""
    return _models_call(n_vars, clauses, False, context, device)


def count_models(n_vars: int, clauses, *, context=None, device: int = 0) -> int:
    """Number of models of the formula (:func:`enumerate_models` without writing them out)."""
    return _models_call(n_vars, clauses, True, context, device)


MAX_SEARCH_VARS = 1024


def _search_call(n_vars, clauses, count_only, context, device):
    if not 1 <= int(n_vars) <= MAX_SEARCH_VARS:
        raise ValueError("model search takes 1..%d variables, got %d" % (MAX_SEARCH_VARS, n_vars))
    from . import _lib
    ctx = context if context is not None else _lib.Context(device)
    try:
        return ctx.enumerate_models_search(int(n_vars), [list(c) for c in clauses], count_only=count_only)
    finally:
        if context is None:
            ctx.close()


def enumerate_models_by_search(n_vars: int, clauses, *, context=None, device: int = 0):
    """Every model of a formula over ``n_vars <= 1024`` variables by ordered search on the GPU
    (``dsat_enumerate_models_search``): ``uint64 [K, ceil(n_vars / 64)]``, word 0 = variables 1..64 (the layout of the
    sampler's keys; ``dist.keys_to_ints`` turns them into ints), ascending.  For ``n_vars <= 63`` the same models as
    :func:`enumerate_models`.  Its cost follows the search tree (which skips every subtree with a failed clause), not
    2^n.  ``context`` and ``device`` as in :func:`enumerate_models`."""
    return _search_call(n_vars, clauses, False, context, device)


def count_models_by_search(n_vars: int, clauses, *, context=None, device: int = 0) -> int:
    """Number of models of the formula (:func:`enumerate_models_by_search` without writing them out)."""
    return _search_call(n_vars, clauses, True, context, device)


def chi_square_likelihood(observed: dict, expected: dict) -> float:
    """p-value of the chi-square test of ``observed`` against ``expected`` (dicts id -> count).
    Ids missing on one side count as zero there; a single shared id is reported as p = 1."""
    if len(observed) == 1 and len(expected) == 1:
        return 1.0
    ids = list(expected) + [k for k in observed if k not in expected]
    obs = [observed.get(k, 0) for k in ids]
    exp = [expected.get(k, 0) for k in ids]
    _, p = stats.chisquare(obs, exp)
    return p


def chi_square_vs_ideal(histogram: dict, solutions, samples_per_solution: float | None = None):
    """Chi-square statistic and p-value of a ``{solution_as_int: count}`` histogram against the uniform
    distribution over ``solutions`` (``diffusion_metrics.py:111,137``: ideal = k per solution)."""
    solutions = list(solutions)
    total = sum(histogram.get(s, 0) for s in solutions)
    if samples_per_solution is None:
        samples_per_solution = total / max(len(solutions), 1)
    obs = [histogram.get(s, 0) for s in solutions]
    exp = [samples_per_solution] * len(solutions)
    if len(solutions) < 2 or total == 0:
        return 0.0, 1.0
    chisq, p = stats.chisquare(obs, exp)
    return float(chisq), float(p)
