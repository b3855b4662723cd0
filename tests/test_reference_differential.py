"""Differential fuzzing of the pure-Python host mirrors against the REFERENCE's own classes (utils/DimacsFile.py,
utils/VariableAssignment.py -- importable without TensorFlow).  The reference is not part of this repository: the tests run
where DIFFUSIONSAT_REFERENCE names a checkout of it and skip elsewhere; the committed golden vectors
(tests/test_host_golden.py) cover the same classes everywhere.  Never part of the GPU tier."""
import contextlib
import io
import os
import sys

import pytest
from hypothesis import given, settings
from hypothesis import strategies as st

REF = os.environ.get("DIFFUSIONSAT_REFERENCE", "")
pytestmark = pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, "utils")),
                                reason="DIFFUSIONSAT_REFERENCE does not name a checkout of the reference project")


def _ref():
    for p in (REF, os.path.join(REF, "utils")):
        if p not in sys.path:
            sys.path.append(p)
    from utils.DimacsFile import DimacsFile as RefDimacs
    from utils.VariableAssignment import VariableAssignment as RefAssignment
    return RefDimacs, RefAssignment


TOKENS = st.sampled_from(["0", "1", "-1", "2", "-2", "3", "7", "-7", "12", "p cnf", "p cnf 3 2", "p cnf 5", "c", "c hello", "v", "v 1 -2",
                          "--", "-- odd", "%", "x", "", " ", "  ", "00", "-0", "+3", "1 -2 0", "2 3 0 4", "p  cnf 4 4"])
LINES = st.lists(st.lists(TOKENS, max_size=5).map(" ".join), max_size=8).map("\n".join)


def _parse(cls, text):
    df = cls()
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            df.load_from_string(text)
    except Exception as exc:        # noqa: BLE001 - the exception type is part of the behaviour
        return ("error", type(exc).__name__)
    return ("ok", df.number_of_vars(), [list(c) for c in df.clauses()], {int(k): bool(v) for k, v in df.b_values.items()})


@settings(max_examples=400, deadline=None)
@given(LINES)
def test_dimacs_parser_agrees_with_the_reference_parser(text):
    from diffusionsat_b200.dimacs import DimacsFile
    RefDimacs, _ = _ref()
    assert _parse(DimacsFile, text) == _parse(RefDimacs, text), repr(text)


@settings(max_examples=200, deadline=None)
@given(st.integers(1, 70).flatmap(lambda n: st.tuples(
    st.just(n),
    st.lists(st.lists(st.integers(1, n).flatmap(lambda v: st.sampled_from([v, -v])), max_size=5), max_size=12),
    st.lists(st.booleans(), min_size=n, max_size=n))))
def test_variable_assignment_agrees_with_the_reference_class(case):
    from diffusionsat_b200.variable_assignment import VariableAssignment
    _, RefAssignment = _ref()
    n, clauses, bits = case
    clauses = [list(c) for c in clauses] + [[n]]             # the largest literal sizes the vector (reference :34-36)
    out = []
    for cls in (VariableAssignment, RefAssignment):
        a = cls(clauses=[list(c) for c in clauses])
        a.assign_all_from_bit_list([float(b) for b in bits])
        b = cls(n, [])
        b.assign_all_from_int(int(a))
        out.append((int(a), bool(a.satisfiable()), str(a), list(a.as_int_list()), b.values() == a.values()))
    assert out[0] == out[1]


@settings(max_examples=150, deadline=None)
@given(st.dictionaries(st.integers(0, 12), st.integers(1, 40), min_size=1, max_size=8),
       st.dictionaries(st.integers(0, 12), st.integers(1, 40), min_size=1, max_size=8))
def test_chi_square_agrees_with_the_reference_function(observed, expected):
    import math
    import warnings
    from diffusionsat_b200.uniformity import chi_square_likelihood
    _ref()
    from utils.chi_square import chi_square_likelihood as ref_chi

    def run(fn):
        try:
            with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
                warnings.simplefilter("ignore")
                return ("ok", float(fn(dict(observed), dict(expected))))
        except Exception as exc:        # noqa: BLE001 - scipy rejects sums that differ; both sides must do the same
            return ("error", type(exc).__name__)
    a, b = run(chi_square_likelihood), run(ref_chi)
    assert a[0] == b[0]
    if a[0] == "ok":
        assert (math.isnan(a[1]) and math.isnan(b[1])) or a[1] == pytest.approx(b[1], rel=1e-12, abs=1e-300)
    else:
        assert a[1] == b[1]
