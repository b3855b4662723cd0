"""Generate tests/golden/differential_golden.json: a fixed, seeded draw from the input grammars of
tests/test_reference_differential.py (DIMACS token soup, VariableAssignment cases, chi-square dict pairs whose key sets or
sums may differ) with the outcome of every case, so that the edge cases the fuzzing explores are checked on every machine.

    DIFFUSIONSAT_REFERENCE=<checkout of the original project> python tests/golden/make_differential_golden.py
    python tests/golden/make_differential_golden.py --mirror

With DIFFUSIONSAT_REFERENCE the outcomes are those of the original's own utils/DimacsFile.py, utils/VariableAssignment.py
and utils/chi_square.py ("source": "reference"); with --mirror they are those of this package's host mirrors
("source": "mirror").  tests/test_host_golden.py compares the host mirrors against the stored outcomes either way.
"""
import contextlib
import io
import json
import os
import sys
import warnings

import numpy as np

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "differential_golden.json")
TOKENS = ["0", "1", "-1", "2", "-2", "3", "7", "-7", "12", "p cnf", "p cnf 3 2", "p cnf 5", "c", "c hello", "v", "v 1 -2",
          "--", "-- odd", "%", "x", "", " ", "  ", "00", "-0", "+3", "1 -2 0", "2 3 0 4", "p  cnf 4 4"]


def draw_cases(seed=2025, n_texts=300, n_assign=120, n_chi=120):
    rng = np.random.default_rng(seed)
    texts = ["\n".join(" ".join(TOKENS[int(t)] for t in rng.integers(0, len(TOKENS), int(rng.integers(0, 6))))
                       for _ in range(int(rng.integers(0, 9)))) for _ in range(n_texts)]
    assign = []
    for _ in range(n_assign):
        n = int(rng.integers(1, 71))
        clauses = [[int(v) if rng.random() < 0.5 else -int(v) for v in rng.integers(1, n + 1, int(rng.integers(0, 6)))]
                   for _ in range(int(rng.integers(0, 13)))]
        assign.append({"n": n, "clauses": clauses, "bits": [int(b) for b in rng.integers(0, 2, n)]})
    chi = []
    for i in range(n_chi):
        pair = [{str(int(k)): int(rng.integers(1, 41)) for k in rng.integers(0, 13, int(rng.integers(1, 9)))}
                for _ in range(2)]
        if i % 3 == 0:          # equal sums (the expected counts a permutation of the observed ones): a p-value, not an error
            keys = list(pair[0])
            pair[1] = dict(zip(keys, (pair[0][k] for k in rng.permutation(keys))))
        chi.append({"observed": pair[0], "expected": pair[1]})
    return {"dimacs": texts, "assignment": assign, "chi_square": chi}


def outcomes(dimacs_cls, assignment_cls, chi_fn, cases):
    """The observable result of every case, in the form the differential tests compare."""
    out = {"dimacs": [], "assignment": [], "chi_square": []}
    for text in cases["dimacs"]:
        df = dimacs_cls()
        try:
            with contextlib.redirect_stdout(io.StringIO()):
                df.load_from_string(text)
            out["dimacs"].append(["ok", df.number_of_vars(), [[int(x) for x in c] for c in df.clauses()],
                                  sorted([int(k), bool(v)] for k, v in df.b_values.items())])
        except Exception as exc:        # noqa: BLE001 - the exception type is part of the behaviour
            out["dimacs"].append(["error", type(exc).__name__])
    for case in cases["assignment"]:
        clauses = [list(c) for c in case["clauses"]] + [[case["n"]]]     # the largest literal sizes the vector
        a = assignment_cls(clauses=[list(c) for c in clauses])
        a.assign_all_from_bit_list([float(b) for b in case["bits"]])
        b = assignment_cls(case["n"], [])
        b.assign_all_from_int(int(a))
        out["assignment"].append([str(int(a)), bool(a.satisfiable()), str(a), [int(x) for x in a.as_int_list()],
                                  bool(b.values() == a.values())])
    for case in cases["chi_square"]:
        obs = {int(k): v for k, v in case["observed"].items()}
        exp = {int(k): v for k, v in case["expected"].items()}
        try:
            with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
                warnings.simplefilter("ignore")
                p = float(chi_fn(dict(obs), dict(exp)))
            out["chi_square"].append(["ok", None if np.isnan(p) else p])
        except Exception as exc:        # noqa: BLE001 - scipy rejects sums that differ; the type must match
            out["chi_square"].append(["error", type(exc).__name__])
    return out


def main():
    ref = os.environ.get("DIFFUSIONSAT_REFERENCE", "")
    if ref:
        sys.path[:0] = [ref, os.path.join(ref, "utils")]
        from utils.DimacsFile import DimacsFile
        from utils.VariableAssignment import VariableAssignment
        from utils.chi_square import chi_square_likelihood
        source = "reference"
    elif "--mirror" in sys.argv:
        sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
        from diffusionsat_b200.dimacs import DimacsFile
        from diffusionsat_b200.uniformity import chi_square_likelihood
        from diffusionsat_b200.variable_assignment import VariableAssignment
        source = "mirror"
    else:
        sys.exit("set DIFFUSIONSAT_REFERENCE to a checkout of the original project, or pass --mirror")
    cases = draw_cases()
    gold = {"source": source, "cases": cases,
            "outcomes": outcomes(DimacsFile, VariableAssignment, chi_square_likelihood, cases)}
    with open(OUT, "w") as handle:
        json.dump(gold, handle, separators=(",", ":"), sort_keys=True)
    print("wrote", OUT, source, {k: len(v) for k, v in cases.items()})


if __name__ == "__main__":
    main()
