"""CPU tests: host-side mirrors and the oracle against golden vectors produced by the reference's own
pure-Python modules (tests/golden/make_golden.py) and the known answers in the reference's tests."""
import json
import os

import numpy as np
import pytest

from diffusionsat_b200 import graph as G
from diffusionsat_b200 import synth
from diffusionsat_b200.dimacs import DimacsFile
from diffusionsat_b200.variable_assignment import VariableAssignment
from oracle import querysat_oracle as O

GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "host_golden.json")))


@pytest.mark.parametrize("case", GOLD["dimacs_parse"], ids=lambda c: repr(c["text"][:18]))
def test_dimacs_parser_matches_reference(case):
    df = DimacsFile()
    if "error" in case:
        with pytest.raises(Exception) as info:
            df.load_from_string(case["text"])
        assert type(info.value).__name__ == case["error"]
        return
    df.load_from_string(case["text"])
    assert df.number_of_vars() == case["n_vars"]
    assert df.clauses() == case["clauses"]
    assert {str(k): v for k, v in df.b_values.items()} == case["b_values"]
    assert str(df) == case["str"]


@pytest.mark.parametrize("case", GOLD["reduce_clauses"], ids=lambda c: str(len(c["clauses"])))
def test_reduce_clauses_matches_reference(case):
    df = DimacsFile(clauses=[list(c) for c in case["clauses"]])
    df.reduce_clauses()
    assert sorted(df.clauses(), key=lambda c: (len(c), c)) == case["reduced_sorted"]
    assert [len(c) for c in df.clauses()] == case["lengths"]          # sorted by length, as the reference


def test_reduce_clauses_reference_known_answers():
    # reference utils/test_DimacsFile.py:3-21
    for clauses, want in (([[1, 2], [1, 2], [3]], [[3], [1, 2]]), ([[1, 2, 3], [1, 2], [3]], [[3], [1, 2]]),
                          ([[1, 2, -3], [1, -2], [1]], [[1]])):
        df = DimacsFile(clauses=clauses)
        df.reduce_clauses()
        assert df.clauses() == want


@pytest.mark.parametrize("case", GOLD["variable_assignment"], ids=lambda c: str(c["n"]))
def test_variable_assignment_matches_reference(case):
    a = VariableAssignment(clauses=case["clauses"]) if case["clauses"] else VariableAssignment(case["n"], [])
    a.assign_all_from_bit_list(case["bits"])
    assert str(int(a)) == case["int"]
    assert a.satisfiable() == case["sat"]
    assert str(a) == case["str"]
    assert a.as_int_list() == case["int_list"]
    b = VariableAssignment(case["n"], [])
    b.assign_all_from_int(int(case["int"]))
    assert b.values() == a.values()
    # the oracle's restatements of the same two functions
    assert str(O.encode_assignment(case["bits"])) == case["int"]
    assert O._satisfiable_py([bool(x) for x in case["bits"]], case["clauses"]) == case["sat"]


def test_variable_assignment_known_answer():
    a = VariableAssignment(3, [])
    a.assign_all_from_int_list([1, 2, 3])
    assert int(a) == 7                                   # reference utils/VariableAssignment.py:109-112


@pytest.mark.parametrize("case", GOLD["adj_indices"], ids=lambda c: str(c["n"]))
def test_adjacency_indices_match_reference(case):
    pos, neg = G.compute_adj_indices(case["clauses"])
    assert pos == case["pos"] and neg == case["neg"]
    # CSR/CSC built for the kernels hold exactly the same multiset of (literal, clause) pairs
    unit = G.build_unit_graph(case["n"], case["clauses"])
    want = sorted([(2 * v, c) for v, c in case["pos"]] + [(2 * v + 1, c) for v, c in case["neg"]])
    csr = sorted((int(unit.cl_lit[e]), j) for j in range(unit.n_clauses)
                 for e in range(unit.cl_rowptr[j], unit.cl_rowptr[j + 1]))
    csc = sorted((l, int(unit.lit_clause[e])) for l in range(2 * unit.n_vars)
                 for e in range(unit.lit_rowptr[l], unit.lit_rowptr[l + 1]))
    assert csr == want and csc == want
    # reference-layout COO regenerated from the unit graph (one chain) equals the reference's lists
    coo, shape = unit.reference_coo(1)
    n = case["n"]
    assert shape == (2 * n, len(case["clauses"]))
    assert coo.tolist() == [list(p) for p in case["pos"]] + [[v + n, c] for v, c in case["neg"]]
    # inside a clause the literals are ordered by the reference literal row (sign*n + var)
    for j in range(unit.n_clauses):
        codes = unit.cl_lit[unit.cl_rowptr[j]:unit.cl_rowptr[j + 1]]
        rows = (codes & 1) * n + (codes >> 1)
        assert np.all(np.diff(rows) >= 0)
    for l in range(2 * n):
        assert np.all(np.diff(unit.lit_clause[unit.lit_rowptr[l]:unit.lit_rowptr[l + 1]]) >= 0)


def test_oracle_graph_layout_matches_reference_indices():
    case = GOLD["adj_indices"][0]
    n, clauses = case["n"], case["clauses"]
    g = O.OracleGraph.copies(n, clauses, 3)
    off_pos = [(v + c * n, j + c * len(clauses)) for c in range(3) for v, j in case["pos"]]
    off_neg = [(v + c * n + 3 * n, j + c * len(clauses)) for c in range(3) for v, j in case["neg"]]
    got = list(zip(g.lit_row.tolist(), g.clause.tolist()))
    assert got == off_pos + off_neg                       # all positives, then all negatives (SatSpecifics.py:24-35)
    unit = G.build_unit_graph(n, clauses)
    coo, shape = unit.reference_coo(3)
    assert coo.tolist() == [list(p) for p in got] and shape == (6 * n, 3 * len(clauses))


@pytest.mark.parametrize("case", GOLD["chi_square"], ids=lambda c: str(len(c["observed"])))
def test_chi_square_matches_reference(case, capsys):
    from diffusionsat_b200.uniformity import chi_square_likelihood
    p = chi_square_likelihood({int(k): v for k, v in case["observed"].items()},
                              {int(k): v for k, v in case["expected"].items()})
    assert p == pytest.approx(case["p"], rel=1e-12, abs=1e-300)


def test_solution_count_known_answer():
    # reference utils/test_AllSolutions.py:6,18 : 14 models
    assert len(synth.enumerate_solutions(5, [[-1, 2], [1, -2], [-3, 4, 5]])) == 14


def test_degree_weights_and_batch_rule():
    n, clauses = synth.random_3sat(30, seed=0)
    assert len(clauses) == 133                           # int(4.258 n + 58.26 n^(-2/3)), data/CNFGen.py:42-43
    unit = G.build_unit_graph(n, clauses)
    deg = unit.lit_degree()
    assert deg.sum() == 399
    np.testing.assert_allclose(unit.degree_weight(), 1 / np.sqrt(np.maximum(deg, 1)), rtol=1e-7)
    np.testing.assert_allclose(unit.var_degree_weight(), 4 / np.sqrt(np.maximum(deg[0::2] + deg[1::2], 1)), rtol=1e-7)
    np.testing.assert_allclose(unit.rev_degree_weight(), 1 / np.sqrt(3.0), rtol=1e-7)
    assert G.chains_per_reference_batch(30, 133) == 103  # floor(20000 / (2n+m)), SURVEY.md section 8
    assert G.chains_per_reference_batch(100, 430) == 31
    assert G.chains_per_reference_batch(250, 1065) == 12
    assert G.chains_per_reference_batch(20000, 1) == 1   # the first formula always fits (data/dimac.py:281)


def test_union_graph_and_reference_coo_roundtrip():
    formulas = [synth.random_ksat_mixed(int(n), int(m), seed=s) for s, (n, m) in enumerate([(5, 9), (3, 4), (8, 20)])]
    union = G.build_union_graph(formulas)
    assert union.n_graphs == 3 and union.var_seg.tolist() == [0, 5, 8, 16] and union.clause_seg.tolist() == [0, 9, 13, 33]
    coo, shape = union.reference_coo(1)
    vg = np.repeat(np.arange(3), [5, 3, 8])
    cg = np.repeat(np.arange(3), [9, 4, 20])
    back = G.unit_graph_from_reference_coo(coo, shape, vg, cg)
    for name in ("cl_rowptr", "cl_lit", "lit_rowptr", "lit_clause", "var_seg", "clause_seg"):
        np.testing.assert_array_equal(getattr(back, name), getattr(union, name))
    og = O.OracleGraph.from_formulas(formulas)
    assert list(zip(og.lit_row.tolist(), og.clause.tolist())) == [tuple(p) for p in coo.tolist()]


def test_is_graph_sat_matches_clause_by_clause_check():
    """Host restatement of reference utils/sat.py:165-180 against a literal-by-literal evaluation."""
    from diffusionsat_b200 import graph as G, synth
    from diffusionsat_b200.query_sat import is_graph_sat
    rng = np.random.default_rng(0)
    formulas = [synth.random_ksat_mixed(int(rng.integers(3, 12)), int(rng.integers(2, 20)), seed=s) for s in range(6)]
    formulas.append((3, [[1], [-1]]))                              # unsatisfiable
    formulas.append((2, [[1, 2], []]))                             # empty clause is never satisfied
    union = G.build_union_graph(formulas)
    coo, shape = union.reference_coo(1)
    vg = np.repeat(np.arange(len(formulas)), [n for n, _ in formulas])
    cg = np.repeat(np.arange(len(formulas)), [len(c) for _, c in formulas])
    for trial in range(5):
        logits = rng.standard_normal(union.n_vars).astype(np.float32)
        logits[rng.integers(0, union.n_vars)] = 0.0                # sigmoid == 0.5 rounds to 0 (half to even)
        got = is_graph_sat(logits, coo, shape, cg, len(formulas))
        off = 0
        for gi, (n, clauses) in enumerate(formulas):
            bits = logits[off:off + n] > 0
            ok = all(any((bits[abs(l) - 1] if l > 0 else not bits[abs(l) - 1]) for l in c) for c in clauses)
            assert got[gi] == float(ok), (trial, gi)
            off += n


def test_sat_checks_match_the_reference_functions_run_over_the_shim():
    """``is_graph_sat`` (host, predict_step) and the oracle's ``is_batch_sat`` (early exit) against flags computed by the
    reference's own ``utils/sat.py:118-124,165-180`` (tests/golden/make_sat_check_golden.py): unsatisfiable formula, empty
    clause, repeated literals, logits of exactly 0 (half-to-even rounding)."""
    import ast
    import os
    import torch
    from diffusionsat_b200 import graph as G
    from diffusionsat_b200.query_sat import is_graph_sat
    from oracle import querysat_oracle as O
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sat_check_golden.npz"))
    formulas = ast.literal_eval(str(gold["formulas"][0]))
    union = G.build_union_graph(formulas)
    coo, shape = union.reference_coo(1)
    cg = np.repeat(np.arange(len(formulas)), [len(c) for _, c in formulas])
    assert gold["graph_sat"].shape == (len(gold["logits"]), len(formulas))
    assert 0 < gold["graph_sat"].sum() < gold["graph_sat"].size               # both outcomes occur
    for z, want in zip(gold["logits"], gold["graph_sat"]):
        np.testing.assert_array_equal(is_graph_sat(z, coo, shape, cg, len(formulas)), want)
    off = 0
    for g, (n_vars, clauses) in enumerate(formulas):
        og = O.OracleGraph.from_formulas([(n_vars, clauses)])
        for t, z in enumerate(gold["logits"]):
            got = float(O.is_batch_sat(torch.from_numpy(z[off:off + n_vars].copy()).reshape(-1, 1), og))
            assert got == float(gold["batch_sat_per_formula"][t, g]), (g, t)
        off += n_vars


def test_input_helpers_match_the_reference_functions_run_over_the_shim():
    """numpy restatements in diffusionsat_b200/query_sat.py against the reference's module-level helpers
    (model/query_sat.py:55-82, tests/golden/make_helper_golden.py) with the same injected uniform draws."""
    import os
    from diffusionsat_b200 import query_sat as Q
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "helper_golden.npz"))
    assert Q.t_power == float(gold["t_power"])
    np.testing.assert_array_equal(Q.randomized_rounding_tf(gold["rr_x"], noise=gold["rr_u"]), gold["rr_out"])
    assert gold["rr_out"][:4, 0].tolist() == [0.0, 1.0, 1.0, 1.0]           # floor(x0 + u) on the boundaries
    for i in range(3):
        np.testing.assert_allclose(Q.distribution_at_time(gold["rr_x"], np.float32(gold["dat_%d_t" % i])),
                                   gold["dat_%d_out" % i], rtol=0, atol=1e-7)
    np.testing.assert_array_equal(Q.add_t_emb(gold["rr_x"], 0.625), gold["emb_out"])

    class Feed:                                     # the generator fed the same uniforms to every call
        def random(self, shape, dtype=np.float32):
            return gold["rr_u"].reshape(shape).astype(dtype)
    for i in range(3):
        got = Q.construct_training_input(gold["cti_bits"], float(gold["cti_%d_t" % i]), rng=Feed())
        np.testing.assert_array_equal(got, gold["cti_%d_out" % i])


def test_batching_rules_match_the_reference_code():
    """``chains_per_reference_batch``, ``pack_batches`` and the variable shift of ``build_union_graph`` against the
    reference's own ``BatchedDimacsDataset`` methods (data/dimac.py:165-174,267-293; tests/golden/make_batching_golden.py)."""
    import json
    import os
    from diffusionsat_b200 import dist as D, graph as G
    gold = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "batching_golden.json")))
    for c in gold["copies"]:
        assert G.sat_node_count(c["n_vars"], c["n_clauses"]) == c["nodes"]
        got = G.chains_per_reference_batch(c["n_vars"], c["n_clauses"], c["max_nodes"])
        assert got == c["first_batch"] and all(b == got for b in c["batch_sizes"]), c
    assert [c["first_batch"] for c in gold["copies"] if c["max_nodes"] == 20000][:3] == [103, 31, 12]     # n = 30, 100, 250

    class Sized:                                    # only len() of the clause list matters to the packing rule
        def __init__(self, m):
            self.m = m

        def __len__(self):
            return self.m
    for m in gold["mixed"]:
        formulas = [(n, Sized(k)) for n, k in m["sizes"]]
        assert D.pack_batches(formulas, m["max_nodes"], drop_overflow=True) == m["batches"]
        ours = D.pack_batches(formulas, m["max_nodes"])
        assert [i for b in ours for i in b] == list(range(len(formulas)))                  # the default loses nothing
        assert ours[0] == m["batches"][0]                                                  # identical up to the first drop
        assert m["dropped"] and m["dropped"][0] == ours[1][0]                               # ... which opens our second batch
    for s in gold["shift"]:
        union = G.build_union_graph([(s["offset"], [[1]] if s["offset"] else []), (3, s["clauses"])]) if s["offset"] \
            else G.build_union_graph([(3, s["clauses"])])
        assert union.clauses[-len(s["clauses"]):] == s["shifted"]


@pytest.mark.parametrize("tag", ["mixed", "edge", "copies"])
def test_batch_tensors_match_the_reference_create_adj_matrices(tag):
    """The reference-layout COO of a union (``UnitGraph.reference_coo``), its way back (``unit_graph_from_reference_coo``) and
    the membership adapters against ``SatSpecifics.create_adj_matrices`` run on ``shift_clause`` + ``compute_adj_indices``
    output (data/SatSpecifics.py:21-69, data/dimac.py:165-170,239-241; tests/golden/make_adjacency_golden.py)."""
    import ast
    import os
    from diffusionsat_b200 import graph as G
    from diffusionsat_b200.query_sat import _coo, _graph_ids
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "adjacency_golden.npz"))
    formulas = ast.literal_eval(str(gold[tag + "_formulas"][0]))
    union = G.build_union_graph(formulas)
    coo, shape = union.reference_coo(1)
    np.testing.assert_array_equal(coo, gold[tag + "_adj_indices"])             # same pairs in the same storage order
    assert tuple(shape) == tuple(gold[tag + "_adj_shape"].tolist())
    # membership matrices -> per-node graph ids
    vg, n_graphs = _graph_ids((gold[tag + "_vg_indices"], gold[tag + "_vg_shape"]), union.n_vars)
    cg, n_graphs_c = _graph_ids((gold[tag + "_cg_indices"], gold[tag + "_cg_shape"]), union.n_clauses)
    assert n_graphs == n_graphs_c == len(formulas)
    np.testing.assert_array_equal(vg, np.repeat(np.arange(len(formulas)), [n for n, _ in formulas]))
    np.testing.assert_array_equal(cg, np.repeat(np.arange(len(formulas)), [len(c) for _, c in formulas]))
    # and back: the graph rebuilt from the reference's tensors is the graph built from the formulas
    idx, shp = _coo((gold[tag + "_adj_indices"], gold[tag + "_adj_shape"]))
    back = G.unit_graph_from_reference_coo(idx, shp, vg, cg)
    for name in ("cl_rowptr", "cl_lit", "lit_rowptr", "lit_clause", "var_seg", "clause_seg"):
        np.testing.assert_array_equal(getattr(back, name), getattr(union, name), err_msg=name)


def test_host_mirrors_match_the_stored_differential_cases():
    """A fixed, seeded draw from the input grammars of the differential fuzz tests (DIMACS token soup, VariableAssignment
    cases, chi-square dict pairs with differing key sets or sums) and the outcome of every case, so that those edge cases
    are checked where the original project is not at hand.  The file's `source` says which implementation produced the
    outcomes (make_differential_golden.py: the original's classes where DIFFUSIONSAT_REFERENCE is set, else the mirrors)."""
    import importlib.util
    import math
    from diffusionsat_b200.uniformity import chi_square_likelihood
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    spec = importlib.util.spec_from_file_location("make_differential_golden", os.path.join(here, "make_differential_golden.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    gold = json.load(open(os.path.join(here, "differential_golden.json")))
    assert gold["cases"] == json.loads(json.dumps(gen.draw_cases()))          # the stored inputs are the generator's draw
    got = gen.outcomes(DimacsFile, VariableAssignment, chi_square_likelihood, gold["cases"])
    want = gold["outcomes"]
    for kind in ("dimacs", "assignment"):
        for case, g, w in zip(gold["cases"][kind], got[kind], want[kind]):
            assert json.loads(json.dumps(g)) == w, (kind, case)
    for case, g, w in zip(gold["cases"]["chi_square"], got["chi_square"], want["chi_square"]):
        assert g[0] == w[0], case
        if g[0] == "error" or w[1] is None or g[1] is None:
            assert g[1] == w[1], case
        else:
            assert math.isclose(g[1], w[1], rel_tol=1e-12, abs_tol=1e-300), case
    assert {k: len(v) for k, v in want.items()} == {k: len(v) for k, v in got.items()} == {"dimacs": 300, "assignment": 120,
                                                                                           "chi_square": 120}
