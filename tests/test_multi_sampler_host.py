"""Host logic of MultiDiffusionSampler with a fake context (no GPU): the launch planner, the union layout handed to
dsat_set_batches (early-exit groups and per-graph noise bases), the row cap, formulas finishing or aborting in different
launches, the per-formula IndexError, and keys trimmed to each formula's word count."""
import numpy as np
import pytest

from diffusionsat_b200 import synth
from diffusionsat_b200.graph import chains_per_reference_batch
from diffusionsat_b200.sampler import MultiDiffusionSampler, ROWS_CAP, chains_for_rate, launch_layout, plan_launch


class _FakeContext:
    """Stands in for _lib.Context: SAT flags come from a per-formula rule keyed by the chain's noise base, keys are the
    global chain id spread over the launch's word count."""

    def __init__(self, sat_rule, words=2):
        self.sat_rule, self.words = sat_rule, words
        self.graph, self.chains = None, 0
        self.launches = []

    def set_sampling(self, mode):
        pass

    def set_graph(self, unit, chains, group_graphs=0):
        self.graph, self.chains = unit, chains

    def set_batches(self, group_seg, noise_base=None):
        self.group_seg, self.noise_base = np.asarray(group_seg), np.asarray(noise_base)
        self.launches.append((self.group_seg.copy(), self.noise_base.copy(), self.graph.n_graphs,
                              set(np.diff(self.graph.var_seg).tolist())))

    def sample_enqueue(self, n_steps, n_rounds, seed=0, chain_offset=0):
        assert chain_offset == 0
        n_per = np.diff(self.graph.var_seg).astype(np.uint64)
        self.chain_ids = self.noise_base // n_per             # global chain id of every copy
        self.n_per = n_per
        self.sat = np.array([self.sat_rule(int(n), int(c)) for n, c in zip(n_per, self.chain_ids)], dtype=np.uint8)

    def sample_fetch_sat(self):
        return self.sat.copy()

    def hist_reduce_segments(self, graph_seg, limits):
        out = []
        for s in range(len(limits)):
            g0 = int(graph_seg[s])
            sel = [g for g in range(g0, g0 + int(limits[s])) if self.sat[g]]
            keys = {}
            for g in sel:
                k = int(self.chain_ids[g]) % 5                  # a few distinct "assignments"
                keys[k] = keys.get(k, 0) + 1
            ks = sorted(keys)
            arr = np.zeros((len(ks), self.words), dtype=np.uint64)
            arr[:, 0] = ks
            out.append((arr, np.array([keys[k] for k in ks], dtype=np.int64)))
        return out, sum(len(v) for v in out)


class _FakeModel:
    def __init__(self, ctx):
        self.ctx, self._graph_key = ctx, None


def _write(tmp_path, specs):
    files = []
    for i, (n, m, seed) in enumerate(specs):
        n_vars, clauses, _ = synth.planted_3sat(n, m, seed=seed)
        p = tmp_path / ("f%d.cnf" % i)
        p.write_text(synth.dimacs_text(n_vars, clauses))
        files.append(str(p))
    return files


def _sampler(monkeypatch, files, ctx, **kw):
    from diffusionsat_b200 import sampler as S
    monkeypatch.setattr(S, "QuerySAT", lambda **a: _FakeModel(ctx))
    return MultiDiffusionSampler(None, files, **kw)


def _solo_reference(n, m_clauses, batch, rule, n_samples, chain_offset=0, rate=0.005):
    """The per-file DiffusionSampler loop (stop rules per reference batch, one batch at a time) on the same rule."""
    from diffusionsat_b200.sampler import consume_batches
    hist, total, sat_total, need, pos, stop = {}, 0, 0, n_samples, chain_offset, False
    while need > 0 and not stop:
        c = chains_for_rate(batch, n, m_clauses, need, sat_total / total if total else None)
        flags = np.array([rule(n, pos + j) for j in range(c)], dtype=np.uint8)
        used, sat_used, stop = consume_batches(flags, batch, need, total, sat_total, rate)
        for j in range(used):
            if flags[j]:
                hist[(pos + j) % 5] = hist.get((pos + j) % 5, 0) + 1
        total, sat_total, need, pos = total + used, sat_total + sat_used, need - sat_used, pos + c
    return hist, total, sat_total, pos - chain_offset, stop


def test_layout_groups_and_noise_bases(tmp_path, monkeypatch):
    files = _write(tmp_path, [(20, 60, 1), (30, 100, 2), (24, 80, 3)])
    ctx = _FakeContext(lambda n, c: 1)
    ms = _sampler(monkeypatch, files, ctx, chain_offset=7, max_nodes_per_batch=300)
    f = ms.formulas
    assert [x.batch_chains for x in f] == [chains_per_reference_batch(20, 60, 300), chains_per_reference_batch(30, 100, 300),
                                           chains_per_reference_batch(24, 80, 300)] == [3, 1, 2]
    f[1].launched = 5                                  # formula 1 already launched 5 chains in this call
    plan = [(0, 7), (1, 3), (2, 4)]                    # 7 chains of a batch-3 formula: groups 3, 3, 1
    graph_seg, group_seg, base = launch_layout(f, plan, chain_offset=7)
    assert graph_seg.tolist() == [0, 7, 10, 14]
    assert group_seg.tolist() == [0, 3, 6, 7, 8, 9, 10, 12, 14]
    want = [(7 + j) * 20 for j in range(7)] + [(7 + 5 + j) * 30 for j in range(3)] + [(7 + j) * 24 for j in range(4)]
    assert base.dtype == np.uint64 and base.tolist() == want


def test_planner_row_cap_and_file_order(tmp_path, monkeypatch):
    files = _write(tmp_path, [(20, 60, 1), (30, 100, 2), (24, 80, 3)])
    ms = _sampler(monkeypatch, files, _FakeContext(lambda n, c: 1), max_nodes_per_batch=300)
    for f in ms.formulas:
        f.start(64)
    full = plan_launch(ms.formulas)
    assert [k for k, _ in full] == [0, 1, 2]
    assert [c for _, c in full] == [f.next_chains() for f in ms.formulas]
    rows = [c * ms.formulas[k].rows_per_chain for k, c in full]
    assert sum(rows) <= ROWS_CAP
    # a cap that holds the first two: the third waits; a cap below the first: the first still goes alone
    assert [k for k, _ in plan_launch(ms.formulas, rows_cap=rows[0] + rows[1])] == [0, 1]
    assert [k for k, _ in plan_launch(ms.formulas, rows_cap=1)] == [0]
    # the second does not fit, so it and everything after it wait, in file order
    assert [k for k, _ in plan_launch(ms.formulas, rows_cap=rows[0] + rows[2])] == [0]
    ms.formulas[0].stopped = True
    assert [k for k, _ in plan_launch(ms.formulas)] == [1, 2]


def test_formulas_finish_and_abort_in_different_launches(tmp_path, monkeypatch):
    files = _write(tmp_path, [(20, 60, 1), (30, 100, 2), (24, 80, 3), (22, 70, 4)])

    def rule(n, c):                     # per formula (keyed by n): every chain, one in seven, only the first, one in three
        return {20: 1, 30: int(c % 7 == 4), 24: int(c == 11), 22: int(c % 3 == 2)}[n]

    ctx = _FakeContext(rule)
    ms = _sampler(monkeypatch, files, ctx, max_nodes_per_batch=300, chain_offset=11)
    need = [40, 25, 10, 0]
    tables = ms.samples_table(need)
    stats, first_call = ms.last_stats, list(ctx.launches)
    assert len(first_call) >= 2
    for k, (n, m) in enumerate([(20, 60), (30, 100), (24, 80), (22, 70)]):
        want, total, sat, launched, stop = _solo_reference(n, m, ms.formulas[k].batch_chains, rule, need[k], chain_offset=11)
        keys, counts = tables[k]
        assert keys.shape[1] == 1                       # trimmed to ceil(n/64) words although the launch had 2
        assert dict(zip(keys[:, 0].tolist(), counts.tolist())) == want, k
        assert (stats[k]["total"], stats[k]["sat"], stats[k]["chains_launched"], stats[k]["stopped_on_rate"]) == \
            (total, sat, launched, stop), k
    assert stats[1]["sat"] == 25 and stats[2]["stopped_on_rate"] and not stats[0]["stopped_on_rate"]
    assert stats[3] == {"total": 0, "sat": 0, "chains_launched": 0, "distinct": 0, "stopped_on_rate": False}
    # formula 0 (20 variables) is done after the first launch and formula 3 asked for nothing: later launches hold neither
    assert first_call[0][3] == {20, 30, 24}
    assert all(sizes <= {30, 24} for _, _, _, sizes in first_call[1:])
    # a second call continues with fresh chains: the same as a solo sampler's second call when launches line up
    again = ms.samples(need)
    assert sum(again[0].values()) == 40 and set(again[0]) == set(range(5))
    assert ms.formulas[0].launched_before == stats[0]["chains_launched"] + ms.last_stats[0]["chains_launched"]
    ms.reset_chains()
    assert [dict(zip(k[:, 0].tolist(), c.tolist())) for k, c in ms.samples_table(need)] == \
        [dict(zip(k[:, 0].tolist(), c.tolist())) for k, c in tables]


def test_index_error_before_any_launch(tmp_path, monkeypatch):
    files = _write(tmp_path, [(20, 60, 1)])
    bad = tmp_path / "bad.cnf"
    bad.write_text("p cnf 4 2\n1 -2 0\n2 3 0\n")        # variable 4 never occurs
    ctx = _FakeContext(lambda n, c: 1)
    ms = _sampler(monkeypatch, files + [str(bad)], ctx, max_nodes_per_batch=300)
    with pytest.raises(IndexError):
        ms.samples(5)
    assert ctx.launches == []
    with pytest.raises(ValueError):
        ms.samples([1, 2, 3])
