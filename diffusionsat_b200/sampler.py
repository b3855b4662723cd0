"""``DiffusionSampler(model_path, dimacs_filename).samples(n)`` on the GPU.

Mirror of reference ``satuniformity/DiffusionSampler.py``: module constants ``:17-21``,
``reverse_distribution_step_theoretic`` ``:29-37``, ``predict`` ``:40-63``, ``diffusion`` ``:78-191``,
``DiffusionSampler.__init__`` ``:197-213``, ``_prepare_checkpoints`` ``:215-227``, ``samples`` ``:229-311``.

Differences that are deliberate and documented in DESIGN.md:

* the dataset detour (solution counting with unigen/approxmc, per-copy DIMACS files, GZIP TFRecords;
  ``data/diffusion_sat_instances.py:80-94``, ``data/dimac.py:129-211``) is replaced by building the CSR/CSC
  arrays of the one formula directly; the batch composition rule is kept (``floor(max_nodes/(2n+m))``
  copies per reference batch, each its own early-exit group);
* several reference batches run in one launch; they are consumed batch by batch in order, with the
  reference's stop rules (exactly ``n`` SAT samples; abort below 0.5 % SAT rate), so the returned
  histogram does not depend on how many batches a launch holds;
* ``model_path`` is the reference's TensorFlow checkpoint directory (read without TensorFlow,
  :mod:`diffusionsat_b200.tf_checkpoint`) or a ``.npz`` from :func:`diffusionsat_b200.weights.save_weights`; a missing file prints
  "Checkpoint not found!" and continues with seeded random weights, as the reference does.
"""

from __future__ import annotations

import numpy as np

from . import _lib
from .dimacs import DimacsFile
from .graph import MAX_NODES_PER_BATCH, build_union_graph, build_unit_graph, chains_per_reference_batch, flatten_formula
from .query_sat import QuerySAT, distribution_at_time, randomized_rounding_tf, t_power
from .variable_assignment import VariableAssignment
from .weights import init_weights, load_weights

use_baseline_sampling = True
test_rounds = 32
diffusion_steps = 32
test_unigen = False
self_supervised = False
ROWS_CAP = 900_000          # variable/clause rows per launch (~20 GB of activations at n=100)


def reverse_distribution_step_theoretic(x, x0, t, t_increment):
    """fp32 numpy restatement of reference ``:29-37`` (``t`` is a Python float, as there)."""
    x = np.asarray(x, dtype=np.float32)
    x0 = np.asarray(x0, dtype=np.float32)
    t1 = np.power(np.float32(t), np.float32(t_power))
    t2 = np.power(np.float32(max(0.0, t - t_increment)), np.float32(t_power))
    x_new = distribution_at_time(x0, t1)
    alpha_t = (np.float32(1) - t1) / (np.float32(1) - t2)
    x_unnormed = distribution_at_time(x, np.float32(1) - alpha_t) * x_new
    return (x_unnormed / (np.sum(x_unnormed, axis=-1, keepdims=True) + np.float32(1e-8))).astype(np.float32)


def _sigmoid(z):
    z = np.asarray(z, dtype=np.float32)
    return (np.float32(1) / (np.float32(1) + np.exp(-z))).astype(np.float32)


def predict(model, model_input, noisy_num, noise_scale, denoised_num=None, **noise):
    if denoised_num is not None:
        raise NotImplementedError("diffusion_step_self is unused by the sampler (self_supervised=False)")
    output = model.diffusion_step(model_input["adj_matrix"], model_input["clauses_graph"],
                                  model_input["variables_graph"], model_input.get("solutions"), noise_scale,
                                  noisy_num, **noise)
    return _sigmoid(output["prediction"]), output


def diffusion(N, model, dataset, step_data, verbose=True, prepare_image=True, *, uniforms=None, labels=None,
              normals=None):
    """Step-by-step reverse process through ``model.diffusion_step`` (one libdsat model call per step).

    ``step_data`` needs ``adjacency_matrix``, ``clauses_graph_adj``, ``variables_graph_adj``,
    ``normal_clauses`` (clause lists per graph) and ``variables_in_graph``.  ``dataset`` is unused
    (the reference only uses it to pick those keys).  Returns ``(mean cum_accuracy, predictions [N_vars],
    var_correct [N_vars])`` like the reference.  The fused whole-run kernel sequence used by
    :class:`DiffusionSampler` is ``Context.sample``; this function exists for API parity and tests.
    """
    model_input = {"adj_matrix": step_data["adjacency_matrix"], "clauses_graph": step_data["clauses_graph_adj"],
                   "variables_graph": step_data["variables_graph_adj"], "solutions": step_data.get("solutions")}
    graphs_n = [int(v) for v in step_data["variables_in_graph"]]
    n_vars = int(sum(graphs_n))
    x = np.zeros((n_vars, 2), dtype=np.float32) + np.float32(0.5)
    fixed_step = [-1] * n_vars
    fixed = [0.0] * n_vars
    cum_accuracy = np.zeros(len(graphs_n))
    predictions = None
    total_accuracy = np.zeros(len(graphs_n), dtype=bool)
    for t in range(N):
        noise_scale = 1 - t / N
        x_noisy = randomized_rounding_tf(x, noise=None if uniforms is None else uniforms[t])
        if use_baseline_sampling:
            x = x_noisy
        extra = {}
        if labels is not None:
            extra["labels"] = labels[t]
        if normals is not None:
            extra["normals"] = normals[t]
        predictions, _ = predict(model, model_input, x_noisy, noise_scale, **extra)
        x = reverse_distribution_step_theoretic(x, np.stack([1 - predictions, predictions], axis=1), noise_scale, 1 / N)
        xx = np.round(predictions)
        shift = 0
        for g, (cur_clauses, cur_n) in enumerate(zip(step_data["normal_clauses"], graphs_n)):
            asgn = VariableAssignment(n_vars=cur_n, clauses=[list(c) for c in cur_clauses])
            asgn.assign_all([bool(b) for b in xx[shift:shift + cur_n]])
            sat = asgn.satisfiable()
            total_accuracy[g] = sat
            if sat and fixed_step[shift] < 0:
                fixed[shift:shift + cur_n] = [float(v) for v in xx[shift:shift + cur_n]]
                fixed_step[shift:shift + cur_n] = [t] * cur_n
            shift += cur_n
        cum_accuracy = np.maximum(cum_accuracy, total_accuracy)
        if verbose:
            print("cum_accuracy:", np.mean(cum_accuracy), "noise_scale:", noise_scale)
    final = np.round(predictions)
    for i in range(n_vars):
        if fixed_step[i] >= 0:
            final[i] = fixed[i]
    var_correct = np.repeat(total_accuracy.astype(np.float32), graphs_n)
    return float(np.mean(cum_accuracy)), final, var_correct


def unpack_assignments(packed: np.ndarray, n_bits: int) -> list:
    """Packed little-endian 64-bit words [G, words] -> Python ints (x1 = bit 0), masked to n_bits."""
    from .dist import keys_to_ints
    return keys_to_ints(np.asarray(packed, dtype=np.uint64), n_bits)


def chains_for_rate(batch: int, n_vars: int, n_clauses: int, still_needed: int, sat_rate: float | None = None) -> int:
    """Chains of one formula's next launch: whole reference batches, as many as the samples still needed are expected to
    take at the SAT rate seen so far (first launch: 50 %, at least four batches), at most ``ROWS_CAP`` rows of the larger
    side."""
    rate = max(sat_rate if sat_rate is not None else 0.5, 0.02)
    batches = max(4, -(-int(still_needed / rate * 1.15 + 1) // batch))
    cap = max(1, ROWS_CAP // max(n_clauses, n_vars, 1) // batch)
    return batch * min(batches, cap)


def check_literals(n_vars: int, clauses):
    """VariableAssignment(clauses=...) sizes its vector by the largest literal (utils/VariableAssignment.py:34-36); for a
    header that declares more variables the reference fails in assign_all_from_bit_list on the first sample -- raised here
    before any GPU work."""
    if n_vars > max((abs(l) for c in clauses for l in c), default=0):
        raise IndexError("list assignment index out of range")


def consume_batches(is_sat: np.ndarray, batch: int, still_needed: int, total: int, sat_total: int,
                    min_sat_rate: float = 0.005):
    """The reference's stop rules (``satuniformity/DiffusionSampler.py:243-307``) applied to the SAT flags of one launch,
    vectorised.  Chains are consumed reference batch by reference batch, in order; before each batch the run stops if
    ``sat_total / total < min_sat_rate`` (``:261-263``); inside a batch it stops right after the sample that completes
    ``still_needed`` (``:305-307``).  Returns ``(chains_consumed, sat_counted, stopped_on_rate)``: the histogram of the
    launch is that of chains ``[0, chains_consumed)``."""
    is_sat = np.asarray(is_sat) != 0
    chains = is_sat.shape[0]
    csum = np.concatenate([[0], np.cumsum(is_sat, dtype=np.int64)])
    pos = 0
    while pos < chains and still_needed > 0:
        if total > 0 and sat_total / total < min_sat_rate:
            return pos, int(csum[pos]), True
        end = min(pos + batch, chains)
        sat_here = int(csum[end] - csum[pos])
        if sat_here >= still_needed:        # the sample that completes the request ends the run inside this batch
            cut = int(np.searchsorted(csum, csum[pos] + still_needed, side="left"))     # first index with that many SAT
            return cut, int(csum[cut]), False
        total += end - pos
        sat_total += sat_here
        still_needed -= sat_here
        pos = end
    return pos, int(csum[pos]), False


class DiffusionSampler:
    """Drop-in for the reference class.  ``precision="fp32"`` (default) runs the Dense layers fp32-accurately on the
    tensor cores; ``"bf16"`` is the faster, stated-separately path.

    Reproducibility: noise is a counter-based Philox stream keyed by ``(seed, global chain id)``.  Every ``samples()``
    call continues with fresh chains (the reference draws fresh TF randomness per call too); a new sampler with the same
    ``seed`` and ``chain_offset`` replays the same chains, and ``reset_chains()`` rewinds this one."""

    def __init__(self, model_path, dimacs_filename, *, device: int = 0, precision: str = "fp32",
                 chains_per_launch: int | None = None, seed: int = 0, chain_offset: int = 0,
                 max_nodes_per_batch: int = MAX_NODES_PER_BATCH, verbose: bool = False, context=None,
                 sampling: str = "inverse_cdf"):
        self.verbose = verbose
        print("model_path is ", model_path)
        weights = self._prepare_checkpoints(model_path)
        test_dimacs = DimacsFile(filename=dimacs_filename)
        test_dimacs.load()
        self.dimacs = test_dimacs
        self.n_vars = test_dimacs.number_of_vars()
        self.clauses = test_dimacs.clauses()
        self.model = QuerySAT(optimizer=None, test_rounds=test_rounds, weights=weights, device=device,
                              precision=precision, seed=seed, context=context,
                              feature_maps=weights.feature_maps, query_maps=weights.query_maps)
        self.ctx = self.model.ctx
        self.ctx.set_sampling(sampling)         # "gumbel": Gumbel-argmax rounding (same distribution, other samples)
        self.unit = build_unit_graph(self.n_vars, self.clauses)
        self.batch_chains = chains_per_reference_batch(self.n_vars, len(self.clauses), max_nodes_per_batch)
        self.chains_per_launch = chains_per_launch
        self.seed = int(seed)
        self.chain_offset = int(chain_offset)   # global id of this sampler's first chain (multi-GPU sharding)
        self.min_sat_rate = 0.005               # reference :261-263; 0 disables the abort (throughput runs)
        self._chains_consumed = 0               # chains launched by earlier samples() calls
        self.last_stats = {}

    def reset_chains(self, chain_offset: int | None = None):
        """Rewind the chain counter (and optionally move the block of global chain ids this sampler draws from)."""
        self._chains_consumed = 0
        if chain_offset is not None:
            self.chain_offset = int(chain_offset)

    def _prepare_checkpoints(self, model_path):
        """Reference ``:215-227``: restore the latest checkpoint, or print "Checkpoint not found!" and go on with
        (seeded) random weights.  Only a missing path counts as "not found": a file that exists but cannot be parsed
        raises, so a reader bug can never turn into silently random weights."""
        import os
        if model_path is None or not (os.path.exists(str(model_path)) or os.path.exists(str(model_path) + ".index")):
            print("Checkpoint not found!")
            return init_weights(seed=1234)
        try:
            weights = load_weights(model_path)
        except FileNotFoundError:              # a directory without a `checkpoint` file / ckpt-N.index
            print("Checkpoint not found!")
            return init_weights(seed=1234)
        print(f"Model restored from {model_path}!")
        return weights

    def _launch_chains(self, still_needed: int, chains_left: int | None = None, sat_rate: float | None = None) -> int:
        """Chains per launch: whole reference batches, bounded by the activation memory.  The reference runs one batch at a
        time until it has enough samples; a launch here holds as many batches as the samples still needed are expected to
        take at the SAT rate seen so far (first launch: 50 %, at least four batches -- small launches are latency-bound, so
        spare chains cost nothing), and batches are consumed in order with the reference's stop rules, so the histogram does
        not depend on the launch size."""
        b = self.batch_chains
        if self.chains_per_launch:
            n = max(b, (self.chains_per_launch // b) * b)
        else:
            n = chains_for_rate(b, self.n_vars, len(self.clauses), still_needed, sat_rate)
            if self.ctx.graph is self.unit and n <= self.ctx.chains <= 2 * n:
                n = self.ctx.chains                         # same shape as the previous launch: buffers and the captured step are kept
        if chains_left is not None:
            n = min(n, max(chains_left, 1))
            if chains_left - n < b:             # a remainder smaller than one reference batch rides along as a last, partial group
                n = max(chains_left, 1)
        return n

    def samples(self, n_samples, *, max_chains: int | None = None):
        """:param n_samples: how many correct samples to generate
        :param max_chains: (extension) stop after this many chains even if fewer samples were found
        :return: the dict solution-as-int => count"""
        from .dist import table_to_dict
        keys, counts = self.samples_table(n_samples, max_chains=max_chains)
        return table_to_dict(keys, counts, self.n_vars)

    def samples_table(self, n_samples, *, max_chains: int | None = None):
        """``samples()`` before the conversion to Python ints: ``(keys [K, words] uint64 ascending, counts [K] int64)``,
        the form ``dist.merge_histograms`` exchanges between GPUs."""
        from .dist import merge_tables
        check_literals(self.n_vars, self.clauses)
        tables = []
        total = sat_total = launched = 0
        still_needed = int(n_samples)
        words = -(-self.n_vars // 64)
        stop = False
        while still_needed > 0 and not stop and (max_chains is None or launched < max_chains):
            chains = self._launch_chains(still_needed, None if max_chains is None else max_chains - launched,
                                         sat_total / total if total else None)
            if self.ctx.graph is not self.unit or self.ctx.chains != chains:
                self.ctx.set_graph(self.unit, chains=chains, group_graphs=self.batch_chains)
                self.model._graph_key = None
            self.ctx.sample_enqueue(diffusion_steps, test_rounds, seed=self.seed,
                                    chain_offset=self.chain_offset + self._chains_consumed + launched)
            is_sat = self.ctx.sample_fetch_sat()
            used, sat_used, stop = consume_batches(is_sat, self.batch_chains, still_needed, total, sat_total,
                                                   self.min_sat_rate)
            if stop:
                print("too many unsat samples; stopping diffusion")
            if sat_used:
                keys, counts, n_sat = self.ctx.hist_reduce(used)        # sort / unique / count on the device
                assert n_sat == sat_used
                tables.append((keys, counts))
            total += used
            sat_total += sat_used
            still_needed -= sat_used
            launched += chains
        self._chains_consumed += launched
        keys, counts = merge_tables(tables, words)
        self.last_stats = {"total": total, "sat": sat_total, "chains_launched": launched, "distinct": int(len(counts))}
        print("success rate: ", sat_total / total if total else 0.0)
        return keys, counts


class _Formula:
    """One file of a MultiDiffusionSampler: its graph data, reference batch size and the progress of the current call."""

    def __init__(self, filename, max_nodes_per_batch):
        dimacs = DimacsFile(filename=filename)
        dimacs.load()
        self.n_vars = dimacs.number_of_vars()
        self.clauses = dimacs.clauses()
        self.flat = flatten_formula(self.n_vars, self.clauses)
        self.batch_chains = chains_per_reference_batch(self.n_vars, len(self.clauses), max_nodes_per_batch)
        self.words = -(-self.n_vars // 64)
        self.launched_before = 0            # chains launched by earlier samples() calls
        self.start(0)

    def start(self, n_samples):
        self.still_needed = int(n_samples)
        self.total = self.sat_total = self.launched = 0
        self.stopped = False
        self.tables = []

    @property
    def active(self) -> bool:
        return self.still_needed > 0 and not self.stopped

    @property
    def rows_per_chain(self) -> int:
        return self.n_vars + len(self.clauses)

    def next_chains(self) -> int:
        return chains_for_rate(self.batch_chains, self.n_vars, len(self.clauses), self.still_needed,
                               self.sat_total / self.total if self.total else None)


def plan_launch(formulas, rows_cap: int = ROWS_CAP):
    """``[(index, chains), ...]`` of the next launch: every active formula in file order with the chains its own
    ``DiffusionSampler`` would launch, while the variable + clause rows stay within ``rows_cap``.  The first active formula
    always goes; the first one that does not fit and every later one wait for the next launch."""
    plan, rows = [], 0
    for k, f in enumerate(formulas):
        if not f.active:
            continue
        c = f.next_chains()
        if plan and rows + c * f.rows_per_chain > rows_cap:
            break
        plan.append((k, c))
        rows += c * f.rows_per_chain
    return plan


def launch_layout(formulas, plan, chain_offset: int):
    """Graph layout of one launch, formula-major (all copies of the first planned formula, then the next ...):
    ``(graph_seg [len(plan)+1], group_seg, noise_base [graphs] uint64)``.  Early-exit groups are runs of the formula's
    reference batch size; copy j of formula k draws the noise of chain ``chain_offset + launched_k + j`` of its own sampler,
    i.e. Philox elements from ``(chain_offset + launched_k + j) * n_k`` on."""
    graph_seg, group_seg, bases = [0], [0], []
    for k, c in plan:
        f = formulas[k]
        g0 = graph_seg[-1]
        group_seg.extend(min(g0 + i, g0 + c) for i in range(f.batch_chains, c + f.batch_chains, f.batch_chains))
        first = chain_offset + f.launched_before + f.launched
        bases.append((np.arange(first, first + c, dtype=np.uint64)) * np.uint64(f.n_vars))
        graph_seg.append(g0 + c)
    noise_base = np.concatenate(bases) if bases else np.zeros(0, dtype=np.uint64)
    return np.asarray(graph_seg, dtype=np.int32), np.asarray(group_seg, dtype=np.int32), noise_base


class MultiDiffusionSampler:
    """``DiffusionSampler.samples`` for many DIMACS files at once: each launch holds reference batches of every formula that
    still needs samples (one disjoint-union graph, ``dsat_set_batches``), so a set of small formulas pays the fixed cost of
    a 32 x 32-round run once per launch instead of once per formula.

    For a fresh sampler ``samples(n)[k]`` equals ``DiffusionSampler(model_path, files[k], ...).samples(n_k)`` built with the
    same ``seed``, ``chain_offset``, ``max_nodes_per_batch``, ``precision`` and ``sampling``: copy j of a formula draws the
    noise of that sampler's chain j, forms the same early-exit groups, and the reference's stop rules are applied per
    formula.  (Bit-identical when the formulas of a launch share the shared-memory PairNorm's thread count; see DESIGN.md.)
    A formula that is done or has aborted gets no chains in later launches."""

    _prepare_checkpoints = DiffusionSampler._prepare_checkpoints

    def __init__(self, model_path, dimacs_filenames, *, device: int = 0, precision: str = "fp32", seed: int = 0,
                 chain_offset: int = 0, max_nodes_per_batch: int = MAX_NODES_PER_BATCH, sampling: str = "inverse_cdf",
                 verbose: bool = False, context=None):
        self.verbose = verbose
        print("model_path is ", model_path)
        weights = self._prepare_checkpoints(model_path)
        self.formulas = [_Formula(f, max_nodes_per_batch) for f in dimacs_filenames]
        self.model = QuerySAT(optimizer=None, test_rounds=test_rounds, weights=weights, device=device,
                              precision=precision, seed=seed, context=context,
                              feature_maps=weights.feature_maps, query_maps=weights.query_maps)
        self.ctx = self.model.ctx
        self.ctx.set_sampling(sampling)
        self.seed = int(seed)
        self.chain_offset = int(chain_offset)
        self.min_sat_rate = 0.005               # reference :261-263, per formula
        self.last_stats = []

    def reset_chains(self, chain_offset: int | None = None):
        """Rewind every formula's chain counter (and optionally move the block of global chain ids)."""
        for f in self.formulas:
            f.launched_before = 0
        if chain_offset is not None:
            self.chain_offset = int(chain_offset)

    def samples(self, n_samples):
        """:param n_samples: correct samples per formula (one int for all, or one per file)
        :return: one dict solution-as-int => count per file, in file order"""
        from .dist import table_to_dict
        return [table_to_dict(keys, counts, f.n_vars)
                for f, (keys, counts) in zip(self.formulas, self.samples_table(n_samples))]

    def samples_table(self, n_samples):
        """``samples()`` before the conversion to Python ints: one ``(keys [K, words_k] uint64 ascending, counts [K] int64)``
        per file, ``words_k = ceil(n_k / 64)``."""
        from .dist import merge_tables
        counts = [int(n_samples)] * len(self.formulas) if np.ndim(n_samples) == 0 else [int(n) for n in n_samples]
        if len(counts) != len(self.formulas):
            raise ValueError("n_samples: one count per file (%d), got %d" % (len(self.formulas), len(counts)))
        for f, n in zip(self.formulas, counts):
            check_literals(f.n_vars, f.clauses)
            f.start(n)
        while True:
            plan = plan_launch(self.formulas)
            if not plan:
                break
            self._launch(plan)
        out, self.last_stats = [], []
        for f in self.formulas:
            f.launched_before += f.launched
            keys, cnt = merge_tables(f.tables, f.words)
            f.tables = []
            out.append((keys, cnt))
            self.last_stats.append({"total": f.total, "sat": f.sat_total, "chains_launched": f.launched,
                                    "distinct": int(len(cnt)), "stopped_on_rate": f.stopped})
            if self.verbose:
                print("success rate: ", f.sat_total / f.total if f.total else 0.0)
        return out

    def _launch(self, plan):
        graph_seg, group_seg, noise_base = launch_layout(self.formulas, plan, self.chain_offset)
        unit = build_union_graph([self.formulas[k].flat for k, c in plan for _ in range(c)])
        self.ctx.set_graph(unit, chains=1)
        self.ctx.set_batches(group_seg, noise_base)
        self.model._graph_key = None
        self.ctx.sample_enqueue(diffusion_steps, test_rounds, seed=self.seed, chain_offset=0)
        is_sat = self.ctx.sample_fetch_sat()
        limits, consumed = [], []
        for i, (k, c) in enumerate(plan):
            f = self.formulas[k]
            used, sat_used, stop = consume_batches(is_sat[graph_seg[i]:graph_seg[i + 1]], f.batch_chains, f.still_needed,
                                                   f.total, f.sat_total, self.min_sat_rate)
            if stop:
                print("too many unsat samples; stopping diffusion")
            limits.append(used)
            consumed.append((f, used, sat_used, stop, c))
        if any(sat_used for _, _, sat_used, _, _ in consumed):
            tables, _ = self.ctx.hist_reduce_segments(graph_seg, limits)       # sort / unique / count per formula on the device
            for (f, _, sat_used, _, _), (keys, counts) in zip(consumed, tables):
                assert int(counts.sum()) == sat_used
                if sat_used:
                    f.tables.append((np.ascontiguousarray(keys[:, :f.words]), counts))
        for f, used, sat_used, stop, c in consumed:
            f.total += used
            f.sat_total += sat_used
            f.still_needed -= sat_used
            f.launched += c
            f.stopped = f.stopped or stop
