#!/usr/bin/env python
"""bench.py -- diffusion samples/sec on hard random 3-SAT n=100 (BASELINE.json configs[1]).

One "step" = one full reverse-diffusion run (32 denoising steps x 32 message-passing rounds, early exit
enabled, reference batch composition of 31 chains per early-exit group) of 4096 chains per GPU.
`value`  : whole-job samples/s with the formula and weights resident in HBM (CUDA events, max over ranks).
`e2e`    : the same through the C ABI with HOST buffers: dsat_set_graph (formula upload) + dsat_sample
           (results copied back) + the histogram merge, wall clock around the call.
`roofline`: the dominant kernel class (the MLP linear ops) from CUDA-event marks on the launching stream.
`message_pass`: the segment-sum SpMM kernels alone on BASELINE configs[4]'s graph (n=10000), HBM GB/s.
`cpu_baseline`: the CPU oracle port of the same path on the host cores (bounded sample).

`precisions`: both MLP arithmetics measured the same way; the top-level `value` / `dtype` are the fp32-accurate path's.
`parity_checked`: one early-exit group of the timed launch re-run on the CPU oracle after the timed region.

`--dump-outputs DIR`: the sampled assignments, SAT flags and latch steps of the last timed run as .npy files; the inputs
(formula, weights, Philox seeds) depend only on the arguments, so two builds can be compared output for output.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision fp32|bf16] [--dump-outputs DIR]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_VARS = 100
CHAINS_PER_GPU = 4096
DIFFUSION_STEPS = 32
ROUNDS = 32
SEED_FORMULA = 0


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks and throttle reasons sampled every 200 ms while the timed region runs."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._drain, daemon=True).start()
        except OSError:
            self.proc = None

    def _drain(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); smax.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


_RESTORE_STDOUT = lambda: None


def formula():
    from diffusionsat_b200 import synth
    return synth.random_3sat(N_VARS, seed=SEED_FORMULA)          # m = int(4.258 n + 58.26 n^(-2/3)) = 428


def mlp_flops_per_round(n_rows, m_rows, f=128, q=128):
    """Algorithmic (unpadded) FLOPs of the eleven linear launches of one round."""
    from diffusionsat_b200.weights import mlp_layer_dims
    dims = mlp_layer_dims(f, q)
    var_side = sum(i * o for name in ("variables_query", "lit_query", "update_gate", "variables_output") for i, o in dims[name])
    clause_side = sum(i * o for i, o in dims["clause_update"])
    return 2.0 * (var_side * n_rows + clause_side * m_rows)


def per_kernel_roofline(class_ms, n_rows, m_rows, precision, peak_tflops, peak_gbs, f=128, q=128):
    """Both roofs for every launch class of one round: executed tensor-core FLOPs (3 bf16 MMAs per product on the
    fp32-accurate path) against the measured bf16 rate, and ALGORITHMIC bytes (every operand row read once, every result row
    written once; weights stay in L2) against the measured copy rate.  Which Dense layers a class covers follows
    run_round (dsat_api.cu): fp32-accurate = whole query MLP (`query_out`), literal layers 1 / 2 / 3 (`v1_hidden`, `lit_2`,
    `lit_3`), clause layers 1 / 2, whole update (`update_3`) and output (`output_2`) MLPs; bf16 = one launch per MLP.
    Operands are hi/lo bf16 planes or fp32 (4 bytes per element) on the fp32-accurate path, bf16 on the bf16 path
    (logits fp32).  Returns {class: {ms, tensor_pipe_frac, hbm_frac, bound}} for the classes that ran."""
    from diffusionsat_b200.weights import mlp_layer_dims
    dims = mlp_layer_dims(f, q)
    pad = lambda x: (x + 15) // 16 * 16
    es = 4 if precision == "fp32" else 2
    v1, vrow = pad(f + 9), pad(f + 9) + 3 * q             # [variables | aux] and the whole variable row (update MLP input)
    macs = lambda layers: sum(i * o for i, o in layers)
    lq, cu = dims["lit_query"], dims["clause_update"]
    if precision == "fp32":
        launches = {      # class: (rows, MACs per row, input columns, output columns)
            "query_out": (n_rows, macs(dims["variables_query"]), v1, 3 * q),
            "v1_hidden": (n_rows, macs(lq[:1]), v1, pad(lq[0][1])),
            "lit_2": (n_rows, macs(lq[1:2]), pad(lq[1][0]), pad(lq[1][1])),
            "lit_3": (n_rows, macs(lq[2:]), pad(lq[2][0]), pad(lq[2][1])),
            "clause_1": (m_rows, macs(cu[:1]), pad(cu[0][0]), pad(cu[0][1])),
            "clause_2": (m_rows, macs(cu[1:]), pad(cu[1][0]), pad(cu[1][1])),
            "update_3": (n_rows, macs(dims["update_gate"]), vrow, f),
            "output_2": (n_rows, macs(dims["variables_output"]), f, 16),
        }
    else:
        launches = {
            "query_out": (n_rows, macs(dims["variables_query"]), v1, 3 * q),
            "lit_3": (n_rows, macs(lq), v1, pad(lq[2][1])),
            "clause_2": (m_rows, macs(cu), pad(cu[0][0]), pad(cu[1][1])),
            "update_3": (n_rows, macs(dims["update_gate"]), vrow, f),
            "output_2": (n_rows, macs(dims["variables_output"]), f, 16 * 4 // es),       # logits are fp32
        }
    mma = 3 if precision == "fp32" else 1
    out = {}
    for name, (rows, mac, cin, cout) in launches.items():
        ms = class_ms.get(name)
        if not ms:
            continue
        tf = mma * 2.0 * rows * mac / (ms / 1e3) / 1e12
        gbs = rows * (cin + cout) * es / (ms / 1e3) / 1e9
        out[name] = {"ms": ms, "tensor_pipe_frac": tf / peak_tflops, "hbm_frac": gbs / peak_gbs,
                     "bound": "tensor" if tf / peak_tflops >= gbs / peak_gbs else "hbm"}
    # PairNorm: read the MLP result, read the old state, write the new state (the variable side also writes the output
    # MLP's input)
    for name, rows, arrays in (("pairnorm_clause", m_rows, 3), ("pairnorm_var", n_rows, 4)):
        ms = class_ms.get(name)
        if ms:
            out[name] = {"ms": ms, "tensor_pipe_frac": 0.0, "hbm_frac": rows * f * es * arrays / (ms / 1e3) / 1e9 / peak_gbs,
                         "bound": "hbm"}
    return out


# ------------------------------------------------------------------------------------ reference arm
def cpu_oracle_rate(batch_chains, dsteps, rounds, threads, repeats=1, warmup=0):
    """samples/s of the CPU oracle port: one reference batch, `dsteps` of 32 denoising steps, scaled."""
    import torch
    from diffusionsat_b200 import weights
    from oracle import querysat_oracle as O
    torch.set_num_threads(threads)
    n, clauses = formula()
    graph = O.OracleGraph.copies(n, clauses, batch_chains)
    w = O.weights_to_torch(weights.init_weights(seed=1234))
    rng = np.random.default_rng(0)
    nt = graph.n_vars
    times = []
    for it in range(warmup + repeats):
        uniforms = torch.from_numpy(rng.random((dsteps, nt)).astype(np.float32))
        labels = torch.from_numpy(rng.integers(0, 2, (dsteps, nt)))
        normals = torch.from_numpy(rng.standard_normal((dsteps, rounds, nt, 4)).astype(np.float32))
        t0 = time.perf_counter()
        O.diffusion(dsteps, graph, w, uniforms, labels, normals, rounds)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    per_full_run = float(np.mean(times)) * (DIFFUSION_STEPS / dsteps)
    return batch_chains / per_full_run, float(np.mean(times))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from diffusionsat_b200.graph import chains_per_reference_batch
    n, clauses = formula()
    batch = chains_per_reference_batch(n, len(clauses))
    threads = os.cpu_count() or 1
    dsteps = 1
    rate, step_s = cpu_oracle_rate(batch, dsteps, ROUNDS, threads, repeats=args.steps, warmup=args.warmup)
    sample = ("%d chains (one reference batch, floor(20000/(2n+m))), %d of %d denoising steps x %d rounds per step, "
              "scaled x%d" % (batch, dsteps, DIFFUSION_STEPS, ROUNDS, DIFFUSION_STEPS // dsteps))
    line = {
        "impl": "reference", "metric": "diffusion samples/sec, 3-SAT n=100", "value": rate, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_s * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "hard random 3-SAT n=100 m=%d, 32 denoising steps x 32 rounds, random-init QuerySAT F=Q=128"
                               % len(clauses)},
        "cpu_baseline": {"value": rate, "unit": "samples/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "TensorFlow 2.4 / TFP 0.12 are not installable offline; this is the torch-CPU oracle port of the reference path",
    }
    _RESTORE_STDOUT()
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ our arm
def message_pass_roofline(ctx, torch, pk):
    """Segment-sum SpMM alone on BASELINE configs[4]'s graph (n=10000, m=43000): sweep over the feature
    width and storage type; the headline entry is F=128 fp32 (the model's width), worst direction."""
    from diffusionsat_b200 import graph, synth
    n, m = 10000, 43000
    nv, clauses = synth.random_3sat(n, m, seed=5)
    unit = graph.build_unit_graph(nv, clauses)
    ctx.set_graph(unit, chains=1, group_graphs=0)
    dev = torch.device("cuda", ctx.device)
    sweep = {}
    for feat, dtype_name, tdt, code in ((128, "f32", torch.float32, 0), (64, "f32", torch.float32, 0),
                                        (256, "f32", torch.float32, 0), (128, "bf16", torch.bfloat16, 1)):
        es = 4 if code == 0 else 2
        chains = max(8, int(3.0e9 / ((2 * n + m) * feat * es)))          # ~3 GB per launch, far beyond L2
        res = {}
        for name, direction, rin, rout in (("clause_from_literal", 0, 2 * n, m), ("literal_from_clause", 1, m, 2 * n)):
            x = torch.randn(chains, rin, feat, device=dev).to(tdt)
            y = torch.empty(chains, rout, feat, device=dev, dtype=tdt)
            torch.cuda.synchronize()
            for _ in range(3):
                ctx.spmm(direction, x.data_ptr(), y.data_ptr(), feat, code, chains)
            ctx.synchronize()
            reps = 5
            ctx.timer_begin()
            for _ in range(reps):
                ctx.spmm(direction, x.data_ptr(), y.data_ptr(), feat, code, chains)
            ms = ctx.timer_end() / reps
            nbytes = (rin + rout) * chains * feat * es + (unit.nnz + rout + 1) * 4
            res[name] = {"gbs": nbytes / ms / 1e6, "ms": ms, "bytes": nbytes, "chains": chains}
            del x, y
        sweep["F%d_%s" % (feat, dtype_name)] = res
    head = sweep["F128_f32"]
    worst = min(head.values(), key=lambda d: d["gbs"])
    return {"bound": "hbm", "achieved": worst["gbs"], "peak": pk["hbm_gbs"], "unit": "GB/s",
            "frac": worst["gbs"] / pk["hbm_gbs"], "traffic": None, "peak_source": pk["source"],
            "workload": "segment-sum SpMM, shared adjacency, 3-SAT n=10000 m=43000, %d chains, F=128 fp32; bytes = "
                        "(R_in+R_out)*C*F*s + (nnz+R_out+1)*4" % worst["chains"],
            "avg_launch_ms": worst["ms"], "bytes_per_launch": worst["bytes"],
            "sweep_gbs": {k: {d: round(v[d]["gbs"], 1) for d in v} for k, v in sweep.items()}}


PRECISION_DTYPE = {"fp32": "f32", "bf16": "bf16"}
PRECISION_KERNEL = {
    "fp32": "x3_mlp_kernel (tcgen05, fp32-accurate: every product = 3 bf16 MMAs on hi/lo planes into one fp32 TMEM accumulator; "
            "7 persistent launches per round)",
    "bf16": "fused_mlp_kernel / fused_mlp_split_kernel (tcgen05 bf16, one persistent launch per MLP, 5 per round)",
}


def ncu_traffic(precision):
    """DRAM bytes per launch of the dominant kernel class from the committed `ncu --set full` capture: NOT measured in this
    run (a run under ncu is never a bench value); `traffic_source` in the line says so."""
    for name in ("r2_traffic.json", "r1_traffic.json"):
        path = os.path.join(ROOT, "profiles", name)
        if os.path.exists(path):
            with open(path) as fh:
                blob = json.load(fh)
            key = {"fp32": "x3_mlp_kernel", "bf16": "fused_mlp_kernel"}[precision]
            if key in blob:
                return blob[key]["dram_bytes_per_launch"], "profiles/" + name
    return None, None


def parity_check(ctx, precision, unit, n, clauses, batch, chains, wts, chain_offset):
    """One early-exit group from the middle of the timed launch, re-run on the CPU oracle with the same Philox noise
    (host restatement, diffusionsat_b200/philox.py), after the timed region: 32 free-running rounds of one model call."""
    import torch
    from diffusionsat_b200 import philox
    from oracle import querysat_oracle as O
    seed, noise_scale = 4242, 0.75
    rng = np.random.default_rng(17)
    bits = rng.integers(0, 2, chains * n).astype(np.float32)
    noisy = np.stack([bits, 1 - bits], axis=1)
    pred, steps, _ = ctx.model_call(noise_scale, noisy, rounds=ROUNDS, seed=seed, chain_offset=chain_offset)
    gmap = ctx.debug_groups()["graph_map"]
    g = (chains // batch) // 2
    c0 = g * batch
    rows = slice(c0 * n, (c0 + batch) * n)
    elems = np.arange((chain_offset + c0) * n, (chain_offset + c0 + batch) * n, dtype=np.uint64)
    labels = philox.labels(seed, elems, 0)
    normals = np.stack([philox.normals(seed, elems, 0, r) for r in range(ROUNDS)])
    graph = O.OracleGraph.copies(n, clauses, batch)
    trace = []
    out = O.model_loop(graph, O.weights_to_torch(wts), noise_scale, torch.from_numpy(noisy[rows]),
                       torch.from_numpy(labels.astype(np.int64)), torch.from_numpy(normals), ROUNDS, trace=trace)
    want = out[0].numpy().astype(np.float64)
    same = np.repeat(gmap[c0:c0 + batch] == trace[-1]["best_graph_map"].numpy(), n)
    got = pred[rows].astype(np.float64)
    rms = float(np.sqrt(np.mean(want ** 2)))
    err = np.abs(got - want)[same]
    tol = 1e-3 if precision == "fp32" else 1e-1
    inside = err <= tol * np.abs(want[same]) + tol * rms
    return {"group": int(g), "chains": int(batch), "of_chains": int(chains), "rounds": ROUNDS, "oracle": "fp32 torch-CPU port",
            "logit_map_agree": float(same.mean()), "max_abs_err_over_rms": float(err.max() / rms) if err.size else None,
            "tolerance": "%g |z| + %g rms(z) per element" % (tol, tol), "elements_inside": float(inside.mean()) if err.size else None,
            "decisions_equal": float(((got > 0) == (want > 0))[same].mean()) if err.size else None,
            "steps_taken_equal": bool(steps[g] == out[1]),
            # fp32: every element inside; bf16 (stated separately): 99 % of the elements inside and 97 % of the decisions equal
            "ok": bool(err.size and steps[g] == out[1] and
                       (inside.all() if precision == "fp32" else
                        inside.mean() >= 0.99 and ((got > 0) == (want > 0))[same].mean() >= 0.97))}


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, n_vars, chain_offset, packed, is_sat, latch_step, sat_any_step):
    """Write what dsat_sample_fetch hands a caller after a run as DIR/<name>.npy: the sampled assignment of every chain
    (0/1 per variable, x1 first), its SAT flag, the denoising step at which it was first satisfied (-1 = never) and the
    any-step SAT flag, all float32, plus the global index of each chain (float64).  Above DUMP_BYTES in all, a fixed
    seeded sample of the chains is written instead, so that two builds can still be compared chain for chain."""
    chains = len(packed)
    rows = np.arange(chains)
    per_chain = 4 * (n_vars + 3) + 8
    if chains * per_chain > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(chains, DUMP_BYTES // per_chain, replace=False))
    bits = np.unpackbits(packed[rows].astype("<u8").view(np.uint8).reshape(len(rows), -1), axis=1, bitorder="little")
    arrays = {"assignment": bits[:, :n_vars].astype(np.float32), "is_sat": is_sat[rows].astype(np.float32),
              "latch_step": latch_step[rows].astype(np.float32), "sat_any_step": sat_any_step[rows].astype(np.float32),
              "chain": (chain_offset + rows).astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)


def measure_precision(ctx, precision, args, world, rank, local_rank, unit, batch, chains, chain_offset, barrier, dist, torch, pk):
    """`value` of one precision: W warm-up + K timed whole reverse-diffusion runs, everything resident, CUDA events on the
    launching stream, max over ranks; then (rank 0) the per-class device time of four rounds for the roofline.  With
    --dump-outputs, rank 0 writes the headline precision's results of the last timed run."""
    from diffusionsat_b200 import _lib
    ctx.set_precision(_lib.PRECISIONS[precision])
    ctx.set_graph(unit, chains=chains, group_graphs=batch)
    steps = args.steps if precision == args.precision else max(1, min(args.steps, 3))
    warmup = args.warmup if precision == args.precision else 3
    for i in range(warmup):
        ctx.sample_enqueue(DIFFUSION_STEPS, ROUNDS, seed=1000 + i, chain_offset=chain_offset)
    ctx.synchronize()
    barrier()
    clocks = ClockSampler(local_rank)
    clocks.start()
    launches0 = ctx.launch_count()
    ctx.timer_begin()
    for i in range(steps):
        ctx.sample_enqueue(DIFFUSION_STEPS, ROUNDS, seed=1000 + warmup + i, chain_offset=chain_offset)
    ms = ctx.timer_end()
    launches = ctx.launch_count() - launches0
    barrier()
    clock_info = clocks.stop()
    if args.dump_outputs and precision == args.precision and rank == 0:
        dump_outputs(args.dump_outputs, unit.n_vars, chain_offset, *ctx.sample_fetch())
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    res = {"value": world * chains * steps / (ms_max / 1e3), "unit": "samples/s", "dtype": PRECISION_DTYPE[precision],
           "steps": steps, "warmup": warmup, "ms_per_step": ms_max / steps, "gpu_launches": int(launches), "clocks": clock_info}
    if rank != 0:
        return res
    prof = ctx.profile_rounds(rounds=4, seed=7)
    total_ms = sum(v[0] for v in prof.values())
    gemm_names = list(_lib.Context.PROFILE_CLASSES[:11])
    gemm_ms = sum(prof[k][0] for k in gemm_names)
    gemm_launches = sum(prof[k][1] for k in gemm_names)
    flops = mlp_flops_per_round(ctx.n_rows, ctx.n_clause_rows) * 4
    achieved_tf = flops / (gemm_ms / 1e3) / 1e12
    peak_tf = pk["bf16_tflops_sustained"]
    traffic, traffic_src = ncu_traffic(precision)
    mma_per_product = 3 if precision == "fp32" else 1
    res["roofline"] = {
        "bound": "tensor", "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf,
        "traffic": traffic, "traffic_source": traffic_src, "peak_source": pk["source"] + " bf16 sustained",
        "kernel": PRECISION_KERNEL[precision], "avg_launch_ms": gemm_ms / max(gemm_launches, 1),
        "share_of_round": gemm_ms / total_ms, "flops_per_launch": flops / max(gemm_launches, 1),
        "bf16_mma_per_algorithmic_product": mma_per_product,
        "tensor_pipe_frac": mma_per_product * achieved_tf / peak_tf,
        "class_ms_per_round": {k: v[0] / 4 for k, v in prof.items() if v[1]}}
    try:        # reporting only: never let it cost the line
        res["roofline"]["per_kernel"] = per_kernel_roofline(res["roofline"]["class_ms_per_round"], ctx.n_rows, ctx.n_clause_rows,
                                                            precision, peak_tf, pk["hbm_gbs"])
    except Exception as exc:
        res["roofline"]["per_kernel_error"] = repr(exc)
    es = 4 if precision == "fp32" else 2
    q = 128
    nnz = unit.nnz
    cg_bytes = ctx.n_rows * 4 * q * es + ctx.n_clause_rows * 2 * q * es + (nnz + unit.n_clauses + 1) * 4
    lg_bytes = ctx.n_clause_rows * 2 * q * es + ctx.n_rows * q * es + ctx.n_rows * 3 * q * es + (nnz + 2 * unit.n_vars + 1) * 4
    res["message_pass_in_model"] = {}
    for name, nbytes in (("clause_gather", cg_bytes), ("literal_gather", lg_bytes)):
        if prof[name][1] == 0:
            continue
        ms_launch = prof[name][0] / prof[name][1]
        res["message_pass_in_model"][name] = {"gbs": nbytes / ms_launch / 1e6, "frac": nbytes / ms_launch / 1e6 / pk["hbm_gbs"],
                                              "ms": ms_launch, "bytes": nbytes}
    return res


def run_ours(args):
    import tempfile
    import torch
    import torch.distributed as dist
    from diffusionsat_b200 import _lib, build, graph, synth, weights
    from diffusionsat_b200 import dist as D
    from diffusionsat_b200.graph import chains_per_reference_batch
    from diffusionsat_b200.sampler import DiffusionSampler

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    build.build()
    pk = peaks()
    ctx = _lib.Context(local_rank)
    wts = weights.init_weights(seed=1234)
    ctx.set_model(wts)
    n, clauses = formula()
    unit = graph.build_unit_graph(n, clauses)
    batch = chains_per_reference_batch(n, len(clauses))
    chains = args.chains
    chain_offset = rank * chains

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # headline precision first (fp32-accurate tensor-core path = the reference's arithmetic), then the other one
    order = [args.precision] + [p for p in ("fp32", "bf16") if p != args.precision]
    if args.single_precision:
        order = order[:1]
    per_precision = {}
    for precision in order:
        per_precision[precision] = measure_precision(ctx, precision, args, world, rank, local_rank, unit, batch, chains,
                                                     chain_offset, barrier, dist, torch, pk)
    head = per_precision[args.precision]

    # end to end through the PUBLIC API: DiffusionSampler(model_path, dimacs).samples(...) with the formula file and the
    # weights file on the host; every step re-uploads the formula, runs `chains` chains (reference batches of 31, stop rule
    # on the SAT rate disabled: random-init weights solve nothing), reduces the histogram on the device and copies the SAT
    # flags and the histogram table back; the ranks' tables are merged over NCCL (all-gather + reduce)
    tmp = tempfile.mkdtemp(prefix="dsat_bench_")
    cnf_path, npz_path = os.path.join(tmp, "formula.cnf"), os.path.join(tmp, "weights.npz")
    with open(cnf_path, "w") as fh:
        fh.write(synth.dimacs_text(n, clauses))
    weights.save_weights(npz_path, wts)
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        sampler = DiffusionSampler(npz_path, cnf_path, context=ctx, precision=args.precision, seed=2000,
                                   chains_per_launch=chains, chain_offset=chain_offset)
    sampler.min_sat_rate = 0.0
    if world > 1:       # untimed warm-up of the merge's collectives (NCCL sets up all-gather / reduce channels on first use)
        D.merge_histograms(np.zeros((0, -(-n // 64)), dtype=np.uint64), np.zeros(0, dtype=np.int64), n)
    barrier()
    e2e_steps = args.steps
    hist_sizes = []
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        ctx.graph = None                                            # forces dsat_set_graph: the formula travels host -> device
        with contextlib.redirect_stdout(io.StringIO()):
            if world == 1:
                hist = sampler.samples(10 ** 9, max_chains=chains)
            else:
                keys, counts = sampler.samples_table(10 ** 9, max_chains=chains)
                hist = D.merge_histograms(keys, counts, n) or {}
        hist_sizes.append(sampler.last_stats["distinct"])
    barrier()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * chains * e2e_steps / float(t.item())
    h2d = int(sum(a.nbytes for a in (unit.cl_rowptr, unit.cl_lit, unit.lit_rowptr, unit.lit_clause, unit.var_seg,
                                     unit.clause_seg)))
    d2h = int(chains + 8 + max(hist_sizes) * (8 * (-(-n // 64)) + 8))          # SAT flags + totals + histogram table
    sat_rate = sampler.last_stats["sat"] / max(sampler.last_stats["total"], 1)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    parity = {}
    if not args.skip_parity:
        for precision in order:
            ctx.set_precision(_lib.PRECISIONS[precision])
            ctx.set_graph(unit, chains=chains, group_graphs=batch)
            parity[precision] = parity_check(ctx, precision, unit, n, clauses, batch, chains, wts, chain_offset)
    ctx.set_precision(_lib.PRECISIONS[args.precision])
    message_pass = None if args.skip_message_pass else message_pass_roofline(ctx, torch, pk)

    # TRAINED fixture weights (tests/golden/trained_small.npz: a short CPU training on n <= 30) on a satisfiable formula of
    # BASELINE configs[0]'s shape (n=30, m=133): formulas do get satisfied here, so the first-SAT latch and the per-group
    # early exit take effect.  (At n=100, ratio 4.28, these weights solve nothing: they never saw that size.)
    trained = None
    cfg1 = None
    fixture = os.path.join(ROOT, "tests", "golden", "trained_small.npz")
    if os.path.exists(fixture) and not args.skip_trained:
        tn, tclauses, _ = synth.planted_3sat(30, 133, seed=0)
        tunit = graph.build_unit_graph(tn, tclauses)
        tbatch = chains_per_reference_batch(tn, len(tclauses))
        tchains = tbatch * 128
        ctx.set_model(weights.load_weights(fixture))
        trained = {"workload": "planted 3-SAT n=30 m=133, %d chains in early-exit groups of %d, 32 x 32" % (tchains, tbatch),
                   "weights": "tests/golden/trained_small.npz"}
        for precision in order:
            ctx.set_precision(_lib.PRECISIONS[precision])
            ctx.set_graph(tunit, chains=tchains, group_graphs=tbatch)
            ctx.sample_enqueue(DIFFUSION_STEPS, ROUNDS, seed=3000, chain_offset=0)
            ctx.synchronize()
            ctx.timer_begin()
            ctx.sample_enqueue(DIFFUSION_STEPS, ROUNDS, seed=3001, chain_offset=0)
            t_ms = ctx.timer_end()
            t_packed, t_sat, t_latch, _ = ctx.sample_fetch()
            trained[precision] = {"samples_per_s": tchains / (t_ms / 1e3), "sat_rate": float(t_sat.mean()),
                                  "distinct_models": int(len(np.unique(t_packed[t_sat.astype(bool)], axis=0))),
                                  "mean_latch_step": float(t_latch[t_latch >= 0].mean()) if (t_latch >= 0).any() else None}
        # BASELINE configs[0]: DiffusionSampler.samples(256) at n=30 through the public API (small-launch regime)
        cnf1 = os.path.join(tmp, "cfg1.cnf")
        with open(cnf1, "w") as fh:
            fh.write(synth.dimacs_text(tn, tclauses))
        cfg1 = {"workload": "planted 3-SAT n=30 m=133, DiffusionSampler.samples(256), trained fixture weights"}
        for precision in order:
            with contextlib.redirect_stdout(io.StringIO()):
                s1 = DiffusionSampler(fixture, cnf1, context=ctx, precision=precision, seed=5)
                s1.samples(256)                                     # warm-up (buffers, plans)
                t1 = time.perf_counter()
                h1 = s1.samples(256)
                dt = time.perf_counter() - t1
            cfg1[precision] = {"seconds": dt, "samples": int(sum(h1.values())), "chains_launched": s1.last_stats["chains_launched"]}
        ctx.set_model(wts)
        ctx.set_precision(_lib.PRECISIONS[args.precision])
        ctx.set_graph(unit, chains=chains, group_graphs=batch)

    cpu = None
    if world == 1 and not args.skip_cpu:
        threads = os.cpu_count() or 1
        cpu_dsteps, cpu_repeats = 4, 5          # about 10 s of CPU work on the box's 16 cores (0.4 s per denoising step)
        rate, secs = cpu_oracle_rate(batch, cpu_dsteps, ROUNDS, threads, repeats=cpu_repeats, warmup=1)
        cpu = {"value": rate, "unit": "samples/s", "cores": threads, "kind": "port",
               "sample": "%d chains (one reference batch), %d of 32 denoising steps x 32 rounds, mean of %d runs after 1 warm-up, "
                         "scaled x%d; %.2f s per denoising step"
                         % (batch, cpu_dsteps, cpu_repeats, DIFFUSION_STEPS // cpu_dsteps, secs / cpu_dsteps)}

    working_set_gb = (ctx.n_rows * 3500 + ctx.n_clause_rows * 850) * (4 if args.precision == "fp32" else 2) / 1e9
    line = {
        "metric": "diffusion samples/sec, 3-SAT n=100", "value": head["value"], "unit": "samples/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": head["dtype"], "data": "synthetic",
        "config": {"workload": "hard random 3-SAT n=100 m=%d (ratio 4.3), %d chains per GPU, 32 denoising steps x 32 rounds, "
                               "random-init QuerySAT F=Q=128, early-exit groups of %d chains" % (len(clauses), chains, batch),
                   "chains_per_gpu": chains, "parallelism": "chains sharded, dp%d" % world,
                   "l2": "activations touched per round ~%.1f GB >> 126 MB L2: inputs larger than L2, no flush needed"
                         % working_set_gb,
                   "precision": args.precision + (" (fp32-accurate Dense layers on tcgen05: 3 split-bf16 MMAs per product; "
                                                  "everything else fp32)" if args.precision == "fp32" else "")},
        "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                "api": "DiffusionSampler(weights.npz, formula.cnf).samples(n, max_chains=%d) + dist.merge_histograms" % chains},
        "gpu_launches": head["gpu_launches"], "clocks": head["clocks"], "roofline": head.get("roofline"),
        "message_pass": message_pass, "message_pass_in_model": head.get("message_pass_in_model"),
        "precisions": {p: {k: v for k, v in r.items()} for p, r in per_precision.items()},
        "parity_checked": parity, "cpu_baseline": cpu, "sat_rate": sat_rate, "trained_weights": trained, "cfg1": cfg1,
    }
    _RESTORE_STDOUT()
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_uf250(args):
    """BASELINE configs[2]: SATLIB-style uf250 shape (n=250, m=1065), `--total-chains` (65536) chains in total sharded over the
    ranks (STRONG scaling), every rank reduces its launches' histograms on the device, one NCCL all-gather + reduce at the end.
    One step = the whole job; wall clock around the public entry (dist.sample_chains_sharded), max over ranks."""
    import torch
    import torch.distributed as dist
    from diffusionsat_b200 import _lib, build, graph, synth, weights
    from diffusionsat_b200 import dist as D
    from diffusionsat_b200.graph import chains_per_reference_batch
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    build.build()
    n, m = 250, 1065
    _, clauses = synth.random_3sat(n, m, seed=250)
    unit = graph.build_unit_graph(n, clauses)
    batch = chains_per_reference_batch(n, m)          # 12
    wts = weights.init_weights(seed=1234)
    ctx = _lib.Context(local_rank)
    ctx.set_model(wts)
    ctx.set_precision(_lib.PRECISIONS[args.precision])
    total = args.total_chains
    per_launch = args.chains_per_launch or 8400

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # warm-up: one launch of the launch size (buffers, plans, the captured step)
    ctx.set_graph(unit, chains=min(per_launch, D.shard_chains(total, world, rank, batch)[1]) or batch, group_graphs=batch)
    ctx.sample_enqueue(2, ROUNDS, seed=1, chain_offset=0)
    ctx.synchronize()
    barrier()
    clocks = ClockSampler(local_rank)
    clocks.start()
    times = []
    stats = None
    for i in range(args.steps):
        barrier()
        t0 = time.perf_counter()
        merged, stats = D.sample_chains_sharded(lambda r: ctx, unit, total, batch, n, DIFFUSION_STEPS, ROUNDS, seed=100 + i,
                                                chains_per_launch=per_launch, return_stats=True)
        barrier()
        times.append(time.perf_counter() - t0)
    clock_info = clocks.stop()
    t = torch.tensor([sum(times)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    secs = float(t.item()) / args.steps
    if rank == 0:
        line = {"metric": "diffusion samples/sec, uf250-shaped 3-SAT n=250 m=1065, %d chains in total" % total,
                "value": total / secs, "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": 1,
                "ms_per_step": secs * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": PRECISION_DTYPE[args.precision], "data": "synthetic",
                "config": {"workload": "BASELINE configs[2]: uf250 shape, %d chains sharded over %d GPUs in launches of <= %d, "
                                       "32 x 32, random-init QuerySAT, early-exit groups of %d, device histogram + NCCL merge"
                                       % (total, world, per_launch, batch), "precision": args.precision},
                "e2e": {"value": total / secs, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                        "api": "dist.sample_chains_sharded (host formula in, merged {int: count} out)"},
                "rank0": stats, "clocks": clock_info, "histogram_size": len(merged)}
        _RESTORE_STDOUT()
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_mixed(args):
    """BASELINE configs[3]: training-shape forward of mixed k-SAT formulas packed into reference batches (<= 20000 nodes), the
    batches dealt to the ranks, logits gathered on rank 0 (dist.forward_formulas_sharded).  Metric: formulas per second."""
    import torch
    import torch.distributed as dist
    from diffusionsat_b200 import _lib, build, synth, weights
    from diffusionsat_b200 import dist as D
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    build.build()
    rng = np.random.default_rng(0)
    formulas = []
    for i in range(args.formulas):          # n ~ U[3,100], k = {1 w.p. .3 | 2} + Geom(.4) (data/k_sat.py:45-46), ratio ~ 4.3
        nv = int(rng.integers(3, 101))
        formulas.append(synth.random_ksat_mixed(nv, max(1, int(4.3 * nv)), seed=1000 + i))
    # what a loader keeps per formula: its clauses laid end to end, once (the reference trains from pre-tensorised TFRecords,
    # data/dimac.py:129-211); batches are then cut, joined and indexed (dsat_graph_build) per step inside the timed region
    from diffusionsat_b200 import graph as G
    formulas = [G.flatten_formula(*f) for f in formulas]
    ctx = _lib.Context(local_rank)
    ctx.set_model(weights.init_weights(seed=1234))
    ctx.set_precision(_lib.PRECISIONS[args.precision])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    D.forward_formulas_sharded(lambda r: ctx, formulas[:200], 0.5, rounds=ROUNDS, seed=0)       # warm-up
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        out = D.forward_formulas_sharded(lambda r: ctx, formulas, 0.5, rounds=ROUNDS, seed=1 + i)
    barrier()
    t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    secs = float(t.item()) / args.steps
    if rank == 0:
        batches = D.pack_batches(formulas)
        nodes = sum(2 * nv + len(cl) for nv, cl in formulas)
        line = {"metric": "training-shape forward, mixed k-SAT formulas/sec", "value": len(formulas) / secs, "unit": "formulas/s",
                "n_gpus": world, "steps": args.steps, "warmup": 1, "ms_per_step": secs * 1e3, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": PRECISION_DTYPE[args.precision], "data": "synthetic",
                "config": {"workload": "BASELINE configs[3]: %d mixed k-SAT formulas (n ~ U[3,100]) = %d nodes in %d reference batches "
                                       "of <= 20000 nodes, one model call (32 rounds) per batch, batches dealt to %d GPUs; "
                                       "formulas pre-flattened once, union graph of every batch built inside the timed region "
                                       "(native dsat_graph_build, on a helper thread under the previous batch's model call)"
                                       % (len(formulas), nodes, len(batches), world), "precision": args.precision},
                "nodes_per_s": nodes / secs, "batches": len(batches)}
        _RESTORE_STDOUT()
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("DSAT_PRECISION", "fp32"), choices=["fp32", "bf16"],
                    help="headline precision: fp32 = fp32-accurate Dense layers on the tensor cores (the reference's arithmetic), "
                         "bf16 = plain bf16 path; the other one is measured too and reported under `precisions`")
    ap.add_argument("--single-precision", action="store_true", help="measure only --precision")
    ap.add_argument("--skip-parity", action="store_true")
    ap.add_argument("--chains", type=int, default=CHAINS_PER_GPU)
    ap.add_argument("--config", default="n100", choices=["n100", "uf250", "mixed"],
                    help="n100 = BASELINE configs[1] (the bench contract); uf250 = configs[2] strong scaling; mixed = configs[3]")
    ap.add_argument("--total-chains", type=int, default=65536, help="uf250: chains in total over all GPUs")
    ap.add_argument("--chains-per-launch", type=int, default=0, help="uf250: cap on the chains per launch and GPU (default 8400)")
    ap.add_argument("--formulas", type=int, default=4000, help="mixed: number of formulas")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-message-pass", action="store_true")
    ap.add_argument("--skip-trained", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="n100: write the results of the last timed run (headline precision) as DIR/<name>.npy; under "
                         "several GPUs only rank 0's chains (chain.npy holds their global indices)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (args.impl != "ours" or args.config != "n100"):
        ap.error("--dump-outputs writes the outputs of the n100 config of --impl ours")
    # Only the JSON line may reach stdout: libraries (NCCL's version banner under torchrun, for one) write there too, so
    # file descriptor 1 points at stderr while the benchmark runs and is restored for the final print.
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    global _RESTORE_STDOUT
    def _RESTORE_STDOUT():
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
    if args.impl == "reference":
        run_reference(args)
    elif args.config == "uf250":
        run_uf250(args)
    elif args.config == "mixed":
        run_mixed(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
