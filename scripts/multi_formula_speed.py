"""Wall time of a set of formulas: the per-file DiffusionSampler loop against one MultiDiffusionSampler, same process.

32 planted 3-SAT formulas, n = 20..60, trained fixture weights, samples(64) each (or the count given).  Both paths are
warmed once, then timed alternately three times; every timed call starts from rewound chain counters, so both compute the
same histograms, which are checked.  Prints the card name and power limit with the numbers.
python scripts/multi_formula_speed.py [precision] [n_samples]"""
import contextlib
import io
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from diffusionsat_b200 import _lib, synth  # noqa: E402
from diffusionsat_b200.sampler import DiffusionSampler, MultiDiffusionSampler  # noqa: E402

prec = sys.argv[1] if len(sys.argv) > 1 else "fp32"
n_samples = int(sys.argv[2]) if len(sys.argv) > 2 else 64
fixture = os.path.join(ROOT, "tests", "golden", "trained_small.npz")
tmp = tempfile.mkdtemp()
files = []
for i, n in enumerate([20 + (40 * i) // 31 for i in range(32)]):
    n_vars, clauses, _ = synth.planted_3sat(n, seed=100 + i)
    path = os.path.join(tmp, "f%02d_n%d.cnf" % (i, n))
    with open(path, "w") as fh:
        fh.write(synth.dimacs_text(n_vars, clauses))
    files.append(path)

try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
except Exception as exc:            # the numbers below still stand; say that the card could not be read
    card = "unknown (%s)" % type(exc).__name__

ctx = _lib.Context(0)
with contextlib.redirect_stdout(io.StringIO()):
    solos = [DiffusionSampler(fixture, f, context=ctx, precision=prec, seed=7) for f in files]
    multi = MultiDiffusionSampler(fixture, files, context=ctx, precision=prec, seed=7)


def run_solo():
    out = []
    for s in solos:
        s.reset_chains()
        out.append(s.samples(n_samples))
    return out


def run_multi():
    multi.reset_chains()
    return multi.samples(n_samples)


def timed(fn):
    with contextlib.redirect_stdout(io.StringIO()):
        ctx.synchronize()
        t0 = time.perf_counter()
        out = fn()
        ctx.synchronize()
        return time.perf_counter() - t0, out


_, want = timed(run_solo)               # warm-up (module load, captured steps, allocations) of both paths
_, got = timed(run_multi)
t_solo, t_multi = [], []
for _ in range(3):
    t, a = timed(run_solo)
    t_solo.append(t)
    t, b = timed(run_multi)
    t_multi.append(t)
    assert a == want and b == got
equal = sum(x == y for x, y in zip(want, got))
print("card: %s" % card)
print("%s, %d formulas (n = 20..60), samples(%d) each" % (prec, len(files), n_samples))
print("per-file DiffusionSampler loop: %s s (median %.3f)" % (["%.3f" % t for t in t_solo], statistics.median(t_solo)))
print("MultiDiffusionSampler:          %s s (median %.3f)" % (["%.3f" % t for t in t_multi], statistics.median(t_multi)))
print("speed-up (median): %.2fx" % (statistics.median(t_solo) / statistics.median(t_multi)))
print("histograms equal to the per-file samplers: %d of %d formulas (formulas of other shared-memory PairNorm classes than "
      "the largest in a launch may differ in the last bits; DESIGN.md); chains launched: per-file %d, multi %d" % (
    equal, len(files), sum(s.last_stats["chains_launched"] for s in solos),
    sum(st["chains_launched"] for st in multi.last_stats)))
