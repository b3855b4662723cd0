"""Device time of exact model enumeration (dsat_enumerate_models: brute force over all 2^n assignments, 2^36 per launch).

Planted 3-SAT at n = 30, 36, 40, 44 (the bench's trained_weights formula is the first) and one formula with many models,
random 3-SAT n = 40 with 80 clauses.  Each formula: one warm-up call, then the count-only call and the full enumeration
as Context.enumerate_models runs it (count pass, scan, emit pass, copy to the host; above 65 536 models a second call with
the exact capacity) timed with CUDA events on the context's stream, three times each (median).  Prints the card name and
power limit with the numbers.
python scripts/model_enumeration_speed.py"""
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

from diffusionsat_b200 import _lib, synth  # noqa: E402

FORMULAS = [("planted_3sat(30, 133, seed=0)", synth.planted_3sat(30, 133, seed=0)[:2]),
            ("planted_3sat(36, seed=1)", synth.planted_3sat(36, seed=1)[:2]),
            ("planted_3sat(40, seed=2)", synth.planted_3sat(40, seed=2)[:2]),
            ("planted_3sat(44, seed=3)", synth.planted_3sat(44, seed=3)[:2]),
            ("random_3sat(40, 80, seed=0)", synth.random_3sat(40, 80, seed=0))]

try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
except Exception as exc:            # the numbers below still stand; say that the card could not be read
    card = "unknown (%s)" % type(exc).__name__

ctx = _lib.Context(0)


def timed(fn, repeats=3):
    ms, out = [], None
    for _ in range(repeats):
        ctx.timer_begin()
        out = fn()
        ms.append(ctx.timer_end())
    return statistics.median(ms), ms, out


print("card: %s" % card)
for name, (n, clauses) in FORMULAS:
    ctx.enumerate_models(n, clauses, count_only=True)                 # warm-up (module load, scratch allocation)
    t_count, all_count, count = timed(lambda: ctx.enumerate_models(n, clauses, count_only=True))
    t_enum, all_enum, models = timed(lambda: ctx.enumerate_models(n, clauses))
    assert len(models) == count and np.all(np.diff(models.astype(np.uint64)) > 0)
    print("%-30s n=%d m=%d  models %d  count-only %.1f ms %s  enumerate %.1f ms %s  %.3g assignments/s (count-only)" % (
        name, n, len(clauses), count, t_count, ["%.1f" % t for t in all_count], t_enum, ["%.1f" % t for t in all_enum],
        2.0 ** n / (t_count / 1e3)))
ctx.close()
