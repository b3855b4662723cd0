"""Device time of model enumeration by ordered search (dsat_enumerate_models_search) next to the brute force
(dsat_enumerate_models).

Both enumerators on the formulas where both run: the planted n = 30/36/40/44 formulas of model_enumeration_speed.py and
random_3sat(40, 80), which has many models and favours the brute force.  The search alone on the 64..100-variable
formulas whose counts the search was checked against, including the bench formula random_3sat(100, seed=0) and
planted_3sat(100, seed=0) (27 M models, about 430 MB of keys).  Each formula and enumerator: one warm-up call, then the
count-only call and the full enumeration as the Context methods run it (above 65 536 models a second call with the exact
capacity; copies to the host included), timed with CUDA events on the context's stream, three times each (median).
Prints the card name and power limit with the numbers.
python scripts/model_search_speed.py"""
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

from diffusionsat_b200 import _lib, synth  # noqa: E402

BOTH = [("planted_3sat(30, 133, seed=0)", synth.planted_3sat(30, 133, seed=0)[:2]),
        ("planted_3sat(36, seed=1)", synth.planted_3sat(36, seed=1)[:2]),
        ("planted_3sat(40, seed=2)", synth.planted_3sat(40, seed=2)[:2]),
        ("planted_3sat(44, seed=3)", synth.planted_3sat(44, seed=3)[:2]),
        ("random_3sat(40, 80, seed=0)", synth.random_3sat(40, 80, seed=0))]
SEARCH_ONLY = [("random_3sat(100, seed=0) bench", synth.random_3sat(100, seed=0)),
               ("random_3sat(100, seed=1)", synth.random_3sat(100, seed=1)),
               ("random_3sat(100, seed=2)", synth.random_3sat(100, seed=2)),
               ("random_3sat(100, seed=3)", synth.random_3sat(100, seed=3)),
               ("random_3sat(80, seed=1)", synth.random_3sat(80, seed=1)),
               ("random_3sat(80, seed=2)", synth.random_3sat(80, seed=2)),
               ("random_3sat(64, seed=1)", synth.random_3sat(64, seed=1)),
               ("random_3sat(64, seed=2)", synth.random_3sat(64, seed=2)),
               ("planted_3sat(64, seed=0)", synth.planted_3sat(64, seed=0)[:2]),
               ("planted_3sat(100, seed=0)", synth.planted_3sat(100, seed=0)[:2])]

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


def run(label, method, n, clauses):
    method(n, clauses, count_only=True)                                # warm-up (module load, scratch allocation)
    t_count, all_count, count = timed(lambda: method(n, clauses, count_only=True))
    t_enum, all_enum, models = timed(lambda: method(n, clauses))
    assert len(models) == count
    print("  %-12s models %9d  count-only %8.2f ms %s  enumerate %8.2f ms %s" % (
        label, count, t_count, ["%.2f" % t for t in all_count], t_enum, ["%.2f" % t for t in all_enum]), flush=True)
    return models


print("card: %s" % card)
for name, (n, clauses) in BOTH:
    print("%s n=%d m=%d" % (name, n, len(clauses)))
    brute = run("brute force", ctx.enumerate_models, n, clauses)
    search = run("search", ctx.enumerate_models_search, n, clauses)
    assert np.array_equal(search[:, 0], brute)
for name, (n, clauses) in SEARCH_ONLY:
    print("%s n=%d m=%d" % (name, n, len(clauses)))
    run("search", ctx.enumerate_models_search, n, clauses)
ctx.close()
