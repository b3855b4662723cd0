"""Small-launch regime (BASELINE configs[0]): wall time of DiffusionSampler.samples(256) at n=30 through the public API.
python scripts/small_case_latency.py [precision]"""
import contextlib, io, os, sys, tempfile, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from diffusionsat_b200 import synth
from diffusionsat_b200.sampler import DiffusionSampler
prec = sys.argv[1] if len(sys.argv) > 1 else "fp32"
fixture = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "trained_small.npz")
n, clauses, _ = synth.planted_3sat(30, 133, seed=0)
cnf = os.path.join(tempfile.mkdtemp(), "f.cnf")
open(cnf, "w").write(synth.dimacs_text(n, clauses))
with contextlib.redirect_stdout(io.StringIO()):
    s = DiffusionSampler(fixture, cnf, precision=prec, seed=5)
    t0 = time.perf_counter(); s.samples(256); cold = time.perf_counter() - t0
    times = []
    for _ in range(3):
        t0 = time.perf_counter(); h = s.samples(256); times.append(time.perf_counter() - t0)
print("%s: samples(256) n=30: cold %.3f s, warm %s s, %d chains launched per call, launches %d" % (
    prec, cold, ["%.3f" % t for t in times], s.last_stats["chains_launched"], s.ctx.launch_count()))
