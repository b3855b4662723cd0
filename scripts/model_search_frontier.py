"""The frontier constants of dsat_model_search.cuh against variants that each change one of them.

Every variant is the library source of this tree with one `constexpr` of dsat_model_search.cuh replaced, compiled with the
flags of diffusionsat_b200/build.py into a temporary directory (all variants at once), and loaded in a process of its
own.  Each formula: one warm-up call, then count-only and full enumeration (Context.enumerate_models_search), CUDA events,
median of 3.  Prints the card name and power limit with the numbers.  The variant without a frontier (levels0) searches
each formula with one warp and skips planted_3sat(100, seed=0), which takes minutes that way.
python scripts/model_search_frontier.py"""
import os
import shutil
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

VARIANTS = [("committed", None, None),
            ("levels0", "MAX_LEVELS = 64;", "MAX_LEVELS = 0;"),
            ("levels16", "MAX_LEVELS = 64;", "MAX_LEVELS = 16;"),
            ("levels32", "MAX_LEVELS = 64;", "MAX_LEVELS = 32;"),
            ("target4k", "FRONTIER_TARGET = 1 << 15;", "FRONTIER_TARGET = 1 << 12;"),
            ("target128k", "FRONTIER_TARGET = 1 << 15;", "FRONTIER_TARGET = 1 << 17;")]


def time_library(lib_path, skip_slow):
    from diffusionsat_b200 import _lib, synth
    _lib._LIB_PATH = lib_path
    ctx = _lib.Context(0)
    formulas = [("bench", synth.random_3sat(100, seed=0)), ("r100s1", synth.random_3sat(100, seed=1)),
                ("r100s2", synth.random_3sat(100, seed=2)), ("p64", synth.planted_3sat(64, seed=0)[:2]),
                ("p44", synth.planted_3sat(44, seed=3)[:2])]
    if not skip_slow:
        formulas.append(("p100", synth.planted_3sat(100, seed=0)[:2]))
    for name, (n, clauses) in formulas:
        ctx.enumerate_models_search(n, clauses, count_only=True)
        res = []
        for count_only in (True, False):
            ms = []
            for _ in range(3):
                ctx.timer_begin()
                ctx.enumerate_models_search(n, clauses, count_only=count_only)
                ms.append(ctx.timer_end())
            res.append(statistics.median(ms))
        print("  %-8s count-only %9.2f ms  enumerate %9.2f ms" % (name, res[0], res[1]), flush=True)
    ctx.close()


def main():
    from diffusionsat_b200 import build
    try:
        card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as exc:
        card = "unknown (%s)" % type(exc).__name__
    print("card: %s" % card)
    tmp = tempfile.mkdtemp(prefix="dsat_frontier_")
    try:
        procs = []
        for name, old, new in VARIANTS:
            src = os.path.join(tmp, name, "pkg", "csrc")               # ../../include as in the tree
            shutil.copytree(build.CSRC, src, ignore=shutil.ignore_patterns("*.so"))
            shutil.copytree(os.path.join(ROOT, "include"), os.path.join(tmp, name, "include"))
            if old is not None:
                path = os.path.join(src, "dsat_model_search.cuh")
                text = open(path).read()
                assert text.count(old) == 1, old
                open(path, "w").write(text.replace(old, new))
            lib = os.path.join(tmp, name, "libdsat.so")
            cmd = [build._nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
                   "-shared", "-o", lib, os.path.join(src, "dsat_api.cu")]
            procs.append((name, old, new, lib, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
        for name, old, new, lib, proc in procs:
            out = proc.communicate()[0]
            if proc.returncode != 0:
                sys.exit("building %s failed:\n%s" % (name, out.decode()[-2000:]))
        for name, old, new, lib, proc in procs:
            print("%s%s" % (name, "" if old is None else "  (%s -> %s)" % (old, new)), flush=True)
            subprocess.run([sys.executable, __file__, lib, "skip_slow" if name == "levels0" else "all"], check=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    if len(sys.argv) == 3:
        time_library(sys.argv[1], sys.argv[2] == "skip_slow")
    else:
        main()
