"""clock64 breakdown of CTA 0 of the seven x3 MLP launches: python scripts/profile_x3.py [chains] [n]"""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from diffusionsat_b200 import _lib, synth, weights, graph
chains = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
n = int(sys.argv[2]) if len(sys.argv) > 2 else 100
ctx = _lib.Context(0); ctx.set_model(weights.init_weights(seed=1234)); ctx.set_precision("fp32")
nv, cl = synth.random_3sat(n, seed=0); ctx.set_graph(graph.build_unit_graph(nv, cl), chains=chains, group_graphs=31)
ctx.profile_rounds(2)
names = ["query", "lit1", "lit2", "lit3", "clause", "update", "output"]
for w in range(7):
    c = ctx.profile_fused(w)
    tot = c[0] or 1
    # "A reads": the wait before accumulating into the half the previous hidden layer's MMAs read their A operand from
    print("%-7s mma warp %9d cyc | waits: accumulator %4.1f%%  A reads %4.1f%%  hidden %4.1f%%  input %4.1f%%  weights %4.1f%% | epilogue warp: tmem_full wait %4.1f%%  hidden epi %4.1f%%  final epi %4.1f%%"
          % (names[w], tot, 100 * c[1] / tot, 100 * c[8] / tot, 100 * c[2] / tot, 100 * c[3] / tot, 100 * c[4] / tot, 100 * c[5] / tot, 100 * c[6] / tot, 100 * c[7] / tot))
