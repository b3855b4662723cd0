"""Uniformity evaluation of the sampler on one formula (SURVEY.md section 8f-2): exact model set on the GPU
(uniformity.enumerate_models up to 63 variables, uniformity.enumerate_models_by_search above, in place of the reference's
unigen/approxmc counting, utils/AllSolutions.py:44-68), `k`
samples per model as in diffusion_metrics.py:111, chi-square against the ideal uniform histogram (utils/chi_square.py).

  python scripts/uniformity_eval.py formula.cnf [weights.npz] [k] [--precision fp32|fp32_simt|bf16]
"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from diffusionsat_b200.dimacs import DimacsFile
from diffusionsat_b200.sampler import DiffusionSampler
from diffusionsat_b200.dist import keys_to_ints
from diffusionsat_b200.uniformity import (MAX_ENUMERATION_VARS, chi_square_likelihood, chi_square_vs_ideal, enumerate_models,
                                          enumerate_models_by_search)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("cnf")
    ap.add_argument("weights", nargs="?", default="no-such-checkpoint")
    ap.add_argument("k", nargs="?", type=int, default=10, help="samples per model")
    ap.add_argument("--precision", default="fp32", help="arithmetic of the Dense layers (default: the product's fp32)")
    args = ap.parse_args()
    df = DimacsFile(filename=args.cnf)
    df.load()
    sampler = DiffusionSampler(args.weights, args.cnf, precision=args.precision)
    n = df.number_of_vars()
    if n <= MAX_ENUMERATION_VARS:
        models = enumerate_models(n, df.clauses(), context=sampler.ctx).tolist()
    else:       # the histogram's keys are ints of the same packed words (sampler.samples -> dist.keys_to_ints)
        models = keys_to_ints(enumerate_models_by_search(n, df.clauses(), context=sampler.ctx), n)
    print("models:", len(models))
    hist = sampler.samples(len(models) * args.k)
    model_set = set(models)
    non_models = sum(c for key, c in hist.items() if key not in model_set)
    hit = sum(1 for key in hist if key in model_set)
    chisq, p = chi_square_vs_ideal(hist, models, samples_per_solution=None)
    print("precision: %s  samples: %d  sampled keys that are not models: %d  models hit: %d of %d  stats: %s" % (
        args.precision, sum(hist.values()), non_models, hit, len(models), sampler.last_stats))
    print("chi-square vs uniform: %.2f (dof %d)  p = %.4g" % (chisq, max(len(models) - 1, 0), p))
    ideal = {m: args.k for m in models}
    if sum(hist.values()) == len(models) * args.k:
        print("reference-style likelihood (utils/chi_square.py):", chi_square_likelihood(hist, ideal))


if __name__ == "__main__":
    main()
