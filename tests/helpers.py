"""Shared fixtures for the parity tests: seeded formulas, weights, noise, oracle runs."""
import numpy as np
import torch

from diffusionsat_b200 import synth, weights as W
from oracle import querysat_oracle as O


def make_weights(feature_maps=128, query_maps=128, seed=7, bias_scale=0.1, lit_hidden=None):
    """Seeded weights; `lit_hidden` narrows the literal MLP's hidden layers (the C ABI takes any consistent widths)."""
    wts = W.init_weights(feature_maps, query_maps, seed=seed, bias_scale=bias_scale)
    if lit_hidden is not None:
        for i in range(3):
            k, b = wts.layers["lit_query/%d" % i]
            k = k[:, :lit_hidden] if i == 0 else k[:lit_hidden, :lit_hidden] if i == 1 else k[:lit_hidden]
            wts.layers["lit_query/%d" % i] = (np.ascontiguousarray(k), b[:lit_hidden] if i < 2 else b)
    return wts


def noise_for(n_rows, rounds, seed, steps=None):
    rng = np.random.default_rng(seed)
    if steps is None:
        return dict(normals=rng.standard_normal((rounds, n_rows, 4)).astype(np.float32),
                    labels=rng.integers(0, 2, n_rows).astype(np.int32),
                    uniform=rng.random(n_rows).astype(np.float32))
    return dict(normals=rng.standard_normal((steps, rounds, n_rows, 4)).astype(np.float32),
                labels=rng.integers(0, 2, (steps, n_rows)).astype(np.int32),
                uniforms=rng.random((steps, n_rows)).astype(np.float32))


def oracle_trace(n_vars, clauses, chains, wts, noise_scale, noisy, noise, rounds, dtype=torch.float32, teacher=None):
    graph = O.OracleGraph.copies(n_vars, clauses, chains)
    w = O.weights_to_torch(wts, dtype)
    trace = []
    out = O.model_loop(graph, w, noise_scale, torch.from_numpy(noisy), torch.from_numpy(noise["labels"].astype(np.int64)),
                       torch.from_numpy(noise["normals"]), rounds, dtype=dtype, trace=trace, teacher=teacher)
    return graph, out, trace


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / (np.max(np.abs(b)) + 1e-12))


def bf16_round(x):
    """Round-to-nearest-even to bfloat16, returned as float32 (numpy has no bf16)."""
    a = np.ascontiguousarray(x, dtype=np.float32)
    bits = a.view(np.uint32).astype(np.uint64)
    rounded = ((bits + 0x7FFF + ((bits >> 16) & 1)) >> 16) << 16
    return rounded.astype(np.uint32).view(np.float32).reshape(a.shape)


def elementwise_excess(got, want, rel, abs_of_rms):
    """max over elements of |got - want| / (rel |want| + abs_of_rms rms(want)); <= 1 means every element is inside."""
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    rms = float(np.sqrt(np.mean(want ** 2))) + 1e-30
    return float(np.max(np.abs(got - want) / (rel * np.abs(want) + abs_of_rms * rms)))
