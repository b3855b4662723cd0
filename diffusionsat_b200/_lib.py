"""ctypes binding of libdsat.so (include/dsat.h) and a thin Python handle over a context.

There is no CPU fallback: importing this module without the built library, or creating a context
without a CUDA device, raises.
"""

from __future__ import annotations

import ctypes as C
import os

import numpy as np

from .graph import UnitGraph
from .weights import QuerySATWeights, flat_layer_names

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc", "libdsat.so")

# dsat_dtype: F32 = fp32 FMA on the CUDA cores, F32_TC = fp32-accurate split-bf16 products on the tensor cores (default),
# BF16 = plain bf16 tensor-core path, BF16_UNFUSED = the same with one kernel per Dense layer
F32, BF16, BF16_UNFUSED, F32_TC = 0, 1, 2, 3
PRECISIONS = {"fp32": F32_TC, "fp32_tc": F32_TC, "fp32_simt": F32, "bf16": BF16, "bf16_unfused": BF16_UNFUSED}

BUFFERS = {name: i for i, name in enumerate(
    ["VROW", "CROW", "H1", "H2", "QS", "LIT", "CH", "COUT", "U1", "U2", "UOUT", "SPRE", "O1", "LOGITS", "OUT", "X"])}

_f32p = C.POINTER(C.c_float)
_i32p = C.POINTER(C.c_int32)
_u64p = C.POINTER(C.c_uint64)
_u8p = C.POINTER(C.c_uint8)
_vp = C.c_void_p

_SIGNATURES = {
    "dsat_version": (C.c_int, []),
    "dsat_build_info": (C.c_int, []),
    "dsat_create": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "dsat_destroy": (None, [_vp]),
    "dsat_last_error": (C.c_char_p, [_vp]),
    "dsat_set_stream": (C.c_int, [_vp, _vp]),
    "dsat_synchronize": (C.c_int, [_vp]),
    "dsat_timer_begin": (C.c_int, [_vp]),
    "dsat_timer_end": (C.c_int, [_vp, _f32p]),
    "dsat_launch_count": (C.c_longlong, [_vp]),
    "dsat_set_model": (C.c_int, [_vp, C.c_int, C.POINTER(_f32p), C.POINTER(_f32p), _i32p, _i32p]),
    "dsat_set_precision": (C.c_int, [_vp, C.c_int]),
    "dsat_set_sampling": (C.c_int, [_vp, C.c_int]),
    "dsat_debug_rounding": (C.c_int, [_vp, C.c_uint64, C.c_int]),
    "dsat_get_precision": (C.c_int, [_vp]),
    "dsat_set_graph": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _i32p, _i32p, _i32p, _i32p, C.c_int, _i32p, _i32p,
                                 C.c_int, C.c_int]),
    "dsat_set_batches": (C.c_int, [_vp, C.c_int, _i32p, _u64p]),
    "dsat_graph_build": (C.c_int, [C.c_int, C.c_int, C.c_longlong, _i32p, _i32p, _i32p, _i32p, _i32p, _i32p, _i32p]),
    "dsat_model_call": (C.c_int, [_vp, C.c_float, _f32p, _i32p, _f32p, C.c_int, C.c_uint64, C.c_uint64, _f32p, _i32p,
                                  _f32p]),
    "dsat_sample": (C.c_int, [_vp, C.c_int, C.c_int, C.c_uint64, C.c_uint64, _f32p, _i32p, _f32p, _u64p, _u8p, _i32p,
                              _u8p]),
    "dsat_sample_enqueue": (C.c_int, [_vp, C.c_int, C.c_int, C.c_uint64, C.c_uint64]),
    "dsat_sample_fetch": (C.c_int, [_vp, _u64p, _u8p, _i32p, _u8p]),
    "dsat_words_per_graph": (C.c_int, [_vp]),
    "dsat_hist_reduce": (C.c_int, [_vp, C.c_int, _u64p, C.POINTER(C.c_int64), C.c_int, _i32p, _i32p]),
    "dsat_hist_reduce_segments": (C.c_int, [_vp, C.c_int, _i32p, _i32p, _u64p, C.POINTER(C.c_int64), C.c_int, _i32p, _i32p]),
    "dsat_spmm": (C.c_int, [_vp, C.c_int, _vp, _vp, C.c_int, C.c_int, C.c_int]),
    "dsat_profile_classes": (C.c_int, []),
    "dsat_profile_fused": (C.c_int, [_vp, C.c_int, C.POINTER(C.c_longlong)]),
    "dsat_profile_rounds": (C.c_int, [_vp, C.c_int, C.c_uint64, _f32p, _i32p]),
    "dsat_tc_linear_test": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _f32p, _f32p, _f32p, C.c_int, C.c_int, _f32p]),
    "dsat_debug_begin": (C.c_int, [_vp, C.c_float, _f32p, _i32p]),
    "dsat_debug_round": (C.c_int, [_vp, C.c_int, _f32p]),
    "dsat_debug_dims": (C.c_int, [_vp, C.c_int, C.POINTER(C.c_longlong), C.POINTER(C.c_int)]),
    "dsat_debug_read": (C.c_int, [_vp, C.c_int, _f32p, C.c_longlong]),
    "dsat_debug_write": (C.c_int, [_vp, C.c_int, _f32p, C.c_longlong]),
    "dsat_debug_groups": (C.c_int, [_vp, _i32p, _i32p, _f32p, _i32p, _i32p]),
    "dsat_debug_mlp": (C.c_int, [_vp, C.c_int]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def library_path() -> str:
    return _LIB_PATH


def load_library():
    """Load libdsat.so and declare every prototype.  Raises if the library was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise RuntimeError(
            "libdsat.so is missing (%s). Build it with `python -m diffusionsat_b200.build`; "
            "diffusionsat_b200 has no CPU fallback." % _LIB_PATH)
    lib = C.CDLL(_LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class DsatError(RuntimeError):
    pass


def _ptr(arr, ctype):
    return arr.ctypes.data_as(C.POINTER(ctype)) if arr is not None else None


def _as(arr, dtype, shape=None):
    if arr is None:
        return None
    out = np.ascontiguousarray(arr, dtype=dtype)
    if shape is not None and tuple(out.shape) != tuple(shape):
        raise ValueError("expected shape %r, got %r" % (tuple(shape), tuple(out.shape)))
    return out


class Context:
    """One libdsat context = one GPU."""

    def __init__(self, device: int = 0):
        self._lib = load_library()
        handle = _vp()
        rc = self._lib.dsat_create(int(device), C.byref(handle))
        if rc != 0 or not handle:
            raise DsatError("dsat_create(device=%d) failed with %d: no usable CUDA device; "
                            "diffusionsat_b200 has no CPU fallback" % (device, rc))
        self._h = handle
        self.device = int(device)
        self.graph = None
        self.chains = 0
        self.feature_maps = self.query_maps = 0

    # ------------------------------------------------------------------ plumbing
    def close(self):
        if getattr(self, "_h", None):
            self._lib.dsat_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            msg = self._lib.dsat_last_error(self._h)
            raise DsatError("libdsat error %d: %s" % (rc, msg.decode() if msg else "?"))

    def set_stream(self, cuda_stream_ptr):
        self._check(self._lib.dsat_set_stream(self._h, _vp(cuda_stream_ptr) if cuda_stream_ptr else None))

    def synchronize(self):
        self._check(self._lib.dsat_synchronize(self._h))

    def timer_begin(self):
        self._check(self._lib.dsat_timer_begin(self._h))

    def timer_end(self) -> float:
        ms = C.c_float(0)
        self._check(self._lib.dsat_timer_end(self._h, C.byref(ms)))
        return float(ms.value)

    def launch_count(self) -> int:
        return int(self._lib.dsat_launch_count(self._h))

    # --------------------------------------------------------------------- setup
    def set_model(self, weights: QuerySATWeights):
        names = flat_layer_names(weights.feature_maps, weights.query_maps)
        kernels = [np.ascontiguousarray(weights.layers[n][0], dtype=np.float32) for n in names]
        biases = [np.ascontiguousarray(weights.layers[n][1], dtype=np.float32) for n in names]
        kp = (_f32p * len(names))(*[_ptr(k, C.c_float) for k in kernels])
        bp = (_f32p * len(names))(*[_ptr(b, C.c_float) for b in biases])
        ins = np.array([k.shape[0] for k in kernels], dtype=np.int32)
        outs = np.array([k.shape[1] for k in kernels], dtype=np.int32)
        self._check(self._lib.dsat_set_model(self._h, len(names), kp, bp, _ptr(ins, C.c_int32), _ptr(outs, C.c_int32)))
        self.feature_maps, self.query_maps = weights.feature_maps, weights.query_maps

    def set_precision(self, dtype):
        """`dtype`: a dsat_dtype code or one of PRECISIONS' names ("fp32" = fp32-accurate tensor-core path)."""
        if isinstance(dtype, str):
            dtype = PRECISIONS[dtype]
        self._check(self._lib.dsat_set_precision(self._h, int(dtype)))

    SAMPLING = {"inverse_cdf": 0, "gumbel": 1}

    def set_sampling(self, mode):
        """"inverse_cdf" = floor(x0 + U) (the reference's live code, default) or "gumbel" = Gumbel-argmax."""
        self._check(self._lib.dsat_set_sampling(self._h, self.SAMPLING[mode] if isinstance(mode, str) else int(mode)))

    def debug_rounding(self, seed=0, step=0):
        self._check(self._lib.dsat_debug_rounding(self._h, C.c_uint64(seed), int(step)))

    def get_precision(self) -> int:
        return int(self._lib.dsat_get_precision(self._h))

    def set_graph(self, graph: UnitGraph, chains: int, group_graphs: int = 0):
        g = graph
        arrs = [np.ascontiguousarray(a, dtype=np.int32) for a in
                (g.cl_rowptr, g.cl_lit, g.lit_rowptr, g.lit_clause, g.var_seg, g.clause_seg)]
        self._check(self._lib.dsat_set_graph(
            self._h, g.n_vars, g.n_clauses, g.nnz, _ptr(arrs[0], C.c_int32), _ptr(arrs[1], C.c_int32),
            _ptr(arrs[2], C.c_int32), _ptr(arrs[3], C.c_int32), g.n_graphs, _ptr(arrs[4], C.c_int32),
            _ptr(arrs[5], C.c_int32), int(chains), int(group_graphs)))
        self.graph, self.chains = g, int(chains)
        self.group_graphs = int(group_graphs) if group_graphs > 0 else g.n_graphs * int(chains)
        self.batch_groups = None

    def set_batches(self, group_seg, noise_base=None):
        """Early-exit groups ``[group_seg[i], group_seg[i+1])`` of the bound graphs and, optionally, the Philox element of
        variable 0 of every graph (``dsat_set_batches``); cleared by the next ``set_graph``."""
        seg = np.ascontiguousarray(group_seg, dtype=np.int32)
        base = None if noise_base is None else np.ascontiguousarray(noise_base, dtype=np.uint64)
        if base is not None and base.shape != (self.total_graphs,):
            raise ValueError("noise_base needs one entry per graph (%d), got %r" % (self.total_graphs, base.shape))
        self._check(self._lib.dsat_set_batches(self._h, int(seg.shape[0]) - 1, _ptr(seg, C.c_int32), _ptr(base, C.c_uint64)))
        self.batch_groups = int(seg.shape[0]) - 1

    # ------------------------------------------------------------------ properties
    @property
    def n_rows(self) -> int:
        return self.graph.n_vars * self.chains

    @property
    def n_clause_rows(self) -> int:
        return self.graph.n_clauses * self.chains

    @property
    def total_graphs(self) -> int:
        return self.graph.n_graphs * self.chains

    @property
    def n_groups(self) -> int:
        if getattr(self, "batch_groups", None):
            return self.batch_groups
        return -(-self.total_graphs // self.group_graphs)

    # ------------------------------------------------------------------------ calls
    def model_call(self, noise_scale, noisy_num, labels=None, normals=None, rounds=32, seed=0, chain_offset=0):
        n = self.n_rows
        noisy = _as(noisy_num, np.float32, (n, 2))
        lab = _as(labels, np.int32, (n,))
        nrm = _as(normals, np.float32, (rounds, n, 4)) if normals is not None else None
        pred = np.empty(n, dtype=np.float32)
        steps = np.empty(self.n_groups, dtype=np.int32)
        loss = np.empty(self.n_groups, dtype=np.float32)
        self._check(self._lib.dsat_model_call(
            self._h, C.c_float(noise_scale), _ptr(noisy, C.c_float), _ptr(lab, C.c_int32), _ptr(nrm, C.c_float),
            int(rounds), C.c_uint64(seed), C.c_uint64(chain_offset), _ptr(pred, C.c_float), _ptr(steps, C.c_int32),
            _ptr(loss, C.c_float)))
        return pred, steps, loss

    def _sample_outputs(self):
        g = self.total_graphs
        words = int(self._lib.dsat_words_per_graph(self._h))
        return (np.empty((g, words), dtype=np.uint64), np.empty(g, dtype=np.uint8), np.empty(g, dtype=np.int32),
                np.empty(g, dtype=np.uint8))

    def sample(self, n_steps=32, n_rounds=32, seed=0, chain_offset=0, uniforms=None, labels=None, normals=None):
        n = self.n_rows
        uni = _as(uniforms, np.float32, (n_steps, n)) if uniforms is not None else None
        lab = _as(labels, np.int32, (n_steps, n)) if labels is not None else None
        nrm = _as(normals, np.float32, (n_steps, n_rounds, n, 4)) if normals is not None else None
        packed, is_sat, latch, sat_any = self._sample_outputs()
        self._check(self._lib.dsat_sample(
            self._h, int(n_steps), int(n_rounds), C.c_uint64(seed), C.c_uint64(chain_offset), _ptr(uni, C.c_float),
            _ptr(lab, C.c_int32), _ptr(nrm, C.c_float), _ptr(packed, C.c_uint64), _ptr(is_sat, C.c_uint8),
            _ptr(latch, C.c_int32), _ptr(sat_any, C.c_uint8)))
        return packed, is_sat, latch, sat_any

    def sample_enqueue(self, n_steps=32, n_rounds=32, seed=0, chain_offset=0):
        self._check(self._lib.dsat_sample_enqueue(self._h, int(n_steps), int(n_rounds), C.c_uint64(seed),
                                                  C.c_uint64(chain_offset)))

    def sample_fetch(self):
        packed, is_sat, latch, sat_any = self._sample_outputs()
        self._check(self._lib.dsat_sample_fetch(self._h, _ptr(packed, C.c_uint64), _ptr(is_sat, C.c_uint8),
                                                _ptr(latch, C.c_int32), _ptr(sat_any, C.c_uint8)))
        return packed, is_sat, latch, sat_any

    def sample_fetch_sat(self) -> np.ndarray:
        """Only the per-chain SAT flags of the last run (the sampler's stop rules need nothing else)."""
        is_sat = np.empty(self.total_graphs, dtype=np.uint8)
        self._check(self._lib.dsat_sample_fetch(self._h, None, _ptr(is_sat, C.c_uint8), None, None))
        return is_sat

    def hist_reduce(self, chain_limit: int = 0):
        """Device-side sort / unique / count of the satisfying assignments of chains ``[0, chain_limit)`` of the last
        run (0 = all): ``(keys [K, words] uint64 ascending, counts [K] int64, n_sat)``."""
        words = int(self._lib.dsat_words_per_graph(self._h))
        cap = self.total_graphs if chain_limit <= 0 else min(int(chain_limit), self.total_graphs)
        keys = np.empty((cap, words), dtype=np.uint64)
        counts = np.empty(cap, dtype=np.int64)
        k, n_sat = C.c_int32(0), C.c_int32(0)
        self._check(self._lib.dsat_hist_reduce(self._h, int(chain_limit), _ptr(keys, C.c_uint64),
                                               counts.ctypes.data_as(C.POINTER(C.c_int64)), cap, C.byref(k), C.byref(n_sat)))
        return keys[:k.value], counts[:k.value], int(n_sat.value)

    def hist_reduce_segments(self, graph_seg, limits):
        """``hist_reduce`` per segment ``[graph_seg[s], graph_seg[s+1])`` of the last run's graphs, counting the first
        ``limits[s]`` of each: ``([(keys [K_s, words] uint64 ascending, counts [K_s] int64) per segment], n_sat)``."""
        seg = np.ascontiguousarray(graph_seg, dtype=np.int32)
        lim = np.ascontiguousarray(limits, dtype=np.int32)
        n_seg = int(seg.shape[0]) - 1
        if lim.shape != (n_seg,):
            raise ValueError("one limit per segment (%d), got %r" % (n_seg, lim.shape))
        words = int(self._lib.dsat_words_per_graph(self._h))
        cap = int(np.minimum(lim, np.diff(seg)).clip(min=0).sum()) if n_seg > 0 else 0
        keys = np.empty((max(cap, 1), words), dtype=np.uint64)
        counts = np.empty(max(cap, 1), dtype=np.int64)
        runs = np.zeros(n_seg + 1, dtype=np.int32)
        n_sat = C.c_int32(0)
        self._check(self._lib.dsat_hist_reduce_segments(self._h, n_seg, _ptr(seg, C.c_int32), _ptr(lim, C.c_int32),
                                                        _ptr(keys, C.c_uint64), counts.ctypes.data_as(C.POINTER(C.c_int64)),
                                                        cap, _ptr(runs, C.c_int32), C.byref(n_sat)))
        return [(keys[runs[s]:runs[s + 1]], counts[runs[s]:runs[s + 1]]) for s in range(n_seg)], int(n_sat.value)

    def spmm(self, direction: int, x_dev_ptr: int, y_dev_ptr: int, feat: int, dtype: int, chains: int):
        self._check(self._lib.dsat_spmm(self._h, int(direction), _vp(x_dev_ptr), _vp(y_dev_ptr), int(feat), int(dtype),
                                        int(chains)))

    PROFILE_CLASSES = ("v1_hidden", "query_out", "lit_2", "lit_3", "clause_1", "clause_2", "update_1", "update_2",
                       "update_3", "output_1", "output_2", "clause_gather", "literal_gather", "pairnorm_clause",
                       "pairnorm_var", "head", "noise")

    def profile_rounds(self, rounds=4, seed=0):
        """{class: (total_ms, launches)} of `rounds` rounds, CUDA events on the launching stream."""
        k = int(self._lib.dsat_profile_classes())
        ms = np.zeros(k, dtype=np.float32)
        cnt = np.zeros(k, dtype=np.int32)
        self._check(self._lib.dsat_profile_rounds(self._h, int(rounds), C.c_uint64(seed), _ptr(ms, C.c_float),
                                                  _ptr(cnt, C.c_int32)))
        return {name: (float(ms[i]), int(cnt[i])) for i, name in enumerate(self.PROFILE_CLASSES[:k])}

    def profile_fused(self, which):
        arr = (C.c_longlong * 16)()
        self._check(self._lib.dsat_profile_fused(self._h, int(which), arr))
        return list(arr)

    def tc_linear_test(self, a, w, bias, epi=0, out_bf16=False):
        """Run the tcgen05 linear kernel alone on host arrays (a [rows,K], w [K,N], bias [N])."""
        a = _as(a, np.float32)
        w = _as(w, np.float32)
        bias = _as(bias, np.float32)
        rows, k = a.shape
        n = w.shape[1]
        out = np.empty((rows, 3 * n if epi == 2 else n), dtype=np.float32)
        self._check(self._lib.dsat_tc_linear_test(self._h, rows, k, n, _ptr(a, C.c_float), _ptr(w, C.c_float),
                                                  _ptr(bias, C.c_float), int(epi), int(bool(out_bf16)),
                                                  _ptr(out, C.c_float)))
        return out

    # ------------------------------------------------------------------------ debug
    def debug_begin(self, noise_scale, noisy_num, labels=None):
        n = self.n_rows
        noisy = _as(noisy_num, np.float32, (n, 2))
        lab = _as(labels, np.int32, (n,))
        self._check(self._lib.dsat_debug_begin(self._h, C.c_float(noise_scale), _ptr(noisy, C.c_float),
                                               _ptr(lab, C.c_int32)))

    def debug_round(self, round_index, normals=None):
        nrm = _as(normals, np.float32, (self.n_rows, 4)) if normals is not None else None
        self._check(self._lib.dsat_debug_round(self._h, int(round_index), _ptr(nrm, C.c_float)))

    def debug_dims(self, name):
        rows, ld = C.c_longlong(0), C.c_int(0)
        self._check(self._lib.dsat_debug_dims(self._h, BUFFERS[name], C.byref(rows), C.byref(ld)))
        return int(rows.value), int(ld.value)

    def debug_read(self, name) -> np.ndarray:
        rows, ld = self.debug_dims(name)
        out = np.empty((rows, ld), dtype=np.float32)
        self._check(self._lib.dsat_debug_read(self._h, BUFFERS[name], _ptr(out, C.c_float), rows * ld))
        return out

    def debug_write(self, name, values):
        rows, ld = self.debug_dims(name)
        arr = _as(values, np.float32, (rows, ld))
        self._check(self._lib.dsat_debug_write(self._h, BUFFERS[name], _ptr(arr, C.c_float), rows * ld))

    MLPS = ("variables_query", "lit_query", "clause_update", "update_gate", "variables_output")

    def debug_mlp(self, which):
        """Run one MLP alone (index or name from MLPS) on the current contents of its input buffer."""
        if isinstance(which, str):
            which = self.MLPS.index(which)
        self._check(self._lib.dsat_debug_mlp(self._h, int(which)))

    def debug_groups(self):
        done = np.empty(self.n_groups, dtype=np.int32)
        steps = np.empty(self.n_groups, dtype=np.int32)
        loss_sum = np.empty(self.n_groups, dtype=np.float32)
        gsat = np.empty(self.total_graphs, dtype=np.int32)
        gmap = np.empty(self.total_graphs, dtype=np.int32)
        self._check(self._lib.dsat_debug_groups(self._h, _ptr(done, C.c_int32), _ptr(steps, C.c_int32),
                                                _ptr(loss_sum, C.c_float), _ptr(gsat, C.c_int32), _ptr(gmap, C.c_int32)))
        return dict(done=done, steps_taken=steps, loss_sum=loss_sum, graph_sat=gsat, graph_map=gmap)
