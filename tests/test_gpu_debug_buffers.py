"""Where each precision keeps the debug buffers, and the launches of one round.

* Round trip: dsat_debug_write of random values, then dsat_debug_read, for every buffer in every precision.  The values come
  back exactly from fp32 storage, rounded to bf16 from bf16 storage, within 2^-17 |v| from hi/lo bf16 planes; a buffer
  the precision does not hold (hidden activations that stay on-chip) raises.
* Launch count of one round: the query and literal MLPs share their first layer on the per-layer paths (one launch)."""
import numpy as np
import pytest

from diffusionsat_b200 import _lib, graph as G, synth
from tests import helpers as H

pytestmark = pytest.mark.gpu

ALL_F32 = {name: "f32" for name in _lib.BUFFERS}
BF16 = dict(ALL_F32, **{name: "bf16" for name in ("VROW", "CROW", "SPRE", "QS", "LIT", "COUT", "UOUT")},
            **{name: None for name in ("H1", "H2", "CH", "U1", "U2", "O1")})
STORAGE = {     # precision -> buffer -> "f32", "bf16", "planes" or None (not held)
    "fp32_simt": ALL_F32,
    "fp32": dict(ALL_F32, **{name: "planes" for name in ("VROW", "CROW", "SPRE", "H2")},
                 **{name: None for name in ("H1", "CH", "U1", "U2", "O1")}),
    "bf16": BF16,
    "bf16_unfused": BF16,
}


def bind(ctx, precision, n_vars=30, chains=4):
    _, clauses = synth.random_3sat(n_vars, seed=0)
    ctx.set_model(H.make_weights(seed=5))
    ctx.set_precision(precision)
    ctx.set_graph(G.build_unit_graph(n_vars, clauses), chains=chains, group_graphs=0)
    return n_vars * chains


@pytest.mark.parametrize("precision", list(STORAGE))
@pytest.mark.parametrize("buffer", list(_lib.BUFFERS))
def test_debug_write_then_read(ctx, precision, buffer):
    bind(ctx, precision)
    store = STORAGE[precision][buffer]
    x = np.random.default_rng(_lib.BUFFERS[buffer]).standard_normal(ctx.debug_dims(buffer)).astype(np.float32)
    if store is None:
        with pytest.raises(_lib.DsatError):
            ctx.debug_write(buffer, x)
        with pytest.raises(_lib.DsatError):
            ctx.debug_read(buffer)
        return
    ctx.debug_write(buffer, x)
    got = ctx.debug_read(buffer)
    if store == "f32":
        np.testing.assert_array_equal(got, x)
    elif store == "bf16":
        np.testing.assert_array_equal(got, H.bf16_round(x))
    else:
        assert np.all(np.abs(got.astype(np.float64) - x) <= 2.0 ** -17 * np.abs(x))


@pytest.mark.parametrize("precision,launches", [("fp32", 14), ("bf16", 12), ("bf16_unfused", 18), ("fp32_simt", 18)])
def test_one_round_launch_count(ctx, precision, launches):
    n_rows = bind(ctx, precision)
    noise = H.noise_for(n_rows, 1, seed=0)
    noisy = np.stack([noise["uniform"], 1.0 - noise["uniform"]], axis=1).astype(np.float32)
    ctx.debug_begin(0.5, noisy, noise["labels"])
    before = ctx.launch_count()
    ctx.debug_round(0, noise["normals"][0])
    assert ctx.launch_count() - before == launches
