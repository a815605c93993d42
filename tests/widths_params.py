"""Parameters of a VectorFieldNet whose branches have their own hidden widths, for the tests of that network.

`init_params_widths` draws exactly what oracle.vector_field.init_params draws (same generator calls in the same order, the same
fan-in scaling and zero-scaled heads), layer by layer with the shapes of exe_flow_matching.layer_shapes: with all six widths
equal it returns the oracle's parameters bit for bit (tests/test_hidden_widths.py checks that)."""
import numpy as np


def shapes(d, widths, F=128):
    (t0, t1), (x0, x1), (xt0, xt1) = widths
    return [(2 * F, t0), (t0, t1), (d, x0), (x0, x1), (t1, d), (x1 + t1, xt0), (xt0, xt1), (xt1, d)]


def init_params_widths(rng: np.random.Generator, d, widths, F=128, head_scale=0.0, dtype=np.float32):
    p = {}
    for i, (fi, fo) in enumerate(shapes(d, widths, F)):
        scale = 1.0 / np.sqrt(fi)
        if i in (4, 7):
            scale *= head_scale
        p[f"Dense_{i}"] = {
            "kernel": (rng.standard_normal((fi, fo)) * scale).astype(dtype),
            "bias": (rng.standard_normal(fo) * 0.01).astype(dtype),
        }
    return {"params": p}
