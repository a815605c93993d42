"""VectorFieldNet with per-branch hidden widths (--hidden_t / --hidden_x / --hidden_xt): the descriptor layout against the header,
the flat parameter layout and its flax-dict round trip, the descriptor the host builds, the depth limit, and the float64 oracle's
algebra for unequal widths.  CPU only; the kernels are checked in tests/test_gpu_hidden_widths.py."""
import ctypes
import os
import subprocess
import tempfile
import textwrap
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import targets as OT, vector_field as VF
from tests.widths_params import init_params_widths

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WIDTHS = {   # ((Ht0, Ht1), (Hx0, Hx1), (Hxt0, Hxt1))
    "4-mode": ((32, 64), (128, 100), (64, 128)),
    "phi-four": ((64, 64), (128, 256), (256, 128)),
    "pines": ((256, 256), (1024, 1024), (1024, 512)),
}


def _net(widths, d=2, F=16):
    from mfm_b200 import exe_flow_matching as E
    (t, x, xt) = widths
    return E.VectorFieldNet(torch.zeros(F), SimpleNamespace(dim=d), list(x), list(t), list(xt))


def test_field_descriptor_offsets_match_header():
    from mfm_b200 import _lib
    code = textwrap.dedent("""
        #include <stdio.h>
        #include <stddef.h>
        #include "mfm_b200.h"
        int main(){ printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(mfm_field_t), offsetof(mfm_field_t, ref_band),
                           offsetof(mfm_field_t, hidden_t), offsetof(mfm_field_t, hidden_x), offsetof(mfm_field_t, hidden_xt),
                           sizeof(((mfm_field_t*)0)->hidden_xt)); return 0; }
    """)
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "t.c"); exe = os.path.join(d, "t")
        open(c, "w").write(code)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        out = [int(v) for v in subprocess.check_output([exe]).decode().split()]
    F = _lib.FieldDesc
    assert out == [ctypes.sizeof(F), F.ref_band.offset, F.hidden_t.offset, F.hidden_x.offset, F.hidden_xt.offset, 8]
    # appended after the last pointer, packed: no older offset moves and the struct grows by exactly the six ints
    assert F.hidden_t.offset == F.ref_band.offset + 8 and ctypes.sizeof(F) == F.hidden_t.offset + 24


@pytest.mark.parametrize("name", list(WIDTHS))
def test_layer_shapes_and_offsets(name):
    from mfm_b200 import exe_flow_matching as E
    (t0, t1), (x0, x1), (xt0, xt1) = w = WIDTHS[name]
    d, F = {"4-mode": 2, "phi-four": 64, "pines": 1600}[name], 128
    H = max(t0, t1, x0, x1, xt0, xt1)
    want = [(2 * F, t0), (t0, t1), (d, x0), (x0, x1), (t1, d), (x1 + t1, xt0), (xt0, xt1), (xt1, d)]
    assert E.layer_shapes(d, H, F, w) == want
    P = E.VectorFieldParams(d, H, F, "cpu", widths=w)
    assert P.hidden == H and P.widths == w and P.shapes == want
    off = 0
    for i, (fi, fo) in enumerate(want):
        assert P.w_off[i] == off and P.w_off[i] % 4 == 0
        off = (off + fi * fo + 3) // 4 * 4
        assert P.b_off[i] == off
        off = (off + fo + 3) // 4 * 4
    assert P.n_params == off == P.flat.numel()
    assert int(P.decay_mask.sum()) == sum(fi * fo for fi, fo in want)


def test_equal_widths_keep_the_layout():
    from mfm_b200 import exe_flow_matching as E
    a = E.VectorFieldParams(64, 128, 128, "cpu")
    b = E.VectorFieldParams(64, 128, 128, "cpu", widths=((128, 128),) * 3)
    assert a.shapes == b.shapes and a.w_off == b.w_off and a.b_off == b.b_off and a.n_params == b.n_params
    assert a.shapes == E.layer_shapes(64, 128, 128)


@pytest.mark.parametrize("name", list(WIDTHS))
def test_flax_dict_round_trip(name):
    from mfm_b200 import exe_flow_matching as E
    w = WIDTHS[name]
    d = {"4-mode": 2, "phi-four": 64, "pines": 1600}[name]
    params = init_params_widths(np.random.default_rng(3), d, w, 128, head_scale=0.1)
    P = E.VectorFieldParams(d, max(max(b) for b in w), 128, "cpu", widths=w).load_dict(params)
    back = P.to_dict()
    for i in range(8):
        for k in ("kernel", "bias"):
            assert np.array_equal(back["params"][f"Dense_{i}"][k], params["params"][f"Dense_{i}"][k]), (i, k)
    # the padding between slices stays zero: nothing of one layer spills into another
    used = np.zeros(P.n_params, bool)
    for i, (fi, fo) in enumerate(P.shapes):
        used[P.w_off[i]:P.w_off[i] + fi * fo] = True
        used[P.b_off[i]:P.b_off[i] + fo] = True
    assert (P.flat.numpy()[~used] == 0).all()


def test_width_initialiser_equals_the_oracle_for_equal_widths():
    for d, H in ((2, 128), (64, 128), (16, 48)):
        a = VF.init_params(np.random.default_rng(11), d, H, 128, head_scale=0.2)
        b = init_params_widths(np.random.default_rng(11), d, ((H, H),) * 3, 128, head_scale=0.2)
        for i in range(8):
            for k in ("kernel", "bias"):
                assert np.array_equal(a["params"][f"Dense_{i}"][k], b["params"][f"Dense_{i}"][k])


def test_descriptor_tail():
    from mfm_b200 import exe_flow_matching as E
    net = _net(((128, 128),) * 3)
    P = E.VectorFieldParams(2, 128, 16, "cpu")
    fd = net.field_desc(P)
    assert fd.hidden == 128 and list(fd.hidden_t) == [0, 0] and list(fd.hidden_x) == [0, 0] and list(fd.hidden_xt) == [0, 0]
    w = WIDTHS["4-mode"]
    net = _net(w)
    assert net.hidden == 128 and net.widths == w
    P = E.VectorFieldParams(2, 128, 16, "cpu", widths=w)
    fd = net.field_desc(P)
    assert [list(fd.hidden_t), list(fd.hidden_x), list(fd.hidden_xt)] == [list(b) for b in w] and fd.hidden == 128
    assert [fd.w_off[i] for i in range(8)] == P.w_off and fd.n_params == P.n_params


def test_equal_width_descriptor_bytes_unchanged():
    """Equal widths given explicitly produce the same descriptor bytes as the equal-width network of before."""
    from mfm_b200 import exe_flow_matching as E
    net = _net(((64, 64),) * 3)
    P1 = E.VectorFieldParams(2, 64, 16, "cpu")
    P2 = E.VectorFieldParams(2, 64, 16, "cpu", widths=((64, 64),) * 3)
    P2.flat = P1.flat
    a, b = net.field_desc(P1), net.field_desc(P2)
    assert bytes(a) == bytes(b)


@pytest.mark.parametrize("depth", [1, 3])
def test_depth_other_than_two_raises(depth):
    from mfm_b200 import exe_flow_matching as E
    for which in range(3):
        ws = [[64, 64], [64, 64], [64, 64]]
        ws[which] = [64] * depth
        with pytest.raises(NotImplementedError, match="two hidden layers per branch"):
            E.VectorFieldNet(torch.zeros(16), SimpleNamespace(dim=2), ws[0], ws[1], ws[2])


def test_bad_widths_raise():
    from mfm_b200 import exe_flow_matching as E
    with pytest.raises(ValueError):
        E.VectorFieldNet(torch.zeros(16), SimpleNamespace(dim=2), [64, 0], [64, 64], [64, 64])
    with pytest.raises(ValueError, match="widest"):
        E.VectorFieldParams(2, 64, 16, "cpu", widths=((32, 32), (128, 64), (64, 64)))


def test_oracle_algebra_for_unequal_widths():
    """The float64 oracle the GPU tests compare with, on an unequal network: its FM gradient against central differences of its
    loss, and its exact divergence against the trace of a finite-difference Jacobian of its field."""
    rng = np.random.default_rng(4)
    d, F = 2, 8
    w = ((5, 7), (6, 4), (9, 3))
    params = init_params_widths(rng, d, w, F, head_scale=0.5, dtype=np.float64)
    omega = rng.standard_normal(F)
    ot = OT.four_mode()
    x = rng.standard_normal((4, d)); t = rng.uniform(size=4); tgt = rng.standard_normal((4, d))
    act = "tanh"                                   # smooth: finite differences are exact to O(h^2)
    loss, g = VF.fm_loss_and_grad(params, omega, x, t, tgt, ot.grad, act=act)
    h = 1e-6
    for i in range(8):
        for k in ("kernel", "bias"):
            a = params["params"][f"Dense_{i}"][k]
            assert g["params"][f"Dense_{i}"][k].shape == a.shape
            idx = tuple(rng.integers(0, s) for s in a.shape)
            old = a[idx]
            a[idx] = old + h; lp, _ = VF.fm_loss_and_grad(params, omega, x, t, tgt, ot.grad, act=act)
            a[idx] = old - h; lm, _ = VF.fm_loss_and_grad(params, omega, x, t, tgt, ot.grad, act=act)
            a[idx] = old
            assert abs((lp - lm) / (2 * h) - g["params"][f"Dense_{i}"][k][idx]) <= 1e-6 * max(1.0, abs(loss)), (i, k)
    v, div = VF.field_and_div(params, omega, x, t, ot, act=act)
    tr = np.zeros(x.shape[0])
    for j in range(d):
        e = np.zeros_like(x); e[:, j] = h
        vp = VF.forward(params, omega, x + e, t, ot.grad, act=act); vm = VF.forward(params, omega, x - e, t, ot.grad, act=act)
        tr += (vp - vm)[:, j] / (2 * h)
    assert np.allclose(div, tr, rtol=1e-6, atol=1e-7)
