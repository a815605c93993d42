"""PhiFourBase as the flow's reference distribution (ref_dist='phifour'): the host band factor, the log-density constant, the
descriptor layout and the registry.  CPU only; the device kernels are checked in tests/test_gpu_ref_dist.py."""
import ctypes
import os
import subprocess
import tempfile
import textwrap

import numpy as np
import pytest
import scipy.linalg

from oracle import targets as OT

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bidiag(l, s):
    return np.diag(l) + np.diag(s[1:], -1)


@pytest.mark.parametrize("d", [2, 16, 64, 1600])
def test_band_factor_matches_oracle(d):
    from mfm_b200.distributions import phi_four_base_band
    ref = OT.PhiFourBase(d)
    l, s, log_norm = phi_four_base_band(d)
    assert s[0] == 0.0 and (l > 0).all()
    L = _bidiag(l, s)
    assert np.abs(L @ L.T - ref.prec).max() <= 1e-10 * np.abs(ref.prec).max()
    chol_cov = scipy.linalg.solve_triangular(L, np.eye(d), lower=True).T            # L^-T
    assert np.abs(chol_cov - ref.chol_cov).max() <= 1e-10 * np.abs(ref.chol_cov).max()
    const = -0.5 * (d * np.log(2 * np.pi) + ref.prior_log_det)
    assert abs(log_norm - const) <= 1e-10 * abs(const)


@pytest.mark.parametrize("d,alpha,beta", [(3, 0.1, 20.0), (64, 0.1, 20.0), (40, 0.3, 2.0)])
def test_sum_of_squares_form_and_back_substitution(d, alpha, beta):
    """The two O(d) row operations the kernels run, restated in float64: the sum-of-squares log-density with the weights stored
    behind the band (beta c, beta / c) equals the oracle's, and the back-substitution x_i = a_i x_{i+1} + z_i / l_i with
    a_i = -s_{i+1} / l_i is sample_model's chol_cov @ z."""
    from mfm_b200.distributions import phi_four_base_band
    ref = OT.PhiFourBase(d, alpha, beta)
    l, s, log_norm = phi_four_base_band(d, alpha, beta)
    c = alpha * d
    x = np.random.default_rng(1).standard_normal((7, d))
    xp = np.pad(x, ((0, 0), (1, 1)))
    q = beta * c * (np.diff(xp, axis=1) ** 2).sum(1) + beta / c * (x ** 2).sum(1)
    assert np.allclose(-0.5 * q + log_norm, ref.loglik(x), rtol=1e-12, atol=1e-10)
    z = np.random.default_rng(2).standard_normal((5, d))
    xs = np.zeros_like(z)
    a = np.zeros(d)
    a[:-1] = -s[1:] / l[:-1]
    for r in range(z.shape[0]):
        nxt = 0.0
        for i in range(d - 1, -1, -1):
            nxt = a[i] * nxt + z[r, i] / l[i]
            xs[r, i] = nxt
    assert np.allclose(xs, z @ ref.chol_cov.T, rtol=1e-12, atol=1e-12)


def test_field_descriptor_offsets_match_header():
    from mfm_b200 import _lib
    code = textwrap.dedent("""
        #include <stdio.h>
        #include <stddef.h>
        #include "mfm_b200.h"
        int main(){ printf("%zu %zu %zu %zu %zu %d %d %d\\n", sizeof(mfm_field_t), offsetof(mfm_field_t, act),
                           offsetof(mfm_field_t, ref_kind), offsetof(mfm_field_t, ref_log_norm), offsetof(mfm_field_t, ref_band),
                           MFM_REF_INDEP_GAUSS, MFM_REF_PHI4_BASE, MFM_REF_BAND_MAX_DIM); return 0; }
    """)
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "t.c"); exe = os.path.join(d, "t")
        open(c, "w").write(code)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        out = [int(v) for v in subprocess.check_output([exe]).decode().split()]
    F = _lib.FieldDesc
    assert out[:5] == [ctypes.sizeof(F), F.act.offset, F.ref_kind.offset, F.ref_log_norm.offset, F.ref_band.offset]
    assert out[5:] == [_lib.REF_INDEP_GAUSS, _lib.REF_PHI4_BASE, _lib.REF_BAND_MAX_DIM]
    # the new fields follow `act`: every older offset is unchanged, and a zero-filled tail means IndepGaussian(ref_mean, ref_std)
    assert F.ref_kind.offset > F.act.offset and _lib.REF_INDEP_GAUSS == 0


def test_phifour_is_registered():
    from mfm_b200 import exe_flow_matching as E
    from mfm_b200.distributions import PhiFourBase
    assert "phifour" in E.ref_dists
    ref = E.ref_dists["phifour"](64, device="cpu")
    assert isinstance(ref, PhiFourBase) and ref.dim == 64 and (ref.alpha, ref.beta) == (0.1, 20.0)
    band = ref.band.numpy().astype(np.float64)
    assert band.shape == (2 * 64 + 2,) and band[63] == 0.0
    assert np.allclose(band[:63], -ref.s[1:] / ref.l[:-1], rtol=1e-7) and np.allclose(band[64:128], 1.0 / ref.l, rtol=1e-7)
    assert np.isclose(band[-2], 20.0 * 6.4) and np.isclose(band[-1], 20.0 / 6.4)


def test_coupled_pbc_raises():
    from mfm_b200.distributions import PhiFourBase
    with pytest.raises(NotImplementedError, match="coupled_pbc"):
        PhiFourBase(16, prior_type="coupled_pbc", device="cpu")
    with pytest.raises(ValueError):
        PhiFourBase(16, prior_type="independent", device="cpu")


def test_reference_only():
    from mfm_b200.distributions import PhiFourBase
    ref = PhiFourBase(8, device="cpu")
    with pytest.raises(NotImplementedError, match="reference distribution only"):
        ref.tempered(1.0)
    with pytest.raises(NotImplementedError, match="reference distribution only"):
        ref._desc(1.0)
