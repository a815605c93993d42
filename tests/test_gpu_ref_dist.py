"""The PhiFourBase reference distribution (ref_dist='phifour', distributions.py:168-226) on the device, against the float64 oracle
oracle.targets.PhiFourBase: mfm_ref_sample / mfm_ref_logprob, the conditional FM batch, the independent flow-MH step, conditional
importance sampling and sample_flow; and bit-identity of everything that does not read the reference distribution."""
import zlib
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import resample as OR, samplers as OS, targets as OT, threefry as tf, vector_field as VF
from tests.helpers import key_dev, make_targets, rel_err, to_dev
from tests.test_gpu_flow import CFG, HEAD_SCALE, _flow, _tol

pytestmark = pytest.mark.gpu


class Ref64(OT.PhiFourBase):
    """The oracle PhiFourBase with its sample_model product in float64 (the draws keep the requested dtype)."""

    def sample(self, keys, dtype=np.float32):
        return tf.vmap_normal(keys, self.dim, dtype).astype(np.float64) @ self.chol_cov.T


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _fm_args(ref_dist="phifour", cond_flow=True):
    return SimpleNamespace(ref_dist=ref_dist, cond_flow=cond_flow, ot_cond_flow=False, sigma=1e-4, adam_beta1=0.9, adam_beta2=0.999,
                           adam_epsilon=1e-8, weight_decay=1e-4, gradient_clip=1.0)


@pytest.fixture(scope="module")
def setups(cuda, lib):
    """test_gpu_flow's configurations (same parameters) with a PhiFourBase reference distribution."""
    from mfm_b200 import distributions as D, exe_flow_matching as E
    out = {}
    for name, ot, dd in make_targets(cuda):
        H, hutch, n_times, clip, n = CFG[name]
        rng = np.random.default_rng(zlib.crc32(name.encode()) % 1000)
        params = VF.init_params(rng, ot.dim, H, 128, head_scale=HEAD_SCALE[name])
        if name == "phi-four":
            params["params"]["Dense_4"]["bias"] = (np.abs(params["params"]["Dense_4"]["bias"]) * 0.2).astype(np.float32)
        omega = rng.standard_normal(128).astype(np.float32)
        model = E.VectorFieldNet(to_dev(omega, cuda), dd, [H, H], [H, H], [H, H], "relu", clip)
        P = E.VectorFieldParams(ot.dim, H, 128, cuda).load_dict(params)
        out[name] = SimpleNamespace(ot=ot, dd=dd, params=params, omega=omega, model=model, P=P, hutch=hutch, n_times=n_times,
                                    clip=clip, n=n, ref=Ref64(ot.dim), ref_d=D.PhiFourBase(ot.dim, device=cuda))
    return out


def _gn(s, nis, ref_dist="phifour"):
    from mfm_b200 import exe_flow_matching as E
    args = SimpleNamespace(hutchs=s.hutch, num_importance_samples=nis, mcmc_per_flow_steps=10, step_size=0.1, ref_dist=ref_dist)
    opts = SimpleNamespace(rtol=1e-5, atol=1e-5, mxstep=1000, n_times=s.n_times)
    return E.create_train_data_gn(s.dd, s.model, opts, args)


# ---- mfm_ref_sample / mfm_ref_logprob -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d", [2, 16, 64, 1600])
def test_ref_sample_matches_oracle(cuda, lib, d):
    from mfm_b200 import distributions as D
    ref_d, ref = D.PhiFourBase(d, device=cuda), Ref64(d)
    n = 64 if d == 1600 else 256
    keys = tf.split(tf.PRNGKey(d), n)
    x = ref_d.sample_model(key_dev(keys, cuda)).cpu().numpy().astype(np.float64)
    x_ref = ref.sample(keys, np.float32)
    err = np.abs(x - x_ref).max(1) / np.abs(x_ref).max(1)
    assert err.max() <= 1e-5, (d, err.max())
    one = ref_d.sample_model(key_dev(keys[3], cuda)).cpu().numpy()            # a single uint32[2] key
    assert np.array_equal(one, x[3].astype(np.float32))


def test_ref_sample_x64_layout(cuda, lib):
    from mfm_b200 import distributions as D
    d, n = 64, 128
    ref_d, ref = D.PhiFourBase(d, device=cuda), Ref64(d)
    keys = tf.split(tf.PRNGKey(9), n)
    lib.mfm_set_rng_x64(1)
    try:
        x = ref_d.sample_model(key_dev(keys, cuda)).cpu().numpy().astype(np.float64)
    finally:
        lib.mfm_set_rng_x64(0)
    x_ref = ref.sample(keys, np.float64)
    assert (np.abs(x - x_ref).max(1) / np.abs(x_ref).max(1)).max() <= 1e-5


@pytest.mark.parametrize("var", [1.0, 5.0])
def test_ref_sample_indep_gauss_is_bit_identical(cuda, lib, var):
    """ref_kind 0 through mfm_ref_sample reproduces IndepGaussian.sample_model (stdgauss, widegauss) bit for bit."""
    from mfm_b200 import _lib, distributions as D
    d, n = 64, 200
    g = D.IndepGaussian(d, var=var, device=cuda)
    keys = key_dev(tf.split(tf.PRNGKey(4), n), cuda)
    fd = _lib.FieldDesc()
    fd.dim = d
    g._fill_ref(fd)
    out = torch.empty(n, d, dtype=torch.float32, device=cuda)
    _lib.check(lib.mfm_ref_sample(fd, keys.data_ptr(), n, out.data_ptr(), _stream()))
    assert torch.equal(out, g.sample_model(keys))


@pytest.mark.parametrize("d", [2, 16, 64, 1600])
def test_ref_logprob_matches_oracle(cuda, lib, d):
    from mfm_b200 import distributions as D
    ref_d, ref = D.PhiFourBase(d, device=cuda), Ref64(d)
    n = 256
    samples = ref_d.sample_model(key_dev(tf.split(tf.PRNGKey(d + 1), n), cuda))
    init = to_dev(np.random.default_rng(d).uniform(-1.0, 1.0, (n, d)), cuda)         # phi-four initial positions
    for x in (samples, init):
        got = ref_d.logprob(x).cpu().numpy().astype(np.float64)
        x64 = x.cpu().numpy().astype(np.float64)
        exp = ref.loglik(x64)
        half_q = np.abs(0.5 * np.einsum("ni,ij,nj->n", x64, ref.prec, x64))
        tol = 1e-5 * (half_q + abs(ref_d.log_norm)) + 1e-6
        assert (np.abs(got - exp) <= tol).all(), (d, np.max(np.abs(got - exp) / tol))
    assert torch.equal(ref_d.loglik(init), ref_d.logprob(init)) and (ref_d.logprior(init) == 0).all()
    assert ref_d.logprob(init[5]).item() == ref_d.logprob(init)[5].item()


def test_error_paths(cuda, lib):
    from mfm_b200 import _lib, distributions as D
    ref_d = D.PhiFourBase(16, device=cuda)
    x = torch.zeros(4, 16, device=cuda)
    out = torch.empty(4, device=cuda)
    keys = key_dev(tf.split(tf.PRNGKey(0), 4), cuda)
    fd = ref_d._ref_desc()
    fd.ref_kind = 7
    assert lib.mfm_ref_logprob(fd, 4, x.data_ptr(), out.data_ptr(), _stream()) == -1          # MFM_ERR_ARG
    assert lib.mfm_ref_sample(fd, keys.data_ptr(), 4, x.data_ptr(), _stream()) == -1
    assert b"ref_kind" in lib.mfm_last_error()
    fd = ref_d._ref_desc()
    fd.ref_band = None
    assert lib.mfm_ref_logprob(fd, 4, x.data_ptr(), out.data_ptr(), _stream()) == -1
    assert b"ref_band" in lib.mfm_last_error()
    fd = ref_d._ref_desc()
    fd.ref_log_norm = float("nan")
    assert lib.mfm_ref_sample(fd, keys.data_ptr(), 4, x.data_ptr(), _stream()) == -1
    fd = ref_d._ref_desc()
    fd.dim = _lib.REF_BAND_MAX_DIM + 1
    assert lib.mfm_ref_sample(fd, keys.data_ptr(), 1, x.data_ptr(), _stream()) == -4            # MFM_ERR_UNSUPPORTED
    fd = _lib.FieldDesc()
    fd.dim = 16
    assert lib.mfm_ref_logprob(fd, 4, x.data_ptr(), out.data_ptr(), _stream()) == -1           # kind 0 with ref_std 0
    assert b"ref_std must be > 0" in lib.mfm_last_error()


# ---- conditional FM batch --------------------------------------------------------------------------------------------------------
def _flat_grads(P, G):
    out = np.zeros(P.n_params)
    for i in range(8):
        k, b = G["params"][f"Dense_{i}"]["kernel"].ravel(), G["params"][f"Dense_{i}"]["bias"].ravel()
        out[P.w_off[i]:P.w_off[i] + k.size] = k
        out[P.b_off[i]:P.b_off[i] + b.size] = b
    return out


def _fm_errors(cuda, s, n, ref_dist="phifour", rng_dtype=np.float32):
    """(loss error, gradient error, per-layer kernel / bias gradient errors) of one FM update against the float64 oracle."""
    from mfm_b200 import exe_flow_matching as E
    state = E.create_train_state(s.model, s.P, E.create_learning_rate_fn(1000, 0, 1e-3), _fm_args(ref_dist))
    x = s.ot.init_positions(tf.PRNGKey(8), n, np.float32).astype(np.float64)
    key = tf.PRNGKey(31337)
    sampler = s.ref.sample if ref_dist == "phifour" else OT.IndepGaussian(s.ot.dim).sample
    times, xt, target = VF.fm_batch(key, x, sampler, 1e-4, rng_dtype=rng_dtype)
    loss_ref, G = VF.fm_loss_and_grad(s.params, s.omega, xt, times, target, s.ot.grad, s.clip)
    loss, grads = state.loss_and_grad(key_dev(key, cuda), to_dev(x, cuda))
    g_ref, g = _flat_grads(s.P, G), grads.cpu().numpy()
    layers = []
    for i in range(8):
        fi, fo = s.P.shapes[i]
        w, b = slice(s.P.w_off[i], s.P.w_off[i] + fi * fo), slice(s.P.b_off[i], s.P.b_off[i] + fo)
        layers.append((rel_err(g[w], g_ref[w]), rel_err(g[b], g_ref[b])))
    return abs(loss.item() - loss_ref) / abs(loss_ref), rel_err(g, g_ref), layers


def _fm_check(cuda, s, n, rng_dtype=np.float32, layer_tol=None):
    loss_err, grad_err, layers = _fm_errors(cuda, s, n, rng_dtype=rng_dtype)
    assert loss_err < 1e-4 and grad_err < 2e-4, (loss_err, grad_err)
    for i, (ew, eb) in enumerate(layers):
        tol = 5e-4 if layer_tol is None else layer_tol[i]
        assert ew < tol[0] if isinstance(tol, tuple) else ew < tol, (i, ew, tol)
        assert eb < tol[1] if isinstance(tol, tuple) else eb < tol, ("bias", i, eb, tol)


@pytest.mark.parametrize("name,n", [("phi-four", 300), ("gmm16", 77)])
def test_fm_loss_and_grad_phifour_ref(cuda, setups, name, n):
    _fm_check(cuda, setups[name], n)


def test_fm_loss_and_grad_phifour_ref_pines(cuda, setups):
    """pines at 300 rows (the scaled-fp16 GEMMs, H = 1024).  Loss and whole gradient to the usual 1e-4 / 2e-4; per layer, 5e-4
    or - where the same update with stdgauss is itself further from the oracle at this shape (the time branch's weight gradient,
    a sum over rows with cancellation) - no more than twice the stdgauss error."""
    s = setups["pines"]
    _, _, base = _fm_errors(cuda, s, 300, ref_dist="stdgauss")
    _fm_check(cuda, s, 300, layer_tol=[(max(5e-4, 2 * ew), max(5e-4, 2 * eb)) for ew, eb in base])


def test_fm_loss_and_grad_phifour_ref_scaled_fp16(cuda, lib, setups):
    """The narrow phi-four network forced onto the scaled-fp16 GEMMs: their operand scales come from the maxima of x_t and of
    the targets that the PhiFourBase batch kernel publishes."""
    lib.mfm_debug_set_h16_min_hidden(0)
    try:
        _fm_check(cuda, setups["phi-four"], 300)
    finally:
        lib.mfm_debug_set_h16_min_hidden(-1)


def test_fm_loss_and_grad_phifour_ref_x64(cuda, lib, setups):
    lib.mfm_set_rng_x64(1)
    try:
        _fm_check(cuda, setups["phi-four"], 300, rng_dtype=np.float64)
    finally:
        lib.mfm_set_rng_x64(0)


def test_fm_sharded_batch_phifour_ref(cuda, setups):
    from mfm_b200 import exe_flow_matching as E
    s = setups["phi-four"]
    state = E.create_train_state(s.model, s.P, E.create_learning_rate_fn(1000, 0, 1e-3), _fm_args())
    n = 96
    x = to_dev(s.ot.init_positions(tf.PRNGKey(8), n, np.float32), cuda)
    key = key_dev(tf.PRNGKey(5), cuda)
    loss, grads = state.loss_and_grad(key, x)
    loss, grads = loss.clone(), grads.clone()
    tot_l, tot_g = 0.0, torch.zeros_like(grads)
    for lo, hi in ((0, 32), (32, 96)):
        l, g = state.loss_and_grad(key, x[lo:hi].contiguous(), chain_offset=lo, n_total=n)
        tot_l += l.item(); tot_g += g
    assert abs(tot_l - loss.item()) < 1e-5 * abs(loss.item())
    assert rel_err(tot_g.cpu().numpy(), grads.cpu().numpy()) < 1e-5


# ---- flow steps and final sampling -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["phi-four", "gmm16"])
def test_indep_flow_mh_step_phifour_ref(cuda, setups, name):
    """independent flow-MH (num_importance_samples < 0, :246-260) with the PhiFourBase proposal: test_flow_mh_step's criteria."""
    s = setups[name]
    n = s.n
    gen, init_fn, _ = _gn(s, -1)
    flow = _flow(s)
    x0 = s.ot.init_positions(tf.PRNGKey(3), n, np.float32).astype(np.float64)
    beta = 0.7
    st_d = init_fn(to_dev(x0, cuda), beta)
    st_o = OS.mala_init(x0, s.ot, beta)
    key = tf.PRNGKey(2024)
    keys = tf.split(key, n)
    dbg, dbg32 = {}, {}
    st_o32 = OS.MALAState(*[a.astype(np.float32) for a in st_o])
    new_o, info_o = OS.indep_flow_mh_step(keys, st_o, s.ot, flow, s.ref, beta, dbg)
    _, info_32 = OS.indep_flow_mh_step(keys, st_o32, s.ot, flow, OT.PhiFourBase(s.ot.dim), beta, dbg32)
    new_d, info_d = gen.flow_step(key_dev(key, cuda), st_d, s.dd.tempered(beta), s.P)
    la, la32 = dbg["log_acc"], dbg32["log_acc"].astype(np.float64)
    err, tol = _tol(info_d.proposed_position.cpu().numpy(), info_o.proposed_position, info_32.proposed_position, 2e-3)
    assert err < tol, (name, err, tol)
    l_mag = np.maximum(np.abs(st_o.logdensity), np.abs(dbg["lp"]))
    ulp = np.spacing(np.maximum(l_mag, 1.0).astype(np.float32)).astype(np.float64)
    fin32 = np.isfinite(la) & np.isfinite(la32) & (np.abs(la) < 80)
    la_tol = np.maximum(1e-3, 4.0 * ulp) + 4.0 * (np.abs(la32 - la)[fin32].max() if fin32.any() else 0.0)
    with np.errstate(over="ignore", divide="ignore"):
        la_d = np.log(info_d.acceptance_rate.cpu().numpy().astype(np.float64))
        logu = np.log(dbg["u"])
    fin = np.isfinite(la) & np.isfinite(la_d) & (np.abs(la) < 80)
    la_err = np.abs(la_d[fin] - la[fin])
    if name == "phi-four":
        e32 = np.abs(la32 - la)[fin32]
        if la_err.size:
            assert np.median(la_err) <= 3.0 * np.median(e32) + 5e-3, (np.median(la_err), np.median(e32))
            assert la_err.max() <= 10.0 * e32.max() + 5e-2, (la_err.max(), e32.max())
        la_tol = np.maximum(la_tol, np.abs(la_d - la) + 1e-6)
    else:
        assert (la_err < la_tol[fin]).all(), (la_err.max(), la_tol[fin][np.argmax(la_err - la_tol[fin])])
    acc_d, acc_o = info_d.is_accepted.cpu().numpy(), info_o.is_accepted
    band = np.abs(la - logu) < la_tol
    assert ((acc_d == acc_o) | band).all(), name
    same = acc_d == acc_o
    err, tol = _tol(new_d.position.cpu().numpy()[same], new_o.position[same], new_o.position[same].astype(np.float32), tol)
    assert err < tol
    assert (info_d.proposed_weight == 0).all()


@pytest.mark.parametrize("name,K", [("gmm16", 4), ("4-mode", 3)])
def test_cis_flow_step_phifour_ref(cuda, setups, name, K):
    """conditional importance sampling (:280-296) with K PhiFourBase reference samples per chain: test_cis_flow_step's criteria."""
    s = setups[name]
    n = s.n
    gen, init_fn, _ = _gn(s, K)
    flow = _flow(s)
    # states the flow maps PhiFourBase's typical set to: from init_positions the pulled-back states lie far outside the narrow
    # reference (d = 2: standard deviations ~0.1), their weights exp(l - logq(u) - V) reach 1e130 and overflow float32
    u0 = s.ref.sample(tf.split(tf.PRNGKey(6), n), np.float32)
    x0, _ = flow.transform_and_logdet(tf.split(tf.PRNGKey(12), n), u0)
    x0 = x0.astype(np.float32).astype(np.float64)
    beta = 0.8
    st_d = init_fn(to_dev(x0, cuda), beta)
    st_o = OS.mala_init(x0, s.ot, beta)
    key = tf.PRNGKey(77)
    new_o, info_o = OS.cis_flow_step(tf.split(key, n), st_o, s.ot, flow, s.ref, K, beta)
    new_d, info_d = gen.flow_step(key_dev(key, cuda), st_d, s.dd.tempered(beta), s.P)
    acc_d, acc_o = info_d.is_accepted.cpu().numpy(), info_o.is_accepted
    w_d, w_o = info_d.acceptance_rate.cpu().numpy().astype(np.float64), info_o.acceptance_rate
    same = (acc_d == acc_o) & (np.abs(w_d - w_o) <= 2e-2 * np.maximum(w_o, 1e-6))
    assert same.sum() >= n - 1, (name, same.sum(), n)
    assert np.allclose(w_d[same], w_o[same], rtol=2e-2)
    assert torch.equal(info_d.proposed_weight, info_d.acceptance_rate)
    err, tol = _tol(new_d.position.cpu().numpy()[same], new_o.position[same], new_o.position[same].astype(np.float32), 2e-3)
    assert err < tol, (name, err, tol)
    ld, lo = new_d.logdensity.cpu().numpy()[same], new_o.logdensity[same]
    assert np.abs(ld - lo).max() <= 2e-3 * max(np.abs(lo).max(), 1.0)
    assert torch.equal(new_d.logdensity_grad, st_d.logdensity_grad)


@pytest.mark.parametrize("hutch", [False, True])
def test_sample_flow_phifour_ref(cuda, lib, hutch):
    """sample_flow (:453-459) with u ~ PhiFourBase and ref_dist.logprob(u) in the weights, against OR.sample_flow."""
    from mfm_b200 import distributions as D, exe_flow_matching as E
    ot = OT.four_mode()
    dd = D.GaussianMixture(ot.modes, ot.covs, ot.weights, device=cuda)
    H, n = 128, 96
    rng = np.random.default_rng(7)
    params = VF.init_params(rng, 2, H, 128, head_scale=0.2)
    omega = rng.standard_normal(128).astype(np.float32)
    model = E.VectorFieldNet(to_dev(omega, cuda), dd, [H, H], [H, H], [H, H], "relu", None)
    P = E.VectorFieldParams(2, H, 128, cuda).load_dict(params)
    args = SimpleNamespace(hutchs=hutch, num_importance_samples=0, mcmc_per_flow_steps=10, step_size=0.2, ref_dist="phifour")
    opts = SimpleNamespace(rtol=1e-5, atol=1e-5, mxstep=1000, n_times=5)
    _, _, transform_and_logdet = E.create_train_data_gn(dd, model, opts, args)
    ref_d = E.ref_dists["phifour"](2, device=cuda)
    key = tf.PRNGKey(3)
    got = E.sample_flow(key_dev(key, cuda), dd, ref_d, transform_and_logdet, P, n)
    flow = OS.Flow(params, omega, ot, hutch, 1e-5, 1e-5, 1000, None, tuple(np.linspace(0, 1, 5)), rng_dtype=np.float32)
    ref = OR.sample_flow(key, ot, Ref64(2), flow, n)
    u = got["u"].cpu().numpy()
    assert np.abs(u - ref["u"]).max() <= 1e-5 * np.abs(ref["u"]).max()
    fs = got["flow_samples"].cpu().numpy()
    assert np.abs(fs - ref["flow_samples"]).max() <= 5e-3 * np.abs(ref["flow_samples"]).max()
    lw, lw_ref = got["log_weights"].cpu().numpy(), ref["log_weights"]
    fin = np.isfinite(lw_ref)
    assert (np.isfinite(lw) == fin).all()
    assert np.abs(lw[fin] - lw_ref[fin]).max() <= 0.05 + 2e-3 * np.abs(lw_ref[fin]).max()
    idx_same_w, _ = OR.choice_indices(tf.split(key)[1], n, n, got["weights"].cpu().numpy())
    idx = got["indices"].cpu().numpy()
    assert np.array_equal(idx, idx_same_w)
    assert (idx == ref["indices"]).mean() >= 0.9
    assert np.array_equal(got["exact_samples"].cpu().numpy(), fs[idx])


# ---- where the reference distribution is not read: bit-identical whatever ref_dist is ---------------------------------------------
def test_rw_flow_mh_and_uncond_fm_ignore_ref_dist(cuda, lib, setups):
    from mfm_b200 import exe_flow_matching as E
    s = setups["phi-four"]
    x0 = to_dev(s.ot.init_positions(tf.PRNGKey(3), s.n, np.float32), cuda)
    key = key_dev(tf.PRNGKey(2024), cuda)
    outs = []
    for ref_dist in ("stdgauss", "phifour"):
        gen, init_fn, _ = _gn(s, 0, ref_dist)
        st = init_fn(x0.clone(), 0.7)
        new, info = gen.flow_step(key, st, s.dd.tempered(0.7), s.P)
        outs.append([*new, info.acceptance_rate, info.is_accepted, info.proposed_position])
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    res = []
    x = to_dev(s.ot.init_positions(tf.PRNGKey(8), 200, np.float32), cuda)
    for ref_dist in ("stdgauss", "phifour"):
        state = E.create_train_state(s.model, s.P, E.create_learning_rate_fn(1000, 0, 1e-3), _fm_args(ref_dist, cond_flow=False))
        l0 = lib.mfm_launch_count()
        loss, grads = state.loss_and_grad(key, x)
        res.append((loss.clone(), grads.clone(), lib.mfm_launch_count() - l0))
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1]) and res[0][2] == res[1][2]
    launches = []
    for ref_dist in ("stdgauss", "phifour"):      # the conditional batch: one kernel either way
        state = E.create_train_state(s.model, s.P, E.create_learning_rate_fn(1000, 0, 1e-3), _fm_args(ref_dist))
        l0 = lib.mfm_launch_count()
        state.loss_and_grad(key, x)
        launches.append(lib.mfm_launch_count() - l0)
    assert launches[0] == launches[1]


@pytest.mark.parametrize("name", ["phi-four", "phi-four-1024"])
def test_graph_replayed_iterations_phifour_ref(cuda, lib, name):
    """HotLoop(graph=True) with ref_dist='phifour': the captured MALA + FM iteration (the PhiFourBase batch kernel inside the
    graph) gives bit-identical chains, parameters and losses to the eager loop, flow-MH iterations (eager) included."""
    from mfm_b200 import distributions as Dm, exe_flow_matching as E, random as mr
    d, n, m, step = {"phi-four": (64, 96, 3, 1e-4), "phi-four-1024": (64, 1024, 3, 1e-4)}[name]
    H, F = 128, 128
    args = SimpleNamespace(hutchs=False, num_importance_samples=-1, mcmc_per_flow_steps=m, step_size=step, ref_dist="phifour",
                           cond_flow=True, ot_cond_flow=False, sigma=1e-4, adam_beta1=0.9, adam_beta2=0.999, adam_epsilon=1e-8,
                           weight_decay=1e-4, gradient_clip=1.0, learning_iter=100, warmup_steps=0, learning_rate=1e-3)
    opts = SimpleNamespace(rtol=1e-5, atol=1e-5, mxstep=1000, n_times=2)
    rng = np.random.default_rng(5)
    shapes = [(2 * F, H), (H, H), (d, H), (H, H), (H, d), (2 * H, H), (H, H), (H, d)]
    params = {"params": {f"Dense_{i}": {"kernel": (rng.standard_normal(s) / np.sqrt(s[0]) * (0.002 if i in (4, 7) else 1.0)).astype(np.float32),
                                        "bias": (rng.standard_normal(s[1]) * 0.01).astype(np.float32)} for i, s in enumerate(shapes)}}
    omega = torch.from_numpy(rng.standard_normal(F).astype(np.float32)).to(cuda)
    x0 = torch.from_numpy(rng.uniform(-1, 1, (n, d)).astype(np.float32)).to(cuda)
    out = []
    for graph in (False, True):
        dist = Dm.PhiFour(d, device=cuda)
        model = E.VectorFieldNet(omega, dist, [H, H], [H, H], [H, H], "relu", None)
        P = E.VectorFieldParams(d, H, F, cuda).load_dict(params)
        loop = E.HotLoop(dist, model, P, args, opts, mr.PRNGKey(21, cuda), x0.clone(), graph=graph)
        losses = [float(loop.iteration().item()) for _ in range(3 * (m + 1) + 2)]
        assert (loop._graph is not None) == graph
        out.append((losses, loop.states.position.clone(), loop.states.logdensity.clone(), P.flat.clone(), loop.key_sample.clone(),
                    loop.last_info.acceptance_rate.clone()))
    assert out[0][0] == out[1][0]
    for a, b in zip(out[0][1:], out[1][1:]):
        assert torch.equal(a, b)


def test_run_phi_four_with_phifour_ref(cuda, lib):
    """run() end to end on the phi-four example with --ref_dist phifour and the independent flow-MH step."""
    from mfm_b200 import multi_modal as MM
    from mfm_b200.distributions import PhiFourBase
    args = MM.parser().parse_args(["--example", "phi-four", "--learning_iter", "4", "--mcmc_per_flow_steps", "1", "--seed", "1",
                                   "--ref_dist", "phifour", "--num_importance_samples", "-1", "--log_every", "1"])
    dist = MM.build(args, device=cuda)
    res = MM.run(dist, args, None, log_every=1)
    assert isinstance(res["loop"].state.ref_dist, PhiFourBase)
    assert len(res["history"]) == 4 and all(np.isfinite(h["loss"]) for h in res["history"])
    assert torch.isfinite(res["loop"].states.position).all()
    assert all(np.isfinite(v) for v in res["table"].values()), res["table"]
