"""What a narrower time branch (--hidden_t 256 256) saves at the pines-scaling shape (65536 chains, d = 1600, F = 128).

Three networks, all relu with grad_clip 1 and the Hutchinson divergence, as bench.py's default configuration:
  default   : --hidden_t / --hidden_x / --hidden_xt all [1024, 1024] (the equal-width descriptor, zero width tail);
  explicit  : the same widths passed through the width tail of the descriptor (must time as `default`: the same kernels run);
  narrow_t  : --hidden_t 256 256, the x and joint branches [1024, 1024].
It times the FM update's loss and gradient (mfm_fm_loss_grad) and one random-walk flow-MH iteration (two adaptive ODE solves
with the divergence), the variants interleaved in one process after a warm-up, with CUDA events over windows of at least
--window seconds per variant; the per-call median of the windows is reported, next to the forward MACs per sample.  The GPU's
name, power limit and maximum SM clock are read with a read-only nvidia-smi query.

    python scripts/hidden_widths_bench.py --out profiles/r03_hidden_widths_bench.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N, D, F = 65536, 1600, 128
VARIANTS = {   # name: (hidden_t, hidden_x, hidden_xt, pass the widths explicitly)
    "default": ([1024, 1024], [1024, 1024], [1024, 1024], False),
    "explicit": ([1024, 1024], [1024, 1024], [1024, 1024], True),
    "narrow_t": ([256, 256], [1024, 1024], [1024, 1024], True),
}


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True, check=True)
    name, power, clock = [v.strip() for v in out.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "clocks_max_sm": clock}


def args_ns():
    return SimpleNamespace(ref_dist="stdgauss", cond_flow=True, ot_cond_flow=False, sigma=1e-4, adam_beta1=0.9, adam_beta2=0.999,
                           adam_epsilon=1e-8, weight_decay=1e-4, gradient_clip=1.0, hutchs=True, num_importance_samples=0,
                           mcmc_per_flow_steps=10, step_size=1e-4)


def forward_macs(shapes):
    return int(sum(fi * fo for fi, fo in shapes))


def setup(dev):
    import torch
    from mfm_b200 import distributions as Dm, exe_flow_matching as E, random as mr
    dist = Dm.LogGaussianCoxPines(D, device=dev)
    rng = np.random.default_rng(0)
    omega = torch.from_numpy(rng.standard_normal(F).astype(np.float32)).to(dev)
    opts = SimpleNamespace(rtol=1e-5, atol=1e-5, mxstep=1000, n_times=2)
    x = (dist._mu_zero + torch.from_numpy(rng.standard_normal((N, D)).astype(np.float32)).to(dev)).contiguous()
    out = {}
    P_default = None
    for name, (ht, hx, hxt, explicit) in VARIANTS.items():
        model = E.VectorFieldNet(omega, dist, hx, ht, hxt, "relu", 1.0)
        if name == "default":
            P = P_default = model.init(mr.PRNGKey(0, dev), head_scale=0.1)
        elif name == "explicit":
            # the same parameters in a buffer laid out from explicit widths (identical offsets)
            P = E.VectorFieldParams(D, model.hidden, F, dev, widths=model.widths)
            P.flat.copy_(P_default.flat)
        else:
            P = model.init(mr.PRNGKey(0, dev), head_scale=0.1)
        if explicit:
            # field_desc leaves the tail zero when the widths are equal: this variant always fills it
            model.field_desc = (lambda P_, flat=None, m=model, f=model.field_desc: _fill_tail(f(P_, flat), m.widths))
        state = E.create_train_state(model, P, E.create_learning_rate_fn(1000, 0, 1e-3), args_ns())
        gen, init_fn, _ = E.create_train_data_gn(dist, model, opts, args_ns())
        out[name] = SimpleNamespace(model=model, P=P, state=state, gen=gen, st=init_fn(x.clone(), 1.0), macs=forward_macs(P.shapes))
    keys = mr.split(mr.PRNGKey(1, dev), 64)
    return SimpleNamespace(dist=dist, x=x, keys=keys, variants=out)


def _fill_tail(fd, widths):
    (fd.hidden_t[0], fd.hidden_t[1]), (fd.hidden_x[0], fd.hidden_x[1]), (fd.hidden_xt[0], fd.hidden_xt[1]) = widths
    return fd


def time_calls(fn, calls):
    import torch
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for i in range(calls):
        fn(i)
    e.record()
    e.synchronize()
    return s.elapsed_time(e) / calls                                   # ms per call


def interleaved(fns, window_s, warm, rounds):
    import torch
    for fn in fns.values():                                            # warm-up (module load, workspaces, weight mirrors)
        for i in range(warm):
            fn(i)
    torch.cuda.synchronize()
    probe = max(time_calls(fns["default"], warm), 1e-3)
    calls = max(2, int(window_s / rounds * 1e3 / probe))
    res = {r: [] for r in fns}
    for _ in range(rounds):
        for r, fn in fns.items():
            res[r].append(time_calls(fn, calls))
    return {r: dict(ms_per_call_median=float(np.median(v)), ms_per_call_windows=[float(t) for t in v], calls_per_window=calls)
            for r, v in res.items()}


def main():
    p = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_hidden_widths_bench.json"))
    p.add_argument("--window", type=float, default=3.0, help="seconds of timed work per variant and workload")
    a = p.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("hidden_widths_bench.py measures on a CUDA device; none found")
    from mfm_b200 import _build, _lib
    _build.build()
    lib = _lib.load()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    S = setup(dev)
    V = S.variants
    result = {"gpu": gpu_info(), "gemm": lib.mfm_gemm_describe().decode(), "chains": N, "d": D, "fourier_dim": F,
              "window_s_per_variant": a.window,
              "variants": {k: {"hidden_t": v[0], "hidden_x": v[1], "hidden_xt": v[2], "width_tail": v[3],
                               "forward_macs_per_sample": V[k].macs} for k, v in VARIANTS.items()}}
    fm = {r: (lambda i, v=v: v.state.loss_and_grad(S.keys[i % 64], S.x)) for r, v in V.items()}
    result["fm_loss_grad"] = interleaved(fm, a.window, 3, 5)
    print("fm_loss_grad", json.dumps(result["fm_loss_grad"]), flush=True)
    lp = S.dist.tempered(1.0)
    mh = {r: (lambda i, v=v: v.gen.flow_step(S.keys[i % 64], v.st, lp, v.P)) for r, v in V.items()}
    result["rw_flow_mh_step"] = interleaved(mh, a.window, 2, 3)
    print("rw_flow_mh_step", json.dumps(result["rw_flow_mh_step"]), flush=True)
    base_macs = V["default"].macs
    summary = {}
    for wl in ("fm_loss_grad", "rw_flow_mh_step"):
        b = result[wl]["default"]["ms_per_call_median"]
        summary[wl] = {k: 100.0 * (b - result[wl][k]["ms_per_call_median"]) / b for k in ("explicit", "narrow_t")}
    summary["forward_macs_saved_pct"] = 100.0 * (base_macs - V["narrow_t"].macs) / base_macs
    result["saving_vs_default_pct"] = summary
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps({"gpu": result["gpu"], "saving_vs_default_pct": summary}))


if __name__ == "__main__":
    main()
