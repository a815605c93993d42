"""Cost of the PhiFourBase reference distribution (--ref_dist phifour) against stdgauss on the device.

Times mfm_fm_loss_grad (the FM update's loss and gradient, which draws x0 from the reference distribution once per outer
iteration) with each reference distribution at two shapes: the phi-four configuration (1024 chains, d = 64, H = 128) and the
pines-scaling shape (65536 chains, d = 1600, H = 1024).  The two variants are interleaved in one process after a warm-up, timed
with CUDA events over windows of at least --window seconds per shape and variant; the per-call median of the windows is
reported.  The batch kernels alone (fm_batch_kernel / fm_batch_phi4_kernel) are timed by torch.profiler in a separate pass, and
the independent flow-MH step (num_importance_samples < 0, which draws its proposal from the reference distribution) at the
phi-four shape.  The GPU's name, power limit and maximum SM clock are read with a read-only nvidia-smi query.

    python scripts/ref_dist_bench.py --out profiles/r03_ref_dist_bench.json
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

SHAPES = {
    "phi-four": dict(n=1024, d=64, H=128, clip=None),
    "pines-scaling": dict(n=65536, d=1600, H=1024, clip=1.0),
}
F = 128


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True, check=True)
    name, power, clock = [v.strip() for v in out.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "clocks_max_sm": clock}


def fm_args(ref_dist, nis=0, hutch=False):
    return SimpleNamespace(ref_dist=ref_dist, cond_flow=True, ot_cond_flow=False, sigma=1e-4, adam_beta1=0.9, adam_beta2=0.999,
                           adam_epsilon=1e-8, weight_decay=1e-4, gradient_clip=1.0, hutchs=hutch, num_importance_samples=nis,
                           mcmc_per_flow_steps=10, step_size=1e-4)


def setup(name, dev):
    import torch
    from mfm_b200 import distributions as D, exe_flow_matching as E, random as mr
    c = SHAPES[name]
    n, d, H = c["n"], c["d"], c["H"]
    dist = D.PhiFour(d, device=dev) if name == "phi-four" else D.LogGaussianCoxPines(d, device=dev)
    rng = np.random.default_rng(0)
    omega = torch.from_numpy(rng.standard_normal(F).astype(np.float32)).to(dev)
    variants = {}
    P = None
    for ref in ("stdgauss", "phifour"):
        model = E.VectorFieldNet(omega, dist, [H, H], [H, H], [H, H], "relu", c["clip"])
        if P is None:
            P = model.init(mr.PRNGKey(0, dev), head_scale=0.1)
        state = E.create_train_state(model, P, E.create_learning_rate_fn(1000, 0, 1e-3), fm_args(ref))
        variants[ref] = SimpleNamespace(model=model, state=state)
    x = (torch.from_numpy(rng.uniform(-1.0, 1.0, (n, d)).astype(np.float32)).to(dev) if name == "phi-four"
         else dist._mu_zero + torch.from_numpy(rng.standard_normal((n, d)).astype(np.float32)).to(dev))
    keys = mr.split(mr.PRNGKey(1, dev), 64)
    return SimpleNamespace(dist=dist, P=P, x=x.contiguous(), keys=keys, variants=variants, n=n, d=d, H=H)


def time_calls(fn, calls):
    import torch
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for i in range(calls):
        fn(i)
    e.record()
    e.synchronize()
    return s.elapsed_time(e) / calls                                   # ms per call


def bench_fm(S, window_s):
    """Interleaved windows: stdgauss, phifour, stdgauss, ... each of at least window_s / rounds seconds."""
    import torch
    fns = {r: (lambda i, v=v: v.state.loss_and_grad(S.keys[i % 64], S.x)) for r, v in S.variants.items()}
    for r, fn in fns.items():                                          # warm-up (module load, workspace, weight mirrors)
        for i in range(5):
            fn(i)
    torch.cuda.synchronize()
    probe = max(time_calls(fns["stdgauss"], 5), 1e-3)
    rounds = 5
    calls = max(5, int(window_s / rounds * 1e3 / probe))
    res = {r: [] for r in fns}
    for _ in range(rounds):
        for r, fn in fns.items():
            res[r].append(time_calls(fn, calls))
    return {r: dict(ms_per_call_median=float(np.median(v)), ms_per_call_windows=[float(t) for t in v], calls_per_window=calls,
                    window_s=float(sum(v) * calls / 1e3)) for r, v in res.items()}


def profile_batch_kernels(S, calls=20):
    import torch
    from torch.profiler import ProfilerActivity, profile
    for v in S.variants.values():
        v.state.loss_and_grad(S.keys[0], S.x)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(calls):
            for v in S.variants.values():
                v.state.loss_and_grad(S.keys[i % 64], S.x)
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if "fm_batch" in ev.key:
            dt = getattr(ev, "device_time_total", None)
            if dt is None:
                dt = ev.cuda_time_total
            out[ev.key.split("(")[0]] = dict(calls=int(ev.count), us_per_call=float(dt) / max(int(ev.count), 1))
    return out


def bench_indep_mh(S, window_s):
    import torch
    from mfm_b200 import exe_flow_matching as E, random as mr
    opts = SimpleNamespace(rtol=1e-5, atol=1e-5, mxstep=1000, n_times=2)
    res = {}
    fns = {}
    for r, v in S.variants.items():
        gen, init_fn, _ = E.create_train_data_gn(S.dist, v.model, opts, fm_args(r, nis=-1))
        st = init_fn(S.x.clone(), 1.0)
        lp = S.dist.tempered(1.0)
        fns[r] = (lambda i, gen=gen, st=st, lp=lp: gen.flow_step(S.keys[i % 64], st, lp, S.P))
    for fn in fns.values():
        for i in range(3):
            fn(i)
    torch.cuda.synchronize()
    probe = max(time_calls(fns["stdgauss"], 3), 1e-3)
    rounds = 3
    calls = max(3, int(window_s / rounds * 1e3 / probe))
    times = {r: [] for r in fns}
    for _ in range(rounds):
        for r, fn in fns.items():
            times[r].append(time_calls(fn, calls))
    for r, v in times.items():
        res[r] = dict(ms_per_call_median=float(np.median(v)), ms_per_call_windows=[float(t) for t in v], calls_per_window=calls)
    return res


def main():
    p = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_ref_dist_bench.json"))
    p.add_argument("--window", type=float, default=1.5, help="seconds of timed work per shape and reference distribution")
    a = p.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("ref_dist_bench.py measures on a CUDA device; none found")
    from mfm_b200 import _build, _lib
    _build.build()
    lib = _lib.load()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    result = {"gpu": gpu_info(), "gemm": lib.mfm_gemm_describe().decode(), "window_s_per_variant": a.window, "shapes": {}}
    for name, c in SHAPES.items():
        S = setup(name, dev)
        r = {"chains": c["n"], "d": c["d"], "hidden": c["H"]}
        r["fm_loss_grad"] = bench_fm(S, a.window)
        base, phi = r["fm_loss_grad"]["stdgauss"]["ms_per_call_median"], r["fm_loss_grad"]["phifour"]["ms_per_call_median"]
        r["fm_loss_grad_overhead_pct"] = 100.0 * (phi - base) / base
        r["batch_kernels_profiler"] = profile_batch_kernels(S)
        if name == "phi-four":
            r["indep_flow_mh_step"] = bench_indep_mh(S, a.window)
            b, q = r["indep_flow_mh_step"]["stdgauss"]["ms_per_call_median"], r["indep_flow_mh_step"]["phifour"]["ms_per_call_median"]
            r["indep_flow_mh_overhead_pct"] = 100.0 * (q - b) / b
        result["shapes"][name] = r
        print(name, json.dumps(r), flush=True)
        del S
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps({"gpu": result["gpu"], "overhead_pct": {k: v["fm_loss_grad_overhead_pct"] for k, v in result["shapes"].items()}}))


if __name__ == "__main__":
    main()
