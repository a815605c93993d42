#!/usr/bin/env python
"""bench.py — chain-steps/sec of the MFM hot path (MALA + flow-MH + FM update).

Contract: `python bench.py --gpus N --steps K --warmup W` (torchrun for N>1) prints ONE JSON line.

Default workload = BASELINE.json configs[4] (SURVEY.md 8(d)): pines-shaped ensemble, 65 536 chains in total,
sharded over the N GPUs (strong scaling: total work fixed), d=1600, H=1024, step 0.01, mcmc_per_flow_steps m,
Hutchinson divergence, rtol=atol=1e-5, beta=1, synthetic positions mu + L eps, "trained-like" MLP fixture (all
kernels ~ N(0, 1/fan_in), heads x0.1, numpy seed 0).  `--config {4-mode,gaussian-mixture,phi-four,pines}` runs the
reference's own four configurations (configs[0..3]) at THEIR shapes on one GPU with the same step definition.

A STEP is one cycle-aligned block of (m+1) outer iterations of the reference loop (exe_flow_matching.py:432-449):
m MALA iterations + 1 flow-MH iteration, EACH followed by one flow-matching AdamW update.
value = n_total * K * (m+1) / seconds  [chain-steps/s].

`--impl reference` times the CPU oracle port of the same path (JAX is not installable here, see DESIGN.md) on the
host cores.  Its step is a BOUNDED SAMPLE of the cycle (a few MALA+FM iterations + one flow-MH+FM iteration on a small
ensemble); the line says what ran (`config.chains_total`, `sample`) and that the cycle rate is composed from the two
measured phase times (`extrapolated: true`).  The `cpu_baseline` object of the default run is ONE such step.

`--dump-outputs DIR` writes what the last timed step handed its caller (chain state, step info, FM loss, updated MLP
parameters) to DIR/<name>.npy in float32, so that two builds can be compared output for output on identical inputs:
every input of a run is a fixed function of the arguments (seeded fixture, seeded keys).  See dump_outputs().
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from types import SimpleNamespace

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

UNIT = "chain-steps/s"
F = 128
# name: chains, d, H, mcmc_per_flow_steps, step size, Hutchinson?, ODE grid, grad clip, CPU sample chains   (SURVEY.md 8 table)
CONFIGS = {
    "4-mode": dict(n=128, d=2, H=128, m=10, step=0.2, hutch=False, n_times=5, clip=None, cpu_n=128,
                   cite="BASELINE.json configs[0]: multi_modal.py --example 4-mode --mcmc_per_flow_steps 10"),
    "gaussian-mixture": dict(n=128, d=2, H=128, m=100, step=0.2, hutch=True, n_times=2, clip=None, cpu_n=128,
                             cite="BASELINE.json configs[1]: --example gaussian-mixture --mcmc_per_flow_steps 100 --hutchs (16 modes)"),
    "phi-four": dict(n=1024, d=64, H=128, m=1000, step=1e-4, hutch=False, n_times=2, clip=None, cpu_n=8,
                     cite="BASELINE.json configs[2]: --example phi-four --mcmc_per_flow_steps 1000 (exact trace)"),
    "pines": dict(n=128, d=1600, H=1024, m=100, step=0.01, hutch=True, n_times=2, clip=1.0, cpu_n=16,
                  cite="BASELINE.json configs[3]: --example pines --mcmc_per_flow_steps 100 --hutchs"),
    "pines-scaling": dict(n=65536, d=1600, H=1024, m=100, step=0.01, hutch=True, n_times=2, clip=1.0, cpu_n=16,
                          cite="BASELINE.json configs[4]: synthetic pines-shaped scaling run, 65536 chains over 1/2/4/8 GPUs"),
}


def metric_name(cfg):
    shape = {"pines-scaling": "pines 40x40", "pines": "pines 40x40 (128 chains)"}.get(cfg, cfg)
    return f"chain-steps/sec (MALA+flow-MH+FM update), {shape}"


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=1)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", type=str, default="b200", choices=["b200", "reference"])
    p.add_argument("--config", type=str, default="pines-scaling", choices=list(CONFIGS))
    p.add_argument("--chains", type=int, default=None, help="total chains over all GPUs (default: the configuration's)")
    p.add_argument("--mcmc_per_flow_steps", dest="m", type=int, default=None)
    p.add_argument("--head_scale", type=float, default=0.1)
    p.add_argument("--warmup_unit", type=str, default="cycle", choices=["iteration", "cycle"],
                   help="a warm-up step is one full cycle (default, = a timed step) or one outer iteration (>=3 of them touch every MALA/FM kernel, and "
                        "one extra flow-MH iteration is then run untimed)")
    p.add_argument("--no_cpu_baseline", action="store_true")
    p.add_argument("--no_e2e", action="store_true")
    p.add_argument("--dump-outputs", dest="dump_outputs", type=str, default=None, metavar="DIR",
                   help="write the outputs of the last timed step to DIR/<name>.npy (float32, a fixed sample of large arrays)")
    a = p.parse_args()
    if a.steps < 1 or a.warmup < 0:
        p.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs and a.impl != "b200":
        p.error("--dump-outputs applies to --impl b200")
    c = CONFIGS[a.config]
    a.chains = a.chains or c["n"]
    a.m = a.m if a.m is not None else c["m"]
    return a


def args_ns(a, learning_iter=10000):
    c = CONFIGS[a.config]
    return SimpleNamespace(hutchs=c["hutch"], num_importance_samples=0, mcmc_per_flow_steps=a.m, step_size=c["step"],
                           ref_dist="stdgauss", cond_flow=True, ot_cond_flow=False, sigma=1e-4, adam_beta1=0.9,
                           adam_beta2=0.999, adam_epsilon=1e-8, weight_decay=1e-4, gradient_clip=1.0,
                           learning_iter=learning_iter, warmup_steps=0, learning_rate=1e-3)


def fixture_params(d, H, head_scale):
    """Trained-like MLP fixture (SURVEY 8d): fixed numpy seed, heads scaled down."""
    rng = np.random.default_rng(0)
    shapes = [(2 * F, H), (H, H), (d, H), (H, H), (H, d), (2 * H, H), (H, H), (H, d)]
    p = {}
    for i, (fi, fo) in enumerate(shapes):
        s = (1.0 / np.sqrt(fi)) * (head_scale if i in (4, 7) else 1.0)
        p[f"Dense_{i}"] = {"kernel": (rng.standard_normal((fi, fo)) * s).astype(np.float32),
                           "bias": (rng.standard_normal(fo) * 0.01).astype(np.float32)}
    omega = rng.standard_normal(F).astype(np.float32)
    return {"params": p}, omega


# ------------------------------------------------------------------------------------------------
# algorithmic work per chain (SURVEY.md 8(d), BASELINE.md 3); 1 MAC = 2 flop
# ------------------------------------------------------------------------------------------------
def flops_per_chain(cfg):
    c = CONFIGS[cfg]
    d, H = c["d"], c["H"]
    P = 2 * F * H + 5 * H * H + 3 * d * H
    T = 2 * d * H + 3 * H * H
    dense_prior = 2 * d * d if d == 1600 else 0                   # pines: x K^-1 (GMM / phi-four: O(d), not counted)
    field = 2 * P + dense_prior + ((2 * T + dense_prior) if c["hutch"] else 2 * d * (3 * H * H + H))
    return dict(mala=dense_prior, fm=6 * P + dense_prior, field=field, logp=dense_prior)


class ClockSampler:
    def __init__(self, gpu_index):
        self.path = tempfile.mktemp(suffix=".csv")
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
            "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown," \
            "clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for nme, v in zip(names, parts[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        os.unlink(self.path)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU oracle (the ONE CPU baseline definition, used by both `--impl reference` and `cpu_baseline`)
# ------------------------------------------------------------------------------------------------
def oracle_target(cfg):
    from oracle import targets as OT
    return {"4-mode": OT.four_mode, "gaussian-mixture": OT.gmm16, "phi-four": lambda: OT.PhiFour(64),
            "pines": lambda: OT.LogGaussianCoxPines(1600), "pines-scaling": lambda: OT.LogGaussianCoxPines(1600)}[cfg]()


class CpuSample:
    """The NumPy oracle (float64, as the reference runs with jax_enable_x64) on a bounded sample of the workload:
    `n` chains of the configuration's shape.  step() = `r` MALA+FM iterations + 1 flow-MH+FM iteration; the cycle rate
    n (m+1) / (m t_mala + t_flow) is composed from the two measured phase times."""

    def __init__(self, cfg, m, head_scale, n=None, r=2):
        from oracle import optim as OO, samplers as OS, targets as OT, threefry as tf, vector_field as VF
        self.OS, self.tf, self.VF = OS, tf, VF
        c = CONFIGS[cfg]
        self.cfg, self.c, self.m, self.r = cfg, c, m, r
        self.n = n or c["cpu_n"]
        self.ot = oracle_target(cfg)
        self.params, self.omega = fixture_params(c["d"], c["H"], head_scale)
        self.ref = OT.IndepGaussian(c["d"])
        self.flow = OS.Flow(self.params, self.omega, self.ot, c["hutch"], 1e-5, 1e-5, 1000, c["clip"], np.linspace(0.0, 1.0, c["n_times"]))
        self.opt = OO.AdamWClipIfFinite(self.params, OO.learning_rate_fn(10000, 0, 1e-3))
        self.st = OS.mala_init(self.ot.init_positions(tf.PRNGKey(1), self.n, np.float64), self.ot)
        self.key = tf.PRNGKey(7)
        self.t_mala, self.t_flow, self.rk = [], [], None
        # torchrun exports OMP_NUM_THREADS=1 to every rank and small-batch NumPy GEMMs do not always gain from threads:
        # the BLAS thread count is set explicitly and calibrated per phase (1 vs all cores) so the CPU gets its best shot
        try:
            from threadpoolctl import threadpool_limits
            self._limits = threadpool_limits
        except Exception:
            self._limits = None
        self.cores_all = os.cpu_count() or 1
        self.th_mala = self._pick(self._mala_fm)
        zc = np.random.default_rng(1).standard_normal((self.n, c["d"]))
        self.th_flow = self._pick(lambda: VF.field_and_div(self.params, self.omega, self.st.position, np.full(self.n, 0.5), self.ot,
                                                           zc if c["hutch"] else None, c["clip"]))

    def _pick(self, fn):
        if self._limits is None:
            return self.cores_all
        best = None
        for cand in sorted({1, self.cores_all}):
            self._limits(limits=cand)
            fn()
            tc = time.perf_counter(); fn(); fn(); tc = time.perf_counter() - tc
            if best is None or tc < best[0]:
                best = (tc, cand)
        return best[1]

    def _fm_update(self, key_step):
        times, xt, target = self.VF.fm_batch(key_step, self.st.position, self.ref.sample, 1e-4)
        _, G = self.VF.fm_loss_and_grad(self.params, self.omega, xt, times, target, self.ot.grad, self.c["clip"])
        self.params = self.opt.update(G, self.params)
        self.flow.params = self.params

    def _mala_fm(self):
        self.key, k1, k2 = self.tf.split(self.key, 3)
        self.st, _, _ = self.OS.mala_step(self.tf.split(k1, self.n), self.st, self.ot, self.c["step"])
        self._fm_update(k2)

    def step(self):
        if self._limits:
            self._limits(limits=self.th_mala)
        t0 = time.perf_counter()
        for _ in range(self.r):
            self._mala_fm()
        self.t_mala.append((time.perf_counter() - t0) / self.r)
        if self._limits:
            self._limits(limits=self.th_flow)
        t0 = time.perf_counter()
        self.key, k1, k2 = self.tf.split(self.key, 3)
        stats = {}
        self.st, _ = self.OS.rw_flow_mh_step(self.tf.split(k1, self.n), self.st, self.ot, self.flow, 1.0, stats)
        self._fm_update(k2)
        self.t_flow.append(time.perf_counter() - t0)
        self.rk = (int(stats["inv"]["n_try"].max()), int(stats["fwd"]["n_try"].max()))

    def reset_timers(self):
        self.t_mala, self.t_flow = [], []

    def rate(self):
        tm, tf_ = float(np.mean(self.t_mala)), float(np.mean(self.t_flow))
        return self.n * (self.m + 1) / (self.m * tm + tf_), tm, tf_

    def describe(self):
        v, tm, tf_ = self.rate()
        c = self.c
        return (f"{self.n} chains (d={c['d']}, H={c['H']}), float64 NumPy oracle port; per step {self.r} MALA+FM iterations ({tm * 1e3:.1f} ms each, "
                f"{self.th_mala} BLAS thread(s)) + 1 flow-MH+FM iteration ({tf_:.2f} s, {self.rk[0]}+{self.rk[1]} RK attempts, {self.th_flow} BLAS thread(s)); "
                f"{len(self.t_flow)} step(s); cycle rate = n (m+1) / (m t_mala + t_flow), m = {self.m}; host has {self.cores_all} cores")

    def cores(self):
        return max(self.th_mala, self.th_flow)


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t0 = time.perf_counter()
    cpu = CpuSample(a.config, a.m, a.head_scale)
    for _ in range(a.warmup):
        cpu.step()
    cpu.reset_timers()
    tw = time.perf_counter()
    for _ in range(a.steps):
        cpu.step()
    wall_timed = time.perf_counter() - tw
    v, tm, tf_ = cpu.rate()
    cfg = workload_config(a, cpu.n)
    cfg["workload"] = f"{cpu.n}-chain sample of: " + cfg["workload"]
    cfg["sample_of_chains_total"] = a.chains
    cfg["step_definition"] = f"SAMPLE step: {cpu.r} MALA+FM iterations + 1 flow-MH+FM iteration on {cpu.n} chains (not a full {a.m}+1 cycle)"
    line = {"metric": metric_name(a.config), "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": 1e3 * wall_timed / max(a.steps, 1), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "impl": "reference", "config": cfg, "extrapolated": True,
            "sample_chains": cpu.n, "iterations_timed": {"mala_fm": cpu.r * a.steps, "flow_mh_fm": a.steps},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cpu.cores(), "kind": "port", "sample": cpu.describe()},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "CPU oracle port (NumPy restatement of the reference; JAX/flax/optax cannot be installed in this image). `value` is the "
                    "per-chain cycle rate composed from the measured phase times of the sample (extrapolated: the sample does not run "
                    f"{a.m} MALA iterations per flow iteration and holds {cpu.n} chains, not {a.chains}); ms_per_step is the measured wall time of one sample step",
            "wall_s": time.perf_counter() - t0}
    print(json.dumps(line), flush=True)


def workload_config(a, n_total):
    c = CONFIGS[a.config]
    big = n_total * c["d"] * 4 > 126e6
    return {"workload": c["cite"], "name": a.config, "chains_total": n_total, "dim": c["d"], "hidden": c["H"], "fourier_dim": F,
            "mcmc_per_flow_steps": a.m, "step_size": c["step"], "divergence": "hutchinson" if c["hutch"] else "exact trace",
            "ode_grid": c["n_times"], "rtol": 1e-5, "atol": 1e-5, "beta": 1.0, "flow_step": "random-walk MH in latent space (reference default)",
            "mlp_params": f"trained-like fixture, heads x{a.head_scale}, numpy seed 0",
            "step_definition": f"{a.m} MALA + 1 flow-MH outer iterations, each followed by one FM AdamW update",
            "l2": (f"inputs larger than L2 (state arrays {n_total * c['d'] * 4 / 2**20:.0f} MiB each)" if big else
                   "state smaller than L2 (the reference's own shape; latency-bound): every iteration rewrites the state and a cycle streams "
                   "the parameter / optimizer buffers, no separate flush"),
            "parallelism": f"chains sharded over {a.gpus} GPU(s), FM-gradient all-reduce (NCCL)"}


def device_dist(cfg, dev):
    from mfm_b200 import distributions as Dm
    from oracle import targets as OT          # constants of the two mixtures only (the fixture the tests use)
    if cfg in ("pines", "pines-scaling"):
        return Dm.LogGaussianCoxPines(1600, device=dev)
    if cfg == "phi-four":
        return Dm.PhiFour(64, device=dev)
    ot = OT.four_mode() if cfg == "4-mode" else OT.gmm16()
    return Dm.GaussianMixture(ot.modes, ot.covs, ot.weights, device=dev)


DUMP_ROWS, DUMP_PARAMS, DUMP_BYTES = 2048, 1 << 20, 64 * 10 ** 6


def dump_outputs(out_dir, loop, loss, n_total, off, world, rank):
    """--dump-outputs: what the last timed step returned to its caller, as float32 DIR/<name>.npy.

    The new chain state (position, logdensity, logdensity_grad), the step's info (acceptance_rate, is_accepted as 0/1,
    proposed_position, proposed_weight), the FM loss of its update and the updated flat MLP parameter vector.  Per-chain
    vectors hold every chain.  [chain, d] arrays hold the rows of DUMP_ROWS chains and `params` DUMP_PARAMS entries, both
    drawn once by numpy seed 0 (sorted, all of them when there are fewer), which keeps the files under DUMP_BYTES at every
    configuration.  Collective when chains are sharded over several ranks; rank 0 writes."""
    import torch
    import torch.distributed as tdist
    dev = loop.states.position.device
    n = loop.n

    def sample(total, k):
        idx = np.arange(total) if total <= k else np.sort(np.random.default_rng(0).choice(total, k, replace=False))
        return torch.from_numpy(idx).to(dev)

    def chains(t, idx):
        # rows `idx` (global chain indices) of a per-chain array: each rank fills the rows of its shard, the others are
        # zero, so the SUM all-reduce is a copy
        out = torch.zeros((idx.numel(),) + tuple(t.shape[1:]), dtype=torch.float32, device=dev)
        own = (idx >= off) & (idx < off + n)
        out[own] = t[idx[own] - off].float()
        if world > 1:
            tdist.all_reduce(out)
        return out.cpu().numpy()

    rows, every = sample(n_total, DUMP_ROWS), torch.arange(n_total, device=dev)
    st, info = loop.states, loop.last_info
    flat = loop.P.flat
    arrays = {"position": chains(st.position, rows), "logdensity": chains(st.logdensity, every),
              "logdensity_grad": chains(st.logdensity_grad, rows),
              "acceptance_rate": chains(info.acceptance_rate, every), "is_accepted": chains(info.is_accepted, every),
              "proposed_position": chains(info.proposed_position, rows), "proposed_weight": chains(info.proposed_weight, every),
              "loss": loss.detach().float().reshape(-1).cpu().numpy(),
              "params": flat[sample(flat.numel(), DUMP_PARAMS)].float().cpu().numpy()}
    total = sum(v.nbytes for v in arrays.values())
    assert total <= DUMP_BYTES, f"--dump-outputs would write {total} bytes"
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        for name, v in arrays.items():
            np.save(os.path.join(out_dir, name + ".npy"), v)


# ------------------------------------------------------------------------------------------------
def main():
    a = parse()
    if a.impl == "reference":
        return run_reference(a)
    # The contract is ONE JSON line on stdout: route everything else that libraries print to fd 1
    # (e.g. NCCL's version banner) to stderr, and keep a private handle for the result line.
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    import torch
    import torch.distributed as tdist
    from mfm_b200 import _lib, exe_flow_matching as E, random as mr

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        tdist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()

    c = CONFIGS[a.config]
    D, H = c["d"], c["H"]
    n_total = a.chains
    assert n_total % world == 0
    n = n_total // world
    off = rank * n
    m = a.m
    cyc = m + 1
    args = args_ns(a)
    opts = SimpleNamespace(rtol=1e-5, atol=1e-5, mxstep=1000, n_times=c["n_times"])

    dist = device_dist(a.config, dev)
    params, omega = fixture_params(D, H, a.head_scale)
    model = E.VectorFieldNet(torch.from_numpy(omega).to(dev), dist, [H, H], [H, H], [H, H], "relu", c["clip"])
    P = E.VectorFieldParams(D, H, F, dev).load_dict(params)

    # synthetic initial positions: this rank's rows of the configuration's own initialize_model (split(key_dist, n_total))
    key0 = mr.PRNGKey(1, dev)
    ks = mr.split(key0, 6)
    key_sample, key_dist = ks[1].clone(), ks[3].clone()
    rows = mr.split(key_dist, n_total)[off:off + n].contiguous()
    if a.config in ("pines", "pines-scaling"):
        eps = mr.normal(rows, (D,))
        pos0 = (dist._mu_zero + eps @ dist._cholesky_gram.T).contiguous()          # mu + L eps (distributions.py:312-314)
        del eps
    elif a.config == "phi-four":
        pos0 = (mr.uniform(rows, (D,)) * 2 - 1).contiguous()                      # distributions.py:162-164
    else:
        pos0 = mr.normal(rows, (D,)).contiguous()                                  # distributions.py:69-71
    del rows

    loop = E.HotLoop(dist, model, P, args, opts, key_sample, pos0, beta=1.0, chain_offset=off, n_total=n_total)

    def sync():
        if world > 1:
            tdist.barrier()
        torch.cuda.synchronize()

    def run_cycle():
        # iterations count+1 .. count+cyc with exactly one flow-MH iteration (count % (m+1) == 0); returns the last loss
        for _ in range(cyc):
            loss = loop.iteration()
        return loss

    # ---- warm-up -------------------------------------------------------------------------------
    if a.warmup_unit == "cycle":
        for _ in range(a.warmup):
            run_cycle()
    else:
        for _ in range(a.warmup):
            loop.iteration()              # MALA + FM update iterations
        # one untimed flow-MH iteration so the ODE kernels are warm too
        loop.count = cyc - 1
        loop.iteration()
        # realign: the timed window must start right after a multiple of (m+1)
        loop.count = 0
    loop.flush()
    sync()

    # ---- timed region --------------------------------------------------------------------------
    sampler = ClockSampler(local) if rank == 0 else None
    launches0 = lib.mfm_launch_count() + loop.replayed_launches
    replays0 = loop.graph_replays
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    flow_stats = []                       # per timed step: the flow iteration's ODE statistics (device tensors, read after the sync)
    sync()
    e0.record()
    for _ in range(a.steps):
        last_loss = run_cycle()
        flow_stats.append(loop.gen.last_stats.get("ode"))
    loop.flush()                          # multi-rank runs pipeline the last AdamW update: it belongs to the timed work
    e1.record()
    sync()
    ms = e0.elapsed_time(e1)
    launches = lib.mfm_launch_count() + loop.replayed_launches - launches0     # kernels launched directly + by CUDA-graph replays
    graph_replays = loop.graph_replays - replays0
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
    ms = float(t.item())
    value = n_total * a.steps * cyc / (ms / 1e3)
    stats_l = [s.cpu() for s in flow_stats if s is not None]
    ode_stats = stats_l[-1][:4].tolist() if stats_l else None
    chain_evals = [int(s[4:6].view(torch.int64).item()) for s in stats_l]          # rows ACTUALLY evaluated (compaction), per step
    if a.dump_outputs:                    # before the phase timings below move the chains on
        dump_outputs(a.dump_outputs, loop, last_loss, n_total, off, world, rank)

    # ---- per-phase timing (MALA iteration, FM update, flow iteration) for the roofline ------------
    def timed(fn, reps):
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); s0.record()
        for _ in range(reps):
            fn()
        s1.record(); torch.cuda.synchronize()
        return s0.elapsed_time(s1) / reps

    fl = flops_per_chain(a.config)
    key_t = mr.PRNGKey(99, dev)
    loop.flush()
    ms_fm = timed(lambda: loop.state.loss_and_grad(key_t, loop.states.position, off, n_total), 3)
    from mfm_b200.bblackjax.mcmc.mala import mala_step
    ms_mala = timed(lambda: mala_step(dist.tempered(1.0), key_t, loop.states, c["step"], False, off, n_total, inplace=True), 3)
    # one whole MALA outer iteration (data generator + FM loss/grad + gradient all-reduce + AdamW), max over ranks
    loop.flush()
    loop.count = 0
    ms_iter = timed(loop.iteration, min(5, m))
    loop.flush()
    t_it = torch.tensor([ms_iter], dtype=torch.float64, device=dev)
    if world > 1:
        tdist.all_reduce(t_it, op=tdist.ReduceOp.MAX)
    ms_iter = float(t_it.item())
    # dominant kernel: the dense-layer GEMM, measured on the FM hidden-layer shape [n,H] x [H,H] with K-major operands
    # (how every forward / backward-data layer calls it): a burst of 10 launches and a sustained run of >= 1 s (the
    # clocks settle under the 1 kW power cap), CUDA events on the launching stream.
    gemm_info = lib.mfm_gemm_describe().decode() if hasattr(lib, "mfm_gemm_describe") else ""
    Ag = torch.randn(n, H, device=dev); Bg = torch.randn(H, H, device=dev) / H ** 0.5; Cg = torch.empty(n, H, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    # as the layers call it: max |A| tracked by A's producer (here: reduced once, outside the timed launches) and the weight
    # operand pre-split once (per parameter update) and loaded by TMA
    a_amax = torch.zeros(1, device=dev)
    _lib.check(lib.mfm_absmax(Ag.data_ptr(), H, n, H, a_amax.data_ptr(), st))
    # ... and A arrives pre-split from the epilogue of the layer that produced it (here: made once by the same split kernel)
    As = torch.empty(n * H + 16, device=dev)
    _lib.check(lib.mfm_gemm_presplit(Ag.data_ptr(), As.data_ptr(), n * H, st))
    gemm = lambda: _lib.check(lib.mfm_gemm_dense(n, H, H, Ag.data_ptr(), H, Bg.data_ptr(), H, None, 0, Cg.data_ptr(), H, a_amax.data_ptr(), None, As.data_ptr(), As.data_ptr() + 4 * n * H, st))
    Bx = torch.empty(2 * H * H, device=dev)
    _lib.check(lib.mfm_gemm_presplit(Bg.data_ptr(), Bx.data_ptr(), H * H, st))
    lib.mfm_gemm_register_mirror(Bg.data_ptr(), H * H, Bx.data_ptr())
    ms_gemm_burst = timed(gemm, 10)
    ms_gemm = timed(gemm, max(10, min(20000, int(1000.0 / ms_gemm_burst))))
    lib.mfm_gemm_register_mirror(None, 0, None)
    gemm_tflops = 2.0 * n * H * H / (ms_gemm * 1e-3) / 1e12
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = float(peaks.get("bf16_tflops_sustained", 1590.0 if not peaks else peaks.get("bf16_tflops", 1590.0)))
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks else "fallback 1590 (of fallback)"
    # whole-step FLOPs from what was executed: FM updates and MALA steps on all n chains, field evaluations on the rows the
    # ODE loop actually evaluated (finished chains are compacted away), read from the device counter of every timed step
    step_flops = a.steps * n * (cyc * fl["fm"] + m * fl["mala"] + fl["logp"]) + sum(chain_evals) * fl["field"]
    step_tflops = step_flops / (ms * 1e-3) / 1e12
    # per-launch DRAM traffic of the dominant kernel: only from an ncu --set full capture of THIS round's kernel at THIS shape
    # (profiles/r02_ncu_traffic.json, written by scripts/ncu_summary.py from the committed capture); otherwise null
    traffic = None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")))
        if tr.get("rows") == n and tr.get("config") == a.config:
            traffic = float(tr["dram_bytes_per_launch"])
    except Exception:
        pass
    roofline = {"bound": "tensor",
                "kernel": f"dense-layer GEMM, FM shape [{n},{H}]x[{H},{H}], K-major operands; {gemm_info}",
                "achieved": gemm_tflops, "peak": peak_tf, "unit": "TFLOP/s", "frac": gemm_tflops / peak_tf,
                "traffic": traffic, "algorithmic_bytes": 2.0 * n * H * 4 + H * H * 4, "peak_source": peak_src,
                "achieved_burst": 2.0 * n * H * H / (ms_gemm_burst * 1e-3) / 1e12,
                "note": "algorithmic fp32 FLOPs (2*M*N*K per launch) / mean launch time over a sustained run (>= 1 s of back-to-back launches, "
                        "CUDA events). fp32-accurate products are emulated on the tensor cores, so the ceiling of the arithmetic is a fraction "
                        "of the bf16 peak (see `kernel` / DESIGN.md 5.1)",
                "whole_step_tflops_per_gpu": step_tflops,
                "whole_step_flops_source": "executed work: n*(FM + MALA) per iteration + device-counted active chain-evaluations of the ODE loops",
                "phase_ms": {"fm_loss_grad": ms_fm, "mala_iteration": ms_mala, "outer_iteration_mala": ms_iter,
                             "outer_iteration_flow": ms / a.steps - m * ms_iter},
                "phase_tflops": {"fm_loss_grad": n * fl["fm"] / (ms_fm * 1e-3) / 1e12,
                                 "mala_iteration": n * fl["mala"] / (ms_mala * 1e-3) / 1e12},
                "mala_state_gbs": n * (20 * D + 28) / (ms_mala * 1e-3) / 1e9}
    del Ag, Bg, Cg, Bx, As

    # ---- end-to-end through the public API with HOST buffers ---------------------------------------
    e2e = None
    if not a.no_e2e:
        host_in = torch.empty((n, D), dtype=torch.float32, pin_memory=True)
        host_in.copy_(loop.states.position)
        host_out = torch.empty((n, D), dtype=torch.float32, pin_memory=True)
        host_loss = torch.empty(1, dtype=torch.float32, pin_memory=True)
        dev_in = torch.empty((n, D), dtype=torch.float32, device=dev)
        loop.count = 0
        sync()
        e0.record()
        for _ in range(a.steps):
            dev_in.copy_(host_in, non_blocking=True)          # H2D: this step's chain positions
            loop.reset_positions(dev_in)                      # public init_fn: logdensity + grad
            loss = None
            for _ in range(cyc):
                loss = loop.iteration()
            loop.flush()
            host_out.copy_(loop.states.position, non_blocking=True)   # D2H: new positions + loss
            host_loss.copy_(loss, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            host_in.copy_(host_out)
        e1.record()
        sync()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
        e2e = {"value": n_total * a.steps * cyc / (float(t.item()) / 1e3), "unit": UNIT,
               "h2d_bytes_per_step": n * D * 4, "d2h_bytes_per_step": n * D * 4 + 4,
               "api": "HotLoop.reset_positions(init_fn) + (m+1) x HotLoop.iteration() per step, pinned host buffers"}

    # ---- CPU baseline (rank 0, N=1 only): ONE sample step of the reference arm's definition ----------
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        cs = CpuSample(a.config, m, a.head_scale)
        cs.step()
        cpu = {"value": cs.rate()[0], "unit": UNIT, "cores": cs.cores(), "kind": "port", "sample": cs.describe()}

    if rank == 0:
        line = {"metric": metric_name(a.config), "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": workload_config(a, n_total), "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
                "graph_replays": int(graph_replays),
                "roofline": roofline, "cpu_baseline": cpu,
                "fm_iterations_per_s": a.steps * cyc / (ms / 1e3),
                "ode_stats_last_flow_step": dict(zip(["accepted", "attempted", "max_attempts_per_chain", "field_evals"],
                                                     ode_stats)) if ode_stats else None,
                "ode_chain_evals_per_step": chain_evals,
                "arithmetic": "dense layers: fp32 products emulated on tensor cores (" + gemm_info + "), fp32 accumulate; everything else fp32",
                "warmup_unit": a.warmup_unit}
        real_stdout.write(json.dumps(line) + "\n")
        real_stdout.flush()
    if world > 1:
        tdist.destroy_process_group()


if __name__ == "__main__":
    main()
