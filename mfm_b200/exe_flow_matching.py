"""Hot-path entry points — B200 drop-in for the reference's exe_flow_matching.py.

Mirrors (same names, argument meaning, return structure):
  VectorFieldNet            exe_flow_matching.py:56-90     (parameter container + apply)
  create_train_state        :93-186   (FM loss, AdamW -> clip -> apply_if_finite)
  create_learning_rate_fn   :189-198
  create_train_data_gn      :201-318  -> (train_data_generator, init_fn, transform_and_logdet)
  run                       :321-450  (hot loop incl. adaptive tempering; post-training metrics/plots
                                        are out of scope, see DESIGN.md)
Everything numeric happens in CUDA kernels behind the C-ABI (include/mfm_b200.h).
"""
from __future__ import annotations

import logging
import os
import time
from types import SimpleNamespace
from typing import Callable, NamedTuple, Optional

import numpy as np
import torch

from . import _lib, parallel, random as mrandom
from .bblackjax.mcmc.mala import MALAInfo, MALAState, init, mala_step
from .distributions import DeviceLogDensity, Distribution, GaussianMixture, IndepGaussian, PhiFourBase

logger = logging.getLogger(__name__)

def _broken_ref(name, why):
    def make(dim, device=None):
        raise TypeError(f"ref_dist='{name}' cannot be constructed in the reference either: {why}")
    return make


# exe_flow_matching.py:48-54.  'bimodal' and 'flat' fail at construction in the reference as coded (GaussianMixture(dim)
# indexes an int, FlatDistribution() misses its argument); they raise here too.  'phifour' is PhiFourBase(dim) with its defaults
# (alpha 0.1, beta 20, prior_type 'coupled'), a Gaussian with a tridiagonal precision that the kernels apply through its band factor.
ref_dists = {
    "stdgauss": lambda dim, device=None: IndepGaussian(dim, device=device),
    "widegauss": lambda dim, device=None: IndepGaussian(dim, var=5.0, device=device),
    "phifour": lambda dim, device=None: PhiFourBase(dim, device=device),
    "bimodal": _broken_ref("bimodal", "GaussianMixture(dim) takes the modes, not a dimension (distributions.py:43-49)"),
    "flat": _broken_ref("flat", "FlatDistribution() is called without its dim argument (exe_flow_matching.py:52)"),
}


def make_ref_dist(args, dim, device=None):
    name = getattr(args, "ref_dist", "stdgauss")
    if name not in ref_dists:
        raise NotImplementedError(f"ref_dist='{name}' is not implemented on device (stdgauss, widegauss, phifour are)")
    return ref_dists[name](dim, device=device)


# ------------------------------------------------------------------------------------------------
# VectorFieldNet
# ------------------------------------------------------------------------------------------------
def branch_widths(hidden_t, hidden_x, hidden_xt):
    """((Ht0, Ht1), (Hx0, Hx1), (Hxt0, Hxt1)) from the three --hidden_* lists.  The device network has exactly two hidden
    layers per branch (flax names Dense_0..Dense_7); each width is free."""
    out = []
    for name, ws in (("hidden_t", hidden_t), ("hidden_x", hidden_x), ("hidden_xt", hidden_xt)):
        ws = [int(w) for w in ws]
        if len(ws) != 2:
            raise NotImplementedError(f"{name} has {len(ws)} layers: the CUDA path implements two hidden layers per branch "
                                      "(depth is the limit; the widths are free)")
        if min(ws) <= 0:
            raise ValueError(f"{name} widths must be positive, got {ws}")
        out.append(tuple(ws))
    return tuple(out)


def layer_shapes(dim: int, hidden: int, fourier_dim: int, widths=None):
    """(in, out) of Dense_0..Dense_7 in flax construction order (exe_flow_matching.py:73-86).  widths: ((Ht0, Ht1), (Hx0, Hx1),
    (Hxt0, Hxt1)) as branch_widths returns it; None: every width is `hidden`.  Dense_5 reads cat = [s_x | s_t]."""
    F, d = fourier_dim, dim
    (t0, t1), (x0, x1), (xt0, xt1) = widths if widths is not None else ((hidden,) * 2,) * 3
    return [(2 * F, t0), (t0, t1), (d, x0), (x0, x1), (t1, d), (x1 + t1, xt0), (xt0, xt1), (xt1, d)]


class VectorFieldParams:
    """Flat fp32 parameter buffer + offsets; converts from/to the flax dict layout
    {'params': {'Dense_i': {'kernel': [in,out], 'bias': [out]}}}.  widths (optional): the per-branch hidden widths
    ((Ht0, Ht1), (Hx0, Hx1), (Hxt0, Hxt1)); `hidden` must then be the widest of them."""

    def __init__(self, dim, hidden, fourier_dim, device, widths=None):
        if widths is not None:
            widths = branch_widths(*widths)
            if hidden != max(max(w) for w in widths):
                raise ValueError(f"hidden={hidden} must be the widest layer of {widths}")
        self.dim, self.hidden, self.fourier_dim = dim, hidden, fourier_dim
        self.widths = widths if widths is not None else ((hidden, hidden),) * 3
        self.shapes = layer_shapes(dim, hidden, fourier_dim, widths)
        self.w_off, self.b_off = [], []
        off = 0
        for fi, fo in self.shapes:
            self.w_off.append(off); off += fi * fo
            off = (off + 3) // 4 * 4                      # 16-byte aligned slices
            self.b_off.append(off); off += fo
            off = (off + 3) // 4 * 4
        self.n_params = off
        self.device = torch.device(device)
        self.flat = torch.zeros(off, dtype=torch.float32, device=self.device)
        mask = torch.zeros(off, dtype=torch.uint8)
        for (fi, fo), wo in zip(self.shapes, self.w_off):
            mask[wo:wo + fi * fo] = 1                     # decay kernels only (decay_mask_fn, :116-127)
        self.decay_mask = mask.to(self.device)

    def kernel(self, i):
        fi, fo = self.shapes[i]
        return self.flat[self.w_off[i]:self.w_off[i] + fi * fo].view(fi, fo)

    def bias(self, i):
        return self.flat[self.b_off[i]:self.b_off[i] + self.shapes[i][1]]

    def load_dict(self, params: dict):
        p = params["params"]
        for i in range(8):
            self.kernel(i).copy_(torch.as_tensor(np.asarray(p[f"Dense_{i}"]["kernel"], np.float32)))
            self.bias(i).copy_(torch.as_tensor(np.asarray(p[f"Dense_{i}"]["bias"], np.float32)))
        return self

    def to_dict(self, flat: Optional[torch.Tensor] = None) -> dict:
        src = self.flat if flat is None else flat
        out = {}
        for i, (fi, fo) in enumerate(self.shapes):
            out[f"Dense_{i}"] = {
                "kernel": src[self.w_off[i]:self.w_off[i] + fi * fo].view(fi, fo).cpu().numpy().copy(),
                "bias": src[self.b_off[i]:self.b_off[i] + fo].cpu().numpy().copy(),
            }
        return {"params": out}


class VectorFieldNet:
    """Device vector field v(x, t) = nn_xt + nn_t * clip(grad logprob(x)) (exe_flow_matching.py:56-90).

    fourier_random is a module attribute (not a parameter), grad_logprob is fixed to the untempered
    target (`jax.grad(dist.logprob)`, :351) and therefore given as the distribution itself."""

    def __init__(self, fourier_random: torch.Tensor, dist: Distribution, hidden_x, hidden_t, hidden_xt,
                 act_fn="relu", grad_clip: Optional[float] = None):
        self.widths = branch_widths(hidden_t, hidden_x, hidden_xt)     # ((Ht0, Ht1), (Hx0, Hx1), (Hxt0, Hxt1))
        if act_fn is torch.relu:
            act_fn = "relu"
        if act_fn not in _lib.ACTIVATIONS:                       # non_lins (:40-46)
            raise KeyError(f"unknown non_linearity {act_fn!r}: one of {sorted(_lib.ACTIVATIONS)}")
        self.act = _lib.ACTIVATIONS[act_fn]
        self.dist = dist
        self.hidden = max(max(w) for w in self.widths)
        self.fourier_random = fourier_random.to(torch.float32).contiguous()
        self.grad_clip = float(grad_clip) if grad_clip else 0.0
        self.ref_mean, self.ref_std = 0.0, 1.0     # reference distribution of the flow (set_ref_dist)
        self.ref = None                            # None: IndepGaussian(ref_mean, ref_std^2)

    def set_ref_dist(self, ref):
        """ref_dists[args.ref_dist](dim) (:149,244): the kernels draw x0 / the independent proposal from it and evaluate
        its log-density, so its parameters travel in the field descriptor."""
        if isinstance(ref, IndepGaussian):
            self.ref_mean, self.ref_std, self.ref = float(ref.mean), float(ref.std), None
        elif isinstance(ref, PhiFourBase):
            if ref.dim != self.dist.dim:
                raise ValueError(f"reference distribution dim {ref.dim} != target dim {self.dist.dim}")
            self.ref_mean, self.ref_std, self.ref = 0.0, 1.0, ref
        else:
            raise NotImplementedError("the device kernels implement the IndepGaussian (stdgauss, widegauss) and PhiFourBase "
                                      "(phifour) reference distributions")
        return self

    def init(self, rng_key, x0=None, t0=None, head_scale: float = 0.0) -> VectorFieldParams:
        """Parameter initialisation.  NOT flax's RNG-folded lecun_normal (a 'next' row): fan-in
        scaled normals from jax.random-compatible streams; nn_t / nn_xt heads are zero-initialised as
        in the reference (:81,86) unless head_scale > 0."""
        P = VectorFieldParams(self.dist.dim, self.hidden, self.fourier_random.numel(), self.fourier_random.device,
                              widths=self.widths)
        keys = mrandom.split(rng_key, 8)
        for i, (fi, fo) in enumerate(P.shapes):
            scale = (1.0 / np.sqrt(fi)) * (head_scale if i in (4, 7) else 1.0)
            if scale > 0:
                P.kernel(i).copy_(mrandom.normal(keys[i], (fi, fo)) * scale)
        return P

    def field_desc(self, P: VectorFieldParams, flat: Optional[torch.Tensor] = None) -> _lib.FieldDesc:
        d = _lib.FieldDesc()
        d.dim, d.hidden, d.fourier_dim = P.dim, P.hidden, P.fourier_dim
        d.params = (P.flat if flat is None else flat).data_ptr()
        for i in range(8):
            d.w_off[i], d.b_off[i] = P.w_off[i], P.b_off[i]
        d.n_params = P.n_params
        d.omega = self.fourier_random.data_ptr()
        d.grad_clip = self.grad_clip
        d.ref_mean, d.ref_std = self.ref_mean, self.ref_std
        d.act = self.act
        if len({w for ws in P.widths for w in ws}) > 1:          # equal widths keep the zero tail: the descriptor of before
            (d.hidden_t[0], d.hidden_t[1]), (d.hidden_x[0], d.hidden_x[1]), (d.hidden_xt[0], d.hidden_xt[1]) = P.widths
        if self.ref is not None:
            self.ref._fill_ref(d)
        return d

    def apply(self, P: VectorFieldParams, x: torch.Tensor, t: torch.Tensor, z: Optional[torch.Tensor] = None,
              hutch: bool = False, want_div: bool = False):
        """Batched model.apply(params, x, t): x [N,d], t [N] -> v [N,d] (and div v [N])."""
        lib = _lib.load()
        n, d = x.shape
        t = t.to(torch.float32).reshape(-1).contiguous()
        if t.numel() == 1:
            t = t.expand(n).contiguous()
        v = torch.empty_like(x)
        div = torch.empty(n, dtype=torch.float32, device=x.device) if want_div else None
        fd, td = self.field_desc(P), self.dist._desc(1.0)
        od = _lib.OdeOpts(1e-5, 1e-5, 1000, 1 if hutch else 0, 2)
        ws = _lib.workspace(lib.mfm_ode_workspace_bytes(fd, td, od, n), x.device, "ode")
        _lib.check(lib.mfm_field_eval(fd, td, od, n, _lib.ptr(x.contiguous()), _lib.ptr(t),
                                      _lib.ptr(z.contiguous()) if z is not None else None, _lib.ptr(v), _lib.ptr(div),
                                      _lib.ptr(ws), ws.numel(), _lib.stream()))
        return (v, div) if want_div else v


# ------------------------------------------------------------------------------------------------
# optimizer / train state
# ------------------------------------------------------------------------------------------------
def create_learning_rate_fn(num_train_steps: int, num_warmup_steps: int, learning_rate: float) -> Callable[[int], float]:
    """Linear warmup then linear decay (exe_flow_matching.py:189-198): optax.join_schedules([linear_schedule(0 -> lr,
    warmup), linear_schedule(lr -> 0, total - warmup)], [warmup]).  optax.linear_schedule with transition_steps <= 0 is the
    constant init_value and join_schedules switches at the boundary, so warmup_steps = 0 is pure decay
    lr * (1 - step / num_train_steps).  The device optimizer evaluates the same schedule from its own step counter."""
    W, T = int(num_warmup_steps), int(num_train_steps)
    if W < 0 or W > T:
        raise ValueError("0 <= warmup_steps <= learning_iter")

    def lin(init, end, steps):
        if steps <= 0:
            return lambda c: init
        return lambda c: (init - end) * (1.0 - min(max(c, 0), steps) / steps) + end

    warm, decay = lin(0.0, learning_rate, W), lin(learning_rate, 0.0, T - W)

    def schedule(step):
        s = int(step)
        return warm(s) if s < W else decay(s - W)

    schedule.base, schedule.total, schedule.warmup = float(learning_rate), T, W
    return schedule


class TrainState:
    """flax TrainState analogue: params + AdamW moments + counters, all on device."""

    def __init__(self, model: VectorFieldNet, params: VectorFieldParams, lr_fn, args):
        self.model, self.P, self.lr_fn, self.args = model, params, lr_fn, args
        self.params = params
        dev = params.flat.device
        self.mu = torch.zeros_like(params.flat)
        self.nu = torch.zeros_like(params.flat)
        self.grads = torch.zeros_like(params.flat)
        self.loss = torch.zeros(1, dtype=torch.float32, device=dev)
        # [adam count, notfinite_count, total_notfinite, last_finite, scratch x4]
        self.opt_state = torch.tensor([0, 0, 0, 1, 0, 0, 0, 0], dtype=torch.int32, device=dev)
        self.step = 0
        self.ref_dist = make_ref_dist(args, params.dim, dev)                    # (:149)
        model.set_ref_dist(self.ref_dist)
        self._pending = None      # gradient all-reduce handles of an update that has not been applied yet


    # loss_fn(rng_key, samples, params) of the reference (flow_matching_loss, :171-179)
    def loss_and_grad(self, rng_key, positions, chain_offset=0, n_total=None, group=None, allreduce=False, defer=False):
        """value_and_grad(loss_fn) on this rank's chains.  allreduce=True additionally sums loss and gradient
        over the ranks of `group` (the loss is a SUM over chains, :178): the backward pass is issued in two
        parts and the all-reduce of the first part's gradients (Dense_4..7, 60 % of the buffer) runs on
        NCCL's stream while the second part computes.  defer=True returns once the LOSS is reduced and leaves
        the gradient all-reduces in flight: `apply_pending()` waits for them and applies the update, which
        lets the caller put parameter-independent work (the next MALA step) under the exchange."""
        assert self._pending is None, "apply_pending() first: the gradient buffer is still being reduced"
        lib = _lib.load()
        a = self.args
        if a.ot_cond_flow:
            raise NotImplementedError("the optimal-transport coupling (ot_cond_flow, ott-jax Sinkhorn) is not on the configured hot path")
        n = positions.shape[0]
        fd, td = self.model.field_desc(self.P), self.model.dist._desc(1.0)
        ws = _lib.workspace(lib.mfm_fm_workspace_bytes(fd, td, n), positions.device, "fm")
        pos = positions.contiguous()

        def part(k):
            _lib.check(lib.mfm_fm_loss_grad_part(fd, td, _lib.ptr(rng_key), n, chain_offset, n_total if n_total is not None else n,
                                                 float(a.sigma), _lib.ptr(pos), _lib.ptr(self.loss), _lib.ptr(self.grads),
                                                 _lib.ptr(ws), ws.numel(), k, _lib.stream()))

        _, world = parallel.world_info(group)
        if not a.cond_flow:
            # flow_fn (:139-147): one ABI call; with several ranks the gradient is reduced in one piece
            _lib.check(lib.mfm_fm_loss_grad_uncond(fd, td, _lib.ptr(rng_key), n, chain_offset, n_total if n_total is not None else n,
                                                   float(a.sigma), _lib.ptr(pos), _lib.ptr(self.loss), _lib.ptr(self.grads),
                                                   _lib.ptr(ws), ws.numel(), _lib.stream()))
            if allreduce and world > 1:
                parallel.allreduce_sum_([self.loss, self.grads], group)
            if defer:
                self._pending = ()
            return self.loss, self.grads
        if not allreduce or world == 1:
            part(0)
            if defer:
                self._pending = ()
            return self.loss, self.grads
        import torch.distributed as tdist
        split = self.P.w_off[4]
        part(1)
        h_tail = tdist.all_reduce(self.grads[split:], op=tdist.ReduceOp.SUM, group=group, async_op=True)
        h_loss = tdist.all_reduce(self.loss, op=tdist.ReduceOp.SUM, group=group, async_op=True)
        part(2)
        h_head = tdist.all_reduce(self.grads[:split], op=tdist.ReduceOp.SUM, group=group, async_op=True)
        h_loss.wait()
        if defer:
            self._pending = (h_tail, h_head)
            return self.loss, self.grads
        for h in (h_tail, h_head):
            h.wait()
        return self.loss, self.grads

    def apply_pending(self):
        """Finish a deferred update: wait (on the stream) for the gradient all-reduces, then AdamW."""
        if self._pending is not None:
            for h in self._pending:
                h.wait()
            self._pending = None
            self.apply_gradients()
        return self

    def apply_gradients(self, grads=None):
        lib = _lib.load()
        a = self.args
        g = self.grads if grads is None else grads
        _lib.check(lib.mfm_adamw_step(_lib.ptr(self.P.flat), _lib.ptr(g), _lib.ptr(self.mu), _lib.ptr(self.nu),
                                      _lib.ptr(self.P.decay_mask), self.P.n_params, _lib.ptr(self.opt_state),
                                      self.lr_fn.base, self.lr_fn.total, self.lr_fn.warmup, a.adam_beta1, a.adam_beta2, a.adam_epsilon,
                                      a.weight_decay, a.gradient_clip, 10, _lib.stream()))
        self.step += 1
        return self


def create_train_state(model: VectorFieldNet, vector_field_param: VectorFieldParams, learning_rate_fn, args) -> TrainState:
    return TrainState(model, vector_field_param, learning_rate_fn, args)


# ------------------------------------------------------------------------------------------------
# MALA / flow-MH data generator
# ------------------------------------------------------------------------------------------------
def create_train_data_gn(dist: Distribution, model: VectorFieldNet, ode_opts, args, chain_offset: int = 0,
                         n_total: Optional[int] = None):
    """Returns (train_data_generator, init_fn, transform_and_logdet) like the reference (:201-318).

    ode_opts: SimpleNamespace(rtol, atol, mxstep, n_times).  chain_offset/n_total describe this
    rank's shard of the ensemble (keys are rows of split(rng_key, n_total))."""
    lib = _lib.load()
    dim = dist.dim
    model.set_ref_dist(make_ref_dist(args, dim, dist.device))                       # (:244)
    opts = _lib.OdeOpts(float(ode_opts.rtol), float(ode_opts.atol), int(ode_opts.mxstep), 1 if args.hutchs else 0,
                        int(ode_opts.n_times))
    n_is = int(args.num_importance_samples)                 # > 0: conditional importance sampling (:280-296, :298)
    variant = _lib.FLOW_INDEP_MH if n_is < 0 else _lib.FLOW_RW_MH
    m = args.mcmc_per_flow_steps
    last_stats = {}

    def _ode(direction, key, sample, P, stats=None):
        """key: uint32[2] shared probe key (as the reference's un-vmapped call) or uint32[N,2]."""
        single = sample.dim() == 1
        x = (sample[None] if single else sample).contiguous()
        n = x.shape[0]
        keys = key if key.dim() == 2 else key[None].expand(n, 2).contiguous()
        y1 = torch.empty_like(x)
        ldj = torch.empty(n, dtype=torch.float32, device=x.device)
        fd, td = model.field_desc(P), dist._desc(1.0)
        ws = _lib.workspace(lib.mfm_ode_workspace_bytes(fd, td, opts, n), x.device, "ode")
        _lib.check(lib.mfm_ode_flow(fd, td, opts, direction, n, _lib.ptr(keys.contiguous()), _lib.ptr(x), _lib.ptr(y1),
                                    _lib.ptr(ldj), _lib.ptr(stats), _lib.ptr(ws), ws.numel(), _lib.stream()))
        return (y1[0], ldj[0]) if single else (y1, ldj)

    def transform_and_logdet(key, ref_sample, vector_field_param, stats=None):
        return _ode(+1, key, ref_sample, vector_field_param, stats)

    def inverse_and_logdet(key, target_sample, vector_field_param, stats=None):
        return _ode(-1, key, target_sample, vector_field_param, stats)

    def flow_step(rng_key, states: MALAState, logprob: DeviceLogDensity, P, per_chain_keys=False, inplace=False):
        x, l, g = states
        if not inplace:
            x, l, g = x.clone(), l.clone(), g.clone()
        n = x.shape[0]
        dev = x.device
        acc_rate = torch.empty(n, dtype=torch.float32, device=dev)
        is_acc = torch.empty(n, dtype=torch.uint8, device=dev)
        prop = torch.empty_like(x)
        weight = torch.empty(n, dtype=torch.float32, device=dev)
        stats = torch.zeros(8, dtype=torch.int32, device=dev)
        fd, td = model.field_desc(P), logprob.desc()
        if n_is > 0:
            ws = _lib.workspace(lib.mfm_flow_cis_workspace_bytes(fd, td, opts, n, n_is), dev, "flow")
            _lib.check(lib.mfm_flow_cis_step(fd, td, opts, n_is, _lib.ptr(rng_key.contiguous()), 1 if per_chain_keys else 0, n, chain_offset,
                                             n_total if n_total is not None else n, _lib.ptr(x), _lib.ptr(l), _lib.ptr(acc_rate),
                                             _lib.ptr(is_acc), _lib.ptr(prop), _lib.ptr(weight), _lib.ptr(stats), _lib.ptr(ws), ws.numel(),
                                             _lib.stream()))
            last_stats["ode"] = stats
            return MALAState(x, l, g), MALAInfo(acc_rate, is_acc.bool(), prop, weight)      # the gradient is kept, as coded (:295)
        ws = _lib.workspace(lib.mfm_flow_mh_workspace_bytes(fd, td, opts, n), dev, "flow")
        _lib.check(lib.mfm_flow_mh_step(fd, td, opts, variant, _lib.ptr(rng_key.contiguous()), 1 if per_chain_keys else 0,
                                        n, chain_offset, n_total if n_total is not None else n, _lib.ptr(x), _lib.ptr(l),
                                        _lib.ptr(g), _lib.ptr(acc_rate), _lib.ptr(is_acc), _lib.ptr(prop), _lib.ptr(weight),
                                        _lib.ptr(stats), _lib.ptr(ws), ws.numel(), _lib.stream()))
        last_stats["ode"] = stats
        return MALAState(x, l, g), MALAInfo(acc_rate, is_acc.bool(), prop, weight)

    def train_data_generator(rng_key, states: MALAState, count: int, vector_field_param, beta: float = 1.0,
                             inplace: bool = False, force: Optional[str] = None):
        """force='mala' / 'flow' (not in the reference): the caller has already decided which branch of the `lax.cond`
        (:304-313) this iteration takes (HotLoop's captured MALA iteration), so `count` is not consulted."""
        logprob = dist.tempered(beta)
        if force is not None:
            is_flow = force == "flow"
        elif 0 < m < 1:
            is_flow = count % (int(1 / m) + 1) != 0          # roles inverted for fractional m (:304-309)
        else:
            is_flow = count % (int(m) + 1) == 0              # :311
        if is_flow:
            return flow_step(rng_key, states, logprob, vector_field_param, inplace=inplace)
        return mala_step(logprob, rng_key, states, args.step_size, per_chain_keys=False, chain_offset=chain_offset,
                         n_total=n_total, inplace=inplace)

    def init_fn(init_positions, beta: float = 1.0):
        return init(init_positions, dist.tempered(beta))

    train_data_generator.flow_step = flow_step
    train_data_generator.inverse_and_logdet = inverse_and_logdet
    train_data_generator.last_stats = last_stats
    return train_data_generator, init_fn, transform_and_logdet


# ------------------------------------------------------------------------------------------------
# hot loop (exe_flow_matching.py:432-449)
# ------------------------------------------------------------------------------------------------
class HotLoop:
    """One rank's share of the reference's training loop: every outer iteration
        key_sample, key_train_gn, key_train_step = split(key_sample, 3)             (:433)
        train_states, infos = train_data_generator(key_train_gn, states, count, params, beta)  (:438)
        state, metrics = train_step(state, train_states.position, key_train_step)   (:439)
    Chains are sharded over ranks (this rank holds [chain_offset, chain_offset+n) of n_total); the
    only exchange is the SUM all-reduce of the flat FM gradient (and the scalar loss)."""

    def __init__(self, dist, model, P, args, ode_opts, key_sample, positions, beta=1.0, chain_offset=0, n_total=None,
                 process_group=None, pipeline=None, graph=None, real_sampler=None):
        import torch.distributed as tdist
        self.dist, self.model, self.P, self.args = dist, model, P, args
        self.n = positions.shape[0]
        self.n_total = n_total if n_total is not None else self.n
        self.chain_offset = chain_offset
        self.pg = process_group
        self.world = tdist.get_world_size(process_group) if (tdist.is_available() and tdist.is_initialized()) else 1
        self.pipeline = (self.world > 1) if pipeline is None else bool(pipeline)
        # MALA + FM-update iterations replayed from a CUDA graph: the latency-bound reference shapes (128 chains x d=2 is
        # 1 KB of state, ~60 launches per iteration) are otherwise bound by host launch overhead.  Off for big ensembles
        # (nothing to gain) and for multi-rank runs (NCCL + pipelined update).
        small = self.n * dist.dim <= (1 << 18)
        self.graph = (small and self.world == 1 and not self.pipeline and os.environ.get("MFM_GRAPH", "1") != "0") if graph is None else bool(graph)
        self._graph, self._graph_loss, self._eager_done, self._graph_ws_gen = None, None, False, -1
        self.graph_replays, self.replayed_launches, self._graph_launches = 0, 0, 0   # diagnostics (bench.py's gpu_launches)
        self.lr_fn = create_learning_rate_fn(args.learning_iter, args.warmup_steps, args.learning_rate)
        self.state = create_train_state(model, P, self.lr_fn, args)
        self.gen, self.init_fn, self.transform_and_logdet = create_train_data_gn(
            dist, model, ode_opts, args, chain_offset=chain_offset, n_total=self.n_total)
        self.beta = float(beta)
        self.key_sample = key_sample.clone()
        # use_real_samples (mcmc_per_flow_steps < 0, :328,382-386): the "data generator" draws from the target itself,
        # real_sampler(uint32[n,2] keys) -> [n,d]; no chains, no log-densities
        self.real_sampler = real_sampler
        if real_sampler is not None:
            self.graph = False
            self.states = MALAState(positions, None, None)
        else:
            self.states = self.init_fn(positions, self.beta)
        self.count = 0
        self.last_info = None

    def reset_positions(self, positions):
        self.states = MALAState(positions, None, None) if self.real_sampler is not None else self.init_fn(positions, self.beta)
        self._graph = None                    # the captured iteration points at the old state arrays

    def _mala_iteration_body(self):
        keys = mrandom.split(self.key_sample, 3)
        # only MALA iterations come here (iteration()): say so explicitly instead of encoding it in a fake count, which
        # cannot be done for fractional mcmc_per_flow_steps (m = 0.5: counts 1 and 2 are both flow iterations)
        self.states, self.last_info = self.gen(keys[1], self.states, self.count, self.P, self.beta, inplace=True, force="mala")
        loss, _ = self.state.loss_and_grad(keys[2], self.states.position, self.chain_offset, self.n_total)
        self.state.apply_gradients()
        self.key_sample.copy_(keys[0])
        return loss

    def _mala_iteration_body_sizing(self):
        """Make every workspace this iteration uses big enough BEFORE a capture (allocation is illegal inside one): the
        size queries are host-only."""
        lib = _lib.load()
        fd, td = self.model.field_desc(self.P), self.dist._desc(1.0)
        dev = self.states.position.device
        _lib.workspace(lib.mfm_fm_workspace_bytes(fd, td, self.n), dev, "fm")
        _lib.workspace(lib.mfm_mala_workspace_bytes(td, self.n), dev, "mala")

    def _graph_iteration(self):
        """MALA iteration through a CUDA graph: the first one runs eagerly (sizes every workspace), the second is captured,
        every later one only replays.  Same kernels, same order, same buffers => bit-identical to the eager loop."""
        if not self._eager_done:
            self._eager_done = True
            return self._mala_iteration_body()
        if self._graph is None or self._graph_beta != self.beta or self._graph_ws_gen != _lib.workspace_generation():
            # (a workspace the captured kernels point into may have been re-allocated by a bigger request elsewhere:
            #  the generation counter says so and the iteration is captured again against the live buffers)
            self._mala_iteration_body_sizing()
            g = torch.cuda.CUDAGraph()
            step = self.state.step
            l0 = _lib.load().mfm_launch_count()
            with torch.cuda.graph(g):
                self._graph_loss = self._mala_iteration_body()
            self._graph_launches = _lib.load().mfm_launch_count() - l0     # kernels one replay launches
            self.state.step = step            # capture records launches, it does not run them
            self._graph, self._graph_beta, self._graph_info = g, self.beta, self.last_info
            self._graph_ws_gen = _lib.workspace_generation()
        self._graph.replay()
        self.graph_replays += 1
        self.replayed_launches += self._graph_launches
        self.state.step += 1
        self.last_info = self._graph_info     # the graph's output buffers (a flow-MH iteration in between replaced the reference)
        return self._graph_loss

    def iteration(self):
        """One outer iteration (exe_flow_matching.py:433-439): data generator, then train_step.

        With several ranks the parameter update is pipelined: the gradient all-reduce of iteration k stays in
        flight while iteration k+1's MALA step runs (a MALA step reads the target only, never the MLP), and AdamW
        is applied right after it, before anything reads the parameters; a flow-MH iteration applies it first.
        Same arithmetic in the same order as the unpipelined loop."""
        self.count += 1
        if self.graph and self.beta >= 1.0 and not self.is_flow_iteration(self.count):   # while tempering the state arrays change every iteration
            return self._graph_iteration()
        keys = mrandom.split(self.key_sample, 3)
        self.key_sample.copy_(keys[0])          # in place: a captured graph reads this buffer
        key_train_gn, key_train_step = keys[1], keys[2]
        if self.real_sampler is not None:
            # train_data_generator = lambda key, *_: vmap(target_gn)(split(key, n_chain))  (:383-385); this rank's rows
            keys_n = mrandom.split(key_train_gn, self.n_total)[self.chain_offset:self.chain_offset + self.n].contiguous()
            self.states = MALAState(self.real_sampler(keys_n).contiguous(), None, None)
            self.last_info = MALAInfo(torch.full((self.n,), float("nan"), device=self.states.position.device), None, None, None)
        else:
            if self.is_flow_iteration(self.count):
                self.state.apply_pending()          # the flow step integrates the CURRENT vector field
            self.states, self.last_info = self.gen(key_train_gn, self.states, self.count, self.P, self.beta, inplace=True)
        self.state.apply_pending()
        pipelined = self.pipeline
        loss, grads = self.state.loss_and_grad(key_train_step, self.states.position, self.chain_offset, self.n_total,
                                               group=self.pg, allreduce=True, defer=pipelined)  # loss is a SUM over chains (:178)
        if not pipelined:
            self.state.apply_gradients()
        return loss

    def flush(self):
        """Apply an update still in flight (call before reading parameters / optimizer state from outside)."""
        self.state.apply_pending()
        return self

    # -- adaptive tempering (exe_flow_matching.py:391-417) ------------------------------------------
    def next_beta(self, prev_beta: float, positions) -> float:
        """beta_fn(prev_beta, vmap(dist.loglik)(positions)) on the whole ensemble."""
        lib = _lib.load()
        _, _, ll = self.dist.tempered(1.0).value_and_grad(positions, want_loglik=True)
        ll = parallel.allgather_chains(ll, self.n_total, self.pg).contiguous()
        prev = torch.tensor([prev_beta], dtype=torch.float32, device=ll.device)
        out = torch.empty(1, dtype=torch.float32, device=ll.device)
        _lib.check(lib.mfm_tempering_beta(_lib.ptr(ll), ll.shape[0], _lib.ptr(prev), float(self.args.alpha), _lib.ptr(out),
                                          _lib.stream()))
        return float(out.item())

    def temper(self):
        """beta_gen (:410-417): while beta < 1 pick the next beta and re-initialise (l, g) under it."""
        self.flush()
        if self.real_sampler is not None:
            return self.beta
        if self.beta < 1.0:
            self.beta = self.next_beta(self.beta, self.states.position)
            self.states = self.init_fn(self.states.position, self.beta)
            self._graph = None                # new state arrays, new temperature
        return self.beta

    def is_flow_iteration(self, count):
        m = self.args.mcmc_per_flow_steps
        if self.real_sampler is not None:
            return False
        return (count % (int(1 / m) + 1) != 0) if 0 < m < 1 else (count % (int(m) + 1) == 0)


# ------------------------------------------------------------------------------------------------
# final sampling + importance resampling (exe_flow_matching.py:389,453-459)
# ------------------------------------------------------------------------------------------------
def sample_flow(key_gen, dist: Distribution, ref_dist, transform_and_logdet, vector_field_param, n_samples: int):
    """The reference's post-training sampling, line for line:
        u = vmap(ref_dist.sample_model)(split(key_gen, n))                       (:389,453)
        key_hutch, key_choice = split(key_gen)                                   (:454; key_gen is reused as coded)
        flow_samples, vols = vmap(lambda u: transform_and_logdet(key_hutch, u, params))(u)   (:455; ONE probe key for all rows)
        log_weights = dist.logprob(flow_samples) - ref_dist.logprob(u) - vols    (:456-457)
        weights = exp(log_weights - max(log_weights))                            (:458)
        exact_samples = random.choice(key_choice, flow_samples, (n,), p=weights) (:459)
    Returns a dict with u, flow_samples, vols, log_weights, weights, exact_samples, indices."""
    lib = _lib.load()
    u = ref_dist.sample_model(mrandom.split(key_gen, n_samples))
    ks = mrandom.split(key_gen)
    key_hutch, key_choice = ks[0].clone(), ks[1].clone()
    flow_samples, vols = transform_and_logdet(key_hutch, u, vector_field_param)
    samples_logdensity = dist.logprob(flow_samples).contiguous()
    ref_logdensity = ref_dist.logprob(u).contiguous()
    log_w = torch.empty(n_samples, dtype=torch.float32, device=u.device)
    w = torch.empty_like(log_w)
    _lib.check(lib.mfm_importance_weights(_lib.ptr(samples_logdensity), _lib.ptr(ref_logdensity), _lib.ptr(vols.contiguous()), n_samples,
                                          _lib.ptr(log_w), _lib.ptr(w), _lib.stream()))
    exact, idx = mrandom.choice(key_choice, flow_samples, (n_samples,), w, return_index=True)
    return {"u": u, "flow_samples": flow_samples, "vols": vols, "samples_logdensity": samples_logdensity, "log_weights": log_w,
            "weights": w, "exact_samples": exact, "indices": idx}


# ------------------------------------------------------------------------------------------------
# run (exe_flow_matching.py:321-488): training loop, final sampling / importance resampling, metric table
# (mean log-density, KSD U/V statistics, MMD against real samples when a target generator is given).  Plots and the
# phi-four magnetisation histogram are out of scope; the function returns what the reference logs.
# ------------------------------------------------------------------------------------------------
def run(dist: Distribution, args, target_gn=None, device=None, log_every: int = 0, final_sampling: bool = True):
    logging.basicConfig(format="%(asctime)s - %(levelname)s - %(name)s - %(message)s", datefmt="%m/%d/%Y %H:%M:%S",
                        level=logging.INFO)
    dev = dist.device if device is None else torch.device(device)
    use_real_samples = args.mcmc_per_flow_steps < 0                                                  # (:328)
    if use_real_samples and target_gn is None:
        raise ValueError("mcmc_per_flow_steps < 0 trains on real samples: a target generator (uint32[n,2] keys -> [n,d]) is required")
    rank, world = parallel.world_info()
    n_total = args.num_chain
    lo, hi = parallel.shard_range(n_total, rank, world)
    iter_per_temp = args.anneal_iter // args.num_anneal_temp                                       # (:331; 0 raises at `count % 0` as in the reference)
    # key_target, key_sample, key_init, key_dist, key_fourier, key_gen = split(PRNGKey(seed), 6)   (:333)
    keys = mrandom.split(mrandom.PRNGKey(args.seed, dev), 6)
    key_sample, key_init, key_dist, key_fourier, key_gen = keys[1], keys[2], keys[3], keys[4], keys[5]
    dist.initialize_model(key_dist, n_total)                                                       # (:334)
    positions = dist.init_params[lo:hi].contiguous()
    fourier_random = args.fourier_std * mrandom.normal(key_fourier, (args.fourier_dim,))           # (:350)
    model = VectorFieldNet(fourier_random, dist, args.hidden_x, args.hidden_t, args.hidden_xt, args.non_linearity,
                           args.gradient_clip if args.dim > 128 else None)                         # (:351)
    P = model.init(key_init)
    ode_opts = SimpleNamespace(rtol=args.rtol, atol=args.atol, mxstep=int(args.mxstep),
                               n_times=5 if args.example == "4-mode" else 2)                       # (:345-349)
    logger.info(f"===== Starting training seed {args.seed} w/ {args.learning_iter} iterations =====")
    loop = HotLoop(dist, model, P, args, ode_opts, key_sample, positions, beta=1.0, chain_offset=lo, n_total=n_total,
                   real_sampler=target_gn if use_real_samples else None)
    if not use_real_samples:
        beta = loop.next_beta(0.0, positions)                                                      # (:426)
        logger.info(f"Initial beta= {beta}")
        loop.beta = beta
        loop.reset_positions(positions)                                                            # (:431)
    t0 = time.time()
    history = []
    for count in range(1, args.learning_iter + 1):                                                 # (:432-449)
        loss = loop.iteration()
        if count % iter_per_temp == 0:
            loop.temper()
        if log_every and (count % log_every == 0 or count == args.learning_iter):
            acc = loop.last_info.acceptance_rate if not use_real_samples else torch.full((2,), float("nan"))
            history.append({"count": count, "loss": float(loss.item()), "learning_rate": loop.lr_fn(count - 1),
                            "acceptance avg.": float(acc.mean().item()), "acceptance std.": float(acc.std(unbiased=False).item()),  # jnp .std(): ddof=0
                            "beta": loop.beta, "train_time": time.time() - t0})
            logger.info(str(history[-1]))
    loop.flush()
    torch.cuda.synchronize()
    train_time = time.time() - t0
    logger.info(f"Final beta= {loop.beta}")
    out = {"train_time": train_time, "final_beta": loop.beta, "history": history, "loop": loop}
    if final_sampling:
        # (:453-459) every rank draws the same eval_iter * num_chain samples (the draw is not sharded)
        from .mcmc_utils import max_mean_disc, stein_disc
        # with a target generator the reference REBINDS key_gen: key_gen, key_loss = split(key_target) (:371), so the real
        # samples and the final sampling both derive from split(key_target)[0]; without one key_gen is the 6th key of :333
        if target_gn is not None:
            key_gen = mrandom.split(keys[0].clone())[0].clone()
        fs = sample_flow(key_gen.clone(), dist, loop.state.ref_dist, loop.transform_and_logdet, P, args.eval_iter * n_total)
        flow_samples, exact_samples = fs["flow_samples"], fs["exact_samples"]
        out.update(flow_samples=flow_samples, exact_samples=exact_samples, weights=fs["weights"])
        # metric table (:463-488): mean log-density and kernelised Stein discrepancy of the flow and the resampled samples
        logpdf = float(fs["samples_logdensity"].mean().item())
        logger.info(f"Logpdf of flow samples= {logpdf}")
        stein = [float(v.item()) for v in stein_disc(flow_samples, dist.logprob)]
        logger.info(f"Stein U, V disc of flow samples= {stein[0]}, {stein[1]}")
        logpdf_ = float(dist.logprob(exact_samples).mean().item())
        logger.info(f"Logpdf of exact samples= {logpdf_}")
        stein_ = [float(v.item()) for v in stein_disc(exact_samples, dist.logprob)]
        logger.info(f"Stein U, V disc of exact samples= {stein_[0]}, {stein_[1]}")
        data = [args.mcmc_per_flow_steps, args.learning_iter, train_time, logpdf, logpdf_, stein[0], stein_[0], stein[1], stein_[1]]
        columns = ["mcmc/flow", "learn iter", "train time", "logpdf", "logpdf*", "KSD U-stat", "KSD U-stat*", "KSD V-stat", "KSD V-stat*"]
        if target_gn is not None:
            # real samples: vmap(target_gn)(split(key_gen, n_iter * n_chain)) with the rebound key_gen (:371-373);
            # target_gn maps uint32[n,2] keys -> [n,d] here
            real_samples = target_gn(mrandom.split(key_gen.clone(), args.eval_iter * n_total))
            mmd = float(max_mean_disc(real_samples, flow_samples).item())
            mmd_ = float(max_mean_disc(real_samples, exact_samples).item())
            logger.info(f"Max mean disc of flow samples= {mmd}")
            logger.info(f"Max mean disc of exact samples= {mmd_}")
            data += [mmd, mmd_]
            columns += ["MMD", "MMD*"]
        out.update(logpdf=logpdf, logpdf_exact=logpdf_, table=dict(zip(columns, data)))
    return out
