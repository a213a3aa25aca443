"""train_step of the reference (nerf_sh/train.py:51-121) on the CUDA library.

    loss_fn + value_and_grad   -> lib.pob_loss_and_grad   (fused tcgen05 forward / dgrad / wgrad)
    lax.pmean(grad, "batch")   -> one torch.distributed all-reduce (NCCL) on the flat [gradient | stats] buffer
    optimizer.apply_gradient   -> lib.pob_adam_update      (flax Adam + operand re-pack)
GraphedTrainStep captures the whole step (jitter draws, kernels, collectives, Adam) in one CUDA graph.

Data parallel layout = one process per GPU; `batch` holds this rank's shard of the global batch
(reference: batch_size is global and split over devices, nerf_sh/nerf/utils.py:518-522, F8).
"""
import collections
import math

import numpy as np
import torch
import torch.distributed as dist

from .._lib import TrainHParams, check, lib, ptr, stream_ptr
from .models import _cuda_f32, ctypes_ref

# nerf_sh/nerf/utils.py:43-50
Stats = collections.namedtuple("Stats", ("loss", "psnr", "loss_c", "loss_sp", "psnr_c", "weight_l2"))


def learning_rate_decay(step, lr_init, lr_final, max_steps, lr_delay_steps=0, lr_delay_mult=1):
    """Learning rate of `step` (nerf_sh/nerf/utils.py:483-515): geometric interpolation from lr_init (step 0) to
    lr_final (step >= max_steps), times a warm-up factor that rises from lr_delay_mult to 1 along a quarter sine
    over the first lr_delay_steps steps."""
    frac = min(max(step / max_steps, 0.0), 1.0)
    lr = math.exp((1.0 - frac) * math.log(lr_init) + frac * math.log(lr_final))
    if lr_delay_steps > 0:
        ramp = math.sin(0.5 * math.pi * min(max(step / lr_delay_steps, 0.0), 1.0))
        lr *= lr_delay_mult + (1.0 - lr_delay_mult) * ramp
    return lr


class TrainState:
    """utils.TrainState(optimizer) (nerf_sh/nerf/utils.py:38-41): parameters live in model.params; the Adam
    moments and the step counter (flax optimizer.state.step) live here."""

    def __init__(self, model):
        self.model = model
        self.m = torch.zeros_like(model.params)
        self.v = torch.zeros_like(model.params)
        self.step = 0
        # gradient buffer: [params | 8 stats] so that the last all-reduce carries both pmean calls
        self.gbuf = torch.zeros(model.params.numel() + 8, dtype=torch.float32, device=model.device)
        # device copy of (lr, step) for replayable graphs
        self.lr_step = torch.zeros(2, dtype=torch.float32, device=model.device)
        self.rng_seed = 20200823 + 7919 * (dist.get_rank() if dist.is_available() and dist.is_initialized() else 0)

    @property
    def grads(self):
        return self.gbuf[:self.model.params.numel()]

    @property
    def stats_raw(self):
        return self.gbuf[self.model.params.numel():]


def default_loss_scale(n_rays):
    """power-of-two scale that keeps the fp16 gradient chain in range: dL/dC = scale*2(C-px)/(3R)."""
    return float(2 ** int(round(math.log2(128.0 * max(1, n_rays)))))


def loss_and_grad(model, state, batch, sparsity_weight=1e-3, sparsity_length=0.05, sparsity_radius=1.5,
                  randomized=True, t_rand=None, u=None, sp_points=None, loss_scale=None, z_fine=None,
                  sigma_noise=None, lr_step_on_device=False):
    """value_and_grad(loss_fn) for this rank's shard; fills state.grads / state.stats_raw (device)."""
    rays = batch["rays"]
    o = _cuda_f32(rays.origins, "rays.origins", 3)
    d = _cuda_f32(rays.directions, "rays.directions", 3)
    v = _cuda_f32(rays.viewdirs, "rays.viewdirs", 3)
    px = _cuda_f32(batch["pixels"], "pixels")[..., :3].contiguous()
    n = o.shape[0]
    use_sp = sparsity_weight > 0.0 and model.sparsity_npoints > 0
    if randomized and t_rand is None and (u is None or model.num_fine_samples == 0) and (sp_points is None or not use_sp):
        # all of the step's draws in one launch of the library's Philox kernel (state.rng_seed, state.step)
        t_rand, u, sp_points = _draw(model, state, n, use_sp, sparsity_radius, lr_step_on_device)
    t_rand, u, upr = model._uniforms(n, randomized, t_rand, u)
    if use_sp:
        if sp_points is None:
            # random.uniform(key, (npoints,3), minval=-radius, maxval=radius)  (train.py:79)
            sp_points = (torch.rand((model.sparsity_npoints, 3), device=model.device) * 2 - 1) * sparsity_radius
        sp_points = _cuda_f32(sp_points, "sp_points", 3)
        if sp_points.shape[0] != model.sparsity_npoints:
            raise ValueError("sp_points must have sparsity_npoints rows")
    z_fine = None if z_fine is None else _cuda_f32(z_fine, "z_fine")   # keep alive until the launch
    noise = model._set_sigma_noise(n, randomized, sigma_noise)          # noqa: F841  (same)
    ws = model.workspace(True)
    hp = TrainHParams(float(sparsity_weight if use_sp else 0.0), float(sparsity_length),
                      float(loss_scale or default_loss_scale(n)))
    check(lib.pob_loss_and_grad(ctypes_ref(model.cfg), ctypes_ref(hp), ptr(model.blobs[0]),
                                ptr(model.blobs[1]) if model.num_mlps == 2 else None, ptr(o), ptr(d), ptr(v),
                                ptr(px), n, ptr(model.z_base), ptr(t_rand), ptr(u), upr,
                                ptr(z_fine), ptr(sp_points) if use_sp else None, ptr(state.grads),
                                ptr(state.stats_raw), ptr(ws), stream_ptr()))
    return n


def _draw(model, state, n, use_sp, sparsity_radius, step_on_device):
    """t_rand [n,Nc], u [n,Nf] ~ U[0,1) and sp_points [npoints,3] ~ U[-radius,radius) of this step, written by
    lib.pob_draw_uniforms into buffers the state owns (replaces random.uniform at model_utils.py:137,262 and
    train.py:79).  The counter is the step number: host value, or state.lr_step[1] when the step is graph-replayed."""
    nc, nf = model.num_coarse_samples, model.num_fine_samples
    nsp = model.sparsity_npoints if use_sp else 0
    key = (n, nsp)
    if getattr(state, "_draw_key", None) != key:
        state._draw_buf = torch.empty(n * nc + n * nf + 3 * nsp, dtype=torch.float32, device=model.device)
        state._draw_key = key
    buf = state._draw_buf
    t_rand = buf[:n * nc].view(n, nc)
    u = buf[n * nc:n * (nc + nf)].view(n, nf) if nf > 0 else None
    sp = buf[n * (nc + nf):].view(nsp, 3) if nsp > 0 else None
    check(lib.pob_draw_uniforms(int(state.rng_seed), float(state.step),
                                ptr(state.lr_step[1:]) if step_on_device else None, ptr(t_rand), n * nc,
                                ptr(u), n * nf, ptr(sp), 3 * nsp, float(sparsity_radius), stream_ptr()))
    return t_rand, u, sp


def stats_from_raw(raw, n_rays, sparsity_weight, sparsity_npoints, two_level, world=1):
    """device sums -> reference Stats (train.py:86-112); `raw` already averaged over ranks."""
    raw = [float(x) for x in raw.tolist()]
    loss = raw[0] / (3.0 * n_rays)
    loss_c = raw[1] / (3.0 * n_rays) if two_level else 0.0
    loss_sp = sparsity_weight * (1.0 - raw[2] / sparsity_npoints) if sparsity_npoints > 0 and sparsity_weight > 0 else 0.0
    psnr = -10.0 * math.log10(loss) if loss > 0 else float("inf")
    psnr_c = (-10.0 * math.log10(loss_c) if loss_c > 0 else float("inf")) if two_level else 0.0
    return Stats(loss, psnr, loss_c, loss_sp, psnr_c, float("nan"))


def _world():
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


def allreduce_gradients(gbuf):
    """lax.pmean(grad) + lax.pmean(stats) (nerf_sh/train.py:117-118) as ONE all-reduce(SUM) on the flat
    [grads | stats] buffer; returns the world size whose reciprocal the caller folds into Adam / stats."""
    world = _world()
    if world > 1:
        dist.all_reduce(gbuf, op=dist.ReduceOp.SUM)
    return world


def shard_batch(batch_size, rank, world):
    """reference semantics: batch_size is global and split evenly over devices (utils.py:518-522,252)."""
    if batch_size % world != 0:
        raise ValueError("Batch size must be divisible by the number of devices.")
    per = batch_size // world
    return rank * per, (rank + 1) * per


def train_step(model, state, batch, lr, sparsity_weight=1e-3, sparsity_length=0.05, sparsity_radius=1.5,
               weight_decay_mult=0.0, randomized=True, t_rand=None, u=None, sp_points=None, loss_scale=None,
               sync_stats=False, lr_step_on_device=False, collective=True):
    """One optimisation step (nerf_sh/train.py:51-121).  Returns Stats when sync_stats (forces a
    device->host read of the six scalars, like the reference's periodic logging), else None."""
    world = _world() if collective else 1     # collective=False: single-rank semantics inside a multi-rank job
    n = loss_and_grad(model, state, batch, sparsity_weight, sparsity_length, sparsity_radius, randomized, t_rand,
                      u, sp_points, loss_scale, lr_step_on_device=lr_step_on_device)
    if world > 1:
        allreduce_gradients(state.gbuf)   # pmean(grad) and pmean(stats) in one bucket
    # weight_l2 = sum(theta^2)/numel  ->  d/dtheta = 2*theta/numel  (train.py:101-108,114)
    wd = 2.0 * weight_decay_mult / model.params.numel() if weight_decay_mult else 0.0
    check(lib.pob_adam_update(model.sh_deg, model.num_mlps, ptr(model.params), ptr(state.grads), ptr(state.m),
                              ptr(state.v), float(lr), float(state.step),
                              ptr(state.lr_step) if lr_step_on_device else None, 1.0 / world, wd,
                              ptr(model.blobs[0]), ptr(model.blobs[1]) if model.num_mlps == 2 else None,
                              stream_ptr()))
    state.step += 1
    if sync_stats:
        raw = state.stats_raw / world
        st = stats_from_raw(raw, n, sparsity_weight, model.sparsity_npoints if sparsity_weight > 0 else 0,
                            model.num_mlps == 2)
        wl2 = float((model.params.double() ** 2).sum() / model.params.numel())
        return st._replace(weight_l2=wl2)
    return None


class GraphedTrainStep:
    """One train_step captured in a CUDA graph (jitter draws, ~30 kernel launches, the gradient all-reduce, Adam,
    operand re-pack) and replayed per step: at 512 rays per GPU (BASELINE's global batch of 4096 on 8 GPUs) the
    launches would otherwise cost as much as the kernels.  The batch lives in static device buffers; the learning
    rate and the step count reach the Adam kernel through a two-float device buffer written before every replay.

        g = GraphedTrainStep(model, state, n_rays)
        g.step(batch, lr)            # batch tensors may be host (pinned) or device; copied into the static buffers
    """

    HYPER_SLOTS = 16

    def __init__(self, model, state, n_rays, sparsity_weight=1e-3, sparsity_length=0.05, sparsity_radius=1.5,
                 weight_decay_mult=0.0, warmup=3, collective=True):
        self.model, self.state, self.n = model, state, int(n_rays)
        dev = model.device
        self.buf = torch.zeros((self.n, 12), dtype=torch.float32, device=dev)       # [o | d | v | px]
        # (lr, step) staging: a ring of pinned slots, each guarded by an event recorded behind its copy, so that the
        # host may queue several replays ahead without overwriting a slot whose copy has not executed yet
        self._host = torch.zeros((self.HYPER_SLOTS, 2), dtype=torch.float32).pin_memory()
        self._host_done = [None] * self.HYPER_SLOTS
        self._slot = 0
        self.kw = dict(sparsity_weight=sparsity_weight, sparsity_length=sparsity_length,
                       sparsity_radius=sparsity_radius, weight_decay_mult=weight_decay_mult, lr_step_on_device=True,
                       collective=collective)
        b = self._batch()
        # warm-up on a side stream (allocations, NCCL communicator, lazy module loads), then capture
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(torch.cuda.current_stream())
        step0 = state.step
        snap = [t.clone() for t in (model.params, state.m, state.v)]
        with torch.cuda.stream(s):
            for _ in range(warmup):
                self._set_hyper(0.0)
                train_step(model, state, b, 0.0, **self.kw)
        torch.cuda.current_stream().wait_stream(s)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            train_step(model, state, b, 0.0, **self.kw)
        # the warm-up / capture steps ran with lr = 0 but still moved the Adam moments: restore
        for t, c in zip((model.params, state.m, state.v), snap):
            t.copy_(c)
        model.repack()
        state.step = step0

    def _batch(self):
        from .models import Rays
        b = self.buf
        return {"rays": Rays(b[:, 0:3], b[:, 3:6], b[:, 6:9]), "pixels": b[:, 9:12]}

    def _set_hyper(self, lr):
        k = self._slot
        self._slot = (k + 1) % self.HYPER_SLOTS
        if self._host_done[k] is not None:
            self._host_done[k].synchronize()
        self._host[k, 0] = float(lr)
        self._host[k, 1] = float(self.state.step)
        self.state.lr_step.copy_(self._host[k], non_blocking=True)
        ev = self._host_done[k] or torch.cuda.Event()
        ev.record()
        self._host_done[k] = ev

    def step(self, batch12, lr):
        """batch12: [n_rays, 12] float32 tensor (origins | directions | viewdirs | pixels), host-pinned or device."""
        self.buf.copy_(batch12, non_blocking=True)
        self._set_hyper(lr)
        self.graph.replay()
        self.state.step += 1
