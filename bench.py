#!/usr/bin/env python
"""bench.py — NeRF-SH SH16 training throughput (BASELINE.json metric) on N B200s of one node.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --gpus 1 --steps 3 --warmup 1     # CPU oracle arm
    python bench.py --gpus 1 --steps 20 --warmup 5 --dump-outputs DIR  # also write the last timed step's outputs

Every timed loop of train steps (the main region, the per-step distribution, the end-to-end loop, the per-kernel
timing and the `strong` / `tt_sh25` extras) runs --steps steps.

Workload (config.workload): BASELINE.json configs[1] — nerf_sh/config/blender (SH16, 64 coarse + 128
fine samples = 256 MLP evaluations per ray, white background, sparsity loss on 10,000 points), synthetic
800x800 random spherical poses, batch 4096 rays per GPU, random-init glorot weights, uniform random
target pixels.  One "step" = one full train_step: forward (both levels), loss, backward, gradient
all-reduce (N > 1), Adam, operand re-pack.  Weak scaling: every rank owns 4096 rays and its own 10,000
sparsity points per step (the reference draws those per device, nerf_sh/train.py:77-83).

`value`  : rays/s with the step's rays already resident in HBM (CUDA events, max over ranks).
`e2e`    : rays/s through the host-facing API with the rays/pixels of every step copied from pinned host
           memory and the step's loss statistics read back to the host inside the timed region.
`roofline`: dominant kernel class (and, under `kernels`, all three), algorithmic GEMM FLOPs (SURVEY.md §8d:
           1,007,104 fwd / 942,592 dgrad / 1,007,104 wgrad FLOP per MLP-sample, SH16) / CUDA-event kernel time,
           vs the measured sustained bf16 tensor peak in MEASURED_PEAKS.json; `step_frac` = the whole step.
`strong`, `tt_sh25`, `c4_extraction`, `c5_octree_opt`, `render_eval`: the other BASELINE configurations, timed after the main
           region on the same ranks (bench_extras.py); skipped with --no-extras.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "NeRF-SH train rays/sec (SH16, 64+128 samp/ray, batch 4096/GPU)"
RAYS = 4096
NC, NF = 64, 128
NSP = 10000
SH_DEG = 3
# algorithmic GEMM FLOPs per MLP-sample, SH16 (BASELINE.md §2)
F_FWD, F_DGRAD, F_WGRAD = 1007104.0, 2 * 471296.0, 1007104.0
SAMPLES_PER_STEP = RAYS * (NC + NC + NF) + NSP          # MLP evaluations per rank per step
FLOP_PER_STEP = SAMPLES_PER_STEP * (F_FWD + F_DGRAD + F_WGRAD)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(tflops=float(p.get("bf16_tflops_sustained", p.get("bf16_tflops"))), src="measured (sustained bf16)")
    return dict(tflops=1400.0, src="fallback (B200_PROFILING.md sustained)")


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = False
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}",
                 "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.samples.append(line.strip())
                if self.stop_flag:
                    break
        except Exception:
            pass

    def stop(self):
        self.stop_flag = True
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass

    def summary(self):
        sm, mx, reasons = [], [], set()
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        busy = sorted(sm)[len(sm) // 2:]
        return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons)}


def run_reference(args):
    """--impl reference: the reference algorithm on the host CPU (oracle port; the reference's JAX path
    cannot run here — no jax/flax in the image).  Each step = one train step on a bounded sample of the
    workload (REF_RAYS rays of the 4096-ray batch, sparsity points scaled alike)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import nerf_sh_oracle as O
    from plenoctree_b200.nerf.rays import random_rays_np   # numpy only: the CPU arm maps no repo .so
    ref_rays = 256
    nsp = max(1, NSP * ref_rays // RAYS)
    torch.set_num_threads(min(os.cpu_count() or 1, 32))   # beyond ~32 threads torch-CPU gets slower here
    cores = torch.get_num_threads()
    fc = O.init_flat_params(SH_DEG, 20200823)
    ff = O.init_flat_params(SH_DEG, 20200824)
    m = [np.zeros_like(fc), np.zeros_like(ff)]
    v = [np.zeros_like(fc), np.zeros_like(ff)]
    cfg = dict(num_coarse_samples=NC, num_fine_samples=NF, near=2.0, far=6.0, white_bkgd=True,
               sparsity_weight=1e-3, sparsity_length=0.05)
    rs = np.random.RandomState(0)

    def step(i):
        nonlocal fc, ff
        o, d, vd, px = random_rays_np(ref_rays, 1000 + i)
        t_rand = rs.uniform(0, 1, size=(ref_rays, NC)).astype(np.float32)
        u = rs.uniform(0, 1, size=(ref_rays, NF)).astype(np.float32)
        sp = rs.uniform(-1.5, 1.5, size=(nsp, 3)).astype(np.float32)
        _, gc, gf = O.loss_and_grads(fc, ff, SH_DEG, (o, d, vd), px, cfg, t_rand, u, sp)
        fc, m[0], v[0] = O.adam_step(fc, gc, m[0], v[0], float(i), 5e-4)
        ff, m[1], v[1] = O.adam_step(ff, gf, m[1], v[1], float(i), 5e-4)

    for i in range(args.warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(args.warmup + i)
    dt = time.perf_counter() - t0
    val = ref_rays * args.steps / dt
    sample = f"{ref_rays} rays x 256 MLP-samples + {nsp} sparsity points per step, torch CPU fp32, {cores} threads"
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "rays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1]: NeRF-SH SH16 training, blender config, synthetic 800x800 random poses",
                   "rays_per_step": ref_rays, "samples_per_ray": "64 coarse + 192 fine", "sparsity_points": nsp},
        "cpu_baseline": {"value": val, "unit": "rays/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def dump_outputs(out_dir, model, state, world):
    """Write what the last timed train_step left its caller, as float32 / float64 .npy files: the updated parameters
    (params), the Adam moments (adam_m, adam_v), the step's rank-averaged gradient (grads) and its Stats
    (stats: loss, psnr, loss_c, loss_sp, psnr_c, weight_l2).  About 16 MB for SH16."""
    from plenoctree_b200.nerf import train as T
    torch.cuda.synchronize()
    st = T.stats_from_raw(state.stats_raw / world, RAYS, 1e-3, NSP, True)
    st = st._replace(weight_l2=float((model.params.double() ** 2).sum() / model.params.numel()))
    arrays = {"params": model.params, "adam_m": state.m, "adam_v": state.v, "grads": state.grads / world}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())
    np.save(os.path.join(out_dir, "stats.npy"), np.array(st, dtype=np.float64))


def cpu_baseline_sample():
    from oracle import nerf_sh_oracle as O
    from plenoctree_b200.nerf.rays import random_rays_np   # numpy only: the CPU arm maps no repo .so
    ref_rays = 256
    nsp = max(1, NSP * ref_rays // RAYS)
    torch.set_num_threads(min(os.cpu_count() or 1, 32))
    cores = torch.get_num_threads()
    fc = O.init_flat_params(SH_DEG, 20200823)
    ff = O.init_flat_params(SH_DEG, 20200824)
    cfg = dict(num_coarse_samples=NC, num_fine_samples=NF, near=2.0, far=6.0, white_bkgd=True,
               sparsity_weight=1e-3, sparsity_length=0.05)
    rs = np.random.RandomState(0)
    times = []
    for i in range(4):
        o, d, vd, px = random_rays_np(ref_rays, 2000 + i)
        t_rand = rs.uniform(0, 1, size=(ref_rays, NC)).astype(np.float32)
        u = rs.uniform(0, 1, size=(ref_rays, NF)).astype(np.float32)
        sp = rs.uniform(-1.5, 1.5, size=(nsp, 3)).astype(np.float32)
        t0 = time.perf_counter()
        _, gc, gf = O.loss_and_grads(fc, ff, SH_DEG, (o, d, vd), px, cfg, t_rand, u, sp)
        O.adam_step(fc, gc, np.zeros_like(fc), np.zeros_like(fc), 0.0, 5e-4)
        O.adam_step(ff, gf, np.zeros_like(ff), np.zeros_like(ff), 0.0, 5e-4)
        times.append(time.perf_counter() - t0)
    best = min(times[1:])
    return {"value": ref_rays / best, "unit": "rays/s", "cores": cores, "kind": "port",
            "sample": f"best of 3 train steps on {ref_rays} rays x 256 MLP-samples + {nsp} sparsity points "
                      f"(same workload, bounded), torch CPU fp32 oracle, {cores} threads"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the strong-scaling / SH25 / extraction / octree extras")
    ap.add_argument("--workload", default="blender", choices=["blender", "tt"],
                    help="blender = BASELINE configs[1] (SH16, near/far 2/6; the default and the quoted metric); "
                         "tt = configs[2] (SH25, near/far 0/4, sparsity radius 5 / length 0.2)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the parameters, Adam moments, gradient and loss statistics of "
                         "the last timed step as DIR/<name>.npy (inputs are seeded: the same arguments give the same "
                         "inputs, so two builds can be compared output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    if args.impl == "reference":
        run_reference(args)
        return

    import torch.distributed as dist
    from plenoctree_b200 import _lib
    from plenoctree_b200.nerf import train as T
    from plenoctree_b200.nerf.models import NerfModel, Rays
    from plenoctree_b200.nerf.rays import random_rays_np

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    K, W = args.steps, args.warmup
    tt = args.workload == "tt"
    sh_deg = 4 if tt else SH_DEG
    near, far = (0.0, 4.0) if tt else (2.0, 6.0)
    sp_len, sp_rad = (0.2, 5.0) if tt else (0.05, 1.5)
    f_scale = (1020928.0 + 2 * 478208.0 + 1020928.0) / (F_FWD + F_DGRAD + F_WGRAD) if tt else 1.0
    model = NerfModel(sh_deg=sh_deg, num_coarse_samples=NC, num_fine_samples=NF, near=near, far=far, white_bkgd=True,
                      max_rays=RAYS, sparsity_npoints=NSP, device=dev)
    model.init_params(20200823)   # same weights on every rank (replicated, train.py:177)
    state = T.TrainState(model)

    # ---- synthetic ray pool: (2K + 2W) batches, different data per rank, host pinned + device copy
    nb = max(2 * (K + W), 800)        # >= 800 batches x 4096 rays x 48 B = 157 MB > the 126 MB L2
    o, d, vd, px = random_rays_np(nb * RAYS, 20200823 + 7919 * rank)
    host = torch.from_numpy(np.concatenate([o, d, vd, px], axis=1)).contiguous().pin_memory()   # [nb*RAYS, 12]
    pool = host.to(dev)                                                                          # HBM resident
    pool_mb = host.numel() * 4 / 1e6
    lr_of = lambda s: float(T.learning_rate_decay(s, 5e-4, 5e-6, 2000000))

    def batch_from(t, i):
        i = (i * 37) % nb                 # stride through the pool: every step touches a fresh region
        b = t[i * RAYS:(i + 1) * RAYS]
        return {"rays": Rays(b[:, 0:3], b[:, 3:6], b[:, 6:9]), "pixels": b[:, 9:12]}

    def step_resident(i):
        T.train_step(model, state, batch_from(pool, i), lr_of(state.step), sparsity_length=sp_len,
                     sparsity_radius=sp_rad)

    # end-to-end loop the way a host trainer drives the API: double-buffered staging, the batch of step i is copied
    # host->device and step i is enqueued, THEN the loss of step i-1 is read (its D2H copy has had a whole step to
    # land), so the device never idles on the host; every step's inputs cross PCIe and every step's loss is read on
    # the host inside the timed region (the last one by e2e_drain, before the closing event).
    stage = [torch.empty((RAYS, 12), dtype=torch.float32, device=dev) for _ in range(2)]
    stats_host = [torch.empty(8, dtype=torch.float32).pin_memory() for _ in range(2)]
    done = [torch.cuda.Event() for _ in range(2)]
    pending = [False, False]
    losses = []

    def e2e_read(slot):
        if pending[slot]:
            done[slot].synchronize()
            losses.append(float(stats_host[slot][0]) / (3.0 * RAYS))
            pending[slot] = False

    def step_e2e(i):
        slot = i & 1
        i = (i * 37) % nb
        st = stage[slot]
        st.copy_(host[i * RAYS:(i + 1) * RAYS], non_blocking=True)                # H2D of this step's batch
        T.train_step(model, state, {"rays": Rays(st[:, 0:3], st[:, 3:6], st[:, 6:9]),
                                    "pixels": st[:, 9:12]}, lr_of(state.step), sparsity_length=sp_len,
                     sparsity_radius=sp_rad)
        stats_host[slot].copy_(state.stats_raw, non_blocking=True)                # D2H of the step's loss sums
        done[slot].record()
        pending[slot] = True
        e2e_read(1 - slot)                                                        # host reads the previous step's loss

    def e2e_drain():
        e2e_read(0)
        e2e_read(1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, first, drain=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            fn(first + i)
        if drain:
            drain()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    # ---- warm-up, then the resident-input measurement with clock sampling ----
    for i in range(W):
        step_resident(i)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    launches0 = _lib.lib.pob_launch_count()
    ms_total = timed(step_resident, W)
    launches = int(_lib.lib.pob_launch_count() - launches0)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model, state, world)
    # ---- per-step distribution over K further steps: every step bracketed by its own pair of events, no host sync
    # inside the loop
    ND = K
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(ND + 1)]
    barrier()
    evs[0].record()
    for i in range(ND):
        step_resident(W + K + i)
        evs[i + 1].record()
    barrier()
    per = sorted(evs[i].elapsed_time(evs[i + 1]) for i in range(ND))
    step_dist = {"steps": ND, "min_ms": per[0], "median_ms": per[ND // 2], "p90_ms": per[int(ND * 0.9)], "max_ms": per[-1],
                 "mean_ms": sum(per) / ND}
    # ---- end-to-end (host buffers) ----
    for i in range(W):
        step_e2e(K + W + i)
    e2e_drain()
    n_before = len(losses)
    ms_e2e = timed(step_e2e, K + 2 * W, e2e_drain)
    assert len(losses) - n_before == K and all(np.isfinite(losses[n_before:])), "e2e loop must read every step's loss"
    if sampler:
        sampler.stop()
    # ---- per-kernel-class timing (CUDA events around every launch), a separate run of K steps ----
    _lib.lib.pob_timing_enable(1)
    nprof = K
    for i in range(nprof):
        step_resident(W + i)
    ms_ph = (ctypes.c_double * 5)()
    n_ph = (ctypes.c_longlong * 5)()
    _lib.lib.pob_timing_read(ms_ph, n_ph)
    _lib.lib.pob_timing_enable(0)
    phases = ["mlp_fwd", "mlp_bwd", "mlp_wgrad", "render_stages", "optimizer"]
    per_step_ms = {p: ms_ph[i] / nprof for i, p in enumerate(phases)}
    if tt:
        alg = {"mlp_fwd": SAMPLES_PER_STEP * 1020928.0, "mlp_bwd": SAMPLES_PER_STEP * 2 * 478208.0,
               "mlp_wgrad": SAMPLES_PER_STEP * 1020928.0}
    else:
        alg = {"mlp_fwd": SAMPLES_PER_STEP * F_FWD, "mlp_bwd": SAMPLES_PER_STEP * F_DGRAD,
               "mlp_wgrad": SAMPLES_PER_STEP * F_WGRAD}
    dom = max(alg, key=lambda k: per_step_ms[k])
    peaks = measured_peaks()
    achieved = alg[dom] / (per_step_ms[dom] * 1e-3) / 1e12
    # dram__bytes_read.sum + dram__bytes_write.sum per kernel class and step, from the committed `ncu --set full`
    # capture of this round (profiles/r2_dram_traffic.json; scaled there to the 4096-ray step)
    traffic_all = {}
    for name in ("r2_dram_traffic.json", "r1_dram_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tpath):
            traffic_all = json.load(open(tpath))
            break
    traffic = traffic_all.get(dom)
    kernels = {k: {"ms_per_step": per_step_ms[k], "algorithmic_flops_per_step": alg[k],
                   "achieved": alg[k] / (per_step_ms[k] * 1e-3) / 1e12,
                   "frac": alg[k] / (per_step_ms[k] * 1e-3) / 1e12 / peaks["tflops"],
                   "traffic": traffic_all.get(k)} for k in alg}

    # ---- the other BASELINE configurations (bounded; never allowed to break the contract line) ----
    extras = {}
    if not args.no_extras:
        import bench_extras as X
        for key, fn in (("strong", lambda: X.strong_scaling(dev, peaks["tflops"], steps=K)),
                        ("tt_sh25", lambda: X.strong_scaling(dev, peaks["tflops"], steps=K, tt=True)),
                        ("c4_extraction", lambda: X.c4_extraction(dev, peaks["tflops"])),
                        ("c5_octree_opt", lambda: X.c5_octree_opt(dev)),
                        ("render_eval", lambda: X.render_eval(dev))):
            try:
                torch.cuda.empty_cache()
                extras[key] = fn()
            except Exception as e:   # noqa: BLE001
                extras[key] = {"error": f"{type(e).__name__}: {e}"[:300]}
                if world > 1:
                    raise   # ranks would desynchronise: fail loudly instead
    if rank == 0:
        value = world * RAYS * K / (ms_total * 1e-3)
        e2e = world * RAYS * K / (ms_e2e * 1e-3)
        line = {
            "metric": METRIC, "value": value, "unit": "rays/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16 operands / f32 accumulate (tcgen05 kind::f16), f32 params+Adam",
            "data": "synthetic",
            "config": {"workload": ("configs[2]: NeRF-SH SH25 training, nerf_sh/config/tt hyper-parameters, synthetic random "
                                    "poses, batch 4096 rays per GPU") if tt else
                                   ("configs[1]: NeRF-SH SH16 training, nerf_sh/config/blender, synthetic 800x800 "
                                    "random poses, batch 4096 rays per GPU"),
                       "rays_per_gpu_per_step": RAYS, "global_batch": RAYS * world,
                       "samples_per_ray": "64 coarse (MLP_0) + 192 fine (MLP_1) = 256 MLP evaluations",
                       "sparsity_points_per_gpu": NSP, "parallelism": f"dp{world}",
                       "l2_policy": f"inputs larger than L2: {pool_mb:.0f} MB ray pool, a fresh batch every step; "
                                    "per-step activation traffic ~17 GB"},
            "e2e": {"value": e2e, "unit": "rays/s", "ms_per_step": ms_e2e / K,
                    "h2d_bytes_per_step": RAYS * 12 * 4, "d2h_bytes_per_step": 8 * 4},
            "gpu_launches": launches,
            "kernel_ms_per_step": per_step_ms,
            "step_ms_distribution": step_dist,
            "step_tflops_algorithmic": FLOP_PER_STEP * f_scale / (ms_total / K * 1e-3) / 1e12,
            "roofline": {"bound": "tensor", "kernel": dom, "achieved": achieved, "peak": peaks["tflops"],
                         "unit": "TFLOP/s", "frac": achieved / peaks["tflops"], "traffic": traffic,
                         "peak_source": peaks["src"],
                         "algorithmic_flops_per_step": alg[dom], "share_of_step": per_step_ms[dom] / sum(per_step_ms.values()),
                         "step_frac": FLOP_PER_STEP * f_scale / (ms_total / K * 1e-3) / 1e12 / peaks["tflops"],
                         "kernels": kernels},
            "clocks": sampler.summary() if sampler else None,
        }
        line.update(extras)
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline_sample()
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
