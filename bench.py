#!/usr/bin/env python
"""bench.py -- the hot path's headline metric on B200 (see BASELINE.json / SURVEY.md §8(d)).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c1|c2|c4|c5] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one forward + backward pass of the hot path over one batch of views of a synthetic scene:
cull -> project -> tile bin / radix sort -> SH composite forward -> composite backward -> projection backward
(-> one NCCL all-reduce of the flat gradient buffer when N > 1).  Default workload = BASELINE config C3, the
configuration the metric is quoted on: 1M Gaussians, 1024x1024, SH degree 3.  With N GPUs each rank renders
one view of its own (weak scaling: per-GPU work fixed) and the gradients of all N views are all-reduced.
Metric: Gaussians x pixels / s = (sum over rendered views of N_gauss*H*W) / time.

`--impl reference` times the reference algorithm's CPU restatement (oracle/, kind "port": the reference has
no CPU path of its own and its CUDA extension is not a CPU implementation) on the host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def usable_cpus() -> int:
    """CPUs this container may actually use: min(affinity, cgroup quota).  The GPU boxes show 128 cores but carry a
    CFS quota (cpu.max 1600000/100000 = 16 CPUs, measured round 1); threads beyond the quota only get the whole
    process throttled in 100 ms slices -- which showed up as random 100-250 ms stalls in the timed loop."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = min(n, max(1, int(int(q) / int(per))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // per))
        except Exception:
            pass
    return n


_IS_REFERENCE_ARM = any(a == "reference" or a == "--impl=reference" for a in sys.argv[1:])
if _IS_REFERENCE_ARM:
    # SET, not setdefault: torch.distributed.run exports OMP_NUM_THREADS=1 to its workers, which crippled the CPU arm
    # of the round-1 scaling runs at N >= 2 (1 core instead of 16).  GSB200_REF_THREADS overrides for experiments.
    os.environ["OMP_NUM_THREADS"] = os.environ.get("GSB200_REF_THREADS", str(usable_cpus()))
    os.environ["MKL_NUM_THREADS"] = os.environ["OMP_NUM_THREADS"]
else:
    # the GPU arm's host work is a few tiny CPU tensor ops per view: an OpenMP pool of 64 spinning workers would
    # only burn the container's CPU quota
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    os.environ.setdefault("MKL_NUM_THREADS", "1")

import torch  # noqa: E402

N_LOOPS = 5  # timed K-step loops per measurement; the median is reported
METRIC = "fwd+bwd Gaussians*pixels/s"
UNIT = "Gaussian*pixel/s"
SH_C = {"c1": 1, "c2": 3, "c3": 4, "c4": 4, "c5": 4}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50, help="steps in each of the five timed loops")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=list(SH_C))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--svec-scale", type=float, default=1.0, help="C5 tile-occupancy sweep")
    ap.add_argument("--clock-period", type=float, default=0.1, help="NVML sampling period in s (0 = off)")
    ap.add_argument("--count-mode", default="auto", choices=["auto", "sync", "async"],
                    help="sync: render_forward waits for N_with_dub (8 bytes) -- the GPU idles whenever the host thread "
                         "is late (CFS throttling of the container shows up as slow loops); async: no host wait, "
                         "capacity-sized tile sort (GSB200_OPT_ASYNC_COUNT); auto (default): async at N=1, sync at "
                         "N>1 (there the sparse all-reduce holds a host wait per step anyway)")
    ap.add_argument("--no-c4-strong", action="store_true", help="skip the C4 strong-scaling sub-record")
    ap.add_argument("--no-ref-ext", action="store_true", help="skip the reference-extension comparison (N=1 only)")
    ap.add_argument("--dense-allreduce", action="store_true",
                    help="N>1: all-reduce the whole flat gradient buffer instead of the rows some view touched")
    ap.add_argument("--plain-grad-buffer", action="store_true",
                    help="N>1: do not allocate the all-reduce operand with ncclMemAlloc / register it")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed loops, write what their last step computed to DIR/<name>.npy (rank 0)")
    return ap.parse_args()


# ------------------------------------------------------------------------------------------------------
# workload
# ------------------------------------------------------------------------------------------------------
def make_views(workload, scene, n_views):
    """(cams, c2ws) for the step.  c4 has its own 8 orbit views; the single-view configs get one extra
    orbit pose per additional rank (azimuth +45 deg each) so that every GPU renders a different view."""
    from gsgen_b200.camera import orbit_c2w

    if workload == "c4":
        return scene.cams, scene.c2ws
    cam = scene.cams[0]
    c2ws = [orbit_c2w(2.5, 15.0 if workload != "c2" else 20.0, (30.0 if workload != "c2" else 45.0) + 45.0 * v)
            for v in range(n_views)]
    return [cam] * n_views, c2ws


def algorithmic_bytes(C, D, D_eff, N, N0, T, H, W):
    """SURVEY.md §8(d) per-stage algorithmic bytes of one view."""
    K = 3 * C * C
    b_inst = 4 + 4 * (7 + K)
    return {
        "preprocess": N0 * 25 + 84 * N,                 # cull + project(+aabb)
        "scan": N0 * 8,
        "bin": N * 20 + D * 12 + D * 24 + D * 8 + T * 8,  # key emit + sort + ranges
        "composite_fwd": D_eff * b_inst + 8 * T + 16 * H * W,
        "composite_bwd": D_eff * b_inst + D_eff * 4 * (7 + K) + 8 * T + 24 * H * W,
        "project_bwd": N * 40 + N * 28 + N * 40,
        "b_inst": b_inst,
    }


class ClockSampler:
    """SM clock / power / throttle reasons sampled from NVML on a background thread (every 10 ms), the same
    counters `nvidia-smi --query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.*` prints.  A thread
    inside this process avoids spawning nvidia-smi next to the timed region (its NVML start-up stalled CUDA calls for
    hundreds of ms in round 1).  mark() returns the sample index; stop(begin, end) summarises that window."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index, period_s=0.01):
        self.gpu_index, self.period = gpu_index, period_s
        self.samples = []  # (sm_mhz, power_w, reasons_bitmask)
        self.ok = False
        self._stop = False
        self.t = None

    def start(self):
        try:
            import threading

            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu_index)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
            self.t = threading.Thread(target=self._run, daemon=True)
            self.t.start()
        except Exception as e:  # pragma: no cover
            self.err = str(e)

    def _run(self):
        nv = self.nv
        while not self._stop:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                try:
                    rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    rs = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.samples.append((sm, pw, rs))
            except Exception:
                pass
            time.sleep(self.period)

    def mark(self):
        return len(self.samples)

    def stop(self, begin=0, end=None):
        self._stop = True
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML unavailable: " + getattr(self, "err", "?")]}
        if self.t is not None:
            self.t.join(timeout=1.0)
        win = self.samples[max(0, begin - 1):(None if end is None else end + 1)]
        if not win:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": ["no samples"]}
        mask = 0
        for _, _, r in win:
            mask |= r
        reasons = sorted(n for b, n in self.REASONS.items() if mask & b)
        return {"sm_mhz": statistics.median(x[0] for x in win), "sm_max_mhz": self.sm_max,
                "power_w_max": max(x[1] for x in win), "samples": len(win), "reasons": reasons,
                "source": "NVML (pynvml), %g s period, window = timed region" % self.period}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_numbers(workload):
    """per-launch numbers of the forward composite from the committed `ncu --set full` capture (profiles/traffic.json):
    DRAM bytes and executed warp instructions.  {} when there is no capture for the workload."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(workload, {})
        except Exception:
            return {}
    return {}


# ------------------------------------------------------------------------------------------------------
# CPU restatement (oracle) -- cpu_baseline leg and the --impl reference arm.  The only place bench.py
# executes oracle/.
# ------------------------------------------------------------------------------------------------------
def cpu_step_factory(workload, scene, cam, c2w, window_frac=1.0):
    import oracle

    C = SH_C[workload]
    ocam = oracle.Cam(cam.fx, cam.fy, cam.cx, cam.cy, cam.w, cam.h, cam.near_plane, cam.far_plane)
    g = torch.Generator().manual_seed(scene.seed + 100)
    gout = torch.randn(cam.h, cam.w, 3, generator=g)
    cfg = oracle.view_cfg(ocam)
    th, tw = cfg["n_tiles_h"], cfg["n_tiles_w"]
    keep = torch.ones(th, tw, dtype=torch.bool)
    if window_frac < 1.0:  # centred window of tiles
        import math

        s = math.sqrt(window_frac)
        hh, ww = max(1, int(round(th * s))), max(1, int(round(tw * s)))
        y0, x0 = (th - hh) // 2, (tw - ww) // 2
        keep[:] = False
        keep[y0:y0 + hh, x0:x0 + ww] = True
    px = 0
    for ty in range(th):
        for tx in range(tw):
            if keep[ty, tx]:
                px += (min(16, cam.h - 16 * ty)) * (min(16, cam.w - 16 * tx))
    keep_flat = keep.view(-1)

    def step():
        """-> (seconds in the per-Gaussian + binning stages incl. their backward, seconds in the window composite fwd+bwd)"""
        t0 = time.perf_counter()
        mean = scene.mean.clone().requires_grad_()
        qvec = scene.qvec.clone().requires_grad_()
        svec = scene.svec.clone().requires_grad_()
        alpha = scene.alpha.clone().requires_grad_()
        sh = scene.sh.clone().requires_grad_()
        normals, pts = oracle.get_frustum(ocam, c2w)
        mask = oracle.cull_bsphere(mean.detach(), svec.detach(), normals, pts, 6.0)
        m, q, s, a = mean[mask].contiguous(), qvec[mask].contiguous(), svec[mask].contiguous(), alpha[mask].contiguous()
        m2, c2, _, dp = oracle.project_gaussians(m, q, s, c2w, True)
        D, tl, br = oracle.tile_culling_aabb_count(m2.detach(), c2.detach(), 16, ocam, 6.0)
        ids, start, end = oracle.tile_culling_aabb_start_end(tl, br, dp.detach(), th, tw, D)
        if window_frac < 1.0:
            start = torch.where(keep_flat, start, torch.full_like(start, -1))
            end = torch.where(keep_flat, end, torch.full_like(end, -1))
        topleft = torch.tensor([-cam.cx / cam.fx, -cam.cy / cam.fy], dtype=torch.float32)
        shm = sh[mask].contiguous()
        # composite forward + backward on detached leaves (timed separately), then the chain rule through the
        # per-Gaussian stages with the gradients it produced
        m2d, c2d = m2.detach().requires_grad_(), c2.detach().requires_grad_()
        shd, ad = shm.detach().requires_grad_(), a.detach().requires_grad_()
        t1 = time.perf_counter()
        rgb = oracle.render_sh(m2d, c2d, shd, ad, start, end, ids, topleft, c2w, C, cfg, None)
        rgb.backward(gradient=gout)
        t2 = time.perf_counter()
        torch.autograd.backward([m2, c2, shm, a], [m2d.grad, c2d.grad, shd.grad, ad.grad])
        t3 = time.perf_counter()
        return (t1 - t0) + (t3 - t2), (t2 - t1)

    return step, px


def run_cpu_baseline(args):
    """cpu_baseline leg: the oracle (CPU restatement of the reference path) timed on the host cores, in a child
    process so that it gets its own OpenMP pool sized to the usable CPUs (the GPU arm runs single-threaded)."""
    n = usable_cpus()
    env = dict(os.environ, OMP_NUM_THREADS=str(n), MKL_NUM_THREADS=str(n), CUDA_VISIBLE_DEVICES="")
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", args.workload, "--steps", "1",
           "--warmup", "0", "--svec-scale", str(args.svec_scale)]
    out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    line = [l for l in out.stdout.splitlines() if l.startswith("{")]
    if not line:
        raise RuntimeError("reference arm printed no JSON: " + out.stderr[-300:])
    d = json.loads(line[-1])
    cb = d["cpu_baseline"]
    cb["seconds_per_step"] = d["ms_per_step"] / 1e3
    return cb


def run_reference_arm(args):
    """--impl reference: the reference algorithm's CPU restatement, same metric/config, K timed steps."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    from gsgen_b200.scenes import make_scene

    oracle.build()
    threads = int(os.environ.get("OMP_NUM_THREADS", usable_cpus()))
    torch.set_num_threads(threads)
    wl = args.workload
    scene = make_scene(wl, svec_scale=args.svec_scale)
    cams, c2ws = make_views(wl, scene, 1)
    cam, c2w = cams[0], c2ws[0]
    # bounded sample.  The per-Gaussian stages (project, 5M-key sort, their backward) do not shrink with a tile window,
    # so a windowed step would understate the reference if its time were divided by the window's pixels only.  Rule:
    # composite the FULL image whenever K+W such steps fit in ~4 minutes (16 usable cores: ~2.1 s/step); otherwise
    # composite a centred window of fraction f and report value = N*H*W / (t_per_gaussian + t_composite / f), i.e. the
    # composite time extrapolated to the whole image.
    total = args.steps + args.warmup
    step, px = cpu_step_factory(wl, scene, cam, c2w, 1.0)
    tp, tc = step()
    frac = 1.0
    if (tp + tc) * total > 240.0:
        for f in (0.25, 1.0 / 16):
            frac = f
            if (tp + tc * f) * total <= 240.0:
                break
        step, px = cpu_step_factory(wl, scene, cam, c2w, frac)
    for _ in range(args.warmup):
        step()
    acc_p = acc_c = 0.0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        a_, b_ = step()
        acc_p += a_
        acc_c += b_
    dt = (time.perf_counter() - t0) / args.steps
    H, W = cam.h, cam.w
    t_full = acc_p / args.steps + (acc_c / args.steps) / frac
    val = scene.N * H * W / t_full
    where = (f"on the FULL image ({px} px)" if frac >= 1.0 else
             f"on a centred window of {frac:.4g} of the tiles ({px} px), extrapolated by 1/{frac:.4g}")
    sample = (f"each step = all per-Gaussian stages + binning on {scene.N} Gaussians (fwd+bwd) + SH composite fwd+bwd "
              f"{where}; measured {dt:.3f} s/step of which {acc_c / args.steps:.3f} s composite; "
              f"value = N*H*W / (t_per_gaussian + t_composite/{frac:.4g})")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": t_full * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(wl, scene, cam), "views_per_step": 1, "parallelism": "cpu-openmp"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_name(wl, scene, cam):
    return (f"{wl}: {scene.N} Gaussians, {cam.w}x{cam.h}, SH deg {SH_C[wl] - 1} (C={SH_C[wl]}), tile 16, "
            f"T_thresh 1e-4, radii 6.0")


# ------------------------------------------------------------------------------------------------------
# ours
# ------------------------------------------------------------------------------------------------------
class Workload:
    """One synthetic scene + its views, replicated parameters, this rank's shard of the views."""

    def __init__(self, args, wl, world, rank, dev, count_mode=None):
        from gsgen_b200.parallel import ViewParallelRenderer, shard_views
        from gsgen_b200.rasterizer import render_view
        from gsgen_b200.scenes import make_scene

        self.args, self.wl, self.world, self.rank, self.dev = args, wl, world, rank, dev
        self.render_view = render_view
        self.C = SH_C[wl]
        self.scene = make_scene(wl, svec_scale=args.svec_scale)
        self.n_views = 8 if wl == "c4" else world
        self.cams, self.c2ws_cpu = make_views(wl, self.scene, self.n_views)
        sc = self.scene
        self.vpr = ViewParallelRenderer(dict(mean=sc.mean, qvec=sc.qvec, svec=sc.svec, alpha=sc.alpha, sh=sc.sh),
                                        self.C, dev, register_nccl=(world > 1 and not args.plain_grad_buffer),
                                        sparse_allreduce=(world > 1 and not args.dense_allreduce))
        self.mine = shard_views(self.n_views, rank, world)
        self.gouts = {}
        for v in self.mine:
            g = torch.Generator().manual_seed(sc.seed + 100 + v)
            self.gouts[v] = torch.randn(self.cams[v].h, self.cams[v].w, 3, generator=g).to(dev)
        self.slot_of = {v: i for i, v in enumerate(self.mine)}  # one library context per in-flight view
        self.count_mode = count_mode or (args.count_mode if args.count_mode != "auto"
                                         else ("async" if world == 1 else "sync"))
        self.async_count = (self.count_mode == "async")
        self.last = {}
        self.overflows = 0

    def render_and_backward(self, params, v):
        from gsgen_b200._lib import TileListOverflow

        # the pose is host data (it comes from the data loader): passing the CPU tensor avoids a D2H sync
        for attempt in range(2):
            out = self.render_view(params["mean"], params["qvec"], params["svec"], params["alpha"], self.c2ws_cpu[v],
                                   self.cams[v], sh=params["sh"], C=self.C, slot=self.slot_of[v],
                                   grad_sink=self.vpr.grad_views, async_count=self.async_count)
            try:
                out["rgb"].backward(gradient=self.gouts[v])
                break
            except TileListOverflow:  # asynchronous-count mode only: capacity was raised, render the view again
                self.overflows += 1
                if attempt:
                    raise
        self.last["rgb"], self.last["aux"] = out["rgb"], out["aux"]

    def step(self):
        self.vpr.step(self.n_views, self.render_and_backward)


DUMP_GRAD_ROWS = 131072  # Gaussians whose gradient rows --dump-outputs writes (all of them when the scene is smaller)


def dump_outputs(out_dir, w):
    """What the timed step hands its caller, as float32 .npy files: the last rendered view's image and the all-reduced
    gradient of every parameter.  The gradients are a fixed seeded sample of DUMP_GRAD_ROWS Gaussians (their indices in
    grad_rows.npy), which keeps the files under 64 MB at the 1M-Gaussian workloads."""
    import numpy as np

    torch.cuda.synchronize()
    os.makedirs(out_dir, exist_ok=True)
    N = w.scene.N
    rows = torch.randperm(N, generator=torch.Generator().manual_seed(0))[:DUMP_GRAD_ROWS].sort().values
    arrays = {"rgb": w.last["rgb"].detach(), "grad_rows": rows.double()}
    for name, g in w.vpr.grad_views.items():
        if name != "touched":
            arrays["grad_" + name] = g.detach()[rows.to(g.device)]
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy())


def timed_loops(args, step, barrier, world, dev, n_loops=3, sampler=None, rank=0):
    """n_loops x (exactly K steps, barrier + synchronize on both sides, CUDA events on the launching stream, max over
    ranks).  Returns [(ms_per_step, mark0, mark1)]."""
    import torch.distributed as dist

    res = []
    for _ in range(n_loops):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier(); torch.cuda.synchronize()
        m0 = sampler.mark() if (sampler is not None and rank == 0) else 0
        e0.record()
        for _ in range(args.steps):
            step()
        e1.record()
        torch.cuda.synchronize(); barrier()
        m1 = sampler.mark() if (sampler is not None and rank == 0) else 0
        t = torch.tensor([e0.elapsed_time(e1) / args.steps], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        res.append((float(t.item()), m0, m1))
    return res


def warm_up(args, step, world, dev):
    """>= 3 untimed steps + ~1.5 s of extra ones: the first backward spawns autograd / CUDA helper threads and the
    container's CPU quota needs a few periods to settle.  The COUNT is agreed across ranks (every step contains a
    collective): max over ranks of a 5-step estimate -- a time-based warm-up dead-locked NCCL at N=8 in round 1."""
    import torch.distributed as dist

    for _ in range(max(3, args.warmup)):
        step()
    torch.cuda.synchronize()
    t_w = time.perf_counter()
    for _ in range(5):
        step()
    torch.cuda.synchronize()
    est = torch.tensor([(time.perf_counter() - t_w) / 5], device=dev)
    if world > 1:
        dist.all_reduce(est, op=dist.ReduceOp.MAX)
    n_extra = int(min(1000, max(10, 1.5 / max(float(est.item()), 1e-4))))
    for _ in range(n_extra):
        step()
    torch.cuda.synchronize()


def roofline_extras(C, n_visible, d_eff, tiles, H, W, traffic, launch_ms, peak_gbs):
    """The two numbers SURVEY.md §8(d) wants NEXT to the contract-definition `achieved`: (ii) the compulsory lower bound
    of the forward composite -- every visible Gaussian's record + payload once, the consumed ids, tile ranges, outputs --
    and (i) the DRAM-side fraction: measured dram__bytes (one ncu launch, `traffic`) / launch time / HBM peak."""
    K = 3 * C * C
    compulsory = n_visible * 4 * (7 + K) + 4 * d_eff + 8 * tiles + 16 * H * W
    out = {"compulsory_bytes": float(compulsory),
           "compulsory_formula": "N_visible*4*(7+3C^2) + 4*D_eff + 8*tiles + 16*H*W (SURVEY.md §8(d)-ii)",
           "compulsory_frac": (compulsory / 1e9) / (launch_ms / 1e3) / peak_gbs if launch_ms > 0 else None}
    if traffic and launch_ms > 0:
        out["dram_gbs"] = (traffic / 1e9) / (launch_ms / 1e3)
        out["dram_frac"] = out["dram_gbs"] / peak_gbs
    return out


def dominant_kernel_roofline(stages, alg_bytes, ncu, peak_gbs, sm_mhz):
    """The same accounting for the kernel that dominates the step (the composite backward: 57 % of it) as `roofline`
    gives for the kernel north_star names (the composite forward): algorithmic bytes / measured launch time / HBM peak,
    the DRAM-side fraction from the committed ncu capture, and the limiter that is actually active -- instruction issue
    and the shared-memory data pipe (DESIGN.md §3.4)."""
    name = max(stages, key=lambda k: stages[k]["ms"])
    ms = stages[name]["ms"]
    out = {"kernel": {"composite_bwd": "k_composite_bwd_sh<C=4,fused>", "composite_fwd": "k_composite_fwd<SH,C=4>"}.get(name, name),
           "stage": name, "share_of_stage_sum": ms / sum(v["ms"] for v in stages.values()), "bound": "hbm",
           "achieved": stages[name]["alg_gbs"], "peak": peak_gbs, "unit": "GB/s",
           "frac": stages[name]["alg_gbs"] / peak_gbs if stages[name]["alg_gbs"] else None,
           "alg_bytes_per_launch": alg_bytes.get(name), "avg_launch_ms": ms,
           "traffic": ncu.get(f"{name}_dram_bytes")}
    if out["traffic"] and ms > 0:
        out["dram_frac"] = (out["traffic"] / 1e9) / (ms / 1e3) / peak_gbs
    inst = ncu.get(f"{name}_warp_inst")
    if inst and ms > 0:
        t_issue = inst / (148 * 4 * sm_mhz * 1e6) * 1e3
        out["issue_roofline"] = {"warp_instructions": inst, "min_ms_at_full_issue": t_issue, "frac": t_issue / ms}
    if ncu.get(f"{name}_smem_wavefront_pct") is not None:
        out["smem_data_pipe_pct_in_capture"] = ncu[f"{name}_smem_wavefront_pct"]
    return out


def allreduce_bytes(vpr):
    """bytes the step's gradient collective(s) carried (sparse: the union's rows + the 1-byte-per-Gaussian mask)"""
    la = vpr.last_allreduce
    if la["mode"] == "sparse":
        return la["rows"] * vpr._row_floats * 4 + vpr.N
    return vpr.grad_bytes() + (vpr.N if getattr(vpr, "sparse", False) else 0)


def time_allreduce(w, barrier, world, dev, reps=10):
    """the gradient all-reduce alone (device time, max over ranks, median of reps); 0 at N=1"""
    import torch.distributed as dist

    if world == 1:
        return 0.0
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier(); torch.cuda.synchronize()
        e0.record()
        w.vpr.all_reduce()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ts.append(float(t.item()))
    return statistics.median(ts)


def measure_e2e(args, w, barrier):
    """The metric through the public API with HOST buffers: every step copies the upstream gradient image from pinned
    host memory (H2D), renders + back-propagates through render_view(), and copies the rendered image to pinned host
    memory (D2H).  Measured twice: everything on the launching stream, and with the two copies on side streams."""
    import torch.distributed as dist

    vpr, mine, cams, c2ws_cpu, C, slot_of, dev, world = w.vpr, w.mine, w.cams, w.c2ws_cpu, w.C, w.slot_of, w.dev, w.world
    render_view = w.render_view
    v0 = mine[0]
    H, W = cams[v0].h, cams[v0].w
    h_c2w = c2ws_cpu[v0].clone().pin_memory()
    h_gout = w.gouts[v0].cpu().pin_memory()
    h_rgb = torch.empty(H, W, 3).pin_memory()
    d_gout = torch.empty_like(w.gouts[v0])

    def view_args(v):
        return (vpr.params["mean"], vpr.params["qvec"], vpr.params["svec"], vpr.params["alpha"],
                h_c2w if v == v0 else c2ws_cpu[v], cams[v])

    # The end-to-end number goes through the public API with its DEFAULTS -- render_view() waits for the duplicate count
    # (16 bytes) once per view -- unless --count-mode async asks otherwise.  (`auto` times the device-resident loops
    # without that wait; measured in the last run of round 2, the side-stream copy schedule hides completely in the
    # synchronous mode, 1.749 vs 1.746 ms, and not in the asynchronous one, 1.861 vs 1.772 ms.)
    e2e_async = (getattr(args, "count_mode", "auto") == "async")
    kw = dict(sh=vpr.params["sh"], C=C, grad_sink=vpr.grad_views, async_count=e2e_async)

    def e2e_step_serial():
        vpr.zero_grad()
        for v in mine:
            d_gout.copy_(h_gout, non_blocking=True)
            out = render_view(*view_args(v), slot=slot_of[v], **kw)
            out["rgb"].backward(gradient=d_gout)
            h_rgb.copy_(out["rgb"].detach(), non_blocking=True)
        vpr.all_reduce()

    # Same bytes, same calls, but the two copies ride their own streams: the upstream-gradient H2D of a view
    # overlaps that view's forward, the image D2H overlaps its backward (PCIe is full duplex; the copy engines
    # are independent of the SMs).  Every step still moves both buffers and the loop ends with all streams joined.
    cs_in, cs_out = torch.cuda.Stream(), torch.cuda.Stream()
    d_gout2 = [torch.empty_like(d_gout), torch.empty_like(d_gout)]
    ev_in = [torch.cuda.Event(), torch.cuda.Event()]
    ev_free = [torch.cuda.Event(), torch.cuda.Event()]
    ev_img = torch.cuda.Event()
    n_copy = [0]

    def e2e_step_pipelined():
        main = torch.cuda.current_stream()
        vpr.zero_grad()
        for v in mine:
            k = n_copy[0] & 1
            n_copy[0] += 1
            with torch.cuda.stream(cs_in):
                cs_in.wait_event(ev_free[k])  # the backward that last read this buffer is done
                d_gout2[k].copy_(h_gout, non_blocking=True)
                ev_in[k].record(cs_in)
            out = render_view(*view_args(v), slot=slot_of[v], **kw)
            rgb = out["rgb"]
            ev_img.record(main)
            with torch.cuda.stream(cs_out):
                cs_out.wait_event(ev_img)
                h_rgb.copy_(rgb.detach(), non_blocking=True)
            rgb.record_stream(cs_out)
            main.wait_event(ev_in[k])
            rgb.backward(gradient=d_gout2[k])
            ev_free[k].record(main)
        vpr.all_reduce()

    def e2e_measure(step_fn):
        for _ in range(3):
            step_fn()

        def joined():
            step_fn()

        runs_ = []
        for _ in range(N_LOOPS):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier(); torch.cuda.synchronize()
            e0.record()
            for _ in range(args.steps):
                joined()
            main = torch.cuda.current_stream()
            main.wait_stream(cs_in); main.wait_stream(cs_out)  # the step's copies belong to the timed region
            e1.record()
            torch.cuda.synchronize(); barrier()
            t2 = torch.tensor([e0.elapsed_time(e1) / args.steps], device=dev)
            if world > 1:
                dist.all_reduce(t2, op=dist.ReduceOp.MAX)
            runs_.append(float(t2.item()))
        return runs_

    serial_runs = e2e_measure(e2e_step_serial)
    mode, e2e_runs, pipe_err = "copies on the launching stream", serial_runs, None
    try:  # every rank takes the same branch: the failure modes (image check) are deterministic per build
        pipe_runs = e2e_measure(e2e_step_pipelined)
        torch.cuda.synchronize()
        # the image that reached the host must be the image the device holds
        v = mine[-1]
        with torch.no_grad():
            ref_img = render_view(*view_args(v), sh=vpr.params["sh"], C=C, slot=slot_of[v])["rgb"]
        img_diff = float((h_rgb.to(dev) - ref_img).abs().max())
        if img_diff != 0.0:
            raise RuntimeError(f"side-stream D2H image differs from the device image by {img_diff}")
        mode, e2e_runs = "copies on side streams (H2D under the forward, D2H under the backward)", pipe_runs
    except RuntimeError as ex:  # report the single-stream number rather than no number
        pipe_err = repr(ex)
    ms_e2e = statistics.median(e2e_runs)
    bi = len(mine) * (h_gout.numel() * 4 + 240)  # gradient image + the by-value camera struct
    bo = len(mine) * h_rgb.numel() * 4
    return {"value": w.n_views * w.scene.N * H * W / (ms_e2e / 1e3), "unit": UNIT, "ms_per_step": ms_e2e,
            "h2d_bytes_per_step": bi, "d2h_bytes_per_step": bo, "ms_per_step_all_runs": e2e_runs,
            "copy_schedule": mode, "count_mode": "async" if e2e_async else "sync",
            "ms_per_step_single_stream": statistics.median(serial_runs),
            "ms_per_step_single_stream_all_runs": serial_runs, "side_stream_error": pipe_err,
            "what": "render_view()+backward through the public API; per step: host camera pose (by-value kernel "
                    "argument) + pinned upstream gradient image H2D, rendered image D2H to pinned memory; Gaussian "
                    "parameters stay resident (they are the model state, like weights); median of five K-step loops"}


class _DeviceStdoutToStderr:
    """The reference extension's kernels `printf` from the device (~150 k lines per C3 comparison: the file-descriptor
    level stdout of the process).  bench.py's stdout contract is ONE JSON line, so fd 1 points at fd 2 while the
    extension runs; the device printf FIFO is drained (synchronize) before fd 1 comes back."""

    def __enter__(self):
        sys.stdout.flush()
        self._saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        try:
            if torch.cuda.is_available():
                torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            try:  # the CUDA runtime writes through C stdio: empty that buffer too while fd 1 still points away
                import ctypes
                ctypes.CDLL(None).fflush(None)
            except Exception:
                pass
            os.dup2(self._saved, 1)
            os.close(self._saved)
        return False


def reference_ext_comparison(w):
    """N=1, OUTSIDE every timed region: the UNMODIFIED reference `_gs` CUDA extension (oracle/_ref/_gs.so, rebuilt for
    sm_100 by oracle/build_ref.sh -- "the kernel to beat", SURVEY.md §0) and libgsb200.so through the same-signature
    ops on the workload's tensors: per-stage ms (median of CUDA-event timed launches)."""
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.exists(os.path.join(ref_dir, "_gs.so")):
        return {"unavailable": "oracle/_ref/_gs.so not built"}
    sys.path.insert(0, ref_dir)
    import _gs as ref

    from gsgen_b200.backend import _backend
    from gsgen_b200.culling import tile_culling_aabb_count
    from gsgen_b200.renderer import project_gaussians

    def timeit(fn, reps=7, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return statistics.median(ts)

    dev = w.dev
    sc = w.scene.to(dev)
    cam, c2w = w.cams[w.mine[0]], w.c2ws_cpu[w.mine[0]]
    C, H, W = w.C, cam.h, cam.w
    th, tw = cam.n_tiles
    normals, pts = cam.get_frustum(c2w)
    normals, pts = normals.to(dev), pts.to(dev)
    mask = torch.zeros(sc.N, dtype=torch.bool, device=dev)
    rmask = torch.zeros(sc.N, dtype=torch.bool, device=dev)
    res = {"what": "unmodified reference _gs ext (sm_100, -DNDEBUG) vs libgsb200 compat ops, same tensors, ms"}
    res["cull"] = {"ours": timeit(lambda: _backend.culling_gaussian_bsphere(sc.mean, sc.qvec, sc.svec, normals, pts, mask, 6.0)),
                   "reference": timeit(lambda: ref.culling_gaussian_bsphere(sc.mean, sc.qvec, sc.svec, normals, pts, rmask, 6.0))}
    m, q, s_ = sc.mean[mask].contiguous(), sc.qvec[mask].contiguous(), sc.svec[mask].contiguous()
    al, sh = sc.alpha[mask].contiguous(), sc.sh[mask].contiguous()
    c2w_d = c2w.to(dev)
    m2, c2, _, dp = project_gaussians(m, q, s_, c2w_d, True)
    m2, c2, dp = m2.contiguous(), c2.contiguous(), dp.contiguous()
    D, tl, br = tile_culling_aabb_count(m2, c2, 16, cam, 6.0)
    mk = lambda: (torch.zeros(D, dtype=torch.int32, device=dev), -torch.ones(th * tw, dtype=torch.int32, device=dev),
                  -torch.ones(th * tw, dtype=torch.int32, device=dev))
    ids, start, end = mk()
    rids, rstart, rend = mk()
    res["bin_sort"] = {"ours": timeit(lambda: _backend.tile_culling_aabb_start_end(tl, br, ids, start, end, dp, th, tw)),
                       "reference": timeit(lambda: ref.tile_culling_aabb_start_end(tl, br, rids, rstart, rend, dp, th, tw))}
    topleft = torch.tensor([-cam.cx / cam.fx, -cam.cy / cam.fy], device=dev)
    common = (16, th, tw, 1.0 / cam.fx, 1.0 / cam.fy, H, W)
    o, ro = torch.zeros(H * W * 3, device=dev), torch.zeros(H * W * 3, device=dev)
    res["sh_composite_fwd"] = {
        "ours": timeit(lambda: _backend.tile_based_vol_rendering_sh(m2, c2, sh, al, start, end, rids, o, topleft, c2w_d,
                                                                    *common, C, 1e-4)),
        "reference": timeit(lambda: ref.tile_based_vol_rendering_sh(m2, c2, sh, al, start, end, rids, ro, topleft, c2w_d,
                                                                    *common, C, 1e-4))}
    res["fwd_max_abs_diff"] = float((o - ro).abs().max())
    go = w.gouts[w.mine[0]].reshape(-1).contiguous()
    z = lambda: (torch.zeros_like(m2), torch.zeros_like(c2), torch.zeros_like(sh), torch.zeros_like(al))
    ga, gb = z(), z()
    res["sh_composite_bwd"] = {
        "ours": timeit(lambda: _backend.tile_based_vol_rendering_backward_sh(m2, c2, sh, al, start, end, rids, ro, *ga,
                                                                             go, topleft, c2w_d, *common, C, 1e-4)),
        "reference": timeit(lambda: ref.tile_based_vol_rendering_backward_sh(m2, c2, sh, al, start, end, rids, ro, *gb,
                                                                             go, topleft, c2w_d, *common, C, 1e-4),
                            reps=3, warm=1)}
    for k, v in res.items():
        if isinstance(v, dict) and "ours" in v:
            v["speedup"] = v["reference"] / v["ours"]
    return res


def run_ours(args):
    import ctypes
    import datetime

    import torch.distributed as dist

    from gsgen_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py --impl ours needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # a mismatched collective must fail fast, not burn GPU time until the default 10-minute watchdog (round 1 lost
        # ~80 GPU-minutes to one hang at N=8)
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=90))

    def barrier():
        if world > 1:
            dist.barrier()

    wl = args.workload
    w = Workload(args, wl, world, rank, dev)
    scene, cams, mine, vpr, C, n_views = w.scene, w.cams, w.mine, w.vpr, w.C, w.n_views
    H, W = cams[0].h, cams[0].w
    step = w.step

    # ---- warm-up (clock sampler already running)
    sampler = ClockSampler(local_rank if "CUDA_VISIBLE_DEVICES" not in os.environ else
                           int(os.environ["CUDA_VISIBLE_DEVICES"].split(",")[local_rank]), args.clock_period)
    if rank == 0 and args.clock_period > 0:
        sampler.start()
        time.sleep(0.5)
    warm_up(args, step, world, dev)
    ctxs = [_lib.ctx(dev, s) for s in w.slot_of.values()]
    hm = (ctypes.c_float * 6)()
    hc = (ctypes.c_int64 * 5)()

    # ---- timed region (the reported value): no instrumentation inside.  Five K-step loops; the MEDIAN is reported and
    # all five are listed (round 1 reported the fastest of three: the GPU boxes throttle the container's CPU in 100 ms CFS
    # slices and a throttled host shows up as a slow loop; the median of five is robust to two such loops, no picking).
    runs = timed_loops(args, step, barrier, world, dev, N_LOOPS, sampler, rank)
    all_runs_ms = [r[0] for r in runs]
    ms_max, mark0, mark1 = sorted(runs, key=lambda r: r[0])[N_LOOPS // 2]
    if args.dump_outputs and rank == 0:  # before anything below runs the step again or all-reduces its gradients
        dump_outputs(args.dump_outputs, w)
    if w.async_count:  # no view of the timed loops may have been truncated: the blocking check of every context
        from gsgen_b200._lib import TileListOverflow
        from gsgen_b200.rasterizer import view_stats

        for s_ in w.slot_of.values():
            try:
                view_stats(dev, s_)
            except TileListOverflow:
                w.overflows += 1
    ar_ms = time_allreduce(w, barrier, world, dev)
    # ---- the same K steps again with every stage bracketed by CUDA events on the launching stream
    # (gsb200_ctx_set_profiling).  Kept out of the headline loop because the bracketing perturbs it (reported).
    for c in ctxs:
        _lib.check(_lib.lib().gsb200_ctx_set_profiling(c, 1))
    step()
    torch.cuda.synchronize()
    for c in ctxs:
        _lib.check(_lib.lib().gsb200_ctx_get_profile(c, hm, hc, 1))
    ms_profiled = timed_loops(args, step, barrier, world, dev, 1)[0][0]

    # ---- stage profile of that loop (events recorded on the launching stream)
    stage_ms = [0.0] * 6
    counts = [0] * 5
    for c in ctxs:
        _lib.check(_lib.lib().gsb200_ctx_get_profile(c, hm, hc, 1))
        for i in range(6):
            stage_ms[i] += float(hm[i])
        for i in range(5):
            counts[i] += int(hc[i])
        _lib.check(_lib.lib().gsb200_ctx_set_profiling(c, 0))
    n_fwd = max(1, counts[0])
    D = counts[2] / n_fwd
    D_eff = counts[3] / n_fwd
    staged = counts[4] / n_fwd
    aux = w.last["aux"]
    N_vis = int(aux["mask"].sum().item())
    th, tw = cams[0].n_tiles
    ab = algorithmic_bytes(C, D, D_eff, N_vis, scene.N, th * tw, H, W)
    names = ["preprocess", "scan", "bin", "composite_fwd", "composite_bwd", "project_bwd"]
    peak, peak_src = measured_peaks()
    stages = {}
    for i, nm in enumerate(names):
        per = stage_ms[i] / n_fwd
        gbs = (ab[nm] / 1e9) / (per / 1e3) if per > 0 else None
        stages[nm] = {"ms": per, "alg_gbs": gbs, "frac_of_hbm_peak": (gbs / peak) if gbs else None}
    fwd_ms = stages["composite_fwd"]["ms"]
    achieved = (ab["composite_fwd"] / 1e9) / (fwd_ms / 1e3) if fwd_ms > 0 else 0.0
    ncu = ncu_numbers(wl)
    roofline = {"kernel": "k_composite_fwd<SH,C=%d>" % C, "bound": "hbm", "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "traffic": ncu.get("composite_fwd_dram_bytes"),
                "peak_source": peak_src, "alg_bytes_per_launch": ab["composite_fwd"], "avg_launch_ms": fwd_ms,
                "alg_bytes_formula": "D_eff*(4+4*(7+3C^2)) + 8*tiles + 16*H*W (SURVEY.md §8(d))"}
    try:  # (never at the price of the bench line)
        roofline.update(roofline_extras(C, N_vis, D_eff, th * tw, H, W, roofline["traffic"], fwd_ms, peak))
    except Exception as ex:
        roofline["extras_error"] = repr(ex)

    # ---- end to end through the public API with host buffers (pinned): per step H2D of the step's inputs
    # (camera pose + upstream gradient image) and D2H of the rendered image
    e2e = None
    if not args.no_e2e:
        try:
            e2e = measure_e2e(args, w, barrier)
        except Exception as ex:  # the bench line must still print; every rank takes the same branch
            e2e = {"value": None, "unit": UNIT, "error": repr(ex)}

    # ---- C4 (north_star's multi-GPU configuration: 500k Gaussians, 8 orbit views 800^2, sharded over the ranks, ONE
    # all-reduce per step): strong scaling sub-record, measured in every default run so that the driver's N=1,2,4,8
    # sweep captures it next to the C3 weak-scaling headline.
    c4 = None
    if wl == "c3" and not args.no_c4_strong and args.svec_scale == 1.0:
        try:
            # the SAME count mode at every N, so that ms(N=1) / ms(N) compares like with like (`auto` would time N = 1
            # asynchronously and N > 1 synchronously); with 8 views per step the host wait is diluted anyway
            w4 = Workload(args, "c4", world, rank, dev,
                          count_mode=("sync" if args.count_mode == "auto" else args.count_mode))
            for _ in range(5):
                w4.step()
            torch.cuda.synchronize()
            r4 = timed_loops(args, w4.step, barrier, world, dev, N_LOOPS)
            ms4 = sorted(x[0] for x in r4)[N_LOOPS // 2]
            cam4 = w4.cams[0]
            c4 = {"workload": workload_name("c4", w4.scene, cam4), "scaling": "strong", "views_per_step": 8,
                  "views_per_gpu": len(w4.mine), "count_mode": w4.count_mode, "ms_per_step": ms4,
                  "ms_per_step_all_runs": [x[0] for x in r4],
                  "value": 8 * w4.scene.N * cam4.h * cam4.w / (ms4 / 1e3), "unit": UNIT,
                  "grad_allreduce_bytes": allreduce_bytes(w4.vpr) if world > 1 else 0,
                  "allreduce": dict(w4.vpr.last_allreduce, of=w4.scene.N) if world > 1 else None,
                  "allreduce_ms": time_allreduce(w4, barrier, world, dev),
                  "allreduce_buffer": w4.vpr.grad_buffer_kind, "tile_list_overflows": w4.overflows,
                  "note": "speed-up over N=1 = ms_per_step(N=1) / ms_per_step(N); north_star target >= 6x at N=8"}
            del w4
            torch.cuda.empty_cache()
        except Exception as ex:
            c4 = {"error": repr(ex)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    time.sleep(0.1)
    clocks = sampler.stop(mark0, mark1)
    # issue-slot roofline of the forward composite (the limiter that is actually active, DESIGN.md §3.3): executed warp
    # instructions of the committed ncu capture / (SMs x 4 schedulers x SM clock)
    inst = ncu.get("composite_fwd_warp_inst")
    sm_mhz = clocks.get("sm_mhz") or 1965.0
    issue = None
    if inst:
        t_issue = inst / (148 * 4 * sm_mhz * 1e6) * 1e3
        issue = {"warp_instructions": inst, "sm_mhz": sm_mhz, "min_ms_at_full_issue": t_issue,
                 "frac": t_issue / fwd_ms if fwd_ms > 0 else None,
                 "source": ncu.get("source", "profiles/traffic.json")}
    roofline["issue_roofline"] = issue
    try:  # (never at the price of the bench line)
        roofline["dominant_kernel"] = dominant_kernel_roofline(stages, ab, ncu, peak, sm_mhz)
    except Exception as ex:
        roofline["dominant_kernel"] = {"error": repr(ex)}
    cpu_base = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            cpu_base = run_cpu_baseline(args)
        except Exception as e:  # the bench line must still print
            cpu_base = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e}"}
    ref_ext = None
    if world == 1 and not args.no_ref_ext:
        try:
            with _DeviceStdoutToStderr():
                ref_ext = reference_ext_comparison(w)
        except Exception as e:
            ref_ext = {"error": repr(e)}
    value = n_views * scene.N * H * W / (ms_max / 1e3)
    # preprocess, fill, emit_tiles, (pad_keys), tile_ranges, composite_fwd, composite_bwd, project_bwd
    my_kernels_per_view = 7 + (1 if w.async_count else 0)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_max, "higher_is_better": True, "scaling": "strong" if wl == "c4" else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(wl, scene, cams[0]), "views_per_step": n_views,
                   "views_per_gpu": len(mine), "parallelism": f"view-dp{world}",
                   "grad_allreduce_bytes": allreduce_bytes(vpr) if world > 1 else 0,
                   "grad_allreduce_dense_bytes": vpr.grad_bytes() if world > 1 else 0,
                   "allreduce": dict(vpr.last_allreduce, of=scene.N) if world > 1 else None,
                   "allreduce_buffer": vpr.grad_buffer_kind if world > 1 else None,
                   "count_mode": w.count_mode,
                   "l2": "no explicit flush: inputs larger than L2 -- per step %.0f MB of Gaussian parameters + as many "
                         "gradients + %.0f MB of sort keys/ids stream through the 126 MB L2"
                         % (vpr.grad_bytes() / 1e6, D * 12 / 1e6)},
        "clocks": clocks,
        "e2e": e2e,
        "gpu_launches": my_kernels_per_view * len(mine) * args.steps,
        "library_launches_note": "plus cub::DeviceScan (2 kernels), 2x cub::DeviceRadixSort onesweep (6 + 4 kernels) and 2 memsets per view",
        "roofline": roofline,
        "stages": stages,
        "allreduce_ms": ar_ms,
        "ms_per_step_with_stage_events": ms_profiled,
        "ms_per_step_all_runs": all_runs_ms,
        "ms_per_step_statistic": "median of five K-step loops",
        "tile_list_overflows": w.overflows,
        "view_stats": {"N_visible": N_vis, "N_with_dub": D, "D_eff": D_eff, "entries_staged_fwd": staged,
                       "tiles": th * tw},
        # SURVEY.md §8(d) number (2): tile-list pairs P = sum_tiles (end - start) * 256 = N_with_dub * 256 per view,
        # identical for the reference and for us when the binning matches (it is bit-exact)
        "tile_list_pairs_per_s": n_views * D * 256.0 / (ms_max / 1e3),
        "c4_strong": c4,
        "cpu_baseline": cpu_base,
        "vs_reference_ext": ref_ext,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
