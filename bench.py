#!/usr/bin/env python
"""bench.py -- rendered MP/s (fwd+bwd) of the mvpraymarch hot path on N B200s.

Metric (BASELINE.json): rendered megapixels (rays) per second, forward + backward, on synthetic
80-view 1024x667 batches of a K=16384, 8^3-voxel subject (SURVEY.md section 8d, config C3), sharded over ranks by
views with one NCCL all-reduce of the primitive gradients per step (section 8e).  One "step" = one
forward + backward pass of the raymarcher over ALL 80 views (strong scaling: the 80 views are split over ranks).

    python bench.py [--gpus N --steps K --warmup W]                 # our CUDA path, N=1 default
    torchrun ... bench.py --gpus N --steps K --warmup W             # N>1: one rank per GPU
    python bench.py --impl reference ...                            # the reference's own CPU autograd path

JSON line keys: the base contract's + "roofline" (dominant kernel), "roofline_forward", "cpu_baseline", "e2e",
"clocks", "gpu_launches".  `oracle/` is only touched in the cpu_baseline / --impl reference legs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

# canonical workload (SURVEY.md section 8d, C3/C4/C5)
VIEWS, H, W, K, T = 80, 1024, 667, 16384, 8
ALPHA_MU, ALPHA_SIGMA = 17.0, 6.0   # ~50 % of the object rays saturate (SURVEY 8d), measured 0.135 / 0.275


_T0 = time.time()


def log(msg):
    """progress to stderr (stdout carries only the JSON line)"""
    print("[bench %7.1fs] %s" % (time.time() - _T0, msg), file=sys.stderr, flush=True)


def algorithmic_bytes(n_views, h, w, k, t):
    """SURVEY.md section 8d: compulsory traffic per pass (every input read once, every output written once)."""
    tpl = k * t ** 3 * 16
    srt = k * 60
    aabb = (2 * k - 1) * 24
    rays_in = h * w * 32
    out = h * w * 28
    fwd = tpl + srt + rays_in + out + aabb
    bwd = (tpl + srt + aabb + rays_in) + h * w * 28 + (tpl + srt)
    return n_views * fwd, n_views * bwd


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU autograd path (mvpraymarch.py:567-633 restated in oracle/torch_ref.py)
# ----------------------------------------------------------------------------------------------------------------
def cpu_autograd_sample(hh=96, ww=64, k=64, t=8, steps=1, warmup=0):
    """Bounded sample of the same kind of workload (head scene, dome camera) on the host cores.
    Returns (MP/s fwd+bwd, seconds per step, description)."""
    from ava256_b200 import scene
    from oracle import torch_ref
    # the loop is ~10^4 small ATen ops: beyond ~16 threads the fork/join cost dominates and it gets slower
    torch.set_num_threads(min(os.cpu_count() or 1, 16))
    s = scene.make_scene(1, hh, ww, k, t, alpha_mu=ALPHA_MU, alpha_sigma=ALPHA_SIGMA)
    stepsize = 2.0 / 16.0          # SURVEY 8d: keeps the autograd graph at ~16 steps
    g = torch.randn(1, hh, ww, 4, generator=torch.Generator().manual_seed(1))
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        torch_ref.raymarch_torch_fwd_bwd(s["raypos"], s["raydir"], stepsize, s["tminmax"], s["primpos"], s["primrot"],
                                         s["primscale"], s["template"], g)
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    sec = sum(times) / len(times)
    desc = "PyTorch autograd raymarch loop (reference mvpraymarch.py:567-633 restated), 1 view %dx%d, K=%d, %d^3, dt=2/16, fp32" % (hh, ww, k, t)
    return hh * ww / sec / 1e6, sec, desc


def workload_config(views, h, w, k, t):
    """`config` of the JSON line: names the workload only, so that both arms (ours, --impl reference) print the same dict."""
    return {"workload": "C3: %d views %dx%d, K=%d, %d^3 RGBA, dt=1/256, one subject (template materialised per view), "
                        "fwd+bwd of the mvpraymarch op" % (views, h, w, k, t),
            "views": views, "height": h, "width": w, "prims": k, "voxels": t,
            "l2": "inputs (%.1f GB template) larger than the 126 MB L2; no explicit flush" % (views * k * t ** 3 * 16 / 1e9)}


def run_reference(args, rank):
    """The reference's own CPU implementation of the path (its PyTorch autograd loop) on the host cores.  Every step is a
    BOUNDED SAMPLE of the workload -- a reduced C1 (1 view 96x64, K=64, 8^3, 16 steps per ray): true C1 (128x128, K=256) takes
    ~40 s per step and runs once in the default arm's `cpu_baseline` leg instead."""
    if rank != 0:
        return
    mps, sec, desc = cpu_autograd_sample(steps=args.steps, warmup=args.warmup)
    cores = torch.get_num_threads()
    line = {
        "impl": "reference", "metric": "rendered MP/s (fwd+bwd)", "value": mps, "unit": "MP/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.views, args.height, args.width, args.prims, args.voxels),
        "sample": "reduced C1: " + desc,
        "cpu_baseline": {"value": mps, "unit": "MP/s", "cores": cores, "kind": "port", "sample": "reduced C1: " + desc},
        "e2e": {"value": mps, "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------
# checker legs of our arm (rank 0, N=1): the UNMODIFIED reference CUDA extension (oracle/_ref, prebuilt) on the same scene
# ----------------------------------------------------------------------------------------------------------------
def ref_cuda_leg(s, stepsize, grad_out, out, grads, chunk=16, reps=7, warm=2):
    """Times the reference kernels (compiled for sm_100 from the reference's sources by oracle/build_ref.py) on the tensors
    the timed region just used, and compares view 0.  The reference launches on legacy stream 0 (= torch's default stream)
    and cudaMalloc/cudaFree's inside compute_aabb (bvh.cu:261-293), so every call is bracketed by device-wide syncs;
    views go in chunks (its int32 strides overflow at N*K*T^3*4 >= 2^31, primsampler.h:31-36).  Returns
    (ref_cuda_baseline dict, parity_check dict) or (None, None) when the extension did not travel to this box."""
    from tests import refext
    if not refext.available():
        return None, None
    m = refext.module()
    names = ("primpos", "primrot", "primscale", "template")
    nv = s["raypos"].shape[0]
    hh, ww = s["raypos"].shape[1:3]
    k = s["primpos"].shape[1]
    dev = s["raypos"].device
    slab = s["template"][0, 0].numel()
    chunk = max(1, min(chunk, nv, (2 ** 31 - 1) // (k * slab)))
    bounds = [(i, min(i + chunk, nv)) for i in range(0, nv, chunk)]
    tree = refext._tree(chunk, k, dev)
    aabb = torch.empty((chunk, 2 * k - 1, 2, 3), device=dev)
    rgba = torch.empty((chunk, hh, ww, 4), device=dev)
    rsat = torch.empty((chunk, hh, ww, 3), device=dev)
    gbuf = [torch.empty_like(s[n][:chunk]) for n in names]

    def ev():
        return torch.cuda.Event(enable_timing=True)

    def one_pass(keep_first=False):
        ta = tf = tb = 0.0
        first = None
        for (a0, a1) in bounds:
            c = a1 - a0
            v = {n: s[n][a0:a1] for n in ("raypos", "raydir", "tminmax") + names}
            so, nc, na = tree[0][:c], tree[1][:c], tree[2][:c]
            rsat[:c].fill_(-1.0)                                   # mvpraymarch.py:147-148 (not timed: torch glue)
            for g_ in gbuf:
                g_[:c].zero_()                                     # mvpraymarch.py:240-246 (not timed)
            torch.cuda.synchronize()
            ea, e0, e1, e2 = ev(), ev(), ev(), ev()
            ea.record()
            m.compute_aabb(v["primpos"], v["primrot"], v["primscale"], so, nc, na, aabb[:c], 0)
            e0.record()
            m.raymarch_forward(v["raypos"], v["raydir"], stepsize, v["tminmax"], so, nc, aabb[:c], v["primpos"], v["primrot"],
                               v["primscale"], v["template"], None, rgba[:c], rsat[:c], None, 0, False, 512, True, True, 8.0, 8.0,
                               0, 0.0, 3, 8, 16)
            e1.record()
            m.raymarch_backward(v["raypos"], v["raydir"], stepsize, v["tminmax"], so, nc, aabb[:c], v["primpos"], gbuf[0][:c],
                                v["primrot"], gbuf[1][:c], v["primscale"], gbuf[2][:c], v["template"], gbuf[3][:c], None, None,
                                rgba[:c], grad_out[a0:a1], rsat[:c], None, 0, False, 512, True, True, 8.0, 8.0, 0, 0.0, 3, 8, 16)
            e2.record()
            torch.cuda.synchronize()
            ta += ea.elapsed_time(e0)
            tf += e0.elapsed_time(e1)
            tb += e1.elapsed_time(e2)
            if keep_first and first is None:
                first = (rgba[0].clone(), rsat[0].clone(), [g_[0].clone() for g_ in gbuf])
        return ta, tf, tb, first

    first = None
    for i in range(warm):
        _, _, _, f_ = one_pass(keep_first=(i == 0))
        first = first or f_
    tas, tfs, tbs = [], [], []
    for _ in range(reps):
        ta, tf, tb, _ = one_pass()
        tas.append(ta)
        tfs.append(tf)
        tbs.append(tb)
    tas.sort()
    tfs.sort()
    tbs.sort()
    aab, fwd, bwd = tas[len(tas) // 2] / nv, tfs[len(tfs) // 2] / nv, tbs[len(tbs) // 2] / nv
    base = {"what": "unmodified reference CUDA extension (oracle/_ref, -arch=sm_100 -use_fast_math), same scene and tensors, "
                    "%d views in chunks of %d; raymarch_forward and raymarch_backward kernels timed alone with CUDA events, "
                    "compute_aabb (with its cudaMalloc / cudaFree, bvh.cu:261-293) separately; its torch allocations and zero-fills "
                    "not timed; median of %d passes after %d warm-ups" % (nv, chunk, reps, warm),
            "fwd_ms_per_view": fwd, "bwd_ms_per_view": bwd, "aabb_ms_per_view": aab,
            "mps": hh * ww / ((fwd + bwd) * 1e-3) / 1e6, "mps_with_aabb": hh * ww / ((aab + fwd + bwd) * 1e-3) / 1e6,
            "fwd_ms_per_view_minmax": [tfs[0] / nv, tfs[-1] / nv], "bwd_ms_per_view_minmax": [tbs[0] / nv, tbs[-1] / nv],
            "aabb_ms_per_view_minmax": [tas[0] / nv, tas[-1] / nv]}

    def rel(a, b):
        return float((a - b).abs().max()) / max(float(b.abs().max()), 1e-30)

    r_rgba, r_sat, r_g = first
    check = {"against": "reference CUDA extension (oracle/_ref), view 0 of the timed tensors",
             "fwd": rel(out[0], r_rgba),
             "satmask_mismatch_frac": float(((r_sat[..., 0] > -1.0) != (out[0][..., 3] >= 1.0)).float().mean()),
             "saturated_frac": float((r_sat[..., 0] > -1.0).float().mean()),
             "grads": {n: rel(g_[0], r_) for n, g_, r_ in zip(names, grads, r_g)},
             "gates": {"fwd": 1e-4, "satmask_mismatch_frac": 1e-4, "grads": 1e-3}}
    check["ok"] = bool(check["fwd"] <= 1e-4 and check["satmask_mismatch_frac"] <= 1e-4 and all(v <= 1e-3 for v in check["grads"].values()))
    return base, check


# ----------------------------------------------------------------------------------------------------------------
# --dump-outputs: the outputs of the timed path, so that two builds can be compared output for output
# ----------------------------------------------------------------------------------------------------------------
DUMP_BYTES = 62_000_000        # all arrays together; with the .npy headers the files stay under 64 MB


def sample_outputs(arrays, budget=DUMP_BYTES, seed=1112):
    """Host float32 copies of the device tensors `arrays` (name -> tensor) within `budget` bytes.  Arrays are taken in order of
    size, each whole if it fits its share of what is left, otherwise as a fixed, seeded sample of its rows (the last axis
    kept whole: RGBA of a pixel or a voxel), sorted by row index -- the same rows in every run with the same arguments."""
    out = {}
    left = budget
    names = sorted(arrays, key=lambda n: arrays[n].numel())
    for i, name in enumerate(names):
        x = arrays[name].detach().float()
        share = left // (len(names) - i)
        if x.numel() * 4 > share:
            rows = x.reshape(-1, x.shape[-1])
            g = torch.Generator().manual_seed(seed + i)
            idx = torch.randint(rows.shape[0], (share // (rows.shape[1] * 4),), generator=g).unique()
            x = rows[idx.to(rows.device)]
        out[name] = x.cpu().numpy()
        left -= out[name].nbytes
    return out


def write_outputs(outdir, arrays):
    import numpy as np
    os.makedirs(outdir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(outdir, name + ".npy"), a)
    log("outputs of the last timed step written to %s (%s)" % (outdir, ", ".join("%s %s" % (n, list(a.shape)) for n, a in arrays.items())))


# ----------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------
def run_ours(args, rank, world):
    from ava256_b200 import lib, parallel, scene
    from ava256_b200.op import mvpraymarch, mvpraymarch_camera
    import ctypes

    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    views, h, w, k, t = args.views, args.height, args.width, args.prims, args.voxels
    assert views % world == 0, "views must divide over ranks"
    nv = views // world                      # contiguous block of views per rank (SURVEY 8e)
    # views are interleaved over the ranks (rank, rank + world, ...): equal coverage per rank (parallel.rank_views)
    vids = parallel.rank_views(views, rank, world, interleave=not args.contiguous_views)
    s = scene.make_scene(nv, h, w, k, t, seed=1112, view_ids=vids, device=dev, alpha_mu=ALPHA_MU, alpha_sigma=ALPHA_SIGMA)
    stepsize = s["stepsize"]
    log("scene ready: %d views/rank %dx%d K=%d T=%d" % (nv, h, w, k, t))
    gen = torch.Generator(device=dev).manual_seed(1112 + rank)
    grad_out = torch.randn(nv, h, w, 4, device=dev, generator=gen)
    leaves = [s[n].requires_grad_(True) for n in ("primpos", "primrot", "primscale", "template")]
    # all-reduced primitive gradients of the subject: double-buffered, the NCCL all-reduce of step i runs under the
    # forward of step i+1 (parallel.GradReducer); every all-reduce is waited for inside the timed region
    red = parallel.GradReducer(k, t, t, t, dev)
    flat = red.bufs[0]
    flat_numel = flat.numel()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        """Returns the images and the flat buffer the subject's (all-reduced) primitive gradients go to."""
        for x in leaves:
            x.grad = None
        out = mvpraymarch(s["raypos"], s["raydir"], stepsize, s["tminmax"], (leaves[0], leaves[1], leaves[2]), leaves[3], None)
        out.backward(grad_out)
        # views of a step share the subject's primitives: local sum over the rank's views, one all-reduce (SURVEY 8e)
        return out, red.reduce(leaves[3].grad, leaves[0].grad, leaves[1].grad, leaves[2].grad)

    for i in range(args.warmup):
        out, _ = step()
        red.finish()
        torch.cuda.synchronize()
        log("warmup step %d done" % i)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        out, out_flat = step()
    red.finish()                 # the compute stream waits for the last all-reduce: it is inside the timed region
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    dump = None
    if args.dump_outputs and rank == 0:
        # what the caller of the timed path receives from its last step: rank 0's images and the subject's reduced gradients
        g_tpl, g_pos, g_rot, g_scale = red.views(out_flat, k, t, t, t)
        dump = sample_outputs({"rayrgba": out.detach(), "grad_template": g_tpl, "grad_primpos": g_pos,
                               "grad_primrot": g_rot, "grad_primscale": g_scale})
    # the collective alone (not overlapped), for the record
    allreduce_ms = None
    if world > 1:
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ea.record()
        for _ in range(5):
            dist.all_reduce(red.bufs[1])
        eb.record()
        barrier()
        ta = torch.tensor([ea.elapsed_time(eb) / 5], device=dev)
        dist.all_reduce(ta, op=dist.ReduceOp.MAX)
        allreduce_ms = float(ta.item())
    log("timed region: %.1f ms for %d steps" % (ms, args.steps))
    clocks = sampler.stop() if rank == 0 else None
    if dump is not None:
        write_outputs(args.dump_outputs, dump)
    tms = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms_step = float(tms.item()) / args.steps
    rank_ms = [ms / args.steps]
    if world > 1:                   # per-rank step times: imbalance between the ranks' view sets is visible in the record
        allms = [torch.zeros(1, device=dev) for _ in range(world)]
        dist.all_gather(allms, torch.tensor([ms / args.steps], device=dev))
        rank_ms = [float(x.item()) for x in allms]
    value = views * h * w / (ms_step * 1e-3) / 1e6
    sat_frac = float((out[..., 3] >= 0.999).float().mean())
    cover = float((out[..., 3] > 0).float().mean())

    # ---- kernel-only timing for the roofline (CUDA events on the launching stream; accel already built) ----
    N_, H_, W_ = s["raypos"].shape[:3]
    wsb = lib.workspace_bytes(N_, H_, W_, k, t, t, t)
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    rgba = torch.empty(N_, H_, W_, 4, device=dev)
    rsat = torch.empty(N_, H_, W_, 3, device=dev)
    raux = torch.empty(N_, H_, W_, 4, dtype=torch.int32, device=dev)
    fa = lib.ForwardArgs()
    fa.shape = lib.Shape(N_, H_, W_, k, t, t, t)
    fa.stepsize, fa.fadescale, fa.fadeexp, fa.flags = stepsize, 8.0, 8.0, 0
    P = lambda x: ctypes.c_void_p(x.data_ptr())  # noqa: E731
    tl = [x.detach() for x in leaves]
    clear_gb = sum(g.numel() for g in tl) * 4 / 1e9
    fa.raypos, fa.raydir, fa.tminmax = P(s["raypos"]), P(s["raydir"]), P(s["tminmax"])
    fa.primpos, fa.primrot, fa.primscale, fa.tplate = P(tl[0]), P(tl[1]), P(tl[2]), P(tl[3])
    fa.rayrgba, fa.raysat, fa.rayaux, fa.workspace, fa.workspace_bytes = P(rgba), P(rsat), P(raux), P(ws), wsb
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    lib.check(lib.LIB.mvp_raymarch_forward(ctypes.byref(fa), stream))          # builds accel
    fa.flags = lib.FLAG_ACCEL_VALID
    gs = [torch.zeros_like(x) for x in tl]
    # the timed forward is the one the op runs: it also zero-fills the backward's gradient buffers on the side
    fa.clear_grad_primpos, fa.clear_grad_primrot, fa.clear_grad_primscale, fa.clear_grad_tplate = P(gs[0]), P(gs[1]), P(gs[2]), P(gs[3])
    ba = lib.BackwardArgs()
    ba.shape, ba.stepsize, ba.fadescale, ba.fadeexp, ba.flags = fa.shape, stepsize, 8.0, 8.0, lib.FLAG_ACCEL_VALID
    ba.raypos, ba.raydir, ba.tminmax = fa.raypos, fa.raydir, fa.tminmax
    ba.primpos, ba.primrot, ba.primscale, ba.tplate = fa.primpos, fa.primrot, fa.primscale, fa.tplate
    ba.grad_rayrgba, ba.raysat, ba.rayaux = P(grad_out), P(rsat), P(raux)
    ba.grad_primpos, ba.grad_primrot, ba.grad_primscale, ba.grad_tplate = P(gs[0]), P(gs[1]), P(gs[2]), P(gs[3])
    ba.workspace, ba.workspace_bytes = P(ws), wsb

    def time_kernel(fn, reps):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    reps = max(2, min(args.steps, 5))
    fwd_ms = time_kernel(lambda: lib.check(lib.LIB.mvp_raymarch_forward(ctypes.byref(fa), stream)), reps)
    bwd_ms = time_kernel(lambda: lib.check(lib.LIB.mvp_raymarch_backward(ctypes.byref(ba), stream)), reps)
    # the same two launches with the rays generated in the kernels' prologue from the camera parameters (mvp_camera) instead of read
    cams_dev = [c_.to(dev) for c_ in scene.make_cameras(nv, h, w, view_ids=vids)]
    cam_struct = lib.Camera(P(cams_dev[0]), P(cams_dev[1]), P(cams_dev[2]), P(cams_dev[3]), scene.VOLRADIUS, 0)
    fa.camera, ba.camera = cam_struct, cam_struct
    fa.raypos = fa.raydir = fa.tminmax = ba.raypos = ba.raydir = ba.tminmax = None
    fa.flags = 0
    lib.check(lib.LIB.mvp_raymarch_forward(ctypes.byref(fa), stream))          # accel from the camera
    fa.flags = lib.FLAG_ACCEL_VALID
    fwd_cam_ms = time_kernel(lambda: lib.check(lib.LIB.mvp_raymarch_forward(ctypes.byref(fa), stream)), reps)
    bwd_cam_ms = time_kernel(lambda: lib.check(lib.LIB.mvp_raymarch_backward(ctypes.byref(ba), stream)), reps)
    del gs, ws
    log("kernel-only: fwd %.2f ms, bwd %.2f ms per launch (%d views)" % (fwd_ms, bwd_ms, nv))

    # ---- second configuration (not the headline, SURVEY 8e "optional fast path"): the subject's primitives passed ONCE,
    # [1,K,...], shared by all views of the rank -- nothing is replicated in HBM, no 10.7 GB zero-fill, no view-sum; the
    # gradients of all views accumulate into the one set, which is what the all-reduce needs anyway ----
    shared_cfg = None
    if not args.no_shared_leg:
        sh = [x.detach()[:1].clone().requires_grad_(True) for x in leaves]

        def shared_step():
            for x in sh:
                x.grad = None
            o_ = mvpraymarch(s["raypos"], s["raydir"], stepsize, s["tminmax"], (sh[0], sh[1], sh[2]), sh[3], None)
            o_.backward(grad_out)
            if world > 1:
                fl = torch.cat([sh[3].grad.reshape(-1), sh[0].grad.reshape(-1), sh[1].grad.reshape(-1), sh[2].grad.reshape(-1)])
                dist.all_reduce(fl)
            return o_

        o_sh = shared_step()
        same = bool(torch.equal(o_sh.detach(), out.detach()))
        barrier()
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        nsh = max(2, min(args.steps, 10))
        ea.record()
        for _ in range(nsh):
            shared_step()
        eb.record()
        barrier()
        tsh = torch.tensor([ea.elapsed_time(eb) / nsh], device=dev)
        if world > 1:
            dist.all_reduce(tsh, op=dist.ReduceOp.MAX)
        shared_cfg = {"what": "same views, the subject's primitives passed once as [1,K,...] (MVP_FLAG_SHARED_PRIMS): no per-view "
                              "copies, gradients of all views accumulate into one set; NOT the headline configuration",
                      "ms_per_step": float(tsh.item()), "value": views * h * w / (float(tsh.item()) * 1e-3) / 1e6, "unit": "MP/s",
                      "images_identical_to_headline_config": same}
        del sh, o_sh
        log("shared-primitive configuration: %.2f ms per step" % shared_cfg["ms_per_step"])

    # ---- third configuration (not the headline either): rays generated inside the render kernels from the camera parameters
    # (SURVEY 8f row 1, op.mvpraymarch_camera): raypos / raydir / tminmax never exist, no camera fit over a ray field ----
    camera_cfg = None
    if not args.no_shared_leg:
        def camera_step():
            for x in leaves:
                x.grad = None
            o_ = mvpraymarch_camera(cams_dev[0], cams_dev[1], cams_dev[2], cams_dev[3], (w, h), scene.VOLRADIUS, stepsize,
                                    (leaves[0], leaves[1], leaves[2]), leaves[3], None)
            o_.backward(grad_out)
            red.reduce(leaves[3].grad, leaves[0].grad, leaves[1].grad, leaves[2].grad)
            return o_

        o_cam = camera_step()
        red.finish()
        torch.cuda.synchronize()
        # the bench scene's ray tensors come from the torch formula on the host (scene.compute_raydirs_host), the kernels' rays from
        # the reference kernel's arithmetic: last-place differences in the rays, so the images agree closely but not bit for bit
        # (bit identity holds against rays from mvp_compute_raydirs: tests/test_gpu_camera_rays.py)
        cam_img_diff = float((o_cam.detach() - out.detach()).abs().max()) / max(float(out.detach().abs().max()), 1e-30)
        barrier()
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ncm = max(2, min(args.steps, 10))
        ea.record()
        for _ in range(ncm):
            camera_step()
        red.finish()
        eb.record()
        barrier()
        tcm = torch.tensor([ea.elapsed_time(eb) / ncm], device=dev)
        if world > 1:
            dist.all_reduce(tcm, op=dist.ReduceOp.MAX)
        camera_cfg = {"what": "same views and per-view primitives as the headline, the rays generated in the render kernels' prologue from "
                              "(viewpos, viewrot, focal, princpt) (mvp_camera; reference: compute_raydirs, utils_kernel.cu:32-46) instead of "
                              "read from raypos / raydir / tminmax; NOT the headline configuration",
                      "ms_per_step": float(tcm.item()), "value": views * h * w / (float(tcm.item()) * 1e-3) / 1e6, "unit": "MP/s",
                      "image_max_rel_diff_vs_host_formula_rays": cam_img_diff,
                      "kernel_ms": {"forward_all_views_per_rank": fwd_cam_ms, "backward_all_views_per_rank": bwd_cam_ms}}
        del o_cam
        out, _ = step()              # the leaves' gradients are those of the headline configuration again (the parity leg reads them)
        red.finish()
        torch.cuda.synchronize()
        log("camera-ray configuration: %.2f ms per step (kernels %.2f + %.2f)" % (camera_cfg["ms_per_step"], fwd_cam_ms, bwd_cam_ms))

    # ---- checker legs (rank 0, single GPU): reference CUDA kernels on the same tensors: timing + parity of view 0 ----
    ref_cuda = parity = None
    if world == 1 and not args.no_check:
        ref_cuda, parity = ref_cuda_leg(s, stepsize, grad_out, out.detach(), [x.grad for x in leaves])
        if ref_cuda is not None:
            log("reference CUDA kernels: fwd %.3f / bwd %.3f ms per view; parity ok=%s" % (ref_cuda["fwd_ms_per_view"], ref_cuda["bwd_ms_per_view"], parity["ok"]))
        else:
            log("reference CUDA extension (oracle/_ref) not on this box: no ref_cuda_baseline / parity_check")

    # ---- end-to-end through the public op with HOST buffers (pinned): H2D of the step's inputs, D2H of the results ----
    # The host hands over, every step: the rays of all views, one subject's primitives/payload and the image
    # gradient; it gets back the rendered images and the view-summed (all-reduced) primitive gradients.  Views are
    # streamed in chunks: H2D of chunk i+1 (copy stream) overlaps fwd+bwd of chunk i (compute stream) and D2H of chunk
    # i-1 (second copy stream) -- all inside the timed region.
    e2e = e2e_cam = None
    if not args.no_e2e:
        host_in = {n: s[n].detach().cpu().pin_memory() for n in ("raypos", "raydir", "tminmax")}
        host_prim = {n: x.detach()[0].cpu().pin_memory() for n, x in zip(("primpos", "primrot", "primscale", "template"), leaves)}
        host_grad = grad_out.cpu().pin_memory()
        host_out = torch.empty(nv, h, w, 4).pin_memory()
        host_flat = torch.empty(flat.numel()).pin_memory()
        h2d = sum(x.numel() * 4 for x in host_in.values()) + sum(x.numel() * 4 for x in host_prim.values()) + host_grad.numel() * 4
        d2h = host_out.numel() * 4 + host_flat.numel() * 4
        # device staging: two full sets (rays, image gradient, the subject's primitives, the reduced-gradient buffer), so the
        # uploads of step i+1 run while step i computes and the downloads of step i run under step i+1
        dev_in = [{n: s[n] for n in host_in}, {n: torch.empty_like(s[n]) for n in host_in}]
        dev_grad = [grad_out, torch.empty_like(grad_out)]
        names = ("primpos", "primrot", "primscale", "template")
        del leaves, tl
        torch.cuda.empty_cache()
        dev_prim = [{n: torch.empty(host_prim[n].shape, device=dev) for n in names} for _ in range(2)]
        flats = red.bufs
        chunk = max(1, min(nv, args.e2e_chunk))
        bounds = [(i, min(i + chunk, nv)) for i in range(0, nv, chunk)]
        s_in, s_out, s_cmp = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.current_stream()
        cmp_done, flat_out_done = [None, None], [None, None]

        from ava256_b200.payload import expand_views, sum_views
        host_cam = [t.pin_memory() for t in scene.make_cameras(nv, h, w, view_ids=vids)]
        dev_cam = [[torch.empty(t.shape, device=dev) for t in host_cam] for _ in range(2)]

        def e2e_step(i, cams=False):
            """cams=False: the host hands over the rays themselves.  cams=True: it hands over the camera parameters (what
            models/autoencoder.py:240 gives compute_raydirs) and the render kernels generate the rays (op.mvpraymarch_camera)."""
            b_ = i & 1
            ev_in = []
            with torch.cuda.stream(s_in):
                if cmp_done[b_] is not None:
                    s_in.wait_event(cmp_done[b_])                  # step i-2 has finished reading this buffer set
                for n in names:
                    dev_prim[b_][n].copy_(host_prim[n], non_blocking=True)
                if cams:
                    for d_, h_ in zip(dev_cam[b_], host_cam):
                        d_.copy_(h_, non_blocking=True)
                for (a0, a1) in bounds:
                    if not cams:
                        for n in host_in:
                            dev_in[b_][n][a0:a1].copy_(host_in[n][a0:a1], non_blocking=True)
                    dev_grad[b_][a0:a1].copy_(host_grad[a0:a1], non_blocking=True)
                    e = torch.cuda.Event()
                    e.record(s_in)
                    ev_in.append(e)
            flat_ = flats[b_]
            if flat_out_done[b_] is not None:
                s_cmp.wait_event(flat_out_done[b_])                # its previous download is over
            flat_.zero_()
            di, pr = dev_in[b_], dev_prim[b_]
            for ci, (a0, a1) in enumerate(bounds):
                s_cmp.wait_event(ev_in[ci])
                nvc = a1 - a0
                lv = [expand_views(pr[n], nvc).requires_grad_(True) for n in names]     # the subject's primitives, per view
                if cams:
                    cp_, cr_, cf_, cpp_ = (t[a0:a1].contiguous() for t in dev_cam[b_])
                    o_ = mvpraymarch_camera(cp_, cr_, cf_, cpp_, (w, h), scene.VOLRADIUS, stepsize, (lv[0], lv[1], lv[2]), lv[3], None)
                else:
                    rp_, rd_, tm_ = di["raypos"][a0:a1], di["raydir"][a0:a1], di["tminmax"][a0:a1]
                    o_ = mvpraymarch(rp_, rd_, stepsize, tm_, (lv[0], lv[1], lv[2]), lv[3], None)
                o_.backward(dev_grad[b_][a0:a1])
                off = 0
                for x in (lv[3], lv[0], lv[1], lv[2]):
                    n_ = x[0].numel()
                    flat_[off:off + n_] += sum_views(x.grad).view(-1)
                    off += n_
                od = o_.detach()
                e = torch.cuda.Event()
                e.record(s_cmp)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(e)
                    host_out[a0:a1].copy_(od, non_blocking=True)
                    od.record_stream(s_out)
            if world > 1:
                dist.all_reduce(flat_)
            e = torch.cuda.Event()
            e.record(s_cmp)
            cmp_done[b_] = e
            with torch.cuda.stream(s_out):
                s_out.wait_event(e)
                host_flat.copy_(flat_, non_blocking=True)
                e2 = torch.cuda.Event()
                e2.record(s_out)
                flat_out_done[b_] = e2

        def e2e_drain():
            s_cmp.wait_stream(s_in)
            s_cmp.wait_stream(s_out)

        log("e2e buffers pinned")
        e2e_step(0)
        e2e_step(1)
        e2e_drain()
        barrier()
        log("e2e warm-up steps done")
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        nrep = max(2, args.steps)
        a.record()
        for i in range(nrep):
            e2e_step(i)
        e2e_drain()                      # every upload, kernel and download of the nrep steps is inside the timed region
        b.record()
        barrier()
        te = torch.tensor([a.elapsed_time(b) / nrep], device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        # same, with camera parameters instead of rays coming from the host (extra key, not the headline)
        e2e_step(0, True)
        e2e_step(1, True)
        e2e_drain()
        barrier()
        a2, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a2.record()
        for i in range(nrep):
            e2e_step(i, True)
        e2e_drain()
        b2.record()
        barrier()
        tc_ = torch.tensor([a2.elapsed_time(b2) / nrep], device=dev)
        if world > 1:
            dist.all_reduce(tc_, op=dist.ReduceOp.MAX)
        h2d_cam = sum(x.numel() * 4 for x in host_cam) + sum(x.numel() * 4 for x in host_prim.values()) + host_grad.numel() * 4
        e2e_cam = {"value": views * h * w / (float(tc_.item()) * 1e-3) / 1e6, "unit": "MP/s", "ms_per_step": float(tc_.item()),
                   "h2d_bytes_per_step": int(h2d_cam * world), "d2h_bytes_per_step": int(d2h * world),
                   "what": "as e2e, but the host hands over camera parameters (viewpos, viewrot, focal, princpt) instead of rays; "
                           "the render kernels generate the rays in their prologue (op.mvpraymarch_camera: compute_raydirs of "
                           "models/autoencoder.py:240 fused into the raymarcher, no ray tensors in HBM)"}
        e2e = {"value": views * h * w / (float(te.item()) * 1e-3) / 1e6, "unit": "MP/s",
               "h2d_bytes_per_step": int(h2d * world), "d2h_bytes_per_step": int(d2h * world),
               "ms_per_step": float(te.item()), "steps": nrep,
               "what": "every step: pinned host rays + one subject's primitives + grad_out -> device, per-view expand (mvp_expand_views), op fwd+bwd, "
                       "view-sum (mvp_sum_views) (+all-reduce), rayrgba + reduced gradients -> pinned host; views streamed in chunks of %d, device "
                       "staging double-buffered so H2D of step i+1 / compute of step i / D2H of step i-1 overlap (three streams); "
                       "%d steps timed back to back, all copies inside the timed region" % (chunk, nrep)}

    log("e2e done")
    if rank != 0:
        return
    peak, peak_src = measured_peaks()
    fb, bb = algorithmic_bytes(nv, h, w, k, t)
    fwd_gbs, bwd_gbs = fb / (fwd_ms * 1e-3) / 1e9, bb / (bwd_ms * 1e-3) / 1e9
    roof_f = {"kernel": "render_forward_kernel", "bound": "hbm", "achieved": fwd_gbs, "peak": peak, "unit": "GB/s",
              "frac": fwd_gbs / peak, "traffic": None, "ms_per_launch": fwd_ms, "algorithmic_bytes_per_launch": fb,
              "peak_source": peak_src}
    roof_b = {"kernel": "render_backward_kernel", "bound": "hbm", "achieved": bwd_gbs, "peak": peak, "unit": "GB/s",
              "frac": bwd_gbs / peak, "traffic": None, "ms_per_launch": bwd_ms, "algorithmic_bytes_per_launch": bb,
              "peak_source": peak_src}
    # traffic (dram bytes per launch): NOT measured in this run (ncu cannot run inside a timed bench); it is the per-view
    # figure of the committed `ncu --set full` capture named in profiles/traffic.json, valid only for the kernel build it
    # names -- reported with its source, or null when the capture is of another build / shape.
    tr = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tr):
        with open(tr) as f:
            tj = json.load(f)
        same_build = tj.get("kernel_build") == lib.LIB.mvp_build_config().decode()
        for r_ in (roof_f, roof_b):
            per_view = tj.get(r_["kernel"], {}).get("dram_bytes_per_view")
            if per_view and (h, w, k, t) == tuple(tj.get("shape", ())) and same_build:
                r_["traffic"] = per_view * nv
                zf = tj.get(r_["kernel"], {}).get("of_which_gradient_zero_fill_per_view")
                if zf:
                    r_["traffic_note"] = ("includes %.1f MB per view of gradient-buffer zero-fill the gradient-mode forward does on the side "
                                          "(clear_grad_*; formerly a memset pass), not algorithmic bytes: %.1f MB per view without it"
                                          % (zf / 1e6, (per_view - zf) / 1e6))
                r_["traffic_source"] = "committed ncu capture %s (per view x %d views), not this run" % (tj.get("source", "profiles/traffic.json"), nv)
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        # SURVEY 8d / BASELINE.json config 1: true C1 (1 x 128x128, K=256, 8^3, ~16 steps per ray), once
        cpu_mps, cpu_sec, cpu_desc = cpu_autograd_sample(128, 128, 256, 8, steps=1, warmup=0)
        cpu = {"value": cpu_mps, "unit": "MP/s", "cores": torch.get_num_threads(), "kind": "port", "sample": "C1: " + cpu_desc + ", 1 step",
               "seconds_per_sample_step": cpu_sec}
    dominant = roof_b if bwd_ms >= fwd_ms else roof_f
    line = {
        "metric": "rendered MP/s (fwd+bwd)", "value": value, "unit": "MP/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(views, h, w, k, t),
        "parallelism": "views sharded over %d rank(s) (%d per rank), interleaved, 1 NCCL all-reduce of %.1f MB primitive grads per step, overlapped with the next step's forward" % (world, nv, flat_numel * 4 / 1e6),
        "kernel_build": lib.LIB.mvp_build_config().decode(),
        "scene": {"alpha_mu": ALPHA_MU, "alpha_sigma": ALPHA_SIGMA, "saturated_ray_frac": sat_frac, "covered_ray_frac": cover},
        "roofline": dominant, "roofline_forward": roof_f, "roofline_backward": roof_b,
        "cpu_baseline": cpu, "ref_cuda_baseline": ref_cuda, "parity_check": parity, "e2e": e2e, "clocks": clocks,
        "shared_primitives_config": shared_cfg, "camera_rays_config": camera_cfg, "e2e_camera_inputs": e2e_cam,
        # this repository's kernels per timed step: accel build + render pair (forward), render pair (backward), 4 x mvp_sum_views
        "gpu_launches": args.steps * (lib.LIB.mvp_forward_launch_count(0) + lib.LIB.mvp_backward_launch_count(lib.FLAG_ACCEL_VALID) + 4),
        "kernel_ms": {"forward_all_views_per_rank": fwd_ms, "backward_all_views_per_rank": bwd_ms,
                      "note": "the forward launch also zero-fills the backward's gradient buffers (clear_grad_*, %.1f GB per rank) "
                              "on the side; those bytes are not counted as algorithmic" % clear_gb},
        "rank_ms_per_step": rank_ms, "allreduce_ms": allreduce_ms,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--views", type=int, default=VIEWS)
    ap.add_argument("--height", type=int, default=H)
    ap.add_argument("--width", type=int, default=W)
    ap.add_argument("--prims", type=int, default=K)
    ap.add_argument("--voxels", type=int, default=T)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--contiguous-views", action="store_true", help="contiguous view blocks per rank instead of interleaved")
    ap.add_argument("--e2e-chunk", type=int, default=20, help="views per pipelined chunk in the e2e measurement")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-shared-leg", action="store_true", help="skip the shared-primitive ([1,K,...]) configuration")
    ap.add_argument("--no-check", action="store_true", help="skip the reference-CUDA legs (ref_cuda_baseline, parity_check)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the images and reduced gradients of the last timed step to "
                    "DIR/<name>.npy (float32; a fixed, seeded sample of the larger arrays, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    if world > 1:
        # keep stdout to the single JSON line: NCCL prints its version banner there at NCCL_DEBUG=VERSION and above
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION", "WARN"):
            os.environ["NCCL_DEBUG"] = "NONE"
        dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ.get("LOCAL_RANK", rank))))
    try:
        run_ours(args, rank, world)
    finally:
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
