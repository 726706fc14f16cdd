"""Times bf16 payloads (C-ABI MVP_FLAG_TPLATE_BF16) on the bench.py scene (C3: 1024x667, K=16384, 8^3, alpha 17/6) at 8 and
80 views, the arms alternated in one process:

  * kernels: mvp_raymarch_forward (gradient mode, accel prebuilt, clearing the gradient buffers like the op does) and
    mvp_raymarch_backward, CUDA events around each launch as in bench.py, for an fp32 template and for its bf16 rounding
    (the same values, so the same samples and the same work);
  * op step (forward + backward through `mvpraymarch`): the bf16 template passed as it is, against the workaround it replaces
    (`template_bf16.float()`, the fp32 op, the gradient cast back to bf16 by autograd);
  * peak memory of one op step of each arm (torch.cuda.max_memory_allocated, and its rise over what was allocated before).

  python scripts/time_bf16_payload.py [--views 8,80] [--steps 5] [--rounds 3] [--out profiles/bf16_payload.json]
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ava256_b200 import lib, scene  # noqa: E402
from ava256_b200.op import mvpraymarch  # noqa: E402

H, W, K, T, ALPHA_MU, ALPHA_SIGMA = 1024, 667, 16384, 8, 17.0, 6.0      # bench.py's scene
P = lambda x: ctypes.c_void_p(x.data_ptr())  # noqa: E731


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    name, power, clk = (x.strip() for x in q.stdout.strip().split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clk, "torch_name": torch.cuda.get_device_name()}


def time_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def kernel_arm(s, tplate, grad_out, bf16):
    """(forward launch, backward launch) through the C-ABI on `tplate`; the accel structure is built once here."""
    N = s["raypos"].shape[0]
    dev = tplate.device
    wsb = lib.workspace_bytes(N, H, W, K, T, T, T)
    st = {"ws": torch.empty(wsb, dtype=torch.uint8, device=dev), "rgba": torch.empty(N, H, W, 4, device=dev),
          "rsat": torch.empty(N, H, W, 3, device=dev), "raux": torch.empty(N, H, W, 4, dtype=torch.int32, device=dev),
          "g": [torch.empty_like(s[k]) for k in ("primpos", "primrot", "primscale")] +
               [torch.empty(tplate.shape, dtype=torch.float32, device=dev)], "tplate": tplate}
    flag = lib.FLAG_TPLATE_BF16 if bf16 else 0
    fa = lib.ForwardArgs()
    fa.shape = lib.Shape(N, H, W, K, T, T, T)
    fa.stepsize, fa.fadescale, fa.fadeexp, fa.flags = s["stepsize"], 8.0, 8.0, flag
    fa.raypos, fa.raydir, fa.tminmax = P(s["raypos"]), P(s["raydir"]), P(s["tminmax"])
    fa.primpos, fa.primrot, fa.primscale, fa.tplate = P(s["primpos"]), P(s["primrot"]), P(s["primscale"]), P(tplate)
    fa.rayrgba, fa.raysat, fa.rayaux, fa.workspace, fa.workspace_bytes = P(st["rgba"]), P(st["rsat"]), P(st["raux"]), P(st["ws"]), wsb
    g = st["g"]
    fa.clear_grad_primpos, fa.clear_grad_primrot, fa.clear_grad_primscale, fa.clear_grad_tplate = P(g[0]), P(g[1]), P(g[2]), P(g[3])
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    lib.check(lib.LIB.mvp_raymarch_forward(ctypes.byref(fa), stream))          # builds the accel structure
    fa.flags = lib.FLAG_ACCEL_VALID | flag
    ba = lib.BackwardArgs()
    ba.shape, ba.stepsize, ba.fadescale, ba.fadeexp, ba.flags = fa.shape, fa.stepsize, 8.0, 8.0, lib.FLAG_ACCEL_VALID | flag
    ba.raypos, ba.raydir, ba.tminmax = fa.raypos, fa.raydir, fa.tminmax
    ba.primpos, ba.primrot, ba.primscale, ba.tplate = fa.primpos, fa.primrot, fa.primscale, fa.tplate
    ba.grad_rayrgba, ba.raysat, ba.rayaux = P(grad_out), P(st["rsat"]), P(st["raux"])
    ba.grad_primpos, ba.grad_primrot, ba.grad_primscale, ba.grad_tplate = P(g[0]), P(g[1]), P(g[2]), P(g[3])
    ba.workspace, ba.workspace_bytes = P(st["ws"]), wsb
    fwd = lambda: lib.check(lib.LIB.mvp_raymarch_forward(ctypes.byref(fa), stream))  # noqa: E731
    bwd = lambda: lib.check(lib.LIB.mvp_raymarch_backward(ctypes.byref(ba), stream))  # noqa: E731
    return fwd, bwd, st


def op_step(s, prims, tleaf, grad_out, workaround):
    for x in prims + [tleaf]:
        x.grad = None
    t = tleaf.float() if workaround else tleaf
    out = mvpraymarch(s["raypos"], s["raydir"], s["stepsize"], s["tminmax"], tuple(prims), t, None)
    out.backward(grad_out)
    return out


def run(n_views, steps, rounds):
    dev = torch.device("cuda")
    s = scene.make_scene(n_views, H, W, K, T, seed=1112, device=dev, alpha_mu=ALPHA_MU, alpha_sigma=ALPHA_SIGMA)
    t16 = s.pop("template").to(torch.bfloat16)
    torch.cuda.empty_cache()
    grad_out = torch.randn(n_views, H, W, 4, device=dev, generator=torch.Generator(device=dev).manual_seed(1112))
    res = {"views": n_views, "H": H, "W": W, "K": K, "T": T, "steps_per_sample": steps, "rounds": rounds}

    # ---- kernels: fp32 template (the bf16 values upcast) vs the bf16 template ----
    t32 = t16.float()
    arms = {"fp32": kernel_arm(s, t32, grad_out, False), "bf16": kernel_arm(s, t16, grad_out, True)}
    kt = {a: {"fwd": [], "bwd": []} for a in arms}
    for _ in range(rounds):
        for a, (fwd, bwd, _) in arms.items():
            kt[a]["fwd"].append(time_ms(fwd, steps))
            kt[a]["bwd"].append(time_ms(bwd, steps))
    fwd, bwd, st32 = arms["fp32"]
    fwd(); bwd()
    _, _, st16 = arms["bf16"]
    fwd16, bwd16, _ = arms["bf16"]
    fwd16(); bwd16()
    torch.cuda.synchronize()
    res["kernel_outputs_identical"] = bool(torch.equal(st32["rgba"], st16["rgba"]))
    res["kernel_grad_template_relerr"] = float((st32["g"][3] - st16["g"][3]).abs().max() / st32["g"][3].abs().max())
    res["kernel_ms"] = {a: {k: {"median": statistics.median(v), "min": min(v), "samples": v} for k, v in d.items()} for a, d in kt.items()}
    del arms, st32, st16, fwd, bwd, fwd16, bwd16, t32
    torch.cuda.empty_cache()

    # ---- op step: bf16 template vs template.float() + fp32 op + gradient cast back ----
    prims = [s[k].requires_grad_(True) for k in ("primpos", "primrot", "primscale")]
    tleaf = t16.requires_grad_(True)
    outs = {}
    for wa in (False, True):                   # warm-up; also the outputs the two arms hand back
        outs[wa] = (op_step(s, prims, tleaf, grad_out, wa).detach(), tleaf.grad.clone())
    torch.cuda.synchronize()
    res["op_outputs_identical"] = bool(torch.equal(outs[False][0], outs[True][0]))
    g0, g1 = outs[False][1].float(), outs[True][1].float()
    res["op_grad_template_dtype"] = str(outs[False][1].dtype)
    res["op_grad_template_max_abs_diff_over_max"] = float((g0 - g1).abs().max() / g1.abs().max())
    del outs, g0, g1
    ot = {"bf16": [], "workaround": []}
    for _ in range(rounds):
        for name, wa in (("bf16", False), ("workaround", True)):
            ot[name].append(time_ms(lambda: op_step(s, prims, tleaf, grad_out, wa), steps))
    res["op_step_ms"] = {k: {"median": statistics.median(v), "min": min(v), "samples": v} for k, v in ot.items()}
    mem = {}
    for name, wa in (("bf16", False), ("workaround", True)):
        for x in prims + [tleaf]:
            x.grad = None
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        op_step(s, prims, tleaf, grad_out, wa)
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated()
        mem[name] = {"max_memory_allocated": peak, "rise_over_inputs": peak - base}
    res["op_step_peak_bytes"] = mem
    res["op_step_peak_saving_bytes"] = mem["workaround"]["max_memory_allocated"] - mem["bf16"]["max_memory_allocated"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--views", default="8,80")
    ap.add_argument("--steps", type=int, default=5, help="launches / op steps per timed sample")
    ap.add_argument("--rounds", type=int, default=3, help="samples per arm, the arms alternated")
    ap.add_argument("--out", default=None, help="JSON file (default: print only)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_bf16_payload.py needs a CUDA device")
    out = {"card": card(), "build_config": lib.LIB.mvp_build_config().decode(), "torch": torch.__version__, "results": []}
    for n in (int(v) for v in args.views.split(",")):
        r = run(n, args.steps, args.rounds)
        out["results"].append(r)
        print(json.dumps({k: r[k] for k in ("views", "kernel_outputs_identical", "op_outputs_identical")}), flush=True)
        for a in ("fp32", "bf16"):
            print("  kernel %-4s fwd %.2f ms  bwd %.2f ms" % (a, r["kernel_ms"][a]["fwd"]["median"], r["kernel_ms"][a]["bwd"]["median"]))
        for a in ("bf16", "workaround"):
            print("  op step %-10s %.2f ms  peak %.2f GB" % (a, r["op_step_ms"][a]["median"], r["op_step_peak_bytes"][a]["max_memory_allocated"] / 1e9))
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(out["card"]))


if __name__ == "__main__":
    main()
