#!/usr/bin/env python
"""Timings of the differentiable render (SmoeRenderer) on one GPU; prints one JSON line.

    python tools/bench_render.py [--workload c3] [--steps 20] [--warmup 3]

The model is the bench.py workload (same image, kernel grid and flags, built by bench.py's own helpers).  Timed,
each pass bracketed by CUDA events on the launching stream with a 256 MB L2 flush write before it (outside the events):
  forward            SmoeRenderer under torch.no_grad() on the training grid (keys, sort, pack, forward)
  forward_backward   forward with the backward state + out.backward(cot): cotangent, backward, finalize, the split of
                     the gradients into the params layout and their accumulation into .grad
  x2_*               the same on a grid with twice the samples per axis (3840x2160 for c3)
  cotangent          smoe_cotangent alone, with GB/s over its algorithmic bytes: grad_r and r read (4C + 4C), the
                     flag read (4), 1 + C plane values written (4 (1 + C)) per pixel
  training_path      the training step's forward / loss / backward launches on the same model (bench.kernel_times)
The GPU's name, power limit and SM clock limit are read in the same run; a number that was not measured is null.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info(index):
    import torch
    info = {"name": torch.cuda.get_device_name(index), "power_limit_w": None, "sm_max_mhz": None}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                            "-i", str(index)], capture_output=True, text=True, timeout=30)
        f = [x.strip() for x in q.stdout.strip().split(",")]
        info["power_limit_w"], info["sm_max_mhz"] = float(f[0]), float(f[1])
    except Exception:
        pass
    return info


def timed(fn, n, warm, flush, before=None):
    """Per-pass device time (ms) of fn(): mean, min, max over n passes."""
    import torch
    for _ in range(warm):
        if before:
            before()
        fn()
    ts = []
    for _ in range(n):
        if before:
            before()
        flush.fill_(1.0)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return {"ms": float(np.mean(ts)), "min_ms": float(np.min(ts)), "max_ms": float(np.max(ts)), "passes": n}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c3")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")

    import torch
    import bench
    import __graft_entry__ as ge
    ge.build()
    from smoe_b200 import Smoe, AdamOptimizer, SmoeRenderer
    from smoe_b200.render import PARAM_KEYS
    from smoe_b200._ffi import check, lib, ptr, stream_ptr

    torch.cuda.set_device(0)
    info = gpu_info(0)
    shape, kgrid, seed, desc = bench.WORKLOADS[args.workload]
    d, Cc = len(shape) - 1, shape[-1]
    img = bench.synth_image(shape, seed)
    m = Smoe(img, kernels_per_dim=kgrid, **bench.SMOE_KW)
    m.set_optimizer(AdamOptimizer(1e-3), AdamOptimizer(1e-5), AdamOptimizer(1.0))
    flags = {k: bench.SMOE_KW[k] for k in ("use_determinant", "train_inverse_cov")}
    p0 = m.get_params()
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")
    line = {"tool": "bench_render", "workload": desc, "kernels": int(m.start_pis), "gpu": info,
            "l2": "256 MB flush write before every timed pass (outside the events)", "timings": {}}

    def leaf(grad):
        return {k: torch.tensor(v, device="cuda", requires_grad=grad) for k, v in p0.items()}

    for tag, grid in (("", [(0, 1, n) for n in shape[:d]]), ("x2_", [(0, 1, 2 * n) for n in shape[:d]])):
        r = SmoeRenderer(grid=grid, channels=Cc, **flags)
        npix = int(np.prod(r.shape))
        p = leaf(True)
        cot = torch.randn(r.shape + (Cc,), device="cuda", generator=torch.Generator("cuda").manual_seed(1))

        def fwd():
            with torch.no_grad():
                r(p)

        def fwd_bwd():
            r(p).backward(cot)

        def clear():
            for k in PARAM_KEYS:
                p[k].grad = None

        t = line["timings"]
        t[tag + "grid"] = list(r.shape)
        t[tag + "forward"] = timed(fwd, args.steps, args.warmup, flush)
        t[tag + "forward_backward"] = timed(fwd_bwd, args.steps, args.warmup, flush, before=clear)
        if tag == "":
            # smoe_cotangent alone, on the state of one forward (re-running it rewrites the flag plane with gr; the
            # traffic is the same)
            out, state = r._forward(tuple(p[k] for k in PARAM_KEYS), keep_state=True)
            pix = state[4]
            L = lib()

            def cotangent():
                check(L.smoe_cotangent(C.byref(r._cfg), C.byref(r._batch), ptr(out), ptr(cot), ptr(pix), stream_ptr()),
                      "smoe_cotangent")

            tc = timed(cotangent, args.steps, args.warmup, flush)
            nbytes = float(npix) * (4 * Cc + 4 * Cc + 4 + 4 * (1 + Cc))
            tc["bytes"] = nbytes
            tc["GBps"] = nbytes / (tc["ms"] / 1e3) / 1e9
            t["cotangent"] = tc
            del out, state, pix
        del r, p, cot
        torch.cuda.empty_cache()
    kt = bench.kernel_times(m, args.steps, with_step=False)
    line["timings"]["training_path"] = {k: kt[k] for k in ("forward_ms", "loss_ms", "loss_GBps", "backward_ms")}
    print(json.dumps(line))


if __name__ == "__main__":
    main()
