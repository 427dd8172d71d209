#!/usr/bin/env python
"""Timings of the spatial Jacobian (SmoePointRenderer.jacobian, SmoeRenderer.jacobian) on one GPU; prints one JSON line.

    python tools/bench_jacobian.py [--steps 20] [--warmup 3]
    python tools/bench_jacobian.py --breakdown       # per-kernel device time of the c3 jacobian() calls instead

Models are bench.py workloads built by bench.py's own helpers: c3 (1920x1080 RGB, 32768 kernels) and c4s (640x360x16
RGB video, 8192 kernels).  Rows:
  c3_shuffled    the 1920x1080 training-grid coordinates in a random order: forward under no_grad, jacobian(), and the
                 route without it -- C evaluations, each a forward, a one-hot cotangent and the coordinate sweep
                 (smoe_point_xgrad), since a call's backward state is consumed once
  c3_grid        the same coordinates in raster order (a uniform grid given as points): forward, jacobian(); and
                 SmoeRenderer on that grid: forward, jacobian() (the grid sweep, smoe_jacobian)
  c3_grid_4k     the same at 3840x2160
  c4s_cloud      640x360x16 points uniform in [0, 1]^3: forward, jacobian()
  c4s_grid       the 640x360x16 grid, as points and through SmoeRenderer
Timing as tools/bench_render.py: CUDA events per pass on the launching stream, a 256 MB L2 flush write before each pass
(outside the events).  The GPU's name, power limit and SM clock limit are read in the same run.  --breakdown runs
torch.profiler (CUDA activity) over --steps jacobian() calls of c3_shuffled and of SmoeRenderer on the c3 grid; a run
of its own, as tracing slows the host.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--breakdown", action="store_true")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")

    import torch
    import bench
    import __graft_entry__ as ge
    from bench_render import gpu_info, timed
    ge.build()
    from smoe_b200 import Smoe, SmoePointRenderer, SmoeRenderer

    torch.cuda.set_device(0)
    line = {"tool": "bench_jacobian", "gpu": gpu_info(0),
            "l2": "256 MB flush write before every timed pass (outside the events)", "models": {}, "timings": {}}
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")
    flags = {k: bench.SMOE_KW[k] for k in ("use_determinant", "train_inverse_cov")}
    gen = np.random.RandomState(7)

    def model(workload):
        shape, kgrid, seed, desc = bench.WORKLOADS[workload]
        m = Smoe(bench.synth_image(shape, seed), kernels_per_dim=kgrid, **bench.SMOE_KW)
        line["models"][workload] = {"workload": desc, "kernels": int(m.start_pis)}
        p = {k: torch.tensor(v, device="cuda") for k, v in m.get_params().items()}
        del m
        torch.cuda.empty_cache()
        return p, shape

    def grid_points(shape):
        axes = [np.linspace(0, 1, n).astype(np.float32) for n in shape]
        return np.stack(np.meshgrid(*axes, indexing="ij"), -1).reshape(-1, len(shape))

    def bench_grid(tag, p, shape, Cc):
        """SmoeRenderer.jacobian on the (0, 1, n) grid of `shape` into the row of the same coordinates as points."""
        r = SmoeRenderer(grid=[(0, 1, n) for n in shape], channels=Cc, **flags)

        def fwd():
            with torch.no_grad():
                r(p)

        row = line["timings"][tag]
        row["grid_forward"] = timed(fwd, args.steps, args.warmup, flush)
        row["grid_jacobian"] = timed(lambda: r.jacobian(p), args.steps, args.warmup, flush)
        row["point_jacobian_over_grid_jacobian"] = row["jacobian"]["ms"] / row["grid_jacobian"]["ms"]
        del r
        torch.cuda.empty_cache()

    def bench_points(tag, p, pts_np, Cc, c_pass=False):
        d = pts_np.shape[1]
        r = SmoePointRenderer(d=d, channels=Cc, **flags)
        x = torch.tensor(pts_np, device="cuda")

        def fwd():
            with torch.no_grad():
                r(p, x)

        row = {"points": int(len(pts_np)), "forward": timed(fwd, args.steps, args.warmup, flush),
               "jacobian": timed(lambda: r.jacobian(p, x), args.steps, args.warmup, flush)}
        if c_pass:
            xg = x.clone().requires_grad_(True)
            onehot = [torch.zeros((len(pts_np), Cc), device="cuda").index_fill_(1, torch.tensor([c], device="cuda"), 1.0)
                      for c in range(Cc)]

            def route():
                for c in range(Cc):
                    xg.grad = None
                    r(p, xg).backward(onehot[c])

            row["c_pass_route"] = timed(route, args.steps, args.warmup, flush)
            row["c_pass_route_over_jacobian"] = row["c_pass_route"]["ms"] / row["jacobian"]["ms"]
        row["jacobian_minus_forward_ms"] = row["jacobian"]["ms"] - row["forward"]["ms"]
        line["timings"][tag] = row
        del r, x
        torch.cuda.empty_cache()

    p3, s3 = model("c3")
    raster = grid_points(s3[:2])
    shuffled = raster[gen.permutation(len(raster))]
    if args.breakdown:
        from torch.profiler import ProfilerActivity, profile
        rp = SmoePointRenderer(d=2, channels=3, **flags)
        rg = SmoeRenderer(grid=[(0, 1, n) for n in s3[:2]], channels=3, **flags)
        x = torch.tensor(shuffled, device="cuda")
        for tag, fn in (("c3_shuffled_jacobian", lambda: rp.jacobian(p3, x)),
                        ("c3_grid_jacobian", lambda: rg.jacobian(p3))):
            for _ in range(args.warmup):
                fn()
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(args.steps):
                    fn()
                torch.cuda.synchronize()
            rows = {e.key[:90]: e.device_time_total / args.steps for e in prof.key_averages() if e.device_time_total > 0}
            line["timings"][tag + "_kernels_us"] = dict(sorted(rows.items(), key=lambda kv: -kv[1]))
            line["timings"][tag + "_kernels_total_us"] = sum(rows.values())
        print(json.dumps(line))
        return
    bench_points("c3_shuffled", p3, shuffled, 3, c_pass=True)
    bench_points("c3_grid", p3, raster, 3)
    bench_grid("c3_grid", p3, s3[:2], 3)
    bench_points("c3_grid_4k", p3, grid_points((2160, 3840)), 3)
    bench_grid("c3_grid_4k", p3, (2160, 3840), 3)
    del p3
    p4, s4 = model("c4s")
    n4 = int(np.prod(s4[:3]))
    bench_points("c4s_cloud", p4, gen.uniform(0, 1, (n4, 3)).astype(np.float32), 3)
    bench_points("c4s_grid", p4, grid_points(s4[:3]), 3)
    bench_grid("c4s_grid", p4, s4[:3], 3)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
