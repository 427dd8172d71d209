#!/usr/bin/env python
"""Timings of SMoE evaluation at arbitrary points (SmoePointRenderer) on one GPU; prints one JSON line.

    python tools/bench_points.py [--steps 20] [--warmup 3]
    python tools/bench_points.py --breakdown         # per-kernel device time of the c3_shuffled forward instead

Models are bench.py workloads built by bench.py's own helpers: c3 (1920x1080 RGB, 32768 kernels) and c4s (640x360x16
RGB video, 8192 kernels).  Point sets:
  c3_raster      the 1920x1080 training-grid coordinates in raster order
  c3_shuffled    the same points in a random order (the op sorts them itself; only its speed may depend on the order)
  c3_random      1920x1080 points uniform in [0, 1]^2
  c3_random_4k   3840x2160 points uniform in [0, 1]^2
  c4s_cloud      640x360x16 points uniform in [0, 1]^3 (times between frames included)
For each: forward under no_grad (keys, sort, gather, pack, forward, scatter), forward + parameter backward, and
forward + parameter and point backward; and SmoeRenderer on the grid of the same size (forward, forward + backward),
for comparison at equal N.  Timing as tools/bench_render.py: CUDA events per pass on the launching stream, a 256 MB
L2 flush write before each pass (outside the events).  The GPU's name, power limit and SM clock limit are read in the
same run.  --breakdown runs torch.profiler (CUDA activity) over --steps no_grad forwards of c3_shuffled and of
SmoeRenderer on the c3 grid and reports each kernel's device time per pass; a run of its own, as tracing slows the host.
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
    from smoe_b200.render import PARAM_KEYS

    torch.cuda.set_device(0)
    line = {"tool": "bench_points", "gpu": gpu_info(0),
            "l2": "256 MB flush write before every timed pass (outside the events)", "models": {}, "timings": {}}
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")
    flags = {k: bench.SMOE_KW[k] for k in ("use_determinant", "train_inverse_cov")}
    gen = np.random.RandomState(7)

    def model(workload):
        shape, kgrid, seed, desc = bench.WORKLOADS[workload]
        m = Smoe(bench.synth_image(shape, seed), kernels_per_dim=kgrid, **bench.SMOE_KW)
        line["models"][workload] = {"workload": desc, "kernels": int(m.start_pis)}
        p = m.get_params()
        del m
        torch.cuda.empty_cache()
        return p, shape

    def grid_points(shape):
        axes = [np.linspace(0, 1, n).astype(np.float32) for n in shape]
        return np.stack(np.meshgrid(*axes, indexing="ij"), -1).reshape(-1, len(shape))

    def leaf(p0, grad):
        return {k: torch.tensor(v, device="cuda", requires_grad=grad) for k, v in p0.items()}

    def clear(*ts):
        def f():
            for t in ts:
                t.grad = None
        return f

    def bench_points(tag, p0, pts_np, Cc):
        d = pts_np.shape[1]
        r = SmoePointRenderer(d=d, channels=Cc, **flags)
        p = leaf(p0, True)
        x = torch.tensor(pts_np, device="cuda")
        xg = x.clone().requires_grad_(True)
        cot = torch.randn((len(pts_np), Cc), device="cuda", generator=torch.Generator("cuda").manual_seed(1))

        def fwd():
            with torch.no_grad():
                r(p, x)

        def fwd_bwd_params():
            r(p, x).backward(cot)

        def fwd_bwd_all():
            r(p, xg).backward(cot)

        pl = [p[k] for k in PARAM_KEYS]
        line["timings"][tag] = {
            "points": int(len(pts_np)),
            "forward": timed(fwd, args.steps, args.warmup, flush),
            "forward_param_backward": timed(fwd_bwd_params, args.steps, args.warmup, flush, before=clear(*pl)),
            "forward_param_point_backward": timed(fwd_bwd_all, args.steps, args.warmup, flush, before=clear(xg, *pl)),
        }
        del r, p, x, xg, cot
        torch.cuda.empty_cache()

    def bench_grid(tag, p0, shape, Cc):
        r = SmoeRenderer(grid=[(0, 1, n) for n in shape], channels=Cc, **flags)
        p = leaf(p0, True)
        cot = torch.randn(r.shape + (Cc,), device="cuda", generator=torch.Generator("cuda").manual_seed(1))

        def fwd():
            with torch.no_grad():
                r(p)

        def fwd_bwd():
            r(p).backward(cot)

        line["timings"][tag] = {"grid": list(r.shape), "forward": timed(fwd, args.steps, args.warmup, flush),
                                "forward_backward": timed(fwd_bwd, args.steps, args.warmup, flush,
                                                          before=clear(*[p[k] for k in PARAM_KEYS]))}
        del r, p, cot
        torch.cuda.empty_cache()

    p3, s3 = model("c3")
    raster = grid_points(s3[:2])
    if args.breakdown:
        from torch.profiler import ProfilerActivity, profile
        p = leaf(p3, False)
        x = torch.tensor(raster[gen.permutation(len(raster))], device="cuda")
        rp = SmoePointRenderer(d=2, channels=3, **flags)
        rg = SmoeRenderer(grid=[(0, 1, n) for n in s3[:2]], channels=3, **flags)
        for tag, fn in (("c3_shuffled_forward", lambda: rp(p, x)), ("c3_grid_renderer_forward", lambda: rg(p))):
            with torch.no_grad():
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
    bench_points("c3_raster", p3, raster, 3)
    bench_points("c3_shuffled", p3, raster[gen.permutation(len(raster))], 3)
    bench_points("c3_random", p3, gen.uniform(0, 1, raster.shape).astype(np.float32), 3)
    bench_grid("c3_grid_renderer", p3, s3[:2], 3)
    n4k = 3840 * 2160
    bench_points("c3_random_4k", p3, gen.uniform(0, 1, (n4k, 2)).astype(np.float32), 3)
    bench_grid("c3_grid_renderer_4k", p3, (2160, 3840), 3)
    p4, s4 = model("c4s")
    n4 = int(np.prod(s4[:3]))
    bench_points("c4s_cloud", p4, gen.uniform(0, 1, (n4, 3)).astype(np.float32), 3)
    bench_grid("c4s_grid_renderer", p4, s4[:3], 3)
    t = line["timings"]
    line["shuffled_forward_over_grid_forward"] = t["c3_shuffled"]["forward"]["ms"] / t["c3_grid_renderer"]["forward"]["ms"]
    print(json.dumps(line))


if __name__ == "__main__":
    main()
