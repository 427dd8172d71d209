#!/usr/bin/env python
"""Timings of the Gauss-Newton diagonal (SmoeRenderer / SmoePointRenderer.gauss_newton_diagonal) on one GPU; prints one
JSON line.

    python tools/bench_gn_diag.py [--steps 20] [--warmup 3]
    python tools/bench_gn_diag.py --breakdown       # per-kernel device time (torch.profiler) on the c3 grid instead

Models are bench.py workloads built by bench.py's own helpers: c3 (1920x1080 RGB, 32768 kernels) and c4s (640x360x16
RGB video, 8192 kernels).  Rows:
  c3_grid         SmoeRenderer on the 1920x1080 training grid
  c3_grid_4k      SmoeRenderer on a 3840x2160 grid of the same model
  c3_shuffled     SmoePointRenderer on the 1920x1080 grid coordinates in a random order
  c4s_grid        SmoeRenderer on the 640x360x16 video grid
Each row times: the forward under no_grad; forward + diagonal (h = 1); forward + backward of a random dL/dr (the
reference cost: the renderer's training-path pair); one Hutchinson sample v * J^T (J v) with a Rademacher v (one
Gauss-Newton product: forward_ad dual inputs that require grad, then the backward of dr).  Then the Hutchinson estimate
given the device time of the exact call (S = max(1, round(t_diagonal / t_sample)) samples) against the exact D: the
median and 90th percentile of |est - D| / D over the entries with D >= 1e-3 max of their tensor.
Timing as tools/bench_render.py: CUDA events per pass on the launching stream, a 256 MB L2 flush write before each pass
(outside the events).  The GPU's name, power limit and SM clock limit are read in the same run.
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

PARAM_KEYS = ("pis", "musX", "A_diagonal", "A_corr", "gamma_e", "nu_e")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--breakdown", action="store_true")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")

    import torch
    import torch.autograd.forward_ad as fwAD
    import bench
    import __graft_entry__ as ge
    from bench_render import gpu_info, timed
    ge.build()
    from smoe_b200 import Smoe, SmoePointRenderer, SmoeRenderer

    torch.cuda.set_device(0)
    line = {"tool": "bench_gn_diag", "gpu": gpu_info(0),
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

    if args.breakdown:
        from torch.profiler import ProfilerActivity, profile
        p3, s3 = model("c3")
        ren = SmoeRenderer(grid=[(0, 1, n) for n in s3[:2]], channels=3, **flags)
        g = torch.randn(tuple(s3[:2]) + (3,), device="cuda")

        def fwd_bwd():
            q = {k: t.detach().requires_grad_(True) for k, t in p3.items()}
            ren(q).backward(g)

        for tag, fn in (("c3_grid_gauss_newton_diagonal", lambda: ren.gauss_newton_diagonal(p3)),
                        ("c3_grid_forward_backward", fwd_bwd)):
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

    def row_for(tag, ren, p, x=None):
        extra = () if x is None else (x,)
        keys = PARAM_KEYS
        rs = np.random.RandomState(5)
        call = ren
        with torch.no_grad():
            r0 = call(p, *extra)
        g = torch.tensor(rs.standard_normal(tuple(r0.shape)).astype(np.float32), device="cuda")
        v = {k: torch.tensor(rs.choice([-1.0, 1.0], t.shape).astype(np.float32), device="cuda") for k, t in p.items()}

        def fwd():
            with torch.no_grad():
                return call(p, *extra)

        def diag():
            return ren.gauss_newton_diagonal(p, *extra)

        def fwd_bwd():
            q = {k: t.detach().requires_grad_(True) for k, t in p.items()}
            call(q, *extra).backward(g)

        def sample(vv):
            q = {k: t.detach().requires_grad_(True) for k, t in p.items()}
            with fwAD.dual_level():
                out = call({k: fwAD.make_dual(q[k], vv[k]) for k in keys}, *extra)
                r, jv = fwAD.unpack_dual(out)
            r.backward(jv)
            return {k: vv[k] * q[k].grad for k in keys}

        row = {"forward": timed(fwd, args.steps, args.warmup, flush),
               "forward_diagonal": timed(diag, args.steps, args.warmup, flush),
               "forward_backward": timed(fwd_bwd, args.steps, args.warmup, flush),
               "hutchinson_sample": timed(lambda: sample(v), args.steps, args.warmup, flush)}
        D = diag()[1]
        S = max(1, int(round(row["forward_diagonal"]["ms"] / row["hutchinson_sample"]["ms"])))
        est = {k: torch.zeros_like(D[k]) for k in keys}
        for s in range(S):
            vs = {k: torch.tensor(rs.choice([-1.0, 1.0], t.shape).astype(np.float32), device="cuda")
                  for k, t in p.items()}
            for k, t in sample(vs).items():
                est[k] += t / S
        errs = []
        for k in keys:
            big = D[k] >= 1e-3 * D[k].max()
            errs.append(((est[k][big] - D[k][big]).abs() / D[k][big]).double().cpu().numpy())
        errs = np.concatenate(errs)
        row["hutchinson_same_time"] = {"samples": S, "median_rel_error": float(np.median(errs)),
                                       "p90_rel_error": float(np.percentile(errs, 90)), "entries": int(errs.size)}
        row["diagonal_over_forward_backward"] = row["forward_diagonal"]["ms"] / row["forward_backward"]["ms"]
        line["timings"][tag] = row
        torch.cuda.empty_cache()

    p3, s3 = model("c3")
    row_for("c3_grid", SmoeRenderer(grid=[(0, 1, n) for n in s3[:2]], channels=3, **flags), p3)
    row_for("c3_grid_4k", SmoeRenderer(grid=[(0, 1, 2160), (0, 1, 3840)], channels=3, **flags), p3)
    axes = [np.linspace(0, 1, n).astype(np.float32) for n in s3[:2]]
    raster = np.stack(np.meshgrid(*axes, indexing="ij"), -1).reshape(-1, 2)
    x = torch.tensor(raster[gen.permutation(len(raster))], device="cuda")
    row_for("c3_shuffled", SmoePointRenderer(d=2, channels=3, **flags), p3, x)
    line["timings"]["c3_shuffled"]["points"] = int(len(raster))
    del p3, x
    p4, s4 = model("c4s")
    row_for("c4s_grid", SmoeRenderer(grid=[(0, 1, n) for n in s4[:3]], channels=3, **flags), p4)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
