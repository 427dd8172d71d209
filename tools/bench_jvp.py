#!/usr/bin/env python
"""Timings of forward mode (Jacobian-vector products of SmoeRenderer and SmoePointRenderer) on one GPU; prints one JSON
line.

    python tools/bench_jvp.py [--steps 20] [--warmup 3]

Models are bench.py workloads built by bench.py's own helpers: c3 (1920x1080 RGB, 32768 kernels) and c4s (640x360x16
RGB video, 8192 kernels).  Rows:
  c3_grid         SmoeRenderer on the 1920x1080 training grid
  c3_grid_4k      SmoeRenderer on a 3840x2160 grid of the same model
  c3_shuffled     SmoePointRenderer on the 1920x1080 grid coordinates in a random order
  c4s_grid        SmoeRenderer on the 640x360x16 video grid
Each row times: the forward under no_grad; forward + JVP with a random tangent on all six parameter tensors (each
entry 0.1 N(0, 1) times the parameter; torch.func.jvp); for points also forward + JVP with a tangent on the points alone; the central-difference route
(two no_grad forwards at p +- h v, h = 1e-3) with its error against the JVP (max |cd - jvp| / max |jvp|); and one
Gauss-Newton product J^T (J v) (forward_ad dual inputs that require grad, then the backward of dr).
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
    line = {"tool": "bench_jvp", "gpu": gpu_info(0),
            "l2": "256 MB flush write before every timed pass (outside the events)", "models": {}, "timings": {}}
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")
    flags = {k: bench.SMOE_KW[k] for k in ("use_determinant", "train_inverse_cov")}
    gen = np.random.RandomState(7)
    H = 1e-3

    def model(workload):
        shape, kgrid, seed, desc = bench.WORKLOADS[workload]
        m = Smoe(bench.synth_image(shape, seed), kernels_per_dim=kgrid, **bench.SMOE_KW)
        line["models"][workload] = {"workload": desc, "kernels": int(m.start_pis)}
        p = {k: torch.tensor(v, device="cuda") for k, v in m.get_params().items()}
        del m
        torch.cuda.empty_cache()
        rs = np.random.RandomState(3)
        # relative tangents, so that p +- h v keeps every pi > 0 (a kernel with pi <= 0 leaves the model)
        v = {k: (t * torch.tensor((0.1 * rs.standard_normal(t.shape)).astype(np.float32), device="cuda"))
             for k, t in p.items()}
        return p, v, shape

    def row_for(tag, call, p, v, x=None, dx=None):
        """call(params[, points]): one renderer call; v: parameter tangents; dx: point tangents (points only)."""
        extra = () if x is None else (x,)
        keys = PARAM_KEYS
        prim = tuple(p[k] for k in keys)
        tan = tuple(v[k] for k in keys)

        def fwd():
            with torch.no_grad():
                return call(p, *extra)

        def jvp():
            return torch.func.jvp(lambda *t: call(dict(zip(keys, t)), *extra), prim, tan)

        def cd():
            with torch.no_grad():
                hi = call({k: p[k] + H * v[k] for k in keys}, *extra)
                lo = call({k: p[k] - H * v[k] for k in keys}, *extra)
            return (hi - lo) / (2 * H)

        def gn():
            q = {k: t.detach().requires_grad_(True) for k, t in p.items()}
            with fwAD.dual_level():
                out = call({k: fwAD.make_dual(q[k], v[k]) for k in keys}, *extra)
                r, jv = fwAD.unpack_dual(out)
            r.backward(jv)
            return [q[k].grad for k in keys]

        row = {"forward": timed(fwd, args.steps, args.warmup, flush), "jvp_params": timed(jvp, args.steps, args.warmup,
                                                                                         flush)}
        if dx is not None:
            row["jvp_points"] = timed(lambda: torch.func.jvp(lambda xx: call(p, xx), (x,), (dx,)), args.steps,
                                      args.warmup, flush)
        row["central_difference"] = timed(cd, args.steps, args.warmup, flush)
        row["gauss_newton_product"] = timed(gn, args.steps, args.warmup, flush)
        jv = jvp()[1].double()
        row["central_difference_error"] = float((cd().double() - jv).abs().max() / jv.abs().max())
        row["jvp_params_minus_forward_ms"] = row["jvp_params"]["ms"] - row["forward"]["ms"]
        line["timings"][tag] = row
        torch.cuda.empty_cache()

    p3, v3, s3 = model("c3")
    r = SmoeRenderer(grid=[(0, 1, n) for n in s3[:2]], channels=3, **flags)
    row_for("c3_grid", r, p3, v3)
    r = SmoeRenderer(grid=[(0, 1, 2160), (0, 1, 3840)], channels=3, **flags)
    row_for("c3_grid_4k", r, p3, v3)
    del r
    axes = [np.linspace(0, 1, n).astype(np.float32) for n in s3[:2]]
    raster = np.stack(np.meshgrid(*axes, indexing="ij"), -1).reshape(-1, 2)
    x = torch.tensor(raster[gen.permutation(len(raster))], device="cuda")
    dx = torch.tensor(gen.standard_normal(tuple(x.shape)).astype(np.float32) * 1e-3, device="cuda")
    row_for("c3_shuffled", SmoePointRenderer(d=2, channels=3, **flags), p3, v3, x, dx)
    line["timings"]["c3_shuffled"]["points"] = int(len(raster))
    del p3, v3, x, dx
    p4, v4, s4 = model("c4s")
    row_for("c4s_grid", SmoeRenderer(grid=[(0, 1, n) for n in s4[:3]], channels=3, **flags), p4, v4)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
