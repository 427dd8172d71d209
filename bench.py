#!/usr/bin/env python
"""bench.py -- SMoE hot-path benchmark (DESIGN.md section "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c1|c2|c3|c4s|c4]
                    [--dump-outputs DIR]

One "step" = one full training iteration of the hot path on the workload: pi-mask compaction,
fused forward (both sweeps), fused backward, statistics -> gradients, Adam, kernel-list upkeep.
Workload (default): BASELINE config 3 -- 1920x1080 RGB, 128x256 kernel grid (32,768 kernels), the
configuration the north-star target is quoted on; it fits one GPU and is the one that shards over
ranks (rows), so every N runs the same total work ("strong" scaling).
metric = pixel.kernel evaluations/s through forward+backward = N_pixels * K_active * steps / time.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (shape, kernels_per_dim, seed, description)
    "c1": ((128, 128, 1), [16, 16], 1001, "128x128x1, 16x16 kernels (config 1)"),
    "c2": ((512, 512, 1), [64, 64], 1002, "512x512x1, 64x64 kernels (config 2)"),
    "c3": ((1080, 1920, 3), [128, 256], 1003, "1920x1080 RGB, 128x256=32768 kernels (config 3)"),
    "c4s": ((360, 640, 16, 3), [16, 32, 16], 1004, "640x360x16 RGB video, 16x32x16=8192 kernels, 3x3 A (config 4 at 1/8 scale)"),
    "c4": ((720, 1280, 32, 3), [32, 64, 32], 1004, "1280x720x32 RGB video, 32x64x32=65536 kernels, 3x3 A (config 4; meant for 2/4/8 GPUs)"),
}
SMOE_KW = dict(use_determinant=True, train_inverse_cov=False, use_yuv=False, normalize_pis=True)


def synth_image(shape, seed):
    """SURVEY.md 8d synthetic pattern, uint8-quantised then /255 (utils.py:126-128)."""
    rs = np.random.RandomState(seed)
    H, W, C = shape[0], shape[1], shape[-1]
    v, u = np.meshgrid(np.linspace(0, 1, H, dtype=np.float32), np.linspace(0, 1, W, dtype=np.float32), indexing="ij")

    def base(uu, vv):
        return (0.5 + 0.25 * np.sin(2 * np.pi * (3 * uu + 2 * vv)) + 0.2 * (uu > vv)
                + 0.15 * np.exp(-((uu - .3) ** 2 + (vv - .6) ** 2) / 0.02)).astype(np.float32)
    shifts = [0.0, 0.11, 0.23]
    if len(shape) == 3:
        img = np.stack([base(u + shifts[c], v) for c in range(C)], axis=-1)
    else:
        ts = np.linspace(0, 1, shape[2])
        img = np.stack([np.stack([base(u + shifts[c] + 0.1 * t, v) for c in range(C)], axis=-1) for t in ts], axis=2)
    img = np.clip(img + 0.03 * rs.standard_normal(img.shape).astype(np.float32), 0, 1)
    return (np.round(img * 255).astype(np.uint8).astype(np.float32) / 255.).astype(np.float32)


def algorithmic_lane_instr(d, C):
    """SURVEY.md 8d: FP32 lane-instructions per evaluation (FMA counted once)."""
    T = d * (d + 1) // 2
    f_fwd = 2 * d + T + 2 + C * (d + 1)
    f_bwd = 4 * d + 2 * T + 6 + 2 * d * C + 3 * C
    return f_fwd, f_bwd


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fd:
            j = json.load(fd)
        return j, "measured"
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------------
# CPU arm: the oracle's restatement of the reference graph on the host cores (TensorFlow is not
# installable offline; see DESIGN.md).  Same materialisation strategy as the reference: broadcast
# (K,N,d,d,d) einsum product, explicit K x N gate matrix, autograd backward, TF-style Adam.
# ----------------------------------------------------------------------------------------------
def cpu_reference_evals_per_s(workload, steps, warmup, budget_s=25.0):
    import torch
    from oracle.model import OracleAdam, OracleSmoe
    shape, kgrid, seed, _ = WORKLOADS[workload]
    d = len(shape) - 1
    # bounded sample of the same workload: a crop of the image with the kernels of the matching
    # crop of the grid (same pixels-per-kernel density), sized for ~1-2 s per step on 8 cores
    frac = {"c1": 1, "c2": 4, "c3": 8, "c4s": 8, "c4": 16}[workload]
    crop = tuple(max(s // frac, 8) for s in shape[:d]) + (shape[-1],)
    kcrop = [max(k // frac, 2) for k in kgrid]
    img = synth_image(shape, seed)[tuple(slice(0, c) for c in crop[:d])]
    torch.set_num_threads(os.cpu_count() or 1)
    m = OracleSmoe(img, kernels_per_dim=kcrop, dtype=torch.float32, einsum_mode="broadcast", **SMOE_KW)
    m.set_optimizer(OracleAdam(1e-3), OracleAdam(1e-5), OracleAdam(1.0))
    evals = int(np.prod(crop[:d])) * int(np.prod(kcrop))
    for _ in range(warmup):
        m.run_batched(train=True)
    times = []
    t_start = time.perf_counter()
    for _ in range(steps):
        t0 = time.perf_counter()
        m.run_batched(train=True)
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_start > budget_s:
            break
    t = float(np.median(times))
    return {"value": evals / t, "unit": "evals/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"crop {crop[:d]} px x {int(np.prod(kcrop))} kernels of {workload} ({evals:.3g} evals/step), "
                      f"median of {len(times)} steps, PyTorch-CPU float32, reference graph restated "
                      f"(TensorFlow unavailable)", "ms_per_step": t * 1e3, "steps": len(times)}, evals


def common_config(workload, world):
    """The workload description both arms print (identical dicts, so the two lines can be paired)."""
    shape, kgrid, _, desc = WORKLOADS[workload]
    d = len(shape) - 1
    return {"workload": desc, "pixels": int(np.prod(shape[:d])), "kernels": int(np.prod(kgrid)), "d": d, "C": shape[-1],
            "batches": 1, "init": "regular grid, pi=1/K, use_determinant", "ranks": world,
            "l2": "GPU arm: 256 MB flush write between timed steps (outside the events); CPU arm: not applicable"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    base, evals = cpu_reference_evals_per_s(args.workload, max(args.steps, 3), max(args.warmup, 1), budget_s=120.0)
    line = {"impl": "reference", "metric": "pixel_kernel_evals_per_s_fwd_bwd", "value": base["value"], "unit": "evals/s",
            "n_gpus": args.gpus, "steps": base["steps"], "warmup": max(args.warmup, 1), "ms_per_step": base["ms_per_step"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": common_config(args.workload, args.gpus),
            "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": base["value"], "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def event_time(fn, n, warm=1):
    """Average device time of fn() over n calls, CUDA events on the launching (current) stream."""
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.mean(ts))


def kernel_times(m, steps, with_step=True):
    """Average launch duration of the forward and backward sweep kernels, CUDA events on the launching stream
    around the C-ABI calls (parameters frozen: no Adam between launches).  Also returns the executed-pair counters
    of ONE such forward + backward (separate, counting instantiation of the kernels; not timed)."""
    import ctypes as C
    import torch
    from smoe_b200._ffi import check, lib, ptr, stream_ptr
    L, st = lib(), stream_ptr()
    b = m._batches[0]
    counts, regs, scal = m._counts[0], m._regsums[0], m._scalars[0]
    ax2 = ptr(m._d_axes[2]) if m.dim_domain == 3 else ptr(None)
    if m._raw_part is None:
        m._raw_part = torch.zeros((m._splits * m.start_pis * m._P,), dtype=torch.float32, device=m.device)
    check(L.smoe_pack(C.byref(m._cfg), ptr(m._theta), ptr(m._mus_grid), ptr(m._qdyn), ptr(m._klist[0]), ptr(m._perm),
                      m.start_pis, ptr(m._packed), ptr(m._indices), ptr(m._pos), ptr(counts), ptr(regs),
                      ptr(m._chunk_bounds), ptr(m._pack_ws), ptr(None), ptr(None), ptr(None), st), "pack")

    def fwd(pc=None):
        m._infl.zero_()
        scal.zero_()
        check(L.smoe_forward(C.byref(m._cfg), C.byref(b), ptr(m._packed), ptr(m._indices), ptr(counts),
                             ptr(m._chunk_bounds), m.start_pis, ptr(None), ptr(m._d_axes[0]), ptr(m._d_axes[1]), ax2,
                             ptr(m._d_res_pre), ptr(None), ptr(m._infl), ptr(m._pix), ptr(m._tile_qmin[0]), ptr(pc), st),
              "forward")

    def loss():
        check(L.smoe_loss(C.byref(m._cfg), C.byref(b), ptr(m._d_res_pre), ptr(m._d_image), ptr(None), ptr(None),
                          ptr(m._d_res), ptr(m._pix), ptr(scal), ptr(m._partials), ptr(m._ticket), st), "loss")

    def bwd(pc=None):
        check(L.smoe_backward(C.byref(m._cfg), C.byref(b), ptr(m._packed), ptr(counts), m.start_pis, ptr(m._pix),
                              ptr(m._tile_qmin[0]), ptr(m._d_axes[0]), ptr(m._d_axes[1]), ax2, m._splits,
                              ptr(m._raw_part), ptr(m._plan), ptr(pc), st), "backward")

    fw, bw, ls = [], [], []
    for _ in range(steps + 1):
        e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        m._infl.zero_()
        scal.zero_()
        e[0].record()
        fwd()
        e[1].record()
        loss()
        e[2].record()
        bwd()
        e[3].record()
        torch.cuda.synchronize()
        fw.append(e[0].elapsed_time(e[1]))
        ls.append(e[1].elapsed_time(e[2]))
        bw.append(e[2].elapsed_time(e[3]))
    fw, bw, ls = fw[1:], bw[1:], ls[1:]
    pc = torch.zeros((8,), dtype=torch.int64, device=m.device)
    fwd(pc)
    loss()
    bwd(pc)
    torch.cuda.synchronize()
    pairs = [int(v) for v in pc.cpu().numpy()]
    # loss stage: elementwise, HBM-bound: r (C f32) + target (C f32) read, res (C f32) + 1 + C planes written, gr plane read
    Cc = m.image.shape[-1]
    loss_bytes = float(np.prod(m._local_shape)) * 4 * (3 * Cc + 2 + Cc)
    out = {"forward_ms": float(np.mean(fw)), "backward_ms": float(np.mean(bw)), "loss_ms": float(np.mean(ls)),
           "loss_GBps": loss_bytes / (float(np.mean(ls)) / 1e3) / 1e9, "other_ms": 0.0, "pairs": pairs,
           "launches_timed": len(fw)}
    if with_step:
        # everything else in a step: pack, finalize / exchange, list upkeep, Adam, memsets
        step = event_time(lambda: m.run_batched(train=True), 5, warm=2)
        out["other_ms"] = max(0.0, step - out["forward_ms"] - out["backward_ms"] - out["loss_ms"])
    return out


def executed_roofline(ker, d, C, peak_tflops):
    """Roofline fraction on the work the kernels actually EXECUTE (lanes x pixels as issued, warp-granular), with the
    algorithmic cost of each part from SURVEY.md 8d: normaliser / gate part 2d+T+2, forward expert part C(d+1),
    backward gate + moment part 4d+2T+6, backward expert part 2dC+3C."""
    T = d * (d + 1) // 2
    f_gate, f_exp, f_bg, f_be = 2 * d + T + 2, C * (d + 1), 4 * d + 2 * T + 6, 2 * d * C + 3 * C
    p = ker["pairs"]
    fwd_li = p[1] * f_gate + p[3] * f_exp
    bwd_li = p[5] * f_bg + p[6] * f_be
    tf = lambda li, ms: li * 2 / (ms / 1e3) / 1e12
    return {"pairs_fwdA_evaluated": p[0], "pairs_fwdA": p[1], "pairs_fwdB_evaluated": p[2], "pairs_fwdB": p[3],
            "pairs_bwd_evaluated": p[4], "pairs_bwd": p[5], "pairs_bwd_expert": p[6],
            "lane_instr_per_pair": {"fwdA": f_gate, "fwdB_expert": f_exp, "bwd_gate_moments": f_bg, "bwd_expert": f_be},
            "frac_forward": tf(fwd_li, ker["forward_ms"]) / peak_tflops,
            "frac_backward": tf(bwd_li, ker["backward_ms"]) / peak_tflops,
            "frac": tf(fwd_li + bwd_li, ker["forward_ms"] + ker["backward_ms"]) / peak_tflops,
            "note": "pairs = lanes x pixels whose ex2 / accumulation part was issued (a warp executes a group for all "
                    "32 lanes when any lane needs it); 'evaluated' = pairs whose logit was computed for the skip test"}


def aux_hbm_pieces(m, img, peaks):
    """HBM-bound pieces on this workload's shapes, algorithmic bytes / device time (north_star: 'reported in GB/s')."""
    import ctypes as C
    import torch
    from smoe_b200._ffi import check, lib, ptr, stream_ptr
    L = lib()
    d, Cc = m.dim_domain, img.shape[-1]
    out = {}
    a = m._d_res.reshape(-1)
    b = m._d_image.reshape(-1)
    dims = (C.c_int32 * 3)(*m._dims3)
    ws = torch.empty((L.smoe_ssim_workspace_bytes(d, dims, Cc) + 7) // 8, dtype=torch.float64, device=m.device)
    o = torch.zeros(4, dtype=torch.float64, device=m.device)
    ms = event_time(lambda: check(L.smoe_ssim(d, dims, Cc, ptr(a), ptr(b), ptr(o), ptr(ws), stream_ptr()), "ssim"), 10, 2)
    alg = 2 * a.numel() * 4
    out["ssim_metric"] = {"ms": ms, "GBps": alg / ms / 1e6, "frac_hbm": alg / ms / 1e6 / peaks["hbm_gbs"]}
    ws2 = torch.empty(1024, dtype=torch.float64, device=m.device)
    o2 = torch.zeros(1, dtype=torch.float64, device=m.device)
    ms = event_time(lambda: check(L.smoe_sqerr(ptr(a), ptr(b), C.c_size_t(a.numel()), ptr(o2), ptr(ws2), stream_ptr()),
                                  "sqerr"), 10, 2)
    out["psnr_sqerr"] = {"ms": ms, "GBps": alg / ms / 1e6, "frac_hbm": alg / ms / 1e6 / peaks["hbm_gbs"]}
    K, P, PK = m.start_pis, m._P, m._PK
    ms = event_time(lambda: check(L.smoe_pack(C.byref(m._cfg), ptr(m._theta), ptr(m._mus_grid), ptr(m._qdyn),
                                              ptr(m._klist[0]), ptr(m._perm), K, ptr(m._packed), ptr(m._indices),
                                              ptr(m._pos), ptr(m._counts[0]), ptr(m._regsums[0]), ptr(m._chunk_bounds),
                                              ptr(m._pack_ws), ptr(None), ptr(None), ptr(None), stream_ptr()), "pack"), 10, 2)
    Ka = int(m._counts[0, 0].item())
    alg = K * (P * 4 + 1 + 4) + Ka * (PK * 4 + 4) + K * 4
    out["compaction"] = {"ms": ms, "K_all": K, "K_active": Ka, "GBps": alg / ms / 1e6,
                         "frac_hbm": alg / ms / 1e6 / peaks["hbm_gbs"]}
    return out


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(m, step_out, out_dir):
    """Writes what the last timed step hands its caller as out_dir/<name>.npy: run_batched's loss, mse and active
    kernel count (float64), the parameters after the step's Adam update, the step's gradients and the kernel
    influence lists (float32).  The inputs are seeded, so two builds run with the same arguments can be compared
    array by array."""
    loss, mse, num_pi, _ = step_out
    arrays = {"loss": np.float64([loss]), "mse": np.float64([mse]), "num_pi": np.float64([num_pi])}
    arrays.update({f"params_{k}": np.asarray(v, np.float32) for k, v in m.get_params().items()})
    arrays.update({f"grads_{k}": np.asarray(v, np.float32) for k, v in m.get_gradients().items()})
    arrays["kernel_list"] = np.stack(m.kernel_list_per_batch).astype(np.float32)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args):
    import torch
    import __graft_entry__ as ge
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local))
    if rank == 0:
        ge.build()
    if world > 1:
        torch.distributed.barrier()
    from smoe_b200 import Smoe, AdamOptimizer

    shape, kgrid, seed, desc = WORKLOADS[args.workload]
    d, C = len(shape) - 1, shape[-1]
    img = synth_image(shape, seed)

    def make(**kw):
        kws = dict(SMOE_KW)
        kws.update(kw)
        mm = Smoe(img, kernels_per_dim=kgrid, **kws)
        mm.set_optimizer(AdamOptimizer(1e-3), AdamOptimizer(1e-5), AdamOptimizer(1.0))
        return mm

    m = make(dense_exec=int(args.dense_exec), eps_bits=int(args.eps_bits))
    N, K = m.num_pixel, m.start_pis
    evals_per_step = float(N) * float(K)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    last_out = [None]           # run_batched's return value of the most recent timed step

    def timed_steps(mm, n, host_image=None, **kw):
        """n steps, each bracketed by its own CUDA events on the launching stream, L2 flushed
        (256 MB write) between steps outside the events; returns per-step ms (max over ranks)."""
        ms = []
        for _ in range(n):
            flush.fill_(1.0)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            if host_image is not None:
                mm.set_image(host_image)          # H2D of this step's pixels, inside the timed region
            last_out[0] = mm.run_batched(train=True, **kw)    # ends with the D2H read of the step's loss scalars + sync
            e1.record()
            torch.cuda.synchronize()
            t = torch.tensor([e0.elapsed_time(e1)], device="cuda")
            if world > 1:
                torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            ms.append(float(t.item()))
        return ms

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    timed_steps(m, max(args.warmup, 3))
    if rank == 0:
        time.sleep(0.3)
        sampler.rows.clear()          # keep only the samples taken from here on
    l0 = m.gpu_launches
    ms = timed_steps(m, args.steps)
    launches = (m.gpu_launches - l0) // max(args.steps, 1)
    n_timed_samples = len(sampler.rows) if rank == 0 else 0
    total_s = sum(ms) / 1e3
    value = evals_per_step * args.steps / total_s
    if args.dump_outputs and rank == 0:
        dump_outputs(m, last_out[0], args.dump_outputs)     # before the legs below move the model on

    # e2e: the same steps through the public API (Smoe.set_image + Smoe.run_batched) with this step's pixels coming
    # from pinned host memory -- the 8-bit pixels as an image file holds them; the /255 conversion (utils.py:126-128)
    # runs in the forward kernel -- and the loss scalars read back to the host
    u8 = np.round(img[m._local_slices] * 255).astype(np.uint8)
    assert np.array_equal(u8.astype(np.float32) / 255., img[m._local_slices])
    host_img = torch.from_numpy(np.ascontiguousarray(u8)).pin_memory()
    timed_steps(m, 3, host_img)
    ms_e2e = timed_steps(m, args.steps, host_img)
    e2e_value = evals_per_step * args.steps / (sum(ms_e2e) / 1e3)
    h2d = host_img.numel() * host_img.element_size()
    d2h = m._host_stats.numel() * 4
    m.set_image(torch.from_numpy(np.ascontiguousarray(img[m._local_slices])))
    torch.cuda.synchronize()

    # per-kernel durations and executed-pair counts of the two sweep kernels (CUDA events on the launching stream)
    ker = kernel_times(m, steps=max(3, min(args.steps, 10)))
    f_fwd, f_bwd = algorithmic_lane_instr(d, C)
    peaks, peak_src = measured_peaks()
    sms = torch.cuda.get_device_properties(local).multi_processor_count
    peak_tflops = sms * 128 * 2 * peaks["sm_max_mhz"] * 1e6 / 1e12
    local_evals = float(np.prod(m._local_shape)) * K
    tfl = lambda ev, F, t_ms: ev * F * 2 / (t_ms / 1e3) / 1e12
    roofline = {"bound": "fp32", "peak": peak_tflops, "unit": "TFLOP/s",
                "peak_source": f"{sms} SMs x 128 FP32 lanes x 2 x sm_max_mhz={peaks['sm_max_mhz']} ({peak_src} MEASURED_PEAKS.json)",
                "algorithmic_lane_instr_per_eval": {"fwd": f_fwd, "bwd": f_bwd},
                "product_mode": {"mode": {0: "exact culling + exact-zero skipping", 1: "every (pixel,kernel) pair executed",
                                          2: "exact-zero skipping only"}[int(args.dense_exec)] +
                                         (f" + epsilon culling 2^-{args.eps_bits}" if args.eps_bits else ""),
                                 "forward_ms": ker["forward_ms"], "backward_ms": ker["backward_ms"],
                                 "loss_ms": ker["loss_ms"], "loss_GBps": ker["loss_GBps"],
                                 "other_ms": ker["other_ms"], "launches_timed": ker["launches_timed"]},
                "executed": executed_roofline(ker, d, C, peak_tflops)}
    # dense_equivalent_speedup: how much faster than a kernel that executes all N*K pairs at 100 % of the FP32 roofline
    # the product-mode step is -- work provably not needed (exact zeros), NOT a roofline fraction
    roofline["dense_equivalent_speedup"] = tfl(local_evals, f_fwd + f_bwd, ker["forward_ms"] + ker["backward_ms"]) / peak_tflops

    # The same two kernels with EVERY (pixel, kernel) pair executed (dense_exec=1): the leg that compares like with
    # like against the algorithmic instruction count, and therefore the roofline fraction of this line.
    if int(args.dense_exec) != 1 and not args.no_dense:
        md = make(dense_exec=1)
        kd = kernel_times(md, steps=5, with_step=False)
        md.close()
        del md
    elif int(args.dense_exec) == 1:
        kd = ker
    else:
        kd = None
    if kd is not None:
        roofline.update({
            "kernel": f"smoe::forward_kernel<{d},{C}> + smoe::backward_kernel<{d},{C}>, dense_exec=1 (every pair executed)",
            "achieved": tfl(local_evals, f_fwd + f_bwd, kd["forward_ms"] + kd["backward_ms"]),
            "dense_forward_ms": kd["forward_ms"], "dense_backward_ms": kd["backward_ms"],
            "dense_launches_timed": kd["launches_timed"],
            "dense_forward": tfl(local_evals, f_fwd, kd["forward_ms"]) / peak_tflops,
            "dense_backward": tfl(local_evals, f_bwd, kd["backward_ms"]) / peak_tflops})
        roofline["frac"] = roofline["achieved"] / peak_tflops
    else:
        roofline.update({"kernel": "executed pairs of the product mode", "achieved": roofline["executed"]["frac"] * peak_tflops,
                         "frac": roofline["executed"]["frac"]})
    tr = os.path.join(ROOT, "profiles", "traffic.json")
    roofline["traffic"] = None
    if os.path.exists(tr):
        with open(tr) as fd:
            roofline["traffic"] = json.load(fd).get(f"{args.workload}@mode{int(args.dense_exec)}@world{world}")

    # a second state of the same workload: after `--pruned-iters` iterations with pis_l1 = 1.0 (pruned, wider kernels)
    states = None
    if args.pruned_iters > 0 and not args.eps_bits:
        for _ in range(args.pruned_iters):
            m.run_batched(train=True, pis_l1=1.0)
        m.update_kernel_list()
        ms_p = timed_steps(m, min(args.steps, 30), pis_l1=1.0)
        kp = kernel_times(m, steps=3, with_step=False)
        _, mse_p, num_pi, _ = m.run_batched(train=False)
        states = {"after_iters": args.pruned_iters, "pis_l1": 1.0, "active_kernels": int(m._counts[0, 0].item()),
                  "num_pi": int(num_pi), "psnr_db": float(10 * np.log10(65536.0 / max(mse_p, 1e-30))),
                  "ms_per_step": float(np.mean(ms_p)), "forward_ms": kp["forward_ms"], "backward_ms": kp["backward_ms"],
                  "value_active": float(N) * int(m._counts[0, 0].item()) / (float(np.mean(ms_p)) / 1e3),
                  "executed": executed_roofline(kp, d, C, peak_tflops)}

    aux = aux_hbm_pieces(m, img, peaks) if not args.no_aux else None

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu, _ = cpu_reference_evals_per_s(args.workload, 5, 1)
        cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
    clocks = None
    if rank == 0:
        clocks = sampler.stop()
        clocks["samples_in_timed_region"] = n_timed_samples
        clocks["window"] = "timed steps, e2e steps, per-kernel timing, dense_exec leg, pruned-state leg and aux pieces"
        if clocks.get("sm_mhz"):
            roofline["frac_at_observed_clock"] = roofline["frac"] * peaks["sm_max_mhz"] / clocks["sm_mhz"]
    if rank == 0:
        cfg = common_config(args.workload, world)
        cfg.update({"parallelism": (f"pixel blocks {'x'.join(str(v) for v in m._block_grid)} over {world} ranks, one "
                                    f"peer-memory exchange fused into grad_finalize per step") if world > 1 else "1 GPU",
                    "dense_exec": int(args.dense_exec), "eps_bits": int(args.eps_bits)})
        line = {"metric": "pixel_kernel_evals_per_s_fwd_bwd", "value": value, "unit": "evals/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": float(np.mean(ms)),
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": cfg, "iters_per_s": args.steps / total_s,
                "e2e": {"value": e2e_value, "unit": "evals/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": float(np.mean(ms_e2e)), "api": "Smoe.set_image(pinned uint8) + Smoe.run_batched(train=True)"},
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "states": states, "aux": aux,
                "cpu_baseline": cpu}
        print(json.dumps(line))
    if world > 1:
        torch.distributed.barrier()
        m.close()
        torch.distributed.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--dense-exec", type=int, default=0,
                    help="0: exact culling + exact-zero skipping (default); 1: execute every pair; 2: skipping only")
    ap.add_argument("--eps-bits", type=int, default=0, help="opt-in epsilon culling: drop terms below 2^-x of the normaliser")
    ap.add_argument("--pruned-iters", type=int, default=300, help="iterations with pis_l1=1 before the second state (0: skip)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-dense", action="store_true", help="skip the dense_exec=1 roofline leg")
    ap.add_argument("--no-aux", action="store_true", help="skip the HBM-bound aux pieces")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
