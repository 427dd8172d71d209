"""SmoePointRenderer.jacobian and SmoeRenderer.jacobian (steered-mixture-of-experts_b200/render.py, csrc/jacobian.cu):
the spatial Jacobian J[..., c, l] = d r_c / d x_l at arbitrary points and on uniform grids, in one CUDA sweep after
the forward.

J is compared with the float64 restatement of the reference graph at the same float32 coordinates (row c of every
point's Jacobian is the coordinate gradient of sum_n r_pre[n, c], since points are independent), with the reverse
path (sum_c g_c J[:, c] is dL/dx for the cotangent g), across the execution modes, and used for the Gauss-Newton
registration it exists for.  The last tests need no device (argument validation, register budget, exports)."""
import os
import re
import shutil
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from conftest import ROOT

PARAM_KEYS = ("pis", "musX", "A_diagonal", "A_corr", "gamma_e", "nu_e")

MODELS = {
    # name: (image shape, kernels per dim, seed)
    "gray": ((32, 40, 1), [6, 8], 7),
    "rgb": ((24, 32, 3), [5, 6], 8),
    "video": ((12, 16, 6, 3), [3, 4, 3], 9),
    "rgb_big": ((96, 160, 3), [24, 40], 6),
}


def _params(name, kw, seed=5):
    """A model's initial parameters with steered kernels, sloped experts and one kernel with pi <= 0."""
    import bench
    from smoe_b200 import Smoe
    shape, k, s = MODELS[name]
    img = bench.synth_image(shape, s)
    d = img.ndim - 1
    p = Smoe(img, kernels_per_dim=k, **kw).get_params()
    rs = np.random.RandomState(seed)
    steer = rs.normal(0, 0.2 * p["A_diagonal"].max(), p["A_corr"].shape).astype(np.float32)
    p["A_corr"] = np.where(np.tril(np.ones((d, d), bool), -1)[None], steer * (0.3 if kw["train_inverse_cov"] else 1.0),
                           0).astype(np.float32)
    p["gamma_e"] = rs.normal(0, 0.3, p["gamma_e"].shape).astype(np.float32)
    p["pis"][3] = -0.1
    return p, d, img.shape[-1]


def _cuda(p, grad=False):
    return {k: torch.tensor(np.asarray(v, np.float32), device="cuda", requires_grad=grad) for k, v in p.items()}


def _rotated_grid(n0, n1, angle=0.4, scale=1.25):
    u, v = np.meshgrid(np.linspace(-0.5, 0.5, n0), np.linspace(-0.5, 0.5, n1), indexing="ij")
    c, s = np.cos(angle) * scale, np.sin(angle) * scale
    return np.stack([0.5 + c * u - s * v, 0.5 + s * u + c * v], -1).astype(np.float32)


def _oracle_jacobian(params, pts, kw, C):
    """float64 graph r_pre (N, C) and Jacobian (N, C, d) at the float32 points, and the points whose gates are not
    within float32 noise of the threshold."""
    from oracle.graph import GraphCfg, ambiguity_margins, graph_forward
    d = params["musX"].shape[1]
    pts = np.asarray(pts, np.float32).reshape(-1, d)
    K = params["pis"].shape[0]
    dom = torch.tensor(pts.astype(np.float64), requires_grad=True)
    cfg = GraphCfg(dim_domain=d, num_channels=C, use_yuv=False, start_pis=K, **kw)
    leaf = {k: torch.tensor(np.asarray(v, np.float64)) for k, v in params.items()}
    out = graph_forward(leaf, np.ones(K, bool), dom, torch.zeros(dom.shape[0], C, dtype=torch.float64), cfg)
    ok = ambiguity_margins(out, cfg)[0] > 1e-3
    J = np.stack([torch.autograd.grad(out["r_pre"][:, c].sum(), dom, retain_graph=True)[0].numpy()
                  for c in range(C)], 1)
    return out["r_pre"].detach().numpy(), J, ok


def _check_against_oracle(p, pts_np, kw, C):
    from smoe_b200 import SmoePointRenderer
    d = pts_np.shape[-1]
    r, J = SmoePointRenderer(d=d, channels=C, **kw).jacobian(_cuda(p), torch.tensor(pts_np, device="cuda"))
    assert r.shape == pts_np.shape[:-1] + (C,) and J.shape == pts_np.shape[:-1] + (C, d)
    r_ref, J_ref, ok = _oracle_jacobian(p, pts_np, kw, C)
    got_r = r.cpu().numpy().reshape(-1, C)
    got_J = J.cpu().numpy().reshape(-1, C, d)
    assert ok.mean() >= 0.97, ok.mean()
    assert np.abs(got_r[ok] - r_ref[ok]).max() <= 1e-5
    err = np.abs(got_J[ok] - J_ref[ok]).max() / max(np.abs(J_ref[ok]).max(), 1e-30)
    assert err <= 1e-4, err
    return got_J


CASES = {
    # name: (model, points as a function of a RandomState, flags)
    "gray_random_det": ("gray", lambda rs: rs.uniform(0, 1, (3000, 2)), dict(use_determinant=True,
                                                                           train_inverse_cov=False)),
    "gray_random_inverse_cov": ("gray", lambda rs: rs.uniform(0, 1, (2000, 2)), dict(use_determinant=False,
                                                                                   train_inverse_cov=True)),
    "rgb_rotated_scaled_grid": ("rgb", lambda rs: _rotated_grid(40, 52), dict(use_determinant=False,
                                                                               train_inverse_cov=True)),
    "rgb_rotated_scaled_grid_det": ("rgb", lambda rs: _rotated_grid(33, 47, angle=-0.9, scale=1.4),
                                    dict(use_determinant=True, train_inverse_cov=False)),
    "video_between_frames": ("video", lambda rs: rs.uniform(0, 1, (2500, 3)), dict(use_determinant=True,
                                                                                 train_inverse_cov=True)),
    "video_random_plain": ("video", lambda rs: rs.uniform(-0.05, 1.05, (1800, 3)), dict(use_determinant=False,
                                                                                      train_inverse_cov=False)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_jacobian_matches_the_float64_graph(name):
    model, pts_of, kw = CASES[name]
    p, d, C = _params(model, kw)
    pts = pts_of(np.random.RandomState(21)).astype(np.float32)
    J = _check_against_oracle(p, pts, kw, C)
    assert np.abs(J).max() > 0


@pytest.mark.gpu
def test_video_jacobian_at_times_between_frames():
    """A 2T-1 sampling of the time axis: every other time lies between two frames of the training video."""
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p, d, C = _params("video", kw)
    g = np.meshgrid(np.linspace(0, 1, 12), np.linspace(0, 1, 16), np.linspace(0, 1, 2 * 6 - 1), indexing="ij")
    _check_against_oracle(p, np.stack(g, -1).astype(np.float32), kw, C)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 511, 513, 1024, 1536])
def test_jacobian_edge_sizes(n):
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p, d, C = _params("rgb", kw)
    pts = np.random.RandomState(n).uniform(0, 1, (max(n, 64), 2)).astype(np.float32)
    if n == 1:                             # one point whose gates are clear of the threshold: ok.all() below
        pts = pts[np.argmax(_oracle_jacobian(p, pts, kw, C)[2])][None]
    _check_against_oracle(p, pts[:n], kw, C)


@pytest.mark.gpu
@pytest.mark.parametrize("C_", [1, 3])
def test_jacobian_agrees_with_the_reverse_path(C_):
    """sum_c g_c J[:, c, :] is the coordinate gradient of the backward for the cotangent g, and jacobian()'s r is the
    grad-enabled forward's output bit for bit."""
    from smoe_b200 import SmoePointRenderer
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p0, d, C = _params("rgb_big" if C_ == 3 else "gray", kw)
    pts_np = np.random.RandomState(3).uniform(-0.1, 1.1, (7000, 2)).astype(np.float32)
    ren = SmoePointRenderer(d=d, channels=C, **kw)
    p = _cuda(p0, grad=True)
    x = torch.tensor(pts_np, device="cuda", requires_grad=True)
    out = ren(p, x)
    g = torch.tensor(np.random.RandomState(4).standard_normal((len(pts_np), C)).astype(np.float32), device="cuda")
    out.backward(g)
    r, J = ren.jacobian(p, x)
    assert not r.requires_grad and not J.requires_grad and r.grad_fn is None and J.grad_fn is None
    assert torch.equal(r, out.detach())
    vjp = torch.einsum("nc,ncl->nl", g.double(), J.double()).cpu().numpy()
    gx = x.grad.double().cpu().numpy()
    assert np.abs(vjp - gx).max() <= 1e-5 * np.abs(gx).max(), np.abs(vjp - gx).max() / np.abs(gx).max()


@pytest.mark.gpu
@pytest.mark.parametrize("cloud", ["clustered", "beyond_unit_square"])
def test_jacobian_modes_and_determinism(cloud):
    """dense_exec 0 (culling + skipping), 1 (every pair), 2 (skipping only), and the same call twice: the same bits."""
    from smoe_b200 import SmoePointRenderer
    kw = dict(use_determinant=False, train_inverse_cov=True)
    p0, d, C = _params("rgb_big", kw)
    rs = np.random.RandomState(8)
    pts_np = (rs.uniform(0.40, 0.46, (5000, 2)) if cloud == "clustered" else rs.uniform(-0.3, 1.3, (6000, 2)))
    pts = torch.tensor(pts_np.astype(np.float32), device="cuda")
    p = _cuda(p0)
    res = [SmoePointRenderer(d=2, channels=C, _dense_exec=mode, **kw).jacobian(p, pts) for mode in (0, 1, 2, 0)]
    for b in (1, 2, 3):
        assert torch.equal(res[0][0], res[b][0]) and torch.equal(res[0][1], res[b][1]), b
    assert res[0][1].abs().max() > 0


@pytest.mark.gpu
def test_jacobian_syncs_nothing_and_runs_only_the_forward_and_its_sweep():
    from torch.profiler import ProfilerActivity, profile
    from smoe_b200 import SmoePointRenderer
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p0, d, C = _params("rgb_big", kw)
    pts = torch.tensor(np.random.RandomState(2).uniform(0, 1, (200000, 2)).astype(np.float32), device="cuda",
                       requires_grad=True)
    ren = SmoePointRenderer(d=2, channels=C, **kw)
    p = _cuda(p0, grad=True)
    ren.jacobian(p, pts)                          # warm-up: allocator, module loading
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        r, J = ren.jacobian(p, pts)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert not r.requires_grad and not J.requires_grad
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ren.jacobian(p, pts)
        torch.cuda.synchronize()
    names = [e.key for e in prof.key_averages()]
    point = [n for n in names if "point_" in n]
    assert any("point_forward_kernel" in n for n in point) and any("point_jacobian_kernel" in n for n in point)
    assert all("point_forward_kernel" in n or "point_jacobian_kernel" in n for n in point), point


GRID_CASES = {
    # name: (model, grid axes as a function of the image shape, flags)
    "rgb_super_resolution_2x": ("rgb", lambda sh: [(0, 1, 2 * sh[0]), (0, 1, 2 * sh[1])],
                                dict(use_determinant=True, train_inverse_cov=False)),
    "gray_crop": ("gray", lambda sh: [(0.2, 0.55, 47), (0.3, 0.8, 61)], dict(use_determinant=False,
                                                                              train_inverse_cov=True)),
    "video_2t_minus_1": ("video", lambda sh: [(0, 1, sh[0]), (0, 1, sh[1]), (0, 1, 2 * sh[2] - 1)],
                         dict(use_determinant=True, train_inverse_cov=True)),
}


def _grid_points(grid, C):
    from smoe_b200.render import plan_grid
    axes = plan_grid(grid, C)[0]
    return np.stack(np.meshgrid(*axes, indexing="ij"), -1)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(GRID_CASES))
def test_grid_jacobian_matches_the_float64_graph_and_the_point_kernel(name):
    from smoe_b200 import SmoePointRenderer, SmoeRenderer
    model, grid_of, kw = GRID_CASES[name]
    p, d, C = _params(model, kw)
    grid = grid_of(MODELS[model][0])
    r, J = SmoeRenderer(grid=grid, channels=C, **kw).jacobian(_cuda(p))
    pts = _grid_points(grid, C)
    assert r.shape == pts.shape[:-1] + (C,) and J.shape == pts.shape[:-1] + (C, d)
    r_ref, J_ref, ok = _oracle_jacobian(p, pts, kw, C)
    got_r, got_J = r.cpu().numpy().reshape(-1, C), J.cpu().numpy().reshape(-1, C, d)
    assert ok.mean() >= 0.97, ok.mean()
    assert np.abs(got_r[ok] - r_ref[ok]).max() <= 1e-5
    assert np.abs(got_J[ok] - J_ref[ok]).max() <= 1e-4 * np.abs(J_ref[ok]).max()
    # the point kernel at the same float32 coordinates (its own tiles, so other roundings of x')
    r_p, J_p = SmoePointRenderer(d=d, channels=C, **kw).jacobian(_cuda(p), torch.tensor(pts, device="cuda"))
    J_p = J_p.cpu().numpy().reshape(-1, C, d)
    assert np.abs(got_J[ok] - J_p[ok]).max() <= 1e-5 * np.abs(J_p[ok]).max()


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["rgb", "video"])
def test_grid_jacobian_r_is_the_render_and_modes_agree(model):
    """On (0, 1, n) axes r is SmoeRenderer's no-grad output bit for bit; dense_exec 0, 1, 2 and a repeat call give
    the same bits."""
    from smoe_b200 import SmoeRenderer
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p0, d, C = _params(model, kw)
    p = _cuda(p0, grad=True)
    grid = [(0, 1, n) for n in MODELS[model][0][:d]]
    with torch.no_grad():
        ref = SmoeRenderer(grid=grid, channels=C, **kw)(p)
    res = [SmoeRenderer(grid=grid, channels=C, _dense_exec=mode, **kw).jacobian(p) for mode in (0, 1, 2, 0)]
    assert not res[0][0].requires_grad and not res[0][1].requires_grad
    assert torch.equal(res[0][0], ref)
    for b in (1, 2, 3):
        assert torch.equal(res[0][0], res[b][0]) and torch.equal(res[0][1], res[b][1]), b
    assert res[0][1].abs().max() > 0


@pytest.mark.gpu
def test_grid_jacobian_syncs_nothing_and_runs_only_the_forward_and_its_sweep():
    from torch.profiler import ProfilerActivity, profile
    from smoe_b200 import SmoeRenderer
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p0, d, C = _params("rgb_big", kw)
    ren = SmoeRenderer(grid=[(0, 1, 480), (0, 1, 800)], channels=C, **kw)
    p = _cuda(p0, grad=True)
    ren.jacobian(p)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        ren.jacobian(p)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ren.jacobian(p)
        torch.cuda.synchronize()
    names = [e.key for e in prof.key_averages() if "smoe::" in e.key]
    assert any("forward_kernel" in n for n in names) and any("grid_jacobian_kernel" in n for n in names)
    assert not any(k in n for n in names for k in ("backward", "cotangent", "xgrad", "loss")), names


@pytest.mark.gpu
def test_gauss_newton_recovers_a_translation():
    """t <- t - (sum J^T J)^-1 sum J^T (r(x + t) - target), sums over points and channels: the registration J is for."""
    from smoe_b200 import SmoePointRenderer
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p0, d, C = _params("rgb_big", kw)
    p = _cuda(p0)
    ren = SmoePointRenderer(d=2, channels=C, **kw)
    g = np.meshgrid(np.linspace(0.15, 0.85, 90), np.linspace(0.15, 0.85, 150), indexing="ij")
    x = torch.tensor(np.stack(g, -1).reshape(-1, 2).astype(np.float32), device="cuda")
    t0 = torch.tensor([0.011, -0.017], device="cuda")
    with torch.no_grad():
        target = ren(p, x + t0)
    t = torch.zeros(2, device="cuda")
    for it in range(10):
        r, J = ren.jacobian(p, x + t)
        J64, res = J.double(), (r - target).double()
        H = torch.einsum("ncl,ncm->lm", J64, J64)
        b = torch.einsum("ncl,nc->l", J64, res)
        t = t - torch.linalg.solve(H, b).float()
        if float((t - t0).norm()) < 2e-4:
            break
    assert float((t - t0).norm()) < 2e-4, (it, t.tolist())


def test_jacobian_argument_validation():
    """jacobian() rejects exactly what a call rejects, with ValueError before any device work (no device needed)."""
    from smoe_b200 import SmoePointRenderer
    ren = SmoePointRenderer.__new__(SmoePointRenderer)       # no device: only the checks run
    ren.d, ren.C, ren.device = 2, 3, torch.device("cpu")
    K = 4
    good = dict(pis=torch.ones(K), musX=torch.zeros(K, 2), A_diagonal=torch.zeros(K, 2, 2),
                A_corr=torch.zeros(K, 2, 2), gamma_e=torch.zeros(K, 2, 3), nu_e=torch.zeros(K, 3))
    pts = torch.zeros(5, 2)
    bad = [
        ({k: v for k, v in good.items() if k != "pis"}, pts),                  # a key missing
        (dict(good, extra=torch.zeros(K)), pts),                               # an extra key
        (dict(good, musX=torch.zeros(K, 3)), pts),                             # shape
        (dict(good, nu_e=torch.zeros(K, 3, dtype=torch.float64)), pts),        # dtype
        (dict(good, gamma_e=np.zeros((K, 2, 3), np.float32)), pts),            # not a tensor
        (dict(good, pis=torch.ones(K, device="meta")), pts),                   # params on another device
        (good, np.zeros((5, 2), np.float32)),                                  # points not a tensor
        (good, torch.zeros(5, 2, dtype=torch.float64)),                        # points dtype
        (good, torch.zeros(5, 3)),                                             # d mismatch
        (good, torch.zeros(0, 2)),                                             # no point
        (good, torch.zeros(5, 2, device="meta")),                              # points on another device
    ]
    for params, x in bad:
        with pytest.raises(ValueError):
            ren.jacobian(params, x)
        with pytest.raises(ValueError):
            ren(params, x)


def test_grid_jacobian_argument_validation():
    """SmoeRenderer.jacobian rejects exactly what a call rejects, with ValueError before any device work."""
    from smoe_b200 import SmoeRenderer
    ren = SmoeRenderer.__new__(SmoeRenderer)                 # no device: only the checks run
    ren.d, ren.C, ren.device = 2, 3, torch.device("cpu")
    K = 4
    good = dict(pis=torch.ones(K), musX=torch.zeros(K, 2), A_diagonal=torch.zeros(K, 2, 2),
                A_corr=torch.zeros(K, 2, 2), gamma_e=torch.zeros(K, 2, 3), nu_e=torch.zeros(K, 3))
    bad = [{k: v for k, v in good.items() if k != "nu_e"}, dict(good, gamma_e=torch.zeros(K, 2, 1)),
           dict(good, pis=torch.ones(K, dtype=torch.float16)), dict(good, musX=torch.zeros(K, 2, device="meta")),
           [1, 2, 3]]
    for params in bad:
        with pytest.raises(ValueError):
            ren.jacobian(params)
        with pytest.raises(ValueError):
            ren(params)


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if cand and os.path.exists(cand):
            return cand
    return None


def test_jacobian_kernels_are_spill_free_within_their_launch_bounds():
    """csrc/jacobian.cu alone for sm_100a with -Xptxas -v: each point and grid (d, C) instantiation spills nothing and uses no more
    registers than its __launch_bounds__ (128 threads; 4 CTAs per SM, 3 at (3, 3)) leave per thread."""
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip("nvcc not found")
    csrc = os.path.join(ROOT, "steered-mixture-of-experts_b200", "csrc")
    with tempfile.TemporaryDirectory() as tmp:
        cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-c",
               "-o", os.path.join(tmp, "jacobian.o"), os.path.join(csrc, "jacobian.cu")]
        r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    seen = {}
    for block in r.stderr.split("Compiling entry function '")[1:]:
        name = block.split("'", 1)[0]
        m = re.search(r"(point|grid)_jacobian_kernelILi(\d)ELi(\d)E", name)
        if m is None:
            continue
        d, C = int(m.group(2)), int(m.group(3))
        regs = int(re.search(r"Used (\d+) registers", block).group(1))
        spill = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", block)
        limit = min(255, 65536 // (128 * (3 if (d, C) == (3, 3) else 4)) // 8 * 8)
        seen[(m.group(1), d, C)] = regs
        assert regs <= limit and spill.groups() == ("0", "0", "0"), (name, regs, limit, spill.groups())
    assert sorted(seen) == [(k, d, C) for k in ("grid", "point") for d in (2, 3) for C in (1, 3)], seen


def test_the_jacobian_call_is_declared_and_exported():
    from smoe_b200 import _ffi
    hdr = open(os.path.join(ROOT, "include", "smoe_b200.h")).read()
    for sym in ("smoe_point_jacobian", "smoe_jacobian"):
        assert re.search(r"\bint " + sym + r"\(", hdr) and sym in _ffi.EXPORTS
        if os.path.exists(_ffi.LIB_PATH):
            import ctypes
            assert hasattr(ctypes.CDLL(_ffi.LIB_PATH), sym)
    assert _ffi.ABI_VERSION == 6
