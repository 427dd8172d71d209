"""SmoePointRenderer (steered-mixture-of-experts_b200/render.py, csrc/points.cu): SMoE evaluation at arbitrary points,
differentiable in the parameters and in the coordinates.

Outputs and gradients are compared with the float64 restatement of the reference graph evaluated at the same float32
coordinates; the last two tests need no device (argument validation, register budget of the point kernels)."""
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
TAU = 0.5 / 256


def _rel(a, b):
    return float(np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)).max() / max(np.abs(b).max(), 1e-30))


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
    p["pis"][3] = -0.1                     # compacted away: no output, zero gradient
    return p, d, img.shape[-1]


def _cuda(p, grad=False):
    return {k: torch.tensor(np.asarray(v, np.float32), device="cuda", requires_grad=grad) for k, v in p.items()}


def _grads_np(p):
    return {k: p[k].grad.cpu().numpy() for k in PARAM_KEYS}


def _oracle(params, pts, cot, kw, C):
    """float64 graph r_pre at the float32 points, and its gradients (params and points) for `cot` zeroed on the points
    within float32 noise of a gate threshold."""
    from oracle.graph import GraphCfg, ambiguity_margins, graph_forward
    pts = np.asarray(pts, np.float32).reshape(-1, params["musX"].shape[1])
    d = pts.shape[1]
    K = params["pis"].shape[0]
    dom = torch.tensor(pts.astype(np.float64), requires_grad=True)
    cfg = GraphCfg(dim_domain=d, num_channels=C, use_yuv=False, start_pis=K, **kw)
    leaf = {k: torch.tensor(np.asarray(v, np.float64), requires_grad=True) for k, v in params.items()}
    out = graph_forward(leaf, np.ones(K, bool), dom, torch.zeros(dom.shape[0], C, dtype=torch.float64), cfg)
    ok = ambiguity_margins(out, cfg)[0] > 1e-3
    cot = np.where(ok[:, None], np.asarray(cot, np.float32).reshape(-1, C), 0).astype(np.float32)
    gr = torch.autograd.grad(out["r_pre"], [leaf[k] for k in PARAM_KEYS] + [dom],
                             grad_outputs=torch.tensor(cot.astype(np.float64)), allow_unused=True)
    g = {k: (np.zeros(leaf[k].shape) if gi is None else gi.numpy()) for k, gi in zip(PARAM_KEYS, gr)}
    return out["r_pre"].detach().numpy(), ok, cot, g, gr[-1].numpy()


def _check_against_oracle(p, pts_np, kw, C, cot_seed=13, min_ok=0.97):
    from smoe_b200 import SmoePointRenderer
    d = pts_np.shape[-1]
    r = SmoePointRenderer(d=d, channels=C, **kw)
    pt = _cuda(p, grad=True)
    pts = torch.tensor(pts_np, device="cuda", requires_grad=True)
    out = r(pt, pts)
    assert out.shape == pts_np.shape[:-1] + (C,)
    cot = np.random.RandomState(cot_seed).standard_normal(out.shape).astype(np.float32)
    ref, ok, cot_used, g_ref, gx_ref = _oracle(p, pts_np, cot, kw, C)
    out.backward(torch.tensor(cot_used.reshape(out.shape), device="cuda"))
    got = out.detach().cpu().numpy().reshape(-1, C)
    assert ok.mean() >= min_ok
    assert np.abs(got[ok] - ref[ok]).max() <= 1e-5
    assert np.abs(got - ref).max() <= 2 * TAU * max(1.0, float(np.abs(ref).max()))     # at most one gate flip
    g = _grads_np(pt)
    for key in PARAM_KEYS:
        assert _rel(g[key], g_ref[key]) < 1e-4, (key, _rel(g[key], g_ref[key]))
    assert all(np.all(g[key][3] == 0) for key in PARAM_KEYS)
    assert np.all(np.triu(g["A_corr"]) == 0)
    assert np.all(g["A_diagonal"] * (1 - np.eye(d)) == 0)
    gx = pts.grad.cpu().numpy().reshape(-1, d)
    assert _rel(gx, gx_ref) < 1e-4, _rel(gx, gx_ref)
    return out


def _rotated_grid(n0, n1, angle=0.4, scale=1.25):
    u, v = np.meshgrid(np.linspace(-0.5, 0.5, n0), np.linspace(-0.5, 0.5, n1), indexing="ij")
    c, s = np.cos(angle) * scale, np.sin(angle) * scale
    return np.stack([0.5 + c * u - s * v, 0.5 + s * u + c * v], -1).astype(np.float32)


CASES = {
    # name: (model, points as a function of a RandomState, flags)
    "gray_uniform_random": ("gray", lambda rs: rs.uniform(0, 1, (3000, 2)),
                            dict(use_determinant=True, train_inverse_cov=False)),
    "gray_uniform_random_plain": ("gray", lambda rs: rs.uniform(0, 1, (2000, 2)),
                                  dict(use_determinant=False, train_inverse_cov=False)),
    "rgb_rotated_scaled_grid": ("rgb", lambda rs: _rotated_grid(40, 52),
                                dict(use_determinant=False, train_inverse_cov=True)),
    "rgb_rotated_scaled_grid_det": ("rgb", lambda rs: _rotated_grid(33, 47, angle=-0.9, scale=1.4),
                                    dict(use_determinant=True, train_inverse_cov=True)),
    "video_random_between_frames": ("video", lambda rs: rs.uniform(0, 1, (2500, 3)),
                                    dict(use_determinant=True, train_inverse_cov=False)),
    "video_random_tic": ("video", lambda rs: rs.uniform(-0.05, 1.05, (1800, 3)),
                         dict(use_determinant=False, train_inverse_cov=True)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_points_match_the_float64_graph(name):
    model, pts_of, kw = CASES[name]
    p, d, C = _params(model, kw)
    pts = pts_of(np.random.RandomState(21)).astype(np.float32)
    _check_against_oracle(p, pts, kw, C)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 511, 513, 1024, 1536])
def test_edge_sizes_match_the_float64_graph(n):
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p, d, C = _params("rgb", kw)
    pts = np.random.RandomState(n).uniform(0, 1, (n, 2)).astype(np.float32)
    _check_against_oracle(p, pts, kw, C, min_ok=0.9 if n > 1 else 0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["identical", "duplicated"])
def test_identical_and_duplicated_points(kind):
    kw = dict(use_determinant=False, train_inverse_cov=False)
    p, d, C = _params("rgb", kw)
    rs = np.random.RandomState(4)
    if kind == "identical":                # one tile with a zero-extent box
        pts = np.tile(np.float32([[0.41, 0.57]]), (700, 1))
    else:
        base = rs.uniform(0, 1, (300, 2)).astype(np.float32)
        pts = base[rs.randint(0, 300, 1400)]
    _check_against_oracle(p, pts, kw, C, min_ok=0.0)


@pytest.mark.gpu
def test_points_shaped_like_an_image():
    kw = dict(use_determinant=True, train_inverse_cov=True)
    p, d, C = _params("rgb", kw)
    pts = _rotated_grid(30, 20)            # (H, W, 2) -> (H, W, 3)
    out = _check_against_oracle(p, pts, kw, C)
    assert out.shape == (30, 20, 3)


@pytest.mark.gpu
def test_points_on_a_grid_agree_with_the_grid_op():
    """The grid's coordinates, shuffled, as points: outputs and parameter gradients match SmoeRenderer."""
    from oracle.graph import GraphCfg, ambiguity_margins, graph_forward
    from smoe_b200 import SmoePointRenderer, SmoeRenderer
    from smoe_b200.render import plan_grid
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p, d, C = _params("rgb_big", kw)
    grid = [(-0.05, 1.05, 70), (0.0, 1.0, 90)]
    axes = plan_grid(grid, C)[0]
    pts = np.stack(np.meshgrid(*axes, indexing="ij"), -1).reshape(-1, 2)
    # gate-ambiguous pixels carry no cotangent, as in the oracle comparisons
    K = p["pis"].shape[0]
    cfg = GraphCfg(dim_domain=2, num_channels=C, use_yuv=False, start_pis=K, **kw)
    o = graph_forward({k: torch.tensor(np.asarray(v, np.float64)) for k, v in p.items()}, np.ones(K, bool),
                      torch.tensor(pts.astype(np.float64)), torch.zeros(len(pts), C, dtype=torch.float64), cfg)
    ok = ambiguity_margins(o, cfg)[0] > 1e-3
    cot = np.where(ok[:, None], np.random.RandomState(3).standard_normal((len(pts), C)), 0).astype(np.float32)
    pg = _cuda(p, grad=True)
    out_g = SmoeRenderer(grid=grid, channels=C, **kw)(pg)
    out_g.backward(torch.tensor(cot.reshape(out_g.shape), device="cuda"))
    perm = np.random.RandomState(5).permutation(len(pts))
    pp = _cuda(p, grad=True)
    out_p = SmoePointRenderer(d=2, channels=C, **kw)(pp, torch.tensor(pts[perm], device="cuda"))
    out_p.backward(torch.tensor(cot[perm], device="cuda"))
    a = out_g.detach().cpu().numpy().reshape(-1, C)
    b = np.empty_like(a)
    b[perm] = out_p.detach().cpu().numpy()
    assert np.abs(a[ok] - b[ok]).max() <= 1e-5
    assert np.abs(a - b).max() <= 2 * TAU * max(1.0, float(np.abs(a).max()))
    gg, gp = _grads_np(pg), _grads_np(pp)
    for key in PARAM_KEYS:
        assert _rel(gp[key], gg[key]) < 1e-4, (key, _rel(gp[key], gg[key]))


@pytest.mark.gpu
@pytest.mark.parametrize("cloud", ["clustered", "beyond_unit_square"])
def test_culling_is_exact(cloud):
    """dense_exec 0 (culling + skipping), 1 (every pair), 2 (skipping only): the same bits for outputs, parameter
    gradients and point gradients."""
    from smoe_b200 import SmoePointRenderer
    kw = dict(use_determinant=False, train_inverse_cov=True)
    p0, d, C = _params("rgb_big", kw)
    rs = np.random.RandomState(8)
    pts_np = (rs.uniform(0.40, 0.46, (5000, 2)) if cloud == "clustered" else rs.uniform(-0.3, 1.3, (6000, 2)))
    pts_np = pts_np.astype(np.float32)
    cot = torch.tensor(rs.standard_normal((len(pts_np), C)).astype(np.float32), device="cuda")
    res = []
    for mode in (0, 1, 2, 0):
        r = SmoePointRenderer(d=2, channels=C, _dense_exec=mode, **kw)
        p = _cuda(p0, grad=True)
        pts = torch.tensor(pts_np, device="cuda", requires_grad=True)
        out = r(p, pts)
        out.backward(cot)
        res.append([out.detach().cpu().numpy(), pts.grad.cpu().numpy()] + [p[k].grad.cpu().numpy() for k in PARAM_KEYS])
    for b in (1, 2, 3):
        for q in range(len(res[0])):
            np.testing.assert_array_equal(res[0][q], res[b][q])
    assert np.abs(res[0][1]).max() > 0 and np.abs(res[0][3]).max() > 0


@pytest.mark.gpu
def test_two_calls_in_one_graph_and_determinism():
    from smoe_b200 import SmoePointRenderer
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p0, d, C = _params("rgb_big", kw)
    rs = np.random.RandomState(1)
    a_np, b_np = rs.uniform(0, 1, (4000, 2)).astype(np.float32), rs.uniform(0.2, 0.7, (2500, 2)).astype(np.float32)
    r = SmoePointRenderer(d=2, channels=C, **kw)

    def f(x):
        return (x.clamp(0, 1) - 0.5).abs().mean()

    def h(x):
        return (x * x).sum() * 1e-3

    def run(both):
        p = _cuda(p0, grad=True)
        a = torch.tensor(a_np, device="cuda", requires_grad=True)
        b = torch.tensor(b_np, device="cuda", requires_grad=True)
        if both is None:
            (f(r(p, a)) + h(r(p, b))).backward()
        elif both == "a":
            f(r(p, a)).backward()
        else:
            h(r(p, b)).backward()
        return _grads_np(p), a.grad, b.grad

    g_ab, ga, gb = run(None)
    g_a, ga1, _ = run("a")
    g_b, _, gb1 = run("b")
    for k in PARAM_KEYS:
        np.testing.assert_array_equal(g_ab[k], g_a[k] + g_b[k], err_msg=k)
    assert torch.equal(ga, ga1) and torch.equal(gb, gb1)
    g_ab2, ga2, gb2 = run(None)                 # the same call twice: the same bits
    for k in PARAM_KEYS:
        np.testing.assert_array_equal(g_ab[k], g_ab2[k], err_msg=k)
    assert torch.equal(ga, ga2) and torch.equal(gb, gb2)
    with torch.no_grad():
        pn = _cuda(p0)
        assert torch.equal(r(pn, torch.tensor(a_np, device="cuda")), r(pn, torch.tensor(a_np, device="cuda")))


@pytest.mark.gpu
def test_no_host_sync_no_state_without_grad_and_only_the_needed_sweeps():
    from torch.profiler import ProfilerActivity, profile
    from smoe_b200 import SmoePointRenderer
    from smoe_b200 import _ffi
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p0, d, C = _params("rgb_big", kw)
    pts_np = np.random.RandomState(2).uniform(0, 1, (200000, 2)).astype(np.float32)
    r = SmoePointRenderer(d=2, channels=C, **kw)
    p = _cuda(p0, grad=True)
    pts = torch.tensor(pts_np, device="cuda", requires_grad=True)
    r(p, pts).sum().backward()                 # warm-up: allocator, module loading
    for k in PARAM_KEYS:
        p[k].grad = None
    pts.grad = None
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        out = r(p, pts)
        (out * out).sum().backward()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert all(p[k].grad is not None for k in PARAM_KEYS) and pts.grad is not None
    del out
    # no backward state under no_grad: the forward is asked for none, and the output holds no graph
    kept = []
    fwd = r._forward
    r._forward = lambda points, ts, keep_state: (kept.append(keep_state), fwd(points, ts, keep_state))[1]
    try:
        with torch.no_grad():
            out = r(p, pts)
        assert out.grad_fn is None and kept == [False]
        out = r(p, pts)
        assert out.grad_fn is not None and kept == [False, True]
    finally:
        del r._forward
    del out
    state_bytes = _ffi.lib().smoe_point_tiles(len(pts_np)) * r._stride * 4
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    with torch.no_grad():
        out = r(p, pts)
    grown = torch.cuda.memory_allocated() - base            # only the output stays (in 512-byte allocator blocks)
    assert out.numel() * 4 <= grown < out.numel() * 4 + 512 and grown < state_bytes, (grown, state_bytes)
    del out

    def kernels(params_grad, points_grad):
        q = _cuda(p0, grad=params_grad)
        x = torch.tensor(pts_np, device="cuda", requires_grad=points_grad)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            r(q, x).sum().backward()
            torch.cuda.synchronize()
        return " ".join(e.key for e in prof.key_averages())

    only_points = kernels(False, True)
    assert "point_xgrad_kernel" in only_points and "point_backward_kernel" not in only_points
    assert "point_plan_kernel" not in only_points
    only_params = kernels(True, False)
    assert "point_backward_kernel" in only_params and "point_xgrad_kernel" not in only_params
    with pytest.raises(RuntimeError):          # a call's backward state is consumed by its one backward
        out = r(p, pts)
        out.sum().backward(retain_graph=True)
        out.sum().backward()


def test_argument_validation():
    """Bad arguments raise ValueError before any device work (no device needed for these)."""
    from smoe_b200.render import MAX_POINTS, SmoePointRenderer, check_points
    for kw in (dict(d=1), dict(d=4), dict(d=True), dict(channels=2), dict(channels=True), dict(precision=0),
               dict(precision=2.5), dict(_dense_exec=3)):
        with pytest.raises(ValueError):
            SmoePointRenderer(**kw)
    cpu = torch.device("cpu")
    assert check_points(torch.zeros(7, 2), 2, cpu) == 7
    assert check_points(torch.zeros(3, 5, 3), 3, cpu) == 15
    bad = [
        (np.zeros((4, 2), np.float32), 2),                       # not a tensor
        (torch.zeros(4, 2, dtype=torch.float64), 2),             # dtype
        (torch.zeros(4, 3), 2),                                  # d mismatch
        (torch.zeros(4), 2),                                     # no coordinate axis of size d
        (torch.zeros(0, 2), 2),                                  # N = 0
        (torch.zeros(()), 2),                                    # a scalar
    ]
    for pts, d in bad:
        with pytest.raises(ValueError):
            check_points(pts, d, cpu)
    big = torch.empty((MAX_POINTS + 1, 2), device="meta")    # no memory: only the shape is read
    with pytest.raises(ValueError):
        check_points(big.to(torch.float32), 2, torch.device("meta"))
    if torch.cuda.is_available():
        with pytest.raises(ValueError):                          # device mismatch
            check_points(torch.zeros(4, 2), 2, torch.device("cuda", 0))


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if cand and os.path.exists(cand):
            return cand
    return None


def test_point_kernels_are_spill_free_within_their_launch_bounds():
    """csrc/points.cu alone for sm_100a with -Xptxas -v: every instantiation spills nothing and uses no more registers
    than its __launch_bounds__ (threads, CTAs per SM) leave per thread."""
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip("nvcc not found")
    csrc = os.path.join(ROOT, "steered-mixture-of-experts_b200", "csrc")
    with tempfile.TemporaryDirectory() as tmp:
        cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-c",
               "-o", os.path.join(tmp, "points.o"), os.path.join(csrc, "points.cu")]
        r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    # kernel -> (threads, resident CTAs per SM) of its __launch_bounds__, as a function of d
    bounds = {"point_forward_kernel": lambda d: (128, 6 if d == 2 else 4), "point_xgrad_kernel": lambda d: (128, 4),
              "point_backward_kernel": lambda d: (64, 8), "point_plan_kernel": lambda d: (128, 1),
              "point_cotangent_kernel": lambda d: (256, 1)}
    seen = {}
    for block in r.stderr.split("Compiling entry function '")[1:]:
        name = block.split("'", 1)[0]
        kern = next((k for k in bounds if k in name), None)
        if kern is None:
            continue
        m = re.search(r"ILi(\d)E", name)
        d = int(m.group(1)) if m and kern != "point_cotangent_kernel" else 2
        regs = int(re.search(r"Used (\d+) registers", block).group(1))
        spill = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", block)
        threads, ctas = bounds[kern](d)
        limit = min(255, 65536 // (threads * ctas) // 8 * 8)
        seen[name] = (regs, limit, tuple(int(g) for g in spill.groups()))
        assert regs <= limit and spill.groups() == ("0", "0", "0"), (name, seen[name])
    counts = {k: sum(k in n for n in seen) for k in bounds}
    assert counts == {"point_forward_kernel": 8, "point_xgrad_kernel": 4, "point_backward_kernel": 8,
                      "point_plan_kernel": 4, "point_cotangent_kernel": 2}, counts
