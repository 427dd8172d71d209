"""Forward mode of SmoeRenderer and SmoePointRenderer (steered-mixture-of-experts_b200/render.py, csrc/jvp.cu):
Jacobian-vector products dr = (d r / d params) v + (d r / d x) xdot under torch.func.jvp and forward_ad, from
smoe_pack_tangent and one CUDA sweep after the forward.

The reference is the forward-mode derivative of the float64 restatement of the reference graph (r_pre), taken with
the double-backward identity J v = d/du <J^T u, v>, at the points whose gates are not within float32 noise of the
threshold.  The JVP is also checked against jacobian() (point tangents), the reverse path (adjoint identity, and a
Gauss-Newton refit of the experts by CG on J^T J), across the execution modes, and inside autograd.  The last tests
need no device (argument validation, register budget, exports)."""
import ctypes
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest
import torch
import torch.autograd.forward_ad as fwAD

from conftest import ROOT
from test_jacobian_gpu import MODELS, _cuda, _grid_points, _nvcc, _params, _rotated_grid

PARAM_KEYS = ("pis", "musX", "A_diagonal", "A_corr", "gamma_e", "nu_e")
GROUPS = {"all": PARAM_KEYS, "pis": ("pis",), "musX": ("musX",), "A": ("A_diagonal", "A_corr"),
          "experts": ("nu_e", "gamma_e")}


def _tangent(p, group, seed=11):
    """A random tangent on the tensors of `group` (zeros elsewhere), numpy float32, the params' layout."""
    rs = np.random.RandomState(seed)
    return {k: (rs.standard_normal(np.shape(v)) * (0.05 if k == "musX" else 0.3) if k in GROUPS[group]
                else np.zeros(np.shape(v))).astype(np.float32) for k, v in p.items()}


def _oracle_jvp(params, pts, kw, C, dparams=None, dpts=None):
    """float64 graph r_pre (N, C) and J v (N, C) at the float32 points for the tangent (dparams, dpts), and the points
    whose gates are not within float32 noise of the threshold."""
    from oracle.graph import GraphCfg, ambiguity_margins, graph_forward
    d = params["musX"].shape[1]
    pts = np.asarray(pts, np.float32).reshape(-1, d)
    K = params["pis"].shape[0]
    dom = torch.tensor(pts.astype(np.float64), requires_grad=True)
    cfg = GraphCfg(dim_domain=d, num_channels=C, use_yuv=False, start_pis=K, **kw)
    leaf = {k: torch.tensor(np.asarray(v, np.float64), requires_grad=True) for k, v in params.items()}
    out = graph_forward(leaf, np.ones(K, bool), dom, torch.zeros(dom.shape[0], C, dtype=torch.float64), cfg)
    ok = ambiguity_margins(out, cfg)[0] > 1e-3
    rp = out["r_pre"]
    ins, vs = [], []
    for k, v in (dparams or {}).items():
        ins.append(leaf[k])
        vs.append(torch.tensor(np.asarray(v, np.float64)))
    if dpts is not None:
        ins.append(dom)
        vs.append(torch.tensor(np.asarray(dpts, np.float64).reshape(-1, d)))
    if not ins:
        return rp.detach().numpy(), np.zeros(tuple(rp.shape)), ok
    u = torch.zeros_like(rp, requires_grad=True)
    g = torch.autograd.grad(rp, ins, grad_outputs=u, create_graph=True, allow_unused=True)
    s = sum((gi * vi).sum() for gi, vi in zip(g, vs) if gi is not None)
    Jv = torch.autograd.grad(s, u, allow_unused=True)[0] if torch.is_tensor(s) and s.requires_grad else None
    Jv = np.zeros(tuple(rp.shape)) if Jv is None else Jv.numpy()
    return rp.detach().numpy(), Jv, ok


def _point_jvp(ren, p, pts, dp=None, dx=None):
    """(r, dr) of a point renderer under torch.func.jvp; dp: params tangent dict (numpy) or None, dx: points tangent."""
    keys = PARAM_KEYS
    pc, x = _cuda(p), torch.tensor(np.asarray(pts, np.float32), device="cuda")
    if dp is None:
        return torch.func.jvp(lambda xx: ren(pc, xx), (x,), (torch.tensor(dx, device="cuda"),))
    primals = tuple(pc[k] for k in keys)
    tangents = tuple(torch.tensor(dp[k], device="cuda") for k in keys)
    if dx is None:
        return torch.func.jvp(lambda *v: ren(dict(zip(keys, v)), x), primals, tangents)
    return torch.func.jvp(lambda xx, *v: ren(dict(zip(keys, v)), xx), (x,) + primals,
                          (torch.tensor(dx, device="cuda"),) + tangents)


def _grid_jvp(ren, p, dp):
    keys = PARAM_KEYS
    pc = _cuda(p)
    return torch.func.jvp(lambda *v: ren(dict(zip(keys, v))), tuple(pc[k] for k in keys),
                          tuple(torch.tensor(dp[k], device="cuda") for k in keys))


def _check(got_r, got_dr, ref_r, ref_dr, ok, C):
    got_r, got_dr = got_r.cpu().numpy().reshape(-1, C), got_dr.cpu().numpy().reshape(-1, C)
    ref_dr = ref_dr.reshape(-1, C)
    assert ok.mean() >= 0.97, ok.mean()
    assert np.abs(got_r[ok] - ref_r[ok]).max() <= 1e-5
    scale = max(np.abs(ref_dr[ok]).max(), 1e-30)
    err = np.abs(got_dr[ok] - ref_dr[ok]).max() / scale
    assert err <= 1e-4, err
    return got_dr


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
@pytest.mark.parametrize("group", list(GROUPS))
@pytest.mark.parametrize("name", list(CASES))
def test_param_jvp_matches_the_float64_graph(name, group):
    """Each chain-rule branch alone (pis, musX, A, experts) and all six tensors together."""
    from smoe_b200 import SmoePointRenderer
    model, pts_of, kw = CASES[name]
    p, d, C = _params(model, kw)
    pts = pts_of(np.random.RandomState(21)).astype(np.float32)
    dp = _tangent(p, group)
    r, dr = _point_jvp(SmoePointRenderer(d=d, channels=C, **kw), p, pts, dp=dp)
    assert dr.shape == r.shape == pts.shape[:-1] + (C,)
    got = _check(r, dr, *_oracle_jvp(p, pts, kw, C, dparams=dp), C)
    assert np.abs(got).max() > 0


@pytest.mark.gpu
def test_param_jvp_with_a_negative_diagonal_under_use_determinant():
    """One kernel with A_ii < 0: the op weighs it by |pi prod A_ii| (the log domain), and d c0 = (dpi / pi +
    sum dA_ll / A_ll) / ln2 holds for that too.  Flipping the sign of column i of A (and of its tangent) leaves A A^T
    and the op unchanged and makes the weight positive: the reference is the graph of the flipped model."""
    from smoe_b200 import SmoePointRenderer
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p, d, C = _params("rgb", kw)
    dp = _tangent(p, "all", seed=5)
    flip = {k: v.copy() for k, v in p.items()}, {k: v.copy() for k, v in dp.items()}
    p["A_diagonal"][7, 1, 1] *= -1.0
    dp["A_diagonal"][7, 1, 1] *= -1.0
    pts = np.random.RandomState(4).uniform(0, 1, (3000, 2)).astype(np.float32)
    r, dr = _point_jvp(SmoePointRenderer(d=d, channels=C, **kw), p, pts, dp=dp)
    _check(r, dr, *_oracle_jvp(flip[0], pts, kw, C, dparams=flip[1]), C)


@pytest.mark.gpu
def test_param_jvp_at_times_between_frames():
    from smoe_b200 import SmoePointRenderer
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p, d, C = _params("video", kw)
    g = np.meshgrid(np.linspace(0, 1, 12), np.linspace(0, 1, 16), np.linspace(0, 1, 2 * 6 - 1), indexing="ij")
    pts = np.stack(g, -1).astype(np.float32)
    dp = _tangent(p, "all")
    r, dr = _point_jvp(SmoePointRenderer(d=d, channels=C, **kw), p, pts, dp=dp)
    _check(r, dr, *_oracle_jvp(p, pts, kw, C, dparams=dp), C)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 511, 513, 1024, 1536])
def test_param_jvp_edge_sizes(n):
    from smoe_b200 import SmoePointRenderer
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p, d, C = _params("rgb", kw)
    pts = np.random.RandomState(n).uniform(0, 1, (max(n, 64), 2)).astype(np.float32)
    dp = _tangent(p, "all")
    if n == 1:                             # one point whose gates are clear of the threshold
        pts = pts[np.argmax(_oracle_jvp(p, pts, kw, C)[2])][None]
    pts = pts[:n]
    r, dr = _point_jvp(SmoePointRenderer(d=d, channels=C, **kw), p, pts, dp=dp)
    _check(r, dr, *_oracle_jvp(p, pts, kw, C, dparams=dp), C)


GRID_CASES = {
    # name: (model, grid axes as a function of the image shape, flags)
    "rgb_training_grid": ("rgb", lambda sh: [(0, 1, sh[0]), (0, 1, sh[1])], dict(use_determinant=False,
                                                                              train_inverse_cov=False)),
    "rgb_super_resolution_2x": ("rgb", lambda sh: [(0, 1, 2 * sh[0]), (0, 1, 2 * sh[1])],
                                dict(use_determinant=True, train_inverse_cov=False)),
    "gray_crop": ("gray", lambda sh: [(0.2, 0.55, 47), (0.3, 0.8, 61)], dict(use_determinant=False,
                                                                              train_inverse_cov=True)),
    "video_2t_minus_1": ("video", lambda sh: [(0, 1, sh[0]), (0, 1, sh[1]), (0, 1, 2 * sh[2] - 1)],
                         dict(use_determinant=True, train_inverse_cov=True)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(GRID_CASES))
def test_grid_jvp_matches_the_float64_graph_and_the_point_kernel(name):
    from smoe_b200 import SmoePointRenderer, SmoeRenderer
    model, grid_of, kw = GRID_CASES[name]
    p, d, C = _params(model, kw)
    grid = grid_of(MODELS[model][0])
    dp = _tangent(p, "all")
    r, dr = _grid_jvp(SmoeRenderer(grid=grid, channels=C, **kw), p, dp)
    pts = _grid_points(grid, C)
    assert r.shape == dr.shape == pts.shape[:-1] + (C,)
    r_ref, dr_ref, ok = _oracle_jvp(p, pts, kw, C, dparams=dp)
    got = _check(r, dr, r_ref, dr_ref, ok, C)
    # the point kernel at the same float32 coordinates (its own tiles, so other roundings of x')
    _, dr_p = _point_jvp(SmoePointRenderer(d=d, channels=C, **kw), p, pts, dp=dp)
    dr_p = dr_p.cpu().numpy().reshape(-1, C)
    assert np.abs(got[ok] - dr_p[ok]).max() <= 1e-5 * np.abs(dr_p[ok]).max()


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["gray", "rgb", "video"])
def test_point_tangents_match_the_jacobian_and_the_graph(model):
    """dr for a tangent on the points alone is einsum(J, xdot) with jacobian()'s J; with parameter tangents too it is
    the sum of both."""
    from smoe_b200 import SmoePointRenderer
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p, d, C = _params(model, kw)
    rs = np.random.RandomState(6)
    pts = rs.uniform(-0.05, 1.05, (2600, d)).astype(np.float32)
    dx = rs.standard_normal(pts.shape).astype(np.float32)
    ren = SmoePointRenderer(d=d, channels=C, **kw)
    r, dr = _point_jvp(ren, p, pts, dx=dx)
    r_ref, dr_ref, ok = _oracle_jvp(p, pts, kw, C, dpts=dx)
    got = _check(r, dr, r_ref, dr_ref, ok, C)
    _, J = ren.jacobian(_cuda(p), torch.tensor(pts, device="cuda"))
    ej = torch.einsum("ncl,nl->nc", J.double(), torch.tensor(dx, device="cuda").double()).cpu().numpy()
    assert np.abs(got - ej).max() <= 1e-5 * np.abs(ej).max()
    dp = _tangent(p, "all")
    r2, dr2 = _point_jvp(ren, p, pts, dp=dp, dx=dx)
    assert torch.equal(r2, r)
    _check(r2, dr2, *_oracle_jvp(p, pts, kw, C, dparams=dp, dpts=dx), C)


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["points", "grid"])
def test_adjoint_identity_with_the_reverse_path(where):
    """<u, J v> = <J^T u, v> with J v from the JVP and J^T u from the existing backward, on rgb_big: 7000 points (with
    point tangents) and a 1080 x 1920 grid."""
    from smoe_b200 import SmoePointRenderer, SmoeRenderer
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p0, d, C = _params("rgb_big", kw)
    dp = _tangent(p0, "all", seed=2)
    rs = np.random.RandomState(9)
    p = _cuda(p0, grad=True)
    v = {k: torch.tensor(dp[k], device="cuda") for k in PARAM_KEYS}
    if where == "points":
        ren = SmoePointRenderer(d=2, channels=C, **kw)
        pts = torch.tensor(rs.uniform(-0.1, 1.1, (7000, 2)).astype(np.float32), device="cuda", requires_grad=True)
        dx = torch.tensor(rs.standard_normal((7000, 2)).astype(np.float32), device="cuda")
        with fwAD.dual_level():
            out = ren({k: fwAD.make_dual(p[k], v[k]) for k in PARAM_KEYS}, fwAD.make_dual(pts, dx))
            prim, jv = fwAD.unpack_dual(out)
    else:
        ren = SmoeRenderer(grid=[(0, 1, 1080), (0, 1, 1920)], channels=C, **kw)
        with fwAD.dual_level():
            out = ren({k: fwAD.make_dual(p[k], v[k]) for k in PARAM_KEYS})
            prim, jv = fwAD.unpack_dual(out)
    u = torch.tensor(rs.standard_normal(tuple(prim.shape)).astype(np.float32), device="cuda")
    prim.backward(u)
    lhs = float((u.double() * jv.double()).sum())
    rhs = sum(float((p[k].grad.double() * v[k].double()).sum()) for k in PARAM_KEYS)
    if where == "points":
        rhs += float((pts.grad.double() * dx.double()).sum())
    assert abs(lhs - rhs) <= 1e-4 * max(abs(lhs), abs(rhs)), (lhs, rhs)


@pytest.mark.gpu
def test_degenerate_tangents():
    """A zero tangent gives dr == 0; tangents on a pi <= 0 kernel and on entries the op never reads (the
    off-diagonal of A_diagonal, the diagonal and upper part of A_corr) change no bit."""
    from smoe_b200 import SmoePointRenderer, SmoeRenderer
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p, d, C = _params("rgb", kw)
    pts = np.random.RandomState(3).uniform(0, 1, (2000, 2)).astype(np.float32)
    ren = SmoePointRenderer(d=2, channels=C, **kw)
    grid = SmoeRenderer(grid=[(0, 1, 48), (0, 1, 64)], channels=C, **kw)
    zero = {k: np.zeros_like(v) for k, v in p.items()}
    assert not _point_jvp(ren, p, pts, dp=zero)[1].any() and not _grid_jvp(grid, p, zero)[1].any()
    assert not _point_jvp(ren, p, pts, dx=np.zeros_like(pts))[1].any()
    dp = _tangent(p, "all")
    noisy = {k: v.copy() for k, v in dp.items()}
    for k in PARAM_KEYS:
        noisy[k][3] += 1.0                                              # kernel 3 has pi <= 0
    noisy["A_diagonal"] += np.where(np.eye(d, dtype=bool), 0, 0.7).astype(np.float32)
    noisy["A_corr"] += np.where(np.tril(np.ones((d, d), bool), -1), 0, -0.4).astype(np.float32)
    assert torch.equal(_point_jvp(ren, p, pts, dp=dp)[1], _point_jvp(ren, p, pts, dp=noisy)[1])
    assert torch.equal(_grid_jvp(grid, p, dp)[1], _grid_jvp(grid, p, noisy)[1])


@pytest.mark.gpu
@pytest.mark.parametrize("cloud", ["clustered", "beyond_unit_square", "crop"])
def test_jvp_modes_and_determinism(cloud):
    """dense_exec 0 (culling + skipping), 1 (every pair), 2 (skipping only), and the same call twice: the same bits."""
    from smoe_b200 import SmoePointRenderer, SmoeRenderer
    kw = dict(use_determinant=False, train_inverse_cov=True)
    p, d, C = _params("rgb_big", kw)
    dp = _tangent(p, "all")
    rs = np.random.RandomState(8)
    if cloud == "crop":
        res = [_grid_jvp(SmoeRenderer(grid=[(0.3, 0.6, 200), (0.25, 0.7, 330)], channels=C, _dense_exec=m, **kw),
                         p, dp) for m in (0, 1, 2, 0)]
    else:
        pts = (rs.uniform(0.40, 0.46, (5000, 2)) if cloud == "clustered" else rs.uniform(-0.3, 1.3, (6000, 2)))
        pts = pts.astype(np.float32)
        dx = rs.standard_normal(pts.shape).astype(np.float32)
        res = [_point_jvp(SmoePointRenderer(d=2, channels=C, _dense_exec=m, **kw), p, pts, dp=dp, dx=dx)
               for m in (0, 1, 2, 0)]
    for b in (1, 2, 3):
        assert torch.equal(res[0][0], res[b][0]) and torch.equal(res[0][1], res[b][1]), b
    assert res[0][1].abs().max() > 0


@pytest.mark.gpu
def test_gauss_newton_refit_of_the_experts_by_cg():
    """r is linear in (nu, gamma) for fixed gates, so L = 1/2 |r - y|^2 is quadratic in them: CG on H v = J^T (J v),
    J v from the JVP and J^T u from the backward, lowers |dL/d(nu, gamma)| by 10^3, and the change of L equals the
    quadratic model g^T delta + 1/2 |J delta|^2."""
    from smoe_b200 import SmoeRenderer
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p0, d, C = _params("rgb", kw)
    shape = MODELS["rgb"][0]
    import bench
    y = torch.tensor(bench.synth_image(shape, 3), device="cuda")
    ren = SmoeRenderer(grid=[(0, 1, shape[0]), (0, 1, shape[1])], channels=C, **kw)
    p = _cuda(p0)
    ex = ("nu_e", "gamma_e")

    def loss_grad(pp):
        q = {k: (t.detach().requires_grad_(k in ex)) for k, t in pp.items()}
        r = ren(q)
        res = (r - y).detach()
        r.backward(res)
        return 0.5 * float((res.double() ** 2).sum()), [q[k].grad.detach() for k in ex], res

    def jvp(v):
        return torch.func.jvp(lambda nu, ga: ren(dict(p, nu_e=nu, gamma_e=ga)), (p["nu_e"], p["gamma_e"]), tuple(v))[1]

    def jtu(u):
        q = {k: (t.detach().requires_grad_(k in ex)) for k, t in p.items()}
        ren(q).backward(u)
        return [q[k].grad.detach() for k in ex]

    def dot(a, b):
        return sum(float((x.double() * z.double()).sum()) for x, z in zip(a, b))

    L0, g0, _ = loss_grad(p)
    x = [torch.zeros_like(t) for t in g0]
    rr = [-t for t in g0]
    s = [t.clone() for t in rr]
    rho = dot(rr, rr)
    for _ in range(300):
        Hs = jtu(jvp(s))
        alpha = rho / dot(s, Hs)
        x = [a + alpha * b for a, b in zip(x, s)]
        rr = [a - alpha * b for a, b in zip(rr, Hs)]
        rho_new = dot(rr, rr)
        if rho_new ** 0.5 < 1e-5 * dot(g0, g0) ** 0.5:
            break
        s = [a + (rho_new / rho) * b for a, b in zip(rr, s)]
        rho = rho_new
    p1 = dict(p, nu_e=p["nu_e"] + x[0], gamma_e=p["gamma_e"] + x[1])
    L1, g1, _ = loss_grad(p1)
    assert dot(g1, g1) ** 0.5 <= 1e-3 * dot(g0, g0) ** 0.5, (dot(g1, g1) ** 0.5, dot(g0, g0) ** 0.5)
    Jd = jvp(x)
    model = dot(g0, x) + 0.5 * float((Jd.double() ** 2).sum())
    assert abs((L1 - L0) - model) <= 1e-3 * abs(model), (L1 - L0, model)


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["points", "grid"])
def test_forward_mode_inside_autograd(where):
    """Dual inputs that also require grad: r is the plain call's, dr is the JVP of a call without gradients, the
    gradients are those of a call without tangents, bit for bit; nothing synchronises with the host and only the
    forward's launches, smoe_pack_tangent and the JVP sweep run."""
    from torch.profiler import ProfilerActivity, profile
    from smoe_b200 import SmoePointRenderer, SmoeRenderer
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p0, d, C = _params("rgb_big", kw)
    dp = _tangent(p0, "all")
    v = {k: torch.tensor(dp[k], device="cuda") for k in PARAM_KEYS}
    rs = np.random.RandomState(1)
    if where == "points":
        ren = SmoePointRenderer(d=2, channels=C, **kw)
        x_np = rs.uniform(0, 1, (200000, 2)).astype(np.float32)
        dx = torch.tensor(rs.standard_normal(x_np.shape).astype(np.float32), device="cuda")
        sweep = "point_jvp_kernel"
    else:
        ren = SmoeRenderer(grid=[(0, 1, 480), (0, 1, 800)], channels=C, **kw)
        sweep = "grid_jvp_kernel"

    def inputs(grad):
        return _cuda(p0, grad=grad), (torch.tensor(x_np, device="cuda", requires_grad=grad) if where == "points"
                                      else None)

    def call(tangents, grad, pre=None):
        p, x = pre or inputs(grad)
        with fwAD.dual_level():
            pd = {k: fwAD.make_dual(p[k], v[k]) for k in PARAM_KEYS} if tangents else p
            args = (pd,) if x is None else (pd, fwAD.make_dual(x, dx) if tangents else x)
            out = ren(*args)
            prim, dr = fwAD.unpack_dual(out)
        return p, x, prim, dr

    _, _, r_plain, _ = call(False, False)
    _, _, r_nograd, dr_nograd = call(True, False)
    p, x, r, dr = call(True, True)
    assert torch.equal(r, r_plain) and torch.equal(r_nograd, r_plain) and torch.equal(dr, dr_nograd)
    g = torch.tensor(rs.standard_normal(tuple(r.shape)).astype(np.float32), device="cuda")
    r.backward(g)
    q, xq, r_ref, _ = call(False, True)
    r_ref.backward(g)
    for k in PARAM_KEYS:
        assert torch.equal(p[k].grad, q[k].grad), k
    if x is not None:
        assert torch.equal(x.grad, xq.grad)
    pre = inputs(False)
    call(True, False, pre)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        call(True, False, pre)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call(True, False, pre)
        torch.cuda.synchronize()
    names = [e.key for e in prof.key_averages() if "smoe::" in e.key]
    assert any(sweep in n for n in names) and any("pack_tangent_kernel" in n for n in names), names
    assert not any(k in n for n in names for k in ("backward", "cotangent", "xgrad", "loss", "jacobian")), names


@pytest.mark.gpu
def test_vmap_and_jacfwd_raise():
    from smoe_b200 import SmoePointRenderer
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p, d, C = _params("gray", kw)
    pc = _cuda(p)
    ren = SmoePointRenderer(d=2, channels=C, **kw)
    x = torch.rand(8, 2, device="cuda")
    with pytest.raises(RuntimeError, match="vmap"):
        torch.func.jacfwd(lambda xx: ren(pc, xx))(x)
    with pytest.raises(RuntimeError, match="vmap"):
        torch.func.vmap(lambda xx: ren(pc, xx))(x[None].expand(3, 8, 2))


def test_tangent_rows_validation():
    """The parameter tangents' theta rows: the layout of pack_model's rows, zeros for a missing tangent, ValueError
    for a shape or a device that is not the parameter's (no device needed)."""
    from smoe_b200.render import tangent_rows, theta_rows
    K, d, C = 5, 2, 3
    rs = np.random.RandomState(0)
    ts = [torch.tensor(rs.standard_normal(s).astype(np.float32)) for s in
          [(K,), (K, d), (K, d, d), (K, d, d), (K, d, C), (K, C)]]
    cpu = torch.device("cpu")
    assert torch.equal(tangent_rows(ts, K, d, C, cpu), theta_rows(ts, d))
    rows = tangent_rows([ts[0]] + [None] * 5, K, d, C, cpu)
    assert rows.shape == (K, 2 + 3 + 1 + C + d * C)
    assert torch.equal(rows[:, 5], ts[0]) and not rows[:, :5].any() and not rows[:, 6:].any()
    for i, bad in [(1, torch.zeros(K, 3)), (4, torch.zeros(K, d, 1)), (0, torch.zeros(K + 1)),
                   (5, torch.zeros(K, C, device="meta"))]:
        dts = [None] * 6
        dts[i] = bad
        with pytest.raises(ValueError):
            tangent_rows(dts, K, d, C, cpu)


def _lib():
    from smoe_b200 import _ffi
    if not os.path.exists(_ffi.LIB_PATH):
        pytest.skip("libsmoe_b200.so is not built")
    return _ffi


def test_jvp_calls_validate_their_arguments_before_any_cuda_work():
    """Every check of the three calls runs on the host: null pointers, d / C, eps_bits, fake quantisation, halo,
    extents, no tangent at all (no device needed: the calls return before touching one)."""
    _ffi = _lib()
    from smoe_b200.render import make_cfg, plan_grid
    L = _ffi.lib()
    fake = ctypes.c_void_p(256)                # never dereferenced: validation fails first
    null = ctypes.c_void_p(0)
    cfg = make_cfg(2, 3, 8, True, False, 0)
    _, _, batch = plan_grid([(0, 1, 32), (0, 1, 40)], 3)

    def pack(c=cfg, **kw):
        a = dict(theta=fake, dtheta=fake, indices=fake, counts=fake, K=10, tangent=fake)
        a.update(kw)
        return L.smoe_pack_tangent(ctypes.byref(c), a["theta"], a["dtheta"], a["indices"], a["counts"], a["K"],
                                   a["tangent"], null)

    def point(c=cfg, **kw):
        a = dict(packed=fake, tangent=fake, counts=fake, cb=fake, K=10, n=100, state=fake, box=fake, r=fake,
                 dx=fake, dr=fake)
        a.update(kw)
        return L.smoe_point_jvp(ctypes.byref(c), a["packed"], a["tangent"], a["counts"], a["cb"], a["K"], a["n"],
                                a["state"], a["box"], a["r"], a["dx"], a["dr"], null)

    def grid(c=cfg, b=batch, **kw):
        a = dict(packed=fake, tangent=fake, counts=fake, cb=fake, K=10, pix=fake, tq=fake, ax0=fake, ax1=fake,
                 ax2=null, rbuf=fake, dr=fake)
        a.update(kw)
        return L.smoe_jvp(ctypes.byref(c), ctypes.byref(b), a["packed"], a["tangent"], a["counts"], a["cb"], a["K"],
                          a["pix"], a["tq"], a["ax0"], a["ax1"], a["ax2"], a["rbuf"], a["dr"], null)

    def variant(**fields):
        c = make_cfg(2, 3, 8, True, False, 0)
        for k, val in fields.items():
            setattr(c, k, val)
        return c

    for call in (pack, point, grid):
        for key in {pack: ("theta", "dtheta", "indices", "counts", "tangent"),
                    point: ("packed", "counts", "cb", "state", "box", "r", "dr"),
                    grid: ("packed", "tangent", "counts", "cb", "pix", "tq", "ax0", "ax1", "rbuf", "dr")}[call]:
            assert call(**{key: null}) != 0, (call.__name__, key)
            assert b"null argument" in L.smoe_last_error()
        assert call(K=0) != 0
        assert call(c=variant(d=4)) != 0 and call(c=variant(C=2)) != 0
        assert call(c=variant(eps_bits=32)) != 0
    assert pack(c=variant(quantization_mode=2)) != 0 and pack(c=variant(quantize_pis=1)) != 0
    assert pack(c=variant(use_diff_center=1)) != 0
    assert point(tangent=null, dx=null) != 0 and b"at least one" in L.smoe_last_error()
    assert point(n=0) != 0
    assert grid(c=variant(d=3)) != 0                       # ax2 missing
    for field, val in (("halo", 2),):
        b = _ffi.Batch.from_buffer_copy(batch)
        setattr(b, field, val)
        assert grid(b=b) != 0
    b = _ffi.Batch.from_buffer_copy(batch)
    b.extent[0] = b.dims[0] + 1
    assert grid(b=b) != 0 and b"outside the image" in L.smoe_last_error()


def test_jvp_kernels_are_spill_free_within_their_launch_bounds():
    """csrc/jvp.cu alone for sm_100a with -Xptxas -v: every point (parameter, point or both tangents) and grid
    instantiation spills nothing and uses no more registers than its __launch_bounds__ (128 threads; with parameter
    tangents 4 CTAs per SM at (2, 1), 3 at (2, 3) and (3, 1), 2 at (3, 3); with point tangents alone 4)."""
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip("nvcc not found")
    csrc = os.path.join(ROOT, "steered-mixture-of-experts_b200", "csrc")
    with tempfile.TemporaryDirectory() as tmp:
        cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-c",
               "-o", os.path.join(tmp, "jvp.o"), os.path.join(csrc, "jvp.cu")]
        r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    ctas = {(2, 1): 4, (2, 3): 3, (3, 1): 3, (3, 3): 2}
    seen = set()
    for block in r.stderr.split("Compiling entry function '")[1:]:
        name = block.split("'", 1)[0]
        m = re.search(r"(point|grid)_jvp_kernelILi(\d)ELi(\d)E(?:Lb(\d)ELb(\d)E)?", name)
        if m is None:
            continue
        d, C = int(m.group(2)), int(m.group(3))
        pt, xt = (m.group(4) or "1") == "1", (m.group(5) or "0") == "1"
        regs = int(re.search(r"Used (\d+) registers", block).group(1))
        spill = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", block)
        limit = min(255, 65536 // (128 * (ctas[(d, C)] if pt else 4)) // 8 * 8)
        seen.add((m.group(1), d, C, pt, xt))
        assert regs <= limit and spill.groups() == ("0", "0", "0"), (name, regs, limit, spill.groups())
    expect = {("grid", d, C, True, False) for d in (2, 3) for C in (1, 3)}
    expect |= {("point", d, C, pt, xt) for d in (2, 3) for C in (1, 3) for pt, xt in ((1, 0), (0, 1), (1, 1))}
    assert seen == {(k, d, C, bool(pt), bool(xt)) for k, d, C, pt, xt in expect}, seen


def test_the_jvp_calls_are_declared_and_exported():
    from smoe_b200 import _ffi
    hdr = open(os.path.join(ROOT, "include", "smoe_b200.h")).read()
    for sym in ("smoe_tangent_stride", "smoe_pack_tangent", "smoe_jvp", "smoe_point_jvp"):
        assert re.search(r"\bint " + sym + r"\(", hdr) and sym in _ffi.EXPORTS
        if os.path.exists(_ffi.LIB_PATH):
            assert hasattr(ctypes.CDLL(_ffi.LIB_PATH), sym)
    if os.path.exists(_ffi.LIB_PATH):
        assert [_ffi.lib().smoe_tangent_stride(d, C) for d in (2, 3) for C in (1, 3)] == [12, 16, 16, 24]
