"""Gauss-Newton diagonal of SmoeRenderer and SmoePointRenderer (steered-mixture-of-experts_b200/render.py,
csrc/gn_diag.cu): D = diag(J^T diag(h) J) in every parameter, from one kernel-stationary CUDA sweep after the forward.

The reference is sum_n sum_c h_c (d r_pre,c / d theta_i)^2 with the float64 restatement of the reference graph's
Jacobian, taken column by column with batched one-hot tangents and the double-backward identity J v = d/du <J^T u, v>;
h is 0 on the samples whose gates are within float32 noise of the threshold.  D is also checked against the library's
own JVP at full size, between the grid and point sweeps, in the weight, across the execution modes, inside the
profiler and as the Jacobi preconditioner of a Gauss-Newton CG refit.  The last tests need no device."""
import ctypes
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from conftest import ROOT
from test_jacobian_gpu import MODELS, _cuda, _grid_points, _nvcc, _params
from test_jvp_gpu import CASES, GRID_CASES

PARAM_KEYS = ("pis", "musX", "A_diagonal", "A_corr", "gamma_e", "nu_e")


def _oracle_diag(params, pts, kw, C, h_of_ok, batch=96):
    """float64 graph r_pre (N, C), the reference diagonal (dict) for the weight h_of_ok(ok) (N, C), and ok."""
    from oracle.graph import GraphCfg, ambiguity_margins, graph_forward
    d = params["musX"].shape[1]
    pts = np.asarray(pts, np.float32).reshape(-1, d)
    K = params["pis"].shape[0]
    dom = torch.tensor(pts.astype(np.float64))
    cfg = GraphCfg(dim_domain=d, num_channels=C, use_yuv=False, start_pis=K, **kw)
    leaf = {k: torch.tensor(np.asarray(params[k], np.float64), requires_grad=True) for k in PARAM_KEYS}
    out = graph_forward(leaf, np.ones(K, bool), dom, torch.zeros(dom.shape[0], C, dtype=torch.float64), cfg)
    ok = ambiguity_margins(out, cfg)[0] > 1e-3
    h = np.asarray(h_of_ok(ok), np.float64)
    rp = out["r_pre"]
    u = torch.zeros_like(rp, requires_grad=True)
    g = torch.autograd.grad(rp, [leaf[k] for k in PARAM_KEYS], grad_outputs=u, create_graph=True, allow_unused=True)
    flat = torch.cat([(gi if gi is not None else torch.zeros_like(leaf[k])).reshape(-1)
                      for k, gi in zip(PARAM_KEYS, g)])
    n = flat.numel()
    hw = torch.tensor(np.broadcast_to(h, tuple(rp.shape)).copy())
    diag = np.zeros(n)
    for s in range(0, n, batch):
        b = min(batch, n - s)
        V = torch.zeros((b, n), dtype=torch.float64)
        V[torch.arange(b), s + torch.arange(b)] = 1.0
        Jc = torch.autograd.grad(flat, u, grad_outputs=V, retain_graph=True, is_grads_batched=True)[0]
        diag[s:s + b] = (hw * Jc ** 2).sum((1, 2)).numpy()
    ref, o = {}, 0
    for k in PARAM_KEYS:
        m = leaf[k].numel()
        ref[k] = diag[o:o + m].reshape(tuple(leaf[k].shape))
        o += m
    return rp.detach().numpy(), ref, ok


def _random_weight(C, seed):
    rs = np.random.RandomState(seed)
    return lambda ok: (rs.uniform(0.5, 2.0, (ok.shape[0], C)) * ok[:, None]).astype(np.float32)


def _check_diag(D, ref, p):
    """Per tensor: max |D - D_ref| <= 1e-4 max |D_ref|, <= 1e-3 relative on entries >= 1e-3 max; entries the op does
    not read and the rows of kernels with pi <= 0 exactly 0."""
    d = p["musX"].shape[1]
    for k in PARAM_KEYS:
        got = D[k].cpu().numpy().astype(np.float64)
        want = ref[k]
        assert got.shape == want.shape and D[k].dtype == torch.float32, k
        scale = np.abs(want).max()
        assert scale > 0, k
        assert np.abs(got - want).max() <= 1e-4 * scale, (k, np.abs(got - want).max() / scale)
        big = np.abs(want) >= 1e-3 * scale
        rel = np.abs(got[big] - want[big]) / np.abs(want[big])
        assert rel.max() <= 1e-3, (k, rel.max())
        assert not got[p["pis"] <= 0].any(), k
    assert not D["A_diagonal"][:, ~torch.eye(d, dtype=torch.bool)].any()
    assert not D["A_corr"][:, ~torch.ones(d, d).tril(-1).bool()].any()


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_point_diagonal_matches_the_float64_graph(name):
    """Gray, RGB and video models, both values of each flag, random points, a rotated and scaled grid, times between
    frames; a random positive weight per sample and channel."""
    from smoe_b200 import SmoePointRenderer
    model, pts_of, kw = CASES[name]
    p, d, C = _params(model, kw)
    pts = pts_of(np.random.RandomState(21)).astype(np.float32)
    r_ref, ref, ok = _oracle_diag(p, pts, kw, C, _random_weight(C, 4))
    h = _random_weight(C, 4)(ok).reshape(pts.shape[:-1] + (C,))
    r, D = SmoePointRenderer(d=d, channels=C, **kw).gauss_newton_diagonal(
        _cuda(p), torch.tensor(pts, device="cuda"), weight=torch.tensor(h, device="cuda"))
    assert not r.requires_grad and not any(t.requires_grad for t in D.values())
    assert np.abs(r.cpu().numpy().reshape(-1, C)[ok] - r_ref[ok]).max() <= 1e-5
    _check_diag(D, ref, p)


@pytest.mark.gpu
def test_point_diagonal_with_a_negative_diagonal_under_use_determinant():
    """A kernel with A_ii < 0 is weighted by |pi prod A_ii|; flipping column i of A leaves the op unchanged and flips
    the sign of the derivatives in that column, so D equals the graph's diagonal of the flipped model."""
    from smoe_b200 import SmoePointRenderer
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p, d, C = _params("rgb", kw)
    flip = {k: v.copy() for k, v in p.items()}
    p["A_diagonal"][7, 1, 1] *= -1.0
    pts = np.random.RandomState(4).uniform(0, 1, (3000, 2)).astype(np.float32)
    _, ref, ok = _oracle_diag(flip, pts, kw, C, _random_weight(C, 2))
    h = _random_weight(C, 2)(ok)
    _, D = SmoePointRenderer(d=d, channels=C, **kw).gauss_newton_diagonal(
        _cuda(p), torch.tensor(pts, device="cuda"), weight=torch.tensor(h, device="cuda"))
    _check_diag(D, ref, p)
    assert D["A_diagonal"][7, 1, 1] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(GRID_CASES))
def test_grid_diagonal_matches_the_graph_and_the_point_sweep(name):
    """The grid sweep against the graph, and against the point sweep on the same float32 coordinates (its own tiles:
    other roundings of x') within 1e-5 of each tensor's max; the grid's r is bitwise the render's."""
    from smoe_b200 import SmoePointRenderer, SmoeRenderer
    model, grid_of, kw = GRID_CASES[name]
    p, d, C = _params(model, kw)
    grid = grid_of(MODELS[model][0])
    pts = _grid_points(grid, C)
    _, ref, ok = _oracle_diag(p, pts, kw, C, _random_weight(C, 9))
    h = torch.tensor(_random_weight(C, 9)(ok).reshape(pts.shape[:-1] + (C,)), device="cuda")
    ren = SmoeRenderer(grid=grid, channels=C, **kw)
    r, D = ren.gauss_newton_diagonal(_cuda(p), weight=h)
    assert torch.equal(r, ren(_cuda(p)))
    _check_diag(D, ref, p)
    _, Dp = SmoePointRenderer(d=d, channels=C, **kw).gauss_newton_diagonal(
        _cuda(p), torch.tensor(pts, device="cuda"), weight=h)
    for k in PARAM_KEYS:
        assert (D[k] - Dp[k]).abs().max() <= 1e-5 * Dp[k].abs().max(), k


@pytest.mark.gpu
def test_diagonal_matches_the_jvp_at_full_size():
    """bench.py's c3 model on its 1920x1080 grid, h = 1: 48 sampled entries over the six tensors, in dense and sparse
    regions, against sum |J e_i|^2 from torch.func.jvp with a one-hot tangent.  An entry may differ only through a
    gate decision within float32 noise of tau; those are counted and must be rare."""
    import bench
    from smoe_b200 import Smoe, SmoeRenderer
    shape, kgrid, seed, _ = bench.WORKLOADS["c3"]
    kw = {k: bench.SMOE_KW[k] for k in ("use_determinant", "train_inverse_cov")}
    m = Smoe(bench.synth_image(shape, seed), kernels_per_dim=kgrid, **bench.SMOE_KW)
    p = {k: torch.tensor(v, device="cuda") for k, v in m.get_params().items()}
    del m
    ren = SmoeRenderer(grid=[(0, 1, n) for n in shape[:2]], channels=3, **kw)
    r, D = ren.gauss_newton_diagonal(p)
    K = p["pis"].shape[0]
    rs = np.random.RandomState(0)
    # kernels with the smallest and the largest footprint-weighted diagonal: sparse and dense regions
    order = torch.argsort(D["nu_e"][:, 0]).cpu().numpy()
    picks = [int(order[i]) for i in rs.randint(K // 4, K, 4)] + [int(order[i]) for i in rs.randint(0, K // 4, 4)]
    entries = []
    for k in picks:
        entries += [("pis", (k,)), ("musX", (k, rs.randint(2))), ("A_diagonal", (k, 1, 1)), ("A_corr", (k, 1, 0)),
                    ("nu_e", (k, rs.randint(3))), ("gamma_e", (k, rs.randint(2), rs.randint(3)))]
    assert len(entries) == 48
    keys = PARAM_KEYS
    prim = tuple(p[k] for k in keys)
    off = 0
    for name, idx in entries:
        tan = tuple(torch.zeros_like(t) for t in prim)
        tan[keys.index(name)][idx] = 1.0
        out, jv = torch.func.jvp(lambda *t: ren(dict(zip(keys, t))), prim, tan)
        assert torch.equal(out, r)
        want = float((jv.double() ** 2).sum())
        got = float(D[name][idx])
        if abs(got - want) > 1e-4 * max(abs(want), 1e-30):
            off += 1
            print(f"{name}{idx}: D {got:.7g}, sum |J e_i|^2 {want:.7g}")
    print(f"{off} of 48 entries differ by more than 1e-4 relative")
    assert off <= 2, off


@pytest.mark.gpu
def test_weights():
    """h = 0 gives D = 0; D(2h) = 2 D(h); a per-channel (C,) weight, the same weight expanded to r's full shape and
    a per-sample weight broadcast over the channels all give the bits of their dense copies."""
    from smoe_b200 import SmoePointRenderer, SmoeRenderer
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p, d, C = _params("rgb", kw)
    pc = _cuda(p)
    ren = SmoeRenderer(grid=[(0, 1, 48), (0, 1, 64)], channels=C, **kw)
    shape = (48, 64, C)
    rs = np.random.RandomState(3)
    h = torch.tensor(rs.uniform(0.5, 2, shape).astype(np.float32), device="cuda")
    _, D0 = ren.gauss_newton_diagonal(pc, weight=torch.zeros(shape, device="cuda"))
    assert not any(t.any() for t in D0.values())
    _, D1 = ren.gauss_newton_diagonal(pc, weight=h)
    _, D2 = ren.gauss_newton_diagonal(pc, weight=2 * h)
    for k in PARAM_KEYS:
        assert (D2[k] - 2 * D1[k]).abs().max() <= 1e-6 * D1[k].abs().max(), k
    hc = torch.tensor([0.5, 2.0, 1.25], device="cuda")
    hn = torch.tensor(rs.uniform(0.5, 2, (48, 64, 1)).astype(np.float32), device="cuda")
    pts = torch.tensor(rs.uniform(0, 1, (1500, 2)).astype(np.float32), device="cuda")
    pren = SmoePointRenderer(d=2, channels=C, **kw)
    for w in (hc, hc.expand(shape), hn):
        a = ren.gauss_newton_diagonal(pc, weight=w)[1]
        b = ren.gauss_newton_diagonal(pc, weight=w.expand(shape).contiguous())[1]
        assert all(torch.equal(a[k], b[k]) for k in PARAM_KEYS)
    a = pren.gauss_newton_diagonal(pc, pts, weight=hc)[1]
    b = pren.gauss_newton_diagonal(pc, pts, weight=hc.expand(1500, C).contiguous())[1]
    assert all(torch.equal(a[k], b[k]) for k in PARAM_KEYS)
    ones = pren.gauss_newton_diagonal(pc, pts)[1]
    assert all(torch.equal(ones[k], pren.gauss_newton_diagonal(pc, pts, weight=torch.ones(C, device="cuda"))[1][k])
               for k in PARAM_KEYS)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["crop", "extrapolating", "clustered"])
def test_modes_and_repeat_calls_give_the_same_bits(case):
    from smoe_b200 import SmoePointRenderer, SmoeRenderer
    kw = dict(use_determinant=False, train_inverse_cov=True)
    p, d, C = _params("rgb_big", kw)
    pc = _cuda(p)
    if case == "clustered":
        pts = torch.tensor(np.random.RandomState(8).uniform(0.40, 0.46, (5000, 2)).astype(np.float32), device="cuda")
        res = [SmoePointRenderer(d=2, channels=C, _dense_exec=m, **kw).gauss_newton_diagonal(pc, pts)
               for m in (0, 1, 2, 0)]
    else:
        grid = [(0.3, 0.6, 200), (0.25, 0.7, 330)] if case == "crop" else [(-0.3, 1.3, 150), (-0.2, 1.2, 260)]
        res = [SmoeRenderer(grid=grid, channels=C, _dense_exec=m, **kw).gauss_newton_diagonal(pc) for m in (0, 1, 2, 0)]
    for b in (1, 2, 3):
        assert torch.equal(res[0][0], res[b][0]), b
        for k in PARAM_KEYS:
            assert torch.equal(res[0][1][k], res[b][1][k]), (b, k)
    assert all(res[0][1][k].abs().max() > 0 for k in PARAM_KEYS)


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["points", "grid"])
def test_no_sync_and_only_the_expected_launches(where):
    from torch.profiler import ProfilerActivity, profile
    from smoe_b200 import SmoePointRenderer, SmoeRenderer
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p, d, C = _params("rgb_big", kw)
    pc = _cuda(p, grad=True)
    if where == "points":
        ren = SmoePointRenderer(d=2, channels=C, **kw)
        x = torch.rand(200000, 2, device="cuda")
        w = torch.rand(200000, C, device="cuda")
        call = lambda: ren.gauss_newton_diagonal(pc, x, weight=w)            # noqa: E731
        expect = ("point_forward_kernel", "point_gn_state_kernel", "point_plan_kernel", "gn_diag_kernel")
    else:
        ren = SmoeRenderer(grid=[(0, 1, 480), (0, 1, 800)], channels=C, **kw)
        w = torch.rand(480, 800, C, device="cuda")
        call = lambda: ren.gauss_newton_diagonal(pc, weight=w)               # noqa: E731
        expect = ("forward_kernel", "gn_state_kernel", "bwd_plan_kernel", "gn_diag_kernel")
    call()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        call()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call()
        torch.cuda.synchronize()
    names = [e.key for e in prof.key_averages() if "smoe::" in e.key]
    for k in expect + ("pack_scatter_kernel", "reduce_splits_kernel", "gn_scatter_kernel"):
        assert any(k in n for n in names), (k, names)
    assert not any(k in n for n in names for k in ("backward_kernel", "cotangent", "xgrad", "loss", "jacobian",
                                                   "finalize", "jvp")), names


@pytest.mark.gpu
def test_jacobi_preconditioned_cg_refit_of_the_experts():
    """The expert refit of test_gauss_newton_refit_of_the_experts_by_cg (H v = J^T (J v) on (nu, gamma), plain CG),
    and the same with the Jacobi preconditioner 1 / max(D, eps) from the diagonal: both reach the 1e-5 residual
    tolerance (within 1500 iterations) and lower |dL/d(nu, gamma)| by 10^3.  Prints both iteration counts; asserts
    convergence, not a speed-up."""
    import bench
    from smoe_b200 import SmoeRenderer
    kw = dict(use_determinant=True, train_inverse_cov=False)
    p0, d, C = _params("rgb", kw)
    shape = MODELS["rgb"][0]
    y = torch.tensor(bench.synth_image(shape, 3), device="cuda")
    ren = SmoeRenderer(grid=[(0, 1, shape[0]), (0, 1, shape[1])], channels=C, **kw)
    p = _cuda(p0)
    ex = ("nu_e", "gamma_e")

    def loss_grad(pp):
        q = {k: (t.detach().requires_grad_(k in ex)) for k, t in pp.items()}
        r = ren(q)
        res = (r - y).detach()
        r.backward(res)
        return [q[k].grad.detach() for k in ex]

    def hvp(v):
        jv = torch.func.jvp(lambda nu, ga: ren(dict(p, nu_e=nu, gamma_e=ga)), (p["nu_e"], p["gamma_e"]), tuple(v))[1]
        q = {k: (t.detach().requires_grad_(k in ex)) for k, t in p.items()}
        ren(q).backward(jv)
        return [q[k].grad.detach() for k in ex]

    def dot(a, b):
        return sum(float((x.double() * z.double()).sum()) for x, z in zip(a, b))

    _, D = ren.gauss_newton_diagonal(p)
    eps = 1e-6 * max(float(D[k].max()) for k in ex)
    minv = [1.0 / D[k].clamp_min(eps) for k in ex]
    g0 = loss_grad(p)

    def cg(precond):
        x = [torch.zeros_like(t) for t in g0]
        rr = [-t for t in g0]
        z = [m * t for m, t in zip(minv, rr)] if precond else rr
        s = [t.clone() for t in z]
        rho = dot(rr, z)
        for it in range(1, 1501):
            Hs = hvp(s)
            alpha = rho / dot(s, Hs)
            x = [a + alpha * b for a, b in zip(x, s)]
            rr = [a - alpha * b for a, b in zip(rr, Hs)]
            res = dot(rr, rr) ** 0.5 / dot(g0, g0) ** 0.5
            if it % 50 == 0:
                print(f"{'Jacobi' if precond else 'plain'} CG, iteration {it}: residual {res:.3e}")
            if res < 1e-5:
                return x, it
            z = [m * t for m, t in zip(minv, rr)] if precond else rr
            rho_new = dot(rr, z)
            s = [a + (rho_new / rho) * b for a, b in zip(z, s)]
            rho = rho_new
        return x, None

    x_plain, n_plain = cg(False)
    x_jac, n_jac = cg(True)
    print(f"CG iterations to a 1e-5 residual: plain {n_plain}, Jacobi-preconditioned {n_jac}")
    assert n_plain is not None and n_jac is not None
    for x in (x_plain, x_jac):
        g1 = loss_grad(dict(p, nu_e=p["nu_e"] + x[0], gamma_e=p["gamma_e"] + x[1]))
        assert dot(g1, g1) ** 0.5 <= 1e-3 * dot(g0, g0) ** 0.5


def test_gauss_newton_diagonal_validates_its_arguments():
    """Bad params, points or weights raise ValueError before any device work (no device needed: the renderer is
    built without its constructor, which needs one)."""
    from smoe_b200.render import SmoePointRenderer, SmoeRenderer, check_weight
    cpu = torch.device("cpu")
    shape = (6, 8, 3)
    assert check_weight(None, shape, cpu) == (None, 0, 0)
    w, ss, sc = check_weight(torch.ones(3), shape, cpu)
    assert (ss, sc) == (0, 1) and w.shape == (48, 3)
    w, ss, sc = check_weight(torch.ones(6, 8, 1), shape, cpu)
    assert (ss, sc) == (1, 0)
    w, ss, sc = check_weight(torch.ones(shape), shape, cpu)
    assert (ss, sc) == (3, 1)
    w, ss, sc = check_weight(torch.ones(8, 6, 3).transpose(0, 1), shape, cpu)           # not viewable: a copy
    assert w.is_contiguous() and (ss, sc) == (3, 1)
    for bad in (np.ones(shape, np.float32), torch.ones(shape, dtype=torch.float64), torch.ones(4),
                torch.ones(6, 8, 3, 2), torch.ones(7, 8, 3), torch.ones(shape, device="meta"), 1.0):
        with pytest.raises(ValueError):
            check_weight(bad, shape, cpu)
    K, d, C = 5, 2, 3
    params = {"pis": torch.ones(K), "musX": torch.zeros(K, d), "A_diagonal": torch.ones(K, d, d),
              "A_corr": torch.zeros(K, d, d), "gamma_e": torch.zeros(K, d, C), "nu_e": torch.zeros(K, C)}
    g = SmoeRenderer.__new__(SmoeRenderer)
    g.d, g.C, g.shape, g.device = d, C, (6, 8), cpu
    pr = SmoePointRenderer.__new__(SmoePointRenderer)
    pr.d, pr.C, pr.device = d, C, cpu
    pts = torch.zeros(10, 2)
    for call in (lambda w: g.gauss_newton_diagonal(params, weight=w),
                 lambda w: pr.gauss_newton_diagonal(params, pts, weight=w)):
        with pytest.raises(ValueError):
            call(torch.ones(5, 3))
        with pytest.raises(ValueError):
            call(torch.ones(3, dtype=torch.float16))
    with pytest.raises(ValueError):
        g.gauss_newton_diagonal(dict(params, pis=torch.ones(K, 1)))
    with pytest.raises(ValueError):
        pr.gauss_newton_diagonal(params, torch.zeros(10, 3))
    with pytest.raises(ValueError):
        pr.gauss_newton_diagonal(params, pts, weight=torch.ones(11, C))


def _lib():
    from smoe_b200 import _ffi
    if not os.path.exists(_ffi.LIB_PATH):
        pytest.skip("libsmoe_b200.so is not built")
    return _ffi


def test_gn_calls_validate_their_arguments_before_any_cuda_work():
    _ffi = _lib()
    from smoe_b200.render import make_cfg, plan_grid
    L = _ffi.lib()
    fake = ctypes.c_void_p(256)
    null = ctypes.c_void_p(0)
    cfg = make_cfg(2, 3, 8, True, False, 0)
    _, _, batch = plan_grid([(0, 1, 32), (0, 1, 40)], 3)
    z = ctypes.c_longlong(0)

    def variant(**fields):
        c = make_cfg(2, 3, 8, True, False, 0)
        for k, val in fields.items():
            setattr(c, k, val)
        return c

    def state(c=cfg, b=batch, **kw):
        a = dict(pix=fake, r=fake, w=null, g=fake)
        a.update(kw)
        return L.smoe_gn_state(ctypes.byref(c), ctypes.byref(b), a["pix"], a["r"], a["w"], z, z, a["g"], null)

    def pstate(c=cfg, **kw):
        a = dict(n=100, st=fake, r=fake, w=null, order=null, g=fake)
        a.update(kw)
        return L.smoe_point_gn_state(ctypes.byref(c), a["n"], a["st"], a["r"], a["w"], a["order"], z, z, a["g"], null)

    def grid(c=cfg, b=batch, **kw):
        a = dict(packed=fake, theta=fake, idx=fake, counts=fake, K=10, g=fake, tq=fake, ax0=fake, ax1=fake, ax2=null,
                 splits=7, part=fake, plan=fake)
        a.update(kw)
        return L.smoe_gn_diag(ctypes.byref(c), ctypes.byref(b), a["packed"], a["theta"], a["idx"], a["counts"], a["K"],
                              a["g"], a["tq"], a["ax0"], a["ax1"], a["ax2"], a["splits"], a["part"], a["plan"], null)

    def point(c=cfg, **kw):
        a = dict(packed=fake, theta=fake, idx=fake, counts=fake, K=10, n=100, g=fake, box=fake, splits=7, part=fake,
                 plan=fake)
        a.update(kw)
        return L.smoe_point_gn_diag(ctypes.byref(c), a["packed"], a["theta"], a["idx"], a["counts"], a["K"], a["n"],
                                    a["g"], a["box"], a["splits"], a["part"], a["plan"], null)

    def scatter(c=cfg, **kw):
        a = dict(raw=fake, idx=fake, counts=fake, K=10, diag=fake)
        a.update(kw)
        return L.smoe_gn_diag_scatter(ctypes.byref(c), a["raw"], a["idx"], a["counts"], a["K"], a["diag"], null)

    nulls = {state: ("pix", "r", "g"), pstate: ("st", "r", "g"),
             grid: ("packed", "theta", "idx", "counts", "g", "tq", "ax0", "ax1", "part", "plan"),
             point: ("packed", "theta", "idx", "counts", "g", "box", "part", "plan"),
             scatter: ("raw", "idx", "counts", "diag")}
    for call, keys in nulls.items():
        for key in keys:
            assert call(**{key: null}) != 0, (call.__name__, key)
            assert b"null argument" in L.smoe_last_error()
        assert call(c=variant(d=4)) != 0 and call(c=variant(C=2)) != 0
    for call in (state, pstate, grid, point):
        assert call(c=variant(eps_bits=32)) != 0
        assert call(c=variant(quantization_mode=2)) != 0 and call(c=variant(use_diff_center=1)) != 0
        assert call(c=variant(radial_as=1)) != 0 and call(c=variant(train_gammas=0)) != 0
    assert pstate(w=fake) != 0 and b"order" in L.smoe_last_error()
    assert pstate(n=0) != 0 and point(n=0) != 0
    for call in (grid, point, scatter):
        assert call(K=0) != 0
    assert grid(splits=0) != 0 and point(splits=0) != 0
    assert grid(c=variant(d=3)) != 0                       # ax2 missing
    for call in (state, grid):
        b = _ffi.Batch.from_buffer_copy(batch)
        b.halo = 2
        assert call(b=b) != 0
        b = _ffi.Batch.from_buffer_copy(batch)
        b.extent[0] = b.dims[0] + 1
        assert call(b=b) != 0 and b"outside the image" in L.smoe_last_error()


def test_gn_kernels_are_spill_free_within_their_launch_bounds():
    """csrc/gn_diag.cu alone for sm_100a with -Xptxas -v: every sweep instantiation (grid and point, each (d, C),
    dense and not) spills nothing and fits backward_kernel's budget of 128 registers (64 threads, 8 CTAs per SM)."""
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip("nvcc not found")
    csrc = os.path.join(ROOT, "steered-mixture-of-experts_b200", "csrc")
    with tempfile.TemporaryDirectory() as tmp:
        cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-c",
               "-o", os.path.join(tmp, "gn_diag.o"), os.path.join(csrc, "gn_diag.cu")]
        r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    seen = set()
    for block in r.stderr.split("Compiling entry function '")[1:]:
        name = block.split("'", 1)[0]
        regs = int(re.search(r"Used (\d+) registers", block).group(1))
        spill = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", block)
        assert spill.groups() == ("0", "0", "0"), (name, spill.groups())
        m = re.search(r"gn_diag_kernelILi(\d)ELi(\d)ELb(\d)ELb(\d)E", name)
        if m is not None:
            assert regs <= 128, (name, regs)
            seen.add(tuple(int(v) for v in m.groups()))
    assert seen == {(d, C, pt, dn) for d in (2, 3) for C in (1, 3) for pt in (0, 1) for dn in (0, 1)}, seen


def test_the_gn_calls_are_declared_and_exported_and_the_abi_is_still_6():
    from smoe_b200 import _ffi
    hdr = open(os.path.join(ROOT, "include", "smoe_b200.h")).read()
    syms = ("smoe_gn_state_stride", "smoe_point_gn_state_stride", "smoe_gn_state", "smoe_point_gn_state",
            "smoe_gn_diag", "smoe_point_gn_diag", "smoe_gn_diag_scatter")
    for sym in syms:
        assert re.search(r"\bint " + sym + r"\(", hdr) and sym in _ffi.EXPORTS, sym
    assert re.search(r"#define SMOE_ABI_VERSION 6\b", hdr) and _ffi.ABI_VERSION == 6
    if os.path.exists(_ffi.LIB_PATH):
        for sym in syms:
            assert hasattr(ctypes.CDLL(_ffi.LIB_PATH), sym)
        L = _ffi.lib()
        assert L.smoe_abi_version() == 6
        assert [L.smoe_point_gn_state_stride(d, C) for d in (2, 3) for C in (1, 3)] == [512 * n for n in (5, 9, 6, 10)]
