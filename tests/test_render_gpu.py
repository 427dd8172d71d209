"""SmoeRenderer (steered-mixture-of-experts_b200/render.py): a differentiable SMoE render on any uniform grid.

On the training grid it must compute the training path's bits, forward and gradient; off it, it is compared with the
float64 restatement of the reference graph.  The last test needs no device: it checks the argument validation."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN

PARAM_KEYS = ("pis", "musX", "A_diagonal", "A_corr", "gamma_e", "nu_e")
TAU = 0.5 / 256


def _rel(a, b):
    return float(np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)).max() / max(np.abs(b).max(), 1e-30))


def _image(case):
    import bench
    if case == "gray":
        return np.load(os.path.join(GOLDEN, "init_cases.npz"))["c1_image"], [16, 16], dict(use_determinant=True,
                                                                                              train_inverse_cov=False)
    if case == "rgb":
        return bench.synth_image((96, 160, 3), 6), [24, 40], dict(use_determinant=False, train_inverse_cov=True)
    return bench.synth_image((40, 48, 16, 3), 5), [10, 12, 4], dict(use_determinant=True, train_inverse_cov=False)


def _steer(p, d, tic, seed=3):
    """Steered kernels and sloped experts, so every part of the gradient is exercised."""
    rs = np.random.RandomState(seed)
    steer = rs.normal(0, 0.2 * p["A_diagonal"].max(), p["A_corr"].shape).astype(np.float32)
    p["A_corr"] = np.where(np.tril(np.ones((d, d), bool), -1)[None], steer * (0.3 if tic else 1.0), 0).astype(np.float32)
    p["gamma_e"] = rs.normal(0, 0.3, p["gamma_e"].shape).astype(np.float32)
    return p


def _model(case):
    from smoe_b200 import Smoe, AdamOptimizer
    img, k, kw = _image(case)
    m = Smoe(img, kernels_per_dim=k, **kw)
    m.set_optimizer(AdamOptimizer(1e-3), AdamOptimizer(1e-5), AdamOptimizer(1.0))
    m.set_params(_steer(m.get_params(), img.ndim - 1, kw["train_inverse_cov"]))
    return m, img, kw


def _cuda(p, grad=False):
    return {k: torch.tensor(np.asarray(v, np.float32), device="cuda", requires_grad=grad) for k, v in p.items()}


def _grads_np(p):
    return {k: p[k].grad.cpu().numpy() for k in PARAM_KEYS}


def _loss_cotangent(m, r):
    """dL/dr of the squared-error loss stage (csrc/forward.cu loss_kernel), in float32 and in its operation order."""
    f32 = np.float32
    C = r.shape[-1]
    two_p = f32(2 ** m.precision)
    eps = f32(m.margin) / two_p
    q_scale = f32(1) / (two_p - f32(1))
    q_inv = f32(1) / q_scale
    tgt = m._d_image.reshape(r.shape)
    rc = r.clamp(0, 1)
    rq = torch.floor(rc * float(q_inv) + 0.5) * float(q_scale)
    diff = rq - tgt
    ad = diff.abs() - float(eps)
    cw = [0.75, 0.125, 0.125][:C] if m.use_yuv else [float(f32(1) / f32(C))] * C
    cw = torch.tensor(cw, dtype=torch.float32, device=r.device)
    inv_count = float(f32(1.0 / m.num_pixel))
    g = 2.0 * ad * torch.sign(diff) * cw * inv_count
    return torch.where((r >= 0) & (r <= 1), g, torch.zeros_like(g))


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["gray", "rgb", "video"])
def test_training_grid_forward_is_bitwise_the_training_path(case):
    from smoe_b200 import SmoeRenderer
    m, img, kw = _model(case)
    d, C = img.ndim - 1, img.shape[-1]
    pre = m.get_pre_clip_reconstruction()
    r = SmoeRenderer(grid=[(0, 1, n) for n in img.shape[:d]], channels=C, **kw)
    with torch.no_grad():
        out = r(_cuda(m.get_params()))
    assert out.shape == img.shape
    np.testing.assert_array_equal(out.cpu().numpy(), pre)
    out_g = r(_cuda(m.get_params(), grad=True))          # the instantiation that also writes the backward state
    np.testing.assert_array_equal(out_g.detach().cpu().numpy(), pre)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["gray", "rgb", "video"])
def test_training_grid_gradients_are_bitwise_the_training_path(case):
    """One training step's gradients == the renderer's, fed the loss stage's dL/dr as the cotangent."""
    from smoe_b200 import SmoeRenderer
    from smoe_b200 import _ffi
    m, img, kw = _model(case)
    d, C = img.ndim - 1, img.shape[-1]
    p0 = m.get_params()
    m.run_batched(train=True, pis_l1=0, u_l1=0)
    g_train = m.get_gradients()
    r_train = m._d_res_pre.reshape(img.shape).clone()
    cot = _loss_cotangent(m, r_train)
    r = SmoeRenderer(grid=[(0, 1, n) for n in img.shape[:d]], channels=C, **kw)
    # diagnostic first: the per-pixel backward state the two paths hand to smoe_backward
    ts = tuple(_cuda(p0)[k] for k in PARAM_KEYS)
    out, state = r._forward(ts, keep_state=True)
    np.testing.assert_array_equal(out.cpu().numpy(), r_train.cpu().numpy())
    r._backward(out, state, cot.contiguous())
    nplanes = (3 + C) * _ffi.TPIX
    mine = state[4].reshape(r._ntiles, -1)[:, :nplanes]
    theirs = m._pix[:state[4].numel()].reshape(r._ntiles, -1)[:, :nplanes]
    np.testing.assert_array_equal(mine.cpu().numpy(), theirs.cpu().numpy())
    # the public op
    p = _cuda(p0, grad=True)
    r(p).backward(cot)
    g = _grads_np(p)
    for k in PARAM_KEYS:
        np.testing.assert_array_equal(g[k], g_train[k], err_msg=k)
    assert np.abs(g["musX"]).max() > 0


def _oracle(params, axes, cot, kw, C):
    """float64 graph r_pre and its gradient for the cotangent `cot`, at the float32 grid coordinates."""
    from oracle.graph import GraphCfg, ambiguity_margins, graph_forward
    d = len(axes)
    K = params["pis"].shape[0]
    grids = np.meshgrid(*[a.astype(np.float64) for a in axes], indexing="ij")
    dom = torch.tensor(np.stack([g.reshape(-1) for g in grids], axis=1))
    cfg = GraphCfg(dim_domain=d, num_channels=C, use_yuv=False, start_pis=K, **kw)
    leaf = {k: torch.tensor(np.asarray(v, np.float64), requires_grad=True) for k, v in params.items()}
    out = graph_forward(leaf, np.ones(K, bool), dom, torch.zeros(dom.shape[0], C, dtype=torch.float64), cfg)
    thr = ambiguity_margins(out, cfg)[0]
    ok = thr > 1e-3
    # pixels within float32 noise of a gate threshold may flip a gate: they carry no cotangent in either run, so the
    # gradients are compared conditional on the same gate decisions
    cot = np.where(ok[:, None], cot.reshape(-1, C), 0).astype(np.float32)
    gr = torch.autograd.grad(out["r_pre"], [leaf[k] for k in PARAM_KEYS],
                             grad_outputs=torch.tensor(cot.astype(np.float64)), allow_unused=True)
    g = {k: (np.zeros(leaf[k].shape) if gi is None else gi.numpy()) for k, gi in zip(PARAM_KEYS, gr)}
    return out["r_pre"].detach().numpy(), ok, cot, g


OFF_GRID = {
    # name: (model case, grid per axis as a function of the image shape, renderer flags)
    "gray_superres_2x": ("gray", lambda s: [(0, 1, 2 * n - 1) for n in s], dict(use_determinant=True,
                                                                                 train_inverse_cov=False)),
    "rgb_zoomed_crop": ("rgb", lambda s: [(0.3, 0.55, n) for n in s], dict(use_determinant=False,
                                                                            train_inverse_cov=True)),
    "rgb_extrapolating": ("rgb", lambda s: [(-0.1, 1.1, n) for n in s], dict(use_determinant=True,
                                                                              train_inverse_cov=True)),
    "gray_extrapolating_plain": ("gray", lambda s: [(-0.1, 1.1, n) for n in s], dict(use_determinant=False,
                                                                                      train_inverse_cov=False)),
    "video_superres_time": ("video_small", lambda s: [(0, 1, s[0]), (0, 1, s[1]), (0, 1, 2 * s[2] - 1)],
                            dict(use_determinant=True, train_inverse_cov=False)),
    "video_one_instant": ("video_small", lambda s: [(0, 1, s[0]), (0, 1, s[1]), (0.37, 0.37, 1)],
                          dict(use_determinant=False, train_inverse_cov=True)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(OFF_GRID))
def test_off_grid_render_and_gradients_match_the_float64_graph(name):
    import bench
    from smoe_b200 import Smoe, SmoeRenderer
    from smoe_b200.render import plan_grid
    case, grid_of, kw = OFF_GRID[name]
    img, k = {"gray": (bench.synth_image((32, 40, 1), 7), [6, 8]), "rgb": (bench.synth_image((24, 32, 3), 8), [5, 6]),
              "video_small": (bench.synth_image((12, 16, 6, 3), 9), [3, 4, 3])}[case]
    d, C = img.ndim - 1, img.shape[-1]
    m = Smoe(img, kernels_per_dim=k, **kw)
    p = _steer(m.get_params(), d, kw["train_inverse_cov"], seed=5)
    p["pis"][3] = -0.1                     # compacted away: no output, zero gradient
    grid = grid_of(img.shape[:d])
    axes = plan_grid(grid, C)[0]
    r = SmoeRenderer(grid=grid, channels=C, **kw)
    pt = _cuda(p, grad=True)
    out = r(pt)
    cot = np.random.RandomState(13).standard_normal(out.shape).astype(np.float32)
    ref, ok, cot_used, g_ref = _oracle(p, axes, cot, kw, C)
    out.backward(torch.tensor(cot_used.reshape(out.shape), device="cuda"))
    got = out.detach().cpu().numpy().reshape(-1, C)
    assert ok.mean() > 0.97
    assert np.abs(got[ok] - ref[ok]).max() <= 1e-5
    assert np.abs(got - ref).max() <= 2 * TAU * max(1.0, float(np.abs(ref).max()))     # at most one gate flip
    g = _grads_np(pt)
    for key in PARAM_KEYS:
        assert _rel(g[key], g_ref[key]) < 1e-4, (key, _rel(g[key], g_ref[key]))
    assert all(np.all(g[key][3] == 0) for key in PARAM_KEYS)
    assert np.all(np.triu(g["A_corr"]) == 0)
    assert np.all(g["A_diagonal"] * (1 - np.eye(d)) == 0)


@pytest.mark.gpu
@pytest.mark.parametrize("grid", [[(0.3, 0.55, 96), (0.3, 0.55, 160)], [(-0.1, 1.1, 96), (-0.1, 1.1, 160)]],
                         ids=["crop", "extrapolating"])
def test_culling_is_exact_off_the_training_grid(grid):
    """dense_exec 0 (culling + skipping), 1 (every pair), 2 (skipping only) give the same bits, on grids whose first
    coordinate is not 0 and whose spacing is not 1/(n-1), with most kernel centres far outside the crop."""
    from smoe_b200 import SmoeRenderer
    m, img, kw = _model("rgb")
    p0 = m.get_params()
    cot = torch.tensor(np.random.RandomState(2).standard_normal((96, 160, 3)).astype(np.float32), device="cuda")
    res = []
    for mode in (0, 1, 2, 0):
        r = SmoeRenderer(grid=grid, channels=3, _dense_exec=mode, **kw)
        p = _cuda(p0, grad=True)
        out = r(p)
        out.backward(cot)
        res.append([out.detach().cpu().numpy()] + [p[k].grad.cpu().numpy() for k in PARAM_KEYS])
    for b in (1, 2, 3):
        for q in range(len(res[0])):
            np.testing.assert_array_equal(res[0][q], res[b][q])
    assert np.abs(res[0][2]).max() > 0


@pytest.mark.gpu
def test_two_renders_in_one_graph():
    from smoe_b200 import SmoeRenderer
    m, img, kw = _model("rgb")
    p0 = m.get_params()
    r1 = SmoeRenderer(grid=[(0, 1, 191), (0, 1, 319)], channels=3, **kw)
    r2 = SmoeRenderer(grid=[(0.2, 0.6, 64), (0.1, 0.5, 80)], channels=3, **kw)

    def f(x):
        return (x.clamp(0, 1) - 0.5).abs().mean()

    def h(x):
        return (x * x).sum() * 1e-3

    p = _cuda(p0, grad=True)
    (f(r1(p)) + h(r2(p))).backward()
    both = _grads_np(p)
    p1, p2 = _cuda(p0, grad=True), _cuda(p0, grad=True)
    f(r1(p1)).backward()
    h(r2(p2)).backward()
    for k in PARAM_KEYS:
        np.testing.assert_array_equal(both[k], (p1[k].grad + p2[k].grad).cpu().numpy(), err_msg=k)


@pytest.mark.gpu
def test_no_host_sync_and_no_backward_state_without_grad():
    from smoe_b200 import SmoeRenderer
    m, img, kw = _model("gray")
    r = SmoeRenderer(grid=[(0, 1, 256), (0, 1, 256)], channels=1, **kw)
    p = _cuda(m.get_params(), grad=True)
    r(p).sum().backward()                   # warm-up: allocator, module loading
    for k in PARAM_KEYS:
        p[k].grad = None
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        out = r(p)
        (out * out).sum().backward()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert all(p[k].grad is not None for k in PARAM_KEYS)
    pix_bytes = r._pix_floats * 4
    del out
    for grad_on in (False, True):
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        with torch.set_grad_enabled(grad_on):
            out = r(p)
        peak = torch.cuda.max_memory_allocated() - base
        del out
        assert (peak >= pix_bytes) if grad_on else (peak < pix_bytes), (grad_on, peak, pix_bytes)
    with pytest.raises(RuntimeError):          # a render's backward state is consumed by its one backward
        out = r(p)
        out.sum().backward(retain_graph=True)
        out.sum().backward()


def test_grid_and_argument_validation():
    from smoe_b200.render import check_params, plan_grid
    axes, tile, b = plan_grid([(0, 1, 1080), (0, 1, 1920)], 3)
    np.testing.assert_array_equal(axes[0], np.linspace(0, 1, 1080).astype(np.float32))
    assert tile == (16, 32, 1) and list(b.dims) == [1080, 1920, 1] and list(b.extent) == [1080, 1920, 1]
    assert list(b.origin) == [0, 0, 0] and b.halo == 0
    axes, tile, b = plan_grid([(0, 1, 40), (0, 1, 48), (0.37, 0.37, 1)], 1)
    assert axes[2].tolist() == [np.float32(0.37)] and tile[0] * tile[1] * tile[2] == 512 and b.dims[2] == 1
    bad = [
        ([(0, 1, 0), (0, 1, 8)], 3),                 # n < 1
        ([(0, 1, 2.5), (0, 1, 8)], 3),               # n not an integer
        ([(1, 0, 8), (0, 1, 8)], 3),                 # reversed bounds
        ([(0.5, 0.5, 8), (0, 1, 8)], 3),             # empty interval with n > 1
        ([(0, float("nan"), 8), (0, 1, 8)], 3),      # not finite
        ([(0, 1, 8)], 3),                            # d = 1
        ([(0, 1, 8)] * 4, 3),                        # d = 4
        ([(0, 1), (0, 1, 8)], 3),                    # not (start, stop, n)
        ([(0, 1, 8), (0, 1, 8)], 2),                 # channels
        ([(0, 1, 65536), (0, 1, 32768)], 1),         # 2^31 pixels
        ([(0, 1, 65535 * 16 + 1), (0, 1, 8)], 1),    # too many tiles along the first axis
    ]
    for grid, C in bad:
        with pytest.raises(ValueError):
            plan_grid(grid, C)
    K, d, C = 5, 2, 3
    good = {"pis": torch.ones(K), "musX": torch.zeros(K, d), "A_diagonal": torch.zeros(K, d, d),
            "A_corr": torch.zeros(K, d, d), "gamma_e": torch.zeros(K, d, C), "nu_e": torch.zeros(K, C)}
    assert len(check_params(good, d, C)) == 6
    variants = [
        {k: v for k, v in good.items() if k != "nu_e"},                          # missing key
        dict(good, extra=torch.zeros(1)),                                         # extra key
        dict(good, musX=torch.zeros(K, 3)),                                       # wrong d
        dict(good, gamma_e=torch.zeros(K, d, 1)),                                 # wrong C
        dict(good, A_corr=torch.zeros(K + 1, d, d)),                              # wrong K
        dict(good, pis=torch.ones(K, 1)),                                         # pis not (K,)
        dict(good, nu_e=torch.zeros(K, C, dtype=torch.float64)),                  # dtype
        dict(good, nu_e=np.zeros((K, C), np.float32)),                            # not a tensor
    ]
    for v in variants:
        with pytest.raises(ValueError):
            check_params(v, d, C)
