"""`SmoeRenderer` and `SmoePointRenderer`: differentiable SMoE evaluation for PyTorch, on any uniform grid and at any
set of points.

The training path (`Smoe.run_batched`) samples the model on the pixel grid of its own image and back-propagates its
own loss.  An SMoE is a continuous function, so a user may want it on another grid -- a finer one
(super-resolution), a crop (zoom), times between frames (video) -- and may want to train it with a loss the library
does not know, or use it as one layer of a larger network.  `SmoeRenderer` is that: a `torch.autograd.Function` over
the same CUDA calls as a training step (smoe_pack, smoe_forward, smoe_backward, smoe_grad_finalize), with the loss
stage replaced by smoe_cotangent, which writes whatever dL/dr autograd hands back.

    r = SmoeRenderer(grid=[(0, 1, 2160), (0, 1, 3840)], channels=3)
    out = r(params)          # (2160, 3840, 3) float32, the mixture r before clip
    loss = (out.clamp(0, 1) - target).abs().mean()
    loss.backward()          # gradients in params[k].grad, the reference's variable layout

Each axis is `(start, stop, n)`: `np.linspace(start, stop, n)` cast to float32, as the training path builds its
coordinates, so `(0, 1, n)` reproduces them bit for bit.  Grids that are not uniform, and any other set of
coordinates, go to `SmoePointRenderer` (below), which also differentiates in the coordinates.  Gates, the threshold
tau = 0.5 / 2^precision (no renormalisation), the determinant, `train_inverse_cov` and the exact culling are the
training path's own kernels.
Fake quantisation, radial A, `use_diff_center` and kernel lists are not part of the op; a caller applies them in
torch to the tensors it passes.  Nothing synchronises with the host, so the op can be captured in a CUDA graph.
"""
from __future__ import annotations

import ctypes as C
import math
from collections.abc import Mapping

import numpy as np
import torch
from torch.autograd.function import once_differentiable

from . import _ffi
from ._ffi import Batch, Cfg, check, lib, ptr, stream_ptr
from .smoe import PARAM_KEYS, a_col, backward_splits, choose_tile, key_scale, theta_offsets

MAX_TILES_AXIS0 = 65535        # the loss / cotangent stages launch one CTA row per tile along the first axis


def plan_grid(grid, channels):
    """(start, stop, n) per axis -> (float32 coordinate axes, tile extents, one smoe_batch over the whole grid).
    Pure host code; raises ValueError for anything the kernels cannot take."""
    if isinstance(channels, bool) or channels not in (1, 3):
        raise ValueError("channels must be 1 or 3")
    try:
        grid = [tuple(ax) for ax in grid]
    except TypeError:
        raise ValueError("grid must be a sequence of (start, stop, n) per axis") from None
    d = len(grid)
    if d not in (2, 3):
        raise ValueError(f"the grid must have 2 (image) or 3 (video) axes, got {d}")
    axes = []
    for a, ax in enumerate(grid):
        if len(ax) != 3:
            raise ValueError(f"axis {a}: expected (start, stop, n), got {ax!r}")
        start, stop, n = ax
        if isinstance(n, bool) or not isinstance(n, (int, np.integer)) or n < 1:
            raise ValueError(f"axis {a}: n must be an integer >= 1, got {n!r}")
        start, stop = float(start), float(stop)
        if not (math.isfinite(start) and math.isfinite(stop)):
            raise ValueError(f"axis {a}: start and stop must be finite")
        x = np.linspace(start, stop, int(n)).astype(np.float32)
        if n > 1 and not x[-1] > x[0]:
            raise ValueError(f"axis {a}: stop must be greater than start (in float32) when n > 1")
        axes.append(x)
    shape = tuple(len(x) for x in axes)
    npix = int(np.prod(shape, dtype=np.int64))
    if npix >= 1 << 31:
        raise ValueError(f"the grid has {npix} pixels; at most 2^31 - 1 are supported")
    tile = choose_tile(d, shape[-1])
    if -(-shape[0] // tile[0]) > MAX_TILES_AXIS0:
        raise ValueError(f"axis 0: at most {MAX_TILES_AXIS0 * tile[0]} samples are supported")
    b = Batch()
    dims = shape + (1,) * (3 - d)
    for a in range(3):
        b.dims[a], b.origin[a], b.extent[a], b.tile[a] = dims[a], 0, dims[a], tile[a]
    b.inv_count = 1.0 / npix
    b.halo = 0
    return axes, tile, b


def check_params(params, d, C):
    """The params dict (the reference's variable layout) -> its six tensors in PARAM_KEYS order; raises ValueError
    for other keys, shapes or dtypes."""
    if not isinstance(params, Mapping) or set(params) != set(PARAM_KEYS):
        got = sorted(params) if isinstance(params, Mapping) else type(params).__name__
        raise ValueError(f"params must have exactly the keys {PARAM_KEYS}, got {got}")
    for k in PARAM_KEYS:
        if not isinstance(params[k], torch.Tensor):
            raise ValueError(f"params[{k!r}] must be a torch.Tensor")
    pis = params["pis"]
    if pis.dim() != 1 or pis.shape[0] < 1:
        raise ValueError(f"pis must have shape (K,) with K >= 1, got {tuple(pis.shape)}")
    K = pis.shape[0]
    expect = dict(pis=(K,), musX=(K, d), A_diagonal=(K, d, d), A_corr=(K, d, d), gamma_e=(K, d, C), nu_e=(K, C))
    for k in PARAM_KEYS:
        t = params[k]
        if tuple(t.shape) != expect[k]:
            raise ValueError(f"params[{k!r}] must have shape {expect[k]}, got {tuple(t.shape)}")
        if t.dtype != torch.float32:
            raise ValueError(f"params[{k!r}] must be float32, got {t.dtype}")
    return tuple(params[k] for k in PARAM_KEYS)


def check_options(precision, dense_exec):
    if isinstance(precision, bool) or not isinstance(precision, (int, np.integer)) or not 1 <= precision <= 30:
        raise ValueError("precision must be an integer in [1, 30]")
    if dense_exec not in (0, 1, 2):
        raise ValueError("_dense_exec must be 0, 1 or 2")


def resolve_device(device, who):
    _ffi.require_cuda()
    dev = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
    if dev.type != "cuda":
        raise ValueError(f"{who} runs on a CUDA device")
    return torch.device("cuda", torch.cuda.current_device()) if dev.index is None else dev


def make_cfg(d, C_, precision, use_determinant, train_inverse_cov, dense_exec):
    """The training path's configuration of a model without quantisation; the loss fields (margin, use_yuv) are not
    read by the calls the renderers make."""
    return Cfg(d=d, C=C_, precision=int(precision), use_determinant=int(bool(use_determinant)),
               train_inverse_cov=int(bool(train_inverse_cov)), train_gammas=1, pis_lb=0.0, pis_ub=1.0, pis_bits=8,
               q_ub=(C.c_float * 5)(*[1.0] * 5), q_bits=(C.c_int32 * 5)(*[8] * 5), dense_exec=int(dense_exec))


def pack_model(cfg, ts, scale):
    """The six parameter tensors -> theta rows, Hilbert keys of the centres (smoe_spatial_keys, per-axis `scale`), a
    stable sort and smoe_pack on the current stream.  Returns (theta, packed, indices, counts, chunk_bounds)."""
    L, st, f32, i32 = lib(), stream_ptr(), torch.float32, torch.int32
    d, Cc = cfg.d, cfg.C
    P, PK = L.smoe_param_count(d, Cc), L.smoe_packed_stride(d, Cc)
    pis, musX, A_diag, A_corr, gamma_e, nu_e = (t.detach() for t in ts)
    dev = pis.device
    K = pis.shape[0]
    A_cols = torch.stack([A_diag[:, l, l] if l == m else A_corr[:, l, m] for l in range(d) for m in range(l + 1)], 1)
    theta = torch.cat([musX, A_cols, pis[:, None], nu_e, gamma_e.reshape(K, d * Cc)], 1).contiguous()
    keys = torch.empty((K,), dtype=torch.int64, device=dev)
    check(L.smoe_spatial_keys(ptr(theta), K, d, P, ptr(None), scale, ptr(keys), st), "smoe_spatial_keys")
    perm = torch.sort(keys, stable=True).indices.to(i32)
    kernel_list = torch.ones((K,), dtype=torch.uint8, device=dev)
    packed = torch.empty((K, PK), dtype=f32, device=dev)
    indices = torch.empty((K,), dtype=i32, device=dev)
    pos = torch.empty((K,), dtype=i32, device=dev)
    counts = torch.empty((4,), dtype=i32, device=dev)
    regsums = torch.empty((2,), dtype=f32, device=dev)
    chunk_bounds = torch.empty(((K + 127) // 128, 12), dtype=f32, device=dev)
    ws = torch.empty(((L.smoe_pack_workspace_bytes(K) + 15) // 4,), dtype=i32, device=dev)
    check(L.smoe_pack(C.byref(cfg), ptr(theta), ptr(None), ptr(None), ptr(kernel_list), ptr(perm), K,
                      ptr(packed), ptr(indices), ptr(pos), ptr(counts), ptr(regsums), ptr(chunk_bounds), ptr(ws),
                      ptr(None), ptr(None), ptr(None), st), "smoe_pack")
    return theta, packed, indices, counts, chunk_bounds


def finalize_grads(cfg, raw_part, splits, plan, theta, indices, counts):
    """smoe_grad_finalize of a backward's statistics without regularisers -> the (K, P) gradient rows of theta."""
    K, P = theta.shape
    grads = torch.zeros((K, P), dtype=torch.float32, device=theta.device)
    check(lib().smoe_grad_finalize(C.byref(cfg), ptr(raw_part), splits, ptr(plan), K, ptr(theta), ptr(None),
                                   ptr(indices), ptr(counts), C.c_float(0.0), C.c_float(float(K)), C.c_float(0.0),
                                   ptr(grads), stream_ptr()), "smoe_grad_finalize")
    return grads


def split_grads(grads, d, Cc):
    """(K, P) gradient rows -> the params-dict layout, in PARAM_KEYS order."""
    o = theta_offsets(d, Cc)
    K = grads.shape[0]
    gA = torch.zeros((K, d, d), dtype=grads.dtype, device=grads.device)
    gC = torch.zeros_like(gA)
    for l in range(d):
        for m in range(l + 1):
            (gA if l == m else gC)[:, l, m] = grads[:, a_col(d, l, m)]
    return (grads[:, o["pi"]].contiguous(), grads[:, 0:d].contiguous(), gA, gC,
            grads[:, o["ga"]:].reshape(K, d, Cc).contiguous(), grads[:, o["nu"]:o["nu"] + Cc].contiguous())


class SmoeRenderer:
    """Differentiable render of an SMoE on a uniform grid; see the module docstring.

    grid      (start, stop, n) per axis: 2 axes (image) or 3 (video; n2 = 1 renders one time instant)
    channels  1 or 3
    use_determinant, train_inverse_cov, precision: as the `Smoe` constructor
    device    the CUDA device of the params (default: the current one)

    `r(params)` takes the dict of CUDA float32 tensors pis (K,), musX (K,d), A_diagonal (K,d,d), A_corr (K,d,d),
    gamma_e (K,d,C), nu_e (K,C) -- only the diagonal of A_diagonal and the strictly-lower part of A_corr are read --
    and returns the mixture r before clip, shape (n0, n1[, n2], C).  Any of the tensors may require grad; gradients
    are zero where a variable is not read and for kernels with pi <= 0, as in the reference's graph.  Every call
    allocates its own state, so several renders can live in one autograd graph.  A render's backward runs once
    (no retain_graph second pass).  `r.jacobian(params)` returns the render with its spatial Jacobian d r_c / d x_l."""

    def __init__(self, grid, channels=3, use_determinant=False, train_inverse_cov=False, precision=8, device=None,
                 _dense_exec=0):
        axes, _, batch = plan_grid(grid, channels)
        check_options(precision, _dense_exec)
        self.device = resolve_device(device, "SmoeRenderer")
        L = lib()
        d = len(axes)
        self.d, self.C = d, int(channels)
        self.shape = tuple(len(x) for x in axes)
        self._batch = batch
        self._cfg = make_cfg(d, self.C, precision, use_determinant, train_inverse_cov, _dense_exec)
        self._key_scale = key_scale(self.shape)
        self._ntiles = L.smoe_num_tiles(C.byref(batch))
        self._pix_floats = self._ntiles * L.smoe_pix_stride(d, self.C, C.byref(batch))
        self._axes = [torch.from_numpy(x).to(self.device) for x in axes]

    def __call__(self, params):
        ts = self._check(params)
        if torch.is_grad_enabled() and any(t.requires_grad for t in ts):
            return _Render.apply(self, *ts)
        with torch.cuda.device(self.device):
            return self._forward(ts, keep_state=False)[0]

    def jacobian(self, params):
        """(r, J): the mixture r before clip on the grid, (n0, n1[, n2], C), and its spatial Jacobian
        J[..., c, l] = d r_c / d x_l, (n0, n1[, n2], C, d), per unit of model coordinate (not per pixel).

        One forward and one CUDA sweep over the forward's per-pixel state (smoe_jacobian).  As with dL/dx of
        `SmoePointRenderer`, the 0/1 gate decision w > tau contributes no term.  Both tensors are returned outside
        autograd (requires_grad=False) whatever the params require: J is not differentiable.  Arguments are validated
        as by a call; nothing synchronises with the host."""
        ts = self._check(params)
        with torch.no_grad(), torch.cuda.device(self.device):
            out, state = self._forward(ts, keep_state=True)
            theta, packed, indices, counts, pix, tile_qmin, chunk_bounds = state
            jac = torch.empty(self.shape + (self.C, self.d), dtype=torch.float32, device=self.device)
            check(lib().smoe_jacobian(C.byref(self._cfg), C.byref(self._batch), ptr(packed), ptr(counts),
                                      ptr(chunk_bounds), theta.shape[0], ptr(pix), ptr(tile_qmin), *self._axis_ptrs(),
                                      ptr(out), ptr(jac), stream_ptr()), "smoe_jacobian")
        return out, jac

    def _check(self, params):
        """ValueError for params that __call__ and jacobian cannot take; returns the six parameter tensors."""
        ts = check_params(params, self.d, self.C)
        for k, t in zip(PARAM_KEYS, ts):
            if t.device != self.device:
                raise ValueError(f"params[{k!r}] is on {t.device}, the renderer on {self.device}")
        return ts

    def _axis_ptrs(self):
        return (ptr(self._axes[0]), ptr(self._axes[1]), ptr(self._axes[2]) if self.d == 3 else ptr(None))

    def _forward(self, ts, keep_state):
        """smoe_spatial_keys + sort + smoe_pack + smoe_forward on the current stream; with keep_state also the
        per-pixel state the backward needs."""
        L, st, dev, f32 = lib(), stream_ptr(), self.device, torch.float32
        Cc = self.C
        theta, packed, indices, counts, chunk_bounds = pack_model(self._cfg, ts, self._key_scale)
        K = theta.shape[0]
        out = torch.empty(self.shape + (Cc,), dtype=f32, device=dev)
        pix = torch.empty((self._pix_floats,), dtype=f32, device=dev) if keep_state else None
        tile_qmin = torch.empty((self._ntiles,), dtype=f32, device=dev) if keep_state else None
        check(L.smoe_forward(C.byref(self._cfg), C.byref(self._batch), ptr(packed), ptr(indices), ptr(counts),
                             ptr(chunk_bounds), K, ptr(None), *self._axis_ptrs(), ptr(out), ptr(None), ptr(None),
                             ptr(pix), ptr(tile_qmin), ptr(None), st), "smoe_forward")
        return out, (theta, packed, indices, counts, pix, tile_qmin, chunk_bounds)

    def _backward(self, out, state, grad_out):
        """smoe_cotangent + smoe_backward + smoe_grad_finalize; returns the (K, P) gradient rows of theta."""
        L, st, dev = lib(), stream_ptr(), self.device
        theta, packed, indices, counts, pix, tile_qmin, _ = state
        K, P = theta.shape
        check(L.smoe_cotangent(C.byref(self._cfg), C.byref(self._batch), ptr(out), ptr(grad_out), ptr(pix), st),
              "smoe_cotangent")
        splits = backward_splits(K, [self._batch])
        raw_part = torch.empty((splits * K * P,), dtype=torch.float32, device=dev)
        plan = torch.empty(((L.smoe_backward_plan_bytes(K, C.byref(self._batch)) + 3) // 4,), dtype=torch.int32,
                           device=dev)
        check(L.smoe_backward(C.byref(self._cfg), C.byref(self._batch), ptr(packed), ptr(counts), K, ptr(pix),
                              ptr(tile_qmin), *self._axis_ptrs(), splits, ptr(raw_part), ptr(plan), ptr(None), st),
              "smoe_backward")
        return finalize_grads(self._cfg, raw_part, splits, plan, theta, indices, counts)


class _Render(torch.autograd.Function):
    @staticmethod
    def forward(ctx, renderer, *ts):
        with torch.cuda.device(renderer.device):
            out, state = renderer._forward(ts, keep_state=True)
        ctx.renderer = renderer
        ctx.state = state
        ctx.save_for_backward(out)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out):
        if ctx.state is None:
            raise RuntimeError("SmoeRenderer: a render's backward runs once (smoe_cotangent consumes the forward's "
                               "per-pixel state); render again for another backward pass")
        (out,) = ctx.saved_tensors
        r = ctx.renderer
        with torch.cuda.device(r.device):
            grads = r._backward(out, ctx.state, grad_out.to(torch.float32).contiguous())
            ctx.state = None
            parts = split_grads(grads, r.d, r.C)
        return (None,) + tuple(g if need else None for g, need in zip(parts, ctx.needs_input_grad[1:]))


MAX_POINTS = 2147483136        # SMOE_POINT_MAX: point indices of the tiles stay below 2^31


def check_points(points, d, device):
    """The points tensor (..., d) -> its row count N; raises ValueError for a type, dtype, device or shape mismatch,
    N = 0 and N > MAX_POINTS."""
    if not isinstance(points, torch.Tensor):
        raise ValueError(f"points must be a torch.Tensor, got {type(points).__name__}")
    if points.dtype != torch.float32:
        raise ValueError(f"points must be float32, got {points.dtype}")
    if points.device != device:
        raise ValueError(f"points are on {points.device}, the renderer on {device}")
    if points.dim() < 1 or points.shape[-1] != d:
        raise ValueError(f"points must have shape (..., {d}), got {tuple(points.shape)}")
    n = points.numel() // d
    if n < 1:
        raise ValueError("points must hold at least one point")
    if n > MAX_POINTS:
        raise ValueError(f"{n} points; at most {MAX_POINTS} are supported")
    return n


class SmoePointRenderer:
    """Differentiable evaluation of an SMoE at arbitrary points, in the parameters and in the coordinates.

    d         2 (image) or 3 (video)
    channels  1 or 3
    use_determinant, train_inverse_cov, precision: as the `Smoe` constructor
    device    the CUDA device of the params and points (default: the current one)

    `r(params, points)` takes the params dict of `SmoeRenderer` and a float32 CUDA tensor of coordinates (..., d) and
    returns the mixture r before clip at every point, (..., C), in the caller's order.  Gradients reach the params as
    with `SmoeRenderer`, and `points` when it requires grad: dL/dx through the gates, the normaliser and the experts
    (the 0/1 gate decision w > tau is a step, whose derivative is 0 almost everywhere).

    Internally the points are sorted along a Hilbert curve over their bounding box (smoe_spatial_keys, a stable sort)
    and gathered into tiles of 512; outputs and point gradients are scattered back.  The order only affects speed,
    never the result.  Coordinates must be finite: a NaN or infinite coordinate is the caller's responsibility (that
    point's values are undefined, and its tile of 512 points is evaluated without culling).  Nothing synchronises with the host.  Under
    no_grad no backward state is allocated; in the backward, the parameter sweep runs only when a parameter needs a
    gradient and the coordinate sweep only when the points do.  A call's backward runs once.  `jacobian(params,
    points)` returns r with its spatial Jacobian d r_c / d x_l."""

    def __init__(self, d=2, channels=3, use_determinant=False, train_inverse_cov=False, precision=8, device=None,
                 _dense_exec=0):
        if isinstance(d, bool) or d not in (2, 3):
            raise ValueError("d must be 2 (image) or 3 (video)")
        if isinstance(channels, bool) or channels not in (1, 3):
            raise ValueError("channels must be 1 or 3")
        check_options(precision, _dense_exec)
        self.device = resolve_device(device, "SmoePointRenderer")
        self.d, self.C = int(d), int(channels)
        self._cfg = make_cfg(self.d, self.C, precision, use_determinant, train_inverse_cov, _dense_exec)
        self._stride = lib().smoe_point_stride(self.d, self.C)
        self._key_scale = key_scale((1,) * self.d)         # model coordinates: one scale on every axis

    def __call__(self, params, points):
        ts = self._check(params, points)
        if torch.is_grad_enabled() and (points.requires_grad or any(t.requires_grad for t in ts)):
            return _PointRender.apply(self, points, *ts)
        with torch.cuda.device(self.device):
            return self._forward(points, ts, keep_state=False)[0]

    def jacobian(self, params, points):
        """(r, J): the mixture r before clip at every point, (..., C), and its spatial Jacobian
        J[..., c, l] = d r_c / d x_l, (..., C, d), both in the caller's order and per unit of model coordinate.

        One forward and one CUDA sweep over the forward's state (smoe_point_jacobian) -- not C reverse passes.  As
        with dL/dx, the 0/1 gate decision w > tau contributes no term.  Both tensors are returned outside autograd
        (requires_grad=False) whatever the inputs require: J is not differentiable.  Arguments are validated as by a
        call; nothing synchronises with the host."""
        ts = self._check(params, points)
        with torch.no_grad(), torch.cuda.device(self.device):
            out, state = self._forward(points, ts, keep_state=True)
            L, st = lib(), stream_ptr()
            theta, packed, indices, counts, chunk_bounds, order, r, pstate, tile_box = state
            n = r.shape[0]
            jac = torch.empty((n, self.C, self.d), dtype=torch.float32, device=self.device)
            check(L.smoe_point_jacobian(C.byref(self._cfg), ptr(packed), ptr(counts), ptr(chunk_bounds), theta.shape[0],
                                        n, ptr(pstate), ptr(tile_box), ptr(r), ptr(jac), st), "smoe_point_jacobian")
            J = torch.empty_like(jac).index_copy_(0, order, jac)
        return out, J.reshape(points.shape[:-1] + (self.C, self.d))

    def _check(self, params, points):
        """ValueError for anything __call__ and jacobian cannot take; returns the six parameter tensors."""
        ts = check_params(params, self.d, self.C)
        for k, t in zip(PARAM_KEYS, ts):
            if t.device != self.device:
                raise ValueError(f"params[{k!r}] is on {t.device}, the renderer on {self.device}")
        check_points(points, self.d, self.device)
        return ts

    def _order(self, pts):
        """Stable Hilbert order of the points over their bounding box (one scale for every axis), on the device."""
        lo = pts.amin(0)
        ext = (pts.amax(0) - lo).amax()
        unit = (pts - lo) * torch.where(ext > 0, 1.0 / ext, torch.ones_like(ext))
        keys = torch.empty((pts.shape[0],), dtype=torch.int64, device=pts.device)
        check(lib().smoe_spatial_keys(ptr(unit.contiguous()), pts.shape[0], self.d, self.d, ptr(None), ptr(None),
                                      ptr(keys), stream_ptr()), "smoe_spatial_keys")
        return torch.sort(keys.to(torch.int32), stable=True).indices       # d * 10 bits: half the radix passes

    def _forward(self, points, ts, keep_state):
        """pack_model + point ordering + smoe_point_forward on the current stream; with keep_state also the point state
        the backward needs."""
        L, st, dev, f32 = lib(), stream_ptr(), self.device, torch.float32
        pts = points.detach().reshape(-1, self.d)
        n = pts.shape[0]
        theta, packed, indices, counts, chunk_bounds = pack_model(self._cfg, ts, self._key_scale)
        K = theta.shape[0]
        order = self._order(pts)
        sp = pts.index_select(0, order).contiguous()
        r = torch.empty((n, self.C), dtype=f32, device=dev)
        ntiles = L.smoe_point_tiles(n)
        state = torch.empty((ntiles * self._stride,), dtype=f32, device=dev) if keep_state else None
        tile_box = torch.empty((ntiles, 8), dtype=f32, device=dev) if keep_state else None
        check(L.smoe_point_forward(C.byref(self._cfg), ptr(packed), ptr(counts), ptr(chunk_bounds), K, ptr(sp), n,
                                   ptr(r), ptr(state), ptr(tile_box), st), "smoe_point_forward")
        out = torch.empty_like(r).index_copy_(0, order, r)
        return out.reshape(points.shape[:-1] + (self.C,)), (theta, packed, indices, counts, chunk_bounds, order, r,
                                                           state, tile_box)

    def _backward(self, state, grad_out, need_params, need_points):
        """smoe_point_cotangent, then smoe_point_backward + smoe_grad_finalize (need_params) and smoe_point_xgrad
        (need_points); returns the (K, P) gradient rows of theta or None, and dL/dx (N, d) or None."""
        L, st, dev, f32 = lib(), stream_ptr(), self.device, torch.float32
        theta, packed, indices, counts, chunk_bounds, order, r, pstate, tile_box = state
        K, P = theta.shape
        n = r.shape[0]
        g = grad_out.reshape(-1, self.C).index_select(0, order).contiguous()
        check(L.smoe_point_cotangent(C.byref(self._cfg), n, ptr(r), ptr(g), ptr(pstate), st), "smoe_point_cotangent")
        grads = gx = None
        if need_params:
            splits = L.smoe_point_splits(K, n)
            raw_part = torch.empty((splits * K * P,), dtype=f32, device=dev)
            plan = torch.empty(((L.smoe_point_plan_bytes(K, n) + 3) // 4,), dtype=torch.int32, device=dev)
            check(L.smoe_point_backward(C.byref(self._cfg), ptr(packed), ptr(counts), K, n, ptr(pstate), ptr(tile_box),
                                        splits, ptr(raw_part), ptr(plan), st), "smoe_point_backward")
            grads = finalize_grads(self._cfg, raw_part, splits, plan, theta, indices, counts)
        if need_points:
            gs = torch.empty((n, self.d), dtype=f32, device=dev)
            check(L.smoe_point_xgrad(C.byref(self._cfg), ptr(packed), ptr(counts), ptr(chunk_bounds), K, n, ptr(pstate),
                                     ptr(tile_box), ptr(gs), st), "smoe_point_xgrad")
            gx = torch.empty_like(gs).index_copy_(0, order, gs)
        return grads, gx


class _PointRender(torch.autograd.Function):
    @staticmethod
    def forward(ctx, renderer, points, *ts):
        with torch.cuda.device(renderer.device):
            out, state = renderer._forward(points, ts, keep_state=True)
        ctx.renderer = renderer
        ctx.state = state
        ctx.points_shape = points.shape
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out):
        if ctx.state is None:
            raise RuntimeError("SmoePointRenderer: a call's backward runs once (smoe_point_cotangent consumes the "
                               "forward's point state); evaluate again for another backward pass")
        r = ctx.renderer
        need_points, need_params = ctx.needs_input_grad[1], any(ctx.needs_input_grad[2:])
        with torch.cuda.device(r.device):
            grads, gx = r._backward(ctx.state, grad_out.to(torch.float32).contiguous(), need_params, need_points)
            ctx.state = None
            parts = split_grads(grads, r.d, r.C) if grads is not None else (None,) * len(PARAM_KEYS)
        return ((None, gx.reshape(ctx.points_shape) if gx is not None else None)
                + tuple(g if need else None for g, need in zip(parts, ctx.needs_input_grad[2:])))
