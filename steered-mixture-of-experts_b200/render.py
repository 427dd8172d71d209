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
import torch.autograd.forward_ad as fwAD
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


def theta_rows(ts, d):
    """The six parameter tensors (PARAM_KEYS order) -> (K, P) theta rows: musX | the diagonal of A_diagonal and the
    strictly-lower part of A_corr, row by row | pis | nu_e | gamma_e.  The entries the op never reads are dropped."""
    pis, musX, A_diag, A_corr, gamma_e, nu_e = ts
    K = pis.shape[0]
    A_cols = torch.stack([A_diag[:, l, l] if l == m else A_corr[:, l, m] for l in range(d) for m in range(l + 1)], 1)
    return torch.cat([musX, A_cols, pis[:, None], nu_e, gamma_e.reshape(K, -1)], 1).contiguous()


def pack_model(cfg, ts, scale):
    """The six parameter tensors -> theta rows, Hilbert keys of the centres (smoe_spatial_keys, per-axis `scale`), a
    stable sort and smoe_pack on the current stream.  Returns (theta, packed, indices, counts, chunk_bounds)."""
    L, st, f32, i32 = lib(), stream_ptr(), torch.float32, torch.int32
    d, Cc = cfg.d, cfg.C
    P, PK = L.smoe_param_count(d, Cc), L.smoe_packed_stride(d, Cc)
    theta = theta_rows([t.detach() for t in ts], d)
    dev = theta.device
    K = theta.shape[0]
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


def tangent_rows(dts, K, d, Cc, device):
    """Forward-mode tangents of the six parameter tensors (None: no tangent) -> their (K, P) theta rows; raises
    ValueError for a shape or device that does not match the parameter's."""
    expect = dict(pis=(K,), musX=(K, d), A_diagonal=(K, d, d), A_corr=(K, d, d), gamma_e=(K, d, Cc), nu_e=(K, Cc))
    rows = []
    for k, dt in zip(PARAM_KEYS, dts):
        if dt is None:
            dt = torch.zeros(expect[k], dtype=torch.float32, device=device)
        elif tuple(dt.shape) != expect[k] or dt.device != device:
            raise ValueError(f"the tangent of {k!r} must have shape {expect[k]} on {device}, got "
                             f"{tuple(dt.shape)} on {dt.device}")
        rows.append(plain(dt).to(torch.float32))
    return theta_rows(rows, d)


def plain(t):
    """The device tensor under a `torch.func` transform's wrappers (a tangent or a saved output inside `jvp`),
    detached: the CUDA calls take its data pointer.  Used under torch._C._DisableFuncTorch(), so that the tensors the
    JVP computes from it stay plain too."""
    while torch._C._functorch.is_functorch_wrapped_tensor(t):
        t = torch._C._functorch.get_unwrapped(t)
    return t.detach()


def pack_tangent(cfg, theta, dts, indices, counts):
    """smoe_pack_tangent on the current stream: the parameter tangents -> one tangent record per packed row."""
    L = lib()
    K = theta.shape[0]
    dtheta = tangent_rows(dts, K, cfg.d, cfg.C, theta.device)
    tangent = torch.empty((K, L.smoe_tangent_stride(cfg.d, cfg.C)), dtype=torch.float32, device=theta.device)
    check(L.smoe_pack_tangent(C.byref(cfg), ptr(theta), ptr(dtheta), ptr(indices), ptr(counts), K, ptr(tangent),
                              stream_ptr()), "smoe_pack_tangent")
    return tangent


def traced(ts):
    """Whether a call must go through autograd: grad mode is on and a tensor requires grad, or a tensor carries a
    forward-mode tangent (a `forward_ad` dual tensor or a `torch.func` transform's tensor), which the no-grad fast
    path would drop."""
    if torch.is_grad_enabled() and any(t.requires_grad for t in ts):
        return True
    return any(torch._C._functorch.is_functorch_wrapped_tensor(t) or fwAD.unpack_dual(t).tangent is not None
               for t in ts)


class _Slot:
    """Hands a call's device state from an autograd Function's forward to its setup_context."""
    __slots__ = ("state",)


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


def check_weight(weight, shape, device):
    """The Gauss-Newton weight h, broadcastable to r's `shape` (..., C) -> (a (samples, C) view or copy, its sample
    stride, its channel stride), or (None, 0, 0) for h = 1; raises ValueError for a type, dtype, device or shape the
    call cannot take.  The values are not checked (that would synchronise)."""
    if weight is None:
        return None, 0, 0
    if not isinstance(weight, torch.Tensor):
        raise ValueError(f"weight must be a torch.Tensor or None, got {type(weight).__name__}")
    if weight.dtype != torch.float32:
        raise ValueError(f"weight must be float32, got {weight.dtype}")
    if weight.device != device:
        raise ValueError(f"weight is on {weight.device}, the renderer on {device}")
    try:
        ok = torch.broadcast_shapes(tuple(weight.shape), tuple(shape)) == tuple(shape)
    except RuntimeError:
        ok = False
    if not ok:
        raise ValueError(f"weight of shape {tuple(weight.shape)} does not broadcast to r's shape {tuple(shape)}")
    w = weight.detach().expand(tuple(shape))
    try:
        w = w.view(-1, shape[-1])                  # per-sample, per-channel or full weights need no copy
    except RuntimeError:
        w = w.reshape(-1, shape[-1]).contiguous()
    return w, w.stride(0), w.stride(1)


def weight_args(w, ss, sc):
    return (C.c_void_p(w.data_ptr()) if w is not None else ptr(None)), C.c_longlong(ss), C.c_longlong(sc)


def gn_finalize(cfg, raw_part, splits, plan, indices, counts, K, P):
    """smoe_reduce_splits + smoe_gn_diag_scatter: the split slabs of a Gauss-Newton diagonal sweep -> (K, P) rows in
    theta's layout and original kernel order, zero for kernels with pi <= 0."""
    L, st, dev = lib(), stream_ptr(), raw_part.device
    raw = torch.empty((K, P), dtype=torch.float32, device=dev)
    check(L.smoe_reduce_splits(C.byref(cfg), ptr(counts), K, splits, ptr(raw_part), ptr(plan), ptr(raw), st),
          "smoe_reduce_splits")
    diag = torch.zeros((K, P), dtype=torch.float32, device=dev)
    check(L.smoe_gn_diag_scatter(C.byref(cfg), ptr(raw), ptr(indices), ptr(counts), K, ptr(diag), st),
          "smoe_gn_diag_scatter")
    return diag


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
    (no retain_graph second pass).  `r.jacobian(params)` returns the render with its spatial Jacobian d r_c / d x_l.

    Forward mode: under `torch.func.jvp` or with `torch.autograd.forward_ad` dual tensors a call also returns the
    Jacobian-vector product dr = (d r / d params) . tangents, from one more CUDA sweep after the forward
    (smoe_pack_tangent + smoe_jvp); r is the plain call's, and the call's backward, if any, is unchanged.  As in
    reverse mode, tangents of kernels with pi <= 0 and of entries the op does not read have no effect, and the 0/1
    gate decision w > tau contributes no term.  `torch.func.vmap` / `jacfwd` have no batching rule.
    `r.gauss_newton_diagonal(params, weight=None)` returns the render with diag(J^T diag(h) J) in every parameter."""

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
        if traced(ts):
            return _Render.apply(self, _Slot(), *ts)
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

    def gauss_newton_diagonal(self, params, weight=None):
        """(r, D): the mixture r before clip on the grid, (n0, n1[, n2], C), bitwise the plain call's, and the
        Gauss-Newton diagonal D = diag(J^T diag(h) J) of J = d r / d params, a dict in the params' layout and dtype.

        `weight` is h, a float32 tensor on the renderer's device broadcastable to r's shape (per sample, per channel or
        both), or None for h = 1, which gives diag(J^T J).  For a loss sum_n,c l(r_c(x_n)), h = l'' gives the
        generalised Gauss-Newton diagonal; for 1/2 |r - y|^2 it is 1.  D is exact for whatever h is given: a Jacobi
        preconditioner for CG, Marquardt's scaling for Levenberg-Marquardt, or the sensitivity of the loss to each
        parameter.  As for the JVP, the 0/1 gate decision w > tau contributes no term; entries the op does not read
        and the rows of kernels with pi <= 0 are 0.  One forward, an elementwise state stage and one kernel-stationary
        CUDA sweep (smoe_gn_state, smoe_gn_diag, smoe_reduce_splits, smoe_gn_diag_scatter).  Both results are returned
        outside autograd.  Arguments are validated as by a call, and `weight`'s shape, dtype and device too; its
        values are not.  Nothing synchronises with the host."""
        ts = self._check(params)
        w, ss, sc = check_weight(weight, self.shape + (self.C,), self.device)
        with torch.no_grad(), torch.cuda.device(self.device):
            out, state = self._forward(ts, keep_state=True)
            L, st, dev = lib(), stream_ptr(), self.device
            theta, packed, indices, counts, pix, tile_qmin, _ = state
            K, P = theta.shape
            gstate = torch.empty((self._ntiles * L.smoe_gn_state_stride(self.d, self.C, C.byref(self._batch)),),
                                 dtype=torch.float32, device=dev)
            check(L.smoe_gn_state(C.byref(self._cfg), C.byref(self._batch), ptr(pix), ptr(out), *weight_args(w, ss, sc),
                                  ptr(gstate), st), "smoe_gn_state")
            splits = backward_splits(K, [self._batch])
            raw_part = torch.empty((splits * K * P,), dtype=torch.float32, device=dev)
            plan = torch.empty(((L.smoe_backward_plan_bytes(K, C.byref(self._batch)) + 3) // 4,), dtype=torch.int32,
                               device=dev)
            check(L.smoe_gn_diag(C.byref(self._cfg), C.byref(self._batch), ptr(packed), ptr(theta), ptr(indices),
                                 ptr(counts), K, ptr(gstate), ptr(tile_qmin), *self._axis_ptrs(), splits, ptr(raw_part),
                                 ptr(plan), st), "smoe_gn_diag")
            diag = gn_finalize(self._cfg, raw_part, splits, plan, indices, counts, K, P)
        return out, dict(zip(PARAM_KEYS, split_grads(diag, self.d, self.C)))

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

    def _jvp(self, out, state, dts):
        """smoe_pack_tangent + smoe_jvp after the forward that left `state`: dr for the parameter tangents dts."""
        theta, packed, indices, counts, pix, tile_qmin, chunk_bounds = state
        tangent = pack_tangent(self._cfg, theta, dts, indices, counts)
        dr = torch.empty_like(out)
        check(lib().smoe_jvp(C.byref(self._cfg), C.byref(self._batch), ptr(packed), ptr(tangent), ptr(counts),
                             ptr(chunk_bounds), theta.shape[0], ptr(pix), ptr(tile_qmin), *self._axis_ptrs(), ptr(out),
                             ptr(dr), stream_ptr()), "smoe_jvp")
        return dr


class _Render(torch.autograd.Function):
    @staticmethod
    def forward(renderer, slot, *ts):
        with torch.cuda.device(renderer.device):
            out, slot.state = renderer._forward(ts, keep_state=True)
        return out

    @staticmethod
    def setup_context(ctx, inputs, output):
        ctx.renderer = inputs[0]
        ctx.state = inputs[1].state
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(output)
        ctx.save_for_forward(output)

    @staticmethod
    def jvp(ctx, _renderer, _slot, *dts):
        (out,) = ctx.saved_tensors
        r = ctx.renderer
        with torch._C._DisableFuncTorch(), torch.cuda.device(r.device):
            return r._jvp(plain(out), ctx.state, dts)

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
        return (None, None) + tuple(g if need else None for g, need in zip(parts, ctx.needs_input_grad[2:]))


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
    points)` returns r with its spatial Jacobian d r_c / d x_l.

    Forward mode: under `torch.func.jvp` or with `torch.autograd.forward_ad` dual tensors, with tangents on the params
    and/or the points, a call also returns dr = (d r / d params) . v + (d r / d x) . xdot from one more CUDA sweep
    after the forward (smoe_pack_tangent when the params carry tangents, then smoe_point_jvp), as `SmoeRenderer`.
    `gauss_newton_diagonal(params, points, weight=None)` returns r with diag(J^T diag(h) J) in every parameter."""

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
        if traced((points,) + ts):
            return _PointRender.apply(self, _Slot(), points, *ts)
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

    def gauss_newton_diagonal(self, params, points, weight=None):
        """(r, D): the mixture r before clip at every point, (..., C) in the caller's order and bitwise the plain
        call's, and the Gauss-Newton diagonal D = diag(J^T diag(h) J) of J = d r / d params, a dict in the params'
        layout and dtype.  `weight` (h) is broadcastable to r's shape, or None for h = 1; see
        `SmoeRenderer.gauss_newton_diagonal`.  One forward, an elementwise state stage and one kernel-stationary CUDA
        sweep (smoe_point_gn_state, smoe_point_gn_diag, smoe_reduce_splits, smoe_gn_diag_scatter), outside autograd;
        nothing synchronises with the host."""
        ts = self._check(params, points)
        w, ss, sc = check_weight(weight, tuple(points.shape[:-1]) + (self.C,), self.device)
        with torch.no_grad(), torch.cuda.device(self.device):
            out, state = self._forward(points, ts, keep_state=True)
            L, st, dev = lib(), stream_ptr(), self.device
            theta, packed, indices, counts, chunk_bounds, order, r, pstate, tile_box = state
            K, P = theta.shape
            n = r.shape[0]
            gstate = torch.empty((L.smoe_point_tiles(n) * L.smoe_point_gn_state_stride(self.d, self.C),),
                                 dtype=torch.float32, device=dev)
            wp, wss, wsc = weight_args(w, ss, sc)
            check(L.smoe_point_gn_state(C.byref(self._cfg), n, ptr(pstate), ptr(r), wp, ptr(order), wss, wsc,
                                        ptr(gstate), st), "smoe_point_gn_state")
            splits = L.smoe_point_splits(K, n)
            raw_part = torch.empty((splits * K * P,), dtype=torch.float32, device=dev)
            plan = torch.empty(((L.smoe_point_plan_bytes(K, n) + 3) // 4,), dtype=torch.int32, device=dev)
            check(L.smoe_point_gn_diag(C.byref(self._cfg), ptr(packed), ptr(theta), ptr(indices), ptr(counts), K, n,
                                       ptr(gstate), ptr(tile_box), splits, ptr(raw_part), ptr(plan), st),
                  "smoe_point_gn_diag")
            diag = gn_finalize(self._cfg, raw_part, splits, plan, indices, counts, K, P)
        return out, dict(zip(PARAM_KEYS, split_grads(diag, self.d, self.C)))

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

    def _jvp(self, state, dpoints, dts):
        """smoe_pack_tangent (parameter tangents) + smoe_point_jvp after the forward that left `state`: dr (N, C) in
        the caller's order for the parameter tangents dts and the point tangents dpoints (None: none)."""
        L, dev, f32 = lib(), self.device, torch.float32
        theta, packed, indices, counts, chunk_bounds, order, r, pstate, tile_box = state
        n = r.shape[0]
        if dpoints is None and all(dt is None for dt in dts):
            return torch.zeros_like(r)
        tangent = pack_tangent(self._cfg, theta, dts, indices, counts) if any(dt is not None for dt in dts) else None
        dxs = None
        if dpoints is not None:
            if dpoints.numel() != n * self.d or dpoints.device != dev:
                raise ValueError(f"the tangent of the points must have {n} x {self.d} values on {dev}")
            dxs = plain(dpoints).to(f32).reshape(-1, self.d).index_select(0, order).contiguous()
        drs = torch.empty((n, self.C), dtype=f32, device=dev)
        check(L.smoe_point_jvp(C.byref(self._cfg), ptr(packed), ptr(tangent), ptr(counts), ptr(chunk_bounds),
                               theta.shape[0], n, ptr(pstate), ptr(tile_box), ptr(r), ptr(dxs), ptr(drs),
                               stream_ptr()), "smoe_point_jvp")
        return torch.empty_like(drs).index_copy_(0, order, drs)


class _PointRender(torch.autograd.Function):
    @staticmethod
    def forward(renderer, slot, points, *ts):
        with torch.cuda.device(renderer.device):
            out, slot.state = renderer._forward(points, ts, keep_state=True)
        return out

    @staticmethod
    def setup_context(ctx, inputs, output):
        ctx.renderer = inputs[0]
        ctx.state = inputs[1].state
        ctx.points_shape = inputs[2].shape
        ctx.set_materialize_grads(False)

    @staticmethod
    def jvp(ctx, _renderer, _slot, dpoints, *dts):
        r = ctx.renderer
        with torch._C._DisableFuncTorch(), torch.cuda.device(r.device):
            return r._jvp(ctx.state, dpoints, dts).reshape(ctx.points_shape[:-1] + (r.C,))

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out):
        if ctx.state is None:
            raise RuntimeError("SmoePointRenderer: a call's backward runs once (smoe_point_cotangent consumes the "
                               "forward's point state); evaluate again for another backward pass")
        r = ctx.renderer
        need_points, need_params = ctx.needs_input_grad[2], any(ctx.needs_input_grad[3:])
        with torch.cuda.device(r.device):
            grads, gx = r._backward(ctx.state, grad_out.to(torch.float32).contiguous(), need_params, need_points)
            ctx.state = None
            parts = split_grads(grads, r.d, r.C) if grads is not None else (None,) * len(PARAM_KEYS)
        return ((None, None, gx.reshape(ctx.points_shape) if gx is not None else None)
                + tuple(g if need else None for g, need in zip(parts, ctx.needs_input_grad[3:])))
