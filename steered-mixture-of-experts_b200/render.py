"""`SmoeRenderer`: a differentiable SMoE render for PyTorch on any uniform grid.

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
coordinates, so `(0, 1, n)` reproduces them bit for bit.  Grids that are not uniform cannot be expressed: the
backward's tile planner relies on uniform spacing.  Gates, the threshold tau = 0.5 / 2^precision (no
renormalisation), the determinant, `train_inverse_cov` and the exact culling are the training path's own kernels.
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
    (no retain_graph second pass)."""

    def __init__(self, grid, channels=3, use_determinant=False, train_inverse_cov=False, precision=8, device=None,
                 _dense_exec=0):
        axes, _, batch = plan_grid(grid, channels)
        if isinstance(precision, bool) or not isinstance(precision, (int, np.integer)) or not 1 <= precision <= 30:
            raise ValueError("precision must be an integer in [1, 30]")
        if _dense_exec not in (0, 1, 2):
            raise ValueError("_dense_exec must be 0, 1 or 2")
        _ffi.require_cuda()
        L = lib()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        if self.device.type != "cuda":
            raise ValueError("SmoeRenderer runs on a CUDA device")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        d = len(axes)
        self.d, self.C = d, int(channels)
        self.shape = tuple(len(x) for x in axes)
        self._batch = batch
        # the training path's configuration of a model without quantisation; the loss fields (margin, use_yuv) are
        # not read by the calls this op makes
        self._cfg = Cfg(d=d, C=self.C, precision=int(precision), use_determinant=int(bool(use_determinant)),
                        train_inverse_cov=int(bool(train_inverse_cov)), train_gammas=1, pis_lb=0.0, pis_ub=1.0,
                        pis_bits=8, q_ub=(C.c_float * 5)(*[1.0] * 5), q_bits=(C.c_int32 * 5)(*[8] * 5),
                        dense_exec=int(_dense_exec))
        self._P, self._PK = L.smoe_param_count(d, self.C), L.smoe_packed_stride(d, self.C)
        self._off = theta_offsets(d, self.C)
        self._key_scale = key_scale(self.shape)
        self._ntiles = L.smoe_num_tiles(C.byref(batch))
        self._pix_floats = self._ntiles * L.smoe_pix_stride(d, self.C, C.byref(batch))
        self._axes = [torch.from_numpy(x).to(self.device) for x in axes]

    def __call__(self, params):
        ts = check_params(params, self.d, self.C)
        for k, t in zip(PARAM_KEYS, ts):
            if t.device != self.device:
                raise ValueError(f"params[{k!r}] is on {t.device}, the renderer on {self.device}")
        if torch.is_grad_enabled() and any(t.requires_grad for t in ts):
            return _Render.apply(self, *ts)
        with torch.cuda.device(self.device):
            return self._forward(ts, keep_state=False)[0]

    def _axis_ptrs(self):
        return (ptr(self._axes[0]), ptr(self._axes[1]), ptr(self._axes[2]) if self.d == 3 else ptr(None))

    def _forward(self, ts, keep_state):
        """smoe_spatial_keys + sort + smoe_pack + smoe_forward on the current stream; with keep_state also the
        per-pixel state the backward needs."""
        L, st, dev, f32, i32 = lib(), stream_ptr(), self.device, torch.float32, torch.int32
        d, Cc, P, PK = self.d, self.C, self._P, self._PK
        pis, musX, A_diag, A_corr, gamma_e, nu_e = (t.detach() for t in ts)
        K = pis.shape[0]
        A_cols = torch.stack([A_diag[:, l, l] if l == m else A_corr[:, l, m] for l in range(d) for m in range(l + 1)], 1)
        theta = torch.cat([musX, A_cols, pis[:, None], nu_e, gamma_e.reshape(K, d * Cc)], 1).contiguous()
        keys = torch.empty((K,), dtype=torch.int64, device=dev)
        check(L.smoe_spatial_keys(ptr(theta), K, d, P, ptr(None), self._key_scale, ptr(keys), st), "smoe_spatial_keys")
        perm = torch.sort(keys, stable=True).indices.to(i32)
        kernel_list = torch.ones((K,), dtype=torch.uint8, device=dev)
        packed = torch.empty((K, PK), dtype=f32, device=dev)
        indices = torch.empty((K,), dtype=i32, device=dev)
        pos = torch.empty((K,), dtype=i32, device=dev)
        counts = torch.empty((4,), dtype=i32, device=dev)
        regsums = torch.empty((2,), dtype=f32, device=dev)
        chunk_bounds = torch.empty(((K + 127) // 128, 12), dtype=f32, device=dev)
        ws = torch.empty(((L.smoe_pack_workspace_bytes(K) + 15) // 4,), dtype=i32, device=dev)
        check(L.smoe_pack(C.byref(self._cfg), ptr(theta), ptr(None), ptr(None), ptr(kernel_list), ptr(perm), K,
                          ptr(packed), ptr(indices), ptr(pos), ptr(counts), ptr(regsums), ptr(chunk_bounds), ptr(ws),
                          ptr(None), ptr(None), ptr(None), st), "smoe_pack")
        out = torch.empty(self.shape + (Cc,), dtype=f32, device=dev)
        pix = torch.empty((self._pix_floats,), dtype=f32, device=dev) if keep_state else None
        tile_qmin = torch.empty((self._ntiles,), dtype=f32, device=dev) if keep_state else None
        check(L.smoe_forward(C.byref(self._cfg), C.byref(self._batch), ptr(packed), ptr(indices), ptr(counts),
                             ptr(chunk_bounds), K, ptr(None), *self._axis_ptrs(), ptr(out), ptr(None), ptr(None),
                             ptr(pix), ptr(tile_qmin), ptr(None), st), "smoe_forward")
        return out, (theta, packed, indices, counts, pix, tile_qmin)

    def _backward(self, out, state, grad_out):
        """smoe_cotangent + smoe_backward + smoe_grad_finalize; returns the (K, P) gradient rows of theta."""
        L, st, dev = lib(), stream_ptr(), self.device
        theta, packed, indices, counts, pix, tile_qmin = state
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
        grads = torch.zeros((K, P), dtype=torch.float32, device=dev)
        check(L.smoe_grad_finalize(C.byref(self._cfg), ptr(raw_part), splits, ptr(plan), K, ptr(theta), ptr(None),
                                   ptr(indices), ptr(counts), C.c_float(0.0), C.c_float(float(K)), C.c_float(0.0),
                                   ptr(grads), st), "smoe_grad_finalize")
        return grads

    def _split_grads(self, grads):
        """(K, P) gradient rows -> the params-dict layout, in PARAM_KEYS order."""
        d, Cc, o = self.d, self.C, self._off
        K = grads.shape[0]
        gA = torch.zeros((K, d, d), dtype=grads.dtype, device=grads.device)
        gC = torch.zeros_like(gA)
        for l in range(d):
            for m in range(l + 1):
                (gA if l == m else gC)[:, l, m] = grads[:, a_col(d, l, m)]
        return (grads[:, o["pi"]].contiguous(), grads[:, 0:d].contiguous(), gA, gC,
                grads[:, o["ga"]:].reshape(K, d, Cc).contiguous(), grads[:, o["nu"]:o["nu"] + Cc].contiguous())


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
            parts = r._split_grads(grads)
        return (None,) + tuple(g if need else None for g, need in zip(parts, ctx.needs_input_grad[1:]))
