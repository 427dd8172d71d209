"""`Smoe`: the reference's model object (smoe.py:37-2578) on top of libsmoe_b200 (sm_100a CUDA).

Same constructor keywords, `set_optimizer` / `train` / `run_batched` / getters, the params dict
(`pis, musX, A_diagonal, A_corr, gamma_e, nu_e`), `kernel_list_per_batch`, history lists and
`qparams` / `rparams` as the reference, so `logger.py`, `plotter.py`, `utils.save_model`,
`quantizer.py` and the `smoe_reconstruction*.py` entry points work against it unchanged.
What changed is everything below `run_batched`: the TensorFlow graph (`init_model`,
smoe.py:331-1064) and `session.run` (smoe.py:1702, 1788) are replaced by hand-written CUDA
kernels called through the C ABI of include/smoe_b200.h.  There is no CPU path.

Deliberate deviations from HEAD (SURVEY.md section 8c, DESIGN.md "Decisions"):
  D1  single-model path only: affines / train_trafo / train_svs / add_kernel_slots>0 /
      dim_domain>=4 raise NotImplementedError (so does radial_as with quantization_mode 3);
      quantization_mode 0-3, quantize_pis, use_diff_center, radial_as, kernel_count_as_norm_l1,
      ssim_opt, overlap_of_batches, loss_mask and sampling_percentage are all on the CUDA path;
  D5  `init_params['A_diagonal'] + init_params['A_corr']` is split back into its diagonal
      (-> A_diagonal) and strictly-lower part (-> A_corr) instead of being stored whole in
      A_diagonal (where the reference's band_part then drops the steering, smoe.py:256, 436, 732);
  the TF leaks `smoe.session.run(smoe.re_assign_*_op)` are replaced by `set_params(dict)`.
"""
from __future__ import annotations

import ctypes as C
import math
from itertools import product

import numpy as np
import torch

import os
import warnings

from . import _ffi
from ._ffi import Adam, Batch, Cfg, Peers, check, lib, ptr, stream_ptr
from .quantizer import quantize_params, rescaler

PARAM_KEYS = ("pis", "musX", "A_diagonal", "A_corr", "gamma_e", "nu_e")


def theta_offsets(d, C):
    """First column of each variable in a theta row (include/smoe_b200.h): musX | A lower triangle | pis | nu_e |
    gamma_e."""
    T = d * (d + 1) // 2
    return dict(mu=0, A=d, pi=d + T, nu=d + T + 1, ga=d + T + 1 + C)


def a_col(d, l, m):
    """Column of A[l, m] (l >= m) in a theta row: the lower triangle, row-major."""
    return d + l * (l + 1) // 2 + m


def choose_tile(d, n_last):
    """Tile extents (product SMOE_TPIX) of a batch of dimension d whose last axis has n_last samples."""
    if d == 2:
        return (_ffi.TPIX // 32, 32, 1)
    # tile[1]*tile[2] must divide 128 and tile[2] must be a multiple of 4 (include/smoe_b200.h)
    t2 = 8 if n_last > 4 else 4
    t1 = 64 // t2
    return (_ffi.TPIX // (t1 * t2), t1, t2)


def key_scale(shape):
    """Per-axis scale of the Hilbert keys (smoe_spatial_keys): n_a / max n, so the curve is isotropic in pixels."""
    nmax = float(max(shape))
    return (C.c_float * 3)(*([n / nmax for n in shape] + [1.0] * (3 - len(shape))))


def backward_splits(k_eff, batches):
    """Pixel splits of smoe_backward for k_eff kernels with work (at least 64) over `batches`; SMOE_SPLITS overrides."""
    return int(os.environ.get("SMOE_SPLITS", 0)) or max(int(lib().smoe_suggest_splits(max(64, k_eff), C.byref(b)))
                                                        for b in batches)


def sliding_window(image, Overlap, BatchSize):
    """Yields (coord, window) over the domain axes, first axis outermost, last innermost, with a
    zero halo of `Overlap` (smoe.py:18-35)."""
    nd = image.ndim - 1
    if nd not in (2, 3):
        return
    pad = np.pad(image, [(Overlap, Overlap)] * nd + [(0, 0)], "constant", constant_values=0)
    starts = [range(0, pad.shape[a] - 2 * Overlap, BatchSize[a]) for a in range(nd)]
    for org in product(*starts):
        sl = tuple(slice(o, o + BatchSize[a] + 2 * Overlap) for a, o in enumerate(org))
        yield np.array(org) - Overlap, pad[sl + (slice(None),)]


class AdamOptimizer:
    """Stand-in for `tf.train.AdamOptimizer(lr)` as the reference constructs it
    (smoe_test.py:84-88); `Smoe.set_optimizer` reads `._lr` (smoe.py:1120)."""

    def __init__(self, learning_rate=0.001, beta1=0.9, beta2=0.999, epsilon=1e-8):
        self._lr = learning_rate
        self._beta1, self._beta2, self._epsilon = beta1, beta2, epsilon
        self._t = 0
        # TF1 keeps beta1_power / beta2_power as float32 variables, multiplied by float32(beta) after every
        # apply_gradients (optimizer `_finish`); lr_t uses the powers BEFORE that update, i.e. beta^t at step t
        self._b1p = np.float32(1.0)
        self._b2p = np.float32(1.0)

    def _step_alpha(self):
        """Advance the beta powers once (one apply_gradients) and return TF's lr_t in float32."""
        f = np.float32
        self._t += 1
        self._b1p = f(self._b1p * f(self._beta1))
        self._b2p = f(self._b2p * f(self._beta2))
        return float(f(self._lr) * np.sqrt(f(1) - self._b2p) / (f(1) - self._b1p))

    def _set_step(self, t):
        """Restore the step count (checkpoint restore): replays the float32 products."""
        f = np.float32
        self._t, self._b1p, self._b2p = 0, f(1.0), f(1.0)
        for _ in range(int(t)):
            self._t += 1
            self._b1p = f(self._b1p * f(self._beta1))
            self._b2p = f(self._b2p * f(self._beta2))


class Smoe:
    def __init__(self, image, kernels_per_dim=None, train_pis=True, init_params=None, start_batches=1,
                 batch_size=None, train_gammas=True, train_musx=True, use_diff_center=False, radial_as=False,
                 use_determinant=False, normalize_pis=True, quantization_mode=0, bit_depths=None,
                 quantize_pis=False, lower_bounds=None, upper_bounds=None, use_yuv=True, only_y_gamma=False,
                 ssim_opt=False, precision=8, add_kernel_slots=0, iter_offset=0, margin=0.5,
                 overlap_of_batches=0, kernel_count_as_norm_l1=False, train_svs=False, affines=None,
                 train_trafo=False, num_params_model=6, train_inverse_cov=True, init_flag=1,
                 only_rec_from_checkpoint=False, loss_mask=None, device=None, dense_exec=False,
                 process_group=None, distributed=None, eps_bits=0, _decoder_only=False, _emulate_shard=None):
        _ffi.require_cuda()
        lib()
        unsupported = {"affines": affines is not None, "train_trafo": train_trafo, "train_svs": train_svs,
                       "add_kernel_slots": add_kernel_slots > 0,
                       # HEAD's mode-3 form for radial kernels clamps the un-shifted scalars to [0, max - min]
                       # (smoe.py:498-504), which is not a usable quantiser
                       "radial_as with quantization_mode 3": radial_as and quantization_mode == 3}
        for k, v in unsupported.items():
            if v:
                raise NotImplementedError(f"{k}: outside the single-model hot path (SURVEY.md 8, decision D1)")
        image = np.ascontiguousarray(np.asarray(image), dtype=np.float32)
        if image.ndim - 1 not in (2, 3):
            raise NotImplementedError("dim_domain must be 2 (image) or 3 (video)")
        if image.shape[-1] not in (1, 3):
            raise NotImplementedError("1 or 3 channels")
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        # --- reference attributes (smoe.py:42-221) ---
        self.use_yuv, self.only_y_gamma, self.ssim_opt = use_yuv, only_y_gamma, ssim_opt
        self.use_diff_center, self.precision = use_diff_center, precision
        self.add_kernel_slots, self.kernel_count_as_norm_l1 = add_kernel_slots, kernel_count_as_norm_l1
        self.qparams = self.rparams = None
        self.losses, self.qlosses, self.losses_history = [], [], []
        self.best_loss = self.best_qloss = None
        self.mses, self.qmses, self.mses_history = [], [], []
        self.best_mse, self.best_qmse = [], []
        self.num_pis, self.num_svs = [], []
        self.iter = iter_offset
        self.valid = self.qvalid = False
        self.reconstruction_image = self.weight_matrix_argmax = None
        self.qreconstruction_image = self.qweight_matrix_argmax = None
        self.train_pis, self.train_gammas, self.train_musx = train_pis, train_gammas, train_musx
        self.radial_as, self.use_determinant = radial_as, use_determinant
        self.quantization_mode, self.bit_depths, self.quantize_pis = quantization_mode, bit_depths, quantize_pis
        self.lower_bounds, self.upper_bounds = lower_bounds, upper_bounds
        self.with_SV, self.train_trafo, self.train_inverse_cov = train_svs, train_trafo, train_inverse_cov
        self.affines, self.loss_mask = affines, loss_mask
        self.only_rec_from_checkpoint = only_rec_from_checkpoint
        self.optimizer1 = self.optimizer2 = self.optimizer3 = None
        self.grad_clip_value_abs = None
        if quantization_mode not in (0, 1, 2, 3):
            raise ValueError("quantization_mode must be 0, 1, 2 or 3")
        if quantization_mode >= 2:
            self.quantize_pis = quantize_pis = True          # smoe.py:474 (and smoe_test.py:36-37)
        if quantize_pis and (lower_bounds is None or upper_bounds is None or bit_depths is None):
            raise ValueError("quantize_pis / quantization_mode 2 need lower_bounds, upper_bounds and bit_depths")

        self.start_batches = start_batches
        self.overlap = int(overlap_of_batches)                # smoe.py:244
        if self.overlap < 0:
            raise ValueError("overlap_of_batches must be >= 0")
        self.eps_bits = int(eps_bits)
        if self.eps_bits and not 24 <= self.eps_bits <= 126:
            raise ValueError("eps_bits must be 0 (exact) or in [24, 126]")
        self.image = image
        self.dim_domain = image.ndim - 1
        self.num_pixel = int(np.prod(image.shape[:self.dim_domain]))
        self.joint_domain_shape = tuple(image.shape[:-1]) + (self.dim_domain + image.shape[-1],)
        self.batch_shape = self.get_batch_shape(start_batches, self.joint_domain_shape)
        d = self.dim_domain
        if batch_size is not None and batch_size[0] is not None:          # smoe.py:231-243
            if len(batch_size) == d:
                self.batch_size_valued = tuple(int(b) for b in batch_size)
            elif len(batch_size) == 1:
                self.batch_size_valued = (int(batch_size[0]),) * d
            else:
                raise ValueError("Required BatchSize doesn't fit to input dimension")
            for ii in range(d):
                if image.shape[ii] % self.batch_size_valued[ii] > 0:
                    raise ValueError("Required BatchSize is not compatible to input dimensions")
        else:
            self.batch_size_valued = tuple(self.batch_shape[:-1])
        if self.overlap > min(self.batch_size_valued):
            # a window narrower than its halo would count partly-halo rows in the loss (the kernels derive the halo
            # from the clipped rectangle); the reference has no such configuration either (smoe_test.py:322-325)
            raise ValueError("overlap_of_batches must not exceed the smallest batch extent")
        self.batch_size = tuple(np.array(self.batch_size_valued) + 2 * self.overlap)
        self.start_batches = int(np.prod(np.ceil(np.array(image.shape[:-1]) / np.array(self.batch_size_valued))))

        assert kernels_per_dim is not None or init_params is not None, \
            "You need to specify the kernel grid size or give initial parameters."
        if init_params:
            self.pis_init = np.asarray(init_params["pis"])
            self.musX_init = np.asarray(init_params["musX"])
            Ad0 = np.asarray(init_params["A_diagonal"])
            if Ad0.ndim == 1:                                   # smoe.py:334-335: a vector of scalars means radial
                self.A_init, self.radial_as = Ad0, True
            else:
                self.A_init = Ad0 + np.asarray(init_params["A_corr"])
            self.gamma_e_init = np.asarray(init_params["gamma_e"])
            self.nu_e_init = np.asarray(init_params["nu_e"])
        else:
            self.generate_kernel_grid(kernels_per_dim)
            # the decoder feeds every expert over the graph (smoe_reconstruction_decoded.py:34-45), so the
            # block-mean initialisation (a Python loop over the full H/4 x W/4 grid) would be dead work
            self.generate_experts(with_means=not _decoder_only)
            self.generate_pis(normalize_pis)
        self.start_pis = int(self.pis_init.size)
        self.kernel_count = self.start_pis
        self.margin = margin

        # --- distributed sharding (SURVEY.md 8e): one rectangular block of pixels per rank ---
        self._pg = process_group
        self._world, self._rank = 1, 0
        self._emulated = _emulate_shard is not None      # profiling aid: the work of rank r of R on one GPU, no exchange
        if self._emulated:
            self._rank, self._world = int(_emulate_shard[0]), int(_emulate_shard[1])
        elif distributed is not False and torch.distributed.is_available() and torch.distributed.is_initialized():
            self._world = torch.distributed.get_world_size(process_group)
            self._rank = torch.distributed.get_rank(process_group)
        d = self.dim_domain
        if self._world > 1:
            if self._world > _ffi.MAX_PEERS:
                raise NotImplementedError(f"at most {_ffi.MAX_PEERS} ranks (one NVSwitch node)")
            if self.start_batches != 1:
                raise NotImplementedError("pixel sharding over ranks needs start_batches == 1")
            # (overlap_of_batches is a no-op here: a sharded model is ONE batch, and a single window has no halo;
            # ssim_opt pulls a ring of neighbour pixels over NVLink, see _init_halo)
            self._blocks = self._choose_blocks(self._world)
            self._block = self._blocks[self._rank]
        else:
            self._block = tuple((0, image.shape[a]) for a in range(d))
            self._blocks = [self._block]
        self._band = self._block[0]

        self._init_device(dense_exec)

    # ------------------------------------------------------------------------------------------
    # initialisers (smoe.py:2146-2242, 2395-2426, 2459-2543)
    # ------------------------------------------------------------------------------------------
    @staticmethod
    def gen_domain(in_, dim_of_input_space=2):
        if isinstance(in_, np.ndarray):
            axes = [np.linspace(0, 1, in_.shape[a]) for a in range(dim_of_input_space)]
            mesh = np.stack(np.meshgrid(*axes, indexing="ij"), axis=-1)
            return np.append(mesh, in_, axis=-1)
        per_dim = [int(in_[a] if len(in_) > 1 else in_[0]) for a in range(dim_of_input_space)]
        axes = [np.linspace((1 / n) / 2, 1 - (1 / n) / 2, n) for n in per_dim]
        mesh = np.stack(np.meshgrid(*axes, indexing="ij"), axis=-1)
        return mesh.reshape(int(np.prod(per_dim)), dim_of_input_space)

    def generate_kernel_grid(self, kernels_per_dim):
        d = self.image.ndim - 1
        self.musX_init = self.gen_domain(list(kernels_per_dim), d)
        per_dim = [kernels_per_dim[a] if len(kernels_per_dim) > 1 else kernels_per_dim[0] for a in range(d)]
        proto = np.diag(np.array([2 * (n + 1) for n in per_dim], dtype=np.float64))
        self.A_init = np.tile(proto, (self.musX_init.shape[0], 1, 1))
        if self.train_inverse_cov:
            self.A_init = self.A_init ** 2

    def generate_experts(self, with_means=True):
        assert self.musX_init is not None, "need musX to generate experts"
        d, Cc = self.dim_domain, self.image.shape[-1]
        K = self.musX_init.shape[0]
        self.gamma_e_init = np.zeros((K, d, Cc))
        if not with_means:
            self.nu_e_init = np.ones((K, Cc)) * 0.5
            return
        half = self.musX_init[0]
        ext = self.image.shape[:d]
        lo = np.empty((K, d), dtype=np.int64)
        hi = np.empty((K, d), dtype=np.int64)
        for a in range(d):          # python round(): half to even, as the reference's int(round(.))
            lo[:, a] = [int(round(v)) for v in (self.musX_init[:, a] - half[a]) * ext[a]]
            hi[:, a] = [int(round(v)) for v in (self.musX_init[:, a] + half[a]) * ext[a]]
        mean = np.empty((K, Cc), dtype=np.float32)
        red = tuple(range(d))
        for k in range(K):
            block = self.image[tuple(slice(lo[k, a], hi[k, a]) for a in range(d))]
            mean[k] = np.mean(block, axis=red)
        self.nu_e_init = mean

    def generate_pis(self, normalize_pis):
        K = self.musX_init.shape[0]
        self.pis_init = np.ones((K,), dtype=np.float32)
        if normalize_pis:
            self.pis_init = self.pis_init / K

    @staticmethod
    def get_batch_shape(desired_batches, joint_domain_shape):
        """Divisor tiling with the smallest batch count >= desired_batches, most cube-like
        (smoe.py:2459-2543; candidate order and tie-breaking as in the reference)."""
        def divisors(n):
            fac, nn, i = {}, n, 2
            while i * i <= nn:
                while nn % i == 0:
                    fac[i] = fac.get(i, 0) + 1
                    nn //= i
                i += 1
            if nn > 1:
                fac[nn] = 1
            out = [1]
            for p in reversed(list(fac.keys())):       # innermost prime varies slowest
                out = [o * p ** e for o in out for e in range(fac[p] + 1)]
            return out
        nd = len(joint_domain_shape)
        factors = [divisors(joint_domain_shape[a]) for a in range(nd - 1)] + [[1]]
        if nd > 4:
            factors[0] = factors[1] = [1]
        shapes = list(product(*factors))
        counts = np.array([np.prod(s[:-1]) for s in shapes], dtype=np.float64)
        diff = counts - desired_batches
        diff[diff < 0] = np.inf
        aimed = counts[int(np.argmin(diff))]
        cand = [s for s, c in zip(shapes, counts) if c == aimed]
        sums = [np.sum(c[2:3]) if len(c) > 4 else np.sum(c) for c in cand]
        div = cand[int(np.argmin(sums))]
        return tuple(int(joint_domain_shape[a] / div[a]) for a in range(nd))

    # ------------------------------------------------------------------------------------------
    # pixel sharding (SURVEY.md 8e): block decomposition
    # ------------------------------------------------------------------------------------------
    def _reach_px(self):
        """Per axis, the distance in pixels over which a kernel's float32 gate can be non-zero (logit within 126
        of its peak), estimated from the median initial steering matrix.  A heuristic that only steers the block
        decomposition and the pixel-split count -- results never depend on it."""
        d = self.dim_domain
        A = np.asarray(self.A_init, dtype=np.float64)
        diag = np.stack([A] * d, 1) if A.ndim == 1 else np.stack([A[:, a, a] for a in range(d)], 1)
        med = np.maximum(np.median(np.abs(diag), axis=0), 1e-6)
        q = 0.72134752 * (med if self.train_inverse_cov else med ** 2)          # diagonal of Qm (log2 domain)
        return [float(np.sqrt(126.0 / q[a]) * max(self.image.shape[a] - 1, 1)) for a in range(d)]

    def _choose_blocks(self, world, halo_weight=0.5):
        """One rectangular block per rank, rank = row-major index in the block grid.  A rank's work grows with its
        block PLUS the strip around it that foreign kernels reach into (the backward visits those tiles, the forward
        sweeps those kernels), so the grid factorisation minimises prod_a (w_a + halo_a) -- 2x4 rather than 8x1 bands
        on a 1080p frame.  The cuts themselves are equal and rounded to the tile grid (no rank gets partial tiles it
        would not have had otherwise): the time of a rank follows its pixel count."""
        d = self.dim_domain
        n = self.image.shape[:d]
        tile = (16, 32) if d == 2 else (8, 8, 8)
        reach = [halo_weight * r for r in self._reach_px()]

        def factorisations(w, k):
            if k == 1:
                yield (w,)
                return
            for f in range(1, w + 1):
                if w % f == 0:
                    for rest in factorisations(w // f, k - 1):
                        yield (f,) + rest

        best, best_cost = None, None
        forced = os.environ.get("SMOE_BLOCK_GRID")              # e.g. "2,4": override the factorisation (experiments)
        if forced:
            best = tuple(int(v) for v in forced.split(","))
            if len(best) != d or int(np.prod(best)) != world:
                raise ValueError("SMOE_BLOCK_GRID must have one factor per domain axis and multiply to the world size")
        for fac in ([] if forced else factorisations(world, d)):
            if any(n[a] // fac[a] < 1 for a in range(d)):
                continue
            cost = 1.0
            for a in range(d):
                eff = (n[a] + reach[a] * (2 * fac[a] - 2)) / fac[a]
                cost *= max(eff, float(tile[a]))                 # a block thinner than a tile still costs a tile
            if best_cost is None or cost < best_cost * (1 - 1e-9):
                best, best_cost = fac, cost
        cuts = []
        for a in range(d):
            r = best[a]
            # equal cuts: measured on configs 3 and 4, a rank's time follows its pixel count far more closely than
            # the number of kernels that reach in from outside (a corner block 1.5x as wide ran 1.7x as long)
            widths = [1.0] * r
            scale = n[a] / sum(widths)
            edges, acc = [0], 0.0
            for i in range(r - 1):
                acc += widths[i] * scale
                e = int(round(acc / tile[a])) * tile[a] if n[a] >= 2 * r * tile[a] else int(round(acc))
                e = min(max(e, edges[-1] + 1), n[a] - (r - 1 - i))
                edges.append(e)
            edges.append(n[a])
            cuts.append(edges)
        self._block_grid = best
        blocks = []
        for idx in product(*[range(best[a]) for a in range(d)]):
            blocks.append(tuple((cuts[a][idx[a]], cuts[a][idx[a] + 1]) for a in range(d)))
        return blocks

    # ------------------------------------------------------------------------------------------
    # device state
    # ------------------------------------------------------------------------------------------
    def _init_device(self, dense_exec):
        dev, f32 = self.device, torch.float32
        d, Cc, K = self.dim_domain, self.image.shape[-1], self.start_pis
        L = lib()
        self._P = L.smoe_param_count(d, Cc)
        self._PK = L.smoe_packed_stride(d, Cc)
        self._T = d * (d + 1) // 2
        self._off = theta_offsets(d, Cc)
        lb3 = float(self.lower_bounds[3]) if self.quantize_pis else 0.0
        ub3 = float(self.upper_bounds[3]) if self.quantize_pis else 1.0
        bits3 = int(self.bit_depths[3]) if self.quantize_pis else 8
        qm2 = self.quantization_mode >= 2
        q_lb = (C.c_float * 5)(*([float(v) for v in self.lower_bounds] if qm2 else [0.0] * 5))
        q_ub = (C.c_float * 5)(*([float(v) for v in self.upper_bounds] if qm2 else [1.0] * 5))
        q_bits = (C.c_int32 * 5)(*([int(v) for v in self.bit_depths] if qm2 else [8] * 5))
        # mode 3: fake-quant ranges from the surviving kernels, computed on the device once per step
        self._qdyn = (torch.zeros((L.smoe_quant_ranges_bytes() + 3) // 4, dtype=torch.int32, device=dev)
                      if self.quantization_mode == 3 else None)
        self._cfg = Cfg(d, Cc, int(self.precision), float(self.margin), int(self.use_determinant),
                        int(self.train_inverse_cov), int(self.use_yuv), int(self.train_gammas),
                        int(self.only_y_gamma), int(self.quantize_pis), lb3, ub3, bits3,
                        int(self.quantization_mode) if qm2 else 0, q_lb, q_ub, q_bits, int(self.use_diff_center),
                        int(self.kernel_count_as_norm_l1), int(bool(self.radial_as)),
                        int(dense_exec),   # dense_exec: 0 cull+skip, 1 dense, 2 skip only
                        int(self.eps_bits))
        if self.eps_bits and int(dense_exec) != 0:
            raise ValueError("eps_bits (opt-in epsilon culling) needs dense_exec == 0")
        # variables
        A0 = np.asarray(self.A_init, dtype=np.float64)
        theta = np.zeros((K, self._P), dtype=np.float32)
        theta[:, 0:d] = 0.0 if self.use_diff_center else self.musX_init      # smoe.py:390-394
        self._mus_grid = (torch.from_numpy(np.ascontiguousarray(self.musX_init, dtype=np.float32)).to(dev)
                          if self.use_diff_center else None)
        if self.radial_as:          # one scalar per kernel on every diagonal entry, A_corr frozen at 0 (smoe.py:429-434)
            a0 = A0 if A0.ndim == 1 else A0[:, 0, 0]
            for l in range(d):
                theta[:, a_col(d, l, l)] = a0
        else:
            for l in range(d):
                for m in range(l + 1):
                    theta[:, a_col(d, l, m)] = A0[:, l, m]
        theta[:, self._off["pi"]] = self.pis_init
        theta[:, self._off["nu"]:self._off["nu"] + Cc] = self.nu_e_init
        theta[:, self._off["ga"]:] = np.asarray(self.gamma_e_init).reshape(K, d * Cc)
        self._theta = torch.from_numpy(theta).to(dev)
        self._theta_best = self._theta.clone()
        self._grads = torch.zeros_like(self._theta)
        self._adam_m = torch.zeros_like(self._theta)
        self._adam_v = torch.zeros_like(self._theta)
        self._group_owner = [None, None, None]
        # image block resident on this rank + coordinate axes (np.linspace -> float32 feed, smoe.py:545)
        blk = self._block
        self._local_slices = tuple(slice(lo, hi) for lo, hi in blk)
        self._local_shape = tuple(hi - lo for lo, hi in blk)
        # The resident buffers cover the block, plus -- for SSIM as the loss on a sharded model -- a ring of 10 pixels
        # around it (clipped to the image): windows that straddle a block border need the neighbours' pixels.
        ring = 10 if (self.ssim_opt and self._world > 1 and not self._emulated) else 0
        self._buf = tuple((max(lo - ring, 0), min(hi + ring, self.image.shape[a])) for a, (lo, hi) in enumerate(blk))
        self._buf_slices = tuple(slice(lo, hi) for lo, hi in self._buf)
        self._buf_shape = tuple(hi - lo for lo, hi in self._buf)
        self._blk_in_buf = tuple(slice(blk[a][0] - self._buf[a][0], blk[a][1] - self._buf[a][0]) for a in range(d))
        self._dims3 = tuple(self._buf_shape) + (1,) * (3 - d)
        self._d_image = torch.from_numpy(np.ascontiguousarray(self.image[self._buf_slices])).to(dev)
        self._d_image_u8 = None
        self._use_u8 = False                                 # set_image() fed 8-bit pixels: the loss stage reads them
        self._copy_stream = self._img_event = None           # set_image()'s host->device copy, overlapped with the forward
        self._img_pending = False
        self._d_loss_mask = None
        if self.loss_mask is not None:                       # per-pixel loss weights (smoe.py:550, 932, 1674-1677)
            lm = np.asarray(self.loss_mask, dtype=np.float32).reshape(self.image.shape[:-1])
            if (lm < 0).any():
                raise ValueError("loss_mask weights must be >= 0")
            self._d_loss_mask = torch.from_numpy(np.ascontiguousarray(lm[self._buf_slices])).to(dev)
        self._d_sample_w = None                              # per-call pixel selection of sampling_percentage < 100
        self.random_sampling_per_batch = None                # None = uniform (smoe.py:271-273)
        axes = [np.linspace(0, 1, self.image.shape[a]).astype(np.float32)[self._buf[a][0]:self._buf[a][1]] for a in range(d)]
        self._d_axes = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in axes]
        self._h_axes = axes
        npx = int(np.prod(self._buf_shape))
        self._res_peer = None
        if ring:
            # the neighbours read this buffer over NVLink: a dedicated, exportable allocation (smoe_peer_alloc)
            self._res_peer = _PeerBuffer(npx * Cc * 4)
            self._d_res = self._res_peer.as_tensor((npx, Cc), dev)
        else:
            self._d_res = torch.zeros((npx, Cc), dtype=f32, device=dev)
        self._d_res_pre = torch.zeros((npx, Cc), dtype=f32, device=dev)      # mixture output before clip (the forward's rbuf)
        self._d_argmax = torch.zeros((npx,), dtype=torch.int32, device=dev)
        # batches (smoe.py:1643: sliding_window order, first axis outermost)
        self._tile = choose_tile(d, self._local_shape[d - 1])
        self._batches = []
        if self._world > 1:
            rects = [(tuple(sl.start for sl in self._blk_in_buf), self._local_shape)]
        else:
            starts = [range(0, self.image.shape[a], self.batch_size_valued[a]) for a in range(d)]
            rects = [(org, self.batch_size_valued) for org in product(*starts)]
        max_tiles = 0
        ov = self.overlap if self._world == 1 else 0        # a sharded model is one batch: no window halo
        self._batch_npix, self._batch_phantom = [], []
        for org, ext in rects:
            b = Batch()
            clipped = False
            for a in range(3):
                b.dims[a] = self._dims3[a]
                # the window plus its overlap halo, clipped to the image (smoe.py:18-35 pads with zeros instead;
                # see _batch_phantom below)
                lo = max(org[a] - ov, 0) if a < d else 0
                hi = min(org[a] + ext[a] + ov, self._dims3[a]) if a < d else 1
                clipped |= a < d and (org[a] - ov < 0 or org[a] + ext[a] + ov > self._dims3[a])
                b.origin[a] = lo
                b.extent[a] = hi - lo
                b.tile[a] = self._tile[a]
            npix = int(np.prod(ext)) if self._world == 1 else self.num_pixel
            b.inv_count = 1.0 / npix
            b.halo = ov
            self._batches.append(b)
            self._batch_npix.append(npix)
            # The reference zero-pads the JOINT domain, coordinates included (smoe.py:20, 28): a window at the image
            # border is fed `overlap` rows of phantom pixels that all sit at coordinate (0,..,0).  They are cropped
            # before the loss and can only add kernels to the window's influence list (smoe.py:829); one extra
            # 1-pixel forward at the image origin reproduces that (pixel 0 IS at coordinate 0).
            self._batch_phantom.append(ov > 0 and clipped)
            max_tiles = max(max_tiles, L.smoe_num_tiles(C.byref(b)))
        self._phantom = None
        if any(self._batch_phantom):
            pb = Batch()
            for a in range(3):
                pb.dims[a], pb.origin[a], pb.extent[a], pb.tile[a] = self._dims3[a], 0, 1, self._tile[a]
            pb.inv_count, pb.halo = 1.0, 0
            self._phantom = (pb, torch.full((1,), _ffi.PIXEL_HALO, dtype=f32, device=dev))
        self._ssim_ws = None
        if self.ssim_opt:
            nbytes = max(L.smoe_ssim_loss_workspace_bytes(C.byref(self._cfg), C.byref(b)) for b in self._batches)
            self._ssim_ws = torch.zeros((nbytes + 7) // 8, dtype=torch.float64, device=dev)
        nb = len(self._batches)
        self._max_tiles = max_tiles
        self._klist = torch.ones((nb, K), dtype=torch.uint8, device=dev)
        self._packed = torch.zeros((K, self._PK), dtype=f32, device=dev)
        self._indices = torch.zeros((K,), dtype=torch.int32, device=dev)
        self._pos = torch.zeros((K,), dtype=torch.int32, device=dev)
        self._perm = torch.zeros((K,), dtype=torch.int32, device=dev)
        self._keys = torch.zeros((K,), dtype=torch.int64, device=dev)
        self._key_scale = key_scale(self.image.shape[:d])
        self._refresh_perm()
        # one block per batch [scalars (NSCAL) | counts (4 x int32) | regulariser sums (2) | pad]: a single
        # device->host copy per run_batched call brings back everything the host needs
        self._stats = torch.zeros((nb, _ffi.STATS_STRIDE), dtype=f32, device=dev)
        self._scalars = self._stats[:, :_ffi.NSCAL]
        self._counts = self._stats.view(torch.int32)[:, _ffi.NSCAL:_ffi.NSCAL + 4]
        self._regsums = self._stats[:, _ffi.NSCAL + 4:_ffi.NSCAL + 6]
        self._infl = torch.zeros((K,), dtype=torch.uint8, device=dev)
        self._pix = torch.zeros((max_tiles * L.smoe_pix_stride(d, Cc, C.byref(self._batches[0])),), dtype=f32, device=dev)
        # per batch: the forward's tile minima of log2 S (culling threshold of the backward; with eps_bits also the
        # PREVIOUS pass's bound for the forward's own sweep A, -inf = "no bound yet, sweep exactly")
        self._tile_qmin = torch.full((nb, max_tiles), -float("inf"), dtype=f32, device=dev)
        self._pair_counts = None        # uint64[8] executed-pair counters, enable_pair_counts()
        self._chunk_bounds = torch.zeros(((K + 127) // 128, 12), dtype=f32, device=dev)
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        self._partials = torch.zeros((8 * max(int(L.smoe_loss_partials(C.byref(b))) for b in self._batches),),
                                     dtype=f32, device=dev)
        self._ticket = torch.zeros((4,), dtype=torch.int32, device=dev)
        self._pack_ws = torch.zeros((L.smoe_pack_workspace_bytes(K) + 15) // 4, dtype=torch.int32, device=dev)
        # Pixel splits of the backward (split s owns tiles s, s+NS, ...): sized for the kernel groups that will have
        # work -- a rank's block is reached by a fraction of the kernels only, and the groups that do not reach it
        # leave after one load -- so that the (group, split) grid still fills the GPU a few waves deep.
        reach = self._reach_px()
        frac = float(np.prod([min(1.0, (self._local_shape[a] + 2 * reach[a]) / (self.image.shape[a] + 2 * reach[a]))
                              for a in range(d)]))
        self._splits = backward_splits(int(K * frac), self._batches)
        self._plan = torch.zeros((max(L.smoe_backward_plan_bytes(K, C.byref(b)) for b in self._batches) + 3) // 4,
                                 dtype=torch.int32, device=dev)
        self._raw_part = None           # allocated on the first training pass
        self._peers = None
        self._halo = self._ssim_region = None
        if self._world > 1 and not self._emulated:
            self._open_peer_windows()
            if self._res_peer is not None:
                self._init_halo()
        self._host_stats = torch.zeros((nb, _ffi.STATS_STRIDE), dtype=f32).pin_memory()
        self._host_f32 = self._host_stats.numpy()                       # views of the pinned block
        self._host_i32 = self._host_stats.view(torch.int32).numpy()
        self._alpha_host = torch.zeros((4,), dtype=f32).pin_memory()
        self._alpha_np = self._alpha_host.numpy()
        self._alpha_dev = torch.zeros((4,), dtype=f32, device=dev)
        self._graphs = {}
        # one CUDA graph per training-step signature, on one GPU and sharded alike (the exchange is stream-ordered
        # kernels over peer memory, DESIGN.md section 5)
        self.use_cuda_graphs = True
        self.gpu_launches = 0

    def _open_peer_windows(self):
        """Allocate this rank's exchange window, swap cudaIpc handles with the other ranks of the node (host
        plumbing: torch.distributed) and map theirs (csrc/exchange.cuh)."""
        L = lib()
        nbytes = L.smoe_xchg_window_bytes(self.start_pis, self._P)
        own = C.c_void_p()
        check(L.smoe_peer_alloc(C.c_size_t(nbytes), C.byref(own)), "smoe_peer_alloc")
        handle = (C.c_ubyte * 64)()
        check(L.smoe_peer_export(own, handle), "smoe_peer_export")
        handles = [None] * self._world
        torch.distributed.all_gather_object(handles, bytes(handle), group=self._pg)
        self._peers = Peers()
        self._peers.world, self._peers.rank = self._world, self._rank
        self._peer_own = own
        for r in range(self._world):
            if r == self._rank:
                self._peers.win[r] = own.value
            else:
                mapped = C.c_void_p()
                buf = (C.c_ubyte * 64).from_buffer_copy(handles[r])
                check(L.smoe_peer_open(buf, C.byref(mapped)), "smoe_peer_open")
                self._peers.win[r] = mapped.value
        torch.cuda.synchronize()
        torch.distributed.barrier(group=self._pg)       # every window exists and is zeroed before anyone signals

    def _init_halo(self):
        """Geometry and peer mappings of the halo pull (smoe_halo_pull) of a sharded SSIM loss."""
        d, Cc = self.dim_domain, self.image.shape[-1]
        handles = [None] * self._world
        torch.distributed.all_gather_object(handles, self._res_peer.handle(), group=self._pg)
        hm = _ffi.HaloMap()
        hm.world, hm.rank, hm.d, hm.C = self._world, self._rank, d, Cc
        for r, blk in enumerate(self._blocks):
            for a in range(3):
                lo, hi = blk[a] if a < d else (0, 1)
                blo = max(lo - 10, 0) if a < d else 0
                bhi = min(hi + 10, self.image.shape[a]) if a < d else 1
                hm.blk_lo[r][a], hm.blk_hi[r][a] = lo, hi
                hm.buf_lo[r][a], hm.buf_dims[r][a] = blo, bhi - blo
            hm.res[r] = self._res_peer.ptr.value if r == self._rank else self._res_peer.open_peer(handles[r])
        self._halo = hm
        reg = _ffi.SsimRegion()
        for a in range(3):
            reg.lo[a], reg.n[a] = 0, self._dims3[a]           # windows centred on every position of the resident buffer
        reg.inv_count = 1.0 / self.num_pixel
        self._ssim_region = reg
        torch.cuda.synchronize()
        torch.distributed.barrier(group=self._pg)

    def close(self):
        """Unmap / free the peer windows of a sharded model (collective: every rank calls it)."""
        if getattr(self, "_peers", None) is None:
            return
        L = lib()
        torch.cuda.synchronize()
        torch.distributed.barrier(group=self._pg)
        for r in range(self._world):
            if r != self._rank:
                L.smoe_peer_close(C.c_void_p(self._peers.win[r]))
        torch.distributed.barrier(group=self._pg)
        L.smoe_peer_free(self._peer_own)
        if self._res_peer is not None:
            self._d_res = None
            self._res_peer.close()
        self._peers = None

    def exchange_status(self):
        """(epoch, error) of this rank's exchange window; error != 0 means a peer never arrived at a barrier."""
        st = (C.c_int32 * 2)()
        check(lib().smoe_xchg_status(C.byref(self._peers), st), "smoe_xchg_status")
        return int(st[0]), int(st[1])

    def enable_pair_counts(self, on=True):
        """Executed-(pixel, kernel)-pair counters of the two sweep kernels (bench / roofline diagnostics; a separate
        kernel instantiation, the default path carries none)."""
        self._pair_counts = torch.zeros((8,), dtype=torch.int64, device=self.device) if on else None
        self._graphs = {}

    def set_image(self, pixels):
        """Feed this rank's block of the target for the following passes (the end-to-end path: a frame arrives in
        host memory every step).  `pixels`: uint8 (as an image file holds them; /255 as utils.py:126-128 happens in
        the forward kernel's epilogue) or float32 in [0,1], shape of the local block, ideally pinned; the copy is
        asynchronous on the current stream."""
        t = pixels if isinstance(pixels, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(pixels))
        if t.shape != self._d_image.shape:
            raise ValueError(f"expected the local block {tuple(self._d_image.shape)}, got {tuple(t.shape)}")
        if t.dtype == torch.uint8:
            if self.ssim_opt:
                raise NotImplementedError("8-bit feed with ssim_opt: feed float32 pixels")
            if self._d_image_u8 is None:
                self._d_image_u8 = torch.empty(self._d_image.shape, dtype=torch.uint8, device=self.device)
            dst, self._use_u8 = self._d_image_u8, True
        elif t.dtype == torch.float32:
            dst, self._use_u8 = self._d_image, False
        else:
            raise ValueError("set_image takes uint8 or float32 pixels")
        if t.is_cuda or not t.is_contiguous():
            raise ValueError("set_image takes a contiguous host tensor (pinned for an asynchronous copy)")
        # The copy runs on its own stream: the next pass's pack and forward sweeps need no target pixels and overlap
        # it; only the loss stage waits for the event (run_batched).  smoe_feed orders it after earlier readers.
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=self.device)
            self._img_event = torch.cuda.Event()
            self._order_event = torch.cuda.Event()
            for ev in (self._img_event, self._order_event):      # torch creates the CUDA event lazily: force it
                ev.record()
            self._feed_handles = (C.c_void_p(self._copy_stream.cuda_stream), C.c_void_p(self._order_event.cuda_event),
                                  C.c_void_p(self._img_event.cuda_event))
        self._feed_src = t                                        # keep the host buffer alive until the copy is consumed
        cs, oe, de = self._feed_handles
        check(lib().smoe_feed(C.c_void_p(dst.data_ptr()), C.c_void_p(t.data_ptr()), C.c_size_t(t.numel() * t.element_size()),
                              stream_ptr(), cs, oe, de), "smoe_feed")
        self._img_pending = True
        self.valid = self.qvalid = False

    def _refresh_perm(self):
        """Spatially coherent packing order (Hilbert-curve order of the current centres, isotropic in pixels): smoe_pack writes the compute
        records in this order, so a forward chunk (128 records) and a backward CTA (64 records) hold neighbours and
        the tile culling bites.  Purely a work-assignment choice -- any order gives the same per-kernel results.
        Keys and sort run on the device (stable sort: ties keep ascending index)."""
        check(lib().smoe_spatial_keys(ptr(self._theta), self.start_pis, self.dim_domain, self._P, ptr(self._mus_grid),
                                      self._key_scale, ptr(self._keys), stream_ptr()), "smoe_spatial_keys")
        # in place: captured CUDA graphs hold the buffer's address
        self._perm.copy_(torch.sort(self._keys, stable=True).indices.to(torch.int32))

    def get_active_indices(self, batch=0):
        """The reference's `indices` of the last pass over `batch` (smoe.py:741-742): ascending original indices of
        the kernels with pi > 0 that are on the batch's kernel list."""
        K = int(self._counts[batch, 0].item())
        return np.sort(self._indices[:K].cpu().numpy())

    def _enable_res_pre(self):
        """The mixture output before clip / output quantisation is always kept (it is what smoe_forward hands to
        smoe_loss; SURVEY.md decision D4 compares reconstructions pre-quantisation).  Kept for callers of round 1."""
        return None

    def get_pre_clip_reconstruction(self):
        self._enable_res_pre()
        self.run_batched(train=False, update_reconstruction=True)
        return self._d_res_pre.reshape(self._buf_shape + (self.image.shape[-1],))[self._blk_in_buf].cpu().numpy()

    # kernel_list_per_batch is exposed as the reference's list of NumPy bool arrays
    @property
    def kernel_list_per_batch(self):
        return [row.astype(bool) for row in self._klist.cpu().numpy()]

    @kernel_list_per_batch.setter
    def kernel_list_per_batch(self, value):
        arr = np.stack([np.asarray(v, dtype=np.uint8) for v in value])
        self._klist.copy_(torch.from_numpy(arr).to(self.device))

    # ------------------------------------------------------------------------------------------
    # optimizers (smoe.py:1079-1204)
    # ------------------------------------------------------------------------------------------
    def set_optimizer(self, optimizer1, optimizer2=None, optimizer3=None, optimizer4=None, optimizer5=None,
                      grad_clip_value_abs=None):
        new = [optimizer1, optimizer2 or optimizer1, optimizer3 or optimizer1]
        self.optimizer1, self.optimizer2, self.optimizer3 = new
        self.grad_clip_value_abs = grad_clip_value_abs
        o = self._off
        cols = {0: list(range(0, o["A"])) + list(range(o["nu"], self._P)), 1: [o["pi"]], 2: list(range(o["A"], o["pi"]))}
        for g in range(3):
            if self._group_owner[g] is not new[g]:          # a new optimizer object gets fresh slots
                idx = torch.tensor(cols[g], device=self.device)
                self._adam_m[:, idx] = 0
                self._adam_v[:, idx] = 0
                self._group_owner[g] = new[g]

    def _adam_prepare(self):
        """Advance the optimizers' beta powers (one apply_gradients each) and stage TF's bias-corrected
        step sizes in pinned host memory; the launch (eager or a replayed CUDA graph) copies them to the
        device, so a captured step never bakes a step count into its kernel arguments."""
        opts = [self.optimizer1, self.optimizer2, self.optimizer3]
        trainable = [True, self.train_pis, True]
        # One apply_gradients per GROUP (smoe.py:1173-1184).  When set_optimizer(opt) aliases one object to all three
        # groups (smoe.py:1080-1090), TF builds three apply_gradients ops on it and each multiplies the shared
        # beta1_power / beta2_power once per step -- the powers advance three times per step and the order of the
        # three ops inside one session.run is unspecified; here they run in group order (1, 2, 3), which is one of
        # TF's valid serialisations (the test-side restatement pins the same order).
        for g, (opt, tr) in enumerate(zip(opts, trainable)):
            on = tr and not opt._lr == 0
            self._alpha_np[g] = opt._step_alpha() if on else 0.0

    def _adam_launch(self, fuse_klist=False):
        hp = Adam()
        for g, opt in enumerate([self.optimizer1, self.optimizer2, self.optimizer3]):
            hp.alpha[g] = 0.0
            hp.beta1[g], hp.beta2[g], hp.epsilon[g] = opt._beta1, opt._beta2, opt._epsilon
        hp.grad_clip = float(self.grad_clip_value_abs) if self.grad_clip_value_abs is not None else 0.0
        hp.train_musx, hp.train_gammas = int(self.train_musx), int(self.train_gammas)
        self._alpha_dev.copy_(self._alpha_host, non_blocking=True)
        check(lib().smoe_adam_step(C.byref(self._cfg), C.byref(hp), ptr(self._alpha_dev), ptr(self._theta),
                                   ptr(self._grads), ptr(self._adam_m), ptr(self._adam_v), self.start_pis,
                                   ptr(self._infl) if fuse_klist else ptr(None),
                                   ptr(self._klist[0]) if fuse_klist else ptr(None), stream_ptr()), "smoe_adam_step")
        self.gpu_launches += 1

    # ------------------------------------------------------------------------------------------
    # the batched executor (smoe.py:1606-1793)
    # ------------------------------------------------------------------------------------------
    def run_batched(self, pis_l1=0, u_l1=0, sv_l1_sub_l2=0, train=True, update_reconstruction=False,
                    with_quantized_params=False, sampling_percentage=100, with_inc=False, train_inc=False,
                    thr_sv=None, use_loss_mask=False):
        if with_inc or train_inc:
            raise NotImplementedError("inc paths are outside the hot path (D1)")
        if train:
            assert self.optimizer1 is not None, "no optimizer found, you have to specify one!"
        sampling = train and not self.ssim_opt and sampling_percentage < 100          # smoe.py:1664
        if use_loss_mask and self._d_loss_mask is None:
            raise ValueError("use_loss_mask needs the loss_mask constructor argument")
        if sampling and use_loss_mask:
            raise ValueError("loss_mask and sampling_percentage < 100 cannot be combined (the reference feeds a "
                             "full-batch mask against the sampled pixels, smoe.py:1666-1677)")
        if self.overlap > 0 and (sampling or use_loss_mask):
            # smoe_test.py:322-325: sampling is "only working if ... batch overlap equal 0"; the mask is sliced
            # with the un-padded window coordinates (smoe.py:1674-1676)
            raise NotImplementedError("sampling_percentage < 100 / use_loss_mask with overlap_of_batches > 0")
        lossw, batches = (self._d_loss_mask if use_loss_mask else None), self._batches
        if sampling:
            lossw, batches = self._draw_samples(sampling_percentage)
        self.valid = False
        if with_quantized_params:
            self.qvalid = False
        K, P = self.start_pis, self._P
        if train and self._raw_part is None:
            self._raw_part = torch.zeros((self._splits * K * P,), dtype=torch.float32, device=self.device)
        if train:
            self._adam_prepare()
        # A plain training step (the hot loop of Smoe.train, smoe.py:1527) is captured once into a CUDA
        # graph and replayed: one graph launch + one stream sync per iteration instead of ~25 launches.
        graphable = (self.use_cuda_graphs and train and not update_reconstruction and not with_quantized_params
                     and not sampling)
        replayed = False
        if graphable:
            key = (float(pis_l1), float(u_l1), self.grad_clip_value_abs, id(self.optimizer1), id(self.optimizer2),
                   id(self.optimizer3), self.optimizer1._lr, self.optimizer2._lr, self.optimizer3._lr,
                   self._use_u8, bool(use_loss_mask))
            state = self._graphs.get(key)
            if state is None:
                self._graphs[key] = "warm"              # first step with this signature runs eagerly
            else:
                if state == "warm":
                    l0 = self.gpu_launches
                    if self._img_pending:               # an event of another stream cannot be awaited inside a capture
                        torch.cuda.current_stream().wait_event(self._img_event)
                        self._img_pending = False
                    torch.cuda.synchronize()
                    try:
                        # two graphs, split where the target pixels are first needed (before the loss stage): a
                        # pending set_image() copy is awaited BETWEEN them, so it overlaps pack + forward
                        graphs = []
                        for phase in (("pre", "post") if len(self._batches) == 1 else ()):
                            g = torch.cuda.CUDAGraph()
                            with torch.cuda.graph(g):
                                self._enqueue(pis_l1, u_l1, True, False, False, lossw=lossw, phase=phase)
                            graphs.append(g)
                        gall = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(gall):
                            self._enqueue(pis_l1, u_l1, True, False, False, lossw=lossw)
                        state = (gall, graphs, (self.gpu_launches - l0) // (2 if graphs else 1))
                    except Exception as exc:
                        # Loud by default: a silent eager fallback would hide a 2x slower step.  A sharded model
                        # cannot fall back at all: its peers would replay a graph while this rank runs eagerly --
                        # same kernels, so still correct, but the failure must be seen.
                        if os.environ.get("SMOE_ALLOW_EAGER", "0") != "1":
                            raise RuntimeError(f"smoe_b200: CUDA graph capture of the training step failed ({exc}); "
                                               "set SMOE_ALLOW_EAGER=1 to run the step eagerly instead") from exc
                        warnings.warn(f"smoe_b200: CUDA graph capture failed ({exc}); running eagerly")
                        self.use_cuda_graphs = False
                        torch.cuda.synchronize()
                        state = None
                    self.gpu_launches = l0
                    if state is not None:
                        self._graphs[key] = state
                if state is not None:
                    if self._img_pending and state[1]:
                        state[1][0].replay()
                        torch.cuda.current_stream().wait_event(self._img_event)
                        self._img_pending = False
                        state[1][1].replay()
                    else:
                        if self._img_pending:
                            torch.cuda.current_stream().wait_event(self._img_event)
                            self._img_pending = False
                        state[0].replay()
                    self.gpu_launches += state[2]
                    replayed = True
        if not replayed:
            self._enqueue(pis_l1, u_l1, train, update_reconstruction, with_quantized_params,
                          lossw=lossw, batches=batches)
        torch.cuda.current_stream().synchronize()
        # plain Python lists: this runs after every step, and NumPy temporaries would cost more than the arithmetic
        h = self._host_f32.tolist()
        hi = self._host_i32.tolist()
        for row, irow in zip(h, hi):
            row[_ffi.NSCAL:_ffi.NSCAL + 4] = irow[_ffi.NSCAL:_ffi.NSCAL + 4]
        norm = float(self.start_pis)
        Cc = self.image.shape[-1]
        loss_val = mse_val = 0.0
        num_pi = -1
        for ii, b in enumerate(batches):
            inv_n = float(b.inv_count)
            if self.ssim_opt:                              # smoe.py:1006-1010
                per = [h[ii][8 + c] / self._batch_npix[ii] for c in range(Cc)]
                ssim = (sum(p * wgt for p, wgt in zip(per, (6, 1, 1))) / 8 if Cc == 3 else per[0]) if self.use_yuv \
                    else sum(per) / Cc
                lp = 1 - ssim
            elif self.use_yuv:                             # smoe.py:933-935
                lp = 6 / 8 * h[ii][0] * inv_n + 1 / 8 * sum(h[ii][c] * inv_n for c in range(1, Cc))
            else:
                lp = sum(h[ii][c] for c in range(Cc)) * inv_n / Cc
            l1n = max(h[ii][_ffi.NSCAL + 1], 1.0) if self.kernel_count_as_norm_l1 else norm      # smoe.py:1022-1025
            loss_b = lp + pis_l1 * h[ii][_ffi.NSCAL + 4] / l1n + u_l1 * h[ii][_ffi.NSCAL + 5]
            mse_b = h[ii][4] * inv_n / Cc * ((2 ** self.precision) ** 2)
            if h[ii][5] > 0:
                loss_b = float("nan")
            frac = 1.0 if self._world > 1 else self._batch_npix[ii] / self.num_pixel
            loss_val += loss_b * frac                       # smoe.py:1758-1759
            mse_val += mse_b * frac
            num_pi = int(h[ii][_ffi.NSCAL + 1])
        self._last_nonpos = int(sum(row[_ffi.NSCAL + 2] for row in h))
        if self._last_nonpos > 0 and not getattr(self, "_warned_nonpos", False):
            # pi * prod(diag A) < 0 with use_determinant: the reference gives such a kernel a NEGATIVE weight n_w
            # (smoe.py:809-820); the log-domain kernels evaluate it with |coef| -- say so once
            warnings.warn(f"smoe_b200: {self._last_nonpos} active kernel(s) have pi * prod(diag A) < 0; they are "
                          "evaluated with the absolute value of that weight (the reference would subtract them)")
            self._warned_nonpos = True
        if update_reconstruction:
            rec, amax = self._gather_reconstruction()
            self._update_sampling_probabilities(rec)
            if with_quantized_params:
                self.qreconstruction_image, self.qweight_matrix_argmax, self.qvalid = rec, amax, True
            else:
                self.reconstruction_image, self.weight_matrix_argmax, self.valid = rec, amax, True
        return loss_val, mse_val, num_pi, 0

    def _draw_samples(self, sampling_percentage):
        """Random pixel sub-sampling of a training pass (smoe.py:1664-1667): per batch, round(N_b * pct / 100)
        pixels drawn without replacement by np.random.choice (the global NumPy generator, as the reference) with
        the error-proportional probabilities of the last reconstruction pass (smoe.py:906-907, 1768-1769).
        Returns the per-pixel selection (1 = fed, SMOE_PIXEL_ABSENT = not fed) and batches whose loss means run
        over the drawn pixels.  A sharded model is the one-batch model of the whole image: every rank draws the SAME
        global sample (same generator state and probabilities on every rank -- seed NumPy identically) and feeds the
        drawn pixels of its own block."""
        d = self.dim_domain
        if self._d_sample_w is None:
            self._d_sample_w = torch.empty(self._buf_shape, dtype=torch.float32, device=self.device)
        w = np.full(self._buf_shape, _ffi.PIXEL_ABSENT, dtype=np.float32)
        batches = []
        self.last_samples = []
        if self._world > 1:
            n = self.num_pixel
            num_samples = int(np.uint32(np.round(n * sampling_percentage / 100)))
            p = self.random_sampling_per_batch[0] if self.random_sampling_per_batch is not None else None
            p = np.ones((n,), dtype=np.float32) / n if p is None else np.asarray(p)
            samples = np.random.choice(n, (num_samples,), replace=False, p=p)
            self.last_samples.append(samples)
            sel = np.full((n,), _ffi.PIXEL_ABSENT, dtype=np.float32)
            sel[samples] = 1.0
            w[self._blk_in_buf] = sel.reshape(self.image.shape[:d])[self._local_slices]
            nb = Batch.from_buffer_copy(self._batches[0])
            nb.inv_count = 1.0 / max(num_samples, 1)
            batches.append(nb)
            self._d_sample_w.copy_(torch.from_numpy(w))
            return self._d_sample_w, batches
        for ii, ((org, ext), b) in enumerate(zip(self._batch_rects(), self._batches)):
            n = int(np.prod(ext))
            num_samples = int(np.uint32(np.round(n * sampling_percentage / 100)))
            p = None if self.random_sampling_per_batch is None else self.random_sampling_per_batch[ii].cpu().numpy()
            if p is None:
                p = np.ones((n,), dtype=np.float32) / n
            samples = np.random.choice(n, (num_samples,), replace=False, p=p)
            self.last_samples.append(samples)
            sel = np.full((n,), _ffi.PIXEL_ABSENT, dtype=np.float32)
            sel[samples] = 1.0
            w[tuple(slice(o, o + e) for o, e in zip(org, ext))] = sel.reshape(ext)
            nb = Batch.from_buffer_copy(b)
            nb.inv_count = 1.0 / max(num_samples, 1)
            batches.append(nb)
        self._d_sample_w.copy_(torch.from_numpy(w))
        return self._d_sample_w, batches

    def _update_sampling_probabilities(self, rec=None):
        """sampl_prob = err_map / sum(err_map) per batch, err_map = mean_c (resq - target)^2 (smoe.py:906-907),
        kept on the device; replaces `random_sampling_per_batch[ii] = results[-1]` (smoe.py:1768-1769).  Sharded: from
        the gathered reconstruction, on the host (identical on every rank)."""
        if self.overlap > 0 and self._world == 1:
            return
        d, Cc = self.dim_domain, self.image.shape[-1]
        if self._world > 1:
            if rec is None or self._emulated:
                return
            err = ((np.asarray(rec, np.float32) - self.image) ** 2).mean(axis=-1).reshape(-1)
            self.random_sampling_per_batch = [err / err.sum()]
            return
        if self._use_u8:
            torch.div(self._d_image_u8.to(torch.float32), 255.0, out=self._d_image)
        err = ((self._d_res.reshape(self._local_shape + (Cc,)) - self._d_image) ** 2).mean(dim=-1)
        probs = []
        for org, ext in self._batch_rects():
            e = err[tuple(slice(o, o + x) for o, x in zip(org, ext))].reshape(-1)
            probs.append(e / e.sum())
        self.random_sampling_per_batch = probs

    def _enqueue(self, pis_l1, u_l1, train, update_reconstruction, with_quantized_params, lossw=None, batches=None,
                 phase="all"):
        """Every launch of one run_batched call, asynchronous on the current stream (capturable, also sharded:
        the exchange is stream-ordered kernels over peer memory).  phase "pre" = everything that needs no target
        pixels (staging, forward), "post" = the rest (loss stage, backward, exchange, finalize, Adam); only one-batch
        passes are split, so that a pending set_image() copy can be awaited between the halves."""
        L, st = lib(), stream_ptr()
        K = self.start_pis
        batches = self._batches if batches is None else batches
        sharded = self._world > 1 and not self._emulated
        pc = ptr(self._pair_counts)
        pre, post = phase in ("all", "pre"), phase in ("all", "post")
        assert phase == "all" or len(batches) == 1
        # (the start-of-pass clears -- gradient accumulators, scalar blocks, influence flags -- ride in smoe_pack)
        fed = with_quantized_params and update_reconstruction
        if fed:
            rp = {k: torch.as_tensor(np.ascontiguousarray(np.asarray(v, dtype=np.float32)), device=self.device)
                  for k, v in self.rparams.items()}
            Kf = int(rp["pis"].shape[0])
            if Kf > K:
                raise ValueError("more fed kernels than model kernels")
            # the fed rows in Hilbert order of their centres, like the variables (device keys + device sort)
            fkeys = torch.empty((Kf,), dtype=torch.int64, device=self.device)
            check(L.smoe_spatial_keys(ptr(rp["musX"]), Kf, self.dim_domain, self.dim_domain, ptr(None), self._key_scale,
                                      ptr(fkeys), st), "smoe_spatial_keys")
            forder = torch.sort(fkeys, stable=True).indices.to(torch.int32)
        norm = float(self.start_pis)
        if pre and self._qdyn is not None and not fed:
            check(L.smoe_quant_ranges(C.byref(self._cfg), ptr(self._theta), K, int(self.train_musx), ptr(self._qdyn), st),
                  "smoe_quant_ranges")
            self.gpu_launches += 2
        ax2 = ptr(self._d_axes[2]) if self.dim_domain == 3 else ptr(None)
        for ii, b in enumerate(batches):
            counts, regs, scal = self._counts[ii], self._regsums[ii], self._scalars[ii]
            tq = self._tile_qmin[ii]
            if pre:
                if fed:
                    check(L.smoe_pack_fed(C.byref(self._cfg), ptr(rp["A"]), ptr(rp["musX"]), ptr(rp["nu_e"]),
                                          ptr(rp["gamma_e"]), ptr(rp["pis"]), ptr(forder), Kf, ptr(self._packed),
                                          ptr(self._indices), ptr(counts), ptr(self._chunk_bounds), ptr(scal),
                                          ptr(self._infl), K, st), "smoe_pack_fed")
                    regs.zero_()
                    self.gpu_launches += 3
                else:
                    check(L.smoe_pack(C.byref(self._cfg), ptr(self._theta), ptr(self._mus_grid), ptr(self._qdyn),
                                      ptr(self._klist[ii]), ptr(self._perm), K, ptr(self._packed),
                                      ptr(self._indices), ptr(self._pos), ptr(counts), ptr(regs), ptr(self._chunk_bounds),
                                      ptr(self._pack_ws), ptr(self._grads) if (train and ii == 0) else ptr(None),
                                      ptr(scal), ptr(self._infl), st), "smoe_pack")
                    self.gpu_launches += 3
                check(L.smoe_forward(C.byref(self._cfg), C.byref(b), ptr(self._packed), ptr(self._indices), ptr(counts),
                                     ptr(self._chunk_bounds), K, ptr(lossw), ptr(self._d_axes[0]), ptr(self._d_axes[1]),
                                     ax2, ptr(self._d_res_pre), ptr(self._d_argmax) if update_reconstruction else ptr(None),
                                     ptr(self._infl), ptr(self._pix) if train else ptr(None), ptr(tq), pc, st),
                      "smoe_forward")
                self.gpu_launches += 1
                if self._batch_phantom[ii]:
                    pb, halo1 = self._phantom
                    check(L.smoe_forward(C.byref(self._cfg), C.byref(pb), ptr(self._packed), ptr(self._indices),
                                         ptr(counts), ptr(self._chunk_bounds), K, ptr(halo1), ptr(self._d_axes[0]),
                                         ptr(self._d_axes[1]), ax2, ptr(self._d_res_pre), ptr(None), ptr(self._infl),
                                         ptr(None), ptr(None), ptr(None), st), "smoe_forward (phantom)")
                    self.gpu_launches += 1
            if not post:
                continue
            if phase == "all" and self._img_pending:      # eager pass right after set_image(): the loss needs the pixels
                torch.cuda.current_stream().wait_event(self._img_event)
                self._img_pending = False
            check(L.smoe_loss(C.byref(self._cfg), C.byref(b), ptr(self._d_res_pre),
                              ptr(None) if self._use_u8 else ptr(self._d_image),
                              ptr(self._d_image_u8) if self._use_u8 else ptr(None), ptr(lossw),
                              # the quantised reconstruction itself is only needed by callers that read it
                              ptr(self._d_res) if (update_reconstruction or self.ssim_opt or not train) else ptr(None),
                              ptr(self._pix) if train else ptr(None), ptr(scal), ptr(self._partials), ptr(self._ticket),
                              st), "smoe_loss")
            self.gpu_launches += 1
            if self.ssim_opt:
                if self._halo is not None:      # sharded: the ring of neighbour pixels around the block, over NVLink
                    check(L.smoe_halo_pull(C.byref(self._peers), C.byref(self._halo), st), "smoe_halo_pull")
                    self.gpu_launches += 1
                check(L.smoe_ssim_loss(C.byref(self._cfg), C.byref(b),
                                       C.byref(self._ssim_region) if self._ssim_region is not None else ptr(None),
                                       ptr(self._d_res), ptr(self._d_image),
                                       ptr(self._d_res_pre), ptr(self._pix) if train else ptr(None), ptr(scal),
                                       ptr(self._ssim_ws), st), "smoe_ssim_loss")
                self.gpu_launches += 2 * self.dim_domain + 2 if train else self.dim_domain + 1
            if train:
                check(L.smoe_backward(C.byref(self._cfg), C.byref(b), ptr(self._packed), ptr(counts), K,
                                      ptr(self._pix), ptr(tq), ptr(self._d_axes[0]), ptr(self._d_axes[1]), ax2,
                                      self._splits, ptr(self._raw_part), ptr(self._plan), pc, st), "smoe_backward")
                self.gpu_launches += 2
            if sharded:
                # the one exchange step (SURVEY.md 8e): publish this rank's sums, then the consumer sums the R
                # windows over NVLink in rank order -- fused into the gradient finalisation on a training pass
                check(L.smoe_xchg_publish(C.byref(self._cfg), C.byref(self._peers), ptr(counts), K, self._splits,
                                          ptr(self._raw_part) if train else ptr(None),
                                          ptr(self._plan) if train else ptr(None), ptr(scal), ptr(self._infl), st),
                      "smoe_xchg_publish")
                self.gpu_launches += 1
                if train:
                    check(L.smoe_grad_finalize_peers(C.byref(self._cfg), C.byref(self._peers), K, ptr(self._theta),
                                                     ptr(self._qdyn), ptr(self._indices), ptr(counts),
                                                     C.c_float(float(pis_l1)), C.c_float(norm), C.c_float(float(u_l1)),
                                                     ptr(self._grads), ptr(scal), ptr(self._infl), st),
                          "smoe_grad_finalize_peers")
                else:
                    check(L.smoe_xchg_reduce_tail(C.byref(self._cfg), C.byref(self._peers), K, ptr(scal),
                                                  ptr(self._infl), st), "smoe_xchg_reduce_tail")
                self.gpu_launches += 1
            elif train:
                check(L.smoe_grad_finalize(C.byref(self._cfg), ptr(self._raw_part), self._splits, ptr(self._plan), K,
                                           ptr(self._theta),
                                           ptr(self._qdyn), ptr(self._indices), ptr(counts), C.c_float(float(pis_l1)),
                                           C.c_float(norm), C.c_float(float(u_l1)), ptr(self._grads), st),
                      "smoe_grad_finalize")
                self.gpu_launches += 1
            # kernel_list <- influential kernels (smoe.py:1763-1766); a one-batch training pass does it inside the Adam launch
            if not with_quantized_params and not (train and len(batches) == 1):
                check(L.smoe_update_kernel_list(ptr(self._infl), ptr(self._klist[ii]), K, st), "smoe_update_kernel_list")
                self.gpu_launches += 1
        if not post:
            return
        if train and self._qdyn is not None:             # clipped gradients of the plain groups -> extreme elements
            check(L.smoe_quant_route(C.byref(self._cfg), ptr(self._theta), ptr(self._qdyn), K, ptr(self._grads), st),
                  "smoe_quant_route")
            self.gpu_launches += 3
        if train:
            self._adam_launch(fuse_klist=len(batches) == 1 and not with_quantized_params)
        # one small device->host read per call: scalars, counts, regulariser sums
        self._host_stats.copy_(self._stats, non_blocking=True)

    def _gather_reconstruction(self):
        Cc = self.image.shape[-1]
        d = self.dim_domain
        res = self._d_res.reshape(self._buf_shape + (Cc,))[self._blk_in_buf]
        amax = self._d_argmax.reshape(self._buf_shape)[self._blk_in_buf]
        if self._world > 1 and not self._emulated:
            # blocks differ in shape: gather through buffers padded to the largest block, then place each block
            mx = tuple(max(hi - lo for lo, hi in (blk[a] for blk in self._blocks)) for a in range(d))
            pad_res = torch.zeros(mx + (Cc,), dtype=res.dtype, device=self.device)
            pad_am = torch.zeros(mx, dtype=amax.dtype, device=self.device)
            own = tuple(slice(0, n) for n in self._local_shape)
            pad_res[own] = res
            pad_am[own] = amax
            out_r = [torch.empty_like(pad_res) for _ in range(self._world)]
            out_a = [torch.empty_like(pad_am) for _ in range(self._world)]
            torch.distributed.all_gather(out_r, pad_res, group=self._pg)
            torch.distributed.all_gather(out_a, pad_am, group=self._pg)
            res = torch.empty(tuple(self.image.shape[:d]) + (Cc,), dtype=res.dtype, device=self.device)
            amax = torch.empty(tuple(self.image.shape[:d]), dtype=amax.dtype, device=self.device)
            for blk, o_r, o_a in zip(self._blocks, out_r, out_a):
                dst = tuple(slice(lo, hi) for lo, hi in blk)
                src = tuple(slice(0, hi - lo) for lo, hi in blk)
                res[dst] = o_r[src]
                amax[dst] = o_a[src]
        rec = res.cpu().numpy()
        am = amax.cpu().numpy().astype(np.float64)
        if (am < 0).any():
            # tf.argmax over the influential kernels returns position 0 when every gate is zero:
            # the lowest-index influential kernel of the batch (smoe.py:833-836, 1716)
            infl_idx = torch.nonzero(self._infl).flatten()
            fill = float(infl_idx.min().item()) if infl_idx.numel() else 0.0
            am[am < 0] = fill
        return rec, am

    # ------------------------------------------------------------------------------------------
    # train loop (smoe.py:1485-1603)
    # ------------------------------------------------------------------------------------------
    def train(self, num_iter, val_iter=100, ukl_iter=None, optimizer1=None, optimizer2=None, optimizer3=None,
              grad_clip_value_abs=None, pis_l1=0, u_l1=0, sv_l1_sub_l2=0, sampling_percentage=100, callbacks=(),
              with_inc=False, train_inc=False, train_orig=True, use_loss_mask=False):
        if ukl_iter is None:
            ukl_iter = val_iter
        if optimizer1:
            self.set_optimizer(optimizer1, optimizer2, optimizer3, grad_clip_value_abs=grad_clip_value_abs)
        assert self.optimizer1 is not None, "no optimizer found, you have to specify one!"
        if self.quantization_mode >= 1:
            self.qparams = quantize_params(self, self.get_params())
        if self.quantization_mode == 1:
            self.rparams = rescaler(self, self.qparams)
            self.best_qloss, self.best_qmse, _, _ = self.run_batched(
                pis_l1=pis_l1, u_l1=u_l1, train=False, update_reconstruction=True, with_quantized_params=True)
            self.qlosses.append((0, self.best_qloss))
            self.qmses.append((0, self.best_qmse))
        self.best_loss, self.best_mse, num_pi, num_sv = self.run_batched(
            pis_l1=pis_l1, u_l1=u_l1, train=False, update_reconstruction=True, use_loss_mask=use_loss_mask)
        self.losses.append((self.iter, self.best_loss))
        self.mses.append((self.iter, self.best_mse))
        self.num_pis.append((self.iter, num_pi))
        self.num_svs.append((self.iter, num_sv))
        for callback in callbacks:
            callback(self)
        loss_val = mse_val = None
        i = 0
        for i in range(1, num_iter + 1):
            self.iter += 1
            try:
                validate = i % val_iter == 0
                update_kl = i % ukl_iter == 0
                loss_val, mse_val, num_pi, num_sv = self.run_batched(
                    pis_l1=pis_l1, u_l1=u_l1, train=train_orig, update_reconstruction=False,
                    sampling_percentage=sampling_percentage, use_loss_mask=use_loss_mask)
                if update_kl:
                    self.update_kernel_list(self.add_kernel_slots)
                    if not validate:
                        loss_val, mse_val, num_pi, num_sv = self.run_batched(
                            pis_l1=pis_l1, u_l1=u_l1, train=False, update_reconstruction=False)
                if validate:
                    self.check_replicas()
                    if self.quantization_mode >= 1:
                        self.qparams = quantize_params(self, self.get_params())
                    if self.quantization_mode == 1:
                        self.rparams = rescaler(self, self.qparams)
                        qloss_val, qmse_val, _, _ = self.run_batched(
                            pis_l1=pis_l1, u_l1=u_l1, train=False, update_reconstruction=True,
                            with_quantized_params=True, use_loss_mask=use_loss_mask)
                    loss_val, mse_val, num_pi, num_sv = self.run_batched(
                        pis_l1=pis_l1, u_l1=u_l1, train=False, update_reconstruction=True,
                        use_loss_mask=use_loss_mask)
                if np.isnan(loss_val) or (len(self.losses) > 0 and loss_val + 1 > (self.losses[0][1] + 100) * 10):
                    print("stop")
                    break
                if validate:
                    if not self.best_loss or loss_val < self.best_loss:
                        self.best_loss = loss_val
                        self._theta_best.copy_(self._theta)       # checkpoint_best_op, smoe.py:861-896
                    self.losses.append((self.iter, loss_val))
                    if not self.best_mse or mse_val < self.best_mse:
                        self.best_mse = mse_val
                    self.mses.append((self.iter, mse_val))
                    if self.quantization_mode == 1:
                        self.qmses.append((i, qmse_val))
                        self.qlosses.append((i, qloss_val))
                    self.num_pis.append((self.iter, num_pi))
                    self.num_svs.append((self.iter, num_sv))
                    for callback in callbacks:
                        callback(self)
            except KeyboardInterrupt:
                break
        self.losses_history.append(self.losses)
        self.mses_history.append(self.mses)
        print("end loss/mse: ", loss_val, "/", mse_val, "@iter: ", i)
        print("best loss/mse: ", self.best_loss, "/", self.best_mse)

    # ------------------------------------------------------------------------------------------
    # kernel lists (smoe.py:2287-2365): OR in every pi>0 kernel with maha < 800 at the 3^d
    # corner / mid points of each batch.  Host-side control, not on the hot path: torch ops.
    # ------------------------------------------------------------------------------------------
    def update_kernel_list(self, add_kernel_slots=0):
        d = self.dim_domain
        A = self._assembled_A()
        mu = self._centres()
        pis = self._effective_pis()
        full_axes = [np.linspace(0, 1, self.image.shape[a]) for a in range(d)]
        rects = self._batch_rects()
        if self._world > 1:
            # A sharded model is the one-batch model of the whole image: every rank probes the WHOLE image rectangle,
            # so the lists stay identical on all ranks (a rank-local probe would give every rank another kernel set,
            # and the exchanged statistics are indexed by packed position).
            rects = [((0,) * d, tuple(self.image.shape[:d]))]
        for ii, (org, ext) in enumerate(rects):
            pts = []
            ov = self.overlap
            padded = ov > 0 and any(org[a] - ov < 0 or org[a] + ext[a] + ov > self.image.shape[a] for a in range(d))
            for a in range(d):
                # min / max of the window's coordinates INCLUDING the overlap halo; the zero padding of border
                # windows sits at coordinate 0 on every axis (smoe.py:18-35, 2324-2330)
                lo = 0.0 if padded else full_axes[a][max(org[a] - ov, 0)]
                hi = full_axes[a][min(org[a] + ext[a] + ov, self.image.shape[a]) - 1]
                pts.append([lo, hi, (lo + hi) / 2])
            probe = torch.tensor(list(product(*pts)), dtype=torch.float32, device=self.device)      # (3^d, d)
            delta = probe[None, :, :] - mu[:, None, :]
            if self.train_inverse_cov:
                maha = torch.einsum("knl,klm,knm->kn", delta, A, delta)
            else:
                y = torch.einsum("klm,knl->knm", A, delta)
                maha = (y * y).sum(-1)
            near = ((maha < 800).any(dim=1) & (pis > 0)).to(torch.uint8)
            self._klist[ii] |= near
        self._refresh_perm()

    def _batch_rects(self):
        d = self.dim_domain
        if self._world > 1:
            return [(tuple(lo for lo, _ in self._block), self._local_shape)]
        starts = [range(0, self.image.shape[a], self.batch_size_valued[a]) for a in range(d)]
        return [(org, self.batch_size_valued) for org in product(*starts)]

    def check_replicas(self):
        """Desync guard of the sharded path (SURVEY.md 8e): every rank must hold bit-identical parameters, Adam state
        and kernel lists (the exchange sums in a fixed rank order, so they are by construction).  Collective; raises
        on any rank that differs from rank 0."""
        if self._world == 1 or self._emulated:
            return True
        sig = torch.stack([t.view(torch.int32).to(torch.int64).sum() for t in
                           (self._theta, self._adam_m, self._adam_v)] + [self._klist.to(torch.int64).sum()])
        ref = sig.clone()
        torch.distributed.broadcast(ref, src=torch.distributed.get_global_rank(self._pg, 0) if self._pg is not None else 0,
                                    group=self._pg)
        ok = torch.tensor([1 if bool((ref == sig).all()) else 0], device=self.device)
        torch.distributed.all_reduce(ok, op=torch.distributed.ReduceOp.MIN, group=self._pg)
        epoch, err = self.exchange_status()
        if ok.item() != 1 or err:
            raise RuntimeError(f"smoe_b200: replicas out of sync on rank {self._rank} (exchange epoch {epoch}, error {err})")
        return True

    def _assembled_A(self):
        d, K = self.dim_domain, self.start_pis
        A = torch.zeros((K, d, d), dtype=torch.float32, device=self.device)
        th = self._effective_theta()
        for l in range(d):
            for m in range(l + 1):
                A[:, l, m] = th[:, a_col(d, l, m)]
                if self.train_inverse_cov and m < l:
                    A[:, m, l] = A[:, l, m]
        return A

    def _effective_pis(self, theta=None):
        theta = self._theta if theta is None else theta
        pis = theta[:, self._off["pi"]]
        if self.quantize_pis:
            pis = _fake_quant_torch(pis, self.lower_bounds[3], self.upper_bounds[3], self.bit_depths[3])
        return pis

    def _effective_theta(self, theta=None):
        """The variables as the graph uses them: fake-quantised per group when quantization_mode == 2
        (smoe.py:482-496); pis also under quantize_pis."""
        theta = self._theta if theta is None else theta
        if self.quantization_mode < 2 and not self.quantize_pis:
            return theta
        if self.quantization_mode == 3:                       # ranges of THIS theta, then the device's own rounding
            L, st = lib(), stream_ptr()
            qd = torch.zeros_like(self._qdyn)
            out = torch.empty_like(theta)
            self._structural = torch.zeros((2,), dtype=torch.float32, device=self.device)
            check(L.smoe_quant_ranges(C.byref(self._cfg), ptr(theta), self.start_pis, int(self.train_musx), ptr(qd), st),
                  "smoe_quant_ranges")
            check(L.smoe_fake_quant_theta(C.byref(self._cfg), ptr(theta), ptr(qd), self.start_pis, ptr(out),
                                          ptr(self._structural), st), "smoe_fake_quant_theta")
            return out
        out = theta.clone()
        o = self._off
        out[:, o["pi"]] = self._effective_pis(theta)
        if self.quantization_mode == 2:
            lb, ub, bd = self.lower_bounds, self.upper_bounds, self.bit_depths
            out[:, 0:o["A"]] = _fake_quant_torch(theta[:, 0:o["A"]], lb[1], ub[1], bd[1])
            out[:, o["A"]:o["pi"]] = _fake_quant_torch(theta[:, o["A"]:o["pi"]], lb[0], ub[0], bd[0])
            out[:, o["nu"]:o["ga"]] = _fake_quant_torch(theta[:, o["nu"]:o["ga"]], lb[2], ub[2], bd[2])
            out[:, o["ga"]:] = _fake_quant_torch(theta[:, o["ga"]:], lb[4], ub[4], bd[4])
        return out

    def _centres(self):
        """Kernel centres as the graph uses them (offsets + grid under use_diff_center, smoe.py:746-747)."""
        mu = self._effective_theta()[:, 0:self.dim_domain]
        return mu + self._mus_grid if self.use_diff_center else mu

    # ------------------------------------------------------------------------------------------
    # params dict (smoe.py:1795-1849), checkpoints (smoe.py:1066-1077)
    # ------------------------------------------------------------------------------------------
    def _params_from(self, theta):
        d, Cc, K, o = self.dim_domain, self.image.shape[-1], self.start_pis, self._off
        pis = self._effective_pis(theta).cpu().numpy().copy()
        th = self._effective_theta(theta).cpu().numpy()        # get_params returns the q* tensors (smoe.py:1796-1798)
        A_diag = np.zeros((K, d, d), dtype=np.float32)
        A_corr = np.zeros((K, d, d), dtype=np.float32)
        if self.quantization_mode == 2:      # the reference fake-quantises the whole (K,d,d) variables (smoe.py:483-486)
            A_diag[:] = A_corr[:] = float(_fake_quant_torch(torch.zeros(1), self.lower_bounds[0], self.upper_bounds[0],
                                                            self.bit_depths[0]))
        elif self.quantization_mode == 3:    # (smoe.py:506-515)
            sv = self._structural.cpu().numpy()
            A_diag[:], A_corr[:] = sv[0], sv[1]
        for l in range(d):
            for m in range(l + 1):
                (A_diag if l == m else A_corr)[:, l, m] = th[:, a_col(d, l, m)]
        if self.radial_as:                                     # the (K,) variable (smoe.py:429-433)
            A_diag = th[:, d].copy()
        return {"pis": pis, "musX": th[:, 0:d].copy(), "A_diagonal": A_diag, "A_corr": A_corr,
                "gamma_e": th[:, o["ga"]:].reshape(K, d, Cc).copy(), "nu_e": th[:, o["nu"]:o["nu"] + Cc].copy()}

    def get_params(self):
        return self._params_from(self._theta)

    def get_best_params(self):
        return self._params_from(self._theta_best)

    def set_params(self, params):
        """Replacement for the reference's `session.run(re_assign_*_op)` pokes: assign any subset of
        the K_all-sized variables."""
        d, Cc, K, o = self.dim_domain, self.image.shape[-1], self.start_pis, self._off
        th = self._theta.cpu().numpy()
        if "musX" in params:
            th[:, 0:d] = params["musX"]
        for l in range(d):
            for m in range(l + 1):
                key = "A_diagonal" if l == m else "A_corr"
                if key in params and self.radial_as:
                    if l == m:
                        a = np.asarray(params[key])
                        th[:, a_col(d, l, m)] = a if a.ndim == 1 else a[:, 0, 0]
                elif key in params:
                    th[:, a_col(d, l, m)] = np.asarray(params[key])[:, l, m]
        if "pis" in params:
            th[:, o["pi"]] = params["pis"]
        if "nu_e" in params:
            th[:, o["nu"]:o["nu"] + Cc] = params["nu_e"]
        if "gamma_e" in params:
            th[:, o["ga"]:] = np.asarray(params["gamma_e"]).reshape(K, d * Cc)
        self._theta.copy_(torch.from_numpy(th).to(self.device))
        if "musX" in params:
            self._refresh_perm()
        self.valid = self.qvalid = False

    def get_gradients(self):
        """Accumulated gradients of the last training pass, in the params-dict layout.  (The reference
        leaves this a stub, smoe.py:1812-1813; exposed here because parity is tested on it.)"""
        d, Cc, K, o = self.dim_domain, self.image.shape[-1], self.start_pis, self._off
        g = self._grads.cpu().numpy()
        A_diag = np.zeros((K, d, d), dtype=np.float32)
        A_corr = np.zeros((K, d, d), dtype=np.float32)
        for l in range(d):
            for m in range(l + 1):
                (A_diag if l == m else A_corr)[:, l, m] = g[:, a_col(d, l, m)]
        if self.radial_as:                  # gradient of the one scalar per kernel (every diagonal entry carries it)
            A_diag = g[:, d].copy()
        return {"pis": g[:, o["pi"]].copy(), "musX": g[:, 0:d].copy(), "A_diagonal": A_diag, "A_corr": A_corr,
                "gamma_e": g[:, o["ga"]:].reshape(K, d, Cc).copy(), "nu_e": g[:, o["nu"]:o["nu"] + Cc].copy()}

    def checkpoint(self, path):
        torch.save({"theta": self._theta.cpu(), "theta_best": self._theta_best.cpu(), "adam_m": self._adam_m.cpu(),
                    "adam_v": self._adam_v.cpu(), "klist": self._klist.cpu(), "iter": self.iter,
                    "adam_t": [o._t if o is not None else 0 for o in (self.optimizer1, self.optimizer2, self.optimizer3)]},
                   path)
        print("Model saved in file: %s" % path)

    def restore(self, path):
        cp = torch.load(path, map_location="cpu")
        for name in ("theta", "theta_best", "adam_m", "adam_v", "klist"):
            getattr(self, "_" + name).copy_(cp[name].to(self.device))
        self.iter = cp["iter"]
        for o, t in zip((self.optimizer1, self.optimizer2, self.optimizer3), cp["adam_t"]):
            if o is not None:
                o._set_step(t)
        self.valid = self.qvalid = False
        print("Model restored from file: %s" % path)

    # ------------------------------------------------------------------------------------------
    # getters (smoe.py:1815-1888)
    # ------------------------------------------------------------------------------------------
    def get_reconstruction(self):
        if not self.valid:
            self.run_batched(train=False, update_reconstruction=True)
        return self.reconstruction_image

    def get_qreconstruction(self):
        if not self.qvalid:
            self.run_batched(train=False, update_reconstruction=True, with_quantized_params=True)
        return self.qreconstruction_image

    def get_weight_matrix_argmax(self):
        if not self.valid:
            self.run_batched(train=False, update_reconstruction=True)
        return self.weight_matrix_argmax

    def get_weight_matrix(self):
        """Dense (K_all, *image.shape[:-1]) gate matrix.  The reference allocates it on EVERY
        run_batched call (smoe.py:1632); here it is materialised only on request, with torch ops
        (not the hot path), and refuses sizes that cannot fit."""
        d, K = self.dim_domain, self.start_pis
        if K * self.num_pixel > 2 ** 31:
            raise MemoryError("dense weight matrix too large; use get_weight_matrix_argmax()")
        if self._world > 1:
            raise NotImplementedError("dense weight matrix on a sharded model")
        out = torch.zeros((K, self.num_pixel), dtype=torch.float32, device=self.device)
        A, mu, pis = self._assembled_A(), self._centres(), self._effective_pis()
        grids = torch.meshgrid(*[torch.linspace(0, 1, n, dtype=torch.float64).to(torch.float32) for n in self.image.shape[:d]],
                               indexing="ij")
        dom_full = torch.stack(grids, dim=-1).to(self.device)
        for ii, (org, ext) in enumerate(self._batch_rects()):
            sl = tuple(slice(o, o + e) for o, e in zip(org, ext))
            dom = dom_full[sl].reshape(-1, d)
            act = (self._klist[ii] > 0) & (pis > 0)
            idx = torch.nonzero(act).flatten()
            delta = dom[None] - mu[idx][:, None]
            if self.train_inverse_cov:
                maha = torch.einsum("knl,klm,knm->kn", delta, A[idx], delta)
            else:
                y = torch.einsum("klm,knl->knm", A[idx], delta)
                maha = (y * y).sum(-1)
            n = torch.exp(-0.5 * maha) * pis[idx][:, None]
            if self.use_determinant:
                n = n * (torch.diagonal(A[idx], dim1=1, dim2=2).prod(-1) / math.sqrt((2 * math.pi) ** d))[:, None]
            w = n / torch.clamp_min(n.sum(0), 10e-12)
            w = w * (w > 0.5 / 2 ** self.precision)
            lin = torch.arange(self.num_pixel, device=self.device).reshape(self.image.shape[:d])[sl].reshape(-1)
            out[idx[:, None], lin[None, :]] = w
        return out.reshape((K,) + tuple(self.image.shape[:d])).cpu().numpy().astype(np.float64)

    def get_best_reconstruction(self):
        raise NotImplementedError

    def get_best_weight_matrix(self):
        raise NotImplementedError

    def get_losses(self):
        return self.losses

    def get_qlosses(self):
        return self.qlosses

    def get_best_loss(self):
        return self.best_loss

    def get_losses_history(self):
        return self.losses_history

    def get_mses(self):
        return self.mses

    def get_qmses(self):
        return self.qmses

    def get_best_mse(self):
        return self.best_mse

    def get_mses_history(self):
        return self.mses_history

    def get_num_pis(self):
        return self.num_pis

    def get_num_svs(self):
        return self.num_svs

    def get_original_image(self):
        return np.squeeze(self.image)

    def get_iter(self):
        return self.iter

    # ------------------------------------------------------------------------------------------
    # GPU metrics (north_star item 4): PSNR from the graph's mse_op, SSIM of ops/image_ops_impl.py
    # ------------------------------------------------------------------------------------------
    def psnr(self, quantized=False):
        from .utils import psnr
        rec = self.get_qreconstruction() if quantized else self.get_reconstruction()
        from .ops.image_ops_impl import mse_gpu
        return psnr(mse_gpu(rec, self.image, device=self.device) * (2 ** self.precision) ** 2, self.precision)

    def ssim(self, quantized=False):
        from .ops.image_ops_impl import smoe_ssim
        rec = self.get_qreconstruction() if quantized else self.get_reconstruction()
        return smoe_ssim(rec, self.image, use_yuv=self.use_yuv, device=self.device)


class _PeerBuffer:
    """A dedicated device allocation that other ranks of the node can map (cudaIpc exports whole allocations, so it
    cannot come from torch's caching allocator): smoe_peer_alloc / _export / _open.  Exposed to torch through the
    CUDA array interface; torch does not own the memory."""

    def __init__(self, nbytes):
        self.nbytes = int(nbytes)
        self.ptr = C.c_void_p()
        check(lib().smoe_peer_alloc(C.c_size_t(self.nbytes), C.byref(self.ptr)), "smoe_peer_alloc")
        self.mapped = []

    def as_tensor(self, shape, device):
        holder = type("_CAI", (), {})()
        holder.__cuda_array_interface__ = {"shape": tuple(int(v) for v in shape), "typestr": "<f4",
                                           "data": (int(self.ptr.value), False), "version": 2, "strides": None}
        self._holder = holder
        return torch.as_tensor(holder, device=device)

    def handle(self):
        h = (C.c_ubyte * 64)()
        check(lib().smoe_peer_export(self.ptr, h), "smoe_peer_export")
        return bytes(h)

    def open_peer(self, handle):
        mapped = C.c_void_p()
        check(lib().smoe_peer_open((C.c_ubyte * 64).from_buffer_copy(handle), C.byref(mapped)), "smoe_peer_open")
        self.mapped.append(mapped)
        return mapped.value

    def close(self):
        for m in self.mapped:
            lib().smoe_peer_close(m)
        self.mapped = []
        if self.ptr:
            lib().smoe_peer_free(self.ptr)
            self.ptr = C.c_void_p()


def _fake_quant_torch(x, mn, mx, bits):
    """TF fake_quant_with_min_max_args values (float32), for get_params (smoe.py:1796-1798)."""
    f = np.float32
    qmax = f(2 ** bits - 1)
    scale = (f(mx) - f(mn)) / qmax
    zp = f(0) - f(mn) / scale
    nzp = f(0) if zp < 0 else (qmax if zp > qmax else f(np.floor(zp + f(0.5))))
    nmin, nmax = float((f(0) - nzp) * scale), float((qmax - nzp) * scale)
    inv = float(f(1) / scale)
    c = torch.clamp(x, nmin, nmax)
    return torch.floor((c - nmin) * inv + 0.5) * float(scale) + nmin
