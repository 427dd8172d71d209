/*
 * smoe_b200.h -- C ABI of libsmoe_b200.so: the B200 (sm_100a) drop-in for the hot path of
 * roljon/Steered-Mixture-of-Experts.
 *
 * The reference has no FFI: its seam is "Python `Smoe` methods <-> one TensorFlow
 * `session.run`" (smoe.py:1702 for the forward/backward graph, smoe.py:1788 for the Adam
 * `train_op`).  Every entry point below replaces one segment of that graph; the reference lines
 * it replaces are cited per function.  Bindings a maintainer of the reference would add are
 * shown in INTEGRATION.md (ctypes, as the reference is Python).
 *
 * Conventions
 *   - every function returns 0 on success, a positive cudaError_t, or a negative SMOE_E_* code;
 *     smoe_last_error() returns a thread-local message for the last failure;
 *   - the library never allocates, frees or retains caller-visible memory: all buffers are device
 *     pointers owned by the caller (float32 / int32 / uint8, contiguous, 16-byte aligned; the scalar blocks,
 *     counts and the tail of the exchange buffer only need their natural 4-byte alignment);
 *   - every launch is asynchronous on the `stream` argument (a cudaStream_t passed as void*);
 *     there is no host synchronisation and no host read-back inside the library;
 *   - the number of active kernels K lives on the device (`counts[0]`), so a training step
 *     never needs a device->host copy to size a launch.
 *
 * Layouts (float32 unless noted; d = dim_domain in {2,3}, C = channels in {1,3},
 * T = d(d+1)/2, P = d + T + 1 + C + d*C, PK = smoe_packed_stride(d,C) = roundup4(P+1+d)):
 *   theta  [K_all][P]  the K_all-sized variables, one row per kernel:
 *                      musX[d] | A lower-tri row-major (l,m), l>=m: diagonal entries are
 *                      A_diagonal_var[l,l], strictly-lower entries are A_corr_var[l,m] | pis |
 *                      nu_e[C] | gamma_e[d][C]
 *   grads, adam_m, adam_v : same shape as theta
 *   packed [K][PK]     compacted compute records (smoe_pack): musX[d] | Qm (upper-tri row-major
 *                      of s*A*A^T, or s*A_sym when train_inverse_cov; s = log2(e)/2) |
 *                      c0 = log2(pi * prod(diag A)/(2pi)^(d/2)) | nu_e[C] | gamma_e[d][C] |
 *                      lam, kap[d] (culling bounds) | pad
 *   image  [H][W]([T])[C]  target colours, the numpy layout of the reference's `image`
 *   axes   ax0[H], ax1[W], ax2[T]  pixel coordinates per axis (np.linspace(0,1,n) cast to f32,
 *                      smoe.py:2412 / the float32 feed at smoe.py:545)
 *   pix    [tiles][smoe_pix_stride]  per-pixel backward state written by the forward and streamed by the
 *                      backward: planes z, qthr, gr, g_c of SMOE_TPIX floats + the row-constant coordinates
 */
#ifndef SMOE_B200_H
#define SMOE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SMOE_ABI_VERSION 6   /* 3: Hilbert-ordered packing (perm argument of smoe_pack, influence flags by ORIGINAL index,
                                smoe_backward without perm/pos), executed-pair counters, eps_bits, peer exchange;
                                4: smoe_cotangent added (additive: every call of version 3 is unchanged);
                                5: the smoe_point_* calls added (additive: every call of version 4 is unchanged);
                                6: smoe_point_jacobian and smoe_jacobian added (additive: every call of version 5 is
                                   unchanged) */
#define SMOE_TPIX 512      /* pixels per tile (compile-time constant of the kernels) */
#define SMOE_NSCAL 16      /* floats in the scalar block */

/* sentinels of the optional per-pixel `loss_weights` of smoe_forward */
#define SMOE_PIXEL_ABSENT (-1.0f)   /* pixel is not part of this run's feed (sampling_percentage < 100)        */
#define SMOE_PIXEL_HALO   (-2.0f)   /* pixel of the overlap halo: forwarded, outside the loss (overlap_of_batches) */

#define SMOE_E_BADARG (-1)
#define SMOE_E_UNSUPPORTED (-2)

/* Static model configuration; field names follow Smoe.__init__ (smoe.py:38-41). */
typedef struct smoe_cfg {
    int32_t d;                 /* dim_domain: 2 (image) or 3 (video)                        */
    int32_t C;                 /* channels: 1 or 3                                          */
    int32_t precision;         /* output bit depth (smoe.py:825, 899, 931, 1053)            */
    float   margin;            /* epsilon = margin / 2^precision (smoe.py:931)              */
    int32_t use_determinant;   /* smoe.py:809-815                                           */
    int32_t train_inverse_cov; /* maha = d^T A d with symmetric A (smoe.py:734-735, 793)    */
    int32_t use_yuv;           /* loss weights 6/8,1/8,1/8 (smoe.py:933-935)                */
    int32_t train_gammas;      /* smoe.py:841-848: gamma ignored in the forward when 0      */
    int32_t only_y_gamma;      /* smoe.py:725-729                                           */
    int32_t quantize_pis;      /* fake-quantise pis before the >0 mask (smoe.py:474-480)    */
    float   pis_lb, pis_ub;    /* lower_bounds[3], upper_bounds[3]                          */
    int32_t pis_bits;          /* bit_depths[3]                                             */
    int32_t quantization_mode; /* 2: every parameter is fake-quantised with the fixed bounds below before use,
                                  gradients pass straight through inside the bounds (smoe.py:482-496);
                                  3: the same with the min / max of the surviving kernels instead of fixed
                                  bounds (smoe.py:497-531; q_bits only, see smoe_quant_ranges);
                                  0/1: parameters are used as they are (mode 1 quantises on the host only) */
    float   q_lb[5], q_ub[5];  /* lower_bounds / upper_bounds in the reference's order: A, musX, nu_e, pis,
                                  gamma_e (smoe_test.py:306-309)                                        */
    int32_t q_bits[5];         /* bit_depths, same order (smoe_test.py:302)                            */
    int32_t use_diff_center;   /* the musX variable holds offsets from a fixed grid (smoe.py:390-394, 746-747) */
    int32_t kernel_count_as_norm_l1; /* L1 on pis normalised by the live kernel count (smoe.py:1022-1025) */
    int32_t radial_as;         /* A = a * I with ONE trainable scalar per kernel and a frozen A_corr = 0
                                  (smoe.py:429-434, 714-721): the d diagonal entries of a theta row are kept
                                  equal -- each receives the sum of the d diagonal gradients -- and the
                                  strictly-lower entries receive none                                    */
    int32_t dense_exec;        /* 0: exact culling + exact-zero skipping (default);
                                  1: execute every (pixel, kernel) pair in full;
                                  2: exact-zero skipping inside the dense sweeps, no tile-level
                                     culling.  Results of the three modes are bit-identical.  */
    int32_t eps_bits;          /* 0 (default): exact.  x > 0: OPT-IN epsilon culling -- (pixel, kernel) terms below
                                  2^-x of the pixel's normaliser are dropped (x in [24, 126]); results then differ
                                  from the exact modes by < 2^-x relative per dropped term                 */
} smoe_cfg;

/* One spatial batch (smoe.py:18-35 sliding_window / one rank's shard) of a resident image. */
typedef struct smoe_batch {
    int32_t dims[3];     /* extents of the resident image buffer (H, W, T); T = 1 when d == 2 */
    int32_t origin[3];   /* first pixel of the batch inside the buffer                         */
    int32_t extent[3];   /* batch extents                                                      */
    int32_t tile[3];     /* tile extents, tile[0]*tile[1]*tile[2] == SMOE_TPIX                 */
    float   inv_count;   /* 1 / number of pixels the loss means run over (smoe.py:927-937);
                            N_batch on one GPU, N_total when pixels are sharded over ranks     */
    int32_t halo;        /* overlap_of_batches: the rectangle is the window PLUS this many halo pixels on every
                            side that is not the image border; halo pixels are forwarded (gates, influence
                            list) and cropped away before the loss (smoe.py:909-923, 985-991)                 */
} smoe_batch;

/* Adam hyper-parameters of the three optimizer groups (smoe.py:1102-1104, smoe_test.py:84-88):
 * group 0 = {nu_e, gamma_e, musX}, 1 = {pis}, 2 = {A_diagonal, A_corr}.  alpha is the
 * bias-corrected step lr*sqrt(1-beta2^t)/(1-beta1^t) of TF1's ApplyAdam; alpha == 0 skips the
 * group (optimizer._lr == 0, smoe.py:1120-1144, or a non-trainable variable). */
typedef struct smoe_adam {
    float alpha[3], beta1[3], beta2[3], epsilon[3];
    float grad_clip;     /* <= 0: off (grad_clip_value_abs, smoe.py:1152-1153) */
    int32_t train_musx;  /* smoe.py:394 */
    int32_t train_gammas;/* smoe.py:389 */
} smoe_adam;

int         smoe_abi_version(void);
const char* smoe_last_error(void);
int         smoe_param_count(int d, int C);      /* P  */
int         smoe_packed_stride(int d, int C);    /* PK */
int         smoe_num_tiles(const smoe_batch* b);
int         smoe_pix_stride(int d, int C, const smoe_batch* b);   /* floats of `pix` per tile */
size_t      smoe_pack_workspace_bytes(int K_all);
size_t      smoe_backward_workspace_bytes(const smoe_cfg* cfg, int K_cap, int num_splits);

/* pi-mask compaction + parameter staging.  Replaces smoe.py:474-480 (optional fake-quant of pis),
 * 732-735 (A assembly), 738-753 (bool_mask = kernel_list & pis>0, indices, 5x boolean_mask) and
 * 1012 (num_pi = count_nonzero(qpis>0)); stable stream compaction of the sequence perm[0..K_all) (perm == NULL:
 * ascending kernel index, the order of the reference's boolean_mask).  The SET {indices[0..K)} is the reference's
 * `indices`; the ORDER is a work-assignment choice: with perm = Hilbert order of the centres (smoe_spatial_keys +
 * a sort), 128 consecutive records (one shared-memory chunk of smoe_forward) and 32 consecutive records (one CTA of
 * smoe_backward) are spatial neighbours, which is what the exact tile culling exploits.
 *   counts[0] = K (active), counts[1] = num_pi, counts[2] = kernels with pi*det <= 0 (unsupported
 *   by the fast path, reported), counts[3] = 0
 *   regsums[0] = sum of active pis, regsums[1] = sum of diag(A) over active kernels (for the
 *   L1 terms of smoe.py:1027, 1044)
 *   chunk_bounds: per 128 consecutive active kernels, bounding box of the centres, smallest
 *   eigenvalue bound and largest c0 -- the coarse level of the exact culling in smoe_forward */
int smoe_pack(const smoe_cfg* cfg, const float* theta, const float* mus_grid /*[K_all][d], use_diff_center only*/,
              const void* quant_ranges /* quantization_mode 3 only, from smoe_quant_ranges */,
              const uint8_t* kernel_list, const int32_t* perm /*[K_all] or NULL*/, int K_all,
              float* packed, int32_t* indices /*[K_all]: original index of packed row k*/,
              int32_t* pos /*[K_all]: packed row of each kernel or -1*/,
              int32_t* counts, float* regsums,
              float* chunk_bounds /*[ceil(K_all/128)][12]*/, void* workspace,
              float* grads_clear /* optional [K_all][P]: zeroed (zero_op of the accumulators, smoe.py:1612-1613) */,
              float* scalars_clear /* optional [SMOE_NSCAL]: zeroed */, uint8_t* infl_clear /* optional [K_all]: zeroed */,
              void* stream);

/* Same staging for parameters that are FED over the compacted tensors (with_quantized_params,
 * smoe.py:1688-1689: rparams A, musX, nu_e, gamma_e, pis of K rows each); no mask, K given. */
int smoe_pack_fed(const smoe_cfg* cfg, const float* A /*[K][d][d]*/, const float* musX, const float* nu_e,
                  const float* gamma_e, const float* pis, const int32_t* order /*[K] or NULL: fed row staged at packed
                  row j (e.g. Hilbert order)*/, int K, float* packed, int32_t* indices /*[K] out: order, or identity*/,
                  int32_t* counts, float* chunk_bounds, float* scalars_clear /*optional*/,
                  uint8_t* infl_clear /*optional [K_all]*/, int K_all, void* stream);

/* Hilbert-curve keys of the kernel centres on a 2^10 grid per axis (centres[i*row_stride + a] (+ grid[i*d + a]),
 * times scale[a] (host array of d floats, or NULL = 1): n_a / max_a n_a makes the curve isotropic in pixels).  Sorting
 * them gives the `perm` of smoe_pack / the `order` of smoe_pack_fed.  Any run of consecutive Hilbert indices is
 * spatially compact, which keeps chunks / CTAs compact after stream compaction shifts the run boundaries. */
int smoe_spatial_keys(const float* centres, int K, int d, int row_stride, const float* grid /*or NULL*/,
                      const float* scale /*host [d] or NULL*/, long long* keys, void* stream);

/* Fused forward over one batch: Mahalanobis logits, gating with the un-renormalised threshold, experts, mixture.
 * Replaces smoe.py:777-858 (kernel values, gates, influence list, argmax, mixture).  The K x N gate matrix is never
 * materialised.  The forward reads NO target pixels: clip, output quantisation and the loss live in smoe_loss, so a
 * step's target may still be on its way from the host while the sweeps run.
 *   rbuf     [dims..][C]  mixture output r BEFORE clip / quantisation (written inside the batch rectangle, not for
 *            halo pixels)
 *   argmax   [dims..] int32, optional: original index of the kernel with the largest gate (ties: the lowest
 *            original index, as tf.argmax over the ascending `indices`), -1 where no gate passed the threshold
 *            (host applies tf.argmax's all-zero convention)
 *   infl     [K_all] uint8, optional, indexed by ORIGINAL kernel index: 1 where the kernel's gate passed the
 *            threshold for some pixel (kernel_list_batch, smoe.py:829); must be zeroed by the caller (smoe_pack can)
 *   pix      optional: per-pixel state for smoe_loss / smoe_backward (planes z, qthr = log2 max(S, 1e-11), and the
 *            "S > 1e-11" flag in the gr plane)
 *   tile_qmin [tiles] (required with pix): min over the tile of qthr, the culling threshold of the backward; with
 *            cfg->eps_bits also READ: the previous pass's value bounds this pass's sweep A
 *   loss_weights [dims..] optional: only its sentinels matter here -- SMOE_PIXEL_ABSENT (the pixel is not fed at all:
 *            random sub-sampling, smoe.py:1664-1667) and SMOE_PIXEL_HALO (forwarded, no output)
 *   pair_counts [8] uint64, optional (NULL in the product path): executed-work counters for the roofline
 *            report, accumulated with integer atomics -- [0] sweep-A pairs whose logit was evaluated, [1] sweep-A
 *            pairs whose ex2 + add was executed, [2] sweep-B pairs evaluated, [3] sweep-B pairs whose expert part
 *            was executed; smoe_backward adds [4] pairs evaluated, [5] pairs whose gate / moment part was executed,
 *            [6] pairs whose expert part was executed (all in lanes x pixels as issued) */
int smoe_forward(const smoe_cfg* cfg, const smoe_batch* batch, const float* packed, const int32_t* indices,
                 const int32_t* counts, const float* chunk_bounds, int K_cap, const float* loss_weights,
                 const float* ax0, const float* ax1, const float* ax2, float* rbuf, int32_t* argmax, uint8_t* infl,
                 float* pix, float* tile_qmin /*[tiles]*/, unsigned long long* pair_counts, void* stream);

/* Loss stage of one batch, after smoe_forward: res = fake_quant(clip(r)) (smoe.py:857, 899), diff = res - target,
 * loss and squared-error sums (smoe.py:905-937, 1053), and -- when pix != NULL -- dL/dr with the straight-through
 * masks of clip and fake-quant: g_c and gr = sum_c g_c r_c (0 where S was clamped, smoe.py:821) into the planes of the
 * backward state.  Elementwise, HBM-bound.
 *   image / image_u8  exactly one: float32 target, or 8-bit pixels as an image file holds them, divided by 255 in
 *            float32 as utils.py:126-128 does
 *   loss_weights [dims..] optional (NULL = weight 1 everywhere): per-pixel weight of the loss term (the `loss_weights`
 *            feed of smoe.py:550, 932, 1674-1677) or a sentinel (absent / halo pixels take no part)
 *   res      [dims..][C]  optional: fake-quantised reconstruction (written inside the batch rectangle, not for halo
 *            pixels); a plain training pass needs only its sums and passes NULL
 *   scalars  [SMOE_NSCAL]: [0..C) sum_n (|diff|-eps)^2 per channel, [4] sum diff^2, [5] non-finite flag; accumulated
 *            (+=) so that batches / ranks can be summed; the caller zeroes it (smoe_pack can)
 *   partials [smoe_loss_partials(batch)][8] scratch, ticket: one int32, zero before the first call */
int smoe_loss_partials(const smoe_batch* batch);
int smoe_loss(const smoe_cfg* cfg, const smoe_batch* batch, const float* rbuf, const float* image,
              const uint8_t* image_u8, const float* loss_weights, float* res, float* pix, float* scalars,
              float* partials, int32_t* ticket, void* stream);

/* Any upstream gradient into the backward state, in place of smoe_loss, after smoe_forward (with pix) and before
 * smoe_backward: the loss is the caller's (a PyTorch loss, a larger network), the library only needs its dL/dr.
 *   grad_r   [dims..][C]  dL/dr with r the mixture output BEFORE clip (the rbuf of smoe_forward), same layout as rbuf
 *   pix      the forward's state: per pixel slot of every tile, g_c = grad_r (0 outside the batch rectangle) and
 *            gr = sum_c g_c r_c (fmaf in channel order from 0, as smoe_loss) where S > 1e-11, else 0 (smoe.py:821)
 * One CTA per tile, the launch geometry of smoe_loss; elementwise, HBM-bound, no reduction, no atomics.  The batch has
 * no halo.  The flag "S > 1e-11" that smoe_forward leaves is consumed: call it once per smoe_forward. */
int smoe_cotangent(const smoe_cfg* cfg, const smoe_batch* batch, const float* rbuf, const float* grad_r, float* pix,
                   void* stream);

/* Fused backward over one batch: recomputes the gates from the per-pixel state and reduces the
 * per-kernel sufficient statistics (sum t, sum t*delta, sum t*delta*delta^T, sum m*w*g,
 * sum m*w*g*x) over the pixels, kernel-stationary, deterministically (no float atomics).
 * Replaces tf.gradients(loss_op, variables) at smoe.py:1148 for the data term.
 *   raw_part [num_splits][K_cap][P]  partial statistics, one slab per pixel split */
int smoe_backward(const smoe_cfg* cfg, const smoe_batch* batch, const float* packed, const int32_t* counts,
                  int K_cap, const float* pix, const float* tile_qmin,
                  const float* ax0, const float* ax1, const float* ax2, int num_splits, float* raw_part,
                  int32_t* plan /* smoe_backward_plan_bytes: [groups] reachable-tile counts | [groups] tile bitmasks,
                  groups of 32 packed kernels; written by a planning pre-pass of this call and read again by
                  smoe_grad_finalize / smoe_reduce_splits / smoe_xchg_publish */,
                  unsigned long long* pair_counts /* optional, see smoe_forward */, void* stream);
size_t smoe_backward_plan_bytes(int K_cap, const smoe_batch* batch);
/*   Thread slot s works on packed row s: the order smoe_pack wrote (any order gives the same per-kernel results;
 *   a spatially coherent one makes the kernels of a warp / CTA neighbours, which is what the tile culling exploits). */
/* number of pixel splits for smoe_backward on this batch (split s owns tiles s, s+NS, ...): a prime that keeps
 * the grid a few waves deep and does not divide the tile-grid extents */
int smoe_suggest_splits(int K_cap, const smoe_batch* batch);

/* ---- evaluation at arbitrary points (csrc/points.cu) ------------------------------------------------------------
 * The model at n_points coordinates points[n][d] instead of on a uniform grid, differentiable in the parameters and in
 * the coordinates.  The points arrive in TILE ORDER: a point tile is a run of SMOE_TPIX consecutive points (the last
 * one may be partial), and culling works on each tile's bounding box, so any order is correct and a spatially coherent
 * one (e.g. sorted along a Hilbert curve with smoe_spatial_keys) is fast.  Coordinates must be finite; a tile with a
 * NaN coordinate culls nothing.  cfg->eps_bits must be 0; cfg->dense_exec 0, 1 and 2 give the same bits.
 *   smoe_point_forward    r[n][C] (before clip) at every point, from the smoe_pack records (chunk bounds included).
 *                         With state != NULL (then tile_box too) also the backward state, per tile of
 *                         smoe_point_stride floats: planes qthr | gr | g_c | tile-centred x'_l of SMOE_TPIX floats,
 *                         and tile_box[tiles][8] = centre[3] | rounded-out half extent[3] | min qthr | 0
 *   smoe_point_cotangent  a caller's dL/dr ([n][C], point order of r) into the state: g_c, and gr = sum_c g_c r_c where
 *                         S > 1e-11, else 0; call it once per smoe_point_forward, before the two calls below
 *   smoe_point_backward   planning pre-pass (every group of 32 packed kernels against every tile box) + kernel-
 *                         stationary sweep into raw_part [num_splits][K_cap][P] and `plan` (smoe_point_plan_bytes), the
 *                         layouts of smoe_backward: smoe_grad_finalize turns them into parameter gradients
 *   smoe_point_xgrad      grad_points[n][d] = dL/dx per point (pixel-stationary, fixed kernel order, no atomics)
 * smoe_point_splits gives num_splits from K_cap and n_points alone. */
#define SMOE_POINT_MAX 2147483136   /* 2^31 - 512: largest n_points */
int    smoe_point_tiles(int n_points);
int    smoe_point_stride(int d, int C);      /* floats of `state` per tile */
size_t smoe_point_plan_bytes(int K_cap, int n_points);
int    smoe_point_splits(int K_cap, int n_points);
int smoe_point_forward(const smoe_cfg* cfg, const float* packed, const int32_t* counts, const float* chunk_bounds,
                       int K_cap, const float* points, int n_points, float* r, float* state /*or NULL*/,
                       float* tile_box /*[tiles][8] with state*/, void* stream);
int smoe_point_cotangent(const smoe_cfg* cfg, int n_points, const float* r, const float* grad_r, float* state,
                         void* stream);
int smoe_point_backward(const smoe_cfg* cfg, const float* packed, const int32_t* counts, int K_cap, int n_points,
                        const float* state, const float* tile_box, int num_splits, float* raw_part, int32_t* plan,
                        void* stream);
int smoe_point_xgrad(const smoe_cfg* cfg, const float* packed, const int32_t* counts, const float* chunk_bounds,
                     int K_cap, int n_points, const float* state, const float* tile_box, float* grad_points,
                     void* stream);

/* ---- spatial Jacobian at arbitrary points and on a grid (csrc/jacobian.cu) -----------------------------------------
 * jac[n][C][d] = d r_c / d x_l at every point (tile order), the derivative of r before clip, from the state and
 * tile_box of a smoe_point_forward call with state and its r ([n][C], tile order).  Call it before
 * smoe_point_cotangent, which overwrites the flag S > 1e-11 the forward leaves in the gr plane.  One pixel-stationary
 * sweep: every kernel above the exact-zero cut, in packed order, no float atomics; as for dL/dx, the 0/1 gate decision
 * w > tau contributes no term.  cfg->eps_bits must be 0; cfg->dense_exec 0, 1 and 2 give the same bits. */
int smoe_point_jacobian(const smoe_cfg* cfg, const float* packed, const int32_t* counts, const float* chunk_bounds,
                        int K_cap, int n_points, const float* state, const float* tile_box, const float* r, float* jac,
                        void* stream);
/* The same Jacobian on a uniform grid: jac[pixel][C][d] in rbuf's layout, per unit of the axes' coordinate, from the
 * pix and tile_qmin of a smoe_forward call on `batch` (which must have halo 0) and its rbuf; the tile geometry and
 * coordinates are recomputed from the batch and the axes as the forward computes them.  Call it before smoe_loss or
 * smoe_cotangent, which overwrite the flag in the gr plane. */
int smoe_jacobian(const smoe_cfg* cfg, const smoe_batch* batch, const float* packed, const int32_t* counts,
                  const float* chunk_bounds, int K_cap, const float* pix, const float* tile_qmin, const float* ax0,
                  const float* ax1, const float* ax2 /*NULL when d == 2*/, const float* rbuf, float* jac, void* stream);

/* ---- Jacobian-vector products: forward-mode derivatives in the parameters and the points (csrc/jvp.cu) ------------
 * dr = (d r / d theta) dtheta + (d r / d x) dpoints, the derivative of r before clip, in one pixel-stationary sweep
 * after the forward, with the Jacobian's culling (the exact-zero cut), fixed packed-kernel order and no float atomics;
 * cfg->dense_exec 0, 1 and 2 give the same bits.  As for dL/dx, the 0/1 gate decision w > tau contributes no term;
 * kernels smoe_pack dropped (pi <= 0) have no tangent.  cfg->eps_bits must be 0.
 *   smoe_pack_tangent  dtheta ([K_all][P], theta's row layout) -> tangent[K_cap][smoe_tangent_stride] in packed order,
 *                      one record per packed row (read through `indices`; K from counts[0] on the device), for the
 *                      theta, indices and counts of a smoe_pack call without fake quantisation or diff centres
 *   smoe_jvp           dr in rbuf's layout on the grid of a smoe_forward call with pix / tile_qmin on `batch` (halo
 *                      0), from its rbuf; call it before smoe_loss or smoe_cotangent (it reads the flag in gr)
 *   smoe_point_jvp     dr[n][C] in tile order from the state, tile_box and r of a smoe_point_forward call with state;
 *                      tangent (parameters) and dpoints ([n][d] tile order) may each be NULL, not both; call it before
 *                      smoe_point_cotangent */
int smoe_tangent_stride(int d, int C);      /* floats per record of `tangent` */
int smoe_pack_tangent(const smoe_cfg* cfg, const float* theta, const float* dtheta, const int32_t* indices,
                      const int32_t* counts, int K_cap, float* tangent, void* stream);
int smoe_jvp(const smoe_cfg* cfg, const smoe_batch* batch, const float* packed, const float* tangent,
             const int32_t* counts, const float* chunk_bounds, int K_cap, const float* pix, const float* tile_qmin,
             const float* ax0, const float* ax1, const float* ax2 /*NULL when d == 2*/, const float* rbuf, float* dr,
             void* stream);
int smoe_point_jvp(const smoe_cfg* cfg, const float* packed, const float* tangent /*or NULL*/, const int32_t* counts,
                   const float* chunk_bounds, int K_cap, int n_points, const float* state, const float* tile_box,
                   const float* r, const float* dpoints /*[n][d] tile order, or NULL*/, float* dr, void* stream);

/* ---- Gauss-Newton diagonal: D = diag(J^T diag(h) J) in every parameter (csrc/gn_diag.cu) -------------------------
 * J = d r / d theta of r before clip, h >= 0 a per-sample, per-channel weight (NULL: h = 1, so D = diag(J^T J); for a
 * loss sum l(r), h = l'' gives the generalised Gauss-Newton diagonal).  Per kernel, P non-negative sums over the
 * samples: ln2^2 w^2 (dq/dtheta_i)^2 sum_c h_c (m E_c - f r_c)^2 for the gate parameters (mu, the A entries the op
 * reads, pi; dq/dtheta_i as smoe_pack_tangent's one-hot tangent logit), h_c m w^2 for nu and h_c m w^2 x_l^2 for gamma.
 * As for the JVP, the 0/1 gate decision w > tau contributes no term and kernels smoe_pack dropped (pi <= 0) have no
 * row.  Kernel-stationary sweep after the forward, with backward_kernel's CTAs, splits and planning pre-pass, no float
 * atomics; cfg->dense_exec 0, 1 and 2 give the same bits.  cfg->eps_bits must be 0; no fake quantisation, diff
 * centres or radial A.  Four stages, in stream order:
 *   smoe_gn_state          after smoe_forward with pix / tile_qmin on `batch` (halo 0) and BEFORE smoe_loss or
 *                          smoe_cotangent, which overwrite the flag S > 1e-11 in the gr plane: writes gstate, per tile
 *                          of smoe_gn_state_stride floats: planes z | qthr | h_c | f r_c of SMOE_TPIX floats, then the
 *                          row coordinates of pix.  weight[sample * stride_sample + c * stride_channel] with sample the
 *                          pixel index of rbuf's layout (strides 0 broadcast), or NULL
 *   smoe_point_gn_state    the same after smoe_point_forward with state, before smoe_point_cotangent: planes
 *                          qthr | h_c | f r_c | x'_l per tile of smoe_point_gn_state_stride floats.  r in tile order;
 *                          the weight is indexed by the caller's row order[i] ([n] int64) of tile slot i
 *   smoe_gn_diag /         planning pre-pass (bwd_plan_kernel / point_plan_kernel) + sweep into raw_part
 *   smoe_point_gn_diag     [num_splits][K_cap][P] in theta's column layout (mu | A lower-tri | pi | nu | gamma), packed
 *                          order, and `plan` (smoe_backward_plan_bytes / smoe_point_plan_bytes; num_splits as for
 *                          smoe_backward / smoe_point_splits).  theta and indices are those of the smoe_pack call.
 *   then smoe_reduce_splits(raw_part, plan) -> raw[K_cap][P], and
 *   smoe_gn_diag_scatter   diag[indices[k]] = raw[k] for the counts[0] packed rows (K on the device); the caller zeroes
 *                          diag[K_all][P] first, so dropped kernels keep 0 rows. */
int smoe_gn_state_stride(int d, int C, const smoe_batch* batch);     /* floats of gstate per grid tile */
int smoe_point_gn_state_stride(int d, int C);                        /* floats of gstate per point tile */
int smoe_gn_state(const smoe_cfg* cfg, const smoe_batch* batch, const float* pix, const float* rbuf,
                  const float* weight /*or NULL*/, long long weight_stride_sample, long long weight_stride_channel,
                  float* gstate, void* stream);
int smoe_point_gn_state(const smoe_cfg* cfg, int n_points, const float* state, const float* r,
                        const float* weight /*or NULL*/, const int64_t* order /*with a weight*/,
                        long long weight_stride_sample, long long weight_stride_channel, float* gstate, void* stream);
int smoe_gn_diag(const smoe_cfg* cfg, const smoe_batch* batch, const float* packed, const float* theta,
                 const int32_t* indices, const int32_t* counts, int K_cap, const float* gstate, const float* tile_qmin,
                 const float* ax0, const float* ax1, const float* ax2 /*NULL when d == 2*/, int num_splits,
                 float* raw_part, int32_t* plan, void* stream);
int smoe_point_gn_diag(const smoe_cfg* cfg, const float* packed, const float* theta, const int32_t* indices,
                       const int32_t* counts, int K_cap, int n_points, const float* gstate, const float* tile_box,
                       int num_splits, float* raw_part, int32_t* plan, void* stream);
int smoe_gn_diag_scatter(const smoe_cfg* cfg, const float* raw, const int32_t* indices, const int32_t* counts,
                         int K_cap, float* diag, void* stream);

/* Fixed-order reduction of the pixel splits: raw[k][j] = sum_s raw_part[s][k][j].  (The buffer a
 * multi-GPU run all-reduces with NCCL.) */
int smoe_reduce_splits(const smoe_cfg* cfg, const int32_t* counts, int K_cap, int num_splits,
                       const float* raw_part, const int32_t* plan /* of the smoe_backward call, or NULL: every slab */,
                       float* raw, void* stream);

/* Statistics -> variable gradients (chain rule through A assembly, pi, determinant; L1 terms of
 * smoe.py:1027, 1044), scattered through `indices` and ACCUMULATED into the K_all-sized `grads`
 * (assign_add, smoe.py:1150).  Also rewrites kernel_list[indices[k]] = infl[k] when infl != NULL
 * (smoe.py:1763-1766). */
int smoe_grad_finalize(const smoe_cfg* cfg, const float* raw, int num_splits,
                       const int32_t* plan /* of the smoe_backward call that wrote `raw`, or NULL: every slab */,
                       int K_cap, const float* theta,
                       const void* quant_ranges /* quantization_mode 3 only */,
                       const int32_t* indices, const int32_t* counts, float pis_l1, float l1_norm /* start_pis */,
                       float u_l1, float* grads, void* stream);

/* quantization_mode 3 (smoe.py:497-531): fake_quant_with_min_max_vars whose min / max are reduce_min / reduce_max
 * over the kernels with a positive (fake-quantised) pi.  smoe_quant_ranges computes those ranges and TF's nudged
 * scales on the device (no host read-back) into an opaque block of smoe_quant_ranges_bytes() that smoe_pack,
 * smoe_grad_finalize, smoe_fake_quant_theta and smoe_quant_route take; call it once per training step, before the
 * first smoe_pack.  A_diagonal (over its diagonal) and nu_e use the shifted form fq(x - min; 0, max - min) + min,
 * A_corr, musX (only when train_musx) and gamma_e the plain form; pis keep their fixed bounds.
 * smoe_quant_route finishes the gradient of the plain groups on the ACCUMULATED `grads`, once per step before
 * smoe_adam_step: elements outside the nudged range lose their gradient to `min` / `max`, i.e. to the extreme
 * elements of the kept kernels (equal shares among ties).
 * smoe_fake_quant_theta writes the variables as the graph uses them (modes 2 and 3 and quantize_pis; what
 * get_params returns, smoe.py:1796-1798); structural[0..1] (optional) receive what the structural zeros of
 * A_diagonal (off-diagonal) and A_corr (diagonal and above) turn into. */
size_t smoe_quant_ranges_bytes(void);
int smoe_quant_ranges(const smoe_cfg* cfg, const float* theta, int K_all, int train_musx, void* quant_ranges,
                      void* stream);
int smoe_quant_route(const smoe_cfg* cfg, const float* theta, const void* quant_ranges /* its scratch part is written */,
                     int K_all, float* grads, void* stream);
int smoe_fake_quant_theta(const smoe_cfg* cfg, const float* theta, const void* quant_ranges, int K_all, float* out,
                          float* structural /*[2]*/, void* stream);

/* kernel_list[i] = 0 for all i, then kernel_list[indices[k]] = influential (smoe.py:1763-1766); with the influence
 * flags indexed by original kernel index this is kernel_list[i] = infl[i]. */
int smoe_update_kernel_list(const uint8_t* infl, uint8_t* kernel_list, int K_all, void* stream);

/* Start of a run_batched pass in one launch: zero the gradient accumulators (zero_op, smoe.py:1612-1613; grads may
 * be NULL for an evaluation pass), the SMOE_NSCAL-float scalar block of each of n_rows batches (row_stride floats
 * apart) and the influence flags (infl may be NULL). */
int smoe_step_begin(float* grads, size_t n_grads, float* scalars, int n_rows, int row_stride, uint8_t* infl, int K,
                    void* stream);

/* ---- pixel-sharded step (SURVEY.md 8e): one exchange per pass, over NVLink peer memory -------------------------
 * Every rank owns a WINDOW of device memory (smoe_xchg_window_bytes) that all ranks of the node have mapped
 * (cudaIpc handles travel through the host plumbing, e.g. torch.distributed.all_gather_object):
 *     [flag block: one epoch slot per rank | epoch | error] [payload 0] [payload 1]
 *     payload = [K_all*P statistics (sum over this rank's pixel splits) | SMOE_NSCAL scalars | K_all influence flags]
 * smoe_xchg_publish fills payload[epoch & 1] (replaces the reference-free "reduce_splits + pack" pair);
 * the CONSUMER -- smoe_grad_finalize_peers on a training pass, smoe_xchg_reduce_tail on an evaluation pass --
 * announces the epoch to every peer (st.release.sys), waits until all ranks have announced it (ld.acquire.sys on
 * its own flag block), then reads the R windows directly and sums them in rank order: a one-shot all-reduce fused
 * into the kernel that needs the result.  All ranks add the same rows in the same order, so gradients, Adam updates
 * and kernel lists are bit-identical on every rank.  No host synchronisation, no library collective; the calls are
 * stream-ordered kernels and can be captured in a CUDA graph.  Every rank must issue the same sequence of
 * publish / consume calls.  A rank that waits ~5 s for a peer sets the error word (smoe_xchg_status) instead of
 * hanging.  This replaces what the reference would do with a gradient all-reduce (there is none in the reference:
 * it is single-process; the exchange is the new step SURVEY.md 8e defines). */
#define SMOE_MAX_PEERS 8
typedef struct smoe_peers {
    int32_t world, rank;
    void*   win[SMOE_MAX_PEERS];   /* win[r]: rank r's window as mapped in THIS process (win[rank] is the local one) */
} smoe_peers;
size_t smoe_xchg_window_bytes(int K_all, int P);
/* The window must be a dedicated allocation (cudaIpc exports whole allocations): the library allocates (and zeroes)
 * it -- the one exception to "never allocates".  export -> 64-byte handle; open -> peer mapping (lazy peer access). */
int smoe_peer_alloc(size_t bytes, void** ptr);
int smoe_peer_free(void* ptr);
int smoe_peer_export(const void* ptr, void* handle64);
int smoe_peer_open(const void* handle64, void** ptr);
int smoe_peer_close(void* ptr);
/* raw_part may be NULL (evaluation pass: only scalars and flags are exchanged). */
int smoe_xchg_publish(const smoe_cfg* cfg, const smoe_peers* peers, const int32_t* counts, int K_all, int num_splits,
                      const float* raw_part, const int32_t* plan /* of smoe_backward, NULL with raw_part == NULL */,
                      const float* scalars, const uint8_t* infl /*[K_all]*/, void* stream);
/* smoe_grad_finalize on the rank-summed statistics; also scalars[0..SMOE_NSCAL) = sum over ranks, infl = any rank. */
int smoe_grad_finalize_peers(const smoe_cfg* cfg, const smoe_peers* peers, int K_cap, const float* theta,
                             const void* quant_ranges, const int32_t* indices, const int32_t* counts, float pis_l1,
                             float l1_norm, float u_l1, float* grads, float* scalars, uint8_t* infl, void* stream);
int smoe_xchg_reduce_tail(const smoe_cfg* cfg, const smoe_peers* peers, int K_all, float* scalars, uint8_t* infl,
                          void* stream);
int smoe_xchg_status(const smoe_peers* peers, int32_t* epoch_and_error /*[2], host memory; synchronous*/);

/* Halo pull for SSIM as the loss on a pixel-sharded model (SURVEY.md 8 f-4: "a 5-pixel halo across shards"; the
 * ring is 10 pixels wide because both the windows of the ring's inner 5 positions and their own 5-pixel support are
 * needed for the gradient of the block's pixels): every rank's `res` buffer covers its block plus the ring and lives
 * in peer-mapped memory (smoe_peer_alloc / _export / _open); after smoe_loss, smoe_halo_pull waits until all ranks
 * have written their blocks (second flag barrier of the windows) and copies the ring from the owners' buffers.
 * Geometry in image coordinates, unused axes [0,1). */
typedef struct smoe_halo_map {
    int32_t world, rank, d, C;
    int32_t blk_lo[SMOE_MAX_PEERS][3], blk_hi[SMOE_MAX_PEERS][3];     /* each rank's block                         */
    int32_t buf_lo[SMOE_MAX_PEERS][3], buf_dims[SMOE_MAX_PEERS][3];   /* each rank's resident buffer: origin, extents */
    void*   res[SMOE_MAX_PEERS];                                      /* each rank's res buffer as mapped here      */
} smoe_halo_map;
int smoe_halo_pull(const smoe_peers* peers, const smoe_halo_map* map, void* stream);

/* Host -> device feed of a pass's target pixels (pinned host memory) on a dedicated copy stream, overlapping whatever
 * the main stream does until smoe_loss: the copy is ordered after the work already enqueued on main_stream
 * (order_event is recorded there and awaited by copy_stream) and done_event fires when the pixels have landed --
 * make the main stream wait for it right before smoe_loss.  The reference feeds its target through the TF feed dict
 * on every session.run (smoe.py:1671-1672, 1702). */
int smoe_feed(void* dst, const void* src_host, size_t bytes, void* main_stream, void* copy_stream,
              void* order_event /* cudaEvent_t */, void* done_event /* cudaEvent_t */);

/* TF1 ApplyAdam on every K_all row (dense, pruned rows included), three groups.  Replaces
 * session.run(train_op) at smoe.py:1788 (apply_gradients at smoe.py:1173-1193). */
int smoe_adam_step(const smoe_cfg* cfg, const smoe_adam* hp, const float* alpha_dev /* optional device [3]:
                   overrides hp->alpha, so that a captured CUDA graph carries no step count */,
                   float* theta, const float* grads, float* adam_m, float* adam_v, int K_all,
                   const uint8_t* infl, uint8_t* kernel_list /* both optional: the same launch also does
                   smoe_update_kernel_list (one-batch models, whose list is rewritten once per step) */, void* stream);

/* custom_ssim (ops/image_ops_impl.py:235-293) as evaluated by the loss graph (smoe.py:993-1010):
 * SYMMETRIC pad 5, 11-tap sigma-1.5 Gaussian window, VALID; out[c] = mean SSIM of channel c.
 * a, b: [dims..][C].  workspace from smoe_ssim_workspace_bytes. */
size_t smoe_ssim_workspace_bytes(int d, const int32_t dims[3], int C);
int    smoe_ssim(int d, const int32_t dims[3], int C, const float* a, const float* b, double* out /*[C]*/,
                 void* workspace, void* stream);

/* SSIM as the training loss (`ssim_opt`, smoe.py:981-1010) on one batch, after smoe_forward and before
 * smoe_backward: per-channel sum over the loss rectangle (the batch minus its halo) of the SSIM map of
 * (res, image), SYMMETRIC-padded by 5 at the rectangle's borders, ACCUMULATED into scalars[8 + c] (the caller
 * divides by the number of positions and forms 1 - sum_c w_c ssim_c); and, when pix != NULL, d loss / d res
 * pushed through the output fake-quant and the clip (straight-through where 0 <= res_pre <= 1) and written
 * over the g_c / gr planes of the backward state that smoe_loss filled for the squared-error loss.
 *   res, image: [dims..][C] as in smoe_loss; res_pre: the rbuf of smoe_forward
 *   region   optional (NULL: the batch's loss rectangle, as above).  Pixel-sharded SSIM: the resident buffers hold the
 *            rank's block PLUS a ring of 10 halo pixels (res pulled from the neighbours by smoe_halo_pull, the target
 *            static); the windows are centred on the positions of `region` (block + ring, clipped to the image, so the
 *            symmetric padding only ever reflects at true image borders), while the SSIM sum and the gradient run over
 *            the batch rectangle only -- every position of the image is counted by exactly one rank, and a window
 *            that straddles a block border sees the neighbour's pixels.  inv_count = 1 / positions of the WHOLE image. */
typedef struct smoe_ssim_region {
    int32_t lo[3], n[3];     /* compute rectangle inside the resident buffer (contains the batch rectangle) */
    float   inv_count;
} smoe_ssim_region;
size_t smoe_ssim_loss_workspace_bytes(const smoe_cfg* cfg, const smoe_batch* batch);
int    smoe_ssim_loss(const smoe_cfg* cfg, const smoe_batch* batch, const smoe_ssim_region* region, const float* res,
                      const float* image, const float* res_pre, float* pix, float* scalars, void* workspace,
                      void* stream);

/* sum over all elements of (a-b)^2 -> out[0] (double accumulation in fixed order);
 * PSNR = 10 log10((2^p)^2 / (mean * (2^p)^2)) on the host (plotter.py:14-15, smoe.py:1053). */
int smoe_sqerr(const float* a, const float* b, size_t n, double* out, void* workspace /* >= 8 KiB */, void* stream);

/* Uniform quantiser of quantizer.py:58-75 / rescale of quantizer.py:124-130 on one tensor of
 * `rows` x `cols` float32 (bounds per column, keepdims semantics of quantizer.py:8-19), IEEE
 * round-to-nearest-even, no FMA contraction: codes are bit-exact with NumPy float32. */
/* `f64` selects the arithmetic NumPy uses at that call site: 0 = float32 (min/max bounds, modes
 * 0/1/3), 1 = float64 (fixed bounds built with np.ones(...)*python_float: mode 2 and quantised
 * pis).  Bounds are passed as double in both cases (float32 values are exact in double); codes /
 * out are float32 arrays when f64 == 0 and float64 arrays when f64 == 1, as in the reference. */
int smoe_quantize(const float* x, const double* lb, const double* ub, int rows, int cols, double step,
                  int f64, void* codes, void* stream);
int smoe_rescale(const void* codes, const double* lb, const double* ub, int rows, int cols, double step,
                 int f64, void* out, void* stream);
/* per-column min / max over rows (np.amin / np.amax axis=0, quantizer.py:8-19), as double */
int smoe_colminmax(const float* x, int rows, int cols, double* lb, double* ub, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SMOE_B200_H */
