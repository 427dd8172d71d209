// Fused SMoE forward (smoe_forward) and the per-pixel loss stage (smoe_loss).  Replace smoe.py:777-858 and
// smoe.py:899-937, 1053.  The forward needs no target pixels: it leaves the mixture output r (before clip) and the
// gate state; smoe_loss then clips, fake-quantises, compares with the target and writes dL/dr for the backward.
// Keeping the two apart lets a step's target arrive from the host WHILE the sweeps run (the end-to-end path).
// smoe_cotangent is the other way into the backward: it writes a caller's dL/dr instead of the library's loss.
//
// Pixel-stationary: a CTA (128 threads, 6 resident per SM for images, 4 for video) owns a spatially compact tile of
// SMOE_TPIX = 512 pixels (4 per thread, in registers) and streams the active kernels past it twice:
//   sweep A  S_n = sum_k 2^{q_k(x_n)}                       (the normaliser of smoe.py:819-821)
//   sweep B  w = 2^{q}/S, m = w > tau, r_c += m*w*E_kc(x)   (smoe.py:823-848; needs the FINAL S,
//            and gates are not renormalised after thresholding, so one sweep is not enough)
// Kernel records arrive in shared memory by TMA bulk copies (cp.async.bulk + mbarrier, double
// buffered) and are re-expressed per tile in tile-centred coordinates, where the whole gate
// logit is one quadratic  q(x') = qc + ql.x' + x'^T qq x'.  The 4 pixels of a thread differ only in
// their first coordinate, so the logit is a parabola  c + (b + qq00 z) z  in z = x'_0 whose
// coefficients cost T+d-2 FFMA once per (thread, kernel) and 2 FFMA per pixel.
// The quadratic form covers both ||A^T(x-mu)||^2 and the train_inverse_cov branch x^T A x.
// The N x K gate matrix is never materialised.  FP32 FFMA + MUFU.EX2; no tensor cores
// (inner dimensions are d = 2..3 and C = 1..3).
//
// Exact work skipping -- every mode returns bit-identical results (tests assert it):
//   * ex2.approx.ftz(q) is exactly +0 for q < -126, and a gate below the threshold multiplies its
//     expert by exactly 0.  Sweep A skips ex2+add for a warp-iteration whose logits are all < -126;
//     sweep B tests the threshold in the log domain, q - log2 S > log2 tau, so it needs no ex2 at all
//     unless a gate passes.                                            (dense_exec = 0 and 2)
//   * Culling: q_k(x) <= c0_k - max(lam_k * dist(x, mu_k)^2, max_l kap_kl * gap_l^2) with lam_k a lower
//     bound of the smallest eigenvalue of Qm_k and kap_kl = 1/(Qm_k^-1)_ll the per-axis bounds.  A chunk of 128
//     kernels whose bound over the tile's box says "all zero"
//     (sweep A: < -126.5; sweep B: < min_n qthr - 0.01) is never loaded, and inside a loaded chunk
//     only the kernels that can matter are re-centred and swept (ordered compaction, so sums keep
//     the order of the dense sweep).  The 0.5 / 0.01 margins cover the rounding of the evaluated
//     logit, which is < 1e-4 there.                                          (dense_exec = 0)
//   * Absorbed terms: sweep A adds the kernels around the tile first (part 1, a geometric rule that is the same in
//     every mode) and everything else afterwards (part 2).  By then S is nearly complete, and a term below half an
//     ulp of the running float32 sum leaves it bit-for-bit unchanged whether it is added or not -- so part 2 is
//     culled against log2 S - 25.5 instead of -126.5.                         (dense_exec = 0 and 2)
#include "smoe_common.cuh"
#include "fwd_records.cuh"

namespace smoe {

// parabola coefficients of q along x'_0 for fixed x'_1.. : q = c + (b + qq00 z) z
template <int D, int C>
__device__ __forceinline__ void parabola(const float* __restrict__ f, const float (&xs)[3], float& c, float& b) {
    using R = Rec<D, C>;
    c = f[R::OC];
#pragma unroll
    for (int l = 1; l < D; ++l) {
        float t = f[R::OL + l];
#pragma unroll
        for (int m = l; m < D; ++m) t = fmaf(f[R::OQ + ut(D, l, m)], xs[m], t);
        c = fmaf(t, xs[l], c);
    }
    b = f[R::OL + 0];
#pragma unroll
    for (int m = 1; m < D; ++m) b = fmaf(f[R::OQ + ut(D, 0, m)], xs[m], b);
}

struct FwdArgs {
    smoe_cfg cfg;
    smoe_batch b;
    const float* packed;
    const int32_t* indices;
    const int32_t* counts;
    const float* chunk_bounds;
    const float* lossw;
    const float* ax[3];
    float* rbuf;
    int32_t* argmax;
    uint8_t* infl;
    float* pix;
    float* tile_qmin;
    unsigned long long* pair_counts;
    int ntiles, nt1, nt2, max_chunks;
    float tau, ltau;
    float eps_cut;          // eps_bits > 0: terms below 2^-eps_cut of the normaliser may be dropped; 0 = exact
};

// COUNT: also count the (pixel, kernel) pairs each sweep evaluates (bench / roofline diagnostics; a separate
// instantiation, so the product path carries no counter).
// AMAX: track the arg-max gate per pixel (only the reconstruction passes ask for it; the training step does not, and
// its instantiation saves the 2 x PPT registers).
#ifndef SMOE_FWD_UNROLL
#define SMOE_FWD_UNROLL 2
#endif
constexpr int kBodyUnroll = SMOE_FWD_UNROLL;
template <int D, int C, bool COUNT, bool AMAX>
__global__ void __launch_bounds__(kThreadsF, (D == 2) ? SMOE_FWD_CTAS_2D : 4) forward_kernel(const FwdArgs a) {
    using R = Rec<D, C>;
    constexpr int PK = pstride(D, C);
    constexpr int PPT = kPixPerThread;
    static_assert(kChunk == kThreadsF, "one kernel of a chunk per thread");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* raw0 = reinterpret_cast<float*>(smem_raw);
    float* raw1 = raw0 + kChunk * PK;
    float* crec = raw1 + kChunk * PK;
    uint64_t* bar = reinterpret_cast<uint64_t*>(crec + kChunk * R::RC);
    float* red = reinterpret_cast<float*>(bar + 2);          // [4 warps][8]
    int* scratch = reinterpret_cast<int*>(red + 32);         // [2][4]
    int* clist = scratch + 8;                                // [max_chunks]

    const int tid = threadIdx.x;
    const int K = a.counts[0];
    const int nchunks = (K + kChunk - 1) / kChunk;
    const int mode = a.cfg.dense_exec;                       // 0 cull+skip, 1 dense, 2 skip only
    const bool cull = mode == 0, skip = mode != 1;
    if (tid == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        fence_barrier_init();
    }
    __syncthreads();
    uint32_t phase0 = 0, phase1 = 0;
    int par = 0;
    unsigned cntA_vis = 0, cntA_ex = 0, cntB_vis = 0, cntB_ex = 0;     // COUNT only

    auto issue = [&](int ci, int buf) {
        int nk = min(kChunk, K - ci * kChunk);
        uint32_t bytes = (uint32_t)nk * PK * 4u;
        fence_proxy_async();
        mbar_expect_tx(&bar[buf], bytes);
        tma_load_1d(buf ? raw1 : raw0, a.packed + (size_t)ci * kChunk * PK, bytes, &bar[buf]);
    };

    const int e1 = a.b.tile[1], e2 = a.b.tile[2];
    for (int tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x) {
        // ---- tile geometry ------------------------------------------------------------
        int tt[3];
        tt[2] = tile % a.nt2;
        tt[1] = (tile / a.nt2) % a.nt1;
        tt[0] = tile / (a.nt2 * a.nt1);
        int lo[3], hi[3];
        float ctr[3], half[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            lo[i] = a.b.origin[i] + tt[i] * a.b.tile[i];
            hi[i] = min(lo[i] + a.b.tile[i], a.b.origin[i] + a.b.extent[i]) - 1;
            const float c0 = (i < D) ? a.ax[i][lo[i]] : 0.f, c1 = (i < D) ? a.ax[i][hi[i]] : 0.f;
            ctr[i] = 0.5f * (c0 + c1);
            half[i] = 0.5f * (c1 - c0) * 1.0001f + 1e-7f;     // box half extent, rounded outwards
        }
        // the thread's PPT pixels: same (i1, i2), rows i0 = p*step + i0_first
        float x0[PPT], xs[3] = {0.f, 0.f, 0.f};
        unsigned okmask = 0;     // bit p: pixel p is inside the batch (and fed); its buffer index is recomputed in the epilogue
        const int gbase12 = ((tid / e2) % e1 + lo[1]) * a.b.dims[2] + (tid % e2 + lo[2]);
        unsigned hmask = 0;      // bit p: pixel p lies in the overlap halo (forwarded, outside the loss crop)
        {
            const int i2 = tid % e2, i1 = (tid / e2) % e1;
            const int g1 = lo[1] + i1, g2 = lo[2] + i2;
            // the halo of overlap_of_batches (smoe.py:909-923) is cropped on every side that is not the image border
            auto in_halo = [&](int ax, int g) {
                const int o = a.b.origin[ax], e = o + a.b.extent[ax];
                return ax < D && ((o > 0 && g < o + a.b.halo) || (e < a.b.dims[ax] && g >= e - a.b.halo));
            };
            const bool h12 = a.b.halo > 0 && (in_halo(1, g1) || in_halo(2, g2));
            if (D > 1) xs[1] = a.ax[1][min(g1, hi[1])] - ctr[1];
            if (D > 2) xs[2] = a.ax[2][min(g2, hi[2])] - ctr[2];
#pragma unroll
            for (int p = 0; p < PPT; ++p) {
                const int j = p * kThreadsF + tid;
                const int i0 = j / (e2 * e1);
                const int g0 = lo[0] + i0;
                const bool ok = g0 <= hi[0] && g1 <= hi[1] && g2 <= hi[2];
                bool fed = ok;
                // a pixel that is not part of this run's feed (random sub-sampling, smoe.py:1664-1667)
                if (a.lossw && ok && a.lossw[g0 * a.b.dims[1] * a.b.dims[2] + gbase12] == SMOE_PIXEL_ABSENT) fed = false;
                if (fed) okmask |= 1u << p;
                if (a.b.halo > 0 && (h12 || in_halo(0, g0))) hmask |= 1u << p;
                x0[p] = a.ax[0][min(g0, hi[0])] - ctr[0];
            }
        }

        // chunk-level culling: ordered list of the chunks whose bound reaches `thr` over this tile.  Sweep A runs in two
        // parts (see there): part 1 takes the NEAR kernels -- those whose logit, by the culling bound, falls by at most
        // kNearCut (log2 units) between the centre and the closest point of the tile's box, a rule that scales with the
        // kernel's own width -- and therefore only the chunks whose bound says they may hold one; part 2 takes all other
        // kernels (any chunk); part 0 = everything.  The split depends on the records and the tile geometry only, not on
        // the execution mode, so the order of summation is the same in every mode.
        auto build_chunk_list = [&](float thr, int part) -> int {
            int n = 0;
            for (int base = 0; base < nchunks; base += kThreadsF) {
                const int ci = base + tid;
                bool need = false;
                if (ci < nchunks) {
                    const float* cb = a.chunk_bounds + (size_t)ci * kCB;
                    float d2 = 0.f, kd = 0.f;
#pragma unroll
                    for (int l = 0; l < D; ++l) {
                        const float mn = cb[l] - ctr[l], mx = cb[3 + l] - ctr[l];
                        const float gap = fmaxf(fmaxf(mn - half[l], -half[l] - mx), 0.f);
                        d2 = fmaf(gap, gap, d2);
                        kd = fmaxf(kd, cb[8 + l] * gap * gap);
                    }
                    const float lam = cb[6], drop = fmaxf(lam * d2, kd);
                    need = part != 1 || !(lam >= 0.f) || !(drop > kNearCut);
                    if (cull && need) need = !(lam >= 0.f) || !(cb[7] - drop < thr);
                }
                int tot;
                const int pos = cta_compact(need, scratch, par, &tot);
                if (need) clist[n + pos] = ci;
                n += tot;
            }
            __syncthreads();
            return n;
        };

        // One sweep over the needed chunks; `body(rec)` is called for every kernel that can matter.  Two CTA
        // barriers per chunk: the one inside cta_compact (which also orders the previous chunk's reads of `crec`
        // before this chunk's writes) and the one that publishes the re-centred records.
        auto sweep = [&](int nlist, float thr, int part, auto&& body) {
            if (tid == 0 && nlist > 0) {
                issue(clist[0], 0);
                if (nlist > 1) issue(clist[1], 1);
            }
            for (int li = 0; li < nlist; ++li) {
                const int buf = li & 1;
                const int ci = clist[li];
                const int nk = min(kChunk, K - ci * kChunk);
                if (buf) { mbar_wait(&bar[1], phase1); phase1 ^= 1; } else { mbar_wait(&bar[0], phase0); phase0 ^= 1; }
                const float* raw = (buf ? raw1 : raw0) + tid * PK;
                bool need = tid < nk;
                float mu[D];
#pragma unroll
                for (int l = 0; l < D; ++l) mu[l] = need ? raw[off_mu(D, C) + l] - ctr[l] : 0.f;
                if (need && (cull || part != 0)) {
                    float d2 = 0.f, kd = 0.f;
#pragma unroll
                    for (int l = 0; l < D; ++l) {
                        const float gap = fmaxf(fabsf(mu[l]) - half[l], 0.f);
                        d2 = fmaf(gap, gap, d2);
                        kd = fmaxf(kd, raw[nparam(D, C) + 1 + l] * gap * gap);
                    }
                    const float lam = raw[nparam(D, C)], drop = fmaxf(lam * d2, kd);
                    if (part != 0) need = (part == 1) == (!(lam >= 0.f) || !(drop > kNearCut));
                    if (need && cull) need = !(lam >= 0.f) || !(raw[off_pi(D, C)] - drop < thr);
                }
                int nneed;
                const int pos = cta_compact(need, scratch, par, &nneed);
                if (need) transform_record<D, C>(raw, mu, ctr, a.indices[ci * kChunk + tid], crec + pos * R::RC);
                __syncthreads();
                if (tid == 0 && li + 2 < nlist) issue(clist[li + 2], buf);
#pragma unroll kBodyUnroll
                for (int kk = 0; kk < nneed; ++kk) body(crec + kk * R::RC);
            }
            __syncthreads();          // the next sweep rebuilds `clist` and re-uses `crec`
        };

        // ---- sweep A: normaliser ------------------------------------------------------
        // Exact mode: a term is skipped only when ex2.approx.ftz returns exactly +0 for it (q < -126).
        // eps mode (opt-in): with L = the tile's minimum of log2 S from the PREVIOUS pass over this batch, terms
        // with q < L - 2 - eps_cut are dropped as well; afterwards min log2 S >= L - 2 is verified (the culled sum
        // is a lower bound of the true one) and the tile is re-swept exactly if the stale L was too optimistic.
        float S[PPT];
        float cutA = -126.5f;
        if (a.eps_cut > 0.f && a.tile_qmin) {
            const float Lprev = a.tile_qmin[tile];
            cutA = fmaxf(cutA, Lprev - 2.0f - a.eps_cut);
            if (!(cutA == cutA)) cutA = -126.5f;
        }
        float Lneed = cutA > -126.5f ? cutA + a.eps_cut : -INFINITY;      // = Lprev - 2
        for (int attempt = 0; attempt < 2; ++attempt) {
#pragma unroll
            for (int p = 0; p < PPT; ++p) S[p] = 0.f;
            float skipA = cutA + 0.5f;
            auto bodyA = [&](const float* rec) {
                float f[4 * R::NG4];
                const float4* r4 = reinterpret_cast<const float4*>(rec);
#pragma unroll
                for (int j = 0; j < R::NG4; ++j) {
                    float4 v = r4[j];
                    f[4 * j] = v.x; f[4 * j + 1] = v.y; f[4 * j + 2] = v.z; f[4 * j + 3] = v.w;
                }
                float cq, bq;
                parabola<D, C>(f, xs, cq, bq);
                float q[PPT];
                float qmax = -INFINITY;
#pragma unroll
                for (int p = 0; p < PPT; ++p) {
                    q[p] = fmaf(fmaf(f[R::OQ], x0[p], bq), x0[p], cq);
                    qmax = fmaxf(qmax, q[p]);
                }
                if (COUNT) cntA_vis += PPT;
                // adding ex2(q) would not change S: it is +0 exactly (q < -126), or -- second part of the sweep --
                // below half an ulp of the running sum (see below)
                if (__builtin_expect(!skip || __any_sync(0xffffffffu, qmax >= skipA), 0)) {
#pragma unroll
                    for (int p = 0; p < PPT; ++p) S[p] += ex2f(q[p]);
                    if (COUNT) cntA_ex += PPT;
                }
            };
            // Part 1: the kernels centred in or right around the tile -- they carry (nearly) all of S.
            sweep(build_chunk_list(cutA, 1), cutA, 1, bodyA);
            // Part 2: all other chunks.  S only grows, and float32 addition absorbs a term below half an ulp of the
            // running sum: with L <= log2 S (now), a term 2^q with q < L - 25 is below 2^(floor(log2 S) - 24), half an ulp of S
            // (the cuts keep 0.25 / 0.5 in hand for the errors of log2f and ex2.approx), and leaves S bit-for-bit unchanged, whether
            // it is added (dense_exec = 1 adds them all, in this same order) or not.  So the remaining kernels are
            // culled against L - 25.5 over the tile instead of -126.5, and a warp skips a kernel when every pixel
            // of it is below its own thread's bound: exact, and most of the far field of sweep A disappears.
            {
                float Lt = INFINITY;
#pragma unroll
                for (int p = 0; p < PPT; ++p)
                    if ((okmask >> p) & 1u) Lt = fminf(Lt, log2f(S[p]));             // log2f(0) = -inf: no bound
                float Lmin = Lt;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) Lmin = fminf(Lmin, __shfl_xor_sync(0xffffffffu, Lmin, o));
                if ((tid & 31) == 0) red[tid >> 5] = Lmin;
                __syncthreads();
                Lmin = fminf(fminf(red[0], red[1]), fminf(red[2], red[3]));
                __syncthreads();
                float cut2 = cutA;
                if (skip && Lmin == Lmin) {
                    cut2 = fmaxf(cutA, Lmin - 25.5f);
                    if (Lt == Lt) skipA = fmaxf(skipA, Lt - 25.25f);
                }
                sweep(build_chunk_list(cut2, 2), cut2, 2, bodyA);
            }
            if (!(Lneed > -INFINITY)) break;                 // exact sweep: done
            float smin = INFINITY;
#pragma unroll
            for (int p = 0; p < PPT; ++p)
                if ((okmask >> p) & 1u) smin = fminf(smin, log2f(fmaxf(S[p], kSFloor)));
            const int bad = __syncthreads_or(smin < Lneed);
            if (!bad) break;
            cutA = -126.5f;                                  // stale bound: exact re-sweep
            Lneed = -INFINITY;
        }

        // ---- sweep B: thresholded gates, experts ----------------------------------------
        float qthr[PPT], r[PPT][C], bestw[PPT];
        int bestk[PPT];
        float qmin = INFINITY;
        unsigned live_mask = 0;          // bit p: S > 1e-11 (smoe.py:821), all that the epilogue needs of S
#pragma unroll
        for (int p = 0; p < PPT; ++p) {
            if (S[p] > kSFloor) live_mask |= 1u << p;
            float Sc = fmaxf(S[p], kSFloor);
            // w = e/S = 2^(q - log2 S) > tau  <=>  q - log2 S > log2 tau = -(precision+1); +inf disables pixels
            // outside the batch.  (qthr holds log2 S: the gate needs no multiplication by tau.)
            qthr[p] = ((okmask >> p) & 1u) ? log2f(Sc) : INFINITY;
            qmin = fminf(qmin, qthr[p]);
            bestw[p] = 0.f;
            bestk[p] = -1;
#pragma unroll
            for (int c = 0; c < C; ++c) r[p][c] = 0.f;
        }
        // tile minimum of qthr: the sweep-B / backward culling threshold
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) qmin = fminf(qmin, __shfl_xor_sync(0xffffffffu, qmin, o));
        if ((tid & 31) == 0) red[tid >> 5] = qmin;
        __syncthreads();
        qmin = fminf(fminf(red[0], red[1]), fminf(red[2], red[3]));
        __syncthreads();
        if (tid == 0 && a.tile_qmin) a.tile_qmin[tile] = qmin;
        {
            const float ltau = a.ltau;                           // log2(tau), an integer
            const float thrB = qmin + ltau - 0.01f;
            const int nlist = build_chunk_list(thrB, 0);
            sweep(nlist, thrB, 0, [&](const float* rec) {
                float f[R::RC];
                const float4* r4 = reinterpret_cast<const float4*>(rec);
#pragma unroll
                for (int j = 0; j < R::NG4; ++j) {
                    float4 v = r4[j];
                    f[4 * j] = v.x; f[4 * j + 1] = v.y; f[4 * j + 2] = v.z; f[4 * j + 3] = v.w;
                }
                float cq, bq;
                parabola<D, C>(f, xs, cq, bq);
                float q[PPT];            // gate logit relative to the pixel's normaliser: q - log2 S
                bool any = false;
#pragma unroll
                for (int p = 0; p < PPT; ++p) {
                    q[p] = fmaf(fmaf(f[R::OQ], x0[p], bq), x0[p], cq) - qthr[p];
                    any |= (q[p] > ltau);
                }
                if (COUNT) cntB_vis += PPT;
                if (__builtin_expect(!skip || __any_sync(0xffffffffu, any), 0)) {
                    if (COUNT) cntB_ex += PPT;
#pragma unroll
                    for (int j = R::NG4; j < (R::OK + 4) / 4; ++j) {
                        float4 v = r4[j];
                        f[4 * j] = v.x; f[4 * j + 1] = v.y; f[4 * j + 2] = v.z; f[4 * j + 3] = v.w;
                    }
                    const int korig = __float_as_int(f[R::OK]);
                    // expert value E_c(x) = nu'_c + gamma_c . x': the part that does not depend on x'_0 once per
                    // (thread, kernel), one FFMA per pixel and channel
                    float Eb[C];
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        Eb[c] = f[R::ONU + c];
#pragma unroll
                        for (int l = 1; l < D; ++l) Eb[c] = fmaf(f[R::OGA + l * C + c], xs[l], Eb[c]);
                    }
#pragma unroll
                    for (int p = 0; p < PPT; ++p) {
                        // w = e/S = 2^(q - log2 S), the form the backward recomputes
                        const float w = ex2f(q[p]);
                        const bool pass = q[p] > ltau;
                        const float wm = pass ? w : 0.f;
#pragma unroll
                        for (int c = 0; c < C; ++c) r[p][c] = fmaf(wm, fmaf(f[R::OGA + c], x0[p], Eb[c]), r[p][c]);
                        // tf.argmax keeps the first maximum in ascending kernel index; records arrive in the
                        // (Hilbert) packing order, so ties are broken on the original index explicitly
                        if (AMAX && pass && (w > bestw[p] || (w == bestw[p] && korig < bestk[p]))) { bestw[p] = w; bestk[p] = korig; }
                    }
                    if (any && a.infl) a.infl[korig] = 1;
                }
            });
        }

        // ---- epilogue: mixture output and gate state for the loss stage / the backward ---------
#pragma unroll
        for (int p = 0; p < PPT; ++p) {
            const int j = p * kThreadsF + tid;
            const bool inb = (okmask >> p) & 1u;
            // linear pixel index in the image buffer (< 2^31, checked by the host)
            const int gpix = (lo[0] + j / (e2 * e1)) * a.b.dims[1] * a.b.dims[2] + gbase12;
            // a pixel of the overlap halo (smoe.py:909-923) is the interior of another window, which writes it
            const bool halo = ((hmask >> p) & 1u) || (a.lossw && inb && a.lossw[gpix] == SMOE_PIXEL_HALO);
            if (inb && !halo) {
#pragma unroll
                for (int c = 0; c < C; ++c) a.rbuf[(size_t)gpix * C + c] = r[p][c];
                if (AMAX) a.argmax[gpix] = bestk[p];
            }
            if (a.pix) {
                // planes [z | qthr | live][512] + row constants; coordinates are stored for every slot.  The gr plane
                // carries "S > 1e-11" (smoe.py:821) to smoe_loss, which replaces it by gr and fills the g_c planes.
                const int RLf = a.b.tile[D - 1];
                float* tp = a.pix + (size_t)tile * pix_stride(D, C, RLf);
                tp[PL_Z * SMOE_TPIX + j] = D == 1 ? x0[p] : xs[D - 1];
                tp[PL_QTHR * SMOE_TPIX + j] = inb ? qthr[p] : INFINITY;   // outside the batch: w = 2^(-inf) = 0
                tp[PL_GR * SMOE_TPIX + j] = (inb && ((live_mask >> p) & 1u)) ? 1.f : 0.f;
                if (D > 1 && j % RLf == 0) {
                    const int row = j / RLf, nrows = SMOE_TPIX / RLf;
                    tp[pix_rowc_offset(C) + row] = x0[p];
#pragma unroll
                    for (int l = 1; l < D - 1; ++l) tp[pix_rowc_offset(C) + l * nrows + row] = xs[l];
                }
            }
        }
    }

    if (COUNT) {
        // executed-pair counters: lanes x pixels per sweep; integer atomics, order-independent
        unsigned long long v[4] = {cntA_vis, cntA_ex, cntB_vis, cntB_ex};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v[q] += __shfl_down_sync(0xffffffffu, v[q], o);
            if ((tid & 31) == 0) atomicAdd(&a.pair_counts[q], v[q]);
        }
    }

}

// ---- loss stage -------------------------------------------------------------------------------------------
// Per pixel of the batch (smoe.py:857, 899-937, 1053): res = fake_quant(clip(r)), diff = res - target, the loss and
// squared-error partial sums, and dL/dr (straight-through where 0 <= r <= 1) for the backward: g_c and gr = sum_c g_c r_c
// into the pixel-state planes the forward prepared.  Elementwise and HBM-bound: reads r (C floats), the target (C bytes
// or floats), writes res (C floats) and 1 + C plane values per pixel.  Persistent grid, one fixed-order partial per CTA,
// summed by the last CTA -- no float atomics, deterministic.
struct LossArgs {
    smoe_cfg cfg;
    smoe_batch b;
    const float* rbuf;
    const float* image;
    const uint8_t* image_u8;
    const float* lossw;
    float* res;
    float* pix;
    float* scalars;
    float* partials;
    int32_t* ticket;
    int ntiles, nt1, nt2, pix_tstride;
    float eps, q_scale, q_inv_scale;
};

template <int C>
__global__ void __launch_bounds__(256) loss_kernel(const LossArgs a) {
    const int tid = threadIdx.x;
    const int e1 = a.b.tile[1], e2 = a.b.tile[2];
    const int D = a.cfg.d;
    float lsum[C];
#pragma unroll
    for (int c = 0; c < C; ++c) lsum[c] = 0.f;
    float sqsum = 0.f;
    int nonfinite = 0;
    {
        // one tile per CTA: blockIdx.y = first tile coordinate, blockIdx.x = the other two (no per-pixel divisions)
        int tt[3], lo[3], hi[3];
        tt[0] = blockIdx.y;
        tt[1] = a.nt2 == 1 ? (int)blockIdx.x : (int)blockIdx.x / a.nt2;
        tt[2] = a.nt2 == 1 ? 0 : (int)blockIdx.x % a.nt2;
        const int tile = (tt[0] * a.nt1 + tt[1]) * a.nt2 + tt[2];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            lo[i] = a.b.origin[i] + tt[i] * a.b.tile[i];
            hi[i] = min(lo[i] + a.b.tile[i], a.b.origin[i] + a.b.extent[i]) - 1;
        }
        auto in_halo = [&](int ax, int g) {
            const int o = a.b.origin[ax], e = o + a.b.extent[ax];
            return ax < D && ((o > 0 && g < o + a.b.halo) || (e < a.b.dims[ax] && g >= e - a.b.halo));
        };
        float* tp = a.pix ? a.pix + (size_t)tile * a.pix_tstride : nullptr;
        // slot j = i0 * (e1 e2) + i1 * e2 + i2 of the tile, as the forward numbers them; 256 is a multiple of e1 e2,
        // so a thread keeps its (i1, i2) and steps through i0
        const int i2 = tid % e2, i1 = (tid / e2) % e1;
        const int g1 = lo[1] + i1, g2 = lo[2] + i2;
        const bool in12 = g1 <= hi[1] && g2 <= hi[2];
        const bool halo12 = a.b.halo > 0 && (in_halo(1, g1) || in_halo(2, g2));
        const int rows_per_pass = 256 / (e1 * e2);
        int g0 = lo[0] + tid / (e1 * e2);
        for (int j = tid; j < SMOE_TPIX; j += 256, g0 += rows_per_pass) {
            bool inb = in12 && g0 <= hi[0];
            const int gpix = inb ? (g0 * a.b.dims[1] + g1) * a.b.dims[2] + g2 : 0;
            // per-pixel loss weight (loss_mask, smoe.py:932, 1674-1677), or a sentinel: pixel not fed at all (random
            // sub-sampling, smoe.py:1664-1667) / fed but cropped away before the loss (overlap halo, smoe.py:909-923)
            const float lwv = (a.lossw && inb) ? a.lossw[gpix] : 1.f;
            if (lwv == SMOE_PIXEL_ABSENT) inb = false;
            const bool halo = lwv == SMOE_PIXEL_HALO || halo12 || (a.b.halo > 0 && in_halo(0, g0));
            float g[C], gr = 0.f;
#pragma unroll
            for (int c = 0; c < C; ++c) g[c] = 0.f;
            if (inb && !halo) {
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const size_t gi = (size_t)gpix * C + c;
                    const float rv = a.rbuf[gi];
                    if (!(fabsf(rv) <= 3.0e38f)) nonfinite = 1;
                    const float rc = fminf(fmaxf(rv, 0.f), 1.f);                        // smoe.py:857
                    const float kq = floorf(__fadd_rn(__fmul_rn(rc, a.q_inv_scale), 0.5f));
                    const float rq = __fmul_rn(kq, a.q_scale);                          // smoe.py:899
                    // 8-bit feed: the /255 of utils.py:126-128 (float32 division) happens here
                    const float tgt = a.image_u8 ? __fdiv_rn((float)a.image_u8[gi], 255.0f) : a.image[gi];
                    const float diff = __fsub_rn(rq, tgt);                              // smoe.py:905
                    const float ad = fabsf(diff) - a.eps;                               // smoe.py:932
                    sqsum = fmaf(diff, diff, sqsum);
                    lsum[c] = a.lossw ? fmaf(ad * ad, lwv, lsum[c]) : fmaf(ad, ad, lsum[c]);
                    const float cw = a.cfg.use_yuv ? (c == 0 ? 0.75f : 0.125f) : (1.0f / C);
                    const float sgn = diff > 0.f ? 1.f : (diff < 0.f ? -1.f : 0.f);
                    const bool ste = (rv >= 0.f) && (rv <= 1.f);                        // clip + fake-quant STE
                    g[c] = ste ? 2.f * ad * sgn * cw * a.b.inv_count : 0.f;
                    if (a.lossw) g[c] *= lwv;
                    gr = fmaf(g[c], rv, gr);
                    if (a.res) a.res[gi] = rq;
                }
            }
            if (tp) {
                const bool live = tp[PL_GR * SMOE_TPIX + j] != 0.f;                      // S > 1e-11, left by the forward
                tp[PL_GR * SMOE_TPIX + j] = live ? gr : 0.f;
#pragma unroll
                for (int c = 0; c < C; ++c) tp[(PL_G + c) * SMOE_TPIX + j] = g[c];
            }
        }
    }
    // partials: warp shuffle -> CTA -> fixed-order sum by the last CTA (thread t adds the CTA partials t, t+256, ...
    // in order, then a fixed tree over the 256 threads)
    __shared__ float red[8][8];
    __shared__ float tree[256];
    __shared__ int s_last;
    const int nblk = gridDim.x * gridDim.y, bid = blockIdx.y * gridDim.x + blockIdx.x;
    float vals[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) vals[q] = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) vals[c] = lsum[c];
    vals[4] = sqsum;
    vals[5] = (float)nonfinite;
#pragma unroll
    for (int q = 0; q < 6; ++q)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) vals[q] += __shfl_down_sync(0xffffffffu, vals[q], o);
    if ((tid & 31) == 0)
#pragma unroll
        for (int q = 0; q < 8; ++q) red[tid >> 5][q] = vals[q];
    __syncthreads();
    if (tid < 8) {
        float s = 0.f;
        for (int wv = 0; wv < 8; ++wv) s += red[wv][tid];
        a.partials[(size_t)bid * 8 + tid] = s;
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = (atomicAdd(a.ticket, 1) == nblk - 1);
    __syncthreads();
    if (s_last) {
        __threadfence();
        for (int q = 0; q < 6; ++q) {
            float s = 0.f;
            for (int bq = tid; bq < nblk; bq += 256) s += __ldcg(&a.partials[(size_t)bq * 8 + q]);
            tree[tid] = s;
            __syncthreads();
            for (int o = 128; o > 0; o >>= 1) {
                if (tid < o) tree[tid] += tree[tid + o];
                __syncthreads();
            }
            if (tid == 0) a.scalars[q] += tree[0];
            __syncthreads();
        }
        if (tid == 0) *a.ticket = 0;
    }
}

// ---- cotangent stage --------------------------------------------------------------------------------------
// The alternative to loss_kernel before the backward when the loss lives outside the library: an arbitrary dL/dr
// (grad_r, same layout as rbuf) goes into the g_c / gr planes of the pixel state.  Same launch geometry and slot
// numbering as loss_kernel, and the same arithmetic for gr (fmaf over the channels in order, from 0), so a grad_r
// equal to what loss_kernel derives yields the same planes bit for bit.  Elementwise, HBM-bound: reads grad_r and r
// (C floats each) and the "S > 1e-11" flag, writes 1 + C plane values per pixel.  No reduction, no atomics.
struct CotArgs {
    smoe_batch b;
    const float* rbuf;
    const float* grad_r;
    float* pix;
    int nt1, nt2, pix_tstride;
};

template <int C>
__global__ void __launch_bounds__(256) cotangent_kernel(const CotArgs a) {
    const int tid = threadIdx.x;
    const int e1 = a.b.tile[1], e2 = a.b.tile[2];
    int tt[3], lo[3], hi[3];
    tt[0] = blockIdx.y;
    tt[1] = a.nt2 == 1 ? (int)blockIdx.x : (int)blockIdx.x / a.nt2;
    tt[2] = a.nt2 == 1 ? 0 : (int)blockIdx.x % a.nt2;
    const int tile = (tt[0] * a.nt1 + tt[1]) * a.nt2 + tt[2];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        lo[i] = a.b.origin[i] + tt[i] * a.b.tile[i];
        hi[i] = min(lo[i] + a.b.tile[i], a.b.origin[i] + a.b.extent[i]) - 1;
    }
    float* tp = a.pix + (size_t)tile * a.pix_tstride;
    const int i2 = tid % e2, i1 = (tid / e2) % e1;
    const int g1 = lo[1] + i1, g2 = lo[2] + i2;
    const bool in12 = g1 <= hi[1] && g2 <= hi[2];
    const int rows_per_pass = 256 / (e1 * e2);
    int g0 = lo[0] + tid / (e1 * e2);
    for (int j = tid; j < SMOE_TPIX; j += 256, g0 += rows_per_pass) {
        const bool inb = in12 && g0 <= hi[0];
        const int gpix = inb ? (g0 * a.b.dims[1] + g1) * a.b.dims[2] + g2 : 0;
        float g[C], gr = 0.f;
#pragma unroll
        for (int c = 0; c < C; ++c) g[c] = 0.f;
        if (inb) {
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const size_t gi = (size_t)gpix * C + c;
                g[c] = a.grad_r[gi];
                gr = fmaf(g[c], a.rbuf[gi], gr);
            }
        }
        // g_c reaches the gate gradients of a clamped pixel too; gr only where S > 1e-11 (smoe.py:821)
        const bool live = tp[PL_GR * SMOE_TPIX + j] != 0.f;
        tp[PL_GR * SMOE_TPIX + j] = live ? gr : 0.f;
#pragma unroll
        for (int c = 0; c < C; ++c) tp[(PL_G + c) * SMOE_TPIX + j] = g[c];
    }
}

template <int D, int C>
static size_t fwd_smem_bytes(int max_chunks) {
    return (size_t)(2 * kChunk * pstride(D, C) + kChunk * Rec<D, C>::RC) * 4 + 2 * 8 + 32 * 4 + 8 * 4 +
           (size_t)max_chunks * 4 + 64;
}

}  // namespace smoe

using namespace smoe;

extern "C" int smoe_forward(const smoe_cfg* cfg, const smoe_batch* batch, const float* packed, const int32_t* indices,
                            const int32_t* counts, const float* chunk_bounds, int K_cap, const float* loss_weights,
                            const float* ax0, const float* ax1, const float* ax2, float* rbuf, int32_t* argmax,
                            uint8_t* infl, float* pix, float* tile_qmin, unsigned long long* pair_counts, void* stream) {
    SMOE_REQUIRE(cfg && batch && packed && indices && counts && chunk_bounds && ax0 && ax1 && rbuf, "null argument");
    SMOE_REQUIRE(K_cap > 0, "K_cap must be positive");
    SMOE_REQUIRE(cfg->d == 2 || ax2, "ax2 required for d == 3");
    SMOE_REQUIRE(batch->tile[0] * batch->tile[1] * batch->tile[2] == SMOE_TPIX, "tile product must be SMOE_TPIX");
    SMOE_REQUIRE(kThreadsF % (batch->tile[1] * batch->tile[2]) == 0 && batch->tile[cfg->d - 1] % 4 == 0,
                 "tile[1]*tile[2] must divide 128 and the last tile extent must be a multiple of 4");
    SMOE_REQUIRE(!pix || tile_qmin, "tile_qmin is required with pix");
    SMOE_REQUIRE(batch->halo >= 0, "negative halo");
    SMOE_REQUIRE(cfg->eps_bits == 0 || (cfg->eps_bits >= 24 && cfg->eps_bits <= 126), "eps_bits must be 0 or in [24, 126]");
    SMOE_REQUIRE(cfg->eps_bits == 0 || cfg->dense_exec == 0, "eps_bits needs dense_exec == 0");
    for (int i = 0; i < 3; ++i)
        SMOE_REQUIRE(batch->extent[i] > 0 && batch->origin[i] >= 0 && batch->origin[i] + batch->extent[i] <= batch->dims[i],
                     "batch rectangle outside the image");
    SMOE_REQUIRE(cfg->d == 3 || (batch->dims[2] == 1 && batch->tile[2] == 1), "d == 2 needs dims[2] == tile[2] == 1");
    SMOE_REQUIRE((long long)batch->dims[0] * batch->dims[1] * batch->dims[2] < (1ll << 31), "more than 2^31 pixels");
    FwdArgs a;
    a.cfg = *cfg;
    a.b = *batch;
    a.packed = packed; a.indices = indices; a.counts = counts; a.chunk_bounds = chunk_bounds;
    a.lossw = loss_weights;
    a.ax[0] = ax0; a.ax[1] = ax1; a.ax[2] = ax2 ? ax2 : ax0;
    a.rbuf = rbuf; a.argmax = argmax; a.infl = infl; a.pix = pix; a.tile_qmin = tile_qmin;
    a.pair_counts = pair_counts;
    a.nt1 = (batch->extent[1] + batch->tile[1] - 1) / batch->tile[1];
    a.nt2 = (batch->extent[2] + batch->tile[2] - 1) / batch->tile[2];
    a.ntiles = smoe_num_tiles(batch);
    a.max_chunks = (K_cap + kChunk - 1) / kChunk;
    const float two_p = (float)(1 << cfg->precision);
    a.tau = 0.5f / two_p;
    a.ltau = -(float)(cfg->precision + 1);          // log2(tau), exact
    a.eps_cut = (float)cfg->eps_bits;
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int per_sm = cfg->d == 2 ? SMOE_FWD_CTAS_2D : 4;          // resident CTAs per SM (matches __launch_bounds__)
    int grid = a.ntiles < per_sm * sms ? a.ntiles : per_sm * sms;
    cudaStream_t st = (cudaStream_t)stream;
#define LAUNCH(D, C, CNT, AM)                                                                                       \
    {                                                                                                               \
        size_t sm = fwd_smem_bytes<D, C>(a.max_chunks);                                                             \
        SMOE_REQUIRE(sm <= 200 * 1024, "too many kernel chunks for the shared-memory chunk list");                  \
        cudaFuncSetAttribute(forward_kernel<D, C, CNT, AM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);  \
        forward_kernel<D, C, CNT, AM><<<grid, kThreadsF, sm, st>>>(a);                                              \
    }
#define CALL(D, C)                                                               \
    if (pair_counts) { if (argmax) LAUNCH(D, C, true, true) else LAUNCH(D, C, true, false) } \
    else { if (argmax) LAUNCH(D, C, false, true) else LAUNCH(D, C, false, false) }
    SMOE_DISPATCH_DC(cfg->d, cfg->C, CALL)
#undef CALL
#undef LAUNCH
    return check_launch("smoe_forward");
}

extern "C" int smoe_loss_partials(const smoe_batch* batch) {
    return batch ? smoe_num_tiles(batch) : 0;          // one CTA per tile; 8 floats each
}

extern "C" int smoe_loss(const smoe_cfg* cfg, const smoe_batch* batch, const float* rbuf, const float* image,
                         const uint8_t* image_u8, const float* loss_weights, float* res, float* pix, float* scalars,
                         float* partials, int32_t* ticket, void* stream) {
    SMOE_REQUIRE(cfg && batch && rbuf && scalars && partials && ticket, "null argument");
    SMOE_REQUIRE((image != nullptr) != (image_u8 != nullptr), "exactly one of image / image_u8");
    SMOE_REQUIRE(batch->tile[0] * batch->tile[1] * batch->tile[2] == SMOE_TPIX, "tile product must be SMOE_TPIX");
    SMOE_REQUIRE(cfg->C == 1 || cfg->C == 3, "1 or 3 channels");
    SMOE_REQUIRE(256 % (batch->tile[1] * batch->tile[2]) == 0, "tile[1]*tile[2] must divide 256");
    LossArgs a;
    a.cfg = *cfg;
    a.b = *batch;
    a.rbuf = rbuf; a.image = image; a.image_u8 = image_u8; a.lossw = loss_weights; a.res = res; a.pix = pix;
    a.scalars = scalars; a.partials = partials; a.ticket = ticket;
    a.nt1 = (batch->extent[1] + batch->tile[1] - 1) / batch->tile[1];
    a.nt2 = (batch->extent[2] + batch->tile[2] - 1) / batch->tile[2];
    a.ntiles = smoe_num_tiles(batch);
    a.pix_tstride = pix_stride(cfg->d, cfg->C, batch->tile[cfg->d - 1]);
    const float two_p = (float)(1 << cfg->precision);
    a.eps = cfg->margin / two_p;
    a.q_scale = 1.0f / (two_p - 1.0f);
    a.q_inv_scale = 1.0f / a.q_scale;
    const int nt0 = a.ntiles / (a.nt1 * a.nt2);
    SMOE_REQUIRE(nt0 <= 65535, "too many tiles along the first axis");
    const dim3 grid(a.nt1 * a.nt2, nt0);
    if (cfg->C == 1) loss_kernel<1><<<grid, 256, 0, (cudaStream_t)stream>>>(a);
    else loss_kernel<3><<<grid, 256, 0, (cudaStream_t)stream>>>(a);
    return check_launch("smoe_loss");
}

extern "C" int smoe_cotangent(const smoe_cfg* cfg, const smoe_batch* batch, const float* rbuf, const float* grad_r,
                              float* pix, void* stream) {
    SMOE_REQUIRE(cfg && batch && rbuf && grad_r && pix, "null argument");
    SMOE_REQUIRE(batch->tile[0] * batch->tile[1] * batch->tile[2] == SMOE_TPIX, "tile product must be SMOE_TPIX");
    SMOE_REQUIRE(batch->halo == 0, "halo must be 0: the cotangent covers the whole batch rectangle");
    SMOE_REQUIRE((cfg->d == 2 || cfg->d == 3) && (cfg->C == 1 || cfg->C == 3), "d in {2, 3} and 1 or 3 channels");
    SMOE_REQUIRE(256 % (batch->tile[1] * batch->tile[2]) == 0, "tile[1]*tile[2] must divide 256");
    CotArgs a;
    a.b = *batch;
    a.rbuf = rbuf; a.grad_r = grad_r; a.pix = pix;
    a.nt1 = (batch->extent[1] + batch->tile[1] - 1) / batch->tile[1];
    a.nt2 = (batch->extent[2] + batch->tile[2] - 1) / batch->tile[2];
    a.pix_tstride = pix_stride(cfg->d, cfg->C, batch->tile[cfg->d - 1]);
    const int nt0 = smoe_num_tiles(batch) / (a.nt1 * a.nt2);
    SMOE_REQUIRE(nt0 <= 65535, "too many tiles along the first axis");
    const dim3 grid(a.nt1 * a.nt2, nt0);
    if (cfg->C == 1) cotangent_kernel<1><<<grid, 256, 0, (cudaStream_t)stream>>>(a);
    else cotangent_kernel<3><<<grid, 256, 0, (cudaStream_t)stream>>>(a);
    return check_launch("smoe_cotangent");
}
