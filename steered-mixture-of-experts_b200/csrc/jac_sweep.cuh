// The chunk sweep of the pixel-stationary derivative kernels (jacobian.cu: the spatial Jacobian; jvp.cu: the
// Jacobian-vector products): smoe_point_xgrad's TMA chunk staging and culling at the exact-zero cut, with an optional
// second record stream (the parameter tangents of smoe_jvp) staged next to the primal chunk.
#pragma once
#include "pt_state.cuh"

namespace smoe {

struct JacArgs {
    smoe_cfg cfg;
    smoe_batch b;              // grid sweeps only
    const float* packed;
    const int32_t* counts;
    const float* chunk_bounds;
    const float* state;        // point sweeps: [ntiles][pt_stride], as smoe_point_forward left it;
                               // grid sweeps: pix [ntiles][pix_stride], as smoe_forward left it
    const float* tile_box;     // point sweeps: [ntiles][kTB]; grid sweeps: tile_qmin [ntiles]
    const float* ax[3];        // grid sweeps only
    const float* r;            // [n][C]: tile order (points) or the grid's rbuf
    float* jac;                // [n][C][d], the layout of r (the Jacobian only)
    int n, ntiles, nt1, nt2;
    float ltau;
};

// Shared memory of a sweep: two raw chunks, the compute records, XF floats of the caller (the tangent chunks of
// smoe_jvp), barriers, `red`, `scratch`, chunk list.
struct JacSmem {
    float *raw0, *raw1, *crec;
    uint64_t* bar;
    int *scratch, *clist;
    uint32_t phase0, phase1;
    int par;
    const float* tangent;          // smoe_jvp: the raw tangent records, staged in traw0 / traw1, re-centred into trec
    float *traw0, *traw1, *trec;
};

template <int D, int C, int XF = 0>
__device__ __forceinline__ JacSmem jac_smem_init() {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    JacSmem s;
    s.raw0 = reinterpret_cast<float*>(smem_raw);
    s.raw1 = s.raw0 + kChunk * pstride(D, C);
    s.crec = s.raw1 + kChunk * pstride(D, C);
    s.bar = reinterpret_cast<uint64_t*>(s.crec + kChunk * Rec<D, C>::RC + XF);
    s.scratch = reinterpret_cast<int*>(reinterpret_cast<float*>(s.bar + 2) + 32);
    s.clist = s.scratch + 8;
    if (threadIdx.x == 0) {
        mbar_init(&s.bar[0], 1);
        mbar_init(&s.bar[1], 1);
        fence_barrier_init();
    }
    __syncthreads();
    s.phase0 = s.phase1 = 0;
    s.par = 0;
    return s;
}

// Raw tangent record of smoe_pack_tangent, one per packed row: d mu | d Qm (upper-tri, log2 units) | d c0 | d nu |
// d gamma at the offsets of a packed record, padded to a multiple of 4 floats (TMA rows of 16 bytes).
__host__ __device__ constexpr int tan_stride(int d, int C) { return (nparam(d, C) + 3) / 4 * 4; }

// Raw tangent record + primal record + tile centre -> the tangent of the tile-centred compute record, in Rec's
// layout: with delta = ctr - mu = -mu', d qq = -dQm, d ql = 2 (Qm dmu - dQm delta),
// d qc = dc0 - delta^T dQm delta + 2 dmu^T Qm delta, d nu' = dnu + dgamma^T ctr, d gamma.
template <int D, int C>
__device__ __forceinline__ void transform_tangent(const float* __restrict__ raw, const float* __restrict__ traw,
                                                  const float (&mu)[D], const float (&ctr)[3], float* __restrict__ dst) {
    using R = Rec<D, C>;
    float out[R::RC];
    float Qm[D][D], dQ[D][D], dmu[D];
#pragma unroll
    for (int l = 0; l < D; ++l) {
        dmu[l] = traw[off_mu(D, C) + l];
#pragma unroll
        for (int m = l; m < D; ++m) {
            Qm[l][m] = Qm[m][l] = raw[off_A(D, C) + ut(D, l, m)];
            dQ[l][m] = dQ[m][l] = traw[off_A(D, C) + ut(D, l, m)];
        }
    }
    float dqc = traw[off_pi(D, C)];
#pragma unroll
    for (int l = 0; l < D; ++l) {
        float a = 0.f, b = 0.f, qd = 0.f;          // (dQm mu')_l, (Qm mu')_l, (Qm dmu)_l
#pragma unroll
        for (int m = 0; m < D; ++m) {
            a = fmaf(dQ[l][m], mu[m], a);
            b = fmaf(Qm[l][m], mu[m], b);
            qd = fmaf(Qm[l][m], dmu[m], qd);
        }
        dqc = fmaf(-mu[l], a, dqc);
        dqc = fmaf(-2.f * dmu[l], b, dqc);
        out[R::OL + l] = 2.f * (qd + a);
#pragma unroll
        for (int m = l; m < D; ++m) out[R::OQ + ut(D, l, m)] = (l == m) ? -dQ[l][m] : -2.f * dQ[l][m];
    }
    out[R::OC] = dqc;
#pragma unroll
    for (int c = 0; c < C; ++c) {
        float nu = traw[off_nu(D, C) + c];
#pragma unroll
        for (int l = 0; l < D; ++l) {
            const float g = traw[off_ga(D, C) + l * C + c];
            nu = fmaf(g, ctr[l], nu);
            out[R::OGA + l * C + c] = g;
        }
        out[R::ONU + c] = nu;
    }
#pragma unroll
    for (int j = R::OK; j < R::RC; ++j) out[j] = 0.f;
    float4* d4 = reinterpret_cast<float4*>(dst);
#pragma unroll
    for (int j = 0; j < R::RC / 4; ++j) d4[j] = make_float4(out[4 * j], out[4 * j + 1], out[4 * j + 2], out[4 * j + 3]);
}

// One tile's sweep, smoe_point_xgrad's staging and culling: the ordered list of chunks whose bound over the box
// (ctr, half) reaches `thr`, TMA double buffering, per-kernel culling and ordered compaction; body(rec) -- with TAN
// body(rec, trec) -- is called for every kernel that can matter, in packed order, with its tile-centred
// record (and its tangent).  With TAN the raw tangent records of smoe_pack_tangent (s.tangent) ride on the primal
// chunk's barrier into s.traw0 / s.traw1 and are re-centred per tile into s.trec.  Ends with a CTA barrier.
template <int D, int C, bool TAN = false, class Body>
__device__ __forceinline__ void jac_sweep(const JacArgs& a, JacSmem& s, int K, bool cull, const float (&ctr)[3],
                                          const float (&half)[3], float thr, Body&& body) {
    using R = Rec<D, C>;
    constexpr int PK = pstride(D, C);
    constexpr int TS = tan_stride(D, C);
    const int tid = threadIdx.x;
    const int nchunks = (K + kChunk - 1) / kChunk;
    auto issue = [&](int ci, int buf) {
        int nk = min(kChunk, K - ci * kChunk);
        uint32_t bytes = (uint32_t)nk * PK * 4u;
        const uint32_t tbytes = TAN ? (uint32_t)nk * TS * 4u : 0u;
        fence_proxy_async();
        mbar_expect_tx(&s.bar[buf], bytes + tbytes);
        tma_load_1d(buf ? s.raw1 : s.raw0, a.packed + (size_t)ci * kChunk * PK, bytes, &s.bar[buf]);
        if constexpr (TAN)
            tma_load_1d(buf ? s.traw1 : s.traw0, s.tangent + (size_t)ci * kChunk * TS, tbytes, &s.bar[buf]);
    };
    int nlist = 0;
    for (int base = 0; base < nchunks; base += kThreadsF) {
        const int ci = base + tid;
        bool need = ci < nchunks;
        if (need && cull) {
            const float* cb = a.chunk_bounds + (size_t)ci * kCB;
            float d2 = 0.f, kd = 0.f;
#pragma unroll
            for (int l = 0; l < D; ++l) {
                const float mn = cb[l] - ctr[l], mx = cb[3 + l] - ctr[l];
                const float gap = fmaxf(fmaxf(mn - half[l], -half[l] - mx), 0.f);
                d2 = fmaf(gap, gap, d2);
                kd = fmaxf(kd, cb[8 + l] * gap * gap);
            }
            const float lam = cb[6];
            need = !(lam >= 0.f) || !(cb[7] - fmaxf(lam * d2, kd) < thr);
        }
        int tot;
        const int pos = cta_compact(need, s.scratch, s.par, &tot);
        if (need) s.clist[nlist + pos] = ci;
        nlist += tot;
    }
    __syncthreads();

    if (tid == 0 && nlist > 0) {
        issue(s.clist[0], 0);
        if (nlist > 1) issue(s.clist[1], 1);
    }
    for (int li = 0; li < nlist; ++li) {
        const int buf = li & 1;
        const int ci = s.clist[li];
        const int nk = min(kChunk, K - ci * kChunk);
        if (buf) { mbar_wait(&s.bar[1], s.phase1); s.phase1 ^= 1; } else { mbar_wait(&s.bar[0], s.phase0); s.phase0 ^= 1; }
        const float* raw = (buf ? s.raw1 : s.raw0) + tid * PK;
        bool need = tid < nk;
        float mu[D];
#pragma unroll
        for (int l = 0; l < D; ++l) mu[l] = need ? raw[off_mu(D, C) + l] - ctr[l] : 0.f;
        if (need && cull) {
            float d2 = 0.f, kd = 0.f;
#pragma unroll
            for (int l = 0; l < D; ++l) {
                const float gap = fmaxf(fabsf(mu[l]) - half[l], 0.f);
                d2 = fmaf(gap, gap, d2);
                kd = fmaxf(kd, raw[nparam(D, C) + 1 + l] * gap * gap);
            }
            const float lam = raw[nparam(D, C)];
            need = !(lam >= 0.f) || !(raw[off_pi(D, C)] - fmaxf(lam * d2, kd) < thr);
        }
        int nneed;
        const int pos = cta_compact(need, s.scratch, s.par, &nneed);
        if (need) {
            transform_record<D, C>(raw, mu, ctr, 0, s.crec + pos * R::RC);
            if constexpr (TAN)
                transform_tangent<D, C>(raw, (buf ? s.traw1 : s.traw0) + tid * TS, mu, ctr, s.trec + pos * R::RC);
        }
        __syncthreads();
        if (tid == 0 && li + 2 < nlist) issue(s.clist[li + 2], buf);
        for (int kk = 0; kk < nneed; ++kk) {
            if constexpr (TAN)
                body(s.crec + kk * R::RC, s.trec + kk * R::RC);
            else
                body(s.crec + kk * R::RC);
        }
    }
    __syncthreads();          // the next tile rebuilds `clist` and re-uses `crec`
}

// record -> registers: the geometry part (NG4 float4), or the rest up to the original index
template <int D, int C>
__device__ __forceinline__ void load_rec(const float* rc, float (&f)[Rec<D, C>::RC], int from, int to) {
    const float4* r4 = reinterpret_cast<const float4*>(rc);
#pragma unroll
    for (int j = from; j < to; ++j) {
        float4 v = r4[j];
        f[4 * j] = v.x; f[4 * j + 1] = v.y; f[4 * j + 2] = v.z; f[4 * j + 3] = v.w;
    }
}

}  // namespace smoe
