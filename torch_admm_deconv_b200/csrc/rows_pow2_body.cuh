// rows_pow2_body.cuh -- body of the specialised row-pass kernel (W in {128, 256, 512}); see rows_pow2.cu for the design notes.
// Included by rows_pow2.cu (the __global__ kernel k_rows_pow2 and its launchers) and by coop_small.cu (the persistent
// cooperative kernel for small, latency-bound batches, which runs the same body as one phase of its iteration loop).
#pragma once
#include "common.cuh"
#include <cstdio>
#include "fft_pow2.cuh"

#ifndef ROWS_ADJ_OCC
#define ROWS_ADJ_OCC 3
#endif
namespace admm {

// w = z - u with z = soft_thresh(q), u = q - z  ==>  w = q - 2 u(q), u = clamp(q) for tau >= 0   (deconv.py:15-16, 104, 114-115)
template <bool NEG> __device__ __forceinline__ float wfunT(float q, float tau) { return fmaf(-2.0f, dual_of<NEG>(q, tau), q); }
__device__ __forceinline__ float2 mk(float2 a, float2 b) { return make_float2(a.x - b.y, a.y + b.x); }       // a + i b
__device__ __forceinline__ float2 mkc(float2 a, float2 b) { return make_float2(a.x + b.y, b.x - a.y); }      // conj(a) + i conj(b)


// pre-clamp state of one row pair (rows a, b) and the q_y of the row below, for columns c, c+1 (+ q_x at c+2)
struct QRegs {
    float2 qxa, qxb, qyb, qyc;
    float qxa2, qxb2;
};

// MODE: ROWS_FULL (one ADMM iteration), ROWS_R2C (real rows -> packed spectrum), ROWS_C2R (packed spectrum -> real
// rows, unnormalised, + optional bias).  The plain modes have no halo: a band is up to 2*NPAIR rows.
// COOP: the body runs inside a persistent cooperative kernel (coop_small.cu) whose earlier phases wrote the data it reads:
// plain (coherent) loads instead of the read-only path, `bid` instead of the block index, shared memory handed in.
// HT: the image height as a compile-time constant (square planes), 0 = run-time value
template <int W, int MODE, bool COOP, int HT = 0>
__device__ __forceinline__ void rows_pow2_body(const RowArgs& a, int H_dyn, int nbands, int pdl, unsigned bid, float2* smem) {
    const int H = HT ? HT : H_dyn;
    auto ldg_f = [](const float* p_) { return COOP ? *p_ : __ldg(p_); };
    auto ldg_f2 = [](const float* p_) {
        return COOP ? *reinterpret_cast<const float2*>(p_) : __ldg(reinterpret_cast<const float2*>(p_));
    };
    auto ldg_c = [](const float2* p_) { return COOP ? *p_ : __ldg(p_); };
    using S = RowSmem<W>;
    using RR = RowRadix<W>;
    constexpr int TPS = S::TPS, NPAIR = S::NPAIR, REGION = S::REGION;
    constexpr int T8 = W / 8;                 // butterflies of the radix-8 edge passes
    constexpr int Wc = W / 2;
    float2* regX = smem;                                    // NPAIR regions
    // v pair m is written over x pair m+1 once every thread has loaded that pair (one barrier per march step),
    // so the divergence needs no second tile and four CTAs fit on an SM
    float2* regV = (MODE == ROWS_FULL || MODE == ROWS_FULL_U || MODE == ROWS_ADJ || MODE == ROWS_FULL_MAP || MODE == ROWS_ADJ_MAP)
                 ? regX + REGION : regX;
    float2* tabs = regX + NPAIR * REGION;
    float2* side = tabs + S::TAB_END;
    const RowMapObj map;

    const int tid = threadIdx.x;
    const int pair = tid / TPS;               // row pair handled by this thread in the FFT phases
    const int t = tid % TPS;
    const int band = bid % nbands;
    const int p = bid / nbands;
    // balanced even band sizes: rows [r0, r1)
    const int hh = H >> 1;
    const int r0 = 2 * ((band * hh) / nbands);
    const int r1 = 2 * (((band + 1) * hh) / nbands);
    const int Rb = r1 - r0;                   // even, <= RMAX (FULL) or 2*NPAIR (plain modes)
    constexpr bool kFull = (MODE == ROWS_FULL || MODE == ROWS_FULL_U || MODE == ROWS_FULL_MAP);
    constexpr bool kStateU = (MODE == ROWS_FULL_U);
    constexpr bool kMap = (MODE == ROWS_FULL_MAP || MODE == ROWS_ADJ_MAP);   // tau per pixel from a.cmap (DESIGN section 11)
    constexpr bool kHalo = (kFull || MODE == ROWS_ADJ || MODE == ROWS_ADJ_MAP);
    const int npx = kHalo ? Rb / 2 + 1 : Rb / 2;   // x pairs (halo modes: rows r0-1 .. r0+Rb)
    const int npv = Rb / 2;                   // v pairs (rows r0 .. r0+Rb-1)
    const int rowbase = kHalo ? r0 - 1 : r0;
    const size_t plane_real = (size_t)p * H * W;
    const size_t plane_spec = (size_t)p * H * Wc;

    // edge-pass butterflies of this thread: j1 = t, j2 = T8 - t   (t == 0: j1 = 0, j2 = T8/2)
    const bool t0 = (t == 0);
    const int j1 = t;
    const int j2 = t0 ? (T8 / 2) : (T8 - t);
    float2 d[kPT];
    float2* myX = regX + pair * REGION;
    // the TPS lanes of one row pair synchronise among themselves only (a warp may hold several pairs, and the
    // last pair of a band can be inactive)
    const unsigned pmask = (TPS >= 32) ? 0xffffffffu
                                       : (((1u << (TPS & 31)) - 1u) << (((tid & 31) / TPS) * TPS));

#ifdef ROWS_STATS
    long long st[6]; st[0] = clock64();
#define ROWS_ST(i) st[i] = clock64()
#else
#define ROWS_ST(i)
#endif
    const bool early_tabs = pdl != 0;
    if (early_tabs) {
        // launched with programmatic stream serialisation (small, latency-bound problems): the tables are built
        // while the previous kernel drains; nothing the previous kernel wrote is touched before pdl_wait()
        pdl_launch_dependents();
        build_tab<W, RR::IB, 8>(tabs + S::TAB_IB, a.tw);
        build_tab<W, RR::IC, 8 * RR::IB>(tabs + S::TAB_IC, a.tw);
        if (!S::kShareB) build_tab<W, RR::FB, RR::FA>(tabs + S::TAB_FB, a.tw);
        if (!S::kShareC) build_tab<W, 8, W / 8>(tabs + S::TAB_FC, a.tw);
        pdl_wait();
    }
    // issue the global loads of the merge first, build the twiddle tables while they are in flight
    float2 A1[4], B1[4], A2[4], B2[4];
    if (MODE != ROWS_R2C && pair < npx) {
        // rows (circular): ia = rowbase + 2*pair, ib = ia + 1
        int ra = rowbase + 2 * pair; if (ra < 0) ra += H; if (ra >= H) ra -= H;
        int rb = ra + 1; if (rb >= H) rb -= H;
        const float2* __restrict__ Sa = a.spec_in + plane_spec + (size_t)ra * Wc;
        const float2* __restrict__ Sb = a.spec_in + plane_spec + (size_t)rb * Wc;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            A1[r] = ldg_c(Sa + j1 + r * T8); B1[r] = ldg_c(Sb + j1 + r * T8);
            A2[r] = ldg_c(Sa + j2 + r * T8); B2[r] = ldg_c(Sb + j2 + r * T8);
        }
    }
    if (!early_tabs) {
        build_tab<W, RR::IB, 8>(tabs + S::TAB_IB, a.tw);
        build_tab<W, RR::IC, 8 * RR::IB>(tabs + S::TAB_IC, a.tw);
        if (!S::kShareB) build_tab<W, RR::FB, RR::FA>(tabs + S::TAB_FB, a.tw);
        if (!S::kShareC) build_tab<W, 8, W / 8>(tabs + S::TAB_FC, a.tw);
    }
    __syncthreads();
    ROWS_ST(1);

    // ------------------------------------------------------------------ C2R: merge + inverse FFT
    if (MODE != ROWS_R2C && pair < npx) {
        // slot (m, r) = d[m + 2r]: m = 0 -> butterfly j1, m = 1 -> butterfly j2; point n = j + r*T8
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            d[0 + 2 * r] = mk(A1[r], B1[r]);
            d[1 + 2 * r] = mk(A2[r], B2[r]);
        }
#pragma unroll
        for (int r = 4; r < 8; ++r) {
            // n = j + r*T8 > W/2: Z[n] = conj(P_a[W-n]) + i conj(P_b[W-n]);  W - n = (T8 - j) + (7 - r) T8
            const float2 g1a = t0 ? A1[(8 - r) & 3] : A2[7 - r];      // t0: W - r*T8 = (8 - r) T8
            const float2 g1b = t0 ? B1[(8 - r) & 3] : B2[7 - r];
            const float2 g2a = t0 ? A2[7 - r] : A1[7 - r];            // t0: j2 = T8/2 is self-paired
            const float2 g2b = t0 ? B2[7 - r] : B1[7 - r];
            d[0 + 2 * r] = mkc(g1a, g1b);
            d[1 + 2 * r] = mkc(g2a, g2b);
        }
        if (t0) {
            // packed column 0 = (DC, Nyquist) of each row, both real
            d[0] = make_float2(A1[0].x, B1[0].x);                      // Z[0]
            d[0 + 2 * 4] = make_float2(A1[0].y, B1[0].y);              // Z[W/2] = Z[4*T8]
        }
        // first inverse pass: radix 8, no twiddles; butterfly j writes positions 8j + r
        {
            float2 v0[8], v1[8];
#pragma unroll
            for (int r = 0; r < 8; ++r) { v0[r] = d[2 * r]; v1[r] = d[1 + 2 * r]; }
            dft8<+1>(v0); dft8<+1>(v1);
            const int b1 = map.base(8 * j1), b2 = map.base(8 * j2);
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                myX[b1 + r] = v0[r];
                myX[b2 + r] = v1[r];
            }
        }
        __syncwarp(pmask);
        pass_load<W>(d, t, myX, map);
        pass_compute<W, RR::IB, 8, +1>(d, t, tabs + S::TAB_IB);
        __syncwarp(pmask);
        pass_store<W, RR::IB, 8>(d, t, myX, map);
        __syncwarp(pmask);
        pass_load<W>(d, t, myX, map);
        pass_compute<W, RR::IC, 8 * RR::IB, +1>(d, t, tabs + S::TAB_IC);
        __syncwarp(pmask);
        pass_store<W, RR::IC, 8 * RR::IB>(d, t, myX, map);      // natural order: myX[at(c)] = (x_a[c], x_b[c])
    }

    if (MODE == ROWS_C2R) {
        // x pairs -> real rows (+ bias): item = (pair, column pair), 8-byte coalesced stores
        __syncthreads();
        constexpr int CP = W / 2;
        float* __restrict__ out = a.real_out + out_plane_offset(a, p, H, W);
        const float bias = a.bias ? __ldg(a.bias) : 0.f;
        const int act = a.act;                                // fused activation(x + b) of the layer (admmdeconv.py:64)
        for (int it = tid; it < npx * CP; it += 256) {
            const int pp = it / CP, c = 2 * (it - pp * CP);
            const int pc = map.at(c);
            const float2 X0 = regX[pp * REGION + pc], X1 = regX[pp * REGION + pc + 1];
            const size_t o = (size_t)(r0 + 2 * pp) * W + c;
            *reinterpret_cast<float2*>(out + o) = make_float2(act_apply(X0.x + bias, act), act_apply(X1.x + bias, act));
            *reinterpret_cast<float2*>(out + o + W) = make_float2(act_apply(X0.y + bias, act), act_apply(X1.y + bias, act));
        }
        return;
    }
    if (MODE == ROWS_R2C) {
        // real rows -> complex pairs (row a + i row b) in the regions the forward FFT reads
        constexpr int CP = W / 2;
        if (!a.r2c_div) {
            const float* __restrict__ in = a.real_in + plane_real;
            const unsigned char* __restrict__ in8 = a.real_in_u8 ? a.real_in_u8 + plane_real : nullptr;
            for (int it = tid; it < npv * CP; it += 256) {
                const int pp = it / CP, c = 2 * (it - pp * CP);
                const int pc = map.at(c);
                const size_t o = (size_t)(r0 + 2 * pp) * W + c;
                float2 ra_, rb_;
                if (in8) {                                    // uint8 image, scaled like etransforms.py:29-31 (x / 255.0)
                    const uchar2 ua = __ldg(reinterpret_cast<const uchar2*>(in8 + o)), ub = __ldg(reinterpret_cast<const uchar2*>(in8 + o + W));
                    ra_ = make_float2((float)ua.x / 255.0f, (float)ua.y / 255.0f);
                    rb_ = make_float2((float)ub.x / 255.0f, (float)ub.y / 255.0f);
                } else {
                    ra_ = ldg_f2(in + o); rb_ = ldg_f2(in + o + W);
                }
                regX[pp * REGION + pc] = make_float2(ra_.x, rb_.x);
                regX[pp * REGION + pc + 1] = make_float2(ra_.y, rb_.y);
            }
        } else {
            // iso=True: the divergence v = Dx^T(k_x q_x) + Dy^T(k_y q_y), k = 2s-1 per pixel (coefficient maps shared by
            // all planes, deconv.py:19-24), is formed while loading, so v never goes through HBM
            const float* __restrict__ qx = a.qx_in + plane_real;
            const float* __restrict__ qy = a.qy_in + plane_real;
            // (backward: xbar = D^T qbar is the same operator with unit coefficients, cmap == NULL)
            const bool unit = (a.cmap == nullptr);
            const float* __restrict__ kx = unit ? qx : a.cmap;          // never dereferenced when unit
            const float* __restrict__ ky = unit ? qx : a.cmap + (size_t)H * W;
            const float2 one2 = make_float2(1.f, 1.f);
            for (int it = tid; it < npv * CP; it += 256) {
                const int pp = it / CP, c = 2 * (it - pp * CP);
                const int pc = map.at(c);
                const int ra_ = r0 + 2 * pp;
                int rc_ = ra_ + 2; if (rc_ >= H) rc_ -= H;
                const int c2 = (c + 2 == W) ? (2 - W) : 2;
                const size_t oa = (size_t)ra_ * W + c, oc = (size_t)rc_ * W + c;
                const float2 xa = ldg_f2(qx + oa), xb = ldg_f2(qx + oa + W);
                const float xa2 = ldg_f(qx + oa + c2), xb2 = ldg_f(qx + oa + W + c2);
                const float2 ya = ldg_f2(qy + oa), yb = ldg_f2(qy + oa + W), yc = ldg_f2(qy + oc);
                const float2 ka = unit ? one2 : ldg_f2(kx + oa), kb = unit ? one2 : ldg_f2(kx + oa + W);
                const float ka2 = unit ? 1.f : ldg_f(kx + oa + c2), kb2 = unit ? 1.f : ldg_f(kx + oa + W + c2);
                const float2 la = unit ? one2 : ldg_f2(ky + oa), lb = unit ? one2 : ldg_f2(ky + oa + W), lc = unit ? one2 : ldg_f2(ky + oc);
                const float wxa0 = ka.x * xa.x, wxa1 = ka.y * xa.y, wxa2 = ka2 * xa2;
                const float wxb0 = kb.x * xb.x, wxb1 = kb.y * xb.y, wxb2 = kb2 * xb2;
                const float wya0 = la.x * ya.x, wya1 = la.y * ya.y, wyb0 = lb.x * yb.x, wyb1 = lb.y * yb.y;
                const float wyc0 = lc.x * yc.x, wyc1 = lc.y * yc.y;
                float va0 = wxa0 - wxa1 + wya0 - wyb0, va1 = wxa1 - wxa2 + wya1 - wyb1;
                float vb0 = wxb0 - wxb1 + wyb0 - wyc0, vb1 = wxb1 - wxb2 + wyb1 - wyc1;
                regX[pp * REGION + pc] = make_float2(va0, vb0);
                regX[pp * REGION + pc + 1] = make_float2(va1, vb1);
            }
        }
    }

    // ------------------------------------------------------------------ prox / dual update / divergence
    // thread = (row group g, column pair cp): columns c, c+1, all v pairs m in [m_lo, m_hi) of the group
    if (kFull) {
        constexpr int CP = W / 2;                              // column pairs per row
        constexpr int NG = 256 / CP;                           // row groups (1 for W = 512)
        const int g = tid / CP;
        const int c = 2 * (tid % CP);
        const int m_lo = (g * npv) / NG, m_hi = ((g + 1) * npv) / NG;
        const float tau = kMap ? 0.f : __ldg(a.lmbd) / __ldg(a.rho);   // deconv.py:44 (maps: read per pixel below)
        const bool have_q = (a.qx_in != nullptr);
        const float* __restrict__ qxi = a.qx_in + plane_real + c;
        const float* __restrict__ qyi = a.qy_in + plane_real + c;
        float* __restrict__ qxo = a.qx_out + plane_real + c;
        float* __restrict__ qyo = a.qy_out + plane_real + c;
        const int c2 = (c + 2 == W) ? (2 - W) : 2;               // offset of column c+2 (circular)
        const int cl = (c == 0) ? W - 1 : c - 1;
        const int pl = map.at(cl), pc = map.at(c), pr2 = map.at((c + 2) & (W - 1));
        const int pc1 = pc + 1;                                  // c is even: c and c+1 share a 16-group

        auto load_q = [&](int m, QRegs& q) {
            // rows a = r0 + 2m, b = a + 1, row below = b + 1 (circular)
            const int ra = r0 + 2 * m;
            int rc = ra + 2; if (rc >= H) rc -= H;
            const float* xa = qxi + (size_t)ra * W;
            const float* ya = qyi + (size_t)ra * W;
            q.qxa = ldg_f2(xa); q.qxa2 = ldg_f(xa + c2);
            q.qxb = ldg_f2(xa + W); q.qxb2 = ldg_f(xa + W + c2);
            q.qyb = ldg_f2(ya + W);
            q.qyc = ldg_f2(qyi + (size_t)rc * W);
        };
        QRegs q0, q1;
        float2 qya = make_float2(0.f, 0.f);
        q0.qxa = q0.qxb = q0.qyb = q0.qyc = make_float2(0.f, 0.f); q0.qxa2 = q0.qxb2 = 0.f;
        q1 = q0;
        if (have_q && m_lo < m_hi) {
            qya = ldg_f2(qyi + (size_t)(r0 + 2 * m_lo) * W);
            load_q(m_lo, q0);
            if (m_lo + 1 < m_hi) load_q(m_lo + 1, q1);
        }
        __syncthreads();                                         // x of every pair is in shared memory
        ROWS_ST(2);

        // The march overwrites x pair m+1 with v pair m.  Inside a warp that is ordered by __syncwarp; the two columns
        // a warp reads from its neighbours' strips are copied to a side buffer first, so warps need no barrier while
        // they march and run at their own pace.
        const int lane = tid & 31, wid = tid >> 5;
        float2* sideW = side + wid * (NPAIR * 2);
        {
            const int cfirst = 2 * ((tid & ~31) % CP);
            const int cL = (cfirst == 0) ? W - 1 : cfirst - 1;
            const int cR = (cfirst + 64) & (W - 1);
            const int nslots = m_hi - m_lo + 1;
            for (int e = lane; e < 2 * nslots; e += 32) {
                const int ps = e >> 1;
                sideW[e] = regX[(m_lo + ps) * REGION + map.at((e & 1) ? cR : cL)];
            }
        }
        __syncwarp();
        // per-lane source of the left / right neighbour columns: edge lanes read the side buffer
        const float2* baseL = (lane == 0) ? sideW : regX + m_lo * REGION + pl;
        const float2* baseR = (lane == 31) ? sideW + 1 : regX + m_lo * REGION + pr2;
        const int strideL = (lane == 0) ? 2 : REGION;
        const int strideR = (lane == 31) ? 2 : REGION;

        const int steps = (npv + NG - 1) / NG;
        // the march, instantiated for tau >= 0 (clamp) and tau < 0 (see dual_of, common.cuh); one uniform branch picks it
        auto march = [&](auto tsign) {
            constexpr bool NEG = decltype(tsign)::neg;
            // previous dual u from the state arrays: stored pre-clamp (q) when a backward may follow, else already clamped
            auto uof = [tau](float s_) { return kStateU ? s_ : dual_of<NEG>(s_, tau); };
            auto sof = [tau](float q_) { return kStateU ? dual_of<NEG>(q_, tau) : q_; };
            auto wfun2 = [](float q_, float tau_) { return wfunT<NEG>(q_, tau_); };
            // pair m holds rows i = 2m (x component) and i = 2m+1 (y component); i = 0 is the halo row r0-1
            const float2* X = regX + m_lo * REGION;
            float2 Pl = baseL[0], P0 = X[pc], P1 = X[pc1], P2 = baseR[0];
            __syncthreads();                                       // every group holds its first pair; side buffers complete
            // q_y and w_y of the first row of the group (row a of pair m_lo)
            float qy0 = P0.y - P0.x + uof(qya.x);
            float qy1 = P1.y - P1.x + uof(qya.y);
            float wy0 = wfun2(qy0, tau), wy1 = wfun2(qy1, tau);
            for (int it = 0; it < steps; ++it) {
                const int m = m_lo + it;
                const bool active = (m < m_hi);
                if (!active) break;
                const QRegs q = q0;
                q0 = q1;
                if (have_q && m + 2 < m_hi) load_q(m + 2, q1);
                X += REGION;
                const float2 Nl = baseL[(it + 1) * strideL], N0 = X[pc], N1 = X[pc1], N2 = baseR[(it + 1) * strideR];
                __syncwarp();                                      // every lane holds pair m+1 before any lane overwrites it
                // row a (band row 2m): x = P.y                                   (deconv.py:108, 111, 114)
                const float qxa0 = P0.y - Pl.y + uof(q.qxa.x);
                const float qxa1 = P1.y - P0.y + uof(q.qxa.y);
                const float qxa2 = P2.y - P1.y + uof(q.qxa2);
                const float wxa0 = wfun2(qxa0, tau), wxa1 = wfun2(qxa1, tau), wxa2 = wfun2(qxa2, tau);
                // row b (band row 2m+1): x = N.x                                 (deconv.py:109, 112, 115)
                const float qyb0 = N0.x - P0.y + uof(q.qyb.x);
                const float qyb1 = N1.x - P1.y + uof(q.qyb.y);
                const float wyb0 = wfun2(qyb0, tau), wyb1 = wfun2(qyb1, tau);
                const float qxb0 = N0.x - Nl.x + uof(q.qxb.x);
                const float qxb1 = N1.x - N0.x + uof(q.qxb.y);
                const float qxb2 = N2.x - N1.x + uof(q.qxb2);
                const float wxb0 = wfun2(qxb0, tau), wxb1 = wfun2(qxb1, tau), wxb2 = wfun2(qxb2, tau);
                // row below b: x = N.y (first row of the next pair, or the halo row r0+Rb)
                const float qyc0 = N0.y - N0.x + uof(q.qyc.x);
                const float qyc1 = N1.y - N1.x + uof(q.qyc.y);
                const float wyc0 = wfun2(qyc0, tau), wyc1 = wfun2(qyc1, tau);
                // v = Dx^T w_x + Dy^T w_y                                         (deconv.py:104)
                const float va0 = wxa0 - wxa1 + wy0 - wyb0;
                const float va1 = wxa1 - wxa2 + wy1 - wyb1;
                const float vb0 = wxb0 - wxb1 + wyb0 - wyc0;
                const float vb1 = wxb1 - wxb2 + wyb1 - wyc1;
                const size_t oa = (size_t)(r0 + 2 * m) * W;
                *reinterpret_cast<float2*>(qxo + oa) = make_float2(sof(qxa0), sof(qxa1));
                *reinterpret_cast<float2*>(qyo + oa) = make_float2(sof(qy0), sof(qy1));
                *reinterpret_cast<float2*>(qxo + oa + W) = make_float2(sof(qxb0), sof(qxb1));
                *reinterpret_cast<float2*>(qyo + oa + W) = make_float2(sof(qyb0), sof(qyb1));
                float2* V = regV + m * REGION;
                V[pc] = make_float2(va0, vb0);
                V[pc1] = make_float2(va1, vb1);
                Pl = Nl; P0 = N0; P1 = N1; P2 = N2;
                qy0 = qyc0; qy1 = qyc1; wy0 = wyc0; wy1 = wyc1;
            }
        };
        // the march with a threshold map: tau of every element read from the map (rows a, b at columns c, c+1, c+2 and
        // the row below at c, c+1; a shared map stays in L2), the dual per element with dual_any (the sign varies)
        auto march_map = [&]() {
            const float* __restrict__ tm = a.cmap + (a.tau_map_planes > 1 ? plane_real : 0) + c;
            auto du = [](float q_, float t_) { return dual_any(q_, t_); };
            auto wf = [](float q_, float t_) { return fmaf(-2.0f, dual_any(q_, t_), q_); };
            const float2* X = regX + m_lo * REGION;
            float2 Pl = baseL[0], P0 = X[pc], P1 = X[pc1], P2 = baseR[0];
            __syncthreads();
            float qy0 = 0.f, qy1 = 0.f, wy0 = 0.f, wy1 = 0.f;
            if (m_lo < m_hi) {
                const float2 t0_ = ldg_f2(tm + (size_t)(r0 + 2 * m_lo) * W);
                qy0 = P0.y - P0.x + du(qya.x, t0_.x);
                qy1 = P1.y - P1.x + du(qya.y, t0_.y);
                wy0 = wf(qy0, t0_.x); wy1 = wf(qy1, t0_.y);
            }
            for (int it = 0; it < steps; ++it) {
                const int m = m_lo + it;
                if (m >= m_hi) break;
                const QRegs q = q0;
                q0 = q1;
                if (have_q && m + 2 < m_hi) load_q(m + 2, q1);
                X += REGION;
                const float2 Nl = baseL[(it + 1) * strideL], N0 = X[pc], N1 = X[pc1], N2 = baseR[(it + 1) * strideR];
                __syncwarp();
                const int ra = r0 + 2 * m;
                int rc = ra + 2; if (rc >= H) rc -= H;
                const float* ta_ = tm + (size_t)ra * W;
                const float2 ta = ldg_f2(ta_), tb = ldg_f2(ta_ + W), tc = ldg_f2(tm + (size_t)rc * W);
                const float ta2 = ldg_f(ta_ + c2), tb2 = ldg_f(ta_ + W + c2);
                const float qxa0 = P0.y - Pl.y + du(q.qxa.x, ta.x);
                const float qxa1 = P1.y - P0.y + du(q.qxa.y, ta.y);
                const float qxa2 = P2.y - P1.y + du(q.qxa2, ta2);
                const float wxa0 = wf(qxa0, ta.x), wxa1 = wf(qxa1, ta.y), wxa2 = wf(qxa2, ta2);
                const float qyb0 = N0.x - P0.y + du(q.qyb.x, tb.x);
                const float qyb1 = N1.x - P1.y + du(q.qyb.y, tb.y);
                const float wyb0 = wf(qyb0, tb.x), wyb1 = wf(qyb1, tb.y);
                const float qxb0 = N0.x - Nl.x + du(q.qxb.x, tb.x);
                const float qxb1 = N1.x - N0.x + du(q.qxb.y, tb.y);
                const float qxb2 = N2.x - N1.x + du(q.qxb2, tb2);
                const float wxb0 = wf(qxb0, tb.x), wxb1 = wf(qxb1, tb.y), wxb2 = wf(qxb2, tb2);
                const float qyc0 = N0.y - N0.x + du(q.qyc.x, tc.x);
                const float qyc1 = N1.y - N1.x + du(q.qyc.y, tc.y);
                const float wyc0 = wf(qyc0, tc.x), wyc1 = wf(qyc1, tc.y);
                const float va0 = wxa0 - wxa1 + wy0 - wyb0;
                const float va1 = wxa1 - wxa2 + wy1 - wyb1;
                const float vb0 = wxb0 - wxb1 + wyb0 - wyc0;
                const float vb1 = wxb1 - wxb2 + wyb1 - wyc1;
                const size_t oa = (size_t)ra * W;
                *reinterpret_cast<float2*>(qxo + oa) = make_float2(qxa0, qxa1);
                *reinterpret_cast<float2*>(qyo + oa) = make_float2(qy0, qy1);
                *reinterpret_cast<float2*>(qxo + oa + W) = make_float2(qxb0, qxb1);
                *reinterpret_cast<float2*>(qyo + oa + W) = make_float2(qyb0, qyb1);
                float2* V = regV + m * REGION;
                V[pc] = make_float2(va0, vb0);
                V[pc1] = make_float2(va1, vb1);
                Pl = Nl; P0 = N0; P1 = N1; P2 = N2;
                qy0 = qyc0; qy1 = qyc1; wy0 = wyc0; wy1 = wyc1;
            }
        };
        if constexpr (kMap) march_map();
        else if (tau < 0.f) march(TauNeg{}); else march(TauPos{});
    }
    // ------------------------------------------------------------------ backward: adjoint of prox / dual / gradient
    // qbar = wbar + 1[|q| < tau] (ubar - 2 wbar) with wbar = D vbar;  xbar = D^T qbar;  new ubar = qbar;
    // taubar += sum (ubar - 2 wbar) 1[|q| >= tau] sign(q)            (SURVEY.md appendix B.1)
    if (MODE == ROWS_ADJ) {
        constexpr int CP = W / 2;
        constexpr int NG = S::kThreads / CP;
        const int g = tid / CP;
        const int c = 2 * (tid % CP);
        const int m_lo = (g * npv) / NG, m_hi = ((g + 1) * npv) / NG;
        const float tau = __ldg(a.lmbd) / __ldg(a.rho);
        const bool have_u = (a.ubx_in != nullptr);
        const float* __restrict__ uxi = a.ubx_in + plane_real + c;
        const float* __restrict__ uyi = a.uby_in + plane_real + c;
        const float* __restrict__ qxs = a.qx_in + plane_real + c;
        const float* __restrict__ qys = a.qy_in + plane_real + c;
        float* __restrict__ uxo = a.ubx_out + plane_real + c;
        float* __restrict__ uyo = a.uby_out + plane_real + c;
        const int c2 = (c + 2 == W) ? (2 - W) : 2;
        const int cl = (c == 0) ? W - 1 : c - 1;
        const int pl = map.at(cl), pc = map.at(c), pr2 = map.at((c + 2) & (W - 1));
        const int pc1 = pc + 1;
        struct ARegs {
            float2 uxa, uxb, uyb, uyc, qxa, qxb, qyb, qyc;
            float uxa2, uxb2, qxa2, qxb2;
        };
        auto load_a = [&](int m, ARegs& q) {
            const int ra = r0 + 2 * m;
            int rc = ra + 2; if (rc >= H) rc -= H;
            const size_t oa = (size_t)ra * W, oc = (size_t)rc * W;
            q.qxa = ldg_f2(qxs + oa); q.qxa2 = ldg_f(qxs + oa + c2);
            q.qxb = ldg_f2(qxs + oa + W); q.qxb2 = ldg_f(qxs + oa + W + c2);
            q.qyb = ldg_f2(qys + oa + W);
            q.qyc = ldg_f2(qys + oc);
            if (have_u) {
                q.uxa = ldg_f2(uxi + oa); q.uxa2 = ldg_f(uxi + oa + c2);
                q.uxb = ldg_f2(uxi + oa + W); q.uxb2 = ldg_f(uxi + oa + W + c2);
                q.uyb = ldg_f2(uyi + oa + W);
                q.uyc = ldg_f2(uyi + oc);
            } else {
                q.uxa = q.uxb = q.uyb = q.uyc = make_float2(0.f, 0.f); q.uxa2 = q.uxb2 = 0.f;
            }
        };
        auto qbar = [tau](float wb, float ub, float q) { return (fabsf(q) < tau) ? (ub - wb) : wb; };
        auto tterm = [tau](float wb, float ub, float q) {
            return (fabsf(q) >= tau) ? (ub - 2.f * wb) * (q > 0.f ? 1.f : (q < 0.f ? -1.f : 0.f)) : 0.f;
        };
        ARegs q0, q1;
        float2 uya = make_float2(0.f, 0.f), qya = make_float2(0.f, 0.f);
        if (m_lo < m_hi) {
            const size_t o0 = (size_t)(r0 + 2 * m_lo) * W;
            qya = ldg_f2(qys + o0);
            if (have_u) uya = ldg_f2(uyi + o0);
            load_a(m_lo, q0);
            if (m_lo + 1 < m_hi) load_a(m_lo + 1, q1); else q1 = q0;
        } else {
            load_a(0, q0); q1 = q0;                                  // idle group: keep the registers defined
        }
        __syncthreads();                                             // vbar rows of every pair are in shared memory

        float tsum = 0.f;
        const int steps = (npv + NG - 1) / NG;
        {
            const float2* X = regX + m_lo * REGION;
            float2 Pl = X[pl], P0 = X[pc], P1 = X[pc1], P2 = X[pr2];
            // first row of the group (row a of pair m_lo): wbar_y = vbar[r] - vbar[r-1]
            float qby0 = qbar(P0.y - P0.x, uya.x, qya.x);
            float qby1 = qbar(P1.y - P1.x, uya.y, qya.y);
            if (m_lo < m_hi) tsum += tterm(P0.y - P0.x, uya.x, qya.x) + tterm(P1.y - P1.x, uya.y, qya.y);
            for (int it = 0; it < steps; ++it) {
                const int m = m_lo + it;
                const bool active = (m < m_hi);
                const ARegs q = q0;
                q0 = q1;
                if (m + 2 < m_hi) load_a(m + 2, q1);
                X += REGION;
                float2 Nl = Pl, N0 = P0, N1 = P1, N2 = P2;
                if (active) { Nl = X[pl]; N0 = X[pc]; N1 = X[pc1]; N2 = X[pr2]; }
                __syncthreads();                                   // every thread holds pair m+1 in registers
                if (!active) continue;
                // row a: vbar = P.y
                const float wxa0 = P0.y - Pl.y, wxa1 = P1.y - P0.y, wxa2 = P2.y - P1.y;
                const float bxa0 = qbar(wxa0, q.uxa.x, q.qxa.x), bxa1 = qbar(wxa1, q.uxa.y, q.qxa.y), bxa2 = qbar(wxa2, q.uxa2, q.qxa2);
                tsum += tterm(wxa0, q.uxa.x, q.qxa.x) + tterm(wxa1, q.uxa.y, q.qxa.y);
                // row b: vbar = N.x
                const float wyb0 = N0.x - P0.y, wyb1 = N1.x - P1.y;
                const float byb0 = qbar(wyb0, q.uyb.x, q.qyb.x), byb1 = qbar(wyb1, q.uyb.y, q.qyb.y);
                tsum += tterm(wyb0, q.uyb.x, q.qyb.x) + tterm(wyb1, q.uyb.y, q.qyb.y);
                const float wxb0 = N0.x - Nl.x, wxb1 = N1.x - N0.x, wxb2 = N2.x - N1.x;
                const float bxb0 = qbar(wxb0, q.uxb.x, q.qxb.x), bxb1 = qbar(wxb1, q.uxb.y, q.qxb.y), bxb2 = qbar(wxb2, q.uxb2, q.qxb2);
                tsum += tterm(wxb0, q.uxb.x, q.qxb.x) + tterm(wxb1, q.uxb.y, q.qxb.y);
                // row below b: vbar = N.y (row a of the next pair, or the halo row r0+Rb)
                const float wyc0 = N0.y - N0.x, wyc1 = N1.y - N1.x;
                const float byc0 = qbar(wyc0, q.uyc.x, q.qyc.x), byc1 = qbar(wyc1, q.uyc.y, q.qyc.y);
                if (m + 1 < m_hi) tsum += tterm(wyc0, q.uyc.x, q.qyc.x) + tterm(wyc1, q.uyc.y, q.qyc.y);
                // xbar = Dx^T qbar_x + Dy^T qbar_y
                const float xa0 = bxa0 - bxa1 + qby0 - byb0;
                const float xa1 = bxa1 - bxa2 + qby1 - byb1;
                const float xb0 = bxb0 - bxb1 + byb0 - byc0;
                const float xb1 = bxb1 - bxb2 + byb1 - byc1;
                const size_t oa = (size_t)(r0 + 2 * m) * W;
                *reinterpret_cast<float2*>(uxo + oa) = make_float2(bxa0, bxa1);
                *reinterpret_cast<float2*>(uyo + oa) = make_float2(qby0, qby1);
                *reinterpret_cast<float2*>(uxo + oa + W) = make_float2(bxb0, bxb1);
                *reinterpret_cast<float2*>(uyo + oa + W) = make_float2(byb0, byb1);
                float2* V = regV + m * REGION;
                V[pc] = make_float2(xa0, xb0);
                V[pc1] = make_float2(xa1, xb1);
                Pl = Nl; P0 = N0; P1 = N1; P2 = N2;
                qby0 = byc0; qby1 = byc1;
            }
        }
        // block reduction of the tau gradient into this CTA's slot (single writer, fixed order: no atomics, so the
        // gradient is bit-identical from run to run; k_bwd_scalars adds the slots in a fixed order)
        __shared__ float tred[8];
        for (int o = 16; o > 0; o >>= 1) tsum += __shfl_down_sync(0xffffffffu, tsum, o);
        if ((tid & 31) == 0) tred[tid >> 5] = tsum;
        __syncthreads();
        if (tid == 0) {
            double s = 0.0;
            for (int w = 0; w < S::kThreads / 32; ++w) s += (double)tred[w];
            a.taubar[bid] += s;
        }
    }
    // the adjoint with a threshold map: masks per element, and each element's tau gradient (its x and y terms) added into
    // a.taubar[plane element] (double, one writer per element and launch: deterministic)
    if constexpr (MODE == ROWS_ADJ_MAP) {
        constexpr int CP = W / 2;
        constexpr int NG = S::kThreads / CP;
        const int g = tid / CP;
        const int c = 2 * (tid % CP);
        const int m_lo = (g * npv) / NG, m_hi = ((g + 1) * npv) / NG;
        const bool have_u = (a.ubx_in != nullptr);
        const float* __restrict__ uxi = a.ubx_in + plane_real + c;
        const float* __restrict__ uyi = a.uby_in + plane_real + c;
        const float* __restrict__ qxs = a.qx_in + plane_real + c;
        const float* __restrict__ qys = a.qy_in + plane_real + c;
        const float* __restrict__ tm = a.cmap + (a.tau_map_planes > 1 ? plane_real : 0) + c;
        float* __restrict__ uxo = a.ubx_out + plane_real + c;
        float* __restrict__ uyo = a.uby_out + plane_real + c;
        double* __restrict__ tbo = a.taubar + plane_real + c;
        const int c2 = (c + 2 == W) ? (2 - W) : 2;
        const int cl = (c == 0) ? W - 1 : c - 1;
        const int pl = map.at(cl), pc = map.at(c), pr2 = map.at((c + 2) & (W - 1));
        const int pc1 = pc + 1;
        auto ld2 = [&](const float* p_, bool ok) { return ok ? ldg_f2(p_) : make_float2(0.f, 0.f); };
        auto qbar = [](float wb, float ub, float q, float t) { return (fabsf(q) < t) ? (ub - wb) : wb; };
        auto tterm = [](float wb, float ub, float q, float t) {
            return (fabsf(q) >= t) ? (ub - 2.f * wb) * (q > 0.f ? 1.f : (q < 0.f ? -1.f : 0.f)) : 0.f;
        };
        float2 tya = make_float2(0.f, 0.f);                        // y terms of row a, carried from the row above
        float qby0 = 0.f, qby1 = 0.f;
        __syncthreads();                                             // vbar rows of every pair are in shared memory
        const float2* X = regX + m_lo * REGION;
        float2 Pl = X[pl], P0 = X[pc], P1 = X[pc1], P2 = X[pr2];
        if (m_lo < m_hi) {
            const size_t o0 = (size_t)(r0 + 2 * m_lo) * W;
            const float2 qya = ldg_f2(qys + o0), uya = ld2(uyi + o0, have_u), t0_ = ldg_f2(tm + o0);
            qby0 = qbar(P0.y - P0.x, uya.x, qya.x, t0_.x);
            qby1 = qbar(P1.y - P1.x, uya.y, qya.y, t0_.y);
            tya = make_float2(tterm(P0.y - P0.x, uya.x, qya.x, t0_.x), tterm(P1.y - P1.x, uya.y, qya.y, t0_.y));
        }
        const int steps = (npv + NG - 1) / NG;
        for (int it = 0; it < steps; ++it) {
            const int m = m_lo + it;
            const bool active = (m < m_hi);
            X += REGION;
            float2 Nl = Pl, N0 = P0, N1 = P1, N2 = P2;
            if (active) { Nl = X[pl]; N0 = X[pc]; N1 = X[pc1]; N2 = X[pr2]; }
            __syncthreads();                                         // every thread holds pair m+1 in registers
            if (!active) continue;
            const int ra = r0 + 2 * m;
            int rc = ra + 2; if (rc >= H) rc -= H;
            const size_t oa = (size_t)ra * W, oc = (size_t)rc * W;
            const float2 qxa = ldg_f2(qxs + oa), qxb = ldg_f2(qxs + oa + W), qyb = ldg_f2(qys + oa + W), qyc = ldg_f2(qys + oc);
            const float qxa2 = ldg_f(qxs + oa + c2), qxb2 = ldg_f(qxs + oa + W + c2);
            const float2 uxa = ld2(uxi + oa, have_u), uxb = ld2(uxi + oa + W, have_u);
            const float2 uyb = ld2(uyi + oa + W, have_u), uyc = ld2(uyi + oc, have_u);
            const float uxa2 = have_u ? ldg_f(uxi + oa + c2) : 0.f, uxb2 = have_u ? ldg_f(uxi + oa + W + c2) : 0.f;
            const float2 ta = ldg_f2(tm + oa), tb = ldg_f2(tm + oa + W), tc = ldg_f2(tm + oc);
            const float ta2 = ldg_f(tm + oa + c2), tb2 = ldg_f(tm + oa + W + c2);
            // row a: vbar = P.y
            const float wxa0 = P0.y - Pl.y, wxa1 = P1.y - P0.y, wxa2 = P2.y - P1.y;
            const float bxa0 = qbar(wxa0, uxa.x, qxa.x, ta.x), bxa1 = qbar(wxa1, uxa.y, qxa.y, ta.y), bxa2 = qbar(wxa2, uxa2, qxa2, ta2);
            const double ga0 = (double)tterm(wxa0, uxa.x, qxa.x, ta.x) + (double)tya.x;
            const double ga1 = (double)tterm(wxa1, uxa.y, qxa.y, ta.y) + (double)tya.y;
            // row b: vbar = N.x
            const float wyb0 = N0.x - P0.y, wyb1 = N1.x - P1.y;
            const float byb0 = qbar(wyb0, uyb.x, qyb.x, tb.x), byb1 = qbar(wyb1, uyb.y, qyb.y, tb.y);
            const float wxb0 = N0.x - Nl.x, wxb1 = N1.x - N0.x, wxb2 = N2.x - N1.x;
            const float bxb0 = qbar(wxb0, uxb.x, qxb.x, tb.x), bxb1 = qbar(wxb1, uxb.y, qxb.y, tb.y), bxb2 = qbar(wxb2, uxb2, qxb2, tb2);
            const double gb0 = (double)tterm(wyb0, uyb.x, qyb.x, tb.x) + (double)tterm(wxb0, uxb.x, qxb.x, tb.x);
            const double gb1 = (double)tterm(wyb1, uyb.y, qyb.y, tb.y) + (double)tterm(wxb1, uxb.y, qxb.y, tb.y);
            // row below b: vbar = N.y; its y terms belong to row a of the next pair (the next group's first row is its own)
            const float wyc0 = N0.y - N0.x, wyc1 = N1.y - N1.x;
            const float byc0 = qbar(wyc0, uyc.x, qyc.x, tc.x), byc1 = qbar(wyc1, uyc.y, qyc.y, tc.y);
            tya = (m + 1 < m_hi) ? make_float2(tterm(wyc0, uyc.x, qyc.x, tc.x), tterm(wyc1, uyc.y, qyc.y, tc.y)) : make_float2(0.f, 0.f);
            const float xa0 = bxa0 - bxa1 + qby0 - byb0;
            const float xa1 = bxa1 - bxa2 + qby1 - byb1;
            const float xb0 = bxb0 - bxb1 + byb0 - byc0;
            const float xb1 = bxb1 - bxb2 + byb1 - byc1;
            *reinterpret_cast<float2*>(uxo + oa) = make_float2(bxa0, bxa1);
            *reinterpret_cast<float2*>(uyo + oa) = make_float2(qby0, qby1);
            *reinterpret_cast<float2*>(uxo + oa + W) = make_float2(bxb0, bxb1);
            *reinterpret_cast<float2*>(uyo + oa + W) = make_float2(byb0, byb1);
            tbo[oa] += ga0; tbo[oa + 1] += ga1; tbo[oa + W] += gb0; tbo[oa + W + 1] += gb1;
            float2* V = regV + m * REGION;
            V[pc] = make_float2(xa0, xb0);
            V[pc1] = make_float2(xa1, xb1);
            Pl = Nl; P0 = N0; P1 = N1; P2 = N2;
            qby0 = byc0; qby1 = byc1;
        }
    }
    __syncthreads();
    ROWS_ST(3);

    // ------------------------------------------------------------------ R2C: forward FFT + split
    auto r2c = [&](float2* regbase, float2* spec_plane) {
    if (pair < npv) {
        float2* myV = regbase + pair * REGION;
        pass_load<W>(d, t, myV, map);
        pass_compute<W, RR::FA, 1, -1>(d, t, nullptr);
        __syncwarp(pmask);
        pass_store<W, RR::FA, 1>(d, t, myV, map);
        __syncwarp(pmask);
        pass_load<W>(d, t, myV, map);
        pass_compute<W, RR::FB, RR::FA, -1>(d, t, tabs + S::TAB_FB);
        __syncwarp(pmask);
        pass_store<W, RR::FB, RR::FA>(d, t, myV, map);
        __syncwarp(pmask);
        // last pass: radix 8, Ns = T8, butterflies j1 and j2; inputs j + r*T8, twiddle k = j
        float2 v0[8], v1[8];
        {
            const int b1 = map.base(j1), b2 = map.base(j2);
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                v0[r] = myV[b1 + RowMapObj::delta(r * T8)];
                v1[r] = myV[b2 + RowMapObj::delta(r * T8)];
            }
        }
        const float2* tabC = tabs + S::TAB_FC;
#pragma unroll
        for (int r = 1; r < 8; ++r) {
            v0[r] = cmul(v0[r], tabC[(r - 1) * T8 + j1]);
            v1[r] = cmul(v1[r], tabC[(r - 1) * T8 + j2]);
        }
        dft8<-1>(v0); dft8<-1>(v1);
        // v0[r] = Z[j1 + r T8], v1[r] = Z[j2 + r T8];  partner of n is W - n
        const int ra = r0 + 2 * pair;
        float2* __restrict__ Oa = spec_plane + (size_t)ra * Wc;
        float2* __restrict__ Ob = Oa + Wc;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            // column c = j1 + r T8 (< W/2)
            const float2 Z1 = v0[r];
            const float2 M1 = t0 ? v0[(8 - r) & 7] : v1[7 - r];
            float2 Xa = make_float2(0.5f * (Z1.x + M1.x), 0.5f * (Z1.y - M1.y));
            float2 Xb = make_float2(0.5f * (Z1.y + M1.y), 0.5f * (M1.x - Z1.x));
            if (r == 0 && t0) {                                        // packed (DC, Nyquist)
                Xa = make_float2(v0[0].x, v0[4].x);
                Xb = make_float2(v0[0].y, v0[4].y);
            }
            Oa[j1 + r * T8] = Xa; Ob[j1 + r * T8] = Xb;
            // column c = j2 + r T8 (< W/2)
            const float2 Z2 = v1[r];
            const float2 M2 = t0 ? v1[7 - r] : v0[7 - r];
            Oa[j2 + r * T8] = make_float2(0.5f * (Z2.x + M2.x), 0.5f * (Z2.y - M2.y));
            Ob[j2 + r * T8] = make_float2(0.5f * (Z2.y + M2.y), 0.5f * (M2.x - Z2.x));
        }
    }
    };
    r2c(regV, a.spec_out + plane_spec);
#ifdef ROWS_STATS
    ROWS_ST(4);
    if (kFull && tid == 0 && (bid % 997) == 7)
        printf("cta %u: tables %lld | spectrum wait + C2R %lld | march %lld | R2C + store %lld | total %lld\n", bid, st[1] - st[0], st[2] - st[1],
               st[3] - st[2], st[4] - st[3], st[4] - st[0]);
#endif

    if (MODE == ROWS_ADJ || MODE == ROWS_ADJ_MAP) {
        // optional second output: v_k = D^T w(q_k) recomputed from the saved pre-clamp state, and its row spectrum
        if (a.qvx != nullptr) {
            constexpr int CP = W / 2;
            constexpr int NG = S::kThreads / CP;
            const int g = tid / CP;
            const int c = 2 * (tid % CP);
            const int m_lo = (g * npv) / NG, m_hi = ((g + 1) * npv) / NG;
            const float tau = kMap ? 0.f : __ldg(a.lmbd) / __ldg(a.rho);
            const float* __restrict__ tm = kMap ? a.cmap + (a.tau_map_planes > 1 ? plane_real : 0) + c : nullptr;
            (void)tm;
            const float* __restrict__ qx = a.qvx + plane_real + c;
            const float* __restrict__ qy = a.qvy + plane_real + c;
            const int c2 = (c + 2 == W) ? (2 - W) : 2;
            const int pc = map.at(c);
            __syncthreads();                                         // every warp finished reading its v region
            for (int m = m_lo; m < m_hi; ++m) {
                const int ra = r0 + 2 * m;
                int rc = ra + 2; if (rc >= H) rc -= H;
                const float* xa = qx + (size_t)ra * W;
                const float2 xa01 = ldg_f2(xa), xb01 = ldg_f2(xa + W);
                const float xa2 = ldg_f(xa + c2), xb2 = ldg_f(xa + W + c2);
                const float2 ya = ldg_f2(qy + (size_t)ra * W), yb = ldg_f2(qy + (size_t)ra * W + W), yc = ldg_f2(qy + (size_t)rc * W);
                auto wfun2 = [](float q_, float tau_) { return fmaf(-2.0f, dual_any(q_, tau_), q_); };
                if constexpr (kMap) {
                    // the threshold of each element from the map: rows a, b at columns c, c+1, c+2 and the row below
                    const float* t_ = tm + (size_t)ra * W;
                    const float2 ta = ldg_f2(t_), tb = ldg_f2(t_ + W), tc = ldg_f2(tm + (size_t)rc * W);
                    const float ta2 = ldg_f(t_ + c2), tb2 = ldg_f(t_ + W + c2);
                    const float wxa0 = wfun2(xa01.x, ta.x), wxa1 = wfun2(xa01.y, ta.y), wxa2 = wfun2(xa2, ta2);
                    const float wxb0 = wfun2(xb01.x, tb.x), wxb1 = wfun2(xb01.y, tb.y), wxb2 = wfun2(xb2, tb2);
                    const float wya0 = wfun2(ya.x, ta.x), wya1 = wfun2(ya.y, ta.y);
                    const float wyb0 = wfun2(yb.x, tb.x), wyb1 = wfun2(yb.y, tb.y);
                    const float wyc0 = wfun2(yc.x, tc.x), wyc1 = wfun2(yc.y, tc.y);
                    regX[m * REGION + pc] = make_float2(wxa0 - wxa1 + wya0 - wyb0, wxb0 - wxb1 + wyb0 - wyc0);
                    regX[m * REGION + pc + 1] = make_float2(wxa1 - wxa2 + wya1 - wyb1, wxb1 - wxb2 + wyb1 - wyc1);
                } else {
                const float wxa0 = wfun2(xa01.x, tau), wxa1 = wfun2(xa01.y, tau), wxa2 = wfun2(xa2, tau);
                const float wxb0 = wfun2(xb01.x, tau), wxb1 = wfun2(xb01.y, tau), wxb2 = wfun2(xb2, tau);
                const float wya0 = wfun2(ya.x, tau), wya1 = wfun2(ya.y, tau);
                const float wyb0 = wfun2(yb.x, tau), wyb1 = wfun2(yb.y, tau);
                const float wyc0 = wfun2(yc.x, tau), wyc1 = wfun2(yc.y, tau);
                regX[m * REGION + pc] = make_float2(wxa0 - wxa1 + wya0 - wyb0, wxb0 - wxb1 + wyb0 - wyc0);
                regX[m * REGION + pc + 1] = make_float2(wxa1 - wxa2 + wya1 - wyb1, wxb1 - wxb2 + wyb1 - wyc1);
                }
            }
            __syncthreads();
            r2c(regX, a.spec_out2 + plane_spec);
        }
    }
}


}  // namespace admm
