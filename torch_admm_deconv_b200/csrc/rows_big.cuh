// rows_big.cuh -- row pass of the ADMM iteration for the LARGE widths on sm_100a: W = 3840 = 15*16*16 (the 2160x3840
// single-frame configuration, BASELINE configs[2]), 1920 = 15*8*16, 2560 = 10*16*16, 1280 = 10*8*16, 1024 = 8*8*16,
// 2048 = 8*16*16, 4096 = 16*16*16, 768 = 8*6*16, 1536 = 8*12*16, 3072 = 12*16*16; plus the plain R2C / C2R passes on the same schedules (k_rows_big_plain).
//
//   packed row spectrum of x_k  --C2R-->  x_k  --prox / dual / divergence-->  v_{k+1}  --R2C-->  packed spectrum
//   (deconv.py:106 irfftn rows, :108-115 Dx/Dy/soft_thresh/dual update, :104 Dx_t/Dy_t + rfftn rows)
//
// One CTA (NT = W/R0 threads; 3840: 256 threads, 128 registers, 2 CTAs/SM) owns a band of Rb (even) image rows of one plane and
// marches down it one row PAIR at a time; the whole CTA works on one complex FFT of length W (two real rows,
// z = row_a + i row_b), 8..16 points per thread in registers.  Three row-pair buffers rotate in shared memory
// (P = x pair m, F = x pair m+1, S = scratch; 3 x 30 KB), every pass reads one and writes another:
//   * inverse FFT of x pair m+1: the first pass (radix 15, every thread) takes its inputs straight from global memory
//     and does the Hermitian merge of the two packed half spectra on the fly (F), pass 2 F -> S, pass 3 S -> F;
//   * spatial step: the thread that owns butterfly j of the first FORWARD pass computes v for exactly the columns
//     j + r W/15 that butterfly consumes, so v never goes through shared memory; x comes from P (rows ra-1, ra) and
//     F (rows ra+1, ra+2), the state from global (128-byte runs per warp, all 75 loads of a thread in one batch);
//     w_x of column c+1 comes from the next lane (shuffle), for a warp's last lane through a small side array;
//   * forward pass 1 -> S, pass 2 S -> P (x pair m is dead by then), pass 3 P -> S, and the split into the two packed
//     half spectra reads S;  P and F swap roles.  7 block barriers per march step.
// q_y of the first row of the next pair is recomputed there (one more 4-byte read per pixel pair, an L2 hit) instead of
// being carried.  Pass-2 twiddles come from a 2 KB shared table, pass-3 twiddles (one set per thread) stay in registers.
// With TILED the packed spectra use the tile-major layout shared with cols_big.cu (common.cuh, kSpecTile).
#pragma once
#include <cstdio>
#include "common.cuh"
#include "fft_big.cuh"

namespace admm {

template <int W> struct RowBig;
// R0 (odd) fixes the thread count NT = W / R0 and the columns a thread owns in the spatial step; pass 2 may have more
// butterflies than threads (looped -- every pass writes a buffer other than the one it reads), pass 3 at most NT.
// PAD: 0 when R0 is odd; R0 when it is even (power-of-two widths): entry n of a row-pair buffer then sits at slot
// n + n/PAD, so the stride-R0 stores of the first passes spread over the banks
template <> struct RowBig<3840> { static constexpr int R0 = 15, R1 = 16, R2 = 16, OCC = 2, PAD = 0; };
template <> struct RowBig<1920> { static constexpr int R0 = 15, R1 = 8,  R2 = 16, OCC = 3, PAD = 0; };   // 3 x 128 threads, 168 registers: faster than 4 x 128 at 128
template <> struct RowBig<1024> { static constexpr int R0 = 8,  R1 = 8,  R2 = 16, OCC = 5, PAD = 8; };     // measured: 5 x 128 threads > 4 > 3 > 6
template <> struct RowBig<2048> { static constexpr int R0 = 8,  R1 = 16, R2 = 16, OCC = 2, PAD = 8; };
template <> struct RowBig<4096> { static constexpr int R0 = 16, R1 = 16, R2 = 16, OCC = 2, PAD = 16; };
template <> struct RowBig<768>  { static constexpr int R0 = 8,  R1 = 6,  R2 = 16, OCC = 6, PAD = 8; };     // 3 * 2^n sizes
template <> struct RowBig<1536> { static constexpr int R0 = 8,  R1 = 12, R2 = 16, OCC = 3, PAD = 8; };
template <> struct RowBig<3072> { static constexpr int R0 = 12, R1 = 16, R2 = 16, OCC = 2, PAD = 12; };
template <> struct RowBig<2560> { static constexpr int R0 = 10, R1 = 16, R2 = 16, OCC = 2, PAD = 10; };   // 1440p
template <> struct RowBig<1280> { static constexpr int R0 = 10, R1 = 8,  R2 = 16, OCC = 4, PAD = 10; };   // 720p (measured: 4 > 3 > 5)

// w = z - u with z = soft_thresh(q), u = q - z  ==>  w = q - 2 u(q), u = clamp(q) for tau >= 0  (deconv.py:15-16, 104, 114-115)

// STATE_U: the state arrays hold the clamped dual u = clamp(q) (inference, nothing saved for a backward) instead of q
// TILED: the packed spectra use the tile-major layout shared with the large column kernel (see common.cuh, spec_tiled)
template <int W, bool STATE_U, bool TILED>
// 1 = bulk L2 prefetch of a march step's state rows at the top of the step (cfg3 row pass 161.9 -> 151.3 us).  The lead matters:
// the same prefetch one whole step (13 us) ahead was measured 3 % SLOWER in round 1 -- at these rates a line that is not used
// within a few microseconds has left the L2 again
#ifndef ROWS_BIG_STATE_PF
#define ROWS_BIG_STATE_PF 1
#endif
// 1 = L2 prefetch of the NEXT step's spectrum rows (first inverse pass) before this step's spatial phase (~6 us ahead)
// (146.5 vs 151.4 us)
#ifndef ROWS_BIG_SPEC_PF
#define ROWS_BIG_SPEC_PF 1
#endif
#ifndef ROWS_BIG_CH
#define ROWS_BIG_CH 15
#endif
__global__ void __launch_bounds__(W / RowBig<W>::R0, RowBig<W>::OCC)
k_rows_big(RowArgs a, int H, int nbands) {
    using RB = RowBig<W>;
    constexpr int R0 = RB::R0, R1 = RB::R1, R2 = RB::R2;
    constexpr int NT = W / R0;
    constexpr int Wc = W / 2;
    constexpr int PAD = RB::PAD;
    constexpr int WB = W + (PAD ? W / PAD : 0);                 // slots per row-pair buffer
    using I1 = BigPass<W, R0, 1, +1, 1, PAD>;
    using I2 = BigPass<W, R1, R0, +1, 1, PAD>;
    using I3 = BigPass<W, R2, R0 * R1, +1, 1, PAD>;
    using F1 = BigPass<W, R0, 1, -1, 1, PAD>;
    using F2 = BigPass<W, R1, R0, -1, 1, PAD>;
    using F3 = BigPass<W, R2, R0 * R1, -1, 1, PAD>;
    auto pm = [](int n) { return PAD ? n + n / (PAD ? PAD : 1) : n; };   // slot of entry n
    constexpr int RMAX = (R1 > R2 ? R1 : R2) > R0 ? (R1 > R2 ? R1 : R2) : R0;
    constexpr int NW = NT / 32;
    constexpr int CH = (R0 % ROWS_BIG_CH == 0) ? ROWS_BIG_CH : R0;        // columns per batch of state loads
    static_assert(NT % 32 == 0 && R0 % CH == 0, "thread / batch layout");
    static_assert(I3::T <= NT && (W / 2) % kSpecTile == 0, "pass-3 twiddles are per thread; whole spectrum tiles");
    constexpr int ROUNDS2 = (I2::T + NT - 1) / NT;
    extern __shared__ float2 smem[];
    float2* P = smem;            // x pair m   (.x = row ra-1, .y = row ra)
    float2* F = smem + WB;       // x pair m+1 (.x = row rb,   .y = row rb+1); P and F swap every march step
    float2* S = smem + 2 * WB;   // scratch: every pass writes a buffer other than the one it reads
    float2* edge = smem + 3 * WB; // w_x of the first column of every warp, per butterfly input r
    // twiddles (forward sign; the inverse passes conjugate): pass 2 (NS = R0) from a compact shared table, entry
    // (r-1) * R0 + k; pass 3 (NS = R0 R1, one distinct set per thread) stays in registers for the whole march
    float2* tab2 = edge + NW * R0;

    const int j = threadIdx.x;
    const int lane = j & 31, warp = j >> 5;
    const int band = blockIdx.x % nbands;
    const int p = blockIdx.x / nbands;
    const int hh = H >> 1;
    const int r0 = 2 * ((band * hh) / nbands);
    const int r1 = 2 * (((band + 1) * hh) / nbands);
    const int npv = (r1 - r0) / 2;
    const size_t plane_real = (size_t)p * H * W;
    const float2* __restrict__ spec = a.spec_in + (size_t)p * H * Wc;
    float2* __restrict__ sout = a.spec_out + (size_t)p * H * Wc;
    const float* __restrict__ qxi = a.qx_in ? a.qx_in + plane_real : nullptr;
    const float* __restrict__ qyi = a.qy_in ? a.qy_in + plane_real : nullptr;
    float* __restrict__ qxo = a.qx_out + plane_real;
    float* __restrict__ qyo = a.qy_out + plane_real;
    const float tau = a.lmbd[0] / a.rho[0];                     // deconv.py:44
    const float2* __restrict__ tw = a.tw;

    float2 v[RMAX];
    for (int i = j; i < (R1 - 1) * R0; i += NT) {
        const int r = i / R0 + 1, k = i - (r - 1) * R0;
        tab2[i] = __ldg(tw + k * r * (W / (R0 * R1)));
    }
    float2 w3[R2 - 1];
#pragma unroll
    for (int r = 1; r < R2; ++r) w3[r - 1] = __ldg(tw + (j < I3::T ? j * r : 0));

    // -DROWS_STATS: per-phase clock cycles of a few CTAs (development instrumentation, tools/README.md)
#ifdef ROWS_STATS
    long long st[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tp = clock64();
#define RB_ST(i) { const long long tn_ = clock64(); st[i] += tn_ - tp; tp = tn_; }
#else
#define RB_ST(i)
#endif
    // inverse FFT of the row pair (rowa, rowb) into dst; the caller guarantees nobody still reads dst
    auto inverse_pair = [&](int rowa, int rowb, float2* __restrict__ dst) {
        const float2* __restrict__ Sa = spec + (size_t)rowa * Wc;
        const float2* __restrict__ Sb = spec + (size_t)rowb * Wc;
        // tile-major: the entries of rows (rowa, rowb) = (odd, even) for one packed column are one float4
        const float4* __restrict__ St = reinterpret_cast<const float4*>(spec) + (size_t)(rowb >> 1) * kSpecTile;
#pragma unroll
        for (int r = 0; r < R0; ++r) {
            const int n = j + r * NT;
            const bool hi = n > Wc;
            const int c = hi ? W - n : (n == Wc ? 0 : n);
            // branch-free (all loads of a thread are in flight together): bins 0 and W/2 are packed in entry 0
            float2 A, B;
            if (TILED) {
                const float4 t = __ldg(St + (size_t)(c / kSpecTile) * (H / 2) * kSpecTile + (c % kSpecTile));
                A = make_float2(t.x, t.y); B = make_float2(t.z, t.w);
            } else {
                A = __ldg(Sa + c); B = __ldg(Sb + c);
            }
            // Z[n] = Xa[n] + i Xb[n];  upper half from the Hermitian symmetry of the two real rows
            float2 z = hi ? make_float2(A.x + B.y, B.x - A.y) : make_float2(A.x - B.y, A.y + B.x);
            if (n == 0) z = make_float2(A.x, B.x);
            if (n == Wc) z = make_float2(A.y, B.y);
            v[r] = z;
        }
        dft_big<R0, +1>(v);
        // dst is free: its last readers (third forward pass of the previous step) are behind a barrier
        I1::store(dst, j, v);
        __syncthreads();                       // also: the split of the previous step has finished reading S
        RB_ST(0);
#pragma unroll
        for (int q = 0; q < ROUNDS2; ++q) {
            const int jj = j + q * NT;
            if (jj < I2::T) { I2::load(dst, jj, v); I2::template butterfly_tab<R0>(v, tab2 + jj % R0); I2::store(S, jj, v); }
        }
        __syncthreads();
        if (j < I3::T) { I3::load(S, j, v); I3::butterfly_reg(v, w3); I3::store(dst, j, v); }
        __syncthreads();
        RB_ST(1);
    };

    { int rm = r0 - 1; if (rm < 0) rm += H; inverse_pair(rm, r0, P); }

    for (int m = 0; m < npv; ++m) {
        const int ra = r0 + 2 * m, rb = ra + 1;
        int rc = rb + 1;
        if (rc >= H) rc -= H;
#if ROWS_BIG_STATE_PF
        // the state rows of this step -> L2 now (one bulk prefetch per row): the spatial step reads them as one exposed batch of
        // 75 loads per thread right after the inverse transform of the next pair, ~4 us from here
        if (qxi && j == 0) {
            const unsigned nb = (unsigned)(W * sizeof(float));
            asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(qxi + (size_t)ra * W), "r"(2 * nb) : "memory");   // rows ra, rb
            asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(qyi + (size_t)ra * W), "r"(2 * nb) : "memory");
            asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(qyi + (size_t)rc * W), "r"(nb) : "memory");
        }
#endif
        inverse_pair(rb, rc, F);

#if ROWS_BIG_SPEC_PF
        if (m + 1 < npv) {
            // rows (rb + 2, rc + 2) = the pair the next step transforms first
            int nb_ = rb + 2, nc_ = rc + 2;
            if (nc_ >= H) nc_ -= H;
            if (TILED) {
                // tile-major: one 128-byte line per 8-column tile holds both rows of the pair
                const char* base = reinterpret_cast<const char*>(reinterpret_cast<const float4*>(spec) + (size_t)(nc_ >> 1) * kSpecTile);
                for (int tl = j; tl < Wc / kSpecTile; tl += NT)
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(base + (size_t)tl * (H / 2) * kSpecTile * sizeof(float4)));
            } else if (j == 0) {
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(spec + (size_t)nb_ * Wc), "r"((unsigned)(Wc * sizeof(float2))) : "memory");
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(spec + (size_t)nc_ * Wc), "r"((unsigned)(Wc * sizeof(float2))) : "memory");
            }
        }
#endif
        // ---- spatial step for the columns of this thread's first forward butterfly
        const size_t oa = (size_t)ra * W, ob = (size_t)rb * W, oc = (size_t)rc * W;
        // the spatial step, instantiated for tau >= 0 (clamp) and tau < 0 (dual_of, common.cuh); one uniform branch
        auto spatial = [&](auto tsign) {
        constexpr bool NEG = decltype(tsign)::neg;
        auto clampf3 = [](float q_, float tau_) { return dual_of<NEG>(q_, tau_); };
        auto wfun3 = [](float q_, float tau_) { return fmaf(-2.0f, dual_of<NEG>(q_, tau_), q_); };
#pragma unroll
        for (int ch = 0; ch < R0; ch += CH) {
            // previous dual (STATE_U) or pre-clamp state of rows ra, rb (x and y field) and of row rc (y field); one
            // batch of loads is in flight before the first use.  Zero on the first iteration.
            float ld[CH][5];
#pragma unroll
            for (int i = 0; i < CH; ++i) {
                const int c = j + (ch + i) * NT;
                if (qxi) {
                    ld[i][0] = __ldg(qxi + oa + c); ld[i][1] = __ldg(qxi + ob + c);
                    ld[i][2] = __ldg(qyi + oa + c); ld[i][3] = __ldg(qyi + ob + c); ld[i][4] = __ldg(qyi + oc + c);
                } else {
                    ld[i][0] = ld[i][1] = ld[i][2] = ld[i][3] = ld[i][4] = 0.f;
                }
            }
#pragma unroll
            for (int i = 0; i < CH; ++i) {
                const int r = ch + i;
                const int c = j + r * NT;
                const int cl = (c == 0) ? W - 1 : c - 1;
                const float2 Pc = P[pm(c)], Pl = P[pm(cl)];
                const float2 Fc = F[pm(c)], Fl = F[pm(cl)];
                const float uxa = STATE_U ? ld[i][0] : clampf3(ld[i][0], tau);
                const float uxb = STATE_U ? ld[i][1] : clampf3(ld[i][1], tau);
                const float uya = STATE_U ? ld[i][2] : clampf3(ld[i][2], tau);
                const float uyb = STATE_U ? ld[i][3] : clampf3(ld[i][3], tau);
                const float uyc = STATE_U ? ld[i][4] : clampf3(ld[i][4], tau);
                const float qx_a = Pc.y - Pl.y + uxa;              // deconv.py:108,111,114
                const float qx_b = Fc.x - Fl.x + uxb;
                const float qy_a = Pc.y - Pc.x + uya;              // deconv.py:109,112,115
                const float qy_b = Fc.x - Pc.y + uyb;
                const float qy_c = Fc.y - Fc.x + uyc;
                const float cxa = clampf3(qx_a, tau), cxb = clampf3(qx_b, tau);
                const float cya = clampf3(qy_a, tau), cyb = clampf3(qy_b, tau);
                qxo[oa + c] = STATE_U ? cxa : qx_a; qxo[ob + c] = STATE_U ? cxb : qx_b;
                qyo[oa + c] = STATE_U ? cya : qy_a; qyo[ob + c] = STATE_U ? cyb : qy_b;
                // w = z - u = q - 2 clamp(q);  v = Dx^T w_x + Dy^T w_y         (deconv.py:104)
                const float wxa = fmaf(-2.0f, cxa, qx_a), wxb = fmaf(-2.0f, cxb, qx_b);
                const float wya = fmaf(-2.0f, cya, qy_a), wyb = fmaf(-2.0f, cyb, qy_b);
                const float wyc = wfun3(qy_c, tau);
                // w_x of column c+1 belongs to the next lane; the warp's last lane gets it through shared memory below
                const float nxa = __shfl_down_sync(0xffffffffu, wxa, 1);
                const float nxb = __shfl_down_sync(0xffffffffu, wxb, 1);
                if (lane == 0) edge[warp * R0 + r] = make_float2(wxa, wxb);
                float va = wxa + wya - wyb, vb = wxb + wyb - wyc;
                if (lane != 31) { va -= nxa; vb -= nxb; }
                v[r] = make_float2(va, vb);
            }
        }
        };
        if (tau < 0.f) spatial(TauNeg{}); else spatial(TauPos{});
        __syncthreads();                       // all reads of P (x pair m) are done, the edge values are visible
        RB_ST(2);
        if (lane == 31) {
            // column c+1 of (warp, r) is lane 0 of the next warp, same r; past the last warp it is thread 0 with r+1
#pragma unroll
            for (int r = 0; r < R0; ++r) {
                const float2 e = (warp + 1 < NW) ? edge[(warp + 1) * R0 + r] : edge[(r + 1) % R0];
                v[r].x -= e.x; v[r].y -= e.y;
            }
        }
        dft_big<R0, -1>(v);
        F1::store(S, j, v);                    // S: last read by the third inverse pass, behind a barrier
        __syncthreads();
#pragma unroll
        for (int q = 0; q < ROUNDS2; ++q) {        // x pair m (in P) is dead
            const int jj = j + q * NT;
            if (jj < F2::T) { F2::load(S, jj, v); F2::template butterfly_tab<R0>(v, tab2 + jj % R0); F2::store(P, jj, v); }
        }
        __syncthreads();
        if (j < F3::T) { F3::load(P, j, v); F3::butterfly_reg(v, w3); F3::store(S, j, v); }
        __syncthreads();
        RB_ST(3);
        // ---- split Z = Va + i Vb into the two packed half spectra
        float2* __restrict__ Oa = sout + (size_t)ra * Wc;
        float2* __restrict__ Ob = sout + (size_t)rb * Wc;
        float4* __restrict__ Ot = reinterpret_cast<float4*>(sout) + (size_t)(ra >> 1) * kSpecTile;   // rows (ra, rb) = (even, odd)
        for (int c = j; c < Wc; c += NT) {
            const float2 Z = S[pm(c)];
            float2 Xa, Xb;
            if (c == 0) {
                const float2 Zn = S[pm(Wc)];
                Xa = make_float2(Z.x, Zn.x);
                Xb = make_float2(Z.y, Zn.y);
            } else {
                const float2 Zm = S[pm(W - c)];
                Xa = make_float2(0.5f * (Z.x + Zm.x), 0.5f * (Z.y - Zm.y));
                Xb = make_float2(0.5f * (Z.y + Zm.y), 0.5f * (Zm.x - Z.x));
            }
            if (TILED) {
                Ot[(size_t)(c / kSpecTile) * (H / 2) * kSpecTile + (c % kSpecTile)] = make_float4(Xa.x, Xa.y, Xb.x, Xb.y);
            } else {
                Oa[c] = Xa; Ob[c] = Xb;
            }
        }
        float2* t = P; P = F; F = t;           // the old P is free; S is still being read until the next barrier
        RB_ST(4);
    }
#ifdef ROWS_STATS
    if (threadIdx.x == 0 && (blockIdx.x % 61) == 5 && npv)
        printf("cta %d, %d row pairs: per pair: spectrum loads + I1 %lld | I2, I3 %lld | state loads + spatial %lld | F1, F2, F3 %lld | split + stores %lld\n",
               blockIdx.x, npv, st[0] / (npv + 1), st[1] / (npv + 1), st[2] / npv, st[3] / npv, st[4] / npv);
#endif
}

// ------------------------------------------------------------------------------------------ plain row passes
// ROWS_C2R: packed spectrum -> real rows (unnormalised, + optional bias);  ROWS_R2C: real rows -> packed spectrum, the
// input either a real field or, with r2c_div = 1, the divergence v = D^T(cmap * q) formed while loading (iso=True forward:
// cmap = 2s-1, deconv.py:19-24,104; NULL = unit coefficients), or with r2c_div = 2 the anisotropic v = D^T(q - 2 dual(q))
// of k_rows_big's spatial step (restart of a checkpointed block, backward.cu).  Same passes and tables as the march kernel, one row
// pair at a time per CTA, no halo.  C2R pairs rows (2k-1, 2k), R2C pairs rows (2k, 2k+1): the pairings of the two
// tile-major spectra (common.cuh, kSpecTile), so both layouts work for either mode.
template <int W, int MODE, bool TILED>
__global__ void __launch_bounds__(W / RowBig<W>::R0, RowBig<W>::OCC)
k_rows_big_plain(RowArgs a, int H, int nbands) {
    using RB = RowBig<W>;
    constexpr int R0 = RB::R0, R1 = RB::R1, R2 = RB::R2;
    constexpr int NT = W / R0;
    constexpr int Wc = W / 2;
    constexpr int PAD = RB::PAD;
    constexpr int WB = W + (PAD ? W / PAD : 0);
    constexpr int DIR = (MODE == ROWS_C2R) ? +1 : -1;
    using P1 = BigPass<W, R0, 1, DIR, 1, PAD>;
    using P2 = BigPass<W, R1, R0, DIR, 1, PAD>;
    using P3 = BigPass<W, R2, R0 * R1, DIR, 1, PAD>;
    constexpr int RMAX = (R1 > R2 ? R1 : R2) > R0 ? (R1 > R2 ? R1 : R2) : R0;
    constexpr int ROUNDS2 = (P2::T + NT - 1) / NT;
    static_assert(P3::T <= NT, "pass-3 twiddles are per thread");
    auto pm = [](int n) { return PAD ? n + n / (PAD ? PAD : 1) : n; };
    extern __shared__ float2 smem[];
    float2* A = smem;
    float2* S = smem + WB;
    float2* tab2 = smem + 2 * WB;
    const int j = threadIdx.x;
    const int band = blockIdx.x % nbands;
    const int p = blockIdx.x / nbands;
    const int hh = H >> 1;
    const int k0 = (band * hh) / nbands, k1 = ((band + 1) * hh) / nbands;
    const size_t plane_real = (size_t)p * H * W;
    const float2* __restrict__ tw = a.tw;
    for (int i = j; i < (R1 - 1) * R0; i += NT) {
        const int r = i / R0 + 1, k = i - (r - 1) * R0;
        tab2[i] = __ldg(tw + k * r * (W / (R0 * R1)));
    }
    float2 w3[R2 - 1];
#pragma unroll
    for (int r = 1; r < R2; ++r) w3[r - 1] = __ldg(tw + (j < P3::T ? j * r : 0));
    float2 v[RMAX];
    // passes 1..3 from the registers of pass 1's inputs; the transform ends in `fin` (A for the first store)
    auto passes = [&]() {
        dft_big<R0, DIR>(v);
        P1::store(A, j, v);
        __syncthreads();
#pragma unroll
        for (int q = 0; q < ROUNDS2; ++q) {
            const int jj = j + q * NT;
            if (jj < P2::T) { P2::load(A, jj, v); P2::template butterfly_tab<R0>(v, tab2 + jj % R0); P2::store(S, jj, v); }
        }
        __syncthreads();
        if (j < P3::T) { P3::load(S, j, v); P3::butterfly_reg(v, w3); P3::store(A, j, v); }
        __syncthreads();
    };

    if (MODE == ROWS_C2R) {
        const float2* __restrict__ spec = a.spec_in + (size_t)p * H * Wc;
        float* __restrict__ out = a.real_out + out_plane_offset(a, p, H, W);
        const float bias = a.bias ? __ldg(a.bias) : 0.f;
        const int act = a.act;
        for (int k = k0; k < k1; ++k) {
            const int rb = 2 * k, ra = (k == 0) ? H - 1 : rb - 1;          // rows (2k-1, 2k)
            const float2* __restrict__ Sa = spec + (size_t)ra * Wc;
            const float2* __restrict__ Sb = spec + (size_t)rb * Wc;
            const float4* __restrict__ St = reinterpret_cast<const float4*>(spec) + (size_t)k * kSpecTile;
#pragma unroll
            for (int r = 0; r < R0; ++r) {
                const int n = j + r * NT;
                const bool hi = n > Wc;
                const int c = hi ? W - n : (n == Wc ? 0 : n);
                float2 X, Y;
                if (TILED) {
                    const float4 t = __ldg(St + (size_t)(c / kSpecTile) * (H / 2) * kSpecTile + (c % kSpecTile));
                    X = make_float2(t.x, t.y); Y = make_float2(t.z, t.w);
                } else {
                    X = __ldg(Sa + c); Y = __ldg(Sb + c);
                }
                float2 z = hi ? make_float2(X.x + Y.y, Y.x - X.y) : make_float2(X.x - Y.y, X.y + Y.x);
                if (n == 0) z = make_float2(X.x, Y.x);
                if (n == Wc) z = make_float2(X.y, Y.y);
                v[r] = z;
            }
            passes();
            for (int c = j; c < W; c += NT) {
                const float2 x = A[pm(c)];
                out[(size_t)ra * W + c] = act_apply(x.x + bias, act);
                out[(size_t)rb * W + c] = act_apply(x.y + bias, act);
            }
            __syncthreads();                   // A is rewritten by the next pair
        }
        return;
    }

    // ROWS_R2C
    float2* __restrict__ sout = a.spec_out + (size_t)p * H * Wc;
    const bool div = a.r2c_div != 0;
    const bool unit = (a.cmap == nullptr);
    const float* __restrict__ in = div ? nullptr : a.real_in + plane_real;
    const unsigned char* __restrict__ in8 = (!div && a.real_in_u8) ? a.real_in_u8 + plane_real : nullptr;
    const float* __restrict__ qx = div ? a.qx_in + plane_real : nullptr;
    const float* __restrict__ qy = div ? a.qy_in + plane_real : nullptr;
    const float* __restrict__ kx = a.cmap;
    const float* __restrict__ ky = unit ? nullptr : a.cmap + (size_t)H * W;
    for (int k = k0; k < k1; ++k) {
        const int ra = 2 * k, rb = ra + 1;                                   // rows (2k, 2k+1)
        int rc = rb + 1; if (rc >= H) rc -= H;
        const size_t oa = (size_t)ra * W, ob = (size_t)rb * W, oc = (size_t)rc * W;
        // r2c_div = 2 (checkpointed backward, restart of a block): v = Dx^T w_x + Dy^T w_y with w = q - 2 dual(q) from the
        // saved pre-clamp state, with the expressions and the association of k_rows_big's spatial step, so the packed
        // spectrum equals the one the march wrote in the forward bit for bit.  One uniform branch on the sign of tau.
        auto aniso_div = [&](auto tsign, float tau) {
            constexpr bool NEG = decltype(tsign)::neg;
            auto wf = [](float q_, float tau_) { return fmaf(-2.0f, dual_of<NEG>(q_, tau_), q_); };
#pragma unroll
            for (int r = 0; r < R0; ++r) {
                const int c = j + r * NT;
                const float wxa = wf(__ldg(qx + oa + c), tau), wxb = wf(__ldg(qx + ob + c), tau);
                const float wya = wf(__ldg(qy + oa + c), tau), wyb = wf(__ldg(qy + ob + c), tau), wyc = wf(__ldg(qy + oc + c), tau);
                // w_x of column c+1 from the next lane; a warp's last lane loads it (fewer loads in flight: no spills)
                float wxar = __shfl_down_sync(0xffffffffu, wxa, 1), wxbr = __shfl_down_sync(0xffffffffu, wxb, 1);
                if ((j & 31) == 31) {
                    const int cr = (c == W - 1) ? 0 : c + 1;
                    wxar = wf(__ldg(qx + oa + cr), tau); wxbr = wf(__ldg(qx + ob + cr), tau);
                }
                v[r] = make_float2(wxa + wya - wyb - wxar, wxb + wyb - wyc - wxbr);   // ((w_x + w_y) - w_y below) - w_x right
            }
        };
        if (a.r2c_div == 2) {
            const float tau = a.lmbd[0] / a.rho[0];                          // as in k_rows_big
            if (tau < 0.f) aniso_div(TauNeg{}, tau); else aniso_div(TauPos{}, tau);
        } else {
#pragma unroll
            for (int r = 0; r < R0; ++r) {
                const int c = j + r * NT;
                if (!div) {
                    v[r] = in8 ? make_float2(ld_u8_div255(in8 + oa + c), ld_u8_div255(in8 + ob + c))
                               : make_float2(__ldg(in + oa + c), __ldg(in + ob + c));
                } else {
                    const int cr = (c == W - 1) ? 0 : c + 1;
                    float xa = __ldg(qx + oa + c), xar = __ldg(qx + oa + cr), xb = __ldg(qx + ob + c), xbr = __ldg(qx + ob + cr);
                    float ya = __ldg(qy + oa + c), yb = __ldg(qy + ob + c), yc = __ldg(qy + oc + c);
                    if (!unit) {
                        xa *= __ldg(kx + oa + c); xar *= __ldg(kx + oa + cr); xb *= __ldg(kx + ob + c); xbr *= __ldg(kx + ob + cr);
                        ya *= __ldg(ky + oa + c); yb *= __ldg(ky + ob + c); yc *= __ldg(ky + oc + c);
                    }
                    v[r] = make_float2(xa - xar + ya - yb, xb - xbr + yb - yc);      // D^T: w_x[c] - w_x[c+1] + w_y[r] - w_y[r+1]
                }
            }
        }
        passes();
        float2* __restrict__ Oa = sout + (size_t)ra * Wc;
        float2* __restrict__ Ob = sout + (size_t)rb * Wc;
        float4* __restrict__ Ot = reinterpret_cast<float4*>(sout) + (size_t)k * kSpecTile;
        for (int c = j; c < Wc; c += NT) {
            const float2 Z = A[pm(c)];
            float2 Xa, Xb;
            if (c == 0) {
                const float2 Zn = A[pm(Wc)];
                Xa = make_float2(Z.x, Zn.x);
                Xb = make_float2(Z.y, Zn.y);
            } else {
                const float2 Zm = A[pm(W - c)];
                Xa = make_float2(0.5f * (Z.x + Zm.x), 0.5f * (Z.y - Zm.y));
                Xb = make_float2(0.5f * (Z.y + Zm.y), 0.5f * (Zm.x - Z.x));
            }
            if (TILED) Ot[(size_t)(c / kSpecTile) * (H / 2) * kSpecTile + (c % kSpecTile)] = make_float4(Xa.x, Xa.y, Xb.x, Xb.y);
            else { Oa[c] = Xa; Ob[c] = Xb; }
        }
        __syncthreads();                       // A is rewritten by the next pair
    }
}

template <int W, int MODE, bool TILED>
static int launch_rows_big_plain_w(const Geometry& g, const RowArgs& a, cudaStream_t st) {
    using RB = RowBig<W>;
    constexpr int NT = W / RB::R0;
    const size_t smem = (size_t)(2 * (W + (RB::PAD ? W / RB::PAD : 0)) + (RB::R1 - 1) * RB::R0) * sizeof(float2);
    static std::atomic<bool> attr_set[64];
    int dev = 0;
    ADMM_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev >= 64 || !attr_set[dev]) {
        ADMM_CUDA_CHECK(cudaFuncSetAttribute(k_rows_big_plain<W, MODE, TILED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        if (dev < 64) attr_set[dev] = true;
    }
    const int occ = (int)std::min<size_t>(RB::OCC, (227 * 1024) / (smem + 1024));
    const int hh = g.H / 2;
    int nbands = std::max(1, std::min(hh, (148 * occ * 2) / g.P));        // about two waves
    dim3 grid((unsigned)((size_t)nbands * g.P));
    ProfScope ps(PROF_OTHER, st);
    k_rows_big_plain<W, MODE, TILED><<<grid, NT, smem, st>>>(a, g.H, nbands);
    ADMM_CUDA_CHECK(cudaGetLastError());
    return 0;
}

template <int W>
static int launch_rows_big_plain_t(RowMode mode, const Geometry& g, const RowArgs& a, cudaStream_t st) {
    if (mode == ROWS_C2R)
        return a.tiled ? launch_rows_big_plain_w<W, ROWS_C2R, true>(g, a, st) : launch_rows_big_plain_w<W, ROWS_C2R, false>(g, a, st);
    return a.tiled ? launch_rows_big_plain_w<W, ROWS_R2C, true>(g, a, st) : launch_rows_big_plain_w<W, ROWS_R2C, false>(g, a, st);
}

template <int W, bool STATE_U, bool TILED>
static int launch_rows_big_w(const Geometry& g, const RowArgs& a, cudaStream_t st) {
    constexpr int NT = W / RowBig<W>::R0;
    using RB = RowBig<W>;
    const size_t smem = (size_t)(3 * (W + (RB::PAD ? W / RB::PAD : 0)) + (NT / 32) * RB::R0 + (RB::R1 - 1) * RB::R0) * sizeof(float2);
    static std::atomic<bool> attr_set[64];
    int dev = 0;
    ADMM_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev < 64 && !attr_set[dev]) {
        ADMM_CUDA_CHECK(cudaFuncSetAttribute(k_rows_big<W, STATE_U, TILED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set[dev] = true;
    } else if (dev >= 64) {
        ADMM_CUDA_CHECK(cudaFuncSetAttribute(k_rows_big<W, STATE_U, TILED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    // one wave: as many bands per plane as fill the resident-CTA slots (3 per SM), even band heights
    const int occ = (int)std::min<size_t>(RB::OCC, (227 * 1024) / (smem + 1024));
    int R = options().rows_per_band;
    int nbands;
    const int hh = g.H / 2;
    if (R > 0) {
        nbands = std::max(1, std::min(hh, (g.H + R - 1) / R));
    } else {
        const int slots = 148 * occ;
        nbands = std::max(1, slots / g.P);
        // at least 8 rows per band (halo = one extra inverse FFT per band), more waves instead when P is large
        nbands = std::min(nbands, std::max(1, hh / 4));
    }
    nbands = std::max(1, std::min(nbands, hh));
    dim3 grid((unsigned)((size_t)nbands * g.P));
    ProfScope ps(PROF_ROWS, st);
    k_rows_big<W, STATE_U, TILED><<<grid, NT, smem, st>>>(a, g.H, nbands);
    ADMM_CUDA_CHECK(cudaGetLastError());
    return 0;
}


// all modes of one width: instantiated in exactly one translation unit (rows_big.cu / rows_big2.cu split the widths so
// that the two files compile in parallel)
template <int W>
static int launch_rows_big_width(RowMode mode, const Geometry& g, const RowArgs& a, cudaStream_t st) {
    if (mode == ROWS_R2C || mode == ROWS_C2R) return launch_rows_big_plain_t<W>(mode, g, a, st);
    if (a.tiled) return mode == ROWS_FULL_U ? launch_rows_big_w<W, true, true>(g, a, st) : launch_rows_big_w<W, false, true>(g, a, st);
    return mode == ROWS_FULL_U ? launch_rows_big_w<W, true, false>(g, a, st) : launch_rows_big_w<W, false, false>(g, a, st);
}

}  // namespace admm
