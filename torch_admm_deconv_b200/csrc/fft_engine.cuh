// fft_engine.cuh -- generic (any length) batched shared-memory FFT for sm_100a.
//
// Layout: NB independent length-N complex sequences live in shared memory "batch fastest":
//     buf[n * BS + b],  n in [0,N), b in [0,NB), BS >= NB.
// Consecutive threads take consecutive b for the same butterfly index, so every shared-memory access of
// a warp is a run of consecutive float2 (conflict-free for any N, any radix) and the twiddle is
// warp-uniform.  The transform is an autosort Stockham: natural order in, natural order out, ping-pong
// between two buffers, one __syncthreads per pass.  Radices 2,3,4,5,8,9,15,16 are unrolled in registers; any
// other prime factor runs a generic O(p^2) pass, so every length is supported (D7 of SURVEY.md: the
// reference transforms exactly (H, W), deconv.py:49,104-106, no padding to a power of two allowed).
//
// This is the fallback / arbitrary-size engine.  The specialised power-of-two kernels are in
// fft_pow2.cuh.  Everything here is templated on the element type V (float2, or double2 for the float64 solve of
// f64.cu); in the double2 layout a warp-wide run is 512 bytes, still conflict-free.
#pragma once
#include <cuda_runtime.h>

namespace admm {

constexpr int kMaxPasses = 24;

struct FftPlan {
    int n;
    int npass;
    int radix[kMaxPasses];
};

__host__ inline bool make_plan(int n, FftPlan& p) {
    p.n = n; p.npass = 0;
    if (n < 1) return false;
    int m = n;
    // big composite radices first (fewest shared-memory passes), then what is left of the powers of 2, 3, 5
    const int pref[9] = {16, 15, 9, 8, 4, 2, 3, 5, 7};
    for (int i = 0; i < 9; ++i) {
        while (m > 1 && m % pref[i] == 0) {
            if (p.npass >= kMaxPasses) return false;
            p.radix[p.npass++] = pref[i]; m /= pref[i];
        }
    }
    for (int f = 11; m > 1; f += 2) {
        while (m % f == 0) {
            if (p.npass >= kMaxPasses) return false;
            p.radix[p.npass++] = f; m /= f;
        }
        if (f > 46341) return false;
    }
    return true;
}

// ---- element types.  The engine runs on float2 (the solver) and double2 (the float64 solve, f64.cu); `real_t<V>` is the
// component type.  The float overloads are the original single-precision code; the double ones mirror them.
template <typename V> struct real_of;
template <> struct real_of<float2> { using type = float; };
template <> struct real_of<double2> { using type = double; };
template <typename V> using real_t = typename real_of<V>::type;
template <typename T> struct cplx_of;
template <> struct cplx_of<float> { using type = float2; };
template <> struct cplx_of<double> { using type = double2; };
template <typename T> using cplx_t = typename cplx_of<T>::type;

__device__ __forceinline__ float2 make_cplx(float x, float y) { return make_float2(x, y); }
__device__ __forceinline__ double2 make_cplx(double x, double y) { return make_double2(x, y); }
// real constants: the float instantiation uses the float literal itself (not a rounded double), so its values are exact
template <typename T> __device__ __forceinline__ constexpr T rconst(float f, double d);
template <> __device__ __forceinline__ constexpr float rconst<float>(float f, double) { return f; }
template <> __device__ __forceinline__ constexpr double rconst<double>(float, double d) { return d; }
#define ADMM_RC(T, x) ::admm::rconst<T>(x##f, x)
__device__ __forceinline__ float xfma(float a, float b, float c) { return fmaf(a, b, c); }
__device__ __forceinline__ double xfma(double a, double b, double c) { return fma(a, b, c); }
__device__ __forceinline__ float xmin(float a, float b) { return fminf(a, b); }
__device__ __forceinline__ double xmin(double a, double b) { return fmin(a, b); }
__device__ __forceinline__ float xmax(float a, float b) { return fmaxf(a, b); }
__device__ __forceinline__ double xmax(double a, double b) { return fmax(a, b); }
__device__ __forceinline__ float xabs(float a) { return fabsf(a); }
__device__ __forceinline__ double xabs(double a) { return fabs(a); }
__device__ __forceinline__ float xsqrt(float a) { return sqrtf(a); }
__device__ __forceinline__ double xsqrt(double a) { return sqrt(a); }

__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
    return make_float2(fmaf(a.x, b.x, -a.y * b.y), fmaf(a.x, b.y, a.y * b.x));
}
__device__ __forceinline__ float2 cconj(float2 a) { return make_float2(a.x, -a.y); }
__device__ __forceinline__ double2 cadd(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ double2 csub(double2 a, double2 b) { return make_double2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ double2 cmul(double2 a, double2 b) {
    return make_double2(fma(a.x, b.x, -a.y * b.y), fma(a.x, b.y, a.y * b.x));
}
__device__ __forceinline__ double2 cconj(double2 a) { return make_double2(a.x, -a.y); }
// multiply by -i*DIR... : DIR=-1 (forward) -> multiply by -i ; DIR=+1 (inverse) -> multiply by +i
template <int DIR, typename V> __device__ __forceinline__ V mul_dir_i(V a) {
    return DIR < 0 ? make_cplx(a.y, -a.x) : make_cplx(-a.y, a.x);
}
// forward twiddle table holds e^{-2 pi i n/N}; the inverse transform conjugates it
template <int DIR, typename V> __device__ __forceinline__ V tw_load(const V* tw, int idx) {
    V w = tw[idx];
    if (DIR > 0) w.y = -w.y;
    return w;
}

// ---------------------------------------------------------------- in-register DFTs, natural order out
template <int DIR, typename V> __device__ __forceinline__ void dft2(V& a, V& b) {
    V t = a; a = cadd(t, b); b = csub(t, b);
}
template <int DIR, typename V> __device__ __forceinline__ void dft3(V* v) {
    using T = real_t<V>;
    const T c = ADMM_RC(T, -0.5), s = ADMM_RC(T, 0.86602540378443864676);
    V t1 = cadd(v[1], v[2]);
    V t2 = make_cplx(xfma(c, t1.x, v[0].x), xfma(c, t1.y, v[0].y));
    V d = csub(v[1], v[2]);
    V t3 = mul_dir_i<DIR>(make_cplx(s * d.x, s * d.y));   // -i s d (fwd) / +i s d (inv)
    v[0] = cadd(v[0], t1);
    v[1] = cadd(t2, t3);
    v[2] = csub(t2, t3);
}
template <int DIR, typename V> __device__ __forceinline__ void dft4(V* v) {
    V t0 = cadd(v[0], v[2]), t1 = csub(v[0], v[2]);
    V t2 = cadd(v[1], v[3]), t3 = mul_dir_i<DIR>(csub(v[1], v[3]));
    v[0] = cadd(t0, t2); v[2] = csub(t0, t2);
    v[1] = cadd(t1, t3); v[3] = csub(t1, t3);
}
template <int DIR, typename V> __device__ __forceinline__ void dft5(V* v) {
    using T = real_t<V>;
    const T c1 = ADMM_RC(T, 0.30901699437494742410), c2 = ADMM_RC(T, -0.80901699437494742410);
    const T s1 = ADMM_RC(T, 0.95105651629515357212), s2 = ADMM_RC(T, 0.58778525229247312917);
    V a1 = cadd(v[1], v[4]), a2 = cadd(v[2], v[3]);
    V b1 = csub(v[1], v[4]), b2 = csub(v[2], v[3]);
    V r1 = make_cplx(v[0].x + c1 * a1.x + c2 * a2.x, v[0].y + c1 * a1.y + c2 * a2.y);
    V r2 = make_cplx(v[0].x + c2 * a1.x + c1 * a2.x, v[0].y + c2 * a1.y + c1 * a2.y);
    V i1 = mul_dir_i<DIR>(make_cplx(s1 * b1.x + s2 * b2.x, s1 * b1.y + s2 * b2.y));
    V i2 = mul_dir_i<DIR>(make_cplx(s2 * b1.x - s1 * b2.x, s2 * b1.y - s1 * b2.y));
    v[0] = cadd(v[0], cadd(a1, a2));
    v[1] = cadd(r1, i1); v[4] = csub(r1, i1);
    v[2] = cadd(r2, i2); v[3] = csub(r2, i2);
}
template <int DIR, typename V> __device__ __forceinline__ void dft8(V* v) {
    using T = real_t<V>;
    const T h = ADMM_RC(T, 0.70710678118654752440);
    // radix-2 stage
    V a0 = cadd(v[0], v[4]), a4 = csub(v[0], v[4]);
    V a1 = cadd(v[1], v[5]), a5 = csub(v[1], v[5]);
    V a2 = cadd(v[2], v[6]), a6 = csub(v[2], v[6]);
    V a3 = cadd(v[3], v[7]), a7 = csub(v[3], v[7]);
    // twiddles w8^k on the odd half: w8 = (1 -+ i)/sqrt2, w8^2 = -+i, w8^3 = (-1 -+ i)/sqrt2
    V t5 = mul_dir_i<DIR>(a5);                       // -+i a5
    a5 = make_cplx(h * (a5.x + t5.x), h * (a5.y + t5.y));   // (1 -+ i)/sqrt2 * a5
    a6 = mul_dir_i<DIR>(a6);
    V t7 = mul_dir_i<DIR>(a7);
    a7 = make_cplx(h * (t7.x - a7.x), h * (t7.y - a7.y));   // (-1 -+ i)/sqrt2 * a7
    // two radix-4 on (a0,a1,a2,a3) and (a4,a5,a6,a7)
    V e[4] = {a0, a1, a2, a3};
    V o[4] = {a4, a5, a6, a7};
    dft4<DIR>(e); dft4<DIR>(o);
    v[0] = e[0]; v[2] = e[1]; v[4] = e[2]; v[6] = e[3];
    v[1] = o[0]; v[3] = o[1]; v[5] = o[2]; v[7] = o[3];
}
// multiply by e^{-+ 2 pi i m / n} given (cos, sin) of the positive angle: forward uses (c, -s), inverse (c, +s)
template <int DIR, typename V> __device__ __forceinline__ V mul_tw(V a, real_t<V> c, real_t<V> s) {
    return DIR < 0 ? make_cplx(xfma(a.x, c, a.y * s), xfma(a.y, c, -a.x * s))
                   : make_cplx(xfma(a.x, c, -a.y * s), xfma(a.y, c, a.x * s));
}
// Composite radices (Cooley-Tukey N1 x N2 in registers, n = N2 n1 + n2, k = k1 + N1 k2): they halve the number of
// shared-memory passes of the mixed-radix sizes (3840 = 16*16*15, 2160 = 16*15*9).
template <int DIR, typename V> __device__ __forceinline__ void dft16(V* v) {
    using T = real_t<V>;
    const T c1 = ADMM_RC(T, 0.92387953251128673848), s1 = ADMM_RC(T, 0.38268343236508978178), h = ADMM_RC(T, 0.70710678118654752440);
    V y[4][4];
#pragma unroll
    for (int n2 = 0; n2 < 4; ++n2) {
        V t[4] = {v[n2], v[n2 + 4], v[n2 + 8], v[n2 + 12]};
        dft4<DIR>(t);
#pragma unroll
        for (int k1 = 0; k1 < 4; ++k1) y[n2][k1] = t[k1];
    }
    // twiddles w16^{n2 k1}
    y[1][1] = mul_tw<DIR>(y[1][1], c1, s1);  y[1][2] = mul_tw<DIR>(y[1][2], h, h);    y[1][3] = mul_tw<DIR>(y[1][3], s1, c1);
    y[2][1] = mul_tw<DIR>(y[2][1], h, h);    y[2][2] = mul_dir_i<DIR>(y[2][2]);       y[2][3] = mul_tw<DIR>(y[2][3], -h, h);
    y[3][1] = mul_tw<DIR>(y[3][1], s1, c1);  y[3][2] = mul_tw<DIR>(y[3][2], -h, h);   y[3][3] = mul_tw<DIR>(y[3][3], -c1, -s1);
#pragma unroll
    for (int k1 = 0; k1 < 4; ++k1) {
        V t[4] = {y[0][k1], y[1][k1], y[2][k1], y[3][k1]};
        dft4<DIR>(t);
#pragma unroll
        for (int k2 = 0; k2 < 4; ++k2) v[k1 + 4 * k2] = t[k2];
    }
}
template <int DIR, typename V> __device__ __forceinline__ void dft9(V* v) {
    using T = real_t<V>;
    V y[3][3];
#pragma unroll
    for (int n2 = 0; n2 < 3; ++n2) {
        V t[3] = {v[n2], v[n2 + 3], v[n2 + 6]};
        dft3<DIR>(t);
#pragma unroll
        for (int k1 = 0; k1 < 3; ++k1) y[n2][k1] = t[k1];
    }
    y[1][1] = mul_tw<DIR>(y[1][1], ADMM_RC(T, 0.76604444311897801345), ADMM_RC(T, 0.64278760968653925190));
    y[1][2] = mul_tw<DIR>(y[1][2], ADMM_RC(T, 0.17364817766693041445), ADMM_RC(T, 0.98480775301220802032));
    y[2][1] = mul_tw<DIR>(y[2][1], ADMM_RC(T, 0.17364817766693041445), ADMM_RC(T, 0.98480775301220802032));
    y[2][2] = mul_tw<DIR>(y[2][2], ADMM_RC(T, -0.93969262078590831688), ADMM_RC(T, 0.34202014332566887944));
#pragma unroll
    for (int k1 = 0; k1 < 3; ++k1) {
        V t[3] = {y[0][k1], y[1][k1], y[2][k1]};
        dft3<DIR>(t);
#pragma unroll
        for (int k2 = 0; k2 < 3; ++k2) v[k1 + 3 * k2] = t[k2];
    }
}
template <int DIR, typename V> __device__ __forceinline__ void dft15(V* v) {
    using T = real_t<V>;
    // N1 = 3 (n1), N2 = 5 (n2): n = 5 n1 + n2, k = k1 + 3 k2
    V y[5][3];
#pragma unroll
    for (int n2 = 0; n2 < 5; ++n2) {
        V t[3] = {v[n2], v[n2 + 5], v[n2 + 10]};
        dft3<DIR>(t);
#pragma unroll
        for (int k1 = 0; k1 < 3; ++k1) y[n2][k1] = t[k1];
    }
    // twiddles w15^{n2 k1}: exponents 1,2 | 2,4 | 3,6 | 4,8
    y[1][1] = mul_tw<DIR>(y[1][1], ADMM_RC(T, 0.91354545764260086660), ADMM_RC(T, 0.40673664307580015276));
    y[1][2] = mul_tw<DIR>(y[1][2], ADMM_RC(T, 0.66913060635885823757), ADMM_RC(T, 0.74314482547739413310));
    y[2][1] = mul_tw<DIR>(y[2][1], ADMM_RC(T, 0.66913060635885823757), ADMM_RC(T, 0.74314482547739413310));
    y[2][2] = mul_tw<DIR>(y[2][2], ADMM_RC(T, -0.10452846326765333207), ADMM_RC(T, 0.99452189536827340088));
    y[3][1] = mul_tw<DIR>(y[3][1], ADMM_RC(T, 0.30901699437494745126), ADMM_RC(T, 0.95105651629515353118));
    y[3][2] = mul_tw<DIR>(y[3][2], ADMM_RC(T, -0.80901699437494734024), ADMM_RC(T, 0.58778525229247324813));
    y[4][1] = mul_tw<DIR>(y[4][1], ADMM_RC(T, -0.10452846326765333207), ADMM_RC(T, 0.99452189536827340088));
    y[4][2] = mul_tw<DIR>(y[4][2], ADMM_RC(T, -0.97814760073380568883), ADMM_RC(T, -0.20791169081775906502));
#pragma unroll
    for (int k1 = 0; k1 < 3; ++k1) {
        V t[5] = {y[0][k1], y[1][k1], y[2][k1], y[3][k1], y[4][k1]};
        dft5<DIR>(t);
#pragma unroll
        for (int k2 = 0; k2 < 5; ++k2) v[k1 + 3 * k2] = t[k2];
    }
}
template <int R, int DIR, typename V> __device__ __forceinline__ void dftR(V* v) {
    if (R == 2) dft2<DIR>(v[0], v[1]);
    else if (R == 3) dft3<DIR>(v);
    else if (R == 4) dft4<DIR>(v);
    else if (R == 5) dft5<DIR>(v);
    else if (R == 8) dft8<DIR>(v);
    else if (R == 9) dft9<DIR>(v);
    else if (R == 15) dft15<DIR>(v);
    else if (R == 16) dft16<DIR>(v);
}

// ---------------------------------------------------------------- one Stockham pass
template <int R, int DIR, typename V>
__device__ __forceinline__ void stockham_pass(const V* __restrict__ src, V* __restrict__ dst,
                                              int N, int Ns, int NB, int BS, const V* __restrict__ tw) {
    const int T = N / R;
    const int tws = N / (Ns * R);
    const int work = T * NB;
    for (int w = threadIdx.x; w < work; w += blockDim.x) {
        const int j = w / NB;
        const int b = w - j * NB;
        const int k = j % Ns;
        V v[R];
#pragma unroll
        for (int r = 0; r < R; ++r) v[r] = src[(j + r * T) * BS + b];
        if (Ns > 1) {
#pragma unroll
            for (int r = 1; r < R; ++r) v[r] = cmul(v[r], tw_load<DIR>(tw, k * r * tws));
        }
        dftR<R, DIR>(v);
        const int j0 = (j - k) * R + k;
#pragma unroll
        for (int r = 0; r < R; ++r) dst[(j0 + r * Ns) * BS + b] = v[r];
    }
}

// generic radix (any prime p): out[m] = sum_r src[j + rT] * w_N^{ r (k + Ns m) N/(Ns p) }
// The direct sum runs in double for both element types: accumulated in float, its rounding error grows with p (5-7x
// that of scipy's fp32 FFT at p = 1021, 23-27x at p = 9677); in double each output is rounded once, when it is stored.
template <int DIR, typename V>
__device__ __forceinline__ void stockham_pass_generic(const V* __restrict__ src, V* __restrict__ dst,
                                                      int N, int R, int Ns, int NB, int BS, const V* __restrict__ tw) {
    const int T = N / R;
    const int tws = N / (Ns * R);
    const int work = T * NB * R;          // one output per work item
    for (int w = threadIdx.x; w < work; w += blockDim.x) {
        const int b = w % NB;
        const int jm = w / NB;
        const int j = jm % T;
        const int m = jm / T;
        const int k = j % Ns;
        const long long step = (long long)(k + Ns * m) * tws;    // < N
        double2 acc = make_double2(0.0, 0.0);
        int idx = 0;
        const int st = (int)(step % N);
        for (int r = 0; r < R; ++r) {
            V x = src[(j + r * T) * BS + b];
            V wv = tw_load<DIR>(tw, idx);
            acc.x = fma((double)x.x, (double)wv.x, fma(-(double)x.y, (double)wv.y, acc.x));
            acc.y = fma((double)x.x, (double)wv.y, fma((double)x.y, (double)wv.x, acc.y));
            idx += st; if (idx >= N) idx -= N;
        }
        const int j0 = (j - k) * R + k;
        dst[(j0 + m * Ns) * BS + b] = make_cplx((real_t<V>)acc.x, (real_t<V>)acc.y);
    }
}

// Transforms NB sequences (see layout above).  The caller must have synchronised after filling `src`.
// Returns the buffer that holds the result (either src or dst); a __syncthreads() has been executed
// after the last pass, so the result is visible to every thread of the block.
template <int DIR, typename V>
__device__ V* fft_batched(V* src, V* dst, const FftPlan& plan, int NB, int BS, const V* __restrict__ tw) {
    const int N = plan.n;
    int Ns = 1;
    for (int p = 0; p < plan.npass; ++p) {
        const int R = plan.radix[p];
        switch (R) {
            case 2: stockham_pass<2, DIR>(src, dst, N, Ns, NB, BS, tw); break;
            case 3: stockham_pass<3, DIR>(src, dst, N, Ns, NB, BS, tw); break;
            case 4: stockham_pass<4, DIR>(src, dst, N, Ns, NB, BS, tw); break;
            case 5: stockham_pass<5, DIR>(src, dst, N, Ns, NB, BS, tw); break;
            case 8: stockham_pass<8, DIR>(src, dst, N, Ns, NB, BS, tw); break;
            case 9: stockham_pass<9, DIR>(src, dst, N, Ns, NB, BS, tw); break;
            case 15: stockham_pass<15, DIR>(src, dst, N, Ns, NB, BS, tw); break;
            case 16: stockham_pass<16, DIR>(src, dst, N, Ns, NB, BS, tw); break;
            default: stockham_pass_generic<DIR>(src, dst, N, R, Ns, NB, BS, tw); break;
        }
        __syncthreads();
        V* t = src; src = dst; dst = t;
        Ns *= R;
    }
    return src;
}

}  // namespace admm
