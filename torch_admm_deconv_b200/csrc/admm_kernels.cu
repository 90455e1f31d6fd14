// admm_kernels.cu -- generic (any H, W) kernels of the ADMM-TV solve for sm_100a.
//
// Per ADMM iteration the solve is two kernels (SURVEY.md section 8d, appendix A.2):
//   k_rows<ROWS_FULL> : packed row spectrum of x --C2R rows--> x --prox/dual/divergence--> v --R2C rows-->
//                       packed row spectrum of v            (reads/writes the pre-clamp state q_x, q_y)
//   k_cols<COLS_ITER> : column FFT --> X = A + Bm * V --> inverse column FFT
// Reference statements covered: deconv.py:104 (divergence + rfftn), :106 (freq_c multiply + irfftn),
// :108-109 (Dx, Dy), :111-112 (soft_thresh), :114-115 (dual update).
//
// State carried between iterations is q = D x + u_prev (pre-clamp); u = clamp(q, +-tau) is rebuilt on
// load, z is never stored (z - u = q - 2 clamp(q)).  The same buffers double as the saved state of the
// backward.
#include "common.cuh"
#include "tables.cuh"

namespace admm {

// ------------------------------------------------------------------------------------------ twiddles
__global__ void k_twiddles(float2* __restrict__ tw, double2* __restrict__ twd, int N) {
    int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    double s, c;
    sincospi(-2.0 * (double)n / (double)N, &s, &c);
    tw[n] = make_float2((float)c, (float)s);
    twd[n] = make_double2(c, s);
}

int launch_twiddles(float2* tw, double2* twd, int N, cudaStream_t st) {
    ProfScope ps(PROF_OTHER, st);
    k_twiddles<<<(N + 255) / 256, 256, 0, st>>>(tw, twd, N);
    ADMM_CUDA_CHECK(cudaGetLastError());
    return 0;
}

// the float64 solve keeps the double table only (same values as k_twiddles' twd)
__global__ void k_twiddles_f64(double2* __restrict__ twd, int N) {
    int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    double s, c;
    sincospi(-2.0 * (double)n / (double)N, &s, &c);
    twd[n] = make_double2(c, s);
}

int launch_twiddles_f64(double2* twd, int N, cudaStream_t st) {
    ProfScope ps(PROF_OTHER, st);
    k_twiddles_f64<<<(N + 255) / 256, 256, 0, st>>>(twd, N);
    ADMM_CUDA_CHECK(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------------------------------ tables
// G[a][v] = sum_b kern[a][b] e^{-2 pi i v b / W},  v in [0, W/2]        (row DFT of the zero-padded PSF)
template <typename T>
__global__ void k_kern_rowdft(const T* __restrict__ kern, int ks, int W,
                              const double2* __restrict__ twWd, double2* __restrict__ G) {
    const int Wh = W / 2 + 1;
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= ks * Wh) return;
    int a = idx / Wh, v = idx - a * Wh;
    double re = 0.0, im = 0.0;
    for (int b = 0; b < ks; ++b) {
        double2 w = twWd[(int)(((long long)v * b) % W)];
        double kv = (double)kern[a * ks + b];
        re += kv * w.x; im += kv * w.y;
    }
    G[idx] = make_double2(re, im);
}

template <typename T>
__global__ void k_tables(int H, int W, int Wc, int ks, const double2* __restrict__ G,
                         const double2* __restrict__ twHd, const double2* __restrict__ twWd,
                         const T* __restrict__ rho_p,
                         T* __restrict__ Bm, T* __restrict__ Bq,
                         cplx_t<T>* __restrict__ Mul, cplx_t<T>* __restrict__ Mq) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= H * Wc) return;
    const int u = idx / Wc, c = idx - u * Wc;
    const double rho = (double)rho_p[0];
    TabEntry e = table_entry(u, c, H, W, ks, G, twHd, twWd, rho);
    if (c > 0) {
        Bm[idx] = (T)e.bm;
        Mul[idx] = make_cplx((T)e.mul.x, (T)e.mul.y);
    } else {
        // packed column 0 carries the DC and the Nyquist column: X = A0 + Bp Z + Bq conj(Z[-u])
        TabEntry n = e;
        if ((W & 1) == 0) n = table_entry(u, W / 2, H, W, ks, G, twHd, twWd, rho);
        Bm[idx] = (T)(0.5 * (e.bm + n.bm));
        Bq[u] = (T)(0.5 * (e.bm - n.bm));
        Mul[idx] = make_cplx((T)(0.5 * (e.mul.x + n.mul.x)), (T)(0.5 * (e.mul.y + n.mul.y)));
        Mq[u] = make_cplx((T)(0.5 * (e.mul.x - n.mul.x)), (T)(0.5 * (e.mul.y - n.mul.y)));
    }
}

template <typename T>
static int launch_tables_t(const Geometry& g, const double2* twWd, const double2* twHd, double2* kdft, T* Bm, T* Bq,
                           cplx_t<T>* Mul, cplx_t<T>* Mq, const T* kern, int ksize, const T* rho, cudaStream_t st) {
    if (ksize > 0) {
        int n = ksize * (g.W / 2 + 1);
        ProfScope ps(PROF_OTHER, st);
        k_kern_rowdft<<<(n + 127) / 128, 128, 0, st>>>(kern, ksize, g.W, twWd, kdft);
        ADMM_CUDA_CHECK(cudaGetLastError());
    }
    int n = g.H * g.Wc;
    ProfScope ps(PROF_OTHER, st);
    k_tables<<<(n + 127) / 128, 128, 0, st>>>(g.H, g.W, g.Wc, ksize, kdft, twHd, twWd, rho, Bm, Bq, Mul, Mq);
    ADMM_CUDA_CHECK(cudaGetLastError());
    return 0;
}

int launch_tables(const Geometry& g, const Workspace& ws, const float* kern, int ksize,
                  const float* rho, cudaStream_t st) {
    return launch_tables_t(g, ws.twWd, ws.twHd, ws.kdft, ws.Bm, ws.Bq, ws.Mul, ws.Mq, kern, ksize, rho, st);
}

int launch_tables_f64(const Geometry& g, const double2* twWd, const double2* twHd, double2* kdft, double* Bm, double* Bq,
                      double2* Mul, double2* Mq, const double* kern, int ksize, const double* rho, cudaStream_t st) {
    return launch_tables_t(g, twWd, twHd, kdft, Bm, Bq, Mul, Mq, kern, ksize, rho, st);
}

// ------------------------------------------------------------------------------------------ row pass
template <typename T> __device__ __forceinline__ T clampf(T q, T tau) { return dual_any(q, tau); }      // u(q), any sign of tau (common.cuh)
// w = z - u with z = soft_thresh(q), u = q - z  ==>  w = q - 2 clamp(q)    (deconv.py:15-16, 104, 114-115)
template <typename T> __device__ __forceinline__ T wfun(T q, T tau) { return xfma(T(-2), clampf(q, tau), q); }
// the fused activation of the layer exists in float only (the float64 solve never sets one)
__device__ __forceinline__ float act_out(float v, int act) { return act_apply(v, act); }
__device__ __forceinline__ double act_out(double v, int) { return v; }

// Two real rows <-> one complex FFT (z = row_a + i row_b).  Merge builds the full complex spectrum of z
// from the two packed half spectra; split is the inverse.
template <typename V>
__device__ __forceinline__ void merge_pairs(const V* __restrict__ S, int H, int W, int Wc, int BS,
                                            int rfirst, int nrows, int NP, V* __restrict__ buf) {
    using T = real_t<V>;
    const bool even = (W & 1) == 0;
    for (int w = threadIdx.x; w < NP * Wc; w += blockDim.x) {
        const int m = w / Wc, c = w - m * Wc;
        int ra = rfirst + 2 * m; ra %= H; if (ra < 0) ra += H;
        V a = S[(size_t)ra * Wc + c];
        V b = make_cplx(T(0), T(0));
        if (2 * m + 1 < nrows) {
            int rb = ra + 1; if (rb >= H) rb -= H;
            b = S[(size_t)rb * Wc + c];
        }
        if (c == 0) {
            buf[m] = make_cplx(a.x, b.x);
            if (even) buf[(W / 2) * BS + m] = make_cplx(a.y, b.y);
        } else {
            buf[c * BS + m] = make_cplx(a.x - b.y, a.y + b.x);
            buf[(W - c) * BS + m] = make_cplx(a.x + b.y, b.x - a.y);
        }
    }
}

template <typename V>
__device__ __forceinline__ void split_pairs(const V* __restrict__ res, int W, int Wc, int BS,
                                            int r0, int Rb, int NP, V* __restrict__ out) {
    using T = real_t<V>;
    const bool even = (W & 1) == 0;
    for (int w = threadIdx.x; w < NP * Wc; w += blockDim.x) {
        const int m = w / Wc, c = w - m * Wc;
        const V Z = res[c * BS + m];
        V Xa, Xb;
        if (c == 0) {
            V Zn = even ? res[(W / 2) * BS + m] : make_cplx(T(0), T(0));
            Xa = make_cplx(Z.x, Zn.x);
            Xb = make_cplx(Z.y, Zn.y);
        } else {
            const V Zm = res[(W - c) * BS + m];
            Xa = make_cplx(T(0.5) * (Z.x + Zm.x), T(0.5) * (Z.y - Zm.y));
            Xb = make_cplx(T(0.5) * (Z.y + Zm.y), T(0.5) * (Zm.x - Z.x));
        }
        out[(size_t)(r0 + 2 * m) * Wc + c] = Xa;
        if (2 * m + 1 < Rb) out[(size_t)(r0 + 2 * m + 1) * Wc + c] = Xb;
    }
}

// Threads per CTA of the generic kernels: float as tuned; double at most 256 (a radix-16 butterfly holds 32 doubles:
// with 512 or 1024 threads the 128 / 64 registers per thread spill, with 256 nothing does)
template <typename T> constexpr int kGenericMaxThreads = sizeof(T) == 4 ? 1024 : 256;

template <int MODE, typename T>
__global__ void __launch_bounds__(kGenericMaxThreads<T>)
k_rows(RowArgsT<T> a, FftPlan plan, int H, int W, int Wc, int R, int BS, int nbands) {
    using V = cplx_t<T>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    V* bufA = reinterpret_cast<V*>(smem_raw);
    V* bufB = bufA + (size_t)W * BS;
    V* tw = bufB + (size_t)W * BS;
    const int band = blockIdx.x % nbands;
    const int p = blockIdx.x / nbands;
    const int r0 = band * R;
    const int Rb = min(R, H - r0);
    const size_t plane_real = (size_t)p * H * W;
    const size_t plane_spec = (size_t)p * H * Wc;
    for (int i = threadIdx.x; i < W; i += blockDim.x) tw[i] = a.tw[i];

    if (MODE == ROWS_R2C) {
        const int NP = (Rb + 1) / 2;
        const T* in = a.real_in + plane_real;
        const unsigned char* in8 = a.real_in_u8 ? a.real_in_u8 + plane_real : nullptr;
        for (int w = threadIdx.x; w < NP * W; w += blockDim.x) {
            const int m = w / W, c = w - m * W;
            const int ra = r0 + 2 * m;
            T xa = in8 ? (T)ld_u8_div255(in8 + (size_t)ra * W + c) : in[(size_t)ra * W + c];
            T xb = (2 * m + 1 < Rb) ? (in8 ? (T)ld_u8_div255(in8 + (size_t)(ra + 1) * W + c) : in[(size_t)(ra + 1) * W + c]) : T(0);
            bufA[c * BS + m] = make_cplx(xa, xb);
        }
        __syncthreads();
        V* res = fft_batched<-1>(bufA, bufB, plan, NP, BS, tw);
        split_pairs(res, W, Wc, BS, r0, Rb, NP, a.spec_out + plane_spec);
        return;
    }

    if (MODE == ROWS_C2R) {
        const int NP = (Rb + 1) / 2;
        merge_pairs(a.spec_in + plane_spec, H, W, Wc, BS, r0, Rb, NP, bufA);
        __syncthreads();
        V* res = fft_batched<+1>(bufA, bufB, plan, NP, BS, tw);
        T* out = a.real_out + out_plane_offset(a, p, H, W);
        const T bias = a.bias ? a.bias[0] : T(0);
        const int act = a.act;
        for (int w = threadIdx.x; w < NP * W; w += blockDim.x) {
            const int m = w / W, c = w - m * W;
            const int ra = r0 + 2 * m;
            const V z = res[c * BS + m];
            out[(size_t)ra * W + c] = act_out(z.x + bias, act);
            if (2 * m + 1 < Rb) out[(size_t)(ra + 1) * W + c] = act_out(z.y + bias, act);
        }
        return;
    }

    if (MODE == ROWS_FULL) {
        // rows r0-1 .. r0+Rb  (Rb + 2 rows, circular), as pairs (i = 2m, 2m+1)
        const int nrows = Rb + 2;
        const int NP = (nrows + 1) / 2;
        merge_pairs(a.spec_in + plane_spec, H, W, Wc, BS, r0 - 1, nrows, NP, bufA);
        __syncthreads();
        V* res = fft_batched<+1>(bufA, bufB, plan, NP, BS, tw);
        V* zb = (res == bufA) ? bufB : bufA;
        const T tau = a.lmbd[0] / a.rho[0];                         // deconv.py:44
        const T* qxi = a.qx_in ? a.qx_in + plane_real : nullptr;
        const T* qyi = a.qy_in ? a.qy_in + plane_real : nullptr;
        T* qxo = a.qx_out + plane_real;
        T* qyo = a.qy_out + plane_real;
        const int NPv = (Rb + 1) / 2;
        for (int w = threadIdx.x; w < NPv * W; w += blockDim.x) {
            const int m = w / W, c = w - m * W;
            const int cl = (c == 0) ? W - 1 : c - 1;
            const int cr = (c == W - 1) ? 0 : c + 1;
            const V P0c = res[c * BS + m],  P1c = res[c * BS + m + 1];
            const V P0l = res[cl * BS + m], P1l = res[cl * BS + m + 1];
            const V P0r = res[cr * BS + m], P1r = res[cr * BS + m + 1];
            const int ra = r0 + 2 * m;
            const bool hasb = (2 * m + 1 < Rb);
            int rb = ra + 1; if (rb >= H) rb -= H;
            int rc = rb + 1; if (rc >= H) rc -= H;
            // previous dual u = clamp(q_prev)   (q_prev == 0 on the first iteration)
            T uxa = 0, uxar = 0, uya = 0, uyb = 0, uxb = 0, uxbr = 0, uyc = 0;
            if (qxi) {
                uxa  = clampf(qxi[(size_t)ra * W + c], tau);
                uxar = clampf(qxi[(size_t)ra * W + cr], tau);
                uya  = clampf(qyi[(size_t)ra * W + c], tau);
                uyb  = clampf(qyi[(size_t)rb * W + c], tau);
                if (hasb) {
                    uxb  = clampf(qxi[(size_t)rb * W + c], tau);
                    uxbr = clampf(qxi[(size_t)rb * W + cr], tau);
                    uyc  = clampf(qyi[(size_t)rc * W + c], tau);
                }
            }
            const T xu = P0c.x;                                  // row ra-1
            const T xa_c = P0c.y, xa_l = P0l.y, xa_r = P0r.y;    // row ra
            const T xb_c = P1c.x, xb_l = P1l.x, xb_r = P1r.x;    // row ra+1
            const T xd = P1c.y;                                  // row ra+2
            const T qx_a  = xa_c - xa_l + uxa;                   // deconv.py:108,111,114
            const T qx_ar = xa_r - xa_c + uxar;
            const T qy_a  = xa_c - xu + uya;                     // deconv.py:109,112,115
            const T qy_b  = xb_c - xa_c + uyb;
            const T va = wfun(qx_a, tau) - wfun(qx_ar, tau) + wfun(qy_a, tau) - wfun(qy_b, tau);   // deconv.py:104
            qxo[(size_t)ra * W + c] = qx_a;
            qyo[(size_t)ra * W + c] = qy_a;
            T vb = 0;
            if (hasb) {
                const T qx_b  = xb_c - xb_l + uxb;
                const T qx_br = xb_r - xb_c + uxbr;
                const T qy_c  = xd - xb_c + uyc;
                vb = wfun(qx_b, tau) - wfun(qx_br, tau) + wfun(qy_b, tau) - wfun(qy_c, tau);
                qxo[(size_t)rb * W + c] = qx_b;
                qyo[(size_t)rb * W + c] = qy_b;
            }
            zb[c * BS + m] = make_cplx(va, vb);
        }
        __syncthreads();
        V* res2 = fft_batched<-1>(zb, res, plan, NPv, BS, tw);
        split_pairs(res2, W, Wc, BS, r0, Rb, NPv, a.spec_out + plane_spec);
        return;
    }
}

template <typename T>
static size_t rows_smem(int W, int BS) { return ((size_t)2 * W * BS + W) * sizeof(cplx_t<T>); }

// the generic engine (any W); float and double
template <typename T>
static int launch_rows_generic(RowMode mode, const Geometry& g, const RowArgsT<T>& a, cudaStream_t st) {
    if (mode == ROWS_ADJ || mode == ROWS_FULL_U) return fail(4, "this row-pass mode exists for power-of-two widths only");
    FftPlan plan;
    if (!make_plan(g.W, plan)) return fail(4, "cannot plan row FFT length");
    const size_t kMax = 227 * 1024;
    const int halo = (mode == ROWS_FULL) ? 2 : 0;
    int R = options().rows_per_band;
    if (R <= 0) R = 16;
    R = std::max(2, std::min(R, g.H + (g.H & 1)));
    R &= ~1;
    int BS = 0;
    for (;; R -= 2) {
        int NP = (R + halo + 1) / 2;
        BS = NP | 1;
        if (rows_smem<T>(g.W, BS) <= kMax) break;
        if (rows_smem<T>(g.W, NP) <= kMax) { BS = NP; break; }
        if (R <= 2) return fail(4, "row FFT does not fit in shared memory (W too large for the generic kernel)");
    }
    // prefer bands that leave >= 2 CTAs per SM when the image is wide
    while (R > 4 && rows_smem<T>(g.W, ((R + halo + 1) / 2) | 1) > 100 * 1024) {
        R -= 2; BS = ((R + halo + 1) / 2) | 1;
    }
    const int nbands = (g.H + R - 1) / R;
    const size_t smem = rows_smem<T>(g.W, BS);
    // one or two fat CTAs per SM need more warps each to keep the SM busy
    const int threads = std::min(kGenericMaxThreads<T>, options().threads > 0 ? options().threads.load()
                                              : (smem > 113 * 1024 ? 1024 : (smem > 75 * 1024 ? 512 : 256)));
    dim3 grid((unsigned)((size_t)nbands * g.P));
    // the opt-in shared-memory limit is a per-device function attribute: raised once to the maximum (the call costs
    // several microseconds of host time, which dominated small problems when it was repeated for every launch)
    int dev_id = 0;
    ADMM_CUDA_CHECK(cudaGetDevice(&dev_id));
#define ADMM_LAUNCH_ROWS(M)                                                                                \
    do {                                                                                                   \
        static std::atomic<bool> attr_set[64];                                                                     \
        if (dev_id >= 64 || !attr_set[dev_id]) {                                                           \
            ADMM_CUDA_CHECK(cudaFuncSetAttribute(k_rows<M, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMax)); \
            if (dev_id < 64) attr_set[dev_id] = true;                                                      \
        }                                                                                                  \
        k_rows<M, T><<<grid, threads, smem, st>>>(a, plan, g.H, g.W, g.Wc, R, BS, nbands);                  \
    } while (0)
    ProfScope ps(mode == ROWS_FULL ? PROF_ROWS : PROF_OTHER, st);
    switch (mode) {
        case ROWS_R2C: ADMM_LAUNCH_ROWS(ROWS_R2C); break;
        case ROWS_C2R: ADMM_LAUNCH_ROWS(ROWS_C2R); break;
        case ROWS_FULL: ADMM_LAUNCH_ROWS(ROWS_FULL); break;
        default: break;
    }
#undef ADMM_LAUNCH_ROWS
    ADMM_CUDA_CHECK(cudaGetLastError());
    return 0;
}

int launch_rows(RowMode mode, const Geometry& g, const RowArgs& a, cudaStream_t st) {
    if (rows_pow2_supported(g)) return launch_rows_pow2(mode, g, a, st);
    if ((mode == ROWS_FULL || mode == ROWS_FULL_U) && rows_big_supported(g)) return launch_rows_big(mode, g, a, st);
    if ((mode == ROWS_R2C || mode == ROWS_C2R) && rows_big_supported(g)) return launch_rows_big_plain(mode, g, a, st);
    return launch_rows_generic(mode, g, a, st);
}

// float64: the generic engine only (no specialised double kernels)
int launch_rows(RowMode mode, const Geometry& g, const RowArgsT<double>& a, cudaStream_t st) {
    return launch_rows_generic(mode, g, a, st);
}

// ------------------------------------------------------------------------------------------ column pass
// Real: float or double (T is the tile width here)
template <int MODE, typename Real>
__global__ void __launch_bounds__(kGenericMaxThreads<Real>)
k_cols(ColArgsT<Real> a, FftPlan plan, int H, int Wc, int T, int ntiles) {
    using V = cplx_t<Real>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    V* bufA = reinterpret_cast<V*>(smem_raw);
    V* bufB = bufA + (size_t)H * T;
    V* tw = bufB + (size_t)H * T;
    const int tile = blockIdx.x % ntiles;
    const int p = blockIdx.x / ntiles;
    const int c0 = tile * T;
    const int Tb = min(T, Wc - c0);
    const size_t plane = (size_t)p * H * Wc;
    for (int i = threadIdx.x; i < H; i += blockDim.x) tw[i] = a.tw[i];
    const V* in = a.spec_in + plane;
    for (int w = threadIdx.x; w < H * T; w += blockDim.x) {
        const int u = w / T, t = w - u * T;
        bufA[w] = (t < Tb) ? in[(size_t)u * Wc + c0 + t] : make_cplx(Real(0), Real(0));
    }
    __syncthreads();
    V* res;
    if (MODE == COLS_FFT_INV) {
        res = fft_batched<+1>(bufA, bufB, plan, T, T, tw);
    } else if (MODE == COLS_BM_INV || MODE == COLS_CMUL_INV || MODE == COLS_INIT_SPEC) {
        res = bufA;                                   // the input already is a full (column-transformed) spectrum
    } else {
        res = fft_batched<-1>(bufA, bufB, plan, T, T, tw);
    }
    if (MODE == COLS_INIT || MODE == COLS_ITER || MODE == COLS_BM_INV || MODE == COLS_CMUL_INV || MODE == COLS_INIT_SPEC) {
        V* other = (res == bufA) ? bufB : bufA;
        V* Ap = (MODE == COLS_INIT || MODE == COLS_ITER || MODE == COLS_INIT_SPEC) ? a.A + plane : nullptr;
        for (int w = threadIdx.x; w < H * T; w += blockDim.x) {
            const int u = w / T, t = w - u * T;
            V o = make_cplx(Real(0), Real(0));
            if (t < Tb) {
                const int c = c0 + t;
                const V Z = res[w];
                if (MODE == COLS_ITER || MODE == COLS_BM_INV) {
                    // X = A + Bm F(v)      (deconv.py:104-106 with freq_c, rho folded into A and Bm)
                    // COLS_BM_INV: the same self-adjoint operator without A (backward: vbar = F^-1[Bm F(xbar)])
                    const V Av = (MODE == COLS_ITER) ? Ap[(size_t)u * Wc + c] : make_cplx(Real(0), Real(0));
                    const Real bm = a.Bm[(size_t)u * Wc + c];
                    o = make_cplx(xfma(bm, Z.x, Av.x), xfma(bm, Z.y, Av.y));
                    if (c == 0) {
                        const int um = (u == 0) ? 0 : H - u;
                        const V Zm = res[um * T + t];
                        const Real bq = a.Bq[u];
                        o.x = xfma(bq, Zm.x, o.x);
                        o.y = xfma(-bq, Zm.y, o.y);
                    }
                } else if (MODE == COLS_CMUL_INV) {
                    // adjoint of A = Mul F(y):  ybar = F^-1[conj(Mul) sum_k F(xbar_k)]
                    o = cmul(cconj(a.Mul[(size_t)u * Wc + c]), Z);
                    if (c == 0) {
                        const int um = (u == 0) ? 0 : H - u;
                        const V Zm = res[um * T + t];
                        o = cadd(o, cmul(cconj(a.Mq[u]), cconj(Zm)));
                    }
                } else {
                    // A = sigma ph F(y) / den   (freq_c * rfftn(H_t(xin)), deconv.py:57,99,104)
                    o = cmul(a.Mul[(size_t)u * Wc + c], Z);
                    if (c == 0) {
                        const int um = (u == 0) ? 0 : H - u;
                        const V Zm = res[um * T + t];
                        o = cadd(o, cmul(a.Mq[u], cconj(Zm)));
                    }
                    Ap[(size_t)u * Wc + c] = o;
                }
            }
            other[w] = o;
        }
        __syncthreads();
        res = fft_batched<+1>(other, res, plan, T, T, tw);
    }
    V* out = a.spec_out + plane;
    for (int w = threadIdx.x; w < H * T; w += blockDim.x) {
        const int u = w / T, t = w - u * T;
        if (t < Tb) out[(size_t)u * Wc + c0 + t] = res[w];
    }
}

template <typename Real>
static size_t cols_smem(int H, int T) { return ((size_t)2 * H * T + H) * sizeof(cplx_t<Real>); }

template <typename Real>
static int launch_cols_generic(ColMode mode, const Geometry& g, const ColArgsT<Real>& a, cudaStream_t st) {
    FftPlan plan;
    if (!make_plan(g.H, plan)) return fail(4, "cannot plan column FFT length");
    const size_t kMax = 227 * 1024;
    int T = options().cols_per_tile;
    if (T <= 0) {
        T = 16;
        while (T > 4 && cols_smem<Real>(g.H, T) > 80 * 1024) T >>= 1;       // keep >= 32-byte global runs
    }
    while (T > 1 && cols_smem<Real>(g.H, T) > kMax) T >>= 1;
    if (cols_smem<Real>(g.H, T) > kMax) return fail(4, "column FFT does not fit in shared memory (H too large for the generic kernel)");
    T = std::min(T, std::max(1, g.Wc));
    const int ntiles = (g.Wc + T - 1) / T;
    const size_t smem = cols_smem<Real>(g.H, T);
    const int threads = std::min(kGenericMaxThreads<Real>, options().threads > 0 ? options().threads.load()
                                              : (smem > 113 * 1024 ? 1024 : (smem > 75 * 1024 ? 512 : 256)));
    dim3 grid((unsigned)((size_t)ntiles * g.P));
    int dev_id = 0;
    ADMM_CUDA_CHECK(cudaGetDevice(&dev_id));
#define ADMM_LAUNCH_COLS(M)                                                                                \
    do {                                                                                                   \
        static std::atomic<bool> attr_set[64];                                                                     \
        if (dev_id >= 64 || !attr_set[dev_id]) {                                                           \
            ADMM_CUDA_CHECK(cudaFuncSetAttribute(k_cols<M, Real>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMax)); \
            if (dev_id < 64) attr_set[dev_id] = true;                                                      \
        }                                                                                                  \
        k_cols<M, Real><<<grid, threads, smem, st>>>(a, plan, g.H, g.Wc, T, ntiles);                        \
    } while (0)
    ProfScope ps(mode == COLS_ITER ? PROF_COLS : PROF_OTHER, st);
    switch (mode) {
        case COLS_FFT_FWD: ADMM_LAUNCH_COLS(COLS_FFT_FWD); break;
        case COLS_FFT_INV: ADMM_LAUNCH_COLS(COLS_FFT_INV); break;
        case COLS_INIT: ADMM_LAUNCH_COLS(COLS_INIT); break;
        case COLS_ITER: ADMM_LAUNCH_COLS(COLS_ITER); break;
        case COLS_BM_INV: ADMM_LAUNCH_COLS(COLS_BM_INV); break;
        case COLS_CMUL_INV: ADMM_LAUNCH_COLS(COLS_CMUL_INV); break;
        case COLS_INIT_SPEC: ADMM_LAUNCH_COLS(COLS_INIT_SPEC); break;
    }
#undef ADMM_LAUNCH_COLS
    ADMM_CUDA_CHECK(cudaGetLastError());
    return 0;
}

int launch_cols(ColMode mode, const Geometry& g, const ColArgs& a, cudaStream_t st) {
    if (cols_pow2_mode_supported(mode) && cols_pow2_supported(g)) return launch_cols_pow2(mode, g, a, st);
    if ((mode == COLS_ITER || mode == COLS_INIT) && cols_big_supported(g)) return launch_cols_big(mode, g, a, st);
    return launch_cols_generic(mode, g, a, st);
}

int launch_cols(ColMode mode, const Geometry& g, const ColArgsT<double>& a, cudaStream_t st) {
    return launch_cols_generic(mode, g, a, st);
}

// float64: whether the generic passes of a solve fit in shared memory (the smallest band / tile the launchers above would
// pick), so that an unsupported size fails before anything is launched
int check_generic_f64(const Geometry& g, bool full_rows) {
    const size_t kMax = 227 * 1024;
    FftPlan plan;
    if (!make_plan(g.W, plan)) return fail(4, "cannot plan row FFT length");
    if (!make_plan(g.H, plan)) return fail(4, "cannot plan column FFT length");
    const int halo = full_rows ? 2 : 0;
    const size_t rows = rows_smem<double>(g.W, (2 + halo + 1) / 2);
    if (rows > kMax)
        return fail(4, "float64 row FFT does not fit in shared memory: W = " + std::to_string(g.W) + " needs " +
                       std::to_string(rows) + " bytes, the limit is " + std::to_string(kMax) +
                       (full_rows ? " (iso = 0 keeps two halo rows: W <= 2905)" : " (W <= 4842)"));
    const size_t cols = cols_smem<double>(g.H, 1);
    if (cols > kMax)
        return fail(4, "float64 column FFT does not fit in shared memory: H = " + std::to_string(g.H) + " needs " +
                       std::to_string(cols) + " bytes, the limit is " + std::to_string(kMax) + " (H <= 4842)");
    return 0;
}

}  // namespace admm
