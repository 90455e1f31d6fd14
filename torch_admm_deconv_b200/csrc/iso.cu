// iso.cu -- spatial kernels of the iso=True (block threshold) mode, forward and backward.
//
// block_thresh (deconv.py:19-20) scales every plane of a pixel by s = max(1 - tau / (n + 1e-15), 0) with
// n = sqrt(sum over (batch, channel) of q^2 + 1e-15) (pixelnorm, deconv.py:23-24), separately for the x and the y
// gradient field.  One thread owns one pixel and walks the planes, so the reduction over planes is sequential,
// deterministic and coalesced along the row.  State carried between iterations: q (pre-prox) plus the two
// H x W norm maps; u = (1 - s) q and w = z - u = (2 s - 1) q are rebuilt from them.
#include "common.cuh"

namespace admm {

template <typename T>
__global__ void k_iso_prox(const T* __restrict__ x, const T* __restrict__ qxp, const T* __restrict__ qyp,
                           const T* __restrict__ n_prev, T* __restrict__ qxn, T* __restrict__ qyn,
                           T* __restrict__ n_new, T* __restrict__ c_new, const T* __restrict__ lmbd,
                           const T* __restrict__ rho, int P, int H, int W, int pdl) {
    // launched with programmatic stream serialisation for small (latency-bound) batches: the next kernel of the iteration
    // may start its prologue (twiddle tables) while this one runs; nothing the previous kernel wrote is read before the wait
    if (pdl) { pdl_launch_dependents(); pdl_wait(); }
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= H * W) return;
    const int r = idx / W, c = idx - r * W;
    const int cl = c == 0 ? W - 1 : c - 1, ru = r == 0 ? H - 1 : r - 1;
    const T tau = lmbd[0] / rho[0];
    T ux_scale = T(0), uy_scale = T(0);                     // u_prev = (1 - s_prev) q_prev
    if (n_prev) {
        ux_scale = T(1) - iso_scale(n_prev[idx], tau);
        uy_scale = T(1) - iso_scale(n_prev[(size_t)H * W + idx], tau);
    }
    T sx = T(0), sy = T(0);
    const size_t HW = (size_t)H * W;
    for (int p = 0; p < P; ++p) {
        const T* X = x + p * HW;
        const T xc = X[idx];
        T qx = xc - X[(size_t)r * W + cl];               // deconv.py:108
        T qy = xc - X[(size_t)ru * W + c];               // deconv.py:109
        if (n_prev) {
            qx += ux_scale * qxp[p * HW + idx];
            qy += uy_scale * qyp[p * HW + idx];
        }
        qxn[p * HW + idx] = qx; qyn[p * HW + idx] = qy;
        sx = xfma(qx, qx, sx); sy = xfma(qy, qy, sy);
    }
    const T nx = xsqrt(sx + iso_eps<T>()), ny = xsqrt(sy + iso_eps<T>());   // deconv.py:23-24
    n_new[idx] = nx;
    n_new[HW + idx] = ny;
    if (c_new) {                                              // w = z - u = (2 s - 1) q : coefficient map for the divergence
        c_new[idx] = T(2) * iso_scale(nx, tau) - T(1);
        c_new[HW + idx] = T(2) * iso_scale(ny, tau) - T(1);
    }
}

// v = Dx^T w_x + Dy^T w_y,  w = z - u = (2 s - 1) q        (deconv.py:104 with z = s q, u = q - z)
// cmap (2s-1 per pixel and field) if given, else rebuilt from the norm maps.  grid = (W/256, H, planes)
template <typename T>
__global__ void k_iso_div(const T* __restrict__ qx, const T* __restrict__ qy, const T* __restrict__ nmap,
                          const T* __restrict__ cmap, T* __restrict__ v, const T* __restrict__ lmbd,
                          const T* __restrict__ rho, int H, int W) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= W) return;
    const int r = blockIdx.y;
    const size_t HW = (size_t)H * W;
    const size_t pl = (size_t)blockIdx.z * HW;
    const int cr = c == W - 1 ? 0 : c + 1, rd = r == H - 1 ? 0 : r + 1;
    const size_t m00 = (size_t)r * W + c, m0r = (size_t)r * W + cr, md0 = (size_t)rd * W + c;
    T kx0, kxr, ky0, kyd;
    if (cmap) {
        kx0 = cmap[m00]; kxr = cmap[m0r]; ky0 = cmap[HW + m00]; kyd = cmap[HW + md0];
    } else {
        const T tau = lmbd[0] / rho[0];
        kx0 = T(2) * iso_scale(nmap[m00], tau) - T(1); kxr = T(2) * iso_scale(nmap[m0r], tau) - T(1);
        ky0 = T(2) * iso_scale(nmap[HW + m00], tau) - T(1); kyd = T(2) * iso_scale(nmap[HW + md0], tau) - T(1);
    }
    v[pl + m00] = (kx0 * qx[pl + m00] - kxr * qx[pl + m0r]) + (ky0 * qy[pl + m00] - kyd * qy[pl + md0]);
}

// backward of the block threshold, one kernel:
//   sb_f[pixel] = sum over planes (2 wbar_f - ubar_f) q_f                                   (reduction over planes)
//   qbar = (2s-1) wbar + (1-s) ubar + act sb tau / (n+eps)^2 q / n ;  taubar += act sb (-1/(n+eps))
// A block owns 32 consecutive pixels; its kIsoPG warps split the planes (plane p -> warp p % kIsoPG) and stream over them
// (unrolled, loads of several planes in flight).  The partial sums meet in shared memory and are added in a fixed order
// (deterministic); then every warp sweeps its planes again to apply the result (vbar / ubar / q are re-read; parking
// the first sweep's terms in shared memory or registers was measured and is not faster: the kernel is bound by the
// latency of its many concurrent plane streams, ~3 TB/s).
constexpr int kIsoPG = 4;
template <bool HAS_U, typename T>
__global__ void __launch_bounds__(32 * kIsoPG)
k_iso_bwd_fused(const T* __restrict__ vb, const T* __restrict__ ubx_in, const T* __restrict__ uby_in,
                const T* __restrict__ qx, const T* __restrict__ qy, const T* __restrict__ nmap,
                T* __restrict__ ubx_out, T* __restrict__ uby_out, const T* __restrict__ lmbd,
                const T* __restrict__ rho, double* __restrict__ taubar, int P, int H, int W, int pdl) {
    if (pdl) { pdl_launch_dependents(); pdl_wait(); }         // see k_iso_prox
    __shared__ T red[kIsoPG][2][32];
    const int tx = threadIdx.x & 31, g = threadIdx.x >> 5;
    const size_t HW = (size_t)H * W;
    const size_t idx = (size_t)blockIdx.x * 32 + tx;
    const bool ok = idx < HW;
    size_t ol = 0, ou = 0;
    if (ok) {
        const int r = (int)(idx / W), c = (int)(idx - (size_t)r * W);
        ol = (size_t)r * W + (c == 0 ? W - 1 : c - 1);
        ou = (size_t)(r == 0 ? H - 1 : r - 1) * W + c;
    }
    T ax = T(0), ay = T(0);
    if (ok) {
#pragma unroll 4
        for (int p = g; p < P; p += kIsoPG) {
            const T* V = vb + p * HW;
            const T v0 = V[idx];
            const T wbx = v0 - V[ol], wby = v0 - V[ou];
            const T ux = HAS_U ? ubx_in[p * HW + idx] : T(0), uy = HAS_U ? uby_in[p * HW + idx] : T(0);
            const T qxv = qx[p * HW + idx], qyv = qy[p * HW + idx];
            const T tX = T(2) * wbx - ux, tY = T(2) * wby - uy;
            ax = xfma(tX, qxv, ax);
            ay = xfma(tY, qyv, ay);
        }
    }
    red[g][0][tx] = ax; red[g][1][tx] = ay;
    __syncthreads();
    double tsum = 0.0;
    if (ok) {
        T sbx = T(0), sby = T(0);
#pragma unroll
        for (int i = 0; i < kIsoPG; ++i) { sbx += red[i][0][tx]; sby += red[i][1][tx]; }
        const T tau = lmbd[0] / rho[0];
        const T nx = nmap[idx], ny = nmap[HW + idx];
        const T sx = iso_scale(nx, tau), sy = iso_scale(ny, tau);
        const T kx = (sx > T(0)) ? sbx * tau / ((nx + iso_eps<T>()) * (nx + iso_eps<T>()) * nx) : T(0);
        const T ky = (sy > T(0)) ? sby * tau / ((ny + iso_eps<T>()) * (ny + iso_eps<T>()) * ny) : T(0);
        if (g == 0) {
            if (sx > T(0)) tsum -= (double)sbx / (double)(nx + iso_eps<T>());
            if (sy > T(0)) tsum -= (double)sby / (double)(ny + iso_eps<T>());
        }
#pragma unroll 4
        for (int p = g; p < P; p += kIsoPG) {
            const T* V = vb + p * HW;
            const T v0 = V[idx];
            const T wbx = v0 - V[ol], wby = v0 - V[ou];
            const T ux = HAS_U ? ubx_in[p * HW + idx] : T(0), uy = HAS_U ? uby_in[p * HW + idx] : T(0);
            // (2s-1) wbar + (1-s) ubar + k q  =  s (2 wbar - ubar) + (ubar - wbar) + k q
            ubx_out[p * HW + idx] = xfma(sx, T(2) * wbx - ux, ux - wbx) + kx * qx[p * HW + idx];
            uby_out[p * HW + idx] = xfma(sy, T(2) * wby - uy, uy - wby) + ky * qy[p * HW + idx];
        }
    }
    if (g == 0) {                                              // warp 0 holds the tau-gradient terms of the 32 pixels
        for (int o = 16; o > 0; o >>= 1) tsum += __shfl_down_sync(0xffffffffu, tsum, o);
        if (tx == 0) taubar[blockIdx.x] += tsum;        // per-block slot, single writer (deterministic)
    }
}

// coefficient map 2s-1 of the divergence (both fields) rebuilt from saved norm maps (backward recompute of v_k)
template <typename T>
__global__ void k_iso_cmap(const T* __restrict__ nmap, T* __restrict__ cmap, const T* __restrict__ lmbd,
                           const T* __restrict__ rho, int n2) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n2) return;
    cmap[i] = T(2) * iso_scale(nmap[i], lmbd[0] / rho[0]) - T(1);
}

template <typename T>
static int launch_iso_cmap_t(const Geometry& g, const T* nmap, T* cmap, const T* lmbd, const T* rho, cudaStream_t st) {
    ProfScope ps(PROF_OTHER, st);
    const int n2 = 2 * g.H * g.W;
    k_iso_cmap<<<(n2 + 255) / 256, 256, 0, st>>>(nmap, cmap, lmbd, rho, n2);
    ADMM_CUDA_CHECK(cudaGetLastError());
    return 0;
}

// xbar = Dx^T a_x + Dy^T a_y
template <typename T>
__global__ void k_div_adjoint(const T* __restrict__ ax, const T* __restrict__ ay, T* __restrict__ xb,
                              int H, int W, size_t total) {
    const size_t HW = (size_t)H * W;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % W);
        const size_t rowi = i / W;
        const int r = (int)(rowi % H);
        const size_t pl = (rowi / H) * HW;
        const int cr = c == W - 1 ? 0 : c + 1, rd = r == H - 1 ? 0 : r + 1;
        const size_t m00 = pl + (size_t)r * W + c;
        xb[m00] = (ax[m00] - ax[pl + (size_t)r * W + cr]) + (ay[m00] - ay[pl + (size_t)rd * W + c]);
    }
}

static int ew_grid(size_t total) { return (int)std::min<size_t>((total + 255) / 256, 148 * 16); }

template <typename T>
static int launch_iso_prox_t(const Geometry& g, const T* x, const T* qx_prev, const T* qy_prev, const T* n_prev,
                             T* qx_new, T* qy_new, T* n_new, T* c_new, const T* lmbd, const T* rho, cudaStream_t st) {
    ProfScope ps(PROF_OTHER, st);
    const int n = g.H * g.W;
    const unsigned nctas = (unsigned)((n + 63) / 64);
    if (options().use_pdl && (size_t)g.P * g.H * g.W <= (size_t)4 << 20) {        // a few waves per kernel: launch latency counts
        ADMM_CUDA_CHECK(launch_pdl(k_iso_prox<T>, dim3(nctas), dim3(64), 0, st, x, qx_prev, qy_prev, n_prev, qx_new, qy_new, n_new, c_new,
                                   lmbd, rho, g.P, g.H, g.W, 1));
    } else {
        k_iso_prox<<<nctas, 64, 0, st>>>(x, qx_prev, qy_prev, n_prev, qx_new, qy_new, n_new, c_new, lmbd, rho, g.P, g.H, g.W, 0);
    }
    ADMM_CUDA_CHECK(cudaGetLastError());
    return 0;
}

template <typename T>
static int launch_iso_div_t(const Geometry& g, const T* qx, const T* qy, const T* nmap, const T* cmap, T* v,
                            const T* lmbd, const T* rho, cudaStream_t st) {
    ProfScope ps(PROF_OTHER, st);
    const int bx = g.W >= 256 ? 256 : (g.W >= 128 ? 128 : 64);
    const dim3 grid((g.W + bx - 1) / bx, g.H, g.P);
    if (g.H > 65535 || g.P > 65535) return fail(4, "iso: H and B*C must be <= 65535");
    k_iso_div<<<grid, bx, 0, st>>>(qx, qy, nmap, cmap, v, lmbd, rho, g.H, g.W);
    ADMM_CUDA_CHECK(cudaGetLastError());
    return 0;
}

template <typename T>
static int launch_iso_bwd_t(const Geometry& g, const T* vb, const T* ubx_in, const T* uby_in, const T* qx,
                            const T* qy, const T* nmap, T* sbmap, T* ubx_out, T* uby_out, T* xb,
                            const T* lmbd, const T* rho, double* taubar, cudaStream_t st) {
    (void)sbmap;                                               // the per-pixel sums stay in shared memory
    ProfScope ps(PROF_OTHER, st);
    const size_t total = (size_t)g.P * g.H * g.W;
    const size_t n = (size_t)g.H * g.W;
    const unsigned nb = (unsigned)((n + 31) / 32);
    const bool pdl = options().use_pdl && total <= ((size_t)4 << 20);
    const T* nullf = nullptr;
    if (ubx_in && uby_in) {
        if (pdl) ADMM_CUDA_CHECK(launch_pdl(k_iso_bwd_fused<true, T>, dim3(nb), dim3(32 * kIsoPG), 0, st, vb, ubx_in, uby_in, qx, qy, nmap,
                                            ubx_out, uby_out, lmbd, rho, taubar, g.P, g.H, g.W, 1));
        else k_iso_bwd_fused<true, T><<<nb, 32 * kIsoPG, 0, st>>>(vb, ubx_in, uby_in, qx, qy, nmap, ubx_out, uby_out, lmbd, rho, taubar,
                                                              g.P, g.H, g.W, 0);
    } else {
        if (pdl) ADMM_CUDA_CHECK(launch_pdl(k_iso_bwd_fused<false, T>, dim3(nb), dim3(32 * kIsoPG), 0, st, vb, nullf, nullf, qx, qy, nmap,
                                            ubx_out, uby_out, lmbd, rho, taubar, g.P, g.H, g.W, 1));
        else k_iso_bwd_fused<false, T><<<nb, 32 * kIsoPG, 0, st>>>(vb, nullptr, nullptr, qx, qy, nmap, ubx_out, uby_out, lmbd, rho,
                                                               taubar, g.P, g.H, g.W, 0);
    }
    ADMM_CUDA_CHECK(cudaGetLastError());
    if (xb) {                                                  // else the caller forms D^T qbar inside its R2C row pass
        k_div_adjoint<<<ew_grid(total), 256, 0, st>>>(ubx_out, uby_out, xb, g.H, g.W, total);
        ADMM_CUDA_CHECK(cudaGetLastError());
    }
    return 0;
}

// ---- threshold maps (lambda maps, DESIGN section 11): the kernels above with tau = tau_map[pixel].  With iso = 1 a map is
// shared by every plane (the block threshold scales all planes of a pixel by one factor), so one thread still owns one
// pixel; the backward adds that pixel's tau gradient into taubar_map[pixel] (one writer per launch: deterministic).
__global__ void k_iso_prox_map(const float* __restrict__ x, const float* __restrict__ qxp, const float* __restrict__ qyp,
                               const float* __restrict__ n_prev, float* __restrict__ qxn, float* __restrict__ qyn,
                               float* __restrict__ n_new, float* __restrict__ c_new, const float* __restrict__ tau_map,
                               int P, int H, int W) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= H * W) return;
    const int r = idx / W, c = idx - r * W;
    const int cl = c == 0 ? W - 1 : c - 1, ru = r == 0 ? H - 1 : r - 1;
    const float tau = tau_map[idx];
    float ux_scale = 0.f, uy_scale = 0.f;
    if (n_prev) {
        ux_scale = 1.f - iso_scale(n_prev[idx], tau);
        uy_scale = 1.f - iso_scale(n_prev[(size_t)H * W + idx], tau);
    }
    float sx = 0.f, sy = 0.f;
    const size_t HW = (size_t)H * W;
    for (int p = 0; p < P; ++p) {
        const float* X = x + p * HW;
        const float xc = X[idx];
        float qx = xc - X[(size_t)r * W + cl];
        float qy = xc - X[(size_t)ru * W + c];
        if (n_prev) {
            qx += ux_scale * qxp[p * HW + idx];
            qy += uy_scale * qyp[p * HW + idx];
        }
        qxn[p * HW + idx] = qx; qyn[p * HW + idx] = qy;
        sx = fmaf(qx, qx, sx); sy = fmaf(qy, qy, sy);
    }
    const float nx = sqrtf(sx + iso_eps<float>()), ny = sqrtf(sy + iso_eps<float>());
    n_new[idx] = nx;
    n_new[HW + idx] = ny;
    if (c_new) {
        c_new[idx] = 2.f * iso_scale(nx, tau) - 1.f;
        c_new[HW + idx] = 2.f * iso_scale(ny, tau) - 1.f;
    }
}

__global__ void k_iso_cmap_map(const float* __restrict__ nmap, float* __restrict__ cmap, const float* __restrict__ tau_map,
                               int HW) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 2 * HW) return;
    cmap[i] = 2.f * iso_scale(nmap[i], tau_map[i < HW ? i : i - HW]) - 1.f;
}

template <bool HAS_U>
__global__ void __launch_bounds__(32 * kIsoPG)
k_iso_bwd_map(const float* __restrict__ vb, const float* __restrict__ ubx_in, const float* __restrict__ uby_in,
              const float* __restrict__ qx, const float* __restrict__ qy, const float* __restrict__ nmap,
              float* __restrict__ ubx_out, float* __restrict__ uby_out, const float* __restrict__ tau_map,
              double* __restrict__ taubar_map, int P, int H, int W) {
    __shared__ float red[kIsoPG][2][32];
    const int tx = threadIdx.x & 31, g = threadIdx.x >> 5;
    const size_t HW = (size_t)H * W;
    const size_t idx = (size_t)blockIdx.x * 32 + tx;
    const bool ok = idx < HW;
    size_t ol = 0, ou = 0;
    if (ok) {
        const int r = (int)(idx / W), c = (int)(idx - (size_t)r * W);
        ol = (size_t)r * W + (c == 0 ? W - 1 : c - 1);
        ou = (size_t)(r == 0 ? H - 1 : r - 1) * W + c;
    }
    float ax = 0.f, ay = 0.f;
    if (ok) {
#pragma unroll 4
        for (int p = g; p < P; p += kIsoPG) {
            const float* V = vb + p * HW;
            const float v0 = V[idx];
            const float wbx = v0 - V[ol], wby = v0 - V[ou];
            const float ux = HAS_U ? ubx_in[p * HW + idx] : 0.f, uy = HAS_U ? uby_in[p * HW + idx] : 0.f;
            ax = fmaf(2.f * wbx - ux, qx[p * HW + idx], ax);
            ay = fmaf(2.f * wby - uy, qy[p * HW + idx], ay);
        }
    }
    red[g][0][tx] = ax; red[g][1][tx] = ay;
    __syncthreads();
    if (!ok) return;
    float sbx = 0.f, sby = 0.f;
#pragma unroll
    for (int i = 0; i < kIsoPG; ++i) { sbx += red[i][0][tx]; sby += red[i][1][tx]; }
    const float tau = tau_map[idx];
    const float nx = nmap[idx], ny = nmap[HW + idx];
    const float sx = iso_scale(nx, tau), sy = iso_scale(ny, tau);
    const float kx = (sx > 0.f) ? sbx * tau / ((nx + iso_eps<float>()) * (nx + iso_eps<float>()) * nx) : 0.f;
    const float ky = (sy > 0.f) ? sby * tau / ((ny + iso_eps<float>()) * (ny + iso_eps<float>()) * ny) : 0.f;
    if (g == 0) {
        double t = 0.0;
        if (sx > 0.f) t -= (double)sbx / (double)(nx + iso_eps<float>());
        if (sy > 0.f) t -= (double)sby / (double)(ny + iso_eps<float>());
        taubar_map[idx] += t;
    }
#pragma unroll 4
    for (int p = g; p < P; p += kIsoPG) {
        const float* V = vb + p * HW;
        const float v0 = V[idx];
        const float wbx = v0 - V[ol], wby = v0 - V[ou];
        const float ux = HAS_U ? ubx_in[p * HW + idx] : 0.f, uy = HAS_U ? uby_in[p * HW + idx] : 0.f;
        ubx_out[p * HW + idx] = fmaf(sx, 2.f * wbx - ux, ux - wbx) + kx * qx[p * HW + idx];
        uby_out[p * HW + idx] = fmaf(sy, 2.f * wby - uy, uy - wby) + ky * qy[p * HW + idx];
    }
}

int launch_iso_prox_map(const Geometry& g, const float* x, const float* qx_prev, const float* qy_prev, const float* n_prev,
                        float* qx_new, float* qy_new, float* n_new, float* c_new, const float* tau_map, cudaStream_t st) {
    ProfScope ps(PROF_OTHER, st);
    const int n = g.H * g.W;
    k_iso_prox_map<<<(unsigned)((n + 63) / 64), 64, 0, st>>>(x, qx_prev, qy_prev, n_prev, qx_new, qy_new, n_new, c_new, tau_map,
                                                             g.P, g.H, g.W);
    ADMM_CUDA_CHECK(cudaGetLastError());
    return 0;
}

int launch_iso_cmap_map(const Geometry& g, const float* nmap, float* cmap, const float* tau_map, cudaStream_t st) {
    ProfScope ps(PROF_OTHER, st);
    const int n = g.H * g.W;
    k_iso_cmap_map<<<(2 * n + 255) / 256, 256, 0, st>>>(nmap, cmap, tau_map, n);
    ADMM_CUDA_CHECK(cudaGetLastError());
    return 0;
}

int launch_iso_bwd_map(const Geometry& g, const float* vb, const float* ubx_in, const float* uby_in, const float* qx,
                       const float* qy, const float* nmap, float* ubx_out, float* uby_out, float* xb, const float* tau_map,
                       double* taubar_map, cudaStream_t st) {
    ProfScope ps(PROF_OTHER, st);
    const size_t total = (size_t)g.P * g.H * g.W;
    const unsigned nb = (unsigned)(((size_t)g.H * g.W + 31) / 32);
    if (ubx_in && uby_in)
        k_iso_bwd_map<true><<<nb, 32 * kIsoPG, 0, st>>>(vb, ubx_in, uby_in, qx, qy, nmap, ubx_out, uby_out, tau_map, taubar_map,
                                                        g.P, g.H, g.W);
    else
        k_iso_bwd_map<false><<<nb, 32 * kIsoPG, 0, st>>>(vb, nullptr, nullptr, qx, qy, nmap, ubx_out, uby_out, tau_map, taubar_map,
                                                         g.P, g.H, g.W);
    ADMM_CUDA_CHECK(cudaGetLastError());
    if (xb) {
        k_div_adjoint<<<ew_grid(total), 256, 0, st>>>(ubx_out, uby_out, xb, g.H, g.W, total);
        ADMM_CUDA_CHECK(cudaGetLastError());
    }
    return 0;
}

// float (the solver) and double (the float64 solve, f64.cu) entry points
#define ADMM_ISO_LAUNCHERS(T)                                                                                              \
    int launch_iso_prox(const Geometry& g, const T* x, const T* qx_prev, const T* qy_prev, const T* n_prev, T* qx_new,     \
                        T* qy_new, T* n_new, T* c_new, const T* lmbd, const T* rho, cudaStream_t st) {                     \
        return launch_iso_prox_t(g, x, qx_prev, qy_prev, n_prev, qx_new, qy_new, n_new, c_new, lmbd, rho, st);             \
    }                                                                                                                      \
    int launch_iso_cmap(const Geometry& g, const T* nmap, T* cmap, const T* lmbd, const T* rho, cudaStream_t st) {         \
        return launch_iso_cmap_t(g, nmap, cmap, lmbd, rho, st);                                                            \
    }                                                                                                                      \
    int launch_iso_div(const Geometry& g, const T* qx, const T* qy, const T* nmap, const T* cmap, T* v, const T* lmbd,     \
                       const T* rho, cudaStream_t st) {                                                                    \
        return launch_iso_div_t(g, qx, qy, nmap, cmap, v, lmbd, rho, st);                                                  \
    }                                                                                                                      \
    int launch_iso_bwd(const Geometry& g, const T* vb, const T* ubx_in, const T* uby_in, const T* qx, const T* qy,         \
                       const T* nmap, T* sbmap, T* ubx_out, T* uby_out, T* xb, const T* lmbd, const T* rho,                \
                       double* taubar, cudaStream_t st) {                                                                  \
        return launch_iso_bwd_t(g, vb, ubx_in, uby_in, qx, qy, nmap, sbmap, ubx_out, uby_out, xb, lmbd, rho, taubar, st);  \
    }
ADMM_ISO_LAUNCHERS(float)
ADMM_ISO_LAUNCHERS(double)
#undef ADMM_ISO_LAUNCHERS

}  // namespace admm
