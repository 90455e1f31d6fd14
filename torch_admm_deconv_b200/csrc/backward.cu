// backward.cu -- hand-derived adjoint of the unrolled ADMM-TV loop (replaces stock autograd through
// deconv.py:103-115).  Derivation and fp64 validation against the reference's autograd: SURVEY.md appendix B,
// oracle/admm_oracle.py:admm_tv_backward, tests/golden/grad_*.npz.
//
// With x_{k+1} = F^-1[A + Bm F(v_k)], q_{k+1} = D x_{k+1} + clamp(q_k), w = q - 2 clamp(q), v_k = D^T w_k, the reverse
// sweep over k = N-1 .. 0 is
//     (k < N-1)  qbar = wbar + 1[|q_{k+1}| < tau] (ubar - 2 wbar);  taubar += sum (ubar - 2 wbar) 1[|q| >= tau] sign(q)
//                xbar = D^T qbar;  ubar <- qbar                       (k = N-1: xbar = grad_out)
//     G = F(xbar);  Gs += G;  C1 += sum_planes conj(G) F(y);  GV += sum_planes conj(G) F(v_k)
//     vbar = F^-1[Bm G];  wbar = D vbar
// and   ybar = F^-1[conj(sigma ph / den) Gs],  rho/lambda/kernel gradients from C1, GV and taubar.
// The forward saved only the pre-clamp fields q_k; v_k is recomputed from q_k and its spectrum from v_k.
// This first version favours reuse (generic FFT passes + elementwise kernels, any H, W) over fusion.
#include <algorithm>
#include <cstring>

#include "../../include/admm_b200.h"
#include "common.cuh"
#include "tables.cuh"

namespace admm {

struct BwdWorkspace {
    float2* ZG; float2* ZV; float2* Gs;     // packed spectra, per plane
    float*  vb; float* xb;                  // real fields
    double2* C1; double2* GV;               // nsplit x H x (W/2+1) partial sums (one slice per plane group, fixed order)
    double2* S;                             // H x (W/2+1)
    double2* Tk;                            // H x ksize
    float2*  GVn;                           // planes x H: Nyquist-column products of the fused column pass
    double*  tau_part;                      // n_tau per-CTA partial sums of the tau gradient (slot = blockIdx.x)
    double*  rho_part;                      // n_rho per-CTA partial sums of the spectral rho gradient
    int nsplit; size_t n_tau, n_rho;
    // checkpointed training (ckpt_interval K >= 2): scratch to re-run one block of the forward
    float*  ck_slots;                       // K-1 slots of [q_x, q_y]
    float2* ck_A; float2* ck_S0; float2* ck_S1;
    float*  ck_v;
    double* taubar_map;                     // threshold maps: per-element tau gradient, accumulated over the sweep
    size_t total;
};

static inline size_t align_up_b(size_t x) { return (x + 255) & ~(size_t)255; }

// tau_map_planes > 0: a solve with a threshold map; its tau-gradient accumulator (one double per element of the sweep's
// terms: P x H x W for iso = 0, H x W for iso = 1) is carved after everything else, so the scalar layout is unchanged
static size_t carve_backward(const Geometry& g, int ksize, int ckpt, char* base, BwdWorkspace* out, int tau_map_planes = 0) {
    size_t off = 0;
    auto take = [&](size_t bytes) { char* p = base ? base + off : nullptr; off += align_up_b(bytes); return p; };
    BwdWorkspace w;
    const size_t HWh = (size_t)g.H * (g.W / 2 + 1);
    w.ZG = (float2*)take(g.spec_bytes);
    w.ZV = (float2*)take(g.spec_bytes);
    w.Gs = (float2*)take(g.spec_bytes);
    w.vb = (float*)take(g.field_bytes);
    w.xb = (float*)take(g.field_bytes);
    // Every reduction of the backward is two-stage and runs in a fixed order (no floating-point atomics): gradients are
    // bit-identical from run to run.  Plane groups for the C1 / GV sums: at most 64, capped at 256 MB of partials.
    w.nsplit = (int)std::max<size_t>(1, std::min<size_t>(std::min(g.P, 64), ((size_t)256 << 20) / (2 * HWh * sizeof(double2))));
    w.C1 = (double2*)take(w.nsplit * HWh * sizeof(double2));
    w.GV = (double2*)take(w.nsplit * HWh * sizeof(double2));
    w.S  = (double2*)take(HWh * sizeof(double2));
    w.Tk = (double2*)take((size_t)g.H * (ksize > 0 ? ksize : 1) * sizeof(double2));
    w.GVn = (float2*)take((size_t)g.P * g.H * sizeof(float2));
    // slot = blockIdx.x of the kernel that produces the partial: fused row pass (<= P * H/2 CTAs), generic spatial
    // kernel (<= 148 * 16), iso kernel (H*W/32)
    w.n_tau = std::max<size_t>(std::max<size_t>((size_t)g.P * (g.H / 2 + 1), 148 * 16), ((size_t)g.H * g.W + 31) / 32);
    w.tau_part = (double*)take(w.n_tau * sizeof(double));
    w.n_rho = (HWh + 127) / 128;
    w.rho_part = (double*)take(w.n_rho * sizeof(double));
    w.ck_slots = nullptr; w.ck_A = w.ck_S0 = w.ck_S1 = nullptr; w.ck_v = nullptr;
    if (ckpt >= 2) {
        w.ck_slots = (float*)take((size_t)(ckpt - 1) * 2 * g.field_bytes);
        w.ck_A = (float2*)take(g.spec_bytes);
        w.ck_S0 = (float2*)take(g.spec_bytes);
        w.ck_S1 = (float2*)take(g.spec_bytes);
        w.ck_v = (float*)take(g.field_bytes);
    }
    w.taubar_map = nullptr;
    if (tau_map_planes > 0)
        w.taubar_map = (double*)take((g.iso ? (size_t)g.H * g.W : (size_t)g.P * g.H * g.W) * sizeof(double));
    w.total = off;
    if (out) *out = w;
    return off;
}

size_t backward_extra_bytes(const Geometry& g, int ksize, int ckpt) { return carve_backward(g, ksize, ckpt, nullptr, nullptr); }

// ------------------------------------------------------------------------------------------ spatial kernels
// Templated on the real type: float for the solver, double for the float64 solve (f64.cu).
template <typename T>
__device__ __forceinline__ T qbar_of(T wb, T ub, T q, T tau) {
    return (xabs(q) < tau) ? (ub - wb) : wb;          // wbar + m (ubar - 2 wbar)
}

// adjoint of prox / dual update / gradient for the state produced by iteration k+1
template <typename T>
__global__ void k_bwd_spatial(const T* __restrict__ vb, const T* __restrict__ ubx_in, const T* __restrict__ uby_in,
                              const T* __restrict__ qx, const T* __restrict__ qy,
                              T* __restrict__ ubx_out, T* __restrict__ uby_out, T* __restrict__ xb,
                              const T* __restrict__ lmbd, const T* __restrict__ rho,
                              double* __restrict__ taubar, int H, int W, size_t total) {
    const T tau = lmbd[0] / rho[0];
    double tsum = 0.0;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(idx % W);
        const size_t rowi = idx / W;
        const int r = (int)(rowi % H);
        const size_t pl = (rowi / H) * (size_t)H * W;
        const int cl = c == 0 ? W - 1 : c - 1, cr = c == W - 1 ? 0 : c + 1;
        const int ru = r == 0 ? H - 1 : r - 1, rd = r == H - 1 ? 0 : r + 1;
        const T* V = vb + pl;
        const T v00 = V[(size_t)r * W + c];
        const T wbx = v00 - V[(size_t)r * W + cl];                       // (Dx vbar)[r][c]
        const T wby = v00 - V[(size_t)ru * W + c];                       // (Dy vbar)[r][c]
        const T wbx_r = V[(size_t)r * W + cr] - v00;                     // (Dx vbar)[r][c+1]
        const T wby_d = V[(size_t)rd * W + c] - v00;                     // (Dy vbar)[r+1][c]
        const size_t i00 = pl + (size_t)r * W + c, i0r = pl + (size_t)r * W + cr, id0 = pl + (size_t)rd * W + c;
        const T ubx = ubx_in ? ubx_in[i00] : T(0), uby = uby_in ? uby_in[i00] : T(0);
        const T ubx_r = ubx_in ? ubx_in[i0r] : T(0), uby_d = uby_in ? uby_in[id0] : T(0);
        const T qx0 = qx[i00], qy0 = qy[i00];
        const T qbx = qbar_of(wbx, ubx, qx0, tau), qby = qbar_of(wby, uby, qy0, tau);
        const T qbx_r = qbar_of(wbx_r, ubx_r, qx[i0r], tau), qby_d = qbar_of(wby_d, uby_d, qy[id0], tau);
        ubx_out[i00] = qbx; uby_out[i00] = qby;
        xb[i00] = (qbx - qbx_r) + (qby - qby_d);                             // Dx^T qbar_x + Dy^T qbar_y
        if (xabs(qx0) >= tau) tsum += (double)((ubx - T(2) * wbx) * (qx0 > T(0) ? T(1) : (qx0 < T(0) ? T(-1) : T(0))));
        if (xabs(qy0) >= tau) tsum += (double)((uby - T(2) * wby) * (qy0 > T(0) ? T(1) : (qy0 < T(0) ? T(-1) : T(0))));
    }
    // block reduction -> this block's slot (single writer; the launches of a sweep are stream-ordered)
    __shared__ double red[32];
    for (int o = 16; o > 0; o >>= 1) tsum += __shfl_down_sync(0xffffffffu, tsum, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = tsum;
    __syncthreads();
    if (threadIdx.x < 32) {
        double v = (threadIdx.x < (blockDim.x + 31) / 32) ? red[threadIdx.x] : 0.0;
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (threadIdx.x == 0) taubar[blockIdx.x] += v;
    }
}

// v = Dx^T w_x + Dy^T w_y with w = q - 2 clamp(q)   (recomputed from the saved pre-clamp state; deconv.py:104)
template <typename T>
__global__ void k_bwd_recompute_v(const T* __restrict__ qx, const T* __restrict__ qy, T* __restrict__ v,
                                  const T* __restrict__ lmbd, const T* __restrict__ rho, int H, int W, size_t total) {
    const T tau = lmbd[0] / rho[0];
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(idx % W);
        const size_t rowi = idx / W;
        const int r = (int)(rowi % H);
        const size_t pl = (rowi / H) * (size_t)H * W;
        const int cr = c == W - 1 ? 0 : c + 1, rd = r == H - 1 ? 0 : r + 1;
        // same operations in the same order as the forward's fused spatial step (rows_pow2.cu, admm_kernels.cu), so a
        // checkpointed backward that restarts the forward from a saved state reproduces its fields bit for bit
        auto wf = [tau](T q) { return xfma(T(-2), dual_any(q, tau), q); };
        const size_t i00 = pl + (size_t)r * W + c;
        v[i00] = wf(qx[i00]) - wf(qx[pl + (size_t)r * W + cr]) + wf(qy[i00]) - wf(qy[pl + (size_t)rd * W + c]);
    }
}

// ---- threshold maps (lambda maps, DESIGN section 11): the two kernels above with tau read per element.  tau of element
// i of plane p is tau_map[(tmp > 1 ? p : 0) H W + pixel]; the tau gradient of element i is added into taubar[i]
// (P x H x W doubles: one writer per element and launch, so the sums are deterministic).  float only.
__device__ __forceinline__ size_t tau_index(size_t i, size_t HW, int tmp) { return tmp > 1 ? i : i % HW; }

__global__ void k_bwd_spatial_map(const float* __restrict__ vb, const float* __restrict__ ubx_in,
                                  const float* __restrict__ uby_in, const float* __restrict__ qx,
                                  const float* __restrict__ qy, float* __restrict__ ubx_out, float* __restrict__ uby_out,
                                  float* __restrict__ xb, const float* __restrict__ tau_map, int tmp,
                                  double* __restrict__ taubar, int H, int W, size_t total) {
    const size_t HW = (size_t)H * W;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(idx % W);
        const size_t rowi = idx / W;
        const int r = (int)(rowi % H);
        const size_t pl = (rowi / H) * HW;
        const int cl = c == 0 ? W - 1 : c - 1, cr = c == W - 1 ? 0 : c + 1;
        const int ru = r == 0 ? H - 1 : r - 1, rd = r == H - 1 ? 0 : r + 1;
        const float* V = vb + pl;
        const float v00 = V[(size_t)r * W + c];
        const float wbx = v00 - V[(size_t)r * W + cl];
        const float wby = v00 - V[(size_t)ru * W + c];
        const float wbx_r = V[(size_t)r * W + cr] - v00;
        const float wby_d = V[(size_t)rd * W + c] - v00;
        const size_t i00 = pl + (size_t)r * W + c, i0r = pl + (size_t)r * W + cr, id0 = pl + (size_t)rd * W + c;
        const float t00 = tau_map[tau_index(i00, HW, tmp)], t0r = tau_map[tau_index(i0r, HW, tmp)];
        const float td0 = tau_map[tau_index(id0, HW, tmp)];
        const float ubx = ubx_in ? ubx_in[i00] : 0.f, uby = uby_in ? uby_in[i00] : 0.f;
        const float ubx_r = ubx_in ? ubx_in[i0r] : 0.f, uby_d = uby_in ? uby_in[id0] : 0.f;
        const float qx0 = qx[i00], qy0 = qy[i00];
        const float qbx = qbar_of(wbx, ubx, qx0, t00), qby = qbar_of(wby, uby, qy0, t00);
        const float qbx_r = qbar_of(wbx_r, ubx_r, qx[i0r], t0r), qby_d = qbar_of(wby_d, uby_d, qy[id0], td0);
        ubx_out[i00] = qbx; uby_out[i00] = qby;
        xb[i00] = (qbx - qbx_r) + (qby - qby_d);
        double t = 0.0;
        if (fabsf(qx0) >= t00) t += (double)((ubx - 2.f * wbx) * (qx0 > 0.f ? 1.f : (qx0 < 0.f ? -1.f : 0.f)));
        if (fabsf(qy0) >= t00) t += (double)((uby - 2.f * wby) * (qy0 > 0.f ? 1.f : (qy0 < 0.f ? -1.f : 0.f)));
        taubar[idx] += t;
    }
}

__global__ void k_bwd_recompute_v_map(const float* __restrict__ qx, const float* __restrict__ qy, float* __restrict__ v,
                                      const float* __restrict__ tau_map, int tmp, int H, int W, size_t total) {
    const size_t HW = (size_t)H * W;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(idx % W);
        const size_t rowi = idx / W;
        const int r = (int)(rowi % H);
        const size_t pl = (rowi / H) * HW;
        const int cr = c == W - 1 ? 0 : c + 1, rd = r == H - 1 ? 0 : r + 1;
        // the operations and order of k_rows<ROWS_FULL_MAP> (admm_kernels.cu), so a checkpointed re-run matches the forward
        const size_t i00 = pl + (size_t)r * W + c, i0r = pl + (size_t)r * W + cr, id0 = pl + (size_t)rd * W + c;
        const float t00 = tau_map[tau_index(i00, HW, tmp)], t0r = tau_map[tau_index(i0r, HW, tmp)];
        const float td0 = tau_map[tau_index(id0, HW, tmp)];
        auto wf = [](float q, float tau) { return fmaf(-2.f, dual_any(q, tau), q); };
        v[i00] = wf(qx[i00], t00) - wf(qx[i0r], t0r) + wf(qy[i00], t00) - wf(qy[id0], td0);
    }
}

// grad_tau in the map's layout: tmp == P copies the per-element sums; a shared map (tmp == 1, n = H x W) adds the planes
// of each pixel in plane order (iso = 1 accumulates per pixel already: nplanes = 1)
__global__ void k_tau_map_grad(const double* __restrict__ taubar, int nplanes, size_t n, float* __restrict__ grad_tau) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        double s = 0.0;
        for (int p = 0; p < nplanes; ++p) s += taubar[(size_t)p * n + i];
        grad_tau[i] = (float)s;
    }
}

// ------------------------------------------------------------------------------------------ spectral accumulation
// Full-spectrum entry (u, v), v in [0, W/2], from a packed column-transformed spectrum (column 0 = DC + i Nyquist).
template <typename V>
__device__ __forceinline__ V unpack_spec(const V* __restrict__ Z, int u, int v, int H, int Wc) {
    using T = real_t<V>;
    if (v >= 1 && v < Wc) return Z[(size_t)u * Wc + v];
    const V z0 = Z[(size_t)u * Wc];
    const V zm = Z[(size_t)((H - u) % H) * Wc];               // conj applied below
    if (v == 0) return make_cplx(T(0.5) * (z0.x + zm.x), T(0.5) * (z0.y - zm.y));
    return make_cplx(T(0.5) * (z0.y + zm.y), T(-0.5) * (z0.x - zm.x));   // Nyquist column: (z0 - conj(zm)) / (2i)
}

template <typename V>
__global__ void k_bwd_accumulate(const V* __restrict__ ZG, const V* __restrict__ ZV, const V* __restrict__ ZY,
                                 V* __restrict__ Gs, double2* __restrict__ C1, double2* __restrict__ GV,
                                 int P, int H, int W, int Wc, int update_gs) {
    // blockIdx.y splits the planes into gridDim.y groups; group y owns slice y of C1 / GV (single writer per entry,
    // accumulated over the stream-ordered launches of a sweep); k_bwd_finalize adds the slices in a fixed order
    const int Wh = W / 2 + 1;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= H * Wh) return;
    const int u = idx / Wh, v = idx - u * Wh;
    const double inv = 1.0 / ((double)H * (double)W);
    double c1x = 0, c1y = 0, gvx = 0, gvy = 0;
    for (int p = blockIdx.y; p < P; p += gridDim.y) {
        const size_t pl = (size_t)p * H * Wc;
        if (update_gs && v < Wc) {
            const size_t e = pl + (size_t)u * Wc + v;
            const V g = ZG[e];
            V s = Gs[e];
            s.x += g.x; s.y += g.y;
            Gs[e] = s;
        }
        if (ZY || ZV) {
            const V g = unpack_spec(ZG + pl, u, v, H, Wc);
            if (ZY) {
                const V y = unpack_spec(ZY + pl, u, v, H, Wc);
                c1x += (double)g.x * y.x + (double)g.y * y.y;             // conj(g) * y
                c1y += (double)g.x * y.y - (double)g.y * y.x;
            }
            if (ZV) {
                const V w = unpack_spec(ZV + pl, u, v, H, Wc);
                gvx += (double)g.x * w.x + (double)g.y * w.y;
                gvy += (double)g.x * w.y - (double)g.y * w.x;
            }
        }
    }
    const size_t sl = (size_t)blockIdx.y * H * Wh + idx;
    if (ZY) { double2 c = C1[sl]; c.x += c1x * inv; c.y += c1y * inv; C1[sl] = c; }
    if (ZV) { double2 c = GV[sl]; c.x += gvx * inv; c.y += gvy * inv; GV[sl] = c; }
}

// GV(u, v) = sum over planes of the per-plane products kept by the fused column pass
__global__ void k_bwd_reduce_gv(const float2* __restrict__ GVp, const float2* __restrict__ GVn, double2* __restrict__ GV,
                                int P, int H, int W, int Wc) {
    const int Wh = W / 2 + 1;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= H * Wh) return;
    const int u = idx / Wh, v = idx - u * Wh;
    double ax = 0, ay = 0;
    for (int p = blockIdx.y; p < P; p += gridDim.y) {
        const float2 e = (v < Wc) ? GVp[((size_t)p * H + u) * Wc + v] : GVn[(size_t)p * H + u];
        ax += e.x; ay += e.y;
    }
    const size_t sl = (size_t)blockIdx.y * H * Wh + idx;
    double2 c = GV[sl]; c.x += ax; c.y += ay; GV[sl] = c;
}

// rho gradient (spectral part) and the kernel-gradient spectrum S(u, v)
template <typename T>
__global__ void k_bwd_finalize(const double2* __restrict__ C1, const double2* __restrict__ GV, int nsplit, double2* __restrict__ S,
                               double* __restrict__ rho_part, int H, int W, int ks, const double2* __restrict__ G,
                               const double2* __restrict__ twHd, const double2* __restrict__ twWd,
                               const T* __restrict__ rho_p) {
    const int Wh = W / 2 + 1;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    double term = 0.0;
    if (idx < H * Wh) {
        const int u = idx / Wh, v = idx - u * Wh;
        const double rho = (double)rho_p[0];
        const SpecEntry e = spec_entry(u, v, H, W, ks, G, twHd, twWd, rho);
        double2 c1 = make_double2(0.0, 0.0), gv = make_double2(0.0, 0.0);
        for (int y = 0; y < nsplit; ++y) {                              // plane groups, fixed order
            const double2 a = C1[(size_t)y * H * Wh + idx], b = GV[(size_t)y * H * Wh + idx];
            c1.x += a.x; c1.y += a.y; gv.x += b.x; gv.y += b.y;
        }
        const double cw = (v == 0 || ((W & 1) == 0 && v == W / 2)) ? 1.0 : 2.0;
        // sp = sigma * ph
        const double2 sp = make_double2(e.sg.x * e.ph.x - e.sg.y * e.ph.y, e.sg.x * e.ph.y + e.sg.y * e.ph.x);
        const double s2 = e.sg.x * e.sg.x + e.sg.y * e.sg.y;
        const double id = 1.0 / e.den;
        // Re[-C1 sp L / den^2 + GV |sigma|^2 / den^2]
        const double re_c1sp = c1.x * sp.x - c1.y * sp.y;
        term = cw * (-re_c1sp * e.L + gv.x * s2) * id * id;
        if (ks > 0) {
            // t1 = C1 ph / den ; R = Re[(C1 sp / den + GV rho / den) / den] ; S = conj(t1) - 2 R sigma
            const double2 t1 = make_double2((c1.x * e.ph.x - c1.y * e.ph.y) * id, (c1.x * e.ph.y + c1.y * e.ph.x) * id);
            const double R = (re_c1sp * id + gv.x * rho * id) * id;
            S[idx] = make_double2(t1.x - 2.0 * R * e.sg.x, -t1.y - 2.0 * R * e.sg.y);
        }
    }
    __shared__ double red[32];
    for (int o = 16; o > 0; o >>= 1) term += __shfl_down_sync(0xffffffffu, term, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = term;
    __syncthreads();
    if (threadIdx.x < 32) {
        double v = (threadIdx.x < (blockDim.x + 31) / 32) ? red[threadIdx.x] : 0.0;
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (threadIdx.x == 0) rho_part[blockIdx.x] = v;
    }
}

// Tk[u][b] = sum_v c(v) S[u][v] e^{+2 pi i v b / W}
__global__ void k_bwd_kgrad_rows(const double2* __restrict__ S, double2* __restrict__ Tk, int H, int W, int ks,
                                 const double2* __restrict__ twWd) {
    const int Wh = W / 2 + 1;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= H * ks) return;
    const int u = idx / ks, b = idx - u * ks;
    double ax = 0, ay = 0;
    for (int v = 0; v < Wh; ++v) {
        const double cw = (v == 0 || ((W & 1) == 0 && v == W / 2)) ? 1.0 : 2.0;
        const double2 s = S[(size_t)u * Wh + v];
        const double2 w = twWd[(int)(((long long)v * b) % W)];        // e^{-i..}; use the conjugate
        ax += cw * (s.x * w.x + s.y * w.y);
        ay += cw * (s.y * w.x - s.x * w.y);
    }
    Tk[idx] = make_double2(ax, ay);
}

// gk[a][b] = sum_u Re(Tk[u][b] e^{+2 pi i u a / H})
template <typename T>
__global__ void k_bwd_kgrad_cols(const double2* __restrict__ Tk, T* __restrict__ gk, int H, int ks,
                                 const double2* __restrict__ twHd) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= ks * ks) return;
    const int a = idx / ks, b = idx - a * ks;
    double acc = 0;
    for (int u = 0; u < H; ++u) {
        const double2 t = Tk[(size_t)u * ks + b];
        const double2 w = twHd[(int)(((long long)u * a) % H)];
        acc += t.x * w.x + t.y * w.y;                                   // Re(t * conj(w))
    }
    gk[idx] = (T)acc;
}

// fixed-order sum of n doubles by one block of 256 threads (strided partials, then a tree)
__device__ double block_sum_256(const double* __restrict__ v, size_t n, double* red) {
    double s = 0.0;
    for (size_t i = threadIdx.x; i < n; i += 256) s += v[i];
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    const double r = red[0];
    __syncthreads();
    return r;
}

template <typename T>
__global__ void __launch_bounds__(256)
k_bwd_scalars(const double* __restrict__ tau_part, size_t n_tau, const double* __restrict__ rho_part, size_t n_rho,
              const T* __restrict__ lmbd, const T* __restrict__ rho, T* __restrict__ grad_lmbd,
              T* __restrict__ grad_rho) {
    __shared__ double red[256];
    const double taubar = block_sum_256(tau_part, n_tau, red);
    const double rhospec = block_sum_256(rho_part, n_rho, red);
    if (threadIdx.x == 0) {
        const double lam = lmbd[0], r = rho[0];
        if (grad_lmbd) grad_lmbd[0] = (T)(taubar / r);
        if (grad_rho) grad_rho[0] = (T)(rhospec - taubar * lam / (r * r));
    }
}

// threshold maps: the rho gradient at fixed tau is the spectral part alone (the tau term goes back through lmbd / rho in
// the caller's autograd)
__global__ void __launch_bounds__(256)
k_bwd_rho_spectral(const double* __restrict__ rho_part, size_t n_rho, float* __restrict__ grad_rho) {
    __shared__ double red[256];
    const double rhospec = block_sum_256(rho_part, n_rho, red);
    if (threadIdx.x == 0) grad_rho[0] = (float)rhospec;
}

static int ew_grid(size_t total) { return (int)std::min<size_t>((total + 255) / 256, 148 * 16); }

// ---- the same kernels in double, for the float64 backward (f64.cu); launch shapes as in run_backward below
int launch_bwd_spatial(const Geometry& g, const double* vb, const double* ubx_in, const double* uby_in, const double* qx,
                       const double* qy, double* ubx_out, double* uby_out, double* xb, const double* lmbd, const double* rho,
                       double* taubar, cudaStream_t st) {
    ProfScope ps(PROF_OTHER, st);
    const size_t fe = (size_t)g.P * g.H * g.W;
    k_bwd_spatial<<<ew_grid(fe), 256, 0, st>>>(vb, ubx_in, uby_in, qx, qy, ubx_out, uby_out, xb, lmbd, rho, taubar, g.H, g.W, fe);
    ADMM_CUDA_CHECK(cudaGetLastError());
    return 0;
}

int launch_bwd_recompute_v(const Geometry& g, const double* qx, const double* qy, double* v, const double* lmbd,
                           const double* rho, cudaStream_t st) {
    ProfScope ps(PROF_OTHER, st);
    const size_t fe = (size_t)g.P * g.H * g.W;
    k_bwd_recompute_v<<<ew_grid(fe), 256, 0, st>>>(qx, qy, v, lmbd, rho, g.H, g.W, fe);
    ADMM_CUDA_CHECK(cudaGetLastError());
    return 0;
}

int launch_bwd_accumulate(const Geometry& g, int nsplit, const double2* ZG, const double2* ZV, const double2* ZY, double2* Gs,
                          double2* C1, double2* GV, int update_gs, cudaStream_t st) {
    ProfScope ps(PROF_OTHER, st);
    const int HWh = g.H * (g.W / 2 + 1);
    k_bwd_accumulate<<<dim3((HWh + 127) / 128, nsplit), 128, 0, st>>>(ZG, ZV, ZY, Gs, C1, GV, g.P, g.H, g.W, g.Wc, update_gs);
    ADMM_CUDA_CHECK(cudaGetLastError());
    return 0;
}

int launch_bwd_finalize(const Geometry& g, const double2* C1, const double2* GV, int nsplit, double2* S, double* rho_part,
                        int ks, const double2* G, const double2* twHd, const double2* twWd, const double* rho, cudaStream_t st) {
    ProfScope ps(PROF_OTHER, st);
    const int HWh = g.H * (g.W / 2 + 1);
    k_bwd_finalize<<<(HWh + 127) / 128, 128, 0, st>>>(C1, GV, nsplit, S, rho_part, g.H, g.W, ks, G, twHd, twWd, rho);
    ADMM_CUDA_CHECK(cudaGetLastError());
    return 0;
}

int launch_bwd_kgrad(const Geometry& g, const double2* S, double2* Tk, int ks, const double2* twWd, const double2* twHd,
                     double* grad_kern, cudaStream_t st) {
    ProfScope ps(PROF_OTHER, st);
    k_bwd_kgrad_rows<<<(g.H * ks + 127) / 128, 128, 0, st>>>(S, Tk, g.H, g.W, ks, twWd);
    ADMM_CUDA_CHECK(cudaGetLastError());
    k_bwd_kgrad_cols<<<(ks * ks + 63) / 64, 64, 0, st>>>(Tk, grad_kern, g.H, ks, twHd);
    ADMM_CUDA_CHECK(cudaGetLastError());
    return 0;
}

int launch_bwd_scalars(const double* tau_part, size_t n_tau, const double* rho_part, size_t n_rho, const double* lmbd,
                       const double* rho, double* grad_lmbd, double* grad_rho, cudaStream_t st) {
    ProfScope ps(PROF_OTHER, st);
    k_bwd_scalars<<<1, 256, 0, st>>>(tau_part, n_tau, rho_part, n_rho, lmbd, rho, grad_lmbd, grad_rho);
    ADMM_CUDA_CHECK(cudaGetLastError());
    return 0;
}

int run_backward(const Geometry& g, const Workspace& ws, const BwdWorkspace& bw, const float* y, const float* grad_out,
                 const float* kern, int ksize, const float* lmbd, const float* rho, int maxit, const float* saved,
                 const float* saved_nmaps, int ckpt,
                 float* grad_y, float* grad_kern, float* grad_lmbd, float* grad_rho, cudaStream_t st,
                 const float* tau_map = nullptr, int tmp = 0, float* grad_tau = nullptr) {
    // tau_map != NULL (lambda maps, DESIGN section 11): tau per element, grad_tau in the map's layout instead of grad_lmbd,
    // grad_rho at fixed tau.  The iterations re-run on the row kernel the forward ran (power-of-two, else generic); the
    // power-of-two widths take the fused adjoint ROWS_ADJ_MAP, the others the elementwise adjoint kernels.
    const size_t fe = (size_t)g.P * g.H * g.W;
    // ---- saved state.  Slot i holds [q_x, q_y] after forward iteration i + 1 (slots 0 .. maxit-2).  Full mode: every
    // slot is in `saved`.  Checkpointed (K = ckpt >= 2): `saved` keeps the slots with (i + 1) % K == 0; the others of a
    // block [bK, (b+1)K) are re-computed into bw.ck_slots by re-running the forward from the checkpoint in front of the
    // block (or from the start for b = 0) when the sweep enters it: about one extra forward in total.
    const int nslots = maxit - 1;
    int cur_block = -1;
    bool ck_A_valid = false;
    auto is_ckpt = [&](int i) { return ckpt >= 2 && ((i + 1) % ckpt) == 0; };
    auto slot_ptr = [&](int i) -> const float* {
        if (ckpt < 2) return saved + (size_t)i * 2 * fe;
        if (is_ckpt(i)) return saved + (size_t)((i + 1) / ckpt - 1) * 2 * fe;
        return bw.ck_slots + (size_t)(i % ckpt) * 2 * fe;
    };
    // The re-run uses the forward's kernels and layouts (abi.cu, solve_planes).  Large-frame row kernel: v is formed inside
    // its R2C from the checkpoint (r2c_div = 2) with the march's operation order; with both large-frame kernels the
    // spectra between them are tile-major and A is item-major (the layout COLS_INIT of cols_big.cu writes and COLS_ITER reads).
    const bool big_rows = rows_big_supported(g) && !tau_map;
    const int tiled = (big_rows && cols_big_supported(g)) ? 1 : 0;
    auto regen_block = [&](int b) -> int {
        RowArgs rr; std::memset(&rr, 0, sizeof(rr));
        ColArgs cc; std::memset(&cc, 0, sizeof(cc));
        rr.tw = ws.twW; rr.lmbd = lmbd; rr.rho = rho;
        cc.tw = ws.twH; cc.A = bw.ck_A; cc.Bm = ws.Bm; cc.Bq = ws.Bq; cc.Bmt = ws.Bmt; cc.Mul = ws.Mul; cc.Mq = ws.Mq;
        const int m0 = b * ckpt;
        const int end = std::min((b + 1) * ckpt - 1, nslots);          // non-checkpoint slots m0 .. end-1
        const float* qprev = nullptr;
        if (b == 0 || !ck_A_valid) {                                     // A = Mul F(y)   (and x_1 for b = 0)
            rr.real_in = y; rr.spec_out = bw.ck_S1;
            if (int e = launch_rows(ROWS_R2C, g, rr, st)) return e;
            cc.spec_in = bw.ck_S1; cc.spec_out = bw.ck_S0; cc.in_tiled = 0; cc.out_tiled = tiled;
            if (int e = launch_cols(COLS_INIT, g, cc, st)) return e;
            ck_A_valid = true;
        }
        if (b > 0) {                                                     // x_{m0+1} from the checkpoint q_{m0}
            qprev = slot_ptr(m0 - 1);
            if (big_rows) {
                RowArgs rv = rr;
                rv.r2c_div = 2; rv.qx_in = qprev; rv.qy_in = qprev + fe; rv.spec_out = bw.ck_S1; rv.tiled = tiled;
                if (int e = launch_rows(ROWS_R2C, g, rv, st)) return e;
            } else {
                {
                    ProfScope ps(PROF_OTHER, st);
                    if (tau_map)
                        k_bwd_recompute_v_map<<<ew_grid(fe), 256, 0, st>>>(qprev, qprev + fe, bw.ck_v, tau_map, tmp, g.H, g.W, fe);
                    else
                        k_bwd_recompute_v<<<ew_grid(fe), 256, 0, st>>>(qprev, qprev + fe, bw.ck_v, lmbd, rho, g.H, g.W, fe);
                    ADMM_CUDA_CHECK(cudaGetLastError());
                }
                rr.real_in = bw.ck_v; rr.spec_out = bw.ck_S1;
                // the restart's spectrum is formed by the R2C of the row kernel the forward ran (generic rows for a map at
                // widths without a power-of-two kernel)
                const bool gen = tau_map && !rows_pow2_supported(g);
                if (int e = gen ? launch_rows_r2c_generic(g, rr, st) : launch_rows(ROWS_R2C, g, rr, st)) return e;
            }
            cc.spec_in = bw.ck_S1; cc.spec_out = bw.ck_S0; cc.in_tiled = tiled; cc.out_tiled = tiled;
            if (int e = launch_cols(COLS_ITER, g, cc, st)) return e;
        }
        rr.tiled = tiled;
        for (int i = m0; i < end; ++i) {
            float* qn = bw.ck_slots + (size_t)(i - m0) * 2 * fe;
            rr.spec_in = bw.ck_S0; rr.spec_out = bw.ck_S1;
            rr.qx_in = qprev; rr.qy_in = qprev ? qprev + fe : nullptr; rr.qx_out = qn; rr.qy_out = qn + fe;
            RowArgs rf = rr;
            if (tau_map) { rf.cmap = tau_map; rf.tau_map_planes = tmp; }
            if (int e = launch_rows(tau_map ? ROWS_FULL_MAP : ROWS_FULL, g, rf, st)) return e;
            if (i + 1 < end) {                                           // another row pass follows: tile-major output
                cc.spec_in = bw.ck_S1; cc.spec_out = bw.ck_S0; cc.in_tiled = tiled; cc.out_tiled = tiled;
                if (int e = launch_cols(COLS_ITER, g, cc, st)) return e;
            }
            qprev = qn;
        }
        return 0;
    };
    auto need_slot = [&](int i) -> int {
        if (ckpt < 2 || is_ckpt(i) || i / ckpt == cur_block) return 0;
        cur_block = i / ckpt;
        return regen_block(cur_block);
    };
    const int HWh = g.H * (g.W / 2 + 1);
    const bool need_spec = (grad_rho != nullptr) || (grad_kern != nullptr && ksize > 0);
    ADMM_CUDA_CHECK(cudaMemsetAsync(bw.Gs, 0, g.spec_bytes, st));
    ADMM_CUDA_CHECK(cudaMemsetAsync(bw.C1, 0, (size_t)bw.nsplit * HWh * sizeof(double2), st));
    ADMM_CUDA_CHECK(cudaMemsetAsync(bw.GV, 0, (size_t)bw.nsplit * HWh * sizeof(double2), st));
    ADMM_CUDA_CHECK(cudaMemsetAsync(bw.tau_part, 0, bw.n_tau * sizeof(double), st));
    ADMM_CUDA_CHECK(cudaMemsetAsync(bw.rho_part, 0, bw.n_rho * sizeof(double), st));
    const size_t n_taubar = g.iso ? (size_t)g.H * g.W : fe;
    if (tau_map) ADMM_CUDA_CHECK(cudaMemsetAsync(bw.taubar_map, 0, n_taubar * sizeof(double), st));

    RowArgs ra; std::memset(&ra, 0, sizeof(ra));
    ColArgs ca; std::memset(&ca, 0, sizeof(ca));
    ra.tw = ws.twW; ra.lmbd = lmbd; ra.rho = rho;
    ca.tw = ws.twH; ca.Bm = ws.Bm; ca.Bq = ws.Bq; ca.Mul = ws.Mul; ca.Mq = ws.Mq;
    float2* ZY = nullptr;
    if (need_spec) {                                    // F(y), packed, kept in the A slot
        ra.real_in = y; ra.spec_out = ws.S1;
        if (int e = launch_rows(ROWS_R2C, g, ra, st)) return e;
        ca.spec_in = ws.S1; ca.spec_out = ws.A;
        if (int e = launch_cols(COLS_FFT_FWD, g, ca, st)) return e;
        ZY = ws.A;
    }
    const float* ubx = nullptr; const float* uby = nullptr;     // ubar = 0 for the last consumed state
    int pp = 0;
    // power-of-two sizes: one fused row pass per iteration (C2R of vbar, adjoint prox/dual/gradient, R2C of xbar, and
    // the recomputed v_k with its R2C); other sizes / iso: elementwise kernels between plain FFT passes
    const bool fused = rows_pow2_supported(g) && !g.iso;
    const bool iso_fused = (rows_pow2_supported(g) || rows_big_supported(g)) && g.iso;   // divergences formed inside the R2C row pass
    const bool cols_fused = cols_adj_supported(g);
    if (cols_fused) {
        ADMM_CUDA_CHECK(cudaMemsetAsync(bw.ZG, 0, g.spec_bytes, st));          // per-plane GV products live in the ZG slot
        ADMM_CUDA_CHECK(cudaMemsetAsync(bw.GVn, 0, (size_t)g.P * g.H * sizeof(float2), st));
    }
    for (int k = maxit - 1; k >= 0; --k) {
        bool zv_in_place = false;
        if (k == maxit - 1) {
            ra.real_in = grad_out; ra.spec_out = ws.S1;
            if (int e = launch_rows(ROWS_R2C, g, ra, st)) return e;
        } else {
            if (int e = need_slot(k)) return e;
            if (need_spec && k >= 1) { if (int e = need_slot(k - 1)) return e; }
            const float* qx = slot_ptr(k);
            const float* qy = qx + fe;
            float* nx = ws.q[pp][0]; float* ny = ws.q[pp][1];
            if (fused) {
                RowArgs aa = ra;
                aa.spec_in = ws.S0; aa.spec_out = ws.S1;
                aa.qx_in = qx; aa.qy_in = qy;
                aa.ubx_in = ubx; aa.uby_in = uby; aa.ubx_out = nx; aa.uby_out = ny;
                aa.taubar = tau_map ? bw.taubar_map : bw.tau_part;     // map: per element, else per CTA
                if (tau_map) { aa.cmap = tau_map; aa.tau_map_planes = tmp; }
                aa.qvx = nullptr; aa.qvy = nullptr; aa.spec_out2 = nullptr;
                if (need_spec && k >= 1) {
                    aa.qvx = slot_ptr(k - 1); aa.qvy = aa.qvx + fe;
                    aa.spec_out2 = bw.ZV;                       // row spectrum of v_k, column-transformed in place below
                    zv_in_place = true;
                }
                if (int e = launch_rows(tau_map ? ROWS_ADJ_MAP : ROWS_ADJ, g, aa, st)) return e;
            } else {
                if (g.iso) {
                    const float* nm = saved_nmaps + (size_t)k * 2 * g.H * g.W;
                    // power-of-two sizes: xbar = D^T qbar is formed inside the R2C row pass (no xbar field in HBM)
                    if (tau_map) {
                        if (int e = launch_iso_bwd_map(g, bw.vb, ubx, uby, qx, qy, nm, nx, ny, iso_fused ? nullptr : bw.xb,
                                                       tau_map, bw.taubar_map, st)) return e;
                    } else if (int e = launch_iso_bwd(g, bw.vb, ubx, uby, qx, qy, nm, ws.sbmap, nx, ny, iso_fused ? nullptr : bw.xb,
                                                      lmbd, rho, bw.tau_part, st)) return e;
                } else {
                    ProfScope ps(PROF_OTHER, st);
                    if (tau_map)
                        k_bwd_spatial_map<<<ew_grid(fe), 256, 0, st>>>(bw.vb, ubx, uby, qx, qy, nx, ny, bw.xb, tau_map, tmp,
                                                                       bw.taubar_map, g.H, g.W, fe);
                    else
                        k_bwd_spatial<<<ew_grid(fe), 256, 0, st>>>(bw.vb, ubx, uby, qx, qy, nx, ny, bw.xb, lmbd, rho, bw.tau_part,
                                                                   g.H, g.W, fe);
                    ADMM_CUDA_CHECK(cudaGetLastError());
                }
                if (g.iso && iso_fused) {
                    RowArgs rd = ra;
                    rd.r2c_div = 1; rd.cmap = nullptr; rd.qx_in = nx; rd.qy_in = ny; rd.spec_out = ws.S1;
                    if (int e = launch_rows(ROWS_R2C, g, rd, st)) return e;
                } else {
                    ra.real_in = bw.xb; ra.spec_out = ws.S1;
                    if (int e = launch_rows(ROWS_R2C, g, ra, st)) return e;
                }
            }
            ubx = nx; uby = ny; pp ^= 1;
        }
        // row spectrum of v_k -> bw.ZV (v_0 = 0)
        const bool has_v = need_spec && k >= 1;
        if (has_v && !zv_in_place) {
            if (int e = need_slot(k - 1)) return e;
            const float* qx = slot_ptr(k - 1);
            if (g.iso && iso_fused) {
                // v_k = D^T((2 s_k - 1) q_k): coefficient map from the saved norms, divergence inside the R2C row pass
                const float* nm = saved_nmaps + (size_t)(k - 1) * 2 * g.H * g.W;
                if (tau_map) {
                    if (int e = launch_iso_cmap_map(g, nm, ws.sbmap, tau_map, st)) return e;
                } else if (int e = launch_iso_cmap(g, nm, ws.sbmap, lmbd, rho, st)) return e;
                RowArgs rd = ra;
                rd.r2c_div = 1; rd.cmap = ws.sbmap; rd.qx_in = qx; rd.qy_in = qx + fe; rd.spec_out = bw.ZV;
                if (int e = launch_rows(ROWS_R2C, g, rd, st)) return e;
            } else if (g.iso) {
                const float* nm = saved_nmaps + (size_t)(k - 1) * 2 * g.H * g.W;
                if (tau_map) {                                  // coefficient map first: k_iso_div then reads no tau
                    if (int e = launch_iso_cmap_map(g, nm, ws.sbmap, tau_map, st)) return e;
                    if (int e = launch_iso_div(g, qx, qx + fe, nm, ws.sbmap, bw.vb, lmbd, rho, st)) return e;
                } else if (int e = launch_iso_div(g, qx, qx + fe, nm, nullptr, bw.vb, lmbd, rho, st)) return e;
            } else {
                ProfScope ps(PROF_OTHER, st);
                if (tau_map)
                    k_bwd_recompute_v_map<<<ew_grid(fe), 256, 0, st>>>(qx, qx + fe, bw.vb, tau_map, tmp, g.H, g.W, fe);
                else
                    k_bwd_recompute_v<<<ew_grid(fe), 256, 0, st>>>(qx, qx + fe, bw.vb, lmbd, rho, g.H, g.W, fe);
                ADMM_CUDA_CHECK(cudaGetLastError());
            }
            if (!(g.iso && iso_fused)) {
                ra.real_in = bw.vb; ra.spec_out = bw.ZV;
                if (int e = launch_rows(ROWS_R2C, g, ra, st)) return e;
            }
        }
        if (cols_fused) {
            // G = F_col(S1); Gs += G; GVp += conj(G) F_col(ZV)/(HW); S0 = F_col^-1[Bm G]   -- one kernel
            if (int e = launch_cols_adj(g, ws.S1, has_v ? bw.ZV : nullptr, bw.Gs, bw.ZG, bw.GVn, k > 0 ? ws.S0 : nullptr,
                                        ws.Bm, ws.Bq, ws.twH, st)) return e;
        } else {
            ca.spec_in = ws.S1; ca.spec_out = bw.ZG;
            if (int e = launch_cols(COLS_FFT_FWD, g, ca, st)) return e;
            const float2* ZV = nullptr;
            if (has_v) {
                ca.spec_in = bw.ZV; ca.spec_out = bw.ZV;        // tile-private: safe in place
                if (int e = launch_cols(COLS_FFT_FWD, g, ca, st)) return e;
                ZV = bw.ZV;
            }
            {
                ProfScope ps(PROF_OTHER, st);
                const dim3 grid((HWh + 127) / 128, bw.nsplit);
                // C1 = sum_planes conj(sum_k G_k) F(y) is formed once after the sweep from Gs; only GV needs every iteration
                k_bwd_accumulate<float2><<<grid, 128, 0, st>>>(bw.ZG, ZV, nullptr, bw.Gs, bw.C1, bw.GV, g.P, g.H, g.W, g.Wc, 1);
                ADMM_CUDA_CHECK(cudaGetLastError());
            }
            if (k > 0) {                                        // vbar = F^-1[Bm G]
                ca.spec_in = bw.ZG; ca.spec_out = ws.S0;
                if (int e = launch_cols(COLS_BM_INV, g, ca, st)) return e;
            }
        }
        if (k > 0 && !fused) {
            ra.spec_in = ws.S0; ra.real_out = bw.vb; ra.bias = nullptr;
            if (int e = launch_rows(ROWS_C2R, g, ra, st)) return e;
        }
    }
    if (cols_fused && need_spec) {
        ProfScope ps(PROF_OTHER, st);
        const dim3 grid((HWh + 127) / 128, bw.nsplit);
        k_bwd_reduce_gv<<<grid, 128, 0, st>>>(bw.ZG, bw.GVn, bw.GV, g.P, g.H, g.W, g.Wc);
        ADMM_CUDA_CHECK(cudaGetLastError());
    }
    if (need_spec) {                                            // C1 = sum_planes conj(Gs) F(y) / (HW)
        ProfScope ps(PROF_OTHER, st);
        const dim3 grid((HWh + 127) / 128, bw.nsplit);
        k_bwd_accumulate<float2><<<grid, 128, 0, st>>>(bw.Gs, nullptr, ZY, bw.Gs, bw.C1, bw.GV, g.P, g.H, g.W, g.Wc, 0);
        ADMM_CUDA_CHECK(cudaGetLastError());
    }
    if (grad_y) {                                               // ybar = F^-1[conj(sigma ph / den) Gs]
        ca.spec_in = bw.Gs; ca.spec_out = ws.S0;
        if (int e = launch_cols(COLS_CMUL_INV, g, ca, st)) return e;
        ra.spec_in = ws.S0; ra.real_out = grad_y; ra.bias = nullptr;
        if (int e = launch_rows(ROWS_C2R, g, ra, st)) return e;
    }
    if (need_spec) {
        ProfScope ps(PROF_OTHER, st);
        k_bwd_finalize<<<(HWh + 127) / 128, 128, 0, st>>>(bw.C1, bw.GV, bw.nsplit, bw.S, bw.rho_part, g.H, g.W, ksize, ws.kdft,
                                                         ws.twHd, ws.twWd, rho);
        ADMM_CUDA_CHECK(cudaGetLastError());
        if (grad_kern && ksize > 0) {
            k_bwd_kgrad_rows<<<(g.H * ksize + 127) / 128, 128, 0, st>>>(bw.S, bw.Tk, g.H, g.W, ksize, ws.twWd);
            ADMM_CUDA_CHECK(cudaGetLastError());
            k_bwd_kgrad_cols<<<(ksize * ksize + 63) / 64, 64, 0, st>>>(bw.Tk, grad_kern, g.H, ksize, ws.twHd);
            ADMM_CUDA_CHECK(cudaGetLastError());
        }
    }
    if (tau_map) {
        ProfScope ps(PROF_OTHER, st);
        if (grad_tau) {
            // iso = 1 accumulated per pixel; iso = 0 per element, added over the planes here for a shared map
            const int nplanes = (!g.iso && tmp == 1) ? g.P : 1;
            const size_t n = n_taubar / nplanes;
            k_tau_map_grad<<<ew_grid(n), 256, 0, st>>>(bw.taubar_map, nplanes, n, grad_tau);
            ADMM_CUDA_CHECK(cudaGetLastError());
        }
        if (grad_rho) {
            k_bwd_rho_spectral<<<1, 256, 0, st>>>(bw.rho_part, bw.n_rho, grad_rho);
            ADMM_CUDA_CHECK(cudaGetLastError());
        }
        return 0;
    }
    if (grad_lmbd || grad_rho) {
        ProfScope ps(PROF_OTHER, st);
        k_bwd_scalars<<<1, 256, 0, st>>>(bw.tau_part, bw.n_tau, bw.rho_part, bw.n_rho, lmbd, rho, grad_lmbd, grad_rho);
        ADMM_CUDA_CHECK(cudaGetLastError());
    }
    return 0;
}

}  // namespace admm

using namespace admm;

namespace admm {
int make_geometry_pub(int planes, int H, int W, Geometry* g);
int check_kernel_pub(int ksize, int H, int W);
}

extern "C" {

size_t admm_query_workspace_backward(int planes, int H, int W, int ksize, int iso, int maxit) {
    return admm_query_workspace_backward_ex(planes, H, W, ksize, iso, maxit, 0);
}

size_t admm_query_workspace_backward_ex(int planes, int H, int W, int ksize, int iso, int maxit, int ckpt_interval) {
    Geometry g;
    if (make_geometry_pub(planes, H, W, &g)) return 0;
    if (check_kernel_pub(ksize, H, W)) return 0;
    g.iso = iso ? 1 : 0;
    if (ckpt_interval >= 2 && !ckpt_supported(g)) return 0;
    return carve_workspace(g, ksize, maxit, nullptr, nullptr) + backward_extra_bytes(g, ksize, ckpt_interval);
}

int admm_tv_backward(const float* y, const float* grad_out, const float* kern, int ksize,
                     const float* lmbd, const float* rho, int B, int C, int H, int W, int iso, int maxit,
                     const void* saved, size_t saved_bytes, void* workspace, size_t workspace_bytes,
                     float* grad_y, float* grad_kern, float* grad_lmbd, float* grad_rho, void* stream) {
    return admm_tv_backward_ex(y, grad_out, kern, ksize, lmbd, rho, B, C, H, W, iso, maxit, saved, saved_bytes, workspace,
                               workspace_bytes, grad_y, grad_kern, grad_lmbd, grad_rho, stream, 0);
}

int admm_tv_backward_ex(const float* y, const float* grad_out, const float* kern, int ksize,
                        const float* lmbd, const float* rho, int B, int C, int H, int W, int iso, int maxit,
                        const void* saved, size_t saved_bytes, void* workspace, size_t workspace_bytes,
                        float* grad_y, float* grad_kern, float* grad_lmbd, float* grad_rho, void* stream, int ckpt_interval) {
    cudaStream_t st = (cudaStream_t)stream;
    const int ckpt = ckpt_interval >= 2 ? ckpt_interval : 0;
    if (!y || !grad_out || !lmbd || !rho) return fail(ADMM_ERR_INVALID, "NULL tensor pointer");
    if (B < 1 || C < 1) return fail(ADMM_ERR_INVALID, "B and C must be >= 1");
    if (maxit < 0) return fail(ADMM_ERR_INVALID, "maxit must be >= 0");
    if (ksize > 0 && !kern) return fail(ADMM_ERR_INVALID, "kern is NULL but ksize > 0");
    Geometry g;
    if (int e = make_geometry_pub(B * C, H, W, &g)) return e;
    if (int e = check_kernel_pub(ksize, H, W)) return e;
    g.iso = iso ? 1 : 0;
    if (maxit == 0) {                                   // output is constant zero: every gradient vanishes
        if (grad_y) ADMM_CUDA_CHECK(cudaMemsetAsync(grad_y, 0, g.field_bytes, st));
        if (grad_kern && ksize > 0) ADMM_CUDA_CHECK(cudaMemsetAsync(grad_kern, 0, (size_t)ksize * ksize * sizeof(float), st));
        if (grad_lmbd) ADMM_CUDA_CHECK(cudaMemsetAsync(grad_lmbd, 0, sizeof(float), st));
        if (grad_rho) ADMM_CUDA_CHECK(cudaMemsetAsync(grad_rho, 0, sizeof(float), st));
        return 0;
    }
    if (int e = check_generic_f32(g, ckpt != 0)) return e;   // the halo row pass runs only to re-run checkpointed blocks
    if (!workspace || ((uintptr_t)workspace & 255)) return fail(ADMM_ERR_WORKSPACE, "workspace is NULL or not 256-byte aligned");
    Workspace ws; BwdWorkspace bw;
    if (ckpt && !ckpt_supported(g)) return fail(ADMM_ERR_UNSUPPORTED, "checkpointed training is not available for this problem");
    const size_t n1 = carve_workspace(g, ksize, maxit, (char*)workspace, &ws);
    const size_t n2 = carve_backward(g, ksize, ckpt, (char*)workspace + n1, &bw);
    if (workspace_bytes < n1 + n2) return fail(ADMM_ERR_WORKSPACE, "workspace too small (use admm_query_workspace_backward_ex)");
    const size_t kept = ckpt ? (size_t)((maxit - 1) / ckpt) : (size_t)(maxit - 1);
    const size_t need_saved = kept * 2 * g.field_bytes
                            + (iso ? (size_t)(maxit - 1) * 2 * H * W * sizeof(float) : 0);
    if (maxit > 1 && need_saved > 0 && (!saved || saved_bytes < need_saved)) return fail(ADMM_ERR_WORKSPACE, "saved state missing or too small");
    if (int e = launch_twiddles(ws.twW, ws.twWd, W, st)) return e;
    if (int e = launch_twiddles(ws.twH, ws.twHd, H, st)) return e;
    if (int e = launch_tables(g, ws, kern, ksize, rho, st)) return e;
    if (cols_big_supported(g))
        if (int e = launch_bm_tiled(g, ws.Bm, ws.Bmt, st)) return e;
    const float* nmaps = (const float*)saved + (size_t)(maxit - 1) * 2 * ((size_t)g.P * H * W);
    return run_backward(g, ws, bw, y, grad_out, kern, ksize, lmbd, rho, maxit, (const float*)saved, nmaps, ckpt,
                        grad_y, grad_kern, grad_lmbd, grad_rho, st);
}

// ---- threshold maps (lambda maps, DESIGN section 11)
size_t admm_query_workspace_backward_map(int planes, int H, int W, int ksize, int iso, int maxit, int ckpt_interval,
                                         int tau_map_planes) {
    Geometry g;
    if (make_geometry_pub(planes, H, W, &g)) return 0;
    if (check_kernel_pub(ksize, H, W)) return 0;
    if (tau_map_planes != 1 && tau_map_planes != planes) return 0;
    if (iso && tau_map_planes != 1) return 0;
    g.iso = iso ? 1 : 0;
    const int ckpt = ckpt_interval >= 2 ? ckpt_interval : 0;
    if (ckpt && !ckpt_supported(g)) return 0;
    return carve_workspace(g, ksize, maxit, nullptr, nullptr) + carve_backward(g, ksize, ckpt, nullptr, nullptr, tau_map_planes);
}

int admm_tv_backward_map(const float* y, const float* grad_out, const float* kern, int ksize,
                         const float* tau_map, int tau_map_planes, const float* rho,
                         int B, int C, int H, int W, int iso, int maxit,
                         const void* saved, size_t saved_bytes, void* workspace, size_t workspace_bytes,
                         float* grad_y, float* grad_kern, float* grad_tau, float* grad_rho, void* stream, int ckpt_interval) {
    cudaStream_t st = (cudaStream_t)stream;
    const int ckpt = ckpt_interval >= 2 ? ckpt_interval : 0;
    if (!y || !grad_out || !rho) return fail(ADMM_ERR_INVALID, "NULL tensor pointer");
    if (B < 1 || C < 1) return fail(ADMM_ERR_INVALID, "B and C must be >= 1");
    if (maxit < 0) return fail(ADMM_ERR_INVALID, "maxit must be >= 0");
    if (ksize > 0 && !kern) return fail(ADMM_ERR_INVALID, "kern is NULL but ksize > 0");
    if (int e = check_tau_map(tau_map, tau_map_planes, B * C, iso)) return e;
    Geometry g;
    if (int e = make_geometry_pub(B * C, H, W, &g)) return e;
    if (int e = check_kernel_pub(ksize, H, W)) return e;
    g.iso = iso ? 1 : 0;
    const size_t map_bytes = (size_t)tau_map_planes * H * W * sizeof(float);
    if (maxit == 0) {
        if (grad_y) ADMM_CUDA_CHECK(cudaMemsetAsync(grad_y, 0, g.field_bytes, st));
        if (grad_kern && ksize > 0) ADMM_CUDA_CHECK(cudaMemsetAsync(grad_kern, 0, (size_t)ksize * ksize * sizeof(float), st));
        if (grad_tau) ADMM_CUDA_CHECK(cudaMemsetAsync(grad_tau, 0, map_bytes, st));
        if (grad_rho) ADMM_CUDA_CHECK(cudaMemsetAsync(grad_rho, 0, sizeof(float), st));
        return 0;
    }
    if (int e = check_generic_f32_map(g, ckpt != 0)) return e;
    if (!workspace || ((uintptr_t)workspace & 255)) return fail(ADMM_ERR_WORKSPACE, "workspace is NULL or not 256-byte aligned");
    if (ckpt && !ckpt_supported(g)) return fail(ADMM_ERR_UNSUPPORTED, "checkpointed training is not available for this problem");
    Workspace ws; BwdWorkspace bw;
    const size_t n1 = carve_workspace(g, ksize, maxit, (char*)workspace, &ws);
    const size_t n2 = carve_backward(g, ksize, ckpt, (char*)workspace + n1, &bw, tau_map_planes);
    if (workspace_bytes < n1 + n2) return fail(ADMM_ERR_WORKSPACE, "workspace too small (use admm_query_workspace_backward_map)");
    const size_t kept = ckpt ? (size_t)((maxit - 1) / ckpt) : (size_t)(maxit - 1);
    const size_t need_saved = kept * 2 * g.field_bytes + (iso ? (size_t)(maxit - 1) * 2 * H * W * sizeof(float) : 0);
    if (maxit > 1 && need_saved > 0 && (!saved || saved_bytes < need_saved)) return fail(ADMM_ERR_WORKSPACE, "saved state missing or too small");
    if (int e = launch_twiddles(ws.twW, ws.twWd, W, st)) return e;
    if (int e = launch_twiddles(ws.twH, ws.twHd, H, st)) return e;
    if (int e = launch_tables(g, ws, kern, ksize, rho, st)) return e;
    if (cols_big_supported(g))
        if (int e = launch_bm_tiled(g, ws.Bm, ws.Bmt, st)) return e;
    const float* nmaps = (const float*)saved + (size_t)(maxit - 1) * 2 * ((size_t)g.P * H * W);
    return run_backward(g, ws, bw, y, grad_out, kern, ksize, nullptr, rho, maxit, (const float*)saved, nmaps, ckpt,
                        grad_y, grad_kern, nullptr, grad_rho, st, tau_map, tau_map_planes, grad_tau);
}

}  // extern "C"
