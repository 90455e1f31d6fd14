// resid.cu -- convergence residuals of the ADMM splitting Dx - z = 0 (Boyd et al. 2011, section 3.3), per plane, from two
// consecutive states of the reduced iteration (DESIGN section 10).  With q_k the pre-threshold state after iteration k:
//     u_k = dual(q_k),  z_k = q_k - u_k,  Dx_k = q_k - u_{k-1}
//     r_k = ||u_k - u_{k-1}||            s_k = rho ||D^T(z_k - z_{k-1})||
//     eps_pri  = sqrt(2HW) atol + rtol max(||Dx_k||, ||z_k||)      eps_dual = sqrt(HW) atol + rtol rho ||D^T u_k||
// k_resid forms every term in the element type with the solver's own dual_of / iso_scale and accumulates the five sums of
// squares in double; each CTA writes its five partial sums to its own slot [plane][block].  k_resid_finalize adds the
// slots of a plane in a fixed order, writes (r, s, eps_pri, eps_dual) and one int "every plane converged".  No atomics:
// the residuals are bit-identical from run to run.
#include <algorithm>
#include <cmath>

#include "common.cuh"

namespace admm {

constexpr int kResidThreads = 256;
constexpr int kResidTerms = 5;          // sums of (u_k - u_{k-1})^2, (D^T dz)^2, (Dx_k)^2, z_k^2, (D^T u_k)^2
constexpr int kResidFinalThreads = 1024;

template <typename T>
struct ResidIn {
    const T* qxp; const T* qyp;         // q_{k-1}; NULL at k = 1 (q_0 = 0)
    const T* qxk; const T* qyk;         // q_k
    const T* np;  const T* nk;          // iso = 1: pixel-norm maps (2 x H x W) of k-1 (NULL at k = 1) and k; iso = 0: NULL
};

__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }      // no contraction into the
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }   // z = q - u that follows

// u = dual(q): clamp / sign(q) tau (dual_of), or (1 - s) q with s from the pixel norm for the block threshold (iso.cu)
template <bool NEG, bool ISO, typename T>
__device__ __forceinline__ T resid_dual(T q, const T* nmap, size_t i, T tau) {
    if (ISO) return nmap ? mul_rn(T(1) - iso_scale(__ldg(nmap + i), tau), q) : T(0);
    return dual_of<NEG>(q, tau);
}

// rows blockIdx.x, blockIdx.x + gridDim.x, ... of one plane; the threads of a CTA stride along the row (H * W < 2^30)
template <bool NEG, bool ISO, typename T>
__device__ __forceinline__ void resid_span(const ResidIn<T>& a, size_t pl, int H, int W, T tau, double* acc) {
    const int HW = H * W;
    for (int r = blockIdx.x; r < H; r += gridDim.x)
    for (int c = threadIdx.x; c < W; c += blockDim.x) {
        const int i = r * W + c;
        // [field][0 = this pixel, 1 = right (x field) / lower (y field) neighbour, circular]
        const int at[2][2] = {{i, r * W + (c == W - 1 ? 0 : c + 1)}, {i, (r == H - 1 ? 0 : r + 1) * W + c}};
        T qk[2][2], uk[2][2], up[2][2], dz[2][2];
#pragma unroll
        for (int f = 0; f < 2; ++f) {
            const T* QK = f ? a.qyk : a.qxk;
            const T* QP = f ? a.qyp : a.qxp;
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int m = at[f][j];
                const T q = __ldg(QK + pl + m);
                const T p = QP ? __ldg(QP + pl + m) : T(0);
                qk[f][j] = q;
                uk[f][j] = resid_dual<NEG, ISO>(q, a.nk, f * HW + m, tau);
                up[f][j] = resid_dual<NEG, ISO>(p, a.np, f * HW + m, tau);
                dz[f][j] = (q - uk[f][j]) - (p - up[f][j]);
            }
        }
#pragma unroll
        for (int f = 0; f < 2; ++f) {
            const T du = uk[f][0] - up[f][0];
            const T dx = qk[f][0] - up[f][0];
            const T z = qk[f][0] - uk[f][0];
            acc[0] += (double)du * (double)du;
            acc[2] += (double)dx * (double)dx;
            acc[3] += (double)z * (double)z;
        }
        const T dtz = (dz[0][0] - dz[0][1]) + (dz[1][0] - dz[1][1]);
        const T dtu = (uk[0][0] - uk[0][1]) + (uk[1][0] - uk[1][1]);
        acc[1] += (double)dtz * (double)dtz;
        acc[4] += (double)dtu * (double)dtu;
    }
}

// grid (blocks per plane, planes); part[(plane * gridDim.x + block) * 5 + term]
template <typename T>
__global__ void __launch_bounds__(kResidThreads)
k_resid(ResidIn<T> a, const T* __restrict__ lmbd, const T* __restrict__ rho, double* __restrict__ part, int H, int W) {
    const T tau = lmbd[0] / rho[0];
    const size_t pl = (size_t)blockIdx.y * H * W;
    double acc[kResidTerms] = {0.0, 0.0, 0.0, 0.0, 0.0};
    if (a.nk) resid_span<false, true>(a, pl, H, W, tau, acc);
    else if (tau < T(0)) resid_span<true, false>(a, pl, H, W, tau, acc);        // warp-uniform, as in the march
    else resid_span<false, false>(a, pl, H, W, tau, acc);
    __shared__ double red[kResidThreads / 32][kResidTerms];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int t = 0; t < kResidTerms; ++t) {
        double v = acc[t];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) red[warp][t] = v;
    }
    __syncthreads();
    if (threadIdx.x < kResidTerms) {
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < kResidThreads / 32; ++w) v += red[w][threadIdx.x];
        part[((size_t)blockIdx.y * gridDim.x + blockIdx.x) * kResidTerms + threadIdx.x] = v;
    }
}

// one CTA; warp w sums the slots of planes w, w + 32, ... (lane l: slots l, l + 32, ..., then a fixed shuffle tree)
template <typename T>
__global__ void __launch_bounds__(kResidFinalThreads)
k_resid_finalize(const double* __restrict__ part, int nblk, int P, const T* __restrict__ rho, double rtol, double atol,
                 double sq_pri, double sq_dual, float* __restrict__ out, int* __restrict__ flag) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const double rh = (double)rho[0];
    int ok = 1;
    for (int p = warp; p < P; p += nw) {
        double s[kResidTerms] = {0.0, 0.0, 0.0, 0.0, 0.0};
        const double* src = part + (size_t)p * nblk * kResidTerms;
#pragma unroll 4
        for (int b = lane; b < nblk; b += 32)
#pragma unroll
            for (int t = 0; t < kResidTerms; ++t) s[t] += src[(size_t)b * kResidTerms + t];
#pragma unroll
        for (int t = 0; t < kResidTerms; ++t)
            for (int o = 16; o > 0; o >>= 1) s[t] += __shfl_xor_sync(0xffffffffu, s[t], o);
        if (lane == 0) {
            const float r = (float)sqrt(s[0]);
            const float sd = (float)(rh * sqrt(s[1]));
            const float ep = (float)(sq_pri * atol + rtol * fmax(sqrt(s[2]), sqrt(s[3])));
            const float ed = (float)(sq_dual * atol + rtol * rh * sqrt(s[4]));
            float4* o = reinterpret_cast<float4*>(out) + p;
            *o = make_float4(r, sd, ep, ed);
            ok &= (r <= ep && sd <= ed) ? 1 : 0;         // the stored fp32 values decide: a history reproduces the stop
        }
    }
    ok = __syncthreads_and(ok);
    if (threadIdx.x == 0) *flag = ok;
}

// CTAs per plane (each takes whole rows): about 2048 CTAs in all, at least 2048 pixels per CTA (8 per thread), at most
// 1024 per plane and one row per CTA
static int resid_blocks(const Geometry& g) {
    const long long HW = (long long)g.H * g.W;
    const long long by_size = std::max(1LL, (HW + 2047) / 2048);
    const long long by_grid = std::max(1LL, (2048LL + g.P - 1) / g.P);
    return (int)std::min(std::min(std::min(by_size, by_grid), 1024LL), (long long)g.H);
}

int resid_checks(int maxit, int every) { return (maxit > 1 && every > 0) ? (maxit - 1) / every : 0; }

static inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

size_t carve_resid(const Geometry& g, int maxit, int every, int early_stop, char* base, ResidBufs* rb) {
    size_t off = 0;
    auto take = [&](size_t bytes) {
        char* p = base ? base + off : nullptr;
        off += align256(bytes);
        return p;
    };
    ResidBufs b;
    b.nblk = resid_blocks(g);
    b.hist = (float*)take((size_t)resid_checks(maxit, every) * g.P * 4 * sizeof(float));
    b.part = (double*)take((size_t)g.P * b.nblk * kResidTerms * sizeof(double));
    b.dflag = (int*)take(sizeof(int));
    b.spare = early_stop ? (float2*)take(g.spec_bytes) : nullptr;
    if (rb) *rb = b;
    return off;
}

int launch_resid(const Geometry& g, const float* qxp, const float* qyp, const float* qxk, const float* qyk,
                 const float* np, const float* nk, const float* lmbd, const float* rho, const ResidBufs& rb, float* out,
                 float rtol, float atol, cudaStream_t st) {
    if (g.P > 65535) return fail(4, "residuals: B*C must be <= 65535");
    ResidIn<float> a;
    a.qxp = qxp; a.qyp = qyp; a.qxk = qxk; a.qyk = qyk; a.np = np; a.nk = nk;
    const double HW = (double)g.H * g.W;
    {
        ProfScope ps(PROF_OTHER, st);
        k_resid<float><<<dim3((unsigned)rb.nblk, (unsigned)g.P), kResidThreads, 0, st>>>(a, lmbd, rho, rb.part, g.H, g.W);
        ADMM_CUDA_CHECK(cudaGetLastError());
    }
    ProfScope ps(PROF_OTHER, st);
    k_resid_finalize<float><<<1, kResidFinalThreads, 0, st>>>(rb.part, rb.nblk, g.P, rho, (double)rtol, (double)atol,
                                                             std::sqrt(2.0 * HW), std::sqrt(HW), out, rb.dflag);
    ADMM_CUDA_CHECK(cudaGetLastError());
    return 0;
}

}  // namespace admm
