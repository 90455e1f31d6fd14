// f64.cu -- the float64 solve: admm_*_f64 of include/admm_b200.h.
//
// The reference computes in xin.dtype (deconv.py:50-67), float64 included.  This file runs that case on the generic engine
// only -- the arbitrary-length Stockham FFT and the generic row / column kernels of admm_kernels.cu, the iso kernels of
// iso.cu and the backward kernels of backward.cu, all instantiated for double.  It is the generic subset of the float32
// solver (abi.cu: solve_planes, backward.cu: run_backward) with double elements: no chunks, cooperative or cluster kernels,
// PDL schedule choices, tiled layouts, shared spectrum or checkpointing, and the float32 solver never branches on it.
//
// Forward, maxit = N >= 1:
//     rows R2C : y -> S1;  cols INIT: S1 -> A, S0
//     N-1 times: rows FULL (iso: C2R -> prox -> div -> R2C): S0 -> S1;  cols ITER: S1 -> S0
//     rows C2R : S0 -> out
// Saved state (same layout as the float32 path, double elements): [slot][q_x, q_y][all planes] for slots 0 .. N-2, then
// for iso = 1 the N-1 pairs of H x W pixel-norm maps.
#include <algorithm>
#include <cstring>

#include "../../include/admm_b200.h"
#include "common.cuh"

namespace admm {

int make_geometry_pub(int planes, int H, int W, Geometry* g);
int check_kernel_pub(int ksize, int H, int W);

namespace {

struct WorkspaceF64 {
    double2* twWd; double2* twHd;      // e^{-2 pi i n/N}
    double2* kdft;                     // k x (W/2+1) row-DFT of the PSF
    double*  Bm; double* Bq;           // H*Wc real (column 0 = Bp), H real
    double2* Mul; double2* Mq;         // H*Wc cplx (column 0 = Mp), H cplx
    double2* S0; double2* S1; double2* A;
    double*  q[2][2];                  // ping-pong pre-clamp state q_x, q_y (inference; backward: ubar)
    double*  xreal; double* vreal;     // iso = 1: x_k and v_{k+1} as real fields
    double*  nmap[2];                  // iso = 1: ping-pong pixel norms, 2 x H x W each
    double*  sbmap;                    // iso = 1: coefficient map 2s-1 of the divergence, 2 x H x W
};

// the generic part of the float32 BwdWorkspace (backward.cu)
struct BwdWorkspaceF64 {
    double2* ZG; double2* ZV; double2* Gs;   // packed spectra, per plane
    double*  vb; double* xb;                 // real fields
    double2* C1; double2* GV;                // nsplit x H x (W/2+1) partial sums (one slice per plane group, fixed order)
    double2* S;                              // H x (W/2+1)
    double2* Tk;                             // H x ksize
    double*  tau_part;                       // per-CTA partial sums of the tau gradient
    double*  rho_part;                       // per-CTA partial sums of the spectral rho gradient
    int nsplit; size_t n_tau, n_rho;
};

inline size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }

struct Carver {
    char* base; size_t off = 0;
    template <class P> P* take(size_t bytes) {
        char* p = base ? base + off : nullptr;
        off += align_up(bytes);
        return (P*)p;
    }
};

int make_geometry_f64(int planes, int H, int W, int iso, Geometry* g) {
    if (int e = make_geometry_pub(planes, H, W, g)) return e;
    g->iso = iso ? 1 : 0;
    g->field_bytes = (size_t)planes * H * W * sizeof(double);
    g->spec_bytes = (size_t)planes * H * g->Wc * sizeof(double2);
    return 0;
}

size_t carve_f64(const Geometry& g, int ksize, char* base, WorkspaceF64* out) {
    Carver c{base};
    WorkspaceF64 w;
    std::memset(&w, 0, sizeof(w));
    const size_t HWc = (size_t)g.H * g.Wc;
    w.twWd = c.take<double2>((size_t)g.W * sizeof(double2));
    w.twHd = c.take<double2>((size_t)g.H * sizeof(double2));
    w.kdft = c.take<double2>((size_t)(ksize > 0 ? ksize : 1) * (g.W / 2 + 1) * sizeof(double2));
    w.Bm   = c.take<double>(HWc * sizeof(double));
    w.Bq   = c.take<double>((size_t)g.H * sizeof(double));
    w.Mul  = c.take<double2>(HWc * sizeof(double2));
    w.Mq   = c.take<double2>((size_t)g.H * sizeof(double2));
    w.S0 = c.take<double2>(g.spec_bytes);
    w.S1 = c.take<double2>(g.spec_bytes);
    w.A  = c.take<double2>(g.spec_bytes);
    for (int i = 0; i < 2; ++i)
        for (int f = 0; f < 2; ++f) w.q[i][f] = c.take<double>(g.field_bytes);
    if (g.iso) {
        const size_t map_bytes = (size_t)2 * g.H * g.W * sizeof(double);
        w.xreal = c.take<double>(g.field_bytes);
        w.vreal = c.take<double>(g.field_bytes);
        w.nmap[0] = c.take<double>(map_bytes);
        w.nmap[1] = c.take<double>(map_bytes);
        w.sbmap = c.take<double>(map_bytes);
    }
    if (out) *out = w;
    return c.off;
}

size_t carve_backward_f64(const Geometry& g, int ksize, char* base, BwdWorkspaceF64* out) {
    Carver c{base};
    BwdWorkspaceF64 w;
    const size_t HWh = (size_t)g.H * (g.W / 2 + 1);
    w.ZG = c.take<double2>(g.spec_bytes);
    w.ZV = c.take<double2>(g.spec_bytes);
    w.Gs = c.take<double2>(g.spec_bytes);
    w.vb = c.take<double>(g.field_bytes);
    w.xb = c.take<double>(g.field_bytes);
    // plane groups of the C1 / GV sums: at most 64, capped at 256 MB of partials (as in backward.cu)
    w.nsplit = (int)std::max<size_t>(1, std::min<size_t>(std::min(g.P, 64), ((size_t)256 << 20) / (2 * HWh * sizeof(double2))));
    w.C1 = c.take<double2>(w.nsplit * HWh * sizeof(double2));
    w.GV = c.take<double2>(w.nsplit * HWh * sizeof(double2));
    w.S  = c.take<double2>(HWh * sizeof(double2));
    w.Tk = c.take<double2>((size_t)g.H * (ksize > 0 ? ksize : 1) * sizeof(double2));
    // slot = blockIdx.x of the kernel that produces the partial: generic spatial kernel (<= 148 * 16), iso kernel (H*W/32)
    w.n_tau = std::max<size_t>(148 * 16, ((size_t)g.H * g.W + 31) / 32);
    w.tau_part = c.take<double>(w.n_tau * sizeof(double));
    w.n_rho = (HWh + 127) / 128;
    w.rho_part = c.take<double>(w.n_rho * sizeof(double));
    if (out) *out = w;
    return c.off;
}

// saved-state bytes the forward writes and the backward reads (without the 256-byte pad of the query)
size_t saved_bytes_f64(const Geometry& g, int maxit) {
    const size_t slots = maxit > 1 ? (size_t)(maxit - 1) : 0;
    return slots * 2 * g.field_bytes + (g.iso ? slots * 2 * (size_t)g.H * g.W * sizeof(double) : 0);
}

int setup_tables(const Geometry& g, const WorkspaceF64& ws, const double* kern, int ksize, const double* rho, cudaStream_t st) {
    if (int e = launch_twiddles_f64(ws.twWd, g.W, st)) return e;
    if (int e = launch_twiddles_f64(ws.twHd, g.H, st)) return e;
    return launch_tables_f64(g, ws.twWd, ws.twHd, ws.kdft, ws.Bm, ws.Bq, ws.Mul, ws.Mq, kern, ksize, rho, st);
}

int forward_f64(const Geometry& g, const WorkspaceF64& ws, const double* y, double* out, const double* lmbd,
                const double* rho, int maxit, double* saved, cudaStream_t st) {
    const size_t fe = (size_t)g.P * g.H * g.W;
    const size_t map = (size_t)2 * g.H * g.W;
    const int slots = maxit - 1;
    RowArgsT<double> ra; std::memset(&ra, 0, sizeof(ra));
    ColArgsT<double> ca; std::memset(&ca, 0, sizeof(ca));
    ra.tw = ws.twWd; ra.lmbd = lmbd; ra.rho = rho;
    ca.tw = ws.twHd; ca.A = ws.A; ca.Bm = ws.Bm; ca.Bq = ws.Bq; ca.Mul = ws.Mul; ca.Mq = ws.Mq;
    ra.real_in = y; ra.spec_out = ws.S1;
    if (int e = launch_rows(ROWS_R2C, g, ra, st)) return e;
    ca.spec_in = ws.S1; ca.spec_out = ws.S0;
    if (int e = launch_cols(COLS_INIT, g, ca, st)) return e;
    const double* qx_prev = nullptr; const double* qy_prev = nullptr;
    for (int it = 1; it < maxit; ++it) {
        double* qx_new = saved ? saved + (size_t)(it - 1) * 2 * fe : ws.q[it & 1][0];
        double* qy_new = saved ? qx_new + fe : ws.q[it & 1][1];
        if (g.iso) {
            // the block threshold couples all planes of a pixel: C2R, per-pixel prox over the planes, divergence, R2C
            const double* n_prev = (it == 1) ? nullptr : (saved ? saved + (size_t)slots * 2 * fe + (size_t)(it - 2) * map
                                                                : ws.nmap[(it - 1) & 1]);
            double* n_new = saved ? saved + (size_t)slots * 2 * fe + (size_t)(it - 1) * map : ws.nmap[it & 1];
            ra.spec_in = ws.S0; ra.real_out = ws.xreal;
            if (int e = launch_rows(ROWS_C2R, g, ra, st)) return e;
            if (int e = launch_iso_prox(g, ws.xreal, qx_prev, qy_prev, n_prev, qx_new, qy_new, n_new, ws.sbmap, lmbd, rho, st))
                return e;
            if (int e = launch_iso_div(g, qx_new, qy_new, n_new, ws.sbmap, ws.vreal, lmbd, rho, st)) return e;
            ra.real_in = ws.vreal; ra.spec_out = ws.S1;
            if (int e = launch_rows(ROWS_R2C, g, ra, st)) return e;
        } else {
            ra.spec_in = ws.S0; ra.spec_out = ws.S1;
            ra.qx_in = qx_prev; ra.qy_in = qy_prev; ra.qx_out = qx_new; ra.qy_out = qy_new;
            if (int e = launch_rows(ROWS_FULL, g, ra, st)) return e;
        }
        ca.spec_in = ws.S1; ca.spec_out = ws.S0;
        if (int e = launch_cols(COLS_ITER, g, ca, st)) return e;
        qx_prev = qx_new; qy_prev = qy_new;
    }
    ra.spec_in = ws.S0; ra.real_out = out;
    return launch_rows(ROWS_C2R, g, ra, st);
}

// The generic branch of run_backward (backward.cu) in double; see the derivation there.
int backward_f64(const Geometry& g, const WorkspaceF64& ws, const BwdWorkspaceF64& bw, const double* y,
                 const double* grad_out, int ksize, const double* lmbd, const double* rho, int maxit, const double* saved,
                 double* grad_y, double* grad_kern, double* grad_lmbd, double* grad_rho, cudaStream_t st) {
    const size_t fe = (size_t)g.P * g.H * g.W;
    const size_t map = (size_t)2 * g.H * g.W;
    const double* nmaps = saved ? saved + (size_t)(maxit - 1) * 2 * fe : nullptr;
    const size_t HWh = (size_t)g.H * (g.W / 2 + 1);
    const bool need_spec = (grad_rho != nullptr) || (grad_kern != nullptr && ksize > 0);
    ADMM_CUDA_CHECK(cudaMemsetAsync(bw.Gs, 0, g.spec_bytes, st));
    ADMM_CUDA_CHECK(cudaMemsetAsync(bw.C1, 0, (size_t)bw.nsplit * HWh * sizeof(double2), st));
    ADMM_CUDA_CHECK(cudaMemsetAsync(bw.GV, 0, (size_t)bw.nsplit * HWh * sizeof(double2), st));
    ADMM_CUDA_CHECK(cudaMemsetAsync(bw.tau_part, 0, bw.n_tau * sizeof(double), st));
    ADMM_CUDA_CHECK(cudaMemsetAsync(bw.rho_part, 0, bw.n_rho * sizeof(double), st));

    RowArgsT<double> ra; std::memset(&ra, 0, sizeof(ra));
    ColArgsT<double> ca; std::memset(&ca, 0, sizeof(ca));
    ra.tw = ws.twWd; ra.lmbd = lmbd; ra.rho = rho;
    ca.tw = ws.twHd; ca.Bm = ws.Bm; ca.Bq = ws.Bq; ca.Mul = ws.Mul; ca.Mq = ws.Mq;
    double2* ZY = nullptr;
    if (need_spec) {                                    // F(y), packed, kept in the A slot
        ra.real_in = y; ra.spec_out = ws.S1;
        if (int e = launch_rows(ROWS_R2C, g, ra, st)) return e;
        ca.spec_in = ws.S1; ca.spec_out = ws.A;
        if (int e = launch_cols(COLS_FFT_FWD, g, ca, st)) return e;
        ZY = ws.A;
    }
    const double* ubx = nullptr; const double* uby = nullptr;   // ubar = 0 for the last consumed state
    int pp = 0;
    for (int k = maxit - 1; k >= 0; --k) {
        if (k == maxit - 1) {
            ra.real_in = grad_out; ra.spec_out = ws.S1;
            if (int e = launch_rows(ROWS_R2C, g, ra, st)) return e;
        } else {
            const double* qx = saved + (size_t)k * 2 * fe;
            const double* qy = qx + fe;
            double* nx = ws.q[pp][0]; double* ny = ws.q[pp][1];
            if (g.iso) {
                if (int e = launch_iso_bwd(g, bw.vb, ubx, uby, qx, qy, nmaps + (size_t)k * map, ws.sbmap, nx, ny, bw.xb,
                                           lmbd, rho, bw.tau_part, st)) return e;
            } else {
                if (int e = launch_bwd_spatial(g, bw.vb, ubx, uby, qx, qy, nx, ny, bw.xb, lmbd, rho, bw.tau_part, st)) return e;
            }
            ra.real_in = bw.xb; ra.spec_out = ws.S1;
            if (int e = launch_rows(ROWS_R2C, g, ra, st)) return e;
            ubx = nx; uby = ny; pp ^= 1;
        }
        // row spectrum of v_k -> bw.ZV (v_0 = 0), recomputed from the saved q_k
        const bool has_v = need_spec && k >= 1;
        if (has_v) {
            const double* qx = saved + (size_t)(k - 1) * 2 * fe;
            if (g.iso) {
                if (int e = launch_iso_div(g, qx, qx + fe, nmaps + (size_t)(k - 1) * map, nullptr, bw.vb, lmbd, rho, st)) return e;
            } else {
                if (int e = launch_bwd_recompute_v(g, qx, qx + fe, bw.vb, lmbd, rho, st)) return e;
            }
            ra.real_in = bw.vb; ra.spec_out = bw.ZV;
            if (int e = launch_rows(ROWS_R2C, g, ra, st)) return e;
        }
        ca.spec_in = ws.S1; ca.spec_out = bw.ZG;
        if (int e = launch_cols(COLS_FFT_FWD, g, ca, st)) return e;
        if (has_v) {
            ca.spec_in = bw.ZV; ca.spec_out = bw.ZV;            // tile-private: safe in place
            if (int e = launch_cols(COLS_FFT_FWD, g, ca, st)) return e;
        }
        if (int e = launch_bwd_accumulate(g, bw.nsplit, bw.ZG, has_v ? bw.ZV : nullptr, nullptr, bw.Gs, bw.C1, bw.GV, 1, st))
            return e;
        if (k > 0) {                                            // vbar = F^-1[Bm G]
            ca.spec_in = bw.ZG; ca.spec_out = ws.S0;
            if (int e = launch_cols(COLS_BM_INV, g, ca, st)) return e;
            ra.spec_in = ws.S0; ra.real_out = bw.vb;
            if (int e = launch_rows(ROWS_C2R, g, ra, st)) return e;
        }
    }
    if (need_spec)                                              // C1 = sum_planes conj(Gs) F(y) / (HW)
        if (int e = launch_bwd_accumulate(g, bw.nsplit, bw.Gs, nullptr, ZY, bw.Gs, bw.C1, bw.GV, 0, st)) return e;
    if (grad_y) {                                               // ybar = F^-1[conj(sigma ph / den) Gs]
        ca.spec_in = bw.Gs; ca.spec_out = ws.S0;
        if (int e = launch_cols(COLS_CMUL_INV, g, ca, st)) return e;
        ra.spec_in = ws.S0; ra.real_out = grad_y;
        if (int e = launch_rows(ROWS_C2R, g, ra, st)) return e;
    }
    if (need_spec) {
        if (int e = launch_bwd_finalize(g, bw.C1, bw.GV, bw.nsplit, bw.S, bw.rho_part, ksize, ws.kdft, ws.twHd, ws.twWd, rho, st))
            return e;
        if (grad_kern && ksize > 0)
            if (int e = launch_bwd_kgrad(g, bw.S, bw.Tk, ksize, ws.twWd, ws.twHd, grad_kern, st)) return e;
    }
    if (grad_lmbd || grad_rho)
        return launch_bwd_scalars(bw.tau_part, bw.n_tau, bw.rho_part, bw.n_rho, lmbd, rho, grad_lmbd, grad_rho, st);
    return 0;
}

// argument checks shared by the two entry points; 0 = go on (maxit >= 1)
int check_call(const void* y, const void* out, const double* kern, int ksize, const double* lmbd, const double* rho, int B,
               int C, int H, int W, int iso, int maxit, Geometry* g) {
    if (!y || !out || !lmbd || !rho) return fail(ADMM_ERR_INVALID, "NULL tensor pointer");
    if (B < 1 || C < 1) return fail(ADMM_ERR_INVALID, "B and C must be >= 1");
    if (maxit < 0) return fail(ADMM_ERR_INVALID, "maxit must be >= 0");
    if (ksize > 0 && !kern) return fail(ADMM_ERR_INVALID, "kern is NULL but ksize > 0");
    if (int e = make_geometry_f64(B * C, H, W, iso, g)) return e;
    return check_kernel_pub(ksize, H, W);
}

}  // namespace
}  // namespace admm

using namespace admm;

extern "C" {

size_t admm_query_workspace_f64(int planes, int H, int W, int ksize, int iso, int maxit) {
    (void)maxit;
    Geometry g;
    if (make_geometry_f64(planes, H, W, iso, &g) || check_kernel_pub(ksize, H, W)) return 0;
    return carve_f64(g, ksize, nullptr, nullptr);
}

size_t admm_query_workspace_backward_f64(int planes, int H, int W, int ksize, int iso, int maxit) {
    (void)maxit;
    Geometry g;
    if (make_geometry_f64(planes, H, W, iso, &g) || check_kernel_pub(ksize, H, W)) return 0;
    return carve_f64(g, ksize, nullptr, nullptr) + carve_backward_f64(g, ksize, nullptr, nullptr);
}

size_t admm_query_saved_f64(int planes, int H, int W, int ksize, int iso, int maxit) {
    Geometry g;
    if (make_geometry_f64(planes, H, W, iso, &g) || check_kernel_pub(ksize, H, W)) return 0;
    return saved_bytes_f64(g, maxit) + 256;
}

int admm_tv_forward_f64(const double* y, double* out, const double* kern, int ksize,
                        const double* lmbd, const double* rho, int B, int C, int H, int W, int iso, int maxit,
                        void* workspace, size_t workspace_bytes, void* saved, size_t saved_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    Geometry g;
    if (int e = check_call(y, out, kern, ksize, lmbd, rho, B, C, H, W, iso, maxit, &g)) return e;
    if (maxit == 0) {                                   // deconv.py:61,103,117: x stays zeros_like(xin)
        ADMM_CUDA_CHECK(cudaMemsetAsync(out, 0, g.field_bytes, st));
        return 0;
    }
    if (int e = check_generic_f64(g, !g.iso && maxit > 1)) return e;
    if (!workspace || ((uintptr_t)workspace & 255)) return fail(ADMM_ERR_WORKSPACE, "workspace is NULL or not 256-byte aligned");
    WorkspaceF64 ws;
    if (workspace_bytes < carve_f64(g, ksize, (char*)workspace, &ws)) return fail(ADMM_ERR_WORKSPACE, "workspace too small");
    if (saved && (((uintptr_t)saved & 255) || saved_bytes < saved_bytes_f64(g, maxit)))
        return fail(ADMM_ERR_WORKSPACE, "saved-state buffer too small or misaligned");
    if (int e = setup_tables(g, ws, kern, ksize, rho, st)) return e;
    return forward_f64(g, ws, y, out, lmbd, rho, maxit, (double*)saved, st);
}

int admm_tv_backward_f64(const double* y, const double* grad_out, const double* kern, int ksize,
                         const double* lmbd, const double* rho, int B, int C, int H, int W, int iso, int maxit,
                         const void* saved, size_t saved_bytes, void* workspace, size_t workspace_bytes,
                         double* grad_y, double* grad_kern, double* grad_lmbd, double* grad_rho, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    Geometry g;
    if (int e = check_call(y, grad_out, kern, ksize, lmbd, rho, B, C, H, W, iso, maxit, &g)) return e;
    if (maxit == 0) {                                   // output is constant zero: every gradient vanishes
        if (grad_y) ADMM_CUDA_CHECK(cudaMemsetAsync(grad_y, 0, g.field_bytes, st));
        if (grad_kern && ksize > 0) ADMM_CUDA_CHECK(cudaMemsetAsync(grad_kern, 0, (size_t)ksize * ksize * sizeof(double), st));
        if (grad_lmbd) ADMM_CUDA_CHECK(cudaMemsetAsync(grad_lmbd, 0, sizeof(double), st));
        if (grad_rho) ADMM_CUDA_CHECK(cudaMemsetAsync(grad_rho, 0, sizeof(double), st));
        return 0;
    }
    if (int e = check_generic_f64(g, false)) return e;  // the backward has no halo row pass
    if (!workspace || ((uintptr_t)workspace & 255)) return fail(ADMM_ERR_WORKSPACE, "workspace is NULL or not 256-byte aligned");
    WorkspaceF64 ws; BwdWorkspaceF64 bw;
    const size_t n1 = carve_f64(g, ksize, (char*)workspace, &ws);
    const size_t n2 = carve_backward_f64(g, ksize, (char*)workspace + n1, &bw);
    if (workspace_bytes < n1 + n2) return fail(ADMM_ERR_WORKSPACE, "workspace too small (use admm_query_workspace_backward_f64)");
    if (maxit > 1 && (!saved || saved_bytes < saved_bytes_f64(g, maxit)))
        return fail(ADMM_ERR_WORKSPACE, "saved state missing or too small");
    if (int e = setup_tables(g, ws, kern, ksize, rho, st)) return e;
    return backward_f64(g, ws, bw, y, grad_out, ksize, lmbd, rho, maxit, (const double*)saved, grad_y, grad_kern, grad_lmbd,
                        grad_rho, st);
}

}  // extern "C"
