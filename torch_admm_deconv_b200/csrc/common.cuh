// common.cuh -- shared declarations of the ADMM-TV library (host side + kernel launchers).
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <cstddef>
#include <cstdint>
#include <string>

#include "fft_engine.cuh"

namespace admm {

// thread-local error text returned by admm_last_error()
void set_error(const std::string& msg);
int  fail(int code, const std::string& msg);

#define ADMM_CUDA_CHECK(expr)                                                                     \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess)                                                                    \
            return ::admm::fail(3, std::string(#expr) + ": " + cudaGetErrorString(_e));            \
    } while (0)

// process-wide tuning knobs (admm_set_option): benchmark / test switches that select between equivalent kernel
// schedules, never between algorithms.  Every field is an atomic, so concurrent host threads (autograd workers, one per
// device) may read them while another thread sets one; a call reads each knob once when it launches.
struct Options {
    std::atomic<int> rows_per_band{0};     // 0 = heuristic
    std::atomic<int> cols_per_tile{0};     // 0 = heuristic
    std::atomic<int> threads{0};           // 0 = heuristic (256 / 512 / 1024 by shared-memory footprint); generic kernels only
    std::atomic<int> force_generic{0};     // 1 = never use the specialised power-of-two kernels
    std::atomic<int> profile{0};           // 1 = bracket every kernel with CUDA events (admm_profile_read)
    std::atomic<int> use_pdl{1};           // 1 = programmatic dependent launch between the iteration kernels
    std::atomic<int> use_big{3};           // bit 0 / bit 1 = large mixed-radix row / column kernels (2160x3840) instead of the generic engine
    std::atomic<int> use_cluster{1};       // 1 = cluster-resident solver (whole solve in one launch) where it applies
    std::atomic<int> use_coop{0};          // persistent cooperative kernel for small batches (coop_small.cu): measured SLOWER than the
                                           // separate launches in 8 of 10 cases, so off; 1 = heuristic, 2 = whenever it applies (tests)
    std::atomic<int> coop_max_melems{2};   // heuristic bound of use_coop = 1: at most this many Mi elements (B*C*H*W / 2^20)
    std::atomic<int> cols_prefetch{0};     // 1 = the column pass prefetches the next resident CTA's input tile into L2
    std::atomic<int> chunk_mb{-1};         // L2-resident plane chunks: working-set budget in MB (0 = off, -1 = heuristic)
};
Options& options();

inline int wc_of(int W) { return (W + 1) / 2; }

// Problem geometry + carved workspace.  All offsets in bytes from the workspace base, 256-B aligned.
struct Geometry {
    int P, H, W, Wc;
    int iso = 0;             // block threshold over (batch, channel): needs real-space scratch fields
    size_t field_bytes;      // P*H*W*4      one real field
    size_t spec_bytes;       // P*H*Wc*8     one packed row spectrum
};

struct Workspace {
    // per-call tables
    float2* twW;  float2* twH;         // e^{-2 pi i n/N}
    double2* twWd; double2* twHd;
    double2* kdft;                     // k x (W/2+1) row-DFT of the PSF
    float*  Bm;   float* Bq;           // H*Wc real (column 0 = Bp), H real
    float*  Bmt;                       // Bm in the tile-major layout of the large column kernel (cols_big.cu)
    float2* Mul;  float2* Mq;          // H*Wc cplx (column 0 = Mp), H cplx
    float2* Mulc; float2* Mqc;         // conj-multiplier tables for the backward (grad wrt y)
    // per-plane buffers
    float2* S0; float2* S1; float2* A;
    float*  q[2][2];                   // ping-pong pre-clamp state q_x,q_y (inference)
    float*  red;                       // reduction scratch (backward)
    // iso=True only
    float*  xreal; float* vreal;       // x_k and v_{k+1} as real fields
    float*  nmap[2];                   // ping-pong pixel norms, 2 x H x W each (x field, y field)
    float*  sbmap;                     // backward: per-pixel sum_{planes} (2 wbar - ubar) q, 2 x H x W
    size_t  total;
};

size_t carve_workspace(const Geometry& g, int ksize, int maxit, char* base, Workspace* ws);
bool   ckpt_supported(const Geometry& g);      // checkpointed training (admm_ext.ckpt_interval) available for this problem

// Programmatic dependent launch: the iteration kernels may start (build their twiddle tables, set up indices) while the
// previous kernel of the stream drains; they call pdl_wait() before touching anything the previous kernel wrote.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// ---- dual of the soft threshold: u = q - soft_thresh(q, tau)   (deconv.py:15-16, 114-115)
// tau >= 0: clamp(q, -tau, tau).  tau < 0 is outside the method's domain but reachable (lmbda and rho are unconstrained
// learnable parameters, admmdeconv.py:26-41): the reference's soft_thresh then returns sign(q)(|q| + |tau|), i.e.
// u = sign(q) tau (0 at q = 0), and its derivative mask |q| < tau is never set -- which is what the backward kernels'
// `fabsf(q) < tau` already gives.  The kernels pick the variant with ONE warp-uniform branch on the sign of tau around
// their spatial step, so the usual case keeps the two-instruction clamp.
template <bool NEG>
__device__ __forceinline__ float dual_of(float q, float tau) {
    if (NEG) return q > 0.f ? tau : (q < 0.f ? -tau : 0.f);
    return fminf(fmaxf(q, -tau), tau);
}
__device__ __forceinline__ float dual_any(float q, float tau) { return tau < 0.f ? dual_of<true>(q, tau) : dual_of<false>(q, tau); }
template <bool NEG>
__device__ __forceinline__ double dual_of(double q, double tau) {
    if (NEG) return q > 0.0 ? tau : (q < 0.0 ? -tau : 0.0);
    return fmin(fmax(q, -tau), tau);
}
__device__ __forceinline__ double dual_any(double q, double tau) { return tau < 0.0 ? dual_of<true>(q, tau) : dual_of<false>(q, tau); }
struct TauPos { static constexpr bool neg = false; };
struct TauNeg { static constexpr bool neg = true; };

// ---- fused layer prologue / epilogue helpers (device)
__device__ __forceinline__ float act_apply(float v, int act) {
    switch (act) {
        case 1: return fmaxf(v, 0.f);                       // relu
        case 2: return 1.f / (1.f + expf(-v));              // sigmoid
        case 3: return tanhf(v);
        default: return v;
    }
}
// offset (floats) of plane p in the output of the last C2R: dense NCHW, or a channel slice of a wider tensor
template <class Args>
__device__ __forceinline__ size_t out_plane_offset(const Args& a, int p, int H, int W) {
    const int pp = p + a.out_p0;
    return a.out_bstride ? (size_t)(pp / a.out_C) * (size_t)a.out_bstride + (size_t)(pp % a.out_C) * H * W : (size_t)pp * H * W;
}
__device__ __forceinline__ float ld_u8_div255(const unsigned char* p) { return (float)__ldg(p) / 255.0f; }

// measurement hooks (abi.cu): every kernel launch goes through ProfScope.  The launch counter is atomic; the event
// lists (only touched when option "profile" is 1) are per device and guarded by a mutex.
enum ProfKind { PROF_ROWS = 0, PROF_COLS = 1, PROF_OTHER = 2 };
int  prof_begin(int kind, cudaStream_t st);            // returns a slot handle (< 0: not recording)
void prof_end(int kind, int slot, cudaStream_t st);
struct ProfScope {
    int kind, slot; cudaStream_t st;
    ProfScope(int k, cudaStream_t s) : kind(k), slot(prof_begin(k, s)), st(s) {}
    ~ProfScope() { if (slot >= 0) prof_end(kind, slot, st); }
};

// ------------------------------------------------------------------ kernel launchers (admm_kernels.cu)
// ROWS_FULL_U: like ROWS_FULL but the state arrays hold the clamped dual u = clamp(q) (inference: nothing is saved for a
// backward, so the clamp on load disappears); power-of-two kernels only
enum RowMode { ROWS_R2C = 0, ROWS_C2R = 1, ROWS_FULL = 2, ROWS_ADJ = 3, ROWS_FULL_U = 4 };
// COLS_INIT_SPEC: like COLS_INIT but the input already is the column-transformed spectrum of y (shared by several solvers)
enum ColMode { COLS_FFT_FWD = 0, COLS_FFT_INV = 1, COLS_INIT = 2, COLS_ITER = 3, COLS_BM_INV = 4, COLS_CMUL_INV = 5, COLS_INIT_SPEC = 6 };

// Arguments of the row and column passes, templated on the real type: T = float for the solver, T = double for the
// float64 solve (f64.cu, generic kernels only).  V = cplx_t<T>.
template <typename T>
struct RowArgsT {
    using V = cplx_t<T>;
    const T*      real_in;    // ROWS_R2C: input rows
    T*            real_out;   // ROWS_C2R: output rows
    const V*      spec_in;    // ROWS_C2R / ROWS_FULL
    V*            spec_out;   // ROWS_R2C / ROWS_FULL
    const T*      qx_in; const T* qy_in;         // ROWS_FULL: previous pre-clamp state (NULL = zeros)
    T*            qx_out; T* qy_out;             // ROWS_FULL
    const T*      lmbd; const T* rho;            // ROWS_FULL: tau = lmbd/rho
    const T*      bias;                          // ROWS_C2R: optional scalar added to the output
    // fused prologue / epilogue of the layer (admm_ext, include/admm_b200.h):
    const unsigned char* real_in_u8;             // ROWS_R2C: uint8 input; the transform sees (float)v / 255 (etransforms.py:29-31)
    int           act;                           // ROWS_C2R: activation on (x + bias) (admmdeconv.py:64): 0 none, 1 relu, 2 sigmoid, 3 tanh
                                                 // (float only: the float64 solve ignores it)
    int           out_C;                         // ROWS_C2R with out_bstride != 0: plane p goes to
    long long     out_bstride;                   //   real_out + (p / out_C) * out_bstride + (p % out_C) * H * W   (channel slice of a wider tensor)
    int           out_p0;                        // ROWS_C2R: index of this launch's first plane in the whole batch (plane chunks)
    const T*      cmap;                          // ROWS_R2C with r2c_div (power-of-two sizes): coefficient maps 2s-1 (2 x H x W),
                                                 // NULL = all ones
    int           r2c_div;                       // ROWS_R2C: the input is v = D^T(cmap * q) built from qx_in / qy_in on the fly;
                                                 // 2 (large-frame kernel only): v = D^T(q - 2 dual(q, lmbd/rho)), the anisotropic step
    // ROWS_ADJ (backward sweep, one fused row pass): spec_in = row spectrum of vbar, qx_in/qy_in = saved q_{k+1},
    // ub*_in = ubar (NULL = zeros), ub*_out = new ubar (= qbar), spec_out = row spectrum of xbar = D^T qbar,
    // taubar accumulates d/dtau; optional second output: qv* = saved q_k -> spec_out2 = row spectrum of v_k
    const T*      ubx_in; const T* uby_in;
    T*            ubx_out; T* uby_out;
    double*       taubar;
    const T*      qvx; const T* qvy;
    V*            spec_out2;
    const V*      tw;
    int tiled;                // large kernels: spec_in / spec_out are tile-major (see kSpecTile)
};
using RowArgs = RowArgsT<float>;

// Tile-major packed spectrum shared by the two large-frame kernels (rows_big.cu <-> cols_big.cu): per plane
// [tile = col / 8][row pair][col % 8][row in pair] float2.  One row pair of one tile is a 128-byte run for the row kernel
// (whole L1 lines, as with the row-major layout), and a column tile is one contiguous 138 KB block of which the column
// kernel takes one half (4 columns: 64-byte runs) per work item.  The spectrum of v (rows -> columns) pairs rows
// (2k, 2k+1); the spectrum of x (columns -> rows) pairs rows (2k-1, 2k), the pairs the row kernel transforms together.
constexpr int kSpecTile = 8;

template <typename T>
struct ColArgsT {
    using V = cplx_t<T>;
    const V*      spec_in;
    V*            spec_out;
    V*            A;          // COLS_INIT: written; COLS_ITER: read.  Private to a kernel family: the power-of-two kernels keep
                              // P0[A] (A after their first inverse pass, cols_pow2_body.cuh), cols_big.cu a tile-major A
    const T*      Bm; const T* Bq;
    const T*      Bmt;        // large column kernel: Bm as [tile][u][4] (A is kept in the same layout there)
    const V*      Mul; const V* Mq;
    const V*      tw;
    int in_tiled, out_tiled;  // large column kernel: layout of spec_in / spec_out
};
using ColArgs = ColArgsT<float>;

int launch_twiddles(float2* tw, double2* twd, int N, cudaStream_t st);
int launch_tables(const Geometry& g, const Workspace& ws, const float* kern, int ksize,
                  const float* rho, cudaStream_t st);
int launch_rows(RowMode mode, const Geometry& g, const RowArgs& a, cudaStream_t st);
int launch_cols(ColMode mode, const Geometry& g, const ColArgs& a, cudaStream_t st);

// fused backward column pass (cols_pow2.cu)
bool cols_adj_supported(const Geometry& g);
int  launch_cols_adj(const Geometry& g, const float2* spec_x, const float2* spec_v, float2* Gs, float2* GVp, float2* GVn,
                     float2* spec_out, const float* Bm, const float* Bq, const float2* tw, cudaStream_t st);

// iso=True (block threshold) spatial kernels (iso.cu)
int launch_iso_prox(const Geometry& g, const float* x, const float* qx_prev, const float* qy_prev, const float* n_prev,
                    float* qx_new, float* qy_new, float* n_new, float* c_new, const float* lmbd, const float* rho,
                    cudaStream_t st);
int launch_iso_cmap(const Geometry& g, const float* nmap, float* cmap, const float* lmbd, const float* rho, cudaStream_t st);
int launch_iso_div(const Geometry& g, const float* qx, const float* qy, const float* nmap, const float* cmap, float* v,
                   const float* lmbd, const float* rho, cudaStream_t st);
int launch_iso_bwd(const Geometry& g, const float* vb, const float* ubx_in, const float* uby_in, const float* qx,
                   const float* qy, const float* nmap, float* sbmap, float* ubx_out, float* uby_out, float* xb,
                   const float* lmbd, const float* rho, double* taubar, cudaStream_t st);

// ------------------------------------------------------------------ float64 solve (f64.cu): the generic kernels in double
int launch_twiddles_f64(double2* twd, int N, cudaStream_t st);
int launch_tables_f64(const Geometry& g, const double2* twWd, const double2* twHd, double2* kdft, double* Bm, double* Bq,
                      double2* Mul, double2* Mq, const double* kern, int ksize, const double* rho, cudaStream_t st);
int launch_rows(RowMode mode, const Geometry& g, const RowArgsT<double>& a, cudaStream_t st);   // R2C, C2R, FULL
int launch_cols(ColMode mode, const Geometry& g, const ColArgsT<double>& a, cudaStream_t st);
int check_generic_f64(const Geometry& g, bool full_rows);       // 0, or ADMM_ERR_UNSUPPORTED with a message
int launch_iso_prox(const Geometry& g, const double* x, const double* qx_prev, const double* qy_prev, const double* n_prev,
                    double* qx_new, double* qy_new, double* n_new, double* c_new, const double* lmbd, const double* rho,
                    cudaStream_t st);
int launch_iso_cmap(const Geometry& g, const double* nmap, double* cmap, const double* lmbd, const double* rho, cudaStream_t st);
int launch_iso_div(const Geometry& g, const double* qx, const double* qy, const double* nmap, const double* cmap, double* v,
                   const double* lmbd, const double* rho, cudaStream_t st);
int launch_iso_bwd(const Geometry& g, const double* vb, const double* ubx_in, const double* uby_in, const double* qx,
                   const double* qy, const double* nmap, double* sbmap, double* ubx_out, double* uby_out, double* xb,
                   const double* lmbd, const double* rho, double* taubar, cudaStream_t st);
// backward.cu: the generic backward kernels in double (the float solver launches them itself)
int launch_bwd_spatial(const Geometry& g, const double* vb, const double* ubx_in, const double* uby_in, const double* qx,
                       const double* qy, double* ubx_out, double* uby_out, double* xb, const double* lmbd, const double* rho,
                       double* taubar, cudaStream_t st);
int launch_bwd_recompute_v(const Geometry& g, const double* qx, const double* qy, double* v, const double* lmbd,
                           const double* rho, cudaStream_t st);
int launch_bwd_accumulate(const Geometry& g, int nsplit, const double2* ZG, const double2* ZV, const double2* ZY, double2* Gs,
                          double2* C1, double2* GV, int update_gs, cudaStream_t st);
int launch_bwd_finalize(const Geometry& g, const double2* C1, const double2* GV, int nsplit, double2* S, double* rho_part,
                        int ks, const double2* G, const double2* twHd, const double2* twWd, const double* rho, cudaStream_t st);
int launch_bwd_kgrad(const Geometry& g, const double2* S, double2* Tk, int ks, const double2* twWd, const double2* twHd,
                     double* grad_kern, cudaStream_t st);
int launch_bwd_scalars(const double* tau_part, size_t n_tau, const double* rho_part, size_t n_rho, const double* lmbd,
                       const double* rho, double* grad_lmbd, double* grad_rho, cudaStream_t st);

// specialised power-of-two kernels (rows_pow2.cu, cols_pow2.cu)
bool rows_pow2_supported(const Geometry& g);
int  launch_rows_pow2(RowMode mode, const Geometry& g, const RowArgs& a, cudaStream_t st);
bool cols_pow2_supported(const Geometry& g);
bool cols_pow2_mode_supported(ColMode mode);
int  launch_cols_pow2(ColMode mode, const Geometry& g, const ColArgs& a, cudaStream_t st);

// cluster-resident solver for small planes (cluster_pow2.cu): the whole solve in one launch, state in distributed shared memory
struct ClusterArgs {
    const float* y; const unsigned char* y8;      // input planes (fp32, or uint8 read as v / 255)
    float* out;                                   // output planes
    const float2* twW; const float2* twH;         // e^{-2 pi i n / N}
    const float* Bm; const float* Bq;             // H x Wc, H          (tables of admm_kernels.cu:k_tables)
    const float2* Mul; const float2* Mq;          // H x Wc, H
    const float* lmbd; const float* rho; const float* bias;
    int act, out_C, out_p0; long long out_bstride;
    int P, maxit;
};

bool cluster_solver_supported(const Geometry& g, int iso, bool training);
bool cluster_solver_preferred(const Geometry& g);
int  launch_cluster_solve(const Geometry& g, const ClusterArgs& a, cudaStream_t st);

// persistent cooperative kernel for small batches (coop_small.cu): iterations 1 .. maxit-1 in one launch, grid.sync between phases
bool coop_solver_supported(const Geometry& g);
bool coop_solver_preferred(const Geometry& g);
int  launch_coop_iterations(const Geometry& g, const Workspace& ws, const float* lmbd, const float* rho, int maxit, cudaStream_t st);

// large mixed-radix sizes (rows_big.cu, cols_big.cu): the 2160x3840 single-frame configuration
bool rows_big_supported(const Geometry& g);
int  launch_rows_big(RowMode mode, const Geometry& g, const RowArgs& a, cudaStream_t st);
int  launch_rows_big_plain(RowMode mode, const Geometry& g, const RowArgs& a, cudaStream_t st);   // ROWS_R2C / ROWS_C2R
bool cols_big_supported(const Geometry& g);
int  launch_cols_big(ColMode mode, const Geometry& g, const ColArgs& a, cudaStream_t st);
int  launch_bm_tiled(const Geometry& g, const float* Bm, float* Bmt, cudaStream_t st);

}  // namespace admm
