/* admm_b200.h -- C ABI of the B200-native ADMM-TV deconvolution hot path.
 *
 * The reference (georgegrosu1/torch-admm-deconv) has NO foreign-function boundary: its hot path
 * is the Python function
 *     fft_admm_tv(xin, lmbd, rho, kern, iso=False, maxit=100)        src/admmtor/eops/deconv.py:35-117
 * called by
 *     ADMMDeconv.forward(x)                                          src/admmtor/elayers/admmdeconv.py:63-64
 * and its backward is stock autograd over that loop.  This header declares the plain-C entry
 * points a binding for that path needs; the Python mirror of the reference API lives in
 * torch_admm_deconv_b200/ and reaches these symbols with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name starts with `host_`;
 *   - image fields are fp32, contiguous NCHW; a "plane" is one (b, c) image, planes = B*C (the *_f64 calls: fp64
 *     everywhere, see "float64 solve" below);
 *   - lmbd / rho are device pointers to ONE float each (learnable parameters: never read on host);
 *   - kern is (ksize x ksize) fp32 row-major, or NULL with ksize == 0 for the TV-denoise branch
 *     (deconv.py:46-47, 86-87);
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); nothing synchronises;
 *   - the library allocates nothing: the caller owns `workspace` (size from admm_query_workspace)
 *     and the optional `saved` state; both must be 256-byte aligned;
 *   - return value 0 = ok; non-zero = error, text available from admm_last_error() (thread-local).
 */
#ifndef ADMM_B200_H
#define ADMM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ADMM_B200_VERSION 300   /* major*10000 + minor*100 + patch */

/* error codes */
#define ADMM_OK                0
#define ADMM_ERR_INVALID       1   /* bad argument (shape, NULL pointer, unsupported size) */
#define ADMM_ERR_WORKSPACE     2   /* workspace / saved buffer too small or misaligned */
#define ADMM_ERR_CUDA          3   /* a CUDA runtime call failed */
#define ADMM_ERR_UNSUPPORTED   4   /* valid request this build cannot run (e.g. FFT does not fit in shared memory) */

int         admm_version(void);
const char* admm_last_error(void);

/* Tuning knobs ("rows_per_band", "cols_per_tile", "threads", "force_generic", ...).  Returns 0 if the
 * key is known.  Process-wide; intended for benchmarks and tests. */
int  admm_set_option(const char* key, int value);
int  admm_get_option(const char* key, int* value);

/* Bytes of scratch needed by admm_tv_forward for this problem (0 on error). */
size_t admm_query_workspace(int planes, int H, int W, int ksize, int iso, int maxit);
/* Bytes of scratch needed by admm_tv_backward (larger than the forward's). */
size_t admm_query_workspace_backward(int planes, int H, int W, int ksize, int iso, int maxit);
/* Bytes of saved state admm_tv_forward writes when `saved != NULL` (consumed by admm_tv_backward). */
size_t admm_query_saved(int planes, int H, int W, int ksize, int iso, int maxit);

/* Replaces fft_admm_tv (deconv.py:35-117): out = last x iterate, zeros when maxit == 0 (deconv.py:61,117).
 *   y, out : (B, C, H, W) fp32     bias: optional device pointer to one float added to out
 *                                  (ADMMDeconv.forward's `+ self.b`, admmdeconv.py:64), or NULL
 *   saved  : NULL for inference; otherwise receives the per-iteration state the backward needs. */
int admm_tv_forward(const float* y, float* out,
                    const float* kern, int ksize,
                    const float* lmbd, const float* rho, const float* bias,
                    int B, int C, int H, int W, int iso, int maxit,
                    void* workspace, size_t workspace_bytes,
                    void* saved, size_t saved_bytes,
                    void* stream);

/* Fused layer prologue / epilogue and output placement, for callers of the layer (ADMMDeconv.forward, admmdeconv.py:64,
 * and the multi-solver containers MultiADMM / Deconvs / ADMMFusion, blocks.py:252-261, deconver.py:8-23,
 * admmfusion.py:28-40).  Zero-initialise, set struct_size = sizeof(admm_ext), fill what is needed. */
#define ADMM_IN_F32        0
#define ADMM_IN_U8_DIV255  1   /* y points to uint8 NCHW; the solve sees (float)y / 255 (eprocessing/etransforms.py:29-31) */
#define ADMM_ACT_NONE      0
#define ADMM_ACT_RELU      1
#define ADMM_ACT_SIGMOID   2
#define ADMM_ACT_TANH      3
typedef struct admm_ext {
    int       struct_size;       /* sizeof(admm_ext) of the caller's header (lets the struct grow) */
    int       in_dtype;          /* ADMM_IN_*: element type of y, converted inside the first row pass */
    int       activation;        /* ADMM_ACT_*: out = act(x + bias), applied by the last row pass (admmdeconv.py:64) */
    int       ckpt_interval;     /* training only: K >= 2 keeps the per-iteration state of every K-th iteration instead of all of
                                    them (memory / recompute trade: the backward re-runs each block of K iterations from its
                                    checkpoint).  0 or 1 = keep every iteration.  iso = 0 only (every frame size, the large
                                    frames of the tile-major kernels included).  Sizes: admm_query_saved_ex,
                                    admm_query_workspace_backward_ex; pass the same K to admm_tv_backward_ex. */
    long long out_batch_stride;  /* floats between consecutive images of `out`; 0 = dense (C*H*W).  With a larger stride the
                                    C planes of image b land at out + b*stride: the channel slice of a concatenated tensor
                                    (torch.cat([admm(x) for admm in admms], dim=1) without the copy) */
    const float* yhat_in;        /* optional: column-transformed packed spectrum of y, as written through yhat_out by an
                                    earlier call on the same y (solvers that share the input skip their R2C + column FFT) */
    float*    yhat_out;          /* optional: receives that spectrum (admm_query_yhat bytes) */
} admm_ext;

size_t admm_query_yhat(int planes, int H, int W);      /* bytes of the shared spectrum buffer (0 on error) */

/* yhat = column-transformed packed row spectrum of y (the F(y) every solver on this input starts from); workspace as
 * for admm_dbg_* (admm_query_workspace(planes, H, W, 0, 0, 1)).  Pass the result as admm_ext.yhat_in. */
int admm_spectrum_forward(const void* y, int in_dtype, float* yhat, int planes, int H, int W,
                          void* workspace, size_t workspace_bytes, void* stream);

/* admm_tv_forward with the extras above; ext == NULL behaves exactly like admm_tv_forward. */
int admm_tv_forward_ex(const void* y, float* out,
                       const float* kern, int ksize,
                       const float* lmbd, const float* rho, const float* bias,
                       int B, int C, int H, int W, int iso, int maxit,
                       void* workspace, size_t workspace_bytes,
                       void* saved, size_t saved_bytes,
                       void* stream, const admm_ext* ext);

/* Checkpointed training (admm_ext.ckpt_interval = K): bytes of saved state and of backward workspace. */
size_t admm_query_saved_ex(int planes, int H, int W, int ksize, int iso, int maxit, int ckpt_interval);
size_t admm_query_workspace_backward_ex(int planes, int H, int W, int ksize, int iso, int maxit, int ckpt_interval);

/* Replaces autograd through deconv.py:103-115.  grad_* outputs may be NULL when not wanted.
 *   grad_out  : (B, C, H, W)        grad_y    : (B, C, H, W)
 *   grad_kern : (ksize, ksize)      grad_lmbd, grad_rho : one float each (overwritten, not accumulated) */
int admm_tv_backward(const float* y, const float* grad_out,
                     const float* kern, int ksize,
                     const float* lmbd, const float* rho,
                     int B, int C, int H, int W, int iso, int maxit,
                     const void* saved, size_t saved_bytes,
                     void* workspace, size_t workspace_bytes,
                     float* grad_y, float* grad_kern, float* grad_lmbd, float* grad_rho,
                     void* stream);

/* admm_tv_backward for a forward that ran with admm_ext.ckpt_interval = K (K <= 1: identical to admm_tv_backward). */
int admm_tv_backward_ex(const float* y, const float* grad_out,
                        const float* kern, int ksize,
                        const float* lmbd, const float* rho,
                        int B, int C, int H, int W, int iso, int maxit,
                        const void* saved, size_t saved_bytes,
                        void* workspace, size_t workspace_bytes,
                        float* grad_y, float* grad_kern, float* grad_lmbd, float* grad_rho,
                        void* stream, int ckpt_interval);

/* ---- float64 solve.  The reference computes in xin.dtype (deconv.py:50-67); these calls are the float32 ones above with
 * double in place of float for every tensor (y, out, kern, lmbd, rho, saved state, gradients), same conventions, error
 * codes and semantics (iso, empty PSF, negative tau, maxit = 0 / 1).  They run on the generic (any H, W) kernels
 * instantiated for double.  Shared memory bounds the size: the column pass needs H <= 4842, the row pass W <= 2905 for
 * iso = 0 with maxit >= 2 (two halo rows) and W <= 4842 otherwise; a larger frame returns ADMM_ERR_UNSUPPORTED before
 * anything is launched.  No bias, activation, uint8 input, shared spectrum or checkpointing.
 * Saved state: [slot][q_x, q_y][all planes] for slots 0 .. maxit-2, then for iso = 1 the maxit-1 pairs of H x W pixel-norm
 * maps, in double (admm_query_saved_f64 = 2 x admm_query_saved - 256: both include one 256-byte pad). */
size_t admm_query_workspace_f64(int planes, int H, int W, int ksize, int iso, int maxit);
size_t admm_query_workspace_backward_f64(int planes, int H, int W, int ksize, int iso, int maxit);
size_t admm_query_saved_f64(int planes, int H, int W, int ksize, int iso, int maxit);
int admm_tv_forward_f64(const double* y, double* out, const double* kern, int ksize,
                        const double* lmbd, const double* rho, int B, int C, int H, int W, int iso, int maxit,
                        void* workspace, size_t workspace_bytes, void* saved, size_t saved_bytes, void* stream);
int admm_tv_backward_f64(const double* y, const double* grad_out, const double* kern, int ksize,
                         const double* lmbd, const double* rho, int B, int C, int H, int W, int iso, int maxit,
                         const void* saved, size_t saved_bytes, void* workspace, size_t workspace_bytes,
                         double* grad_y, double* grad_kern, double* grad_lmbd, double* grad_rho, void* stream);

/* ---- measurement hooks (bench.py): per-kernel-class device time from CUDA events recorded on the launch
 * stream when option "profile" is 1, and the number of kernels launched since the last reset.
 *   kind: 0 = row pass (C2R + prox/dual/divergence + R2C), 1 = column pass (FFT, A + Bm*V, iFFT), 2 = other */
int admm_profile_reset(void);
int admm_profile_read(int kind, double* total_ms, int* launches);   /* synchronises the recorded events */
long long admm_launch_count(void);

/* ---- stage-level entry points (used by the parity tests to localise errors; same kernels) ----
 * Packed row spectrum: per plane H x Wc complex64, Wc = (W+1)/2; entry [r][0] = (Re DC, Re Nyquist). */
int admm_dbg_rows_r2c(const float* real_in, float* rowspec_out, int planes, int H, int W,
                      void* workspace, size_t workspace_bytes, void* stream);
int admm_dbg_rows_c2r(const float* rowspec_in, float* real_out, int planes, int H, int W,
                      void* workspace, size_t workspace_bytes, void* stream);   /* unnormalised */
int admm_dbg_cols_fft(const float* rowspec_in, float* rowspec_out, int planes, int H, int W, int inverse,
                      void* workspace, size_t workspace_bytes, void* stream);   /* unnormalised */

#ifdef __cplusplus
}
#endif
#endif /* ADMM_B200_H */
