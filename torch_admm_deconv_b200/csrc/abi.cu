// abi.cu -- extern "C" entry points declared in include/admm_b200.h.
//
// Kernel launch sequence of admm_tv_forward (replaces fft_admm_tv, deconv.py:35-117), maxit = N >= 1:
//     twiddles, tables                                  deconv.py:44-57   (per call, like the reference)
//     rows R2C : y -> S1                                 deconv.py:104     (rfftn of H_t(xin), once)
//     cols INIT: S1 -> A, S0 = iFFT_col(A)                                (x_1 = F^-1[A]; z = u = 0)
//     repeat N-1 times:
//         rows FULL: S0 -> x_k -> q_k, v_{k+1} -> S1      deconv.py:106-115, 104
//         cols ITER: S1 -> S0                             deconv.py:104-106
//     rows C2R : S0 -> out (+ bias)                       deconv.py:117, admmdeconv.py:64
#include <algorithm>
#include <atomic>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/admm_b200.h"
#include "common.cuh"

namespace admm {

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
int fail(int code, const std::string& msg) { g_err = msg; return code; }

Options& options() {
    static Options o;
    return o;
}

// ---- measurement hooks -------------------------------------------------------------------------
// launch counter: atomic.  Event pairs: one list per (device, kind), created lazily, guarded by a mutex; nothing here is
// touched on the launch path unless option "profile" is 1.
static constexpr int kMaxProfEvents = 16384;
static constexpr int kMaxProfDevices = 16;
struct ProfList {
    std::vector<cudaEvent_t> ev;          // 2 per recorded launch
    int used = 0;                         // launches recorded since the last reset
};
static std::mutex g_prof_mu;
static ProfList g_prof[kMaxProfDevices][3];
static std::atomic<long long> g_launches{0};

int prof_begin(int kind, cudaStream_t st) {
    g_launches.fetch_add(1, std::memory_order_relaxed);
    if (!options().profile) return -1;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxProfDevices) return -1;
    std::lock_guard<std::mutex> lk(g_prof_mu);
    ProfList& L = g_prof[dev][kind];
    if (L.used >= kMaxProfEvents) return -1;
    const int i = L.used;
    while ((int)L.ev.size() < 2 * (i + 1)) {
        cudaEvent_t e;
        if (cudaEventCreate(&e) != cudaSuccess) return -1;
        L.ev.push_back(e);
    }
    cudaEventRecord(L.ev[2 * i], st);
    L.used = i + 1;
    return dev * kMaxProfEvents + i;
}

void prof_end(int kind, int slot, cudaStream_t st) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    ProfList& L = g_prof[slot / kMaxProfEvents][kind];
    const int i = slot % kMaxProfEvents;
    if (i < L.used && 2 * i + 1 < (int)L.ev.size()) cudaEventRecord(L.ev[2 * i + 1], st);
}

static inline size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }

size_t carve_workspace(const Geometry& g, int ksize, int maxit, char* base, Workspace* ws) {
    size_t off = 0;
    auto take = [&](size_t bytes) {
        char* p = base ? base + off : nullptr;
        off += align_up(bytes);
        return p;
    };
    Workspace w;
    std::memset(&w, 0, sizeof(w));
    const size_t HWc = (size_t)g.H * g.Wc;
    w.twW  = (float2*)take((size_t)g.W * sizeof(float2));
    w.twH  = (float2*)take((size_t)g.H * sizeof(float2));
    w.twWd = (double2*)take((size_t)g.W * sizeof(double2));
    w.twHd = (double2*)take((size_t)g.H * sizeof(double2));
    w.kdft = (double2*)take((size_t)(ksize > 0 ? ksize : 1) * (g.W / 2 + 1) * sizeof(double2));
    w.Bm   = (float*)take(HWc * sizeof(float));
    w.Bq   = (float*)take((size_t)g.H * sizeof(float));
    w.Bmt  = (float*)take(HWc * sizeof(float));
    w.Mul  = (float2*)take(HWc * sizeof(float2));
    w.Mq   = (float2*)take((size_t)g.H * sizeof(float2));
    w.Mulc = nullptr; w.Mqc = nullptr;
    w.S0 = (float2*)take(g.spec_bytes);
    w.S1 = (float2*)take(g.spec_bytes);
    w.A  = (float2*)take(g.spec_bytes);
    for (int i = 0; i < 2; ++i)
        for (int f = 0; f < 2; ++f) w.q[i][f] = (float*)take(g.field_bytes);
    w.red = (float*)take(4096);
    if (g.iso) {
        const size_t map_bytes = (size_t)2 * g.H * g.W * sizeof(float);
        w.xreal = (float*)take(g.field_bytes);
        w.vreal = (float*)take(g.field_bytes);
        w.nmap[0] = (float*)take(map_bytes);
        w.nmap[1] = (float*)take(map_bytes);
        w.sbmap = (float*)take(map_bytes);
    }
    w.total = off;
    if (ws) *ws = w;
    return off;
}

static int make_geometry(int planes, int H, int W, Geometry* g) {
    if (planes < 1) return fail(ADMM_ERR_INVALID, "planes (B*C) must be >= 1");
    if (H < 2 || W < 2) return fail(ADMM_ERR_INVALID, "H and W must be >= 2");
    if ((long long)H * W > (1LL << 30)) return fail(ADMM_ERR_INVALID, "image too large");
    g->P = planes; g->H = H; g->W = W; g->Wc = wc_of(W);
    g->field_bytes = (size_t)planes * H * W * sizeof(float);
    g->spec_bytes = (size_t)planes * H * g->Wc * sizeof(float2);
    return 0;
}

static int check_kernel(int ksize, int H, int W) {
    if (ksize < 0) return fail(ADMM_ERR_INVALID, "ksize must be >= 0");
    if (ksize > H || ksize > W) return fail(ADMM_ERR_INVALID, "PSF larger than the image");
    return 0;
}

int make_geometry_pub(int planes, int H, int W, Geometry* g) { return make_geometry(planes, H, W, g); }
// checkpointed training re-runs blocks of the forward inside the backward (backward.cu, regen_block), on every kernel
// route of iso = 0; the iso = 1 state (pixel-norm maps of every iteration) has no restart
bool ckpt_supported(const Geometry& g) { return !g.iso; }
int check_kernel_pub(int ksize, int H, int W) { return check_kernel(ksize, H, W); }

}  // namespace admm

using namespace admm;

// Default L2 working-set budget of a plane chunk (MB); see admm_tv_forward_ex.  B200: 126 MB L2.
static constexpr int kDefaultChunkMB = 0;

// All iterations for the planes of one chunk (gc.P planes starting at plane p0 of the batch described by gall).
static int solve_planes(const Geometry& g, const Geometry& gall, const Workspace& ws, const float* y, const unsigned char* y8,
                        float* out, int p0, int C, const float* kern, int ksize, const float* lmbd, const float* rho,
                        const float* bias, int maxit, float* saved, size_t fe_all, int slots, size_t map_floats,
                        const admm_ext& ext, size_t off_spec, cudaStream_t st) {
    const int H = g.H, W = g.W;
    const bool iso = g.iso != 0;
    (void)kern; (void)ksize; (void)gall;
    RowArgs ra; std::memset(&ra, 0, sizeof(ra));
    ColArgs ca; std::memset(&ca, 0, sizeof(ca));
    ra.tw = ws.twW; ra.lmbd = lmbd; ra.rho = rho;
    ca.tw = ws.twH; ca.A = ws.A; ca.Bm = ws.Bm; ca.Bq = ws.Bq; ca.Bmt = ws.Bmt; ca.Mul = ws.Mul; ca.Mq = ws.Mq;

    // 2160x3840 frames: between the two large kernels the packed spectra travel tile-major (common.cuh, kSpecTile);
    // the generic R2C before the loop and C2R after it keep the row-major layout
    const bool tiled = rows_big_supported(g) && cols_big_supported(g);
    if (!ext.yhat_in) {
        ra.real_in = y; ra.real_in_u8 = y8; ra.spec_out = ws.S1;
        if (int e = launch_rows(ROWS_R2C, g, ra, st)) return e;
        ra.real_in_u8 = nullptr;
    }
    ca.in_tiled = 0; ca.out_tiled = (tiled && maxit > 1) ? 1 : 0;
    if (ext.yhat_in || ext.yhat_out) {
        // several solvers on the same input (MultiADMM / Deconvs / ADMMFusion): F(y) is computed once and every solver
        // starts from it, A = Mul_s F(y)
        const float2* yh = ext.yhat_in ? (const float2*)ext.yhat_in + off_spec : nullptr;
        if (!yh) {
            ca.spec_in = ws.S1; ca.spec_out = (float2*)ext.yhat_out + off_spec;
            if (int e = launch_cols(COLS_FFT_FWD, g, ca, st)) return e;
            yh = (const float2*)ext.yhat_out + off_spec;
        }
        ca.spec_in = yh; ca.spec_out = ws.S0;
        if (int e = launch_cols(COLS_INIT_SPEC, g, ca, st)) return e;
    } else {
        ca.spec_in = ws.S1; ca.spec_out = ws.S0;
        if (int e = launch_cols(COLS_INIT, g, ca, st)) return e;
    }

    const float* qx_prev = nullptr; const float* qy_prev = nullptr;
    // small, latency-bound batches (inference): iterations 1 .. maxit-1 in ONE cooperative launch (coop_small.cu)
    const bool coop = !saved && maxit > 1 && !tiled && coop_solver_supported(g) && coop_solver_preferred(g);
    if (coop) {
        if (int e = launch_coop_iterations(g, ws, lmbd, rho, maxit, st)) return e;
    }
    for (int it = 1; it < maxit && !coop; ++it) {
        float* qx_new; float* qy_new;
        const int K = ext.ckpt_interval;
        if (saved && K >= 2 && (it % K) != 0) {        // checkpointed training: this iteration's state is not kept
            qx_new = ws.q[it & 1][0]; qy_new = ws.q[it & 1][1];
        } else if (saved) {                            // layout [slot][field][all planes of the batch]; `saved` points at plane p0
            const int slot = (K >= 2) ? it / K - 1 : it - 1;
            qx_new = saved + (size_t)slot * 2 * fe_all;
            qy_new = qx_new + fe_all;
        } else {
            qx_new = ws.q[it & 1][0]; qy_new = ws.q[it & 1][1];
        }
        if (iso) {
            // block threshold couples all planes of a pixel (pixelnorm over dims (0,1), deconv.py:19-24): the row
            // pass is split into C2R, a per-pixel prox over the planes, the divergence, and R2C   (never chunked)
            const float* n_prev = (it == 1) ? nullptr
                                : (saved ? saved + (size_t)slots * 2 * fe_all + (size_t)(it - 2) * map_floats : ws.nmap[(it - 1) & 1]);
            float* n_new = saved ? saved + (size_t)slots * 2 * fe_all + (size_t)(it - 1) * map_floats : ws.nmap[it & 1];
            ra.spec_in = ws.S0; ra.real_out = ws.xreal; ra.bias = nullptr; ra.tiled = tiled ? 1 : 0;
            if (int e = launch_rows(ROWS_C2R, g, ra, st)) return e;
            if (int e = launch_iso_prox(g, ws.xreal, qx_prev, qy_prev, n_prev, qx_new, qy_new, n_new, ws.sbmap, lmbd, rho, st)) return e;
            if (rows_pow2_supported(g) || rows_big_supported(g)) {   // divergence fused into the R2C row pass
                RowArgs rb = ra;
                rb.r2c_div = 1; rb.cmap = ws.sbmap; rb.qx_in = qx_new; rb.qy_in = qy_new; rb.spec_out = ws.S1;
                if (int e = launch_rows(ROWS_R2C, g, rb, st)) return e;
            } else {
                if (int e = launch_iso_div(g, qx_new, qy_new, n_new, ws.sbmap, ws.vreal, lmbd, rho, st)) return e;
                ra.real_in = ws.vreal; ra.spec_out = ws.S1;
                if (int e = launch_rows(ROWS_R2C, g, ra, st)) return e;
            }
        } else {
            ra.spec_in = ws.S0; ra.spec_out = ws.S1;
            ra.qx_in = qx_prev; ra.qy_in = qy_prev; ra.qx_out = qx_new; ra.qy_out = qy_new;
            ra.tiled = tiled ? 1 : 0;
            // inference on the specialised kernels keeps the clamped dual as state (no clamp on reload)
            const RowMode fm = (!saved && (rows_pow2_supported(g) || rows_big_supported(g))) ? ROWS_FULL_U : ROWS_FULL;
            if (int e = launch_rows(fm, g, ra, st)) return e;
        }
        ca.spec_in = ws.S1; ca.spec_out = ws.S0;
        ca.in_tiled = tiled ? 1 : 0; ca.out_tiled = (tiled && it + 1 < maxit) ? 1 : 0;
        if (int e = launch_cols(COLS_ITER, g, ca, st)) return e;
        qx_prev = qx_new; qy_prev = qy_new;
    }
    ra.spec_in = ws.S0; ra.real_out = out; ra.bias = bias; ra.tiled = 0;
    ra.act = ext.activation; ra.out_C = C; ra.out_p0 = p0;
    ra.out_bstride = (ext.out_batch_stride == (long long)C * H * W) ? 0 : ext.out_batch_stride;
    if (int e = launch_rows(ROWS_C2R, g, ra, st)) return e;
    return 0;
}

// maxit == 0: the solve returns zeros and the layer computes act(0 + b); image blockIdx.y starts at out + y * stride
__global__ void k_fill_scalar(float* __restrict__ out, const float* __restrict__ value, int act, size_t n, size_t stride) {
    const float v = act_apply(value ? value[0] : 0.f, act);
    float* o = out + (size_t)blockIdx.y * stride;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) o[i] = v;
}

extern "C" {

int admm_version(void) { return ADMM_B200_VERSION; }
const char* admm_last_error(void) { return g_err.c_str(); }

int admm_set_option(const char* key, int value) {
    if (!key) return 1;
    Options& o = options();
    if (!std::strcmp(key, "rows_per_band")) { o.rows_per_band = value; return 0; }
    if (!std::strcmp(key, "cols_per_tile")) { o.cols_per_tile = value; return 0; }
    if (!std::strcmp(key, "threads")) {
        if (value != 0 && (value < 32 || value > 1024 || value % 32)) return 1;
        o.threads = value; return 0;
    }
    if (!std::strcmp(key, "force_generic")) { o.force_generic = value; return 0; }
    if (!std::strcmp(key, "profile")) { o.profile = value ? 1 : 0; return 0; }
    if (!std::strcmp(key, "use_big")) { o.use_big = value & 3; return 0; }
    if (!std::strcmp(key, "use_pdl")) { o.use_pdl = value ? 1 : 0; return 0; }
    if (!std::strcmp(key, "use_cluster")) { o.use_cluster = value; return 0; }     // 0 off, 1 heuristic, 2 always
    if (!std::strcmp(key, "chunk_mb")) { o.chunk_mb = value; return 0; }
    if (!std::strcmp(key, "cols_prefetch")) { o.cols_prefetch = value ? 1 : 0; return 0; }
    if (!std::strcmp(key, "use_coop")) { o.use_coop = value; return 0; }                  // 0 off, 1 heuristic, 2 always
    if (!std::strcmp(key, "coop_max_melems")) { o.coop_max_melems = value; return 0; }
    return 1;
}

int admm_profile_reset(void) {
    {
        std::lock_guard<std::mutex> lk(g_prof_mu);
        for (int d = 0; d < kMaxProfDevices; ++d)
            for (int k = 0; k < 3; ++k) g_prof[d][k].used = 0;
    }
    g_launches.store(0);
    return 0;
}

int admm_profile_read(int kind, double* total_ms, int* launches) {
    if (kind < 0 || kind > 2 || !total_ms || !launches) return fail(ADMM_ERR_INVALID, "bad profile query");
    int dev = 0;
    ADMM_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= kMaxProfDevices) return fail(ADMM_ERR_INVALID, "profile: device index out of range");
    std::lock_guard<std::mutex> lk(g_prof_mu);
    ProfList& L = g_prof[dev][kind];
    double tot = 0.0;
    for (int i = 0; i < L.used; ++i) {
        ADMM_CUDA_CHECK(cudaEventSynchronize(L.ev[2 * i + 1]));
        float ms = 0.f;
        ADMM_CUDA_CHECK(cudaEventElapsedTime(&ms, L.ev[2 * i], L.ev[2 * i + 1]));
        tot += ms;
    }
    *total_ms = tot; *launches = L.used;
    return 0;
}

long long admm_launch_count(void) { return g_launches.load(); }

int admm_get_option(const char* key, int* value) {
    if (!key || !value) return 1;
    Options& o = options();
    if (!std::strcmp(key, "rows_per_band")) { *value = o.rows_per_band; return 0; }
    if (!std::strcmp(key, "cols_per_tile")) { *value = o.cols_per_tile; return 0; }
    if (!std::strcmp(key, "threads")) { *value = o.threads; return 0; }
    if (!std::strcmp(key, "force_generic")) { *value = o.force_generic; return 0; }
    if (!std::strcmp(key, "profile")) { *value = o.profile; return 0; }
    if (!std::strcmp(key, "use_big")) { *value = o.use_big; return 0; }
    if (!std::strcmp(key, "use_pdl")) { *value = o.use_pdl; return 0; }
    if (!std::strcmp(key, "use_cluster")) { *value = o.use_cluster; return 0; }
    if (!std::strcmp(key, "chunk_mb")) { *value = o.chunk_mb; return 0; }
    if (!std::strcmp(key, "cols_prefetch")) { *value = o.cols_prefetch; return 0; }
    if (!std::strcmp(key, "use_coop")) { *value = o.use_coop; return 0; }
    if (!std::strcmp(key, "coop_max_melems")) { *value = o.coop_max_melems; return 0; }
    return 1;
}

size_t admm_query_workspace(int planes, int H, int W, int ksize, int iso, int maxit) {
    Geometry g;
    if (make_geometry(planes, H, W, &g)) return 0;
    if (check_kernel(ksize, H, W)) return 0;
    g.iso = iso ? 1 : 0;
    return carve_workspace(g, ksize, maxit, nullptr, nullptr);
}

size_t admm_query_saved(int planes, int H, int W, int ksize, int iso, int maxit) {
    return admm_query_saved_ex(planes, H, W, ksize, iso, maxit, 0);
}

size_t admm_query_saved_ex(int planes, int H, int W, int ksize, int iso, int maxit, int ckpt_interval) {
    Geometry g;
    if (make_geometry(planes, H, W, &g)) return 0;
    (void)ksize;
    // q_x, q_y of iterations 1 .. maxit-1 (the prox after the last x-update is never consumed);
    // iso=True additionally keeps the two pixel-norm maps of every iteration.
    // Checkpointed (K >= 2, iso = 0): only the slots i with (i + 1) % K == 0 are kept.
    int slots = maxit > 1 ? maxit - 1 : 0;
    if (ckpt_interval >= 2) {
        g.iso = iso ? 1 : 0;
        if (!ckpt_supported(g)) return 0;
        slots = slots / ckpt_interval;
    }
    size_t n = (size_t)slots * 2 * g.field_bytes + 256;
    if (iso) n += (size_t)slots * 2 * H * W * sizeof(float);
    return n;
}

int admm_tv_forward(const float* y, float* out, const float* kern, int ksize,
                    const float* lmbd, const float* rho, const float* bias,
                    int B, int C, int H, int W, int iso, int maxit,
                    void* workspace, size_t workspace_bytes, void* saved, size_t saved_bytes,
                    void* stream) {
    return admm_tv_forward_ex(y, out, kern, ksize, lmbd, rho, bias, B, C, H, W, iso, maxit, workspace, workspace_bytes,
                              saved, saved_bytes, stream, nullptr);
}

size_t admm_query_yhat(int planes, int H, int W) {
    Geometry g;
    if (make_geometry(planes, H, W, &g)) return 0;
    g.iso = 0;
    if (cols_big_supported(g)) return 0;     // the large-frame column kernel keeps its own layouts: no shared spectrum there
    return g.spec_bytes;
}

int admm_tv_forward_ex(const void* y_any, float* out, const float* kern, int ksize,
                       const float* lmbd, const float* rho, const float* bias,
                       int B, int C, int H, int W, int iso, int maxit,
                       void* workspace, size_t workspace_bytes, void* saved, size_t saved_bytes,
                       void* stream, const admm_ext* ext_in) {
    cudaStream_t st = (cudaStream_t)stream;
    admm_ext ext;
    std::memset(&ext, 0, sizeof(ext));
    if (ext_in) {
        if (ext_in->struct_size < (int)(4 * sizeof(int)) || ext_in->struct_size > (int)sizeof(admm_ext))
            return fail(ADMM_ERR_INVALID, "admm_ext.struct_size does not match this library");
        std::memcpy(&ext, ext_in, (size_t)ext_in->struct_size);
    }
    if (ext.in_dtype != ADMM_IN_F32 && ext.in_dtype != ADMM_IN_U8_DIV255) return fail(ADMM_ERR_INVALID, "unknown admm_ext.in_dtype");
    if (ext.activation < ADMM_ACT_NONE || ext.activation > ADMM_ACT_TANH) return fail(ADMM_ERR_INVALID, "unknown admm_ext.activation");
    if (ext.out_batch_stride != 0 && ext.out_batch_stride < (long long)C * H * W)
        return fail(ADMM_ERR_INVALID, "admm_ext.out_batch_stride is smaller than one image (C*H*W floats)");
    const float* y = (ext.in_dtype == ADMM_IN_F32) ? (const float*)y_any : nullptr;
    const unsigned char* y8 = (ext.in_dtype == ADMM_IN_U8_DIV255) ? (const unsigned char*)y_any : nullptr;
    if (!y_any || !out || !lmbd || !rho) return fail(ADMM_ERR_INVALID, "NULL tensor pointer");
    if (B < 1 || C < 1) return fail(ADMM_ERR_INVALID, "B and C must be >= 1");
    if (maxit < 0) return fail(ADMM_ERR_INVALID, "maxit must be >= 0");
    if (ksize > 0 && !kern) return fail(ADMM_ERR_INVALID, "kern is NULL but ksize > 0");
    Geometry g;
    if (int e = make_geometry(B * C, H, W, &g)) return e;
    if (int e = check_kernel(ksize, H, W)) return e;
    g.iso = iso ? 1 : 0;
    if (maxit == 0) {                                   // deconv.py:61,103,117: x stays zeros_like(xin) ...
        const size_t img = (size_t)C * H * W;            // ... and ADMMDeconv.forward still applies act(0 + b) (admmdeconv.py:64)
        const size_t stride = ext.out_batch_stride ? (size_t)ext.out_batch_stride : img;
        if (bias || ext.activation != ADMM_ACT_NONE) {
            ProfScope ps(PROF_OTHER, st);
            k_fill_scalar<<<dim3((unsigned)std::min<size_t>((img + 1023) / 1024, 148 * 8), (unsigned)B), 256, 0, st>>>(
                out, bias, ext.activation, img, stride);
            ADMM_CUDA_CHECK(cudaGetLastError());
        } else if (stride == img) {
            ADMM_CUDA_CHECK(cudaMemsetAsync(out, 0, g.field_bytes, st));
        } else {
            ADMM_CUDA_CHECK(cudaMemset2DAsync(out, stride * sizeof(float), 0, img * sizeof(float), (size_t)B, st));
        }
        return 0;
    }
    if (!workspace || ((uintptr_t)workspace & 255)) return fail(ADMM_ERR_WORKSPACE, "workspace is NULL or not 256-byte aligned");
    Workspace ws;
    const size_t need = carve_workspace(g, ksize, maxit, (char*)workspace, &ws);
    if (workspace_bytes < need) return fail(ADMM_ERR_WORKSPACE, "workspace too small");
    const int slots = maxit - 1;
    const size_t map_floats = (size_t)2 * H * W;
    const int ckpt = (saved && ext.ckpt_interval >= 2) ? ext.ckpt_interval : 0;
    if (ckpt && !ckpt_supported(g))
        return fail(ADMM_ERR_UNSUPPORTED, "checkpointed training (admm_ext.ckpt_interval) is not available for iso = 1");
    if (saved) {
        const size_t kept = ckpt ? (size_t)(slots / ckpt) : (size_t)slots;
        const size_t need_saved = kept * 2 * g.field_bytes + (iso ? (size_t)slots * map_floats * sizeof(float) : 0);
        if (((uintptr_t)saved & 255) || saved_bytes < need_saved)
            return fail(ADMM_ERR_WORKSPACE, "saved-state buffer too small or misaligned");
    }
    if (int e = launch_twiddles(ws.twW, ws.twWd, W, st)) return e;
    if (int e = launch_twiddles(ws.twH, ws.twHd, H, st)) return e;
    if (int e = launch_tables(g, ws, kern, ksize, rho, st)) return e;
    if (cols_big_supported(g))
        if (int e = launch_bm_tiled(g, ws.Bm, ws.Bmt, st)) return e;

    if ((ext.yhat_in || ext.yhat_out) && cols_big_supported(g))
        return fail(ADMM_ERR_UNSUPPORTED, "shared spectrum (admm_ext.yhat_*) is not available for this frame size (admm_query_yhat returns 0)");

    // ---- one or a few small planes: the cluster-resident solver runs the whole solve in one launch (cluster_pow2.cu)
    if (!saved && !ext.yhat_in && !ext.yhat_out && cluster_solver_supported(g, iso, false) && cluster_solver_preferred(g)) {
        ClusterArgs ka; std::memset(&ka, 0, sizeof(ka));
        ka.y = y; ka.y8 = y8; ka.out = out; ka.twW = ws.twW; ka.twH = ws.twH; ka.Bm = ws.Bm; ka.Bq = ws.Bq; ka.Mul = ws.Mul; ka.Mq = ws.Mq;
        ka.lmbd = lmbd; ka.rho = rho; ka.bias = bias; ka.act = ext.activation; ka.out_C = C; ka.out_p0 = 0;
        ka.out_bstride = (ext.out_batch_stride == (long long)C * H * W) ? 0 : ext.out_batch_stride;
        ka.P = g.P; ka.maxit = maxit;
        return launch_cluster_solve(g, ka, st);
    }

    // ---- L2-resident plane chunks.  For iso=False the planes are independent (deconv.py:103-115 couples nothing across
    // (b, c)), so the loop nest can be chunk-major: all maxit iterations for a group of planes whose working set (S0, S1,
    // A and the ping-pong state, 7 fields per plane) fits the 126 MB L2, then the next group, re-using the same workspace
    // addresses.  After the first iteration of a chunk both kernels of an iteration find their operands in L2 and HBM
    // sees y, x and (training) the saved state only.
    const size_t fe_all = (size_t)g.P * H * W;          // floats per field, whole batch
    int chunkP = g.P;
    {
        int mb = options().chunk_mb;
        if (mb < 0) mb = kDefaultChunkMB;
        const size_t per_plane = (size_t)H * W * sizeof(float) * 7;
        if (mb > 0 && !iso && maxit > 2) {
            const size_t fit = ((size_t)mb << 20) / per_plane;
            if (fit >= 1 && (int)fit < g.P) {
                // balanced chunks, each at least a wave's worth of work when possible
                const int nchunks = (int)((g.P + fit - 1) / fit);
                chunkP = (g.P + nchunks - 1) / nchunks;
            }
        }
    }
    for (int p0 = 0; p0 < g.P; p0 += chunkP) {
        Geometry gc = g;
        gc.P = std::min(chunkP, g.P - p0);
        gc.field_bytes = (size_t)gc.P * H * W * sizeof(float);
        gc.spec_bytes = (size_t)gc.P * H * g.Wc * sizeof(float2);
        const size_t off_real = (size_t)p0 * H * W, off_spec = (size_t)p0 * H * g.Wc;
        if (int e = solve_planes(gc, g, ws, y ? y + off_real : nullptr, y8 ? y8 + off_real : nullptr, out, p0, C, kern, ksize,
                                 lmbd, rho, bias, maxit, saved ? (float*)saved + off_real : nullptr, fe_all, slots, map_floats,
                                 ext, off_spec, st)) return e;
    }
    return 0;
}

static int dbg_setup(int planes, int H, int W, void* workspace, size_t workspace_bytes, Geometry* g, Workspace* ws,
                     cudaStream_t st) {
    if (int e = make_geometry(planes, H, W, g)) return e;
    if (!workspace || ((uintptr_t)workspace & 255)) return fail(ADMM_ERR_WORKSPACE, "workspace is NULL or misaligned");
    const size_t need = carve_workspace(*g, 0, 1, (char*)workspace, ws);
    if (workspace_bytes < need) return fail(ADMM_ERR_WORKSPACE, "workspace too small");
    if (int e = launch_twiddles(ws->twW, ws->twWd, W, st)) return e;
    if (int e = launch_twiddles(ws->twH, ws->twHd, H, st)) return e;
    return 0;
}

int admm_spectrum_forward(const void* y, int in_dtype, float* yhat, int planes, int H, int W,
                          void* workspace, size_t workspace_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (!y || !yhat) return fail(ADMM_ERR_INVALID, "NULL tensor pointer");
    if (in_dtype != ADMM_IN_F32 && in_dtype != ADMM_IN_U8_DIV255) return fail(ADMM_ERR_INVALID, "unknown in_dtype");
    Geometry g; Workspace ws;
    if (int e = dbg_setup(planes, H, W, workspace, workspace_bytes, &g, &ws, st)) return e;
    if (cols_big_supported(g)) return fail(ADMM_ERR_UNSUPPORTED, "shared spectrum is not available for this frame size");
    RowArgs ra; std::memset(&ra, 0, sizeof(ra));
    ra.tw = ws.twW; ra.spec_out = ws.S1;
    if (in_dtype == ADMM_IN_F32) ra.real_in = (const float*)y; else ra.real_in_u8 = (const unsigned char*)y;
    if (int e = launch_rows(ROWS_R2C, g, ra, st)) return e;
    ColArgs ca; std::memset(&ca, 0, sizeof(ca));
    ca.tw = ws.twH; ca.spec_in = ws.S1; ca.spec_out = (float2*)yhat;
    return launch_cols(COLS_FFT_FWD, g, ca, st);
}

int admm_dbg_rows_r2c(const float* real_in, float* rowspec_out, int planes, int H, int W,
                      void* workspace, size_t workspace_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    Geometry g; Workspace ws;
    if (int e = dbg_setup(planes, H, W, workspace, workspace_bytes, &g, &ws, st)) return e;
    RowArgs ra; std::memset(&ra, 0, sizeof(ra));
    ra.tw = ws.twW; ra.real_in = real_in; ra.spec_out = (float2*)rowspec_out;
    return launch_rows(ROWS_R2C, g, ra, st);
}

int admm_dbg_rows_c2r(const float* rowspec_in, float* real_out, int planes, int H, int W,
                      void* workspace, size_t workspace_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    Geometry g; Workspace ws;
    if (int e = dbg_setup(planes, H, W, workspace, workspace_bytes, &g, &ws, st)) return e;
    RowArgs ra; std::memset(&ra, 0, sizeof(ra));
    ra.tw = ws.twW; ra.spec_in = (const float2*)rowspec_in; ra.real_out = real_out;
    return launch_rows(ROWS_C2R, g, ra, st);
}

int admm_dbg_cols_fft(const float* rowspec_in, float* rowspec_out, int planes, int H, int W, int inverse,
                      void* workspace, size_t workspace_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    Geometry g; Workspace ws;
    if (int e = dbg_setup(planes, H, W, workspace, workspace_bytes, &g, &ws, st)) return e;
    ColArgs ca; std::memset(&ca, 0, sizeof(ca));
    ca.tw = ws.twH; ca.spec_in = (const float2*)rowspec_in; ca.spec_out = (float2*)rowspec_out;
    return launch_cols(inverse ? COLS_FFT_INV : COLS_FFT_FWD, g, ca, st);
}

}  // extern "C"
