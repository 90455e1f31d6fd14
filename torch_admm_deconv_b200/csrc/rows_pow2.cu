// rows_pow2.cu -- specialised row-pass kernel of the ADMM iteration for W in {128, 256, 512} (sm_100a).
//
//   packed row spectrum of x_k  --C2R-->  x_k  --prox / dual / divergence-->  v_{k+1}  --R2C-->  packed spectrum
//   (deconv.py:106 irfftn rows, :108-115 Dx/Dy/soft_thresh/dual update, :104 Dx_t/Dy_t + rfftn rows)
//
// One CTA (256 threads) owns a band of Rb image rows of one plane plus one halo row above and below.
// Two image rows share one complex FFT (z = row_a + i row_b); TPS = W/16 consecutive threads of one warp
// own one row pair and keep 16 complex points each in registers, so the FFT passes need only __syncwarp.
// The first inverse pass and the last forward pass give every thread the two butterflies j and W/8 - j:
// the Hermitian merge (two packed half spectra -> full spectrum of z) and split (back) then happen
// entirely in registers and the global accesses are 256-byte coalesced runs, 8 bytes per lane.
// The spatial step marches down the band: a thread owns two adjacent columns, carries x and w_y of the
// previous row in registers and loads the pre-clamp state two row pairs ahead of its use.
#include "rows_pow2_body.cuh"

namespace admm {

// the marching modes: ROWS_FULL, ROWS_FULL_U, ROWS_ADJ and their threshold-map variants (one halo row above and below)
template <int MODE> constexpr bool kRowsIter = (MODE == ROWS_FULL || MODE == ROWS_FULL_U || MODE == ROWS_ADJ ||
                                                MODE == ROWS_FULL_MAP || MODE == ROWS_ADJ_MAP);
// CTAs per SM the kernel is built for: 4, the adjoint ROWS_ADJ_OCC; the map modes carry the map's values on top of the
// state and are built for 3 (no spills)
template <int MODE> constexpr int kRowsOcc = (MODE == ROWS_ADJ) ? ROWS_ADJ_OCC : (MODE == ROWS_FULL_MAP || MODE == ROWS_ADJ_MAP) ? 3 : 4;

template <int W, int MODE, int HT>
__global__ void __launch_bounds__(256, kRowsOcc<MODE>)
k_rows_pow2(RowArgs a, int H, int nbands, int pdl) {
    extern __shared__ float2 smem[];
    rows_pow2_body<W, MODE, false, HT>(a, H, nbands, pdl, blockIdx.x, smem);
}


// HT = W for the iteration kernels (forward and backward) on square planes, else 0 (run-time height)
template <int W, int MODE, int HT>
static int launch_rows_pow2_h(const Geometry& g, const RowArgs& a, cudaStream_t st) {
    using S = RowSmem<W>;
    constexpr int rmax = kRowsIter<MODE> ? S::RMAX : 2 * S::NPAIR;
    int nbands = (g.H + rmax - 1) / rmax;
    // few planes (latency-bound problems such as a single image): cut thinner bands so that every SM gets a CTA
    const int want = (2 * 148 + g.P - 1) / g.P;
    if (nbands < want) nbands = std::min(g.H / 2, want);
    if (options().rows_per_band >= 0) {
        // wave balance (rows_per_band = -1 switches it off): with a few hundred to a few thousand CTAs the last, partly
        // filled wave costs as much as a full one; thinner bands (more CTAs, one more halo pair each in the marching
        // modes) can fill it.  Model: waves x (rows per band + halo).
        constexpr int halo = kRowsIter<MODE> ? 2 : 0;
        const long slots = 148L * kRowsOcc<MODE>;
        auto cost = [&](int nb) { return ((long)nb * g.P + slots - 1) / slots * ((g.H + nb - 1) / nb + halo); };
        int best = nbands;
        for (int nb = nbands + 1; nb <= std::min(g.H / 2, 2 * nbands); ++nb)
            if (cost(nb) < cost(best)) best = nb;
        if (cost(best) * 20 <= cost(nbands) * 19) nbands = best;          // only for a gain of 5 % or more
    }
    if (options().rows_per_band > 0)                       // tuning knob: thinner bands than the kernel's maximum
        nbands = std::min(g.H / 2, std::max(nbands, (g.H + options().rows_per_band - 1) / options().rows_per_band));
    // the opt-in shared-memory limit is a per-device function attribute: remember which devices have it
    static std::atomic<bool> attr_set_dev[64];
    int dev_id = 0;
    cudaGetDevice(&dev_id);
    std::atomic<bool>& attr_set = attr_set_dev[dev_id & 63];
    if (!attr_set) {
        ADMM_CUDA_CHECK(cudaFuncSetAttribute(k_rows_pow2<W, MODE, HT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::bytes));
        attr_set = true;
    }
    ProfScope ps((MODE == ROWS_FULL || MODE == ROWS_FULL_U || MODE == ROWS_FULL_MAP) ? PROF_ROWS : PROF_OTHER, st);
    // programmatic dependent launch pays off when a kernel is a wave or two (launch / drain latency dominates)
    const size_t nctas = (size_t)nbands * g.P;
    if (options().use_pdl && nctas <= 148 * 8) {
        ADMM_CUDA_CHECK(launch_pdl(k_rows_pow2<W, MODE, HT>, dim3((unsigned)nctas), dim3(256), S::bytes, st, a, g.H, nbands, 1));
    } else {
        k_rows_pow2<W, MODE, HT><<<(unsigned)nctas, 256, S::bytes, st>>>(a, g.H, nbands, 0);
    }
    ADMM_CUDA_CHECK(cudaGetLastError());
    return 0;
}

template <int W, int MODE>
static int launch_rows_pow2_m(const Geometry& g, const RowArgs& a, cudaStream_t st) {
    constexpr bool iter = kRowsIter<MODE>;
    if (iter && g.H == W) return launch_rows_pow2_h<W, MODE, (iter ? W : 0)>(g, a, st);
    return launch_rows_pow2_h<W, MODE, 0>(g, a, st);
}

template <int W>
static int launch_rows_pow2_t(RowMode mode, const Geometry& g, const RowArgs& a, cudaStream_t st) {
    switch (mode) {
        case ROWS_FULL: return launch_rows_pow2_m<W, ROWS_FULL>(g, a, st);
        case ROWS_R2C: return launch_rows_pow2_m<W, ROWS_R2C>(g, a, st);
        case ROWS_C2R: return launch_rows_pow2_m<W, ROWS_C2R>(g, a, st);
        case ROWS_ADJ: return launch_rows_pow2_m<W, ROWS_ADJ>(g, a, st);
        case ROWS_FULL_U: return launch_rows_pow2_m<W, ROWS_FULL_U>(g, a, st);
        case ROWS_FULL_MAP: return launch_rows_pow2_m<W, ROWS_FULL_MAP>(g, a, st);
        case ROWS_ADJ_MAP: return launch_rows_pow2_m<W, ROWS_ADJ_MAP>(g, a, st);
    }
    return fail(4, "rows_pow2: bad mode");
}

bool rows_pow2_supported(const Geometry& g) {
    if (options().force_generic) return false;
    if (g.H & 1) return false;
    return g.W == 128 || g.W == 256 || g.W == 512;
}

int launch_rows_pow2(RowMode mode, const Geometry& g, const RowArgs& a, cudaStream_t st) {
    switch (g.W) {
        case 128: return launch_rows_pow2_t<128>(mode, g, a, st);
        case 256: return launch_rows_pow2_t<256>(mode, g, a, st);
        case 512: return launch_rows_pow2_t<512>(mode, g, a, st);
    }
    return fail(4, "rows_pow2: unsupported width");
}

}  // namespace admm
