// K3 (general form): one CTA per window.  magnitude of the half spectrum -> mean / sample sigma -> threshold ->
// strict local maxima -> flexible (prominence) or rigid (resolution) picker -> fixed-size peak record.
// The spectrum is read once from HBM; magnitudes live in shared memory (or in a global workspace for N > 2^14/2^15).
//
// Reference behaviour reproduced (paths relative to the reference checkout):
//   utils/get_peak_prominence.py:149-226 get_top_peaks_prominence (+ :32-54 calculate_prominence,
//       :89-112 calculate_half_power_width_prominenceBased)
//   utils/get_peak_resolution.py:80-128 get_top_peaks_resolution (+ :30-44 width_half_magnitude, :48-62 resolution)
// Every comparison the reference makes in fp64 is made here with individually rounded fp64 operations in the same
// order; round(x, 4) is emulated exactly (round_dec4).  fp32 instantiations keep magnitudes/prominences in fp32 and
// evaluate the statistics and the damping / exclusion / zeroing arithmetic in fp64.
#include <math_constants.h>

#include <algorithm>

#include "common.cuh"
#include "peaks_common.cuh"
#include "peaks_window.cuh"

namespace {

// One CTA per window; with a repair list (list[0] = count, list[1..] = window ids, written by the fp32 fast kernel) the
// CTAs stride over the listed windows instead.
template <typename T, bool SMEM, bool FLEX>
__global__ void __launch_bounds__(SMEM ? 256 : 1024) peaks_kernel(const typename vec2<T>::type *__restrict__ spec, int64_t n, int half, int64_t batch,
                             double fs_all, const double *__restrict__ d_fs, int k, int rec_cap,
                             unsigned char *__restrict__ recs, unsigned char *__restrict__ ws,
                             const int *__restrict__ list) {
    for (int64_t it = blockIdx.x;; it += gridDim.x) {
        int64_t win = it;
        if (list) {
            if (it >= list[0]) break;
            win = list[1 + it];
        } else if (it >= batch) {
            break;
        }
        if (FLEX) peaks_prominence_window<T, SMEM>(win, spec, n, half, fs_all, d_fs, k, rec_cap, recs, ws, win);
        else peaks_resolution_window<T, SMEM>(win, spec, n, half, fs_all, d_fs, k, rec_cap, recs, ws, win);
        __syncthreads();
    }
}

// ---- module-public helper functions of the reference, on a caller-supplied magnitude list ---------------------------
// out[0] = calculate_prominence(mags, idx); out[1] = half-power bin count for prominence prom_in; out[2] = width_half_magnitude
__global__ void mag_helpers_kernel(const double *__restrict__ mags, int n, int idx, double prom_in, double *out) {
    double prom = warp_prominence<double>(mags, n, idx);
    if (threadIdx.x == 0) {
        out[0] = prom;
        out[1] = (double)half_power_bins<double>(mags, n, prom_in, idx);
        out[2] = (double)half_height_bins<double>(mags, n, idx);
    }
}

}  // namespace

template <typename T>
size_t peaks_mag_workspace_bytes(apda_ctx *ctx, int64_t n, int64_t batch) {
    if (peaks_large_supports(n) && !ctx->generic_only) return peaks_large_workspace_bytes<T>(n, batch);
    Layout lay = make_layout<T>((int)(n / 2));
    if (lay.bytes + 4096 <= (size_t)ctx->smem_optin) return 0;
    return lay.bytes * (size_t)batch;
}
template size_t peaks_mag_workspace_bytes<double>(apda_ctx *, int64_t, int64_t);
template size_t peaks_mag_workspace_bytes<float>(apda_ctx *, int64_t, int64_t);

template <typename T>
static int launch_peaks_general(apda_ctx *ctx, cudaStream_t st, const T *d_spec, int64_t n, int64_t batch, double fs,
                                const double *d_fs, int k, int rec_cap, int flexible, void *d_rec, void *d_mag_ws,
                                const int *list) {
    using V2 = typename vec2<T>::type;
    const int half = (int)(n / 2);
    const Layout lay = make_layout<T>(half);
    const bool in_smem = lay.bytes + 4096 <= (size_t)ctx->smem_optin;
    const V2 *spec = reinterpret_cast<const V2 *>(d_spec);
    unsigned char *recs = reinterpret_cast<unsigned char *>(d_rec);
    unsigned char *ws = reinterpret_cast<unsigned char *>(d_mag_ws);
    const unsigned grid = list ? (unsigned)std::min<int64_t>(batch, 2 * (int64_t)ctx->sm_count) : (unsigned)batch;
    if (in_smem) {
        auto kern = flexible ? peaks_kernel<T, true, true> : peaks_kernel<T, true, false>;
        APDA_FUNC_SMEM(ctx, kern, lay.bytes);
        kern<<<grid, 256, lay.bytes, st>>>(spec, n, half, batch, fs, d_fs, k, rec_cap, recs, nullptr, list);
    } else {
        if (!ws) {
            apda_set_error("launch_peaks: magnitude workspace missing for n=%lld", (long long)n);
            return APDA_ERR_INVALID;
        }
        auto kern = flexible ? peaks_kernel<T, false, true> : peaks_kernel<T, false, false>;
        kern<<<grid, 1024, 0, st>>>(spec, n, half, batch, fs, d_fs, k, rec_cap, recs, ws, list);
    }
    ctx->launches++;
    APDA_CUDA(cudaGetLastError());
    return APDA_OK;
}

template <typename T>
int launch_peaks_general_listed(apda_ctx *ctx, cudaStream_t st, const T *d_spec, int64_t n, int64_t batch, double fs,
                                const double *d_fs, int k, int rec_cap, int flexible, void *d_rec, const int *list) {
    return launch_peaks_general<T>(ctx, st, d_spec, n, batch, fs, d_fs, k, rec_cap, flexible, d_rec, nullptr, list);
}
template int launch_peaks_general_listed<float>(apda_ctx *, cudaStream_t, const float *, int64_t, int64_t, double,
                                                const double *, int, int, int, void *, const int *);
template int launch_peaks_general_listed<double>(apda_ctx *, cudaStream_t, const double *, int64_t, int64_t, double,
                                                 const double *, int, int, int, void *, const int *);

template <typename T>
int launch_peaks(apda_ctx *ctx, cudaStream_t st, const T *d_spec, int64_t n, int64_t batch, double fs,
                 const double *d_fs, int k, int rec_cap, int flexible, void *d_rec, void *d_mag_ws) {
    using V2 = typename vec2<T>::type;
    if (sizeof(T) == 4 && !ctx->generic_only && peaks_f32_fast_supports(n, k, rec_cap))
        return launch_peaks_f32_fast(ctx, st, reinterpret_cast<const float *>(d_spec), n, batch, fs, d_fs, k, flexible,
                                     d_rec);
    if (sizeof(T) == 8 && !ctx->generic_only && peaks_f64_fast_supports(n, k, rec_cap))
        return launch_peaks_f64_fast(ctx, st, reinterpret_cast<const double *>(d_spec), n, batch, fs, d_fs, k, flexible,
                                     d_rec);
    if (peaks_large_supports(n) && !ctx->generic_only && d_mag_ws)
        return launch_peaks_large<T>(ctx, st, d_spec, n, batch, fs, d_fs, k, rec_cap, flexible, d_rec, d_mag_ws);
    return launch_peaks_general<T>(ctx, st, d_spec, n, batch, fs, d_fs, k, rec_cap, flexible, d_rec, d_mag_ws, nullptr);
}
template int launch_peaks<double>(apda_ctx *, cudaStream_t, const double *, int64_t, int64_t, double, const double *, int,
                                  int, int, void *, void *);
template int launch_peaks<float>(apda_ctx *, cudaStream_t, const float *, int64_t, int64_t, double, const double *, int,
                                 int, int, void *, void *);

int launch_mag_helpers_f64(apda_ctx *ctx, cudaStream_t st, const double *d_mags, int64_t n, int64_t idx, double prom_in,
                           double *d_out3) {
    mag_helpers_kernel<<<1, 32, 0, st>>>(d_mags, (int)n, (int)idx, prom_in, d_out3);
    ctx->launches++;
    APDA_CUDA(cudaGetLastError());
    return APDA_OK;
}
