// K1 (general form): one CTA per window, the whole transform resident in shared memory.
//
//   load n_samples reals -> exact median (block radix select) -> centre -> bit-reversed scatter with zero padding
//   -> log2(N) radix-2 DIT stages on the reference's dataflow graph -> bin 0 := 0 -> coalesced store of N bins.
//
// Reference behaviour reproduced (paths relative to the reference checkout):
//   metrics/fft_iterativa.py:5-11 (median), :13-22 (pad after centring), :24-36 (bit reversal),
//   :38-70 (butterflies, twiddle recurrence -> host-built table), :85 (DC bin zeroed).
// The fp64 instantiation uses individually rounded multiplies/adds (no FMA) in the reference's operation order, so
// the spectrum is bit-identical to the reference.  The fp32 instantiation of this general kernel serves the sizes
// the specialised fp32 kernels (fft_f32_fast.cu) do not cover.
#include <math_constants.h>

#include <algorithm>

#include "common.cuh"
#include "fft_smem.cuh"

namespace {

// One CTA per window.  nv (optional): per-window sample counts of a ragged batch; list (optional): list[0] = count,
// list[1..] = the windows to process (grid-stride), used for the ragged windows the specialised kernels skip.
template <typename T, bool FAITHFUL, bool COMPLEX_IN>
__global__ void __launch_bounds__(kThreads)
fft_smem_kernel(const T *__restrict__ samples, int n_samples, int64_t ld, int N, int logN,
                const typename vec2<T>::type *__restrict__ tw, typename vec2<T>::type *__restrict__ spec, int center,
                const int *__restrict__ nv, const int *__restrict__ list) {
    if (!list) {
        const int64_t win = blockIdx.x;
        fft_smem_window<T, FAITHFUL, COMPLEX_IN>(win, samples, nv ? nv[win] : n_samples, ld, N, logN, tw, spec, center,
                                                 win);
        return;
    }
    for (int it = blockIdx.x; it < list[0]; it += gridDim.x) {
        const int64_t win = list[1 + it];
        fft_smem_window<T, FAITHFUL, COMPLEX_IN>(win, samples, nv[win], ld, N, logN, tw, spec, center, win);
        __syncthreads();
    }
}

// remove_dc_component on one list (metrics/fft_iterativa.py:5-11): out[i] = in[i] - median(in)
__global__ void __launch_bounds__(kThreads) center_kernel(const double *__restrict__ in, int n, double *__restrict__ out,
                                                          uint64_t *keys) {
    __shared__ unsigned hist[256];
    __shared__ unsigned bcast[2];
    double med = block_median<double, uint64_t>(in, keys, n, hist, bcast);
    for (int i = threadIdx.x; i < n; i += kThreads) out[i] = sub_rn(in[i], med);
}

template <typename T>
size_t smem_bytes_for(int64_t N, bool complex_in) {
    // transform (+ raw samples for real input)
    return complex_in ? (size_t)N * 2 * sizeof(T) : (size_t)N * 3 * sizeof(T);
}

}  // namespace

template <typename T>
int64_t fft_smem_max_n(apda_ctx *ctx) {
    int64_t n = 2;
    while (smem_bytes_for<T>(n * 2, false) + 2048 <= (size_t)ctx->smem_optin) n *= 2;
    return n;
}
template int64_t fft_smem_max_n<double>(apda_ctx *);
template int64_t fft_smem_max_n<float>(apda_ctx *);

template <typename T>
int launch_fft_smem(apda_ctx *ctx, cudaStream_t st, const T *d_samples, int64_t n_samples, int64_t ld, int64_t batch,
                    int64_t N, int flags, T *d_spec, bool complex_input, const int *d_nv, const int *d_list) {
    using V2 = typename vec2<T>::type;
    TwiddleTables tw;
    APDA_TRY(apda_get_twiddles(ctx, N, &tw));
    const V2 *twp = sizeof(T) == 8 ? reinterpret_cast<const V2 *>(tw.d64) : reinterpret_cast<const V2 *>(tw.d32);
    size_t smem = smem_bytes_for<T>(N, complex_input);
    if (smem + 2048 > (size_t)ctx->smem_optin) {
        apda_set_error("fft_smem: N=%lld does not fit shared memory", (long long)N);
        return APDA_ERR_UNSUPPORTED;
    }
    constexpr bool kFaithful = sizeof(T) == 8;
    auto kern = complex_input ? fft_smem_kernel<T, kFaithful, true> : fft_smem_kernel<T, kFaithful, false>;
    APDA_FUNC_SMEM(ctx, kern, smem);
    int logN = ilog2_i64(N);
    // grid.x is limited to 2^31-1 windows per launch, far above any batch that fits HBM
    const unsigned grid = d_list ? (unsigned)std::min<int64_t>(batch, 2 * (int64_t)ctx->sm_count) : (unsigned)batch;
    kern<<<grid, kThreads, smem, st>>>(d_samples, (int)n_samples, ld, (int)N, logN, twp, reinterpret_cast<V2 *>(d_spec),
                                       flags, d_nv, d_list);
    ctx->launches++;
    APDA_CUDA(cudaGetLastError());
    return APDA_OK;
}
template int launch_fft_smem<double>(apda_ctx *, cudaStream_t, const double *, int64_t, int64_t, int64_t, int64_t, int,
                                     double *, bool, const int *, const int *);
template int launch_fft_smem<float>(apda_ctx *, cudaStream_t, const float *, int64_t, int64_t, int64_t, int64_t, int,
                                    float *, bool, const int *, const int *);

int launch_center_f64(apda_ctx *ctx, cudaStream_t st, const double *d_in, int64_t n, double *d_out) {
    // keys live in global scratch right behind the output (caller reserves 2*n doubles at d_out)
    center_kernel<<<1, kThreads, 0, st>>>(d_in, (int)n, d_out, reinterpret_cast<uint64_t *>(d_out + n));
    ctx->launches++;
    APDA_CUDA(cudaGetLastError());
    return APDA_OK;
}
