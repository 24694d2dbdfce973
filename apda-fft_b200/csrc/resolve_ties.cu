// fp32 tie resolver (apda_resolve_fp32_ties_*): the windows whose record status is exactly APDA_STATUS_FP32_TIE are
// re-run through the fp64 bit-faithful path on their own fp32 samples, widened to double at the load, and their records
// replaced.  Every other byte of the record table is left alone.
//
//   tie_list_kernel      status words of the records -> device list of the tied windows (list[0] = count)
//   resolve_ties_kernel  persistent CTAs walk the list: K1-general (fp64, faithful) into a spectrum slot owned by the CTA,
//                        then K3-general (fp64) from that slot into the window's record, with the window's own fs
//
// Widening is exact, so the median, the transform and the picker see exactly the fp64 path's inputs: the record is the one
// apda_analyze_f64_dev (apda_analyze_ragged_f64_dev with per-window counts) writes for the widened samples.
#include <algorithm>

#include "common.cuh"
#include "fft_smem.cuh"
#include "peaks_window.cuh"

namespace {

__global__ void tie_list_kernel(const unsigned char *__restrict__ recs, int64_t rec_bytes, int64_t batch,
                                int *__restrict__ list) {
    for (int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < batch; w += (int64_t)gridDim.x * blockDim.x)
        if (reinterpret_cast<const int *>(recs + w * rec_bytes)[1] == APDA_STATUS_FP32_TIE)
            list[1 + atomicAdd(&list[0], 1)] = (int)w;
}

// slots: gridDim.x spectra of N bins, one per CTA.  nv (optional): per-window sample counts of a ragged batch.
template <bool FLEX>
__global__ void __launch_bounds__(kThreads)
resolve_ties_kernel(const float *__restrict__ samples, const int *__restrict__ nv, int n_samples, int64_t ld, int N,
                    int logN, const double2 *__restrict__ tw, double2 *slots, int center, double fs_all,
                    const double *__restrict__ d_fs, int k, int rec_cap, unsigned char *__restrict__ recs,
                    const int *__restrict__ list) {
    const int64_t slot = blockIdx.x;
    for (int it = blockIdx.x; it < list[0]; it += gridDim.x) {
        const int64_t win = list[1 + it];
        const int n = nv ? nv[win] : n_samples;
        fft_smem_window<double, true, false, float>(win, samples, n, ld, N, logN, tw, slots, center, slot);
        __syncthreads();  // the slot is complete and visible to the whole CTA; the shared memory is the picker's now
        if (FLEX) peaks_prominence_window<double, true>(win, slots, N, N / 2, fs_all, d_fs, k, rec_cap, recs, nullptr, slot);
        else peaks_resolution_window<double, true>(win, slots, N, N / 2, fs_all, d_fs, k, rec_cap, recs, nullptr, slot);
        if (nv && threadIdx.x == 0 && n != N) {  // the status bits ragged_status_kernel (api.cu) sets on the fp64 path
            int64_t p = 1;
            while (p < n) p <<= 1;
            int *hdr = reinterpret_cast<int *>(recs + win * APDA_REC_BYTES(rec_cap));
            if (n <= 0) {
                hdr[0] = 0;
                hdr[1] |= APDA_STATUS_EMPTY;
            } else if (p != N) {
                hdr[1] |= APDA_STATUS_OTHER_LENGTH;
            }
        }
        __syncthreads();
    }
}

unsigned resolve_grid(apda_ctx *ctx, int64_t batch) { return (unsigned)std::min<int64_t>(batch, 2 * (int64_t)ctx->sm_count); }

}  // namespace

size_t resolve_ties_slot_bytes(apda_ctx *ctx, int64_t N, int64_t batch) {
    return (size_t)resolve_grid(ctx, batch) * (size_t)N * sizeof(double2);
}

int launch_resolve_ties(apda_ctx *ctx, cudaStream_t st, const float *d_samples, const int *d_nv, int64_t n_samples,
                        int64_t ld, int64_t batch, int64_t N, int center, int flexible, double fs, const double *d_fs,
                        int k, int rec_cap, void *d_rec, int *d_list, void *d_slots) {
    TwiddleTables tw;
    APDA_TRY(apda_get_twiddles(ctx, N, &tw));
    unsigned char *recs = reinterpret_cast<unsigned char *>(d_rec);
    const unsigned scan = (unsigned)std::min<int64_t>((batch + 255) / 256, 32 * (int64_t)ctx->sm_count);
    tie_list_kernel<<<scan, 256, 0, st>>>(recs, APDA_REC_BYTES(rec_cap), batch, d_list);
    ctx->launches++;
    APDA_CUDA(cudaGetLastError());
    const size_t smem = std::max<size_t>((size_t)N * 3 * sizeof(double), make_layout<double>((int)(N / 2)).bytes);
    auto kern = flexible ? resolve_ties_kernel<true> : resolve_ties_kernel<false>;
    APDA_FUNC_SMEM(ctx, kern, smem);
    kern<<<resolve_grid(ctx, batch), kThreads, smem, st>>>(d_samples, d_nv, (int)n_samples, ld, (int)N, ilog2_i64(N), tw.d64,
                                                           reinterpret_cast<double2 *>(d_slots), center, fs, d_fs, k, rec_cap,
                                                           recs, d_list);
    ctx->launches++;
    APDA_CUDA(cudaGetLastError());
    return APDA_OK;
}
