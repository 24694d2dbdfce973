// C ABI of libapda_b200.so (declared in include/apda_b200.h): context, twiddle tables, dispatch, host pipelines.
#include <errno.h>
#include <fcntl.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "common.cuh"

// ---------------------------------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

void apda_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
int apda_cuda_fail(cudaError_t e, const char *what) {
    apda_set_error("CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
    return APDA_ERR_CUDA;
}
extern "C" const char *apda_last_error(void) { return g_err; }
extern "C" int apda_version(void) { return 103; }

int apda_reserve(void **buf, size_t *have, size_t need) {
    if (need <= *have) return APDA_OK;
    if (*buf) APDA_CUDA(cudaFree(*buf));
    *buf = nullptr;
    *have = 0;
    size_t want = need + need / 8;
    cudaError_t e = cudaMalloc(buf, want);
    if (e != cudaSuccess) {
        want = need;
        e = cudaMalloc(buf, want);
    }
    if (e != cudaSuccess) {
        apda_set_error("cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
        (void)cudaGetLastError();
        return APDA_ERR_NOMEM;
    }
    *have = want;
    return APDA_OK;
}

int apda_pdl_mask() {
    static const int mask = [] {
        const char *e = getenv("APDA_PDL");
        return e && e[0] ? atoi(e) : 15;
    }();
    return mask;
}

int apda_func_smem(const void *kernel, int device, size_t bytes) {
    static std::mutex mu;
    static std::map<std::pair<int, const void *>, size_t> done;
    std::lock_guard<std::mutex> lock(mu);
    size_t &have = done[std::make_pair(device, kernel)];
    if (bytes <= have) return APDA_OK;
    APDA_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    have = bytes;
    return APDA_OK;
}

static int stream_list(cudaStream_t st, int **buf, size_t *have, int64_t batch, int **out) {
    const size_t need = ((size_t)batch + 1) * sizeof(int);
    if (need > *have) {
        APDA_CUDA(cudaStreamSynchronize(st));  // the old list may still be read by kernels queued on this stream
        APDA_TRY(apda_reserve((void **)buf, have, need));
    }
    APDA_CUDA(cudaMemsetAsync(*buf, 0, sizeof(int), st));
    *out = *buf;
    return APDA_OK;
}
int apda_repair_list(apda_ctx *ctx, cudaStream_t st, int64_t batch, int **out) {
    auto &l = ctx->stream_lists[st];
    return stream_list(st, &l.repair, &l.repair_bytes, batch, out);
}
int apda_ragged_list(apda_ctx *ctx, cudaStream_t st, int64_t batch, int **out) {
    auto &l = ctx->stream_lists[st];
    return stream_list(st, &l.ragged, &l.ragged_bytes, batch, out);
}
int apda_tie_list(apda_ctx *ctx, cudaStream_t st, int64_t batch, int **out) {
    auto &l = ctx->stream_lists[st];
    return stream_list(st, &l.ties, &l.ties_bytes, batch, out);
}

// ---------------------------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------------------------
extern "C" int apda_ctx_create(int device, apda_ctx **out) {
    if (!out) {
        apda_set_error("apda_ctx_create: out is NULL");
        return APDA_ERR_INVALID;
    }
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        apda_set_error("no CUDA device available (%s); libapda_b200 has no CPU fallback",
                       e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        (void)cudaGetLastError();
        return APDA_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= count) {
        apda_set_error("device %d out of range [0, %d)", device, count);
        return APDA_ERR_INVALID;
    }
    cudaDeviceProp prop;
    APDA_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        apda_set_error("device %d (%s) is compute capability %d.%d; this library is built for sm_100a only", device,
                       prop.name, prop.major, prop.minor);
        return APDA_ERR_NO_DEVICE;
    }
    APDA_CUDA(cudaSetDevice(device));
    apda_ctx *ctx = new apda_ctx();
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = (int)prop.sharedMemPerBlockOptin;
    APDA_CUDA(cudaDeviceGetAttribute(&ctx->clock_khz, cudaDevAttrClockRate, device));
    APDA_CUDA(cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking));
    ctx->stream = ctx->own_stream;
    for (int i = 0; i < 2; ++i) {
        APDA_CUDA(cudaStreamCreateWithFlags(&ctx->pipe[i], cudaStreamNonBlocking));
    }
    *out = ctx;
    return APDA_OK;
}

extern "C" int apda_ctx_destroy(apda_ctx *ctx) {
    if (!ctx) return APDA_OK;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    for (auto &kv : ctx->twiddles) {
        cudaFree(kv.second.d64);
        cudaFree(kv.second.d32);
    }
    fft_f32_fast_release(ctx);
    cudaFree(ctx->ws);
    cudaFree(ctx->ws_small);
    for (auto &kv : ctx->stream_lists) {
        cudaFree(kv.second.repair);
        cudaFree(kv.second.ragged);
        cudaFree(kv.second.ties);
        cudaFree(kv.second.jsonl);
    }
    for (auto &kv : ctx->stream_scratch) cudaFree(kv.second.first);
    for (int i = 0; i < 2; ++i) {
        cudaFree(ctx->ws_pipe[i]);
        cudaFreeHost(ctx->log_stage[i]);
        if (ctx->pipe[i]) cudaStreamDestroy(ctx->pipe[i]);
    }
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
    return APDA_OK;
}

extern "C" int apda_ctx_set_stream(apda_ctx *ctx, void *cuda_stream) {
    if (!ctx) return APDA_ERR_INVALID;
    ctx->stream = (cudaStream_t)cuda_stream;
    return APDA_OK;
}

extern "C" int apda_ctx_reset_stream(apda_ctx *ctx) {
    if (!ctx) return APDA_ERR_INVALID;
    ctx->stream = ctx->own_stream;
    return APDA_OK;
}

extern "C" int apda_ctx_set_generic_only(apda_ctx *ctx, int on) {
    if (!ctx) return APDA_ERR_INVALID;
    ctx->generic_only = on ? 1 : 0;
    return APDA_OK;
}

extern "C" int apda_sync(apda_ctx *ctx) {
    if (!ctx) return APDA_ERR_INVALID;
    APDA_CUDA(cudaStreamSynchronize(ctx->stream));
    return APDA_OK;
}

extern "C" int64_t apda_launch_count(apda_ctx *ctx) { return ctx ? ctx->launches : 0; }

// ---------------------------------------------------------------------------------------------------------------
// twiddle tables: the reference's recurrence (metrics/fft_iterativa.py:53,57,68) evaluated on the host with the same
// libm cos/sin CPython's cmath.exp calls and separately rounded complex products, uploaded once per N.
// ---------------------------------------------------------------------------------------------------------------
int apda_get_twiddles(apda_ctx *ctx, int64_t N, TwiddleTables *out) {
    auto it = ctx->twiddles.find(N);
    if (it != ctx->twiddles.end()) {
        *out = it->second;
        return APDA_OK;
    }
    const size_t cnt = (size_t)std::max<int64_t>(N - 1, 1);
    std::vector<double2> h(cnt);
    std::vector<float2> hf(cnt);
    h[0] = make_double2(1.0, 0.0);
    const double pi = 3.141592653589793;  // cmath.pi
    for (int64_t half = 1; half < N; half <<= 1) {
        const double theta = (-2.0 * pi) / (double)(2 * half);
        const volatile double cr = cos(theta), ci = sin(theta);
        double wr = 1.0, wi = 0.0;
        double2 *t = h.data() + (half - 1);
        for (int64_t j = 0; j < half; ++j) {
            t[j] = make_double2(wr, wi);
            // volatile temporaries: every product and sum rounds on its own, as Python's complex product does
            volatile double a = wr * cr, b = wi * ci, c = wr * ci, d = wi * cr;
            double nr = a - b, ni = c + d;
            wr = nr;
            wi = ni;
        }
    }
    for (size_t i = 0; i < cnt; ++i) hf[i] = make_float2((float)h[i].x, (float)h[i].y);
    TwiddleTables tw;
    APDA_CUDA(cudaMalloc(&tw.d64, cnt * sizeof(double2)));
    APDA_CUDA(cudaMalloc(&tw.d32, cnt * sizeof(float2)));
    APDA_CUDA(cudaMemcpy(tw.d64, h.data(), cnt * sizeof(double2), cudaMemcpyHostToDevice));
    APDA_CUDA(cudaMemcpy(tw.d32, hf.data(), cnt * sizeof(float2), cudaMemcpyHostToDevice));
    ctx->twiddles[N] = tw;
    *out = tw;
    return APDA_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// argument checks and dispatch
// ---------------------------------------------------------------------------------------------------------------
static int check_fft_args(apda_ctx *ctx, const void *in, int64_t n_samples, int64_t ld, int64_t batch, int64_t N,
                          int flags, const void *out) {
    if (!ctx || !in || !out) {
        apda_set_error("fft: NULL argument");
        return APDA_ERR_INVALID;
    }
    if (batch < 0 || batch > 0x7fffffff) {
        apda_set_error("fft: batch %lld out of range", (long long)batch);
        return APDA_ERR_INVALID;
    }
    if (!is_pow2_i64(N) || N < 2 || N > (int64_t(1) << 30)) {
        apda_set_error("fft: N=%lld must be a power of two in [2, 2^30]", (long long)N);
        return APDA_ERR_INVALID;
    }
    if (n_samples < 1 || n_samples > N || ld < n_samples) {
        apda_set_error("fft: need 1 <= n_samples (%lld) <= N (%lld) and ld (%lld) >= n_samples", (long long)n_samples,
                       (long long)N, (long long)ld);
        return APDA_ERR_INVALID;
    }
    if (flags != APDA_CENTER_MEDIAN && flags != APDA_CENTER_MEAN && flags != APDA_CENTER_NONE) {
        apda_set_error("fft: unknown flags %d", flags);
        return APDA_ERR_INVALID;
    }
    if (flags == APDA_CENTER_MEAN && n_samples != N) {
        apda_set_error("fft: APDA_CENTER_MEAN is only legal when n_samples == N (padding needs the exact median)");
        return APDA_ERR_INVALID;
    }
    return APDA_OK;
}

static int check_peaks_args(apda_ctx *ctx, const void *spec, int64_t n, int64_t batch, int k, int rec_cap,
                            const void *rec) {
    if (!ctx || !spec || !rec) {
        apda_set_error("peaks: NULL argument");
        return APDA_ERR_INVALID;
    }
    if (batch < 0 || batch > 0x7fffffff || n < 0 || n > (int64_t(1) << 31)) {
        apda_set_error("peaks: batch/n out of range");
        return APDA_ERR_INVALID;
    }
    if (n / 2 < 1) {
        apda_set_error("mean requires at least one data point");
        return APDA_ERR_STATS_MEAN;
    }
    if (n / 2 < 2) {
        apda_set_error("stdev requires at least two data points");
        return APDA_ERR_STATS_STDEV;
    }
    // a window holds at most n/8 + 8 peaks (candidates are strict local maxima above mean + 2 sigma: < 20 % of the
    // half spectrum's bins by Cantelli's inequality), so wider records than that are never needed
    if (k < 1 || rec_cap < k || (rec_cap > APDA_MAX_REC_CAP && (int64_t)rec_cap > APDA_MAX_PEAKS(n))) {
        apda_set_error("peaks: need 1 <= k (%d) <= rec_cap (%d) <= max(%d, n/8 + 8 = %lld)", k, rec_cap, APDA_MAX_REC_CAP,
                       (long long)APDA_MAX_PEAKS(n));
        return APDA_ERR_INVALID;
    }
    return APDA_OK;
}

template <typename T>
static int fft_dispatch(apda_ctx *ctx, cudaStream_t st, const T *d_samples, int64_t n_samples, int64_t ld,
                        int64_t batch, int64_t N, int flags, T *d_spec, bool complex_in, bool half_out = false) {
    if (batch == 0) return APDA_OK;
    if (sizeof(T) == 8 && flags == APDA_CENTER_MEAN) {
        apda_set_error("fft: APDA_CENTER_MEAN is an fp32-only option; the fp64 path is bit-faithful to the reference");
        return APDA_ERR_INVALID;
    }
    if (sizeof(T) == 4 && !complex_in && !ctx->generic_only && fft_f32_fast_supports(N))
        return launch_fft_f32_fast(ctx, st, reinterpret_cast<const float *>(d_samples), n_samples, ld, batch, N, flags,
                                   reinterpret_cast<float *>(d_spec), nullptr, half_out);
    if (sizeof(T) == 8 && !complex_in && !ctx->generic_only && fft_f64_fast_supports(N))
        return launch_fft_f64_fast(ctx, st, reinterpret_cast<const double *>(d_samples), n_samples, ld, batch, N, flags,
                                   reinterpret_cast<double *>(d_spec));
    // largest N that goes to the one-CTA-per-window kernel: fp32 N = 16384 fits its shared memory, but two K2 passes are
    // faster there (277 vs 483 ns per window); APDA_SMEM_MAXN overrides for A/B runs
    static const int64_t smem_cap = [] {
        const char *e = getenv("APDA_SMEM_MAXN");
        return e && e[0] ? (int64_t)atoll(e) : (int64_t)8192;
    }();
    if (N <= std::min(fft_smem_max_n<T>(ctx), smem_cap))
        return launch_fft_smem<T>(ctx, st, d_samples, n_samples, ld, batch, N, flags, d_spec, complex_in);
    return launch_fft_large<T>(ctx, st, d_samples, n_samples, ld, batch, N, flags, d_spec, complex_in);
}

template <typename T>
static int peaks_dispatch(apda_ctx *ctx, cudaStream_t st, const T *d_spec, int64_t n, int64_t batch, double fs,
                          const double *d_fs, int k, int rec_cap, int flexible, void *d_rec, void **ws, size_t *ws_bytes,
                          size_t ws_offset) {
    if (batch == 0) return APDA_OK;
    size_t need = peaks_mag_workspace_bytes<T>(ctx, n, batch);
    void *mag_ws = nullptr;
    if (need) {
        if (*ws_bytes < ws_offset + need) {
            apda_set_error("peaks: internal workspace too small");
            return APDA_ERR_NOMEM;
        }
        mag_ws = (char *)*ws + ws_offset;
    }
    return launch_peaks<T>(ctx, st, d_spec, n, batch, fs, d_fs, k, rec_cap, flexible, d_rec, mag_ws);
}

static inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// ---------------------------------------------------------------------------------------------------------------
// ragged batches: per-window sample counts (windows that lost samples to inf/nan filtering, text logs of different
// lengths).  Windows with the common length n_max run on the specialised kernels; the others are listed on the device
// and go through the general kernel with their own length.  No host synchronisation anywhere.
// ---------------------------------------------------------------------------------------------------------------
__global__ void ragged_list_kernel(const int *__restrict__ nv, int64_t batch, int n_max, int *__restrict__ list) {
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w < batch && nv[w] != n_max) list[1 + atomicAdd(&list[0], 1)] = (int)w;
}

// record status of ragged windows: bit 2 = the window's own padded length differs from the batch N (the reference would
// transform at that other length), bit 3 = empty window (the reference's pickers raise StatisticsError on start_fft([]))
__global__ void ragged_status_kernel(const int *__restrict__ nv, int64_t batch, int64_t N,
                                     unsigned char *__restrict__ recs, int64_t rec_bytes) {
    for (int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < batch; w += (int64_t)gridDim.x * blockDim.x) {
        const int n = nv[w];
        if (n == N) continue;
        int64_t p = 1;
        while (p < n) p <<= 1;
        int *hdr = reinterpret_cast<int *>(recs + (int64_t)w * rec_bytes);
        if (n <= 0) {
            hdr[0] = 0;
            hdr[1] |= 8;
        } else if (p != N) {
            hdr[1] |= 4;
        }
    }
}

template <typename T>
static int fft_dispatch_ragged(apda_ctx *ctx, cudaStream_t st, const T *d_samples, const int *d_nv, int64_t n_max,
                               int64_t ld, int64_t batch, int64_t N, int flags, T *d_spec) {
    if (batch == 0) return APDA_OK;
    if (N > fft_smem_max_n<T>(ctx)) {
        apda_set_error("ragged batches are offered for N <= %lld", (long long)fft_smem_max_n<T>(ctx));
        return APDA_ERR_UNSUPPORTED;
    }
    if (flags == APDA_CENTER_MEAN) {
        apda_set_error("ragged batches need the exact median (padding): APDA_CENTER_MEAN is not legal");
        return APDA_ERR_INVALID;
    }
    const bool fast32 = sizeof(T) == 4 && !ctx->generic_only && fft_f32_fast_supports(N);
    const bool fast64 = sizeof(T) == 8 && !ctx->generic_only && fft_f64_fast_supports(N);
    if (!fast32 && !fast64)
        return launch_fft_smem<T>(ctx, st, d_samples, n_max, ld, batch, N, flags, d_spec, false, d_nv, nullptr);
    int *ragged = nullptr;
    APDA_TRY(apda_ragged_list(ctx, st, batch, &ragged));
    ragged_list_kernel<<<(unsigned)((batch + 255) / 256), 256, 0, st>>>(d_nv, batch, (int)n_max, ragged);
    ctx->launches++;
    if (fast32)
        APDA_TRY(launch_fft_f32_fast(ctx, st, reinterpret_cast<const float *>(d_samples), n_max, ld, batch, N, flags,
                                     reinterpret_cast<float *>(d_spec), d_nv));
    else
        APDA_TRY(launch_fft_f64_fast(ctx, st, reinterpret_cast<const double *>(d_samples), n_max, ld, batch, N, flags,
                                     reinterpret_cast<double *>(d_spec), d_nv));
    return launch_fft_smem<T>(ctx, st, d_samples, n_max, ld, batch, N, flags, d_spec, false, d_nv, ragged);
}

static int check_ragged_args(apda_ctx *ctx, const void *in, const void *nv, int64_t n_max, int64_t ld, int64_t batch,
                             int64_t N, int flags, const void *out) {
    if (!nv) {
        apda_set_error("ragged: n_valid array is NULL");
        return APDA_ERR_INVALID;
    }
    return check_fft_args(ctx, in, n_max, ld, batch, N, flags, out);
}

template <typename T>
static int analyze_ragged_dev(apda_ctx *ctx, cudaStream_t st, const T *d_samples, const int *d_nv, int64_t n_max, int64_t ld,
                              int64_t batch, int64_t N, int flags, int flexible, double fs, const double *d_fs, int k,
                              int rec_cap, T *d_spec, void *d_rec, void **ws, size_t *ws_bytes, size_t ws_off) {
    APDA_TRY(fft_dispatch_ragged<T>(ctx, st, d_samples, d_nv, n_max, ld, batch, N, flags, d_spec));
    APDA_TRY(peaks_dispatch<T>(ctx, st, d_spec, N, batch, fs, d_fs, k, rec_cap, flexible, d_rec, ws, ws_bytes, ws_off));
    if (batch > 0) {  // every ragged path (specialised or general kernels): the status bits only depend on d_nv
        const unsigned blocks = (unsigned)std::min<int64_t>((batch + 255) / 256, 1024);
        ragged_status_kernel<<<blocks, 256, 0, st>>>(d_nv, batch, N, reinterpret_cast<unsigned char *>(d_rec),
                                                     APDA_REC_BYTES(rec_cap));
        ctx->launches++;
        APDA_CUDA(cudaGetLastError());
    }
    return APDA_OK;
}


// ---------------------------------------------------------------------------------------------------------------
// device-pointer entry points
// ---------------------------------------------------------------------------------------------------------------
template <typename T>
static int fft_dev(apda_ctx *ctx, const T *d_samples, int64_t n_samples, int64_t ld, int64_t batch, int64_t N, int flags,
                   T *d_spec) {
    APDA_TRY(check_fft_args(ctx, d_samples, n_samples, ld, batch, N, flags, d_spec));
    APDA_CUDA(cudaSetDevice(ctx->device));
    return fft_dispatch<T>(ctx, ctx->stream, d_samples, n_samples, ld, batch, N, flags, d_spec, false);
}
extern "C" int apda_fft_f64_dev(apda_ctx *ctx, const double *d_samples, int64_t n_samples, int64_t ld, int64_t batch,
                                int64_t N, int flags, double *d_spec) {
    return fft_dev<double>(ctx, d_samples, n_samples, ld, batch, N, flags, d_spec);
}
extern "C" int apda_fft_f32_dev(apda_ctx *ctx, const float *d_samples, int64_t n_samples, int64_t ld, int64_t batch,
                                int64_t N, int flags, float *d_spec) {
    return fft_dev<float>(ctx, d_samples, n_samples, ld, batch, N, flags, d_spec);
}

template <typename T>
static int peaks_dev(apda_ctx *ctx, const T *d_spec, int64_t n, int64_t batch, double fs, const double *d_fs, int k,
                     int rec_cap, int flexible, void *d_rec) {
    APDA_TRY(check_peaks_args(ctx, d_spec, n, batch, k, rec_cap, d_rec));
    APDA_CUDA(cudaSetDevice(ctx->device));
    size_t need = peaks_mag_workspace_bytes<T>(ctx, n, batch);
    if (need) {
        if (need > ctx->ws_bytes) APDA_CUDA(cudaStreamSynchronize(ctx->stream));  // old workspace may be in use
        APDA_TRY(apda_reserve(&ctx->ws, &ctx->ws_bytes, need));
    }
    return peaks_dispatch<T>(ctx, ctx->stream, d_spec, n, batch, fs, d_fs, k, rec_cap, flexible, d_rec, &ctx->ws,
                             &ctx->ws_bytes, 0);
}
extern "C" int apda_peaks_prominence_f64_dev(apda_ctx *ctx, const double *d_spec, int64_t n, int64_t batch, double fs,
                                             const double *d_fs, int k, int rec_cap, void *d_rec) {
    return peaks_dev<double>(ctx, d_spec, n, batch, fs, d_fs, k, rec_cap, 1, d_rec);
}
extern "C" int apda_peaks_prominence_f32_dev(apda_ctx *ctx, const float *d_spec, int64_t n, int64_t batch, double fs,
                                             const double *d_fs, int k, int rec_cap, void *d_rec) {
    return peaks_dev<float>(ctx, d_spec, n, batch, fs, d_fs, k, rec_cap, 1, d_rec);
}
extern "C" int apda_peaks_resolution_f64_dev(apda_ctx *ctx, const double *d_spec, int64_t n, int64_t batch, double fs,
                                             const double *d_fs, int k, int rec_cap, void *d_rec) {
    return peaks_dev<double>(ctx, d_spec, n, batch, fs, d_fs, k, rec_cap, 0, d_rec);
}
extern "C" int apda_peaks_resolution_f32_dev(apda_ctx *ctx, const float *d_spec, int64_t n, int64_t batch, double fs,
                                             const double *d_fs, int k, int rec_cap, void *d_rec) {
    return peaks_dev<float>(ctx, d_spec, n, batch, fs, d_fs, k, rec_cap, 0, d_rec);
}

template <typename T>
static int analyze_dev(apda_ctx *ctx, const T *d_samples, int64_t n_samples, int64_t ld, int64_t batch, int64_t N,
                       int flags, int flexible, double fs, const double *d_fs, int k, int rec_cap, T *d_spec_ws,
                       void *d_rec) {
    APDA_TRY(check_fft_args(ctx, d_samples, n_samples, ld, batch, N, flags, d_rec));
    APDA_TRY(check_peaks_args(ctx, d_samples, N, batch, k, rec_cap, d_rec));
    APDA_CUDA(cudaSetDevice(ctx->device));
    const size_t spec_bytes = d_spec_ws ? 0 : align256((size_t)batch * (size_t)N * 2 * sizeof(T));
    const size_t mag_bytes = peaks_mag_workspace_bytes<T>(ctx, N, batch);
    if (spec_bytes + mag_bytes > ctx->ws_bytes) {
        APDA_CUDA(cudaStreamSynchronize(ctx->stream));
        APDA_TRY(apda_reserve(&ctx->ws, &ctx->ws_bytes, spec_bytes + mag_bytes));
    }
    T *spec = d_spec_ws ? d_spec_ws : reinterpret_cast<T *>(ctx->ws);
    // the library's own workspace only ever feeds the picker: K1 skips the upper half of the spectrum there (a caller's
    // d_spec_ws receives all N bins, as apda_fft_* would write them)
    APDA_TRY(fft_dispatch<T>(ctx, ctx->stream, d_samples, n_samples, ld, batch, N, flags, spec, false, d_spec_ws == nullptr));
    return peaks_dispatch<T>(ctx, ctx->stream, spec, N, batch, fs, d_fs, k, rec_cap, flexible, d_rec, &ctx->ws,
                             &ctx->ws_bytes, spec_bytes);
}
extern "C" int apda_analyze_f64_dev(apda_ctx *ctx, const double *d_samples, int64_t n_samples, int64_t ld,
                                    int64_t batch, int64_t N, int flags, int flexible, double fs, const double *d_fs,
                                    int k, int rec_cap, double *d_spec_ws, void *d_rec) {
    return analyze_dev<double>(ctx, d_samples, n_samples, ld, batch, N, flags, flexible, fs, d_fs, k, rec_cap, d_spec_ws,
                               d_rec);
}
extern "C" int apda_analyze_f32_dev(apda_ctx *ctx, const float *d_samples, int64_t n_samples, int64_t ld, int64_t batch,
                                    int64_t N, int flags, int flexible, double fs, const double *d_fs, int k,
                                    int rec_cap, float *d_spec_ws, void *d_rec) {
    return analyze_dev<float>(ctx, d_samples, n_samples, ld, batch, N, flags, flexible, fs, d_fs, k, rec_cap, d_spec_ws,
                              d_rec);
}

template <typename T>
static int fft_ragged_dev(apda_ctx *ctx, const T *d_samples, const int32_t *d_nv, int64_t n_max, int64_t ld, int64_t batch,
                          int64_t N, int flags, T *d_spec) {
    APDA_TRY(check_ragged_args(ctx, d_samples, d_nv, n_max, ld, batch, N, flags, d_spec));
    APDA_CUDA(cudaSetDevice(ctx->device));
    return fft_dispatch_ragged<T>(ctx, ctx->stream, d_samples, d_nv, n_max, ld, batch, N, flags, d_spec);
}
extern "C" int apda_fft_ragged_f64_dev(apda_ctx *ctx, const double *d_samples, const int32_t *d_n_valid, int64_t n_max,
                                       int64_t ld, int64_t batch, int64_t N, int flags, double *d_spec) {
    return fft_ragged_dev<double>(ctx, d_samples, d_n_valid, n_max, ld, batch, N, flags, d_spec);
}
extern "C" int apda_fft_ragged_f32_dev(apda_ctx *ctx, const float *d_samples, const int32_t *d_n_valid, int64_t n_max,
                                       int64_t ld, int64_t batch, int64_t N, int flags, float *d_spec) {
    return fft_ragged_dev<float>(ctx, d_samples, d_n_valid, n_max, ld, batch, N, flags, d_spec);
}

template <typename T>
static int analyze_ragged_entry(apda_ctx *ctx, const T *d_samples, const int32_t *d_nv, int64_t n_max, int64_t ld,
                                int64_t batch, int64_t N, int flags, int flexible, double fs, const double *d_fs, int k,
                                int rec_cap, T *d_spec_ws, void *d_rec) {
    APDA_TRY(check_ragged_args(ctx, d_samples, d_nv, n_max, ld, batch, N, flags, d_rec));
    APDA_TRY(check_peaks_args(ctx, d_samples, N, batch, k, rec_cap, d_rec));
    APDA_CUDA(cudaSetDevice(ctx->device));
    const size_t spec_bytes = d_spec_ws ? 0 : align256((size_t)batch * (size_t)N * 2 * sizeof(T));
    const size_t mag_bytes = peaks_mag_workspace_bytes<T>(ctx, N, batch);
    if (spec_bytes + mag_bytes > ctx->ws_bytes) {
        APDA_CUDA(cudaStreamSynchronize(ctx->stream));
        APDA_TRY(apda_reserve(&ctx->ws, &ctx->ws_bytes, spec_bytes + mag_bytes));
    }
    T *spec = d_spec_ws ? d_spec_ws : reinterpret_cast<T *>(ctx->ws);
    return analyze_ragged_dev<T>(ctx, ctx->stream, d_samples, d_nv, n_max, ld, batch, N, flags, flexible, fs, d_fs, k, rec_cap,
                                 spec, d_rec, &ctx->ws, &ctx->ws_bytes, spec_bytes);
}
extern "C" int apda_analyze_ragged_f64_dev(apda_ctx *ctx, const double *d_samples, const int32_t *d_n_valid, int64_t n_max,
                                           int64_t ld, int64_t batch, int64_t N, int flags, int flexible, double fs,
                                           const double *d_fs, int k, int rec_cap, double *d_spec_ws, void *d_rec) {
    return analyze_ragged_entry<double>(ctx, d_samples, d_n_valid, n_max, ld, batch, N, flags, flexible, fs, d_fs, k, rec_cap,
                                        d_spec_ws, d_rec);
}
extern "C" int apda_analyze_ragged_f32_dev(apda_ctx *ctx, const float *d_samples, const int32_t *d_n_valid, int64_t n_max,
                                           int64_t ld, int64_t batch, int64_t N, int flags, int flexible, double fs,
                                           const double *d_fs, int k, int rec_cap, float *d_spec_ws, void *d_rec) {
    return analyze_ragged_entry<float>(ctx, d_samples, d_n_valid, n_max, ld, batch, N, flags, flexible, fs, d_fs, k, rec_cap,
                                       d_spec_ws, d_rec);
}

// ---------------------------------------------------------------------------------------------------------------
// host-pointer entry points: chunked two-stream pipeline (H2D of chunk c+1 overlaps the kernels / D2H of chunk c)
// ---------------------------------------------------------------------------------------------------------------
enum HostMode { kFftOnly, kPeaksOnly, kAnalyze, kFused };

template <typename T>
static int host_pipeline(apda_ctx *ctx, HostMode mode, const T *h_in, int64_t n_samples, int64_t ld, int64_t batch,
                         int64_t N, int flags, int flexible, double fs, const double *h_fs, int k, int rec_cap,
                         bool complex_in, T *h_spec_out, void *h_rec_out) {
    APDA_CUDA(cudaSetDevice(ctx->device));
    if (batch == 0) return APDA_OK;
    const size_t rec_bytes = (size_t)APDA_REC_BYTES(rec_cap);
    const size_t in_elems = mode == kPeaksOnly ? (size_t)N * 2 : (complex_in ? (size_t)N * 2 : (size_t)n_samples);
    const size_t in_ld = mode == kPeaksOnly ? (size_t)N * 2 : (complex_in ? (size_t)N * 2 : (size_t)ld);
    const size_t spec_elems = (size_t)N * 2;
    // chunk: ~96 MB of spectrum per stream, at least one window
    int64_t chunk = std::max<int64_t>(1, (int64_t)((96u << 20) / ((mode == kFused ? in_elems : spec_elems) * sizeof(T))));
    chunk = std::min<int64_t>(chunk, batch);
    if (batch > chunk && batch < 2 * chunk) chunk = (batch + 1) / 2;

    const size_t in_bytes = align256(chunk * in_elems * sizeof(T));
    const size_t spec_bytes = (mode == kPeaksOnly || mode == kFused) ? 0 : align256(chunk * spec_elems * sizeof(T));
    const size_t recs_bytes = mode == kFftOnly ? 0 : align256(chunk * rec_bytes);
    const size_t fs_bytes = (h_fs && mode != kFftOnly) ? align256(chunk * sizeof(double)) : 0;
    const size_t mag_bytes = (mode == kFftOnly || mode == kFused) ? 0 : align256(peaks_mag_workspace_bytes<T>(ctx, N, chunk));
    const size_t total = in_bytes + spec_bytes + recs_bytes + fs_bytes + mag_bytes;
    for (int s = 0; s < 2; ++s) {
        if (total > ctx->ws_pipe_bytes[s]) {
            APDA_CUDA(cudaStreamSynchronize(ctx->pipe[s]));
            APDA_TRY(apda_reserve(&ctx->ws_pipe[s], &ctx->ws_pipe_bytes[s], total));
        }
        if (batch <= chunk) break;  // single chunk: one stream is enough
    }

    // one chunk; an error returns from the lambda only, so the caller below always drains both streams before it
    // reports (async copies from / into the caller's buffers must not outlive the call)
    auto run_chunk = [&](int c, int64_t done, int64_t cnt) -> int {
        const int s = c & 1;
        cudaStream_t st = ctx->pipe[s];
        char *base = (char *)ctx->ws_pipe[s];
        T *d_in = (T *)base;
        T *d_spec = (T *)(base + in_bytes);
        void *d_rec = base + in_bytes + spec_bytes;
        double *d_fs = fs_bytes ? (double *)(base + in_bytes + spec_bytes + recs_bytes) : nullptr;
        void *mag_ws = mag_bytes ? base + in_bytes + spec_bytes + recs_bytes + fs_bytes : nullptr;
        size_t mag_have = mag_bytes;

        const T *src = h_in + (size_t)done * in_ld;
        if (in_ld == in_elems) {
            APDA_CUDA(cudaMemcpyAsync(d_in, src, cnt * in_elems * sizeof(T), cudaMemcpyHostToDevice, st));
        } else {
            APDA_CUDA(cudaMemcpy2DAsync(d_in, in_elems * sizeof(T), src, in_ld * sizeof(T), in_elems * sizeof(T), cnt,
                                        cudaMemcpyHostToDevice, st));
        }
        if (d_fs) APDA_CUDA(cudaMemcpyAsync(d_fs, h_fs + done, cnt * sizeof(double), cudaMemcpyHostToDevice, st));

        const T *spec_for_peaks = d_in;
        if (mode == kFused) {
            APDA_TRY(launch_fused_f32(ctx, st, reinterpret_cast<const float *>(d_in), n_samples, (int64_t)in_elems, cnt, N,
                                      flags, flexible, fs, d_fs, k, d_rec));
            APDA_CUDA(cudaMemcpyAsync((char *)h_rec_out + (size_t)done * rec_bytes, d_rec, cnt * rec_bytes,
                                      cudaMemcpyDeviceToHost, st));
            return APDA_OK;
        }
        if (mode != kPeaksOnly) {
            APDA_TRY(fft_dispatch<T>(ctx, st, d_in, n_samples, (int64_t)in_elems, cnt, N, flags, d_spec, complex_in,
                                     mode == kAnalyze));
            spec_for_peaks = d_spec;
            if (mode == kFftOnly)
                APDA_CUDA(cudaMemcpyAsync(h_spec_out + (size_t)done * spec_elems, d_spec, cnt * spec_elems * sizeof(T),
                                          cudaMemcpyDeviceToHost, st));
        }
        if (mode != kFftOnly) {
            APDA_TRY(peaks_dispatch<T>(ctx, st, spec_for_peaks, N, cnt, fs, d_fs, k, rec_cap, flexible, d_rec, &mag_ws,
                                       &mag_have, 0));
            APDA_CUDA(cudaMemcpyAsync((char *)h_rec_out + (size_t)done * rec_bytes, d_rec, cnt * rec_bytes,
                                      cudaMemcpyDeviceToHost, st));
        }
        return APDA_OK;
    };
    int status = APDA_OK;
    int c = 0;
    for (int64_t done = 0; done < batch && status == APDA_OK; ++c) {
        const int64_t cnt = std::min<int64_t>(chunk, batch - done);
        status = run_chunk(c, done, cnt);
        done += cnt;
    }
    cudaError_t e0 = cudaStreamSynchronize(ctx->pipe[0]);
    cudaError_t e1 = cudaStreamSynchronize(ctx->pipe[1]);
    if (status != APDA_OK) return status;
    if (e0 != cudaSuccess) return apda_cuda_fail(e0, "host pipeline (stream 0)");
    if (e1 != cudaSuccess) return apda_cuda_fail(e1, "host pipeline (stream 1)");
    return APDA_OK;
}

extern "C" int apda_fft_f64_host(apda_ctx *ctx, const double *h_samples, int64_t n_samples, int64_t ld, int64_t batch,
                                 int64_t N, int flags, double *h_spec) {
    APDA_TRY(check_fft_args(ctx, h_samples, n_samples, ld, batch, N, flags, h_spec));
    return host_pipeline<double>(ctx, kFftOnly, h_samples, n_samples, ld, batch, N, flags, 0, 0.0, nullptr, 1, 5, false,
                                 h_spec, nullptr);
}
extern "C" int apda_fft_f32_host(apda_ctx *ctx, const float *h_samples, int64_t n_samples, int64_t ld, int64_t batch,
                                 int64_t N, int flags, float *h_spec) {
    APDA_TRY(check_fft_args(ctx, h_samples, n_samples, ld, batch, N, flags, h_spec));
    return host_pipeline<float>(ctx, kFftOnly, h_samples, n_samples, ld, batch, N, flags, 0, 0.0, nullptr, 1, 5, false,
                                h_spec, nullptr);
}
extern "C" int apda_fft_c2c_f64_host(apda_ctx *ctx, const double *h_in, int64_t batch, int64_t N, double *h_out) {
    APDA_TRY(check_fft_args(ctx, h_in, N, N, batch, N, APDA_CENTER_NONE, h_out));
    return host_pipeline<double>(ctx, kFftOnly, h_in, N, N, batch, N, APDA_CENTER_NONE, 0, 0.0, nullptr, 1, 5, true,
                                 h_out, nullptr);
}
extern "C" int apda_peaks_prominence_f64_host(apda_ctx *ctx, const double *h_spec, int64_t n, int64_t batch, double fs,
                                              const double *h_fs, int k, int rec_cap, void *h_rec) {
    APDA_TRY(check_peaks_args(ctx, h_spec, n, batch, k, rec_cap, h_rec));
    return host_pipeline<double>(ctx, kPeaksOnly, h_spec, 0, 0, batch, n, 0, 1, fs, h_fs, k, rec_cap, false, nullptr,
                                 h_rec);
}
extern "C" int apda_peaks_resolution_f64_host(apda_ctx *ctx, const double *h_spec, int64_t n, int64_t batch, double fs,
                                              const double *h_fs, int k, int rec_cap, void *h_rec) {
    APDA_TRY(check_peaks_args(ctx, h_spec, n, batch, k, rec_cap, h_rec));
    return host_pipeline<double>(ctx, kPeaksOnly, h_spec, 0, 0, batch, n, 0, 0, fs, h_fs, k, rec_cap, false, nullptr,
                                 h_rec);
}
extern "C" int apda_peaks_prominence_f32_host(apda_ctx *ctx, const float *h_spec, int64_t n, int64_t batch, double fs,
                                              const double *h_fs, int k, int rec_cap, void *h_rec) {
    APDA_TRY(check_peaks_args(ctx, h_spec, n, batch, k, rec_cap, h_rec));
    return host_pipeline<float>(ctx, kPeaksOnly, h_spec, 0, 0, batch, n, 0, 1, fs, h_fs, k, rec_cap, false, nullptr,
                                h_rec);
}
extern "C" int apda_peaks_resolution_f32_host(apda_ctx *ctx, const float *h_spec, int64_t n, int64_t batch, double fs,
                                              const double *h_fs, int k, int rec_cap, void *h_rec) {
    APDA_TRY(check_peaks_args(ctx, h_spec, n, batch, k, rec_cap, h_rec));
    return host_pipeline<float>(ctx, kPeaksOnly, h_spec, 0, 0, batch, n, 0, 0, fs, h_fs, k, rec_cap, false, nullptr,
                                h_rec);
}
extern "C" int apda_analyze_f64_host(apda_ctx *ctx, const double *h_samples, int64_t n_samples, int64_t ld,
                                     int64_t batch, int64_t N, int flags, int flexible, double fs, const double *h_fs,
                                     int k, int rec_cap, void *h_rec) {
    APDA_TRY(check_fft_args(ctx, h_samples, n_samples, ld, batch, N, flags, h_rec));
    APDA_TRY(check_peaks_args(ctx, h_samples, N, batch, k, rec_cap, h_rec));
    return host_pipeline<double>(ctx, kAnalyze, h_samples, n_samples, ld, batch, N, flags, flexible, fs, h_fs, k, rec_cap,
                                 false, nullptr, h_rec);
}
extern "C" int apda_analyze_f32_host(apda_ctx *ctx, const float *h_samples, int64_t n_samples, int64_t ld, int64_t batch,
                                     int64_t N, int flags, int flexible, double fs, const double *h_fs, int k,
                                     int rec_cap, void *h_rec) {
    APDA_TRY(check_fft_args(ctx, h_samples, n_samples, ld, batch, N, flags, h_rec));
    APDA_TRY(check_peaks_args(ctx, h_samples, N, batch, k, rec_cap, h_rec));
    return host_pipeline<float>(ctx, kAnalyze, h_samples, n_samples, ld, batch, N, flags, flexible, fs, h_fs, k, rec_cap,
                                false, nullptr, h_rec);
}

// ---------------------------------------------------------------------------------------------------------------
// one host process, several GPUs: the batch is sharded contiguously over the contexts (SURVEY 8e: rank r of G owns
// windows [r*ceil(B/G), ...)), one host thread per context runs the chunked host pipeline on its shard, and every
// device copies its records straight into its rows of the caller's table - the "gather to rank 0" of a single-process
// host needs no collective at all.  (Multi-process fleets use the peer record table below, or NCCL in the host language.)
// ---------------------------------------------------------------------------------------------------------------
template <typename T>
static int multi_analyze_host(apda_ctx **ctxs, int n_ctx, const T *h_samples, int64_t n_samples, int64_t ld, int64_t batch,
                              int64_t N, int flags, int flexible, double fs, const double *h_fs, int k, int rec_cap,
                              void *h_rec) {
    if (!ctxs || n_ctx < 1 || n_ctx > 64) {
        apda_set_error("multi_analyze: need 1..64 contexts");
        return APDA_ERR_INVALID;
    }
    for (int i = 0; i < n_ctx; ++i) {
        if (!ctxs[i]) {
            apda_set_error("multi_analyze: context %d is NULL", i);
            return APDA_ERR_INVALID;
        }
        for (int j = 0; j < i; ++j)
            if (ctxs[j] == ctxs[i]) {
                apda_set_error("multi_analyze: context %d is listed twice (a context belongs to one thread)", i);
                return APDA_ERR_INVALID;
            }
    }
    APDA_TRY(check_fft_args(ctxs[0], h_samples, n_samples, ld, batch, N, flags, h_rec));
    APDA_TRY(check_peaks_args(ctxs[0], h_samples, N, batch, k, rec_cap, h_rec));
    const int64_t per = (batch + n_ctx - 1) / n_ctx;
    const size_t rec_bytes = (size_t)APDA_REC_BYTES(rec_cap);
    std::vector<int> status((size_t)n_ctx, APDA_OK);
    std::vector<std::string> message((size_t)n_ctx);
    std::vector<std::thread> workers;
    for (int r = 0; r < n_ctx; ++r) {
        const int64_t lo = std::min<int64_t>(batch, r * per), hi = std::min<int64_t>(batch, lo + per);
        if (hi <= lo) continue;
        workers.emplace_back([&, r, lo, hi] {
            status[(size_t)r] = host_pipeline<T>(ctxs[r], kAnalyze, h_samples + (size_t)lo * (size_t)ld, n_samples, ld, hi - lo, N,
                                                 flags, flexible, fs, h_fs ? h_fs + lo : nullptr, k, rec_cap, false, nullptr,
                                                 (char *)h_rec + (size_t)lo * rec_bytes);
            if (status[(size_t)r] != APDA_OK) message[(size_t)r] = apda_last_error();  // the worker's thread-local message
        });
    }
    for (auto &w : workers) w.join();
    for (int r = 0; r < n_ctx; ++r)
        if (status[(size_t)r] != APDA_OK) {
            apda_set_error("multi_analyze: context %d (device %d): %s", r, ctxs[r]->device, message[(size_t)r].c_str());
            return status[(size_t)r];
        }
    return APDA_OK;
}
extern "C" int apda_multi_analyze_f32_host(apda_ctx **ctxs, int n_ctx, const float *h_samples, int64_t n_samples, int64_t ld,
                                           int64_t batch, int64_t N, int flags, int flexible, double fs, const double *h_fs,
                                           int k, int rec_cap, void *h_rec) {
    return multi_analyze_host<float>(ctxs, n_ctx, h_samples, n_samples, ld, batch, N, flags, flexible, fs, h_fs, k, rec_cap, h_rec);
}
extern "C" int apda_multi_analyze_f64_host(apda_ctx **ctxs, int n_ctx, const double *h_samples, int64_t n_samples, int64_t ld,
                                           int64_t batch, int64_t N, int flags, int flexible, double fs, const double *h_fs,
                                           int k, int rec_cap, void *h_rec) {
    return multi_analyze_host<double>(ctxs, n_ctx, h_samples, n_samples, ld, batch, N, flags, flexible, fs, h_fs, k, rec_cap, h_rec);
}

static int check_fused_args(int64_t N, int flags, int k, int rec_cap) {
    if (!fft_f32_fast_supports(N) || rec_cap != 5 || k < 1 || k > 5) {
        apda_set_error("analyze_fused_f32: needs N in {1024, 2048, 4096, 8192}, 1 <= k <= 5 and 128-byte records (rec_cap 5)");
        return APDA_ERR_UNSUPPORTED;
    }
    if (flags == APDA_CENTER_NONE) {
        apda_set_error("analyze_fused_f32: APDA_CENTER_NONE is not offered by the fused kernel");
        return APDA_ERR_UNSUPPORTED;
    }
    return APDA_OK;
}

extern "C" int apda_analyze_fused_f32_dev(apda_ctx *ctx, const float *d_samples, int64_t n_samples, int64_t ld,
                                          int64_t batch, int64_t N, int flags, int flexible, double fs,
                                          const double *d_fs, int k, int rec_cap, void *d_rec) {
    APDA_TRY(check_fft_args(ctx, d_samples, n_samples, ld, batch, N, flags, d_rec));
    APDA_TRY(check_peaks_args(ctx, d_samples, N, batch, k, rec_cap, d_rec));
    APDA_TRY(check_fused_args(N, flags, k, rec_cap));
    APDA_CUDA(cudaSetDevice(ctx->device));
    if (batch == 0) return APDA_OK;
    return launch_fused_f32(ctx, ctx->stream, d_samples, n_samples, ld, batch, N, flags, flexible, fs, d_fs, k, d_rec);
}

extern "C" int apda_analyze_fused_f32_host(apda_ctx *ctx, const float *h_samples, int64_t n_samples, int64_t ld,
                                           int64_t batch, int64_t N, int flags, int flexible, double fs,
                                           const double *h_fs, int k, int rec_cap, void *h_rec) {
    APDA_TRY(check_fft_args(ctx, h_samples, n_samples, ld, batch, N, flags, h_rec));
    APDA_TRY(check_peaks_args(ctx, h_samples, N, batch, k, rec_cap, h_rec));
    APDA_TRY(check_fused_args(N, flags, k, rec_cap));
    return host_pipeline<float>(ctx, kFused, h_samples, n_samples, ld, batch, N, flags, flexible, fs, h_fs, k, rec_cap, false,
                                nullptr, h_rec);
}

// ---------------------------------------------------------------------------------------------------------------
// fp32 tie resolution: records with status exactly APDA_STATUS_FP32_TIE get the fp64 path's record of the widened samples
// ---------------------------------------------------------------------------------------------------------------
static int check_resolve_args(apda_ctx *ctx, const float *samples, int64_t n_samples, int64_t ld, int64_t batch, int64_t N,
                              int flags, int k, int rec_cap, const void *rec) {
    APDA_TRY(check_fft_args(ctx, samples, n_samples, ld, batch, N, flags, rec));
    return check_peaks_args(ctx, samples, N, batch, k, rec_cap, rec);
}
// the fp64 reference centres with the exact median; APDA_CENTER_MEAN (full-length windows only) is its fp32 shortcut
static int resolve_center(int flags) { return flags == APDA_CENTER_MEAN ? APDA_CENTER_MEDIAN : flags; }

extern "C" int apda_resolve_fp32_ties_dev(apda_ctx *ctx, const float *d_samples, const int32_t *d_n_valid,
                                          int64_t n_samples, int64_t ld, int64_t batch, int64_t N, int flags, int flexible,
                                          double fs, const double *d_fs, int k, int rec_cap, void *d_rec) {
    APDA_TRY(check_resolve_args(ctx, d_samples, n_samples, ld, batch, N, flags, k, rec_cap, d_rec));
    APDA_CUDA(cudaSetDevice(ctx->device));
    if (N > fft_smem_max_n<double>(ctx)) {
        apda_set_error("resolve_fp32_ties_dev: N=%lld > %lld does not fit one CTA in fp64 (use apda_resolve_fp32_ties_host)",
                       (long long)N, (long long)fft_smem_max_n<double>(ctx));
        return APDA_ERR_UNSUPPORTED;
    }
    if (batch == 0) return APDA_OK;
    const size_t slots = resolve_ties_slot_bytes(ctx, N, batch);
    if (slots > ctx->ws_bytes) {
        APDA_CUDA(cudaStreamSynchronize(ctx->stream));  // old workspace may be in use
        APDA_TRY(apda_reserve(&ctx->ws, &ctx->ws_bytes, slots));
    }
    int *list = nullptr;
    APDA_TRY(apda_tie_list(ctx, ctx->stream, batch, &list));
    return launch_resolve_ties(ctx, ctx->stream, d_samples, d_n_valid, n_samples, ld, batch, N, resolve_center(flags), flexible,
                               fs, d_fs, k, rec_cap, d_rec, list, ctx->ws);
}

extern "C" int apda_resolve_fp32_ties_host(apda_ctx *ctx, const float *h_samples, const int32_t *h_n_valid,
                                           int64_t n_samples, int64_t ld, int64_t batch, int64_t N, int flags, int flexible,
                                           double fs, const double *h_fs, int k, int rec_cap, void *h_rec) {
    APDA_TRY(check_resolve_args(ctx, h_samples, n_samples, ld, batch, N, flags, k, rec_cap, h_rec));
    APDA_CUDA(cudaSetDevice(ctx->device));
    const bool on_device = N <= fft_smem_max_n<double>(ctx);
    if (!on_device && h_n_valid) {
        apda_set_error("ragged batches are offered for N <= %lld", (long long)fft_smem_max_n<double>(ctx));
        return APDA_ERR_UNSUPPORTED;
    }
    const int center = resolve_center(flags);
    const size_t rec_bytes = (size_t)APDA_REC_BYTES(rec_cap);
    unsigned char *recs = reinterpret_cast<unsigned char *>(h_rec);
    std::vector<int64_t> tied;
    for (int64_t w = 0; w < batch; ++w) {
        int32_t status;
        memcpy(&status, recs + (size_t)w * rec_bytes + 4, sizeof(status));
        if (status == APDA_STATUS_FP32_TIE) tied.push_back(w);
    }
    const int64_t cnt = (int64_t)tied.size();
    if (cnt == 0) return APDA_OK;

    if (!on_device) {  // the fp64 analysis pipeline on the gathered, widened windows
        std::vector<double> x((size_t)cnt * (size_t)n_samples), f(h_fs ? (size_t)cnt : 0);
        std::vector<unsigned char> r((size_t)cnt * rec_bytes);
        for (int64_t i = 0; i < cnt; ++i) {
            const float *src = h_samples + (size_t)tied[(size_t)i] * (size_t)ld;
            std::copy(src, src + n_samples, x.begin() + (size_t)i * (size_t)n_samples);
            if (h_fs) f[(size_t)i] = h_fs[tied[(size_t)i]];
        }
        APDA_TRY(host_pipeline<double>(ctx, kAnalyze, x.data(), n_samples, n_samples, cnt, N, center, flexible, fs,
                                       h_fs ? f.data() : nullptr, k, rec_cap, false, nullptr, r.data()));
        for (int64_t i = 0; i < cnt; ++i)
            memcpy(recs + (size_t)tied[(size_t)i] * rec_bytes, r.data() + (size_t)i * rec_bytes, rec_bytes);
        return APDA_OK;
    }

    // the device resolver on the gathered windows (every uploaded record is tied, so every one is listed), in chunks of
    // about 96 MB of samples on the first pipeline stream
    int64_t chunk = std::max<int64_t>(1, (int64_t)((96u << 20) / ((size_t)n_samples * sizeof(float))));
    chunk = std::min<int64_t>(chunk, cnt);
    const size_t in_b = align256((size_t)chunk * (size_t)n_samples * sizeof(float)), rec_b = align256((size_t)chunk * rec_bytes);
    const size_t fs_b = h_fs ? align256((size_t)chunk * sizeof(double)) : 0, nv_b = h_n_valid ? align256((size_t)chunk * sizeof(int)) : 0;
    const size_t total = in_b + rec_b + fs_b + nv_b + resolve_ties_slot_bytes(ctx, N, chunk);
    cudaStream_t st = ctx->pipe[0];
    if (total > ctx->ws_pipe_bytes[0]) {
        APDA_CUDA(cudaStreamSynchronize(st));
        APDA_TRY(apda_reserve(&ctx->ws_pipe[0], &ctx->ws_pipe_bytes[0], total));
    }
    char *base = (char *)ctx->ws_pipe[0];
    float *d_in = (float *)base;
    unsigned char *d_rec = (unsigned char *)(base + in_b);
    double *d_fs = h_fs ? (double *)(base + in_b + rec_b) : nullptr;
    int *d_nv = h_n_valid ? (int *)(base + in_b + rec_b + fs_b) : nullptr;
    void *d_slots = base + in_b + rec_b + fs_b + nv_b;
    std::vector<float> x((size_t)chunk * (size_t)n_samples);
    std::vector<unsigned char> r((size_t)chunk * rec_bytes);
    std::vector<double> f(h_fs ? (size_t)chunk : 0);
    std::vector<int> nv(h_n_valid ? (size_t)chunk : 0);
    // one chunk; an error returns from the lambda only, so the stream is always drained before the host buffers go
    auto run_chunk = [&](int64_t done, int64_t c) -> int {
        for (int64_t i = 0; i < c; ++i) {
            const int64_t w = tied[(size_t)(done + i)];
            const float *src = h_samples + (size_t)w * (size_t)ld;
            std::copy(src, src + n_samples, x.begin() + (size_t)i * (size_t)n_samples);
            memcpy(r.data() + (size_t)i * rec_bytes, recs + (size_t)w * rec_bytes, rec_bytes);
            if (h_fs) f[(size_t)i] = h_fs[w];
            if (h_n_valid) nv[(size_t)i] = h_n_valid[w];
        }
        APDA_CUDA(cudaMemcpyAsync(d_in, x.data(), (size_t)c * (size_t)n_samples * sizeof(float), cudaMemcpyHostToDevice, st));
        APDA_CUDA(cudaMemcpyAsync(d_rec, r.data(), (size_t)c * rec_bytes, cudaMemcpyHostToDevice, st));
        if (d_fs) APDA_CUDA(cudaMemcpyAsync(d_fs, f.data(), (size_t)c * sizeof(double), cudaMemcpyHostToDevice, st));
        if (d_nv) APDA_CUDA(cudaMemcpyAsync(d_nv, nv.data(), (size_t)c * sizeof(int), cudaMemcpyHostToDevice, st));
        int *list = nullptr;
        APDA_TRY(apda_tie_list(ctx, st, c, &list));
        APDA_TRY(launch_resolve_ties(ctx, st, d_in, d_nv, n_samples, n_samples, c, N, center, flexible, fs, d_fs, k, rec_cap,
                                     d_rec, list, d_slots));
        APDA_CUDA(cudaMemcpyAsync(r.data(), d_rec, (size_t)c * rec_bytes, cudaMemcpyDeviceToHost, st));
        return APDA_OK;
    };
    for (int64_t done = 0; done < cnt; done += chunk) {
        const int64_t c = std::min<int64_t>(chunk, cnt - done);
        const int status = run_chunk(done, c);
        const cudaError_t e = cudaStreamSynchronize(st);
        if (status != APDA_OK) return status;
        if (e != cudaSuccess) return apda_cuda_fail(e, "resolve_fp32_ties_host");
        for (int64_t i = 0; i < c; ++i)
            memcpy(recs + (size_t)tied[(size_t)(done + i)] * rec_bytes, r.data() + (size_t)i * rec_bytes, rec_bytes);
    }
    return APDA_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// wire-format ingest: 2 bytes per sample over PCIe instead of 4/8
// ---------------------------------------------------------------------------------------------------------------
static int check_wire_args(apda_ctx *ctx, const void *payload, const void *fv, int64_t n_max, int64_t ld_bytes,
                           int64_t batch, const void *out) {
    if (!ctx || !payload || !fv || !out || n_max < 1 || n_max > (int64_t(1) << 24) || ld_bytes < 2 * n_max || batch < 0 ||
        batch > 0x7fffffff) {
        apda_set_error("wire16: bad arguments (need payload, first_value, out, 1 <= n_max, ld_bytes >= 2*n_max)");
        return APDA_ERR_INVALID;
    }
    return APDA_OK;
}

template <typename T>
static int decode_wire16_dev(apda_ctx *ctx, const uint8_t *d_payload, int64_t n_max, int64_t ld_bytes, int64_t batch,
                             const double *d_first_value, T *d_samples, int64_t ld_out, int32_t *d_n_valid) {
    APDA_TRY(check_wire_args(ctx, d_payload, d_first_value, n_max, ld_bytes, batch, d_samples));
    if (!d_n_valid || ld_out < n_max) {
        apda_set_error("wire16: n_valid is NULL or ld_out < n_max");
        return APDA_ERR_INVALID;
    }
    APDA_CUDA(cudaSetDevice(ctx->device));
    return launch_decode_wire16<T>(ctx, ctx->stream, d_payload, n_max, ld_bytes, batch, d_first_value, d_samples, ld_out,
                                   d_n_valid);
}
extern "C" int apda_decode_wire16_f64_dev(apda_ctx *ctx, const uint8_t *d_payload, int64_t n_max, int64_t ld_bytes,
                                          int64_t batch, const double *d_first_value, double *d_samples, int64_t ld_out,
                                          int32_t *d_n_valid) {
    return decode_wire16_dev<double>(ctx, d_payload, n_max, ld_bytes, batch, d_first_value, d_samples, ld_out, d_n_valid);
}
extern "C" int apda_decode_wire16_f32_dev(apda_ctx *ctx, const uint8_t *d_payload, int64_t n_max, int64_t ld_bytes,
                                          int64_t batch, const double *d_first_value, float *d_samples, int64_t ld_out,
                                          int32_t *d_n_valid) {
    return decode_wire16_dev<float>(ctx, d_payload, n_max, ld_bytes, batch, d_first_value, d_samples, ld_out, d_n_valid);
}

// host payload -> (optionally) host samples and/or host records; chunked over the two pipeline streams
template <typename T>
static int wire16_host(apda_ctx *ctx, const uint8_t *h_payload, int64_t n_max, int64_t ld_bytes, int64_t batch,
                       const double *h_first_value, T *h_samples_out, int32_t *h_n_valid_out, bool analyze, int64_t N,
                       int flags, int flexible, double fs, const double *h_fs, int k, int rec_cap, void *h_rec) {
    APDA_CUDA(cudaSetDevice(ctx->device));
    if (batch == 0) return APDA_OK;
    const size_t rec_bytes = (size_t)APDA_REC_BYTES(rec_cap);
    const size_t per_window = analyze ? (size_t)N * 2 * sizeof(T) : (size_t)n_max * sizeof(T);
    int64_t chunk = std::max<int64_t>(1, (int64_t)((96u << 20) / per_window));
    chunk = std::min<int64_t>(chunk, batch);
    if (batch > chunk && batch < 2 * chunk) chunk = (batch + 1) / 2;
    const size_t pay_b = align256(chunk * (size_t)n_max * 2), fv_b = align256(chunk * sizeof(double));
    const size_t smp_b = align256(chunk * (size_t)n_max * sizeof(T)), nv_b = align256(chunk * sizeof(int));
    const size_t spec_b = analyze ? align256(chunk * (size_t)N * 2 * sizeof(T)) : 0;
    const size_t recs_b = analyze ? align256(chunk * rec_bytes) : 0;
    const size_t fs_b = (analyze && h_fs) ? align256(chunk * sizeof(double)) : 0;
    const size_t mag_b = analyze ? align256(peaks_mag_workspace_bytes<T>(ctx, N, chunk)) : 0;
    const size_t total = pay_b + fv_b + smp_b + nv_b + spec_b + recs_b + fs_b + mag_b;
    for (int s = 0; s < 2; ++s) {
        if (total > ctx->ws_pipe_bytes[s]) {
            APDA_CUDA(cudaStreamSynchronize(ctx->pipe[s]));
            APDA_TRY(apda_reserve(&ctx->ws_pipe[s], &ctx->ws_pipe_bytes[s], total));
        }
        if (batch <= chunk) break;
    }
    auto run_chunk = [&](int c, int64_t done, int64_t cnt) -> int {  // see host_pipeline: errors never skip the drain
        const int s = c & 1;
        cudaStream_t st = ctx->pipe[s];
        char *base = (char *)ctx->ws_pipe[s];
        unsigned char *d_pay = (unsigned char *)base;
        double *d_fv = (double *)(base + pay_b);
        T *d_smp = (T *)(base + pay_b + fv_b);
        int *d_nv = (int *)(base + pay_b + fv_b + smp_b);
        T *d_spec = (T *)(base + pay_b + fv_b + smp_b + nv_b);
        void *d_rec = base + pay_b + fv_b + smp_b + nv_b + spec_b;
        double *d_fs = fs_b ? (double *)(base + pay_b + fv_b + smp_b + nv_b + spec_b + recs_b) : nullptr;
        void *mag_ws = mag_b ? base + pay_b + fv_b + smp_b + nv_b + spec_b + recs_b + fs_b : nullptr;
        size_t mag_have = mag_b;
        if (ld_bytes == 2 * n_max)
            APDA_CUDA(cudaMemcpyAsync(d_pay, h_payload + (size_t)done * ld_bytes, cnt * (size_t)n_max * 2,
                                      cudaMemcpyHostToDevice, st));
        else
            APDA_CUDA(cudaMemcpy2DAsync(d_pay, (size_t)n_max * 2, h_payload + (size_t)done * ld_bytes, ld_bytes,
                                        (size_t)n_max * 2, cnt, cudaMemcpyHostToDevice, st));
        APDA_CUDA(cudaMemcpyAsync(d_fv, h_first_value + done, cnt * sizeof(double), cudaMemcpyHostToDevice, st));
        if (d_fs) APDA_CUDA(cudaMemcpyAsync(d_fs, h_fs + done, cnt * sizeof(double), cudaMemcpyHostToDevice, st));
        APDA_TRY(launch_decode_wire16<T>(ctx, st, d_pay, n_max, (int64_t)n_max * 2, cnt, d_fv, d_smp, n_max, d_nv));
        if (h_samples_out)
            APDA_CUDA(cudaMemcpyAsync(h_samples_out + (size_t)done * n_max, d_smp, cnt * (size_t)n_max * sizeof(T),
                                      cudaMemcpyDeviceToHost, st));
        if (h_n_valid_out)
            APDA_CUDA(cudaMemcpyAsync(h_n_valid_out + done, d_nv, cnt * sizeof(int), cudaMemcpyDeviceToHost, st));
        if (analyze) {
            APDA_TRY(analyze_ragged_dev<T>(ctx, st, d_smp, d_nv, n_max, n_max, cnt, N, flags, flexible, fs, d_fs, k, rec_cap,
                                           d_spec, d_rec, &mag_ws, &mag_have, 0));
            APDA_CUDA(cudaMemcpyAsync((char *)h_rec + (size_t)done * rec_bytes, d_rec, cnt * rec_bytes,
                                      cudaMemcpyDeviceToHost, st));
        }
        return APDA_OK;
    };
    int status = APDA_OK;
    int c = 0;
    for (int64_t done = 0; done < batch && status == APDA_OK; ++c) {
        const int64_t cnt = std::min<int64_t>(chunk, batch - done);
        status = run_chunk(c, done, cnt);
        done += cnt;
    }
    cudaError_t e0 = cudaStreamSynchronize(ctx->pipe[0]);
    cudaError_t e1 = cudaStreamSynchronize(ctx->pipe[1]);
    if (status != APDA_OK) return status;
    if (e0 != cudaSuccess) return apda_cuda_fail(e0, "wire16 pipeline (stream 0)");
    if (e1 != cudaSuccess) return apda_cuda_fail(e1, "wire16 pipeline (stream 1)");
    return APDA_OK;
}

extern "C" int apda_decode_wire16_f64_host(apda_ctx *ctx, const uint8_t *h_payload, int64_t n_max, int64_t ld_bytes,
                                           int64_t batch, const double *h_first_value, double *h_samples,
                                           int32_t *h_n_valid) {
    APDA_TRY(check_wire_args(ctx, h_payload, h_first_value, n_max, ld_bytes, batch, h_samples));
    return wire16_host<double>(ctx, h_payload, n_max, ld_bytes, batch, h_first_value, h_samples, h_n_valid, false, 0, 0, 0,
                               0.0, nullptr, 1, 5, nullptr);
}
template <typename T>
static int analyze_wire16_host(apda_ctx *ctx, const uint8_t *h_payload, int64_t n_max, int64_t ld_bytes, int64_t batch,
                               const double *h_first_value, int64_t N, int flags, int flexible, double fs,
                               const double *h_fs, int k, int rec_cap, void *h_rec) {
    APDA_TRY(check_wire_args(ctx, h_payload, h_first_value, n_max, ld_bytes, batch, h_rec));
    APDA_TRY(check_fft_args(ctx, h_payload, n_max, n_max, batch, N, flags, h_rec));
    APDA_TRY(check_peaks_args(ctx, h_payload, N, batch, k, rec_cap, h_rec));
    return wire16_host<T>(ctx, h_payload, n_max, ld_bytes, batch, h_first_value, nullptr, nullptr, true, N, flags, flexible, fs,
                          h_fs, k, rec_cap, h_rec);
}
extern "C" int apda_analyze_wire16_f64_host(apda_ctx *ctx, const uint8_t *h_payload, int64_t n_max, int64_t ld_bytes,
                                            int64_t batch, const double *h_first_value, int64_t N, int flags,
                                            int flexible, double fs, const double *h_fs, int k, int rec_cap,
                                            void *h_rec) {
    return analyze_wire16_host<double>(ctx, h_payload, n_max, ld_bytes, batch, h_first_value, N, flags, flexible, fs, h_fs, k,
                                       rec_cap, h_rec);
}
extern "C" int apda_analyze_wire16_f32_host(apda_ctx *ctx, const uint8_t *h_payload, int64_t n_max, int64_t ld_bytes,
                                            int64_t batch, const double *h_first_value, int64_t N, int flags,
                                            int flexible, double fs, const double *h_fs, int k, int rec_cap,
                                            void *h_rec) {
    return analyze_wire16_host<float>(ctx, h_payload, n_max, ld_bytes, batch, h_first_value, N, flags, flexible, fs, h_fs, k,
                                      rec_cap, h_rec);
}

// ---------------------------------------------------------------------------------------------------------------
// text ingest: the sample lines of many sensor logs -> samples (-> records) on the device
// ---------------------------------------------------------------------------------------------------------------
template <typename T>
static int text_host(apda_ctx *ctx, const char *h_text, const int64_t *h_offsets, int64_t batch, int64_t n_max,
                     T *h_samples_out, int32_t *h_n_valid, int32_t *h_flags, bool analyze, int64_t N, int flags,
                     int flexible, double fs, const double *h_fs, int k, int rec_cap, void *h_rec) {
    if (!ctx || !h_text || !h_offsets || !h_n_valid || !h_flags || batch < 0 || batch > 0x7fffffff || n_max < 1) {
        apda_set_error("text ingest: bad arguments");
        return APDA_ERR_INVALID;
    }
    APDA_CUDA(cudaSetDevice(ctx->device));
    if (batch == 0) return APDA_OK;
    const size_t rec_bytes = (size_t)APDA_REC_BYTES(rec_cap);
    const size_t per_window = analyze ? (size_t)N * 2 * sizeof(T) : (size_t)n_max * sizeof(T);
    int64_t chunk = std::max<int64_t>(1, (int64_t)((96u << 20) / per_window));
    chunk = std::min<int64_t>(chunk, batch);
    if (batch > chunk && batch < 2 * chunk) chunk = (batch + 1) / 2;
    size_t max_text = 0;  // largest text span of a chunk
    for (int64_t d = 0; d < batch; d += chunk)
        max_text = std::max<size_t>(max_text, (size_t)(h_offsets[std::min(batch, d + chunk)] - h_offsets[d]));
    const size_t txt_b = align256(max_text + 16), off_b = align256((chunk + 1) * sizeof(int64_t));
    const size_t smp_b = align256(chunk * (size_t)n_max * sizeof(T)), nv_b = align256(chunk * sizeof(int));
    const size_t fl_b = align256(chunk * sizeof(int));
    const size_t spec_b = analyze ? align256(chunk * (size_t)N * 2 * sizeof(T)) : 0;
    const size_t recs_b = analyze ? align256(chunk * rec_bytes) : 0;
    const size_t fs_b = (analyze && h_fs) ? align256(chunk * sizeof(double)) : 0;
    const size_t mag_b = analyze ? align256(peaks_mag_workspace_bytes<T>(ctx, N, chunk)) : 0;
    const size_t total = txt_b + off_b + smp_b + nv_b + fl_b + spec_b + recs_b + fs_b + mag_b;
    for (int s = 0; s < 2; ++s) {
        if (total > ctx->ws_pipe_bytes[s]) {
            APDA_CUDA(cudaStreamSynchronize(ctx->pipe[s]));
            APDA_TRY(apda_reserve(&ctx->ws_pipe[s], &ctx->ws_pipe_bytes[s], total));
        }
        if (batch <= chunk) break;
    }
    // chunk-relative offsets: one host vector per chunk, alive until the drain below (the H2D copies read them
    // asynchronously), so no chunk has to wait for the previous one on its stream
    std::vector<std::vector<int64_t>> rel((size_t)((batch + chunk - 1) / chunk));
    auto run_chunk = [&](int c, int64_t done, int64_t cnt) -> int {  // see host_pipeline: errors never skip the drain
        const int s = c & 1;
        cudaStream_t st = ctx->pipe[s];
        char *base = (char *)ctx->ws_pipe[s];
        char *d_txt = base;
        int64_t *d_off = (int64_t *)(base + txt_b);
        T *d_smp = (T *)(base + txt_b + off_b);
        int *d_nv = (int *)(base + txt_b + off_b + smp_b);
        int *d_fl = (int *)(base + txt_b + off_b + smp_b + nv_b);
        T *d_spec = (T *)(base + txt_b + off_b + smp_b + nv_b + fl_b);
        void *d_rec = base + txt_b + off_b + smp_b + nv_b + fl_b + spec_b;
        double *d_fs = fs_b ? (double *)(base + txt_b + off_b + smp_b + nv_b + fl_b + spec_b + recs_b) : nullptr;
        void *mag_ws = mag_b ? base + txt_b + off_b + smp_b + nv_b + fl_b + spec_b + recs_b + fs_b : nullptr;
        size_t mag_have = mag_b;
        std::vector<int64_t> &r = rel[(size_t)c];
        r.resize((size_t)cnt + 1);
        for (int64_t i = 0; i <= cnt; ++i) r[(size_t)i] = h_offsets[done + i] - h_offsets[done];
        APDA_CUDA(cudaMemcpyAsync(d_txt, h_text + h_offsets[done], (size_t)r[(size_t)cnt], cudaMemcpyHostToDevice, st));
        APDA_CUDA(cudaMemcpyAsync(d_off, r.data(), (size_t)(cnt + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        if (d_fs) APDA_CUDA(cudaMemcpyAsync(d_fs, h_fs + done, cnt * sizeof(double), cudaMemcpyHostToDevice, st));
        APDA_TRY(launch_parse_samples<T>(ctx, st, d_txt, d_off, cnt, n_max, d_smp, d_nv, d_fl));
        if (h_samples_out)
            APDA_CUDA(cudaMemcpyAsync(h_samples_out + (size_t)done * n_max, d_smp, cnt * (size_t)n_max * sizeof(T),
                                      cudaMemcpyDeviceToHost, st));
        APDA_CUDA(cudaMemcpyAsync(h_n_valid + done, d_nv, cnt * sizeof(int), cudaMemcpyDeviceToHost, st));
        APDA_CUDA(cudaMemcpyAsync(h_flags + done, d_fl, cnt * sizeof(int), cudaMemcpyDeviceToHost, st));
        if (analyze) {
            APDA_TRY(analyze_ragged_dev<T>(ctx, st, d_smp, d_nv, n_max, n_max, cnt, N, flags, flexible, fs, d_fs, k, rec_cap,
                                           d_spec, d_rec, &mag_ws, &mag_have, 0));
            APDA_CUDA(cudaMemcpyAsync((char *)h_rec + (size_t)done * rec_bytes, d_rec, cnt * rec_bytes,
                                      cudaMemcpyDeviceToHost, st));
        }
        return APDA_OK;
    };
    int status = APDA_OK;
    int c = 0;
    for (int64_t done = 0; done < batch && status == APDA_OK; ++c) {
        const int64_t cnt = std::min<int64_t>(chunk, batch - done);
        status = run_chunk(c, done, cnt);
        done += cnt;
    }
    cudaError_t e0 = cudaStreamSynchronize(ctx->pipe[0]);
    cudaError_t e1 = cudaStreamSynchronize(ctx->pipe[1]);
    if (status != APDA_OK) return status;
    if (e0 != cudaSuccess) return apda_cuda_fail(e0, "text pipeline (stream 0)");
    if (e1 != cudaSuccess) return apda_cuda_fail(e1, "text pipeline (stream 1)");
    return APDA_OK;
}

extern "C" int apda_parse_samples_f64_host(apda_ctx *ctx, const char *h_text, const int64_t *h_offsets, int64_t batch,
                                           int64_t n_max, double *h_samples, int32_t *h_n_valid, int32_t *h_flags) {
    if (!h_samples) {
        apda_set_error("parse_samples: output is NULL");
        return APDA_ERR_INVALID;
    }
    return text_host<double>(ctx, h_text, h_offsets, batch, n_max, h_samples, h_n_valid, h_flags, false, 0, 0, 0, 0.0, nullptr,
                             1, 5, nullptr);
}
template <typename T>
static int analyze_text_host(apda_ctx *ctx, const char *h_text, const int64_t *h_offsets, int64_t batch, int64_t n_max,
                             int64_t N, int flags, int flexible, double fs, const double *h_fs, int k, int rec_cap,
                             void *h_rec, int32_t *h_n_valid, int32_t *h_flags) {
    APDA_TRY(check_fft_args(ctx, h_text, n_max, n_max, batch, N, flags, h_rec));
    APDA_TRY(check_peaks_args(ctx, h_text, N, batch, k, rec_cap, h_rec));
    return text_host<T>(ctx, h_text, h_offsets, batch, n_max, nullptr, h_n_valid, h_flags, true, N, flags, flexible, fs, h_fs, k,
                        rec_cap, h_rec);
}
extern "C" int apda_analyze_text_f64_host(apda_ctx *ctx, const char *h_text, const int64_t *h_offsets, int64_t batch,
                                          int64_t n_max, int64_t N, int flags, int flexible, double fs,
                                          const double *h_fs, int k, int rec_cap, void *h_rec, int32_t *h_n_valid,
                                          int32_t *h_flags) {
    return analyze_text_host<double>(ctx, h_text, h_offsets, batch, n_max, N, flags, flexible, fs, h_fs, k, rec_cap, h_rec,
                                     h_n_valid, h_flags);
}
extern "C" int apda_analyze_text_f32_host(apda_ctx *ctx, const char *h_text, const int64_t *h_offsets, int64_t batch,
                                          int64_t n_max, int64_t N, int flags, int flexible, double fs,
                                          const double *h_fs, int k, int rec_cap, void *h_rec, int32_t *h_n_valid,
                                          int32_t *h_flags) {
    return analyze_text_host<float>(ctx, h_text, h_offsets, batch, n_max, N, flags, flexible, fs, h_fs, k, rec_cap, h_rec,
                                    h_n_valid, h_flags);
}

// ---------------------------------------------------------------------------------------------------------------
// whole sensor logs: paths -> file bytes in pinned staging (reader threads) -> header layout, samples, records on the
// device.  The host never looks inside a file.
// ---------------------------------------------------------------------------------------------------------------
namespace {

// Fork-join reader threads: run(n, fn) calls fn(0 .. n-1) on min(16, hardware threads, n) threads and returns at
// once; join() (also run by the destructor, so every error path joins) waits for them.  A thread that cannot be
// created leaves its share to the others; with none at all the caller's thread does the work inside run().
class ReaderThreads {
   public:
    ~ReaderThreads() { join(); }
    void run(int64_t n, std::function<void(int64_t)> fn) {
        join();
        next_ = 0;
        n_ = n;
        fn_ = std::move(fn);
        const unsigned hw = std::thread::hardware_concurrency();
        const int64_t want = std::min<int64_t>(n, std::min(16u, hw ? hw : 1u));
        for (int64_t i = 0; i < want; ++i) {
            try {
                threads_.emplace_back([this] { work(); });
            } catch (...) {
                break;
            }
        }
        if (threads_.empty()) work();
    }
    void join() {
        for (auto &t : threads_) t.join();
        threads_.clear();
    }

   private:
    void work() {
        for (int64_t i; (i = next_.fetch_add(1)) < n_;) fn_(i);
    }
    std::atomic<int64_t> next_{0};
    int64_t n_ = 0;
    std::function<void(int64_t)> fn_;
    std::vector<std::thread> threads_;
};

// size of a regular file, or -1 (missing, unreadable, directory, device, fifo ...)
int64_t log_file_size(const char *path) {
    struct stat sb;
    if (stat(path, &sb) != 0 || !S_ISREG(sb.st_mode)) return -1;
    return (int64_t)sb.st_size;
}

// the whole file into dst; false unless it is still a regular file of exactly `size` bytes and every byte was read
bool read_log_file(const char *path, char *dst, int64_t size) {
    const int fd = open(path, O_RDONLY | O_CLOEXEC | O_NONBLOCK);
    if (fd < 0) return false;
    struct stat sb;
    bool ok = fstat(fd, &sb) == 0 && S_ISREG(sb.st_mode) && (int64_t)sb.st_size == size;
    for (int64_t got = 0; ok && got < size;) {
        const ssize_t r = pread(fd, dst + got, (size_t)(size - got), (off_t)got);
        if (r < 0 && errno == EINTR) continue;
        if (r <= 0) ok = false;
        else got += r;
    }
    close(fd);
    return ok;
}

int reserve_pinned(cudaStream_t user, void **buf, size_t *have, size_t need) {
    if (need <= *have) return APDA_OK;
    APDA_CUDA(cudaStreamSynchronize(user));  // the old buffer may still feed a copy on this stream
    if (*buf) APDA_CUDA(cudaFreeHost(*buf));
    *buf = nullptr;
    *have = 0;
    const cudaError_t e = cudaHostAlloc(buf, need, cudaHostAllocDefault);
    if (e != cudaSuccess) {
        *buf = nullptr;
        apda_set_error("cudaHostAlloc(%zu) failed: %s", need, cudaGetErrorString(e));
        (void)cudaGetLastError();
        return APDA_ERR_NOMEM;
    }
    *have = need;
    return APDA_OK;
}

}  // namespace

// a chunk holds at most this many file bytes (a larger file is a chunk of its own)
static const int64_t kLogChunkBytes = int64_t(64) << 20;

template <typename T>
static int analyze_logs_host(apda_ctx *ctx, const char *const *paths, int64_t n_files, int64_t N, int flags, int flexible,
                             int k, int rec_cap, void *h_rec, double *h_fs, int32_t *h_n_valid, int32_t *h_flags,
                             char *h_head) {
    if (!ctx || !paths || !h_rec || !h_fs || !h_n_valid || !h_flags || !h_head || n_files < 0 || n_files > 0x7fffffff) {
        apda_set_error("analyze_logs: bad arguments (NULL buffer or n_files out of range)");
        return APDA_ERR_INVALID;
    }
    if (!is_pow2_i64(N) || N < 4 || N > fft_smem_max_n<T>(ctx)) {
        apda_set_error("analyze_logs: N=%lld must be a power of two in [4, %lld]", (long long)N,
                       (long long)fft_smem_max_n<T>(ctx));
        return APDA_ERR_INVALID;
    }
    if (flags != APDA_CENTER_MEDIAN && flags != APDA_CENTER_NONE) {
        apda_set_error("analyze_logs: flags must be APDA_CENTER_MEDIAN or APDA_CENTER_NONE");
        return APDA_ERR_INVALID;
    }
    APDA_TRY(check_peaks_args(ctx, h_rec, N, n_files, k, rec_cap, h_rec));
    for (int64_t b = 0; b < n_files; ++b)
        if (!paths[b]) {
            apda_set_error("analyze_logs: paths[%lld] is NULL", (long long)b);
            return APDA_ERR_INVALID;
        }
    APDA_CUDA(cudaSetDevice(ctx->device));
    if (n_files == 0) return APDA_OK;
    const size_t rec_bytes = (size_t)APDA_REC_BYTES(rec_cap);

    ReaderThreads readers;
    std::vector<int64_t> size((size_t)n_files);
    readers.run(n_files, [&](int64_t b) { size[(size_t)b] = log_file_size(paths[b]); });
    readers.join();

    // chunks: at most kLogChunkBytes of text and as many files as ~96 MB of spectra hold
    const int64_t max_files = std::max<int64_t>(1, (int64_t)((96u << 20) / ((size_t)N * 2 * sizeof(T))));
    std::vector<int64_t> first;  // first file of every chunk, then n_files
    int64_t max_text = 0, max_cnt = 0;
    for (int64_t b = 0, bytes = 0; b < n_files; ++b) {
        const int64_t s = std::max<int64_t>(size[(size_t)b], 0);
        if (first.empty() || b - first.back() == max_files || (b > first.back() && bytes + s > kLogChunkBytes)) {
            first.push_back(b);
            bytes = 0;
        }
        bytes += s;
        max_text = std::max(max_text, bytes);
        max_cnt = std::max(max_cnt, b - first.back() + 1);
    }
    first.push_back(n_files);
    const int64_t n_chunks = (int64_t)first.size() - 1;

    // device workspace of one chunk (per stream) and pinned staging: text, then the chunk-relative offsets
    const size_t txt_b = align256((size_t)max_text + 16), off_b = align256((size_t)(max_cnt + 1) * sizeof(int64_t));
    const size_t start_b = align256((size_t)max_cnt * sizeof(int64_t)), fs_b = align256((size_t)max_cnt * sizeof(double));
    const size_t int_b = align256((size_t)max_cnt * sizeof(int)), head_b = align256((size_t)max_cnt * APDA_LOG_HEAD_BYTES);
    const size_t smp_b = align256((size_t)max_cnt * (size_t)N * sizeof(T));
    const size_t spec_b = align256((size_t)max_cnt * (size_t)N * 2 * sizeof(T)), recs_b = align256((size_t)max_cnt * rec_bytes);
    const size_t mag_b = align256(peaks_mag_workspace_bytes<T>(ctx, N, max_cnt));
    const size_t total = txt_b + off_b + start_b + fs_b + 3 * int_b + head_b + smp_b + spec_b + recs_b + mag_b;
    for (int s = 0; s < 2 && s < n_chunks; ++s) {
        if (total > ctx->ws_pipe_bytes[s]) {
            APDA_CUDA(cudaStreamSynchronize(ctx->pipe[s]));
            APDA_TRY(apda_reserve(&ctx->ws_pipe[s], &ctx->ws_pipe_bytes[s], total));
        }
        APDA_TRY(reserve_pinned(ctx->pipe[s], &ctx->log_stage[s], &ctx->log_stage_bytes[s], txt_b + off_b));
    }

    std::vector<char> unread((size_t)n_files, 0);
    // reader threads put chunk c's files into staging buffer c & 1 (returns at once; readers.join() waits)
    auto fill = [&](int64_t c) {
        char *stage = (char *)ctx->log_stage[c & 1];
        int64_t *off = (int64_t *)(stage + txt_b);
        const int64_t lo = first[(size_t)c], cnt = first[(size_t)c + 1] - lo;
        off[0] = 0;
        for (int64_t i = 0; i < cnt; ++i) off[i + 1] = off[i] + std::max<int64_t>(size[(size_t)(lo + i)], 0);
        readers.run(cnt, [&, stage, off, lo](int64_t i) {
            const int64_t b = lo + i;
            if (size[(size_t)b] < 0 || !read_log_file(paths[b], stage + off[i], size[(size_t)b])) unread[(size_t)b] = 1;
        });
    };
    auto run_chunk = [&](int64_t c) -> int {  // see host_pipeline: errors never skip the drain
        const int s = (int)(c & 1);
        cudaStream_t st = ctx->pipe[s];
        const int64_t lo = first[(size_t)c], cnt = first[(size_t)c + 1] - lo;
        const char *stage = (const char *)ctx->log_stage[s];
        const int64_t *off = (const int64_t *)(stage + txt_b);
        char *p = (char *)ctx->ws_pipe[s];
        char *d_txt = p;                   p += txt_b;
        int64_t *d_off = (int64_t *)p;     p += off_b;
        int64_t *d_start = (int64_t *)p;   p += start_b;
        double *d_fs = (double *)p;        p += fs_b;
        int *d_fl = (int *)p;              p += int_b;
        int *d_pfl = (int *)p;             p += int_b;
        int *d_nv = (int *)p;              p += int_b;
        char *d_head = p;                  p += head_b;
        T *d_smp = (T *)p;                 p += smp_b;
        T *d_spec = (T *)p;                p += spec_b;
        void *d_rec = p;                   p += recs_b;
        void *mag_ws = mag_b ? (void *)p : nullptr;
        size_t mag_have = mag_b;
        APDA_CUDA(cudaMemcpyAsync(d_txt, stage, (size_t)off[cnt], cudaMemcpyHostToDevice, st));
        APDA_CUDA(cudaMemcpyAsync(d_off, off, (size_t)(cnt + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        APDA_TRY(launch_log_layout(ctx, st, d_txt, d_off, cnt, d_start, d_fs, d_fl, d_head));
        APDA_TRY(launch_parse_samples<T>(ctx, st, d_txt, d_off, cnt, N, d_smp, d_nv, d_pfl, d_start));
        APDA_TRY(analyze_ragged_dev<T>(ctx, st, d_smp, d_nv, N, N, cnt, N, flags, flexible, 0.0, d_fs, k, rec_cap, d_spec,
                                       d_rec, &mag_ws, &mag_have, 0));
        APDA_TRY(launch_log_finish(ctx, st, cnt, d_fl, d_pfl, d_rec, rec_cap));
        APDA_CUDA(cudaMemcpyAsync((char *)h_rec + (size_t)lo * rec_bytes, d_rec, (size_t)cnt * rec_bytes,
                                  cudaMemcpyDeviceToHost, st));
        APDA_CUDA(cudaMemcpyAsync(h_fs + lo, d_fs, (size_t)cnt * sizeof(double), cudaMemcpyDeviceToHost, st));
        APDA_CUDA(cudaMemcpyAsync(h_n_valid + lo, d_nv, (size_t)cnt * sizeof(int), cudaMemcpyDeviceToHost, st));
        APDA_CUDA(cudaMemcpyAsync(h_flags + lo, d_fl, (size_t)cnt * sizeof(int), cudaMemcpyDeviceToHost, st));
        APDA_CUDA(cudaMemcpyAsync(h_head + (size_t)lo * APDA_LOG_HEAD_BYTES, d_head, (size_t)cnt * APDA_LOG_HEAD_BYTES,
                                  cudaMemcpyDeviceToHost, st));
        return APDA_OK;
    };
    fill(0);
    readers.join();
    int status = APDA_OK;
    for (int64_t c = 0; c < n_chunks && status == APDA_OK; ++c) {
        if (c + 1 < n_chunks) {
            // staging buffer (c + 1) & 1 fed chunk c - 1, whose copies were enqueued on the same stream
            const cudaError_t e = cudaStreamSynchronize(ctx->pipe[(c + 1) & 1]);
            if (e != cudaSuccess) {
                status = apda_cuda_fail(e, "analyze_logs (staging reuse)");
                break;
            }
            fill(c + 1);
        }
        status = run_chunk(c);
        readers.join();
    }
    readers.join();
    cudaError_t e0 = cudaStreamSynchronize(ctx->pipe[0]);
    cudaError_t e1 = cudaStreamSynchronize(ctx->pipe[1]);
    if (status != APDA_OK) return status;
    if (e0 != cudaSuccess) return apda_cuda_fail(e0, "analyze_logs (stream 0)");
    if (e1 != cudaSuccess) return apda_cuda_fail(e1, "analyze_logs (stream 1)");
    for (int64_t b = 0; b < n_files; ++b) {
        if (!unread[(size_t)b]) continue;
        h_flags[b] = 16;
        h_fs[b] = 0.0;
        h_n_valid[b] = 0;
        memset(h_head + (size_t)b * APDA_LOG_HEAD_BYTES, 0, APDA_LOG_HEAD_BYTES);
        char *rec = (char *)h_rec + (size_t)b * rec_bytes;  // the empty record, status 0
        const int32_t hdr[2] = {0, 0};
        const apda_peak none{-1, 0, 0.0, 0.0};
        memcpy(rec, hdr, sizeof(hdr));
        for (int i = 0; i < rec_cap; ++i) memcpy(rec + 8 + (size_t)i * sizeof(apda_peak), &none, sizeof(none));
    }
    return APDA_OK;
}
extern "C" int apda_analyze_logs_f64_host(apda_ctx *ctx, const char *const *paths, int64_t n_files, int64_t N, int flags,
                                          int flexible, int k, int rec_cap, void *h_rec, double *h_fs, int32_t *h_n_valid,
                                          int32_t *h_flags, char *h_head) {
    return analyze_logs_host<double>(ctx, paths, n_files, N, flags, flexible, k, rec_cap, h_rec, h_fs, h_n_valid, h_flags,
                                     h_head);
}
extern "C" int apda_analyze_logs_f32_host(apda_ctx *ctx, const char *const *paths, int64_t n_files, int64_t N, int flags,
                                          int flexible, int k, int rec_cap, void *h_rec, double *h_fs, int32_t *h_n_valid,
                                          int32_t *h_flags, char *h_head) {
    return analyze_logs_host<float>(ctx, paths, n_files, N, flags, flexible, k, rec_cap, h_rec, h_fs, h_n_valid, h_flags,
                                    h_head);
}

// ---------------------------------------------------------------------------------------------------------------
// record presentation: the reference's rounded peak fields and the fleet JSONL rows, computed on the device
// ---------------------------------------------------------------------------------------------------------------
static int check_present_args(apda_ctx *ctx, const void *rec, int rec_cap, int64_t batch, int64_t n, int k,
                              int64_t first_window) {
    if (!ctx || !rec) {
        apda_set_error("present: NULL context or records");
        return APDA_ERR_INVALID;
    }
    if ((uintptr_t)rec % 8) {
        apda_set_error("present: records must be 8-byte aligned");
        return APDA_ERR_INVALID;
    }
    if (!is_pow2_i64(n) || n < 4 || n > (int64_t(1) << 30)) {
        apda_set_error("present: n=%lld must be a power of two in [4, 2^30]", (long long)n);
        return APDA_ERR_INVALID;
    }
    if (rec_cap < 1 || (rec_cap > APDA_MAX_REC_CAP && (int64_t)rec_cap > APDA_MAX_PEAKS(n))) {
        apda_set_error("present: need 1 <= rec_cap (%d) <= max(%d, n/8 + 8 = %lld)", rec_cap, APDA_MAX_REC_CAP,
                       (long long)APDA_MAX_PEAKS(n));
        return APDA_ERR_INVALID;
    }
    if (k < 1 || k > rec_cap) {
        apda_set_error("present: need 1 <= k (%d) <= rec_cap (%d)", k, rec_cap);
        return APDA_ERR_INVALID;
    }
    if (batch < 0 || batch > 0x7fffffff) {
        apda_set_error("present: batch %lld out of range", (long long)batch);
        return APDA_ERR_INVALID;
    }
    if (first_window < 0 || first_window > INT64_MAX - batch) {
        apda_set_error("present: first_window %lld must be >= 0 and first_window + batch must fit int64",
                       (long long)first_window);
        return APDA_ERR_INVALID;
    }
    return APDA_OK;
}

extern "C" int apda_present_dev(apda_ctx *ctx, const void *d_rec, int rec_cap, int64_t batch, int64_t n, double fs,
                                const double *d_fs, int flexible, int k, int32_t *d_idx, double *d_freq, double *d_mag,
                                double *d_prominence, double *d_damping, double *d_q) {
    APDA_TRY(check_present_args(ctx, d_rec, rec_cap, batch, n, k, 0));
    APDA_CUDA(cudaSetDevice(ctx->device));
    return launch_present_columns(ctx, ctx->stream, d_rec, rec_cap, batch, n, fs, d_fs, flexible, k, d_idx, d_freq, d_mag,
                                  d_prominence, d_damping, d_q);
}

extern "C" int apda_present_host(apda_ctx *ctx, const void *h_rec, int rec_cap, int64_t batch, int64_t n, double fs,
                                 const double *h_fs, int flexible, int k, int32_t *h_idx, double *h_freq, double *h_mag,
                                 double *h_prominence, double *h_damping, double *h_q) {
    APDA_TRY(check_present_args(ctx, h_rec, rec_cap, batch, n, k, 0));
    APDA_CUDA(cudaSetDevice(ctx->device));
    if (batch == 0) return APDA_OK;
    double *h_col[5] = {h_freq, h_mag, h_prominence, h_damping, h_q};
    int ncol = 0;
    for (double *c : h_col) ncol += c != nullptr;
    const size_t rec_bytes = (size_t)APDA_REC_BYTES(rec_cap);
    const size_t per_window = rec_bytes + (h_fs ? 8 : 0) + (size_t)k * ((h_idx ? 4 : 0) + 8 * ncol);
    // chunk: ~64 MB of staging per stream, at least one window
    int64_t chunk = std::min<int64_t>(batch, std::max<int64_t>(1, (int64_t)((64u << 20) / per_window)));
    if (batch > chunk && batch < 2 * chunk) chunk = (batch + 1) / 2;
    const size_t rec_b = align256((size_t)chunk * rec_bytes), fs_b = h_fs ? align256((size_t)chunk * 8) : 0;
    const size_t idx_b = h_idx ? align256((size_t)chunk * k * 4) : 0, col_b = align256((size_t)chunk * k * 8);
    const size_t total = rec_b + fs_b + idx_b + col_b * ncol;
    for (int s = 0; s < 2; ++s) {
        if (total > ctx->ws_pipe_bytes[s]) {
            APDA_CUDA(cudaStreamSynchronize(ctx->pipe[s]));
            APDA_TRY(apda_reserve(&ctx->ws_pipe[s], &ctx->ws_pipe_bytes[s], total));
        }
        if (batch <= chunk) break;
    }
    // an error returns from the lambda only, so both streams are drained before the caller's buffers are released
    auto run_chunk = [&](int c, int64_t done, int64_t cnt) -> int {
        cudaStream_t st = ctx->pipe[c & 1];
        char *base = (char *)ctx->ws_pipe[c & 1];
        void *d_rec = base;
        double *d_fs = h_fs ? (double *)(base + rec_b) : nullptr;
        int32_t *d_idx = h_idx ? (int32_t *)(base + rec_b + fs_b) : nullptr;
        double *d_col[5] = {};
        char *p = base + rec_b + fs_b + idx_b;
        for (int i = 0; i < 5; ++i)
            if (h_col[i]) {
                d_col[i] = (double *)p;
                p += col_b;
            }
        APDA_CUDA(cudaMemcpyAsync(d_rec, (const char *)h_rec + (size_t)done * rec_bytes, (size_t)cnt * rec_bytes,
                                  cudaMemcpyHostToDevice, st));
        if (d_fs) APDA_CUDA(cudaMemcpyAsync(d_fs, h_fs + done, (size_t)cnt * 8, cudaMemcpyHostToDevice, st));
        APDA_TRY(launch_present_columns(ctx, st, d_rec, rec_cap, cnt, n, fs, d_fs, flexible, k, d_idx, d_col[0], d_col[1],
                                        d_col[2], d_col[3], d_col[4]));
        const size_t slots = (size_t)cnt * k, first = (size_t)done * k;
        if (h_idx) APDA_CUDA(cudaMemcpyAsync(h_idx + first, d_idx, slots * 4, cudaMemcpyDeviceToHost, st));
        for (int i = 0; i < 5; ++i)
            if (h_col[i]) APDA_CUDA(cudaMemcpyAsync(h_col[i] + first, d_col[i], slots * 8, cudaMemcpyDeviceToHost, st));
        return APDA_OK;
    };
    int status = APDA_OK;
    int c = 0;
    for (int64_t done = 0; done < batch && status == APDA_OK; ++c) {
        const int64_t cnt = std::min<int64_t>(chunk, batch - done);
        status = run_chunk(c, done, cnt);
        done += cnt;
    }
    cudaError_t e0 = cudaStreamSynchronize(ctx->pipe[0]);
    cudaError_t e1 = cudaStreamSynchronize(ctx->pipe[1]);
    if (status != APDA_OK) return status;
    if (e0 != cudaSuccess) return apda_cuda_fail(e0, "present_host (stream 0)");
    if (e1 != cudaSuccess) return apda_cuda_fail(e1, "present_host (stream 1)");
    return APDA_OK;
}

extern "C" int apda_fleet_jsonl_dev(apda_ctx *ctx, const void *d_rec, int rec_cap, int64_t batch, int64_t n, double fs,
                                    const double *d_fs, int flexible, int k, int64_t first_window, char *d_text,
                                    int64_t text_cap, int64_t *d_offsets) {
    APDA_TRY(check_present_args(ctx, d_rec, rec_cap, batch, n, k, first_window));
    if (!d_text || !d_offsets) {
        apda_set_error("fleet_jsonl: NULL text or offsets");
        return APDA_ERR_INVALID;
    }
    // the exact size is only known on the device: the buffer must hold the bound of every row
    if (text_cap < 0 || text_cap / APDA_JSONL_ROW_BYTES(k) < batch) {
        apda_set_error("fleet_jsonl_dev: text_cap %lld < batch (%lld) * APDA_JSONL_ROW_BYTES(%d) = %lld bytes",
                       (long long)text_cap, (long long)batch, k, (long long)(batch * APDA_JSONL_ROW_BYTES(k)));
        return APDA_ERR_INVALID;
    }
    APDA_CUDA(cudaSetDevice(ctx->device));
    if (batch == 0) return APDA_OK;
    auto &l = ctx->stream_lists[ctx->stream];
    const size_t need = fleet_jsonl_scratch_bytes(batch);
    if (need > l.jsonl_bytes) {
        APDA_CUDA(cudaStreamSynchronize(ctx->stream));  // the old scratch may still be in use on this stream
        APDA_TRY(apda_reserve((void **)&l.jsonl, &l.jsonl_bytes, need));
    }
    return launch_fleet_jsonl(ctx, ctx->stream, d_rec, rec_cap, batch, n, fs, d_fs, flexible, k, first_window, d_text,
                              d_offsets, l.jsonl);
}

extern "C" int apda_fleet_jsonl_host(apda_ctx *ctx, const void *h_rec, int rec_cap, int64_t batch, int64_t n, double fs,
                                     const double *h_fs, int flexible, int k, int64_t first_window, char *h_text,
                                     int64_t text_cap, int64_t *h_offsets) {
    APDA_TRY(check_present_args(ctx, h_rec, rec_cap, batch, n, k, first_window));
    if (!h_text || !h_offsets || text_cap < 0) {
        apda_set_error("fleet_jsonl: NULL text or offsets, or text_cap < 0");
        return APDA_ERR_INVALID;
    }
    APDA_CUDA(cudaSetDevice(ctx->device));
    h_offsets[0] = 0;
    if (batch == 0) return APDA_OK;
    const size_t rec_bytes = (size_t)APDA_REC_BYTES(rec_cap), row_bytes = (size_t)APDA_JSONL_ROW_BYTES(k);
    const size_t per_window = rec_bytes + (h_fs ? 8 : 0) + 8 + row_bytes;
    const int64_t chunk = std::min<int64_t>(batch, std::max<int64_t>(1, (int64_t)((96u << 20) / per_window)));
    const size_t rec_b = align256((size_t)chunk * rec_bytes), fs_b = h_fs ? align256((size_t)chunk * 8) : 0;
    const size_t off_b = align256((size_t)(chunk + 1) * 8), scan_b = align256(fleet_jsonl_scratch_bytes(chunk));
    const size_t total = rec_b + fs_b + off_b + scan_b + (size_t)chunk * row_bytes;
    cudaStream_t st = ctx->pipe[0];
    if (total > ctx->ws_pipe_bytes[0]) {
        APDA_CUDA(cudaStreamSynchronize(st));
        APDA_TRY(apda_reserve(&ctx->ws_pipe[0], &ctx->ws_pipe_bytes[0], total));
    }
    char *base = (char *)ctx->ws_pipe[0];
    void *d_rec = base;
    double *d_fs = h_fs ? (double *)(base + rec_b) : nullptr;
    int64_t *d_off = (int64_t *)(base + rec_b + fs_b);
    int64_t *d_scan = (int64_t *)(base + rec_b + fs_b + off_b);
    char *d_text = base + rec_b + fs_b + off_b + scan_b;
    std::vector<int64_t> off((size_t)chunk + 1);
    // one chunk at a time: its rows' total decides whether (and where) its text may be copied out; every error path
    // drains the stream before the host buffers go
    int64_t written = 0;
    for (int64_t done = 0; done < batch;) {
        const int64_t cnt = std::min<int64_t>(chunk, batch - done);
        int status = [&]() -> int {
            APDA_CUDA(cudaMemcpyAsync(d_rec, (const char *)h_rec + (size_t)done * rec_bytes, (size_t)cnt * rec_bytes,
                                      cudaMemcpyHostToDevice, st));
            if (d_fs) APDA_CUDA(cudaMemcpyAsync(d_fs, h_fs + done, (size_t)cnt * 8, cudaMemcpyHostToDevice, st));
            APDA_TRY(launch_fleet_jsonl(ctx, st, d_rec, rec_cap, cnt, n, fs, d_fs, flexible, k, first_window + done,
                                        d_text, d_off, d_scan));
            APDA_CUDA(cudaMemcpyAsync(off.data(), d_off, (size_t)(cnt + 1) * 8, cudaMemcpyDeviceToHost, st));
            return APDA_OK;
        }();
        cudaError_t e = cudaStreamSynchronize(st);
        if (status != APDA_OK) return status;
        if (e != cudaSuccess) return apda_cuda_fail(e, "fleet_jsonl_host");
        if (off[(size_t)cnt] > text_cap - written) {
            apda_set_error("fleet_jsonl_host: text_cap %lld is smaller than the %lld bytes of rows 0 .. %lld",
                           (long long)text_cap, (long long)(written + off[(size_t)cnt]), (long long)(done + cnt - 1));
            return APDA_ERR_INVALID;
        }
        status = [&]() -> int {
            APDA_CUDA(cudaMemcpyAsync(h_text + written, d_text, (size_t)off[(size_t)cnt], cudaMemcpyDeviceToHost, st));
            return APDA_OK;
        }();
        e = cudaStreamSynchronize(st);
        if (status != APDA_OK) return status;
        if (e != cudaSuccess) return apda_cuda_fail(e, "fleet_jsonl_host");
        for (int64_t i = 1; i <= cnt; ++i) h_offsets[done + i] = written + off[(size_t)i];
        written += off[(size_t)cnt];
        done += cnt;
    }
    return APDA_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// small helpers on host lists
// ---------------------------------------------------------------------------------------------------------------
extern "C" int apda_center_f64_host(apda_ctx *ctx, const double *h_in, int64_t n, double *h_out) {
    if (!ctx || !h_in || !h_out || n < 1 || n > (int64_t(1) << 28)) {
        apda_set_error("center: bad arguments");
        return APDA_ERR_INVALID;
    }
    APDA_CUDA(cudaSetDevice(ctx->device));
    APDA_TRY(apda_reserve(&ctx->ws_small, &ctx->ws_small_bytes, (size_t)n * 3 * sizeof(double)));
    double *d_in = (double *)ctx->ws_small, *d_out = d_in + n;
    cudaStream_t st = ctx->pipe[0];
    APDA_CUDA(cudaMemcpyAsync(d_in, h_in, n * sizeof(double), cudaMemcpyHostToDevice, st));
    APDA_TRY(launch_center_f64(ctx, st, d_in, n, d_out));
    APDA_CUDA(cudaMemcpyAsync(h_out, d_out, n * sizeof(double), cudaMemcpyDeviceToHost, st));
    APDA_CUDA(cudaStreamSynchronize(st));
    return APDA_OK;
}

static int mag_helpers(apda_ctx *ctx, const double *h_mags, int64_t n, int64_t idx, double prom_in, double out3[3]) {
    if (!ctx || !h_mags || n < 1 || idx < 0 || idx >= n || n > (int64_t(1) << 30)) {
        apda_set_error("magnitude helper: bad arguments (n=%lld idx=%lld)", (long long)n, (long long)idx);
        return APDA_ERR_INVALID;
    }
    APDA_CUDA(cudaSetDevice(ctx->device));
    APDA_TRY(apda_reserve(&ctx->ws_small, &ctx->ws_small_bytes, (size_t)(n + 4) * sizeof(double)));
    double *d_mags = (double *)ctx->ws_small, *d_out = d_mags + n;
    cudaStream_t st = ctx->pipe[0];
    APDA_CUDA(cudaMemcpyAsync(d_mags, h_mags, n * sizeof(double), cudaMemcpyHostToDevice, st));
    APDA_TRY(launch_mag_helpers_f64(ctx, st, d_mags, n, idx, prom_in, d_out));
    APDA_CUDA(cudaMemcpyAsync(out3, d_out, 3 * sizeof(double), cudaMemcpyDeviceToHost, st));
    APDA_CUDA(cudaStreamSynchronize(st));
    return APDA_OK;
}
extern "C" int apda_prominence_f64_host(apda_ctx *ctx, const double *h_mags, int64_t n, int64_t idx, double *out) {
    double r[3];
    APDA_TRY(mag_helpers(ctx, h_mags, n, idx, 0.0, r));
    *out = r[0];
    return APDA_OK;
}
extern "C" int apda_half_power_bins_f64_host(apda_ctx *ctx, const double *h_mags, int64_t n, double prominence,
                                             int64_t idx, int64_t *bins) {
    double r[3];
    APDA_TRY(mag_helpers(ctx, h_mags, n, idx, prominence, r));
    *bins = (int64_t)r[1];
    return APDA_OK;
}
extern "C" int apda_half_height_bins_f64_host(apda_ctx *ctx, const double *h_mags, int64_t n, int64_t idx,
                                              int64_t *bins) {
    double r[3];
    APDA_TRY(mag_helpers(ctx, h_mags, n, idx, 0.0, r));
    *bins = (int64_t)r[2];
    return APDA_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// synthetic input
// ---------------------------------------------------------------------------------------------------------------
extern "C" int apda_synth_f64_dev(apda_ctx *ctx, int64_t first_window, int64_t count, int64_t N, uint64_t seed,
                                  int on_bin, double *d_out) {
    if (!ctx || !d_out || count < 0 || N < 2) return APDA_ERR_INVALID;
    APDA_CUDA(cudaSetDevice(ctx->device));
    return launch_synth<double>(ctx, ctx->stream, first_window, count, N, seed, on_bin, d_out);
}
extern "C" int apda_synth_f32_dev(apda_ctx *ctx, int64_t first_window, int64_t count, int64_t N, uint64_t seed,
                                  int on_bin, float *d_out) {
    if (!ctx || !d_out || count < 0 || N < 2) return APDA_ERR_INVALID;
    APDA_CUDA(cudaSetDevice(ctx->device));
    return launch_synth<float>(ctx, ctx->stream, first_window, count, N, seed, on_bin, d_out);
}

// ---------------------------------------------------------------------------------------------------------------
// fleet record table in peer memory (SURVEY 8e): rank 0 owns one table for the whole fleet; every other rank maps it
// through CUDA IPC and its K3 kernels store their 128-byte records straight into their rows over NVLink - the
// "gather" is fused into the producing kernel's epilogue store and needs no collective, no staging copy and no SMs.
// ---------------------------------------------------------------------------------------------------------------
extern "C" int apda_peer_table_create(apda_ctx *ctx, int64_t bytes, void **d_table, unsigned char *handle64) {
    if (!ctx || !d_table || !handle64 || bytes <= 0) return APDA_ERR_INVALID;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size is part of the ABI");
    APDA_CUDA(cudaSetDevice(ctx->device));
    void *p = nullptr;
    APDA_CUDA(cudaMalloc(&p, (size_t)bytes));
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) {
        cudaFree(p);
        return apda_cuda_fail(e, "cudaIpcGetMemHandle");
    }
    memcpy(handle64, &h, 64);
    *d_table = p;
    return APDA_OK;
}
extern "C" int apda_peer_table_open(apda_ctx *ctx, const unsigned char *handle64, void **d_table) {
    if (!ctx || !d_table || !handle64) return APDA_ERR_INVALID;
    APDA_CUDA(cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    void *p = nullptr;
    APDA_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    *d_table = p;
    return APDA_OK;
}
extern "C" int apda_peer_table_close(apda_ctx *ctx, void *d_table) {
    if (!ctx || !d_table) return APDA_ERR_INVALID;
    APDA_CUDA(cudaSetDevice(ctx->device));
    APDA_CUDA(cudaIpcCloseMemHandle(d_table));
    return APDA_OK;
}
extern "C" int apda_peer_table_destroy(apda_ctx *ctx, void *d_table) {
    if (!ctx || !d_table) return APDA_ERR_INVALID;
    APDA_CUDA(cudaSetDevice(ctx->device));
    APDA_CUDA(cudaFree(d_table));
    return APDA_OK;
}

// Completion flags of the peer table: one 32-bit step counter per rank, living in the owner's memory next to the rows.
// A producer rank enqueues apda_peer_signal after its pickers (release at system scope: the records it stored over
// NVLink are visible before the flag), the owner enqueues apda_peer_wait (acquire) before it consumes the table - the
// whole exchange stays on the device timelines, no host synchronisation, no collective.
namespace {
__global__ void peer_signal_kernel(unsigned *flag, unsigned value) {
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(flag), "r"(value) : "memory");
}
__global__ void peer_wait_kernel(const unsigned *flags, int world, unsigned value, long long timeout_cycles,
                                 int *timed_out) {
    const int r = threadIdx.x;
    if (r == 0) *timed_out = 0;  // the word reports THIS wait, not an earlier one
    __syncwarp();
    if (r >= world) return;
    const long long t0 = clock64();
    while (true) {
        unsigned v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + r) : "memory");
        if ((int)(v - value) >= 0) break;
        if (clock64() - t0 > timeout_cycles) {  // a peer died: never hang the device
            atomicExch(timed_out, 1);
            break;
        }
        __nanosleep(200);
    }
}
}  // namespace

extern "C" int apda_peer_signal(apda_ctx *ctx, void *d_flag, uint32_t value) {
    if (!ctx || !d_flag) return APDA_ERR_INVALID;
    APDA_CUDA(cudaSetDevice(ctx->device));
    peer_signal_kernel<<<1, 1, 0, ctx->stream>>>(reinterpret_cast<unsigned *>(d_flag), value);
    ctx->launches++;
    APDA_CUDA(cudaGetLastError());
    return APDA_OK;
}
extern "C" int apda_peer_wait(apda_ctx *ctx, const void *d_flags, int world, uint32_t value, double timeout_s,
                              int *d_timed_out) {
    if (!ctx || !d_flags || !d_timed_out || world < 1 || world > 32) return APDA_ERR_INVALID;
    APDA_CUDA(cudaSetDevice(ctx->device));
    peer_wait_kernel<<<1, 32, 0, ctx->stream>>>(reinterpret_cast<const unsigned *>(d_flags), world, value,
                                               (long long)(timeout_s * 1e3 * (double)ctx->clock_khz), d_timed_out);
    ctx->launches++;
    APDA_CUDA(cudaGetLastError());
    return APDA_OK;
}
