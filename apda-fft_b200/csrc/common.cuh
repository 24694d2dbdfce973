// Shared device/host helpers of libapda_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include <map>
#include <mutex>
#include <utility>
#include <vector>
#include <string>

#include "../../include/apda_b200.h"

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
struct TwiddleTables {
    double2 *d64 = nullptr;  // N-1 entries: stage with half-span h occupies [h-1, 2h-1)  (reference recurrence values)
    float2 *d32 = nullptr;   // same table rounded to fp32
};

struct apda_ctx {
    int device = 0;
    int sm_count = 0;
    int smem_optin = 0;
    int clock_khz = 0;  // SM clock (cached: querying cudaDevAttrClockRate per call costs about a millisecond)
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;  // stream the _dev entry points enqueue on
    cudaStream_t pipe[2] = {nullptr, nullptr};
    std::map<int64_t, TwiddleTables> twiddles;
    void *ws = nullptr;  // grow-only workspace for the _dev entry points (spectrum for analyze, mags for large N)
    size_t ws_bytes = 0;
    void *ws_pipe[2] = {nullptr, nullptr};
    size_t ws_pipe_bytes[2] = {0, 0};
    void *ws_small = nullptr;  // per-window fs array etc.
    size_t ws_small_bytes = 0;
    int64_t launches = 0;
    std::map<cudaStream_t, std::pair<void *, size_t>> stream_scratch;  // K2 median state, one per stream
    // device-side window lists ([0] = count, [1..] = window ids), one set PER STREAM: the two host-pipeline streams run
    // chunks concurrently, so a list shared by the context would be zeroed / appended to by one chunk while the other
    // chunk's kernels still read it
    struct StreamLists {
        int *ragged = nullptr;  // ragged batches: windows whose length differs from the batch's common length
        size_t ragged_bytes = 0;
        int *repair = nullptr;  // K3 fast path: windows handed over to the general kernel
        size_t repair_bytes = 0;
        int *ties = nullptr;  // fp32 tie resolver: windows whose record status is APDA_STATUS_FP32_TIE
        size_t ties_bytes = 0;
        int64_t *jsonl = nullptr;  // fleet JSONL rows: per-block byte counts, then their prefixes
        size_t jsonl_bytes = 0;
    };
    std::map<cudaStream_t, StreamLists> stream_lists;
    int generic_only = 0;  // debug/test switch: bypass the specialised fp32 kernels
    // pinned staging of apda_analyze_logs_*_host, one per pipeline stream: file bytes, then the chunk's offsets
    void *log_stage[2] = {nullptr, nullptr};
    size_t log_stage_bytes[2] = {0, 0};
};

void apda_set_error(const char *fmt, ...);
int apda_cuda_fail(cudaError_t e, const char *what);
#define APDA_CUDA(call)                                            \
    do {                                                           \
        cudaError_t _e = (call);                                   \
        if (_e != cudaSuccess) return apda_cuda_fail(_e, #call);   \
    } while (0)
#define APDA_TRY(call)                 \
    do {                               \
        int _s = (call);               \
        if (_s != APDA_OK) return _s;  \
    } while (0)

// ---- programmatic dependent launch (chains of short dependent kernels: K2's median + passes, K3-large) ---------------
// A kernel launched through apda_launch_pdl may become resident while the kernel in front of it in the stream drains
// (that kernel lets it go with pdl_trigger(), or implicitly when it ends); it must call pdl_wait() before its first
// global-memory access: the wait returns when the kernel in front has completed and its writes are visible.  Both
// instructions are no-ops in a kernel launched the ordinary way.  APDA_PDL=<mask> selects the kernel groups that get the attribute (0: none; A/B runs).
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#endif
enum { APDA_PDL_MEDIAN = 1, APDA_PDL_HEAD = 2, APDA_PDL_TAIL = 4, APDA_PDL_K3 = 8 };
int apda_pdl_mask();  // APDA_PDL environment variable (default: every group)
template <typename... KArgs, typename... Args>
inline cudaError_t apda_launch_pdl(int group, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                   Args &&...args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr{};
    attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr.val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = &attr;
    cfg.numAttrs = (apda_pdl_mask() & group) ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(std::forward<Args>(args))...);
}

int apda_get_twiddles(apda_ctx *ctx, int64_t N, TwiddleTables *out);
int apda_reserve(void **buf, size_t *have, size_t need);
// cudaFuncAttributeMaxDynamicSharedMemorySize, set once per (device, kernel): the attribute call is a driver round trip that
// a launch on the hot path (a few hundred microseconds of GPU work per step in the strong-scaled fleet sweep) should not pay
int apda_func_smem(const void *kernel, int device, size_t bytes);
#define APDA_FUNC_SMEM(ctx, kernel, bytes) APDA_TRY(apda_func_smem(reinterpret_cast<const void *>(kernel), (ctx)->device, (size_t)(bytes)))
// per-stream window lists of `batch + 1` ints, zero count enqueued on `st` (see apda_ctx::stream_lists)
int apda_repair_list(apda_ctx *ctx, cudaStream_t st, int64_t batch, int **out);
int apda_ragged_list(apda_ctx *ctx, cudaStream_t st, int64_t batch, int **out);
int apda_tie_list(apda_ctx *ctx, cudaStream_t st, int64_t batch, int **out);

static inline int ilog2_i64(int64_t v) {
    int l = 0;
    while ((int64_t(1) << l) < v) ++l;
    return l;
}
static inline bool is_pow2_i64(int64_t v) { return v > 0 && (v & (v - 1)) == 0; }

// launchers implemented in the kernel translation units
template <typename T>
int launch_fft_smem(apda_ctx *ctx, cudaStream_t st, const T *d_samples, int64_t n_samples, int64_t ld, int64_t batch,
                    int64_t N, int flags, T *d_spec, bool complex_input, const int *d_nv = nullptr,
                    const int *d_list = nullptr);
template <typename T>
int launch_fft_large(apda_ctx *ctx, cudaStream_t st, const T *d_samples, int64_t n_samples, int64_t ld, int64_t batch,
                     int64_t N, int flags, T *d_spec, bool complex_input);
template <typename T>
int launch_peaks(apda_ctx *ctx, cudaStream_t st, const T *d_spec, int64_t n, int64_t batch, double fs,
                 const double *d_fs, int k, int rec_cap, int flexible, void *d_rec, void *d_mag_ws);
template <typename T>
size_t peaks_mag_workspace_bytes(apda_ctx *ctx, int64_t n, int64_t batch);
template <typename T>
int launch_synth(apda_ctx *ctx, cudaStream_t st, int64_t first, int64_t count, int64_t N, uint64_t seed, int on_bin,
                 T *d_out);
template <typename T>
int64_t fft_smem_max_n(apda_ctx *ctx);
bool fft_f32_fast_supports(int64_t N);
int launch_fft_f32_fast(apda_ctx *ctx, cudaStream_t st, const float *d_samples, int64_t n_samples, int64_t ld,
                        int64_t batch, int64_t N, int flags, float *d_spec, const int *d_nv = nullptr, bool half_out = false);
void fft_f32_fast_release(apda_ctx *ctx);
int launch_fused_f32(apda_ctx *ctx, cudaStream_t st, const float *d_samples, int64_t n_samples, int64_t ld, int64_t batch,
                     int64_t N, int flags, int flexible, double fs, const double *d_fs, int k, void *d_rec);
template <typename T>
int launch_decode_wire16(apda_ctx *ctx, cudaStream_t st, const unsigned char *d_payload, int64_t n_max, int64_t ld_bytes,
                         int64_t batch, const double *d_first_value, T *d_samples, int64_t ld_out, int *d_n_valid);
// d_starts: where each log's sample region begins (NULL: at d_offsets[b]); it ends at d_offsets[b + 1]
template <typename T>
int launch_parse_samples(apda_ctx *ctx, cudaStream_t st, const char *d_text, const int64_t *d_offsets, int64_t batch,
                         int64_t ld, T *d_samples, int *d_n_valid, int *d_flags, const int64_t *d_starts = nullptr);
// whole .log files (text_ingest.cu): header layout, sampling rate and header bytes; then the flags / empty records
int launch_log_layout(apda_ctx *ctx, cudaStream_t st, const char *d_text, const int64_t *d_offsets, int64_t batch,
                      int64_t *d_starts, double *d_fs, int *d_flags, char *d_head);
int launch_log_finish(apda_ctx *ctx, cudaStream_t st, int64_t batch, int *d_flags, const int *d_parse_flags, void *d_rec,
                      int rec_cap);
bool fft_f64_fast_supports(int64_t N);
int launch_fft_f64_fast(apda_ctx *ctx, cudaStream_t st, const double *d_samples, int64_t n_samples, int64_t ld,
                        int64_t batch, int64_t N, int flags, double *d_spec, const int *d_nv = nullptr);
bool peaks_f32_fast_supports(int64_t n, int k, int rec_cap);
bool peaks_large_supports(int64_t n);
template <typename T>
size_t peaks_large_workspace_bytes(int64_t n, int64_t batch);
template <typename T>
int launch_peaks_large(apda_ctx *ctx, cudaStream_t st, const T *d_spec, int64_t n, int64_t batch, double fs,
                       const double *d_fs, int k, int rec_cap, int flexible, void *d_rec, void *ws);
template <typename T>
int launch_peaks_general_listed(apda_ctx *ctx, cudaStream_t st, const T *d_spec, int64_t n, int64_t batch, double fs,
                                const double *d_fs, int k, int rec_cap, int flexible, void *d_rec, const int *list);
bool peaks_f64_fast_supports(int64_t n, int k, int rec_cap);
int launch_peaks_f64_fast(apda_ctx *ctx, cudaStream_t st, const double *d_spec, int64_t n, int64_t batch, double fs,
                          const double *d_fs, int k, int flexible, void *d_rec);
int launch_peaks_f32_fast(apda_ctx *ctx, cudaStream_t st, const float *d_spec, int64_t n, int64_t batch, double fs,
                          const double *d_fs, int k, int flexible, void *d_rec);
int launch_center_f64(apda_ctx *ctx, cudaStream_t st, const double *d_in, int64_t n, double *d_out);
int launch_mag_helpers_f64(apda_ctx *ctx, cudaStream_t st, const double *d_mags, int64_t n, int64_t idx, double prom_in,
                           double *d_out3);
// fp32 tie resolver (resolve_ties.cu): d_slots holds resolve_ties_slot_bytes(ctx, N, batch) bytes of spectrum slots
size_t resolve_ties_slot_bytes(apda_ctx *ctx, int64_t N, int64_t batch);
int launch_resolve_ties(apda_ctx *ctx, cudaStream_t st, const float *d_samples, const int *d_nv, int64_t n_samples,
                        int64_t ld, int64_t batch, int64_t N, int center, int flexible, double fs, const double *d_fs,
                        int k, int rec_cap, void *d_rec, int *d_list, void *d_slots);
// record presentation (present.cu): reference-rounded columns, fleet JSONL rows (d_scratch: fleet_jsonl_scratch_bytes)
int launch_present_columns(apda_ctx *ctx, cudaStream_t st, const void *d_rec, int rec_cap, int64_t batch, int64_t n,
                           double fs, const double *d_fs, int flexible, int k, int32_t *d_idx, double *d_freq,
                           double *d_mag, double *d_prom, double *d_damp, double *d_q);
size_t fleet_jsonl_scratch_bytes(int64_t batch);
int launch_fleet_jsonl(apda_ctx *ctx, cudaStream_t st, const void *d_rec, int rec_cap, int64_t batch, int64_t n, double fs,
                       const double *d_fs, int flexible, int k, int64_t first_window, char *d_text, int64_t *d_offsets,
                       int64_t *d_scratch);

// ---------------------------------------------------------------------------------------------------------------
// device side
// ---------------------------------------------------------------------------------------------------------------
#ifdef __CUDACC__

template <typename T>
struct vec2;
template <>
struct vec2<double> {
    using type = double2;
};
template <>
struct vec2<float> {
    using type = float2;
};

// Individually rounded IEEE operations: the compiler may never contract these into FMAs.  Every place where the
// reference's Python float arithmetic decides a comparison or feeds the fp64 bit-exact spectrum goes through them.
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub_rn(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double div_rn(double a, double b) { return __ddiv_rn(a, b); }
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float sub_rn(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float div_rn(float a, float b) { return __fdiv_rn(a, b); }

// |re + i*im| with the operation sequence of glibc 2.39's hypot (Borges' correction, non-FMA kernel), which is what
// CPython's abs(complex) calls: bit-identical to the reference for fp64 (checked in tests).  The huge/tiny scaling
// branches of glibc are kept so the full double range behaves the same.
__device__ __forceinline__ double hypot_kernel_rn(double ax, double ay) {
    double h = __dsqrt_rn(add_rn(mul_rn(ax, ax), mul_rn(ay, ay)));
    double t1, t2;
    if (h <= mul_rn(2.0, ay)) {
        double delta = sub_rn(h, ay);
        t1 = mul_rn(ax, sub_rn(mul_rn(2.0, delta), ax));
        t2 = mul_rn(sub_rn(delta, mul_rn(2.0, sub_rn(ax, ay))), delta);
    } else {
        double delta = sub_rn(h, ax);
        t1 = mul_rn(mul_rn(2.0, delta), sub_rn(ax, mul_rn(2.0, ay)));
        t2 = add_rn(mul_rn(sub_rn(mul_rn(4.0, delta), ay), ay), mul_rn(delta, delta));
    }
    return sub_rn(h, div_rn(add_rn(t1, t2), mul_rn(2.0, h)));
}
__device__ __forceinline__ double magnitude(double re, double im) {
    double x = fabs(re), y = fabs(im);
    if (!(x <= 1.7976931348623157e308) || !(y <= 1.7976931348623157e308)) {  // inf / nan
        if (isinf(x) || isinf(y)) return CUDART_INF;
        return x + y;
    }
    double ax = x < y ? y : x;
    double ay = x < y ? x : y;
    const double EPS = 0x1p-54, LARGE = 0x1p+511, TINY = 0x1p-459, SCALE = 0x1p-600;
    if (ax > LARGE) {
        if (ay <= mul_rn(ax, EPS)) return add_rn(ax, ay);
        return div_rn(hypot_kernel_rn(mul_rn(ax, SCALE), mul_rn(ay, SCALE)), SCALE);
    }
    if (ay < TINY) {
        if (ax >= div_rn(ay, EPS)) return add_rn(ax, ay);
        return mul_rn(hypot_kernel_rn(div_rn(ax, SCALE), div_rn(ay, SCALE)), SCALE);
    }
    if (ax >= div_rn(ay, EPS)) return add_rn(ax, ay);
    return hypot_kernel_rn(ax, ay);
}
__device__ __forceinline__ float magnitude(float re, float im) { return sqrtf(fmaf(re, re, im * im)); }

// Blackwell packed fp32 arithmetic (FADD2 / FMUL2 / FFMA2): one instruction per (re, im) pair.  ptxas folds a pair made of
// one register twice, (a, a), into the scalar-broadcast operand form, so a complex product is two packed instructions.
__device__ __forceinline__ unsigned long long f2bits(float2 v) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(v.x), "f"(v.y));
    return r;
}
__device__ __forceinline__ float2 f2from(unsigned long long b) {
    float2 r;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(b));
    return r;
}
__device__ __forceinline__ float2 f2add(float2 a, float2 b) {
    unsigned long long r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(f2bits(a)), "l"(f2bits(b)));
    return f2from(r);
}
__device__ __forceinline__ float2 f2sub(float2 a, float2 b) {
    unsigned long long r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(f2bits(a)), "l"(f2bits(b)));
    return f2from(r);
}
__device__ __forceinline__ float2 f2mul(float2 a, float2 b) {
    unsigned long long r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(f2bits(a)), "l"(f2bits(b)));
    return f2from(r);
}
__device__ __forceinline__ float2 f2fma(float2 a, float2 b, float2 c) {
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(f2bits(a)), "l"(f2bits(b)), "l"(f2bits(c)));
    return f2from(r);
}

// order-preserving integer keys of IEEE values (radix select)
__device__ __forceinline__ uint64_t ordered_key(double v) {
    uint64_t b = (uint64_t)__double_as_longlong(v);
    return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double key_value(uint64_t k, double) {
    uint64_t b = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)b);
}
__device__ __forceinline__ uint32_t ordered_key(float v) {
    uint32_t b = __float_as_uint(v);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key_value(uint32_t k, float) {
    uint32_t b = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
    return __uint_as_float(b);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// double-double helpers (error-free transformations) for the fp64 statistics
struct dd {
    double hi, lo;
};
__device__ __forceinline__ dd two_sum(double a, double b) {
    double s = add_rn(a, b);
    double bb = sub_rn(s, a);
    double e = add_rn(sub_rn(a, sub_rn(s, bb)), sub_rn(b, bb));
    return {s, e};
}
__device__ __forceinline__ dd dd_add(dd a, dd b) {
    dd s = two_sum(a.hi, b.hi);
    dd t = two_sum(a.lo, b.lo);
    double c = add_rn(s.lo, t.hi);
    dd v = two_sum(s.hi, c);
    double w = add_rn(t.lo, v.lo);
    return two_sum(v.hi, w);
}
__device__ __forceinline__ dd dd_add_d(dd a, double b) {
    dd s = two_sum(a.hi, b);
    double w = add_rn(s.lo, a.lo);
    return two_sum(s.hi, w);
}
__device__ __forceinline__ dd two_prod(double a, double b) {
    double p = mul_rn(a, b);
    return {p, __fma_rn(a, b, -p)};
}
__device__ __forceinline__ dd dd_mul(dd a, dd b) {
    dd p = two_prod(a.hi, b.hi);
    double c = add_rn(mul_rn(a.hi, b.lo), mul_rn(a.lo, b.hi));
    return two_sum(p.hi, add_rn(p.lo, c));
}
__device__ __forceinline__ dd dd_neg(dd a) { return {-a.hi, -a.lo}; }
__device__ __forceinline__ dd dd_div_d(dd a, double b) {  // a / b, b exact double
    double q1 = div_rn(a.hi, b);
    dd p = two_prod(q1, b);
    dd r = dd_add(a, dd_neg(p));
    double q2 = div_rn(r.hi, b);
    dd p2 = two_prod(q2, b);
    dd r2 = dd_add(r, dd_neg(p2));
    double q3 = div_rn(r2.hi, b);
    dd q = two_sum(q1, q2);
    return dd_add_d(q, q3);
}
__device__ __forceinline__ double dd_sqrt_to_double(dd a) {  // correctly rounded sqrt(a) for all but ~2^-50 of inputs
    if (!(a.hi > 0.0)) return 0.0;
    double s = __dsqrt_rn(a.hi);
    dd s2 = two_prod(s, s);
    dd r = dd_add(a, dd_neg(s2));
    return add_rn(s, div_rn(r.hi, mul_rn(2.0, s)));
}
// approximate reciprocal / square root (one MUFU each) for values that only STEER an exact algorithm (selection pivots)
__device__ __forceinline__ float rcp_approx(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float sqrt_approx(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
// Ask L2 for the bytes [p, p + bytes) of a window a LATER CTA will stream (128-byte lines dealt out to the callers), so
// that its loads find the data on chip instead of waiting a DRAM round trip; `ahead` = windows resident on the whole GPU.
#ifndef APDA_L2_PREFETCH
#define APDA_L2_PREFETCH 1
#endif
__device__ __forceinline__ unsigned sm_count_reg() {
    unsigned n;
    asm("mov.u32 %0, %%nsmid;" : "=r"(n));
    return n;
}
__device__ __forceinline__ void l2_prefetch_span(const void *p, int bytes, int tid, int nthreads) {
    const char *c = reinterpret_cast<const char *>(p);
    for (int off = tid * 128; off < bytes; off += nthreads * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(c + off));
}
#endif  // __CUDACC__
