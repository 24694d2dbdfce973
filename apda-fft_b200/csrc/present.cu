// Presentation of record tables (SURVEY 8f rank 4): records -> the values the reference's consumers read, computed on the
// device with Python's float semantics.
//
//   present_columns_kernel  one thread per (window, slot): the fields of records.prominence_dicts (flexible picker) or
//                           records.resolution_dicts (rigid picker) as doubles, in the reference's operation order
//   jsonl_length_kernel     one thread per window: the byte length of its records.write_fleet_jsonl row; block sums
//   jsonl_scan_kernel       one CTA: exclusive scan of the block sums
//   jsonl_write_kernel      one thread per window: row offset (block scan + block prefix), then the row's text
//
// round(x, d) for d = 2, 4 is CPython's: the exact value x * 10^d rounded half to even to an integer n (the product and its
// FMA residual decide), then the correctly rounded n / 10^d; once |n| >= 2^53 the result is x itself (x then lies within
// half an ulp of n / 10^d).  The text is repr() of each float (repr.cuh) in json.dumps' layout.
#include "common.cuh"
#include "repr.cuh"

namespace {

__device__ __forceinline__ double py_round(double x, double p) {
    const double hi = mul_rn(x, p);
    const double lo = __fma_rn(x, p, -hi);
    double n = rint(hi);
    const double d = sub_rn(hi, n);
    if (d == 0.5 && lo > 0.0) n = add_rn(n, 1.0);
    if (d == -0.5 && lo < 0.0) n = sub_rn(n, 1.0);
    if (!(fabs(n) < 9007199254740992.0)) return x;  // also inf and nan
    return div_rn(n, p);
}

struct Slot {
    int idx;
    double freq, mag, prominence, damping, q;
};

// slot j < count of window w (records.py operation order; Python ints convert to double exactly)
__device__ __forceinline__ Slot present_slot(const unsigned char *rec, double fs, double n, int flexible, int j) {
    const unsigned char *pk = rec + 8 + 24 * j;
    const int2 iw = *reinterpret_cast<const int2 *>(pk);
    const double mag = *reinterpret_cast<const double *>(pk + 8);
    const double df = div_rn(fs, n);
    const double fn = mul_rn((double)iw.x, df);
    Slot s;
    s.idx = iw.x;
    if (flexible) {
        const double q = div_rn(fn, mul_rn((double)iw.y, df));
        const double damping = div_rn(1.0, mul_rn(2.0, q));
        s.freq = py_round(fn, 1e4);
        s.mag = py_round(mag, 1e4);
        s.prominence = *reinterpret_cast<const double *>(pk + 16);
        s.damping = py_round(mul_rn(damping, 100.0), 1e2);
        s.q = py_round(q, 1e2);
    } else {
        s.freq = fn;
        s.mag = mag;
        s.prominence = s.damping = s.q = CUDART_NAN;
    }
    return s;
}

__device__ __forceinline__ int peaks_shown(const unsigned char *rec, int k) {
    return min(max(*reinterpret_cast<const int *>(rec), 0), k);
}

__global__ void __launch_bounds__(256)
present_columns_kernel(const unsigned char *__restrict__ recs, int64_t rec_bytes, int64_t slots, int k, double n, double fs,
                       const double *__restrict__ d_fs, int flexible, int32_t *__restrict__ o_idx,
                       double *__restrict__ o_freq, double *__restrict__ o_mag, double *__restrict__ o_prom,
                       double *__restrict__ o_damp, double *__restrict__ o_q) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= slots) return;
    const int64_t w = t / k;
    const int j = (int)(t - w * k);
    const unsigned char *rec = recs + w * rec_bytes;
    Slot s{-1, CUDART_NAN, CUDART_NAN, CUDART_NAN, CUDART_NAN, CUDART_NAN};
    if (j < peaks_shown(rec, k)) s = present_slot(rec, d_fs ? d_fs[w] : fs, n, flexible, j);
    if (o_idx) o_idx[t] = s.idx;
    if (o_freq) o_freq[t] = s.freq;
    if (o_mag) o_mag[t] = s.mag;
    if (o_prom) o_prom[t] = s.prominence;
    if (o_damp) o_damp[t] = s.damping;
    if (o_q) o_q[t] = s.q;
}

// json.dumps({"window": first_window + w, "fft_freqs": [...], "fft_mags": [...]}) + "\n", missing peaks as 0.0
template <class O>
__device__ void put_row(O &o, const unsigned char *rec, double fs, double n, int flexible, int k, int64_t window) {
    const int shown = peaks_shown(rec, k);
    repr::put_lit(o, "{\"window\": ");
    repr::put_int(o, (uint64_t)window);
    repr::put_lit(o, ", \"fft_freqs\": [");
    for (int j = 0; j < k; ++j) {
        if (j) repr::put_lit(o, ", ");
        repr::put_double(o, j < shown ? present_slot(rec, fs, n, flexible, j).freq : 0.0);
    }
    repr::put_lit(o, "], \"fft_mags\": [");
    for (int j = 0; j < k; ++j) {
        if (j) repr::put_lit(o, ", ");
        repr::put_double(o, j < shown ? present_slot(rec, fs, n, flexible, j).mag : 0.0);
    }
    repr::put_lit(o, "]}\n");
}

constexpr int kRowThreads = 256;

__device__ __forceinline__ int64_t block_sum(int64_t v, int64_t *warp_tot) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) warp_tot[warp] = v;
    __syncthreads();
    int64_t s = 0;
#pragma unroll
    for (int i = 0; i < kRowThreads / 32; ++i) s += warp_tot[i];
    return s;
}

__global__ void __launch_bounds__(kRowThreads)
jsonl_length_kernel(const unsigned char *__restrict__ recs, int64_t rec_bytes, int64_t batch, int k, double n, double fs,
                    const double *__restrict__ d_fs, int flexible, int64_t first_window, int64_t *__restrict__ offsets,
                    int64_t *__restrict__ block_sums) {
    __shared__ int64_t warp_tot[kRowThreads / 32];
    const int64_t w = (int64_t)blockIdx.x * kRowThreads + threadIdx.x;
    repr::Count c;
    if (w < batch) {
        put_row(c, recs + w * rec_bytes, d_fs ? d_fs[w] : fs, n, flexible, k, first_window + w);
        offsets[w + 1] = c.n;
    }
    const int64_t s = block_sum(c.n, warp_tot);
    if (threadIdx.x == 0) block_sums[blockIdx.x] = s;
}

// in place: block_sums[b] := sum of block_sums[0 .. b)
__global__ void __launch_bounds__(1024) jsonl_scan_kernel(int64_t *__restrict__ block_sums, int64_t nblocks) {
    __shared__ int64_t warp_tot[32];
    __shared__ int64_t carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int64_t base = 0; base < nblocks; base += 1024) {
        const int64_t i = base + threadIdx.x;
        const int64_t v = i < nblocks ? block_sums[i] : 0;
        int64_t incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) warp_tot[warp] = incl;
        __syncthreads();
        int64_t before = carry, total = carry;
        for (int x = 0; x < 32; ++x) {
            if (x < warp) before += warp_tot[x];
            total += warp_tot[x];
        }
        if (i < nblocks) block_sums[i] = before + incl - v;
        __syncthreads();
        if (threadIdx.x == 0) carry = total;
        __syncthreads();
    }
}

// offsets[w + 1] holds row w's length on entry and its end on exit; each thread rewrites only its own entry
__global__ void __launch_bounds__(kRowThreads)
jsonl_write_kernel(const unsigned char *__restrict__ recs, int64_t rec_bytes, int64_t batch, int k, double n, double fs,
                   const double *__restrict__ d_fs, int flexible, int64_t first_window, int64_t *__restrict__ offsets,
                   const int64_t *__restrict__ block_prefix, char *__restrict__ text) {
    __shared__ int64_t warp_incl[kRowThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t w = (int64_t)blockIdx.x * kRowThreads + threadIdx.x;
    const int64_t len = w < batch ? offsets[w + 1] : 0;
    int64_t incl = len;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int64_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) warp_incl[warp] = incl;
    __syncthreads();
    int64_t end = block_prefix[blockIdx.x] + incl;
    for (int x = 0; x < warp; ++x) end += warp_incl[x];
    if (w >= batch) return;
    offsets[w + 1] = end;
    if (w == 0) offsets[0] = 0;
    repr::Write out{text + (end - len)};
    put_row(out, recs + w * rec_bytes, d_fs ? d_fs[w] : fs, n, flexible, k, first_window + w);
}

}  // namespace

int launch_present_columns(apda_ctx *ctx, cudaStream_t st, const void *d_rec, int rec_cap, int64_t batch, int64_t n,
                           double fs, const double *d_fs, int flexible, int k, int32_t *d_idx, double *d_freq,
                           double *d_mag, double *d_prom, double *d_damp, double *d_q) {
    const int64_t slots = batch * k;
    if (slots == 0) return APDA_OK;
    present_columns_kernel<<<(unsigned)((slots + 255) / 256), 256, 0, st>>>(
        reinterpret_cast<const unsigned char *>(d_rec), APDA_REC_BYTES(rec_cap), slots, k, (double)n, fs, d_fs, flexible,
        d_idx, d_freq, d_mag, d_prom, d_damp, d_q);
    ctx->launches++;
    APDA_CUDA(cudaGetLastError());
    return APDA_OK;
}

size_t fleet_jsonl_scratch_bytes(int64_t batch) {
    return (size_t)((batch + kRowThreads - 1) / kRowThreads) * sizeof(int64_t);
}

int launch_fleet_jsonl(apda_ctx *ctx, cudaStream_t st, const void *d_rec, int rec_cap, int64_t batch, int64_t n, double fs,
                       const double *d_fs, int flexible, int k, int64_t first_window, char *d_text, int64_t *d_offsets,
                       int64_t *d_scratch) {
    if (batch == 0) return APDA_OK;
    const int64_t nblocks = (batch + kRowThreads - 1) / kRowThreads;
    const unsigned char *recs = reinterpret_cast<const unsigned char *>(d_rec);
    const int64_t rec_bytes = APDA_REC_BYTES(rec_cap);
    jsonl_length_kernel<<<(unsigned)nblocks, kRowThreads, 0, st>>>(recs, rec_bytes, batch, k, (double)n, fs, d_fs, flexible,
                                                                   first_window, d_offsets, d_scratch);
    ctx->launches++;
    APDA_CUDA(cudaGetLastError());
    jsonl_scan_kernel<<<1, 1024, 0, st>>>(d_scratch, nblocks);
    ctx->launches++;
    APDA_CUDA(cudaGetLastError());
    jsonl_write_kernel<<<(unsigned)nblocks, kRowThreads, 0, st>>>(recs, rec_bytes, batch, k, (double)n, fs, d_fs, flexible,
                                                                  first_window, d_offsets, d_scratch, d_text);
    ctx->launches++;
    APDA_CUDA(cudaGetLastError());
    return APDA_OK;
}
