// K2: multi-pass FFT for transforms longer than 2^13 in both precisions (N = 2^14 ... 2^30, any batch).
//
// The reference's radix-2 DIT dataflow graph (metrics/fft_iterativa.py:38-70) is cut into P passes of q_p stages
// (sum q_p = log2 N, q_p <= 10 fp64 / 11 fp32).  Every pass moves the data through HBM exactly once:
//
//   head pass  (stages 1..q_1)   In bit-reversed order the first q_1 stages act on contiguous blocks of 2^q_1
//              outputs whose inputs are the samples j = j_hi * 2^(n-q_1) + j_lo with j_lo fixed: a COLUMN of the
//              input viewed as a [2^q_1][2^(n-q_1)] matrix.  A CTA takes C adjacent columns (C*sizeof(T)-byte
//              coalesced row segments), centres / pads / bit-reverses on the way into shared memory, runs the
//              stages on C contiguous column arrays and writes each column out as one contiguous block.
//   tail passes (stages s0+1..s0+q) act on index bits [s0, s0+q): a tile is [2^q rows (stride 2^s0)][C adjacent
//              columns], loaded and stored in place with coalesced C-element row segments; the stage twiddles
//              T_s[(r mod 2^(t-1)) * 2^s0 + column] are read coalesced from the recurrence table.
//
// The butterflies use the same host-built recurrence twiddle table and the same individually rounded operations as
// K1, so the fp64 result is bit-identical to the reference for every N (the table is what makes N >= 2^16 match to
// 1e-12: the reference's own twiddle drift reaches 3e-10 at N = 2^24).  fp32 runs the same passes on the rounded table.
// The exact median of up to 2^30 samples is a multi-CTA radix select (histogram passes over HBM).
#include <cuda.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>

#include "common.cuh"

#ifndef APDA_K2_HEAD_UNR
#define APDA_K2_HEAD_UNR 8  // gather loads in flight per thread in the head pass
#endif

namespace {

constexpr int kThreads = 512;  // default CTA size; the pass kernels are templated on it (NT)

template <typename T>
__device__ __forceinline__ void butterfly(typename vec2<T>::type &u, typename vec2<T>::type &v,
                                          const typename vec2<T>::type w) {
    // v*w with Python's complex product (ac-bd, ad+bc), then u+v, u-v; every operation rounds on its own
    const T vr = sub_rn(mul_rn(v.x, w.x), mul_rn(v.y, w.y));
    const T vi = add_rn(mul_rn(v.x, w.y), mul_rn(v.y, w.x));
    typename vec2<T>::type a, b;
    a.x = add_rn(u.x, vr);
    a.y = add_rn(u.y, vi);
    b.x = sub_rn(u.x, vr);
    b.y = sub_rn(u.y, vi);
    u = a;
    v = b;
}

// fp32 butterfly (tolerance path, not bit-exact): packed arithmetic, the product v*w as two packed instructions
//   v*w = v.x * (w.x, w.y) + v.y * (-w.y, w.x);   wr = (-w.y, w.x) is prepared once per twiddle
__device__ __forceinline__ void butterfly_f32(float2 &u, float2 &v, const float2 w, const float2 wr) {
    const float2 vw = f2fma(make_float2(v.y, v.y), wr, f2mul(make_float2(v.x, v.x), w));
    const float2 a = f2add(u, vw), b = f2sub(u, vw);
    u = a;
    v = b;
}

// QR radix-2 stages (t0+1 .. t0+QR of this pass) on 2^QR register-resident values per work item: one shared-memory round
// trip and one barrier per QR stages instead of per stage, 2^QR - 1 twiddle loads per QR * 2^(QR-1) butterflies.
// Element (row r, column c) of the pass's working set lives at tile[r * rs + c * cs]; rows r = (hi << (t0+QR)) + (k << t0) + jr.
// Twiddle of stage t for row r: T_{s0+t}[((r mod 2^(t-1)) << s0) + lo0 + c]  (head pass: s0 = 0 and no column term - its
// columns are independent sub-transforms).  fp64: the reference's dataflow graph with individually rounded operations
// (bit-exact); fp32: the same graph with packed arithmetic.
template <typename T, int QR, bool HEAD, int NT>
__device__ __forceinline__ void stage_round(typename vec2<T>::type *tile, int rs, int cs, int logC, int q, int t0,
                                            const typename vec2<T>::type *__restrict__ tw, int s0, int64_t lo0, int tid) {
    using V2 = typename vec2<T>::type;
    constexpr int R = 1 << QR;
    const int items = 1 << (logC + q - QR);
    for (int item = tid; item < items; item += NT) {
        const int c = item & ((1 << logC) - 1), rest = item >> logC;
        const int jr = rest & ((1 << t0) - 1), hi = rest >> t0;
        V2 *p = tile + (((hi << (t0 + QR)) + jr) * rs + c * cs);  // a tile holds < 2^15 elements: 32-bit index arithmetic
        const int kstride = rs << t0;
        V2 v[R];
#pragma unroll
        for (int k = 0; k < R; ++k) v[k] = p[k * kstride];
        // twiddle indices fit 32 bits (the table of N <= 2^30 has N - 1 entries): one 64-bit pointer add per load
        const unsigned tw_row = ((unsigned)jr << s0) + (HEAD ? 0u : (unsigned)lo0 + (unsigned)c);
        const unsigned tw_step = 1u << (t0 + s0);
#pragma unroll
        for (int u = 1; u <= QR; ++u) {
            const int t = t0 + u;  // stage of this pass (1-based): pairs rows that differ in bit t-1
            const V2 *tab = tw + (((1u << (s0 + t - 1)) - 1u) + tw_row);
            V2 w[R / 2];
#pragma unroll
            for (int m = 0; m < (1 << (u - 1)); ++m) w[m] = __ldg(tab + m * tw_step);
            if constexpr (sizeof(T) == 4) {
                V2 wr[R / 2];
#pragma unroll
                for (int m = 0; m < (1 << (u - 1)); ++m) wr[m] = make_float2(-w[m].y, w[m].x);
#pragma unroll
                for (int k = 0; k < R; ++k)
                    if ((k & (1 << (u - 1))) == 0)
                        butterfly_f32(v[k], v[k + (1 << (u - 1))], w[k & ((1 << (u - 1)) - 1)], wr[k & ((1 << (u - 1)) - 1)]);
            } else {
#pragma unroll
                for (int k = 0; k < R; ++k)
                    if ((k & (1 << (u - 1))) == 0) butterfly<T>(v[k], v[k + (1 << (u - 1))], w[k & ((1 << (u - 1)) - 1)]);
            }
        }
#pragma unroll
        for (int k = 0; k < R; ++k) p[k * kstride] = v[k];
    }
}

// all q stages of a pass in ceil(q / QMAX) rounds of nearly equal size (QMAX = 3 stages on 8 values per thread in fp64,
// 4 stages on 16 values in fp32, where the registers allow it), one barrier per round
template <typename T, bool HEAD, int NT>
__device__ __forceinline__ void run_stages(typename vec2<T>::type *tile, int rs, int cs, int logC, int q,
                                           const typename vec2<T>::type *__restrict__ tw, int s0, int64_t lo0, int tid) {
    constexpr int QMAX = sizeof(T) == 4 ? 4 : 3;
    const int rounds = (q + QMAX - 1) / QMAX, base = q / rounds, rem = q % rounds;
    int t0 = 0;
    for (int r = 0; r < rounds; ++r) {
        const int qr = base + (r < rem ? 1 : 0);
        if constexpr (sizeof(T) == 4) {
            if (qr == 4) stage_round<T, 4, HEAD, NT>(tile, rs, cs, logC, q, t0, tw, s0, lo0, tid);
        }
        if (qr == 3) stage_round<T, 3, HEAD, NT>(tile, rs, cs, logC, q, t0, tw, s0, lo0, tid);
        else if (qr == 2) stage_round<T, 2, HEAD, NT>(tile, rs, cs, logC, q, t0, tw, s0, lo0, tid);
        else if (qr == 1) stage_round<T, 1, HEAD, NT>(tile, rs, cs, logC, q, t0, tw, s0, lo0, tid);
        __syncthreads();
        t0 += qr;
    }
}

// ---- head pass ------------------------------------------------------------------------------------------------------
template <typename T, bool COMPLEX_IN, int NT>
__global__ void __launch_bounds__(NT)
large_head_kernel(const T *__restrict__ samples, int64_t n_samples, int64_t ld, int n, int q, int C,
                  const typename vec2<T>::type *__restrict__ tw, typename vec2<T>::type *__restrict__ spec,
                  const T *__restrict__ med_ptr) {
    using V2 = typename vec2<T>::type;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    pdl_trigger();
    pdl_wait();
    V2 *work = reinterpret_cast<V2 *>(smem_raw);
    const int LDW = (1 << q) + 1;
    const int tid = threadIdx.x;
    const int64_t win = blockIdx.y;
    const int64_t N = (int64_t)1 << n;
    const int64_t lo0 = (int64_t)blockIdx.x * C;
    const T med = med_ptr ? med_ptr[win] : T(0);
    const int rows = 1 << q;

    const int logC = 31 - __clz(C);  // C is a power of two
    // eight loads of a thread are issued before the first of them is used: the gather's rows are 2^(n-q) samples apart, so
    // every load is its own DRAM burst and the pass lives on memory-level parallelism
    constexpr int UNR = APDA_K2_HEAD_UNR;
    const int total = C << q;
    for (int e0 = tid; e0 < total; e0 += NT * UNR) {
        V2 val[UNR];
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const int e = e0 + u * NT;
            const int c = e & (C - 1), jh = e >> logC;
            const int64_t j = ((int64_t)jh << (n - q)) + lo0 + c;
            val[u].x = T(0);
            val[u].y = T(0);
            if (e < total) {
                if (COMPLEX_IN) val[u] = reinterpret_cast<const V2 *>(samples)[win * N + j];
                else if (j < n_samples) val[u].x = samples[win * ld + j];
            }
        }
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const int e = e0 + u * NT;
            if (e < total) {
                const int c = e & (C - 1), jh = e >> logC;
                const int64_t j = ((int64_t)jh << (n - q)) + lo0 + c;
                if (!COMPLEX_IN && j < n_samples) val[u].x = sub_rn(val[u].x, med);
                const int il = (int)(__brev((unsigned)jh) >> (32 - q));
                work[c * LDW + il] = val[u];
            }
        }
    }
    __syncthreads();

    run_stages<T, true, NT>(work, 1, LDW, logC, q, tw, 0, 0, tid);

    V2 *out = spec + win * N;
    for (int e = tid; e < (C << q); e += NT) {
        const int c = e >> q, il = e & (rows - 1);
        const int64_t ih = (int64_t)(__brev((unsigned)(lo0 + c)) >> (32 - (n - q)));
        out[(ih << q) + il] = work[c * LDW + il];
    }
}

// ---- tail passes ----------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kThreads)
large_tail_kernel(typename vec2<T>::type *__restrict__ spec, int n, int s0, int q, int C,
                  const typename vec2<T>::type *__restrict__ tw, int zero_dc) {
    using V2 = typename vec2<T>::type;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    pdl_trigger();
    pdl_wait();
    V2 *tile = reinterpret_cast<V2 *>(smem_raw);
    const int LD = C + 1;
    const int tid = threadIdx.x;
    const int64_t N = (int64_t)1 << n;
    const int64_t tiles_lo = ((int64_t)1 << s0) / C;
    const int64_t hi = blockIdx.x / tiles_lo;
    const int64_t lo0 = (blockIdx.x % tiles_lo) * C;
    V2 *base = spec + (int64_t)blockIdx.y * N + (hi << (s0 + q)) + lo0;
    const int rows = 1 << q;

    const int logC = 31 - __clz(C);  // C is a power of two
    for (int e = tid; e < (C << q); e += kThreads) {
        const int c = e & (C - 1), r = e >> logC;
        tile[r * LD + c] = base[((int64_t)r << s0) + c];
    }
    __syncthreads();

    run_stages<T, false, kThreads>(tile, LD, 1, logC, q, tw, s0, lo0, tid);

    for (int e = tid; e < (C << q); e += kThreads) {
        const int c = e & (C - 1), r = e >> logC;
        V2 val = tile[r * LD + c];
        if (zero_dc && hi == 0 && lo0 == 0 && r == 0 && c == 0) val.x = val.y = T(0);  // reference: res[0] = 0
        base[((int64_t)r << s0) + c] = val;
    }
    (void)rows;
}

// ---- tail pass, TMA staged -----------------------------------------------------------------------------------------
// Same arithmetic as large_tail_kernel; the [2^q][C] tile is brought in by cp.async.bulk.tensor (one elected thread,
// completion on an mbarrier) and written back in place by a bulk tensor store, so no thread spends registers or LSU
// issue slots on the HBM traffic.  The tensor map views the spectra as [batch * n_hi][2^q][2^s0] complex values
// (innermost dimension counted in scalars: 2 per complex value).
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// NT threads, MINB resident CTAs per SM: several tiles per SM in flight are what overlaps the bulk load of one tile with
// the butterflies of another and the bulk store of a third (a CTA alone runs load -> compute -> store back to back)
template <typename T, int NT, int MINB>
__global__ void __launch_bounds__(NT, MINB)
large_tail_tma_kernel(const __grid_constant__ CUtensorMap tmap, int n, int s0, int q, int C,
                      const typename vec2<T>::type *__restrict__ tw, int zero_dc) {
    using V2 = typename vec2<T>::type;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ __align__(8) unsigned long long bar;
    // TMA wants a 128-byte aligned shared-memory destination; the dynamic segment only promises 16
    V2 *tile = reinterpret_cast<V2 *>(smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u));
    const int tid = threadIdx.x;
    const int64_t tiles_lo = ((int64_t)1 << s0) / C;
    const int64_t n_hi = (int64_t)1 << (n - s0 - q);
    const int64_t hi = blockIdx.x / tiles_lo;
    const int64_t lo0 = (blockIdx.x % tiles_lo) * C;
    const int rows = 1 << q;
    const int box_rows = rows < 256 ? rows : 256;
    const int c0 = (int)(2 * lo0), c2 = (int)((int64_t)blockIdx.y * n_hi + hi);
    const uint32_t bar_a = smem_u32(&bar);

    pdl_trigger();
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_a));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    pdl_wait();  // the pass in front wrote this tile
    __syncthreads();
    if (tid == 0) {
        const uint32_t bytes = (uint32_t)((size_t)rows * C * sizeof(V2));
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"(bytes) : "memory");
        for (int r0 = 0; r0 < rows; r0 += box_rows) {
            const uint32_t dst = smem_u32(tile + (size_t)r0 * C);
            asm volatile(
                "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                ::"r"(dst), "l"(reinterpret_cast<uint64_t>(&tmap)), "r"(c0), "r"(r0), "r"(c2), "r"(bar_a)
                : "memory");
        }
    }
    {  // every thread waits for the tile (phase 0 of the barrier)
        uint32_t done = 0;
        while (!done) {
            asm volatile(
                "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                : "=r"(done)
                : "r"(bar_a), "r"(0u)
                : "memory");
        }
    }

    run_stages<T, false, NT>(tile, C, 1, 31 - __clz(C), q, tw, s0, lo0, tid);
    if (zero_dc && hi == 0 && lo0 == 0 && tid == 0) tile[0].x = tile[0].y = T(0);  // reference: res[0] = 0
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to the bulk store
    __syncthreads();
    if (tid == 0) {
        for (int r0 = 0; r0 < rows; r0 += box_rows) {
            const uint32_t src = smem_u32(tile + (size_t)r0 * C);
            asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%1, %2, %3}], [%4];" ::"l"(
                             reinterpret_cast<uint64_t>(&tmap)),
                         "r"(c0), "r"(r0), "r"(c2), "r"(src)
                         : "memory");
        }
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        // the CTA may retire as soon as the bulk store has READ the tile out of shared memory (its slot can then be handed to
        // the next tile); the global writes themselves complete before the kernel does
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn lookup_encode_fn() {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    EncodeTiledFn fn = nullptr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
        fn = reinterpret_cast<EncodeTiledFn>(p);
    (void)cudaGetLastError();
    return fn;
}
static EncodeTiledFn get_encode_fn() {
    static const EncodeTiledFn fn = lookup_encode_fn();  // initialised once, thread-safe
    return fn;
}

// tensor map of one tail pass; false if the driver entry point is missing or rejects the shape (caller falls back)
template <typename T>
static bool make_tail_tmap(CUtensorMap *tm, T *d_spec, int n, int s0, int q, int C, int64_t batch) {
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)2 << s0, (cuuint64_t)1 << q, (cuuint64_t)batch << (n - s0 - q)};
    const cuuint64_t strides[2] = {((cuuint64_t)1 << s0) * 2 * sizeof(T), ((cuuint64_t)1 << (s0 + q)) * 2 * sizeof(T)};
    const cuuint32_t box[3] = {(cuuint32_t)(2 * C), (cuuint32_t)std::min(1 << q, 256), 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUtensorMapDataType dt = sizeof(T) == 8 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
    if (box[0] > 256 || dims[2] >= ((cuuint64_t)1 << 32)) return false;
    return enc(tm, dt, 3, d_spec, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
               CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// ---- exact median of one long window: MSB-first 8-bit radix select with HBM histogram passes -----------------------
template <typename T>
struct KeyT;
template <>
struct KeyT<double> {
    using type = uint64_t;
};
template <>
struct KeyT<float> {
    using type = uint32_t;
};

struct SelectState {            // device resident
    unsigned long long prefix;  // key bits decided so far
    unsigned long long mask;
    long long rank;             // rank still to resolve inside the prefix bucket
    unsigned hist[256];
    unsigned long long found[2];  // lower / upper middle keys
    // compaction after the first two digit passes: the bucket that holds the median, copied out
    unsigned long long above_min;  // smallest key in the buckets above it
    unsigned long long m;          // elements in the bucket
};

template <typename T>
__global__ void __launch_bounds__(256) select_hist_kernel(const T *__restrict__ x, int64_t n, int shift, SelectState *st) {
    using K = typename KeyT<T>::type;
    __shared__ unsigned h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    const K prefix = (K)st->prefix, mask = (K)st->mask;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const K k = ordered_key(x[i]);
        if ((k & mask) == prefix) atomicAdd(&h[(unsigned)(k >> shift) & 255u], 1u);
    }
    __syncthreads();
    if (h[threadIdx.x]) atomicAdd(&st->hist[threadIdx.x], h[threadIdx.x]);
}

__global__ void __launch_bounds__(256) select_pick_kernel(SelectState *st, int shift, int which, int last) {
    // 256 threads: inclusive scan of the digit histogram, the digit whose cumulative count first exceeds the rank wins
    __shared__ unsigned long long cum[256];
    const int d = threadIdx.x;
    const unsigned mine = st->hist[d];
    cum[d] = mine;
    __syncthreads();
    for (int o = 1; o < 256; o <<= 1) {
        const unsigned long long add = d >= o ? cum[d - o] : 0ull;
        __syncthreads();
        cum[d] += add;
        __syncthreads();
    }
    const long long rank = st->rank;
    const unsigned long long before = cum[d] - mine;
    const bool winner = rank >= (long long)before && rank < (long long)cum[d];
    const bool none = d == 255 && rank >= (long long)cum[255];  // cannot happen for a consistent state: keep digit 255
    __syncthreads();
    st->hist[d] = 0;
    if (winner || none) {
        st->rank = rank - (long long)(none ? cum[254] : before);
        st->prefix |= (unsigned long long)d << shift;
        st->mask |= 255ull << shift;
        if (last) st->found[which] = st->prefix;
    }
}

__global__ void select_reset_kernel(SelectState *st, long long rank) {
    if (threadIdx.x == 0) {
        st->prefix = 0;
        st->mask = 0;
        st->rank = rank;
        st->above_min = ~0ull;
        st->m = 0;
    }
    st->hist[threadIdx.x] = 0;
}

// upper middle order statistic from the lower one in a single pass: it equals the lower key when that key is
// duplicated across the midpoint, else it is the smallest key above it
template <typename T>
__global__ void __launch_bounds__(256) select_upper_kernel(const T *__restrict__ x, int64_t n, SelectState *st) {
    using K = typename KeyT<T>::type;
    const K lo = (K)st->found[0];
    unsigned long long le = 0, above = ~0ull;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const K k = ordered_key(x[i]);
        le += (k <= lo);
        if (k > lo && (unsigned long long)k < above) above = (unsigned long long)k;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        le += __shfl_xor_sync(0xffffffffu, le, o);
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, above, o);
        above = other < above ? other : above;
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&st->prefix, le);       // prefix / mask are free after the digit passes: reuse as count / min
        atomicMin(&st->mask, above);
    }
}

template <typename T>
__global__ void select_finish_kernel(SelectState *st, int64_t n, T *med_out) {
    using K = typename KeyT<T>::type;
    const K lo = (K)st->found[0];
    const K hi = ((long long)st->prefix >= (long long)(n / 2 + 1)) ? lo : (K)st->mask;
    const T a = key_value(lo, T(0)), b = key_value(hi, T(0));
    *med_out = div_rn(add_rn(a, b), T(2));  // statistics.median: middle value, or (a + b) / 2 for even n
}

__global__ void select_prepare_upper_kernel(SelectState *st) {
    st->prefix = 0;
    st->mask = ~0ull;
}

// ---- exact median of one long window: sampled bracket + linear buckets (2 passes over the window) -----------------------
// The MSB digits of floating-point keys are a poor histogram (sign and exponent: nearly every sample of a sensor window
// falls into two or three of the 256 bins, and the shared-memory atomics serialise).  Instead:
//   sample   one CTA draws 1024 stratified pseudo-random samples and takes, from a linear histogram of them, a value
//            bracket [lo, hi) around the sample median that is ~16 sigma of the sampling error wide (about a quarter of
//            the window), or the single plateau value if the middle of the sample is one repeated value;
//   count    one pass over the window (128-bit loads): samples below the bracket are counted, samples inside it go
//            into 4096 LINEAR buckets (a monotone map, so buckets are ordered like the values);
//   compact  every CTA first re-derives, from the bucket counts, the bucket (or the region below / above the bracket,
//            should the sample have missed) that holds the lower middle order statistic and its rank inside; the
//            second pass then copies that bucket out (warp-aggregated append; typically a few hundred values) and
//            records the smallest value after it;
//   finish   one CTA ranks the copy (directly when it is small, else by an 8-bit radix select on the keys; immediate
//            when all copied values are equal), finds the upper middle value (same key if duplicated across the
//            midpoint, else the next key, inside the copy or after it) and writes statistics.median.
// Exact for any input: the bracket only steers where the resolution goes.
constexpr int kBrBuckets = 4096;
constexpr int kBrSample = 1024;
// threads per CTA of the two streaming kernels: 256 for short windows (more CTAs), 1024 for long ones (the per-CTA
// histogram clear / flush and the per-CTA pick are paid 148 x 2 times instead of 148 x 8 times)
constexpr int kBrThreadsSmall = 256, kBrThreadsLarge = 1024;

template <typename T>
struct BracketState {  // device resident, one per stream
    T lo, hi, scale;            // bracket [lo, hi), scale = buckets / (hi - lo)
    int mode;                   // winning region: -1 below the bracket, 0..B-1 a bucket, B at or above hi
    long long rank;             // rank of the lower middle order statistic inside the winning region
    unsigned long long below;   // samples < lo
    unsigned long long m;       // samples copied out
    unsigned long long above_min, kmin, kmax;  // smallest key after the region; smallest / largest key copied
    unsigned hist[kBrBuckets];
};

template <typename T>
__device__ __forceinline__ int br_bucket(T x, T lo, T scale) {  // for lo <= x < hi
    const int b = (int)(sub_rn(x, lo) * scale);  // monotone in x; NaN -> 0
    return b < 0 ? 0 : (b >= kBrBuckets ? kBrBuckets - 1 : b);
}
template <typename T>
__device__ __forceinline__ T next_above_t(T v) {
    T n = key_value(ordered_key(v) + 1, T(0));
    if (!(n > v)) n = key_value(ordered_key(v) + 2, T(0));  // -0.0 -> +0.0 compares equal
    return n;
}
__device__ __forceinline__ unsigned block_scan_incl_1024(unsigned v, unsigned *warp_tot /* 32 */) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += t;
    }
    if (lane == 31) warp_tot[warp] = v;
    __syncthreads();
    if (warp == 0) {
        unsigned w = warp_tot[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned t = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += t;
        }
        warp_tot[lane] = w;
    }
    __syncthreads();
    return v + (warp ? warp_tot[warp - 1] : 0u);
}

template <typename T>
__global__ void __launch_bounds__(1024) br_sample_kernel(const T *__restrict__ x, int64_t n, BracketState<T> *st, int64_t ld) {
    x += (int64_t)blockIdx.y * ld;  // blockIdx.y: window of the batch (its own state, bucket copy and result)
    st += blockIdx.y;
    __shared__ unsigned bins[1024];
    __shared__ unsigned wt[32];
    __shared__ T red_min[32], red_max[32];
    __shared__ int s_a, s_b;
    pdl_trigger();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int S = (int)(n < kBrSample ? n : kBrSample);
    const int64_t g = n / S;  // stratum size (>= 1)
    T v = T(0), mn = CUDART_INF, mx = -CUDART_INF;
    if (tid < S) {
        unsigned h = (unsigned)tid * 2654435761u;  // position inside the stratum: a hash, so periodic signals cannot alias
        h ^= h >> 15;
        h *= 2246822519u;
        h ^= h >> 13;
        v = x[(int64_t)tid * g + (int64_t)(h % (unsigned long long)g)];
        mn = mx = v;
    }
    bins[tid] = 0;
    for (int i = tid; i < kBrBuckets; i += 1024) st->hist[i] = 0;
    if (tid == 0) {
        s_a = 0;
        s_b = 1023;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const T a = __shfl_xor_sync(0xffffffffu, mn, o), b = __shfl_xor_sync(0xffffffffu, mx, o);
        mn = a < mn ? a : mn;
        mx = b > mx ? b : mx;
    }
    if (lane == 0) {
        red_min[warp] = mn;
        red_max[warp] = mx;
    }
    __syncthreads();
    for (int w = 0; w < 32; ++w) {
        mn = red_min[w] < mn ? red_min[w] : mn;
        mx = red_max[w] > mx ? red_max[w] : mx;
    }
    const T width = sub_rn(mx, mn);
    const bool flat = !(width > T(0)) || !(width < CUDART_INF);  // one value (or no finite range): bracket = that value
    const T sc = flat ? T(0) : T(1024) / width;
    if (!flat && tid < S) {
        int b = (int)(sub_rn(v, mn) * sc);
        b = b < 0 ? 0 : (b > 1023 ? 1023 : b);
        atomicAdd(&bins[b], 1u);
    }
    __syncthreads();
    // sample ranks S/2 -+ S/8: the population rank of a sample order statistic is off by ~N/(2 sqrt(S)) = N/64
    const unsigned mine = bins[tid];
    const unsigned cum = block_scan_incl_1024(mine, wt);
    const unsigned r0 = (unsigned)(S / 2 - S / 8), r1 = (unsigned)(S / 2 + S / 8);
    if (mine && cum - mine <= r0 && r0 < cum) s_a = tid;
    if (mine && cum - mine <= r1 && r1 < cum) s_b = tid;
    __syncthreads();
    if (tid == 0) {
        T lo = mn, hi = next_above_t(mn);
        if (!flat) {
            const int a = s_a, b = s_b;
            lo = add_rn(mn, (T)a * (width / T(1024)));
            hi = add_rn(mn, (T)(b + 1) * (width / T(1024)));
            if (a == 0) lo = mn;
            if (!(hi > lo)) hi = next_above_t(lo);
        }
        const T w2 = sub_rn(hi, lo);
        st->lo = lo;
        st->hi = hi;
        st->scale = (w2 > T(0) && (T)kBrBuckets / w2 < CUDART_INF) ? (T)kBrBuckets / w2 : T(0);  // 0: everything inside -> bucket 0
        st->mode = 0;
        st->rank = 0;
        st->below = 0;
        st->m = 0;
        st->above_min = ~0ull;
        st->kmin = ~0ull;
        st->kmax = 0ull;
    }
}

// One pass over x[0, n) with 128-bit loads, four in flight per thread (and the next four requested ahead): body(e, valid) sees E = 4 * 16/sizeof(T) elements
// per call (bit u of `valid`: e[u] is a sample).  Warp-uniform trip count (the bodies use warp collectives); the
// few samples before the first / after the last aligned 16-byte vector go through the same body, one per lane.
template <typename T, int NT, typename Body>
__device__ __forceinline__ void br_stream(const T *__restrict__ x, int64_t n, Body body) {
    constexpr int VEC = 16 / (int)sizeof(T), UNR = 4, E = VEC * UNR;
    const uintptr_t addr = reinterpret_cast<uintptr_t>(x);
    int64_t a0 = (int64_t)(((16 - (addr & 15)) & 15) / sizeof(T));  // first element on a 16-byte boundary
    if (a0 > n) a0 = n;
    const int64_t nvec = (n - a0) / VEC;
    const int4 *xv = reinterpret_cast<const int4 *>(x + a0);
    const int64_t per_it = (int64_t)gridDim.x * NT * UNR;
    // software pipeline: the next trip's four vectors are requested before the current ones are processed
    int4 nxt[UNR];
    auto fetch = [&](int64_t it0) {
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const int64_t iv = it0 + ((int64_t)blockIdx.x * UNR + u) * NT + threadIdx.x;
            nxt[u] = make_int4(0, 0, 0, 0);
            if (iv < nvec) nxt[u] = __ldg(xv + iv);
        }
    };
    if (nvec > 0) fetch(0);
    for (int64_t it0 = 0; it0 < nvec; it0 += per_it) {
        T e[E];
        unsigned valid = 0;
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const int64_t iv = it0 + ((int64_t)blockIdx.x * UNR + u) * NT + threadIdx.x;
            if (iv < nvec) valid |= ((1u << VEC) - 1u) << (u * VEC);
            const T *p = reinterpret_cast<const T *>(&nxt[u]);
#pragma unroll
            for (int q = 0; q < VEC; ++q) e[u * VEC + q] = p[q];
        }
        if (it0 + per_it < nvec) fetch(it0 + per_it);
        body(e, valid);
    }
    if (blockIdx.x == 0 && threadIdx.x < 32) {  // leftovers: < VEC in front, < VEC behind
        const int64_t tail0 = a0 + nvec * VEC;
        const int64_t left = a0 + (n - tail0);
        T e[E];
#pragma unroll
        for (int u = 0; u < E; ++u) e[u] = T(0);
        unsigned valid = 0;
        if ((int64_t)threadIdx.x < left) {
            const int64_t i = (int64_t)threadIdx.x < a0 ? (int64_t)threadIdx.x : tail0 + ((int64_t)threadIdx.x - a0);
            e[0] = x[i];
            valid = 1u;
        }
        body(e, valid);
    }
}

template <typename T, int NT>
__global__ void __launch_bounds__(NT) br_count_kernel(const T *__restrict__ x, int64_t n, BracketState<T> *st, int64_t ld) {
    x += (int64_t)blockIdx.y * ld;
    st += blockIdx.y;
    constexpr int E = 4 * 16 / (int)sizeof(T);
    __shared__ unsigned h[kBrBuckets];
    pdl_trigger();
    for (int i = threadIdx.x; i < kBrBuckets; i += NT) h[i] = 0;
    pdl_wait();  // the bracket comes from br_sample_kernel
    __syncthreads();
    const T lo = st->lo, hi = st->hi, scale = st->scale;
    unsigned below = 0;
    // Per 128-bit vector: two comparisons per sample decide below / inside / above (three quarters of a window are
    // outside the bracket and take nothing else); the buckets of a vector that is inside are computed together, and a
    // vector that falls into ONE bucket (smooth signals) costs one atomic.
    br_stream<T, NT>(x, n, [&](const T (&e)[E], unsigned valid) {
        constexpr int VEC = 16 / (int)sizeof(T);
#pragma unroll
        for (int v = 0; v < E / VEC; ++v) {
            const unsigned vmask = (valid >> (v * VEC)) & ((1u << VEC) - 1u);
            if (!vmask) continue;
            const bool full = vmask == (1u << VEC) - 1u;  // else: a leftover sample in slot 0
            bool in[VEC];
            bool any = false;
#pragma unroll
            for (int q = 0; q < VEC; ++q) {
                const T xq = e[v * VEC + q];
                const bool ok = q == 0 || full;
                const bool lt = ok && xq < lo;
                in[q] = ok && !(xq < lo) && !(xq >= hi);
                below += lt;
                any |= in[q];
            }
            if (!any) continue;
            int bk[VEC];
            bool same = true;
#pragma unroll
            for (int q = 0; q < VEC; ++q) {
                bk[q] = in[q] ? br_bucket<T>(e[v * VEC + q], lo, scale) : -1 - q;
                same &= bk[q] == bk[0];
            }
            if (same) {
                atomicAdd(&h[bk[0]], (unsigned)VEC);
            } else {
#pragma unroll
                for (int q = 0; q < VEC; ++q)
                    if (in[q]) atomicAdd(&h[bk[q]], 1u);
            }
        }
    });
    below = __reduce_add_sync(0xffffffffu, below);
    if ((threadIdx.x & 31) == 0 && below) atomicAdd(&st->below, (unsigned long long)below);
    __syncthreads();
    unsigned mine[kBrBuckets / NT];  // all shared-memory reads first: the reductions then go out back to back
#pragma unroll
    for (int u = 0; u < kBrBuckets / NT; ++u) mine[u] = h[threadIdx.x + u * NT];
#pragma unroll
    for (int u = 0; u < kBrBuckets / NT; ++u)
        if (mine[u]) atomicAdd(&st->hist[threadIdx.x + u * NT], mine[u]);
}

template <typename T, int NT>
__global__ void __launch_bounds__(NT) br_compact_kernel(const T *__restrict__ x, int64_t n, BracketState<T> *st,
                                                               T *__restrict__ bucket, int64_t ld) {
    x += (int64_t)blockIdx.y * ld;
    st += blockIdx.y;
    bucket += (int64_t)blockIdx.y * n;
    constexpr int E = 4 * 16 / (int)sizeof(T);
    constexpr int PER = kBrBuckets / NT;
    __shared__ unsigned long long wsum[NT / 32];
    __shared__ int s_mode;
    __shared__ long long s_rank;
    __shared__ unsigned long long blk[3][NT / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    pdl_trigger();
    pdl_wait();
    // ---- pick: which region holds rank (n-1)/2, and the rank inside it (every CTA derives the same answer) ----------
    {
        unsigned long long mine = 0;
        unsigned cnt[PER];
#pragma unroll
        for (int u = 0; u < PER; ++u) {
            cnt[u] = st->hist[threadIdx.x * PER + u];
            mine += cnt[u];
        }
        unsigned long long incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) wsum[warp] = incl;
        __syncthreads();
        unsigned long long ahead = 0, inside = 0;
        for (int w = 0; w < NT / 32; ++w) {
            if (w < warp) ahead += wsum[w];
            inside += wsum[w];
        }
        const long long r_lo = (long long)((n - 1) / 2), below = (long long)st->below;
        if (threadIdx.x == 0) {
            if (r_lo < below) {
                s_mode = -1;
                s_rank = r_lo;
            } else if (r_lo >= below + (long long)inside) {
                s_mode = kBrBuckets;
                s_rank = r_lo - below - (long long)inside;
            }
        }
        long long acc = below + (long long)(ahead + incl - mine);  // samples ahead of this thread's first bucket
        if (r_lo >= acc && r_lo < acc + (long long)mine) {
#pragma unroll
            for (int u = 0; u < PER; ++u) {
                if (r_lo >= acc && r_lo < acc + (long long)cnt[u]) {
                    s_mode = threadIdx.x * PER + u;
                    s_rank = r_lo - acc;
                }
                acc += cnt[u];
            }
        }
        __syncthreads();
    }
    const int mode = s_mode;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        st->mode = mode;
        st->rank = s_rank;
    }
    // ---- compact ---------------------------------------------------------------------------------------------------
    const T lo = st->lo, hi = st->hi, scale = st->scale;
    T amin = CUDART_INF;                       // smallest value after the region
    unsigned long long kmin = ~0ull, kmax = 0ull;  // key range of the copied values
    br_stream<T, NT>(x, n, [&](const T (&e)[E], unsigned valid) {
        constexpr int VEC = 16 / (int)sizeof(T);
        unsigned take = 0;
#pragma unroll
        for (int v = 0; v < E / VEC; ++v) {
            const unsigned vmask = (valid >> (v * VEC)) & ((1u << VEC) - 1u);
            if (!vmask) continue;
            const bool full = vmask == (1u << VEC) - 1u;
            if (mode >= 0 && mode < kBrBuckets) {  // the usual case: one bucket of the bracket
                bool in[VEC];
                bool any = false;
#pragma unroll
                for (int q = 0; q < VEC; ++q) {
                    const T xq = e[v * VEC + q];
                    const bool ok = q == 0 || full;
                    in[q] = ok && !(xq < lo) && !(xq >= hi);
                    if (ok && xq >= hi && xq < amin) amin = xq;
                    any |= in[q];
                }
                if (!any) continue;
#pragma unroll
                for (int q = 0; q < VEC; ++q) {
                    if (!in[q]) continue;
                    const T xq = e[v * VEC + q];
                    const int r = br_bucket<T>(xq, lo, scale);
                    if (r == mode) take |= 1u << (v * VEC + q);
                    else if (r > mode && xq < amin) amin = xq;
                }
            } else if (mode < 0) {  // the sample missed: the middle lies below the bracket
#pragma unroll
                for (int q = 0; q < VEC; ++q) {
                    const T xq = e[v * VEC + q];
                    const bool ok = q == 0 || full;
                    if (ok && xq < lo) take |= 1u << (v * VEC + q);
                    else if (ok && xq < amin) amin = xq;
                }
            } else {  // ... or at / above its upper end
#pragma unroll
                for (int q = 0; q < VEC; ++q)
                    if ((q == 0 || full) && e[v * VEC + q] >= hi) take |= 1u << (v * VEC + q);
            }
        }
        if (!__any_sync(0xffffffffu, take != 0)) return;
        unsigned incl = (unsigned)__popc(take);  // offsets inside the warp's append
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        const unsigned total = __shfl_sync(0xffffffffu, incl, 31);
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(&st->m, (unsigned long long)total);
        base = __shfl_sync(0xffffffffu, base, 0) + (incl - (unsigned)__popc(take));
#pragma unroll
        for (int u = 0; u < E; ++u) {
            if ((take >> u) & 1u) {
                bucket[base++] = e[u];
                const unsigned long long k = (unsigned long long)ordered_key(e[u]);
                kmin = k < kmin ? k : kmin;
                kmax = k > kmax ? k : kmax;
            }
        }
    });
    unsigned long long above = amin < CUDART_INF ? (unsigned long long)ordered_key(amin) : ~0ull;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long a = __shfl_xor_sync(0xffffffffu, above, o), b = __shfl_xor_sync(0xffffffffu, kmin, o),
                                 c = __shfl_xor_sync(0xffffffffu, kmax, o);
        above = a < above ? a : above;
        kmin = b < kmin ? b : kmin;
        kmax = c > kmax ? c : kmax;
    }
    if (lane == 0) {
        blk[0][warp] = above;
        blk[1][warp] = kmin;
        blk[2][warp] = kmax;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < NT / 32; ++w) {
            above = blk[0][w] < above ? blk[0][w] : above;
            kmin = blk[1][w] < kmin ? blk[1][w] : kmin;
            kmax = blk[2][w] > kmax ? blk[2][w] : kmax;
        }
        if (above != ~0ull) atomicMin(&st->above_min, above);
        if (kmin != ~0ull) atomicMin(&st->kmin, kmin);
        if (kmax != 0ull) atomicMax(&st->kmax, kmax);
    }
}

// rank `st->rank` of the copied region, the upper middle value and statistics.median itself, one CTA
template <typename T>
__global__ void __launch_bounds__(1024) br_finish_kernel(const T *__restrict__ bucket, BracketState<T> *st, int64_t n,
                                                          T *med_out) {
    bucket += (int64_t)blockIdx.y * n;
    st += blockIdx.y;
    med_out += blockIdx.y;
    using K = typename KeyT<T>::type;
    constexpr int kDirect = 256;  // copies up to this size are ranked directly (m^2 comparisons)
    __shared__ K keys[kDirect];
    __shared__ unsigned h[256];
    __shared__ unsigned wt[32];
    __shared__ unsigned long long s_prefix, s_mask, s_le, s_above, s_lo;
    __shared__ long long s_rank;
    pdl_trigger();
    pdl_wait();
    const long long m = (long long)st->m;
    const long long rank0 = st->rank;
    if (threadIdx.x == 0) {
        s_prefix = 0;
        s_mask = 0;
        s_rank = rank0;
        s_le = 0;
        s_above = ~0ull;
        s_lo = 0;
    }
    __syncthreads();
    K lo_key;
    if (st->kmin == st->kmax) {  // every copied value is the same (plateaus, constant windows)
        lo_key = (K)st->kmin;
        if (threadIdx.x == 0) s_le = (unsigned long long)m;
        __syncthreads();
    } else if (m <= kDirect) {
        // direct ranking: thread i counts the keys below its own (ties by position); two keys per thread
        for (int i = threadIdx.x; i < (int)m; i += 1024) keys[i] = ordered_key(bucket[i]);
        __syncthreads();
        for (int i = threadIdx.x; i < (int)m; i += 1024) {
            const K mine = keys[i];
            int below = 0, le = 0;
            K next = ~(K)0;
            for (int j = 0; j < (int)m; ++j) {
                const K o = keys[j];
                below += (o < mine) || (o == mine && j < i);
                le += o <= mine;
                if (o > mine && o < next) next = o;
            }
            if (below == (int)rank0) {  // exactly one thread: ranks with the position tie-break are a permutation
                s_lo = (unsigned long long)mine;
                s_le = (unsigned long long)le;
                s_above = next == ~(K)0 ? ~0ull : (unsigned long long)next;
            }
        }
        __syncthreads();
        lo_key = (K)s_lo;
    } else {
        // the copied keys agree in every bit above the highest one in which the smallest and largest differ: the digit
        // passes start at that byte
        const int top = 63 - __clzll((long long)(st->kmin ^ st->kmax));
        const int shift0 = (top / 8) * 8;
        if (threadIdx.x == 0) {
            const unsigned long long keep = shift0 + 8 >= 64 ? 0ull : ~((1ull << (shift0 + 8)) - 1ull);
            s_prefix = st->kmin & keep;
            s_mask = keep;
        }
        __syncthreads();
        for (int shift = shift0; shift >= 0; shift -= 8) {
            if (threadIdx.x < 256) h[threadIdx.x] = 0;
            __syncthreads();
            const K prefix = (K)s_prefix, mask = (K)s_mask;
            int cur = -1;
            unsigned run = 0;
            for (long long i = threadIdx.x; i < m; i += blockDim.x) {
                const K k = ordered_key(bucket[i]);
                if ((k & mask) == prefix) {
                    const int d = (int)((k >> shift) & 255u);
                    if (d == cur) {
                        ++run;
                    } else {
                        if (run) atomicAdd(&h[cur], run);
                        cur = d;
                        run = 1;
                    }
                }
            }
            if (run) atomicAdd(&h[cur], run);
            __syncthreads();
            const unsigned mine = threadIdx.x < 256 ? h[threadIdx.x] : 0u;
            const unsigned cum = block_scan_incl_1024(mine, wt);
            const long long rank = s_rank;
            __syncthreads();
            if (threadIdx.x < 256 && mine && rank >= (long long)(cum - mine) && rank < (long long)cum) {
                s_rank = rank - (long long)(cum - mine);
                s_prefix |= (unsigned long long)threadIdx.x << shift;
                s_mask |= 255ull << shift;
            }
            __syncthreads();
        }
        lo_key = (K)s_prefix;
        unsigned long long le = 0, above = ~0ull;
        for (long long i = threadIdx.x; i < m; i += blockDim.x) {
            const K k = ordered_key(bucket[i]);
            le += (k <= lo_key);
            if (k > lo_key && (unsigned long long)k < above) above = (unsigned long long)k;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            le += __shfl_xor_sync(0xffffffffu, le, o);
            const unsigned long long other = __shfl_xor_sync(0xffffffffu, above, o);
            above = other < above ? other : above;
        }
        if ((threadIdx.x & 31) == 0) {
            atomicAdd(&s_le, le);
            atomicMin(&s_above, above);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        // samples ahead of the copied region: the lower middle's global rank minus its rank inside the region
        const long long before = (long long)((n - 1) / 2) - rank0;
        const unsigned long long up = s_above < st->above_min ? s_above : st->above_min;
        const K hi_key = (before + (long long)s_le >= (long long)(n / 2 + 1)) ? lo_key : (K)up;
        const T a = key_value(lo_key, T(0)), b = key_value(hi_key, T(0));
        *med_out = div_rn(add_rn(a, b), T(2));  // statistics.median: middle value, or (a + b) / 2 for even n
    }
}

// windows of one call that share a launch set (blockIdx.y): a batch of 2^14 ... 2^17-point windows is launch bound otherwise
template <typename T>
static int64_t median_windows(int64_t n, int64_t batch) {
    const int64_t fit = std::max<int64_t>(1, ((int64_t)256 << 20) / std::max<int64_t>(1, n * (int64_t)sizeof(T)));
    return std::max<int64_t>(1, std::min<int64_t>(batch, std::min<int64_t>(fit, 256)));
}

// medians of `wins` windows (rows of d_x, `ld` apart): states[wins], d_bucket[wins * n], d_med[wins]
template <typename T>
int large_median(apda_ctx *ctx, cudaStream_t st, const T *d_x, int64_t n, int64_t ld, int64_t wins, void *state_raw, T *d_med,
                 T *d_bucket) {
    BracketState<T> *state = reinterpret_cast<BracketState<T> *>(state_raw);
    const bool big = n * (int64_t)sizeof(T) >= (int64_t)16 << 20;
    const int nt = big ? kBrThreadsLarge : kBrThreadsSmall;
    const int64_t per_cta = (int64_t)nt * 4 * (16 / (int)sizeof(T));  // samples per CTA and trip
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((n + per_cta - 1) / per_cta, (int64_t)ctx->sm_count * (2048 / nt)));
    const dim3 one(1, (unsigned)wins), many((unsigned)grid, (unsigned)wins);
    br_sample_kernel<T><<<one, 1024, 0, st>>>(d_x, n, state, ld);
    if (big) {
        APDA_CUDA(apda_launch_pdl(APDA_PDL_MEDIAN, br_count_kernel<T, kBrThreadsLarge>, many, dim3(nt), 0, st, d_x, n, state, ld));
        APDA_CUDA(apda_launch_pdl(APDA_PDL_MEDIAN, br_compact_kernel<T, kBrThreadsLarge>, many, dim3(nt), 0, st, d_x, n, state, d_bucket, ld));
    } else {
        APDA_CUDA(apda_launch_pdl(APDA_PDL_MEDIAN, br_count_kernel<T, kBrThreadsSmall>, many, dim3(nt), 0, st, d_x, n, state, ld));
        APDA_CUDA(apda_launch_pdl(APDA_PDL_MEDIAN, br_compact_kernel<T, kBrThreadsSmall>, many, dim3(nt), 0, st, d_x, n, state, d_bucket, ld));
    }
    APDA_CUDA(apda_launch_pdl(APDA_PDL_MEDIAN, br_finish_kernel<T>, one, dim3(1024), 0, st, (const T *)d_bucket, state, n, d_med));
    ctx->launches += 4;
    APDA_CUDA(cudaGetLastError());
    return APDA_OK;
}

// the earlier form (eight full histogram passes + one pass for the upper middle); kept as the reference implementation for
// apda_ctx_set_generic_only
template <typename T>
int large_median_passes(apda_ctx *ctx, cudaStream_t st, const T *d_x, int64_t n, SelectState *state, T *d_med) {
    const int bits = (int)sizeof(T) * 8;
    const int grid = (int)std::min<int64_t>((n + 255) / 256, (int64_t)ctx->sm_count * 8);
    select_reset_kernel<<<1, 256, 0, st>>>(state, (long long)((n - 1) / 2));
    for (int shift = bits - 8; shift >= 0; shift -= 8) {
        select_hist_kernel<T><<<grid, 256, 0, st>>>(d_x, n, shift, state);
        select_pick_kernel<<<1, 256, 0, st>>>(state, shift, 0, shift == 0);
        ctx->launches += 2;
    }
    select_prepare_upper_kernel<<<1, 1, 0, st>>>(state);
    select_upper_kernel<T><<<grid, 256, 0, st>>>(d_x, n, state);
    select_finish_kernel<T><<<1, 1, 0, st>>>(state, n, d_med);
    ctx->launches += 4;
    APDA_CUDA(cudaGetLastError());
    return APDA_OK;
}

struct PassPlan {
    int npass;
    int q[8];
};
static PassPlan make_plan(int n, int qmax) {
    PassPlan p;
    p.npass = (n + qmax - 1) / qmax;
    if (p.npass < 2) p.npass = 2;
    const int base = n / p.npass, rem = n % p.npass;
    for (int i = 0; i < p.npass; ++i) p.q[i] = base + (i < rem ? 1 : 0);
    return p;
}

// Tuning of the pass structure.  Defaults are the measured best on B200 (DESIGN.md, K2); the environment variables exist
// for same-box A/B runs (scripts/k2_ab.py) and are read once per process.
//   qmax      most radix-2 stages per pass (tile rows = 2^q)
//   max_tile  complex elements per shared-memory tile (rows * columns)
//   nt        threads per CTA of the tail passes;  minb: resident CTAs per SM the kernel is compiled for
struct K2Tune {
    int qmax, max_tile, nt, minb;
};
static int env_int(const char *name, int dflt) {
    const char *v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
}
template <typename T>
static K2Tune k2_tune() {
    static const K2Tune t = [] {
        K2Tune d;
        d.qmax = 10;  // fp32 could hold 2^11-row tiles, but 2^22 runs 22 % faster as (8, 7, 7) than as (11, 11)
        d.max_tile = sizeof(T) == 8 ? 4096 : 8192;  // 64 KB tiles
        d.nt = 256;  // 3 CTAs x 256 threads leave 85 registers per thread: 8 complex fp64 / 16 complex fp32 values in flight
        d.minb = 3;
        const char *sfx = sizeof(T) == 8 ? "64" : "32";
        char name[32];
        snprintf(name, sizeof(name), "APDA_K2_QMAX%s", sfx);
        d.qmax = env_int(name, d.qmax);
        snprintf(name, sizeof(name), "APDA_K2_TILE%s", sfx);
        d.max_tile = env_int(name, d.max_tile);
        snprintf(name, sizeof(name), "APDA_K2_NT%s", sfx);
        d.nt = env_int(name, d.nt);
        snprintf(name, sizeof(name), "APDA_K2_MINB%s", sfx);
        d.minb = env_int(name, d.minb);
        return d;
    }();
    return t;
}

// A pass whose grid fits the chip in one wave is launched the ordinary way: its dependent's CTAs would become resident
// at once and (measured, 2^20: 23 -> 39 us for the two passes) slow the pass down; with several waves the dependent
// only enters while the last wave drains (2^22: 71 -> 65 us, 2^24: 240 -> 235 us).
static int pass_pdl_group(const apda_ctx *ctx, dim3 grid, int group) {
    return (int64_t)grid.x * grid.y > 3 * (int64_t)ctx->sm_count ? group : 0;
}

template <typename T, int NT, int MINB>
static int launch_tail_tma(apda_ctx *ctx, cudaStream_t st, dim3 grid, size_t smem, const CUtensorMap &tm, int n, int s0, int q, int C,
                           const typename vec2<T>::type *twp, int zero_dc) {
    APDA_FUNC_SMEM(ctx, (large_tail_tma_kernel<T, NT, MINB>), smem);
    APDA_CUDA(apda_launch_pdl(pass_pdl_group(ctx, grid, APDA_PDL_TAIL), large_tail_tma_kernel<T, NT, MINB>, grid, dim3(NT), smem, st, tm, n,
                              s0, q, C, twp, zero_dc));
    return APDA_OK;
}

template <typename T, bool CPLX, int NT>
static int launch_head(apda_ctx *ctx, cudaStream_t st, dim3 grid, size_t smem, const T *d_samples, int64_t n_samples, int64_t ld, int n, int q,
                       int C, const typename vec2<T>::type *twp, typename vec2<T>::type *spec, const T *d_med) {
    APDA_FUNC_SMEM(ctx, (large_head_kernel<T, CPLX, NT>), smem);
    APDA_CUDA(apda_launch_pdl(pass_pdl_group(ctx, grid, APDA_PDL_HEAD), large_head_kernel<T, CPLX, NT>, grid, dim3(NT), smem, st, d_samples,
                              n_samples, ld, n, q, C, twp, spec, d_med));
    return APDA_OK;
}

// head pass and tail passes of `batch` <= 65535 windows (gridDim.y); d_med: the windows' centring constants or NULL
template <typename T>
static int large_passes(apda_ctx *ctx, cudaStream_t st, const T *d_samples, int64_t n_samples, int64_t ld, int64_t batch, int n,
                        const PassPlan &plan, int max_tile, const K2Tune &tune, const typename vec2<T>::type *twp, T *d_spec,
                        const T *d_med, bool complex_input) {
    using V2 = typename vec2<T>::type;
    {  // head pass
        const int q = plan.q[0];
        const int64_t cols = (int64_t)1 << (n - q);
        const int C = (int)std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>(max_tile >> q, 64), cols));
        const size_t smem = (size_t)C * ((1u << q) + 1) * sizeof(V2);
        dim3 grid((unsigned)(cols / C), (unsigned)batch);
        V2 *spec = reinterpret_cast<V2 *>(d_spec);
        // a tile that leaves room for one CTA per SM gets the most threads; otherwise 256 threads, so that three CTAs per
        // SM fit the register file (74 registers in fp32: 16 complex values per thread)
        const int hnt = smem > (96u << 10) ? 1024 : 256;
        if (complex_input) {
            if (hnt == 1024) APDA_TRY((launch_head<T, true, 1024>(ctx, st, grid, smem, d_samples, n_samples, ld, n, q, C, twp, spec, d_med)));
            else APDA_TRY((launch_head<T, true, 256>(ctx, st, grid, smem, d_samples, n_samples, ld, n, q, C, twp, spec, d_med)));
        } else {
            if (hnt == 1024) APDA_TRY((launch_head<T, false, 1024>(ctx, st, grid, smem, d_samples, n_samples, ld, n, q, C, twp, spec, d_med)));
            else APDA_TRY((launch_head<T, false, 256>(ctx, st, grid, smem, d_samples, n_samples, ld, n, q, C, twp, spec, d_med)));
        }
        ctx->launches++;
        APDA_CUDA(cudaGetLastError());
    }
    int s0 = plan.q[0];
    for (int p = 1; p < plan.npass; ++p) {
        const int q = plan.q[p];
        const int64_t cols = (int64_t)1 << s0;
        const int C = (int)std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>(max_tile >> q, 64), cols));
        const int64_t tiles = (cols / C) * ((int64_t)1 << (n - s0 - q));
        dim3 grid((unsigned)tiles, (unsigned)batch);
        const int zero_dc = (!complex_input && p == plan.npass - 1) ? 1 : 0;
        CUtensorMap tm;
        const size_t tma_smem = (size_t)C * (1u << q) * sizeof(V2) + 128;
        if (!ctx->generic_only && C * sizeof(V2) >= 16 && tma_smem <= (size_t)ctx->smem_optin &&
            make_tail_tmap<T>(&tm, d_spec, n, s0, q, C, batch)) {
            const bool one_per_sm = tma_smem > (size_t)ctx->smem_optin / 2;
            const int nt = one_per_sm ? std::max(tune.nt, 512) : tune.nt;
            if (nt >= 1024) APDA_TRY((launch_tail_tma<T, 1024, 1>(ctx, st, grid, tma_smem, tm, n, s0, q, C, twp, zero_dc)));
            else if (nt >= 512 && (one_per_sm || tune.minb <= 1)) APDA_TRY((launch_tail_tma<T, 512, 1>(ctx, st, grid, tma_smem, tm, n, s0, q, C, twp, zero_dc)));
            else if (nt >= 512 && tune.minb == 2) APDA_TRY((launch_tail_tma<T, 512, 2>(ctx, st, grid, tma_smem, tm, n, s0, q, C, twp, zero_dc)));
            else if (nt >= 512) APDA_TRY((launch_tail_tma<T, 512, 3>(ctx, st, grid, tma_smem, tm, n, s0, q, C, twp, zero_dc)));
            else if (tune.minb <= 2) APDA_TRY((launch_tail_tma<T, 256, 2>(ctx, st, grid, tma_smem, tm, n, s0, q, C, twp, zero_dc)));
            else APDA_TRY((launch_tail_tma<T, 256, 3>(ctx, st, grid, tma_smem, tm, n, s0, q, C, twp, zero_dc)));
        } else {
            const size_t smem = (size_t)(C + 1) * (1u << q) * sizeof(V2);
            if (smem > (size_t)ctx->smem_optin) {
                apda_set_error("fft_large: tile of 2^%d x %d does not fit shared memory", q, C);
                return APDA_ERR_UNSUPPORTED;
            }
            APDA_FUNC_SMEM(ctx, large_tail_kernel<T>, smem);
            APDA_CUDA(apda_launch_pdl(pass_pdl_group(ctx, grid, APDA_PDL_TAIL), large_tail_kernel<T>, grid, dim3(kThreads), smem, st,
                                      reinterpret_cast<V2 *>(d_spec), n, s0, q, C, twp, zero_dc));
        }
        ctx->launches++;
        APDA_CUDA(cudaGetLastError());
        s0 += q;
    }
    return APDA_OK;
}

}  // namespace

template <typename T>
int launch_fft_large(apda_ctx *ctx, cudaStream_t st, const T *d_samples, int64_t n_samples, int64_t ld, int64_t batch,
                     int64_t N, int flags, T *d_spec, bool complex_input) {
    using V2 = typename vec2<T>::type;
    const int n = ilog2_i64(N);
    if (n > 30) {
        apda_set_error("fft_large: N=2^%d outside the supported range", n);
        return APDA_ERR_UNSUPPORTED;
    }
    TwiddleTables tw;
    APDA_TRY(apda_get_twiddles(ctx, N, &tw));
    const V2 *twp = sizeof(T) == 8 ? reinterpret_cast<const V2 *>(tw.d64) : reinterpret_cast<const V2 *>(tw.d32);
    const K2Tune tune = k2_tune<T>();
    const int max_tile = tune.max_tile;  // complex elements per tile: 64 KB tiles let 3 CTAs per SM overlap load, compute and store
    const PassPlan plan = make_plan(n, tune.qmax);

    // centring constant per window
    T *d_med = nullptr;
    if (!complex_input && flags != APDA_CENTER_NONE) {
        // per-stream scratch: the two host-pipeline streams may run long transforms concurrently
        const size_t med_bytes = ((size_t)batch * sizeof(T) + 255) & ~(size_t)255;
        const int64_t wins = ctx->generic_only ? 1 : median_windows<T>(n_samples, batch);
        const size_t state_bytes = (std::max(sizeof(BracketState<T>) * (size_t)wins, sizeof(SelectState)) + 255) & ~(size_t)255;
        // states, medians, bucket copies (worst case: all samples of every window of a launch set)
        const size_t need = state_bytes + med_bytes + (size_t)wins * (size_t)n_samples * sizeof(T);
        auto &slot = ctx->stream_scratch[st];
        if (need > slot.second) {
            APDA_CUDA(cudaStreamSynchronize(st));
            APDA_TRY(apda_reserve(&slot.first, &slot.second, need));
        }
        SelectState *state = reinterpret_cast<SelectState *>(slot.first);
        d_med = reinterpret_cast<T *>(reinterpret_cast<char *>(slot.first) + state_bytes);
        T *d_bucket = reinterpret_cast<T *>(reinterpret_cast<char *>(slot.first) + state_bytes + med_bytes);
        if (ctx->generic_only) {
            for (int64_t w = 0; w < batch; ++w)
                APDA_TRY(large_median_passes<T>(ctx, st, d_samples + w * ld, n_samples, state, d_med + w));
        } else {
            for (int64_t w0 = 0; w0 < batch; w0 += wins)
                APDA_TRY(large_median<T>(ctx, st, d_samples + w0 * ld, n_samples, ld, std::min<int64_t>(wins, batch - w0), slot.first,
                                         d_med + w0, d_bucket));
        }
    }

    // head and tail passes put the windows on gridDim.y (at most 65535): longer batches run in launch sets of that many
    // windows, each with its own samples, spectra, centring constants and tensor maps
    constexpr int64_t kMaxSet = 65535;
    for (int64_t w0 = 0; w0 < batch; w0 += kMaxSet) {
        const int64_t wb = std::min<int64_t>(kMaxSet, batch - w0);
        const T *x = d_samples + w0 * (complex_input ? 2 * N : ld);
        T *y = d_spec + w0 * 2 * N;
        const T *med = d_med ? d_med + w0 : nullptr;
        APDA_TRY(large_passes<T>(ctx, st, x, n_samples, ld, wb, n, plan, max_tile, tune, twp, y, med, complex_input));
    }
    return APDA_OK;
}
template int launch_fft_large<double>(apda_ctx *, cudaStream_t, const double *, int64_t, int64_t, int64_t, int64_t, int,
                                      double *, bool);
template int launch_fft_large<float>(apda_ctx *, cudaStream_t, const float *, int64_t, int64_t, int64_t, int64_t, int,
                                     float *, bool);
