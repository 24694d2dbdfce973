// K1-general's building blocks (exact block median, one window's radix-2 transform in shared memory), shared by
// fft_smem.cu and the fp32 tie resolver (resolve_ties.cu).  See fft_smem.cu for the reference behaviour reproduced.
#pragma once
#include <math_constants.h>

#include "common.cuh"

namespace {

constexpr int kThreads = 256;

// ---- exact order statistic: MSB-first 8-bit radix select over order-preserving keys held in shared memory --------
template <typename K>
__device__ K block_select_rank(const K *keys, int n, int rank, unsigned *hist /*256*/, unsigned *bcast /*2*/) {
    constexpr int kBits = sizeof(K) * 8;
    K prefix = 0, mask = 0;
    for (int shift = kBits - 8; shift >= 0; shift -= 8) {
        for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
        __syncthreads();
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            K k = keys[i];
            if ((k & mask) == prefix) atomicAdd(&hist[(unsigned)(k >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (threadIdx.x < 32) {  // warp 0: find the digit whose cumulative count crosses `rank`
            unsigned lane = threadIdx.x;
            unsigned local[8], s = 0;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                local[q] = hist[lane * 8 + q];
                s += local[q];
            }
            unsigned incl = s;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= (unsigned)o) incl += t;
            }
            unsigned excl = incl - s;
            if ((unsigned)rank >= excl && (unsigned)rank < incl) {
                unsigned c = excl;
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    if ((unsigned)rank >= c && (unsigned)rank < c + local[q]) {
                        bcast[0] = lane * 8 + q;
                        bcast[1] = (unsigned)rank - c;
                    }
                    c += local[q];
                }
            }
        }
        __syncthreads();
        prefix |= (K)bcast[0] << shift;
        mask |= (K)255 << shift;
        rank = (int)bcast[1];
        __syncthreads();
    }
    return prefix;
}

// statistics.median of vals[0..n): odd -> middle order statistic, even -> (a + b) / 2 of the two middle ones.
template <typename T, typename K>
__device__ T block_median(const T *vals, K *keys, int n, unsigned *hist, unsigned *bcast) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) keys[i] = ordered_key(vals[i]);
    __syncthreads();
    if (n & 1) return key_value(block_select_rank<K>(keys, n, n / 2, hist, bcast), T(0));
    K lo = block_select_rank<K>(keys, n, n / 2 - 1, hist, bcast);
    // upper middle: equals lo when lo is duplicated across the midpoint, else the smallest key above lo
    unsigned le = 0;
    K above = ~(K)0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        K k = keys[i];
        le += (k <= lo);
        if (k > lo && k < above) above = k;
    }
    if (threadIdx.x == 0) {
        bcast[0] = 0;
        hist[0] = 0xffffffffu;
        hist[1] = 0xffffffffu;
    }
    __syncthreads();
    atomicAdd(&bcast[0], le);
    if (sizeof(K) == 8) {
        // 64-bit min via two 32-bit rounds (high word, then low word among matching highs)
        atomicMin(&hist[0], (unsigned)((uint64_t)above >> 32));
        __syncthreads();
        if ((unsigned)((uint64_t)above >> 32) == hist[0]) atomicMin(&hist[1], (unsigned)above);
    } else {
        atomicMin(&hist[1], (unsigned)above);
    }
    __syncthreads();
    K hi_key = (bcast[0] >= (unsigned)(n / 2 + 1)) ? lo
               : (sizeof(K) == 8 ? (K)(((uint64_t)hist[0] << 32) | hist[1]) : (K)hist[1]);
    __syncthreads();
    T a = key_value(lo, T(0)), b = key_value(hi_key, T(0));
    return div_rn(add_rn(a, b), T(2));
}

template <typename T>
struct KeyOf;
template <>
struct KeyOf<double> {
    using type = uint64_t;
};
template <>
struct KeyOf<float> {
    using type = uint32_t;
};

// ---- K1 general kernel -------------------------------------------------------------------------------------------
// dynamic shared memory: N complex<T> (transform; doubles as the select-key buffer) followed by N T (raw samples).
// Real rows of S (S = float, T = double: fp32 samples widened exactly at the load) are read from samples + win*ld; the
// spectrum goes to spec + spec_win*N.
template <typename T, bool FAITHFUL, bool COMPLEX_IN, typename S = T>
__device__ void fft_smem_window(const int64_t win, const S *__restrict__ samples, int n_samples, int64_t ld, int N, int logN,
                                const typename vec2<T>::type *__restrict__ tw,
                                typename vec2<T>::type *__restrict__ spec, int center, const int64_t spec_win) {
    using V2 = typename vec2<T>::type;
    using K = typename KeyOf<T>::type;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ unsigned hist[256];
    __shared__ unsigned bcast[2];
    __shared__ double red[kThreads / 32];
    V2 *y = reinterpret_cast<V2 *>(smem_raw);
    const int tid = threadIdx.x;

    if (COMPLEX_IN) {
        const V2 *x = reinterpret_cast<const V2 *>(samples) + win * (int64_t)N;
        for (int i = tid; i < N; i += kThreads) y[i] = x[__brev((unsigned)i) >> (32 - logN)];
    } else {
        T *raw = reinterpret_cast<T *>(y + N);
        K *keys = reinterpret_cast<K *>(y);  // the transform buffer is free until the scatter below
        const S *x = samples + win * ld;
        for (int i = tid; i < n_samples; i += kThreads) raw[i] = x[i];
        __syncthreads();
        T med = T(0);
        if (n_samples == 0) {
            // ragged batches only: an empty window (the reference returns [0]; flagged in the record status)
        } else if (center == APDA_CENTER_MEDIAN) {
            med = block_median<T, K>(raw, keys, n_samples, hist, bcast);
        } else if (center == APDA_CENTER_MEAN) {
            double s = 0.0;
            for (int i = tid; i < n_samples; i += kThreads) s += (double)raw[i];
            s = warp_sum(s);
            if ((tid & 31) == 0) red[tid >> 5] = s;
            __syncthreads();
            double tot = 0.0;
            for (int w = 0; w < kThreads / 32; ++w) tot += red[w];
            med = (T)(tot / (double)n_samples);
        }
        for (int i = tid; i < N; i += kThreads) {
            int src = (int)(__brev((unsigned)i) >> (32 - logN));
            V2 v;
            v.x = src < n_samples ? sub_rn(raw[src], med) : T(0);
            v.y = T(0);
            y[i] = v;
        }
    }
    __syncthreads();

    for (int s = 0; s < logN; ++s) {
        const int half = 1 << s;
        const V2 *t = tw + (half - 1);
        for (int b = tid; b < (N >> 1); b += kThreads) {
            int j = b & (half - 1);
            int lo = ((b >> s) << (s + 1)) + j;
            int hi = lo + half;
            V2 w = __ldg(t + j);
            V2 u = y[lo], v = y[hi], p, q;
            T vr, vi;
            if (FAITHFUL) {
                vr = sub_rn(mul_rn(v.x, w.x), mul_rn(v.y, w.y));
                vi = add_rn(mul_rn(v.x, w.y), mul_rn(v.y, w.x));
            } else {
                vr = v.x * w.x - v.y * w.y;
                vi = v.x * w.y + v.y * w.x;
            }
            p.x = add_rn(u.x, vr);
            p.y = add_rn(u.y, vi);
            q.x = sub_rn(u.x, vr);
            q.y = sub_rn(u.y, vi);
            y[lo] = p;
            y[hi] = q;
        }
        __syncthreads();
    }

    V2 *out = spec + spec_win * (int64_t)N;
    for (int i = tid; i < N; i += kThreads) {
        V2 v = y[i];
        if (!COMPLEX_IN && i == 0) v.x = v.y = T(0);
        out[i] = v;
    }
}

}  // namespace
