// K3-general's per-window pickers (magnitudes -> statistics -> candidates -> flexible / rigid picker -> record), shared
// by peaks.cu and the fp32 tie resolver (resolve_ties.cu).  See peaks.cu for the reference behaviour reproduced.
#pragma once
#include <math_constants.h>

#include "common.cuh"
#include "peaks_common.cuh"

namespace {

template <typename T>
__device__ void load_magnitudes(const typename vec2<T>::type *spec, T *mags, int half) {
    // four independent loads in flight per thread before the (long) magnitude arithmetic consumes them
    const int step = blockDim.x;
    int i = threadIdx.x;
    for (; i + 3 * step < half; i += 4 * step) {
        typename vec2<T>::type v0 = spec[i], v1 = spec[i + step], v2 = spec[i + 2 * step], v3 = spec[i + 3 * step];
        mags[i] = magnitude(v0.x, v0.y);
        mags[i + step] = magnitude(v1.x, v1.y);
        mags[i + 2 * step] = magnitude(v2.x, v2.y);
        mags[i + 3 * step] = magnitude(v3.x, v3.y);
    }
    for (; i < half; i += step) {
        typename vec2<T>::type v = spec[i];
        mags[i] = magnitude(v.x, v.y);
    }
    __syncthreads();
}

struct Layout {  // per-window scratch: magnitudes, candidate indices, surviving candidates
    size_t mags_off, cand_off, found_off, acc_off, bytes;
    int cap;
};
template <typename T>
__host__ __device__ inline Layout make_layout(int half) {
    Layout l;
    l.cap = half / 4 + 8;  // bins above mean+2*sigma are < 20 % of all bins (Cantelli), local maxima at most half of those
    l.mags_off = 0;
    size_t o = ((size_t)half * sizeof(T) + 15) & ~(size_t)15;
    l.found_off = o;
    o += (size_t)l.cap * sizeof(Found);
    l.cand_off = o;
    o += (size_t)l.cap * sizeof(int);
    l.acc_off = o;  // accepted peaks (slot / bin index): any k up to cap, not a fixed-size array
    o += (size_t)l.cap * sizeof(int);
    l.bytes = (o + 15) & ~(size_t)15;
    return l;
}

// ---- flexible-structure picker ------------------------------------------------------------------------------------
template <typename T, bool SMEM>
__device__ void peaks_prominence_window(const int64_t win, const typename vec2<T>::type *__restrict__ spec, int64_t n,
                                        int half, double fs_all, const double *__restrict__ d_fs, int k, int rec_cap,
                                        unsigned char *__restrict__ recs, unsigned char *__restrict__ ws,
                                        const int64_t spec_win) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ dd red[64];
    __shared__ Stats stats_s;
    __shared__ int ncand_s, nfound_s;
    const Layout lay = make_layout<T>(half);
    unsigned char *base = SMEM ? smem_raw : ws + (size_t)blockIdx.x * lay.bytes;
    T *mags = reinterpret_cast<T *>(base + lay.mags_off);
    Found *found = reinterpret_cast<Found *>(base + lay.found_off);
    int *cand = reinterpret_cast<int *>(base + lay.cand_off);
    int *acc_slot = reinterpret_cast<int *>(base + lay.acc_off);
    const int tid = threadIdx.x;
    unsigned char *rec = recs + win * APDA_REC_BYTES(rec_cap);
    const double fs = d_fs ? d_fs[win] : fs_all;
    const double df = div_rn(fs, (double)n);

    __shared__ int tie_s;
    if (tid == 0) ncand_s = nfound_s = tie_s = 0;
    load_magnitudes<T>(spec + spec_win * n, mags, half);
    const Stats st = block_stats<T>(mags, half, red, &stats_s);

    for (int j = 1 + tid; j < half - 1; j += blockDim.x) {
        T m = mags[j];
        if (m > mags[j - 1] && m > mags[j + 1] && (double)m > st.thr) {
            int pos = atomicAdd(&ncand_s, 1);
            if (pos < lay.cap) cand[pos] = j;
        }
        if (sizeof(T) == 4 && fp32_tie_top(mags, half, j, m, st.thr)) tie_s = 1;
    }
    __syncthreads();
    const int ncand = min(ncand_s, lay.cap);
    int status = (ncand_s > lay.cap ? APDA_STATUS_TRUNCATED : 0) | (tie_s ? APDA_STATUS_FP32_TIE : 0);

    const int warp = tid >> 5, nwarp = blockDim.x >> 5, lane = tid & 31;
    const double half_sd = mul_rn(0.5, st.sd);
    for (int c = warp; c < ncand; c += nwarp) {
        const int j = cand[c];
        const T prom = warp_prominence<T>(mags, half, j);
        if (!((double)prom > half_sd)) continue;
        const int bins = half_power_bins<T>(mags, half, prom, j);
        const double width_hz = mul_rn((double)bins, df);
        if (!(width_hz > 0.0)) continue;
        const double fn = mul_rn((double)j, df);
        const double q = div_rn(fn, width_hz);
        const double damping = div_rn(1.0, mul_rn(2.0, q));
        if (0.001 <= damping && damping <= 0.07 && lane == 0) {
            int pos = atomicAdd(&nfound_s, 1);
            Found f;
            f.rmag = round_dec4((double)mags[j]);
            f.prom = (double)prom;
            f.idx = j;
            f.width = bins;
            found[pos] = f;  // pos < cap because nfound <= ncand
        }
    }
    __syncthreads();

    // sorted(candidates, key=rounded mag, reverse=True) is stable, so ties keep ascending idx; the greedy "hump"
    // exclusion then walks that order.  Warp 0 extracts the order one element at a time.
    if (warp == 0) {
        const int nfound = nfound_s;
        int na = 0;
        double prev_mag = CUDART_INF;
        int prev_idx = -1;
        while (na < k) {
            double best = -1.0;
            int best_idx = 0x7fffffff, best_e = -1;
            for (int e = lane; e < nfound; e += 32) {
                double r = found[e].rmag;
                int ix = found[e].idx;
                bool after_prev = r < prev_mag || (r == prev_mag && ix > prev_idx);
                if (after_prev && (r > best || (r == best && ix < best_idx))) {
                    best = r;
                    best_idx = ix;
                    best_e = e;
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                double r = __shfl_xor_sync(0xffffffffu, best, o);
                int ix = __shfl_xor_sync(0xffffffffu, best_idx, o);
                int e = __shfl_xor_sync(0xffffffffu, best_e, o);
                if (e >= 0 && (best_e < 0 || r > best || (r == best && ix < best_idx))) {
                    best = r;
                    best_idx = ix;
                    best_e = e;
                }
            }
            if (best_e < 0) break;
            prev_mag = best;
            prev_idx = best_idx;
            const double cf = round_dec4(mul_rn((double)best_idx, df));
            bool hump = false;
            for (int a = 0; a < na && !hump; ++a) {
                const double af = round_dec4(mul_rn((double)found[acc_slot[a]].idx, df));
                const double rel = div_rn(fabs(sub_rn(cf, af)), af);
                if (rel < 0.05) {
                    const double ratio = div_rn(found[best_e].prom, best);
                    if (ratio < 0.10) hump = true;
                }
            }
            if (!hump) {
                if (lane == 0) acc_slot[na] = best_e;
                ++na;
            }
            __syncwarp();
        }
        if (lane == 0) {
            write_rec_header(rec, na, status);
            for (int a = 0; a < rec_cap; ++a) {
                if (a < na) {
                    const Found f = found[acc_slot[a]];
                    write_rec_peak(rec, a, f.idx, f.width, (double)mags[f.idx], f.prom);
                } else {
                    write_rec_peak(rec, a, -1, 0, 0.0, 0.0);
                }
            }
        }
    }
}

// ---- rigid-structure picker -----------------------------------------------------------------------------------------
template <typename T, bool SMEM>
__device__ void peaks_resolution_window(const int64_t win, const typename vec2<T>::type *__restrict__ spec, int64_t n,
                                        int half, double fs_all, const double *__restrict__ d_fs, int k, int rec_cap,
                                        unsigned char *__restrict__ recs, unsigned char *__restrict__ ws,
                                        const int64_t spec_win) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ dd red[64];
    __shared__ Stats stats_s;
    __shared__ double best_m[32];
    __shared__ int best_j[32];
    __shared__ int ctl[4];  // chosen idx, zero start, zero end, accepted count
    const Layout lay = make_layout<T>(half);
    unsigned char *base = SMEM ? smem_raw : ws + (size_t)blockIdx.x * lay.bytes;
    T *mags = reinterpret_cast<T *>(base + lay.mags_off);
    int *acc_idx = reinterpret_cast<int *>(base + lay.acc_off);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = blockDim.x >> 5;
    unsigned char *rec = recs + win * APDA_REC_BYTES(rec_cap);
    const double fs = d_fs ? d_fs[win] : fs_all;
    const double df = div_rn(fs, (double)n);
    const double distance = sub_rn(mul_rn(2.0, df), mul_rn(1.0, df));  // frequencies[2] - frequencies[1]

    load_magnitudes<T>(spec + spec_win * n, mags, half);
    const Stats st = block_stats<T>(mags, half, red, &stats_s);
    __shared__ int tie_s;
    if (tid == 0) ctl[3] = tie_s = 0;
    __syncthreads();
    if (sizeof(T) == 4) {  // on the original magnitudes (the zeroing below makes equal bins of its own)
        for (int j = 1 + tid; j < half - 1; j += blockDim.x)
            if (fp32_tie_top(mags, half, j, mags[j], st.thr)) tie_s = 1;
        __syncthreads();
    }

    while (true) {
        // arg-max over strict local maxima above the threshold; ties resolve to the lowest index (first wins)
        double bm = -1.0;
        int bj = -1;
        for (int j = 1 + tid; j < half - 1; j += blockDim.x) {
            T m = mags[j];
            if (m > mags[j - 1] && m > mags[j + 1] && (double)m > bm && (double)m > st.thr) {
                bm = (double)m;
                bj = j;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            double m2 = __shfl_xor_sync(0xffffffffu, bm, o);
            int j2 = __shfl_xor_sync(0xffffffffu, bj, o);
            if (j2 >= 0 && (bj < 0 || m2 > bm || (m2 == bm && j2 < bj))) {
                bm = m2;
                bj = j2;
            }
        }
        if (lane == 0) {
            best_m[warp] = bm;
            best_j[warp] = bj;
        }
        __syncthreads();
        if (tid == 0) {
            for (int w = 1; w < nwarp; ++w) {
                if (best_j[w] >= 0 && (bj < 0 || best_m[w] > bm || (best_m[w] == bm && best_j[w] < bj))) {
                    bm = best_m[w];
                    bj = best_j[w];
                }
            }
            ctl[0] = bj;
            if (bj >= 0) {
                int na = ctl[3];
                const double f = mul_rn((double)bj, df);
                const int w2 = half_height_bins<T>(mags, half, bj);
                bool separated = true;
                for (int a = 0; a < na && separated; ++a) {
                    const int w1 = half_height_bins<T>(mags, half, acc_idx[a]);
                    double rs = 0.0;
                    if (w1 + w2 != 0) {
                        int dist = bj - acc_idx[a];
                        if (dist < 0) dist = -dist;
                        rs = div_rn(mul_rn(1.18, (double)dist), (double)(w1 + w2));
                    }
                    if (!(rs >= 1.5)) separated = false;
                }
                if (separated) {
                    acc_idx[na] = bj;
                    write_rec_peak(rec, na, bj, w2, bm, 0.0);
                    ctl[3] = na + 1;
                }
                double reach_d = rint(div_rn(mul_rn(f, 0.02), distance));  // Python round(): half to even
                if (!(reach_d >= 0.0)) reach_d = 0.0;
                if (reach_d > (double)half) reach_d = (double)half;
                const int reach = (int)reach_d;
                ctl[1] = max(0, bj - reach);
                ctl[2] = min(half, bj + reach + 1);
            }
        }
        __syncthreads();
        if (ctl[0] < 0) break;
        for (int j = ctl[1] + tid; j < ctl[2]; j += blockDim.x) mags[j] = T(0);
        const bool full = ctl[3] >= k;
        __syncthreads();
        if (full) break;
    }
    if (tid == 0) {
        const int na = ctl[3];
        write_rec_header(rec, na, tie_s ? APDA_STATUS_FP32_TIE : 0);
        for (int a = na; a < rec_cap; ++a) write_rec_peak(rec, a, -1, 0, 0.0, 0.0);
    }
}

}  // namespace
