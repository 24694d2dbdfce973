// Batched ingest of sensor .log sample lines (SURVEY 8f rank 2): many logs' sample regions -> sample arrays on the
// device, without a Python float() per token.
//
// Reference behaviour reproduced (utils/load_data.py:67-80): the region after the four header lines is split into lines
// (universal newlines) and each line at ';'; every non-empty piece goes through float(); pieces that do not parse and
// non-finite values are dropped; the rest are the samples, in file order.
// Device grammar (decided exactly): optional sign, digits with at most one '.', at most 15 significant digits and 22
// fractional digits -> value = M / 10^f with one correctly rounded division (both exact in binary64), which is what
// float() returns for such text (the sensor logs are written with "%8.6f", protocol_decoder.py:174).  Pieces that
// contain a character float() could never accept in a finite number are dropped; pieces float() might accept in a
// form the kernel does not decide (exponents, '_' digit separators, > 15 significant digits, non-ASCII) raise flag
// bit 0 for that log, and the host re-parses that log with float() (apda-fft_b200/utils/load_data.py).
#include "common.cuh"

namespace {

__device__ __forceinline__ bool is_delim(unsigned char c) { return c == ';' || c == '\n' || c == '\r'; }
__device__ __forceinline__ bool is_space(unsigned char c) { return c == ' ' || (c >= 9 && c <= 13) || (c >= 28 && c <= 31); }

// classify / parse the piece text[b, e): 1 = sample (value in *out), 0 = dropped, -1 = undecided (host fallback)
__device__ int parse_piece(const unsigned char *text, int64_t b, int64_t e, double *out) {
    while (b < e && is_space(text[b])) ++b;
    while (e > b && is_space(text[e - 1])) --e;
    if (b == e) return 0;  // float('') / float(' ') -> ValueError
    bool only_numeric_chars = true, non_ascii = false;
    for (int64_t i = b; i < e; ++i) {
        const unsigned char c = text[i];
        if (c >= 0x80) non_ascii = true;
        if (!((c >= '0' && c <= '9') || c == '+' || c == '-' || c == '.' || c == '_' || c == 'e' || c == 'E'))
            only_numeric_chars = false;
    }
    if (non_ascii) return -1;           // e.g. non-ASCII digits are legal for float()
    if (!only_numeric_chars) return 0;  // letters other than e/E: "nan", "inf", markers -> never a finite float
    int64_t i = b;
    bool neg = false;
    if (text[i] == '+' || text[i] == '-') {
        neg = text[i] == '-';
        ++i;
    }
    unsigned long long m = 0;
    int sig = 0, frac = 0, ndig = 0;
    bool seen_dot = false;
    for (; i < e; ++i) {
        const unsigned char c = text[i];
        if (c >= '0' && c <= '9') {
            ++ndig;
            if (m != 0 || c != '0') ++sig;
            if (sig > 15) return -1;
            m = m * 10ull + (unsigned long long)(c - '0');
            if (seen_dot) ++frac;
        } else if (c == '.' && !seen_dot) {
            seen_dot = true;
        } else {
            return -1;  // exponent, '_', second '.', inner sign: float() decides on the host
        }
    }
    if (ndig == 0) return 0;  // "+", ".", "-." -> ValueError
    if (frac > 22) return -1;
    double p = 1.0;
    for (int q = 0; q < frac; ++q) p *= 10.0;  // exact up to 1e22
    const double v = frac ? div_rn((double)m, p) : (double)m;
    *out = neg ? -v : v;
    return 1;
}

// log b's sample region is text[starts ? starts[b] : offsets[b], offsets[b + 1])
template <typename T>
__global__ void __launch_bounds__(256)
parse_samples_kernel(const unsigned char *__restrict__ text, const int64_t *__restrict__ offsets,
                     const int64_t *__restrict__ starts, int64_t ld, T *__restrict__ samples, int *__restrict__ n_valid,
                     int *__restrict__ flags) {
    __shared__ int warp_tot[8];
    __shared__ int flag_s;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t win = blockIdx.x;
    const int64_t r0 = starts ? starts[win] : offsets[win], r1 = offsets[win + 1];
    const int64_t per = (r1 - r0 + 255) / 256;
    const int64_t a = min(r0 + tid * per, r1), z = min(a + per, r1);
    if (tid == 0) flag_s = 0;
    __syncthreads();
    int cnt = 0, flag = 0;
    double v;
    for (int pass = 0; pass < 2; ++pass) {
        int pos = 0;
        if (pass == 1) {
            int incl = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
            }
            if (lane == 31) warp_tot[warp] = incl;
            __syncthreads();
            int base = 0, total = 0;
#pragma unroll
            for (int w = 0; w < 8; ++w) {
                if (w < warp) base += warp_tot[w];
                total += warp_tot[w];
            }
            pos = base + incl - cnt;
            if (tid == 0) {
                n_valid[win] = total < ld ? total : (int)ld;
                if (total > ld) atomicOr(&flag_s, 2);
            }
        }
        for (int64_t p = a; p < z; ++p) {
            // a piece belongs to the thread in whose range it starts
            if (is_delim(text[p]) || (p > r0 && !is_delim(text[p - 1]))) continue;
            int64_t q = p;
            while (q < r1 && !is_delim(text[q])) ++q;
            const int kind = parse_piece(text, p, q, &v);
            if (pass == 0) {
                if (kind == 1 && fabs(v) <= 1.7976931348623157e308) ++cnt;
                if (kind < 0) flag = 1;
            } else if (kind == 1 && fabs(v) <= 1.7976931348623157e308) {
                if (pos < ld) samples[win * ld + pos] = (T)v;
                ++pos;
            }
        }
        if (pass == 0 && flag) atomicOr(&flag_s, 1);
    }
    __syncthreads();
    if (tid == 0) flags[win] = flag_s;
}

// Whole .log files (utils/load_data.py:64-70 load_sensor): file b is text[offsets[b], offsets[b + 1]).  One warp per
// file reads at most APDA_LOG_HEAD_BYTES + 1 bytes of it:
//   - the ends of the first four lines with universal newlines ("\r", "\n", "\r\n"; load_data.split_log);
//   - flag 4 when no fifth line follows (load_sensor returns None);
//   - flag 8 when the header is not decided here: no fourth line end within APDA_LOG_HEAD_BYTES - 1 bytes, a byte
//     >= 0x80 or NUL in it (load_sensor decodes UTF-8 first), fewer than 4 ';' fields on line 0, or a rate field that
//     is not decided by parse_piece once every " Hz" is removed (float(rate.replace(" Hz", "")), load_data.py:42);
//   - starts[b]: where the sample region begins (offsets[b + 1], i.e. empty, when a flag is set), fs[b] (0 when a flag
//     is set) and the header bytes, NUL-padded to APDA_LOG_HEAD_BYTES (all zero when a flag is set).
constexpr int kRateChars = 64;  // longest rate field (after the " Hz" removal) the device decides

__global__ void __launch_bounds__(256)
log_layout_kernel(const unsigned char *__restrict__ text, const int64_t *__restrict__ offsets, int64_t batch,
                  int64_t *__restrict__ starts, double *__restrict__ fs, int *__restrict__ lflags,
                  unsigned char *__restrict__ head) {
    __shared__ unsigned char rate_s[8][kRateChars];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int64_t w = (int64_t)blockIdx.x * 8 + wib;
    if (w >= batch) return;  // whole warps only
    const int64_t o0 = offsets[w], o1 = offsets[w + 1];
    const int64_t lim = min(o1, o0 + APDA_LOG_HEAD_BYTES);
    int lines = 0;
    int64_t end = -1, e0 = -1;  // end of the 4th line's terminator, start of line 0's terminator
    bool bad = false;           // non-ASCII or NUL byte in the header
    for (int64_t base = o0; base < lim && end < 0; base += 32) {
        const int64_t p = base + lane;
        const unsigned char c = p < lim ? text[p] : 0;
        const bool term = p < lim && (c == '\r' || (c == '\n' && !(p > o0 && text[p - 1] == '\r')));
        const unsigned tm = __ballot_sync(0xffffffffu, term);
        const unsigned bm = __ballot_sync(0xffffffffu, p < lim && (c >= 0x80 || c == 0));
        if (lines == 0 && tm) e0 = base + __ffs(tm) - 1;
        if (lines + __popc(tm) >= 4) {
            unsigned m = tm;
            for (int i = lines; i < 3; ++i) m &= m - 1;  // drop the terminators of lines 1..3 still in this word
            const int t = __ffs(m) - 1;
            const int64_t tp = base + t;
            end = tp + ((text[tp] == '\r' && tp + 1 < o1 && text[tp + 1] == '\n') ? 2 : 1);
            bad = bad || (bm & ((2u << t) - 1u)) != 0;
        } else {
            lines += __popc(tm);
            bad = bad || bm != 0;
        }
    }
    int flag;
    if (end < 0)
        flag = (lim == o1 && !bad) ? 4 : 8;  // the whole file holds fewer than 4 line ends / the header is too long
    else if (end == o1)
        flag = bad ? 8 : 4;
    else
        flag = (bad || end - o0 > APDA_LOG_HEAD_BYTES - 1) ? 8 : 0;

    double rate = 0.0;
    if (flag == 0) {
        // line 0 is [o0, e0); field 2 (the rate) lies between its 2nd and 3rd ';'
        int semis = 0;
        int64_t f0 = -1, f1 = -1;
        for (int64_t base = o0; base < e0 && f1 < 0; base += 32) {
            const int64_t p = base + lane;
            unsigned m = __ballot_sync(0xffffffffu, p < e0 && text[p] == ';');
            while (m && f1 < 0) {
                const int t = __ffs(m) - 1;
                m &= m - 1;
                if (++semis == 2) f0 = base + t + 1;
                else if (semis == 3) f1 = base + t;
            }
        }
        int ok = 0;
        if (f1 >= 0 && lane == 0) {
            unsigned char *r = rate_s[wib];
            int n = 0;
            bool fits = true;
            for (int64_t p = f0; p < f1;) {
                if (p + 2 < f1 && text[p] == ' ' && text[p + 1] == 'H' && text[p + 2] == 'z') {
                    p += 3;
                    continue;
                }
                if (n == kRateChars) {
                    fits = false;
                    break;
                }
                r[n++] = text[p++];
            }
            ok = fits && parse_piece(r, 0, n, &rate) == 1;  // 0: float() raises or gives nan/inf; -1: not decided
        }
        ok = __shfl_sync(0xffffffffu, ok, 0);
        rate = __shfl_sync(0xffffffffu, rate, 0);
        if (!ok) flag = 8;
    }
    const int64_t hlen = flag ? 0 : end - o0;
    unsigned char *h = head + w * APDA_LOG_HEAD_BYTES;
    for (int i = lane; i < APDA_LOG_HEAD_BYTES; i += 32) h[i] = i < hlen ? text[o0 + i] : 0;
    if (lane == 0) {
        starts[w] = flag ? o1 : end;
        fs[w] = flag ? 0.0 : rate;
        lflags[w] = flag;
    }
}

// flags := layout flags | parse flags; a log with any flag gets the empty record (count 0, every slot idx -1 and zeros)
// with status APDA_STATUS_OTHER_LENGTH for "more than N samples" and APDA_STATUS_EMPTY for "fewer than 5 lines"
__global__ void log_finish_kernel(int64_t batch, int *__restrict__ lflags, const int *__restrict__ pflags,
                                  unsigned char *__restrict__ recs, int rec_cap) {
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= batch) return;
    const int fl = lflags[w] | pflags[w];
    lflags[w] = fl;
    if (!fl) return;
    unsigned char *rec = recs + w * APDA_REC_BYTES(rec_cap);
    int *hdr = reinterpret_cast<int *>(rec);
    hdr[0] = 0;
    hdr[1] = ((fl & 2) ? APDA_STATUS_OTHER_LENGTH : 0) | ((fl & 4) ? APDA_STATUS_EMPTY : 0);
    apda_peak *pk = reinterpret_cast<apda_peak *>(rec + 8);
    for (int i = 0; i < rec_cap; ++i) pk[i] = apda_peak{-1, 0, 0.0, 0.0};
}

}  // namespace

template <typename T>
int launch_parse_samples(apda_ctx *ctx, cudaStream_t st, const char *d_text, const int64_t *d_offsets, int64_t batch,
                         int64_t ld, T *d_samples, int *d_n_valid, int *d_flags, const int64_t *d_starts) {
    if (batch == 0) return APDA_OK;
    parse_samples_kernel<T><<<(unsigned)batch, 256, 0, st>>>(reinterpret_cast<const unsigned char *>(d_text), d_offsets,
                                                            d_starts, ld, d_samples, d_n_valid, d_flags);
    ctx->launches++;
    APDA_CUDA(cudaGetLastError());
    return APDA_OK;
}
template int launch_parse_samples<double>(apda_ctx *, cudaStream_t, const char *, const int64_t *, int64_t, int64_t,
                                          double *, int *, int *, const int64_t *);
template int launch_parse_samples<float>(apda_ctx *, cudaStream_t, const char *, const int64_t *, int64_t, int64_t, float *,
                                         int *, int *, const int64_t *);

int launch_log_layout(apda_ctx *ctx, cudaStream_t st, const char *d_text, const int64_t *d_offsets, int64_t batch,
                      int64_t *d_starts, double *d_fs, int *d_flags, char *d_head) {
    if (batch == 0) return APDA_OK;
    log_layout_kernel<<<(unsigned)((batch + 7) / 8), 256, 0, st>>>(reinterpret_cast<const unsigned char *>(d_text), d_offsets,
                                                                   batch, d_starts, d_fs, d_flags,
                                                                   reinterpret_cast<unsigned char *>(d_head));
    ctx->launches++;
    APDA_CUDA(cudaGetLastError());
    return APDA_OK;
}

int launch_log_finish(apda_ctx *ctx, cudaStream_t st, int64_t batch, int *d_flags, const int *d_parse_flags, void *d_rec,
                      int rec_cap) {
    if (batch == 0) return APDA_OK;
    log_finish_kernel<<<(unsigned)((batch + 255) / 256), 256, 0, st>>>(batch, d_flags, d_parse_flags,
                                                                       reinterpret_cast<unsigned char *>(d_rec), rec_cap);
    ctx->launches++;
    APDA_CUDA(cudaGetLastError());
    return APDA_OK;
}
