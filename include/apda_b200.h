/* apda_b200.h - C ABI of libapda_b200.so: the B200 (sm_100a) implementation of APDA-FFT's spectral hot path.
 *
 * The reference (Copojacaab/APDA-FFT) has no FFI layer: its hot path is three plain-Python modules.  Each entry
 * point below names the reference interface it stands in for (paths relative to the reference checkout); the
 * Python mirror in apda-fft_b200/{metrics,utils}/ binds them with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - every function returns an int status: APDA_OK (0) or a negative APDA_ERR_*; apda_last_error() gives the
 *     thread-local message of the last failure.  No exceptions, no exit(), no CPU fallback: without an sm_100
 *     device apda_ctx_create fails with APDA_ERR_NO_DEVICE.
 *   - an apda_ctx belongs to one host thread and one device.  "_dev" entry points take DEVICE pointers, enqueue
 *     on the context stream and return without synchronising (apda_sync waits).  "_host" entry points take HOST
 *     pointers, run H2D -> kernels -> D2H in a chunked two-stream pipeline and return when the results are in
 *     the caller's buffers.
 *   - spectra are interleaved (re, im) pairs, N bins per window, window b at offset b*2*N reals.
 *   - N is a power of two; n_samples <= N real samples per window are median-centred, then zero padded to N.
 */
#ifndef APDA_B200_H
#define APDA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define APDA_OK 0
#define APDA_ERR_INVALID (-1)      /* bad argument (NULL, non power-of-two N, n_samples > N, k out of range ...) */
#define APDA_ERR_NO_DEVICE (-2)    /* no CUDA device / not compute capability 10.x */
#define APDA_ERR_CUDA (-3)         /* a CUDA runtime call or kernel failed; message holds cudaGetErrorString */
#define APDA_ERR_NOMEM (-4)
#define APDA_ERR_UNSUPPORTED (-5)  /* size outside what the kernels cover */
#define APDA_ERR_STATS_MEAN (-6)   /* half spectrum empty: reference raises StatisticsError('mean requires at least one data point') */
#define APDA_ERR_STATS_STDEV (-7)  /* half spectrum has 1 bin: StatisticsError('stdev requires at least two data points') */

/* flags of apda_fft_* */
#define APDA_CENTER_MEDIAN 0  /* exact statistics.median of the n_samples real samples (reference behaviour, default) */
#define APDA_CENTER_MEAN 1    /* fp32 only, only legal when n_samples == N: block mean; bins >= 1 are unaffected (DESIGN.md) */
#define APDA_CENTER_NONE 2    /* input already centred by the caller */

/* One detected peak.  width_bins: flexible picker = max(right-left,1) of the half-power walk;
 * rigid picker = half-height width of the candidate when it was accepted.  prominence is 0 for the rigid picker. */
typedef struct apda_peak {
    int32_t idx;
    int32_t width_bins;
    double mag;        /* raw |X[idx]| (fp32 paths widen to double) */
    double prominence; /* raw, flexible picker only */
} apda_peak; /* 24 bytes */

/* Fixed 128-byte per-window record (rec_cap == 5).  For rec_cap != 5 a record is 8 + 24*rec_cap bytes with the
 * same header.  Peaks are in the reference's output order (flexible: descending rounded magnitude; rigid: discovery). */
typedef struct apda_peak_rec {
    int32_t count;  /* peaks found (<= k) */
    int32_t status; /* 0 ok, else a set of APDA_STATUS_* bits: the record is not (known to be) reference-equivalent */
    apda_peak pk[5];
} apda_peak_rec;

#define APDA_STATUS_TRUNCATED 1     /* internal candidate list overflowed (result truncated; unreachable by Cantelli's bound) */
#define APDA_STATUS_OTHER_LENGTH 4  /* ragged batch: the window's own padded length differs from N */
#define APDA_STATUS_EMPTY 8         /* ragged batch: empty window (the reference's pickers raise StatisticsError) */
#define APDA_STATUS_FP32_TIE 16     /* fp32 pickers (N <= 2^15): two adjacent bins above the threshold are equal in fp32 and form
                                     * the top of a peak; the strict local-maximum test reports no peak there, the fp64
                                     * reference (whose magnitudes differ below fp32 resolution) reports one.
                                     * apda_resolve_fp32_ties_{dev,host} replace such records by the fp64 path's.  Plateaus
                                     * of three or more equal bins are not flagged, so they are not resolved either. */
#define APDA_REC_BYTES(rec_cap) (8 + 24 * (int64_t)(rec_cap))
#define APDA_MAX_REC_CAP 64
/* Most peaks one window of n bins can report (candidates are strict local maxima above mean + 2 sigma of the half
 * spectrum: fewer than 20 % of its bins): the reference accepts any k (utils/get_peak_prominence.py:149,223,
 * utils/get_peak_resolution.py:80,94), so records may be as wide as max(APDA_MAX_REC_CAP, APDA_MAX_PEAKS(n)). */
#define APDA_MAX_PEAKS(n) ((int64_t)(n) / 8 + 8)

typedef struct apda_ctx apda_ctx;

/* ---- context ---------------------------------------------------------------------------------------------- */
int apda_ctx_create(int device, apda_ctx **out);
int apda_ctx_destroy(apda_ctx *ctx);
/* Run the _dev entry points on a caller-owned CUDA stream (e.g. torch.cuda.current_stream().cuda_stream; the value 0
 * is CUDA's legacy default stream).  apda_ctx_reset_stream goes back to the context's own non-blocking stream. */
int apda_ctx_set_stream(apda_ctx *ctx, void *cuda_stream);
int apda_ctx_reset_stream(apda_ctx *ctx);
/* Test/debug switch: on != 0 routes fp32 work through the general kernels instead of the specialised N=1024..8192 ones. */
int apda_ctx_set_generic_only(apda_ctx *ctx, int on);
int apda_sync(apda_ctx *ctx);
const char *apda_last_error(void);
int apda_version(void);
/* number of kernels this library has launched through ctx since creation (bench.py's gpu_launches) */
int64_t apda_launch_count(apda_ctx *ctx);

/* ---- K1/K2: FFT --------------------------------------------------------------------------------------------
 * replaces metrics/fft_iterativa.py:74-87 start_fft(samples, fs): median centre (:5-11), zero pad (:13-22),
 * bit reversal (:24-36), radix-2 DIT butterflies with the recurrence twiddles (:38-70), bin 0 := 0 (:85).
 * f64 is bit-faithful to the reference (no FMA, host-built recurrence twiddle table).  f32 is the fast path.
 * N <= 2^13 runs one shared-memory kernel per window batch in both precisions; N = 2^14 ... 2^30 runs the multi-pass
 * kernels (K2), for any batch.  fp32 N = 2^14 fits the shared-memory kernel too, but only ragged batches use it there. */
int apda_fft_f64_dev(apda_ctx *ctx, const double *d_samples, int64_t n_samples, int64_t ld, int64_t batch,
                     int64_t N, int flags, double *d_spec);
int apda_fft_f32_dev(apda_ctx *ctx, const float *d_samples, int64_t n_samples, int64_t ld, int64_t batch,
                     int64_t N, int flags, float *d_spec);
int apda_fft_f64_host(apda_ctx *ctx, const double *h_samples, int64_t n_samples, int64_t ld, int64_t batch,
                      int64_t N, int flags, double *h_spec);
int apda_fft_f32_host(apda_ctx *ctx, const float *h_samples, int64_t n_samples, int64_t ld, int64_t batch,
                      int64_t N, int flags, float *h_spec);
/* replaces metrics/fft_iterativa.py:38-70 fft(x) on complex input (no centring, no DC zeroing), N = 2^k */
int apda_fft_c2c_f64_host(apda_ctx *ctx, const double *h_in, int64_t batch, int64_t N, double *h_out);
/* replaces metrics/fft_iterativa.py:5-11 remove_dc_component(samples) */
int apda_center_f64_host(apda_ctx *ctx, const double *h_in, int64_t n, double *h_out);

/* ---- K3: peak pickers --------------------------------------------------------------------------------------
 * n = bins per window in the spectrum (the pickers read bins [0, n/2)); fs: one value for all windows when
 * d_fs/h_fs is NULL.  k <= rec_cap <= max(APDA_MAX_REC_CAP, APDA_MAX_PEAKS(n)); out: batch records of
 * APDA_REC_BYTES(rec_cap).
 * prominence: replaces utils/get_peak_prominence.py:149-226 get_top_peaks_prominence(res_fft, fs, k=4)
 * resolution: replaces utils/get_peak_resolution.py:80-128 get_top_peaks_resolution(fft_res, fs, k=5) */
int apda_peaks_prominence_f64_dev(apda_ctx *ctx, const double *d_spec, int64_t n, int64_t batch, double fs,
                                  const double *d_fs, int k, int rec_cap, void *d_rec);
int apda_peaks_prominence_f32_dev(apda_ctx *ctx, const float *d_spec, int64_t n, int64_t batch, double fs,
                                  const double *d_fs, int k, int rec_cap, void *d_rec);
int apda_peaks_resolution_f64_dev(apda_ctx *ctx, const double *d_spec, int64_t n, int64_t batch, double fs,
                                  const double *d_fs, int k, int rec_cap, void *d_rec);
int apda_peaks_resolution_f32_dev(apda_ctx *ctx, const float *d_spec, int64_t n, int64_t batch, double fs,
                                  const double *d_fs, int k, int rec_cap, void *d_rec);
int apda_peaks_prominence_f64_host(apda_ctx *ctx, const double *h_spec, int64_t n, int64_t batch, double fs,
                                   const double *h_fs, int k, int rec_cap, void *h_rec);
int apda_peaks_resolution_f64_host(apda_ctx *ctx, const double *h_spec, int64_t n, int64_t batch, double fs,
                                   const double *h_fs, int k, int rec_cap, void *h_rec);
int apda_peaks_prominence_f32_host(apda_ctx *ctx, const float *h_spec, int64_t n, int64_t batch, double fs,
                                   const double *h_fs, int k, int rec_cap, void *h_rec);
int apda_peaks_resolution_f32_host(apda_ctx *ctx, const float *h_spec, int64_t n, int64_t batch, double fs,
                                   const double *h_fs, int k, int rec_cap, void *h_rec);

/* ---- pipeline: samples -> records, spectra never leave HBM -------------------------------------------------
 * replaces the body of GT_FFT_v5.py:635-642 (start_fft followed by the picker selected by is_flexibile_structure).
 * flexible != 0 -> prominence picker, else resolution picker.  d_spec_ws: caller-provided spectrum workspace of
 * batch*2*N reals (it then holds the N-bin spectra apda_fft_* would write), or NULL to use the context's own - in which
 * case the fp32 FFT kernel only writes the bins [0, N/2) the pickers read (SURVEY.md 8d "half-spectrum pipeline":
 * 3*s*N + 128 bytes of HBM traffic per window instead of 4*s*N + 128; same records). */
int apda_analyze_f64_dev(apda_ctx *ctx, const double *d_samples, int64_t n_samples, int64_t ld, int64_t batch,
                         int64_t N, int flags, int flexible, double fs, const double *d_fs, int k, int rec_cap,
                         double *d_spec_ws, void *d_rec);
int apda_analyze_f32_dev(apda_ctx *ctx, const float *d_samples, int64_t n_samples, int64_t ld, int64_t batch,
                         int64_t N, int flags, int flexible, double fs, const double *d_fs, int k, int rec_cap,
                         float *d_spec_ws, void *d_rec);
int apda_analyze_f64_host(apda_ctx *ctx, const double *h_samples, int64_t n_samples, int64_t ld, int64_t batch,
                          int64_t N, int flags, int flexible, double fs, const double *h_fs, int k, int rec_cap,
                          void *h_rec);
int apda_analyze_f32_host(apda_ctx *ctx, const float *h_samples, int64_t n_samples, int64_t ld, int64_t batch,
                          int64_t N, int flags, int flexible, double fs, const double *h_fs, int k, int rec_cap,
                          void *h_rec);

/* One host process, several GPUs (SURVEY.md 8e; nothing like it in the reference, which analyses one file at a time,
 * GT_FFT_v5.py:466,620): ctxs[0..n_ctx) are contexts of different devices (or several contexts of one device), each owned
 * by this call for its duration.  The batch is sharded contiguously (context r: windows [r*ceil(batch/n_ctx), ...)), one
 * host thread per context runs the chunked pipeline of apda_analyze_*_host on its shard, and every device writes its
 * records into its rows of h_rec - the table a gather to rank 0 would produce, in window order, with no collective. */
int apda_multi_analyze_f32_host(apda_ctx **ctxs, int n_ctx, const float *h_samples, int64_t n_samples, int64_t ld,
                                int64_t batch, int64_t N, int flags, int flexible, double fs, const double *h_fs, int k,
                                int rec_cap, void *h_rec);
int apda_multi_analyze_f64_host(apda_ctx **ctxs, int n_ctx, const double *h_samples, int64_t n_samples, int64_t ld,
                                int64_t batch, int64_t N, int flags, int flexible, double fs, const double *h_fs, int k,
                                int rec_cap, void *h_rec);

/* Ragged batches: window b holds d_n_valid[b] <= n_max <= N samples (rows of ld reals); everything stays on the device
 * and nothing synchronises.  Windows of the common length n_max run on the specialised kernels, the others on the
 * general kernel with their own length.  Record status bit 2 (4): the window's own padded length differs from N (the
 * reference would transform it at that length); bit 3 (8): empty window.  Used by the ingest paths (wire decode, text
 * logs), where non-finite samples are dropped per window as utils/load_data.py:72-80 does. */
int apda_fft_ragged_f64_dev(apda_ctx *ctx, const double *d_samples, const int32_t *d_n_valid, int64_t n_max, int64_t ld,
                            int64_t batch, int64_t N, int flags, double *d_spec);
int apda_fft_ragged_f32_dev(apda_ctx *ctx, const float *d_samples, const int32_t *d_n_valid, int64_t n_max, int64_t ld,
                            int64_t batch, int64_t N, int flags, float *d_spec);
int apda_analyze_ragged_f64_dev(apda_ctx *ctx, const double *d_samples, const int32_t *d_n_valid, int64_t n_max,
                                int64_t ld, int64_t batch, int64_t N, int flags, int flexible, double fs,
                                const double *d_fs, int k, int rec_cap, double *d_spec_ws, void *d_rec);
int apda_analyze_ragged_f32_dev(apda_ctx *ctx, const float *d_samples, const int32_t *d_n_valid, int64_t n_max, int64_t ld,
                                int64_t batch, int64_t N, int flags, int flexible, double fs, const double *d_fs, int k,
                                int rec_cap, float *d_spec_ws, void *d_rec);

/* ---- wire-format ingest (SURVEY.md 8f rank 3) ------------------------------------------------------------------
 * replaces protocol_decoder.py:116-175 (decode_float_v2 / decode_samples: 16-bit samples, high byte first, + the axis
 * baseline first_value, formatted "%8.6f") together with the float() read-back of utils/load_data.py:67-80 (non-finite
 * tokens dropped): payload row b (n_max samples, 2 bytes each, rows ld_bytes apart) -> the samples the reference's FFT
 * would have loaded, compacted, with their count in n_valid[b].  fp64 results are bit-identical to the reference chain.
 * apda_analyze_wire16_* continues into the ragged pipeline (records as apda_analyze_*; 2 bytes per sample over PCIe). */
int apda_decode_wire16_f64_dev(apda_ctx *ctx, const uint8_t *d_payload, int64_t n_max, int64_t ld_bytes, int64_t batch,
                               const double *d_first_value, double *d_samples, int64_t ld_out, int32_t *d_n_valid);
int apda_decode_wire16_f32_dev(apda_ctx *ctx, const uint8_t *d_payload, int64_t n_max, int64_t ld_bytes, int64_t batch,
                               const double *d_first_value, float *d_samples, int64_t ld_out, int32_t *d_n_valid);
int apda_decode_wire16_f64_host(apda_ctx *ctx, const uint8_t *h_payload, int64_t n_max, int64_t ld_bytes, int64_t batch,
                                const double *h_first_value, double *h_samples, int32_t *h_n_valid);
int apda_analyze_wire16_f64_host(apda_ctx *ctx, const uint8_t *h_payload, int64_t n_max, int64_t ld_bytes, int64_t batch,
                                 const double *h_first_value, int64_t N, int flags, int flexible, double fs,
                                 const double *h_fs, int k, int rec_cap, void *h_rec);
int apda_analyze_wire16_f32_host(apda_ctx *ctx, const uint8_t *h_payload, int64_t n_max, int64_t ld_bytes, int64_t batch,
                                 const double *h_first_value, int64_t N, int flags, int flexible, double fs,
                                 const double *h_fs, int k, int rec_cap, void *h_rec);

/* ---- text ingest (SURVEY.md 8f rank 2) ---------------------------------------------------------------------------
 * replaces the sample loop of utils/load_data.py:67-80 for many sensor logs at once.  h_text holds the logs' sample
 * regions (everything after the four header lines) back to back; log b is h_text[h_offsets[b] .. h_offsets[b+1]).
 * Pieces between ';' / newlines are parsed like float() and non-finite / unparsable ones dropped; log b yields
 * h_n_valid[b] <= n_max samples.  h_flags[b] bit 0: the log holds a piece in a float() syntax the kernel does not
 * decide (exponent, '_', > 15 significant digits, non-ASCII): re-parse that log on the host; bit 1: more than n_max
 * samples (truncated).  apda_analyze_text_* continues into the ragged pipeline without moving the samples to the host. */
int apda_parse_samples_f64_host(apda_ctx *ctx, const char *h_text, const int64_t *h_offsets, int64_t batch, int64_t n_max,
                                double *h_samples, int32_t *h_n_valid, int32_t *h_flags);
int apda_analyze_text_f64_host(apda_ctx *ctx, const char *h_text, const int64_t *h_offsets, int64_t batch, int64_t n_max,
                               int64_t N, int flags, int flexible, double fs, const double *h_fs, int k, int rec_cap,
                               void *h_rec, int32_t *h_n_valid, int32_t *h_flags);
int apda_analyze_text_f32_host(apda_ctx *ctx, const char *h_text, const int64_t *h_offsets, int64_t batch, int64_t n_max,
                               int64_t N, int flags, int flexible, double fs, const double *h_fs, int k, int rec_cap,
                               void *h_rec, int32_t *h_n_valid, int32_t *h_flags);

/* ---- whole sensor logs -----------------------------------------------------------------------------------------
 * replaces utils/load_data.py:64-70 load_sensor(path) followed by start_fft + picker (GT_FFT_v5.py:635-642) for many
 * .log files at once.  The host only reads bytes: reader threads (min(16, hardware threads), all joined before the call
 * returns) pread whole files into pinned staging buffers owned by the context, chunk c + 1 while the two pipeline
 * streams process chunk c.  The header layout, the sampling rate and the samples are decoded on the device.
 * Per file b:
 *   h_fs[b]       rate of header line 0, float(rate.replace(" Hz", "")) (bit-equal to Python)
 *   h_n_valid[b]  samples parsed (at most N)
 *   h_head[b]     the bytes of the four header lines (line ends included), NUL-padded to APDA_LOG_HEAD_BYTES
 *   h_rec[b]      the record of apda_analyze_ragged_*_dev at n_max = ld = N on the file's samples with fs = h_fs[b]
 *                 (windows that pad to another length carry APDA_STATUS_OTHER_LENGTH, empty ones APDA_STATUS_EMPTY)
 * h_flags[b] (a record of a file with a non-zero flag is not an analysis result: count 0, every slot idx -1 and zeros):
 *   1   a sample piece in a float() syntax the device does not decide (exponent, '_', > 15 significant digits,
 *       non-ASCII): status 0, re-read the file on the host
 *   2   more than N samples: status APDA_STATUS_OTHER_LENGTH
 *   4   fewer than 5 lines (load_sensor returns None): status APDA_STATUS_EMPTY
 *   8   header not decided on the device (no 4th line end within APDA_LOG_HEAD_BYTES - 1 bytes, a non-ASCII or NUL byte
 *       in it, fewer than 4 ';' fields on line 0, a rate field outside the sample grammar once " Hz" is removed):
 *       status 0, re-read the file on the host
 *   16  the path is not a regular file, or could not be opened or read whole: status 0
 * With flag 4, 8 or 16 h_fs, h_n_valid and h_head are 0.  N: a power of two from 4 up to the ragged batches' limit (on a
 * B200 8192 in fp64, 16384 in fp32); flags: APDA_CENTER_MEDIAN or APDA_CENTER_NONE.  Use _f64 where the reference's
 * samples matter: they are the fp64 parse (fp32 records are not tie-resolved). */
#define APDA_LOG_HEAD_BYTES 1024
int apda_analyze_logs_f64_host(apda_ctx *ctx, const char *const *paths, int64_t n_files, int64_t N, int flags,
                               int flexible, int k, int rec_cap, void *h_rec, double *h_fs, int32_t *h_n_valid,
                               int32_t *h_flags, char *h_head);
int apda_analyze_logs_f32_host(apda_ctx *ctx, const char *const *paths, int64_t n_files, int64_t N, int flags,
                               int flexible, int k, int rec_cap, void *h_rec, double *h_fs, int32_t *h_n_valid,
                               int32_t *h_flags, char *h_head);

/* Fused window -> record kernel (fp32, N in {1024, 2048, 4096, 8192}, k <= 5, rec_cap == 5): same records as
 * apda_analyze_f32_*, but the spectrum never exists in memory (HBM traffic s*N + 128 bytes per window instead of
 * 4*s*N + 128).  A throughput variant for fleets that only need the peak tables (SURVEY.md 8f rank 1); the drop-in
 * start_fft contract stays with the pipeline entry points above. */
int apda_analyze_fused_f32_dev(apda_ctx *ctx, const float *d_samples, int64_t n_samples, int64_t ld, int64_t batch,
                               int64_t N, int flags, int flexible, double fs, const double *d_fs, int k, int rec_cap,
                               void *d_rec);
int apda_analyze_fused_f32_host(apda_ctx *ctx, const float *h_samples, int64_t n_samples, int64_t ld, int64_t batch,
                                int64_t N, int flags, int flexible, double fs, const double *h_fs, int k, int rec_cap,
                                void *h_rec);

/* ---- fp32 tie resolution -----------------------------------------------------------------------------------------
 * Replace the record of every window whose status is exactly APDA_STATUS_FP32_TIE with the record the fp64 path computes
 * from the same samples widened to double; the records are a table written by any fp32 picker route (apda_analyze_f32_*,
 * apda_analyze_ragged_f32_dev, apda_analyze_fused_f32_*, or apda_fft_f32_* followed by apda_peaks_*_f32_*) for these
 * samples and these arguments.
 *   - Only status == 16 is re-run.  A record with 16 together with other bits (e.g. APDA_STATUS_OTHER_LENGTH) keeps every
 *     byte, and so does every other record.  Samples are read-only; no byte outside the replaced records is written.
 *   - The new record is byte-equal to what apda_analyze_f64_dev (apda_analyze_ragged_f64_dev when n_valid is given)
 *     writes for that window's samples widened to double, with the same n_samples, ld, N, k, rec_cap and flexible, and
 *     fs = d_fs ? d_fs[w] : fs.
 *   - APDA_CENTER_MEDIAN and APDA_CENTER_NONE are passed through; APDA_CENTER_MEAN (legal only at n_samples == N) becomes
 *     APDA_CENTER_MEDIAN, the reference's centring.
 *   - _dev enqueues on the context stream and does not synchronise the host (except when it grows its workspace, as the
 *     other _dev calls do); it serves N <= 8192 on a B200 and returns APDA_ERR_UNSUPPORTED above.  d_rec may be a peer
 *     table slice: call it after the picker and before apda_peer_signal.
 *   - _host covers every N the fp64 analysis supports (ragged batches: N <= 8192): it scans h_rec, uploads only the
 *     flagged rows, resolves them and writes their records back.
 * Not covered: the wire-16 and text ingest (there the reference's samples are the fp64 decode, not the fp32 values: use
 * their _f64 entry points), and the apda_peaks_* entry points (no samples). */
int apda_resolve_fp32_ties_dev(apda_ctx *ctx, const float *d_samples, const int32_t *d_n_valid /* NULL: n_samples */,
                               int64_t n_samples, int64_t ld, int64_t batch, int64_t N, int flags, int flexible,
                               double fs, const double *d_fs, int k, int rec_cap, void *d_rec);
int apda_resolve_fp32_ties_host(apda_ctx *ctx, const float *h_samples, const int32_t *h_n_valid,
                                int64_t n_samples, int64_t ld, int64_t batch, int64_t N, int flags, int flexible,
                                double fs, const double *h_fs, int k, int rec_cap, void *h_rec);

/* ---- picker helpers on a magnitude array (module-public functions of the reference) --------------------------
 * utils/get_peak_prominence.py:32-54 calculate_prominence(magnitudes, peak_idx) */
int apda_prominence_f64_host(apda_ctx *ctx, const double *h_mags, int64_t n, int64_t idx, double *out);
/* utils/get_peak_prominence.py:89-112 calculate_half_power_width_prominenceBased: returns the bin count; Hz = bins*(fs/n) */
int apda_half_power_bins_f64_host(apda_ctx *ctx, const double *h_mags, int64_t n, double prominence, int64_t idx,
                                  int64_t *bins);
/* utils/get_peak_resolution.py:30-44 width_half_magnitude(magnitudes, peak_idx) */
int apda_half_height_bins_f64_host(apda_ctx *ctx, const double *h_mags, int64_t n, int64_t idx, int64_t *bins);

/* ---- synthetic fleet windows generated on the device (SURVEY.md Appendix B.2; bench input only) -------------- */
int apda_synth_f64_dev(apda_ctx *ctx, int64_t first_window, int64_t count, int64_t N, uint64_t seed, int on_bin,
                       double *d_out);
int apda_synth_f32_dev(apda_ctx *ctx, int64_t first_window, int64_t count, int64_t N, uint64_t seed, int on_bin,
                       float *d_out);

/* ---- fleet record table in peer memory (multi-GPU sweep; nothing like it exists in the reference, whose
 * work_flow_fft stores one dict per sensor in fft_dict, GT_FFT_v5.py:644-659) -------------------------------------
 * One process per GPU.  The destination rank creates the table (bytes = total windows * record size) and hands the
 * 64-byte handle to the other processes (any channel); they open it and pass `table + first_window * record size` as
 * d_rec to apda_peaks_* / apda_analyze_*: the K3 kernels then store their records straight into the owner's memory
 * over NVLink.  After every rank has synchronised its stream (and a process barrier) the owner reads the full table
 * in window order.  Same-node GPUs with peer access only (NVSwitch); open fails with APDA_ERR_CUDA otherwise. */
int apda_peer_table_create(apda_ctx *ctx, int64_t bytes, void **d_table, unsigned char *handle64);
int apda_peer_table_open(apda_ctx *ctx, const unsigned char *handle64, void **d_table);
int apda_peer_table_close(apda_ctx *ctx, void *d_table);    /* importer side */
int apda_peer_table_destroy(apda_ctx *ctx, void *d_table);  /* owner side */
/* Completion on the device timelines: every rank owns one uint32 step counter in the owner's memory (the caller
 * reserves them, e.g. behind the rows).  apda_peer_signal (producer, after its pickers, same stream) publishes
 * `value` with release semantics at system scope; apda_peer_wait (owner) holds the stream until all `world` counters
 * have reached `value` (acquire); *d_timed_out is 0 afterwards, or 1 if the wait gave up after timeout_s seconds instead
 * of hanging.  The same pair serves the back-pressure direction: the owner signals an "acknowledged step" counter once it
 * has consumed a step's table, and a producer waits on it (world = 1) before it overwrites rows the owner may still be
 * reading (apda-fft_b200/fleet.py: PeerRecordTable double-buffers the table by step parity). */
int apda_peer_signal(apda_ctx *ctx, void *d_flag, uint32_t value);
int apda_peer_wait(apda_ctx *ctx, const void *d_flags, int world, uint32_t value, double timeout_s, int *d_timed_out);

#ifdef __cplusplus
}
#endif
#endif /* APDA_B200_H */
