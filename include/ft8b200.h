/* ft8b200.h -- C ABI of libft8b200.so, the B200-native (sm_100a) implementation of the
 * rtlsdr-ft8d receive-and-decode hot path.
 *
 * Two layers, both `extern "C"`, plain pointers and sizes only:
 *
 *  (1) DROP-IN entry points carrying the reference's own names, signatures and struct
 *      layouts, taking HOST pointers exactly as the reference's callers pass them.  Each one
 *      cites the reference interface it replaces.  A daemon built from the reference's
 *      rtlsdr_ft8d.c links against this library instead of compiling ft8_lib/ft8/decode.c etc.
 *      (see INTEGRATION.md for the exact binding).
 *
 *  (2) BATCHED entry points (`ft8b200_*`) taking DEVICE pointers, used by the benchmarks, the
 *      multi-GPU driver and the parity tests: many independent 15 s slots / receiver streams per
 *      launch.  Layer (1) is implemented on top of layer (2).
 *
 * There is no CPU fallback: every entry point runs CUDA kernels and reports failure when no
 * sm_100 device is usable (ft8b200_last_error()).
 */
#ifndef FT8B200_H
#define FT8B200_H

#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------
 * ABI types, byte-for-byte those of the reference
 * ---------------------------------------------------------------------------------------- */

/* Included from the REFERENCE's own sources (INTEGRATION.md) this header must not define what their headers already
 * have: ft8_lib's constants.h / decode.h are recognised by their include guards; rtlsdr_ft8d.h uses #pragma once, so a
 * translation unit that has included it defines FT8B200_WITH_RTLSDR_FT8D_H before including this header. */
#ifndef _INCLUDE_CONSTANTS_H_
/* replaces: ft8_lib/ft8/constants.h:6-10 */
typedef enum { PROTO_FT4, PROTO_FT8 } ftx_protocol_t;
#endif

#ifndef _INCLUDE_DECODE_H_
/* replaces: ft8_lib/ft8/decode.h:15-25 (40 bytes; mag @24, block_stride @32, protocol @36) */
typedef struct {
    int max_blocks;
    int num_blocks;
    int num_bins;
    int time_osr;
    int freq_osr;
    uint8_t *mag; /* uint8_t[blocks][time_osr][freq_osr][num_bins], HOST memory */
    int block_stride;
    ftx_protocol_t protocol;
} waterfall_t;

/* replaces: ft8_lib/ft8/decode.h:29-36 (8 bytes) */
typedef struct {
    int16_t score;
    int16_t time_offset;
    int16_t freq_offset;
    uint8_t time_sub;
    uint8_t freq_sub;
} candidate_t;

/* replaces: ft8_lib/ft8/decode.h:39-44 (28 bytes; hash @26) */
typedef struct {
    char text[25];
    uint16_t hash;
} message_t;

/* replaces: ft8_lib/ft8/decode.h:47-53 (12 bytes) */
typedef struct {
    int ldpc_errors;
    uint16_t crc_extracted;
    uint16_t crc_calculated;
    int unpack_status;
} decode_status_t;
#endif

#ifndef FT8B200_WITH_RTLSDR_FT8D_H
/* replaces: rtlsdr_ft8d.h:136-141 (28 bytes) */
struct decoder_results {
    char call[13];
    char loc[7];
    int32_t freq;
    int32_t snr;
};
#endif

/* replaces: ft8_lib/decode_ft8.c:82-90 (defined inside the .c in the reference) */
typedef struct {
    float f_min;
    float f_max;
    int sample_rate;
    int time_osr;
    int freq_osr;
    ftx_protocol_t protocol;
} monitor_config_t;

/* replaces: ft8_lib/decode_ft8.c:94-109.  Same leading fields as the reference so code that
 * reads me->wf / block_size keeps working; the two kiss_fft housekeeping pointers of the
 * reference are replaced by one opaque device-side handle of the same total size. */
typedef struct {
    float symbol_period;
    int block_size;
    int subblock_size;
    int nfft;
    float fft_norm;
    float *window;     /* host copy of the Hann window (nfft floats) */
    float *last_frame; /* host copy of the sliding analysis frame (nfft floats) */
    waterfall_t wf;    /* wf.mag is HOST memory, refreshed after every monitor_process() */
    float max_mag;
    void *fft_work; /* opaque: device state of this monitor */
    void *fft_cfg;  /* unused, kept for layout compatibility */
} monitor_t;

/* ------------------------------------------------------------------------------------------
 * (1) drop-in entry points (host pointers)
 * ---------------------------------------------------------------------------------------- */

/* replaces: static rtlsdr_callback(), rtlsdr_ft8d.c:76-202 (type rtlsdr_read_async_cb_t).
 * `samples_count` bytes of interleaved uint8 I/Q, a multiple of 8.  The bytes are consumed
 * before returning.  ctx == NULL selects the process-wide default stream (the reference keeps
 * its state in function statics); otherwise ctx is a ft8b200_stream_t* from
 * ft8b200_stream_create(), which is how many receivers share one process.  Unlike the
 * reference the caller's buffer is NOT modified. */
#ifndef FT8B200_WITH_RTLSDR_FT8D_H /* rtlsdr_ft8d.h:144 declares it itself -- `static` there: drop that word, the definition now lives here */
void rtlsdr_callback(unsigned char *samples, uint32_t samples_count, void *ctx);
#endif

/* replaces: initFFTW()/freeFFTW(), rtlsdr_ft8d.c:314-347: creates / destroys the default
 * context (device tables, workspaces).  Every other entry point creates it on demand. */
#ifndef FT8B200_WITH_RTLSDR_FT8D_H /* declared (without prototype) at rtlsdr_ft8d.h:155-156 */
void initFFTW(void);
void freeFFTW(void);
#endif

/* replaces: ft8_subsystem(), rtlsdr_ft8d.c:1387-1524.  48000 conditioned samples per rail;
 * samples_len is ignored exactly like the reference ignores it (:1393); decodes[] must hold
 * K_MAX_MESSAGES (50) records; *n_results counts ALL unique messages, CQ or not. */
#ifndef FT8B200_WITH_RTLSDR_FT8D_H /* rtlsdr_ft8d.h:164 */
void ft8_subsystem(float *iSamples, float *qSamples, uint32_t samples_len, struct decoder_results *decodes, int32_t *n_results);
#endif

/* replaces: ft8_find_sync(), ft8_lib/ft8/decode.h:63 / decode.c:173-234 */
#ifndef _INCLUDE_DECODE_H_
int ft8_find_sync(const waterfall_t *power, int num_candidates, candidate_t heap[], int min_score);
#endif

/* replaces: ft8_decode(), ft8_lib/ft8/decode.h:72 / decode.c:316-376.  On early failure the
 * later fields of *status are left unwritten, as in the reference. */
#ifndef _INCLUDE_DECODE_H_
bool ft8_decode(const waterfall_t *power, const candidate_t *cand, message_t *message, int max_iterations, decode_status_t *status);
#endif

/* replaces: waterfall_init()/waterfall_free(), ft8_lib/decode_ft8.c:63-79 */
void waterfall_init(waterfall_t *me, int max_blocks, int num_bins, int time_osr, int freq_osr);
void waterfall_free(waterfall_t *me);

/* replaces: monitor_init/process/reset/free, ft8_lib/decode_ft8.c:111-224 */
void monitor_init(monitor_t *me, const monitor_config_t *cfg);
void monitor_process(monitor_t *me, const float *frame);
void monitor_reset(monitor_t *me);
void monitor_free(monitor_t *me);
/* B200-side extension of the monitor: DEFERRED mode.  monitor_process() as the reference defines it is a copy-launch-copy-
 * synchronise round trip per 160 ms block (93 per recording).  With ft8b200_monitor_set_deferred(me, 1) -- or FT8B200_MONITOR_DEFERRED=1
 * in the environment at monitor_init() -- it only appends the block on the host; all pending blocks are transformed in ONE launch when
 * the waterfall is needed: ft8_find_sync() / ft8_decode() on me->wf do it themselves, as do monitor_reset(), monitor_free() and
 * ft8b200_monitor_flush() (returns the number of blocks transformed).  The only observable difference: between a monitor_process()
 * and the next flush, me->wf.mag and me->max_mag do not yet include the appended blocks (me->wf.num_blocks does).  decode_ft8's
 * main() reads max_mag once, after its loop (decode_ft8.c:301): a flush there keeps its output identical. */
int ft8b200_monitor_set_deferred(monitor_t *me, int on);
int ft8b200_monitor_flush(monitor_t *me);

/* ------------------------------------------------------------------------------------------
 * (2) batched entry points (device pointers unless the name says _host)
 * All return 0 on success, a negative FT8B200_E* code otherwise; ft8b200_last_error() has text.
 * `stream` is a cudaStream_t passed as void* (NULL = the context's own stream).
 * ---------------------------------------------------------------------------------------- */
#define FT8B200_OK 0
#define FT8B200_ENODEV (-1)   /* no usable sm_100 device / CUDA runtime error at init */
#define FT8B200_EINVAL (-2)   /* bad argument */
#define FT8B200_ECUDA (-3)    /* a CUDA call or kernel failed */
#define FT8B200_ENOMEM (-4)
#define FT8B200_EBUSY (-5)    /* ft8b200_pipe_submit*: every lane is in flight, collect a batch first */

#define FT8B200_SLOT_SAMPLES 48000  /* 15 s at 3200 sps per rail (rtlsdr_ft8d.h:34-35) */
#define FT8B200_DECIM 751           /* input samples per output sample (rtlsdr_ft8d.c:156-160) */
#define FT8B200_WF_BYTES 94208      /* daemon waterfall bytes per slot (rtlsdr_ft8d.h:54) */
#define FT8B200_RAW_SLOT_BYTES 72000000
/* Batch sizes: the entry points that take slots of 3200 sps samples, waterfalls, candidates or audio (process_slots /
 * _conditioned, condition, waterfall, find_sync, decode, osd, spots, monitor_waterfall, synth_*, the pipe's submit_slots,
 * the stream and file calls) accept any n_slots >= 1 the device memory holds; beyond 65 535 slots their per-slot kernels
 * run as several launches.  The raw-IQ entry points (decimate, decimate_streams, process_raw, process_raw_streams and the
 * pipe and cluster submits built on them) refuse more than FT8B200_MAX_RAW_ROWS streams or output rows per call with
 * FT8B200_EINVAL: that many raw slots are 4.7 TB. */
#define FT8B200_MAX_RAW_ROWS 65535

typedef struct ft8b200_ctx ft8b200_ctx_t;
typedef struct ft8b200_stream ft8b200_stream_t;
typedef struct ft8b200_pipe ft8b200_pipe_t;

typedef struct {
    int device;          /* CUDA device ordinal */
    int max_slots;       /* largest batch the workspaces are sized for */
    int max_candidates;  /* K_MAX_CANDIDATES: 120 (daemon), 500 (crowded band) */
    int max_messages;    /* K_MAX_MESSAGES: 50 (daemon), 200 (crowded band) */
    int min_score;       /* K_MIN_SCORE: 10 */
    int ldpc_iterations; /* K_LDPC_ITERS: 20 */
} ft8b200_config_t;

const char *ft8b200_last_error(void);
const char *ft8b200_version(void);
void ft8b200_default_config(ft8b200_config_t *cfg);
ft8b200_ctx_t *ft8b200_create(const ft8b200_config_t *cfg);
void ft8b200_destroy(ft8b200_ctx_t *ctx);
void *ft8b200_cuda_stream(ft8b200_ctx_t *ctx);
int ft8b200_sync(ft8b200_ctx_t *ctx);
/* number of kernels this library has launched since the context was created */
uint64_t ft8b200_kernel_launches(ft8b200_ctx_t *ctx);

/* a1-a3: n_streams independent receiver streams, each `bytes_per_stream` bytes of uint8 IQ
 * (multiple of 16, 16-byte aligned, streams `stream_stride_bytes` apart), decimated from zero
 * filter state.  Writes, per stream, floor(bytes/2/751) outputs (<= 48000) into
 * d_i/d_q[stream*48000 ...], zero-fills the rest of the 48000, stores the output count in
 * d_count[stream] and max(|I|,|Q|) in d_peak[stream] (the input of decoder()'s normalisation,
 * rtlsdr_ft8d.c:248-258).  d_y2 (optional, int32[n_streams][48000][2]) receives the integer
 * CIC output before the FIR. */
int ft8b200_decimate(ft8b200_ctx_t *ctx, const uint8_t *d_iq, size_t bytes_per_stream, size_t stream_stride_bytes, int n_streams,
                     float *d_i, float *d_q, uint32_t *d_count, float *d_peak, int32_t *d_y2, void *stream);

/* Continuous receiver streams cut into consecutive slots (BASELINE config #5): stream s holds slots_per_stream x
 * bytes_per_slot bytes of one receiver; the decimator runs THROUGH the slot boundaries (filter history is the real
 * preceding samples) and output row s*slots_per_stream + g receives the samples whose decimation instant falls into
 * slot g -- 47 936 or 47 937 per 72 000 000-byte slot, exactly what rx_state's buffers hold when main() flips them every
 * 15 s between callbacks (rtlsdr_ft8d.c:1339-1354).  Output arrays have n_streams*slots_per_stream rows. */
int ft8b200_decimate_streams(ft8b200_ctx_t *ctx, const uint8_t *d_iq, size_t bytes_per_stream, size_t stream_stride_bytes, int n_streams,
                             int slots_per_stream, size_t bytes_per_slot, float *d_i, float *d_q, uint32_t *d_count, float *d_peak,
                             int32_t *d_y2, void *stream);

/* a4: in-place decoder() conditioning of n_slots x 48000 samples using d_peak (rtlsdr_ft8d.c:242-263) */
int ft8b200_condition(ft8b200_ctx_t *ctx, float *d_i, float *d_q, const float *d_peak, int n_slots, void *stream);

/* a5: daemon waterfall.  d_peak may be NULL (samples already conditioned); otherwise the
 * conditioning scale (float)(0.5/max(peak,1e-24)) is applied on load. d_mag: n_slots x 94208. */
int ft8b200_waterfall(ft8b200_ctx_t *ctx, const float *d_i, const float *d_q, const float *d_peak, int n_slots, uint8_t *d_mag, void *stream);

/* a7-a8: per slot, candidate list sorted exactly like ft8_find_sync(). d_cand: n_slots x max_candidates,
 * d_ncand: n_slots.  Waterfall geometry as in waterfall_t (all slots share it). */
int ft8b200_find_sync(ft8b200_ctx_t *ctx, const uint8_t *d_mag, size_t slot_stride_bytes, int n_slots, int num_blocks, int num_bins,
                      int time_osr, int freq_osr, candidate_t *d_cand, int *d_ncand, void *stream);

/* a9-a14: decode every candidate of every slot.  Outputs are n_slots x max_candidates arrays:
 * d_ok (uint8: 1 = message decoded), d_stage (uint8: 1 = stopped at LDPC, 2 = at CRC, 3 = at unpack, 4 = done:
 * which decode_status_t fields the reference would have written), d_status, d_msg; optional d_plain
 * (uint8[...][174]) and d_llr (float[...][174], the normalised LLRs fed to the BP decoder). */
int ft8b200_decode(ft8b200_ctx_t *ctx, const uint8_t *d_mag, size_t slot_stride_bytes, int n_slots, int num_blocks, int num_bins,
                   int time_osr, int freq_osr, const candidate_t *d_cand, const int *d_ncand, uint8_t *d_ok, uint8_t *d_stage,
                   decode_status_t *d_status, message_t *d_msg, uint8_t *d_plain, float *d_llr, void *stream);

/* Ordered-statistics decoding (OSD, DESIGN.md section 2.4.1) of the candidates belief propagation leaves undecoded (stage 1: no zero
 * syndrome, stage 2: CRC mismatch).  order: 0 = off (default), 1 = the most reliable basis' hard decisions and every single flip
 * (92 codewords), 2 = also every pair among its 32 least reliable positions (588); anything else is FT8B200_EINVAL.  The least-metric
 * codeword is accepted when its CRC holds, it differs from the hard decision in at most max_hard_errors bits and it unpacks.
 * max_hard_errors < 0 selects FT8B200_OSD_DEFAULT_MAX_HARD: the largest cap that decoded at most 2 messages on 4096 noise-only
 * daemon slots (K = 120) at order 2 (tools/perf_osd.py; profiles/perf_osd.json).
 * The process_* calls, ft8b200_decode and the whole-recording calls honour it; off, every output and launch is as without it. */
#define FT8B200_OSD_DEFAULT_MAX_HARD 174
int ft8b200_set_osd(ft8b200_ctx_t *ctx, int order, int max_hard_errors);
/* Stage-wise OSD with the context's order, cap and protocol: upgrades the n_slots x max_candidates outputs of ft8b200_decode in
 * place (d_llr = its normalised LLRs).  An accepted codeword makes the entry ok = 1, stage = 4, status.ldpc_errors = 0 with the
 * codeword's CRC fields, msg as a BP decode would, d_plain (optional) = the codeword; a rejected one changes none of them.
 * d_osd: 0 = not attempted (stage 3/4, beyond d_ncand, a non-finite LLR or order 0), 1 = attempted and rejected, 2 = decoded by OSD.
 * d_osd_hard: the winner's hard-decision distance, -1 when not attempted.  d_osd_cw (optional, uint8[...][174]): the winner whether
 * or not it was accepted (zeros when not attempted). */
int ft8b200_osd(ft8b200_ctx_t *ctx, const float *d_llr, int n_slots, const int *d_ncand, uint8_t *d_ok, uint8_t *d_stage,
                decode_status_t *d_status, message_t *d_msg, uint8_t *d_plain, uint8_t *d_osd, int32_t *d_osd_hard, uint8_t *d_osd_cw,
                void *stream);
/* d_osd / d_osd_hard (as above) of the last process_* or decode batch run with OSD on (n_slots x max_candidates); NULL before that */
int ft8b200_osd_workspace(ft8b200_ctx_t *ctx, uint8_t **d_osd, int32_t **d_osd_hard);
/* Multi-pass decoding (DESIGN.md section 2.4.2) on the daemon path -- every process_raw*, process_slots / process_conditioned call,
 * and through them the pipe, the cluster, the drop-in ft8_subsystem, the stream and .iq file paths.  passes = 1 (default) decodes
 * a slot once, exactly as without this call.  With 2 or 3, after each pass the messages the spot table accepted as new in that
 * pass (in acceptance order; duplicates and messages dropped by a full table are not) are subtracted from the pass's input as
 * unit-amplitude GFSK waveforms (ft8b200_subtract), and the residual is searched again: waterfall with the slot's original peak
 * scale, find_sync (same max_candidates and min_score), decode (+ OSD when on), and the spot table in append mode -- it keeps the
 * slot's earlier records, de-duplicates against every earlier pass by hash and text, and appends new records behind them (freq and
 * snr from the new candidate).  A slot with nothing new in a pass is not searched again.  Pass 1's outputs (records, workspace
 * rows) are those of passes = 1; the later passes only append.  The later passes use their own context workspaces, allocated only
 * with passes > 1.  ft8b200_stage_times reports subtraction + later passes as a seventh stage.
 * Out of scope: the 12 kHz audio entry points (ft8b200_decode_audio, decode_ft8 and the monitor), whose geometry differs.
 * Any passes other than 1, 2 or 3 is FT8B200_EINVAL. */
int ft8b200_set_passes(ft8b200_ctx_t *ctx, int passes);
/* Stage-wise subtraction of decoded FT8 messages from daemon slots (3200 sps complex, FT8B200_SLOT_SAMPLES floats per slot row,
 * dense).  Slot s has d_nmsg[s] (clamped to 0 ... max_messages) messages: d_cand[s][j] (candidate_t, max_messages per slot)
 * and d_cw[s][j] (174 bytes, one codeword bit per byte, ft8b200_decode's d_plain order).  Each message's start sample and tone-0
 * frequency follow from its candidate (s0 = 512 time_offset + 256 time_sub + 256, f0 = 3.125 (2 freq_offset + freq_sub) Hz);
 * the GFSK reference is refined on the INPUT slot over dt = -128 ... +128 samples (step 16) x df = -8 ... +8 steps of 6.25/32 Hz,
 * then dt +- 8 samples at the chosen df, and d_grid[s][j] = {dt in samples, df in steps} receives the result.  The messages are
 * then subtracted in list order, each with the amplitude of the residual against it smoothed by a 1025-tap Hann window:
 * d_ri / d_rq (same layout as d_i / d_q; may be d_i / d_q themselves, not otherwise overlapping) receive the residual.
 * The subtraction is linear in the samples, so no peak scale is needed: conditioned or unconditioned slots give the residual of
 * what was passed in.  tests/subtract_ref.py is the float64 definition. */
int ft8b200_subtract(ft8b200_ctx_t *ctx, const float *d_i, const float *d_q, int n_slots, const candidate_t *d_cand, const uint8_t *d_cw,
                     const int32_t *d_nmsg, float *d_ri, float *d_rq, int32_t *d_grid, void *stream);

/* a15: the daemon's duplicate table + CQ filter, one slot per thread.  d_results: n_slots x max_messages
 * (zeroed here first), d_nresults: n_slots; optional first-seen unique message log: d_umsg (n_slots x
 * max_messages message_t), d_ufreq (float), d_uscore (int32), d_ucand (int32, optional: index of the candidate
 * that produced the entry). */
int ft8b200_spots(ft8b200_ctx_t *ctx, int n_slots, int freq_osr, const candidate_t *d_cand, const int *d_ncand, const uint8_t *d_ok,
                  const message_t *d_msg, struct decoder_results *d_results, int32_t *d_nresults, message_t *d_umsg, float *d_ufreq,
                  int32_t *d_uscore, int32_t *d_ucand, void *stream);

/* Whole path on device buffers owned by the context: raw uint8 IQ (d_iq != NULL) or conditioned
 * 3200 sps samples (d_i/d_q) -> decoder_results.  Results stay on the device (ft8b200_results_device)
 * until fetched. */
int ft8b200_process_raw(ft8b200_ctx_t *ctx, const uint8_t *d_iq, size_t bytes_per_stream, size_t stream_stride_bytes, int n_slots, void *stream);
/* whole path over continuous streams (see ft8b200_decimate_streams): n_streams*slots_per_stream result rows */
int ft8b200_process_raw_streams(ft8b200_ctx_t *ctx, const uint8_t *d_iq, size_t bytes_per_stream, size_t stream_stride_bytes, int n_streams,
                                int slots_per_stream, size_t bytes_per_slot, void *stream);
/* n_slots x 48000 conditioned samples per rail; d_i and d_q must be 16-byte aligned (as for ft8b200_waterfall), otherwise
 * FT8B200_EINVAL before anything is queued.  The same holds for ft8b200_process_conditioned and ft8b200_pipe_submit_slots. */
int ft8b200_process_slots(ft8b200_ctx_t *ctx, const float *d_i, const float *d_q, int n_slots, void *stream);
/* same, but the samples are NOT yet conditioned: d_peak[slot] = max(|I|,|Q|) and decoder()'s 0.5/peak scale is applied on load */
int ft8b200_process_conditioned(ft8b200_ctx_t *ctx, const float *d_i, const float *d_q, const float *d_peak, int n_slots, void *stream);
/* Per-stage device timing of the process_* calls: when enabled, CUDA events are recorded on the launching
 * stream between stages; ms[0..5] = block sums, comb+FIR, waterfall, sync, decode, spots (-1 = stage not run). */
int ft8b200_set_profiling(ft8b200_ctx_t *ctx, int on);
/* groups >= 2: ft8b200_process_raw splits the batch into that many slot groups and runs the compute-bound back end of
 * one group on a high-priority side stream while the HBM-bound decimator of the next group runs on the caller's stream
 * (default 0 = off; results are identical either way; only worthwhile when a group still holds >= ~64 slots). */
int ft8b200_set_overlap(ft8b200_ctx_t *ctx, int groups);
int ft8b200_stage_times(ft8b200_ctx_t *ctx, float *ms, int n);
/* begin/end of each stage of the last process_* call in ms since `ref_event` (a timing cudaEvent_t recorded earlier) */
int ft8b200_stage_marks(ft8b200_ctx_t *ctx, void *ref_event, float *begin_ms, float *end_ms, int n);
/* on: ft8b200_process_raw runs its back end (waterfall ... spots) on the context's high-priority side stream even for a
 * single slot group, and ft8b200_front_event() returns the cudaEvent_t (as void*) recorded on the launching stream right
 * after the decimator of the last call -- what ft8b200_pipe_t chains its lanes with. */
int ft8b200_set_side_backend(ft8b200_ctx_t *ctx, int on);
/* Protocol that ft8b200_find_sync / ft8b200_decode score and demap: PROTO_FT8 (default) or PROTO_FT4 (ft4_sync_score,
 * ft4_extract_likelihood and the descrambling of decode.c:110-171,236-263,355-363).  The drop-in ft8_find_sync / ft8_decode
 * take it from waterfall_t.protocol like the reference; the daemon path (ft8b200_process_*) is FT8 by definition. */
int ft8b200_set_protocol(ft8b200_ctx_t *ctx, int protocol);
/* Which cic_block_sums kernel the decimator uses: 0 = streaming (one warp per super-block, whole-GPU grid),
 * >= 1 = persistent bulk-copy kernel (one CTA per SM: a producer thread feeding a shared-memory ring with cp.async.bulk,
 * consumer warps doing the arithmetic) which leaves most of each SM free for the back-end kernels of another batch.
 * Results are identical. */
int ft8b200_set_decimator_variant(ft8b200_ctx_t *ctx, int variant);
/* Which belief-propagation kernel ft8b200_decode and the process_* calls use (process-wide): 0 = node-centred (default: a lane
 * owns a variable / a check row, Pade evaluations with the in-range division sequence inlined), 1 = edge-centred (a lane
 * per edge).  Results are identical; 1 exists for comparison.  Also settable as FT8B200_DECODE_VARIANT=1 in the environment. */
int ft8b200_set_decode_variant(int variant);
/* Device self-check of variant 0's inlined fast_tanh / fast_atanh (ldpc.c:220-251) against the same expressions with the full
 * IEEE division, over ALL 2^32 float bit patterns.  counts5[0] = tanh mismatches, [1] = atanh mismatches for |x| <= 2 or NaN
 * (the argument is a product of tanh values), [2] = atanh mismatches elsewhere, [3], [4] = how many patterns took the full
 * division (tanh, atanh).  [0..2] must be 0. */
int ft8b200_selfcheck_pade(ft8b200_ctx_t *ctx, uint64_t *counts5);
/* Device self-check of the waterfall kernel's dB quantiser (replaces: 10*log10f + (int)(2*db+240) + clamp, rtlsdr_ft8d.c:1416,1425-1427):
 * every non-negative float bit pattern and every NaN through the kernel's straight-line form (MUFU.LG2 estimate, one load of the two
 * host-computed step thresholds around it, two compares) against a search over all 256 thresholds.  counts3[0] = mismatches (must be 0),
 * [1] = inputs whose estimate needed the +-1 correction, [2] = inputs whose estimate was off by more than one (must be 0). */
int ft8b200_selfcheck_quantiser(ft8b200_ctx_t *ctx, uint64_t *counts3);
/* Device self-check hook for the message unpacker (a13): n 77-bit payloads (10 bytes each, MSB first, host) through the
 * kernel-side unpack77 (replaces: unpack77, ft8_lib/ft8/unpack.c:396-427 and everything under it), one thread each.
 * h_text32: n x 32 chars (NUL-padded; empty when rejected), h_status: unpack77's return value (0, -1, -2).  Exists so that
 * every message type and reject path can be fuzzed against the CPU checker without a waterfall in front of it. */
int ft8b200_unpack77_batch(ft8b200_ctx_t *ctx, const uint8_t *h_payloads, int n, char *h_text32, int32_t *h_status);
/* Run the context's work on caller-owned streams (cudaStream_t as void*): `front_stream` replaces the context's launching
 * stream, `back_stream` its back-end side stream, whose kernels size their persistent grids for `back_sm_count` SMs.
 * NULL restores the context's own stream.  Used by ft8b200_pipe_set_partition with green-context streams. */
int ft8b200_set_partition_streams(ft8b200_ctx_t *ctx, void *front_stream, void *back_stream, int back_sm_count);
/* With partition streams set: 0 (default) = the comb+FIR pass runs on the back-end SM set with the rest of the back end,
 * 1 = it stays on the front set directly behind cic_block_sums (it is a whole-GPU grid that takes 5x longer on a small back
 * partition, but on the front set it queues ahead of the next batch's block sums).  Which is better depends on how the two
 * sides balance: ft8b200_pipe_autotune measures it. */
int ft8b200_set_comb_front(ft8b200_ctx_t *ctx, int on);
void *ft8b200_front_event(ft8b200_ctx_t *ctx);
/* One-shot: the cic_block_sums kernel of the NEXT ft8b200_process_raw* call on this context starts only after `cuda_event` (a
 * cudaEvent_t) has completed; the call's buffer initialisation ahead of it does not wait.  What ft8b200_pipe_t chains its lanes with. */
int ft8b200_set_front_wait(ft8b200_ctx_t *ctx, void *cuda_event);
/* The same for the back end: ft8b200_back_event() = the cudaEvent_t recorded on the back-end stream behind the spot table of the last
 * ft8b200_process_raw* call (NULL unless ft8b200_set_side_backend is on); ft8b200_set_back_wait: one-shot, the back end (comb+FIR when
 * it runs on the back set, waterfall ... spots) of the NEXT call starts only after `cuda_event`.  ft8b200_pipe_t chains the lanes'
 * back ends with it on an SM partition: two batches' back ends sharing a back partition that one of them fills slow each other
 * down, and a partition that is only just large enough then falls behind for good (measured: 24 back-end SMs, 1.417 ms per batch
 * while the backlog was under one batch, 1.547 once it was not). */
void *ft8b200_back_event(ft8b200_ctx_t *ctx);
int ft8b200_set_back_wait(ft8b200_ctx_t *ctx, void *cuda_event);
/* device pointers to the last batch's outputs: results (n_slots x max_messages), counts (n_slots) */
int ft8b200_results_device(ft8b200_ctx_t *ctx, struct decoder_results **d_results, int32_t **d_nresults);
int ft8b200_fetch_results(ft8b200_ctx_t *ctx, int n_slots, struct decoder_results *h_results, int32_t *h_nresults, void *stream);
/* same without the final synchronisation: h_results/h_nresults must be pinned and are valid once `stream` reaches this point */
int ft8b200_fetch_results_async(ft8b200_ctx_t *ctx, int n_slots, struct decoder_results *h_results, int32_t *h_nresults, void *stream);
/* intermediate device buffers of the last batch (for tests / profiling): any pointer may be NULL */
int ft8b200_workspace(ft8b200_ctx_t *ctx, float **d_i, float **d_q, float **d_peak, uint8_t **d_mag, candidate_t **d_cand, int **d_ncand,
                      uint8_t **d_ok, decode_status_t **d_status, message_t **d_msg);

/* Same, host buffers in / host results out (H2D + kernels + D2H): the end-to-end call. */
int ft8b200_process_raw_host(ft8b200_ctx_t *ctx, const uint8_t *h_iq, size_t bytes_per_stream, int n_slots,
                             struct decoder_results *h_results, int32_t *h_nresults);
int ft8b200_process_slots_host(ft8b200_ctx_t *ctx, const float *h_i, const float *h_q, int n_slots,
                               struct decoder_results *h_results, int32_t *h_nresults);

/* Pipelined executor: `depth` lanes (contexts) on one GPU keep that many batches in flight, in order.  The HBM-bound
 * decimator of batch n+1 runs while the compute-bound back end of batch n finishes on a high-priority stream; host input
 * is copied H2D on the lane's own stream (overlapping the previous batch's kernels); spot records come back through
 * pinned buffers, so the host blocks only in ft8b200_pipe_collect().  This is the daemon's "receive slot n+1 while slot
 * n decodes" double buffering (rtlsdr_ft8d.c:221-285,1336-1354) across batches.  Results are identical to
 * ft8b200_process_raw + ft8b200_fetch_results.
 *   submit*  : 0, FT8B200_EBUSY when `depth` batches are already in flight, or another error (ft8b200_pipe_error)
 *   collect  : waits for the OLDEST batch in flight, copies its records out, returns its slot count (>0) or an error (<0)
 * Device input passed to ft8b200_pipe_submit must be complete (synchronised) and stay untouched until collected;
 * host input of ft8b200_pipe_submit_host should be pinned (cudaHostAlloc/cudaHostRegister) for the copy to be async. */
ft8b200_pipe_t *ft8b200_pipe_create(const ft8b200_config_t *cfg, int depth);
/* FT8B200_PIPE_OVERLAP (default): as described above.  FT8B200_PIPE_SERIAL: the kernels of batch n+1 start when batch n
 * has completed, so only H2D copies, D2H of the records and host work overlap the kernels (each kernel then runs alone
 * on the GPU, which is what the per-kernel roofline is quoted for).  decimator_variant >= 0 also selects the
 * cic_block_sums kernel of every lane (ft8b200_set_decimator_variant), -1 leaves it. */
#define FT8B200_PIPE_OVERLAP 0
#define FT8B200_PIPE_SERIAL 1
int ft8b200_pipe_set_mode(ft8b200_pipe_t *p, int mode, int decimator_variant);
/* Spatial partition (CUDA green contexts, resolved from the driver at run time): the HBM-bound front end (cic_block_sums,
 * comb+FIR) of batch n+1 runs on one disjoint set of SMs while the issue/latency-bound back end (waterfall, sync, LDPC,
 * spots) of batch n runs on the other `back_sms` SMs (rounded up by the driver to its granularity, 8 SMs on sm_100; the
 * sizes actually provisioned come back through front_sms/back_sms, either may be NULL).  Implies FT8B200_PIPE_OVERLAP.
 * back_sms == 0 removes the partition.  Results are identical in every mode.  Needs depth >= 2 and no batch in flight.
 * SM layout: back_sms + 1000 * layout.  layout 0 = the driver's split by count (the first back_sms SMs of its enumeration, the rest
 * in front).  layout 1..6 = the SMs are split into the driver's groups of 8 and the back partition is composed of groups spread
 * over the enumeration (1: evenly from the first group, 2: evenly, centred, 3: the last groups, 4: every second group, 5: spread
 * neighbouring pairs, 6: the first groups), the front end gets every other group plus the remainder.  An HBM-bound front end
 * that loses whole GPCs loses their ports into the L2 fabric as well as their SMs; which layout is best depends on the GPU's
 * floor-sweeping, so ft8b200_pipe_autotune accepts encoded candidates and measures them. */
int ft8b200_pipe_set_partition(ft8b200_pipe_t *p, int back_sms, int *front_sms, int *back_sms_out);
/* Diagnostic: the hardware SM ids (%smid) the front (which = 0) or back (which = 1) partition runs on, as a 256-bit mask
 * (mask8[id / 32] bit id % 32); without a partition, the SMs of the whole GPU. */
int ft8b200_pipe_partition_smids(ft8b200_pipe_t *p, int which, uint32_t *mask8);
/* Chooses the partition by measurement: for every back_sms in `candidates` (0 = no partition, serial kernels) and both placements
 * of the comb+FIR pass, batches of the caller's device-resident input (as for ft8b200_pipe_submit) are pushed through the executor
 * and the STEADY-STATE interval between completed batches is timed: `batches` / 2 batches run first, untimed (a back partition that
 * is too small only throttles the front end once the lanes' slack is used up), then `batches` are timed from completion to
 * completion.  Of the settings within 0.3 % of the fastest the one with the largest back partition is left in place and reported
 * (best_back_sms, best_comb_front, ms per batch of each point in ms_out[2 * n_candidates], comb_front = 0 first; any of the three
 * may be NULL).  The split that balances the HBM-bound front end against the issue-bound back end depends on the batch's candidate
 * load and on the box; nothing in the results does. */
/* With an SM partition: on = the back end of batch n+1 starts only when the back end of batch n has finished (the front ends are
 * always chained).  Off (default) the back ends of consecutive batches may share the back partition when a backlog has built up,
 * which is the better executor when the back end falls behind; on is what ft8b200_pipe_autotune compares partitions with (it
 * shows within a dozen batches whether ONE batch's back end fits under the next batch's block sums) and restores afterwards.
 * Results are identical either way.  Not while batches are in flight. */
int ft8b200_pipe_set_back_chain(ft8b200_pipe_t *p, int on);
/* ft8b200_set_osd on every lane (a cluster's pipes through ft8b200_cluster_pipe).  FT8B200_EBUSY while batches are in flight;
 * ft8b200_osd_workspace of a lane is not exposed: the pipe returns spot records only. */
int ft8b200_pipe_set_osd(ft8b200_pipe_t *p, int order, int max_hard_errors);
/* ft8b200_set_passes on every lane (a cluster's pipes through ft8b200_cluster_pipe).  FT8B200_EBUSY while batches are in flight. */
int ft8b200_pipe_set_passes(ft8b200_pipe_t *p, int passes);
int ft8b200_pipe_autotune(ft8b200_pipe_t *p, const uint8_t *d_iq, size_t bytes_per_stream, size_t stream_stride_bytes, int n_slots,
                          const int *candidates, int n_candidates, int batches, int *best_back_sms, int *best_comb_front, float *ms_out);
void ft8b200_pipe_destroy(ft8b200_pipe_t *p);
const char *ft8b200_pipe_error(ft8b200_pipe_t *p);
int ft8b200_pipe_depth(ft8b200_pipe_t *p);
int ft8b200_pipe_in_flight(ft8b200_pipe_t *p);
int ft8b200_pipe_submit(ft8b200_pipe_t *p, const uint8_t *d_iq, size_t bytes_per_stream, size_t stream_stride_bytes, int n_slots);
int ft8b200_pipe_submit_host(ft8b200_pipe_t *p, const uint8_t *h_iq, size_t bytes_per_stream, int n_slots);
/* continuous receiver streams cut into consecutive slots (BASELINE config #5, see ft8b200_process_raw_streams): the batch has
 * n_streams * slots_per_stream result rows */
int ft8b200_pipe_submit_streams(ft8b200_pipe_t *p, const uint8_t *d_iq, size_t bytes_per_stream, size_t stream_stride_bytes, int n_streams,
                                int slots_per_stream, size_t bytes_per_slot);
/* The same executor fed at the OTHER boundary of the path, the input of ft8_subsystem() (rtlsdr_ft8d.h:164): n_slots x 48000 float
 * samples per rail at 3200 sps.  _host: conditioned samples in (pinned) host memory, copied H2D on the lane's stream; device form:
 * d_peak == NULL for conditioned samples, else decoder()'s 0.5/peak scale is applied on load.  384 KB per slot instead of 72 MB:
 * this is the call for hosts that decimate elsewhere (or replay .iq/.c2 recordings).  Use a pipe without an SM partition.
 * d_i and d_q must be 16-byte aligned; a refused batch is not in flight. */
int ft8b200_pipe_submit_slots(ft8b200_pipe_t *p, const float *d_i, const float *d_q, const float *d_peak, int n_slots);
int ft8b200_pipe_submit_slots_host(ft8b200_pipe_t *p, const float *h_i, const float *h_q, int n_slots);
int ft8b200_pipe_collect(ft8b200_pipe_t *p, struct decoder_results *h_results, int32_t *h_nresults, int capacity_slots);
/* same wait, but hands out the DEVICE buffers of the oldest batch (n_slots x max_messages records, n_slots counts) instead of
 * copying to the host -- for a collective on the records (NCCL all_gather).  They stay valid until that lane is submitted
 * to again, i.e. finish (synchronise) the collective before the next ft8b200_pipe_submit*. */
int ft8b200_pipe_collect_device(ft8b200_pipe_t *p, struct decoder_results **d_results, int32_t **d_nresults);
/* One-shot stream dependency: the kernels of the NEXT submitted batch start only after `cuda_event` (a cudaEvent_t recorded by
 * the caller, e.g. behind an NCCL all_gather that reads the device buffers handed out by ft8b200_pipe_collect_device) has
 * completed -- ordering on the device, no host synchronisation. */
int ft8b200_pipe_depend_on(ft8b200_pipe_t *p, void *cuda_event);
/* per-stage device times summed over the batches collected since profiling was switched on (ms[0..5] as ft8b200_stage_times) */
int ft8b200_pipe_set_profiling(ft8b200_pipe_t *p, int on);
int ft8b200_pipe_stage_times(ft8b200_pipe_t *p, double *ms, int n, uint64_t *batches);
/* device timeline of those batches: 12 floats each (begin, end of the six stages, ms since profiling was switched on);
 * returns how many batches were written.  Shows what actually overlapped. */
int ft8b200_pipe_timeline(ft8b200_pipe_t *p, float *out, int max_batches);
uint64_t ft8b200_pipe_kernel_launches(ft8b200_pipe_t *p);

/* ---- every GPU of one box from ONE process (csrc/cluster.cu) --------------------------------------------------------------------
 * The path shards by independent slot or receiver stream (no data-path collective); a cluster owns one ft8b200_pipe_t per device
 * and the only exchange is the one BASELINE.json names: the decoded-spot records of a step are gathered with one grouped
 * ncclAllGather over NVLink on a side stream per device, device 0's copy is read to the host and handed out in (device, slot)
 * order.  NCCL is loaded at run time (libnccl.so.2); with a single device none is needed, with several and no NCCL the cluster
 * cannot be created.  A step = one batch per device; up to `depth` steps may be in flight before the oldest is collected. */
typedef struct ft8b200_cluster ft8b200_cluster_t;
/* n_devices <= 0: all visible devices (ordinals 0..n-1).  NULL on failure (reason on stderr and in ft8b200_last_error()). */
ft8b200_cluster_t *ft8b200_cluster_create(const ft8b200_config_t *cfg, int n_devices, int depth);
void ft8b200_cluster_destroy(ft8b200_cluster_t *c);
const char *ft8b200_cluster_error(ft8b200_cluster_t *c);
int ft8b200_cluster_devices(ft8b200_cluster_t *c);
int ft8b200_cluster_in_flight(ft8b200_cluster_t *c);
/* device `device_index`'s executor, and a utility context on that device (ft8b200_synth_*, ft8b200_device_malloc) */
ft8b200_pipe_t *ft8b200_cluster_pipe(ft8b200_cluster_t *c, int device_index);
ft8b200_ctx_t *ft8b200_cluster_ctx(ft8b200_cluster_t *c, int device_index);
/* contiguous block of n_items (slots or streams) that device `device_index` owns: blocks of ceil(n / devices) */
int ft8b200_cluster_shard(ft8b200_cluster_t *c, int n_items, int device_index, int *first, int *count);
/* One step from device-resident input: d_iq[d] on device d holds n_per_device[d] slots (0 = that device sits the step out). */
int ft8b200_cluster_submit(ft8b200_cluster_t *c, const uint8_t *const *d_iq, size_t bytes_per_stream, size_t stream_stride_bytes, const int *n_slots_per_device);
/* ... or n_streams_per_device[d] continuous receiver streams cut into slots_per_stream consecutive slots (BASELINE config #5) */
int ft8b200_cluster_submit_streams(ft8b200_cluster_t *c, const uint8_t *const *d_iq, size_t bytes_per_stream, size_t stream_stride_bytes,
                                   const int *n_streams_per_device, int slots_per_stream, size_t bytes_per_slot);
/* One step from (pinned) host memory: n_slots independent slots, sharded in contiguous blocks (ft8b200_cluster_shard) */
int ft8b200_cluster_submit_host(ft8b200_cluster_t *c, const uint8_t *h_iq, size_t bytes_per_stream, int n_slots);
/* Oldest step: records of all devices in (device, slot) order; returns the number of slots (>= 0) or an error (< 0). */
int ft8b200_cluster_collect(ft8b200_cluster_t *c, struct decoder_results *h_results, int32_t *h_nresults, int capacity_slots);
uint64_t ft8b200_cluster_gathers(ft8b200_cluster_t *c);          /* NCCL all-gathers issued so far */
int ft8b200_cluster_nccl_version(ft8b200_cluster_t *c);          /* e.g. 22809; 0 for a single-device cluster */
uint64_t ft8b200_cluster_kernel_launches(ft8b200_cluster_t *c);
/* device memory on the context's device for callers without the CUDA headers (the C host program); NULL on failure */
void *ft8b200_device_malloc(ft8b200_ctx_t *ctx, size_t bytes);
void ft8b200_device_free(ft8b200_ctx_t *ctx, void *p);

/* Receiver streams for rtlsdr_callback(): persistent decimator state, double-buffered 15 s slots.
 * flip / count / fetch / decode accept s == NULL for the process-wide default stream, the one that
 * rtlsdr_callback(..., ctx = NULL) feeds (the reference registers its callback with a NULL ctx, rtlsdr_ft8d.c:214);
 * freeFFTW() destroys it together with the default context. */
ft8b200_stream_t *ft8b200_stream_create(ft8b200_ctx_t *ctx);
void ft8b200_stream_destroy(ft8b200_stream_t *s);
/* what main() does every 15 s (rtlsdr_ft8d.c:1339-1354): close the current slot buffer, start the next */
int ft8b200_stream_flip(ft8b200_stream_t *s);
/* samples collected so far in the slot being filled (rx_state.iqIndex[bufferIndex]) */
uint32_t ft8b200_stream_count(ft8b200_stream_t *s);
/* the slot closed by the last flip: copy its (unconditioned) samples to the host, return their number */
int ft8b200_stream_fetch(ft8b200_stream_t *s, float *h_i, float *h_q, uint32_t *n_valid);
/* decoder() (rtlsdr_ft8d.c:221-285) for the slot closed by the last flip: skip if < 12 s, condition, decode */
int ft8b200_stream_decode(ft8b200_stream_t *s, struct decoder_results *h_results, int32_t *h_nresults);

/* ---- on-disk formats and whole recordings (csrc/files.cu) --------------------------------------------------------
 * Readers return the samples UNSCALED plus their peak max(|I|,|Q|): the reference's "normalise @ -3 dB" is applied on the
 * device (ft8b200_process_conditioned / ft8b200_condition).  Buffers hold 48000 floats; the tail is zero-filled.
 * replaces: readRawIQfile / readC2file (rtlsdr_ft8d.c:744-856), load_wav (ft8_lib/common/wave.c:66-128). */
int ft8b200_read_iq_file(const char *path, float *h_i, float *h_q, float *peak);                      /* -> pairs read, 0 = cannot open */
int ft8b200_read_c2_file(const char *path, float *h_i, float *h_q, float *peak, double *dial_freq, int *type, char *name15);
int ft8b200_load_wav(float *signal, int *num_samples, int *sample_rate, const char *path);            /* load_wav()'s contract; -3 = cannot open */
int ft8b200_load_wav_s16(int16_t *raw_s16, float *signal, int *num_samples, int *sample_rate, const char *path);
/* decodeRecordedFile() (rtlsdr_ft8d.c:859-887) for a batch of .iq / .c2 files: n x max_messages records, n counts */
int ft8b200_decode_iq_files(ft8b200_ctx_t *ctx, const char *const *paths, int n, struct decoder_results *h_results, int32_t *h_nresults,
                            int32_t *h_samples);
/* one line of decode_ft8's output: "000000 %3d %+4.2f %4.0f ~  %s" = score, time_sec, freq_hz, text (decode_ft8.c:399-401) */
typedef struct {
    char text[25];
    uint16_t hash;
    int16_t score;
    float time_sec;
    float freq_hz;
} ft8b200_decoded_t;
/* decode_ft8 main() (ft8_lib/decode_ft8.c:272-409) for n device-resident float recordings / n WAV files, FT8 or FT4:
 * h_out holds max_out_per_recording (>= max_messages) entries per recording, first-seen unique messages in candidate order. */
int ft8b200_decode_audio(ft8b200_ctx_t *ctx, const float *d_audio, size_t stride, int n_samples, int n, int sample_rate, int protocol,
                         ft8b200_decoded_t *h_out, int32_t *h_count, int max_out_per_recording);
int ft8b200_decode_wav_files(ft8b200_ctx_t *ctx, const char *const *paths, int n, int protocol, ft8b200_decoded_t *h_out, int32_t *h_count,
                             int max_out_per_recording, int32_t *h_status);
int ft8b200_get_config(ft8b200_ctx_t *ctx, ft8b200_config_t *cfg);

/* ---- device-side signal synthesis (csrc/synth.cu): the step before the path -------------------------------------
 * message -> 77-bit payload (host) -> CRC/LDPC/Gray/Costas symbols -> phase-continuous FSK + noise (device).
 * replaces for benchmarking/testing: pack77 (ft8_lib/ft8/pack.c), ft8_encode/ft4_encode (ft8/encode.c:22-195) and the
 * modulators of decoderSelfTest (rtlsdr_ft8d.c:937-955) / gen_ft8 (gen_ft8.c:28-102).  The waveform generator is integer
 * (32-bit phase accumulators, table cosine, counter-hash noise) so that a CPU twin reproduces it bit for bit. */
typedef struct {
    uint8_t payload[10];  /* 77-bit message, MSB first (ft8b200_pack77_std or any packer) */
    uint8_t reserved[2];  /* [0]: 0 = plain FSK as decoderSelfTest() sends it (rtlsdr_ft8d.c:937-955), 1 = GFSK as gen_ft8 does (gen_ft8.c:28-102:
                           *      Gaussian-smoothed frequency, BT 2 (FT8) / 1 (FT4), extended end symbols, raised-cosine ramps); [1]: 0 */
    float f0_hz;          /* frequency of tone 0 as the decoder will see it */
    float t0_sec;         /* start of symbol 0 */
    float amp;            /* raw path: amplitude in LSB; float paths: linear amplitude */
} ft8b200_signal_t;
int ft8b200_pack77_std(const char *call_to, const char *call_de, const char *extra, uint8_t *payload10);
/* replaces: pack77(), ft8_lib/ft8/pack.c:284-301 (what decoderSelfTest() and gen_ft8 call): a standard message when both call
 * fields pack (pack77_1, :167-218: "CQ K1JT FN20QI" packs as FN20), else 13 characters of free text (packtext77, :220-282).
 * Host code.  Returns 0 = standard message, 1 = free text, -1 = NULL argument (the reference returns 0 in both cases). */
int ft8b200_pack77(const char *msg, uint8_t *payload10);
/* n payloads (10 bytes each, host) -> n x 105 channel symbols (host; FT8 uses the first 79), computed on the device */
int ft8b200_encode_tones(ft8b200_ctx_t *ctx, const uint8_t *h_payloads, int n, int protocol, uint8_t *h_tones);
/* Slot s holds signals h_first[s] .. h_first[s+1]-1 (h_first has n_slots+1 entries).  Noise stream of slot s is selected by
 * (seed, first_slot_index + s): a batch generated in pieces or on several GPUs equals one generated at once. */
int ft8b200_synth_raw(ft8b200_ctx_t *ctx, const ft8b200_signal_t *h_signals, const int *h_first, int n_slots, float noise_lsb, uint64_t seed,
                      int first_slot_index, uint8_t *d_iq, size_t slot_stride_bytes, size_t bytes_per_slot, void *stream);
int ft8b200_synth_slots(ft8b200_ctx_t *ctx, const ft8b200_signal_t *h_signals, const int *h_first, int n_slots, float noise_sigma, uint64_t seed,
                        int first_slot_index, float *d_i, float *d_q, size_t slot_stride_samples, int n_samples, void *stream);
int ft8b200_synth_audio(ft8b200_ctx_t *ctx, const ft8b200_signal_t *h_signals, const int *h_first, int n_slots, int protocol, float noise_sigma,
                        uint64_t seed, int first_slot_index, float *d_audio, size_t slot_stride_samples, int n_samples, void *stream);

/* 12 kHz monitor waterfall, batched: n_slots x n_samples real audio -> u8[n_slots][blocks][time_osr][freq_osr][bins] */
int ft8b200_monitor_waterfall(ft8b200_ctx_t *ctx, const float *d_audio, size_t slot_stride_samples, int n_samples, int n_slots,
                              int sample_rate, int time_osr, int freq_osr, int protocol, uint8_t *d_mag, size_t mag_slot_stride,
                              int *num_blocks_out, void *stream);

/* ------------------------------------------------------------------------------------------
 * Reporting records: the step after the hot path (SURVEY.md section 8f rank 4).  HOST code, no sockets: these
 * build the bytes / strings the daemon's reporters emit; sending them stays with the caller.
 * ---------------------------------------------------------------------------------------- */

/* replaces: rtlsdr_ft8d.h:130-134 (24 bytes) -- dial frequency and identity of the receiving station */
#ifndef FT8B200_WITH_RTLSDR_FT8D_H
struct decoder_options {
    uint32_t freq;
    char rcall[13];
    char rloc[7];
};
#endif

/* The four form fields webClusterSpots() posts for one spot (buffer sizes of rtlsdr_ft8d.c:599-602; longer values truncate) */
typedef struct {
    char mycall[16]; /* "_mycall" */
    char dxcall[12]; /* "_dxcall" */
    char freq[10];   /* "_freq": kHz, "%8f" of a float */
    char info[100];  /* "_info":  "M2M FT8 [<rx locator> - <tx locator>]" */
} ft8b200_cluster_form_t;

#define FT8B200_PSK_MAX_DATAGRAM 1600

/* replaces: postSpots(), rtlsdr_ft8d.c:365-552 (the packet-building part; the UDP send at :554-582 stays with the caller).
 * One PSKreporter IPFIX datagram: header, the two template sets, the receiver record (call, locator, app_version) and one
 * sender record per spot (call, dial + freq, (int8)snr - 20, "FT8", locator, source 1, unixtime), until the sender set has
 * grown past 1200 bytes.  app_version NULL = ft8b200_report_app_version().  The reference uses sequence 1 and a per-process
 * rand() id.  Returns the datagram length, or -1 (bad argument / `cap` too small; FT8B200_PSK_MAX_DATAGRAM always fits). */
int ft8b200_pskreporter_datagram(const struct decoder_results *spots, uint32_t n_spots, const struct decoder_options *station,
                                 const char *app_version, uint32_t unixtime, uint32_t sequence, uint32_t random_id, uint8_t *out,
                                 size_t cap, uint32_t *n_reported);
/* The same for the records of a batch (the layout ft8b200_fetch_results / ft8b200_pipe_collect return: spots[n_slots][max_messages],
 * n_spots[n_slots]): datagram s at out + s*stride, its length in lengths[s] (0 for a slot without spots, which sends nothing);
 * sequence numbers count up from first_sequence over the datagrams actually built.  Returns the number of datagrams, or -1. */
int ft8b200_pskreporter_batch(const struct decoder_results *spots, const int32_t *n_spots, int n_slots, int max_messages,
                              const struct decoder_options *station, const char *app_version, const uint32_t *unixtime,
                              uint32_t first_sequence, uint32_t random_id, uint8_t *out, size_t stride, int32_t *lengths);
/* replaces: the field formatting of webClusterSpots(), rtlsdr_ft8d.c:603-606 (the curl POST stays with the caller) */
int ft8b200_webcluster_form(const struct decoder_results *spot, const struct decoder_options *station, ft8b200_cluster_form_t *form);
/* replaces: printSpots(), rtlsdr_ft8d.c:635-663: the console table (or the "No spot <UTC time>" line) into `out`.
 * Returns the number of characters needed, excluding the terminator (snprintf convention), or -1. */
int ft8b200_format_spots(const struct decoder_results *spots, uint32_t n_spots, uint32_t dial_freq, uint32_t unixtime, char *out, size_t cap);
const char *ft8b200_report_app_version(void);

#ifdef __cplusplus
}
#endif
#endif /* FT8B200_H */
