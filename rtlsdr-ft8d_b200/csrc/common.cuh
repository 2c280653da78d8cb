// common.cuh -- internal declarations shared by the kernels and the C-ABI layer of libft8b200.so.
// Nothing in csrc/ includes, links or calls anything under oracle/.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

#include "../../include/ft8b200.h"

namespace ft8b200 {

constexpr int kSlot = FT8B200_SLOT_SAMPLES;  // 48000
constexpr int kDecim = FT8B200_DECIM;        // 751
constexpr int kWfBytes = FT8B200_WF_BYTES;   // 94208
constexpr int kNfft = 1024;
constexpr int kFrames = 184;                 // 92 blocks x 2 time subdivisions
constexpr int kFirTaps = 57;
constexpr int kLdpcN = 174, kLdpcK = 91, kLdpcM = 83, kLdpcEdges = 522;

// per 751-sample block: sum s, sum i*s for the I and Q rails after the fs/4 mixer (int32, wrapping)
struct __align__(16) BlockSums { int32_t s0i, s1i, s0q, s1q; };

// ---- tables uploaded once per context (built on the host with the host libm, see tables.cu) ----
struct DeviceTables {
    float *window1024;     // sinf((float)((M_PI/1024)*i))               rtlsdr_ft8d.c:331-334
    float2 *twiddle1024;   // ((float)cos, (float)sin)(-2*pi*k/1024)      kiss_fft.c:351-357
    float *db_thresholds;  // [257] smallest x with quantise(x) >= k       rtlsdr_ft8d.c:1416,1425-1427
    float *wf_blob;        // the three tables above re-laid-out for waterfall1024_kernel (build_waterfall_tables)
    // monitor (12 kHz) tables, built lazily per nfft
    float *mon_window;     // fft_norm-free Hann, nfft floats
    float2 *mon_twiddle;   // nfft/2 complex twiddles
    float2 *mon_super;     // nfft/4 "super twiddles" of kiss_fftr
    int mon_nfft;
};

// ---- launchers (each returns cudaGetLastError()) ----
// gridDim.y limit: launches that put the slot (or stream) in blockIdx.y cover at most this many rows each; the slot-wise
// launchers run larger batches as consecutive launches, the raw-IQ entry points refuse more rows (FT8B200_MAX_RAW_ROWS)
constexpr int kMaxGridRows = 65535;
constexpr int kHistBlocks = 59; // block sums a flush needs from before its first block: 56 FIR taps + 3 comb delays
constexpr int kK1StreamingDense = -1;   // `variant` of launch_cic_block_sums: the streaming kernel at 5 CTAs per SM (for a launch that owns only part of the SMs)
cudaError_t launch_cic_block_sums(const uint8_t *d_iq, size_t stream_stride_bytes, int n_streams, int blocks_per_stream, BlockSums *d_sums,
                                  size_t sums_stride, int variant, int sm_count, cudaStream_t st, int *launches);
cudaError_t launch_cic_block_sums_generic(const uint8_t *d_iq_first_block, size_t stream_stride_bytes, int n_streams, uint32_t phase0, int n_blocks,
                                          BlockSums *d_sums_first_block, size_t sums_stride, cudaStream_t st, int *launches);
cudaError_t launch_cic_comb_fir(const BlockSums *d_sums, size_t sums_stride, int n_blocks, int out_offset, bool zero_fill, int n_streams,
                                float *d_i, float *d_q, uint32_t *d_count, float *d_peak, int32_t *d_y2, cudaStream_t st,
                                int *launches, int segs = 1, long long seg_samples = 0);
cudaError_t upload_fir_constants();  // once per device, synchronised (called by ft8b200_create / ft8b200_stream_create)
cudaError_t launch_shift_history(BlockSums *d_sums_with_prefix, int n_blocks, cudaStream_t st, int *launches);
cudaError_t launch_condition(float *d_i, float *d_q, const float *d_peak, int n_slots, cudaStream_t st, int *launches);
cudaError_t launch_waterfall(const DeviceTables &t, const float *d_i, const float *d_q, const float *d_peak, int n_slots, uint8_t *d_mag,
                             int sm_count, cudaStream_t st, int *launches);
void build_waterfall_tables(const float *window, const float2 *tw, const float *thr257, float *blob);
int waterfall_blob_floats();
cudaError_t upload_waterfall_constants(const float *blob_host);
cudaError_t run_quantiser_check(const float *d_thr257, unsigned long long *h_counts3, int sm_count, cudaStream_t st);
constexpr int kListCap = 1024;               // survivor words per slot handed from the score kernels to the selection (4 KB)
size_t find_sync_list_bytes(int n_slots);    // size of `d_lists`: per-slot counters + survivor lists
cudaError_t launch_find_sync(const uint8_t *d_mag, size_t slot_stride, int n_slots, int num_blocks, int num_bins, int time_osr, int freq_osr,
                             int protocol, int max_cand, int min_score, candidate_t *d_cand, int *d_ncand, int16_t *d_scores, uint32_t *d_lists,
                             uint32_t *d_work, unsigned int *d_work_total, int sm_count, cudaStream_t st, int *launches);
cudaError_t launch_decode(const uint8_t *d_mag, size_t slot_stride, int n_slots, int num_blocks, int num_bins, int time_osr, int freq_osr,
                          int protocol, int max_cand, int max_iters, const candidate_t *d_cand, const int *d_ncand, uint8_t *d_ok, uint8_t *d_stage,
                          decode_status_t *d_status, message_t *d_msg, uint8_t *d_plain, float *d_llr, const uint32_t *d_work,
                          unsigned int *d_work_total, int sm_count, cudaStream_t st, int *launches);
cudaError_t launch_spots(int n_slots, int max_cand, int max_msgs, int min_score, int freq_osr, const candidate_t *d_cand, const int *d_ncand,
                         const uint8_t *d_ok, const message_t *d_msg, struct decoder_results *d_results, int32_t *d_nresults,
                         message_t *d_umsg, float *d_ufreq, int32_t *d_uscore, int32_t *d_ucand, int16_t *d_table, cudaStream_t st, int *launches,
                         bool append = false, int32_t *d_first = nullptr);
// append (a later pass of multi-pass decoding): keep the slot's records and the log d_umsg/d_ufreq/d_uscore/d_ucand (required) of the
// earlier passes, de-duplicate against the log and append behind it.  d_first (optional): the slot's record count before this call.
// ordered-statistics decoding of the entries BP left at stage 1 or 2 (order 0: nothing attempted); with d_work the entries of the
// find_sync work list, otherwise all n_slots * max_cand.  *d_next: the pull counter, zeroed by the caller.
cudaError_t launch_osd(int n_slots, int max_cand, int protocol, int order, int max_hard, const float *d_llr, const int *d_ncand, uint8_t *d_ok,
                       uint8_t *d_stage, decode_status_t *d_status, message_t *d_msg, uint8_t *d_plain, uint8_t *d_osd, int32_t *d_osd_hard,
                       uint8_t *d_osd_cw, const uint32_t *d_work, const unsigned int *d_work_total, unsigned int *d_next, int sm_count,
                       cudaStream_t st, int *launches);
// subtract.cu: refinement + subtraction of decoded messages (multi-pass decoding).  Entry j in [lo, hi) of slot s is row
// (d_row ? d_row[s * list_stride + j] : j) of d_cand / d_cw (cand_stride rows per slot); d_grid (int32 [n_slots][list_stride][2])
// receives its refined (dt samples, df steps); y = x minus every listed message (y may be x).  zero_idle: a slot with no entry
// gets y = 0.  d_scratch: subtract_scratch_bytes.
cudaError_t upload_subtract_tables();
size_t subtract_scratch_bytes(int n_slots, int sm_count);
cudaError_t launch_subtract(const float *d_xi, const float *d_xq, float *d_yi, float *d_yq, int n_slots, const candidate_t *d_cand,
                            const uint8_t *d_cw, int cand_stride, const int32_t *d_row, const int32_t *d_lo, const int32_t *d_hi, int list_stride,
                            int32_t *d_grid, float2 *d_scratch, bool zero_idle, int sm_count, cudaStream_t st, int *launches);
// BP again on d_llr, with the hypothesis' codeword positions forced, for the entries the decoders before left at stage 1 or 2
// (on = 0: nothing attempted): a-priori decoding with cq_hypothesis(), fine-sync decoding with nothing forced (Hypothesis{}).
// d_flag / d_hard get every entry's outcome.  Work list as launch_osd; with d_next the warps pull entries from that counter (zeroed by
// the caller), without it they take a fixed stride.
struct Hypothesis {
    uint32_t mask[3], val[3];  // the forced codeword positions (bits 0-95) and their values
    uint32_t scr[3];           // the FT4 scramble of message bits 0-76, which the CQ gate undoes
    int cq_gate;               // accept only a plausible CQ: standard call_2, no R, a locator or none
};
Hypothesis cq_hypothesis(int protocol);  // "CQ ??? ???"
cudaError_t launch_rebp(int n_slots, int max_cand, int protocol, const Hypothesis &hyp, int on, int max_hard, int max_iters, const float *d_llr,
                        const int *d_ncand, uint8_t *d_ok, uint8_t *d_stage, decode_status_t *d_status, message_t *d_msg, uint8_t *d_plain,
                        uint8_t *d_flag, int32_t *d_hard, const uint32_t *d_work, const unsigned int *d_work_total, unsigned int *d_next,
                        int sm_count, cudaStream_t st, int *launches);
// fine-sync decoding, front half (finesync.cu): for the entries BP, OSD and AP left at stage 1 or 2 (on = 0: nothing attempted), the
// Costas search on the slots d_xi / d_xq (kSlot floats per slot) and the refined LLRs into d_llr ([n_slots][max_cand][174]) and d_grid
// ([n_slots][max_cand][2]), for the entries it attempts only; deep = 1 also writes sets b and c (DESIGN.md section 2.4.6) into d_llr_b
// and d_llr_c, laid out as d_llr.  Work list as launch_osd, *d_next: its pull counter, zeroed by the caller.  launch_rebp on d_llr is
// the back half.
cudaError_t upload_finesync_tables();
cudaError_t launch_finesync(int n_slots, int max_cand, int on, int deep, const float *d_xi, const float *d_xq, const candidate_t *d_cand,
                            const int *d_ncand, const uint8_t *d_stage, float *d_llr, float *d_llr_b, float *d_llr_c, int32_t *d_grid,
                            const uint32_t *d_work, const unsigned int *d_work_total, unsigned int *d_next, int sm_count, cudaStream_t st,
                            int *launches);
// deep mode's last step: the n entries' flag / hard rows of retry step i (0 ... 7, at d_flag / d_hard + i * n; bit i of `steps` = it
// ran) folded into d_fs / d_fs_hard, and d_how (0 = not decoded by fine sync, 1 + 3 set + decoder) written for every entry
cudaError_t launch_finesync_merge(size_t n, unsigned int steps, const uint8_t *d_flag, const int32_t *d_hard, uint8_t *d_fs, int32_t *d_fs_hard,
                                  uint8_t *d_how, int sm_count, cudaStream_t st, int *launches);
cudaError_t launch_unpack77_batch(const uint8_t *d_payloads, int n, char *d_text32, int32_t *d_status, cudaStream_t st, int *launches);
cudaError_t upload_ldpc_tables();
void set_decode_variant(int v);  // 0 = node-centred belief propagation (default), 1 = edge-centred
int decode_variant();
cudaError_t run_pade_check(unsigned long long *h_counts5, int sm_count, cudaStream_t st);

// api.cu: the context's device ordinal; find_sync / decode with an explicit protocol (independent of ft8b200_set_protocol)
int ctx_device(ft8b200_ctx_t *ctx);
// A failed CUDA runtime call also stays behind as the runtime's "last error" until somebody reads it -- the host application's next
// check (torch's, the daemon's own) would then report OUR failure as its own.  Every error path of the library goes through here:
// the reason goes to ft8b200_last_error(), the runtime's error state is cleared (a sticky error survives that, as it should),
// and FT8B200_ECUDA is returned.  e == cudaSuccess: whatever the runtime holds as its last error is taken instead.
int cuda_error(cudaError_t e, const char *where);
int api_error(int code, const char *why);   // `code` back, `why` into ft8b200_last_error()
int bad_argument(const char *func);        // FT8B200_EINVAL, "<func>: bad argument" into ft8b200_last_error()
#define FT8B200_BAD_ARG() ::ft8b200::bad_argument(__func__)
#define FT8B200_CUDA_FAIL() ::ft8b200::cuda_error(cudaSuccess, __func__)
int ctx_sm_count(ft8b200_ctx_t *ctx);
int find_sync_proto(ft8b200_ctx_t *ctx, int protocol, const uint8_t *d_mag, size_t slot_stride_bytes, int n_slots, int num_blocks, int num_bins,
                    int time_osr, int freq_osr, candidate_t *d_cand, int *d_ncand, void *stream);
int decode_proto(ft8b200_ctx_t *ctx, int protocol, const uint8_t *d_mag, size_t slot_stride_bytes, int n_slots, int num_blocks, int num_bins, int time_osr,
                 int freq_osr, const candidate_t *d_cand, const int *d_ncand, uint8_t *d_ok, uint8_t *d_stage, decode_status_t *d_status,
                 message_t *d_msg, uint8_t *d_plain, float *d_llr, void *stream);

// host-side table builders (tables.cu)
void build_window1024(float *w);
void build_twiddles(int n, float2 *tw);
void build_db_thresholds(float *t257);
void build_fir(float *z57);

}  // namespace ft8b200
