// api.cu -- the C ABI of libft8b200.so (include/ft8b200.h): contexts, workspaces, the batched device
// entry points and the whole-path pipelines.  Host-side C++ only; every numeric step is a CUDA kernel
// launched from here (decimator.cu, waterfall.cu, sync.cu, decode.cu).  No CPU fallback exists.
#include "common.cuh"

#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <string>
#include <vector>

using namespace ft8b200;

namespace {
thread_local std::string g_err;
int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}
int cuda_fail(cudaError_t e, const char *what) {
    const cudaError_t held = cudaGetLastError();   // read = clear (see cuda_error in common.cuh)
    if (e == cudaSuccess) e = held;
    g_err = std::string(what) + ": " + (e == cudaSuccess ? "failed" : cudaGetErrorString(e));
    return FT8B200_ECUDA;
}
#define CU(call)                                              \
    do {                                                      \
        cudaError_t e__ = (call);                             \
        if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
    } while (0)

struct DevBuf {
    void *p = nullptr;
    size_t bytes = 0;
    int ensure(size_t need) {
        if (need <= bytes) return 0;
        if (p) cudaFree(p);
        p = nullptr;
        bytes = 0;
        cudaError_t e = cudaMalloc(&p, need);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc");
        bytes = need;
        return 0;
    }
    // for buffers a kernel may read ahead of what was written into them (the selection fetches a slot's first 32 survivor words
    // together with the count that says how many of them exist): defined contents from the start
    int ensure_zeroed(size_t need) {
        if (need <= bytes) return 0;
        const int rc = ensure(need);
        if (rc) return rc;
        cudaError_t e = cudaMemset(p, 0, bytes);
        if (e == cudaSuccess) e = cudaStreamSynchronize(0);
        return e == cudaSuccess ? 0 : cuda_fail(e, "cudaMemset");
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        bytes = 0;
    }
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
    template <class T> T *at(size_t n) const { return p ? as<T>() + n : nullptr; }
};

// The per-candidate rows of one pass over S slots of K candidates: what find_sync and BP write, the codewords multi-pass decoding
// subtracts (plain), the LLRs OSD and AP read, the flag and hard-distance pair of each retry decoder (OSD, AP, fine sync), and which
// step of deep fine sync decoded a candidate (fs_how).  A buffer whose option is off is not allocated.
struct Rows {
    DevBuf mag, cand, ncand, ok, stage, status, msg, plain, llr, osd, osd_hard, ap, ap_hard, fs, fs_hard, fs_how;
    // the rows of slots s0...: every pointer moved to slot s0, nullptr for a buffer that does not exist or (llr, plain) is not used
    struct View {
        uint8_t *mag; candidate_t *cand; int *ncand; uint8_t *ok, *stage; decode_status_t *status; message_t *msg; uint8_t *plain; float *llr;
        uint8_t *osd; int32_t *osd_hard; uint8_t *ap; int32_t *ap_hard; uint8_t *fs; int32_t *fs_hard; uint8_t *fs_how;
    };
    // the LLRs and the pair of each retry decoder that is on
    int ensure_retry(size_t S, size_t K, bool osd_on, bool ap_on, bool fs_on, bool deep_on) {
        const size_t E = S * K;
        int rc;
        if ((osd_on || ap_on) && (rc = llr.ensure(E * kLdpcN * sizeof(float)))) return rc;
        if (osd_on && ((rc = osd.ensure(E)) || (rc = osd_hard.ensure(E * sizeof(int32_t))))) return rc;
        if (ap_on && ((rc = ap.ensure(E)) || (rc = ap_hard.ensure(E * sizeof(int32_t))))) return rc;
        if (fs_on && ((rc = fs.ensure(E)) || (rc = fs_hard.ensure(E * sizeof(int32_t))))) return rc;
        if (deep_on && (rc = fs_how.ensure(E))) return rc;
        return 0;
    }
    int ensure(size_t S, size_t K, bool osd_on, bool ap_on, bool fs_on, bool deep_on, bool need_plain) {
        int rc;
        if ((rc = mag.ensure(S * kWfBytes)) || (rc = cand.ensure(S * K * sizeof(candidate_t))) || (rc = ncand.ensure(S * sizeof(int)))) return rc;
        if ((rc = ok.ensure(S * K)) || (rc = stage.ensure(S * K)) || (rc = status.ensure(S * K * sizeof(decode_status_t)))) return rc;
        if ((rc = msg.ensure(S * K * sizeof(message_t)))) return rc;
        if (need_plain && (rc = plain.ensure(S * K * kLdpcN))) return rc;
        return ensure_retry(S, K, osd_on, ap_on, fs_on, deep_on);
    }
    void release() {
        for (DevBuf *b : {&mag, &cand, &ncand, &ok, &stage, &status, &msg, &plain, &llr, &osd, &osd_hard, &ap, &ap_hard, &fs, &fs_hard, &fs_how})
            b->release();
    }
    View at(int s0, size_t K, bool llr_on, bool plain_on) const {
        const size_t o = (size_t)s0 * K;
        return {mag.at<uint8_t>((size_t)s0 * kWfBytes), cand.at<candidate_t>(o), ncand.at<int>(s0), ok.at<uint8_t>(o), stage.at<uint8_t>(o),
                status.at<decode_status_t>(o), msg.at<message_t>(o), plain_on ? plain.at<uint8_t>(o * kLdpcN) : nullptr,
                llr_on ? llr.at<float>(o * kLdpcN) : nullptr, osd.at<uint8_t>(o), osd_hard.at<int32_t>(o), ap.at<uint8_t>(o),
                ap_hard.at<int32_t>(o), fs.at<uint8_t>(o), fs_hard.at<int32_t>(o), fs_how.at<uint8_t>(o)};
    }
};
}  // namespace

constexpr int kMaxGroups = 16;

struct ft8b200_ctx {
    ft8b200_config_t cfg;
    cudaStream_t stream = nullptr;         // effective launching stream: own_stream, or the front-end partition's stream
    cudaStream_t own_stream = nullptr;
    DeviceTables tb = {};
    int launches = 0;
    uint64_t launches_total = 0;
    int sm_count = 0;
    // workspaces (grown on demand); pass1: the per-candidate rows of the path's first pass, and of the stage-wise retry decoders
    DevBuf raw, sums, si, sq, peak, count, results, nresults, table, lists, scores, work, work_total;
    Rows pass1;
    // the retry decoders after BP, each 0 = off: ordered-statistics decoding (ft8b200_set_osd), a-priori decoding of "CQ ??? ???"
    // (ft8b200_set_ap) and fine-sync decoding (ft8b200_set_finesync), whose refined LLRs and grid points fs_llr / fs_grid are
    // scratch between finesync_kernel and the BP after it, shared by all passes
    int osd_order = 0;
    int osd_max_hard = FT8B200_OSD_DEFAULT_MAX_HARD;
    int ap_on = 0;
    int ap_max_hard = FT8B200_AP_DEFAULT_MAX_HARD;
    int fs_on = 0;
    int fs_max_hard = FT8B200_FINESYNC_DEFAULT_MAX_HARD;
    DevBuf fs_llr, fs_grid;
    // deep fine sync (ft8b200_set_finesync_deep), 0 = off: with fine sync on, the nsym = 2 and 3 sets and OSD / AP on the refined sets.
    // Scratch, for slots s0 ... s0 + n at offset s0: sets b and c (deep_llr, [2][n][K][174]) and the flag / hard rows of the 8 extra
    // retry steps (deep_flag, deep_hard, [8][n][K])
    int fs_deep = 0;
    int fs_deep_max_hard = FT8B200_FINESYNC_DEEP_DEFAULT_MAX_HARD;
    DevBuf deep_llr, deep_flag, deep_hard;
    // multi-pass decoding (ft8b200_set_passes): 1 = off.  With passes > 1: the slot's log of accepted messages across passes
    // (ulog/ufreq/uscore/ucand, first = record count before the last pass), the refined grid points, the residual slots (ri/rq), and
    // the rows of the later passes
    int passes = 1;
    DevBuf ulog, ufreq, uscore, ucand, first, grid, ri, rq, sub_scratch;
    Rows later;
    // optional per-stage timing of the last process_* call (CUDA events on the launching stream)
    bool profiling = false;
    int overlap = 0;                       // number of slot groups ft8b200_process_raw pipelines (0/1 = off)
    int protocol = PROTO_FT8;              // what ft8b200_find_sync / ft8b200_decode score and demap (ft8b200_set_protocol)
    int k1_variant = 0;                    // 0 = streaming cic_block_sums kernel, >= 1 = persistent bulk-copy kernel (shape index)
    bool side_back = false;                // back end on the high-priority side stream even with a single group (pipe lanes)
    bool comb_front = false;               // with an SM partition: comb+FIR stays on the front partition (ft8b200_set_comb_front)
    cudaEvent_t front_wait = nullptr;      // one-shot: the next process_raw's block sums wait for it (ft8b200_set_front_wait), its memsets do not
    cudaEvent_t ev_front = nullptr;        // recorded on the launching stream right after the last process_raw's cic_block_sums
    cudaEvent_t ev_k1 = nullptr;
    cudaEvent_t ev_back = nullptr;         // recorded on the back-end stream behind the last process_raw's spot table (ft8b200_back_event)
    cudaEvent_t back_wait = nullptr;       // one-shot: the next process_raw's back end waits for it (ft8b200_set_back_wait)
    cudaEvent_t ev[7][kMaxGroups][2] = {};   // stage 6: subtraction and the later passes (passes > 1)
    bool ev_valid[7][kMaxGroups] = {};
    cudaStream_t aux = nullptr;            // high-priority side stream for the back end of a slot group
    cudaStream_t own_aux = nullptr;
    int sm_back = 0;                       // SMs the back-end kernels size their persistent grids for (0 = sm_count)
    cudaEvent_t ev_join = nullptr;
    cudaEvent_t ev_group[kMaxGroups] = {};
    std::mutex mu;
};

namespace {

int ctx_enter(ft8b200_ctx_t *ctx) {
    if (!ctx) return fail(FT8B200_EINVAL, "null context");
    cudaError_t e = cudaSetDevice(ctx->cfg.device);
    if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
    return 0;
}
cudaStream_t pick(ft8b200_ctx_t *ctx, void *stream) { return stream ? reinterpret_cast<cudaStream_t>(stream) : ctx->stream; }
void tally(ft8b200_ctx_t *ctx) {
    ctx->launches_total += (uint64_t)ctx->launches;
    ctx->launches = 0;
}

int ensure_slot_buffers(ft8b200_ctx_t *ctx, int n_slots) {
    const size_t K = (size_t)ctx->cfg.max_candidates, M = (size_t)ctx->cfg.max_messages, S = (size_t)n_slots;
    const bool multi = ctx->passes > 1;
    int rc;
    const bool deep = ctx->fs_on && ctx->fs_deep;
    if ((rc = ctx->pass1.ensure(S, K, ctx->osd_order, ctx->ap_on, ctx->fs_on, deep, multi))) return rc;
    if ((rc = ctx->results.ensure(S * M * sizeof(struct decoder_results)))) return rc;
    if ((rc = ctx->nresults.ensure(S * sizeof(int32_t)))) return rc;
    if ((rc = ctx->table.ensure(S * M * sizeof(int16_t)))) return rc;
    if (ctx->fs_on && ((rc = ctx->fs_llr.ensure(S * K * kLdpcN * sizeof(float))) || (rc = ctx->fs_grid.ensure(S * K * 2 * sizeof(int32_t))))) return rc;
    if (deep && ((rc = ctx->deep_llr.ensure(2 * S * K * kLdpcN * sizeof(float))) || (rc = ctx->deep_flag.ensure(8 * S * K)) ||
                 (rc = ctx->deep_hard.ensure(8 * S * K * sizeof(int32_t)))))
        return rc;
    if (!multi) return 0;
    if ((rc = ctx->later.ensure(S, K, ctx->osd_order, ctx->ap_on, ctx->fs_on, deep, true))) return rc;
    if ((rc = ctx->ulog.ensure(S * M * sizeof(message_t))) || (rc = ctx->ufreq.ensure(S * M * sizeof(float)))) return rc;
    if ((rc = ctx->uscore.ensure(S * M * sizeof(int32_t))) || (rc = ctx->ucand.ensure(S * M * sizeof(int32_t)))) return rc;
    if ((rc = ctx->first.ensure(S * sizeof(int32_t))) || (rc = ctx->grid.ensure(S * M * 2 * sizeof(int32_t)))) return rc;
    if ((rc = ctx->ri.ensure(S * kSlot * sizeof(float))) || (rc = ctx->rq.ensure(S * kSlot * sizeof(float)))) return rc;
    return ctx->sub_scratch.ensure(subtract_scratch_bytes(n_slots, ctx->sm_count));
}

int ensure_scratch(ft8b200_ctx_t *ctx, int npos, int n_slots) {
    int rc0 = ctx->scores.ensure((size_t)n_slots * npos * sizeof(int16_t));
    if (rc0) return rc0;
    if ((rc0 = ctx->lists.ensure_zeroed(find_sync_list_bytes(n_slots)))) return rc0;   // survivor lists, score kernel -> selection
    if ((rc0 = ctx->work.ensure((size_t)n_slots * ctx->cfg.max_candidates * sizeof(uint32_t)))) return rc0;
    if ((rc0 = ctx->work_total.ensure(5 * sizeof(unsigned int)))) return rc0;
    return 0;
}

// Deep fine sync (DESIGN.md section 2.4.6) after the BP on set a (llr[0]) of n slots: OSD and AP on set a, then BP, OSD and AP on sets
// b and c, each where it is on and on what the steps before left at stage 1 or 2, capped at min(its own cap, the deep cap), their
// outcomes into step i's rows of flag / hard ([8][n][K]); then the merge into fs / fs_hard / fs_how.  Every step walks its entries in
// a fixed stride, so none needs a pull counter.
int launch_deep(ft8b200_ctx_t *ctx, const Rows::View &r, int n, const float *const (&llr)[3], uint8_t *flag, int32_t *hard, uint8_t *fs,
                int32_t *fs_hard, uint8_t *fs_how, const uint32_t *work, const unsigned int *total, int sms, cudaStream_t st) {
    const int K = ctx->cfg.max_candidates, iters = ctx->cfg.ldpc_iterations, cap = ctx->fs_deep_max_hard;
    const size_t nk = (size_t)n * K;
    unsigned int steps = 0;
    for (int set = 0; set < 3; ++set) {
        for (int dec = set ? 0 : 1; dec < 3; ++dec) {   // BP, OSD, AP; set a's BP has run
            const int i = 3 * set + dec - 1;
            uint8_t *f = flag + i * nk;
            int32_t *h = hard + i * nk;
            if (dec == 0) {
                CU(launch_rebp(n, K, PROTO_FT8, Hypothesis{}, 1, std::min(ctx->fs_max_hard, cap), iters, llr[set], r.ncand, r.ok, r.stage, r.status, r.msg,
                               r.plain, f, h, work, total, nullptr, sms, st, &ctx->launches));
            } else if (dec == 1) {
                if (!ctx->osd_order) continue;
                CU(launch_osd(n, K, PROTO_FT8, ctx->osd_order, std::min(ctx->osd_max_hard, cap), llr[set], r.ncand, r.ok, r.stage, r.status, r.msg, r.plain,
                              f, h, nullptr, work, total, nullptr, sms, st, &ctx->launches));
            } else {
                if (!ctx->ap_on) continue;
                CU(launch_rebp(n, K, PROTO_FT8, cq_hypothesis(PROTO_FT8), 1, std::min(ctx->ap_max_hard, cap), iters, llr[set], r.ncand, r.ok, r.stage,
                               r.status, r.msg, r.plain, f, h, work, total, nullptr, sms, st, &ctx->launches));
            }
            steps |= 1u << i;
        }
    }
    CU(launch_finesync_merge(nk, steps, flag, hard, fs, fs_hard, fs_how, sms, st, &ctx->launches));
    return 0;
}

// What runs after BP on the rows r of n slots starting at slot s0: OSD, AP and fine sync, each where it is on, each on what the ones
// before it left at stage 1 or 2.  With the work list (the whole path) they visit its entries and find_sync has zeroed their pull
// counters, words [2] - [4] of work_total; without it (ft8b200_decode) they visit every entry and the counters they use are zeroed
// here.  Fine sync demodulates the slot samples xi / xq (kSlot floats per slot); without samples it does not run.  Deep fine sync
// (launch_deep) follows it where on.
int launch_retries(ft8b200_ctx_t *ctx, int protocol, const Rows::View &r, int s0, int n, const float *xi, const float *xq, const uint32_t *work,
                   int sms, cudaStream_t st) {
    const int K = ctx->cfg.max_candidates, iters = ctx->cfg.ldpc_iterations;
    unsigned int *counters = ctx->work_total.as<unsigned int>();
    const unsigned int *total = work ? counters : nullptr;
    if (ctx->osd_order) {
        if (!work) CU(cudaMemsetAsync(counters + 2, 0, sizeof(unsigned int), st));
        CU(launch_osd(n, K, protocol, ctx->osd_order, ctx->osd_max_hard, r.llr, r.ncand, r.ok, r.stage, r.status, r.msg, r.plain, r.osd, r.osd_hard,
                      nullptr, work, total, counters + 2, sms, st, &ctx->launches));
    }
    if (ctx->ap_on) {
        if (!work) CU(cudaMemsetAsync(counters + 3, 0, sizeof(unsigned int), st));
        CU(launch_rebp(n, K, protocol, cq_hypothesis(protocol), 1, ctx->ap_max_hard, iters, r.llr, r.ncand, r.ok, r.stage, r.status, r.msg, r.plain,
                       r.ap, r.ap_hard, work, total, counters + 3, sms, st, &ctx->launches));
    }
    if (ctx->fs_on && xi) {  // (finesync_kernel demodulates FT8)
        float *fs_llr = ctx->fs_llr.as<float>() + (size_t)s0 * K * kLdpcN;
        const bool deep = ctx->fs_deep;
        float *deep_llr = deep ? ctx->deep_llr.as<float>() + 2 * (size_t)s0 * K * kLdpcN : nullptr;
        const size_t set_floats = (size_t)n * K * kLdpcN;
        if (!work) CU(cudaMemsetAsync(counters + 4, 0, sizeof(unsigned int), st));
        CU(launch_finesync(n, K, 1, deep, xi, xq, r.cand, r.ncand, r.stage, fs_llr, deep_llr, deep ? deep_llr + set_floats : nullptr,
                           ctx->fs_grid.as<int32_t>() + (size_t)s0 * K * 2, work, total, counters + 4, sms, st, &ctx->launches));
        CU(launch_rebp(n, K, PROTO_FT8, Hypothesis{}, 1, ctx->fs_max_hard, iters, fs_llr, r.ncand, r.ok, r.stage, r.status, r.msg, r.plain, r.fs,
                       r.fs_hard, work, total, nullptr, sms, st, &ctx->launches));
        if (deep) {
            const float *const sets[3] = {fs_llr, deep_llr, deep_llr + set_floats};
            if (int rc = launch_deep(ctx, r, n, sets, ctx->deep_flag.as<uint8_t>() + 8 * (size_t)s0 * K, ctx->deep_hard.as<int32_t>() + 8 * (size_t)s0 * K,
                                     r.fs, r.fs_hard, r.fs_how, work, total, sms, st))
                return rc;
        }
    }
    return 0;
}

}  // namespace

extern "C" {

const char *ft8b200_last_error(void) { return g_err.c_str(); }
const char *ft8b200_version(void) { return "ft8b200 0.1 (sm_100a)"; }

void ft8b200_default_config(ft8b200_config_t *cfg) {
    if (!cfg) return;
    cfg->device = 0;
    cfg->max_slots = 1;
    cfg->max_candidates = 120;  // K_MAX_CANDIDATES, rtlsdr_ft8d.h:46
    cfg->max_messages = 50;     // K_MAX_MESSAGES,   rtlsdr_ft8d.h:48
    cfg->min_score = 10;        // K_MIN_SCORE,      rtlsdr_ft8d.h:45
    cfg->ldpc_iterations = 20;  // K_LDPC_ITERS,     rtlsdr_ft8d.h:47
}

ft8b200_ctx_t *ft8b200_create(const ft8b200_config_t *cfg_in) {
    ft8b200_config_t cfg;
    ft8b200_default_config(&cfg);
    if (cfg_in) cfg = *cfg_in;
    if (cfg.max_candidates < 1 || cfg.max_candidates > 30000 || cfg.max_messages < 1 || cfg.max_messages > 30000 || cfg.ldpc_iterations < 0) {
        fail(FT8B200_EINVAL, "bad configuration");
        return nullptr;
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev <= 0) {
        g_err = std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                " (libft8b200 has no CPU fallback)";
        return nullptr;
    }
    if (cfg.device < 0 || cfg.device >= ndev) {
        fail(FT8B200_EINVAL, "device ordinal out of range");
        return nullptr;
    }
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, cfg.device)) != cudaSuccess) { cuda_fail(e, "cudaGetDeviceProperties"); return nullptr; }
    if (prop.major != 10) {
        g_err = "device " + std::to_string(cfg.device) + " is sm_" + std::to_string(prop.major) + std::to_string(prop.minor) +
                "; libft8b200 is built for sm_100a only and has no fallback";
        return nullptr;
    }
    if ((e = cudaSetDevice(cfg.device)) != cudaSuccess) { cuda_fail(e, "cudaSetDevice"); return nullptr; }
    ft8b200_ctx_t *ctx = new ft8b200_ctx();
    ctx->cfg = cfg;
    ctx->sm_count = prop.multiProcessorCount;
    if (const char *e = getenv("FT8B200_K1")) ctx->k1_variant = atoi(e);  // experiments; ft8b200_set_decimator_variant is the API
    bool okc = true;
    // non-blocking: work queued here must not serialise with whatever the host application does on the legacy NULL stream
    // (e.g. a synchronous cudaMemcpy of gathered records would otherwise wait for every batch in flight)
    okc = okc && cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) == cudaSuccess;
    ctx->stream = ctx->own_stream;
    // tables, built with the host libm exactly as the reference builds them
    std::vector<float> win(kNfft), thr(257);
    std::vector<float2> tw(kNfft);
    build_window1024(win.data());
    build_twiddles(kNfft, tw.data());
    build_db_thresholds(thr.data());
    okc = okc && cudaMalloc(&ctx->tb.window1024, kNfft * sizeof(float)) == cudaSuccess;
    okc = okc && cudaMalloc(&ctx->tb.twiddle1024, kNfft * sizeof(float2)) == cudaSuccess;
    okc = okc && cudaMalloc(&ctx->tb.db_thresholds, 257 * sizeof(float)) == cudaSuccess;
    okc = okc && cudaMemcpy(ctx->tb.window1024, win.data(), kNfft * sizeof(float), cudaMemcpyHostToDevice) == cudaSuccess;
    okc = okc && cudaMemcpy(ctx->tb.twiddle1024, tw.data(), kNfft * sizeof(float2), cudaMemcpyHostToDevice) == cudaSuccess;
    okc = okc && cudaMemcpy(ctx->tb.db_thresholds, thr.data(), 257 * sizeof(float), cudaMemcpyHostToDevice) == cudaSuccess;
    okc = okc && upload_fir_constants() == cudaSuccess;
    okc = okc && upload_ldpc_tables() == cudaSuccess;
    okc = okc && upload_subtract_tables() == cudaSuccess;
    okc = okc && upload_finesync_tables() == cudaSuccess;
    {
        std::vector<float> blob(waterfall_blob_floats());
        build_waterfall_tables(win.data(), tw.data(), thr.data(), blob.data());
        okc = okc && cudaMalloc(&ctx->tb.wf_blob, blob.size() * sizeof(float)) == cudaSuccess;
        okc = okc && cudaMemcpy(ctx->tb.wf_blob, blob.data(), blob.size() * sizeof(float), cudaMemcpyHostToDevice) == cudaSuccess;
        okc = okc && upload_waterfall_constants(blob.data()) == cudaSuccess;
    }
    if (!okc) {
        cuda_fail(cudaGetLastError(), "context initialisation");
        ft8b200_destroy(ctx);
        return nullptr;
    }
    return ctx;
}

void ft8b200_destroy(ft8b200_ctx_t *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->cfg.device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->own_stream) { cudaStreamSynchronize(ctx->own_stream); cudaStreamDestroy(ctx->own_stream); }
    for (auto &s : ctx->ev) for (auto &g : s) for (cudaEvent_t e : g) if (e) cudaEventDestroy(e);
    if (ctx->aux) cudaStreamSynchronize(ctx->aux);
    if (ctx->own_aux) { cudaStreamSynchronize(ctx->own_aux); cudaStreamDestroy(ctx->own_aux); }
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    if (ctx->ev_k1) cudaEventDestroy(ctx->ev_k1);
    if (ctx->ev_back) cudaEventDestroy(ctx->ev_back);
    for (cudaEvent_t e : ctx->ev_group) if (e) cudaEventDestroy(e);
    cudaFree(ctx->tb.window1024); cudaFree(ctx->tb.twiddle1024); cudaFree(ctx->tb.db_thresholds); cudaFree(ctx->tb.wf_blob);
    cudaFree(ctx->tb.mon_window); cudaFree(ctx->tb.mon_twiddle); cudaFree(ctx->tb.mon_super);
    DevBuf *bufs[] = {&ctx->raw, &ctx->sums, &ctx->si, &ctx->sq, &ctx->peak, &ctx->count, &ctx->results, &ctx->nresults, &ctx->table, &ctx->lists,
                      &ctx->scores, &ctx->work, &ctx->work_total, &ctx->fs_llr, &ctx->fs_grid, &ctx->deep_llr, &ctx->deep_flag, &ctx->deep_hard,
                      &ctx->ulog, &ctx->ufreq, &ctx->uscore, &ctx->ucand, &ctx->first, &ctx->grid, &ctx->ri, &ctx->rq, &ctx->sub_scratch};
    for (DevBuf *b : bufs) b->release();
    ctx->pass1.release();
    ctx->later.release();
    delete ctx;
}

int ft8b200_get_config(ft8b200_ctx_t *ctx, ft8b200_config_t *cfg) {
    if (!ctx || !cfg) return fail(FT8B200_EINVAL, "ft8b200_get_config: null argument");
    *cfg = ctx->cfg;
    return 0;
}

void *ft8b200_cuda_stream(ft8b200_ctx_t *ctx) { return ctx ? ctx->stream : nullptr; }
int ft8b200_sync(ft8b200_ctx_t *ctx) {
    int rc = ctx_enter(ctx);
    if (rc) return rc;
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}
uint64_t ft8b200_kernel_launches(ft8b200_ctx_t *ctx) { return ctx ? ctx->launches_total : 0; }

static int decimate_impl(ft8b200_ctx_t *ctx, const uint8_t *d_iq, size_t bytes_per_stream, size_t stream_stride_bytes, int n_streams, int segs,
                         size_t seg_bytes, float *d_i, float *d_q, uint32_t *d_count, float *d_peak, int32_t *d_y2, void *stream) {
    int rc = ctx_enter(ctx);
    if (rc) return rc;
    if (!d_iq || !d_i || !d_q || n_streams < 1) return fail(FT8B200_EINVAL, "ft8b200_decimate: null buffer or n_streams < 1");
    if ((bytes_per_stream & 7) || (stream_stride_bytes & 15) || (((size_t)d_iq) & 15))
        return fail(FT8B200_EINVAL, "ft8b200_decimate: byte counts must be multiples of 8, stream stride and base 16-byte aligned");
    if (segs < 1 || (segs > 1 && (seg_bytes < 8 || (seg_bytes & 7) || seg_bytes * (size_t)segs > bytes_per_stream || seg_bytes / 2 / kDecim + 1 > (size_t)kSlot)))
        return fail(FT8B200_EINVAL, "ft8b200_decimate_streams: slots_per_stream * bytes_per_slot must fit the stream, bytes_per_slot a multiple of 8 and <= one 48000-sample slot");
    if ((long long)n_streams * segs > FT8B200_MAX_RAW_ROWS)
        return fail(FT8B200_EINVAL, "ft8b200_decimate: more than FT8B200_MAX_RAW_ROWS (65535) streams or output rows in one call; split the batch");
    const int blocks = (int)((bytes_per_stream / 2) / kDecim);
    // the 128-bit loads of the last super-block may read up to 14 bytes past the last complete block
    if ((size_t)(blocks / 8) * 12016 > bytes_per_stream) return fail(FT8B200_EINVAL, "internal: super-block overrun");
    std::lock_guard<std::mutex> lk(ctx->mu);
    cudaStream_t st = pick(ctx, stream);
    const size_t sstride = (size_t)blocks + kHistBlocks;
    if ((rc = ctx->sums.ensure((size_t)n_streams * sstride * sizeof(BlockSums)))) return rc;
    if (d_peak) CU(cudaMemsetAsync(d_peak, 0, sizeof(float) * n_streams * segs, st));
    // fresh filter state: the history prefix of every stream is zero
    CU(cudaMemset2DAsync(ctx->sums.p, sstride * sizeof(BlockSums), 0, kHistBlocks * sizeof(BlockSums), n_streams, st));
    BlockSums *s0 = ctx->sums.as<BlockSums>() + kHistBlocks;
    CU(launch_cic_block_sums(d_iq, stream_stride_bytes, n_streams, blocks, s0, sstride, ctx->k1_variant, ctx->sm_count, st, &ctx->launches));
    CU(launch_cic_comb_fir(s0, sstride, blocks, 0, true, n_streams, d_i, d_q, d_count, d_peak, d_y2, st, &ctx->launches, segs,
                           (long long)(seg_bytes / 2)));
    tally(ctx);
    return 0;
}

int ft8b200_decimate(ft8b200_ctx_t *ctx, const uint8_t *d_iq, size_t bytes_per_stream, size_t stream_stride_bytes, int n_streams, float *d_i,
                     float *d_q, uint32_t *d_count, float *d_peak, int32_t *d_y2, void *stream) {
    return decimate_impl(ctx, d_iq, bytes_per_stream, stream_stride_bytes, n_streams, 1, 0, d_i, d_q, d_count, d_peak, d_y2, stream);
}

int ft8b200_decimate_streams(ft8b200_ctx_t *ctx, const uint8_t *d_iq, size_t bytes_per_stream, size_t stream_stride_bytes, int n_streams,
                             int slots_per_stream, size_t bytes_per_slot, float *d_i, float *d_q, uint32_t *d_count, float *d_peak, int32_t *d_y2,
                             void *stream) {
    return decimate_impl(ctx, d_iq, bytes_per_stream, stream_stride_bytes, n_streams, slots_per_stream, bytes_per_slot, d_i, d_q, d_count, d_peak,
                         d_y2, stream);
}

int ft8b200_condition(ft8b200_ctx_t *ctx, float *d_i, float *d_q, const float *d_peak, int n_slots, void *stream) {
    int rc = ctx_enter(ctx);
    if (rc) return rc;
    if (!d_i || !d_q || !d_peak || n_slots < 1) return fail(FT8B200_EINVAL, "ft8b200_condition: bad argument");
    CU(launch_condition(d_i, d_q, d_peak, n_slots, pick(ctx, stream), &ctx->launches));
    tally(ctx);
    return 0;
}

int ft8b200_waterfall(ft8b200_ctx_t *ctx, const float *d_i, const float *d_q, const float *d_peak, int n_slots, uint8_t *d_mag, void *stream) {
    int rc = ctx_enter(ctx);
    if (rc) return rc;
    if (!d_i || !d_q || !d_mag || n_slots < 1) return fail(FT8B200_EINVAL, "ft8b200_waterfall: bad argument");
    if ((((size_t)d_mag) | ((size_t)d_i) | ((size_t)d_q)) & 15) return fail(FT8B200_EINVAL, "ft8b200_waterfall: d_i, d_q and d_mag must be 16-byte aligned");
    CU(launch_waterfall(ctx->tb, d_i, d_q, d_peak, n_slots, d_mag, ctx->sm_count, pick(ctx, stream), &ctx->launches));
    tally(ctx);
    return 0;
}

}  // extern "C"

// find_sync / decode with an explicit protocol (the C entry points use the context's, ft8b200_set_protocol): what the whole-
// recording calls of files.cu use, so that they neither change nor depend on the protocol selected for the stage-wise API
namespace ft8b200 {
int cuda_error(cudaError_t e, const char *where) { return cuda_fail(e, where); }
int api_error(int code, const char *why) { return fail(code, why); }
int bad_argument(const char *func) { return fail(FT8B200_EINVAL, std::string(func) + ": bad argument"); }
int ctx_device(ft8b200_ctx_t *ctx) { return ctx ? ctx->cfg.device : -1; }
int ctx_sm_count(ft8b200_ctx_t *ctx) { return ctx ? ctx->sm_count : 0; }

int find_sync_proto(ft8b200_ctx_t *ctx, int protocol, const uint8_t *d_mag, size_t slot_stride_bytes, int n_slots, int num_blocks, int num_bins,
                    int time_osr, int freq_osr, candidate_t *d_cand, int *d_ncand, void *stream) {
    int rc = ctx_enter(ctx);
    if (rc) return rc;
    if (!d_mag || !d_cand || !d_ncand || n_slots < 1 || num_blocks < 1 || num_bins < 8 || time_osr < 1 || freq_osr < 1)
        return fail(FT8B200_EINVAL, "ft8b200_find_sync: bad argument");
    const long npos = (long)time_osr * freq_osr * 36 * (num_bins - 7);
    if (npos >= (1l << 20)) return fail(FT8B200_EINVAL, "ft8b200_find_sync: waterfall too large (position index exceeds 20 bits)");
    std::lock_guard<std::mutex> lk(ctx->mu);
    if ((rc = ensure_scratch(ctx, (int)npos, n_slots))) return rc;
    CU(launch_find_sync(d_mag, slot_stride_bytes, n_slots, num_blocks, num_bins, time_osr, freq_osr, protocol, ctx->cfg.max_candidates, ctx->cfg.min_score,
                        d_cand, d_ncand, ctx->scores.as<int16_t>(), ctx->lists.as<uint32_t>(), nullptr, nullptr, ctx->sm_count,
                        pick(ctx, stream), &ctx->launches));
    tally(ctx);
    return 0;
}

int decode_proto(ft8b200_ctx_t *ctx, int protocol, const uint8_t *d_mag, size_t slot_stride_bytes, int n_slots, int num_blocks, int num_bins, int time_osr,
                 int freq_osr, const candidate_t *d_cand, const int *d_ncand, uint8_t *d_ok, uint8_t *d_stage, decode_status_t *d_status,
                 message_t *d_msg, uint8_t *d_plain, float *d_llr, void *stream) {
    int rc = ctx_enter(ctx);
    if (rc) return rc;
    if (!d_mag || !d_cand || !d_ncand || !d_ok || !d_stage || !d_status || !d_msg || n_slots < 1)
        return fail(FT8B200_EINVAL, "ft8b200_decode: bad argument");
    std::lock_guard<std::mutex> lk(ctx->mu);
    if ((rc = ctx->work_total.ensure(5 * sizeof(unsigned int)))) return rc;
    cudaStream_t st = pick(ctx, stream);
    unsigned int *pull = nullptr;
    if (decode_variant() == 0 && (size_t)n_slots * ctx->cfg.max_candidates > 8u * 4u * (size_t)ctx->sm_count) {
        // more candidates than resident warps: let the warps pull them (counter = word [1], see launch_decode)
        pull = ctx->work_total.as<unsigned int>();
        CU(cudaMemsetAsync(pull, 0, 4 * sizeof(unsigned int), st));
    }
    // OSD's and AP's outputs go to pass 1's rows (ft8b200_osd_workspace, ft8b200_ap_workspace), and so do the LLRs when the caller
    // passes none; everything else is the caller's
    if ((rc = ctx->pass1.ensure_retry((size_t)n_slots, (size_t)ctx->cfg.max_candidates, ctx->osd_order, ctx->ap_on, false, false))) return rc;
    Rows::View r = ctx->pass1.at(0, ctx->cfg.max_candidates, ctx->osd_order || ctx->ap_on, false);
    r.cand = const_cast<candidate_t *>(d_cand);  // the retry decoders only read the candidates
    r.ncand = const_cast<int *>(d_ncand);
    r.ok = d_ok; r.stage = d_stage; r.status = d_status; r.msg = d_msg; r.plain = d_plain;
    if (d_llr) r.llr = d_llr;
    CU(launch_decode(d_mag, slot_stride_bytes, n_slots, num_blocks, num_bins, time_osr, freq_osr, protocol, ctx->cfg.max_candidates, ctx->cfg.ldpc_iterations,
                     d_cand, d_ncand, d_ok, d_stage, d_status, d_msg, d_plain, r.llr, nullptr, pull, ctx->sm_count, st, &ctx->launches));
    // no slot samples: the stage-wise decode runs OSD and AP; fine sync is its own entry point (ft8b200_finesync)
    if ((rc = launch_retries(ctx, protocol, r, 0, n_slots, nullptr, nullptr, nullptr, ctx->sm_count, st))) return rc;
    tally(ctx);
    return 0;
}
}  // namespace ft8b200

extern "C" {

int ft8b200_find_sync(ft8b200_ctx_t *ctx, const uint8_t *d_mag, size_t slot_stride_bytes, int n_slots, int num_blocks, int num_bins, int time_osr,
                      int freq_osr, candidate_t *d_cand, int *d_ncand, void *stream) {
    if (!ctx) return fail(FT8B200_EINVAL, "null context");
    return find_sync_proto(ctx, ctx->protocol, d_mag, slot_stride_bytes, n_slots, num_blocks, num_bins, time_osr, freq_osr, d_cand, d_ncand, stream);
}

int ft8b200_decode(ft8b200_ctx_t *ctx, const uint8_t *d_mag, size_t slot_stride_bytes, int n_slots, int num_blocks, int num_bins, int time_osr,
                   int freq_osr, const candidate_t *d_cand, const int *d_ncand, uint8_t *d_ok, uint8_t *d_stage, decode_status_t *d_status,
                   message_t *d_msg, uint8_t *d_plain, float *d_llr, void *stream) {
    if (!ctx) return fail(FT8B200_EINVAL, "null context");
    return decode_proto(ctx, ctx->protocol, d_mag, slot_stride_bytes, n_slots, num_blocks, num_bins, time_osr, freq_osr, d_cand, d_ncand, d_ok, d_stage,
                        d_status, d_msg, d_plain, d_llr, stream);
}

int ft8b200_spots(ft8b200_ctx_t *ctx, int n_slots, int freq_osr, const candidate_t *d_cand, const int *d_ncand, const uint8_t *d_ok,
                  const message_t *d_msg, struct decoder_results *d_results, int32_t *d_nresults, message_t *d_umsg, float *d_ufreq,
                  int32_t *d_uscore, int32_t *d_ucand, void *stream) {
    int rc = ctx_enter(ctx);
    if (rc) return rc;
    if (!d_cand || !d_ncand || !d_ok || !d_msg || !d_results || !d_nresults || n_slots < 1) return fail(FT8B200_EINVAL, "ft8b200_spots: bad argument");
    if (d_umsg && (!d_ufreq || !d_uscore)) return fail(FT8B200_EINVAL, "ft8b200_spots: d_umsg needs d_ufreq and d_uscore");
    std::lock_guard<std::mutex> lk(ctx->mu);
    if ((rc = ctx->table.ensure((size_t)n_slots * ctx->cfg.max_messages * sizeof(int16_t)))) return rc;
    CU(launch_spots(n_slots, ctx->cfg.max_candidates, ctx->cfg.max_messages, ctx->cfg.min_score, freq_osr, d_cand, d_ncand, d_ok, d_msg, d_results,
                    d_nresults, d_umsg, d_ufreq, d_uscore, d_ucand, ctx->table.as<int16_t>(), pick(ctx, stream), &ctx->launches));
    tally(ctx);
    return 0;
}

int ft8b200_set_osd(ft8b200_ctx_t *ctx, int order, int max_hard_errors) {
    if (!ctx || order < 0 || order > 2) return fail(FT8B200_EINVAL, "ft8b200_set_osd: order 0 (off), 1 or 2");
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->osd_order = order;
    ctx->osd_max_hard = max_hard_errors < 0 ? FT8B200_OSD_DEFAULT_MAX_HARD : max_hard_errors;
    return 0;
}

int ft8b200_set_ap(ft8b200_ctx_t *ctx, int on, int max_hard_errors) {
    if (!ctx) return fail(FT8B200_EINVAL, "null context");
    if (on != 0 && on != 1) return fail(FT8B200_EINVAL, "ft8b200_set_ap: on must be 0 (off, the default) or 1");
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->ap_on = on;
    ctx->ap_max_hard = max_hard_errors < 0 ? FT8B200_AP_DEFAULT_MAX_HARD : max_hard_errors;
    return 0;
}

int ft8b200_set_finesync(ft8b200_ctx_t *ctx, int on, int max_hard_errors) {
    if (!ctx) return fail(FT8B200_EINVAL, "null context");
    if (on != 0 && on != 1) return fail(FT8B200_EINVAL, "ft8b200_set_finesync: on must be 0 (off, the default) or 1");
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->fs_on = on;
    ctx->fs_max_hard = max_hard_errors < 0 ? FT8B200_FINESYNC_DEFAULT_MAX_HARD : max_hard_errors;
    return 0;
}

int ft8b200_set_finesync_deep(ft8b200_ctx_t *ctx, int on, int max_hard_errors) {
    if (!ctx) return fail(FT8B200_EINVAL, "null context");
    if (on != 0 && on != 1) return fail(FT8B200_EINVAL, "ft8b200_set_finesync_deep: on must be 0 (off, the default) or 1");
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->fs_deep = on;
    ctx->fs_deep_max_hard = max_hard_errors < 0 ? FT8B200_FINESYNC_DEEP_DEFAULT_MAX_HARD : max_hard_errors;
    return 0;
}

int ft8b200_set_passes(ft8b200_ctx_t *ctx, int passes) {
    if (!ctx) return fail(FT8B200_EINVAL, "null context");
    if (passes < 1 || passes > 3) return fail(FT8B200_EINVAL, "ft8b200_set_passes: passes must be 1 (one pass, the default), 2 or 3");
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->passes = passes;
    return 0;
}

int ft8b200_subtract(ft8b200_ctx_t *ctx, const float *d_i, const float *d_q, int n_slots, const candidate_t *d_cand, const uint8_t *d_cw,
                     const int32_t *d_nmsg, float *d_ri, float *d_rq, int32_t *d_grid, void *stream) {
    int rc = ctx_enter(ctx);
    if (rc) return rc;
    if (!d_i || !d_q || !d_cand || !d_cw || !d_nmsg || !d_ri || !d_rq || !d_grid || n_slots < 1 || n_slots > FT8B200_MAX_RAW_ROWS)
        return fail(FT8B200_EINVAL, "ft8b200_subtract: null buffer or n_slots outside 1 ... 65535");
    if ((((size_t)d_i) | ((size_t)d_q) | ((size_t)d_ri) | ((size_t)d_rq)) & 3) return fail(FT8B200_EINVAL, "ft8b200_subtract: float buffers must be 4-byte aligned");
    std::lock_guard<std::mutex> lk(ctx->mu);
    if ((rc = ctx->sub_scratch.ensure(subtract_scratch_bytes(n_slots, ctx->sm_count)))) return rc;
    const int M = ctx->cfg.max_messages;
    CU(launch_subtract(d_i, d_q, d_ri, d_rq, n_slots, d_cand, d_cw, M, nullptr, nullptr, d_nmsg, M, d_grid, ctx->sub_scratch.as<float2>(), false,
                       ctx->sm_count, pick(ctx, stream), &ctx->launches));
    tally(ctx);
    return 0;
}

int ft8b200_osd(ft8b200_ctx_t *ctx, const float *d_llr, int n_slots, const int *d_ncand, uint8_t *d_ok, uint8_t *d_stage, decode_status_t *d_status,
                message_t *d_msg, uint8_t *d_plain, uint8_t *d_osd, int32_t *d_osd_hard, uint8_t *d_osd_cw, void *stream) {
    int rc = ctx_enter(ctx);
    if (rc) return rc;
    if (!d_llr || !d_ncand || !d_ok || !d_stage || !d_status || !d_msg || !d_osd || !d_osd_hard || n_slots < 1)
        return fail(FT8B200_EINVAL, "ft8b200_osd: bad argument");
    std::lock_guard<std::mutex> lk(ctx->mu);
    if ((rc = ctx->work_total.ensure(5 * sizeof(unsigned int)))) return rc;
    cudaStream_t st = pick(ctx, stream);
    unsigned int *next = ctx->work_total.as<unsigned int>() + 2;
    CU(cudaMemsetAsync(next, 0, sizeof(unsigned int), st));
    CU(launch_osd(n_slots, ctx->cfg.max_candidates, ctx->protocol, ctx->osd_order, ctx->osd_max_hard, d_llr, d_ncand, d_ok, d_stage, d_status, d_msg,
                  d_plain, d_osd, d_osd_hard, d_osd_cw, nullptr, nullptr, next, ctx->sm_count, st, &ctx->launches));
    tally(ctx);
    return 0;
}

int ft8b200_osd_workspace(ft8b200_ctx_t *ctx, uint8_t **d_osd, int32_t **d_osd_hard) {
    if (!ctx) return fail(FT8B200_EINVAL, "null context");
    if (d_osd) *d_osd = ctx->pass1.osd.as<uint8_t>();
    if (d_osd_hard) *d_osd_hard = ctx->pass1.osd_hard.as<int32_t>();
    return 0;
}

int ft8b200_ap(ft8b200_ctx_t *ctx, const float *d_llr, int n_slots, const int *d_ncand, uint8_t *d_ok, uint8_t *d_stage, decode_status_t *d_status,
               message_t *d_msg, uint8_t *d_plain, uint8_t *d_ap, int32_t *d_ap_hard, void *stream) {
    int rc = ctx_enter(ctx);
    if (rc) return rc;
    if (!d_llr || !d_ncand || !d_ok || !d_stage || !d_status || !d_msg || !d_ap || !d_ap_hard || n_slots < 1)
        return fail(FT8B200_EINVAL, "ft8b200_ap: bad argument");
    std::lock_guard<std::mutex> lk(ctx->mu);
    if ((rc = ctx->work_total.ensure(5 * sizeof(unsigned int)))) return rc;
    cudaStream_t st = pick(ctx, stream);
    unsigned int *next = ctx->work_total.as<unsigned int>() + 3;
    CU(cudaMemsetAsync(next, 0, sizeof(unsigned int), st));
    CU(launch_rebp(n_slots, ctx->cfg.max_candidates, ctx->protocol, cq_hypothesis(ctx->protocol), ctx->ap_on, ctx->ap_max_hard, ctx->cfg.ldpc_iterations,
                   d_llr, d_ncand, d_ok, d_stage, d_status, d_msg, d_plain, d_ap, d_ap_hard, nullptr, nullptr, next, ctx->sm_count, st, &ctx->launches));
    tally(ctx);
    return 0;
}

int ft8b200_ap_workspace(ft8b200_ctx_t *ctx, uint8_t **d_ap, int32_t **d_ap_hard) {
    if (!ctx) return fail(FT8B200_EINVAL, "null context");
    if (d_ap) *d_ap = ctx->pass1.ap.as<uint8_t>();
    if (d_ap_hard) *d_ap_hard = ctx->pass1.ap_hard.as<int32_t>();
    return 0;
}

int ft8b200_finesync(ft8b200_ctx_t *ctx, const float *d_i, const float *d_q, int n_slots, const candidate_t *d_cand, const int *d_ncand, uint8_t *d_ok,
                     uint8_t *d_stage, decode_status_t *d_status, message_t *d_msg, uint8_t *d_plain, uint8_t *d_fs, int32_t *d_fs_hard,
                     int32_t *d_fs_grid, float *d_fs_llr, void *stream) {
    int rc = ctx_enter(ctx);
    if (rc) return rc;
    if (!d_i || !d_q || !d_cand || !d_ncand || !d_ok || !d_stage || !d_status || !d_msg || !d_fs || !d_fs_hard || !d_fs_grid || n_slots < 1 ||
        n_slots > FT8B200_MAX_RAW_ROWS)
        return fail(FT8B200_EINVAL, "ft8b200_finesync: null buffer or n_slots outside 1 ... 65535");
    if ((((size_t)d_i) | ((size_t)d_q) | ((size_t)d_fs_llr)) & 3) return fail(FT8B200_EINVAL, "ft8b200_finesync: float buffers must be 4-byte aligned");
    std::lock_guard<std::mutex> lk(ctx->mu);
    if ((rc = ctx->work_total.ensure(5 * sizeof(unsigned int)))) return rc;
    const int K = ctx->cfg.max_candidates;
    const size_t nk = (size_t)n_slots * K;
    if (!d_fs_llr) {
        if ((rc = ctx->fs_llr.ensure(nk * kLdpcN * sizeof(float)))) return rc;
        d_fs_llr = ctx->fs_llr.as<float>();
    }
    // deep mode: sets b and c and the extra steps' rows in the context's scratch, fs_how into pass 1's row (ft8b200_finesync_deep_workspace)
    const bool deep = ctx->fs_on && ctx->fs_deep;
    if (deep && ((rc = ctx->deep_llr.ensure(2 * nk * kLdpcN * sizeof(float))) || (rc = ctx->deep_flag.ensure(8 * nk)) ||
                 (rc = ctx->deep_hard.ensure(8 * nk * sizeof(int32_t))) || (rc = ctx->pass1.fs_how.ensure(nk))))
        return rc;
    float *deep_llr = deep ? ctx->deep_llr.as<float>() : nullptr;
    cudaStream_t st = pick(ctx, stream);
    unsigned int *next = ctx->work_total.as<unsigned int>() + 4;
    CU(cudaMemsetAsync(next, 0, sizeof(unsigned int), st));
    CU(launch_finesync(n_slots, K, ctx->fs_on, deep, d_i, d_q, d_cand, d_ncand, d_stage, d_fs_llr, deep_llr, deep ? deep_llr + nk * kLdpcN : nullptr,
                       d_fs_grid, nullptr, nullptr, next, ctx->sm_count, st, &ctx->launches));
    CU(launch_rebp(n_slots, K, PROTO_FT8, Hypothesis{}, ctx->fs_on, ctx->fs_max_hard, ctx->cfg.ldpc_iterations, d_fs_llr, d_ncand, d_ok, d_stage, d_status,
                   d_msg, d_plain, d_fs, d_fs_hard, nullptr, nullptr, nullptr, ctx->sm_count, st, &ctx->launches));
    if (deep) {
        Rows::View r = {};
        r.ncand = const_cast<int *>(d_ncand);   // the retry decoders only read the counts
        r.ok = d_ok; r.stage = d_stage; r.status = d_status; r.msg = d_msg; r.plain = d_plain;
        const float *const sets[3] = {d_fs_llr, deep_llr, deep_llr + nk * kLdpcN};
        if ((rc = launch_deep(ctx, r, n_slots, sets, ctx->deep_flag.as<uint8_t>(), ctx->deep_hard.as<int32_t>(), d_fs, d_fs_hard,
                              ctx->pass1.fs_how.as<uint8_t>(), nullptr, nullptr, ctx->sm_count, st)))
            return rc;
    }
    tally(ctx);
    return 0;
}

int ft8b200_finesync_sets(ft8b200_ctx_t *ctx, const float *d_i, const float *d_q, int n_slots, const candidate_t *d_cand, const int *d_ncand,
                          const uint8_t *d_stage, int32_t *d_grid, float *d_llr_sets, void *stream) {
    int rc = ctx_enter(ctx);
    if (rc) return rc;
    if (!d_i || !d_q || !d_cand || !d_ncand || !d_stage || !d_grid || !d_llr_sets || n_slots < 1 || n_slots > FT8B200_MAX_RAW_ROWS)
        return fail(FT8B200_EINVAL, "ft8b200_finesync_sets: null buffer or n_slots outside 1 ... 65535");
    if ((((size_t)d_i) | ((size_t)d_q) | ((size_t)d_grid) | ((size_t)d_llr_sets)) & 3)
        return fail(FT8B200_EINVAL, "ft8b200_finesync_sets: d_i, d_q, d_grid and d_llr_sets must be 4-byte aligned");
    std::lock_guard<std::mutex> lk(ctx->mu);
    if ((rc = ctx->work_total.ensure(5 * sizeof(unsigned int)))) return rc;
    cudaStream_t st = pick(ctx, stream);
    unsigned int *next = ctx->work_total.as<unsigned int>() + 4;
    CU(cudaMemsetAsync(next, 0, sizeof(unsigned int), st));
    const size_t set_floats = (size_t)n_slots * ctx->cfg.max_candidates * kLdpcN;
    CU(launch_finesync(n_slots, ctx->cfg.max_candidates, 1, 1, d_i, d_q, d_cand, d_ncand, d_stage, d_llr_sets, d_llr_sets + set_floats,
                       d_llr_sets + 2 * set_floats, d_grid, nullptr, nullptr, next, ctx->sm_count, st, &ctx->launches));
    tally(ctx);
    return 0;
}

int ft8b200_finesync_deep_workspace(ft8b200_ctx_t *ctx, uint8_t **d_fs_how) {
    if (!ctx) return fail(FT8B200_EINVAL, "null context");
    if (d_fs_how) *d_fs_how = ctx->pass1.fs_how.as<uint8_t>();
    return 0;
}

int ft8b200_finesync_workspace(ft8b200_ctx_t *ctx, uint8_t **d_fs, int32_t **d_fs_hard) {
    if (!ctx) return fail(FT8B200_EINVAL, "null context");
    if (d_fs) *d_fs = ctx->pass1.fs.as<uint8_t>();
    if (d_fs_hard) *d_fs_hard = ctx->pass1.fs_hard.as<int32_t>();
    return 0;
}

// ---- per-stage timing: one event pair per (stage, group); stage times are summed over the groups -------------
static void mark(ft8b200_ctx_t *ctx, int stage, int group, bool end, cudaStream_t st) {
    if (!ctx->profiling || group >= kMaxGroups) return;
    cudaEvent_t &e = ctx->ev[stage][group][end ? 1 : 0];
    if (!e) cudaEventCreate(&e);
    const bool ok = cudaEventRecord(e, st) == cudaSuccess;
    if (end) ctx->ev_valid[stage][group] = ok && ctx->ev_valid[stage][group];
    else ctx->ev_valid[stage][group] = ok;
}
static void clear_marks(ft8b200_ctx_t *ctx) {
    for (auto &s : ctx->ev_valid) for (bool &v : s) v = false;
}

// waterfall -> sync -> decode -> spots for slots [s0, s0+n) of the context buffers, all on `st`; with passes > 1 the decoded
// messages are then subtracted and the residual searched again (later_passes)
static int later_passes(ft8b200_ctx_t *ctx, const Rows::View &p1, const float *d_i, const float *d_q, const float *d_peak, int s0, int n, int sms,
                        cudaStream_t st);
static int run_back_end(ft8b200_ctx_t *ctx, const float *d_i, const float *d_q, const float *d_peak, int s0, int n, int group, cudaStream_t st) {
    const size_t K = (size_t)ctx->cfg.max_candidates, M = (size_t)ctx->cfg.max_messages;
    const bool multi = ctx->passes > 1;
    const Rows::View r = ctx->pass1.at(s0, K, ctx->osd_order || ctx->ap_on, multi);  // plain: the codewords subtraction needs
    const float *xi = d_i + (size_t)s0 * kSlot, *xq = d_q + (size_t)s0 * kSlot;
    uint32_t *work = ctx->work.as<uint32_t>();
    unsigned int *work_total = ctx->work_total.as<unsigned int>();
    const int sms = (ctx->sm_back > 0 && st == ctx->aux) ? ctx->sm_back : ctx->sm_count;  // persistent grids fit the back-end partition
    mark(ctx, 2, group, false, st);
    // decoder()'s normalisation (when d_peak != NULL) is applied on load inside the waterfall kernel
    CU(launch_waterfall(ctx->tb, xi, xq, d_peak ? d_peak + s0 : nullptr, n, r.mag, sms, st, &ctx->launches));
    mark(ctx, 2, group, true, st);
    mark(ctx, 3, group, false, st);
    CU(launch_find_sync(r.mag, kWfBytes, n, 92, 256, 2, 2, PROTO_FT8, ctx->cfg.max_candidates, ctx->cfg.min_score, r.cand, r.ncand,
                        ctx->scores.as<int16_t>(), ctx->lists.as<uint32_t>(), work, work_total, sms, st, &ctx->launches));
    mark(ctx, 3, group, true, st);
    mark(ctx, 4, group, false, st);
    CU(launch_decode(r.mag, kWfBytes, n, 92, 256, 2, 2, PROTO_FT8, ctx->cfg.max_candidates, ctx->cfg.ldpc_iterations, r.cand, r.ncand, r.ok, r.stage,
                     r.status, r.msg, r.plain, r.llr, work, work_total, sms, st, &ctx->launches));
    if (int rc = launch_retries(ctx, PROTO_FT8, r, s0, n, xi, xq, work, sms, st)) return rc;
    mark(ctx, 4, group, true, st);
    mark(ctx, 5, group, false, st);
    if (!multi) {
        CU(launch_spots(n, ctx->cfg.max_candidates, ctx->cfg.max_messages, ctx->cfg.min_score, 2, r.cand, r.ncand, r.ok, r.msg,
                        ctx->results.as<struct decoder_results>() + (size_t)s0 * M, ctx->nresults.as<int32_t>() + s0, nullptr, nullptr, nullptr, nullptr,
                        ctx->table.as<int16_t>() + (size_t)s0 * M, st, &ctx->launches));
    } else {   // the same table, which also logs what it accepts, in order, for the subtraction and the later passes' de-duplication
        CU(launch_spots(n, ctx->cfg.max_candidates, ctx->cfg.max_messages, ctx->cfg.min_score, 2, r.cand, r.ncand, r.ok, r.msg,
                        ctx->results.as<struct decoder_results>() + (size_t)s0 * M, ctx->nresults.as<int32_t>() + s0, ctx->ulog.as<message_t>() + (size_t)s0 * M,
                        ctx->ufreq.as<float>() + (size_t)s0 * M, ctx->uscore.as<int32_t>() + (size_t)s0 * M, ctx->ucand.as<int32_t>() + (size_t)s0 * M,
                        ctx->table.as<int16_t>() + (size_t)s0 * M, st, &ctx->launches, false, ctx->first.as<int32_t>() + s0));
    }
    mark(ctx, 5, group, true, st);
    if (multi) {
        mark(ctx, 6, group, false, st);
        if (int rc = later_passes(ctx, r, d_i, d_q, d_peak, s0, n, sms, st)) return rc;
        mark(ctx, 6, group, true, st);
    }
    return 0;
}

// Pass p >= 2 (DESIGN.md section 2.4.2): the messages pass p - 1 accepted as new (log entries [first, nresults) of each slot) are
// refined on that pass's input x and subtracted from it into the residual slots (in place from pass 3 on); a slot with none gets a
// zero residual and so no candidates.  The residual goes through waterfall (with the slot's original peak scale: the quantiser is
// absolute), sync, decode and the retry decoders (launch_retries: OSD, AP and fine sync on the residual, where on) into the later-pass
// rows, and the spot table appends what is new.  p1: pass 1's rows of these slots.
static int later_passes(ft8b200_ctx_t *ctx, const Rows::View &p1, const float *d_i, const float *d_q, const float *d_peak, int s0, int n, int sms,
                        cudaStream_t st) {
    const size_t K = (size_t)ctx->cfg.max_candidates, M = (size_t)ctx->cfg.max_messages;
    const float *xi = d_i + (size_t)s0 * kSlot, *xq = d_q + (size_t)s0 * kSlot;
    float *ri = ctx->ri.as<float>() + (size_t)s0 * kSlot, *rq = ctx->rq.as<float>() + (size_t)s0 * kSlot;
    const Rows::View r = ctx->later.at(s0, K, ctx->osd_order || ctx->ap_on, true);
    const candidate_t *prev_cand = p1.cand;
    const uint8_t *prev_plain = p1.plain;
    uint32_t *work = ctx->work.as<uint32_t>();
    unsigned int *work_total = ctx->work_total.as<unsigned int>();
    int32_t *first = ctx->first.as<int32_t>() + s0, *nres = ctx->nresults.as<int32_t>() + s0, *ucand = ctx->ucand.as<int32_t>() + (size_t)s0 * M;
    for (int p = 2; p <= ctx->passes; ++p) {
        CU(launch_subtract(xi, xq, ri, rq, n, prev_cand, prev_plain, (int)K, ucand, first, nres, (int)M, ctx->grid.as<int32_t>() + (size_t)s0 * M * 2,
                           ctx->sub_scratch.as<float2>(), true, sms, st, &ctx->launches));
        xi = ri;
        xq = rq;
        CU(launch_waterfall(ctx->tb, ri, rq, d_peak ? d_peak + s0 : nullptr, n, r.mag, sms, st, &ctx->launches));
        CU(launch_find_sync(r.mag, kWfBytes, n, 92, 256, 2, 2, PROTO_FT8, ctx->cfg.max_candidates, ctx->cfg.min_score, r.cand, r.ncand,
                            ctx->scores.as<int16_t>(), ctx->lists.as<uint32_t>(), work, work_total, sms, st, &ctx->launches));
        CU(launch_decode(r.mag, kWfBytes, n, 92, 256, 2, 2, PROTO_FT8, ctx->cfg.max_candidates, ctx->cfg.ldpc_iterations, r.cand, r.ncand, r.ok, r.stage,
                         r.status, r.msg, r.plain, r.llr, work, work_total, sms, st, &ctx->launches));
        if (int rc = launch_retries(ctx, PROTO_FT8, r, s0, n, ri, rq, work, sms, st)) return rc;
        CU(launch_spots(n, ctx->cfg.max_candidates, ctx->cfg.max_messages, ctx->cfg.min_score, 2, r.cand, r.ncand, r.ok, r.msg,
                        ctx->results.as<struct decoder_results>() + (size_t)s0 * M, nres, ctx->ulog.as<message_t>() + (size_t)s0 * M,
                        ctx->ufreq.as<float>() + (size_t)s0 * M, ctx->uscore.as<int32_t>() + (size_t)s0 * M, ucand, ctx->table.as<int16_t>() + (size_t)s0 * M,
                        st, &ctx->launches, true, first));
        prev_cand = r.cand;
        prev_plain = r.plain;
    }
    return 0;
}

static int ensure_aux(ft8b200_ctx_t *ctx) {
    if (!ctx->aux) {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);  // hi is the numerically lowest = highest priority
        CU(cudaStreamCreateWithPriority(&ctx->own_aux, cudaStreamNonBlocking, hi));
        ctx->aux = ctx->own_aux;
    }
    if (!ctx->ev_join) {
        CU(cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&ctx->ev_k1, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&ctx->ev_back, cudaEventDisableTiming));
        for (cudaEvent_t &e : ctx->ev_group) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    return 0;
}

static int process_raw_impl(ft8b200_ctx_t *ctx, const uint8_t *d_iq, size_t bytes_per_stream, size_t stream_stride_bytes, int n_slots, int segs,
                            size_t seg_bytes, void *stream) {
    int rc = ctx_enter(ctx);
    if (rc) return rc;
    if (!d_iq || n_slots < 1) return fail(FT8B200_EINVAL, "ft8b200_process_raw: bad argument");
    if ((bytes_per_stream & 7) || (stream_stride_bytes & 15) || (((size_t)d_iq) & 15))
        return fail(FT8B200_EINVAL, "ft8b200_process_raw: byte counts must be multiples of 8, stream stride and base 16-byte aligned");
    if (segs < 1 || (segs > 1 && (seg_bytes < 8 || (seg_bytes & 7) || seg_bytes * (size_t)segs > bytes_per_stream || seg_bytes / 2 / kDecim + 1 > (size_t)kSlot)))
        return fail(FT8B200_EINVAL, "ft8b200_process_raw_streams: slots_per_stream * bytes_per_slot must fit the stream, bytes_per_slot a multiple of 8 and <= one 48000-sample slot");
    if ((long long)n_slots * segs > FT8B200_MAX_RAW_ROWS)
        return fail(FT8B200_EINVAL, "ft8b200_process_raw: more than FT8B200_MAX_RAW_ROWS (65535) streams or result rows in one call; split the batch");
    std::lock_guard<std::mutex> lk(ctx->mu);
    cudaStream_t st = pick(ctx, stream);
    const int blocks = (int)((bytes_per_stream / 2) / kDecim);
    const int n_rows = n_slots * segs;  // 15 s slots to decode: (receiver stream, consecutive slot)
    if ((rc = ensure_slot_buffers(ctx, n_rows))) return rc;
    const size_t sstride = (size_t)blocks + kHistBlocks;
    if ((rc = ctx->sums.ensure((size_t)n_slots * sstride * sizeof(BlockSums)))) return rc;
    if ((rc = ctx->si.ensure((size_t)n_rows * kSlot * sizeof(float)))) return rc;
    if ((rc = ctx->sq.ensure((size_t)n_rows * kSlot * sizeof(float)))) return rc;
    if ((rc = ctx->peak.ensure((size_t)n_rows * sizeof(float)))) return rc;
    if ((rc = ctx->count.ensure((size_t)n_rows * sizeof(uint32_t)))) return rc;
    // Slot groups: the HBM-bound front end (block sums, comb+FIR) of group g+1 runs on the caller's stream while the
    // compute-bound back end (waterfall, sync, LDPC, spots) of group g runs on a high-priority side stream.
    int n_groups = 1;
    if (ctx->overlap > 1 && n_slots >= 2 * ctx->overlap) {
        n_groups = ctx->overlap;  // a group must stay large enough for the back end to fill the machine
        if (n_groups > kMaxGroups) n_groups = kMaxGroups;
    }
    const int per = (n_slots + n_groups - 1) / n_groups;
    const int npos = 2 * 2 * 36 * (256 - 7);
    if ((rc = ensure_scratch(ctx, npos, per * segs))) return rc;
    cudaStream_t back = st;
    const bool side = n_groups > 1 || ctx->side_back;
    if (side) {
        if ((rc = ensure_aux(ctx))) return rc;
        back = ctx->aux;
        CU(cudaEventRecord(ctx->ev_join, st));           // the side stream starts after everything already queued on st
        CU(cudaStreamWaitEvent(back, ctx->ev_join, 0));
        if (ctx->back_wait) {  // the executor's second chain: back ends of consecutive batches (other lanes' streams) never share their SMs
            CU(cudaStreamWaitEvent(back, ctx->back_wait, 0));
        }
    }
    ctx->back_wait = nullptr;
    clear_marks(ctx);
    CU(cudaMemsetAsync(ctx->peak.p, 0, sizeof(float) * n_rows, st));
    CU(cudaMemset2DAsync(ctx->sums.p, sstride * sizeof(BlockSums), 0, kHistBlocks * sizeof(BlockSums), n_slots, st));  // fresh filter state
    if (ctx->front_wait) {  // the executor's chain: the previous batch's block sums must have finished -- the two memsets above need not wait for that
        CU(cudaStreamWaitEvent(st, ctx->front_wait, 0));
        ctx->front_wait = nullptr;
    }
    for (int g = 0, s0 = 0; s0 < n_slots; ++g, s0 += per) {
        const int n = (n_slots - s0) < per ? (n_slots - s0) : per;
        const int r0 = s0 * segs, nr = n * segs;
        BlockSums *sg = ctx->sums.as<BlockSums>() + (size_t)s0 * sstride + kHistBlocks;
        mark(ctx, 0, g, false, st);
        CU(launch_cic_block_sums(d_iq + (size_t)s0 * stream_stride_bytes, stream_stride_bytes, n, blocks, sg, sstride,
                                 (ctx->k1_variant == 0 && ctx->sm_back > 0) ? kK1StreamingDense : ctx->k1_variant,   // on a front partition: see cic_block_sums_kernel
                                 ctx->sm_count, st, &ctx->launches));
        mark(ctx, 0, g, true, st);
        if (side && s0 + per >= n_slots) {
            // the next batch's block sums (another lane) may start now: comb+FIR below is 2 % of the front end's bytes and
            // fills the ramp-up of that kernel instead of leaving the memory system idle between batches
            CU(cudaEventRecord(ctx->ev_k1, st));
            ctx->ev_front = ctx->ev_k1;
        }
        // With an SM partition the comb+FIR pass belongs to the back end's SM set: it is a whole-GPU grid, and on the front
        // set its CTAs would queue ahead of the next batch's block sums (measured: the two then run back to back).
        cudaStream_t fst = st;
        if (side && ctx->sm_back > 0 && !ctx->comb_front) {
            CU(cudaEventRecord(ctx->ev_group[g], st));
            CU(cudaStreamWaitEvent(back, ctx->ev_group[g], 0));
            fst = back;
        }
        mark(ctx, 1, g, false, fst);
        CU(launch_cic_comb_fir(sg, sstride, blocks, 0, true, n, ctx->si.as<float>() + (size_t)r0 * kSlot,
                               ctx->sq.as<float>() + (size_t)r0 * kSlot, ctx->count.as<uint32_t>() + r0, ctx->peak.as<float>() + r0, nullptr, fst,
                               &ctx->launches, segs, (long long)(seg_bytes / 2)));
        mark(ctx, 1, g, true, fst);
        if (side && fst == st) {
            CU(cudaEventRecord(ctx->ev_group[g], st));
            CU(cudaStreamWaitEvent(back, ctx->ev_group[g], 0));
        }
        if ((rc = run_back_end(ctx, ctx->si.as<float>(), ctx->sq.as<float>(), ctx->peak.as<float>(), r0, nr, g, back))) return rc;
    }
    if (side) {  // results are ready, in stream order, when this call's work on st completes
        CU(cudaEventRecord(ctx->ev_back, back));
        CU(cudaEventRecord(ctx->ev_join, back));
        CU(cudaStreamWaitEvent(st, ctx->ev_join, 0));
    }
    tally(ctx);
    return 0;
}

int ft8b200_process_raw(ft8b200_ctx_t *ctx, const uint8_t *d_iq, size_t bytes_per_stream, size_t stream_stride_bytes, int n_slots, void *stream) {
    return process_raw_impl(ctx, d_iq, bytes_per_stream, stream_stride_bytes, n_slots, 1, 0, stream);
}

int ft8b200_process_raw_streams(ft8b200_ctx_t *ctx, const uint8_t *d_iq, size_t bytes_per_stream, size_t stream_stride_bytes, int n_streams,
                                int slots_per_stream, size_t bytes_per_slot, void *stream) {
    return process_raw_impl(ctx, d_iq, bytes_per_stream, stream_stride_bytes, n_streams, slots_per_stream, bytes_per_slot, stream);
}

int ft8b200_process_slots(ft8b200_ctx_t *ctx, const float *d_i, const float *d_q, int n_slots, void *stream) {
    return ft8b200_process_conditioned(ctx, d_i, d_q, nullptr, n_slots, stream);
}

int ft8b200_process_conditioned(ft8b200_ctx_t *ctx, const float *d_i, const float *d_q, const float *d_peak, int n_slots, void *stream) {
    int rc = ctx_enter(ctx);
    if (rc) return rc;
    if (!d_i || !d_q || n_slots < 1) return fail(FT8B200_EINVAL, "ft8b200_process_slots: bad argument");
    // the waterfall kernel reads the samples with 16-byte cp.async (as ft8b200_waterfall requires): refused before anything is queued
    if ((((size_t)d_i) | ((size_t)d_q)) & 15) return fail(FT8B200_EINVAL, "ft8b200_process_slots: d_i and d_q must be 16-byte aligned");
    std::lock_guard<std::mutex> lk(ctx->mu);
    cudaStream_t st = pick(ctx, stream);
    if ((rc = ensure_slot_buffers(ctx, n_slots))) return rc;
    if ((rc = ensure_scratch(ctx, 2 * 2 * 36 * (256 - 7), n_slots))) return rc;
    clear_marks(ctx);
    rc = run_back_end(ctx, d_i, d_q, d_peak, 0, n_slots, 0, st);
    tally(ctx);
    return rc;
}

int ft8b200_set_profiling(ft8b200_ctx_t *ctx, int on) {
    if (!ctx) return fail(FT8B200_EINVAL, "null context");
    ctx->profiling = on != 0;
    return 0;
}

int ft8b200_set_overlap(ft8b200_ctx_t *ctx, int on) {
    if (!ctx) return fail(FT8B200_EINVAL, "null context");
    ctx->overlap = on;
    return 0;
}

int ft8b200_set_side_backend(ft8b200_ctx_t *ctx, int on) {
    if (!ctx) return fail(FT8B200_EINVAL, "null context");
    ctx->side_back = on != 0;
    if (!on) ctx->ev_front = nullptr;
    return 0;
}

int ft8b200_set_front_wait(ft8b200_ctx_t *ctx, void *cuda_event) {
    if (!ctx) return fail(FT8B200_EINVAL, "null context");
    ctx->front_wait = reinterpret_cast<cudaEvent_t>(cuda_event);
    return 0;
}

int ft8b200_set_back_wait(ft8b200_ctx_t *ctx, void *cuda_event) {
    if (!ctx) return fail(FT8B200_EINVAL, "null context");
    ctx->back_wait = reinterpret_cast<cudaEvent_t>(cuda_event);
    return 0;
}

void *ft8b200_back_event(ft8b200_ctx_t *ctx) { return ctx && ctx->side_back ? ctx->ev_back : nullptr; }

int ft8b200_set_comb_front(ft8b200_ctx_t *ctx, int on) {
    if (!ctx) return fail(FT8B200_EINVAL, "null context");
    ctx->comb_front = on != 0;
    return 0;
}

int ft8b200_set_partition_streams(ft8b200_ctx_t *ctx, void *front_stream, void *back_stream, int back_sm_count) {
    if (!ctx) return fail(FT8B200_EINVAL, "null context");
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->aux) cudaStreamSynchronize(ctx->aux);
    ctx->stream = front_stream ? reinterpret_cast<cudaStream_t>(front_stream) : ctx->own_stream;
    ctx->aux = back_stream ? reinterpret_cast<cudaStream_t>(back_stream) : ctx->own_aux;
    ctx->sm_back = back_stream ? back_sm_count : 0;
    return 0;
}

int ft8b200_set_protocol(ft8b200_ctx_t *ctx, int protocol) {
    if (!ctx || (protocol != PROTO_FT4 && protocol != PROTO_FT8)) return fail(FT8B200_EINVAL, "ft8b200_set_protocol: PROTO_FT4 or PROTO_FT8");
    ctx->protocol = protocol;
    return 0;
}

int ft8b200_set_decimator_variant(ft8b200_ctx_t *ctx, int variant) {
    if (!ctx || variant < 0 || variant > 6) return fail(FT8B200_EINVAL, "ft8b200_set_decimator_variant: bad argument");
    ctx->k1_variant = variant;
    return 0;
}

int ft8b200_set_decode_variant(int variant) {
    if (variant != 0 && variant != 1) return fail(FT8B200_EINVAL, "ft8b200_set_decode_variant: 0 (node-centred) or 1 (edge-centred)");
    set_decode_variant(variant);
    return 0;
}

int ft8b200_selfcheck_pade(ft8b200_ctx_t *ctx, uint64_t *counts5) {
    if (!ctx || !counts5) return fail(FT8B200_EINVAL, "ft8b200_selfcheck_pade: bad argument");
    unsigned long long c[5] = {0, 0, 0, 0, 0};
    if (int rc = ctx_enter(ctx)) return rc;
    cudaError_t e = run_pade_check(c, ctx->sm_count, ctx->stream);
    if (e != cudaSuccess) return cuda_fail(e, __func__);
    for (int k = 0; k < 5; ++k) counts5[k] = c[k];
    return 0;
}

int ft8b200_selfcheck_quantiser(ft8b200_ctx_t *ctx, uint64_t *counts3) {
    if (!ctx || !counts3) return fail(FT8B200_EINVAL, "ft8b200_selfcheck_quantiser: bad argument");
    if (int rc = ctx_enter(ctx)) return rc;
    unsigned long long c[3] = {0, 0, 0};
    cudaError_t e = run_quantiser_check(ctx->tb.db_thresholds, c, ctx->sm_count, ctx->stream);
    if (e != cudaSuccess) return cuda_fail(e, __func__);
    for (int k = 0; k < 3; ++k) counts3[k] = c[k];
    return 0;
}

int ft8b200_unpack77_batch(ft8b200_ctx_t *ctx, const uint8_t *h_payloads, int n, char *h_text32, int32_t *h_status) {
    int rc = ctx_enter(ctx);
    if (rc) return rc;
    if (!h_payloads || !h_text32 || !h_status || n < 1) return fail(FT8B200_EINVAL, "ft8b200_unpack77_batch: bad argument");
    std::lock_guard<std::mutex> lk(ctx->mu);
    uint8_t *d_in = nullptr;
    char *d_text = nullptr;
    int32_t *d_st = nullptr;
    cudaStream_t st = ctx->stream;
    cudaError_t e = cudaMallocAsync(reinterpret_cast<void **>(&d_in), (size_t)n * 10, st);
    if (e == cudaSuccess) e = cudaMallocAsync(reinterpret_cast<void **>(&d_text), (size_t)n * 32, st);
    if (e == cudaSuccess) e = cudaMallocAsync(reinterpret_cast<void **>(&d_st), (size_t)n * sizeof(int32_t), st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_in, h_payloads, (size_t)n * 10, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = launch_unpack77_batch(d_in, n, d_text, d_st, st, &ctx->launches);
    if (e == cudaSuccess) e = cudaMemcpyAsync(h_text32, d_text, (size_t)n * 32, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(h_status, d_st, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, st);
    if (d_in) cudaFreeAsync(d_in, st);
    if (d_text) cudaFreeAsync(d_text, st);
    if (d_st) cudaFreeAsync(d_st, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    tally(ctx);
    if (e != cudaSuccess) return cuda_fail(e, "ft8b200_unpack77_batch");
    return 0;
}

void *ft8b200_front_event(ft8b200_ctx_t *ctx) { return ctx ? ctx->ev_front : nullptr; }

// ms[0..5] = block sums, comb+FIR, waterfall, sync, decode, spots of the last process_* call, summed over its slot
// groups (-1 = stage not run).  With overlap on, front-end and back-end stages run concurrently: the sum of the stage
// times then exceeds the wall time of the call.  ms[6] (written only when n >= 7 and passes > 1): subtraction and the later passes.
int ft8b200_stage_times(ft8b200_ctx_t *ctx, float *ms, int n) {
    int rc = ctx_enter(ctx);
    if (rc) return rc;
    if (!ms || n < 6) return fail(FT8B200_EINVAL, "ft8b200_stage_times: need room for 6 floats");
    const int stages = (n >= 7 && ctx->passes > 1) ? 7 : 6;
    for (int k = 0; k < stages; ++k) {
        float total = 0.0f;
        bool any = false;
        for (int g = 0; g < kMaxGroups; ++g) {
            if (!ctx->ev_valid[k][g]) continue;
            float t = 0.0f;
            CU(cudaEventSynchronize(ctx->ev[k][g][1]));
            CU(cudaEventElapsedTime(&t, ctx->ev[k][g][0], ctx->ev[k][g][1]));
            total += t;
            any = true;
        }
        ms[k] = any ? total : -1.0f;
    }
    return 0;
}

// Timeline of the last process_* call: begin_ms[k] / end_ms[k] = device time of stage k's first start / last end mark,
// measured from `ref_event` (a timing-enabled cudaEvent_t recorded earlier by the caller); -1 = stage not run.
int ft8b200_stage_marks(ft8b200_ctx_t *ctx, void *ref_event, float *begin_ms, float *end_ms, int n) {
    int rc = ctx_enter(ctx);
    if (rc) return rc;
    if (!ref_event || !begin_ms || !end_ms || n < 6) return fail(FT8B200_EINVAL, "ft8b200_stage_marks: bad argument");
    cudaEvent_t ref = reinterpret_cast<cudaEvent_t>(ref_event);
    for (int k = 0; k < 6; ++k) {
        float b = -1.0f, e = -1.0f;
        for (int g = 0; g < kMaxGroups; ++g) {
            if (!ctx->ev_valid[k][g]) continue;
            float t0 = 0.0f, t1 = 0.0f;
            CU(cudaEventSynchronize(ctx->ev[k][g][1]));
            CU(cudaEventElapsedTime(&t0, ref, ctx->ev[k][g][0]));
            CU(cudaEventElapsedTime(&t1, ref, ctx->ev[k][g][1]));
            if (b < 0.0f || t0 < b) b = t0;
            if (t1 > e) e = t1;
        }
        begin_ms[k] = b;
        end_ms[k] = e;
    }
    return 0;
}

int ft8b200_results_device(ft8b200_ctx_t *ctx, struct decoder_results **d_results, int32_t **d_nresults) {
    if (!ctx) return fail(FT8B200_EINVAL, "null context");
    if (d_results) *d_results = ctx->results.as<struct decoder_results>();
    if (d_nresults) *d_nresults = ctx->nresults.as<int32_t>();
    return 0;
}

int ft8b200_fetch_results(ft8b200_ctx_t *ctx, int n_slots, struct decoder_results *h_results, int32_t *h_nresults, void *stream) {
    int rc = ctx_enter(ctx);
    if (rc) return rc;
    if (!h_results || !h_nresults || n_slots < 1) return fail(FT8B200_EINVAL, "ft8b200_fetch_results: bad argument");
    cudaStream_t st = pick(ctx, stream);
    const size_t M = (size_t)ctx->cfg.max_messages;
    if (ctx->results.bytes < (size_t)n_slots * M * sizeof(struct decoder_results)) return fail(FT8B200_EINVAL, "ft8b200_fetch_results: no such batch");
    CU(cudaMemcpyAsync(h_results, ctx->results.p, (size_t)n_slots * M * sizeof(struct decoder_results), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(h_nresults, ctx->nresults.p, (size_t)n_slots * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return 0;
}

int ft8b200_fetch_results_async(ft8b200_ctx_t *ctx, int n_slots, struct decoder_results *h_results, int32_t *h_nresults, void *stream) {
    int rc = ctx_enter(ctx);
    if (rc) return rc;
    if (!h_results || !h_nresults || n_slots < 1) return fail(FT8B200_EINVAL, "ft8b200_fetch_results_async: bad argument");
    cudaStream_t st = pick(ctx, stream);
    const size_t M = (size_t)ctx->cfg.max_messages;
    if (ctx->results.bytes < (size_t)n_slots * M * sizeof(struct decoder_results)) return fail(FT8B200_EINVAL, "ft8b200_fetch_results_async: no such batch");
    CU(cudaMemcpyAsync(h_results, ctx->results.p, (size_t)n_slots * M * sizeof(struct decoder_results), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(h_nresults, ctx->nresults.p, (size_t)n_slots * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    return 0;
}

int ft8b200_workspace(ft8b200_ctx_t *ctx, float **d_i, float **d_q, float **d_peak, uint8_t **d_mag, candidate_t **d_cand, int **d_ncand,
                      uint8_t **d_ok, decode_status_t **d_status, message_t **d_msg) {
    if (!ctx) return fail(FT8B200_EINVAL, "null context");
    if (d_i) *d_i = ctx->si.as<float>();
    if (d_q) *d_q = ctx->sq.as<float>();
    if (d_peak) *d_peak = ctx->peak.as<float>();
    if (d_mag) *d_mag = ctx->pass1.mag.as<uint8_t>();
    if (d_cand) *d_cand = ctx->pass1.cand.as<candidate_t>();
    if (d_ncand) *d_ncand = ctx->pass1.ncand.as<int>();
    if (d_ok) *d_ok = ctx->pass1.ok.as<uint8_t>();
    if (d_status) *d_status = ctx->pass1.status.as<decode_status_t>();
    if (d_msg) *d_msg = ctx->pass1.msg.as<message_t>();
    return 0;
}

int ft8b200_process_raw_host(ft8b200_ctx_t *ctx, const uint8_t *h_iq, size_t bytes_per_stream, int n_slots, struct decoder_results *h_results,
                             int32_t *h_nresults) {
    int rc = ctx_enter(ctx);
    if (rc) return rc;
    if (!h_iq || n_slots < 1 || (bytes_per_stream & 7)) return fail(FT8B200_EINVAL, "ft8b200_process_raw_host: bad argument");
    const size_t stride = (bytes_per_stream + 15) & ~(size_t)15;
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        if ((rc = ctx->raw.ensure(stride * n_slots + 16))) return rc;
    }
    if (stride == bytes_per_stream) {
        CU(cudaMemcpyAsync(ctx->raw.p, h_iq, bytes_per_stream * n_slots, cudaMemcpyHostToDevice, ctx->stream));
    } else {
        CU(cudaMemcpy2DAsync(ctx->raw.p, stride, h_iq, bytes_per_stream, bytes_per_stream, n_slots, cudaMemcpyHostToDevice, ctx->stream));
    }
    if ((rc = ft8b200_process_raw(ctx, ctx->raw.as<uint8_t>(), bytes_per_stream, stride, n_slots, nullptr))) return rc;
    return ft8b200_fetch_results(ctx, n_slots, h_results, h_nresults, nullptr);
}

int ft8b200_process_slots_host(ft8b200_ctx_t *ctx, const float *h_i, const float *h_q, int n_slots, struct decoder_results *h_results,
                               int32_t *h_nresults) {
    int rc = ctx_enter(ctx);
    if (rc) return rc;
    if (!h_i || !h_q || n_slots < 1) return fail(FT8B200_EINVAL, "ft8b200_process_slots_host: bad argument");
    const size_t bytes = (size_t)n_slots * kSlot * sizeof(float);
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        if ((rc = ctx->si.ensure(bytes))) return rc;
        if ((rc = ctx->sq.ensure(bytes))) return rc;
    }
    CU(cudaMemcpyAsync(ctx->si.p, h_i, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(ctx->sq.p, h_q, bytes, cudaMemcpyHostToDevice, ctx->stream));
    if ((rc = ft8b200_process_slots(ctx, ctx->si.as<float>(), ctx->sq.as<float>(), n_slots, nullptr))) return rc;
    return ft8b200_fetch_results(ctx, n_slots, h_results, h_nresults, nullptr);
}

}  // extern "C"
