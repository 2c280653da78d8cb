// dropin.cu -- the reference's own entry points (names, signatures, struct layouts) implemented on
// top of the batched device API.  These take HOST pointers, exactly what the reference's callers pass:
//   ft8_subsystem()            rtlsdr_ft8d.c:1387-1524   (caller: decoder() :274, decodeRecordedFile :878, decoderSelfTest :961)
//   ft8_find_sync()/ft8_decode ft8_lib/ft8/decode.h:63,72 (callers: ft8_subsystem :1450,1476; decode_ft8.c:305,330)
//   initFFTW()/freeFFTW()      rtlsdr_ft8d.c:314-347
//   waterfall_init()/free()    ft8_lib/decode_ft8.c:63-79
// rtlsdr_callback() lives in streams.cu, monitor_*() in monitor.cu.
#include "common.cuh"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <string>
#include <vector>

using namespace ft8b200;

namespace ft8b200 {
ft8b200_ctx_t *default_ctx();
void default_ctx_release();
void default_stream_release();
void monitor_flush_for_mag(const uint8_t *mag);
}

namespace {
std::mutex g_mu;
ft8b200_ctx_t *g_ctx = nullptr;

// The per-candidate ft8_decode() call pattern is hostile to a GPU, so ft8_find_sync() decodes all the
// candidates it returns in the same visit and keeps the answers; ft8_decode() then only looks them up.
// The cache is keyed by the waterfall's geometry, its host pointer and a FINGERPRINT of its content: ft8_find_sync()
// reads every byte anyway (it copies them to the device) and takes the fingerprint then; each of the up to K ft8_decode()
// calls that follow re-takes it -- 1/16 of the bytes, in 64-byte pieces spread evenly over the buffer plus its last piece
// (6 KB of the daemon's 94 KB, 22 KB of the 12 kHz monitor's 357 KB) instead of re-hashing the whole waterfall per
// candidate.  A caller that rewrites the waterfall in place between the two calls (a new slot, another
// monitor_process() block) changes those pieces or the geometry and gets a fresh decode; FT8B200_DROPIN_FULL_HASH=1 in
// the environment hashes every byte on every call instead.
struct DecodeCache {
    bool valid = false;
    uint64_t key = 0;
    const uint8_t *host_ptr = nullptr;
    int iters = 0;
    int nb = 0, nbins = 0, tosr = 0, fosr = 0, proto = 1;
    std::vector<candidate_t> cand;
    std::vector<uint8_t> ok, stage;
    std::vector<decode_status_t> status;
    std::vector<message_t> msg;
} g_cache;

uint64_t hash_bytes(const uint8_t *p, size_t n) {
    uint64_t h0 = 0x9E3779B97F4A7C15ull, h1 = 0xC2B2AE3D27D4EB4Full, h2 = 0x165667B19E3779F9ull, h3 = 0x27D4EB2F165667C5ull;
    size_t k = 0;
    for (; k + 32 <= n; k += 32) {
        uint64_t w[4];
        memcpy(w, p + k, 32);
        h0 = (h0 ^ w[0]) * 0x100000001B3ull; h0 ^= h0 >> 29;
        h1 = (h1 ^ w[1]) * 0x100000001B3ull; h1 ^= h1 >> 31;
        h2 = (h2 ^ w[2]) * 0x100000001B3ull; h2 ^= h2 >> 27;
        h3 = (h3 ^ w[3]) * 0x100000001B3ull; h3 ^= h3 >> 33;
    }
    for (; k < n; ++k) { h0 = (h0 ^ p[k]) * 0x100000001B3ull; }
    uint64_t h = h0 ^ (h1 * 3) ^ (h2 * 5) ^ (h3 * 7) ^ (uint64_t)n;
    h ^= h >> 32; h *= 0xD6E8FEB86659FD93ull; h ^= h >> 32;
    return h;
}

bool full_hash_mode() {
    static const bool on = [] { const char *e = getenv("FT8B200_DROPIN_FULL_HASH"); return e && atoi(e) != 0; }();
    return on;
}
// content fingerprint: every 16th 64-byte piece and the last one (or every byte in full-hash mode / for small buffers)
uint64_t fingerprint(const uint8_t *p, size_t n) {
    if (full_hash_mode() || n < 4096) return hash_bytes(p, n);
    uint64_t h = 0x9E3779B97F4A7C15ull ^ (uint64_t)n;
    for (size_t o = 0; o + 64 <= n; o += 1024) h = (h ^ hash_bytes(p + o, 64)) * 0x100000001B3ull;
    return (h ^ hash_bytes(p + n - 64, 64)) * 0x100000001B3ull;
}

struct Scratch {  // device buffers of the drop-in calls (separate from the batched workspaces)
    uint8_t *mag = nullptr; size_t mag_bytes = 0;
    candidate_t *cand = nullptr; int *ncand = nullptr; uint8_t *ok = nullptr, *stage = nullptr;
    decode_status_t *status = nullptr; message_t *msg = nullptr; size_t k_alloc = 0;
} g_s;

bool ensure_scratch(size_t mag_bytes, size_t k) {
    if (mag_bytes > g_s.mag_bytes) {
        cudaFree(g_s.mag);
        if (cudaMalloc(&g_s.mag, mag_bytes + 16) != cudaSuccess) { g_s.mag = nullptr; g_s.mag_bytes = 0; return false; }
        g_s.mag_bytes = mag_bytes;
    }
    if (k > g_s.k_alloc) {
        cudaFree(g_s.cand); cudaFree(g_s.ncand); cudaFree(g_s.ok); cudaFree(g_s.stage); cudaFree(g_s.status); cudaFree(g_s.msg);
        bool okc = cudaMalloc(&g_s.cand, k * sizeof(candidate_t)) == cudaSuccess && cudaMalloc(&g_s.ncand, sizeof(int)) == cudaSuccess &&
                   cudaMalloc(&g_s.ok, k) == cudaSuccess && cudaMalloc(&g_s.stage, k) == cudaSuccess &&
                   cudaMalloc(&g_s.status, k * sizeof(decode_status_t)) == cudaSuccess && cudaMalloc(&g_s.msg, k * sizeof(message_t)) == cudaSuccess;
        if (!okc) { g_s.k_alloc = 0; return false; }
        g_s.k_alloc = k;
    }
    return true;
}

void die(const char *where) {
    // The reference's entry points have no error channel; a GPU failure here must not look like "no decodes".
    fprintf(stderr, "libft8b200: %s failed: %s\n", where, ft8b200_last_error());
    abort();
}

// <name>=<0 or 1> and <name>_MAX_HARD=<cap> switch a decoder and cap its hard distance; anything but an integer, a switch other
// than 0 or 1, or a cap above 174 stops the program
void set_from_env(ft8b200_ctx_t *ctx, const char *name, int (*set)(ft8b200_ctx_t *, int, int)) {
    const std::string cap_name = std::string(name) + "_MAX_HARD";
    const char *v = getenv(name), *cap = getenv(cap_name.c_str());
    if (!v) return;
    char *end = nullptr, *cap_end = nullptr;
    const long on = strtol(v, &end, 10), c = cap ? strtol(cap, &cap_end, 10) : -1;
    if (!*v || *end || (cap && (!*cap || *cap_end)) || on < 0 || on > 1 || c > 174 || set(ctx, (int)on, (int)c) != 0)
        die((std::string(name) + " (0 or 1) / " + cap_name + " (an integer up to 174; negative = the default)").c_str());
}
}  // namespace

namespace ft8b200 {
ft8b200_ctx_t *default_ctx() {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!g_ctx) {
        ft8b200_config_t cfg;
        ft8b200_default_config(&cfg);
        const char *dev = getenv("FT8B200_DEVICE");
        if (dev) cfg.device = atoi(dev);
        g_ctx = ft8b200_create(&cfg);
        if (!g_ctx) die("ft8b200_create (default context)");
        // deeper decoding for a relinked program without code changes: FT8B200_OSD=<order>, FT8B200_OSD_MAX_HARD=<cap> (INTEGRATION.md)
        const char *osd = getenv("FT8B200_OSD"), *cap = getenv("FT8B200_OSD_MAX_HARD");
        if (osd && ft8b200_set_osd(g_ctx, atoi(osd), cap ? atoi(cap) : -1) != 0) die("FT8B200_OSD (0, 1 or 2)");
        // a-priori decoding of CQ calls, fine-sync decoding and its deep mode (INTEGRATION.md)
        set_from_env(g_ctx, "FT8B200_AP", ft8b200_set_ap);
        set_from_env(g_ctx, "FT8B200_FINESYNC", ft8b200_set_finesync);
        set_from_env(g_ctx, "FT8B200_FINESYNC_DEEP", ft8b200_set_finesync_deep);
        // multi-pass decoding with signal subtraction: FT8B200_PASSES=<1, 2 or 3>
        const char *passes = getenv("FT8B200_PASSES");
        if (passes && ft8b200_set_passes(g_ctx, atoi(passes)) != 0) die("FT8B200_PASSES (1, 2 or 3)");
    }
    return g_ctx;
}
void default_ctx_release() {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_ctx) {
        cudaFree(g_s.mag); cudaFree(g_s.cand); cudaFree(g_s.ncand); cudaFree(g_s.ok); cudaFree(g_s.stage); cudaFree(g_s.status); cudaFree(g_s.msg);
        g_s = Scratch();
        g_cache = DecodeCache();
        ft8b200_destroy(g_ctx);
        g_ctx = nullptr;
    }
}
}  // namespace ft8b200

extern "C" {

void initFFTW(void) { (void)default_ctx(); }
void freeFFTW(void) { default_stream_release(); default_ctx_release(); }

void ft8_subsystem(float *iSamples, float *qSamples, uint32_t samples_len, struct decoder_results *decodes, int32_t *n_results) {
    (void)samples_len;  // the reference ignores it too (rtlsdr_ft8d.c:1393)
    ft8b200_ctx_t *ctx = default_ctx();
    ft8b200_config_t cfg;
    ft8b200_default_config(&cfg);
    std::vector<struct decoder_results> tmp((size_t)cfg.max_messages);
    int32_t n = 0;
    if (ft8b200_process_slots_host(ctx, iSamples, qSamples, 1, tmp.data(), &n) != 0) die("ft8_subsystem");
    // The reference writes decodes[k] only for "CQ ..." messages and leaves the other slots as they were
    // (rtlsdr_ft8d.c:1509-1520); the kernel marks written records with a non-empty call.
    for (int k = 0; k < n && k < cfg.max_messages; ++k)
        if (tmp[(size_t)k].call[0]) decodes[k] = tmp[(size_t)k];
    *n_results = n;
}

int ft8_find_sync(const waterfall_t *power, int num_candidates, candidate_t heap[], int min_score) {
    ft8b200_ctx_t *ctx = default_ctx();
    if (power->protocol != PROTO_FT8 && power->protocol != PROTO_FT4) {
        fprintf(stderr, "libft8b200: ft8_find_sync: unknown protocol %d\n", (int)power->protocol);
        abort();
    }
    if (num_candidates <= 0) return 0;
    if (power->num_bins < 8) return 0;   // the reference's `freq_offset + 7 < num_bins` loop never runs (decode.c:189)
    monitor_flush_for_mag(power->mag);   // a deferred monitor (ft8b200_monitor_set_deferred) transforms its pending blocks now
    std::lock_guard<std::mutex> lk(g_mu);
    if (cudaSetDevice(ctx_device(ctx)) != cudaSuccess) die("ft8_find_sync (cudaSetDevice)");  // the decoder thread's current device may differ
    const size_t bytes = (size_t)power->num_blocks * power->block_stride;
    if (!ensure_scratch(bytes, (size_t)num_candidates)) die("ft8_find_sync (device allocation)");
    cudaStream_t st = (cudaStream_t)ft8b200_cuda_stream(ctx);
    if (cudaMemcpyAsync(g_s.mag, power->mag, bytes, cudaMemcpyHostToDevice, st) != cudaSuccess) die("ft8_find_sync (H2D)");
    // a private context view with the caller's K / min_score
    int launches = 0;
    const int npos = power->time_osr * power->freq_osr * 36 * (power->num_bins - 7);
    static uint32_t *lists = nullptr;   // survivor list of the one slot (score kernel -> selection)
    static int16_t *scores = nullptr;
    static int scratch_npos = 0;
    if (!lists && (cudaMalloc(&lists, find_sync_list_bytes(1)) != cudaSuccess || cudaMemset(lists, 0, find_sync_list_bytes(1)) != cudaSuccess ||
                   cudaStreamSynchronize(0) != cudaSuccess)) die("ft8_find_sync (scratch)");   // zeroed: the selection reads a slot's first words ahead of its count
    if (npos > scratch_npos) {
        cudaFree(scores);
        if (cudaMalloc(&scores, (size_t)npos * sizeof(int16_t)) != cudaSuccess) die("ft8_find_sync (scratch)");
        scratch_npos = npos;
    }
    if (launch_find_sync(g_s.mag, bytes, 1, power->num_blocks, power->num_bins, power->time_osr, power->freq_osr, (int)power->protocol, num_candidates, min_score,
                         g_s.cand, g_s.ncand, scores, lists, nullptr, nullptr, ctx_sm_count(ctx), st, &launches) != cudaSuccess) die("ft8_find_sync (kernel)");
    // decode everything now; ft8_decode() will look the answers up
    ft8b200_config_t cfg;
    ft8b200_default_config(&cfg);
    if (launch_decode(g_s.mag, bytes, 1, power->num_blocks, power->num_bins, power->time_osr, power->freq_osr, (int)power->protocol, num_candidates, cfg.ldpc_iterations,
                      g_s.cand, g_s.ncand, g_s.ok, g_s.stage, g_s.status, g_s.msg, nullptr, nullptr, nullptr, nullptr, ctx_sm_count(ctx), st, &launches) != cudaSuccess)
        die("ft8_find_sync (decode kernel)");
    int n = 0;
    g_cache.cand.resize((size_t)num_candidates); g_cache.ok.resize((size_t)num_candidates); g_cache.stage.resize((size_t)num_candidates);
    g_cache.status.resize((size_t)num_candidates); g_cache.msg.resize((size_t)num_candidates);
    bool okc = cudaMemcpyAsync(&n, g_s.ncand, sizeof(int), cudaMemcpyDeviceToHost, st) == cudaSuccess &&
               cudaMemcpyAsync(g_cache.cand.data(), g_s.cand, sizeof(candidate_t) * num_candidates, cudaMemcpyDeviceToHost, st) == cudaSuccess &&
               cudaMemcpyAsync(g_cache.ok.data(), g_s.ok, (size_t)num_candidates, cudaMemcpyDeviceToHost, st) == cudaSuccess &&
               cudaMemcpyAsync(g_cache.stage.data(), g_s.stage, (size_t)num_candidates, cudaMemcpyDeviceToHost, st) == cudaSuccess &&
               cudaMemcpyAsync(g_cache.status.data(), g_s.status, sizeof(decode_status_t) * num_candidates, cudaMemcpyDeviceToHost, st) == cudaSuccess &&
               cudaMemcpyAsync(g_cache.msg.data(), g_s.msg, sizeof(message_t) * num_candidates, cudaMemcpyDeviceToHost, st) == cudaSuccess &&
               cudaStreamSynchronize(st) == cudaSuccess;
    if (!okc) die("ft8_find_sync (D2H)");
    g_cache.cand.resize((size_t)n); g_cache.ok.resize((size_t)n); g_cache.stage.resize((size_t)n);
    g_cache.status.resize((size_t)n); g_cache.msg.resize((size_t)n);
    g_cache.key = fingerprint(power->mag, bytes);
    g_cache.host_ptr = power->mag;
    g_cache.iters = cfg.ldpc_iterations;
    g_cache.nb = power->num_blocks; g_cache.nbins = power->num_bins; g_cache.tosr = power->time_osr; g_cache.fosr = power->freq_osr;
    g_cache.proto = (int)power->protocol;
    g_cache.valid = true;
    memcpy(heap, g_cache.cand.data(), sizeof(candidate_t) * (size_t)n);
    return n;
}

static void write_status(decode_status_t *status, const decode_status_t &s, int stage) {
    // the reference fills the fields progressively and returns early (decode.c:329-369)
    status->ldpc_errors = s.ldpc_errors;
    if (stage >= 2) { status->crc_extracted = s.crc_extracted; status->crc_calculated = s.crc_calculated; }
    if (stage >= 3) status->unpack_status = s.unpack_status;
}

bool ft8_decode(const waterfall_t *power, const candidate_t *cand, message_t *message, int max_iterations, decode_status_t *status) {
    ft8b200_ctx_t *ctx = default_ctx();
    if (power->protocol != PROTO_FT8 && power->protocol != PROTO_FT4) {
        fprintf(stderr, "libft8b200: ft8_decode: unknown protocol %d\n", (int)power->protocol);
        abort();
    }
    monitor_flush_for_mag(power->mag);
    std::lock_guard<std::mutex> lk(g_mu);
    if (cudaSetDevice(ctx_device(ctx)) != cudaSuccess) die("ft8_decode (cudaSetDevice)");
    const size_t bytes = (size_t)power->num_blocks * power->block_stride;
    if (g_cache.valid && g_cache.host_ptr == power->mag && g_cache.iters == max_iterations && g_cache.nb == power->num_blocks &&
        g_cache.nbins == power->num_bins && g_cache.tosr == power->time_osr && g_cache.fosr == power->freq_osr && g_cache.proto == (int)power->protocol &&
        g_cache.key == fingerprint(power->mag, bytes)) {
        for (size_t k = 0; k < g_cache.cand.size(); ++k) {
            if (memcmp(&g_cache.cand[k], cand, sizeof(candidate_t)) == 0) {
                write_status(status, g_cache.status[k], g_cache.stage[k]);
                if (g_cache.ok[k]) { *message = g_cache.msg[k]; return true; }
                return false;
            }
        }
    }
    // not cached: decode this one candidate
    if (!ensure_scratch(bytes, 1)) die("ft8_decode (device allocation)");
    cudaStream_t st = (cudaStream_t)ft8b200_cuda_stream(ctx);
    int launches = 0, one = 1;
    uint8_t okv = 0, stage = 0;
    decode_status_t s;
    message_t m;
    bool okc = cudaMemcpyAsync(g_s.mag, power->mag, bytes, cudaMemcpyHostToDevice, st) == cudaSuccess &&
               cudaMemcpyAsync(g_s.cand, cand, sizeof(candidate_t), cudaMemcpyHostToDevice, st) == cudaSuccess &&
               cudaMemcpyAsync(g_s.ncand, &one, sizeof(int), cudaMemcpyHostToDevice, st) == cudaSuccess &&
               launch_decode(g_s.mag, bytes, 1, power->num_blocks, power->num_bins, power->time_osr, power->freq_osr, (int)power->protocol, 1, max_iterations, g_s.cand,
                             g_s.ncand, g_s.ok, g_s.stage, g_s.status, g_s.msg, nullptr, nullptr, nullptr, nullptr, ctx_sm_count(ctx), st, &launches) == cudaSuccess &&
               cudaMemcpyAsync(&okv, g_s.ok, 1, cudaMemcpyDeviceToHost, st) == cudaSuccess &&
               cudaMemcpyAsync(&stage, g_s.stage, 1, cudaMemcpyDeviceToHost, st) == cudaSuccess &&
               cudaMemcpyAsync(&s, g_s.status, sizeof(s), cudaMemcpyDeviceToHost, st) == cudaSuccess &&
               cudaMemcpyAsync(&m, g_s.msg, sizeof(m), cudaMemcpyDeviceToHost, st) == cudaSuccess && cudaStreamSynchronize(st) == cudaSuccess;
    if (!okc) die("ft8_decode");
    g_cache.valid = false;  // the device copy of the waterfall changed
    write_status(status, s, stage);
    if (okv) { *message = m; return true; }
    return false;
}

void waterfall_init(waterfall_t *me, int max_blocks, int num_bins, int time_osr, int freq_osr) {
    const size_t mag_size = (size_t)max_blocks * time_osr * freq_osr * num_bins;
    me->max_blocks = max_blocks;
    me->num_blocks = 0;
    me->num_bins = num_bins;
    me->time_osr = time_osr;
    me->freq_osr = freq_osr;
    me->block_stride = time_osr * freq_osr * num_bins;
    me->mag = (uint8_t *)malloc(mag_size);
}

void waterfall_free(waterfall_t *me) { free(me->mag); me->mag = nullptr; }

}  // extern "C"
