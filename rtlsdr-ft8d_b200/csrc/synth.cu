// synth.cu -- device-side signal synthesis: the step BEFORE the path (SURVEY.md section 8f rank 3), so that benchmark and
// test inputs of any size are produced where they are consumed instead of on the host.
//   message -> 77-bit payload (host, ft8b200_pack77_std: the standard-message packer of ft8_lib/ft8/pack.c:20-232)
//   payload -> CRC-14 -> LDPC(174,91) parity -> Gray/Costas channel symbols   (device; ft8_encode / ft4_encode,
//              ft8_lib/ft8/encode.c:22-195)
//   symbols -> phase-continuous FSK + noise as
//                * raw RTL-SDR bytes: uint8 I/Q at 2.4 Msps, the tone sequence placed at (f - 600 kHz) so that the daemon's
//                  fs/4 mixer lands it at f (BASELINE configs #2, #5),
//                * complex baseband float at 3200 sps (what ft8_subsystem() consumes; configs #1, #3, #4),
//                * real float audio at 12 kHz (ft8_lib's monitor path; FT8 or FT4).
// The reference's own modulators (decoderSelfTest, rtlsdr_ft8d.c:937-955; gen_ft8.c:28-102) use rand() and libm per sample
// and cannot be reproduced bit for bit on another machine.  This generator is defined so that it CAN be: a 32-bit phase
// accumulator per signal (frequency words computed once on the host in double), a host-built cosine table, and noise from a
// counter hash (splitmix64 of seed/slot/sample index; sum of uniform bytes ~ Gaussian).  oracle/ft8_oracle_synth.c is its
// CPU twin; tests assert the two produce identical bytes / float bit patterns, and that the signals decode.
//
// GFSK (ft8b200_signal_t.reserved[0] = 1; gen_ft8.c:28-102): the frequency of symbol i is smoothed by the Gaussian pulse of
// gfsk_pulse() (three symbols long, BT = 2 for FT8, 1 for FT4), the first and last symbol are extended by a copy of themselves,
// and the first and last eighth of a symbol are ramped by a raised cosine.  The reference integrates the smoothed frequency
// sample by sample (phi += dphi[k]); here the pulse is an INTEGER table q[j] = round(pulse[j] * tone-spacing word) with prefix
// sums P[m], so that the phase of any sample is a closed form of at most three table entries --
//     phase(s L + j) = pstart[s] + j fw0 + t[s+1] P[j] + t[s] (P[j+L] - P[L]) + t[s-1] (P[j+2L] - P[2L]),   t[-1] = t[0], t[n] = t[n-1]
// -- every thread computes its own samples, and the CPU twin reproduces the waveform bit for bit.
#include "common.cuh"
#include "ft8_tables.h"

#include <math.h>
#include <string.h>

#include <mutex>
#include <vector>

using namespace ft8b200;

namespace {

constexpr int kMaxSym = 105;
constexpr int kLutBits = 12, kLut = 1 << kLutBits;  // 4096-entry cosine table

struct SigDev {
    long long s0;            // first sample of symbol 0
    uint32_t fw[8];          // frequency word of each tone: round(f / fs * 2^32), wraps for negative f
    uint32_t pstart[kMaxSym];  // phase at the first sample of every symbol
    float amp;               // linear amplitude (float paths)
    int32_t amp_q8;          // amplitude in LSB * 256 (raw path)
    int32_t n_sym;           // 79 (FT8) or 105 (FT4)
    uint8_t payload[10];
    uint8_t ft4;
    uint8_t gfsk;            // 0 = plain FSK (decoderSelfTest, rtlsdr_ft8d.c:937-955), 1 = GFSK (gen_ft8.c:49-102)
    uint8_t tones[kMaxSym];
};

// integer GFSK pulse of one layout (symbol length L): prefix sums P[0..3L], the raised-cosine ramp of L/8 samples
struct GfskDev {
    const uint32_t *P;
    const float *env_f;      // (1 - cosf(2 pi i / (2 n_ramp))) / 2
    const int32_t *env_q15;  // the same * 32768, rounded
    uint32_t p1, p2, p3;     // P[L], P[2L], P[3L]
};

__constant__ uint8_t c_gen[kLdpcM][12];   // the protocol tables of ft8_tables.h, uploaded by ensure_tables()
__constant__ uint8_t c_costas8[7], c_gray8[8], c_costas4[4][4], c_gray4[4], c_xor4[10];
__device__ float g_lut_f[kLut];     // (float)cos(2*pi*i/4096)
__device__ int16_t g_lut_q14[kLut]; // lround(16384*cos(2*pi*i/4096))

__host__ __device__ inline uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
__host__ __device__ inline uint64_t slot_key(uint64_t seed, int slot) { return splitmix64(seed + 0x632BE59BD9B4E019ull * (uint64_t)(slot + 1)); }
__host__ __device__ inline int byte_sum4(uint32_t w) { return (int)(w & 255u) + (int)((w >> 8) & 255u) + (int)((w >> 16) & 255u) + (int)(w >> 24); }

__device__ uint32_t crc14_dev(const uint8_t *msg, int num_bits) {  // ftx_compute_crc, crc.c:10-38
    uint32_t rem = 0;
    for (int b = 0, byte = 0; b < num_bits; ++b) {
        if ((b & 7) == 0) rem ^= ((uint32_t)msg[byte++] << 6);
        rem = (rem & 0x2000u) ? (((rem << 1) ^ 0x2757u) & 0xffffu) : ((rem << 1) & 0xffffu);
    }
    return rem & 0x3FFFu;
}

// one thread per signal: channel symbols + per-symbol start phases
__global__ void synth_prepare_kernel(SigDev *sigs, int n, int sym_len, GfskDev gf) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    SigDev &s = sigs[t];
    uint8_t a91[12];
    for (int k = 0; k < 10; ++k) a91[k] = s.payload[k] ^ (s.ft4 ? c_xor4[k] : 0);  // FT4 scrambles first (encode.c:131-136)
    a91[9] &= 0xF8; a91[10] = 0; a91[11] = 0;
    const uint32_t crc = crc14_dev(a91, 82);                                        // ftx_add_crc, crc.c:45-63
    a91[9] |= (uint8_t)(crc >> 11);
    a91[10] = (uint8_t)(crc >> 3);
    a91[11] = (uint8_t)(crc << 5);
    uint8_t bits[kLdpcN];
    for (int k = 0; k < kLdpcK; ++k) bits[k] = (a91[k >> 3] >> (7 - (k & 7))) & 1;
    for (int r = 0; r < kLdpcM; ++r) {                                              // encode174, encode.c:22-63
        int acc = 0;
        for (int b = 0; b < 12; ++b) acc ^= __popc((unsigned)(a91[b] & c_gen[r][b]));
        bits[kLdpcK + r] = (uint8_t)(acc & 1);
    }
    int k = 0;
    if (s.ft4) {
        s.n_sym = 105;
        for (int i = 0; i < 105; ++i) {
            uint8_t tone;
            if (i == 0 || i == 104) tone = 0;
            else if (i < 5) tone = c_costas4[0][i - 1];
            else if (i >= 34 && i < 38) tone = c_costas4[1][i - 34];
            else if (i >= 67 && i < 71) tone = c_costas4[2][i - 67];
            else if (i >= 100) tone = c_costas4[3][i - 100];
            else { tone = c_gray4[(bits[k] << 1) | bits[k + 1]]; k += 2; }
            s.tones[i] = tone;
        }
    } else {
        s.n_sym = 79;
        for (int i = 0; i < 79; ++i) {
            uint8_t tone;
            if (i < 7) tone = c_costas8[i];
            else if (i >= 36 && i < 43) tone = c_costas8[i - 36];
            else if (i >= 72) tone = c_costas8[i - 72];
            else { tone = c_gray8[(bits[k] << 2) | (bits[k + 1] << 1) | bits[k + 2]]; k += 3; }
            s.tones[i] = tone;
        }
    }
    uint32_t ph = 0;
    for (int i = 0; i < s.n_sym; ++i) {
        s.pstart[i] = ph;
        if (s.gfsk) {  // a symbol's worth of: tone 0, the tail of the previous pulse, the middle of this one, the head of the next
            const uint32_t tp = s.tones[i > 0 ? i - 1 : 0], tc = s.tones[i], tn = s.tones[i + 1 < s.n_sym ? i + 1 : i];
            ph += (uint32_t)sym_len * s.fw[0] + tn * gf.p1 + tc * (gf.p2 - gf.p1) + tp * (gf.p3 - gf.p2);
        } else {
            ph += (uint32_t)sym_len * s.fw[s.tones[i]];
        }
    }
}

// phase of signal `s` at sample n, or false when the signal is silent there; ramp = index into the GFSK envelope table or -1
template <int kSymLen>
__device__ __forceinline__ bool phase_at(const SigDev &s, long long n, const GfskDev &gf, uint32_t &ph, int &ramp) {
    const long long rel = n - s.s0;
    const long long total = (long long)s.n_sym * kSymLen;
    if (rel < 0 || rel >= total) return false;
    const int k = (int)(rel / kSymLen);
    const uint32_t j = (uint32_t)(rel - (long long)k * kSymLen);
    ramp = -1;
    if (s.gfsk) {
        const uint32_t tp = s.tones[k > 0 ? k - 1 : 0], tc = s.tones[k], tn = s.tones[k + 1 < s.n_sym ? k + 1 : k];
        ph = s.pstart[k] + j * s.fw[0] + tn * gf.P[j] + tc * (gf.P[j + kSymLen] - gf.p1) + tp * (gf.P[j + 2 * kSymLen] - gf.p2);
        constexpr int kRamp = kSymLen / 8;
        if (rel < kRamp) ramp = (int)rel;
        else if (rel >= total - kRamp) ramp = (int)(total - 1 - rel);
    } else {
        ph = s.pstart[k] + j * s.fw[s.tones[k]];
    }
    return true;
}

// raw RTL bytes: 8 complex samples (16 bytes) per thread
__global__ void __launch_bounds__(256)
synth_raw_kernel(const SigDev *__restrict__ sigs, const int *__restrict__ first, GfskDev gf, int noise_q8, uint64_t seed, int slot0,
                 uint8_t *__restrict__ out, size_t slot_stride, long long n_samples) {
    const int slot = blockIdx.y;
    const long long n0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 8;
    if (n0 >= n_samples) return;
    const uint64_t key = slot_key(seed, slot0 + slot);
    const int a = first[slot], b = first[slot + 1];
    uint32_t w[4] = {0, 0, 0, 0};
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        const long long n = n0 + u;
        int vi = 0, vq = 0;
        for (int g = a; g < b; ++g) {
            uint32_t ph;
            int ramp;
            if (!phase_at<384000>(sigs[g], n, gf, ph, ramp)) continue;
            const int idx = (int)(ph >> (32 - kLutBits));
            int amp = sigs[g].amp_q8;
            if (ramp >= 0) amp = (int)(((long long)amp * gf.env_q15[ramp] + 16384) >> 15);
            vi += (amp * (int)g_lut_q14[idx] + (1 << 21)) >> 22;                          // amp * cos
            vq += (amp * (int)g_lut_q14[(idx - kLut / 4) & (kLut - 1)] + (1 << 21)) >> 22;  // amp * sin
        }
        const uint64_t h = splitmix64(key + (uint64_t)n);
        const int ni = ((byte_sum4((uint32_t)h) - 510) * noise_q8 + (1 << 15)) >> 16;
        const int nq = ((byte_sum4((uint32_t)(h >> 32)) - 510) * noise_q8 + (1 << 15)) >> 16;
        int bi = 128 + vi + ni, bq = 128 + vq + nq;
        bi = bi < 0 ? 0 : (bi > 255 ? 255 : bi);
        bq = bq < 0 ? 0 : (bq > 255 ? 255 : bq);
        if (n < n_samples) w[u >> 1] |= ((uint32_t)bi | ((uint32_t)bq << 8)) << (16 * (u & 1));
    }
    uint8_t *dst = out + (size_t)slot * slot_stride + (size_t)n0 * 2;
    if (n0 + 8 <= n_samples) {
        *reinterpret_cast<uint4 *>(dst) = make_uint4(w[0], w[1], w[2], w[3]);
    } else {
        for (int u = 0; u < 8 && n0 + u < n_samples; ++u) {
            const uint32_t v = w[u >> 1] >> (16 * (u & 1));
            dst[2 * u] = (uint8_t)v;
            dst[2 * u + 1] = (uint8_t)(v >> 8);
        }
    }
}

// float paths: complex baseband (kComplex) or real audio; one sample per thread
template <int kSymLen, bool kComplex>
__global__ void __launch_bounds__(256)
synth_float_kernel(const SigDev *__restrict__ sigs, const int *__restrict__ first, GfskDev gf, float noise_scale, uint64_t seed, int slot0,
                   float *__restrict__ out_i, float *__restrict__ out_q, size_t slot_stride, int n_samples) {
    const int slot = blockIdx.y;
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= n_samples) return;
    const uint64_t key = slot_key(seed, slot0 + slot);
    // noise first (the host twin adds in the same order): (sum of 8 uniform bytes - 1020) * noise_scale per rail
    const uint64_t h0 = splitmix64(key + 2ull * (uint64_t)n);
    float vi = __fmul_rn((float)(byte_sum4((uint32_t)h0) + byte_sum4((uint32_t)(h0 >> 32)) - 1020), noise_scale);
    float vq = 0.0f;
    if (kComplex) {
        const uint64_t h1 = splitmix64(key + 2ull * (uint64_t)n + 1ull);
        vq = __fmul_rn((float)(byte_sum4((uint32_t)h1) + byte_sum4((uint32_t)(h1 >> 32)) - 1020), noise_scale);
    }
    for (int g = first[slot]; g < first[slot + 1]; ++g) {
        uint32_t ph;
        int ramp;
        if (!phase_at<kSymLen>(sigs[g], (long long)n, gf, ph, ramp)) continue;
        const int idx = (int)(ph >> (32 - kLutBits));
        const float amp = ramp >= 0 ? __fmul_rn(sigs[g].amp, gf.env_f[ramp]) : sigs[g].amp;
        vi = __fadd_rn(vi, __fmul_rn(amp, g_lut_f[idx]));
        if (kComplex) vq = __fadd_rn(vq, __fmul_rn(amp, g_lut_f[(idx - kLut / 4) & (kLut - 1)]));
    }
    out_i[(size_t)slot * slot_stride + n] = vi;
    if (kComplex) out_q[(size_t)slot * slot_stride + n] = vq;
}

bool g_tables_ready[64] = {};
cudaError_t ensure_tables() {
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    if (g_tables_ready[dev]) return cudaSuccess;
    static float lut_f[kLut];
    static int16_t lut_q[kLut];
    for (int i = 0; i < kLut; ++i) {
        const double c = cos(2.0 * M_PI * (double)i / (double)kLut);
        lut_f[i] = (float)c;
        lut_q[i] = (int16_t)lround(16384.0 * c);
    }
    cudaError_t e = cudaMemcpyToSymbol(g_lut_f, lut_f, sizeof(lut_f));
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(g_lut_q14, lut_q, sizeof(lut_q));
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(c_gen, kFt8tGen, sizeof(c_gen));
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(c_costas8, kFt8tCostas, sizeof(c_costas8));
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(c_gray8, kFt8tGray, sizeof(c_gray8));
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(c_costas4, kFt4tCostas, sizeof(c_costas4));
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(c_gray4, kFt4tGray, sizeof(c_gray4));
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(c_xor4, kFt4tXor, sizeof(c_xor4));
    if (e == cudaSuccess) g_tables_ready[dev] = true;
    return e;
}

// The integer GFSK pulse of one layout, per device.  pulse[j] is gfsk_pulse()'s own float expression (gen_ft8.c:28-38, erff of the
// host libm); q[j] = round(pulse[j] * step) with step = the tone spacing as a phase word; P = prefix sums (wrapping uint32).
struct GfskTab { uint32_t *d_P = nullptr; float *d_env_f = nullptr; int32_t *d_env_q = nullptr; uint32_t p1 = 0, p2 = 0, p3 = 0; bool ready = false; };
GfskTab g_gfsk[64][4];  // [device][layout: 0 raw, 1 3200 sps, 2 12 kHz FT8, 3 12 kHz FT4]

void build_gfsk_host(int L, float bt, uint32_t step, std::vector<uint32_t> &P, std::vector<float> &env_f, std::vector<int32_t> &env_q) {
    P.assign((size_t)3 * L + 1, 0u);
    uint32_t acc = 0;
    for (int j = 0; j < 3 * L; ++j) {
        const float t = j / (float)L - 1.5f;
        const float arg1 = 5.336446f * bt * (t + 0.5f), arg2 = 5.336446f * bt * (t - 0.5f);   // GFSK_CONST_K, gen_ft8.c:19
        const float pulse = (erff(arg1) - erff(arg2)) / 2;
        P[(size_t)j] = acc;
        acc += (uint32_t)llround((double)pulse * (double)step);
    }
    P[(size_t)3 * L] = acc;
    const int n_ramp = L / 8;
    env_f.resize((size_t)n_ramp);
    env_q.resize((size_t)n_ramp);
    for (int i = 0; i < n_ramp; ++i) {
        env_f[(size_t)i] = (1 - cosf(2 * (float)M_PI * i / (2 * n_ramp))) / 2;   // gen_ft8.c:96-101
        env_q[(size_t)i] = (int32_t)lround((double)env_f[(size_t)i] * 32768.0);
    }
}

struct Layout { double fs; int sym_len; double tone_hz; double f_shift; };
Layout layout_of(int kind, int protocol) {
    if (kind == 0) return {2400000.0, 384000, 6.25, -600000.0};                  // raw bytes (FT8 only)
    if (kind == 1) return {3200.0, 512, 6.25, 0.0};                              // 3200 sps complex (FT8 only)
    return protocol == PROTO_FT4 ? Layout{12000.0, 576, 1.0 / 0.048, 0.0} : Layout{12000.0, 1920, 6.25, 0.0};  // 12 kHz audio
}

// the GFSK tables of a layout on the current device (built and uploaded on first use; empty descriptor on failure)
std::mutex g_gfsk_mu;
GfskDev gfsk_tables(int kind, int protocol) {
    GfskDev out = {nullptr, nullptr, nullptr, 0, 0, 0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return out;
    const int slot = kind == 0 ? 0 : (kind == 1 ? 1 : (protocol == PROTO_FT4 ? 3 : 2));
    std::lock_guard<std::mutex> lk(g_gfsk_mu);
    GfskTab &t = g_gfsk[dev][slot];
    if (!t.ready) {
        const Layout L = layout_of(kind, protocol);
        const uint32_t step = (uint32_t)llround(L.tone_hz / L.fs * 4294967296.0);
        std::vector<uint32_t> P;
        std::vector<float> ef;
        std::vector<int32_t> eq;
        build_gfsk_host(L.sym_len, (kind == 2 && protocol == PROTO_FT4) ? 1.0f : 2.0f, step, P, ef, eq);   // FT8_SYMBOL_BT / FT4_SYMBOL_BT, gen_ft8.c:16-17
        const bool ok = cudaMalloc(&t.d_P, P.size() * sizeof(uint32_t)) == cudaSuccess && cudaMalloc(&t.d_env_f, ef.size() * sizeof(float)) == cudaSuccess &&
                        cudaMalloc(&t.d_env_q, eq.size() * sizeof(int32_t)) == cudaSuccess &&
                        cudaMemcpy(t.d_P, P.data(), P.size() * sizeof(uint32_t), cudaMemcpyHostToDevice) == cudaSuccess &&
                        cudaMemcpy(t.d_env_f, ef.data(), ef.size() * sizeof(float), cudaMemcpyHostToDevice) == cudaSuccess &&
                        cudaMemcpy(t.d_env_q, eq.data(), eq.size() * sizeof(int32_t), cudaMemcpyHostToDevice) == cudaSuccess;
        if (!ok) return out;
        t.p1 = P[(size_t)L.sym_len]; t.p2 = P[(size_t)2 * L.sym_len]; t.p3 = P[(size_t)3 * L.sym_len];
        t.ready = true;
    }
    out.P = t.d_P; out.env_f = t.d_env_f; out.env_q15 = t.d_env_q; out.p1 = t.p1; out.p2 = t.p2; out.p3 = t.p3;
    return out;
}

// host descriptors -> device descriptors (frequency words in double, once per signal), then the prepare kernel
int upload_signals(const ft8b200_signal_t *h_signals, const int *h_first, int n_slots, int kind, int protocol, SigDev **d_sigs, int **d_first,
                   GfskDev *gf_out, cudaStream_t st) {
    if (!h_signals && h_first[n_slots] > 0) return FT8B200_BAD_ARG();
    const int n = h_first[n_slots];
    const Layout L = layout_of(kind, protocol);
    bool any_gfsk = false;
    for (int g = 0; g < n; ++g) any_gfsk = any_gfsk || h_signals[g].reserved[0] != 0;
    GfskDev gf = {nullptr, nullptr, nullptr, 0, 0, 0};
    if (any_gfsk) {
        gf = gfsk_tables(kind, protocol);
        if (!gf.P) return FT8B200_ENOMEM;
    }
    if (gf_out) *gf_out = gf;
    std::vector<SigDev> host((size_t)(n > 0 ? n : 1));
    memset(host.data(), 0, host.size() * sizeof(SigDev));
    for (int g = 0; g < n; ++g) {
        const ft8b200_signal_t &s = h_signals[g];
        SigDev &d = host[(size_t)g];
        d.s0 = llround((double)s.t0_sec * L.fs);
        for (int t = 0; t < 8; ++t) {
            const double f = (double)s.f0_hz + t * L.tone_hz + L.f_shift;
            d.fw[t] = (uint32_t)(int64_t)llround(f / L.fs * 4294967296.0);
        }
        d.amp = s.amp;
        d.amp_q8 = (int32_t)lround((double)s.amp * 256.0);
        memcpy(d.payload, s.payload, 10);
        d.ft4 = (kind == 2 && protocol == PROTO_FT4) ? 1 : 0;
        d.gfsk = s.reserved[0] != 0 ? 1 : 0;
    }
    if (cudaMalloc(d_sigs, host.size() * sizeof(SigDev)) != cudaSuccess) return FT8B200_ENOMEM;
    if (cudaMalloc(d_first, sizeof(int) * (size_t)(n_slots + 1)) != cudaSuccess) { cudaFree(*d_sigs); return FT8B200_ENOMEM; }
    bool ok = ensure_tables() == cudaSuccess &&
              cudaMemcpyAsync(*d_sigs, host.data(), host.size() * sizeof(SigDev), cudaMemcpyHostToDevice, st) == cudaSuccess &&
              cudaMemcpyAsync(*d_first, h_first, sizeof(int) * (size_t)(n_slots + 1), cudaMemcpyHostToDevice, st) == cudaSuccess;
    if (ok && n > 0) {
        synth_prepare_kernel<<<(n + 127) / 128, 128, 0, st>>>(*d_sigs, n, L.sym_len, gf);
        ok = cudaGetLastError() == cudaSuccess;
    }
    // the pageable host vector must outlive the async copies
    ok = ok && cudaStreamSynchronize(st) == cudaSuccess;
    if (!ok) { cudaFree(*d_sigs); cudaFree(*d_first); return FT8B200_CUDA_FAIL(); }
    return 0;
}

bool check_first(const int *h_first, int n_slots) {
    if (!h_first || n_slots < 1 || h_first[0] != 0) return false;
    for (int s = 0; s < n_slots; ++s) if (h_first[s + 1] < h_first[s]) return false;
    return true;
}

}  // namespace

extern "C" {

// Standard (type 1) message: "<to> <de> <extra>", to/de = standard call signs or DE/QRZ/CQ, extra = grid (AA00), report
// (+NN/-NN/R+NN/R-NN), RRR, RR73, 73 or "".  ref: pack77_1 / pack28 / packgrid, ft8_lib/ft8/pack.c:20-232.
// Returns 0, or -1 if a field is not representable (non-standard call signs are out of scope here).
static int pack_call28(const char *call, uint32_t *out) {
    if (!strcmp(call, "DE")) { *out = 0; return 0; }
    if (!strcmp(call, "QRZ")) { *out = 1; return 0; }
    if (!strcmp(call, "CQ")) { *out = 2; return 0; }
    const size_t n = strlen(call);
    char c6[7] = "      ";
    if (n >= 3 && n <= 6 && call[2] >= '0' && call[2] <= '9') memcpy(c6, call, n);
    else if (n >= 2 && n <= 5 && call[1] >= '0' && call[1] <= '9') memcpy(c6 + 1, call, n);
    else return -1;
    static const char *A1 = " 0123456789ABCDEFGHIJKLMNOPQRSTUVWXYZ", *A2 = "0123456789ABCDEFGHIJKLMNOPQRSTUVWXYZ", *A3 = "0123456789",
                      *A4 = " ABCDEFGHIJKLMNOPQRSTUVWXYZ";
    const char *tabs[6] = {A1, A2, A3, A4, A4, A4};
    const int bases[6] = {37, 36, 10, 27, 27, 27};
    uint32_t v = 0;
    for (int k = 0; k < 6; ++k) {
        const char *p = strchr(tabs[k], c6[k]);
        if (!p || !c6[k]) return -1;
        v = v * (uint32_t)bases[k] + (uint32_t)(p - tabs[k]);
    }
    *out = 2063592u + 4194304u + v;
    return 0;
}

int ft8b200_pack77_std(const char *call_to, const char *call_de, const char *extra, uint8_t *payload10) {
    if (!call_to || !call_de || !extra || !payload10) return -1;
    uint32_t a, d, g;
    if (pack_call28(call_to, &a) || pack_call28(call_de, &d)) return -1;
    const size_t n = strlen(extra);
    if (n == 0) g = 32401;
    else if (!strcmp(extra, "RRR")) g = 32402;
    else if (!strcmp(extra, "RR73")) g = 32403;
    else if (!strcmp(extra, "73")) g = 32404;
    else if (n == 4 && extra[0] >= 'A' && extra[0] <= 'R' && extra[1] >= 'A' && extra[1] <= 'R' && extra[2] >= '0' && extra[2] <= '9' &&
             extra[3] >= '0' && extra[3] <= '9')
        g = (uint32_t)(((extra[0] - 'A') * 18 + (extra[1] - 'A')) * 100 + (extra[2] - '0') * 10 + (extra[3] - '0'));
    else {
        const bool r = extra[0] == 'R';
        char *end = nullptr;
        const long v = strtol(extra + (r ? 1 : 0), &end, 10);
        if (!end || *end || v < -35 || v > 99) return -1;
        g = (uint32_t)(32400 + 35 + v) | (r ? 0x8000u : 0u);
    }
    a <<= 1; d <<= 1; g &= 0xFFFFu;
    const uint32_t b[10] = {a >> 21, a >> 13, a >> 5, (a << 3) | (d >> 26), d >> 18, d >> 10, d >> 2, (d << 6) | (g >> 10), g >> 2, (g << 6) | (1u << 3)};
    for (int k = 0; k < 10; ++k) payload10[k] = (uint8_t)b[k];
    return 0;
}

// ---- pack77(): message text -> 77-bit payload, the whole of ft8_lib/ft8/pack.c:284-301 -------------------------------
// A standard message ("<call|DE|QRZ|CQ> <call> [grid | report | RRR | RR73 | 73]", pack77_1 :167-218) when both call fields
// pack, otherwise 13 characters of free text (packtext77 :220-282).  The reference's quirks are kept because they decide
// which bits go on the air: the third field is whatever follows the second blank ("FN20QI" packs as FN20; a field that is
// neither a grid nor a keyword goes through dd_to_int() unchecked), special tokens need their trailing blank, the 3DA0 and
// 3X prefix rewrites, and free text maps every character outside the 42-symbol alphabet (lower case included) to a blank.
namespace {

bool has_prefix(const char *s, const char *prefix) { return strncmp(s, prefix, strlen(prefix)) == 0; }
bool digit(char c) { return c >= '0' && c <= '9'; }
bool letter(char c) { return (c >= 'A' && c <= 'Z') || (c >= 'a' && c <= 'z'); }
int index_in(const char *alphabet, char c) {
    if (!c) return -1;
    const char *hit = strchr(alphabet, c);
    return hit ? (int)(hit - alphabet) : -1;
}

// pack28(), pack.c:22-98: `field` points INTO the message, the field ends at the next blank or at the end of the string
long field_to_n28(const char *field) {
    if (has_prefix(field, "DE ")) return 0;
    if (has_prefix(field, "QRZ ")) return 1;
    if (has_prefix(field, "CQ ")) return 2;
    int len = 0;
    while (field[len] && field[len] != ' ') ++len;
    auto at = [&](int k) { return k <= len ? field[k] : '\0'; };  // field[len] is the delimiter; nothing is read beyond it
    char c6[6] = {' ', ' ', ' ', ' ', ' ', ' '};
    if (has_prefix(field, "3DA0") && len <= 7) {          // Swaziland: 3DA0XYZ -> 3D0XYZ
        memcpy(c6, "3D0", 3);
        memcpy(c6 + 3, field + 4, (size_t)(len - 4));
    } else if (has_prefix(field, "3X") && letter(at(2)) && len <= 7) {  // Guinea: 3XA0XYZ -> QA0XYZ
        c6[0] = 'Q';
        memcpy(c6 + 1, field + 2, (size_t)(len - 2));
    } else if (digit(at(2)) && len <= 6) {
        memcpy(c6, field, (size_t)len);
    } else if (digit(at(1)) && len <= 5) {
        memcpy(c6 + 1, field, (size_t)len);
    }
    static const char *const alphabets[6] = {" 0123456789ABCDEFGHIJKLMNOPQRSTUVWXYZ", "0123456789ABCDEFGHIJKLMNOPQRSTUVWXYZ", "0123456789",
                                             " ABCDEFGHIJKLMNOPQRSTUVWXYZ", " ABCDEFGHIJKLMNOPQRSTUVWXYZ", " ABCDEFGHIJKLMNOPQRSTUVWXYZ"};
    static const long radix[6] = {37, 36, 10, 27, 27, 27};
    long n = 0;
    for (int k = 0; k < 6; ++k) {
        const int q = index_in(alphabets[k], c6[k]);
        if (q < 0) return -1;
        n = n * radix[k] + q;
    }
    return 2063592L + 4194304L + n;  // NTOKENS + MAX22 + n28
}

// dd_to_int(str, 3), text.c:103-131: optional sign, then digits while fewer than 3 characters have been consumed
int report_value(const char *s) {
    const bool neg = s[0] == '-';
    int k = (neg || s[0] == '+') ? 1 : 0, v = 0;
    for (; k < 3 && digit(s[k]); ++k) v = v * 10 + (s[k] - '0');
    return neg ? -v : v;
}

// packgrid(), pack.c:122-164: `rest` = everything after the second blank, or NULL when there is none
uint16_t third_field(const char *rest) {
    if (!rest) return 32401;
    if (!strcmp(rest, "RRR")) return 32402;
    if (!strcmp(rest, "RR73")) return 32403;
    if (!strcmp(rest, "73")) return 32404;
    if (rest[0] >= 'A' && rest[0] <= 'R' && rest[1] >= 'A' && rest[1] <= 'R' && digit(rest[2]) && digit(rest[3]))
        return (uint16_t)(((rest[0] - 'A') * 18 + (rest[1] - 'A')) * 100 + (rest[2] - '0') * 10 + (rest[3] - '0'));
    if (rest[0] == 'R') return (uint16_t)((32400 + (uint16_t)(35 + report_value(rest + 1))) | 0x8000);
    return (uint16_t)(32400 + (uint16_t)(35 + report_value(rest)));
}

}  // namespace

int ft8b200_pack77(const char *msg, uint8_t *payload10) {
    if (!msg || !payload10) return -1;
    const char *blank1 = strchr(msg, ' ');
    if (blank1) {
        const long a = field_to_n28(msg), d = field_to_n28(blank1 + 1);
        if (a >= 0 && d >= 0) {
            const char *blank2 = strchr(blank1 + 1, ' ');
            const uint32_t g = third_field(blank2 ? blank2 + 1 : nullptr);
            const uint32_t a29 = (uint32_t)a << 1, d29 = (uint32_t)d << 1;  // ipa = ipb = 0
            const uint32_t b[10] = {a29 >> 21, a29 >> 13, a29 >> 5, (a29 << 3) | (d29 >> 26), d29 >> 18, d29 >> 10, d29 >> 2, (d29 << 6) | (g >> 10), g >> 2,
                                    (g << 6) | (1u << 3)};  // i3 = 1
            for (int k = 0; k < 10; ++k) payload10[k] = (uint8_t)b[k];
            return 0;
        }
    }
    // free text, i3 = 0, n3 = 0: 13 base-42 digits as a 71-bit number, left-aligned in the first 72 bits
    while (*msg == ' ') ++msg;
    int len = (int)strlen(msg);
    while (len > 0 && msg[len - 1] == ' ') --len;
    unsigned __int128 v = 0;
    for (int k = 0; k < 13; ++k) {
        const int q = k < len ? index_in(" 0123456789ABCDEFGHIJKLMNOPQRSTUVWXYZ+-./?", msg[k]) : 0;
        v = v * 42 + (unsigned)(q > 0 ? q : 0);
    }
    v <<= 1;
    for (int k = 8; k >= 0; --k, v >>= 8) payload10[k] = (uint8_t)v;
    payload10[9] = 0;
    return 1;
}

// channel symbols of n payloads (10 bytes each) on the device: d_tones = n x 105 bytes (FT8 fills the first 79)
int ft8b200_encode_tones(ft8b200_ctx_t *ctx, const uint8_t *h_payloads, int n, int protocol, uint8_t *h_tones) {
    if (!ctx || !h_payloads || !h_tones || n < 1 || (protocol != PROTO_FT4 && protocol != PROTO_FT8)) return FT8B200_BAD_ARG();
    std::vector<ft8b200_signal_t> sig((size_t)n);
    std::vector<int> first((size_t)n + 1);
    memset(sig.data(), 0, sig.size() * sizeof(ft8b200_signal_t));
    for (int k = 0; k < n; ++k) { memcpy(sig[(size_t)k].payload, h_payloads + 10 * (size_t)k, 10); first[(size_t)k] = k; }
    first[(size_t)n] = n;
    if (cudaSetDevice(ctx_device(ctx)) != cudaSuccess) return FT8B200_CUDA_FAIL();  // tables (per device) and buffers belong to the context's device
    cudaStream_t st = (cudaStream_t)ft8b200_cuda_stream(ctx);
    SigDev *d_sigs = nullptr;
    int *d_first = nullptr;
    int rc = upload_signals(sig.data(), first.data(), n, 2, protocol, &d_sigs, &d_first, nullptr, st);
    if (rc) return rc;
    std::vector<SigDev> back((size_t)n);
    const bool ok = cudaMemcpy(back.data(), d_sigs, sizeof(SigDev) * (size_t)n, cudaMemcpyDeviceToHost) == cudaSuccess;
    cudaFree(d_sigs); cudaFree(d_first);
    if (!ok) return FT8B200_CUDA_FAIL();
    for (int k = 0; k < n; ++k) memcpy(h_tones + (size_t)k * kMaxSym, back[(size_t)k].tones, kMaxSym);
    return 0;
}

// h_first[s] .. h_first[s+1] = the signals of slot s (h_first has n_slots+1 entries, h_first[0] = 0).
// seed/first_slot_index select the noise: slot s uses the stream of slot index first_slot_index + s, so a batch generated
// in pieces (or on several GPUs) is identical to one generated at once.
int ft8b200_synth_raw(ft8b200_ctx_t *ctx, const ft8b200_signal_t *h_signals, const int *h_first, int n_slots, float noise_lsb, uint64_t seed,
                      int first_slot_index, uint8_t *d_iq, size_t slot_stride_bytes, size_t bytes_per_slot, void *stream) {
    if (!ctx || !d_iq || !check_first(h_first, n_slots) || (bytes_per_slot & 1) || slot_stride_bytes < bytes_per_slot || (slot_stride_bytes & 15) ||
        (((size_t)d_iq) & 15))
        return FT8B200_BAD_ARG();
    if (cudaSetDevice(ctx_device(ctx)) != cudaSuccess) return FT8B200_CUDA_FAIL();
    cudaStream_t st = stream ? (cudaStream_t)stream : (cudaStream_t)ft8b200_cuda_stream(ctx);
    SigDev *d_sigs = nullptr;
    int *d_first = nullptr;
    GfskDev gf;
    int rc = upload_signals(h_signals, h_first, n_slots, 0, PROTO_FT8, &d_sigs, &d_first, &gf, st);
    if (rc) return rc;
    const long long n_samples = (long long)(bytes_per_slot / 2);
    const int noise_q8 = (int)lround((double)noise_lsb * 65536.0 / 147.79715829474123);  // sigma of a sum of 4 uniform bytes
    bool ok = true;
    for (int s0 = 0; ok && s0 < n_slots; s0 += kMaxGridRows) {   // the slot is blockIdx.y
        const int rows = n_slots - s0 < kMaxGridRows ? n_slots - s0 : kMaxGridRows;
        dim3 grid((unsigned)((n_samples + 8 * 256 - 1) / (8 * 256)), (unsigned)rows);
        synth_raw_kernel<<<grid, 256, 0, st>>>(d_sigs, d_first + s0, gf, noise_q8, seed, first_slot_index + s0, d_iq + (size_t)s0 * slot_stride_bytes,
                                               slot_stride_bytes, n_samples);
        ok = cudaGetLastError() == cudaSuccess;
    }
    ok = ok && cudaStreamSynchronize(st) == cudaSuccess;
    cudaFree(d_sigs); cudaFree(d_first);
    return ok ? 0 : FT8B200_CUDA_FAIL();
}

// kind 1: complex baseband at 3200 sps (d_q != NULL, 48000 samples per slot typical); kind 2: real audio at 12 kHz
static int synth_float(ft8b200_ctx_t *ctx, int kind, int protocol, const ft8b200_signal_t *h_signals, const int *h_first, int n_slots,
                       float noise_sigma, uint64_t seed, int first_slot_index, float *d_i, float *d_q, size_t slot_stride, int n_samples, void *stream) {
    if (!ctx || !d_i || (kind == 1 && !d_q) || !check_first(h_first, n_slots) || n_samples < 1 || slot_stride < (size_t)n_samples) return FT8B200_BAD_ARG();
    if (cudaSetDevice(ctx_device(ctx)) != cudaSuccess) return FT8B200_CUDA_FAIL();
    cudaStream_t st = stream ? (cudaStream_t)stream : (cudaStream_t)ft8b200_cuda_stream(ctx);
    SigDev *d_sigs = nullptr;
    int *d_first = nullptr;
    GfskDev gf;
    int rc = upload_signals(h_signals, h_first, n_slots, kind, protocol, &d_sigs, &d_first, &gf, st);
    if (rc) return rc;
    const float scale = (float)((double)noise_sigma / 209.02153956946134);  // sigma of a sum of 8 uniform bytes
    bool ok = true;
    for (int s0 = 0; ok && s0 < n_slots; s0 += kMaxGridRows) {   // the slot is blockIdx.y
        const int rows = n_slots - s0 < kMaxGridRows ? n_slots - s0 : kMaxGridRows;
        dim3 grid((unsigned)((n_samples + 255) / 256), (unsigned)rows);
        const int *first = d_first + s0;
        float *oi = d_i + (size_t)s0 * slot_stride, *oq = d_q ? d_q + (size_t)s0 * slot_stride : nullptr;
        if (kind == 1) synth_float_kernel<512, true><<<grid, 256, 0, st>>>(d_sigs, first, gf, scale, seed, first_slot_index + s0, oi, oq, slot_stride, n_samples);
        else if (protocol == PROTO_FT4) synth_float_kernel<576, false><<<grid, 256, 0, st>>>(d_sigs, first, gf, scale, seed, first_slot_index + s0, oi, nullptr, slot_stride, n_samples);
        else synth_float_kernel<1920, false><<<grid, 256, 0, st>>>(d_sigs, first, gf, scale, seed, first_slot_index + s0, oi, nullptr, slot_stride, n_samples);
        ok = cudaGetLastError() == cudaSuccess;
    }
    ok = ok && cudaStreamSynchronize(st) == cudaSuccess;
    cudaFree(d_sigs); cudaFree(d_first);
    return ok ? 0 : FT8B200_CUDA_FAIL();
}

int ft8b200_synth_slots(ft8b200_ctx_t *ctx, const ft8b200_signal_t *h_signals, const int *h_first, int n_slots, float noise_sigma, uint64_t seed,
                        int first_slot_index, float *d_i, float *d_q, size_t slot_stride_samples, int n_samples, void *stream) {
    return synth_float(ctx, 1, PROTO_FT8, h_signals, h_first, n_slots, noise_sigma, seed, first_slot_index, d_i, d_q, slot_stride_samples, n_samples, stream);
}

int ft8b200_synth_audio(ft8b200_ctx_t *ctx, const ft8b200_signal_t *h_signals, const int *h_first, int n_slots, int protocol, float noise_sigma,
                        uint64_t seed, int first_slot_index, float *d_audio, size_t slot_stride_samples, int n_samples, void *stream) {
    if (protocol != PROTO_FT4 && protocol != PROTO_FT8) return FT8B200_BAD_ARG();
    return synth_float(ctx, 2, protocol, h_signals, h_first, n_slots, noise_sigma, seed, first_slot_index, d_audio, nullptr, slot_stride_samples, n_samples, stream);
}

}  // extern "C"
