// finesync.cu -- the front half of fine-sync decoding (DESIGN.md section 2.4.4, ft8b200_set_finesync, ft8b200_finesync): for every
// candidate that BP, OSD and AP left at stage 1 or 2, a (dt, df) search against the Costas arrays on the slot's 3200 sps samples and
// the symbol-synchronous spectra at the winner, turned into the reference's LLRs.  The back half (belief propagation and the gates)
// is rebp_kernel in decode.cu with nothing forced.  tests/finesync_ref.py is the float64 definition this kernel is held to.
//
// For a candidate with nominal start s0 and tone-0 frequency f0 (slot_search.cuh):
//   S(s, f) = sum over the 21 Costas symbols k of |sum_{m < 512} x[s + 512 k + m] exp(-2 pi i (f + 6.25 costas[k]) m / 3200)|^2
//   coarse: dt = -256, -240 ... +256 (33) x df = -8 ... +8 steps of 6.25/32 Hz (17), on sub-block sums (slot_search.cuh);
//   fine:   dt +- 8 samples at that df, exact; ties to the lower dt, then the lower df.
//   c[k][j] = sum_{m < 512} x[s* + 512 k + m] exp(-2 pi i (f* + 6.25 j) m / 3200), k < 79, j < 8; E = mean |c|^2;
//   v = 10 log10(|c|^2 / E + 1e-12), the max-log bit metrics of extract_llrs over v, normalised as a10 (scale sqrt(24 / var)).
// E = 0 (nothing of the span inside the slot, or a silent one) writes NaN LLRs: the back half then does not attempt the candidate.
// Deep mode (finesync_kernel<true>, DESIGN.md section 2.4.6, tests/finesync_deep_ref.py) also writes sets b and c, the nsym = 2 and 3
// coherent metrics: c'[k][j] = c[k][j] exp(-2 pi i f* 512 k / 3200) (one time origin for every symbol), and per group of g consecutive
// data symbols of a half A(b) = |sum_t c'[sym_t][gray[b_t]]| over the 8^g patterns, bit LLR = max A (bit 1) - max A (bit 0).
#include "common.cuh"
#include "ft8_tables.h"
#include "slot_search.cuh"

#include <math.h>

using namespace ft8b200;
using namespace ft8b200::slot_search;

namespace {

constexpr int kThreads = 256;
constexpr int kDtCoarse = 33, kCoarseStep = 16, kDtReach = 256;   // coarse dt = -256 ... +256
constexpr int kFine = 17;                                          // fine dt = coarse +- 8
constexpr int kCostasSyms = 21;
constexpr int kCoarsePoints = kDtCoarse * kDfPoints;               // 561
// Shared-memory layouts that keep a warp's accesses on distinct banks: the coarse stage's samples and tone carry one pad element per
// 8 (a lane per sub-block reads elements 8 apart), the rows of sub-block sums and rotations one per row of 64.
constexpr int kRow = kBlocks + 1;
constexpr int kCoarseSpan = kSym + 2 * kDtReach;                   // 1024 samples around a Costas symbol
__device__ __forceinline__ int pad8(int n) { return n + (n >> 3); }

__constant__ uint8_t c_costas[7], c_gray[8];

struct FsArgs {
    int n_slots, max_cand, on;
    const float *xi, *xq;            // slot s: xi + s * kSlot
    const candidate_t *cand; const int *ncand; const uint8_t *stage;
    float *llr;                      // [n_slots][max_cand][174]
    int32_t *grid;                   // [n_slots][max_cand][2]: dt samples, df steps
    const uint32_t *work; const unsigned int *work_total; unsigned int *next;
    float *llr_b, *llr_c;            // deep mode: sets b (nsym = 2) and c (nsym = 3), laid out as llr
};

// x[n] exp(-2 pi i f m / fs) needs the phase of f m / fs: formed in double, only its fractional cycle goes through sincospif
__device__ __forceinline__ float2 tone(double f_hz, int m) {
    const double cyc = f_hz / kFs * (double)m;
    float sn, cs;
    sincospif(2.0f * (float)(cyc - floor(cyc)), &sn, &cs);
    return make_float2(cs, sn);
}

__device__ __forceinline__ int costas_symbol(int q) { return q < 7 ? q : (q < 14 ? q + 29 : q + 58); }   // 0-6, 36-42, 72-78

// Deep mode, one group of G consecutive data symbols starting at symbol sym0, on one warp: lane l takes the patterns l, l + 32 ...
// (pattern p: symbol t carries Gray index (p >> 3 (G - 1 - t)) & 7, so bit q of the group is bit 3 G - 1 - q of p), keeps the
// largest A with each bit 1 and 0, and the warp takes the maxima of those (max is exact, so the result does not depend on the order).
// raw[q] = the group's unnormalised LLRs, written by lane 0.
template <int G>
__device__ __forceinline__ void group_llrs(const float2 *C, int sym0, int lane, float *raw) {
    float m1[3 * G], m0[3 * G];
#pragma unroll
    for (int q = 0; q < 3 * G; ++q) m1[q] = m0[q] = 0.0f;
    for (int p = lane; p < (1 << (3 * G)); p += 32) {
        float re = 0.0f, im = 0.0f;
#pragma unroll
        for (int t = 0; t < G; ++t) {
            const float2 z = C[(sym0 + t) * 8 + c_gray[(p >> (3 * (G - 1 - t))) & 7]];
            re += z.x;
            im += z.y;
        }
        const float A = sqrtf(re * re + im * im);
#pragma unroll
        for (int q = 0; q < 3 * G; ++q) {
            if ((p >> (3 * G - 1 - q)) & 1) m1[q] = fmaxf(m1[q], A);
            else m0[q] = fmaxf(m0[q], A);
        }
    }
#pragma unroll
    for (int q = 0; q < 3 * G; ++q) {   // A >= 0: its bit pattern orders as an unsigned integer
        const float hi = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(m1[q])));
        const float lo = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(m0[q])));
        if (lane == 0) raw[q] = hi - lo;
    }
}

// Deep mode: sets b and c of one candidate from the symbol-referenced spectra C [79][8] and the tone powers P (for E), the whole CTA.
// The groups of a half start at its first data symbol; the last takes what remains (nsym = 2: 14 pairs and a single, nsym = 3: 9
// triples and a pair).  The 30 + 20 groups go to the warps in turn, then warps 0 and 1 normalise sets b and c as set a is (a10).
__device__ void deep_sets(const FsArgs &a, size_t oidx, const float2 *C, const float *P, float *raw) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int task = warp; task < 50; task += kThreads / 32) {
        const int set = task < 30 ? 0 : 1, nsym = 2 + set, u = task - 30 * set, per = set ? 10 : 15;
        const int half = u / per, g = u - half * per;
        const int s = 29 * half + nsym * g, G = min(nsym, 29 - nsym * g);   // first data symbol of the group, its size
        const int sym0 = s + (s < 29 ? 7 : 14);
        float *out = raw + set * kLdpcN + 3 * s;
        if (G == 3) group_llrs<3>(C, sym0, lane, out);
        else if (G == 2) group_llrs<2>(C, sym0, lane, out);
        else group_llrs<1>(C, sym0, lane, out);
    }
    __syncthreads();
    if (warp < 2) {
        double e = 0.0;
        for (int q = lane; q < kNsym * 8; q += 32) e += (double)P[q];
        for (int o = 16; o > 0; o >>= 1) e += __shfl_xor_sync(0xffffffffu, e, o);
        const float *l = raw + warp * kLdpcN;
        double sum = 0.0, sum2 = 0.0;
        for (int i = lane; i < kLdpcN; i += 32) { sum += l[i]; sum2 += (double)l[i] * l[i]; }
        for (int o = 16; o > 0; o >>= 1) {
            sum += __shfl_xor_sync(0xffffffffu, sum, o);
            sum2 += __shfl_xor_sync(0xffffffffu, sum2, o);
        }
        const double var = (sum2 - sum * sum / 174.0) / 174.0;
        const double scale = sqrt(24.0 / var);
        float *dst = (warp ? a.llr_c : a.llr_b) + oidx * kLdpcN;
        for (int i = lane; i < kLdpcN; i += 32) dst[i] = e > 0.0 ? (float)(l[i] * scale) : __int_as_float(0x7fc00000);
    }
}

// one candidate, the whole CTA
template <bool kDeep>
__device__ void finesync_one(const FsArgs &a, size_t oidx, int slot, const float2 *w, float2 *xs, float2 *rs, float2 *bs, double *metric,
                             float *P, int *pick) {
    const int tid = threadIdx.x;
    const candidate_t cand = a.cand[oidx];
    const float *xi = a.xi + (size_t)slot * kSlot, *xq = a.xq + (size_t)slot * kSlot;
    const int s_nom = nominal_start(cand);
    const double f0 = nominal_f0(cand);

    // ---- coarse: 33 dt x 17 df, each thread owns up to three grid points and sums them over the 21 symbols in order
    double acc[3] = {0.0, 0.0, 0.0};
    for (int q = 0; q < kCostasSyms; ++q) {
        const int k = costas_symbol(q);
        const long long base = (long long)s_nom + (long long)kSym * k - kDtReach;
        const double fk = f0 + kToneHz * c_costas[q % 7];
        for (int i = tid; i < kCoarseSpan; i += blockDim.x) xs[pad8(i)] = load_x(xi, xq, base + i);
        for (int i = tid; i < kSym; i += blockDim.x) rs[pad8(i)] = tone(fk, i);
        __syncthreads();
        for (int p = tid; p < kDtCoarse * kBlocks; p += blockDim.x) {
            const int d = p / kBlocks, b = p - d * kBlocks;
            float2 s = make_float2(0.0f, 0.0f);
            for (int i = 0; i < kBlk; ++i) {
                const float2 z = cmul_conj(xs[pad8(d * kCoarseStep + kBlk * b + i)], rs[pad8(kBlk * b + i)]);
                s.x += z.x;
                s.y += z.y;
            }
            bs[d * kRow + b] = s;
        }
        __syncthreads();
        for (int u = 0; u < 3; ++u) {
            const int p = tid + u * blockDim.x;
            if (p >= kCoarsePoints) break;
            const int d = p / kDfPoints, f = p - d * kDfPoints;
            acc[u] += rotated_power(bs + d * kRow, w + f * kRow);
        }
        __syncthreads();
    }
    for (int u = 0; u < 3; ++u)
        if (tid + u * blockDim.x < kCoarsePoints) metric[tid + u * blockDim.x] = acc[u];
    __syncthreads();
    if (tid == 0) {
        const int best = pick_max(metric, kCoarsePoints);
        pick[0] = -kDtReach + kCoarseStep * (best / kDfPoints);
        pick[1] = best % kDfPoints - 8;
    }
    __syncthreads();
    const int dt_c = pick[0], df_i = pick[1];
    const double f = f0 + df_i * kDfStep;

    // ---- fine: dt_c - 8 ... dt_c + 8 at df, exact symbol sums (16 chunks of 32 samples x 17 dt, then the chunks in order)
    float2 *part = bs;
    double acc2 = 0.0;
    for (int q = 0; q < kCostasSyms; ++q) {
        const int k = costas_symbol(q);
        const long long base = (long long)s_nom + dt_c + (long long)kSym * k - 8;
        const double fk = f + kToneHz * c_costas[q % 7];
        for (int i = tid; i < kSym + 16; i += blockDim.x) xs[i] = load_x(xi, xq, base + i);
        for (int i = tid; i < kSym; i += blockDim.x) rs[i] = tone(fk, i);
        __syncthreads();
        for (int p = tid; p < kFine * 16; p += blockDim.x) {
            const int c = p / kFine, d = p - c * kFine;
            float2 s = make_float2(0.0f, 0.0f);
            for (int i = 0; i < 32; ++i) {
                const float2 z = cmul_conj(xs[d + 32 * c + i], rs[32 * c + i]);
                s.x += z.x;
                s.y += z.y;
            }
            part[p] = s;
        }
        __syncthreads();
        if (tid < kFine) {
            float re = 0.0f, im = 0.0f;
            for (int c = 0; c < 16; ++c) { re += part[c * kFine + tid].x; im += part[c * kFine + tid].y; }
            acc2 += (double)re * re + (double)im * im;
        }
        __syncthreads();
    }
    if (tid < kFine) metric[tid] = acc2;
    __syncthreads();
    if (tid == 0) {
        const int dt = dt_c + pick_max(metric, kFine) - 8;
        pick[0] = dt;
        int32_t *g = a.grid + oidx * 2;
        g[0] = dt;
        g[1] = df_i;
    }
    __syncthreads();

    // ---- spectra at s* = s0 + dt, f* = f: every symbol is downmixed by f* (rs), then 8 bins of a 512-point DFT (tw: 6.25 Hz = fs / 512)
    const long long s_star = (long long)s_nom + pick[0];
    float2 *tw = bs, *sp = bs + kSym;
    for (int i = tid; i < kSym; i += blockDim.x) {
        rs[i] = tone(f, i);
        double sn, cs;
        sincospi(2.0 * i / kSym, &sn, &cs);
        tw[i] = make_float2((float)cs, (float)sn);
    }
    const int j = tid >> 5, lane = tid & 31;   // 8 tones x 32 lanes, lane l sums samples l, l + 32 ... l + 480
    for (int k = 0; k < kNsym; ++k) {
        const long long base = s_star + (long long)kSym * k;
        __syncthreads();   // rs / tw written, and the previous symbol's xs and sp read
        for (int i = tid; i < kSym; i += blockDim.x) xs[i] = cmul_conj(load_x(xi, xq, base + i), rs[i]);
        __syncthreads();
        float2 s = make_float2(0.0f, 0.0f);
        for (int i = lane; i < kSym; i += 32) {
            const float2 z = cmul_conj(xs[i], tw[(j * i) & (kSym - 1)]);
            s.x += z.x;
            s.y += z.y;
        }
        sp[tid] = s;
        __syncthreads();
        if (tid < 8) {
            float re = 0.0f, im = 0.0f;
            for (int c = 0; c < 32; ++c) { re += sp[tid * 32 + c].x; im += sp[tid * 32 + c].y; }
            P[k * 8 + tid] = (float)((double)re * re + (double)im * im);
            if (kDeep) bs[kSym + 256 + k * 8 + tid] = cmul_conj(make_float2(re, im), tone(f, kSym * k));   // c'[k][tid]
        }
    }
    __syncthreads();

    // ---- LLRs (warp 0): v in dB against the mean power, the max-log metrics of extract_llrs, a10's normalisation
    if (tid < 32) {
        double e = 0.0;
        for (int q = lane; q < kNsym * 8; q += 32) e += (double)P[q];
        for (int o = 16; o > 0; o >>= 1) e += __shfl_xor_sync(0xffffffffu, e, o);   // butterfly: every lane the same sum
        e /= (double)(kNsym * 8);
        float *out = a.llr + oidx * kLdpcN;
        double l[2][3], sum = 0.0, sum2 = 0.0;
        for (int r = 0; r < 2; ++r) {
            const int s = lane + 32 * r;
            if (s >= 58) break;
            const int sym = s + (s < 29 ? 7 : 14);
            double v[8];
            for (int q = 0; q < 8; ++q) v[q] = 10.0 * log10((double)P[sym * 8 + c_gray[q]] / e + 1e-12);
            l[r][0] = fmax(fmax(v[4], v[5]), fmax(v[6], v[7])) - fmax(fmax(v[0], v[1]), fmax(v[2], v[3]));
            l[r][1] = fmax(fmax(v[2], v[3]), fmax(v[6], v[7])) - fmax(fmax(v[0], v[1]), fmax(v[4], v[5]));
            l[r][2] = fmax(fmax(v[1], v[3]), fmax(v[5], v[7])) - fmax(fmax(v[0], v[2]), fmax(v[4], v[6]));
            for (int i = 0; i < 3; ++i) { sum += l[r][i]; sum2 += l[r][i] * l[r][i]; }
        }
        for (int o = 16; o > 0; o >>= 1) {
            sum += __shfl_xor_sync(0xffffffffu, sum, o);
            sum2 += __shfl_xor_sync(0xffffffffu, sum2, o);
        }
        const double var = (sum2 - sum * sum / 174.0) / 174.0;
        const double scale = sqrt(24.0 / var);
        for (int r = 0; r < 2; ++r) {
            const int s = lane + 32 * r;
            if (s >= 58) break;
            for (int i = 0; i < 3; ++i) out[3 * s + i] = e > 0.0 ? (float)(l[r][i] * scale) : __int_as_float(0x7fc00000);
        }
    }
    // c' sits behind tw and sp in bs, the raw LLRs of sets b and c in metric: both dead by now
    if (kDeep) deep_sets(a, oidx, bs + kSym + 256, P, reinterpret_cast<float *>(metric));
}

// one CTA per candidate left at stage 1 or 2; a persistent grid whose CTAs pull entries from *a.next (zeroed by the caller)
template <bool kDeep>
__global__ void __launch_bounds__(kThreads) finesync_kernel(const FsArgs a) {
    __shared__ float2 w[kDfPoints * kRow];
    __shared__ float2 xs[kCoarseSpan + kCoarseSpan / 8];
    __shared__ float2 rs[kSym + kSym / 8];
    __shared__ float2 bs[kDtCoarse * kRow];
    __shared__ double metric[kCoarsePoints];
    __shared__ float P[kNsym * 8];
    __shared__ int pick[2];
    __shared__ unsigned int s_item;
    if (!a.on) return;
    fill_rotations(w, kRow);
    const unsigned int total = a.work ? *a.work_total : (unsigned int)a.n_slots * (unsigned int)a.max_cand;
    for (unsigned int item = blockIdx.x; item < total;) {
        const size_t oidx = a.work ? (size_t)a.work[item] : (size_t)item;   // list entries are slot * max_cand + candidate
        const int slot = (int)(oidx / (size_t)a.max_cand), c = (int)(oidx - (size_t)slot * a.max_cand);
        const int stage = a.stage[oidx];
        __syncthreads();   // the previous item's shared state is no longer read; w is written
        if (c < a.ncand[slot] && (stage == 1 || stage == 2)) finesync_one<kDeep>(a, oidx, slot, w, xs, rs, bs, metric, P, pick);
        if (threadIdx.x == 0) s_item = gridDim.x + atomicAdd(a.next, 1u);
        __syncthreads();
        item = s_item;
    }
}

// Deep mode: folds the flag / hard rows of the retries on the refined sets into the candidate's fs / fs_hard and fs_how.  Step i
// (0 ... 7: OSD and AP on set a, then BP, OSD and AP on set b and on set c) has its rows at flag / hard + i * n and ran when bit i of
// `steps` is set.  At most one step accepts (each runs only on what the ones before left at stage 1 or 2).
__global__ void finesync_merge_kernel(size_t n, unsigned int steps, const uint8_t *flag, const int32_t *hard, uint8_t *fs, int32_t *fs_hard,
                                      uint8_t *how) {
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
        uint8_t h = fs[e] == 2 ? 1 : 0;
        for (int i = 0; i < 8; ++i) {
            if (((steps >> i) & 1u) && flag[i * n + e] == 2) {
                fs[e] = 2;
                fs_hard[e] = hard[i * n + e];
                h = (uint8_t)(2 + i);
            }
        }
        how[e] = h;
    }
}

}  // namespace

namespace ft8b200 {

cudaError_t upload_finesync_tables() {
    cudaError_t e = cudaMemcpyToSymbol(c_costas, kFt8tCostas, sizeof(kFt8tCostas));
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(c_gray, kFt8tGray, sizeof(kFt8tGray));
    return e;
}

cudaError_t launch_finesync(int n_slots, int max_cand, int on, int deep, const float *d_xi, const float *d_xq, const candidate_t *d_cand,
                            const int *d_ncand, const uint8_t *d_stage, float *d_llr, float *d_llr_b, float *d_llr_c, int32_t *d_grid,
                            const uint32_t *d_work, const unsigned int *d_work_total, unsigned int *d_next, int sm_count, cudaStream_t st,
                            int *launches) {
    const FsArgs a = {n_slots, max_cand, on, d_xi, d_xq, d_cand, d_ncand, d_stage, d_llr, d_grid, d_work, d_work_total, d_next, d_llr_b, d_llr_c};
    // persistent grid, 4 CTAs per SM it may use; a CTA skips the entries at stage 3 or 4 and pulls the next
    size_t blocks = (size_t)n_slots * max_cand;
    if (sm_count > 0 && blocks > (size_t)(4 * sm_count)) blocks = (size_t)(4 * sm_count);
    if (deep) finesync_kernel<true><<<(unsigned)blocks, kThreads, 0, st>>>(a);
    else finesync_kernel<false><<<(unsigned)blocks, kThreads, 0, st>>>(a);
    ++*launches;
    return cudaGetLastError();
}

cudaError_t launch_finesync_merge(size_t n, unsigned int steps, const uint8_t *d_flag, const int32_t *d_hard, uint8_t *d_fs, int32_t *d_fs_hard,
                                  uint8_t *d_how, int sm_count, cudaStream_t st, int *launches) {
    size_t blocks = (n + 255) / 256;
    if (sm_count > 0 && blocks > (size_t)(8 * sm_count)) blocks = (size_t)(8 * sm_count);
    finesync_merge_kernel<<<(unsigned)blocks, 256, 0, st>>>(n, steps, d_flag, d_hard, d_fs, d_fs_hard, d_how);
    ++*launches;
    return cudaGetLastError();
}

}  // namespace ft8b200
