// slot_search.cuh -- the daemon slot's geometry and the (dt, df) search machinery shared by refine_kernel (subtract.cu: against a
// decoded message's GFSK waveform) and finesync_kernel (finesync.cu: against the Costas arrays alone).
#pragma once
#include "common.cuh"

namespace ft8b200 {
namespace slot_search {

constexpr int kSym = 512, kNsym = 79, kSpan = kSym * kNsym;   // 40448 samples
constexpr double kFs = 3200.0, kToneHz = 6.25;
constexpr int kDfPoints = 17;              // df = -8 ... +8 steps
constexpr double kDfStep = kToneHz / 32.0; // df step (Hz)
constexpr int kBlk = 8;                    // coarse stages: symbol sums are formed from sub-blocks of 8 samples
constexpr int kBlocks = kSym / kBlk;       // 64

// the candidate's nominal start sample and tone-0 frequency: the waterfall's 1024-point frames at hop 256 are 3.125 Hz wide, and a
// frame is centred on the symbol it scores (tests/subtract_ref.py nominal)
__device__ __forceinline__ int nominal_start(const candidate_t &c) { return kSym * c.time_offset + (kSym / 2) * c.time_sub + kSym / 2; }
__device__ __forceinline__ double nominal_f0(const candidate_t &c) { return 3.125 * (2 * c.freq_offset + c.freq_sub); }

// sample n of a slot, zero outside [0, kSlot)
__device__ __forceinline__ float2 load_x(const float *xi, const float *xq, long long n) {
    return (n >= 0 && n < kSlot) ? make_float2(xi[n], xq[n]) : make_float2(0.0f, 0.0f);
}

__device__ __forceinline__ float2 cmul_conj(float2 a, float2 b) {  // a * conj(b)
    return make_float2(a.x * b.x + a.y * b.y, a.y * b.x - a.x * b.y);
}

// Coarse stages: a symbol sum at df = 0 is formed from sub-block sums B_b over 8 samples, and the symbol sum at df is then
// sum_b B_b w_df[b] with w_df[b] = exp(-2 pi i df (8 b + 3.5) / fs).  Against the exact sum this drops each sub-block's own
// rotation exp(-2 pi i df (i - 3.5) / fs), |angle| <= 2 pi 1.5625 3.5 / 3200 = 0.0107 rad at the largest df.
// w: kDfPoints rows of kBlocks, row f at w + f * stride, filled by the whole CTA (no barrier here).
__device__ __forceinline__ void fill_rotations(float2 *w, int stride) {
    for (int q = threadIdx.x; q < kDfPoints * kBlocks; q += blockDim.x) {
        const int f = q / kBlocks, b = q - f * kBlocks;
        double sn, cs;
        sincospi(-2.0 * (f - 8) * kDfStep * (kBlk * b + 0.5 * (kBlk - 1)) / kFs, &sn, &cs);
        w[f * stride + b] = make_float2((float)cs, (float)sn);
    }
}

// |sum_b bs[b] w[b]|^2 over the kBlocks sub-blocks of one symbol, in a fixed order
__device__ __forceinline__ double rotated_power(const float2 *bs, const float2 *w) {
    float re = 0.0f, im = 0.0f;
    for (int b = 0; b < kBlocks; ++b) {
        const float2 a = bs[b], c = w[b];
        re += a.x * c.x - a.y * c.y;
        im += a.x * c.y + a.y * c.x;
    }
    return (double)re * re + (double)im * im;
}

// index of the largest of m[0, n): strict comparison, so ties keep the lower index (in C order of a (dt, df) array: the lower dt,
// then the lower df)
__device__ __forceinline__ int pick_max(const double *m, int n) {
    int best = 0;
    for (int p = 1; p < n; ++p)
        if (m[p] > m[best]) best = p;
    return best;
}

}  // namespace slot_search
}  // namespace ft8b200
