// subtract.cu -- signal subtraction for multi-pass decoding on the daemon path (DESIGN.md section 2.4.2, ft8b200_set_passes,
// ft8b200_subtract).  tests/subtract_ref.py is the float64 definition these kernels are held to.
//
// For every decoded message of a slot: the 79 channel tones of its codeword (Costas arrays + Gray map), its nominal start sample
// s0 = 512 time_offset + 256 time_sub + 256 and tone-0 frequency f0 = 3.125 (2 freq_offset + freq_sub) Hz (the waterfall's
// framing: 1024-point frames at hop 256 whose centre meets the symbol's centre), and the unit-amplitude GFSK waveform r gen_ft8
// sends (BT = 2, extended end symbols, raised-cosine ramps, 6.25 Hz spacing, 512 samples a symbol) starting at s0 + dt with
// tone 0 at f0 + df.
//   refine_kernel (one CTA per message): maximise M = sum_k |sum_{n in symbol k} x[n] conj(r[n])|^2 over dt = -128, -112 ... 128
//       x df = -8 ... 8 steps of 6.25/32 Hz, then over dt +- 8 samples at that df; ties to the lower dt, then the lower df.
//   subtract_kernel (one CTA per slot, messages in list order): c = y conj(r) over the signal's span, a = c smoothed by a
//       1025-tap Hann window normalised by the taps inside the span, y -= a r.
// The phase of r is formed in double (closed form of the integrated GFSK pulse, as synth.cu does in integers) and only its
// fractional cycle goes through sincospif: the synthesiser's 4096-entry cosine table would leave 1.5e-3 of the signal behind.
#include "common.cuh"
#include "ft8_tables.h"
#include "slot_search.cuh"

#include <math.h>

using namespace ft8b200;

namespace {

using namespace ft8b200::slot_search;
constexpr int kGrid = kDfPoints;           // points per axis of every search stage
constexpr int kCoarseStep = 16;            // coarse dt step (samples); the coarse dt grid is -128 ... +128
constexpr int kHalfWin = 512;              // smoothing window: 1025 taps, h[k] = cos^2(pi k / 1026), |k| <= 512
constexpr double kWinW = 2.0 * 3.14159265358979323846 / 1026.0;
constexpr int kChunk = 2048;               // smoothing: outputs per chunk; its halo of 2 x 512 samples is scanned with it
constexpr int kHalo = kChunk + 2 * kHalfWin;
constexpr int kRefineThreads = 256, kSubThreads = 512;

__constant__ uint8_t c_costas[7], c_gray[8];
__device__ double g_pd[3 * kSym + 1];      // prefix sums of gfsk_pulse (BT = 2): g_pd[j] = sum_{i < j} pulse[i]

// per-message state shared by both kernels
struct MsgShared {
    uint8_t tones[kNsym];
    double pst[kNsym];   // integrated pulse (tone units) at the first sample of every symbol
};

__device__ void load_message(MsgShared &ms, const uint8_t *cw) {
    const int t = threadIdx.x;
    if (t < kNsym) {
        uint8_t tone;
        if (t < 7) tone = c_costas[t];
        else if (t >= 36 && t < 43) tone = c_costas[t - 36];
        else if (t >= 72) tone = c_costas[t - 72];
        else {
            const int k = 3 * (t < 36 ? t - 7 : t - 14);
            tone = c_gray[((cw[k] & 1) << 2) | ((cw[k + 1] & 1) << 1) | (cw[k + 2] & 1)];
        }
        ms.tones[t] = tone;
    }
    __syncthreads();
    if (t == 0) {
        const double p1 = g_pd[kSym], p2 = g_pd[2 * kSym], p3 = g_pd[3 * kSym];
        double acc = 0.0;
        for (int s = 0; s < kNsym; ++s) {
            ms.pst[s] = acc;
            const int tp = ms.tones[s > 0 ? s - 1 : 0], tc = ms.tones[s], tn = ms.tones[s + 1 < kNsym ? s + 1 : s];
            acc += tn * p1 + tc * (p2 - p1) + tp * (p3 - p2);
        }
    }
    __syncthreads();
}

// r[m], m in [0, kSpan): unit-amplitude GFSK with tone 0 at f_hz
__device__ __forceinline__ float2 ref_sample(const MsgShared &ms, int m, double f_hz) {
    const int s = m / kSym, j = m - s * kSym;
    const int tp = ms.tones[s > 0 ? s - 1 : 0], tc = ms.tones[s], tn = ms.tones[s + 1 < kNsym ? s + 1 : s];
    const double pulse = ms.pst[s] + tn * g_pd[j] + tc * (g_pd[j + kSym] - g_pd[kSym]) + tp * (g_pd[j + 2 * kSym] - g_pd[2 * kSym]);
    const double cyc = f_hz / kFs * (double)m + kToneHz / kFs * pulse;
    const float frac = (float)(cyc - floor(cyc));
    float sn, cs;
    sincospif(2.0f * frac, &sn, &cs);
    constexpr int kRamp = kSym / 8;
    float env = 1.0f;
    if (m < kRamp) env = (float)(0.5 - 0.5 * cospi((double)m / kRamp));
    else if (m >= kSpan - kRamp) env = (float)(0.5 - 0.5 * cospi((double)(kSpan - 1 - m) / kRamp));
    return make_float2(env * cs, env * sn);
}

struct MsgList {
    const candidate_t *cand;  // slot s, row r: cand[s * cand_stride + r]
    const uint8_t *cw;        // 174 bytes per row, indexed as cand
    int cand_stride;
    const int32_t *row;       // optional: entry j of slot s is row row[s * list_stride + j] (else row j)
    const int32_t *lo;        // optional: first entry of slot s (else 0)
    const int32_t *hi;        // entries [lo, hi) of slot s
    int list_stride;
};

__device__ __forceinline__ void list_range(const MsgList &L, int s, int &lo, int &hi) {
    lo = L.lo ? L.lo[s] : 0;
    hi = L.hi[s];
    if (hi > L.list_stride) hi = L.list_stride;   // counts from outside the library: never past the slot's own rows
    if (lo < 0) lo = 0;
}
__device__ __forceinline__ bool list_entry(const MsgList &L, int s, int j, candidate_t &c, const uint8_t *&cw) {
    const int r = L.row ? L.row[(size_t)s * L.list_stride + j] : j;
    if (r < 0 || r >= L.cand_stride) return false;
    const size_t o = (size_t)s * L.cand_stride + r;
    c = L.cand[o];
    cw = L.cw + o * kLdpcN;
    return true;
}
// Coarse stage: for each symbol the 17 dt candidates are downmixed by r at df = 0 and summed over sub-blocks of 8 samples, then
// rotated to each df (slot_search.cuh).  On a message's own waveform the dropped rotation within a sub-block is a factor
// sinc(pi df 8 / fs) = 1 - 5e-6 at the largest df that is nearly common to all points.  The fine stage, at one df, is exact.
__global__ void __launch_bounds__(kRefineThreads) refine_kernel(const float *__restrict__ x_i, const float *__restrict__ x_q, int n_slots, MsgList L,
                                                                int32_t *__restrict__ grid_out) {
    __shared__ MsgShared ms;
    __shared__ float2 xs[kSym + 2 * 128];
    __shared__ float2 rs[kSym];
    __shared__ float2 bs[kGrid * kBlocks];
    __shared__ float2 w[kGrid * kBlocks];
    __shared__ float2 part[kGrid * 16];
    __shared__ double metric[kGrid * kGrid];
    __shared__ int pick[2];
    const int tid = threadIdx.x;
    fill_rotations(w, kBlocks);
    const long long total = (long long)n_slots * L.list_stride;
    for (long long item = blockIdx.x; item < total; item += gridDim.x) {
        const int s = (int)(item % n_slots), j = (int)(item / n_slots);   // entry j of every slot before entry j + 1 of any
        int lo, hi;
        list_range(L, s, lo, hi);
        if (j < lo || j >= hi) continue;
        candidate_t cand;
        const uint8_t *cw;
        if (!list_entry(L, s, j, cand, cw)) continue;
        __syncthreads();   // the previous item's shared state is no longer read
        load_message(ms, cw);
        const float *xi = x_i + (size_t)s * kSlot, *xq = x_q + (size_t)s * kSlot;
        const int s_nom = nominal_start(cand);
        const double f0 = nominal_f0(cand);

        double acc[2] = {0.0, 0.0};
        for (int k = 0; k < kNsym; ++k) {
            const long long base = (long long)s_nom + (long long)kSym * k;
            for (int i = tid; i < kSym + 256; i += blockDim.x) xs[i] = load_x(xi, xq, base - 128 + i);
            for (int i = tid; i < kSym; i += blockDim.x) rs[i] = ref_sample(ms, kSym * k + i, f0);
            __syncthreads();
            for (int q = tid; q < kGrid * kBlocks; q += blockDim.x) {
                const int d = q / kBlocks, b = q - d * kBlocks;
                float2 a = make_float2(0.0f, 0.0f);
                for (int i = 0; i < kBlk; ++i) {
                    const float2 z = cmul_conj(xs[d * kCoarseStep + kBlk * b + i], rs[kBlk * b + i]);
                    a.x += z.x;
                    a.y += z.y;
                }
                bs[q] = a;
            }
            __syncthreads();
            for (int u = 0; u < 2; ++u) {
                const int p = tid + u * blockDim.x;
                if (p >= kGrid * kGrid) break;
                const int d = p / kGrid, f = p - d * kGrid;
                acc[u] += rotated_power(bs + d * kBlocks, w + f * kBlocks);
            }
            __syncthreads();
        }
        for (int u = 0; u < 2; ++u)
            if (tid + u * blockDim.x < kGrid * kGrid) metric[tid + u * blockDim.x] = acc[u];
        __syncthreads();
        if (tid == 0) {
            const int best = pick_max(metric, kGrid * kGrid);
            pick[0] = -128 + kCoarseStep * (best / kGrid);
            pick[1] = best % kGrid - 8;
        }
        __syncthreads();
        const int dt_c = pick[0], df_i = pick[1];
        const double f = f0 + df_i * kDfStep;

        double acc2 = 0.0;
        for (int k = 0; k < kNsym; ++k) {
            const long long base = (long long)s_nom + dt_c + (long long)kSym * k;
            for (int i = tid; i < kSym + 16; i += blockDim.x) xs[i] = load_x(xi, xq, base - 8 + i);
            for (int i = tid; i < kSym; i += blockDim.x) rs[i] = ref_sample(ms, kSym * k + i, f);
            __syncthreads();
            for (int q = tid; q < kGrid * 16; q += blockDim.x) {
                const int d = q / 16, c = q - d * 16;
                float2 a = make_float2(0.0f, 0.0f);
                for (int i = 0; i < 32; ++i) {
                    const float2 z = cmul_conj(xs[d + 32 * c + i], rs[32 * c + i]);
                    a.x += z.x;
                    a.y += z.y;
                }
                part[q] = a;
            }
            __syncthreads();
            if (tid < kGrid) {
                float re = 0.0f, im = 0.0f;
                for (int c = 0; c < 16; ++c) { re += part[tid * 16 + c].x; im += part[tid * 16 + c].y; }
                acc2 += (double)re * re + (double)im * im;
            }
            __syncthreads();
        }
        if (tid < kGrid) metric[tid] = acc2;
        __syncthreads();
        if (tid == 0) {
            const int best = pick_max(metric, kGrid);
            int32_t *g = grid_out + ((size_t)s * L.list_stride + j) * 2;
            g[0] = dt_c + best - 8;
            g[1] = df_i;
        }
    }
}

// inclusive prefix sums of three double2 arrays of n <= kHalo elements, in a fixed order (deterministic)
__device__ void scan3(double2 *a0, double2 *a1, double2 *a2, int n, double2 *warp_tot) {
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nw = blockDim.x >> 5;
    constexpr int kPer = (kHalo + kSubThreads - 1) / kSubThreads;
    const int b = tid * kPer, e = min(b + kPer, n);
    double2 *arr[3] = {a0, a1, a2};
    double2 run[3];
    for (int v = 0; v < 3; ++v) {
        double2 r = make_double2(0.0, 0.0);
        for (int i = b; i < e; ++i) { r.x += arr[v][i].x; r.y += arr[v][i].y; arr[v][i] = r; }
        run[v] = r;
    }
    // exclusive scan of the thread totals: within the warp by shuffles, then over the warps
    double2 incl[3];
    for (int v = 0; v < 3; ++v) {
        double2 x = run[v];
        for (int o = 1; o < 32; o <<= 1) {
            const double ux = __shfl_up_sync(0xffffffffu, x.x, o), uy = __shfl_up_sync(0xffffffffu, x.y, o);
            if (lane >= o) { x.x += ux; x.y += uy; }
        }
        incl[v] = x;
        if (lane == 31) warp_tot[v * 32 + wid] = x;
    }
    __syncthreads();
    if (tid < 3) {
        double2 r = make_double2(0.0, 0.0);
        for (int q = 0; q < nw; ++q) { const double2 t = warp_tot[tid * 32 + q]; warp_tot[tid * 32 + q] = r; r.x += t.x; r.y += t.y; }
    }
    __syncthreads();
    for (int v = 0; v < 3; ++v) {
        const double2 wo = warp_tot[v * 32 + wid];
        const double ox = wo.x + incl[v].x - run[v].x, oy = wo.y + incl[v].y - run[v].y;
        for (int i = b; i < e; ++i) { arr[v][i].x += ox; arr[v][i].y += oy; }
    }
    __syncthreads();
}

// sum of h[k] = 0.5 + 0.5 cos(w k) over k = p ... q
__device__ __forceinline__ double window_sum(int p, int q) {
    return 0.5 * (q - p + 1) + 0.5 * (sin(kWinW * (q + 0.5)) - sin(kWinW * (p - 0.5))) / (2.0 * sin(0.5 * kWinW));
}

__global__ void __launch_bounds__(kSubThreads) subtract_kernel(const float *__restrict__ x_i, const float *__restrict__ x_q, float *y_i, float *y_q,
                                                               int n_slots, MsgList L, const int32_t *__restrict__ grid, float2 *scratch,
                                                               int zero_idle) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double2 *u0 = reinterpret_cast<double2 *>(smem_raw), *up = u0 + kHalo, *um = up + kHalo, *warp_tot = um + kHalo;
    __shared__ MsgShared ms;
    const int tid = threadIdx.x;
    float2 *c = scratch + (size_t)blockIdx.x * kSpan;
    const double h_full = window_sum(-kHalfWin, kHalfWin);
    for (int s = blockIdx.x; s < n_slots; s += gridDim.x) {
        int lo, hi;
        list_range(L, s, lo, hi);
        float *yi = y_i + (size_t)s * kSlot, *yq = y_q + (size_t)s * kSlot;
        const float *xi = x_i + (size_t)s * kSlot, *xq = x_q + (size_t)s * kSlot;
        if (zero_idle && hi <= lo) {   // nothing new in this pass: the slot is not searched again
            for (int n = tid; n < kSlot; n += blockDim.x) { yi[n] = 0.0f; yq[n] = 0.0f; }
            continue;
        }
        if (xi != yi)
            for (int n = tid; n < kSlot; n += blockDim.x) { yi[n] = xi[n]; yq[n] = xq[n]; }
        __syncthreads();
        for (int j = lo; j < hi; ++j) {
            candidate_t cand;
            const uint8_t *cw;
            if (!list_entry(L, s, j, cand, cw)) continue;
            load_message(ms, cw);
            const int32_t *g = grid + ((size_t)s * L.list_stride + j) * 2;
            const long long S = (long long)nominal_start(cand) + g[0];
            const double f = nominal_f0(cand) + g[1] * kDfStep;
            const int n_lo = (int)max(S, 0ll), n_hi = (int)min(S + kSpan, (long long)kSlot);
            if (n_lo >= n_hi) { __syncthreads(); continue; }
            for (int n = n_lo + tid; n < n_hi; n += blockDim.x) c[n - S] = cmul_conj(make_float2(yi[n], yq[n]), ref_sample(ms, (int)(n - S), f));
            __syncthreads();
            for (int n0 = n_lo; n0 < n_hi; n0 += kChunk) {
                const int a = max(n0 - kHalfWin, n_lo), b = min(n0 + kChunk + kHalfWin, n_hi), len = b - a;
                for (int i = tid; i < len; i += blockDim.x) {
                    const float2 cv = c[a + i - S];
                    double sn, cs;
                    sincospi(2.0 * (a + i - n0) / 1026.0, &sn, &cs);   // e^{i w (m - n0)}
                    u0[i] = make_double2(cv.x, cv.y);
                    up[i] = make_double2(cv.x * cs - cv.y * sn, cv.x * sn + cv.y * cs);
                    um[i] = make_double2(cv.x * cs + cv.y * sn, cv.y * cs - cv.x * sn);
                }
                __syncthreads();
                scan3(u0, up, um, len, warp_tot);
                const int n1 = min(n0 + kChunk, n_hi);
                for (int n = n0 + tid; n < n1; n += blockDim.x) {
                    const int ka = max(n - kHalfWin, n_lo), kb = min(n + kHalfWin, n_hi - 1);
                    const int ia = ka - a, ib = kb - a;
                    double2 s0 = u0[ib], sp = up[ib], sm = um[ib];
                    if (ia > 0) {
                        s0.x -= u0[ia - 1].x; s0.y -= u0[ia - 1].y;
                        sp.x -= up[ia - 1].x; sp.y -= up[ia - 1].y;
                        sm.x -= um[ia - 1].x; sm.y -= um[ia - 1].y;
                    }
                    double sn, cs;
                    sincospi(2.0 * (n - n0) / 1026.0, &sn, &cs);   // e^{i w (n - n0)}
                    // sum_m h[m - n] c[m] = 0.5 S0 + 0.25 e^{-i w n} S+ + 0.25 e^{i w n} S-
                    const double ar = 0.5 * s0.x + 0.25 * (sp.x * cs + sp.y * sn) + 0.25 * (sm.x * cs - sm.y * sn);
                    const double ai = 0.5 * s0.y + 0.25 * (sp.y * cs - sp.x * sn) + 0.25 * (sm.y * cs + sm.x * sn);
                    const double hn = (ka == n - kHalfWin && kb == n + kHalfWin) ? h_full : window_sum(ka - n, kb - n);
                    const float2 r = ref_sample(ms, (int)(n - S), f);
                    const float amr = (float)(ar / hn), ami = (float)(ai / hn);
                    yi[n] -= amr * r.x - ami * r.y;
                    yq[n] -= amr * r.y + ami * r.x;
                }
                __syncthreads();
            }
        }
        __syncthreads();
    }
}

constexpr size_t kSubSmem = (size_t)(3 * kHalo + 96) * sizeof(double2);

}  // namespace

namespace ft8b200 {

cudaError_t upload_subtract_tables() {
    double pd[3 * kSym + 1];
    const double c = 3.14159265358979323846 * sqrt(2.0 / log(2.0)), bt = 2.0;
    double acc = 0.0;
    for (int j = 0; j < 3 * kSym; ++j) {
        pd[j] = acc;
        const double t = (double)j / kSym - 1.5;
        acc += (erf(c * bt * (t + 0.5)) - erf(c * bt * (t - 0.5))) / 2.0;
    }
    pd[3 * kSym] = acc;
    cudaError_t e = cudaMemcpyToSymbol(g_pd, pd, sizeof(pd));
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(c_costas, kFt8tCostas, sizeof(kFt8tCostas));
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(c_gray, kFt8tGray, sizeof(kFt8tGray));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(subtract_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSubSmem);
    return e;
}

size_t subtract_scratch_bytes(int n_slots, int sm_count) {
    const int ctas = n_slots < sm_count ? n_slots : sm_count;
    return (size_t)(ctas > 0 ? ctas : 1) * kSpan * sizeof(float2);
}

cudaError_t launch_subtract(const float *d_xi, const float *d_xq, float *d_yi, float *d_yq, int n_slots, const candidate_t *d_cand,
                            const uint8_t *d_cw, int cand_stride, const int32_t *d_row, const int32_t *d_lo, const int32_t *d_hi, int list_stride,
                            int32_t *d_grid, float2 *d_scratch, bool zero_idle, int sm_count, cudaStream_t st, int *launches) {
    const MsgList L = {d_cand, d_cw, cand_stride, d_row, d_lo, d_hi, list_stride};
    const int sms = sm_count > 0 ? sm_count : 1;
    long long items = (long long)n_slots * list_stride;
    const int rgrid = (int)(items < 4ll * sms ? items : 4ll * sms);
    refine_kernel<<<rgrid, kRefineThreads, 0, st>>>(d_xi, d_xq, n_slots, L, d_grid);
    ++*launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const int sgrid = n_slots < sms ? n_slots : sms;   // subtract_scratch_bytes sizes the scratch for this grid
    subtract_kernel<<<sgrid, kSubThreads, kSubSmem, st>>>(d_xi, d_xq, d_yi, d_yq, n_slots, L, d_grid, d_scratch, zero_idle ? 1 : 0);
    ++*launches;
    return cudaGetLastError();
}

}  // namespace ft8b200
