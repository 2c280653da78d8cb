// waterfall.cu -- windowed STFT -> uint8 dB waterfall of one 15 s slot (daemon path, 3200 sps complex).
// Replaces the FFTW loop of ft8_subsystem(), /root/reference/rtlsdr_ft8d.c:1395-1435 (+ window :331-334).
//
// 184 frames per slot (92 blocks x 2 time subdivisions), 1024-point complex FFT each, hop 256.
// The FFT is a register/shared-memory radix-4 decimation-in-time transform whose butterflies perform the same
// float operations, in the same order, as the reference's vendored kiss_fft (kf_bfly4,
// ft8_lib/fft/kiss_fft.c:38-84 with C_MUL of _kiss_fft_guts.h:81-83) -- 1024 = 4^5, so kiss_fft uses
// five radix-4 passes over a base-4 digit-reversed input -- which makes the spectrum, and therefore
// every waterfall byte, bit-identical to the CPU path that uses kiss_fft.  (The reference daemon itself
// links FFTW3f, an external library whose rounding depends on its plan; see DESIGN.md.)
// Magnitude -> dB -> uint8 is fused into the last pass; log10f is replaced by a comparison against the
// 255 host-computed step thresholds of the reference's quantiser (tables.cu), which is exact.
//
// Execution shape: PERSISTENT CTAs, 3 per SM.  A work item is a group of 4 consecutive frames of one slot
// (they overlap by 75 %: 1792 input samples); every CTA walks a contiguous range of groups.  Per CTA lifetime the
// twiddle/window/threshold tables are loaded into shared memory once; per group the 1024 new input samples arrive by
// cp.async into a 3-chunk ring while the previous group is being transformed, so no warp ever waits on a global load
// inside the transform.  64 threads own a frame (16 points each: stages {m=1,m=4}, {m=16,m=64}, {m=256}); the two
// exchanges go through an XOR-swizzled float2 buffer (conflict-free in all three access patterns) and are ordered by
// 64-thread named barriers, so the four frames of a CTA drift apart instead of meeting at __syncthreads.
//
// Round 2: the exchange buffer is addressed by 32-bit shared addresses built so that every access is `R ^ imm` or
// `[R + imm]` with a per-thread register R computed once per CTA lifetime (the swizzle XORs bits 3..6 of a 128-byte
// aligned row, everything else is additive above bit 6) -- one LOP3 or nothing per access instead of the 4-5 integer
// instructions per access the index expression compiled to; the quantiser is straight-line code: the MUFU.LG2 estimate is
// within one step of the answer for every float (ft8b200_selfcheck_quantiser sweeps all bit patterns), so ONE 64-bit load
// of {thr[k], thr[k+1]} and two compares settle it -- no loops, no branches, half the (randomly addressed, hence
// bank-conflicting) threshold loads.
#include "common.cuh"

namespace ft8b200 {
namespace {

constexpr int kThreads = 256;
constexpr int kFramesPerCta = 4;
constexpr int kGroupsPerSlot = kFrames / kFramesPerCta;  // 46
constexpr int kChunk = 1024;                             // input samples per ring chunk (= hop * frames per group)
constexpr int kCtasPerSm = 3;
constexpr uint32_t kRingBytes = 3u * kChunk * 4u;        // one rail of the ring
constexpr int kOutSkew = 16, kOutPitch = 512 + kOutSkew;

struct cpx { float r, i; };
__device__ __forceinline__ cpx cmul(cpx a, float2 b) {  // C_MUL: each product rounded, then the add
    cpx m;
    m.r = __fsub_rn(__fmul_rn(a.r, b.x), __fmul_rn(a.i, b.y));
    m.i = __fadd_rn(__fmul_rn(a.r, b.y), __fmul_rn(a.i, b.x));
    return m;
}
__device__ __forceinline__ cpx cadd(cpx a, cpx b) { return cpx{__fadd_rn(a.r, b.r), __fadd_rn(a.i, b.i)}; }
__device__ __forceinline__ cpx csub(cpx a, cpx b) { return cpx{__fsub_rn(a.r, b.r), __fsub_rn(a.i, b.i)}; }

// shared-memory accesses by 32-bit shared address (constant parts of `a` fold into the instruction's immediate offset)
__device__ __forceinline__ float2 lds64(uint32_t a) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a));
    return v;
}
__device__ __forceinline__ float lds32(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts64(uint32_t a, float x, float y) { asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(a), "f"(x), "f"(y) : "memory"); }
__device__ __forceinline__ void sts8(uint32_t a, int v) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// Exact replacement of clamp((int)(2*(10*log10f(x))+240),0,255): the count of step thresholds <= x.  k0 = the MUFU.LG2
// estimate clamped to [0, 255]; the answer is k0 - 1, k0 or k0 + 1 for every x >= 0 (and NaN gives 0, +inf gives 256 -> byte 0,
// which is what the reference's (int) conversion of +-inf / NaN ends up as on x86): one 64-bit load of {thr[k0], thr[k0+1]}.
__device__ __forceinline__ int quantise_estimate(float x) {
    int k = (int)__fmaf_rn(6.0206f, __log2f(x), 240.0f);  // an estimate: any rounding will do (ft8b200_selfcheck_quantiser proves the +-1 bound for THIS form)
    return k < 0 ? 0 : (k > 255 ? 255 : k);
}
__device__ __forceinline__ int quantise(float x, uint32_t thr2_base) {
    const int k = quantise_estimate(x);
    const float2 lh = lds64(thr2_base + 8u * (uint32_t)k);  // thr[0] = 0, thr[256] = +inf
    return k + (x >= lh.y ? 1 : 0) - (x < lh.x ? 1 : 0);
}

// radix-4 butterfly of kf_bfly4 (forward), twiddled inputs a,b,c already formed
__device__ __forceinline__ void bfly4(cpx &f0, cpx &f1, cpx &f2, cpx &f3, const cpx a, const cpx b, const cpx c) {
    const cpx d5 = csub(f0, b);
    f0 = cadd(f0, b);
    const cpx s3 = cadd(a, c);
    const cpx s4 = csub(a, c);
    f2 = csub(f0, s3);
    f0 = cadd(f0, s3);
    f1.r = __fadd_rn(d5.r, s4.i); f1.i = __fsub_rn(d5.i, s4.r);
    f3.r = __fsub_rn(d5.r, s4.i); f3.i = __fadd_rn(d5.i, s4.r);
}
// kiss_fft multiplies by twiddle 0 = (1, -0) like by any other.  For a finite input the product equals the input except
// possibly for the sign of a zero, which cannot reach |X|^2.  For a non-finite one it does not: inf * -0 is NaN, so kiss_fft
// turns (inf, y) into (inf, NaN) where skipping keeps (inf, y).  That cannot change a byte either: every bin such a frame
// reaches is then inf or NaN (no other twiddle has an exact zero component), and the quantiser maps both to 0
// (test_non_finite_and_extreme_float_slots).  So index-0 twiddles are skipped WHERE THAT IS KNOWN AT COMPILE TIME (pass A).
// Where it depends on the lane (i0 == 0 in pass B, i == 0 in pass C) the multiplication is simply performed, as kiss_fft
// does: a per-lane special case made every warp execute both the twiddled and the untwiddled butterfly (2 of its 32 lanes
// took the short path), which cost pass B half as much again as the arithmetic it saved.
__device__ __forceinline__ void bfly4_tw(cpx &f0, cpx &f1, cpx &f2, cpx &f3, float2 t1, float2 t2, float2 t3, bool trivial) {
    if (trivial) bfly4(f0, f1, f2, f3, f1, f2, f3);
    else bfly4(f0, f1, f2, f3, cmul(f1, t1), cmul(f2, t2), cmul(f3, t3));
}

// stage m=4 twiddles tw[64 q (k+1)], q = 1..3: the same for every thread -> constant bank operands
__constant__ float2 c_tw_a[3][3];

// Exchange buffer: element o of a frame's 1024-point array lives at (o & ~15) | ((o & 15) ^ ((o >> 6) & 15)) (float2 units).
// Pass A writes 16 consecutive elements per thread, pass B reads/writes stride-16 and stride-64 sets, pass C reads stride 256;
// with this swizzle the 16 lanes of every half-warp hit 16 different 8-byte bank pairs in all of them.  In bytes the swizzle
// XORs bits 3..6 of an address whose row (bits >= 7) is untouched, so with a 128-byte aligned buffer
//   pass A:  (RA ^ 8j),                       RA = (base + 128 p)          | 8 (t & 15)
//   pass B:  (RB ^ 8c) + 512 c + 128 a,       RB = (base + 2048 bq)        | (8 i0 ^ 32 bq)
//   pass C:  (RC ^ 8(u + 4q)) + 512 u + 2048 q,  RC = (base + 8 (t & 48))  | 8 (t & 15)
struct WfSmem {
    float2 ex[kFramesPerCta][1024];    // first: 128-byte aligned (checked at kernel start)
    float ring_i[3 * kChunk], ring_q[3 * kChunk];  // input samples, chunk c of the slot in ring slot c % 3
    float2 tw_c[768];                  // tw[k], k < 768: last stage uses tw[i], tw[2i], tw[3i], i < 256
    float2 tw_b2[4][3][16];            // tw[4 (k+1) (i0 + 16 a)]: stage m=64
    float win[16][64];                 // window[n(j, t)]: pass A's 16 window values of thread t
    float2 thr2[256];                  // {thr[k], thr[k+1]}: the step thresholds around estimate k
    float2 tw_2[256];                  // tw[2 i], i < 256, compact: read at stride 2 out of tw_c the 16 lanes of a half-warp would share 8 bank pairs
    uint8_t out[kFramesPerCta][kOutPitch];  // the frame's 512 bytes; the second 256 start 16 bytes later (kOutSkew): the two rows a warp writes fall on different banks
};

__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void frame_barrier(int fr) { asm volatile("bar.sync %0, 64;" ::"r"(fr + 1) : "memory"); }

// layout of the table blob built by build_waterfall_tables(): floats.  [kBlobTwC, kBlobTwB1) mirrors WfSmem from tw_c on.
constexpr int kBlobTwC = 0, kBlobTwB2 = kBlobTwC + 768 * 2, kBlobWin = kBlobTwB2 + 4 * 3 * 16 * 2, kBlobThr2 = kBlobWin + 16 * 64,
              kBlobTw2 = kBlobThr2 + 256 * 2, kBlobTwB1 = kBlobTw2 + 256 * 2, kBlobTwA = kBlobTwB1 + 3 * 16 * 2, kBlobFloats = kBlobTwA + 9 * 2;

__global__ void __launch_bounds__(kThreads, kCtasPerSm)
waterfall1024_kernel(const float *__restrict__ d_i, const float *__restrict__ d_q, const float *__restrict__ peak,
                     const float *__restrict__ blob, int total_groups, uint8_t *__restrict__ mag) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    WfSmem &sm = *reinterpret_cast<WfSmem *>(smem_raw);
    const int tid = threadIdx.x;
    const int g_begin = (int)((long long)blockIdx.x * total_groups / gridDim.x);
    const int g_end = (int)((long long)(blockIdx.x + 1) * total_groups / gridDim.x);
    if (g_begin >= g_end) return;
    if (smem_u32(smem_raw) & 127u) __trap();  // the XOR addressing below relies on it

    // ---- once per CTA: tables -> shared memory (contiguous in the blob in WfSmem order), stage m=16 twiddles -> registers
    {
        const float4 *src = reinterpret_cast<const float4 *>(blob);
        float4 *dst = reinterpret_cast<float4 *>(&sm.tw_c[0]);
        for (int k = tid; k < kBlobTwB1 / 4; k += kThreads) dst[k] = __ldg(src + k);
    }
    const int fr = tid >> 6, t = tid & 63;
    const int i0 = t & 15, bq = t >> 4;  // pass B coordinates
    float2 tb1[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) tb1[k] = __ldg(reinterpret_cast<const float2 *>(blob + kBlobTwB1) + k * 16 + i0);
    // pass A coordinates: this thread transforms the 16 elements o = 16 p + j, which come from input n = rev2(j)*64 + r3
    // (base-4 digit reversal, kf_work's leaf copy order); p and r3 are digit reversals of each other.  The lane -> p map is
    // chosen so that both the input reads (bank = r3 mod 32) and the swizzled float2 writes are conflict-free.
    const int r3 = ((t >> 4) << 4) | ((t & 3) << 2) | ((t >> 2) & 3);
    const int p = (((t >> 2) & 3) << 4) | ((t & 3) << 2) | (t >> 4);
    // per-thread address registers, valid for the CTA's lifetime (see the table above WfSmem)
    const uint32_t ex_b = smem_u32(sm.ex[fr]);
    const uint32_t RA = (ex_b + 128u * (uint32_t)p) | (8u * (uint32_t)(t & 15));
    const uint32_t RB = (ex_b + 2048u * (uint32_t)bq) | ((8u * (uint32_t)i0) ^ (32u * (uint32_t)bq));
    const uint32_t RC = (ex_b + 8u * (uint32_t)(t & 48)) | (8u * (uint32_t)(t & 15));
    const uint32_t Rwin = smem_u32(&sm.win[0][t]);                       // + 256 j
    const uint32_t Rtb2 = smem_u32(&sm.tw_b2[0][0][i0]);                  // + 128 (3 a + k)
    const uint32_t Rtc1 = smem_u32(sm.tw_c) + 8u * (uint32_t)t;          // tw[i],  i = t + 64 u: + 512 u
    const uint32_t Rtc2 = smem_u32(sm.tw_2) + 8u * (uint32_t)t;          // tw[2i] = tw_2[i]:     + 512 u
    const uint32_t Rtc3 = smem_u32(sm.tw_c) + 24u * (uint32_t)t;         // tw[3i]:               + 1536 u
    const uint32_t Rout = smem_u32(sm.out[fr]) + (256u + kOutSkew) * (uint32_t)(t & 1) + (uint32_t)(t >> 1);  // + 32 u (+ 128)
    const uint32_t thr_b = smem_u32(sm.thr2);
    const uint32_t ring_b = smem_u32(sm.ring_i) + 4u * (uint32_t)(256 * fr + r3);  // sample 256 fr + r3 of ring slot 0, I rail

    auto load_chunk = [&](int slot, int chunk) {  // 1024 samples (the slot's last chunk, 46, holds 896), one 16-byte piece per thread and rail
        const int s = chunk * kChunk + tid * 4;
        if (s < kSlot) {
            cp_async16(&sm.ring_i[(chunk % 3) * kChunk + tid * 4], d_i + (size_t)slot * kSlot + s);
            cp_async16(&sm.ring_q[(chunk % 3) * kChunk + tid * 4], d_q + (size_t)slot * kSlot + s);
        }
    };

    float scale = 1.0f;
    for (int G = g_begin; G < g_end; ++G) {
        const int slot = G / kGroupsPerSlot, g = G - slot * kGroupsPerSlot;
        if (G == g_begin || g == 0) {  // (re)start of a slot: both chunks of this group are fetched now
            __syncthreads();           // the ring may still be read by the previous group
            load_chunk(slot, g);
            load_chunk(slot, g + 1);
            cp_async_commit();
            scale = 1.0f;
            if (peak != nullptr) {  // decoder(): maxSig = 0.5 / max(1e-24f, peak), rtlsdr_ft8d.c:249-259
                float pk = __ldg(peak + slot);
                if (!(pk > 1e-24f)) pk = 1e-24f;
                scale = __double2float_rn(__ddiv_rn(0.5, (double)pk));
            }
        }
        cp_async_wait_all();
        __syncthreads();  // this group's samples are visible to everyone; everyone is done with the group before
        if (g + 1 < kGroupsPerSlot && G + 1 < g_end) {  // next group's new chunk, in flight during this group's transform
            load_chunk(slot, g + 2);
            cp_async_commit();
        }
        // the group's samples 0..1791 start at ring slot g % 3 and run on into slot (g + 1) % 3: sample s lives at byte
        // 4096 gm + 4 s of the rail, minus the rail's size once that passes its end.  s = 256 fr + 64 c + r3 with 4 r3 < 256, so
        // "past the end" is 16 gm + 4 fr + c >= 48: the same for every lane of a warp.
        // c = 4 (j & 3) + (j >> 2) and the test only involves c >> 2 = j & 3: four base addresses per group, then immediates.
        const int gm = g % 3;
        const uint32_t G0 = ring_b + 4096u * (uint32_t)gm;
        uint32_t Gq[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) Gq[q] = (4 * gm + fr + q >= 12) ? G0 - kRingBytes : G0;

        cpx e[16];
        {   // pass A: stages m=1 and m=4 on 16 consecutive (digit-reversed) points
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const int c = ((j & 3) << 2) | (j >> 2);
                const uint32_t a = Gq[j & 3] + 256u * (uint32_t)c;
                const float xi = lds32(a), xq = lds32(a + kRingBytes);
                const float w = lds32(Rwin + 256u * (uint32_t)j);
                e[j].r = __fmul_rn(__fmul_rn(xi, scale), w);            // decoder()'s scale, then the window (x * 1.0f is exact)
                e[j].i = __fmul_rn(__fmul_rn(xq, scale), w);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) bfly4(e[4 * q], e[4 * q + 1], e[4 * q + 2], e[4 * q + 3], e[4 * q + 1], e[4 * q + 2], e[4 * q + 3]);
            bfly4(e[0], e[4], e[8], e[12], e[4], e[8], e[12]);
#pragma unroll
            for (int q = 1; q < 4; ++q) bfly4_tw(e[q], e[q + 4], e[q + 8], e[q + 12], c_tw_a[q - 1][0], c_tw_a[q - 1][1], c_tw_a[q - 1][2], false);
#pragma unroll
            for (int j = 0; j < 16; ++j) sts64(RA ^ (8u * (uint32_t)j), e[j].r, e[j].i);  // swz(16 p + j): (o >> 6) & 15 == t & 15
        }
        frame_barrier(fr);
        {   // pass B: points 256 b + i0 + 16 a + 64 c: stages m=16 (over a) and m=64 (over c)
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const uint32_t rb = (RB ^ (8u * (uint32_t)c)) + 512u * (uint32_t)c;
#pragma unroll
                for (int a = 0; a < 4; ++a) {
                    const float2 v = lds64(rb + 128u * (uint32_t)a);
                    e[4 * c + a].r = v.x; e[4 * c + a].i = v.y;
                }
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) bfly4_tw(e[4 * c], e[4 * c + 1], e[4 * c + 2], e[4 * c + 3], tb1[0], tb1[1], tb1[2], false);
#pragma unroll
            for (int a = 0; a < 4; ++a)
                bfly4_tw(e[a], e[4 + a], e[8 + a], e[12 + a], lds64(Rtb2 + 128u * (uint32_t)(3 * a)), lds64(Rtb2 + 128u * (uint32_t)(3 * a + 1)),
                         lds64(Rtb2 + 128u * (uint32_t)(3 * a + 2)), false);
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const uint32_t rb = (RB ^ (8u * (uint32_t)c)) + 512u * (uint32_t)c;
#pragma unroll
                for (int a = 0; a < 4; ++a) sts64(rb + 128u * (uint32_t)a, e[4 * c + a].r, e[4 * c + a].i);
            }
        }
        frame_barrier(fr);
        {   // pass C: last stage (m = 256); only bins i and i+256 are kept (the daemon stores bins 0..511)
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float2 v0 = lds64((RC ^ (8u * (uint32_t)u)) + 512u * (uint32_t)u);
                const float2 v1 = lds64((RC ^ (8u * (uint32_t)(u + 4))) + 512u * (uint32_t)u + 2048u);
                const float2 v2 = lds64((RC ^ (8u * (uint32_t)(u + 8))) + 512u * (uint32_t)u + 4096u);
                const float2 v3 = lds64((RC ^ (8u * (uint32_t)(u + 12))) + 512u * (uint32_t)u + 6144u);
                cpx f0{v0.x, v0.y}, f1{v1.x, v1.y}, f2{v2.x, v2.y}, f3{v3.x, v3.y};
                const cpx a = cmul(f1, lds64(Rtc1 + 512u * (uint32_t)u));
                const cpx b = cmul(f2, lds64(Rtc2 + 512u * (uint32_t)u));
                const cpx c = cmul(f3, lds64(Rtc3 + 1536u * (uint32_t)u));
                const cpx d5 = csub(f0, b);
                f0 = cadd(f0, b);
                const cpx s3 = cadd(a, c);
                const cpx s4 = csub(a, c);
                f0 = cadd(f0, s3);
                f1.r = __fadd_rn(d5.r, s4.i); f1.i = __fsub_rn(d5.i, s4.r);
                // mag2 * 4.0f / (NFFT*NFFT) then 1E-12f + ..., rtlsdr_ft8d.c:1415-1416 (the divide by 2^20 is an exact scaling)
                const float m0 = __fadd_rn(__fmul_rn(f0.r, f0.r), __fmul_rn(f0.i, f0.i));
                const float m1 = __fadd_rn(__fmul_rn(f1.r, f1.r), __fmul_rn(f1.i, f1.i));
                const float x0 = __fadd_rn(1E-12f, __fmul_rn(__fmul_rn(m0, 4.0f), 9.5367431640625e-07f));
                const float x1 = __fadd_rn(1E-12f, __fmul_rn(__fmul_rn(m1, 4.0f), 9.5367431640625e-07f));
                // layout [freq_sub][bin]: FFT bin 2*bin+freq_sub, rtlsdr_ft8d.c:1420-1428 -> byte (i & 1) * 256 + (i >> 1), and + 128 for bin i + 256
                sts8(Rout + 32u * (uint32_t)u, quantise(x0, thr_b));
                sts8(Rout + 32u * (uint32_t)u + 128u, quantise(x1, thr_b));
            }
        }
        frame_barrier(fr);
        if (t < 32) {  // the frame's 512 bytes, 16 per lane
            uint4 *dst = reinterpret_cast<uint4 *>(mag + (size_t)slot * kWfBytes + (size_t)(g * kFramesPerCta + fr) * 512);
            dst[t] = reinterpret_cast<const uint4 *>(sm.out[fr])[t < 16 ? t : t + kOutSkew / 16];
        }
    }
}

// ft8b200_selfcheck_quantiser: every non-negative float bit pattern (+inf included) and every NaN through quantise() against a
// binary search over the 256 thresholds: counts[0] = mismatches, counts[1] = inputs whose estimate was off by one (took the
// correction), counts[2] = inputs whose estimate was off by MORE than one (must be 0: the straight-line form relies on it)
__global__ void quantise_check_kernel(const float *__restrict__ thr257, unsigned long long *counts) {
    __shared__ float2 s_thr2[256];
    __shared__ float s_thr[257];
    for (int k = threadIdx.x; k < 257; k += blockDim.x) s_thr[k] = thr257[k];
    for (int k = threadIdx.x; k < 256; k += blockDim.x) s_thr2[k] = make_float2(thr257[k], thr257[k + 1]);
    __syncthreads();
    const uint32_t base = smem_u32(s_thr2);
    unsigned long long bad = 0, corrected = 0, far = 0;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long b = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; b < (1ull << 32); b += stride) {
        const uint32_t bits = (uint32_t)b;
        const float x = __uint_as_float(bits);
        if ((bits >> 31) && !(x != x)) continue;  // negative numbers cannot occur (x = 1e-12f + a sum of squares); NaNs of either sign can
        int want = 0;                             // count of thresholds thr[1..256] <= x
        if (x == x) {
            int lo = 0, hi = 256;                 // invariant: thr[lo] <= x (thr[0] = 0), thr[hi + 1]... search the largest k with thr[k] <= x
            while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (s_thr[mid] <= x) lo = mid; else hi = mid - 1; }
            want = lo;
        }
        const int got = quantise(x, base);
        bad += (uint8_t)got != (uint8_t)want;
        const int est = quantise_estimate(x);
        const int d = est - want;
        if (x == x && want <= 255) { corrected += d != 0; far += (d < -1 || d > 1); }
    }
    if (bad) atomicAdd(counts + 0, bad);
    atomicAdd(counts + 1, corrected);
    if (far) atomicAdd(counts + 2, far);
}

}  // namespace

// Host side of the table blob (layout: kBlob* above).  window/twiddles/thresholds are the host-libm tables of tables.cu.
void build_waterfall_tables(const float *window, const float2 *tw, const float *thr257, float *blob) {
    float2 *twc = reinterpret_cast<float2 *>(blob + kBlobTwC);
    for (int k = 0; k < 768; ++k) twc[k] = tw[k];
    float2 *b2 = reinterpret_cast<float2 *>(blob + kBlobTwB2);
    for (int a = 0; a < 4; ++a)
        for (int k = 0; k < 3; ++k)
            for (int i0 = 0; i0 < 16; ++i0) b2[(a * 3 + k) * 16 + i0] = tw[4 * (k + 1) * (i0 + 16 * a)];
    for (int j = 0; j < 16; ++j)
        for (int t = 0; t < 64; ++t) {
            const int c = ((j & 3) << 2) | (j >> 2);
            const int r3 = ((t >> 4) << 4) | ((t & 3) << 2) | ((t >> 2) & 3);
            blob[kBlobWin + j * 64 + t] = window[c * 64 + r3];
        }
    for (int k = 0; k < 256; ++k) { blob[kBlobThr2 + 2 * k] = thr257[k]; blob[kBlobThr2 + 2 * k + 1] = thr257[k + 1]; }
    float2 *t2 = reinterpret_cast<float2 *>(blob + kBlobTw2);
    for (int i = 0; i < 256; ++i) t2[i] = tw[2 * i];
    float2 *b1 = reinterpret_cast<float2 *>(blob + kBlobTwB1);
    for (int k = 0; k < 3; ++k)
        for (int i0 = 0; i0 < 16; ++i0) b1[k * 16 + i0] = tw[16 * (k + 1) * i0];
    float2 *ta = reinterpret_cast<float2 *>(blob + kBlobTwA);
    for (int q = 1; q < 4; ++q)
        for (int k = 0; k < 3; ++k) ta[(q - 1) * 3 + k] = tw[64 * q * (k + 1)];
}
int waterfall_blob_floats() { return kBlobFloats; }
cudaError_t upload_waterfall_constants(const float *blob_host) {
    return cudaMemcpyToSymbol(c_tw_a, blob_host + kBlobTwA, sizeof(float2) * 9);
}

cudaError_t launch_waterfall(const DeviceTables &tb, const float *d_i, const float *d_q, const float *d_peak, int n_slots, uint8_t *d_mag,
                             int sm_count, cudaStream_t st, int *launches) {
    static_assert(kFrames % kFramesPerCta == 0, "184 frames = 46 groups of 4");
    static_assert(offsetof(WfSmem, tw_b2) - offsetof(WfSmem, tw_c) == kBlobTwB2 * 4 && offsetof(WfSmem, win) - offsetof(WfSmem, tw_c) == kBlobWin * 4 &&
                      offsetof(WfSmem, thr2) - offsetof(WfSmem, tw_c) == kBlobThr2 * 4 && offsetof(WfSmem, tw_2) - offsetof(WfSmem, tw_c) == kBlobTw2 * 4 &&
                      offsetof(WfSmem, out) - offsetof(WfSmem, tw_c) == kBlobTwB1 * 4 && offsetof(WfSmem, out) % 16 == 0 && kOutPitch % 16 == 0,
                  "the blob's shared-memory part mirrors WfSmem from tw_c on");
    static_assert(offsetof(WfSmem, ex) == 0 && offsetof(WfSmem, tw_c) % 16 == 0 && offsetof(WfSmem, ring_q) - offsetof(WfSmem, ring_i) == kRingBytes, "WfSmem layout");
    static_assert(kBlobTwB1 % 4 == 0, "blob is copied in 16-byte pieces");
    cudaError_t e = cudaFuncSetAttribute(waterfall1024_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(WfSmem));
    if (e != cudaSuccess) return e;
    const int total = n_slots * kGroupsPerSlot;
    int grid = sm_count * kCtasPerSm;
    if (grid > total) grid = total;
    waterfall1024_kernel<<<grid, kThreads, sizeof(WfSmem), st>>>(d_i, d_q, d_peak, tb.wf_blob, total, d_mag);
    ++*launches;
    return cudaGetLastError();
}

// all float bit patterns the quantiser can see through the kernel's quantise() against a search over the thresholds
cudaError_t run_quantiser_check(const float *d_thr257, unsigned long long *h_counts3, int sm_count, cudaStream_t st) {
    unsigned long long *d = nullptr;
    cudaError_t err = cudaMalloc(&d, 3 * sizeof(unsigned long long));
    if (err != cudaSuccess) return err;
    cudaMemsetAsync(d, 0, 3 * sizeof(unsigned long long), st);
    quantise_check_kernel<<<(sm_count > 0 ? sm_count : 1) * 16, 256, 0, st>>>(d_thr257, d);
    err = cudaMemcpyAsync(h_counts3, d, 3 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st);
    if (err == cudaSuccess) err = cudaStreamSynchronize(st);
    cudaFree(d);
    return err;
}

}  // namespace ft8b200
