// decimator.cu -- uint8 IQ @ 2.4 Msps -> float I/Q @ 3200 sps (fs/4 mixer, CIC N=2 R=751 M=2, 57-tap FIR).
// Replaces rtlsdr_callback(), /root/reference/rtlsdr_ft8d.c:76-202, for whole batches of streams.
//
// Design (B200-first, not a translation of the sample-by-sample loop):
//   The two integrators + two combs of the reference are, exactly and in wrapping int32 arithmetic,
//   a 3003-tap triangular FIR sampled every 751 inputs (SURVEY.md section 8 a2).  Splitting the input
//   into 751-sample blocks b with S0_b = sum s, S1_b = sum i*s (i = index inside the block):
//       y2[k] = (751*S0_k - S1_k) + (1502*S0_{k-1} - S1_{k-1}) + (751*S0_{k-2} + S1_{k-2}) + S1_{k-3}
//   so the only pass over the 72 MB/slot input is a streaming reduction (kernel 1, HBM-bound:
//   2 B/sample in, 16 B/751 samples out), and everything order-sensitive (the float FIR, the
//   double-precision scale) happens on the 751x smaller block-sum array (kernel 2).
//
//   Kernel 1 maps one warp to one "super-block" of 8 blocks = 6008 samples = 12016 B = exactly 751
//   16-byte chunks, so every lane issues aligned, fully coalesced 128-bit loads and the block layout
//   inside a super-block is a compile-time constant (the 24 warp-iterations are fully unrolled).
//   The mixer (multiply sample n by j^n, with the reference's wrapping int8 negate: -(-128) == -128)
//   is done four bytes at a time: bytes are regrouped by PRMT into {I-rail plain, I-rail negated,
//   Q-rail plain, Q-rail negated} words, the negated words get a carry-free per-byte two's-complement
//   (3 ALU ops), and S0/S1 partial sums are DP4A dot products with constant weight words.  Values are
//   kept as unsigned bytes v+128; the -128 offsets are constants per block.  Block totals are warp
//   reductions (REDUX), one per finished block.  The 7 chunks per super-block that straddle a block
//   boundary are first attributed whole to the earlier block and corrected afterwards by 7 lanes.
#include "common.cuh"

#include <stdlib.h>

#include <atomic>
#include <mutex>

namespace ft8b200 {

namespace {

constexpr int kChunksPerSuper = 751;          // 16-byte chunks per super-block
constexpr int kSuperBytes = 12016;            // 8 * 751 * 2
constexpr uint32_t kOnes = 0x01010101u;
// sample index (0..7 inside the chunk) of each byte of the regrouped words
constexpr uint32_t kW_IP = 0x07040300u;  // I rail, plain   : samples 0,3,4,7  (bytes I0,Q3,I4,Q7)
constexpr uint32_t kW_IN = 0x06050201u;  // I rail, negated : samples 1,2,5,6  (bytes Q1,I2,Q5,I6)
constexpr uint32_t kW_QP = 0x05040100u;  // Q rail, plain   : samples 0,1,4,5  (bytes Q0,I1,Q4,I5)
constexpr uint32_t kW_QN = 0x07060302u;  // Q rail, negated : samples 2,3,6,7  (bytes Q2,I3,Q6,I7)
constexpr uint32_t kOff0 = 128u * 751u;                 // sum of the +128 offsets over a block
constexpr uint32_t kOff1 = 128u * (750u * 751u / 2u);   // sum of i*128

struct Acc { uint32_t s0i, s1i, s0q, s1q; };

__device__ __forceinline__ uint4 ldg_stream(const uint4 *p) {
    uint4 v;
    // (an L2 evict-first policy on these loads -- so that what the back end re-reads a millisecond later stays resident -- was
    // measured and changes nothing: 1.483-1.490 against 1.486-1.523 ms per 128 slots on 116 SMs, profiles/k1_prefetch_r2zb.txt)
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}

// per-byte two's complement (mod 256) of all four bytes, no carries between bytes
__device__ __forceinline__ uint32_t neg4(uint32_t u) { return (0x80808080u - (u & 0x7f7f7f7fu)) ^ (~u & 0x80808080u); }

// regroup one 16-byte chunk (samples 0..7 as I0 Q0 I1 Q1 ...) into the four rail words
__device__ __forceinline__ void regroup(const uint4 w, uint32_t &ip, uint32_t &in, uint32_t &qp, uint32_t &qn) {
    qp = __byte_perm(w.x, w.z, 0x6521);                 // Q0 I1 Q4 I5
    qn = neg4(__byte_perm(w.y, w.w, 0x6521));           // -(Q2 I3 Q6 I7)
    const uint32_t t01 = __byte_perm(w.x, w.y, 0x4370); // I0 Q3 Q1 I2
    const uint32_t t23 = __byte_perm(w.z, w.w, 0x4370); // I4 Q7 Q5 I6
    ip = __byte_perm(t01, t23, 0x5410);                 // I0 Q3 I4 Q7
    in = neg4(__byte_perm(t01, t23, 0x7632));           // -(Q1 I2 Q5 I6)
}

template <int K>
struct IterInfo {
    static constexpr int c0 = 32 * K;
    static constexpr int nvalid = (kChunksPerSuper - c0) < 32 ? (kChunksPerSuper - c0) : 32;
    static constexpr int bF = (8 * c0) / kDecim;                      // block of lane 0's chunk
    static constexpr int bL = (8 * (c0 + nvalid - 1)) / kDecim;       // block of the last valid lane's chunk
    static constexpr bool trans = (bL != bF);
    static constexpr int Lk = trans ? ((kDecim * (bF + 1) - 1) / 8 - c0) : 31;  // last lane still in block bF
    static constexpr int bN = (c0 + 32 < kChunksPerSuper) ? (8 * (c0 + 32)) / kDecim : 8;
    static constexpr bool flush = (bN > bF);                          // block bF is complete after this iteration
    static constexpr int ibase = 8 * c0 - kDecim * bF;                // in-block index of lane 0's first sample
};

// kSmem: the super-block has been staged in shared memory (bulk-copy kernel) instead of being streamed from global
template <bool kSmem>
__device__ __forceinline__ uint4 ld_chunk(const uint4 *p) {
    if (kSmem) return *p;  // LDS.128, consecutive lanes -> consecutive 16-byte chunks: conflict-free
    return ldg_stream(p);
}

template <int K, bool kSmem = false>
__device__ __forceinline__ uint4 load_chunk(const uint4 *base, int lane) {
    using I = IterInfo<K>;
    if (I::nvalid == 32 || lane < I::nvalid) return ld_chunk<kSmem>(base + I::c0 + lane);
    return make_uint4(0u, 0u, 0u, 0u);  // contributes nothing to the unsigned sums
}

template <int K>
__device__ __forceinline__ void process_chunk(const uint4 w, int lane, uint32_t lane8, Acc &A, Acc &B, uint4 *wsums) {
    using I = IterInfo<K>;
    uint32_t ip, in, qp, qn;
    regroup(w, ip, in, qp, qn);
    const uint32_t u0i = __dp4a(ip, kOnes, __dp4a(in, kOnes, 0u));
    const uint32_t u0q = __dp4a(qp, kOnes, __dp4a(qn, kOnes, 0u));
    if (!I::trans) {
        const uint32_t i0 = lane8 + (uint32_t)I::ibase;
        A.s0i += u0i;
        A.s0q += u0q;
        A.s1i = __dp4a(ip, kW_IP, __dp4a(in, kW_IN, A.s1i + i0 * u0i));
        A.s1q = __dp4a(qp, kW_QP, __dp4a(qn, kW_QN, A.s1q + i0 * u0q));
    } else {
        const bool later = lane > I::Lk;  // this lane's chunk starts in block bF+1
        const uint32_t i0 = lane8 + (uint32_t)I::ibase - (later ? (uint32_t)kDecim : 0u);
        const uint32_t u1i = __dp4a(ip, kW_IP, __dp4a(in, kW_IN, i0 * u0i));
        const uint32_t u1q = __dp4a(qp, kW_QP, __dp4a(qn, kW_QN, i0 * u0q));
        if (later) { B.s0i += u0i; B.s0q += u0q; B.s1i += u1i; B.s1q += u1q; }
        else       { A.s0i += u0i; A.s0q += u0q; A.s1i += u1i; A.s1q += u1q; }
    }
    if (I::flush) {
        uint4 t;
        t.x = __reduce_add_sync(0xffffffffu, A.s0i);
        t.y = __reduce_add_sync(0xffffffffu, A.s1i);
        t.z = __reduce_add_sync(0xffffffffu, A.s0q);
        t.w = __reduce_add_sync(0xffffffffu, A.s1q);
        if (lane == 0) wsums[I::bF] = t;
        A = B;
        B.s0i = B.s1i = B.s0q = B.s1q = 0u;
    }
}

template <int G, bool kSmem = false>
__device__ __forceinline__ void load_group(uint4 (&buf)[4], const uint4 *base, int lane) {
    buf[0] = load_chunk<4 * G + 0, kSmem>(base, lane);
    buf[1] = load_chunk<4 * G + 1, kSmem>(base, lane);
    buf[2] = load_chunk<4 * G + 2, kSmem>(base, lane);
    buf[3] = load_chunk<4 * G + 3, kSmem>(base, lane);
}
template <int G>
__device__ __forceinline__ void process_group(const uint4 (&buf)[4], int lane, uint32_t lane8, Acc &A, Acc &B, uint4 *wsums) {
    process_chunk<4 * G + 0>(buf[0], lane, lane8, A, B, wsums);
    process_chunk<4 * G + 1>(buf[1], lane, lane8, A, B, wsums);
    process_chunk<4 * G + 2>(buf[2], lane, lane8, A, B, wsums);
    process_chunk<4 * G + 3>(buf[3], lane, lane8, A, B, wsums);
}

// byte masks (0xFF where the sample of that byte is >= t) for the four rail words, t = 1..7
__device__ __forceinline__ uint32_t tail_mask(uint32_t sample_idx_word, uint32_t t) {
    uint32_t m = 0;
#pragma unroll
    for (int b = 0; b < 4; ++b)
        if (((sample_idx_word >> (8 * b)) & 0xffu) >= t) m |= 0xffu << (8 * b);
    return m;
}

// One warp, one super-block: 8 block sums into out[0..7].  `base` = the super-block's 751 chunks (global or staged in
// shared memory); `wsums` = 8 x uint4 of per-warp shared scratch.  `release` (kSmem only) is called once every read of
// the staged copy has completed, so the producer may refill the stage while the results are still being written.
template <bool kSmem, class Release>
__device__ __forceinline__ void super_block_sums(const uint4 *base, int lane, uint4 *wsums, BlockSums *__restrict__ out, Release release) {
    const uint32_t lane8 = 8u * (uint32_t)lane;
    Acc A = {0u, 0u, 0u, 0u}, B = {0u, 0u, 0u, 0u};
    uint4 b0[4], b1[4];
    load_group<0, kSmem>(b0, base, lane);
    load_group<1, kSmem>(b1, base, lane);
    process_group<0>(b0, lane, lane8, A, B, wsums);
    load_group<2, kSmem>(b0, base, lane);
    process_group<1>(b1, lane, lane8, A, B, wsums);
    load_group<3, kSmem>(b1, base, lane);
    process_group<2>(b0, lane, lane8, A, B, wsums);
    load_group<4, kSmem>(b0, base, lane);
    process_group<3>(b1, lane, lane8, A, B, wsums);
    load_group<5, kSmem>(b1, base, lane);
    // Boundary fix-up operand: the chunk holding sample 751*beta (beta = 1..7) is summed whole into block beta-1
    // with in-block indices >= 751; its tail (samples t >= t*) is moved into block beta below.
    uint4 wfix = make_uint4(0u, 0u, 0u, 0u);
    uint32_t tstar = 0;
    if (lane < 7) {
        const uint32_t beta = (uint32_t)lane + 1u;
        const uint32_t cstar = (kDecim * beta) >> 3;
        tstar = kDecim * beta - 8u * cstar;  // = 8 - beta, never 0 for beta < 8
        wfix = ld_chunk<kSmem>(base + cstar);
    }
    release();
    process_group<4>(b0, lane, lane8, A, B, wsums);
    process_group<5>(b1, lane, lane8, A, B, wsums);
    __syncwarp();

    uint32_t t0i = 0, t1i = 0, t0q = 0, t1q = 0;
    if (lane < 7) {
        uint32_t ip, in, qp, qn;
        regroup(wfix, ip, in, qp, qn);
        const uint32_t mip = tail_mask(kW_IP, tstar), min_ = tail_mask(kW_IN, tstar);
        const uint32_t mqp = tail_mask(kW_QP, tstar), mqn = tail_mask(kW_QN, tstar);
        t0i = __dp4a(ip, kOnes & mip, __dp4a(in, kOnes & min_, 0u));
        t1i = __dp4a(ip, kW_IP & mip, __dp4a(in, kW_IN & min_, 0u));
        t0q = __dp4a(qp, kOnes & mqp, __dp4a(qn, kOnes & mqn, 0u));
        t1q = __dp4a(qp, kW_QP & mqp, __dp4a(qn, kW_QN & mqn, 0u));
        // leave block beta-1: those samples carried index (751 - t*) + t
        uint4 v = wsums[lane];
        const uint32_t ib = (uint32_t)kDecim - tstar;
        v.x -= t0i; v.y -= ib * t0i + t1i; v.z -= t0q; v.w -= ib * t0q + t1q;
        wsums[lane] = v;
    }
    __syncwarp();
    if (lane < 7) {  // enter block beta with index t - t*
        uint4 v = wsums[lane + 1];
        v.x += t0i; v.y += t1i - tstar * t0i; v.z += t0q; v.w += t1q - tstar * t0q;
        wsums[lane + 1] = v;
    }
    __syncwarp();
    if (lane < 8) {
        const uint4 v = wsums[lane];
        BlockSums o;
        o.s0i = (int32_t)(v.x - kOff0); o.s1i = (int32_t)(v.y - kOff1);
        o.s0q = (int32_t)(v.z - kOff0); o.s1q = (int32_t)(v.w - kOff1);
        out[lane] = o;
    }
    __syncwarp();  // wsums is reused by this warp's next super-block
}

constexpr int kWarpsPerCta = 8;

// Kernel 1: block sums of full, 16-byte aligned super-blocks.  One warp per super-block.
// kMinCtas = 4: 58 registers, 4 CTAs per SM -- the fastest form on the whole GPU (1.372 ms per 128 slots).  kMinCtas = 5: 48 registers
// (five spilled words), 5 CTAs per SM = a quarter more loads in flight per SM: 1.1 % slower on 148 SMs, but on the 116 SMs the
// SM-partitioned executor leaves it -- fewer SMs have to carry the same bytes in flight -- 0.8 % faster (1.463 -> 1.450 ms), and the
// same at the clocks the power cap allows in a long run (launch_cic_block_sums takes the choice from its caller).
template <int kMinCtas>
__global__ void __launch_bounds__(kWarpsPerCta * 32, kMinCtas)
cic_block_sums_kernel(const uint8_t *__restrict__ iq, size_t stream_stride_bytes, int supers_per_stream, size_t sums_stride,
                      BlockSums *__restrict__ sums) {
    __shared__ uint4 s_sums[kWarpsPerCta][8];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int sb = blockIdx.x * kWarpsPerCta + warp;
    if (sb >= supers_per_stream) return;  // whole warp leaves together
    const int stream = blockIdx.y;
    const uint4 *base = reinterpret_cast<const uint4 *>(iq + (size_t)stream * stream_stride_bytes + (size_t)sb * kSuperBytes);
    uint4 *wsums = s_sums[warp];
    super_block_sums<false>(base, lane, wsums, sums + (size_t)stream * sums_stride + (size_t)sb * 8, [] {});
}

// ---- Kernel 1, bulk-copy variant: persistent CTAs, one producer thread + kC consumer warps, kS-stage shared-memory ring ----
// The streaming variant above needs ~1500 resident threads per SM to keep enough loads in flight (128 B per thread), so
// nothing else fits on the SM while it runs.  Here the bytes in flight live in shared memory instead of registers: one
// elected thread issues 12 016-byte cp.async.bulk copies (the TMA engine, SASS UBLKCP) into a ring of kS stages guarded by
// full/empty mbarriers, and kC consumer warps pull staged super-blocks off the ring (LDS.128) and run the same
// PRMT/DP4A/REDUX arithmetic.  One CTA per SM with (kC+1) warps and kS x 12 KB of shared memory sustains the same HBM
// rate and leaves most of the SM's threads, registers and shared memory to the back-end kernels of the previous batch
// (ft8b200_pipe_t overlaps them).  Work is handed out dynamically (global counter, kGrab super-blocks at a time) so SMs
// that are slowed down by co-resident CTAs simply take fewer super-blocks.
constexpr int kStageBytes = 12032;  // 12016 rounded up to a multiple of 128
constexpr int kGrab = 8;

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

template <int kC, int kS>
__global__ void __launch_bounds__((kC + 1) * 32, 1)
cic_block_sums_tma_kernel(const uint8_t *__restrict__ iq, size_t stream_stride_bytes, int supers_per_stream, int total_supers, size_t sums_stride,
                          BlockSums *__restrict__ sums, unsigned int *__restrict__ work_counter) {
    extern __shared__ __align__(128) uint8_t s_ring[];  // kS stages of kStageBytes
    __shared__ __align__(8) uint64_t s_full[kS], s_empty[kS];
    __shared__ int s_item[kS];                    // global super-block index staged in each stage (-1 = no more work)
    __shared__ unsigned int s_next;               // CTA-local sequence number handed to the consumer warps
    __shared__ volatile unsigned int s_issued;    // items the producer has armed so far (consumers never wait on a stage before that)
    __shared__ uint4 s_sums[kC][8];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int k = 0; k < kS; ++k) { mbar_init(&s_full[k], 1); mbar_init(&s_empty[k], 1); }
        s_next = 0;
        s_issued = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();

    if (warp == kC) {  // ---- producer: one thread
        if (lane != 0) return;
        uint32_t j = 0;
        auto src_of = [&](unsigned int item) {
            const unsigned int stream = item / (unsigned int)supers_per_stream, sb = item - stream * (unsigned int)supers_per_stream;
            return iq + (size_t)stream * stream_stride_bytes + (size_t)sb * kSuperBytes;
        };
        // (Requesting the next run into L2 with cp.async.bulk.prefetch.L2 was measured and dropped: 3.4 TB/s instead of 5.3.)
        unsigned int cur = 0, have = 0;
        for (;;) {
            if (have == 0) { cur = atomicAdd(work_counter, (unsigned int)kGrab); have = kGrab; }
            const unsigned int item = cur++;
            --have;
            if (item >= (unsigned int)total_supers) break;
            const uint32_t st = j % kS, ph = (j / kS) & 1u;
            mbar_wait(&s_empty[st], ph ^ 1u);
            s_item[st] = (int)item;
            mbar_arrive_expect_tx(&s_full[st], (uint32_t)kSuperBytes);
            bulk_g2s(s_ring + (size_t)st * kStageBytes, src_of(item), (uint32_t)kSuperBytes, &s_full[st]);
            ++j;
            __threadfence_block();
            s_issued = j;
        }
        for (int c = 0; c < kC; ++c, ++j) {  // one end marker per consumer warp
            const uint32_t st = j % kS, ph = (j / kS) & 1u;
            mbar_wait(&s_empty[st], ph ^ 1u);
            s_item[st] = -1;
            mbar_arrive(&s_full[st]);
            __threadfence_block();
            s_issued = j + 1;
        }
        // every producer has made its last grab once all of them got here: the last one re-arms the counters for the
        // next launch that uses this pair (no memset node between launches)
        if (atomicAdd(work_counter + 1, 1u) == gridDim.x - 1) { work_counter[0] = 0u; work_counter[1] = 0u; }
        return;
    }

    // ---- consumers
    uint4 *wsums = s_sums[warp];
    for (;;) {
        unsigned int j = 0;
        if (lane == 0) j = atomicAdd(&s_next, 1u);
        j = __shfl_sync(0xffffffffu, j, 0);
        const uint32_t st = j % kS, ph = (j / kS) & 1u;
        // A parity wait is only exact when the waiter is at most one phase ahead of the barrier.  Consumers claim items
        // freely, so first wait until the producer has armed item j (then full[st] is in exactly phase j / kS).
        while (s_issued <= j) __nanosleep(32);
        mbar_wait(&s_full[st], ph);
        const int item = s_item[st];
        uint64_t *empty = &s_empty[st];
        if (item < 0) {  // end marker: hand the stage back (the producer may need it for another warp's marker) and leave
            if (lane == 0) mbar_arrive(empty);
            break;
        }
        const int stream = item / supers_per_stream, sb = item - stream * supers_per_stream;
        super_block_sums<true>(reinterpret_cast<const uint4 *>(s_ring + (size_t)st * kStageBytes), lane, wsums,
                               sums + (size_t)stream * sums_stride + (size_t)sb * 8, [empty, lane] {
                                   __syncwarp();  // every lane's shared-memory reads of this stage have been issued and returned
                                   if (lane == 0) mbar_arrive(empty);
                               });
    }
}

// Generic block sums: one warp per 751-sample block, 2-byte loads, any block range / alignment.
// Used for the blocks a stream has outside its full, aligned super-blocks (ragged batch tails and the
// rtlsdr_callback() streams, whose flushes start and end anywhere).  `iq` points at the first byte of the
// first block of stream 0; `phase0` is (global index of that block's first sample) & 3 for the fs/4 mixer.
__global__ void __launch_bounds__(256)
cic_block_sums_generic_kernel(const uint8_t *__restrict__ iq, size_t stream_stride_bytes, uint32_t phase0, int n_blocks, size_t sums_stride,
                              BlockSums *__restrict__ sums) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int rel = blockIdx.x * 8 + warp;
    if (rel >= n_blocks) return;
    const int stream = blockIdx.y;
    const uchar2 *p = reinterpret_cast<const uchar2 *>(iq + (size_t)stream * stream_stride_bytes) + (size_t)rel * kDecim;
    const uint32_t ph = (phase0 + 3u * (uint32_t)rel) & 3u;  // 751 == 3 (mod 4)
    uint32_t s0i = 0, s1i = 0, s0q = 0, s1q = 0;
    for (uint32_t i = lane; i < (uint32_t)kDecim; i += 32) {
        const uchar2 v = p[i];
        const uint32_t a = v.x, b = v.y;
        const uint32_t na = (0u - a) & 0xffu, nb = (0u - b) & 0xffu;  // wrapping int8 negate, offset-128 domain
        uint32_t mi, mq;
        switch ((ph + i) & 3u) {
        case 0: mi = a; mq = b; break;
        case 1: mi = nb; mq = a; break;
        case 2: mi = na; mq = nb; break;
        default: mi = b; mq = na; break;
        }
        s0i += mi; s1i += i * mi; s0q += mq; s1q += i * mq;
    }
    s0i = __reduce_add_sync(0xffffffffu, s0i);
    s1i = __reduce_add_sync(0xffffffffu, s1i);
    s0q = __reduce_add_sync(0xffffffffu, s0q);
    s1q = __reduce_add_sync(0xffffffffu, s1q);
    if (lane == 0) {
        BlockSums o;
        o.s0i = (int32_t)(s0i - kOff0); o.s1i = (int32_t)(s1i - kOff1);
        o.s0q = (int32_t)(s0q - kOff0); o.s1q = (int32_t)(s1q - kOff1);
        sums[(size_t)stream * sums_stride + rel] = o;
    }
}

// Kernel 2: comb (closed form over 4 consecutive block sums) + 57-tap FIR + scale + peak.
// ref: rtlsdr_ft8d.c:162-200.  One CTA = kTilesPerCta tiles of 512 consecutive outputs of one row.
// (FT8B200_COMB_THREADS / FT8B200_COMB_TILES: build-time shape for A/B runs, tools/perf_combfir.py)
#ifndef FT8B200_COMB_THREADS
#define FT8B200_COMB_THREADS 128
#endif
#ifndef FT8B200_COMB_TILES
#define FT8B200_COMB_TILES 2
#endif
constexpr int kPerThread = 4;      // outputs per thread
constexpr int kTileThreads = FT8B200_COMB_THREADS;
constexpr int kTilesPerCta = FT8B200_COMB_TILES;   // consecutive tiles one CTA walks (the next tile's block sums prefetched)
constexpr int kTile = kTileThreads * kPerThread;  // 512 outputs per CTA
constexpr int kHist = kFirTaps - 1;  // 56 FIR history samples; they need kHistBlocks = 56 + 3 block sums

// n_blocks new blocks per stream -> outputs [out_offset, out_offset + n_blocks) of the stream's 48000-sample
// slot buffer (outputs past 48000 are dropped but the filter keeps running, rtlsdr_ft8d.c:196-200).
// zero_fill: also clear [out_offset + n_blocks, 48000) -- what decoder() does before it normalises (:243-246).
// Each thread produces kPerThread consecutive outputs from a register window of the (float)y2 history, so the
// 57-tap FIR costs one shared load per ~4 taps; coefficients sit in constant memory (uniform broadcast).

// (float)((double)sum / (32768.0 * 750)), rtlsdr_ft8d.c:197-198, without the FP64 divide: 24 576 000 = 375 * 2^16, and a float
// quotient sum/375 can neither be nor come within 2^-34 (relative) of a midpoint between two floats (sum has 24 significant
// bits, 375 * midpoint has >= 25 and is odd in its last place), so rounding the exact quotient once to float equals rounding it
// to double first; the 2^-16 is exact while the result stays normal.  Verified over every float mantissa on the CPU
// (tests/test_oracle_golden.py::test_fir_scale_identity); tiny inputs (never produced by the filter) take the FP64 form.
__device__ __forceinline__ float scale_out(float sum) {
    if (fabsf(sum) < 1e-20f) return __double2float_rn(__ddiv_rn((double)sum, 32768.0 * 750));
    return __fmul_rn(__fdiv_rn(sum, 375.0f), 1.52587890625e-05f);
}

// The I and Q rails run the same 57 taps, so a tap is ONE packed multiply and ONE packed add over the {I, Q} pair (SASS FFMA2 with
// a zero addend / FADD2): per lane the same IEEE round-to-nearest product and sum as the scalar FMUL / FADD, 456 instead of 912
// instructions per thread.  A packed instruction keeps the FP32 pipe busy for two cycles but the scheduler for one
// (tools/f32x2_issue_probe.cu: 8 FADD2 + 8 IADD take the 16 cycles of 8 FADD2 alone), so the kernel's other ~600 instructions per
// thread issue in its shadow: 80 -> 70 us per 128 slots on the whole GPU, 0.46 -> 0.35 ms on a 32-SM back partition
// (profiles/perf_combfir_r2y.json) -- once the {I, Q} layout's bank conflicts were gone (swz() below): with them the packed form
// measured exactly as fast as the scalar one.
__constant__ float2 c_fir2[kFirTaps];  // {z[j], z[j]}

// ptxas 12.9 CONTRACTS mul.rn.f32x2 followed by add.rn.f32x2 into one FFMA2 -- with explicit .rn on both and with -fmad=false, which
// it honours for the scalar forms -- and a fused tap does not round the product (tools/f32x2_contract_probe.cu shows the SASS).
// Written as two fused multiply-adds it does not: RN(w * c + 0) IS the rounded product, RN(p * 1 + acc) IS the rounded sum, and
// ptxas turns the second into FADD2 without merging it into the first.  (The only case where w * c + 0 and w * c differ is a
// product of -0, which becomes +0; the accumulator starts at +0 and a sum is -0 only when both terms are, so it never is -0 on
// either path and x + (+0) = x + (-0) for every other x: results are identical bit for bit.)  tests/test_abi.py checks the
// built kernel's SASS for exactly this shape: 57 x kPerThread FFMA2 with an RZ addend and as many FADD2, no other FFMA2.
__device__ __forceinline__ unsigned long long mul2_rn(unsigned long long a, unsigned long long b) {
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(0ull));
    return r;
}
__device__ __forceinline__ unsigned long long add2_rn(unsigned long long a, unsigned long long b) {
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(b), "l"(0x3f8000003f800000ull), "l"(a));   // b * {1, 1} + a
    return r;
}

// Shared-memory placement of the {I, Q} samples: 16-byte chunk c (samples 2c, 2c+1) lives at chunk c ^ ((c >> 3) & 1).  A thread's
// window starts 32 bytes after its neighbour's, so without the swap the 128-bit loads of threads i and i + 4 of a quarter-warp hit
// the same banks (2-way conflict on every load: 5.9 M conflicts per 128-slot launch, the shared-memory data pipe 96 % busy); with it
// every quarter-warp covers all 32 banks, for every window position (checked exhaustively in tests/test_abi.py::test_fir_window_placement_is_conflict_free).
__device__ __forceinline__ unsigned swz(unsigned c) { return c ^ ((c >> 3) & 1u); }

template <int kN>
__device__ __forceinline__ void fir_window2(const float2 *__restrict__ y, unsigned chunk0, float (&acc_i)[kN], float (&acc_q)[kN]) {
    // y[0 .. kN+55] = {(float)Iy2, (float)Qy2}: acc[o] = sum_j y[o+j]*z[j], strictly sequential in j, product rounded before the
    // add (no FMA): rtlsdr_ft8d.c:179-192 for both rails at once
    unsigned long long w[kN + kHist], acc[kN];
#pragma unroll
    for (int v = 0; v < (kN + kHist) / 2; ++v) {
        const unsigned c = chunk0 + v;   // 16-byte chunk {y[2c], y[2c+1]}
        const ulonglong2 q = reinterpret_cast<const ulonglong2 *>(y)[swz(c)];
        w[2 * v] = q.x; w[2 * v + 1] = q.y;
    }
#pragma unroll
    for (int o = 0; o < kN; ++o) acc[o] = 0ull;  // {0.0f, 0.0f}
#pragma unroll
    for (int j = 0; j < kFirTaps; ++j) {
        const unsigned long long c = *reinterpret_cast<const unsigned long long *>(&c_fir2[j]);
#pragma unroll
        for (int o = 0; o < kN; ++o) acc[o] = add2_rn(acc[o], mul2_rn(w[o + j], c));
    }
#pragma unroll
    for (int o = 0; o < kN; ++o) {
        acc_i[o] = __uint_as_float((unsigned int)(acc[o] & 0xffffffffull));
        acc_q[o] = __uint_as_float((unsigned int)(acc[o] >> 32));
    }
}

// Slot segments of a continuous stream (BASELINE config #5: consecutive 15 s slots of one receiver): with segs > 1 the
// row blockIdx.y is (stream, segment); segment g takes the outputs whose decimation instant 750 + 751*k falls inside
// input samples [g*seg_samples, (g+1)*seg_samples) -- what the daemon gets when main() flips the rx buffer every 15 s
// between two callbacks (rtlsdr_ft8d.c:1339-1354) -- i.e. 47 936 or 47 937 outputs per slot.  Because the filter has no
// integrator state, a segment simply starts reading block sums further into the stream; its FIR/comb history is the
// real preceding blocks.
__device__ __forceinline__ int seg_first_block(int seg, long long seg_samples) {
    const long long first_sample = (long long)seg * seg_samples;
    return first_sample <= 750 ? 0 : (int)((first_sample - 750 + kDecim - 1) / kDecim);
}

// One CTA walks kTilesPerCta consecutive tiles of a row.  The block sums of a tile (k0-59 .. k0+kTile-1) go to shared memory with
// 16-byte cp.async copies -- all of a tile's global reads in flight at once, no registers held -- and the NEXT tile's copies are
// issued before the current tile is filtered, so after a CTA's first tile no warp waits for global memory.  (The loop this
// replaces loaded four block sums per output and waited for them trip by trip, five dependent round trips to L2/HBM per CTA: a
// third of the kernel's stall samples, profiles/ncu_lines_cic_comb_fir_kernel_r2v.txt.)
__device__ __forceinline__ void stage_block_sums(BlockSums *s_b, const BlockSums *__restrict__ s, int k0, int n_blocks) {
    // `s` points at this flush's block 0; the kHistBlocks entries before it hold the previous blocks of the stream (zeros for a
    // fresh filter state), so no lower index test is needed
    for (int i = threadIdx.x; i < kTile + kHistBlocks; i += kTileThreads) {
        const int kk = k0 - kHistBlocks + i;
        if (kk < n_blocks) {
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(&s_b[i])), "l"(s + kk) : "memory");
        } else {
            s_b[i] = BlockSums{0, 0, 0, 0};
        }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
}

__global__ void __launch_bounds__(kTileThreads)
cic_comb_fir_kernel(const BlockSums *__restrict__ sums, size_t sums_stride, int n_blocks, int out_offset, int zero_fill, int segs,
                    long long seg_samples, int n_tiles, float *__restrict__ out_i, float *__restrict__ out_q, uint32_t *__restrict__ count,
                    float *__restrict__ peak, int32_t *__restrict__ y2_out) {
    __shared__ __align__(16) float2 s_y[kTile + kHist];  // {(float)Iy2, (float)Qy2}, rtlsdr_ft8d.c:189-190
    __shared__ __align__(16) BlockSums s_b[kTilesPerCta > 1 ? 2 : 1][kTile + kHistBlocks];
    const int stream = blockIdx.y;  // output row: (receiver stream, segment)
    const BlockSums *s = sums + (size_t)(stream / segs) * sums_stride;
    if (segs > 1) {
        const int seg = stream % segs;
        const int b0 = seg_first_block(seg, seg_samples);
        int b1 = seg_first_block(seg + 1, seg_samples);
        if (b1 > n_blocks) b1 = n_blocks;
        n_blocks = b1 > b0 ? b1 - b0 : 0;
        s += b0;
    }
    const int tile0 = blockIdx.x * kTilesPerCta;
    int tile_end = tile0 + kTilesPerCta;
    if (tile_end > n_tiles) tile_end = n_tiles;
    float m = 0.0f;   // the row's peak over this CTA's tiles
    stage_block_sums(s_b[0], s, tile0 * kTile, n_blocks);
    for (int tile = tile0; tile < tile_end; ++tile) {
        const int k0 = tile * kTile;
        const BlockSums *sb = s_b[(tile - tile0) & (kTilesPerCta > 1 ? 1 : 0)];
        if (kTilesPerCta > 1 && tile + 1 < tile_end) {
            // the other buffer was last read by the comb of tile - 1, which every thread left through the barrier behind it
            stage_block_sums(s_b[(tile + 1 - tile0) & 1], s, k0 + kTile, n_blocks);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();   // this tile's block sums have landed; every thread is done with the previous tile's s_y
        // comb, rtlsdr_ft8d.c:162-176 in closed form over 4 consecutive block sums (DESIGN 2.1):
        //   y2[k] = (751 S0 - S1)[k] + (1502 S0 - S1)[k-1] + (751 S0 + S1)[k-2] + S1[k-3]   (mod 2^32)
        for (int idx = threadIdx.x; idx < kTile + kHist; idx += kTileThreads) {
            const int k = k0 - kHist + idx;  // >= -56: inside the history prefix
            int32_t yi = 0, yq = 0;
            if (k < n_blocks) {
                const BlockSums c0 = sb[idx + 3], c1 = sb[idx + 2], c2 = sb[idx + 1], c3 = sb[idx];
                yi = (int32_t)((751u * (uint32_t)c0.s0i - (uint32_t)c0.s1i) + (1502u * (uint32_t)c1.s0i - (uint32_t)c1.s1i) +
                               (751u * (uint32_t)c2.s0i + (uint32_t)c2.s1i) + (uint32_t)c3.s1i);
                yq = (int32_t)((751u * (uint32_t)c0.s0q - (uint32_t)c0.s1q) + (1502u * (uint32_t)c1.s0q - (uint32_t)c1.s1q) +
                               (751u * (uint32_t)c2.s0q + (uint32_t)c2.s1q) + (uint32_t)c3.s1q);
            }
            s_y[2 * swz((unsigned)idx >> 1) + (idx & 1)] = make_float2(__int2float_rn(yi), __int2float_rn(yq));
            if (y2_out && k >= k0 && k < n_blocks && out_offset + k < kSlot) {
                y2_out[((size_t)stream * kSlot + out_offset + k) * 2 + 0] = yi;
                y2_out[((size_t)stream * kSlot + out_offset + k) * 2 + 1] = yq;
            }
        }
        __syncthreads();
        const int kb = k0 + threadIdx.x * kPerThread;  // first of this thread's outputs
        float vi[kPerThread], vq[kPerThread];
#pragma unroll
        for (int o = 0; o < kPerThread; ++o) { vi[o] = 0.0f; vq[o] = 0.0f; }
        if (kb < n_blocks && out_offset + kb < kSlot) {
            float ai[kPerThread], aq[kPerThread];
            fir_window2<kPerThread>(s_y, threadIdx.x * (kPerThread / 2), ai, aq);
#pragma unroll
            for (int o = 0; o < kPerThread; ++o) {
                if (kb + o < n_blocks) {
                    vi[o] = scale_out(ai[o]);  // rtlsdr_ft8d.c:197-198
                    vq[o] = scale_out(aq[o]);
                }
            }
        }
#pragma unroll
        for (int o = 0; o < kPerThread; ++o) {
            const int k = kb + o, pos = out_offset + k;
            if (pos < kSlot && (k < n_blocks || zero_fill)) {
                out_i[(size_t)stream * kSlot + pos] = vi[o];
                out_q[(size_t)stream * kSlot + pos] = vq[o];
            }
            m = fmaxf(m, fmaxf(fabsf(vi[o]), fabsf(vq[o])));
        }
    }
#pragma unroll
    for (int sh = 16; sh > 0; sh >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, sh));
    if ((threadIdx.x & 31) == 0 && peak && m > 0.0f) atomicMax(reinterpret_cast<unsigned int *>(peak + stream), __float_as_uint(m));
    if (count && blockIdx.x == 0 && threadIdx.x == 0) {
        const int n_out = out_offset + n_blocks;
        count[stream] = (uint32_t)(n_out < kSlot ? n_out : kSlot);
    }
}

// keep the last kHistBlocks sums of a flush as the history prefix of the next one (regions may overlap)
__global__ void shift_history_kernel(BlockSums *sums, int n_blocks) {
    // sums points at the history prefix: entries [0, kHistBlocks) history, [kHistBlocks, kHistBlocks + n_blocks) new
    const int t = threadIdx.x;
    BlockSums v = {};
    if (t < kHistBlocks) v = sums[n_blocks + t];
    __syncthreads();
    if (t < kHistBlocks) sums[t] = v;
}

// a4 as a standalone pass (the fused pipeline applies the scale inside the waterfall load instead)
__global__ void condition_kernel(float *__restrict__ d_i, float *__restrict__ d_q, const float *__restrict__ peak) {
    const int slot = blockIdx.y;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    float p = peak[slot];
    if (!(p > 1e-24f)) p = 1e-24f;
    const float scale = __double2float_rn(__ddiv_rn(0.5, (double)p));
    if (k < kSlot) {
        d_i[(size_t)slot * kSlot + k] = __fmul_rn(d_i[(size_t)slot * kSlot + k], scale);
        d_q[(size_t)slot * kSlot + k] = __fmul_rn(d_q[(size_t)slot * kSlot + k], scale);
    }
}

}  // namespace

// counter pairs {next super-block, finished CTAs} for the bulk-copy kernel: zeroed once, re-armed by the kernel itself
constexpr int kCounterPairs = 256;
static unsigned int *counter_pool(int dev) {
    static unsigned int *pool[64] = {};
    if (dev < 0 || dev >= 64) return nullptr;
    if (!pool[dev]) {
        if (cudaMalloc(&pool[dev], kCounterPairs * 2 * sizeof(unsigned int)) != cudaSuccess) return nullptr;
        cudaMemset(pool[dev], 0, kCounterPairs * 2 * sizeof(unsigned int));
    }
    return pool[dev];
}

template <int kC, int kS>
static cudaError_t launch_tma(const uint8_t *d_iq, size_t stream_stride_bytes, int n_streams, int supers, BlockSums *d_sums, size_t sums_stride,
                              int sm_count, unsigned int *counter, cudaStream_t st) {
    const int smem = kS * kStageBytes;
    {   // the opt-in is per device (and cheap): set it on whichever device is current, every time
        cudaError_t e = cudaFuncSetAttribute(cic_block_sums_tma_kernel<kC, kS>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
    }
    const long total = (long)supers * n_streams;
    int grid = sm_count;
    if ((long)grid * kC > total) grid = (int)((total + kC - 1) / kC);
    cic_block_sums_tma_kernel<kC, kS><<<grid, (kC + 1) * 32, smem, st>>>(d_iq, stream_stride_bytes, supers, (int)total, sums_stride, d_sums, counter);
    return cudaGetLastError();
}

// Block sums of `blocks_per_stream` blocks per stream, streams starting at a super-block boundary of their
// sample stream (mixer phase 0).  d_sums points at block 0 of stream 0 (history prefix before it).
// variant 0: streaming kernel (one warp per super-block, grid over all of them); variant >= 1: persistent bulk-copy
// kernel (shape selected by the variant number), for running underneath other kernels.
cudaError_t launch_cic_block_sums(const uint8_t *d_iq, size_t stream_stride_bytes, int n_streams, int blocks_per_stream, BlockSums *d_sums,
                                  size_t sums_stride, int variant, int sm_count, cudaStream_t st, int *launches) {
    const int supers = blocks_per_stream / 8;
    if (supers > 0 && variant >= 1 && (long)supers * n_streams < (1l << 31)) {   // (kK1StreamingDense is negative: the streaming branch below)
        static std::atomic<unsigned int> next_pair{0};  // contexts and lanes on any host thread draw from one pool
        int dev = 0;
        cudaGetDevice(&dev);
        unsigned int *pool = counter_pool(dev);
        if (!pool) return cudaErrorMemoryAllocation;
        unsigned int *counter = pool + 2 * (next_pair.fetch_add(1u) % kCounterPairs);
        cudaError_t e;
        switch (variant) {
        case 2: e = launch_tma<12, 8>(d_iq, stream_stride_bytes, n_streams, supers, d_sums, sums_stride, sm_count, counter, st); break;
        case 3: e = launch_tma<16, 8>(d_iq, stream_stride_bytes, n_streams, supers, d_sums, sums_stride, sm_count, counter, st); break;
        case 4: e = launch_tma<6, 4>(d_iq, stream_stride_bytes, n_streams, supers, d_sums, sums_stride, sm_count, counter, st); break;
        case 5: e = launch_tma<8, 10>(d_iq, stream_stride_bytes, n_streams, supers, d_sums, sums_stride, sm_count, counter, st); break;
        case 6: e = launch_tma<16, 12>(d_iq, stream_stride_bytes, n_streams, supers, d_sums, sums_stride, sm_count, counter, st); break;
        default: e = launch_tma<8, 6>(d_iq, stream_stride_bytes, n_streams, supers, d_sums, sums_stride, sm_count, counter, st); break;
        }
        if (e != cudaSuccess) return e;
        ++*launches;
    } else if (supers > 0) {
        dim3 grid((supers + kWarpsPerCta - 1) / kWarpsPerCta, n_streams);
        // (Requesting the rest of a warp's super-block into L2 at its start -- prefetch.global.L2, one 128-byte line per lane, SASS CCTL.PF2 --
        // was measured in the last session of round 2 and dropped like the bulk prefetch of the ring variant: 1.48 -> 1.65 ms per 128
        // slots with 4 KB, 1.73 with 8 KB requested ahead on 116 SMs, 1.375 -> 1.645 on the whole GPU; profiles/k1_prefetch_r2zb.txt.)
        if (variant == kK1StreamingDense) cic_block_sums_kernel<5><<<grid, kWarpsPerCta * 32, 0, st>>>(d_iq, stream_stride_bytes, supers, sums_stride, d_sums);
        else cic_block_sums_kernel<4><<<grid, kWarpsPerCta * 32, 0, st>>>(d_iq, stream_stride_bytes, supers, sums_stride, d_sums);
        ++*launches;
    }
    const int rest = blocks_per_stream - supers * 8;
    if (rest > 0) {
        dim3 grid((rest + 7) / 8, n_streams);
        cic_block_sums_generic_kernel<<<grid, 256, 0, st>>>(d_iq + (size_t)supers * kSuperBytes, stream_stride_bytes, 0u, rest, sums_stride,
                                                            d_sums + (size_t)supers * 8);
        ++*launches;
    }
    return cudaGetLastError();
}

cudaError_t launch_cic_block_sums_generic(const uint8_t *d_iq_first_block, size_t stream_stride_bytes, int n_streams, uint32_t phase0, int n_blocks,
                                          BlockSums *d_sums_first_block, size_t sums_stride, cudaStream_t st, int *launches) {
    if (n_blocks > 0) {
        dim3 grid((n_blocks + 7) / 8, n_streams);
        cic_block_sums_generic_kernel<<<grid, 256, 0, st>>>(d_iq_first_block, stream_stride_bytes, phase0, n_blocks, sums_stride, d_sums_first_block);
        ++*launches;
    }
    return cudaGetLastError();
}

cudaError_t launch_cic_comb_fir(const BlockSums *d_sums, size_t sums_stride, int n_blocks, int out_offset, bool zero_fill, int n_streams,
                                float *d_i, float *d_q, uint32_t *d_count, float *d_peak, int32_t *d_y2, cudaStream_t st,
                                int *launches, int segs, long long seg_samples) {
    int span = n_blocks;
    if (segs > 1) span = (int)(seg_samples / kDecim) + 2;  // outputs of one segment
    if (zero_fill && kSlot - out_offset > span) span = kSlot - out_offset;
    if (span <= 0) return cudaSuccess;
    if (segs < 1) segs = 1;
    const int n_tiles = (span + kTile - 1) / kTile;
    dim3 grid((n_tiles + kTilesPerCta - 1) / kTilesPerCta, n_streams * segs);
    cic_comb_fir_kernel<<<grid, kTileThreads, 0, st>>>(d_sums, sums_stride, n_blocks, out_offset, zero_fill ? 1 : 0, segs, seg_samples, n_tiles, d_i,
                                                       d_q, d_count, d_peak, d_y2);
    ++*launches;
    return cudaGetLastError();
}

// The 57 FIR coefficients live in constant memory: uploaded once per device when a context or stream is created on it
// (ft8b200_create / ft8b200_stream_create), with a device synchronisation behind the copy -- never lazily next to the first
// launch, where a pageable copy on the legacy stream would not be ordered against a non-blocking stream.
cudaError_t upload_fir_constants() {
    static std::mutex mu;
    static bool done[64] = {};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    std::lock_guard<std::mutex> lk(mu);
    if (done[dev]) return cudaSuccess;
    float z[kFirTaps];
    build_fir(z);
    float2 z2[kFirTaps];
    for (int j = 0; j < kFirTaps; ++j) z2[j] = make_float2(z[j], z[j]);
    e = cudaMemcpyToSymbol(c_fir2, z2, sizeof(z2));
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess) done[dev] = true;
    return e;
}

cudaError_t launch_shift_history(BlockSums *d_sums_with_prefix, int n_blocks, cudaStream_t st, int *launches) {
    shift_history_kernel<<<1, 64, 0, st>>>(d_sums_with_prefix, n_blocks);
    ++*launches;
    return cudaGetLastError();
}

cudaError_t launch_condition(float *d_i, float *d_q, const float *d_peak, int n_slots, cudaStream_t st, int *launches) {
    for (int s0 = 0; s0 < n_slots; s0 += kMaxGridRows) {   // the slot is blockIdx.y
        const int rows = n_slots - s0 < kMaxGridRows ? n_slots - s0 : kMaxGridRows;
        const size_t o = (size_t)s0 * kSlot;
        condition_kernel<<<dim3((kSlot + 255) / 256, rows), 256, 0, st>>>(d_i + o, d_q + o, d_peak + s0);
        ++*launches;
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

}  // namespace ft8b200
