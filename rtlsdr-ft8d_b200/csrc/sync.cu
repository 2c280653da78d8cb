// sync.cu -- Costas 7x7 sync scoring over the whole waterfall + exact top-K candidate selection.
// Replaces ft8_find_sync() / ft8_sync_score() / heapify_*(), /root/reference/ft8_lib/ft8/decode.c:35-108,
// 173-234, 388-435.
//
// The score kernels (a few CTAs per slot) stage their part of the slot's waterfall in shared memory, score their share of the
// tosr*fosr*36*(bins-7) positions, store the scores in the reference's loop order (time_sub, freq_sub, time_offset,
// freq_offset) and append every position with score >= min_score to the slot's survivor list.  sync_select_kernel (one small
// CTA per slot) sorts the survivors back into loop order and one thread replays the reference's min-heap insertions and the
// final heap sort over them.  The replay is what makes the retained set at the cut score and the order among equal scores
// identical to the reference (they depend on heap history).  The surviving candidates are also appended to a flat work list
// for the decode kernel.
#include "common.cuh"

namespace ft8b200 {
namespace {

constexpr int kSyncThreads = 128;  // small CTAs: the heap replay is one thread's latency, so many slots should be resident per SM

struct Geo { int nb, nbins, tosr, fosr, stride, nfo, npos; uint32_t nfo_magic, fosr_magic; };  // x / d == umulhi(x, magic) for x < 2^20, d < 2^12

// A heap entry is the survivor word itself: (position << 12) | (score & 0xfff) -- position = index in the reference's loop
// order (< 2^20), score sign-extended from 12 bits.  Comparisons look at the score only, exactly like the reference's
// heap[a].score < heap[b].score, so equal scores compare equal whatever their position.
__device__ __forceinline__ int ent_score(uint32_t v) { return ((int)(v << 20)) >> 20; }

// ref: heapify_down, decode.c:388-415 -- the element at the root sinks while a child is STRICTLY smaller (left child first,
// the right one only if smaller than the left).  "Hole" form of the reference's swap chain: the sinking element is always
// the one compared against, so moving children up and storing it once at the end performs the same comparisons and leaves
// the same array.  Both children are loaded before either is examined (one shared-memory latency per level, not two).
__device__ __forceinline__ void sift_down(uint32_t *h, int n) {
    const uint32_t x = h[0];
    const int xs = ent_score(x);
    int cur = 0;
    for (;;) {
        const int l = 2 * cur + 1, r = l + 1;
        if (l >= n) break;
        const uint32_t vl = h[l], vr = h[r < n ? r : l];
        int ps = xs, pick = cur;
        uint32_t pv = x;
        if (ent_score(vl) < ps) { ps = ent_score(vl); pick = l; pv = vl; }
        if (r < n && ent_score(vr) < ps) { pick = r; pv = vr; }
        if (pick == cur) break;
        h[cur] = pv;
        cur = pick;
    }
    h[cur] = x;
}
// ref: heapify_up, decode.c:417-435 -- the last element rises while STRICTLY smaller than its parent
__device__ __forceinline__ void sift_up(uint32_t *h, int n, uint32_t x) {
    const int xs = ent_score(x);
    int cur = n - 1;
    while (cur > 0) {
        const int par = (cur - 1) >> 1;
        const uint32_t pv = h[par];
        if (xs >= ent_score(pv)) break;
        h[cur] = pv;
        cur = par;
    }
    h[cur] = x;
}

// The exact top-K selection of one slot (ref: ft8_find_sync, decode.c:173-234).
//
// The reference visits the positions in loop order and keeps a min-heap of the best K: push while there is room; once the heap
// is full a position enters only if its score is STRICTLY above the root's, evicting the root; a final heap sort orders the
// result.  Which positions are retained at the cut score, and the order among equal scores, depend on that history, so the
// pushes/evictions are replayed by one thread exactly as the reference performs them -- but ONLY those: a position that fails
// `score >= min_score` (or, with a full heap, `score > root`) is a no-op in the reference and is skipped wholesale here.
//
// Survivors come from the score kernels themselves: every position with score >= min_score is appended (warp-aggregated
// atomicAdd) to the slot's list as (position << 12) | score.  The list is unordered, but positions are distinct, so sorting the
// 32-bit words ascending restores the reference's visiting order (bitonic sort in shared memory).  A slot with more than
// kListCap survivors (min_score <= 0 on noise: every other position) takes the scan path instead: warp 0 walks the score array
// in position order, 256 positions per step, and tests them against `min_score` (heap not full) or the root (full) -- still no
// serial step for a position that does nothing.  Neither path needs a scratch list in global memory.
//
// Tried and measured in round 2, not kept: running the selection as the TAIL of the score kernel (the last CTA of a slot to
// finish, found with one atomic counter per slot, selects for that slot).  It saves a launch, but a tail holds a score CTA's
// 73 KB of shared memory while one thread replays the heap: equal at 128 slots (57.5 vs 57.3 us for the stage), 12 % slower at
// 4096 (1.261 vs 1.123 ms), where the separate kernel keeps 16 small CTAs per SM in flight and their serial parts overlap.
struct SelArgs {
    uint32_t *lists;          // [n_slots][kListCap] survivor words
    int *count;               // [n_slots] survivors appended (may exceed kListCap: overflow -> scan path)
    int max_cand, min_score;
    candidate_t *cand_out;    // [n_slots][max_cand]
    int *ncand_out;           // [n_slots]
    uint32_t *work;           // flat decode work list (may be null)
    unsigned int *work_total; // its counter
};

__device__ __forceinline__ uint32_t survivor_word(int pos, int score) { return ((uint32_t)pos << 12) | ((uint32_t)score & 0xfffu); }

// Called by all 32 lanes of a warp (converged).  `s_over` is a per-CTA flag in shared memory: once a CTA has seen the slot's
// count pass kListCap it stops issuing atomics (the count only has to END above the cap for the selection to take the scan path).
__device__ __forceinline__ void emit_survivor(const SelArgs &sa, int slot, bool pass, uint32_t word, volatile int *s_over) {
    const unsigned b = __ballot_sync(0xffffffffu, pass);
    if (b == 0) return;
    const int lane = threadIdx.x & 31, leader = __ffs((int)b) - 1, n = __popc(b);
    int base = 0;
    if (lane == leader) {
        base = *s_over ? kListCap : atomicAdd(sa.count + slot, n);
        if (base + n > kListCap) *s_over = 1;
    }
    base = __shfl_sync(0xffffffffu, base, leader);
    if (pass) {
        const int at = base + __popc(b & ((1u << lane) - 1u));
        if (at < kListCap) sa.lists[(size_t)slot * kListCap + at] = word;
    }
}

// ref: the pop + push of a full heap, decode.c:203-216 (last element to the root, sift down, newcomer appended, sift up)
__device__ __forceinline__ void heap_replace_root(uint32_t *heap, int max_cand, uint32_t word) {
    heap[0] = heap[max_cand - 1];
    sift_down(heap, max_cand - 1);
    sift_up(heap, max_cand, word);
}

// `dyn` = at least max_cand*4 (16-byte aligned up) + kListCap*4 bytes of shared memory, free for this call.  All kThreads threads
// of the CTA call it.  Scores and list words come from the score kernel: read through L2 (__ldcg), they are used once.
template <int kThreads>
__device__ void select_slot(const int16_t *__restrict__ scores, const Geo &g, const SelArgs &sa, int slot, uint8_t *dyn) {
    __shared__ int s_total, s_base;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int max_cand = sa.max_cand, min_score = sa.min_score;
    uint32_t *heap = reinterpret_cast<uint32_t *>(dyn);
    uint32_t *surv = reinterpret_cast<uint32_t *>(dyn + (((size_t)max_cand * 4 + 15) & ~(size_t)15));
    // warp 0 fetches the first 32 list words together with the count (one L2 round trip instead of two for the usual slot)
    const uint32_t first = warp == 0 ? __ldcg(sa.lists + (size_t)slot * kListCap + lane) : 0u;
    const int n_list = __ldcg(sa.count + slot);
    const bool listed = n_list <= kListCap, small = n_list <= 32;

    if (listed && !small) {
        // the slot's survivors, sorted by position (= by word: positions are distinct and sit in the high bits)
        int m = 64;
        while (m < n_list) m <<= 1;
        for (int i = tid; i < m; i += kThreads) surv[i] = i < n_list ? __ldcg(sa.lists + (size_t)slot * kListCap + i) : 0xffffffffu;
        __syncthreads();
        for (int k = 2; k <= m; k <<= 1)
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int i = tid; i < m; i += kThreads) {
                    const int ixj = i ^ j;
                    if (ixj > i) {
                        const uint32_t a = surv[i], b = surv[ixj];
                        if (((i & k) == 0) ? (a > b) : (a < b)) { surv[i] = b; surv[ixj] = a; }
                    }
                }
                __syncthreads();
            }
    }

    if (warp == 0) {
        int n = 0;
        if (small) {  // the usual slot (a few signals): sorted in registers, no block barrier before the replay
            uint32_t v = lane < n_list ? first : 0xffffffffu;
#pragma unroll
            for (int k = 2; k <= 32; k <<= 1)
#pragma unroll
                for (int j = k >> 1; j > 0; j >>= 1) {
                    const uint32_t o = __shfl_xor_sync(0xffffffffu, v, j);
                    const bool keep_min = ((lane & j) == 0) == ((lane & k) == 0);
                    v = keep_min ? (v < o ? v : o) : (v > o ? v : o);
                }
            surv[lane] = v;
            __syncwarp();
        }
        if (max_cand > 0 && listed) {
            // (a) room in the heap: every survivor is pushed (one thread; nothing to skip)
            const int n_fill = n_list < max_cand ? n_list : max_cand;
            if (lane == 0)
                for (int e = 0; e < n_fill; ++e) sift_up(heap, e + 1, surv[e]);
            n = n_fill;
            // (b) heap full: 32 survivors per step against the root score, which only ever rises
            if (n_list > max_cand) {
                __syncwarp();
                int root = __shfl_sync(0xffffffffu, lane == 0 ? ent_score(heap[0]) : 0, 0);   // only lane 0 touches the heap
                for (int base = max_cand; base < n_list; base += 32) {
                    const int e = base + lane;
                    const uint32_t v = e < n_list ? surv[e] : 0u;
                    const int sc = ent_score(v);
                    unsigned todo = __ballot_sync(0xffffffffu, e < n_list && sc > root);
                    while (todo) {
                        const int src = __ffs((int)todo) - 1;
                        const uint32_t vv = __shfl_sync(0xffffffffu, v, src);
                        if (lane == 0) {
                            heap_replace_root(heap, max_cand, vv);
                            root = ent_score(heap[0]);
                        }
                        root = __shfl_sync(0xffffffffu, root, 0);
                        todo &= ~((2u << src) - 1u);                                   // lanes up to src are settled
                        todo &= __ballot_sync(0xffffffffu, e < n_list && sc > root);   // the others face the new root
                    }
                }
            }
        } else if (max_cand > 0) {
            // scan path: 8 consecutive positions per lane and step (256 per warp step), four steps of loads in flight;
            // `need` = the score a position must reach to act: min_score while the heap has room, root + 1 once it is full
            const bool vec = (g.npos & 7) == 0 && (((size_t)scores) & 15) == 0;
            auto load8 = [&](int base) -> uint4 {   // eight int16 scores, packed as they lie in memory
                const int p0 = base + 8 * lane;
                if (p0 >= g.npos) return make_uint4(0u, 0u, 0u, 0u);
                if (vec) return __ldcg(reinterpret_cast<const uint4 *>(scores + p0));
                uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    if (p0 + j < g.npos) w[j >> 1] |= ((uint32_t)(uint16_t)__ldcg(scores + p0 + j)) << (16 * (j & 1));
                return make_uint4(w[0], w[1], w[2], w[3]);
            };
            int need = min_score;
            uint4 ring[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) ring[u] = load8(256 * u);
            for (int base0 = 0; base0 < g.npos; base0 += 1024) {
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int base = base0 + 256 * u;
                    if (base >= g.npos) break;
                    const uint4 raw = ring[u];
                    ring[u] = load8(base + 1024);
                    const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
                    int cur[8];
#pragma unroll
                    for (int j = 0; j < 4; ++j) { cur[2 * j] = (int)(short)(w[j] & 0xffffu); cur[2 * j + 1] = (int)(short)(w[j] >> 16); }
                    const int left = g.npos - (base + 8 * lane);                   // positions of this lane inside the slot
                    const unsigned valid = left >= 8 ? 0xffu : (left > 0 ? (1u << left) - 1u : 0u);
                    unsigned m = 0;
#pragma unroll
                    for (int j = 0; j < 8; ++j) m |= (cur[j] >= need ? 1u : 0u) << j;
                    m &= valid;
                    unsigned lanes = __ballot_sync(0xffffffffu, m != 0);
                    while (lanes) {
                        const int src = __ffs((int)lanes) - 1;
                        const int j = __ffs((int)__shfl_sync(0xffffffffu, m, src)) - 1;
                        int mine = 0;
#pragma unroll
                        for (int q = 0; q < 8; ++q) mine = q == j ? cur[q] : mine;
                        const int sc = __shfl_sync(0xffffffffu, mine, src);
                        if (lane == 0) {
                            const uint32_t word = survivor_word(base + 8 * src + j, sc);
                            if (n < max_cand) sift_up(heap, n + 1, word);
                            else heap_replace_root(heap, max_cand, word);
                        }
                        if (n < max_cand) ++n;
                        if (n == max_cand) {
                            int root = lane == 0 ? ent_score(heap[0]) : 0;
                            root = __shfl_sync(0xffffffffu, root, 0);
                            need = root + 1;                                          // strictly above the root
                        }
                        if (lane == src) m &= ~((2u << j) - 1u);                      // this lane's positions up to j are settled
                        unsigned still = 0;
#pragma unroll
                        for (int q = 0; q < 8; ++q) still |= (cur[q] >= need ? 1u : 0u) << q;
                        m &= still;
                        lanes = __ballot_sync(0xffffffffu, m != 0);
                    }
                }
            }
        }
        if (lane == 0) {
            for (int rest = n; rest > 1;) {  // heap sort -> descending score (decode.c:219-231)
                const uint32_t t = heap[rest - 1]; heap[rest - 1] = heap[0]; heap[0] = t;
                --rest;
                sift_down(heap, rest);
            }
            s_total = n;
            sa.ncand_out[slot] = n;
            s_base = (sa.work && n > 0) ? (int)atomicAdd(sa.work_total, (unsigned int)n) : 0;
        }
    }
    __syncthreads();
    {
        // position -> (time_sub, freq_sub, time_offset, freq_offset), by all threads, off the serial path
        const int n = s_total;
        unsigned long long *dst = reinterpret_cast<unsigned long long *>(sa.cand_out + (size_t)slot * max_cand);
        for (int k = tid; k < max_cand; k += kThreads) {
            unsigned long long c = 0ull;
            if (k < n) {  // candidate_t as one 64-bit word: score | time_offset<<16 | freq_offset<<32 | time_sub<<48 | freq_sub<<56
                const uint32_t v = heap[k];
                const int score = ent_score(v), p = (int)(v >> 12);
                int q = g.nfo_magic ? (int)__umulhi((uint32_t)p, g.nfo_magic) : p;   // p / nfo (exact: p < 2^20, nfo < 2^12; magic 0 = divide by 1)
                const int fo = p - q * g.nfo;
                const int q36 = q / 36;
                const int to = q - 36 * q36 - 12;
                const int ts = g.fosr_magic ? (int)__umulhi((uint32_t)q36, g.fosr_magic) : q36, fs = q36 - ts * g.fosr;
                c = ((unsigned long long)(uint16_t)(short)score) | ((unsigned long long)(uint16_t)(short)to << 16) |
                    ((unsigned long long)(uint16_t)(short)fo << 32) | ((unsigned long long)(uint8_t)ts << 48) | ((unsigned long long)(uint8_t)fs << 56);
            }
            dst[k] = c;
        }
        if (sa.work)
            for (int k = tid; k < n; k += kThreads) sa.work[s_base + k] = (uint32_t)slot * (uint32_t)max_cand + (uint32_t)k;
    }
    __syncthreads();
}

// One CTA per slot (looping over slots).
__global__ void __launch_bounds__(kSyncThreads, 8)
sync_select_kernel(const int16_t *__restrict__ scores_all, int n_slots, Geo g, SelArgs sa) {
    extern __shared__ __align__(16) uint8_t smem[];
    for (int slot = blockIdx.x; slot < n_slots; slot += gridDim.x) select_slot<kSyncThreads>(scores_all + (size_t)slot * g.npos, g, sa, slot, smem);
}

// Phase 1: score every position.  For a fixed (time_sub, freq_sub) every byte a score touches lies in ONE sub-plane of
// the waterfall: mag[((row*tosr + ts)*fosr + fs)*nbins + bin] for row < nb, bin < nbins (nb x nbins bytes: 23.5 KB for
// the daemon geometry, 89 KB for the 12 kHz monitor).  grid = (planes * splits, slots): a CTA stages its plane compactly
// in shared memory ([row][bin]) and scores the positions of that plane for its share of the 36 time offsets; thread t
// owns frequency offsets t, t + blockDim, ... so a warp reads 32 consecutive bytes per access (one wavefront) and the
// row-range tests are uniform across the CTA.  Scores go to global memory as int16 in the reference's loop order.
constexpr int kScoreThreads = 256;

// ref: ft8_sync_score(), decode.c:44-108 / ft4_sync_score(), decode.c:110-171, on the compact plane (`nbins` = row pitch)
// FT8: 3 groups of 7 symbols at 0, 36, 72 sharing one Costas array, 8 tones.  FT4: 4 groups of 4 symbols at 1, 34, 67,
// 100, one Costas array per group, 4 tones.
template <int kBins, bool kFt4>
__device__ __forceinline__ int sync_score_plane(const uint8_t *__restrict__ plane, int nb, int nbins_rt, int to, int fo) {
    const int nbins = kBins > 0 ? kBins : nbins_rt;
    constexpr int kGroups = kFt4 ? 4 : 3, kLen = kFt4 ? 4 : 7, kFirst = kFt4 ? 1 : 0, kStep = kFt4 ? 33 : 36, kTop = kFt4 ? 3 : 7;
    constexpr int kCostas8[7] = {3, 1, 4, 0, 6, 5, 2};
    constexpr int kCostas4[4][4] = {{0, 1, 3, 2}, {1, 0, 2, 3}, {2, 3, 1, 0}, {3, 2, 0, 1}};
    int score = 0, terms = 0;
#pragma unroll
    for (int grp = 0; grp < kGroups; ++grp) {
#pragma unroll
        for (int k = 0; k < kLen; ++k) {
            const int row = to + kFirst + kStep * grp + k;
            if (row < 0) continue;
            if (row >= nb) break;  // leaves this group only, like the reference's inner `break`
            const int tone = kFt4 ? kCostas4[grp][k < 4 ? k : 0] : kCostas8[k];
            const uint8_t *p = plane + row * nbins + fo + tone;
            const int centre = p[0];
            if (tone > 0) { score += centre - p[-1]; ++terms; }
            if (tone < kTop) { score += centre - p[1]; ++terms; }
            if (k > 0 && row > 0) { score += centre - p[-nbins]; ++terms; }
            if (k + 1 < kLen && row + 1 < nb) { score += centre - p[nbins]; ++terms; }
        }
    }
    if (terms > 0) score /= terms;  // truncating division
    return score;
}

template <int kBins, bool kStage, bool kFt4>
__global__ void __launch_bounds__(kScoreThreads)
sync_score_kernel(const uint8_t *__restrict__ mag_all, size_t slot_stride, Geo g, int splits, int to_per_cta, int16_t *__restrict__ scores_all,
                  SelArgs sa) {
    extern __shared__ __align__(16) uint8_t smem[];
    __shared__ int s_over;
    const int tid = threadIdx.x;
    if (tid == 0) s_over = 0;
    if (!kStage) __syncthreads();
    const int slot = blockIdx.y;
    const int plane_id = blockIdx.x / splits, split = blockIdx.x - plane_id * splits;  // plane_id = ts*fosr + fs
    const int nbins = kBins > 0 ? kBins : g.nbins;
    const uint8_t *gplane = mag_all + (size_t)slot * slot_stride + (size_t)plane_id * nbins;  // row r at gplane + r*stride
    const int to0 = -12 + split * to_per_cta;
    int to1 = to0 + to_per_cta;
    if (to1 > 24) to1 = 24;
    const uint8_t *plane;
    int pitch;
    if (kStage) {
        // rows this CTA can touch: [to0 - 1, (to1 - 1) + last sync symbol + 1], clipped (last sync symbol: 78 FT8, 103 FT4)
        int r0 = to0 - 1, r1 = to1 + (kFt4 ? 104 : 79);
        if (r0 < 0) r0 = 0;
        if (r1 > g.nb) r1 = g.nb;
        if (((((size_t)gplane) | (size_t)g.stride | (size_t)nbins) & 15) == 0) {
            const int vec_per_row = nbins >> 4;
            for (int v = tid; v < (r1 - r0) * vec_per_row; v += kScoreThreads) {
                const int r = r0 + v / vec_per_row, c = v - (v / vec_per_row) * vec_per_row;
                reinterpret_cast<uint4 *>(smem + (size_t)r * nbins)[c] = __ldg(reinterpret_cast<const uint4 *>(gplane + (size_t)r * g.stride) + c);
            }
        } else {
            for (int v = tid; v < (r1 - r0) * nbins; v += kScoreThreads) {
                const int r = r0 + v / nbins, c = v - (v / nbins) * nbins;
                smem[(size_t)r * nbins + c] = gplane[(size_t)r * g.stride + c];
            }
        }
        plane = smem;
        pitch = nbins;
        __syncthreads();
    } else {
        plane = gplane;
        pitch = g.stride;
    }
    const int pos0 = plane_id * 36 * g.nfo;
    int16_t *scores = scores_all + (size_t)slot * g.npos + pos0;
    for (int to = to0; to < to1; ++to) {
        for (int f0 = 0; f0 < g.nfo; f0 += kScoreThreads) {   // CTA-uniform trip count: emit_survivor() is a whole-warp call
            const int fo = f0 + tid;
            int sc = 0;
            if (fo < g.nfo) {
                sc = kStage ? sync_score_plane<kBins, kFt4>(plane, g.nb, pitch, to, fo) : sync_score_plane<0, kFt4>(plane, g.nb, pitch, to, fo);
                scores[(to + 12) * g.nfo + fo] = (int16_t)sc;  // stored as int16_t in candidate_t
            }
            emit_survivor(sa, slot, fo < g.nfo && sc >= sa.min_score, survivor_word(pos0 + (to + 12) * g.nfo + fo, sc), &s_over);
        }
    }
}

// FT8 fast path.  Every term of a score is a difference between a cell P[r][c] and one of its four neighbours, and WHICH
// neighbours take part depends only on the Costas index k (k = 0 has no earlier symbol, k = 6 no later one, k = 3 is tone 0
// and has no lower neighbour; tone 7 never occurs) and on the row being the first/last of the waterfall.  So the CTA first
// turns its tile of the plane into four 16-bit planes, with a = P - P[c+1], b = P - P[c-1], u = r > 0 ? P - P[r-1] : 0,
// d = r + 1 < nb ? P - P[r+1] : 0:
//     W0 = a + b + d   (k = 0)     Wm = a + b + u + d   (k = 1,2,4,5)     W3 = a + u + d   (k = 3)     W6 = a + b + u   (k = 6)
// each stored with a bias of +256 per difference (so two cells are computed per 32-bit integer operation without borrows between the halves)
// and with 12 rows before and >= 10 rows after the waterfall holding the biased zero: the reference's `row < 0 -> continue` and
// `row >= nb -> break` become zero contributions, and a score is 21 loads at compile-time offsets plus 21 adds, minus the 75 biases.
// The number of terms it is divided by depends on the time offset only (exact truncating division by multiply-high).
// The sums are the same integers as the reference's, so the scores are too.
// grid = (planes * tiles, slots); a tile is kTileF frequency offsets (all 36 time offsets, all rows).
constexpr int kTileF = 64;
constexpr int kTilePitch = kTileF + 8;   // 16-bit elements per derived row (71 needed: fo .. fo + 6), 18 groups of 4
constexpr int kRawPitch = kTileF + 32;   // raw bytes per row: columns fo0 - 16 .. fo0 + 79, whole 16-byte chunks of the waterfall row
constexpr int kRawLead = 16;             // columns staged before fo0 (4 are needed; 16 keeps the chunks aligned)
constexpr int kPadBefore = 12;           // time offsets start at -12
constexpr uint32_t kBias4 = 0x04000400u; // biased zero of the four-difference plane (two cells): 4 x 256
constexpr uint32_t kBias3 = 0x03000300u; // ... of the three-difference planes
constexpr int kBiasPerScore = 3 * (4 * 1024 + 3 * 768);  // 3 groups x (k = 1,2,4,5 on Wm, k = 0,3,6 on W0/W3/W6)
__host__ __device__ constexpr int fast_rows(int nb) { return kPadBefore + (nb > 102 ? nb : 102); }  // last row touched: 23 + 72 + 6

// Number of terms a score at time offset to = ti - 12 is divided by (ft8_sync_score's num_average), as 2^32 / terms + 1 for the
// multiply-high division (0: one term or none, no division).  It depends on the waterfall's height only, so the host fills it
// in once per launch (computed by 36 threads of every CTA it was a serial prologue the other 220 threads waited for: 22 % of
// the kernel's stall samples).
struct TermMagic { uint32_t m[36]; };
static TermMagic term_magic(int nb) {
    TermMagic tm;
    for (int ti = 0; ti < 36; ++ti) {
        const int to = ti - 12;
        int terms = 0;
        for (int grp = 0; grp < 3; ++grp)
            for (int k = 0; k < 7; ++k) {
                const int row = to + 36 * grp + k;
                if (row < 0) continue;
                if (row >= nb) break;
                terms += (k == 3 ? 1 : 2) + ((k > 0 && row > 0) ? 1 : 0) + ((k < 6 && row + 1 < nb) ? 1 : 0);
            }
        tm.m[ti] = terms > 1 ? (0xffffffffu / (uint32_t)terms + 1u) : 0u;
    }
    return tm;
}

// two 16-bit lanes per word, every lane stays non-negative: a' = P + 256 - N in [1, 511]
__device__ __forceinline__ uint32_t diff2(uint32_t p2, uint32_t n2) { return p2 + 0x01000100u - n2; }

__global__ void __launch_bounds__(kScoreThreads)
sync_score_ft8_kernel(const uint8_t *__restrict__ mag_all, size_t slot_stride, Geo g, int tiles, int16_t *__restrict__ scores_all, SelArgs sa,
                      const TermMagic tm) {
    extern __shared__ __align__(16) uint8_t smem[];
    __shared__ int s_over;
    const int tid = threadIdx.x, slot = blockIdx.y;
    if (tid == 0) s_over = 0;
    const int plane_id = blockIdx.x / tiles, tile = blockIdx.x - plane_id * tiles;
    const int fo0 = tile * kTileF;
    const int nb = g.nb, nbins = g.nbins;
    const int rows = fast_rows(nb);
    uint8_t *raw = smem;                                                   // [nb][kRawPitch]
    uint16_t *w0 = reinterpret_cast<uint16_t *>(smem + (((size_t)nb * kRawPitch + 15) & ~(size_t)15));
    const int plane_elems = rows * kTilePitch;
    const uint8_t *gplane = mag_all + (size_t)slot * slot_stride + (size_t)plane_id * nbins;  // row r at gplane + r*stride

    // raw tile: columns [fo0 - 16, fo0 + 80), zero outside [0, nbins).  All of a thread's copies are in flight at once (cp.async):
    // with one load -> one store per loop trip this phase was 30 % of the kernel (a chain of L2 round trips per thread).
    constexpr int kWordsPerRow = kRawPitch / 4;
    if (((((size_t)gplane) | (size_t)g.stride | (size_t)nbins) & 15) == 0) {
        constexpr int kChunks = kRawPitch / 16, kRowsPerTrip = kScoreThreads / kChunks;   // 6 chunks per row, 42 rows per trip
        if (tid < kChunks * kRowsPerTrip) {
            const int r0 = tid / kChunks, j = tid - r0 * kChunks;
            const int c = fo0 - kRawLead + 16 * j;
            const bool inside = c >= 0 && c + 16 <= nbins;   // nbins and c are multiples of 16: a chunk is never split
            for (int r = r0; r < nb; r += kRowsPerTrip) {
                uint8_t *dst = raw + (size_t)r * kRawPitch + 16 * j;
                if (inside) {
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)),
                                 "l"(gplane + (size_t)r * g.stride + c) : "memory");
                } else {
                    *reinterpret_cast<uint4 *>(dst) = make_uint4(0u, 0u, 0u, 0u);
                }
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
    } else {
        for (int v = tid; v < nb * kWordsPerRow; v += kScoreThreads) {
            const int r = v / kWordsPerRow, wi = v - r * kWordsPerRow;
            const int c = fo0 - kRawLead + 4 * wi;
            uint32_t word = 0;
            if (c >= 0 && c + 4 <= nbins) word = __ldg(reinterpret_cast<const uint32_t *>(gplane + (size_t)r * g.stride + c));
            reinterpret_cast<uint32_t *>(raw + (size_t)r * kRawPitch)[wi] = word;
        }
    }
    __syncthreads();
    constexpr int kGroups = kTilePitch / 4;  // 18 groups of 4 cells per row
    constexpr int kPrepRows = kScoreThreads / kGroups;   // 14 rows per trip (252 threads busy): no division inside the loop
    const int rp0 = tid / kGroups, q = tid - rp0 * kGroups;
    for (int rp = rp0; rp < rows && rp0 < kPrepRows; rp += kPrepRows) {
        const int r = rp - kPadBefore;
        uint2 o0, om, o3, o6;
        if (r < 0 || r >= nb) {
            om = make_uint2(kBias4, kBias4);
            o0 = o3 = o6 = make_uint2(kBias3, kBias3);
        } else {
            // words: [0] left, [1] the 4 cells (columns fo0 + 4q ..), [2] right
            const uint32_t *row = reinterpret_cast<const uint32_t *>(raw + (size_t)r * kRawPitch) + (kRawLead / 4 - 1) + q;
            const uint32_t wl = row[0], wc = row[1], wr = row[2];
            const uint32_t p01 = __byte_perm(wc, 0u, 0x4140), p23 = __byte_perm(wc, 0u, 0x4342);    // (P0,P1) (P2,P3) as 16-bit lanes
            const uint32_t l01 = __byte_perm(p01, wl, 0x1017), l23 = __byte_perm(wc, 0u, 0x4241);   // (P-1,P0) (P1,P2); p01/p23 supply the zero bytes
            const uint32_t r23 = __byte_perm(p23, wr, 0x1412);                                      // (P3,P4)
            const uint32_t a01 = diff2(p01, l23), a23 = diff2(p23, r23);   // P - right neighbour (right of (P0,P1) is (P1,P2))
            const uint32_t b01 = diff2(p01, l01), b23 = diff2(p23, l23);   // P - left neighbour
            uint32_t u01 = 0x01000100u, u23 = 0x01000100u, d01 = 0x01000100u, d23 = 0x01000100u;
            if (r > 0) {
                const uint32_t wu = row[-kWordsPerRow + 1];
                u01 = diff2(p01, __byte_perm(wu, 0u, 0x4140)); u23 = diff2(p23, __byte_perm(wu, 0u, 0x4342));
            }
            if (r + 1 < nb) {
                const uint32_t wd = row[kWordsPerRow + 1];
                d01 = diff2(p01, __byte_perm(wd, 0u, 0x4140)); d23 = diff2(p23, __byte_perm(wd, 0u, 0x4342));
            }
            const uint32_t ab01 = a01 + b01, ab23 = a23 + b23, ud01 = u01 + d01, ud23 = u23 + d23;
            o0 = make_uint2(ab01 + d01, ab23 + d23);
            om = make_uint2(ab01 + ud01, ab23 + ud23);
            o3 = make_uint2(a01 + ud01, a23 + ud23);
            o6 = make_uint2(ab01 + u01, ab23 + u23);
        }
        uint2 *dst = reinterpret_cast<uint2 *>(w0 + (size_t)rp * kTilePitch) + q;
        dst[0] = o0;
        dst[plane_elems / 4] = om;
        dst[2 * (plane_elems / 4)] = o3;
        dst[3 * (plane_elems / 4)] = o6;
    }
    __syncthreads();
    const int fl = tid & (kTileF - 1), fo = fo0 + fl;
    const bool valid = fo < g.nfo;   // the other threads of the last tile still score (cells inside the tile) but store nothing
    const int pos0 = plane_id * 36 * g.nfo;
    int16_t *scores = scores_all + (size_t)slot * g.npos + pos0;
    constexpr int kCostas8[7] = {3, 1, 4, 0, 6, 5, 2};
    // A thread scores its frequency offset at kPerThread time offsets ti0, ti0 + 4, ... (warp-uniform; padded row = ti + 36 grp + k).
    // Fully unrolled: the 21 x 9 loads are immediates off four base registers.  Survivors are rare, so they are looked for once
    // per thread after the loop (one ballot per warp) instead of once per score.
    constexpr int kTiStep = kScoreThreads / kTileF, kPerThread = 36 / kTiStep;
    static_assert(kTiStep * kPerThread == 36, "time offsets must divide evenly among the threads of a column");
    const int ti0 = tid / kTileF;
    const uint16_t *b0 = w0 + ti0 * kTilePitch + fl, *bm = b0 + plane_elems, *b3 = bm + plane_elems, *b6 = b3 + plane_elems;
    int16_t *out = scores + ti0 * g.nfo + fo;
    const int out_step = kTiStep * g.nfo;
    int sc[kPerThread];
    bool any = false;
#pragma unroll
    for (int i = 0; i < kPerThread; ++i) {
        const int row0 = i * kTiStep * kTilePitch;
        int sum = 0;
#pragma unroll
        for (int grp = 0; grp < 3; ++grp) {
#pragma unroll
            for (int k = 0; k < 7; ++k) {
                const uint16_t *w = k == 0 ? b0 : (k == 3 ? b3 : (k == 6 ? b6 : bm));
                sum += w[row0 + (36 * grp + k) * kTilePitch + kCostas8[k]];
            }
        }
        int score = sum - kBiasPerScore;
        const uint32_t magic = tm.m[ti0 + i * kTiStep];
        if (magic) {  // truncating division by the number of terms
            const uint32_t mag_q = __umulhi((uint32_t)abs(score), magic);
            score = score < 0 ? -(int)mag_q : (int)mag_q;
        }
        sc[i] = score;
        if (valid) out[i * out_step] = (int16_t)score;
        any |= score >= sa.min_score;
    }
    if (__ballot_sync(0xffffffffu, any && valid)) {
#pragma unroll
        for (int i = 0; i < kPerThread; ++i)
            emit_survivor(sa, slot, valid && sc[i] >= sa.min_score, survivor_word(pos0 + (ti0 + i * kTiStep) * g.nfo + fo, sc[i]), &s_over);
    }
}

}  // namespace

size_t find_sync_list_bytes(int n_slots) { return ((size_t)n_slots + (size_t)n_slots * kListCap) * sizeof(uint32_t); }

cudaError_t launch_find_sync(const uint8_t *d_mag, size_t slot_stride, int n_slots, int num_blocks, int num_bins, int time_osr, int freq_osr,
                             int protocol, int max_cand, int min_score, candidate_t *d_cand, int *d_ncand, int16_t *d_scores, uint32_t *d_lists,
                             uint32_t *d_work, unsigned int *d_work_total, int sm_count, cudaStream_t st, int *launches) {
    Geo g;
    g.nb = num_blocks; g.nbins = num_bins; g.tosr = time_osr; g.fosr = freq_osr;
    g.stride = time_osr * freq_osr * num_bins;
    g.nfo = num_bins - 7;
    g.npos = time_osr * freq_osr * 36 * g.nfo;
    if (g.nfo < 1) {
        // fewer than 8 bins: the reference's `freq_offset + 7 < num_bins` loop (decode.c:189) never runs -> no candidates, no error
        cudaError_t e0 = cudaMemsetAsync(d_ncand, 0, (size_t)n_slots * sizeof(int), st);
        if (e0 == cudaSuccess && d_work_total) e0 = cudaMemsetAsync(d_work_total, 0, 5 * sizeof(unsigned int), st);
        return e0;
    }
    if (g.nfo >= 4096 || freq_osr >= 4096 || g.npos >= (1 << 20)) return cudaErrorInvalidValue;
    g.nfo_magic = g.nfo > 1 ? 0xffffffffu / (uint32_t)g.nfo + 1u : 0u;   // 0: division by 1
    g.fosr_magic = freq_osr > 1 ? 0xffffffffu / (uint32_t)freq_osr + 1u : 0u;
    SelArgs sa;
    sa.count = reinterpret_cast<int *>(d_lists);                  // layout: count[n_slots] | words[n_slots][kListCap]
    sa.lists = d_lists + n_slots;
    sa.max_cand = max_cand; sa.min_score = min_score;
    sa.cand_out = d_cand; sa.ncand_out = d_ncand;
    sa.work = d_work; sa.work_total = d_work_total;
    cudaError_t e = cudaMemsetAsync(sa.count, 0, (size_t)n_slots * sizeof(int), st);
    if (e != cudaSuccess) return e;
    // one CTA per (slot, sub-plane, share of the 36 time offsets); enough CTAs to fill the machine for small batches
    const int planes = time_osr * freq_osr;
    int splits = (4 * sm_count + n_slots * planes - 1) / (n_slots * planes);
    if (splits > 6) splits = 6;
    if (splits < 1) splits = 1;
    const int to_per_cta = (36 + splits - 1) / splits;
    splits = (36 + to_per_cta - 1) / to_per_cta;
    const size_t staged = ((size_t)g.nb * g.nbins + 15) & ~(size_t)15;
    const bool ft4 = protocol == PROTO_FT4;
    const size_t fast_smem = (((size_t)g.nb * kRawPitch + 15) & ~(size_t)15) + (size_t)4 * fast_rows(g.nb) * kTilePitch * sizeof(int16_t);
    // the slot is blockIdx.y: a batch of more than kMaxGridRows slots is scored by consecutive launches, each over slots
    // [s0, s0 + rows) with its pointers moved to slot s0 (one launch, exactly as before, for every smaller batch)
    for (int s0 = 0; s0 < n_slots; s0 += kMaxGridRows) {
        const int rows = n_slots - s0 < kMaxGridRows ? n_slots - s0 : kMaxGridRows;
        const uint8_t *mag = d_mag + (size_t)s0 * slot_stride;
        int16_t *scores = d_scores + (size_t)s0 * g.npos;
        SelArgs sc = sa;
        sc.count += s0;
        sc.lists += (size_t)s0 * kListCap;
        const dim3 grid(planes * splits, rows);
        if (!ft4 && fast_smem <= 96 * 1024 && (((size_t)d_mag | slot_stride | (size_t)g.stride | (size_t)g.nbins) & 3) == 0) {
            // FT8 fast path: derived int16 planes per (plane, tile of 64 frequency offsets)
            const int tiles = (g.nfo + kTileF - 1) / kTileF;
            e = cudaFuncSetAttribute(sync_score_ft8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
            if (e != cudaSuccess) return e;
            sync_score_ft8_kernel<<<dim3(planes * tiles, rows), kScoreThreads, fast_smem, st>>>(mag, slot_stride, g, tiles, scores, sc, term_magic(g.nb));
        } else if (staged <= 200 * 1024) {
            if (g.nbins == 256 && !ft4) {
                sync_score_kernel<256, true, false><<<grid, kScoreThreads, staged, st>>>(mag, slot_stride, g, splits, to_per_cta, scores, sc);
            } else {
                auto kern = ft4 ? sync_score_kernel<0, true, true> : sync_score_kernel<0, true, false>;
                if (staged > 48 * 1024 && (e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)staged)) != cudaSuccess) return e;
                kern<<<grid, kScoreThreads, staged, st>>>(mag, slot_stride, g, splits, to_per_cta, scores, sc);
            }
        } else {
            auto kern = ft4 ? sync_score_kernel<0, false, true> : sync_score_kernel<0, false, false>;
            kern<<<grid, kScoreThreads, 0, st>>>(mag, slot_stride, g, splits, to_per_cta, scores, sc);
        }
        ++*launches;
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    if (d_work_total) {
        // [0] items, [1] next item (decode_kernel), [2] - [4] the pull counters of OSD, AP (osd_kernel, rebp_kernel) and finesync_kernel
        e = cudaMemsetAsync(d_work_total, 0, 5 * sizeof(unsigned int), st);
        if (e != cudaSuccess) return e;
    }
    // the selection's shared memory: heap + survivors
    const size_t sel_smem = (((size_t)max_cand * 4 + 15) & ~(size_t)15) + (size_t)kListCap * sizeof(uint32_t);
    if (sel_smem > 200 * 1024) return cudaErrorInvalidValue;
    int sgrid = sm_count * 12;  // 128-thread CTAs looping over the slots
    if (sgrid > n_slots) sgrid = n_slots;
    if (sel_smem > 48 * 1024 && (e = cudaFuncSetAttribute(sync_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sel_smem)) != cudaSuccess) return e;
    sync_select_kernel<<<sgrid, kSyncThreads, sel_smem, st>>>(d_scores, n_slots, g, sa);
    ++*launches;
    return cudaGetLastError();
}

}  // namespace ft8b200
