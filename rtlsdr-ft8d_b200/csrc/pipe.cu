// pipe.cu -- ft8b200_pipe_t: a small in-order executor that keeps several slot batches in flight on one GPU.
//
// Why: one batch through ft8b200_process_raw() is an HBM-bound front end (cic_block_sums + comb/FIR, ~11 us per slot)
// followed by a latency/issue-bound back end (waterfall, sync, LDPC, spot table) that uses almost no DRAM bandwidth.
// Run back to back they leave the memory system idle for a third of the step, and every step also pays the host's
// launch latency and the blocking D2H of the spot records.  The pipe owns `depth` lanes (one ft8b200_ctx_t each: private
// workspaces, a launching stream and a high-priority side stream for the back end) and chains them so that
//   * the front end of batch n+1 starts as soon as the front end of batch n has been issued and finished
//     (front ends never compete with each other for DRAM),
//   * the back end of batch n runs on its lane's high-priority stream underneath the front end of batch n+1,
//   * host input (ft8b200_pipe_submit_host) is copied H2D on the lane's own stream, so the PCIe copy of batch n+1
//     overlaps all of batch n's kernels, and
//   * spot records return through pinned per-lane buffers with an async D2H; the host only blocks in collect().
// Results are bit-identical to the unpipelined calls (tests/test_gpu_parity.py::test_pipe_*): the kernels and their
// per-batch buffers are the same, only the stream topology differs.
//
// Reference counterpart: the daemon's double-buffered rx_state + decoder thread (rtlsdr_ft8d.c:221-285, 1336-1354),
// i.e. "receive slot n+1 while slot n decodes" -- here across batches of slots on one GPU.
#include "common.cuh"

#include <cuda.h>  // types and prototypes only: the driver entry points are resolved through cudaGetDriverEntryPoint, libcuda is not linked
#include <stdlib.h>
#include <string.h>

#include <chrono>
#include <mutex>
#include <string>
#include <vector>

namespace {

struct Lane {
    ft8b200_ctx_t *ctx = nullptr;
    cudaStream_t st = nullptr;
    uint8_t *d_raw = nullptr;
    size_t raw_bytes = 0;
    float *d_fi = nullptr, *d_fq = nullptr;   // host-submitted 3200 sps slots (ft8b200_pipe_submit_slots_host)
    size_t f_slots = 0;
    struct decoder_results *h_res = nullptr;
    int32_t *h_n = nullptr;
    size_t res_slots = 0;
    cudaEvent_t done = nullptr;
    int n_slots = 0;
    CUstream part_front = nullptr, part_back = nullptr;  // streams of the two SM partitions (ft8b200_pipe_set_partition)
};

// Spatial partition of the GPU (CUDA green contexts): the HBM-bound front end (cic_block_sums, comb+FIR) of batch n+1 owns
// `front_sms` SMs, the issue/latency-bound back end (waterfall, sync, LDPC, spots) of batch n owns the other `back_sms`.
// Time-sharing the same SMs was measured not to pay (the back-end CTAs displace decimator CTAs, whose loads in flight are
// what saturates HBM); with disjoint SM sets the decimator keeps its residency and the back end runs in its shadow.
struct Partition {
    CUgreenCtx front = nullptr, back = nullptr;
    int front_sms = 0, back_sms = 0;
};

struct DriverApi {
    decltype(&cuDeviceGet) DeviceGet = nullptr;
    decltype(&cuDeviceGetDevResource) DeviceGetDevResource = nullptr;
    decltype(&cuDevSmResourceSplitByCount) DevSmResourceSplitByCount = nullptr;
    decltype(&cuDevResourceGenerateDesc) DevResourceGenerateDesc = nullptr;
    decltype(&cuGreenCtxCreate) GreenCtxCreate = nullptr;
    decltype(&cuGreenCtxDestroy) GreenCtxDestroy = nullptr;
    decltype(&cuGreenCtxStreamCreate) GreenCtxStreamCreate = nullptr;
    decltype(&cuStreamDestroy) StreamDestroy = nullptr;
    bool ok = false;
};

const DriverApi &driver_api() {
    static DriverApi api = [] {
        DriverApi a;
        bool ok = true;
        auto get = [&](const char *name, void **fn) {
            cudaDriverEntryPointQueryResult q;
            if (cudaGetDriverEntryPoint(name, fn, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess || !*fn) ok = false;
        };
        get("cuDeviceGet", reinterpret_cast<void **>(&a.DeviceGet));
        get("cuDeviceGetDevResource", reinterpret_cast<void **>(&a.DeviceGetDevResource));
        get("cuDevSmResourceSplitByCount", reinterpret_cast<void **>(&a.DevSmResourceSplitByCount));
        get("cuDevResourceGenerateDesc", reinterpret_cast<void **>(&a.DevResourceGenerateDesc));
        get("cuGreenCtxCreate", reinterpret_cast<void **>(&a.GreenCtxCreate));
        get("cuGreenCtxDestroy", reinterpret_cast<void **>(&a.GreenCtxDestroy));
        get("cuGreenCtxStreamCreate", reinterpret_cast<void **>(&a.GreenCtxStreamCreate));
        get("cuStreamDestroy", reinterpret_cast<void **>(&a.StreamDestroy));
        a.ok = ok;
        return a;
    }();
    return api;
}

// Green contexts are created once per (device, requested split) and kept for the life of the process: the driver (580.159) does not
// give back the ~4 MiB of device memory a green context holds when cuGreenCtxDestroy is called (tools/greenctx_leak_probe.cu: 8 MiB
// per create/destroy of a front/back pair, with or without streams and launches), so a pipe that is re-partitioned -- the autotune
// walks six splits -- or created and destroyed repeatedly would grow without bound.  Pipes on the same device with the same split
// share the pair (they are confined to the same SM sets, which is what the split asks for); only the lanes' streams are per pipe.
struct CachedPartition {
    int device = 0, back_req = 0;
    Partition part;
};
std::mutex g_part_mu;
std::vector<CachedPartition> g_parts;

}  // namespace

struct ft8b200_pipe {
    ft8b200_config_t cfg;
    std::vector<Lane> lanes;
    int head = 0;    // oldest batch in flight
    int count = 0;   // batches in flight
    cudaEvent_t prev_front = nullptr;  // front-end-done event of the most recently submitted batch
    cudaEvent_t prev_done = nullptr;   // completion event of the most recently submitted batch
    cudaEvent_t prev_back = nullptr;   // back-end-done event of the most recently submitted raw batch
    bool chain_back = false;           // back ends of consecutive batches serialised on the back partition (ft8b200_pipe_set_back_chain)
    int mode = FT8B200_PIPE_OVERLAP;
    cudaEvent_t dependency = nullptr;  // one-shot: the next submit's kernels wait for this event (ft8b200_pipe_depend_on)
    bool profiling = false;
    double stage_ms[6] = {0, 0, 0, 0, 0, 0};
    uint64_t batches = 0, slots = 0;
    cudaEvent_t t_ref = nullptr;           // recorded when profiling is switched on: origin of the timeline
    std::vector<float> timeline;           // 12 floats per collected batch: begin/end of the 6 stages, ms since t_ref
    Partition part;
    std::string err;
};

namespace {

int pfail(ft8b200_pipe_t *p, int code, const std::string &msg) {
    p->err = msg;
    return code;
}

// a decoder setting for every lane's context; refused while batches are in flight.  `func`: the setter's name, for the message
template <class Set>
int set_lanes(ft8b200_pipe_t *p, const char *func, Set set) {
    if (p->count) return pfail(p, FT8B200_EBUSY, std::string(func) + ": batches in flight");
    for (Lane &l : p->lanes)
        if (int rc = set(l.ctx)) return rc;
    return 0;
}

#define PCU(call)                                                                                   \
    do {                                                                                            \
        cudaError_t e__ = (call);                                                                   \
        if (e__ != cudaSuccess) { (void)cudaGetLastError(); return pfail(p, FT8B200_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e__)); } \
    } while (0)

int lane_results(ft8b200_pipe_t *p, Lane &l, int n_slots) {
    if ((size_t)n_slots <= l.res_slots) return 0;
    if (l.h_res) cudaFreeHost(l.h_res);
    if (l.h_n) cudaFreeHost(l.h_n);
    l.h_res = nullptr; l.h_n = nullptr; l.res_slots = 0;
    PCU(cudaMallocHost(&l.h_res, (size_t)n_slots * p->cfg.max_messages * sizeof(struct decoder_results)));
    PCU(cudaMallocHost(&l.h_n, (size_t)n_slots * sizeof(int32_t)));
    l.res_slots = (size_t)n_slots;
    return 0;
}

// queue one batch on the next free lane; `h_iq` (host) or `d_iq` (device) holds the raw IQ.  segs > 1: the n_slots streams are
// continuous receivers cut into `segs` consecutive slots of seg_bytes each (ft8b200_process_raw_streams): n_slots * segs result rows
int submit(ft8b200_pipe_t *p, const uint8_t *h_iq, const uint8_t *d_iq, size_t bytes_per_stream, size_t stride, int n_slots, int segs = 1,
           size_t seg_bytes = 0) {
    if (!p) return FT8B200_BAD_ARG();
    if ((!h_iq && !d_iq) || n_slots < 1 || (bytes_per_stream & 7) || segs < 1) return pfail(p, FT8B200_EINVAL, "ft8b200_pipe_submit: bad argument");
    if ((long long)n_slots * segs > FT8B200_MAX_RAW_ROWS)   // before the host copy and the pinned record buffers are sized for it
        return pfail(p, FT8B200_EINVAL, "ft8b200_pipe_submit: more than FT8B200_MAX_RAW_ROWS (65535) streams or result rows in one batch; split it");
    const int n_rows = n_slots * segs;
    if (p->count == (int)p->lanes.size()) return pfail(p, FT8B200_EBUSY, "ft8b200_pipe_submit: every lane is in flight, collect first");
    PCU(cudaSetDevice(p->cfg.device));
    Lane &l = p->lanes[(p->head + p->count) % p->lanes.size()];
    int rc = lane_results(p, l, n_rows);
    if (rc) return rc;
    if (h_iq) {
        stride = (bytes_per_stream + 15) & ~(size_t)15;
        const size_t need = stride * (size_t)n_slots + 16;
        if (need > l.raw_bytes) {
            if (l.d_raw) cudaFree(l.d_raw);
            l.d_raw = nullptr; l.raw_bytes = 0;
            PCU(cudaMalloc(&l.d_raw, need));
            l.raw_bytes = need;
        }
        if (stride == bytes_per_stream) PCU(cudaMemcpyAsync(l.d_raw, h_iq, bytes_per_stream * n_slots, cudaMemcpyHostToDevice, l.st));
        else PCU(cudaMemcpy2DAsync(l.d_raw, stride, h_iq, bytes_per_stream, bytes_per_stream, n_slots, cudaMemcpyHostToDevice, l.st));
        d_iq = l.d_raw;
    }
    if (p->dependency) {  // e.g. a collective still reading this lane's previous results
        PCU(cudaStreamWaitEvent(l.st, p->dependency, 0));
        p->dependency = nullptr;
    }
    if (p->mode == FT8B200_PIPE_OVERLAP) {
        // front ends are serialised across lanes: this batch's decimator starts when the previous batch's has finished (the wait is
        // placed by the context right in front of its block-sum kernel, behind the memsets that prepare the batch's buffers)
        // (measured in round 2: without the chain consecutive block-sum kernels fill each other's tails and the step gains 0.8 %, but
        // their per-launch times then overlap and no longer say what the kernel achieves -- kept chained)
        if (p->prev_front) ft8b200_set_front_wait(l.ctx, p->prev_front);
        // Optionally (ft8b200_pipe_set_back_chain; the autotune's probe) so are the back ends on an SM partition.  Unchained, the back
        // ends of two batches share the back partition whenever a backlog has built up, and fill each other's tails: a partition that
        // is too small for one batch's back end then looks fine for the first ~70 batches (24 SMs: 1.417 ms per batch in a 72-batch
        // probe, 1.58 in the long run) -- chained, it shows what one back end costs within a dozen batches (1.65).  Unchained is the
        // better executor when the back end does fall behind (81.0 k against 77.4 k slots/s at 24 SMs) and the same when it does not
        // (85.2 / 85.3 k at 32), so that is how batches run; the chain is how partitions are compared.
        if (p->chain_back && p->part.back && p->prev_back) ft8b200_set_back_wait(l.ctx, p->prev_back);
    } else if (p->prev_done) {
        // kernels of consecutive batches never share the GPU; only copies and host work overlap them
        PCU(cudaStreamWaitEvent(l.st, p->prev_done, 0));
    }
    rc = segs > 1 ? ft8b200_process_raw_streams(l.ctx, d_iq, bytes_per_stream, stride, n_slots, segs, seg_bytes, nullptr)
                  : ft8b200_process_raw(l.ctx, d_iq, bytes_per_stream, stride, n_slots, nullptr);
    if (rc) return pfail(p, rc, ft8b200_last_error());
    p->prev_front = reinterpret_cast<cudaEvent_t>(ft8b200_front_event(l.ctx));
    p->prev_back = reinterpret_cast<cudaEvent_t>(ft8b200_back_event(l.ctx));
    if ((rc = ft8b200_fetch_results_async(l.ctx, n_rows, l.h_res, l.h_n, nullptr))) return pfail(p, rc, ft8b200_last_error());
    PCU(cudaEventRecord(l.done, l.st));
    p->prev_done = l.done;
    l.n_slots = n_rows;
    ++p->count;
    return 0;
}

// queue one batch of 3200 sps slots (BASELINE configs #1/#3/#4: the input of ft8_subsystem()) on the next free lane:
// host samples are copied H2D on the lane's stream, then waterfall -> sync -> decode -> spots, records back through the
// lane's pinned buffers.  d_peak != NULL: the samples are unconditioned, decoder()'s 0.5/peak scale is applied on load.
int submit_slots(ft8b200_pipe_t *p, const float *h_i, const float *h_q, const float *d_i, const float *d_q, const float *d_peak, int n_slots) {
    if (!p) return FT8B200_BAD_ARG();
    if (!((h_i && h_q) || (d_i && d_q)) || n_slots < 1) return pfail(p, FT8B200_EINVAL, "ft8b200_pipe_submit_slots: bad argument");
    if (p->count == (int)p->lanes.size()) return pfail(p, FT8B200_EBUSY, "ft8b200_pipe_submit_slots: every lane is in flight, collect first");
    PCU(cudaSetDevice(p->cfg.device));
    Lane &l = p->lanes[(p->head + p->count) % p->lanes.size()];
    int rc = lane_results(p, l, n_slots);
    if (rc) return rc;
    if (h_i) {
        if ((size_t)n_slots > l.f_slots) {
            if (l.d_fi) cudaFree(l.d_fi);
            if (l.d_fq) cudaFree(l.d_fq);
            l.d_fi = l.d_fq = nullptr; l.f_slots = 0;
            PCU(cudaMalloc(&l.d_fi, (size_t)n_slots * ft8b200::kSlot * sizeof(float)));
            PCU(cudaMalloc(&l.d_fq, (size_t)n_slots * ft8b200::kSlot * sizeof(float)));
            l.f_slots = (size_t)n_slots;
        }
        const size_t bytes = (size_t)n_slots * ft8b200::kSlot * sizeof(float);
        PCU(cudaMemcpyAsync(l.d_fi, h_i, bytes, cudaMemcpyHostToDevice, l.st));
        PCU(cudaMemcpyAsync(l.d_fq, h_q, bytes, cudaMemcpyHostToDevice, l.st));
        d_i = l.d_fi; d_q = l.d_fq; d_peak = nullptr;
    }
    if (p->dependency) {
        PCU(cudaStreamWaitEvent(l.st, p->dependency, 0));
        p->dependency = nullptr;
    }
    // there is no HBM-bound front end to keep apart here: in SERIAL mode batches follow each other, otherwise the lanes'
    // streams simply run side by side (copies of batch n+1 under the kernels of batch n)
    if (p->mode == FT8B200_PIPE_SERIAL && p->prev_done) PCU(cudaStreamWaitEvent(l.st, p->prev_done, 0));
    if ((rc = ft8b200_process_conditioned(l.ctx, d_i, d_q, d_peak, n_slots, nullptr))) return pfail(p, rc, ft8b200_last_error());
    p->prev_front = nullptr;
    p->prev_back = nullptr;
    if ((rc = ft8b200_fetch_results_async(l.ctx, n_slots, l.h_res, l.h_n, nullptr))) return pfail(p, rc, ft8b200_last_error());
    PCU(cudaEventRecord(l.done, l.st));
    p->prev_done = l.done;
    l.n_slots = n_slots;
    ++p->count;
    return 0;
}

__global__ void smid_probe_kernel(unsigned int *mask) {
    unsigned int id;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(id));
    const long long t0 = clock64();
    while (clock64() - t0 < 30000) { }   // hold the SM long enough for the grid to spread over every SM of the partition
    if (threadIdx.x == 0 && id < 256) atomicOr(mask + (id >> 5), 1u << (id & 31));
}

}  // namespace

extern "C" {

ft8b200_pipe_t *ft8b200_pipe_create(const ft8b200_config_t *cfg_in, int depth) {
    if (depth < 1 || depth > 8) return nullptr;
    ft8b200_pipe_t *p = new ft8b200_pipe();
    ft8b200_default_config(&p->cfg);
    if (cfg_in) p->cfg = *cfg_in;
    p->lanes.resize((size_t)depth);
    for (Lane &l : p->lanes) {
        l.ctx = ft8b200_create(&p->cfg);  // fails (NULL + ft8b200_last_error) without an sm_100 device: no fallback
        if (!l.ctx || cudaEventCreateWithFlags(&l.done, cudaEventDisableTiming) != cudaSuccess) {
            ft8b200_pipe_destroy(p);
            return nullptr;
        }
        l.st = reinterpret_cast<cudaStream_t>(ft8b200_cuda_stream(l.ctx));
        ft8b200_set_side_backend(l.ctx, depth > 1);
    }
    return p;
}

static void partition_release(ft8b200_pipe_t *p);

int ft8b200_pipe_set_mode(ft8b200_pipe_t *p, int mode, int decimator_variant) {
    if (!p || (mode != FT8B200_PIPE_OVERLAP && mode != FT8B200_PIPE_SERIAL)) return FT8B200_BAD_ARG();
    if (p->count) return pfail(p, FT8B200_EBUSY, "ft8b200_pipe_set_mode: batches in flight");
    if (p->part.front || p->part.back) partition_release(p);  // both modes time-share the whole GPU
    p->mode = mode;
    for (Lane &l : p->lanes) {
        ft8b200_set_side_backend(l.ctx, mode == FT8B200_PIPE_OVERLAP && p->lanes.size() > 1);
        if (decimator_variant >= 0 && ft8b200_set_decimator_variant(l.ctx, decimator_variant)) return pfail(p, FT8B200_EINVAL, ft8b200_last_error());
    }
    p->prev_front = nullptr;
    p->prev_back = nullptr;
    return 0;
}

// drop the SM partition: lanes go back to their own streams, the partition's streams are destroyed
static void partition_release(ft8b200_pipe_t *p) {
    const DriverApi &d = driver_api();
    for (Lane &l : p->lanes) {
        if (!l.part_front && !l.part_back) continue;
        if (l.ctx) {
            ft8b200_set_partition_streams(l.ctx, nullptr, nullptr, 0);  // synchronises both streams first
            l.st = reinterpret_cast<cudaStream_t>(ft8b200_cuda_stream(l.ctx));
        }
        if (l.part_front) d.StreamDestroy(l.part_front);
        if (l.part_back) d.StreamDestroy(l.part_back);
        l.part_front = l.part_back = nullptr;
    }
    p->part = Partition();   // the green contexts stay in g_parts (see CachedPartition)
}

// Which SMs the back partition gets.  Asked for ONE group of back_sms SMs, cuDevSmResourceSplitByCount returns the first groups of its
// enumeration and the rest as the remainder; layout > 0 (encoded by the caller as back_sms + 1000 * layout) asks the driver for groups
// of 8 instead and composes the back partition from groups picked over the enumeration, the front end from all the others plus the
// remainder (cuDevResourceGenerateDesc accepts several SM resources of one split).  Written to find out whether the partitioned
// block-sum kernel's box-to-box spread (0.96-1.00 of the copy peak; alone it is 1.03 everywhere) comes from which SMs it is left with.
// It does not: on a B200 a group of 8 is already one TPC from each of four GPCs (%smid 0,1,16,17,32,33,48,49 ...), the driver's own
// 32 SMs are 8 from each of the four 16-SM GPCs, and no layout beats that outside the probe's noise (profiles/part_layout_r2u.json).
static int pick_groups(int layout, int n_groups, int n_back, int *idx) {
    if (n_back < 1 || n_back >= n_groups) return -1;
    for (int i = 0; i < n_back; ++i) {
        int g;
        switch (layout) {
            case 1: g = (i * n_groups) / n_back; break;                       // evenly spread from the first group
            case 2: g = ((2 * i + 1) * n_groups) / (2 * n_back); break;       // evenly spread, centred
            case 3: g = n_groups - n_back + i; break;                         // the last groups
            case 4: g = 2 * i; break;                                         // every second group from the first
            case 5: g = (i & 1) + (i / 2) * (2 * n_groups / n_back); break;   // neighbouring pairs, spread
            case 6: g = i; break;                                             // the first groups (what layout 0 does, as a control)
            default: return -1;
        }
        if (g < 0 || g >= n_groups) return -1;
        for (int k = 0; k < i; ++k) if (idx[k] == g) return -1;
        idx[i] = g;
    }
    return 0;
}

int ft8b200_pipe_set_partition(ft8b200_pipe_t *p, int back_sms, int *front_sms_out, int *back_sms_out) {
    if (!p || back_sms < 0) return FT8B200_BAD_ARG();
    if (p->count) return pfail(p, FT8B200_EBUSY, "ft8b200_pipe_set_partition: batches in flight");
    PCU(cudaSetDevice(p->cfg.device));
    const DriverApi &d = driver_api();
    if (p->part.front || p->part.back) partition_release(p);
    p->prev_front = nullptr;
    p->prev_back = nullptr;
    const int back_req = back_sms;           // cache key: size and layout
    const int layout = back_sms / 1000;
    back_sms %= 1000;
    if (layout > 6 || (layout > 0 && back_sms == 0)) return pfail(p, FT8B200_EINVAL, "ft8b200_pipe_set_partition: no such SM layout");
    if (back_sms == 0) {
        if (front_sms_out) *front_sms_out = 0;
        if (back_sms_out) *back_sms_out = 0;
        return 0;
    }
    if (p->lanes.size() < 2) return pfail(p, FT8B200_EINVAL, "ft8b200_pipe_set_partition: needs a pipe of depth >= 2");
    if (!d.ok) return pfail(p, FT8B200_ECUDA, "ft8b200_pipe_set_partition: the CUDA driver does not export the green-context API");
#define PDRV(call)                                                                                                  \
    do {                                                                                                            \
        CUresult r__ = (call);                                                                                      \
        if (r__ != CUDA_SUCCESS) {                                                                                  \
            partition_release(p);                                                                                   \
            return pfail(p, FT8B200_ECUDA, std::string(#call) + ": CUresult " + std::to_string((int)r__));          \
        }                                                                                                           \
    } while (0)
    {
        std::lock_guard<std::mutex> lk(g_part_mu);
        const CachedPartition *hit = nullptr;
        for (const CachedPartition &c : g_parts)
            if (c.device == p->cfg.device && c.back_req == back_req) hit = &c;
        if (!hit) {
            CUdevice dev;
            PDRV(d.DeviceGet(&dev, p->cfg.device));
            CUdevResource all;
            PDRV(d.DeviceGetDevResource(dev, &all, CU_DEV_RESOURCE_TYPE_SM));
            if ((unsigned)back_sms >= all.sm.smCount) return pfail(p, FT8B200_EINVAL, "ft8b200_pipe_set_partition: back_sms must leave SMs for the front end");
            CUdevResourceDesc dfront, dback;
            unsigned int n_front_sms = 0, n_back_sms = 0;
            if (layout == 0) {
                CUdevResource back, front;
                unsigned int groups = 1;
                // a size that is not a multiple of the co-scheduling granularity (8 SMs on sm_100) is split TPC-wise (2 SMs): none of the
                // back-end kernels launches thread-block clusters, which is all the coarser granularity guarantees
                const unsigned int flags = (back_sms % 8) ? CU_DEV_SM_RESOURCE_SPLIT_IGNORE_SM_COSCHEDULING : 0;
                PDRV(d.DevSmResourceSplitByCount(&back, &groups, &all, &front, flags, (unsigned)back_sms));  // rounds up to the granularity
                if (groups != 1 || front.sm.smCount == 0) return pfail(p, FT8B200_ECUDA, "ft8b200_pipe_set_partition: the driver could not split the SMs that way");
                PDRV(d.DevResourceGenerateDesc(&dback, &back, 1));
                PDRV(d.DevResourceGenerateDesc(&dfront, &front, 1));
                n_front_sms = front.sm.smCount;
                n_back_sms = back.sm.smCount;
            } else {
                constexpr unsigned kGran = 8, kMaxGroups = 64;
                CUdevResource grp[kMaxGroups], rem, sel_back[kMaxGroups], sel_front[kMaxGroups + 1];
                unsigned int groups = all.sm.smCount / kGran;
                if (groups > kMaxGroups) groups = kMaxGroups;
                memset(&rem, 0, sizeof(rem));
                PDRV(d.DevSmResourceSplitByCount(grp, &groups, &all, &rem, 0, kGran));
                const int n_back = (back_sms + (int)kGran - 1) / (int)kGran;
                int idx[kMaxGroups];
                if (groups < 2 || pick_groups(layout, (int)groups, n_back, idx))
                    return pfail(p, FT8B200_EINVAL, "ft8b200_pipe_set_partition: no such layout for this split");
                unsigned nb = 0, nf = 0;
                for (unsigned g = 0; g < groups; ++g) {
                    bool is_back = false;
                    for (int k = 0; k < n_back; ++k) is_back |= idx[k] == (int)g;
                    if (is_back) { sel_back[nb++] = grp[g]; n_back_sms += grp[g].sm.smCount; }
                    else { sel_front[nf++] = grp[g]; n_front_sms += grp[g].sm.smCount; }
                }
                if (rem.type == CU_DEV_RESOURCE_TYPE_SM && rem.sm.smCount > 0) { sel_front[nf++] = rem; n_front_sms += rem.sm.smCount; }
                PDRV(d.DevResourceGenerateDesc(&dback, sel_back, nb));
                PDRV(d.DevResourceGenerateDesc(&dfront, sel_front, nf));
            }
            CachedPartition c;
            c.device = p->cfg.device;
            c.back_req = back_req;
            PDRV(d.GreenCtxCreate(&c.part.back, dback, dev, CU_GREEN_CTX_DEFAULT_STREAM));
            CUresult rf = d.GreenCtxCreate(&c.part.front, dfront, dev, CU_GREEN_CTX_DEFAULT_STREAM);
            if (rf != CUDA_SUCCESS) {
                d.GreenCtxDestroy(c.part.back);
                return pfail(p, FT8B200_ECUDA, "cuGreenCtxCreate (front): CUresult " + std::to_string((int)rf));
            }
            c.part.front_sms = (int)n_front_sms;
            c.part.back_sms = (int)n_back_sms;
            g_parts.push_back(c);
            hit = &g_parts.back();
        }
        p->part = hit->part;
    }
    for (Lane &l : p->lanes) {
        PDRV(d.GreenCtxStreamCreate(&l.part_front, p->part.front, CU_STREAM_NON_BLOCKING, 0));
        PDRV(d.GreenCtxStreamCreate(&l.part_back, p->part.back, CU_STREAM_NON_BLOCKING, 0));
        int rc = ft8b200_set_partition_streams(l.ctx, l.part_front, l.part_back, p->part.back_sms);
        if (rc) { partition_release(p); return pfail(p, rc, ft8b200_last_error()); }
        l.st = reinterpret_cast<cudaStream_t>(ft8b200_cuda_stream(l.ctx));
        ft8b200_set_side_backend(l.ctx, 1);
    }
#undef PDRV
    p->mode = FT8B200_PIPE_OVERLAP;
    if (front_sms_out) *front_sms_out = p->part.front_sms;
    if (back_sms_out) *back_sms_out = p->part.back_sms;
    return 0;
}

int ft8b200_pipe_set_back_chain(ft8b200_pipe_t *p, int on) {
    if (!p) return FT8B200_BAD_ARG();
    if (p->count) return pfail(p, FT8B200_EBUSY, "ft8b200_pipe_set_back_chain: batches in flight");
    p->chain_back = on != 0;
    p->prev_back = nullptr;
    return 0;
}

int ft8b200_pipe_set_osd(ft8b200_pipe_t *p, int order, int max_hard_errors) {
    if (!p || order < 0 || order > 2) return FT8B200_BAD_ARG();
    return set_lanes(p, __func__, [&](ft8b200_ctx_t *c) { return ft8b200_set_osd(c, order, max_hard_errors); });
}

int ft8b200_pipe_set_ap(ft8b200_pipe_t *p, int on, int max_hard_errors) {
    if (!p || (on != 0 && on != 1)) return FT8B200_BAD_ARG();
    return set_lanes(p, __func__, [&](ft8b200_ctx_t *c) { return ft8b200_set_ap(c, on, max_hard_errors); });
}

int ft8b200_pipe_set_finesync(ft8b200_pipe_t *p, int on, int max_hard_errors) {
    if (!p || (on != 0 && on != 1)) return FT8B200_BAD_ARG();
    return set_lanes(p, __func__, [&](ft8b200_ctx_t *c) { return ft8b200_set_finesync(c, on, max_hard_errors); });
}

int ft8b200_pipe_set_finesync_deep(ft8b200_pipe_t *p, int on, int max_hard_errors) {
    if (!p || (on != 0 && on != 1)) return FT8B200_BAD_ARG();
    return set_lanes(p, __func__, [&](ft8b200_ctx_t *c) { return ft8b200_set_finesync_deep(c, on, max_hard_errors); });
}

int ft8b200_pipe_set_passes(ft8b200_pipe_t *p, int passes) {
    if (!p) return FT8B200_BAD_ARG();
    if (passes < 1 || passes > 3) return pfail(p, FT8B200_EINVAL, "ft8b200_pipe_set_passes: passes must be 1, 2 or 3");
    return set_lanes(p, __func__, [&](ft8b200_ctx_t *c) { return ft8b200_set_passes(c, passes); });
}

int ft8b200_pipe_autotune(ft8b200_pipe_t *p, const uint8_t *d_iq, size_t bytes_per_stream, size_t stream_stride_bytes, int n_slots,
                          const int *candidates, int n_candidates, int batches, int *best_back_sms, int *best_comb_front, float *ms_out) {
    if (!p || !d_iq || !candidates || n_candidates < 1 || n_slots < 1) return FT8B200_BAD_ARG();
    if (p->count) return pfail(p, FT8B200_EBUSY, "ft8b200_pipe_autotune: batches in flight");
    if (batches < (int)p->lanes.size() + 2) batches = (int)p->lanes.size() + 2;
    PCU(cudaSetDevice(p->cfg.device));
    std::vector<struct decoder_results> res((size_t)n_slots * p->cfg.max_messages);
    std::vector<int32_t> cnt((size_t)n_slots);
    float best = -1.0f;
    int best_sms = 0, best_comb = 0, rc = 0;
    std::vector<float> all_ms((size_t)2 * (size_t)n_candidates, -1.0f);
    const bool chain_was = p->chain_back;
    p->chain_back = true;   // one batch's back end at a time while partitions are compared (see submit())
    struct Restore { ft8b200_pipe_t *p; bool v; ~Restore() { p->chain_back = v; p->prev_back = nullptr; } } restore{p, chain_was};
    auto apply = [&](int sms, int comb) -> int {
        int r = ft8b200_pipe_set_partition(p, sms, nullptr, nullptr);
        if (r) return r;
        if (sms == 0 && (r = ft8b200_pipe_set_mode(p, FT8B200_PIPE_SERIAL, -1))) return r;
        for (Lane &l : p->lanes) ft8b200_set_comb_front(l.ctx, comb);
        return 0;
    };
    for (int c = 0; c < n_candidates && !rc; ++c) {
        for (int comb = 0; comb < 2 && !rc; ++comb) {
            float ms = -1.0f;
            if (candidates[c] == 0 && comb == 1) { if (ms_out) ms_out[2 * c + 1] = -1.0f; continue; }  // no partition: the placement means nothing
            if (apply(candidates[c], comb) != 0) { if (ms_out) ms_out[2 * c + comb] = -1.0f; continue; }   // e.g. a split the driver refuses
            for (int pass = 0; pass < 2 && !rc; ++pass) {  // pass 0 warms the lanes' workspaces up
                int submitted = 0, collected = 0;
                // What is timed is the STEADY-STATE interval between completed batches.  The start of a run is not representative either
                // way: its first `depth` batches still find free lanes and an idle back end, which flatters a back partition that is too
                // small (its backlog only shows once the lanes have run out), and the backlog of those first batches then drains in a
                // burst; the end of a run adds the last batch's back end, which a short probe spreads over few batches.  So the clock
                // starts when as many batches as the probe times have been collected before it (a back end that is 10 % too slow needs
                // ~15 batches to use up the lanes' slack) (collect returns on a batch's completion event) and
                // stops at the last completion; nothing after it is waited for.
                const int lead = batches / 2 > (int)p->lanes.size() ? batches / 2 : (int)p->lanes.size();
                const int n = pass == 0 ? (int)p->lanes.size() : batches + lead;
                std::chrono::steady_clock::time_point t0, t1;
                while (collected < n && !rc) {
                    while (submitted < n && p->count < (int)p->lanes.size() && !rc) {
                        rc = submit(p, nullptr, d_iq, bytes_per_stream, stream_stride_bytes, n_slots);
                        ++submitted;
                    }
                    if (rc) break;
                    const int got = ft8b200_pipe_collect(p, res.data(), cnt.data(), n_slots);
                    if (got < 0) rc = got;
                    ++collected;
                    if (collected == lead) t0 = std::chrono::steady_clock::now();
                }
                if (pass == 1 && !rc) {
                    t1 = std::chrono::steady_clock::now();
                    ms = std::chrono::duration<float, std::milli>(t1 - t0).count() / (float)batches;
                }
            }
            if (ms_out) ms_out[2 * c + comb] = ms;
            all_ms[(size_t)(2 * c + comb)] = rc ? -1.0f : ms;
            if (!rc && ms > 0.0f && (best < 0.0f || ms < best)) best = ms;
        }
    }
    if (rc) return rc;
    if (best < 0.0f) return pfail(p, FT8B200_ECUDA, "ft8b200_pipe_autotune: no candidate could be measured");
    // Points within 0.3 % of the fastest are the same within the probe's noise; among them the LARGEST back-end partition is kept (a
    // back end that only just hides under the next batch's block sums is the one a busier slot mix tips over).  The probe itself has
    // to be long: timed over 12 batches from the start of a run, 24 SMs looked 0.1 % faster than 32 and then ran a 20-step bench at
    // 81.1 k slots/s instead of 85.5 k -- the too-small partition's backlog only throttles the front end once the lanes' slack is gone.
    float kept = -1.0f;
    for (int c = 0; c < n_candidates; ++c)
        for (int comb = 0; comb < 2; ++comb) {
            const float ms = all_ms[(size_t)(2 * c + comb)];
            if (ms <= 0.0f || ms > best * 1.003f) continue;
            // (size = candidate % 1000; the thousands carry the SM layout, see ft8b200_pipe_set_partition)
            if (kept < 0.0f || candidates[c] % 1000 > best_sms % 1000 || (candidates[c] % 1000 == best_sms % 1000 && ms < kept)) { kept = ms; best_sms = candidates[c]; best_comb = comb; }
        }
    if ((rc = apply(best_sms, best_comb))) return rc;
    if (best_back_sms) *best_back_sms = best_sms;
    if (best_comb_front) *best_comb_front = best_comb;
    return 0;
}

// Diagnostic: which SMs (hardware %smid) the front (which = 0) or back (which = 1) partition runs on, as a 256-bit mask.
int ft8b200_pipe_partition_smids(ft8b200_pipe_t *p, int which, uint32_t *mask8) {
    if (!p || !mask8 || which < 0 || which > 1) return FT8B200_BAD_ARG();
    if (p->count) return pfail(p, FT8B200_EBUSY, "ft8b200_pipe_partition_smids: batches in flight");
    PCU(cudaSetDevice(p->cfg.device));
    Lane &l = p->lanes[0];
    cudaStream_t st = reinterpret_cast<cudaStream_t>(which ? l.part_back : l.part_front);
    if (!st) st = l.st;  // no partition: the whole GPU
    unsigned int *d_mask = nullptr;
    PCU(cudaMalloc(&d_mask, 8 * sizeof(unsigned int)));
    cudaMemsetAsync(d_mask, 0, 8 * sizeof(unsigned int), st);
    smid_probe_kernel<<<2048, 1024, 0, st>>>(d_mask);
    cudaError_t e = cudaMemcpyAsync(mask8, d_mask, 8 * sizeof(unsigned int), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(d_mask);
    if (e != cudaSuccess) { (void)cudaGetLastError(); return pfail(p, FT8B200_ECUDA, std::string("ft8b200_pipe_partition_smids: ") + cudaGetErrorString(e)); }
    return 0;
}

void ft8b200_pipe_destroy(ft8b200_pipe_t *p) {
    if (!p) return;
    cudaSetDevice(p->cfg.device);
    partition_release(p);
    for (Lane &l : p->lanes) {
        if (l.st) cudaStreamSynchronize(l.st);
        if (l.ctx) ft8b200_destroy(l.ctx);
        if (l.done) cudaEventDestroy(l.done);
        if (l.d_raw) cudaFree(l.d_raw);
        if (l.d_fi) cudaFree(l.d_fi);
        if (l.d_fq) cudaFree(l.d_fq);
        if (l.h_res) cudaFreeHost(l.h_res);
        if (l.h_n) cudaFreeHost(l.h_n);
    }
    if (p->t_ref) cudaEventDestroy(p->t_ref);
    delete p;
}

const char *ft8b200_pipe_error(ft8b200_pipe_t *p) { return p ? p->err.c_str() : "null pipe"; }
int ft8b200_pipe_depth(ft8b200_pipe_t *p) { return p ? (int)p->lanes.size() : 0; }
int ft8b200_pipe_in_flight(ft8b200_pipe_t *p) { return p ? p->count : 0; }

int ft8b200_pipe_submit(ft8b200_pipe_t *p, const uint8_t *d_iq, size_t bytes_per_stream, size_t stream_stride_bytes, int n_slots) {
    return submit(p, nullptr, d_iq, bytes_per_stream, stream_stride_bytes, n_slots);
}

int ft8b200_pipe_submit_host(ft8b200_pipe_t *p, const uint8_t *h_iq, size_t bytes_per_stream, int n_slots) {
    return submit(p, h_iq, nullptr, bytes_per_stream, bytes_per_stream, n_slots);
}

int ft8b200_pipe_submit_streams(ft8b200_pipe_t *p, const uint8_t *d_iq, size_t bytes_per_stream, size_t stream_stride_bytes, int n_streams,
                                int slots_per_stream, size_t bytes_per_slot) {
    return submit(p, nullptr, d_iq, bytes_per_stream, stream_stride_bytes, n_streams, slots_per_stream, bytes_per_slot);
}

int ft8b200_pipe_submit_slots(ft8b200_pipe_t *p, const float *d_i, const float *d_q, const float *d_peak, int n_slots) {
    return submit_slots(p, nullptr, nullptr, d_i, d_q, d_peak, n_slots);
}

int ft8b200_pipe_submit_slots_host(ft8b200_pipe_t *p, const float *h_i, const float *h_q, int n_slots) {
    return submit_slots(p, h_i, h_q, nullptr, nullptr, nullptr, n_slots);
}

static int pop(ft8b200_pipe_t *p, struct decoder_results *h_results, int32_t *h_nresults, int capacity_slots, struct decoder_results **d_results,
               int32_t **d_nresults) {
    if (!p) return FT8B200_BAD_ARG();
    if (p->count == 0) return pfail(p, FT8B200_EINVAL, "ft8b200_pipe_collect: nothing in flight");
    Lane &l = p->lanes[p->head];
    if (h_results && (capacity_slots < l.n_slots || !h_nresults)) return pfail(p, FT8B200_EINVAL, "ft8b200_pipe_collect: result buffers too small");
    PCU(cudaSetDevice(p->cfg.device));
    PCU(cudaEventSynchronize(l.done));
    if (h_results) {
        memcpy(h_results, l.h_res, (size_t)l.n_slots * p->cfg.max_messages * sizeof(struct decoder_results));
        memcpy(h_nresults, l.h_n, (size_t)l.n_slots * sizeof(int32_t));
    }
    if (d_results || d_nresults) {
        int rc = ft8b200_results_device(l.ctx, d_results, d_nresults);
        if (rc) return pfail(p, rc, ft8b200_last_error());
    }
    if (p->profiling) {
        float ms[6];
        if (ft8b200_stage_times(l.ctx, ms, 6) == 0)
            for (int k = 0; k < 6; ++k) if (ms[k] > 0) p->stage_ms[k] += ms[k];
        float tb[6], te[6];
        if (p->t_ref && ft8b200_stage_marks(l.ctx, p->t_ref, tb, te, 6) == 0)
            for (int k = 0; k < 6; ++k) { p->timeline.push_back(tb[k]); p->timeline.push_back(te[k]); }
    }
    ++p->batches;
    p->slots += (uint64_t)l.n_slots;
    p->head = (p->head + 1) % (int)p->lanes.size();
    --p->count;
    return l.n_slots;
}

int ft8b200_pipe_collect(ft8b200_pipe_t *p, struct decoder_results *h_results, int32_t *h_nresults, int capacity_slots) {
    if (!h_results || !h_nresults) return p ? pfail(p, FT8B200_EINVAL, "ft8b200_pipe_collect: null result buffer") : FT8B200_EINVAL;
    return pop(p, h_results, h_nresults, capacity_slots, nullptr, nullptr);
}

int ft8b200_pipe_collect_device(ft8b200_pipe_t *p, struct decoder_results **d_results, int32_t **d_nresults) {
    return pop(p, nullptr, nullptr, 0, d_results, d_nresults);
}

int ft8b200_pipe_depend_on(ft8b200_pipe_t *p, void *cuda_event) {
    if (!p) return FT8B200_BAD_ARG();
    p->dependency = reinterpret_cast<cudaEvent_t>(cuda_event);
    return 0;
}

int ft8b200_pipe_set_profiling(ft8b200_pipe_t *p, int on) {
    if (!p) return FT8B200_BAD_ARG();
    p->profiling = on != 0;
    for (Lane &l : p->lanes) ft8b200_set_profiling(l.ctx, on);
    for (double &v : p->stage_ms) v = 0.0;
    p->batches = 0;
    p->slots = 0;
    p->timeline.clear();
    if (on) {
        PCU(cudaSetDevice(p->cfg.device));
        if (!p->t_ref) PCU(cudaEventCreate(&p->t_ref));
        PCU(cudaEventRecord(p->t_ref, p->lanes[0].st));
    }
    return 0;
}

// Device timeline of the batches collected since profiling was switched on: 12 floats per batch (begin, end of block sums,
// comb+FIR, waterfall, sync, decode, spots in ms since that moment).  Returns the number of batches written (<= max_batches).
int ft8b200_pipe_timeline(ft8b200_pipe_t *p, float *out, int max_batches) {
    if (!p || !out || max_batches < 0) return FT8B200_BAD_ARG();
    int n = (int)(p->timeline.size() / 12);
    if (n > max_batches) n = max_batches;
    memcpy(out, p->timeline.data(), (size_t)n * 12 * sizeof(float));
    return n;
}

// sums over the batches collected since profiling was switched on: ms[0..5] as ft8b200_stage_times, *batches = how many
int ft8b200_pipe_stage_times(ft8b200_pipe_t *p, double *ms, int n, uint64_t *batches) {
    if (!p || !ms || n < 6) return FT8B200_BAD_ARG();
    for (int k = 0; k < 6; ++k) ms[k] = p->stage_ms[k];
    if (batches) *batches = p->batches;
    return 0;
}

uint64_t ft8b200_pipe_kernel_launches(ft8b200_pipe_t *p) {
    uint64_t n = 0;
    if (p) for (Lane &l : p->lanes) n += ft8b200_kernel_launches(l.ctx);
    return n;
}

}  // extern "C"
