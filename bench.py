#!/usr/bin/env python3
"""bench.py -- FT8 15 s-slots decoded per second, from raw 2.4 Msps uint8 RTL IQ (BASELINE.json config #2:
one 15 s slot = 36 M complex samples through the full CIC+FIR decimation and FT8 decode), batched.

  python bench.py --gpus N --steps K --warmup W                     this repository's CUDA path (one process per GPU)
  python bench.py --impl reference --gpus N --steps K --warmup W    the reference's own CPU implementation, all host cores
  python bench.py ... --dump-outputs DIR                            + the spot records of the last timed step as DIR/*.npy

A "step" is one pass of the whole hot path (decimate -> condition -> waterfall -> Costas sync/top-K ->
LLR/LDPC/CRC/unpack -> spot table) over one batch of synthetic slots.  `value` times it with the batch already
resident in HBM (the batch is larger than L2); `e2e` times the same path through the C-ABI call that takes HOST
buffers (pinned), host->device copies, the device->host read of the spot records and -- on several GPUs -- the NCCL
gather of the records inside the timed region.  `e2e_slots` is the same at the path's other boundary (the input of
ft8_subsystem(): 3200 sps float slots from host memory).  `roofline` is for the dominant kernel (cic_block_sums,
HBM-bound), timed live with CUDA events on the launching stream; `roofline_extra` times every kernel of the path in one
serial, un-partitioned pass; `configs` carries the other BASELINE configurations (#1 as single-slot latency through the
literal drop-in calls, #3 on both waterfall paths, #4 strong-scaled over the GPUs with the gather, #5 sharded by receiver
stream), each with the CPU reference on a sample beside it and a parity flag; `cpu_baseline` is the CPU checker
(oracle/_ref = the unmodified reference when it was built, else the restatement) timed on this box's host cores on a
bounded sample of the headline batch.  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

RAW_SLOT_BYTES = 72_000_000
ALGO_BYTES_PER_SLOT = 72_000_000 + 47_936 * 8  # SURVEY.md section 8d: 2 B/sample in + 8 B per output
WF_BYTES_PER_SLOT = 384_000 + 94_208           # SURVEY 8d: waterfall A reads the slot, writes the uint8 waterfall
MON_BYTES_PER_SLOT = 720_000 + 357_120         # SURVEY 8d: waterfall B (12 kHz monitor)
COMB_BYTES_PER_SLOT = 47_936 * 16 + 384_000    # comb+FIR: block sums (int32x4 per block) in, two float rails out
WF_FP32_PER_SLOT = 8.9e6                       # DESIGN.md 2.2: FP32 instructions (thread level) bit-exact kiss_fft arithmetic needs per slot
METRIC = "FT8 15s-slots decoded/sec from raw 2.4 Msps uint8 IQ"


# --------------------------------------------------------------------------------------------- inputs
def slot_params(seed: int):
    """Deterministic message / frequency / time offset of synthetic slot `seed`."""
    from tools import synth
    rng = np.random.Generator(np.random.PCG64(0xF78 + seed))
    to, de, ex = synth.random_message(rng)
    if seed % 2 == 0:
        to = "CQ"
        ex = synth.random_grid(rng)
    return dict(text=f"{to} {de} {ex}", f_hz=float(rng.uniform(200.0, 1400.0)), t0=float(0.5 + rng.uniform(-0.3, 0.3)),
                amp=20.0, noise=30.0)


def gen_batch(n_slots: int, first_seed: int, device, ctx=None):
    """n_slots x 72 MB of uint8 IQ made ON THE DEVICE by the library's synthesiser (csrc/synth.cu): one FT8 message per
    slot as phase-continuous 8-FSK at (f - 600 kHz), 20 LSB over 30 LSB of noise, offset 128, saturating."""
    from ft8b200_loader import load
    pkg = load()
    own = ctx is None
    if own:
        ctx = pkg.Context(device.index or 0)
    params = [slot_params(first_seed + s) for s in range(n_slots)]
    sig = pkg.make_signals((pkg.pack77_std(*p["text"].split()), p["f_hz"], p["t0"], p["amp"]) for p in params)
    buf = ctx.synth_raw(sig, np.arange(n_slots + 1, dtype=np.int32), params[0]["noise"], 0xF78, first_slot_index=first_seed)
    if own:
        ctx.close()
    return buf, [p["text"] for p in params]


def slot_ok(text: str, res_row, n: int) -> bool:
    """The slot's own message came back: CQ messages with their call sign in decoder_results; other messages only count
    as a decode (rtlsdr_ft8d.c:1509-1520 writes records for CQ messages only)."""
    if n < 1:
        return False
    to, de = text.split()[:2]
    return to != "CQ" or any(r["call"] == de.encode() for r in res_row[:n])


def count_ok(texts, res, nres) -> int:
    return sum(1 for s in range(len(texts)) if slot_ok(texts[s], res[s], int(nres[s])))


# --------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock / throttle-reason sampling DURING the timed region: NVML polled every 2 ms from a thread
    (nvidia-smi -lms cannot resolve a region that lasts milliseconds)."""
    REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.stop_flag = False
        self.thread = None
        self.max_mhz = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(visible.split(",")[self.gpu]) if visible and visible.split(",")[self.gpu].isdigit() else self.gpu
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception:
            return

        def loop():
            while not self.stop_flag:
                try:
                    mhz = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                    try:
                        why = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                    except Exception:
                        why = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    self.rows.append((time.time(), float(mhz), int(why)))
                except Exception:
                    pass
                time.sleep(0.002)

        self.thread = threading.Thread(target=loop, daemon=True)
        self.thread.start()

    def stop(self):
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=1)

    def summary(self, t0: float, t1: float):
        rows = [r for r in self.rows if t0 <= r[0] <= t1]
        if not rows:  # region shorter than one poll: take the nearest samples
            rows = sorted(self.rows, key=lambda r: abs(r[0] - 0.5 * (t0 + t1)))[:3]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        why = 0
        for r in rows:
            why |= r[2]
        return {"sm_mhz": float(np.median([r[1] for r in rows])), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(k for k, bit in self.REASONS.items() if why & bit), "samples": len(rows)}


# --------------------------------------------------------------------------------------------- CPU arms
_CPU_SLOTS = None  # numpy uint8 [n, 72e6], shared with forked workers


def cpu_kind():
    from oracle.pyoracle import Reference
    return "reference" if Reference.available("k120") else "port"


_CPU_PHASE_S = {"decimator": 0.0, "decode": 0.0}   # seconds spent per phase by _cpu_one_slot in THIS process (single-thread baseline)


def _cpu_one_slot(idx: int):
    """Raw slot -> spots on the CPU: rtlsdr_callback() in 65536-byte calls, decoder() conditioning, ft8_subsystem()."""
    from oracle.pyoracle import Oracle, Reference
    raw = _CPU_SLOTS[idx]
    orc = Oracle()
    t0 = time.perf_counter()
    if cpu_kind() == "reference":
        ref = Reference("k120", fresh=True)  # private copy: the daemon's decimator state is function-static
        for o in range(0, raw.size, 65536):
            ref.callback(raw[o:o + 65536])
        i_s, q_s, n = ref.rx()
        t1 = time.perf_counter()
        i_s, q_s, _ = orc.condition(i_s, q_s, n)  # decoder() itself is thread-bound in the daemon (rtlsdr_ft8d.c:221-285)
        count = int(ref.subsystem(i_s, q_s)["n"])
    else:
        oi, oq = orc.decimate_slot(raw)
        t1 = time.perf_counter()
        i_s = np.zeros(48000, np.float32); q_s = np.zeros(48000, np.float32)
        i_s[:oi.size] = oi; q_s[:oq.size] = oq
        i_s, q_s, _ = orc.condition(i_s, q_s, oi.size)
        count = int(orc.subsystem(i_s, q_s)["n"])
    _CPU_PHASE_S["decimator"] += t1 - t0
    _CPU_PHASE_S["decode"] += time.perf_counter() - t1
    return count


def _cpu_synth_slot(idx: int):
    """Slot `idx` of the bench batch into _CPU_SLOTS (shared memory), by the CPU twin of ft8b200_synth_raw."""
    from oracle.pyoracle import Oracle, signal_dtype
    orc = Oracle()
    p = slot_params(idx)
    sig = np.zeros(1, signal_dtype)
    sig[0]["payload"] = np.frombuffer(orc.pack_std(*p["text"].split()), np.uint8)
    sig[0]["f0_hz"], sig[0]["t0_sec"], sig[0]["amp"] = p["f_hz"], p["t0"], p["amp"]
    _CPU_SLOTS[idx] = orc.synth_raw(sig, p["noise"], 0xF78, idx, RAW_SLOT_BYTES // 2)
    return 0


def cpu_run(n_slots: int, workers: int):
    """Seconds to push slots 0..n_slots-1 of _CPU_SLOTS through the CPU path with `workers` processes."""
    t0 = time.perf_counter()
    if workers <= 1:
        out = [_cpu_one_slot(k) for k in range(n_slots)]
    else:
        import multiprocessing as mp
        with mp.get_context("fork").Pool(workers) as pool:
            out = pool.map(_cpu_one_slot, range(n_slots), chunksize=1)
    return time.perf_counter() - t0, out


# --------------------------------------------------------------------------------------------- helpers
_JSON_FD = None


def bind_to_gpu_numa(local: int):
    """Run this rank on the CPUs of the NUMA node its GPU hangs off, so that the pinned host buffers of the e2e measurement
    (first touch) are local to the PCIe root the copies go through.  Returns a note for `config`, or None when it does not apply."""
    if os.environ.get("BENCH_NUMA", "1") == "0":
        return "off"
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bus = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return "GPU %s on NUMA node %d: rank bound to its %d CPUs" % (bus, node, len(cpus))
    except Exception as exc:
        return "not bound (%s)" % type(exc).__name__


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(line.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, line)


class Env:
    """What every part of the CUDA arm needs: torch, the harness package, rank/world, device, timing helpers."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        from ft8b200_loader import load
        self.torch, self.dist, self.pkg, self.args = torch, dist, load(), args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.device = torch.device("cuda", self.local)
        self.numa = bind_to_gpu_numa(self.local)
        if self.world > 1:
            # the all_gather of the spot records must not queue behind the decimator's 190k-CTA grid: high-priority NCCL stream
            opts = dist.ProcessGroupNCCL.Options()
            opts.is_high_priority_stream = True
            dist.init_process_group("nccl", device_id=self.device, pg_options=opts)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, ms: float) -> float:
        if self.world == 1:
            return float(ms)
        t = self.torch.tensor([ms], dtype=self.torch.float64, device=self.device)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, v: int) -> int:
        if self.world == 1:
            return int(v)
        t = self.torch.tensor([v], dtype=self.torch.int64, device=self.device)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return int(t.item())

    def timed(self, fn, steps: int):
        """barrier + sync | CUDA events around fn(steps) | barrier + sync -> ms, max over ranks."""
        e0 = self.torch.cuda.Event(enable_timing=True); e1 = self.torch.cuda.Event(enable_timing=True)
        self.barrier()
        t0 = time.time()
        e0.record()
        out = fn(steps)
        e1.record()
        self.barrier()
        t1 = time.time()
        return self.max_over_ranks(e0.elapsed_time(e1)), out, (t0, t1)

    def gather_records(self, res_dev, nres_dev):
        """ONE NCCL all_gather each for a batch's decoder_results (uint8[n, M, 28] device tensor) and counts (int32[n]);
        -> (uint8[world*n, M, 28], int32[world*n]) device tensors (the local ones when there is one rank)."""
        if self.world == 1:
            return res_dev, nres_dev
        g_res = self.torch.empty((self.world * res_dev.shape[0],) + tuple(res_dev.shape[1:]), dtype=res_dev.dtype, device=self.device)
        g_n = self.torch.empty(self.world * nres_dev.shape[0], dtype=nres_dev.dtype, device=self.device)
        self.dist.all_gather_into_tensor(g_res, res_dev.contiguous())
        self.dist.all_gather_into_tensor(g_n, nres_dev.contiguous())
        return g_res, g_n


class StepGather:
    """Multi-GPU: the spot records of a step's executor batches are staged on the device (a local copy, so a lane is free again
    as soon as its records are copied) and gathered to every rank with ONE NCCL all_gather per step; rank 0 reads them on the
    host through pinned double buffers without blocking its submit loop."""

    def __init__(self, env: Env, pipe, chunks: int, bc: int):
        from tools.shard import stage_row_bytes
        torch = env.torch
        self.env, self.pipe, self.chunks, self.bc, self.M = env, pipe, chunks, bc, pipe.M
        row = stage_row_bytes(bc, pipe.M)
        self.stage = torch.empty((chunks, row), dtype=torch.uint8, device=env.device)  # per batch: records, then counts
        self.gathered = torch.empty((env.world, chunks, row), dtype=torch.uint8, device=env.device)
        self.copied = torch.cuda.Event()
        self.host_rec = [torch.empty(self.gathered.shape, dtype=torch.uint8).pin_memory() for _ in range(2)] if env.rank == 0 else None
        self.host_ev = [torch.cuda.Event(), torch.cuda.Event()]
        self.n_staged = 0

    def collect(self):
        """Oldest batch in flight -> staged; after the step's last batch: all_gather + async read on rank 0."""
        from tools.shard import stage_batch
        res_dev, nres_dev = self.pipe.collect_device()
        stage_batch(self.stage, self.n_staged % self.chunks, res_dev, nres_dev, self.bc, self.M)
        self.copied.record()
        self.pipe.depend_on(self.copied)   # the lane's buffers are rewritten only after they have been copied out (ordered on the device)
        self.n_staged += 1
        if self.n_staged % self.chunks == 0:
            self.env.dist.all_gather_into_tensor(self.gathered.view(-1), self.stage.view(-1))   # spot records over NVLink, once per step
            if self.env.rank == 0:
                i = (self.n_staged // self.chunks - 1) % 2
                self.host_ev[i].synchronize()   # the copy issued two steps ago (long finished) owns this buffer
                self.host_rec[i].copy_(self.gathered, non_blocking=True)
                self.host_ev[i].record()

    def last(self):
        """rank 0: records of the last gathered step, all ranks, in (rank, slot) order; None elsewhere."""
        from tools.shard import unpack_gathered
        if self.env.rank != 0 or self.n_staged < self.chunks:
            return None
        i = (self.n_staged // self.chunks - 1) % 2
        self.host_ev[i].synchronize()
        res, nres = unpack_gathered(self.host_rec[i].numpy(), self.env.world, self.chunks, self.bc, self.M)
        from ft8b200_loader import load
        return res.view(load().result_dtype).reshape(res.shape[0], self.M), nres


def run_steps(env: Env, pipe, submit, steps: int, chunks: int, bc: int, gather: StepGather | None):
    """`steps` passes, each `chunks` executor batches (submit(c) queues batch c); every batch's spot records are read back
    (one rank) or staged + gathered (several).  Returns the last pass's records in slot order (gathered: rank 0 only)."""
    outs = []

    def collect():
        if gather is not None:
            gather.collect()
        else:
            outs.append(pipe.collect(bc))

    for _ in range(steps):
        for c in range(chunks):
            if pipe.in_flight() == pipe.depth:
                collect()
            submit(c)
    while pipe.in_flight():
        collect()
    if gather is not None:
        return gather.last()
    last = outs[-chunks:]
    return np.concatenate([np.asarray(o[0]) for o in last]), np.concatenate([np.asarray(o[1]) for o in last])


def records_equal(a, b) -> bool:
    return bool(np.array_equal(np.asarray(a[1]), np.asarray(b[1])) and np.asarray(a[0]).tobytes() == np.asarray(b[0]).tobytes())


DUMP_MAX_BYTES = 64_000_000   # all files together, .npy headers included
DUMP_HEADER_BYTES = 256       # allowance per .npy header (numpy writes 128 bytes for these arrays)


def dump_outputs(path: str, res, nres, result_dtype):
    """Write what the caller of the timed path received in its last step -- per slot, the spot count and the decoder_results
    records -- as float arrays under `path`, so two builds can be compared output for output on the same inputs.  Records past
    a slot's count carry no result and are written as zeros.  Text fields are written one float32 per byte.  Where all slots
    would not fit in DUMP_MAX_BYTES a fixed, seeded sample of slots is written; slot_index.npy names the slots either way."""
    res = np.asarray(res).view(result_dtype)
    nres = np.asarray(nres, np.int64)
    n_slots, m = res.shape
    slot_bytes = m * (8 + 8 + 4 * (result_dtype["call"].itemsize + result_dtype["loc"].itemsize)) + 16
    budget = DUMP_MAX_BYTES - 6 * DUMP_HEADER_BYTES   # six files
    idx = np.arange(n_slots)
    if n_slots * slot_bytes > budget:
        idx = np.sort(np.random.default_rng(0).choice(n_slots, budget // slot_bytes, replace=False))
    res, nres = res[idx].copy(), nres[idx]
    res[np.arange(m)[None, :] >= nres[:, None]] = np.zeros((), result_dtype)
    os.makedirs(path, exist_ok=True)
    arrays = {"slot_index": idx.astype(np.float64), "n_results": nres.astype(np.float64),
              "freq": res["freq"].astype(np.float64), "snr": res["snr"].astype(np.float64)}
    for name in ("call", "loc"):
        arrays[name] = np.ascontiguousarray(res[name]).view(np.uint8).reshape(res.shape + (-1,)).astype(np.float32)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


# --------------------------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--slots", type=int, default=512, help="15 s slots per GPU per step (36.9 GB of raw IQ per GPU at 512)")
    ap.add_argument("--e2e-slots", type=int, default=8, help="raw slots per step of the host-buffer (e2e) measurement")
    ap.add_argument("--chunks", type=int, default=4, help="executor batches per step: a step's slots are submitted to ft8b200_pipe_t in this many batches")
    ap.add_argument("--depth", type=int, default=3, help="batches in flight in the pipelined executor")
    ap.add_argument("--back-sms", type=int, default=-1, help="SMs of the back-end partition (waterfall/sync/LDPC of batch n next to the decimator of batch n+1 on the "
                                                             "other SMs); -1 = measure 24/32/40 and both comb+FIR placements at start-up and keep the fastest "
                                                             "(ft8b200_pipe_autotune); 0 = no partition, kernels of consecutive batches run serially")
    ap.add_argument("--overlap", action="store_true", help="(without a partition) let the back end of batch n time-share the GPU with the decimator of batch n+1")
    ap.add_argument("--k1-variant", type=int, default=0, help="0 = streaming cic_block_sums kernel, 1..6 = bulk-copy (TMA) variants")
    ap.add_argument("--cpu-slots", type=int, default=96, help="bounded CPU-baseline sample (slots)")
    ap.add_argument("--cluster", action="store_true", help="single-process arm: all --gpus devices driven from THIS process through ft8b200_cluster_t "
                                                          "(records gathered by the library's own NCCL all-gather); not launched under torchrun")
    ap.add_argument("--chain-back", action="store_true", help="A/B: with an SM partition, back ends of consecutive batches run one at a time (ft8b200_pipe_set_back_chain)")
    ap.add_argument("--no-configs", action="store_true", help="skip the other BASELINE configurations (configs, e2e_slots, roofline_extra)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the spot records of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.cluster):
        ap.error("--dump-outputs applies to the CUDA arm without --cluster")
    args.warmup = max(args.warmup, 3)
    # stdout carries exactly ONE line, the JSON: anything a library prints to fd 1 on the way (NCCL's version banner at
    # communicator creation, for one) is sent to stderr, and the JSON line is written to the original stdout at the end
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    config = {"workload": "BASELINE config #2 batched: %d x (one 15 s slot of raw 2.4 Msps uint8 RTL IQ, 36 M complex samples, one FT8 message "
                          "at 20 LSB over 30 LSB noise) per GPU per step -> CIC+FIR decimation -> decoder() conditioning -> waterfall -> "
                          "sync (K=120) -> LDPC/CRC/unpack -> spot table" % args.slots,
              "slots_per_gpu_per_step": args.slots, "input_bytes_per_step_per_gpu": args.slots * RAW_SLOT_BYTES,
              "l2": "inputs larger than L2 (%.1f GB per step per GPU vs 126 MB)" % (args.slots * RAW_SLOT_BYTES / 1e9),
              "max_candidates": 120, "max_messages": 50, "ldpc_iterations": 20,
              "parallelism": "slots sharded across GPUs, no data-path collective; "
              "spot records gathered with one NCCL all_gather per step" if world > 1 else "single GPU"}

    if args.impl == "reference":
        return reference_arm(args, rank, world, config)
    if args.cluster:
        return cluster_arm(args, config)

    env = Env(args)
    run_info = {}   # how THIS arm ran the workload (executor, SM split, CPU binding): `config` itself only names the workload and is the same in every arm
    torch, dist, pkg = env.torch, env.dist, env.pkg
    device, local = env.device, env.local
    if env.numa:
        run_info["numa"] = env.numa

    B = args.slots
    if args.chunks < 1 or B % args.chunks:
        raise SystemExit("--slots must be a multiple of --chunks")
    Bc = B // args.chunks   # slots per executor batch
    batch, texts = gen_batch(B, 100_000 * rank, device)
    torch.cuda.synchronize()
    # The product's batch executor (ft8b200_pipe_t): `depth` batches in flight; in SERIAL mode the kernels of consecutive
    # batches never share the GPU (each kernel is timed alone), only D2H of the records and host work overlap them.
    pipe = pkg.Pipe(local, args.depth)
    pipe.set_mode(serial=not args.overlap, decimator_variant=args.k1_variant)
    mode_txt = "overlap (time-shared)" if args.overlap else "serial (kernels of consecutive batches do not share the GPU)"
    if args.back_sms != 0:
        # green contexts: disjoint SM sets for the HBM-bound decimator and the issue-bound back end (ft8b200_pipe_set_partition)
        try:
            if args.back_sms < 0:
                pipe.set_profiling(True)   # the timed region records stage events: the probe must carry the same (small) per-stage cost
                tuned = pipe.autotune(batch[:Bc], Bc, candidates=(24, 32, 40), batches=48)
                run_info["sm_partition"] = {"chosen_by": "ft8b200_pipe_autotune (ms per %d-slot batch at each point)" % Bc, **tuned}
                mode_txt = "SM partition: back end of batch n on %d SMs (comb+FIR on the %s set), decimator of batch n+1 on the others" % (
                    tuned["back_sms"], "front" if tuned["comb_front"] else "back")
            else:
                run_info["sm_partition"] = dict(zip(("front_sms", "back_sms"), pipe.set_partition(args.back_sms)))
                mode_txt = "SM partition: back end of batch n on >= %d SMs, decimator of batch n+1 on the others" % args.back_sms
        except Exception as exc:  # a driver without green contexts: same kernels, consecutive batches back to back on the whole GPU
            run_info["sm_partition"] = "unavailable (%s): running serial" % exc
            pipe.set_mode(serial=True, decimator_variant=args.k1_variant)
            args.back_sms = 0
    if args.chain_back and args.back_sms != 0:
        pipe.set_back_chain(True)
        mode_txt += ", back ends chained"
    run_info["executor"] = "ft8b200_pipe_t depth %d, %d batches of %d slots per step, %s" % (args.depth, args.chunks, Bc, mode_txt)
    M = pipe.M

    gather = StepGather(env, pipe, args.chunks, Bc) if world > 1 and not os.environ.get("BENCH_NOGATHER") else None
    submit_dev = lambda c: pipe.submit(batch[c * Bc:(c + 1) * Bc], Bc)
    out = run_steps(env, pipe, submit_dev, args.warmup, args.chunks, Bc, gather)

    # ---- correctness guard: every synthetic slot must decode to its own message -- on every rank, through both result paths
    local_res, local_nres = run_steps(env, pipe, submit_dev, 1, args.chunks, Bc, None)   # this rank's records through the host-collect path
    n_good_local = count_ok(texts, local_res, local_nres)
    n_good = env.sum_over_ranks(n_good_local)
    verify = {"slots_decoded_to_their_own_message": n_good, "of": world * B}
    if world > 1:
        # rank 0 holds the gathered records of every rank (staged on the device, one all_gather per step): they must equal what each
        # rank collects locally through ft8b200_pipe_collect, and every rank's slot must carry that rank's own message
        t_res = torch.from_numpy(np.ascontiguousarray(local_res).view(np.uint8).reshape(B, M * 28)).to(device)
        t_n = torch.from_numpy(np.ascontiguousarray(local_nres, np.int32)).to(device)
        all_res, all_n = env.gather_records(t_res, t_n)
        if rank == 0 and out is not None:
            g_res, g_n = out
            ref_res = all_res.cpu().numpy().view(pkg.result_dtype).reshape(world * B, M)
            ref_n = all_n.cpu().numpy()
            verify["gathered_records_equal_each_ranks_local_records"] = records_equal((g_res, g_n), (ref_res, ref_n))
            all_texts = [slot_params(100_000 * r + s)["text"] for r in range(world) for s in range(B)]
            verify["gathered_slots_decoded_to_their_own_message"] = count_ok(all_texts, g_res, g_n)
    res, nres = local_res, local_nres

    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    pipe.set_profiling(True)
    launches0 = pipe.launches()
    ms, last_step, (t_wall0, t_wall1) = env.timed(lambda k: run_steps(env, pipe, submit_dev, k, args.chunks, Bc, gather), args.steps)
    launches = pipe.launches() - launches0
    stage_acc, n_prof = pipe.stage_times()
    pipe.set_profiling(False)
    if args.dump_outputs and rank == 0 and last_step is not None:
        dump_outputs(args.dump_outputs, *last_step, pkg.result_dtype)
    value = world * B * args.steps / (ms * 1e-3)
    clocks = sampler.summary(t_wall0, t_wall1)

    # ---- e2e: host buffers in, host results out, through the C-ABI calls that take HOST memory; several GPUs: + the gather
    Be = min(args.e2e_slots, B)
    host = torch.empty((Be, RAW_SLOT_BYTES), dtype=torch.uint8, pin_memory=True)
    host.copy_(batch[:Be])
    host_np = host.numpy()
    gather_e = StepGather(env, pipe, 1, Be) if gather is not None else None
    submit_host = lambda c: pipe.submit_host(host_np, Be)
    run_steps(env, pipe, submit_host, args.warmup, 1, Be, gather_e)
    ms_e2e, out_e2e, _ = env.timed(lambda k: run_steps(env, pipe, submit_host, k, 1, Be, gather_e), args.steps)
    sampler.stop()
    if world == 1:
        same_e2e = records_equal(out_e2e, (res[:Be], nres[:Be]))
    else:
        flag = 1
        if rank == 0:
            g_res, g_n = out_e2e
            ref_res = all_res.cpu().numpy().view(pkg.result_dtype).reshape(world, B, M)[:, :Be].reshape(world * Be, M)
            ref_n = all_n.cpu().numpy().reshape(world, B)[:, :Be].reshape(-1)
            flag = int(records_equal((g_res, g_n), (ref_res, ref_n)))
        same_e2e = bool(env.sum_over_ranks(flag) == world)
    e2e = {"value": world * Be * args.steps / (ms_e2e * 1e-3), "unit": "slots/s", "h2d_bytes_per_step": Be * RAW_SLOT_BYTES,
           "d2h_bytes_per_step": Be * (M * 28 + 4) * (world if rank == 0 and world > 1 else 1), "slots_per_step": Be,
           "same_results_as_device_path": same_e2e,
           "h2d_gbs": world * Be * RAW_SLOT_BYTES * args.steps / (ms_e2e * 1e-3) / 1e9,
           "api": "ft8b200_pipe_submit_host / ft8b200_pipe_collect%s (pinned host IQ in, decoder_results out, %d batches in flight)" % (
               "_device + one NCCL all_gather of the records per step, read on rank 0" if world > 1 else "", pipe.depth)}
    try:
        hc = json.load(open(os.path.join(ROOT, "profiles", "h2d_ceiling_r2.json")))
        e2e["host_ceiling_gbs"] = hc.get("by_gpus", {}).get(str(world))
        e2e["host_ceiling_source"] = "profiles/h2d_ceiling_r2.json (tools/h2d_probe.py: %s)" % hc.get("what", "")
    except Exception:
        pass

    # ---- roofline of the dominant kernel (cic_block_sums): algorithmic bytes / CUDA-event time
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_source = "MEASURED_PEAKS.json hbm_gbs (measured, burst copy)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    n_prof = max(n_prof, 1)
    k1_ms = stage_acc.get("block_sums", 0.0) / n_prof
    k2_ms = stage_acc.get("comb_fir", 0.0) / n_prof
    achieved = Bc * ALGO_BYTES_PER_SLOT / (k1_ms * 1e-3) / 1e9 if k1_ms > 0 else None
    roofline = {"kernel": "cic_block_sums_kernel", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": (achieved / peak) if achieved else None, "traffic": None, "peak_source": peak_source,
                "algorithmic_bytes_per_launch": Bc * ALGO_BYTES_PER_SLOT, "slots_per_launch": Bc, "launch_ms": k1_ms,
                "decimator_ms_incl_comb_fir": k1_ms + k2_ms,
                "decimator_msps": Bc * 36.0 / ((k1_ms + k2_ms) * 1e-3) if k1_ms > 0 else None,
                "timed": "CUDA events around every launch of the kernel inside the timed region (%d launches)" % n_prof,
                "stage_ms_per_launch": {k: v / n_prof for k, v in stage_acc.items()},
                "stage_note": "with an SM partition the back-end stages (comb_fir ... spots) run on the back-end SMs concurrently with the "
                              "next batch's block sums: their times overlap it and do not add to the step" if args.back_sms != 0 else "stages run back to back"}
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic_r2.json")))  # one `ncu --set full` capture, per slot
        roofline["traffic"] = tr.get("dram_bytes_per_slot", 0) * Bc or None
        roofline["traffic_source"] = tr.get("source")
    except Exception:
        pass

    out = {"metric": METRIC, "value": value, "unit": "slots/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32+f32",
           "data": "synthetic (generated on the device by ft8b200_synth_raw)", "config": config, "run": run_info, "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
           "decoded_ok_slots_in_first_batch": n_good_local, "verify": verify}

    pipe.close()
    if not args.no_configs:
        from tools import bench_configs as bc
        sm_mhz = clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965.0
        if rank == 0:
            out["roofline_extra"] = bc.roofline_extra(env, batch, min(Bc, 128), peak, peak_source, sm_mhz)
        env.barrier()
        configs = {}
        configs["c5_streams"] = bc.config5(env, batch, texts)
        del batch, host
        torch.cuda.empty_cache()
        configs["c4_slots_sharded"], slots_host = bc.config4(env, args.steps)
        out["e2e_slots"] = bc.e2e_slots(env, slots_host, args.steps, args.depth)
        if world == 1:
            configs["c3_daemon_k500"] = bc.config3_daemon(env)
            configs["c3_monitor_12k"] = bc.config3_monitor(env)
            configs["c1_single_slot_latency"] = bc.config1_latency(env)
        out["configs"] = configs
        # re-created for the CPU baseline sample below
        batch = None

    if rank == 0 and world == 1:
        global _CPU_SLOTS
        n_cpu = min(args.cpu_slots, B)
        if batch is None:
            batch, _ = gen_batch(n_cpu, 0, device)
        _CPU_SLOTS = batch[:n_cpu].cpu().numpy()
        _CPU_PHASE_S["decimator"] = _CPU_PHASE_S["decode"] = 0.0
        secs, n_dec = cpu_run(n_cpu, 1)
        gpu_n = [int(x) for x in nres[:n_cpu]]
        out["cpu_baseline"] = {"value": n_cpu / secs, "unit": "slots/s", "cores": 1, "kind": cpu_kind(),
                               "sample": "%d of the step's %d slots, single thread: rtlsdr_callback in 65536-byte calls + decoder() "
                                         "conditioning + ft8_subsystem (%.2f s)" % (n_cpu, B, secs),
                               "same_spot_counts_as_gpu": n_dec == gpu_n,
                               # SURVEY 8d (i), (ii): the two halves of the path on one host thread
                               "decimator_msps": n_cpu * (RAW_SLOT_BYTES // 2) / max(_CPU_PHASE_S["decimator"], 1e-9) / 1e6,
                               "decode_slots_per_s": n_cpu / max(_CPU_PHASE_S["decode"], 1e-9)}
    if rank == 0:
        emit(out)
    if world > 1:
        dist.destroy_process_group()
    return 0


def cluster_arm(args, config):
    """The library's own multi-GPU plane: ONE process, ft8b200_cluster_t over args.gpus devices (one executor per device, spot records
    of every step gathered with the library's grouped ncclAllGather and read on the host).  Same workload and step as the headline;
    torch only allocates nothing here -- the inputs are made by each device's context.  Timed on the host clock between
    synchronisations of every device (one process drives all of them, so there is no per-rank clock to take the maximum of)."""
    import torch
    from ft8b200_loader import load
    pkg = load()
    B, Bc = args.slots, args.slots // args.chunks
    cl = pkg.Cluster(args.gpus, args.depth)
    n = cl.n
    bufs, texts = [], []
    for d in range(n):
        b, t = gen_batch(B, 100_000 * d, torch.device("cuda", d), cl.ctx(d))
        bufs.append(b); texts += t
    part = []
    for d in range(n):
        p = cl.pipe(d)
        p.set_mode(serial=True)
        try:
            part.append(p.autotune(bufs[d][:Bc], Bc, candidates=(24, 32, 40), batches=48) if args.back_sms < 0 else
                        (dict(zip(("front_sms", "back_sms"), p.set_partition(args.back_sms))) if args.back_sms > 0 else "serial"))
        except Exception as exc:
            part.append("unavailable (%s)" % exc)

    def sync_all():
        for d in range(n):
            torch.cuda.synchronize(d)

    def run(steps):
        outs = []
        for _ in range(steps):
            for c in range(args.chunks):
                if cl.in_flight() == cl.depth:
                    outs.append(cl.collect(n * Bc))
                cl.submit([bufs[d][c * Bc:(c + 1) * Bc] for d in range(n)], [Bc] * n)
        while cl.in_flight():
            outs.append(cl.collect(n * Bc))
        return outs[-args.chunks:]

    last = run(args.warmup)
    # records of a step come back chunk by chunk, each in (device, slot) order
    n_good = 0
    for c, (res, nres) in enumerate(last):
        for d in range(n):
            for k in range(Bc):
                n_good += slot_ok(texts[d * B + c * Bc + k], res[d * Bc + k], int(nres[d * Bc + k]))
    launches0 = cl.launches()
    gathers0 = cl.gathers()
    sync_all()
    t0 = time.perf_counter()
    run(args.steps)
    sync_all()
    secs = time.perf_counter() - t0
    cfg = dict(config)
    run_info = {"parallelism": "ONE process, ft8b200_cluster_t: %d devices, slots sharded by device, records gathered by the library (grouped ncclAllGather, NCCL %d)" % (n, cl.nccl_version()),
                "executor": "one ft8b200_pipe_t of depth %d per device, %d batches of %d slots per device per step" % (args.depth, args.chunks, Bc),
                "sm_partition": part}
    out = {"impl": "cluster", "metric": METRIC, "value": n * B * args.steps / secs, "unit": "slots/s", "n_gpus": n, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": secs / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32+f32",
           "data": "synthetic (generated on each device by ft8b200_synth_raw)", "config": cfg, "run": run_info, "gpu_launches": int(cl.launches() - launches0),
           "nccl_gathers": int(cl.gathers() - gathers0), "verify": {"slots_decoded_to_their_own_message": int(n_good), "of": n * B},
           "timed": "host clock between synchronisations of all devices"}
    cl.close()
    emit(out)
    return 0


def reference_arm(args, rank, world, config):
    """The reference's own CPU implementation of the path on this box's host cores (rank 0 only)."""
    if rank != 0:
        return 0
    global _CPU_SLOTS
    cores = os.cpu_count() or 1
    n = max(4 * cores, 16)  # a few slots per worker per step
    # Inputs: the same synthetic slots as the CUDA arm, made by the synthesiser's bit-identical CPU twin (oracle/ft8_oracle_synth.c)
    # in the worker processes -- nothing of libft8b200 and no GPU is involved anywhere in this arm.
    try:
        import multiprocessing as mp
        shared = mp.RawArray("B", n * RAW_SLOT_BYTES)
        _CPU_SLOTS = np.frombuffer(shared, np.uint8).reshape(n, RAW_SLOT_BYTES)
        with mp.get_context("fork").Pool(cores) as pool:
            pool.map(_cpu_synth_slot, range(n), chunksize=1)
    except Exception as exc:  # pragma: no cover
        emit({"impl": "reference", "unavailable": f"input synthesis failed: {exc}"})
        return 0
    for _ in range(min(args.warmup, 1)):
        cpu_run(min(n, cores), cores)
    t = 0.0
    for _ in range(args.steps):
        secs, _ = cpu_run(n, cores)
        t += secs
    value = n * args.steps / t
    kind = cpu_kind()
    cfg = dict(config)   # the workload, word for word what the CUDA arm prints
    run_info = {"executor": "n/a (CPU arm)", "reference_sample": "%d slots per step over %d worker processes" % (n, cores)}
    out = {"impl": "reference", "metric": METRIC, "value": value, "unit": "slots/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": t / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32+f32",
           "data": "synthetic (same slots as the CUDA arm, made on the host by the synthesiser's bit-identical CPU twin)", "config": cfg, "run": run_info,
           "cpu_baseline": {"value": value, "unit": "slots/s", "cores": cores, "kind": kind,
                            "sample": "%d slots per step, one forked process per slot on %d cores (the reference itself is single-threaded)" % (n, cores)},
           "e2e": {"value": value, "unit": "slots/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(out)
    return 0


if __name__ == "__main__":
    sys.exit(main())
