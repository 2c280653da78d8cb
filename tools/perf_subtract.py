#!/usr/bin/env python3
"""Gain and cost of multi-pass decoding with signal subtraction (DESIGN.md section 2.4.2) on the GPU -> profiles/perf_subtract.json.

  * gain: transmitted messages decoded at passes 1 / 2 / 3 on seeded crowded GFSK slots (10 / 20 / 40 / 60 CQ messages a slot,
    SNR uniform in -20 ... -8 dB, tone-0 frequency uniform in 100 ... 1500 Hz so that signals overlap, DT 0.5 +- 0.3 s);
  * false decodes: records that were never transmitted on those slots, and on 4096 seeded noise-only slots;
  * cost: device time of subtraction + later passes (ft8b200_stage_times' seventh stage) per 128-slot batch, for bench.py's
    workload (raw IQ, process_raw) and for 128 crowded slots of 40 messages;
  * executor throughput: wall time per batch of the partitioned pipe at passes 1 and 2.
The card's name and power limit are read in the same run.
usage: python tools/perf_subtract.py [out.json]"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

from tools import synth  # noqa: E402


def amp_for(snr_db, sigma=1.0):
    """Amplitude of a 3200 sps complex signal at snr_db in 2500 Hz against noise of sigma per rail."""
    return float(np.sqrt(2.0 * sigma ** 2 * (2500.0 / 3200.0) * 10.0 ** (snr_db / 10.0)))


def crowded_items(pkg, n_slots, n_signals, seed, snr_lo=-20.0, snr_hi=-8.0):
    """Seeded CQ messages -> (signal_dtype array, first int32[n_slots + 1], [set of (call, loc) bytes per slot])."""
    rng = np.random.Generator(np.random.PCG64(seed))
    items, sent = [], []
    for _ in range(n_slots):
        here = set()
        for _ in range(n_signals):
            call, loc = synth.random_call(rng), synth.random_grid(rng)
            items.append((pkg.pack77_std("CQ", call, loc), float(rng.uniform(100.0, 1500.0)), float(0.5 + rng.uniform(-0.3, 0.3)),
                          amp_for(float(rng.uniform(snr_lo, snr_hi)))))
            here.add((call.encode(), loc.encode()))
        sent.append(here)
    return pkg.make_signals(items, gfsk=True), np.arange(0, n_slots * n_signals + 1, n_signals, dtype=np.int32), sent


def crowded_slots(pkg, ctx, n_slots, n_signals, seed, **kw):
    """Device slots (I, Q float32 [n, 48000], noise sigma 1) + the transmitted (call, loc) sets."""
    sig, first, sent = crowded_items(pkg, n_slots, n_signals, seed, **kw)
    d_i, d_q = ctx.synth_slots(sig, first, 1.0, seed)
    return d_i, d_q, sent


def score(res, nres, sent):
    """(decoded transmitted messages, records never transmitted) over the slots."""
    good = bad = 0
    for s in range(len(sent)):
        got = {(bytes(r["call"]), bytes(r["loc"])) for r in res[s][:int(nres[s])]}
        good += len(got & sent[s])
        bad += sum((bytes(r["call"]), bytes(r["loc"])) not in sent[s] for r in res[s][:int(nres[s])])
    return good, bad


def run_conditioned(ctx, d_i, d_q):
    import torch
    peak = torch.maximum(d_i.abs().amax(1), d_q.abs().amax(1)).contiguous()
    ctx.process_conditioned(d_i, d_q, peak)
    return ctx.fetch_results(d_i.shape[0])


def gain(pkg, n_slots=128, crowding=(10, 20, 40, 60)):
    rows = []
    for n_sig in crowding:
        row = {"signals_per_slot": n_sig, "slots": n_slots, "transmitted": n_slots * n_sig}
        for passes in (1, 2, 3):
            ctx = pkg.Context(0)
            ctx.set_passes(passes)
            d_i, d_q, sent = crowded_slots(pkg, ctx, n_slots, n_sig, 0x5B7 + n_sig)
            good, bad = score(*run_conditioned(ctx, d_i, d_q), sent)
            row[f"passes{passes}"] = {"decoded": good, "never_transmitted": bad}
            ctx.close()
        rows.append(row)
        print(row, flush=True)
    return rows


def noise_only(pkg, n_slots=4096, batch=1024):
    out = {}
    for passes in (1, 2, 3):
        ctx = pkg.Context(0)
        ctx.set_passes(passes)
        n = 0
        for b0 in range(0, n_slots, batch):
            d_i, d_q = ctx.synth_slots(pkg.make_signals([]), np.zeros(batch + 1, np.int32), 1.0, 0x0D5E, first_slot_index=b0)
            _, nres = run_conditioned(ctx, d_i, d_q)
            n += int(nres.sum())
        out[f"passes{passes}_records"] = n
        ctx.close()
    print("noise", out, flush=True)
    return out


def cost(pkg, reps=10):
    import torch
    import bench
    dev = torch.device("cuda:0")
    batch, _ = bench.gen_batch(128, 0, dev)
    out = {}
    tmp = pkg.Context(0)
    ci, cq, _ = crowded_slots(pkg, tmp, 128, 40, 0xC057)
    tmp.close()
    cp = torch.maximum(ci.abs().amax(1), cq.abs().amax(1)).contiguous()
    for name, run in (("bench_128_raw_slots", lambda c: c.process_raw(batch, 128)),
                      ("crowded_128_slots_40_signals", lambda c: c.process_conditioned(ci, cq, cp))):
        res = {}
        for passes in (1, 2, 3):
            ctx = pkg.Context(0)
            ctx.set_passes(passes)
            ctx.set_profiling(True)
            for _ in range(3):
                run(ctx)
            torch.cuda.synchronize()
            later, total = [], []
            for _ in range(reps):
                run(ctx)
                t = ctx.stage_times()
                later.append(t.get("later_passes", 0.0))
                total.append(sum(v for k, v in t.items() if k in ("waterfall", "sync", "decode", "spots", "later_passes") and v > 0))
            res[f"passes{passes}"] = {"later_passes_ms_median": float(np.median(later)), "back_end_ms_median": float(np.median(total))}
            ctx.close()
        out[name] = res
        print(name, res, flush=True)
    return out


def pipe_times(pkg, back_sms=40, batches=24):
    import torch
    import bench
    batch, _ = bench.gen_batch(128, 0, torch.device("cuda:0"))
    out = {"back_sms_requested": back_sms, "slots_per_batch": 128}
    for passes in (1, 2):
        p = pkg.Pipe(0, depth=3)
        out["provisioned"] = p.set_partition(back_sms)
        p.set_passes(passes)
        for _ in range(4):
            p.submit(batch, 128)
            p.collect(128)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(batches):
            if p.in_flight() == 3:
                p.collect(128)
            p.submit(batch, 128)
        while p.in_flight():
            p.collect(128)
        out[f"passes{passes}_ms_per_batch"] = (time.perf_counter() - t0) * 1e3 / batches
        p.close()
    print("pipe", out, flush=True)
    return out


def main():
    from ft8b200_loader import load
    pkg = load()
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "perf_subtract.json")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    out = {"gpu": gpu}
    out["gain"] = gain(pkg)
    out["false_decodes_4096_noise_slots"] = noise_only(pkg)
    out["cost_per_128_slot_batch"] = cost(pkg)
    out["pipe_partitioned"] = pipe_times(pkg)
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
