#!/usr/bin/env python3
"""Gain, false decodes and cost of deep fine sync (DESIGN.md section 2.4.6) on the GPU -> profiles/perf_finesync_deep.json.

  * false decodes on 4096 seeded noise-only daemon slots (K = 120) with OSD {0, 2} x AP {0, 1}, fine sync and deep mode on, from cap
    174 down (noise_sweep): the default cap (FT8B200_FINESYNC_DEEP_DEFAULT_MAX_HARD) is the largest at which deep mode decodes nothing;
  * decode rate against SNR (-16 ... -24 dB, 512 seeded single-signal GFSK slots per point, synthesised on the device) with
    BP + fine sync and BP + OSD order 2 + AP + fine sync, each without and with deep mode, for plain CQ messages and for non-CQ
    messages, with every decoded message that was never transmitted counted and the new decodes broken down by fs_how;
  * 128 crowded slots of 40 GFSK CQ messages (-24 ... -8 dB) at passes 1 and 2, fine sync on, deep mode off and on;
  * the decode stage's device time (ft8b200_set_profiling) for a 128-slot batch of bench.py's workload and for 32 crowded slots at
    K = 500 / M = 200, and the partitioned pipe's wall time per batch, deep mode off and on;
  * with --parent-lib PATH: bench.py (deep mode off, the default) alternated with the parent build in one run.
usage: python tools/perf_finesync_deep.py [out.json] [--parent-lib PATH] [--sections noise,cost,gain,crowded,bench] [--quick]"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from tools import ft8enc, synth  # noqa: E402
from tools.perf_ap import message_set  # noqa: E402
from tools.perf_finesync import bench_ab, candidate_outputs, pkg  # noqa: E402
from tools.perf_osd import _Arr, amp_for  # noqa: E402

DEV = torch.device("cuda:0")
# (label, OSD order, AP, deep); fine sync is on in all of them
CONFIGS = (("bp_fs", 0, 0, 0), ("bp_fs_deep", 0, 0, 1), ("osd2_ap_fs", 2, 1, 0), ("osd2_ap_fs_deep", 2, 1, 1))
HOW = {1 + 3 * s + d: f"{'abc'[s]}_{('bp', 'osd', 'ap')[d]}" for s in range(3) for d in range(3)}


def make_ctx(osd, ap, deep, cap, **cfg):
    ctx = pkg.Context(0, **cfg)
    ctx.set_osd(osd, -1)
    ctx.set_ap(ap, -1)
    ctx.set_finesync(1, -1)
    ctx.set_finesync_deep(deep, cap)
    return ctx


def run_slots(ctx, d_i, d_q):
    peak = torch.maximum(d_i.abs().amax(1), d_q.abs().amax(1)).contiguous()
    ctx.process_conditioned(d_i, d_q, peak)
    torch.cuda.synchronize()
    n = d_i.shape[0]
    ok, msg, fs, hard = candidate_outputs(ctx, n)
    p = ctx.finesync_deep_workspace_ptrs()
    how = torch.as_tensor(_Arr(p, (n, ctx.K), "|u1"), device=DEV).cpu().numpy() if p else np.zeros((n, ctx.K), np.uint8)
    how = np.where(ok > 0, how, 0)
    return ok, msg, fs, hard, how


def noise_at(cap, n_slots, batch):
    out = {}
    for osd in (0, 2):
        for ap in (0, 1):
            ctx = make_ctx(osd, ap, 1, cap)
            deep, fs_a, other = [], 0, 0
            for b0 in range(0, n_slots, batch):
                d_i, d_q = ctx.synth_slots(pkg.make_signals([]), np.zeros(batch + 1, np.int32), 1.0, 0x0D5E, first_slot_index=b0)
                ok, msg, fs, hard, how = run_slots(ctx, d_i, d_q)
                for s, k in zip(*np.nonzero(ok)):
                    if how[s, k] >= 2:
                        deep.append([b0 + int(s), bytes(msg[s, k]["text"]).decode(), HOW[int(how[s, k])], int(hard[s, k])])
                    elif fs[s, k] == 2:
                        fs_a += 1
                    else:
                        other += 1
            ctx.close()
            hards = np.array([d[3] for d in deep], np.int64)
            out[f"osd{osd}_ap{ap}"] = {"deep_decodes": deep, "set_a_bp_decodes": fs_a, "other_decodes": other,
                                        "deep_decodes_by_cap": {int(c): int((hards <= c).sum()) for c in range(cap + 1)}}
            print("noise", cap, osd, ap, len(deep), fs_a, other, flush=True)
    return out


def noise_sweep(n_slots=4096, batch=1024):
    """-> ({cap: runs}, default cap).  A run at cap c gives the decodes at every cap from the largest decoded hard distance up to c
    (the steps before the one that accepted rejected for reasons other than the cap); below it a later step may accept instead, so
    the candidate cap just below the smallest decoded distance is run again until a run decodes nothing."""
    runs, cap = {}, 174
    while cap >= 0:
        r = noise_at(cap, n_slots, batch)
        runs[cap] = r
        hards = [d[3] for v in r.values() for d in v["deep_decodes"]]
        if not hards:
            break
        cap = min(hards) - 1
    return runs, cap


def gain_row(kind, snr, cap, per_point=512):
    texts, sig = message_set(kind, snr, per_point)
    row = {"snr_db": snr, "slots": per_point}
    for name, osd, ap, deep in CONFIGS:
        ctx = make_ctx(osd, ap, deep, cap)
        d_i, d_q = ctx.synth_slots(sig, np.arange(per_point + 1, dtype=np.int32), 1.0, 0xF5E + snr + (0 if kind == "cq" else 99), first_slot_index=0)
        ok, msg, fs, _, how = run_slots(ctx, d_i, d_q)
        good = bad = 0
        by_how, bad_by = {}, {}
        for s in range(per_point):
            got = {bytes(msg[s, k]["text"]).decode() for k in np.flatnonzero(ok[s])}
            good += texts[s] in got
            bad += len(got - {texts[s]})
            for k in np.flatnonzero(ok[s]):   # which step decoded a message that was never transmitted
                if bytes(msg[s, k]["text"]).decode() != texts[s]:
                    h = HOW.get(int(how[s, k]), "before_fine_sync") if fs[s, k] == 2 else "before_fine_sync"
                    bad_by[h] = bad_by.get(h, 0) + 1
            if texts[s] in got:
                # the step that decoded the transmitted message where nothing before deep mode's steps did
                ks = [k for k in np.flatnonzero(ok[s]) if bytes(msg[s, k]["text"]).decode() == texts[s]]
                if all(how[s, k] >= 2 for k in ks):
                    h = HOW[int(min(how[s, k] for k in ks))]
                    by_how[h] = by_how.get(h, 0) + 1
        row[name] = {"decoded": good, "rate": good / per_point, "never_transmitted": bad, "decoded_only_by_deep_steps": by_how,
                     "never_transmitted_by_step": bad_by}
        ctx.close()
    return row


def gain_sweep(cap, snrs, per_point):
    out = {}
    for kind in ("cq", "non_cq"):
        rows = []
        for snr in snrs:
            rows.append(gain_row(kind, snr, cap, per_point))
            print(kind, rows[-1], flush=True)
        out[kind] = rows
    return out


def crowded(cap, n_slots=128, per_slot=40):
    rng = np.random.Generator(np.random.PCG64(0xC40))
    items, sent = [], []
    for _ in range(n_slots):
        keys = set()
        for _ in range(per_slot):
            call, grid = synth.random_call(rng), synth.random_grid(rng)
            keys.add((call, grid))
            items.append((pkg.pack77_std("CQ", call, grid), float(rng.uniform(100, 2400)), float(0.5 + rng.uniform(-0.3, 0.3)),
                          amp_for(float(rng.uniform(-24, -8)))))
        sent.append(keys)
    first = np.arange(0, n_slots * per_slot + 1, per_slot, dtype=np.int32)
    out = {"slots": n_slots, "messages_per_slot": per_slot, "fine_sync": 1}
    for passes in (1, 2):
        for deep in (0, 1):
            ctx = make_ctx(0, 0, deep, cap)
            ctx.set_passes(passes)
            d_i, d_q = ctx.synth_slots(pkg.make_signals(items, gfsk=True), first, 1.0, 0xC40)
            peak = torch.maximum(d_i.abs().amax(1), d_q.abs().amax(1)).contiguous()
            ctx.process_conditioned(d_i, d_q, peak)
            res, nres = ctx.fetch_results(n_slots)
            good = bad = 0
            for s in range(n_slots):
                for r in res[s][:int(nres[s])]:
                    key = (r["call"].decode(), r["loc"].decode())
                    good += key in sent[s]
                    bad += key not in sent[s]
            out[f"passes{passes}_deep{deep}"] = {"transmitted_decoded": good, "never_transmitted": bad}
            print("crowded", passes, deep, good, bad, flush=True)
            ctx.close()
    return out


def stage4_times(cap, reps=10):
    out = {}
    batch, _ = bench.gen_batch(128, 0, DEV)
    rng_slots = [synth.crowded_band(ft8enc, 60, 500 + s)[:2] for s in range(32)]
    peaks = [max(np.abs(i).max(), np.abs(q).max()) for i, q in rng_slots]
    ci = torch.from_numpy(np.stack([i for i, _ in rng_slots])).to(DEV)
    cq = torch.from_numpy(np.stack([q for _, q in rng_slots])).to(DEV)
    cp = torch.tensor(peaks, dtype=torch.float32, device=DEV)
    for name, K, M, run in (("headline_128_raw_slots_k120", 120, 50, lambda c: c.process_raw(batch, 128)),
                            ("config3_32_crowded_slots_k500", 500, 200, lambda c: c.process_conditioned(ci, cq, cp))):
        res = {}
        for label, osd, ap, deep in CONFIGS:
            ctx = make_ctx(osd, ap, deep, cap, max_candidates=K, max_messages=M)
            ctx.set_profiling(True)
            for _ in range(3):
                run(ctx)
            torch.cuda.synchronize()
            ts = []
            for _ in range(reps):
                run(ctx)
                ts.append(ctx.stage_times()["decode"])
            res[label] = {"decode_stage_ms_median": float(np.median(ts)), "decode_stage_ms_min": float(np.min(ts))}
            ctx.close()
        out[name] = res
        print(name, res, flush=True)
    return out


def pipe_times(cap, back_sms=40, batches=24):
    batch, _ = bench.gen_batch(128, 0, DEV)
    out = {"back_sms_requested": back_sms, "depth": 3, "slots_per_batch": 128, "fine_sync": 1}
    for deep in (0, 1, 0, 1):  # alternated, twice each
        p = pkg.Pipe(0, depth=3)
        out["provisioned"] = p.set_partition(back_sms)
        p.set_finesync(1, -1)
        p.set_finesync_deep(deep, cap)
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
        out.setdefault(f"deep{deep}_ms_per_batch", []).append((time.perf_counter() - t0) * 1e3 / batches)
        p.close()
    print("pipe", out, flush=True)
    return out


def main():
    argv = sys.argv[1:]
    opt = {}
    for name in ("--parent-lib", "--sections"):
        if name in argv:
            i = argv.index(name)
            opt[name] = argv[i + 1]
            del argv[i:i + 2]
    parent = opt.get("--parent-lib")
    # what to measure; the results are merged into an existing file, so that the sections can run in separate invocations
    sections = opt.get("--sections", "noise,cost,gain,crowded,bench").split(",")
    quick = "--quick" in argv   # a rehearsal at toy sizes
    argv = [a for a in argv if a != "--quick"]
    path = argv[0] if argv else os.path.join(ROOT, "profiles", "perf_finesync_deep.json")
    out = json.load(open(path)) if os.path.exists(path) else {}
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    out.setdefault("gpu_by_section", {}).update({sec: gpu for sec in sections})
    if "noise" in sections:
        noise, cap = noise_sweep(n_slots=64, batch=64) if quick else noise_sweep()
        out.update(default_max_hard=cap, false_decodes_4096_noise_slots_k120_by_run_cap=noise)
        print("default cap", cap, flush=True)
    cap = max(out.get("default_max_hard", 174), 0)
    if "cost" in sections:
        out["decode_stage_time"] = stage4_times(cap, reps=2 if quick else 10)
        out["pipe_partitioned"] = pipe_times(cap, batches=4 if quick else 24)
    if "gain" in sections:
        out["gain"] = gain_sweep(cap, [-19] if quick else range(-16, -25, -1), 16 if quick else 512)
        out["never_transmitted_from_deep"] = sum(r["bp_fs_deep"]["never_transmitted"] - r["bp_fs"]["never_transmitted"]
                                                 + r["osd2_ap_fs_deep"]["never_transmitted"] - r["osd2_ap_fs"]["never_transmitted"]
                                                 for rows in out["gain"].values() for r in rows)
        out["gain_sum_over_snrs"] = {k: sum(r[k]["decoded"] for r in out["gain"]["cq"] + out["gain"]["non_cq"]) for k, *_ in CONFIGS}
    if "crowded" in sections:
        out["crowded"] = crowded(cap, n_slots=8 if quick else 128)
    if "bench" in sections and parent:
        out["bench_ab"] = bench_ab(parent, steps=3 if quick else 20, warmup=1 if quick else 5)
        out["bench_ab"]["what"] = out["bench_ab"]["what"].replace("fine sync off (the default)", "fine sync and deep mode off (the defaults)")
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
