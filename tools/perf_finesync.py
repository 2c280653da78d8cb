#!/usr/bin/env python3
"""Gain, false decodes and cost of fine-sync decoding (DESIGN.md section 2.4.4) on the GPU -> profiles/perf_finesync.json.

  * false decodes on 4096 seeded noise-only daemon slots (K = 120) against the hard-distance cap: the default cap
    (FT8B200_FINESYNC_DEFAULT_MAX_HARD) is the largest one at which fine sync decodes nothing;
  * decode rate against SNR (-16 ... -24 dB, 512 seeded single-signal GFSK slots per point, synthesised on the device) with BP alone,
    BP + fine sync, BP + OSD order 2 + AP and BP + OSD order 2 + AP + fine sync at that cap, for plain CQ messages and for non-CQ
    messages, with every decoded message that was never transmitted counted;
  * 128 crowded slots of 40 GFSK CQ messages (-24 ... -8 dB) at passes 1 and 2, fine sync off and on: transmitted messages in the
    spot records and records of messages never transmitted;
  * the decode stage's device time (ft8b200_set_profiling, which brackets BP, OSD, AP and fine sync) for a 128-slot batch of
    bench.py's workload and for 32 crowded slots at K = 500 / M = 200;
  * wall time per batch of the partitioned pipe (depth 3, 40 back-end SMs) with fine sync off and on;
  * with --parent-lib PATH: bench.py (fine sync off, the default) alternated with the parent build in one run.
usage: python tools/perf_finesync.py [out.json] [--parent-lib PATH]"""
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
from ft8b200_loader import load  # noqa: E402
from oracle.pyoracle import msg_dtype  # noqa: E402
from tools import ft8enc, synth  # noqa: E402
from tools.perf_ap import message_set  # noqa: E402
from tools.perf_osd import _Arr, amp_for  # noqa: E402

pkg = load()
DEV = torch.device("cuda:0")
CONFIGS = (("bp", 0, 0, 0), ("bp_fs", 0, 0, 1), ("osd2_ap", 2, 1, 0), ("osd2_ap_fs", 2, 1, 1))


def candidate_outputs(ctx, n_slots):
    """(ok, msg, fs, fs_hard) of pass 1 of the last batch, on the host; entries past a slot's candidate count zeroed."""
    w = ctx.workspace_ptrs()
    K = ctx.K
    ok = torch.as_tensor(_Arr(w["ok"], (n_slots, K), "|u1"), device=DEV).cpu().numpy()
    msg = torch.as_tensor(_Arr(w["msg"], (n_slots, K, 28), "|u1"), device=DEV).cpu().numpy().view(msg_dtype).reshape(n_slots, K)
    ncand = torch.as_tensor(_Arr(w["ncand"], (n_slots,), "<i4"), device=DEV).cpu().numpy()
    a, b = ctx.finesync_workspace_ptrs()
    fs = torch.as_tensor(_Arr(a, (n_slots, K), "|u1"), device=DEV).cpu().numpy() if a else np.zeros((n_slots, K), np.uint8)
    hard = torch.as_tensor(_Arr(b, (n_slots, K), "<i4"), device=DEV).cpu().numpy() if b else np.full((n_slots, K), -1, np.int32)
    for s in range(n_slots):
        ok[s, ncand[s]:] = 0
        fs[s, ncand[s]:] = 0
    return ok, msg, fs, hard


def run_slots(ctx, d_i, d_q):
    peak = torch.maximum(d_i.abs().amax(1), d_q.abs().amax(1)).contiguous()
    ctx.process_conditioned(d_i, d_q, peak)
    torch.cuda.synchronize()
    return candidate_outputs(ctx, d_i.shape[0])


def noise_sweep(n_slots=4096, batch=1024, caps=range(0, 175)):
    """Fine-sync decodes on noise-only slots at every cap: one run at cap 174 gives them all (the cap is the last gate), a message
    counting at cap c when one of its candidates decoded at a hard distance <= c."""
    ctx = pkg.Context(0)
    ctx.set_finesync(1, 174)
    other, hard_of, attempted = set(), {}, 0
    for b0 in range(0, n_slots, batch):
        d_i, d_q = ctx.synth_slots(pkg.make_signals([]), np.zeros(batch + 1, np.int32), 1.0, 0x0D5E, first_slot_index=b0)
        ok, msg, fs, hard = run_slots(ctx, d_i, d_q)
        attempted += int((fs > 0).sum())
        for s, k in zip(*np.nonzero(ok)):
            key = (b0 + s, bytes(msg[s, k]["text"]).decode())
            if fs[s, k] == 2:
                hard_of[key] = min(hard_of.get(key, 999), int(hard[s, k]))
            else:
                other.add(key)
    ctx.close()
    hards = np.array(sorted(hard_of.values()), np.int64)
    out = {"candidates_attempted": attempted, "bp_decodes": len(other), "fs_decodes_by_cap": {int(c): int((hards <= c).sum()) for c in caps},
           "fs_decodes_at_cap_174": sorted([s, t, h] for (s, t), h in hard_of.items())}
    ok_caps = [c for c in caps if out["fs_decodes_by_cap"][c] == 0]
    return out, max(ok_caps) if ok_caps else -1


def gain_row(kind, snr, cap, per_point=512, configs=CONFIGS):
    texts, sig = message_set(kind, snr, per_point)
    row = {"snr_db": snr, "slots": per_point}
    for name, osd, ap, fs_on in configs:
        ctx = pkg.Context(0)
        ctx.set_osd(osd, -1)
        ctx.set_ap(ap, -1)
        ctx.set_finesync(fs_on, cap)
        d_i, d_q = ctx.synth_slots(sig, np.arange(per_point + 1, dtype=np.int32), 1.0, 0xF5E + snr + (0 if kind == "cq" else 99), first_slot_index=0)
        ok, msg, fs, _ = run_slots(ctx, d_i, d_q)
        good = bad = by_fs = 0
        for s in range(per_point):
            got = {bytes(msg[s, k]["text"]).decode() for k in np.flatnonzero(ok[s])}
            other = {bytes(msg[s, k]["text"]).decode() for k in np.flatnonzero(ok[s] & (fs[s] != 2))}
            good += texts[s] in got
            by_fs += texts[s] in got and texts[s] not in other
            bad += len(got - {texts[s]})
        row[name] = {"decoded": good, "rate": good / per_point, "never_transmitted": bad, "decoded_only_by_fs": by_fs}
        ctx.close()
    return row


def gain_sweep(cap, snrs=range(-16, -25, -1)):
    out = {}
    for kind in ("cq", "non_cq"):
        rows = []
        for snr in snrs:
            rows.append(gain_row(kind, snr, cap))
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
    out = {"slots": n_slots, "messages_per_slot": per_slot}
    for passes in (1, 2):
        for fs_on in (0, 1):
            ctx = pkg.Context(0)
            ctx.set_passes(passes)
            ctx.set_finesync(fs_on, cap)
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
            out[f"passes{passes}_fs{fs_on}"] = {"transmitted_decoded": good, "never_transmitted": bad}
            print("crowded", passes, fs_on, good, bad, flush=True)
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
        for label, osd, ap, fs_on in CONFIGS:
            ctx = pkg.Context(0, max_candidates=K, max_messages=M)
            ctx.set_osd(osd, -1)
            ctx.set_ap(ap, -1)
            ctx.set_finesync(fs_on, cap)
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
    out = {"back_sms_requested": back_sms, "depth": 3, "slots_per_batch": 128}
    for fs_on in (0, 1, 0, 1):  # alternated, twice each
        p = pkg.Pipe(0, depth=3)
        out["provisioned"] = p.set_partition(back_sms)
        p.set_finesync(fs_on, cap)
        for _ in range(4):
            p.submit(batch, 128)
            p.collect(128)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k in range(batches):
            if p.in_flight() == 3:
                p.collect(128)
            p.submit(batch, 128)
        while p.in_flight():
            p.collect(128)
        out.setdefault(f"fs{fs_on}_ms_per_batch", []).append((time.perf_counter() - t0) * 1e3 / batches)
        p.close()
    print("pipe", out, flush=True)
    return out


def bench_ab(parent_lib, steps=20, warmup=5):
    """bench.py with this tree's library and with the parent's (FT8B200_LIB_PATH), alternated, fine sync off."""
    args = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup), "--cpu-slots", "8", "--no-configs"]
    out = {"what": " ".join(["bench.py"] + args[2:]) + ", fine sync off (the default), this tree against the parent build, alternated in one run",
           "order": [], "slots_per_s": {}}
    for rep in (1, 2):
        for who in ("new", "parent"):
            env = dict(os.environ)
            if who == "parent":
                env["FT8B200_LIB_PATH"] = parent_lib
            p = subprocess.run(args, env=env, capture_output=True, text=True, cwd=ROOT)
            line = [ln for ln in p.stdout.splitlines() if ln.startswith("{")][-1]
            key = f"{who}_{rep}"
            out["order"].append(key)
            out["slots_per_s"][key] = json.loads(line)["value"]
            print("bench", key, out["slots_per_s"][key], flush=True)
    return out


def main():
    argv = sys.argv[1:]
    parent = None
    if "--parent-lib" in argv:
        i = argv.index("--parent-lib")
        parent = argv[i + 1]
        del argv[i:i + 2]
    path = argv[0] if argv else os.path.join(ROOT, "profiles", "perf_finesync.json")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    noise, cap = noise_sweep()
    print("noise", {c: n for c, n in noise["fs_decodes_by_cap"].items() if n}, "default cap", cap, flush=True)
    out = {"gpu": gpu, "default_max_hard": cap, "false_decodes_4096_noise_slots_k120": noise}
    out["decode_stage_time"] = stage4_times(cap)
    out["pipe_partitioned"] = pipe_times(cap)
    out["gain"] = gain_sweep(cap)
    out["never_transmitted_from_fs"] = sum(r["bp_fs"]["never_transmitted"] - r["bp"]["never_transmitted"]
                                           + r["osd2_ap_fs"]["never_transmitted"] - r["osd2_ap"]["never_transmitted"]
                                           for rows in out["gain"].values() for r in rows)
    out["gain_minus18_to_minus20"] = {k: sum(r[k]["decoded"] for r in out["gain"]["cq"] + out["gain"]["non_cq"] if -20 <= r["snr_db"] <= -18)
                                      for k, *_ in CONFIGS}
    out["crowded"] = crowded(cap)
    if parent:
        out["bench_ab"] = bench_ab(parent)
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
