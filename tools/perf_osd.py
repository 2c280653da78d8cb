#!/usr/bin/env python3
"""Cost and gain of ordered-statistics decoding (OSD, DESIGN.md section 2.4.1) on the GPU -> profiles/perf_osd.json.

  * false decodes on 4096 seeded noise-only daemon slots (K = 120) at orders 1 and 2 against the hard-distance cap: the default
    cap (FT8B200_OSD_DEFAULT_MAX_HARD) is the largest one with at most 2 OSD-decoded messages at order 2;
  * decode rate against SNR (-16 ... -26 dB, 512 seeded single-signal slots per point, synthesised on the device) with OSD off,
    at order 1 and at order 2 with that cap, and the messages decoded that were never transmitted;
  * the decode stage's device time (ft8b200_set_profiling, which brackets BP and OSD) for a 128-slot batch of bench.py's
    workload and for 32 crowded slots at K = 500 / M = 200 (BASELINE config #3);
  * wall time per batch of the partitioned pipe with OSD off and on.
usage: python tools/perf_osd.py [out.json]"""
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

pkg = load()
DEV = torch.device("cuda:0")


class _Arr:
    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2}


def candidate_outputs(ctx, n_slots):
    """(ok, msg, osd, osd_hard) of the last batch, on the host."""
    w = ctx.workspace_ptrs()
    K = ctx.K
    ok = torch.as_tensor(_Arr(w["ok"], (n_slots, K), "|u1"), device=DEV).cpu().numpy()
    msg = torch.as_tensor(_Arr(w["msg"], (n_slots, K, 28), "|u1"), device=DEV).cpu().numpy().view(msg_dtype).reshape(n_slots, K)
    ncand = torch.as_tensor(_Arr(w["ncand"], (n_slots,), "<i4"), device=DEV).cpu().numpy()
    a, b = ctx.osd_workspace_ptrs()
    osd = torch.as_tensor(_Arr(a, (n_slots, K), "|u1"), device=DEV).cpu().numpy() if a else np.zeros((n_slots, K), np.uint8)
    hard = torch.as_tensor(_Arr(b, (n_slots, K), "<i4"), device=DEV).cpu().numpy() if b else np.full((n_slots, K), -1, np.int32)
    for s in range(n_slots):  # entries past a slot's candidate count hold stale rows
        ok[s, ncand[s]:] = 0
        osd[s, ncand[s]:] = 0
    return ok, msg, osd, hard


def run_slots(ctx, d_i, d_q):
    peak = torch.maximum(d_i.abs().amax(1), d_q.abs().amax(1)).contiguous()
    ctx.process_conditioned(d_i, d_q, peak)
    torch.cuda.synchronize()
    return candidate_outputs(ctx, d_i.shape[0])


def amp_for(snr_db, sigma=1.0):
    return float(np.sqrt(2.0 * sigma ** 2 * (2500.0 / 3200.0) * 10.0 ** (snr_db / 10.0)))


def noise_sweep(n_slots=4096, batch=1024, caps=range(0, 175)):
    out = {}
    for order in (1, 2):
        ctx = pkg.Context(0)
        ctx.set_osd(order, 174)  # no cap: the winner does not depend on it, so one run gives every cap
        bp, hards = set(), []
        for b0 in range(0, n_slots, batch):
            first = np.zeros(batch + 1, np.int32)
            d_i, d_q = ctx.synth_slots(pkg.make_signals([]), first, 1.0, 0x0D5E, first_slot_index=b0)
            ok, msg, osd, hard = run_slots(ctx, d_i, d_q)
            seen = set()
            for s, k in zip(*np.nonzero(ok)):
                key = (b0 + s, bytes(msg[s, k]["text"]))
                if osd[s, k] == 2:
                    if key not in seen:
                        seen.add(key)
                        hards.append(int(hard[s, k]))
                else:
                    bp.add(key)
        ctx.close()
        hards = np.array(hards, np.int64)
        out[f"order{order}"] = {"bp_decodes": len(bp), "osd_decodes_by_cap": {int(c): int((hards <= c).sum()) for c in caps},
                                "osd_winner_hard_distances": sorted(int(h) for h in hards)}
    ok_caps = [c for c, n in out["order2"]["osd_decodes_by_cap"].items() if n <= 2]
    default = max(ok_caps) if ok_caps else 0
    return out, default


def sensitivity(cap, snrs=range(-16, -27, -1), per_point=512):
    rows = []
    for snr in snrs:
        rng = np.random.Generator(np.random.PCG64(0x05D + 1000 * (-snr)))
        texts, items = [], []
        for s in range(per_point):
            to, de, ex = synth.random_message(rng)
            texts.append(f"{to} {de} {ex}")
            items.append((pkg.pack77_std(to, de, ex), float(rng.uniform(300.0, 1300.0)), float(0.5 + rng.uniform(-0.3, 0.3)), amp_for(snr)))
        sig = pkg.make_signals(items, gfsk=True)
        row = {"snr_db": snr, "slots": per_point}
        for order in (0, 1, 2):
            ctx = pkg.Context(0)
            ctx.set_osd(order, cap)
            d_i, d_q = ctx.synth_slots(sig, np.arange(per_point + 1, dtype=np.int32), 1.0, 0x5E45 + snr, first_slot_index=0)
            ok, msg, osd, _ = run_slots(ctx, d_i, d_q)
            good = bad = by_osd = 0
            for s in range(per_point):
                got = {bytes(msg[s, k]["text"]).decode() for k in np.flatnonzero(ok[s])}
                osd_got = {bytes(msg[s, k]["text"]).decode() for k in np.flatnonzero(osd[s] == 2)}
                good += texts[s] in got
                by_osd += texts[s] in osd_got and texts[s] not in {bytes(msg[s, k]["text"]).decode() for k in np.flatnonzero(ok[s] & (osd[s] != 2))}
                bad += len(got - {texts[s]})
            row[f"order{order}"] = {"decoded": good, "rate": good / per_point, "never_transmitted": bad, "decoded_only_by_osd": by_osd}
            ctx.close()
        rows.append(row)
        print(row, flush=True)
    return rows


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
        for order in (0, 1, 2):
            ctx = pkg.Context(0, max_candidates=K, max_messages=M)
            ctx.set_osd(order, cap)
            ctx.set_profiling(True)
            for _ in range(3):
                run(ctx)
            torch.cuda.synchronize()
            ts = []
            for _ in range(reps):
                run(ctx)
                ts.append(ctx.stage_times()["decode"])
            res[f"order{order}"] = {"decode_stage_ms_median": float(np.median(ts)), "decode_stage_ms_min": float(np.min(ts))}
            ctx.close()
        out[name] = res
        print(name, res, flush=True)
    return out


def pipe_times(cap, back_sms=40, batches=24):
    batch, _ = bench.gen_batch(128, 0, DEV)
    out = {"back_sms_requested": back_sms, "slots_per_batch": 128}
    for order in (0, 2):
        p = pkg.Pipe(0, depth=3)
        out["provisioned"] = p.set_partition(back_sms)
        p.set_osd(order, cap)
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
        ms = (time.perf_counter() - t0) * 1e3 / batches
        out[f"order{order}_ms_per_batch"] = ms
        p.close()
    print("pipe", out, flush=True)
    return out


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "perf_osd.json")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    noise, cap = noise_sweep()
    print("noise", {k: v["osd_decodes_by_cap"] for k, v in noise.items()}, "default cap", cap, flush=True)
    out = {"gpu": gpu, "default_max_hard": cap, "false_decodes_4096_noise_slots_k120": noise}
    out["decode_stage_time"] = stage4_times(cap)
    out["pipe_partitioned"] = pipe_times(cap)
    out["sensitivity"] = sensitivity(cap)
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
