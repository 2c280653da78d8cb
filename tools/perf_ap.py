#!/usr/bin/env python3
"""Cost and gain of a-priori (AP) decoding of "CQ ??? ???" (DESIGN.md section 2.4.3) on the GPU -> profiles/perf_ap.json.

  * false decodes on 4096 seeded noise-only daemon slots (K = 120) against the hard-distance cap, with OSD off and at order 2: the
    default cap (FT8B200_AP_DEFAULT_MAX_HARD) is the largest one at which AP decodes nothing in either;
  * decode rate against SNR (-16 ... -24 dB, 512 seeded single-signal GFSK slots per point, synthesised on the device) with BP
    alone, BP + AP, BP + OSD order 2 and BP + OSD order 2 + AP at that cap, for plain CQ messages and for non-CQ messages
    ("K1ABC W9XYZ FN42" forms), with every decoded message that was never transmitted counted;
  * the decode stage's device time (ft8b200_set_profiling, which brackets BP, OSD and AP) for a 128-slot batch of bench.py's
    workload and for 32 crowded slots at K = 500 / M = 200;
  * wall time per batch of the partitioned pipe (depth 3, 40 back-end SMs) with AP off and on.
usage: python tools/perf_ap.py [out.json]"""
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
from tools.perf_osd import _Arr, amp_for  # noqa: E402

pkg = load()
DEV = torch.device("cuda:0")
CONFIGS = (("bp", 0, 0), ("bp_ap", 0, 1), ("osd2", 2, 0), ("osd2_ap", 2, 1))


def candidate_outputs(ctx, n_slots):
    """(ok, msg, ap, ap_hard) of the last batch, on the host; entries past a slot's candidate count zeroed."""
    w = ctx.workspace_ptrs()
    K = ctx.K
    ok = torch.as_tensor(_Arr(w["ok"], (n_slots, K), "|u1"), device=DEV).cpu().numpy()
    msg = torch.as_tensor(_Arr(w["msg"], (n_slots, K, 28), "|u1"), device=DEV).cpu().numpy().view(msg_dtype).reshape(n_slots, K)
    ncand = torch.as_tensor(_Arr(w["ncand"], (n_slots,), "<i4"), device=DEV).cpu().numpy()
    a, b = ctx.ap_workspace_ptrs()
    ap = torch.as_tensor(_Arr(a, (n_slots, K), "|u1"), device=DEV).cpu().numpy() if a else np.zeros((n_slots, K), np.uint8)
    hard = torch.as_tensor(_Arr(b, (n_slots, K), "<i4"), device=DEV).cpu().numpy() if b else np.full((n_slots, K), -1, np.int32)
    for s in range(n_slots):
        ok[s, ncand[s]:] = 0
        ap[s, ncand[s]:] = 0
    return ok, msg, ap, hard


def run_slots(ctx, d_i, d_q):
    peak = torch.maximum(d_i.abs().amax(1), d_q.abs().amax(1)).contiguous()
    ctx.process_conditioned(d_i, d_q, peak)
    torch.cuda.synchronize()
    return candidate_outputs(ctx, d_i.shape[0])


def noise_sweep(n_slots=4096, batch=1024, caps=range(0, 175)):
    """AP-decoded messages on noise-only slots at every cap: one run at cap 174 gives them all (the cap is the only gate that
    depends on it), a message counting at cap c when one of its candidates decoded at a hard distance <= c."""
    out = {}
    for osd in (0, 2):
        ctx = pkg.Context(0)
        ctx.set_osd(osd, -1)
        ctx.set_ap(1, 174)
        other, hard_of = set(), {}
        for b0 in range(0, n_slots, batch):
            d_i, d_q = ctx.synth_slots(pkg.make_signals([]), np.zeros(batch + 1, np.int32), 1.0, 0x0D5E, first_slot_index=b0)
            ok, msg, ap, hard = run_slots(ctx, d_i, d_q)
            for s, k in zip(*np.nonzero(ok)):
                key = (b0 + s, bytes(msg[s, k]["text"]).decode())
                if ap[s, k] == 2:
                    hard_of[key] = min(hard_of.get(key, 999), int(hard[s, k]))
                else:
                    other.add(key)
        ctx.close()
        hards = np.array(sorted(hard_of.values()), np.int64)
        out[f"osd{osd}"] = {"bp_or_osd_decodes": len(other), "ap_decodes_by_cap": {int(c): int((hards <= c).sum()) for c in caps},
                            "ap_decodes_at_cap_174": sorted([s, t, h] for (s, t), h in hard_of.items())}
    ok_caps = [c for c in caps if all(out[k]["ap_decodes_by_cap"][c] == 0 for k in out)]
    return out, max(ok_caps) if ok_caps else 0


def message_set(kind, snr, per_point):
    rng = np.random.Generator(np.random.PCG64(0xA9 + 1000 * (-snr) + (0 if kind == "cq" else 7)))
    texts, items = [], []
    for _ in range(per_point):
        to = "CQ" if kind == "cq" else synth.random_call(rng)
        de, ex = synth.random_call(rng), synth.random_grid(rng)
        texts.append(f"{to} {de} {ex}")
        items.append((pkg.pack77_std(to, de, ex), float(rng.uniform(300.0, 1300.0)), float(0.5 + rng.uniform(-0.3, 0.3)), amp_for(snr)))
    return texts, pkg.make_signals(items, gfsk=True)


def gain_row(kind, snr, cap, per_point=512, configs=CONFIGS):
    texts, sig = message_set(kind, snr, per_point)
    row = {"snr_db": snr, "slots": per_point}
    for name, osd, ap in configs:
        ctx = pkg.Context(0)
        ctx.set_osd(osd, -1)
        ctx.set_ap(ap, cap)
        d_i, d_q = ctx.synth_slots(sig, np.arange(per_point + 1, dtype=np.int32), 1.0, 0xA95E + snr + (0 if kind == "cq" else 99), first_slot_index=0)
        ok, msg, apo, _ = run_slots(ctx, d_i, d_q)
        good = bad = by_ap = 0
        for s in range(per_point):
            got = {bytes(msg[s, k]["text"]).decode() for k in np.flatnonzero(ok[s])}
            other = {bytes(msg[s, k]["text"]).decode() for k in np.flatnonzero(ok[s] & (apo[s] != 2))}
            good += texts[s] in got
            by_ap += texts[s] in got and texts[s] not in other
            bad += len(got - {texts[s]})
        row[name] = {"decoded": good, "rate": good / per_point, "never_transmitted": bad, "decoded_only_by_ap": by_ap}
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


def never_transmitted_added_by_ap(gain):
    """never-transmitted messages with AP on minus those of the same configuration with AP off, over the sweep"""
    return sum(r["bp_ap"]["never_transmitted"] - r["bp"]["never_transmitted"] + r["osd2_ap"]["never_transmitted"] - r["osd2"]["never_transmitted"]
               for rows in gain.values() for r in rows)


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
        for label, osd, ap in CONFIGS:
            ctx = pkg.Context(0, max_candidates=K, max_messages=M)
            ctx.set_osd(osd, -1)
            ctx.set_ap(ap, cap)
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
    for ap in (0, 1, 0, 1):  # alternated, twice each
        p = pkg.Pipe(0, depth=3)
        out["provisioned"] = p.set_partition(back_sms)
        p.set_ap(ap, cap)
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
        out.setdefault(f"ap{ap}_ms_per_batch", []).append((time.perf_counter() - t0) * 1e3 / batches)
        p.close()
    print("pipe", out, flush=True)
    return out


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "perf_ap.json")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    noise, cap = noise_sweep()
    print("noise", {k: {c: n for c, n in v["ap_decodes_by_cap"].items() if n} for k, v in noise.items()}, "default cap", cap, flush=True)
    out = {"gpu": gpu, "default_max_hard": cap, "false_decodes_4096_noise_slots_k120": noise}
    out["decode_stage_time"] = stage4_times(cap)
    out["pipe_partitioned"] = pipe_times(cap)
    out["gain"] = gain_sweep(cap)
    out["never_transmitted_added_by_ap"] = never_transmitted_added_by_ap(out["gain"])
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
