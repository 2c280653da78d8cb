#!/usr/bin/env python3
"""The decoders after BP (OSD, AP, fine sync) and the later passes: this tree's library against a parent build, alternated in one
run -> profiles/perf_decode_chain_ab.json.

Workloads: {off, OSD order 2, AP, fine sync, OSD 2 + AP + fine sync} x passes {1, 3}, each on bench.py's 128-slot raw batch (K = 120)
and on 32 crowded slots (60 GFSK signals each, K = 500 / M = 200).  Each library runs in a subprocess of its own (the parent's through
FT8B200_LIB_PATH), twice, in the order new, parent, new, parent.  A subprocess reports per workload:
  * a SHA-256 over the spot records and pass 1's rows (ok, status, msg, the OSD / AP / fine-sync flags and hard distances) of every
    slot's candidates: it must be the same for both libraries;
  * stage_times()["decode"] (BP and the decoders after it) and ["later_passes"] over 10 timed batches after 3 warm-up ones, medians:
    the new library's must lie within the spread between the two runs of the same library.
Then bench.py (every option off) alternated the same way.  The GPU's name and power limit are read in the same run.
usage: python tools/perf_decode_chain_ab.py --parent-lib PATH [out.json]"""
import hashlib
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

OPTIONS = (("off", 0, 0, 0), ("osd2", 2, 0, 0), ("ap", 0, 1, 0), ("fs", 0, 0, 1), ("osd2_ap_fs", 2, 1, 1))
PASSES = (1, 3)


def worker(crowded_npz, out_path, warmup=3, reps=10):
    import torch

    import bench
    from ft8b200_loader import load
    from tools.perf_osd import _Arr

    pkg = load()
    dev = torch.device("cuda:0")
    raw, _ = bench.gen_batch(128, 0, dev)
    d = np.load(crowded_npz)
    ci, cq = torch.from_numpy(d["i"]).to(dev), torch.from_numpy(d["q"]).to(dev)
    cp = torch.maximum(ci.abs().amax(1), cq.abs().amax(1)).contiguous()
    shapes = (("raw128_k120", 128, 120, 50, lambda c: c.process_raw(raw, 128)),
              ("crowded32_k500", 32, 500, 200, lambda c: c.process_conditioned(ci, cq, cp)))
    host = lambda ptr, shape, t: torch.as_tensor(_Arr(ptr, shape, t), device=dev).cpu().numpy()
    out = {}
    for shape, n, K, M, run in shapes:
        for label, osd, ap, fs in OPTIONS:
            for passes in PASSES:
                ctx = pkg.Context(0, max_candidates=K, max_messages=M)
                ctx.set_osd(osd, -1)
                ctx.set_ap(ap, -1)
                ctx.set_finesync(fs, -1)
                ctx.set_passes(passes)
                ctx.set_profiling(True)
                for _ in range(warmup):
                    run(ctx)
                torch.cuda.synchronize()
                dec, later = [], []
                for _ in range(reps):
                    run(ctx)
                    t = ctx.stage_times()
                    dec.append(t["decode"])
                    later.append(t.get("later_passes", 0.0))
                res, nres = ctx.fetch_results(n)
                w = ctx.workspace_ptrs()
                ncand = host(w["ncand"], (n,), "<i4")
                rows = [host(w["ok"], (n, K), "|u1"), host(w["status"], (n, K, 12), "|u1"), host(w["msg"], (n, K, 28), "|u1")]
                for a, b in (ctx.osd_workspace_ptrs(), ctx.ap_workspace_ptrs(), ctx.finesync_workspace_ptrs()):
                    if a:
                        rows += [host(a, (n, K), "|u1"), host(b, (n, K), "<i4")]
                h = hashlib.sha256(np.ascontiguousarray(nres).tobytes() + np.ascontiguousarray(res).tobytes())
                for s in range(n):
                    for r in rows:
                        h.update(np.ascontiguousarray(r[s, :ncand[s]]).tobytes())
                key = f"{shape}/{label}/passes{passes}"
                out[key] = {"sha256": h.hexdigest(), "spots": int(nres.sum()), "candidates": int(ncand.sum()),
                            "decode_ms_median": float(np.median(dec)), "later_passes_ms_median": float(np.median(later))}
                print(key, out[key], flush=True)
                ctx.close()
    with open(out_path, "w") as f:
        json.dump(out, f)


def run_worker(lib, crowded_npz, tmp, tag):
    env = dict(os.environ)
    if lib:
        env["FT8B200_LIB_PATH"] = lib
    path = os.path.join(tmp, tag + ".json")
    p = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", crowded_npz, path], env=env, cwd=ROOT, capture_output=True, text=True)
    if p.returncode != 0:
        raise RuntimeError(f"{tag}: {p.stderr[-3000:]}")
    with open(path) as f:
        return json.load(f)


def bench_ab(parent_lib, steps=20, warmup=5):
    args = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup), "--cpu-slots", "8", "--no-configs"]
    out = {"what": " ".join(["bench.py"] + args[2:]) + ", every option off, alternated", "slots_per_s": {}}
    for rep in (1, 2):
        for who, lib in (("new", None), ("parent", parent_lib)):
            env = dict(os.environ)
            if lib:
                env["FT8B200_LIB_PATH"] = lib
            p = subprocess.run(args, env=env, capture_output=True, text=True, cwd=ROOT)
            line = [ln for ln in p.stdout.splitlines() if ln.startswith("{")][-1]
            out["slots_per_s"][f"{who}_{rep}"] = json.loads(line)["value"]
            print("bench", who, rep, out["slots_per_s"][f"{who}_{rep}"], flush=True)
    return out


def main():
    argv = sys.argv[1:]
    if argv and argv[0] == "--worker":
        return worker(argv[1], argv[2])
    i = argv.index("--parent-lib")
    parent = os.path.abspath(argv[i + 1])
    del argv[i:i + 2]
    path = argv[0] if argv else os.path.join(ROOT, "profiles", "perf_decode_chain_ab.json")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    from tools import ft8enc, synth
    slots = [synth.crowded_band(ft8enc, 60, 500 + s)[:2] for s in range(32)]
    out = {"gpu": gpu, "order": ["new_1", "parent_1", "new_2", "parent_2"], "runs": {}}
    with tempfile.TemporaryDirectory() as tmp:
        crowded_npz = os.path.join(tmp, "crowded.npz")
        np.savez(crowded_npz, i=np.stack([a for a, _ in slots]), q=np.stack([b for _, b in slots]))
        for tag in out["order"]:
            out["runs"][tag] = run_worker(parent if tag.startswith("parent") else None, crowded_npz, tmp, tag)
    runs = out["runs"]
    keys = [k for k in runs["new_1"] if "/" in k]
    summary, same = {}, True
    for k in keys:
        digests = {runs[t][k]["sha256"] for t in out["order"]}
        row = {"identical": len(digests) == 1}
        same = same and row["identical"]
        for m in ("decode_ms_median", "later_passes_ms_median"):
            new = [runs[t][k][m] for t in ("new_1", "new_2")]
            par = [runs[t][k][m] for t in ("parent_1", "parent_2")]
            row[m] = {"new": new, "parent": par, "new_over_parent": float(np.mean(new) / np.mean(par)) if np.mean(par) > 0 else None}
        summary[k] = row
    out["summary"] = summary
    out["all_outputs_identical"] = same
    out["bench_ab"] = bench_ab(parent)
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print("all outputs identical:", same)
    print("wrote", path)


if __name__ == "__main__":
    main()
