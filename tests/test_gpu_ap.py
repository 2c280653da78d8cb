"""A-priori (AP) decoding of "CQ ??? ???" on the B200 against the CPU restatement (orc_ap and the _ap forms of orc_decode /
orc_subsystem, tests/support/ap_oracle.c), byte for byte, and against a composition of the stage-wise entry points with multi-pass
decoding.  Every test creates its own contexts and pipes: the session contexts of the other suites never have AP switched on."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import test_gpu_multipass as mp
from conftest import ROOT
from oracle.pyoracle import cand_dtype, msg_dtype, result_dtype, status_dtype
from test_ap import KNOWN, fuzz_ap_llrs, oracle  # noqa: F401 (oracle: the fixture with the OSD and AP forms)
from test_gpu_osd import expected_finish
from tools import ft8enc, synth

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
DEV = torch.device("cuda:0")


@pytest.fixture(scope="module")
def default_cap(pkg):
    hdr = open(os.path.join(ROOT, "include", "ft8b200.h")).read()
    return int(re.search(r"#define FT8B200_AP_DEFAULT_MAX_HARD (\d+)", hdr).group(1))


@pytest.fixture(scope="module")
def osd_cap(pkg):
    hdr = open(os.path.join(ROOT, "include", "ft8b200.h")).read()
    return int(re.search(r"#define FT8B200_OSD_DEFAULT_MAX_HARD (\d+)", hdr).group(1))


@pytest.mark.parametrize("protocol", [1, 0], ids=["ft8", "ft4"])
def test_stage_entry_matches_oracle(pkg, oracle, protocol, default_cap):
    """7 680 fuzzed LLR vectors (noise, noisy CQ codewords, reversed known positions, non-CQ codewords, ties, +-0, 1 % non-finite)
    at stages 1-4 and past ncand, through ft8b200_ap at three caps and with AP off."""
    K, S = 120, 64
    llrs = fuzz_ap_llrs(oracle, S * K, 4321 + protocol, protocol).reshape(S, K, 174)
    rng = np.random.default_rng(6)
    bad = rng.random((S, K)) < 0.01
    llrs[bad, rng.integers(0, 174, int(bad.sum()))] = rng.choice([np.nan, np.inf, -np.inf], int(bad.sum()))
    stage0 = np.where(rng.random((S, K)) < 0.8, rng.integers(1, 3, (S, K)), rng.integers(3, 5, (S, K))).astype(np.uint8)
    ncand = rng.integers(K - 10, K + 1, S).astype(np.int32)
    want = [[oracle.ap(llrs[s, k], 174, protocol) for k in range(K)] for s in range(S)]  # the cap is the only gate that depends on it
    ctx = pkg.Context(0, max_candidates=K)
    ctx.set_protocol(protocol)
    d_llr = torch.from_numpy(llrs).to(DEV)
    d_ncand = torch.from_numpy(ncand).to(DEV)
    sentinel_st = rng.integers(0, 256, (S, K, 12), dtype=np.uint8)
    sentinel_msg = rng.integers(0, 256, (S, K, 28), dtype=np.uint8)
    sentinel_plain = rng.integers(0, 2, (S, K, 174), dtype=np.uint8)
    try:
        for on, cap in ((1, 20), (1, 60), (1, default_cap), (0, 174)):
            ctx.set_ap(on, cap)
            ok = torch.zeros((S, K), dtype=torch.uint8, device=DEV)
            stage = torch.from_numpy(stage0).to(DEV)
            status = torch.from_numpy(sentinel_st).to(DEV)
            msg = torch.from_numpy(sentinel_msg).to(DEV)
            plain = torch.from_numpy(sentinel_plain).to(DEV)
            ap, hard = ctx.ap(d_llr, d_ncand, ok, stage, status, msg, plain)
            torch.cuda.synchronize()
            ap, hard = ap.cpu().numpy(), hard.cpu().numpy()
            ok, stage, status, msg, plain = ok.cpu().numpy(), stage.cpu().numpy(), status.cpu().numpy(), msg.cpu().numpy(), plain.cpu().numpy()
            accepted = rejected = 0
            for s in range(S):
                for k in range(K):
                    w = want[s][k]
                    attempted = on and k < ncand[s] and stage0[s, k] in (1, 2) and w[0] >= 0
                    if not attempted:
                        assert ap[s, k] == 0 and hard[s, k] == -1, (on, cap, s, k)
                        acc = False
                    else:
                        acc = w[0] == 1 and w[2] <= cap
                        assert ap[s, k] == (2 if acc else 1) and hard[s, k] == w[2], (cap, s, k, ap[s, k], hard[s, k], w[0], w[2])
                        rejected += not acc
                    if acc:
                        accepted += 1
                        est, emsg = expected_finish(oracle, w[1], protocol)
                        assert ok[s, k] == 1 and stage[s, k] == 4 and status[s, k].tobytes() == est and msg[s, k].tobytes() == emsg, (s, k)
                        assert np.array_equal(plain[s, k], w[1])
                    else:
                        assert ok[s, k] == 0 and stage[s, k] == stage0[s, k] and np.array_equal(status[s, k], sentinel_st[s, k])
                        assert np.array_equal(msg[s, k], sentinel_msg[s, k]) and np.array_equal(plain[s, k], sentinel_plain[s, k])
            if on:
                assert accepted > 100 and rejected > 100, (cap, accepted, rejected)
    finally:
        ctx.close()


@pytest.fixture(scope="module")
def weak_cq_slots(oracle):
    """48 seeded slots of 1-8 CQ signals at -21 ... -17 dB (plain 8-FSK), conditioned."""
    out = []
    for s in range(48):
        rng = np.random.default_rng(900 + s)
        sig = [(ft8enc.tones(ft8enc.pack_std("CQ", synth.random_call(rng), synth.random_grid(rng))), float(rng.uniform(100, 1500)),
                float(0.5 + rng.uniform(-0.3, 0.3)), float(rng.uniform(-21.0, -17.0))) for _ in range(1 + s % 8)]
        i_s, q_s = synth.slot_f32(sig, 900 + s)
        out.append(tuple(oracle.condition(i_s, q_s, 48000)[:2]))
    return np.stack([a for a, _ in out]), np.stack([b for _, b in out])


class _Arr:
    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2}


def ctx_outputs(ctx, n):
    w = ctx.workspace_ptrs()
    K = ctx.K
    g = lambda p, shp, t: torch.as_tensor(_Arr(p, shp, t), device=DEV).cpu().numpy()
    a, b = ctx.ap_workspace_ptrs()
    return dict(ok=g(w["ok"], (n, K), "|u1"), ncand=g(w["ncand"], (n,), "<i4"), cand=g(w["cand"], (n, K * 8), "|u1").view(cand_dtype),
                status=g(w["status"], (n, K * 12), "|u1").view(status_dtype), msg=g(w["msg"], (n, K * 28), "|u1").view(msg_dtype),
                ap=g(a, (n, K), "|u1") if a else None, hard=g(b, (n, K), "<i4") if b else None, mag=g(w["mag"], (n, 94208), "|u1"))


@pytest.mark.parametrize("osd", [0, 2])
def test_whole_path_matches_oracle(pkg, oracle, weak_cq_slots, osd, default_cap, osd_cap):
    hi, hq = weak_cq_slots
    n = hi.shape[0]
    ctx = pkg.Context(0)
    try:
        ctx.set_osd(osd, -1)
        ctx.set_ap(1, -1)
        res, nres = ctx.process_slots_host(hi, hq)
        o = ctx_outputs(ctx, n)
        by_ap = 0
        for s in range(n):
            ref = oracle.subsystem_ap(hi[s], hq[s], osd, osd_cap, 1, default_cap)
            assert int(nres[s]) == ref["n"] and res[s].tobytes() == ref["results"].tobytes(), s
            for k in range(int(o["ncand"][s])):
                d = oracle.decode_ap(o["mag"][s], o["cand"][s, k], osd, osd_cap, 1, default_cap)
                assert o["ok"][s, k] == d["ok"] and o["ap"][s, k] == d["ap"] and o["hard"][s, k] == d["ap_hard"], (s, k)
                if d["ok"]:
                    assert o["status"][s, k].tobytes() == d["status"].tobytes() and o["msg"][s, k]["text"] == d["msg"]["text"]
                by_ap += d["ap"] == 2
        assert by_ap >= 1
    finally:
        ctx.close()


def test_k500_and_pipe_with_and_without_partition(pkg, oracle, weak_cq_slots, default_cap, osd_cap):
    hi, hq = weak_cq_slots
    c5 = pkg.Context(0, max_candidates=500, max_messages=200)
    c5.set_ap(1, -1)
    res, nres = c5.process_slots_host(hi[:8], hq[:8])
    for s in range(8):
        ref = oracle.subsystem_ap(hi[s], hq[s], 0, osd_cap, 1, default_cap, max_cand=500, max_msgs=200)
        assert int(nres[s]) == ref["n"] and res[s].tobytes() == ref["results"].tobytes(), s
    c5.close()
    c = pkg.Context(0)
    c.set_osd(2, -1)
    c.set_ap(1, -1)
    want_res, want_n = c.process_slots_host(hi[:16], hq[:16])
    c.close()
    for back in (0, 40):
        p = pkg.Pipe(0, depth=2)
        if back:
            p.set_partition(back)
        p.set_osd(2, -1)
        p.set_ap(1, -1)
        p.submit_slots_host(hi[:16], hq[:16])
        assert p.in_flight() == 1
        with pytest.raises(pkg.Ft8Error):
            p.set_ap(0, -1)  # EBUSY while a batch is in flight
        got_res, got_n = p.collect(16)
        assert np.array_equal(got_n, want_n) and got_res.tobytes() == want_res.tobytes()
        p.close()


def test_off_means_untouched(pkg, weak_cq_slots):
    """AP off: outputs, launch counts and device memory as a context that never called set_ap; on, every BP decode is unchanged."""
    hi, hq = weak_cq_slots
    fresh = pkg.Context(0)
    r0, n0 = fresh.process_slots_host(hi, hq)
    o0 = ctx_outputs(fresh, 48)
    l0 = fresh.launches()
    assert fresh.ap_workspace_ptrs() == (0, 0)
    used = []
    for c in (pkg.Context(0), pkg.Context(0)):  # device memory a batch allocates: a context that never called set_ap, then one set off
        if used:
            c.set_ap(0, 30)
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        r2, n2 = c.process_slots_host(hi, hq)
        torch.cuda.synchronize()
        used.append(free0 - torch.cuda.mem_get_info()[0])
        off = c
    assert abs(used[1] - used[0]) <= (2 << 20), used
    assert off.launches() == l0 and off.ap_workspace_ptrs() == (0, 0)
    assert np.array_equal(n0, n2) and r0.tobytes() == r2.tobytes()
    toggled = pkg.Context(0)
    toggled.set_ap(1, -1)
    toggled.process_slots_host(hi, hq)
    o2 = ctx_outputs(toggled, 48)
    toggled.set_ap(0, -1)
    l1 = toggled.launches()
    r1, n1 = toggled.process_slots_host(hi, hq)
    o1 = ctx_outputs(toggled, 48)
    assert toggled.launches() - l1 == l0 and np.array_equal(n0, n1) and r0.tobytes() == r1.tobytes()
    for key in ("ok", "cand", "status", "msg"):
        for s in range(48):
            nc = int(o0["ncand"][s])
            assert o0[key][s][:nc].tobytes() == o1[key][s][:nc].tobytes(), (key, s)
    for s in range(48):
        nc = int(o0["ncand"][s])
        bp = np.flatnonzero(o0["ok"][s, :nc])
        assert np.all(o2["ok"][s, bp] == 1) and np.all(o2["ap"][s, bp] == 0)
        assert o2["status"][s, bp].tobytes() == o0["status"][s, bp].tobytes() and o2["msg"][s, bp].tobytes() == o0["msg"][s, bp].tobytes()
    for c in (fresh, off, toggled):
        c.close()


def test_argument_checks(pkg):
    ctx = pkg.Context(0)
    for on in (-1, 2, 7):
        with pytest.raises(pkg.Ft8Error):
            ctx.set_ap(on, -1)
    ctx.set_ap(1, -1)
    ctx.set_ap(0, 0)
    llr = torch.zeros((1, ctx.K, 174), dtype=torch.float32, device=DEV)
    ncand = torch.zeros(1, dtype=torch.int32, device=DEV)
    u8 = torch.zeros((1, ctx.K), dtype=torch.uint8, device=DEV)
    status = torch.zeros((1, ctx.K, 12), dtype=torch.uint8, device=DEV)
    msg = torch.zeros((1, ctx.K, 28), dtype=torch.uint8, device=DEV)
    hard = torch.zeros((1, ctx.K), dtype=torch.int32, device=DEV)
    full = [llr, ncand, u8, u8, status, msg, None, u8.clone(), hard]  # ft8b200_ap's buffers after n_slots; plain is optional
    for drop in (0, 1, 2, 3, 4, 5, 7, 8):
        args = [None if q == drop else t for q, t in enumerate(full)]
        with pytest.raises(pkg.Ft8Error):
            ctx._chk(ctx.L.ft8b200_ap(pkg.C.c_void_p(ctx.h), pkg._p(args[0]), 1, *[pkg._p(t) for t in args[1:]], None))
    with pytest.raises(pkg.Ft8Error):  # n_slots < 1
        ctx._chk(ctx.L.ft8b200_ap(pkg.C.c_void_p(ctx.h), pkg._p(llr), 0, *[pkg._p(t) for t in full[1:]], None))
    ctx.close()
    p = pkg.Pipe(0, depth=2)
    with pytest.raises(pkg.Ft8Error):
        p.set_ap(2, -1)
    p.set_ap(1, -1)
    p.close()


_DROPIN = r'''
import sys, numpy as np
sys.path.insert(0, sys.argv[1])
from ft8b200_loader import load
pkg = load()
d = np.load(sys.argv[2])
out = []
for s in range(d["i"].shape[0]):
    dec = np.zeros(50, pkg.result_dtype)
    _, n = pkg.ft8_subsystem(d["i"][s], d["q"][s], dec)
    out.append((n, dec.tobytes()))
np.save(sys.argv[3], np.array([o[1] for o in out], dtype=object), allow_pickle=True)
np.save(sys.argv[3] + ".n.npy", np.array([o[0] for o in out]))
'''


def test_dropin_reads_the_environment(pkg, weak_cq_slots, tmp_path):
    hi, hq = weak_cq_slots
    np.savez(tmp_path / "slots.npz", i=hi[:12], q=hq[:12])
    script = tmp_path / "dropin.py"
    script.write_text(_DROPIN)
    run = lambda env: subprocess.run([sys.executable, str(script), ROOT, str(tmp_path / "slots.npz"), str(tmp_path / "out.npy")], env=env,
                                     capture_output=True, text=True, timeout=600)
    base = {k: v for k, v in os.environ.items() if not k.startswith("FT8B200_")}
    for bad in ("2", "x", ""):
        p = run(dict(base, FT8B200_AP=bad))
        assert p.returncode != 0 and "FT8B200_AP" in p.stderr, bad
    p = run(dict(base, FT8B200_AP="1"))
    assert p.returncode == 0, p.stderr[-2000:]
    got = np.load(tmp_path / "out.npy", allow_pickle=True)
    got_n = np.load(tmp_path / "out.npy.n.npy")
    ctx = pkg.Context(0)
    ctx.set_ap(1, -1)
    for s in range(12):
        res, nres = ctx.process_slots_host(hi[s:s + 1], hq[s:s + 1])
        want = np.zeros(50, result_dtype)
        for k in range(int(nres[0])):
            if res[0][k]["call"]:
                want[k] = res[0][k]
        assert got_n[s] == nres[0] and got[s] == want.tobytes(), s
    ctx.close()


def stage_with_ap(c, x_i, x_q, peak, osd):
    """test_gpu_multipass.stage on a context with AP on: waterfall -> find_sync -> ft8b200_decode, which runs OSD (when on) and then
    AP, AP decodes writing their word into plain; AP's outputs from the context's workspace."""
    mag = c.waterfall(x_i, x_q, peak)
    cand, ncand = c.find_sync(mag)
    ok, stg, status, msg, plain, llr = c.decode(mag, cand, ncand, want_plain=True, want_llr=True)
    torch.cuda.synchronize()
    n = x_i.shape[0]
    ap = torch.as_tensor(_Arr(c.ap_workspace_ptrs()[0], (n, c.K), "|u1"), device=DEV).clone()
    R = dict(cand=cand.cpu().numpy().view(cand_dtype).reshape(n, c.K), ncand=ncand.cpu().numpy(), ok=ok.cpu().numpy(), status=status.cpu().numpy(),
             msg=msg.cpu().numpy().view(msg_dtype).reshape(n, c.K), plain=plain.cpu().numpy())
    APS.append((ap.cpu().numpy(), R))
    return R


APS = []


@pytest.fixture(scope="module")
def cq_slots(pkg):
    """24 device slots of 6-20 CQ messages at -22 ... -16 dB (GFSK, noise 1.0) with their peaks."""
    rng = np.random.Generator(np.random.PCG64(0xA95))
    slots = [[(pkg.pack77_std("CQ", synth.random_call(rng), synth.random_grid(rng)), float(rng.uniform(100, 1500)), float(0.5 + rng.uniform(-0.3, 0.3)),
               mp.amp_for(float(rng.uniform(-22, -16)))) for _ in range(int(rng.integers(6, 21)))] for _ in range(24)]
    first = np.cumsum([0] + [len(s) for s in slots]).astype(np.int32)
    ctx = pkg.Context(0)
    d_i, d_q = ctx.synth_slots(pkg.make_signals([it for s in slots for it in s], gfsk=True), first, 1.0, 0xA95)
    peak = torch.maximum(d_i.abs().amax(1), d_q.abs().amax(1)).contiguous()
    torch.cuda.synchronize()
    ctx.close()
    return d_i, d_q, peak


@pytest.mark.parametrize("osd", [0, 2])
def test_multipass_composes_and_subtracts_ap_decodes(pkg, oracle, cq_slots, osd, monkeypatch):
    """passes = 1, 2 and 3 with AP equal the composition of the stage-wise entries with AP after OSD in every pass: pass-1 rows byte
    for byte (so pass 1 of passes = 2 is passes = 1), and the records, which after pass 1 depend on every AP-decoded message's plain
    row having been subtracted.  Each AP-decoded plain row is the codeword of its message."""
    d_i, d_q, peak = cq_slots
    n = d_i.shape[0]
    cfg = mp.cfg_of("default")
    monkeypatch.setattr(mp, "stage", stage_with_ap)
    ref = pkg.Context(0, **cfg)
    ref.set_osd(osd, -1)
    ref.set_ap(1, -1)
    st = mp.new_stats()
    APS.clear()
    one = None
    for passes in (1, 2, 3):
        ctx = pkg.Context(0, **cfg)
        ctx.set_osd(osd, -1)
        ctx.set_ap(1, -1)
        ctx.set_passes(passes)
        ctx.process_conditioned(d_i, d_q, peak)
        got = ctx.fetch_results(n)
        R1, wres, wnres = mp.compose(ref, oracle, d_i, d_q, peak, passes, osd, cfg, st)
        mp.check_pass1(ctx, n, R1)
        mp.check_records(got, (wres, wnres), (osd, passes))
        if passes == 1:
            one = got
        else:  # the later passes only append
            for s in range(n):
                k = int(one[1][s])
                assert got[0][s][:k].tobytes() == one[0][s][:k].tobytes(), (passes, s)
        ctx.close()
    ref.close()
    decoded = 0
    for ap, R in APS:
        for s, k in zip(*np.nonzero(ap == 2)):
            text = bytes(R["msg"][s, k]["text"]).decode().split()
            assert text[0] == "CQ" and len(text) in (2, 3)
            cw = ft8enc.encode174(ft8enc.pack_std("CQ", text[1], text[2] if len(text) == 3 else ""))
            assert np.array_equal(R["plain"][s, k], cw), text
            decoded += 1
    assert decoded >= 3 and st["appended_in_pass2"] >= 1


def _perf():
    with open(os.path.join(ROOT, "profiles", "perf_ap.json")) as f:
        return json.load(f)


def test_gain_and_no_false_records_as_measured(pkg):
    """The seeded rows of tools/perf_ap.py at the SNR where AP gained most, recomputed: the same counts, AP decodes strictly more
    transmitted CQ messages than BP alone, and nothing never transmitted on the CQ and the non-CQ set."""
    from tools import perf_ap
    perf = _perf()
    rows = perf["gain"]["cq"]
    best = max(rows, key=lambda r: r["bp_ap"]["decoded"] - r["bp"]["decoded"])
    cap = perf["default_max_hard"]
    for kind in ("cq", "non_cq"):
        want = next(r for r in perf["gain"][kind] if r["snr_db"] == best["snr_db"])
        got = perf_ap.gain_row(kind, best["snr_db"], cap, configs=(("bp", 0, 0), ("bp_ap", 0, 1)))
        for name in ("bp", "bp_ap"):
            assert got[name] == want[name], (kind, name, got[name], want[name])
            assert got[name]["never_transmitted"] == 0
        if kind == "cq":
            assert got["bp_ap"]["decoded"] > got["bp"]["decoded"]
        else:
            assert got["bp_ap"]["decoded_only_by_ap"] == 0


def test_nothing_on_noise_at_the_default_cap(pkg, default_cap):
    from tools import perf_ap
    assert _perf()["default_max_hard"] == default_cap
    ctx = pkg.Context(0)
    ctx.set_ap(1, -1)
    found = set()
    d_i, d_q = ctx.synth_slots(pkg.make_signals([]), np.zeros(1025, np.int32), 1.0, 0x0D5E, first_slot_index=0)
    ok, msg, ap, _ = perf_ap.run_slots(ctx, d_i, d_q)
    found |= {(s, bytes(msg[s, k]["text"])) for s, k in zip(*np.nonzero(ap == 2))}
    ctx.close()
    assert not found, found
