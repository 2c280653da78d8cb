"""Ordered-statistics decoding (OSD) on the B200 against the CPU restatement (orc_osd and the _osd forms of orc_decode / orc_subsystem,
tests/support/osd_oracle.c), byte for byte.  Every test creates its own contexts and pipes: the session contexts of the other suites
never have OSD switched on."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from oracle.pyoracle import cand_dtype, msg_dtype, result_dtype, status_dtype
from test_osd import FT4_XOR, fuzz_llrs, oracle  # noqa: F401 (oracle: the fixture with the OSD forms)
from tools import ft8enc, synth

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
DEV = torch.device("cuda:0")


def view(t, dt):
    a = t.cpu().numpy()
    return a.view(dt).reshape(a.shape[:-1])


@pytest.fixture(scope="module")
def default_cap(pkg):
    import re
    hdr = open(os.path.join(ROOT, "include", "ft8b200.h")).read()
    return int(re.search(r"#define FT8B200_OSD_DEFAULT_MAX_HARD (\d+)", hdr).group(1))


def expected_finish(oracle, cw, protocol):
    """status and message bytes finish() writes for an accepted codeword."""
    a = np.packbits(np.concatenate([cw[:91], np.zeros(5, np.uint8)])).tobytes()
    crc = int("".join(map(str, cw[77:91])), 2)
    p = bytes(x ^ y for x, y in zip(a[:10], FT4_XOR)) if protocol == 0 else a[:10]
    rc, text = oracle.unpack77(p[:9] + bytes([p[9] & 0xF8]))
    st = np.zeros(1, status_dtype)
    st[0] = (0, crc, crc, rc)
    m = np.zeros(1, msg_dtype)
    m[0]["text"] = text.encode()[:24]
    m[0]["hash"] = crc
    return st.tobytes(), m.tobytes()


@pytest.mark.parametrize("protocol", [1, 0], ids=["ft8", "ft4"])
def test_stage_entry_matches_oracle(pkg, oracle, protocol, default_cap):
    """20 000 fuzzed LLR vectors (Gaussian, noisy codewords, ties, +-0, early dependent columns, 1 % non-finite) at stage 1, plus
    entries at stage 2-4 and past ncand, through ft8b200_osd at orders 1 and 2 and three caps."""
    K, S = 125, 160
    llrs = fuzz_llrs(oracle, S * K, 1234 + protocol).reshape(S, K, 174)
    rng = np.random.default_rng(5)
    bad = rng.random((S, K)) < 0.01
    llrs[bad, rng.integers(0, 174, int(bad.sum()))] = rng.choice([np.nan, np.inf, -np.inf], int(bad.sum()))
    stage0 = np.where(rng.random((S, K)) < 0.85, 1, rng.integers(2, 5, (S, K))).astype(np.uint8)
    ncand = rng.integers(K - 10, K + 1, S).astype(np.int32)
    want = {}
    for order in (1, 2):
        want[order] = [[oracle.osd(llrs[s, k], order, 174, protocol) for k in range(K)] for s in range(S)]
    ctx = pkg.Context(0, max_candidates=K)
    ctx.set_protocol(protocol)
    d_llr = torch.from_numpy(llrs).to(DEV)
    d_ncand = torch.from_numpy(ncand).to(DEV)
    sentinel_st = rng.integers(0, 256, (S, K, 12), dtype=np.uint8)
    sentinel_msg = rng.integers(0, 256, (S, K, 28), dtype=np.uint8)
    sentinel_plain = rng.integers(0, 2, (S, K, 174), dtype=np.uint8)
    try:
        for order in (1, 2):
            for cap in (10, 26, default_cap):
                ctx.set_osd(order, cap)
                ok = torch.zeros((S, K), dtype=torch.uint8, device=DEV)
                stage = torch.from_numpy(stage0).to(DEV)
                status = torch.from_numpy(sentinel_st).to(DEV)
                msg = torch.from_numpy(sentinel_msg).to(DEV)
                plain = torch.from_numpy(sentinel_plain).to(DEV)
                osd, hard, cw = ctx.osd(d_llr, d_ncand, ok, stage, status, msg, plain, want_cw=True)
                torch.cuda.synchronize()
                osd, hard, cw = osd.cpu().numpy(), hard.cpu().numpy(), cw.cpu().numpy()
                ok, stage, status, msg, plain = ok.cpu().numpy(), stage.cpu().numpy(), status.cpu().numpy(), msg.cpu().numpy(), plain.cpu().numpy()
                accepted = 0
                for s in range(S):
                    for k in range(K):
                        w = want[order][s][k]
                        attempted = k < ncand[s] and stage0[s, k] in (1, 2) and w[0] >= 0
                        if not attempted:
                            assert osd[s, k] == 0 and hard[s, k] == -1 and not cw[s, k].any(), (order, cap, s, k)
                            acc = False
                        else:
                            acc = w[0] == 1 and w[2] <= cap
                            assert osd[s, k] == (2 if acc else 1) and hard[s, k] == w[2] and np.array_equal(cw[s, k], w[1]), (order, cap, s, k)
                        if acc:
                            accepted += 1
                            est, emsg = expected_finish(oracle, w[1], protocol)
                            assert ok[s, k] == 1 and stage[s, k] == 4 and status[s, k].tobytes() == est and msg[s, k].tobytes() == emsg, (s, k)
                            assert np.array_equal(plain[s, k], w[1])
                        else:
                            assert ok[s, k] == 0 and stage[s, k] == stage0[s, k] and np.array_equal(status[s, k], sentinel_st[s, k])
                            assert np.array_equal(msg[s, k], sentinel_msg[s, k]) and np.array_equal(plain[s, k], sentinel_plain[s, k])
                assert accepted > 100
    finally:
        ctx.close()


@pytest.fixture(scope="module")
def weak_slots(oracle):
    """64 seeded slots of 1-30 overlapping 8-FSK signals at -26 ... -14 dB, conditioned."""
    out = []
    for s in range(64):
        n = 1 + (s * 7) % 30
        i_s, q_s, _ = synth.crowded_band(ft8enc, n, 700 + s, snr_lo=-26.0, snr_hi=-14.0)
        out.append(tuple(oracle.condition(i_s, q_s, 48000)[:2]))
    return np.stack([a for a, _ in out]), np.stack([b for _, b in out])


def ctx_outputs(ctx, n):
    w = ctx.workspace_ptrs()

    class _Arr:
        def __init__(self, ptr, shape, typestr):
            self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2}
    K = ctx.K
    g = lambda p, shp, t: torch.as_tensor(_Arr(p, shp, t), device=DEV).cpu().numpy()
    a, b = ctx.osd_workspace_ptrs()
    return dict(ok=g(w["ok"], (n, K), "|u1"), ncand=g(w["ncand"], (n,), "<i4"), cand=g(w["cand"], (n, K * 8), "|u1").view(cand_dtype),
                status=g(w["status"], (n, K * 12), "|u1").view(status_dtype), msg=g(w["msg"], (n, K * 28), "|u1").view(msg_dtype),
                osd=g(a, (n, K), "|u1") if a else None, hard=g(b, (n, K), "<i4") if b else None, mag=g(w["mag"], (n, 94208), "|u1"))


@pytest.mark.parametrize("order", [1, 2])
def test_whole_path_matches_oracle(pkg, oracle, weak_slots, order, default_cap):
    hi, hq = weak_slots
    n = 64 if order == 2 else 24
    ctx = pkg.Context(0)
    try:
        ctx.set_osd(order, -1)
        res, nres = ctx.process_slots_host(hi[:n], hq[:n])
        o = ctx_outputs(ctx, n)
        by_osd = 0
        for s in range(n):
            ref = oracle.subsystem_osd(hi[s], hq[s], order, default_cap)
            assert int(nres[s]) == ref["n"] and res[s].tobytes() == ref["results"].tobytes(), s
            for k in range(int(o["ncand"][s])):
                d = oracle.decode_osd(o["mag"][s], o["cand"][s, k], order, default_cap)
                assert o["ok"][s, k] == d["ok"] and o["osd"][s, k] == d["osd"] and o["hard"][s, k] == d["osd_hard"], (s, k)
                if d["ok"]:
                    assert o["status"][s, k].tobytes() == d["status"].tobytes() and o["msg"][s, k]["text"] == d["msg"]["text"]
                by_osd += d["osd"] == 2
        assert by_osd >= 1
    finally:
        ctx.close()


def test_k500_and_pipe_with_and_without_partition(pkg, oracle, weak_slots, default_cap):
    hi, hq = weak_slots
    c5 = pkg.Context(0, max_candidates=500, max_messages=200)
    c5.set_osd(2, -1)
    res, nres = c5.process_slots_host(hi[:8], hq[:8])
    for s in range(8):
        ref = oracle.subsystem_osd(hi[s], hq[s], 2, default_cap, max_cand=500, max_msgs=200)
        assert int(nres[s]) == ref["n"] and res[s].tobytes() == ref["results"].tobytes(), s
    c5.close()
    c = pkg.Context(0)
    c.set_osd(2, -1)
    want_res, want_n = c.process_slots_host(hi[:16], hq[:16])
    c.close()
    for back in (0, 40):
        p = pkg.Pipe(0, depth=2)
        if back:
            p.set_partition(back)
        p.set_osd(2, -1)
        p.submit_slots_host(hi[:16], hq[:16])
        assert p.in_flight() == 1
        with pytest.raises(pkg.Ft8Error):
            p.set_osd(1, -1)  # EBUSY while a batch is in flight
        got_res, got_n = p.collect(16)
        assert np.array_equal(got_n, want_n) and got_res.tobytes() == want_res.tobytes()
        p.close()


def test_off_means_untouched_and_bp_decodes_unchanged(pkg, weak_slots):
    hi, hq = weak_slots
    fresh = pkg.Context(0)
    r0, n0 = fresh.process_slots_host(hi, hq)
    o0 = ctx_outputs(fresh, 64)
    l0 = fresh.launches()
    toggled = pkg.Context(0)
    toggled.set_osd(2, -1)
    toggled.process_slots_host(hi, hq)
    o2 = ctx_outputs(toggled, 64)
    toggled.set_osd(0, -1)
    l1 = toggled.launches()
    r1, n1 = toggled.process_slots_host(hi, hq)
    o1 = ctx_outputs(toggled, 64)
    assert toggled.launches() - l1 == l0 and np.array_equal(n0, n1) and r0.tobytes() == r1.tobytes()
    assert np.array_equal(o0["ncand"], o1["ncand"])
    for key in ("ok", "cand", "status", "msg"):
        for s in range(64):
            nc = int(o0["ncand"][s])
            assert o0[key][s][:nc].tobytes() == o1[key][s][:nc].tobytes(), (key, s)
    # with OSD on, every BP decode is unchanged and every message decoded without OSD is still decoded
    for s in range(64):
        nc = int(o0["ncand"][s])
        bp = np.flatnonzero(o0["ok"][s, :nc])
        assert np.all(o2["ok"][s, bp] == 1) and np.all(o2["osd"][s, bp] == 0)
        assert o2["status"][s, bp].tobytes() == o0["status"][s, bp].tobytes() and o2["msg"][s, bp].tobytes() == o0["msg"][s, bp].tobytes()
    fresh.close()
    toggled.close()


def test_flat_waterfall_gives_no_attempt(pkg):
    ctx = pkg.Context(0)
    ctx.set_osd(2, -1)
    mag = torch.full((1, 94208), 77, dtype=torch.uint8, device=DEV)
    cand = np.zeros((1, ctx.K), cand_dtype)
    cand[0, :3] = [(20, 0, 10, 0, 0), (20, 5, 100, 1, 1), (20, -3, 200, 0, 1)]
    d_cand = torch.from_numpy(cand.view(np.uint8).reshape(1, ctx.K, 8)).to(DEV)
    ncand = torch.tensor([3], dtype=torch.int32, device=DEV)
    ok, stage, status, msg, plain, llr = ctx.decode(mag, d_cand, ncand, want_llr=True)
    assert torch.isnan(llr[0, :3]).any(dim=1).all()
    osd, hard, _ = ctx.osd(llr, ncand, ok, stage, status, msg)
    torch.cuda.synchronize()
    assert not osd.any() and (hard == -1).all() and not ok.any()
    ctx.close()


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


def test_dropin_reads_the_environment(pkg, weak_slots, tmp_path):
    hi, hq = weak_slots
    np.savez(tmp_path / "slots.npz", i=hi[:12], q=hq[:12])
    script = tmp_path / "dropin.py"
    script.write_text(_DROPIN)
    env = dict(os.environ, FT8B200_OSD="1")
    env.pop("FT8B200_OSD_MAX_HARD", None)
    p = subprocess.run([sys.executable, str(script), ROOT, str(tmp_path / "slots.npz"), str(tmp_path / "out.npy")], env=env, capture_output=True,
                       text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    got = np.load(tmp_path / "out.npy", allow_pickle=True)
    got_n = np.load(tmp_path / "out.npy.n.npy")
    ctx = pkg.Context(0)
    ctx.set_osd(1, -1)
    for s in range(12):
        res, nres = ctx.process_slots_host(hi[s:s + 1], hq[s:s + 1])
        want = np.zeros(50, result_dtype)
        for k in range(int(nres[0])):
            if res[0][k]["call"]:
                want[k] = res[0][k]
        assert got_n[s] == nres[0] and got[s] == want.tobytes(), s
    ctx.close()


def _decode_rate(pkg, order, snr, n=512, seed=0x5EED):
    from tools.perf_osd import amp_for, run_slots
    rng = np.random.Generator(np.random.PCG64(seed + 100 * (-snr)))
    texts, items = [], []
    for _ in range(n):
        to, de, ex = synth.random_message(rng)
        texts.append(f"{to} {de} {ex}")
        items.append((pkg.pack77_std(to, de, ex), float(rng.uniform(300.0, 1300.0)), float(0.5 + rng.uniform(-0.3, 0.3)), amp_for(snr)))
    ctx = pkg.Context(0)
    ctx.set_osd(order, -1)
    d_i, d_q = ctx.synth_slots(pkg.make_signals(items, gfsk=True), np.arange(n + 1, dtype=np.int32), 1.0, seed + snr)
    ok, msg, _, _ = run_slots(ctx, d_i, d_q)
    ctx.close()
    return sum(texts[s] in {bytes(msg[s, k]["text"]).decode() for k in np.flatnonzero(ok[s])} for s in range(n)) / n


def test_osd_decodes_deeper_and_stays_clean_on_noise(pkg):
    from tools.perf_osd import run_slots
    snr = next(s for s in range(-18, -27, -1) if 0.10 <= _decode_rate(pkg, 0, s) <= 0.60)
    for order in (1, 2):
        assert _decode_rate(pkg, order, snr) > _decode_rate(pkg, 0, snr), (order, snr)
    ctx = pkg.Context(0)
    ctx.set_osd(2, -1)
    found = set()
    for b0 in range(0, 4096, 1024):
        d_i, d_q = ctx.synth_slots(pkg.make_signals([]), np.zeros(1025, np.int32), 1.0, 0x0D5E, first_slot_index=b0)
        ok, msg, osd, _ = run_slots(ctx, d_i, d_q)
        found |= {(b0 + s, bytes(msg[s, k]["text"])) for s, k in zip(*np.nonzero(osd == 2))}
    ctx.close()
    assert len(found) <= 2, found
