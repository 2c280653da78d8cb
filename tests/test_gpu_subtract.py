"""Multi-pass decoding with signal subtraction (ft8b200_set_passes, ft8b200_subtract) on the B200: the kernels against the float64
definition (tests/subtract_ref.py), pass 1 against passes = 1, the gain on crowded GFSK slots, and every entry point.  Every test
creates its own contexts and pipes: the session contexts of the other suites stay at passes = 1."""
import os
import subprocess
import sys

import numpy as np
import pytest

import subtract_ref as sr
from conftest import ROOT
from oracle.pyoracle import cand_dtype
from ref64 import bits_from_tones
from tools.perf_subtract import crowded_items, crowded_slots, run_conditioned, score

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
DEV = torch.device("cuda:0")


class _Arr:
    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2}


def pass1_rows(ctx, n):
    w = ctx.workspace_ptrs()
    K = ctx.K
    g = lambda p, shp, t: torch.as_tensor(_Arr(p, shp, t), device=DEV).cpu().numpy()
    ncand = g(w["ncand"], (n,), "<i4")
    rows = dict(cand=g(w["cand"], (n, K * 8), "|u1"), ok=g(w["ok"], (n, K), "|u1"), status=g(w["status"], (n, K * 12), "|u1"),
                msg=g(w["msg"], (n, K * 28), "|u1"))
    out = {"ncand": ncand}
    for key, a in rows.items():   # rows past a slot's candidate count are stale
        per = a.shape[1] // K
        out[key] = [a[s, :int(ncand[s]) * per].tobytes() for s in range(n)]
    return out


@pytest.fixture(scope="module")
def crowded(pkg):
    """64 seeded slots of 10-60 overlapping GFSK CQ messages at -20 ... -8 dB (device), and what each slot carries."""
    ctx = pkg.Context(0)
    parts = [crowded_slots(pkg, ctx, 16, n_sig, 0xC0 + n_sig) for n_sig in (10, 20, 40, 60)]
    ctx.close()
    return torch.cat([p[0] for p in parts]), torch.cat([p[1] for p in parts]), sum((p[2] for p in parts), [])


def run_passes(pkg, slots, passes, osd=0):
    d_i, d_q, _ = slots
    ctx = pkg.Context(0)
    ctx.set_osd(osd, -1)
    if passes is not None:
        ctx.set_passes(passes)
    res, nres = run_conditioned(ctx, d_i, d_q)
    out = dict(res=res, nres=nres, rows=pass1_rows(ctx, d_i.shape[0]), launches=ctx.launches(), ctx=ctx)
    return out


def test_arguments_are_checked(pkg):
    ctx = pkg.Context(0)
    for bad in (0, 4, -1):
        with pytest.raises(pkg.Ft8Error, match="passes must be 1"):
            ctx.set_passes(bad)
    ctx.close()
    p = pkg.Pipe(0, depth=2)
    with pytest.raises(pkg.Ft8Error):
        p.set_passes(4)
    h = np.zeros((4, 48000), np.float32)
    p.submit_slots_host(h, h)
    with pytest.raises(pkg.Ft8Error, match="in flight"):
        p.set_passes(2)
    p.collect(4)
    p.set_passes(2)
    p.close()


def test_off_means_off(pkg, crowded):
    never = run_passes(pkg, crowded, None)
    one = run_passes(pkg, crowded, 1)
    for o in (never, one):
        o["ctx"].close()
    assert one["launches"] == never["launches"]
    assert np.array_equal(one["nres"], never["nres"]) and one["res"].tobytes() == never["res"].tobytes()
    assert one["rows"]["ncand"].tobytes() == never["rows"]["ncand"].tobytes()
    for key in ("cand", "ok", "status", "msg"):
        assert one["rows"][key] == never["rows"][key], key
    # a context that ran with passes = 3 and is set back to 1 allocates nothing more and launches what a fresh one does
    ctx = pkg.Context(0)
    ctx.set_passes(3)
    run_conditioned(ctx, crowded[0][:8], crowded[1][:8])
    ctx.set_passes(1)
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    l0 = ctx.launches()
    fresh = pkg.Context(0)
    fresh.process_slots(crowded[0][:8], crowded[1][:8])
    lf = fresh.launches()
    fresh.close()
    res, nres = run_conditioned(ctx, crowded[0][:8], crowded[1][:8])
    torch.cuda.synchronize()
    assert ctx.launches() - l0 == lf and torch.cuda.mem_get_info()[0] >= free0 - (2 << 20)
    assert np.array_equal(nres, never["nres"][:8]) and res.tobytes() == never["res"][:8].tobytes()
    ctx.close()


def check_prefix(base, multi):
    assert multi["rows"]["ncand"].tobytes() == base["rows"]["ncand"].tobytes()
    for key in ("cand", "ok", "status", "msg"):
        assert multi["rows"][key] == base["rows"][key], key
    n1, nm = base["nres"], multi["nres"]
    assert np.all(nm >= n1)
    for s in range(n1.size):
        assert multi["res"][s][:n1[s]].tobytes() == base["res"][s][:n1[s]].tobytes(), s


def test_pass1_is_a_prefix_and_later_passes_gain(pkg, crowded):
    sent = crowded[2]
    runs = {p: run_passes(pkg, crowded, p) for p in (1, 2, 3)}
    for r in runs.values():
        r["ctx"].close()
    good = {}
    for p in (1, 2, 3):
        if p > 1:
            check_prefix(runs[1], runs[p])
            check_prefix(runs[p - 1], runs[p])
        g, bad = score(runs[p]["res"], runs[p]["nres"], sent)
        assert bad == 0, (p, bad)
        good[p] = g
    assert good[2] > good[1] and good[3] >= good[2], good


def test_with_osd_keeps_the_prefix(pkg, crowded):
    part = (crowded[0][:32], crowded[1][:32], crowded[2][:32])
    base = run_passes(pkg, part, 1, osd=2)
    multi = run_passes(pkg, part, 3, osd=2)
    check_prefix(base, multi)
    assert score(multi["res"], multi["nres"], part[2])[1] == 0
    multi["ctx"].set_profiling(True)
    run_conditioned(multi["ctx"], part[0], part[1])
    assert multi["ctx"].stage_times()["later_passes"] > 0
    base["ctx"].set_profiling(True)
    run_conditioned(base["ctx"], part[0], part[1])
    assert "later_passes" not in base["ctx"].stage_times()
    base["ctx"].close()
    multi["ctx"].close()


def test_deterministic_and_batch_invariant(pkg, crowded):
    d_i, d_q, _ = crowded
    ctx = pkg.Context(0)
    ctx.set_passes(3)
    idx = torch.arange(128, device=DEV) % 64
    big_i, big_q = d_i[idx].contiguous(), d_q[idx].contiguous()
    r1, n1 = run_conditioned(ctx, big_i, big_q)
    r2, n2 = run_conditioned(ctx, big_i, big_q)
    assert np.array_equal(n1, n2) and r1.tobytes() == r2.tobytes()
    for s in (0, 17, 40, 63):
        ra, na = run_conditioned(ctx, d_i[s:s + 1].contiguous(), d_q[s:s + 1].contiguous())
        for pos in (s, s + 64):
            assert na[0] == n1[pos] and ra[0].tobytes() == r1[pos].tobytes(), (s, pos)
    ctx.close()


@pytest.fixture(scope="module")
def raw_slot(pkg):
    """One crowded raw-IQ slot (2.4 Msps bytes, GFSK) of 40 CQ messages, and what it carries."""
    sig, first, sent = crowded_items(pkg, 1, 40, 0xAA55)
    sig["amp"] = [np.sqrt(2 * 900.0 * 2500 / 2.4e6 * 10 ** (snr / 10.0)) for snr in np.random.default_rng(7).uniform(-18, -6, sig.size)]
    ctx = pkg.Context(0)
    iq = ctx.synth_raw(sig, first, 30.0, 0xAA55)
    d_i, d_q, cnt, peak, _ = ctx.decimate(iq, 1, pkg.RAW_SLOT_BYTES, stride=iq.stride(0))
    ctx.condition(d_i, d_q, peak)
    torch.cuda.synchronize()
    ctx.close()
    return iq, d_i.cpu().numpy(), d_q.cpu().numpy(), sent


def test_every_entry_gains_on_a_raw_slot(pkg, raw_slot, tmp_path):
    iq, hi, hq, sent = raw_slot
    got = {}
    for passes in (1, 2):
        ctx = pkg.Context(0)
        ctx.set_passes(passes)
        ctx.process_raw(iq, 1, stride=iq.stride(0))
        got[passes] = ctx.fetch_results(1)
        ctx.close()
    g1, b1 = score(*got[1], sent)
    g2, b2 = score(*got[2], sent)
    assert g2 > g1 and b2 == 0, (g1, g2, b2)
    for back in (0, 40):
        p = pkg.Pipe(0, depth=2)
        if back:
            p.set_partition(back)
        p.set_passes(2)
        p.submit(iq, 1, stride=iq.stride(0))
        res, nres = p.collect(1)
        p.close()
        assert np.array_equal(nres, got[2][1]) and res.tobytes() == got[2][0].tobytes(), back
    # the drop-in ft8_subsystem on the decimated, conditioned slot, with the option from the environment
    np.savez(tmp_path / "slot.npz", i=hi, q=hq)
    script = tmp_path / "dropin.py"
    script.write_text(_DROPIN)
    ctx = pkg.Context(0)
    want = {}
    for passes in (1, 2):
        ctx.set_passes(passes)
        want[passes] = ctx.process_slots_host(hi, hq)
    ctx.close()
    assert want[2][1][0] > want[1][1][0]
    env = dict(os.environ, FT8B200_PASSES="2")
    p = subprocess.run([sys.executable, str(script), ROOT, str(tmp_path / "slot.npz")], env=env, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    n, recs = p.stdout.strip().splitlines()[-1].split(" ", 1)
    res, nres = want[2]
    calls = {bytes(r["call"]) for r in res[0][:nres[0]] if r["call"]}
    assert int(n) == nres[0] and set(recs.split(",")) - {""} == {c.decode() for c in calls}
    env["FT8B200_PASSES"] = "4"
    p = subprocess.run([sys.executable, str(script), ROOT, str(tmp_path / "slot.npz")], env=env, capture_output=True, text=True, timeout=600)
    assert p.returncode != 0 and "FT8B200_PASSES" in p.stderr


_DROPIN = r'''
import sys, numpy as np
sys.path.insert(0, sys.argv[1])
from ft8b200_loader import load
pkg = load()
d = np.load(sys.argv[2])
dec = np.zeros(50, pkg.result_dtype)
_, n = pkg.ft8_subsystem(d["i"][0], d["q"][0], dec)
print(n, ",".join(bytes(r["call"]).decode() for r in dec[:n] if r["call"]))
'''


def host_candidate(oracle, i, q):
    ci, cq, _ = oracle.condition(i, q, 48000)
    return oracle.find_sync(oracle.waterfall(ci, cq))[0]


def on_grid(oracle, f0, t0):
    """(f0, t0) moved onto the refinement grid of the candidate the signal gets (so that the coarse metric has one clear best:
    neighbours 16 samples or 6.25/32 Hz away score 3.2e-3 lower), or None when moving it changes the candidate."""
    from test_subtract import gfsk_slot, strongest_candidate
    x, _ = gfsk_slot(oracle, [("CQ", "K1ABC", "FN20", f0, t0, 1.0)])
    c = strongest_candidate(oracle, x)
    s_nom, f_nom = sr.nominal(c)
    start = s_nom + 16 * int(np.clip(round((int(np.float32(t0) * 3200.0 + 0.5) - s_nom) / 16), -8, 8))
    f1 = f_nom + sr.DF_STEP * int(np.clip(round((f0 - f_nom) / sr.DF_STEP), -8, 8))
    t1 = float(np.float32((start + 0.25) / 3200.0))
    x, _ = gfsk_slot(oracle, [("CQ", "K1ABC", "FN20", f1, t1, 1.0)])
    if tuple(strongest_candidate(oracle, x)) != tuple(c) or int(np.float32(t1) * 3200.0 + 0.5) != start:
        return None
    return f1, t1


def test_stage_entry_matches_the_float64_definition(pkg, oracle):
    """ft8b200_subtract against subtract_ref on device-synthesised GFSK, and the residual, with the kernel's grid, to 1e-4 of the
    peak.  Grid points: wherever the reference's coarse best and second best differ by more than 1e-3 (relative) the kernel's
    point must be the reference's.  The fine stage's neighbours, one sample apart, differ by only 2e-5 on GFSK (its smooth tone
    changes); that stage is exact in the kernel up to float32 rounding of 32-term partial sums (~1e-6 relative), so it is held
    to the reference wherever its gap exceeds 1e-5.  Everywhere the kernel's point must score within 1e-3 of the reference's
    best.  The nominal position is pinned: on the noiseless slots the refined start is the synthesised one."""
    rng = np.random.default_rng(11)
    specs = []   # per slot: list of (f0, t0, amp); noiseless slots first
    while len(specs) < 6:
        f0t0 = on_grid(oracle, float(rng.uniform(200, 1400)), float(rng.uniform(0.3, 1.2)))
        if f0t0:
            specs.append([(f0t0[0], f0t0[1], 1.0)])
    for k in range(2):
        specs.append([(float(rng.uniform(200, 1400)), float(rng.uniform(0.3, 1.2)), 1.0)])
    specs.append([(700.0, 0.5, 1.0), (760.0, 0.62, 0.5)])
    specs.append([(900.0, 0.7, 1.0), (904.0, 0.9, 0.7), (1300.0, 0.4, 0.3)])
    specs.append([])
    n = len(specs)
    ctx = pkg.Context(0)
    M = ctx.M
    items, first = [], [0]
    for sp in specs:
        for f0, t0, amp in sp:
            call = "K1ABC" if len(sp) == 1 and len(items) < 6 else f"K{len(items)}ABC"
            items.append((pkg.pack77_std("CQ", call, "FN20"), f0, t0, amp))
        first.append(len(items))
    sig = pkg.make_signals(items, gfsk=True)
    d_i, d_q = ctx.synth_slots(sig, np.array(first, np.int32), 0.0, 3)
    noisy_i, noisy_q = ctx.synth_slots(sig, np.array(first, np.int32), 0.05, 3)
    kept = {}
    for slots_i, slots_q, noiseless in ((d_i, d_q, True), (noisy_i, noisy_q, False)):
        hi, hq = slots_i.cpu().numpy(), slots_q.cpu().numpy()
        cand = np.zeros((n, M), cand_dtype)
        cw = np.zeros((n, M, 174), np.uint8)
        nmsg = np.zeros(n, np.int32)
        for s, sp in enumerate(specs):
            for j in range(len(sp)):
                g = first[s] + j
                one = pkg.make_signals([items[g]], gfsk=True)   # each message's candidate from its own slot
                a_i, a_q = ctx.synth_slots(one, np.array([0, 1], np.int32), 0.0, 3)
                cand[s, j] = host_candidate(oracle, a_i[0].cpu().numpy(), a_q[0].cpu().numpy())
                cw[s, j] = bits_from_tones(oracle.tones(items[g][0]))
            nmsg[s] = len(sp)
        d_cand = torch.from_numpy(cand.view(np.uint8).reshape(n, M, 8)).to(DEV)
        ri, rq, grid = ctx.subtract(slots_i, slots_q, d_cand, torch.from_numpy(cw).to(DEV), torch.from_numpy(nmsg).to(DEV))
        torch.cuda.synchronize()
        ri, rq, grid = ri.cpu().numpy(), rq.cpu().numpy(), grid.cpu().numpy()
        kept[noiseless] = (ri, rq, grid, d_cand, cw, nmsg)
        checked = 0
        for s, sp in enumerate(specs):
            x = hi[s].astype(np.float64) + 1j * hq[s].astype(np.float64)
            msgs = [(cand[s, j], cw[s, j]) for j in range(len(sp))]
            for j, (c, w) in enumerate(msgs):
                (dt, df), (coarse, fine) = sr.refine(x, c, w, with_metrics=True)
                cs, fs_ = np.sort(coarse.ravel()), np.sort(fine)
                if (cs[-1] - cs[-2]) > 1e-3 * cs[-1] and (fs_[-1] - fs_[-2]) > 1e-5 * fs_[-1]:
                    assert tuple(grid[s, j]) == (dt, df), (s, j, grid[s, j], dt, df)
                    checked += 1
                s0, f0 = sr.nominal(c)
                r = sr.reference(sr.tones_from_codeword(w), f0 + grid[s, j, 1] * sr.DF_STEP)
                assert sr.metric(x, s0 + grid[s, j, 0], r) >= (1 - 1e-3) * fs_[-1], (s, j)
                if noiseless and len(sp) == 1:
                    s0, _ = sr.nominal(c)
                    assert s0 + grid[s, j, 0] == int(np.float32(sp[j][1]) * 3200.0 + 0.5), (s, j)
            y, _ = sr.subtract(x, msgs, grids=[tuple(grid[s, j]) for j in range(len(sp))])
            peak = max(np.abs(hi[s]).max(), np.abs(hq[s]).max(), 1e-30)
            err = max(np.abs(ri[s] - y.real).max(), np.abs(rq[s] - y.imag).max())
            # float32 slots, r from a double phase through sincospif (~1e-7), the window sums in double: 1e-4 of the peak has room
            assert err <= 1e-4 * peak, (s, err / peak)
            if not sp:
                assert np.array_equal(ri[s], hi[s]) and np.array_equal(rq[s], hq[s])
        assert checked >= 6
    # in place (the residual over the input) gives the same bytes
    ri, rq, grid, d_cand, cw, nmsg = kept[True]
    a, b = d_i.clone(), d_q.clone()
    _, _, g2 = ctx.subtract(a, b, d_cand, torch.from_numpy(cw).to(DEV), torch.from_numpy(nmsg).to(DEV), out=(a, b))
    torch.cuda.synchronize()
    ctx.close()
    assert np.array_equal(g2.cpu().numpy(), grid) and np.array_equal(a.cpu().numpy(), ri) and np.array_equal(b.cpu().numpy(), rq)
