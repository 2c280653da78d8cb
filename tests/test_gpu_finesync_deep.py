"""Deep fine sync (ft8b200_set_finesync_deep, ft8b200_finesync_sets; DESIGN.md section 2.4.6) on the B200: the three refined LLR sets
against fine sync's own outputs and the float64 definition (tests/finesync_deep_ref.py), the retry chain on them byte for byte against
the CPU restatements of BP, OSD and AP, that deep mode off changes nothing, and every daemon entry against a composition of the
stage-wise calls.  Every test creates its own contexts and pipes."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import finesync_deep_ref as dr
import finesync_ref as fr
import subtract_ref as sr
import test_gpu_finesync as tgf
import test_gpu_multipass as mp
from conftest import ROOT
from oracle.pyoracle import cand_dtype, result_dtype
from test_ap import oracle  # noqa: F401 (the oracle fixture with the OSD and AP forms)
from test_gpu_ap import _Arr
from test_gpu_osd import expected_finish
from tools import synth

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
DEV = torch.device("cuda:0")
LLR_TOL = 1e-2   # float32 sums against float64, as test_gpu_finesync's


def caps_of():
    hdr = open(os.path.join(ROOT, "include", "ft8b200.h")).read()
    get = lambda name: int(re.search(r"#define FT8B200_%s_DEFAULT_MAX_HARD (\d+)" % name, hdr).group(1))
    return dict(deep=get("FINESYNC_DEEP"), fs=get("FINESYNC"), osd=get("OSD"), ap=get("AP"))


@pytest.fixture(scope="module")
def hand_slots():
    """8 slots (noise sigma 1 per rail): six with one GFSK CQ at about -13 ... -24 dB, two noise-only; 16 hand-placed candidates per slot
    (up to 16 live), half of them near the truth, and some stage 3/4 entries that must be left alone."""
    rng = np.random.Generator(np.random.PCG64(0xDEE9))
    K = 16
    starts = [1600, -20000, 30000, 27476, -10000, 2500]
    amps = [0.3, 0.15, 0.1, 0.085, 0.08, 0.2]
    xs, cands = [], np.zeros((8, K), cand_dtype)
    for s in range(8):
        x = rng.standard_normal(sr.SLOT) + 1j * rng.standard_normal(sr.SLOT)
        truth = None
        if s < 6:
            truth = (starts[s], float(rng.uniform(300, 1300)))
            x = x + tgf.gfsk(truth[0], truth[1], amps[s], rng)
        xs.append(x.astype(np.complex64))
        for k in range(K):
            if truth is not None and k < 8:
                s0 = 256 + 256 * round((truth[0] + rng.integers(-200, 201) - 256) / 256)
                f0s = int(round(truth[1] / 3.125 + rng.uniform(-0.45, 0.45)))
            else:
                s0 = 256 + 256 * int(rng.integers(-157, 187))
                f0s = int(rng.integers(60, 480))
            cands[s, k] = tgf.cand_rec(s0, f0s)
    stage0 = np.where(rng.random((8, K)) < 0.85, rng.integers(1, 3, (8, K)), rng.integers(3, 5, (8, K))).astype(np.uint8)
    ncand = np.array([14, 16, 12, 16, 15, 16, 13, 16], np.int32)
    return np.stack(xs), cands, stage0, ncand


def to_dev(x, cands, stage0, ncand):
    S, K = stage0.shape
    return (torch.from_numpy(np.ascontiguousarray(x.real, np.float32)).to(DEV), torch.from_numpy(np.ascontiguousarray(x.imag, np.float32)).to(DEV),
            torch.from_numpy(cands.view(np.uint8).reshape(S, K, 8).copy()).to(DEV), torch.from_numpy(ncand).to(DEV), torch.from_numpy(stage0).to(DEV))


def sets_of(ctx, x, cands, stage0, ncand):
    d_i, d_q, c, nc, st = to_dev(x, cands, stage0, ncand)
    grid, llr = ctx.finesync_sets(d_i, d_q, c, nc, st)
    torch.cuda.synchronize()
    return grid.cpu().numpy(), llr.cpu().numpy()


def fs_how(ctx, n):
    p = ctx.finesync_deep_workspace_ptrs()
    return torch.as_tensor(_Arr(p, (n, ctx.K), "|u1"), device=DEV).cpu().numpy() if p else None


def test_front_half_matches_finesync_and_the_definition(pkg, hand_slots):
    x, cands, stage0, ncand = hand_slots
    ctx = pkg.Context(0, max_candidates=16)
    ctx.set_finesync(1, -1)
    grid, sets = sets_of(ctx, x, cands, stage0, ncand)
    _, out = tgf.run_stage(pkg, ctx, x, cands, stage0, ncand)
    ctx.close()
    live = (np.arange(16)[None, :] < ncand[:, None]) & np.isin(stage0, (1, 2))
    assert np.array_equal(grid.view(np.uint32), out["grid"].view(np.uint32))
    assert np.array_equal(sets[0].view(np.uint32), out["llr"].view(np.uint32))   # set a: fine sync's LLRs bit for bit
    assert np.all(grid[~live] == 0) and np.all(sets[:, ~live] == 0)
    checked = 0
    for s, k in zip(*np.nonzero(live)):
        want = dr.sets_at(x[s].astype(np.complex128), cands[s, k], int(grid[s, k, 0]), int(grid[s, k, 1]))
        for j in (1, 2):
            assert np.array_equal(np.isfinite(want[j]), np.isfinite(sets[j, s, k])), (s, k, j)
            if fr.attempted(want[j]):
                np.testing.assert_allclose(sets[j, s, k], want[j], atol=LLR_TOL, rtol=0, err_msg=str((s, k, j)))
                checked += 1
    assert checked >= 150, checked


def expected_chain(oracle, sets, caps, dcap, osd, ap):
    """-> (fs, fs_hard, fs_how, codeword or None) of the retry chain on one candidate at stage 1 or 2 with these LLR sets; caps: the
    fine-sync, OSD and AP caps."""
    fs, hard, cw = tgf.expected_back_half(oracle, sets[0], caps["fs"])
    if fs == 2:
        return fs, hard, 1, cw
    for i, (j, dec) in enumerate([(0, 1), (0, 2), (1, 0), (1, 1), (1, 2), (2, 0), (2, 1), (2, 2)]):
        llr = sets[j]
        if dec == 0:
            f, h, w = tgf.expected_back_half(oracle, llr, min(caps["fs"], dcap))
            acc = f == 2
        elif dec == 1:
            if not osd:
                continue
            a, w, h, _ = oracle.osd(llr, osd, min(caps["osd"], dcap))
            acc = a == 1
        else:
            if not ap:
                continue
            a, w, h = oracle.ap(llr, min(caps["ap"], dcap))
            acc = a == 1
        if acc:
            return 2, h, 2 + i, w
    return fs, hard, 0, None


def test_back_half_byte_for_byte(pkg, oracle, hand_slots):
    """On the kernel's own sets at deep caps {0, 12, default} x OSD {0, 2} x AP {0, 1}, and once with fine sync's own cap at 0 (so that
    the later steps get candidates set a's BP would take): fs, fs_hard, fs_how, ok, stage, status, msg and plain equal the CPU chain
    (orc_bp_decode, orc_osd, orc_ap, finish()), and sentinels elsewhere, past ncand included, are untouched."""
    x, cands, stage0, ncand = hand_slots
    S, K = stage0.shape
    caps = caps_of()
    ctx = pkg.Context(0, max_candidates=K)
    _, sets = sets_of(ctx, x, cands, stage0, ncand)
    ctx.close()
    hows = {}
    runs = [(dcap, osd, ap, caps["fs"]) for dcap in (0, 12, caps["deep"]) for osd in (0, 2) for ap in (0, 1)] + [(caps["deep"], 2, 1, 0)]
    for dcap, osd, ap, fs_cap in runs:
        caps = dict(caps, fs=fs_cap)
        ctx = pkg.Context(0, max_candidates=K)
        ctx.set_finesync(1, fs_cap)
        ctx.set_finesync_deep(1, dcap)
        ctx.set_osd(osd, -1)
        ctx.set_ap(ap, -1)
        sent, out = tgf.run_stage(pkg, ctx, x, cands, stage0, ncand, rng_seed=dcap + 7 * osd + ap + fs_cap)
        how = fs_how(ctx, S)
        ctx.close()
        for s in range(S):
            for k in range(K):
                if k >= ncand[s] or stage0[s, k] not in (1, 2):
                    w = (0, -1, 0, None)
                else:
                    w = expected_chain(oracle, sets[:, s, k], caps, dcap, osd, ap)
                got = (out["fs"][s, k], out["hard"][s, k], how[s, k])
                assert got == w[:3], (dcap, osd, ap, s, k, got, w[:3])
                hows[w[2]] = hows.get(w[2], 0) + 1
                if w[3] is not None:
                    est, emsg = expected_finish(oracle, w[3], 1)
                    assert out["ok"][s, k] == 1 and out["stage"][s, k] == 4
                    assert out["status"][s, k].tobytes() == est and out["msg"][s, k].tobytes() == emsg
                    assert np.array_equal(out["plain"][s, k], w[3])
                else:
                    for key in ("ok", "stage", "status", "msg", "plain"):
                        assert np.array_equal(out[key][s, k], sent[key][s, k]), (dcap, osd, ap, s, k, key)
    assert hows.get(1, 0) >= 10 and sum(v for h, v in hows.items() if h >= 2) >= 1, hows


@pytest.fixture(scope="module")
def weak_slots(pkg):
    """48 device slots of 1-8 GFSK CQ and non-CQ messages at -24 ... -17 dB (noise 1.0) with their peaks."""
    rng = np.random.Generator(np.random.PCG64(0xDEE51))
    slots = []
    for s in range(48):
        sp = []
        for _ in range(1 + s % 8):
            to = "CQ" if rng.random() < 0.6 else synth.random_call(rng)
            sp.append((pkg.pack77_std(to, synth.random_call(rng), synth.random_grid(rng)), float(rng.uniform(100, 1500)),
                       float(0.5 + rng.uniform(-0.3, 0.3)), mp.amp_for(float(rng.uniform(-24, -17)))))
        slots.append(sp)
    first = np.cumsum([0] + [len(sp) for sp in slots]).astype(np.int32)
    ctx = pkg.Context(0)
    d_i, d_q = ctx.synth_slots(pkg.make_signals([it for sp in slots for it in sp], gfsk=True), first, 1.0, 0xDEE51)
    peak = torch.maximum(d_i.abs().amax(1), d_q.abs().amax(1)).contiguous()
    torch.cuda.synchronize()
    ctx.close()
    return d_i, d_q, peak


def test_off_is_untouched(pkg, weak_slots, hand_slots):
    """Deep mode off, or on with fine sync off: records, rows and launch counts as a context that never called the setter, nothing
    allocated, and no fs_how row."""
    d_i, d_q, peak = weak_slots
    n = d_i.shape[0]
    for fs_on in (0, 1):
        fresh = pkg.Context(0)
        fresh.set_finesync(fs_on, -1)
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        fresh.process_conditioned(d_i, d_q, peak)
        r0, o0, l0 = fresh.fetch_results(n), tgf.outputs(fresh, n), fresh.launches()
        torch.cuda.synchronize()
        used0 = free0 - torch.cuda.mem_get_info()[0]
        variants = [(0, 12)] + ([(1, -1)] if not fs_on else [])
        for on, cap in variants:
            c = pkg.Context(0)
            c.set_finesync(fs_on, -1)
            c.set_finesync_deep(on, cap)
            torch.cuda.synchronize()
            free0 = torch.cuda.mem_get_info()[0]
            c.process_conditioned(d_i, d_q, peak)
            r1, o1 = c.fetch_results(n), tgf.outputs(c, n)
            torch.cuda.synchronize()
            assert abs((free0 - torch.cuda.mem_get_info()[0]) - used0) <= (2 << 20), (fs_on, on)
            assert c.launches() == l0 and c.finesync_deep_workspace_ptrs() == 0, (fs_on, on)
            mp.check_records(r1, r0, (fs_on, on))
            assert np.array_equal(o0["ncand"], o1["ncand"])
            for key in o0:
                assert (o0[key] is None) == (o1[key] is None), (fs_on, on, key)
                if key == "ncand" or o0[key] is None:
                    continue
                for s in range(n):   # the rows of live candidates: entries past ncand hold whatever the buffer held
                    nc = int(o0["ncand"][s]) * (8 if key == "cand" else 1)
                    assert np.array_equal(o0[key][s, :nc], o1[key][s, :nc]), (fs_on, on, key, s)
            c.close()
        fresh.close()
    x, cands, stage0, ncand = hand_slots
    ctx = pkg.Context(0, max_candidates=16)
    ctx.set_finesync_deep(1, -1)   # fine sync off: the stage-wise entry attempts nothing and allocates no fs_how row
    sent, out = tgf.run_stage(pkg, ctx, x, cands, stage0, ncand)
    assert np.all(out["fs"] == 0) and np.all(out["hard"] == -1) and ctx.finesync_deep_workspace_ptrs() == 0
    for key in ("ok", "stage", "status", "msg", "plain"):
        assert np.array_equal(out[key], sent[key]), key
    for on in (-1, 2, 7):
        with pytest.raises(pkg.Ft8Error):
            ctx.set_finesync_deep(on, -1)
    ctx.close()


@pytest.mark.parametrize("osd,ap", [(0, 0), (2, 1)])
def test_pass1_superset(pkg, weak_slots, osd, ap):
    """Every pass-1 row decoded with deep mode off is decoded identically with it on; every other row stays as it was (fs and fs_hard
    included) or becomes a fine-sync decode with fs_how >= 2."""
    d_i, d_q, peak = weak_slots
    n = d_i.shape[0]
    outs = []
    for deep in (0, 1):
        c = pkg.Context(0)
        c.set_osd(osd, -1)
        c.set_ap(ap, -1)
        c.set_finesync(1, -1)
        c.set_finesync_deep(deep, -1)
        c.process_conditioned(d_i, d_q, peak)
        outs.append((tgf.outputs(c, n), fs_how(c, n)))
        c.close()
    (ob, _), (o1, how) = outs
    assert np.array_equal(ob["ncand"], o1["ncand"]) and np.array_equal(ob["cand"], o1["cand"])
    new = 0
    for s in range(n):
        for k in range(int(ob["ncand"][s])):
            same = all(np.array_equal(ob[key][s, k], o1[key][s, k]) for key in ("ok", "status", "msg"))
            if how[s, k] >= 2:
                assert ob["ok"][s, k] == 0 and o1["ok"][s, k] == 1 and o1["fs"][s, k] == 2, (s, k)
                new += 1
            else:
                assert same and ob["fs"][s, k] == o1["fs"][s, k] and ob["hard"][s, k] == o1["hard"][s, k], (s, k)
                assert how[s, k] == (1 if o1["fs"][s, k] == 2 else 0), (s, k)
    print("deep decodes", osd, ap, new)


@pytest.mark.parametrize("osd,ap", [(0, 0), (2, 1)])
def test_conditioned_and_slots_compose(pkg, oracle, weak_slots, osd, ap, monkeypatch):
    """process_conditioned and process_slots at passes 1, 2 and 3 with deep fine sync equal the composition of the stage-wise entries
    (ft8b200_decode, ft8b200_finesync with deep mode, spots): pass-1 rows byte for byte and the records."""
    d_i, d_q, peak = weak_slots
    n = d_i.shape[0]
    c_i, c_q = d_i.clone(), d_q.clone()
    cond = pkg.Context(0)
    cond.condition(c_i, c_q, peak.clone())
    cond.close()
    cfg = mp.cfg_of("default")
    monkeypatch.setattr(mp, "stage", tgf.stage_with_fs)

    def make():
        c = pkg.Context(0, **cfg)
        c.set_osd(osd, -1)
        c.set_ap(ap, -1)
        c.set_finesync(1, -1)
        c.set_finesync_deep(1, -1)
        return c
    ref = make()
    st = mp.new_stats()
    tgf.FS.clear()
    for passes in (1, 2, 3):
        for entry, (x_i, x_q, pk) in (("conditioned", (d_i, d_q, peak)), ("slots", (c_i, c_q, None))):
            if entry == "slots" and passes == 3:
                continue
            ctx = make()
            ctx.set_passes(passes)
            if pk is None:
                ctx.process_slots(x_i, x_q)
            else:
                ctx.process_conditioned(x_i, x_q, pk)
            got = ctx.fetch_results(n)
            R1, wres, wnres = mp.compose(ref, oracle, x_i, x_q, pk, passes, osd, cfg, st)
            mp.check_pass1(ctx, n, R1)
            mp.check_records(got, (wres, wnres), (osd, ap, passes, entry))
            ctx.close()
    ref.close()
    assert tgf.fs_decodes_are_codewords() >= 3 and st["appended_in_pass2"] >= 1


def test_raw_entries_and_pipes(pkg, oracle, monkeypatch):
    """process_raw in 4 overlap groups and process_raw_streams at passes 2 with OSD 2, AP and deep fine sync equal the composition on the
    decimated slots; a pipe with and without an SM partition equals process_raw batch by batch, and its setter is EBUSY in flight."""
    sig, first = mp.fixture_items(pkg, 0x7E13, n_crowded=4, specials_first=True)
    sig["amp"] *= np.float32(1.2 * np.sqrt(2 * 900.0 * 2500 / 2.4e6) / np.sqrt(2 * 2500 / 3200.0))
    c0 = pkg.Context(0)
    raw = c0.synth_raw(sig, first, 30.0, 0x7E13)
    torch.cuda.synchronize()
    c0.close()
    n = raw.shape[0]
    cfg = mp.cfg_of("default")
    monkeypatch.setattr(mp, "stage", tgf.stage_with_fs)

    def make(c):
        c.set_osd(2, -1)
        c.set_ap(1, -1)
        c.set_finesync(1, -1)
        c.set_finesync_deep(1, -1)
        return c
    ref = make(pkg.Context(0))
    st = mp.new_stats()
    ctx = make(pkg.Context(0))
    ctx.set_passes(2)
    for run in ("overlap", "streams"):
        if run == "overlap":
            ctx.set_overlap(4)
            ctx.process_raw(raw, n, stride=raw.stride(0))
        else:
            ctx.set_overlap(0)
            ctx.process_raw_streams(raw, n // 2, 2, stride=2 * raw.stride(0))
        got = ctx.fetch_results(n)
        x_i, x_q, pk = mp.workspace_slots(ctx, n)
        R1, wres, wnres = mp.compose(ref, oracle, x_i, x_q, pk, 2, 2, cfg, st)
        mp.check_pass1(ctx, n, R1)
        mp.check_records(got, (wres, wnres), run)
    want = []
    for b in range(2):
        ctx.process_raw(raw[4 * b:4 * b + 4], 4, stride=raw.stride(0))
        want.append(ctx.fetch_results(4))
    ctx.close()
    ref.close()
    for back in (0, 40):
        p = pkg.Pipe(0, depth=2)
        if back:
            p.set_partition(back)
        make(p)
        p.set_passes(2)
        with pytest.raises(pkg.Ft8Error):
            p.set_finesync_deep(2, -1)
        p.submit(raw[:4], 4, stride=raw.stride(0))
        with pytest.raises(pkg.Ft8Error):
            p.set_finesync_deep(0, -1)   # EBUSY while a batch is in flight
        p.submit(raw[4:8], 4, stride=raw.stride(0))
        got = [p.collect(4) for _ in range(2)]
        p.close()
        for b in range(2):
            mp.check_records(got[b], want[b], ("pipe", back, b))


def test_dropin_environment_and_iq_files(pkg, oracle, weak_slots, tmp_path):
    d_i, d_q, peak = weak_slots
    hi = (d_i[:12] * (0.5 / peak[:12, None])).cpu().numpy()
    hq = (d_q[:12] * (0.5 / peak[:12, None])).cpu().numpy()
    np.savez(tmp_path / "slots.npz", i=hi, q=hq)
    script = tmp_path / "dropin.py"
    script.write_text(tgf._DROPIN)
    run = lambda env: subprocess.run([sys.executable, str(script), ROOT, str(tmp_path / "slots.npz"), str(tmp_path / "out.npy")], env=env,
                                     capture_output=True, text=True, timeout=600)
    base = {k: v for k, v in os.environ.items() if not k.startswith("FT8B200_")}
    base["FT8B200_FINESYNC"] = "1"
    for bad in ({"FT8B200_FINESYNC_DEEP": "2"}, {"FT8B200_FINESYNC_DEEP": "x"},
                {"FT8B200_FINESYNC_DEEP": "1", "FT8B200_FINESYNC_DEEP_MAX_HARD": "175"}):
        p = run(dict(base, **bad))
        assert p.returncode != 0 and "FT8B200_FINESYNC_DEEP" in p.stderr, bad
    p = run(dict(base, FT8B200_FINESYNC_DEEP="1", FT8B200_FINESYNC_DEEP_MAX_HARD="60"))
    assert p.returncode == 0, p.stderr[-2000:]
    got = np.load(tmp_path / "out.npy", allow_pickle=True)
    got_n = np.load(tmp_path / "out.npy.n.npy")
    ctx = pkg.Context(0)
    ctx.set_finesync(1, -1)
    ctx.set_finesync_deep(1, 60)
    for s in range(12):
        res, nres = ctx.process_slots_host(hi[s:s + 1], hq[s:s + 1])
        want = np.zeros(50, result_dtype)
        for k in range(int(nres[0])):
            if res[0][k]["call"]:
                want[k] = res[0][k]
        assert got_n[s] == nres[0] and got[s] == want.tobytes(), s
    paths = []
    for s in range(4):
        inter = np.empty(2 * sr.SLOT, np.float32)
        inter[0::2], inter[1::2] = hi[s] * 3.0, -hq[s] * 3.0
        path = tmp_path / f"s{s}.iq"
        inter.tofile(path)
        paths.append(str(path))
    res, nres, _ = pkg.decode_iq_files(ctx, paths)
    for s in range(4):
        inter = np.fromfile(paths[s], np.float32)
        ci, cq, _ = oracle.condition(inter[0::2].copy(), -inter[1::2], sr.SLOT)
        w, wn = ctx.process_slots_host(ci[None], cq[None])
        assert nres[s] == wn[0] and res[s].tobytes() == w[0].tobytes(), s
    ctx.close()


def test_shapes_and_argument_checks(pkg, hand_slots):
    """More than 2 x SMs slots (300 copies of the hand slots): every slot's sets, grid and chain outputs equal those of the slot run alone;
    misaligned or out-of-range arguments to ft8b200_finesync_sets are refused with nothing written."""
    x, cands, stage0, ncand = hand_slots
    ctx = pkg.Context(0, max_candidates=16)
    ctx.set_finesync(1, -1)
    ctx.set_finesync_deep(1, -1)
    ctx.set_osd(2, -1)
    ctx.set_ap(1, -1)
    alone = []
    for s in range(8):
        g, l = sets_of(ctx, x[s:s + 1], cands[s:s + 1], stage0[s:s + 1], ncand[s:s + 1])
        _, o = tgf.run_stage(pkg, ctx, x[s:s + 1], cands[s:s + 1], stage0[s:s + 1], ncand[s:s + 1])
        alone.append((g, l, o, fs_how(ctx, 1)))
    idx = np.arange(8 * (300 // 8 + 1)) % 8
    g, l = sets_of(ctx, x[idx], cands[idx], stage0[idx], ncand[idx])
    _, big = tgf.run_stage(pkg, ctx, x[idx], cands[idx], stage0[idx], ncand[idx])
    how = fs_how(ctx, idx.size)
    for r, s in enumerate(idx):
        ag, al, ao, ah = alone[s]
        assert np.array_equal(g[r], ag[0]) and np.array_equal(l[:, r].view(np.uint32), al[:, 0].view(np.uint32)), (r, s)
        assert np.array_equal(how[r], ah[0]), (r, s)
        for key in ("fs", "hard", "grid"):
            assert np.array_equal(big[key][r], ao[key][0]), (r, s, key)
        dec = big["fs"][r] == 2
        for key in ("ok", "stage", "status", "msg", "plain"):
            assert np.array_equal(big[key][r][dec], ao[key][0][dec]), (r, s, key)
    K = 16
    d = torch.zeros((2, sr.SLOT + 1), dtype=torch.float32, device=DEV)
    c = torch.zeros((1, K, 8), dtype=torch.uint8, device=DEV)
    nc = torch.full((1,), K, dtype=torch.int32, device=DEV)
    st = torch.ones((1, K), dtype=torch.uint8, device=DEV)
    grid = torch.full((1, K, 2), 7, dtype=torch.int32, device=DEV)
    llr = torch.full((3, 1, K, 174), 7.0, dtype=torch.float32, device=DEV)
    call = lambda xi, xq, n, gp, lp: ctx._chk(ctx.L.ft8b200_finesync_sets(pkg.C.c_void_p(ctx.h), pkg.C.c_void_p(xi), pkg.C.c_void_p(xq), n, pkg._p(c),
                                                                          pkg._p(nc), pkg._p(st), pkg.C.c_void_p(gp), pkg.C.c_void_p(lp), None))
    base, gp, lp = d.data_ptr(), grid.data_ptr(), llr.data_ptr()
    for args in ((base + 2, base + 4 * 48001, 1, gp, lp), (base, base + 4 * 48001 + 1, 1, gp, lp), (base, base + 4 * 48001, 1, gp + 2, lp),
                 (base, base + 4 * 48001, 1, gp, lp + 2), (base, base + 4 * 48001, 0, gp, lp), (base, base + 4 * 48001, 65536, gp, lp),
                 (0, base, 1, gp, lp), (base, base + 4 * 48001, 1, 0, lp), (base, base + 4 * 48001, 1, gp, 0)):
        with pytest.raises(pkg.Ft8Error):
            call(*args)
    torch.cuda.synchronize()
    assert bool(torch.all(grid == 7)) and bool(torch.all(llr == 7.0))
    ctx.close()
