"""Fine-sync decoding (ft8b200_set_finesync, ft8b200_finesync; DESIGN.md section 2.4.4) on the B200: the front half against the
float64 definition (tests/finesync_ref.py), the back half byte for byte against the CPU restatement of BP and the gates, that only
candidates at stage 1 or 2 change, and every daemon entry against a composition of the stage-wise calls.  Every test creates its own
contexts and pipes: the session contexts of the other suites never have fine sync switched on."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import finesync_ref as fr
import subtract_ref as sr
import test_gpu_multipass as mp
from conftest import ROOT
from oracle.pyoracle import cand_dtype, msg_dtype, result_dtype, status_dtype
from ref64 import crc_ok, gfsk_phase
from test_gpu_ap import _Arr
from test_gpu_osd import expected_finish
from tools import ft8enc, synth

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
DEV = torch.device("cuda:0")

# Grid parity bounds.  The coarse stage evaluates S on 8-sample sub-block sums rotated to each df (slot_search.cuh), which drops a
# rotation of at most 0.0107 rad within a sub-block.  coarse_subblock restates that approximation in float64, and err = max over the
# grid of |S_sub - S| bounds how far it moves any grid point: where float64's best coarse metric beats the runner-up by more than
# 2 err (+ FLOAT_GAP of float32 rounding), the coarse choice is the same.  The fine stage is exact: float32 sums of 512 products are
# within ~1e-6 relative of float64, so a gap above FLOAT_GAP = 1e-4 fixes the final dt.
FLOAT_GAP = 1e-4
# LLR tolerance: float32 symbol sums against float64, through 10 log10 of the power; a nearly cancelled bin loses relative accuracy,
# and the normalised LLRs are O(1).
LLR_TOL = 1e-2


@pytest.fixture(scope="module")
def default_cap(pkg):
    hdr = open(os.path.join(ROOT, "include", "ft8b200.h")).read()
    return int(re.search(r"#define FT8B200_FINESYNC_DEFAULT_MAX_HARD (\d+)", hdr).group(1))


def gfsk(start, f_hz, amp, rng):
    p = ft8enc.pack_std("CQ", synth.random_call(rng), synth.random_grid(rng))
    phase, env = gfsk_phase(ft8enc.tones(p), sr.SYM, sr.FS, f_hz, sr.TONE_HZ, 2.0)
    x = np.zeros(sr.SLOT, np.complex128)
    n = start + np.arange(phase.size)
    inside = (n >= 0) & (n < sr.SLOT)
    x[n[inside]] = amp * env[inside] * np.exp(1j * phase[inside])
    return x


def coarse_subblock(x, cand):
    """The coarse stage as finesync_kernel computes it, in float64: per Costas symbol and coarse dt the sub-block sums at df = 0,
    rotated to each df by exp(-2 pi i df (8 b + 3.5) / fs) -> [33, 17]."""
    s0, f0 = sr.nominal(cand)
    b = np.arange(64)
    w = np.exp(-2j * np.pi * (sr.DF_STEPS[:, None] * sr.DF_STEP) * (8 * b[None, :] + 3.5) / sr.FS)   # [17, 64]
    m = np.arange(sr.SYM)
    out = np.zeros((33, 17))
    for k, c in zip(fr.COSTAS_SYMS, fr.COSTAS_TONES):
        idx = s0 + 512 * k - 256 + np.arange(1024)
        win = np.where((idx >= 0) & (idx < sr.SLOT), x[np.clip(idx, 0, sr.SLOT - 1)], 0)
        r = np.exp(-2j * np.pi * (f0 + sr.TONE_HZ * c) * m / sr.FS)
        B = np.stack([(win[16 * d:16 * d + 512] * r).reshape(64, 8).sum(1) for d in range(33)])   # [33, 64]
        out += np.abs(B @ w.T) ** 2
    return out


def cand_rec(s0, f0_steps, score=20):
    c = np.zeros(1, cand_dtype)
    to, ts = divmod(s0 - 256, 512)
    fo, fs = divmod(f0_steps, 2)
    c[0] = (score, to, fo, ts // 256, fs)
    return c[0]


@pytest.fixture(scope="module")
def hand_slots():
    """8 slots (noise sigma 1 per rail): six with one GFSK CQ at -12 ... -23 dB in 2500 Hz, true starts from -40 000 to 47 700 samples,
    two noise-only; 16 hand-placed candidates per slot (up to 14 live): nominal positions within the grid's reach of the truth,
    others anywhere from -40 000 to +47 700, and a few stage 3/4 entries that must be left alone."""
    rng = np.random.Generator(np.random.PCG64(0xF5))
    K = 16
    starts = [1600, -20000, 30000, 27476, -10000, 2500]
    amps = [0.3, 0.15, 0.12, 0.1, 0.09, 0.2]
    xs, cands, truth = [], np.zeros((8, K), cand_dtype), []
    for s in range(8):
        x = (rng.standard_normal(sr.SLOT) + 1j * rng.standard_normal(sr.SLOT))
        if s < 6:
            f_true = float(rng.uniform(300, 1300))
            x = x + gfsk(starts[s], f_true, amps[s], rng)
            truth.append((starts[s], f_true))
        else:
            truth.append(None)
        xs.append(x.astype(np.complex64))
        for k in range(K):
            if truth[-1] is not None and k < 8:
                st0, ft = truth[-1]
                s0 = 256 + 256 * round((st0 + rng.integers(-200, 201) - 256) / 256)
                f0s = int(round(ft / 3.125 + rng.uniform(-0.45, 0.45)))
            else:
                s0 = 256 + 256 * int(rng.integers(-157, 187))   # -39 936 ... 47 616
                f0s = int(rng.integers(60, 480))
            cands[s, k] = cand_rec(s0, f0s)
    x = np.stack(xs)
    stage0 = np.where(rng.random((8, K)) < 0.85, rng.integers(1, 3, (8, K)), rng.integers(3, 5, (8, K))).astype(np.uint8)
    ncand = np.array([14, 16, 12, 16, 15, 16, 13, 16], np.int32)
    return x, cands, stage0, ncand, truth


def run_stage(pkg, ctx, x, cands, stage0, ncand, rng_seed=1):
    S, K = stage0.shape
    rng = np.random.default_rng(rng_seed)
    d_i = torch.from_numpy(np.ascontiguousarray(x.real, np.float32)).to(DEV)
    d_q = torch.from_numpy(np.ascontiguousarray(x.imag, np.float32)).to(DEV)
    sent = dict(ok=np.zeros((S, K), np.uint8), stage=stage0.copy(), status=rng.integers(0, 256, (S, K, 12), dtype=np.uint8),
                msg=rng.integers(0, 256, (S, K, 28), dtype=np.uint8), plain=rng.integers(0, 2, (S, K, 174), dtype=np.uint8))
    t = {k: torch.from_numpy(v.copy()).to(DEV) for k, v in sent.items()}
    c = torch.from_numpy(cands.view(np.uint8).reshape(S, K, 8).copy()).to(DEV)
    nc = torch.from_numpy(ncand).to(DEV)
    fs, hard, grid, llr = ctx.finesync(d_i, d_q, c, nc, t["ok"], t["stage"], t["status"], t["msg"], t["plain"], want_llr=True)
    torch.cuda.synchronize()
    out = {k: v.cpu().numpy() for k, v in t.items()}
    out.update(fs=fs.cpu().numpy(), hard=hard.cpu().numpy(), grid=grid.cpu().numpy(), llr=llr.cpu().numpy())
    return sent, out


def test_front_half_matches_the_definition(pkg, hand_slots, default_cap):
    x, cands, stage0, ncand, truth = hand_slots
    ctx = pkg.Context(0, max_candidates=16)
    ctx.set_finesync(1, -1)
    _, out = run_stage(pkg, ctx, x, cands, stage0, ncand)
    ctx.close()
    exact = coarse_only = llr_checked = near_truth = sub_checked = 0
    errs = []
    for s in range(x.shape[0]):
        xs = x[s].astype(np.complex128)
        for k in range(int(ncand[s])):
            if stage0[s, k] not in (1, 2):
                assert np.all(out["grid"][s, k] == 0) and np.all(out["llr"][s, k] == 0), (s, k)
                continue
            (dt, df), (coarse, fine) = fr.search(xs, cands[s, k], with_metrics=True)
            gdt, gdf = (int(v) for v in out["grid"][s, k])
            top = np.sort(coarse.reshape(-1))[::-1]
            sub = coarse_subblock(xs, cands[s, k])
            err = float(np.max(np.abs(sub - coarse)))
            errs.append(err / top[0] if top[0] > 0 else 0.0)
            ts = np.sort(sub.reshape(-1))[::-1]
            if ts[0] - ts[1] > FLOAT_GAP * ts[0]:   # the kernel's own approximation, restated: only float32 rounding apart
                i, j = sr.pick(sub)
                assert gdf == sr.DF_STEPS[j] and abs(gdt - fr.DT_COARSE[i]) <= 8, (s, k, (gdt, gdf), (i, j))
                sub_checked += 1
            if top[0] - top[1] > 2 * err + FLOAT_GAP * top[0]:
                assert gdf == df and abs(gdt - dt) <= 8, (s, k, (gdt, gdf), (dt, df))
                tf = np.sort(fine)[::-1]
                if tf[0] - tf[1] > FLOAT_GAP * tf[0]:
                    assert gdt == dt, (s, k, gdt, dt)
                    exact += 1
                else:
                    coarse_only += 1
            # the LLRs at the kernel's own grid point
            s0, f0 = sr.nominal(cands[s, k])
            want = fr.llrs_from_power(fr.spectra(xs, s0 + gdt, f0 + gdf * sr.DF_STEP))
            got = out["llr"][s, k]
            assert np.array_equal(np.isfinite(want), np.isfinite(got)), (s, k)
            if fr.attempted(want):
                np.testing.assert_allclose(got, want, atol=LLR_TOL, rtol=0, err_msg=str((s, k)))
                llr_checked += 1
            if truth[s] is not None and k < 8 and abs(s0 + gdt - truth[s][0]) <= 8:
                near_truth += 1
    assert exact >= 10 and sub_checked >= 60 and llr_checked >= 60 and near_truth >= 15, \
        (exact, coarse_only, sub_checked, llr_checked, near_truth, np.percentile(errs, [50, 90, 100]))


def expected_back_half(oracle, llr, cap):
    """-> (fs, hard, codeword or None) of rebp_kernel (fine sync: nothing forced) for one candidate at stage 1 or 2 with these LLRs."""
    if not np.all(np.isfinite(llr)):
        return 0, -1, None
    plain, err = oracle.bp_decode(llr, 20)
    hard = int(np.sum(plain != (llr > 0)))
    if err != 0 or not crc_ok(plain):
        return 1, hard, None
    a = np.packbits(np.concatenate([plain[:91], np.zeros(5, np.uint8)])).tobytes()
    rc, _ = oracle.unpack77(a[:9] + bytes([a[9] & 0xF8]))
    if rc < 0 or hard > cap:
        return 1, hard, None
    return 2, hard, plain


def test_back_half_byte_for_byte(pkg, oracle, hand_slots, default_cap):
    """Given the kernel's own refined LLRs: fs, fs_hard, ok, stage, status, msg and plain equal the CPU restatement of BP (orc_bp_decode),
    finish() and the hard-distance gate at three caps; sentinels in every entry fine sync leaves alone, past ncand included."""
    x, cands, stage0, ncand, _ = hand_slots
    S, K = stage0.shape
    decoded_at = {}
    for cap in (0, 12, default_cap):
        ctx = pkg.Context(0, max_candidates=K)
        ctx.set_finesync(1, cap)
        sent, out = run_stage(pkg, ctx, x, cands, stage0, ncand, rng_seed=cap)
        ctx.close()
        acc = rej = 0
        for s in range(S):
            for k in range(K):
                if k >= ncand[s] or stage0[s, k] not in (1, 2):
                    w = (0, -1, None)
                else:
                    w = expected_back_half(oracle, out["llr"][s, k], cap)
                assert (out["fs"][s, k], out["hard"][s, k]) == w[:2], (cap, s, k, out["fs"][s, k], out["hard"][s, k], w[:2])
                if w[0] == 2:
                    est, emsg = expected_finish(oracle, w[2], 1)
                    assert out["ok"][s, k] == 1 and out["stage"][s, k] == 4
                    assert out["status"][s, k].tobytes() == est and out["msg"][s, k].tobytes() == emsg and np.array_equal(out["plain"][s, k], w[2])
                    acc += 1
                else:
                    for key in ("ok", "stage", "status", "msg", "plain"):
                        assert np.array_equal(out[key][s, k], sent[key][s, k]), (cap, s, k, key)
                    rej += w[0] == 1
        decoded_at[cap] = acc
        assert rej >= 20, (cap, rej)
    assert decoded_at[default_cap] >= 5, decoded_at


def test_off_and_argument_checks(pkg, hand_slots):
    x, cands, stage0, ncand, _ = hand_slots
    ctx = pkg.Context(0, max_candidates=16)
    for on in (-1, 2, 7):
        with pytest.raises(pkg.Ft8Error):
            ctx.set_finesync(on, -1)
    sent, out = run_stage(pkg, ctx, x, cands, stage0, ncand)   # off: nothing attempted, nothing written but fs / fs_hard
    assert np.all(out["fs"] == 0) and np.all(out["hard"] == -1) and np.all(out["grid"] == 0) and np.all(out["llr"] == 0)
    for key in ("ok", "stage", "status", "msg", "plain"):
        assert np.array_equal(out[key], sent[key]), key
    ctx.set_finesync(1, -1)
    S, K = stage0.shape
    d = torch.zeros((2, sr.SLOT + 1), dtype=torch.float32, device=DEV)
    u8 = torch.zeros((1, K), dtype=torch.uint8, device=DEV)
    marks = [torch.full((1, K), 7, dtype=torch.uint8, device=DEV), torch.full((1, K), 7, dtype=torch.int32, device=DEV),
             torch.full((1, K, 2), 7, dtype=torch.int32, device=DEV), torch.full((1, K, 174), 7.0, dtype=torch.float32, device=DEV)]
    c = torch.zeros((1, K, 8), dtype=torch.uint8, device=DEV)
    nc = torch.full((1,), K, dtype=torch.int32, device=DEV)
    st = torch.zeros((1, K, 12), dtype=torch.uint8, device=DEV)
    ms = torch.zeros((1, K, 28), dtype=torch.uint8, device=DEV)
    call = lambda xi, xq, n, llr: ctx._chk(ctx.L.ft8b200_finesync(pkg.C.c_void_p(ctx.h), pkg.C.c_void_p(xi), pkg.C.c_void_p(xq), n, pkg._p(c), pkg._p(nc),
                                                                   pkg._p(u8), pkg._p(u8), pkg._p(st), pkg._p(ms), None, pkg._p(marks[0]), pkg._p(marks[1]),
                                                                   pkg._p(marks[2]), pkg.C.c_void_p(llr), None))
    base = d.data_ptr()
    for args in ((base + 2, base + 4 * 48001, 1, 0), (base, base + 4 * 48001 + 1, 1, 0), (base, base + 4 * 48001, 1, marks[3].data_ptr() + 2),
                 (base, base + 4 * 48001, 0, 0), (base, base + 4 * 48001, 65536, 0), (0, base, 1, 0)):
        with pytest.raises(pkg.Ft8Error):
            call(*args)
    torch.cuda.synchronize()
    assert all(bool(torch.all(m == 7)) for m in marks)   # refused: nothing written
    ctx.close()
    p = pkg.Pipe(0, depth=2)
    with pytest.raises(pkg.Ft8Error):
        p.set_finesync(2, -1)
    p.set_finesync(1, -1)
    p.close()


@pytest.fixture(scope="module")
def weak_slots(pkg):
    """48 device slots of 1-8 GFSK CQ and non-CQ messages at -23 ... -17 dB (noise 1.0) with their peaks."""
    rng = np.random.Generator(np.random.PCG64(0xF51))
    slots = []
    for s in range(48):
        sp = []
        for _ in range(1 + s % 8):
            to = "CQ" if rng.random() < 0.6 else synth.random_call(rng)
            sp.append((pkg.pack77_std(to, synth.random_call(rng), synth.random_grid(rng)), float(rng.uniform(100, 1500)),
                       float(0.5 + rng.uniform(-0.3, 0.3)), mp.amp_for(float(rng.uniform(-23, -17)))))
        slots.append(sp)
    first = np.cumsum([0] + [len(sp) for sp in slots]).astype(np.int32)
    ctx = pkg.Context(0)
    d_i, d_q = ctx.synth_slots(pkg.make_signals([it for sp in slots for it in sp], gfsk=True), first, 1.0, 0xF51)
    peak = torch.maximum(d_i.abs().amax(1), d_q.abs().amax(1)).contiguous()
    torch.cuda.synchronize()
    ctx.close()
    return d_i, d_q, peak


def outputs(ctx, n):
    w = ctx.workspace_ptrs()
    K = ctx.K
    g = lambda p, shp, t: torch.as_tensor(_Arr(p, shp, t), device=DEV).cpu().numpy()
    a, b = ctx.finesync_workspace_ptrs()
    return dict(ok=g(w["ok"], (n, K), "|u1"), ncand=g(w["ncand"], (n,), "<i4"), cand=g(w["cand"], (n, K * 8), "|u1"),
                status=g(w["status"], (n, K * 12), "|u1").reshape(n, K, 12), msg=g(w["msg"], (n, K * 28), "|u1").reshape(n, K, 28),
                fs=g(a, (n, K), "|u1") if a else None, hard=g(b, (n, K), "<i4") if b else None)


def test_only_stage_1_2_change_and_off_is_untouched(pkg, weak_slots):
    """Off: records, rows and launch counts as a context that never called set_finesync, and nothing allocated.  On: the candidate
    lists are the same, every row BP (or OSD, AP) decoded or left at stage 3 is byte-identical, and the others either stay as they
    were or become fine-sync decodes."""
    d_i, d_q, peak = weak_slots
    n = d_i.shape[0]
    fresh = pkg.Context(0)
    fresh.process_conditioned(d_i, d_q, peak)
    r0 = fresh.fetch_results(n)
    o0 = outputs(fresh, n)
    l0 = fresh.launches()
    assert fresh.finesync_workspace_ptrs() == (0, 0)
    used = []
    for c in (pkg.Context(0), pkg.Context(0)):
        if used:
            c.set_finesync(0, 30)
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        c.process_conditioned(d_i, d_q, peak)
        r2 = c.fetch_results(n)
        torch.cuda.synchronize()
        used.append(free0 - torch.cuda.mem_get_info()[0])
        off = c
    assert abs(used[1] - used[0]) <= (2 << 20), used
    assert off.launches() == l0 and off.finesync_workspace_ptrs() == (0, 0)
    mp.check_records(r2, r0, "off")
    for osd, ap in ((0, 0), (2, 1)):
        base = pkg.Context(0)
        base.set_osd(osd, -1)
        base.set_ap(ap, -1)
        base.process_conditioned(d_i, d_q, peak)
        ob = outputs(base, n)
        on = pkg.Context(0)
        on.set_osd(osd, -1)
        on.set_ap(ap, -1)
        on.set_finesync(1, -1)
        on.process_conditioned(d_i, d_q, peak)
        o1 = outputs(on, n)
        assert np.array_equal(ob["ncand"], o1["ncand"]) and np.array_equal(ob["cand"], o1["cand"])
        by_fs = 0
        for s in range(n):
            nc = int(ob["ncand"][s])
            for k in range(nc):
                same = all(np.array_equal(ob[key][s, k], o1[key][s, k]) for key in ("ok", "status", "msg"))
                if ob["ok"][s, k] or o1["fs"][s, k] != 2:
                    assert same and o1["fs"][s, k] != 2, (osd, s, k)
                else:
                    assert o1["ok"][s, k] == 1 and ob["ok"][s, k] == 0
                    by_fs += 1
        assert by_fs >= 1, (osd, by_fs)
        base.close()
        on.close()
    for c in (fresh, off):
        c.close()


def stage_with_fs(c, x_i, x_q, peak, osd):
    """test_gpu_multipass.stage on a context with fine sync on: waterfall -> find_sync -> ft8b200_decode (which runs OSD and AP when
    they are on) -> ft8b200_finesync on the pass's own samples, fine-sync decodes writing their word into plain."""
    mag = c.waterfall(x_i, x_q, peak)
    cand, ncand = c.find_sync(mag)
    ok, stg, status, msg, plain, llr = c.decode(mag, cand, ncand, want_plain=True, want_llr=True)
    fs, _, _, _ = c.finesync(x_i, x_q, cand, ncand, ok, stg, status, msg, plain)
    torch.cuda.synchronize()
    n = x_i.shape[0]
    R = dict(cand=cand.cpu().numpy().view(cand_dtype).reshape(n, c.K), ncand=ncand.cpu().numpy(), ok=ok.cpu().numpy(), status=status.cpu().numpy(),
             msg=msg.cpu().numpy().view(msg_dtype).reshape(n, c.K), plain=plain.cpu().numpy())
    FS.append((fs.cpu().numpy(), R))
    return R


FS = []


def fs_decodes_are_codewords():
    decoded = 0
    for fs, R in FS:
        for s, k in zip(*np.nonzero(fs == 2)):
            text = bytes(R["msg"][s, k]["text"]).decode().split()
            if len(text) == 3 and text[0] == "CQ":
                assert np.array_equal(R["plain"][s, k], ft8enc.encode174(ft8enc.pack_std(*text))), text
            decoded += 1
    return decoded


@pytest.mark.parametrize("osd,ap", [(0, 0), (2, 1)])
def test_conditioned_and_slots_compose(pkg, oracle, weak_slots, osd, ap, monkeypatch):
    """process_conditioned and process_slots at passes 1, 2 and 3 equal the composition of the stage-wise entries with fine sync after
    AP in every pass: pass-1 rows byte for byte and the records, which after pass 1 depend on every fine-sync decode's plain row
    having been subtracted."""
    d_i, d_q, peak = weak_slots
    n = d_i.shape[0]
    c_i, c_q = d_i.clone(), d_q.clone()
    cond = pkg.Context(0)
    cond.condition(c_i, c_q, peak.clone())
    cond.close()
    cfg = mp.cfg_of("default")
    monkeypatch.setattr(mp, "stage", stage_with_fs)
    ref = pkg.Context(0, **cfg)
    ref.set_osd(osd, -1)
    ref.set_ap(ap, -1)
    ref.set_finesync(1, -1)
    st = mp.new_stats()
    FS.clear()
    for passes in (1, 2, 3):
        for entry, (x_i, x_q, pk) in (("conditioned", (d_i, d_q, peak)), ("slots", (c_i, c_q, None))):
            if entry == "slots" and passes == 3:
                continue
            ctx = pkg.Context(0, **cfg)
            ctx.set_osd(osd, -1)
            ctx.set_ap(ap, -1)
            ctx.set_finesync(1, -1)
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
    assert fs_decodes_are_codewords() >= 3 and st["appended_in_pass2"] >= 1


def test_raw_entries_and_pipes(pkg, oracle, monkeypatch):
    """process_raw in 4 overlap groups and process_raw_streams at passes 2 with OSD 2 and AP equal the composition on the decimated
    slots; a pipe with and without an SM partition equals process_raw batch by batch."""
    sig, first = mp.fixture_items(pkg, 0x7E12, n_crowded=4, specials_first=True)
    sig["amp"] *= np.float32(1.2 * np.sqrt(2 * 900.0 * 2500 / 2.4e6) / np.sqrt(2 * 2500 / 3200.0))
    c0 = pkg.Context(0)
    raw = c0.synth_raw(sig, first, 30.0, 0x7E12)
    torch.cuda.synchronize()
    c0.close()
    n = raw.shape[0]
    cfg = mp.cfg_of("default")
    monkeypatch.setattr(mp, "stage", stage_with_fs)
    ref = pkg.Context(0)
    ref.set_osd(2, -1)
    ref.set_ap(1, -1)
    ref.set_finesync(1, -1)
    st = mp.new_stats()
    FS.clear()
    ctx = pkg.Context(0)
    ctx.set_osd(2, -1)
    ctx.set_ap(1, -1)
    ctx.set_finesync(1, -1)
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
        p.set_osd(2, -1)
        p.set_ap(1, -1)
        p.set_finesync(1, -1)
        p.set_passes(2)
        p.submit(raw[:4], 4, stride=raw.stride(0))
        with pytest.raises(pkg.Ft8Error):
            p.set_finesync(0, -1)   # EBUSY while a batch is in flight
        p.submit(raw[4:8], 4, stride=raw.stride(0))
        got = [p.collect(4) for _ in range(2)]
        p.close()
        for b in range(2):
            mp.check_records(got[b], want[b], ("pipe", back, b))


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


def test_dropin_environment_and_iq_files(pkg, oracle, weak_slots, tmp_path):
    d_i, d_q, peak = weak_slots
    hi = (d_i[:12] * (0.5 / peak[:12, None])).cpu().numpy()
    hq = (d_q[:12] * (0.5 / peak[:12, None])).cpu().numpy()
    np.savez(tmp_path / "slots.npz", i=hi, q=hq)
    script = tmp_path / "dropin.py"
    script.write_text(_DROPIN)
    run = lambda env: subprocess.run([sys.executable, str(script), ROOT, str(tmp_path / "slots.npz"), str(tmp_path / "out.npy")], env=env,
                                     capture_output=True, text=True, timeout=600)
    base = {k: v for k, v in os.environ.items() if not k.startswith("FT8B200_")}
    for bad in ({"FT8B200_FINESYNC": "2"}, {"FT8B200_FINESYNC": "x"}, {"FT8B200_FINESYNC": ""},
                {"FT8B200_FINESYNC": "1", "FT8B200_FINESYNC_MAX_HARD": "175"}):
        p = run(dict(base, **bad))
        assert p.returncode != 0 and "FT8B200_FINESYNC" in p.stderr, bad
    p = run(dict(base, FT8B200_FINESYNC="1"))
    assert p.returncode == 0, p.stderr[-2000:]
    got = np.load(tmp_path / "out.npy", allow_pickle=True)
    got_n = np.load(tmp_path / "out.npy.n.npy")
    ctx = pkg.Context(0)
    ctx.set_finesync(1, -1)
    for s in range(12):
        res, nres = ctx.process_slots_host(hi[s:s + 1], hq[s:s + 1])
        want = np.zeros(50, result_dtype)
        for k in range(int(nres[0])):
            if res[0][k]["call"]:
                want[k] = res[0][k]
        assert got_n[s] == nres[0] and got[s] == want.tobytes(), s
    # .iq recordings: readRawIQfile's normalisation, then the daemon path with fine sync
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
        ci, cq, _ = oracle.condition(inter[0::2].copy(), -inter[1::2], sr.SLOT)   # readRawIQfile's normalisation
        w, wn = ctx.process_slots_host(ci[None], cq[None])
        assert nres[s] == wn[0] and res[s].tobytes() == w[0].tobytes(), s
    ctx.close()


def test_shapes_and_batch_invariance(pkg, hand_slots):
    """Grids below the persistent cap (K = 4, 3 slots) and above it, more than 2 x SMs slots (300 copies of the hand slots): every
    slot's outputs equal those of the same slot run alone."""
    x, cands, stage0, ncand, _ = hand_slots
    ctx = pkg.Context(0, max_candidates=16)
    ctx.set_finesync(1, -1)
    alone = [run_stage(pkg, ctx, x[s:s + 1], cands[s:s + 1], stage0[s:s + 1], ncand[s:s + 1])[1] for s in range(8)]
    reps = 300 // 8 + 1
    idx = np.arange(8 * reps) % 8
    _, big = run_stage(pkg, ctx, x[idx], cands[idx], stage0[idx], ncand[idx])
    for r, s in enumerate(idx):
        for key in ("fs", "hard", "grid", "llr"):
            assert np.array_equal(big[key][r], alone[s][key][0], equal_nan=key == "llr"), (r, s, key)
        dec = big["fs"][r] == 2
        for key in ("ok", "stage", "status", "msg", "plain"):
            assert np.array_equal(big[key][r][dec], alone[s][key][0][dec]), (r, s, key)
    ctx.close()
    small = pkg.Context(0, max_candidates=4)
    small.set_finesync(1, -1)
    _, o = run_stage(pkg, small, x[:3], cands[:3, :4], stage0[:3, :4], np.minimum(ncand[:3], 4))
    for s in range(3):
        for key in ("fs", "hard", "grid"):
            assert np.array_equal(o[key][s], alone[s][key][0][:4]), (s, key)
    small.close()
