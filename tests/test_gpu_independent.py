"""The kernels against independent references (tests/ref64.py): float64 DFTs and sample loops, exact integer sync scores,
the LDPC checks of the source text, a fresh CRC-14 and the transmitted messages themselves.

The rest of the GPU suite compares the kernels bit for bit with the C restatement in oracle/, which shares
csrc/ft8_tables.h with them; those tests cannot see a mistake that both make.  These tests can.  They pin what the
restatement cannot vouch for on its own: FT4 sync, demapper and descrambling, the 12 kHz monitor at other rates and
oversampling (including kiss_fft's generic radix-7 stage), sync scores on every geometry, LLRs, the synthesiser's
symbols and waveforms.  They deliberately do not re-implement the heap's tie order, belief propagation's iteration-by-
iteration bits or unpack77's text: the assertions are chosen so that a wrong score, range, threshold, bit or check fails
without them.

Bars are the north-star tolerances: waterfall cells +-1 LSB on at most 0.01 % of the cells, decimator floats within
1e-5 of the row's largest output, LLRs within 2e-6 of the candidate's largest LLR, GFSK within 2e-3 of the amplitude.
The worst deviation each test saw is printed (pytest -s)."""

import numpy as np
import pytest

import ref64
from conftest import golden
from oracle.pyoracle import cand_dtype, status_dtype
from tools import ft8enc, synth

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

WINDOW = golden("kat")["window"]


def dev():
    return torch.device("cuda:0")


def view(t, dt):
    a = t.cpu().numpy()
    return a.view(dt).reshape(a.shape[:-1])


def report(what, value):
    print(f"\n[independent] {what}: {value}")


def cell_diff(got, ref, what):
    """The waterfall bar: every cell within one step; at most 0.01 % of the cells differ among those a float32 FFT can
    resolve (ref64.RESOLVABLE).  ref = (cells, resolvable mask).  -> (differing resolvable cells, differing cells)."""
    ref, ok = ref
    d = got.astype(np.int64) - ref.astype(np.int64)
    n = int((d[ok] != 0).sum())
    assert np.abs(d).max(initial=0) <= 1, f"{what}: a cell is off by {int(np.abs(d).max())} steps"
    assert n <= ref.size // 10000, f"{what}: {n} of {ref.size} cells differ"
    return n, int((d != 0).sum())


# ------------------------------------------------------------------------------------------- 1. decimator vs the sample loop
def check_decimator_row(gi, gq, gy2, cnt, peak, ref, first=0):
    y2, fi, fq = ref
    n = int(cnt)
    assert np.array_equal(gy2[:n].astype(np.int64), y2[first:first + n]), "comb outputs must be exact"
    worst = 0.0
    for g, r in ((gi, fi), (gq, fq)):
        r = r[first:first + n]
        scale = np.abs(r).max(initial=0.0)
        err = np.abs(g[:n].astype(np.float64) - r).max(initial=0.0)
        assert err <= 1e-5 * scale, (err, scale)
        worst = max(worst, err / scale if scale else 0.0)
        assert not g[n:].any(), "the tail of the 48 000-sample buffer is zero"
    assert float(peak) == float(max(np.abs(gi[:n]).max(initial=0), np.abs(gq[:n]).max(initial=0)))
    return worst


def test_decimator_vs_sample_loop(pkg, ctx):
    """Three rows of about one second with runs of 0x00, 0x80 and 0xFF (the int8 negate wraps at 0x00), and one full
    72 MB slot (one message in noise) made on the device."""
    rng = np.random.default_rng(2024)
    nbytes = 2 * 751 * 3200 + 608      # a multiple of 16 with a ragged last block
    iq = rng.integers(0, 256, size=(3, nbytes), dtype=np.uint8)
    for r, v in enumerate((0x00, 0x80, 0xFF)):
        for s in range(0, nbytes, 200_000):
            iq[r, s:s + 20_000 + 1000 * r] = v
    iq[1, ::2][::7] = 0x00
    d_i, d_q, cnt, peak, y2 = ctx.decimate(torch.from_numpy(iq).to(dev()), 3, nbytes, want_y2=True)
    worst = 0.0
    for r in range(3):
        ref = ref64.decimate(iq[r])
        assert int(cnt[r]) == ref[0].shape[0] == nbytes // 2 // 751
        worst = max(worst, check_decimator_row(d_i[r].cpu().numpy(), d_q[r].cpu().numpy(), y2[r].cpu().numpy(), cnt[r], peak[r], ref))
    g = pkg.make_signals([(pkg.pack77_std("CQ", "K1JT", "FN20"), 900.0, 0.4, 25.0)])
    raw = ctx.synth_raw(g, [0, 1], 30.0, 77)
    d_i, d_q, cnt, peak, y2 = ctx.decimate(raw, 1, 72_000_000, stride=raw.stride(0), want_y2=True)
    host = raw[0, :72_000_000].cpu().numpy()
    ref = ref64.decimate(host)
    assert int(cnt[0]) == 47936 == ref[0].shape[0]
    worst = max(worst, check_decimator_row(d_i[0].cpu().numpy(), d_q[0].cpu().numpy(), y2[0].cpu().numpy(), cnt[0], peak[0], ref))
    report("decimator worst |gpu - ref| / max|ref|", worst)


def test_decimate_streams_vs_one_continuous_loop(ctx):
    """Receivers x consecutive slots: row (r, s) holds exactly the outputs of ONE continuous sample loop over receiver r whose
    instant 750 + 751 k falls into slot s, with the real preceding samples as filter history."""
    n_streams, slots, bps = 2, 6, 2 * 751 * 330 + 804   # 402 samples past a whole number of outputs per slot
    rng = np.random.default_rng(5)
    iq = rng.integers(0, 256, size=(n_streams, slots * bps), dtype=np.uint8)
    iq[1, : bps // 2] = 0x80
    d_i, d_q, cnt, peak, y2 = ctx.decimate_streams(torch.from_numpy(iq).to(dev()), n_streams, slots, bps, want_y2=True)
    rows = ref64.slot_rows(bps // 2, slots)
    assert len({c for _, c in rows}) > 1, "the decimation phase drifts across these slots"
    for r in range(n_streams):
        ref = ref64.decimate(iq[r])
        for s, (first, count) in enumerate(rows):
            k = r * slots + s
            assert int(cnt[k]) == count, (r, s)
            check_decimator_row(d_i[k].cpu().numpy(), d_q[k].cpu().numpy(), y2[k].cpu().numpy(), cnt[k], peak[k], ref, first)
    # the full-size slot: 47 936 outputs per 36 000 000 samples, 47 937 in every 12th slot (36e6 mod 751 = 64)
    full = [c for _, c in ref64.slot_rows(36_000_000, 24)]
    assert [s for s, c in enumerate(full) if c == 47937] == [11, 23] and set(full) == {47936, 47937}


# ------------------------------------------------------------------------------------------- 2. daemon waterfall vs a float64 DFT
def _tone(f_hz, amp=0.4, n=48000, fs=3200.0):
    t = np.arange(n) / fs
    return (amp * np.cos(2 * np.pi * f_hz * t)).astype(np.float32), (amp * np.sin(2 * np.pi * f_hz * t)).astype(np.float32)


def _cond(i_s, q_s):
    s = np.float32(0.5 / max(np.abs(i_s).max(), np.abs(q_s).max(), 1e-24))
    return i_s * s, q_s * s


def _sig(f0, t0, snr, msg=("CQ", "K1JT", "FN20")):
    return (ft8enc.tones(ft8enc.pack_std(*msg)), f0, t0, snr)


@pytest.fixture(scope="module")
def daemon_slots():
    """(name, I, Q) conditioned slots, and (name, I, Q, peak) unconditioned ones."""
    z = np.zeros(48000, np.float32)
    cond = [("crowded", *_cond(*synth.crowded_band(ft8enc, 40, 17)[:2])),
            ("one signal", *_cond(*synth.slot_f32([_sig(700.0, 0.5, -10.0)], 7))),
            ("noise", *_cond(*synth.slot_f32([], 11))),
            ("silence", z, z),
            ("tone on a bin centre", *_tone(100 * 3.125)),
            ("tone between bins", *_tone(100.5 * 3.125)),
            ("DC", np.full(48000, 0.3, np.float32), np.full(48000, -0.2, np.float32)),
            ("band edges", *_cond(*synth.slot_f32([_sig(3.0, 0.2, 0.0), _sig(1553.0, 1.0, 0.0, ("K1ABC", "W9XYZ", "-15"))], 13))),
            ("tone at the top bin", *_tone(1597.0))]
    raw = []
    i_s, q_s = synth.slot_f32([_sig(400.0, 0.3, -5.0)], 21)
    raw.append(("peak 3.7e-3", i_s * np.float32(3.7e-3), q_s * np.float32(3.7e-3), float(max(np.abs(i_s).max(), np.abs(q_s).max()) * np.float32(3.7e-3))))
    i_s, q_s = synth.slot_f32([_sig(900.0, 0.8, 10.0), _sig(1200.0, 0.1, 10.0)], 22)
    raw.append(("understated peak: cells clamp at 255", i_s * np.float32(40.0), q_s * np.float32(40.0), 0.5))
    return cond, raw


def test_daemon_waterfall_vs_dft(ctx, daemon_slots):
    cond, raw = daemon_slots
    worst = {}
    hi = np.stack([s[1] for s in cond]); hq = np.stack([s[2] for s in cond])
    mag = ctx.waterfall(torch.from_numpy(hi).to(dev()), torch.from_numpy(hq).to(dev())).cpu().numpy()
    for s, (name, i_s, q_s) in enumerate(cond):
        worst[name] = cell_diff(mag[s], ref64.daemon_waterfall(i_s, q_s, WINDOW, resolvable=True), name)
    hi = np.stack([s[1] for s in raw]); hq = np.stack([s[2] for s in raw])
    peak = torch.tensor([s[3] for s in raw], dtype=torch.float32, device=dev())
    mag = ctx.waterfall(torch.from_numpy(hi).to(dev()), torch.from_numpy(hq).to(dev()), peak).cpu().numpy()
    for s, (name, i_s, q_s, pk) in enumerate(raw):
        ref = ref64.daemon_waterfall(i_s, q_s, WINDOW, peak=np.float32(pk), resolvable=True)
        worst[name] = cell_diff(mag[s], ref, name)
    assert (mag[1] == 255).sum() > 1000, "the loud slot reaches the top of the quantiser"
    assert not ref64.daemon_waterfall(*cond[3][1:], WINDOW).any()
    report("daemon waterfall (differing resolvable cells, differing cells) per slot, of 94 208", worst)


# ------------------------------------------------------------------------------------------- 3. monitor waterfall vs float64 rfft
def _recordings(rate, protocol, seed):
    """Noise with signals, a clipped full-scale s16 square wave, and silence."""
    n = int(rate * (15.0 if protocol == 1 else 7.5))
    rng = np.random.default_rng(seed)
    t = np.arange(n) / rate
    a = 0.05 * rng.standard_normal(n)
    for f, t0, amp in ((0.07 * rate, 0.4, 0.2), (0.19 * rate, 1.3, 0.1), (0.31 * rate + 3.3, 0.0, 0.05)):
        a += amp * np.cos(2 * np.pi * f * t + 0.3) * (t >= t0)
    sq = np.clip(np.sign(np.sin(2 * np.pi * 441.0 * t + 0.1)) * 40000, -32768, 32767).astype(np.int16).astype(np.float32) / np.float32(32768.0)
    return np.stack([a.astype(np.float32), sq, np.zeros(n, np.float32)])


@pytest.mark.parametrize("rate,tosr,fosr,proto", [(12000, 2, 2, 1), (12000, 2, 2, 0), (12000, 1, 1, 1), (8000, 2, 2, 1), (8000, 1, 2, 0),
                                                  (11025, 2, 2, 1), (11025, 1, 1, 1)])
def test_monitor_waterfall_vs_rfft(ctx, rate, tosr, fosr, proto):
    """12 kHz FT8 (3840-point frames) and FT4 (1152), 8 kHz, and 11 025 Hz whose frames have a factor 7 (kiss_fft's generic
    butterfly); time and frequency oversampling 1 and 2."""
    audio = _recordings(rate, proto, rate + tosr + 10 * fosr + proto)
    mag, nb = ctx.monitor_waterfall(torch.from_numpy(audio).to(dev()), rate, tosr, fosr, proto)
    mag = mag.cpu().numpy()
    worst = []
    for s in range(audio.shape[0]):
        ref, rnb, _, ok = ref64.monitor_waterfall(audio[s], rate, tosr, fosr, proto, resolvable=True)
        assert nb == rnb
        worst.append(cell_diff(mag[s][: ref.size], (ref, ok), f"recording {s}"))
    report(f"monitor {rate} Hz tosr {tosr} fosr {fosr} proto {proto}: (differing resolvable cells, differing cells) per recording, of {mag.shape[1]}", worst)


@pytest.mark.parametrize("rate", [12000, 11025])
def test_monitor_max_mag_vs_float64(pkg, rate):
    """monitor_process() block by block: max_mag within 0.01 dB of the float64 maximum of 10 log10(x)."""
    audio = _recordings(rate, 1, 3)[0]
    mon = pkg.Monitor(rate, 2, 2, 1)
    bs = mon.me.block_size
    for o in range(0, audio.size - bs + 1, bs):
        mon.process(audio[o:o + bs])
    ref, nb, max_db, ok = ref64.monitor_waterfall(audio, rate, 2, 2, 1, resolvable=True)
    assert mon.me.wf.num_blocks == nb
    cell_diff(mon.mag(), (ref, ok), "drop-in monitor")
    assert abs(float(mon.me.max_mag) - max_db) <= 0.01, (float(mon.me.max_mag), max_db)
    report(f"monitor max_mag at {rate} Hz: |gpu - float64| dB", abs(float(mon.me.max_mag) - max_db))
    mon.close()


# ------------------------------------------------------------------------------------------- 4. sync scores vs exact integers
GEOMETRIES = {"daemon": (dict(num_blocks=92, num_bins=256, time_osr=2, freq_osr=2), 1),
              "ft8_12k": (dict(num_blocks=93, num_bins=960, time_osr=2, freq_osr=2), 1),
              "ft4": (dict(num_blocks=156, num_bins=288, time_osr=2, freq_osr=2), 0),
              "odd": (dict(num_blocks=60, num_bins=78, time_osr=1, freq_osr=3), 1),
              "narrow": (dict(num_blocks=95, num_bins=8, time_osr=1, freq_osr=1), 1)}


def _cells(dims):
    return dims["num_blocks"] * dims["time_osr"] * dims["freq_osr"] * dims["num_bins"]


def ft4_audio(pkg, ctx, seed, n=6):
    """FT4 recording made by the device synthesiser: n CQ messages, (texts, f0s, t0s)."""
    rng = np.random.default_rng(seed)
    items, texts = [], []
    f0s = 300.0 + 330.0 * np.arange(n) + rng.uniform(0, 40, n)
    t0s = rng.uniform(0.2, 1.0, n)
    for k in range(n):
        _, de, ex = synth.random_message(rng)
        ex = synth.random_grid(rng)
        items.append((pkg.pack77_std("CQ", de, ex), float(f0s[k]), float(t0s[k]), 0.1))
        texts.append(f"CQ {de} {ex}")
    d_a = ctx.synth_audio(pkg.make_signals(items), [0, n], 0, 0.05, seed, n_samples=90_000)
    return d_a, texts, f0s.astype(np.float32), t0s.astype(np.float32)


@pytest.fixture(scope="module")
def waterfalls(pkg, ctx, daemon_slots):
    """Per geometry: uint8 [n, cells] = real (where the geometry has a source), random bytes, ties everywhere, constant."""
    rng = np.random.default_rng(99)
    cond, _ = daemon_slots
    out = {}
    for name, (dims, proto) in GEOMETRIES.items():
        cells = _cells(dims)
        mags = [rng.integers(0, 256, cells, dtype=np.uint8), (rng.integers(0, 2, cells) * 255).astype(np.uint8), np.full(cells, 77, np.uint8)]
        if name == "daemon":
            hi = np.stack([cond[0][1], cond[1][1]]); hq = np.stack([cond[0][2], cond[1][2]])
            mags = list(ctx.waterfall(torch.from_numpy(hi).to(dev()), torch.from_numpy(hq).to(dev())).cpu().numpy()) + mags
        elif name == "ft8_12k":
            sigs = [(ft8enc.tones(ft8enc.pack_std("CQ", "K1JT", "FN20")), 1200.0, 0.5, 0.1), (ft8enc.tones(ft8enc.pack_std("CQ", "W9XYZ", "EN37")), 2100.0, 1.1, 0.05)]
            m, nb = ctx.monitor_waterfall(torch.from_numpy(synth.audio_12k(sigs, 3)[None]).to(dev()))
            mags = [m[0].cpu().numpy()[:cells]] + mags
        elif name == "ft4":
            d_a, _, _, _ = ft4_audio(pkg, ctx, 11)
            m, nb = ctx.monitor_waterfall(d_a, protocol=0)
            assert nb == dims["num_blocks"]
            mags = [m[0].cpu().numpy()[:cells]] + mags
        out[name] = np.stack(mags)
    return out


@pytest.mark.parametrize("geometry", list(GEOMETRIES))
def test_sync_scores_vs_integer_restatement(pkg, waterfalls, geometry):
    """Every GPU candidate's score is the exact score at its position; positions are distinct and scores do not increase
    down the list; ncand = min(K, positions with score >= min_score); the GPU's scores are the top ncand scores."""
    dims, proto = GEOMETRIES[geometry]
    mags = waterfalls[geometry]
    every = [ref64.sync_scores(m, protocol=proto, **dims) for m in mags]       # [ts, fs, 36, nfo]
    nfo = dims["num_bins"] - 7
    d_mag = torch.from_numpy(mags).to(dev())
    for K in (1, 7, 120, 500):
        for min_score in (0, 10):
            c = pkg.Context(0, max_candidates=K, max_messages=50, min_score=min_score)
            c.set_protocol(proto)
            cand, ncand = c.find_sync(d_mag, **dims)
            g = view(cand, cand_dtype)
            for s in range(mags.shape[0]):
                n = int(ncand[s])
                sc = every[s].reshape(-1)
                assert n == min(K, int((sc >= min_score).sum())), (K, min_score, s)
                cd = g[s, :n]
                assert ((cd["time_offset"] >= -12) & (cd["time_offset"] < 24) & (cd["freq_offset"] >= 0) & (cd["freq_offset"] < nfo)).all()
                assert ((cd["time_sub"] < dims["time_osr"]) & (cd["freq_sub"] < dims["freq_osr"])).all()
                pos = ((cd["time_sub"].astype(np.int64) * dims["freq_osr"] + cd["freq_sub"]) * 36 + cd["time_offset"] + 12) * nfo + cd["freq_offset"]
                assert np.array_equal(cd["score"], sc[pos]), (K, min_score, s)
                assert np.unique(pos).size == n
                assert (np.diff(cd["score"].astype(np.int64)) <= 0).all()
                assert np.array_equal(cd["score"], np.sort(sc)[::-1][:n])
            c.close()


# ------------------------------------------------------------------------------------------- 5./6. LLRs, decodes vs the code
def _llr_check(mags, cands, ncand, llr, dims, proto):
    worst, nan_seen = 0.0, 0
    for s in range(mags.shape[0]):
        for k in range(int(ncand[s])):
            ref, var = ref64.llrs(mags[s], cands[s, k], protocol=proto, **dims)
            g = llr[s, k]
            assert np.array_equal(np.isnan(g), np.isnan(ref)), (s, k)
            if var == 0:
                assert np.isnan(g).all()
                nan_seen += 1
                continue
            scale = np.abs(ref).max()
            err = np.abs(g.astype(np.float64) - ref).max()
            assert err <= 2e-6 * scale, (s, k, err, scale)
            worst = max(worst, err / scale)
    return worst, nan_seen


def _check_decodes(ok, stage, status, plain, ncand, n_slots, proto, msg_bits=None):
    n_ok = 0
    st = view(status, status_dtype)
    for s in range(n_slots):
        for k in range(int(ncand[s])):
            if not int(ok[s, k]):
                continue
            bits = plain[s, k]
            assert ref64.checks_satisfied(bits), (s, k)
            assert ref64.crc_ok(bits), (s, k)
            assert int(st[s, k]["ldpc_errors"]) == 0 and int(stage[s, k]) == 4
            n_ok += 1
    return n_ok


@pytest.fixture(params=[0, 1], ids=["bp_nodes", "bp_edges"])
def bp_variant(request, pkg):
    pkg.set_decode_variant(request.param)
    yield request.param
    pkg.set_decode_variant(0)


@pytest.mark.parametrize("geometry", ["daemon", "ft8_12k", "ft4"])
def test_llrs_and_decodes_vs_independent_references(pkg, waterfalls, geometry, bp_variant):
    """Candidates from find_sync on real and random waterfalls: LLRs against the float64 demapper; every decoded word (ok = 1)
    satisfies all 83 checks of the source text and carries the CRC-14 of its 77 message bits."""
    dims, proto = GEOMETRIES[geometry]
    mags = waterfalls[geometry]
    c = pkg.Context(0, max_candidates=120, max_messages=50, min_score=10)
    c.set_protocol(proto)
    d_mag = torch.from_numpy(mags).to(dev())
    cand, ncand = c.find_sync(d_mag, **dims)
    ok, stage, status, msg, plain, llr = c.decode(d_mag, cand, ncand, want_plain=True, want_llr=True, **dims)
    ncand = ncand.cpu().numpy()
    worst, _ = _llr_check(mags, view(cand, cand_dtype), ncand, llr.cpu().numpy(), dims, proto)
    n_ok = _check_decodes(ok.cpu().numpy(), stage.cpu().numpy(), status, plain.cpu().numpy(), ncand, mags.shape[0], proto)
    assert n_ok >= (1 if geometry == "ft8_12k" else 3)
    report(f"LLR worst relative error, {geometry}, {n_ok} decodes checked", worst)
    c.close()


def test_llrs_on_degenerate_waterfalls(ctx, waterfalls):
    """Hand-placed candidates over both time edges on a flat waterfall (var = 0: NaN), one flat except a row, and a real one."""
    dims = GEOMETRIES["daemon"][0]
    flat = np.full(94208, 77, np.uint8)
    one_row = flat.copy().reshape(92, 2, 2, 256)
    one_row[40] = np.random.default_rng(4).integers(0, 256, size=(2, 2, 256), dtype=np.uint8)
    mags = np.stack([flat, one_row.reshape(-1), waterfalls["daemon"][0]])
    picks = [(20, 0, 10, 0, 0), (20, -12, 100, 1, 1), (20, 23, 248, 1, 0), (20, 5, 0, 0, 1), (20, -7, 33, 0, 0), (20, 17, 200, 1, 1)]
    cands = np.zeros((3, ctx.K), cand_dtype)
    cands[:, : len(picks)] = np.array(picks, cand_dtype)
    ncand = np.full(3, len(picks), np.int32)
    _, _, _, _, _, llr = ctx.decode(torch.from_numpy(mags).to(dev()), torch.from_numpy(cands.view(np.uint8).reshape(3, ctx.K, 8)).to(dev()),
                                    torch.from_numpy(ncand).to(dev()), want_llr=True)
    worst, nan_seen = _llr_check(mags, cands, ncand, llr.cpu().numpy(), dims, 1)
    assert nan_seen >= len(picks), "every candidate on the flat waterfall has var = 0"
    report("LLR worst relative error, hand-placed candidates", worst)


# ------------------------------------------------------------------------------------------- 7. end to end vs the transmitted messages
def _cq_signals(pkg, rng, n, f_lo, f_hi, t_lo, t_hi, amp, gfsk=False):
    """n CQ messages at distinct calls, f0 at least 60 Hz apart (an FT8 signal is 50 Hz wide)."""
    edges = np.linspace(f_lo, f_hi, n + 1)
    items, truth = [], {}
    while len(items) < n:
        _, de, _ = synth.random_message(rng)
        if de in truth or len(de) > 6:
            continue
        k = len(items)
        f0 = float(rng.uniform(edges[k], edges[k + 1] - 60.0))
        grid = synth.random_grid(rng)
        items.append((pkg.pack77_std("CQ", de, grid), f0, float(rng.uniform(t_lo, t_hi)), amp))
        truth[de] = (grid, f0)
    return pkg.make_signals(items, gfsk=gfsk), truth


def _check_spots(res, nres, truth):
    got = {}
    for r in res[: int(nres)]:
        if r["call"]:
            got[r["call"].decode()] = (r["loc"].decode(), int(r["freq"]))
    assert set(got) == set(truth), (sorted(got), sorted(truth))
    for call, (loc, f) in got.items():
        assert loc == truth[call][0]
        assert abs(f - truth[call][1]) <= 6.25, (call, f, truth[call][1])


def test_raw_slots_decode_the_transmitted_messages(pkg, ctx):
    rng = np.random.default_rng(41)
    sigs, truths, first = [], [], [0]
    for _ in range(2):
        g, t = _cq_signals(pkg, rng, 4, 200.0, 1500.0, 0.2, 1.2, 25.0)
        sigs.append(g); truths.append(t); first.append(first[-1] + g.size)
    raw = ctx.synth_raw(np.concatenate(sigs), first, 30.0, 3)
    ctx.process_raw(raw, 2, stride=raw.stride(0))
    res, nres = ctx.fetch_results(2)
    for s in range(2):
        _check_spots(res[s], nres[s], truths[s])


def test_float_slots_decode_the_transmitted_messages(pkg, ctx):
    rng = np.random.default_rng(42)
    n_slots = 64
    sigs, truths, first = [], [], [0]
    for s in range(n_slots):
        g, t = _cq_signals(pkg, rng, 3, 150.0, 1500.0, 0.2, 1.5, 0.5, gfsk=bool(s & 1))
        sigs.append(g); truths.append(t); first.append(first[-1] + g.size)
    d_i, d_q = ctx.synth_slots(np.concatenate(sigs), first, 1.0, 9)
    peak = torch.maximum(d_i.abs().amax(1), d_q.abs().amax(1))
    ctx.process_conditioned(d_i, d_q, peak)
    res, nres = ctx.fetch_results(n_slots)
    for s in range(n_slots):
        _check_spots(res[s], nres[s], truths[s])


@pytest.mark.parametrize("proto", [1, 0], ids=["ft8", "ft4"])
def test_12k_recordings_decode_the_transmitted_messages(pkg, ctx, proto):
    """decode_ft8's chain on recordings made by the synthesiser: the message set, frequency within one tone spacing, and
    time within half a symbol of t0 + one symbol period.  (decode_ft8 reports the block whose frame -- two blocks long, ending
    half a block into the next symbol -- is centred on the first symbol, so its times run one symbol behind the signal start.)"""
    period, spacing = (0.16, 6.25) if proto == 1 else (0.048, 1 / 0.048)
    rng = np.random.default_rng(43 + proto)
    recs, truths = [], []
    for _ in range(3):
        if proto == 1:
            g, t = _cq_signals(pkg, rng, 5, 300.0, 2700.0, 0.2, 1.2, 0.1)
        else:
            g, t = _cq_signals(pkg, rng, 5, 300.0, 2700.0, 0.2, 1.0, 0.1)
            for k in range(g.size):            # FT4 signals are 83 Hz wide
                g[k]["f0_hz"] = 300.0 + 450.0 * k + float(rng.uniform(0, 50))
            t = {de: (v[0], float(g[k]["f0_hz"])) for k, (de, v) in enumerate(t.items())}
        recs.append(g); truths.append((t, g))
    first = np.cumsum([0] + [g.size for g in recs])
    d_a = ctx.synth_audio(np.concatenate(recs), first, proto, 0.05, 7, n_samples=180_000 if proto == 1 else 90_000)
    outs = pkg.decode_audio(ctx, d_a, 12000, proto)
    worst_t = 0.0
    for (t, g), out in zip(truths, outs):
        want = {f"CQ {de} {v[0]}": k for k, (de, v) in enumerate(t.items())}
        got = {r["text"].decode(): r for r in out}
        assert set(got) == set(want), (sorted(got), sorted(want))
        for text, r in got.items():
            k = want[text]
            assert abs(float(r["freq_hz"]) - float(g[k]["f0_hz"])) <= spacing
            dt = float(r["time_sec"]) - (float(g[k]["t0_sec"]) + period)
            assert abs(dt) <= period / 2, (text, float(r["time_sec"]), float(g[k]["t0_sec"]))
            worst_t = max(worst_t, abs(dt) / period)
    report(f"12 kHz proto {proto}: worst |time - (t0 + symbol)| in symbols", worst_t)


# ------------------------------------------------------------------------------------------- 8. synthesiser vs float64 FSK/GFSK
def test_encode_tones_vs_protocol(pkg, ctx):
    """Costas symbols at their places; Gray-decoding the data symbols gives a codeword of the source text's checks with the
    CRC of its message bits, whose message bits are the payload (FT4: after descrambling)."""
    rng = np.random.default_rng(17)
    payloads = np.stack([np.frombuffer(pkg.pack77_std(*synth.random_message(rng)), np.uint8) for _ in range(100)])
    for proto in (1, 0):
        tones = ctx.encode_tones(payloads, proto)
        assert tones.shape[1] == (79 if proto == 1 else 105)
        for k in range(payloads.shape[0]):
            t = tones[k]
            for pos, tone in ref64.costas_positions(proto).items():
                assert t[pos] == tone, (proto, k, pos)
            if proto == 0:
                assert t[0] == 0 and t[104] == 0
            bits = ref64.bits_from_tones(t, proto)
            assert ref64.checks_satisfied(bits) and ref64.crc_ok(bits), (proto, k)
            msg = ref64.descramble77(bits) if proto == 0 else np.packbits(np.r_[bits[:77], np.zeros(3, np.int64)].astype(np.uint8)).tobytes()
            assert msg == payloads[k].tobytes(), (proto, k)


def test_fsk_symbols_peak_at_their_tones(pkg, ctx):
    """Plain FSK, no noise: the float64 DFT of each 512-sample symbol is largest at f0 + 6.25 tone."""
    rng = np.random.default_rng(5)
    items = [(pkg.pack77_std(*synth.random_message(rng)), float(f0), 0.25, 0.3) for f0 in (201.3, 777.0)]
    g = pkg.make_signals(items)
    d_i, d_q = ctx.synth_slots(g, [0, 1, 2], 0.0, 1)
    tones = ctx.encode_tones(np.stack([np.frombuffer(x[0], np.uint8) for x in items]), 1)
    x = (d_i.cpu().numpy().astype(np.float64) + 1j * d_q.cpu().numpy().astype(np.float64))
    n = np.arange(512)
    for s, (_, f0, t0, _) in enumerate(items):
        s0 = int(round(t0 * 3200))
        basis = np.exp(-2j * np.pi * (f0 + 6.25 * np.arange(8))[:, None] * n[None, :] / 3200.0)
        for k in range(79):
            seg = x[s, s0 + 512 * k: s0 + 512 * (k + 1)]
            assert int(np.argmax(np.abs(basis @ seg))) == tones[s, k], (s, k)


@pytest.mark.parametrize("form", ["slots_ft8", "audio_ft8", "audio_ft4"])
def test_gfsk_vs_continuous_float64(pkg, ctx, form):
    """GFSK (reserved[0] = 1) against the continuous float64 form: erf pulse with BT 2 (FT8) / 1 (FT4), first and last symbol
    extended, raised-cosine ramps over 1/8 symbol.  Phase starts at 0 at round(t0 fs)."""
    rng = np.random.default_rng(61)
    proto = 0 if form == "audio_ft4" else 1
    fs, L, spacing, bt = (3200.0, 512, 6.25, 2.0) if form == "slots_ft8" else (12000.0, 1920, 6.25, 2.0) if proto == 1 else (12000.0, 576, 1 / 0.048, 1.0)
    amp = 0.37
    items = [(pkg.pack77_std(*synth.random_message(rng)), float(rng.uniform(300, 1300)), float(rng.uniform(0.1, 0.9)), amp) for _ in range(3)]
    g = pkg.make_signals(items, gfsk=True)
    first = [0, 1, 2, 3]
    if form == "slots_ft8":
        d_i, d_q = ctx.synth_slots(g, first, 0.0, 1)
        got = d_i.cpu().numpy().astype(np.float64) + 1j * d_q.cpu().numpy().astype(np.float64)
    else:
        got = ctx.synth_audio(g, first, proto, 0.0, 1, n_samples=180_000 if proto == 1 else 90_000).cpu().numpy().astype(np.float64)
    tones = ctx.encode_tones(np.stack([np.frombuffer(x[0], np.uint8) for x in items]), proto)
    worst = 0.0
    for s in range(3):
        f0, t0 = float(np.float32(items[s][1])), float(np.float32(items[s][2]))
        phase, env = ref64.gfsk_phase(tones[s], L, fs, f0, spacing, bt)
        s0 = int(round(t0 * fs))
        want = np.zeros(got.shape[1], got.dtype)
        seg = amp * env * (np.exp(1j * phase) if form == "slots_ft8" else np.cos(phase))
        end = min(got.shape[1], s0 + seg.size)
        want[s0:end] = seg[: end - s0]
        err = np.abs(got[s] - want).max() / amp
        assert err <= 2e-3, (form, s, err)
        worst = max(worst, err)
    report(f"GFSK {form}: worst |gpu - float64| / amplitude", worst)
