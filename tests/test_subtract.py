"""The float64 definition of signal subtraction (tests/subtract_ref.py) on noiseless GFSK from the synthesiser's CPU twin
(oracle/ft8_oracle_synth.c), and its window and tie rules on hand-made inputs.  No GPU needed."""
import numpy as np
import pytest

import subtract_ref as sr
from ref64 import bits_from_tones

SIG = np.dtype([("payload", "u1", 10), ("reserved", "u1", 2), ("f0_hz", "<f4"), ("t0_sec", "<f4"), ("amp", "<f4")])


def gfsk_slot(oracle, items, noise=0.0, seed=1):
    """items: (call_to, call_de, extra, f0_hz, t0_sec, amp) -> (complex slot, [codeword per item])."""
    sig = np.zeros(len(items), SIG)
    cws = []
    for k, (to, de, ex, f0, t0, amp) in enumerate(items):
        p = oracle.pack_std(to, de, ex)
        sig[k]["payload"] = np.frombuffer(p, np.uint8)
        sig[k]["reserved"][0] = 1
        sig[k]["f0_hz"], sig[k]["t0_sec"], sig[k]["amp"] = f0, t0, amp
        cws.append(bits_from_tones(oracle.tones(p)))
    i, q = oracle.synth_float(1, False, sig, noise, seed, 0, sr.SLOT)
    return i.astype(np.float64) + 1j * q.astype(np.float64), cws


def strongest_candidate(oracle, x):
    i, q, _ = oracle.condition(x.real.astype(np.float32), x.imag.astype(np.float32), sr.SLOT)
    return oracle.find_sync(oracle.waterfall(i, q))[0]


@pytest.mark.parametrize("f0,t0", [(703.3, 0.537), (1211.0, 0.47), (350.7, 1.02)])
def test_removes_a_noiseless_signal(oracle, f0, t0):
    x, (cw,) = gfsk_slot(oracle, [("CQ", "K1JT", "FN20", f0, t0, 1.0)])
    cand = strongest_candidate(oracle, x)
    s0, f_nom = sr.nominal(cand)
    true_start = int(np.float32(t0) * 3200.0 + 0.5)
    assert abs(true_start - s0) <= 136 and abs(np.float32(f0) - f_nom) <= 1.5625 + 1e-6   # within reach of the grid
    y, [(dt, df)] = sr.subtract(x, [(cand, cw)])
    assert s0 + dt == true_start
    assert abs(f_nom + df * sr.DF_STEP - float(np.float32(f0))) <= sr.DF_STEP
    span = slice(max(true_start, 0), min(true_start + sr.SPAN, sr.SLOT))
    e_sig, e_res = np.sum(np.abs(x[span]) ** 2), np.sum(np.abs(y[span]) ** 2)
    assert 10 * np.log10(e_res / e_sig) <= -25.0
    assert np.array_equal(y[:span.start], x[:span.start]) and np.array_equal(y[span.stop:], x[span.stop:])


def test_nominal_position_pins_the_waterfall_framing(oracle):
    """s0 / f0 of the candidate are within half a quantisation step of the synthesised start and frequency."""
    for f0, t0 in [(500.0, 0.5), (503.1, 0.53), (777.7, 0.57), (1000.0, 0.62), (333.3, 1.1), (1500.0, 0.38)]:
        x, _ = gfsk_slot(oracle, [("CQ", "K1JT", "FN20", f0, t0, 1.0)])
        s0, f_nom = sr.nominal(strongest_candidate(oracle, x))
        assert -128 <= round(t0 * 3200) - s0 <= 160 and abs(f_nom - f0) <= 1.5625 + 1e-3, (f0, t0, s0, f_nom)


@pytest.mark.parametrize("sep_hz,max_db", [(10.0, 1.0), (60.0, 0.1)])
def test_neighbour_is_left_alone(oracle, sep_hz, max_db):
    """Removing one of two equal signals sep_hz apart changes the other's coherent energy by less than max_db.  10 Hz apart the
    8-FSK tones of the two overlap within the 0.32 s window's main lobe (+-6.25 Hz) for part of the slot, and the amplitude
    estimate takes up some of the neighbour (0.6 dB); beyond the 50 Hz signal bandwidth it takes up none (< 0.001 dB)."""
    a = ("CQ", "K1JT", "FN20", 700.0, 0.5, 1.0)
    b = ("CQ", "W1AW", "FN31", 700.0 + sep_hz, 0.62, 1.0)
    x, (cwa, _) = gfsk_slot(oracle, [a, b])
    xa, _ = gfsk_slot(oracle, [a])
    xb, _ = gfsk_slot(oracle, [b])
    y, _ = sr.subtract(x, [(strongest_candidate(oracle, xa), cwa)])
    start = round(0.62 * 3200)
    span = slice(start, start + sr.SPAN)
    proj = np.vdot(xb[span], y[span]) / np.vdot(xb[span], xb[span])   # the residual projected on b's own waveform
    assert abs(20 * np.log10(abs(proj))) < max_db


def test_window_is_edge_corrected():
    assert sr.WINDOW.size == 1025 and np.all(sr.WINDOW > 0) and np.isclose(sr.WINDOW[512], 1.0)
    for n in (1, 300, 1025, 5000):
        for v in (1.0, 2.5 - 0.5j):
            assert np.allclose(sr.smooth(np.full(n, v)), v, rtol=0, atol=1e-12)   # a constant is kept to the span's edges
    rng = np.random.default_rng(3)
    c = rng.standard_normal(3000) + 1j * rng.standard_normal(3000)
    a = sr.smooth(c)
    for n in (0, 17, 511, 512, 1500, 2488, 2999):
        k = np.arange(max(n - 512, 0), min(n + 513, c.size))
        h = sr.WINDOW[k - n + 512]
        assert np.isclose(a[n], np.sum(h * c[k]) / np.sum(h), rtol=1e-12, atol=1e-12)
    # a linear ramp is kept away from the edges (the window is symmetric)
    ramp = np.arange(4000, dtype=np.float64)
    assert np.allclose(sr.smooth(ramp)[512:-512], ramp[512:-512], atol=1e-8)


def test_grid_tie_rule():
    m = np.ones((17, 17))
    assert sr.pick(m) == (0, 0)
    m[3, 5] = m[3, 2] = 2.0
    assert sr.pick(m) == (3, 2)
    m[2, 9] = m[5, 1] = 3.0
    assert sr.pick(m) == (2, 9)
    f = np.zeros(17)
    f[[4, 11]] = 1.0
    assert sr.pick(f) == (4,)


def test_tones_from_codeword_match_the_encoder(oracle):
    p = oracle.pack_std("CQ", "DL1ABC", "JO62")
    tones = oracle.tones(p)
    assert np.array_equal(sr.tones_from_codeword(bits_from_tones(tones)), tones)


# ------------------------------------------------------------------------------------------- spans that cross a slot edge
@pytest.mark.parametrize("f0,t0", [(703.3, -0.8), (1211.0, -0.3), (350.7, -0.05), (903.1, 2.4), (1402.2, 3.0), (512.9, 3.6)])
def test_removes_a_noiseless_signal_at_a_slot_edge(oracle, f0, t0):
    """A signal whose span hangs over the start (DT < 0) or the end (DT > 2.36 s) of the slot, as sync reports them on the air
    (time_offset -12 ... 23, so starts -5888 ... 12288).  Refinement finds the synthesised start and frequency from the in-slot part
    alone, subtraction removes that part to -25 dB, and no sample outside it changes."""
    x, (cw,) = gfsk_slot(oracle, [("CQ", "K1JT", "FN20", f0, t0, 1.0)])
    true_start = int(np.round(np.float64(np.float32(t0)) * 3200.0))
    assert true_start < 0 or true_start + sr.SPAN > sr.SLOT   # the span does cross an edge
    cand = strongest_candidate(oracle, x)
    s0, f_nom = sr.nominal(cand)
    assert abs(true_start - s0) <= 136 and abs(np.float32(f0) - f_nom) <= 1.5625 + 1e-6
    y, [(dt, df)] = sr.subtract(x, [(cand, cw)])
    assert s0 + dt == true_start
    assert abs(f_nom + df * sr.DF_STEP - float(np.float32(f0))) <= sr.DF_STEP
    span = slice(max(true_start, 0), min(true_start + sr.SPAN, sr.SLOT))
    e_sig, e_res = np.sum(np.abs(x[span]) ** 2), np.sum(np.abs(y[span]) ** 2)
    assert 10 * np.log10(e_res / e_sig) <= -25.0, 10 * np.log10(e_res / e_sig)
    assert np.array_equal(y[:span.start], x[:span.start]) and np.array_equal(y[span.stop:], x[span.stop:])


@pytest.mark.parametrize("n", [1, 2, 511, 512, 1024, 1025])
def test_smooth_on_spans_shorter_than_the_window(n):
    """A span that a slot edge clips to fewer samples than the 1025-tap window: a constant is kept, and every output is the
    taps inside the span times c over the sum of those taps."""
    for v in (1.0, -3.25 + 0.75j):
        assert np.allclose(sr.smooth(np.full(n, v)), v, rtol=0, atol=1e-12)
    rng = np.random.default_rng(n)
    c = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    a = sr.smooth(c)
    for m in sorted({0, n // 2, n - 1}):
        k = np.arange(max(m - 512, 0), min(m + 513, n))
        h = sr.WINDOW[k - m + 512]
        assert np.isclose(a[m], np.sum(h * c[k]) / np.sum(h), rtol=1e-12, atol=1e-12)


# ------------------------------------------------------------------------------------------- step 1: which messages are new
def _fuzz_pass(rng, pool, n_rows, p_pool=0.8, score_lo=-5):
    """One pass's decode results for one slot: rows drawn from pool (hash, text) with random ok and score."""
    from oracle.pyoracle import cand_dtype, msg_dtype
    cand = np.zeros(n_rows, cand_dtype)
    msg = np.zeros(n_rows, msg_dtype)
    cand["score"] = rng.integers(score_lo, 40, n_rows)
    cand["time_offset"] = rng.integers(-12, 24, n_rows)
    cand["freq_offset"] = rng.integers(0, 249, n_rows)
    cand["time_sub"] = rng.integers(0, 2, n_rows)
    cand["freq_sub"] = rng.integers(0, 2, n_rows)
    ok = (rng.random(n_rows) < p_pool).astype(np.uint8)
    for k in range(n_rows):
        h, text = pool[int(rng.integers(len(pool)))]
        msg[k]["hash"], msg[k]["text"] = h, text
    return cand, ok, msg


def _pool(rng, n, hashes):
    """n distinct messages; hashes from a small set so that different texts clash on a hash and on a table cell.  Some texts
    carry bytes after their NUL, which the table ignores: the same message with other bytes there is the same message."""
    out = []
    for k in range(n):
        text = (b"CQ K%dAB FN%02d" % (k, k % 100)) if k % 3 else (b"K%dAB W9XYZ RR73" % k)
        out.append((int(hashes[k % len(hashes)]), text))
    tails = [(h, t + b"\0" + bytes(rng.integers(65, 90, 3, dtype=np.uint8))) for h, t in out[:4]]
    return out + tails


def _check_accept_against_orc_spots(oracle, passes, max_msgs, min_score):
    log = []
    acc = []
    for cand, ok, msg in passes:
        acc.append(sr.accept((cand, ok, msg), log, max_msgs, min_score))
    cat = [np.concatenate([p[j] for p in passes]) for j in range(3)]
    want = oracle.spots(*cat, max_msgs=max_msgs, min_score=min_score)
    assert [sr.message_key(m) for m in want["msgs"]] == log
    rows = [(p, k) for p, a in enumerate(acc) for k in a]
    cands = np.array([passes[p][0][k] for p, k in rows], passes[0][0].dtype)
    freq = ((cands["freq_offset"].astype(np.float32) + cands["freq_sub"].astype(np.float32) / np.float32(2)) * np.float32(6.25)).astype(np.float32)
    assert np.array_equal(want["freq_hz"], freq) and np.array_equal(want["score"], cands["score"].astype(np.int32))
    assert want["n"] == len(log)
    return acc, log


@pytest.mark.parametrize("max_msgs", [1, 8, 50])
@pytest.mark.parametrize("fills", ["pass1", "pass2", "never"])
def test_accept_is_the_spot_table_over_passes(oracle, max_msgs, fills):
    """accept() over 2-3 passes equals orc_spots' unique-message log (the reference's own table loop) over the concatenated
    passes: the same messages in the same order, with their frequencies and scores.  Covered: hash clashes with different texts,
    duplicates within a pass and across passes, and a table that fills in pass 1, in pass 2, or never."""
    rng = np.random.default_rng(1000 * max_msgs + len(fills))
    n_pool = 3 * max_msgs + 4 if fills != "never" else max_msgs   # "never": no more distinct messages than the table holds
    seen_cross = seen_within = seen_clash = 0
    for trial in range(40):
        pool = _pool(rng, n_pool, rng.integers(0, 4 * max_msgs + 1, max(n_pool // 2, 1)))
        n_passes = 2 + trial % 2
        if fills == "pass1":
            sizes = [int(rng.integers(4 * max_msgs, 4 * max_msgs + 20))] + [int(rng.integers(0, 30)) for _ in range(n_passes - 1)]
        elif fills == "pass2":
            sizes = [int(rng.integers(0, max(max_msgs // 2, 1)))] + [int(rng.integers(4 * max_msgs, 4 * max_msgs + 20)) for _ in range(n_passes - 1)]
        else:
            sizes = [int(rng.integers(0, 30)) for _ in range(n_passes)]
        filling = {"pass1": 0, "pass2": 1}.get(fills)   # the pass that fills the table: every row of it is live
        passes = [_fuzz_pass(rng, pool, n, *((1.0, 10) if p == filling else ())) for p, n in enumerate(sizes)]
        for min_score in (10, 0):
            log = []
            n_after = []
            keys = []
            for cand, ok, msg in passes:
                live = [sr.message_key(msg[k]) for k in range(len(cand)) if ok[k] and cand[k]["score"] >= min_score]
                seen_cross += len(set(live) & set(log))
                seen_within += len(live) - len(set(live))
                keys.append(live)
                sr.accept((cand, ok, msg), log, max_msgs, min_score)
                n_after.append(len(log))
            _check_accept_against_orc_spots(oracle, passes, max_msgs, min_score)
            allkeys = {k for ks in keys for k in ks}
            seen_clash += len(allkeys) - len({h for h, _ in allkeys})
            if min_score == 10:
                if fills == "pass1":
                    assert n_after[0] == max_msgs
                elif fills == "pass2":
                    assert n_after[0] < max_msgs and n_after[1] == max_msgs
            if fills == "never":
                assert n_after[-1] == len(allkeys)   # nothing was dropped for lack of room
    assert seen_within and (seen_cross or max_msgs == 1 and fills != "never") and (seen_clash or max_msgs == 1)

