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
