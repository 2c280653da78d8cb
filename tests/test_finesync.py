"""The float64 definition of fine-sync decoding's front half (tests/finesync_ref.py) on noiseless GFSK placed by hand with
ref64.gfsk_phase, and its tie, edge and empty-slot rules.  No GPU needed."""
import numpy as np
import pytest

import finesync_ref as fr
import subtract_ref as sr
from ref64 import gfsk_phase
from tools import ft8enc

PAYLOAD = ft8enc.pack_std("CQ", "K1JT", "FN20")
CW = ft8enc.encode174(PAYLOAD)
TONES = ft8enc.tones(PAYLOAD)


def cand_at(s0, f0_steps):
    """A candidate whose nominal start is s0 (256 plus a multiple of 256) and tone-0 frequency 3.125 f0_steps Hz."""
    to, ts = divmod(s0 - 256, 512)
    assert ts in (0, 256)
    fo, fs = divmod(f0_steps, 2)
    return {"time_offset": to, "time_sub": ts // 256, "freq_offset": fo, "freq_sub": fs}


def slot_with(start, f_hz, tones=TONES, amp=1.0):
    """A noiseless unit-amplitude GFSK signal starting at sample `start` (may hang over either end) with tone 0 at f_hz."""
    phase, env = gfsk_phase(tones, sr.SYM, sr.FS, f_hz, sr.TONE_HZ, 2.0)
    x = np.zeros(sr.SLOT, np.complex128)
    n = start + np.arange(phase.size)
    inside = (n >= 0) & (n < sr.SLOT)
    x[n[inside]] = amp * env[inside] * np.exp(1j * phase[inside])
    return x


S0, F0_STEPS = 512 * 4 + 256, 2 * 160 + 1   # nominal 0.72 s, 1003.125 Hz
CAND = cand_at(S0, F0_STEPS)


def test_candidate_helper_is_the_nominal_position():
    assert sr.nominal(CAND) == (S0, 3.125 * F0_STEPS)


@pytest.mark.parametrize("dt", [-256, -241, -123, -8, 0, 5, 77, 161, 250, 256])
@pytest.mark.parametrize("df_hz", [-1.5625, -0.8, 0.0, 0.33, 1.5625])
def test_recovers_start_and_frequency_inside_the_grid(dt, df_hz):
    s0, f0 = sr.nominal(CAND)
    x = slot_with(s0 + dt, f0 + df_hz)
    (gdt, gdf), (coarse, fine) = fr.search(x, CAND, with_metrics=True)
    assert coarse.shape == (33, 17) and fine.shape == (17,)
    assert abs(gdt - dt) <= 8, (dt, df_hz, gdt, gdf)
    assert abs(gdf * sr.DF_STEP - df_hz) <= sr.DF_STEP + 1e-9, (dt, df_hz, gdt, gdf)


@pytest.mark.parametrize("dt,df_hz", [(-272, 0.0), (272, 0.0), (0, -1.5625 - sr.DF_STEP), (0, 1.5625 + sr.DF_STEP), (272, 1.5625 + sr.DF_STEP)])
def test_one_step_outside_the_grid_stays_on_its_edge(dt, df_hz):
    """Truth one step beyond the grid: the search returns a point of the grid, on the edge nearest the truth."""
    s0, f0 = sr.nominal(CAND)
    gdt, gdf = fr.search(slot_with(s0 + dt, f0 + df_hz), CAND)
    assert -264 <= gdt <= 264 and -8 <= gdf <= 8
    if abs(dt) > 256:
        assert abs(gdt - dt) <= 16 and np.sign(gdt) == np.sign(dt)
    if abs(df_hz) > 1.5625:
        assert gdf == 8 * np.sign(df_hz)


@pytest.mark.parametrize("dt,df_hz", [(0, 0.0), (-123, 0.7), (161, -1.2)])
def test_hard_decisions_at_the_true_alignment_are_the_codeword(dt, df_hz):
    s0, f0 = sr.nominal(CAND)
    x = slot_with(s0 + dt, f0 + df_hz)
    llr = fr.llrs_from_power(fr.spectra(x, s0 + dt, f0 + df_hz))
    assert fr.attempted(llr)
    assert np.array_equal((llr > 0).astype(np.uint8), CW)
    assert np.isclose(np.sum(llr * llr) - np.sum(llr) ** 2 / 174, 24 * 174)   # normalised: variance 24
    # and through the whole front half, from the nominal position
    (gdt, gdf), llr2 = fr.finesync(x, CAND)
    assert np.array_equal((llr2 > 0).astype(np.uint8), CW), (gdt, gdf)


def test_tie_rule():
    """Equal metrics go to the lower dt index, then the lower df index: pick on constructed arrays, and an all-zero slot, whose
    metrics are all equal, ends on the first point of both stages."""
    m = np.zeros((33, 17))
    m[4, 9] = m[4, 2] = m[20, 0] = 3.0
    assert sr.pick(m) == (4, 2)
    m[3, 16] = 3.0
    assert sr.pick(m) == (3, 16)
    assert sr.pick(np.array([1.0, 2.0, 2.0, 0.5])) == (1,)
    x = np.zeros(sr.SLOT, np.complex128)
    assert fr.search(x, CAND) == (-256 - 8, -8)


@pytest.mark.parametrize("start", [-30000, -5888, 12288, 20000])
def test_spans_over_the_slot_edges_are_zero_filled(start):
    """Symbols outside [0, 48000) read zeros, and a signal hanging over either end is still found from the Costas groups inside."""
    seg = fr.symbols(np.arange(sr.SLOT) + 1.0, start)
    idx = start + np.arange(79 * 512)
    assert np.array_equal(seg.reshape(-1), np.where((idx >= 0) & (idx < sr.SLOT), idx + 1.0, 0.0))
    s0 = 256 + 256 * round((start - 77 - 256) / 256)   # a nominal start on the waterfall's grid, within 205 samples of the truth
    cand = cand_at(s0, F0_STEPS)
    x = slot_with(start, 3.125 * F0_STEPS + 0.4)
    dt, df = fr.search(x, cand)
    assert abs(s0 + dt - start) <= 8 and abs(df * sr.DF_STEP - 0.4) <= sr.DF_STEP
    (_, _), llr = fr.finesync(x, cand)
    assert fr.attempted(llr)


def test_empty_slot_and_span_outside_are_not_attempted():
    x = np.zeros(sr.SLOT, np.complex128)
    (_, _), llr = fr.finesync(x, CAND)
    assert not fr.attempted(llr)
    y = slot_with(S0, 1003.125)
    far = cand_at(256 + 512 * 200, F0_STEPS)   # span wholly after the slot, the grid's reach included
    (_, _), llr = fr.finesync(y, far)
    assert not fr.attempted(llr)
