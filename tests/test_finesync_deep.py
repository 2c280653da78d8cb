"""The float64 definition of deep fine sync's LLR sets (tests/finesync_deep_ref.py) on noiseless GFSK placed by hand with
ref64.gfsk_phase: the nsym = 2 and 3 coherent sets recover the codeword, ignore the carrier phase, cover every bit once, and their
vectorised max-log equals a brute-force loop.  No GPU needed."""
import numpy as np
import pytest

import finesync_deep_ref as dr
import finesync_ref as fr
import subtract_ref as sr
from ref64 import FT8_DATA
from test_finesync import CAND, CW, cand_at, slot_with


def noise(seed):
    return np.array([1, 1j]) @ np.random.default_rng(seed).standard_normal((2, sr.SLOT))


@pytest.mark.parametrize("dt", [0, -123, 161])
@pytest.mark.parametrize("df_hz", [0.0, -sr.DF_STEP, 0.7 * sr.DF_STEP, sr.DF_STEP])
def test_coherent_sets_recover_the_codeword(dt, df_hz):
    """The hard decisions of sets b and c at the true alignment, and at the grid point the search picks with a start error of dt and
    a frequency error of up to one df step, are the codeword."""
    s0, f0 = sr.nominal(CAND)
    x = slot_with(s0 + dt, f0 + df_hz)
    if dt == 0 and df_hz == 0.0:
        llr = dr.sets_at(x, CAND, 0, 0)
    else:
        (gdt, _), llr = dr.finesync_sets(x, CAND)
        assert abs(gdt - dt) <= 8
    assert np.all(np.isfinite(llr))
    for k in (1, 2):
        assert np.array_equal((llr[k] > 0).astype(np.uint8), CW), (k, np.nonzero((llr[k] > 0) != CW)[0])


def test_set_a_is_fine_syncs_set():
    s0, f0 = sr.nominal(CAND)
    x = slot_with(s0 + 40, f0 + 0.3) + 0.3 * noise(5)
    (dt, df), a = fr.finesync(x, CAND)
    (dt2, df2), sets = dr.finesync_sets(x, CAND)
    assert (dt, df) == (dt2, df2)
    np.testing.assert_allclose(sets[0], a, rtol=0, atol=1e-9)


def test_constant_phase_rotation_leaves_sets_b_and_c():
    s0, f0 = sr.nominal(CAND)
    x = slot_with(s0 - 30, f0 + 0.5) + 0.5 * noise(6)
    base = dr.sets_at(x, CAND, -32, 3)
    for theta in (0.3, 1.9, -2.7):
        rot = dr.sets_at(x * np.exp(1j * theta), CAND, -32, 3)
        np.testing.assert_allclose(rot[1:], base[1:], rtol=0, atol=1e-9)


@pytest.mark.parametrize("nsym,sizes", [(2, [2] * 14 + [1]), (3, [3] * 9 + [2])])
def test_grouping_covers_every_bit_once(nsym, sizes):
    gs = dr.groups(nsym)
    assert [g for _, g in gs] == sizes * 2
    assert [s for s, _ in gs][:1] == [0] and gs[len(sizes)][0] == 29   # each half starts at its first data symbol
    bits = np.concatenate([np.arange(3 * s, 3 * (s + g)) for s, g in gs])
    assert np.array_equal(np.sort(bits), np.arange(174)) and np.array_equal(bits, np.arange(174))
    syms = np.concatenate([FT8_DATA[s:s + g] for s, g in gs])
    assert np.array_equal(syms, FT8_DATA)
    for s, g in gs:   # no group reaches across a Costas array
        assert FT8_DATA[s + g - 1] - FT8_DATA[s] == g - 1


@pytest.mark.parametrize("g", [1, 2, 3])
def test_vectorised_max_log_equals_the_loop(g):
    rng = np.random.default_rng(10 + g)
    for _ in range(3):
        cp = rng.standard_normal((79, 8)) + 1j * rng.standard_normal((79, 8))
        syms = FT8_DATA[rng.integers(0, 58 - g) + np.arange(g)]
        np.testing.assert_allclose(dr.group_llrs(cp, syms), dr.group_llrs_loop(cp, syms), rtol=0, atol=1e-12)


def test_empty_slots_and_spans_outside_are_not_attempted():
    (_, _), sets = dr.finesync_sets(np.zeros(sr.SLOT, np.complex128), CAND)
    assert not any(fr.attempted(s) for s in sets)
    far = cand_at(256 + 512 * 200, 2 * 160)   # nominal start 102 656: the whole span lies past the slot's end
    x = slot_with(1000, 1000.0)
    (_, _), sets = dr.finesync_sets(x, far)
    assert not any(fr.attempted(s) for s in sets)
