"""Float64 definition of deep fine sync's LLR sets (DESIGN.md section 2.4.6); finesync_kernel<true> in csrc/finesync.cu is held to it.

For one candidate of a daemon slot x, at fine sync's grid point (finesync_ref.search: s* = s0 + dt, f* = f0 + df):
- coherent spectra c'[k][j] = sum_{m < 512} x[s* + 512 k + m] exp(-2 pi i (f* (512 k + m) + 6.25 j m) / 3200), k < 79, j < 8: fine
  sync's c[k][j] times exp(-2 pi i f* 512 k / 3200), so that every symbol refers to one time origin (|c'| = |c|);
- set a: finesync_ref.llrs_from_power(|c'|^2), fine sync's dB set;
- sets b, c (nsym = 2, 3): each half of 29 data symbols (7-35, 43-71) split into groups of nsym consecutive symbols from its first
  one, the last taking what remains; for a group of g symbols and each of the 8^g patterns b, A(b) = |sum_t c'[sym_t][gray[b_t]]|;
  the LLR of each of the group's 3 g bits (3 per symbol, MSB first) is max A over the patterns with the bit 1 minus max A over those
  with it 0; the 174 values normalised by sqrt(24 / var) as set a;
- E = mean |c'|^2 = 0 or any non-finite value: that set is not attempted.
This module imports finesync_ref, subtract_ref and ref64 and nothing of the library or the oracle."""
import itertools

import numpy as np

import finesync_ref as fr
from ref64 import FT8_DATA, FT8_GRAY
from subtract_ref import DF_STEP, FS, NSYM, SYM, TONE_HZ, nominal

_M = np.arange(SYM)


def coherent_spectra(x, start, f):
    """c'[k][j], complex [79, 8]."""
    seg = fr.symbols(x, start)
    ph = np.exp(-2j * np.pi * (f + TONE_HZ * np.arange(8))[:, None] * _M[None, :] / FS)   # [8, 512]
    return (seg @ ph.T) * np.exp(-2j * np.pi * f * SYM * np.arange(NSYM) / FS)[:, None]


def groups(nsym):
    """-> [(first data symbol index 0 ... 57, g)] in bit order."""
    return [(29 * h + s, min(nsym, 29 - s)) for h in range(2) for s in range(0, 29, nsym)]


def _patterns(g):
    """-> (b [8^g, g] in C order, bits [8^g, 3 g]: bit q = bit 2 - q % 3 of b[q // 3])."""
    b = np.indices((8,) * g).reshape(g, -1).T
    bits = ((b[:, :, None] >> np.array([2, 1, 0])) & 1).reshape(b.shape[0], 3 * g)
    return b, bits


def group_llrs(cp, syms):
    """The 3 g unnormalised max-log LLRs of the group of data symbols syms, vectorised over the 8^g patterns."""
    b, bits = _patterns(len(syms))
    a = np.abs(sum(cp[s, FT8_GRAY[b[:, t]]] for t, s in enumerate(syms)))
    return np.array([a[bits[:, q] == 1].max() - a[bits[:, q] == 0].max() for q in range(bits.shape[1])])


def group_llrs_loop(cp, syms):
    """group_llrs as a plain loop over the patterns (the test's brute force)."""
    g = len(syms)
    best = np.full((3 * g, 2), -np.inf)
    for b in itertools.product(range(8), repeat=g):
        a = abs(sum(cp[s, FT8_GRAY[bt]] for s, bt in zip(syms, b)))
        for q in range(3 * g):
            v = (b[q // 3] >> (2 - q % 3)) & 1
            best[q, v] = max(best[q, v], a)
    return best[:, 1] - best[:, 0]


def normalise(raw, e):
    if e == 0 or not np.isfinite(e):
        return np.full(174, np.nan)
    var = (np.sum(raw * raw) - np.sum(raw) ** 2 / 174.0) / 174.0
    with np.errstate(divide="ignore", invalid="ignore"):
        return raw * np.sqrt(24.0 / var)


def coherent_llrs(cp, nsym):
    """Set b (nsym = 2) or c (nsym = 3) from c' -> 174 normalised LLRs (NaN when E = 0)."""
    raw = np.concatenate([group_llrs(cp, FT8_DATA[s:s + g]) for s, g in groups(nsym)])
    return normalise(raw, float(np.mean(np.abs(cp) ** 2)))


def llr_sets(cp):
    """-> float64 [3, 174]: sets a, b, c from c'."""
    return np.stack([fr.llrs_from_power(np.abs(cp) ** 2), coherent_llrs(cp, 2), coherent_llrs(cp, 3)])


def sets_at(x, cand, dt, df):
    s0, f0 = nominal(cand)
    return llr_sets(coherent_spectra(np.asarray(x, np.complex128), s0 + dt, f0 + df * DF_STEP))


def finesync_sets(x, cand):
    """-> ((dt, df), llr [3, 174]); a set is not attempted when it has a non-finite entry (fr.attempted)."""
    x = np.asarray(x, np.complex128)
    dt, df = fr.search(x, cand)
    return (dt, df), sets_at(x, cand, dt, df)
