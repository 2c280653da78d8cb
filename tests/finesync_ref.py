"""Float64 definition of fine-sync decoding's front half (DESIGN.md section 2.4.4); csrc/finesync.cu is held to it.

For one candidate of a daemon slot x (3200 sps complex, 48 000 samples, zero outside [0, 48000)):
- nominal position s0, f0: subtract_ref.nominal;
- Costas metric S(s, f) = sum over the 21 Costas symbols k (0-6, 36-42, 72-78) of
  |sum_{m < 512} x[s + 512 k + m] exp(-2 pi i (f + 6.25 costas[k]) m / 3200)|^2 -- pure tones, the data tones being unknown;
- grid: coarse dt = -256, -240 ... +256 (33) x df = -8 ... +8 steps of 6.25/32 Hz (17), then dt_c + (-8 ... +8) at that df; ties to
  the lower dt index, then the lower df index (subtract_ref.pick);
- spectra at s* = s0 + dt, f* = f0 + df: c[k][j] = sum_{m < 512} x[s* + 512 k + m] exp(-2 pi i (f* + 6.25 j) m / 3200), k < 79, j < 8;
  E = mean |c|^2 (E = 0: not attempted);
- LLRs: v = 10 log10(|c|^2 / E + 1e-12), the max-log bit metrics of ref64.llrs over v (data symbols 7-35 and 43-71, Gray map, the
  same bit order) and its normalisation sqrt(24 / var); a non-finite LLR: not attempted.
The back half is the BP of decode_kernel on these LLRs with the acceptance gates of the header (zero syndrome, CRC, unpack, hard
distance <= cap).  This module imports ref64 and subtract_ref and nothing of the library or the oracle."""
import numpy as np

from ref64 import FT8_COSTAS, FT8_DATA, FT8_GRAY, FT8_SYNC_AT
from subtract_ref import DF_STEP, DF_STEPS, FS, NSYM, SYM, TONE_HZ, nominal, pick

DT_COARSE = np.arange(-256, 257, 16)    # 33 points
DT_FINE = np.arange(-8, 9)
COSTAS_SYMS = np.array([g0 + k for g0 in FT8_SYNC_AT for k in range(7)])
COSTAS_TONES = np.tile(FT8_COSTAS, 3)
_M = np.arange(SYM)


def symbols(x, start, n_sym=NSYM):
    """x over [start, start + 512 n_sym) as [n_sym, 512], zero outside the slot."""
    x = np.asarray(x, np.complex128)
    idx = start + np.arange(n_sym * SYM)
    inside = (idx >= 0) & (idx < x.size)
    seg = np.zeros(idx.size, np.complex128)
    seg[inside] = x[idx[inside]]
    return seg.reshape(n_sym, SYM)


def costas_metric(x, s, f):
    seg = symbols(x, s)[COSTAS_SYMS]
    ph = np.exp(-2j * np.pi * (f + TONE_HZ * COSTAS_TONES)[:, None] * _M[None, :] / FS)
    return float((np.abs((seg * ph).sum(axis=1)) ** 2).sum())


def search(x, cand, with_metrics=False):
    """-> (dt samples, df steps) [, (coarse metric [33, 17], fine metric [17])]."""
    s0, f0 = nominal(cand)
    coarse = np.array([[costas_metric(x, s0 + dt, f0 + d * DF_STEP) for d in DF_STEPS] for dt in DT_COARSE])
    i, j = pick(coarse)
    dt_c, df = int(DT_COARSE[i]), int(DF_STEPS[j])
    fine = np.array([costas_metric(x, s0 + dt_c + d, f0 + df * DF_STEP) for d in DT_FINE])
    dt = dt_c + int(DT_FINE[pick(fine)[0]])
    return ((dt, df), (coarse, fine)) if with_metrics else (dt, df)


def spectra(x, start, f):
    """|c[k][j]|^2, [79, 8]."""
    seg = symbols(x, start)
    ph = np.exp(-2j * np.pi * (f + TONE_HZ * np.arange(8))[:, None] * _M[None, :] / FS)   # [8, 512]
    return np.abs(seg @ ph.T) ** 2


def llrs_from_power(p):
    """[79, 8] tone powers -> 174 normalised LLRs (NaN when the mean power is 0)."""
    e = p.mean()
    if e == 0:
        return np.full(174, np.nan)
    v = 10.0 * np.log10(p / e + 1e-12)
    out = np.zeros((FT8_DATA.size, 3))
    for k, sym in enumerate(FT8_DATA):
        s = v[sym, FT8_GRAY]                                    # s[j] = metric of the tone that carries bits j
        for i in range(3):
            one = (np.arange(8) >> (2 - i)) & 1
            out[k, i] = s[one == 1].max() - s[one == 0].max()
    x = out.reshape(-1)
    var = (np.sum(x * x) - np.sum(x) ** 2 / 174.0) / 174.0
    with np.errstate(divide="ignore", invalid="ignore"):
        return x * np.sqrt(24.0 / var)


def finesync(x, cand):
    """-> ((dt, df), llr [174]); llr has a non-finite entry when the candidate is not attempted."""
    x = np.asarray(x, np.complex128)
    dt, df = search(x, cand)
    s0, f0 = nominal(cand)
    return (dt, df), llrs_from_power(spectra(x, s0 + dt, f0 + df * DF_STEP))


def attempted(llr):
    return bool(np.all(np.isfinite(llr)))
