"""Float64 definition of signal subtraction for multi-pass decoding (DESIGN.md section 2.4.2); csrc/subtract.cu is held to it.

For one daemon slot x (3200 sps complex, 48 000 samples) and a list of decoded messages (candidate + 174-bit codeword):
- tones: the 79 FT8 channel tones of the codeword (Costas arrays + Gray map, ref64's constants);
- nominal position: start sample s0 = 512 time_offset + 256 time_sub + 256 and tone-0 frequency f0 = 3.125 (2 freq_offset +
  freq_sub) Hz -- the waterfall's 1024-point frames at hop 256 are 3.125 Hz wide, and a frame is centred on the symbol it scores;
- reference r_{dt,df}: unit-amplitude GFSK as gen_ft8 sends it (ref64.gfsk_phase: BT = 2, extended end symbols, raised-cosine
  ramps), starting at s0 + dt with tone 0 at f0 + df;
- refinement, on x itself: M = sum_k |sum_{n in symbol k} x[n] conj(r[n])|^2 (samples outside the slot skipped), maximised over
  dt = -128, -112 ... +128 x df = -8 ... +8 steps of 6.25/32 Hz, then over dt + (-8 ... +8) at that df; ties to the lower dt
  index, then the lower df index;
- subtraction, in list order on the running residual y (from y = x): over the message's span (its 79 symbols within the slot)
  c = y conj(r), a = c smoothed by h[k] = cos^2(pi k / 1026), |k| <= 512, normalised by the taps inside the span, y -= a r.
Which messages a pass subtracts is step 1 of the multi-pass definition (accept): the ones the spot table accepted as new.
This module imports ref64 (gfsk_phase and the protocol constants) and nothing of the library or the oracle."""
import numpy as np
from scipy.signal import fftconvolve

from ref64 import FT8_COSTAS, FT8_DATA, FT8_GRAY, FT8_SYNC_AT, gfsk_phase

FS = 3200.0
SYM = 512
NSYM = 79
SPAN = SYM * NSYM
SLOT = 48000
TONE_HZ = 6.25
DT_COARSE = np.arange(-128, 129, 16)    # 17 points
DF_STEPS = np.arange(-8, 9)             # 17 points of DF_STEP
DF_STEP = TONE_HZ / 32.0
DT_FINE = np.arange(-8, 9)
WINDOW = np.cos(np.pi * np.arange(-512, 513) / 1026.0) ** 2   # 1025 taps, 0.32 s


def tones_from_codeword(cw):
    cw = np.asarray(cw, np.int64)
    tones = np.zeros(NSYM, np.int64)
    for g0 in FT8_SYNC_AT:
        tones[g0:g0 + 7] = FT8_COSTAS
    v = cw.reshape(58, 3) @ np.array([4, 2, 1])
    tones[FT8_DATA] = FT8_GRAY[v]
    return tones


def nominal(cand):
    """(start sample, tone-0 frequency in Hz) of a candidate (cand_dtype record or dict-like)."""
    s0 = 512 * int(cand["time_offset"]) + 256 * int(cand["time_sub"]) + 256
    f0 = 3.125 * (2 * int(cand["freq_offset"]) + int(cand["freq_sub"]))
    return s0, f0


def reference(tones, f_hz):
    phase, env = gfsk_phase(tones, SYM, FS, f_hz, TONE_HZ, 2.0)
    return env * np.exp(1j * phase)


def _window_of(x, start):
    """x over [start, start + SPAN), zero outside the slot; and the mask of samples inside it."""
    idx = start + np.arange(SPAN)
    inside = (idx >= 0) & (idx < x.size)
    seg = np.zeros(SPAN, np.complex128)
    seg[inside] = x[idx[inside]]
    return seg, inside


def metric(x, start, r):
    seg, _ = _window_of(x, start)
    return float((np.abs((seg * np.conj(r)).reshape(NSYM, SYM).sum(axis=1)) ** 2).sum())


def pick(m):
    """Index of the largest entry of a metric array in C order: ties go to the lower first index, then the lower second."""
    m = np.asarray(m)
    return np.unravel_index(int(np.argmax(m)), m.shape)


def refine(x, cand, cw, with_metrics=False):
    """-> (dt samples, df steps) [, (coarse metric [17, 17], fine metric [17])]."""
    x = np.asarray(x, np.complex128)
    tones = tones_from_codeword(cw)
    s0, f0 = nominal(cand)
    refs = [reference(tones, f0 + d * DF_STEP) for d in DF_STEPS]
    coarse = np.array([[metric(x, s0 + dt, r) for r in refs] for dt in DT_COARSE])
    i, j = pick(coarse)
    dt_c, df = int(DT_COARSE[i]), int(DF_STEPS[j])
    fine = np.array([metric(x, s0 + dt_c + d, refs[j]) for d in DT_FINE])
    dt = dt_c + int(DT_FINE[pick(fine)[0]])
    return ((dt, df), (coarse, fine)) if with_metrics else (dt, df)


def smooth(c):
    """Edge-corrected Hann smoothing of c (the signal's span): sum of the taps inside the span times c, over the sum of those taps."""
    c = np.asarray(c, np.complex128)
    num = fftconvolve(c, WINDOW, mode="same")
    den = fftconvolve(np.ones(c.size), WINDOW, mode="same")
    return num / den


def message_key(msg):
    """(hash, text up to its first NUL) of a msg_dtype record: what the spot table tells messages apart by."""
    return int(msg["hash"]), bytes(msg["text"]).split(b"\0")[0]


def accept(rows, log, max_msgs, min_score):
    """Step 1 of a pass: the rows (cand, ok, msg: one slot's candidates of one pass, cand_dtype / uint8 / msg_dtype) the spot table
    accepts as new, in candidate order.  A row is live when ok is set and its score is >= min_score; it is accepted when its key is
    not in log (the keys accepted by earlier passes and earlier rows) and log holds fewer than max_msgs keys.  With linear probing
    and no deletions that is exactly the table's behaviour, a full table included.  Extends log; returns the accepted row indices."""
    cand, ok, msg = rows
    seen = set(log)
    out = []
    for k in range(len(cand)):
        if not ok[k] or int(cand[k]["score"]) < min_score:
            continue
        key = message_key(msg[k])
        if key in seen or len(log) >= max_msgs:
            continue
        seen.add(key)
        log.append(key)
        out.append(k)
    return out


def subtract(x, msgs, grids=None):
    """x: complex slot; msgs: list of (cand, cw) in subtraction order.  -> (residual, [(dt, df) per message]).  grids: use these
    grid points instead of refining (to hold the subtraction alone to a kernel's choice)."""
    x = np.asarray(x, np.complex128)
    if grids is None:
        grids = [refine(x, cand, cw) for cand, cw in msgs]   # all on x: the messages refine independently
    y = x.copy()
    for (cand, cw), (dt, df) in zip(msgs, grids):
        s0, f0 = nominal(cand)
        start = s0 + dt
        r = reference(tones_from_codeword(cw), f0 + df * DF_STEP)
        lo, hi = max(start, 0), min(start + SPAN, x.size)
        if lo >= hi:
            continue
        rr = r[lo - start:hi - start]
        a = smooth(y[lo:hi] * np.conj(rr))
        y[lo:hi] -= a * rr
    return y, grids
