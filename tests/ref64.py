"""Independent numpy references for the GPU stages: float64 arithmetic, or exact integers where the operation is integer.

The GPU parity tests compare the kernels bit for bit with oracle/libft8oracle.so, a plain-C restatement of the reference
that shares csrc/ft8_tables.h with the kernels.  A change that moves kernel and restatement away from FT8/FT4 in the same
way passes those tests.  The functions here restate each stage from the protocol definitions instead, so that
tests/test_gpu_independent.py and tests/test_tables_independent.py hold the kernels to FT8/FT4 themselves.

Independence rules (what keeps these references from sharing a mistake with the kernels):
- This module does not import oracle.pyoracle or the library, and does not read csrc/ft8_tables.h.
- Protocol constants are written out below from the FT8/FT4 definitions.
- The LDPC(174,91) checks come from tools/ldpc_174_91_nm.txt, the source text the header is generated from.
- The CRC-14 is implemented here as plain polynomial division; it is checked against tests/golden/kat.npz["crc_test3"],
  which the unmodified reference computed.
- The daemon's FFT window is kat.npz["window"], which the reference recorded.
- The FFTs are numpy's float64 ones, not kiss_fft's float arithmetic, so results may differ from the kernels' by the
  north-star allowances (waterfall cells +-1 LSB on <= 0.01 % of cells, decimator floats 1e-5 relative), never by more.
"""
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# ---- protocol constants (FT8/FT4 definitions) -------------------------------------------------------------------------
FT8_COSTAS = np.array([3, 1, 4, 0, 6, 5, 2])
FT8_GRAY = np.array([0, 1, 3, 2, 5, 6, 4, 7])              # 3 bits -> tone
FT4_COSTAS = np.array([[0, 1, 3, 2], [1, 0, 2, 3], [2, 3, 1, 0], [3, 2, 0, 1]])
FT4_GRAY = np.array([0, 1, 3, 2])                           # 2 bits -> tone
FT8_SYNC_AT = (0, 36, 72)                                   # first symbol of each 7-symbol Costas group
FT8_DATA = np.r_[7:36, 43:72]                               # 58 data symbols
FT4_SYNC_AT = (1, 34, 67, 100)                              # first symbol of each 4-symbol Costas group
FT4_DATA = np.r_[5:34, 38:67, 71:100]                       # 87 data symbols
FT4_XOR = bytes([0x4A, 0x5E, 0x89, 0xB4, 0xB0, 0x8A, 0x79, 0x55, 0xBE, 0x28])   # FT4 scrambling vector over the 77 message bits
CRC14_POLY = 0x2757                                         # x^14 + x^13 + x^10 + x^9 + x^8 + x^6 + x^4 + x^2 + x + 1, top bit implied

# The daemon's CIC compensation filter (rtlsdr_ft8d.c:93-110): 57 taps, symmetric about tap 28 = 0.5, stored as float.
_FIR_HALF = [-0.0025719973, 0.0010118403, 0.0009110571, -0.0034940765, 0.0069713409, -0.0114242790, 0.0167023466,
             -0.0223683056, 0.0276808966, -0.0316243672, 0.0329894230, -0.0305042011, 0.0230074504, -0.0096499429,
             -0.0098950502, 0.0352349632, -0.0650990428, 0.0972406918, -0.1284211497, 0.1544893973, -0.1705667465,
             0.1713383321, -0.1514501610, 0.1060148823, -0.0312560926, -0.0745846391, 0.2096088743, -0.3638689868]
FIR = np.float32(_FIR_HALF + [0.5] + _FIR_HALF[::-1]).astype(np.float64)
DECIM = 751                  # keep one integrator output in 751 (2.4 Msps -> 3195.7 sps)
DECIM_SCALE = 32768.0 * 750  # = 24 576 000


def ldpc_checks():
    """int array [83, 7] of 0-origin variable indices, -1 = unused (tools/ldpc_174_91_nm.txt)."""
    rows = []
    with open(os.path.join(ROOT, "tools", "ldpc_174_91_nm.txt")) as f:
        for line in f:
            if line.strip() and not line.startswith("#"):
                rows.append([int(v) - 1 for v in line.split()])
    return np.array(rows)


def parity_matrix():
    """H as uint8 [83, 174] over GF(2)."""
    nm = ldpc_checks()
    H = np.zeros((nm.shape[0], 174), np.uint8)
    for m, row in enumerate(nm):
        H[m, row[row >= 0]] = 1
    return H


def checks_satisfied(bits174) -> np.ndarray:
    """bool per word: every one of the 83 checks has even parity.  bits174: [..., 174] of 0/1."""
    b = np.asarray(bits174, np.int64)
    return ((b @ parity_matrix().T.astype(np.int64)) % 2 == 0).all(axis=-1)


def crc14_bits(bits) -> int:
    """CRC-14 of a bit sequence (MSB first): the remainder of bits(x) * x^14 modulo the generator."""
    reg = 0
    for b in bits:
        fb = ((reg >> 13) & 1) ^ int(b)
        reg = (reg << 1) & 0x3FFF
        if fb:
            reg ^= CRC14_POLY
    return reg


def crc14_bytes(data: bytes, num_bits: int) -> int:
    return crc14_bits(np.unpackbits(np.frombuffer(bytes(data), np.uint8))[:num_bits])


def crc_ok(bits174) -> bool:
    """Bits 77..90 are the CRC-14 of the 77 message bits followed by 5 zero bits."""
    b = np.asarray(bits174, np.int64)
    want = int("".join(str(int(x)) for x in b[77:91]), 2)
    return crc14_bits(np.r_[b[:77], np.zeros(5, np.int64)]) == want


# ---- decimator (rtlsdr_ft8d.c:76-202) ---------------------------------------------------------------------------------
def _neg8(v):
    """int8 negate with two's-complement wrap: -(-128) = -128."""
    return np.where(v == -128, -128, -v)


def mix(iq_u8):
    """fs/4 mixer: complex sample n times j^n, on int8 rails (byte ^ 0x80).  -> (I, Q) int64."""
    iq = np.asarray(iq_u8, np.uint8)
    n = iq.size // 2
    a = iq[0:2 * n:2].astype(np.int64) - 128
    b = iq[1:2 * n:2].astype(np.int64) - 128
    ph = np.arange(n) & 3
    mi = np.select([ph == 0, ph == 1, ph == 2], [a, _neg8(b), _neg8(a)], b)
    mq = np.select([ph == 0, ph == 1, ph == 2], [b, a, _neg8(b)], _neg8(a))
    return mi, mq


def _wrap32(x):
    return ((np.asarray(x, np.int64) + 2 ** 31) % 2 ** 32 - 2 ** 31).astype(np.int64)


def decimate(iq_u8):
    """The sample loop: two integrators, keep every 751st value (sample 750 + 751 k), two combs with delay 2, all mod 2^32,
    then the 57-tap FIR in float64 over the int32 comb outputs (zero history) and / 24 576 000.
    -> (y2 int64 [n, 2] holding int32 values, I float64 [n], Q float64 [n])."""
    out = []
    for rail in mix(iq_u8):
        x2 = np.cumsum(np.cumsum(rail))[DECIM - 1::DECIM]          # exact in int64 for any slot size used here
        y1 = x2 - np.r_[0, 0, x2[:-2]][: x2.size]
        y2 = _wrap32(y1 - np.r_[0, 0, y1[:-2]][: y1.size])
        out.append(y2)
    y2 = np.stack(out, axis=1)
    f = []
    for r in range(2):
        full = np.convolve(y2[:, r].astype(np.float64), FIR[::-1])[: y2.shape[0]]   # out[k] = sum_j FIR[j] * y2[k - 56 + j]
        f.append(full / DECIM_SCALE)
    return y2, f[0], f[1]


def slot_rows(n_samples_per_slot: int, slots: int):
    """For one continuous stream cut into slots of n samples: (first, count) output indices per slot -- the outputs whose
    decimation instant 750 + 751 k falls into [s n, (s + 1) n)."""
    first = [max(0, -((DECIM - 1 - s * n_samples_per_slot) // DECIM)) for s in range(slots + 1)]
    return [(first[s], first[s + 1] - first[s]) for s in range(slots)]


# ---- waterfalls ---------------------------------------------------------------------------------------------------------
# A float32 FFT -- the reference's kiss_fft, to which the kernels are bit-identical, as much as any other -- carries rounding
# noise of about float epsilon (6e-8) times the frame's largest bin amplitude.  80 dB below that bin in power a cell's value is
# still known to about 1e-3, which the quantiser's 0.5 dB steps absorb at the 0.01 % rate; further down, for example in the
# sidelobes of a pure tone or a square wave, the float32 noise decides on which side of a step a cell lands.  The +-1 LSB bar
# holds everywhere; the 0.01 % count is taken over the cells within RESOLVABLE of their frame's largest bin.
RESOLVABLE = 1e-8
# -------------------------------------------------------------------------------------------------------
def quantise(x):
    """clamp(trunc(20 log10(x) + 240), 0, 255) in float64 (x > 0)."""
    v = np.trunc(20.0 * np.log10(np.asarray(x, np.float64)) + 240.0)
    return np.clip(v, 0, 255).astype(np.uint8)


def daemon_waterfall(i_s, q_s, window, peak=None, resolvable=False):
    """Daemon waterfall (rtlsdr_ft8d.c:1395-1435): frames of 1024 at 512 blk + 256 ts, the recorded window, FFT index 2 b + fs
    -> uint8 [92, 2, 2, 256] flattened.  peak: decoder()'s conditioning 0.5 / peak applied first.
    resolvable: also return the cells a float32 FFT can resolve (see RESOLVABLE)."""
    x = np.asarray(i_s, np.float64) + 1j * np.asarray(q_s, np.float64)
    if peak is not None:
        x = x * (0.5 / float(peak))
    starts = (512 * np.arange(92)[:, None] + 256 * np.arange(2)[None, :]).reshape(-1)
    frames = x[starts[:, None] + np.arange(1024)[None, :]] * np.asarray(window, np.float64)[None, :]
    X = np.fft.fft(frames, axis=1)
    p2 = X.real ** 2 + X.imag ** 2
    top = p2.max(axis=1, keepdims=True)
    p2 = p2[:, :512].reshape(92, 2, 256, 2).transpose(0, 1, 3, 2)         # [blk, ts, fs, b]
    q = quantise(1e-12 + p2 * 4.0 / 2.0 ** 20).reshape(-1)
    if not resolvable:
        return q
    return q, (p2 >= RESOLVABLE * top.reshape(92, 2, 1, 1)).reshape(-1)


def monitor_geometry(sample_rate, time_osr, freq_osr, protocol):
    period = np.float32(0.048 if protocol == 0 else 0.160)
    block = int(np.float32(sample_rate) * period)
    return dict(block=block, hop=block // time_osr, nfft=block * freq_osr, num_bins=int(np.float32(sample_rate) * period / 2),
                max_blocks=int(np.float32(7.5 if protocol == 0 else 15.0) / period))


def monitor_waterfall(audio, sample_rate=12000, time_osr=2, freq_osr=2, protocol=1, resolvable=False):
    """ft8_lib's monitor (decode_ft8.c:35-39, 162-218) in float64: Hann (sin^2) window over the last nfft samples (history
    starts at zero), fft_norm = 2 / nfft, real FFT, cell (blk, ts, fs, b) = bin b freq_osr + fs, x = 1e-12 + |X|^2.
    -> (uint8 cells flattened, num_blocks, max over the cells of 10 log10(x), floored at -120[, resolvable cells])."""
    g = monitor_geometry(sample_rate, time_osr, freq_osr, protocol)
    a = np.asarray(audio, np.float64)
    nb = min(g["max_blocks"], a.size // g["block"])
    nfft, hop = g["nfft"], g["hop"]
    padded = np.r_[np.zeros(nfft), a]
    ends = nfft + hop * (np.arange(nb * time_osr) + 1)
    frames = padded[ends[:, None] - nfft + np.arange(nfft)[None, :]]
    win = np.sin(np.pi * np.arange(nfft) / nfft) ** 2
    X = np.fft.rfft(frames * win[None, :] * (2.0 / nfft), axis=1)
    top = (X.real ** 2 + X.imag ** 2).max(axis=1).reshape(nb, time_osr, 1, 1)
    X = X[:, : g["num_bins"] * freq_osr].reshape(nb, time_osr, g["num_bins"], freq_osr).transpose(0, 1, 3, 2)
    p2 = X.real ** 2 + X.imag ** 2
    x = 1e-12 + p2
    max_db = max(-120.0, float(10.0 * np.log10(x).max())) if nb else -120.0
    q = quantise(x).reshape(-1)
    if not resolvable:
        return q, nb, max_db
    return q, nb, max_db, (p2 >= RESOLVABLE * top).reshape(-1)


# ---- sync scores (ft8_lib decode.c:35-171) ----------------------------------------------------------------------------
def sync_scores(mag, num_blocks, num_bins, time_osr, freq_osr, protocol=1):
    """Score of every position, exact integers: int16 [time_osr, freq_osr, 36 (to = -12 .. 23), num_bins - 7], in the
    reference's loop order when flattened.  Each Costas symbol adds a - neighbour for the tone below and above (when that
    tone exists) and the same bin one symbol earlier and later (inside the group and inside the waterfall); rows below 0
    are skipped, a row >= num_blocks ends its group; the sum is divided by the number of terms, truncating toward zero."""
    P = np.asarray(mag, np.int64)[: num_blocks * time_osr * freq_osr * num_bins].reshape(num_blocks, time_osr, freq_osr, num_bins)
    P = P.transpose(1, 2, 0, 3)                                         # [ts, fs, row, bin]
    nfo = num_bins - 7
    fo = np.arange(nfo)
    if protocol == 1:
        groups = [(g0, FT8_COSTAS, 8) for g0 in FT8_SYNC_AT]
    else:
        groups = [(g0, FT4_COSTAS[k], 4) for k, g0 in enumerate(FT4_SYNC_AT)]
    out = np.zeros((time_osr, freq_osr, 36, nfo), np.int16)
    for ti, to in enumerate(range(-12, 24)):
        total = np.zeros((time_osr, freq_osr, nfo), np.int64)
        terms = 0
        for g0, costas, ntones in groups:
            for k, tone in enumerate(costas):
                row = to + g0 + k
                if row < 0:
                    continue
                if row >= num_blocks:
                    break
                a = P[:, :, row, fo + tone]
                if tone > 0:
                    total += a - P[:, :, row, fo + tone - 1]; terms += 1
                if tone < ntones - 1:
                    total += a - P[:, :, row, fo + tone + 1]; terms += 1
                if k > 0 and row > 0:
                    total += a - P[:, :, row - 1, fo + tone]; terms += 1
                if k + 1 < len(costas) and row + 1 < num_blocks:
                    total += a - P[:, :, row + 1, fo + tone]; terms += 1
        if terms:
            total = np.sign(total) * (np.abs(total) // terms)
        out[:, :, ti, :] = total.astype(np.int16)
    return out


# ---- LLRs (ft8_lib decode.c:265-314) ----------------------------------------------------------------------------------
def llrs(mag, cand, num_blocks, num_bins, time_osr, freq_osr, protocol=1):
    """Max-log demapper over the Gray-mapped tones (FT8 58 x 3 bits, FT4 87 x 2), 0 for symbols outside the waterfall, then
    normalised: var over the 174 values, gain sqrt(24 / var) (NaN everywhere when var = 0).  -> (float64 [174], var)."""
    P = np.asarray(mag, np.float64)[: num_blocks * time_osr * freq_osr * num_bins].reshape(num_blocks, time_osr, freq_osr, num_bins)
    to, fo, ts, fs = int(cand["time_offset"]), int(cand["freq_offset"]), int(cand["time_sub"]), int(cand["freq_sub"])
    if protocol == 1:
        data, gray, nbits = FT8_DATA, FT8_GRAY, 3
    else:
        data, gray, nbits = FT4_DATA, FT4_GRAY, 2
    out = np.zeros((data.size, nbits))
    for k, sym in enumerate(data):
        row = to + sym
        if row < 0 or row >= num_blocks:
            continue
        s = P[row, ts, fs, fo + gray]                                   # s[j] = power of the tone that carries bits j
        for i in range(nbits):
            one = (np.arange(2 ** nbits) >> (nbits - 1 - i)) & 1
            out[k, i] = s[one == 1].max() - s[one == 0].max()
    x = out.reshape(-1)
    var = (np.sum(x * x) - np.sum(x) ** 2 / 174.0) / 174.0
    with np.errstate(divide="ignore", invalid="ignore"):
        return x * np.sqrt(24.0 / var), var


# ---- channel symbols --------------------------------------------------------------------------------------------------
def bits_from_tones(tones, protocol=1):
    """Gray-decode the data symbols of a tone sequence -> 174 bits (MSB of each symbol first)."""
    t = np.asarray(tones, np.int64)
    if protocol == 1:
        data, gray, nbits = t[FT8_DATA], FT8_GRAY, 3
    else:
        data, gray, nbits = t[FT4_DATA], FT4_GRAY, 2
    inv = np.argsort(gray)                                              # tone -> bits
    v = inv[data]
    return ((v[:, None] >> np.arange(nbits - 1, -1, -1)[None, :]) & 1).reshape(-1)


def descramble77(bits174):
    """FT4: the 77 message bits of a codeword XOR the scrambling vector -> 10 payload bytes (last 3 bits zero)."""
    b = np.asarray(bits174[:77], np.uint8) ^ np.unpackbits(np.frombuffer(FT4_XOR, np.uint8))[:77]
    return np.packbits(np.r_[b, np.zeros(3, np.uint8)]).tobytes()


def costas_positions(protocol=1):
    """{symbol index: tone} of the sync symbols."""
    if protocol == 1:
        return {g0 + k: int(t) for g0 in FT8_SYNC_AT for k, t in enumerate(FT8_COSTAS)}
    return {g0 + k: int(t) for grp, g0 in enumerate(FT4_SYNC_AT) for k, t in enumerate(FT4_COSTAS[grp])}


# ---- synthesis --------------------------------------------------------------------------------------------------------
def gfsk_phase(tones, sym_len, fs, f0, spacing, bt):
    """Continuous-phase GFSK (gen_ft8.c:28-102) in float64: the frequency of symbol i is smoothed by the erf pulse
    (three symbols long, bandwidth-time product bt), the first and last symbol are extended by a copy of themselves, and the
    phase is the running sum of the per-sample phase steps from 0.  -> (phase [n_sym sym_len], envelope of the same length:
    raised-cosine ramps over the first and last eighth of a symbol)."""
    t = np.asarray(tones, np.float64)
    n_sym, L = t.size, sym_len
    j = np.arange(3 * L)
    tt = j / L - 1.5
    c = np.pi * np.sqrt(2.0 / np.log(2.0))
    from scipy.special import erf
    pulse = (erf(c * bt * (tt + 0.5)) - erf(c * bt * (tt - 0.5))) / 2.0
    dphi = np.full((n_sym + 2) * L, 2 * np.pi * f0 / fs)
    ext = np.r_[t[0], t, t[-1]]                                         # symbol i of ext starts at (i - 1) L in dphi
    peak = 2 * np.pi * spacing / fs
    for i, tone in enumerate(ext):
        lo = (i - 1) * L
        a, b = max(lo, 0), min(lo + 3 * L, dphi.size)
        dphi[a:b] += peak * tone * pulse[a - lo:b - lo]
    steps = dphi[L:L + n_sym * L]
    phase = np.r_[0.0, np.cumsum(steps[:-1])]
    env = np.ones(n_sym * L)
    n_ramp = L // 8
    r = (1 - np.cos(2 * np.pi * np.arange(n_ramp) / (2 * n_ramp))) / 2
    env[:n_ramp] = r
    env[n_sym * L - 1 - np.arange(n_ramp)] = r
    return phase, env
