"""The generated protocol tables (csrc/ft8_tables.h, and the oracle's copy) against the FT8/FT4 definitions written out in
tests/ref64.py and the LDPC source text tools/ldpc_174_91_nm.txt -- not against anything derived from the header itself.
No GPU needed."""
import os
import re

import numpy as np
import pytest

import ref64

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADERS = [os.path.join(ROOT, "rtlsdr-ft8d_b200", "csrc", "ft8_tables.h"), os.path.join(ROOT, "oracle", "ft8_tables.h")]


def header_array(path, name):
    """Integer values of `static const uint8_t <name>[...] = {...};` in file order."""
    with open(path) as f:
        text = f.read()
    m = re.search(r"\b%s\s*(\[[^=]*)=\s*\{(.*?)\};" % re.escape(name), text, re.S)
    assert m, f"{name} not found in {path}"
    dims = [int(d) for d in re.findall(r"\[(\d+)\]", m.group(1))]
    vals = [int(v, 0) for v in re.findall(r"0x[0-9a-fA-F]+|\d+", m.group(2))]
    return np.array(vals).reshape(dims)


@pytest.fixture(scope="module", params=HEADERS, ids=["csrc", "oracle"])
def header(request):
    return request.param


def test_crc14_matches_the_reference():
    """The independent CRC-14 against the value the unmodified reference computed (kat.npz["crc_test3"])."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "kat.npz"))
    assert ref64.crc14_bytes(bytes([0x11, 0, 0, 0, 0, 0x0E, 0x10, 0x04, 0x01, 0x00, 0, 0]), 76) == int(g["crc_test3"][0])


def test_ldpc_source_text_shape():
    """Every variable is in exactly 3 checks; 24 checks have weight 7 and 59 weight 6; no variable twice in a check."""
    nm = ref64.ldpc_checks()
    assert nm.shape == (83, 7)
    w = (nm >= 0).sum(axis=1)
    assert (w == 7).sum() == 24 and (w == 6).sum() == 59
    H = ref64.parity_matrix()
    assert (H.sum(axis=0) == 3).all() and H.sum() == (nm >= 0).sum()


def test_check_rows_equal_the_source_text(header):
    nm_txt = ref64.ldpc_checks() + 1                      # back to 1-origin, 0 = unused
    assert np.array_equal(header_array(header, "kFt8tNm"), nm_txt)
    assert np.array_equal(header_array(header, "kFt8tNumRows"), (nm_txt > 0).sum(axis=1))


def test_variable_lists_are_the_transpose(header):
    """kFt8tMn[n] lists, in ascending order, the 3 checks variable n takes part in."""
    H = ref64.parity_matrix()
    mn = header_array(header, "kFt8tMn")
    assert mn.shape == (174, 3)
    want = np.array([np.flatnonzero(H[:, n]) + 1 for n in range(174)])
    assert np.array_equal(mn, want)


def test_generator_satisfies_every_check(header):
    """G H^T = 0 over GF(2): the codeword of every unit message (bit j set, parity = bit j of each generator row) passes all
    83 checks, and the parity part has full rank (so the code is the one the checks define)."""
    gen = header_array(header, "kFt8tGen").astype(np.uint8)
    par = np.unpackbits(gen, axis=1)[:, :91]             # [83 parity bits, 91 message bits], MSB first
    G = np.concatenate([np.eye(91, dtype=np.uint8), par.T], axis=1)   # [91, 174] systematic generator
    H = ref64.parity_matrix()
    assert not ((G.astype(np.int64) @ H.T.astype(np.int64)) % 2).any()
    assert ref64.checks_satisfied(G).all()


def test_costas_and_gray_are_the_published_constants(header):
    assert np.array_equal(header_array(header, "kFt8tCostas"), ref64.FT8_COSTAS)
    assert np.array_equal(header_array(header, "kFt8tGray"), ref64.FT8_GRAY)
    assert np.array_equal(header_array(header, "kFt4tCostas"), ref64.FT4_COSTAS)
    assert np.array_equal(header_array(header, "kFt4tGray"), ref64.FT4_GRAY)
    assert bytes(header_array(header, "kFt4tXor").astype(np.uint8)) == ref64.FT4_XOR


def test_kernel_copies_of_the_constants():
    """Two kernels spell the Costas arrays and the FT8 Gray map out instead of including the header."""
    with open(os.path.join(ROOT, "rtlsdr-ft8d_b200", "csrc", "sync.cu")) as f:
        sync = f.read()
    c8 = re.findall(r"kCostas8\[7\]\s*=\s*\{([^}]*)\}", sync)
    assert c8 and all([int(v) for v in c.split(",")] == list(ref64.FT8_COSTAS) for c in c8)
    c4 = re.findall(r"kCostas4\[4\]\[4\]\s*=\s*\{(.*?)\};", sync, re.S)
    assert c4 and all(np.array_equal(np.array([int(v) for v in re.findall(r"\d+", c)]).reshape(4, 4), ref64.FT4_COSTAS) for c in c4)
    with open(os.path.join(ROOT, "rtlsdr-ft8d_b200", "csrc", "decode.cu")) as f:
        dec = f.read()
    g8 = re.findall(r"c_gray\[8\]\s*=\s*\{([^}]*)\}", dec)
    assert g8 and [int(v) for v in g8[0].split(",")] == list(ref64.FT8_GRAY)


def test_channel_symbol_layout():
    """The layout constants themselves: 58 FT8 / 87 FT4 data symbols that, with the sync symbols, tile 79 / 103 symbols
    (FT4 adds a ramp symbol at each end: 105)."""
    s8 = set(ref64.costas_positions(1))
    assert len(ref64.FT8_DATA) * 3 == 174 and s8.isdisjoint(ref64.FT8_DATA) and s8 | set(ref64.FT8_DATA) == set(range(79))
    s4 = set(ref64.costas_positions(0))
    assert len(ref64.FT4_DATA) * 2 == 174 and s4.isdisjoint(ref64.FT4_DATA) and s4 | set(ref64.FT4_DATA) == set(range(1, 104))


# ---- belief propagation: Pade constants and the oracle's decoder against float64 ------------------------------------------
def _pade_forms(path):
    """{function name: (numerator, denominator, clamp or None)} of every tanh/atanh Pade form in a source file: the C
    expressions of `a` and `b` evaluated on polynomials in x (so __fmul_rn / __fadd_rn nesting and implicit 1 coefficients
    read as written), coefficients ascending in powers of x."""
    P = np.polynomial.Polynomial
    with open(path) as f:
        text = f.read()
    out = {}
    for m in re.finditer(r"float\s+(a?tanh_(?:inl|pade))\s*\(([^)]*)\)\s*\{(.*?)\n\}", text, re.S):
        name, body = m.group(1), m.group(3)
        x = P([0.0, 1.0])
        env = {"x": x, "x2": x * x, "__fmul_rn": lambda p, q: p * q, "__fadd_rn": lambda p, q: p + q}
        poly = []
        for var in ("a", "b"):
            expr = re.search(r"const float %s = (.*?);" % var, body, re.S).group(1)
            poly.append(tuple(int(round(c)) for c in eval(re.sub(r"(\d+\.\d*)f\b", r"\1", expr), env).coef))
        lo = re.findall(r"x\s*<\s*-(\d+\.\d+)f", body)
        hi = re.findall(r"x\s*>\s*(\d+\.\d+)f", body)
        out[name] = (poly[0], poly[1], (float(lo[0]), float(hi[0])) if lo else None)
    return out


@pytest.mark.parametrize("path", ["rtlsdr-ft8d_b200/csrc/decode.cu", "oracle/ft8_oracle_codec.c"])
def test_pade_constants_vs_taylor_series(path):
    """fast_tanh / fast_atanh in the kernels (the inlined and the plain forms) and in the oracle are the [5/4] Pade
    approximants derived here from the Taylor series: x(945 + 105x^2 + x^4)/(945 + 420x^2 + 15x^4) and
    x(945 - 735x^2 + 64x^4)/(945 - 1050x^2 + 225x^4); tanh is clamped to -+1 beyond 4.97."""
    tanh, atanh = ref64.pade_coefficients("tanh"), ref64.pade_coefficients("atanh")
    assert tanh == ((0, 945, 0, 105, 0, 1), (945, 0, 420, 0, 15)) and atanh == ((0, 945, 0, -735, 0, 64), (945, 0, -1050, 0, 225))
    forms = _pade_forms(os.path.join(ROOT, path))
    want = {"tanh_pade", "atanh_pade"} | ({"tanh_inl", "atanh_inl"} if path.endswith(".cu") else set())
    assert set(forms) == want, sorted(forms)
    for name, (num, den, clamp) in forms.items():
        ref = atanh if name.startswith("atanh") else tanh
        assert (num, den) == ref, (name, num, den)
        assert clamp == (None if name.startswith("atanh") else (ref64.TANH_CLAMP, ref64.TANH_CLAMP)), (name, clamp)


def test_oracle_bp_vs_float64(oracle):
    """orc_bp_decode (bit-equal to both BP kernels) against ref64.bp_decode64 under the agreement rule, on noisy codewords,
    Gaussian noise, few magnitudes (ties), +-0 and saturated values, at n = 0 .. 100 rounds.

    Calibration of the rule (ref64.TAU, TAU_LONG, LONG_ROUNDS), measured here and on the daemon slots of tests/test_gpu_bp.py:
    - 1000 of these vectors x 9 counts: the oracle's plain and ldpc_errors equal float64's for all 9000 pairs, resolved or
      not.  The vectors with +-0 give exact-zero posteriors, which no margin resolves.  Here (409 vectors x 9 counts) 76 % of
      the pairs are resolved, 87 % of those with n <= 5.
    - 569 find_sync candidates of six daemon slots x 14 counts: every pair agrees up to n = 50; at n = 100, 5 candidates whose
      float64 run never converges end on a different hard decision (same ldpc_errors), with posteriors no closer to zero than
      6e-4 x max|llr|.  Hence TAU_LONG = 1e-2 from round 51 on.  Resolved: 83 % of all pairs, 93 % of those with n <= 5."""
    from test_osd import fuzz_llrs
    llrs = fuzz_llrs(oracle, 400, 3)
    sat = np.where(np.arange(174) % 3 == 0, 1e30, -3.0).astype(np.float32) * np.where(np.arange(174) % 2, 1, -1)
    llrs = np.concatenate([llrs, sat[None], np.float32(np.sign(llrs[1::50]) * 30.0)])
    traj = ref64.bp_decode64(llrs, 100)
    pairs = resolved = pairs_small = resolved_small = 0
    for n in (0, 1, 2, 3, 5, 10, 20, 50, 100):
        plain, errors, margin = ref64.bp_resolved(traj, llrs, n)
        for c in range(llrs.shape[0]):
            op, oe = oracle.bp_decode(llrs[c], n)
            if margin[c] >= 1:
                assert np.array_equal(op, plain[c]) and oe == errors[c], (n, c, oe, int(errors[c]), float(margin[c]))
            pairs += 1; resolved += margin[c] >= 1
            if n <= 5:
                pairs_small += 1; resolved_small += margin[c] >= 1
    print(f"\n[bp] oracle vs float64: resolved {resolved}/{pairs}, n <= 5: {resolved_small}/{pairs_small}")
    assert resolved >= 0.7 * pairs and resolved_small >= 0.75 * pairs_small
    assert (traj["stop"] == 1).any() and ((traj["stop"] > 1) & ~traj["zero"]).any() and (traj["stop"] == 0).any()
