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
