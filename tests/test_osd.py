"""Ordered-statistics decoding (OSD): the CPU restatement orc_osd (tests/support/osd_oracle.c) against an independent numpy
implementation of the definition (DESIGN.md section 2.4.1).  The reference has no OSD, so this is what pins the restatement; the
GPU kernel is then held to it byte for byte (tests/test_gpu_osd.py).  No GPU needed."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from oracle.pyoracle import WF_BYTES, Oracle, SlotReport, _ptr, cand_dtype, make_wf, msg_dtype, result_dtype, status_dtype

N, K, M = 174, 91, 83


def _table(name, rows):
    src = open(os.path.join(ROOT, "oracle", "ft8_tables.h")).read()
    body = src[src.index(name):]
    body = body[body.index("{") + 1:body.index("};")]
    vals = [int(v, 0) for v in re.findall(r"0x[0-9a-fA-F]+|\d+", body)]
    return np.array(vals, np.int64).reshape(rows, -1)


GEN = _table("kFt8tGen[83][12]", 83)
NM = _table("kFt8tNm[83][7]", 83)
FT4_XOR = bytes(int(v) for v in _table("kFt4tXor[10]", 10).ravel())
# G = [I_91 | P]: row k is the codeword of message bit k
P = np.array([[(GEN[r][k >> 3] >> (7 - (k & 7))) & 1 for r in range(M)] for k in range(K)], np.uint8)
G = np.concatenate([np.eye(K, dtype=np.uint8), P], axis=1)
H = np.zeros((M, N), np.uint8)
for r in range(M):
    for v in NM[r]:
        if v:
            H[r, v - 1] = 1


def crc14(bits82):
    """CRC-14, polynomial 0x2757, MSB first, over 82 bits (the 77 message bits and 5 zeros)."""
    rem = 0
    for b in bits82:
        rem = ((rem << 1) | int(b))
        if rem & 0x4000:
            rem ^= 0x4000 | 0x2757
    for _ in range(14):
        rem <<= 1
        if rem & 0x4000:
            rem ^= 0x4000 | 0x2757
    return rem & 0x3FFF


def gf2_inv(a):
    n = a.shape[0]
    m = np.concatenate([a.copy(), np.eye(n, dtype=np.uint8)], axis=1)
    for c in range(n):
        piv = c + int(np.flatnonzero(m[c:, c])[0])
        m[[c, piv]] = m[[piv, c]]
        rows = np.flatnonzero(m[:, c])
        rows = rows[rows != c]
        m[rows] ^= m[c]
    return m[:, n:]


def ref_osd(llr, order, max_hard, oracle, protocol=1):
    """The definition, independently: (accepted -1/0/1, codeword, hard distance, D)."""
    llr = np.asarray(llr, np.float32)
    if order == 0 or not np.all(np.isfinite(llr)):
        return -1, None, None, None
    mag = llr.view(np.uint32) & 0x7FFFFFFF
    perm = np.lexsort((np.arange(N), -mag.astype(np.int64)))  # |llr| descending, then index ascending
    h = (llr > 0).astype(np.uint8)
    q = (np.minimum(np.abs(llr), np.float32(255.0)) * np.float32(256.0)).astype(np.uint32).astype(np.int64)
    basis, mrb = {}, []  # xor basis of the columns taken so far, keyed by leading bit
    for col in perm:
        v = int("".join(map(str, G[:, col])), 2)
        while v:
            top = v.bit_length() - 1
            if top not in basis:
                basis[top] = v
                mrb.append(int(col))
                break
            v ^= basis[top]
        if len(mrb) == K:
            break
    mrb = np.array(mrb)
    ainv = gf2_inv(G[:, mrb].T.copy())  # message m = A^-1 u for MRB values u: G[:, mrb]^T m = u
    u0 = h[mrb]
    pats = [u0.copy()]
    for t in range(K):
        u = u0.copy(); u[t] ^= 1; pats.append(u)
    if order == 2:
        lo = np.arange(K - 32, K)
        for i in range(32):
            for j in range(i + 1, 32):
                u = u0.copy(); u[lo[i]] ^= 1; u[lo[j]] ^= 1; pats.append(u)
    U = np.array(pats, np.int64)
    msgs = (ainv.astype(np.int64) @ U.T % 2).T
    cws = (msgs @ G.astype(np.int64) % 2).astype(np.uint8)
    d = (cws != h) @ q
    win = int(np.argmin(d))  # first minimum = lower pattern index
    cw = cws[win]
    hard = int(np.sum(cw != h))
    msg = cw[:77]
    ok = hard <= max_hard and crc14(np.concatenate([msg, np.zeros(5, np.uint8)])) == int("".join(map(str, cw[77:91])), 2)
    if ok:
        a = np.packbits(np.concatenate([msg, np.zeros(3, np.uint8)])).tobytes()
        if protocol == 0:
            a = bytes(x ^ y for x, y in zip(a, FT4_XOR))
        a = a[:9] + bytes([a[9] & 0xF8])
        ok = oracle.unpack77(a)[0] >= 0
    return int(ok), cw, hard, int(d[win])


class OsdOracle(Oracle):
    """The oracle plus the OSD restatement: tests/support/osd_oracle.c compiled with the oracle's sources and flags."""

    def __init__(self, workdir):
        super().__init__()
        srcs = [os.path.join(ROOT, "tests", "support", "osd_oracle.c")] + \
            [os.path.join(ROOT, "oracle", f) for f in ("ft8_oracle.c", "ft8_oracle_codec.c", "ft8_oracle_synth.c", "ft8_oracle_report.c")]
        so = os.path.join(str(workdir), "libosdoracle.so")
        subprocess.check_call([os.environ.get("CC", "gcc"), "-O3", "-std=gnu17", "-ffp-contract=off", "-fwrapv", "-fPIC", "-w", "-shared",
                               "-I" + os.path.join(ROOT, "oracle"), "-o", so] + srcs + ["-lm"])
        self.osd_lib = C.CDLL(so)

    def osd(self, llr, order, max_hard, protocol=1):
        """orc_osd -> (accepted: -1 not attempted / 0 / 1, codeword uint8[174], hard distance, metric D)."""
        llr = np.ascontiguousarray(llr, np.float32)
        cw = np.zeros(174, np.uint8)
        hard, dist = C.c_int(0), C.c_uint32(0)
        acc = self.osd_lib.orc_osd(_ptr(llr), int(order), int(max_hard), int(protocol), _ptr(cw), C.byref(hard), C.byref(dist))
        return int(acc), cw, hard.value, dist.value

    def decode_osd(self, mag, cand, order, max_hard, max_iters=20, **dims):
        """orc_decode_osd -> decode()'s dict plus osd (0 not attempted, 1 rejected, 2 decoded) and osd_hard."""
        wf = make_wf(mag, **dims)
        c = np.array([cand], cand_dtype)
        msg = np.zeros(1, msg_dtype)
        st = np.frombuffer(bytes([0xA5]) * 12, status_dtype).copy()
        llr = np.zeros(174, np.float32)
        plain = np.zeros(174, np.uint8)
        osd, hard = C.c_uint8(0), C.c_int(0)
        ok = self.osd_lib.orc_decode_osd(C.byref(wf), _ptr(c), max_iters, int(order), int(max_hard), _ptr(msg), _ptr(st), _ptr(llr),
                                         _ptr(plain), C.byref(osd), C.byref(hard))
        return dict(ok=int(ok), msg=msg[0], status=st[0], llr=llr, plain=plain, osd=osd.value, osd_hard=hard.value)

    def subsystem_osd(self, i_s, q_s, order, max_hard, max_cand=120, max_msgs=50, min_score=10, iters=20):
        """orc_subsystem_osd: subsystem() with OSD where BP stopped at stage 1 or 2."""
        i_s = np.ascontiguousarray(i_s, np.float32)
        q_s = np.ascontiguousarray(q_s, np.float32)
        res = np.zeros(max_msgs, result_dtype)
        rep = SlotReport()
        wf = np.zeros(WF_BYTES, np.uint8)
        cands = np.zeros(max_cand, cand_dtype)
        n = self.osd_lib.orc_subsystem_osd(_ptr(i_s), _ptr(q_s), max_cand, max_msgs, min_score, iters, int(order), int(max_hard), _ptr(res),
                                           C.byref(rep), _ptr(wf), _ptr(cands))
        return self._slot_dict(n, res, rep, cands, wf)

    def decode_waterfall_osd(self, mag, order, max_hard, max_cand=120, max_msgs=50, min_score=10, iters=20, **dims):
        wf = make_wf(mag, **dims)
        res = np.zeros(max_msgs, result_dtype)
        rep = SlotReport()
        cands = np.zeros(max_cand, cand_dtype)
        n = self.osd_lib.orc_decode_waterfall_osd(C.byref(wf), max_cand, max_msgs, min_score, iters, int(order), int(max_hard), _ptr(res),
                                                  C.byref(rep), _ptr(cands))
        return self._slot_dict(n, res, rep, cands, mag)


@pytest.fixture(scope="module")
def oracle(tmp_path_factory):
    """Overrides the session oracle in the OSD test modules: the same restatement plus the OSD forms."""
    return OsdOracle(tmp_path_factory.mktemp("osd_oracle"))


def codeword(oracle, rng):
    payload = bytes(rng.integers(0, 256, 10, dtype=np.uint8))
    return oracle.encode174(payload)


def fuzz_llrs(oracle, n, seed):
    """n LLR vectors: Gaussian noise, noisy codewords, a few magnitudes (ties), +-0, and an early dependent column."""
    rng = np.random.default_rng(seed)
    out = []
    for k in range(n):
        kind = k % 5
        if kind == 0:
            x = rng.normal(0, 2.5, N)
        elif kind == 1:  # a codeword through noise: most winners pass the CRC
            c = codeword(oracle, rng).astype(np.float64)
            x = (2 * c - 1) * rng.uniform(1.0, 3.0) + rng.normal(0, rng.uniform(0.8, 2.2), N)
        elif kind == 2:  # few magnitudes: ties everywhere
            c = codeword(oracle, rng).astype(np.float64)
            flip = rng.random(N) < rng.uniform(0.0, 0.15)
            x = np.where(flip, 1 - 2 * c, 2 * c - 1) * rng.choice([0.5, 1.0, 2.0, 4.0], N)
        elif kind == 3:  # +0 and -0 among them
            x = rng.normal(0, 3.0, N)
            z = rng.random(N) < 0.2
            x[z] = np.where(rng.random(int(z.sum())) < 0.5, 0.0, -0.0)
        else:  # parity column 91 + r right behind the message bits it depends on: dependent early in the order
            r = int(rng.integers(0, M))
            x = rng.normal(0, 1.0, N)
            dep = np.flatnonzero(P[:, r])
            x[dep] = np.sign(rng.normal(size=dep.size)) * rng.uniform(20, 30, dep.size)
            x[K + r] = 19.0 * (1 if rng.random() < 0.5 else -1)
        out.append(np.asarray(x, np.float32))
    return np.array(out, np.float32)


@pytest.mark.parametrize("order", [1, 2])
def test_restatement_equals_independent_implementation(oracle, order):
    llrs = fuzz_llrs(oracle, 1000, 7 + order)
    accepted = 0
    for cap in (10, 26, 174):
        for x in (llrs if cap == 26 else llrs[::4]):
            got = oracle.osd(x, order, cap)
            want = ref_osd(x, order, cap, oracle)
            assert got[0] == want[0]
            assert np.array_equal(got[1], want[1]) and got[2] == want[2] and got[3] == want[3]
            accepted += got[0] == 1
    assert accepted > 50  # the acceptance path is exercised, not only rejections


def test_restatement_ft4_descrambles_before_unpacking(oracle):
    llrs = fuzz_llrs(oracle, 300, 99)
    for x in llrs:
        for proto in (0, 1):
            got = oracle.osd(x, 1, 40, proto)
            want = ref_osd(x, 1, 40, oracle, proto)
            assert got[0] == want[0] and np.array_equal(got[1], want[1])


def test_every_winner_is_a_codeword(oracle):
    for x in fuzz_llrs(oracle, 400, 3):
        acc, cw, _, _ = oracle.osd(x, 2, 174)
        assert acc >= 0 and not np.any(H.astype(np.int64) @ cw % 2), "winner violates a parity check of kFt8tNm"


@pytest.mark.parametrize("order,flips", [(1, 1), (2, 2)])
def test_errors_in_the_least_reliable_basis_positions_are_corrected(oracle, order, flips):
    rng = np.random.default_rng(order)
    for _ in range(50):
        c = codeword(oracle, rng)
        x = ((2 * c.astype(np.float32) - 1) * rng.uniform(3.0, 6.0, N)).astype(np.float32)
        # the MRB is decided by magnitudes alone: find it, then flip the signs of its least reliable positions, keeping them there
        mag = x.view(np.uint32) & 0x7FFFFFFF
        perm = np.lexsort((np.arange(N), -mag.astype(np.int64)))
        basis, mrb = {}, []
        for col in perm:
            v = int("".join(map(str, G[:, col])), 2)
            while v:
                top = v.bit_length() - 1
                if top not in basis:
                    basis[top] = v; mrb.append(int(col)); break
                v ^= basis[top]
            if len(mrb) == K:
                break
        bad = rng.choice(mrb[K - 32:], flips, replace=False)
        x[bad] = -x[bad]
        acc, cw, hard, _ = oracle.osd(x, order, 174)
        assert acc >= 0 and np.array_equal(cw, c) and hard == flips


def test_non_finite_llrs_are_not_attempted(oracle):
    x = fuzz_llrs(oracle, 3, 5)[1]
    for bad in (np.nan, np.inf, -np.inf):
        y = x.copy(); y[17] = bad
        assert oracle.osd(y, 1, 174)[0] == -1 and oracle.osd(y, 2, 174)[0] == -1
    assert oracle.osd(x, 0, 174)[0] == -1


def test_order_zero_forms_equal_the_plain_decoder(oracle):
    from tools import ft8enc, synth
    sig = [(ft8enc.tones(ft8enc.pack_std("CQ", "K1JT", "FN20")), 700.0, 0.5, -21.0),
           (ft8enc.tones(ft8enc.pack_std("CQ", "W1AW", "FN31")), 1200.0, 1.1, -14.0)]
    i_s, q_s = synth.slot_f32(sig, 11)
    i_s, q_s, _ = oracle.condition(i_s, q_s, 48000)
    a, b = oracle.subsystem(i_s, q_s), oracle.subsystem_osd(i_s, q_s, 0, 0)
    assert a["n"] == b["n"] and a["results"].tobytes() == b["results"].tobytes() and a["msgs"].tobytes() == b["msgs"].tobytes()
    for c in a["cands"][:40]:
        d, e = oracle.decode(a["wf"], c), oracle.decode_osd(a["wf"], c, 0, 0)
        assert d["ok"] == e["ok"] and d["status"].tobytes() == e["status"].tobytes() and np.array_equal(d["plain"], e["plain"])
        assert e["osd"] == 0 and e["osd_hard"] == -1
