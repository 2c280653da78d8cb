"""A-priori (AP) decoding of "CQ ??? ???": the CPU restatement orc_ap (tests/support/ap_oracle.c) against an independent numpy
implementation of the definition's forcing and acceptance steps (DESIGN.md section 2.4.3; BP itself is orc_bp_decode, pinned
elsewhere), the hypothesis against the encoder, and constructed cases.  The GPU kernel is then held to orc_ap byte for byte
(tests/test_gpu_ap.py).  No GPU needed."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from oracle.pyoracle import WF_BYTES, _ptr, cand_dtype, make_wf, msg_dtype, result_dtype, status_dtype
from test_osd import FT4_XOR, H, OsdOracle, codeword, crc14
from tools import ft8enc, synth

N = 174
KNOWN = np.r_[0:29, 74:77]
NTOK, MAX22 = 2063592, 4194304


class ApOracle(OsdOracle):
    """The OSD oracle plus the AP restatement: tests/support/ap_oracle.c (which includes osd_oracle.c) with the oracle's sources."""

    def __init__(self, workdir):
        super().__init__(workdir)
        srcs = [os.path.join(ROOT, "tests", "support", "ap_oracle.c")] + \
            [os.path.join(ROOT, "oracle", f) for f in ("ft8_oracle.c", "ft8_oracle_codec.c", "ft8_oracle_synth.c", "ft8_oracle_report.c")]
        so = os.path.join(str(workdir), "libaporacle.so")
        subprocess.check_call([os.environ.get("CC", "gcc"), "-O3", "-std=gnu17", "-ffp-contract=off", "-fwrapv", "-fPIC", "-w", "-shared",
                               "-I" + os.path.join(ROOT, "oracle"), "-I" + os.path.join(ROOT, "tests", "support"), "-o", so] + srcs + ["-lm"])
        self.ap_lib = C.CDLL(so)

    def hypothesis(self, protocol=1):
        mask, val = np.zeros(N, np.uint8), np.zeros(N, np.uint8)
        self.ap_lib.orc_ap_hypothesis(int(protocol), _ptr(mask), _ptr(val))
        return mask, val

    def ap(self, llr, max_hard, protocol=1, max_iters=20):
        """orc_ap -> (accepted: -1 not attempted / 0 / 1, BP's final word uint8[174], hard distance)."""
        llr = np.ascontiguousarray(llr, np.float32)
        cw = np.zeros(N, np.uint8)
        hard = C.c_int(0)
        acc = self.ap_lib.orc_ap(_ptr(llr), int(max_iters), int(max_hard), int(protocol), _ptr(cw), C.byref(hard))
        return int(acc), cw, hard.value

    def decode_ap(self, mag, cand, osd_order, osd_max_hard, ap_on, ap_max_hard, max_iters=20, **dims):
        """orc_decode_ap -> decode()'s dict plus osd / osd_hard and ap (0 not attempted, 1 rejected, 2 decoded) / ap_hard."""
        wf = make_wf(mag, **dims)
        c = np.array([cand], cand_dtype)
        msg = np.zeros(1, msg_dtype)
        st = np.frombuffer(bytes([0xA5]) * 12, status_dtype).copy()
        llr = np.zeros(N, np.float32)
        plain = np.zeros(N, np.uint8)
        osd, ohard, ap, ahard = C.c_uint8(0), C.c_int(0), C.c_uint8(0), C.c_int(0)
        ok = self.ap_lib.orc_decode_ap(C.byref(wf), _ptr(c), max_iters, int(osd_order), int(osd_max_hard), int(ap_on), int(ap_max_hard), _ptr(msg),
                                       _ptr(st), _ptr(llr), _ptr(plain), C.byref(osd), C.byref(ohard), C.byref(ap), C.byref(ahard))
        return dict(ok=int(ok), msg=msg[0], status=st[0], llr=llr, plain=plain, osd=osd.value, osd_hard=ohard.value, ap=ap.value, ap_hard=ahard.value)

    def subsystem_ap(self, i_s, q_s, osd_order, osd_max_hard, ap_on, ap_max_hard, max_cand=120, max_msgs=50, min_score=10, iters=20):
        """orc_subsystem_ap: subsystem() with OSD and then AP where they leave a candidate at stage 1 or 2."""
        i_s = np.ascontiguousarray(i_s, np.float32)
        q_s = np.ascontiguousarray(q_s, np.float32)
        res = np.zeros(max_msgs, result_dtype)
        from oracle.pyoracle import SlotReport
        rep = SlotReport()
        wf = np.zeros(WF_BYTES, np.uint8)
        cands = np.zeros(max_cand, cand_dtype)
        n = self.ap_lib.orc_subsystem_ap(_ptr(i_s), _ptr(q_s), max_cand, max_msgs, min_score, iters, int(osd_order), int(osd_max_hard), int(ap_on),
                                         int(ap_max_hard), _ptr(res), C.byref(rep), _ptr(wf), _ptr(cands))
        return self._slot_dict(n, res, rep, cands, wf)


@pytest.fixture(scope="module")
def oracle(tmp_path_factory):
    """Overrides the session oracle in the AP test modules: the same restatement plus the OSD and AP forms."""
    return ApOracle(tmp_path_factory.mktemp("ap_oracle"))


def bits77(payload):
    return np.unpackbits(np.frombuffer(payload[:10], np.uint8))[:77]


def scramble(payload):
    """FT4: the 77 message bits XORed with kFt4tXor before CRC and FEC."""
    return bytes(x ^ y for x, y in zip(payload[:10], FT4_XOR))


def cq_codeword(oracle, rng, protocol=1, extra=None):
    to, de, ex = "CQ", synth.random_call(rng), synth.random_grid(rng) if extra is None else extra
    p = ft8enc.pack_std(to, de, ex)
    return oracle.encode174(scramble(p) if protocol == 0 else p), f"CQ {de} {ex}".strip()


def fuzz_ap_llrs(oracle, n, seed, protocol=1):
    """n LLR vectors: noise, noisy CQ codewords (BP fails on many, AP recovers some), CQ codewords with the known positions
    reversed, noisy non-CQ codewords, ties and +-0."""
    rng = np.random.default_rng(seed)
    out = []
    for k in range(n):
        kind = k % 5
        if kind == 0:
            x = rng.normal(0, 2.5, N)
        elif kind in (1, 2):
            c = cq_codeword(oracle, rng, protocol)[0].astype(np.float64)
            x = (2 * c - 1) * rng.uniform(0.8, 2.0) + rng.normal(0, rng.uniform(1.2, 2.6), N)
            if kind == 2:
                x[KNOWN] = -x[KNOWN]
        elif kind == 3:
            c = codeword(oracle, rng).astype(np.float64)
            x = (2 * c - 1) * rng.uniform(1.0, 2.5) + rng.normal(0, rng.uniform(0.8, 2.2), N)
        else:
            c = cq_codeword(oracle, rng, protocol)[0].astype(np.float64)
            flip = rng.random(N) < rng.uniform(0.0, 0.25)
            x = np.where(flip, 1 - 2 * c, 2 * c - 1) * rng.choice([0.5, 1.0, 2.0, 4.0], N)
            z = rng.random(N) < 0.05
            x[z] = np.where(rng.random(int(z.sum())) < 0.5, 0.0, -0.0)
        out.append(np.asarray(x, np.float32))
    return np.array(out, np.float32)


def ref_ap(llr, max_hard, oracle, protocol=1, max_iters=20):
    """Steps 1, 2, 4 and 5 of the definition, independently; step 3 is orc_bp_decode.  -> (accepted -1/0/1, word, hard)."""
    llr = np.asarray(llr, np.float32)
    if not np.all(np.isfinite(llr)):
        return -1, None, None
    hyp = np.zeros(77, np.uint8)
    hyp[:29] = [int(b) for b in format(4, "029b")]  # c28 = 2 (CQ) << 1 | r1 = 0
    hyp[74:77] = [0, 0, 1]                           # i3 = 1
    scr = np.unpackbits(np.frombuffer(FT4_XOR, np.uint8))[:77] if protocol == 0 else np.zeros(77, np.uint8)
    forced_bits = (hyp ^ scr)[KNOWN]
    apmag = np.float32(np.max(np.abs(llr))) * np.float32(1.01)
    y = llr.copy()
    y[KNOWN] = np.where(forced_bits == 1, apmag, -apmag).astype(np.float32)
    word, errors = oracle.bp_decode(y, max_iters)
    hard = int(np.sum(word != (llr > 0)))
    msg = word[:77] ^ scr
    ok = errors == 0 and np.array_equal(word[KNOWN], forced_bits) and hard <= max_hard
    ok = ok and crc14(np.concatenate([word[:77], np.zeros(5, np.uint8)])) == int("".join(map(str, word[77:91])), 2)
    n28b = int("".join(map(str, msg[29:57])), 2)
    g15 = int("".join(map(str, msg[59:74])), 2)
    ok = ok and n28b >= NTOK + MAX22 and msg[58] == 0 and (g15 <= 32400 or g15 == 32401)
    if ok:
        a = np.packbits(np.concatenate([msg, np.zeros(3, np.uint8)])).tobytes()
        ok = oracle.unpack77(a)[0] >= 0
    return int(ok), word, hard


def test_hypothesis_is_every_plain_cq_and_no_other_form(oracle):
    mask, val = oracle.hypothesis(1)
    assert np.array_equal(np.flatnonzero(mask), KNOWN)
    mask4, val4 = oracle.hypothesis(0)
    scr = np.unpackbits(np.frombuffer(FT4_XOR, np.uint8))[:77]
    assert np.array_equal(mask4, mask) and np.array_equal(val4[KNOWN], val[KNOWN] ^ scr[KNOWN])
    rng = np.random.default_rng(11)
    n_cq = n_other = 0
    for _ in range(3000):
        to, de, ex = synth.random_message(rng)
        b = bits77(ft8enc.pack_std(to, de, ex))
        same = np.array_equal(b[KNOWN], val[KNOWN])
        assert same == (to == "CQ"), (to, de, ex)
        n_cq += to == "CQ"
        n_other += to != "CQ"
    assert n_cq >= 1000 and n_other >= 1000
    payloads, labels = synth.payload_fuzz(3, 4000)
    for p, lab in zip(payloads, labels):
        p = bytes(p)
        rc, text = oracle.unpack77(p[:9] + bytes([p[9] & 0xF8]))
        if np.array_equal(bits77(p)[KNOWN], val[KNOWN]):
            assert lab.startswith("std_token") and (rc < 0 or text.startswith("CQ ")), (lab, text)  # call_2 is not part of it
        if lab.startswith(("std_cq_nnn", "std_cq_aaaa")) or (rc >= 0 and not text.startswith("CQ ")):
            assert not np.array_equal(bits77(p)[KNOWN], val[KNOWN]), (lab, text)
    call, grid = ft8enc._pack_call("K1ABC"), ft8enc._pack_extra("FN42")
    for text, n28a in (("CQ 123 K1ABC FN42", 3 + 123), ("CQ DX K1ABC FN42", 1003 + 4 * 27 + 24), ("CQ TEST K1ABC FN42", 1003 + ((20 * 27 + 5) * 27 + 19) * 27 + 20),
                       ("QRZ K1ABC FN42", 1), ("DE K1ABC FN42", 0), ("W9XYZ K1ABC FN42", ft8enc._pack_call("W9XYZ"))):
        p = std_payload(n28a, call, 0, grid)
        assert oracle.unpack77(p[:9] + bytes([p[9] & 0xF8]))[1].strip() == text
        assert not np.array_equal(bits77(p)[KNOWN], val[KNOWN]), text
    p = std_payload(2, call, 0, grid, i3=2)  # "CQ K1ABC FN42" of type i3 = 2 (/P calls) is not the hypothesis either
    assert oracle.unpack77(p[:9] + bytes([p[9] & 0xF8]))[1].strip() == "CQ K1ABC FN42" and not np.array_equal(bits77(p)[KNOWN], val[KNOWN])


@pytest.mark.parametrize("protocol", [1, 0], ids=["ft8", "ft4"])
def test_restatement_equals_independent_implementation(oracle, protocol):
    llrs = fuzz_ap_llrs(oracle, 1000, 21 + protocol, protocol)
    accepted = rejected = 0
    for cap in (20, 60, 174):
        for x in (llrs if cap == 60 else llrs[::4]):
            got = oracle.ap(x, cap, protocol)
            want = ref_ap(x, cap, oracle, protocol)
            assert got[0] == want[0] and np.array_equal(got[1], want[1]) and got[2] == want[2]
            accepted += got[0] == 1
            rejected += got[0] == 0
    assert accepted > 50 and rejected > 50  # both paths are exercised


def test_reversed_known_positions_are_recovered(oracle):
    """A CQ codeword with the LLRs of its 32 known positions reversed: BP alone fails, AP decodes it."""
    for protocol in (1, 0):
        rng = np.random.default_rng(40 + protocol)
        recovered = 0
        for _ in range(40):
            c, text = cq_codeword(oracle, rng, protocol)
            x = ((2 * c.astype(np.float32) - 1) * rng.uniform(2.0, 4.0, N)).astype(np.float32)
            x[KNOWN] = -x[KNOWN]
            _, errors = oracle.bp_decode(x)
            acc, word, hard = oracle.ap(x, 174, protocol)
            if errors == 0:
                continue
            assert acc == 1 and np.array_equal(word, c) and hard == 32, text
            recovered += 1
        assert recovered >= 30


def test_non_finite_llrs_are_not_attempted(oracle):
    x = fuzz_ap_llrs(oracle, 3, 5)[1]
    for bad in (np.nan, np.inf, -np.inf):
        y = x.copy(); y[100] = bad
        assert oracle.ap(y, 174)[0] == -1 and oracle.ap(y, 174, 0)[0] == -1


def test_cap_is_inclusive(oracle):
    rng = np.random.default_rng(8)
    c, _ = cq_codeword(oracle, rng)
    x = ((2 * c.astype(np.float32) - 1) * 3.0).astype(np.float32)
    x[KNOWN[:7]] = -x[KNOWN[:7]]
    acc, word, hard = oracle.ap(x, 174)
    assert acc == 1 and np.array_equal(word, c) and hard == 7
    assert oracle.ap(x, 7)[0] == 1
    acc, word6, hard6 = oracle.ap(x, 6)  # one over the cap: rejected, same word
    assert acc == 0 and np.array_equal(word6, c) and hard6 == 7


def std_payload(n28a, n28b, ir, g15, i3=1):
    from tools.synth import bits_to_payload
    return bytes(bits_to_payload([(n28a, 28), (0, 1), (n28b, 28), (0, 1), (ir, 1), (g15, 15), (i3, 3)]))


@pytest.mark.parametrize("text,n28b,ir,g15", [("CQ <...> FN42", NTOK + 12345, 0, None), ("CQ K1ABC R FN42", None, 1, None),
                                             ("CQ K1ABC RR73", None, 0, 32403), ("CQ K1ABC +05", None, 0, 32400 + 35 + 5),
                                             ("CQ K1ABC RRR", None, 0, 32402), ("CQ K1ABC 73", None, 0, 32404)])
def test_implausible_cq_words_are_rejected(oracle, text, n28b, ir, g15):
    call = ft8enc._pack_call("K1ABC")
    p = std_payload(2, call if n28b is None else n28b, ir, ft8enc._pack_extra("FN42") if g15 is None else g15)
    rc, got = oracle.unpack77(p[:9] + bytes([p[9] & 0xF8]))
    assert rc >= 0 and got.strip() == text
    for payload, want in ((p, 0), (std_payload(2, call, 0, ft8enc._pack_extra("FN42")), 1), (std_payload(2, call, 0, 32401), 1)):
        c = oracle.encode174(payload)
        x = ((2 * c.astype(np.float32) - 1) * 3.0).astype(np.float32)
        x[KNOWN[:5]] = -x[KNOWN[:5]]  # BP alone stops at the CRC or the syndrome; AP's word is the codeword
        acc, word, hard = oracle.ap(x, 174)
        assert np.array_equal(word, c) and hard == 5 and acc == want, oracle.unpack77(payload[:9] + bytes([payload[9] & 0xF8]))


def test_every_accepted_word_is_a_codeword(oracle):
    for protocol in (1, 0):
        for x in fuzz_ap_llrs(oracle, 300, 77, protocol):
            acc, word, _ = oracle.ap(x, 174, protocol)
            if acc == 1:
                assert not np.any(H.astype(np.int64) @ word % 2)


def test_ap_off_forms_equal_the_osd_forms(oracle):
    sig = [(ft8enc.tones(ft8enc.pack_std("CQ", "K1JT", "FN20")), 700.0, 0.5, -21.0),
           (ft8enc.tones(ft8enc.pack_std("CQ", "W1AW", "FN31")), 1200.0, 1.1, -14.0),
           (ft8enc.tones(ft8enc.pack_std("K1ABC", "W9XYZ", "EN37")), 400.0, 0.3, -20.0)]
    i_s, q_s = synth.slot_f32(sig, 12)
    i_s, q_s, _ = oracle.condition(i_s, q_s, 48000)
    for order in (0, 2):
        a, b = oracle.subsystem_osd(i_s, q_s, order, 174), oracle.subsystem_ap(i_s, q_s, order, 174, 0, 174)
        assert a["n"] == b["n"] and a["results"].tobytes() == b["results"].tobytes() and a["msgs"].tobytes() == b["msgs"].tobytes()
        for c in a["cands"][:40]:
            d, e = oracle.decode_osd(a["wf"], c, order, 174), oracle.decode_ap(a["wf"], c, order, 174, 0, 174)
            assert d["ok"] == e["ok"] and d["status"].tobytes() == e["status"].tobytes() and np.array_equal(d["plain"], e["plain"])
            assert d["osd"] == e["osd"] and e["ap"] == 0 and e["ap_hard"] == -1


def test_ap_on_only_adds_decodes(oracle):
    """With AP on, every candidate BP or OSD decoded is unchanged, and an AP decode is a plausible CQ whose plain row is the word."""
    rng = np.random.default_rng(3)
    n_ap = 0
    for s in range(6):
        sig = [(ft8enc.tones(ft8enc.pack_std("CQ", synth.random_call(rng), synth.random_grid(rng))), float(rng.uniform(300, 1300)), 0.5, -19.0)
               for _ in range(3)]
        i_s, q_s = synth.slot_f32(sig, 300 + s)
        i_s, q_s, _ = oracle.condition(i_s, q_s, 48000)
        a = oracle.subsystem_osd(i_s, q_s, 0, 174)
        for c in a["cands"]:
            d, e = oracle.decode_osd(a["wf"], c, 0, 174), oracle.decode_ap(a["wf"], c, 0, 174, 1, 174)
            if d["ok"]:
                assert e["ok"] and e["ap"] == 0 and d["status"].tobytes() == e["status"].tobytes()
            elif e["ap"] == 2:
                n_ap += 1
                assert e["ok"] and e["msg"]["text"].startswith(b"CQ ") and e["status"]["ldpc_errors"] == 0
                assert not np.any(H.astype(np.int64) @ e["plain"] % 2)
    assert n_ap >= 1
