"""ctypes bindings for the CPU checkers under oracle/.  TEST INFRASTRUCTURE ONLY.

Two libraries:
  * ``Oracle``  -> oracle/libft8oracle.so, this repository's C restatement (always buildable:
    ``make -C oracle restate``; built on demand here).
  * ``Reference`` -> oracle/_ref/libref_{k120,k500}.so, the UNMODIFIED reference compiled from
    /root/reference by oracle/Makefile (present only where it was built; optional).
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module.  The product library never touches it.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
N_SLOT = 48000
WF_BYTES = 94208

cand_dtype = np.dtype([("score", "<i2"), ("time_offset", "<i2"), ("freq_offset", "<i2"), ("time_sub", "u1"), ("freq_sub", "u1")])
msg_dtype = np.dtype([("text", "S25"), ("_pad", "u1"), ("hash", "<u2")])
status_dtype = np.dtype([("ldpc_errors", "<i4"), ("crc_extracted", "<u2"), ("crc_calculated", "<u2"), ("unpack_status", "<i4")])
result_dtype = np.dtype([("call", "S13"), ("loc", "S7"), ("freq", "<i4"), ("snr", "<i4")])
assert cand_dtype.itemsize == 8 and msg_dtype.itemsize == 28 and status_dtype.itemsize == 12 and result_dtype.itemsize == 28


class WaterfallT(C.Structure):
    _fields_ = [("max_blocks", C.c_int), ("num_blocks", C.c_int), ("num_bins", C.c_int), ("time_osr", C.c_int),
                ("freq_osr", C.c_int), ("mag", C.c_void_p), ("block_stride", C.c_int), ("protocol", C.c_int)]


assert C.sizeof(WaterfallT) == 40


class DecimState(C.Structure):
    _fields_ = [("ints", C.c_int32 * 12), ("decim_index", C.c_uint32), ("fir_i", C.c_float * 56), ("fir_q", C.c_float * 56),
                ("n_out", C.c_uint64)]


class SlotReport(C.Structure):
    _fields_ = [("n_cand", C.c_int), ("n_unique", C.c_int), ("msgs", C.c_uint8 * (28 * 512)), ("freq_hz", C.c_float * 512),
                ("score", C.c_int * 512)]


signal_dtype = np.dtype([("payload", "u1", 10), ("reserved", "u1", 2), ("f0_hz", "<f4"), ("t0_sec", "<f4"), ("amp", "<f4")])
assert signal_dtype.itemsize == 24


def _ptr(a, t=C.c_void_p):
    return a.ctypes.data_as(t)


def reference_dir() -> str:
    """Where oracle/Makefile looks for the reference's sources: $REF, else the Makefile's default."""
    if os.environ.get("REF"):
        return os.environ["REF"]
    with open(os.path.join(HERE, "Makefile")) as f:
        for line in f:
            if line.startswith("REF") and "?=" in line:
                return line.split("?=", 1)[1].strip()
    raise RuntimeError("oracle/Makefile sets no REF")


def build_restatement(force: bool = False) -> str:
    so = os.path.join(HERE, "libft8oracle.so")
    srcs = [os.path.join(HERE, f) for f in ("ft8_oracle.c", "ft8_oracle_codec.c", "ft8_oracle_synth.c", "ft8_oracle_report.c", "ft8_oracle.h", "ft8_tables.h")]
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["make", "-C", HERE, "restate"], stdout=subprocess.DEVNULL)
    return so


def make_wf(mag: np.ndarray, num_blocks=92, num_bins=256, time_osr=2, freq_osr=2, protocol=1) -> WaterfallT:
    assert mag.dtype == np.uint8 and mag.flags.c_contiguous
    return WaterfallT(num_blocks, num_blocks, num_bins, time_osr, freq_osr, mag.ctypes.data, time_osr * freq_osr * num_bins, protocol)


class Oracle:
    """The restatement (oracle/ft8_oracle.c)."""

    def __init__(self):
        self.lib = L = C.CDLL(build_restatement())
        L.orc_fir_coefs.restype = C.POINTER(C.c_float)
        L.orc_condition.restype = C.c_float
        L.orc_quantize_db.restype = C.c_uint8
        L.orc_quantize_db.argtypes = [C.c_float]
        L.orc_crc14.restype = C.c_uint16
        L.orc_monitor_new.restype = C.c_void_p
        L.orc_monitor_mag.restype = C.POINTER(C.c_uint8)
        L.orc_monitor_max_mag.restype = C.c_float
        for f in ("orc_monitor_free", "orc_monitor_process", "orc_monitor_reset", "orc_monitor_info", "orc_monitor_mag", "orc_monitor_max_mag"):
            getattr(L, f).argtypes = [C.c_void_p] + ([C.c_void_p] if f in ("orc_monitor_process", "orc_monitor_info") else [])

    # -- decimator ------------------------------------------------------------------
    def fir(self) -> np.ndarray:
        return np.ctypeslib.as_array(self.lib.orc_fir_coefs(), shape=(57,)).copy()

    def new_decim(self) -> DecimState:
        st = DecimState()
        self.lib.orc_decim_reset(C.byref(st))
        return st

    def decim_feed(self, st: DecimState, iq: np.ndarray, cap: int, want_y2=False):
        """Feed one callback's worth of bytes; returns (I, Q[, y2i, y2q]) produced by this call (<= cap)."""
        iq = np.ascontiguousarray(iq, dtype=np.uint8)
        assert iq.size % 8 == 0
        i_out = np.zeros(cap, np.float32)
        q_out = np.zeros(cap, np.float32)
        y2i = np.zeros(cap, np.int32) if want_y2 else None
        y2q = np.zeros(cap, np.int32) if want_y2 else None
        cnt = C.c_size_t(0)
        self.lib.orc_decim_feed(C.byref(st), _ptr(iq), C.c_size_t(iq.size), _ptr(i_out), _ptr(q_out),
                                _ptr(y2i) if want_y2 else None, _ptr(y2q) if want_y2 else None, C.c_size_t(cap), C.byref(cnt))
        n = cnt.value
        return (i_out[:n], q_out[:n], y2i[:n], y2q[:n]) if want_y2 else (i_out[:n], q_out[:n])

    def decimate_slot(self, iq: np.ndarray, chunk=65536, want_y2=False):
        """A whole stream from zero state in `chunk`-byte callbacks (as librtlsdr delivers them)."""
        st = self.new_decim()
        outs = []
        for o in range(0, iq.size, chunk):
            outs.append(self.decim_feed(st, iq[o:o + chunk], (chunk // 2) // 751 + 2, want_y2))
        return tuple(np.concatenate([o[k] for o in outs]) for k in range(4 if want_y2 else 2))

    def condition(self, i_s: np.ndarray, q_s: np.ndarray, n_valid: int):
        i2 = np.array(i_s, np.float32, copy=True)
        q2 = np.array(q_s, np.float32, copy=True)
        scale = self.lib.orc_condition(_ptr(i2), _ptr(q2), C.c_size_t(n_valid), C.c_size_t(i2.size))
        return i2, q2, np.float32(scale)

    # -- waterfall -------------------------------------------------------------------
    def sine_window(self, n=1024):
        w = np.zeros(n, np.float32)
        self.lib.orc_sine_window(_ptr(w), n)
        return w

    def fft_c2c(self, x: np.ndarray) -> np.ndarray:
        x = np.ascontiguousarray(x, np.complex64)
        y = np.zeros_like(x)
        self.lib.orc_fft_c2c(x.size, _ptr(x), _ptr(y))
        return y

    def fft_r2c(self, x: np.ndarray) -> np.ndarray:
        x = np.ascontiguousarray(x, np.float32)
        y = np.zeros(x.size // 2 + 1, np.complex64)
        self.lib.orc_fft_r2c(x.size, _ptr(x), _ptr(y))
        return y

    def db_thresholds(self) -> np.ndarray:
        t = np.zeros(257, np.float32)
        self.lib.orc_db_thresholds(_ptr(t))
        return t

    def quantize_db(self, x: float) -> int:
        return int(self.lib.orc_quantize_db(C.c_float(x)))

    def waterfall(self, i_s, q_s) -> np.ndarray:
        i_s = np.ascontiguousarray(i_s, np.float32)
        q_s = np.ascontiguousarray(q_s, np.float32)
        assert i_s.size == N_SLOT and q_s.size == N_SLOT
        mag = np.zeros(WF_BYTES, np.uint8)
        self.lib.orc_waterfall_daemon(_ptr(i_s), _ptr(q_s), _ptr(mag))
        return mag

    def monitor_waterfall(self, audio: np.ndarray, sample_rate=12000, time_osr=2, freq_osr=2, protocol=1):
        """Run the 12 kHz monitor over `audio`; returns (mag, info[9], max_mag)."""
        audio = np.ascontiguousarray(audio, np.float32)
        m = self.lib.orc_monitor_new(sample_rate, time_osr, freq_osr, protocol)
        info = np.zeros(9, np.int32)
        self.lib.orc_monitor_info(m, _ptr(info))
        bs = int(info[0])
        for o in range(0, audio.size - bs + 1, bs):
            self.lib.orc_monitor_process(m, _ptr(audio[o:o + bs]))
        self.lib.orc_monitor_info(m, _ptr(info))
        nbytes = int(info[4]) * int(info[8])
        mag = np.ctypeslib.as_array(self.lib.orc_monitor_mag(m), shape=(int(info[3]) * int(info[8]),))[:nbytes].copy()
        mx = float(self.lib.orc_monitor_max_mag(m))
        self.lib.orc_monitor_free(m)
        return mag, info, mx

    # -- sync / decode ----------------------------------------------------------------
    def find_sync(self, mag, max_cand=120, min_score=10, **dims) -> np.ndarray:
        wf = make_wf(mag, **dims)
        heap = np.zeros(max_cand, cand_dtype)
        n = self.lib.orc_find_sync(C.byref(wf), max_cand, _ptr(heap), min_score)
        return heap[:n]

    def sync_score(self, mag, cand, **dims) -> int:
        wf = make_wf(mag, **dims)
        c = np.array([cand], cand_dtype)
        return int(self.lib.orc_sync_score(C.byref(wf), _ptr(c)))

    def decode(self, mag, cand, max_iters=20, **dims):
        """-> dict(ok, msg, status, llr, plain); status pre-filled with 0xA5 like the reference tap."""
        wf = make_wf(mag, **dims)
        c = np.array([cand], cand_dtype)
        msg = np.zeros(1, msg_dtype)
        st = np.frombuffer(bytes([0xA5]) * 12, status_dtype).copy()
        llr = np.zeros(174, np.float32)
        plain = np.zeros(174, np.uint8)
        ok = self.lib.orc_decode(C.byref(wf), _ptr(c), max_iters, _ptr(msg), _ptr(st), _ptr(llr), _ptr(plain))
        return dict(ok=int(ok), msg=msg[0], status=st[0], llr=llr, plain=plain)

    def bp_decode(self, llr, max_iters=20):
        llr = np.ascontiguousarray(llr, np.float32)
        plain = np.zeros(174, np.uint8)
        err = C.c_int(0)
        self.lib.orc_bp_decode(_ptr(llr), max_iters, _ptr(plain), C.byref(err))
        return plain, err.value

    def crc14(self, data: bytes, nbits: int) -> int:
        return int(self.lib.orc_crc14(data, nbits))

    def unpack77(self, a77: bytes):
        buf = C.create_string_buffer(64)
        rc = self.lib.orc_unpack77(a77, buf)
        return rc, buf.value.decode("ascii", "replace")

    def subsystem(self, i_s, q_s, max_cand=120, max_msgs=50, min_score=10, iters=20):
        """ft8_subsystem() restated -> dict(n, results, report(msgs,freq,score), wf, cands)."""
        i_s = np.ascontiguousarray(i_s, np.float32)
        q_s = np.ascontiguousarray(q_s, np.float32)
        res = np.zeros(max_msgs, result_dtype)
        rep = SlotReport()
        wf = np.zeros(WF_BYTES, np.uint8)
        cands = np.zeros(max_cand, cand_dtype)
        n = self.lib.orc_subsystem(_ptr(i_s), _ptr(q_s), max_cand, max_msgs, min_score, iters, _ptr(res), C.byref(rep), _ptr(wf), _ptr(cands))
        return self._slot_dict(n, res, rep, cands, wf)

    def decode_waterfall(self, mag, max_cand=120, max_msgs=50, min_score=10, iters=20, **dims):
        wf = make_wf(mag, **dims)
        res = np.zeros(max_msgs, result_dtype)
        rep = SlotReport()
        cands = np.zeros(max_cand, cand_dtype)
        n = self.lib.orc_decode_waterfall(C.byref(wf), max_cand, max_msgs, min_score, iters, _ptr(res), C.byref(rep), _ptr(cands))
        return self._slot_dict(n, res, rep, cands, mag)

    def spots(self, cands, ok, msgs, max_msgs=50, min_score=10, freq_osr=2):
        """The duplicate table + CQ filter alone (rtlsdr_ft8d.c:1467-1522) over hand-made decode results."""
        cands = np.ascontiguousarray(cands, cand_dtype)
        ok = np.ascontiguousarray(ok, np.uint8)
        msgs = np.ascontiguousarray(msgs, msg_dtype)
        assert cands.size == ok.size == msgs.size
        res = np.zeros(max_msgs, result_dtype)
        rep = SlotReport()
        n = self.lib.orc_spots(_ptr(cands), _ptr(ok), _ptr(msgs), cands.size, max_msgs, min_score, freq_osr, _ptr(res), C.byref(rep))
        rep.n_cand = cands.size
        return self._slot_dict(n, res, rep, cands, None)

    @staticmethod
    def _slot_dict(n, res, rep, cands, wf):
        k = min(rep.n_unique, 512)
        msgs = np.frombuffer(bytes(rep.msgs), msg_dtype)[:k].copy()
        return dict(n=n, results=res, msgs=msgs, freq_hz=np.array(rep.freq_hz[:k], np.float32), score=np.array(rep.score[:k], np.int32),
                    cands=cands[:rep.n_cand].copy(), wf=wf)

    def decode_ft8_lines(self, audio: np.ndarray, sample_rate=12000, protocol=1, max_cand=120, min_score=10, iters=20, max_msgs=50):
        """decode_ft8's main() (ft8_lib/decode_ft8.c:296-406) on one recording -> its stdout lines:
        monitor waterfall, ft8_find_sync, then per candidate ft8_decode + the hash table of first-seen unique messages."""
        mag, info, _ = self.monitor_waterfall(audio, sample_rate, 2, 2, protocol)
        dims = dict(num_blocks=int(info[4]), num_bins=int(info[5]), time_osr=2, freq_osr=2, protocol=protocol)
        if dims["num_blocks"] == 0:
            return []
        sp = np.float32(0.048 if protocol == 0 else 0.160)
        table = [None] * max_msgs
        lines = []
        for c in self.find_sync(mag, max_cand, min_score, **dims):
            if c["score"] < min_score:
                continue
            freq = (np.float32(c["freq_offset"]) + np.float32(c["freq_sub"]) / np.float32(2)) / sp
            tsec = (np.float32(c["time_offset"]) + np.float32(c["time_sub"]) / np.float32(2)) * sp
            d = self.decode(mag, c, iters, **dims)
            if not d["ok"]:
                continue
            h, text = int(d["msg"]["hash"]), d["msg"]["text"]
            idx = h % max_msgs
            dup = False
            for _ in range(max_msgs):
                if table[idx] is None:
                    break
                if table[idx] == (h, text):
                    dup = True
                    break
                idx = (idx + 1) % max_msgs
            else:
                continue  # table full: the reference would spin forever (decode_ft8.c:369-388)
            if dup:
                continue
            table[idx] = (h, text)
            lines.append("000000 %3d %+4.2f %4.0f ~  %s" % (int(c["score"]), float(tsec), float(freq), text.decode()))
        return lines

    # -- CPU twin of the device signal synthesiser (csrc/synth.cu) ------------------------------------
    def synth_raw(self, signals: np.ndarray, noise_lsb: float, seed: int, slot_index: int, n_samples: int) -> np.ndarray:
        """signals: array of signal_dtype -> uint8[2*n_samples] interleaved I,Q (one slot)."""
        signals = np.ascontiguousarray(signals, signal_dtype)
        out = np.zeros(2 * n_samples, np.uint8)
        self.lib.orc_synth_raw(_ptr(signals), signals.size, C.c_float(noise_lsb), C.c_uint64(seed), slot_index, _ptr(out), C.c_longlong(n_samples))
        return out

    def synth_float(self, kind: int, ft4: bool, signals: np.ndarray, noise_sigma: float, seed: int, slot_index: int, n_samples: int):
        """kind 1: complex 3200 sps -> (I, Q); kind 2: real 12 kHz audio -> (x, None)."""
        signals = np.ascontiguousarray(signals, signal_dtype)
        oi = np.zeros(n_samples, np.float32)
        oq = np.zeros(n_samples, np.float32) if kind == 1 else None
        self.lib.orc_synth_float(kind, int(ft4), _ptr(signals), signals.size, C.c_float(noise_sigma), C.c_uint64(seed), slot_index, _ptr(oi),
                                 _ptr(oq) if oq is not None else None, n_samples)
        return oi, oq

    # -- reporting formats (ft8_oracle_report.c) -----------------------------------------------------------
    def pskreporter_datagram(self, spots: np.ndarray, rcall: str, rloc: str, dial_freq: int, app_version: str, unixtime: int,
                             sequence: int = 1, random_id: int = 0) -> bytes:
        spots = np.ascontiguousarray(spots, result_dtype)
        out = C.create_string_buffer(4096)
        n = self.lib.orc_pskreporter_datagram(_ptr(spots), C.c_uint32(spots.size), rcall.encode(), rloc.encode(), C.c_uint32(dial_freq),
                                              app_version.encode(), C.c_uint32(unixtime), C.c_uint32(sequence), C.c_uint32(random_id), out)
        return out.raw[:n]

    def webcluster_form(self, spot: np.ndarray, rcall: str, rloc: str, dial_freq: int) -> dict:
        spot = np.ascontiguousarray(spot, result_dtype).reshape(1)
        out = C.create_string_buffer(4 * 112)
        self.lib.orc_webcluster_form(_ptr(spot), rcall.encode(), rloc.encode(), C.c_uint32(dial_freq), out)
        return {k: out.raw[i * 112:(i + 1) * 112].split(b"\0")[0] for i, k in enumerate(("_mycall", "_dxcall", "_freq", "_info"))}

    def print_spots(self, spots: np.ndarray, dial_freq: int, unixtime: int) -> str:
        spots = np.ascontiguousarray(spots, result_dtype)
        out = C.create_string_buffer(1 << 16)
        self.lib.orc_print_spots(_ptr(spots), C.c_uint32(spots.size), C.c_uint32(dial_freq), C.c_uint32(unixtime), out, C.c_size_t(1 << 16))
        return out.value.decode()

    # -- encoder ----------------------------------------------------------------------
    def pack_std(self, call_to: str, call_de: str, extra: str) -> bytes:
        b = C.create_string_buffer(10)
        rc = self.lib.orc_pack_std(call_to.encode(), call_de.encode(), extra.encode(), b)
        if rc < 0:
            raise ValueError(f"cannot pack {call_to} {call_de} {extra}")
        return b.raw

    def pack_text(self, text: str) -> bytes:
        b = C.create_string_buffer(10)
        self.lib.orc_pack_text(text.encode(), b)
        return b.raw

    def pack77(self, msg: str):
        """pack77() restated (pack.c:284-301): (payload, kind) with kind 0 = standard message, 1 = free text."""
        b = C.create_string_buffer(10)
        kind = self.lib.orc_pack77(msg.encode(), b)
        return b.raw, int(kind)

    def tones(self, payload: bytes) -> np.ndarray:
        t = np.zeros(79, np.uint8)
        self.lib.orc_encode_tones(payload, _ptr(t))
        return t

    def encode174(self, payload: bytes) -> np.ndarray:
        t = np.zeros(174, np.uint8)
        self.lib.orc_encode174(payload, _ptr(t))
        return t


class Reference:
    """The unmodified reference (oracle/_ref/libref_k*.so).  `fresh=True` loads a private copy of the
    .so so the daemon's function-static decimator state starts from zero (one stream per copy)."""

    TAP_MAX = 1024

    def __init__(self, variant="k120", fresh=False):
        path = os.path.join(HERE, "_ref", f"libref_{variant}.so")
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        if fresh:
            fd, tmp = tempfile.mkstemp(suffix=".so", prefix="libref_")
            os.close(fd)
            shutil.copy(path, tmp)
            self.lib = C.CDLL(tmp)
            os.unlink(tmp)
        else:
            self.lib = C.CDLL(path)
        L = self.lib
        L.ref_taps_ptr.restype = C.c_void_p
        L.ref_rx_count.restype = C.c_uint32
        L.ref_window.restype = C.POINTER(C.c_float)
        L.ref_crc.restype = C.c_uint32
        L.ref_init()
        self.kmax = L.ref_k_max_candidates()
        self.mmax = L.ref_k_max_messages()
        T = self.TAP_MAX
        self.taps_dtype = np.dtype([
            ("wf_bytes", "<i4"), ("wf_dims", "<i4", 6), ("n_cand", "<i4"), ("n_decode_calls", "<i4"), ("n_bp_calls", "<i4"),
            ("cand", cand_dtype, T), ("dec_cand", cand_dtype, T), ("dec_ok", "<i4", T), ("dec_status", status_dtype, T),
            ("dec_msg", msg_dtype, T), ("llr", "<f4", (T, 174)), ("plain", "u1", (T, 174)), ("bp_errors", "<i4", T),
            ("wf", "u1", 93 * 2 * 2 * 960)])
        assert self.taps_dtype.itemsize == L.ref_taps_size(), (self.taps_dtype.itemsize, L.ref_taps_size())

    @staticmethod
    def available(variant="k120") -> bool:
        return os.path.exists(os.path.join(HERE, "_ref", f"libref_{variant}.so"))

    def taps(self):
        buf = (C.c_uint8 * self.taps_dtype.itemsize).from_address(self.lib.ref_taps_ptr())
        return np.frombuffer(buf, self.taps_dtype)[0]

    def window(self):
        return np.ctypeslib.as_array(self.lib.ref_window(), shape=(1024,)).copy()

    def callback(self, iq: np.ndarray):
        buf = np.array(iq, np.uint8, copy=True)  # the reference mixes in place
        self.lib.ref_callback(_ptr(buf), C.c_uint32(buf.size))

    def rx(self, which=None):
        if which is None:
            which = self.lib.ref_rx_buffer_index()
        n = self.lib.ref_rx_count(which)
        i_s = np.zeros(N_SLOT, np.float32)
        q_s = np.zeros(N_SLOT, np.float32)
        self.lib.ref_rx_copy(which, _ptr(i_s), _ptr(q_s), C.c_uint32(N_SLOT))
        return i_s, q_s, int(n)

    def flip(self):
        self.lib.ref_rx_flip()

    def subsystem(self, i_s, q_s):
        i_s = np.array(i_s, np.float32, copy=True)
        q_s = np.array(q_s, np.float32, copy=True)
        res = np.zeros(self.mmax, result_dtype)
        n = self.lib.ref_subsystem(_ptr(i_s), _ptr(q_s), _ptr(res), self.mmax)
        t = self.taps()
        nc = int(t["n_cand"])
        nd = int(t["n_decode_calls"])
        return dict(n=n, results=res, wf=t["wf"][:int(t["wf_bytes"])].copy(), cands=t["cand"][:nc].copy(),
                    dec_ok=t["dec_ok"][:nd].copy(), dec_status=t["dec_status"][:nd].copy(), dec_msg=t["dec_msg"][:nd].copy(),
                    llr=t["llr"][:nd].copy(), plain=t["plain"][:nd].copy(), bp_errors=t["bp_errors"][:nd].copy())

    def subsystem_scripted(self, cands, ok, msgs):
        """The reference's own candidate loop / table / CQ filter (rtlsdr_ft8d.c:1452-1523) over a hand-made candidate list and
        hand-made ft8_decode() answers -> (n_results, decoder_results[K_MAX_MESSAGES])."""
        cands = np.ascontiguousarray(cands, cand_dtype)
        ok = np.ascontiguousarray(ok, np.int32)
        msgs = np.ascontiguousarray(msgs, msg_dtype)
        assert cands.size == ok.size == msgs.size <= min(self.kmax, self.TAP_MAX)
        res = np.zeros(self.mmax, result_dtype)
        n = self.lib.ref_subsystem_scripted(_ptr(cands), _ptr(ok), _ptr(msgs), cands.size, _ptr(res), self.mmax)
        return int(n), res

    def time_subsystem(self, i_s, q_s, reps=9):
        """Wall-clock (ms per call, timed inside the C harness) of decoder()'s conditioning + ft8_subsystem on one slot."""
        i_s = np.ascontiguousarray(i_s, np.float32); q_s = np.ascontiguousarray(q_s, np.float32)
        ms = np.zeros(reps, np.float64)
        n = self.lib.ref_time_subsystem(_ptr(i_s), _ptr(q_s), reps, _ptr(ms))
        return ms, int(n)

    def time_receive(self, raw):
        """Wall-clock (ms) of one raw slot through rtlsdr_callback (65536-byte calls) + flip + conditioning + ft8_subsystem."""
        buf = np.array(raw, np.uint8, copy=True)
        ms = C.c_double(0)
        n = self.lib.ref_time_receive(_ptr(buf), C.c_uint32(buf.size), C.byref(ms))
        return float(ms.value), int(n)

    def find_sync(self, mag, max_cand=120, min_score=10, num_blocks=92, num_bins=256, time_osr=2, freq_osr=2, protocol=1):
        mag = np.ascontiguousarray(mag, np.uint8)
        heap = np.zeros(max_cand, cand_dtype)
        n = self.lib.ref_find_sync(_ptr(mag), num_blocks, num_bins, time_osr, freq_osr, protocol, max_cand, _ptr(heap), min_score)
        return heap[:n]

    def decode(self, mag, cand, max_iters=20, num_blocks=92, num_bins=256, time_osr=2, freq_osr=2, protocol=1):
        mag = np.ascontiguousarray(mag, np.uint8)
        c = np.array([cand], cand_dtype)
        msg = np.zeros(1, msg_dtype)
        st = np.zeros(1, status_dtype)
        llr = np.zeros(174, np.float32)
        plain = np.zeros(174, np.uint8)
        ok = self.lib.ref_decode(_ptr(mag), num_blocks, num_bins, time_osr, freq_osr, protocol, _ptr(c), max_iters, _ptr(msg), _ptr(st), _ptr(llr), _ptr(plain))
        return dict(ok=int(ok), msg=msg[0], status=st[0], llr=llr, plain=plain)

    def bp_decode(self, llr, max_iters=20):
        llr = np.ascontiguousarray(llr, np.float32)
        plain = np.zeros(174, np.uint8)
        err = C.c_int(0)
        self.lib.ref_bp_decode(_ptr(llr), max_iters, _ptr(plain), C.byref(err))
        return plain, err.value

    def pack77(self, text: str) -> bytes:
        b = C.create_string_buffer(12)
        self.lib.ref_pack77(text.encode(), b)
        return b.raw[:10]

    def tones(self, payload: bytes) -> np.ndarray:
        t = np.zeros(79, np.uint8)
        self.lib.ref_encode(payload, _ptr(t))
        return t

    def unpack77(self, a77: bytes):
        buf = C.create_string_buffer(64)
        rc = self.lib.ref_unpack77(a77, buf)
        return rc, buf.value.decode("ascii", "replace")

    def crc(self, data: bytes, nbits: int) -> int:
        return int(self.lib.ref_crc(data, nbits))


class ReferenceMonitor:
    """ft8_lib's 12 kHz monitor path, unmodified (oracle/_ref/libref_mon.so)."""

    def __init__(self):
        path = os.path.join(HERE, "_ref", "libref_mon.so")
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        self.lib = L = C.CDLL(path)
        L.refmon_new.restype = C.c_void_p
        L.refmon_new.argtypes = [C.c_float, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int]
        L.refmon_mag.restype = C.POINTER(C.c_uint8)
        L.refmon_max_mag.restype = C.c_float
        for f in ("refmon_delete", "refmon_reset", "refmon_mag", "refmon_max_mag"):
            getattr(L, f).argtypes = [C.c_void_p]
        L.refmon_process.argtypes = [C.c_void_p, C.c_void_p]
        L.refmon_info.argtypes = [C.c_void_p, C.c_void_p]
        L.refmon_find_sync.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        L.refmon_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]

    @staticmethod
    def available() -> bool:
        return os.path.exists(os.path.join(HERE, "_ref", "libref_mon.so"))

    def waterfall(self, audio, sample_rate=12000, time_osr=2, freq_osr=2, protocol=1):
        audio = np.ascontiguousarray(audio, np.float32)
        m = self.lib.refmon_new(100.0, 3000.0, sample_rate, time_osr, freq_osr, protocol)
        info = np.zeros(9, np.int32)
        self.lib.refmon_info(m, _ptr(info))
        bs = int(info[0])
        for o in range(0, audio.size - bs + 1, bs):
            self.lib.refmon_process(m, _ptr(audio[o:o + bs]))
        self.lib.refmon_info(m, _ptr(info))
        nbytes = int(info[4]) * int(info[8])
        mag = np.ctypeslib.as_array(self.lib.refmon_mag(m), shape=(nbytes,)).copy()
        mx = float(self.lib.refmon_max_mag(m))
        self.lib.refmon_delete(m)
        return mag, info, mx

    def fftr(self, x):
        x = np.ascontiguousarray(x, np.float32)
        y = np.zeros(x.size // 2 + 1, np.complex64)
        self.lib.refmon_fftr(x.size, _ptr(x), _ptr(y))
        return y

    def decode_ft8_stdout(self, wav_path: str, ft4: bool = False):
        """Run the reference's own main() (decode_ft8 [-ft4] file.wav) in-process and return its stdout lines."""
        import tempfile
        args = [b"decode_ft8"] + ([b"-ft4"] if ft4 else []) + [wav_path.encode()]
        argv = (C.c_char_p * (len(args) + 1))(*args, None)
        libc = C.CDLL(None)
        libc.fflush(None)
        with tempfile.TemporaryFile() as tmp:
            saved, saved_err = os.dup(1), os.dup(2)
            devnull = os.open(os.devnull, os.O_WRONLY)
            os.dup2(tmp.fileno(), 1)
            os.dup2(devnull, 2)  # LOG(LOG_INFO, ...) chatter
            try:
                rc = self.lib.ref_decode_ft8_main(len(args), argv)
                libc.fflush(None)
            finally:
                os.dup2(saved, 1)
                os.dup2(saved_err, 2)
                os.close(saved); os.close(saved_err); os.close(devnull)
            tmp.seek(0)
            out = tmp.read().decode("ascii", "replace")
        if rc != 0:
            raise IOError(f"decode_ft8 main -> {rc}")
        return [l for l in out.splitlines() if l.startswith("000000")]

    def load_wav(self, path, max_samples=15 * 12000):
        sig = np.zeros(max_samples, np.float32)
        n = C.c_int(max_samples)
        sr = C.c_int(0)
        rc = self.lib.refmon_load_wav(path.encode(), _ptr(sig), C.byref(n), C.byref(sr))
        if rc < 0:
            raise IOError(f"load_wav({path}) -> {rc}")
        return sig[:n.value].copy(), sr.value


class ReferenceGen:
    """ft8_lib's gen_ft8.c (gfsk_pulse / synth_gfsk), unmodified (oracle/_ref/libref_gen.so)."""

    def __init__(self):
        path = os.path.join(HERE, "_ref", "libref_gen.so")
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        self.lib = C.CDLL(path)

    @staticmethod
    def available() -> bool:
        return os.path.exists(os.path.join(HERE, "_ref", "libref_gen.so"))

    def pulse(self, n_spsym: int, bt: float) -> np.ndarray:
        out = np.zeros(3 * n_spsym, np.float32)
        self.lib.refgen_pulse(n_spsym, C.c_float(bt), _ptr(out))
        return out

    def synth_gfsk(self, tones: np.ndarray, f0: float, bt: float, symbol_period: float, rate: int) -> np.ndarray:
        tones = np.ascontiguousarray(tones, np.uint8)
        n_spsym = int(0.5 + rate * symbol_period)
        out = np.zeros(tones.size * n_spsym, np.float32)
        self.lib.refgen_synth(_ptr(tones), tones.size, C.c_float(f0), C.c_float(bt), C.c_float(symbol_period), rate, _ptr(out))
        return out


class ReferenceReport:
    """The reference daemon's own reporting functions (postSpots / webClusterSpots / printSpots) with network, clock and stdout
    captured (oracle/_ref/libref_report.so, see ref_report_harness.c for the two lines edited in a temp copy)."""

    def __init__(self):
        path = os.path.join(HERE, "_ref", "libref_report.so")
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        self.lib = L = C.CDLL(path)
        L.ref_report_app_version.restype = C.c_char_p
        self.app_version = L.ref_report_app_version().decode()
        self.max_messages = L.ref_report_max_messages()

    @staticmethod
    def available() -> bool:
        return os.path.exists(os.path.join(HERE, "_ref", "libref_report.so"))

    def post_spots(self, spots: np.ndarray, rcall: str, rloc: str, dial_freq: int, unixtime: int) -> bytes:
        """-> the datagram postSpots() hands to send(); bytes 12..15 are the process-wide rand() id."""
        spots = np.ascontiguousarray(spots, result_dtype)
        assert spots.size <= self.max_messages
        out = C.create_string_buffer(4096)
        n = self.lib.ref_post_spots(_ptr(spots), C.c_uint32(spots.size), rcall.encode(), rloc.encode(), C.c_uint32(dial_freq), C.c_uint32(unixtime), out, 4096)
        return out.raw[:n] if n > 0 else b""

    def print_spots(self, spots: np.ndarray, dial_freq: int, unixtime: int) -> str:
        spots = np.ascontiguousarray(spots, result_dtype)
        out = C.create_string_buffer(1 << 16)
        self.lib.ref_print_spots(_ptr(spots), C.c_uint32(spots.size), C.c_uint32(dial_freq), C.c_uint32(unixtime), out, 1 << 16)
        return out.value.decode()

    def webcluster(self, spots: np.ndarray, rcall: str, rloc: str, dial_freq: int) -> list:
        """-> one {field name: value} dict per spot, as passed to curl_formadd()."""
        spots = np.ascontiguousarray(spots, result_dtype)
        out = C.create_string_buffer(224 * 4 * max(spots.size, 1))
        k = self.lib.ref_webcluster_spots(_ptr(spots), C.c_uint32(spots.size), rcall.encode(), rloc.encode(), C.c_uint32(dial_freq), out, 4 * max(spots.size, 1))
        pairs = [(out.raw[(2 * i) * 112:(2 * i + 1) * 112].split(b"\0")[0].decode(), out.raw[(2 * i + 1) * 112:(2 * i + 2) * 112].split(b"\0")[0]) for i in range(k)]
        return [dict(pairs[4 * j:4 * j + 4]) for j in range(k // 4)]
