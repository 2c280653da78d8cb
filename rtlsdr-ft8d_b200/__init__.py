"""rtlsdr-ft8d_b200 -- Python harness binding for libft8b200.so (the sm_100a implementation of the
rtlsdr-ft8d receive-and-decode hot path).

The product is the C-ABI shared library built from ``csrc/`` (see ``include/ft8b200.h``); this module
only loads it with ctypes and moves torch device tensors in and out, for the tests and benchmarks.
PyTorch is plumbing here (device memory, streams, torch.distributed), not the compute path.
There is no fallback: if the library is missing or no B200 is visible, calls raise.

The directory name contains a hyphen (it mirrors the reference's name), so import it through
``ft8b200_loader.load()`` at the repository root, which registers it as ``rtlsdr_ft8d_b200``.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FT8B200_LIB_PATH") or os.path.join(PKG_DIR, "libft8b200.so")  # override: A/B runs of an older build (tools/)

N_SLOT = 48000
WF_BYTES = 94208
RAW_SLOT_BYTES = 72_000_000

cand_dtype = np.dtype([("score", "<i2"), ("time_offset", "<i2"), ("freq_offset", "<i2"), ("time_sub", "u1"), ("freq_sub", "u1")])
msg_dtype = np.dtype([("text", "S25"), ("_pad", "u1"), ("hash", "<u2")])
status_dtype = np.dtype([("ldpc_errors", "<i4"), ("crc_extracted", "<u2"), ("crc_calculated", "<u2"), ("unpack_status", "<i4")])
result_dtype = np.dtype([("call", "S13"), ("loc", "S7"), ("freq", "<i4"), ("snr", "<i4")])


signal_dtype = np.dtype([("payload", "u1", 10), ("reserved", "u1", 2), ("f0_hz", "<f4"), ("t0_sec", "<f4"), ("amp", "<f4")])


def pack77_std(call_to: str, call_de: str, extra: str) -> bytes:
    """Standard (type 1) message -> 10-byte payload (host code of csrc/synth.cu); raises ValueError if not representable."""
    b = C.create_string_buffer(10)
    if lib().ft8b200_pack77_std(call_to.encode(), call_de.encode(), extra.encode(), b) != 0:
        raise ValueError(f"cannot pack {call_to} {call_de} {extra}")
    return b.raw


def pack77(msg: str):
    """pack77() of ft8_lib (pack.c:284-301): message text -> (10-byte payload, kind) with kind 0 = standard, 1 = free text."""
    b = C.create_string_buffer(10)
    kind = lib().ft8b200_pack77(msg.encode(), b)
    if kind < 0:
        raise ValueError("ft8b200_pack77")
    return b.raw, kind


def make_signals(items, gfsk: bool = False):
    """items: iterable of (payload bytes, f0_hz, t0_sec, amp) -> signal_dtype array.  gfsk: Gaussian-smoothed frequency, extended end
    symbols and ramps as gen_ft8 sends them (gen_ft8.c:28-102) instead of the self-test's plain FSK."""
    items = list(items)
    out = np.zeros(len(items), signal_dtype)
    out["reserved"][:, 0] = 1 if gfsk else 0
    for k, (payload, f0, t0, amp) in enumerate(items):
        out[k]["payload"] = np.frombuffer(payload, np.uint8)
        out[k]["f0_hz"], out[k]["t0_sec"], out[k]["amp"] = f0, t0, amp
    return out


class Config(C.Structure):
    _fields_ = [("device", C.c_int), ("max_slots", C.c_int), ("max_candidates", C.c_int), ("max_messages", C.c_int),
                ("min_score", C.c_int), ("ldpc_iterations", C.c_int)]


class WaterfallT(C.Structure):
    _fields_ = [("max_blocks", C.c_int), ("num_blocks", C.c_int), ("num_bins", C.c_int), ("time_osr", C.c_int),
                ("freq_osr", C.c_int), ("mag", C.c_void_p), ("block_stride", C.c_int), ("protocol", C.c_int)]


class MonitorConfig(C.Structure):
    _fields_ = [("f_min", C.c_float), ("f_max", C.c_float), ("sample_rate", C.c_int), ("time_osr", C.c_int), ("freq_osr", C.c_int),
                ("protocol", C.c_int)]


class MonitorT(C.Structure):
    _fields_ = [("symbol_period", C.c_float), ("block_size", C.c_int), ("subblock_size", C.c_int), ("nfft", C.c_int), ("fft_norm", C.c_float),
                ("window", C.c_void_p), ("last_frame", C.c_void_p), ("wf", WaterfallT), ("max_mag", C.c_float), ("fft_work", C.c_void_p),
                ("fft_cfg", C.c_void_p)]


def build(force: bool = False) -> str:
    """Compile csrc/*.cu into libft8b200.so for sm_100a (nvcc cross-compiles without a GPU)."""
    args = ["make", "-C", PKG_DIR, "-j8"]
    if force:
        subprocess.check_call(["make", "-C", PKG_DIR, "clean"], stdout=subprocess.DEVNULL)
    subprocess.check_call(args, stdout=subprocess.DEVNULL)
    return LIB_PATH


_lib = None


def lib() -> C.CDLL:
    """Load libft8b200.so (building it if the .so is absent). Raises if it cannot be loaded."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            build()
        L = C.CDLL(LIB_PATH)
        L.ft8b200_last_error.restype = C.c_char_p
        L.ft8b200_version.restype = C.c_char_p
        L.ft8b200_create.restype = C.c_void_p
        L.ft8b200_create.argtypes = [C.c_void_p]
        L.ft8b200_cuda_stream.restype = C.c_void_p
        L.ft8b200_kernel_launches.restype = C.c_uint64
        if hasattr(L, "ft8b200_stream_create"):
            L.ft8b200_stream_create.restype = C.c_void_p
            L.ft8b200_stream_count.restype = C.c_uint32
        L.ft8_decode.restype = C.c_bool
        for name in ("ft8b200_destroy", "ft8b200_cuda_stream", "ft8b200_sync", "ft8b200_kernel_launches", "ft8b200_stream_create",
                     "ft8b200_stream_destroy", "ft8b200_stream_flip", "ft8b200_stream_count"):
            if hasattr(L, name):
                getattr(L, name).argtypes = [C.c_void_p]
        _lib = L
    return _lib


def set_decode_variant(variant: int):
    """0 = node-centred belief propagation (default), 1 = edge-centred; process-wide."""
    if lib().ft8b200_set_decode_variant(int(variant)) != 0:
        raise ValueError(lib().ft8b200_last_error().decode())


class Ft8Error(RuntimeError):
    pass


def _p(t):
    """Device/host pointer of a torch tensor or numpy array (None -> NULL)."""
    if t is None:
        return C.c_void_p(0)
    if isinstance(t, np.ndarray):
        return C.c_void_p(t.ctypes.data)
    return C.c_void_p(t.data_ptr())


def _st(stream):
    """cudaStream_t to launch on: an explicit handle, or (default) torch's current stream so that the
    library's kernels are ordered with the torch ops that produced/consume the tensors."""
    if stream is None:
        import torch
        stream = torch.cuda.current_stream().cuda_stream
        if stream == 0:
            stream = 1  # cudaStreamLegacy: NULL means "the context's own stream" in the C ABI
    return C.c_void_p(stream)


class Context:
    """One ft8b200_ctx_t on one device. All tensors passed in must live on that device and be contiguous."""

    def __init__(self, device: int = 0, max_candidates: int = 120, max_messages: int = 50, min_score: int = 10, ldpc_iterations: int = 20):
        self.L = lib()
        self.cfg = Config(device, 1, max_candidates, max_messages, min_score, ldpc_iterations)
        self.h = self.L.ft8b200_create(C.byref(self.cfg))
        if not self.h:
            raise Ft8Error(self.L.ft8b200_last_error().decode())
        self.device = device
        self.K = max_candidates
        self.M = max_messages

    @classmethod
    def borrow(cls, handle: int, device: int, max_candidates: int = 120, max_messages: int = 50):
        """A non-owning view of a context created elsewhere (ft8b200_cluster_ctx): close() leaves it alone."""
        self = cls.__new__(cls)
        self.L = lib()
        self.h, self.device, self.K, self.M, self.borrowed = handle, device, max_candidates, max_messages, True
        return self

    def close(self):
        if self.h and not getattr(self, "borrowed", False):
            self.L.ft8b200_destroy(C.c_void_p(self.h))
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc != 0:
            raise Ft8Error(f"ft8b200 error {rc}: {self.L.ft8b200_last_error().decode()}")

    def sync(self):
        self._chk(self.L.ft8b200_sync(C.c_void_p(self.h)))

    @property
    def cuda_stream(self) -> int:
        return int(self.L.ft8b200_cuda_stream(C.c_void_p(self.h)) or 0)

    def launches(self) -> int:
        return int(self.L.ft8b200_kernel_launches(C.c_void_p(self.h)))

    # ---- stage-wise (device tensors) -------------------------------------------------------------
    def decimate(self, iq, n_streams: int, bytes_per_stream: int, stride: int | None = None, want_y2: bool = False, stream: int | None = None):
        import torch
        dev = iq.device
        stride = bytes_per_stream if stride is None else stride
        d_i = torch.empty((n_streams, N_SLOT), dtype=torch.float32, device=dev)
        d_q = torch.empty_like(d_i)
        cnt = torch.zeros(n_streams, dtype=torch.int32, device=dev)
        peak = torch.zeros(n_streams, dtype=torch.float32, device=dev)
        y2 = torch.zeros((n_streams, N_SLOT, 2), dtype=torch.int32, device=dev) if want_y2 else None
        self._chk(self.L.ft8b200_decimate(C.c_void_p(self.h), _p(iq), C.c_size_t(bytes_per_stream), C.c_size_t(stride), n_streams, _p(d_i), _p(d_q),
                                          _p(cnt), _p(peak), _p(y2), _st(stream)))
        return d_i, d_q, cnt, peak, y2

    def decimate_streams(self, iq, n_streams: int, slots_per_stream: int, bytes_per_slot: int, bytes_per_stream: int | None = None,
                         stride: int | None = None, want_y2: bool = False, stream: int | None = None):
        """Continuous streams cut into consecutive slots: rows = n_streams * slots_per_stream."""
        import torch
        dev = iq.device
        bytes_per_stream = slots_per_stream * bytes_per_slot if bytes_per_stream is None else bytes_per_stream
        stride = bytes_per_stream if stride is None else stride
        rows = n_streams * slots_per_stream
        d_i = torch.empty((rows, N_SLOT), dtype=torch.float32, device=dev)
        d_q = torch.empty_like(d_i)
        cnt = torch.zeros(rows, dtype=torch.int32, device=dev)
        peak = torch.zeros(rows, dtype=torch.float32, device=dev)
        y2 = torch.zeros((rows, N_SLOT, 2), dtype=torch.int32, device=dev) if want_y2 else None
        self._chk(self.L.ft8b200_decimate_streams(C.c_void_p(self.h), _p(iq), C.c_size_t(bytes_per_stream), C.c_size_t(stride), n_streams,
                                                  slots_per_stream, C.c_size_t(bytes_per_slot), _p(d_i), _p(d_q), _p(cnt), _p(peak), _p(y2), _st(stream)))
        return d_i, d_q, cnt, peak, y2

    def process_raw_streams(self, iq, n_streams: int, slots_per_stream: int, bytes_per_slot: int = RAW_SLOT_BYTES, bytes_per_stream: int | None = None,
                            stride: int | None = None, stream: int | None = None):
        bytes_per_stream = slots_per_stream * bytes_per_slot if bytes_per_stream is None else bytes_per_stream
        stride = bytes_per_stream if stride is None else stride
        self._chk(self.L.ft8b200_process_raw_streams(C.c_void_p(self.h), _p(iq), C.c_size_t(bytes_per_stream), C.c_size_t(stride), n_streams,
                                                     slots_per_stream, C.c_size_t(bytes_per_slot), _st(stream)))

    def condition(self, d_i, d_q, peak, stream: int | None = None):
        self._chk(self.L.ft8b200_condition(C.c_void_p(self.h), _p(d_i), _p(d_q), _p(peak), d_i.shape[0], _st(stream)))

    def waterfall(self, d_i, d_q, peak=None, stream: int | None = None):
        import torch
        n = d_i.shape[0]
        mag = torch.empty((n, WF_BYTES), dtype=torch.uint8, device=d_i.device)
        self._chk(self.L.ft8b200_waterfall(C.c_void_p(self.h), _p(d_i), _p(d_q), _p(peak), n, _p(mag), _st(stream)))
        return mag

    def find_sync(self, mag, num_blocks=92, num_bins=256, time_osr=2, freq_osr=2, stream: int | None = None):
        import torch
        n = mag.shape[0]
        cand = torch.zeros((n, self.K, 8), dtype=torch.uint8, device=mag.device)
        ncand = torch.zeros(n, dtype=torch.int32, device=mag.device)
        self._chk(self.L.ft8b200_find_sync(C.c_void_p(self.h), _p(mag), C.c_size_t(mag.stride(0)), n, num_blocks, num_bins, time_osr, freq_osr,
                                           _p(cand), _p(ncand), _st(stream)))
        return cand, ncand

    def decode(self, mag, cand, ncand, num_blocks=92, num_bins=256, time_osr=2, freq_osr=2, want_plain=False, want_llr=False, stream: int | None = None):
        import torch
        n = mag.shape[0]
        dev = mag.device
        ok = torch.zeros((n, self.K), dtype=torch.uint8, device=dev)
        stage = torch.zeros((n, self.K), dtype=torch.uint8, device=dev)
        status = torch.zeros((n, self.K, 12), dtype=torch.uint8, device=dev)
        msg = torch.zeros((n, self.K, 28), dtype=torch.uint8, device=dev)
        plain = torch.zeros((n, self.K, 174), dtype=torch.uint8, device=dev) if want_plain else None
        llr = torch.zeros((n, self.K, 174), dtype=torch.float32, device=dev) if want_llr else None
        self._chk(self.L.ft8b200_decode(C.c_void_p(self.h), _p(mag), C.c_size_t(mag.stride(0)), n, num_blocks, num_bins, time_osr, freq_osr,
                                        _p(cand), _p(ncand), _p(ok), _p(stage), _p(status), _p(msg), _p(plain), _p(llr), _st(stream)))
        return ok, stage, status, msg, plain, llr

    def set_osd(self, order: int, max_hard_errors: int = -1):
        """Ordered-statistics decoding after BP: order 0 (off), 1 or 2; max_hard_errors < 0 = FT8B200_OSD_DEFAULT_MAX_HARD."""
        self._chk(self.L.ft8b200_set_osd(C.c_void_p(self.h), int(order), int(max_hard_errors)))

    def osd(self, llr, ncand, ok, stage, status, msg, plain=None, want_cw=False, stream: int | None = None):
        """Stage-wise OSD over ft8b200_decode's outputs (updated in place) -> (osd uint8[n, K], osd_hard int32[n, K], cw uint8[n, K, 174] or None)."""
        import torch
        n = llr.shape[0]
        dev = llr.device
        osd = torch.zeros((n, self.K), dtype=torch.uint8, device=dev)
        hard = torch.zeros((n, self.K), dtype=torch.int32, device=dev)
        cw = torch.zeros((n, self.K, 174), dtype=torch.uint8, device=dev) if want_cw else None
        self._chk(self.L.ft8b200_osd(C.c_void_p(self.h), _p(llr), n, _p(ncand), _p(ok), _p(stage), _p(status), _p(msg), _p(plain), _p(osd), _p(hard),
                                     _p(cw), _st(stream)))
        return osd, hard, cw

    def set_ap(self, on: int, max_hard_errors: int = -1):
        """A-priori decoding of "CQ ??? ???" after BP and OSD: 0 (off) or 1; max_hard_errors < 0 = FT8B200_AP_DEFAULT_MAX_HARD."""
        self._chk(self.L.ft8b200_set_ap(C.c_void_p(self.h), int(on), int(max_hard_errors)))

    def ap(self, llr, ncand, ok, stage, status, msg, plain=None, stream: int | None = None):
        """Stage-wise AP over ft8b200_decode's (and ft8b200_osd's) outputs, updated in place -> (ap uint8[n, K], ap_hard int32[n, K])."""
        import torch
        n = llr.shape[0]
        dev = llr.device
        ap = torch.zeros((n, self.K), dtype=torch.uint8, device=dev)
        hard = torch.zeros((n, self.K), dtype=torch.int32, device=dev)
        self._chk(self.L.ft8b200_ap(C.c_void_p(self.h), _p(llr), n, _p(ncand), _p(ok), _p(stage), _p(status), _p(msg), _p(plain), _p(ap), _p(hard),
                                    _st(stream)))
        return ap, hard

    def ap_workspace_ptrs(self):
        """Device pointers (ap, ap_hard) of the last batch decoded with AP on (0 before that)."""
        a, b = C.c_void_p(0), C.c_void_p(0)
        self._chk(self.L.ft8b200_ap_workspace(C.c_void_p(self.h), C.byref(a), C.byref(b)))
        return a.value or 0, b.value or 0

    def set_finesync(self, on: int, max_hard_errors: int = -1):
        """Fine-sync decoding after BP, OSD and AP: 0 (off) or 1; max_hard_errors < 0 = FT8B200_FINESYNC_DEFAULT_MAX_HARD."""
        self._chk(self.L.ft8b200_set_finesync(C.c_void_p(self.h), int(on), int(max_hard_errors)))

    def finesync(self, d_i, d_q, cand, ncand, ok, stage, status, msg, plain=None, want_llr=False, stream: int | None = None):
        """Stage-wise fine sync on slots d_i / d_q float32 [n, 48000] over ft8b200_decode's (and OSD's, AP's) outputs, updated in place
        -> (fs uint8[n, K], fs_hard int32[n, K], grid int32[n, K, 2] of (dt samples, df steps), llr float32[n, K, 174] or None); grid
        and llr are written for the candidates at stage 1 or 2 only (zeros elsewhere)."""
        import torch
        n = d_i.shape[0]
        dev = d_i.device
        fs = torch.zeros((n, self.K), dtype=torch.uint8, device=dev)
        hard = torch.zeros((n, self.K), dtype=torch.int32, device=dev)
        grid = torch.zeros((n, self.K, 2), dtype=torch.int32, device=dev)
        llr = torch.zeros((n, self.K, 174), dtype=torch.float32, device=dev) if want_llr else None
        self._chk(self.L.ft8b200_finesync(C.c_void_p(self.h), _p(d_i), _p(d_q), n, _p(cand), _p(ncand), _p(ok), _p(stage), _p(status), _p(msg),
                                          _p(plain), _p(fs), _p(hard), _p(grid), _p(llr), _st(stream)))
        return fs, hard, grid, llr

    def finesync_workspace_ptrs(self):
        """Device pointers (fs, fs_hard) of pass 1 of the last batch decoded with fine sync on (0 before that)."""
        a, b = C.c_void_p(0), C.c_void_p(0)
        self._chk(self.L.ft8b200_finesync_workspace(C.c_void_p(self.h), C.byref(a), C.byref(b)))
        return a.value or 0, b.value or 0

    def set_finesync_deep(self, on: int, max_hard_errors: int = -1):
        """Deep fine sync (sets a, b, c and OSD / AP on them; only while fine sync is on): 0 (off) or 1; max_hard_errors < 0 =
        FT8B200_FINESYNC_DEEP_DEFAULT_MAX_HARD."""
        self._chk(self.L.ft8b200_set_finesync_deep(C.c_void_p(self.h), int(on), int(max_hard_errors)))

    def finesync_sets(self, d_i, d_q, cand, ncand, stage, stream: int | None = None):
        """Deep fine sync's front half on slots d_i / d_q float32 [n, 48000] -> (grid int32[n, K, 2], llr float32[3, n, K, 174] of sets
        a, b, c), written for the candidates at stage 1 or 2 only (zeros elsewhere)."""
        import torch
        n = d_i.shape[0]
        dev = d_i.device
        grid = torch.zeros((n, self.K, 2), dtype=torch.int32, device=dev)
        llr = torch.zeros((3, n, self.K, 174), dtype=torch.float32, device=dev)
        self._chk(self.L.ft8b200_finesync_sets(C.c_void_p(self.h), _p(d_i), _p(d_q), n, _p(cand), _p(ncand), _p(stage), _p(grid), _p(llr),
                                               _st(stream)))
        return grid, llr

    def finesync_deep_workspace_ptrs(self):
        """Device pointer of fs_how (uint8 [n, K]; 0 = not a fine-sync decode, else 1 + 3 set + decoder) of pass 1 of the last batch, or
        stage-wise ft8b200_finesync, run with deep fine sync (0 before that)."""
        a = C.c_void_p(0)
        self._chk(self.L.ft8b200_finesync_deep_workspace(C.c_void_p(self.h), C.byref(a)))
        return a.value or 0

    def set_passes(self, passes: int):
        """Multi-pass decoding with signal subtraction on the daemon path: 1 (default, one pass), 2 or 3 (ft8b200_set_passes)."""
        self._chk(self.L.ft8b200_set_passes(C.c_void_p(self.h), int(passes)))

    def subtract(self, d_i, d_q, cand, cw, nmsg, out=None, stream: int | None = None):
        """Stage-wise ft8b200_subtract: slots float32 [n, 48000] (I, Q), per slot up to M messages -- cand uint8 [n, M, 8]
        (candidate_t), cw uint8 [n, M, 174] (codeword bits), nmsg int32 [n] -> (residual I, residual Q, grid int32 [n, M, 2] of
        (dt samples, df steps)).  out = (ri, rq) to write the residual into (may be d_i, d_q)."""
        import torch
        n = d_i.shape[0]
        ri, rq = out if out is not None else (torch.empty_like(d_i), torch.empty_like(d_q))
        grid = torch.zeros((n, self.M, 2), dtype=torch.int32, device=d_i.device)
        self._chk(self.L.ft8b200_subtract(C.c_void_p(self.h), _p(d_i), _p(d_q), n, _p(cand), _p(cw), _p(nmsg), _p(ri), _p(rq), _p(grid), _st(stream)))
        return ri, rq, grid

    def osd_workspace_ptrs(self):
        """Device pointers (osd, osd_hard) of the last batch decoded with OSD on (0 before that)."""
        a, b = C.c_void_p(0), C.c_void_p(0)
        self._chk(self.L.ft8b200_osd_workspace(C.c_void_p(self.h), C.byref(a), C.byref(b)))
        return a.value or 0, b.value or 0

    def spots(self, cand, ncand, ok, msg, freq_osr=2, want_log=True, stream: int | None = None):
        import torch
        n = cand.shape[0]
        dev = cand.device
        res = torch.zeros((n, self.M, 28), dtype=torch.uint8, device=dev)
        nres = torch.zeros(n, dtype=torch.int32, device=dev)
        umsg = torch.zeros((n, self.M, 28), dtype=torch.uint8, device=dev) if want_log else None
        ufreq = torch.zeros((n, self.M), dtype=torch.float32, device=dev) if want_log else None
        uscore = torch.zeros((n, self.M), dtype=torch.int32, device=dev) if want_log else None
        self._chk(self.L.ft8b200_spots(C.c_void_p(self.h), n, freq_osr, _p(cand), _p(ncand), _p(ok), _p(msg), _p(res), _p(nres), _p(umsg), _p(ufreq),
                                       _p(uscore), C.c_void_p(0), _st(stream)))
        return res, nres, umsg, ufreq, uscore

    def monitor_waterfall(self, audio, sample_rate=12000, time_osr=2, freq_osr=2, protocol=1, stream: int | None = None):
        """Batched 12 kHz monitor: audio float32 [n_slots, n_samples] on device -> (mag uint8 [n_slots, bytes], num_blocks)."""
        import torch
        n_slots, n_samples = audio.shape
        block = int(np.float32(sample_rate) * np.float32(0.048 if protocol == 0 else 0.160))
        bins = int(np.float32(sample_rate) * np.float32(0.048 if protocol == 0 else 0.160) / 2)
        max_blocks = int(np.float32(7.5 if protocol == 0 else 15.0) / np.float32(0.048 if protocol == 0 else 0.160))
        nb = min(max_blocks, n_samples // block)
        stride = time_osr * freq_osr * bins
        mag = torch.zeros((n_slots, max(nb, 1) * stride), dtype=torch.uint8, device=audio.device)
        out_nb = C.c_int(0)
        self._chk(self.L.ft8b200_monitor_waterfall(C.c_void_p(self.h), _p(audio), C.c_size_t(audio.stride(0)), n_samples, n_slots, sample_rate, time_osr,
                                                   freq_osr, protocol, _p(mag), C.c_size_t(mag.stride(0)), C.byref(out_nb), _st(stream)))
        return mag, out_nb.value

    # ---- device-side signal synthesis (csrc/synth.cu) ---------------------------------------------------
    @staticmethod
    def _sig_args(signals, first):
        signals = np.ascontiguousarray(signals, signal_dtype)
        first = np.ascontiguousarray(first, np.int32)
        assert first[0] == 0 and first[-1] == signals.size
        return signals, first

    def synth_raw(self, signals, first, noise_lsb: float, seed: int, first_slot_index: int = 0, bytes_per_slot: int = RAW_SLOT_BYTES, out=None):
        """signals: signal_dtype array, first: int32[n_slots+1] -> uint8 device tensor [n_slots, bytes_per_slot] of raw RTL IQ."""
        import torch
        signals, first = self._sig_args(signals, first)
        n_slots = first.size - 1
        stride = (bytes_per_slot + 15) // 16 * 16
        if out is None:
            out = torch.empty((n_slots, stride), dtype=torch.uint8, device=torch.device("cuda", self.device))
        self._chk(self.L.ft8b200_synth_raw(C.c_void_p(self.h), _p(signals), _p(first), n_slots, C.c_float(noise_lsb), C.c_uint64(seed), first_slot_index,
                                           _p(out), C.c_size_t(out.stride(0)), C.c_size_t(bytes_per_slot), _st(None)))
        return out

    def synth_slots(self, signals, first, noise_sigma: float, seed: int, first_slot_index: int = 0, n_samples: int = N_SLOT):
        import torch
        signals, first = self._sig_args(signals, first)
        n_slots = first.size - 1
        d_i = torch.empty((n_slots, n_samples), dtype=torch.float32, device=torch.device("cuda", self.device))
        d_q = torch.empty_like(d_i)
        self._chk(self.L.ft8b200_synth_slots(C.c_void_p(self.h), _p(signals), _p(first), n_slots, C.c_float(noise_sigma), C.c_uint64(seed), first_slot_index,
                                             _p(d_i), _p(d_q), C.c_size_t(n_samples), n_samples, _st(None)))
        return d_i, d_q

    def synth_audio(self, signals, first, protocol: int, noise_sigma: float, seed: int, first_slot_index: int = 0, n_samples: int = 180_000):
        import torch
        signals, first = self._sig_args(signals, first)
        n_slots = first.size - 1
        d_a = torch.empty((n_slots, n_samples), dtype=torch.float32, device=torch.device("cuda", self.device))
        self._chk(self.L.ft8b200_synth_audio(C.c_void_p(self.h), _p(signals), _p(first), n_slots, protocol, C.c_float(noise_sigma), C.c_uint64(seed),
                                             first_slot_index, _p(d_a), C.c_size_t(n_samples), n_samples, _st(None)))
        return d_a

    def encode_tones(self, payloads, protocol: int = 1) -> np.ndarray:
        payloads = np.ascontiguousarray(payloads, np.uint8).reshape(-1, 10)
        tones = np.zeros((payloads.shape[0], 105), np.uint8)
        self._chk(self.L.ft8b200_encode_tones(C.c_void_p(self.h), _p(payloads), payloads.shape[0], protocol, _p(tones)))
        return tones[:, :79] if protocol == 1 else tones

    # ---- whole path ----------------------------------------------------------------------------------
    def process_raw(self, iq, n_slots: int, bytes_per_stream: int = RAW_SLOT_BYTES, stride: int | None = None, stream: int | None = None):
        stride = bytes_per_stream if stride is None else stride
        self._chk(self.L.ft8b200_process_raw(C.c_void_p(self.h), _p(iq), C.c_size_t(bytes_per_stream), C.c_size_t(stride), n_slots, _st(stream)))

    def process_slots(self, d_i, d_q, stream: int | None = None):
        self._chk(self.L.ft8b200_process_slots(C.c_void_p(self.h), _p(d_i), _p(d_q), d_i.shape[0], _st(stream)))

    def process_conditioned(self, d_i, d_q, peak, stream: int | None = None):
        """Unconditioned samples + their peak max(|I|,|Q|) per slot: decoder()'s 0.5/peak scale is applied on load."""
        self._chk(self.L.ft8b200_process_conditioned(C.c_void_p(self.h), _p(d_i), _p(d_q), _p(peak), d_i.shape[0], _st(stream)))

    def fetch_results(self, n_slots: int, stream: int | None = None, out=None):
        """Records of the last batch -> host.  out = (result_dtype[n, M], int32[n]) arrays to fill (e.g. views of pinned memory:
        the copy then runs at the link's rate instead of through the driver's staging buffer); fresh arrays otherwise."""
        res, nres = out if out is not None else (np.zeros((n_slots, self.M), result_dtype), np.zeros(n_slots, np.int32))
        assert res.dtype == result_dtype and res.shape == (n_slots, self.M) and nres.dtype == np.int32 and nres.shape == (n_slots,)
        self._chk(self.L.ft8b200_fetch_results(C.c_void_p(self.h), n_slots, _p(res), _p(nres), _st(stream)))
        return res, nres

    def set_profiling(self, on: bool):
        self._chk(self.L.ft8b200_set_profiling(C.c_void_p(self.h), int(on)))

    def set_protocol(self, protocol: int):
        """0 = FT4, 1 = FT8 (ftx_protocol_t) for find_sync / decode."""
        self._chk(self.L.ft8b200_set_protocol(C.c_void_p(self.h), int(protocol)))

    def set_decimator_variant(self, variant: int):
        """0 = streaming cic_block_sums kernel; >= 1 = persistent bulk-copy (TMA) kernel, shape index 1..6."""
        self._chk(self.L.ft8b200_set_decimator_variant(C.c_void_p(self.h), int(variant)))

    def selfcheck_pade(self):
        """All 2^32 float patterns through variant 0's inlined tanh/atanh vs the full-division expressions: 5 counters."""
        c = (C.c_uint64 * 5)()
        self._chk(self.L.ft8b200_selfcheck_pade(C.c_void_p(self.h), c))
        return [int(v) for v in c]

    def selfcheck_quantiser(self):
        """All float patterns the dB quantiser can see, straight-line kernel form vs threshold search: (mismatches, corrected, far)."""
        c = (C.c_uint64 * 3)()
        self._chk(self.L.ft8b200_selfcheck_quantiser(C.c_void_p(self.h), c))
        return [int(v) for v in c]

    def unpack77_batch(self, payloads):
        """n 77-bit payloads (uint8 [n, 10]) through the device unpacker -> (list of texts, int32 status[n])."""
        payloads = np.ascontiguousarray(payloads, np.uint8).reshape(-1, 10)
        n = payloads.shape[0]
        text = np.zeros((n, 32), np.uint8)
        status = np.zeros(n, np.int32)
        self._chk(self.L.ft8b200_unpack77_batch(C.c_void_p(self.h), _p(payloads), n, _p(text), _p(status)))
        return [bytes(t).split(b"\0")[0].decode("ascii", "replace") for t in text], status

    def set_overlap(self, groups: int):
        self._chk(self.L.ft8b200_set_overlap(C.c_void_p(self.h), int(groups)))

    def stage_times(self):
        """ms per stage of the last process_* call: dict(block_sums, comb_fir, waterfall, sync, decode, spots), and later_passes
        (subtraction + passes 2 and 3) when the context decodes in more than one pass."""
        ms = (C.c_float * 7)(*([-2.0] * 7))
        self._chk(self.L.ft8b200_stage_times(C.c_void_p(self.h), ms, 7))
        names = ("block_sums", "comb_fir", "waterfall", "sync", "decode", "spots", "later_passes")
        return {k: float(x) for k, x in zip(names, ms) if x != -2.0}

    def results_device_ptrs(self):
        a, b = C.c_void_p(0), C.c_void_p(0)
        self._chk(self.L.ft8b200_results_device(C.c_void_p(self.h), C.byref(a), C.byref(b)))
        return a.value, b.value

    def results_tensors(self, n_slots: int):
        """Zero-copy torch views of the last batch's device-resident outputs: (uint8[n, M, 28], int32[n])."""
        import torch
        a, b = self.results_device_ptrs()

        class _Arr:
            def __init__(self, ptr, shape, typestr):
                self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2}

        dev = torch.device("cuda", self.device)
        return (torch.as_tensor(_Arr(a, (n_slots, self.M, 28), "|u1"), device=dev), torch.as_tensor(_Arr(b, (n_slots,), "<i4"), device=dev))

    def workspace_ptrs(self):
        ptrs = [C.c_void_p(0) for _ in range(9)]
        self._chk(self.L.ft8b200_workspace(C.c_void_p(self.h), *[C.byref(p) for p in ptrs]))
        names = ("i", "q", "peak", "mag", "cand", "ncand", "ok", "status", "msg")
        return {k: p.value for k, p in zip(names, ptrs)}

    def process_raw_host(self, iq_host: np.ndarray, n_slots: int, bytes_per_stream: int = RAW_SLOT_BYTES):
        res = np.zeros((n_slots, self.M), result_dtype)
        nres = np.zeros(n_slots, np.int32)
        self._chk(self.L.ft8b200_process_raw_host(C.c_void_p(self.h), _p(iq_host), C.c_size_t(bytes_per_stream), n_slots, _p(res), _p(nres)))
        return res, nres

    def process_slots_host(self, i_host: np.ndarray, q_host: np.ndarray):
        n = i_host.shape[0]
        res = np.zeros((n, self.M), result_dtype)
        nres = np.zeros(n, np.int32)
        self._chk(self.L.ft8b200_process_slots_host(C.c_void_p(self.h), _p(i_host), _p(q_host), n, _p(res), _p(nres)))
        return res, nres


class Pipe:
    """ft8b200_pipe_t: `depth` batches in flight on one GPU (see include/ft8b200.h)."""

    def __init__(self, device: int = 0, depth: int = 2, max_candidates: int = 120, max_messages: int = 50, min_score: int = 10,
                 ldpc_iterations: int = 20):
        self.L = lib()
        self.L.ft8b200_pipe_create.restype = C.c_void_p
        self.L.ft8b200_pipe_error.restype = C.c_char_p
        self.L.ft8b200_pipe_kernel_launches.restype = C.c_uint64
        self.cfg = Config(device, 1, max_candidates, max_messages, min_score, ldpc_iterations)
        self.h = self.L.ft8b200_pipe_create(C.byref(self.cfg), depth)
        if not self.h:
            raise Ft8Error(self.L.ft8b200_last_error().decode())
        self.depth = depth
        self.M = max_messages

    @classmethod
    def borrow(cls, handle: int, device: int, depth: int, max_messages: int = 50):
        """A non-owning view of a pipe created elsewhere (ft8b200_cluster_pipe)."""
        self = cls.__new__(cls)
        self.L = lib()
        self.L.ft8b200_pipe_error.restype = C.c_char_p
        self.L.ft8b200_pipe_kernel_launches.restype = C.c_uint64
        self.cfg = Config(device, 1, 120, max_messages, 10, 20)
        self.h, self.depth, self.M, self.borrowed = handle, depth, max_messages, True
        return self

    def close(self):
        if self.h and not getattr(self, "borrowed", False):
            self.L.ft8b200_pipe_destroy(C.c_void_p(self.h))
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc < 0:
            raise Ft8Error(f"ft8b200 pipe error {rc}: {self.L.ft8b200_pipe_error(C.c_void_p(self.h)).decode()}")
        return rc

    def in_flight(self) -> int:
        return self.L.ft8b200_pipe_in_flight(C.c_void_p(self.h))

    def depend_on(self, event):
        """event: torch.cuda.Event already recorded; the next submitted batch waits for it on the device."""
        self._chk(self.L.ft8b200_pipe_depend_on(C.c_void_p(self.h), C.c_void_p(event.cuda_event)))

    def set_mode(self, serial: bool, decimator_variant: int = -1):
        self._chk(self.L.ft8b200_pipe_set_mode(C.c_void_p(self.h), 1 if serial else 0, int(decimator_variant)))

    def timeline(self, max_batches: int = 64):
        """float32[n, 6, 2]: begin/end (ms since set_profiling(True)) of the six stages of each collected batch."""
        out = np.zeros((max_batches, 6, 2), np.float32)
        n = self._chk(self.L.ft8b200_pipe_timeline(C.c_void_p(self.h), _p(out), max_batches))
        return out[:n]

    def set_partition(self, back_sms: int):
        """Disjoint SM sets (green contexts) for the front end of batch n+1 and the back end of batch n; 0 removes it.
        Returns (front_sms, back_sms) as provisioned by the driver."""
        f, b = C.c_int(0), C.c_int(0)
        self._chk(self.L.ft8b200_pipe_set_partition(C.c_void_p(self.h), int(back_sms), C.byref(f), C.byref(b)))
        return f.value, b.value

    def set_osd(self, order: int, max_hard_errors: int = -1):
        """Context.set_osd on every lane; not while batches are in flight."""
        self._chk(self.L.ft8b200_pipe_set_osd(C.c_void_p(self.h), int(order), int(max_hard_errors)))

    def set_ap(self, on: int, max_hard_errors: int = -1):
        """Context.set_ap on every lane; not while batches are in flight."""
        self._chk(self.L.ft8b200_pipe_set_ap(C.c_void_p(self.h), int(on), int(max_hard_errors)))

    def set_finesync(self, on: int, max_hard_errors: int = -1):
        """Context.set_finesync on every lane; not while batches are in flight."""
        self._chk(self.L.ft8b200_pipe_set_finesync(C.c_void_p(self.h), int(on), int(max_hard_errors)))

    def set_finesync_deep(self, on: int, max_hard_errors: int = -1):
        """Context.set_finesync_deep on every lane; not while batches are in flight."""
        self._chk(self.L.ft8b200_pipe_set_finesync_deep(C.c_void_p(self.h), int(on), int(max_hard_errors)))

    def set_passes(self, passes: int):
        """Context.set_passes on every lane; not while batches are in flight."""
        self._chk(self.L.ft8b200_pipe_set_passes(C.c_void_p(self.h), int(passes)))

    def set_back_chain(self, on: bool):
        """Back ends of consecutive batches serialised on the back partition (what the autotune probes with)."""
        self._chk(self.L.ft8b200_pipe_set_back_chain(C.c_void_p(self.h), int(on)))

    def partition_smids(self, which: int):
        """Hardware SM ids (%smid) the front (0) / back (1) partition runs on (diagnostic)."""
        m = (C.c_uint32 * 8)()
        self._chk(self.L.ft8b200_pipe_partition_smids(C.c_void_p(self.h), int(which), m))
        return [32 * w + b for w in range(8) for b in range(32) if (m[w] >> b) & 1]

    def autotune(self, iq, n_slots: int, candidates=(24, 32, 40), batches: int = 12, bytes_per_stream: int = RAW_SLOT_BYTES, stride: int | None = None):
        """ft8b200_pipe_autotune: measure every (back_sms, comb+FIR placement) point on `iq`, keep the fastest.
        -> dict(back_sms, comb_front, points={(back_sms, comb_front): ms_per_batch})."""
        stride = bytes_per_stream if stride is None else stride
        cand = (C.c_int * len(candidates))(*candidates)
        ms = (C.c_float * (2 * len(candidates)))()
        b, cf = C.c_int(0), C.c_int(0)
        self._chk(self.L.ft8b200_pipe_autotune(C.c_void_p(self.h), _p(iq), C.c_size_t(bytes_per_stream), C.c_size_t(stride), n_slots, cand, len(candidates),
                                               batches, C.byref(b), C.byref(cf), ms))
        return {"back_sms": b.value, "comb_front": cf.value,
                "points": {"%d/%s" % (s, "front" if k else "back"): float(ms[2 * i + k]) for i, s in enumerate(candidates) for k in (0, 1) if ms[2 * i + k] > 0}}

    def submit(self, iq, n_slots: int, bytes_per_stream: int = RAW_SLOT_BYTES, stride: int | None = None):
        """iq: device tensor (already complete on the device) -> queued on the next lane."""
        stride = bytes_per_stream if stride is None else stride
        self._chk(self.L.ft8b200_pipe_submit(C.c_void_p(self.h), _p(iq), C.c_size_t(bytes_per_stream), C.c_size_t(stride), n_slots))

    def submit_streams(self, iq, n_streams: int, slots_per_stream: int, bytes_per_slot: int = RAW_SLOT_BYTES, stride: int | None = None):
        """iq: device tensor of n_streams receiver streams, each slots_per_stream consecutive slots (decimator state carried through
        the slot boundaries) -> one batch of n_streams * slots_per_stream slots, records in (stream, slot) order."""
        bytes_per_stream = slots_per_stream * bytes_per_slot
        stride = bytes_per_stream if stride is None else stride
        self._chk(self.L.ft8b200_pipe_submit_streams(C.c_void_p(self.h), _p(iq), C.c_size_t(bytes_per_stream), C.c_size_t(stride), n_streams,
                                                     slots_per_stream, C.c_size_t(bytes_per_slot)))

    def submit_host(self, iq_host, n_slots: int, bytes_per_stream: int = RAW_SLOT_BYTES):
        self._chk(self.L.ft8b200_pipe_submit_host(C.c_void_p(self.h), _p(iq_host), C.c_size_t(bytes_per_stream), n_slots))

    def submit_slots(self, d_i, d_q, peak=None):
        """Device tensors float32 [n, 48000] per rail (peak: unconditioned samples + their max per slot)."""
        self._chk(self.L.ft8b200_pipe_submit_slots(C.c_void_p(self.h), _p(d_i), _p(d_q), _p(peak), d_i.shape[0]))

    def submit_slots_host(self, h_i, h_q):
        """Conditioned samples in (pinned) host memory: numpy float32 [n, 48000] per rail."""
        self._chk(self.L.ft8b200_pipe_submit_slots_host(C.c_void_p(self.h), _p(h_i), _p(h_q), h_i.shape[0]))

    def collect(self, capacity_slots: int):
        res = np.zeros((capacity_slots, self.M), result_dtype)
        nres = np.zeros(capacity_slots, np.int32)
        n = self._chk(self.L.ft8b200_pipe_collect(C.c_void_p(self.h), _p(res), _p(nres), capacity_slots))
        return res[:n], nres[:n]

    def collect_device(self):
        """Oldest batch as zero-copy torch views of the lane's device buffers: (uint8[n, M, 28], int32[n])."""
        import torch
        a, b = C.c_void_p(0), C.c_void_p(0)
        n = self._chk(self.L.ft8b200_pipe_collect_device(C.c_void_p(self.h), C.byref(a), C.byref(b)))

        class _Arr:
            def __init__(self, ptr, shape, typestr):
                self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2}

        dev = torch.device("cuda", self.cfg.device)
        return (torch.as_tensor(_Arr(a.value, (n, self.M, 28), "|u1"), device=dev), torch.as_tensor(_Arr(b.value, (n,), "<i4"), device=dev))

    def set_profiling(self, on: bool):
        self._chk(self.L.ft8b200_pipe_set_profiling(C.c_void_p(self.h), int(on)))

    def stage_times(self):
        """(dict of summed ms per stage, number of batches) since profiling was switched on."""
        ms = (C.c_double * 6)()
        nb = C.c_uint64(0)
        self._chk(self.L.ft8b200_pipe_stage_times(C.c_void_p(self.h), ms, 6, C.byref(nb)))
        return dict(zip(("block_sums", "comb_fir", "waterfall", "sync", "decode", "spots"), [float(x) for x in ms])), int(nb.value)

    def launches(self) -> int:
        return int(self.L.ft8b200_pipe_kernel_launches(C.c_void_p(self.h)))


class Cluster:
    """ft8b200_cluster_t: every visible GPU from ONE process, spot records gathered with NCCL (see include/ft8b200.h)."""

    def __init__(self, n_devices: int = 0, depth: int = 2, max_candidates: int = 120, max_messages: int = 50, min_score: int = 10, ldpc_iterations: int = 20):
        self.L = L = lib()
        L.ft8b200_cluster_create.restype = C.c_void_p
        L.ft8b200_cluster_error.restype = C.c_char_p
        L.ft8b200_cluster_ctx.restype = C.c_void_p
        L.ft8b200_cluster_pipe.restype = C.c_void_p
        L.ft8b200_cluster_gathers.restype = C.c_uint64
        L.ft8b200_cluster_kernel_launches.restype = C.c_uint64
        self.cfg = Config(0, 1, max_candidates, max_messages, min_score, ldpc_iterations)
        self.h = L.ft8b200_cluster_create(C.byref(self.cfg), n_devices, depth)
        if not self.h:
            raise Ft8Error(L.ft8b200_last_error().decode() or "ft8b200_cluster_create failed (see stderr)")
        self.n = L.ft8b200_cluster_devices(C.c_void_p(self.h))
        self.depth, self.K, self.M = depth, max_candidates, max_messages

    def close(self):
        if self.h:
            self.L.ft8b200_cluster_destroy(C.c_void_p(self.h))
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc < 0:
            raise Ft8Error(f"ft8b200 cluster error {rc}: {self.L.ft8b200_cluster_error(C.c_void_p(self.h)).decode()}")
        return rc

    def ctx(self, d: int) -> "Context":
        return Context.borrow(self.L.ft8b200_cluster_ctx(C.c_void_p(self.h), d), d, self.K, self.M)

    def pipe(self, d: int) -> "Pipe":
        return Pipe.borrow(self.L.ft8b200_cluster_pipe(C.c_void_p(self.h), d), d, self.depth, self.M)

    def shard(self, n_items: int, d: int):
        a, b = C.c_int(0), C.c_int(0)
        self._chk(self.L.ft8b200_cluster_shard(C.c_void_p(self.h), n_items, d, C.byref(a), C.byref(b)))
        return a.value, b.value

    def in_flight(self) -> int:
        return self.L.ft8b200_cluster_in_flight(C.c_void_p(self.h))

    def submit(self, tensors, counts, bytes_per_stream: int = RAW_SLOT_BYTES, stride: int | None = None, slots_per_stream: int = 1, bytes_per_slot: int = RAW_SLOT_BYTES):
        """tensors[d]: uint8 device tensor on device d (or None when counts[d] == 0)."""
        stride = bytes_per_stream if stride is None else stride
        ptrs = (C.c_void_p * self.n)(*[(t.data_ptr() if t is not None else 0) for t in tensors])
        cnt = (C.c_int * self.n)(*counts)
        if slots_per_stream > 1:
            self._chk(self.L.ft8b200_cluster_submit_streams(C.c_void_p(self.h), ptrs, C.c_size_t(bytes_per_stream), C.c_size_t(stride), cnt, slots_per_stream, C.c_size_t(bytes_per_slot)))
        else:
            self._chk(self.L.ft8b200_cluster_submit(C.c_void_p(self.h), ptrs, C.c_size_t(bytes_per_stream), C.c_size_t(stride), cnt))

    def submit_host(self, iq_host, n_slots: int, bytes_per_stream: int = RAW_SLOT_BYTES):
        self._chk(self.L.ft8b200_cluster_submit_host(C.c_void_p(self.h), _p(iq_host), C.c_size_t(bytes_per_stream), n_slots))

    def collect(self, capacity_slots: int):
        res = np.zeros((capacity_slots, self.M), result_dtype)
        nres = np.zeros(capacity_slots, np.int32)
        n = self._chk(self.L.ft8b200_cluster_collect(C.c_void_p(self.h), _p(res), _p(nres), capacity_slots))
        return res[:n], nres[:n]

    def gathers(self) -> int:
        return int(self.L.ft8b200_cluster_gathers(C.c_void_p(self.h)))

    def nccl_version(self) -> int:
        return int(self.L.ft8b200_cluster_nccl_version(C.c_void_p(self.h)))

    def launches(self) -> int:
        return int(self.L.ft8b200_cluster_kernel_launches(C.c_void_p(self.h)))


class Stream:
    """One receiver stream (ft8b200_stream_t): what rtlsdr_callback() feeds.  Mirrors the daemon's rx_state."""

    def __init__(self, ctx: Context):
        self.L = ctx.L
        self.ctx = ctx
        self.h = self.L.ft8b200_stream_create(C.c_void_p(ctx.h))
        if not self.h:
            raise Ft8Error(self.L.ft8b200_last_error().decode())

    def close(self):
        if self.h:
            self.L.ft8b200_stream_destroy(C.c_void_p(self.h))
            self.h = None

    def callback(self, buf: np.ndarray):
        """rtlsdr_callback(samples, samples_count, ctx) with ctx = this stream."""
        buf = np.ascontiguousarray(buf, np.uint8)
        self.L.rtlsdr_callback(_p(buf), C.c_uint32(buf.size), C.c_void_p(self.h))

    def flip(self):
        rc = self.L.ft8b200_stream_flip(C.c_void_p(self.h))
        if rc:
            raise Ft8Error(f"ft8b200_stream_flip -> {rc}")

    def count(self) -> int:
        return int(self.L.ft8b200_stream_count(C.c_void_p(self.h)))

    def fetch(self):
        i_s = np.zeros(N_SLOT, np.float32)
        q_s = np.zeros(N_SLOT, np.float32)
        n = C.c_uint32(0)
        rc = self.L.ft8b200_stream_fetch(C.c_void_p(self.h), _p(i_s), _p(q_s), C.byref(n))
        if rc:
            raise Ft8Error(f"ft8b200_stream_fetch -> {rc}")
        return i_s, q_s, int(n.value)

    def decode(self):
        res = np.zeros(self.ctx.M, result_dtype)
        n = C.c_int32(0)
        rc = self.L.ft8b200_stream_decode(C.c_void_p(self.h), _p(res), C.byref(n))
        if rc:
            raise Ft8Error(f"ft8b200_stream_decode -> {rc}: {self.L.ft8b200_last_error().decode()}")
        return res, int(n.value)


class Monitor:
    """monitor_init/process/reset/free with the reference's monitor_t / monitor_config_t (ft8_lib/decode_ft8.c:82-224)."""

    def __init__(self, sample_rate=12000, time_osr=2, freq_osr=2, protocol=1, f_min=100.0, f_max=3000.0):
        self.L = lib()
        self.cfg = MonitorConfig(f_min, f_max, sample_rate, time_osr, freq_osr, protocol)
        self.me = MonitorT()
        self.L.monitor_init(C.byref(self.me), C.byref(self.cfg))
        self.open = True

    def process(self, frame: np.ndarray):
        frame = np.ascontiguousarray(frame, np.float32)
        assert frame.size == self.me.block_size
        self.L.monitor_process(C.byref(self.me), _p(frame))

    def reset(self):
        self.L.monitor_reset(C.byref(self.me))

    def set_deferred(self, on: bool):
        """ft8b200_monitor_set_deferred: process() only appends; the pending blocks are transformed at find_sync/decode/flush."""
        if self.L.ft8b200_monitor_set_deferred(C.byref(self.me), int(on)) != 0:
            raise Ft8Error("ft8b200_monitor_set_deferred")

    def flush(self) -> int:
        return self.L.ft8b200_monitor_flush(C.byref(self.me))

    def mag(self) -> np.ndarray:
        n = self.me.wf.num_blocks * self.me.wf.block_stride
        return np.ctypeslib.as_array(C.cast(self.me.wf.mag, C.POINTER(C.c_uint8)), shape=(n,)).copy()

    def find_sync(self, num_candidates=120, min_score=10):
        heap = np.zeros(num_candidates, cand_dtype)
        n = self.L.ft8_find_sync(C.byref(self.me.wf), num_candidates, _p(heap), min_score)
        return heap[:n]

    def decode(self, cand, max_iterations=20):
        c = np.array([cand], cand_dtype)
        msg = np.zeros(1, msg_dtype)
        st = np.frombuffer(bytes([0xA5]) * 12, status_dtype).copy()
        ok = self.L.ft8_decode(C.byref(self.me.wf), _p(c), _p(msg), max_iterations, _p(st))
        return bool(ok), msg[0], st[0]

    def close(self):
        if self.open:
            self.L.monitor_free(C.byref(self.me))
            self.open = False


# ---- the reference-named drop-in entry points (host pointers) ---------------------------------------
def rtlsdr_callback(samples: np.ndarray):
    """rtlsdr_callback(samples, samples_count, NULL): the process-wide default stream, as in the reference."""
    buf = np.ascontiguousarray(samples, np.uint8)
    lib().rtlsdr_callback(_p(buf), C.c_uint32(buf.size), C.c_void_p(0))


def ft8_subsystem(i_samples: np.ndarray, q_samples: np.ndarray, decodes: np.ndarray | None = None):
    """ft8_subsystem(float*, float*, uint32_t, struct decoder_results*, int32_t*) on host arrays."""
    L = lib()
    i_s = np.ascontiguousarray(i_samples, np.float32)
    q_s = np.ascontiguousarray(q_samples, np.float32)
    if decodes is None:
        decodes = np.zeros(50, result_dtype)
    n = C.c_int32(0)
    L.ft8_subsystem(_p(i_s), _p(q_s), C.c_uint32(N_SLOT), _p(decodes), C.byref(n))
    return decodes, n.value


def ft8_find_sync(mag: np.ndarray, num_candidates=120, min_score=10, num_blocks=92, num_bins=256, time_osr=2, freq_osr=2, protocol=1):
    L = lib()
    mag = np.ascontiguousarray(mag, np.uint8)
    wf = WaterfallT(num_blocks, num_blocks, num_bins, time_osr, freq_osr, mag.ctypes.data, time_osr * freq_osr * num_bins, protocol)
    heap = np.zeros(num_candidates, cand_dtype)
    n = L.ft8_find_sync(C.byref(wf), num_candidates, _p(heap), min_score)
    return heap[:n]


def ft8_decode(mag: np.ndarray, cand, max_iterations=20, num_blocks=92, num_bins=256, time_osr=2, freq_osr=2, protocol=1):
    L = lib()
    mag = np.ascontiguousarray(mag, np.uint8)
    wf = WaterfallT(num_blocks, num_blocks, num_bins, time_osr, freq_osr, mag.ctypes.data, time_osr * freq_osr * num_bins, protocol)
    c = np.array([cand], cand_dtype)
    msg = np.zeros(1, msg_dtype)
    st = np.frombuffer(bytes([0xA5]) * 12, status_dtype).copy()
    ok = L.ft8_decode(C.byref(wf), _p(c), _p(msg), max_iterations, _p(st))
    return bool(ok), msg[0], st[0]


# ---- on-disk formats and whole recordings (csrc/files.cu) -------------------------------------------------
decoded_dtype = np.dtype([("text", "S25"), ("_pad", "u1"), ("hash", "<u2"), ("score", "<i2"), ("_pad2", "<u2"), ("time_sec", "<f4"), ("freq_hz", "<f4")])
assert decoded_dtype.itemsize == 40


def read_iq_file(path: str):
    """-> (I[48000], Q[48000], n_pairs, peak): unscaled samples of a .iq recording (readRawIQfile without its normalisation)."""
    i_s = np.zeros(N_SLOT, np.float32); q_s = np.zeros(N_SLOT, np.float32)
    peak = C.c_float(0)
    n = lib().ft8b200_read_iq_file(path.encode(), _p(i_s), _p(q_s), C.byref(peak))
    return i_s, q_s, int(n), float(peak.value)


def read_c2_file(path: str):
    i_s = np.zeros(N_SLOT, np.float32); q_s = np.zeros(N_SLOT, np.float32)
    peak, freq, ty = C.c_float(0), C.c_double(0), C.c_int(0)
    name = C.create_string_buffer(15)
    n = lib().ft8b200_read_c2_file(path.encode(), _p(i_s), _p(q_s), C.byref(peak), C.byref(freq), C.byref(ty), name)
    return i_s, q_s, int(n), float(peak.value), float(freq.value), int(ty.value), name.raw[:14]


def load_wav(path: str, max_samples: int = 15 * 12000):
    """load_wav() of ft8_lib/common/wave.c: -> (float32 signal, sample_rate); raises IOError(code) like a negative return."""
    sig = np.zeros(max_samples, np.float32)
    n, sr = C.c_int(max_samples), C.c_int(0)
    rc = lib().ft8b200_load_wav(_p(sig), C.byref(n), C.byref(sr), path.encode())
    if rc < 0:
        raise IOError(rc)
    return sig[:n.value].copy(), int(sr.value)


def _paths(paths):
    arr = (C.c_char_p * len(paths))(*[p.encode() for p in paths])
    return arr


def decode_iq_files(ctx: Context, paths):
    n = len(paths)
    res = np.zeros((n, ctx.M), result_dtype)
    nres = np.zeros(n, np.int32)
    ns = np.zeros(n, np.int32)
    ctx._chk(ctx.L.ft8b200_decode_iq_files(C.c_void_p(ctx.h), _paths(paths), n, _p(res), _p(nres), _p(ns)))
    return res, nres, ns


def decode_audio(ctx: Context, audio, sample_rate=12000, protocol=1):
    """audio: float32 device tensor [n, n_samples] -> list of decoded_dtype arrays (decode_ft8's output per recording)."""
    n, n_samples = audio.shape
    out = np.zeros((n, ctx.M), decoded_dtype)
    cnt = np.zeros(n, np.int32)
    ctx._chk(ctx.L.ft8b200_decode_audio(C.c_void_p(ctx.h), _p(audio), C.c_size_t(audio.stride(0)), n_samples, n, sample_rate, protocol, _p(out), _p(cnt), ctx.M))
    return [out[k, :cnt[k]] for k in range(n)]


def decode_wav_files(ctx: Context, paths, protocol=1):
    n = len(paths)
    out = np.zeros((n, ctx.M), decoded_dtype)
    cnt = np.zeros(n, np.int32)
    status = np.zeros(n, np.int32)
    ctx._chk(ctx.L.ft8b200_decode_wav_files(C.c_void_p(ctx.h), _paths(paths), n, protocol, _p(out), _p(cnt), ctx.M, _p(status)))
    return [out[k, :cnt[k]] for k in range(n)], status


def format_decoded(rec) -> str:
    """One line of decode_ft8's stdout (decode_ft8.c:401)."""
    return "000000 %3d %+4.2f %4.0f ~  %s" % (int(rec["score"]), float(rec["time_sec"]), float(rec["freq_hz"]), rec["text"].decode())


# ---- reporting records (csrc/report.cu): host code, no GPU involved ---------------------------------------
options_dtype = np.dtype([("freq", "<u4"), ("rcall", "S13"), ("rloc", "S7")])
cluster_form_dtype = np.dtype([("mycall", "S16"), ("dxcall", "S12"), ("freq", "S10"), ("info", "S100")])
PSK_MAX_DATAGRAM = 1600


def station(rcall: str, rloc: str, dial_freq: int) -> np.ndarray:
    """struct decoder_options (rtlsdr_ft8d.h:130-134) as a 1-element array."""
    o = np.zeros(1, options_dtype)
    o[0] = (dial_freq, rcall.encode(), rloc.encode())
    return o


def pskreporter_datagram(spots: np.ndarray, opt: np.ndarray, unixtime: int, sequence: int = 1, random_id: int = 0, app_version: str | None = None,
                         cap: int = PSK_MAX_DATAGRAM):
    """-> (datagram bytes, number of spots it carries); raises Ft8Error when `cap` is too small."""
    spots = np.ascontiguousarray(spots, result_dtype)
    out = np.zeros(cap, np.uint8)
    used = C.c_uint32(0)
    n = lib().ft8b200_pskreporter_datagram(_p(spots), C.c_uint32(spots.size), _p(opt), None if app_version is None else app_version.encode(),
                                           C.c_uint32(unixtime), C.c_uint32(sequence), C.c_uint32(random_id), _p(out), C.c_size_t(cap), C.byref(used))
    if n < 0:
        raise Ft8Error("ft8b200_pskreporter_datagram failed (bad argument or buffer too small)")
    return out[:n].tobytes(), used.value


def pskreporter_batch(res: np.ndarray, nres: np.ndarray, opt: np.ndarray, unixtime, first_sequence: int = 1, random_id: int = 0,
                      app_version: str | None = None):
    """Records of a batch (fetch_results / Pipe.collect layout) -> list of datagrams (b"" for slots without spots)."""
    res = np.ascontiguousarray(res, result_dtype)
    n_slots, M = res.shape
    nres = np.ascontiguousarray(nres, np.int32)
    ut = np.ascontiguousarray(np.broadcast_to(np.asarray(unixtime, np.uint32), (n_slots,)))
    out = np.zeros((n_slots, PSK_MAX_DATAGRAM), np.uint8)
    lens = np.zeros(n_slots, np.int32)
    k = lib().ft8b200_pskreporter_batch(_p(res), _p(nres), n_slots, M, _p(opt), None if app_version is None else app_version.encode(), _p(ut),
                                        C.c_uint32(first_sequence), C.c_uint32(random_id), _p(out), C.c_size_t(PSK_MAX_DATAGRAM), _p(lens))
    if k < 0:
        raise Ft8Error("ft8b200_pskreporter_batch failed")
    return [out[s, :lens[s]].tobytes() for s in range(n_slots)], k


def webcluster_form(spot: np.ndarray, opt: np.ndarray) -> dict:
    spot = np.ascontiguousarray(spot, result_dtype).reshape(1)
    f = np.zeros(1, cluster_form_dtype)
    if lib().ft8b200_webcluster_form(_p(spot), _p(opt), _p(f)) != 0:
        raise Ft8Error("ft8b200_webcluster_form failed")
    return {"_mycall": f[0]["mycall"], "_dxcall": f[0]["dxcall"], "_freq": f[0]["freq"], "_info": f[0]["info"]}


def format_spots(spots: np.ndarray, dial_freq: int, unixtime: int) -> str:
    spots = np.ascontiguousarray(spots, result_dtype)
    need = lib().ft8b200_format_spots(_p(spots), C.c_uint32(spots.size), C.c_uint32(dial_freq), C.c_uint32(unixtime), None, C.c_size_t(0))
    buf = C.create_string_buffer(need + 1)
    lib().ft8b200_format_spots(_p(spots), C.c_uint32(spots.size), C.c_uint32(dial_freq), C.c_uint32(unixtime), buf, C.c_size_t(need + 1))
    return buf.value.decode()


def lib_app_version() -> str:
    L = lib()
    L.ft8b200_report_app_version.restype = C.c_char_p
    return L.ft8b200_report_app_version().decode()
