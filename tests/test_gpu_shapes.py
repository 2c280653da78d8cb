"""The device entry points at the batch sizes and memory layouts that select their code paths, against the CPU oracle.

The parity suite feeds every kernel densely packed tensors with 256-byte-aligned bases and batches of 1-64 slots.  The launch
functions choose different code by batch size x SM count (decode: one CTA row per slot, or a persistent grid whose warps pull
entries; sync: how many time offsets a CTA scores) and by pointer and stride alignment (sync: the FT8 fast kernel, or staged
kernels that load 16 bytes or one byte at a time, or no staging at all; monitor: float2 or scalar loads, uint4 or byte stores).
Here each of those paths is compared with the oracle byte for byte, and torch.profiler (CUDA activity) shows which kernel and
which grid actually ran, so that a mis-computed threshold fails instead of passing vacuously.  Batches of more than 65 535
slots (the gridDim.y limit) and misaligned float slots are checked too."""
import ctypes as C
import json
import re

import numpy as np
import pytest

from oracle.pyoracle import cand_dtype, msg_dtype, result_dtype, status_dtype
from test_osd import OsdOracle, fuzz_llrs
from tools import ft8enc, synth

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

DEV = torch.device("cuda:0")
EINVAL = -2
MAX_ROWS = 65535
DAEMON = dict(num_blocks=92, num_bins=256, time_osr=2, freq_osr=2)
GEOMETRIES = {  # dims, protocol
    "ft8_daemon": (DAEMON, 1),
    "ft8_12k": (dict(num_blocks=93, num_bins=960, time_osr=2, freq_osr=2), 1),
    "ft4": (dict(num_blocks=156, num_bins=288, time_osr=2, freq_osr=2), 0),
}
SENT = dict(ok=0xEE, stage=0xEE, status=0xA5, msg=0x5A, plain=0x77)
SENT_LLR = np.int32(0x7FC0DEAD)   # a NaN no kernel produces


# ------------------------------------------------------------------------------------------- helpers
def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def cells(dims):
    return dims["num_blocks"] * dims["time_osr"] * dims["freq_osr"] * dims["num_bins"]


def _p(t):
    return C.c_void_p(0) if t is None else C.c_void_p(t.data_ptr())


def _stream():
    s = torch.cuda.current_stream().cuda_stream
    return C.c_void_p(s if s else 1)   # NULL would be the context's own stream; 1 = cudaStreamLegacy


def last_error(pkg):
    return pkg.lib().ft8b200_last_error().decode()


def as_np(t, dt):
    a = t.cpu().numpy()
    return a.view(dt).reshape(a.shape[:-1])


def profiled(fn, tmp_path, tag):
    """Run fn() under torch.profiler (CUDA activity) -> (fn's result, [(kernel name, grid)] in launch order)."""
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    path = tmp_path / f"{tag}.json"
    prof.export_chrome_trace(str(path))
    events = json.loads(path.read_text())["traceEvents"]
    ks = [(e["name"], tuple(e.get("args", {}).get("grid", ()))) for e in events if e.get("cat") == "kernel"]
    path.unlink()
    return out, ks


SYNC_KINDS = {   # demangled names of the four sync score kernels
    "fast": re.compile(r"sync_score_ft8_kernel\("),
    "staged256": re.compile(r"sync_score_kernel<256, ?true, ?false>"),
    "staged": re.compile(r"sync_score_kernel<0, ?true, ?(true|false)>"),
    "unstaged": re.compile(r"sync_score_kernel<0, ?false, ?(true|false)>"),
}


def sync_kind(ks):
    found = [(k, g) for name, g in ks for k, rx in SYNC_KINDS.items() if rx.search(name)]
    assert len(found) >= 1, f"no sync score kernel among {[n for n, _ in ks]}"
    return found


def std_sig(f0=700.0, t0=0.5, snr=-10.0, msg=("CQ", "K1JT", "FN20")):
    return (ft8enc.tones(ft8enc.pack_std(*msg)), f0, t0, snr)


def conditioned(oracle, sigs, seed):
    i_s, q_s = synth.slot_f32(sigs, seed)
    return oracle.condition(i_s, q_s, 48000)[:2]


def distinct_mags(oracle, dims, rng, real=None):
    """Three waterfalls that give many candidates and different ones: random bytes, a narrow band of values, a ramp;
    `real` (a daemon waterfall with signals) replaces the narrow band."""
    n = cells(dims)
    ramp = np.clip(np.arange(n) // max(n // 230, 1) + rng.integers(0, 24, n), 0, 255).astype(np.uint8)
    second = real if real is not None else rng.integers(100, 104, n, dtype=np.uint8)
    return np.stack([rng.integers(0, 256, n, dtype=np.uint8), second, ramp])


def strided(dense, base_offset, stride):
    """A view of `dense` (rows x cols) whose first byte sits `base_offset` bytes past a 256-byte-aligned allocation and
    whose rows are `stride` elements apart."""
    rows, cols = dense.shape
    item = dense.element_size()
    assert base_offset % item == 0
    buf = torch.zeros(base_offset // item + rows * stride + 16, dtype=dense.dtype, device=DEV)
    v = buf[base_offset // item: base_offset // item + rows * stride].view(rows, stride)[:, :cols]
    v.copy_(dense)
    return v


def expected_entry(oracle, mag, cand, dims, protocol):
    """Every byte ft8b200_decode writes for one candidate: ok, stage, status (fields the reference leaves unwritten are 0),
    message (all 28 bytes, zero unless decoded), hard decisions and normalised LLRs."""
    d = oracle.decode(mag, cand, protocol=protocol, **dims)
    s = d["status"]
    stage = 1 if s["ldpc_errors"] > 0 else 2 if s["crc_extracted"] != s["crc_calculated"] else 4 if d["ok"] else 3
    st = np.zeros(1, status_dtype)
    st[0] = (s["ldpc_errors"], s["crc_extracted"] if stage >= 2 else 0, s["crc_calculated"] if stage >= 2 else 0,
             s["unpack_status"] if stage >= 3 else 0)
    m = np.zeros(1, msg_dtype)
    if d["ok"]:
        m[0]["text"], m[0]["hash"] = d["msg"]["text"], d["msg"]["hash"]
    assert not np.isnan(d["llr"]).any()
    return d["ok"], stage, st.view(np.uint8), m.view(np.uint8), d["plain"], d["llr"].view(np.int32)


class Ref:
    """Oracle outputs for the first K candidates of a few distinct waterfalls, as (W, K, ...) arrays."""

    def __init__(self, oracle, mags, cands, dims, protocol):
        W, K = cands.shape
        self.ok = np.zeros((W, K), np.uint8); self.stage = np.zeros((W, K), np.uint8)
        self.status = np.zeros((W, K, 12), np.uint8); self.msg = np.zeros((W, K, 28), np.uint8)
        self.plain = np.zeros((W, K, 174), np.uint8); self.llr = np.zeros((W, K, 174), np.int32)
        self.cands = cands
        for w in range(W):
            for k in range(K):
                (self.ok[w, k], self.stage[w, k], self.status[w, k], self.msg[w, k], self.plain[w, k],
                 self.llr[w, k]) = expected_entry(oracle, mags[w], cands[w, k], dims, protocol)


def first_diff(a, b):
    idx = np.argwhere(a != b)
    return tuple(idx[0]) if idx.size else None


@pytest.fixture(params=[0, 1], ids=["bp_nodes", "bp_edges"])
def bp_variant(request, pkg):
    """Both belief-propagation kernels (ft8b200_set_decode_variant): node-centred (default) and edge-centred."""
    pkg.set_decode_variant(request.param)
    yield request.param
    pkg.set_decode_variant(0)


@pytest.fixture(scope="module")
def daemon(oracle):
    """Three distinct daemon waterfalls (one message, a crowded band, random bytes), their 500 best-scoring positions as
    candidates (min_score below every score) and the oracle's decode of each of them."""
    real = oracle.waterfall(*conditioned(oracle, [std_sig()], 7))
    i_s, q_s, _ = synth.crowded_band(ft8enc, 25, 5, snr_lo=-18, snr_hi=0)
    crowded = oracle.waterfall(*oracle.condition(i_s, q_s, 48000)[:2])
    mags = np.stack([real, crowded, np.random.default_rng(1).integers(0, 256, 94208, dtype=np.uint8)])
    cands = np.stack([oracle.find_sync(m, max_cand=500, min_score=-1000) for m in mags])
    ref = Ref(oracle, mags, cands, DAEMON, 1)
    assert ref.ok[0].any() and ref.ok[1].sum() >= 5 and not ref.ok[2].any()
    return mags, ref


# ------------------------------------------------------------------------------------------- 1. decode modes
def decode_raw(c, mag, cand, ncand, n, dims, want_extra=True):
    """ft8b200_decode through the C entry with sentinel-filled outputs."""
    K = c.K
    out = dict(ok=torch.full((n, K), SENT["ok"], dtype=torch.uint8, device=DEV),
               stage=torch.full((n, K), SENT["stage"], dtype=torch.uint8, device=DEV),
               status=torch.full((n, K, 12), SENT["status"], dtype=torch.uint8, device=DEV),
               msg=torch.full((n, K, 28), SENT["msg"], dtype=torch.uint8, device=DEV))
    if want_extra:
        out["plain"] = torch.full((n, K, 174), SENT["plain"], dtype=torch.uint8, device=DEV)
        out["llr"] = torch.full((n, K, 174), int(SENT_LLR), dtype=torch.int32, device=DEV)
    rc = c.L.ft8b200_decode(C.c_void_p(c.h), _p(mag), C.c_size_t(mag.stride(0)), n, dims["num_blocks"], dims["num_bins"], dims["time_osr"],
                            dims["freq_osr"], _p(cand), _p(ncand), _p(out["ok"]), _p(out["stage"]), _p(out["status"]), _p(out["msg"]),
                            _p(out.get("plain")), _p(out.get("llr")), _stream())
    assert rc == 0, c.L.ft8b200_last_error().decode()
    return out


def check_against_ref(out, ref, w_of, ncand):
    """Every byte of every entry: the oracle's for c < ncand[s], ok = stage = 0 and the sentinels untouched past it."""
    n, K = out["ok"].shape
    live = np.arange(K)[None, :] < ncand[:, None]
    exp = dict(ok=np.where(live, ref.ok[w_of, :K], 0), stage=np.where(live, ref.stage[w_of, :K], 0),
               status=np.where(live[..., None], ref.status[w_of, :K], SENT["status"]),
               msg=np.where(live[..., None], ref.msg[w_of, :K], SENT["msg"]))
    if "plain" in out:
        exp["plain"] = np.where(live[..., None], ref.plain[w_of, :K], SENT["plain"])
        exp["llr"] = np.where(live[..., None], ref.llr[w_of, :K], SENT_LLR)
    for key, e in exp.items():
        g = out[key].cpu().numpy()
        assert np.array_equal(g, e), f"{key}: first difference at (slot, cand, ...) = {first_diff(g, e)}"


@pytest.mark.parametrize("where", ["T-1", "T", "T+1", "2T+7", "8T"])
@pytest.mark.parametrize("K", [1, 7, 120, 500])
def test_decode_grid_and_pull_modes_pin_every_byte(pkg, daemon, bp_variant, K, where, tmp_path):
    """ft8b200_decode with n x K around T = 32 x SMs, where the node-centred kernel switches from a (candidate group, slot)
    grid to a persistent grid whose warps pull all n x K entries; ncand runs from 0 to K.  Every output byte of every entry,
    past ncand included, against the oracle; the profiler shows which kernel and which grid ran."""
    mags, ref = daemon
    T = 32 * sm_count()
    target = {"T-1": T - 1, "T": T, "T+1": T + 1, "2T+7": 2 * T + 7, "8T": 8 * T}[where]
    n = target // K if where in ("T-1", "T") else -(-target // K)
    assert n >= 1
    W = mags.shape[0]
    w_of = np.arange(n) % W
    ncand = ((np.arange(n) * 37 + 3) % (K + 1)).astype(np.int32)
    ncand[0] = K
    if n > 1:
        ncand[-1] = 0
    c = pkg.Context(0, max_candidates=K)
    try:
        d_mag = torch.from_numpy(mags).to(DEV)[torch.from_numpy(w_of).to(DEV)]
        d_cand = torch.from_numpy(np.ascontiguousarray(ref.cands[w_of, :K]).view(np.uint8).reshape(n, K, 8)).to(DEV)
        d_ncand = torch.from_numpy(ncand).to(DEV)
        out, ks = profiled(lambda: decode_raw(c, d_mag, d_cand, d_ncand, n, DAEMON), tmp_path, f"decode_{K}_{where}")
        dk = [(name, g) for name, g in ks if re.search(r"decode_(edges_)?kernel\(", name)]
        assert len(dk) == 1, dk
        name, grid = dk[0]
        pull = bp_variant == 0 and n * K > T
        if bp_variant == 1:
            assert "decode_edges_kernel(" in name and grid[:2] == (-(-K // 8), n), (name, grid)
        elif pull:
            assert "decode_edges" not in name and grid[1] == 1 and 1 <= grid[0] <= 4 * sm_count(), (name, grid)
        else:
            assert "decode_edges" not in name and grid[:2] == (-(-K // 8), n), (name, grid)
        check_against_ref(out, ref, w_of, ncand)
    finally:
        c.close()


@pytest.mark.parametrize("size", ["small", "above_T"])
def test_work_list_mode_matches_stage_wise_decode(pkg, oracle, bp_variant, size):
    """process_slots decodes from the flat work list the sync selection writes.  Its candidates, ok, status and message bytes
    equal find_sync + ft8b200_decode on the same waterfalls, and its spot records equal the oracle's ft8_subsystem()."""
    n = 3 if size == "small" else 2 * 32 * sm_count() // 120 + 7
    slots = [conditioned(oracle, [std_sig()], 7), conditioned(oracle, [std_sig(1200.0, 1.0, -5.0, ("K1ABC", "W9XYZ", "RR73"))], 9),
             conditioned(oracle, [], 11)]
    W = len(slots)
    w_of = np.arange(n) % W
    hi = np.stack([s[0] for s in slots])[w_of]
    hq = np.stack([s[1] for s in slots])[w_of]
    c = pkg.Context(0)
    try:
        d_i, d_q = torch.from_numpy(hi).to(DEV), torch.from_numpy(hq).to(DEV)
        c.process_slots(d_i, d_q)
        c.sync()
        w = c.workspace_ptrs()
        K = c.K

        class _Arr:
            def __init__(self, ptr, shape, typestr):
                self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2}
        g = lambda key, shape, t: torch.as_tensor(_Arr(w[key], shape, t), device=DEV).clone()
        ws = dict(cand=g("cand", (n, K, 8), "|u1"), ncand=g("ncand", (n,), "<i4"), ok=g("ok", (n, K), "|u1"), status=g("status", (n, K, 12), "|u1"),
                  msg=g("msg", (n, K, 28), "|u1"), mag=g("mag", (n, 94208), "|u1"))
        res, nres = c.fetch_results(n)
        mag = c.waterfall(d_i, d_q)
        cand, ncand = c.find_sync(mag)
        out = decode_raw(c, mag, cand, ncand, n, DAEMON, want_extra=False)
        torch.cuda.synchronize()
        assert torch.equal(ws["mag"], mag) and torch.equal(ws["ncand"], ncand)
        nc = ncand.cpu().numpy()
        live = torch.from_numpy(np.arange(K)[None, :] < nc[:, None]).to(DEV)
        assert torch.equal(ws["cand"][live], cand[live])
        assert torch.equal(ws["ok"], out["ok"])
        assert torch.equal(ws["status"][live], out["status"][live]) and torch.equal(ws["msg"][live], out["msg"][live])
        for s in range(W):
            o = oracle.subsystem(*slots[s])
            for t in range(s, n, W):
                assert nres[t] == o["n"] and res[t].tobytes() == o["results"].tobytes(), t
        assert nres[0] >= 1 and nres[1] >= 1
    finally:
        c.close()


# ------------------------------------------------------------------------------------------- 2. sync at every split
def splits_to_per_cta(n, sms, planes):
    s = min(6, max(1, -(-4 * sms // (n * planes))))
    return -(-36 // s)


@pytest.mark.parametrize("to_per_cta", [6, 8, 9, 12, 18, 36])
@pytest.mark.parametrize("geometry", list(GEOMETRIES))
def test_sync_scores_every_split(pkg, oracle, geometry, to_per_cta, tmp_path):
    """The staged score kernels give a CTA 36 / splits time offsets, splits chosen from the batch size and the SM count.  Batch
    sizes are picked so that each of 6, 8, 9, 12, 18 and 36 offsets per CTA occurs; FT8 waterfalls are passed at a 1-byte offset
    so that the staged kernels (not the FT8 fast kernel) run.  Candidates equal the oracle's in content and order."""
    dims, proto = GEOMETRIES[geometry]
    planes = dims["time_osr"] * dims["freq_osr"]
    sms = sm_count()
    n = next(k for k in range(1, 8 * sms) if splits_to_per_cta(k, sms, planes) == to_per_cta)
    mags = distinct_mags(oracle, dims, np.random.default_rng(20 + n))
    W = mags.shape[0]
    w_of = np.arange(n) % W
    dense = torch.from_numpy(mags).to(DEV)[torch.from_numpy(w_of).to(DEV)]
    mag = strided(dense, 1 if proto == 1 else 0, dense.shape[1])
    c = pkg.Context(0)
    try:
        c.set_protocol(proto)
        (cand, ncand), ks = profiled(lambda: c.find_sync(mag, **dims), tmp_path, f"sync_{geometry}_{n}")
        found = sync_kind(ks)
        splits = -(-36 // to_per_cta)
        assert [k for k, _ in found] == ["staged256" if dims["num_bins"] == 256 and proto == 1 else "staged"], found
        assert found[0][1][:2] == (planes * splits, n), (found, splits)
        g = as_np(cand, cand_dtype)
        nc = ncand.cpu().numpy()
        for w in range(W):
            o = oracle.find_sync(mags[w], max_cand=c.K, min_score=10, protocol=proto, **dims)
            for s in range(w, n, W):
                assert nc[s] == o.size and g[s, : o.size].tobytes() == o.tobytes(), (geometry, n, s)
    finally:
        c.close()


# ------------------------------------------------------------------------------------------- 3. layouts
LAYOUT_GEOMETRIES = dict(GEOMETRIES, ft8_wide=(dict(num_blocks=93, num_bins=2400, time_osr=2, freq_osr=2), 1),
                         ft4_wide=(dict(num_blocks=156, num_bins=1400, time_osr=2, freq_osr=2), 0))


@pytest.mark.parametrize("geometry", list(LAYOUT_GEOMETRIES))
def test_waterfall_layouts_find_sync_decode_spots(pkg, oracle, daemon, geometry, tmp_path):
    """find_sync, decode and spots on waterfall views at base offsets of 1, 2, 3, 4, 8 and 16 bytes and slot strides of the slot's
    size + 1, 2, 4, 8 and 16 bytes give the bytes of the dense call, which equals the oracle candidate by candidate.  Over the
    geometries every sync score kernel runs: the FT8 fast kernel (4-byte aligned FT8), the 256-bin staged kernel (misaligned
    daemon waterfalls), the generic staged kernel with 16-byte and with byte loads (FT4, misaligned 12 kHz FT8) and the unstaged
    kernel (waterfalls too large to stage)."""
    dims, proto = LAYOUT_GEOMETRIES[geometry]
    rng = np.random.default_rng(sum(map(ord, geometry)))
    mags = daemon[0] if geometry == "ft8_daemon" else distinct_mags(oracle, dims, rng)
    W = mags.shape[0]
    n = 5
    w_of = np.arange(n) % W
    dense = torch.from_numpy(mags).to(DEV)[torch.from_numpy(w_of).to(DEV)].contiguous()
    c = pkg.Context(0)
    c.set_protocol(proto)
    seen = set()

    def run(mag, tag):
        def go():
            cand, ncand = c.find_sync(mag, **dims)
            dec = c.decode(mag, cand, ncand, want_plain=True, want_llr=True, **dims)
            sp = c.spots(cand, ncand, dec[0], dec[3], freq_osr=dims["freq_osr"])
            return [cand, ncand, *dec[:5], dec[5].view(torch.int32), *sp]
        out, ks = profiled(go, tmp_path, tag)
        kinds = sync_kind(ks)
        seen.update(k for k, _ in kinds)
        return out, kinds[0][0]

    try:
        base, kind = run(dense, "dense")
        assert kind == ("fast" if proto == 1 else "unstaged" if "wide" in geometry else "staged"), kind
        # the dense call against the oracle, candidate by candidate
        cand, ncand, ok, stage, status, msg, plain, llr = base[:8]
        g_c, nc = as_np(cand, cand_dtype), ncand.cpu().numpy()
        for w in range(W):
            o = oracle.find_sync(mags[w], max_cand=c.K, min_score=10, protocol=proto, **dims)
            assert nc[w] == o.size and g_c[w, : o.size].tobytes() == o.tobytes(), w
            for k in range(o.size):
                e_ok, e_stage, e_st, e_msg, e_plain, e_llr = expected_entry(oracle, mags[w], o[k], dims, proto)
                assert (int(ok[w, k]), int(stage[w, k])) == (e_ok, e_stage), (w, k)
                assert np.array_equal(status[w, k].cpu().numpy(), e_st) and np.array_equal(msg[w, k].cpu().numpy(), e_msg), (w, k)
                assert np.array_equal(plain[w, k].cpu().numpy(), e_plain), (w, k)
                assert np.array_equal(llr[w, k].cpu().numpy(), e_llr), (w, k)
        for s in range(W, n):
            for t in base:
                assert torch.equal(t[s], t[s % W])
        for off in (1, 2, 3, 4, 8, 16):
            for extra in (1, 2, 4, 8, 16):
                out, _ = run(strided(dense, off, dense.shape[1] + extra), f"o{off}_{extra}")
                for k, (a, b) in enumerate(zip(out, base)):
                    assert torch.equal(a, b), (geometry, off, extra, k)
        want = {"ft8_daemon": {"fast", "staged256"}, "ft8_12k": {"fast", "staged"}, "ft4": {"staged"}, "ft8_wide": {"fast", "unstaged"},
                "ft4_wide": {"unstaged"}}[geometry]
        assert seen == want, seen
    finally:
        c.close()


MONITOR_CASES = {  # sample rate, protocol, odd n_samples
    "ft8_12k": (12000, 1, 180_001),
    "ft4_12k": (12000, 0, 90_001),
    "ft8_11025": (11025, 1, 165_375),
}


@pytest.mark.parametrize("case", list(MONITOR_CASES))
def test_monitor_audio_and_output_layouts(pkg, oracle, case):
    """ft8b200_monitor_waterfall with audio views at odd float offsets and odd slot strides (scalar loads where float2 loads
    would be misaligned) and with an output at a 3-byte offset whose slot stride is no multiple of 16 (byte stores): the same
    bytes as the dense call, which equals the oracle's monitor slot by slot."""
    rate, proto, ns = MONITOR_CASES[case]
    rng = np.random.default_rng(rate + proto)
    W, n = 3, 5
    rows = (rng.standard_normal((W, ns)) * np.array([[0.1], [0.003], [1.0]])).astype(np.float32)
    dense = torch.from_numpy(rows[np.arange(n) % W]).to(DEV)
    c = pkg.Context(0)
    try:
        base, nb = c.monitor_waterfall(dense, sample_rate=rate, protocol=proto)
        torch.cuda.synchronize()
        b = base.cpu().numpy()
        for w in range(W):
            ref, info, _ = oracle.monitor_waterfall(rows[w], sample_rate=rate, protocol=proto)
            assert nb == int(info[4]) and nb > 0
            for s in range(w, n, W):
                assert np.array_equal(b[s], ref), (case, s, int((b[s] != ref).sum()))
        for off, extra in ((1, 0), (1, 1), (3, 2), (0, 1), (5, 7)):
            view = strided(dense, 4 * off, ns + extra)
            got, nb2 = c.monitor_waterfall(view, sample_rate=rate, protocol=proto)
            assert nb2 == nb and torch.equal(got, base), (case, off, extra)
        # misaligned output, slot stride not a multiple of 16
        per = base.shape[1]
        out = torch.full((3 + n * (per + 5) + 16,), 0xCD, dtype=torch.uint8, device=DEV)
        d_out = C.c_void_p(out.data_ptr() + 3)
        view = strided(dense, 4, ns + 1)
        nbo = C.c_int(0)
        rc = c.L.ft8b200_monitor_waterfall(C.c_void_p(c.h), _p(view), C.c_size_t(view.stride(0)), ns, n, rate, 2, 2, proto, d_out, C.c_size_t(per + 5),
                                           C.byref(nbo), _stream())
        assert rc == 0, last_error(pkg)
        torch.cuda.synchronize()
        o = out.cpu().numpy()
        assert nbo.value == nb and (o[:3] == 0xCD).all()
        for s in range(n):
            row = o[3 + s * (per + 5): 3 + s * (per + 5) + per + 5]
            assert np.array_equal(row[:per], b[s]) and (row[per:] == 0xCD).all(), (case, s)
    finally:
        c.close()


# ------------------------------------------------------------------------------------------- 4. OSD with an uncapped grid
@pytest.fixture(scope="module")
def osd_oracle(tmp_path_factory):
    return OsdOracle(tmp_path_factory.mktemp("osd_oracle_shapes"))


@pytest.mark.parametrize("protocol", [1, 0], ids=["ft8", "ft4"])
def test_osd_stage_entry_small_batch(pkg, osd_oracle, protocol, tmp_path):
    """ft8b200_osd with few entries: its grid is ceil(n x K / 8) CTAs, below the 2 x SMs cap every larger test runs at.
    Every entry against orc_osd; entries at stage 3/4 or past ncand are left alone."""
    S, K = 3, 125   # 375 entries: 47 CTAs, below the cap on any GPU with 24 or more SMs
    llrs = fuzz_llrs(osd_oracle, S * K, 77 + protocol).reshape(S, K, 174)
    rng = np.random.default_rng(6)
    stage0 = np.where(rng.random((S, K)) < 0.8, 1, rng.integers(2, 5, (S, K))).astype(np.uint8)
    ncand = np.array([K, K - 5, 0], np.int32)
    ctx = pkg.Context(0, max_candidates=K)
    try:
        ctx.set_protocol(protocol)
        for order in (1, 2):
            ctx.set_osd(order, 174)
            want = [[osd_oracle.osd(llrs[s, k], order, 174, protocol) for k in range(K)] for s in range(S)]
            ok = torch.zeros((S, K), dtype=torch.uint8, device=DEV)
            stage = torch.from_numpy(stage0).to(DEV)
            status = torch.full((S, K, 12), 0xA5, dtype=torch.uint8, device=DEV)
            msg = torch.full((S, K, 28), 0x5A, dtype=torch.uint8, device=DEV)
            (osd, hard, cw), ks = profiled(lambda: ctx.osd(torch.from_numpy(llrs).to(DEV), torch.from_numpy(ncand).to(DEV), ok, stage, status, msg,
                                                           want_cw=True), tmp_path, f"osd{order}")
            grids = [g for name, g in ks if "osd_kernel" in name]
            assert grids == [(-(-S * K // 8), 1, 1)] and grids[0][0] < 2 * sm_count(), grids
            osd, hard, cw, okn, stn = osd.cpu().numpy(), hard.cpu().numpy(), cw.cpu().numpy(), ok.cpu().numpy(), stage.cpu().numpy()
            accepted = 0
            for s in range(S):
                for k in range(K):
                    w = want[s][k]
                    if k < ncand[s] and stage0[s, k] in (1, 2) and w[0] >= 0:
                        acc = w[0] == 1
                        assert osd[s, k] == (2 if acc else 1) and hard[s, k] == w[2] and np.array_equal(cw[s, k], w[1]), (order, s, k)
                        accepted += acc
                        assert (okn[s, k], stn[s, k]) == ((1, 4) if acc else (0, stage0[s, k])), (order, s, k)
                    else:
                        assert osd[s, k] == 0 and hard[s, k] == -1 and not cw[s, k].any(), (order, s, k)
                        assert okn[s, k] == 0 and stn[s, k] == stage0[s, k], (order, s, k)
            assert accepted >= 3
    finally:
        ctx.close()


# ------------------------------------------------------------------------------------------- 5. more than 65 535 slots
@pytest.fixture(scope="module")
def daemon120(oracle, daemon):
    """The daemon waterfalls' own candidate lists (K = 120, min_score 10), the oracle's decode of each and its spot records."""
    mags = daemon[0]
    lists = [oracle.find_sync(m, max_cand=120, min_score=10) for m in mags]
    out = []
    for w, m in enumerate(mags):
        ents = [expected_entry(oracle, m, cd, DAEMON, 1)[:4] for cd in lists[w]]
        out.append((lists[w], ents, oracle.decode_waterfall(m)))
    return out


@pytest.mark.parametrize("n", [65537, 70001])
def test_find_sync_decode_spots_beyond_65535_slots(pkg, daemon, daemon120, bp_variant, n):
    """find_sync, decode and spots on more slots than gridDim.y holds: slots 0, 65534 ... 65537 and the last equal the oracle
    and every slot equals the slot it is a copy of."""
    mags = daemon[0]
    W = mags.shape[0]
    w_of = torch.arange(n, device=DEV) % W
    c = pkg.Context(0)
    try:
        d_mag = torch.from_numpy(mags).to(DEV)[w_of]
        cand, ncand = c.find_sync(d_mag)
        ok, stage, status, msg, _, _ = c.decode(d_mag, cand, ncand)
        res, nres, umsg, ufreq, uscore = c.spots(cand, ncand, ok, msg)
        torch.cuda.synchronize()
        del d_mag
        for t in (cand, ncand, ok, stage, status, msg, res, nres, umsg, ufreq, uscore):
            assert torch.equal(t, t[:W][w_of])
        for s in sorted({0, 65534, 65535, 65536, min(65537, n - 1), n - 1}):
            w = s % W
            lst, ents, o = daemon120[w]
            assert int(ncand[s]) == len(lst) and as_np(cand[s], cand_dtype)[: len(lst)].tobytes() == lst.tobytes(), s
            for k, (e_ok, e_stage, e_st, e_msg) in enumerate(ents):
                assert (int(ok[s, k]), int(stage[s, k])) == (e_ok, e_stage), (s, k)
                assert np.array_equal(status[s, k].cpu().numpy(), e_st) and np.array_equal(msg[s, k].cpu().numpy(), e_msg), (s, k)
            assert int(nres[s]) == o["n"] and as_np(res[s], result_dtype).tobytes() == o["results"].tobytes(), s
        assert int(nres[0]) >= 1 and int(nres[65536 - 65536 % W]) >= 1
    finally:
        c.close()
        torch.cuda.empty_cache()


def test_synth_audio_and_condition_beyond_65535_slots(pkg, oracle):
    """synth_audio (short recordings) and condition at 65 537 slots: slots on both sides of the 65 535-row launch boundary
    equal the CPU twin, and a piece generated on its own equals the same rows of the whole batch."""
    n, ns = 65537, 700
    with_sig = (0, 65534, 65535, 65536)
    first = np.zeros(n + 1, np.int32)
    for s in with_sig:
        first[s + 1:] += 1
    sig = pkg.make_signals([(pkg.pack77_std("CQ", "K1JT", "FN20"), 500.0 + 100 * k, 0.0, 0.3) for k in range(len(with_sig))])
    c = pkg.Context(0)
    try:
        a = c.synth_audio(sig, first, 1, 0.1, 42, first_slot_index=3, n_samples=ns)
        part = c.synth_audio(sig[1:], first[65530:n + 1] - first[65530], 1, 0.1, 42, first_slot_index=3 + 65530, n_samples=ns)
        torch.cuda.synchronize()
        assert torch.equal(part.view(torch.int32), a[65530:].view(torch.int32))
        for s in (0, 1, 65533, 65534, 65535, 65536):
            x, _ = oracle.synth_float(2, False, sig[first[s]:first[s + 1]], 0.1, 42, 3 + s, ns)
            assert np.array_equal(a[s].cpu().numpy().view(np.int32), x.view(np.int32)), s
        del a, part
        # condition: three distinct slots tiled over 65 537 rows
        rows = [synth.slot_f32([std_sig()], 31 + k) for k in range(3)]
        scale = np.float32([1.0, 3.7e-3, 250.0])
        hi = np.stack([r[0] * f for r, f in zip(rows, scale)]).astype(np.float32)
        hq = np.stack([r[1] * f for r, f in zip(rows, scale)]).astype(np.float32)
        peak = np.maximum(np.abs(hi).max(1), np.abs(hq).max(1)).astype(np.float32)
        w_of = torch.arange(n, device=DEV) % 3
        d_i, d_q = torch.from_numpy(hi).to(DEV)[w_of], torch.from_numpy(hq).to(DEV)[w_of]
        c.condition(d_i, d_q, torch.from_numpy(peak).to(DEV)[w_of])
        torch.cuda.synchronize()
        for w in range(3):
            ei, eq, _ = oracle.condition(hi[w], hq[w], 48000)
            ti, tq = torch.from_numpy(ei).to(DEV).view(torch.int32), torch.from_numpy(eq).to(DEV).view(torch.int32)
            assert bool((d_i[w::3].view(torch.int32) == ti).all()) and bool((d_q[w::3].view(torch.int32) == tq).all()), w
    finally:
        c.close()
        torch.cuda.empty_cache()


def test_process_conditioned_beyond_65535_slots(pkg, oracle):
    """One process_conditioned of 65 537 mostly silent slots; the slots with a message sit on both sides of the launch boundary."""
    n = 65537
    free, _ = torch.cuda.mem_get_info()
    if free < 48 * 2 ** 30:
        pytest.skip(f"needs about 35 GB of device memory, {free / 2 ** 30:.1f} GB free")
    i_s, q_s = synth.slot_f32([std_sig(900.0, 0.5, -5.0, ("K1ABC", "W9XYZ", "FN42"))], 17)
    i_s *= np.float32(2.5e-2); q_s *= np.float32(2.5e-2)
    pk = np.float32(max(np.abs(i_s).max(), np.abs(q_s).max()))
    o = oracle.subsystem(*oracle.condition(i_s, q_s, 48000)[:2])
    assert o["n"] >= 1
    loud = (0, 65534, 65535, 65536)
    c = pkg.Context(0)
    d_i = d_q = None
    try:
        d_i = torch.zeros((n, 48000), dtype=torch.float32, device=DEV)
        d_q = torch.zeros_like(d_i)
        peak = torch.zeros(n, dtype=torch.float32, device=DEV)
        for s in loud:
            d_i[s] = torch.from_numpy(i_s).to(DEV); d_q[s] = torch.from_numpy(q_s).to(DEV); peak[s] = float(pk)
        c.process_conditioned(d_i, d_q, peak)
        res, nres = c.fetch_results(n)
        for s in loud:
            assert nres[s] == o["n"] and res[s].tobytes() == o["results"].tobytes(), s
        quiet = np.ones(n, bool)
        quiet[list(loud)] = False
        assert not nres[quiet].any() and not res[quiet].view(np.uint8).any()
    finally:
        c.close()
        del d_i, d_q
        torch.cuda.empty_cache()


def test_raw_entries_refuse_more_than_65535_rows_and_keep_working(pkg, oracle):
    """The raw-IQ entry points take at most 65 535 streams or output rows per call (65 536 raw slots are 4.7 TB): decimate,
    decimate_streams, process_raw, process_raw_streams and the pipe's submits return FT8B200_EINVAL with a reason before anything
    runs.  The context and the pipe decode normally afterwards."""
    n = MAX_ROWS + 1
    c = pkg.Context(0)
    p = pkg.Pipe(0, depth=2)
    L, h, ph = c.L, C.c_void_p(c.h), C.c_void_p(p.h)
    try:
        iq = torch.zeros(4096, dtype=torch.uint8, device=DEV)
        f = torch.zeros(4096, dtype=torch.float32, device=DEV)
        st = _stream()
        rcs = {
            "decimate": L.ft8b200_decimate(h, _p(iq), C.c_size_t(16), C.c_size_t(16), n, _p(f), _p(f), _p(f), _p(f), None, st),
            "decimate_streams": L.ft8b200_decimate_streams(h, _p(iq), C.c_size_t(8 * n), C.c_size_t(8 * n), 1, n, C.c_size_t(8), _p(f), _p(f),
                                                           _p(f), _p(f), None, st),
            "process_raw": L.ft8b200_process_raw(h, _p(iq), C.c_size_t(16), C.c_size_t(16), n, st),
            "process_raw_streams": L.ft8b200_process_raw_streams(h, _p(iq), C.c_size_t(8 * n), C.c_size_t(8 * n), 1, n, C.c_size_t(8), st),
        }
        for name, rc in rcs.items():
            assert rc == EINVAL and "65535" in last_error(pkg), (name, rc, last_error(pkg))
        rc = L.ft8b200_pipe_submit(ph, _p(iq), C.c_size_t(16), C.c_size_t(16), n)
        assert rc == EINVAL and "65535" in L.ft8b200_pipe_error(ph).decode()
        rc = L.ft8b200_pipe_submit_streams(ph, _p(iq), C.c_size_t(8 * n), C.c_size_t(8 * n), 1, n, C.c_size_t(8))
        assert rc == EINVAL and "65535" in L.ft8b200_pipe_error(ph).decode()
        assert p.in_flight() == 0
        check_context_and_pipe_decode(c, p, oracle)
    finally:
        p.close()
        c.close()


def check_context_and_pipe_decode(c, p, oracle):
    i_s, q_s = conditioned(oracle, [std_sig()], 7)
    o = oracle.subsystem(i_s, q_s)
    assert o["n"] >= 1
    d_i, d_q = torch.from_numpy(i_s[None]).to(DEV), torch.from_numpy(q_s[None]).to(DEV)
    c.process_slots(d_i, d_q)
    res, nres = c.fetch_results(1)
    assert nres[0] == o["n"] and res[0].tobytes() == o["results"].tobytes()
    torch.cuda.synchronize()
    p.submit_slots(d_i, d_q)
    res, nres = p.collect(1)
    assert nres[0] == o["n"] and res[0].tobytes() == o["results"].tobytes()
    assert p.in_flight() == 0


# ------------------------------------------------------------------------------------------- 6. misaligned float slots
def test_misaligned_float_slots_are_refused(pkg, oracle):
    """process_slots, process_conditioned and the pipe's submit_slots with d_i or d_q 4 bytes off a 16-byte boundary return
    FT8B200_EINVAL with a reason (the waterfall kernel reads the samples with 16-byte copies); nothing is left in flight and
    the context and the pipe decode normally afterwards."""
    c = pkg.Context(0)
    p = pkg.Pipe(0, depth=2)
    L, h, ph = c.L, C.c_void_p(c.h), C.c_void_p(p.h)
    try:
        buf = torch.zeros(2 * 48000 + 16, dtype=torch.float32, device=DEV)
        good = torch.zeros((1, 48000), dtype=torch.float32, device=DEV)
        off = buf[1:1 + 48000].view(1, 48000)
        assert off.data_ptr() % 16 == 4 and good.data_ptr() % 16 == 0
        peak = torch.ones(1, dtype=torch.float32, device=DEV)
        st = _stream()
        for name, rc in (("process_slots d_i", L.ft8b200_process_slots(h, _p(off), _p(good), 1, st)),
                         ("process_slots d_q", L.ft8b200_process_slots(h, _p(good), _p(off), 1, st)),
                         ("process_conditioned d_i", L.ft8b200_process_conditioned(h, _p(off), _p(good), _p(peak), 1, st)),
                         ("process_conditioned d_q", L.ft8b200_process_conditioned(h, _p(good), _p(off), _p(peak), 1, st))):
            assert rc == EINVAL and "16-byte" in last_error(pkg), (name, rc)
        for args in ((off, good, None), (good, off, peak)):
            rc = L.ft8b200_pipe_submit_slots(ph, *[_p(a) for a in args], 1)
            assert rc == EINVAL and "16-byte" in L.ft8b200_pipe_error(ph).decode(), rc
            assert p.in_flight() == 0
        check_context_and_pipe_decode(c, p, oracle)
    finally:
        p.close()
        c.close()
