"""Belief propagation (a11: decode_kernel and decode_edges_kernel) against the float64 flooding decoder of tests/ref64.py,
round by round, and the LDPC iteration count through every entry point that takes it.

After n rounds the kernels write the last hard decision (`plain`) and the minimum parity error count (`ldpc_errors`), so
decoding the same candidates with ldpc_iterations = 0, 1, 2, ... shows their state round by round.  Each n is compared
  - byte for byte with the oracle at the same n (ok, stage, status, message, plain; LLRs bitwise, and equal for every n),
  - with ref64.bp_decode64 under the agreement rule below,
  - with invariants that need no reference: ldpc_errors never increases with n, a word once decoded stays decoded to the
    same bits and text, and n = 0 gives ldpc_errors = 83, stage 1, ok 0.

Agreement rule (ref64.TAU, ref64.bp_resolved).  The kernels are float32; the reference is float64.  A (candidate, n) pair
is resolved when every posterior of every round the float64 run executes up to n stays clear of zero by a margin.  For a
resolved pair the kernel's plain and ldpc_errors equal the reference's at n, and its stage is 1 when the reference leaves
parity errors, 2 when the reference's word fails the CRC-14, and 3 or 4 when it passes.  The margins and the resolved-fraction
bars were calibrated with the oracle (bit-equal to the kernels) against the same reference, on the CPU:
tests/test_tables_independent.py::test_oracle_bp_vs_float64.  The worst case is printed with -s."""
import numpy as np
import pytest

import ref64
from oracle.pyoracle import cand_dtype, msg_dtype, status_dtype
from tools import ft8enc, synth

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

DEV = torch.device("cuda:0")
ITERS = (0, 1, 2, 3, 4, 5, 7, 10, 15, 20, 25, 35, 50, 100)
DAEMON = dict(num_blocks=92, num_bins=256, time_osr=2, freq_osr=2)
FT8_12K = dict(num_blocks=93, num_bins=960, time_osr=2, freq_osr=2)
FT4_12K = dict(num_blocks=156, num_bins=288, time_osr=2, freq_osr=2)
# crowded_band seeds at -24 .. -14 dB whose candidates include words that float64 BP decodes only after round 20
LATE_SEEDS = (201, 203, 210, 212, 214)


def report(what, value):
    print(f"\n[bp] {what}: {value}")


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def as_np(t, dt):
    a = t.cpu().numpy()
    return a.view(dt).reshape(a.shape[:-1])


@pytest.fixture(params=[0, 1], ids=["bp_nodes", "bp_edges"])
def bp_variant(request, pkg):
    pkg.set_decode_variant(request.param)
    yield request.param
    pkg.set_decode_variant(0)


# ------------------------------------------------------------------------------------------- expectations
def oracle_entry(oracle, mag, cand, n, dims, protocol):
    """Every byte ft8b200_decode writes for one candidate after n rounds, from the oracle: ok, stage, status (fields the
    reference leaves unwritten are 0), message (zero unless decoded), plain, LLRs."""
    d = oracle.decode(mag, cand, max_iters=n, protocol=protocol, **dims)
    s = d["status"]
    stage = 1 if s["ldpc_errors"] > 0 else 2 if s["crc_extracted"] != s["crc_calculated"] else 4 if d["ok"] else 3
    st = np.zeros(1, status_dtype)
    st[0] = (s["ldpc_errors"], s["crc_extracted"] if stage >= 2 else 0, s["crc_calculated"] if stage >= 2 else 0, s["unpack_status"] if stage >= 3 else 0)
    m = np.zeros(1, msg_dtype)
    if d["ok"]:
        m[0]["text"], m[0]["hash"] = d["msg"]["text"], d["msg"]["hash"]
    return d["ok"], stage, st.view(np.uint8), m.view(np.uint8), d["plain"], d["llr"]


class Case:
    """Waterfalls of one geometry, their candidates, and per n of ITERS the oracle's outputs for every live candidate,
    flattened in (slot, candidate) order; plus the float64 trajectory of the oracle's LLRs."""

    def __init__(self, oracle, name, mags, cands, ncand, dims, protocol, iters=ITERS):
        self.name, self.mags, self.cands, self.ncand, self.dims, self.protocol = name, mags, cands, ncand, dims, protocol
        self.where = [(s, k) for s in range(mags.shape[0]) for k in range(int(ncand[s]))]
        self.iters = iters
        E = len(self.where)
        self.ok = np.zeros((len(iters), E), np.uint8); self.stage = np.zeros((len(iters), E), np.uint8)
        self.status = np.zeros((len(iters), E, 12), np.uint8); self.msg = np.zeros((len(iters), E, 28), np.uint8)
        self.plain = np.zeros((len(iters), E, 174), np.uint8); self.llr = np.zeros((E, 174), np.float32)
        for i, n in enumerate(iters):
            for e, (s, k) in enumerate(self.where):
                (self.ok[i, e], self.stage[i, e], self.status[i, e], self.msg[i, e], self.plain[i, e], llr) = \
                    oracle_entry(oracle, mags[s], cands[s, k], n, dims, protocol)
                if i == 0:
                    self.llr[e] = llr
        self.traj = ref64.bp_decode64(self.llr, max(iters))

    def live(self, t):
        """[S, K, ...] device output -> [E, ...] numpy over the live candidates."""
        a = t.cpu().numpy()
        return np.stack([a[s, k] for s, k in self.where]) if self.where else a.reshape((0,) + a.shape[2:])


def sub_traj(traj, sel):
    """bp_decode64's trajectory restricted to the candidates `sel`."""
    return {k: (v[:, sel] if k in ("bits", "errors", "margin", "ran") else v[sel]) for k, v in traj.items()}


class Agreement:
    """The agreement rule's tallies over many (candidate, n) pairs."""

    def __init__(self):
        self.pairs = self.resolved = self.pairs_small = self.resolved_small = 0
        self.worst = np.inf

    def check(self, traj, llr, n, plain, errors, stage, what):
        rp, re_, margin = ref64.bp_resolved(traj, llr, n)
        res = margin >= 1
        for e in np.flatnonzero(res):
            assert np.array_equal(plain[e], rp[e]) and int(errors[e]) == int(re_[e]), \
                f"{what} n={n} candidate {e}: kernel (errors {int(errors[e])}) differs from float64 BP (errors {int(re_[e])}, margin {margin[e]:.3g})"
            want = (1,) if re_[e] > 0 else (3, 4) if ref64.crc_ok(rp[e]) else (2,)
            assert int(stage[e]) in want, (what, n, e, int(stage[e]), want)
        self.pairs += res.size; self.resolved += int(res.sum())
        if n <= 5:
            self.pairs_small += res.size; self.resolved_small += int(res.sum())
        if res.any():
            self.worst = min(self.worst, float(margin[res].min()))

    def finish(self, what, bar, bar_small):
        f = self.resolved / max(self.pairs, 1)
        fs = self.resolved_small / self.pairs_small if self.pairs_small else 1.0
        report(f"{what}: resolved pairs", f"{self.resolved}/{self.pairs} = {f:.4f} (n <= 5: {fs:.4f}); smallest margin of a resolved pair "
               f"{self.worst:.3g} x its bar")
        assert f >= bar and fs >= bar_small, (f, fs)


# ------------------------------------------------------------------------------------------- inputs
def _cond(oracle, i_s, q_s):
    return tuple(oracle.condition(i_s, q_s, 48000)[:2])


@pytest.fixture(scope="module")
def daemon_raw():
    """Unconditioned daemon slots: one with strong signals (words whose hard decision is already a codeword) and
    LATE_SEEDS at -24 .. -14 dB (words that need many rounds, and many that never converge)."""
    slots = [synth.crowded_band(ft8enc, 15, 300, snr_lo=-6, snr_hi=6)[:2]]
    slots += [synth.crowded_band(ft8enc, 40, s, snr_lo=-24, snr_hi=-14)[:2] for s in LATE_SEEDS]
    return slots


def ft4_audio(pkg, ctx, seed, n=6):
    """FT4 recording made by the device synthesiser: n CQ messages near the threshold."""
    rng = np.random.default_rng(seed)
    items = []
    for k in range(n):
        _, de, _ = synth.random_message(rng)
        items.append((pkg.pack77_std("CQ", de, synth.random_grid(rng)), 300.0 + 330.0 * k + float(rng.uniform(0, 40)), float(rng.uniform(0.2, 1.0)),
                      float(rng.uniform(0.01, 0.05))))
    return ctx.synth_audio(pkg.make_signals(items), [0, n], 0, 0.05, seed, n_samples=90_000)


def ft8_12k_audio(seed):
    rng = np.random.default_rng(seed)
    sigs = [(ft8enc.tones(ft8enc.pack_std("CQ", de, synth.random_grid(rng))), 300.0 + 400.0 * k + float(rng.uniform(0, 50)),
             float(rng.uniform(0.2, 1.2)), float(rng.uniform(0.005, 0.03)))
            for k, de in enumerate(("K1JT", "W9XYZ", "K1ABC", "DL1AAA", "JA1XYZ", "G4ABC"))]
    return synth.audio_12k(sigs, seed)


@pytest.fixture(scope="module")
def cases(pkg, ctx, oracle, daemon_raw):
    """Case per geometry: daemon slots (GPU waterfall of the conditioned slots), a 12 kHz FT8 and an FT4 recording
    (GPU monitor), candidates from the GPU find_sync at K = 120."""
    out = {}
    c = pkg.Context(0, max_candidates=120, max_messages=50, min_score=10)
    try:
        cond = [_cond(oracle, *s) for s in daemon_raw]
        hi = np.stack([s[0] for s in cond]); hq = np.stack([s[1] for s in cond])
        mag = c.waterfall(torch.from_numpy(hi).to(DEV), torch.from_numpy(hq).to(DEV))
        srcs = [("daemon", mag, DAEMON, 1)]
        m, nb = c.monitor_waterfall(torch.from_numpy(ft8_12k_audio(5)[None]).to(DEV))
        assert nb == FT8_12K["num_blocks"]
        srcs.append(("ft8_12k", m[:, : FT8_12K["num_blocks"] * 2 * 2 * 960].contiguous(), FT8_12K, 1))
        m, nb = c.monitor_waterfall(ft4_audio(pkg, c, 13), protocol=0)
        assert nb == FT4_12K["num_blocks"]
        srcs.append(("ft4", m[:, : FT4_12K["num_blocks"] * 2 * 2 * 288].contiguous(), FT4_12K, 0))
        for name, d_mag, dims, proto in srcs:
            c.set_protocol(proto)
            cand, ncand = c.find_sync(d_mag, **dims)
            out[name] = (Case(oracle, name, d_mag.cpu().numpy(), as_np(cand, cand_dtype), ncand.cpu().numpy(), dims, proto), d_mag, cand, ncand)
    finally:
        c.close()
    out["daemon_cond"] = cond
    return out


# ------------------------------------------------------------------------------------------- a. trajectories
def test_bp_trajectories(pkg, cases, bp_variant):
    """Every n of ITERS on daemon slots, a 12 kHz FT8 and an FT4 recording, under both kernels."""
    ctxs = {n: pkg.Context(0, max_candidates=120, max_messages=50, min_score=10, ldpc_iterations=n) for n in ITERS}
    agree = Agreement()
    try:
        for name in ("daemon", "ft8_12k", "ft4"):
            case, d_mag, cand, ncand = cases[name]
            got = {}
            for n in ITERS:
                c = ctxs[n]
                c.set_protocol(case.protocol)
                ok, stage, status, msg, plain, llr = c.decode(d_mag, cand, ncand, want_plain=True, want_llr=True, **case.dims)
                got[n] = dict(ok=case.live(ok), stage=case.live(stage), status=case.live(status), msg=case.live(msg), plain=case.live(plain),
                              llr=case.live(llr))
            for i, n in enumerate(ITERS):
                g = got[n]
                assert np.array_equal(g["llr"].view(np.uint32), case.llr.view(np.uint32)), (name, n, "LLRs differ from the oracle's")
                for key in ("ok", "stage", "status", "msg", "plain"):
                    want = getattr(case, key)[i]
                    bad = np.argwhere(g[key] != want)
                    assert not bad.size, f"{name} n={n}: {key} differs from the oracle's at candidate {case.where[bad[0][0]]}"
                errors = g["status"][:, :4].copy().view(np.int32)[:, 0]
                agree.check(case.traj, case.llr, n, g["plain"], errors, g["stage"], name)
            # invariants that need no reference
            errs = np.stack([got[n]["status"][:, :4].copy().view(np.int32)[:, 0] for n in ITERS])
            assert (np.diff(errs, axis=0) <= 0).all(), f"{name}: ldpc_errors grew with n"
            assert (errs[0] == 83).all() and (got[0]["stage"] == 1).all() and not got[0]["ok"].any() and not got[0]["plain"].any()
            for i, n in enumerate(ITERS):
                for m in ITERS[i + 1:]:
                    done = got[n]["ok"] == 1
                    assert (got[m]["ok"][done] == 1).all() and np.array_equal(got[m]["plain"][done], got[n]["plain"][done]) \
                        and np.array_equal(got[m]["msg"][done], got[n]["msg"][done]), (name, n, m)
        # coverage: the float64 run converges in round 1, 2-5, 6-20 and 21-100 for several candidates each, and never for some
        s = np.concatenate([cases[k][0].traj["stop"] for k in ("daemon", "ft8_12k", "ft4")])
        z = np.concatenate([cases[k][0].traj["zero"] for k in ("daemon", "ft8_12k", "ft4")])
        conv = (s > 0) & ~z
        groups = {"1": conv & (s == 1), "2-5": conv & (s >= 2) & (s <= 5), "6-20": conv & (s >= 6) & (s <= 20), "21-100": conv & (s > 20)}
        counts = {k: int(v.sum()) for k, v in groups.items()}
        report(f"convergence round of float64 BP over {s.size} candidates", dict(counts, never=int((s == 0).sum())))
        assert all(v >= 5 for v in counts.values()) and (s == 0).sum() >= 1, counts
        agree.finish(f"trajectories, {'nodes' if bp_variant == 0 else 'edges'}", 0.75, 0.85)
    finally:
        for c in ctxs.values():
            c.close()


# ------------------------------------------------------------------------------------------- b. decode modes
@pytest.mark.parametrize("n", [1, 20, 50])
@pytest.mark.parametrize("mode", ["grid", "pull"])
def test_bp_decode_modes(pkg, cases, bp_variant, mode, n):
    """The (candidate group, slot) grid below slots x K = 32 x SMs and the node kernel's pull counter above it, on the
    daemon slots repeated.  The mode follows from slots x K and the kernel variant alone; test_gpu_shapes.py shows with the
    profiler which kernel and grid these sizes select.  This file does not profile: a profiling session early in a pytest
    process left the traces of later sessions without their first kernels."""
    case, d_mag, cand, ncand = cases["daemon"]
    S = case.mags.shape[0]
    T = 32 * sm_count()
    n_slots = S if mode == "grid" else T // 120 + 1 + S
    assert (n_slots * 120 > T) == (mode == "pull")
    w_of = torch.arange(n_slots, device=DEV) % S
    c = pkg.Context(0, max_candidates=120, ldpc_iterations=n)
    try:
        ok, stage, status, msg, plain, llr = c.decode(d_mag[w_of].contiguous(), cand[w_of].contiguous(), ncand[w_of].contiguous(),
                                                      want_plain=True, want_llr=True)
        i = ITERS.index(n)
        agree = Agreement()
        for r in range(n_slots):
            sel = [e for e, (s, _) in enumerate(case.where) if s == r % S]
            ks_ = [case.where[e][1] for e in sel]
            for key, t in (("ok", ok), ("stage", stage), ("status", status), ("msg", msg), ("plain", plain)):
                assert np.array_equal(t[r].cpu().numpy()[ks_], getattr(case, key)[i][sel]), (mode, n, r, key)
            g_plain = plain[r].cpu().numpy()[ks_]
            errors = status[r].cpu().numpy()[ks_][:, :4].copy().view(np.int32)[:, 0]
            agree.check(sub_traj(case.traj, sel), case.llr[sel], n, g_plain, errors, stage[r].cpu().numpy()[ks_], f"{mode} slot {r}")
        agree.finish(f"{mode} n={n}", 0.75, 0.85)
    finally:
        c.close()


@pytest.mark.parametrize("n", [1, 20, 50])
def test_bp_work_list(pkg, oracle, cases, n):
    """process_slots decodes from the work list the sync selection writes: its ok, status and message bytes equal the
    oracle's at n, its ldpc_errors follow the agreement rule, and its spot records equal ft8_subsystem() at n."""
    case, _, _, ncand = cases["daemon"]
    cond = cases["daemon_cond"]
    S = len(cond)
    c = pkg.Context(0, ldpc_iterations=n)
    try:
        d_i = torch.from_numpy(np.stack([s[0] for s in cond])).to(DEV)
        d_q = torch.from_numpy(np.stack([s[1] for s in cond])).to(DEV)
        c.process_slots(d_i, d_q)
        c.sync()
        w = c.workspace_ptrs()

        class _Arr:
            def __init__(self, ptr, shape, typestr):
                self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2}
        g = lambda key, shape: torch.as_tensor(_Arr(w[key], shape, "|u1"), device=DEV).clone()
        ok, status, msg = g("ok", (S, c.K)), g("status", (S, c.K, 12)), g("msg", (S, c.K, 28))
        res, nres = c.fetch_results(S)
        i = ITERS.index(n)
        assert np.array_equal(case.live(ok), case.ok[i]) and np.array_equal(case.live(status), case.status[i]) and np.array_equal(case.live(msg), case.msg[i])
        errors = case.live(status)[:, :4].copy().view(np.int32)[:, 0]
        rp, re_, margin = ref64.bp_resolved(case.traj, case.llr, n)
        res_ = margin >= 1
        assert np.array_equal(errors[res_], re_[res_]) and res_.mean() >= 0.75, res_.mean()
        for s in range(S):
            o = oracle.subsystem(*cond[s], iters=n)
            assert nres[s] == o["n"] and res[s].tobytes() == o["results"].tobytes(), s
    finally:
        c.close()


# ------------------------------------------------------------------------------------------- c. hand-made edges
@pytest.mark.parametrize("n", [1, 100])
def test_bp_hand_made_waterfalls(pkg, oracle, daemon_raw, bp_variant, n):
    """Every data symbol at tone 0 (LLRs of one sign: the hard decision is the all-zero word and BP gives up before any
    check), saturated cells (messages reach the tanh clamp), one live row, and a flat waterfall (NaN LLRs)."""
    rng = np.random.default_rng(8)
    tone0 = rng.integers(40, 70, 94208).astype(np.uint8).reshape(92, 2, 2, 256)
    tone0[:, :, :, 30] = 220
    flat = np.full(94208, 77, np.uint8)
    one_row = flat.copy().reshape(92, 2, 2, 256)
    one_row[40] = rng.integers(0, 256, size=(2, 2, 256), dtype=np.uint8)
    i_s, q_s = _cond(oracle, *daemon_raw[0])
    sat = oracle.waterfall(i_s * np.float32(400.0), q_s * np.float32(400.0))
    assert (sat == 255).sum() > 10000
    mags = np.stack([tone0.reshape(-1), flat, one_row.reshape(-1), sat])
    K = 120
    cands = np.zeros((4, K), cand_dtype)
    picks = [(20, 0, 30, 0, 0), (20, 5, 30, 1, 1), (20, -12, 100, 1, 1), (20, 23, 248, 1, 0), (20, -7, 33, 0, 0)]
    cands[:3, : len(picks)] = np.array(picks, cand_dtype)
    found = oracle.find_sync(sat, K, 10)
    cands[3, : found.size] = found
    ncand = np.array([len(picks)] * 3 + [found.size], np.int32)
    case = Case(oracle, "edges", mags, cands, ncand, DAEMON, 1, iters=(n,))
    c = pkg.Context(0, max_candidates=K, ldpc_iterations=n)
    try:
        ok, stage, status, msg, plain, llr = c.decode(torch.from_numpy(mags).to(DEV), torch.from_numpy(cands.view(np.uint8).reshape(4, K, 8)).to(DEV),
                                                      torch.from_numpy(ncand).to(DEV), want_plain=True, want_llr=True)
        g = dict(ok=case.live(ok), stage=case.live(stage), status=case.live(status), msg=case.live(msg), plain=case.live(plain))
        gl = case.live(llr)
        assert np.array_equal(np.isnan(gl), np.isnan(case.llr)) and np.array_equal(np.nan_to_num(gl).view(np.uint32), np.nan_to_num(case.llr).view(np.uint32))
        for key, v in g.items():
            assert np.array_equal(v, getattr(case, key)[0]), key
        errors = g["status"][:, :4].copy().view(np.int32)[:, 0]
        agree = Agreement()
        agree.check(case.traj, case.llr, n, g["plain"], errors, g["stage"], "hand-made")
        # tone 0: every LLR negative, all-zero word, 83 errors
        assert (case.llr[:2] < 0).all() and not g["plain"][:2].any() and (errors[:2] == 83).all() and (g["stage"][:2] == 1).all()
        # flat: NaN LLRs, all-zero word, 83 errors
        flat_e = [e for e, (s, _) in enumerate(case.where) if s == 1]
        assert np.isnan(case.llr[flat_e]).all() and not g["plain"][flat_e].any() and (errors[flat_e] == 83).all()
        # saturated: some messages start beyond the clamp (|llr| / 2 > 4.97 in round 1)
        sat_e = [e for e, (s, _) in enumerate(case.where) if s == 3]
        assert (np.abs(case.llr[sat_e]) > 2 * ref64.TANH_CLAMP).any()
    finally:
        c.close()


# ------------------------------------------------------------------------------------------- d. every entry point
@pytest.fixture(scope="module")
def raw_case(oracle):
    """One raw 2.4 Msps slot with two messages, and the oracle's conditioned decimation of it."""
    sigs = [(ft8enc.tones(ft8enc.pack_std("CQ", "K1JT", "FN20")), 800.0, 0.5, 20.0), (ft8enc.tones(ft8enc.pack_std("CQ", "W9XYZ", "EN37")), 1200.0, 0.8, 3.0)]
    raw = synth.raw_u8(sigs, 3)
    oi, oq = oracle.decimate_slot(raw)
    ri = np.zeros(48000, np.float32); rq = np.zeros(48000, np.float32)
    ri[:oi.size] = oi; rq[:oq.size] = oq
    return raw, tuple(oracle.condition(ri, rq, oi.size)[:2])


def _same_records(res, nres, want, what):
    for s, o in enumerate(want):
        assert nres[s] == o["n"] and res[s].tobytes() == o["results"].tobytes(), (what, s)


@pytest.mark.parametrize("n", [0, 1, 7, 50])
def test_iteration_count_reaches_every_entry_point(pkg, ctx, oracle, cases, daemon_raw, raw_case, n):
    """ldpc_iterations = n through process_conditioned, process_slots, process_raw, a pipe, a one-device cluster and
    ft8b200_decode_audio: spot records byte-equal to the oracle's ft8_subsystem() / decode_ft8 at n."""
    cond = cases["daemon_cond"][:3]
    want = [oracle.subsystem(i, q, iters=n) for i, q in cond]
    raw, raw_cond = raw_case
    want_raw = [oracle.subsystem(*raw_cond, iters=n)]
    d_i = torch.from_numpy(np.stack([s[0] for s in cond])).to(DEV)
    d_q = torch.from_numpy(np.stack([s[1] for s in cond])).to(DEV)
    d_raw = torch.from_numpy(raw[None]).to(DEV)
    c = pkg.Context(0, ldpc_iterations=n)
    try:
        c.process_slots(d_i, d_q)
        _same_records(*c.fetch_results(3), want, "process_slots")
        ri = np.stack([s[0] for s in daemon_raw[:3]]); rq = np.stack([s[1] for s in daemon_raw[:3]])
        peak = torch.from_numpy(np.maximum(np.abs(ri).max(1), np.abs(rq).max(1)).astype(np.float32)).to(DEV)
        c.process_conditioned(torch.from_numpy(ri).to(DEV), torch.from_numpy(rq).to(DEV), peak)
        _same_records(*c.fetch_results(3), want, "process_conditioned")
        c.process_raw(d_raw, 1)
        _same_records(*c.fetch_results(1), want_raw, "process_raw")
        audio = [(1, ft8_12k_audio(5)), (0, ft4_audio(pkg, ctx, 13).cpu().numpy()[0])]
        n_lines = 0
        for proto, a in audio:
            got = [pkg.format_decoded(r) for r in pkg.decode_audio(c, torch.from_numpy(a[None]).to(DEV), 12000, proto)[0]]
            assert got == oracle.decode_ft8_lines(a, 12000, protocol=proto, iters=n), proto
            n_lines += len(got)
    finally:
        c.close()
    p = pkg.Pipe(0, 2, ldpc_iterations=n)
    try:
        p.submit_slots(d_i, d_q)
        _same_records(*p.collect(3), want, "pipe")
    finally:
        p.close()
    cl = pkg.Cluster(1, 2, ldpc_iterations=n)
    try:
        cl.submit([d_raw], [1])
        _same_records(*cl.collect(1), want_raw, "cluster")
    finally:
        cl.close()
    spots = sum(o["n"] for o in want + want_raw)
    assert (spots == 0 and n_lines == 0) if n == 0 else spots >= 2, (n, spots, n_lines)


# ------------------------------------------------------------------------------------------- e. the drop-in cache
def test_dropin_cache_keys_on_iteration_count(pkg, oracle, cases):
    """ft8_find_sync decodes and caches at the default 20 rounds; ft8_decode with max_iterations 1, 5, 20, 50, 20 on the
    same waterfall and candidates answers each count as the oracle does, the second 20 included."""
    case = cases["daemon"][0]
    mag = np.ascontiguousarray(case.mags[1])
    heap = pkg.ft8_find_sync(mag, 120, 10)
    o = oracle.find_sync(mag, 120, 10)
    assert np.array_equal(heap.view(cand_dtype), o)
    answers = {}
    for it in (1, 5, 20, 50, 20):
        got = []
        for cd in o:
            ok, msg, st = pkg.ft8_decode(mag, cd, it)
            d = oracle.decode(mag, cd, max_iters=it)
            assert ok == bool(d["ok"]) and st.tobytes() == d["status"].tobytes(), (it, cd)
            if ok:
                assert msg.tobytes() == d["msg"].tobytes(), (it, cd)
            got.append(st.tobytes() + (msg.tobytes() if ok else b""))
        answers.setdefault(it, got)
        assert answers[it] == got
    assert answers[1] != answers[5] != answers[20] != answers[50], "the counts give different answers on this slot"
