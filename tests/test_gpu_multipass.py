"""Multi-pass decoding on the daemon path (ft8b200_set_passes, later_passes in csrc/api.cu) against a composition of its stages
(DESIGN.md section 2.4.2).  The composition runs the stage-wise entry points -- waterfall with the slot's original peak, find_sync,
decode, OSD, subtract -- on a second context with the same configuration, and decides which messages each pass subtracts with
subtract_ref.accept, the spot table's rule.  The daemon's records must equal orc_spots over every pass's rows, byte for byte: the
kernels are the same, deterministic and batch-invariant, so there is no tolerance."""
import numpy as np
import pytest

import subtract_ref as sr
from oracle.pyoracle import cand_dtype, msg_dtype, result_dtype
from test_gpu_subtract import _Arr, pass1_rows
from tools import synth
from tools.perf_subtract import amp_for

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
DEV = torch.device("cuda:0")

CONFIGS = {"default": dict(), "k500_m200": dict(max_candidates=500, max_messages=200), "m8": dict(max_messages=8),
           "min_score0": dict(min_score=0)}
STATS = {}   # non-vacuity counts, summed over the matrix (test_the_matrix_reaches_every_case)


def cfg_of(name):
    c = dict(max_candidates=120, max_messages=50, min_score=10)
    c.update(CONFIGS[name])
    return c


def fixture_items(pkg, seed, n_crowded=12, specials_first=False):
    """Seeded GFSK messages for noise 1.0 -> (signal_dtype array, first int32[n + 1]).  Slots: n_crowded of 10-60 CQ messages at
    -20 ... -8 dB and t0 0.5 +- 0.3 s, a quarter of them with about a third of their signals at t0 in [-0.8, -0.1] or [2.4, 3.2] s;
    the same message twice, 200 Hz apart; non-CQ standard messages with a few CQs; noise only; one strong message (these four
    first with specials_first)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    slots = []
    for s in range(n_crowded):
        edge = s % 4 == 1
        sp = []
        for _ in range(int(rng.integers(10, 61))):
            t0 = 0.5 + rng.uniform(-0.3, 0.3)
            if edge and rng.random() < 0.35:
                t0 = rng.uniform(-0.8, -0.1) if rng.random() < 0.5 else rng.uniform(2.4, 3.2)
            sp.append((pkg.pack77_std("CQ", synth.random_call(rng), synth.random_grid(rng)), float(rng.uniform(100, 1500)), float(t0),
                       amp_for(float(rng.uniform(-20, -8)))))
        slots.append(sp)
    dup = pkg.pack77_std("CQ", "K1DUP", "FN42")
    slots.append([(dup, 800.0, 0.5, amp_for(-9.0)), (dup, 1000.0, 0.62, amp_for(-10.0))]
                 + [(pkg.pack77_std("CQ", synth.random_call(rng), synth.random_grid(rng)), float(rng.uniform(100, 1500)), 0.5, amp_for(-14.0))
                    for _ in range(6)])
    non_cq = [("K1ABC", "W9XYZ", "RR73"), ("W9XYZ", "K1ABC", "R-12"), ("DL1ABC", "G4XYZ", "JO62"), ("G4XYZ", "DL1ABC", "73"),
              ("JA1ABC", "VK2XYZ", "-08"), ("VK2XYZ", "JA1ABC", "QF56")]
    slots.append([(pkg.pack77_std(*m), 200.0 + 180.0 * k, 0.4 + 0.05 * k, amp_for(-12.0)) for k, m in enumerate(non_cq)]
                 + [(pkg.pack77_std("CQ", synth.random_call(rng), synth.random_grid(rng)), 300.0 + 180.0 * k, 0.6, amp_for(-11.0)) for k in range(5)])
    slots.append([])
    slots.append([(pkg.pack77_std("CQ", "W1AW", "FN31"), 1234.5, 0.55, amp_for(0.0))])
    if specials_first:
        slots = slots[-1:] + slots[n_crowded:-1] + slots[:n_crowded]
    items = [it for sp in slots for it in sp]
    first = np.cumsum([0] + [len(sp) for sp in slots]).astype(np.int32)
    return pkg.make_signals(items, gfsk=True), first


def filling_slot(pkg, ctx, n_sig, seed):
    """One slot of n_sig CQ messages (-20 ... -8 dB, noise 1.0) whose first pass accepts 7 messages and whose second pass an 8th:
    an 8-message table fills during pass 2 (seeds found by running both passes)."""
    rng = np.random.Generator(np.random.PCG64(100 * seed + n_sig))
    items = [(pkg.pack77_std("CQ", synth.random_call(rng), synth.random_grid(rng)), float(rng.uniform(100, 1500)), float(0.5 + rng.uniform(-0.3, 0.3)),
              amp_for(float(rng.uniform(-20, -8)))) for _ in range(n_sig)]
    return ctx.synth_slots(pkg.make_signals(items, gfsk=True), np.array([0, n_sig], np.int32), 1.0, seed)


@pytest.fixture(scope="module")
def slots(pkg):
    """Device slots (noise 1.0): raw samples and their peaks, and the same slots conditioned (for process_slots, which takes no peak)."""
    sig, first = fixture_items(pkg, 0x3A55)
    ctx = pkg.Context(0)
    parts = [ctx.synth_slots(sig, first, 1.0, 0x3A55), filling_slot(pkg, ctx, 10, 3), filling_slot(pkg, ctx, 12, 1)]
    d_i, d_q = torch.cat([a for a, _ in parts]).contiguous(), torch.cat([b for _, b in parts]).contiguous()
    peak = torch.maximum(d_i.abs().amax(1), d_q.abs().amax(1)).contiguous()
    c_i, c_q = d_i.clone(), d_q.clone()
    ctx.condition(c_i, c_q, peak.clone())
    torch.cuda.synchronize()
    ctx.close()
    return d_i, d_q, peak, c_i, c_q


@pytest.fixture(scope="module")
def raw(pkg):
    """8 raw 2.4 Msps slots (GFSK, the same kinds of slot as above but fewer crowded ones), the special slots first so that the first
    overlap group decodes something.  6 dB stronger than the float slots against noise of 30 LSB: at their levels the crowded raw
    slots decode next to nothing."""
    sig, first = fixture_items(pkg, 0x7E11, n_crowded=4, specials_first=True)
    sig["amp"] *= np.float32(2.0 * np.sqrt(2 * 900.0 * 2500 / 2.4e6) / np.sqrt(2 * 2500 / 3200.0))
    ctx = pkg.Context(0)
    iq = ctx.synth_raw(sig, first, 30.0, 0x7E11)
    torch.cuda.synchronize()
    ctx.close()
    return iq


def stage(c, x_i, x_q, peak, osd):
    """Pass rows of one batch from the stage-wise entries: waterfall -> find_sync -> decode (+ OSD)."""
    mag = c.waterfall(x_i, x_q, peak)
    cand, ncand = c.find_sync(mag)
    ok, stg, status, msg, plain, llr = c.decode(mag, cand, ncand, want_plain=True, want_llr=bool(osd))
    if osd:
        c.osd(llr, ncand, ok, stg, status, msg, plain=plain)
    torch.cuda.synchronize()
    n = x_i.shape[0]
    return dict(cand=cand.cpu().numpy().view(cand_dtype).reshape(n, c.K), ncand=ncand.cpu().numpy(), ok=ok.cpu().numpy(),
                status=status.cpu().numpy(), msg=msg.cpu().numpy().view(msg_dtype).reshape(n, c.K), plain=plain.cpu().numpy())


def compose(c, oracle, x_i, x_q, peak, passes, osd, cfg, stats):
    """The definition of passes 1 ... `passes` on a batch -> (pass-1 rows, expected records, expected counts)."""
    n, M = x_i.shape[0], cfg["max_messages"]
    R = stage(c, x_i, x_q, peak, osd)
    first_rows = R
    logs = [[] for _ in range(n)]
    rows = [[] for _ in range(n)]   # per slot: (cand, ok, msg) of every pass
    acc = []
    for s in range(n):
        nc = int(R["ncand"][s])
        rows[s].append((R["cand"][s, :nc], R["ok"][s, :nc], R["msg"][s, :nc]))
        acc.append(sr.accept(rows[s][-1], logs[s], M, cfg["min_score"]))
    full_after_1 = [len(lg) == M for lg in logs]
    for p in range(2, passes + 1):
        cand = np.zeros((n, M), cand_dtype)
        cw = np.zeros((n, M, 174), np.uint8)
        nmsg = np.array([len(a) for a in acc], np.int32)
        for s in range(n):
            for j, k in enumerate(acc[s]):
                cand[s, j], cw[s, j] = R["cand"][s, k], R["plain"][s, k]
                stats["non_cq_subtracted"] += not bytes(R["msg"][s, k]["text"]).startswith(b"CQ ")
        y_i, y_q, grid = c.subtract(x_i, x_q, torch.from_numpy(cand.view(np.uint8).reshape(n, M, 8)).to(DEV), torch.from_numpy(cw).to(DEV),
                                    torch.from_numpy(nmsg).to(DEV))
        idle = torch.from_numpy(nmsg == 0).to(DEV)
        y_i[idle] = 0.0
        y_q[idle] = 0.0
        stats[f"idle_at_pass{p}"] += int((nmsg == 0).sum())
        g = grid.cpu().numpy()
        for s in range(n):
            for j in range(int(nmsg[s])):
                S = sr.nominal(cand[s, j])[0] + int(g[s, j, 0])
                stats["crosses_start"] += S < 0 < S + sr.SPAN
                stats["crosses_end"] += S < sr.SLOT < S + sr.SPAN
        R = stage(c, y_i, y_q, peak, osd)
        for s in range(n):
            nc = int(R["ncand"][s])
            pr = (R["cand"][s, :nc], R["ok"][s, :nc], R["msg"][s, :nc])
            earlier = set(logs[s])
            live = [sr.message_key(pr[2][k]) for k in range(nc) if pr[1][k] and pr[0][k]["score"] >= cfg["min_score"]]
            stats["cross_pass_duplicates"] += sum(key in earlier for key in live)
            rows[s].append(pr)
            before = len(logs[s])
            acc[s] = sr.accept(pr, logs[s], M, cfg["min_score"])
            stats[f"appended_in_pass{p}"] += len(acc[s])
            if p == 2 and M == 8:
                stats["m8_full_after_pass1"] += full_after_1[s]
                stats["m8_fills_in_pass2"] += before < M and len(logs[s]) == M
        x_i, x_q = y_i, y_q
    res = np.zeros((n, M), result_dtype)
    nres = np.zeros(n, np.int32)
    for s in range(n):
        cat = [np.concatenate([r[j] for r in rows[s]]) for j in range(3)]
        o = oracle.spots(*cat, max_msgs=M, min_score=cfg["min_score"])
        res[s], nres[s] = o["results"], o["n"]
        assert [sr.message_key(m) for m in o["msgs"]] == logs[s]
    return first_rows, res, nres


def pass1_counts(R, cfg):
    return np.array([len(sr.accept((R["cand"][s, :nc], R["ok"][s, :nc], R["msg"][s, :nc]), [], cfg["max_messages"], cfg["min_score"]))
                     for s, nc in enumerate(R["ncand"])])


def check_pass1(ctx, n, R):
    got = pass1_rows(ctx, n)
    assert np.array_equal(got["ncand"], R["ncand"])
    for s in range(n):
        nc = int(R["ncand"][s])
        assert got["cand"][s] == R["cand"][s, :nc].tobytes() and got["ok"][s] == R["ok"][s, :nc].tobytes(), s
        assert got["status"][s] == R["status"][s, :nc].tobytes() and got["msg"][s] == R["msg"][s, :nc].tobytes(), s


def check_records(got, want, what):
    (res, nres), (wres, wnres) = got, want
    assert np.array_equal(nres, wnres), (what, nres, wnres)
    for s in range(len(nres)):
        assert res[s].tobytes() == wres[s].tobytes(), (what, s)


def new_stats():
    keys = ("appended_in_pass2", "appended_in_pass3", "crosses_start", "crosses_end", "cross_pass_duplicates", "non_cq_subtracted",
            "idle_at_pass2", "idle_at_pass3", "m8_full_after_pass1", "m8_fills_in_pass2", "runs")
    return {k: 0 for k in keys}


def tally(stats):
    for k, v in stats.items():
        STATS[k] = STATS.get(k, 0) + v


@pytest.mark.parametrize("osd", [0, 2])
@pytest.mark.parametrize("config", list(CONFIGS))
def test_process_conditioned_and_slots_compose(pkg, oracle, slots, config, osd):
    """process_conditioned (with the slots' peak) and process_slots (conditioned slots, no peak) at passes 2 and 3 equal the
    composition of their stages: pass-1 rows byte for byte, and the records with their counts and the gaps non-CQ messages leave."""
    d_i, d_q, peak, c_i, c_q = slots
    n = d_i.shape[0]
    cfg = cfg_of(config)
    st = new_stats()
    ref = pkg.Context(0, **cfg)
    ref.set_osd(osd, -1)
    for passes in (2, 3):
        for entry, (x_i, x_q, pk) in (("conditioned", (d_i, d_q, peak)), ("slots", (c_i, c_q, None))):
            ctx = pkg.Context(0, **cfg)
            ctx.set_osd(osd, -1)
            ctx.set_passes(passes)
            if pk is None:
                ctx.process_slots(x_i, x_q)
            else:
                ctx.process_conditioned(x_i, x_q, pk)
            got = ctx.fetch_results(n)
            R1, wres, wnres = compose(ref, oracle, x_i, x_q, pk, passes, osd, cfg, st)
            check_pass1(ctx, n, R1)
            ctx.close()
            check_records(got, (wres, wnres), (config, osd, passes, entry))
            st["runs"] += 1
    ref.close()
    tally(st)


def workspace_slots(ctx, n):
    w = ctx.workspace_ptrs()
    g = lambda key, shape, t: torch.as_tensor(_Arr(w[key], shape, t), device=DEV).clone()
    return g("i", (n, sr.SLOT), "<f4"), g("q", (n, sr.SLOT), "<f4"), g("peak", (n,), "<f4")


@pytest.mark.parametrize("osd", [0, 2])
def test_raw_entries_compose(pkg, oracle, raw, osd):
    """process_raw on 8 raw slots in 4 overlap groups (the later passes run on slot offsets s0 != 0), process_raw_streams with 2
    slots a stream, and a pipe (depth 2, no partition and 40 back-end SMs) over two batches: each equals the composition on the
    decimated slots and peaks it read back, and the pipe equals the context."""
    n = raw.shape[0]
    cfg = cfg_of("default")
    st = new_stats()
    ref = pkg.Context(0)
    ref.set_osd(osd, -1)
    group0_first = later_groups_gain = 0
    for passes in (2, 3):
        ctx = pkg.Context(0)
        ctx.set_osd(osd, -1)
        ctx.set_passes(passes)
        ctx.set_overlap(4)
        ctx.process_raw(raw, n, stride=raw.stride(0))
        got = ctx.fetch_results(n)
        x_i, x_q, pk = workspace_slots(ctx, n)
        R1, wres, wnres = compose(ref, oracle, x_i, x_q, pk, passes, osd, cfg, st)
        check_pass1(ctx, n, R1)
        check_records(got, (wres, wnres), ("process_raw overlap", osd, passes))
        n1 = pass1_counts(R1, cfg)
        group0_first += int(n1[:2].sum())                  # the first group's log is not empty ...
        later_groups_gain += int((wnres[2:] > n1[2:]).sum())   # ... and groups at s0 != 0 append in later passes
        st["runs"] += 1
        ctx.set_overlap(0)
        ctx.process_raw_streams(raw, n // 2, 2, stride=2 * raw.stride(0))
        got = ctx.fetch_results(n)
        x_i, x_q, pk = workspace_slots(ctx, n)
        R1, wres, wnres = compose(ref, oracle, x_i, x_q, pk, passes, osd, cfg, st)
        check_pass1(ctx, n, R1)
        check_records(got, (wres, wnres), ("process_raw_streams", osd, passes))
        st["runs"] += 1
        ctx.close()
    ref.close()
    # the pipe: per batch the records of process_raw on the same slots (which the overlap run above pins to the composition)
    ctx = pkg.Context(0)
    ctx.set_osd(osd, -1)
    ctx.set_passes(3)
    want = []
    for b in range(2):
        ctx.process_raw(raw[4 * b:4 * b + 4], 4, stride=raw.stride(0))
        want.append(ctx.fetch_results(4))
    ctx.set_overlap(4)
    ctx.process_raw(raw, n, stride=raw.stride(0))
    whole = ctx.fetch_results(n)
    ctx.close()
    check_records(whole, (np.concatenate([w[0] for w in want]), np.concatenate([w[1] for w in want])), ("batch invariance", osd))
    for back in (0, 40):
        p = pkg.Pipe(0, depth=2)
        if back:
            p.set_partition(back)
        p.set_osd(osd, -1)
        p.set_passes(3)
        for b in range(2):
            p.submit(raw[4 * b:4 * b + 4], 4, stride=raw.stride(0))
        got = [p.collect(4) for _ in range(2)]
        p.close()
        for b in range(2):
            check_records(got[b], want[b], ("pipe", back, b))
    assert group0_first > 0 and later_groups_gain > 0, (group0_first, later_groups_gain)
    tally(st)


def test_edge_centred_bp_composes(pkg, oracle, slots):
    """The same composition at passes = 3 under the edge-centred BP kernel (process-wide, restored afterwards)."""
    d_i, d_q, peak, _, _ = slots
    n = d_i.shape[0]
    cfg = cfg_of("default")
    st = new_stats()
    pkg.set_decode_variant(1)
    try:
        ctx, ref = pkg.Context(0), pkg.Context(0)
        ctx.set_passes(3)
        ctx.process_conditioned(d_i, d_q, peak)
        got = ctx.fetch_results(n)
        R1, wres, wnres = compose(ref, oracle, d_i, d_q, peak, 3, 0, cfg, st)
        check_pass1(ctx, n, R1)
        check_records(got, (wres, wnres), "edge-centred")
        ctx.close()
        ref.close()
    finally:
        pkg.set_decode_variant(0)
    st["runs"] += 1
    tally(st)


def test_the_matrix_reaches_every_case():
    """Summed over the runs above: records appended in pass 2 and in pass 3, subtracted spans over each slot edge, a cross-pass
    duplicate, a non-CQ message subtracted, idle slots at pass 2 and 3, and the 8-message table full after pass 1 in some slot
    and filling during pass 2 in another."""
    if STATS.get("runs", 0) < len(CONFIGS) * 2 * 4 + 2 * 4 + 1:
        pytest.skip("runs only after the whole matrix of this module")
    for k, v in STATS.items():
        assert v > 0, (k, STATS)
