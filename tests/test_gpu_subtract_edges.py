"""ft8b200_subtract (csrc/subtract.cu) against the float64 definition (tests/subtract_ref.py) where the kernels clip, clamp and loop:
spans hanging over either end of the slot or lying wholly outside it, the ends of the band, full message lists, list counts from
outside the library, batches larger than the persistent grids, and unaligned float views.  Candidates are made by hand (the
nominal position nearest the synthesised start and frequency, which puts the truth within +-128 samples and +-1.5625 Hz, inside
the grid's reach), so that a span can be put anywhere; signals are device-synthesised GFSK, noiseless and with noise 0.05."""
import ctypes as C

import numpy as np
import pytest

import subtract_ref as sr
from oracle.pyoracle import cand_dtype
from ref64 import bits_from_tones

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
DEV = torch.device("cuda:0")
EINVAL = -2

START_EDGE = [-40148, -30000, -5888, -600, -1, 100]       # 300 in-slot samples ... sync's earliest ... the coarse grid reaches before 0
END_EDGE = [7452, 7553, 12288, 20000, 47700]              # the grid reaches past the end ... first crossing ... sync's latest ... 300 in slot
IN_SLOT = [1, 511, 1024, 1025, 2047, 2048, 2049, 4097]    # around the 512-sample halo and the 2048-sample chunk of subtract_kernel


def nearest_cand(start, f_hz, score=20):
    """The candidate whose nominal position (subtract_ref.nominal) is nearest a start sample and a tone-0 frequency."""
    c = np.zeros((), cand_dtype)
    m = int(round((start - 256) / 256))
    k = int(round(f_hz / 3.125))
    c["time_offset"], c["time_sub"], c["freq_offset"], c["freq_sub"], c["score"] = m // 2, m % 2, k // 2, k % 2, score
    return c


def t0_of(start):
    """A float32 t0 the synthesiser rounds to `start` samples at 3200 sps."""
    t0 = float(np.float32((start + 0.25) / 3200.0))
    assert int(np.round(np.float64(np.float32(t0)) * 3200.0)) == start
    return t0


class Batch:
    """Slots of hand-placed messages: specs[s] = list of (start sample, f0 Hz, amp); cand / cw / nmsg as ft8b200_subtract takes them."""

    def __init__(self, pkg, ctx, specs, noise, seed, cands=None):
        self.n, self.M = len(specs), ctx.M
        items, first = [], [0]
        for s, sp in enumerate(specs):
            for j, (start, f0, amp) in enumerate(sp):
                items.append((pkg.pack77_std("CQ", f"K{(s * 7 + j) % 10}{chr(65 + s % 26)}{chr(65 + j % 26)}", "FN20"), f0, t0_of(start), amp))
            first.append(len(items))
        sig = pkg.make_signals(items, gfsk=True)
        self.d_i, self.d_q = ctx.synth_slots(sig, np.array(first, np.int32), noise, seed)
        self.cand = np.zeros((self.n, self.M), cand_dtype)
        self.cw = np.zeros((self.n, self.M, 174), np.uint8)
        self.nmsg = np.array([len(sp) for sp in specs], np.int32)
        tones = ctx.encode_tones(np.stack([np.frombuffer(it[0], np.uint8) for it in items])) if items else None
        for s, sp in enumerate(specs):
            for j, (start, f0, _) in enumerate(sp):
                self.cand[s, j] = nearest_cand(start, f0) if cands is None else cands[s][j]
                self.cw[s, j] = bits_from_tones(tones[first[s] + j])
        self.hi, self.hq = self.d_i.cpu().numpy(), self.d_q.cpu().numpy()

    def device(self, order=None):
        cand, cw = self.cand, self.cw
        if order is not None:
            cand, cw = cand[:, order], cw[:, order]
        return (torch.from_numpy(np.ascontiguousarray(cand).view(np.uint8).reshape(self.n, self.M, 8)).to(DEV),
                torch.from_numpy(np.ascontiguousarray(cw)).to(DEV))

    def run(self, ctx, nmsg=None, order=None):
        d_cand, d_cw = self.device(order)
        nm = torch.from_numpy(self.nmsg if nmsg is None else np.asarray(nmsg, np.int32)).to(DEV)
        ri, rq, grid = ctx.subtract(self.d_i, self.d_q, d_cand, d_cw, nm)
        torch.cuda.synchronize()
        return ri.cpu().numpy(), rq.cpu().numpy(), grid.cpu().numpy()

    def x(self, s):
        return self.hi[s].astype(np.float64) + 1j * self.hq[s].astype(np.float64)


def check_metric(x, cand, cw, g):
    """The kernel's grid point g scores within 1e-3 of the float64 best, and is the float64 point wherever the coarse gap is above
    1e-3 and the fine gap above 1e-5 (the bars of test_gpu_subtract.py and their reasons).  -> (pinned, float64 point)."""
    (dt, df), (coarse, fine) = sr.refine(x, cand, cw, with_metrics=True)
    cs, fs_ = np.sort(coarse.ravel()), np.sort(fine)
    pinned = (cs[-1] - cs[-2]) > 1e-3 * cs[-1] and (fs_[-1] - fs_[-2]) > 1e-5 * fs_[-1]
    if pinned:
        assert tuple(g) == (dt, df), (tuple(g), dt, df)
    s0, f0 = sr.nominal(cand)
    r = sr.reference(sr.tones_from_codeword(cw), f0 + g[1] * sr.DF_STEP)
    assert sr.metric(x, s0 + g[0], r) >= (1 - 1e-3) * fs_[-1]
    return pinned, (dt, df)


def check_residual(b, s, ri, rq, grid, order=None):
    """The residual against subtract_ref.subtract with the kernel's grid, to 1e-4 of the slot's peak."""
    js = list(range(int(b.nmsg[s]))) if order is None else list(order[:int(b.nmsg[s])])
    msgs = [(b.cand[s, j], b.cw[s, j]) for j in js]
    y, _ = sr.subtract(b.x(s), msgs, grids=[tuple(grid[s, k]) for k in range(len(js))])
    peak = max(np.abs(b.hi[s]).max(), np.abs(b.hq[s]).max(), 1e-30)
    err = max(np.abs(ri[s] - y.real).max(), np.abs(rq[s] - y.imag).max())
    assert err <= 1e-4 * peak, (s, err / peak)
    return err / peak


@pytest.mark.parametrize("noise", [0.0, 0.05])
def test_spans_across_the_slot_edges(pkg, noise):
    """One message a slot, its true start at or near either slot edge: the refinement's zero fill and the subtraction's clipped
    span, chunk placement and window normaliser against the float64 definition.  On the noiseless slots whose tone-0 frequency is on
    the grid the refined start is the synthesised one wherever float64 refinement finds it (it moves a start by one sample when that
    makes the in-slot part whole symbols)."""
    rng = np.random.default_rng(21)
    starts = START_EDGE + END_EDGE + [L - sr.SPAN for L in IN_SLOT] + [sr.SLOT - L for L in IN_SLOT]
    specs = []
    for st in starts:
        f_nom = sr.nominal(nearest_cand(st, float(rng.uniform(200, 1400))))[1]
        specs.append([(st, f_nom + sr.DF_STEP * int(rng.integers(-7, 8)), 1.0)])   # on the df grid of its own candidate
    ctx = pkg.Context(0)
    b = Batch(pkg, ctx, specs, noise, 5)
    ri, rq, grid = b.run(ctx)
    ctx.close()
    pinned, crossing, lengths = 0, 0, []
    for s, [(st, f, _)] in enumerate(specs):
        p, _ = check_metric(b.x(s), b.cand[s, 0], b.cw[s, 0], grid[s, 0])
        pinned += p
        check_residual(b, s, ri, rq, grid)
        S = sr.nominal(b.cand[s, 0])[0] + int(grid[s, 0, 0])
        lo = min(max(S, 0), sr.SLOT)
        hi = max(min(S + sr.SPAN, sr.SLOT), lo)
        assert np.array_equal(ri[s, :lo], b.hi[s, :lo]) and np.array_equal(ri[s, hi:], b.hi[s, hi:]), s   # outside the span: untouched
        assert np.array_equal(rq[s, :lo], b.hq[s, :lo]) and np.array_equal(rq[s, hi:], b.hq[s, hi:]), s
        crossing += S < 0 or S + sr.SPAN > sr.SLOT
        lengths.append(hi - lo)
        if noise == 0.0 and p:
            true_len = min(st + sr.SPAN, sr.SLOT) - max(st, 0)
            if st in START_EDGE[1:] + END_EDGE[:-1]:
                assert S == st, (st, S)
            elif true_len >= 511:
                assert abs(S - st) <= 1, (st, S)
    assert pinned >= len(specs) // 2 and crossing >= len(specs) - 4, (pinned, crossing)
    # clipped spans shorter than the window, and spans clipped in the middle of a symbol (the normaliser's edge cases)
    assert any(0 < n < 1025 for n in lengths) and any(0 < n < sr.SPAN and n % 512 for n in lengths), lengths


@pytest.mark.parametrize("noise", [0.0, 0.05])
def test_spans_outside_the_slot_and_band_ends(pkg, noise):
    """A candidate whose every grid point lies wholly before or after the slot leaves the residual equal to the input byte for byte,
    with the grid at (-136, -8): the tie rule on all-zero metrics, which subtract_ref.refine gives too.  At the band's ends the grid
    reaches negative frequencies (freq_offset 0) and 1598 Hz (freq_offset 248, freq_sub 1); both against the float64 definition."""
    ctx = pkg.Context(0)
    outside = [nearest_cand(-40704, 700.0), nearest_cand(48384, 900.0), nearest_cand(-80000, 500.0), nearest_cand(60000, 300.0)]
    for c in outside:
        assert sr.nominal(c)[0] + 136 + sr.SPAN <= 0 or sr.nominal(c)[0] - 136 >= sr.SLOT
    specs = [[(4000, 700.0, 1.0), (5000, 900.0, 0.5)], [(4000, 3.125 / 16, 1.0)], [(3000, 1553.125 + 8 * sr.DF_STEP, 1.0)],
             [(2000, 1.5625, 0.8), (3100, 1553.125 - 3 * sr.DF_STEP, 0.6)]]
    cands = [outside[:2], [nearest_cand(4000, 0.0)], [nearest_cand(3000, 1553.125)], [nearest_cand(2000, 0.0), nearest_cand(3100, 1553.125)]]
    assert (cands[2][0]["freq_offset"], cands[2][0]["freq_sub"]) == (248, 1) and cands[1][0]["freq_offset"] == 0
    b = Batch(pkg, ctx, specs, noise, 9, cands=cands)
    b.cand[0, 2:4] = outside[2:]   # four messages in slot 0, none of them in it
    b.cw[0, 2:4] = b.cw[0, :2]
    b.nmsg[0] = 4
    ri, rq, grid = b.run(ctx)
    ctx.close()
    assert np.array_equal(ri[0], b.hi[0]) and np.array_equal(rq[0], b.hq[0])
    for j in range(4):
        assert tuple(grid[0, j]) == (-136, -8) == sr.refine(b.x(0), b.cand[0, j], b.cw[0, j]), j
    for s in (1, 2, 3):
        for j in range(int(b.nmsg[s])):
            check_metric(b.x(s), b.cand[s, j], b.cw[s, j], grid[s, j])
        check_residual(b, s, ri, rq, grid)


def crowded_specs(rng, n_slots, n_msgs, edge_share=0.25):
    specs = []
    for _ in range(n_slots):
        sp = []
        for _ in range(n_msgs):
            u = rng.random()
            st = int(rng.integers(-2560, -320)) if u < edge_share / 2 else int(rng.integers(7680, 10240)) if u < edge_share else int(rng.integers(640, 2560))
            sp.append((st, float(rng.uniform(100, 1500)), float(rng.uniform(0.3, 1.0))))
        specs.append(sp)
    return specs


def test_full_lists_clamps_and_order(pkg):
    """Two slots of exactly M = 50 crowded messages (some over the slot edges) against subtract_ref.subtract with the kernel's grid;
    the metric bar on 12 of each slot's messages (float64 refinement is the slow part).  A count above M gives the bytes of M, counts
    of -1 and 0 leave the input as it is, and the same messages in reverse order match the definition in that order."""
    rng = np.random.default_rng(33)
    ctx = pkg.Context(0)
    M = ctx.M
    specs = crowded_specs(rng, 2, M)
    b = Batch(pkg, ctx, specs, 0.05, 17)
    ri, rq, grid = b.run(ctx)
    for s in range(2):
        check_residual(b, s, ri, rq, grid)
        for j in rng.choice(M, 12, replace=False):
            check_metric(b.x(s), b.cand[s, j], b.cw[s, j], grid[s, j])
    over = b.run(ctx, nmsg=[M + 5, M + 5])
    assert all(np.array_equal(a, c) for a, c in zip(over, (ri, rq, grid)))
    for cnt in (-1, 0):
        ni, nq, ng = b.run(ctx, nmsg=[cnt, cnt])
        assert np.array_equal(ni, b.hi) and np.array_equal(nq, b.hq) and not ng.any()
    rev = np.arange(M)[::-1]
    vi, vq, vg = b.run(ctx, order=rev)
    ctx.close()
    assert np.array_equal(vg, grid[:, rev])   # every message refines on the input alone
    for s in range(2):
        check_residual(b, s, vi, vq, vg, order=rev)
    assert not np.array_equal(vi, ri)   # the order does matter to the bytes


def test_batches_beyond_the_persistent_grids(pkg):
    """2 x SMs + 5 slots of 1-3 messages: refine_kernel's item loop (grid 4 x SMs) and subtract_kernel's slot loop (grid SMs, one
    scratch row per CTA reused across slots) both run more than once a CTA.  Every slot's residual and grid equal a single-slot
    call and an in-place call byte for byte; 12 slots, the first and the last among them, against the float64 definition."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = 2 * sms + 5
    rng = np.random.default_rng(44)
    specs = [crowded_specs(rng, 1, int(rng.integers(1, 4)), edge_share=0.5)[0] for _ in range(n)]
    ctx = pkg.Context(0)
    assert n * ctx.M > 4 * sms
    b = Batch(pkg, ctx, specs, 0.05, 23)
    ri, rq, grid = b.run(ctx)
    d_cand, d_cw = b.device()
    d_n = torch.from_numpy(b.nmsg).to(DEV)
    for s in range(n):
        a_i, a_q, a_g = ctx.subtract(b.d_i[s:s + 1], b.d_q[s:s + 1], d_cand[s:s + 1], d_cw[s:s + 1], d_n[s:s + 1])
        torch.cuda.synchronize()
        assert np.array_equal(a_i.cpu().numpy()[0], ri[s]) and np.array_equal(a_q.cpu().numpy()[0], rq[s]), s
        assert np.array_equal(a_g.cpu().numpy()[0], grid[s]), s
    xi, xq = b.d_i.clone(), b.d_q.clone()
    _, _, g2 = ctx.subtract(xi, xq, d_cand, d_cw, d_n, out=(xi, xq))
    torch.cuda.synchronize()
    ctx.close()
    assert np.array_equal(xi.cpu().numpy(), ri) and np.array_equal(xq.cpu().numpy(), rq) and np.array_equal(g2.cpu().numpy(), grid)
    for s in sorted({0, n - 1} | set(rng.choice(np.arange(1, n - 1), 10, replace=False).tolist())):
        for j in range(int(b.nmsg[s])):
            check_metric(b.x(s), b.cand[s, j], b.cw[s, j], grid[s, j])
        check_residual(b, s, ri, rq, grid)


def test_unaligned_views_and_refusals(pkg):
    """Views one float off a 16-byte boundary (rows still 48 000 floats apart) give the aligned call's bytes.  A pointer 2 bytes
    off, n_slots of 0 or 65 536, and null buffers are refused with FT8B200_EINVAL and a reason, and nothing is written."""
    rng = np.random.default_rng(55)
    ctx = pkg.Context(0)
    b = Batch(pkg, ctx, crowded_specs(rng, 3, 3, edge_share=0.5), 0.05, 29)
    ri, rq, grid = b.run(ctx)
    d_cand, d_cw = b.device()
    d_n = torch.from_numpy(b.nmsg).to(DEV)
    N = 3 * sr.SLOT

    def off_view(src):
        buf = torch.zeros(N + 1, dtype=torch.float32, device=DEV)
        v = buf[1:].view(3, sr.SLOT)
        if src is not None:
            v.copy_(src)
        assert v.data_ptr() % 16 == 4
        return v
    oi, oq, yi, yq = off_view(b.d_i), off_view(b.d_q), off_view(None), off_view(None)
    _, _, g = ctx.subtract(oi, oq, d_cand, d_cw, d_n, out=(yi, yq))
    torch.cuda.synchronize()
    assert np.array_equal(yi.cpu().numpy(), ri) and np.array_equal(yq.cpu().numpy(), rq) and np.array_equal(g.cpu().numpy(), grid)

    L, h = ctx.L, C.c_void_p(ctx.h)
    s = torch.cuda.current_stream().cuda_stream
    st = C.c_void_p(s if s else 1)
    raw = torch.zeros(N * 4 + 64, dtype=torch.uint8, device=DEV)
    mis = C.c_void_p(raw.data_ptr() + 2)
    out_i = torch.full((3, sr.SLOT), 7.0, dtype=torch.float32, device=DEV)
    out_q = torch.full((3, sr.SLOT), 7.0, dtype=torch.float32, device=DEV)
    out_g = torch.full((3, ctx.M, 2), 123, dtype=torch.int32, device=DEV)
    P = lambda t: C.c_void_p(t.data_ptr())
    good = dict(i=P(b.d_i), q=P(b.d_q), n=3, cand=P(d_cand), cw=P(d_cw), nmsg=P(d_n), ri=P(out_i), rq=P(out_q), grid=P(out_g))
    cases = [("i", mis, "aligned"), ("q", mis, "aligned"), ("ri", mis, "aligned"), ("rq", mis, "aligned"), ("n", 0, "n_slots"),
             ("n", 65536, "n_slots")] + [(k, C.c_void_p(0), "null") for k in ("i", "q", "cand", "cw", "nmsg", "ri", "rq", "grid")]
    for key, val, why in cases:
        a = dict(good, **{key: val})
        rc = L.ft8b200_subtract(h, a["i"], a["q"], a["n"], a["cand"], a["cw"], a["nmsg"], a["ri"], a["rq"], a["grid"], st)
        assert rc == EINVAL and why in pkg.lib().ft8b200_last_error().decode(), (key, rc)
    torch.cuda.synchronize()
    assert bool((out_i == 7.0).all()) and bool((out_q == 7.0).all()) and bool((out_g == 123).all()) and not raw.any()
    ctx.close()
