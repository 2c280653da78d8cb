"""Pins the CPU restatement (oracle/ft8_oracle*.c) against the UNMODIFIED reference compiled from its sources
(oracle/_ref/libref_*.so, `make -C oracle ref`).  Skipped where the reference build is absent (the committed golden
fixtures in tests/golden/ cover that case: tests/test_oracle_golden.py)."""
import numpy as np
import pytest

from conftest import bits_equal, golden
from oracle.pyoracle import Reference, ReferenceMonitor, cand_dtype
from tools import ft8enc, synth

needs_reference = pytest.mark.skipif(not (Reference.available("k120") and Reference.available("k500") and ReferenceMonitor.available()),
                                     reason="oracle/_ref not built (make -C oracle ref needs the reference's sources)")


@needs_reference
def test_reference_selftest_runs():
    """decoderSelfTest() (rtlsdr_ft8d.c:913-972): the reference decodes its own 'CQ K1JT FN20QI' signal."""
    assert Reference("k120").lib.ref_selftest() == 1


@needs_reference
def test_decimator_streaming_vs_rtlsdr_callback(oracle):
    ref = Reference("k120", fresh=True)
    rng = np.random.default_rng(3)
    iq = rng.integers(0, 256, size=65536 * 40, dtype=np.uint8)
    iq[::977] = 0
    iq[5::1201] = 255
    st = oracle.new_decim()
    outs = []
    sizes = [65536] * 20 + [8, 16, 751 * 8, 65536 - 8 - 16 - 751 * 8] + [65536] * 19
    o = 0
    for s in sizes:
        chunk = iq[o:o + s]; o += s
        ref.callback(chunk)
        outs.append(oracle.decim_feed(st, chunk, 100))
    i_s = np.concatenate([x[0] for x in outs]); q_s = np.concatenate([x[1] for x in outs])
    ri, rq, n = ref.rx()
    assert n == i_s.size == 1745
    assert bits_equal(ri[:n], i_s) and bits_equal(rq[:n], q_s)


@needs_reference
def test_buffer_stops_at_48000_but_filter_keeps_running(oracle):
    """rtlsdr_ft8d.c:196-200: outputs beyond 48000 are dropped; after the flip the state continues."""
    ref = Reference("k120", fresh=True)
    rng = np.random.default_rng(4)
    n_bytes = 2 * 751 * 48100
    n_bytes -= n_bytes % 65536
    iq = rng.integers(96, 160, size=n_bytes + 65536 * 4, dtype=np.uint8)
    st = oracle.new_decim()
    got_i = []
    for o in range(0, n_bytes, 65536):
        ref.callback(iq[o:o + 65536])
        got_i.append(oracle.decim_feed(st, iq[o:o + 65536], 64)[0])
    got_i = np.concatenate(got_i)
    ri, rq, n = ref.rx()
    assert n == 48000 and got_i.size > 48000
    assert bits_equal(ri, got_i[:48000])
    ref.flip()
    more = []
    for o in range(n_bytes, iq.size, 65536):
        ref.callback(iq[o:o + 65536])
        more.append(oracle.decim_feed(st, iq[o:o + 65536], 64)[0])
    more = np.concatenate(more)
    ri, rq, n = ref.rx()
    assert n == more.size and bits_equal(ri[:n], more)


@needs_reference
@pytest.mark.parametrize("variant,n_sig,seed", [("k120", 1, 7), ("k120", 25, 5), ("k500", 60, 99), ("k120", 60, 1234), ("k120", 0, 11)])
def test_subsystem_all_taps(oracle, variant, n_sig, seed):
    ref = Reference(variant)
    if n_sig == 1:
        i_s, q_s = synth.slot_f32([(ft8enc.tones(ft8enc.pack_std("CQ", "K1JT", "FN20")), 700.0, 0.5, -10.0)], seed)
    elif n_sig == 0:
        i_s, q_s = synth.slot_f32([], seed)
    else:
        i_s, q_s, _ = synth.crowded_band(ft8enc, n_sig, seed)
    i_s, q_s, _ = oracle.condition(i_s, q_s, 48000)
    r = ref.subsystem(i_s, q_s)
    o = oracle.subsystem(i_s, q_s, max_cand=ref.kmax, max_msgs=ref.mmax)
    assert np.array_equal(o["wf"], r["wf"])
    assert np.array_equal(o["cands"], r["cands"].view(cand_dtype))
    assert o["n"] == r["n"] and o["results"].tobytes() == r["results"].tobytes()
    for k, c in enumerate(r["cands"]):
        d = oracle.decode(r["wf"], c)
        assert d["ok"] == r["dec_ok"][k]
        assert bits_equal(d["llr"], r["llr"][k]) and np.array_equal(d["plain"], r["plain"][k])
        assert d["status"].tobytes() == r["dec_status"][k].tobytes()
        assert d["msg"].tobytes() == r["dec_msg"][k].tobytes()


@needs_reference
def test_find_sync_on_random_waterfalls(oracle):
    """Heap eviction and tie-breaking paths: random bytes make thousands of positions pass min_score."""
    ref = Reference("k120")
    rng = np.random.default_rng(3)
    for lo, hi, k, ms in [(0, 256, 120, 10), (60, 90, 120, 10), (0, 256, 7, 0), (100, 110, 500, 1)]:
        mag = rng.integers(lo, hi, size=94208, dtype=np.uint8)
        assert np.array_equal(oracle.find_sync(mag, k, ms), ref.find_sync(mag, k, ms).view(cand_dtype))


@needs_reference
def test_bp_decode_fuzz(oracle):
    ref = Reference("k120")
    rng = np.random.default_rng(6)
    for trial in range(60):
        bits = oracle.encode174(bytes(rng.integers(0, 256, 10, dtype=np.uint8)))
        llr = ((bits.astype(np.float32) * 2 - 1) * 4.0 + rng.standard_normal(174).astype(np.float32) * (1.0 + 0.1 * trial)).astype(np.float32)
        for iters in (20, 3):
            po, eo = oracle.bp_decode(llr, iters)
            pr, er = ref.bp_decode(llr, iters)
            assert eo == er and np.array_equal(po, pr)
    for llr in (np.zeros(174, np.float32), np.full(174, -3.0, np.float32), np.full(174, np.nan, np.float32)):
        po, eo = oracle.bp_decode(llr)
        pr, er = ref.bp_decode(llr)
        assert eo == er and np.array_equal(po, pr)


@needs_reference
def test_unpack77_fuzz(oracle):
    """All message types the reference unpacks (0.0 free text, 0.5 telemetry, 1/2 standard, 4 nonstandard) + rejects."""
    ref = Reference("k120")
    rng = np.random.default_rng(7)
    for i3 in range(8):
        for _ in range(400):
            a = bytearray(rng.integers(0, 256, 12, dtype=np.uint8))
            a[9] = (a[9] & 0xC7) | (i3 << 3)
            rc_o, t_o = oracle.unpack77(bytes(a))
            rc_r, t_r = ref.unpack77(bytes(a))
            assert rc_o == rc_r
            if rc_r >= 0:
                assert t_o == t_r, (bytes(a).hex(), t_o, t_r)
    for n28 in list(range(0, 1100)) + [532443, 532444, 2063591, 2063592, 2063592 + 4194303, 2063592 + 4194304]:
        v = (n28 << 1)
        a = bytearray(12)
        a[0] = (v >> 21) & 0xFF; a[1] = (v >> 13) & 0xFF; a[2] = (v >> 5) & 0xFF; a[3] = ((v << 3) & 0xF8) | 0x01
        a[4] = 0x23; a[5] = 0x45; a[9] = 1 << 3
        assert oracle.unpack77(bytes(a)) == ref.unpack77(bytes(a))


@needs_reference
def test_unpack77_stratified_vs_reference(oracle):
    """tools/synth.py::payload_fuzz (the generator the GPU tests use for the device unpacker): every token class, flag, report
    form and reject path -- oracle == reference on 60 000 payloads."""
    ref = Reference("k120")
    payloads, labels = synth.payload_fuzz(20261, 60_000)
    for a, lab in zip(payloads, labels):
        b = bytes(a) + b"\0\0"
        rc_o, t_o = oracle.unpack77(b)
        rc_r, t_r = ref.unpack77(b)
        assert rc_o == rc_r and (rc_r < 0 or t_o == t_r), (lab, b.hex(), rc_o, t_o, rc_r, t_r)


@needs_reference
def test_spots_vs_reference_loop(oracle):
    """The duplicate table / CQ filter restated in orc_spots() against the reference's OWN loop (ft8_subsystem, rtlsdr_ft8d.c:
    1452-1523) fed hand-made candidates and ft8_decode() answers through the scripted taps of oracle/ref_harness.c: 2-token CQ
    ("(null)" locator), "CQ DX ..." tokenisation, %.12s / %.6s truncation, hash clashes with different text, duplicates,
    low-score and failed candidates, a table one short of full; plus 200 random scripts."""
    from test_gpu_messages import spots_cases, _msg
    ref = Reference("k120")
    for name, c, okv, m, max_msgs, defined in spots_cases():
        if not defined:
            continue
        n, res = ref.subsystem_scripted(c, okv, m)
        o = oracle.spots(c, okv, m, max_msgs=max_msgs, min_score=10)
        assert n == o["n"] and res.tobytes() == o["results"].tobytes(), name
    rng = np.random.default_rng(5)
    calls = ["K1JT", "W9XYZ", "PA0ABC", "PJ4/K1ABC", "DX", "TEST", "<...>", "3DA0XYZ/P"]
    for _ in range(200):
        k = int(rng.integers(1, 60))
        c = np.zeros(k, cand_dtype)
        c["score"] = np.sort(rng.integers(5, 40, k))[::-1]
        c["freq_offset"] = rng.integers(0, 249, k); c["freq_sub"] = rng.integers(0, 2, k)
        texts = ["%s %s %s" % (rng.choice(["CQ", "CQ", "QRZ", "K1ABC", "CQ DX"]), rng.choice(calls), rng.choice(["FN20", "RR73", "-15", ""])) for _ in range(k)]
        texts = [t.strip() for t in texts]
        m = np.array([_msg(t, int(rng.integers(0, 60))) for t in texts])   # few hash values: clashes are the rule
        okv = (rng.random(k) < 0.8).astype(np.uint8)
        live = {(t, int(h)) for t, h, o_, s_ in zip(texts, m["hash"], okv, c["score"]) if o_ and s_ >= 10}
        if len(live) >= 50:
            continue   # the reference never returns from a full table
        n, res = ref.subsystem_scripted(c, okv, m)
        o = oracle.spots(c, okv, m)
        assert n == o["n"] and res.tobytes() == o["results"].tobytes(), texts


@needs_reference
def test_gfsk_twin_vs_reference_synth_gfsk(oracle):
    """The synthesiser's GFSK mode (integer pulse table, closed-form phase; oracle/ft8_oracle_synth.c is the bit-identical twin
    of csrc/synth.cu) against ft8_lib's own synth_gfsk() (gen_ft8.c:49-102) at the same sample rate: the quadrature rail of the
    complex 3200 sps waveform is sin(phase), which is what the reference emits -- same smoothed frequency, same extended end
    symbols, same ramps, to within the 4096-entry phase table and the reference's float phase accumulator."""
    from oracle.pyoracle import ReferenceGen, signal_dtype
    if not ReferenceGen.available():
        pytest.skip("oracle/_ref/libref_gen.so not built")
    gen = ReferenceGen()
    for k, msg in enumerate([("CQ", "K1JT", "FN20"), ("K1ABC", "W9XYZ", "RR73")]):
        sig = np.zeros(1, signal_dtype)
        sig[0]["payload"] = np.frombuffer(oracle.pack_std(*msg), np.uint8)
        sig[0]["reserved"][0] = 1
        sig[0]["f0_hz"], sig[0]["t0_sec"], sig[0]["amp"] = 400.0 + 311.0 * k, 0.0, 1.0
        wi, wq = oracle.synth_float(1, False, sig, 0.0, 1, 0, 79 * 512)
        ref = gen.synth_gfsk(oracle.tones(sig[0]["payload"].tobytes()), float(sig[0]["f0_hz"]), 2.0, 0.16, 3200)
        assert ref.size == wq.size == 79 * 512
        err = np.abs(wq.astype(np.float64) - ref.astype(np.float64))
        assert err.max() < 0.02 and np.sqrt((err ** 2).mean()) < 0.005, (err.max(), np.sqrt((err ** 2).mean()))
        assert abs(wi[0]) < 1e-6 and abs(wi[10]) < 0.07          # ramped start: the envelope reaches 1 only after 64 samples (0.059 at sample 10)
        # plain FSK of the same message differs (phase discontinuities in frequency at every symbol boundary)
        sig[0]["reserved"][0] = 0
        _, fq = oracle.synth_float(1, False, sig, 0.0, 1, 0, 79 * 512)
        assert np.abs(fq.astype(np.float64) - ref).max() > 0.5
    # FT4 / 12 kHz: BT = 1, 576 samples per symbol; the real-audio rail is cos(phase): compare instantaneous frequency instead
    p8, p4 = gen.pulse(512, 2.0), gen.pulse(576, 1.0)
    assert abs(float(p8.sum()) - 512.0) < 0.5 and abs(float(p4.sum()) - 576.0) < 0.5   # a pulse integrates to one symbol of deviation


@needs_reference
def test_oracle_pack77_vs_reference(oracle):
    """The restated pack77() (oracle/ft8_oracle_codec.c) against the reference's on 20 000 message texts."""
    ref = Reference("k120")
    for m in synth.pack77_fuzz_messages(29, 20000):
        assert oracle.pack77(m)[0] == ref.pack77(m), repr(m)


@needs_reference
def test_library_pack77_vs_reference(pkg):
    """ft8b200_pack77 (host code of the library) against the reference's own pack77() (pack.c:284-301) on 20 000 message texts:
    standard / free-text choice and every payload byte, quirks included ("FN20QI" packs as FN20, unchecked reports, 3DA0/3X)."""
    ref = Reference("k120")
    n_std = 0
    for m in synth.pack77_fuzz_messages(23, 20000):
        got, kind = pkg.pack77(m)
        assert got == ref.pack77(m), repr(m)
        n_std += kind == 0
    assert 5000 < n_std < 15000


@needs_reference
def test_encoder_and_crc_vs_reference(oracle):
    ref = Reference("k120")
    rng = np.random.default_rng(8)
    for _ in range(200):
        to, de, ex = synth.random_message(rng)
        text = f"{to} {de} {ex}".strip()
        p_ref = ref.pack77(text)
        assert oracle.pack_std(to, de, ex) == p_ref == ft8enc.pack_std(to, de, ex), text
        assert np.array_equal(oracle.tones(p_ref), ref.tones(p_ref)) and np.array_equal(ft8enc.tones(p_ref), ref.tones(p_ref))
        blob = bytes(rng.integers(0, 256, 12, dtype=np.uint8))
        for nbits in (76, 77, 82, 96):
            assert oracle.crc14(blob, nbits) == ref.crc(blob, nbits) == ft8enc.crc14(blob, nbits)
    assert oracle.pack_text("HELLO WORLD") == ref.pack77("HELLO WORLD")


@needs_reference
def test_fft_vs_kiss(oracle):
    mon = ReferenceMonitor()
    rng = np.random.default_rng(9)
    for n in (3840, 1152, 128, 960, 60, 3528, 14112, 154, 442, 202, 98):   # the last six: kf_bfly_generic (radix 7, 11, 13, 17, 101)
        x = rng.standard_normal(n).astype(np.float32)
        assert np.array_equal(oracle.fft_r2c(x).view(np.uint32), mon.fftr(x).view(np.uint32)), n


@needs_reference
def test_monitor_vs_reference(oracle):
    mon = ReferenceMonitor()
    sigs = [(ft8enc.tones(ft8enc.pack_std("CQ", "K1JT", "FN20")), 1200.0, 0.5, 0.1), (ft8enc.tones(ft8enc.pack_std("K1ABC", "W9XYZ", "-15")), 2100.0, 1.1, 0.05)]
    a = synth.audio_12k(sigs, 3)
    mo, io, xo = oracle.monitor_waterfall(a)
    mr, ir, xr = mon.waterfall(a)
    assert np.array_equal(io, ir) and np.array_equal(mo, mr) and np.float32(xo) == np.float32(xr)


def test_log10f_quantiser_is_monotone_over_the_whole_input_range(oracle):
    """The kernels replace log10f by the step thresholds; that is exact iff the host quantiser is monotone.
    Checked exhaustively in C over every float in [1e-12, 1e7] would take ~10 s; here: every float within 64 ulp of
    each threshold plus 2M log-uniform samples, sorted, must quantise to a non-decreasing sequence."""
    thr = oracle.db_thresholds()
    near = []
    for t in thr[1:256]:
        u = np.float32(t).view(np.uint32)
        near.append((np.arange(-64, 65, dtype=np.int64) + int(u)).astype(np.uint32).view(np.float32))
    rng = np.random.default_rng(0)
    xs = np.concatenate(near + [np.exp(rng.uniform(np.log(1e-12), np.log(1e7), 200000)).astype(np.float32)])
    xs.sort()
    q = np.array([oracle.quantize_db(float(x)) for x in xs])
    assert np.all(np.diff(q) >= 0)
    assert np.array_equal(q, np.searchsorted(thr[1:256], xs, side="right"))


def ft4_audio(seed, n=5):
    rng = np.random.default_rng(seed)
    sigs, texts = [], []
    for k in range(n):
        to, de, ex = synth.random_message(rng)
        if k % 2 == 0:
            to = "CQ"
        sigs.append((ft8enc.tones_ft4(ft8enc.pack_std(to, de, ex)), float(rng.uniform(300.0, 2600.0)), float(0.3 + rng.uniform(0.0, 0.9)),
                     float(rng.uniform(0.03, 0.15))))
        texts.append(f"{to} {de} {ex}")
    return synth.audio_12k(sigs, seed, n_samples=90_000, symbol_period=0.048), texts


@needs_reference
def test_ft4_vs_reference(oracle):
    """FT4 through the restatement == the unmodified reference at every tap: encoder tones, the 7.5 s / 576-sample
    monitor waterfall (kiss_fftr 1152), ft4_sync_score + heap order, 87x2 LLRs, LDPC, CRC, descrambling, text."""
    ref = Reference("k120")
    mon = ReferenceMonitor()
    # encoder: Python restatement vs the oracle's C vs (through decode) the reference
    payload = ft8enc.pack_std("CQ", "K1JT", "FN20")
    t4 = np.zeros(105, np.uint8)
    oracle.lib.orc_encode_tones_ft4(payload, t4.ctypes.data_as(__import__("ctypes").c_void_p))
    assert np.array_equal(t4, ft8enc.tones_ft4(payload))
    decoded_any = 0
    for seed in (1, 2):
        audio, texts = ft4_audio(seed)
        mo, io, xo = oracle.monitor_waterfall(audio, protocol=0)
        mr, ir, xr = mon.waterfall(audio, protocol=0)
        assert np.array_equal(io, ir) and np.array_equal(mo, mr) and np.float32(xo) == np.float32(xr)
        assert int(io[0]) == 576 and int(io[2]) == 1152 and int(io[5]) == 288
        dims = dict(num_blocks=int(io[4]), num_bins=int(io[5]), time_osr=2, freq_osr=2, protocol=0)
        for K, ms in ((120, 10), (40, 0)):
            co = oracle.find_sync(mo, K, ms, **dims)
            cr = ref.find_sync(mo, K, ms, **dims)
            assert co.tobytes() == cr.tobytes()
        got = set()
        for c in co[:60]:
            do, dr = oracle.decode(mo, c, 20, **dims), ref.decode(mo, c, 20, **dims)
            assert do["ok"] == dr["ok"]
            assert np.array_equal(do["llr"].view(np.uint32), dr["llr"].view(np.uint32)) and np.array_equal(do["plain"], dr["plain"])
            assert do["status"]["ldpc_errors"] == dr["status"]["ldpc_errors"]
            if do["ok"]:
                assert do["msg"].tobytes() == dr["msg"].tobytes() and do["status"].tobytes() == dr["status"].tobytes()
                got.add(do["msg"]["text"].decode())
        decoded_any += len(got & set(texts))
    assert decoded_any >= 4, "the synthetic FT4 signals must actually decode"


def stored_recordings(tmp_path):
    """tests/golden/recordings_12k.npz -- three of the reference's own real-world recordings and the stdout lines of its
    decode_ft8 on them -- written back as 16-bit mono WAV files: -> [(path, lines)]."""
    import wave
    g = golden("recordings_12k")
    out = []
    for k, (pcm, lines) in enumerate(zip(g["pcm"], g["lines"])):
        path = str(tmp_path / f"rec{k}.wav")
        with wave.open(path, "wb") as w:
            w.setnchannels(1); w.setsampwidth(2); w.setframerate(12000)
            w.writeframes(np.ascontiguousarray(pcm, np.int16).tobytes())
        out.append((path, str(lines).split("\n")))
    return out


@needs_reference
def test_decode_ft8_main_on_the_reference_recordings(oracle, tmp_path):
    """The reference's own main() (`decode_ft8 file.wav`, stdout captured) on the stored real-world recordings == the
    restatement's chain (monitor waterfall -> find_sync -> decode -> unique-message table), line for line: score, time,
    frequency and text of every decode, in order -- and both == the lines stored with the recordings (47 lines)."""
    mon = ReferenceMonitor()
    total = 0
    for p, stored in stored_recordings(tmp_path):
        ref = mon.decode_ft8_stdout(p)
        sig, sr = mon.load_wav(p)
        assert oracle.decode_ft8_lines(sig, sr) == ref == stored, p
        total += len(ref)
    assert total == 47


@needs_reference
def test_file_loaders_vs_reference(pkg, oracle, tmp_path):
    """The library's host-side readers against the reference's readRawIQfile / readC2file / load_wav on the same files
    (the reference normalises on the host; the library returns unscaled samples + peak and scales on the device, so the
    comparison applies decoder()'s scale expression here)."""
    import ctypes as C
    ref = Reference("k120")
    i_s, q_s = synth.slot_f32([(ft8enc.tones(ft8enc.pack_std("CQ", "K1JT", "FN20")), 700.0, 0.5, -3.0)], 5)
    i_s *= 3.7; q_s *= 3.7
    inter = np.empty(2 * 40000, np.float32)
    inter[0::2] = i_s[:40000]; inter[1::2] = -q_s[:40000]
    iq_path, c2_path = str(tmp_path / "a.iq"), str(tmp_path / "b.c2")
    inter.tofile(iq_path)
    with open(c2_path, "wb") as f:
        f.write(b"210101_0000.c2"[:14].ljust(14, b"\0") + np.int32(2).tobytes() + np.float64(14.074).tobytes() + inter.tobytes())
    for path, reader in ((iq_path, "readRawIQfile"), (c2_path, "readC2file")):
        ri = np.zeros(48000, np.float32); rq = np.zeros(48000, np.float32)
        n_ref = getattr(ref.lib, reader)(ri.ctypes.data_as(C.c_void_p), rq.ctypes.data_as(C.c_void_p), path.encode())
        got = pkg.read_iq_file(path) if path.endswith(".iq") else pkg.read_c2_file(path)
        gi, gq, n, peak = got[:4]
        assert n == n_ref == 40000
        scale = np.float32(0.5 / max(np.float64(np.float32(1e-24)), np.float64(peak)))
        assert bits_equal(gi * scale, ri) and bits_equal(gq * scale, rq)
        assert not gi[n:].any() and not gq[n:].any()
    assert pkg.read_c2_file(c2_path)[4:] == (14.074, 2, b"210101_0000.c2")
    assert pkg.read_iq_file(str(tmp_path / "missing.iq"))[2] == 0
    mon = ReferenceMonitor()
    for p, _ in stored_recordings(tmp_path):
        a, sr = pkg.load_wav(p)
        b, sr2 = mon.load_wav(p)
        assert sr == sr2 == 12000 and bits_equal(a, b)
