"""GPU parity tests: the CUDA library, called through its C ABI, against the CPU oracle.

Bar (north star): decoded NIDs / TSBK / LC / voice frames and their sample indices bit-exact;
FEC decoders bit-exact; discriminator / boxcar samples within 1e-4 absolute of the oracle
(full scale is +-4.8, so 2e-5 of full scale)."""
import numpy as np
import p25_spec as S
import pytest
from tools import p25tx as tx
from util import check_against_truth, events_key, oracle_events

pytestmark = pytest.mark.gpu
BB_TOL = 1e-4


@pytest.fixture(scope="module")
def p25():
    import p25rx_b200
    return p25rx_b200


def _streams_baseband(kind: str, n: int, length: int | None = None):
    rows, truth = [], []
    for s in range(n):
        st = tx.control_channel(100 + s, 3, lead_idle=20 + 7 * s) if kind == "control" else tx.traffic_channel(200 + s, 1, lead_idle=20 + 5 * s)
        bb, _ = tx.baseband_48k(st.dibits, snr_db=22 if s % 2 else None, dc=0.01 * (s % 3), seed=s, timing_offset=(s * 1.7) % 10)
        rows.append(bb)
        truth.append(tx.expected_events(st))
    length = length or min(len(r) for r in rows)
    return np.stack([r[:length] for r in rows]), truth


# ------------------------------------------------------------------ FEC decoders
def test_fec_decoders_bit_exact(p25, oracle):
    import ctypes as C
    O = oracle.lib()
    ctx = p25.Context(1, max_chunk_samples=1024)
    rng = np.random.default_rng(0)
    n = 20000
    # BCH: codewords with 0..15 errors plus random words
    words = np.zeros(n, dtype=np.uint64)
    for i in range(n):
        w = S.bch_encode(int(rng.integers(0, 65536)))
        for p in rng.choice(63, int(rng.integers(0, 16)), replace=False):
            w ^= 1 << int(p)
        words[i] = w if i % 5 else int(rng.integers(0, 1 << 63))
    for gk in (0, 12):    # per-thread decoder, then the warp-cooperative form the walker uses
        data, nerr = ctx.fec_selftest(gk, words)
        for i in range(0, n, 7):
            od, on = C.c_uint16(), C.c_int()
            ok = O.p25o_bch_decode(int(words[i]), C.byref(od), C.byref(on))
            assert (nerr[i] >= 0) == bool(ok), (gk, i)
            if ok:
                assert nerr[i] == on.value and data[i] == od.value, (gk, i)
    # short codes: random words (every syndrome class is exercised)
    for kind, name, bits in ((1, "golay23", 23), (2, "golay24", 24), (3, "golay18", 18), (4, "hamming15", 15),
                             (5, "hamming10", 10), (6, "cyclic16", 16)):
        w = rng.integers(0, 1 << bits, n).astype(np.uint32)
        data, nerr = ctx.fec_selftest(kind, w)
        fo = getattr(O, f"p25o_{name}_decode")
        for i in range(0, n, 5):
            a = C.c_uint32()
            assert fo(int(w[i]), C.byref(a)) == nerr[i] and a.value == data[i], (name, i)
    # Reed-Solomon
    for (nn, kk) in (S.RS_SHORT, S.RS_MED, S.RS_LONG):
        t = (nn - kk) // 2
        blocks = np.zeros((4000, nn), dtype=np.uint8)
        for i in range(len(blocks)):
            cw = S.rs_encode([int(x) for x in rng.integers(0, 64, kk)], nn, kk)
            for p in rng.choice(nn, int(rng.integers(0, t + 3)), replace=False):
                cw[int(p)] ^= int(rng.integers(1, 64))
            blocks[i] = cw if i % 4 else rng.integers(0, 64, nn)
        ref = blocks.copy()
        got = [ctx.fec_selftest(gk, blocks.copy(), nn, kk) for gk in (7, 10)]
        for i in range(len(ref)):
            r = O.p25o_rs_decode(ref[i].ctypes.data_as(C.c_void_p), nn, kk)
            for fixed, nerr in got:
                assert r == nerr[i] and (ref[i] == fixed.reshape(-1, nn)[i]).all(), (nn, kk, i)
    # trellis + IMBE
    blocks = np.zeros((4000, 98), dtype=np.uint8)
    for i in range(len(blocks)):
        d = S.tsbk_block_dibits(rng.integers(0, 256, 12).astype(np.uint8).tobytes()).copy()
        for p in rng.choice(196, int(rng.integers(0, 20)), replace=False):
            d[int(p) // 2] ^= 2 >> (int(p) & 1)
        blocks[i] = d if i % 5 else rng.integers(0, 4, 98)
    got = [ctx.fec_selftest(gk, blocks) for gk in (8, 13)]
    for i in range(len(blocks)):
        o = np.zeros(12, np.uint8)
        r = O.p25o_trellis_half_decode(blocks[i].ctypes.data_as(C.c_void_p), o.ctypes.data_as(C.c_void_p))
        for out, nerr in got:
            assert r == nerr[i] and (r < 0 or (o == out[i]).all()), i
    blocks = np.zeros((4000, 72), dtype=np.uint8)
    for i in range(len(blocks)):
        d = S.imbe_encode([int(rng.integers(0, 1 << b)) for b in S.IMBE_U_BITS]).copy()
        for p in rng.choice(144, int(rng.integers(0, 14)), replace=False):
            d[int(p) // 2] ^= 2 >> (int(p) & 1)
        blocks[i] = d
    got = [ctx.fec_selftest(gk, blocks)[0] for gk in (9, 11)]
    for i in range(len(blocks)):
        c, e = np.zeros(8, np.uint32), np.zeros(7, np.uint32)
        O.p25o_imbe_decode(blocks[i].ctypes.data_as(C.c_void_p), c.ctypes.data_as(C.c_void_p), e.ctypes.data_as(C.c_void_p))
        for out in got:
            assert (out[i, :8] == c).all() and (out[i, 8:] == e).all(), i
    ctx.close()


# ------------------------------------------------------------------ decode (Surface 2)
@pytest.mark.parametrize("kind", ["control", "traffic"])
@pytest.mark.parametrize("chunk", [None, 3277, 8192, 1000])
def test_decode_bit_exact(p25, oracle, kind, chunk):
    bb, truth = _streams_baseband(kind, 9)
    ref, ref_stats = oracle_events(oracle, bb)
    ctx = p25.Context(len(bb), max_chunk_samples=1024, max_baseband=bb.shape[1])
    rx = p25.MessageReceiver(ctx)
    if chunk is None:
        ev = rx.feed(bb)
    else:
        ev = np.concatenate([rx.feed(bb[:, i:i + chunk]) for i in range(0, bb.shape[1], chunk)])
        ev = ev[np.lexsort((ev["sample"], ev["stream"]))]
    assert events_key(ev) == events_key(ref)
    for s in range(len(bb)):
        assert (ctx.stats(s) == ref_stats[s]).all(), s
    check_against_truth(ev, truth[0][: np.count_nonzero(ev["stream"] == 0)], 0)
    ctx.close()


def test_decode_noise_and_garbage(p25, oracle):
    """Low SNR, noise-only and constant streams: whatever the oracle decides, the GPU decides."""
    rng = np.random.default_rng(3)
    rows = []
    for s in range(12):
        st = tx.traffic_channel(300 + s, 1) if s % 2 else tx.control_channel(300 + s, 4)
        bb, _ = tx.baseband_48k(st.dibits, snr_db=[4, 6, 8, 10, 12, 15][s % 6], seed=s, dc=0.02)
        rows.append(bb)
    n = min(len(r) for r in rows)
    rows = [r[:n] for r in rows]
    rows.append(rng.normal(0, 0.6, n).astype(np.float32))
    rows.append(np.zeros(n, dtype=np.float32))
    rows.append(np.full(n, 0.3, dtype=np.float32))
    bb = np.stack(rows)
    ref, ref_stats = oracle_events(oracle, bb)
    ctx = p25.Context(len(bb), max_chunk_samples=1024, max_baseband=bb.shape[1])
    ev = p25.MessageReceiver(ctx).feed(bb)
    assert events_key(ev) == events_key(ref)
    assert np.count_nonzero(ev["kind"] == 0) > 0          # the error paths were exercised
    for s in range(len(bb)):
        assert (ctx.stats(s) == ref_stats[s]).all()
    ctx.close()


def test_resync_and_stats_clear(p25, oracle):
    bb, _ = _streams_baseband("control", 3)
    cut = 2000
    ctx = p25.Context(3, max_chunk_samples=1024, max_baseband=bb.shape[1])
    rx = p25.MessageReceiver(ctx)
    ev1 = rx.feed(bb[:, :cut])
    rx.resync(1)
    ev2 = rx.feed(bb[:, cut:])
    ref = []
    for s in range(3):
        o = oracle.MessageReceiver(stream=s)
        ref.append(o.feed(bb[s, :cut]))
        if s == 1:
            o.resync()
        ref.append(o.feed(bb[s, cut:]))
    ref = np.concatenate(ref)
    got = np.concatenate([ev1, ev2])
    got = got[np.lexsort((got["sample"], got["stream"]))]
    ref = ref[np.lexsort((ref["sample"], ref["stream"]))]
    assert events_key(got) == events_key(ref)
    assert ctx.stats(0, clear=True)[0, 0] > 0 and ctx.stats(0)[:, [0, 1, 3]].sum() == 0
    ctx.close()


# ------------------------------------------------------------------ demod (Surface 1)
@pytest.mark.parametrize("fmt,dec", [("cf32", 5), ("u8", 5), ("cf32", 50), ("u8", 50)])
@pytest.mark.parametrize("chunk", [16384, 30000, 4999])
def test_demod_within_tolerance(p25, oracle, fmt, dec, chunk):
    fs = 240_000 * (dec // 5)
    S_ = 5
    rows = []
    for s in range(S_):
        st = tx.control_channel(400 + s, 2)
        rows.append(tx.modulate_iq(st.dibits, fs, snr_db=25, cfo_hz=50.0 * s, seed=s)[: 4 * chunk + 123])
    n = min(len(r) for r in rows)
    iq = np.stack([r[:n] for r in rows])
    if fmt == "u8":
        data = np.stack([tx.iq_to_u8(r) for r in iq])
        ofmt, gfmt = oracle.FMT_U8, p25.FMT_U8_IQ
    else:
        data, ofmt, gfmt = iq, oracle.FMT_CF32, p25.FMT_CF32_IQ
    ctx = p25.Context(S_, fmt=gfmt, decimation=dec, max_chunk_samples=chunk)
    chains = [oracle.DemodChain(ofmt, dec == 50) for _ in range(S_)]
    per = 2 if fmt == "u8" else 1
    worst = 0.0
    for i in range(0, n, chunk):
        m = min(chunk, n - i)
        part = np.ascontiguousarray(data[:, per * i: per * (i + m)])
        bb, n_out, pw = ctx.demod(part, m, want_power=True)
        for s in range(S_):
            ref, pref = chains[s].feed(part[s], want_power=True)
            assert len(ref) == n_out
            if n_out:
                worst = max(worst, float(np.max(np.abs(bb[s] - ref))))
                assert abs(pw[s] - pref) < 1e-2
    assert worst < BB_TOL, worst
    ctx.close()


def test_demod_odd_chunks_and_device_input(p25, oracle):
    """Odd chunk lengths force the unaligned load path; a torch CUDA tensor is used without a host copy."""
    import torch
    st = tx.control_channel(500, 3)
    iq = tx.modulate_iq(st.dibits, 240_000, snr_db=25, seed=1)[:40001]
    assert len(iq) == 40001
    ctx = p25.Context(2, fmt=p25.FMT_CF32_IQ, decimation=5, max_chunk_samples=20000)
    chains = [oracle.DemodChain(oracle.FMT_CF32, False) for _ in range(2)]
    pos = 0
    for m in (777, 12345, 20000, 6879):
        part = np.ascontiguousarray(np.stack([iq[pos:pos + m], iq[pos:pos + m][::-1]]))
        dev = torch.from_numpy(part.view(np.float32)).cuda()
        torch.cuda.synchronize()      # the library reads the buffer on its own stream
        bb, n_out, _ = ctx.demod(dev, m)
        for s in range(2):
            ref = chains[s].feed(part[s])
            assert len(ref) == n_out and np.max(np.abs(bb[s] - ref)) < BB_TOL
        pos += m
    ctx.close()


# ------------------------------------------------------------------ end to end (the hot path)
@pytest.mark.parametrize("fmt,dec", [("cf32", 50), ("u8", 5), ("cf32", 5)])
def test_process_iq_to_events(p25, oracle, fmt, dec):
    fs = 240_000 * (dec // 5)
    S_ = 6
    rows, truth = [], []
    for s in range(S_):
        st = tx.control_channel(600 + s, 3) if s % 2 == 0 else tx.traffic_channel(600 + s, 1)
        rows.append(tx.modulate_iq(st.dibits[: 2200], fs, snr_db=20, cfo_hz=-120.0 + 60 * s, timing_offset=1.3 * s, seed=s))
        truth.append(tx.expected_events(st))
    n = min(len(r) for r in rows)
    iq = np.stack([r[:n] for r in rows])
    if fmt == "u8":
        data = np.stack([tx.iq_to_u8(r) for r in iq])
        ofmt, gfmt = oracle.FMT_U8, p25.FMT_U8_IQ
    else:
        data, ofmt, gfmt = iq, oracle.FMT_CF32, p25.FMT_CF32_IQ
    chunk = 16384 * (dec // 5)
    ctx = p25.Context(S_, fmt=gfmt, decimation=dec, max_chunk_samples=chunk)
    per = 2 if fmt == "u8" else 1
    got = []
    for i in range(0, n, chunk):
        m = min(chunk, n - i)
        ctx.process(np.ascontiguousarray(data[:, per * i: per * (i + m)]), m)
        got.append(ctx.poll())
    got = np.concatenate(got)
    got = got[np.lexsort((got["sample"], got["stream"]))]
    ref = []
    for s in range(S_):
        bb = oracle.DemodChain(ofmt, dec == 50).feed(data[s])
        ref.append(oracle.MessageReceiver(stream=s).feed(bb))
    ref = np.concatenate(ref)
    assert events_key(got) == events_key(ref)
    assert len(got) > 40
    ctx.close()


def test_golden_fixtures(p25):
    """Committed fixtures (tests/golden/make_golden.py): input baseband -> expected events."""
    import os
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "decode_golden.npz"))
    bb, exp = g["baseband"].astype(np.float32), g["events"]
    ctx = p25.Context(bb.shape[0], max_chunk_samples=1024, max_baseband=bb.shape[1])
    ev = p25.MessageReceiver(ctx).feed(bb)
    assert events_key(ev) == events_key(exp.view(p25.EVENT_DTYPE).reshape(-1))
    ctx.close()
    # demod fixture: u8 IQ in the reference's chunking -> baseband and power (generic kernel, then the /5 fast kernel)
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "demod_golden.npz"))
    iq, exp, pw = g["iq_u8"], g["baseband"], g["power_dbm"]
    ctx = p25.Context(1, fmt=p25.FMT_U8_IQ, decimation=5, max_chunk_samples=16384)
    got, gpw = [], []
    for a, b in ((0, 16384), (16384, 32768), (32768, 40_000)):
        bb, _, p = ctx.demod(np.ascontiguousarray(iq[None, 2 * a: 2 * b]), b - a, want_power=True)
        got.append(bb[0])
        gpw.append(p[0])
    assert np.max(np.abs(np.concatenate(got) - exp)) < BB_TOL and np.max(np.abs(np.array(gpw) - pw)) < 1e-2
    ctx.close()
    # channelizer fixture: capture -> spectra of the last 8 output times, 96 channels
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "pfb_golden.npz"))
    cap = g["capture"]
    ctx = p25.Context(1536, fmt=p25.FMT_CF32_IQ, decimation=400, max_chunk_samples=len(cap))
    ctx.keep_spectra(True)
    ctx.demod(np.ascontiguousarray(cap[None, :]), len(cap), want_baseband=False)
    y = ctx.channelizer_output()[0]
    got = y[g["rows"]][:, g["channels"]]
    assert np.max(np.abs(got - g["spectra"])) < 2e-5 * np.max(np.abs(g["spectra"]))
    ctx.close()


def test_full_size_properties(p25):
    """BASELINE configs[1] scale (1,024 streams): every stream is a circular shift of one of 8 seeds,
    so decoded payload multisets must be identical across the streams that share a seed."""
    base = []
    for s in range(8):
        st = tx.control_channel(700 + s, 6, lead_idle=30)
        base.append(tx.baseband_48k(st.dibits, snr_db=20, seed=s)[0][:22000])
    S_ = 1024
    bb = np.stack([np.roll(base[s % 8], 360 * 10 * (s // 8 % 4)) for s in range(S_)])
    ctx = p25.Context(S_, max_chunk_samples=1024, max_baseband=bb.shape[1])
    ev = p25.MessageReceiver(ctx).feed(bb)
    assert (np.diff(ev["stream"].astype(np.int64)) >= 0).all()
    per = {}
    for s in range(S_):
        e = ev[ev["stream"] == s]
        assert (np.diff(e["sample"].astype(np.int64)) > 0).all()
        key = sorted(bytes(x["payload"][:12]) for x in e[e["kind"] == 7])
        per.setdefault((s % 8, s // 8 % 4), key)
        assert key == per[(s % 8, s // 8 % 4)]
        assert len(key) >= 12
    ctx.close()


# ------------------------------------------------------------------ BASELINE.json configs[3]: voice at low SNR with CFO
def _voice_streams(n_streams: int, pairs: int):
    """SURVEY.md section 8d cfg4: HDU, alternating LDU1/LDU2, TDULC; SNR swept over {6, 8, 10, 12, 15} dB."""
    return [tx.traffic_channel(4000 + s, pairs) for s in range(n_streams)], [6, 8, 10, 12, 15]


def test_cfg4_voice_low_snr_decode_bit_exact(p25, oracle):
    """256 traffic-channel streams at 6..15 dB: every Golay / Hamming / RS / cyclic path runs with real errors
    and failures; events, payloads (IMBE u0..u7 + error counts, LC, ES, LSD, HDU) and all stats are bit-exact."""
    S_ = 256
    streams, snrs = _voice_streams(S_, 2)
    rows = [tx.baseband_48k(st.dibits, snr_db=snrs[s % 5], seed=s, dc=0.01 * ((s % 7) - 3), timing_offset=0.37 * (s % 10))[0]
            for s, st in enumerate(streams)]
    n = min(len(r) for r in rows)
    bb = np.stack([r[:n] for r in rows])
    ref, ref_stats = oracle_events(oracle, bb)
    ctx = p25.Context(S_, max_chunk_samples=1024, max_baseband=8192)
    rx = p25.MessageReceiver(ctx)
    ev = np.concatenate([rx.feed(bb[:, i:i + 8192]) for i in range(0, n, 8192)])   # the replay block size (src/replay.rs:27)
    ev = ev[np.lexsort((ev["sample"], ev["stream"]))]
    assert events_key(ev) == events_key(ref)
    got_stats = np.stack([ctx.stats(s) for s in range(S_)])
    assert (got_stats == np.stack(ref_stats)).all()
    kinds = np.bincount(ev["kind"], minlength=9)
    assert kinds[p25.EV_VOICE_FRAME] > 30 * S_ and kinds[p25.EV_ERROR] > 0 and kinds[p25.EV_LINK_CONTROL] > 0
    fam = got_stats.sum(axis=0)                  # every voice-path code family saw words and corrected bits
    for f in ("golayStd", "golayExt", "golayShort", "hammingStd", "hammingShort", "rsShort", "rsMed", "rsLong", "cyclic", "bch"):
        i = p25.STATS_FAMILIES.index(f)
        assert fam[i, 0] > 0 and fam[i, 3] > 0, f
    ctx.close()


def test_cfg4_voice_iq_cfo_end_to_end(p25, oracle):
    """The same signals as 240 kS/s u8 IQ with +-300 Hz carrier offset through the whole path (ddc_fm /5 fast kernel +
    walker) against the oracle chain.  The front ends agree to ~1e-6, so slicer decisions can differ only on samples
    that sit within that distance of a threshold: the event lists must agree except for a stated, tiny fraction."""
    S_ = 40
    streams, snrs = _voice_streams(S_, 1)
    rng = np.random.default_rng(44)
    rows = [tx.iq_to_u8(tx.modulate_iq(st.dibits, 240_000, snr_db=snrs[s % 5] + 6.0, cfo_hz=float(rng.uniform(-300, 300)), seed=s))
            for s, st in enumerate(streams)]
    n = min(len(r) for r in rows) // 2 // 16384 * 16384
    data = np.stack([r[: 2 * n] for r in rows])
    ctx = p25.Context(S_, fmt=p25.FMT_U8_IQ, decimation=5, max_chunk_samples=16384)
    got = []
    for i in range(0, n, 16384):                                        # the reference's SDR chunk (src/consts.rs:6)
        ctx.process(np.ascontiguousarray(data[:, 2 * i: 2 * (i + 16384)]), 16384)
        got.append(ctx.poll())
    got = np.concatenate(got)
    got = got[np.lexsort((got["sample"], got["stream"]))]
    ref = []
    for s in range(S_):
        bb = oracle.DemodChain(oracle.FMT_U8, False).feed(data[s])
        ref.append(oracle.MessageReceiver(stream=s).feed(bb))
    ref = np.concatenate(ref)
    a, b = set(events_key(got)), set(events_key(ref))
    diff = len(a ^ b)
    assert len(ref) > 25 * S_
    assert diff <= max(2, len(ref) // 500), f"{diff} of {len(ref)} events differ"
    ctx.close()


# ------------------------------------------------------------------ BASELINE.json configs[2]: wideband channelizer
def test_channelizer_spectra_baseband_and_events(p25, oracle):
    """19.2 MS/s capture -> 1,536 channels (pfb.cu) against oracle/pfb_oracle.py + the reference's 48 kHz chain:
    channel spectra and occupied-channel baseband within the FP32 tolerance, decoded events identical, carried state
    across unequal chunks."""
    from oracle import pfb_oracle as pfb
    occupied = {3: 0.05, 100: 0.04, 767: 0.05, 768: 0.03, 1000: 0.05, 1535: 0.04}
    chans = {k: (tx.control_channel(800 + k, 2, lead_idle=20 + k % 30).dibits, amp, 40.0 * ((k % 5) - 2))
             for k, amp in occupied.items()}
    n_out_total = 2 * 3600 + 700
    n = n_out_total * 400
    cap = tx.wideband_capture(chans, n, noise_db=-55.0, seed=3)
    ref_y = pfb.channelize(cap)                                   # [n_out][1536] complex128
    ref_c = pfb.channel_filter(ref_y)                             # what the kernels deliver: the channel filter is folded in
    ctx = p25.Context(1536, fmt=p25.FMT_CF32_IQ, decimation=400, max_chunk_samples=1_600_000, event_slots=64)
    ctx.keep_spectra(True)
    got_y, got_bb, pos = [], [], 0
    for m in (1_000_000, 1_555_556, n - 2_555_556):               # unequal, not multiples of 400
        bb, n_out, _ = ctx.demod(np.ascontiguousarray(cap[None, pos:pos + m]), m)
        got_y.append(ctx.channelizer_output()[0])
        got_bb.append(bb)
        ctx.decode()
        pos += m
    ev = ctx.poll()
    got_y = np.concatenate(got_y)
    got_bb = np.concatenate(got_bb, axis=1)
    assert got_y.shape == ref_c.shape == (n_out_total, 1536)
    scale = np.max(np.abs(ref_c))
    assert np.max(np.abs(got_y - ref_c)) < 2e-5 * scale, np.max(np.abs(got_y - ref_c)) / scale
    oracle.lib().p25o_set_always_correlate(0)
    ref_ev = []
    for k in range(1536):
        chain = oracle.DemodChain(oracle.FMT_CF32, 2)
        rbb = chain.feed(ref_y[:, k].astype(np.complex64))
        ref_ev.append(oracle.MessageReceiver(stream=k).feed(rbb))
        if k in occupied:     # carrier present from sample ~0 on: the discriminator is well conditioned
            assert np.max(np.abs(got_bb[k, 200:] - rbb[200:])) < BB_TOL, k
    ref_ev = np.concatenate(ref_ev)
    ev = ev[np.lexsort((ev["sample"], ev["stream"]))]
    assert events_key(ev) == events_key(ref_ev)
    # noise-only channels yield false syncs (errors, the odd NID that random bits happen to BCH-decode to) identically
    # in both; trunking payloads come from the occupied channels only
    good = ev[ev["kind"] == p25.EV_TSBK]
    assert sorted(set(int(s) for s in good["stream"])) == sorted(occupied)
    assert np.count_nonzero(ev["kind"] == p25.EV_TSBK) == 6 * len(occupied)
    ctx.close()


# ------------------------------------------------------------------ the reference's own driver shapes (host mirrors)
def test_replay_receiver_reads_baseband_files_like_replay_rs(p25, oracle, tmp_path):
    """src/replay.rs:26-57: f32le 48 kHz files read in 32,768-byte blocks, VoiceFrames handed to the audio sink,
    stats merged.  Three recordings replayed at once against the oracle fed the same files."""
    from p25rx_b200 import consumers as co
    files = []
    for s in range(3):
        st = tx.traffic_channel(900 + s, 2) if s != 1 else tx.control_channel(900 + s, 5)
        bb, _ = tx.baseband_48k(st.dibits, snr_db=14, seed=s)
        path = tmp_path / f"rec{s}.f32"
        with open(path, "wb") as f:
            co.write_baseband(f, bb[:18000 + 1111 * s])      # unequal lengths: replay ends with the shortest recording
        files.append(path)
    voice = []
    rr = p25.ReplayReceiver(n_streams=3, on_voice_frame=lambda e: voice.append((int(e["stream"]), int(e["sample"]))))
    handles = [open(pth, "rb") for pth in files]
    got = rr.replay(handles)
    got = got[np.lexsort((got["sample"], got["stream"]))]
    ref = []
    for s, pth in enumerate(files):
        o = oracle.MessageReceiver(stream=s)
        with open(pth, "rb") as f:
            data = np.concatenate(list(co.read_baseband_blocks(f)))[:18000]
        ref.append(o.feed(data))
    ref = np.concatenate(ref)
    ref = ref[np.lexsort((ref["sample"], ref["stream"]))]
    assert events_key(got) == events_key(ref)
    assert len(voice) == np.count_nonzero(ref["kind"] == p25.EV_VOICE_FRAME) > 10
    rr.ctx.close()


def test_demod_task_reports_power_every_fourth_chunk(p25, oracle):
    """src/demod.rs:62-119 with the SDR's 32,768-byte chunks (src/consts.rs:6): baseband every chunk, signal power on
    every 4th (Throttler::new(4), src/demod.rs:67, :95-101), equal to the oracle's power_dbm (src/demod.rs:123-134)."""
    st = tx.control_channel(77, 9)
    raw = tx.iq_to_u8(tx.modulate_iq(st.dibits, 240_000, snr_db=25, seed=2, amplitude=0.3))
    n_chunks = len(raw) // 32768
    assert n_chunks >= 9
    ctx = p25.Context(2, fmt=p25.FMT_U8_IQ, decimation=5, max_chunk_samples=16384)
    task = p25.DemodTask(ctx)
    chain = oracle.DemodChain(oracle.FMT_U8, False)
    lens = []
    for i in range(9):
        chunk = raw[i * 32768:(i + 1) * 32768]
        bb, pw = task.run_chunk(np.stack([chunk, chunk]))
        ref, pref = chain.feed(chunk, want_power=True)
        lens.append(bb.shape[1])
        assert bb.shape[1] == len(ref) and np.max(np.abs(bb[0] - ref)) < BB_TOL and np.array_equal(bb[0], bb[1])
        assert (pw is not None) == (i % 4 == 0)
        if pw is not None:
            assert abs(pw[0] - pref) < 1e-2 and abs(pw[0] - (30 + 10 * np.log10(0.09))) < 1.0
    assert set(lens) == {3276, 3277} and sum(lens) == 9 * 16384 // 5      # phase carried across chunks (SURVEY 8a a2)
    ctx.close()


# ------------------------------------------------------------------ error behaviour of the boundary (SURVEY 8b: codes, never abort)
def test_abi_error_codes_and_edge_sizes(p25, oracle):
    ctx = p25.Context(2, fmt=p25.FMT_CF32_IQ, decimation=5, max_chunk_samples=4096, event_slots=4)
    with pytest.raises(p25.P25Error) as e:                      # chunk larger than configured
        ctx.demod(np.zeros((2, 5000), dtype=np.complex64), 5000)
    assert e.value.status == -1 and "max_chunk_samples" in str(e.value)
    with pytest.raises(p25.P25Error) as e:                      # decode(NULL) with nothing demodulated
        ctx.decode()
    assert e.value.status == -3
    with pytest.raises(p25.P25Error) as e:
        ctx.resync(7)                                           # no such stream
    assert e.value.status == -1
    # empty and tiny chunks are legal and keep the decimator phase
    bb, n_out, _ = ctx.demod(np.zeros((2, 0), dtype=np.complex64), 0)
    assert n_out == 0 and bb.shape == (2, 0)
    total = 0
    for m in (3, 1, 4, 2, 7):
        bb, n_out, _ = ctx.demod(np.zeros((2, m), dtype=np.complex64), m)
        total += n_out
    assert total == 17 // 5
    ctx.decode()
    assert len(ctx.poll()) == 0
    # more events than slots: the surplus is dropped and reported, the context stays usable
    st = tx.control_channel(5, 6)
    bb, _ = tx.baseband_48k(st.dibits, snr_db=20, seed=1)
    ctx2 = p25.Context(1, max_chunk_samples=1024, max_baseband=len(bb), event_slots=4)
    ctx2.decode(bb[None, :])
    with pytest.raises(p25.P25Error) as e:
        ctx2.poll()
    assert e.value.status == -4
    ctx2.decode(bb[None, :2000])
    assert len(ctx2.poll()) <= 4
    with pytest.raises(p25.P25Error):
        p25.Context(1000, fmt=p25.FMT_CF32_IQ, decimation=400, max_chunk_samples=4000)   # not a multiple of 1536 channels
    with pytest.raises(p25.P25Error):
        p25.Context(4, decimation=7)
    ctx.close()
    ctx2.close()


# ------------------------------------------------------------------ BASELINE.json configs[4] at full size
def test_cfg5_full_size_properties(p25):
    """65,536 streams of u8 IQ at 240 kS/s (the reference's own format) through the whole path in two chunks, at the
    size the oracle cannot follow: size-independent properties instead.  Every stream is a circular shift of one of
    16 phase-continuous transmissions, so (a) the events arrive ordered by (stream, sample), (b) every decoded TSBK
    passes its CRC, (c) streams that share a transmission decode the same multiset of TSBKs whatever their shift,
    (d) per-stream Viterbi word counts equal the TSBK events + errors, and (e) a second context fed the same input in
    one chunk instead of two yields the identical event list (chunking invariance, generic + fast kernels mixed)."""
    import torch
    from tools.shape_bench import base_streams, tile_on_device
    from p25rx_b200 import consumers as co
    S_, n_base = 65536, 16
    base = base_streams("control", 240_000, n_base, 20.0)                    # [16][36000] complex64, periodic
    n = base.shape[1]
    b8 = np.stack([tx.iq_to_u8(b).reshape(n, 2) for b in base])
    one = tile_on_device(torch.from_numpy(b8).cuda(), S_)                     # [S][n][2] u8
    dev = torch.cat([one, one[:, : n // 2]], dim=1).contiguous()              # 1.5 periods per stream
    total = dev.shape[1]
    cut = 22_016                                                             # multiple of 8: aligned fast path for chunk 2
    ctx = p25.Context(S_, fmt=p25.FMT_U8_IQ, decimation=5, max_chunk_samples=total, event_slots=64)
    part1, part2 = dev[:, :cut].contiguous(), dev[:, cut:].contiguous()
    torch.cuda.synchronize()          # the library works on its own stream: the caller's producers must be done (C ABI contract)
    ctx.process(part1, cut)
    ev1 = ctx.poll()
    ctx.process(part2, total - cut)
    ev = np.concatenate([ev1, ctx.poll()])
    ev = ev[np.lexsort((ev["sample"], ev["stream"]))]
    tsbk = ev[ev["kind"] == p25.EV_TSBK]
    assert len(tsbk) >= 6 * S_                                               # at least two whole TSDUs per stream
    pl = tsbk["payload"][:, :12].astype(np.uint32)
    # (b) CRC of every TSBK, vectorised: recompute over the first 10 bytes
    crc = np.zeros(len(pl), dtype=np.uint32)
    for i in range(10):
        crc ^= pl[:, i] << 8
        for _ in range(8):
            crc = np.where(crc & 0x8000, ((crc << 1) ^ 0x1021) & 0xFFFF, (crc << 1) & 0xFFFF)
    good = (crc ^ 0xFFFF) == (pl[:, 10] << 8 | pl[:, 11])
    # the streams of one transmission share its noise, so a block the noise corrupts fails in all 4,096 of them:
    # bound the failures per transmission instead of overall
    assert good.mean() > 0.98, good.mean()
    # (c) the set of distinct CRC-valid TSBKs of a stream depends only on its transmission
    key = (pl[:, :8] * (np.arange(1, 9, dtype=np.uint32) * 2654435761 % 1000003)).sum(axis=1) % (1 << 31)
    streams = tsbk["stream"].astype(np.int64)
    for b in range(n_base):
        m = ((streams % n_base) == b) & good
        uniq = np.unique(np.stack([streams[m], key[m].astype(np.int64)], axis=1), axis=0)
        counts = np.bincount((uniq[:, 0] // n_base).astype(np.int64), minlength=S_ // n_base)
        assert counts.min() == counts.max() >= 5, (b, counts.min(), counts.max())    # 2 TSDUs x 3 distinct blocks
        ref_set = set(uniq[uniq[:, 0] == uniq[0, 0], 1].tolist())
        assert set(uniq[:, 1].tolist()) == ref_set
    # (d) stats of a few streams
    for s in (0, 1, 4097, 65535):
        st = ctx.stats(s)
        e = ev[ev["stream"] == s]
        vit = p25.STATS_FAMILIES.index("viterbiDibit")
        assert st[vit, 0] == np.count_nonzero(e["kind"] == p25.EV_TSBK) + np.count_nonzero(
            (e["kind"] == p25.EV_ERROR) & (e["payload"][:, 0] == 3))
    ctx.close()
    # (e) chunking invariance on a slice of the streams
    sub = dev[:4096].contiguous()
    torch.cuda.synchronize()
    c1 = p25.Context(4096, fmt=p25.FMT_U8_IQ, decimation=5, max_chunk_samples=total, event_slots=64)
    c1.process(sub, total)
    one_shot = c1.poll()
    c1.close()
    two = ev[ev["stream"] < 4096]
    assert events_key(one_shot) == events_key(two)
    assert co.TsbkFields(bytes(tsbk[good]["payload"][0][:12])).crc_valid()


def test_demod_weak_and_strong_u8_signals(p25, oracle):
    """The /5 u8 kernel works in byte units centred on 128 and restores the 0.5-LSB offset as a constant after the
    filters: check the tolerance where that matters most -- a carrier of only +-4 LSB -- and near full scale."""
    st = tx.control_channel(321, 3)
    S_ = 4
    amps = [0.03, 0.06, 0.5, 0.95]
    rows = [tx.iq_to_u8(tx.modulate_iq(st.dibits, 240_000, snr_db=25, cfo_hz=200.0 * (s - 1.5), seed=s, amplitude=a))
            for s, a in enumerate(amps)]
    n = min(len(r) for r in rows) // 2 // 8 * 8
    data = np.stack([r[: 2 * n] for r in rows])
    ctx = p25.Context(S_, fmt=p25.FMT_U8_IQ, decimation=5, max_chunk_samples=n)
    cut = 16384
    got, pws = [], []
    for a, b in ((0, cut), (cut, n)):                              # generic kernel, then the warp kernel
        bb, _, pw = ctx.demod(np.ascontiguousarray(data[:, 2 * a: 2 * b]), b - a, want_power=True)
        got.append(bb)
        pws.append(pw)
    got = np.concatenate(got, axis=1)
    for s in range(S_):
        chain = oracle.DemodChain(oracle.FMT_U8, False)
        r1, p1 = chain.feed(data[s, : 2 * cut], want_power=True)
        r2, p2 = chain.feed(data[s, 2 * cut:], want_power=True)
        ref = np.concatenate([r1, r2])
        assert np.max(np.abs(got[s] - ref)) < BB_TOL, (amps[s], float(np.max(np.abs(got[s] - ref))))
        assert abs(pws[0][s] - p1) < 1e-2 and abs(pws[1][s] - p2) < 1e-2
    ctx.close()


def test_replay_tool_prints_consumer_view(p25, tmp_path):
    """tools/p25replay.py: the `p25rx -r FILE` shape as a command, JSON lines with the fields the consumers read."""
    import json
    import os
    import subprocess
    import sys
    from p25rx_b200 import consumers as co
    st = tx.control_channel(55, 3)
    bb, _ = tx.baseband_48k(st.dibits, snr_db=22, seed=3)
    f32 = tmp_path / "cc.f32"
    with open(f32, "wb") as f:
        co.write_baseband(f, bb)
    raw = tx.iq_to_u8(tx.modulate_iq(st.dibits, 240_000, snr_db=25, seed=4, amplitude=0.4))
    u8 = tmp_path / "cc.u8"
    raw[: 32768 * (len(raw) // 32768)].tofile(u8)
    tool = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "p25replay.py")
    for argv, n_tsbk in (([str(f32)], 9), (["--iq", str(u8)], 6)):
        r = subprocess.run([sys.executable, tool] + argv, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-1500:]
        lines = [json.loads(x) for x in r.stdout.splitlines()]
        tsbk = [x for x in lines if x["event"] == "TrunkingControl"]
        assert len(tsbk) >= n_tsbk and all(x["crc_valid"] and x["mfg"] == 0 for x in tsbk)
        assert [x for x in lines if x["event"] == "PacketNID"][0]["nac"] == 0x293
        stats = [x for x in lines if x["event"] == "stats"][0]["stats"]
        assert stats["viterbiDibit"]["totalWords"] == len(tsbk) and stats["bch"]["totalWords"] >= 2
        if "--iq" in argv:
            assert any(x["event"] == "sigPower" for x in lines)
