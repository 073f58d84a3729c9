"""GPU parity tests added in round 2 (VERDICT r1 "Next round" items 1, 2, 3, 6, 8): the CUDA library, through its C ABI,
against (a) the oracle at the geometries bench.py times, on a deterministic sample of streams, (b) decoders that share
neither text nor algorithm with the device code (spec/p25_refdec.py), (c) itself across its two event formats, input
residencies and host threads."""
import ctypes as C
import os
import threading

import numpy as np
import p25_refdec as R
import p25_spec as S
import pytest
from tools import p25tx as tx
from util import events_key, oracle_events

pytestmark = pytest.mark.gpu
BB_TOL = 1e-4


@pytest.fixture(scope="module")
def p25():
    import p25rx_b200
    return p25rx_b200


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


# ------------------------------------------------------------------ FEC: device decoders vs independent decoders
def test_fec_device_vs_independent_decoders(p25, oracle):
    """Every device decoder (per-thread forms and the warp-cooperative forms the walker uses) against spec/p25_refdec.py:
    exhaustive nearest-code-word search, Euclid + Vandermonde Reed-Solomon, numpy dynamic-programme trellis decoding."""
    ctx = p25.Context(1, max_chunk_samples=1024)
    rng = np.random.default_rng(21)
    # BCH(63,16,23)
    words = np.zeros(3000, dtype=np.uint64)
    for i in range(len(words)):
        w = S.bch_encode(int(rng.integers(0, 65536)))
        for p in rng.choice(63, int(rng.integers(0, 16)), replace=False):
            w ^= 1 << int(p)
        words[i] = w if i % 5 else int(rng.integers(0, 1 << 63))
    ref_d, ref_n = R.bch_decode(words)
    for gk in (0, 12):
        d, n = ctx.fec_selftest(gk, words)
        assert (n == ref_n).all(), gk
        assert (d[ref_n >= 0] == ref_d[ref_n >= 0]).all(), gk
    # short binary codes on random words (every coset)
    for kind, name, bits in ((1, "golay23", 23), (2, "golay24", 24), (3, "golay18", 18), (4, "hamming15", 15), (5, "hamming10", 10),
                             (6, "cyclic16", 16)):
        w = rng.integers(0, 1 << bits, 20000).astype(np.uint32)
        d, n = ctx.fec_selftest(kind, w)
        ref_d, ref_n = getattr(R, f"{name}_decode")(w)
        assert (n == ref_n).all(), name
        sel = ref_n >= 0 if name == "golay24" else slice(None)
        assert (d[sel] == ref_d[sel]).all(), name
    # Reed-Solomon
    for (nn, kk) in (S.RS_SHORT, S.RS_MED, S.RS_LONG):
        t = (nn - kk) // 2
        blocks = np.zeros((600, nn), dtype=np.uint8)
        for i in range(len(blocks)):
            cw = S.rs_encode([int(x) for x in rng.integers(0, 64, kk)], nn, kk)
            for p in rng.choice(nn, int(rng.integers(0, t + 3)), replace=False):
                cw[int(p)] ^= int(rng.integers(1, 64))
            blocks[i] = cw if i % 4 else rng.integers(0, 64, nn)
        got = [ctx.fec_selftest(gk, blocks.copy(), nn, kk) for gk in (7, 10)]
        for i in range(len(blocks)):
            ref, rn = R.rs_decode([int(x) for x in blocks[i]], nn, kk)
            for fixed, nerr in got:
                assert nerr[i] == rn and list(fixed.reshape(-1, nn)[i]) == ref, (nn, kk, i)
    # trellis codes: 1/2 rate (kinds 8, 13) and 3/4 rate (kinds 14, 15)
    for enc, nbytes, max_err, kinds, dec in ((S.tsbk_block_dibits, 12, 20, (8, 13), R.trellis_half_decode),
                                             (S.pdu_block34_dibits, 18, 9, (14, 15), R.trellis_34_decode)):
        blocks = np.zeros((3000, 98), dtype=np.uint8)
        for i in range(len(blocks)):
            d = enc(rng.integers(0, 256, nbytes).astype(np.uint8).tobytes()).copy()
            for p in rng.choice(196, int(rng.integers(0, max_err)), replace=False):
                d[int(p) // 2] ^= 2 >> (int(p) & 1)
            blocks[i] = d if i % 5 else rng.integers(0, 4, 98)
        ref, met = dec(blocks)
        assert (met >= 0).sum() > 500 and (met < 0).sum() > 500
        for gk in kinds:
            out, nerr = ctx.fec_selftest(gk, blocks)
            assert (nerr == met).all(), gk
            assert (out[met >= 0] == ref[met >= 0]).all(), gk
    # 3/4 rate also against the oracle's C++ decoder
    O = oracle.lib()
    out, nerr = ctx.fec_selftest(15, blocks)
    for i in range(0, len(blocks), 3):
        o = np.zeros(18, np.uint8)
        r = O.p25o_trellis_34_decode(_p(blocks[i]), _p(o))
        assert r == nerr[i] and (r < 0 or (o == out[i]).all()), i
    # IMBE frames
    blocks = np.zeros((400, 72), dtype=np.uint8)
    for i in range(len(blocks)):
        d = S.imbe_encode([int(rng.integers(0, 1 << b)) for b in S.IMBE_U_BITS]).copy()
        for p in rng.choice(144, int(rng.integers(0, 14)), replace=False):
            d[int(p) // 2] ^= 2 >> (int(p) & 1)
        blocks[i] = d
    got = [ctx.fec_selftest(gk, blocks)[0] for gk in (9, 11)]
    for i in range(len(blocks)):
        u, err = R.imbe_decode(blocks[i])
        for out in got:
            assert list(out[i, :8]) == u and list(out[i, 8:]) == err, i
    ctx.close()


# ------------------------------------------------------------------ a9.9: packet data units, 3/4-rate trellis
def test_pdu_decode_bit_exact(p25, oracle):
    """Packet data traffic at 8..20 dB: PacketNIDs, ViterbiDibit / ViterbiTribit errors, sample indices and every stats
    family equal to the oracle; the viterbiTribit family (src/hub.rs:570) sees words, corrections and failures."""
    S_ = 48
    snrs = [8, 9, 10, 12, 14, 20]
    rows = [tx.baseband_48k(tx.data_channel(5000 + s, 8).dibits, snr_db=snrs[s % 6], seed=s, dc=0.01 * (s % 3),
                            timing_offset=0.4 * (s % 9))[0] for s in range(S_)]
    n = min(len(r) for r in rows)
    bb = np.stack([r[:n] for r in rows])
    ref, ref_stats = oracle_events(oracle, bb)
    ctx = p25.Context(S_, max_chunk_samples=1024, max_baseband=8192)
    rx = p25.MessageReceiver(ctx)
    ev = np.concatenate([rx.feed(bb[:, i:i + 8192]) for i in range(0, n, 8192)])
    ev = ev[np.lexsort((ev["sample"], ev["stream"]))]
    assert events_key(ev) == events_key(ref)
    got_stats = np.stack([ctx.stats(s) for s in range(S_)])
    assert (got_stats == np.stack(ref_stats)).all()
    tri = got_stats[:, p25.STATS_FAMILIES.index("viterbiTribit")].sum(axis=0)
    assert tri[0] > 100 and tri[1] > 0 and tri[3] > 0, tri                 # words, failed words, corrected bits
    codes = ev[ev["kind"] == p25.EV_ERROR]["payload"][:, 0]
    assert (codes == 4).any() and (codes == 3).any()                       # ViterbiTribit and ViterbiDibit errors
    ctx.close()


# ------------------------------------------------------------------ packed, asynchronous event drain
def test_packed_poll_matches_records_and_runs_async(p25, oracle):
    """p25cu_poll_start / p25cu_poll_packed: the variable-length records, unpacked on the host, equal the 80-byte records
    of p25cu_poll; a poll started after chunk k is collected after chunk k+1 was queued; a host buffer too small for the
    drain delivers the rest with the next poll (`more`)."""
    S_ = 24
    rows = []
    for s in range(S_):
        st = tx.traffic_channel(6000 + s, 1) if s % 3 == 0 else tx.control_channel(6000 + s, 5)
        rows.append(tx.baseband_48k(st.dibits, snr_db=12 + s % 9, seed=s)[0])
    n = min(len(r) for r in rows) // 4096 * 4096
    bb = np.stack([r[:n] for r in rows])
    ref, _ = oracle_events(oracle, bb)
    a = p25.Context(S_, max_chunk_samples=1024, max_baseband=4096)
    got, n_bytes = [], 0
    for k, i in enumerate(range(0, n, 4096)):
        a.decode(bb[:, i:i + 4096])
        a.poll_start()                                   # drain of chunk k queued behind its walker
        if k:
            w, ne, more = a.poll_packed()                # collects the drain of chunk k - 1
            assert not more
            got.append(a.unpack(w, ne))
            n_bytes += 4 * len(w)
    w, ne, more = a.poll_packed()
    got.append(a.unpack(w, ne))
    n_bytes += 4 * len(w)
    ev = np.concatenate(got)
    ev = ev[np.lexsort((ev["sample"], ev["stream"]))]
    assert events_key(ev) == events_key(ref)
    assert n_bytes < 0.62 * 80 * len(ref)               # voice frames dominate this mix; control channels pack 3.6x
    with pytest.raises(p25.P25Error) as e:               # the two formats cannot be interleaved mid-drain
        a.poll_start()
        a.poll()
    assert e.value.status == -3
    a.poll_packed()
    a.close()
    # a tiny host buffer: the drain comes in pieces, nothing is lost, per-poll order stays (stream, sample)
    os.environ["P25CU_POLL_RING_WORDS"] = "256"
    try:
        b = p25.Context(S_, max_chunk_samples=1024, max_baseband=n)
        b.decode(bb)
        pieces, rounds = [], 0
        while True:
            w, ne, more = b.poll_packed()
            pieces.append(b.unpack(w, ne))
            rounds += 1
            if not more:
                break
        assert rounds > 3
        for pc in pieces:
            assert (np.diff(pc["stream"].astype(np.int64)) >= 0).all()
        ev = np.concatenate(pieces)
        ev = ev[np.lexsort((ev["sample"], ev["stream"]))]
        assert events_key(ev) == events_key(ref)
        b.close()
    finally:
        del os.environ["P25CU_POLL_RING_WORDS"]


# ------------------------------------------------------------------ host buffers, call-sequence rules
def test_pinned_host_buffers_and_sequence_rules(p25, oracle):
    """p25cu_host_alloc / p25cu_host_register: chunks handed over from pinned memory may be refilled as soon as the call
    returns (double-buffered staging on a copy stream); results equal the oracle's.  demod, demod, decode(NULL) once
    decoding has begun is a call-sequence error instead of a silently skipped chunk."""
    S_, chunk, n_chunks = 6, 16384, 5
    rows = [tx.iq_to_u8(tx.modulate_iq(tx.control_channel(7000 + s, 6).dibits, 240_000, snr_db=20, cfo_hz=30.0 * s, seed=s))
            for s in range(S_)]
    assert min(len(r) for r in rows) >= 2 * chunk * n_chunks
    data = np.stack([r[: 2 * chunk * n_chunks] for r in rows])
    ctx = p25.Context(S_, fmt=p25.FMT_U8_IQ, decimation=5, max_chunk_samples=chunk)
    pinned = ctx.host_alloc((S_, 2 * chunk), np.uint8)
    own = np.zeros((S_, 2 * chunk), dtype=np.uint8)
    ctx.host_register(own)
    got = []
    for c in range(n_chunks):
        buf = pinned if c % 2 == 0 else own
        buf[:] = data[:, 2 * chunk * c: 2 * chunk * (c + 1)]
        ctx.process(buf, chunk)
        buf[:] = 0x55                                   # the call has returned: the buffer is the caller's again
        got.append(ctx.poll())
    got = np.concatenate(got)
    got = got[np.lexsort((got["sample"], got["stream"]))]
    ref = np.concatenate([oracle.MessageReceiver(stream=s).feed(oracle.DemodChain(oracle.FMT_U8, False).feed(data[s])) for s in range(S_)])
    assert events_key(got) == events_key(ref) and len(ref) > 60
    ctx.host_unregister(own)
    ctx.host_free(pinned)
    part = np.ascontiguousarray(data[:, : 2 * chunk])
    ctx.demod(part, chunk, want_baseband=False)
    ctx.demod(part, chunk, want_baseband=False)
    with pytest.raises(p25.P25Error) as e:
        ctx.decode()
    assert e.value.status == -3 and "demodulated chunks" in str(e.value)
    ctx.close()
    demod_only = p25.Context(2, fmt=p25.FMT_U8_IQ, decimation=5, max_chunk_samples=chunk)   # never decodes: no rule applies
    for _ in range(3):
        demod_only.demod(np.ascontiguousarray(data[:2, : 2 * chunk]), chunk)
    demod_only.close()


# ------------------------------------------------------------------ oracle-pinned parity at the benchmarked geometries
def _sampled_compare(p25, oracle, ctx, dev, base, n, fmt_u8, decim, sample, n_steps, n_base=16):
    """Run n_steps x p25cu_process over the device-resident batch; after each step read the sampled streams' baseband
    back; compare baseband and events of the sampled streams with one oracle chain + receiver per stream."""
    import torch
    per = 2 if fmt_u8 else 1
    torch.cuda.synchronize()
    bbs = {s: [] for s in sample}
    evs = []
    n_out = n // decim
    for k in range(n_steps):
        ctx.process(dev, n)
        for s in sample:
            bbs[s].append(ctx.read_baseband(s, n_out))
        e = ctx.poll()
        evs.append(e[np.isin(e["stream"], sample)])
    ev = np.concatenate(evs)
    ev = ev[np.lexsort((ev["sample"], ev["stream"]))]
    worst, ref = 0.0, []
    for s in sample:
        row = np.roll(base[s % n_base], -((s // n_base) * 5003 % n), axis=0)
        row = row.reshape(-1) if fmt_u8 else row.reshape(n, 2).view(np.complex64).reshape(n)
        chain = oracle.DemodChain(oracle.FMT_U8 if fmt_u8 else oracle.FMT_CF32, decim == 50)
        rx = oracle.MessageReceiver(stream=s)
        for k in range(n_steps):
            obb = chain.feed(row)
            assert len(obb) == n_out
            worst = max(worst, float(np.max(np.abs(obb - bbs[s][k]))))
            ref.append(rx.feed(obb))
    ref = np.concatenate(ref)
    assert per and worst < BB_TOL, worst
    a, b = set(events_key(ev)), set(events_key(ref))
    assert len(ref) >= 6 * len(sample) * (n_steps - 1)
    # the two front ends agree to ~1e-6: a slicer decision can differ only on a sample that close to a threshold
    assert len(a ^ b) <= len(ref) // 500, (len(a ^ b), len(ref))
    return worst, len(ref)


def test_cfg2_bench_geometry_sampled_against_oracle(p25, oracle):
    """BASELINE configs[1] exactly as bench.py times it -- 1,024 cf32 streams x 360,000 samples, /50, persistent grid with
    the 7/8 static share and the ticketed remainder -- three consecutive steps; 72 streams (first, last, every kind of
    CTA-boundary straddler in the static part, streams of the ticketed part) sample-for-sample against the oracle."""
    import torch
    from bench import Workload
    from tools.shape_bench import tile_on_device
    wl = Workload("cfg2", 1)
    base = wl.base()                                                         # [16][360000][2] float32
    S_, n = wl.streams, wl.n
    dev = tile_on_device(torch.from_numpy(base).cuda(), S_)
    ctx = p25.Context(S_, fmt=p25.FMT_CF32_IQ, decimation=50, max_chunk_samples=n, event_slots=64)
    bps, grid = 113, 148 * 3                                                  # blocks per stream, CTAs (3 per SM)
    n_static = (S_ * bps // grid) * 7 // 8
    straddlers = sorted({(n_static * b) // bps for b in range(1, grid, 8)})   # streams a static share begins inside
    sample = sorted(set([0, 1, 2, S_ - 2, S_ - 1] + straddlers + list(range((n_static * grid) // bps, S_, 9))))
    assert len(sample) >= 64
    worst, n_ev = _sampled_compare(p25, oracle, ctx, dev, base, n, False, 50, sample, 3)
    print(f"cfg2 geometry: {len(sample)} streams, {n_ev} events identical, max |baseband - oracle| = {worst:.2e}")
    ctx.close()


def test_cfg2_u8_bench_geometry_sampled_against_oracle(p25, oracle):
    """The same batch in the reference's own sample format (u8 IQ at 2.4 MS/s, 2 B/sample): the u8 /50 stream kernel."""
    import torch
    from bench import Workload
    from tools.shape_bench import tile_on_device
    wl = Workload("cfg2u8", 1)
    base = wl.base()                                                         # [16][360000][2] uint8
    S_, n = wl.streams, wl.n
    dev = tile_on_device(torch.from_numpy(base).cuda(), S_)
    ctx = p25.Context(S_, fmt=p25.FMT_U8_IQ, decimation=50, max_chunk_samples=n, event_slots=64)
    sample = sorted(set([0, 1, S_ - 1] + list(range(3, S_, 16))))
    worst, n_ev = _sampled_compare(p25, oracle, ctx, dev, base, n, True, 50, sample, 3)
    print(f"cfg2 u8 geometry: {len(sample)} streams, {n_ev} events, max |baseband - oracle| = {worst:.2e}")
    ctx.close()


def test_cfg5_bench_geometry_sampled_against_oracle(p25, oracle):
    """BASELINE configs[4] as bench.py times it -- 65,536 u8 streams x 36,000 samples, /5, warp-autonomous kernel whose
    warps enter streams mid-way -- three steps (generic kernel, then the fast one twice); 80 streams incl. warp-share
    boundaries against the oracle."""
    import torch
    from bench import Workload
    from tools.shape_bench import tile_on_device
    wl = Workload("cfg5", 1)
    base = wl.base()                                                         # [16][36000][2] uint8
    S_, n = wl.streams, wl.n
    dev = tile_on_device(torch.from_numpy(base).cuda(), S_)
    ctx = p25.Context(S_, fmt=p25.FMT_U8_IQ, decimation=5, max_chunk_samples=n, event_slots=64)
    ips, gw_total = (n // 5 + 123) // 124, 148 * 5 * 4                        # iterations per stream, warps in the grid
    total = S_ * ips
    straddlers = sorted({(total * g // gw_total) // ips for g in range(1, gw_total, 61)})
    sample = sorted(set([0, 1, S_ - 1, 4097, 32768] + straddlers + list(range(7, S_, 4999))))
    assert len(sample) >= 64
    worst, n_ev = _sampled_compare(p25, oracle, ctx, dev, base, n, True, 5, sample, 3)
    print(f"cfg5 geometry: {len(sample)} streams, {n_ev} events, max |baseband - oracle| = {worst:.2e}")
    ctx.close()


# ------------------------------------------------------------------ one process, several contexts and host threads
def _thread_job(p25, device, fmt, decim, data, chunk, overlap, out, key):
    try:
        ctx = p25.Context(data.shape[0], fmt=fmt, decimation=decim, max_chunk_samples=chunk, device=device)
        ctx.set_overlap(overlap)
        per = 2 if fmt == p25.FMT_U8_IQ else 1
        got = []
        n = data.shape[1] // per
        for i in range(0, n, chunk):
            ctx.process(np.ascontiguousarray(data[:, per * i: per * (i + chunk)]), chunk)
            got.append(ctx.poll())
        ev = np.concatenate(got)
        out[key] = ev[np.lexsort((ev["sample"], ev["stream"]))]
        ctx.close()
    except Exception as e:       # surfaced by the main thread
        out[key] = e


def _two_context_case(p25, oracle, devices):
    S_, chunk, n_chunks = 40, 16384, 4
    jobs = []
    for j, dev_id in enumerate(devices):
        u8 = j % 2 == 0
        fs, decim = (240_000, 5) if u8 else (2_400_000, 50)
        ck = chunk if u8 else chunk * 10
        rows = []
        for s in range(S_ if u8 else 6):
            st = tx.traffic_channel(8000 + 100 * j + s, 1) if s % 2 else tx.control_channel(8000 + 100 * j + s, 4)
            iq = tx.modulate_iq(st.dibits, fs, snr_db=18, cfo_hz=25.0 * s, seed=s + j)[: ck * n_chunks]
            assert len(iq) == ck * n_chunks
            rows.append(tx.iq_to_u8(iq) if u8 else iq)
        jobs.append((dev_id, p25.FMT_U8_IQ if u8 else p25.FMT_CF32_IQ, decim, np.stack(rows), ck, j % 2 == 1))
    out = {}
    threads = [threading.Thread(target=_thread_job, args=(p25, d, f, dc, data, ck, ov, out, j))
               for j, (d, f, dc, data, ck, ov) in enumerate(jobs)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for j, (d, f, dc, data, ck, ov) in enumerate(jobs):
        assert not isinstance(out[j], Exception), out[j]
        ofmt = oracle.FMT_U8 if f == p25.FMT_U8_IQ else oracle.FMT_CF32
        ref = np.concatenate([oracle.MessageReceiver(stream=s).feed(oracle.DemodChain(ofmt, dc == 50).feed(data[s]))
                              for s in range(data.shape[0])])
        a, b = set(events_key(out[j])), set(events_key(ref))
        assert len(ref) > 50 and len(a ^ b) <= len(ref) // 500, (j, len(a ^ b), len(ref))


def test_two_contexts_two_threads_one_device(p25, oracle):
    """Two contexts on device 0 driven from two host threads at once, different formats, kernels and overlap settings
    (the walker's carve-out preference flips between them): each equals the oracle."""
    _two_context_case(p25, oracle, [0, 0, 0, 0])


def test_contexts_on_two_devices_in_one_process(p25, oracle):
    """SURVEY 8e / reference src/main.rs:254-293 (one process, named threads): one context per GPU in ONE process, each on
    its own host thread, fast kernels with opted-in dynamic shared memory on both devices."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    _two_context_case(p25, oracle, [1, 0, 1, 0])


# ------------------------------------------------------------------ walker: tensor-pipe sync prefilter
def test_sync_prefilter_never_changes_the_decoded_output(p25, oracle, monkeypatch):
    """The TF32 prefilter of the sync search (decode_walk.cu sync_prefilter) may only skip search steps that hold no
    position above the detector's threshold.  Streams at 3..20 dB (many near-threshold correlations), gaps of silence
    and pure noise, odd chunk sizes: events, sample indices and stats with the prefilter forced on equal those with it
    off and the oracle's."""
    S_ = 40
    rows = []
    rng = np.random.default_rng(11)
    for s in range(S_):
        if s % 5 == 4:
            bb = (0.8 * rng.standard_normal(40000)).astype(np.float32)                     # nothing but noise
        else:
            st = tx.control_channel(6000 + s, 3, lead_idle=5 * s) if s % 2 else tx.traffic_channel(6000 + s, 1, lead_idle=3 * s)
            bb = tx.baseband_48k(st.dibits, snr_db=[3, 4, 5, 6, 8, 20][s % 6], seed=s, dc=0.02 * (s % 4), timing_offset=0.3 * (s % 7))[0]
            if s % 3 == 0:
                bb = np.concatenate([np.zeros(1500 + 77 * s, np.float32), bb])             # silence first: energy 0 windows
        rows.append(bb)
    n = min(len(r) for r in rows)
    bb = np.stack([r[:n] for r in rows])
    ref, ref_stats = oracle_events(oracle, bb)
    got = {}
    for flag in ("1", "0"):
        monkeypatch.setenv("P25CU_WALK_PREFILTER", flag)
        ctx = p25.Context(S_, max_chunk_samples=1024, max_baseband=5003)
        rx = p25.MessageReceiver(ctx)
        ev = np.concatenate([rx.feed(bb[:, i:i + 5003]) for i in range(0, n, 5003)])
        got[flag] = (ev[np.lexsort((ev["sample"], ev["stream"]))], np.stack([ctx.stats(s) for s in range(S_)]))
        ctx.close()
    assert len(ref) > 200
    for flag in ("1", "0"):
        assert events_key(got[flag][0]) == events_key(ref), flag
        assert (got[flag][1] == np.stack(ref_stats)).all(), flag


def test_cfg3_bench_geometry_sampled_against_oracle(p25, oracle):
    """BASELINE configs[2] as bench.py times it -- 8 wideband captures x 2,880,000 samples through the cluster channelizer
    kernel (9 runs of 800 output times per capture, each with its own warm-up from the carried tail), two consecutive
    steps -- 12 sampled (capture, channel) streams against the definition: mix down, 6,144-tap prototype, keep every 400th
    (scipy upfirdn, float64), then the oracle's 48 kHz chain and receiver.  Occupied channels: baseband within the FP32
    tolerance; all sampled streams: events identical."""
    import torch
    from scipy import signal
    from bench import Workload
    wl = Workload("cfg3", 1)
    n, caps = wl.n, wl.rows
    dev = wl.device_input(0)
    ctx = p25.Context(wl.streams, fmt=p25.FMT_CF32_IQ, decimation=400, max_chunk_samples=n, event_slots=64)
    n_steps, got_ev = 2, []
    for _ in range(n_steps):
        ctx.process(dev, n)
        got_ev.append(ctx.poll())
    n_out = n // 400
    ev = np.concatenate(got_ev)
    h = S.taps_pfb().astype(np.float64)
    occupied = [(37 * i + 5) % 1536 for i in range(64)]
    idle = [k for k in range(1536) if k not in occupied]
    sample = [(c, k) for c in (0, 3, 7) for k in (occupied[0], occupied[31], occupied[63], idle[5 + 100 * c])]
    oracle.lib().p25o_set_always_correlate(0)
    nn = np.arange(n_steps * n)
    ref_ev, worst = [], 0.0
    for c, k in sample:
        x = np.tile(wl.oracle_row(c).astype(np.complex128), n_steps)                      # both steps of this capture
        xm = x * np.exp(-2j * np.pi * ((k * nn) % 1536) / 1536.0)
        y = signal.upfirdn(h, np.concatenate([[0.0], xm]), up=1, down=400)[1:n_steps * n // 400 + 1]   # newest input 400 m + 399
        rbb = oracle.DemodChain(oracle.FMT_CF32, 2).feed(y.astype(np.complex64))
        s_id = c * 1536 + k
        ref_ev.append(oracle.MessageReceiver(stream=s_id).feed(rbb))
        if k in occupied:                                                                  # second step: what the device still holds
            bb = ctx.read_baseband(s_id, n_out)
            worst = max(worst, float(np.max(np.abs(bb - rbb[n_out:]))))
    ref_ev = np.concatenate(ref_ev)
    ref_ev = ref_ev[np.lexsort((ref_ev["sample"], ref_ev["stream"]))]
    ids = [c * 1536 + k for c, k in sample]
    got = ev[np.isin(ev["stream"], ids)]
    got = got[np.lexsort((got["sample"], got["stream"]))]
    assert worst < BB_TOL, worst
    assert len(ref_ev) >= 9 * 6 and events_key(got) == events_key(ref_ev)
    ctx.close()


def test_channelizer_is_invariant_under_chunking(p25, oracle):
    """The cluster kernel recomputes its warm-up (c[m-1], nine discriminator values) from the carried input tail at the
    start of every run.  Two captures fed as one chunk and as a ragged sequence (1 sample, less than one output, not a
    multiple of 400, a chunk with no output at all ...) must give the same spectra (to rounding: the order in which a
    window's sixteen slots are summed depends on where the run started), the same baseband on the occupied channels and
    the same events."""
    rng = np.random.default_rng(21)
    st = tx.control_channel(4242, 2, lead_idle=10)
    n = (len(st.dibits) * 10 + 300) * 400 + 37
    cap0 = tx.wideband_capture({7: (st.dibits, 0.05, 20.0), 1530: (st.dibits, 0.03, -35.0)}, n, noise_db=-50.0, seed=5)
    cap1 = (0.02 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))).astype(np.complex64)
    caps = np.stack([cap0.astype(np.complex64), cap1])

    def run(chunks):
        ctx = p25.Context(2 * 1536, fmt=p25.FMT_CF32_IQ, decimation=400, max_chunk_samples=max(chunks), event_slots=32)
        ctx.keep_spectra(True)
        ys, bbs, pos, n_tot = [], [], 0, 0
        for m in chunks:
            bb, n_out, _ = ctx.demod(np.ascontiguousarray(caps[:, pos:pos + m]), m)
            if n_out:
                ys.append(ctx.channelizer_output())
                bbs.append(bb)
            ctx.decode()
            pos += m
            n_tot += n_out
        ev = ctx.poll()
        ctx.close()
        return np.concatenate(ys, axis=1), np.concatenate(bbs, axis=1), n_tot, ev[np.lexsort((ev["sample"], ev["stream"]))]

    whole = run([n])
    ragged = run([1, 398, 1, 400, 401, 7, 3, 40000, 799, 12345, n - (1 + 398 + 1 + 400 + 401 + 7 + 3 + 40000 + 799 + 12345)])
    assert whole[2] == ragged[2] == n // 400
    scale = float(np.max(np.abs(whole[0])))
    assert np.max(np.abs(whole[0] - ragged[0])) < 2e-6 * scale, np.max(np.abs(whole[0] - ragged[0])) / scale
    for k in (7, 1530):
        assert np.max(np.abs(whole[1][k, 200:] - ragged[1][k, 200:])) < BB_TOL, k
    busy = lambda e: e[np.isin(e["stream"], (7, 1530))]
    assert events_key(busy(whole[3])) == events_key(busy(ragged[3])) and len(busy(whole[3])) >= 8, len(busy(whole[3]))


# ------------------------------------------------------------------ integer-tensor-pipe decimators: chunk phases and edge sizes
@pytest.mark.parametrize("dec,chunks", [
    (5, [16384, 1312, 1320, 2568, 5128, 20000, 1312, 8]),          # 1312 = the carried tail: the smallest fast-path chunk
    (50, [16384, 3264, 3272, 6648, 12808, 40000, 3264, 8, 1608, 3264]),   # 1608: shorter than the tail
])
def test_u8_imma_kernels_chunk_phases_and_minimal_chunks(p25, oracle, dec, chunks):
    """w5i / w50i (u8, decimator stages as u8 x s8 mma.sync on the raw bytes): a chunk sequence that walks the slice's
    alignment inside its 16-byte group through every value it can take, with chunks as short as the carried tail (one warp
    iteration per stream: warm-up + one partial iteration), one of a single 16-byte group (generic kernel between two
    fast ones), seven streams (a ragged share of the flattened work space), power requested on alternate chunks (both
    template instantiations).  /50 also feeds an aligned chunk with outputs but shorter than the tail, which the FFMA2
    stream kernel fast::p25_ddc_fm_stream_kernel<u8> serves, and then a w50i chunk that starts from the tail it carried.
    Baseband <= 1e-4 of the oracle's, power <= 0.01 dB."""
    fs = 240_000 * (dec // 5)
    S_ = 7
    total = sum(chunks)
    rows = []
    for s in range(S_):
        st = tx.control_channel(700 + s, 3)
        iq = tx.modulate_iq(st.dibits, fs, snr_db=22, cfo_hz=60.0 * (s - 3), seed=40 + s, amplitude=[0.02, 0.1, 0.3, 0.5, 0.7, 0.9, 0.97][s])
        assert len(iq) >= total
        rows.append(tx.iq_to_u8(iq[:total]))
    data = np.stack(rows)
    ctx = p25.Context(S_, fmt=p25.FMT_U8_IQ, decimation=dec, max_chunk_samples=max(chunks))
    chains = [oracle.DemodChain(oracle.FMT_U8, dec == 50) for _ in range(S_)]
    pos, worst = 0, 0.0
    for i, m in enumerate(chunks):
        part = np.ascontiguousarray(data[:, 2 * pos: 2 * (pos + m)])
        want_pw = i % 2 == 1
        bb, n_out, pw = ctx.demod(part, m, want_power=want_pw)
        for s in range(S_):
            ref = chains[s].feed(part[s], want_power=want_pw)
            if want_pw:
                ref, pref = ref
                if n_out:
                    assert abs(pw[s] - pref) < 1e-2, (i, s, pw[s], pref)
                else:                                   # a chunk without outputs: power_dbm of nothing is -inf on both sides
                    assert not np.isfinite(pw[s]) and not np.isfinite(pref)
            assert len(ref) == n_out
            if n_out:
                worst = max(worst, float(np.max(np.abs(bb[s] - ref))))
        pos += m
    assert worst < BB_TOL, worst
    ctx.close()
