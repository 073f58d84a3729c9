"""Every demod kernel route and the power output against the float64 chain (oracle/demod_f64.py).

The older demod tests compare with the float32 C++ oracle at 1e-4 (the oracle the walker is bit-exact to).  That bar has
about 300x headroom over the kernels' rounding, enough for a kernel that loses a channel-filter or front-stage tap to
pass.  The bars here are set from the other side: the CPU tests below show, for every stimulus and chunk plan the GPU
tests use, that

  * zeroing any single tap (|h| > 1e-12) of the front, decimator or channel filter moves the baseband of the chunks each
    kernel route serves by at least MARGIN x BB_BAR (max-abs over the conditioned outputs);
  * leaving one output out of a chunk's power sum, or counting one twice, moves the reported power by at least
    MARGIN x PW_BAR (relative, linear).  The device divides the sum by the chunk's output count, so a dropped or
    doubled output j moves the mean by |c_j|^2 / sum |c|^2: the check takes the smallest such share among the outputs
    each mutant can hit (the first and last output of the chunk; any output for a doubled one; every output of the
    period for the bench geometries, whose streams are shifted by every multiple of D);
  * the float32 oracle itself sits within BB_BAR / MARGIN of the float64 chain, and the conditioning rule keeps >= 99 %
    of the outputs.

The mutant family is single taps of the spec filters.  w5i and w50i do not run those taps directly: they run
hand-built integer tables (w50i's 290-tap cascade g = hd (*) hf, whose individual taps are often below 1e-6), and a
one-entry error in such a table is not a spec-tap mutant, so these bars need not catch it.  Those tables are pinned bit
for bit by tests/test_w5i_dataflow.py (test_library_tables_equal_the_model, through tests/hostcheck/imma_hostcheck.cpp)
instead.

The GPU tests then hold every route to BB_BAR / PW_BAR and print what they measure.  Where a carrier fades towards zero
the discriminator's rounding error grows like 1/|c|; those outputs are excluded by demod_f64.conditioned(), a rule
computed from the reference, never by per-stream skips."""
import numpy as np
import pytest
from oracle import demod_f64 as F
from tools import p25tx as tx

BB_BAR = 1.5e-6          # baseband, absolute (full scale +-4.8)
PW_BAR = 1e-5            # power, relative in linear units (4.3e-5 dB)
CH_PW_BAR = 1e-5         # channelizer power of the occupied channels, relative
MARGIN = 4
FS = {5: 240_000, 50: 2_400_000}
HT = {5: 1312, 50: 3264}  # carried input tail per decimation (ddc_fm.cu Cfg<FRONT>::HT)


# ------------------------------------------------------------------ stimuli
def _bursts(n: int, fs: int, centres, width_s: float = 1e-3, gain: float = 2.0, period: int | None = None) -> np.ndarray:
    """Amplitude envelope 1 + gain * (Gaussian bursts at the given sample positions), optionally periodic in `period`."""
    t = np.arange(n, dtype=np.float64)
    env = np.ones(n)
    w = width_s * fs
    for c in centres:
        d = t - c
        if period:
            d = (d + period / 2) % period - period / 2
        env += gain * np.exp(-0.5 * (d / w) ** 2)
    return env


# (amplitude, carrier offset Hz, SNR dB, power bursts): +-4 LSB to near full scale in u8 terms
SWEEP_ROWS = [(0.5, 0.0, 25, False), (0.9, 300.0, 25, False), (0.03, -200.0, 30, False), (0.06, 150.0, 22, False),
              (0.3, 0.0, 25, True), (0.7, -450.0, 25, False), (0.25, 80.0, 20, True), (0.85, 600.0, 20, False)]

# Chunk plans: (input samples, power requested, route).  Routes follow p25cu_launch_ddc (ddc_fm.cu):
#   /5:  chunks with outputs, aligned rows (even cf32 / multiple-of-8 u8 length) and a0 >= 1312, of any length
#        -> w5 (cf32) / w5i (u8); anything else (the first chunk, odd lengths) -> generic p25_ddc_fm_kernel<false, FMT>
#   /50 cf32: aligned rows and an even a0 -> fast::p25_ddc_fm_stream_kernel, else generic <true, cf32>
#   /50 u8: aligned rows and a0 >= 3264, of any length -> w50i; else generic <true, u8>
# The generic kernel splits a stream into segments when a chunk has >= 16 blocks of outputs (ddc_fm.cu): the first
# chunk of each plan is one segment, the second several.  The warp kernels also take chunks shorter than the carried
# tail (1,312 / 3,264 samples), down to one or two outputs, and carry the tail of such a chunk from the old tail and
# the chunk; the chunk after each one starts from that tail.
PLANS = {
    ("cf32", 5): [(777, True, "generic"), (30001, True, "generic_seg"), (16384, True, "w5"), (1312, False, "w5"),
                  (1304, True, "w5"), (6, False, "w5"), (650, True, "w5")],
    ("u8", 5): [(777, True, "generic"), (30001, False, "generic_seg"), (16384, True, "w5i_pw"), (16384, False, "w5i"),
                (1312, True, "w5i_pw"), (1304, False, "w5i"), (8, True, "w5i_pw"), (648, False, "w5i")],
    ("cf32", 50): [(47999, True, "generic"), (100001, False, "generic_seg"), (40000, True, "fast"), (40000, False, "fast")],
    ("u8", 50): [(47999, True, "generic"), (100001, True, "generic_seg"), (40000, True, "w50i_pw"), (40000, False, "w50i")] +
                [(3256, i % 2 == 0, "w50i_pw" if i % 2 == 0 else "w50i") for i in range(6)] + [(3264, True, "w50i_pw")],
}

# route -> the kernel the profiler must see
KERNELS = {("cf32", 5, "generic"): "p25_ddc_fm_kernel<false,1>", ("u8", 5, "generic"): "p25_ddc_fm_kernel<false,0>",
           ("cf32", 50, "generic"): "p25_ddc_fm_kernel<true,1>", ("u8", 50, "generic"): "p25_ddc_fm_kernel<true,0>",
           ("cf32", 5, "w5"): "w5::p25_ddc5_warp_kernel", ("u8", 5, "w5i_pw"): "w5i::p25_ddc5_imma_kernel<true>",
           ("u8", 5, "w5i"): "w5i::p25_ddc5_imma_kernel<false>", ("cf32", 50, "fast"): "fast::p25_ddc_fm_stream_kernel",
           ("u8", 50, "w50i_pw"): "w50i::p25_ddc50_imma_kernel<true>",
           ("u8", 50, "w50i"): "w50i::p25_ddc50_imma_kernel<false>"}


def _route(fmt: str, dec: int, a0: int, n: int) -> str:
    """p25cu_launch_ddc's choice for a chunk of n samples at absolute input sample a0 (rows 16-byte aligned in memory)."""
    u8 = fmt == "u8"
    aligned = n % (8 if u8 else 2) == 0
    n_out = (a0 + n) // dec - a0 // dec
    if dec == 5 and aligned and n_out > 0 and a0 >= HT[5]:
        return "w5i" if u8 else "w5"
    if dec == 50 and not u8 and aligned and a0 % 2 == 0 and n_out > 0:
        return "fast"
    if dec == 50 and u8 and aligned and n_out > 0 and a0 >= HT[50]:
        return "w50i"
    return "generic"


def _generic_segments(dec: int, n_out: int, n_streams: int, n_sm: int) -> int:
    """The generic kernel's segment split (its launcher in ddc_fm.cu)."""
    mb = 64 if dec == 50 else 256
    iters = -(-n_out // mb)
    want = max(1, min(n_sm * 16 // n_streams, iters // 8))
    seg_out = -(-iters // want) * mb
    return -(-n_out // seg_out) if n_out else 1


def _sweep_inputs(fmt: str, dec: int):
    """The route sweep's streams: (device input rows [S][n] in the context's format, complex128 rows the float64 chain
    sees).  Power bursts sit on the plan's chunk boundaries, so the first and last outputs of a chunk carry a large share
    of its power."""
    fs, plan = FS[dec], PLANS[(fmt, dec)]
    total = sum(m for m, _, _ in plan)
    edges = np.cumsum([0] + [m for m, _, _ in plan])
    dev, x = [], []
    for s, (amp, cfo, snr, bursts) in enumerate(SWEEP_ROWS):
        st = tx.control_channel(1400 + s, 4)
        iq = tx.modulate_iq(st.dibits, fs, snr_db=snr, cfo_hz=cfo, seed=60 + s, amplitude=amp)
        assert len(iq) >= total
        iq = iq[:total].astype(np.complex128)
        if bursts:
            iq = iq * _bursts(total, fs, edges)
        iq = iq.astype(np.complex64)
        if fmt == "u8":
            raw = tx.iq_to_u8(iq)
            dev.append(raw)
            x.append(F.u8_to_c128(raw))
        else:
            dev.append(iq)
            x.append(iq.astype(np.complex128))
    return np.stack(dev), x


def _chunk_slices(plan, dec):
    out, a0 = [], 0
    for m, pw, route in plan:
        out.append((a0, m, pw, route, F.chunk_outputs(a0, m, dec)))
        a0 += m
    return out


# bench geometries: workload -> (format, decimation, streams, samples per step)
BENCH = {"cfg2": ("cf32", 50, 1024, 360_000), "cfg2u8": ("u8", 50, 1024, 360_000), "cfg5": ("u8", 5, 65536, 36_000)}
N_BASE = 16


def _bench_bases(name: str):
    """16 periodic base rows: tools/shape_bench.base_streams (what bench.py feeds), the upper half with a periodic burst
    envelope.  Returns (device rows [16][n][2] in the workload's format, complex128 rows, n)."""
    from tools.shape_bench import base_streams
    fmt, dec, _, n = BENCH[name]
    base = base_streams("control", FS[dec], N_BASE, 20.0).astype(np.complex128)
    assert base.shape[1] == n
    rows, x = [], []
    for b in range(N_BASE):
        iq = base[b]
        if b >= N_BASE // 2:
            iq = iq * _bursts(n, FS[dec], [n * (j + 0.5) / (b - 6) for j in range(b - 6)], gain=0.75, period=n)
        iq = iq.astype(np.complex64)
        if fmt == "u8":
            raw = tx.iq_to_u8(iq)
            rows.append(raw.reshape(n, 2))
            x.append(F.u8_to_c128(raw))
        else:
            rows.append(iq.view(np.float32).reshape(n, 2))
            x.append(iq.astype(np.complex128))
    return np.stack(rows), x, n


def _steady_state(x: np.ndarray, dec: int) -> dict:
    """Stages of two periods of a periodic input: the outputs of the second period are the steady state."""
    return F.stages(np.tile(x, 2), dec)


def _bench_shift(s, N: int):
    """Stream s of a bench geometry is base s % 16 advanced by this many outputs (the input by D times as many samples).
    s: an int or an integer tensor of stream ids."""
    return (s // N_BASE) * 1009 % N


# ------------------------------------------------------------------ CPU: the reference and the bars are sound
def _feed_chunks(oracle, fmt, dec, raw, chunks):
    ch = oracle.DemodChain(oracle.FMT_U8 if fmt == "u8" else oracle.FMT_CF32, dec == 50)
    per = 2 if fmt == "u8" else 1
    out, pos = [], 0
    for m in chunks:
        out.append(ch.feed(raw[per * pos: per * (pos + m)], want_power=True))
        pos += m
    return out


@pytest.mark.parametrize("fmt,dec", [("cf32", 5), ("u8", 5), ("cf32", 50), ("u8", 50)])
def test_float64_chain_matches_oracle_conventions(oracle, fmt, dec):
    """Decimator phase, stream-start zeros and the u8 table: the float64 chain equals the float32 oracle within 3e-7 on
    the conditioned outputs of every chunk (a first chunk, odd lengths, a chunk without outputs), and power within the
    oracle's own sequential float32 summation error (n_out x 2^-24 relative)."""
    fs = FS[dec]
    chunks = [3, 1, dec + 1, dec - 2, 4999 * (dec // 5), 2, 16383 * (dec // 5), 1001]
    total = sum(chunks)
    iq = tx.modulate_iq(tx.control_channel(1300, 3).dibits, fs, snr_db=25, cfo_hz=120.0, seed=9, amplitude=0.4)[:total]
    assert len(iq) == total
    raw = tx.iq_to_u8(iq) if fmt == "u8" else iq
    x = F.u8_to_c128(raw) if fmt == "u8" else iq.astype(np.complex128)
    c, bb = F.chain(x, dec)
    assert len(bb) == total // dec
    mask = F.conditioned(c)
    assert mask.mean() > 0.98
    a0, n_empty = 0, 0
    for m, (obb, opw) in zip(chunks, _feed_chunks(oracle, fmt, dec, raw, chunks)):
        sl = F.chunk_outputs(a0, m, dec)
        assert len(obb) == sl.stop - sl.start
        ref_pw = F.chunk_power_dbm(c, a0, m, dec)
        if len(obb) == 0:
            n_empty += 1
            assert not np.isfinite(opw) and not np.isfinite(ref_pw)
        else:
            err = np.abs(obb - bb[sl])[mask[sl]]
            assert err.size == 0 or err.max() < 3e-7, (m, err.max())
            rel = abs(10 ** ((opw - ref_pw) / 10) - 1)
            assert rel < len(obb) * 2.0 ** -24 + 2e-6, (m, rel)
        a0 += m
    assert n_empty >= 1


def test_tap_mutant_shortcut_equals_zeroed_taps():
    """demod_f64.tap_mutant (the linear shortcut the sensitivity checks use) equals chain() with the tap zeroed."""
    rng = np.random.default_rng(3)
    x = rng.standard_normal(20000) + 1j * rng.standard_normal(20000)
    s = F.stages(x, 50)
    for stage, k in (("front", 0), ("front", 31), ("decim", 24), ("decim", 7), ("chan", 0), ("chan", 40)):
        t = s["taps"][stage].copy()
        t[k] = 0.0
        c_ref, bb_ref = F.chain(x, 50, {stage: t})
        c, bb = F.tap_mutant(s, stage, k)
        assert np.max(np.abs(c - c_ref)) < 1e-12 and np.max(np.abs(bb - bb_ref)) < 1e-9, (stage, k)


def _weakest_tap_mutant(s: dict, dec: int, groups: dict):
    """groups: name -> boolean mask over the outputs.  Returns name -> (max |baseband change| of the single-tap mutant
    that changes that group least, stage, tap)."""
    out = {g: (np.inf, None, None) for g in groups}
    for stage in (("front", "decim", "chan") if dec == 50 else ("decim", "chan")):
        for k in np.nonzero(np.abs(s["taps"][stage]) > 1e-12)[0]:
            _, bb = F.tap_mutant(s, stage, int(k))
            d = np.abs(bb - s["bb"])
            for g, m in groups.items():
                v = float(d[m].max()) if m.any() else 0.0
                if v < out[g][0]:
                    out[g] = (v, stage, int(k))
    return out


@pytest.mark.parametrize("fmt,dec", [("cf32", 5), ("u8", 5), ("cf32", 50), ("u8", 50)])
def test_route_sweep_bars_separate_mutants(oracle, fmt, dec):
    """For the route sweep's streams and chunk plan: every single-tap mutant moves each route's conditioned outputs by
    >= MARGIN x BB_BAR (a kernel route is wrong for every stream at once, so the distance is the largest over the streams
    that route served); dropping a chunk's first or last output from the power sum, or doubling any of its outputs,
    moves the power by >= MARGIN x PW_BAR; the float32 oracle is within BB_BAR / MARGIN; the mask keeps >= 99 %."""
    plan = PLANS[(fmt, dec)]
    dev, xs = _sweep_inputs(fmt, dec)
    chunks = _chunk_slices(plan, dec)
    routes = sorted({r for _, _, _, r, _ in chunks})
    worst_mut = {r: 0.0 for r in routes}
    kept = []
    for s, x in enumerate(xs):
        st = F.stages(x, dec)
        c, bb = st["c"], st["bb"]
        mask = F.conditioned(c)
        kept.append(mask[F.BOXCAR:].mean())
        groups = {}
        for _, _, _, r, sl in chunks:
            g = groups.setdefault(r, np.zeros(len(bb), bool))
            g[sl] = mask[sl]
        for r, (v, _, _) in _weakest_tap_mutant(st, dec, groups).items():
            worst_mut[r] = max(worst_mut[r], v)
        obb = np.concatenate([o for o, _ in _feed_chunks(oracle, fmt, dec, dev[s], [m for m, _, _ in plan])])
        assert np.max(np.abs(obb - bb)[mask]) <= BB_BAR / MARGIN, s
        p = np.abs(c) ** 2
        for a0, m, pw, r, sl in chunks:
            if not pw or sl.stop == sl.start:
                continue
            # covers the first, the last and any doubled output; the outputs the mask leaves out (the filters filling
            # at the stream start) carry next to no power, and no power bar can see them dropped
            share = p[sl][mask[sl]].min() / p[sl].sum()
            assert share >= MARGIN * PW_BAR, (s, r, a0, share)
    print(f"{fmt} /{dec} weakest single-tap mutant per route: " + ", ".join(f"{r} {v:.2e}" for r, v in worst_mut.items()))
    for r, v in worst_mut.items():
        assert v >= MARGIN * BB_BAR, (r, v)
    assert min(kept) >= 0.99, kept


@pytest.mark.parametrize("name", sorted(BENCH))
def test_bench_geometry_bars_separate_mutants(oracle, name):
    """The same three checks for the 16 periodic bases of each bench geometry, in steady state (one period after one
    period of warm-up): every stream is a base shifted by a whole number of outputs, so over all streams every output
    of the period is some chunk's first and last output."""
    fmt, dec, _, n = BENCH[name]
    rows, xs, _ = _bench_bases(name)
    N = n // dec
    worst = np.inf
    for b, x in enumerate(xs):
        st = _steady_state(x, dec)
        c, bb = st["c"], st["bb"]
        mask = F.conditioned(c)
        mask[:N] = False
        assert mask[N:].mean() >= 0.99, (b, mask[N:].mean())
        v = _weakest_tap_mutant(st, dec, {"all": mask})["all"]
        worst = min(worst, v[0])
        assert v[0] >= MARGIN * BB_BAR, (b, v)
        p = np.abs(c[N:]) ** 2
        assert p.min() / p.sum() >= MARGIN * PW_BAR, (b, p.min() / p.sum())
        raw = rows[b].reshape(-1) if fmt == "u8" else rows[b].reshape(-1).view(np.complex64)
        obb = oracle.DemodChain(oracle.FMT_U8 if fmt == "u8" else oracle.FMT_CF32, dec == 50).feed(np.tile(raw, 2))
        assert np.max(np.abs(obb - bb)[mask]) <= BB_BAR / MARGIN, b
    print(f"{name}: weakest single-tap mutant over the 16 bases {worst:.2e}")


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def p25():
    import p25rx_b200
    return p25rx_b200


def _rel_power(got_dbm, ref_dbm):
    return np.abs(10.0 ** ((np.asarray(got_dbm, np.float64) - ref_dbm) / 10.0) - 1.0)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,dec", [("cf32", 5), ("u8", 5), ("cf32", 50), ("u8", 50)])
def test_route_sweep_against_float64(p25, fmt, dec):
    """Every kernel route of p25cu_launch_ddc (see PLANS), eight streams from +-4 LSB to near full scale with carrier
    offsets and power bursts: baseband within BB_BAR of the float64 chain on the conditioned outputs, power within
    PW_BAR (relative) of the float64 mean |c|^2."""
    plan = PLANS[(fmt, dec)]
    dev, xs = _sweep_inputs(fmt, dec)
    S_ = len(xs)
    refs = [F.chain(x, dec) for x in xs]
    masks = [F.conditioned(c) for c, _ in refs]
    import torch
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    ctx = p25.Context(S_, fmt=p25.FMT_U8_IQ if fmt == "u8" else p25.FMT_CF32_IQ, decimation=dec,
                      max_chunk_samples=max(m for m, _, _ in plan))
    per = 2 if fmt == "u8" else 1
    bb_err, pw_err = {}, {}
    for a0, m, want_pw, route, sl in _chunk_slices(plan, dec):
        assert _route(fmt, dec, a0, m) == route.split("_")[0], (a0, m, route)
        if route.startswith("generic"):
            assert (_generic_segments(dec, sl.stop - sl.start, S_, n_sm) > 1) == (route == "generic_seg"), (a0, m)
        bb, n_out, pw = ctx.demod(np.ascontiguousarray(dev[:, per * a0: per * (a0 + m)]), m, want_power=want_pw)
        assert n_out == sl.stop - sl.start
        for s in range(S_):
            (c, rbb), mk = refs[s], masks[s][sl]
            if mk.any():
                bb_err[route] = max(bb_err.get(route, 0.0), float(np.max(np.abs(bb[s] - rbb[sl])[mk])))
            if want_pw:
                pw_err[route] = max(pw_err.get(route, 0.0), float(_rel_power(pw[s], F.chunk_power_dbm(c, a0, m, dec))))
    ctx.close()
    print(f"{fmt} /{dec}: max |baseband - float64| " + ", ".join(f"{r} {v:.2e}" for r, v in sorted(bb_err.items())) +
          "; power relative " + ", ".join(f"{r} {v:.2e}" for r, v in sorted(pw_err.items())))
    assert max(bb_err.values()) < BB_BAR, bb_err
    assert max(pw_err.values()) < PW_BAR, pw_err


@pytest.mark.gpu
def test_route_table_kernels_ran(p25):
    """torch.profiler (CUDA activities) around one demod call per chunk of every plan: each chunk launched the kernel its
    route names, and nothing else from ddc_fm.cu."""
    from torch.profiler import ProfilerActivity, profile
    seen = []
    for (fmt, dec), plan in PLANS.items():
        dev, _ = _sweep_inputs(fmt, dec)
        per = 2 if fmt == "u8" else 1
        ctx = p25.Context(dev.shape[0], fmt=p25.FMT_U8_IQ if fmt == "u8" else p25.FMT_CF32_IQ, decimation=dec,
                          max_chunk_samples=max(m for m, _, _ in plan))
        for a0, m, want_pw, route, _ in _chunk_slices(plan, dec):
            part = np.ascontiguousarray(dev[:, per * a0: per * (a0 + m)])
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                ctx.demod(part, m, want_power=want_pw)
                ctx.sync()
            names = {e.name.replace(" ", "") for e in prof.events() if "ddc" in e.name}
            want = KERNELS[(fmt, dec, route.replace("_seg", ""))]
            assert any(want in nm for nm in names), (fmt, dec, a0, m, route, names)
            assert len(names) == 1, names
            seen.append(want)
        ctx.close()
    assert set(seen) == set(KERNELS.values())
    print("kernels seen: " + ", ".join(sorted(set(seen))))


def _tile_by_outputs(base_dev, S_: int, dec: int):
    """dev[s] = base[s % 16] advanced by _bench_shift(s) outputs (a multiple of D input samples), built in slabs."""
    import torch
    B, n = base_dev.shape[0], base_dev.shape[1]
    assert B == N_BASE
    N = n // dec
    dev = torch.empty((S_,) + tuple(base_dev.shape[1:]), dtype=base_dev.dtype, device=base_dev.device)
    ar = torch.arange(n, device=base_dev.device)
    slab = max(1, (1 << 27) // n)
    for s0 in range(0, S_, slab):
        g = torch.arange(s0, min(S_, s0 + slab), device=base_dev.device)
        sh = _bench_shift(g, N) * dec
        dev[s0:s0 + len(g)] = base_dev[(g % B)[:, None], (ar[None, :] + sh[:, None]) % n]
    return dev


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(BENCH))
def test_bench_geometry_every_stream_against_float64(p25, name):
    """The bench geometries (persistent grids, warps and static shares that enter streams mid-way, the /50 static +
    ticket split) with power: three steps of demod(want_power=True).  From step 2 on every output of every stream is a
    cyclic shift of its base's steady-state float64 output and every stream's power equals its base's: all streams'
    baseband and power are checked, so a dropped or doubled iteration anywhere in the work split fails."""
    import torch
    fmt, dec, S_, n = BENCH[name]
    rows, xs, _ = _bench_bases(name)
    N = n // dec
    ref_bb, ref_mask, ref_pw = [], [], []
    for x in xs:
        st = _steady_state(x, dec)
        c = st["c"]
        mask = F.conditioned(c)
        ref_bb.append(st["bb"][N:])
        ref_mask.append(mask[N:])
        ref_pw.append(F.chunk_power_dbm(c, n, n, dec))
    gpu = torch.device("cuda")
    rbb = torch.from_numpy(np.stack(ref_bb)).to(gpu)
    rmask = torch.from_numpy(np.stack(ref_mask)).to(gpu)
    dev = _tile_by_outputs(torch.from_numpy(rows).to(gpu), S_, dec)
    ctx = p25.Context(S_, fmt=p25.FMT_U8_IQ if fmt == "u8" else p25.FMT_CF32_IQ, decimation=dec, max_chunk_samples=n)
    torch.cuda.synchronize()           # the library reads the input on its own stream
    sid = torch.arange(S_, device=gpu)
    shift = _bench_shift(sid, N)
    col = torch.arange(N, device=gpu)
    bb_worst, pw_worst = 0.0, 0.0
    for step in range(3):
        bb, n_out, pw = ctx.demod(dev, n, want_power=True)
        assert n_out == N
        if step == 0:
            continue
        slab = max(1, (1 << 26) // N)
        for s0 in range(0, S_, slab):
            s1 = min(S_, s0 + slab)
            got = torch.from_numpy(bb[s0:s1]).to(gpu).double()
            idx = (col[None, :] + shift[s0:s1, None]) % N
            b = (sid[s0:s1] % N_BASE)[:, None]
            err = torch.where(rmask[b, idx], (got - rbb[b, idx]).abs(), torch.zeros((), dtype=torch.float64, device=gpu))
            bb_worst = max(bb_worst, float(err.max()))
        rel = _rel_power(pw, np.array(ref_pw)[np.arange(S_) % N_BASE])
        pw_worst = max(pw_worst, float(rel.max()))
    ctx.close()
    del dev
    print(f"{name}: {S_} streams, steps 2-3, max |baseband - float64| = {bb_worst:.2e}, power relative {pw_worst:.2e}")
    assert bb_worst < BB_BAR and pw_worst < PW_BAR, (bb_worst, pw_worst)


CH_CHUNKS_HEAD = [1, 398, 1, 400, 401, 7, 3, 40000, 799, 12345]


def _channelizer_capture():
    st = tx.control_channel(4343, 2, lead_idle=10)
    n = (len(st.dibits) * 10 - 100) * 400 + 37                 # the carriers are on from the first sample to the last
    occupied = {7: 0.05, 400: 0.03, 767: 0.04, 1100: 0.05, 1530: 0.03}
    cap = tx.wideband_capture({k: (st.dibits, a, 15.0 * (k % 7 - 3)) for k, a in occupied.items()}, n, noise_db=-50.0, seed=8)
    env = _bursts(n, 19_200_000, np.cumsum(CH_CHUNKS_HEAD), width_s=4e-4, gain=2.0)
    return (cap.astype(np.complex128) * env).astype(np.complex64), occupied


@pytest.mark.gpu
def test_channelizer_power_every_channel(p25):
    """Channelizer power: a capture with an amplitude envelope (bursts on the chunk boundaries), ragged chunks (one
    sample, less than one output, not multiples of 400, chunks without outputs), all 1,536 channels' power of every chunk
    against the mean |channel_filter(channelize(x))|^2 over the chunk's outputs.  Occupied channels within CH_PW_BAR
    relative; idle channels, and every channel while the filters fill at the stream start, within the absolute error
    that the 2e-5 spectra bar allows: |P - P_ref| <= 2 sqrt(P_ref) e + e^2 with e = 2e-5 of the spectra's full scale."""
    from oracle import pfb_oracle as pfb
    cap, occupied = _channelizer_capture()
    n = len(cap)
    chunks = CH_CHUNKS_HEAD + [n - sum(CH_CHUNKS_HEAD)]
    ref_c = pfb.channel_filter(pfb.channelize(cap))            # [n_out][1536]
    e = 2e-5 * float(np.max(np.abs(ref_c)))
    mask = F.conditioned(ref_c[:, sorted(occupied)[0]])
    ctx = p25.Context(1536, fmt=p25.FMT_CF32_IQ, decimation=400, max_chunk_samples=max(chunks))
    occ = np.array(sorted(occupied))
    idle = np.setdiff1d(np.arange(1536), occ)
    pos, occ_worst, idle_worst, n_checked = 0, 0.0, 0.0, 0
    for m in chunks:
        _, n_out, pw = ctx.demod(np.ascontiguousarray(cap[None, pos:pos + m]), m, want_baseband=False, want_power=True)
        sl = F.chunk_outputs(pos, m, 400)
        assert n_out == sl.stop - sl.start
        if n_out == 0:
            assert not np.isfinite(pw).any()
        else:
            p_ref = np.mean(np.abs(ref_c[sl]) ** 2, axis=0)
            p_got = 10.0 ** ((pw.astype(np.float64) - 30.0) / 10.0)
            absolute = np.abs(p_got - p_ref) / (2 * np.sqrt(p_ref) * e + e * e)
            abs_ch = np.arange(1536)
            if mask[sl].any():           # past the filters' fill at the stream start
                occ_worst = max(occ_worst, float(np.max(np.abs(p_got[occ] / p_ref[occ] - 1))))
                abs_ch = idle
            idle_worst = max(idle_worst, float(np.max(absolute[abs_ch])))
            n_checked += 1
        pos += m
    ctx.close()
    print(f"channelizer power: {n_checked} chunks, occupied relative {occ_worst:.2e}, idle {idle_worst:.2f} of the bar")
    assert n_checked >= 7
    assert occ_worst < CH_PW_BAR and idle_worst < 1.0, (occ_worst, idle_worst)


def test_channelizer_power_bar_separates_mutants():
    """The occupied channels of the channelizer capture: dropping the first or last output of a chunk, or doubling any,
    moves that channel's power by >= MARGIN x CH_PW_BAR."""
    from oracle import pfb_oracle as pfb
    cap, occupied = _channelizer_capture()
    n = len(cap)
    chunks = CH_CHUNKS_HEAD + [n - sum(CH_CHUNKS_HEAD)]
    c = pfb.channel_filter(pfb.channelize(cap))[:, sorted(occupied)]
    p = np.abs(c) ** 2
    mask = np.stack([F.conditioned(c[:, j]) for j in range(c.shape[1])], axis=1)
    pos, n_checked = 0, 0
    for m in chunks:
        sl = F.chunk_outputs(pos, m, 400)
        for j in range(c.shape[1]):
            if mask[sl, j].any():        # the outputs while the filters fill carry next to no power
                share = p[sl, j][mask[sl, j]].min() / p[sl, j].sum()
                assert share >= MARGIN * CH_PW_BAR, (pos, m, j, share)
                n_checked += 1
        pos += m
    assert n_checked >= 4 * c.shape[1]
