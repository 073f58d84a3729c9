"""The wideband channelizer (pfb.cu, p25_pfbc_kernel) against the float64 fused polyphase form (oracle/pfb_oracle.py).

Per-output max-abs bars cannot see most of the 22,144-tap equivalent prototype: zeroing tap i moves an output by about
|h_i| |x|, while float32 rounding moves it by ~1.5e-8 |x|, so every tap below ~2e-4 of the peak would drop out unseen.
These tests pool over many outputs instead:

  * TAP IDENTIFICATION.  The inverse DFT is invertible, so the delivered spectra give back every output time's branch
    sums; per branch, a least-squares fit against the input recovers the taps the kernel actually applied, each with a
    standard error sigma_i.  Every coefficient must lie within TAP_Z sigma_i (plus REL_TAP |h_i|, below) of the device
    table h32, and the coefficients of the sample a window may hold early (p = -1) and of a sixteenth slot (p = 15)
    within TAP_Z sigma_i of zero.  The CPU part shows the estimator is exact in float64, that it returns each tap
    mutant exactly, and that >= 99 % of the taps are resolved (|h_i| >= MARGIN (TAP_Z sigma_i + REL_TAP |h_i|)) at the
    noise level NOISE_REL of a float32 model of the kernel; the rest are all below 1e-7 of the peak.
  * EVERY OUTPUT.  Every channel of every output time -- stream start, chunk starts, run starts, tail -- within
    OUT_BAR of the local input level (|x|rms over the LE samples behind the output).
  * BASEBAND, BOTH KERNEL PATHS.  The discriminator and boxcar after the channelizer (the production path that packs two
    output times per atan2, and the per-time path the spectra hook selects) against the float64 discriminator and boxcar
    of the float64 spectra: carrier channels within BB_BAR (conditioned outputs once the filters have filled), every
    output of every channel within bb_bound (the error OUT_BAR allows through the discriminator, plus the atan2 and
    boxcar rounding; a discriminator value within that error of +-pi may land on the other side, a whole 2 pi).  The CPU
    part shows that a discriminator restarted at a run start, a wrong pair hand-off, a 9- or 11-term boxcar or a warm-up
    one output short each move a carrier's baseband by >= MARGIN x bb_bound.

Noise model (test_noise_model_and_resolved_taps): channelize_f32 -- float32 branch sums, complex64 FFT -- on the device
tests' stimuli.  NOISE_REL is 3x its weighted branch-sum residual rms on the white noise, OUT_BAR 3x its largest spectra
error per stimulus, both relative to |x|rms.  REL_TAP: the kernel's inverse DFT is a fixed linear map built from float32
constants (twiddles, sqrt(1/2), cos(pi/6)); each input passes at most six of them, each within 2^-24, so the map differs
from the exact DFT by at most ~6 x 2^-24 relative, and its diagonal scales each identified tap by that much at most (the
float32 model shows up to 7e-8, the B200 4.4e-8).  2^-21 covers that bound.

What these bars cannot reach: taps below the resolved threshold (all < 1e-7 of the peak, printed by the CPU test); a
time-variant fault confined to one tail-tap slot at one run start (a few products out of millions: the fit pools over all
output times, the per-output bar sees |h_i| |x| only for taps above ~2e-4 of the peak); and, on the carriers, baseband
errors between BB_BAR and bb_bound: at the carrier stimulus' OUT_BAR the worst case of bb_bound reaches a few BB_BAR, so
BB_BAR is held directly there, not derived from the spectra bar."""
import numpy as np
import p25_spec as S
import pytest
from oracle import demod_f64 as F
from oracle import pfb_oracle as PO
from test_demod_f64 import BB_BAR, CH_CHUNKS_HEAD, MARGIN, _channelizer_capture

N, M = PO.N, PO.M
TAP_Z = 6
REL_TAP = 2.0 ** -21          # relative allowance of an identified tap: the float32 constants of the inverse DFT
NOISE_REL = 2.5e-10           # branch-sum residual rms / |x|rms: 3x the float32 model (test_noise_model_and_resolved_taps)
# per-output spectra error / local |x|rms, per stimulus: 3x the float32 model's largest.  A capture of a few strong
# carriers puts its energy into few channels and its largest rounding errors are ~7x those of white noise at the same
# |x|rms (the rms error is the same), so each stimulus has its own bar.
OUT_BAR = {"white": 5.0e-8, "carrier": 4.0e-7}
ATAN2_RAD, ATAN2_REL = 2e-7, 1.5e-7   # kernel atan2 error (float32 products + polynomial) <= 2e-7 + 1.5e-7 |angle| rad
FILL = -(-PO.LE // PO.M) + 10           # output times until the prototype and the boxcar lie inside the stream
FM_GAIN = float(S.FM_GAIN)

# identification stimulus: complex white Gaussian noise at three levels (|x|rms), ragged chunks
LEVELS = (0.02, 0.07, 0.3)
T_ID = 6000
N_ID = M * T_ID + 211                                        # ends with a partial output time


def _id_chunks(n: int):
    head = CH_CHUNKS_HEAD + [600_011, 3, 999_997]
    return head + [n - sum(head)]


def _id_captures():
    xs = []
    for i, lv in enumerate(LEVELS):
        rng = np.random.default_rng(500 + i)
        x = lv / np.sqrt(2) * (rng.standard_normal(N_ID) + 1j * rng.standard_normal(N_ID))
        xs.append(x.astype(np.complex64))
    return xs


def _carrier_chunks(n: int):
    return CH_CHUNKS_HEAD + [n - sum(CH_CHUNKS_HEAD)]


# ------------------------------------------------------------------ the baseband bound
def _box_sum(a: np.ndarray, lo: int, hi: int) -> np.ndarray:
    """s[m] = sum_{j = m - lo .. m - hi} a[j] along axis 0 (a[j] = 0 for j < 0)."""
    cs = np.concatenate([np.zeros((lo + 1,) + a.shape[1:]), np.cumsum(a, axis=0)])   # cs[j + lo + 1] = a[0] + .. + a[j]
    m = np.arange(len(a))
    return cs[m - hi + lo + 1] - cs[m]


def _disc(c: np.ndarray) -> np.ndarray:
    """Discriminator values d[m] = FM_GAIN arg(c[m] conj(c[m-1])), c[-1] = 0, along axis 0."""
    prev = np.concatenate([np.zeros_like(c[:1]), c[:-1]])
    return np.angle(c * np.conj(prev)) * FM_GAIN


def discriminate(c: np.ndarray) -> np.ndarray:
    """demod_f64.discriminate along axis 0 of [n_out][channels]."""
    return _box_sum(_disc(c), F.BOXCAR - 1, 0) / F.BOXCAR


def bb_bound(c: np.ndarray, xrms: np.ndarray, out_bar: float):
    """The largest baseband error a spectra error within out_bar x xrms[m] allows at each output of c [n_out][channels]
    (float64 reference spectra), and where that bound is defined: every discriminator input c[m-10 .. m] has
    E <= 0.1 |c| (then arg moves by at most asin(E / |c|) <= 1.002 E / |c|).  c[m-10] and c[m] enter one discriminator
    value of the 10-term boxcar, c[m-9 .. m-1] two.  Added: the kernel's atan2 error, the mean over the ten values of
    (ATAN2_RAD + ATAN2_REL |angle|) x FM_GAIN (a float32 model of atan2_branchfree over 4 M random arguments stays within
    0.74 of that envelope; a flat 2e-7 rad would not hold near |angle| = pi, where float32 itself rounds to 1.2e-7), and
    the float32 rounding of FM_GAIN x angle, the boxcar tree and the 1/10 scale."""
    a = np.abs(c)
    e = out_bar * np.asarray(xrms)[:, None] / np.maximum(a, 1e-300)
    ok = e <= 0.1
    w = _box_sum(e, 10, 0) + _box_sum(e, 9, 1)                             # weights 1, 2 x 9, 1
    d = _disc(c)
    bb = _box_sum(d, 9, 0) / F.BOXCAR
    rnd = 2.0 ** -24 * _box_sum(np.abs(d), 9, 0) + 4e-8 * np.abs(bb)
    at2 = (ATAN2_RAD * F.BOXCAR + ATAN2_REL * _box_sum(np.abs(d), 9, 0) / FM_GAIN) * FM_GAIN / F.BOXCAR
    bound = FM_GAIN / F.BOXCAR * 1.002 * w + at2 + rnd
    defined = (_box_sum((~ok).astype(np.float64), 10, 0) == 0) & (np.arange(len(c)) >= F.BOXCAR)[:, None]
    return bound, defined


# ------------------------------------------------------------------ CPU: the reference, the estimator, the bars
def test_channelize_taps_equals_fused_and_two_stage():
    """channelize_taps with the device table equals channelize_fused (the same sums), and with the unrounded heq the
    two-stage definition channel_filter(channelize(x)), to 1e-12 of the output scale: stream start, an m0, the tail."""
    rng = np.random.default_rng(7)
    n = M * 140 + 321
    x = 0.1 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    got = PO.channelize_taps(x)
    ref = PO.channelize_fused(x)
    scale = np.max(np.abs(ref))
    assert got.shape == ref.shape == (140, N)
    assert np.max(np.abs(got - ref)) <= 1e-12 * scale
    heq = np.zeros(PO.LE)
    heq[: len(PO.equivalent_prototype())] = PO.equivalent_prototype()
    two = PO.channel_filter(PO.channelize(x))
    assert np.max(np.abs(PO.channelize_taps(x, heq) - two)) <= 1e-12 * scale
    assert np.max(np.abs(PO.channelize_taps(x, m0=61, n_out=70) - got[61:131])) <= 1e-12 * scale


def _coef_table(h: np.ndarray, early=None, late=None) -> np.ndarray:
    """[17][N] coefficients p = -1 .. 15 for a tap table h (LE) and optional early / sixteenth-slot rows."""
    out = np.zeros((PO.P_HI - PO.P_LO, N))
    out[1:1 + PO.PE] = h.reshape(PO.PE, N)
    if early is not None:
        out[0] = early
    if late is not None:
        out[-1] = late
    return out


def _mutant_spectra(x: np.ndarray, coef: np.ndarray, m0: int, n_out: int, comp: tuple | None = None) -> np.ndarray:
    """Spectra of a channelizer whose branch r applies coef[p + 1][r] to x[n_m - r - N p], p = -1 .. 15.
    comp = (r, p, hr): that one product uses hr on the real part of x only (a one-component tap)."""
    xp = np.concatenate([np.zeros(PO.LE + N, dtype=np.complex128), x, np.zeros(N, dtype=np.complex128)])
    nm = M * (m0 + np.arange(n_out)) + M - 1
    v = np.zeros((n_out, N), dtype=np.complex128)
    r = np.arange(N)
    for k, p in enumerate(range(PO.P_LO, PO.P_HI)):
        v += coef[k][None, :] * xp[(PO.LE + N + nm)[:, None] - r[None, :] - N * p]
    if comp is not None:
        rr, p, hr = comp
        v[:, rr] += hr * xp[PO.LE + N + nm - rr - N * p].real
    return np.fft.ifft(np.take_along_axis(v, (r[None, :] + nm[:, None]) % N, axis=1), axis=1) * N


def test_identify_taps_is_exact_and_returns_each_mutant():
    """In float64 the estimator returns h32 to 1e-13 of the peak, and a mutant's taps exactly: a zeroed tail tap, a
    scaled tap, a tap moved to another branch, a tap moved to the other parity of its branch, non-zero p = -1 and
    p = 15 coefficients; a tap applied to the real part of x only comes back as a non-real coefficient (h/2) with a
    residual far above NOISE_REL."""
    rng = np.random.default_rng(11)
    n = M * 600 + 99
    x = 0.07 / np.sqrt(2) * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    h = PO.device_taps()
    peak = np.max(np.abs(h))
    fit = PO.identify_taps(x, PO.channelize_taps(x), 0, scale=0.07)
    assert np.max(np.abs(fit.table() - h)) <= 1e-13 * peak
    assert np.max(np.abs(fit.coef[0])) <= 1e-13 * peak and np.max(np.abs(fit.coef[-1])) <= 1e-13 * peak
    tail = int(np.nonzero(np.abs(h) > 0)[0][-1])                # the last non-zero tap
    big = int(np.argmax(np.abs(h)))
    mutants = {}
    hz = h.copy(); hz[tail] = 0.0
    mutants["zeroed tail tap"] = _coef_table(hz)
    hs = h.copy(); hs[big] *= 1.5
    mutants["scaled tap"] = _coef_table(hs)
    hb = h.copy(); hb[big + 1] += hb[big]; hb[big] = 0.0
    mutants["tap on the wrong branch"] = _coef_table(hb)
    hp = h.copy(); hp[big + N] += hp[big]; hp[big] = 0.0
    mutants["tap on the wrong parity (p)"] = _coef_table(hp)
    early = np.zeros(N); early[17] = h[big]
    mutants["early sample p = -1"] = _coef_table(h, early=early)
    late = np.zeros(N); late[1000] = h[1000 + 14 * N] + 1e-9
    mutants["sixteenth slot p = 15"] = _coef_table(h, late=late)
    for name, coef in mutants.items():
        c = _mutant_spectra(x, coef, 0, 600)
        f = PO.identify_taps(x, c, 0, scale=0.07)
        assert np.max(np.abs(f.coef - coef)) <= 1e-13 * peak, name
    r_, p_ = big % N, big // N
    coef = _coef_table(h)
    coef[p_ + 1][r_] = 0.0
    f = PO.identify_taps(x, _mutant_spectra(x, coef, 0, 600, comp=(r_, p_, h[big])), 0, scale=0.07)
    got = f.coef[p_ + 1][r_]
    assert abs(got.real - h[big] / 2) < 0.05 * h[big] and f.resid_rms > 1e3 * NOISE_REL, (got, f.resid_rms)


def _model_error(x: np.ndarray, n_out: int) -> tuple:
    ref = PO.channelize_taps(x, n_out=n_out)
    em = PO.channelize_f32(x, n_out=n_out).astype(np.complex128)
    return float(np.max(np.abs(em - ref) / PO.window_rms(x, 0, n_out)[:, None])), em


def _noise_model():
    """channelize_f32 on the first 1,000 output times of each identification capture and on the whole carrier capture:
    (largest per-output spectra error / local |x|rms per stimulus, weighted branch-sum residual rms of the fit, largest
    relative tap bias of taps > 1e-4, worst z)."""
    xs = [x.astype(np.complex128) for x in _id_captures()]
    n_em = 1000
    out_max, cs = {"white": 0.0}, []
    for x in xs:
        e, em = _model_error(x, n_em)
        out_max["white"] = max(out_max["white"], e)
        cs.append(em)
    cap, _ = _channelizer_capture()
    out_max["carrier"] = _model_error(cap.astype(np.complex128), len(cap) // M)[0]
    fit = PO.identify_taps(xs, cs, 0, scale=list(LEVELS))
    coef = _coef_table(PO.device_taps())
    big = np.abs(coef) > 1e-4
    bias = float(np.max(np.abs(fit.coef - coef)[big] / np.abs(coef[big])))
    z = np.max(np.maximum(np.abs(fit.coef - coef) - REL_TAP * np.abs(coef), 0) / fit.sigma)
    return out_max, fit.resid_rms, bias, float(z), n_em * len(xs)


def test_noise_model_and_resolved_taps():
    """NOISE_REL and OUT_BAR are 3x the float32 model's residual and largest errors (within 10 %); the model itself passes
    the identification bar; with sigma_i from NOISE_REL for the device test's stimulus (3 captures x 6,000 output
    times), >= 99 % of the 22,144 taps are resolved and every unresolved tap is below 1e-7 of the peak."""
    out_max, resid, bias, z, n_em = _noise_model()
    print(f"\nfloat32 model: spectra error max " +
          ", ".join(f"{k} {v:.3e} |x|rms (OUT_BAR {OUT_BAR[k]:.1e} = {OUT_BAR[k] / v:.2f}x)" for k, v in out_max.items()) +
          f"; {n_em} white-noise output times: branch-sum residual rms {resid:.3e} |x|rms (NOISE_REL {NOISE_REL:.1e} = "
          f"{NOISE_REL / resid:.2f}x), largest relative tap bias {bias:.1e} (REL_TAP {REL_TAP:.1e}), worst z {z:.2f}")
    for k, v in out_max.items():
        assert 2.7 <= OUT_BAR[k] / v <= 3.3, k
    assert 2.7 <= NOISE_REL / resid <= 3.3
    assert bias < REL_TAP and z <= TAP_Z
    xs = [x.astype(np.complex128) for x in _id_captures()]
    sig = PO.tap_sigma(xs, 0, T_ID, NOISE_REL, scale=list(LEVELS))
    h = PO.device_taps()
    peak = np.max(np.abs(h))
    sig_t = sig[1:1 + PO.PE].reshape(-1)
    n_taps = len(PO.equivalent_prototype())
    real = np.arange(PO.LE) < n_taps
    resolved = np.abs(h) >= MARGIN * (TAP_Z * sig_t + REL_TAP * np.abs(h))
    n_res = int(np.count_nonzero(resolved & real))
    worst_unres = float(np.max(np.abs(h[real & ~resolved]), initial=0.0)) / peak
    print(f"sigma {np.median(sig_t):.2e} (median), resolved taps {n_res} of {n_taps}, largest unresolved tap "
          f"{worst_unres:.2e} of the peak")
    assert n_res >= 0.99 * n_taps
    assert n_res == RESOLVED_TAPS
    assert worst_unres < 1e-7


RESOLVED_TAPS = 21994         # pinned: test_noise_model_and_resolved_taps


def _carrier_reference():
    cap, occupied = _channelizer_capture()
    x = cap.astype(np.complex128)
    n_out = len(x) // M
    return x, PO.channelize_taps(x), PO.window_rms(x, 0, n_out), sorted(occupied)


def _carrier_mask(c: np.ndarray) -> np.ndarray:
    """Where a carrier channel is held to BB_BAR: its conditioned outputs once the filters have filled (m >= FILL).  While
    they fill, |c| ramps up from zero and the bar OUT_BAR allows more; there the output is held to bb_bound only."""
    mk = F.conditioned(c)
    mk[:FILL] = False
    return mk


def test_bb_bound_on_carriers():
    """On the carrier capture's occupied channels the derived bound is defined on every conditioned output, and on >= 90 %
    of every channel's outputs.  It does not stay within BB_BAR: at the carrier stimulus' OUT_BAR the worst case, every
    discriminator input off by the full bar in the worst direction, reaches a few BB_BAR.  The carriers are held to BB_BAR
    directly (the bar of tests/test_demod_f64.py) and every output to bb_bound."""
    x, c, xr, occ = _carrier_reference()
    bound, defined = bb_bound(c, xr, OUT_BAR["carrier"])
    worst = 0.0
    for k in occ:
        assert np.all(defined[F.conditioned(c[:, k]), k]), k
        mk = _carrier_mask(c[:, k])
        worst = max(worst, float(np.max(bound[mk, k])))
    print(f"\nlargest bb_bound on the carriers' conditioned outputs past the fill {worst:.2e} (BB_BAR {BB_BAR:.1e})")
    assert defined[:, occ].mean(axis=0).min() >= 0.9


def _box(d: np.ndarray, lo: int, hi: int) -> np.ndarray:
    return _box_sum(d, lo, hi) / F.BOXCAR


def test_48k_mutants_exceed_the_bound():
    """Each fault of the 48 kHz side, restated on the float64 chain of the carrier capture, moves the baseband of some
    carrier channel's conditioned output by >= MARGIN x bb_bound: at >= 90 % of the possible run starts for the
    discriminator restart (c[m-1] = 0), the zeroed boxcar history and the warm-up one output short; on both parities for
    the pair hand-off from c[m-2]; anywhere for a 9- or 11-term boxcar."""
    x, c, xr, occ = _carrier_reference()
    c = c[:, occ]
    bound, _ = bb_bound(c, xr, OUT_BAR["carrier"])
    mask = np.stack([_carrier_mask(c[:, j]) for j in range(c.shape[1])], axis=1)
    lim = np.where(mask, MARGIN * bound, np.inf)
    d = _disc(c)
    bb = _box(d, 9, 0)
    T = len(c)
    starts = np.arange(2 * F.BOXCAR + 2, T - 2 * F.BOXCAR)

    def hit(delta, rows):
        return bool(np.any(np.abs(delta) >= lim[rows]))

    out = {}
    # discriminator restarted at b: d[b] = 0, seen by bb[b .. b+9]
    out["restart c[m-1] = 0"] = np.mean([hit(np.broadcast_to(d[b], (10, d.shape[1])) / F.BOXCAR, slice(b, b + 10))
                                         for b in starts])
    # boxcar history zeroed at b: bb[m], m = b .. b+8, loses d[m-9 .. b-1]
    cs = np.cumsum(d, axis=0)

    def hist_delta(b):
        m = np.arange(b, b + 9)
        return (cs[b - 1][None, :] - cs[m - 10]) / F.BOXCAR
    out["boxcar history zeroed"] = np.mean([hit(hist_delta(b), slice(b, b + 9)) for b in starts])
    # warm-up one output short: bb[b] loses d[b-9]
    out["warm-up one short"] = np.mean([hit(d[b - 9][None, :] / F.BOXCAR, slice(b, b + 1)) for b in starts])
    ratio = {}
    for par in (0, 1):
        prev2 = np.concatenate([np.zeros_like(c[:2]), c[:-2]])
        dm = d.copy()
        sel = np.arange(T) % 2 == par
        dm[sel] = np.angle(c[sel] * np.conj(prev2[sel])) * FM_GAIN
        ratio[f"pair hand-off c[m-2], parity {par}"] = np.abs(_box(dm, 9, 0) - bb) / lim
    ratio["9-term boxcar"] = np.abs(_box(d, 8, 0) - bb) / lim
    ratio["11-term boxcar"] = np.abs(_box(d, 10, 0) - bb) / lim
    print()
    for name, frac in out.items():
        print(f"{name}: caught at {100 * frac:.1f} % of {len(starts)} run starts")
    for name, r in ratio.items():
        print(f"{name}: largest change {float(np.max(r[np.isfinite(r)])):.1f} x MARGIN x bb_bound")
    for name, frac in out.items():
        assert frac >= 0.9, (name, frac)
    for name, r in ratio.items():
        assert np.max(r[np.isfinite(r)]) >= 1.0, name


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def p25():
    import p25rx_b200
    return p25rx_b200


def _run(p25, caps, chunks, spectra: bool):
    """All captures [C][n] through one channelizer context in the given chunks.  Returns (baseband [C * N][n_out],
    spectra [C][n_out][N] or None)."""
    C = len(caps)
    ctx = p25.Context(C * N, fmt=p25.FMT_CF32_IQ, decimation=M, max_chunk_samples=max(chunks))
    ctx.keep_spectra(spectra)
    bbs, ys, pos = [], [], 0
    arr = np.stack(caps)
    for m in chunks:
        bb, n_out, _ = ctx.demod(np.ascontiguousarray(arr[:, pos:pos + m]), m)
        bbs.append(bb)
        if spectra and n_out:
            ys.append(ctx.channelizer_output())
        pos += m
    ctx.close()
    return np.concatenate(bbs, axis=1), (np.concatenate(ys, axis=1) if spectra else None)


@pytest.fixture(scope="module")
def runs(p25):
    """The identification captures and the carrier capture, each through the kernel with the spectra kept (per-time
    path) and without (paired-atan2 path), with their float64 references."""
    ids = _id_captures()
    cap, occupied = _channelizer_capture()
    out = {}
    for name, caps, chunks, occ in (("white", ids, _id_chunks(N_ID), []),
                                    ("carrier", [cap], _carrier_chunks(len(cap)), sorted(occupied))):
        bb_slow, y = _run(p25, caps, chunks, True)
        bb_fast, _ = _run(p25, caps, chunks, False)
        xs = [c.astype(np.complex128) for c in caps]
        out[name] = dict(xs=xs, y=y, bb_slow=bb_slow, bb_fast=bb_fast, occ=occ)
    return out


@pytest.mark.gpu
def test_tap_identification(runs):
    """The taps the kernel applied, recovered from its spectra over 3 x 6,000 output times of white noise at three
    levels: every coefficient (the 23,040 table entries, padding included, and the p = -1 / p = 15 slots of all 1,536
    branches) within TAP_Z sigma_i + REL_TAP |h32_i| of the table; the residual within NOISE_REL."""
    r = runs["white"]
    fit = PO.identify_taps(r["xs"], [y for y in r["y"]], 0, scale=list(LEVELS))
    coef = _coef_table(PO.device_taps())
    dev = np.abs(fit.coef - coef)
    z = np.maximum(dev - REL_TAP * np.abs(coef), 0) / fit.sigma
    zr = dev / fit.sigma
    w = np.unravel_index(int(np.argmax(z)), z.shape)
    print(f"\ntap identification: worst z {z.max():.2f} at p = {w[0] - 1}, r = {w[1]} (without the REL_TAP allowance "
          f"{zr.max():.1f}); largest relative deviation of taps > 1e-4 "
          f"{float(np.max(dev[np.abs(coef) > 1e-4] / np.abs(coef[np.abs(coef) > 1e-4]))):.1e}; residual rms "
          f"{fit.resid_rms:.3e} |x|rms (NOISE_REL {NOISE_REL:.1e}); median sigma {np.median(fit.sigma):.2e}")
    assert fit.coef.shape == (17, N)
    assert z.max() <= TAP_Z, (z.max(), w)
    assert fit.resid_rms <= NOISE_REL


@pytest.mark.gpu
def test_every_output_against_float64(runs):
    """Every channel of every output time of both stimuli (stream start, chunk and run starts, the tail) within OUT_BAR
    of the float64 fused form, relative to the local |x|rms."""
    worst = {}
    for name, r in runs.items():
        for i, x in enumerate(r["xs"]):
            y = r["y"][i]
            n_out = len(x) // M
            assert y.shape == (n_out, N)
            ref = PO.channelize_taps(x, n_out=n_out)
            err = np.abs(y.astype(np.complex128) - ref) / PO.window_rms(x, 0, n_out)[:, None]
            worst[f"{name}{i}"] = float(err.max())
            assert worst[f"{name}{i}"] <= OUT_BAR[name], (name, i, worst)
    print("\nspectra error / local |x|rms: " + ", ".join(f"{k} {v:.2e}" for k, v in worst.items()) +
          f" (OUT_BAR {OUT_BAR})")


def _check_baseband(bb: np.ndarray, c: np.ndarray, xr: np.ndarray, out_bar: float, occ, where: str, stats: dict,
                    skip: int = 0):
    """bb [n_out][channels] from the kernel against discriminate(c)[skip:] (c has `skip` lead-in outputs): carriers
    within BB_BAR on conditioned outputs past the filters' fill, every output within bb_bound where it is defined, the
    bound defined on >= 90 % of each channel's outputs."""
    assert skip == 0 or skip >= FILL
    ref = discriminate(c)[skip:]
    bound, defined = bb_bound(c, xr, out_bar)
    bound, defined = bound[skip:], defined[skip:]
    err = np.abs(bb.astype(np.float64) - ref)
    # a discriminator value within the atan2 allowance of +-pi may come out on the other side: each such value of the
    # boxcar window may move the output by a whole 2 pi FM_GAIN / 10
    q = 2 * np.pi * FM_GAIN / F.BOXCAR
    e = out_bar * np.asarray(xr)[:, None] / np.maximum(np.abs(c), 1e-300)
    tol = 1.002 * (e + np.concatenate([np.zeros_like(e[:1]), e[:-1]])) + ATAN2_RAD + ATAN2_REL * np.pi
    near = _box_sum((np.pi - np.abs(_disc(c) / FM_GAIN) <= tol).astype(np.float64), 9, 0)[skip:]
    wraps = np.rint(err / q)
    err = np.where(wraps <= near, np.abs(err - wraps * q), err)
    assert defined.mean(axis=0).min() >= 0.9, where
    over = float(np.max(np.where(defined, err / bound, 0.0)))
    car = 0.0
    for k in occ:
        mk = _carrier_mask(c[:, k])[skip:]
        car = max(car, float(np.max(err[mk, k])))
    stats[where] = (car, over)
    assert over <= 1.0, (where, over)
    assert car <= BB_BAR, (where, car)


@pytest.mark.gpu
def test_baseband_both_paths(runs):
    """Baseband of every channel, both kernel paths, against the float64 chain (see _check_baseband); the two paths agree
    within twice the largest atan2 allowance on the carriers' conditioned outputs."""
    stats, pair = {}, 0.0
    for name, r in runs.items():
        for i, x in enumerate(r["xs"]):
            n_out = len(x) // M
            c = PO.channelize_taps(x, n_out=n_out)
            xr = PO.window_rms(x, 0, n_out)
            fast = r["bb_fast"][i * N:(i + 1) * N].T
            slow = r["bb_slow"][i * N:(i + 1) * N].T
            _check_baseband(fast, c, xr, OUT_BAR[name], r["occ"], f"{name}{i} paired", stats)
            _check_baseband(slow, c, xr, OUT_BAR[name], r["occ"], f"{name}{i} per-time", stats)
            for k in r["occ"]:
                mk = _carrier_mask(c[:, k])
                pair = max(pair, float(np.max(np.abs(fast[mk, k].astype(np.float64) - slow[mk, k]))))
    print("\nbaseband (carriers max |err|, max err / bb_bound): " +
          ", ".join(f"{k} {a:.2e} {b:.2f}" for k, (a, b) in stats.items()) + f"; paths differ by {pair:.2e}")
    assert pair <= 2 * (ATAN2_RAD + ATAN2_REL * np.pi) * FM_GAIN


@pytest.mark.gpu
def test_cfg3_every_stream_against_float64(p25):
    """The cfg3 bench geometry as bench.py runs it: 8 captures x 2,880,000 samples, two steps through process()
    (spectra not kept).  The second step's baseband of all 12,288 streams against the float64 chain with the bars of
    test_baseband_both_paths.  Capture g is the periodic base advanced by 77 g output times, so its steady-state spectra
    are the base's shifted and turned by a constant phase per channel, which the discriminator does not see."""
    import torch
    from bench import Workload
    wl = Workload("cfg3", 1)
    n, caps = wl.n, wl.rows
    T = n // M
    assert all(wl.shift(g) == M * 77 * g % n for g in range(caps))
    dev = wl.device_input(0)
    ctx = p25.Context(wl.streams, fmt=p25.FMT_CF32_IQ, decimation=M, max_chunk_samples=n, event_slots=64)
    torch.cuda.synchronize()
    for _ in range(2):
        ctx.process(dev, n)
        ctx.poll()
    del dev
    base = np.ascontiguousarray(wl.base()[0]).view(np.complex64).reshape(-1).astype(np.complex128)
    pre = FILL
    c = PO.channelize_taps(np.tile(base, 2), m0=T - pre, n_out=T + pre)      # steady state, FILL lead-in
    xr = PO.window_rms(np.tile(base, 2), T - pre, T + pre)
    occ = sorted((37 * i + 5) % N for i in range(64))
    stats = {}
    for g in range(caps):
        # output j of the step is period position (j + 77 g) mod T, with the pre positions before it as lead-in
        cg = np.roll(c[pre:], -77 * g, axis=0)
        cg = np.concatenate([cg[-pre:], cg])
        xg = np.roll(xr[pre:], -77 * g)
        xg = np.concatenate([xg[-pre:], xg])
        rows = np.stack([ctx.read_baseband(g * N + k, T) for k in range(N)], axis=1)   # [T][N]
        _check_baseband(rows, cg, xg, OUT_BAR["carrier"], occ, f"cap{g}", stats, skip=pre)
    ctx.close()
    print("\ncfg3 baseband (carriers max |err|, max err / bb_bound): " +
          ", ".join(f"{k} {a:.2e} {b:.2f}" for k, (a, b) in stats.items()))
