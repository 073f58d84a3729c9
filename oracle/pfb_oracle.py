"""CPU restatement of the wideband channelizer (float64 numpy).

ORACLE -- TEST INFRASTRUCTURE ONLY.  The reference (kchmck/p25rx) has no channelizer: one RTL-SDR tuner, one
channel, retuned by hopping (reference src/sdr.rs:61-68, src/recv.rs:127-137); BASELINE.json configs[2] asks for
one, so its behaviour is defined by spec/p25_spec.py (PFB_* constants, taps_pfb) and restated here twice:

  channel_direct  the definition: mix down by k * 12.5 kHz, prototype low-pass, keep every 400th output
  channelize      the same numbers through the polyphase identity and numpy's FFT

tests/test_pfb_oracle.py checks the two against each other; the GPU kernels (p25rx_b200/csrc/pfb.cu) are
checked against channelize().  Everything after the channelizer is the reference's own 48 kHz chain
(oracle.pyoracle.DemodChain(..., front=2)).
"""
from __future__ import annotations

import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", "spec"))
import p25_spec as S  # noqa: E402

N, M, P = S.PFB_CHANNELS, S.PFB_DECIM, S.PFB_TAPS_PER_BRANCH
L = N * P


def _taps() -> np.ndarray:
    return S.taps_pfb().astype(np.float64)


def channel_direct(x: np.ndarray, k: int, m: np.ndarray) -> np.ndarray:
    """y_k[m] = sum_i h[i] x[n_m - i] exp(-2j pi k (n_m - i) / N), n_m = M m + M - 1; x[n] = 0 for n < 0."""
    h = _taps()
    x = np.asarray(x, dtype=np.complex128)
    out = np.zeros(len(m), dtype=np.complex128)
    i = np.arange(L)
    for j, mm in enumerate(np.asarray(m)):
        idx = M * int(mm) + M - 1 - i
        ok = idx >= 0
        xs = np.zeros(L, dtype=np.complex128)
        xs[ok] = x[idx[ok]]
        ph = np.exp(-2j * np.pi * ((k * idx) % N) / N)
        out[j] = np.sum(h * xs * ph)
    return out


def channelize(x: np.ndarray, m0: int = 0, n_out: int | None = None) -> np.ndarray:
    """All channels for output times m0 .. m0 + n_out - 1: returns [n_out][N] complex128.
    x holds the stream from absolute sample 0 (zeros before it)."""
    h = _taps().reshape(P, N)                       # h[p][r] = h[r + N p]
    x = np.asarray(x, dtype=np.complex128)
    if n_out is None:
        n_out = len(x) // M - m0
    xp = np.concatenate([np.zeros(L, dtype=np.complex128), x])   # xp[L + n] = x[n]
    out = np.empty((n_out, N), dtype=np.complex128)
    r = np.arange(N)
    for j in range(n_out):
        nm = M * (m0 + j) + M - 1
        win = xp[L + nm - L + 1: L + nm + 1][::-1]              # win[i] = x[nm - i], i = 0 .. L-1
        v = np.sum(h * win.reshape(P, N), axis=0)               # v[r] = sum_p h[r + N p] x[nm - r - N p]
        u = v[(r + nm) % N]
        out[j] = np.fft.ifft(u) * N                             # sum_q u[q] exp(+2j pi k q / N)
    return out


def channel_filter(y: np.ndarray) -> np.ndarray:
    """The reference's channel-select FIR (src/demod.rs:93) down every channel column of y [n_out][N], zeros before the
    stream start: c_k[m] = sum_j hc[j] y_k[m - j].  This is what the CUDA kernels deliver as channel spectra: they fold
    the filter into the polyphase prototype (p25rx_b200/csrc/pfb.cu)."""
    hc = S.taps_chan().astype(np.float64)
    y = np.asarray(y, dtype=np.complex128)
    out = np.zeros_like(y)
    for j, h in enumerate(hc[: len(y)]):
        out[j:] += h * y[: len(y) - j]
    return out


def equivalent_prototype() -> np.ndarray:
    """heq = hp (*) upsample(hc, M): the prototype whose polyphase channelizer output equals channel_filter(channelize(x))."""
    hp, hc = _taps(), S.taps_chan().astype(np.float64)
    heq = np.zeros(L + M * (len(hc) - 1), dtype=np.float64)
    for j, h in enumerate(hc):
        heq[M * j: M * j + L] += h * hp
    return heq


def channelize_fused(x: np.ndarray, m0: int = 0, n_out: int | None = None) -> np.ndarray:
    """channel_filter(channelize(x)) computed the way the kernels do: one polyphase pass with the equivalent prototype
    (15 taps per branch), float32-rounded taps like the device table."""
    heq = equivalent_prototype()
    PE = -(-len(heq) // N)
    h = np.zeros(PE * N)
    h[: len(heq)] = heq.astype(np.float32).astype(np.float64)
    h = h.reshape(PE, N)
    LE = PE * N
    x = np.asarray(x, dtype=np.complex128)
    if n_out is None:
        n_out = len(x) // M - m0
    xp = np.concatenate([np.zeros(LE, dtype=np.complex128), x])
    out = np.empty((n_out, N), dtype=np.complex128)
    r = np.arange(N)
    for j in range(n_out):
        nm = M * (m0 + j) + M - 1
        win = xp[nm + 1: LE + nm + 1][::-1]                     # win[i] = x[nm - i], i = 0 .. LE-1
        v = np.sum(h * win.reshape(PE, N), axis=0)
        out[j] = np.fft.ifft(v[(r + nm) % N]) * N
    return out


# ------------------------------------------------------------------ the fused form, vectorised, for any tap vector
PE = 15                                   # taps per branch of the equivalent prototype (pfb.cu PE)
LE = PE * N                               # 23,040: the equivalent prototype zero-padded (pfb.cu LE)
P_LO, P_HI = -1, PE + 1                   # coefficient slots identify_taps fits per branch: p = -1 .. 15


def device_taps() -> np.ndarray:
    """The kernels' tap table h32 (float64 copy of float32 values, length LE): heq rounded once to float32, accumulated in
    double in the order p25cu_pfb_upload uses (pfb.cu), the padding zero."""
    heq = equivalent_prototype()
    h = np.zeros(LE)
    h[: len(heq)] = heq.astype(np.float32)
    return h


def _windows(xp: np.ndarray, off: int, nm0: int, T: int) -> np.ndarray:
    """View X[t, p, r] = xp[off + nm0 + M t - r - N p] (no copy): the LE samples behind output times nm0, nm0 + M, ..."""
    s = xp.strides[0]
    assert off + nm0 - (LE - 1) >= 0 and off + nm0 + M * (T - 1) < len(xp)
    return np.lib.stride_tricks.as_strided(xp[off + nm0:], shape=(T, PE, N), strides=(M * s, -N * s, -s), writeable=False)


def channelize_taps(x: np.ndarray, h: np.ndarray | None = None, m0: int = 0, n_out: int | None = None,
                    block: int = 256) -> np.ndarray:
    """c[m][k] = sum_i h[i] x[n_m - i] exp(-2j pi k (n_m - i) / N), n_m = M m + M - 1, for m = m0 .. m0 + n_out - 1:
    [n_out][N] complex128.  h has LE taps (default device_taps()); x holds the stream from absolute sample 0 (zeros
    before it).  The fused polyphase form of channelize_fused, over blocks of output times at once."""
    H = (device_taps() if h is None else np.asarray(h, dtype=np.float64)).reshape(PE, N)
    x = np.asarray(x, dtype=np.complex128)
    if n_out is None:
        n_out = len(x) // M - m0
    assert len(x) >= M * (m0 + n_out), "x must reach the newest sample of the last output time"
    xp = np.concatenate([np.zeros(LE, dtype=np.complex128), x])
    out = np.empty((n_out, N), dtype=np.complex128)
    r = np.arange(N)
    for j0 in range(0, n_out, block):
        T = min(block, n_out - j0)
        nm = M * (m0 + j0 + np.arange(T)) + M - 1
        X = _windows(xp, LE, int(nm[0]), T)
        v = H[0] * X[:, 0, :]
        for p in range(1, PE):
            v += H[p] * X[:, p, :]                              # v[t][r] = sum_p h[r + N p] x[n_m - r - N p]
        u = np.take_along_axis(v, (r[None, :] + nm[:, None]) % N, axis=1)
        out[j0: j0 + T] = np.fft.ifft(u, axis=1) * N
    return out


def channelize_f32(x: np.ndarray, m0: int = 0, n_out: int | None = None, block: int = 256) -> np.ndarray:
    """A float32 model of the kernel's arithmetic for the noise model of the device tests: channelize_taps with the
    branch sums accumulated in float32 and a complex64 inverse FFT (scipy keeps the precision).  Not the kernel's
    operation order, only its precision."""
    from scipy import fft as sfft
    H = device_taps().astype(np.float32).reshape(PE, N)
    x = np.asarray(x, dtype=np.complex64)
    if n_out is None:
        n_out = len(x) // M - m0
    xp = np.concatenate([np.zeros(LE, dtype=np.complex64), x])
    out = np.empty((n_out, N), dtype=np.complex64)
    r = np.arange(N)
    for j0 in range(0, n_out, block):
        T = min(block, n_out - j0)
        nm = M * (m0 + j0 + np.arange(T)) + M - 1
        X = _windows(xp, LE, int(nm[0]), T)
        v = H[0] * X[:, 0, :]
        for p in range(1, PE):
            v = v + H[p] * X[:, p, :]
        u = np.take_along_axis(v, (r[None, :] + nm[:, None]) % N, axis=1)
        out[j0: j0 + T] = sfft.ifft(u, axis=1, norm="forward")
    return out


def window_rms(x: np.ndarray, m0: int, n_out: int) -> np.ndarray:
    """|x|rms over the LE samples behind each output time (zeros before the stream start): the scale of that output's
    float32 rounding error."""
    p = np.concatenate([np.zeros(LE + 1), np.cumsum(np.abs(np.asarray(x, dtype=np.complex128)) ** 2)])   # p[LE + n + 1]
    nm = M * (m0 + np.arange(n_out)) + M - 1
    return np.sqrt((p[LE + nm + 1] - p[nm + 1]) / LE)


def branch_sums(c: np.ndarray, m0: int) -> np.ndarray:
    """Invert the inverse DFT: v_m[r] = fft(c[m])[(r - n_m) mod N] / N, [n_out][N] complex128."""
    c = np.asarray(c)
    nm = M * (m0 + np.arange(len(c))) + M - 1
    V = np.fft.fft(c.astype(np.complex128), axis=1) / N
    return np.take_along_axis(V, (np.arange(N)[None, :] - nm[:, None]) % N, axis=1)


class TapFit:
    """identify_taps' result.  coef[p - P_LO][r]: the complex coefficient of x[n_m - r - N p], p = -1 .. 15; table():
    the LE entries h[r + N p], p = 0 .. 14; sigma: the standard error of each coefficient (|complex| error); resid: the
    weighted residual rms per output time, per capture; resid_rms over all."""

    def __init__(self, coef, sigma, resid, resid_rms):
        self.coef, self.sigma, self.resid, self.resid_rms = coef, sigma, resid, resid_rms

    def table(self, a: np.ndarray | None = None) -> np.ndarray:
        a = self.coef if a is None else a
        return a[-P_LO: -P_LO + PE].reshape(-1)


def _regressors(xps, nms, ws, rb: np.ndarray) -> np.ndarray:
    """A[b, row, p - P_LO] = w x[n_m - r_b - N p] over all captures' rows, for the branches rb."""
    P_ = np.arange(P_LO, P_HI)
    out = []
    for xp, nm, w in zip(xps, nms, ws):
        idx = (LE + N + nm)[None, :, None] - rb[:, None, None] - N * P_[None, None, :]
        out.append(xp[idx] * w[None, :, None])
    return np.concatenate(out, axis=1)


def _prep(x, m0, n_rows, scale):
    xs = x if isinstance(x, (list, tuple)) else [x]
    m0s = m0 if isinstance(m0, (list, tuple)) else [m0] * len(xs)
    scales = scale if isinstance(scale, (list, tuple)) else [scale] * len(xs)
    xps, nms, ws = [], [], []
    for xx, mm, nr, sc in zip(xs, m0s, n_rows, scales):
        xx = np.asarray(xx, dtype=np.complex128)
        xps.append(np.concatenate([np.zeros(LE + N, dtype=np.complex128), xx, np.zeros(N, dtype=np.complex128)]))
        nms.append(M * (mm + np.arange(nr)) + M - 1)
        ws.append(np.broadcast_to(1.0 / np.asarray(sc, dtype=np.float64), (nr,)))
    return xps, nms, ws, m0s


def tap_sigma(x, m0, n_out, noise: float, scale=1.0, branch_block: int = 16) -> np.ndarray:
    """The standard error identify_taps would give each coefficient [17][N] if the weighted residual had rms `noise`:
    noise * sqrt(diag((A^H A)^-1)) per branch.  x, m0, n_out and scale may be lists (one entry per capture)."""
    n_caps = len(x) if isinstance(x, (list, tuple)) else 1
    ns = n_out if isinstance(n_out, (list, tuple)) else [n_out] * n_caps
    xps, nms, ws, _ = _prep(x, m0, ns, scale)
    out = np.empty((P_HI - P_LO, N))
    for r0 in range(0, N, branch_block):
        rb = np.arange(r0, min(N, r0 + branch_block))
        A = _regressors(xps, nms, ws, rb)
        G = np.conj(np.swapaxes(A, 1, 2)) @ A
        out[:, rb] = noise * np.sqrt(np.diagonal(np.linalg.inv(G), axis1=1, axis2=2).real).T
    return out


def identify_taps(x, c, m0=0, scale=1.0, branch_block: int = 16) -> TapFit:
    """The effective taps of a channelizer from its delivered spectra c[m][k] (output times m0 ..): per branch r, the
    complex least-squares coefficients of x[n_m - r - N p], p = -1 .. 15, against the branch sums v_m[r] recovered by
    branch_sums().  p = 0 .. 14 are the table's taps; p = -1 (a sample after n_m) and p = 15 (a sixteenth, older slot)
    must come out zero, and a tap applied to one component of x only comes out non-real.  Rows are weighted by 1/scale
    (the capture's |x|rms), so the residual is in units of the input level.  x, c, m0 and scale may be lists, one entry
    per capture (fitted together).  Works in blocks of branch_block branches (~80 MB for 18,000 rows)."""
    cs = c if isinstance(c, (list, tuple)) else [c]
    xps, nms, ws, m0s = _prep(x, m0, [len(cc) for cc in cs], scale)
    vs = [branch_sums(cc, mm) * w[:, None] for cc, mm, w in zip(cs, m0s, ws)]
    n_rows = sum(len(v) for v in vs)
    K = P_HI - P_LO
    coef = np.empty((K, N), dtype=np.complex128)
    sigma = np.empty((K, N))
    res2 = [np.zeros(len(v)) for v in vs]
    for r0 in range(0, N, branch_block):
        rb = np.arange(r0, min(N, r0 + branch_block))
        A = _regressors(xps, nms, ws, rb)                                    # [B][rows][17]
        y = np.concatenate([v[:, rb] for v in vs], axis=0).T[:, :, None]     # [B][rows][1]
        AH = np.conj(np.swapaxes(A, 1, 2))
        Gi = np.linalg.inv(AH @ A)
        a = Gi @ (AH @ y)
        e = (y - A @ a)[:, :, 0]                                             # [B][rows]
        s2 = np.sum(np.abs(e) ** 2, axis=1) / (n_rows - K)
        coef[:, rb] = a[:, :, 0].T
        sigma[:, rb] = np.sqrt(s2[:, None] * np.diagonal(Gi, axis1=1, axis2=2).real).T
        row = 0
        for i, v in enumerate(vs):
            res2[i] += np.sum(np.abs(e[:, row: row + len(v)]) ** 2, axis=0)
            row += len(v)
    resid = [np.sqrt(r2 / N) for r2 in res2]
    return TapFit(coef, sigma, resid, float(np.sqrt(sum(np.sum(r2) for r2 in res2) / (n_rows * N))))
