"""Float64 restatement of the demod chain (reference src/demod.rs:82-134).

ORACLE -- TEST INFRASTRUCTURE ONLY.  The C++ oracle (pyoracle.DemodChain) runs the chain in float32, sample by sample,
like the reference; this module computes the same numbers in float64 with whole-array filters, so that the CUDA
kernels can be held to a bar well below the float32 oracle's own rounding (tests/test_demod_f64.py).

Conventions (those of the oracle's Decimator and FmDemod):
  * x holds the stream from absolute sample 0; in front of it the stream is complex zero (for u8 input too: no byte
    encodes 0.0, the zeros are not the LUT value of any byte).
  * /5 stage:  yd[m] = sum_k hd[k] x[5 m + 4 - k];  /10 front stage (2.4 MS/s input): ya[j] = sum_k hf[k] x[10 j + 9 - k].
  * channel filter on every 48 kHz sample: c[m] = sum_k hc[k] yd[m - k].  Power is computed on c.
  * discriminator d[m] = arg(c[m] conj(c[m - 1])) * FM_GAIN, c[-1] = 0; baseband = 10-term mean of d.
"""
from __future__ import annotations

import os
import sys

import numpy as np
from scipy import signal

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", "spec"))
import p25_spec as S  # noqa: E402

BOXCAR = S.BOXCAR_LEN


def spec_taps() -> dict:
    """The fp32-rounded spec taps the kernels and the C++ oracle use, as float64."""
    return {"front": S.taps_front().astype(np.float64), "decim": S.taps_decim().astype(np.float64),
            "chan": S.taps_chan().astype(np.float64)}


def u8_to_c128(raw: np.ndarray) -> np.ndarray:
    """Interleaved u8 IQ bytes -> complex128 through the spec's table."""
    lut = S.iq_lut().astype(np.float64)
    raw = np.asarray(raw, dtype=np.uint8).reshape(-1)
    return lut[raw[0::2]] + 1j * lut[raw[1::2]]


def discriminate(c: np.ndarray) -> np.ndarray:
    """FM discriminator (c[-1] = 0) and the 10-term boxcar."""
    prev = np.concatenate([[0.0], c[:-1]])
    d = np.angle(c * np.conj(prev)) * float(S.FM_GAIN)
    return signal.lfilter(np.ones(BOXCAR) / BOXCAR, 1.0, d)


# stage name -> (decimation, phase of the newest input): output j reads the stage input at D j + phase - k
_STAGE = {"front": (10, 9), "decim": (5, 4), "chan": (1, 0)}


def stages(x: np.ndarray, dec: int, taps: dict | None = None) -> dict:
    """Every stage's input and output: {"front": x (dec 50 only), "decim": 240 kS/s, "chan": 48 kS/s, "c", "bb"};
    each stage name keys that stage's input."""
    assert dec in (5, 50), dec
    h = spec_taps()
    if taps:
        h.update({k: np.asarray(v, dtype=np.float64) for k, v in taps.items()})
    out = {"taps": h}
    y = np.asarray(x, dtype=np.complex128)
    for st in (("front", "decim", "chan") if dec == 50 else ("decim", "chan")):
        out[st] = y
        D, ph = _STAGE[st]
        y = signal.lfilter(h[st], 1.0, y)[ph::D]
    out["c"], out["bb"] = y, discriminate(y)
    return out


def chain(x: np.ndarray, dec: int, taps: dict | None = None):
    """x: complex128 from absolute sample 0; dec: 5 (240 kS/s input) or 50 (2.4 MS/s input).
    taps optionally overrides "front", "decim" and/or "chan".  Returns (c, baseband): the channel-filter output and the
    boxcar output, len(x) // dec samples each."""
    s = stages(x, dec, taps)
    return s["c"], s["bb"]


def tap_mutant(s: dict, stage: str, k: int):
    """chain() with tap k of `stage` set to zero, from the stages() of the unmutated chain: the stage is linear, so its
    output loses h[k] times its input delayed by k; the stages after it are recomputed.  Returns (c, baseband)."""
    D, ph = _STAGE[stage]
    xin, h = s[stage], s["taps"][stage]
    order = [st for st in ("front", "decim", "chan") if st in s]
    nxt = order.index(stage) + 1
    y_ref = s[order[nxt]] if nxt < len(order) else s["c"]
    idx = D * np.arange(len(y_ref)) + ph - k
    y = y_ref - h[k] * np.where(idx >= 0, xin[np.maximum(idx, 0)], 0)
    for st in order[nxt:]:
        Ds, phs = _STAGE[st]
        y = signal.lfilter(s["taps"][st], 1.0, y)[phs::Ds]
    return y, discriminate(y)


def chunk_outputs(a0: int, n: int, dec: int) -> slice:
    """The outputs a chunk of n input samples starting at absolute input sample a0 delivers."""
    return slice(a0 // dec, (a0 + n) // dec)


def chunk_power_dbm(c: np.ndarray, a0: int, n: int, dec: int) -> float:
    """Mean |c|^2 over the chunk's outputs in dBm (R = 1 ohm), as p25cu_demod reports it; -inf for a chunk without one."""
    cc = c[chunk_outputs(a0, n, dec)]
    if len(cc) == 0:
        return -np.inf
    return 30.0 + 10.0 * np.log10(np.mean(np.abs(cc) ** 2))


def conditioned(c: np.ndarray) -> np.ndarray:
    """Outputs whose discriminator inputs c[m-10 .. m] all have |c| >= 0.1 rms(|c|) (c = 0 in front of the stream):
    where the carrier fades towards zero the discriminator's rounding error grows like 1/|c|, so a bar stated in
    absolute baseband units applies to the other outputs only."""
    a = np.abs(c)
    bad = (a < 0.1 * np.sqrt(np.mean(a ** 2))).astype(np.int64)
    cs = np.concatenate([np.zeros(BOXCAR + 1, np.int64), np.cumsum(bad)])   # cs[j + 11] = bad[0] + ... + bad[j]
    m = np.arange(len(c))
    n_bad = cs[m + BOXCAR + 1] - cs[m]                                        # bad[m - 10 .. m]
    return (n_bad == 0) & (m >= BOXCAR)
