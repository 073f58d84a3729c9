"""Oracle demod chain (reference src/demod.rs:82-114) against the float64 restatement (oracle/demod_f64.py)."""
import numpy as np
import pytest
from oracle import demod_f64 as F
from tools import p25tx as tx
from util import check_against_truth


@pytest.mark.parametrize("front", [False, True])
def test_cf32_chain_matches_scipy(oracle, front):
    fs = 2_400_000 if front else 240_000
    st = tx.control_channel(1, 1)
    iq = tx.modulate_iq(st.dibits, fs, snr_db=30, cfo_hz=100.0, seed=1)[: fs // 20]
    got = oracle.DemodChain(oracle.FMT_CF32, front).feed(iq)
    ref = F.chain(iq, 50 if front else 5)[1]
    assert len(got) == len(iq) // (50 if front else 5)
    assert np.max(np.abs(got - ref[: len(got)])) < 2e-5


def test_u8_chain_and_lut(oracle):
    st = tx.control_channel(2, 1)
    iq = tx.modulate_iq(st.dibits, 240_000, snr_db=30, seed=2)[:16384]
    u8 = tx.iq_to_u8(iq)
    got = oracle.DemodChain(oracle.FMT_U8, False).feed(u8)
    ref = F.chain(F.u8_to_c128(u8), 5)[1]
    assert len(got) == 3276                      # floor(16384 / 5), reference src/demod.rs:87
    assert np.max(np.abs(got - ref[:3276])) < 2e-5


def test_chunking_and_phase_carry(oracle):
    """16,384 is not a multiple of 5: the decimator phase must persist (reference src/demod.rs:87)."""
    st = tx.control_channel(3, 5)
    iq = tx.modulate_iq(st.dibits, 240_000, snr_db=25, seed=3)[: 5 * 16384]
    assert len(iq) == 5 * 16384
    whole = oracle.DemodChain(oracle.FMT_CF32, False).feed(iq)
    dc = oracle.DemodChain(oracle.FMT_CF32, False)
    parts = [dc.feed(iq[i:i + 16384]) for i in range(0, len(iq), 16384)]
    assert [len(p) for p in parts] == [3276, 3277, 3277, 3277, 3277]
    assert np.array_equal(np.concatenate(parts), whole)


def test_power_dbm(oracle):
    n = 16384
    iq = (0.25 * np.exp(2j * np.pi * 1000 * np.arange(n) / 240000)).astype(np.complex64)
    _, p = oracle.DemodChain(oracle.FMT_CF32, False).feed(iq, want_power=True)
    assert abs(p - (30 + 10 * np.log10(0.25 ** 2))) < 0.2     # reference src/demod.rs:123-134


@pytest.mark.parametrize("fmt,front", [("cf32", False), ("u8", False), ("cf32", True)])
def test_iq_to_events(oracle, fmt, front):
    fs = 2_400_000 if front else 240_000
    st = tx.control_channel(4, 3)
    iq = tx.modulate_iq(st.dibits, fs, snr_db=20, cfo_hz=150.0, timing_offset=2.5, seed=5)
    if fmt == "u8":
        bb = oracle.DemodChain(oracle.FMT_U8, front).feed(tx.iq_to_u8(iq))
    else:
        bb = oracle.DemodChain(oracle.FMT_CF32, front).feed(iq)
    check_against_truth(oracle.MessageReceiver().feed(bb), tx.expected_events(st))
