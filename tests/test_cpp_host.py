"""The C++ host layer (include/p25cu.hpp): builds everywhere, runs on the GPU box in the reference's driver shapes."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "spec"))

from tools import p25tx as tx  # noqa: E402


def build_host_main(out_dir):
    """Link tests/cpp/p25host_main.cpp against the built library into out_dir: the source tree may be read-only."""
    lib_dir = os.path.join(ROOT, "p25rx_b200")
    exe = os.path.join(str(out_dir), "p25host_main")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-Wextra", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "p25host_main.cpp"), "-o", exe,
                           "-L", lib_dir, "-lp25cu", f"-Wl,-rpath,{lib_dir}"])
    return exe


def test_cpp_host_layer_compiles_and_links(tmp_path):
    import p25rx_b200
    p25rx_b200.build()
    exe = build_host_main(tmp_path)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 2 and "usage" in r.stderr            # no GPU work without arguments


def _parse(out: str):
    ev, pw, bb, st, voice = [], [], [], {}, None
    for line in out.splitlines():
        t = line.split()
        if t[0] == "E":
            ev.append((int(t[1]), int(t[2]), int(t[3]), bytes.fromhex(t[5]) if len(t) > 5 else b""))
        elif t[0] == "P":
            pw.append((int(t[1]), int(t[2]), float(t[3])))
        elif t[0] == "B":
            bb.append((int(t[1]), int(t[2])))
        elif t[0] == "S":
            st[t[1]] = (int(t[2]), int(t[3]), int(t[4]))
        elif t[0] == "V":
            voice = int(t[1])
    return ev, pw, bb, st, voice


@pytest.mark.gpu
def test_cpp_replay_receiver_matches_oracle(tmp_path):
    from oracle import pyoracle as po
    from p25rx_b200 import consumers as co
    exe = build_host_main(tmp_path)
    paths, ref, ref_stats, n_voice = [], [], np.zeros((12, 4), dtype=np.uint64), 0
    po.lib().p25o_set_always_correlate(0)
    for s in range(3):
        st = tx.traffic_channel(700 + s, 2) if s != 1 else tx.control_channel(700 + s, 6)
        bb, _ = tx.baseband_48k(st.dibits, snr_db=13, seed=s)
        bb = bb[:20000]
        path = tmp_path / f"r{s}.f32"
        with open(path, "wb") as f:
            co.write_baseband(f, bb)
        paths.append(str(path))
        o = po.MessageReceiver(stream=s)
        e = o.feed(bb)
        ref += [(int(x["stream"]), int(x["sample"]), int(x["kind"]), bytes(x["payload"][: int(x["len"])])) for x in e]
        ref_stats += o.stats()
        n_voice += int(np.count_nonzero(e["kind"] == 6))
    r = subprocess.run([exe, "replay"] + paths, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    ev, _, _, st, voice = _parse(r.stdout)
    assert sorted(ev) == sorted(ref) and voice == n_voice > 10
    # per stream the delivery order is feed()'s order
    for s in range(3):
        samples = [e[1] for e in ev if e[0] == s]
        assert samples == sorted(samples)
    from p25rx_b200 import STATS_FAMILIES
    for i, name in enumerate(STATS_FAMILIES):
        assert st[name] == (int(ref_stats[i, 0]), int(ref_stats[i, 1]), int(ref_stats[i, 3])), name


@pytest.mark.gpu
def test_cpp_demod_task_and_receiver_match_oracle(tmp_path):
    from oracle import pyoracle as po
    exe = build_host_main(tmp_path)
    po.lib().p25o_set_always_correlate(0)
    paths, ref, ref_pw, n_chunks = [], [], {}, 6
    for s in range(2):
        st = tx.control_channel(720 + s, 8)
        raw = tx.iq_to_u8(tx.modulate_iq(st.dibits, 240_000, snr_db=24, cfo_hz=35.0 * s, seed=s, amplitude=0.4))
        raw = raw[: 32768 * n_chunks + 1000]                      # a trailing partial chunk is dropped
        path = tmp_path / f"iq{s}.u8"
        raw.tofile(path)
        paths.append(str(path))
        chain, o = po.DemodChain(po.FMT_U8, False), po.MessageReceiver(stream=s)
        for c in range(n_chunks):
            bb, pw = chain.feed(raw[32768 * c: 32768 * (c + 1)], want_power=True)
            ref_pw[(c, s)] = pw
            ref += [(int(x["stream"]), int(x["sample"]), int(x["kind"]), bytes(x["payload"][: int(x["len"])])) for x in o.feed(bb)]
    r = subprocess.run([exe, "sdr"] + paths, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    ev, pw, bb, st, _ = _parse(r.stdout)
    assert sorted(ev) == sorted(ref) and len(ev) > 30
    assert [n for _, n in bb] == [(16384 * (c + 1)) // 5 - (16384 * c) // 5 for c in range(n_chunks)]   # 3276 / 3277
    assert sorted({c for c, _, _ in pw}) == [0, 4]                # every 4th chunk (src/demod.rs:67)
    for c, s, v in pw:
        assert abs(v - ref_pw[(c, s)]) < 1e-2
    assert st["viterbiDibit"][0] == sum(1 for e in ev if e[2] == 7)


# ------------------------------------------------------------------ SURVEY 8f rank 2 in the compiled host layer
def _chan_params(ident, base_hz=851_012_500, spacing_hz=12_500, bw_hz=12_500, offset=(1, 45)):
    v = (ident << 60) | ((bw_hz // 125) << 51) | (((0x100 if offset[0] > 0 else 0) | offset[1]) << 42) | ((spacing_hz // 125) << 32) | (base_hz // 5)
    return v.to_bytes(8, "big")


def _consumer_units():
    """TSBKs and link-control words whose fields the reference's consumers read (src/recv.rs:237-342, src/hub.rs:346-443)."""
    ch = lambda ident, number: ((ident << 12) | number).to_bytes(2, "big")
    sysid, wacn = 0x2A5, 0xBEE07
    status = bytes([0x11, 0x10 | (sysid >> 8), sysid & 0xFF, 0x07, 0x21]) + ch(1, 0x155) + bytes([0x70])
    tsbks = [
        (0x3D, _chan_params(1)),                                                            # ChannelParamsUpdate
        (0x00, bytes([0x04]) + ch(1, 0x123) + (0x4567).to_bytes(2, "big") + (0xABCDEF).to_bytes(3, "big")),   # GroupVoiceGrant
        (0x02, ch(1, 0x010) + (100).to_bytes(2, "big") + ch(2, 0x020) + (200).to_bytes(2, "big")),           # update: id 2 unknown
        (0x02, ch(1, 0x011) + (0xFFFF).to_bytes(2, "big") + ch(1, 0x012) + (0x0001).to_bytes(2, "big")),     # Everybody / Default: skipped
        (0x3A, status), (0x3C, status),                                                     # RfssStatus, AdjacentSite
        (0x3B, bytes([0x11, wacn >> 12, (wacn >> 4) & 0xFF, ((wacn & 0xF) << 4) | (sysid >> 8), sysid & 0xFF]) + ch(1, 0x155) + bytes([0x70])),
        (0x39, bytes([0x07, 0x21]) + ch(1, 0x200) + bytes([0x70]) + ch(3, 0x201) + bytes([0x70])),            # AltControl: id 3 unknown
        (0x2B, bytes([0x01, 0x12, 0x34, 0x07, 0x21]) + (0x00BEEF).to_bytes(3, "big")),       # LocRegResponse
        (0x2C, bytes([0x20 | (sysid >> 8), sysid & 0xFF]) + (0x123456).to_bytes(3, "big") + (0x654321).to_bytes(3, "big")),
        (0x2F, bytes([0x00, wacn >> 12, (wacn >> 4) & 0xFF, ((wacn & 0xF) << 4) | (sysid >> 8), sysid & 0xFF]) + (0x00CAFE).to_bytes(3, "big")),
        (0x15, bytes(8)),                                                                   # unknown opcode: ignored
    ]
    lcs = [bytes([0x00, 0x00, 0x00, 0x00, 0x45, 0x67, 0xAB, 0xCD, 0xEF]),                  # GroupVoiceTraffic -> srcUnit
           bytes([0x02]) + ch(1, 0x030) + (300).to_bytes(2, "big") + ch(1, 0x031) + (301).to_bytes(2, "big"),   # GroupVoiceUpdate
           bytes([0x23]) + status, bytes([0x0F]) + bytes(8)]
    return tsbks, lcs


def _consumer_events():
    """The same units as a drained event array (for the Python side) and as `fields` arguments (for the C++ side)."""
    from p25rx_b200 import EVENT_DTYPE
    tsbks, lcs = _consumer_units()
    rows = [(7, tx.make_tsbk(op, 0, pl, last=False)) for op, pl in tsbks]
    rows.insert(3, (7, tx.make_tsbk(0x00, 0, tsbks[1][1], last=False, bad_crc=True)))       # CRC failure: dropped
    rows.insert(4, (7, tx.make_tsbk(0x00, 0x90, tsbks[1][1], last=False)))                  # manufacturer-specific: dropped
    rows += [(3, lcs[0]), (3, lcs[1]), (8, lcs[2]), (8, lcs[3])]
    ev = np.zeros(len(rows), dtype=EVENT_DTYPE)
    for i, (k, pl) in enumerate(rows):
        ev[i]["kind"], ev[i]["sample"], ev[i]["len"] = k, i, len(pl)
        ev[i]["payload"][: len(pl)] = np.frombuffer(pl, dtype=np.uint8)
    return ev, [f"{k}:{pl.hex()}" for k, pl in rows]


def _parse_consumer(out: str):
    import json
    tg = [tuple(int(x) for x in line.split()[1:5]) for line in out.splitlines() if line.startswith("T ")]
    hub = [(int(line.split()[1]), json.loads(line.split(" ", 2)[2])) for line in out.splitlines() if line.startswith("H ")]
    return tg, hub


def test_cpp_consumer_fields_match_python_adapters(tmp_path):
    """include/p25cu.hpp TsbkFields / LinkControlFields / fields:: / ChannelParamsMap / RecvConsumer against
    p25rx_b200/consumers.py on hand-built payloads (no GPU): talkgroups with their traffic-channel frequency and the
    hub's status JSON, including what must be dropped (bad CRC, manufacturer id, reserved talkgroups, unknown channel ids)."""
    import json
    import p25rx_b200
    from p25rx_b200 import consumers as co
    p25rx_b200.build()
    exe = build_host_main(tmp_path)
    ev, argv = _consumer_events()
    r = subprocess.run([exe, "fields"] + argv, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    tg, hub = _parse_consumer(r.stdout)
    ptg, phub = co.consume(ev)
    assert tg == ptg and [t[2] for t in tg] == [0x4567, 100, 300, 301]
    assert tg[0][3] == 851_012_500 + 12_500 * 0x123
    assert hub == [(s, json.loads(j)) for s, j in phub]
    names = [h[1]["event"] for h in hub]
    assert names == ["rfssStatus", "adjacentSite", "networkStatus", "altControl", "locReg", "unitReg", "unitDereg", "srcUnit", "rfssStatus"]
    assert hub[2][1]["payload"] == {"area": 0x11, "wacn": 0xBEE07, "system": 0x2A5}
    assert hub[1][1]["payload"]["freq"] == 851_012_500 + 12_500 * 0x155 and hub[7][1]["payload"] == 0xABCDEF


@pytest.mark.gpu
def test_cpp_consumer_view_of_decoded_streams(tmp_path):
    """The consumer view end to end on the GPU path: recordings carrying those TSBKs and link-control words, decoded by
    the CUDA library; p25host_main's RecvConsumer output must equal consumers.consume() over the Python host layer's
    events of the same files."""
    import json
    import p25rx_b200 as p25
    from p25rx_b200 import consumers as co
    exe = build_host_main(tmp_path)
    tsbks, lcs = _consumer_units()
    units = []
    for i in range(0, len(tsbks), 3):
        grp = tsbks[i:i + 3]
        units.append(tx.tsdu(0x293, [tx.make_tsbk(op, 0, pl, last=(j == len(grp) - 1)) for j, (op, pl) in enumerate(grp)]))
    rng = np.random.default_rng(9)
    voice = [tx.hdu(0x293, bytes(9), 0, 0x80, 0, 0x4567),
             tx.ldu(0x293, 1, [tx.random_imbe(rng) for _ in range(9)], lcs[0], (1, 2)),
             tx.ldu(0x293, 2, [tx.random_imbe(rng) for _ in range(9)], bytes(9) + bytes([0x80, 0, 0]), (3, 4)),
             tx.ldu(0x293, 1, [tx.random_imbe(rng) for _ in range(9)], lcs[1], (5, 6)),
             tx.tdulc(0x293, lcs[2])]
    paths = []
    # stream 1 learns channel id 1 from its own TSDU before the link-control update arrives (one RecvTask per stream)
    bbs = [tx.baseband_48k(tx.concat_units(us, lead_idle=30, gap_idle=12).dibits, snr_db=22, seed=s)[0]
           for s, us in enumerate((units, [tx.tsdu(0x293, [tx.make_tsbk(0x3D, 0, _chan_params(1), last=True)])] + voice))]
    n = max(len(b) for b in bbs)           # replay ends with the shortest recording: pad with an idle carrier
    for s, bb in enumerate(bbs):
        bb = np.concatenate([bb, np.zeros(n - len(bb), dtype=np.float32)])
        path = tmp_path / f"c{s}.f32"
        with open(path, "wb") as f:
            co.write_baseband(f, bb)
        paths.append(str(path))
    r = subprocess.run([exe, "consumer"] + paths, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    tg, hub = _parse_consumer(r.stdout)
    rr = p25.ReplayReceiver(n_streams=2)
    ev = rr.replay([open(pth, "rb") for pth in paths])
    rr.ctx.close()
    ev = ev[np.lexsort((ev["sample"], ev["stream"]))]
    ptg, phub = co.consume(ev)
    assert tg == ptg and hub == [(s, json.loads(j)) for s, j in phub]
    assert {t[2] for t in tg} == {0x4567, 100, 300, 301}
    assert {h[1]["event"] for h in hub} >= {"rfssStatus", "adjacentSite", "networkStatus", "altControl", "locReg", "unitReg", "unitDereg", "srcUnit"}
