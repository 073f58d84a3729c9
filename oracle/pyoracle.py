"""ctypes binding of the CPU oracle (oracle/libp25oracle.so).

ORACLE -- TEST INFRASTRUCTURE ONLY.  PARITY UNPINNED (see p25_oracle.hpp).
Importable from tests/, __graft_entry__.smoke() and bench.py's CPU legs only; the
product package p25rx_b200 never imports this module.
"""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

FMT_U8, FMT_CF32 = 0, 1

EVENT_DTYPE = np.dtype([("stream", "<u4"), ("kind", "<u4"), ("sample", "<u8"), ("len", "<u4"),
                        ("payload", "u1", (60,))], align=True)
assert EVENT_DTYPE.itemsize == 80


_native_dir: str | None = None


def build(native: bool = False) -> str:
    """(Re)build the oracle if its sources are newer than the library.  The -march=native copy is built once per process
    into a temporary directory: it fits only the host it was compiled on, and the source tree may be read-only."""
    global _native_dir
    if native:
        if _native_dir is None:
            d = tempfile.mkdtemp(prefix="p25oracle-")
            atexit.register(shutil.rmtree, d, ignore_errors=True)
            subprocess.check_call(["make", "-C", HERE, "native", "NATIVE_LIB=" + os.path.join(d, "libp25oracle_native.so")],
                                  stdout=subprocess.DEVNULL)
            _native_dir = d
        return os.path.join(_native_dir, "libp25oracle_native.so")
    path = os.path.join(HERE, "libp25oracle.so")
    srcs = [os.path.join(HERE, f) for f in ("p25_oracle.cpp", "p25_oracle.hpp", "p25_tables.h", "Makefile")]
    if not os.path.exists(path) or any(os.path.getmtime(s) > os.path.getmtime(path) for s in srcs):
        subprocess.check_call(["make", "-C", HERE, "all"], stdout=subprocess.DEVNULL)
    return path


_libs: dict[bool, C.CDLL] = {}


def lib(native: bool = False) -> C.CDLL:
    if native in _libs:
        return _libs[native]
    L = C.CDLL(build(native))
    vp, sz, u32p, fp = C.c_void_p, C.c_size_t, C.POINTER(C.c_uint32), C.POINTER(C.c_float)
    L.p25o_demod_new.restype = vp
    L.p25o_demod_new.argtypes = [C.c_int, C.c_int]
    L.p25o_demod_free.argtypes = [vp]
    L.p25o_demod_feed.restype = sz
    L.p25o_demod_feed.argtypes = [vp, vp, sz, vp, fp]
    L.p25o_recv_new.restype = vp
    L.p25o_recv_free.argtypes = [vp]
    L.p25o_recv_resync.argtypes = [vp]
    L.p25o_recv_state.argtypes = [vp]
    L.p25o_recv_feed.restype = sz
    L.p25o_recv_feed.argtypes = [vp, vp, sz, vp, sz, C.c_uint32]
    L.p25o_recv_stats.argtypes = [vp, vp, C.c_int]
    L.p25o_bch_decode.argtypes = [C.c_uint64, C.POINTER(C.c_uint16), C.POINTER(C.c_int)]
    for n in ("golay23", "golay24", "golay18", "hamming15", "hamming10", "cyclic16"):
        getattr(L, f"p25o_{n}_decode").argtypes = [C.c_uint32, u32p]
    L.p25o_rs_decode.argtypes = [vp, C.c_int, C.c_int]
    L.p25o_trellis_half_decode.argtypes = [vp, vp]
    L.p25o_trellis_34_decode.argtypes = [vp, vp]
    L.p25o_imbe_decode.argtypes = [vp, vp, vp]
    L.p25o_crc_ccitt.restype = C.c_uint32
    L.p25o_crc_ccitt.argtypes = [vp, C.c_int]
    L.p25o_batch_run.restype = sz
    L.p25o_batch_run.argtypes = [C.c_int, C.c_int, vp, sz, sz, C.c_int, vp, sz, vp]
    L.p25o_set_always_correlate.argtypes = [C.c_int]
    _libs[native] = L
    return L


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


class DemodChain:
    """One stream's DemodTask::run body (reference src/demod.rs:70-117)."""

    def __init__(self, fmt: int, front, native: bool = False):
        """front: False / 0 = reference chain (/5), True / 1 = /10 front stage first (2.4 MS/s input),
        2 = input already at 48 kS/s (a channelizer output): 48 kHz stages only."""
        self._L = lib(native)
        self._h = self._L.p25o_demod_new(fmt, int(front))
        self.fmt, self.front = fmt, int(front)

    def __del__(self):
        if getattr(self, "_h", None):
            self._L.p25o_demod_free(self._h)
            self._h = None

    def feed(self, iq: np.ndarray, want_power: bool = False):
        if self.fmt == FMT_U8:
            iq = np.ascontiguousarray(iq, dtype=np.uint8)
            n = iq.size // 2
        else:
            iq = np.ascontiguousarray(iq, dtype=np.complex64)
            n = iq.size
        out = np.empty(n // {0: 5, 1: 50, 2: 1}[self.front] + 2, dtype=np.float32)
        p = C.c_float(0)
        m = self._L.p25o_demod_feed(self._h, _ptr(iq), n, _ptr(out), C.byref(p) if want_power else None)
        return (out[:m], p.value) if want_power else out[:m]


class MessageReceiver:
    """p25::message::receiver::MessageReceiver as driven by reference src/replay.rs:40-57."""

    def __init__(self, stream: int = 0, native: bool = False):
        self._L = lib(native)
        self._h = self._L.p25o_recv_new()
        self.stream = stream

    def __del__(self):
        if getattr(self, "_h", None):
            self._L.p25o_recv_free(self._h)
            self._h = None

    def feed(self, samples: np.ndarray, cap: int | None = None) -> np.ndarray:
        s = np.ascontiguousarray(samples, dtype=np.float32)
        cap = cap or (s.size // 400 + 64)
        ev = np.zeros(cap, dtype=EVENT_DTYPE)
        n = self._L.p25o_recv_feed(self._h, _ptr(s), s.size, _ptr(ev), cap, self.stream)
        if n > cap:
            raise RuntimeError(f"event buffer too small: {n} > {cap}")
        return ev[:n]

    def resync(self):
        self._L.p25o_recv_resync(self._h)

    @property
    def state(self) -> int:
        return self._L.p25o_recv_state(self._h)

    def stats(self, clear: bool = False) -> np.ndarray:
        out = np.zeros((12, 4), dtype=np.uint64)
        self._L.p25o_recv_stats(self._h, _ptr(out), int(clear))
        return out


def batch_run(fmt: int, front: bool, iq: np.ndarray, n_streams: int, n_per_stream: int, threads: int,
              cap_per_stream: int = 0, native: bool = False):
    """S independent (DemodChain + MessageReceiver) pairs over `threads` host threads."""
    L = lib(native)
    counts = np.zeros(n_streams, dtype=np.uint32)
    ev = np.zeros(max(1, n_streams * cap_per_stream), dtype=EVENT_DTYPE)
    total = L.p25o_batch_run(fmt, int(front), _ptr(iq), n_streams, n_per_stream, threads,
                             _ptr(ev) if cap_per_stream else None, cap_per_stream, _ptr(counts))
    return total, counts, ev.reshape(n_streams, -1) if cap_per_stream else None
