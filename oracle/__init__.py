"""ctypes loader for the CPU oracle (oracle/jsdr_oracle.c).

TEST INFRASTRUCTURE ONLY.  Importable from tests/, __graft_entry__.smoke()
and bench.py's cpu_baseline / --impl reference legs; never from the product
package.  See oracle/jsdr_oracle.h for the parity status of each function.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libjsdr_oracle.so")
INT_MIN = -2147483648


def build(force: bool = False) -> str:
    src = os.path.join(_HERE, "jsdr_oracle.c")
    hdr = os.path.join(_HERE, "jsdr_oracle.h")
    stale = (not os.path.exists(_SO)) or any(
        os.path.getmtime(f) > os.path.getmtime(_SO) for f in (src, hdr))
    if force or stale:
        subprocess.check_call(["make", "-C", _HERE, "-s"] + (["-B"] if force else []))
    return _SO


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.orc_bpsk_sizeof.restype = C.c_int
        _lib.orc_fir_filter.restype = C.c_int
        _lib.orc_fec_decode.restype = C.c_int
        _lib.orc_fec_table_probe.restype = C.c_int
        _lib.orc_baseline_fft_s16.restype = C.c_int
        _lib.orc_baseline_mixdecim_s16.restype = C.c_int
        _lib.orc_baseline_pipeline_s16.restype = C.c_int
    return _lib


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


# ---------------------------------------------------------------- ingest
def s16_to_float(raw: np.ndarray, ic: int = 0, qc: int = 0, chns: int = 2) -> np.ndarray:
    """JavaAudio.java:276-293."""
    raw = np.ascontiguousarray(raw, dtype=np.int16).ravel()
    nframes = raw.size // chns
    out = np.empty(2 * nframes, dtype=np.float32)
    lib().orc_s16_to_float(_p(raw, C.c_int16), nframes, chns, ic, qc, _p(out, C.c_float))
    return out


# ---------------------------------------------------------------- DFT / fft.java
def dft_f64(x: np.ndarray, inverse: bool = False, direct: bool = False) -> np.ndarray:
    x = np.ascontiguousarray(x, dtype=np.complex128)
    n = x.size
    out = np.empty(n, dtype=np.complex128)
    fn = lib().orc_dft_direct_f64 if direct else lib().orc_dft_f64
    fn(_p(x.view(np.float64), C.c_double), _p(out.view(np.float64), C.c_double), n, int(inverse))
    return out


def fft_receive(buf: np.ndarray, rate: int, f32plan: bool = False):
    """fft.java:190-224.  Returns (psd[n+2] float32, peak_bin)."""
    buf = np.ascontiguousarray(buf, dtype=np.float32).ravel()
    n = buf.size // 2
    psd = np.empty(n + 2, dtype=np.float32)
    pk = C.c_int(0)
    fn = lib().orc_fft_receive_f32plan if f32plan else lib().orc_fft_receive
    fn(_p(buf, C.c_float), n, rate, _p(psd, C.c_float), C.byref(pk))
    return psd, pk.value


def fft_power_f64(buf: np.ndarray) -> np.ndarray:
    buf = np.ascontiguousarray(buf, dtype=np.float32).ravel()
    n = buf.size // 2
    pw = np.empty(n, dtype=np.float64)
    lib().orc_fft_power_f64(_p(buf, C.c_float), n, _p(pw, C.c_double))
    return pw


# ---------------------------------------------------------------- fir.java
class _FirS(C.Structure):
    _fields_ = [("wfir", C.c_double * 21), ("fir", C.c_int * 21), ("fof", C.c_int)]


class Fir:
    """fir.java:169-228 (weights / filter / complex_gen / complex_mod)."""

    def __init__(self, rate: float = 44100.0):
        self.s = _FirS()
        self.rate = C.c_float(rate)
        lib().orc_fir_init(C.byref(self.s))

    def weights(self, f1: int, f2: int) -> np.ndarray:
        lib().orc_fir_weights(C.byref(self.s), f1, f2, self.rate)
        return np.array(self.s.wfir[:], dtype=np.float64)

    def filter(self, x: np.ndarray) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.int32)
        out = np.empty_like(x)
        lib().orc_fir_filter_block(C.byref(self.s), _p(x, C.c_int), _p(out, C.c_int), x.size)
        return out

    def complex_gen(self, freq: int, n0: int, count: int) -> np.ndarray:
        wav = (C.c_int * 2)(freq, n0)
        sig = (C.c_int * 2)()
        out = np.empty((count, 2), dtype=np.int32)
        for i in range(count):
            lib().orc_fir_complex_gen(sig, wav, self.rate)
            out[i, 0], out[i, 1] = sig[0], sig[1]
        return out


def complex_mod(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.int32).reshape(-1, 2)
    b = np.ascontiguousarray(b, dtype=np.int32).reshape(-1, 2)
    out = np.empty_like(a)
    aa, bb, oo = (C.c_int * 2)(), (C.c_int * 2)(), (C.c_int * 2)()
    for i in range(a.shape[0]):
        aa[0], aa[1] = int(a[i, 0]), int(a[i, 1])
        bb[0], bb[1] = int(b[i, 0]), int(b[i, 1])
        lib().orc_fir_complex_mod(aa, bb, oo)
        out[i, 0], out[i, 1] = oo[0], oo[1]
    return out


# ---------------------------------------------------------------- demod.java
class _DemodS(C.Structure):
    _fields_ = [("wfir", C.c_float * 21), ("fir", C.c_float * 42), ("fof", C.c_int),
                ("car", C.c_float), ("phi", C.c_float), ("dofir", C.c_int),
                ("dodwn", C.c_int), ("rate", C.c_int)]


class Demod:
    """demod.java:341-434 (weights / filter / FIR + NCO part of receive)."""

    def __init__(self, rate: int, dofir: bool = True, dodwn: bool = True):
        self.s = _DemodS()
        lib().orc_demod_init(C.byref(self.s), rate)
        self.s.dofir, self.s.dodwn = int(dofir), int(dodwn)

    def weights(self, flo: int, fhi: int) -> np.ndarray:
        lib().orc_demod_weights(C.byref(self.s), flo, fhi)
        return np.array(self.s.wfir[:], dtype=np.float32)

    def receive(self, buf: np.ndarray) -> np.ndarray:
        buf = np.ascontiguousarray(buf, dtype=np.float32).ravel()
        out = np.empty_like(buf)
        lib().orc_demod_receive(C.byref(self.s), _p(buf, C.c_float), buf.size // 2, _p(out, C.c_float))
        return out


def demod_phases(phi, car0, n: int) -> np.ndarray:
    """demod.java:427-429 alone: float32[n + 1], the car of each of n samples from car0 and the
    value carried after them."""
    out = np.empty(n + 1, dtype=np.float32)
    lib().orc_demod_phases(C.c_float(phi), C.c_float(car0), int(n), _p(out, C.c_float))
    return out


def demod_detect(sam: np.ndarray, mode: int, rate: int, doagc: bool, lilq: np.ndarray):
    """demod.java:405-481 on the FIR/NCO output; lilq (float32[2]) is updated in place.
    Returns (audio int16[n], max_avg float32[2])."""
    sam = np.ascontiguousarray(sam, dtype=np.float32).ravel()
    n = sam.size // 2
    audio = np.empty(n, dtype=np.int16)
    ma = np.empty(2, dtype=np.float32)
    lib().orc_demod_detect(_p(sam, C.c_float), n, mode, rate, int(doagc), _p(lilq, C.c_float),
                           _p(audio, C.c_int16), _p(ma, C.c_float))
    return audio, ma


def waterfall_row(psd: np.ndarray, width: int, peak_rgb: int = 0x00FFFF) -> np.ndarray:
    """waterfall.java:90-107 for one published psd row (float[n+2])."""
    psd = np.ascontiguousarray(psd, dtype=np.float32).ravel()
    pix = np.empty(width, dtype=np.int32)
    lib().orc_waterfall_row(_p(psd, C.c_float), psd.size - 2, width, C.c_uint32(peak_rgb), _p(pix, C.c_int32))
    return pix


# ---------------------------------------------------------------- FUNcubeBPSKDemod.java
class _BpskS(C.Structure):
    _fields_ = [
        ("rate", C.c_int), ("D", C.c_int),
        ("tuning", C.c_double), ("tuPhaseInc", C.c_double), ("tuPhase", C.c_double),
        ("ds_ntaps", C.c_int),
        ("dsFilter", C.c_double * 128), ("dsBuf", C.c_double * 256),
        ("dsPos", C.c_int), ("dsCnt", C.c_int),
        ("vcoPhase", C.c_double), ("dmBuf", C.c_double * 130), ("dmPos", C.c_int),
        ("dmEnergy", C.c_double * 10),
        ("dmBitPos", C.c_int), ("dmPeakPos", C.c_int), ("dmNewPeak", C.c_int),
        ("dmEnergyOut", C.c_double), ("dmBitPhase", C.c_double), ("dmLastIQ", C.c_double * 2),
        ("energy1", C.c_double), ("energy2", C.c_double),
        ("cntRaw", C.c_int64), ("cntDS", C.c_int64), ("cntBit", C.c_int64),
        ("cntFEC", C.c_int64), ("cntDec", C.c_int64),
        ("dmCorr", C.c_int), ("dmMaxCorr", C.c_int), ("dmErrBits", C.c_int), ("decodeOK", C.c_int),
        ("dmFECCorr", C.c_int8 * 5200), ("decoded", C.c_uint8 * 256),
        ("do_fec", C.c_int), ("stages", C.c_int), ("doUp", C.c_int),
        ("avePeakPower", C.c_double), ("aveCentreBin", C.c_double), ("centreBin", C.c_int),
        ("sinTab", C.c_double * 256), ("cosTab", C.c_double * 256),
        ("cap_ds", C.POINTER(C.c_double)), ("cap_ds_n", C.c_int), ("cap_ds_max", C.c_int),
        ("cap_dm", C.POINTER(C.c_double)), ("cap_dm_n", C.c_int), ("cap_dm_max", C.c_int),
        ("cap_bits", C.POINTER(C.c_int8)), ("cap_bit_at", C.POINTER(C.c_int64)),
        ("cap_bits_n", C.c_int), ("cap_bits_max", C.c_int),
        ("cap_frames", C.POINTER(C.c_uint8)), ("cap_frames_n", C.c_int), ("cap_frames_max", C.c_int),
    ]


class Bpsk:
    """FUNcubeBPSKDemod.java:366-595 for one tuner."""

    def __init__(self, rate: int, tuning: float = 12000.0, do_fec: bool = False,
                 ds_taps: np.ndarray | None = None, stages: int = 3):
        assert C.sizeof(_BpskS) == lib().orc_bpsk_sizeof(), "struct layout drift"
        self.s = _BpskS()
        lib().orc_bpsk_init(C.byref(self.s), rate, C.c_double(tuning))
        self.s.do_fec = int(do_fec)
        self.s.stages = stages
        if ds_taps is not None:
            t = np.ascontiguousarray(ds_taps, dtype=np.float64)
            lib().orc_bpsk_set_ds_filter(C.byref(self.s), _p(t, C.c_double), t.size)

    def set_tuning(self, hz: float):
        lib().orc_bpsk_set_tuning(C.byref(self.s), C.c_double(hz))

    def receive(self, buf: np.ndarray, autotune: bool = False) -> dict:
        """One IAudioHandler.receive(buf) call; returns what this block produced."""
        buf = np.ascontiguousarray(buf, dtype=np.float32).ravel()
        n = buf.size // 2
        nds = n // max(self.s.D, 1) + 2
        ds = np.zeros((nds, 2), dtype=np.float64)
        dm = np.zeros((nds, 2), dtype=np.float64)
        bits = np.zeros(nds, dtype=np.int8)
        bit_at = np.zeros(nds, dtype=np.int64)
        frames = np.zeros((8, 256), dtype=np.uint8)
        s = self.s
        s.cap_ds, s.cap_ds_n, s.cap_ds_max = _p(ds, C.c_double), 0, nds
        s.cap_dm, s.cap_dm_n, s.cap_dm_max = _p(dm, C.c_double), 0, nds
        s.cap_bits, s.cap_bit_at = _p(bits, C.c_int8), _p(bit_at, C.c_int64)
        s.cap_bits_n, s.cap_bits_max = 0, nds
        s.cap_frames, s.cap_frames_n, s.cap_frames_max = _p(frames, C.c_uint8), 0, 8
        fn = lib().orc_bpsk_receive_fft if autotune else lib().orc_bpsk_receive
        fn(C.byref(s), _p(buf, C.c_float), n)
        out = dict(ds=ds[:s.cap_ds_n].copy(), dm=dm[:s.cap_dm_n].copy(),
                   bits=bits[:s.cap_bits_n].copy(), bit_at=bit_at[:s.cap_bits_n].copy(),
                   frames=frames[:s.cap_frames_n].copy(), centre_bin=int(s.centreBin))
        s.cap_ds = s.cap_dm = None
        s.cap_bits = None
        s.cap_bit_at = None
        s.cap_frames = None
        return out

    def counters(self) -> dict:
        s = self.s
        return dict(raw=s.cntRaw, ds=s.cntDS, bit=s.cntBit, fec=s.cntFEC, dec=s.cntDec)


def default_taps():
    ds = np.empty(27, dtype=np.float64)
    dm = np.empty(65, dtype=np.float64)
    lib().orc_bpsk_default_taps(_p(ds, C.c_double), _p(dm, C.c_double))
    return ds, dm


def sync_vector() -> np.ndarray:
    out = np.empty(65, dtype=np.int8)
    lib().orc_sync_vector(_p(out, C.c_int8))
    return out


# ---------------------------------------------------------------- FECDecoder.java
def fec_sync_lfsr() -> np.ndarray:
    out = np.empty(65, dtype=np.uint8)
    lib().orc_fec_sync_lfsr(_p(out, C.c_uint8))
    return out


def fec_encode(data: np.ndarray) -> np.ndarray:
    data = np.ascontiguousarray(data, dtype=np.uint8)
    assert data.size == 256
    sym = np.empty(5200, dtype=np.uint8)
    lib().orc_fec_encode(_p(data, C.c_uint8), _p(sym, C.c_uint8))
    return sym


def fec_decode(raw: np.ndarray):
    raw = np.ascontiguousarray(raw, dtype=np.uint8)
    assert raw.size == 5200
    out = np.zeros(256, dtype=np.uint8)
    rc = lib().orc_fec_decode(_p(raw, C.c_uint8), _p(out, C.c_uint8))
    return rc, out


def rs_decode(cw: np.ndarray):
    """decode_rs_8 (FECDecoder.java:325-519) on one 255-symbol word: (return value, word after)."""
    cw = np.array(cw, dtype=np.uint8)
    assert cw.size == 255
    rc = lib().orc_rs_decode(_p(cw, C.c_uint8))
    return rc, cw


def fec_table_probe(which: int, idx: int) -> int:
    return lib().orc_fec_table_probe(which, idx)


# ---------------------------------------------------------------- CPU baseline drivers
def baseline_set_fft_mode(mode: int):
    """0: FFT plan rebuilt per block (what fft.java:194 does); 1: cached plan, modulo-free loops."""
    lib().orc_baseline_set_fft_mode(int(mode))


def baseline_fft_s16(raw: np.ndarray, n: int, rate: int, nthreads: int):
    raw = np.ascontiguousarray(raw, dtype=np.int16).ravel()
    nblocks = raw.size // (2 * n)
    psd = np.empty((nblocks, n + 2), dtype=np.float32)
    used = lib().orc_baseline_fft_s16(_p(raw, C.c_int16), nblocks, n, rate, _p(psd, C.c_float), nthreads)
    return psd, used


def baseline_mixdecim_s16(raw: np.ndarray, nchan: int, rate: int, tuning: np.ndarray,
                          taps: np.ndarray | None, nthreads: int):
    raw = np.ascontiguousarray(raw, dtype=np.int16).ravel()
    nsamples = raw.size // (2 * nchan)
    D = rate // 9600
    tuning = np.ascontiguousarray(tuning, dtype=np.float64)
    out = np.zeros((nchan, nsamples // D, 2), dtype=np.float64)
    tp = None
    nt = 0
    if taps is not None:
        taps = np.ascontiguousarray(taps, dtype=np.float64)
        tp, nt = _p(taps, C.c_double), taps.size
    used = lib().orc_baseline_mixdecim_s16(_p(raw, C.c_int16), nchan, nsamples, rate,
                                           _p(tuning, C.c_double), tp, nt,
                                           _p(out, C.c_double), nthreads)
    return out, used


def baseline_pipeline_s16(raw: np.ndarray, nchan: int, nblocks: int, n: int, rate: int,
                          tuning: np.ndarray, taps: np.ndarray | None, nthreads: int):
    """The benchmark pipeline on the CPU: per (channel, block) JavaAudio conversion,
    fft.receive (plan rebuilt per block, fft.java:194) and tuner + decimator."""
    raw = np.ascontiguousarray(raw, dtype=np.int16).ravel()
    assert raw.size == nchan * nblocks * n * 2
    D = rate // 9600
    tuning = np.ascontiguousarray(tuning, dtype=np.float64)
    psd = np.empty((nchan * nblocks, n + 2), dtype=np.float32)
    ds = np.zeros((nchan, nblocks * n // D, 2), dtype=np.float64)
    tp, nt = None, 0
    if taps is not None:
        taps = np.ascontiguousarray(taps, dtype=np.float64)
        tp, nt = _p(taps, C.c_double), taps.size
    used = lib().orc_baseline_pipeline_s16(_p(raw, C.c_int16), nchan, nblocks, n, rate,
                                           _p(tuning, C.c_double), tp, nt,
                                           _p(psd, C.c_float), _p(ds, C.c_double), nthreads)
    return psd, ds, used
