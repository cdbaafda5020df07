"""Host-side binding of libjsdrcuda.so (ctypes), shaped like java-sdr's handlers.

The reference's host language is Java; no JDK exists in this image, so the
handler classes that the Java shim provides (INTEGRATION.md) are mirrored here
over the same C ABI (include/jsdrcuda.h):

    AudioDescriptor          AudioDescriptor.java:3-15
    Publish                  the IPublish bus, jsdr.java:118-147
    fft                      fft.java            receive(float[]) -> "fft-psd"
    FUNcubeBPSKDemod         FUNcubeBPSKDemod.java   (a bank of tuners)
    demod                    demod.java          receive: FIR + NCO, detectors, AGC (float or s16 IQ)
    fir                      fir.java            weights/filter/complex_gen/complex_mod

There is no CPU path: importing works anywhere (so the symbol table can be
checked without a GPU), but creating a Context without a CUDA device raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)                      # java-sdr_b200/
_SO = os.path.join(_ROOT, "libjsdrcuda.so")
HEADER = os.path.join(os.path.dirname(_ROOT), "include", "jsdrcuda.h")

MEM_HOST, MEM_DEVICE = 0, 1
PREC_F64, PREC_F32 = 0, 1
KERNEL_AUTO, KERNEL_TILE, KERNEL_STREAM = 0, 1, 2
INT_MIN = -2147483648


class JsdrError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"jsdrcuda error {code}: {msg}")
        self.code = code


def build(force: bool = False) -> str:
    """Compile csrc/ for sm_100a into java-sdr_b200/libjsdrcuda.so (in tree)."""
    args = ["make", "-C", os.path.join(_ROOT, "csrc"), "-s", "-j8"]
    if force:
        args.append("-B")
    subprocess.check_call(args)
    return _SO


_lib = None

_i, _i64, _f, _d, _vp = C.c_int, C.c_int64, C.c_float, C.c_double, C.c_void_p
_pp = C.POINTER(C.c_void_p)

# name -> argtypes; everything returns int except jsdr_last_error
_SIGS = {
    "jsdr_abi_version": [],
    "jsdr_device_count": [C.POINTER(_i)],
    "jsdr_ctx_create": [_i, _pp],
    "jsdr_ctx_destroy": [_vp],
    "jsdr_ctx_sync": [_vp],
    "jsdr_ctx_launch_count": [_vp, C.POINTER(_i64)],
    "jsdr_ctx_profile": [_vp, _i],
    "jsdr_ctx_profile_read": [_vp, _vp, _vp, _i],
    "jsdr_host_alloc": [_vp, C.c_size_t, _pp],
    "jsdr_host_free": [_vp, _vp],
    "jsdr_dev_alloc": [_vp, C.c_size_t, _pp],
    "jsdr_dev_free": [_vp, _vp],
    "jsdr_memcpy_h2d": [_vp, _vp, _vp, C.c_size_t],
    "jsdr_memcpy_d2h": [_vp, _vp, _vp, C.c_size_t],
    "jsdr_memset_dev": [_vp, _vp, _i, C.c_size_t],
    "jsdr_timer_start": [_vp],
    "jsdr_timer_stop_ms": [_vp, C.POINTER(_f)],
    "jsdr_fft_supported": [_i],
    "jsdr_fft_create": [_vp, _i, _i, _i, _pp],
    "jsdr_fft_destroy": [_vp],
    "jsdr_fft_receive_f32": [_vp, _vp, _i, _vp, _vp, _i],
    "jsdr_fft_receive_s16": [_vp, _vp, _i, _i, _i, _vp, _vp, _i],
    "jsdr_fft_forward_f32": [_vp, _vp, _i, _vp, _i],
    "jsdr_fft_set_window": [_vp, _vp],
    "jsdr_bpsk_create": [_vp, _i, _i, _vp, _i, _pp],
    "jsdr_bpsk_destroy": [_vp],
    "jsdr_bpsk_set_stages": [_vp, _i],
    "jsdr_bpsk_set_tuning": [_vp, _i, _d],
    "jsdr_bpsk_set_autotune": [_vp, _i, _i],
    "jsdr_bpsk_read_centre": [_vp, _vp],
    "jsdr_bpsk_enable_fec": [_vp, _vp, _i],
    "jsdr_bpsk_read_frames": [_vp, _vp, _vp, _vp, _vp, _vp, _i],
    "jsdr_bpsk_read_fec_counters": [_vp, _vp, _vp],
    "jsdr_bpsk_set_precision": [_vp, _i],
    "jsdr_bpsk_set_kernel": [_vp, _i],
    "jsdr_bpsk_set_ds_filter": [_vp, _vp, _i],
    "jsdr_bpsk_receive_f32": [_vp, _vp, _i, _i64, _i],
    "jsdr_bpsk_receive_s16": [_vp, _vp, _i, _i64, _i, _i, _i],
    "jsdr_bpsk_last_counts": [_vp, C.POINTER(C.c_int32)],
    "jsdr_bpsk_read_ds": [_vp, _vp, _i],
    "jsdr_bpsk_read_ds_async": [_vp, _vp, _i],
    "jsdr_bpsk_read_dm": [_vp, _vp, _i],
    "jsdr_bpsk_read_bits": [_vp, _vp, _vp, _vp, _i, _i],
    "jsdr_bpsk_read_counters": [_vp, _vp],
    "jsdr_bpsk_ds_device_ptr": [_vp, _pp],
    "jsdr_demod_create": [_vp, _i, _i, _i, _pp],
    "jsdr_demod_destroy": [_vp],
    "jsdr_demod_weights": [_vp, _i, _i, _i],
    "jsdr_demod_get_weights": [_vp, _i, _vp],
    "jsdr_demod_set_flags": [_vp, _i, _i],
    "jsdr_demod_receive_f32": [_vp, _vp, _i, _i64, _vp, _i],
    "jsdr_demod_set_mode": [_vp, _i, _i],
    "jsdr_demod_receive_audio_f32": [_vp, _vp, _i, _i64, _vp, _vp, _i],
    "jsdr_demod_receive_s16": [_vp, _vp, _i, _i64, _i, _i, _vp, _i],
    "jsdr_demod_receive_audio_s16": [_vp, _vp, _i, _i64, _i, _i, _vp, _vp, _i],
    "jsdr_waterfall_rows": [_vp, _vp, _i, _i, _i, C.c_uint32, _vp, _i],
    "jsdr_fir_design": [_i, _i, _f, _vp],
    "jsdr_fir_nco_table": [_i, _f, _vp],
    "jsdr_fir_create": [_vp, _i, _i, _pp],
    "jsdr_fir_destroy": [_vp],
    "jsdr_fir_set_weights": [_vp, _i, _vp],
    "jsdr_fir_filter_i32": [_vp, _vp, _i, _i64, _vp, _i],
    "jsdr_fir_complex_mod_i32": [_vp, _vp, _vp, _vp, _i64, _i],
    "jsdr_pump_receive_s16": [_vp, _vp, _vp, _i, _i, _i, _vp, _vp, _i],
    "jsdr_pump_waterfall_s16": [_vp, _vp, _vp, _i, _i, _i, _i, C.c_uint32, _vp, _vp, _vp, _i],
    "jsdr_pump_demod_s16": [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _i],
    "jsdr_probe_table": [_i, _vp, _i],
    "jsdr_probe_taps": [_vp, _vp],
    "jsdr_probe_scout_thresholds": [_d, C.POINTER(_d), C.POINTER(_d)],
}
EXPORTS = sorted(list(_SIGS) + ["jsdr_last_error"])


def lib() -> C.CDLL:
    """Load libjsdrcuda.so.  Fails loudly if the CUDA extension has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            raise ImportError(f"{_SO} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(there is no CPU fallback)")
        # JSDR_LIB: another build of the same library (kernel experiments, tools/kbench.py)
        _lib = C.CDLL(os.environ.get("JSDR_LIB") or _SO)
        for name, args in _SIGS.items():
            fn = getattr(_lib, name, None)
            if fn is None:
                if os.environ.get("JSDR_LIB"):      # an older experiment build may lack newer entry points
                    continue
                raise ImportError(f"{_SO} does not export {name}: rebuild it")
            fn.argtypes = args
            fn.restype = C.c_int
        _lib.jsdr_last_error.restype = C.c_char_p
        _lib.jsdr_last_error.argtypes = []
    return _lib


def _ck(rc: int):
    if rc != 0:
        raise JsdrError(rc, lib().jsdr_last_error().decode("utf-8", "replace"))


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(_vp)
    if isinstance(a, DevBuf):
        return _vp(a.ptr)
    return _vp(int(a))


# ---------------------------------------------------------------------------- contracts
class AudioDescriptor:
    """AudioDescriptor.java:3-15."""

    def __init__(self, rate: int, bits: int = 16, chns: int = 2, size: int = 4, blen: int | None = None):
        self.rate, self.bits, self.chns, self.size = rate, bits, chns, size
        self.blen = rate * size // 10 if blen is None else blen      # JavaAudio.java:59

    @property
    def samples(self) -> int:
        return self.blen // self.size


class Publish:
    """The IPublish bus (IPublish.java, implemented at jsdr.java:118-147):
    setPublish stores the value and notifies listeners synchronously."""

    def __init__(self):
        self._vals, self._listeners = {}, []

    def setPublish(self, key, val):
        self._vals[key] = val
        for l in list(self._listeners):
            l(key, val) if callable(l) else l.notify(key, val)

    def getPublish(self, key, default=None):
        return self._vals.get(key, default)

    def listen(self, l):
        self._listeners.append(l)

    def unlisten(self, l):
        self._listeners.remove(l)


class DevBuf:
    """A device allocation owned by a Context."""

    def __init__(self, ctx: "Context", nbytes: int):
        self.ctx, self.nbytes = ctx, int(nbytes)
        p = C.c_void_p()
        _ck(lib().jsdr_dev_alloc(ctx.h, self.nbytes, C.byref(p)))
        self.ptr = p.value

    def upload(self, a: np.ndarray, offset: int = 0):
        a = np.ascontiguousarray(a)
        assert offset + a.nbytes <= self.nbytes
        _ck(lib().jsdr_memcpy_h2d(self.ctx.h, _vp(self.ptr + offset), a.ctypes.data_as(_vp), a.nbytes))

    def download(self, dtype, count: int, offset: int = 0) -> np.ndarray:
        out = np.empty(count, dtype=dtype)
        assert offset + out.nbytes <= self.nbytes
        _ck(lib().jsdr_memcpy_d2h(self.ctx.h, out.ctypes.data_as(_vp), _vp(self.ptr + offset), out.nbytes))
        return out

    def free(self):
        if self.ptr:
            lib().jsdr_dev_free(self.ctx.h, _vp(self.ptr))
            self.ptr = 0


class Context:
    def __init__(self, device: int = 0):
        h = C.c_void_p()
        _ck(lib().jsdr_ctx_create(device, C.byref(h)))
        self.h = h
        self.device = device

    def close(self):
        if self.h:
            lib().jsdr_ctx_destroy(self.h)
            self.h = None

    def sync(self):
        _ck(lib().jsdr_ctx_sync(self.h))

    def launch_count(self) -> int:
        n = C.c_int64()
        _ck(lib().jsdr_ctx_launch_count(self.h, C.byref(n)))
        return n.value

    KINDS = ("fft", "mixdecim", "matched", "timing", "scout", "other", "demod", "fir", "detect", "waterfall", "sync", "fec")

    def profile(self, enable: bool = True):
        """Bracket every kernel launch with CUDA events on its own stream (bench.py)."""
        _ck(lib().jsdr_ctx_profile(self.h, int(enable)))

    def profile_read(self) -> dict:
        """{kind: (total ms, launches)} since the last read; waits for the device."""
        ms = np.zeros(len(self.KINDS), dtype=np.float64)
        cnt = np.zeros(len(self.KINDS), dtype=np.int64)
        _ck(lib().jsdr_ctx_profile_read(self.h, _ptr(ms), _ptr(cnt), len(self.KINDS)))
        return {k: (float(ms[i]), int(cnt[i])) for i, k in enumerate(self.KINDS)}

    def dev_alloc(self, nbytes: int) -> DevBuf:
        return DevBuf(self, nbytes)

    def host_alloc(self, shape, dtype) -> np.ndarray:
        """Pinned host array (the ring buffers handed to Java as MemorySegments)."""
        dtype = np.dtype(dtype)
        n = int(np.prod(shape))
        p = C.c_void_p()
        _ck(lib().jsdr_host_alloc(self.h, n * dtype.itemsize, C.byref(p)))
        buf = (C.c_char * (n * dtype.itemsize)).from_address(p.value)
        return np.frombuffer(buf, dtype=dtype, count=n).reshape(shape)

    def host_free(self, a: np.ndarray):
        lib().jsdr_host_free(self.h, _vp(a.ctypes.data))

    def timer_start(self):
        _ck(lib().jsdr_timer_start(self.h))

    def timer_stop_ms(self) -> float:
        ms = C.c_float()
        _ck(lib().jsdr_timer_stop_ms(self.h, C.byref(ms)))
        return ms.value


def device_count() -> int:
    n = C.c_int()
    _ck(lib().jsdr_device_count(C.byref(n)))
    return n.value


def design_lowpass(ntaps: int, cutoff_hz: float, rate: int) -> np.ndarray:
    """Hamming windowed-sinc low-pass by the demod.java:356-366 formula (band
    -cutoff..+cutoff) in double: the 64-tap decimator shape of BASELINE config 4."""
    ord_ = ntaps - 1
    nlo, nhi = -cutoff_hz / rate, cutoff_hz / rate
    w = np.empty(ntaps, dtype=np.float64)
    for n in range(ntaps):
        d = n - ord_ / 2.0
        if d == 0:
            w[n] = 2.0 * (nhi - nlo)
        else:
            w[n] = (np.sin(2 * np.pi * nhi * d) - np.sin(2 * np.pi * nlo * d)) / (np.pi * d)
        w[n] *= 0.54 - 0.46 * np.cos(2 * np.pi * n / ord_)
    return w


def fft_supported(n: int) -> bool:
    return bool(lib().jsdr_fft_supported(n))


# ---------------------------------------------------------------------------- fft.java
class fft:
    """fft.java: receive(buf) publishes "fft-psd" = float[N+2] (fft.java:190-228).

    `max_batch` > 1 lets one call carry many independent blocks (BASELINE config 3).
    """

    def __init__(self, ctx: Context, publish: Publish | None, adsc: AudioDescriptor, max_batch: int = 1,
                 n: int | None = None):
        self.ctx, self.publish, self.adsc = ctx, publish, adsc
        self.n = adsc.samples if n is None else n          # dat.length/2, fft.java:67
        self.max_batch = max_batch
        h = C.c_void_p()
        _ck(lib().jsdr_fft_create(ctx.h, self.n, adsc.rate, max_batch, C.byref(h)))
        self.h = h
        self.psd = np.zeros(self.n + 2, dtype=np.float32)   # reused every block, like fft.java:68
        self.peak_bin = -1

    def close(self):
        if self.h:
            lib().jsdr_fft_destroy(self.h)
            self.h = None

    def receive(self, buf: np.ndarray):
        """IAudioHandler.receive(float[] buf): one block of 2N floats."""
        buf = np.ascontiguousarray(buf, dtype=np.float32).ravel()
        if buf.size != 2 * self.n:
            raise ValueError("buf must hold 2*N floats")
        pk = np.zeros(1, dtype=np.int32)
        _ck(lib().jsdr_fft_receive_f32(self.h, _ptr(buf), 1, _ptr(self.psd), _ptr(pk), MEM_HOST))
        self.peak_bin = int(pk[0])
        if self.publish is not None:
            self.publish.setPublish("fft-psd", self.psd)     # fft.java:226
        return self.psd

    def receive_raw(self, raw: np.ndarray, ic: int = 0, qc: int = 0):
        """IRawHandler.receive(byte[] buf): s16le IQ, converted on the device."""
        raw = np.ascontiguousarray(raw).view(np.int16).ravel()
        if raw.size != 2 * self.n:
            raise ValueError("raw must hold 2*N int16")
        pk = np.zeros(1, dtype=np.int32)
        _ck(lib().jsdr_fft_receive_s16(self.h, _ptr(raw), 1, ic, qc, _ptr(self.psd), _ptr(pk), MEM_HOST))
        self.peak_bin = int(pk[0])
        if self.publish is not None:
            self.publish.setPublish("fft-psd", self.psd)
        return self.psd

    def receive_batch(self, bufs: np.ndarray, s16: bool = False, ic: int = 0, qc: int = 0):
        """Many blocks at once: returns (psd[batch, N+2], peak_bin[batch])."""
        a = np.ascontiguousarray(bufs, dtype=np.int16 if s16 else np.float32).reshape(-1, 2 * self.n)
        batch = a.shape[0]
        psd = np.empty((batch, self.n + 2), dtype=np.float32)
        pk = np.empty(batch, dtype=np.int32)
        if s16:
            _ck(lib().jsdr_fft_receive_s16(self.h, _ptr(a), batch, ic, qc, _ptr(psd), _ptr(pk), MEM_HOST))
        else:
            _ck(lib().jsdr_fft_receive_f32(self.h, _ptr(a), batch, _ptr(psd), _ptr(pk), MEM_HOST))
        return psd, pk

    def forward(self, bufs: np.ndarray) -> np.ndarray:
        """The spectrum complexForward leaves in dat[] (fft.java:195), per block."""
        a = np.ascontiguousarray(bufs, dtype=np.float32).reshape(-1, 2 * self.n)
        out = np.empty_like(a)
        _ck(lib().jsdr_fft_forward_f32(self.h, _ptr(a), a.shape[0], _ptr(out), MEM_HOST))
        return out.view(np.complex64).reshape(a.shape[0], self.n)

    def set_window(self, win):
        """fft.java's win[] (:72-73) applied ahead of the transform (jsdr_fft_set_window): every
        later call multiplies sample t of each block by win[t], float[N]; None removes it.
        Stream-ordered: device-memory calls already enqueued keep the window they were enqueued with."""
        if win is None:
            _ck(lib().jsdr_fft_set_window(self.h, None))
            return
        w = np.ascontiguousarray(win, dtype=np.float32).ravel()
        if w.size != self.n:
            raise ValueError("win must hold N floats")
        _ck(lib().jsdr_fft_set_window(self.h, _ptr(w)))

    # device-resident entry points (bench.py)
    def receive_dev(self, d_in, batch: int, d_psd, d_peak=None, s16: bool = True, ic: int = 0, qc: int = 0):
        if s16:
            _ck(lib().jsdr_fft_receive_s16(self.h, _ptr(d_in), batch, ic, qc, _ptr(d_psd), _ptr(d_peak), MEM_DEVICE))
        else:
            _ck(lib().jsdr_fft_receive_f32(self.h, _ptr(d_in), batch, _ptr(d_psd), _ptr(d_peak), MEM_DEVICE))


# ---------------------------------------------------------------------------- FUNcubeBPSKDemod.java
class FUNcubeBPSKDemod:
    """A bank of FUNcube tuners; receive(buf) is doBufferTune for every channel
    (FUNcubeBPSKDemod.java:358-379).  `tuning` is one value per channel
    (config key "FUNcube<i>-bpsk-tuning", default 12000, :195)."""

    def __init__(self, ctx: Context, publish: Publish | None, adsc: AudioDescriptor, tuning=(12000.0,),
                 max_block: int | None = None, stages: int = 3, name: str = "FUNcube"):
        self.ctx, self.publish, self.adsc, self.name = ctx, publish, adsc, name
        self.tuning = np.ascontiguousarray(tuning, dtype=np.float64).ravel()
        self.nchan = self.tuning.size
        self.max_block = adsc.samples if max_block is None else max_block
        self.D = adsc.rate // 9600
        h = C.c_void_p()
        _ck(lib().jsdr_bpsk_create(ctx.h, adsc.rate, self.nchan, _ptr(self.tuning), self.max_block, C.byref(h)))
        self.h = h
        self.stages = stages
        _ck(lib().jsdr_bpsk_set_stages(h, stages))

    def close(self):
        if self.h:
            lib().jsdr_bpsk_destroy(self.h)
            self.h = None

    def set_tuning(self, chan: int, hz: float):
        _ck(lib().jsdr_bpsk_set_tuning(self.h, chan, hz))
        self.tuning[chan] = hz

    def set_autotune(self, dofft: bool, upper: bool = False):
        """doBufferFFT instead of doBufferTune (config "FUNcube<i>-bpsk-dofft" / "-upper")."""
        self.dofft = bool(dofft)
        _ck(lib().jsdr_bpsk_set_autotune(self.h, int(dofft), int(upper)))

    def centre_bins(self) -> np.ndarray:
        out = np.zeros(self.nchan, dtype=np.int32)
        _ck(lib().jsdr_bpsk_read_centre(self.h, _ptr(out)))
        return out

    def enable_fec(self, mettab: np.ndarray, max_frames: int = 64):
        """Sync correlator + FECDecode behind the bits (:553-574, FECDecoder.java:703-852).
        mettab: FECDecoder's metric table, int16[2, 256]."""
        t = np.ascontiguousarray(mettab, dtype=np.int16).reshape(2, 256)
        self._max_frames = max_frames
        _ck(lib().jsdr_bpsk_enable_fec(self.h, _ptr(t), max_frames))

    def read_frames(self):
        """[(channel, bit_index, errors, data uint8[256])] of the last receive, by (channel, bit)."""
        mf = self._max_frames
        n = np.zeros(1, dtype=np.int32)
        chan = np.zeros(mf, dtype=np.int32)
        at = np.zeros(mf, dtype=np.int64)
        err = np.zeros(mf, dtype=np.int32)
        data = np.zeros((mf, 256), dtype=np.uint8)
        _ck(lib().jsdr_bpsk_read_frames(self.h, _ptr(n), _ptr(chan), _ptr(at), _ptr(err), _ptr(data), mf))
        k = min(int(n[0]), mf)
        return [(int(chan[i]), int(at[i]), int(err[i]), data[i].copy()) for i in range(k)]

    def fec_counters(self):
        a = np.zeros(self.nchan, dtype=np.int64)
        d = np.zeros(self.nchan, dtype=np.int64)
        _ck(lib().jsdr_bpsk_read_fec_counters(self.h, _ptr(a), _ptr(d)))
        return a, d

    def set_precision(self, precision: int):
        _ck(lib().jsdr_bpsk_set_precision(self.h, precision))

    def set_kernel(self, mode: int):
        _ck(lib().jsdr_bpsk_set_kernel(self.h, mode))

    def set_ds_filter(self, taps: np.ndarray):
        t = np.ascontiguousarray(taps, dtype=np.float64)
        _ck(lib().jsdr_bpsk_set_ds_filter(self.h, _ptr(t), t.size))

    def _stride(self, total: int, n: int, shared: bool) -> int:
        return 0 if shared else n

    def receive(self, buf: np.ndarray, shared: bool | None = None):
        """float IQ.  buf is [2*S] (one stream fanned out to all tuners) or [nchan, 2*S]."""
        a = np.ascontiguousarray(buf, dtype=np.float32)
        if shared is None:
            shared = a.ndim == 1 or a.shape[0] == 1 and self.nchan > 1
        S = a.size // 2 if shared else a.size // (2 * self.nchan)
        _ck(lib().jsdr_bpsk_receive_f32(self.h, _ptr(a), S, 0 if shared else S, MEM_HOST))
        self._published()

    def receive_raw(self, raw: np.ndarray, ic: int = 0, qc: int = 0, shared: bool | None = None):
        a = np.ascontiguousarray(raw).view(np.int16)
        if shared is None:
            shared = a.ndim == 1 or a.shape[0] == 1 and self.nchan > 1
        S = a.size // 2 if shared else a.size // (2 * self.nchan)
        _ck(lib().jsdr_bpsk_receive_s16(self.h, _ptr(a), S, 0 if shared else S, ic, qc, MEM_HOST))
        self._published()

    def receive_dev(self, d_in, S: int, chan_stride: int, s16: bool = True, ic: int = 0, qc: int = 0):
        if s16:
            _ck(lib().jsdr_bpsk_receive_s16(self.h, _ptr(d_in), S, chan_stride, ic, qc, MEM_DEVICE))
        else:
            _ck(lib().jsdr_bpsk_receive_f32(self.h, _ptr(d_in), S, chan_stride, MEM_DEVICE))

    def _published(self):
        if self.publish is None:
            return
        if getattr(self, "dofft", False):                     # :455-456
            centre = self.centre_bins()
            for c in range(self.nchan):
                self.publish.setPublish(f"{self.name}{c}-bpsk-tune", -1)
                self.publish.setPublish(f"{self.name}{c}-bpsk-centre", int(centre[c]))
        else:                                                 # :377-378
            for c in range(self.nchan):
                self.publish.setPublish(f"{self.name}{c}-bpsk-centre", -1)
                self.publish.setPublish(f"{self.name}{c}-bpsk-tune", int(self.tuning[c]))

    def last_nds(self) -> int:
        n = C.c_int32()
        _ck(lib().jsdr_bpsk_last_counts(self.h, C.byref(n)))
        return n.value

    def read_ds(self) -> np.ndarray:
        n = self.last_nds()
        out = np.empty((self.nchan, n, 2), dtype=np.float64)
        _ck(lib().jsdr_bpsk_read_ds(self.h, _ptr(out), MEM_HOST))
        return out

    def read_ds_async(self, out: np.ndarray) -> int:
        """Start the copy of the decimated rows into `out` (pinned host memory, at least
        nchan x last_nds x 2 doubles) and return last_nds at once; the rows are there after
        Context.sync().  The copy overlaps the next block's upload."""
        n = self.last_nds()
        assert out.dtype == np.float64 and out.size >= self.nchan * n * 2
        _ck(lib().jsdr_bpsk_read_ds_async(self.h, _ptr(out), MEM_HOST))
        return n

    def read_dm(self) -> np.ndarray:
        n = self.last_nds()
        out = np.empty((self.nchan, n, 2), dtype=np.float64)
        _ck(lib().jsdr_bpsk_read_dm(self.h, _ptr(out), MEM_HOST))
        return out

    def read_bits(self):
        """Returns (list of int8 arrays per channel, list of int64 sample indices)."""
        mb = max(self.last_nds(), 1)
        bits = np.zeros((self.nchan, mb), dtype=np.int8)
        at = np.zeros((self.nchan, mb), dtype=np.int64)
        nb = np.zeros(self.nchan, dtype=np.int32)
        _ck(lib().jsdr_bpsk_read_bits(self.h, _ptr(bits), _ptr(at), _ptr(nb), mb, MEM_HOST))
        return [bits[c, :nb[c]].copy() for c in range(self.nchan)], [at[c, :nb[c]].copy() for c in range(self.nchan)]

    def counters(self) -> np.ndarray:
        out = np.zeros((self.nchan, 4), dtype=np.int64)
        _ck(lib().jsdr_bpsk_read_counters(self.h, _ptr(out)))
        return out


# ---------------------------------------------------------------------------- demod.java
class demod:
    """FIR band-pass + NCO down-shift of demod.receive (demod.java:410-434)."""

    def __init__(self, ctx: Context, adsc: AudioDescriptor, nchan: int = 1, max_block: int | None = None,
                 dofir: bool = True, dodwn: bool = True):
        self.ctx, self.adsc, self.nchan = ctx, adsc, nchan
        self.max_block = adsc.samples if max_block is None else max_block
        h = C.c_void_p()
        _ck(lib().jsdr_demod_create(ctx.h, adsc.rate, nchan, self.max_block, C.byref(h)))
        self.h = h
        _ck(lib().jsdr_demod_set_flags(h, int(dofir), int(dodwn)))

    def close(self):
        if self.h:
            lib().jsdr_demod_destroy(self.h)
            self.h = None

    def weights(self, flo: int, fhi: int, chan: int = 0) -> np.ndarray:
        _ck(lib().jsdr_demod_weights(self.h, chan, flo, fhi))
        w = np.empty(21, dtype=np.float32)
        _ck(lib().jsdr_demod_get_weights(self.h, chan, _ptr(w)))
        return w

    def set_flags(self, dofir: bool, dodwn: bool):
        _ck(lib().jsdr_demod_set_flags(self.h, int(dofir), int(dodwn)))

    def receive(self, buf: np.ndarray, shared: bool | None = None) -> np.ndarray:
        a = np.ascontiguousarray(buf, dtype=np.float32)
        if shared is None:
            shared = a.ndim == 1
        S = a.size // 2 if shared else a.size // (2 * self.nchan)
        out = np.empty((self.nchan, 2 * S), dtype=np.float32)
        _ck(lib().jsdr_demod_receive_f32(self.h, _ptr(a), S, 0 if shared else S, _ptr(out), MEM_HOST))
        return out


    MODE_OFF, MODE_RAW, MODE_AM, MODE_NFM, MODE_WFM = range(5)     # demod.java:39-43

    def set_mode(self, mode: int, doagc: bool = False):
        _ck(lib().jsdr_demod_set_mode(self.h, mode, int(doagc)))

    def receive_audio(self, buf: np.ndarray, shared: bool | None = None):
        """The whole of demod.receive (:398-481): returns (s16 audio [nchan, S], max_avg [nchan, 2])."""
        a = np.ascontiguousarray(buf, dtype=np.float32)
        if shared is None:
            shared = a.ndim == 1
        S = a.size // 2 if shared else a.size // (2 * self.nchan)
        audio = np.empty((self.nchan, S), dtype=np.int16)
        ma = np.empty((self.nchan, 2), dtype=np.float32)
        _ck(lib().jsdr_demod_receive_audio_f32(self.h, _ptr(a), S, 0 if shared else S, _ptr(audio), _ptr(ma), MEM_HOST))
        return audio, ma

    def _raw(self, raw, shared):
        a = np.ascontiguousarray(raw).view(np.int16)
        if shared is None:
            shared = a.ndim == 1
        S = a.size // 2 if shared else a.size // (2 * self.nchan)
        return a, S, 0 if shared else S

    def receive_raw(self, raw: np.ndarray, ic: int = 0, qc: int = 0, shared: bool | None = None) -> np.ndarray:
        """receive() on s16 IQ (IRawHandler), converted on the device as JavaAudio.java:276-293 does."""
        a, S, stride = self._raw(raw, shared)
        out = np.empty((self.nchan, 2 * S), dtype=np.float32)
        _ck(lib().jsdr_demod_receive_s16(self.h, _ptr(a), S, stride, ic, qc, _ptr(out), MEM_HOST))
        return out

    def receive_audio_raw(self, raw: np.ndarray, ic: int = 0, qc: int = 0, shared: bool | None = None):
        """receive_audio() on s16 IQ: returns (s16 audio [nchan, S], max_avg [nchan, 2])."""
        a, S, stride = self._raw(raw, shared)
        audio = np.empty((self.nchan, S), dtype=np.int16)
        ma = np.empty((self.nchan, 2), dtype=np.float32)
        _ck(lib().jsdr_demod_receive_audio_s16(self.h, _ptr(a), S, stride, ic, qc, _ptr(audio), _ptr(ma), MEM_HOST))
        return audio, ma


def waterfall_rows(ctx: "Context", psd: np.ndarray, width: int, peak_rgb: int = 0x00FFFF) -> np.ndarray:
    """waterfall.paintLine (waterfall.java:90-107) for rows of published "fft-psd" arrays."""
    a = np.ascontiguousarray(psd, dtype=np.float32)
    a = a.reshape(-1, a.shape[-1])
    pix = np.empty((a.shape[0], width), dtype=np.int32)
    _ck(lib().jsdr_waterfall_rows(ctx.h, _ptr(a), a.shape[1] - 2, a.shape[0], width, peak_rgb, _ptr(pix), MEM_HOST))
    return pix


# ---------------------------------------------------------------------------- fir.java
class fir:
    """fir.java's arithmetic: weights (:169-195), filter (:198-211),
    complex_gen (:221-228), complex_mod (:214-218)."""

    def __init__(self, ctx: Context, rate: float = 44100.0, nchan: int = 1, max_block: int = 65536):
        self.ctx, self.rate, self.nchan = ctx, float(rate), nchan
        h = C.c_void_p()
        _ck(lib().jsdr_fir_create(ctx.h, nchan, max_block, C.byref(h)))
        self.h = h

    def close(self):
        if self.h:
            lib().jsdr_fir_destroy(self.h)
            self.h = None

    def weights(self, f1: int, f2: int, chan: int = 0) -> np.ndarray:
        w = np.empty(21, dtype=np.float64)
        _ck(lib().jsdr_fir_design(f1, f2, self.rate, _ptr(w)))
        _ck(lib().jsdr_fir_set_weights(self.h, chan, _ptr(w)))
        return w

    def filter(self, x: np.ndarray, shared: bool | None = None) -> np.ndarray:
        a = np.ascontiguousarray(x, dtype=np.int32)
        if shared is None:
            shared = a.ndim == 1
        S = a.size if shared else a.size // self.nchan
        out = np.empty((self.nchan, S), dtype=np.int32)
        _ck(lib().jsdr_fir_filter_i32(self.h, _ptr(a), S, 0 if shared else S, _ptr(out), MEM_HOST))
        return out

    def complex_gen(self, freq: int) -> np.ndarray:
        """One period ((int)rate samples) of the integer NCO."""
        t = np.empty((int(self.rate), 2), dtype=np.int32)
        _ck(lib().jsdr_fir_nco_table(freq, self.rate, _ptr(t)))
        return t

    def complex_mod(self, a: np.ndarray, b: np.ndarray) -> np.ndarray:
        a = np.ascontiguousarray(a, dtype=np.int32).reshape(-1, 2)
        b = np.ascontiguousarray(b, dtype=np.int32).reshape(-1, 2)
        out = np.empty_like(a)
        _ck(lib().jsdr_fir_complex_mod_i32(self.ctx.h, _ptr(a), _ptr(b), _ptr(out), a.shape[0], MEM_HOST))
        return out


# ---------------------------------------------------------------------------- the pump
def pump_receive_s16(f: fft, b: FUNcubeBPSKDemod, raw, nblocks: int, psd, peak_bin=None, mem: int = MEM_HOST,
                     ic: int = 0, qc: int = 0):
    """JavaAudio.run's fan-out (JavaAudio.java:262-304) for [nchan][nblocks*N] s16 IQ; ic/qc are
    the I/Q DC corrections of JavaAudio.java:281-288, seen by both handlers."""
    _ck(lib().jsdr_pump_receive_s16(f.h, b.h, _ptr(raw), nblocks, ic, qc, _ptr(psd), _ptr(peak_bin), mem))


def pump_waterfall_s16(f: fft, b: FUNcubeBPSKDemod, raw, nblocks: int, width: int, pixels, peak, peak_bin=None,
                       mem: int = MEM_HOST, ic: int = 0, qc: int = 0, peak_rgb: int = 0x00ffff):
    """The pump with waterfall.java's paintLine (:90-107) on the device: pixel rows
    [nchan*nblocks][width] int32 and peak [nchan*nblocks][2] float32 instead of the PSD."""
    _ck(lib().jsdr_pump_waterfall_s16(f.h, b.h, _ptr(raw), nblocks, ic, qc, width, peak_rgb, _ptr(pixels), _ptr(peak),
                                      _ptr(peak_bin), mem))


def pump_demod_s16(f: fft, b: FUNcubeBPSKDemod, d: demod, raw, nblocks: int, psd, audio, max_avg=None, peak_bin=None,
                   mem: int = MEM_HOST, ic: int = 0, qc: int = 0):
    """JavaAudio.run's whole fan-out (JavaAudio.java:298-304): the pump plus the demod handler.
    audio is [nchan][nblocks*N] int16; max_avg (optional) [nchan][nblocks][2] float32, per block."""
    _ck(lib().jsdr_pump_demod_s16(f.h, b.h, d.h, _ptr(raw), nblocks, ic, qc, _ptr(psd), _ptr(peak_bin), _ptr(audio),
                                  _ptr(max_avg), mem))


# ---------------------------------------------------------------------------- constant tables
_TABLE_SIZES = {"Partab": (0, 256), "Syms": (1, 128), "Scrambler": (2, 320), "ALPHA_TO": (3, 256),
                "INDEX_OF": (4, 256), "RS_poly": (5, 16), "SYNC_VECTOR": (6, 65)}


def probe_table(name: str) -> np.ndarray:
    """A table the library builds for itself (jsdr_probe_table), by its name in the reference
    (FECDecoder.java:40-181,544-546; FUNcubeBPSKDemod.java:79-81).  No device needed."""
    which, n = _TABLE_SIZES[name]
    out = np.empty(n, dtype=np.int32)
    _ck(lib().jsdr_probe_table(which, _ptr(out), n))
    return out


def probe_scout_thresholds(inc: float):
    """(th1, th2) of the tuner-phase replay for one increment (jsdr_probe_scout_thresholds)."""
    a, b = _d(), _d()
    _ck(lib().jsdr_probe_scout_thresholds(inc, C.byref(a), C.byref(b)))
    return a.value, b.value


def probe_taps():
    """(dsFilter[27], dmFilter[65]) as the kernels use them (FUNcubeBPSKDemod.java:27-77)."""
    ds, dm = np.empty(27), np.empty(65)
    _ck(lib().jsdr_probe_taps(_ptr(ds), _ptr(dm)))
    return ds, dm
