#!/usr/bin/env python
"""Kernel-level timings on one GPU (CUDA events on the library's stream).
  python tools/kbench.py mix   [nchan] [S]      tuner+decimator: tile / stream f64 / stream f32
  python tools/kbench.py fft   [n ...]          FFT+PSD per length (s16 and f32 input)
  python tools/kbench.py other                  demod.java FIR+NCO, detectors, fir.java int FIR, waterfall rows, frame stage
  python tools/kbench.py demod [nchan] [S]      demod FIR+NCO and NFM / AM audio, f32 against s16 input, alternated
  python tools/kbench.py pumpdemod [nchan] [nblk] [n]   the pump with and without the demod handler, alternated
  python tools/kbench.py duty                   the reference's duty: fft + demod (NFM) + two tuners, per 100 ms block
  python tools/kbench.py window [n ...]         FFT+PSD with and without jsdr_fft_set_window, alternated (s16 and f32)
Prints achieved GB/s of algorithmic bytes and the fraction of MEASURED_PEAKS.json."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "java-sdr_b200")):
    sys.path.insert(0, p)
import jsdrcuda as J

try:
    PEAK = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
except Exception:
    PEAK = 6650.0


def time_ms(ctx, fn, reps=5, warm=2):
    for _ in range(warm):
        fn()
    ctx.sync()
    ctx.timer_start()
    for _ in range(reps):
        fn()
    return ctx.timer_stop_ms() / reps


def mix(nchan=4096, S=131072, rate=192000, ntaps=64):
    ctx = J.Context(0)
    D = rate // 9600
    rng = np.random.default_rng(1)
    tun = rng.uniform(2000, 90000, nchan)
    taps = J.design_lowpass(ntaps, 4800.0, rate) if ntaps != 27 else None
    d_raw = ctx.dev_alloc(nchan * S * 4)
    tile = rng.integers(-20000, 20000, (64, 2 * S)).astype(np.int16)
    for c0 in range(0, nchan, 64):
        d_raw.upload(tile[: min(64, nchan - c0)], offset=c0 * S * 4)
    bytes_ = nchan * S * 4 + nchan * (S // D) * 16
    for name, kern, prec in (("tile f64", J.KERNEL_TILE, J.PREC_F64), ("stream f64", J.KERNEL_STREAM, J.PREC_F64),
                             ("stream f32", J.KERNEL_STREAM, J.PREC_F32)):
        bank = J.FUNcubeBPSKDemod(ctx, None, J.AudioDescriptor(rate), tuning=tun, max_block=S, stages=1)
        if taps is not None:
            bank.set_ds_filter(taps)
        bank.set_kernel(kern)
        bank.set_precision(prec)
        ms = time_ms(ctx, lambda: bank.receive_dev(d_raw, S, S, s16=True))
        gbs = bytes_ / ms / 1e6
        print(f"mix {name:10s} nchan={nchan} S={S} taps={ntaps} D={D}: {ms:8.3f} ms  {nchan * S / ms / 1e3:9.1f} Msamples/s  "
              f"{gbs:7.1f} GB/s  frac {gbs / PEAK:.3f}", flush=True)
        bank.close()
    # float input (IAudioHandler path), half the channels to keep the resident batch the same size
    nf = nchan // 2
    d_f = ctx.dev_alloc(nf * S * 8)
    tf = (tile[:64].astype(np.float32) / 32767.0)
    for c0 in range(0, nf, 64):
        d_f.upload(tf[: min(64, nf - c0)], offset=c0 * S * 8)
    for name, prec in (("stream f64", J.PREC_F64), ("stream f32", J.PREC_F32)):
        bank = J.FUNcubeBPSKDemod(ctx, None, J.AudioDescriptor(rate), tuning=tun[:nf], max_block=S, stages=1)
        if taps is not None:
            bank.set_ds_filter(taps)
        bank.set_precision(prec)
        ms = time_ms(ctx, lambda: bank.receive_dev(d_f, S, S, s16=False))
        b = nf * S * 8 + nf * (S // D) * 16
        print(f"mix {name:10s} FLOAT IN nchan={nf} S={S}: {ms:8.3f} ms  {nf * S / ms / 1e3:9.1f} Msamples/s  "
              f"{b / ms / 1e6:7.1f} GB/s  frac {b / ms / 1e6 / PEAK:.3f}", flush=True)
        bank.close()
    ctx.close()


def fft(ns, total=None):
    # KBENCH_TOTAL: samples per launch (default 2^28); KBENCH_FILL=0: random data only
    # in the first 8 MB (the rest of a fresh allocation reads as zeros: no arg-max work, less power)
    total = total or int(os.environ.get("KBENCH_TOTAL", 1 << 28))
    fill = os.environ.get("KBENCH_FILL", "1") != "0"
    ctx = J.Context(0)
    rng = np.random.default_rng(2)
    for n in ns:
        batch = max(1, total // n)
        f = J.fft(ctx, None, J.AudioDescriptor(192000), max_batch=batch, n=n)
        d_in = ctx.dev_alloc(batch * n * 8)
        tile = rng.integers(-20000, 20000, 1 << 22).astype(np.int16)
        d_in.upload(tile)
        if fill:
            for off in range(tile.nbytes, batch * n * 4, tile.nbytes):
                d_in.upload(tile[: min(tile.size, (batch * n * 4 - off) // 2)], offset=off)
        d_psd = ctx.dev_alloc(batch * (n + 2) * 4)
        d_pk = ctx.dev_alloc(batch * 4)
        for s16 in (True, False):
            ms = time_ms(ctx, lambda: f.receive_dev(d_in, batch, d_psd, d_pk, s16=s16))
            b = batch * n * ((4 if s16 else 8) + 4)
            print(f"fft n={n:6d} batch={batch:7d} {'s16' if s16 else 'f32'}: {ms:8.3f} ms  {batch * n / ms / 1e3:9.1f} Msamples/s  "
                  f"{b / ms / 1e6:7.1f} GB/s  frac {b / ms / 1e6 / PEAK:.3f}", flush=True)
        for d in (d_in, d_psd, d_pk):
            d.free()
        f.close()
    ctx.close()


def chain(nchan=4096, S=131072, rate=192000):
    """Full FUNcube chain (tuner, 27-tap decimator, matched filter, bit timing) per stage count."""
    ctx = J.Context(0)
    rng = np.random.default_rng(1)
    tun = rng.uniform(2000, 90000, nchan)
    d_raw = ctx.dev_alloc(nchan * S * 4)
    tile = rng.integers(-20000, 20000, (64, 2 * S)).astype(np.int16)
    for c0 in range(0, nchan, 64):
        d_raw.upload(tile[: min(64, nchan - c0)], offset=c0 * S * 4)
    for stages in (1, 2, 3):
        bank = J.FUNcubeBPSKDemod(ctx, None, J.AudioDescriptor(rate), tuning=tun, max_block=S, stages=stages)
        ctx.profile(True)
        ms = time_ms(ctx, lambda: bank.receive_dev(d_raw, S, S, s16=True))
        prof = ctx.profile_read()
        ctx.profile(False)
        per = {k: round(v[0] / max(v[1], 1), 3) for k, v in prof.items() if v[1]}
        print(f"chain stages={stages} nchan={nchan} S={S}: {ms:8.3f} ms  {nchan * S / ms / 1e3:9.1f} Msamples/s  per-kernel ms {per}", flush=True)
        bank.close()
    ctx.close()


def pump(nchan=4096, nblk=128, n=4096, rate=192000, reps=6):
    """BASELINE config 5's step (FFT + PSD per block, tuner + 64-tap decimator) through
    jsdr_pump_receive_s16 with device buffers: step time and per-kernel event times."""
    ctx = J.Context(0)
    S = nblk * n
    rng = np.random.default_rng(3)
    tun = rng.uniform(2000, 90000, nchan)
    d_raw = ctx.dev_alloc(nchan * S * 4)
    tile = rng.integers(-20000, 20000, (16, 2 * S)).astype(np.int16)
    for c0 in range(0, nchan, 16):
        d_raw.upload(tile[: min(16, nchan - c0)], offset=c0 * S * 4)
    adsc = J.AudioDescriptor(rate)
    bank = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tun, max_block=S, stages=1)
    bank.set_ds_filter(J.design_lowpass(64, 4800.0, rate))
    f = J.fft(ctx, None, adsc, max_batch=nchan * nblk, n=n)
    d_psd = ctx.dev_alloc(nchan * nblk * (n + 2) * 4)
    d_pk = ctx.dev_alloc(nchan * nblk * 4)
    step = lambda: J.pump_receive_s16(f, bank, d_raw, nblk, d_psd, d_pk, mem=J.MEM_DEVICE)
    for _ in range(3):
        step()
    ctx.sync()
    ctx.profile(True)
    ctx.timer_start()
    for _ in range(reps):
        step()
    ms = ctx.timer_stop_ms() / reps
    prof = ctx.profile_read()
    ctx.profile(False)
    per = {k: round(v[0] / max(v[1], 1), 3) for k, v in prof.items() if v[1]}
    print(f"pump nchan={nchan} nblk={nblk} n={n}: {ms:8.3f} ms/step  {nchan * S / ms / 1e3:9.1f} Msamples/s  per-kernel ms {per}", flush=True)
    ctx.close()


def other(nchan=1024, S=131072, rate=192000):
    """The remaining kernels of the path, device-resident, per-kernel CUDA-event times and the
    achieved GB/s of their algorithmic bytes: demod.java FIR + NCO (:410-434), its detectors
    + AGC + s16 (:448-481), fir.java's int FIR (:198-211), waterfall.java's paintLine (:90-107),
    and the frame stage (sync correlator + FECDecode, FUNcubeBPSKDemod.java:553-574)."""
    import ctypes as C
    L = J.lib()
    ctx = J.Context(0)
    rng = np.random.default_rng(4)
    adsc = J.AudioDescriptor(rate)

    def timed(kind, fn, bytes_, label, reps=5):
        for _ in range(2):
            fn()
        ctx.sync()
        ctx.profile(True)
        ctx.profile_read()
        for _ in range(reps):
            fn()
        prof = ctx.profile_read()
        ctx.profile(False)
        ms = prof[kind][0] / max(prof[kind][1], 1)
        gbs = bytes_ / ms / 1e6
        print(f"{label:58s} {ms:8.4f} ms/launch  {gbs:7.1f} GB/s  frac {gbs / PEAK:.3f}", flush=True)

    # ---- demod.java: 21-tap complex FIR (float, reference order) + float NCO, then detectors
    tile = rng.uniform(-1, 1, (16, 2 * S)).astype(np.float32)
    d_iq = ctx.dev_alloc(nchan * S * 8)
    for c0 in range(0, nchan, 16):
        d_iq.upload(tile[: min(16, nchan - c0)], offset=c0 * S * 8)
    d_out = ctx.dev_alloc(nchan * S * 8)
    dm = J.demod(ctx, adsc, nchan=nchan, max_block=S)
    for c in range(nchan):
        dm.weights(3000, 6000, chan=c)
    dm.set_flags(True, True)
    timed("demod", lambda: J._ck(L.jsdr_demod_receive_f32(dm.h, J._ptr(d_iq), S, S, J._ptr(d_out), J.MEM_DEVICE)),
          nchan * S * 16, f"demod FIR+NCO      nchan={nchan} S={S} (8 B in + 8 B out)")
    d_aud = ctx.dev_alloc(nchan * S * 2)
    d_ma = ctx.dev_alloc(nchan * 8)
    for mode, name in ((2, "AM"), (3, "NFM")):
        dm.set_mode(mode, True)
        timed("detect", lambda: J._ck(L.jsdr_demod_receive_audio_f32(dm.h, J._ptr(d_iq), S, S, J._ptr(d_aud), J._ptr(d_ma), J.MEM_DEVICE)),
              nchan * S * 10, f"demod detect {name:3s}+AGC+s16 nchan={nchan} S={S} (8 B in + 2 B out)")
    dm.close()
    # ---- fir.java: int samples x double taps
    f = J.fir(ctx, float(rate), nchan=nchan, max_block=S)
    for c in range(nchan):
        f.weights(3000, 6000, chan=c)
    d_ii = ctx.dev_alloc(nchan * S * 4)
    ti = rng.integers(-30000, 30000, (16, S)).astype(np.int32)
    for c0 in range(0, nchan, 16):
        d_ii.upload(ti[: min(16, nchan - c0)], offset=c0 * S * 4)
    timed("fir", lambda: J._ck(L.jsdr_fir_filter_i32(f.h, J._ptr(d_ii), S, S, J._ptr(d_out), J.MEM_DEVICE)),
          nchan * S * 8, f"fir.java int FIR    nchan={nchan} S={S} (4 B in + 4 B out)")
    f.close()
    # ---- waterfall rows from a resident PSD
    n, rows, width = 4096, 65536, 1024
    d_psd = ctx.dev_alloc(rows * (n + 2) * 4)
    prow = rng.uniform(-100, 0, (64, n + 2)).astype(np.float32)
    for r0 in range(0, rows, 64):
        d_psd.upload(prow, offset=r0 * (n + 2) * 4)
    d_pix = ctx.dev_alloc(rows * width * 4)
    timed("waterfall", lambda: J._ck(L.jsdr_waterfall_rows(ctx.h, J._ptr(d_psd), n, rows, width, 0x00ffff, J._ptr(d_pix), J.MEM_DEVICE)),
          rows * ((n + 2) * 4 + width * 4), f"waterfall rows      rows={rows} n={n} width={width}")
    for d in (d_iq, d_out, d_aud, d_ma, d_ii, d_psd, d_pix):
        d.free()
    # ---- frame stage: config-2 frames on one shared stream, every tuner of the bank on the signal
    import oracle as O
    from oracle import siggen
    r2 = 96000
    nt = 256
    pl = siggen.random_payloads(3)
    sig = siggen.make_iq_s16(pl, rate=r2, ebn0_db=13.0, pad_to=9600)
    blk = 9600 * 8
    sig = sig[: (sig.size // (2 * blk)) * 2 * blk]
    bank = J.FUNcubeBPSKDemod(ctx, None, J.AudioDescriptor(r2), tuning=np.full(nt, 12000.0), max_block=blk, stages=3)
    mett = np.array([[O.fec_table_probe(6 + r, i) for i in range(256)] for r in range(2)], dtype=np.int16)
    bank.enable_fec(mett, max_frames=nt * 2)
    ctx.profile(True)
    ctx.profile_read()
    nframes = 0
    for k in range(sig.size // (2 * blk)):
        bank.receive_raw(sig[2 * k * blk: 2 * (k + 1) * blk], shared=True)
        nframes += len(bank.read_frames())
    prof = ctx.profile_read()
    ctx.profile(False)
    per = {k: (round(v[0], 3), v[1]) for k, v in prof.items() if v[1]}
    fec_ms, fec_n = prof["fec"]
    print(f"frame stage: {nt} tuners x {sig.size // 2} samples, {nframes} frames decoded; k_fec_decode {fec_ms:.3f} ms over {fec_n} launches "
          f"({1000 * fec_ms / max(nframes, 1):.1f} us per frame at {nt} frames per launch), k_sync {prof['sync'][0]:.3f} ms; all kernels (ms, launches): {per}", flush=True)
    bank.close()
    ctx.close()


def detect(S=32768, rate=192000):
    """demod.java's AM detector + running mean + AGC + s16 (:448-481) against the bank width: the
    running mean is one sequential chain per channel, so the time of a launch is the chain's
    (S samples) as long as the channels fit the machine in one wave (148 SMs x 8 CTAs)."""
    import ctypes as C
    L = J.lib()
    ctx = J.Context(0)
    rng = np.random.default_rng(4)
    adsc = J.AudioDescriptor(rate)
    tile = rng.uniform(-1, 1, (16, 2 * S)).astype(np.float32)
    for nchan in (74, 148, 296, 592, 1184, 2368, 4736):
        d_iq = ctx.dev_alloc(nchan * S * 8)
        for c0 in range(0, nchan, 16):
            d_iq.upload(tile[: min(16, nchan - c0)], offset=c0 * S * 8)
        d_aud = ctx.dev_alloc(nchan * S * 2)
        d_ma = ctx.dev_alloc(nchan * 8)
        dm = J.demod(ctx, adsc, nchan=nchan, max_block=S, dofir=False, dodwn=False)
        for mode, name in ((2, "AM"), (3, "NFM")):
            dm.set_mode(mode, True)
            fn = lambda: J._ck(L.jsdr_demod_receive_audio_f32(dm.h, J._ptr(d_iq), S, S, J._ptr(d_aud), J._ptr(d_ma), J.MEM_DEVICE))
            for _ in range(2):
                fn()
            ctx.sync()
            ctx.profile(True)
            ctx.profile_read()
            for _ in range(5):
                fn()
            prof = ctx.profile_read()
            ctx.profile(False)
            ms = prof["detect"][0] / max(prof["detect"][1], 1)
            gbs = nchan * S * 10 / ms / 1e6
            print(f"detect {name:3s} nchan={nchan:5d} S={S}: {ms:8.4f} ms/launch  {1e6 * ms / S:7.2f} ns per sample of a channel  "
                  f"{gbs:7.1f} GB/s  frac {gbs / PEAK:.3f}", flush=True)
        dm.close()
        for b in (d_iq, d_aud, d_ma):
            b.free()
    ctx.close()


def demod(nchan=1024, S=131072, rate=192000, rounds=4):
    """demod.java's FIR + NCO (:410-434) and the whole receive (NFM, AM with AGC) on float IQ
    (8 B per sample in) against s16 IQ (4 B in, converted as JavaAudio.java:276-293 does), same
    samples, alternated round by round; per-kernel CUDA-event times."""
    L = J.lib()
    ctx = J.Context(0)
    rng = np.random.default_rng(4)
    adsc = J.AudioDescriptor(rate)
    raw = rng.integers(-20000, 20000, (16, 2 * S)).astype(np.int16)
    d_raw, d_iq = ctx.dev_alloc(nchan * S * 4), ctx.dev_alloc(nchan * S * 8)
    fl = np.stack([r.astype(np.float32) / np.float32(32767.0) for r in raw])
    for c0 in range(0, nchan, 16):
        d_raw.upload(raw[: min(16, nchan - c0)], offset=c0 * S * 4)
        d_iq.upload(fl[: min(16, nchan - c0)], offset=c0 * S * 8)
    d_out, d_aud, d_ma = ctx.dev_alloc(nchan * S * 8), ctx.dev_alloc(nchan * S * 2), ctx.dev_alloc(nchan * 8)
    dm = J.demod(ctx, adsc, nchan=nchan, max_block=S)
    for c in range(nchan):
        dm.weights(3000, 6000, chan=c)
    P = J._ptr
    legs = [("FIR+NCO", None, "demod",
             lambda: L.jsdr_demod_receive_f32(dm.h, P(d_iq), S, S, P(d_out), J.MEM_DEVICE),
             lambda: L.jsdr_demod_receive_s16(dm.h, P(d_raw), S, S, 0, 0, P(d_out), J.MEM_DEVICE))]
    for mode, name in ((3, "NFM"), (2, "AM")):
        legs.append((f"audio {name}+AGC", mode, None,
                     lambda: L.jsdr_demod_receive_audio_f32(dm.h, P(d_iq), S, S, P(d_aud), P(d_ma), J.MEM_DEVICE),
                     lambda: L.jsdr_demod_receive_audio_s16(dm.h, P(d_raw), S, S, 0, 0, P(d_aud), P(d_ma), J.MEM_DEVICE)))
    res = {}
    for r in range(rounds):
        for label, mode, kind, f32, s16 in legs:
            if mode is not None:
                dm.set_mode(mode, True)
            for form, fn in (("f32", f32), ("s16", s16)) if r % 2 == 0 else (("s16", s16), ("f32", f32)):
                for _ in range(2):
                    J._ck(fn())
                ctx.sync()
                ctx.profile(True)
                ctx.profile_read()
                ctx.timer_start()
                for _ in range(5):
                    J._ck(fn())
                ms = ctx.timer_stop_ms() / 5
                prof = ctx.profile_read()
                ctx.profile(False)
                k = {kk: round(v[0] / max(v[1], 1), 4) for kk, v in prof.items() if v[1]}
                res.setdefault((label, form), []).append((ms, k))
                print(f"round {r} {label:16s} {form} nchan={nchan} S={S}: {ms:8.4f} ms/call  per-kernel ms {k}", flush=True)
    print("summary (min .. max over rounds; k_demod = 'demod', k_detect = 'detect'):")
    for (label, form), v in res.items():
        calls = [x[0] for x in v]
        kd = [x[1].get("demod", 0.0) for x in v]
        kt = [x[1].get("detect", 0.0) for x in v]
        inb = nchan * S * (4 if form == "s16" else 8)
        gbs = (inb + nchan * S * 8) / min(kd) / 1e6
        print(f"  {label:16s} {form}: call {min(calls):.4f} .. {max(calls):.4f} ms   k_demod {min(kd):.4f} .. {max(kd):.4f} ms "
              f"({gbs:.0f} GB/s in+out, frac {gbs / PEAK:.3f})" + (f"   k_detect {min(kt):.4f} .. {max(kt):.4f} ms" if any(kt) else ""),
              flush=True)
    for x in (d_raw, d_iq, d_out, d_aud, d_ma):
        x.free()
    dm.close()
    ctx.close()


def pumpdemod(nchan=1024, nblk=32, n=4096, rate=192000, rounds=4, reps=6):
    """jsdr_pump_receive_s16 (fft + tuner bank, 64-tap decimator, stages 1) against
    jsdr_pump_demod_s16 (the same plus demod in NFM with AGC) on one resident batch of
    [nchan][nblk*n] s16, device buffers, alternated round by round."""
    ctx = J.Context(0)
    S = nblk * n
    rng = np.random.default_rng(3)
    tun = rng.uniform(2000, 90000, nchan)
    d_raw = ctx.dev_alloc(nchan * S * 4)
    tile = rng.integers(-20000, 20000, (16, 2 * S)).astype(np.int16)
    for c0 in range(0, nchan, 16):
        d_raw.upload(tile[: min(16, nchan - c0)], offset=c0 * S * 4)
    adsc = J.AudioDescriptor(rate)
    bank = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tun, max_block=S, stages=1)
    bank.set_ds_filter(J.design_lowpass(64, 4800.0, rate))
    f = J.fft(ctx, None, adsc, max_batch=nchan * nblk, n=n)
    dm = J.demod(ctx, adsc, nchan=nchan, max_block=S)
    for c in range(nchan):
        dm.weights(3000, 6000, chan=c)
    dm.set_mode(J.demod.MODE_NFM, True)
    d_psd, d_pk = ctx.dev_alloc(nchan * nblk * (n + 2) * 4), ctx.dev_alloc(nchan * nblk * 4)
    d_aud, d_ma = ctx.dev_alloc(nchan * S * 2), ctx.dev_alloc(nchan * nblk * 8)
    steps = {"fft+bank": lambda: J.pump_receive_s16(f, bank, d_raw, nblk, d_psd, d_pk, mem=J.MEM_DEVICE),
             "fft+demod+bank": lambda: J.pump_demod_s16(f, bank, dm, d_raw, nblk, d_psd, d_aud, d_ma, d_pk, mem=J.MEM_DEVICE)}
    res = {}
    for r in range(rounds):
        for name in (list(steps) if r % 2 == 0 else list(steps)[::-1]):
            step = steps[name]
            for _ in range(3):
                step()
            ctx.sync()
            ctx.profile(True)
            ctx.profile_read()
            ctx.profile(False)
            ctx.timer_start()
            for _ in range(reps):
                step()
            ms = ctx.timer_stop_ms() / reps
            ctx.profile(True)
            step()
            prof = ctx.profile_read()
            ctx.profile(False)
            per = {k: round(v[0] / max(v[1], 1), 3) for k, v in prof.items() if v[1]}
            res.setdefault(name, []).append(ms)
            print(f"round {r} pump {name:15s} nchan={nchan} nblk={nblk} n={n}: {ms:8.3f} ms/step  "
                  f"{nchan * S / ms / 1e3:9.1f} Msamples/s  per-kernel ms (profiled step) {per}", flush=True)
    for name, v in res.items():
        print(f"summary pump {name:15s}: {min(v):.3f} .. {max(v):.3f} ms/step", flush=True)
    ctx.close()


def duty(rate=192000, calls=230, warm=30):
    """The reference's own duty (jsdr.java:475-483): ONE stream, one block of rate/10 samples per
    100 ms, the fft handler, the demod handler (NFM) and two FUNcube tuners to bit decisions, host
    buffers, per call through the C ABI, in the form of bench.py's latency leg: the three handlers
    one by one (fft.receive_raw, demod.receive_audio_raw, bank.receive_raw + read_bits) against
    jsdr_pump_demod_s16 (one call; then read_bits), each timed per block, p50 / p99."""
    import time
    ctx = J.Context(0)
    n = rate // 10
    adsc = J.AudioDescriptor(rate)
    rng = np.random.default_rng(5)
    blk = rng.integers(-8000, 8000, 2 * n).astype(np.int16)
    f = J.fft(ctx, None, adsc, max_batch=2, n=n)
    f2 = J.fft(ctx, None, adsc, max_batch=2, n=n)
    bank = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=[12000.0, 14000.0], max_block=n, stages=3)
    bank2 = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=[12000.0, 14000.0], max_block=n, stages=3)
    dm = J.demod(ctx, adsc, nchan=1, max_block=n)
    dm.weights(9000, 15000)
    dm.set_mode(J.demod.MODE_NFM, True)
    # the pump's demod needs one channel per tuner: the two rows of the batch are the same stream
    dm2 = J.demod(ctx, adsc, nchan=2, max_block=n)
    for c in range(2):
        dm2.weights(9000, 15000, chan=c)
    dm2.set_mode(J.demod.MODE_NFM, True)
    two = np.ascontiguousarray(np.stack([blk, blk]))
    psd = np.empty((2, n + 2), np.float32)
    pk = np.empty(2, np.int32)
    aud = np.empty((2, n), np.int16)
    ma = np.empty((2, 1, 2), np.float32)
    t_sep, t_pump = [], []
    for i in range(calls):
        t0 = time.perf_counter()
        f.receive_raw(blk)
        dm.receive_audio_raw(blk)
        bank.receive_raw(blk, shared=True)
        bank.read_bits()
        t1 = time.perf_counter()
        J.pump_demod_s16(f2, bank2, dm2, two, 1, psd, aud, ma, pk)
        bank2.read_bits()
        t2 = time.perf_counter()
        if i >= warm:
            t_sep.append((t1 - t0) * 1e6)
            t_pump.append((t2 - t1) * 1e6)
    pct = lambda v, q: round(float(np.percentile(v, q)), 1)
    out = {"unit": "us", "block": f"N={n} s16 IQ (one 100 ms block at {rate} S/s), MEM_HOST, {calls - warm} calls after {warm} warm-up",
           "handlers_one_by_one_fft_demodNFM_2tuners_to_bits": {"p50": pct(t_sep, 50), "p99": pct(t_sep, 99)},
           "pump_demod_s16_then_read_bits": {"p50": pct(t_pump, 50), "p99": pct(t_pump, 99)},
           "budget_us": 100000,
           "note": "one by one: jsdr_fft_receive_s16, jsdr_demod_receive_audio_s16 (1 channel), jsdr_bpsk_receive_s16 (shared "
                   "stream, 2 tuners) + jsdr_bpsk_read_bits; pump: jsdr_pump_demod_s16 with the block as the row of each of "
                   "the 2 channels (FFT of both rows, demod of both) + jsdr_bpsk_read_bits; includes the ctypes call overhead"}
    print("duty " + json.dumps(out), flush=True)
    for h in (f, f2, bank, bank2, dm, dm2):
        h.close()
    ctx.close()


def card():
    """The device's name and power limit, read in the same run as the numbers they qualify."""
    import subprocess
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:
        q = f"unknown ({e})"
    return f"{name}, power limit / max SM clock: {q}"


def window(ns, total=1 << 31, rounds=4, reps=5):
    """jsdr_fft_set_window: the windowed FFT + PSD against the unwindowed one on the same
    device-resident batch of `total` samples (s16 and f32 input), alternated round by round so
    that both see the same clocks; per call the CUDA-event time of the FFT kernels (JSDR_K_FFT,
    summed over the launches of one call) and of the whole call on the stream."""
    print(f"window: {card()}", flush=True)
    ctx = J.Context(0)
    rng = np.random.default_rng(7)
    tile = rng.integers(-20000, 20000, 1 << 25).astype(np.int16)          # 64 MB
    res = {}
    for n in ns:
        batch = max(1, total // n)
        d_in = ctx.dev_alloc(batch * n * 8)
        for off in range(0, batch * n * 8, tile.nbytes):
            d_in.upload(tile[: min(tile.size, (batch * n * 8 - off) // 2)], offset=off)
        d_psd, d_pk = ctx.dev_alloc(batch * (n + 2) * 4), ctx.dev_alloc(batch * 4)
        adsc = J.AudioDescriptor(192000)
        plain = J.fft(ctx, None, adsc, max_batch=batch, n=n)
        win = J.fft(ctx, None, adsc, max_batch=batch, n=n)
        t = np.arange(n)
        win.set_window((0.54 - 0.46 * np.cos(2.0 * np.pi * t / n)).astype(np.float32))
        legs = {"plain": plain, "hamming": win}
        for r in range(rounds):
            for s16 in (True, False):
                for name in (list(legs) if r % 2 == 0 else list(legs)[::-1]):
                    f = legs[name]
                    fn = lambda: f.receive_dev(d_in, batch, d_psd, d_pk, s16=s16)
                    for _ in range(2):
                        fn()
                    ctx.sync()
                    ctx.profile(True)
                    ctx.profile_read()
                    ctx.timer_start()
                    for _ in range(reps):
                        fn()
                    ms = ctx.timer_stop_ms() / reps
                    prof = ctx.profile_read()
                    ctx.profile(False)
                    kms = prof["fft"][0] / reps
                    fmt = "s16" if s16 else "f32"
                    res.setdefault((n, fmt, name), []).append((kms, ms))
                    print(f"round {r} n={n:6d} batch={batch:7d} {fmt} {name:8s}: FFT kernels {kms:8.3f} ms  call {ms:8.3f} ms",
                          flush=True)
        for d in (d_in, d_psd, d_pk):
            d.free()
        plain.close()
        win.close()
    # (the four-step pair of 65536 runs its chunks on two streams: there the summed kernel time
    # exceeds the call, and the call time is the one to compare)
    print(f"summary ({total} samples per call; min .. max over {rounds} rounds of {reps} calls; {card()}):")
    for n in ns:
        for fmt in ("s16", "f32"):
            for i, what in ((0, "FFT kernels"), (1, "call")):
                p = [v[i] for v in res[(n, fmt, "plain")]]
                w = [v[i] for v in res[(n, fmt, "hamming")]]
                b = (total // n) * n * ((4 if fmt == "s16" else 8) + 4)
                print(f"  n={n:6d} {fmt} {what:11s}: unwindowed {min(p):8.3f} .. {max(p):8.3f} ms   windowed {min(w):8.3f} .. "
                      f"{max(w):8.3f} ms   ratio of minima {min(w) / min(p):.3f}   windowed {b / min(w) / 1e6:7.1f} GB/s of input + PSD",
                      flush=True)
    ctx.close()


if __name__ == "__main__":
    what = sys.argv[1] if len(sys.argv) > 1 else "mix"
    if what == "mix":
        a = [int(x) for x in sys.argv[2:]]
        mix(*a)
    elif what == "pump":
        pump(*[int(x) for x in sys.argv[2:]])
    elif what == "chain":
        chain(*[int(x) for x in sys.argv[2:]])
    elif what == "other":
        other(*[int(x) for x in sys.argv[2:]])
    elif what == "detect":
        detect(*[int(x) for x in sys.argv[2:]])
    elif what == "demod":
        demod(*[int(x) for x in sys.argv[2:]])
    elif what == "pumpdemod":
        pumpdemod(*[int(x) for x in sys.argv[2:]])
    elif what == "duty":
        duty(*[int(x) for x in sys.argv[2:]])
    elif what == "window":
        window([int(x) for x in sys.argv[2:]] or [4096, 19200, 65536])
    else:
        fft([int(x) for x in sys.argv[2:]] or [256, 1024, 4096, 9600, 16384, 19200])

