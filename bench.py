#!/usr/bin/env python
"""bench.py — Msamples/s (complex IQ) through mix + FIR + FFT on B200.

One step = one pass of the hot path over one batch of synthetic s16 IQ
(BASELINE config 4/5): for every channel, every block goes to the fft handler
(FFT + PSD, fft.java:190-228) and the whole stream goes through the FUNcube
tuner + decimating FIR (FUNcubeBPSKDemod.java:382-397, 467-492), via the C ABI's
jsdr_pump_receive_s16 — the batched form of JavaAudio.run's fan-out.

  value   whole-job Msamples/s with the batch resident in HBM
  e2e     the same call with HOST (pinned) buffers: H2D of the raw IQ and D2H of
          the published PSD + a decimated-output read inside the timed region
  roofline  the dominant kernel (FFT+PSD) timed alone with CUDA events
  cpu_baseline  the oracle port of the same pipeline on the host cores (rank 0, N=1)

`--impl reference` times the CPU port only (no JVM / JTransforms jar exists in this
image, so the reference's own Java cannot be run; see DESIGN.md).

Launch: python bench.py [--gpus N --steps K --warmup W]; for N>1 under
torch.distributed.run, one rank per GPU, no data-path collective (channels shard).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "java-sdr_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

RATE = 192000
D = RATE // 9600


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--channels", type=int, default=4096, help="independent streams per GPU")
    ap.add_argument("--fft-n", type=int, default=4096, help="block length (complex samples)")
    ap.add_argument("--blocks", type=int, default=128, help="blocks per channel per step")
    ap.add_argument("--taps", type=int, default=64, help="decimator taps (config 4: 64)")
    ap.add_argument("--precision", default="f64", choices=["f64", "f32"],
                    help="tuner+decimator arithmetic of the headline run: f64 = the reference's binary64, bit-exact")
    ap.add_argument("--e2e-channels", type=int, default=256)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--main-only", action="store_true",
                    help="only the timed step (for ncu runs): skips the variants, latency, e2e and CPU legs; prints a short line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0) as DIR/<name>.npy: a fixed, "
                         "seeded sample of PSD rows, peak bins and decimated channels, at most 64 MB in all")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def measured_traffic():
    """DRAM bytes per input sample of the two data kernels, from the committed ncu --set full
    captures (profiles/traffic.json; written by tools/ncu_summary.py runs)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def workload_name(a):
    return (f"config5: {a.channels} ch x {a.blocks} blk x N={a.fft_n} s16 IQ @192kS/s per GPU "
            f"({a.channels * a.blocks * a.fft_n} samples): FFT+PSD per block + NCO mix + {a.taps}-tap FIR decimate x{D}")


def synth_tile(nchan, S, seed):
    """Synthetic FUNcube-shaped IQ: a BPSK-like carrier near each channel's tuning in noise."""
    rng = np.random.Generator(np.random.PCG64(seed))
    out = rng.integers(-6000, 6000, size=(nchan, 2 * S), dtype=np.int16)
    t = np.arange(S)
    car = (8000 * np.cos(2 * np.pi * 13200.0 / RATE * t)).astype(np.int16)
    sar = (8000 * np.sin(2 * np.pi * 13200.0 / RATE * t)).astype(np.int16)
    out[:, 0::2] += car
    out[:, 1::2] += sar
    return out


def sample_rows(nrows, ncols, itemsize, budget, seed):
    """A fixed, seeded set of rows (ascending) and a leading run of columns of an nrows x ncols
    output, together at most `budget` bytes."""
    rng = np.random.Generator(np.random.PCG64(seed))
    k = int(min(nrows, max(1, budget // max(1, ncols * itemsize))))
    rows = np.sort(rng.choice(nrows, k, replace=False))
    return rows, int(min(ncols, budget // (k * itemsize)))


# bytes per dumped file as stored (PSD float32, peak bins and decimated rows float64):
# 60 MiB = 62.9e6 bytes in all, which leaves room for the .npy headers under 64 MB
DUMP_BUDGET = {"psd": 24 << 20, "peak_bin": 4 << 20, "ds": 32 << 20}


def dump_plan(batch, n, nchan, nds):
    """{name: (rows, cols, itemsize)}: the sample dump_outputs takes of each output of the pump,
    PSD [batch][n+2], peak bins [batch] and decimated rows [nchan][nds] complex."""
    shapes = {"psd": (batch, n + 2, 4), "peak_bin": (batch, 1, 8), "ds": (nchan, nds, 16)}
    return {k: sample_rows(r, c, size, DUMP_BUDGET[k], seed) + (size,)
            for seed, (k, (r, c, size)) in enumerate(shapes.items(), 1)}


def dump_outputs(out_dir, bank, d_psd, d_peak, batch, n):
    """What the caller of jsdr_pump_receive_s16 receives from the last step, sampled by dump_plan."""
    os.makedirs(out_dir, exist_ok=True)
    ds = bank.read_ds()
    plan = dump_plan(batch, n, ds.shape[0], ds.shape[1])
    rows, cols, _ = plan["psd"]
    psd = np.stack([d_psd.download(np.float32, cols, offset=int(r) * (n + 2) * 4) for r in rows])
    rows, _, _ = plan["peak_bin"]
    peak = d_peak.download(np.int32, batch)[rows].astype(np.float64)
    rows, cols, _ = plan["ds"]
    for name, v in (("psd", psd), ("peak_bin", peak), ("ds", ds[rows, :cols])):
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(v))


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md's clocks line).
    NVML from a thread of this process every ~4 ms (no start-up delay, so even a 150 ms region
    gets dozens of samples); `nvidia-smi -lms 20` is the fall-back when NVML cannot be loaded,
    and then start() waits for its first row (a fresh box can take seconds to produce it)."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.rows, self.proc, self.nvml, self.th = device, [], None, None, None
        self.source = None
        self._stop = threading.Event()

    @staticmethod
    def physical_index(local):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        ids = [v.strip() for v in vis.split(",") if v.strip()]
        if local < len(ids) and ids[local].isdigit():
            return int(ids[local])
        return local

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.physical_index(self.device))
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            pynvml.nvmlDeviceGetClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.nvml, self.source = pynvml, "nvml"
            self.th = threading.Thread(target=self._poll_nvml, daemon=True)
            self.th.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.physical_index(self.device))],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi"
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
            t_end = time.time() + 15.0
            while not self.rows and time.time() < t_end and self.proc.poll() is None:
                time.sleep(0.02)
        except Exception:
            self.proc = None

    def _poll_nvml(self):
        n = self.nvml
        names = (("hw_slowdown", n.nvmlClocksEventReasonHwSlowdown),
                 ("hw_thermal_slowdown", n.nvmlClocksEventReasonHwThermalSlowdown),
                 ("sw_thermal_slowdown", n.nvmlClocksEventReasonSwThermalSlowdown),
                 ("sw_power_cap", n.nvmlClocksEventReasonSwPowerCap))
        while not self._stop.is_set():
            try:
                sm = float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM))
                try:
                    mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                r = ["", sm, self.mx, "", ""] + ["Active" if mask & bit else "Not Active" for _, bit in names]
                self.rows.append((time.time(), r))
            except Exception:
                pass
            self._stop.wait(0.004)

    def _read(self):
        import datetime
        for line in self.proc.stdout:
            r = [c.strip() for c in line.split(",")]
            try:        # nvidia-smi's own timestamp (its stdout reaches us in bursts)
                ts = datetime.datetime.strptime(r[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except Exception:
                ts = time.time()
            self.rows.append((ts, r))

    def window(self, t0, t1):
        """Keep the samples taken inside the timed region (host clock, 30 ms slack)."""
        self.t0, self.t1 = t0 - 0.03, t1 + 0.03

    def stop(self):
        if self.nvml is not None:
            self._stop.set()
            self.th.join(timeout=1.0)
        elif self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
            try:
                self.th.join(timeout=1.0)
            except Exception:
                pass
        else:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["no NVML and no nvidia-smi on this host"]}
        sm, mx, reasons = [], [], set()
        t0, t1 = getattr(self, "t0", None), getattr(self, "t1", None)
        rows = [(ts, r) for ts, r in self.rows if t0 is None or t0 <= ts <= t1]
        scope = "timed region"
        if len(rows) < 3:   # too short a region for the sampling period: everything since before the warm-up
            rows, scope = self.rows, "warm-up + timed region"
        for ts, r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if str(v).lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "scope": scope, "source": self.source, "reasons": sorted(reasons)}


def cpu_pipeline(a, seconds, nthreads):
    """The oracle port of the same pipeline on a bounded sample; returns the cpu_baseline object.
    Timed with the FFT plan cached per thread and modulo-free loops (oracle fft mode 1): that is
    MORE favourable to the CPU than the reference's own code, which builds a new FloatFFT_1D for
    every block (fft.java:194); the plan-per-block form is timed on a short sample beside it."""
    import oracle as O
    from oracle import siggen
    taps = siggen.lowpass_taps(a.taps, 4800.0, RATE)
    nblk = 1
    probe_ch = max(nthreads, 1) * 2
    rng = np.random.Generator(np.random.PCG64(7))
    def run(nch):
        raw = synth_tile(nch, nblk * a.fft_n, 99)
        tun = rng.uniform(2000, 90000, nch)
        t0 = time.perf_counter()
        _, _, used = O.baseline_pipeline_s16(raw, nch, nblk, a.fft_n, RATE, tun, taps, nthreads)
        return time.perf_counter() - t0, used
    O.baseline_set_fft_mode(1)
    dt, used = run(probe_ch)
    per_ch = dt / probe_ch
    nch = int(max(probe_ch, min(seconds / max(per_ch, 1e-9), 200000)))
    nch = (nch // max(nthreads, 1)) * max(nthreads, 1)
    dt, used = run(nch)
    v = nch * nblk * a.fft_n / dt / 1e6
    O.baseline_set_fft_mode(0)
    nch0 = max(probe_ch, nch // 8)
    dt0, _ = run(nch0)
    v0 = nch0 * nblk * a.fft_n / dt0 / 1e6
    return {"value": round(v, 3), "unit": "Msamples/s", "cores": used, "kind": "port",
            "sample": f"{nch} channels x {nblk} block x N={a.fft_n} of the same pipeline "
                      f"(s16->float, float FFT + PSD, tuner + {a.taps}-tap decimator), "
                      f"{dt:.1f} s on {used} threads; C port of the Java arithmetic (no JVM in this image), "
                      f"FFT plan cached per thread",
            "plan_per_block": {"value": round(v0, 3), "unit": "Msamples/s",
                               "note": "the same with the FFT plan and twiddle table rebuilt for every block, "
                                       "as fft.java:194 does (new FloatFFT_1D per receive)"}}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    nthreads = os.cpu_count() or 1
    per_step = max(2.0, min(20.0, 120.0 / max(a.steps + a.warmup, 1)))
    for _ in range(a.warmup):
        cpu_pipeline(a, min(per_step, 2.0), nthreads)
    vals, last = [], None
    t0 = time.perf_counter()
    for _ in range(a.steps):
        last = cpu_pipeline(a, per_step, nthreads)
        vals.append(last["value"])
    wall = time.perf_counter() - t0
    v = float(np.mean(vals))
    last["value"] = round(v, 3)
    line = {"impl": "reference", "metric": "Msamples/s (complex IQ) through mix+FIR+FFT", "value": round(v, 3),
            "unit": "Msamples/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": round(1000 * wall / max(a.steps, 1), 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(a), "note": "CPU port of the reference on the host cores, bounded sample per step"},
            "cpu_baseline": last,
            "e2e": {"value": round(v, 3), "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    a = parse()
    if a.impl == "reference":
        run_reference(a)
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    import jsdrcuda as J

    ctx = J.Context(local)
    adsc = J.AudioDescriptor(RATE)
    n, nblk, nchan = a.fft_n, a.blocks, a.channels
    S = n * nblk
    batch = nchan * nblk
    samples = nchan * S

    # weak scaling: every rank owns a.channels channels of a (world * a.channels)-channel bank;
    # a channel's tuning depends on its global index only (jsdrcuda/sharding.py)
    from jsdrcuda import sharding
    first, _ = sharding.partition(world * nchan, world, rank)
    tuning = sharding.channel_tuning(first, nchan)
    taps = J.design_lowpass(a.taps, 4800.0, RATE)

    f = J.fft(ctx, None, adsc, max_batch=batch, n=n)
    bank = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tuning, max_block=S, stages=1)
    bank.set_ds_filter(taps)
    bank.set_precision(J.PREC_F32 if a.precision == "f32" else J.PREC_F64)

    d_raw = ctx.dev_alloc(samples * 4)
    d_psd = ctx.dev_alloc(batch * (n + 2) * 4)
    d_peak = ctx.dev_alloc(batch * 4)
    # fill the resident batch from a 64-channel synthetic tile
    tile_ch = min(64, nchan)
    tile = synth_tile(tile_ch, S, 1000 + rank)
    for c0 in range(0, nchan, tile_ch):
        k = min(tile_ch, nchan - c0)
        d_raw.upload(tile[:k], offset=c0 * S * 4)

    def step():
        J.pump_receive_s16(f, bank, d_raw, nblk, d_psd, d_peak, mem=J.MEM_DEVICE)

    def barrier():
        ctx.sync()
        if dist is not None:
            dist.barrier()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()          # nvidia-smi needs a moment to start: begin before the warm-up
    for _ in range(a.warmup):
        step()
    barrier()
    l0 = ctx.launch_count()
    ctx.profile(True)            # CUDA events around every kernel launch, on the stream it is launched on
    ctx.profile_read()
    t_wall0 = time.time()
    ctx.timer_start()
    for _ in range(a.steps):
        step()
    ms = ctx.timer_stop_ms()
    sampler.window(t_wall0, time.time())
    launches = ctx.launch_count() - l0
    kern = ctx.profile_read()    # {kind: (total ms, launches)} inside the timed region
    ctx.profile(False)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, bank, d_psd, d_peak, batch, n)
    fft_ms = kern["fft"][0] / max(kern["fft"][1], 1)
    mix_ms = kern["mixdecim"][0] / max(kern["mixdecim"][1], 1)
    scout_ms = kern["scout"][0] / max(kern["scout"][1], 1)

    if a.main_only:
        if rank == 0:
            print(json.dumps({"main_only": True, "ms_per_step": round(ms / a.steps, 4), "fft_ms": round(fft_ms, 4),
                              "mixdecim_ms": round(mix_ms, 4), "scout_ms": round(scout_ms, 4), "gpu_launches": int(launches)}), flush=True)
        for h in (f, bank):
            h.close()
        ctx.close()
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- the FFT kernel with the SMs to itself (no phase scout beside it), for the record
    ctx.sync()
    for _ in range(2):
        f.receive_dev(d_raw, batch, d_psd, d_peak, s16=True)
    ctx.sync()
    ctx.timer_start()
    for _ in range(5):
        f.receive_dev(d_raw, batch, d_psd, d_peak, s16=True)
    fft_alone_ms = ctx.timer_stop_ms() / 5

    # ---- the other decimator arithmetic, same pipeline, for the record (rank-local, few steps)
    other = "f32" if a.precision == "f64" else "f64"
    bank.set_precision(J.PREC_F32 if other == "f32" else J.PREC_F64)
    for _ in range(2):
        step()
    ctx.sync()
    ctx.timer_start()
    for _ in range(max(2, a.steps // 2)):
        step()
    other_ms = ctx.timer_stop_ms() / max(2, a.steps // 2)
    bank.set_precision(J.PREC_F32 if a.precision == "f32" else J.PREC_F64)

    # ---- BASELINE config 4 on its own: NCO mix + 64-tap FIR decimation of every channel, no FFT
    for _ in range(2):
        bank.receive_dev(d_raw, S, S, s16=True)
    ctx.sync()
    ctx.timer_start()
    for _ in range(3):
        bank.receive_dev(d_raw, S, S, s16=True)
    mixonly_ms = ctx.timer_stop_ms() / 3

    # ---- the whole FUNcube chain to bits (27-tap decimator, matched filter, bit timing) on the
    # same resident batch, for the record: the reference's own receiver shape at 192 kS/s
    bank_c = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tuning, max_block=S, stages=3)
    for _ in range(2):
        bank_c.receive_dev(d_raw, S, S, s16=True)
    ctx.sync()
    ctx.timer_start()
    for _ in range(3):
        bank_c.receive_dev(d_raw, S, S, s16=True)
    chain_ms = ctx.timer_stop_ms() / 3
    bank_c.close()

    # ---- the same step at the reference's own block lengths, N = rate/10 (fft.java:67,
    # JavaAudio.java:59): 19200 at 192 kS/s (D = 20) and 9600 at 96 kS/s (D = 10), same resident batch
    # (as many whole blocks per channel as fit in the 2^31-sample buffer)
    def rate10_variant(vrate):
        vn = vrate // 10
        vblk = S // vn
        vS = vblk * vn
        vadsc = J.AudioDescriptor(vrate)
        vf = J.fft(ctx, None, vadsc, max_batch=nchan * vblk, n=vn)
        vbank = J.FUNcubeBPSKDemod(ctx, None, vadsc, tuning=tuning * (vrate / RATE), max_block=vS, stages=1)
        vtaps = a.taps if vrate == RATE else 27          # 96 kS/s: the reference's own 27-tap low-pass (:27-55)
        if vtaps != 27:
            vbank.set_ds_filter(J.design_lowpass(vtaps, 4800.0, vrate))
        vbank.set_precision(J.PREC_F32 if a.precision == "f32" else J.PREC_F64)
        vstep = lambda: J.pump_receive_s16(vf, vbank, d_raw, vblk, d_psd, d_peak, mem=J.MEM_DEVICE)
        for _ in range(3):
            vstep()
        ctx.sync()
        ctx.profile(True)
        ctx.profile_read()
        ctx.timer_start()
        reps = max(3, a.steps // 4)
        for _ in range(reps):
            vstep()
        vms = ctx.timer_stop_ms() / reps
        vk = ctx.profile_read()
        ctx.profile(False)
        vf.close()
        vbank.close()
        return {"n": vn, "rate": vrate, "blocks": vblk, "samples": nchan * vS, "ms": vms, "taps": vtaps,
                "fft_ms": vk["fft"][0] / max(vk["fft"][1], 1), "mix_ms": vk["mixdecim"][0] / max(vk["mixdecim"][1], 1)}
    v192 = rate10_variant(192000)
    v96 = rate10_variant(96000)

    # ---- latency at the reference's operating point: ONE stream, one block of rate/10 samples
    # per 100 ms (JavaAudio.java:231-233), the fft handler and two FUNcube tuners on it
    # (jsdr.java:476,479), host buffers, results back in host memory — per call, through the C ABI
    lat = None
    if rank == 0:
        ln = RATE // 10
        f_l = J.fft(ctx, None, adsc, max_batch=1, n=ln)
        bank_l = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=[12000.0, 14000.0], max_block=ln, stages=3)
        blk = synth_tile(1, ln, 5)[0]
        t_fft, t_bpsk = [], []
        for i in range(230):
            t0 = time.perf_counter()
            f_l.receive_raw(blk)
            t1 = time.perf_counter()
            bank_l.receive_raw(blk, shared=True)
            bank_l.read_bits()
            t2 = time.perf_counter()
            if i >= 30:
                t_fft.append((t1 - t0) * 1e6)
                t_bpsk.append((t2 - t1) * 1e6)
        f_l.close()
        bank_l.close()
        pct = lambda v, q: round(float(np.percentile(v, q)), 1)
        lat = {"unit": "us", "block": f"N={ln} s16 IQ (one 100 ms block at 192 kS/s), MEM_HOST, 200 calls after 30 warm-up",
               "fft_receive_s16": {"p50": pct(t_fft, 50), "p99": pct(t_fft, 99)},
               "bpsk_receive_s16_2_tuners_to_bits": {"p50": pct(t_bpsk, 50), "p99": pct(t_bpsk, 99)},
               "budget_us": 100000,
               "note": "jsdr_fft_receive_s16 (H2D, FFT+PSD, D2H) and jsdr_bpsk_receive_s16 + jsdr_bpsk_read_bits "
                       "(shared stream, tuner .. bit decisions) as the patched java-sdr handlers call them; "
                       "includes the ctypes call overhead"}

    # ---- end to end through the C ABI with host (pinned) buffers
    e_ch = min(a.e2e_channels, nchan)
    e_batch = e_ch * nblk
    bank_e = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tuning[:e_ch], max_block=S, stages=1)
    bank_e.set_ds_filter(taps)
    f_e = J.fft(ctx, None, adsc, max_batch=e_batch, n=n)
    h_raw = ctx.host_alloc((e_ch, 2 * S), np.int16)
    h_psd = ctx.host_alloc((e_batch, n + 2), np.float32)
    h_pk = ctx.host_alloc((e_batch,), np.int32)
    h_ds = ctx.host_alloc((e_ch, S // D + 1, 2), np.float64)   # the carry makes the count vary by one per call
    h_raw[:] = tile[np.arange(e_ch) % tile_ch]
    def e2e_step():
        J.pump_receive_s16(f_e, bank_e, h_raw, nblk, h_psd, h_pk, mem=J.MEM_HOST)   # H2D raw, D2H PSD inside
        # D2H of the decimated output on the download stream: it drains beside the next step's
        # upload (PCIe is full duplex); the sync that closes the timed region waits for the last one
        bank_e.read_ds_async(h_ds)
    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        e2e_step()
    ctx.sync()
    e2e_s = (time.perf_counter() - t0) / a.steps
    e2e_samples = e_ch * S
    h2d = h_raw.nbytes
    d2h = h_psd.nbytes + h_pk.nbytes + h_ds.nbytes
    # the same with waterfall.java's paintLine on the device: pixel rows come back instead of the PSD
    WF_W = 1024
    h_pix = ctx.host_alloc((e_batch, WF_W), np.int32)
    h_peak = ctx.host_alloc((e_batch, 2), np.float32)
    def e2e_wf_step():
        J.pump_waterfall_s16(f_e, bank_e, h_raw, nblk, WF_W, h_pix, h_peak, h_pk, mem=J.MEM_HOST)
        bank_e.read_ds_async(h_ds)
    for _ in range(2):
        e2e_wf_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        e2e_wf_step()
    ctx.sync()
    e2e_wf_s = (time.perf_counter() - t0) / a.steps
    d2h_wf = h_pix.nbytes + h_peak.nbytes + h_pk.nbytes + h_ds.nbytes

    # ---- reduce over ranks: max time, summed work
    t_step = ms / a.steps
    dev = None
    if dist is not None:
        import torch
        dev = torch.device("cuda", local)
    (t_step, fft_ms, mix_ms, e2e_s, other_ms, scout_ms, chain_ms, mixonly_ms, v192["ms"], v192["fft_ms"], v96["ms"],
     v96["fft_ms"], e2e_wf_s), launches = sharding.reduce_timing(
        dist, dev, [t_step, fft_ms, mix_ms, e2e_s, other_ms, scout_ms, chain_ms, mixonly_ms, v192["ms"], v192["fft_ms"],
                    v96["ms"], v96["fft_ms"], e2e_wf_s], launches)
    launches = int(launches)

    if rank == 0:
        peak, peak_src = peaks()
        value = world * samples / (t_step * 1e-3) / 1e6
        nout = nchan * (S // D)
        fft_bytes = samples * 8 + batch * 8            # s16 in (4 B) + float PSD out (4 B) per sample, + 2 floats per block
        mix_bytes = samples * 4 + nout * 16            # s16 in + complex double out
        step_bytes = samples * 4 + samples * 4 + nout * 16
        traffic = measured_traffic()
        kernels = [
            {"kernel": "k_mixdecim_stream (NCO mix + %d-tap FIR decimate x%d, %s)" % (a.taps, D, a.precision),
             "ms_per_launch": round(mix_ms, 4), "algorithmic_bytes_per_launch": mix_bytes,
             "traffic": traffic.get("mixdecim_bytes_per_sample") and int(traffic["mixdecim_bytes_per_sample"] * samples)},
            {"kernel": "fft_kernel (FFT N=%d + PSD, s16 in)" % n,
             "ms_per_launch": round(fft_ms, 4), "algorithmic_bytes_per_launch": fft_bytes,
             "traffic": traffic.get("fft_bytes_per_sample") and int(traffic["fft_bytes_per_sample"] * samples)},
        ]
        for k in kernels:
            k["achieved"] = round(k["algorithmic_bytes_per_launch"] / (k["ms_per_launch"] * 1e-3) / 1e9, 1)
            k["frac"] = round(k["achieved"] / peak, 4)
        kernels.sort(key=lambda k: -k["ms_per_launch"])
        dom = kernels[0]
        line = {
            "metric": "Msamples/s (complex IQ) through mix+FIR+FFT",
            "value": round(value, 1), "unit": "Msamples/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": round(t_step, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 (FFT/PSD) + %s (tuner/decimator%s)" % (a.precision, ", reference order, bit-exact" if a.precision == "f64" else ""),
            "data": "synthetic",
            "config": {"workload": workload_name(a), "channels_per_gpu": nchan, "blocks_per_channel": nblk,
                       "fft_n": n, "rate": RATE, "decimation": D, "taps": a.taps,
                       "l2": "inputs larger than L2 (%.1f GiB resident per GPU)" % (samples * 4 / 2 ** 30),
                       "sharding": "channels split across ranks, no collective"},
            "roofline": {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["achieved"],
                         "peak": peak, "unit": "GB/s", "frac": dom["frac"], "traffic": dom["traffic"],
                         "peak_source": peak_src + " copy bandwidth (MEASURED_PEAKS.json)",
                         "algorithmic_bytes_per_launch": dom["algorithmic_bytes_per_launch"],
                         "ms_per_launch": dom["ms_per_launch"],
                         "timing": "CUDA events around each launch on its own stream, averaged over the timed region",
                         "fft_kernel_alone": {"ms_per_launch": round(fft_alone_ms, 4),
                                              "achieved": round(fft_bytes / (fft_alone_ms * 1e-3) / 1e9, 1),
                                              "frac": round(fft_bytes / (fft_alone_ms * 1e-3) / 1e9 / peak, 4),
                                              "note": "same launch outside the pipeline (rank 0): in the step the phase scout "
                                                      "of the next block holds 16 SMs beside it"},
                         "other_kernels": kernels[1:] + [{"kernel": "k_tuner_scout (exact tuner phase replay, side stream, overlapped)",
                                                          "ms_per_launch": round(scout_ms, 4)}],
                         "pipeline": {"algorithmic_bytes_per_step_fused": step_bytes,
                                      "achieved": round(step_bytes / (t_step * 1e-3) / 1e9, 1),
                                      "frac": round(step_bytes / (t_step * 1e-3) / 1e9 / peak, 4),
                                      "note": "4 B in (read once) + 4 B PSD + 16/D B decimated out per sample"}},
            "variants": {"decimator_" + other: {"value": round(world * samples / (other_ms * 1e-3) / 1e6, 1),
                                                "unit": "Msamples/s", "ms_per_step": round(other_ms, 4),
                                                "note": "same pipeline with the tuner+decimator in %s" % other},
                         "tuner_decimator_only": {"value": round(world * samples / (mixonly_ms * 1e-3) / 1e6, 1),
                                                  "unit": "Msamples/s", "ms_per_step": round(mixonly_ms, 4),
                                                  "frac_of_hbm_peak": round((samples * 4 + nout * 16) / (mixonly_ms * 1e-3) / 1e9 / peak, 4),
                                                  "note": "BASELINE config 4 alone: NCO mix + %d-tap FIR decimate x%d (%s), "
                                                          "4 + 16/D algorithmic bytes per sample" % (a.taps, D, a.precision)},
                         **{"fft_n%d" % v["n"]: {
                             "value": round(world * v["samples"] / (v["ms"] * 1e-3) / 1e6, 1), "unit": "Msamples/s",
                             "ms_per_step": round(v["ms"], 4),
                             "fft_ms_per_launch": round(v["fft_ms"], 4),
                             "fft_frac_of_hbm_peak": round((v["samples"] * 8 + nchan * v["blocks"] * 8) / (v["fft_ms"] * 1e-3) / 1e9 / peak, 4),
                             "pipeline_frac_of_hbm_peak": round((v["samples"] * 8 + nchan * (v["blocks"] * v["n"] // (v["rate"] // 9600)) * 16)
                                                                / (v["ms"] * 1e-3) / 1e9 / peak, 4),
                             "note": "the same step at the reference's own block length N = rate/10 (fft.java:67): %d ch x %d blk x "
                                     "N=%d @ %d kS/s, %d-tap decimate x%d" % (nchan, v["blocks"], v["n"], v["rate"] // 1000, v["taps"], v["rate"] // 9600)}
                            for v in (v192, v96)},
                         "e2e_waterfall_rows": {"value": round(world * e2e_samples / e2e_wf_s / 1e6, 1), "unit": "Msamples/s",
                                                "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h_wf),
                                                "note": "e2e with waterfall.java's paintLine on the device (jsdr_pump_waterfall_s16, "
                                                        "%d-pixel rows): pixel rows + peak values + decimated rows return instead of the PSD" % WF_W},
                         "funcube_chain_to_bits": {"value": round(world * samples / (chain_ms * 1e-3) / 1e6, 1),
                                                   "unit": "Msamples/s", "ms_per_step": round(chain_ms, 4),
                                                   "note": "tuner + 27-tap decimator + 65-tap matched filter + bit timing "
                                                           "(FUNcubeBPSKDemod.java:382-595), bit-exact, same resident batch"}},
            "e2e": {"value": round(world * e2e_samples / e2e_s / 1e6, 1), "unit": "Msamples/s",
                    "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "sample": f"{e_ch} channels x {nblk} blocks per rank through jsdr_pump_receive_s16 + jsdr_bpsk_read_ds with pinned host buffers"},
            "latency": lat,
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        if not a.no_cpu and world == 1:
            line["cpu_baseline"] = cpu_pipeline(a, a.cpu_seconds, os.cpu_count() or 1)
        print(json.dumps(line), flush=True)

    for h in (f, bank, f_e, bank_e):
        h.close()
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
