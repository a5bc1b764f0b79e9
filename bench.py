#!/usr/bin/env python3
"""bench.py -- throughput of the STFT phase-vocoder hot path on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W          (N > 1: launched by torch.distributed.run)
  python bench.py --impl reference ...                   the reference's own CPU implementation
  python bench.py ... --dump-outputs DIR                 also save the last timed step's output (DIR/output.npy)

Workload (BASELINE.json configs[1]): batch 1024 stereo streams per GPU, 48 kHz presetDefault,
0.8x time-stretch (outputSamples = 0.8 * inputSamples, cmd/main.cpp:27,37 semantics), synthetic
harmonic audio.  One STEP = one process() call over the whole batch carrying 32 blocks per stream
(46 080 output / 57 600 input samples per channel = 0.96 s of output audio).
Metric: audio output samples per second, counted per channel (batch * channels * outputSamples / t).

* value      device-resident: inputs already in HBM, CUDA events on the engine's stream;
* e2e        the same call through the host-buffer C ABI (b200s_process) from/to PINNED host memory,
             host->device and device->host copies inside the timed region;
* roofline   algorithmic bytes (SURVEY.md section 8(d): 129.2 B per output sample for this config)
             over the measured device time, against MEASURED_PEAKS.json's HBM copy bandwidth;
* cpu_baseline  the reference's own binary (oracle/_ref, kind "reference") on the host cores.
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
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SR = 48000
CHANNELS = 2
BATCH_PER_GPU = 1024
BLOCKS_PER_STEP = 32
RATIO_OUT = 0.8  # output length / input length
# SURVEY.md section 8(d): compulsory HBM traffic per block-channel for this configuration
# (input read + history append + 2 analysis gathers + output/energy state + OLA ring + output)
ALGO_BYTES_PER_BLOCK_CHANNEL = 186048
# --config 3 / 4 (not the driver's default): BASELINE configs[2] / [3] on one GPU, rate 1
# (no re-analysis: 209 280 B per block-channel, SURVEY.md section 8(d))
EXTRA = {3: dict(channels=1, semitones=7.0, tonality=8000.0 / 48000, formant=False, algo=209280,
                 name="BASELINE configs[2]: batch=1024/GPU mono 48 kHz presetDefault, +7 semitones, 8 kHz tonality limit"),
         4: dict(channels=2, semitones=12.0, tonality=0.0, formant=True, algo=209280,
                 name="BASELINE configs[3]: stereo 48 kHz presetDefault, +12 semitones, formant compensation, base 200 Hz")}
METRIC = "audio output samples/sec (batched streams, per channel)"


def workload(batch):
    H = int(SR * 0.03)
    n_out = BLOCKS_PER_STEP * H
    n_in = int(round(n_out / RATIO_OUT))
    return {"batch": batch, "channels": CHANNELS, "n_in": n_in, "n_out": n_out, "interval": H,
            "samples_per_step": batch * CHANNELS * n_out}


def config_dict(w, n_gpus):
    return {"workload": "BASELINE configs[1]: batch=%d stereo 48 kHz presetDefault, 0.8x time-stretch, per GPU" % BATCH_PER_GPU,
            "global_batch": w["batch"] * n_gpus, "batch_per_gpu": w["batch"], "channels": CHANNELS, "sample_rate": SR,
            "preset": "presetDefault", "out_over_in": RATIO_OUT, "blocks_per_step": BLOCKS_PER_STEP,
            "output_samples_per_step": w["n_out"], "input_samples_per_step": w["n_in"],
            "parallelism": "streams sharded contiguously, %d rank(s), no data-path collective" % n_gpus,
            "l2": "inputs (%.0f MB/step, 3 rotating buffers) larger than L2" % (w["batch"] * CHANNELS * w["n_in"] * 4 / 1e6)}


def synth_input(batch, n, seed0=0):
    """[batch][C][n] float32; cheap vectorised version of tests/signals.harmonic (seed = stream)."""
    t = np.arange(n, dtype=np.float64) / SR
    s = (np.arange(batch) + seed0)[:, None, None]
    c = np.arange(CHANNELS)[None, :, None]
    f0 = 110.0 * (1 + 0.01 * (s % 97)) * (1 + 0.05 * c)
    ph = 2 * np.pi * f0 * t[None, None, :] + 3 * np.sin(2 * np.pi * 0.7 * t)[None, None, :]
    x = np.zeros((batch, CHANNELS, n))
    for k in range(6):
        x += np.sin((k + 1) * ph) / (k + 1)
    x *= (1 + 0.3 * np.sin(2 * np.pi * 2 * t))[None, None, :] * 0.2
    rng = np.random.default_rng(1234 + seed0)
    x += 0.01 * rng.standard_normal(x.shape)
    return x.astype(np.float32)


DUMP_STREAMS = 64


def dump_outputs(out_dir, y_dev):
    """DIR/output.npy: what the last timed process() call returned, float32 [streams][channels][samples], for a fixed
    seeded sample of DUMP_STREAMS streams of the batch in ascending order (the whole batch when it is smaller), so that
    two builds run with the same arguments can be compared output for output."""
    import torch

    streams = np.sort(np.random.default_rng(0).choice(y_dev.shape[0], min(DUMP_STREAMS, y_dev.shape[0]), replace=False))
    y = y_dev[torch.from_numpy(streams).to(y_dev.device)].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "output.npy"), y)


# ------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML polled every ~2 ms from a thread (the timed
    region of the default run is ~50 ms, shorter than one nvidia-smi period); nvidia-smi -lms as the fallback."""
    Q = "clocks.sm,clocks.max.sm,clocks.mem,power.draw,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []
        self.nvml, self.handle, self.stop_flag, self.samples, self.mask, self.max_mhz = None, None, False, [], 0, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                self.samples.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
                self.mask |= int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nvml:
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml:
            self.stop_flag = True
            self.th.join(timeout=1)
            return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                    "reasons": sorted(nm for bit, nm in self.REASONS.items() if self.mask & bit), "samples": len(self.samples),
                    "source": "NVML, 2 ms polling during the timed region"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [v.strip() for v in ln.split(",")]
            if len(p) < 8:
                continue
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
            except ValueError:
                continue
            for nm, v in zip(names, p[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi -lms 100"}


# ------------------------------------------------------------------------------------ host cores / NUMA
def host_cores():
    """The CPUs this process may actually use: affinity mask, cgroup CPU quota, physical cores (os.cpu_count() is none
    of these: on a leased box it reports every logical CPU of the host)."""
    aff = sorted(os.sched_getaffinity(0))
    quota = None
    try:  # cgroup v2
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:  # cgroup v1
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    phys = set()
    try:
        cur = {}
        for ln in list(open("/proc/cpuinfo")) + [""]:
            if ":" in ln:
                k, v = [t.strip() for t in ln.split(":", 1)]
                cur[k] = v
            elif not ln.strip() and cur:
                if int(cur.get("processor", -1)) in aff:
                    phys.add((cur.get("physical id", "0"), cur.get("core id", cur.get("processor"))))
                cur = {}
    except Exception:
        pass
    usable = len(aff)
    if quota is not None:
        usable = max(1, min(usable, int(quota + 0.5)))
    return {"logical_cpus": os.cpu_count(), "affinity_cpus": len(aff), "cgroup_quota_cpus": quota,
            "physical_cores_in_affinity": len(phys) or None, "usable": usable}


def bind_to_gpu_numa(index):
    """Pin this rank (and therefore the first-touch placement of the pinned host buffers it allocates afterwards) to
    the CPUs local to its GPU.  GPUs 0-3 / 4-7 of an 8-GPU HGX box hang off different sockets; without this every rank's
    staging memory lands on whichever node the launcher ran on and half of the PCIe traffic crosses the socket link."""
    info = {"bound": False}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n_words = ((os.cpu_count() or 64) + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        cur = os.sched_getaffinity(0)
        want = cpus & cur
        info["gpu_local_cpus"] = len(cpus)
        try:
            bus = pynvml.nvmlDeviceGetPciInfo(h).busId
            bus = bus.decode() if isinstance(bus, bytes) else bus
            info["numa_node"] = int(open("/sys/bus/pci/devices/%s/numa_node" % bus.lower()[-12:]).read())
        except Exception:
            info["numa_node"] = None
        if want and want != cur:
            os.sched_setaffinity(0, want)
            info["bound"] = True
        info["cpus_after"] = len(os.sched_getaffinity(0))
    except Exception as ex:  # noqa: BLE001
        info["error"] = str(ex)[-120:]
    return info


# ------------------------------------------------------------------------------------ CPU reference
_CPU_INPUT = {}


def cpu_reference_run(n_streams, seconds_per_stream, threads, fast=False):
    """The reference's own implementation of this workload on the host cores.
    kind "reference": the shipped WASM binary translated to C (oracle/_ref/libwasm_stretch.so, gcc -O2 -ffp-contract=off;
    fast=True: the same translation built -O3 -ffast-math -mavx2 -mfma, BASELINE.md section 3);
    falls back to the oracle restatement ("port") only if that file is absent.
    Timed: the process() calls only (instance creation and presetDefault excluded), wall clock of the thread pool."""
    import ctypes

    from oracle import hdrref, wasmref

    H = int(SR * 0.03)
    n_out_total = int(seconds_per_stream * SR) // H * H
    chunk = 480  # BASELINE.md section 3: 480-sample output chunks
    n_in_total = int(round(n_out_total / RATIO_OUT))
    # a pool of 64 distinct synthetic streams, tiled over the batch (generating 1024 distinct ones costs several times
    # the timed run itself; the reference's cost does not depend on the data)
    key = (n_streams, n_in_total)
    if _CPU_INPUT.get("key") != key:
        pool = synth_input(min(n_streams, 64), n_in_total)
        _CPU_INPUT["x"] = np.ascontiguousarray(np.tile(pool, ((n_streams + len(pool) - 1) // len(pool), 1, 1))[:n_streams])
        _CPU_INPUT["key"] = key
    x = _CPU_INPUT["x"]
    wall_total = None
    fast_path = os.path.join(os.path.dirname(wasmref.lib_path()), "libwasm_stretch_fast.so")
    if wasmref.available() and (not fast or os.path.exists(fast_path)):
        # native pthread pool, one reference instance per stream (oracle/ref_bench.c)
        L = ctypes.CDLL(fast_path if fast else wasmref.lib_path())
        L.refbench_run2.restype = ctypes.c_double
        L.refbench_run2.argtypes = [ctypes.c_int] * 3 + [ctypes.c_float, ctypes.c_int, ctypes.c_float, ctypes.c_float] + \
            [ctypes.c_int] * 3 + [ctypes.c_void_p, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]
        chk, proc = ctypes.c_double(0), ctypes.c_double(0)
        wall_total = L.refbench_run2(threads, n_streams, CHANNELS, float(SR), 0, 0.0, 0.0, n_in_total, n_out_total, chunk,
                                     x.ctypes.data, ctypes.byref(chk), ctypes.byref(proc))
        dt = proc.value
        kind = "reference"
        how = "native pthread pool over the reference's shipped binary (oracle/_ref, WASM->C, gcc %s)" % \
            ("-O3 -ffast-math -mavx2 -mfma" if fast else "-O2 -ffp-contract=off")
    elif fast:
        return None
    else:
        from concurrent.futures import ThreadPoolExecutor

        def one(s):
            o = hdrref.CpuStretch("orc")
            o.presetDefault(CHANNELS, float(SR))
            i = done = 0
            while done < n_out_total:
                co = min(chunk, n_out_total - done)
                ci = int(round((done + co) / RATIO_OUT)) - i
                o.process(x[s][:, i:i + ci], co)
                i += ci
                done += co

        t0 = time.perf_counter()
        with ThreadPoolExecutor(max_workers=threads) as ex:
            list(ex.map(one, range(n_streams)))
        dt = time.perf_counter() - t0
        kind, how = "port", "oracle restatement (double-precision FFT) via ctypes threads"
    total = n_streams * CHANNELS * n_out_total
    return {"value": total / dt, "unit": "samples/s", "cores": threads, "per_core": total / dt / threads, "kind": kind,
            "wall_s_process_only": dt, "wall_s_with_instance_creation": wall_total,
            "sample": "%d streams x %.1f s stereo 48 kHz presetDefault 0.8x, 480-sample calls, %d threads, %.2f s inside process(); %s"
                      % (n_streams, seconds_per_stream, threads, dt, how)}


def cpu_baseline_report(n_streams_per_thread, seconds_per_stream):
    """cpu_baseline object of the JSON line: thread count = the CPUs this process may really use (affinity and cgroup
    quota, not os.cpu_count()), per-core and aggregate figures, and the -O3 -ffast-math build beside the -O2 one."""
    hc = host_cores()
    threads = hc["usable"]
    n = max(n_streams_per_thread * threads, 64)
    r = cpu_reference_run(n, seconds_per_stream, threads)
    r["host"] = hc
    f = cpu_reference_run(n, seconds_per_stream, threads, fast=True)
    if f:
        r["fast_math_build"] = {"value": f["value"], "per_core": f["per_core"], "sample": f["sample"]}
    return r


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    hc = host_cores()
    threads = hc["usable"]
    vals, t_all = [], []
    n_streams = max(threads * 2, 64)
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        r = cpu_reference_run(n_streams, 10.0, threads)  # a bounded sample of the workload per step: 10 s of audio per stream
        if i >= args.warmup:
            vals.append(r["value"])
            t_all.append(time.perf_counter() - t0)
    v = float(np.mean(vals))
    w = workload(BATCH_PER_GPU)
    r["value"] = v
    r["per_core"] = v / threads
    r["host"] = hc
    f = cpu_reference_run(n_streams, 10.0, threads, fast=True)
    if f:
        r["fast_math_build"] = {"value": f["value"], "per_core": f["per_core"], "sample": f["sample"]}
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": v, "unit": "samples/s", "n_gpus": args.gpus,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.mean(t_all)) * 1e3,
                      "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                      "config": config_dict(w, args.gpus), "cpu_baseline": r,
                      "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


# ------------------------------------------------------------------------------------ 16-bit PCM boundary probe
def pcm16_probe(args):
    """Child process of the default run (never the measured arm itself): the same workload through
    b200s_process_pcm16 -- int16 host buffers, conversions on the device, half the PCIe bytes -- streamed like `e2e`."""
    import torch

    from signalsmith_stretch_b200 import BatchStretch, build_library

    build_library()
    torch.cuda.set_device(0)
    w = workload(args.batch)
    eng = BatchStretch(args.batch, device=0)
    eng.presetDefault(CHANNELS, float(SR))
    eng.reserve(w["n_in"], w["n_out"])
    pool = synth_input(min(args.batch, 64), 3 * w["n_in"])
    x = np.tile(pool, ((args.batch + len(pool) - 1) // len(pool), 1, 1))[:args.batch]
    x16 = np.clip(np.round(x * 32768), -32768, 32767).astype(np.int16)
    xs = [torch.from_numpy(np.ascontiguousarray(x16[:, :, k * w["n_in"]:(k + 1) * w["n_in"]])).pin_memory() for k in range(3)]
    ys = [torch.empty((args.batch, CHANNELS, w["n_out"]), dtype=torch.int16).pin_memory() for _ in range(3)]
    for i in range(3):
        eng.process_pcm16_ptr(xs[i % 3].data_ptr(), w["n_in"], ys[i % 3].data_ptr(), w["n_out"], wait=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(args.steps):
        eng.process_pcm16_ptr(xs[i % 3].data_ptr(), w["n_in"], ys[i % 3].data_ptr(), w["n_out"], wait=False)
    eng.synchronize()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    print(json.dumps({"value": w["samples_per_step"] * args.steps / dt, "unit": "samples/s", "ms_per_step": dt / args.steps * 1e3,
                      "h2d_bytes_per_step": int(xs[0].numel() * 2), "d2h_bytes_per_step": int(ys[0].numel() * 2),
                      "timed": "host wall clock around %d pipelined b200s_process_pcm16() calls + synchronize (int16 host buffers, conversions on the device)" % args.steps}))


# ------------------------------------------------------------------------------------ config 5: ratio x preset sweep
SWEEP_RATIOS = [(2, 1), (3, 2), (5, 4), (1, 1), (4, 5), (2, 3), (1, 2)]  # input / output length: 0.5x ... 2.0x stretch
SWEEP_BATCH = 4096


def algo_bytes_block_channel(B, H, K, in_over_out):
    """SURVEY.md section 8(d): compulsory HBM bytes per block-channel (r = 1 when the previous block is re-analysed)."""
    h_in = H * in_over_out
    r = 1 if abs(h_in - H) > 1 else 0
    return 4 * h_in + 4 * h_in + 4 * B * (1 + r) + 16 * K + 16 * K * (1 - r) + 8 * K + 8 * B + 4 * H


def run_sweep(args):
    """BASELINE configs[4]: stretch ratio 0.5x ... 2.0x  x  {presetDefault, presetCheaper}, batch 4096 mono, one GPU.
    One JSON line per point (device-resident, CUDA events, 32 blocks per call); not the driver's default run."""
    import torch

    from signalsmith_stretch_b200 import BatchStretch, build_library

    build_library()
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak = float(json.load(open(peaks_path))["hbm_gbs"]) if os.path.exists(peaks_path) else 6650.0
    global CHANNELS
    CHANNELS = 1
    batch = args.batch if args.batch != BATCH_PER_GPU else SWEEP_BATCH
    for preset in ("presetDefault", "presetCheaper"):
        for num, den in SWEEP_RATIOS:
            if args.sweep_filter and args.sweep_filter not in "%s:%d/%d" % (preset, num, den):
                continue
            eng = BatchStretch(batch, device=0)
            getattr(eng, preset)(1, float(SR))
            B, H, K = eng.blockSamples(), eng.intervalSamples(), eng.bands()
            n_out = BLOCKS_PER_STEP * H
            n_in = n_out * num // den
            assert n_in * den == n_out * num
            eng.reserve(n_in, n_out)
            pool = synth_input(64, 3 * n_in)
            x = np.tile(pool, ((batch + 63) // 64, 1, 1))[:batch]
            xd = [torch.from_numpy(np.ascontiguousarray(x[:, :, k * n_in:(k + 1) * n_in])).to(dev) for k in range(3)]
            yd = torch.empty((batch, 1, n_out), dtype=torch.float32, device=dev)
            for i in range(max(args.warmup, 3)):
                eng.process(xd[i % 3], n_out, out=yd)
            eng.synchronize()
            eng.timer_start()
            for i in range(args.steps):
                eng.process(xd[i % 3], n_out, out=yd)
            ms = eng.timer_stop() / args.steps
            eng.profile_begin()
            for i in range(2):
                eng.process(xd[i % 3], n_out, out=yd)
            prof = eng.profile_end()
            kern = {k: v[0] / max(v[1], 1) for k, v in prof.items()}
            unserved = eng.unserved_random_blocks()
            algo = algo_bytes_block_channel(B, H, K, num / den)
            achieved = algo * batch * BLOCKS_PER_STEP / (ms * 1e-3) / 1e9
            print(json.dumps({
                "metric": METRIC, "value": batch * n_out / (ms * 1e-3), "unit": "samples/s", "n_gpus": 1, "steps": args.steps,
                "ms_per_step": ms, "dtype": "f32", "data": "synthetic",
                "config": {"workload": "BASELINE configs[4] sweep point: batch=%d mono 48 kHz %s, input/output = %d/%d (%.3gx stretch)"
                                       % (batch, preset, num, den, den / num),
                           "preset": preset, "in_over_out": num / den, "block": B, "interval": H, "bands": K, "blocks_per_step": BLOCKS_PER_STEP},
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "algo_bytes_per_block_channel": algo, "algo_bytes_per_output_sample": algo / H, "kernel_ms_per_step": kern},
                "unserved_random_blocks": unserved}), flush=True)
            del eng, xd, yd
            torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------ live / streaming caller
def run_live(args):
    """SURVEY.md 8(f) rank 4: the reference's live wrapper (web/web-wrapper.js:215-332: seek + process(0, 128) per audio
    quantum) as a batched server loop (signalsmith_stretch_b200/live.py), batch 1024 stereo, every stream its own rate.
    Host wall clock: the loop includes the per-quantum window gathering on the host, like the worklet's."""
    import torch

    from signalsmith_stretch_b200 import BatchStretch, build_library
    from signalsmith_stretch_b200.live import LiveBatch

    build_library()
    torch.cuda.set_device(0)
    batch, quantum = args.batch, 128
    eng = BatchStretch(batch, device=0)
    eng.presetDefault(CHANNELS, float(SR))
    live = LiveBatch(eng, float(SR))
    pool = synth_input(64, 4 * SR)
    for s in range(batch):
        live.add_buffers(s, pool[s % 64])
        live.start(s, when=0.0, offset=0.05 * (s % 7), rate=0.6 + 0.1 * (s % 9))
    for _ in range(20):
        live.process(quantum)
    eng.synchronize()
    n = max(args.steps, 10) * 20
    t0 = time.perf_counter()
    t_gpu = 0.0
    for _ in range(n):
        live.process(quantum)
    eng.synchronize()
    dt = time.perf_counter() - t0
    print(json.dumps({"metric": "live quanta/s (seek + process(0, 128) per quantum for every stream)", "value": n / dt, "unit": "quanta/s",
                      "streams": batch, "channels": CHANNELS, "quantum": quantum, "stream_quanta_per_s": n * batch / dt,
                      "realtime_streams_sustained": n * batch / dt / (SR / quantum),
                      "output_samples_per_s_per_channel": n * batch * CHANNELS * quantum / dt, "ms_per_quantum": dt / n * 1e3,
                      "timed": "host wall clock over %d quanta incl. the host-side window gathering, H2D of the seek windows and D2H of the output" % n}))


# ------------------------------------------------------------------------------------ GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH_PER_GPU, help="streams per GPU (default: the BASELINE config)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs (ncu): device-resident steps only; the JSON line then has no e2e / per-kernel split")
    ap.add_argument("--sub-batches", type=int, default=0, help="device-resident path: split the batch over N prioritised CUDA streams (experiment)")
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5], help="BASELINE config (default 2 = the headline; 5 = the ratio x preset sweep, one line per point)")
    ap.add_argument("--pcm16-probe", action="store_true", help="internal: child process measuring the 16-bit PCM boundary")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the child runs of BASELINE configs[2] / [3]")
    ap.add_argument("--sweep-filter", default="", help="config 5: only the points whose 'preset:num/den' contains this string (e.g. presetDefault:5/4)")
    ap.add_argument("--live", action="store_true", help="the live / streaming caller (seek + process(0, 128) per quantum), batch 1024 stereo")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the last timed step's output of the device-resident path to DIR/output.npy (float32, %d sampled streams)" % DUMP_STREAMS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.live or args.config == 5 or args.impl == "reference"):
        ap.error("--dump-outputs applies to the device-resident path of --config 2, 3 or 4")
    if args.pcm16_probe:
        pcm16_probe(args)
        return
    if args.live:
        run_live(args)
        return
    if args.config == 5:
        run_sweep(args)
        return
    if args.config != 2:
        global CHANNELS, RATIO_OUT, ALGO_BYTES_PER_BLOCK_CHANNEL
        CHANNELS, RATIO_OUT, ALGO_BYTES_PER_BLOCK_CHANNEL = EXTRA[args.config]["channels"], 1.0, EXTRA[args.config]["algo"]
        args.no_cpu_baseline = True
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist

    from signalsmith_stretch_b200 import BatchStretch, build_library
    from signalsmith_stretch_b200.shard import reduce_throughput, shard_range

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 arm has no CPU path (use --impl reference for the CPU baseline)")
    build_library()
    orig_affinity = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa(local_rank)  # before the pinned host buffers are allocated (first touch)
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)

    w = workload(args.batch)
    lo, _hi = shard_range(args.batch * world, rank, world)  # this rank's streams of the global batch
    eng = BatchStretch(args.batch, device=local_rank)
    eng.presetDefault(CHANNELS, float(SR))
    if args.config != 2:
        eng.setTransposeSemitones(EXTRA[args.config]["semitones"], EXTRA[args.config]["tonality"])
        if EXTRA[args.config]["formant"]:
            eng.setFormantFactor(1.0, True)
            eng.setFormantBase(200.0 / SR)
    eng.reserve(w["n_in"], w["n_out"])
    if args.sub_batches > 1:
        eng.set_sub_batches(args.sub_batches)

    # three distinct input buffers (each >> L2), consecutive seconds of each stream's audio
    x_host = synth_input(args.batch, 3 * w["n_in"], seed0=lo)
    x_dev = [torch.from_numpy(np.ascontiguousarray(x_host[:, :, k * w["n_in"]:(k + 1) * w["n_in"]])).to(dev) for k in range(3)]
    y_dev = torch.empty((args.batch, CHANNELS, w["n_out"]), dtype=torch.float32, device=dev)
    x_pin = [torch.from_numpy(np.ascontiguousarray(x_host[:, :, k * w["n_in"]:(k + 1) * w["n_in"]])).pin_memory() for k in range(3)]
    y_pin = torch.empty((args.batch, CHANNELS, w["n_out"]), dtype=torch.float32).pin_memory()
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident: warm-up, then exactly K timed steps
    for i in range(args.warmup):
        eng.process(x_dev[i % 3], w["n_out"], out=y_dev)
    eng.synchronize()
    barrier()
    clocks = ClockSampler(local_rank)
    clocks.start()
    launches0 = eng.kernel_launches()
    eng.timer_start()
    for i in range(args.steps):
        eng.process(x_dev[i % 3], w["n_out"], out=y_dev)
    ms = eng.timer_stop()
    launches = eng.kernel_launches() - launches0
    barrier()
    clk = clocks.stop()
    total, tmax = reduce_throughput(w["samples_per_step"] * args.steps, ms / 1e3, dist if world > 1 else None, dev)
    value = total / tmax
    if args.dump_outputs and rank == 0:  # y_dev still holds the last timed step; later passes overwrite it
        dump_outputs(args.dump_outputs, y_dev)

    if args.no_e2e:
        if rank == 0:
            pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
            pkv = float(json.load(open(pk))["hbm_gbs"]) if os.path.exists(pk) else 6650.0
            ach = ALGO_BYTES_PER_BLOCK_CHANNEL * args.batch * CHANNELS * BLOCKS_PER_STEP / (tmax / args.steps) / 1e9
            print(json.dumps({"metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
                              "ms_per_step": tmax / args.steps * 1e3, "gpu_launches": int(launches),
                              "roofline_frac": ach / pkv, "algo_bytes_per_block_channel": ALGO_BYTES_PER_BLOCK_CHANNEL,
                              "workload": EXTRA[args.config]["name"] if args.config in EXTRA else "BASELINE configs[1]",
                              "note": "--no-e2e run (device-resident only)"}))
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- end to end through the host-buffer C ABI: pinned host in, pinned host out, copies timed.
    # (a) e2e: the streaming form a server uses -- b200s_process_async, chunk after chunk, three buffer sets in
    #     rotation, one synchronize at the end; every byte of every step crosses PCIe inside the timed region.
    # (b) e2e_sync: one blocking b200s_process() per step (the reference's own call shape).
    y_pins = [y_pin] + [torch.empty_like(y_pin).pin_memory() for _ in range(2)]
    for i in range(2):
        eng.process_host_ptr(x_pin[i % 3].data_ptr(), w["n_in"], y_pin.data_ptr(), w["n_out"])
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        eng.process_host_ptr(x_pin[i % 3].data_ptr(), w["n_in"], y_pin.data_ptr(), w["n_out"])
    torch.cuda.synchronize()
    wall_sync = time.perf_counter() - t0
    barrier()
    t0 = time.perf_counter()
    eng.timer_start()
    for i in range(args.steps):
        eng.process_host_ptr_async(x_pin[i % 3].data_ptr(), w["n_in"], y_pins[i % 3].data_ptr(), w["n_out"])
    ms_e2e_dev = eng.timer_stop()
    eng.synchronize()
    torch.cuda.synchronize()
    wall_e2e = time.perf_counter() - t0
    barrier()
    tot_e, t_e = reduce_throughput(w["samples_per_step"] * args.steps, max(wall_e2e, ms_e2e_dev / 1e3), dist if world > 1 else None, dev)
    tot_s, t_s = reduce_throughput(w["samples_per_step"] * args.steps, wall_sync, dist if world > 1 else None, dev)
    e2e = {"value": tot_e / t_e, "unit": "samples/s",
           "h2d_bytes_per_step": int(x_pin[0].numel() * 4), "d2h_bytes_per_step": int(y_pin.numel() * 4),
           "ms_per_step": t_e / args.steps * 1e3,
           "h2d_gbs_per_rank": x_pin[0].numel() * 4 / (t_e / args.steps) / 1e9, "d2h_gbs_per_rank": y_pin.numel() * 4 / (t_e / args.steps) / 1e9,
           "numa": numa,
           "timed": "host wall clock around %d pipelined b200s_process_async() calls + synchronize, pinned H2D + D2H of every step inside" % args.steps,
           "sync_call": {"value": tot_s / t_s, "ms_per_step": t_s / args.steps * 1e3, "timed": "one blocking b200s_process() per step"}}

    # ---- per-kernel device time (separate pass, CUDA events around every kernel of process())
    eng.profile_begin()
    nprof = min(args.steps, 4)
    for i in range(nprof):
        eng.process(x_dev[i % 3], w["n_out"], out=y_dev)
    prof = eng.profile_end()
    kern = {k: v[0] / max(v[1], 1) for k, v in prof.items()}
    ksum = sum(kern.values())
    dominant = max(kern, key=kern.get)

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    algo_bytes_step = ALGO_BYTES_PER_BLOCK_CHANNEL * args.batch * CHANNELS * BLOCKS_PER_STEP
    ms_step_dev = ms / args.steps
    achieved = algo_bytes_step / (ms_step_dev * 1e-3) / 1e9
    # measured DRAM traffic of the three large kernels for this workload (ncu --set full, committed under profiles/);
    # only meaningful for the default configuration and batch
    traffic, kernel_dram = None, None
    tpath = os.path.join(ROOT, "profiles", "r01_traffic.json")
    if args.config == 2 and args.batch == BATCH_PER_GPU and os.path.exists(tpath):
        tj = json.load(open(tpath))
        traffic = float(tj["total_bytes_per_step"])
        # measured DRAM bytes of each large kernel / its measured duration in THIS run: how close each one is to the HBM bound
        kernel_dram = {k: {"dram_gbs": v / (kern[k] * 1e-3) / 1e9, "frac_of_peak": v / (kern[k] * 1e-3) / 1e9 / peak}
                       for k, v in tj["dram_bytes_per_launch"].items() if kern.get(k, 0) > 0}
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": "profiles/r01_traffic.json: dram read+write bytes per step of analyse+chain+synth (ncu --set full); algorithmic bytes per step: %d" % algo_bytes_step,
                "peak_source": peak_src,
                "scope": "whole process() launch sequence (the path is not yet one fused kernel): "
                         "%d algorithmic bytes per block-channel (SURVEY.md 8(d)) x %d block-channels per step / device time per step"
                         % (ALGO_BYTES_PER_BLOCK_CHANNEL, args.batch * CHANNELS * BLOCKS_PER_STEP),
                "kernel_ms_per_step": kern, "kernel_dram": kernel_dram, "kernel_share": {k: v / ksum for k, v in kern.items()}, "dominant_kernel": dominant}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        os.sched_setaffinity(0, orig_affinity)  # the CPU baseline uses every CPU of the lease, not only the GPU-local ones
        cpu = cpu_baseline_report(2, 10.0)

    # the 16-bit PCM boundary (not the reference's float call: reported beside `e2e`, never instead of it), measured in a
    # child process so that nothing it does can take the line above with it
    e2e_pcm16 = None
    if rank == 0 and world == 1 and args.config == 2:
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--pcm16-probe", "--steps", str(args.steps), "--batch", str(args.batch)],
                               capture_output=True, text=True, timeout=240)
            e2e_pcm16 = json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 else {"unavailable": (r.stderr or "failed")[-200:]}
        except Exception as ex:  # noqa: BLE001
            e2e_pcm16 = {"unavailable": str(ex)[-200:]}

    # BASELINE configs[2] / [3] (frequency map; formants) on this GPU, device-resident, in child processes: reported beside
    # the headline (never instead of it) so that the driver's record carries them too
    other_configs = None
    if rank == 0 and world == 1 and args.config == 2 and not args.no_other_configs:
        other_configs = {}
        for c in (3, 4):
            try:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--config", str(c), "--steps", str(args.steps), "--no-e2e"],
                                   capture_output=True, text=True, timeout=240)
                other_configs["config%d" % c] = json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 else {"unavailable": (r.stderr or "failed")[-200:]}
            except Exception as ex:  # noqa: BLE001
                other_configs["config%d" % c] = {"unavailable": str(ex)[-200:]}

    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": tmax / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": dict(config_dict(w, world), **({} if args.config == 2 else {"workload": EXTRA[args.config]["name"]})), "clocks": clk,
            "e2e": e2e, "e2e_pcm16": e2e_pcm16, "other_configs": other_configs, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
