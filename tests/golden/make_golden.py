#!/usr/bin/env python3
"""Generates tests/golden/*.npz from the REFERENCE (run in the build container, where
/root/reference exists and oracle/_ref has been built by `make -C oracle ref`):

  * `wasm`: the reference's own shipped binary (web/emscripten/main.js:9) translated to C
            -- authoritative for STFT + non-formant process (SURVEY.md section 0.5);
  * `hdr` : the unmodified reference header on the oracle's stand-in STFT
            -- authoritative for formants / flush / seek API sequences.

Each fixture: the first 16 blocks (+ latency) of output for one stream of a BASELINE config,
driven with 480-sample output chunks, plus the input and the KATs of SURVEY.md section 8(c).
Outputs too long to store whole are kept as a SHA-256 digest (bit-exact checks) or as an evenly
spaced sample (statistical checks): see `header_cases` and `bench_shape`.  The tests need only
these files, never the reference itself.

  python tests/golden/make_golden.py [configs] [header_cases] [bench_shape]   (default: all)
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

import signals  # noqa: E402
from oracle.hdrref import CpuStretch  # noqa: E402
from oracle.wasmref import WasmStretch  # noqa: E402


def record(out, key, y, n_sample=512):
    out[key + "_shape"] = np.array(y.shape)
    out[key + "_sha256"] = signals.digest(y)
    out[key + "_sample"] = y.reshape(-1)[signals.sample_positions(y.size, n_sample)]


def header_cases():
    """tests/test_oracle_pinning.py: the header on signals.HEADER_CASES and on the API sequence."""
    out = {}
    x = signals.header_case_input()
    for i, (cfg, ratio, chunk) in enumerate(signals.HEADER_CASES):
        h = CpuStretch("hdr")
        cfg(h)
        record(out, "case%d" % i, signals.run_single(h, x, ratio, chunk))
    record(out, "api_sequence", signals.header_api_sequence(CpuStretch("hdr")))
    np.savez_compressed(os.path.join(HERE, "reference_header_cases.npz"), **out)


def bench_shape():
    """tests/test_gpu_parity.py::test_benchmark_shape_vs_oracle: the shipped binary on stream 0 of config 2 at the
    benchmark's shape (three calls of 32 blocks), 4096 evenly spaced positions per channel."""
    cfg, C, sr, ratio, _ = signals.CONFIGS["config2_stereo_0p8x"]
    n_out = 32 * int(sr * 0.03)
    n_in = int(round(n_out / ratio))
    x = np.stack([signals.harmonic(3 * n_in, sr, 0, c) for c in range(C)])
    w = WasmStretch()
    cfg(w)
    y = signals.run_single(w, x, ratio, n_out)
    idx = signals.sample_positions(y.shape[-1], 4096)
    np.savez_compressed(os.path.join(HERE, "config2_bench_shape_wasm.npz"), x_sha256=signals.digest(x), wasm=y[:, idx])


def main():
    what = sys.argv[1:] or ["configs", "header_cases", "bench_shape"]
    if "header_cases" in what:
        header_cases()
    if "bench_shape" in what:
        bench_shape()
    if "configs" in what:
        configs()


def configs():
    for name, (cfg, C, sr, ratio, kind) in signals.CONFIGS.items():
        H = int(sr * 0.03) if "cheaper" not in name else int(sr * 0.04)
        n_out = 16 * H + 2 * int(sr * 0.12)
        n_in = int(round(n_out / ratio))
        x = signals.batch(kind, 1, C, n_in, sr)[0]
        out = {"x": x, "ratio": ratio, "chunk": 480, "sr": sr}
        h = CpuStretch("hdr")
        cfg(h)
        out["hdr"] = signals.run_single(h, x, ratio, 480)
        if "formant" not in name:
            w = WasmStretch()
            cfg(w)
            out["wasm"] = signals.run_single(w, x, ratio, 480)
            d = out["wasm"] - out["hdr"]
            print("%-22s wasm-vs-hdr rms %.2e" % (name, np.sqrt(np.mean(d ** 2))))
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    # KATs (SURVEY.md section 8(c) items 1-3)
    kat = {}
    h = CpuStretch("hdr")
    h.presetDefault(1, 48000.0)
    win = h.state("window")
    kat["window_48k_default"] = win[[0, 1440, 2879, 2880, 5759]]
    kat["window_argmax"] = np.array([int(win.argmax())])
    w = WasmStretch()
    w.presetDefault(1, 48000.0)
    p = w.mem_u32(6460)[0]
    kat["window_48k_default_wasm"] = w.mem_f32(p, 5760)[[0, 1440, 2879, 2880, 5759]]
    p = w.mem_u32(6420)[0]
    kat["wp_after_configure_wasm"] = w.mem_f32(p, 5760)[[0, 1439, 1440, 2880, 5759]]
    lat = []
    for preset, srr in (("presetDefault", 44100.0), ("presetDefault", 48000.0), ("presetCheaper", 44100.0), ("presetCheaper", 48000.0),
                        ("presetDefault", 96000.0), ("presetDefault", 16000.0)):
        w = WasmStretch()
        getattr(w, preset)(1, srr)
        lat.append([w.blockSamples(), w.intervalSamples(), w.inputLatency(), w.outputLatency()])
    kat["latency_table_wasm"] = np.array(lat)
    # seek + process + flush(<= interval) sequence (header == wasm for this path)
    x = signals.harmonic(12000, 48000)[None]
    seqs = {}
    for key, o in (("hdr", CpuStretch("hdr")), ("wasm", WasmStretch())):
        o.presetDefault(1, 48000.0)
        o.setTransposeSemitones(3, 0)
        o.seek(x[:, :2880], 1.0)
        a = o.process(x[:, 2880:2880 + 7200], 7200)
        b = o.flush(1440) if key == "wasm" else o.flush(1440, 1.0)
        seqs[key] = np.concatenate([a, b], axis=1)
    kat["seek_process_flush_x"] = x
    kat["seek_process_flush_hdr"] = seqs["hdr"]
    kat["seek_process_flush_wasm"] = seqs["wasm"]
    np.savez_compressed(os.path.join(HERE, "kats.npz"), **kat)
    print("golden vectors written to", HERE)


if __name__ == "__main__":
    main()
