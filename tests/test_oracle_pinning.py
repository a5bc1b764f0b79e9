"""Pins the oracle (oracle/stretch_oracle.cpp) to the reference: golden vectors and digests generated
from the reference's own binary / header (tests/golden/make_golden.py).  CPU only."""
import os

import numpy as np
import pytest

import signals

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def rms(a):
    return float(np.sqrt(np.mean(np.square(a, dtype=np.float64))))


@pytest.mark.parametrize("name", list(signals.CONFIGS))
def test_oracle_matches_reference_header_golden(oracle_port, name):
    """Reference header (unmodified) on the stand-in STFT: the oracle is bit-exact against it."""
    g = np.load(os.path.join(GOLD, name + ".npz"))
    o = oracle_port()
    signals.CONFIGS[name][0](o)
    y = signals.run_single(o, g["x"], float(g["ratio"]), int(g["chunk"]))
    assert y.shape == g["hdr"].shape
    # same libm / compiler on the GPU box image; allow 1e-6 in case sinf/cosf differ by an ulp
    assert np.abs(y - g["hdr"]).max() <= 1e-6


@pytest.mark.parametrize("name", [n for n in signals.CONFIGS if "formant" not in n])
def test_oracle_matches_reference_binary_golden(oracle_port, name):
    """The reference's shipped WASM binary (-O3 -ffast-math, float FFT): agreement to float
    precision over the short horizon; the identity config at any length (SURVEY.md 8(c))."""
    g = np.load(os.path.join(GOLD, name + ".npz"))
    o = oracle_port()
    cfg, C, sr, ratio, _ = signals.CONFIGS[name]
    cfg(o)
    y = signals.run_single(o, g["x"], float(g["ratio"]), int(g["chunk"]))
    H = o.intervalSamples()
    lat = o.outputLatency() + int(o.inputLatency() * ratio)
    d = y - g["wasm"]
    if name == "identity":
        assert rms(d) <= 1e-6
    else:
        first = d[:, : lat + 8 * H]
        assert rms(first) <= 1e-4, "short-horizon disagreement with the reference binary"
        assert rms(d) <= 1e-3  # the reference's own regression criterion (-60 dB, cmd/main-dev.cpp:215-232)


def test_kats(oracle_port):
    k = np.load(os.path.join(GOLD, "kats.npz"))
    o = oracle_port()
    o.presetDefault(1, 48000.0)
    win = o.state("window")
    assert np.abs(win[[0, 1440, 2879, 2880, 5759]] - k["window_48k_default_wasm"]).max() < 5e-6
    assert int(win.argmax()) == int(k["window_argmax"][0]) == 2879
    assert abs(win[0] - 0.015485264) < 5e-6 and abs(win[2880] - 0.8161286) < 5e-6  # SURVEY 8(c) item 2
    wp = o.state("windowProducts")  # pending order: index i <-> ring position i + interval
    ref = k["wp_after_configure_wasm"]  # ring positions [0, 1439, 1440, 2880, 5759]
    assert abs(wp[0] - ref[2]) / ref[2] < 1e-5 and abs(wp[1440] - ref[3]) / ref[3] < 1e-5
    assert abs(wp[5759 - 1440] - ref[4]) / ref[4] < 1e-5
    assert ref[0] == np.float32(1e-30) and wp[5759] == np.float32(1e-30)
    presets = [("presetDefault", 44100.0), ("presetDefault", 48000.0), ("presetCheaper", 44100.0), ("presetCheaper", 48000.0),
               ("presetDefault", 96000.0), ("presetDefault", 16000.0)]
    for (preset, sr), row in zip(presets, k["latency_table_wasm"]):
        o = oracle_port()
        getattr(o, preset)(1, sr)
        assert [o.blockSamples(), o.intervalSamples(), o.inputLatency(), o.outputLatency()] == list(row)


def test_seek_process_flush_sequence(oracle_port):
    k = np.load(os.path.join(GOLD, "kats.npz"))
    x = k["seek_process_flush_x"]
    o = oracle_port()
    o.presetDefault(1, 48000.0)
    o.setTransposeSemitones(3, 0)
    o.seek(x[:, :2880], 1.0)
    y = np.concatenate([o.process(x[:, 2880:2880 + 7200], 7200), o.flush(1440, 1.0)], axis=1)
    assert np.abs(y - k["seek_process_flush_hdr"]).max() <= 1e-6
    assert rms(y - k["seek_process_flush_wasm"]) <= 1e-4


def test_identity_is_a_pure_delay(oracle_port):
    o = oracle_port()
    o.presetDefault(1, 48000.0)
    x = signals.harmonic(3 * 5760, 48000)[None]
    y = signals.run_single(o, x, 1.0, 1000)
    lat = o.inputLatency() + o.outputLatency()
    assert rms(y[:, lat:] - x[:, :-lat]) <= 1e-6
    assert np.abs(y[:, :lat]).max() <= 1e-6


def test_chunk_size_invariance(oracle_port):
    x = signals.harmonic(20000, 48000)[None]
    ys = []
    for chunk in (64, 480, 5000):
        o = oracle_port()
        signals.cfg_config3(o)
        ys.append(signals.run_single(o, x, 1.0, chunk))
    assert np.array_equal(ys[0], ys[1]) and np.array_equal(ys[0], ys[2])


# ---- bit-exact checks against the reference header's outputs, stored as digests (tests/golden/make_golden.py) ----
def _assert_matches_record(y, g, key):
    assert list(y.shape) == list(g[key + "_shape"]), (key, y.shape)
    idx = signals.sample_positions(y.size, g[key + "_sample"].size)
    d = np.abs(y.reshape(-1)[idx] - g[key + "_sample"]).max()
    assert np.array_equal(signals.digest(y), g[key + "_sha256"]), "%s differs from the reference header: max diff %g on %d sampled positions" % (key, d, idx.size)


def test_live_oracle_bit_exact_vs_reference_header(oracle_port):
    g = np.load(os.path.join(GOLD, "reference_header_cases.npz"))
    x = signals.header_case_input()
    for i, (cfg, ratio, chunk) in enumerate(signals.HEADER_CASES):
        o = oracle_port()
        cfg(o)
        _assert_matches_record(signals.run_single(o, x, ratio, chunk), g, "case%d" % i)


def test_live_api_sequence_vs_reference_header(oracle_port):
    g = np.load(os.path.join(GOLD, "reference_header_cases.npz"))
    _assert_matches_record(signals.header_api_sequence(oracle_port()), g, "api_sequence")
