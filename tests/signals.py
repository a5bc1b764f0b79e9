"""Deterministic synthetic audio used by tests, golden vectors and bench.py (SURVEY.md section 8(d))."""
import hashlib

import numpy as np


def sweep(n, sr, c=0):
    """Exponential sine sweep 100*(1+0.5c) Hz -> x80 over the duration, amplitude 0.5."""
    t = np.arange(n) / sr
    dur = max(n / sr, 1e-9)
    f0 = 100.0 * (1 + 0.5 * c)
    k = np.log(80.0) / dur
    ph = 2 * np.pi * f0 * (np.exp(k * t) - 1) / k
    return (0.5 * np.sin(ph + c)).astype(np.float32)


def harmonic(n, sr, s=0, c=0):
    """11-partial tone with vibrato + tremolo + a little noise; seed = stream index."""
    rng = np.random.default_rng(7 + s + 100 * c)
    t = np.arange(n) / sr
    f0 = 110.0 * (1 + 0.01 * (s % 97)) * (1 + 0.05 * c)
    ph = 2 * np.pi * f0 * t + 3 * np.sin(2 * np.pi * 0.7 * t)
    x = sum(np.sin((k + 1) * ph) / (k + 1) for k in range(11))
    x = x * (1 + 0.3 * np.sin(2 * np.pi * 2 * t)) * 0.2 + 0.01 * rng.standard_normal(n)
    return x.astype(np.float32)


def batch(kind, S, C, n, sr):
    gen = sweep if kind == "sweep" else harmonic
    if kind == "sweep":
        return np.stack([np.stack([sweep(n, sr, c) * (1 - 0.3 * (s % 3) / 3) for c in range(C)]) for s in range(S)])
    return np.stack([np.stack([gen(n, sr, s, c) for c in range(C)]) for s in range(S)])


def chunks(n_in, ratio_out, chunk_out):
    """(in_start, in_len, out_len) per call so that every call keeps the exact in/out ratio."""
    n_out = int(round(n_in * ratio_out))
    i = o = 0
    res = []
    while o < n_out:
        co = min(chunk_out, n_out - o)
        ci = min(int(round((o + co) / ratio_out)), n_in) - i
        res.append((i, ci, co))
        i += ci
        o += co
    return res


def run_single(obj, x, ratio_out, chunk_out):
    """Drive a one-stream object (oracle / reference drivers): x [C][n] -> [C][n_out]."""
    outs = [obj.process(x[:, i:i + ci], co) for i, ci, co in chunks(x.shape[-1], ratio_out, chunk_out)]
    return np.concatenate(outs, axis=-1)


def run_batch(obj, x, ratio_out, chunk_out):
    """Drive a BatchStretch: x [S][C][n] -> [S][C][n_out]."""
    outs = [np.array(obj.process(x[:, :, i:i + ci], co)) for i, ci, co in chunks(x.shape[-1], ratio_out, chunk_out)]
    return np.concatenate(outs, axis=-1)


# ---- compact golden records of long outputs: an exact digest plus an evenly spaced sample for diagnostics
def digest(y):
    """SHA-256 of float32 samples; -0.0 counts as 0.0, so equal digests mean np.array_equal."""
    y = np.ascontiguousarray(np.asarray(y, np.float32) + np.float32(0), "<f4")
    return np.frombuffer(hashlib.sha256(y.tobytes()).digest(), np.uint8)


def sample_positions(n, k):
    """k evenly spaced positions in [0, n)."""
    return np.unique(np.linspace(0, n - 1, min(n, k)).round().astype(np.int64))


# piecewise-linear frequency maps (setFreqMap with a tabulated function; frequencies as multiples of the sample rate)
PWL_MONOTONE = (np.array([0.0, 0.02, 0.08, 0.2, 0.5], np.float32), np.array([0.0, 0.03, 0.1, 0.21, 0.5], np.float32))
# not monotone: the band between 0.06 and 0.1 folds back below what the band under it maps to, so consecutive peaks can
# have DEcreasing output bins (updateOutputMap's segments then overwrite each other in peak order, :896-911)
PWL_FOLDING = (np.array([0.0, 0.06, 0.1, 0.25, 0.5], np.float32), np.array([0.0, 0.09, 0.07, 0.3, 0.5], np.float32))


# named configurations (BASELINE.json configs, scaled down where noted)
def cfg_identity(o):
    o.presetDefault(1, 48000.0)


def cfg_config1(o):  # mono 44.1k presetDefault, +12 st, tonality 8 kHz (cmd/main.cpp:26 default)
    o.presetDefault(1, 44100.0)
    o.setTransposeSemitones(12, 8000 / 44100)


def cfg_config2(o):  # stereo 48k presetDefault, 0.8x time-stretch
    o.presetDefault(2, 48000.0)


def cfg_config3(o):  # mono 48k +7 st with 8 kHz tonality limit
    o.presetDefault(1, 48000.0)
    o.setTransposeSemitones(7, 8000 / 48000)


def cfg_config4(o):  # stereo +12 st with formant compensation, base 200 Hz
    o.presetDefault(2, 48000.0)
    o.setTransposeSemitones(12, 0)
    o.setFormantFactor(1, True)
    o.setFormantBase(200 / 48000)


def cfg_cheaper(o):  # presetCheaper (split by default), config 5 corner
    o.presetCheaper(1, 48000.0)


CONFIGS = {
    # name: (configure fn, channels, sample rate, out/in ratio, signal kind)
    "identity": (cfg_identity, 1, 48000, 1.0, "harmonic"),
    "config1_12st_44k": (cfg_config1, 1, 44100, 1.0, "sweep"),
    "config2_stereo_0p8x": (cfg_config2, 2, 48000, 0.8, "harmonic"),
    "config3_7st_ton8k": (cfg_config3, 1, 48000, 1.0, "harmonic"),
    "config4_formant": (cfg_config4, 2, 48000, 1.0, "harmonic"),
    "config5_cheaper_2x": (cfg_cheaper, 1, 48000, 2.0, "harmonic"),
}


# the oracle against the unmodified reference header, beyond the golden configurations: (configure fn, out/in ratio,
# output chunk), all on header_case_input()
HEADER_CASES = [
    (lambda o: (o.presetDefault(2, 48000.0), o.setTransposeSemitones(-5, 0)), 1.5, 4800),
    (lambda o: (o.presetCheaper(2, 48000.0, False), o.setTransposeSemitones(4, 0.2), o.setFormantSemitones(3, False), o.setFormantBase(0)), 1.0, 480),
    (lambda o: (o.configure(2, 1000, 250, True), o.setFreqMapQuadratic(1.2, 0.5)), 0.9, 333),
    (lambda o: o.presetDefault(2, 44100.0), 2.5, 441),  # > 2x: exercises the RNG path of the header
    # setFreqMap with a piecewise-linear function: monotone, and one that folds back (non-monotone output map)
    (lambda o: (o.configure(2, 1000, 250, False), o.setFreqMapTable(*PWL_MONOTONE)), 1.0, 500),
    (lambda o: (o.presetDefault(2, 48000.0), o.setFreqMapTable(*PWL_FOLDING)), 1.25, 2880),
]


def header_case_input():
    return np.stack([harmonic(30000, 48000, 1, 0), harmonic(30000, 48000, 1, 1)])


def header_api_sequence(o):
    """seek / silence bypass / flush / reset / outputSeek / exact on a one-stream CPU object, outputs concatenated."""
    x = harmonic(60000, 48000)[None]
    o.presetDefault(1, 48000.0)
    o.setTransposeSemitones(3, 0)
    outs = []
    o.seek(x[:, :3000], 1.0)
    outs.append(o.process(x[:, 3000:7800], 4800))
    z = np.zeros((1, 30000), np.float32)
    outs += [o.process(z[:, :12000], 12000), o.process(z[:, :4000], 4000), o.process(z[:, :4000], 5000)]
    outs.append(o.process(x[:, 8000:17600], 9000))
    outs.append(o.flush(1000, 1.0))
    outs.append(o.process(x[:, 20000:24800], 4800))
    outs.append(o.flush(5000, 1.1))
    o.reset()
    outs.append(o.process(x[:, 20000:24800], 2400))
    o.outputSeek(x[:, : o.outputSeekLength(1.3)])
    outs.append(o.process(x[:, 5000:11240], 4800))
    outs.append(o.exact(x[:, :40000], 50000)[1])
    return np.concatenate(outs, axis=1)
