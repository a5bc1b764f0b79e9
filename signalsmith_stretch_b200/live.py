"""LiveBatch -- the reference's live / streaming caller (web/web-wrapper.js:215-332, its AudioWorklet processor in
buffer-playback mode) as a batched server loop over the B200 C ABI (SURVEY.md section 8(f) rank 4).

One `LiveBatch` drives S independent streams of one `BatchStretch` engine.  Every stream has what one worklet has:
  * audio appended with `add_buffers` (web-wrapper.js:163-169) and dropped with `drop_buffers` (:137-162);
  * a TIME MAP: a list of segments {output, input, rate, active, loopStart, loopEnd} edited with `schedule` / `start` /
    `stop` (:45-108, including `adjustPrevious`), looked up per audio quantum (:227-231);
  * per quantum, the segment's input position at the quantum's output time (+ latencies, loop wrap :271-279), the
    `bufferLength = inputLatency + outputLatency` samples that END there taken from the audio with zero padding on both
    sides (:282-311), and then -- exactly like the worklet, which "constantly seeks" (:313) -- `seek(window, rate)`
    followed by `process(0, quantum)` (:314-315).
The batch makes ONE seek + ONE `b200s_process(0, n)` call per quantum for all streams, each stream with its own window
and its own rate.  Two ways to hand over the windows:
  * bank mode (default on a GPU): the streams' audio lives in a DEVICE bank [S][C][capacity] (uploaded once by
    `add_buffers`); per quantum only S window positions and S rates cross PCIe and `b200s_live_seek` cuts the windows
    out of the bank inside the seek kernel.  The per-quantum position arithmetic is vectorised over the streams.
  * host mode: the windows are gathered on the host and uploaded (`b200s_seek_rates`), 47 MB per quantum at batch 1024 --
    what S separate worklets do; kept for engines without a bank (the one-stream oracle adapter of the tests).
When no stream is active the quantum is `process(zeros, n)` for the batch, as :247-253.  Difference from S separate
worklets, by construction of a batch call: in a quantum where SOME streams are active, a stopped stream is fed a silent
seek window instead of `n` zero samples appended to its history (its tail is then the synthesis ring's, up to one block
shorter).  Parameters (transpose / formants) are batch-wide, as in the C ABI.
"""
import numpy as np

__all__ = ["LiveBatch"]


def _segment():
    return dict(active=False, input=0.0, output=0.0, rate=1.0, loopStart=0.0, loopEnd=0.0)  # :17-29


class LiveBatch:
    def __init__(self, engine, sample_rate, bank="auto", capacity=0):
        """bank: "torch" (CUDA tensor), "numpy" (the emulated library's "device" memory is host memory) or None for host
        mode; "auto" (default): "torch" when the engine has b200s_live_seek and a GPU is there, else host mode."""
        self.eng, self.sr = engine, float(sample_rate)
        self.S, self.C = engine.batch, engine.channels()
        self.buffer_length = engine.inputLatency() + engine.outputLatency()  # :205-207
        self.in_lat_s = engine.inputLatency() / self.sr
        self.out_lat_s = engine.outputLatency() / self.sr
        self.time_maps = [[_segment()] for _ in range(self.S)]
        self.current_sample = 0  # currentTime * sampleRate of the audio context
        if bank == "auto":
            bank = None
            if hasattr(engine, "live_seek"):
                try:
                    import torch

                    bank = "torch" if torch.cuda.is_available() else None
                except ImportError:
                    pass
        self.bank_kind = bank
        self.audio_start = np.zeros(self.S, np.int64)  # sample index of the first stored sample (audioBuffersStart)
        self.audio_len = np.zeros(self.S, np.int64)
        if bank:
            self._cap = 0
            self._bank = None
            self._grow(max(int(capacity), 1))
        else:
            self._audio = [np.zeros((self.C, 0), np.float32) for _ in range(self.S)]
            self._win = np.zeros((self.S, self.C, self.buffer_length), np.float32)
        # the current segment of every stream as arrays (refreshed from the time map when it changes)
        z = np.zeros(self.S)
        self._in, self._out, self._rate, self._ls, self._le = z.copy(), z.copy(), z + 1.0, z.copy(), z.copy()
        self._active = np.zeros(self.S, bool)
        self._next = np.full(self.S, np.inf)  # output time at which the next segment takes over

    @property
    def current_time(self):
        return self.current_sample / self.sr

    # ---- audio storage ----
    def _grow(self, cap):
        if cap <= self._cap:
            return
        cap = max(cap, 2 * self._cap)
        if self.bank_kind == "torch":
            import torch

            new = torch.zeros((self.S, self.C, cap), dtype=torch.float32, device="cuda")
            if self._bank is not None:
                new[:, :, : self._cap] = self._bank
        else:
            new = np.zeros((self.S, self.C, cap), np.float32)
            if self._bank is not None:
                new[:, :, : self._cap] = self._bank
        self._bank, self._cap = new, cap

    def add_buffers(self, s, samples):  # :163-169
        x = np.ascontiguousarray(np.asarray(samples, np.float32).reshape(self.C, -1))
        n, at = x.shape[1], int(self.audio_len[s])
        if self.bank_kind:
            self._grow(at + n)
            if self.bank_kind == "torch":
                import torch

                self._bank[s, :, at:at + n] = torch.from_numpy(x).to(self._bank.device)
            else:
                self._bank[s, :, at:at + n] = x
        else:
            self._audio[s] = np.concatenate([self._audio[s], x], axis=1)
        self.audio_len[s] += n
        return (self.audio_start[s] + self.audio_len[s]) / self.sr

    def drop_buffers(self, s, to_seconds=None):  # :137-162 (sample-accurate instead of whole buffers)
        if to_seconds is None:
            n = int(self.audio_len[s])
            new_start = 0
        else:
            n = max(0, min(int(self.audio_len[s]), int(to_seconds * self.sr) - int(self.audio_start[s])))
            new_start = int(self.audio_start[s]) + n
        if self.bank_kind:
            keep = int(self.audio_len[s]) - n
            if keep > 0:
                self._bank[s, :, :keep] = self._bank[s, :, n:n + keep].clone() if self.bank_kind == "torch" else self._bank[s, :, n:n + keep].copy()
            self._bank[s, :, keep:int(self.audio_len[s])] = 0
        else:
            self._audio[s] = self._audio[s][:, n:]
        self.audio_len[s] -= n
        self.audio_start[s] = new_start
        return self.audio_start[s] / self.sr, (self.audio_start[s] + self.audio_len[s]) / self.sr

    # ---- remote methods of the worklet, per stream ----
    def _to_map(self, s):
        self.time_maps[s][0]["input"] = float(self._in[s])  # (the loop wrap of :275-278 edits the current segment)

    def _from_map(self, s):
        tm = self.time_maps[s]
        seg = tm[0]
        self._in[s], self._out[s], self._rate[s] = seg["input"], seg["output"], seg["rate"]
        self._ls[s], self._le[s], self._active[s] = seg["loopStart"], seg["loopEnd"], seg["active"]
        self._next[s] = tm[1]["output"] if len(tm) > 1 else np.inf

    def schedule(self, s, obj_in, adjust_previous=False):
        """Insert a time-map point for stream `s` (semantics of the worklet's `schedule`, web-wrapper.js:67-108).
        `obj_in`: any of outputTime (default: now), input, rate, active, loopStart, loopEnd.  Points at or after the new
        one are discarded; fields that are not given are inherited from the earliest discarded point (else from the last
        point of the map); a missing `input` is that point's playback extrapolated to the new time (or stands still if it
        was stopped).  adjust_previous: re-aim the preceding
        segment so that it arrives exactly at the new point (its start is first moved up to "now" if already passed)."""
        self._to_map(s)
        points = self.time_maps[s]
        t_new = float(obj_in.get("outputTime", self.current_time))
        # the map is ordered by output time.  The new point is derived from the earliest point it replaces (the worklet pops
        # from the end and keeps the last one popped), or from the last point of the map if it replaces none
        keep = [pt for pt in points if pt["output"] < t_new]
        replaced = [pt for pt in points if pt["output"] >= t_new]
        parent = replaced[0] if replaced else keep[-1]
        fresh = dict(parent)
        fresh["output"] = t_new
        given = {k: v for k, v in obj_in.items() if k != "outputTime"}
        fresh.update(given)
        if given.get("input") is None:
            speed = parent["rate"] if parent["active"] else 0.0
            fresh["input"] = parent["input"] + (fresh["output"] - parent["output"]) * speed  # (`output` may have been given explicitly: stop(when))
        points[:] = keep + [fresh]
        if adjust_previous and len(points) >= 2:
            before = points[-2]
            now = self.current_time
            if before["output"] < now:  # already playing: its remaining part starts now, from where it has got to
                before["input"] += (now - before["output"]) * (before["rate"] if before["active"] else 0.0)
                before["output"] = now
            span = fresh["output"] - before["output"]
            if span != 0:  # (a zero-length segment is never looked up; JavaScript would store Infinity there)
                before["rate"] = (fresh["input"] - before["input"]) / span
        # points that have been superseded by a later one at or before t_new are history
        while len(points) > 1 and points[1]["output"] <= t_new:
            del points[0]
        self._from_map(s)
        return fresh

    def start(self, s, when=None, offset=0.0, duration=None, rate=1.0):  # :49-66
        obj = dict(active=True, input=offset, output=self.current_time + self.out_lat_s if when is None else when, rate=rate)
        res = self.schedule(s, obj)
        if duration is not None:
            self.stop(s, obj["output"] + duration)
        return res

    def stop(self, s, when=None):  # :45-48
        return self.schedule(s, dict(active=False, output=self.current_time if when is None else when))

    # ---- one audio quantum for every stream (:215-332) ----
    def process(self, n_out=128):
        """Render the next quantum: returns [S][C][n_out]."""
        output_time = self.current_time + self.out_lat_s  # :226
        for s in np.nonzero(self._next <= output_time)[0]:  # streams whose next segment takes over now (:227-230)
            tm = self.time_maps[s]
            while len(tm) > 1 and tm[1]["output"] <= output_time:
                tm.pop(0)
            self._from_map(s)
        if not self._active.any():  # :247-253 for the whole batch
            y = self.eng.process(np.zeros((self.S, self.C, n_out), np.float32), n_out)
        else:
            # :271-281, all streams at once: input position of the quantum, loop wrap, window end in samples
            input_time = self._in + (output_time - self._out) * self._rate
            loop = self._le - self._ls
            wrap = self._active & (loop > 0) & (input_time >= self._le)
            self._in = np.where(wrap, self._in - loop, self._in)
            input_time = np.where(wrap, input_time - loop, input_time) + self.in_lat_s
            ends = np.floor(input_time * self.sr + 0.5).astype(np.int64)  # Math.round
            rates = np.where(self._active, self._rate, 1.0)
            if self.bank_kind:
                # window = bank[end - bufferLength, end) with zeros outside the stored audio; a stopped stream gets a window
                # that lies entirely before its audio
                rel = np.where(self._active, ends - self.audio_start, -1)
                ptr = self._bank.data_ptr() if self.bank_kind == "torch" else self._bank.ctypes.data
                self.eng.live_seek(ptr, self._cap, rel, self.buffer_length, rates)
            else:
                for s in range(self.S):
                    self._win[s] = 0
                    if self._active[s]:
                        lo, hi = int(ends[s]) - self.buffer_length, int(ends[s])
                        a0, a1 = int(self.audio_start[s]), int(self.audio_start[s] + self.audio_len[s])
                        c0, c1 = max(lo, a0), min(hi, a1)
                        if c1 > c0:
                            self._win[s][:, c0 - lo:c1 - lo] = self._audio[s][:, c0 - a0:c1 - a0]
                self.eng.seek(self._win, rates)                                    # :314
            y = self.eng.process(np.zeros((self.S, self.C, 0), np.float32), n_out)  # :315
        self.current_sample += n_out
        return np.array(y)
