"""One pass of the feature hot path over a batch of 6 s analysis windows with
every buffer preallocated: the unit BASELINE.json's metric counts.

Per window (reference flow, training.py:265-449 restricted to the hot path):
    K1  STFT magnitude of the window audio          (util_audio.py:127-148)
    K2  constant-Q magnitudes of the window audio   (util_audio.py:424-429)
    K1  STFT magnitude of the rendered guessed note (util_audio.py:237)
    K3  align / scale / subtract / ReLU, then dB    (util_audio.py:238-259, :179)
        The guess is scaled by the WINDOW's own maximum: `section` (training.py:284) runs before anything has
        evaluated the song's `ref_mag` (first use: training.py:336), so the window's `_ref_mag` is None and its first
        `subtract` takes `max(window mag)` over the window's 516 columns (K3 reduces K1's per-frame maxima).

The window is the first `n_frames` STFT columns of its clip, which is what
`section(..., duration_in_frames=timing_frames)` (training.py:284) keeps.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib, ops
from .util_audio import note_to_hz


def seconds_to_frames(time, n_frames, sr, wf_len):
    """util_audio.py:264, same float64 operation order."""
    return int(np.floor(time * n_frames * sr / wf_len))


class WindowFeaturePipeline:
    def __init__(self, n_windows, window_samples=264600, guess_samples=65024, sr=44100,
                 n_fft=2048, hop=512, cqt_lowest="C1", cqt_bins=84, cqt_bpo=12, n_frames=None,
                 device=None, cqt_impl=0):
        self.dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.dev.index is None:
            self.dev = torch.device("cuda", torch.cuda.current_device())
        self.W, self.ns, self.ng, self.sr = n_windows, window_samples, guess_samples, sr
        self.stft = ops.get_stft_plan(n_fft, hop, True, device=self.dev)
        self.cqt = ops.get_cqt_plan(sr, hop, note_to_hz(cqt_lowest), cqt_bins, cqt_bpo, 2, device=self.dev)
        self.cqt_impl = cqt_impl
        self.nb = self.stft.n_bins
        self.P = ops.frame_pitch(self.nb)
        self.T_clip = self.stft.num_frames(window_samples)          # 517 for 6 s @ 2048/512
        self.T = n_frames if n_frames is not None else int(window_samples // hop)   # 516 = int(6*sr/hop)
        if self.T > self.T_clip:
            raise ValueError("window frames exceed the clip's STFT columns")
        self.Tg = self.stft.num_frames(guess_samples)
        self.Tc = self.cqt.num_frames(window_samples)
        self.Pc = ops.frame_pitch(cqt_bins)
        d, f32 = self.dev, torch.float32
        W = n_windows
        self.mag = torch.empty((W, self.T_clip, self.P), device=d, dtype=f32)
        # zeros: the dB pass writes the window's T rows only, and rows [T, T_clip) must not hold stale device memory
        self.D = torch.zeros((W, self.T_clip, self.P), device=d, dtype=f32)
        self.frame_max = torch.empty((W, self.T_clip), device=d, dtype=f32)
        self.clip_max = torch.empty((W,), device=d, dtype=f32)
        self.gmag = torch.empty((W, 1, self.Tg, self.P), device=d, dtype=f32)
        self.gmax = torch.empty((W,), device=d, dtype=f32)
        self.C = torch.empty((W, self.Tc, self.Pc), device=d, dtype=f32)
        self.ref = torch.empty((W,), device=d, dtype=f32)
        self.offs_w = torch.arange(W, device=d, dtype=torch.int64) * window_samples
        self.lens_w = torch.full((W,), window_samples, device=d, dtype=torch.int64)
        self.offs_g = torch.arange(W, device=d, dtype=torch.int64) * guess_samples
        self.lens_g = torch.full((W,), guess_samples, device=d, dtype=torch.int64)
        lib = _lib.lib()
        nbytes = lib.saga_cqt_workspace_bytes(self.cqt.handle, W, window_samples)
        self.ws = torch.empty(((nbytes + 255) // 256) * 256, device=d, dtype=torch.uint8)
        self._lib = lib
        # host side of the e2e path (pinned), allocated on demand
        self._host = None
        self._streams = None
        self._cqt_stream = None
        # "serial": one stream, kernel after kernel (default: fastest, 2.99 ms per bench step);
        # "chains": the CQT chain forked onto a second stream (3.12 ms); "db_with_contraction": the contraction
        # held back to run beside the dB pass (3.13 ms) -- profiles/microbench/schedule_variants_b200.txt.
        # Every kernel of the step fills the GPU by itself, and the pairs that could share an SM (tensor-core
        # contraction + dB pass) take as long together as one after the other (db_umma_overlap_b200.txt).
        self.schedule = "serial"

    # algorithmic work per window (DESIGN.md / SURVEY.md section 8d)
    def stft_bytes_per_window(self):
        return 4 * (self.ns + self.T_clip * self.nb) + 4 * (self.ng + self.Tg * self.nb)

    def subtract_bytes_per_window(self):
        return 4 * self.nb * (2 * self.T + self.Tg)          # read mag + read guess + write one output

    def cqt_flops_per_window(self):
        return self.Tc * sum(8 * o["n_filters"] * (o["n_fft"] // 2 + 1) for o in self.cqt.octaves)

    def run(self, *args, **kwargs):
        """See `_run`; executed with the pipeline's device current (plans, buffers and streams live there)."""
        with torch.cuda.device(self.dev):
            return self._run(*args, **kwargs)

    def run_host(self, *args, **kwargs):
        with torch.cuda.device(self.dev):
            return self._run_host(*args, **kwargs)

    def _run(self, wav, guess_wav, offset_frames, events=None, w0=0, w1=None, overlap=True, parts=("stft", "cqt")):
        """wav [W, window_samples], guess_wav [W, guess_samples] CUDA float32 contiguous,
        offset_frames [W,1] int32 CUDA.  Results land in self.mag (subtracted,
        in place), self.D, self.C, self.ref.  `events`: optional list that
        receives (stage, start_event, end_event) on the current stream (stages then run
        one after the other).  `w0:w1` restricts the pass to that window range (chunked use).

        The path is two independent chains -- STFT(window) -> STFT(guess) -> subtract/dB, and
        decimation cascade -> CQT contraction -- that only share the read-only audio.  `self.schedule`
        picks how they are enqueued: "serial" (default) on the caller's stream one after the other;
        "chains" / "db_with_contraction" fork the CQT chain onto a second stream (needs `overlap`
        and no per-stage timing) and join it at the end.  Measured on B200 the forked schedules are
        4 % slower: each kernel saturates the SMs' registers or shared memory on its own, so the block
        scheduler time-slices whole SMs and the interleaving only adds tail effects and L2 thrash."""
        w1 = self.W if w1 is None else w1
        p = lambda t: C.c_void_p(t[w0:].data_ptr())
        q = lambda t: C.c_void_p(t.data_ptr())
        main = torch.cuda.current_stream(self.dev)
        st = C.c_void_p(main.cuda_stream)
        lib, W = self._lib, w1 - w0
        fork = overlap and events is None and self.schedule != "serial"
        if fork:
            if self._cqt_stream is None:
                self._cqt_stream = torch.cuda.Stream(device=self.dev)
            side = self._cqt_stream
            ev = torch.cuda.Event()
            ev.record(main)
            side.wait_event(ev)
            st_cqt = C.c_void_p(side.cuda_stream)
        else:
            st_cqt = st

        def stage(name, fn):
            if events is None:
                return fn()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            events.append((name, a, b))

        if "stft" in parts:
            stage("stft", lambda: _lib.check(lib.saga_stft_exec(
                self.stft.handle, p(wav), q(self.offs_w), q(self.lens_w), W, self.ns, p(self.mag), None, None,
                self.P, self.T_clip * self.P, p(self.frame_max), p(self.clip_max), st)))
        def cqt(flags):
            _lib.check(lib.saga_cqt_exec(
                self.cqt.handle, p(wav), q(self.offs_w), None, W, self.ns, p(self.C), None,
                self.Pc, self.Tc * self.Pc, q(self.ws), self.ws.numel(), self.cqt_impl | flags, st_cqt))
        def guess_stft():
            _lib.check(lib.saga_stft_exec(
                self.stft.handle, p(guess_wav), q(self.offs_g), q(self.lens_g), W, self.ng, p(self.gmag), None,
                None, self.P, self.Tg * self.P, None, p(self.gmax), st))

        def subtract(phase):
            _lib.check(lib.saga_subtract_db_exec(
                p(self.mag), None, self.T_clip * self.P, p(self.gmag), None, self.Tg * self.P, None, self.Tg,
                p(offset_frames), None, p(self.gmax), None, p(self.frame_max), self.T_clip,
                _lib.SUB_NORMALIZE | _lib.SUB_RELU | phase, p(self.D), p(self.ref), W, 1, self.nb, self.T, self.P,
                1e-5, 80.0, st))

        if events is not None:       # timed separately: decimation cascade, then the kernel-bank contraction
            stage("cqt_cascade", lambda: cqt(0x100))
            stage("cqt_contract", lambda: cqt(0x200))
            stage("stft_guess", guess_stft)
            stage("subtract_db", lambda: subtract(0))
        elif fork and self.schedule == "db_with_contraction":
            # cascade beside the two STFTs and the chain; then the tensor-core contraction (one 208 KB CTA per SM,
            # 17 % of the DRAM bandwidth) beside the HBM-bound dB pass (no shared memory, 30 registers): the only
            # two kernels of the step that fit on an SM together
            cqt(0x100)
            guess_stft()
            subtract(_lib.SUB_SKIP_DB)
            ev2 = torch.cuda.Event()
            ev2.record(main)
            side.wait_event(ev2)
            cqt(0x200)
            subtract(_lib.SUB_ONLY_DB)
        else:
            if "cqt" in parts:
                cqt(0)          # on the side stream when forked (st_cqt)
            if "stft" in parts:
                guess_stft()
                subtract(0)
        if fork:
            ev = torch.cuda.Event()
            ev.record(side)
            main.wait_event(ev)

    # ---- end-to-end: host buffers in, host results out -----------------------------
    def host_buffers(self):
        if self._host is None:
            pin = dict(pin_memory=True)
            self._host = dict(
                wav=torch.empty((self.W, self.ns), dtype=torch.float32, **pin),
                guess=torch.empty((self.W, self.ng), dtype=torch.float32, **pin),
                offs=torch.empty((self.W, 1), dtype=torch.int32, **pin),
                C=torch.empty((self.W, self.Tc, self.Pc), dtype=torch.float32, **pin),
                ref=torch.empty((self.W,), dtype=torch.float32, **pin),
                d_wav=torch.empty((self.W, self.ns), device=self.dev, dtype=torch.float32),
                d_guess=torch.empty((self.W, self.ng), device=self.dev, dtype=torch.float32),
                d_offs=torch.empty((self.W, 1), device=self.dev, dtype=torch.int32))
        return self._host

    def host_pcm_buffers(self):
        """Extra buffers of the PCM-ingest variant of the e2e path: the windows and the rendered guesses
        as int16 PCM plus the float64 factor of util_audio.py:781 per clip (pinned host + device).
        `wav_div` [W] float64: the divisor of each WINDOW.  The reference divides a render by the peak of the whole
        song before it is cut into windows (util_audio.py:781, then :784 / `section`), so a window's divisor is its
        song's max|pcm|, which the caller knows and the window alone does not: fill it in.  Entries <= 0 (the default)
        fall back to the window's own peak, found on the device -- right only for clips that ARE whole renders, like
        the single-note guesses, which always use their own peak."""
        h = self.host_buffers()
        if "wav_pcm" not in h:
            pin, d = dict(pin_memory=True), self.dev
            h.update(
                wav_pcm=torch.empty((self.W, self.ns), dtype=torch.int16, **pin),
                guess_pcm=torch.empty((self.W, self.ng), dtype=torch.int16, **pin),
                mul=torch.ones((2, self.W), dtype=torch.float64, **pin),
                wav_div=torch.zeros((self.W,), dtype=torch.float64, **pin),
                d_wav_div=torch.empty((self.W,), device=d, dtype=torch.float64),
                d_wav_pcm=torch.empty((self.W, self.ns), device=d, dtype=torch.int16),
                d_guess_pcm=torch.empty((self.W, self.ng), device=d, dtype=torch.int16),
                d_mul=torch.empty((2, self.W), device=d, dtype=torch.float64),
                d_peak=torch.empty((2, self.W), device=d, dtype=torch.int32))
        return h

    def _run_host(self, chunks=6, pcm16=False, returns="cqt"):
        """Pinned host inputs -> device -> hot path -> features back on the host
        (CQT magnitudes + post-subtraction ref_mag; the subtracted window and its dB
        image stay resident for the next loop iteration, as in training.py:449).

        The batch is cut into `chunks` window ranges; H2D copies, kernels and D2H
        copies run on three streams so PCIe transfers overlap the compute (the
        path is PCIe-bound: 1.3 MB of audio in per window).

        `pcm16`: the host holds the audio as 16-bit PCM (what fluidsynth and the audio files deliver,
        util_audio.py:894 / :964) plus the per-clip float64 factor; K0 rebuilds the reference's float
        waveform `pcm * mul / max|pcm|` (util_audio.py:781) on the device, which halves the PCIe bytes."""
        h = self.host_pcm_buffers() if pcm16 else self.host_buffers()
        feats = returns == "features"
        if feats:
            self.feature_buffers()
        elif returns != "cqt":
            raise ValueError("returns must be 'cqt' or 'features'")
        if self._streams is None:
            self._streams = [torch.cuda.Stream(device=self.dev) for _ in range(3)]
            self._last_compute = None
        s_in, s_cmp, s_out = self._streams
        cur = torch.cuda.current_stream(self.dev)
        start = torch.cuda.Event()
        start.record(cur)
        s_in.wait_event(start)
        s_cmp.wait_event(start)
        s_out.wait_event(start)
        n = max(1, min(chunks, self.W))
        bounds = [(i * self.W // n, (i + 1) * self.W // n) for i in range(n)]
        song_div = pcm16 and bool((h["wav_div"] > 0).all())
        ev_in, ev_cmp = [], []
        with torch.cuda.stream(s_in):
            if pcm16:
                h["d_mul"].copy_(h["mul"], non_blocking=True)
                h["d_wav_div"].copy_(h["wav_div"], non_blocking=True)
            for a, b in bounds:
                if pcm16:
                    h["d_wav_pcm"][a:b].copy_(h["wav_pcm"][a:b], non_blocking=True)
                    h["d_guess_pcm"][a:b].copy_(h["guess_pcm"][a:b], non_blocking=True)
                else:
                    h["d_wav"][a:b].copy_(h["wav"][a:b], non_blocking=True)
                    h["d_guess"][a:b].copy_(h["guess"][a:b], non_blocking=True)
                h["d_offs"][a:b].copy_(h["offs"][a:b], non_blocking=True)
                e = torch.cuda.Event()
                e.record(s_in)
                ev_in.append(e)
        with torch.cuda.stream(s_cmp):
            for (a, b), e in zip(bounds, ev_in):
                s_cmp.wait_event(e)
                if pcm16:
                    for k, (src, dst) in enumerate((("d_wav_pcm", "d_wav"), ("d_guess_pcm", "d_guess"))):
                        if k == 0 and song_div:
                            div = h["d_wav_div"][a:b]                  # the song's peak (util_audio.py:781)
                        else:
                            div = ops.pcm16_absmax(h[src][a:b], out=h["d_peak"][k, a:b])
                        ops.pcm16_to_wave(h[src][a:b], mul=h["d_mul"][k, a:b], div=div, out=h[dst][a:b])
                self._run(h["d_wav"], h["d_guess"], h["d_offs"], w0=a, w1=b)
                if feats:
                    self._reduce_features(h, a, b)
                e2 = torch.cuda.Event()
                e2.record(s_cmp)
                ev_cmp.append(e2)
        with torch.cuda.stream(s_out):
            for (a, b), e in zip(bounds, ev_cmp):
                s_out.wait_event(e)
                if feats:
                    for k in ("D8", "C8", "timing"):
                        h[k][a:b].copy_(h["d_" + k][a:b], non_blocking=True)
                else:
                    h["C"][a:b].copy_(self.C[a:b], non_blocking=True)
                h["ref"][a:b].copy_(self.ref[a:b], non_blocking=True)
        done = torch.cuda.Event()
        done.record(s_out)
        cur.wait_event(done)
        cur.wait_event(ev_in[-1])

    # ---- reduced, classifier-ready outputs of the e2e path (K5 on the device) ----------------------
    FEATURE_COLS = 8          # pitch_frames / instrument_frames of the reference (util_train_test.py:41-59)
    TIMING_BANDS = 20         # timing_bands

    def feature_buffers(self):
        """Device + pinned host buffers of `run_host(returns="features")`: per window
        D8 [8, P]   the dB image's 8 columns from the guessed note's onset frame (util_audio.py:176-180 -> :469-507),
        C8 [8, Pc]  the same columns of the constant-Q magnitudes (util_audio.py:431-434),
        timing [T, 20] compress_bands of the subtracted magnitude / song ref_mag (training.py:333-336),
        ref [1]     post-subtraction ref_mag."""
        h = self.host_buffers()
        if "D8" not in h:
            pin, d, n = dict(pin_memory=True), self.dev, self.FEATURE_COLS
            Pb = ops.frame_pitch(self.TIMING_BANDS)
            shapes = dict(D8=(self.W, n, self.P), C8=(self.W, n, self.Pc), timing=(self.W, self.T, Pb))
            for k, shp in shapes.items():
                h["d_" + k] = torch.empty(shp, device=d, dtype=torch.float32)
                h[k] = torch.empty(shp, dtype=torch.float32, **pin)
            h["cols"] = torch.arange(n, device=d, dtype=torch.int32).reshape(1, n)
            from .util_audio import band_edges
            h["edges"] = band_edges(self.nb, self.TIMING_BANDS)
            h["inv_song"] = torch.empty((self.W,), device=d, dtype=torch.float32)
        return h

    def _reduce_features(self, h, a, b):
        """K5 on windows [a, b): what the classifiers consume instead of the full CQT / dB images."""
        src = h["d_offs"][a:b] + h["cols"]                               # onset frame + 0..7   (index bookkeeping)
        src_d = torch.where(src < self.T, src, torch.full_like(src, -1))
        src_c = torch.where(src < self.Tc, src, torch.full_like(src, -1))
        ops.gather_frames_batch(self.D[a:b, :self.T], self.nb, src_d, out=h["d_D8"][a:b])
        ops.gather_frames_batch(self.C[a:b], self.cqt.n_bins, src_c, out=h["d_C8"][a:b])
        torch.reciprocal(self.clip_max[a:b], out=h["inv_song"][a:b])
        ops.compress_bands_batch(self.mag[a:b, :self.T], self.nb, h["edges"], inv_scale=h["inv_song"][a:b],
                                 out=h["d_timing"][a:b])

    def h2d_bytes(self, pcm16=False):
        if pcm16:
            return self.W * (2 * (self.ns + self.ng) + 4 + 16 + 8)
        return 4 * self.W * (self.ns + self.ng + 1)

    def d2h_bytes(self, returns="cqt"):
        if returns == "features":
            n = self.FEATURE_COLS
            return 4 * self.W * (n * self.P + n * self.Pc + self.T * ops.frame_pitch(self.TIMING_BANDS) + 1)
        return 4 * self.W * (self.Tc * self.Pc + 1)
