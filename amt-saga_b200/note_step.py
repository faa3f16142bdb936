"""Batched form of ONE iteration of the reference's per-note loop, in the reference's own order, for W
analysis windows at once (one note per window and step):

    training.py:333-336   C_timing      = _resize(compress_bands(audio_w.mag, 20), 258) / song ref_mag      K5
    training.py:337       audio_sw      = audio_w.resize(onset, duration, 8, ['mag', 'ph'])                  K5
    training.py:340-346   C_sw_pitch / C_sw_inst = audio_w.slice_C(...)/ref_C     (174 @ 24, 348 @ 48 per octave)   K4 + K2
    training.py:347-363   F_sw_inst_foc(_const)(_log10), ph                                                   K5
    training.py:365-388   C_sw_inst_foc / _foc_const (348 @ 192 per octave), C_velocity (36 @ 24)            K2
    training.py:426       ac_note_guessed = audio_complete(render(note), N)                                   K1
    training.py:449       audio_w.subtract(ac_note_guessed, offset=onset)                                     K3

`audio_w.slice_C` reads `audio_w.wf`, which after the first subtraction is `librosa.istft(mag * ph)`
(util_audio.py:88-106, length hop * (T - 1)): every step but the first therefore starts with K4 on the
subtracted windows.  Every subtraction scales the guess by the window's CURRENT maximum: `section` (training.py:284)
runs before the song's ref_mag is first evaluated (training.py:336), so it copies an empty `_ref_mag`, and the `mag`
setter resets it after each subtraction (a stale copied value can be modelled with `load(window_ref_mag=...)`).

The state (subtracted magnitudes, original phases, waveforms) stays on the device between steps; the eleven
classifier tensors come back as `[W, bands, frames]` CUDA tensors (`batches.py` stacks them for the models).
Host work per step is the float64 time -> frame arithmetic of util_audio.py:264 (vectorised, same operation
order) and the `_resize` index maps.  Windows whose note needs a CQT that librosa would refuse (pass band beyond
Nyquist) are reported in `valid` instead of raising, so one bad note does not lose the batch.
"""
import bisect

import numpy as np
import torch

from . import ops
from .cqt_plan import ParameterError
from .util_audio import band_edges, midi_to_hz, note_to_midi


class NoteStepBatch:
    def __init__(self, n_windows, sr=44100, n_fft=4096, hop_length=None, timing_frames=258, timing_bands=20,
                 pitch_frames=8, instrument_frames=8, pitch_bins_per_tone=2, instrument_bins_per_tone=4,
                 instrument_bands=348, bins_velocity=36, device=None):
        self.W, self.sr, self.N = int(n_windows), sr, int(n_fft)
        self.hl = int(hop_length) if hop_length is not None else self.N // 4
        self.T = int(timing_frames)
        self.timing_bands = timing_bands
        self.pitch_frames, self.instrument_frames = pitch_frames, instrument_frames
        self.pitch_bpt, self.inst_bpt = pitch_bins_per_tone, instrument_bins_per_tone
        self.instrument_bands, self.bins_velocity = instrument_bands, bins_velocity
        self.dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.stft = ops.get_stft_plan(self.N, self.hl, True, device=self.dev)
        self.nb = self.stft.n_bins
        self._fft_freq = np.linspace(0, float(sr) / 2, int(1 + self.N // 2), endpoint=True)   # util_audio.py:67
        self.mag = self.ph = self.wav = self.wav_lens = None
        self.state = None          # [W] int8: AUDIO / SYNCED / DIRTY / FULL (what `wav` holds, below)
        self._dirty = None         # frames changed by the last subtract of the DIRTY windows
        self.incremental_istft = True   # False: every rebuild of `wav` inverts all T frames (A/B twin)
        self.share_cascade = True       # False: every pitch group runs its own decimation cascade; "per_plan": shared
                                        # cascade but one contraction launch per pitch (A/B twins)
        self._tone_fft = None
        self._plan_frames = {}     # (note shape, distinct window lengths) -> [128 pitches, lengths] frame counts
        self.full_cqt = False      # True: every slice_C transforms all 258 columns like the reference (A/B twin)

    # What `wav[w, :wav_lens[w]]` holds -- the class's `_wf` and what the next step has to do to it:
    AUDIO = 0    # real audio: not subtracted since `load` or since a slide of a window that had a waveform
    SYNCED = 1   # the iSTFT of the current rows (rebuilt, no subtraction since)
    DIRTY = 2    # the iSTFT of the rows before the last subtraction: the next step patches the frames it changed
    FULL = 3     # stale (a subtraction of AUDIO rows, two subtractions, or a slide of a stale window): full iSTFT

    @property
    def _wav_synced(self):
        """Some window's `wav` is an iSTFT the next subtraction can patch incrementally."""
        return self.state is not None and bool(((self.state == self.SYNCED) | (self.state == self.DIRTY)).any())

    # ------------------------------------------------------------------ helpers (host, float64)
    def midi_tone_to_FFT(self, tone):          # util_audio.py:278-284
        ind = bisect.bisect_right(self._fft_freq, midi_to_hz(tone)) - 1
        return 0 if ind == 0 else ind - 1

    def _frames(self, seconds):
        """util_audio.py:264 for every window: floor(time * T * sr / len(wf)), float64, that order."""
        x = np.asarray(seconds, dtype=np.float64) * self.T * self.sr / self.wav_lens
        return np.floor(x).astype(np.int64)

    def _lens_arg(self, order=None):
        """`lens` for the CQT entries: None when every window fills the buffer (the dense path)."""
        if (self.wav_lens == self.wav.shape[1]).all():
            return None
        return self.wav_lens if order is None else self.wav_lens[order]

    @staticmethod
    def _length_ok(plan, lens):
        """Per window: does librosa accept a signal of this length for `plan` (check_length, per distinct length)."""
        u, inv = np.unique(np.asarray(lens, dtype=np.int64), return_inverse=True)
        ok = np.ones(len(u), dtype=bool)
        for i, n in enumerate(u):
            try:
                plan.check_length(int(n))
            except ParameterError:
                ok[i] = False
        return ok[inv.reshape(-1)]

    _resize_tables = {}

    @classmethod
    def _resize_map(cls, s, t, n_src, target):
        """Source column of every output column of `_resize(P[:, s:t], target)` for each window (numpy slice
        clipping included); -1 = the all-zero result of an empty slice.  `_resize` of a slice of n columns only
        depends on n up to `target` (n >= target keeps the first `target` columns): one table row per n."""
        tbl = cls._resize_tables.get(target)
        if tbl is None:
            tbl = np.stack([ops.resize_indices(n, target) for n in range(target + 1)]).astype(np.int32)
            cls._resize_tables[target] = tbl
        a_c = np.clip(np.asarray(s, dtype=np.int64), 0, n_src)
        b_c = np.clip(np.asarray(t, dtype=np.int64), 0, n_src)
        idx = tbl[np.minimum(np.maximum(b_c - a_c, 0), target)]
        return np.where(idx >= 0, idx + a_c[:, None], -1).astype(np.int32)

    def _upload(self, host):
        """All of a step's small index tables in ONE pinned staging buffer and one asynchronous copy (a pageable
        torch.as_tensor per table is a blocking copy behind everything queued on the stream: 62 of them made the
        step host-bound).  Returns {name: int32 device view}."""
        sizes = [(k, v.shape, int(v.size)) for k, v in host.items()]
        total = sum(n for _, _, n in sizes)
        stage = torch.empty(total, dtype=torch.int32, pin_memory=True)
        flat = stage.numpy()
        o = 0
        for (k, _, n) in sizes:
            flat[o:o + n] = np.asarray(host[k], dtype=np.int32).reshape(-1)
            o += n
        dbuf = stage.to(self.dev, non_blocking=True)
        out, o = {}, 0
        for (k, shape, n) in sizes:
            out[k] = dbuf[o:o + n].view(shape)
            o += n
        return out

    # ------------------------------------------------------------------ state
    def load(self, mag_storage, phase_storage, wav, song_ref_mag, ref_C, window_ref_mag=None, wav_lens=None):
        """Windows as `mid_wf.section(offset, None, timing_frames)` leaves them (training.py:284):
        mag_storage / phase_storage: frame-major [W, T, P] (columns of the SONG's STFT), wav [W, L] the matching
        waveform slices, song_ref_mag [W] = mid_wf.ref_mag (the features' normaliser, training.py:336),
        ref_C [W, 3] = (ref_C_1, ref_C_inst, ref_C_foc).  window_ref_mag: the `_ref_mag` the section carries -- None
        (default) when the song's had not been evaluated yet at `section` time, which is training.py's order: the
        first subtraction then scales by the window's own maximum; pass the song's to model a stale copy.
        wav_lens [W]: the length of each window's waveform (what the class's `len(wf)` is) when `wav` is a padded batch
        of windows of different lengths; None = every window is wav.shape[1] samples."""
        f32 = lambda x: torch.as_tensor(np.asarray(x, dtype=np.float32) if not isinstance(x, torch.Tensor) else x,
                                        device=self.dev).to(torch.float32).contiguous()
        if mag_storage.shape[:2] != (self.W, self.T) or phase_storage.shape != mag_storage.shape:
            raise ValueError("expected [W, T, P] magnitude and phase storage")
        self.mag, self.ph = mag_storage.contiguous(), phase_storage.contiguous()
        self.wav = wav.to(device=self.dev, dtype=torch.float32).contiguous()
        if wav_lens is None:
            self.wav_lens = np.full(self.W, self.wav.shape[1], dtype=np.int64)
        else:
            self.wav_lens = np.asarray(wav_lens.cpu() if isinstance(wav_lens, torch.Tensor) else wav_lens,
                                       dtype=np.int64).reshape(-1).copy()
            if self.wav_lens.shape != (self.W,) or (self.wav_lens < 1).any() or (self.wav_lens > self.wav.shape[1]).any():
                raise ValueError("wav_lens must be [W] with 1 <= len <= wav.shape[1]")
        self.song_ref = f32(song_ref_mag)
        self.inv_song_ref = 1.0 / self.song_ref
        rc = np.asarray(ref_C.cpu() if isinstance(ref_C, torch.Tensor) else ref_C, dtype=np.float64).reshape(self.W, 3)
        self.inv_ref_C = [f32(1.0 / rc[:, i]) for i in range(3)]
        # the `ref_mag` the next subtraction of each window scales by (< 0: the window's maximum at that moment)
        if window_ref_mag is None:
            _, self._ref_init = ops.subtract_db_batch(self.mag, None, None, self.nb, want_D=False)   # max of each window
        else:
            self._ref_init = f32(window_ref_mag)   # `section` copied a cached ref_mag (util_audio.py:323)
        self._ref_given = np.full(self.W, window_ref_mag is not None)
        self.state = np.full(self.W, self.AUDIO, dtype=np.int8)
        self._dirty = None

    # ------------------------------------------------------------------ one batched step
    def _cqt_prepare(self, L, lowest_midi, nbins, bpt, s, t, n_cols):
        """Host side of one slice_C shape for windows of L[w] samples: the plan, which windows librosa accepts, the
        first column each window needs and the `_resize` map relative to it (frame-window form) or absolute (full
        transform)."""
        plan = ops.get_cqt_plan(self.sr, self.hl, midi_to_hz(lowest_midi), int(nbins), int(12 * bpt), 2, device=self.dev)
        L = np.broadcast_to(np.asarray(L, dtype=np.int64), np.shape(s))
        ok = self._length_ok(plan, L)
        u, inv = np.unique(L, return_inverse=True)
        Tc = np.array([plan.num_frames(int(n)) for n in u], dtype=np.int64)[inv.reshape(-1)]
        src = self._resize_map(s, t, Tc, n_cols)                                     # C[:, s:t] -> _resize
        windowed = n_cols <= 8 and not self.full_cqt
        # whatever t - s is, `_resize` keeps columns of [s, s + n_cols): contract only those (K2 frame window)
        first = np.clip(s, 0, np.maximum(Tc - 1, 0)).astype(np.int32)
        rel = np.where(src >= 0, src - first[:, None], -1).astype(np.int32) if windowed else src
        assert not windowed or rel.max(initial=-1) < n_cols
        return plan, windowed, first, rel, ok

    def _cqt_run(self, wav, plan, windowed, first_dev, rel_dev, n_cols, nbins, inv_ref, lens=None):
        if windowed:
            C = ops.cqt_frames_batch(wav, plan, first_dev, n_cols, lens=lens)        # [W', n_cols, Pc]
        else:
            C = ops.cqt_batch(wav, plan, lens=lens)["mag_storage"]                   # [W', Tc, Pc]
        return ops.gather_frames_batch(C, nbins, rel_dev, inv_ref)                   # / ref_C

    def _cqt_columns(self, wav, lowest_midi, nbins, bpt, s, t, n_cols, inv_ref):
        plan, windowed, first, rel, ok = self._cqt_prepare(wav.shape[1], lowest_midi, nbins, bpt, s, t, n_cols)
        if not ok.all():
            plan.check_length(int(wav.shape[1]))
        d = self._upload({"first": first, "rel": rel})
        return self._cqt_run(wav, plan, windowed, d["first"], d["rel"], n_cols, nbins, inv_ref)

    def _pitch_groups(self, p_s, L_s, nbins, bpt, shift):
        """Runs [a, b) of equal pitch in the pitch-sorted windows with the plan of the note-relative shape (lowest note
        pitch + shift); None where librosa refuses the plan.  Also the windows librosa refuses (plan or length)."""
        W = len(p_s)
        groups, a, refused = [], 0, np.zeros(W, dtype=bool)
        while a < W:
            b = a + int(np.searchsorted(p_s[a:], p_s[a], side="right"))
            try:
                plan = ops.get_cqt_plan(self.sr, self.hl, midi_to_hz(int(p_s[a]) + shift), int(nbins), int(12 * bpt), 2,
                                        device=self.dev)
                ok = self._length_ok(plan, L_s[a:b])
                if not ok.any():
                    plan.check_length(int(L_s[a]))
                refused[a:b] = ~ok
                groups.append((a, b, plan))
            except ParameterError:      # librosa: "Filter pass-band lies beyond Nyquist" -> the loop skips the file
                refused[a:b] = True
                groups.append((a, b, None))
            a = b
        return groups, refused

    def _note_frames(self, si, groups, starts, p_s, Tc0, u_len, inv_len):
        """Frames of each (pitch-sorted) window's transform for note-relative shape si: the plan's count, which early
        decimation can make 1 + L // hop + 1.  A table per shape and set of window lengths holds each pitch's counts,
        so a step only computes the pitches it has not seen (0 = unknown; refused plans keep Tc0 = 1 + L // hop)."""
        key = (si, u_len.tobytes())
        tab = self._plan_frames.get(key)
        if tab is None:
            tab = self._plan_frames[key] = np.zeros((128, len(u_len)), dtype=np.int64)
        if p_s[0] < 0 or p_s[-1] > 127:          # (sorted) pitches outside MIDI's range: no table, every group computed
            Tc = Tc0.copy()
            for a, b, plan in groups:
                if plan is not None:
                    Tc[a:b] = np.array([plan.num_frames(int(n)) for n in u_len], dtype=np.int64)[inv_len[a:b]]
            return Tc
        for g in np.flatnonzero(tab[p_s[starts], 0] == 0):
            a, b, plan = groups[g]
            if plan is not None:
                tab[p_s[a]] = [plan.num_frames(int(n)) for n in u_len]
        known = tab[p_s, inv_len]
        return np.where(known > 0, known, Tc0)

    def step(self, onset, duration, pitch, guess_wav, guess_lens=None, subtract=True):
        """onset / duration (seconds, relative to the window) and MIDI pitch per window (host arrays, [W]);
        guess_wav [W, Lg]: the rendered guessed notes (device float32; `guess_lens` for ragged renders).
        Returns the note_sample tensors (util_train_test.py:177-209) as [W, bands, frames] CUDA tensors plus
        `valid` [W] (bool, host) and `offset_frames` [W]; then subtracts the guesses (training.py:449)."""
        W = self.W
        onset = np.asarray(onset, dtype=np.float64).reshape(W)
        duration = np.asarray(duration, dtype=np.float64).reshape(W)
        pitch = np.asarray(pitch, dtype=np.int64).reshape(W)
        if (self.state >= self.DIRTY).any():
            # util_audio.py:88-106: wf is rebuilt from the subtracted magnitude and the original phase
            self._rebuild_wav()
        s, t = self._frames(onset), self._frames(onset + duration)
        out = {}
        Lw = self.wav_lens
        lens = self._lens_arg()
        a0, c8 = note_to_midi("A0"), note_to_midi("C8")
        nf = self.instrument_frames
        # ---- host: every index table of the step, then ONE upload ------------------------------------------
        if self._tone_fft is None:
            self._tone_fft = np.array([self.midi_tone_to_FFT(p) for p in range(128)], dtype=np.int32)
        host = {"sw_src": self._resize_map(s, t, self.T, self.pitch_frames),
                "b_note": self._tone_fft[np.clip(pitch, 0, 127)]}
        const_shapes = (("C_sw_pitch", a0, (c8 - a0) * self.pitch_bpt, self.pitch_bpt, self.pitch_frames, 0),
                        ("C_sw_inst", a0, (c8 - a0) * self.inst_bpt, self.inst_bpt, nf, 1),
                        ("C_sw_inst_foc_const", 60, self.instrument_bands, self.inst_bpt * 4, nf, 2))
        const_plans = {}
        valid = np.ones(W, dtype=bool)
        for name, low, nbins, bpt, n_cols, _ in const_shapes:
            plan, windowed, first, rel, ok = self._cqt_prepare(Lw, low, nbins, bpt, s, t, n_cols)
            const_plans[name] = (plan, windowed, ok)
            valid &= ok
            host["first_" + name], host["rel_" + name] = first, rel
        # the two note-relative transforms have one kernel bank per pitch: windows are sorted by pitch once, every
        # pitch group contracts its <= 8 columns straight into its slice of ONE compact buffer, and one gather
        # (C[:, s:t] -> _resize -> / ref_C_foc) serves all windows
        order = np.argsort(pitch, kind="stable")
        host["order"], host["inv_order"] = order, np.argsort(order)
        s_s, t_s, p_s = s[order], t[order], pitch[order]
        L_s = Lw[order]
        lens_s = self._lens_arg(order)
        part = (lambda a, b: None) if lens_s is None else (lambda a, b: lens_s[a:b])
        full = self.full_cqt
        # the `_resize` maps for 1 + L // hop frames; a note-relative plan with early decimation can have one frame more,
        # and the windows whose slice reaches that frame get their own rows below
        Tc0 = 1 + L_s // self.hl
        src0 = self._resize_map(s_s, t_s, Tc0, nf)
        first0 = np.clip(s_s, 0, np.maximum(Tc0 - 1, 0)).astype(np.int32)
        host["first_s"] = first0
        host["rel_s"] = src0 if full else np.where(src0 >= 0, src0 - first0[:, None], -1)
        off = np.maximum(s, 0).astype(np.int32)       # util_audio.py:248 with attack_compensation 0
        host["off"] = off
        d = self._upload(host)
        # ---- device ---------------------------------------------------------------------------------------------
        # -- timing classifier input (training.py:333-336)
        edges = band_edges(self.nb, self.timing_bands)
        ct = ops.compress_bands_batch(self.mag, self.nb, edges, inv_scale=self.inv_song_ref)
        out["C_timing"] = ct[:, :, :self.timing_bands].transpose(1, 2)              # T == timing_frames: _resize is the identity
        # -- short window (training.py:337, :347-363)
        b_const = self.midi_tone_to_FFT(60)
        fc = ops.short_window_features_batch(self.mag, None, d["sw_src"], b_const, self.instrument_bands, self.nb,
                                             self.inv_song_ref)
        out["F_sw_inst_foc_const"], out["F_sw_inst_foc_const_log10"] = fc["lin"], fc["log"]
        fn = ops.short_window_features_batch(self.mag, self.ph, d["sw_src"], d["b_note"], self.instrument_bands, self.nb,
                                             self.inv_song_ref, want_phase=True)
        out["F_sw_inst_foc"], out["F_sw_inst_foc_log10"], out["ph"] = fn["lin"], fn["log"], fn["phase"]
        # -- constant-Q inputs (training.py:340-346, :365-388); filter_scale 2 (util_audio.py:426)
        for name, low, nbins, bpt, n_cols, ref_i in const_shapes:
            plan, windowed, ok = const_plans[name]
            out[name] = self._cqt_run(self.wav, plan, windowed, d["first_" + name], d["rel_" + name], n_cols, nbins,
                                      self.inv_ref_C[ref_i], lens=lens)
            if not ok.all():        # librosa refuses these windows' lengths: the loop skips their files
                out[name][torch.as_tensor(~ok, device=self.dev)] = float("nan")
        wav_s = self.wav.index_select(0, d["order"])
        inv_ref_s = self.inv_ref_C[2].index_select(0, d["order"])
        res = []
        if len(self._plan_frames) > 256:       # windows of ever new lengths (song walks): keep the cache bounded
            self._plan_frames.clear()
        if lens_s is None:
            u_len, inv_len = L_s[:1], np.zeros(W, dtype=np.int64)
        else:
            u_len, inv_len = np.unique(L_s, return_inverse=True)
            inv_len = inv_len.reshape(-1)
        starts = np.flatnonzero(np.r_[True, p_s[1:] != p_s[:-1]])      # the pitch groups' first windows
        note_shapes = ((self.instrument_bands, self.inst_bpt * 4, 0), (self.bins_velocity, 2, -10))
        for si, (nbins, bpt, shift) in enumerate(note_shapes):
            P = ops.frame_pitch(nbins)
            groups, refused = self._pitch_groups(p_s, L_s, nbins, bpt, shift)
            Tc = self._note_frames(si, groups, starts, p_s, Tc0, u_len, inv_len)
            first_dev, rel_dev = d["first_s"], d["rel_s"]
            r = np.flatnonzero((Tc != Tc0) & (np.maximum(s_s, t_s) >= np.minimum(Tc, Tc0) - 1))
            if len(r):
                src = self._resize_map(s_s[r], t_s[r], Tc[r], nf)
                first = np.clip(s_s[r], 0, np.maximum(Tc[r] - 1, 0))
                u = self._upload({"r": r, "first": first, "rel": src if full else np.where(src >= 0, src - first[:, None], -1)})
                rows = u["r"].long()
                first_dev = first_dev.index_copy(0, rows, u["first"])
                rel_dev = rel_dev.index_copy(0, rows, u["rel"])
            buf = torch.zeros((W, int(Tc.max()) if full else nf, P), device=self.dev, dtype=torch.float32)
            i = 0
            while i < len(groups):
                a, b, plan = groups[i]
                if plan is None:
                    i += 1
                    continue
                if full:
                    C = ops.cqt_batch(wav_s[a:b], plan, lens=part(a, b))["mag_storage"]
                    buf[a:b, :C.shape[1]] = C
                    i += 1
                    continue
                # consecutive pitches of equal geometry (early factor, levels, kernel length) decimate the audio the same
                # way: ONE cascade for the whole run, then one contraction per pitch with its own bank
                j = i
                while self.share_cascade and j + 1 < len(groups) and groups[j + 1][2] is not None and \
                        groups[j + 1][2].geometry() == plan.geometry():
                    j += 1
                if j == i:
                    ops.cqt_frames_batch(wav_s[a:b], plan, first_dev[a:b], nf, lens=part(a, b), out=buf[a:b])
                else:
                    A, B = a, groups[j][1]
                    token = ops.cqt_cascade_shared(wav_s[A:B], plan, lens=part(A, B))
                    run = groups[i:j + 1]
                    if self.share_cascade == "per_plan":      # one contraction launch per pitch (A/B twin)
                        for (ga, gb, gp) in run:
                            ops.cqt_frames_from_cascade(token, gp, ga - A, gb - ga, first_dev[ga:gb], nf, buf[ga:gb])
                    else:                                     # all pitches of the run in ~one launch per 10 banks
                        ops.cqt_frames_from_cascade_multi(token, [g_[2] for g_ in run], [g_[0] - A for g_ in run],
                                                          [g_[1] - g_[0] for g_ in run], first_dev[A:B], nf, buf[A:B])
                i = j + 1
            if refused.any():
                valid[order[refused]] = False
                buf[torch.as_tensor(refused, device=self.dev)] = float("nan")
            g = ops.gather_frames_batch(buf, nbins, rel_dev, inv_ref_s)
            res.append(g.index_select(0, d["inv_order"]))
        foc, vel = res
        out["C_sw_inst_foc"], out["C_velocity"] = foc, vel
        out["valid"], out["offset_frames"] = valid, off
        if subtract:
            self.subtract(guess_wav, off, guess_lens, offset_dev=d["off"])
        return out

    def _rebuild_wav(self):
        """`wf` after a subtraction (util_audio.py:88-106: istft of magnitude x phase).  The first rebuild inverts every
        frame (the window's original audio is not an iSTFT).  From then on `wav` IS the iSTFT of the previous
        magnitudes and a subtraction changes frames [o, o + tg) only: with n_fft = 4 hops a sample depends on 4
        frames, so the samples that change are [(o - 2) hop, (o + tg + 2) hop), computed from frames
        [o - 4, o + tg + 4): gather those rows, invert them (K4 on ~1/4 of the frames) and patch that sample range.
        Same frames, same accumulation order per sample: the patched waveform equals the full rebuild.
        Per window: FULL windows are inverted whole, DIRTY ones patched, AUDIO / SYNCED ones left alone -- at most one
        K4 call of each kind for the batch.  The [W, L] buffer grows if hop * (T - 1) is wider than it."""
        d = self._dirty
        full, dirty = self.state == self.FULL, self.state == self.DIRTY
        if dirty.any() and (d is None or not self.incremental_istft or d["F"] >= self.T):
            full, dirty = full | dirty, np.zeros_like(dirty)
        Li = self.hl * (self.T - 1)
        if full.all():
            self.wav = ops.istft_batch(self.stft, mag=self.mag, phase=self.ph, n_bins=self.nb)
        else:
            if self.wav.shape[1] < Li:
                self.wav = torch.nn.functional.pad(self.wav, (0, Li - self.wav.shape[1]))
            if dirty.any() and d["any"]:
                F, hop = d["F"], self.hl
                y = ops.istft_batch(self.stft, mag=self.mag, phase=self.ph, n_bins=self.nb, frame0=d["fa32"], n_frames=F)   # [W, (F-1) hop]
                idx = d["fa"][:, None] * hop + torch.arange(y.shape[1], device=self.dev)   # global sample of every sub sample
                keep = (idx >= d["lo"][:, None]) & (idx < d["hi"][:, None])
                self.wav.scatter_(1, idx, torch.where(keep, y, self.wav.gather(1, idx)))
            if full.any():
                sel = torch.as_tensor(np.flatnonzero(full), device=self.dev)
                y = ops.istft_batch(self.stft, mag=self.mag.index_select(0, sel), phase=self.ph.index_select(0, sel),
                                    n_bins=self.nb)
                self.wav.index_copy_(0, sel, torch.nn.functional.pad(y, (0, self.wav.shape[1] - y.shape[1])))
        self.wav_lens[full | dirty] = Li
        self.state[full | dirty] = self.SYNCED
        self._dirty = None

    def wf(self):
        """The class's `wf` getter for every window: pending rebuilds run now (the next step then has none) and
        (wav [W, L], wav_lens [W] host) come back.  Like reading `audio_w.wf`, it leaves each window holding its
        waveform, so a slide before the next subtraction cuts that waveform instead of dropping it."""
        if (self.state >= self.DIRTY).any():
            self._rebuild_wav()
        return self.wav, self.wav_lens.copy()

    def ref_mag(self):
        """The class's `ref_mag` getter for every window (util_audio.py:170-174): the window's current maximum unless
        one is cached, and caches it -- a slide keeps a cached value (slice / concat do not touch `_ref_mag`), so the
        next subtraction scales by it instead of by the slid window's maximum.  Returns [W] float32 CUDA."""
        need = ~self._ref_given
        if need.any():
            _, cur = ops.subtract_db_batch(self.mag, None, None, self.nb, want_D=False)   # max of each window now
            self._ref_init = torch.where(torch.as_tensor(need, device=self.dev), cur, self._ref_init)
            self._ref_given[:] = True
        return self._ref_init

    def _apply_slide(self, m, song_idx, g, song_mag, song_phase, song_wav, song_lens=None):
        """State side of a half-window slide (training.py:317-328) of windows m (host, distinct), with the host
        geometry `song_setup.slide_geometry` gives: the rows (one slide-kernel launch), the waveforms and the
        per-window state.  A window that holds a waveform (AUDIO / SYNCED) keeps `wf[a:b]` of it followed by the new
        half's samples, one gather for all of them; any other window's `wf` is None in the class and becomes FULL: the
        next step inverts all T rows.  song_mag None: the songs are held as waveforms (song_wav [S, L], song_lens [S])
        and the new halves' rows are computed from them."""
        h = self.T // 2
        m = np.asarray(m, dtype=np.int64)
        if song_mag is None:
            # with no live song rows the kernel only moves rows [h, 2h) down (and zeroes them): it never reads song
            # storage, so the window storages stand in for it; the new halves then go straight into rows [h, 2h)
            none = np.zeros(len(m), dtype=np.int64)
            ops.window_slide_batch(self.mag, self.ph, self.nb, h, m, none, none, none, self.mag, self.ph)
            ops.stft_rows_batch(song_wav, self.stft, g["tfs"], h, lens=song_lens, clip_rows=song_idx, out=self.mag,
                                phase_out=self.ph, dst_clip=m, dst_row0=h)
        else:
            ops.window_slide_batch(self.mag, self.ph, self.nb, h, m, song_idx, np.where(g["rows"] > 0, g["tfs"], 0),
                                   g["rows"], song_mag, song_phase)
        has_wf = (self.state[m] == self.AUDIO) | (self.state[m] == self.SYNCED)
        a, keep, n_copy, new_len = g["a"], g["keep"], g["n_copy"], g["wav_len"]
        w0 = g["w0"]
        ma = np.flatnonzero(has_wf)
        cat = None
        if len(ma):
            Lc = int(new_len[ma].max())
            d = self._upload({"row": m[ma], "a": a[ma], "keep": keep[ma], "song": np.asarray(song_idx)[ma],
                              "w0": np.asarray(w0)[ma], "n_copy": np.asarray(n_copy)[ma]})
            j = torch.arange(Lc, device=self.dev)[None, :]
            kp, nc = d["keep"].long()[:, None], d["n_copy"].long()[:, None]
            old = self.wav[d["row"].long()[:, None], (d["a"].long()[:, None] + j).clamp(max=self.wav.shape[1] - 1)]
            new = song_wav[d["song"].long()[:, None], (d["w0"].long()[:, None] + j - kp).clamp(0, song_wav.shape[1] - 1)]
            cat = torch.where(j < kp, old, torch.where((j >= kp) & (j < kp + nc), new, 0.0))
        width = max(self.wav.shape[1], int(new_len.max()))
        if width > self.wav.shape[1]:
            self.wav = torch.nn.functional.pad(self.wav, (0, width - self.wav.shape[1]))
        if cat is not None:
            self.wav.index_copy_(0, d["row"].long(), torch.nn.functional.pad(cat, (0, width - cat.shape[1])))
        self.wav_lens[m] = new_len
        self.state[m] = np.where(has_wf, self.AUDIO, self.FULL).astype(np.int8)
        # slice / concat keep `_ref_mag`: a copied one stays; None (subtracted, or never set) is the max at the next
        # subtraction, which after the slide is the slid window's (util_audio.py:170-174)
        drop = m[~self._ref_given[m]]
        if len(drop):
            self._ref_init = self._ref_init.index_fill(0, torch.as_tensor(drop, device=self.dev), -1.0)

    def _apply_refill(self, slots, wav, wav_lens, song_ref_mag, ref_C):
        """State side of SongBatch.refill: windows `slots` (host, distinct), whose rows the caller has written, now hold
        a fresh section -- waveform wav [n, >= max(wav_lens)], song_ref_mag [n], ref_C [n, 3] -- in the state `load`
        leaves (AUDIO, the window's own maximum at its first subtraction).  The other windows keep theirs, bit for bit.
        A refilled window that was DIRTY must leave the pending patch: `_rebuild_wav` writes its sample range
        [lo, hi) into every window, so that range is emptied (hi = lo) -- otherwise the old rows' samples would land
        in the new song's audio."""
        slots = np.asarray(slots, dtype=np.int64)
        sl = torch.as_tensor(slots, device=self.dev)
        wav = wav.to(device=self.dev, dtype=torch.float32)
        width = max(self.wav.shape[1], wav.shape[1])
        if width > self.wav.shape[1]:
            self.wav = torch.nn.functional.pad(self.wav, (0, width - self.wav.shape[1]))
        self.wav.index_copy_(0, sl, torch.nn.functional.pad(wav, (0, width - wav.shape[1])))
        self.wav_lens[slots] = np.asarray(wav_lens, dtype=np.int64)
        ref = song_ref_mag.to(device=self.dev, dtype=torch.float32)
        self.song_ref = self.song_ref.index_copy(0, sl, ref)
        self.inv_song_ref = self.inv_song_ref.index_copy(0, sl, 1.0 / ref)
        rc = np.asarray(ref_C, dtype=np.float64).reshape(len(slots), 3)
        self.inv_ref_C = [c.index_copy(0, sl, torch.as_tensor((1.0 / rc[:, i]).astype(np.float32), device=self.dev))
                          for i, c in enumerate(self.inv_ref_C)]
        self._ref_init = self._ref_init.index_fill(0, sl, -1.0)
        self._ref_given[slots] = False
        self.state[slots] = self.AUDIO
        if self._dirty is not None:
            self._dirty["hi"] = self._dirty["hi"].index_copy(0, sl, self._dirty["lo"].index_select(0, sl))

    @staticmethod
    def _dirty_ranges(offset_frames, guess_frames, T, N, hop):
        """Frames [o, o + tg) of a T-frame centred STFT (n_fft N, hop) changed.  Returns (F, fa, lo, hi, tg): the
        samples [lo, hi) of the hop (T - 1)-sample iSTFT that depend on them, and per window the first row fa of an
        F-row block whose own iSTFT reproduces those samples exactly (every frame that reaches them is in the block,
        or the block touches the true edge of the window)."""
        m = N // (2 * hop)                               # frames on either side of floor(n / hop) that reach sample n
        o = np.clip(np.asarray(offset_frames, dtype=np.int64), 0, T)
        tg = np.minimum(np.asarray(guess_frames, dtype=np.int64), T - o)
        F = int(min(T, int(tg.max(initial=0)) + 4 * m))
        fa = np.clip(o - 2 * m, 0, T - F)
        L = hop * (T - 1)
        lo = np.clip((o - m) * hop, 0, L)
        hi = np.where(tg > 0, np.clip((o + tg + m) * hop, 0, L), lo)
        return F, fa, lo, hi, tg

    def _mark_dirty(self, offset_frames, guess_frames):
        """Host side of the incremental rebuild: per SYNCED window the frame range the subtraction touched.  Any other
        window's `wav` is audio, or already stale (a second subtraction before the rebuild): it is inverted whole."""
        syn = self.state == self.SYNCED
        self.state = np.where(syn, self.DIRTY, self.FULL).astype(np.int8)
        if not syn.any():
            self._dirty = None
            return
        tg_in = np.where(syn, np.asarray(guess_frames, dtype=np.int64), 0)
        F, fa, lo, hi, tg = self._dirty_ranges(offset_frames, tg_in, self.T, self.N, self.hl)
        dev = self._upload({"fa": fa, "lo": lo, "hi": hi})
        self._dirty = {"F": F, "any": bool((tg > 0).any()), "fa32": dev["fa"], "fa": dev["fa"].long(), "lo": dev["lo"].long(),
                       "hi": dev["hi"].long()}

    def subtract(self, guess_wav, offset_frames, guess_lens=None, offset_dev=None):
        """training.py:426 + :449: STFT of the rendered notes (K1), then align / scale / subtract / ReLU (K3)."""
        g = ops.stft_batch(guess_wav, self.stft, lens=guess_lens, want_max=True)
        gm = g["mag_storage"]
        frames = None
        if guess_lens is not None:
            frames = torch.as_tensor([self.stft.num_frames(int(n)) for n in np.asarray(guess_lens)], dtype=torch.int32,
                                     device=self.dev).reshape(self.W, 1)
        if int(np.max(offset_frames)) > self.T:
            raise ValueError("negative dimensions are not allowed")      # numpy's error for zeros((bins, T - off - ...))
        self._mark_dirty(offset_frames, [self.stft.num_frames(int(n)) for n in np.asarray(guess_lens)] if guess_lens is not None
                         else np.full(self.W, self.stft.num_frames(int(guess_wav.shape[1]))))
        _, self.ref = ops.subtract_db_batch(
            self.mag, gm.unsqueeze(1),
            (offset_dev if offset_dev is not None else torch.as_tensor(offset_frames, dtype=torch.int32)).reshape(self.W, 1), self.nb,
            guess_ref=g["clip_max"].reshape(self.W, 1), ref_init=self._ref_init,
            guess_frames=frames,
            normalize=True, relu=True, want_D=False)
        # the `mag` setter dropped the copied ref_mag (util_audio.py:149-153); the next subtraction scales by the max
        self._ref_init = self.ref
        self._ref_given[:] = False
