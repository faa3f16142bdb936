"""Batched form of the producer loop's per-song setup (training.py:265-284) for S songs of different lengths:

    training.py:265-269   mid_wf = audio_complete(song, N); mid_wf.mag                  K1 (ragged batch)
    training.py:266       spectral flatness gate (songs above 0.3 are skipped)         K1 by-product + flatness kernel
    training.py:271-282   ref_C_1 / ref_C_inst / ref_C_foc = np.max(slice_C(0, dur, T))  K2 peak mode (no image)
    training.py:284       audio_w = mid_wf.section(offset, None, 258)                   row / sample gathers
    training.py:317-328   half-window slide (section + slice + concat)                  slide kernel + one sample gather
    training.py:289       fft_bin_min_const = midi_tone_to_FFT(60)
    training.py:336       song ref_mag                                                  K1 by-product

`slice_C(0, dur, T)` `_resize`s `C[:, 0:t]` to T columns, which only repeats or drops columns: its maximum is the
maximum of |C| over bins and columns [0, t), with t = floor(dur * T * sr / len) (util_audio.py:264) -- T - 1 for some
lengths, and then the last column is not part of it.  `ops.cqt_peak_batch` computes exactly that per song.

Songs the class would refuse (an empty buffer; a length librosa's CQT rejects, on which training.py:291-294 skips
the file) come back with `valid = False` and NaN normalisers instead of raising, so one bad file does not lose the
batch.  The float64 frame arithmetic below is the class's, operation for operation, vectorised over songs.
"""
import bisect

import numpy as np
import torch

from . import ops
from .cqt_plan import ParameterError
from .util_audio import midi_to_hz, note_to_hz, note_to_midi


# ---------------------------------------------------------------------------------- host frame arithmetic (float64)
def song_frames(lens, hop):
    """Frames of the centred song STFT: 1 + len // hop (0 for an empty song)."""
    lens = np.asarray(lens, dtype=np.int64)
    return np.where(lens > 0, 1 + lens // hop, 0)


def song_durations(T, lens, sr):
    """`_frames_to_seconds(T)` = T / T / sr * len (util_audio.py:269-272); NaN for an empty song."""
    T = np.asarray(T, dtype=np.int64)
    with np.errstate(invalid="ignore", divide="ignore"):
        return T / T / sr * np.asarray(lens, dtype=np.int64)


def seconds_to_frames(seconds, T, lens, sr):
    """`_seconds_to_frames` (util_audio.py:264): floor(time * T * sr / len), float64, that order."""
    with np.errstate(invalid="ignore", divide="ignore"):      # an empty song: NaN -> an arbitrary int, never used
        x = np.asarray(seconds, dtype=np.float64) * np.asarray(T, dtype=np.int64) * sr / np.asarray(lens, dtype=np.int64)
        return np.floor(x).astype(np.int64)


def frames_to_seconds(frames, T, lens, sr):
    return np.asarray(frames, dtype=np.int64) / np.asarray(T, dtype=np.int64) / sr * np.asarray(lens, dtype=np.int64)


def section_geometry(T, lens, offset_s, n_frames, sr):
    """`section(offset, None, n_frames)` of songs with T frames and `lens` samples (util_audio.py:286-328).
    Returns dict of int64 arrays: tfs / tfe (frame range), w0 / w1 (sample range), n_copy (samples copied from the
    song), pad (zeros appended: w1 - n_copy when the slice comes out short, (sic) util_audio.py:306) and wav_len."""
    T, lens = np.asarray(T, dtype=np.int64), np.asarray(lens, dtype=np.int64)
    tfs = seconds_to_frames(offset_s, T, lens, sr)
    tfe = tfs + int(n_frames)
    w0 = np.floor(frames_to_seconds(tfs, T, lens, sr) * sr).astype(np.int64)
    w1 = np.floor(frames_to_seconds(tfe, T, lens, sr) * sr).astype(np.int64)
    n_copy = np.maximum(np.minimum(w1, lens) - w0, 0)
    pad = np.where(n_copy < w1 - w0, w1 - n_copy, 0)
    return dict(tfs=tfs, tfe=tfe, w0=w0, w1=w1, n_copy=n_copy, pad=pad, wav_len=n_copy + pad)


def slide_geometry(T, wav_len, has_wf, T_song, song_len, offset_s, half_seconds, sr, hop):
    """Host side of the loop's half-window slide (training.py:317-328) of windows with T rows, waveforms of wav_len
    samples (has_wf: the class's `_wf` is not None) and offsets offset_s, in songs of T_song frames / song_len samples:
        offset += half_seconds; new = section(offset + half_seconds, None, h); slice(h, 2h); concat(new)
    Returns section_geometry's entries for the new half plus offset_s (the new offset), a / b (`slice`'s sample
    range, util_audio.py:351-365, python slice clipping), keep (= b - a samples kept), rows (live song rows of the
    new half), past_end (tfs > T_song: the class appends more than h columns) and wav_len (the window's new waveform
    length: keep + n_copy + pad with a waveform, hop (T - 1) -- the next iSTFT -- without)."""
    if T % 2:
        raise ValueError("slice(h, 2h) + concat of an odd T = %d leaves T - 1 frames" % T)
    h = T // 2
    L = np.asarray(wav_len, dtype=np.int64)
    T_song = np.asarray(T_song, dtype=np.int64)
    off = np.asarray(offset_s, dtype=np.float64) + half_seconds
    g = section_geometry(T_song, song_len, off + half_seconds, h, sr)
    a = np.minimum((h / T / sr * L * sr).astype(np.int64), L)
    b = np.minimum((2 * h / T / sr * L * sr).astype(np.int64), L)
    keep = np.maximum(b - a, 0)
    g.update(offset_s=off, a=a, b=b, keep=keep, rows=np.clip(T_song - g["tfs"], 0, h), past_end=g["tfs"] > T_song,
             wav_len=np.where(has_wf, keep + g["n_copy"] + g["pad"], hop * (T - 1)))
    return g


# ---------------------------------------------------------------------------------- windows
class SongWindows:
    """What `mid_wf.section(offset, None, n_frames)` leaves, for W windows of a SongBatch:
    mag / phase: frame-major storage [W, n_frames, P] (float32 / complex64), zero past the song's end;
    wav [W, max(wav_len)] float32, zero after each window's `wav_len[w]` samples; song_idx, offset_s (float64 [W],
    the window's offset in seconds, training.py's `offset`), and the host geometry of `section_geometry` (tfs, tfe,
    w0, w1, n_copy, pad, wav_len).  A window that starts past the song's end has n_frames zero rows here; the
    class's copy has tfe - T columns there ((sic) util_audio.py:318-321).  After `SongBatch.slide` the geometry
    entries of a slid window describe the half it appended, and wav_len is the window's whole waveform."""

    def __init__(self, mag, phase, wav, song_idx, geometry, offset_s):
        self.mag, self.phase, self.wav, self.song_idx = mag, phase, wav, song_idx
        self.geometry = geometry
        self.wav_len = geometry["wav_len"]
        self.offset_s = np.array(offset_s, dtype=np.float64)

    def stacked_wav(self):
        """[W, L] waveforms for NoteStepBatch.load, which takes windows of one length only."""
        lens = np.unique(self.wav_len)
        if len(lens) != 1:
            raise ValueError("windows have different waveform lengths %s: load them in separate batches" % lens.tolist())
        return self.wav[:, :int(lens[0])]


# ---------------------------------------------------------------------------------- songs
class SongBatch:
    """training.py:265-284 for a batch of songs.  The hyper-parameters are NoteStepBatch's: n_fft, hop (N / 4), sr,
    pitch_frames (slice_C's `magnitude_only` argument at training.py:271-282, truthy there) and the bins per tone of
    the three whole-song CQTs (87 x 1, 87 x 4 and 87 x 16 bins from A0, i.e. 12 / 48 / 192 bins per octave).

    hold: what the batch keeps of each song between calls.
      "stft"      the whole song STFT, mag / phase [S, T_max, P] (24 624 B per frame at n_fft 4096: 6x the float32
                  waveform); `section`, `slide` and `refill` gather their rows from it.
      "waveform"  the waveforms only (mag / phase are None); `section`, `slide` and `refill` compute the rows they need
                  with a frame-range STFT of the song (ops.stft_rows_batch).  Every row, waveform and normaliser equals
                  hold="stft"'s bit for bit.  For corpora whose STFT does not fit the device."""

    HOLDS = ("stft", "waveform")
    chunk_bytes = 1 << 28      # hold="waveform" setup: magnitude scratch per chunk of frames, samples per CQT call

    def __init__(self, sr=44100, n_fft=4096, hop_length=None, pitch_frames=8, bins_per_tone=(1, 4, 16),
                 flatness_threshold=0.3, lowest_note="A0", highest_note="C8", device=None, hold="stft"):
        if hold not in self.HOLDS:
            raise ValueError("hold must be one of %s, not %r" % (self.HOLDS, hold))
        self.hold = hold
        self.sr, self.N = sr, int(n_fft)
        self.hl = int(hop_length) if hop_length is not None else self.N // 4
        if not pitch_frames:
            raise ValueError("the whole-song CQTs are magnitudes (slice_C's magnitude_only is truthy at training.py:271-282)")
        self.pitch_frames = pitch_frames
        self.bins_per_tone = tuple(bins_per_tone)
        self.flatness_threshold = float(flatness_threshold)
        self.dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.stft = ops.get_stft_plan(self.N, self.hl, True, device=self.dev)
        self.nb = self.stft.n_bins
        low, high = note_to_midi(lowest_note), note_to_midi(highest_note)
        self.cqt_plans = [ops.get_cqt_plan(sr, self.hl, note_to_hz(lowest_note), int((high - low) * bpt), int(12 * bpt), 2,
                                           device=self.dev) for bpt in self.bins_per_tone]
        fft_freq = np.linspace(0, float(sr) / 2, int(1 + self.N // 2), endpoint=True)    # util_audio.py:67
        ind = bisect.bisect_right(fft_freq, midi_to_hz(60)) - 1                           # util_audio.py:278-284
        self.fft_bin_min_const = 0 if ind == 0 else ind - 1                                 # training.py:289

    def _wave_in(self, songs, lens):
        """[S, L_max] float32 device batch + host int64 lens."""
        if isinstance(songs, torch.Tensor):
            if not songs.is_cuda or songs.dim() != 2:
                raise ValueError("songs must be a [S, L_max] CUDA tensor or a list of host arrays")
            wav = songs.to(device=self.dev, dtype=torch.float32).contiguous()
            lens = np.full(wav.shape[0], wav.shape[1], dtype=np.int64) if lens is None else \
                np.asarray(lens.cpu() if isinstance(lens, torch.Tensor) else lens, dtype=np.int64)
            if lens.shape != (wav.shape[0],) or (lens < 0).any() or (lens > wav.shape[1]).any():
                raise ValueError("lens must be [S] with 0 <= len <= songs.shape[1]")
            return wav, lens
        if lens is not None:
            raise ValueError("lens go with a padded [S, L_max] tensor; a list of songs carries its own lengths")
        # float64 host songs are cast to float32 on the device, as audio_complete._wave_in does
        ts = [torch.as_tensor(np.asarray(s)).to(device=self.dev, dtype=torch.float32).reshape(-1) for s in songs]
        lens = np.array([t.numel() for t in ts], dtype=np.int64)
        wav = torch.zeros((len(ts), max(int(lens.max(initial=0)), 1)), device=self.dev, dtype=torch.float32)
        for i, t in enumerate(ts):
            wav[i, :t.numel()] = t
        return wav, lens

    def setup(self, songs, lens=None):
        """Runs training.py:265-284 for every song.  Sets (host arrays unless noted):
        T [S] frames, song_dur [S] float64, flatness [S] float64, keep [S] (flatness <= threshold), valid [S],
        ref_mag [S] float32 CUDA (the song's ref_mag), ref_C [S, 3] float64 (NaN where not valid), ref_cols [S] (the
        column range [0, ref_cols) of the whole-song CQT maxima), and under hold="stft" the song STFT as frame-major
        storage mag / phase [S, T_max, P] (zero past each song's end; None under hold="waveform").  Returns self."""
        wav, lens = self._wave_in(songs, lens)
        S = wav.shape[0]
        self.wav, self.lens = wav, lens
        self.T = song_frames(lens, self.hl)
        if self.hold == "stft":
            # -- song STFT (training.py:269) and ref_mag (:336): one ragged K1 call
            r = ops.stft_batch(wav, self.stft, lens=lens, want_phase=True, want_max=True)
            self.mag, self.phase, self.ref_mag = r["mag_storage"], r["phase_storage"], r["clip_max"]
            T_max = self.mag.shape[1]
            if T_max > 0:
                flat = ops.spectral_flatness_batch(self.mag, self.nb)
        else:
            self.mag = self.phase = None
            T_max = int(self.T.max(initial=0))
            self.ref_mag, flat = self._song_frames_walk(T_max)
        # -- flatness gate (:266): mean over each song's own frames (a zero frame past the end would count as 1)
        if T_max > 0:
            flat = flat.double()
            T_dev = torch.as_tensor(self.T, device=self.dev)
            mask = torch.arange(T_max, device=self.dev)[None, :] < T_dev[:, None]
            self.flatness = (torch.where(mask, flat, 0.0).sum(1) / T_dev).cpu().numpy()
        else:
            self.flatness = np.full(S, np.nan)
        self.keep = self.flatness <= self.flatness_threshold
        # -- durations and the column range of the whole-song maxima (:271-282)
        self.song_dur = song_durations(self.T, lens, self.sr)
        self.ref_cols = np.where(lens > 0, seconds_to_frames(self.song_dur, self.T, lens, self.sr), 0)
        # -- songs the class refuses: an empty buffer, or a length one of the CQTs rejects (librosa ParameterError)
        self.valid = lens > 0
        for plan in self.cqt_plans:
            for s in np.flatnonzero(self.valid):
                try:
                    plan.check_length(int(lens[s]))
                except ParameterError:
                    self.valid[s] = False
        # -- ref_C (:271-282): the three CQT peaks over columns [0, ref_cols); refused songs take no part
        lens_c = np.where(self.valid, lens, 0)
        lo = np.zeros(S, dtype=np.int32)
        hi = np.where(self.valid, self.ref_cols, 0).astype(np.int32)
        if self.hold == "stft":
            peaks = [ops.cqt_peak_batch(wav, plan, lo, hi, lens=lens_c) for plan in self.cqt_plans]
        else:
            # groups of songs of about chunk_bytes of samples: the CQT workspace scales with the songs of a call and
            # would otherwise match the waveforms in size.  A clip's peak does not depend on the other clips of its call.
            g = max(1, self.chunk_bytes // (4 * wav.shape[1]))
            peaks = [torch.cat([ops.cqt_peak_batch(wav[s:s + g], plan, lo[s:s + g], hi[s:s + g], lens=lens_c[s:s + g])
                                for s in range(0, S, g)]) for plan in self.cqt_plans]
        self.ref_C = torch.stack(peaks, dim=1).double().cpu().numpy()
        self.ref_C[~self.valid] = np.nan
        return self

    def _song_frames_walk(self, T_max):
        """hold="waveform" setup: the song STFT in chunks of frames, magnitudes only, through one reused buffer.
        Returns ref_mag [S] (the maximum accumulates over the chunks) and the per-frame flatness [S, T_max] float32.
        Both are per-frame quantities, so they equal hold="stft"'s bit for bit; the masked mean then runs once over
        the whole table, in hold="stft"'s summation order."""
        S = self.wav.shape[0]
        ref = torch.zeros(S, device=self.dev, dtype=torch.float32)
        if T_max == 0:
            return ref, None
        P = ops.frame_pitch(self.nb)
        ch = max(1, min(T_max, self.chunk_bytes // (4 * P * S)))
        buf = torch.empty(S * ch * P, device=self.dev, dtype=torch.float32)
        flat = torch.empty((S, T_max), device=self.dev, dtype=torch.float32)
        for c0 in range(0, T_max, ch):
            n = min(ch, T_max - c0)
            m = buf[:S * n * P].view(S, n, P)
            ops.stft_rows_batch(self.wav, self.stft, c0, n, lens=self.lens, out=m, clip_max=ref)
            flat[:, c0:c0 + n] = ops.spectral_flatness_batch(m, self.nb)
        return ref, flat

    def _section_rows(self, song_idx, tfs, n_frames):
        """Rows tfs .. tfs + n_frames - 1 of songs song_idx, zero past each song's end: [n, n_frames, P] mag / phase."""
        if self.hold == "waveform":
            r = ops.stft_rows_batch(self.wav, self.stft, tfs, n_frames, lens=self.lens, clip_rows=song_idx, phase_out=True)
            return r["mag_storage"], r["phase_storage"]
        T = self.T[song_idx]
        T_max = self.mag.shape[1]
        sel = torch.as_tensor(song_idx, device=self.dev)
        # frame rows tfs .. tfs + n_frames - 1, zero where they are past the song's end
        rows = torch.as_tensor(tfs, device=self.dev)[:, None] + torch.arange(int(n_frames), device=self.dev)[None, :]
        live = rows < torch.as_tensor(T, device=self.dev)[:, None]
        rows_c = rows.clamp(max=max(T_max - 1, 0))
        mag = torch.where(live[..., None], self.mag[sel[:, None], rows_c], 0.0)
        phase = torch.where(live[..., None], self.phase[sel[:, None], rows_c], torch.zeros((), dtype=self.phase.dtype,
                                                                                           device=self.dev))
        return mag.contiguous(), phase.contiguous()

    def _section_wav(self, song_idx, g):
        """Samples [w0, w0 + n_copy) of songs song_idx, then zeros up to wav_len: [n, max(wav_len)]."""
        sel = torch.as_tensor(song_idx, device=self.dev)
        Lw = max(int(g["wav_len"].max(initial=0)), 1)
        idx = torch.as_tensor(g["w0"], device=self.dev)[:, None] + torch.arange(Lw, device=self.dev)[None, :]
        take = torch.arange(Lw, device=self.dev)[None, :] < torch.as_tensor(g["n_copy"], device=self.dev)[:, None]
        return torch.where(take, self.wav[sel[:, None], idx.clamp(0, self.wav.shape[1] - 1)], 0.0)

    def section(self, song_idx, offset_s, n_frames=258):
        """`mid_wf.section(offset, None, n_frames)` (training.py:284, util_audio.py:286-328) of song song_idx[w] at
        offset_s[w] seconds, for W windows.  Returns SongWindows."""
        song_idx = np.asarray(song_idx, dtype=np.int64).reshape(-1)
        offset_s = np.broadcast_to(np.asarray(offset_s, dtype=np.float64), song_idx.shape)
        if (song_idx < 0).any() or (song_idx >= len(self.lens)).any():
            raise ValueError("song index out of range")
        if not self.valid[song_idx].all():
            raise ValueError("windows of songs that are not valid (empty or refused by the CQT)")
        if (offset_s < 0).any():
            raise ValueError("offsets must be >= 0")
        T, lens = self.T[song_idx], self.lens[song_idx]
        g = section_geometry(T, lens, offset_s, n_frames, self.sr)
        g["song_idx"] = song_idx
        mag, phase = self._section_rows(song_idx, g["tfs"], n_frames)
        return SongWindows(mag, phase, self._section_wav(song_idx, g), song_idx, g, offset_s)

    def load_into(self, step, windows):
        """NoteStepBatch.load with each window's song normalisers: song_ref_mag and ref_C.  window_ref_mag stays None:
        `section` (training.py:284) runs before the song's ref_mag is first evaluated (:336).  Windows may have
        waveforms of different lengths (songs of different len / T ratios)."""
        idx = windows.song_idx
        step.load(windows.mag, windows.phase, windows.wav,
                  self.ref_mag.index_select(0, torch.as_tensor(idx, device=self.dev)), self.ref_C[idx],
                  wav_lens=windows.wav_len)
        return step

    def slide(self, step, windows, mask, half_seconds=3.0):
        """training.py:317-328 for the windows where `mask` is set, on the state `load_into` gave `step`:
            offset += half_seconds
            new = mid_wf.section(offset + half_seconds, None, h)      # h = T // 2 rows of the song
            audio_w.slice(h, 2h); audio_w.concat(new)
        Rows: one slide-kernel launch for all masked windows (under hold="waveform" the kernel only moves the rows down,
        and one frame-range STFT of the songs writes the new halves).  Waveforms: a window that holds one (no subtraction since
        it was loaded or last slid, or `step.wf()` was read since) keeps `wf[a:b]` plus the new half's samples, a
        ragged length; any other window is inverted whole by the next step.  Updates windows.offset_s, the geometry and
        wav_len of the slid windows.  Calling it twice before a step slides twice, as the loop does.
        Returns a bool mask [W] of the windows whose new half starts past the song's end (tfs > T_song): the class
        then appends tfe - T_song > h zero columns ((sic) util_audio.py:318-321), a window this batch cannot hold.
        Their rows are zero-filled as `section` does, and from there on they differ from the class's."""
        W, T = step.W, step.T
        if T % 2:
            raise ValueError("slice(h, 2h) + concat of an odd T = %d leaves T - 1 frames" % T)
        self._check_step(step)
        mask = np.asarray(mask, dtype=bool).reshape(-1)
        if mask.shape != (W,) or len(windows.song_idx) != W:
            raise ValueError("mask must be [W], one entry per window of the batch")
        past = np.zeros(W, dtype=bool)
        m = np.flatnonzero(mask)
        if not len(m):
            return past
        sidx = windows.song_idx[m]
        has_wf = (step.state[m] == step.AUDIO) | (step.state[m] == step.SYNCED)
        g = slide_geometry(T, step.wav_lens[m], has_wf, self.T[sidx], self.lens[sidx], windows.offset_s[m], half_seconds,
                           self.sr, self.hl)
        step._apply_slide(m, sidx, g, self.mag, self.phase, self.wav, song_lens=self.lens)
        windows.offset_s[m] = g["offset_s"]
        windows.wav_len = windows.geometry["wav_len"] = step.wav_lens.copy()
        for k in ("tfs", "tfe", "w0", "w1", "n_copy", "pad"):
            windows.geometry[k][m] = g[k]
        past[m] = g["past_end"]
        return past

    def _check_step(self, step):
        if step.hl != self.hl or step.sr != self.sr:
            raise ValueError("the step and the songs must share hop and sample rate")
        if self.hold == "waveform" and step.N != self.N:
            raise ValueError("the step and the songs must share n_fft")

    def refill(self, step, windows, slots, song_idx, offset_s=0.0):
        """Slot slots[i] of the batch `load_into` gave `step` now holds `section(song_idx[i], offset_s[i], step.T)`:
        exactly what `section` + `load_into` give a fresh batch -- rows, waveform, song normalisers, the window's own
        maximum as the first subtraction's ref_mag, state AUDIO -- while every other slot is left as it was, bit for
        bit.  For a walk over more songs than slots: a slot whose song's notes are done, or whose slide went past the
        song's end, takes the next song.  Updates windows.song_idx, offset_s, the geometry and wav_len of those slots.
        Rows: one frame-range STFT straight into step.mag / step.ph (hold="waveform"), or a gather from the song STFT
        (hold="stft")."""
        slots = np.asarray(slots, dtype=np.int64).reshape(-1)
        song_idx = np.asarray(song_idx, dtype=np.int64).reshape(-1)
        offset_s = np.broadcast_to(np.asarray(offset_s, dtype=np.float64), song_idx.shape).copy()
        if slots.shape != song_idx.shape:
            raise ValueError("one song per refilled slot")
        if ((slots < 0) | (slots >= step.W)).any() or len(np.unique(slots)) != len(slots):
            raise ValueError("slots must be distinct indices in [0, %d)" % step.W)
        if ((song_idx < 0) | (song_idx >= len(self.lens))).any():
            raise ValueError("song index out of range")
        if not self.valid[song_idx].all():
            raise ValueError("songs that are not valid (empty or refused by the CQT)")
        if (offset_s < 0).any():
            raise ValueError("offsets must be >= 0")
        if len(windows.song_idx) != step.W:
            raise ValueError("windows must be the batch's, one entry per slot")
        self._check_step(step)
        if not len(slots):
            return
        g = section_geometry(self.T[song_idx], self.lens[song_idx], offset_s, step.T, self.sr)
        if self.hold == "waveform":
            ops.stft_rows_batch(self.wav, self.stft, g["tfs"], step.T, lens=self.lens, clip_rows=song_idx, out=step.mag,
                                phase_out=step.ph, dst_clip=slots)
        else:
            mag, phase = self._section_rows(song_idx, g["tfs"], step.T)
            sl = torch.as_tensor(slots, device=self.dev)
            step.mag.index_copy_(0, sl, mag)
            step.ph.index_copy_(0, sl, phase)
        step._apply_refill(slots, self._section_wav(song_idx, g), g["wav_len"],
                           self.ref_mag.index_select(0, torch.as_tensor(song_idx, device=self.dev)), self.ref_C[song_idx])
        windows.song_idx = windows.song_idx.copy()
        windows.song_idx[slots] = song_idx
        windows.geometry["song_idx"] = windows.song_idx
        windows.offset_s[slots] = offset_s
        for k in ("tfs", "tfe", "w0", "w1", "n_copy", "pad"):
            windows.geometry[k][slots] = g[k]
        windows.wav_len = windows.geometry["wav_len"] = step.wav_lens.copy()
