"""A float64 replay of ONE `NoteStepBatch.step` for one window, from the state the step starts from (CPU only).

`snapshot(step, windows)` copies what a window's step depends on: magnitude / phase rows, waveform, what the waveform
holds (`state`), the level the next subtraction scales the guess by, and the song normalisers.  `replay(...)` then
recomputes everything the step returns for that window, in float64, from the reference's own definitions:

* frame arithmetic, `_resize` and the FFT bin of a pitch: `oracle.audio_oracle.AudioOracle` (util_audio.py:261-409);
* the waveform: the float64 iSTFT of mag x phase when the step rebuilds it (util_audio.py:88-106), else the window's;
* C_timing, F_sw_inst_foc(_const)(_log10), ph: band means and `section_power` (training.py:333-363);
* the five constant-Q outputs: the plan's decimation cascade and banks contracted in float64 (`device_model`, pinned
  against the oracle's multi-rate CQT in test_cqt_plan_host.py), only at the <= 8 columns `_resize` keeps; a plan
  librosa refuses means NaN and `valid = False`;
* the subtraction (util_audio.py:221-259): float64 STFT of the guess, scaled to the window's level, aligned, clipped,
  subtracted, ReLU.

Nothing here accumulates earlier steps, so every step of a walk is checked on its own."""
import functools

import numpy as np
from scipy.signal import fftconvolve

import amt_saga_b200  # noqa: F401
from amt_saga_b200.cqt_plan import CqtPlan, ParameterError
from oracle import spectral as osp
from oracle.audio_oracle import AudioOracle
from oracle.spectral import reflect_index

SR, N, HOP = 44100, 4096, 1024
A0, C8 = 21, 108


# ------------------------------------------------------------------------------------------ constant-Q model (float64)
def fir_decimate(x, taps, factor):
    """The device cascade's FIR decimator: zero-padded symmetric filter, every `factor`-th output, ceil(n / factor)
    outputs of which the last is zero when n is not a multiple of `factor`."""
    S = len(taps) - 1
    n_full, n_out = len(x) // factor, -(-len(x) // factor)
    h = np.concatenate([taps[:0:-1], taps]).astype(np.float64)     # symmetric: convolution == correlation
    xp = np.concatenate([np.zeros(S), np.asarray(x, dtype=np.float64), np.zeros(S + factor)])
    y = np.zeros(n_out)
    y[:n_full] = fftconvolve(xp, h, mode="valid")[:factor * n_full:factor]
    return y


class Cascade:
    """The decimated levels of one signal, shared by every plan with the same early factor (the taps of a factor are
    fixed, kaiser_fast_taps)."""

    def __init__(self, y):
        self.y = np.asarray(y, dtype=np.float64)
        self._lv = {}

    def level(self, plan, l):
        key = (plan.early_factor, l)
        if key not in self._lv:
            if l == 0:
                self._lv[key] = fir_decimate(self.y, plan.early_taps, plan.early_factor) if plan.early_factor > 1 \
                    else self.y
            else:
                self._lv[key] = fir_decimate(self.level(plan, l - 1), plan.half_taps, 2)
        return self._lv[key]


def device_model(plan, y, first=0, n_cols=None, cascade=None):
    """Complex CQT [n_bins, n_cols] of the columns [first, first + n_cols) (clipped to the transform's frames) of the
    plan's algorithm: decimate with its FIR taps, reflect-indexed strided frames of every octave's level, dense
    contraction with its banks, all in float64."""
    cascade = Cascade(y) if cascade is None else cascade
    T = plan.num_frames(len(cascade.y))
    cols = np.arange(first, T if n_cols is None else min(T, first + n_cols))
    C = np.zeros((plan.n_bins, len(cols)), dtype=np.complex128)
    for o in plan.octaves:
        sig = cascade.level(plan, o["level"])
        n = np.arange(o["n_fft"])
        idx = reflect_index(cols[:, None] * o["hop"] + n[None, :] - o["n_fft"] // 2, len(sig))
        out = sig[idx] @ o["bank"].astype(np.float64)          # [cols, 2 * n_filters]
        for f in range(o["n_filters"]):
            b = o["first_bin"] + f
            if 0 <= b < plan.n_bins:
                C[b] = out[:, 2 * f] + 1j * out[:, 2 * f + 1]
    return C


@functools.lru_cache(maxsize=None)
def cqt_plan(lowest_midi, n_bins, bins_per_octave):
    """The step's plan for a slice_C shape (filter_scale 2, util_audio.py:426), host arrays only; None when librosa
    refuses it (pass band beyond Nyquist)."""
    try:
        return CqtPlan(SR, HOP, float(osp.midi_to_hz(lowest_midi)), int(n_bins), int(bins_per_octave), filter_scale=2,
                       create_device_plan=False)
    except ParameterError:
        return None


# ------------------------------------------------------------------------------------------ state before a step
def snapshot(step, windows):
    """What `step.step` reads of windows `windows`, taken before the call: device clones of their rows and waveforms
    and host copies of the rest.  `window_state(snap, i)` gives the i-th listed window's state on the host."""
    import torch
    windows = np.asarray(windows, dtype=np.int64)
    sel = torch.as_tensor(windows, device=step.dev)
    given = step._ref_given[windows]
    ref_init = step._ref_init.index_select(0, sel).cpu().numpy()
    return dict(windows=windows, nb=step.nb, T=step.T, mag=step.mag.index_select(0, sel),
                ph=step.ph.index_select(0, sel), wav=step.wav.index_select(0, sel), wav_lens=step.wav_lens[windows].copy(),
                state=step.state[windows].copy(), ref_init=np.where(given, ref_init, -1.0),
                song_ref=step.song_ref.index_select(0, sel).cpu().numpy(),
                ref_C=np.stack([1.0 / r.index_select(0, sel).double().cpu().numpy() for r in step.inv_ref_C], axis=1))


def window_state(snap, i):
    mag = snap["mag"][i, :, :snap["nb"]].cpu().numpy()
    ref = float(snap["ref_init"][i])
    return dict(mag=mag, ph=snap["ph"][i, :, :snap["nb"]].cpu().numpy(),
                wav=snap["wav"][i, :int(snap["wav_lens"][i])].cpu().numpy(), state=int(snap["state"][i]),
                # the level the subtraction scales by: a cached ref_mag, else the window's maximum at that moment
                level=ref if ref >= 0 else float(mag.max()),
                song_ref=float(snap["song_ref"][i]), ref_C=snap["ref_C"][i], T=snap["T"])


# ------------------------------------------------------------------------------------------ one step, float64
def _waveform(st):
    if st["state"] >= 2:       # DIRTY / FULL: util_audio.py:88-106, istft(mag * ph), length hop (T - 1)
        F = st["mag"].T.astype(np.float64) * st["ph"].T.astype(np.complex128)
        return osp.istft(F, hop_length=HOP, dtype=np.float64)
    return st["wav"].astype(np.float64)


def _slice_C(oracle, casc, onset, duration, lowest_midi, n_bins, bpo, n_cols=8):
    """`audio_w.slice_C(onset, duration, n_cols, ...)` (util_audio.py:411-434) with the plan's float64 model, only at
    the columns `_resize` keeps.  None: librosa refuses the plan or the length."""
    plan = cqt_plan(lowest_midi, n_bins, bpo)
    if plan is None:
        return None
    try:
        plan.check_length(len(casc.y))
    except ParameterError:
        return None
    Tc = plan.num_frames(len(casc.y))
    s = oracle._seconds_to_frames(onset)
    t = oracle._seconds_to_frames(onset + duration)
    C = np.zeros((n_bins, Tc))
    a = min(max(s, 0), Tc)
    b = min(max(t, a), Tc, a + n_cols)           # `_resize` of C[:, s:t] reads no column past s + n_cols
    if b > a:
        C[:, a:b] = np.abs(device_model(plan, None, a, b - a, cascade=casc))
    return AudioOracle._resize(C[:, s:t], n_cols)


def _log_feature(p):
    with np.errstate(invalid="ignore", divide="ignore"):
        v = np.log10(p * 1000 + 1)
        return v / np.max(v)                      # all-zero slice: 0 / 0 = NaN, as in numpy


def replay(st, onset, duration, pitch, guess, instrument_bands=348, bins_velocity=36):
    """Everything `step` returns for one window, plus `mag_after` [bins, T] (the magnitudes after the subtraction)."""
    T = st["T"]
    y = _waveform(st)
    o = AudioOracle(y, N)
    o._v["mag"], o._v["ph"] = st["mag"].T.astype(np.float64), st["ph"].T.astype(np.complex128)
    r = {"wav_len": len(y)}
    song_ref, ref_C = st["song_ref"], st["ref_C"]
    # -- training.py:333-336
    r["C_timing"] = AudioOracle._resize(AudioOracle.compress_bands(o.mag, 20), T) / song_ref
    # -- training.py:337, :347-363
    sw = o.resize(onset, duration, 8, attribs=["mag", "ph"])
    lo_c = o.midi_tone_to_FFT(60)
    fc = sw.section_power("mag", lo_c, lo_c + instrument_bands)
    r["F_sw_inst_foc_const"], r["F_sw_inst_foc_const_log10"] = fc / song_ref, _log_feature(fc)
    lo = o.midi_tone_to_FFT(pitch)
    ff = sw.section_power("mag", lo, lo + instrument_bands)
    r["F_sw_inst_foc"], r["F_sw_inst_foc_log10"] = ff / song_ref, _log_feature(ff)
    r["ph"] = (np.angle(sw.section_power("ph", lo, lo + instrument_bands)) + 3.15) / 6.3
    r["sw_mag"], r["fft_bin_min"] = sw.mag, lo
    # -- training.py:340-346, :365-388 (filter_scale 2)
    casc = Cascade(y)
    shapes = (("C_sw_pitch", A0, (C8 - A0) * 2, 24, 0), ("C_sw_inst", A0, (C8 - A0) * 4, 48, 1),
              ("C_sw_inst_foc", pitch, instrument_bands, 192, 2), ("C_sw_inst_foc_const", 60, instrument_bands, 192, 2),
              ("C_velocity", pitch - 10, bins_velocity, 24, 2))
    valid = True
    for name, low, nbins, bpo, ref_i in shapes:
        C = _slice_C(o, casc, onset, duration, low, nbins, bpo)
        if C is None:
            valid = False
            C = np.full((nbins, 8), np.nan)
        r[name] = C / ref_C[ref_i]
    r["valid"] = valid
    # -- training.py:426 + :449: util_audio.py:221-259 with a float64 STFT of the guess
    gm = np.abs(osp.stft(np.asarray(guess, dtype=np.float64), n_fft=N, hop_length=HOP, dtype=np.complex128))
    gm *= st["level"] / gm.max()
    off = max(o._seconds_to_frames(onset), 0)
    r["offset_frames"] = off
    gm = gm[:, :max(T - off, 0)]
    pad = np.zeros((gm.shape[0], T))
    pad[:, off:off + gm.shape[1]] = gm
    r["mag_after"] = np.maximum(o.mag - pad, 0.0)
    return r


# ------------------------------------------------------------------------------------------ comparison
TOL = 1e-4
# The step transforms a float32 waveform: after a subtraction it is K4's float32 iSTFT, whose rounding (~6e-8 of the
# window's peak) puts a CQT noise floor near 1e-8 of the song's CQT peak, to which ref_C normalises.  Constant-Q outputs
# whose peak is under CQT_FLOOR are therefore held to TOL * CQT_FLOOR = 1e-7 absolute (an 8-column slice of a subtracted
# window at a high pitch can be all noise: 1e-7..1e-17 on a B200).
CQT_FLOOR = 1e-3
NAMES = ("C_timing", "C_sw_pitch", "C_sw_inst", "F_sw_inst_foc", "F_sw_inst_foc_log10", "F_sw_inst_foc_const",
         "F_sw_inst_foc_const_log10", "C_sw_inst_foc", "C_sw_inst_foc_const", "C_velocity")


def compare(got, ref, song_ref):
    """Errors of one window's step outputs `got` (host arrays, the step's layout) against `ref = replay(...)`, each over
    its tolerance (<= 1 passes): features and CQT outputs within TOL of the reference's peak (for the CQT outputs at
    least CQT_FLOOR, in units of ref_C), the log features within
    the TOL error propagated through log10, phasors within 2e-3 on bins above 1e-3 of the window's peak, the
    subtracted magnitudes within TOL * song_ref.  NaN masks must be equal (else the ratio is inf)."""
    err = {}
    for name in NAMES:
        v, r = np.asarray(got[name], dtype=np.float64), ref[name]
        if v.shape != r.shape:
            raise AssertionError("%s: shape %s, reference %s" % (name, v.shape, r.shape))
        nan = np.isnan(r)
        if not np.array_equal(np.isnan(v), nan):
            err[name] = np.inf
            continue
        if nan.all():
            err[name] = 0.0
            continue
        d = np.abs(v - r)[~nan]
        if name.endswith("_log10"):
            src = ref[name[:-len("_log10")]][~nan] * song_ref
            tol = TOL * song_ref * 1000 / (np.log(10) * (1000 * src + 1)) / np.log10(1000 * src.max() + 1) + 1e-6
            err[name] = float((d / tol).max())
        else:
            peak = np.abs(r[~nan]).max()
            if name.startswith("C_") and name != "C_timing":
                peak = max(peak, CQT_FLOOR)
            err[name] = float(d.max() / (TOL * peak)) if peak > 0 else (0.0 if d.max() == 0 else np.inf)
    m, lo = ref["sw_mag"], int(ref["fft_bin_min"])
    strong = np.zeros(ref["ph"].shape, dtype=bool)
    rows = min(strong.shape[0], m.shape[0] - lo)
    strong[:rows] = m[lo:lo + rows] > 1e-3 * m.max()
    d = np.abs(np.exp(1j * (np.asarray(got["ph"]) * 6.3 - 3.15)) - np.exp(1j * (ref["ph"] * 6.3 - 3.15)))
    err["ph"] = float(d[strong].max() / 2e-3) if strong.any() else 0.0
    err["mag_after"] = float(np.abs(np.asarray(got["mag_after"], dtype=np.float64) - ref["mag_after"]).max()
                             / (TOL * song_ref))
    return err
