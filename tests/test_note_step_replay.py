"""The batched per-note step (`NoteStepBatch.step`) over every key of the piano and at the benchmark's batch size, each
window of each step against a float64 replay of that step (tests/step_replay.py), and the K5 feature entries at their
edges against float64.

* 88 keys: 178 windows of 12 songs through three steps, with `wf()` and a slide of a quarter of the windows between the
  first two, so that the steps see audio, synced, incrementally patched and fully rebuilt waveforms of ragged lengths.
  Onsets on frame 0, T - 1 and T and zero durations; pitches 116 and 127, whose 348-bin / 192-per-octave plan librosa
  refuses; the 12-pitch geometry run 93..104 of that plan, which takes two contraction launches.
* the same run alone (12 windows): split-K and two launches together;
* refused pitches: NaN exactly in their refused outputs, and the other windows as in a batch without them;
* the benchmark's shape: 600 windows of 264168 samples over pitches 21..108, one step, a sample of windows replayed.
"""
import math

import numpy as np
import pytest

import amt_saga_b200  # noqa: F401
from tests import step_replay as R

SR, N, HOP, T = 44100, 4096, 1024, 258
OUT_NAMES = R.NAMES + ("ph",)


def _cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _onset_at_frame(k, wav_len):
    """An onset (seconds) that `_seconds_to_frames` maps to frame k of a window of wav_len samples."""
    return (k + 0.5) * wav_len / (T * SR)


def _step_lens(step):
    """The waveform length each window's next step works on (a pending rebuild makes it hop (T - 1))."""
    return np.where(step.state >= step.DIRTY, HOP * (T - 1), step.wav_lens)


def _foc_runs(pitches):
    """Pitch runs of equal 348 / 192 geometry over the distinct pitches of a batch, in the order the step walks them,
    and the plans one launch holds (64 column groups over the groups per plan)."""
    runs, prev = [], None
    for p in sorted(set(int(x) for x in pitches)):
        plan = R.cqt_plan(p, 348, 192)
        g = None if plan is None else plan.geometry()
        if g is not None and g == prev:
            runs[-1].append(p)
        elif g is not None:
            runs.append([p])
        prev = g
    plan = R.cqt_plan(93, 348, 192)
    gpp = sum(math.ceil(2 * o["n_filters"] / 128) for o in plan.octaves)
    return runs, 64 // gpp


def _run_and_replay(torch, step, onset, dur, pitch, guess, glens, windows, key, worst):
    """One step of every window, then the replay of the listed ones; the worst error ratio per output goes to
    `worst` (name -> (ratio, key, window))."""
    snap = R.snapshot(step, windows)
    out = step.step(onset, dur, pitch, guess, guess_lens=glens)
    host = {k: out[k].cpu().numpy() for k in OUT_NAMES}
    g_host = guess.cpu().numpy()
    for i, w in enumerate(windows):
        st = R.window_state(snap, i)
        ref = R.replay(st, onset[w], dur[w], int(pitch[w]), g_host[w, :int(glens[w])])
        assert bool(out["valid"][w]) == ref["valid"], (key, w, int(pitch[w]))
        assert int(out["offset_frames"][w]) == ref["offset_frames"], (key, w)
        got = {k: host[k][w] for k in OUT_NAMES}
        got["mag_after"] = step.mag[w, :, :step.nb].T.cpu().numpy()
        for name, e in R.compare(got, ref, st["song_ref"]).items():
            if name not in worst or e > worst[name][0]:
                worst[name] = (e, key, int(w))
            if e > 1:
                a, b_ = np.asarray(got[name], dtype=np.float64), ref[name]
                j = np.unravel_index(np.nanargmax(np.abs(a - b_)), a.shape)
                print("%s window %d pitch %d %s: error / tolerance %.3g; state %d, %d samples, onset frame %d, "
                      "duration %.3f s; peak %.4g (reference) %.4g (step); at %s %.4g (reference) %.4g (step)"
                      % (key, w, pitch[w], name, e, st["state"], ref["wav_len"], ref["offset_frames"], dur[w],
                         np.nanmax(np.abs(b_)), np.nanmax(np.abs(a)), j, b_[j], a[j]))
    return out


def _report(title, worst):
    print("\n%s: worst error / tolerance per output" % title)
    for name, (e, key, w) in sorted(worst.items()):
        print("  %-26s %.3e  (%s, window %d)" % (name, e, key, w))
    bad = {k: v for k, v in worst.items() if not v[0] <= 1.0}
    assert not bad, bad


# --------------------------------------------------------------------------- 88 keys
@pytest.fixture(scope="module")
def songs12():
    """12 songs of 20-90 s, set up as the producer loop does, and 178 windows over them: two per key 21..108, then
    pitches 116 and 127."""
    torch = _cuda()
    from amt_saga_b200 import synth
    from amt_saga_b200.song_setup import SongBatch
    rng = np.random.default_rng(88)
    secs = np.concatenate([[20.0, 90.0], rng.uniform(20.0, 90.0, 10)])
    lens = (secs * SR).astype(np.int64)
    wav = synth.piano_batch(range(12), int(lens.max()), SR, n_notes=160, seed_base=8800, device="cuda")
    b = SongBatch().setup(wav, lens=lens)
    assert b.valid.all()
    pitch = np.concatenate([np.repeat(np.arange(21, 109), 2), [116, 127]])
    W = len(pitch)
    song = np.arange(W) % 12
    offs = rng.uniform(0.0, secs[song] - 6.5)
    return dict(b=b, pitch=pitch, song=song, offs=offs, W=W)


def _notes(rng, step, W, edges):
    """Onsets / durations of one step: random, then the edge cases on windows `edges` (5 of them): onset on frame 0,
    on frame T - 1, on frame T (nothing left to subtract), a zero duration, and frame T - 1 with a zero duration."""
    lens = _step_lens(step)
    onset = rng.uniform(0.0, 5.8, W)
    dur = rng.uniform(0.05, 1.2, W)
    e0, e1, e2, e3, e4 = edges
    onset[e0] = 0.0
    onset[e1] = _onset_at_frame(T - 1, lens[e1])
    onset[e2] = _onset_at_frame(T, lens[e2])
    dur[e3] = 0.0
    onset[e4], dur[e4] = _onset_at_frame(T - 1, lens[e4]), 0.0
    return onset, dur


def _guesses(torch, rng, W, seed):
    from amt_saga_b200 import synth
    glens = rng.integers(int(0.2 * SR), int(1.6 * SR), W)
    guess = synth.piano_batch(range(W), int(glens.max()), SR, n_notes=1, seed_base=seed, device="cuda")
    return guess, glens


@pytest.mark.gpu
def test_all_88_keys_through_steps_and_a_slide_against_the_float64_replay(songs12):
    torch = _cuda()
    from amt_saga_b200.note_step import NoteStepBatch
    b, pitch, W = songs12["b"], songs12["pitch"], songs12["W"]
    runs, per_launch = _foc_runs(pitch)
    print("\n348/192 geometry runs over the batch's pitches: %s; %d plans per launch"
          % ([(r[0], r[-1]) for r in runs], per_launch))
    assert max(len(r) for r in runs) > per_launch          # a run that needs a second contraction launch
    win = b.section(songs12["song"], songs12["offs"], T)
    step = b.load_into(NoteStepBatch(W), win)
    rng = np.random.default_rng(881)
    worst = {}
    seen = set()
    for k in range(3):
        if k == 1:
            step.wf()                                          # the loop reads wf: a slide then cuts the waveform
            mask = rng.random(W) < 0.25
            b.slide(step, win, mask)
            assert 30 <= mask.sum() <= 60
        seen |= set(step.state.tolist())
        onset, dur = _notes(rng, step, W, edges=[5 * k + i for i in (0, 40, 80, 120, 160)])
        guess, glens = _guesses(torch, rng, W, 9000 + 1000 * k)
        out = _run_and_replay(torch, step, onset, dur, pitch, guess, glens, np.arange(W), "step %d" % k, worst)
        assert not out["valid"][-2:].any() and out["valid"][:-2].all()
    assert seen == {step.AUDIO, step.SYNCED, step.DIRTY, step.FULL}
    _report("88 keys, 3 steps x %d windows" % W, worst)


@pytest.mark.gpu
def test_a_twelve_pitch_run_alone_splits_k_over_two_launches(songs12):
    """Pitches 93..104 share one geometry of the 348 / 192 plan: 12 plans of 6 column groups, 10 per launch.  With one
    window each the first launch has 10 x 6 tiles, far fewer than the SMs, so the step splits K as well."""
    torch = _cuda()
    from amt_saga_b200.note_step import NoteStepBatch
    b = songs12["b"]
    pitch = np.arange(93, 105)
    W = len(pitch)
    runs, per_launch = _foc_runs(pitch)
    assert [len(r) for r in runs] == [12] and per_launch == 10
    win = b.section(np.arange(W), np.random.default_rng(93).uniform(0.0, 13.0, W), T)
    step = b.load_into(NoteStepBatch(W), win)
    rng = np.random.default_rng(931)
    worst = {}
    for k in range(2):
        onset, dur = rng.uniform(0.0, 5.8, W), rng.uniform(0.05, 1.2, W)
        guess, glens = _guesses(torch, rng, W, 9300 + 100 * k)
        _run_and_replay(torch, step, onset, dur, pitch, guess, glens, np.arange(W), "step %d" % k, worst)
    _report("pitches 93..104, 2 steps x %d windows" % W, worst)


@pytest.mark.gpu
def test_refused_pitches_are_nan_and_do_not_change_the_other_windows(songs12):
    """Windows at 116 and 127 (a 348 / 192 plan past Nyquist) come back invalid with NaN in exactly the outputs of the
    refused plans; every other window equals the same batch without them (to 2e-6 of its peak: a different batch can
    split K differently)."""
    torch = _cuda()
    from amt_saga_b200.note_step import NoteStepBatch
    b, pitch, W = songs12["b"], songs12["pitch"], songs12["W"]
    keep = np.arange(W - 2)
    rng = np.random.default_rng(116)
    onset, dur = rng.uniform(0.3, 5.0, W), rng.uniform(0.2, 1.0, W)
    guess, glens = _guesses(torch, rng, W, 11600)
    outs, mags = [], []
    for sel in (np.arange(W), keep):
        win = b.section(songs12["song"][sel], songs12["offs"][sel], T)
        step = b.load_into(NoteStepBatch(len(sel)), win)
        outs.append(step.step(onset[sel], dur[sel], pitch[sel], guess[sel].contiguous(), guess_lens=glens[sel]))
        mags.append(step.mag[:, :, :step.nb])
    full, part = outs
    assert not full["valid"][-2:].any() and full["valid"][:-2].all() and part["valid"].all()
    for w in (W - 2, W - 1):
        p = int(pitch[w])
        refused = {"C_sw_inst_foc": R.cqt_plan(p, 348, 192) is None, "C_velocity": R.cqt_plan(p - 10, 36, 24) is None}
        assert refused["C_sw_inst_foc"]
        for name in OUT_NAMES:
            nan = torch.isnan(full[name][w])
            assert bool(nan.all()) if refused.get(name, False) else not bool(nan.any()), (p, name)
    worst = 0.0
    keep_d = torch.as_tensor(keep, device="cuda")
    for name in OUT_NAMES:
        a, c = full[name].index_select(0, keep_d).double(), part[name].double()
        assert torch.equal(torch.isnan(a), torch.isnan(c)), name
        a, c = torch.nan_to_num(a), torch.nan_to_num(c)
        peak = c.abs().flatten(1).amax(1).clamp_min(1e-30)
        err = float(((a - c).abs().flatten(1).amax(1) / peak).max())
        worst = max(worst, err)
        assert err <= 2e-6, (name, err)
    d = float((mags[0].index_select(0, keep_d) - mags[1]).abs().max())
    assert d <= 2e-6 * float(mags[1].abs().max()), d
    print("\nrefused pitches: the other %d windows within %.2e of their peaks of the batch without them" % (W - 2, worst))


# --------------------------------------------------------------------------- the benchmark's shape
@pytest.mark.gpu
def test_bench_shape_600_windows_over_88_keys_against_the_float64_replay():
    """bench.py's `timed(21, 109)`: 600 windows of 264168 samples loaded from their own STFT, pitches drawn from
    21..108, one step.  Replayed: a seeded sample of 48 windows, the first and the last, and every window of the
    12-pitch run 93..104."""
    torch = _cuda()
    from amt_saga_b200 import ops, synth
    from amt_saga_b200.note_step import NoteStepBatch
    W, L = 600, 264168
    wav = synth.piano_batch(range(W), L, SR, seed_base=50000, device="cuda")
    plan = ops.get_stft_plan(N, HOP, True, device="cuda")
    r = ops.stft_batch(wav, plan, want_phase=True)
    step = NoteStepBatch(W)
    step.load(r["mag_storage"][:, :T].contiguous(), r["phase_storage"][:, :T].contiguous(), wav, r["clip_max"],
              np.ones((W, 3)))
    del r
    guess = synth.piano_batch(range(W), 54277, SR, n_notes=1, seed_base=90000, device="cuda")
    glens = np.full(W, 54277)
    rg = np.random.default_rng(600)
    onset, dur, pitch = rg.uniform(0, 5.0, W), rg.uniform(0.2, 1.2, W), rg.integers(21, 109, W)
    runs, per_launch = _foc_runs(pitch)
    assert max(len(r_) for r_ in runs) > per_launch
    sample = set(rg.choice(W, 48, replace=False).tolist()) | {0, W - 1} | set(np.flatnonzero((pitch >= 93) & (pitch <= 104)).tolist())
    worst = {}
    _run_and_replay(torch, step, onset, dur, pitch, guess, glens, np.array(sorted(sample)), "bench step", worst)
    _report("bench shape, %d of %d windows replayed" % (len(sample), W), worst)


# --------------------------------------------------------------------------- K5 entries at their edges
def _garbage_storage(torch, rng, W, T_, nb, P, value):
    """Frame-major [W, T_, P] float32 with random rows and `value` in the padding columns [nb, P)."""
    x = rng.random((W, T_, P)).astype(np.float32) ** 3
    x[..., nb:] = value
    return x, torch.as_tensor(x, device="cuda")


@pytest.mark.gpu
def test_compress_bands_batch_edges_against_float64():
    """An empty band (NaN, np.mean of an empty slice), 128 bands (the most the kernel takes), per-window inv_scale,
    W > 1 with garbage in the padding columns."""
    torch = _cuda()
    from amt_saga_b200 import ops
    rng = np.random.default_rng(5)
    W, T_, nb = 3, 11, 1000
    P = ops.frame_pitch(nb)
    x, xd = _garbage_storage(torch, rng, W, T_, nb, P, 1e6)
    edges = np.sort(rng.choice(np.arange(1, nb), 127, replace=False))
    edges = np.concatenate([[0], edges, [nb]]).astype(np.int64)
    edges[50] = edges[49]                                   # band 49 is empty
    inv = np.array([0.5, 2.0, 1.0 / 3.0], dtype=np.float32)
    for scale in (None, inv):
        out = ops.compress_bands_batch(xd, nb, edges, inv_scale=None if scale is None else torch.as_tensor(scale, device="cuda"))
        got = out[:, :, :128].double().cpu().numpy()
        assert not out[:, :, 128:].any()
        s = np.ones(W) if scale is None else scale.astype(np.float64)
        for b_ in range(128):
            lo, hi = edges[b_], edges[b_ + 1]
            want = (x[:, :, lo:hi].astype(np.float64).mean(axis=2) if hi > lo else np.full((W, T_), np.nan)) * s[:, None]
            if hi == lo:
                assert np.isnan(got[:, :, b_]).all()
            else:
                assert np.abs(got[:, :, b_] - want).max() <= 2e-6 * np.abs(want).max(), b_


@pytest.mark.gpu
@pytest.mark.parametrize("n_rows,n_cols", [(37, 7), (348, 8), (5, 3)])
def test_short_window_features_batch_edges_against_float64(n_rows, n_cols):
    """Per-window band_min / inv_ref tensors; band_min + n_rows past n_bins (those rows are zero, whatever the padding
    columns hold); an all-zero tile (0 / 0 = NaN in the log feature, as numpy); -1 columns; n_rows x n_cols not a
    multiple of the 256 threads."""
    torch = _cuda()
    from amt_saga_b200 import ops
    rng = np.random.default_rng(n_rows * n_cols)
    W, T_, nb = 5, 9, 2049
    P = ops.frame_pitch(nb)
    assert P > nb
    x, xd = _garbage_storage(torch, rng, W, T_, nb, P, 7.0)
    ang = rng.uniform(-np.pi, np.pi, (W, T_, P))
    ph = np.exp(1j * ang).astype(np.complex64)
    ph[..., nb:] = 3.0 + 4.0j
    phd = torch.as_tensor(ph, device="cuda")
    src = rng.integers(0, T_, (W, n_cols)).astype(np.int32)
    src[0, 0] = src[4, -1] = -1
    src[2] = -1                                              # all-zero tile
    band_min = np.array([0, nb - n_rows // 2, 17, nb - 1, 900], dtype=np.int32)
    inv_ref = np.array([1.0, 0.25, 3.0, 1e-3, 10.0], dtype=np.float32)
    r = ops.short_window_features_batch(xd, phd, src, torch.as_tensor(band_min, device="cuda"), n_rows, nb,
                                        torch.as_tensor(inv_ref, device="cuda"), want_phase=True)
    for w in range(W):
        m = np.zeros((n_rows, n_cols))
        a = np.zeros((n_rows, n_cols))
        for j in range(n_cols):
            if src[w, j] < 0:
                continue
            rows = np.arange(band_min[w], min(band_min[w] + n_rows, nb))
            m[:len(rows), j] = x[w, src[w, j], rows]
            a[:len(rows), j] = np.angle(ph[w, src[w, j], rows].astype(np.complex128))
        lin = m * float(inv_ref[w])
        with np.errstate(invalid="ignore"):
            lg = np.log10(1000 * m + 1) / np.log10(1000 * m + 1).max()
        pha = (a + 3.15) / 6.3
        g_lin, g_log, g_ph = (r[k][w].double().cpu().numpy() for k in ("lin", "log", "phase"))
        assert np.abs(g_lin - lin).max() <= 1e-6 * np.abs(lin).max(), w
        assert np.array_equal(np.isnan(g_log), np.isnan(lg)), w
        if not np.isnan(lg).any():
            assert np.abs(g_log - lg).max() <= 2e-6, w
        else:
            assert w == 2
        assert np.abs(g_ph - pha).max() <= 2e-6, w


@pytest.mark.gpu
def test_gather_frames_batch_edges_against_float64():
    """-1 columns (zeros), with and without a per-window scale; the output's padding columns written as zero."""
    torch = _cuda()
    from amt_saga_b200 import ops
    rng = np.random.default_rng(9)
    W, T_, nb, n_cols = 4, 13, 348, 8
    P = ops.frame_pitch(nb)
    x, xd = _garbage_storage(torch, rng, W, T_, nb, P, -5.0)
    src = rng.integers(-1, T_, (W, n_cols)).astype(np.int32)
    src[1] = -1
    src[3, -1] = T_ - 1
    scale = np.array([1.0, 2.0, 1.0 / 7.0, 1e3], dtype=np.float32)
    Po = ops.frame_pitch(nb)
    for sc in (None, scale):
        out = torch.full((W, n_cols, Po), float("nan"), device="cuda")
        v = ops.gather_frames_batch(xd, nb, src, None if sc is None else torch.as_tensor(sc, device="cuda"), out=out)
        got = v.cpu().numpy()
        s = np.ones(W) if sc is None else sc.astype(np.float64)
        want = np.zeros((W, nb, n_cols))
        for w in range(W):
            for j in range(n_cols):
                if src[w, j] >= 0:
                    want[w, :, j] = x[w, src[w, j], :nb].astype(np.float64) * s[w]
        assert np.array_equal(got, want.astype(np.float32))     # one float32 product: exact
        assert not out[:, :, nb:].any()


@pytest.mark.gpu
def test_spectral_flatness_batch_edges_against_float64():
    """Silent frames (every bin under amin: flatness 1), garbage in the padding columns, and ragged songs whose frames
    past their end are masked out of the mean as SongBatch.setup does."""
    torch = _cuda()
    from amt_saga_b200 import ops
    rng = np.random.default_rng(12)
    S, T_, nb = 3, 40, 2049
    P = ops.frame_pitch(nb)
    x, _ = _garbage_storage(torch, rng, S, T_, nb, P, 1e3)
    frames = np.array([T_, 17, 1])
    for s in range(S):
        x[s, frames[s]:, :nb] = 0.0
    x[0, 5] = 0.0
    x[0, 5, nb:] = 1e3
    x[1, 3, :nb] = 1e-7                                        # under amin = 1e-10 once squared
    xd = torch.as_tensor(x, device="cuda")
    amin = 1e-10
    flat = ops.spectral_flatness_batch(xd, nb, amin).double().cpu().numpy()
    p = np.maximum(amin, x[..., :nb].astype(np.float64) ** 2)
    want = np.exp(np.log(p).mean(axis=2)) / p.mean(axis=2)
    assert np.abs(flat - want).max() <= 1e-5 * np.abs(want).max()
    assert abs(flat[0, 5] - 1.0) <= 1e-6 and abs(flat[1, 3] - 1.0) <= 1e-6
    # ragged songs, one with a silent stretch: SongBatch.setup averages each over its own frames only
    from amt_saga_b200.song_setup import SongBatch
    from oracle import spectral as osp
    from tests.synth import piano_clip
    songs = [piano_clip(70, 5 * SR), piano_clip(71, 3 * SR + 517), piano_clip(72, 2 * SR)]
    songs[2][SR // 2:SR + SR // 2] = 0.0
    b = SongBatch().setup(songs)
    for y, got in zip(songs, b.flatness):
        Sm = np.abs(osp.stft(y.astype(np.float64), n_fft=N, hop_length=HOP, dtype=np.complex128))
        p = np.maximum(amin, Sm ** 2)
        want = np.mean(np.exp(np.log(p).mean(axis=0)) / p.mean(axis=0))
        assert abs(got - want) <= 1e-4, (got, want)


# --------------------------------------------------------------------------- the replay against the oracle container
def _oracle_step(aw, song_ref, onset, dur, pitch, clip):
    """tests/ref_loop.py:104-144 on the oracle container (full-window CQTs, float32 STFT / iSTFT as the reference)."""
    from oracle import cqt as ocqt
    from oracle.audio_oracle import AudioOracle
    from tests.ref_loop import midi_to_note
    r = {"C_timing": AudioOracle._resize(AudioOracle.compress_bands(aw.mag, 20), T) / song_ref}
    sw = aw.resize(onset, dur, 8, attribs=["mag", "ph"])
    lo_c, lo = aw.midi_tone_to_FFT(60), aw.midi_tone_to_FFT(pitch)
    fc, ff = sw.section_power("mag", lo_c, lo_c + 348), sw.section_power("mag", lo, lo + 348)
    r["F_sw_inst_foc_const"], r["F_sw_inst_foc_const_log10"] = fc / song_ref, R._log_feature(fc)
    r["F_sw_inst_foc"], r["F_sw_inst_foc_log10"] = ff / song_ref, R._log_feature(ff)
    r["ph"] = (np.angle(sw.section_power("ph", lo, lo + 348)) + 3.15) / 6.3
    r["sw_mag"], r["fft_bin_min"] = sw.mag, lo
    r["valid"] = True
    for name, kw in (("C_sw_pitch", dict(bins_per_tone=2)), ("C_sw_inst", dict(bins_per_tone=4)),
                     ("C_sw_inst_foc", dict(bins_per_tone=16, highest_note=None, nbins=348, lowest_note=midi_to_note(pitch))),
                     ("C_sw_inst_foc_const", dict(bins_per_tone=16, highest_note=None, nbins=348, lowest_note="C4")),
                     ("C_velocity", dict(bins_per_tone=2, highest_note=None, nbins=36, lowest_note=midi_to_note(pitch - 10)))):
        try:
            r[name] = aw.slice_C(onset, dur, 8, **kw)
        except ocqt.ParameterError:
            r[name] = np.full((kw.get("nbins") or {2: 174, 4: 348}[kw["bins_per_tone"]], 8), np.nan)
            r["valid"] = False
    r["offset_frames"] = max(aw._seconds_to_frames(onset), 0)
    aw.subtract(type(aw)(clip, N), offset=onset)
    r["mag_after"] = aw.mag
    return r


@pytest.mark.parametrize("pitch", [21, 60, 98, 116])
def test_replay_equals_the_oracle_container_over_two_steps(pitch):
    """The replay's shortcuts (CQT columns kept by `_resize` only, the subtraction level, the waveform it starts from)
    against the oracle container driven through two steps of the loop, on the CPU: the first step starts from the
    window's audio, the second from the iSTFT of the subtracted rows.  Onsets on frame 0, T - 1 and T, and a zero
    duration."""
    from oracle.audio_oracle import AudioOracle
    from tests.synth import piano_clip
    song = AudioOracle(piano_clip(40 + pitch, int(9.3 * SR), n_notes=30), N)
    song_ref = float(song.ref_mag)
    worst = 0.0
    for k, (frame, dur) in enumerate(((0, 0.6), (T - 1, 0.4), (T, 0.5), (100, 0.0))):
        aw = song.section(1.7, None, T)
        clips = [piano_clip(50 + k + 10 * i, int(0.8 * SR), n_notes=1, pitch_range=(60, 60)) for i in range(2)]
        for i, clip in enumerate(clips):
            wf = aw.wf                                     # materialises the iSTFT on the second step
            onset = _onset_at_frame(frame, len(wf)) if frame else 0.0
            st = dict(mag=aw.mag.T.astype(np.float32), ph=aw.ph.T.astype(np.complex64), wav=wf, state=0 if i == 0 else 3,
                      level=float(aw.ref_mag), song_ref=song_ref, ref_C=np.ones(3), T=T)
            got = R.replay(st, onset, dur, pitch, clip)
            want = _oracle_step(aw, song_ref, onset, dur, pitch, clip)
            key = (pitch, frame, dur, i)
            assert got["valid"] == want["valid"] == (pitch < 116), key
            assert got["offset_frames"] == want["offset_frames"] == frame, key
            assert got["wav_len"] == len(wf), key
            errs = R.compare({k_: want[k_] for k_ in OUT_NAMES + ("mag_after",)}, got, song_ref)
            # half of what the GPU step is allowed: the oracle's own iSTFT accumulates in float32, which shows in the
            # weak high bands of a subtracted window (C_sw_inst_foc at 98: 0.35)
            assert max(errs.values()) <= 0.5, (key, errs)
            worst = max(worst, max(errs.values()))
    print("\npitch %d: replay against the oracle container, worst error / tolerance %.3e" % (pitch, worst))
