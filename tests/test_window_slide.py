"""Half-window slides and windows of different lengths in the batched per-note step (SongBatch.slide,
NoteStepBatch's per-window state, saga_window_slide_exec / ops.window_slide_batch).

* no GPU: the slide's float64 geometry against the oracle container (bit-identical to the reference's class) over
  about 200 song lengths and chains of slides, with and without a subtraction before them; the C entry's argument
  checks; odd window lengths refused;
* GPU: the kernel against a torch gather; the golden FULL song (notes 0 and 1, a slide, note 2) in a batch with two
  other songs; eight songs walked through steps and slides against the CUDA class; ragged windows without slides.
"""
import ctypes as C
import os

import numpy as np
import pytest

import amt_saga_b200  # noqa: F401
from amt_saga_b200 import _lib
from amt_saga_b200 import song_setup as ss
from oracle.audio_oracle import AudioOracle
from tests import ref_loop as L
from tests.golden.make_ref_class_golden import FULL, FULL_COLS, NOTE_STEPS
from tests.synth import piano_clip
from tests.test_song_setup import _lengths

GOLD = os.path.join(os.path.dirname(__file__), "golden")
MAG_TOL = 1e-4
SR, N, HOP, T, H = 44100, 4096, 1024, 258, 129


# --------------------------------------------------------------------------- no GPU
def _oracle_slide(song, win, offset):
    """tests/ref_loop.py:98-102."""
    offset += 3.0
    new = song.section(offset + 3.0, None, H)
    win.slice(H, 2 * H)
    win.concat(new)
    return offset


def test_slide_geometry_equals_the_class_over_song_lengths_and_chains():
    lens = [n for n in _lengths() if n >= 2 * HOP]
    assert len(lens) >= 180
    rng = np.random.default_rng(5)
    for n in lens:
        wf = (np.arange(n, dtype=np.float64) % 991 + 1.0).astype(np.float32)
        song = AudioOracle(wf, N)
        song.mag
        Ts = song.shape[1]
        dur = n / SR
        starts = sorted({0.0, float(rng.uniform(0, dur)), max(dur - 6.0, 0.0), max(dur - 3.0, 0.0), dur + 1.0})
        for subtracted in (False, True):
            for off0 in starts:
                win = song.section(off0, None, T)
                if win.shape[1] != T:            # starts past the song's end: SongBatch.section's case, not a slide's
                    continue
                if subtracted:
                    win.mag = win.mag            # what a subtraction does to the window's waveform: `_wf` dropped
                wl = len(win._v["wf"]) if win._v["wf"] is not None else HOP * (T - 1)
                off = off0
                for k in range(3):               # chains of one, two and three slides
                    has_wf = win._v["wf"] is not None
                    g = ss.slide_geometry(T, [wl], [has_wf], [Ts], [n], [off], 3.0, SR, HOP)
                    if has_wf:
                        wlen = len(win._v["wf"])
                        assert g["a"][0] == min(int(win._frames_to_seconds(H) * SR), wlen)
                        assert g["b"][0] == min(int(win._frames_to_seconds(2 * H) * SR), wlen)
                    off = _oracle_slide(song, win, off)
                    assert g["offset_s"][0] == off
                    assert g["tfs"][0] == song._seconds_to_frames(off + 3.0)
                    assert bool(g["past_end"][0]) == (win.shape[1] > T), (n, off0, k)
                    if win.shape[1] > T:
                        break                    # the batch cannot hold that window: it is reported, not continued
                    got = win._v["wf"]
                    assert (got is not None) == has_wf
                    wl = len(got) if got is not None else HOP * (T - 1)
                    assert g["wav_len"][0] == wl, (n, off0, subtracted, k)
                    if got is not None:
                        nc, kp = int(g["n_copy"][0]), int(g["keep"][0])
                        assert np.array_equal(got[kp:kp + nc], wf[g["w0"][0]:g["w0"][0] + nc])
                        assert not got[kp + nc:].any()


def test_odd_window_length_is_refused():
    with pytest.raises(ValueError):
        ss.slide_geometry(257, [1000], [True], [300], [300000], [0.0], 3.0, SR, HOP)


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__
    __graft_entry__.build()
    return _lib.lib()


def test_slide_entry_argument_errors_do_not_need_a_device(lib):
    one = C.c_void_p(256)                 # never dereferenced: the checks come first
    P = 2052

    def call(mag=one, phase=one, n_windows=4, n_frames=T, half=H, n_bins=2049, pitch=P, stride=T * P, lst=one, n_list=2,
             song_mag=one, song_phase=one, song_stride=300 * P):
        return lib.saga_window_slide_exec(mag, phase, n_windows, n_frames, half, n_bins, pitch, stride, lst, lst, lst,
                                          lst, n_list, song_mag, song_phase, song_stride, None)

    for k in ("mag", "phase", "lst", "song_mag", "song_phase"):
        assert call(**{k: None}) == _lib.SAGA_ERR_INVALID
        assert b"null argument" in lib.saga_last_error_string()
    for kw, word in ((dict(half=0), b"half"), (dict(half=130), b"half"), (dict(n_bins=2053), b"n_bins"),
                     (dict(pitch=2050, stride=T * 2050), b"multiple of 4"), (dict(n_list=-1), b"negative"),
                     (dict(n_windows=-1), b"negative"), (dict(n_list=5), b"more listed"),
                     (dict(stride=T * P - 4), b"stride"), (dict(mag=C.c_void_p(260)), b"aligned")):
        assert call(**kw) == _lib.SAGA_ERR_INVALID, kw
        assert word in lib.saga_last_error_string(), (kw, lib.saga_last_error_string())
    assert call(n_list=0) == _lib.SAGA_OK           # nothing listed: nothing launched


# --------------------------------------------------------------------------- GPU
def _cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


@pytest.mark.gpu
def test_slide_kernel_equals_a_torch_gather():
    torch = _cuda()
    from amt_saga_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(3)
    W, S, Ts, nb, P = 9, 4, 300, 2049, 2060           # P > n_bins + 3: whole padding chunks too
    mag = torch.rand((W, T, P), device="cuda", generator=g)
    ph = torch.complex(torch.rand((W, T, P), device="cuda", generator=g), torch.rand((W, T, P), device="cuda", generator=g))
    mag[..., nb:] = 0
    ph[..., nb:] = 0
    smag = torch.rand((S, Ts, P), device="cuda", generator=g)
    sph = torch.complex(torch.rand((S, Ts, P), device="cuda", generator=g), torch.rand((S, Ts, P), device="cuda", generator=g))
    smag[..., nb:] = 0
    sph[..., nb:] = 0
    win = np.array([7, 0, 3, 4, 8])
    sidx = np.array([1, 3, 0, 1, 2])
    row0 = np.array([10, 200, 0, 250, 290])
    rows = np.clip(Ts - row0, 0, H)                   # windows 0, 3 and 4 run out of song rows partway
    rows[2] = 0                                       # a new half past the song's end: all zero
    assert (rows < H).sum() == 4
    want_m, want_p = mag.clone(), ph.clone()
    for i, w in enumerate(win):
        want_m[w, :H], want_p[w, :H] = mag[w, H:2 * H], ph[w, H:2 * H]
        want_m[w, H:2 * H], want_p[w, H:2 * H] = 0, 0
        r = int(rows[i])
        want_m[w, H:H + r], want_p[w, H:H + r] = smag[sidx[i], row0[i]:row0[i] + r], sph[sidx[i], row0[i]:row0[i] + r]
    ops.window_slide_batch(mag, ph, nb, H, win, sidx, row0, rows, smag, sph)
    assert torch.equal(mag, want_m) and torch.equal(ph, want_p)
    assert not mag[..., nb:].any() and not ph[..., nb:].any()
    with pytest.raises(ValueError):
        ops.window_slide_batch(mag, ph, nb, H, [1, 1], [0, 0], [0, 0], [H, H], smag, sph)   # repeated window


def _stack_guesses(torch, clips):
    lens = np.array([len(c) for c in clips])
    g = np.zeros((len(clips), lens.max()), dtype=np.float32)
    for w, c in enumerate(clips):
        g[w, :len(c)] = c
    return torch.as_tensor(g, device="cuda"), lens


NAMES = {"C_timing": "C_timing", "C_sw_pitch": "C_sw_pitch", "C_sw_inst": "C_sw_inst", "F_sw_inst_foc": "F_foc",
         "F_sw_inst_foc_log10": "F_foc_log10", "F_sw_inst_foc_const": "F_const",
         "F_sw_inst_foc_const_log10": "F_const_log10", "C_sw_inst_foc": "C_foc", "C_sw_inst_foc_const": "C_foc_const",
         "C_velocity": "C_velocity"}


def _check_features(out, w, ref, peak, key=""):
    """The tolerances of test_note_step.py: 1e-4 of peak, the log10 formula, phasors 2e-3 on strong bins."""
    for mine, theirs in NAMES.items():
        v, r = out[mine][w].cpu().numpy(), ref[theirs]
        assert v.shape == r.shape, (key, mine, v.shape, r.shape)
        if theirs.endswith("_log10"):
            src = ref[theirs.replace("_log10", "")].astype(np.float64) * peak
            tol = MAG_TOL * peak * 1000 / (np.log(10) * (1000 * src + 1)) / np.log10(1000 * src.max() + 1) + 1e-6
            assert (np.abs(v - r) <= tol).all(), (key, mine)
        else:
            assert np.abs(v - r).max() <= MAG_TOL * np.abs(r).max(), (key, mine, float(np.abs(v - r).max()))
    m, lo = ref["sw_mag"], int(ref["fft_bin_min"])
    strong = np.zeros(ref["ph"].shape, dtype=bool)
    rows = min(strong.shape[0], m.shape[0] - lo)
    strong[:rows] = m[lo:lo + rows] > 1e-3 * m.max()
    d = np.abs(np.exp(1j * (out["ph"][w].cpu().numpy() * 6.3 - 3.15)) - np.exp(1j * (ref["ph"] * 6.3 - 3.15)))
    assert d[strong].max() <= 2e-3, key


@pytest.mark.gpu
def test_golden_full_song_through_steps_and_a_slide_in_a_mixed_batch():
    """ref_class_loop_full.npz: the FULL song (10 s) with notes 0 and 1, a slide, note 2, as tests/ref_loop.py drives
    the reference's class -- which reads `ref_mag` and `wf` after every subtraction, so the slide keeps the cached
    ref_mag and cuts the rebuilt waveform: `ref_mag()` and `wf()` do the same here.  Two other songs of other lengths
    share the batch."""
    torch = _cuda()
    from amt_saga_b200.note_step import NoteStepBatch
    gold = dict(np.load(os.path.join(GOLD, "ref_class_loop_full.npz")))
    song, clips = L.make_inputs(FULL["seed"], FULL["seconds"], FULL["notes"])
    others = [piano_clip(31, int(SR * 13.3), n_notes=50), piano_clip(32, int(SR * 8.7), n_notes=30)]
    b = ss.SongBatch().setup([song] + others)
    win = b.section([0, 1, 2], [0.0, 0.0, 0.0], T)
    assert len(set(win.wav_len.tolist())) == 3
    step = b.load_into(NoteStepBatch(3), win)
    peak = float(gold["song_ref_mag"])
    assert abs(float(b.ref_mag[0]) - peak) <= 2e-5 * peak
    for n, (onset, dur, pitch) in enumerate(FULL["notes"]):
        key = "n%d_" % n
        if n == FULL["slide_after"]:
            past = b.slide(step, win, [True, True, True])
            assert not past.any()
            assert np.array_equal(np.array([step.nb, step.T]), gold[key + "slid_shape"])
        guess, glens = _stack_guesses(torch, [clips[n]] * 3)
        out = step.step([onset] * 3, [dur] * 3, [pitch] * 3, guess, guess_lens=glens)
        assert out["valid"].all()
        assert out["offset_frames"][0] == gold[key + "off_frames"]
        _check_features(out, 0, {k[len(key):]: v for k, v in gold.items() if k.startswith(key)}, peak, key)
        ref = step.ref_mag()                     # ref_loop.py:146 and :147 read both after the subtraction
        _, wl = step.wf()
        assert wl[0] == gold[key + "wf_len_after"]
        mag_after = step.mag[0, :, :2049].T.cpu().numpy()
        assert np.abs(mag_after[:, FULL_COLS] - gold[key + "mag_after__cols"]).max() <= MAG_TOL * peak
        assert np.abs(mag_after.sum(axis=0, dtype=np.float64) - gold[key + "mag_after__colsum"]).max() \
            <= 1e-4 * gold[key + "mag_after__colsum"].max()
        assert abs(float(ref[0]) - float(gold[key + "ref_after"])) <= 2e-5 * float(gold[key + "ref_after"])


# ---- the CUDA class driven per window in the loop's order (training.py:317-449, no reads between the steps)
def _class_step(ua, aw, onset, dur, pitch, clip, song_ref, ref_C):
    """tests/ref_loop.py:104-144 on one window of the CUDA class, returning what the batched step returns.  Nothing
    reads `wf` or `ref_mag` after the subtraction (training.py does not), so the class state is training.py's."""
    AC = ua.audio_complete
    r = {}
    ct = AC.compress_bands(aw.mag, bands=20)
    r["C_timing"] = L.host(AC._resize(ct, T)) / song_ref
    sw = aw.resize(onset, dur, 8, attribs=["mag", "ph"])
    r["sw_mag"] = L.host(sw.mag)
    r["C_sw_pitch"] = L.host(aw.slice_C(onset, dur, 8, bins_per_tone=2)) / ref_C[0]
    r["C_sw_inst"] = L.host(aw.slice_C(onset, dur, 8, bins_per_tone=4)) / ref_C[1]
    lo_c = aw.midi_tone_to_FFT(60)
    fc = L.host(sw.section_power("mag", lo_c, lo_c + 348))
    r["F_const"] = fc / song_ref
    r["F_const_log10"] = np.log10(fc * 1000 + 1) / np.max(np.log10(fc * 1000 + 1))
    lo = aw.midi_tone_to_FFT(pitch)
    r["fft_bin_min"] = lo
    ff = L.host(sw.section_power("mag", lo, lo + 348))
    r["F_foc"] = ff / song_ref
    r["F_foc_log10"] = np.log10(ff * 1000 + 1) / np.max(np.log10(ff * 1000 + 1))
    r["ph"] = (np.angle(L.host(sw.section_power("ph", lo, lo + 348))) + 3.15) / 6.3
    r["C_foc"] = L.host(aw.slice_C(onset, dur, 8, bins_per_tone=16, highest_note=None, nbins=348,
                                   lowest_note=L.midi_to_note(pitch))) / ref_C[2]
    r["C_foc_const"] = L.host(aw.slice_C(onset, dur, 8, bins_per_tone=16, highest_note=None, nbins=348,
                                         lowest_note=L.midi_to_note(60))) / ref_C[2]
    r["C_velocity"] = L.host(aw.slice_C(onset, dur, 8, bins_per_tone=2, highest_note=None, nbins=36,
                                        lowest_note=L.midi_to_note(pitch - 10))) / ref_C[2]
    r["wav_len"] = int(aw._wf.shape[0])            # the waveform slice_C used (materialised by it)
    r["off_frames"] = aw._seconds_to_frames(onset)
    aw.subtract(AC(clip, N), offset=onset)
    return r


# (seconds, slides before each of four notes): two slides before the first note (audio slides, ragged lengths); a slide
# after two subtractions; a new half overhanging the song's end (the waveform grows, sic); a new half past the end
# (flagged); never; alternating; audio then stale; two stale slides in a row
WALK = [(12.0, (2, 0, 0, 0)), (20.0, (0, 0, 1, 0)), (8.5, (1, 0, 0, 0)), (8.0, (1, 1, 0, 0)), (30.0, (0, 0, 0, 0)),
        (40.0, (0, 1, 0, 1)), (15.0, (1, 0, 1, 0)), (25.0, (0, 0, 2, 0))]


@pytest.mark.gpu
def test_song_walk_against_the_cuda_class():
    torch = _cuda()
    from amt_saga_b200 import util_audio as ua
    from amt_saga_b200.note_step import NoteStepBatch
    W = len(WALK)
    rng = np.random.default_rng(17)
    songs = [piano_clip(600 + w, int(SR * sec), n_notes=int(4 * sec)) for w, (sec, _) in enumerate(WALK)]
    notes = [[(float(rng.uniform(0.05, 5.0)), float(rng.uniform(0.3, 1.0)), int(rng.integers(40, 80))) for _ in range(4)]
             for _ in range(W)]
    clips = [[piano_clip(700 + 10 * w + k, int(SR * (notes[w][k][1] + 0.3)), n_notes=1,
                         pitch_range=(notes[w][k][2], notes[w][k][2])) for k in range(4)] for w in range(W)]
    b = ss.SongBatch().setup(songs)
    win = b.section(np.arange(W), np.zeros(W), T)
    step = b.load_into(NoteStepBatch(W), win)
    song_ref = b.ref_mag.double().cpu().numpy()
    mids = [ua.audio_complete(s, N) for s in songs]
    for m in mids:
        m.mag
    aws = [m.section(0, None, T) for m in mids]
    offs = [0.0] * W
    gone = np.zeros(W, dtype=bool)                     # flagged: the class's window has more than T columns
    for k in range(4):
        for rep in range(2):
            mask = np.array([WALK[w][1][k] > rep for w in range(W)])
            if not mask.any():
                continue
            past = b.slide(step, win, mask)
            for w in np.flatnonzero(mask):
                offs[w] = _oracle_slide(mids[w], aws[w], offs[w])
                assert bool(past[w]) == (aws[w].shape[1] > T), (w, k)
                assert win.offset_s[w] == offs[w]
            gone |= past
        assert gone.tolist() == [False, False, False, k >= 1, False, False, False, False]
        guess, glens = _stack_guesses(torch, [clips[w][k] for w in range(W)])
        nk = [notes[w][k] for w in range(W)]
        out = step.step([x[0] for x in nk], [x[1] for x in nk], [x[2] for x in nk], guess, guess_lens=glens)
        lens_used = step.wav_lens.copy()
        for w in np.flatnonzero(~gone):
            key = "w%d step %d" % (w, k)
            r = _class_step(ua, aws[w], *nk[w], clips[w][k], float(song_ref[w]), b.ref_C[w])
            assert out["valid"][w]
            assert out["offset_frames"][w] == r["off_frames"], key
            assert lens_used[w] == r["wav_len"], key
            _check_features(out, w, r, float(song_ref[w]), key)
            mine = step.mag[w, :, :2049]
            theirs = aws[w]._mag.st[:, :2049]
            assert float((mine - theirs).abs().max()) <= MAG_TOL * float(song_ref[w]), key
            assert abs(float(step.ref[w]) - float(aws[w]._max_hint.reshape(-1)[0])) <= 2e-5 * float(step.ref[w]), key


@pytest.mark.gpu
def test_ragged_windows_without_slides_against_the_cuda_class():
    """Windows of songs of different lengths at offset 0 through load_into (one wav length was required before)."""
    torch = _cuda()
    from amt_saga_b200 import util_audio as ua
    from amt_saga_b200.note_step import NoteStepBatch
    secs = [60.0, 60.02, 61.0, 18.3]
    songs = [piano_clip(900 + i, int(SR * s), n_notes=40) for i, s in enumerate(secs)]
    W = len(songs)
    b = ss.SongBatch().setup(songs)
    win = b.section(np.arange(W), np.zeros(W), T)
    assert len(set(win.wav_len.tolist())) == W
    step = b.load_into(NoteStepBatch(W), win)
    song_ref = b.ref_mag.double().cpu().numpy()
    aws = []
    for s in songs:
        m = ua.audio_complete(s, N)
        m.mag
        aws.append(m.section(0, None, T))
    notes = [[(0.4, 0.5, 45), (2.0, 0.8, 60), (4.4, 0.6, 70), (5.5, 0.4, 52)],
             [(3.3, 0.9, 76), (0.1, 0.5, 33), (1.5, 1.0, 64), (2.9, 0.7, 58)]]
    for k in range(2):
        clips = [piano_clip(950 + 10 * k + w, int(SR * (notes[k][w][1] + 0.3)), n_notes=1,
                            pitch_range=(notes[k][w][2], notes[k][w][2])) for w in range(W)]
        guess, glens = _stack_guesses(torch, clips)
        nk = notes[k]
        out = step.step([x[0] for x in nk], [x[1] for x in nk], [x[2] for x in nk], guess, guess_lens=glens)
        lens_used = step.wav_lens.copy()
        for w in range(W):
            r = _class_step(ua, aws[w], *nk[w], clips[w], float(song_ref[w]), b.ref_C[w])
            assert out["offset_frames"][w] == r["off_frames"] and lens_used[w] == r["wav_len"], (w, k)
            _check_features(out, w, r, float(song_ref[w]), (w, k))
            assert float((step.mag[w, :, :2049] - aws[w]._mag.st[:, :2049]).abs().max()) <= MAG_TOL * float(song_ref[w])
