"""Songs held as waveforms in the song walk: the frame-range STFT (saga_stft_rows_exec / ops.stft_rows_batch),
SongBatch(hold="waveform") and SongBatch.refill.

* no GPU: the C entry's argument checks; an unknown hold refused; refill's refusals before any device work;
* GPU: rows against the full STFT (bit for bit) over the kernel shapes, ragged and unaligned clips, frame ranges at
  the start, middle, straddling and past the end, a destination permutation; hold="waveform" against hold="stft" on
  the same songs (setup, section, the song walk of test_window_slide.py, refills); memory after setup; a corpus walk
  with refills against the CUDA class; a refill of a window with a pending incremental patch.
"""
import ctypes as C
import types

import numpy as np
import pytest

import amt_saga_b200  # noqa: F401
from amt_saga_b200 import _lib
from amt_saga_b200 import song_setup as ss
from tests.synth import piano_clip
from tests.test_song_setup import _golden_songs
from tests.test_window_slide import (MAG_TOL, WALK, _check_features, _class_step, _oracle_slide, _stack_guesses)

SR, N, HOP, T, H = 44100, 4096, 1024, 258, 129


# --------------------------------------------------------------------------- no GPU
@pytest.fixture(scope="module")
def lib():
    import __graft_entry__
    __graft_entry__.build()
    return _lib.lib()


class _PlanHead(C.Structure):
    """The leading fields of saga_stft_plan (stft_plan.cuh): the checks read n_bins = M + 1 from it."""
    _fields_ = [("n_fft", C.c_int), ("hop", C.c_int), ("center", C.c_int), ("M", C.c_int), ("pad", C.c_int * 64)]


def test_rows_entry_argument_errors_do_not_need_a_device(lib):
    plan = _PlanHead(N, HOP, 1, N // 2)
    one = C.c_void_p(256)                 # never dereferenced: the checks come first
    P = 2052

    def call(p=C.cast(C.pointer(plan), C.c_void_p), wav=one, offs=one, lens=one, n_clips=3, frame0=one, n_frames=40,
             dst=None, row0=0, out_frames=T, mag=one, pitch=P, stride=T * P):
        return lib.saga_stft_rows_exec(p, wav, offs, lens, n_clips, frame0, n_frames, dst, row0, out_frames, mag, None,
                                       pitch, stride, None, None)

    for k in ("p", "wav", "offs", "lens", "frame0", "mag"):
        assert call(**{k: None}) == _lib.SAGA_ERR_INVALID
        assert b"null argument" in lib.saga_last_error_string()
    for kw, word in ((dict(n_clips=-1), b"n_clips < 0"), (dict(n_frames=0), b"n_frames 0 <= 0"),
                     (dict(pitch=2048, stride=T * 2048), b"frame_pitch 2048 < n_bins 2049"),
                     (dict(row0=-1), b"dst_row0 -1"), (dict(row0=T - 39), b"outside the 258 output rows"),
                     (dict(stride=T * P - 1), b"out_clip_stride")):
        assert call(**kw) == _lib.SAGA_ERR_INVALID, kw
        assert word in lib.saga_last_error_string(), (kw, lib.saga_last_error_string())
    assert call(n_clips=0) == _lib.SAGA_OK        # nothing to do: nothing launched
    assert call(n_clips=0, row0=T - 40) == _lib.SAGA_OK


def test_unknown_hold_is_refused():
    with pytest.raises(ValueError, match="hold"):
        ss.SongBatch(hold="bogus")


def test_refill_refuses_bad_slots_and_songs_before_the_device():
    b = object.__new__(ss.SongBatch)      # host fields only: a refusal must not reach the device
    b.hold, b.sr, b.hl, b.N = "waveform", SR, HOP, N
    b.lens = np.array([SR * 10, SR * 12, 0])
    b.T = ss.song_frames(b.lens, HOP)
    b.valid = b.lens > 0
    step = types.SimpleNamespace(W=4, T=T, hl=HOP, sr=SR, N=N)
    win = types.SimpleNamespace(song_idx=np.zeros(4, dtype=np.int64))
    for slots, songs, word in (([1, 1], [0, 1], "distinct"), ([4], [0], "distinct"), ([-1], [0], "distinct"),
                               ([0, 2], [0, 3], "out of range"), ([0], [-1], "out of range"), ([3], [2], "not valid"),
                               ([0, 1], [0], "one song")):
        with pytest.raises(ValueError, match=word):
            b.refill(step, win, slots, songs)
    with pytest.raises(ValueError, match="offsets"):
        b.refill(step, win, [0], [1], offset_s=-1.0)


# --------------------------------------------------------------------------- GPU
def _cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop,opts", [(4096, 1024, {}), (4096, 1024, {"SAGA_STFT_NO_EO": "1"}), (1024, 256, {}),
                                            (2048, 512, {"SAGA_STFT_RING": "0"})],
                         ids=["4096_eo", "4096_three_pass", "1024", "2048_generic"])
def test_rows_equal_the_full_stft(n_fft, hop, opts):
    """Rows of stft_rows_batch against saga_stft_exec's rows (torch.equal, magnitude and phasor, padding included).
    n_fft 2048 / hop 512: stft_exec runs the ring kernel by default, the rows entry the generic kernel, which is
    stft_exec's SAGA_STFT_RING=0 twin."""
    torch = _cuda()
    from amt_saga_b200 import ops
    plan = ops.get_stft_plan(n_fft, hop, True)
    P = ops.frame_pitch(plan.n_bins)
    g = torch.Generator(device="cuda").manual_seed(11)
    lens = np.array([hop * 61 + 7, hop * 40, hop * 97 + 301, n_fft // 2 + 5, hop * 23 + 1])
    n = len(lens)
    # rows of an odd width starting 3 floats into the buffer: the clips start at unaligned offsets, each differently
    width = int(lens.max()) + 10
    width += 1 - width % 2
    base = torch.rand((n, width), device="cuda", generator=g) * 2 - 1
    wav = base[:, 3:3 + int(lens.max()) + 1]
    for i, L in enumerate(lens):
        wav[i, L:] = 0
    with ops.options(**opts):
        ref = ops.stft_batch(wav, plan, lens=lens, want_phase=True, want_max=True)
    rm, rp = ref["mag_storage"], ref["phase_storage"]
    Tc = 1 + lens // hop
    nf = 40
    starts = {"start": np.zeros(n, dtype=np.int64), "mid": Tc // 3, "straddle": np.maximum(Tc - 13, 0), "past": Tc + 3}
    with ops.options(**{k: v for k, v in opts.items() if k != "SAGA_STFT_RING"}):
        for name, f0 in starts.items():
            r = ops.stft_rows_batch(wav, plan, f0, nf, lens=lens, phase_out=True)
            m, p = r["mag_storage"], r["phase_storage"]
            for c in range(n):
                live = int(np.clip(Tc[c] - f0[c], 0, nf))
                assert torch.equal(m[c, :live], rm[c, f0[c]:f0[c] + live]), (name, c)
                assert torch.equal(p[c, :live], rp[c, f0[c]:f0[c] + live]), (name, c)
                assert not m[c, live:].any() and not p[c, live:].any(), (name, c)
        # a destination permutation with dst_row0 > 0: rows outside the target keep a sentinel
        perm, row0 = np.array([3, 0, 4, 1, 2]), 5
        out = torch.full((n, nf + row0 + 4, P), 7.0, device="cuda")
        ph = torch.full((n, nf + row0 + 4, P), 7 + 7j, device="cuda", dtype=torch.complex64)
        f0 = starts["straddle"]
        ops.stft_rows_batch(wav, plan, f0, nf, lens=lens, out=out, phase_out=ph, dst_clip=perm, dst_row0=row0)
        for c in range(n):
            d, live = perm[c], int(np.clip(Tc[c] - f0[c], 0, nf))
            assert torch.equal(out[d, row0:row0 + live], rm[c, f0[c]:f0[c] + live])
            assert torch.equal(ph[d, row0:row0 + live], rp[c, f0[c]:f0[c] + live])
            assert not out[d, row0 + live:row0 + nf].any() and not ph[d, row0 + live:row0 + nf].any()
            assert (out[d, :row0] == 7).all() and (out[d, row0 + nf:] == 7).all()
            assert (ph[d, :row0] == 7 + 7j).all() and (ph[d, row0 + nf:] == 7 + 7j).all()
        # clip_max accumulated over chunks of frames (not zeroed by the entry) = stft_exec's ref_mag
        cm = torch.zeros(n, device="cuda")
        for c0 in range(0, int(Tc.max()), 37):
            ops.stft_rows_batch(wav, plan, c0, 37, lens=lens, clip_max=cm)
        assert torch.equal(cm, ref["clip_max"])


def _walk_songs():
    """The five golden songs plus ragged synthetic ones (one shorter than a window, one not a whole number of hops)."""
    songs, _ = _golden_songs()
    extra = [piano_clip(1200 + i, int(SR * s) + d, n_notes=int(3 * s)) for i, (s, d) in
             enumerate(((5.1, 0), (13.7, 333), (22.0, 1), (31.3, 517)))]
    return songs + extra


def _snapshot(step):
    """A copy of everything the next step starts from."""
    return {"mag": step.mag.clone(), "ph": step.ph.clone(), "wav": step.wav.clone(), "wav_lens": step.wav_lens.copy(),
            "state": step.state.copy(), "song_ref": step.song_ref.clone(), "inv_song_ref": step.inv_song_ref.clone(),
            "inv_ref_C": [c.clone() for c in step.inv_ref_C], "ref_init": step._ref_init.clone(),
            "ref_given": step._ref_given.copy()}


def _assert_equal_state(torch, a, b, key):
    for k in a:
        x, y = a[k], b[k]
        if isinstance(x, list):
            assert all(torch.equal(u, v) for u, v in zip(x, y)), (key, k)
        elif isinstance(x, torch.Tensor):
            assert x.shape == y.shape and torch.equal(x, y), (key, k)
        else:
            assert np.array_equal(x, y), (key, k)


@pytest.mark.gpu
def test_waveform_hold_equals_stft_hold():
    """Setup, section, WALK (test_window_slide.py's slides and steps) and then refills, under both holds on the same
    songs.  The step state is compared with torch.equal after every step.  Step outputs: the STFT-held walk runs twice;
    an output equal in those two runs must be equal under hold="waveform"; one that is not deterministic from run to
    run is held to test_note_step.py's 1e-4 of its peak (and reported)."""
    torch = _cuda()
    from amt_saga_b200.note_step import NoteStepBatch
    songs = _walk_songs()
    bs = ss.SongBatch(hold="stft").setup(songs)
    bw = ss.SongBatch(hold="waveform")
    bw.chunk_bytes = 16 << 20       # several chunks of frames (227 here) and of songs (2 per CQT peak call)
    bw.setup(songs)
    assert bw.mag is None and bw.phase is None
    for k in ("T", "song_dur", "flatness", "keep", "valid", "ref_C", "ref_cols"):
        assert np.array_equal(getattr(bs, k), getattr(bw, k), equal_nan=getattr(bs, k).dtype.kind == "f"), k
    assert torch.equal(bs.ref_mag, bw.ref_mag)
    assert np.isfinite(bw.flatness).all()
    S = len(songs)
    offs = np.array([0.0, 1.3, 2.0, 0.5, 5.0, 0.0, 9.1, 17.9, 30.0])       # incl. one past the end, one straddling
    idx = np.arange(S)
    ws, ww = bs.section(idx, offs, T), bw.section(idx, offs, T)
    for k in ("mag", "phase", "wav"):
        assert torch.equal(getattr(ws, k), getattr(ww, k)), k
    assert all(np.array_equal(ws.geometry[k], ww.geometry[k]) for k in ws.geometry)

    # WALK on eight of the songs (one per WALK entry; lengths as given there)
    W = len(WALK)
    rng = np.random.default_rng(17)
    wsongs = [piano_clip(600 + w, int(SR * sec), n_notes=int(4 * sec)) for w, (sec, _) in enumerate(WALK)]
    notes = [[(float(rng.uniform(0.05, 5.0)), float(rng.uniform(0.3, 1.0)), int(rng.integers(40, 80))) for _ in range(4)]
             for _ in range(W)]
    clips = [[piano_clip(700 + 10 * w + k, int(SR * (notes[w][k][1] + 0.3)), n_notes=1,
                         pitch_range=(notes[w][k][2], notes[w][k][2])) for k in range(4)] for w in range(W)]
    runs = {}
    for name, hold in (("stft", "stft"), ("stft_again", "stft"), ("waveform", "waveform")):
        b = ss.SongBatch(hold=hold).setup(wsongs)
        win = b.section(np.arange(W), np.zeros(W), T)
        step = b.load_into(NoteStepBatch(W), win)
        outs, states = [], []
        for k in range(5):
            if k == 4:      # refills: a finished slot (0), a slot whose slide went past the end (3), one at an offset
                b.refill(step, win, [0, 3, 6], [2, 1, 7], [0.0, 2.5, 11.0])
            else:
                for rep in range(2):
                    mask = np.array([WALK[w][1][k] > rep for w in range(W)])
                    if mask.any():
                        b.slide(step, win, mask)
            states.append(_snapshot(step))
            kk = min(k, 3)
            guess, glens = _stack_guesses(torch, [clips[w][kk] for w in range(W)])
            nk = [notes[w][kk] for w in range(W)]
            out = step.step([x[0] for x in nk], [x[1] for x in nk], [x[2] for x in nk], guess, guess_lens=glens)
            outs.append(out)
            states.append(_snapshot(step))
        runs[name] = (outs, states, win)
    assert np.array_equal(runs["stft"][2].song_idx, runs["waveform"][2].song_idx)
    assert np.array_equal(runs["stft"][2].offset_s, runs["waveform"][2].offset_s)
    for i, (a, b) in enumerate(zip(runs["stft"][1], runs["waveform"][1])):
        _assert_equal_state(torch, a, b, "state %d" % i)
    nondet = set()
    for k, (a, a2, b) in enumerate(zip(runs["stft"][0], runs["stft_again"][0], runs["waveform"][0])):
        for key in a:
            x, x2, y = a[key], a2[key], b[key]
            if not isinstance(x, torch.Tensor):
                assert np.array_equal(x, y), (k, key)
            elif torch.equal(x, x2):
                assert torch.equal(x, y), (k, key)
            else:
                nondet.add(key)
                peak = float(x.abs().nan_to_num().max())
                assert float((x - y).abs().nan_to_num().max()) <= 1e-4 * peak, (k, key)
    print("outputs not deterministic from run to run (held to 1e-4 of peak):", sorted(nondet) or "none")


@pytest.mark.gpu
def test_waveform_hold_memory_after_setup():
    """After a hold="waveform" setup the batch holds its waveforms and [S, T_max] tables, not the [S, T_max, P] STFT
    (24 624 B per frame at n_fft 4096 against 4 096 B of float32 waveform: 6x)."""
    torch = _cuda()
    from amt_saga_b200 import ops
    songs = [piano_clip(1300 + i, int(SR * s), n_notes=int(2 * s)) for i, s in enumerate((60.0, 45.5, 71.2, 38.9))]
    ss.SongBatch(hold="waveform").setup(songs)        # plans and the CQT workspace, which later setups share
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    b = ss.SongBatch(hold="waveform").setup(songs)
    torch.cuda.synchronize()
    used = torch.cuda.memory_allocated() - base
    S, L_max = b.wav.shape
    T_max = int(b.T.max())
    bound = 4 * S * L_max + 4 * 8 * S * T_max + (2 << 20)        # waveforms + a few [S, T_max] tables + small tensors
    stft_bytes = S * T_max * ops.frame_pitch(b.nb) * 12             # mag + phase of hold="stft"
    print("hold=waveform after setup: %.1f MB (bound %.1f MB); hold=stft's song STFT alone: %.1f MB"
          % (used / 1e6, bound / 1e6, stft_bytes / 1e6))
    assert used <= bound
    assert stft_bytes >= 5 * bound


@pytest.mark.gpu
def test_corpus_walk_with_refills_against_the_cuda_class():
    """12 songs of 8-40 s through W = 4 slots under hold="waveform", with slides.  A slot takes the next song when its
    song's notes are done or its slide went past the song's end.  Every note's features are checked against the CUDA
    class driven song by song (test_window_slide.py's tolerances)."""
    torch = _cuda()
    from amt_saga_b200 import util_audio as ua
    from amt_saga_b200.note_step import NoteStepBatch
    rng = np.random.default_rng(23)
    secs = [8.0, 40.0, 12.5, 8.7, 20.0, 33.3, 8.4, 15.0, 26.0, 10.0, 18.2, 37.0]
    S, W = len(secs), 4
    songs = [piano_clip(1400 + i, int(SR * s), n_notes=int(3 * s)) for i, s in enumerate(secs)]
    n_notes = rng.integers(2, 5, size=S)
    notes = [[(float(rng.uniform(0.3, 1.0)), int(rng.integers(40, 80))) for _ in range(n_notes[s])] for s in range(S)]
    slides = [[int(rng.integers(0, 3)) if k else 0 for k in range(n_notes[s])] for s in range(S)]
    slides[0][1] = slides[3][1] = 2                   # 8 s and 9 s songs: the second slide goes past the end
    clips = [[piano_clip(1500 + 10 * s + k, int(SR * (notes[s][k][0] + 0.3)), n_notes=1,
                         pitch_range=(notes[s][k][1], notes[s][k][1])) for k in range(n_notes[s])] for s in range(S)]
    b = ss.SongBatch(hold="waveform").setup(songs)
    song_ref = b.ref_mag.double().cpu().numpy()
    cur = list(range(W))
    win = b.section(cur, np.zeros(W), T)
    step = b.load_into(NoteStepBatch(W), win)
    queue = list(range(W, S))

    def class_window(s):
        m = ua.audio_complete(songs[s], N)
        m.mag
        return m, m.section(0, None, T)
    cls = {s: class_window(s) for s in cur}
    k_note, offs, done = [0] * W, [0.0] * W, [False] * W
    checked, refilled, went_past, skipped = 0, 0, 0, 0
    while not all(done) or queue:
        fill = [w for w in range(W) if done[w]][:len(queue)]
        if fill:
            new = [queue.pop(0) for _ in fill]
            b.refill(step, win, fill, new)
            for w, s in zip(fill, new):
                cur[w], k_note[w], offs[w], done[w] = s, 0, 0.0, False
                cls[s] = class_window(s)
                assert win.song_idx[w] == s and win.offset_s[w] == 0.0
            refilled += len(fill)
        if all(done):
            break
        for rep in range(2):
            mask = np.array([not done[w] and slides[cur[w]][k_note[w]] > rep for w in range(W)])
            if not mask.any():
                continue
            past = b.slide(step, win, mask)
            for w in np.flatnonzero(mask):
                m, aw = cls[cur[w]]
                offs[w] = _oracle_slide(m, aw, offs[w])
                assert bool(past[w]) == (aw.shape[1] > T), (cur[w], k_note[w])
                if past[w]:
                    done[w] = True
                    went_past += 1
                    skipped += n_notes[cur[w]] - k_note[w]
        live = [w for w in range(W) if not done[w]]
        # onsets inside the song's remaining audio (a slide not past the end leaves at least 3 s of it): a note in the
        # silence after a short song's end has 0 / 0 log10 features in the class as well
        nk = [(float(rng.uniform(0.05, min(5.0, secs[cur[w]] - offs[w] - 1.2))),) + notes[cur[w]][k_note[w]]
              if not done[w] else (0.5, 0.5, 60) for w in range(W)]
        ck = [clips[cur[w]][k_note[w]] if not done[w] else clips[0][0] for w in range(W)]
        guess, glens = _stack_guesses(torch, ck)
        out = step.step([x[0] for x in nk], [x[1] for x in nk], [x[2] for x in nk], guess, guess_lens=glens)
        lens_used = step.wav_lens.copy()
        for w in live:
            s = cur[w]
            key = "song %d note %d" % (s, k_note[w])
            aw = cls[s][1]
            r = _class_step(ua, aw, *nk[w], ck[w], float(song_ref[s]), b.ref_C[s])
            assert out["valid"][w], key
            assert out["offset_frames"][w] == r["off_frames"], key
            assert lens_used[w] == r["wav_len"], key
            _check_features(out, w, r, float(song_ref[s]), key)
            assert float((step.mag[w, :, :2049] - aw._mag.st[:, :2049]).abs().max()) <= MAG_TOL * float(song_ref[s]), key
            checked += 1
            k_note[w] += 1
            if k_note[w] == n_notes[s]:
                done[w] = True
    assert checked + skipped == int(n_notes.sum())
    assert refilled == S - W and went_past >= 2
    print("corpus walk: %d notes checked, %d refills, %d slides past the end" % (checked, refilled, went_past))


@pytest.mark.gpu
def test_refill_of_a_window_with_a_pending_patch():
    """A slot subtracted in the last step is DIRTY: the next rebuild patches a sample range of it, and that patch is
    written over every window whose range covers the sample.  Refilling the slot must drop its range: its waveform is
    then the section's, and the other slots' waveforms are those of the same run without the refill."""
    torch = _cuda()
    from amt_saga_b200.note_step import NoteStepBatch
    songs = [piano_clip(1600 + i, int(SR * s), n_notes=int(3 * s)) for i, s in enumerate((14.0, 11.0, 17.5, 9.3))]
    clip = piano_clip(1650, int(SR * 0.8), n_notes=1, pitch_range=(57, 57))
    wavs = {}
    for refill in (False, True):
        b = ss.SongBatch(hold="waveform").setup(songs)
        win = b.section([0, 1, 2], [0.0, 0.0, 0.0], T)
        step = b.load_into(NoteStepBatch(3), win)
        guess, glens = _stack_guesses(torch, [clip] * 3)
        for onset in (1.0, 2.5):        # the first step leaves FULL windows; the second rebuilds (SYNCED), then DIRTY
            step.step([onset] * 3, [0.5] * 3, [57] * 3, guess, guess_lens=glens)
        assert (step.state == step.DIRTY).all() and step._dirty is not None
        if refill:
            b.refill(step, win, [1], [3], [1.5])
            assert step.state.tolist() == [step.DIRTY, step.AUDIO, step.DIRTY]
        wavs[refill] = step.wf()
    (w0, l0), (w1, l1) = wavs[False], wavs[True]
    sec = b.section([3], [1.5], T)
    assert l1[1] == sec.wav_len[0]
    assert torch.equal(w1[1, :l1[1]], sec.wav[0, :l1[1]])
    for w in (0, 2):
        assert l0[w] == l1[w] and torch.equal(w0[w, :l0[w]], w1[w, :l1[w]]), w
