"""Batched per-note step (amt_saga_b200.note_step.NoteStepBatch) against the reference's OWN class: the golden
vectors were produced by /root/reference/util_audio.py driven through the producer loop of training.py:265-449
(tests/golden/make_ref_class_golden.py::note_steps, three songs x two notes, N 4096 / hop 1024 / 258 frames)."""
import os

import numpy as np
import pytest

from oracle.audio_oracle import AudioOracle
from tests import ref_loop as L
from tests.golden.make_ref_class_golden import FULL_COLS, NOTE_STEPS

GOLD = os.path.join(os.path.dirname(__file__), "golden")
MAG_TOL = 1e-4


def test_resize_map_equals_reference_resize_on_column_indices():
    """Host logic: the index map must pick exactly the columns `_resize(P[:, s:t], target)` returns."""
    import amt_saga_b200  # noqa: F401
    from amt_saga_b200.note_step import NoteStepBatch
    rng = np.random.default_rng(1)
    P = np.arange(258, dtype=np.float64)[None, :] + 1.0       # column j holds j + 1 (0 marks "zeros")
    s = rng.integers(0, 270, size=200)                        # onsets are >= 0: frames never negative
    t = s + rng.integers(-2, 40, size=200)
    t[t < 0] = 0
    for target in (8, 258):
        m = NoteStepBatch._resize_map(s, t, 258, target)
        for i in range(len(s)):
            want = AudioOracle._resize(P[:, s[i]:t[i]], target)[0]
            got = np.where(m[i] >= 0, m[i] + 1.0, 0.0)
            assert np.array_equal(got, want), (s[i], t[i], target)


@pytest.mark.gpu
@pytest.mark.parametrize("full_cqt", [False, True], ids=["frame_window_cqt", "full_window_cqt"])
def test_batched_note_step_matches_reference_class_golden(full_cqt):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import amt_saga_b200  # noqa: F401
    from amt_saga_b200 import util_audio as ua
    from amt_saga_b200.note_step import NoteStepBatch
    W = len(NOTE_STEPS)
    gold = {}
    for w in range(W):
        gold.update(np.load(os.path.join(GOLD, "ref_class_note_steps_w%d.npz" % w)))
    songs, clips = zip(*[L.make_inputs(c["seed"], c["seconds"], c["notes"]) for c in NOTE_STEPS])
    # windows exactly as `mid_wf.section(0, None, 258)` leaves them (training.py:284)
    mags, phs, wavs = [], [], []
    for song in songs:
        a = ua.audio_complete(song, 4096)
        a.mag
        w = a.section(0, None, 258)
        mags.append(w._mag.st), phs.append(w._ph.st), wavs.append(w._wf)
    assert len({int(x.numel()) for x in wavs}) == 1
    batch = NoteStepBatch(W)
    batch.full_cqt = full_cqt
    batch.load(torch.stack(mags), torch.stack(phs), torch.stack(wavs),
               [float(gold["w%d_song_ref_mag" % w]) for w in range(W)], np.stack([gold["w%d_ref_C" % w] for w in range(W)]))
    names = {"C_timing": "C_timing", "C_sw_pitch": "C_sw_pitch", "C_sw_inst": "C_sw_inst", "F_sw_inst_foc": "F_foc",
             "F_sw_inst_foc_log10": "F_foc_log10", "F_sw_inst_foc_const": "F_const",
             "F_sw_inst_foc_const_log10": "F_const_log10", "C_sw_inst_foc": "C_foc", "C_sw_inst_foc_const": "C_foc_const",
             "C_velocity": "C_velocity"}
    for n in range(2):
        notes = [c["notes"][n] for c in NOTE_STEPS]
        lens = np.array([len(clips[w][n]) for w in range(W)])
        g = np.zeros((W, lens.max()), dtype=np.float32)
        for w in range(W):
            g[w, :lens[w]] = clips[w][n]
        out = batch.step([x[0] for x in notes], [x[1] for x in notes], [x[2] for x in notes],
                         torch.as_tensor(g, device="cuda"), guess_lens=lens)
        assert out["valid"].all()
        for w in range(W):
            key = "w%d_n%d_" % (w, n)
            peak = float(gold["w%d_song_ref_mag" % w])
            assert out["offset_frames"][w] == gold[key + "off_frames"]          # frame indexing: exact
            for mine, theirs in names.items():
                v, ref = out[mine][w].cpu().numpy(), gold[key + theirs]
                assert v.shape == ref.shape, (mine, v.shape, ref.shape)
                if theirs.endswith("_log10"):
                    src = gold[key + theirs.replace("_log10", "")].astype(np.float64) * peak
                    tol = MAG_TOL * peak * 1000 / (np.log(10) * (1000 * src + 1)) / np.log10(1000 * src.max() + 1) + 1e-6
                    assert (np.abs(v - ref) <= tol).all(), (key, mine)
                else:
                    assert np.abs(v - ref).max() <= MAG_TOL * np.abs(ref).max(), (key, mine, float(np.abs(v - ref).max()))
            # phase feature: compare phasors where the short-window magnitude is not noise
            m, lo = gold[key + "sw_mag"], int(gold[key + "fft_bin_min"])
            strong = np.zeros(gold[key + "ph"].shape, dtype=bool)
            rows = min(strong.shape[0], m.shape[0] - lo)
            strong[:rows] = m[lo:lo + rows] > 1e-3 * m.max()
            d = np.abs(np.exp(1j * (out["ph"][w].cpu().numpy() * 6.3 - 3.15)) - np.exp(1j * (gold[key + "ph"] * 6.3 - 3.15)))
            assert d[strong].max() <= 2e-3
            # state after the subtraction (training.py:449)
            mag_after = batch.mag[w, :, :2049].T.cpu().numpy()
            ref_cols = gold[key + "mag_after__cols"]
            assert np.abs(mag_after[:, FULL_COLS] - ref_cols).max() <= MAG_TOL * peak
            assert np.abs(mag_after.sum(axis=0, dtype=np.float64) - gold[key + "mag_after__colsum"]).max() \
                <= 1e-4 * gold[key + "mag_after__colsum"].max()
            assert abs(float(batch.ref[w]) - float(gold[key + "ref_after"])) <= 2e-5 * float(gold[key + "ref_after"])
    # after a subtraction the next step's waveform is the iSTFT of mag * ph: hop * (T - 1) samples
    batch.step([0.5] * W, [0.5] * W, [60] * W, torch.zeros((W, 8192), device="cuda"), subtract=False)
    assert batch.wav.shape[1] == 1024 * 257 == int(gold["w0_n1_wf_len_after"])


@pytest.mark.gpu
def test_incremental_wave_rebuild_equals_full_istft():
    """After the first subtraction `wav` is an iSTFT, and a subtraction only changes frames [o, o + tg): the note step
    then re-inverts just the rows around them and patches the sample range they reach (util_audio.py:88-106 rebuilds
    everything).  Four steps with ragged guesses, onsets at the window start, in the middle and hanging over the end:
    the patched waveform and every feature must equal the full rebuild's."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import amt_saga_b200  # noqa: F401
    from amt_saga_b200 import ops, synth
    from amt_saga_b200.note_step import NoteStepBatch
    dev = torch.device("cuda")
    W, Lw = 6, 264168
    wav = synth.piano_batch(range(W), Lw, 44100, seed_base=4000, device=dev)
    plan = ops.get_stft_plan(4096, 1024, True)
    r = ops.stft_batch(wav, plan, want_phase=True)
    guess = synth.piano_batch(range(W), 54277, 44100, n_notes=1, seed_base=7000, device=dev)
    lens = np.array([54277, 30000, 54277, 8192, 41000, 54277])
    onsets = [np.array([0.0, 0.5, 2.0, 3.1, 5.6, 5.99]), np.array([5.9, 0.0, 1.0, 4.0, 2.5, 0.2]),
              np.array([1.5, 5.5, 0.01, 2.2, 0.0, 4.9]), np.array([3.0, 3.0, 3.0, 3.0, 3.0, 3.0])]
    outs = {}
    for inc in (True, False):
        b = NoteStepBatch(W)
        b.incremental_istft = inc
        b.load(r["mag_storage"][:, :258].clone(), r["phase_storage"][:, :258].clone(), wav, r["clip_max"], np.ones((W, 3)))
        seq = []
        for k, on in enumerate(onsets):
            o = b.step(on, np.full(W, 0.6), np.array([50, 60, 45, 72, 50, 60]) + k, guess, guess_lens=lens)
            seq.append((b.wav.clone(), {n: v.clone() for n, v in o.items() if isinstance(v, torch.Tensor)}))
        outs[inc] = seq
        used_patch = b._wav_synced
    assert used_patch
    for k in range(len(onsets)):
        wa, fa = outs[True][k]
        wb, fb = outs[False][k]
        assert wa.shape == wb.shape
        assert float((wa - wb).abs().max()) <= 1e-6 * float(wb.abs().max()), k
        for n in fb:
            assert torch.allclose(fa[n], fb[n], rtol=0, atol=1e-6 * max(float(fb[n].abs().max()), 1e-30)), (k, n)
    assert torch.equal(outs[True][1][0], outs[False][1][0])        # step 2 inverts everything in both modes


@pytest.mark.gpu
def test_shared_cascade_across_pitches_is_bit_identical():
    """Pitches of equal CQT geometry share one decimation cascade in the batched step (saga_cqt_frames_shared_exec:
    cascade once for the run of windows, one contraction per pitch on its clip range); with `share_cascade = False`
    every pitch group runs the whole transform on its own.  Same kernels on the same data: equal bit for bit when
    every pitch still gets its own contraction launch ("per_plan"); the default packs a run's pitches into one launch
    (saga_cqt_frames_shared_multi_exec), whose K split and hence summation order differ: 2e-6 of peak.  40 windows over
    23 pitches in every geometry class the note-relative transforms meet."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import amt_saga_b200  # noqa: F401
    from amt_saga_b200 import ops, synth
    from amt_saga_b200.note_step import NoteStepBatch
    dev = torch.device("cuda")
    W, Lw = 40, 264168
    wav = synth.piano_batch(range(W), Lw, 44100, seed_base=8000, device=dev)
    plan = ops.get_stft_plan(4096, 1024, True)
    r = ops.stft_batch(wav, plan, want_phase=True)
    guess = synth.piano_batch(range(W), 54277, 44100, n_notes=1, seed_base=9000, device=dev)
    rng = np.random.default_rng(5)
    pitch = np.concatenate([np.arange(30, 96, 3), rng.integers(30, 96, W - 22)])
    onset = rng.uniform(0, 5.5, W)
    geoms = set()
    outs = {}
    for share in (True, "per_plan", False):
        b = NoteStepBatch(W)
        b.share_cascade = share
        b.load(r["mag_storage"][:, :258].clone(), r["phase_storage"][:, :258].clone(), wav, r["clip_max"], np.ones((W, 3)))
        o1 = b.step(onset, np.full(W, 0.5), pitch, guess)
        o2 = b.step(onset[::-1].copy(), np.full(W, 0.7), pitch[::-1].copy(), guess)
        outs[share] = (o1, o2)
    for p in np.unique(pitch):
        geoms.add(ops.get_cqt_plan(44100, 1024, 440.0 * 2.0 ** ((int(p) - 69) / 12.0), 348, 192, 2).geometry())
    assert 1 < len(geoms) < len(np.unique(pitch))        # several pitches per geometry, several geometries
    for mode in (True, "per_plan"):
        for k in range(2):
            assert (outs[mode][k]["valid"] == outs[False][k]["valid"]).all()
            for n in ("C_sw_inst_foc", "C_velocity", "C_sw_pitch"):
                a_, b_ = torch.nan_to_num(outs[mode][k][n]), torch.nan_to_num(outs[False][k][n])
                if mode == "per_plan":      # same launches on the same data
                    assert torch.equal(a_, b_), (mode, k, n)
                else:                       # one launch for a run of pitches: a different K split, i.e. summation order
                    assert float((a_ - b_).abs().max()) <= 2e-6 * float(b_.abs().max()), (mode, k, n)


@pytest.mark.gpu
def test_shared_cascade_entry_points_reject_mismatched_plans():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import ctypes as C
    import amt_saga_b200  # noqa: F401
    from amt_saga_b200 import ops, synth, _lib
    wav = synth.piano_batch(range(4), 264168, 44100, seed_base=1, device="cuda")
    hz = lambda m: 440.0 * 2.0 ** ((m - 69) / 12.0)
    p_a, p_b = ops.get_cqt_plan(44100, 1024, hz(50), 36, 24, 2), ops.get_cqt_plan(44100, 1024, hz(51), 36, 24, 2)
    p_far = ops.get_cqt_plan(44100, 1024, hz(80), 36, 24, 2)
    assert p_a.geometry() == p_b.geometry() != p_far.geometry()
    tok = ops.cqt_cascade_shared(wav, p_a)
    first = torch.zeros(4, dtype=torch.int32, device="cuda")
    out = torch.zeros((4, 8, ops.frame_pitch(36)), device="cuda")
    ops.cqt_frames_from_cascade_multi(tok, [p_a, p_b], [0, 2], [2, 2], first, 8, out)
    ref = torch.cat([ops.cqt_frames_batch(wav[:2], p_a, first[:2]), ops.cqt_frames_batch(wav[2:], p_b, first[2:])])
    assert float((out - ref).abs().max()) <= 2e-6 * float(ref.max())
    tok = ops.cqt_cascade_shared(wav, p_a)
    with pytest.raises(ValueError):
        ops.cqt_frames_from_cascade_multi(tok, [p_a, p_far], [0, 2], [2, 2], first, 8, out)       # another geometry
    with pytest.raises(ValueError):
        ops.cqt_frames_from_cascade_multi(tok, [p_a, p_b], [0, 1], [2, 2], first, 8, out)         # ranges do not tile
    with pytest.raises(ValueError):
        ops.cqt_frames_from_cascade(tok, p_far, 0, 4, first, 8, out)
    # the C entry checks the geometry itself (a caller that bypasses the wrapper)
    lib = _lib.lib()
    handles = (C.c_void_p * 2)(p_a.handle, p_far.handle)
    cf, cc = np.array([0, 2], dtype=np.int32), np.array([2, 2], dtype=np.int32)
    rc = lib.saga_cqt_frames_shared_multi_exec(handles, 2, cf.ctypes.data_as(C.c_void_p), cc.ctypes.data_as(C.c_void_p),
                                               C.c_void_p(tok["wav"].data_ptr()), C.c_void_p(tok["offs"].data_ptr()), None, 4,
                                               tok["max_len"], C.c_void_p(first.data_ptr()), 8, C.c_void_p(out.data_ptr()),
                                               out.shape[2], 8 * out.shape[2], C.c_void_p(tok["ws"].data_ptr()),
                                               tok["ws"].numel(), None)
    assert rc == -1 and b"geometry" in lib.saga_last_error_string()


def test_dirty_ranges_cover_exactly_what_a_changed_frame_range_reaches():
    """Host logic of the incremental waveform rebuild, against a brute-force dependency map of the centred iSTFT:
    sample n of the trimmed output sums the frames t with t hop <= n + N/2 < t hop + N."""
    import amt_saga_b200  # noqa: F401
    from amt_saga_b200.note_step import NoteStepBatch
    rng = np.random.default_rng(3)
    for N, hop, T in ((4096, 1024, 258), (2048, 512, 40), (4096, 1024, 9), (1024, 256, 33)):
        L = hop * (T - 1)
        n = np.arange(L)
        t_lo = np.maximum(0, -(-(n + N // 2 - N + 1) // hop))                    # first / last frame reaching sample n
        t_hi = np.minimum(T - 1, (n + N // 2) // hop)
        o = np.concatenate([[0, 0, T - 1, T, T + 3, 1], rng.integers(0, T + 2, 40)])
        tg = np.concatenate([[1, T, 5, 4, 2, 0], rng.integers(0, 60, 40)])
        F, fa, lo, hi, tg_c = NoteStepBatch._dirty_ranges(o, tg, T, N, hop)
        assert 1 <= F <= T and np.all(fa >= 0) and np.all(fa + F <= T)
        for i in range(len(o)):
            oc, tc = min(int(o[i]), T), int(tg_c[i])
            touched = (t_hi >= oc) & (t_lo <= oc + tc - 1) if tc > 0 else np.zeros(L, dtype=bool)
            if touched.any():
                assert lo[i] <= n[touched].min() and n[touched].max() < hi[i]          # every affected sample is patched
                # and every patched sample is computable from the block: all frames reaching it lie inside
                # [fa, fa + F), or the missing ones do not exist (true window edge)
                p = n[lo[i]:hi[i]]
                assert np.all(t_lo[p] >= fa[i]) and np.all(t_hi[p] <= fa[i] + F - 1)
            else:
                assert hi[i] <= lo[i] or tc > 0
