"""Batched song setup (amt_saga_b200.song_setup.SongBatch, training.py:265-284) and the constant-Q peak of a column
range per clip (saga_cqt_peak_exec / ops.cqt_peak_batch).

* no GPU: the float64 frame arithmetic of SongBatch against the oracle container (bit-identical to the reference's
  class) one song at a time, and the argument checks of the new C entries;
* GPU: one ragged batch of the five golden songs against the reference class's normalisers, the peak against the
  maximum of the full transform (packed rows against padded ones, batch against single songs, streamed kernel
  against the fp32 one), `section` against the class's, the whole chain into NoteStepBatch, and refused songs.
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
from tests.golden.make_ref_class_golden import FULL, FULL_COLS, NOTE_STEPS, SMALL

GOLD = os.path.join(os.path.dirname(__file__), "golden")
MAG_TOL = 1e-4
SR, N, HOP = 44100, 4096, 1024


# --------------------------------------------------------------------------- no GPU
def _lengths():
    rng = np.random.default_rng(11)
    lens = [1, 2, 100, 1023, 1024, 1025, 2047, 2048, 2049, 4095, 4096, 4097, 10000]
    for k in (3, 7, 50, 129, 258, 259, 300):                 # at and around multiples of the hop
        lens += [k * HOP - 1, k * HOP, k * HOP + 1]
    lens += list(rng.integers(5000, 400000, 200 - len(lens)))
    return sorted(set(int(x) for x in lens))


def test_host_frame_arithmetic_equals_the_class_song_by_song():
    lens = _lengths()
    assert len(lens) >= 190
    rng = np.random.default_rng(3)
    for n in lens:
        wf = (np.arange(n, dtype=np.float64) % 997 + 1.0).astype(np.float32)     # no zero sample: the copy is visible
        o = AudioOracle(wf, N)
        T = o.shape[1]
        assert ss.song_frames([n], HOP)[0] == T
        dur = ss.song_durations([T], [n], SR)[0]
        want_dur = o._frames_to_seconds(T)                                      # ref_loop.py:77
        assert dur == want_dur and np.float64(dur).tobytes() == np.float64(want_dur).tobytes()
        assert ss.seconds_to_frames([dur], [T], [n], SR)[0] == o._seconds_to_frames(want_dur)     # ref_C columns
        dur_s = n / SR
        offsets = [0.0, dur_s / 2, rng.uniform(0, dur_s), dur_s - 258 * HOP / SR, dur_s, dur_s + 0.5]
        offsets = [x for x in offsets if x >= 0]
        g = ss.section_geometry(np.full(len(offsets), T), np.full(len(offsets), n), offsets, 258, SR)
        for i, off in enumerate(offsets):
            tfs = o._seconds_to_frames(off)
            tfe = tfs + 258
            assert (g["tfs"][i], g["tfe"][i]) == (tfs, tfe)
            assert g["w0"][i] == int(np.floor(o._frames_to_seconds(tfs) * o.sr))
            assert g["w1"][i] == int(np.floor(o._frames_to_seconds(tfe) * o.sr))
            w = o.section(off, None, 258).wf
            nc = int(g["n_copy"][i])
            assert w.shape[0] == g["wav_len"][i] == nc + g["pad"][i], (n, off)
            assert np.array_equal(w[:nc], wf[g["w0"][i]:g["w0"][i] + nc]) and not w[nc:].any(), (n, off)
    assert ss.song_frames([0], HOP)[0] == 0 and np.isnan(ss.song_durations([0], [0], SR)[0])


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__
    __graft_entry__.build()
    return _lib.lib()


def test_peak_entry_argument_errors_do_not_need_a_device(lib):
    one = C.c_void_p(256)                 # never dereferenced: the checks come first
    lo = hi = peak = ws = one
    assert lib.saga_cqt_peak_exec(None, one, one, None, 1, 1000, lo, hi, peak, ws, 1 << 20, None) == _lib.SAGA_ERR_INVALID
    assert b"cqt_peak_exec" in lib.saga_last_error_string()
    for k in range(4):                    # null col_lo, col_hi, peak_out, workspace
        args = [lo, hi, peak, ws]
        args[k] = None
        assert lib.saga_cqt_peak_exec(one, one, one, None, 1, 1000, *args, 1 << 20, None) == _lib.SAGA_ERR_INVALID
        assert b"null argument" in lib.saga_last_error_string()
    assert lib.saga_cqt_peak_exec(one, one, one, None, -1, 1000, lo, hi, peak, ws, 1 << 20, None) == _lib.SAGA_ERR_INVALID
    assert b"n_clips" in lib.saga_last_error_string()
    assert lib.saga_cqt_peak_workspace_bytes(None, 4, 1000) == 256
    with pytest.raises(ValueError):
        _lib.check(_lib.SAGA_ERR_INVALID, amt_saga_b200.cqt_plan.ParameterError)


# --------------------------------------------------------------------------- GPU
def _cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _golden_songs():
    """The five songs of the golden files: SMALL (3.2 s), FULL (10 s) and the three NOTE_STEPS songs (7 s)."""
    cfgs = [SMALL, FULL] + NOTE_STEPS
    gold = [dict(np.load(os.path.join(GOLD, "ref_class_loop_small.npz"))),
            dict(np.load(os.path.join(GOLD, "ref_class_loop_full.npz")))]
    for w in range(len(NOTE_STEPS)):
        g = np.load(os.path.join(GOLD, "ref_class_note_steps_w%d.npz" % w))
        gold.append({"song_ref_mag": g["w%d_song_ref_mag" % w], "ref_C": g["w%d_ref_C" % w]})
    songs = [L.make_inputs(c["seed"], c["seconds"], c["notes"])[0] for c in cfgs]
    return songs, gold


@pytest.mark.gpu
def test_ragged_song_batch_matches_reference_class_golden():
    _cuda()
    songs, gold = _golden_songs()
    assert len({len(s) for s in songs}) == 3
    b = ss.SongBatch().setup(songs)
    assert b.valid.all() and b.keep.all()
    got = {"flatness": b.flatness, "song_dur": b.song_dur, "song_ref_mag": b.ref_mag.double().cpu().numpy(),
           "ref_C": b.ref_C}
    for i, g in enumerate(gold):
        for k in ("flatness", "song_dur", "song_ref_mag", "ref_C"):
            if k not in g:
                continue
            v, ref = np.asarray(got[k][i], dtype=np.float64), np.asarray(g[k], dtype=np.float64)
            assert v.shape == ref.shape, (i, k)
            assert np.abs(v - ref).max() <= MAG_TOL * np.abs(ref).max(), (i, k, v, ref)
        if "fft_bin_min_const" in g:
            assert b.fft_bin_min_const == int(g["fft_bin_min_const"])


def _ragged(torch, seconds, seed):
    from amt_saga_b200 import synth
    lens = np.array([int(s * SR) for s in seconds])
    wav = synth.piano_batch(range(len(lens)), int(lens.max()), SR, seed_base=seed, device="cuda")
    for i, n in enumerate(lens):
        wav[i, n:] = 0
    return wav, lens


@pytest.mark.gpu
@pytest.mark.parametrize("stream", [None, "0"], ids=["default", "fp32_contraction"])
def test_cqt_peak_equals_max_of_the_full_transform(stream):
    """Packed rows without an image against the padded, materialised transform: same per-row arithmetic, and a maximum
    does not depend on the order, so the numbers are equal.  Batched against one song at a time: packing leaks
    nothing between clips."""
    torch = _cuda()
    from amt_saga_b200 import ops
    from amt_saga_b200.util_audio import note_to_hz
    wav, lens = _ragged(torch, (0.5, 3.0, 37.0, 61.0), 500)
    rng = np.random.default_rng(9)
    with ops.options(SAGA_CQT_STREAM=stream):
        for bpt in (1, 4, 16):
            plan = ops.get_cqt_plan(SR, HOP, note_to_hz("A0"), 87 * bpt, 12 * bpt, 2)
            Tc = np.array([plan.num_frames(int(n)) for n in lens])
            first = int(rng.integers(0, Tc[0]))
            lo = np.array([first, 5, int(rng.integers(0, Tc[2] // 2)), Tc[3] - 7])
            hi = np.array([first, Tc[1] + 40, int(rng.integers(Tc[2] // 2, Tc[2])), Tc[3] + 100])  # empty, past the end
            peak = ops.cqt_peak_batch(wav, plan, lo, hi, lens=lens)
            mag = ops.cqt_batch(wav, plan, lens=lens)["mag_storage"]
            want = torch.zeros(4, device="cuda")
            for c in range(4):
                a, e = max(int(lo[c]), 0), min(int(hi[c]), int(Tc[c]))
                if e > a:
                    want[c] = mag[c, a:e, :plan.n_bins].max()
            assert torch.equal(peak, want), (bpt, peak, want)
            assert float(want[1]) > 0 and float(want[0]) == 0
            single = torch.cat([ops.cqt_peak_batch(wav[c:c + 1, :lens[c]], plan, lo[c:c + 1], hi[c:c + 1]) for c in range(4)])
            assert torch.equal(peak, single), (bpt, peak, single)


@pytest.mark.gpu
def test_section_equals_the_class_section():
    torch = _cuda()
    from amt_saga_b200 import util_audio as ua
    songs, _ = _golden_songs()
    b = ss.SongBatch().setup(songs)
    idx, offs = [], []
    for s, song in enumerate(songs):
        d = len(song) / SR
        for off in (0.0, d / 3, d - 2.0):         # the last one hangs over the end
            idx.append(s)
            offs.append(max(off, 0.0))
    win = b.section(idx, offs, 258)
    assert (win.geometry["tfe"] > b.T[np.array(idx)]).any()
    for w, (s, off) in enumerate(zip(idx, offs)):
        a = ua.audio_complete(songs[s], N)
        a.mag
        ref = a.section(off, None, 258)
        assert torch.equal(win.mag[w], ref._mag.st), (s, off)
        assert torch.equal(win.phase[w], ref._ph.st), (s, off)
        assert torch.equal(win.wav[w, :int(win.wav_len[w])], ref._wf), (s, off)
        assert not win.wav[w, int(win.wav_len[w]):].any()


@pytest.mark.gpu
def test_song_batch_into_note_step_matches_reference_class_golden():
    """NOTE_STEPS songs -> SongBatch -> section(0, 258) -> NoteStepBatch.load with the normalisers SongBatch computed;
    two steps against the reference class's golden vectors (the checks of test_note_step.py)."""
    torch = _cuda()
    from amt_saga_b200.note_step import NoteStepBatch
    W = len(NOTE_STEPS)
    gold = {}
    for w in range(W):
        gold.update(np.load(os.path.join(GOLD, "ref_class_note_steps_w%d.npz" % w)))
    songs, clips = zip(*[L.make_inputs(c["seed"], c["seconds"], c["notes"]) for c in NOTE_STEPS])
    b = ss.SongBatch().setup(list(songs))
    win = b.section(np.arange(W), np.zeros(W), 258)
    step = b.load_into(NoteStepBatch(W), win)
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
        out = step.step([x[0] for x in notes], [x[1] for x in notes], [x[2] for x in notes],
                        torch.as_tensor(g, device="cuda"), guess_lens=lens)
        assert out["valid"].all()
        for w in range(W):
            key = "w%d_n%d_" % (w, n)
            peak = float(gold["w%d_song_ref_mag" % w])
            assert out["offset_frames"][w] == gold[key + "off_frames"]
            for mine, theirs in names.items():
                v, ref = out[mine][w].cpu().numpy(), gold[key + theirs]
                assert v.shape == ref.shape, (mine, v.shape, ref.shape)
                if theirs.endswith("_log10"):
                    src = gold[key + theirs.replace("_log10", "")].astype(np.float64) * peak
                    tol = MAG_TOL * peak * 1000 / (np.log(10) * (1000 * src + 1)) / np.log10(1000 * src.max() + 1) + 1e-6
                    assert (np.abs(v - ref) <= tol).all(), (key, mine)
                else:
                    assert np.abs(v - ref).max() <= MAG_TOL * np.abs(ref).max(), (key, mine, float(np.abs(v - ref).max()))
            m, lo = gold[key + "sw_mag"], int(gold[key + "fft_bin_min"])
            strong = np.zeros(gold[key + "ph"].shape, dtype=bool)
            rows = min(strong.shape[0], m.shape[0] - lo)
            strong[:rows] = m[lo:lo + rows] > 1e-3 * m.max()
            d = np.abs(np.exp(1j * (out["ph"][w].cpu().numpy() * 6.3 - 3.15)) - np.exp(1j * (gold[key + "ph"] * 6.3 - 3.15)))
            assert d[strong].max() <= 2e-3
            mag_after = step.mag[w, :, :2049].T.cpu().numpy()
            assert np.abs(mag_after[:, FULL_COLS] - gold[key + "mag_after__cols"]).max() <= MAG_TOL * peak
            assert abs(float(step.ref[w]) - float(gold[key + "ref_after"])) <= 2e-5 * float(gold[key + "ref_after"])


@pytest.mark.gpu
def test_refused_and_silent_songs_in_a_batch():
    """An empty song and one too short for the CQTs come back not valid with NaN normalisers; an all-zero song is valid
    with ref_C 0 and is gated out (its flatness is 1).  The other songs' results are those of a batch without them."""
    torch = _cuda()
    wav, lens = _ragged(torch, (3.0, 5.5), 700)
    good = ss.SongBatch().setup(wav, lens)
    L_max = wav.shape[1]
    mixed = torch.zeros((5, L_max), device="cuda")
    mixed[0], mixed[3] = wav[0], wav[1]
    mixed[2, :100] = wav[0, :100]
    mlens = np.array([lens[0], 0, 100, lens[1], 2 * SR])
    b = ss.SongBatch().setup(mixed, mlens)
    assert b.valid.tolist() == [True, False, False, True, True]
    assert np.isnan(b.ref_C[1:3]).all()
    assert np.array_equal(b.ref_C[4], np.zeros(3)) and abs(b.flatness[4] - 1.0) < 1e-6 and not b.keep[4]
    for i, j in ((0, 0), (3, 1)):
        assert np.array_equal(b.ref_C[i], good.ref_C[j])
        assert b.flatness[i] == good.flatness[j] and b.song_dur[i] == good.song_dur[j] and b.keep[i] == good.keep[j]
        assert float(b.ref_mag[i]) == float(good.ref_mag[j])
        assert torch.equal(b.mag[i, :good.T[j]], good.mag[j, :good.T[j]])
