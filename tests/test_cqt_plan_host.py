"""The product's host-side CQT plan (amt-saga_b200/cqt_plan.py) folds librosa's
"rect FFT x sparsified basis" into time-domain banks.  Here the DEVICE algorithm
(decimate with the FIR taps, reflect-indexed strided frames, dense contraction)
is replayed in float64 numpy from the plan's own arrays and must reproduce the
oracle's multi-rate CQT -- proving the formulation, independent of any GPU."""
import numpy as np
import pytest

import amt_saga_b200  # noqa: F401
from amt_saga_b200.cqt_plan import CqtPlan, ParameterError, kaiser_fast_taps
from oracle import cqt as ocqt
from oracle import resample as ors
from oracle.spectral import midi_to_hz, note_to_hz
from tests.step_replay import device_model


CASES = [
    # (sr, hop, lowest note, n_bins, bins_per_octave)  -- filter_scale = 2 as util_audio.py:426
    (16000, 512, "C1", 84, 12),      # BASELINE cfg1
    (44100, 512, "C1", 84, 12),      # cfg3
    (44100, 1024, "A0", 87, 12),     # ref_C_1 (training.py:271): n_bins not a multiple of bpo
    (44100, 1024, "A0", 174, 24),    # C_sw_pitch (training.py:340)
    (44100, 1024, "D3", 36, 24),     # C_velocity (training.py:382): early factor 16
    # the per-note step's heavy shapes (note_step.py), the plans tests/step_replay.py replays it with
    (44100, 1024, "A0", 348, 48),    # C_sw_inst (training.py:344)
    (44100, 1024, "C4", 348, 192),   # C_sw_inst_foc_const (training.py:375)
    (44100, 1024, 93, 348, 192),     # C_sw_inst_foc at A6: the 12-pitch geometry run 93..104, no early decimation
    (44100, 1024, 11, 36, 24),       # C_velocity of A0 (pitch - 10): early factor 128
]


@pytest.mark.parametrize("sr,hop,low,n_bins,bpo", CASES)
def test_folded_banks_reproduce_oracle_cqt(sr, hop, low, n_bins, bpo):
    rng = np.random.default_rng(7)
    n = 3 * sr // 2 + 37
    t = np.arange(n)
    y = 0.4 * np.sin(2 * np.pi * 220.0 * t / sr) + 0.2 * np.sin(2 * np.pi * 1318.5 * t / sr) \
        + 0.05 * rng.standard_normal(n)
    fmin = note_to_hz(low) if isinstance(low, str) else float(midi_to_hz(low))     # a note name or a MIDI number
    ref = ocqt.cqt(y, sr=sr, hop_length=hop, fmin=fmin, n_bins=n_bins, bins_per_octave=bpo,
                   filter_scale=2)
    plan = CqtPlan(sr, hop, fmin, n_bins, bpo, filter_scale=2, create_device_plan=False)
    got = device_model(plan, y)
    assert got.shape == ref.shape
    assert plan.num_frames(n) == ref.shape[1]
    peak = np.abs(ref).max()
    assert np.abs(got - ref).max() <= 2e-6 * peak


def test_taps_match_oracle_resampler():
    for D in (2, 4, 8, 16):
        assert np.allclose(kaiser_fast_taps(D), ors.decimation_taps(D) * np.sqrt(D), rtol=0, atol=1e-15)


def test_plan_geometry_cfg3():
    plan = CqtPlan(44100, 512, note_to_hz("C1"), 84, 12, filter_scale=2, create_device_plan=False)
    assert plan.early_factor == 2 and len(plan.octaves) == 7
    assert [o["hop"] for o in plan.octaves] == [256, 128, 64, 32, 16, 8, 4]
    assert all(o["n_fft"] == 512 and o["n_filters"] == 12 for o in plan.octaves)
    assert [o["first_bin"] for o in plan.octaves] == [72, 60, 48, 36, 24, 12, 0]


def test_errors_like_librosa():
    with pytest.raises(ParameterError):   # hop not divisible by 2^(n_octaves-1)
        CqtPlan(44100, 100, note_to_hz("C1"), 84, 12, filter_scale=2, create_device_plan=False)
    with pytest.raises(ParameterError):   # pass-band beyond Nyquist
        CqtPlan(8000, 512, note_to_hz("C1"), 96, 12, filter_scale=2, create_device_plan=False)
    with pytest.raises(ocqt.ParameterError):
        ocqt.cqt(np.zeros(4000), sr=8000, hop_length=512, fmin=note_to_hz("C1"), n_bins=96,
                 filter_scale=2)


def test_note_relative_plans_fall_into_few_contiguous_geometry_classes():
    """The batched per-note step shares one decimation cascade between pitches whose plans have the same geometry
    (CqtPlan.geometry(): early factor, levels, hops, kernel lengths) and walks the windows in pitch order: over the 88
    keys the two note-relative shapes of training.py:366-388 must fall into a handful of classes, each a contiguous
    pitch range (a class that came back later would only cost an extra cascade, never a wrong result)."""
    from amt_saga_b200.cqt_plan import CqtPlan, ParameterError
    for nbins, bpo, shift in ((348, 192, 0), (36, 24, -10)):
        seq = []
        for midi in range(21, 109):
            try:
                seq.append(CqtPlan(44100, 1024, 440.0 * 2.0 ** ((midi + shift - 69) / 12.0), nbins, bpo, filter_scale=2,
                                   create_device_plan=False).geometry())
            except ParameterError:
                seq.append(None)            # pass-band beyond Nyquist: the producer loop skips the note
        runs = [g for i, g in enumerate(seq) if g is not None and (i == 0 or seq[i - 1] != g)]
        classes = {g for g in seq if g is not None}
        assert 2 <= len(classes) <= 16, len(classes)
        assert len(runs) == len(classes)                      # contiguous: every class is ONE run in pitch order
        valid = [g for g in seq if g is not None]
        assert len(valid) >= 40
