"""Pins against the reference's OWN outputs.

`subtraction_demo/<name>_test{,_guess,_sub}.flac` are waveforms the reference wrote itself
(`test_snippets.py:473-514`, saved through `util_audio.py:520-527`): the mix, the
guessed note, and `istft(relu(mag - shifted normalised guess) * ph)`.  Decoded with the test-only
FLAC reader they pin  STFT -> magphase -> ref_mag -> subtract -> iSTFT  end to end: the oracle (and,
on a GPU, the CUDA path through the C ABI) must reproduce `_sub` from `_test` and `_guess` to the
24-bit quantisation of the files.  One triple is committed as tests/golden/ref_subtraction_piano.npz
(tests/golden/make_reference_pins.py); the others are checked when SAGA_REFERENCE_DIR names a
checkout of the original project.
"""
import json
import os

import numpy as np
import pytest

from oracle import ref_class
from oracle.audio_oracle import AudioOracle
from tests.flac_reader import read_flac

GOLD = os.path.join(os.path.dirname(__file__), "golden")
DEMO = os.path.join(ref_class.REFERENCE_DIR, "subtraction_demo", "")
SCALE = float(1 << 23)
# both inputs and the output went through 24-bit rounding: the residual is a few LSB at most and about
# a third of an LSB rms (measured: tests/golden/ref_subtraction_pins.json)
MAX_LSB, RMS_LSB = 4.0, 0.6

with open(os.path.join(GOLD, "ref_subtraction_pins.json")) as _fh:
    PINS = json.load(_fh)


def _residual_lsb(wave, sub_pcm):
    wave = np.asarray(wave, dtype=np.float64)
    assert wave.shape == sub_pcm.shape                     # iSTFT length hop*(T-1) = 1024*129
    e = np.abs(wave * SCALE - sub_pcm)
    return float(e.max()), float(np.sqrt((e ** 2).mean()))


def _oracle_sub(test_pcm, guess_pcm, pin):
    ac = AudioOracle((test_pcm / SCALE).astype(np.float32), pin["n_fft"])
    acg = AudioOracle((guess_pcm / SCALE).astype(np.float32), pin["n_fft"])
    s = ac.clone()
    s.subtract(acg, offset=pin["offset"], attack_compensation=pin["attack_compensation"],
               normalize=pin["normalize"])
    return s.wf


def test_oracle_reproduces_reference_subtraction_committed():
    z = np.load(os.path.join(GOLD, "ref_subtraction_piano.npz"))
    assert [len(z["test"]), len(z["guess"]), len(z["sub"])] == PINS["piano"]["samples"] == [132300, 88200, 132096]
    mx, rms = _residual_lsb(_oracle_sub(z["test"], z["guess"], PINS["piano"]), z["sub"])
    assert mx <= MAX_LSB and rms <= RMS_LSB, (mx, rms)


def test_wrong_parameters_do_not_reproduce_it():
    """The pin is sharp: without the normalisation the residual is five orders of magnitude larger."""
    z = np.load(os.path.join(GOLD, "ref_subtraction_piano.npz"))
    pin = dict(PINS["piano"], normalize=False)
    mx, _ = _residual_lsb(_oracle_sub(z["test"], z["guess"], pin), z["sub"])
    assert mx > 1e4


needs_fixtures = pytest.mark.skipif(not (ref_class.REFERENCE_DIR and os.path.isdir(DEMO)),
                                    reason="needs the original project's FLAC fixtures: set SAGA_REFERENCE_DIR")


@needs_fixtures
@pytest.mark.parametrize("name", sorted(PINS))
def test_oracle_reproduces_reference_subtraction_from_flac(name):
    pcm = {}
    for part in ("test", "test_guess", "test_sub"):
        pcm[part], sr, bps = read_flac(DEMO + "%s_%s.flac" % (name, part))    # checks CRC-16s and the MD5
        assert (sr, bps) == (44100, 24)
    if name == "piano":
        z = np.load(os.path.join(GOLD, "ref_subtraction_piano.npz"))
        assert np.array_equal(z["test"], pcm["test"]) and np.array_equal(z["sub"], pcm["test_sub"])
    mx, rms = _residual_lsb(_oracle_sub(pcm["test"], pcm["test_guess"], PINS[name]), pcm["test_sub"])
    assert mx <= MAX_LSB and rms <= RMS_LSB, (mx, rms)


@needs_fixtures
def test_fixture_lengths_pin_resize_targets():
    """short_window_demo/{j}/sw_{j}_*.flac hold exactly 1024*(j-1) samples: `_resize` returned j frames
    (test_snippets.py:1204-1211) and istft yields hop*(T-1) samples."""
    root = os.path.join(ref_class.REFERENCE_DIR, "short_window_demo", "")
    for j in (6, 8, 10, 15, 20):
        pcm, sr, bps = read_flac(root + "%d/sw_%d_0.flac" % (j, j))
        assert len(pcm) == 1024 * (j - 1) and sr == 44100


@pytest.mark.gpu
def test_cuda_path_reproduces_reference_subtraction():
    """The product path (audio_complete over the C ABI: K1 STFT, K3 subtract, K4 iSTFT, all on the
    device) against the reference's own output."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import amt_saga_b200  # noqa: F401
    from amt_saga_b200.util_audio import audio_complete
    z = np.load(os.path.join(GOLD, "ref_subtraction_piano.npz"))
    pin = PINS["piano"]
    ac = audio_complete((z["test"] / SCALE).astype(np.float32), pin["n_fft"])
    acg = audio_complete((z["guess"] / SCALE).astype(np.float32), pin["n_fft"])
    s = ac.clone()
    s.subtract(acg, offset=pin["offset"], attack_compensation=pin["attack_compensation"],
               normalize=pin["normalize"])
    wf = s.wf
    wf = wf.detach().cpu().numpy() if hasattr(wf, "detach") else np.asarray(wf)
    mx, rms = _residual_lsb(wf, z["sub"])
    # fp32 FFTs on the device instead of the reference's float64: one more LSB of slack
    assert mx <= MAX_LSB + 1.0 and rms <= RMS_LSB, (mx, rms)
