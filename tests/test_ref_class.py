"""Parity against the reference's OWN class.

`oracle/ref_class.py` imports `/root/reference/util_audio.py` unmodified (stub modules for
matplotlib / magenta / soundfile, librosa entry points bound to oracle.spectral / oracle.cqt) and
`tests/ref_loop.py` drives it through the producer loop of `training.py:265-449`.

* here (CPU, /root/reference mounted): `AudioOracle` == reference class, bit for bit, on every
  intermediate of the loop and on the property setters -- so the restated container is the
  reference's code in behaviour, and only librosa/resampy remain restated;
* anywhere (CPU): `AudioOracle` == the committed golden vectors that class produced
  (tests/golden/make_ref_class_golden.py);
* GPU box: the CUDA `audio_complete` vs those golden vectors within north_star's tolerances
  (magnitudes 1e-4 of the peak, dB 0.01 above the floor, frame indexing exact).
"""
import os

import numpy as np
import pytest

from oracle import ref_class
from oracle.audio_oracle import AudioOracle
from tests import ref_loop as L
from tests.golden.make_ref_class_golden import FULL, FULL_COLS, SMALL, thin, thin_small

GOLD = os.path.join(os.path.dirname(__file__), "golden")
needs_reference = pytest.mark.skipif(not ref_class.available(),
                                     reason="needs the original project's source: set SAGA_REFERENCE_DIR")
MAG_TOL, DB_TOL = 1e-4, 0.01


def _run(AC, cfg, dtype=np.float64):
    p = L.small_params(cfg["timing_frames"]) if cfg["timing_frames"] != 258 else L.Params
    song, clips = L.make_inputs(cfg["seed"], cfg["seconds"], cfg["notes"], dtype=dtype)
    return L.run_loop(AC, song, cfg["notes"], clips, p, slide_after=cfg["slide_after"])


def _assert_identical(a, b):
    assert sorted(a) == sorted(b)
    for k in a:
        assert a[k].shape == b[k].shape and a[k].dtype == b[k].dtype, k
        assert np.array_equal(a[k], b[k], equal_nan=True), k


# --------------------------------------------------------------------------- CPU
@needs_reference
def test_reference_class_imports_unmodified():
    m = ref_class.load()
    assert os.path.samefile(m.__file__, os.path.join(ref_class.REFERENCE_DIR, "util_audio.py"))
    ac = m.audio_complete(np.zeros(8192), 4096)
    assert ac.hl == 1024 and ac.shape == (2049, 9)          # util_audio.py:65, T = 1 + n // hop


@needs_reference
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_oracle_container_equals_reference_class_on_the_producer_loop(dtype):
    ref = _run(ref_class.load().audio_complete, SMALL, dtype)
    ora = _run(AudioOracle, SMALL, dtype)
    _assert_identical(ref, ora)
    assert ref["n0_C_sw_pitch"].shape == (174, 8) and ref["n0_C_foc"].shape == (348, 8)
    assert ref["n0_C_velocity"].shape == (36, 8) and ref["n0_C_timing"].shape == (20, 64)
    assert ref["n2_wf_len_after"] == 1024 * 63               # hidden iSTFT length hop * (T - 1)


@needs_reference
def test_oracle_container_equals_reference_class_on_setters_and_errors():
    song, _ = L.make_inputs(3, 1.0, [])
    y = song.astype(np.float32)[:40000]
    _assert_identical(L.run_setters(ref_class.load().audio_complete, y), L.run_setters(AudioOracle, y))
    for AC in (ref_class.load().audio_complete, AudioOracle):
        a = AC(y, 2048)
        with pytest.raises(ValueError, match="Requested attribute does not exist"):
            a._P("nope")
        with pytest.raises(ValueError, match="Invalid attribute requested"):
            a.resize(0, 0.1, 8, attribs=["zzz"])


@needs_reference
def test_static_helpers_equal_reference_class():
    R = ref_class.load().audio_complete
    rng = np.random.default_rng(5)
    for t in (0, 1, 2, 3, 5, 7, 8, 9, 30):
        P = rng.standard_normal((6, t)).astype(np.float32)
        for target in (8, 258):
            a, b = R._resize(P, target), AudioOracle._resize(P, target)
            assert a.shape == b.shape and np.array_equal(a, b)
    S = np.abs(rng.standard_normal((2049, 12))).astype(np.float32)
    for bands, log in ((20, True), (80, True), (13, False)):
        assert np.array_equal(R.compress_bands(S, bands, log), AudioOracle.compress_bands(S, bands, log))
    for tone in (21, 60, 69, 108):
        assert R(None, 4096).midi_tone_to_FFT(tone) == AudioOracle(None, 4096).midi_tone_to_FFT(tone)


def test_oracle_matches_committed_reference_class_golden_small():
    g = dict(np.load(os.path.join(GOLD, "ref_class_loop_small.npz")))
    _assert_identical(g, thin_small(_run(AudioOracle, SMALL)))


def test_oracle_matches_committed_reference_class_golden_setters():
    g = dict(np.load(os.path.join(GOLD, "ref_class_setters.npz")))
    song, _ = L.make_inputs(3, 1.0, [])
    _assert_identical(g, L.run_setters(AudioOracle, song.astype(np.float32)[:40000]))


# --------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def cuda_class():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import amt_saga_b200  # noqa: F401
    from amt_saga_b200 import util_audio
    return util_audio.audio_complete


EXACT = ("off_frames", "wf_len_after", "fft_bin_min", "fft_bin_min_const", "slid_shape", "wf_final__len", "shape")


def _compare_with_golden(got, gold):
    """north_star tolerances; every key of the golden file is checked."""
    assert sorted(got) == sorted(gold)
    peak = float(gold["song_ref_mag"]) if "song_ref_mag" in gold else None
    for k, g in gold.items():
        v = got[k]
        assert v.shape == g.shape, k
        base = k.split("_", 1)[1] if k[0] == "n" and k[1].isdigit() else k
        if base.endswith("__sha256"):   # bit patterns: checked on the CPU container only
            continue
        if base in EXACT:
            assert np.array_equal(v, g), k
        elif base == "D_final" or base.startswith("D_final__c"):
            if base.endswith("__colsum"):
                continue
            above = g > -79.9          # ref = current max after a subtraction: 0 dB is the top
            assert np.abs(v[above] - g[above]).max() <= DB_TOL, k
        elif base == "ph":
            # (angle + 3.15) / 6.3 of a unit phasor: ill-conditioned where the bin is empty and
            # 2 pi-periodic; compare the phasors where the short-window magnitude is not noise
            m = gold[k[:-2] + "sw_mag"]
            lo = int(gold[k[:-2] + "fft_bin_min"])
            mm = np.zeros(g.shape)
            rows = min(g.shape[0], m.shape[0] - lo)
            mm[:rows] = m[lo:lo + rows]
            strong = mm > 1e-3 * m.max()
            d = np.abs(np.exp(1j * (v * 6.3 - 3.15)) - np.exp(1j * (g * 6.3 - 3.15)))
            assert d[strong].max() <= 2e-3, k
        elif base in ("F_foc_log10", "F_const_log10"):
            # log10(1000 x + 1) / max: error amplification 1000 / (ln10 (1000 x + 1)) <= 434 x the
            # 1e-4-of-peak magnitude tolerance, relative to a maximum of log10(1000 peak' + 1)
            src = gold[k.replace("_log10", "")] * peak
            lmax = np.log10(1000 * src.max() + 1)
            tol = MAG_TOL * peak * 1000 / (np.log(10) * (1000 * src + 1)) / lmax + 1e-6
            assert (np.abs(v - g) <= tol).all(), k
        else:
            scale = np.abs(g).max()
            assert np.abs(v - g).max() <= MAG_TOL * max(scale, 1e-30), (k, float(np.abs(v - g).max()), float(scale))


@pytest.mark.gpu
def test_cuda_class_matches_reference_class_golden_small(cuda_class):
    gold = dict(np.load(os.path.join(GOLD, "ref_class_loop_small.npz")))
    _compare_with_golden(thin_small(_run(cuda_class, SMALL)), gold)


@pytest.mark.gpu
def test_cuda_class_matches_reference_class_golden_full_shape(cuda_class):
    """The reference's real shape (N 4096, hop 1024, 258-frame window, float64 waveforms)."""
    gold = dict(np.load(os.path.join(GOLD, "ref_class_loop_full.npz")))
    got = thin(_run(cuda_class, FULL))
    assert got["n0_mag_after__cols"].shape == (2049, len(FULL_COLS))
    _compare_with_golden(got, gold)


@pytest.mark.gpu
def test_cuda_class_matches_reference_class_golden_setters(cuda_class):
    gold = dict(np.load(os.path.join(GOLD, "ref_class_setters.npz")))
    song, _ = L.make_inputs(3, 1.0, [])
    got = L.run_setters(cuda_class, song.astype(np.float32)[:40000])
    assert sorted(got) == sorted(gold)
    for k, g in gold.items():
        if k == "shape":
            assert np.array_equal(got[k], g)
        elif k == "D0":
            above = g > g.max() - 79.9
            assert np.abs(got[k][above] - g[above]).max() <= DB_TOL
        else:
            assert np.abs(got[k] - g).max() <= MAG_TOL * np.abs(g).max(), k
