"""Oracle (TEST INFRASTRUCTURE): the reference's OWN `util_audio.audio_complete`
class, imported unmodified from /root/reference and run in this container.

The reference is pure Python, so nothing is compiled: this is the Python form of
`oracle/_ref` (the task's "a Python reference can be imported in THIS container
to validate the restatement and to generate golden vectors").  Recipe:

* `/root/reference/util_audio.py` is executed as-is by importlib (never copied),
* while it is being imported, `sys.modules` holds empty stand-ins for the
  packages it imports at module level but that the hot path never calls
  (`matplotlib.pyplot`, `magenta.music.midi_io`, `magenta.protobuf.music_pb2`,
  `soundfile`; `fluidsynth` is already optional, util_audio.py:22-26),
* `librosa` is a module object whose entry points used by `audio_complete`
  (util_audio.py:67, :92, :101, :127, :147, :179, :281, :331, :421-426) are
  bound to the numpy restatements in `oracle.spectral` / `oracle.cqt` -- the
  ONLY layer that remains restated (librosa 0.6.3 / resampy 0.2.x are not
  installed and there is no network),
* the module's `np` is a thin proxy of numpy that answers `np.int` with `int`
  (util_audio.py:451; removed from numpy >= 1.24) -- numpy itself is untouched.

Every line of `audio_complete` (lazy properties and their invalidation rules,
`subtract`, `_seconds_to_frames`, `section/slice/concat`, `_resize/resize`,
`slice_C`, `compress_bands`, `section_power`, `midi_tone_to_FFT`, `clone`) is
therefore the reference's code.  `/root/reference` does not exist on the GPU
box: `available()` is False there, tests that need the class skip, and the GPU
tests use the golden vectors `tests/golden/make_ref_class_golden.py` generated
from this class here.
"""
import importlib.util
import os
import sys
import types

import numpy as _np

from . import cqt as _cqt
from . import spectral as _sp

# a checkout of the original project (its util_audio.py and fixture directories); unset: not available
REFERENCE_DIR = os.environ.get("SAGA_REFERENCE_DIR", "")
_mod = None


def available():
    return bool(REFERENCE_DIR) and os.path.isfile(os.path.join(REFERENCE_DIR, "util_audio.py"))


class _NumpyWithInt:
    """numpy, plus the `np.int` alias the reference still uses."""
    int = int

    def __getattr__(self, name):
        return getattr(_np, name)


def _librosa_shim():
    """Module object with the librosa entry points util_audio.py touches."""
    lr = types.ModuleType("librosa")
    core = types.ModuleType("librosa.core")
    feature = types.ModuleType("librosa.feature")
    for m in (lr, core):
        m.stft = _sp.stft
        m.istft = _sp.istft
        m.magphase = _sp.magphase
        m.amplitude_to_db = _sp.amplitude_to_db
        m.db_to_amplitude = _sp.db_to_amplitude
        m.fft_frequencies = _sp.fft_frequencies
        m.midi_to_hz = _sp.midi_to_hz
        m.note_to_midi = _sp.note_to_midi
        m.note_to_hz = _sp.note_to_hz
        m.midi_to_note = _sp.midi_to_note
        m.cqt = _cqt.cqt
    feature.spectral_flatness = _sp.spectral_flatness
    lr.core, lr.feature = core, feature
    lr.__version__ = "0.6.3-restated"
    return {"librosa": lr, "librosa.core": core, "librosa.feature": feature}


def _stubs():
    names = ["matplotlib", "matplotlib.pyplot", "magenta", "magenta.music", "magenta.music.midi_io",
             "magenta.protobuf", "magenta.protobuf.music_pb2", "soundfile"]
    mods = {n: types.ModuleType(n) for n in names}
    for n, m in mods.items():
        if "." in n:
            parent, leaf = n.rsplit(".", 1)
            setattr(mods[parent], leaf, m)
    mods.update(_librosa_shim())
    return mods


def load():
    """Import the original project's util_audio.py (once) and return the module."""
    global _mod
    if _mod is not None:
        return _mod
    if not available():
        raise FileNotFoundError("SAGA_REFERENCE_DIR does not name the original project's source (%r)" % REFERENCE_DIR)
    stand_ins = _stubs()
    saved = {n: sys.modules.get(n) for n in stand_ins}
    sys.modules.update(stand_ins)
    try:
        spec = importlib.util.spec_from_file_location(
            "_saga_reference_util_audio", os.path.join(REFERENCE_DIR, "util_audio.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        for n, old in saved.items():
            if old is None:
                sys.modules.pop(n, None)
            else:
                sys.modules[n] = old
    mod.np = _NumpyWithInt()
    _mod = mod
    return mod


def audio_complete(*args, **kwargs):
    """Construct the reference's class (util_audio.py:32)."""
    return load().audio_complete(*args, **kwargs)
