"""ctypes binding of include/saga_b200.h.  There is NO fallback: if the CUDA
library is missing or a call fails, this raises."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libsaga_b200.so")

SAGA_OK, SAGA_ERR_INVALID, SAGA_ERR_UNSUPPORTED, SAGA_ERR_CUDA, SAGA_ERR_NOMEM = 0, -1, -2, -3, -4
SUB_NORMALIZE, SUB_RELU, SUB_OFFSETS_ALIGNED = 1, 2, 4
SUB_SKIP_DB, SUB_ONLY_DB = 0x100, 0x200


class SagaError(RuntimeError):
    """CUDA / resource failure inside libsaga_b200."""


class SagaUnsupported(NotImplementedError):
    pass


class CqtOctave(C.Structure):
    _fields_ = [("level", C.c_int), ("hop", C.c_int), ("n_fft", C.c_int), ("n_filters", C.c_int),
                ("first_bin", C.c_int), ("bank_host", C.POINTER(C.c_float))]


class CqtDesc(C.Structure):
    _fields_ = [("n_bins", C.c_int), ("hop", C.c_int), ("early_factor", C.c_int),
                ("n_early_taps", C.c_int), ("early_taps_host", C.POINTER(C.c_float)),
                ("n_half_taps", C.c_int), ("half_taps_host", C.POINTER(C.c_float)),
                ("n_octaves", C.c_int), ("octaves", C.POINTER(CqtOctave))]


_P, _I, _L, _F, _D = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double

# name -> (restype, argtypes); must list every symbol include/saga_b200.h declares
SIGNATURES = {
    "saga_last_error_string": (C.c_char_p, []),
    "saga_abi_version": (_I, []),
    "saga_launch_count": (_L, []),
    "saga_set_option": (_I, [C.c_char_p, C.c_char_p]),
    "saga_get_option": (C.c_char_p, [C.c_char_p]),
    "saga_pcm16_absmax_exec": (_I, [_P, _L, _I, _I, _L, _P, _P]),
    "saga_pcm16_ingest_exec": (_I, [_P, _L, _I, _P, _L, _I, _L, _P, _P, _P, _D, _D, _P]),
    "saga_stft_plan_create": (_I, [C.POINTER(_P), _I, _I, _I, _P]),
    "saga_stft_plan_destroy": (_I, [_P]),
    "saga_stft_num_frames": (_L, [_P, _L]),
    "saga_stft_exec": (_I, [_P, _P, _P, _P, _I, _L, _P, _P, _P, _L, _L, _P, _P, _P]),
    "saga_istft_exec": (_I, [_P, _P, _P, _P, _I, _I, _L, _L, _P, _L, _P]),
    "saga_istft_rows_exec": (_I, [_P, _P, _P, _P, _I, _P, _I, _L, _L, _P, _L, _P]),
    "saga_subtract_db_exec": (_I, [_P, _P, _L, _P, _P, _L, _P, _I, _P, _P, _P, _P, _P, _L, _I, _P, _P,
                                   _I, _I, _I, _I, _L, _F, _F, _P]),
    "saga_amplitude_to_db_exec": (_I, [_P, _P, _P, _I, _I, _I, _L, _L, _F, _F, _P]),
    "saga_cqt_plan_create": (_I, [C.POINTER(_P), C.POINTER(CqtDesc)]),
    "saga_cqt_plan_destroy": (_I, [_P]),
    "saga_cqt_num_frames": (_L, [_P, _L]),
    "saga_cqt_workspace_bytes": (_L, [_P, _I, _L]),
    "saga_cqt_exec": (_I, [_P, _P, _P, _P, _I, _L, _P, _P, _L, _L, _P, _L, _I, _P]),
    "saga_cqt_frames_exec": (_I, [_P, _P, _P, _P, _I, _L, _P, _I, _P, _L, _L, _P, _L, _P]),
    "saga_cqt_frames_shared_exec": (_I, [_P, _P, _P, _P, _I, _L, _I, _I, _I, _P, _I, _P, _L, _L, _P, _L, _P]),
    "saga_cqt_frames_shared_multi_exec": (_I, [_P, _I, _P, _P, _P, _P, _P, _I, _L, _P, _I, _P, _L, _L, _P, _L, _P]),
    "saga_cqt_peak_workspace_bytes": (_L, [_P, _I, _L]),
    "saga_cqt_peak_exec": (_I, [_P, _P, _P, _P, _I, _L, _P, _P, _P, _P, _L, _P]),
    "saga_compress_bands_exec": (_I, [_P, _P, _P, _I, _I, _I, _L, _L, _L, _L, _P, _P]),
    "saga_short_window_exec": (_I, [_P, _P, _P, _I, _I, _I, _I, _L, _F, _P, _P, _P, _L, _P]),
    "saga_short_window_batch_exec": (_I, [_P, _P, _L, _L, _P, _I, _P, _I, _I, _I, _P, _F, _P, _P, _P, _L, _L, _I, _P]),
    "saga_gather_frames_exec": (_I, [_P, _P, _P, _P, _I, _I, _I, _L, _L, _L, _L, _P]),
    "saga_spectral_flatness_exec": (_I, [_P, _P, _I, _I, _I, _L, _L, _F, _P]),
}

_lib = None


def lib():
    """Load (once) and return the ctypes handle.  Raises if the .so is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SagaError(
                "libsaga_b200.so not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback)")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def check(rc, exc_invalid=ValueError):
    """Map a status code to the exception the reference's callers expect:
    invalid arguments -> ValueError (librosa ParameterError is a ValueError),
    anything else -> SagaError."""
    if rc == SAGA_OK:
        return
    msg = lib().saga_last_error_string().decode("utf-8", "replace")
    if rc == SAGA_ERR_INVALID:
        raise exc_invalid(msg)
    if rc == SAGA_ERR_UNSUPPORTED:
        raise SagaUnsupported(msg)
    raise SagaError("saga_b200 error %d: %s" % (rc, msg))
