"""Batched entry points over the C ABI (include/saga_b200.h).

torch is the carrier only: it owns device memory and the stream; every
arithmetic step is a call into libsaga_b200.so.  Tensors returned as
"[..., bins, frames]" are strided views of FRAME-MAJOR storage
([..., frames, pitch], bins contiguous) -- i.e. Fortran order, the layout
librosa.stft itself returns.
"""
import contextlib
import ctypes as C
import os

import numpy as np
import torch

from . import _lib
from .cqt_plan import CqtPlan, ParameterError  # noqa: F401


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _stream(t=None):
    """The current stream OF THE TENSOR'S DEVICE (not of whichever device happens to be current)."""
    return C.c_void_p(torch.cuda.current_stream(None if t is None else t.device).cuda_stream)


def _dev_index(device=None):
    if device is None:
        return torch.cuda.current_device()
    d = torch.device(device)
    return d.index if d.index is not None else torch.cuda.current_device()


@contextlib.contextmanager
def _on(t, plan=None):
    """Make the tensor's device current for the allocations and the launch inside, and refuse a plan whose
    tables live on another device (kernels would read foreign pointers)."""
    if plan is not None and getattr(plan, "device_index", None) not in (None, t.device.index):
        raise ValueError("plan was created for cuda:%d but the data is on %s; use get_*_plan(..., device=...)"
                         % (plan.device_index, t.device))
    with torch.cuda.device(t.device):
        yield


def _require_cuda(t, name):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise TypeError("%s must be a CUDA tensor (there is no CPU path)" % name)


def frame_pitch(n_bins):
    """Row pitch (floats) of frame-major storage: n_bins rounded up to 16 bytes."""
    return (n_bins + 3) & ~3


def bins_frames_view(storage, n_bins):
    """[..., T, pitch] frame-major storage -> [..., n_bins, T] view."""
    return storage[..., :n_bins].transpose(-1, -2)


def storage_of(view):
    """Inverse of bins_frames_view for tensors produced by this module: returns
    the frame-major [..., T, n_bins(+pad)] tensor sharing memory with `view`,
    or None when `view` is not laid out that way."""
    t = view.transpose(-1, -2)
    if t.stride(-1) != 1:
        return None
    return t


# ---------------------------------------------------------------------------
# K1 / K4 plans
# ---------------------------------------------------------------------------
class StftPlan:
    def __init__(self, n_fft, hop_length, center=True, window=None, device=None):
        self.n_fft, self.hop, self.center = int(n_fft), int(hop_length), bool(center)
        self.n_bins = self.n_fft // 2 + 1
        win = None
        if window is not None:
            w = np.ascontiguousarray(np.asarray(window, dtype=np.float32))
            if w.shape != (self.n_fft,):
                raise ValueError("window must have n_fft entries")
            win = w.ctypes.data_as(C.c_void_p)
        h = C.c_void_p()
        self.device_index = _dev_index(device)
        with torch.cuda.device(self.device_index):      # the plan's tables are allocated on the current device
            _lib.check(_lib.lib().saga_stft_plan_create(C.byref(h), self.n_fft, self.hop,
                                                        int(self.center), win))
        self._h = h

    @property
    def handle(self):
        return self._h

    def num_frames(self, n):
        if n <= 0:
            return 0
        if self.center:
            return 1 + n // self.hop
        return 1 + (n - self.n_fft) // self.hop if n >= self.n_fft else 0

    def __del__(self):
        try:
            if self._h is not None:
                _lib.lib().saga_stft_plan_destroy(self._h)
                self._h = None
        except Exception:
            pass


# Plan cache.  A plan owns device tables, so the key carries the DEVICE it was built on and the PROCESS that
# built it: a worker forked by the reference's `Pool(...)` (training.py:623) must not reuse (or destroy) handles
# that belong to its parent's CUDA context.
_plans = {}
_tables = {}


def _forget_foreign(cache):
    pid = os.getpid()
    for k in [k for k in cache if k[0] != pid]:
        v = cache.pop(k)
        if hasattr(v, "_h"):
            v._h = None          # never call *_destroy on another process's handle


def _cached_plan(key, device, make):
    idx = _dev_index(device)
    k = (os.getpid(), idx) + key
    plan = _plans.get(k)
    if plan is None:
        _forget_foreign(_plans)
        plan = make(idx)
        _plans[k] = plan
    return plan


def get_stft_plan(n_fft, hop_length, center=True, device=None):
    return _cached_plan(("stft", int(n_fft), int(hop_length), bool(center)), device,
                        lambda idx: StftPlan(n_fft, hop_length, center, device=idx))


def get_cqt_plan(sr, hop_length, fmin, n_bins, bins_per_octave, filter_scale=2, device=None):
    def make(idx):
        with torch.cuda.device(idx):
            plan = CqtPlan(sr, hop_length, fmin, n_bins, bins_per_octave, filter_scale=filter_scale)
        plan.device_index = idx
        return plan
    return _cached_plan(("cqt", sr, int(hop_length), float(fmin), int(n_bins), int(bins_per_octave), filter_scale),
                        device, make)


def _clip_table(wav, lens):
    """(wav2d, offsets int64 dev, lens int64 dev, max_len host)."""
    _require_cuda(wav, "wav")
    if wav.dtype != torch.float32:
        wav = wav.float()
    if wav.dim() == 1:
        wav = wav.unsqueeze(0)
    if wav.dim() != 2 or wav.stride(1) != 1:
        wav = wav.contiguous()
    n_clips, width = wav.shape
    if lens is None:
        # the offset / length tables of a dense batch depend on its geometry only: built once per
        # (process, device, geometry) instead of three torch launches per call
        key = (os.getpid(), wav.device.index, n_clips, wav.stride(0), width)
        tab = _tables.get(key)
        if tab is None:
            _forget_foreign(_tables)
            if len(_tables) > 256:
                _tables.clear()
            tab = (torch.arange(n_clips, device=wav.device, dtype=torch.int64) * wav.stride(0),
                   torch.full((n_clips,), width, device=wav.device, dtype=torch.int64))
            _tables[key] = tab
        return wav, tab[0], tab[1], width
    offs = torch.arange(n_clips, device=wav.device, dtype=torch.int64) * wav.stride(0)
    if lens is None:
        max_len = width
        lens_dev = torch.full((n_clips,), width, device=wav.device, dtype=torch.int64)
    else:
        lens_host = np.asarray(lens.cpu() if isinstance(lens, torch.Tensor) else lens, dtype=np.int64)
        if lens_host.shape != (n_clips,) or (lens_host > width).any() or (lens_host < 0).any():
            raise ValueError("lens must be [n_clips] with 0 <= len <= wav.shape[1]")
        max_len = int(lens_host.max()) if n_clips else 0
        lens_dev = torch.as_tensor(lens_host, device=wav.device)
    return wav, offs, lens_dev, max_len


def stft_batch(wav, plan, lens=None, want_phase=False, want_complex=False, want_max=True):
    """K1.  wav: CUDA float32 [clips, samples] (or [samples]); ragged clips via
    `lens`.  Returns a dict:
        mag        [clips, n_bins, T] float32 view (frame-major storage)
        phase / F  complex64 views when requested
        frame_max  [clips, T],  clip_max [clips]  (clip_max == reference ref_mag)
    """
    wav, offs, lens_dev, max_len = _clip_table(wav, lens)
    n_clips = wav.shape[0]
    T = plan.num_frames(max_len)
    P = frame_pitch(plan.n_bins)
    dev = wav.device
    alloc = torch.empty if lens is None else torch.zeros
    mag = alloc((n_clips, T, P), device=dev, dtype=torch.float32)
    ph = alloc((n_clips, T, P, 2), device=dev, dtype=torch.float32) if want_phase else None
    cx = alloc((n_clips, T, P, 2), device=dev, dtype=torch.float32) if want_complex else None
    fmax = alloc((n_clips, max(T, 1)), device=dev, dtype=torch.float32) if want_max else None
    cmax = torch.zeros((n_clips,), device=dev, dtype=torch.float32) if want_max else None
    with _on(wav, plan):
        _lib.check(_lib.lib().saga_stft_exec(plan.handle, _ptr(wav), _ptr(offs), _ptr(lens_dev), n_clips,
                                             max_len, _ptr(mag), _ptr(ph), _ptr(cx), P, T * P,
                                             _ptr(fmax), _ptr(cmax), _stream(wav)))
    out = {"mag": bins_frames_view(mag, plan.n_bins), "mag_storage": mag}
    if want_phase:
        out["phase_storage"] = torch.view_as_complex(ph)
        out["phase"] = bins_frames_view(out["phase_storage"], plan.n_bins)
    if want_complex:
        out["F_storage"] = torch.view_as_complex(cx)
        out["F"] = bins_frames_view(out["F_storage"], plan.n_bins)
    if want_max:
        out["frame_max"], out["clip_max"] = fmax[:, :T], cmax
    return out


def istft_batch(plan, F=None, mag=None, phase=None, n_bins=None, frame0=None, n_frames=None):
    """K4 on frame-major storage [clips, T, P] (rows = frames).  Either complex
    `F`, or float `mag` and complex unit-phasor `phase` with identical strides.
    Returns [clips, hop*(T-1)] (centred) float32.
    frame0 (int32 device tensor [clips]) + n_frames: invert only rows [frame0[c], frame0[c] + n_frames) of every clip
    (saga_istft_rows_exec); the caller guarantees frame0[c] + n_frames <= T."""
    n_bins = plan.n_bins if n_bins is None else n_bins
    if n_bins != plan.n_bins:
        raise ValueError("spectrogram has %d bins, plan expects %d" % (n_bins, plan.n_bins))

    def prep(x, dtype):
        _require_cuda(x, "spectrogram")
        if x.dim() == 2:
            x = x.unsqueeze(0)
        if x.dtype != dtype:
            x = x.to(dtype)
        if x.stride(2) != 1 or x.shape[2] < n_bins:
            raise ValueError("expected frame-major storage [clips, T, P>=n_bins]")
        if x.shape[0] > 1 and x.stride(0) < x.stride(1) * x.shape[1]:
            x = x.contiguous()
        return x

    if F is not None:
        s = prep(F, torch.complex64)
        args = (_ptr(torch.view_as_real(s)), None, None)
    else:
        s = prep(mag, torch.float32)
        p = prep(phase, torch.complex64)
        if s.stride() != p.stride():
            s, p = s.contiguous(), p.contiguous()
        args = (None, _ptr(s), _ptr(torch.view_as_real(p)))
    n_clips, T, _ = s.shape
    pitch = s.stride(1) if T > 1 else s.shape[2]
    cstride = s.stride(0) if n_clips > 1 else T * pitch
    Tn = T if frame0 is None else int(n_frames)
    if frame0 is not None and not (0 < Tn <= T):
        raise ValueError("n_frames must be in 1..T")
    out_len = plan.hop * (Tn - 1) + (0 if plan.center else plan.n_fft)
    wav = torch.empty((n_clips, max(out_len, 0)), device=s.device, dtype=torch.float32)
    with _on(s, plan):
        if frame0 is None:
            _lib.check(_lib.lib().saga_istft_exec(plan.handle, args[0], args[1], args[2], n_clips, T, pitch,
                                                  cstride, _ptr(wav), wav.stride(0), _stream(s)))
        else:
            f0 = frame0.to(device=s.device, dtype=torch.int32).contiguous()
            if f0.shape != (n_clips,):
                raise ValueError("frame0 must be [clips]")
            _lib.check(_lib.lib().saga_istft_rows_exec(plan.handle, args[0], args[1], args[2], n_clips, _ptr(f0), Tn, pitch,
                                                       cstride, _ptr(wav), wav.stride(0), _stream(s)))
    return wav


# ---------------------------------------------------------------------------
# K2
# ---------------------------------------------------------------------------
_workspaces = {}


def _workspace(nbytes, device):
    key = (os.getpid(), device.index if device.index is not None else torch.cuda.current_device())
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty((nbytes + 255) // 256 * 256, device=device, dtype=torch.uint8)
        _workspaces[key] = ws
    return ws


def cqt_batch(wav, plan, lens=None, want_complex=False, impl=0, fill=None):
    """K2.  Returns dict(mag=[clips, n_bins, T] view, C=complex view if requested).
    `fill` (tests): value the outputs are set to before the call, so that an element the kernels
    failed to write cannot hide behind stale allocator contents."""
    wav, offs, lens_dev, max_len = _clip_table(wav, lens)
    n_clips = wav.shape[0]
    lib = _lib.lib()
    T = plan.num_frames(max_len)
    P = frame_pitch(plan.n_bins)
    dev = wav.device
    alloc = torch.empty if lens is None else torch.zeros
    mag = alloc((n_clips, T, P), device=dev, dtype=torch.float32)
    cx = alloc((n_clips, T, P, 2), device=dev, dtype=torch.float32) if want_complex else None
    if fill is not None:
        mag.fill_(fill)
        if cx is not None:
            cx.fill_(fill)
    nbytes = lib.saga_cqt_workspace_bytes(plan.handle, n_clips, max_len)
    ws = _workspace(nbytes, dev)
    with _on(wav, plan):
        _lib.check(lib.saga_cqt_exec(plan.handle, _ptr(wav), _ptr(offs), _ptr(lens_dev) if lens is not None else None,
                                     n_clips, max_len,
                                     _ptr(mag), _ptr(cx), P, T * P, _ptr(ws), ws.numel(), impl, _stream(wav)),
                   ParameterError)
    out = {"mag": bins_frames_view(mag, plan.n_bins), "mag_storage": mag}
    if want_complex:
        out["C"] = bins_frames_view(torch.view_as_complex(cx), plan.n_bins)
    return out


def cqt_peak_batch(wav, plan, col_lo, col_hi, lens=None):
    """saga_cqt_peak_exec: per clip, max |C| over every bin and the frames col_lo[c] <= t < min(col_hi[c], T_c)
    (0 for an empty range) -- np.max of `C[:, lo:hi]` without the image.  col_lo / col_hi: int sequences or tensors
    [clips].  Returns a float32 CUDA tensor [clips]."""
    wav, offs, lens_dev, max_len = _clip_table(wav, lens)
    n_clips = wav.shape[0]
    lib = _lib.lib()
    dev = wav.device

    def cols(x, name):
        t = torch.as_tensor(np.ascontiguousarray(x, dtype=np.int32), device=dev) \
            if not isinstance(x, torch.Tensor) else x.to(device=dev, dtype=torch.int32).contiguous()
        if t.shape != (n_clips,):
            raise ValueError("%s must be [clips]" % name)
        return t
    lo, hi = cols(col_lo, "col_lo"), cols(col_hi, "col_hi")
    peak = torch.empty((n_clips,), device=dev, dtype=torch.float32)
    nbytes = lib.saga_cqt_peak_workspace_bytes(plan.handle, n_clips, max_len)
    ws = _workspace(nbytes, dev)
    with _on(wav, plan):
        _lib.check(lib.saga_cqt_peak_exec(plan.handle, _ptr(wav), _ptr(offs), _ptr(lens_dev) if lens is not None else None,
                                          n_clips, max_len, _ptr(lo), _ptr(hi), _ptr(peak), _ptr(ws), ws.numel(),
                                          _stream(wav)), ParameterError)
    return peak


def cqt_frames_batch(wav, plan, frame_first, frame_count=8, lens=None, out=None):
    """saga_cqt_frames_exec: only columns [frame_first[c], frame_first[c] + frame_count) of each clip's CQT
    magnitude (what slice_C + _resize keep).  Returns compact frame-major storage [clips, frame_count, P]
    (`out`: write into this preallocated contiguous slice instead)."""
    wav, offs, lens_dev, max_len = _clip_table(wav, lens)
    n_clips = wav.shape[0]
    lib = _lib.lib()
    P = frame_pitch(plan.n_bins)
    dev = wav.device
    first = torch.as_tensor(np.ascontiguousarray(frame_first, dtype=np.int32), device=dev) \
        if not isinstance(frame_first, torch.Tensor) else frame_first.to(device=dev, dtype=torch.int32).contiguous()
    if first.shape != (n_clips,):
        raise ValueError("frame_first must be [clips]")
    if out is None:
        out = torch.empty((n_clips, int(frame_count), P), device=dev, dtype=torch.float32)
    elif out.shape != (n_clips, int(frame_count), P) or not out.is_contiguous() or out.dtype != torch.float32:
        raise ValueError("out must be contiguous float32 [clips, frame_count, %d]" % P)
    nbytes = lib.saga_cqt_workspace_bytes(plan.handle, n_clips, max_len)
    ws = _workspace(nbytes, dev)
    with _on(wav, plan):
        _lib.check(lib.saga_cqt_frames_exec(plan.handle, _ptr(wav), _ptr(offs), _ptr(lens_dev) if lens is not None else None,
                                            n_clips, max_len, _ptr(first), int(frame_count), _ptr(out), P,
                                            int(frame_count) * P, _ptr(ws), ws.numel(), _stream(wav)), ParameterError)
    return out


def cqt_cascade_shared(wav, plan, lens=None):
    """Phase 1 of saga_cqt_frames_shared_exec: decimation cascade + reflect margins of the whole batch, once, for every
    plan of `plan.geometry()`.  Returns the token `cqt_frames_from_cascade` takes; the (per-device, shared) workspace
    must not be used by another CQT call in between."""
    wav, offs, lens_dev, max_len = _clip_table(wav, lens)
    n_clips = wav.shape[0]
    lib = _lib.lib()
    nbytes = lib.saga_cqt_workspace_bytes(plan.handle, n_clips, max_len)
    ws = _workspace(nbytes, wav.device)
    lens_ptr = _ptr(lens_dev) if lens is not None else None
    with _on(wav, plan):
        _lib.check(lib.saga_cqt_frames_shared_exec(plan.handle, _ptr(wav), _ptr(offs), lens_ptr, n_clips, max_len, 1, 0, n_clips,
                                                   None, 0, None, 0, 0, _ptr(ws), ws.numel(), _stream(wav)), ParameterError)
    return dict(wav=wav, offs=offs, lens_ptr=lens_ptr, n_clips=n_clips, max_len=max_len, ws=ws, geometry=plan.geometry(),
                keep=lens_dev)


def cqt_frames_from_cascade(token, plan, clip_first, n_clips, frame_first, frame_count, out):
    """Phase 2: `frame_count` columns from frame_first[c] for clips [clip_first, clip_first + n_clips) of the cascade
    batch, with THIS plan's bank.  frame_first: int32 device tensor [n_clips]; out: contiguous [n_clips, frame_count, P]."""
    if plan.geometry() != token["geometry"]:
        raise ValueError("plan geometry differs from the cascade's")
    P = frame_pitch(plan.n_bins)
    if out.shape != (n_clips, int(frame_count), P) or not out.is_contiguous() or out.dtype != torch.float32:
        raise ValueError("out must be contiguous float32 [clips, frame_count, %d]" % P)
    first = frame_first.to(device=out.device, dtype=torch.int32).contiguous()
    if first.shape != (n_clips,):
        raise ValueError("frame_first must be [clips]")
    wav = token["wav"]
    with _on(wav, plan):
        _lib.check(_lib.lib().saga_cqt_frames_shared_exec(
            plan.handle, _ptr(wav), _ptr(token["offs"]), token["lens_ptr"], token["n_clips"], token["max_len"], 2,
            int(clip_first), int(n_clips), _ptr(first), int(frame_count), _ptr(out), P, int(frame_count) * P,
            _ptr(token["ws"]), token["ws"].numel(), _stream(wav)), ParameterError)
    return out


def cqt_frames_from_cascade_multi(token, plans, clip_first, clip_count, frame_first, frame_count, out):
    """Phase 2 for several plans of the cascade's geometry in one call (saga_cqt_frames_shared_multi_exec): plan i
    contracts clips [clip_first[i], clip_first[i] + clip_count[i]) of the cascade batch; together they must cover every
    clip once.  frame_first: int32 device tensor [batch]; out: contiguous [batch, frame_count, P]."""
    n = token["n_clips"]
    P = frame_pitch(plans[0].n_bins)
    for pl in plans:
        if pl.geometry() != token["geometry"]:
            raise ValueError("plan geometry differs from the cascade's")
    if out.shape != (n, int(frame_count), P) or not out.is_contiguous() or out.dtype != torch.float32:
        raise ValueError("out must be contiguous float32 [batch, frame_count, %d]" % P)
    first = frame_first.to(device=out.device, dtype=torch.int32).contiguous()
    if first.shape != (n,):
        raise ValueError("frame_first must be [batch]")
    cf = np.ascontiguousarray(clip_first, dtype=np.int32)
    cc = np.ascontiguousarray(clip_count, dtype=np.int32)
    order = np.argsort(cf)
    if len(cf) != len(plans) or int(cc.sum()) != n or np.any(np.cumsum(cc[order]) - cc[order] != cf[order]):
        raise ValueError("the plans' clip ranges must tile the batch")
    handles = (C.c_void_p * len(plans))(*[pl.handle for pl in plans])
    wav = token["wav"]
    with _on(wav, plans[0]):
        _lib.check(_lib.lib().saga_cqt_frames_shared_multi_exec(
            handles, len(plans), cf.ctypes.data_as(C.c_void_p), cc.ctypes.data_as(C.c_void_p), _ptr(wav), _ptr(token["offs"]),
            token["lens_ptr"], n, token["max_len"], _ptr(first), int(frame_count), _ptr(out), P, int(frame_count) * P,
            _ptr(token["ws"]), token["ws"].numel(), _stream(wav)), ParameterError)
    return out


# ---------------------------------------------------------------------------
# K3
# ---------------------------------------------------------------------------
def subtract_db_batch(win, guesses, offset_frames, n_bins, overkill=None, guess_ref=None,
                      ref_init=None, guess_frames=None, normalize=True, relu=True, want_D=True,
                      amin=1e-5, top_db=80.0, frame_max=None, D_out=None):
    """K3 on frame-major storage.
        win      [W, T, P] float32, modified in place (P = frame pitch >= n_bins)
        frame_max optional [W, >=T] per-frame maxima of `win` (stft_batch's by-product)
        guesses  [W, S, Tg, P] float32 (S sequential steps per window)
        offset_frames [W, S] int32 column offsets
    Returns (D storage [W, T, P] or None, ref [W] = max of each final window)."""
    _require_cuda(win, "win")
    if win.dim() != 3 or win.stride(2) != 1 or win.stride(1) < n_bins or win.dtype != torch.float32:
        raise ValueError("win must be frame-major float32 storage [W, T, P]")
    W, T, _ = win.shape
    P = win.stride(1)
    if W > 1 and win.stride(0) < T * P:
        raise ValueError("overlapping windows")
    S = 0
    Tg = 0
    if guesses is not None:
        _require_cuda(guesses, "guesses")
        if guesses.dim() != 4 or guesses.stride(3) != 1 or guesses.stride(2) != P or not guesses.is_contiguous():
            raise ValueError("guesses must be contiguous [W, S, Tg, P] with the window's pitch")
        S, Tg = guesses.shape[1], guesses.shape[2]
        offset_frames = offset_frames.to(device=win.device, dtype=torch.int32).contiguous()
    f32 = lambda x: None if x is None else x.to(device=win.device, dtype=torch.float32).contiguous()
    overkill, guess_ref, ref_init = f32(overkill), f32(guess_ref), f32(ref_init)
    if guess_frames is not None:
        guess_frames = guess_frames.to(device=win.device, dtype=torch.int32).contiguous()
    D = None
    if want_D:
        D = D_out if D_out is not None else torch.empty_strided(win.shape, win.stride(), device=win.device,
                                                               dtype=win.dtype)
        if D.stride() != win.stride() or D.shape != win.shape:
            raise ValueError("D_out must have the window tensor's shape and strides")
    fm_stride = 0
    if frame_max is not None:
        _require_cuda(frame_max, "frame_max")
        if frame_max.dim() != 2 or frame_max.shape[0] != W or frame_max.shape[1] < T or \
                frame_max.stride(1) != 1 or frame_max.dtype != torch.float32:
            raise ValueError("frame_max must be float32 [W, >=T]")
        fm_stride = frame_max.stride(0)
    ref = torch.empty((W,), device=win.device, dtype=torch.float32)
    flags = (_lib.SUB_NORMALIZE if normalize else 0) | (_lib.SUB_RELU if relu else 0)
    with _on(win):
        _lib.check(_lib.lib().saga_subtract_db_exec(
            _ptr(win), None, win.stride(0) if W > 1 else T * P, _ptr(guesses), None,
            Tg * P, _ptr(guess_frames), Tg, _ptr(offset_frames), _ptr(overkill), _ptr(guess_ref),
            _ptr(ref_init), _ptr(frame_max), fm_stride, flags, _ptr(D), _ptr(ref), W, S, n_bins, T, P,
            float(amin), float(top_db if top_db is not None else -1.0), _stream(win)))
    return D, ref


def amplitude_to_db_batch(mag_storage, n_bins, ref=None, amin=1e-5, top_db=80.0):
    """librosa.amplitude_to_db on frame-major storage [clips, T, P]; ref: [clips]
    tensor (negative entries => the clip's own max) or None (=> max)."""
    _require_cuda(mag_storage, "mag")
    m = mag_storage
    if m.dim() == 2:
        m = m.unsqueeze(0)
    if m.stride(2) != 1 or m.dtype != torch.float32:
        raise ValueError("mag must be frame-major float32 storage")
    n_clips, T, _ = m.shape
    P = m.stride(1)
    D = torch.empty_strided(m.shape, m.stride(), device=m.device, dtype=torch.float32)
    if ref is not None:
        ref = ref.to(device=m.device, dtype=torch.float32).contiguous()
    with _on(m):
        _lib.check(_lib.lib().saga_amplitude_to_db_exec(
            _ptr(m), _ptr(D), _ptr(ref), n_clips, n_bins, T, P, m.stride(0) if n_clips > 1 else T * P,
            float(amin), float(top_db if top_db is not None else -1.0), _stream(m)))
    return D


# ---------------------------------------------------------------------------
# K0: PCM ingest
# ---------------------------------------------------------------------------
def pcm16_absmax(pcm, channel_stride=1, out=None):
    """np.abs(pcm).max() per clip (int32 CUDA tensor) of int16 PCM [clips, samples*channel_stride];
    channel_stride=2 looks at the left channel of interleaved stereo (util_audio.py:894 `[::2]`)."""
    _require_cuda(pcm, "pcm")
    if pcm.dtype != torch.int16 or pcm.dim() != 2 or pcm.stride(1) != 1:
        raise TypeError("pcm must be a [clips, samples] int16 CUDA tensor with contiguous rows")
    n_clips, width = pcm.shape
    n = (width + channel_stride - 1) // channel_stride
    if out is None:
        out = torch.empty((n_clips,), device=pcm.device, dtype=torch.int32)
    if n_clips == 0:
        return out
    if n == 0:
        return out.zero_()
    with _on(pcm):
        _lib.check(_lib.lib().saga_pcm16_absmax_exec(_ptr(pcm), pcm.stride(0), channel_stride, n_clips, n,
                                                     _ptr(out), _stream(pcm)))
    return out


def pcm16_to_wave(pcm, mul=1.0, div=32768.0, channel_stride=1, out=None):
    """float32( (float64(pcm) * mul) / div ) per clip: the one scaling the reference applies to its PCM
    (util_audio.py:776-781 for fluidsynth renders, soundfile's /32768 for files), bit-exact.
    mul / div: python floats, or per-clip CUDA tensors (float64; div may also be the int32 tensor
    pcm16_absmax returns, i.e. `/ np.abs(wf).max()`)."""
    _require_cuda(pcm, "pcm")
    if pcm.dtype != torch.int16 or pcm.dim() != 2 or pcm.stride(1) != 1:
        raise TypeError("pcm must be a [clips, samples] int16 CUDA tensor with contiguous rows")
    n_clips, width = pcm.shape
    n = (width + channel_stride - 1) // channel_stride
    if out is None:
        out = torch.empty((n_clips, n), device=pcm.device, dtype=torch.float32)
    elif out.dtype != torch.float32 or out.shape != (n_clips, n) or out.stride(1) != 1:
        raise ValueError("out must be float32 [clips, samples] with contiguous rows")
    if n_clips == 0 or n == 0:
        return out
    mul_t = div_t = peak_t = None
    mul_all = div_all = 1.0
    if isinstance(mul, torch.Tensor):
        mul_t = mul.to(device=pcm.device, dtype=torch.float64).contiguous()
    else:
        mul_all = float(mul)
    if isinstance(div, torch.Tensor):
        if div.dtype == torch.int32:
            peak_t = div.to(device=pcm.device).contiguous()
        else:
            div_t = div.to(device=pcm.device, dtype=torch.float64).contiguous()
    else:
        div_all = float(div)
    for t in (mul_t, div_t, peak_t):
        if t is not None and t.shape != (n_clips,):
            raise ValueError("per-clip scales must be [clips]")
    with _on(pcm):
        _lib.check(_lib.lib().saga_pcm16_ingest_exec(_ptr(pcm), pcm.stride(0), channel_stride, _ptr(out), out.stride(0),
                                                     n_clips, n, _ptr(mul_t), _ptr(div_t), _ptr(peak_t),
                                                     mul_all, div_all, _stream(pcm)))
    return out


def launch_count():
    return int(_lib.lib().saga_launch_count())


@contextlib.contextmanager
def options(**kv):
    """Temporarily set library switches (saga_set_option), e.g. `with ops.options(SAGA_SUB_NO_CLUSTER="1"):`.
    The previous values are restored on exit; None unsets."""
    lib = _lib.lib()
    old = {k: lib.saga_get_option(k.encode()) for k in kv}
    try:
        for k, v in kv.items():
            _lib.check(lib.saga_set_option(k.encode(), None if v is None else str(v).encode()))
        yield
    finally:
        for k, v in old.items():
            lib.saga_set_option(k.encode(), v)


# ---------------------------------------------------------------------------
# K5: classifier feature gather
# ---------------------------------------------------------------------------
def compress_bands_batch(mag_storage, n_bins, edges, inv_scale=None, out=None):
    """util_audio.compress_bands on frame-major storage [clips, T, P]: returns
    frame-major [clips, T, Pb] whose [..., :n_bands].transpose is [bands, frames]."""
    _require_cuda(mag_storage, "mag")
    m = mag_storage if mag_storage.dim() == 3 else mag_storage.unsqueeze(0)
    if m.stride(2) != 1 or m.dtype != torch.float32:
        raise ValueError("mag must be frame-major float32 storage")
    edges = np.ascontiguousarray(np.asarray(edges, dtype=np.int32))
    n_bands = len(edges) - 1
    if edges[-1] > n_bins:
        raise ValueError("band edge beyond the spectrum")
    n_clips, T, _ = m.shape
    P = m.stride(1) if T > 1 else m.shape[2]
    Pb = frame_pitch(n_bands)
    if out is None:
        out = torch.empty((n_clips, T, Pb), device=m.device, dtype=torch.float32)
    elif out.shape != (n_clips, T, Pb) or not out.is_contiguous():
        raise ValueError("out must be contiguous [clips, T, %d]" % Pb)
    if inv_scale is not None:
        inv_scale = inv_scale.to(device=m.device, dtype=torch.float32).contiguous()
    with _on(m):
        _lib.check(_lib.lib().saga_compress_bands_exec(
            _ptr(m), _ptr(out), edges.ctypes.data_as(C.c_void_p), n_bands, n_clips, T, P,
            m.stride(0) if n_clips > 1 else T * P, Pb, T * Pb, _ptr(inv_scale), _stream(m)))
    return out


def resize_indices(t, target):
    """Source column of every output column of util_audio._resize (util_audio.py:384-409);
    -1 marks the all-zero result of an empty slice."""
    if t == 0:
        return np.full(target, -1, dtype=np.int32)
    if t == target:
        return np.arange(target, dtype=np.int32)
    if t < 3:
        return np.array([0] + [t - 1] * (target - 1), dtype=np.int32)
    if t < target:
        lim = min(1, int(np.round(t / 3)))
        reps = int(np.floor((target - 2 * lim) / (t - 2 * lim)))
        mid = list(range(lim, t - lim)) * reps
        tail = target - len(mid) - lim
        return np.array(list(range(lim)) + mid + list(range(t - tail, t)), dtype=np.int32)
    return np.arange(target, dtype=np.int32)


def short_window_features(mag_st, phase_st, src_frames, band_min, n_rows, n_bins, inv_ref=1.0,
                          want_lin=True, want_log=True, want_phase=False):
    """One launch for resize + section_power + normalisations (training.py:337-363).
    mag_st / phase_st: frame-major [T, P] storage of ONE window; src_frames: int32
    window-frame index per output column (-1 = zeros).  Returns a dict of
    [n_rows, n_cols] views (lin, log, phase)."""
    _require_cuda(mag_st, "mag")
    src = torch.as_tensor(np.asarray(src_frames, dtype=np.int32), device=mag_st.device)
    n_cols = int(src.numel())
    P = mag_st.stride(0) if mag_st.shape[0] > 1 else mag_st.shape[1]
    Po = frame_pitch(n_rows)
    mk = lambda on: torch.zeros((n_cols, Po), device=mag_st.device, dtype=torch.float32) if on else None
    lin, log, pha = mk(want_lin), mk(want_log), mk(want_phase)
    ph_ptr = None
    if want_phase:
        if phase_st is None or phase_st.stride(0) != mag_st.stride(0):
            raise ValueError("phase storage must match the magnitude storage")
        ph_ptr = _ptr(torch.view_as_real(phase_st))
    with _on(mag_st):
        _lib.check(_lib.lib().saga_short_window_exec(
            _ptr(mag_st), ph_ptr, _ptr(src), n_cols, int(band_min), int(n_rows), int(n_bins), P, float(inv_ref),
            _ptr(lin), _ptr(log), _ptr(pha), Po, _stream(mag_st)))
    view = lambda x: None if x is None else x[:, :n_rows].transpose(0, 1)
    return {"lin": view(lin), "log": view(log), "phase": view(pha)}


def short_window_features_batch(mag_st, phase_st, src_frames, band_min, n_rows, n_bins, inv_ref,
                                want_lin=True, want_log=True, want_phase=False):
    """saga_short_window_batch_exec: the short-window block of training.py:337-363 for W windows at once.
    mag_st [W, T, P] float32 (phase_st complex64, same strides); src_frames int32 [W, n_cols] (host or device;
    -1 = zeros); band_min: int or int32 [W]; inv_ref: float or float32 [W] device.  Returns a dict of
    [W, n_rows, n_cols] views (lin, log, phase)."""
    _require_cuda(mag_st, "mag")
    W, T, _ = mag_st.shape
    dev = mag_st.device
    src = torch.as_tensor(np.ascontiguousarray(src_frames, dtype=np.int32), device=dev) \
        if not isinstance(src_frames, torch.Tensor) else src_frames.to(device=dev, dtype=torch.int32).contiguous()
    n_cols = int(src.shape[1])
    P = mag_st.stride(1) if T > 1 else mag_st.shape[2]
    cs = mag_st.stride(0) if W > 1 else T * P
    Po = frame_pitch(n_rows)
    mk = lambda on: torch.empty((W, n_cols, Po), device=dev, dtype=torch.float32) if on else None
    lin, log, pha = mk(want_lin), mk(want_log), mk(want_phase)
    ph_ptr = None
    if want_phase:
        if phase_st is None or phase_st.stride() != mag_st.stride():
            raise ValueError("phase storage must match the magnitude storage")
        ph_ptr = _ptr(torch.view_as_real(phase_st))
    if isinstance(band_min, torch.Tensor):
        bm_dev, bm_all = band_min.to(device=dev, dtype=torch.int32).contiguous(), 0
    else:
        bm_dev, bm_all = (None, int(band_min)) if np.isscalar(band_min) else \
            (torch.as_tensor(np.asarray(band_min, dtype=np.int32), device=dev), 0)
    ir_dev, ir_all = (None, float(inv_ref)) if not isinstance(inv_ref, torch.Tensor) else \
        (inv_ref.to(device=dev, dtype=torch.float32).contiguous(), 1.0)
    with _on(mag_st):
        _lib.check(_lib.lib().saga_short_window_batch_exec(
            _ptr(mag_st), ph_ptr, cs, P, _ptr(src), n_cols, _ptr(bm_dev), bm_all, int(n_rows), int(n_bins),
            _ptr(ir_dev), ir_all, _ptr(lin), _ptr(log), _ptr(pha), Po, n_cols * Po, W, _stream(mag_st)))
    view = lambda x: None if x is None else x[:, :, :n_rows].transpose(1, 2)
    return {"lin": view(lin), "log": view(log), "phase": view(pha)}


def gather_frames_batch(storage, n_bins, src_frames, scale=None, out=None):
    """saga_gather_frames_exec: out[w][:, j] = in[w][:, src[w, j]] * scale[w] (src -1 => zeros): `C[:, s:t]` +
    `_resize` + `/ ref` of util_audio.slice_C for a batch.  storage [W, T, P] frame-major; returns the
    [W, n_bins, n_cols] view of frame-major [W, n_cols, Pout] storage."""
    _require_cuda(storage, "storage")
    W, T, _ = storage.shape
    dev = storage.device
    src = torch.as_tensor(np.ascontiguousarray(src_frames, dtype=np.int32), device=dev) \
        if not isinstance(src_frames, torch.Tensor) else src_frames.to(device=dev, dtype=torch.int32).contiguous()
    n_cols = int(src.shape[1])
    P = storage.stride(1) if T > 1 else storage.shape[2]
    cs = storage.stride(0) if W > 1 else T * P
    Po = frame_pitch(n_bins)
    if out is None:
        out = torch.empty((W, n_cols, Po), device=dev, dtype=torch.float32)
    elif out.shape != (W, n_cols, Po) or not out.is_contiguous():
        raise ValueError("out must be contiguous [W, n_cols, %d]" % Po)
    if scale is not None:
        scale = scale.to(device=dev, dtype=torch.float32).contiguous()
    with _on(storage):
        _lib.check(_lib.lib().saga_gather_frames_exec(_ptr(storage), _ptr(src), _ptr(scale), _ptr(out), W, n_cols,
                                                      int(n_bins), P, cs, Po, n_cols * Po, _stream(storage)))
    return out[:, :, :n_bins].transpose(1, 2)


def spectral_flatness_batch(mag_storage, n_bins, amin=1e-10):
    """librosa.feature.spectral_flatness(power=2) per frame: [clips, T]."""
    m = mag_storage if mag_storage.dim() == 3 else mag_storage.unsqueeze(0)
    _require_cuda(m, "mag")
    n_clips, T, _ = m.shape
    P = m.stride(1) if T > 1 else m.shape[2]
    out = torch.empty((n_clips, T), device=m.device, dtype=torch.float32)
    with _on(m):
        _lib.check(_lib.lib().saga_spectral_flatness_exec(
            _ptr(m), _ptr(out), n_clips, n_bins, T, P, m.stride(0) if n_clips > 1 else T * P, float(amin), _stream(m)))
    return out
