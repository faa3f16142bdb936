"""Batched song setup (SongBatch, training.py:265-284) on 32 seeded songs of 60-300 s (ragged), with a per-stage
breakdown, the constant-Q peak mode against materialise-then-reduce, and the whole batch against the per-song class
loop of tests/ref_loop.py:74-94.

    python profiles/microbench/song_setup_bench.py [n_songs]

The songs are synth.piano_batch at the longest length, cut by `lens`: 32 x 300 s of float32 is 1.7 GB, far larger
than the 126 MB L2, so no stage reads its input from L2 left behind by the previous one.  Times are CUDA events
around 3 calls after a warm-up call of the same shapes (class loop: host clock around one pass ending in a
synchronise, after one warm-up song).  1392/192 algorithmic rate: 50.34 Mflop per frame (SURVEY Appendix B) times the
frames each path contracts: the packed peak mode contracts sum T_c, the whole transform n_songs x T_max."""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import amt_saga_b200  # noqa: E402,F401
from amt_saga_b200 import ops, synth  # noqa: E402
from amt_saga_b200 import util_audio as ua  # noqa: E402
from amt_saga_b200.song_setup import SongBatch  # noqa: E402

MFLOP_192 = 50.34e6
SR = 44100


def gpu_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def timed(fn, n=3):
    fn()
    torch.cuda.synchronize()
    a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    e.record()
    torch.cuda.synchronize()
    return a.elapsed_time(e) / n


def column_max(mag_storage, n_bins, hi):
    """materialise-then-reduce: max over bins, then over frames [0, hi) of each song"""
    fm = mag_storage[..., :n_bins].amax(dim=2)                                        # [S, T_max]
    keep = torch.arange(fm.shape[1], device=fm.device)[None, :] < hi[:, None]
    return torch.where(keep, fm, 0.0).amax(dim=1)


def class_loop(wav, lens):
    """tests/ref_loop.py:74-94 per song with the CUDA class: flatness, mag, three slice_C maxima, section, ref_mag"""
    out = []
    for s in range(len(lens)):
        a = ua.audio_complete(wav[s, :int(lens[s])], 4096)
        flat = a.spectral_flatness()
        a.mag
        T = a.shape[1]
        dur = a._frames_to_seconds(T)
        rc = [float(np.max(a.slice_C(0, dur, T, 8, bins_per_tone=b).cpu().numpy())) for b in (1, 4, 16)]
        a.section(0, None, 258)
        a.midi_tone_to_FFT(60)
        out.append((flat, dur, rc, float(a.ref_mag)))
    return out


def main():
    S = int(sys.argv[1]) if len(sys.argv) > 1 else 32
    torch.cuda.set_device(0)
    res = {"gpu": gpu_line(), "songs": S}
    rng = np.random.default_rng(2026)
    lens = (rng.uniform(60, 300, S) * SR).astype(np.int64)
    lens[0] = 300 * SR                                                                  # the range's both ends
    lens[1] = 60 * SR
    wav = synth.piano_batch(range(S), int(lens.max()), SR, seed_base=31000, device="cuda")
    torch.cuda.synchronize()
    res["seconds_total"] = round(float(lens.sum()) / SR, 1)
    res["input_GB"] = round(wav.numel() * 4 / 1e9, 2)

    b = SongBatch()
    b.setup(wav, lens)                                                                  # warm-up: plans, workspaces
    torch.cuda.synchronize()
    stft = b.stft
    stages = {}
    stages["stft"] = timed(lambda: ops.stft_batch(wav, stft, lens=lens, want_phase=True, want_max=True))
    r = ops.stft_batch(wav, stft, lens=lens, want_phase=True, want_max=True)
    T_dev = torch.as_tensor(b.T, device="cuda")

    def flatness():
        f = ops.spectral_flatness_batch(r["mag_storage"], b.nb).double()
        mask = torch.arange(f.shape[1], device="cuda")[None, :] < T_dev[:, None]
        return torch.where(mask, f, 0.0).sum(1) / T_dev
    stages["flatness"] = timed(flatness)
    lo = np.zeros(S, dtype=np.int32)
    hi = b.ref_cols.astype(np.int32)
    hi_dev = torch.as_tensor(hi, device="cuda")
    names = ("peak_87_12", "peak_348_48", "peak_1392_192")
    for name, plan in zip(names, b.cqt_plans):
        stages[name] = timed(lambda: ops.cqt_peak_batch(wav, plan, lo, hi, lens=lens))
    res["stages_ms"] = {k: round(v, 3) for k, v in stages.items()}

    p192 = b.cqt_plans[2]
    frames_packed = int(sum(p192.num_frames(int(n)) for n in lens))
    frames_padded = S * p192.num_frames(int(lens.max()))
    res["sum_frames_1392_192"] = frames_packed
    res["padded_frames_1392_192"] = frames_padded
    res["peak_1392_192_algorithmic_TFLOPs"] = round(frames_packed * MFLOP_192 / (stages["peak_1392_192"] * 1e-3) / 1e12, 1)

    # packed rows, no image  vs  padded rows, image written, then a column-range max
    cmp = {}
    for name, plan in zip(names, b.cqt_plans):
        t_img = timed(lambda: column_max(ops.cqt_batch(wav, plan, lens=lens)["mag_storage"], plan.n_bins, hi_dev))
        want = column_max(ops.cqt_batch(wav, plan, lens=lens)["mag_storage"], plan.n_bins, hi_dev)
        got = ops.cqt_peak_batch(wav, plan, lo, hi, lens=lens)
        cmp[name] = {"peak_ms": round(stages[name], 3), "cqt_batch_plus_max_ms": round(t_img, 3),
                     "speedup": round(t_img / stages[name], 2), "equal": bool(torch.equal(got, want))}
    cmp["peak_1392_192"]["cqt_batch_algorithmic_TFLOPs_on_padded_frames"] = round(
        frames_padded * MFLOP_192 / (cmp["peak_1392_192"]["cqt_batch_plus_max_ms"] * 1e-3) / 1e12, 1)
    res["peak_vs_materialise"] = cmp
    torch.cuda.empty_cache()

    # the whole batch against the per-song class loop
    res["song_batch_ms"] = round(timed(lambda: b.setup(wav, lens)), 2)
    class_loop(wav[:1], lens[:1])                                                       # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ref = class_loop(wav, lens)
    torch.cuda.synchronize()
    res["class_loop_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
    res["class_loop_over_song_batch"] = round(res["class_loop_ms"] / res["song_batch_ms"], 1)
    b.setup(wav, lens)
    rel = lambda a_, b_: float(np.max(np.abs(np.asarray(a_) - np.asarray(b_)) / np.maximum(np.abs(np.asarray(b_)), 1e-30)))
    res["max_rel_diff_vs_class"] = {
        "flatness": rel(b.flatness, [x[0] for x in ref]),
        "song_dur": rel(b.song_dur, [x[1] for x in ref]),
        "ref_C": rel(b.ref_C, [x[2] for x in ref]),
        "ref_mag": rel(b.ref_mag.double().cpu().numpy(), [x[3] for x in ref])}
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
