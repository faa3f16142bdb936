"""Songs walked through the batched per-note step with half-window slides (SongBatch.slide, training.py:317-328):
W seeded songs of 30-180 s (ragged), one window per song, through steps and slides.

    python profiles/microbench/song_walk_bench.py [--windows 128] [--compare-tree DIR] [--out FILE]

Reports
* the slide kernel (saga_window_slide_exec) for all W windows: CUDA events over 50 launches, against its algorithmic
  bytes 2 h P 12 read + 2 h P 12 written per window (h = 129, P = 2052), as a fraction of the HBM copy peak DESIGN.md
  uses (6 543 GB/s, MEASURED_PEAKS.json).  W x 12.7 MB is far larger than the 126 MB L2;
* a step (wall clock around the host call, synchronised) without slides, and with a slide of a random quarter of the
  windows before it (the slide included in the time);
* microseconds per note against the CUDA class driven window by window (4 songs, 3 notes each);
* bench.py's `per_note_batched` (uniform-length windows, the path this change must not slow) from this tree and, with
  --compare-tree, from another checkout, alternating, in the same run.
The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import amt_saga_b200  # noqa: E402,F401
from amt_saga_b200 import ops, synth  # noqa: E402
from amt_saga_b200 import util_audio as ua  # noqa: E402
from amt_saga_b200.note_step import NoteStepBatch  # noqa: E402
from amt_saga_b200.song_setup import SongBatch  # noqa: E402

SR, HBM_PEAK = 44100, 6543e9


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown (%s)" % q.stderr.strip()[:80]


def notes(rng, W):
    return rng.uniform(0.05, 5.0, W), rng.uniform(0.2, 1.2, W), rng.integers(40, 80, W)


def per_note_batched(tree):
    """bench.py's per-note figure from `tree` (its own build), extras only."""
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    subprocess.run([sys.executable, "-c", "import __graft_entry__ as g; g.build()"], cwd=tree, env=env, check=True,
                   capture_output=True)
    r = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", "10", "--warmup", "3", "--cpu-windows", "0",
                        "--e2e-steps", "3", "--no-ref-shape"], cwd=tree, env=env, capture_output=True, text=True)
    for line in r.stdout.splitlines()[::-1]:
        if line.startswith("{"):
            return json.loads(line).get("per_note_batched")
    return {"error": (r.stderr or r.stdout)[-300:]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=128)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--compare-tree", default=None)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    W = args.windows
    res = {"card": card(), "windows": W}
    rng = np.random.default_rng(1)
    secs = rng.uniform(30.0, 180.0, W)
    lens = (secs * SR).astype(np.int64)
    wav = synth.piano_batch(range(W), int(lens.max()), SR, n_notes=200, seed_base=31000, device=dev)
    b = SongBatch(device=dev).setup(wav, lens)
    win = b.section(np.arange(W), np.zeros(W), 258)
    step = b.load_into(NoteStepBatch(W, device=dev), win)
    res["distinct_window_lengths"] = int(len(np.unique(win.wav_len)))
    guess = synth.piano_batch(range(W), 54277, SR, n_notes=1, seed_base=32000, device=dev)

    # -- the slide kernel alone (rows only), all W windows per launch
    h, P = 129, step.mag.shape[2]
    row0 = np.zeros(W, dtype=np.int64)
    rows = np.full(W, h)
    args_k = (step.mag, step.ph, step.nb, h, np.arange(W), np.arange(W), row0, rows, b.mag, b.phase)
    ops.window_slide_batch(*args_k)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(50):
        ops.window_slide_batch(*args_k)
    ev[1].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1]) / 50
    nbytes = W * 4 * h * P * 12
    res["slide_kernel"] = {"ms": ms, "algorithmic_bytes": nbytes, "TBps": nbytes / (ms * 1e-3) / 1e12,
                           "fraction_of_hbm_peak": nbytes / (ms * 1e-3) / HBM_PEAK}

    # -- steps, with and without a quarter of the windows sliding first (reload: the kernel loop above moved rows)
    win = b.section(np.arange(W), np.zeros(W), 258)
    step = b.load_into(NoteStepBatch(W, device=dev), win)
    for i in range(3):                                          # plans of every pitch, the full and patched iSTFT
        step.step(*notes(np.random.default_rng(100 + i), W), guess)

    def timed(slide):
        r = np.random.default_rng(7)
        torch.cuda.synchronize()
        t0, t_slide = time.perf_counter(), 0.0
        for i in range(args.steps):
            if slide:
                mask = np.zeros(W, dtype=bool)
                mask[r.choice(W, W // 4, replace=False)] = True
                mask &= win.offset_s + 9.0 < lens / SR         # keep the walk inside the songs
                torch.cuda.synchronize()
                t1 = time.perf_counter()
                b.slide(step, win, mask)
                torch.cuda.synchronize()
                t_slide += time.perf_counter() - t1
            step.step(*notes(r, W), guess)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / args.steps * 1e3, t_slide / args.steps * 1e3
    ms_plain, _ = timed(False)
    ms_slide, ms_slide_only = timed(True)
    ms_plain2, _ = timed(False)
    res["step"] = {"ms_no_slide": [ms_plain, ms_plain2], "ms_quarter_sliding": ms_slide,
                   "ms_of_which_slide_call": ms_slide_only, "us_per_note_no_slide": ms_plain / W * 1e3,
                   "us_per_note_quarter_sliding": ms_slide / W * 1e3, "steps": args.steps,
                   "timing": "wall clock around the host calls, synchronised"}

    # -- the CUDA class window by window (4 songs, 3 notes each, one slide before the third)
    n_cls, t_cls, count = 4, 0.0, 0
    for s in range(n_cls):
        mid = ua.audio_complete(wav[s, :int(lens[s])], 4096)
        mid.mag
        aw = mid.section(0, None, 258)
        g = ua.audio_complete(guess[s], 4096)
        r = np.random.default_rng(200 + s)
        for k in range(3):
            on, du, pi = float(r.uniform(0.05, 5.0)), float(r.uniform(0.2, 1.2)), int(r.integers(40, 80))
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            if k == 2:
                new = mid.section(6.0, None, 129)
                aw.slice(129, 258)
                aw.concat(new)
            ua.audio_complete.compress_bands(aw.mag, bands=20)
            sw = aw.resize(on, du, 8, attribs=["mag", "ph"])
            sw.section_power("mag", 23, 371)
            for bpt, low, nb in ((2, "A0", None), (4, "A0", None), (16, ua.midi_to_note(pi), 348),
                                 (16, "C4", 348), (2, ua.midi_to_note(pi - 10), 36)):
                aw.slice_C(on, du, 8, bins_per_tone=bpt, lowest_note=low, nbins=nb,
                           highest_note=None if nb else "C8")
            aw.subtract(g, offset=on)
            torch.cuda.synchronize()
            if s or k:                                          # the first note builds plans
                t_cls += time.perf_counter() - t0
                count += 1
    res["class_per_window"] = {"us_per_note": t_cls / count * 1e6, "notes": count,
                               "note": "the CUDA drop-in class, one window and one note at a time, synchronised"}

    # -- bench.py per_note_batched, this tree and the other one alternating
    if args.compare_tree:
        runs = []
        for tree in (args.compare_tree, ROOT, args.compare_tree, ROOT):
            p = per_note_batched(tree)
            runs.append({"tree": "compare" if tree == args.compare_tree else "this", "per_note_batched": p})
        res["bench_per_note_batched"] = runs
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
