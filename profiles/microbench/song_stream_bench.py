"""Songs held as waveforms (SongBatch(hold="waveform")) against songs held as their STFT (hold="stft"), on
song_walk_bench.py's W seeded songs of 30-180 s, one window per song; both holds in one process, alternating.

    python profiles/microbench/song_stream_bench.py [--windows 128] [--corpus 512] [--compare-tree DIR] [--out FILE]

Reports, per hold and repetition:
* torch.cuda.max_memory_allocated after setup and over a walk (the input waveforms included: both holds share them);
* setup time (wall clock, synchronised);
* the slide call for a random quarter of the windows, and a step with that quarter sliding first (wall clock around the
  host calls, synchronised), and a step without slides;
then
* ops.stft_rows_batch alone at a slide's shape (h = 129 new rows for each of the W windows, magnitude + phasor):
  CUDA events over 50 launches, against its algorithmic bytes -- samples read ((h - 1) hop + N) 4 plus rows written
  h P 12 per clip -- as a fraction of the HBM copy peak DESIGN.md uses (6 543 GB/s);
* a corpus walk under hold="waveform": --corpus songs through W slots, 4 notes per song with a slide before every
  second note; a slot takes the next song (SongBatch.refill) when its notes are done or its slide went past the end.
  Notes per second, wall clock, synchronised, after a warm-up walk of the first W songs;
* bench.py's `per_note_batched` from this tree and, with --compare-tree, another checkout, alternating.
The card's name and power limit are read in the same run."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from song_walk_bench import ROOT, HBM_PEAK, SR, card, notes, per_note_batched  # noqa: E402
from amt_saga_b200 import _lib, ops, synth  # noqa: E402
from amt_saga_b200.note_step import NoteStepBatch  # noqa: E402
from amt_saga_b200.song_setup import SongBatch  # noqa: E402


def sync_ms(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


def hold_run(hold, wav, lens, guess, steps, dev):
    W = wav.shape[0]
    ops._workspaces.clear()        # the CQT workspace a previous run left: each hold is measured as if it ran alone
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    r = {}
    ms, b = sync_ms(lambda: SongBatch(device=dev, hold=hold).setup(wav, lens))
    r["setup_ms"] = ms
    r["max_memory_allocated_setup_GB"] = torch.cuda.max_memory_allocated() / 1e9
    r["memory_allocated_after_setup_GB"] = torch.cuda.memory_allocated() / 1e9
    win = b.section(np.arange(W), np.zeros(W), 258)
    step = b.load_into(NoteStepBatch(W, device=dev), win)
    for i in range(3):                                         # plans of every pitch, the full and patched iSTFT
        step.step(*notes(np.random.default_rng(100 + i), W), guess)
    rng = np.random.default_rng(7)
    t_plain, t_slide, t_call = [], [], []
    for i in range(steps):
        mask = np.zeros(W, dtype=bool)
        mask[rng.choice(W, W // 4, replace=False)] = True
        mask &= win.offset_s + 9.0 < lens / SR                 # keep the walk inside the songs
        n = notes(rng, W)
        if i % 2:
            t_plain.append(sync_ms(lambda: step.step(*n, guess))[0])
        else:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            t_call.append(sync_ms(lambda: b.slide(step, win, mask))[0])
            step.step(*n, guess)
            torch.cuda.synchronize()
            t_slide.append((time.perf_counter() - t0) * 1e3)
    r["ms_slide_call"] = float(np.median(t_call))
    r["ms_step_quarter_sliding"] = float(np.median(t_slide))
    r["ms_step_no_slide"] = float(np.median(t_plain))
    r["max_memory_allocated_walk_GB"] = torch.cuda.max_memory_allocated() / 1e9
    del step, win, b
    return r


def rows_kernel(wav, lens, dev):
    """stft_rows_batch at a slide's shape: frames [t, t + 129) of every song, written as rows [129, 258)."""
    W = wav.shape[0]
    plan = ops.get_stft_plan(4096, 1024, True, device=dev)
    P = ops.frame_pitch(plan.n_bins)
    h = 129
    out = torch.empty((W, 258, P), device=dev)
    ph = torch.empty((W, 258, P), device=dev, dtype=torch.complex64)
    T = 1 + lens // 1024
    f0 = torch.as_tensor(np.random.default_rng(3).integers(0, T - h), device=dev, dtype=torch.int32)
    offs = torch.arange(W, device=dev, dtype=torch.int64) * wav.stride(0)
    lens_dev = torch.as_tensor(lens, device=dev)

    def run():      # the C entry with device tables built once: the kernel, not the per-call table upload
        _lib.check(_lib.lib().saga_stft_rows_exec(
            plan.handle, ops._ptr(wav), ops._ptr(offs), ops._ptr(lens_dev), W, ops._ptr(f0), h, None, h, 258,
            ops._ptr(out), ops._ptr(torch.view_as_real(ph)), P, 258 * P, None, ops._stream(wav)))
    run()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(50):
        run()
    ev[1].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1]) / 50
    nbytes = W * (((h - 1) * 1024 + 4096) * 4 + h * P * 12)
    return {"ms": ms, "frames": W * h, "ns_per_frame": ms * 1e6 / (W * h), "algorithmic_bytes": nbytes,
            "TBps": nbytes / (ms * 1e-3) / 1e12, "fraction_of_hbm_peak": nbytes / (ms * 1e-3) / HBM_PEAK,
            "note": "the W windows' new halves at random song offsets; each launch reads %.0f MB of samples and writes "
                    "%.0f MB of rows, above the 126 MB L2" % (W * ((h - 1) * 1024 + 4096) * 4 / 1e6, W * h * P * 12 / 1e6)}


def corpus_walk(wav, lens, W, guess, dev, n_songs, notes_per_song=4):
    """Songs 0 .. n_songs - 1 through W slots; a slot is refilled when its song's notes are done or its slide went past
    the song's end.  Returns (notes stepped for live songs, steps, refills, seconds)."""
    b = SongBatch(device=dev, hold="waveform").setup(wav[:n_songs], lens[:n_songs])
    win = b.section(np.arange(W), np.zeros(W), 258)
    step = b.load_into(NoteStepBatch(W, device=dev), win)
    cur, k = np.arange(W), np.zeros(W, dtype=np.int64)
    done = np.zeros(W, dtype=bool)
    nxt, n_notes, n_steps, n_refill = W, 0, 0, 0
    rng = np.random.default_rng(11)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    while True:
        fill = np.flatnonzero(done)[:max(0, n_songs - nxt)]
        if len(fill):
            b.refill(step, win, fill, np.arange(nxt, nxt + len(fill)))
            cur[fill], k[fill], done[fill] = np.arange(nxt, nxt + len(fill)), 0, False
            nxt += len(fill)
            n_refill += len(fill)
        if done.all():
            break
        mask = ~done & (k % 2 == 1)
        if mask.any():
            done |= b.slide(step, win, mask)
        step.step(*notes(rng, W), guess)
        n_notes += int((~done).sum())
        n_steps += 1
        k[~done] += 1
        done |= k >= notes_per_song
    torch.cuda.synchronize()
    return n_notes, n_steps, n_refill, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=128)
    ap.add_argument("--corpus", type=int, default=512)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--compare-tree", default=None)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    W = args.windows
    res = {"card": card(), "windows": W}
    rng = np.random.default_rng(1)                              # song_walk_bench.py's songs
    secs = rng.uniform(30.0, 180.0, W)
    lens = (secs * SR).astype(np.int64)
    wav = synth.piano_batch(range(W), int(lens.max()), SR, n_notes=200, seed_base=31000, device=dev)
    guess = synth.piano_batch(range(W), 54277, SR, n_notes=1, seed_base=32000, device=dev)
    res["song_frames"] = int((1 + lens // 1024).sum())
    res["input_waveforms_GB"] = wav.numel() * 4 / 1e9
    runs = []
    for rep in range(args.reps):
        for hold in ("stft", "waveform"):
            runs.append(dict(hold=hold, rep=rep, **hold_run(hold, wav, lens, guess, args.steps, dev)))
    res["holds"] = runs
    by = {h: [r for r in runs if r["hold"] == h] for h in ("stft", "waveform")}
    res["summary"] = {
        "peak_memory_ratio_stft_over_waveform": float(np.median([s["max_memory_allocated_walk_GB"] for s in by["stft"]])
                                                      / np.median([w["max_memory_allocated_walk_GB"] for w in by["waveform"]])),
        "step_quarter_sliding_waveform_over_stft": float(np.median([w["ms_step_quarter_sliding"] for w in by["waveform"]])
                                                         / np.median([s["ms_step_quarter_sliding"] for s in by["stft"]])),
        "slide_call_waveform_over_stft": float(np.median([w["ms_slide_call"] for w in by["waveform"]])
                                               / np.median([s["ms_slide_call"] for s in by["stft"]]))}
    torch.cuda.empty_cache()
    res["stft_rows_kernel"] = rows_kernel(wav, lens, dev)
    del wav
    torch.cuda.empty_cache()

    # -- corpus walk: song_walk's recipe for --corpus songs (the first W are the songs above)
    secs_c = np.random.default_rng(1).uniform(30.0, 180.0, args.corpus)
    lens_c = (secs_c * SR).astype(np.int64)
    wav_c = synth.piano_batch(range(args.corpus), int(lens_c.max()), SR, n_notes=200, seed_base=31000, device=dev)
    corpus_walk(wav_c, lens_c, W, guess, dev, 2 * W)            # warm-up: plans of every pitch and shape
    ops._workspaces.clear()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    n_notes, n_steps, n_refill, sec = corpus_walk(wav_c, lens_c, W, guess, dev, args.corpus)
    res["corpus_walk"] = {"songs": args.corpus, "slots": W, "notes": n_notes, "steps": n_steps, "refills": n_refill,
                          "seconds": sec, "notes_per_s": n_notes / sec,
                          "max_memory_allocated_GB": torch.cuda.max_memory_allocated() / 1e9,
                          "input_waveforms_GB": wav_c.numel() * 4 / 1e9,
                          "timing": "wall clock from the first step to the last refill, synchronised at both ends; "
                                    "setup not included"}
    del wav_c
    torch.cuda.empty_cache()

    if args.compare_tree:
        res["bench_per_note_batched"] = [
            {"tree": "compare" if tree == args.compare_tree else "this", "per_note_batched": per_note_batched(tree)}
            for tree in (args.compare_tree, ROOT, args.compare_tree, ROOT)]
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
