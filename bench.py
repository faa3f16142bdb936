#!/usr/bin/env python
"""Throughput of the AMT-SAGA feature hot path (STFT + CQT + generative-subtract
+ dB) in window-features/s -- BASELINE.json's metric -- on N B200s.

  python bench.py [--gpus N] [--steps K] [--warmup W]          this repo's CUDA path
  python bench.py ... --dump-outputs DIR                       also write the last timed step's outputs
                                                               (seeded inputs: comparable across builds)
  python bench.py --impl reference ...                         the reference's CPU path
                                                               (oracle port: the reference
                                                               itself cannot be imported here)
One "step" = one pass over 1 h of synthetic 44.1 kHz audio held as 600 analysis
windows of 6 s (per GPU: weak scaling, windows are independent).  `value` times
the step with inputs resident in HBM; `e2e` times it from pinned host buffers
through the same public API with the H2D / D2H copies inside the timed region.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries exactly one JSON line: keep NCCL's banner / debug output on stderr
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

SR, N_FFT, HOP = 44100, 2048, 512
WIN_SAMPLES = 6 * SR            # 264600 -> 517 STFT columns, window = first 516
GUESS_SAMPLES = 65024           # single rendered note -> 128 columns
METRIC = "window-features/sec (STFT+CQT+subtract)"


def guess_offsets(n_windows, seed=7):
    """onset ~ U(0, 6 s) -> frame offset with util_audio.py:264 semantics, len(wf) = hop*(T-1)."""
    rng = np.random.default_rng(seed)
    t = rng.uniform(0, 6.0, n_windows)
    T = WIN_SAMPLES // HOP
    return np.floor(t * T * SR / (HOP * (T - 1))).astype(np.int32).reshape(-1, 1)


# ----------------------------------------------------------------------------- CPU reference arm
_BLAS_LIMIT = None
_CPU_INPUTS = None      # [(window wave, guess wave, onset seconds)], filled in the parent BEFORE the timer / the fork


def _cpu_class():
    """The class that plays `util_audio.audio_complete` on the CPU arm: the reference's own class when
    /root/reference is mounted (build container), else `AudioOracle`, which tests/test_ref_class.py proves
    bit-identical to it on the producer loop.  librosa / resampy underneath are the numpy restatement in both."""
    from oracle import ref_class
    if ref_class.available():
        return ref_class.load().audio_complete, "reference"
    from oracle.audio_oracle import AudioOracle
    return AudioOracle, "port"


def cpu_prepare(n_windows, seed0=50000):
    """Synthesise the CPU arm's inputs (same generator and seeds as the GPU arm).  NOT timed: the GPU arm
    synthesises outside its timed region too."""
    global _CPU_INPUTS
    from tests.synth import piano_clip
    rng = np.random.default_rng(7)
    onsets = rng.uniform(0, 6.0, n_windows)
    _CPU_INPUTS = [(piano_clip(seed0 + i, WIN_SAMPLES), piano_clip(90000 + seed0 + i, GUESS_SAMPLES, n_notes=1),
                    float(onsets[i])) for i in range(n_windows)]


def _cpu_window(i):
    """One window-feature on the CPU, through the reference's class interface (util_audio.py:32):
    STFT magnitude, CQT 84/12, one guessed-note subtraction, dB.  Returns the seconds of compute."""
    global _BLAS_LIMIT
    if _BLAS_LIMIT is None:      # one BLAS / OpenMP thread per process: `cores` = threads actually used
        try:
            from threadpoolctl import threadpool_limits
            _BLAS_LIMIT = threadpool_limits(limits=1)
        except Exception:
            _BLAS_LIMIT = False
    AC, _ = _cpu_class()
    y, g, onset = _CPU_INPUTS[i]
    T = WIN_SAMPLES // HOP
    t0 = time.perf_counter()
    song = AC(y, N_FFT, hop_length=HOP, sample_rate=SR)
    song.mag                                                          # util_audio.py:147 (STFT + magphase)
    C = song.slice_C(0, song._frames_to_seconds(song.shape[1]), song.shape[1], bins_per_tone=1,
                     lowest_note="C1", nbins=84)                      # util_audio.py:411-434 (CQT 84/12, fs 2)
    w = song.section(0, None, T)                                      # the 516-frame window (training.py:284)
    w.subtract(AC(g, N_FFT, hop_length=HOP, sample_rate=SR), offset=onset)   # util_audio.py:221-259
    D = w.D                                                           # util_audio.py:176-180
    return time.perf_counter() - t0, float(C[0, 0] + D[0, 0])


def cpu_sample(n_windows, pool=None):
    """windows/s over `n_windows` prepared windows (wall clock of the compute only; inputs are resident)."""
    t0 = time.perf_counter()
    if pool is not None:
        inner = pool.map(_cpu_window, range(n_windows), chunksize=1)
    else:
        inner = [_cpu_window(i) for i in range(n_windows)]
    wall = time.perf_counter() - t0
    return n_windows / wall, wall, sum(t for t, _ in inner)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    os.environ["OMP_NUM_THREADS"] = "1"
    import multiprocessing as mp
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    procs = max(1, min(cores, 64))
    per_step = procs                       # one window per worker per step: a bounded sample of the 600-window step
    _, kind = _cpu_class()
    cpu_prepare(per_step)                  # inputs synthesised here, before the fork and before any timer
    _cpu_window(0)                         # import / table warm-up in the parent (inherited by the forked workers)
    # ONE pool for the whole run, like the reference's Pool(synth_worker_count) (training.py:623): worker
    # start-up is not part of a step
    busy = 0.0
    with mp.get_context("fork").Pool(procs) as pool:
        for _ in range(max(args.warmup, 1)):
            cpu_sample(per_step, pool)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            busy += cpu_sample(per_step, pool)[2]
        dt = time.perf_counter() - t0
    value = per_step * args.steps / dt
    sample = ("%d of the step's 6 s windows per step (1 per worker, %d single-threaded workers = the box's usable logical "
              "CPUs) x %d steps; inputs synthesised before the timer; %.2f s of compute per window inside a worker, "
              "%.1f workers busy on average" % (per_step, procs, args.steps, busy / (per_step * args.steps), busy / dt))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "window-features/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD_NAME, "windows_per_step": per_step,
                   "note": "the reference's audio_complete interface (util_audio.py:32) on the CPU: "
                           + ("its own class imported from /root/reference (oracle/ref_class.py)" if kind == "reference" else
                              "AudioOracle, bit-identical to the reference's class (tests/test_ref_class.py; /root/reference "
                              "is not on this box)")
                           + " over the numpy restatement of librosa 0.6.3 / resampy (not installable here), under one "
                             "multiprocessing.Pool like training.py:623"},
        "cpu_baseline": {"value": value, "unit": "window-features/s", "cores": procs, "kind": kind,
                         "sample": sample},
        "e2e": {"value": value, "unit": "window-features/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


WORKLOAD_NAME = ("cfg2: 1 h synthetic 44.1 kHz audio per GPU as 600 x 6 s windows; STFT n_fft=2048 hop=512 "
                 "+ CQT 84 bins/12 per octave + 1 guessed-note subtract + dB per window")


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            pass

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons, pw = [], [], set(), []
        for ln in self.f.read().splitlines():
            c = [x.strip() for x in ln.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2])); pw.append(float(c[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            busy = [s for s, p in zip(sm, pw) if p >= 0.5 * max(pw)] or sm
            out.update(sm_mhz=float(np.median(busy)), sm_max_mhz=float(max(mx)), samples=len(sm),
                       power_w_max=float(max(pw)))
        out["reasons"] = sorted(reasons)
        return out



# ----------------------------------------------------------------------------- extra measurements (N = 1)
def measure_tf32_peak(torch, dev, n=8192, iters=10):
    """SURVEY 8(d): the tensor fraction of a TF32 kernel is quoted against a TF32 GEMM measured the same way
    as MEASURED_PEAKS.json's bf16 figure (torch.matmul, 8192^3, best of `iters`, CUDA events)."""
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        a = torch.randn((n, n), device=dev)
        b = torch.randn((n, n), device=dev)
        c = torch.empty((n, n), device=dev)
        for _ in range(3):
            torch.matmul(a, b, out=c)
        torch.cuda.synchronize()
        best = 1e30
        for _ in range(iters):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b, out=c)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return 2.0 * n ** 3 / best / 1e9
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def measure_cfg4(torch, ops, dev, hbm_peak, n_windows=4096, steps=5):
    """BASELINE config 4: 4096 windows [1025, 516] x 16 guessed-note spectrograms [1025, 128], applied sequentially per
    window (current-max ref at every step), ReLU, then dB -- through K3's chain kernel.  Random magnitudes of the right
    shapes (timing; the arithmetic is bit-exact against numpy in tests/test_gpu_parity.py)."""
    B, T, Tg, S = 1025, 516, 128, 16
    P = ops.frame_pitch(B)
    g = torch.Generator(device=dev).manual_seed(1)
    win = torch.rand((n_windows, T, P), device=dev, generator=g)
    base = win.clone()
    gue = torch.rand((n_windows, S, Tg, P), device=dev, generator=g)
    offs = torch.randint(0, T, (n_windows, S), device=dev, generator=g, dtype=torch.int32)
    D = torch.empty_like(win)
    gref = gue.amax(dim=(2, 3))
    ms = []
    for i in range(steps + 1):
        win.copy_(base)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        ops.subtract_db_batch(win, gue, offs, B, D_out=D, guess_ref=gref)
        b.record()
        torch.cuda.synchronize()
        if i:
            ms.append(a.elapsed_time(b))
    t = sorted(ms)[len(ms) // 2]
    alg = n_windows * 4 * B * (2 * T + S * Tg)      # read mag + read 16 guesses + write one output (SURVEY 8d)
    del win, base, gue, D
    torch.cuda.empty_cache()
    return {"workload": "cfg4: %d windows x 16 guesses, subtract chain + dB" % n_windows, "ms": t,
            "windows_per_s": n_windows / t * 1e3, "GBps": alg / t / 1e6, "frac": alg / t / 1e6 / hbm_peak,
            "bound": "hbm", "kernel": "subtract_chain_cluster_kernel (K3, 16 sequential steps + dB)",
            "algorithmic_bytes": alg, "steps": steps}


def measure_note_step(torch, ops, synth, dev, n_windows=600, steps=5):
    """One batched iteration of the reference's per-note loop in ITS order (training.py:333-449) for 600 windows of
    its own shape (N 4096, hop 1024, 258 frames): K4 iSTFT of the subtracted windows -> the five slice_C shapes -> K5 ->
    guess STFT -> K3 (amt_saga_b200.note_step.NoteStepBatch; parity vs the reference's class: tests/test_note_step.py)."""
    from amt_saga_b200.note_step import NoteStepBatch
    L = 264168
    wav = synth.piano_batch(range(n_windows), L, SR, seed_base=50000, device=dev)
    plan = ops.get_stft_plan(4096, 1024, True, device=dev)
    r = ops.stft_batch(wav, plan, want_phase=True)
    b = NoteStepBatch(n_windows, device=dev)
    b.load(r["mag_storage"][:, :258].contiguous(), r["phase_storage"][:, :258].contiguous(), wav, r["clip_max"],
           np.ones((n_windows, 3)))
    guess = synth.piano_batch(range(n_windows), 54277, SR, n_notes=1, seed_base=90000, device=dev)

    def one(seed, lo=48, hi=72):
        rg = np.random.default_rng(seed)
        b.step(rg.uniform(0, 5.0, n_windows), rg.uniform(0.2, 1.2, n_windows), rg.integers(lo, hi, n_windows), guess)

    def timed(lo, hi):
        for i in range(3):          # builds (and caches) the note-relative CQT plans (one bank per pitch)
            one(i, lo, hi)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(steps):
            one(10 + i, lo, hi)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / steps * 1e3
    ms = timed(48, 72)
    ms88 = timed(21, 109)           # every key of the piano: many small pitch groups
    del b, wav, guess, r
    torch.cuda.empty_cache()
    return {"workload": "one per-note iteration of training.py:333-449 for %d windows (N 4096, hop 1024, 258 frames, 24 "
                        "distinct pitches): iSTFT + 5 CQT shapes + K5 + guess STFT + subtract" % n_windows,
            "ms_per_step": ms, "us_per_note": ms / n_windows * 1e3, "notes_per_s": n_windows / ms * 1e3,
            "ms_per_step_88_pitches": ms88, "us_per_note_88_pitches": ms88 / n_windows * 1e3,
            "timing": "wall clock around the host call (includes the per-pitch host loop), synchronised",
            "unbatched_class_ms_per_note": 1.02, "unbatched_class_ms_per_note_round1": 2.97, "steps": steps}


# ----------------------------------------------------------------------------- GPU arm
DUMP_WINDOWS = 8        # mag + D of 8 windows: 34 MB of float32


def dump_outputs(torch, pipe, out_dir, seed=0):
    """Write what the last step returned to its caller as float32 `out_dir/<name>.npy`: `ref` [W], the
    post-subtraction ref_mag of every window, and for a fixed seeded sample of DUMP_WINDOWS windows (ascending
    window order) `mag` [n, frames, bins], the subtracted STFT magnitude, `D` [n, frames, bins], its dB image, and
    `C` [n, frames, cqt bins], the constant-Q magnitudes.  The inputs are seeded as well, so two builds run with
    the same arguments can be compared file by file."""
    os.makedirs(out_dir, exist_ok=True)
    idx = np.sort(np.random.default_rng(seed).choice(pipe.W, size=min(DUMP_WINDOWS, pipe.W), replace=False))
    sel = torch.as_tensor(idx, device=pipe.dev)
    out = {"ref": pipe.ref, "mag": pipe.mag[sel, :pipe.T, :pipe.nb], "D": pipe.D[sel, :pipe.T, :pipe.nb],
           "C": pipe.C[sel, :, :pipe.cqt.n_bins]}
    for name, t in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.to(torch.float32).cpu().numpy())


def bind_to_gpu_cpus(local):
    """Pin this rank to the CPUs NVML reports as local to its GPU, so that the pinned host buffers of the end-to-end
    path are allocated (first touch) on the GPU's own NUMA node and the H2D copies of eight ranks do not all cross
    one inter-socket link.  Best effort: returns a short description for the bench line, None if nothing was done."""
    try:
        import pynvml
        pynvml.nvmlInit()
        # torch's device `local` is CUDA_VISIBLE_DEVICES-relative: resolve it through the PCI bus id
        import torch
        bus = torch.cuda.get_device_properties(local).pci_bus_id if hasattr(torch.cuda.get_device_properties(local), "pci_bus_id") else None
        h = None
        if bus is not None:
            for i in range(pynvml.nvmlDeviceGetCount()):
                hi = pynvml.nvmlDeviceGetHandleByIndex(i)
                if pynvml.nvmlDeviceGetPciInfo(hi).bus == bus:
                    h = hi
                    break
        if h is None:
            h = pynvml.nvmlDeviceGetHandleByIndex(local)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        usable = cpus & set(os.sched_getaffinity(0))
        if not usable or usable == set(os.sched_getaffinity(0)):
            return None if not usable else "gpu-local cpus = all usable cpus (%d)" % len(usable)
        os.sched_setaffinity(0, usable)
        return "bound to %d gpu-local cpus (NVML affinity)" % len(usable)
    except Exception as e:      # no NVML, no permission: run unbound
        return "unbound (%s)" % type(e).__name__


def run_saga(args):
    import torch
    import torch.distributed as dist
    import amt_saga_b200  # noqa: F401
    from amt_saga_b200 import ops, synth
    from amt_saga_b200.pipeline import WindowFeaturePipeline

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout must carry exactly ONE JSON line, but native libraries write there too (NCCL prints its
    # version banner on fd 1 whatever NCCL_DEBUG_FILE says): park the real stdout, point fd 1 at stderr
    # for the run, and write the result line to the parked descriptor at the end
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback for the product path)")
    torch.cuda.set_device(local)
    numa = bind_to_gpu_cpus(local)      # before any pinned allocation: first touch puts the buffers next to the GPU
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    W = args.windows
    pipe = WindowFeaturePipeline(W, WIN_SAMPLES, GUESS_SAMPLES, SR, N_FFT, HOP, device=dev,
                                 cqt_impl=args.cqt_impl)
    # rank r owns windows [r*W, (r+1)*W): contiguous block partition, generated on device
    ids = range(rank * W, (rank + 1) * W)
    wav = synth.piano_batch(ids, WIN_SAMPLES, SR, seed_base=50000, device=dev)
    guess = synth.piano_batch(ids, GUESS_SAMPLES, SR, n_notes=1, seed_base=90000, device=dev)
    offs = torch.as_tensor(guess_offsets(W, seed=7 + rank), device=dev)
    gathered = torch.empty((world * W,), device=dev, dtype=torch.float32) if world > 1 else None

    def step(events=None):
        pipe.run(wav, guess, offs, events)
        if world > 1:     # collection only: per-window ref_mag gathered over NVLink
            dist.all_gather_into_tensor(gathered, pipe.ref)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    launches0 = ops.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    launches = ops.launch_count() - launches0
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:     # before the passes below overwrite the pipeline's buffers
        dump_outputs(torch, pipe, args.dump_outputs)
    # per-kernel durations for the roofline: the same steps again with the two chains of the path run one
    # after the other (in the timed loop above the CQT chain overlaps the STFT / subtract chain on a second
    # stream, so a kernel's own duration cannot be read off there)
    events = []
    stage_steps = max(3, min(args.steps, 20))
    for _ in range(stage_steps):
        step(events)
    barrier()
    stage_ms = {}
    for name, a, b in events:
        stage_ms[name] = stage_ms.get(name, 0.0) + a.elapsed_time(b)
    stage_ms = {k: v / stage_steps for k, v in stage_ms.items()}

    # ---- end to end from pinned host memory ----------------------------------------------
    h = pipe.host_buffers()
    h["wav"].copy_(wav); h["guess"].copy_(guess); h["offs"].copy_(offs)
    torch.cuda.synchronize()
    e2e_steps = max(3, min(args.steps, args.e2e_steps))
    RET = "features"      # D2H = what the classifiers consume (K5 on the device), not the raw CQT image
    for _ in range(2):
        pipe.run_host(args.e2e_chunks, returns=RET)
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(e2e_steps):
        pipe.run_host(args.e2e_chunks, returns=RET)
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)

    # ---- the same, with the host holding 16-bit PCM (what fluidsynth / the audio files deliver): K0 rebuilds the
    # reference's `pcm * (vel/128)**4 / max|pcm|` float waveform on the device, half the H2D bytes.  Reported
    # beside `e2e` (whose float32 host buffers are the contract), not instead of it.
    hp = pipe.host_pcm_buffers()
    for src, key in ((wav, "wav_pcm"), (guess, "guess_pcm")):
        peak = src.abs().amax(dim=1, keepdim=True).clamp_min(1e-12)
        hp[key].copy_((src / peak * 32767.0).round().to(torch.int16))
    vel = torch.as_tensor(np.random.default_rng(11 + rank).integers(30, 121, size=(2, W)), dtype=torch.float64)
    hp["mul"].copy_((vel / 128.0) ** 4)
    torch.cuda.synchronize()
    for _ in range(2):
        pipe.run_host(args.e2e_chunks, pcm16=True, returns=RET)
    barrier()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = ops.launch_count()
    g0.record()
    for _ in range(e2e_steps):
        pipe.run_host(args.e2e_chunks, pcm16=True, returns=RET)
    g1.record()
    barrier()
    ms_pcm = g0.elapsed_time(g1)
    pcm_launches = (ops.launch_count() - l0) // e2e_steps
    clocks = sampler.stop() if sampler else None

    t = torch.tensor([ms, ms_e2e, ms_pcm], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e, ms_pcm = float(t[0]), float(t[1]), float(t[2])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    ms_step = ms / args.steps
    value = world * W / (ms_step * 1e-3)
    e2e_value = world * W / (ms_e2e / e2e_steps * 1e-3)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json, burst copy)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    # per-stage algorithmic work (DESIGN.md section 4)
    stft_bytes = W * 4 * (pipe.ns + pipe.T_clip * pipe.nb)
    gst_bytes = W * 4 * (pipe.ng + pipe.Tg * pipe.nb)
    sub_bytes = W * pipe.subtract_bytes_per_window()
    cqt_flops = W * pipe.cqt_flops_per_window()
    casc_bytes = W * 4 * pipe.ns * 2          # each level read once, written once at half the length: <= 2x the input
    tpeak_bf16 = float(peaks.get("bf16_tflops_sustained", 1400.0))
    tpeak = measure_tf32_peak(torch, dev)       # the contraction runs kind::tf32: quote it against a TF32 GEMM
    stages = {
        "stft": {"ms": stage_ms.get("stft"), "bound": "hbm", "GBps": stft_bytes / stage_ms["stft"] / 1e6},
        "stft_guess": {"ms": stage_ms.get("stft_guess"), "bound": "hbm", "GBps": gst_bytes / stage_ms["stft_guess"] / 1e6},
        "subtract_db": {"ms": stage_ms.get("subtract_db"), "bound": "hbm", "GBps": sub_bytes / stage_ms["subtract_db"] / 1e6},
        "cqt_cascade": {"ms": stage_ms.get("cqt_cascade"), "bound": "hbm", "GBps": casc_bytes / stage_ms["cqt_cascade"] / 1e6},
        "cqt_contract": {"ms": stage_ms.get("cqt_contract"), "bound": "tensor",
                         "TFLOPs_algorithmic": cqt_flops / stage_ms["cqt_contract"] / 1e9,
                         # per 24 useful columns the kernel issues one N=48 ([hi|lo] bank) and one N=32 MMA
                         "TFLOPs_issued_tf32": cqt_flops * (80.0 / 24.0) / stage_ms["cqt_contract"] / 1e9},
    }
    traffic = {}
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        pass
    kernels = {"stft": "stft_ring_kernel<19,20> (K1 ring kernel, window batch)", "stft_guess": "stft_ring_kernel<19,20> (K1 ring kernel, guess batch)",
               "subtract_db": "subtract_single_flat_kernel + window_db_lean_kernel<256,12> (K3)",
               "cqt_cascade": "decimate2x2_kernel x 2 + decimate2_kernel x 3 + cqt_pad_kernel (K2a)",
               "cqt_contract": "cqt_umma_kernel (tcgen05) + cqt_tail_kernel (K2b)"}
    for k, v in stages.items():
        v["frac"] = (v["GBps"] / hbm_peak) if v["bound"] == "hbm" else (v["TFLOPs_algorithmic"] / tpeak)
        v["kernel"] = kernels.get(k, k)
        v["traffic"] = traffic.get(k, {}).get("bytes")     # ncu DRAM bytes per launch (profiles/traffic.json)
    dom = max(stage_ms, key=stage_ms.get)
    tr = traffic.get(dom, {}).get("bytes")
    if stages[dom]["bound"] == "tensor":
        roof = {"kernel": "cqt_umma_kernel (tcgen05 kernel-bank contraction)", "bound": "tensor",
                "achieved": stages[dom]["TFLOPs_algorithmic"], "peak": tpeak, "unit": "TFLOP/s",
                "frac": stages[dom]["frac"], "traffic": tr,
                "peak_source": "TF32 torch.matmul 8192^3 measured in this run",
                "note": "algorithmic flops = 172704/frame (SURVEY 8d); the 3xTF32 split issues 3.33x that (N=48 main + N=32 correction MMA per 24 useful columns); "
                        "an SS-mode tcgen05.mma is paced by the SMEM bytes it reads: 44-48 cycles for N<=64 (profiles/microbench)"}
    else:
        ach = stages[dom]["GBps"]
        roof = {"kernel": kernels.get(dom, dom), "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                "frac": ach / hbm_peak, "traffic": tr, "peak_source": peak_src}

    # ---- the same step at the reference's own default analysis shape (main.py: N=4096, hop=1024; CQT 87 bins from A0,
    # training.py:271), reported beside the BASELINE shape; never the headline
    ref_shape = None
    if world == 1 and not args.no_ref_shape:
        try:
            p2 = WindowFeaturePipeline(W, WIN_SAMPLES, GUESS_SAMPLES, SR, 4096, 1024, cqt_lowest="A0", cqt_bins=87,
                                       cqt_bpo=12, device=dev)
            offs2 = torch.div(offs, 2, rounding_mode="floor").to(torch.int32)
            for _ in range(3):
                p2.run(wav, guess, offs2)
            torch.cuda.synchronize()
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n2 = max(3, min(args.steps, 30))
            r0.record()
            for _ in range(n2):
                p2.run(wav, guess, offs2)
            r1.record()
            torch.cuda.synchronize()
            ms2 = r0.elapsed_time(r1) / n2
            ref_shape = {"shape": "n_fft 4096, hop 1024, 258 frames per window, CQT 87 bins from A0 (12 per octave)",
                         "value": W / (ms2 * 1e-3), "unit": "window-features/s", "ms_per_step": ms2, "steps": n2}
            del p2
        except Exception as e:      # informational only
            ref_shape = {"error": repr(e)[:200]}

    cfg4 = note_step = None
    if world == 1 and not args.no_extras:
        for name, fn in (("cfg4", lambda: measure_cfg4(torch, ops, dev, hbm_peak)),
                         ("note", lambda: measure_note_step(torch, ops, synth, dev))):
            try:
                res = fn()
            except Exception as e:      # reported beside the headline, never instead of it
                res = {"error": repr(e)[:300]}
            if name == "cfg4":
                cfg4 = res
            else:
                note_step = res

    cpu = None
    if world == 1 and args.cpu_windows > 0:
        cpu_prepare(args.cpu_windows)          # synthesis is outside the timer, as on the GPU arm
        _cpu_window(0)
        v, wall, _ = cpu_sample(args.cpu_windows)
        cpu = {"value": v, "unit": "window-features/s", "cores": 1, "kind": _cpu_class()[1],
               "sample": "%d of the step's 6 s windows through the reference's audio_complete interface on the numpy "
                         "restatement of librosa 0.6.3, 1 process, 1 thread, inputs resident (%.1f s)" % (args.cpu_windows, wall)}
    line = {
        "metric": METRIC, "value": value, "unit": "window-features/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD_NAME, "windows_per_gpu": W, "frames_per_window": pipe.T,
                   "frames_per_s": world * W * pipe.T / (ms_step * 1e-3),
                   "l2": "inputs 635 MB/step per GPU > 126 MB L2 (no flush needed)",
                   "parallelism": "window shards, 1 process/GPU, no collective on the path",
                   "streams": "schedule=%s (kernels of a step enqueued on one stream; forking the CQT chain onto a second "
                              "stream measured 4 %% slower); `stages` are timed in a separate pass with events between "
                              "the kernels (sum %.3f ms)" % (pipe.schedule, sum(stage_ms.values())),
                   "cqt_impl": args.cqt_impl},
        "e2e": {"value": e2e_value, "unit": "window-features/s", "h2d_bytes_per_step": pipe.h2d_bytes(),
                "d2h_bytes_per_step": pipe.d2h_bytes(RET), "steps": e2e_steps,
                "ms_per_step": ms_e2e / e2e_steps,
                "returns": "per window, reduced on the device by K5: the log-dB image's 8 columns from the guessed note's "
                           "onset [8 x 1025], the CQT's same 8 columns [8 x 84], compress_bands(subtracted mag)/ref [516 x 20], "
                           "post-subtraction ref_mag (the shapes the classifiers take, util_train_test.py:39-59)",
                "overlap": "%d window chunks on 3 streams (H2D | kernels | D2H)" % args.e2e_chunks,
                "h2d_GBps_aggregate": world * pipe.h2d_bytes() / (ms_e2e / e2e_steps * 1e-3) / 1e9,
                "host_affinity": numa},
        "e2e_pcm16": {"value": world * W / (ms_pcm / e2e_steps * 1e-3), "unit": "window-features/s",
                      "h2d_bytes_per_step": pipe.h2d_bytes(pcm16=True), "d2h_bytes_per_step": pipe.d2h_bytes(RET),
                      "steps": e2e_steps, "ms_per_step": ms_pcm / e2e_steps, "launches_per_step": int(pcm_launches),
                      "note": "same call with int16 PCM + per-clip float64 factor in pinned host memory (the form in which "
                              "fluidsynth / soundfile deliver audio, util_audio.py:894/:964); K0 (pcm16_absmax + pcm16_ingest "
                              "kernels) rebuilds float32(pcm*mul/max|pcm|) = util_audio.py:781 on the device, bit-exact; "
                              "`e2e` above keeps float32 host buffers"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roof,
        "stages": stages,
        "cpu_baseline": cpu,
        "reference_default_shape": ref_shape,
        "cfg4": cfg4,
        "per_note_batched": note_step,
        "tensor_peaks": {"tf32_tflops_measured_here": tpeak, "bf16_tflops_sustained": tpeak_bf16,
                         "how": "torch.matmul 8192^3, allow_tf32, best of 10 (CUDA events); bf16 from MEASURED_PEAKS.json"},
    }
    sys.stdout.flush()
    os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()



# ----------------------------------------------------------------------------- BASELINE config 5
def run_cfg5(args):
    """Corpus-scale sharded feature extraction: `hours` x 360 clips of 10 s (SURVEY 8d: clip c = piano generator with
    seed 1234 + c), contiguous clip ranges per rank, generated ON DEVICE in 1 h chunks (the 127 GB of input never
    exist at once), STFT magnitude (2048 / 512) + CQT (84 bins, 12 per octave) per clip, of which only a per-clip
    checksum is kept.  No collective on the path; one all_gather of the checksums at the end.  Prints ONE JSON line:
    clips/s end to end (generation included) and for the feature kernels alone, and the gathered checksum, which must
    be identical for every GPU count."""
    import torch
    import torch.distributed as dist
    import amt_saga_b200  # noqa: F401
    from amt_saga_b200 import ops, shard, synth
    from amt_saga_b200.util_audio import note_to_hz

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    clips_total = int(round(args.cfg5_hours * 360))
    ns, chunk = 441000, 360
    lo, hi = shard.shard_range(clips_total, rank, world)
    sp = ops.get_stft_plan(N_FFT, HOP, True, device=dev)
    cp = ops.get_cqt_plan(SR, HOP, note_to_hz("C1"), 84, 12, 2, device=dev)

    def features(ids):
        wav = synth.piano_batch(ids, ns, SR, seed_base=1234, device=dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        m = ops.stft_batch(wav, sp, want_max=False)["mag_storage"]
        c = ops.cqt_batch(wav, cp)["mag_storage"]
        b.record()
        # per-clip checksum of the exact bit patterns (wraps in int64: order-independent, partition-independent)
        cs = m.view(torch.int32).to(torch.int64).sum(dim=(1, 2)) + 31 * c.view(torch.int32).to(torch.int64).sum(dim=(1, 2))
        return cs, (a, b), m.shape[1]

    features(list(range(min(4, max(hi - lo, 1)))))       # warm-up: plans, allocator
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    parts, evs, frames = [], [], 0
    for a, b in shard.chunks(lo, hi, chunk):
        cs, ev, T = features(list(range(a, b)))
        parts.append(cs)
        evs.append(ev)
        frames += (b - a) * T
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    kern_ms = sum(a.elapsed_time(b) for a, b in evs)
    local_cs = torch.cat(parts) if parts else torch.zeros(0, device=dev, dtype=torch.int64)
    allcs = shard.gather_ragged(local_cs) if world > 1 else local_cs
    t = torch.tensor([wall, kern_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    wall, kern_ms = float(t[0]), float(t[1])
    if rank == 0:
        assert allcs.numel() == clips_total
        total = int(allcs.sum().item())
        line = {"metric": "clips/s (cfg5: sharded STFT + CQT over a generated corpus)", "value": clips_total / wall,
                "unit": "clips/s", "n_gpus": world, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic (generated on device per shard, seeds 1234 + clip id)",
                "config": {"workload": "cfg5: %.1f h = %d clips of 10 s at 44.1 kHz, 1 h chunks, STFT 2048/512 + CQT 84/12, "
                                       "per-clip checksums gathered" % (args.cfg5_hours, clips_total),
                           "partition": "contiguous clip ranges per rank, no collective on the path"},
                "wall_s": wall, "hours_of_audio_per_s": args.cfg5_hours / wall,
                "feature_kernels_only": {"ms": kern_ms, "clips_per_s": (hi - lo) * world / kern_ms * 1e3,
                                         "note": "CUDA events around K1 + K2 of every chunk on the slowest rank; the rest of "
                                                 "the wall time is the on-device audio generator"},
                "checksum": total, "checksum_clip0": int(allcs[0].item()), "checksum_last": int(allcs[-1].item())}
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="saga", choices=["saga", "reference"])
    ap.add_argument("--windows", type=int, default=600, help="6 s windows per GPU per step (600 = 1 h)")
    ap.add_argument("--cpu-windows", type=int, default=48, help="windows in the cpu_baseline sample (0 = skip)")
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--cqt-impl", type=int, default=0)
    ap.add_argument("--e2e-chunks", type=int, default=12, help="window chunks for H2D/compute/D2H overlap")
    ap.add_argument("--no-ref-shape", action="store_true", help="skip the extra pass at the reference's default n_fft/hop")
    ap.add_argument("--no-extras", action="store_true", help="skip the cfg4 chain and batched per-note measurements")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (float32; "
                         "ref_mag of every window, mag / D / C of a fixed sample of %d windows)" % DUMP_WINDOWS)
    ap.add_argument("--cfg5-hours", type=float, default=0.0,
                    help="BASELINE config 5 instead of the step bench: this many hours of synthetic audio (360 clips of 10 s per "
                         "hour), block-partitioned over the ranks, generated on device in 1 h chunks, STFT + CQT, checksum gathered")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    elif args.cfg5_hours > 0:
        run_cfg5(args)
    else:
        run_saga(args)


if __name__ == "__main__":
    main()
