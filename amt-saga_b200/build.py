"""Build the saga_b200 C-ABI shared library in-tree with nvcc for sm_100a.

The .so lands next to this file (git-ignored, but it travels to the GPU box
with the gpurun snapshot).  No torch.utils.cpp_extension / JIT cache involved.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libsaga_b200.so")
SOURCES = ["api.cu", "stft.cu", "stft_ring.cu", "istft_ring.cu", "subtract_db.cu", "cqt.cu", "cqt_umma.cu", "cqt_umma_stream.cu", "features.cu", "ingest.cu", "window_slide.cu"]
NVCC_FLAGS = ["-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-shared", "-Xcompiler", "-fPIC", "-lcuda"]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    deps.append(os.path.join(HERE, "..", "include", "saga_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile csrc/*.cu into libsaga_b200.so (sm_100a). Returns the path.
    The translation units are compiled in parallel (host-only linkage between them), then linked."""
    if not force and not _stale():
        return LIB
    import concurrent.futures
    import tempfile
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    compile_flags = [f for f in NVCC_FLAGS if f not in ("-shared", "-lcuda")]
    with tempfile.TemporaryDirectory(prefix="saga_build_") as tmp:
        def one(src):
            obj = os.path.join(tmp, src.replace(".cu", ".o"))
            cmd = [nvcc] + compile_flags + (["-Xptxas", "-v"] if verbose else []) + \
                ["-c", os.path.join(CSRC, src), "-o", obj]
            return obj, subprocess.run(cmd, capture_output=True, text=True)
        with concurrent.futures.ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 1)) as pool:
            results = list(pool.map(one, SOURCES))
        for obj, res in results:
            if res.returncode != 0:
                sys.stderr.write(res.stdout + res.stderr)
                raise RuntimeError("nvcc failed building libsaga_b200.so")
            if verbose:
                sys.stderr.write(res.stderr)
        link = [nvcc, "-shared", "-Xcompiler", "-fPIC", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + \
            [obj for obj, _ in results] + ["-lcuda"]
        res = subprocess.run(link, capture_output=True, text=True)
        if res.returncode != 0:
            sys.stderr.write(res.stdout + res.stderr)
            raise RuntimeError("nvcc failed linking libsaga_b200.so")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
