"""Build the CUDA library in-tree with nvcc for sm_100a (no JIT cache, no torch extension machinery).

The shared object lands in ``chainer-speech-recognition_b200/_lib/libb200ctc.so`` so that it travels
with the repository snapshot to the GPU box (it is git-ignored, not gpurun-ignored).
"""
import fcntl
import hashlib
import os
import shutil
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "_lib")
SO_PATH = os.path.join(LIBDIR, "libb200ctc.so")
STAMP = os.path.join(LIBDIR, "libb200ctc.stamp")
SOURCES = ["api.cu", "host_cache.cu", "softmax_gather.cu", "lattice.cu", "gradient.cu", "greedy_error.cu", "layernorm_loss.cu",
           "viterbi.cu"]
HEADERS = ["common.cuh", "kernels.h", "row_ring.cuh", "prep.cuh", os.path.join("..", "..", "include", "b200ctc.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared", "-cudart", "shared"]


def find_nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    return None


def source_hash():
    h = hashlib.sha256()
    for name in SOURCES + HEADERS:
        with open(os.path.join(CSRC, name), "rb") as f:
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def is_current():
    if not (os.path.exists(SO_PATH) and os.path.exists(STAMP)):
        return False
    with open(STAMP) as f:
        return f.read().strip() == source_hash()


def build(force=False, verbose=False):
    """Compile csrc/*.cu -> _lib/libb200ctc.so.  Returns the path.  Raises if nvcc is missing.

    Safe against concurrent callers: an exclusive lock on _lib/.build.lock serialises them, the compiler writes to a
    temporary file in the same directory and the result is renamed into place (a process that has the old file
    mapped keeps it), so nobody ever dlopens a half-written library."""
    if not force and is_current():
        return SO_PATH
    nvcc = find_nvcc()
    if nvcc is None:
        raise RuntimeError("nvcc not found: cannot build libb200ctc.so (and there is no CPU fallback)")
    os.makedirs(LIBDIR, exist_ok=True)
    with open(os.path.join(LIBDIR, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and is_current():                 # another process built it while we waited
                return SO_PATH
            env = dict(os.environ)
            env.pop("CC", None)      # the image exports a broken CC wrapper; let nvcc find the PATH g++
            env.pop("CXX", None)
            fd, tmp = tempfile.mkstemp(prefix="libb200ctc.", suffix=".so.tmp", dir=LIBDIR)
            os.close(fd)
            try:
                cmd = [nvcc] + NVCC_FLAGS + ["-o", tmp] + [os.path.join(CSRC, s) for s in SOURCES]
                if verbose:
                    print(" ".join(cmd))
                subprocess.check_call(cmd, env=env, cwd=CSRC)
                os.chmod(tmp, 0o755)
                os.replace(tmp, SO_PATH)
            finally:
                if os.path.exists(tmp):
                    os.unlink(tmp)
            with open(STAMP + ".tmp", "w") as f:
                f.write(source_hash())
            os.replace(STAMP + ".tmp", STAMP)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return SO_PATH


if __name__ == "__main__":
    print(build(force=True, verbose=True))
