"""Build libsupnerf_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).  Every source is compiled to its
own object file in parallel (only those older than their source or than any header), then linked."""
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "_build")
LIB = os.path.join(HERE, "libsupnerf_b200.so")
SOURCES = ["api.cu", "composite.cu", "sampler.cu", "latent.cu", "mlp_f32.cu", "mlp_tc.cu", "mlp_tc2.cu", "decoder.cu", "render.cu", "loss.cu",
           "compact.cu", "scene.cu", "refine.cu", "render_batch.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC"]  # no --use_fast_math: sinf/expf accuracy is part of parity
NVCC_FLAGS += os.environ.get("SNB_EXTRA_NVCC_FLAGS", "").split()   # tuning builds only (e.g. -DSNB_EXP_... timing experiments)


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _headers():
    hs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    return hs + [os.path.join(os.path.dirname(HERE), "include", "supnerf_b200.h")]


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + _headers()
    return any(os.path.getmtime(d) > t for d in deps)


def _flags_changed():
    """True when the objects on disk were compiled with other flags (a tuning build left behind): everything is rebuilt."""
    stamp = os.path.join(OBJ, "flags.txt")
    want = " ".join(NVCC_FLAGS)
    have = open(stamp).read() if os.path.exists(stamp) else None
    if have == want:
        return False
    os.makedirs(OBJ, exist_ok=True)
    open(stamp, "w").write(want)
    return have is not None or os.path.exists(LIB) and bool(os.environ.get("SNB_EXTRA_NVCC_FLAGS"))


def build(force=False, verbose=False):
    force = force or _flags_changed()
    if not force and not needs_build():
        return LIB
    os.makedirs(OBJ, exist_ok=True)
    nvcc = _nvcc()
    hdr_time = max(os.path.getmtime(h) for h in _headers())

    def compile_one(src):
        s, o = os.path.join(CSRC, src), os.path.join(OBJ, src[:-3] + ".o")
        if not force and os.path.exists(o) and os.path.getmtime(o) > max(os.path.getmtime(s), hdr_time):
            return o, ""
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed on %s:\n%s%s" % (src, r.stdout, r.stderr))
        return o, r.stderr

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 4)) as ex:
        results = list(ex.map(compile_one, SOURCES))
    if verbose:
        for _, err in results:
            sys.stderr.write(err)
    tmp = LIB + ".tmp"
    # -cudart shared: the static runtime would embed the names of every runtime entry point (ADVICE r1) in the .so
    r = subprocess.run([nvcc, "-shared", "-cudart", "shared", "-o", tmp] + [o for o, _ in results], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    os.replace(tmp, LIB)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
