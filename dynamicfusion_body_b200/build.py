"""Build libdfb_b200.so in-tree with nvcc for sm_100a (B200).  `python -m dynamicfusion_body_b200.build`

Every translation unit is compiled to its own object (in parallel, cached under csrc/_obj/ by modification time) and the
objects are linked into the shared library, so touching one kernel file recompiles only that file."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

_PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_PKG, "csrc")
OBJ = os.path.join(CSRC, "_obj")
OUT = os.path.join(_PKG, "libdfb_b200.so")
SOURCES = ["common.cu", "tsdf.cu", "knn.cu", "gn.cu", "graph.cu", "mc.cu", "comm.cu", "step.cu", "render.cu", "track.cu", "raycast.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC"]


def _headers():
    return [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".h")] + [os.path.join(os.path.dirname(_PKG), "include", "dfb.h")]


def _stale():
    if not os.path.isfile(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in SOURCES] + _headers()
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, extra_flags=(), out=None):
    out = out or OUT
    if not force and out == OUT and not _stale():
        return OUT
    nvcc = os.environ.get("NVCC", "nvcc")
    os.makedirs(OBJ, exist_ok=True)
    tag = ("_" + "_".join(f.replace("-", "").replace("=", "") for f in extra_flags)) if extra_flags else ""
    hdr_t = max(os.path.getmtime(h) for h in _headers())
    jobs = []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        obj = os.path.join(OBJ, s[:-3] + tag + ".o")
        if force or verbose or not os.path.isfile(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), hdr_t):
            jobs.append((src, obj))

    def compile_one(job):
        src, obj = job
        cmd = [nvcc] + NVCC_FLAGS + list(extra_flags) + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
        return job, subprocess.run(cmd, capture_output=True, text=True)

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        for (src, obj), res in ex.map(compile_one, jobs):
            if res.returncode != 0:
                sys.stderr.write(res.stdout + res.stderr)
                raise RuntimeError("nvcc failed compiling %s" % os.path.basename(src))
            if verbose:
                sys.stderr.write(res.stderr)
    objs = [os.path.join(OBJ, s[:-3] + tag + ".o") for s in SOURCES]
    res = subprocess.run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a"] + objs + ["-o", out, "-ldl"], capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed linking libdfb_b200.so")
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
