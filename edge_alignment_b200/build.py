"""Builds edge_alignment_b200/libea_b200.so with nvcc for sm_100a (in-tree, so it travels with gpurun)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libea_b200.so")
SOURCES = ["ea_cabi.cu", "ea_solve.cu", "ea_preprocess.cu", "ea_canny_edt.cu", "ea_tracker.cu", "ea_shard.cu", "ea_views.cu", "ea_views_batch.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC,-Wall,-Wno-unused-function", "--expt-relaxed-constexpr",
              "-I", os.path.join(ROOT, "include"), "-I", CSRC]


def nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError("nvcc not found")


def needs_build():
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(ROOT, "include", "ea_cabi.h"), __file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return SO
    os.makedirs(os.path.join(HERE, "_obj"), exist_ok=True)
    objs = []
    procs = []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        if not os.path.exists(src):
            continue
        obj = os.path.join(HERE, "_obj", s.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    cmd = [nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", SO] + objs + ["-lcudart", "-ldl"]
    subprocess.check_call(cmd)
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
