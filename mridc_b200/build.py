"""Build recipe for libmridc_b200.so (hand-written CUDA for sm_100a, C-ABI in include/mridc_b200.h) and
libmridc_b200_espirit.so (coil-sensitivity estimation, C-ABI in include/mridc_b200_espirit.h).

The library is built IN-TREE (mridc_b200/libmridc_b200.so) with nvcc so that it travels with the source
snapshot to the GPU box; nvcc cross-compiles without a GPU.  `python -m mridc_b200.build` or
`__graft_entry__.build()`.
"""
import hashlib
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libmridc_b200.so")
STAMP = os.path.join(PKG_DIR, "csrc", ".build_stamp")
SOURCES = ["core.cu", "fft.cu", "dc.cu", "conv.cu", "unet.cu", "conv_tc.cu", "conv_tc2.cu", "qmri.cu", "metrics.cu"]
# ESPIRiT library: a library of its own (no core.cu); its transforms come from libmridc_b200.so through Python
ESPIRIT_SOURCES = ["espirit.cu"]
ESPIRIT_HEADER = os.path.join(PKG_DIR, "..", "include", "mridc_b200_espirit.h")
ESPIRIT_LIB_PATH = os.path.join(PKG_DIR, "libmridc_b200_espirit.so")
ESPIRIT_STAMP = os.path.join(PKG_DIR, "csrc", ".build_stamp_espirit")
# tools-only library (tools/libmridc_b200_tools.so): the tensor-core kernels with their per-role cycle counters and role
# switches compiled in (-DMRB_TC_PROF) plus the tcgen05 issue micro-benchmark; never loaded by the package
TOOLS_SOURCES = ["core.cu", "conv_tc.cu", "conv_tc2.cu", "conv.cu", "tc_microbench.cu"]
TOOLS_LIB_PATH = os.path.join(PKG_DIR, "..", "tools", "libmridc_b200_tools.so")
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
] + os.environ.get("MRIDC_B200_NVCC_EXTRA", "").split()  # extra nvcc flags for experiments (part of the build digest)


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; cannot build libmridc_b200.so")


def _digest():
    h = hashlib.sha256()
    for root, _, files in sorted(os.walk(CSRC)):
        for f in sorted(files):
            if f.endswith((".cu", ".cuh", ".h")) and f not in ESPIRIT_SOURCES:
                with open(os.path.join(root, f), "rb") as fh:
                    h.update(f.encode() + b"\0" + fh.read())
    with open(os.path.join(PKG_DIR, "..", "include", "mridc_b200.h"), "rb") as fh:
        h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS + SOURCES).encode())
    return h.hexdigest()


def _espirit_digest():
    h = hashlib.sha256()
    for f in ESPIRIT_SOURCES:
        with open(os.path.join(CSRC, f), "rb") as fh:
            h.update(f.encode() + b"\0" + fh.read())
    with open(ESPIRIT_HEADER, "rb") as fh:
        h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def _fresh(path, stamp, digest):
    if os.path.exists(path) and os.path.exists(stamp):
        with open(stamp) as fh:
            return fh.read().strip() == digest
    return False


def build(force=False, verbose=False):
    """Compile every CUDA source for sm_100a: libmridc_b200.so and libmridc_b200_espirit.so. Returns the path of the
    first."""
    digest = _digest()
    if force or not _fresh(LIB_PATH, STAMP, digest):
        _compile(SOURCES, LIB_PATH, os.path.join(PKG_DIR, "csrc", "build"), verbose)
        with open(STAMP, "w") as fh:
            fh.write(digest)
    digest = _espirit_digest()
    if force or not _fresh(ESPIRIT_LIB_PATH, ESPIRIT_STAMP, digest):
        _compile(ESPIRIT_SOURCES, ESPIRIT_LIB_PATH, os.path.join(PKG_DIR, "csrc", "build", "espirit"), verbose)
        with open(ESPIRIT_STAMP, "w") as fh:
            fh.write(digest)
    return LIB_PATH


def _compile(sources, lib_path, objdir, verbose):
    nvcc = _nvcc()
    os.makedirs(objdir, exist_ok=True)
    procs = []
    objs = []
    for src in sources:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            failed = True
            sys.stderr.write("nvcc failed on %s:\n%s\n" % (src, out))
        elif verbose or "warning" in out:
            sys.stderr.write(out)
    if failed:
        raise RuntimeError("nvcc compilation failed")
    cmd = [nvcc, "-shared", "-Wno-deprecated-gpu-targets", "-o", lib_path] + objs + ["-lcudart"]
    subprocess.check_call(cmd)


def build_tools():
    """tools/libmridc_b200_tools.so: profiling build of the tensor-core kernels (see TOOLS_SOURCES)."""
    nvcc = _nvcc()
    objdir = os.path.join(PKG_DIR, "csrc", "build", "tools")
    os.makedirs(objdir, exist_ok=True)
    objs, procs = [], []
    for src in TOOLS_SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc] + NVCC_FLAGS + ["-DMRB_TC_PROF", "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError("nvcc failed on %s:\n%s" % (src, out))
    subprocess.check_call([nvcc, "-shared", "-Wno-deprecated-gpu-targets", "-o", TOOLS_LIB_PATH] + objs + ["-lcudart"])
    return TOOLS_LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
    if "--tools" in sys.argv:
        print(build_tools())
