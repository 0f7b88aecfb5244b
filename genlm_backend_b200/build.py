"""Build recipe for the in-tree C-ABI library ``libgenlm_trie_b200.so`` (nvcc, sm_100a only).

``python -m genlm_backend_b200.build`` compiles ``csrc/*.cpp`` and ``csrc/*.cu`` into
``genlm_backend_b200/libgenlm_trie_b200.so``.  nvcc cross-compiles without a GPU, so this runs in the
dev container; the built library travels to the GPU box with the source tree (it is git-ignored).
"""
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
# GT_LIB_NAME / GT_NVCC_DEFINES: build (and load) an experimental variant next to the default library, e.g.
#   GT_LIB_NAME=libgt_cw8.so GT_NVCC_DEFINES=-DGT_COMPUTE_WARPS=8 python genlm_backend_b200/build.py
LIB_NAME = os.environ.get("GT_LIB_NAME", "libgenlm_trie_b200.so")
LIB_PATH = os.path.join(PKG_DIR, LIB_NAME)
EXTRA_DEFINES = os.environ.get("GT_NVCC_DEFINES", "").split()
INCLUDE = os.path.join(os.path.dirname(PKG_DIR), "include")

SOURCES = ["trie_builder.cpp", "trie_plan.cpp", "device_plan.cu", "mass_kernels.cu", "token_mask_kernels.cu",
           "child_kernels.cu", "sampler_kernels.cu"]
HEADERS = [os.path.join(CSRC, h) for h in ("trie_internal.h", "trie_device.cuh", "philox.cuh")] + [
    os.path.join(INCLUDE, "genlm_trie_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC,-O3,-Wall,-Wno-unknown-pragmas",
    "--expt-relaxed-constexpr",
]


def _nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: the CUDA toolkit is required to build " + LIB_NAME)
    return exe


def needs_build():
    if not os.path.exists(LIB_PATH):
        return True
    built = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + HEADERS + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > built for d in deps)


def build(force=False, verbose=False):
    """Compile the library if any source is newer than it.  Returns the path of the .so."""
    if not force and not needs_build():
        return LIB_PATH
    nvcc = _nvcc()
    objdir = os.path.join(PKG_DIR, "build", os.path.splitext(LIB_NAME)[0])
    os.makedirs(objdir, exist_ok=True)
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, os.path.splitext(src)[0] + ".o")
        cmd = [nvcc] + NVCC_FLAGS + EXTRA_DEFINES + ["-I", INCLUDE, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd), flush=True)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(out)
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed building " + LIB_NAME)
    tmp = LIB_PATH + ".tmp"
    link = [nvcc, "-shared", "-o", tmp] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static", "-ldl"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError("link failed for " + LIB_NAME)
    os.replace(tmp, LIB_PATH)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
