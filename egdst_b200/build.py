"""nvcc driver: one sm_100a shared library per generated model image.

Replaces the ``mex`` invocations of the reference's compile step (@egdstmodel/compile.m:754-819):
the user's exec strings, translated by ``codegen.emit_devspec``, are compiled *into* the solver and
simulator kernels (``egdst_b200/csrc``).  Libraries are kept in-tree under ``egdst_b200/_lib/<key>/``
(git-ignored, but they travel to the GPU box) and are keyed by the generated source, so models that
differ only in run-time properties (grid sizes, horizon, parameter values) share one image.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess

from . import codegen

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(ROOT, "include")
LIBROOT = os.environ.get("EGDST_B200_LIB_DIR", os.path.join(HERE, "_lib"))

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--shared", "-fmad=false"] + os.environ.get("EGDST_NVCC_EXTRA", "").split()

_SOURCES = ["egdst_capi.cu", "egdst_capi_sim.inc", "egdst_common.cuh", "egdst_envelope.cuh", "egdst_loglik.cuh",
            "egdst_numerics.cuh", "egdst_period.cuh", "egdst_simulator.cuh", "egdst_solver.cuh", "egdst_tables.cuh"]


def source_digest() -> str:
    h = hashlib.sha1()
    for name in _SOURCES:
        with open(os.path.join(CSRC, name), "rb") as f:
            h.update(f.read())
    for name in ("egdst_b200.h", "egdst_modelctx.h"):
        with open(os.path.join(INCLUDE, name), "rb") as f:
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()[:12]


def library_path(model) -> str:
    key = codegen.model_key(model)
    return os.path.join(LIBROOT, key, "libegdst_b200_%s.so" % key)


def find_nvcc() -> str:
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.isfile(nvcc):
        raise RuntimeError("nvcc not found: the egdst_b200 model library can only be built with the CUDA toolkit")
    return nvcc


def build_model_library(model, force: bool = False, verbose: bool = False) -> str:
    """Generate modelspec_dev.h and compile the model image.  Returns the library path."""
    key = codegen.model_key(model)
    path = library_path(model)
    outdir = os.path.dirname(path)
    stamp = os.path.join(outdir, "build.stamp")
    digest = source_digest()
    if not force and os.path.isfile(path) and os.path.isfile(stamp) and open(stamp).read().strip() == digest:
        return path
    os.makedirs(outdir, exist_ok=True)
    with open(os.path.join(outdir, "modelspec_dev.h"), "w") as f:
        f.write(codegen.emit_devspec(model))
    cmd = [find_nvcc()] + NVCC_FLAGS + ["-I" + outdir, "-I" + INCLUDE, "-I" + CSRC,
                                        '-DEGDST_MODEL_KEY="%s"' % key,
                                        os.path.join(CSRC, "egdst_capi.cu"), "-o", path]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed for model '%s':\n%s\n%s" % (model.label, res.stdout, res.stderr))
    if verbose:
        print(res.stderr)
    with open(stamp, "w") as f:
        f.write(digest + "\n")
    return path
