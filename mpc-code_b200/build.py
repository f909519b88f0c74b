"""Compile the per-problem CUDA library (generated model header + hand-written kernels) for sm_100a.

One shared object per problem, kept in-tree under ``mpc-code_b200/_build/`` and keyed by a hash of
the generated header and the kernel sources, so a second build of the same problem is a no-op.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import tempfile

from .devicegen import generate_header

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
INCLUDE = os.path.join(os.path.dirname(PKG_DIR), "include")
BUILD_DIR = os.path.join(PKG_DIR, "_build")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]
_SOURCES = ("mpcb_api.cu", "mpcb_device.cuh", "mpcb_ocp.cuh", "mpcb_target.cuh", "mpcb_sens.cuh")


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: the CUDA library cannot be built (there is no CPU fallback)")
    return exe


def build_dir_for(path: str, artefact: str) -> str:
    """Where to keep ``artefact``: ``path`` (in the tree) when it is already there or ``path`` can be written, else a
    per-user directory under the system temporary directory, so that a read-only tree compiles what it lacks there."""
    if os.path.exists(os.path.join(path, artefact)):
        return path
    probe = path
    while not os.path.exists(probe):
        probe = os.path.dirname(probe)
    if os.access(probe, os.W_OK):
        return path
    return os.path.join(tempfile.gettempdir(), "mpc_code_b200_%d" % os.getuid(), os.path.basename(os.path.dirname(path)))


def source_digest(header_text: str) -> str:
    hsh = hashlib.sha256(header_text.encode())
    for name in _SOURCES:
        with open(os.path.join(CSRC, name), "rb") as fh:
            hsh.update(fh.read())
    with open(os.path.join(INCLUDE, "mpcb.h"), "rb") as fh:
        hsh.update(fh.read())
    hsh.update(" ".join(NVCC_FLAGS).encode())
    return hsh.hexdigest()[:16]


def build_library(name: str, prob, ss_spec, ocp_spec, verbose: bool = False, extra_flags=()) -> dict:
    """Generate the header and compile; returns ``{"so": path, "header": path, "gen": generate_header(...)}``.

    ``MPCB_EXTRA_FLAGS`` (environment, space separated) appends nvcc flags - used by the tuning scripts to try
    kernel mappings (e.g. ``-DMPCB_KKT_LANES=32``)."""
    extra_flags = tuple(extra_flags) + tuple(os.environ.get("MPCB_EXTRA_FLAGS", "").split())
    gen = generate_header(prob, ss_spec, ocp_spec)
    digest = source_digest(gen["text"] + " ".join(extra_flags))
    base = build_dir_for(BUILD_DIR, "libmpcb_%s_%s.so" % (name, digest))
    work = os.path.join(base, "%s_%s" % (name, digest))
    so_path = os.path.join(base, "libmpcb_%s_%s.so" % (name, digest))
    header = os.path.join(work, "mpcb_model.h")
    os.makedirs(work, exist_ok=True)
    if not os.path.exists(header):          # published atomically: several ranks may start on a cold _build at once
        tmp_h = header + ".tmp%d" % os.getpid()
        with open(tmp_h, "w") as fh:
            fh.write(gen["text"])
        os.replace(tmp_h, header)
    if not os.path.exists(so_path):
        tmp = so_path + ".tmp%d" % os.getpid()
        cmd = [_nvcc(), *NVCC_FLAGS, *extra_flags, "-I", work, "-I", CSRC, "-I", INCLUDE,
               "-o", tmp, os.path.join(CSRC, "mpcb_api.cu")]
        if verbose:
            cmd.insert(1, "-Xptxas"); cmd.insert(2, "-v")
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("nvcc failed:\n%s\n%s" % (" ".join(cmd), res.stderr[-4000:]))
        if verbose:
            print(res.stderr)
        os.replace(tmp, so_path)
    return dict(so=so_path, header=header, gen=gen, digest=digest)
