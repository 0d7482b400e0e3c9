"""Builds rustsasa_b200/libsasa_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "csrc", "sasa_api.cu")
DEPS = [os.path.join(HERE, "csrc", f) for f in ("sasa_api.cu", "sasa_device.cuh", "sasa_tight.cuh", "sasa_cap.cuh", "sasa_small.cuh", "sasa_large.cuh", "sasa_pair_sums.cuh")]
DEPS.append(os.path.join(os.path.dirname(HERE), "include", "sasa_b200.h"))
OUT = os.path.join(HERE, "libsasa_b200.so")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC,-fvisibility=hidden", "-shared", "--cudart", "static"]


def needs_build() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(d) > t for d in DEPS)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return OUT
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", OUT, SRC]
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose:
        print(r.stdout)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + r.stdout)
    return OUT


HOST_DIR = os.path.join(HERE, "csrc", "host")
HOST_SRCS = [os.path.join(HOST_DIR, f) for f in ("structure.cpp", "options.cpp", "writers.cpp", "capi.cpp")]
HOST_OUT = os.path.join(HERE, "libsasa_b200_host.so")
CLI_OUT = os.path.join(HERE, "sasa_b200_cli")
HOST_HDRS = [os.path.join(os.path.dirname(HERE), "include", f) for f in ("sasa_b200.h", "sasa_b200.hpp")]
PROTOR = os.path.join(os.path.dirname(HERE), "radii", "protor.config")
PROTOR_INC = os.path.join(HOST_DIR, "protor_config.inc")


def build_host(force: bool = False) -> str:
    """C++ host layer (include/sasa_b200.hpp) + the sasa_b200_cli binary; plain g++, links the C ABI library only."""
    build()
    deps = HOST_SRCS + HOST_HDRS + [os.path.join(HOST_DIR, "cli.cpp"), PROTOR, OUT]
    if not force and os.path.exists(HOST_OUT) and os.path.exists(CLI_OUT):
        t = min(os.path.getmtime(HOST_OUT), os.path.getmtime(CLI_OUT))
        if all(os.path.getmtime(d) <= t for d in deps):
            return HOST_OUT
    # the ProtOr table is embedded like the reference's include_str! (src/utils/consts.rs:22-29)
    with open(PROTOR) as fh:
        text = fh.read()
    assert ')PROTOR"' not in text
    with open(PROTOR_INC, "w") as fh:
        fh.write('R"PROTOR(' + text + ')PROTOR"\n')
    gxx = os.environ.get("CXX_HOST", "/usr/bin/g++")
    common = [gxx, "-O2", "-std=c++17", "-fPIC", "-fvisibility=hidden", "-Wall", "-pthread"]
    link = ["-L" + HERE, "-lsasa_b200", "-Wl,-rpath,$ORIGIN"]
    for cmd in (common + ["-shared", "-o", HOST_OUT] + HOST_SRCS + link,
                common + ["-o", CLI_OUT, os.path.join(HOST_DIR, "cli.cpp")] + HOST_SRCS[:3] + link):
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if r.returncode != 0:
            raise RuntimeError("g++ failed:\n" + r.stdout)
    return HOST_OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
    print(build_host(force="--force" in sys.argv))
