"""In-tree build of the CUDA engine (liburmb.so) and host tools for sm_100a."""
from __future__ import annotations

import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")


def _stale(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources if os.path.exists(s))


def is_current():
    """True when liburmb.so and the host tools are up to date with their sources (make -q: nothing is built)."""
    return subprocess.call(["make", "-q", "-C", CSRC], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL) == 0


def build_engine(force=False, verbose=False):
    """nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo ... -> urmap_b200/liburmb.so (+ bin/urmap_b200)."""
    out = None if verbose else subprocess.DEVNULL
    args = ["make", "-j4", "-C", CSRC]
    if force:
        args.append("-B")
    subprocess.check_call(args, stdout=out)
    return os.path.join(HERE, "liburmb.so")
