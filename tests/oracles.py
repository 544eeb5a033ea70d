"""Loaders for the CPU checkers under oracle/ (TEST INFRASTRUCTURE; the product never imports this)."""
import ctypes
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pathtracer_b200._abi import Lib  # noqa: E402

REF_SO = os.path.join(ROOT, "oracle", "_ref", "libptb_ref.so")
PORT_SO = os.path.join(ROOT, "oracle", "port", "libptb_port.so")
_cache = {}


def reference_dir():
    """The checkout of the reference (nbonneel/pathtracer) that PTB_REFERENCE_DIR names, or None.  The repository holds only the
    reference's outputs (tests/golden/); its sources, and oracle/_ref built from them, come from there or not at all."""
    d = os.environ.get("PTB_REFERENCE_DIR")
    return d if d and os.path.isdir(d) else None


def build_ref():
    """Compile oracle/_ref from reference_dir() (oracle/build_ref.py)."""
    subprocess.check_call([sys.executable, os.path.join(ROOT, "oracle", "build_ref.py"), reference_dir()])


def ref_lib():
    """oracle/_ref: the reference's own sources compiled headless (None if it was never built)."""
    if "ref" not in _cache:
        if not os.path.exists(REF_SO) and reference_dir():
            build_ref()
        _cache["ref"] = Lib(ctypes.CDLL(REF_SO, mode=ctypes.RTLD_LOCAL), "ref_") if os.path.exists(REF_SO) else None
    return _cache["ref"]


def port_lib():
    """oracle/port: plain-C restatement; always buildable (gcc only)."""
    if "port" not in _cache:
        if not os.path.exists(PORT_SO):
            subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle", "port"), "-s"])
        _cache["port"] = Lib(ctypes.CDLL(PORT_SO, mode=ctypes.RTLD_LOCAL), "orc_")
    return _cache["port"]

DEVSIM_SO = os.path.join(ROOT, "tests", "devsim", "libptb_devsim.so")


def devsim_lib():
    """tests/devsim: the DEVICE headers compiled for the host (debugging aid, see devsim.cpp)."""
    if "sim" not in _cache:
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "tests", "devsim"), "-s"])
        _cache["sim"] = Lib(ctypes.CDLL(DEVSIM_SO, mode=ctypes.RTLD_LOCAL), "sim_")
    return _cache["sim"]
