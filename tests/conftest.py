import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")
REFERENCE_PINS = os.path.join(GOLDEN, "reference_pins.json")

GOLDEN_CASES = [
    "hw4", "reflectance", "dof", "spherelight", "spheres_blur", "checkertexture", "checkertexture_nogloss",
    "texture", "textureog", "window", "staircase", "rectprism", "checkercylinder", "chkpt2_mocap", "boundary_mocap",
    # the slab-box prism classes (SURVEY 8a a14): the reference's own `prismcyl` scene, and scenes that put RectPrism /
    # RectPrismWithCylinder / RectPrismWithHoles in front of its constructors (tests/golden/make_golden.py)
    "prismcyl", "prism_box", "prism_cyl", "prism_cyl_side", "prism_holes", "prism_holes_back",
]
# In the reference a hit on the wall of a prism's hole WRITES the hole's colour into the prism for good (geometry.cpp:1650,
# 2005, 2044): every later ray sees it, so its picture depends on the order the pixels are rendered in.  The oracle
# reproduces that to the bit under DRT_ORACLE_Q19=persist (sequential mode only); by default -- and in the CUDA path -- the
# colour belongs to the hit that set it (DESIGN.md, Q19).
Q19_CASES = {"prism_cyl", "prism_cyl_side", "prism_holes", "prism_holes_back"}


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run with -m gpu on the B200 box)")


@pytest.fixture(scope="session")
def oracle_lib():
    """Build (if needed) and return the path of oracle/liboracle.so -- the checker, never the product."""
    so = os.path.join(ROOT, "oracle", "liboracle.so")
    srcs = [os.path.join(ROOT, "oracle", f) for f in ("drt_oracle.cpp", "drt_skeleton_oracle.cpp")]
    if not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(src) for src in srcs):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "liboracle.so"])
    return so


def load_case(name):
    from distraytracer_b200.scene import load_fixture
    return load_fixture(os.path.join(GOLDEN, name + ".npz"))


def _digest(*arrays):
    """SHA-256 over dtypes, shapes and bytes; every NaN is hashed as the same quiet NaN (equal_nan comparisons)."""
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        if a.dtype.kind == "f":
            a = np.where(np.isnan(a), np.array(np.nan, dtype=a.dtype), a)
        h.update(repr((a.dtype.str, a.shape)).encode()); h.update(a.tobytes())
    return h.hexdigest()


def assert_pinned(key, *arrays, matched_reference):
    """`arrays` equal, to the bit, the ones whose digest tests/golden/reference_pins.json holds for `key`: the compiled
    reference's output for that case (provenance: tests/golden/README.md).  With DRT_RECORD_PINS=1 the digest is stored
    instead, and only for arrays the caller has just found equal to the live reference's (`matched_reference`): a pin
    never records what the restatement alone computes."""
    pins = json.load(open(REFERENCE_PINS)) if os.path.exists(REFERENCE_PINS) else {}
    if os.environ.get("DRT_RECORD_PINS"):
        if not matched_reference:
            pytest.fail(f"{key}: recording a pin needs the compiled reference (oracle/_ref and the reference tree)")
        pins[key] = _digest(*arrays)
        with open(REFERENCE_PINS, "w") as f:
            json.dump(dict(sorted(pins.items())), f, indent=0)
            f.write("\n")
        return
    assert key in pins, f"no stored pin for {key}"
    assert _digest(*arrays) == pins[key], f"{key}: the restatement no longer reproduces the reference's output"
