"""ctypes bindings of the pcl::CropBox statements used by the tests (TEST INFRASTRUCTURE ONLY):
  crop_box      the C++ oracle, tests/crop_box_oracle.cpp (cmo_crop_box);
  pcl_crop_box  the real PCL class behind tests/crop_box_pcl_ref.cpp (cmp_crop_box), where PCL is installed.
Both are compiled on first use into a per-user directory under the system temporary directory, keyed by the hash of the
source and flags, so the repository tree is never written."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# the flags of oracle/Makefile: no -march / -ffast-math / FMA contraction, so float mul/add round separately
CXXFLAGS = ["-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-Wall", "-Wextra"]
_LIBS = {}
_WHY = ""


def _build(src: str, extra_flags=()) -> str:
    flags = CXXFLAGS + list(extra_flags)
    text = open(src, "rb").read()
    key = hashlib.sha256(text + " ".join(flags).encode()).hexdigest()[:16]
    d = os.path.join(tempfile.gettempdir(), "cm_crop_box_oracle_%d" % os.getuid())
    os.makedirs(d, exist_ok=True)
    so = os.path.join(d, "%s_%s.so" % (os.path.splitext(os.path.basename(src))[0], key))
    if not os.path.exists(so):
        tmp = so + ".%d.tmp" % os.getpid()
        subprocess.run([os.environ.get("CXX", "g++")] + flags + ["-o", tmp, src], check=True, capture_output=True, text=True)
        os.replace(tmp, so)
    return so


class CmoCropBox(C.Structure):
    _fields_ = [("min", C.c_float * 3), ("max", C.c_float * 3), ("translation", C.c_float * 3), ("rotation", C.c_float * 3),
                ("transform", C.c_float * 12), ("negative", C.c_int32), ("reserved", C.c_int32)]


def make_crop_box(box: dict) -> CmoCropBox:
    """box: dict(min, max, translation=0, rotation=0 (roll, pitch, yaw), transform=identity 3x4, negative=False)."""
    b = CmoCropBox()
    t = np.asarray(box.get("transform", np.eye(3, 4)), np.float32).reshape(-1)[:12]
    for k in range(3):
        b.min[k] = float(np.float32(box["min"][k])); b.max[k] = float(np.float32(box["max"][k]))
        b.translation[k] = float(np.float32(box.get("translation", (0, 0, 0))[k]))
        b.rotation[k] = float(np.float32(box.get("rotation", (0, 0, 0))[k]))
    for k in range(12):
        b.transform[k] = float(t[k])
    b.negative = int(bool(box.get("negative", False)))
    return b


def _lib():
    if "cmo" not in _LIBS:
        L = C.CDLL(_build(os.path.join(HERE, "crop_box_oracle.cpp")))
        L.cmo_crop_box.restype = C.c_int64
        L.cmo_crop_box.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.POINTER(CmoCropBox), C.c_void_p]
        _LIBS["cmo"] = L
    return _LIBS["cmo"]


def crop_box(xyzi: np.ndarray, is_dense: bool, box: dict) -> np.ndarray:
    """One pcl::CropBox stage (cmo_crop_box): indices of the kept points, in input order."""
    xyzi = np.ascontiguousarray(xyzi, np.float32).reshape(-1, 4)
    idx = np.empty(max(len(xyzi), 1), np.int32)
    b = make_crop_box(box)
    k = _lib().cmo_crop_box(xyzi.ctypes.data, len(xyzi), int(bool(is_dense)), C.byref(b), idx.ctypes.data)
    return idx[:k].copy()


# ---- the real PCL ------------------------------------------------------------------------------------------------------------
def pcl_available() -> bool:
    """Builds the real-PCL wrapper when pkg-config finds PCL's filters module (>= 1.8); never raises."""
    global _WHY
    if "pcl" in _LIBS:
        return True
    if not shutil.which("pkg-config"):
        _WHY = "pkg-config not found"
        return False
    mods = None
    for ver in ("1.8", "1.9", "1.10", "1.11", "1.12", "1.13", "1.14"):
        m = ["pcl_filters-" + ver, "pcl_common-" + ver, "eigen3"]
        if subprocess.run(["pkg-config", "--exists"] + m).returncode == 0:
            mods = m
            break
    if mods is None:
        _WHY = "PCL >= 1.8 not found by pkg-config (pcl_filters)"
        return False
    flags = subprocess.run(["pkg-config", "--cflags", "--libs"] + mods, capture_output=True, text=True).stdout.split()
    try:
        L = C.CDLL(_build(os.path.join(HERE, "crop_box_pcl_ref.cpp"), flags))
    except (subprocess.CalledProcessError, OSError) as e:
        _WHY = "building tests/crop_box_pcl_ref.cpp failed: %s" % (getattr(e, "stderr", "") or e)[-400:]
        return False
    L.cmp_crop_box.restype = C.c_int64
    _LIBS["pcl"] = L
    return True


def pcl_why_not() -> str:
    return _WHY or "the real-PCL CropBox wrapper is not built"


def pcl_crop_box(xyzi, is_dense, box) -> np.ndarray:
    """pcl::CropBox itself: indices kept. box as for crop_box."""
    xyzi = np.ascontiguousarray(xyzi, np.float32).reshape(-1, 4)
    b = np.concatenate([np.asarray(box[k], np.float32).reshape(-1) for k in ("min", "max", "translation", "rotation")] +
                       [np.asarray(box["transform"], np.float32).reshape(-1)[:12]]).astype(np.float32)
    idx = np.empty(max(len(xyzi), 1), np.int32)
    k = _LIBS["pcl"].cmp_crop_box(xyzi.ctypes.data_as(C.c_void_p), C.c_int64(len(xyzi)), int(bool(is_dense)),
                                  b.ctypes.data_as(C.c_void_p), int(bool(box["negative"])), idx.ctypes.data_as(C.c_void_p))
    return idx[:k].copy()
