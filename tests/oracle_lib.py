"""ctypes binding of the CPU oracle (oracle/libsift_oracle.so) -- TEST INFRASTRUCTURE.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may import this.
"""
from __future__ import annotations

import ctypes as C
import os
import struct
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
LIB_PATH = os.path.join(ORACLE_DIR, "libsift_oracle.so")

MODE = {"popsift": 0, "opencv": 1, "vlfeat": 2}
NORM = {"rootsift": 0, "classic": 1}


class OrcConfig(C.Structure):
    _fields_ = [("octaves", C.c_int32), ("levels", C.c_int32), ("sigma", C.c_float),
                ("edge_limit", C.c_float), ("threshold", C.c_float), ("upscale", C.c_float),
                ("initial_blur", C.c_float), ("has_initial_blur", C.c_int32),
                ("sift_mode", C.c_int32), ("norm_mode", C.c_int32), ("norm_multi", C.c_int32),
                ("max_extrema", C.c_int32), ("scaling_mode", C.c_int32), ("gauss_direct", C.c_int32), ("gauss_relative", C.c_int32), ("gauss_fixed", C.c_int32)]


class OrcGaussTable(C.Structure):
    _fields_ = [("filter", C.c_float * (12 * 32)), ("sigma", C.c_float * 12), ("span", C.c_int32 * 12)]


class OrcTables(C.Structure):
    _fields_ = [("inc", OrcGaussTable), ("dd_filter0", C.c_float * 32), ("dd_sigma0", C.c_float),
                ("dd_span0", C.c_int32), ("peak_threshold", C.c_float), ("sigma_k", C.c_float),
                ("dd_filter", C.c_float * (20 * 32)), ("dd_sigma", C.c_float * 20), ("dd_span", C.c_int32 * 20),
                ("abs_o0", OrcGaussTable), ("inc_ifilter", C.c_float * (12 * 32)), ("inc_ispan", C.c_int32 * 12),
                ("abs_oN", OrcGaussTable)]


FEATURE_DTYPE = np.dtype([("octave", "<i4"), ("x", "<f4"), ("y", "<f4"), ("sigma", "<f4"),
                          ("num_ori", "<i4"), ("ori", "<f4", (4,)), ("pad", "<i4"),
                          ("desc_idx", "<i8", (4,))])
assert FEATURE_DTYPE.itemsize == 72

_lib = None


def build_oracle() -> None:
    subprocess.check_call(["make", "-s", "-C", ORACLE_DIR, "libsift_oracle.so"])


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < os.path.getmtime(
                os.path.join(ORACLE_DIR, "sift_oracle.c")):
            build_oracle()
        L = C.CDLL(LIB_PATH)
        L.orc_create.restype = C.c_void_p
        L.orc_create.argtypes = [C.POINTER(OrcConfig), C.c_int, C.c_int]
        L.orc_destroy.argtypes = [C.c_void_p]
        L.orc_run_u8.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.orc_run_f32.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.orc_tex_f32.restype = C.c_float
        L.orc_tex_f32.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_float]
        L.orc_num_octaves.argtypes = [C.c_void_p]
        L.orc_octave_dims.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        L.orc_gauss_plane.restype = C.POINTER(C.c_float)
        L.orc_gauss_plane.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.orc_dog_plane.restype = C.POINTER(C.c_float)
        L.orc_dog_plane.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.orc_get_tables.restype = C.POINTER(OrcTables)
        L.orc_get_tables.argtypes = [C.c_void_p]
        L.orc_num_extrema.argtypes = [C.c_void_p]
        L.orc_get_extrema.argtypes = [C.c_void_p, C.c_void_p]
        L.orc_counts.argtypes = [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        L.orc_download.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_compute_tables.argtypes = [C.POINTER(OrcConfig), C.POINTER(OrcTables)]
        L.orc_geometry.argtypes = [C.POINTER(OrcConfig), C.c_int, C.c_int, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        L.orc_default_config.argtypes = [C.POINTER(OrcConfig)]
        L.orc_tex_u8.restype = C.c_float
        L.orc_tex_u8.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_float]
        L.orc_set_threads.argtypes = [C.c_int]
        _lib = L
    return _lib


def make_config(**kw) -> OrcConfig:
    c = OrcConfig()
    lib().orc_default_config(C.byref(c))
    for k, v in kw.items():
        if k == "mode":
            c.sift_mode = MODE[v]
        elif k == "norm":
            c.norm_mode = NORM[v]
        elif k == "downsampling":
            c.upscale = -float(v)
        elif k == "initial_blur":
            c.initial_blur = float(v)
            c.has_initial_blur = int(v != 0.0)          # Config::setInitialBlur (reference sift_conf.cu:246-255)
        else:
            assert hasattr(c, k), k
            setattr(c, k, v)
    return c


class Oracle:
    """One oracle context for a fixed config and image size."""

    def __init__(self, cfg: OrcConfig, w: int, h: int):
        self.cfg, self.w, self.h = cfg, w, h
        self.ctx = lib().orc_create(C.byref(cfg), w, h)
        if not self.ctx:
            raise RuntimeError("orc_create failed (sigma > 2 or too many levels)")

    def close(self):
        if self.ctx:
            lib().orc_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        self.close()

    def run(self, img: np.ndarray, stages: int = 15) -> None:
        """uint8 image -> ByteImages path; float32 image (values in [0,1]) -> FloatImages path"""
        assert img.shape == (self.h, self.w)
        if img.dtype == np.float32:
            img = np.ascontiguousarray(img)
            lib().orc_run_f32(self.ctx, img.ctypes.data, stages)
            return
        img = np.ascontiguousarray(img, dtype=np.uint8)
        lib().orc_run_u8(self.ctx, img.ctypes.data, stages)

    @property
    def num_octaves(self) -> int:
        return lib().orc_num_octaves(self.ctx)

    def dims(self, o: int):
        W, H = C.c_int32(), C.c_int32()
        lib().orc_octave_dims(self.ctx, o, C.byref(W), C.byref(H))
        return W.value, H.value

    def gauss(self, o: int, l: int) -> np.ndarray:
        W, H = self.dims(o)
        p = lib().orc_gauss_plane(self.ctx, o, l)
        return np.ctypeslib.as_array(p, shape=(H, W)).copy()

    def dog(self, o: int, l: int) -> np.ndarray:
        W, H = self.dims(o)
        p = lib().orc_dog_plane(self.ctx, o, l)
        return np.ctypeslib.as_array(p, shape=(H, W)).copy()

    def tables(self) -> OrcTables:
        return lib().orc_get_tables(self.ctx).contents

    def extrema(self) -> np.ndarray:
        n = lib().orc_num_extrema(self.ctx)
        out = np.zeros((n, 5), dtype=np.float32)
        if n:
            lib().orc_get_extrema(self.ctx, out.ctypes.data)
        return out

    def features(self):
        nf, nd = C.c_int32(), C.c_int32()
        lib().orc_counts(self.ctx, C.byref(nf), C.byref(nd))
        feat = np.zeros(nf.value, dtype=FEATURE_DTYPE)
        desc = np.zeros((nd.value, 128), dtype=np.float32)
        lib().orc_download(self.ctx, feat.ctypes.data, desc.ctypes.data)
        return feat, desc


# ---- readers for files written by the reference (oracle/ref_driver.cpp, write_plane_2d.cu:142-178)

def read_ref_dump(path: str) -> np.ndarray:
    with open(path, "rb") as f:
        data = f.read()
    nl1 = data.index(b"\n")
    assert data[:nl1] == b"floats"
    nl2 = data.index(b"\n", nl1 + 1)
    cols, rows = (int(t) for t in data[nl1 + 1:nl2].split())
    return np.frombuffer(data, dtype="<f4", count=rows * cols, offset=nl2 + 1).reshape(rows, cols).copy()


REF_FEATURE_DTYPE = np.dtype([("octave", "<i4"), ("x", "<f4"), ("y", "<f4"), ("sigma", "<f4"),
                              ("num_ori", "<i4"), ("ori", "<f4", (4,)), ("desc_idx", "<i4", (4,))])


def read_ref_features(path: str, with_rev: bool = False):
    """features.bin written by oracle/ref_driver.cpp -> (feat[REF_FEATURE_DTYPE], desc[n,128]);
    with_rev: also the descriptor -> feature reverse map that --match runs append ("PSR1")."""
    with open(path, "rb") as f:
        data = f.read()
    assert data[:4] == b"PSF1"
    nf, nd = struct.unpack_from("<ii", data, 4)
    feat = np.frombuffer(data, dtype=REF_FEATURE_DTYPE, count=nf, offset=12).copy()
    off = 12 + nf * REF_FEATURE_DTYPE.itemsize
    desc = np.frombuffer(data, dtype="<f4", count=nd * 128, offset=off).reshape(nd, 128).copy()
    if not with_rev:
        return feat, desc
    off += nd * 512
    assert data[off:off + 4] == b"PSR1"
    rev = np.frombuffer(data, dtype="<i4", count=nd, offset=off + 4).copy()
    return feat, desc, rev


def run_key(w: int, h: int, seed: int, args) -> str:
    """key of a reference run on make_frame(w, h, seed) with these ref_dump arguments in tests/golden/ref_runs.json"""
    return "%dx%d_s%d %s" % (w, h, seed, " ".join(args))


def flatten(feat, desc):
    """-> array [n_desc, 4] of (x, y, sigma, theta) and the matching descriptors, one row per
    (feature, orientation)."""
    rows, idx = [], []
    for f in feat:
        for k in range(int(f["num_ori"])):
            rows.append((f["x"], f["y"], f["sigma"], f["ori"][k]))
            idx.append(int(f["desc_idx"][k]))
    kp = np.array(rows, dtype=np.float64).reshape(-1, 4)
    return kp, desc[np.array(idx, dtype=np.int64)] if len(idx) else desc[:0]
