"""Helpers for tests/test_slot_state_and_device_input.py: device-resident input frames, a bit-exact digest of everything
a slot computed for one frame, the library's own fresh-context run of a frame, and the mixed-geometry frame sequence.

    python tests/slot_state.py mixed      # JSON digests of the mixed sequence (host input), one per frame

The command line exists so that the sequence can run in a process of its own, under the library's process-wide
switches (POPSIFT_B200_GRAPH=0)."""
from __future__ import annotations

import ctypes as C
import functools
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for _p in (HERE, ROOT):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import compare  # noqa: E402
from popsift_b200 import api  # noqa: E402
from popsift_b200.synth import affine_set, make_frame  # noqa: E402

PS_ERR_ARG, PS_ERR_TOO_LARGE = -1, -3


def u8_pitch(w):
    """row pitch of the slot's own 8-bit image buffer: rows start 4-byte aligned"""
    return (w + 3) & ~3


class DevImage:
    """An 8-bit frame in a ps_dev_alloc buffer: row r starts at byte `offset + r * pitch` of the buffer.  Every other
    byte of the buffer (the pitch padding, the bytes before the first row and after the last) holds `pad`: one byte
    value, or random bytes for pad=None.  A copy that reads any of them changes the result."""

    def __init__(self, lib, img, pitch=None, offset=0, pad=0xFF, seed=0):
        self.lib = lib
        self.h, self.w = img.shape
        self.pitch = self.w if pitch is None else pitch
        self.offset = offset
        self.size = offset + self.pitch * self.h + 64
        self.base = lib.ps_dev_alloc(self.size)
        assert self.base, "ps_dev_alloc failed"
        self.write(img, pad, seed)

    @property
    def ptr(self):
        return self.base + self.offset

    def write(self, img, pad=0xFF, seed=0):
        """the whole buffer, synchronously (ps_host_to_dev)"""
        if pad is None:
            buf = np.random.default_rng(seed).integers(0, 256, self.size, dtype=np.uint8)
        else:
            buf = np.full(self.size, pad, np.uint8)
        buf[self.offset:self.offset + self.pitch * self.h].reshape(self.h, self.pitch)[:, :self.w] = img
        assert self.lib.ps_host_to_dev(self.base, buf.ctypes.data, self.size) == 0

    def free(self):
        if self.base:
            self.lib.ps_dev_free(self.base)
            self.base = None


def submit(ps, slot, img=None, dev=None):
    """one frame into `slot` of the api.PopSift `ps` through the C ABI: ps_submit_dev_u8 from `dev`, else ps_submit_f32
    or ps_submit_u8 by the dtype of `img`"""
    L = ps._lib
    if dev is not None:
        rc = L.ps_submit_dev_u8(ps._ctx, slot, dev.ptr, dev.pitch, dev.w, dev.h)
    else:
        img = np.ascontiguousarray(img)
        h, w = img.shape
        fn = L.ps_submit_f32 if img.dtype == np.float32 else L.ps_submit_u8
        rc = fn(ps._ctx, slot, img.ctypes.data, w, h)
    ps._check(rc)


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _bits(a):
    """float32 bits with -0.0 folded into 0.0"""
    return (np.asarray(a, np.float32) + np.float32(0)).view(np.uint32)


def feature_digest(feats):
    """(sha256 of the sorted feature table, sha256 of the descriptors in that order): features and descriptors bit for
    bit, independent of the order the library emitted them in"""
    t, order = compare._feature_table(feats.feat)
    nk = feats.feat["num_ori"][order].astype(np.int64)
    f_in = np.repeat(order, nk)
    k = np.arange(nk.sum()) - np.repeat(np.cumsum(nk) - nk, nk)
    desc = feats.desc[feats.desc_idx[f_in, k]] if len(f_in) else feats.desc[:0]
    return _sha(t[order]), _sha(desc)


def extrema_digest(ext):
    """sha256 of the sorted extremum records without idx_ori (the position of the first descriptor, which depends on
    the order the extrema were found in) and with the orientation slots beyond num_ori zeroed"""
    t = np.zeros((len(ext), 10), np.uint32)
    for j, name in enumerate(("x", "y", "sigma")):
        t[:, j] = _bits(ext[name])
    for j, name in enumerate(("lpos", "octave", "num_ori"), 3):
        t[:, j] = ext[name].astype(np.int32).view(np.uint32)
    t[:, 6:] = _bits(np.where(np.arange(4)[None, :] < ext["num_ori"][:, None], ext["ori"], 0))
    return _sha(t[np.lexsort(t.T[::-1])])


def snapshot(ps, slot, octaves=None):
    """everything `slot` computed for its last frame -> (digest dict, Features).  The digest holds the counts and the
    sha256 of every Gaussian and DoG plane of the first `octaves` octaves (all for None), of the extrema and of the
    features and descriptors; two frames computed the same bits iff their digests are equal.  Collecting the result
    goes through ps_counts, which must return 0."""
    feats = api.SiftJob(ps, slot).get()
    levels = max(2, ps._config.levels)
    geo = ps.slot_geometry(slot)
    planes = {}
    for oc in range(len(geo) if octaves is None else min(octaves, len(geo))):
        for lv in range(levels + 3):
            planes["g%d_%d" % (oc, lv)] = _sha(ps.plane(slot, oc, lv))
        for lv in range(levels + 2):
            planes["d%d_%d" % (oc, lv)] = _sha(ps.plane(slot, oc, lv, dog=True))
    fd, dd = feature_digest(feats)
    d = {"counts": [feats.getFeatureCount(), feats.getDescriptorCount()], "geometry": [list(g) for g in geo],
         "planes": planes, "extrema": extrema_digest(ps.extrema(slot)), "features": fd, "descriptors": dd}
    return d, feats


def differences(got, want):
    """names of the digest entries that differ (planes one by one)"""
    out = [k for k in got if k != "planes" and got[k] != want.get(k)]
    gp, wp = got["planes"], want["planes"]
    out += ["plane " + k for k in sorted(set(gp) | set(wp)) if gp.get(k) != wp.get(k)]
    return out


# ---- configurations and frames, by name (so that fresh-context results can be cached) ----------------------------

def config(name):
    """"default" (popsift::Config defaults), "vlfeat" (VLFeat mode, classic norm), "bench" (bench.py's octaves=5,
    levels=3)"""
    c = api.Config()
    if name == "vlfeat":
        c.setMode("vlfeat")
        c.setNormMode("classic")
    elif name == "bench":
        c.setOctaves(5)
        c.setLevels(3)
    else:
        assert name == "default", name
    return c


@functools.lru_cache(None)
def _affine_images():
    return [im for im, _ in affine_set()]


@functools.lru_cache(None)
def frame(name):
    """"WxH_sSEED": make_frame(W, H, SEED); "affineK": image K of the affine set; "flatWxH": constant 128;
    "f32:NAME": frame NAME / 256 as float32 (popsift-demo --float-mode)"""
    if name.startswith("f32:"):
        return frame(name[4:]).astype(np.float32) / np.float32(256.0)
    if name.startswith("affine"):
        return _affine_images()[int(name[6:]) - 1]
    if name.startswith("flat"):
        w, h = map(int, name[4:].split("x"))
        return np.full((h, w), 128, np.uint8)
    size, seed = name.split("_s")
    w, h = map(int, size.split("x"))
    return make_frame(w, h, int(seed))


@functools.lru_cache(None)
def fresh(cfg_name, frame_name, octaves=None):
    """digest of the library's plain run of a frame: a new context of exactly the frame's size, one slot, one
    ps_submit_u8 (ps_submit_f32 for float frames).  The reference result for anything that reuses slot state."""
    img = frame(frame_name)
    h, w = img.shape
    ps = api.PopSift(config(cfg_name), max_width=w, max_height=h, slots=1)
    try:
        submit(ps, 0, img)
        return snapshot(ps, 0, octaves)[0]
    finally:
        ps.uninit()


# ---- one context, many geometries -------------------------------------------------------------------------------------

MIXED_SLOTS = 3
MIXED_MAX = (1920, 1080)
# Frame i goes to slot i % 3.  Slot 0 runs 1920x1080 directly, captures it, replays it, then takes 97x61 and comes back
# to 1920x1080, which replays the graph captured three frames earlier.  Slot 1 has a 1920x1080 graph when 1919x1080
# arrives: same height, other width.  Slot 2 captures 800x640 on the second affine image and replays it on the first
# after 641x479.
MIXED = ["1920x1080_s101", "1920x1080_s101", "affine1",
         "1920x1080_s101", "1920x1080_s101", "affine2",
         "1920x1080_s101", "1919x1080_s103", "641x479_s5",
         "97x61_s13", "32x32_s14", "affine1",
         "1920x1080_s101", "1919x1080_s103", "641x479_s5",
         "1920x1080_s101"]
MIXED_OCTAVES = 2
MIXED_REFERENCE = {"1920x1080_s101": "1920x1080_s101 --mode vlfeat --norm classic",
                   "affine1": "affine1 --mode vlfeat --norm classic", "affine2": "affine2 --mode vlfeat --norm classic"}


def run_mixed(device_input=False):
    """the MIXED sequence through one VLFeat / classic context of 1920x1080 with 3 slots, MIXED_SLOTS frames in flight;
    from device buffers (pitch u8_pitch(w) + 29, first row 1 byte into the buffer, random padding) when device_input.
    Returns [(digest, Features)] in frame order."""
    ps = api.PopSift(config("vlfeat"), max_width=MIXED_MAX[0], max_height=MIXED_MAX[1], slots=MIXED_SLOTS)
    devs = {}
    try:
        if device_input:
            for k, name in enumerate(sorted(set(MIXED))):
                img = frame(name)
                devs[name] = DevImage(ps._lib, img, pitch=u8_pitch(img.shape[1]) + 29, offset=1, pad=None, seed=k)
        out = [None] * len(MIXED)
        pending = {}
        for i, name in enumerate(MIXED):
            s = i % MIXED_SLOTS
            if s in pending:
                out[pending.pop(s)] = snapshot(ps, s, MIXED_OCTAVES)
            submit(ps, s, frame(name), devs.get(name))
            pending[s] = i
        for s, i in sorted(pending.items(), key=lambda kv: kv[1]):
            out[i] = snapshot(ps, s, MIXED_OCTAVES)
        return out
    finally:
        for d in devs.values():
            d.free()
        ps.uninit()


if __name__ == "__main__":
    if sys.argv[1:] != ["mixed"]:
        raise SystemExit("usage: python tests/slot_state.py mixed")
    print(json.dumps([d for d, _ in run_mixed()]))
