"""GPU tests of the state a slot carries from one frame to the next, and of device-resident input (ps_submit_dev_u8).

A slot keeps its captured CUDA graph (keyed on width, height and image type), the geometry it last ran directly, buffers
regrown after an overflow, and planes, candidate lists and an 8-bit image buffer that are zeroed once at ps_create and
afterwards hold whatever the previous frames left there.  Every frame below must give exactly the bits of the library's
plain run of the same frame (slot_state.fresh: a new context of the frame's size, one slot, ps_submit_u8), and where the
reference's own run of the frame is pinned (tests/golden/ref_runs.json), the reference's result."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import compare
import slot_state as ss
from popsift_b200 import api
from slot_state import DevImage, differences, fresh, frame, snapshot, submit, u8_pitch
from test_gpu_parity import assert_planes_same_as_reference, assert_same_as_reference, mk_cfg, ref_run

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def assert_same(got, want, what):
    bad = differences(got, want)
    assert not bad, (what, bad[:12])


# ---- 1. device input equals host input --------------------------------------------------------------------------------

@pytest.mark.parametrize("w,h,seed", [(641, 479, 5), (97, 61, 13), (33, 17, 15), (1919, 1079, 16), (5000, 96, 28)])
def test_device_input_equals_host_input(w, h, seed):
    """ps_submit_dev_u8 from buffers whose row pitch is w, w + 1, the slot's own pitch + 29 and 2w, with the first row
    0, 1 or 3 bytes into the buffer and the padding filled with 0xFF or random bytes: every Gaussian and DoG plane, the
    extrema, the features and the descriptors are those of ps_submit_u8 in a fresh context, bit for bit.  (641 and 97
    are not multiples of 4: the slot's own rows are padded.)"""
    name = "%dx%d_s%d" % (w, h, seed)
    img = frame(name)
    want = fresh("default", name)
    ps = api.PopSift(ss.config("default"), max_width=w, max_height=h, slots=1)
    try:
        k = 0
        for pitch in (w, w + 1, u8_pitch(w) + 29, 2 * w):
            for offset in (0, 1, 3):
                dev = DevImage(ps._lib, img, pitch, offset, pad=0xFF if k % 2 else None, seed=k)
                try:
                    submit(ps, 0, dev=dev)
                    got, _ = snapshot(ps, 0)
                finally:
                    dev.free()
                assert_same(got, want, ("pitch", pitch, "offset", offset))
                k += 1
    finally:
        ps.uninit()


def _reference_cfg(extra):
    c = mk_cfg("vlfeat", "classic") if "--mode" in extra else mk_cfg()
    if "--octaves" in extra:
        c.setOctaves(int(extra[extra.index("--octaves") + 1]))
    if "--downsampling" in extra:
        c.setDownsampling(float(extra[extra.index("--downsampling") + 1]))
    if "--gauss-mode" in extra:
        c.setGaussMode(extra[extra.index("--gauss-mode") + 1])
    if "--direct-scaling" in extra:
        c.setScalingMode(0)
    return c


@pytest.mark.parametrize("w,h,seed,extra,octaves", [
    (641, 479, 26, "--octaves 2 --downsampling 1", 2),                                  # launch_level0_u8, halved odd extent
    (5000, 96, 28, "--octaves 2", 2),                                                   # launch_level0_u8, wider than 4096
    (640, 480, 35, "--mode vlfeat --norm classic --gauss-mode relative", 3),            # launch_level0_rows_u8
    (640, 480, 37, "--mode vlfeat --norm classic --gauss-mode fixed9", 3),              # launch_fixed_level0_u8
    (640, 480, 37, "--mode vlfeat --norm classic --gauss-mode fixed15", 3),
    (640, 480, 33, "--mode vlfeat --norm classic --gauss-mode vlfeat-direct", 2),       # launch_level0_abs_u8
    (640, 480, 31, "--mode vlfeat --norm classic --direct-scaling", 3),                 # launch_level0_u8, every octave
])
def test_device_input_reproduces_reference_runs(w, h, seed, extra, octaves):
    """Every level-0 kernel that reads the slot's 8-bit image, fed through ps_submit_dev_u8 from a buffer with a pitch
    of the slot's own pitch + 29, the first row 3 bytes in and random padding: the Gaussian planes the reference dumped
    under --log (sha256), its feature and descriptor counts, and where pinned its keypoints and sampled descriptors."""
    args = extra.split()
    key = "%dx%d_s%d %s" % (w, h, seed, " ".join(["--log"] + args))
    ps = api.PopSift(_reference_cfg(args), max_width=w, max_height=h, slots=1)
    dev = DevImage(ps._lib, frame("%dx%d_s%d" % (w, h, seed)), u8_pitch(w) + 29, 3, pad=None, seed=seed)
    try:
        submit(ps, 0, dev=dev)
        feats = api.SiftJob(ps, 0).get()
        assert_planes_same_as_reference(ps, key, octaves)
        assert [feats.getFeatureCount(), feats.getDescriptorCount()] == ref_run(key)["counts"], key
        if "digest" in ref_run(key):
            assert_same_as_reference(feats, key)
    finally:
        dev.free()
        ps.uninit()


# ---- 2. the benchmark's timed loop ------------------------------------------------------------------------------------

def test_benchmark_loop_device_input_matches_reference(tmp_path):
    """bench.run_ours' step_dev restated: 4 slots round robin over the 32 frames of bench.synth_frames(32, 0) in device
    memory, ps_submit_dev_u8 -> ps_counts -> ps_download, each frame's results into a region of its own in one
    page-locked block.  Two passes take every slot through direct launches, capture and replay; in the second every
    frame is the reference's (keypoints bit for bit, counts, sampled descriptors) and its Feature::desc pointers land in
    its own region.  bench.dump_outputs then writes what the reference's per-frame digests can be rebuilt from."""
    import torch
    import bench
    L = api.load_library()
    torch.cuda.set_device(0)
    cfg = ss.config("bench")
    frames = bench.synth_frames(bench.FRAMES_PER_STEP, 0)
    keys = ["bench%d --octaves 5 --levels 3" % i for i in range(len(frames))]
    ref = [ref_run(k) for k in keys]
    slots = 4
    ctx = L.ps_create(0, C.byref(cfg._c), bench.W, bench.H, slots)
    assert ctx, L.ps_last_error(None).decode()
    dev_frames = [torch.from_numpy(f).cuda() for f in frames]
    torch.cuda.synchronize()
    n_feat, n_desc = (sum(r["counts"][j] for r in ref) for j in (0, 1))
    scratch = api._PinnedBlock(L, n_feat, n_desc)
    keep = api._PinnedBlock(L, n_feat + 1024, n_desc + 1024)
    nf, nd = C.c_int32(), C.c_int32()

    def chk(rc):
        assert rc == 0, (rc, L.ps_last_error(ctx).decode())

    def step(regions):
        tot_f = tot_d = 0
        inflight = []

        def fetch(s0):
            nonlocal tot_f, tot_d
            chk(L.ps_counts(ctx, s0, C.byref(nf), C.byref(nd)))
            if regions is None:
                chk(L.ps_download(ctx, s0, scratch.pf, scratch.pd))
            else:
                assert tot_f + nf.value <= keep.n_feat and tot_d + nd.value <= keep.n_desc
                chk(L.ps_download(ctx, s0, keep.pf + 72 * tot_f, keep.pd + 512 * tot_d))
                regions.append((tot_f, nf.value, tot_d, nd.value))
            tot_f += nf.value
            tot_d += nd.value

        for i, df in enumerate(dev_frames):
            s = i % slots
            if len(inflight) == slots:
                fetch(inflight.pop(0))
            chk(L.ps_submit_dev_u8(ctx, s, df.data_ptr(), bench.W, bench.W, bench.H))
            inflight.append(s)
        for s0 in inflight:
            fetch(s0)
        return [tot_f, tot_d]

    regions = []
    try:
        assert step(None) == [n_feat, n_desc]
        assert step(regions) == [n_feat, n_desc] == [453753, 522542]
    finally:
        L.ps_destroy(ctx)
        scratch.free()
    del dev_frames
    try:
        per_frame = []
        for i, (f0, n, d0, m) in enumerate(regions):
            feat, desc = keep.feat[f0:f0 + n], keep.desc[d0:d0 + m]
            base = keep.pd + 512 * d0
            used = np.arange(4)[None, :] < feat["num_ori"][:, None]
            ptr = feat["desc_ptr"].astype(np.int64)
            assert (ptr[~used] == 0).all(), i
            off = ptr[used] - base
            assert ((off >= 0) & (off < 512 * m) & (off % 512 == 0)).all(), ("Feature::desc outside the frame's region", i)
            assert_same_as_reference(api.Features(feat, desc), keys[i])
            per_frame.append((feat, desc, base))

        bench.dump_outputs(str(tmp_path), per_frame)
        counts = np.load(str(tmp_path / "counts.npy"))
        table = np.load(str(tmp_path / "features.npy"))
        dumped = np.load(str(tmp_path / "descriptors.npy"))
        rows = np.load(str(tmp_path / "descriptor_rows.npy")).astype(np.int64)
        assert counts.tolist() == [r["counts"] for r in ref]
        assert len(table) == n_feat and len(dumped) == len(rows) > 0
        for i in range(len(frames)):
            t = table[table[:, 0] == i]
            f = np.zeros(len(t), api.FEATURE_DTYPE)
            f["octave"], f["x"], f["y"], f["sigma"], f["num_ori"] = t[:, 1], t[:, 2], t[:, 3], t[:, 4], t[:, 5]
            f["ori"] = t[:, 6:]
            assert compare.keypoint_digest(f) == ref[i]["digest"], ("features.npy", i)
        # every sampled row of descriptors.npy is the in-memory descriptor that descriptor_rows.npy names
        where = {}
        for i, (feat, desc, _) in enumerate(per_frame):
            ft = api.Features(feat, desc)
            n = feat["num_ori"]
            t = np.zeros((len(feat), 10), np.float32)
            t[:, 0] = i
            t[:, 1:6] = np.stack([feat["octave"], feat["x"], feat["y"], feat["sigma"], n], 1)
            t[:, 6:] = np.where(np.arange(4)[None, :] < n[:, None], feat["ori"], np.float32(0))
            for j in range(len(t)):
                where[t[j].tobytes()] = (i, j, ft.desc_idx[j])
        for s, (r, k) in enumerate(rows):
            i, j, didx = where[table[r].tobytes()]
            assert 0 <= k < table[r, 5], (s, r, k)
            want = per_frame[i][1][didx[k]]
            assert np.array_equal(dumped[s].view(np.uint32), want.view(np.uint32)), ("descriptors.npy row", s, "frame", i)
    finally:
        keep.free()


# ---- 3. mixed geometries in one context -------------------------------------------------------------------------------

_mixed = {}


def mixed(device_input):
    if device_input not in _mixed:
        _mixed[device_input] = ss.run_mixed(device_input)
    return _mixed[device_input]


@pytest.mark.parametrize("device_input", [False, True], ids=["host", "device"])
def test_mixed_geometries_in_one_context(device_input):
    """One 1920x1080 VLFeat / classic context with 3 slots runs ss.MIXED: large -> small -> large, two widths of one
    height, graphs replayed after other geometries ran in the slot.  Every frame equals its fresh-context run bit for
    bit (planes of octaves 0-1, extrema, features, descriptors), and the frames the reference ran are the reference's."""
    out = mixed(device_input)
    for i, (name, (got, feats)) in enumerate(zip(ss.MIXED, out)):
        assert_same(got, fresh("vlfeat", name, ss.MIXED_OCTAVES), (i, name, "slot %d" % (i % ss.MIXED_SLOTS)))
        if name in ss.MIXED_REFERENCE:
            assert_same_as_reference(feats, ss.MIXED_REFERENCE[name])
    assert len({d["counts"][0] for d, _ in out}) > 3       # the sequence really mixes different frames


def test_u8_and_float_images_alternating_in_one_slot():
    """u8 and float images of one size alternate in one slot: the graph key includes the image type.  The sequence
    replays a u8 graph after a float frame ran directly, captures a float graph over it, and so on; every frame equals
    the fresh u8 or float run."""
    name = "640x480_s1"
    seq = ["u8", "u8", "u8", "f32", "u8", "f32", "f32", "u8", "f32", "f32"]
    want = {"u8": fresh("vlfeat", name, 2), "f32": fresh("vlfeat", "f32:" + name, 2)}
    assert want["u8"]["features"] != want["f32"]["features"]
    ps = api.PopSift(ss.config("vlfeat"), max_width=640, max_height=480, slots=1)
    try:
        for i, kind in enumerate(seq):
            submit(ps, 0, frame(name if kind == "u8" else "f32:" + name))
            assert_same(snapshot(ps, 0, 2)[0], want[kind], (i, kind))
    finally:
        ps.uninit()


# ---- 4. graph replay and direct launches ------------------------------------------------------------------------------

def test_mixed_sequence_without_graphs_gives_the_same_bits():
    """POPSIFT_B200_GRAPH=0 (read once per process, hence a child process) issues every launch directly: the mixed
    sequence gives the same digests frame by frame as the in-process run with graph capture and replay."""
    env = dict(os.environ, POPSIFT_B200_GRAPH="0")
    out = subprocess.run([sys.executable, os.path.join(HERE, "slot_state.py"), "mixed"], env=env, capture_output=True,
                         text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    direct = json.loads(out.stdout.strip().splitlines()[-1])
    graphed = [d for d, _ in mixed(False)]
    assert len(direct) == len(graphed) == len(ss.MIXED)
    for i, (a, b) in enumerate(zip(direct, graphed)):
        assert_same(a, b, (i, ss.MIXED[i]))


# ---- 5. regrow inside a replayed graph --------------------------------------------------------------------------------

@pytest.mark.parametrize("device_input", [False, True], ids=["host", "device"])
def test_regrow_after_a_replayed_graph_overflows(device_input, monkeypatch):
    """Extremum and descriptor buffers of 64 records (POPSIFT_B200_INIT_CAP, read by ps_create).  A constant frame runs
    directly, is captured and replayed without overflow; a textured frame of the same size then replays that graph,
    overflows, and ps_counts grows the buffers and re-runs the tail; the next textured frame is captured again with the
    new buffers and the one after replays it; a constant frame replays the new graph.  ps_counts returns 0 every time
    and every result is the fresh-context run's (made with the default capacities)."""
    flat, tex = "flat640x480", "640x480_s1"
    want = {n: fresh("vlfeat", n, 2) for n in (flat, tex)}
    assert want[flat]["counts"] == [0, 0] and want[tex]["counts"][0] > 64
    monkeypatch.setenv("POPSIFT_B200_INIT_CAP", "64")
    ps = api.PopSift(ss.config("vlfeat"), max_width=640, max_height=480, slots=1)
    devs = {}
    try:
        if device_input:
            devs = {n: DevImage(ps._lib, frame(n), 700, 1, pad=None, seed=k) for k, n in enumerate((flat, tex))}
        for i, n in enumerate([flat, flat, flat, tex, tex, tex, flat]):
            submit(ps, 0, frame(n), devs.get(n))
            assert_same(snapshot(ps, 0, 2)[0], want[n], (i, n))
    finally:
        for d in devs.values():
            d.free()
        ps.uninit()


# ---- 6. ps_wait_input covers device input -----------------------------------------------------------------------------

def test_wait_input_covers_device_input():
    """The slot's stream is held up by a ~0.1 s sleep kernel; frame X is submitted from a device buffer, ps_wait_input
    returns, and the buffer is overwritten with frame Y.  ps_wait_input must not return before the slot has copied X,
    so the result is X's."""
    import torch
    torch.cuda.set_device(0)
    w, h = 640, 480
    x, y = "640x480_s51", "640x480_s52"
    want = {n: fresh("vlfeat", n, 1) for n in (x, y)}
    assert want[x]["features"] != want[y]["features"]
    ps = api.PopSift(ss.config("vlfeat"), max_width=w, max_height=h, slots=1)
    L = ps._lib
    dev = DevImage(L, frame(x), u8_pitch(w) + 29, 1)
    try:
        for _ in range(2):                    # first frame direct, second captured: X below replays the graph
            submit(ps, 0, frame(y))
            snapshot(ps, 0, 0)
        st = torch.cuda.ExternalStream(L.ps_slot_stream(ps._ctx, 0))
        with torch.cuda.stream(st):
            torch.cuda._sleep(200_000_000)    # about 0.1 s at the B200's clocks
        submit(ps, 0, dev=dev)
        assert L.ps_wait_input(ps._ctx, 0) == 0
        dev.write(frame(y))
        got = snapshot(ps, 0, 1)[0]
        assert differences(got, want[y]), \
            "the result equals frame Y's: ps_wait_input returned before the slot had copied the device image"
        assert_same(got, want[x], "frame X")
    finally:
        dev.free()
        ps.uninit()


# ---- 7. argument checks on the device path ----------------------------------------------------------------------------

def test_device_input_argument_checks():
    """pitch < w and a null pointer are argument errors, an image wider than the context is PS_ERR_TOO_LARGE; none of
    them disturbs the slot: the next valid submit (direct, captured, replayed) gives the fresh-context result."""
    w, h = 320, 240
    name = "320x240_s61"
    want = fresh("vlfeat", name, 1)
    ps = api.PopSift(ss.config("vlfeat"), max_width=w, max_height=h, slots=1)
    L = ps._lib
    dev = DevImage(L, frame(name), 2 * w, 0)
    try:
        refusals = [((dev.ptr, w - 1, w, h), ss.PS_ERR_ARG, "pitch"),
                    ((None, w, w, h), ss.PS_ERR_ARG, "bad argument"),
                    ((dev.ptr, 2 * w, w + 1, h), ss.PS_ERR_TOO_LARGE, "exceeds")]
        for args, code, text in refusals:
            assert L.ps_submit_dev_u8(ps._ctx, 0, *args) == code, (args, L.ps_last_error(ps._ctx).decode())
            assert text in L.ps_last_error(ps._ctx).decode(), args
            submit(ps, 0, dev=dev)
            assert_same(snapshot(ps, 0, 1)[0], want, args)
    finally:
        dev.free()
        ps.uninit()
