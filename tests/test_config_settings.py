"""The detection settings a user can change -- Config::setThreshold, setEdgeLimit, setInitialBlur,
setNormalizationMultiplier and the per-octave extremum cap (ps_config.max_extrema) -- at values where they change the
result: threshold 0 (very many extrema), OpenCV mode whose floored peak threshold is 0 (every DoG sample passes the
pre-test) or 2, threshold 0.5 (nothing found), edge limit 0 ((0 + 1)^2 / 0 = inf, nothing rejected), an initial blur above
the level-0 sigma (the |sigma0^2 - blur^2| branch), descriptors scaled by 2^m, and a cap that bites.

Each run is compared with the CPU oracle on the same frame (planes and extrema bit for bit, counts, descriptors) and with the
reference's run of the same settings (tests/golden/ref_runs.json, made by tests/golden/make_ref_runs.py).

Run as a script (python tests/test_config_settings.py W H SEED [ref_dump arguments]) it prints the feature count, the
descriptor count and compare.keypoint_digest of make_frame(W, H, SEED) under those settings."""
import functools
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import compare
import oracle_lib as ol
from popsift_b200 import api
from popsift_b200.synth import make_frame

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
G = os.path.join(HERE, "golden")
F1_MIN, L2_MAX = 0.99, 1e-3

VL = ["--mode", "vlfeat", "--norm", "classic"]
# (w, h, seed, ref_dump arguments): the reference runs of tests/golden/make_ref_runs.py for these settings
RUNS = [
    (640, 480, 3, VL + ["--threshold", "0"]),
    (640, 480, 3, ["--mode", "opencv", "--norm", "classic", "--threshold", "0.02"]),     # floor(0.02 * 127.5 / 3) = 0
    (640, 480, 3, ["--mode", "opencv", "--threshold", "0.05"]),                          # floor(2.125) = 2
    (640, 480, 3, ["--mode", "popsift", "--threshold", "0.5"]),                          # nothing passes
] + [(640, 480, 3, VL + ["--edge-limit", x]) for x in ("0", "2.5", "50")] + [
    (640, 480, 5, ["--log", "--initial-blur", "0"]),
    (640, 480, 5, ["--log", "--initial-blur", "1.0"]),                                   # 1.0 * 2 > sigma 1.6
    (640, 480, 5, ["--log", "--initial-blur", "0.3", "--downsampling", "0"]),
    (640, 480, 5, ["--log", "--initial-blur", "1.0", "--direct-scaling"] + VL),
    (640, 480, 5, ["--log", "--initial-blur", "1.0", "--gauss-mode", "vlfeat-direct"] + VL),
    (640, 480, 5, ["--log", "--initial-blur", "0", "--gauss-mode", "relative"] + VL),
    (640, 480, 1, ["--norm-multi", "9"]),
    (640, 480, 1, ["--norm", "classic", "--norm-multi", "9"]),
    (640, 480, 1, ["--norm-multi", "-3"]),
    (640, 480, 1, ["--desc-mode", "grid", "--norm-multi", "9"]),
]


def settings(args):
    """ref_dump arguments -> (this library's Config, the oracle's make_config keywords, the normalization multiplier)"""
    c, okw, m = api.Config(), {}, 0
    it = iter(args)
    for a in it:
        if a == "--log":
            continue
        if a == "--direct-scaling":
            c.setScalingMode(0)                      # Config::ScaleDirect
            okw["scaling_mode"] = 1
            continue
        v = next(it)
        if a == "--mode":
            c.setMode(v); okw["mode"] = v
        elif a == "--norm":
            c.setNormMode("RootSift" if v == "rootsift" else "classic"); okw["norm"] = v
        elif a == "--threshold":
            c.setThreshold(float(v)); okw["threshold"] = float(v)
        elif a == "--edge-limit":
            c.setEdgeLimit(float(v)); okw["edge_limit"] = float(v)
        elif a == "--initial-blur":
            c.setInitialBlur(float(v)); okw["initial_blur"] = float(v)
        elif a == "--downsampling":
            c.setDownsampling(float(v)); okw["downsampling"] = float(v)
        elif a == "--gauss-mode":
            c.setGaussMode(v); okw[{"vlfeat-direct": "gauss_direct", "relative": "gauss_relative"}[v]] = 1
        elif a == "--norm-multi":
            m = int(v); c.setNormalizationMultiplier(m); okw["norm_multi"] = m
        elif a == "--desc-mode":
            c.setDescMode(v)                         # the oracle computes the default (loop) descriptors only
        else:
            raise AssertionError(a)
    return c, okw, m


def run_gpu(img, cfg):
    h, w = img.shape
    ps = api.PopSift(cfg, max_width=w, max_height=h, slots=1)
    return ps, ps.enqueue(w, h, img).get()


@functools.lru_cache(None)
def _ref_runs():
    with open(os.path.join(G, "ref_runs.json")) as fh:
        return json.load(fh), np.load(os.path.join(G, "ref_runs_desc.npz"))


def assert_same_as_reference(ps, feats, key, l2_max):
    """the reference's run `key`: identical counts, keypoints and orientations bit for bit, each sampled descriptor within
    l2_max, and for --log runs the Gaussian planes of octaves 0..2 with the reference's shapes and sha256"""
    rec, z = _ref_runs()[0][key], _ref_runs()[1]
    assert [feats.getFeatureCount(), feats.getDescriptorCount()] == rec["counts"], (key, rec["counts"])
    assert compare.keypoint_digest(feats.feat) == rec["digest"], key
    l2 = compare.sampled_descriptor_l2(feats.feat, feats.desc, feats.desc_idx, z[key + "|keys"], z[key + "|desc"])
    assert (l2 < l2_max).all(), (key, l2.max(initial=0))
    bad = []
    for name, p in rec.get("planes", {}).items():
        _, oc, l = name.split("_")
        g = ps.plane(0, int(oc), int(l))
        if list(g.shape) != p["shape"] or hashlib.sha256(g.tobytes()).hexdigest() != p["sha256"]:
            bad.append(name)
    assert not bad, (key, bad)


def extrema_set(ps):
    return sorted((int(e["octave"]), float(e["x"]), float(e["y"]), int(e["lpos"])) for e in ps.extrema(0))


def oracle_extrema_set(o):
    return sorted((int(e[4]), float(e[0]), float(e[1]), int(e[3])) for e in o.extrema())


@pytest.mark.parametrize("w,h,seed,args", RUNS)
def test_setting_vs_oracle_and_reference(w, h, seed, args):
    """planes (every octave for the initial-blur runs, octaves 0 and 2 otherwise) and extrema bit-exact against the
    oracle, the same counts and descriptors; the same keypoints, sampled descriptors and plane hashes as the reference.
    Descriptor tolerances scale with the 2^m the descriptors are scaled by."""
    img = make_frame(w, h, seed)
    cfg, okw, m = settings(args)
    ps, feats = run_gpu(img, cfg)
    o = ol.Oracle(ol.make_config(**okw), w, h)
    o.run(img)
    L = 3
    octaves = range(o.num_octaves) if "--initial-blur" in args else (0, 2)
    bad = []
    for oc in octaves:
        bad += [("g", oc, l) for l in range(L + 3) if not np.array_equal(ps.plane(0, oc, l), o.gauss(oc, l))]
        bad += [("d", oc, l) for l in range(L + 2) if not np.array_equal(ps.plane(0, oc, l, dog=True), o.dog(oc, l))]
    assert not bad, bad
    assert extrema_set(ps) == oracle_extrema_set(o)
    of, od = o.features()
    assert (feats.getFeatureCount(), feats.getDescriptorCount()) == (len(of), len(od))
    if len(od):
        r = compare.report(*feats.keypoints(), *ol.flatten(of, od))
        assert r["f1"] >= F1_MIN, r
        if "--desc-mode" not in args:
            assert r["desc_l2_max"] < L2_MAX * 2.0 ** m, r
    o.close()
    assert_same_as_reference(ps, feats, ol.run_key(w, h, seed, args), L2_MAX * 2.0 ** m)
    ps.uninit()


def test_settings_reach_their_edge_cases():
    """the runs above really are at the edges they are meant for (counts of the reference's runs)"""
    runs = _ref_runs()[0]
    n = lambda *args: runs[ol.run_key(640, 480, 3, list(args))]["counts"][0]
    assert n(*VL, "--threshold", "0") > 1000
    assert n("--mode", "opencv", "--norm", "classic", "--threshold", "0.02") > 1000
    assert n("--mode", "popsift", "--threshold", "0.5") == 0
    assert n(*VL, "--edge-limit", "0") >= n(*VL, "--edge-limit", "50") > n(*VL, "--edge-limit", "2.5") > 0


def sorted_output(feats):
    """(feature table in sorted order, descriptors in the matching (feature, orientation) order)"""
    t, order = compare._feature_table(feats.feat)
    idx = [int(feats.desc_idx[i, j]) for i in order for j in range(int(feats.feat["num_ori"][i]))]
    return t[order], feats.desc[idx]


@pytest.mark.parametrize("dm", ["loop", "iloop", "grid", "igrid", "notile"])
def test_norm_multiplier_is_an_exact_power_of_two_scale(dm):
    """scalbnf is exact: with setNormalizationMultiplier(m) every descriptor of every mode equals the m = 0 descriptor
    times 2^m bit for bit (RootSift and classic), and the keypoints do not change"""
    img = make_frame(640, 480, 1)
    for norm in ("RootSift", "classic"):
        out = {}
        for m in (0, 9, -3):
            cfg = api.Config()
            cfg.setDescMode(dm)
            cfg.setNormMode(norm)
            cfg.setNormalizationMultiplier(m)
            ps, feats = run_gpu(img, cfg)
            out[m] = sorted_output(feats)
            ps.uninit()
        t0, d0 = out[0]
        assert len(d0) > 100
        for m in (9, -3):
            t, d = out[m]
            assert np.array_equal(t, t0), (dm, norm, m)
            assert np.array_equal(d, d0 * np.float32(2.0 ** m)), (dm, norm, m, float(np.abs(d - d0 * np.float32(2.0 ** m)).max()))


def _descriptor_keys(fd):
    """one key per device descriptor: (feature table row, orientation slot), from the reverse map"""
    feat, _, rev = fd.to_host()
    t, _ = compare._feature_table(feat)
    base = fd.getDescriptors()
    keys = []
    for d, f in enumerate(rev):
        q = [k for k in range(int(feat["num_ori"][f])) if (int(feat["desc_ptr"][f, k]) - base) // 512 == d]
        assert len(q) == 1, (d, f)
        keys.append(tuple(t[f].tolist()) + (q[0],))
    return keys


def test_matcher_on_scaled_descriptors():
    """squared distances scale by exactly 2^(2m): FeaturesDev::match in MatchingMode with norm_multi 9 gives the same
    (best, second, accept) as with norm_multi 0, in keypoint terms (the two runs may emit extrema in another order)"""
    w, h = 640, 480
    ims = [make_frame(w, h, 1), make_frame(w, h, 2)]
    rows = {}
    for m in (0, 9):
        cfg = api.Config()
        cfg.setNormalizationMultiplier(m)
        pm = api.PopSift(cfg, mode=api.Config.MatchingMode, max_width=w, max_height=h, slots=2)
        fds = [pm.enqueue(w, h, im).getDev() for im in ims]
        kl, kr = _descriptor_keys(fds[0]), _descriptor_keys(fds[1])
        for flags in (api.FeaturesDev.MATCH_EXACT, api.FeaturesDev.MATCH_TENSOR):
            mm = fds[0].match(fds[1], flags)
            rows[m, flags] = sorted((kl[i], kr[b], kr[s], int(a)) for i, (b, s, a) in enumerate(mm.tolist()))
        del fds
        pm.uninit()
    for flags in (api.FeaturesDev.MATCH_EXACT, api.FeaturesDev.MATCH_TENSOR):
        assert rows[9, flags] == rows[0, flags], flags
        assert sum(r[3] for r in rows[0, flags]) > 10
    assert rows[0, api.FeaturesDev.MATCH_EXACT] == rows[0, api.FeaturesDev.MATCH_TENSOR]


def _frame_in_subprocess(env_extra, w, h, seed, args):
    env = dict(os.environ, **env_extra)
    env["PYTHONPATH"] = os.pathsep.join([ROOT, HERE] + [p for p in env.get("PYTHONPATH", "").split(os.pathsep) if p])
    out = subprocess.run([sys.executable, os.path.abspath(__file__), str(w), str(h), str(seed)] + args,
                         env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    nf, nd, digest = out.stdout.split()[-3:]
    return int(nf), int(nd), digest


@pytest.mark.parametrize("args", [VL + ["--threshold", "0"], ["--mode", "opencv", "--norm", "classic", "--threshold", "0.02"]])
def test_candidate_path_equals_dense_scan_at_low_threshold(args):
    """At a peak threshold of 0 (OpenCV mode floors 0.02 * 127.5 / 3 to 0) the pyramid kernels report nearly every DoG sample
    as a candidate: the candidate-driven extrema stage must still find exactly the dense scan's keypoints
    (POPSIFT_B200_DENSE_SCAN is read once per process, so the dense scan runs in a child process)."""
    w, h, seed = 640, 480, 3
    ps, feats = run_gpu(make_frame(w, h, seed), settings(args)[0])
    here = (feats.getFeatureCount(), feats.getDescriptorCount(), compare.keypoint_digest(feats.feat))
    ps.uninit()
    assert here[0] > 200
    assert _frame_in_subprocess({"POPSIFT_B200_DENSE_SCAN": "1"}, w, h, seed, args) == here


def test_extremum_cap_keeps_a_subset_and_regrows_the_slot():
    """ps_config.max_extrema = 200 on a frame whose uncapped oracle finds [480, 1073, 541, 73, 17] extrema per octave at
    threshold 0: per-octave feature counts are min(count, 200), every kept extremum is one of the uncapped oracle's (octave,
    x, y, lpos) bit for bit, and every kept feature and descriptor is the oracle's.  The slot's buffers start at 2 x 200
    records and 690 are needed, so this also grows them (regrow_slot) with a small cap; no PopSiftError."""
    w, h, cap = 640, 480, 200
    img = make_frame(w, h, 3)
    cfg = api.Config()
    cfg.setThreshold(0.0)
    cfg._c.max_extrema = cap
    ps, feats = run_gpu(img, cfg)
    o = ol.Oracle(ol.make_config(threshold=0.0), w, h)
    o.run(img)
    full = o.extrema()
    per_oct = np.bincount(full[:, 4].astype(int))
    assert per_oct.tolist() == [480, 1073, 541, 73, 17]
    want = np.minimum(per_oct, cap)
    assert np.bincount(feats.feat["octave"], minlength=len(want)).tolist() == want.tolist()
    kept = extrema_set(ps)
    assert len(kept) == want.sum() == 690
    assert set(kept) <= set(oracle_extrema_set(o))
    r = compare.report(*feats.keypoints(), *ol.flatten(*o.features()))
    assert r["precision"] == 1.0 and r["desc_l2_max"] < L2_MAX, r
    o.close()
    ps.uninit()


def test_initial_blur_zero_means_no_assumed_blur():
    """setInitialBlur(0) clears hasInitialBlur (reference sift_conf.cu:246-255): level 0 is blurred by the full sigma, the
    oracle's has_initial_blur = 0 planes, not the default's"""
    w, h = 256, 192
    img = make_frame(w, h, 3)
    cfg = api.Config()
    assert cfg.hasInitialBlur()
    cfg.setInitialBlur(0.0)
    assert not cfg.hasInitialBlur() and cfg.getInitialBlur() == 0.0
    ps, _ = run_gpu(img, cfg)
    o = ol.Oracle(ol.make_config(has_initial_blur=0), w, h)
    o.run(img, 1)
    for oc in range(o.num_octaves):
        for l in range(6):
            assert np.array_equal(ps.plane(0, oc, l), o.gauss(oc, l)), (oc, l)
    ps0, _ = run_gpu(img, api.Config())
    assert not np.array_equal(ps0.plane(0, 0, 0), ps.plane(0, 0, 0))
    ps0.uninit(); ps.uninit(); o.close()


if __name__ == "__main__":
    w, h, seed = (int(v) for v in sys.argv[1:4])
    ps, feats = run_gpu(make_frame(w, h, seed), settings(sys.argv[4:])[0])
    print(feats.getFeatureCount(), feats.getDescriptorCount(), compare.keypoint_digest(feats.feat))
    ps.uninit()
