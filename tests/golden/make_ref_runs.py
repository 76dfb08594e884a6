"""Fixtures of the reference runs the GPU tests compare with: runs the UNMODIFIED reference (oracle/_ref/ref_dump, which
`make -C oracle ref` builds from the reference's sources) on a B200 on the tests' seeded frames and keeps what the tests
compare, small enough to commit.

    python tests/golden/make_ref_runs.py [OUT_DIR]        # default OUT_DIR: tests/golden

Fixtures:
  ref_runs.json       per run, keyed by oracle_lib.run_key(w, h, seed, args): feature / descriptor counts; the sha256 of the keypoint
                      set (compare.keypoint_digest: keypoints and orientations bit for bit); the sha256 and shape of the
                      Gaussian planes of octaves 0..2 from --log runs; and the repeatability / matching scores of the
                      affine set computed from the reference's full outputs
  ref_runs_desc.npz   per run with a descriptor sample: <key>|keys [k, 5] (octave, x, y, sigma, theta) and <key>|desc
                      [k, 128], drawn by compare.descriptor_sample (seed 0)
  feat_<name>.npz     the full features (feat, in ref_dump's record layout) and descriptors (desc) of the FULL_F256 runs
"""
import glob
import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [os.path.dirname(HERE), ROOT]
import compare  # noqa: E402
import oracle_lib as ol  # noqa: E402
from popsift_b200.synth import affine_set, make_frame, write_pgm  # noqa: E402

REF = os.path.join(ROOT, "oracle", "_ref", "ref_dump")
SAMPLE = 8          # descriptors kept per run (1 per frame of the benchmark workload)


# (w, h, seed, ref_dump arguments, descriptors sampled) of every run on a make_frame() frame
RUNS = [
    # tests/test_gpu_parity.py::test_live_against_reference_library
    (1920, 1080, 101, ["--mode", "vlfeat", "--norm", "classic"], SAMPLE),
    (1920, 1080, 102, ["--mode", "popsift", "--norm", "rootsift"], SAMPLE),
    (800, 600, 21, ["--mode", "vlfeat", "--norm", "classic", "--downsampling", "0"], SAMPLE),
    (3840, 2160, 7, ["--mode", "vlfeat", "--norm", "classic", "--octaves", "5"], SAMPLE),
    (800, 600, 22, ["--mode", "vlfeat", "--norm", "classic", "--gauss-mode", "opencv"], SAMPLE),
    (640, 480, 23, ["--mode", "popsift", "--norm", "rootsift", "--gauss-mode", "opencv", "--sigma", "1.2", "--levels", "4"], SAMPLE),
    (700, 500, 24, ["--mode", "vlfeat", "--norm", "classic", "--downsampling", "-0.5"], SAMPLE),
    (640, 480, 25, ["--mode", "popsift", "--norm", "rootsift", "--downsampling", "0.5"], SAMPLE),
    (641, 479, 26, ["--mode", "vlfeat", "--norm", "classic", "--downsampling", "1"], SAMPLE),
    # test_descriptor_modes_vs_reference
] + [(640, 480, 1, ["--desc-mode", dm], SAMPLE) for dm in ("iloop", "grid", "igrid", "notile")] + [
    # test_level0_planes_bit_exact_vs_live_reference
    (700, 500, 24, ["--log", "--octaves", "2", "--downsampling", "-0.5"], 0),
    (640, 480, 27, ["--log", "--octaves", "2", "--downsampling", "-1.5"], 0),
    (641, 479, 26, ["--log", "--octaves", "2", "--downsampling", "1"], 0),
    (5000, 96, 28, ["--log", "--octaves", "2"], 0),
    (4096, 64, 29, ["--log", "--octaves", "2"], 0),
    (1000, 700, 30, ["--log", "--octaves", "2", "--downsampling", "0"], 0),
    # test_direct_scaling_vs_oracle_and_live_reference, test_gauss_mode_*_vs_oracle_and_live_reference (the features of the
    # first two are committed in full: feat_f640_direct.npz, feat_f640_vlfeat_direct.npz)
    (640, 480, 31, ["--log", "--mode", "vlfeat", "--norm", "classic", "--direct-scaling"], 0),
    (640, 480, 33, ["--log", "--mode", "vlfeat", "--norm", "classic", "--gauss-mode", "vlfeat-direct"], 0),
    (640, 480, 35, ["--log", "--mode", "vlfeat", "--norm", "classic", "--gauss-mode", "relative"], SAMPLE),
    (640, 480, 37, ["--log", "--mode", "vlfeat", "--norm", "classic", "--gauss-mode", "fixed9"], SAMPLE),
    (640, 480, 37, ["--log", "--mode", "vlfeat", "--norm", "classic", "--gauss-mode", "fixed15"], SAMPLE),
    # test_direct_scaling_with_every_gauss_mode
] + [(512, 384, 39, ["--log", "--mode", "vlfeat", "--norm", "classic", "--gauss-mode", g, "--direct-scaling"], 0)
     for g in ("relative", "fixed9", "fixed15", "vlfeat-direct")] + [
    # tests/test_config_settings.py: threshold (OpenCV mode floors the peak threshold: 0.02 -> 0, 0.05 -> 2), edge limit,
    # initial blur (above the level-0 sigma at 1.0 with the default up-scale; 0 = no assumed blur), normalization multiplier
    (640, 480, 3, ["--mode", "vlfeat", "--norm", "classic", "--threshold", "0"], SAMPLE),
    (640, 480, 3, ["--mode", "opencv", "--norm", "classic", "--threshold", "0.02"], SAMPLE),
    (640, 480, 3, ["--mode", "opencv", "--threshold", "0.05"], SAMPLE),
    (640, 480, 3, ["--mode", "popsift", "--threshold", "0.5"], SAMPLE),
] + [(640, 480, 3, ["--mode", "vlfeat", "--norm", "classic", "--edge-limit", x], SAMPLE) for x in ("0", "2.5", "50")] + [
    (640, 480, 5, ["--log", "--initial-blur", "0"], SAMPLE),
    (640, 480, 5, ["--log", "--initial-blur", "1.0"], SAMPLE),
    (640, 480, 5, ["--log", "--initial-blur", "0.3", "--downsampling", "0"], SAMPLE),
    (640, 480, 5, ["--log", "--initial-blur", "1.0", "--direct-scaling", "--mode", "vlfeat", "--norm", "classic"], SAMPLE),
    (640, 480, 5, ["--log", "--initial-blur", "1.0", "--gauss-mode", "vlfeat-direct", "--mode", "vlfeat", "--norm", "classic"], SAMPLE),
    (640, 480, 5, ["--log", "--initial-blur", "0", "--gauss-mode", "relative", "--mode", "vlfeat", "--norm", "classic"], SAMPLE),
    (640, 480, 1, ["--norm-multi", "9"], SAMPLE),
    (640, 480, 1, ["--norm", "classic", "--norm-multi", "9"], SAMPLE),
    (640, 480, 1, ["--norm-multi", "-3"], SAMPLE),
    (640, 480, 1, ["--desc-mode", "grid", "--norm-multi", "9"], SAMPLE),
]

# (name, ref_dump arguments) of the runs on make_frame(256, 192, 3) whose features and descriptors are kept in full as
# feat_<name>.npz (tests/test_oracle_golden.py::test_features_vs_reference)
FULL_F256 = [
    ("f256_threshold0", ["--mode", "vlfeat", "--norm", "classic", "--threshold", "0"]),
    ("f256_opencv_threshold002", ["--mode", "opencv", "--norm", "classic", "--threshold", "0.02"]),
    ("f256_edge_limit2_5", ["--mode", "vlfeat", "--norm", "classic", "--edge-limit", "2.5"]),
    ("f256_initial_blur1", ["--initial-blur", "1.0"]),
    ("f256_norm_multi9", ["--norm-multi", "9"]),
]


def record(out_bin, k, logdir=None):
    feat, desc = ol.read_ref_features(out_bin)
    rec = {"counts": [len(feat), len(desc)]}
    sample = None
    if k:
        rec["digest"] = compare.keypoint_digest(feat)
        sample = compare.descriptor_sample(feat, desc, feat["desc_idx"], k)
    if logdir:
        planes = {}
        for fn in sorted(glob.glob(os.path.join(logdir, "dir-octave-dump", "pyramid-o-*-l-*.dump"))):
            b = os.path.basename(fn)
            oc, l = int(b.split("-o-")[1].split("-")[0]), int(b.split("-l-")[1].split(".")[0])
            if oc < 3:
                p = ol.read_ref_dump(fn)
                planes["g_%d_%d" % (oc, l)] = {"shape": list(p.shape), "sha256": hashlib.sha256(p.tobytes()).hexdigest()}
        rec["planes"] = planes
    return rec, sample, (feat, desc)


def main(out_dir):
    assert os.path.exists(REF), "build the reference first: make -C oracle ref"
    os.makedirs(out_dir, exist_ok=True)
    runs, samples = {}, {}

    def keep(key, rec, sample):
        runs[key] = rec
        if sample is not None:
            samples[key + "|keys"], samples[key + "|desc"] = sample
        print(key, rec["counts"], flush=True)

    with tempfile.TemporaryDirectory() as td:
        for n, (w, h, seed, args, k) in enumerate(RUNS):
            wd = os.path.join(td, "r%d" % n)
            os.makedirs(wd)
            write_pgm(os.path.join(wd, "f.pgm"), make_frame(w, h, seed))
            subprocess.run([REF, "-i", "f.pgm", "-o", "f.bin"] + args, cwd=wd, check=True, capture_output=True)
            rec, sample, _ = record(os.path.join(wd, "f.bin"), k, wd if "--log" in args else None)
            keep(ol.run_key(w, h, seed, args), rec, sample)
        write_pgm(os.path.join(td, "f256.pgm"), make_frame(256, 192, 3))
        for name, args in FULL_F256:
            out = os.path.join(td, name + ".bin")
            subprocess.run([REF, "-i", os.path.join(td, "f256.pgm"), "-o", out] + args, check=True, capture_output=True)
            feat, desc = ol.read_ref_features(out)
            np.savez_compressed(os.path.join(out_dir, "feat_%s.npz" % name), feat=feat, desc=desc.astype(np.float32))
            print(name, [len(feat), len(desc)], flush=True)
        # test_affine_set_per_keypoint_diff_and_repeatability: the six images of the affine set, VLFeat mode
        aset, full = affine_set(), []
        for i, (im, _) in enumerate(aset, 1):
            pgm, out = os.path.join(td, "a%d.pgm" % i), os.path.join(td, "a%d.bin" % i)
            write_pgm(pgm, im)
            args = ["--mode", "vlfeat", "--norm", "classic"]
            subprocess.run([REF, "-i", pgm, "-o", out] + args, check=True, capture_output=True)
            rec, sample, (feat, desc) = record(out, SAMPLE)
            keep("affine%d %s" % (i, " ".join(args)), rec, sample)
            full.append(ol.flatten(feat, desc))
        runs["affine_scores"] = [compare.affine_scores(*full[0], *full[k], aset[k][1]) for k in range(1, 6)]
        # test_benchmark_workload_matches_reference_exactly: the 32 frames bench.py times, default Config, octaves 5, levels 3
        import bench
        args = ["--octaves", "5", "--levels", "3"]
        cmd = [REF, "-o", os.path.join(td, "bench")] + args
        for i, f in enumerate(bench.synth_frames(32, 0)):
            write_pgm(os.path.join(td, "b%d.pgm" % i), f)
            cmd += ["-i", os.path.join(td, "b%d.pgm" % i)]
        subprocess.run(cmd, check=True, capture_output=True)
        for i in range(32):
            rec, sample, _ = record(os.path.join(td, "bench.%d" % i), 1)
            keep("bench%d %s" % (i, " ".join(args)), rec, sample)
    with open(os.path.join(out_dir, "ref_runs.json"), "w") as fh:       # one run per line
        fh.write("{\n%s\n}\n" % ",\n".join("%s: %s" % (json.dumps(k), json.dumps(runs[k], sort_keys=True)) for k in sorted(runs)))
    np.savez_compressed(os.path.join(out_dir, "ref_runs_desc.npz"), **samples)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else HERE)
