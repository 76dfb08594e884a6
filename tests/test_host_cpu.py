"""CPU-only checks of the product's host side: the C-ABI library loads, exports every symbol
include/popsift_b200.h declares, and its GPU-free host logic (tables, geometry, Config) agrees with
the oracle.  No compute call needs a GPU here."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import oracle_lib as ol
from popsift_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "popsift_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(ps_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    L = api.load_library()
    for name in sorted(declared):
        assert hasattr(L, name), "libpopsift_b200.so does not export %s" % name
    assert declared == set(api.EXPORTS)
    assert L.ps_abi_version() == 3


def test_struct_sizes_match_reference_layouts():
    # popsift::Feature is 72 bytes, Descriptor 512 (SURVEY appendix C)
    assert api.FEATURE_DTYPE.itemsize == 72
    assert api.EXTREMUM_DTYPE.itemsize == 44
    assert C.sizeof(api.PsConfig) == 18 * 4      # ABI 2: + scaling mode and the three grid-filter fields


CFGS = [dict(), dict(downsampling=0), dict(levels=4), dict(sigma=1.2, levels=5), dict(initial_blur=0.0),
        dict(downsampling=-2), dict(levels=2, sigma=2.0), dict(gauss_relative=1), dict(gauss_relative=1, levels=4, sigma=1.3),
        dict(gauss_fixed=4), dict(gauss_fixed=7)]


def _mk(kw):
    c = api.Config()
    o = dict(kw)
    if "downsampling" in o:
        c.setDownsampling(o["downsampling"])
    if "levels" in o:
        c.setLevels(o["levels"])
    if "sigma" in o:
        c.setSigma(o["sigma"])
    if "initial_blur" in o:
        c.setInitialBlur(o["initial_blur"])
    if o.get("gauss_relative"):
        c.setGaussMode("relative")
    if o.get("gauss_fixed"):
        c.setGaussMode("fixed9" if o["gauss_fixed"] == 4 else "fixed15")
    oc = ol.make_config(**{k: v for k, v in kw.items() if k != "initial_blur"})
    if "initial_blur" in kw:
        oc.initial_blur = kw["initial_blur"]
        oc.has_initial_blur = 0 if kw["initial_blur"] == 0 else 1
    return c, oc


@pytest.mark.parametrize("kw", CFGS)
def test_gauss_tables_bit_identical_to_oracle(kw):
    c, oc = _mk(kw)
    t = c.gauss_tables()
    ot = ol.OrcTables()
    assert ol.lib().orc_compute_tables(C.byref(oc), C.byref(ot)) == 0
    assert list(t.inc_span) == list(ot.inc.span)
    assert np.array_equal(np.frombuffer(t.inc_filter, np.uint32), np.frombuffer(ot.inc.filter, np.uint32))
    assert np.array_equal(np.frombuffer(t.inc_sigma, np.uint32), np.frombuffer(ot.inc.sigma, np.uint32))
    assert np.array_equal(np.frombuffer(t.dd_filter0, np.uint32), np.frombuffer(ot.dd_filter0, np.uint32))
    assert t.dd_span0 == ot.dd_span0
    # the direct-downscaling rows of every octave (Config::ScaleDirect); row 0 is the classic one
    assert list(t.dd_span) == list(ot.dd_span) and t.dd_span[0] == t.dd_span0
    assert np.array_equal(np.frombuffer(t.dd_filter, np.uint32), np.frombuffer(ot.dd_filter, np.uint32))
    assert np.array_equal(np.frombuffer(t.dd_filter, np.uint32)[:32], np.frombuffer(t.dd_filter0, np.uint32))
    # levels >= 1 from level 0 of the same octave (--gauss-mode fixed9 / fixed15)
    assert list(t.absn_span) == list(ot.abs_oN.span)
    assert np.array_equal(np.frombuffer(t.absn_filter, np.uint32), np.frombuffer(ot.abs_oN.filter, np.uint32))
    # the rows transformed for interpolated fetches (--gauss-mode relative)
    assert list(t.inc_ispan) == list(ot.inc_ispan)
    assert np.array_equal(np.frombuffer(t.inc_ifilter, np.uint32), np.frombuffer(ot.inc_ifilter, np.uint32))
    # the absolute rows of octave 0 (--gauss-mode vlfeat-direct)
    assert list(t.abs_span) == list(ot.abs_o0.span)
    assert np.array_equal(np.frombuffer(t.abs_filter, np.uint32), np.frombuffer(ot.abs_o0.filter, np.uint32))
    assert t.peak_threshold == ot.peak_threshold and t.sigma_k == ot.sigma_k


def test_default_tables_have_the_surveyed_spans():
    t = api.Config().gauss_tables()
    # SURVEY 8: taps 11,11,15,17,21,27 -> spans 6,6,8,9,11,14
    assert list(t.inc_span)[:6] == [6, 6, 8, 9, 11, 14]
    assert abs(t.peak_threshold - 1.7) < 1e-6


@pytest.mark.parametrize("w,h,kw,expect", [
    (640, 480, {}, [(1280, 960), (640, 480), (320, 240), (160, 120), (80, 60), (40, 30), (20, 15)]),
    (1920, 1080, {}, [(3840, 2160), (1920, 1080), (960, 540), (480, 270), (240, 135), (120, 68), (60, 34), (30, 17), (15, 9)]),
    (3840, 2160, {"downsampling": 0, "octaves": 5}, [(3840, 2160), (1920, 1080), (960, 540), (480, 270), (240, 135)]),
    (641, 479, {}, None),
    (17, 33, {}, None),
])
def test_geometry_matches_oracle_and_survey(w, h, kw, expect):
    c = api.Config()
    if "downsampling" in kw:
        c.setDownsampling(kw["downsampling"])
    if "octaves" in kw:
        c.setOctaves(kw["octaves"])
    g = c.geometry(w, h)
    oc = ol.make_config(**kw)
    W = (C.c_int32 * 20)()
    H = (C.c_int32 * 20)()
    n = ol.lib().orc_geometry(C.byref(oc), w, h, W, H)
    assert g == [(W[i], H[i]) for i in range(n)]
    if expect:
        assert g == expect


def test_config_mirrors_reference_semantics():
    a, b = api.Config(), api.Config()
    assert a == b
    b.setDescMode("grid")          # not part of equal() (reference sift_conf.cu:286-304)
    assert a == b
    b.setNormMode("classic")
    assert not (a == b)
    with pytest.raises(api.PopSiftError):
        a.setGaussMode("nonsense")
    with pytest.raises(api.PopSiftError):
        a.setNormMode("L2")
    a.setInitialBlur(0.0)
    assert not a.hasInitialBlur()
    assert abs(api.Config().getPeakThreshold() - 1.7) < 1e-6
    c = api.Config(); c.setSigma(2.5)
    with pytest.raises(api.PopSiftError):
        c.gauss_tables()           # reference gauss_filter.cu:131-137 rejects sigma > 2


def test_no_cpu_fallback_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(api.PopSiftError) as ei:
        api.PopSift(api.Config(), max_width=64, max_height=64)
    assert "no CUDA device" in str(ei.value) or "CUDA" in str(ei.value)


def test_fast_unorm16_division_is_exact_for_every_r16():
    """k_pyramid_march.cu::unorm16_to_float: q = x*c; q += c*fma(-q, 65535, x) with c = RN(1/65535) equals the
    correctly rounded x/65535 (what the texture unit returns) for all 65536 inputs."""
    from fractions import Fraction

    def rn32(fr):
        f = np.float32(float(fr))
        cands = [f, np.nextafter(f, np.float32(np.inf)), np.nextafter(f, np.float32(-np.inf))]
        return min(cands, key=lambda c: (abs(Fraction(float(c)) - fr), int(c.view(np.uint32)) & 1))

    def fma32(a, b, c):
        return rn32(Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c)))

    c = np.array([0x37800080], dtype=np.uint32).view(np.float32)[0]
    assert c == np.float32(1.0) / np.float32(65535.0)
    for r in list(range(0, 65536, 7)) + [1, 2, 255, 256, 257, 65534, 65535] + [(257 * s + 2) >> 2 for s in range(1021)]:
        x = np.float32(r)
        q = np.float32(x * c)
        q2 = fma32(fma32(-q, np.float32(65535.0), x), c, q)
        assert q2 == rn32(Fraction(r, 65535)), r


def test_march_partition_covers_every_row_once():
    """The pyramid kernels' strip x segment partition (k_partition.h): host sweep over plane sizes."""
    import subprocess
    from popsift_b200 import build as B
    B.build()
    out = subprocess.run([B.PART_CHECK], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    assert out.stdout.startswith("OK"), out.stdout
    # the 4K workload fills all 592 slots of one wave
    assert "B=592" in out.stdout, out.stdout


def test_descriptor_fast_math_bounds():
    """The descriptor kernel (k_desc.cu) replaces atan2f and the float->int conversions by cheaper forms.
    float32 emulation of the same formulas: the atan2 polynomial stays within 1e-6 rad of atan2, and the
    magic-number floor / fixed-point conversions are exact on their whole input range."""
    rng = np.random.default_rng(5)
    f32 = np.float32
    # fast_atan2: a = min/max, degree-6 polynomial in a^2 (coefficients as in k_desc.cu)
    coef = [0.006811764091253281, -0.03360414132475853, 0.07962359488010406, -0.1323333978652954,
            0.19807815551757812, -0.3331736922264099, 0.9999961256980896]
    y = rng.uniform(-255, 255, 200000).astype(f32)
    x = rng.uniform(-255, 255, 200000).astype(f32)
    ax, ay = np.abs(x), np.abs(y)
    mx, mn = np.maximum(ax, ay), np.minimum(ax, ay)
    a = np.where(mx > f32(1e-30), mn / np.where(mx > 0, mx, 1), f32(0)).astype(f32)
    s = (a * a).astype(f32)
    p = np.full_like(a, f32(coef[0]))
    for c in coef[1:]:
        p = (p * s + f32(c)).astype(f32)
    r = (p * a).astype(f32)
    r = np.where(ay > ax, f32(1.57079632679489662) - r, r).astype(f32)
    r = np.where(x < 0, f32(3.14159265358979323846) - r, r).astype(f32)
    r = np.copysign(r, y)
    err = np.abs(r.astype(np.float64) - np.arctan2(y.astype(np.float64), x.astype(np.float64)))
    assert err.max() < 1e-6, err.max()
    # floor_bits: v + 1.5 * 2^23 rounded DOWN keeps floor(v) in the low mantissa bits (two's complement)
    v = np.concatenate([rng.uniform(-40, 40, 100000), np.arange(-16, 17), np.arange(-16, 17) - 1e-4]).astype(f32)
    magic = np.float64(12582912.0)
    summed = np.floor(v.astype(np.float64) + magic)              # exact real sum, then round toward -inf to an integer ulp
    bits = summed.astype(f32).view(np.uint32)
    assert np.array_equal(summed.astype(f32).astype(np.float64), summed)   # representable: ulp is 1 in [2^23, 2^24)
    fl = np.floor(v.astype(np.float64)).astype(np.int64)
    assert np.array_equal((bits & 7).astype(np.int64), fl & 7)
    assert np.array_equal(summed - magic, fl.astype(np.float64))
    # fix_bits: round(w * c) for 0 <= w * c < 2^23 through fma(w, c, 2^23)
    w = rng.uniform(0, 360 * 16384, 100000).astype(f32)
    c = rng.uniform(0, 1, 100000).astype(f32)
    prod = w.astype(np.float64) * c.astype(np.float64)
    fixed = (np.rint(prod + 8388608.0).astype(f32).view(np.uint32) & 0x7FFFFF).astype(np.float64)
    assert np.array_equal(fixed, np.rint(prod))
    assert (360.0 * 16384) < 2 ** 23


def _ref_pgm_gray(kind, maxval, samples, w, h):
    """What the reference reader returns (reference src/application/pgmread.cpp:126-250, as compiled with
    RGB2GRAY_IN_INT): P2/P3 values and 16-bit P5 values are scaled by 255.0/maxval (truncating), 8-bit P5
    bytes are taken as they are, colour becomes (4899 r + 9617 g + 1868 b) >> 14 truncated to 8 bits, and
    P6 samples enter the weights unscaled (8- or 16-bit)."""
    s = np.asarray(samples, np.int64)
    def scale(v):
        return v if maxval == 255 else (v * 255.0 / maxval).astype(np.int64)
    if kind == 2:
        return scale(s).astype(np.uint8)
    if kind == 5:
        return s.astype(np.uint8) if maxval < 256 else (s * 255.0 / maxval).astype(np.int64).astype(np.uint8)
    rgb = (scale(s) & 0xff if kind == 3 else s).reshape(-1, 3)
    return ((4899 * rgb[:, 0] + 9617 * rgb[:, 1] + 1868 * rgb[:, 2]) >> 14).astype(np.uint8)


@pytest.mark.parametrize("kind,maxval", [(2, 255), (2, 1023), (3, 255), (3, 15), (5, 255), (5, 100), (5, 65535),
                                         (6, 255), (6, 65535)])
def test_netpbm_reader_matches_reference_conversions(tmp_path, kind, maxval):
    """popsift-demo's reader (csrc/app/pgmread.cpp) on generated P2 / P3 / P5 / P6 files, comments included."""
    import subprocess
    from popsift_b200 import build as B
    B.build()
    rng = np.random.default_rng(kind * 1000 + maxval)
    w, h = 7, 5
    ch = 3 if kind in (3, 6) else 1
    samples = rng.integers(0, maxval + 1, w * h * ch)
    path = str(tmp_path / "img.pnm")
    header = ("P%d\n# a comment\n%d %d\n# another\n%d\n" % (kind, w, h, maxval)).encode()
    with open(path, "wb") as f:
        f.write(header)
        if kind in (2, 3):
            f.write((" ".join(str(int(v)) for v in samples) + "\n").encode())
        elif maxval < 256:
            f.write(samples.astype(np.uint8).tobytes())
        else:
            f.write(samples.astype("<u2").tobytes())      # the reference reads 16-bit samples in host order
    out = subprocess.run([B.PGM_CHECK, path], capture_output=True, text=True, timeout=60)
    assert out.returncode == 0, out.stdout + out.stderr
    lines = out.stdout.split("\n")
    assert lines[0].split() == [str(w), str(h)]
    got = np.frombuffer(bytes.fromhex(lines[1]), np.uint8)
    want = _ref_pgm_gray(kind, maxval, samples, w, h)
    assert np.array_equal(got, want), (got, want)


def test_match_oracle_on_constructed_descriptors():
    """tests/match_oracle.py (restatement of the reference matcher, groundwork for SURVEY 8f rank 2): right
    descriptors built from the left ones with known perturbations give known best / second / accept."""
    import match_oracle as mo
    rng = np.random.default_rng(3)
    left = rng.uniform(0, 1, (6, 128)).astype(np.float32)
    left /= np.linalg.norm(left, axis=1, keepdims=True)
    right = np.zeros((8, 128), np.float32)
    perm = [3, 0, 5, 1, 4, 2]
    for i, p in enumerate(perm):
        right[i] = left[p] + np.float32(0.01) * rng.standard_normal(128).astype(np.float32)     # near copy of left[p]
    right[6] = left[0] + np.float32(0.011) * rng.standard_normal(128).astype(np.float32)        # a second near copy of left[0]
    right[7] = rng.uniform(0, 1, 128).astype(np.float32)
    m = mo.match(left, right)
    inv = {p: i for i, p in enumerate(perm)}
    for l in range(6):
        assert m[l, 0] == inv[l] or (l == 0 and m[l, 0] in (inv[0], 6))
    assert set(m[0, :2]) == {inv[0], 6} and m[0, 2] == 0          # two equally good candidates: ratio test rejects
    assert all(m[l, 2] == 1 for l in range(1, 6))                 # unique near copies: accepted
    # the matrix-product form agrees on this well-separated set
    assert np.array_equal(mo.match(left, right, exact_order=False)[:, [0, 2]], m[:, [0, 2]])
    assert mo.match(left, right[:0]).tolist() == [[0, 0, 0]] * 6


def test_result_arrays_keep_their_page_locked_block_alive():
    """ADVICE r1: `d = job.get().desc` must stay valid after the Features object is gone.  The arrays' base
    objects hold a lease on the block; it returns to the pool (or is freed after uninit) only when the last
    view dies.  Checked with a stand-in allocator, no GPU needed."""
    import gc

    class FakeLib:
        def __init__(self):
            self.live, self.bufs = set(), {}

        def ps_host_alloc(self, n):
            b = (C.c_uint8 * max(n, 1))()
            a = C.addressof(b)
            self.live.add(a); self.bufs[a] = b
            return a

        def ps_host_free(self, p):
            self.live.discard(p)

    L = FakeLib()
    pool = api._Pool()
    f, d = api._leased_views(pool, api._PinnedBlock(L, 10, 10), 3, 2)
    row = d[1]
    del f, d
    gc.collect()
    assert pool.blocks == [] and len(L.live) == 2          # still leased: a view is alive
    row[:] = 1.0                                           # and writable memory
    del row
    gc.collect()
    assert len(pool.blocks) == 1                           # recycled
    f, d = api._leased_views(pool, pool.blocks.pop(), 1, 1)
    pool.close()                                           # PopSift.uninit() while a result is still referenced
    assert len(L.live) == 2
    del f, d
    gc.collect()
    assert not L.live                                      # freed when the last view died


def test_level0_plan_follows_the_texture_coordinate_model():
    """ps_debug_level0_plan (host arithmetic, the same tex_axis the kernels run) against a numpy restatement of the
    measured coordinate model: the benchmark's 2x geometries keep the byte-tile kernel, other power-of-two ratios share
    fetches, everything else -- non-integer scale factors, odd extents halved, non-power-of-two widths beyond 4096
    at 2x -- fetches per tap."""
    f32 = np.float32

    def tex_axis(c, n):
        c = np.clip(c, f32(-1), f32(2)).astype(np.float32)
        q = np.floor(c * f32(2097152.0)).astype(np.int64)
        I = np.clip(((q * n + 4096) >> 13) - 128, -128, n * 256 - 128)
        i, a = I >> 8, I & 255
        i0, i1 = np.clip(i, 0, n - 1), np.clip(i + 1, 0, n - 1)
        a = np.where(i0 == i1, 0, a)
        return i0, np.where(a == 0, i0, i1), a

    def centre(X, shift, N0):
        return ((X.astype(np.float32) + f32(shift)) / f32(N0)).astype(np.float32)

    def shared(w, W, shift, R):
        X = np.arange(W)
        cx = centre(X, shift, W)
        for off in range(-R, R + 1):
            rel = f32(abs(off)) / f32(W)
            A = tex_axis((cx - rel if off < 0 else cx + rel).astype(np.float32), w)
            B = tex_axis(centre(X + off, shift, W), w)
            if any((a != b).any() for a, b in zip(A, B)):
                return False
        return True

    L = api.load_library()
    expect_fixed = {(3840, 2160, 1.0): 0, (1920, 1080, 1.0): 0, (4096, 2160, 1.0): 0, (640, 480, 0.0): 1, (640, 480, -1.0): 1,
                    (640, 480, 2.0): 1, (640, 480, 0.5): 2, (641, 479, -1.0): 2, (5000, 96, 1.0): 2}
    for (w, h, up), want in expect_fixed.items():
        W, H = int(np.ceil(f32(w) * f32(2.0 ** up))), int(np.ceil(f32(h) * f32(2.0 ** up)))
        shift = float(f32(0.5) * f32(2.0 ** up))
        got = L.ps_debug_level0_plan(w, h, W, H, shift, 4)
        assert got == want, (w, h, up, got, want)
        assert (got != 2) == shared(w, W, shift, 4), (w, h, up)


def test_shipped_sass_uses_tma_and_tcgen05():
    """The claims of DESIGN.md about the hardware paths, checked on the built library itself (cuobjdump, no GPU needed):
    every column-marching level kernel stages its rows with the TMA unit (UTMALDG + mbarrier SYNCS), its column pass is packed
    FFMA2, and the matcher issues tcgen05 MMAs (UTCHMMA) with TMEM loads (LDTM).  Only the variants that run are shipped: one
    orientation kernel, one tensor-core matcher, one candidate extrema kernel per SIFT mode, and level kernels without
    programmatic-dependent-launch instructions (ACQBULK / PREEXIT)."""
    import shutil
    import sys as _sys
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    lib = os.path.join(ROOT, "popsift_b200", "lib", "libpopsift_b200.so")
    if not os.path.exists(lib):
        pytest.skip("library not built")
    _sys.path.insert(0, os.path.join(ROOT, "tools"))
    import sass_hist
    k = sass_hist.histogram(lib)
    level = {n: c for n, c in k.items() if "march_level_kernel" in n}
    assert len(level) >= 50
    for n, c in level.items():
        assert c["UTMALDG"] > 0 and c["SYNCS"] > 0 and c["FFMA2"] > 0, n
        assert c["LDGSTS"] == 0, n                       # no cp.async staging left in the level kernels
        assert c["ACQBULK"] == 0 and c["PREEXIT"] == 0, n
    tc = {n: c for n, c in k.items() if "match_tc_kernel" in n}
    assert len(tc) == 1 and all(c["UTCHMMA"] > 0 and c["LDTM"] > 0 and c["UTMALDG"] > 0 for c in tc.values())
    assert sum("orientation_kernel" in n for n in k) == 1
    assert sum("cand_extrema_kernel" in n for n in k) == 3


def test_runtime_switches_are_the_documented_ones():
    """The POPSIFT_B200_* environment variables the library reads (getenv under popsift_b200/csrc) are exactly the ones
    INTEGRATION.md section 5 lists, apart from the two that Python code reads: POPSIFT_B200_LIB (api.py) and
    POPSIFT_BENCH_SLOTS (bench.py)."""
    read = set()
    for dp, _, fs in os.walk(os.path.join(ROOT, "popsift_b200", "csrc")):
        for f in fs:
            with open(os.path.join(dp, f), errors="replace") as fh:
                read |= set(re.findall(r'getenv\("(POPSIFT_B200_\w+)"\)', fh.read()))
    with open(os.path.join(ROOT, "INTEGRATION.md")) as fh:
        sec = fh.read().split("\n## 5.")[1].split("\n## ")[0]
    listed = set()
    for ln in sec.splitlines():
        if ln.startswith("| `"):
            listed |= set(re.findall(r"`(POPSIFT_\w+?)[=`]", ln.split(" | ")[0]))
    python_side = {"POPSIFT_B200_LIB": "popsift_b200/api.py", "POPSIFT_BENCH_SLOTS": "bench.py"}
    for name, path in python_side.items():
        with open(os.path.join(ROOT, path)) as fh:
            assert name in fh.read(), (name, path)
    assert read, "no getenv calls found"
    assert listed - set(python_side) == read, (sorted(listed - set(python_side) - read), sorted(read - listed))


def test_print_gauss_tables_text():
    """Config::setPrintGaussTables() / --print-gauss-tables: the reference's printout (header of init_filter and
    print_gauss_filter_symbol(10), gauss_filter.cu:24-121,146-161) rebuilt from this library's tables -- same sections, same
    row format `level taps sigma: values`, values to 8 decimals, rows longer than 10 columns end with `...`."""
    c = api.Config()
    txt = c.gauss_tables_text()
    assert txt.startswith("\nUpscaling factor: 1.000000 (i.e. original image is scaled by a factor of 2.000000)\n")
    assert "    Initial sigma is 1.600000\n    Input blurriness is assumed to be 0.500000 (scaled to 1.000000)\n" in txt
    for head in ("Gauss tables\n      level span sigma : center value -> edge value\n    relative sigma\n",
                 "Gauss tables for hardware interpolation\n", "      absolute filters octave 0 (compute level 0, all other levels directly from level 0)\n",
                 "      absolute filters other octaves\n", "    level 0-filters for direct downscaling\n"):
        assert head in txt, head
    t = c.gauss_tables()
    # first incremental row: "      0 11 1.248999: 0.32525530 ..." (span 6 -> 11 taps, 6 values)
    row0 = [ln for ln in txt.splitlines() if ln.startswith("      0 %d " % (2 * t.inc_span[0] - 1))][0]
    vals = row0.split(": ")[1].split()
    assert len(vals) == t.inc_span[0] and vals[0] == "%0.8f" % t.inc_filter[0] and row0.split()[2] == "%2.6f:" % t.inc_sigma[0]
    # level 5 has 14 taps a side: only 10 printed
    row5 = [ln for ln in txt.splitlines() if ln.startswith("      5 %d " % (2 * t.inc_span[5] - 1))][0]
    assert row5.endswith("...") and len(row5.split(": ")[1].split()) == 11
    assert txt.count("\n") > 6 * 4 + 20       # four tables of levels + 3 rows and the 20 rows of the dd table
