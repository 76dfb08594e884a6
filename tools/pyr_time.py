"""Times the pyramid stage and each octave-0 launch at 4K (CUDA events, L2 flushed) -- roofline helper."""
import ctypes as C, os, sys, statistics
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from popsift_b200 import api
from popsift_b200.synth import make_frame
W, H = (int(sys.argv[1]), int(sys.argv[2])) if len(sys.argv) > 2 else (3840, 2160)
octv = int(sys.argv[3]) if len(sys.argv) > 3 else 5
L = api.load_library()
cfg = api.Config(); cfg.setOctaves(octv)
ctx = L.ps_create(0, C.byref(cfg._c), W, H, 1)
img = torch.from_numpy(make_frame(W, H, 7)).cuda()
nf, nd = C.c_int32(), C.c_int32()
assert L.ps_submit_dev_u8(ctx, 0, img.data_ptr(), W, W, H) == 0
assert L.ps_counts(ctx, 0, C.byref(nf), C.byref(nd)) == 0
st = torch.cuda.ExternalStream(L.ps_slot_stream(ctx, 0))
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
geo = cfg.geometry(W, H)
def timeit(fn, n=10, warm=3):
    ts = []
    for it in range(warm + n):
        with torch.cuda.stream(st):
            flush.fill_(it & 255)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st); fn(); b.record(st); b.synchronize()
        if it >= warm: ts.append(a.elapsed_time(b))
    return statistics.median(ts)
t = timeit(lambda: L.ps_run_pyramid_only(ctx, 0))
sumwh = sum(w * h for w, h in geo)
print("env TILE=%s" % os.environ.get("POPSIFT_B200_TILE_KERNELS"))
print("pyramid stage: %.3f ms  -> %.0f GB/s algorithmic (68 B/px, %d px)" % (t, 68 * sumwh / t / 1e6, sumwh))
for o in range(min(2, len(geo))):
    for l in range(0 if o == 0 else 1, 6):
        tl = timeit(lambda: L.ps_run_level_only(ctx, 0, o, l), n=6, warm=2)
        px = geo[o][0] * geo[o][1]
        b = (8.25 if l == 0 else 12) * px
        print("  octave %d level %d: %.3f ms  %.0f GB/s" % (o, l, tl, b / tl / 1e6))
L.ps_destroy(ctx)
