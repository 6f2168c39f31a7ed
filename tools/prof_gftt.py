"""Profiling helper: one 24 MP goodFeaturesToTrack call (config-2 parameters) after a warm-up call.

    python tools/prof_gftt.py [maxCorners] [--ksize G ...]

With --ksize, times the call for each Sobel aperture G (cv2's gradientSize: -1 = Scharr, 1, 3, 5, 7) with CUDA events after
warm-up and prints the card name and power limit beside the times: on the u8 frame, then on the same frame as float32
(I / 255, the float path's front end)."""
import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from iceberg_tracking_code_b200 import cv, synthetic as syn

args = sys.argv[1:]
ksizes = []
if "--ksize" in args:
    i = args.index("--ksize")
    ksizes = [int(v) for v in args[i + 1:]]
    args = args[:i]
H, W = 4000, 6000
base = syn.base_texture(H, W, 7, device="cuda")
g = syn.frame_gray(base, 0)
del base
maxc = int(args[0]) if args else 20000

if ksizes:
    import subprocess
    try:
        card = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        print("card:", card.strip().splitlines()[torch.cuda.current_device()])
    except Exception as e:                                  # noqa: BLE001
        print("card:", torch.cuda.get_device_name(), "(power limit unreadable: %s)" % e)
    gf = g.float() / 255.0
    for img, kind in ((g, "u8"), (gf, "float32")):
        for ks in ksizes:
            gp = dict(maxCorners=maxc, qualityLevel=0.007, minDistance=10, blockSize=10, gradientSize=ks)
            for _ in range(3):
                cv.goodFeaturesToTrack(img, **gp)
            reps, ts = 20, []
            for _ in range(reps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); p = cv.goodFeaturesToTrack(img, **gp); e1.record(); e1.synchronize()
                ts.append(e0.elapsed_time(e1))
            ts.sort()
            print("%-7s gradientSize %2d: median %.3f ms  min %.3f ms  (%d calls)  corners %s" % (
                kind, ks, ts[reps // 2], ts[0], reps, None if p is None else p.shape[0]))
    sys.exit(0)

for it in range(3):
    torch.cuda.synchronize(); t0 = time.perf_counter()
    p = cv.goodFeaturesToTrack(g, maxCorners=maxc, qualityLevel=0.007, minDistance=10, blockSize=10)
    torch.cuda.synchronize(); print("gftt ms", (time.perf_counter() - t0) * 1e3, None if p is None else tuple(p.shape))

# phase stamps of the select kernel (GfttCounters.tstamp: after 6+2+64+4096 uint32)
import numpy as np
ws = cv._gftt_workspace(g.device, H, W)[0]
off = (8 + 64 + 4096) * 4
ts = ws[off:off + 16 * 8].cpu().numpy().view(np.uint64).astype(np.int64)
names = {0: "start", 1: "hist+zero", 2: "bins", 3: "select", 4: "pass4", 5: "pass5", 6: "pass6", 7: "pass7", 8: "pos+cells", 9: "cull", 10: "write"}
prev = ts[0]
for i in range(1, 11):
    if ts[i] >= ts[0] and ts[i] > 0:
        print("  %-10s +%6.1f us (at %6.1f)" % (names[i], (ts[i] - prev) / 1e3, (ts[i] - ts[0]) / 1e3)); prev = ts[i]
