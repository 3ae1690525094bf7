import sys, time
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import numpy as np
import face_alignment_cvpr_2012_b200 as crf
from face_alignment_cvpr_2012_b200 import workloads as wl
gm = crf.Model(packed=str(wl.staged_model_path()))
crops, _ = wl.make_crops(64)
for hs, fs in ((1, 1), (4, 3)):
    ctx = crf.Context(gm, 0, crf._options(None, hp_stride=hs, ffd_stride=fs))
    for n in (1, 4, 16):
        for _ in range(5):
            ctx.analyze_crops(crops[:n])
        ctx.set_profiling(True, False); ctx.reset_counters()
        reps = 20
        for _ in range(reps):
            ctx.analyze_crops(crops[:n])
        ms, _ = ctx.stage_ms()
        ctx.set_profiling(False, False)
        t = time.perf_counter()
        for _ in range(reps):
            ctx.analyze_crops(crops[:n])
        print(f"strides {hs}/{fs} n={n}: {(time.perf_counter() - t) / reps * 1e3:.3f} ms/call;", {k: round(v / reps, 4) for k, v in ms.items()}, flush=True)
