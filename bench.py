#!/usr/bin/env python
"""Benchmark of the CRF inference hot path (BASELINE.json: face crops/sec, head pose + 10-pt FFD).

Workload (configs[1]): a batch of 4096 synthetic 100x100 face crops per GPU, head-pose forest + FFD forest,
dense stride-1 patches.  One step = one pass of the whole path over the batch.  Faces shard across GPUs with no
collective on the data path (weak scaling: every rank owns its own batch); the barrier and the max-over-ranks
reduction are the only torch.distributed calls.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--faces F] [--dump-outputs DIR]

`value`  : whole-job faces/s with the crops already resident in HBM (crf_analyze_crops_device), CUDA events on
           the library's stream, max over ranks.
`e2e`    : the same metric through the reference-facing C-ABI call with HOST buffers (crf_analyze_crops):
           pinned host crops -> H2D -> path -> D2H of the crf_face_t results, every step.
`roofline`: the dominant kernel (FFD forest traversal, k_traverse_win2).  achieved / peak / frac are the contract's
           HBM-EQUIVALENT figure: algorithmic bytes (SURVEY §8d: 48 B per node test + 4 B per leaf written) / the kernel's
           CUDA-event duration inside the timed region, against the measured HBM copy peak.  The gathers are served from a
           shared-memory window, so this is NOT a DRAM roofline (it exceeds 1); `roofline.physical` holds what bounds the
           kernel physically: shared-memory wavefronts per second against the SMs' LSU pipe (wavefronts per node test from
           the committed ncu capture of this build x the node tests counted live), the DRAM fraction, and the issue rate.
`kernels`: the other kernel groups, each against the unit that bounds it (executed FFMA for the Gabor bank, bytes for
           votes / MeanShift).
`other_workloads`: C2 at the reference's default strides, C3 (64 frames 1080p x 16 faces, crf_analyze_batch with host frames), C4 (head-pose
           forest only, 65 536 crops) and C5 (64 mixed-resolution images up to 4K, one call per image), each with its own CPU sample; `strong`: 32 768 C2 crops split over the ranks, records gathered on
           rank 0 inside the timed region; `single_caller`: crf_multi_* (one process, one host thread per GPU).
`cpu_baseline` / `--impl reference`: the reference's ThreadPool CPU path on the box's host cores, on a bounded sample of
           the same workload: oracle/_ref (the reference's own sources compiled against type stand-ins, `kind` "reference")
           when its text archives are staged, and the oracle port (`kind` "port"); the FASTER of the two is the headline,
           so the GPU / CPU ratio is not inflated by the stand-in's unoptimised filter2D.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "face crops/sec (head pose + 10-pt FFD)"
UNIT = "faces/s"
CROP = 100
WORKLOAD = "C2: batch of 4096 synthetic 100x100 face crops per GPU, head-pose forest + FFD forest, dense stride-1 patches"


print_line = print   # replaced in main() by a writer on the original stdout


def ncu_counters():
    """Per-kernel counters of this build from its committed `ncu --set full` capture (profiles/r2_counters.json, written by
    tools/ncu_counters.py from the round's own .ncu-rep, with the git head of the capture): DRAM bytes per launch, shared-memory
    wavefronts per node test, issue rate.  bench.py cannot run under ncu, so these per-unit figures are scaled by the work
    counted live."""
    for name in ("r2_counters.json",):
        p = ROOT / "profiles" / name
        if p.exists():
            try:
                return json.loads(p.read_text()), name
            except Exception:
                pass
    return None, None


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return json.loads(p.read_text()), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.th.join(timeout=2)
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx = float(r[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def load_models(need_gpu: bool, need_oracle: bool):
    """Staged packed image of the shipped forests if present, else seeded random forests in the same format."""
    from face_alignment_cvpr_2012_b200 import workloads as wl
    packed = wl.staged_model_path()
    gm = om = None
    if packed:
        tag = "pretrained trees_headpose + trees_ffd (packed image)"
        if need_gpu:
            import face_alignment_cvpr_2012_b200 as crf
            gm = crf.Model(packed=str(packed))
        if need_oracle:
            from oracle import oracle as O
            om = O.Model(packed=str(packed))
    else:
        import tempfile
        from face_alignment_cvpr_2012_b200 import synthetic_model as sm
        d = tempfile.mkdtemp(prefix="crf_synth_")
        hp, ffd = sm.write_model(d, seed=7, hp_depth=12, ffd_depth=13, leaf_prob=0.1)   # ~0.5 M nodes: tens of seconds to write and parse
        tag = "random-init forests of the shipped shape (staged/model.crfb200 absent)"
        if need_gpu:
            import face_alignment_cvpr_2012_b200 as crf
            gm = crf.Model(hp, ffd, 15, 20)
        if need_oracle:
            from oracle import oracle as O
            om = O.Model(hp, ffd, 15, 20)
    return gm, om, tag


def cpu_sample(om, items, hp_stride: int, ffd_stride: int, budget_s: float, max_faces: int, headpose_only: bool = False):
    """Reference-shaped CPU path of the oracle port (per-face ThreadPool over patches / Gabor filters) on all host cores.
    items: list of (bgr image, box)."""
    from oracle import oracle as O
    cores = O.hardware_concurrency()
    n, t0, ms = 0, time.perf_counter(), []
    while n < min(max_faces, len(items)) and (time.perf_counter() - t0) < budget_s:
        t1 = time.perf_counter()
        om.analyze_face(items[n][0], items[n][1], hp_stride, ffd_stride, threads=cores, headpose_only=headpose_only)
        ms.append((time.perf_counter() - t1) * 1e3); n += 1
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": UNIT, "cores": cores, "kind": "port", "faces": n, "p50_ms_per_face": float(np.median(ms))}


_REF_FF = None


def ref_forest():
    """The real reference (oracle/_ref) when its library and the text archives are staged; None otherwise."""
    global _REF_FF
    if _REF_FF is not None:
        return _REF_FF or None
    _REF_FF = False
    try:
        from oracle import ref as R
        hp, ffd = ROOT / "staged" / "trees_headpose", ROOT / "staged" / "trees_ffd"
        if not hp.exists() and R.REF_DATA is not None:
            hp, ffd = R.REF_DATA / "trees_headpose", R.REF_DATA / "trees_ffd"
        if R.available() and hp.exists() and ffd.exists():
            _REF_FF = R.FaceForest(str(hp), str(ffd))
    except Exception as e:  # noqa: BLE001
        print("reference build unavailable:", e, file=sys.stderr)
    return _REF_FF or None


def ref_sample(items, hp_stride: int, ffd_stride: int, budget_s: float, max_faces: int):
    """The same sample through the reference's own FaceForest::analyzeFace (its ThreadPool sizes itself to the host)."""
    ff = ref_forest()
    if ff is None:
        return None
    from oracle import oracle as O
    ff.set_strides(hp_stride, ffd_stride)
    n, t0, ms = 0, time.perf_counter(), []
    while n < min(max_faces, len(items)) and (time.perf_counter() - t0) < budget_s:
        t1 = time.perf_counter()
        ff.analyze_face(items[n][0], items[n][1])
        ms.append((time.perf_counter() - t1) * 1e3); n += 1
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": UNIT, "cores": O.hardware_concurrency(), "kind": "reference", "faces": n, "p50_ms_per_face": float(np.median(ms))}


def cv2_channel_ms(items, n: int = 3):
    """The channel stage alone through cv2 with all host threads (SURVEY 8d asks for it beside the port's): ms per face."""
    try:
        import cv2
        from oracle import oracle as O
        cv2.setNumThreads(O.hardware_concurrency())
        bank = O.gabor_bank()
        ts = []
        for img, box in items[:n]:
            x, y, w, h = box
            sw, sh, _ = O.scaled_size(w, h)
            t0 = time.perf_counter()
            g = cv2.resize(cv2.cvtColor(img, cv2.COLOR_BGR2GRAY)[y:y + h, x:x + w], (sw, sh), interpolation=cv2.INTER_LINEAR)
            cv2.integral(g, sdepth=cv2.CV_32F)
            for re, im in bank:
                r = cv2.filter2D(g, cv2.CV_32F, re); i = cv2.filter2D(g, cv2.CV_32F, im)
                m = cv2.pow(cv2.add(cv2.pow(i, 2), cv2.pow(r, 2)), 0.5)
                cv2.integral(cv2.convertScaleAbs(cv2.normalize(m, None, 0, 1, cv2.NORM_MINMAX), alpha=255), sdepth=cv2.CV_32F)
            cv2.integral(cv2.Sobel(g, cv2.CV_8U, 0, 1), sdepth=cv2.CV_32F); cv2.integral(cv2.Sobel(g, cv2.CV_8U, 1, 0), sdepth=cv2.CV_32F)
            ts.append((time.perf_counter() - t0) * 1e3)
        t0 = time.perf_counter()
        for img, box in items[:n]:
            x, y, w, h = box
            sw, sh, _ = O.scaled_size(w, h)
            O.channels(O.resize(O.bgr2gray(img)[y:y + h, x:x + w], sh, sw), threads=O.hardware_concurrency())
        port = (time.perf_counter() - t0) * 1e3 / max(len(items[:n]), 1)
        return {"cv2_ms_per_face": float(np.median(ts)), "port_ms_per_face": port}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def cpu_baseline(om, items, hp_stride: int, ffd_stride: int, budget_s: float, max_faces: int, what: str, headpose_only: bool = False):
    """Port and (when staged) the real reference on the same sample; the faster one is the headline.  headpose_only (C4): the port only —
    the reference's analyzeFace has no way to stop after getHeadPoseVotesMT."""
    port = cpu_sample(om, items, hp_stride, ffd_stride, budget_s, max_faces, headpose_only)
    ref = None if headpose_only else ref_sample(items, hp_stride, ffd_stride, budget_s, max_faces)
    best = dict(ref if (ref and ref["value"] > port["value"]) else port)
    best["sample"] = f"first {best['faces']} faces of {what} (strides {hp_stride}/{ffd_stride}), one face at a time, ThreadPool over {best['cores']} host threads per face"
    best["port"] = {k: port[k] for k in ("value", "faces", "p50_ms_per_face")}
    best["reference_build"] = {k: ref[k] for k in ("value", "faces", "p50_ms_per_face")} if ref else "oracle/_ref or its text archives not staged on this box"
    ch = cv2_channel_ms(items)
    best["channel_stage"] = ch
    # SURVEY 8d: use the faster channel implementation, so the speed-up is not inflated
    if best["kind"] == "port" and "cv2_ms_per_face" in ch and ch["cv2_ms_per_face"] < ch["port_ms_per_face"]:
        per_face = 1e3 / best["value"] - ch["port_ms_per_face"] + ch["cv2_ms_per_face"]
        best["value_with_port_channels"] = best["value"]
        best["value"] = 1e3 / per_face
        best["sample"] += "; channel stage re-timed through cv2 (faster than the port's)"
    return best


def run_reference(args, rank: int, world: int):
    if rank != 0:
        return 0
    from face_alignment_cvpr_2012_b200 import workloads as wl
    _, om, mtag = load_models(False, True)
    crops, dtag = wl.make_crops(64)
    items = [(c, (0, 0, CROP, CROP)) for c in crops]
    budget = max(3.0, min(12.0, 100.0 / max(args.steps + args.warmup, 1)))
    rates, last = [], None
    for s in range(args.warmup + args.steps):
        last = cpu_baseline(om, items, 1, 1, budget, 16, "the C2 batch")
        if s >= args.warmup:
            rates.append(last["value"])
    v = float(np.mean(rates))
    last["value"] = v
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * 4096 / v, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+int32", "data": dtag + "; " + mtag,
        "config": {"workload": WORKLOAD, "faces_per_gpu": args.faces, "hp_stride": 1, "ffd_stride": 1},
        "p50_ms_per_face": last["p50_ms_per_face"],
        "cpu_baseline": last,
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "CPU arm: the faster of oracle/_ref (the reference's own sources, built against OpenCV/Boost type stand-ins) and the oracle port, all host "
                "threads, one face at a time as the reference's mains do; each step is a bounded sample and ms_per_step extrapolates its rate to 4096 faces",
    }
    print_line(json.dumps(line))
    return 0


# FFMA the Gabor kernels execute per output pixel (2 flops each), counted from their loop structure: for a K x K kernel in separable
# form the row pass does (7 x 2 + 1) K multiply-adds on the (BAND + K - 1) rows a BAND-row band needs (BAND = 32, the library default; the
# 125-row crops of this workload take 4 bands of 32 rows), the column pass (7 x 4 + 1) K; the 7 x 7 scale is the direct sum, 49 taps x 7
# orientations x (re, im) with separately rounded multiply and add.
GABOR_BAND = 32
GABOR_EXECUTED_FLOP_PER_PIXEL = sum(2 * (15 * K * (GABOR_BAND - 1 + K) / GABOR_BAND + 29 * K) for K in (9, 13, 19, 25)) + 2 * 49 * 7 * 2


DUMP_BYTES = 60_000_000   # keeps a dump, .npy headers included, under 64 MB


def dump_outputs(out_dir: str, rec: np.ndarray) -> None:
    """--dump-outputs: the records the last timed step returned, one float64 array per crf_face_t field (DIR/<field>.npy,
    first axis = face, in batch order), so that two builds can be compared output for output on the same seeded inputs.
    Above DUMP_BYTES in all, a fixed seeded sample of the faces is written instead and DIR/face_index.npy lists them."""
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    per_face = 8 * sum(int(np.prod(rec.dtype[n].shape)) for n in rec.dtype.names)
    idx = np.arange(len(rec))
    if per_face * len(rec) > DUMP_BYTES:
        keep = DUMP_BYTES // (per_face + 8)
        idx = np.sort(np.random.default_rng(0).choice(len(rec), keep, replace=False))
        np.save(d / "face_index.npy", idx.astype(np.float64))
    for name in rec.dtype.names:
        np.save(d / f"{name}.npy", rec[name][idx].astype(np.float64))


def other_workloads(crf, wl, torch, gm, om, local_rank, dev, crops, args):
    """The other BASELINE configurations that the reference actually runs at (its default strides 4 / 3), on one GPU, each with a CPU
    sample of the same inputs: C2's crops at the default strides, and C3 (64 frames 1080p x 16 faces) through crf_analyze_batch."""
    out = {}
    F = len(crops)
    try:
        ctx = crf.Context(gm, local_rank, crf._options(None))
        h = torch.from_numpy(crops).pin_memory()
        rec = np.zeros(F, crf.FACE_DTYPE)
        for _ in range(3):
            ctx.analyze_crops_ptr(h.data_ptr(), F, CROP, CROP, rec)
        ctx.set_profiling(True, False); ctx.reset_counters()
        t0 = time.perf_counter()
        for _ in range(3):
            ctx.analyze_crops_ptr(h.data_ptr(), F, CROP, CROP, rec)
        dt = (time.perf_counter() - t0) / 3
        sm, _ = ctx.stage_ms()
        out["C2_default_strides"] = {"workload": f"{F} crops 100x100, reference default strides 4/3, crf_analyze_crops with pinned host buffers", "value": F / dt, "unit": UNIT,
                                     "ms_per_pass": 1e3 * dt, "stages_ms_per_pass": {k: v / 3 for k, v in sm.items()}}
        if om is not None:
            out["C2_default_strides"]["cpu_baseline"] = cpu_baseline(om, [(c, (0, 0, CROP, CROP)) for c in crops[:64]], 4, 3, 5.0, 64, "the same crops")
        frames, boxes, iob, tag = wl.make_frames(args.c3_frames, seed=2013)
        fr = torch.from_numpy(frames).pin_memory().numpy()
        for _ in range(2):
            ctx.analyze_batch(fr, boxes, iob)
        ctx.reset_counters()
        t0 = time.perf_counter()
        for _ in range(3):
            ctx.analyze_batch(fr, boxes, iob)
        dt = (time.perf_counter() - t0) / 3
        cnt = ctx.counters()
        one = [ctx.analyze_batch(fr[i:i + 1], boxes[iob == i], np.zeros(int((iob == i).sum()), np.int32)) for i in range(2)]   # warm the single-frame shapes
        t0 = time.perf_counter()
        for i in range(min(16, len(fr))):
            ctx.analyze_batch(fr[i:i + 1], boxes[iob == i], np.zeros(int((iob == i).sum()), np.int32))
        per_frame = (time.perf_counter() - t0) / min(16, len(fr))
        out["C3"] = {"workload": f"{len(fr)} frames 1080x1920 with {len(boxes)} faces in all (16 non-overlapping boxes per frame requested, boxes given), reference default strides, one crf_analyze_batch call with pinned host frames",
                     "value": len(boxes) / dt, "unit": UNIT, "frames_per_s": len(fr) / dt, "ms_per_pass": 1e3 * dt, "ms_per_frame_when_called_frame_by_frame": 1e3 * per_frame,
                     "h2d_bytes_per_pass": cnt["h2d_bytes"] // 3, "d2h_bytes_per_pass": cnt["d2h_bytes"] // 3, "data": tag}
        if om is not None:
            out["C3"]["cpu_baseline"] = cpu_baseline(om, [(frames[i], tuple(int(v) for v in b)) for b, i in zip(boxes, iob)], 4, 3, 5.0, 64, "the same frames")
        del one
        # C4: head-pose forest only on 65 536 crops at the reference's stride 4 (stops after getHeadPoseVotesMT): 16 calls on this rank's pinned
        # 4096-crop block, so that the host memory of the default run stays small; the path's cost does not depend on the content
        hp_rec = np.zeros(F, crf.FACE_DTYPE)
        ctx.analyze_crops_ptr(h.data_ptr(), F, CROP, CROP, hp_rec, headpose_only=True)
        ncall = max(1, 65536 // F)
        t0 = time.perf_counter()
        for _ in range(ncall):
            ctx.analyze_crops_ptr(h.data_ptr(), F, CROP, CROP, hp_rec, headpose_only=True)
        dt = time.perf_counter() - t0
        out["C4"] = {"workload": f"head-pose forest only, {ncall * F} crops 100x100 as {ncall} crf_headpose_crops calls of {F} pinned host crops, stride 4", "value": ncall * F / dt,
                     "unit": UNIT, "ms_per_call": 1e3 * dt / ncall}
        if om is not None:
            out["C4"]["cpu_baseline"] = cpu_baseline(om, [(c, (0, 0, CROP, CROP)) for c in crops[:64]], 4, 3, 3.0, 64, "the same crops, head pose only", headpose_only=True)
        # C5: 64 mixed-resolution images (480p .. 4K, 1-8 boxes each, widths 64..1500), one crf_analyze_faces call per image, pageable host frames
        imgs, tag5 = wl.make_mixed(args.c5_images, seed=2015)
        nfaces5 = sum(len(bx) for _, bx in imgs)
        for fr5, bx5 in imgs[:5]:
            ctx.analyze_faces(fr5, bx5)
        t0 = time.perf_counter()
        for fr5, bx5 in imgs:
            ctx.analyze_faces(fr5, bx5)
        dt = time.perf_counter() - t0
        out["C5"] = {"workload": f"{len(imgs)} mixed-resolution images (480p .. 4K) with {nfaces5} faces in all, one crf_analyze_faces call per image, pageable host frames, reference default strides",
                     "value": nfaces5 / dt, "unit": UNIT, "images_per_s": len(imgs) / dt, "ms_per_image": 1e3 * dt / len(imgs), "data": tag5}
        if om is not None:
            items5 = [(fr5, tuple(int(v) for v in b)) for fr5, bx5 in imgs for b in bx5]
            out["C5"]["cpu_baseline"] = cpu_baseline(om, items5, 4, 3, 3.0, 32, "the same images")
        ctx.close()
    except Exception as e:  # noqa: BLE001
        out["error"] = str(e)
    return out


def single_caller(crf, torch, gm, crops, args):
    """SURVEY 8(e) as one process: crf_multi_* with one context and one host thread per visible GPU, the C2 batch of every GPU in
    ONE call from this caller, records written into one array.  Under torchrun the other ranks wait at the final barrier meanwhile."""
    try:
        ndev = torch.cuda.device_count()
        if ndev < 2:
            return {"n_gpus": ndev, "skipped": "one visible GPU: the single-context numbers above are this path"}
        F = len(crops)
        mc = crf.MultiContext(gm, list(range(ndev)), crf._options(None, hp_stride=1, ffd_stride=1, max_chunk=args.chunk))
        h = torch.from_numpy(np.concatenate([crops] * ndev)).pin_memory()
        rec = np.zeros(F * ndev, crf.FACE_DTYPE)
        for _ in range(2):
            mc.analyze_crops_ptr(h.data_ptr(), F * ndev, CROP, CROP, rec)
        t0 = time.perf_counter()
        for _ in range(3):
            mc.analyze_crops_ptr(h.data_ptr(), F * ndev, CROP, CROP, rec)
        dt = (time.perf_counter() - t0) / 3
        mc.close()
        return {"n_gpus": ndev, "value": F * ndev / dt, "unit": UNIT, "ms_per_pass": 1e3 * dt, "faces_per_call": F * ndev,
                "note": "one process, crf_multi_analyze_crops: host thread + context per GPU, contiguous shards, pinned host crops in, records out"}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def run_b200(args, rank: int, world: int, local_rank: int):
    import torch
    import face_alignment_cvpr_2012_b200 as crf
    from face_alignment_cvpr_2012_b200 import capi, workloads as wl

    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    gm, om, mtag = load_models(True, rank == 0 and not args.no_cpu)
    F = args.faces
    crops, dtag = wl.make_crops(F, seed=2012 + rank)
    opt = crf._options(None, hp_stride=1, ffd_stride=1, max_chunk=args.chunk)
    ctx = crf.Context(gm, local_rank, opt)
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)

    # device-resident arm
    d_crops = torch.from_numpy(crops).to(dev)
    d_out = torch.empty(F * crf.FACE_DTYPE.itemsize, dtype=torch.uint8, device=dev)
    # host arm: pinned crops and results
    h_crops = torch.from_numpy(crops).pin_memory()
    h_out = np.zeros(F, crf.FACE_DTYPE)
    torch.cuda.synchronize()

    def step_device():
        ctx.analyze_crops_device(d_crops.data_ptr(), F, CROP, CROP, d_out.data_ptr())

    def step_host():
        ctx.analyze_crops_ptr(h_crops.data_ptr(), F, CROP, CROP, h_out)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    host_group = dist.new_group(backend="gloo") if dist is not None else None

    # ---- work counters of one step (exact, counted on the device; outside the timed region)
    ctx.set_profiling(False, True)
    ctx.reset_counters()
    step_device()
    work = ctx.counters()
    ctx.set_profiling(True, False)
    for _ in range(args.warmup):
        step_device()
    ctx.reset_counters()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step_device()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_out.cpu().numpy().view(crf.FACE_DTYPE))
    stage_ms, stage_launches = ctx.stage_ms()
    launches = ctx.counters()["kernel_launches"]
    clocks = sampler.stop() if rank == 0 else None

    # ---- end to end through the host-buffer C-ABI call
    for _ in range(max(1, min(args.warmup, 2))):
        step_host()
    ctx.reset_counters()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_host()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    cnt = ctx.counters()

    if dist is not None:
        t = torch.tensor([ms, e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_s = float(t[0]), float(t[1])

    # ---- strong scaling: 32 768 C2 crops in total, split over the ranks, records gathered on rank 0 inside the timed region
    strong = None
    try:
        total = args.strong_faces
        if total > 0:
            per = total // world
            reps = -(-per // F)
            big = torch.from_numpy(np.concatenate([crops] * reps)[:per]).pin_memory()   # the rank's own batch, repeated: the path's cost does not depend on the content
            mine = np.zeros(per, crf.FACE_DTYPE)
            gg = dist.new_group(backend="gloo") if dist is not None else None

            def strong_step():
                ctx.analyze_crops_ptr(big.data_ptr(), per, CROP, CROP, mine)
                if dist is None:
                    return mine
                parts = [None] * world if rank == 0 else None
                dist.gather_object(mine, parts, dst=0, group=gg)   # host gather of ~236 B per face, no device collective
                return np.concatenate(parts) if rank == 0 else None

            strong_step()
            barrier()
            t0 = time.perf_counter()
            for _ in range(2):
                allrec = strong_step()
            st = time.perf_counter() - t0
            barrier()
            if dist is not None:
                tt = torch.tensor([st], dtype=torch.float64, device=dev)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                st = float(tt[0])
            if rank == 0:
                strong = {"faces_total": per * world, "value": per * world * 2 / st, "unit": UNIT, "ms_per_pass": 1e3 * st / 2, "scaling": "strong",
                          "gathered_records": int(len(allrec)), "note": "host buffers -> H2D -> path -> D2H -> records of all ranks gathered on rank 0 (gloo), all inside the timed region"}
            del big
    except Exception as e:  # noqa: BLE001
        strong = {"error": str(e)}

    if rank == 0:
        peaks, peak_kind = measured_peaks()
        value = world * F * args.steps / (ms * 1e-3)
        e2e = world * F * args.steps / e2e_s
        per_step = {k: v / args.steps for k, v in stage_ms.items()}
        sm_clock = (clocks or {}).get("sm_mhz") or peaks.get("sm_max_mhz", 1965.0)
        n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
        counters, counters_src = ncu_counters()
        # dominant kernel: FFD forest traversal
        ffd_ms, hp_ms, gabor_ms = per_step["ffd_traverse"], per_step["hp_traverse"], per_step["gabor"]
        alg_bytes = 48 * work["ffd_node_tests"] + 4 * work["ffd_traversals"]
        achieved = alg_bytes / (ffd_ms * 1e-3) / 1e9 if ffd_ms > 0 else 0.0
        launches_ffd = max(stage_launches["ffd_traverse"] // args.steps, 1)

        def physical(kernel_key, tests, t_ms):
            """What bounds a window-traversal launch physically, from the committed ncu capture of this build scaled by live counts."""
            if not counters or kernel_key not in counters or t_ms <= 0:
                return None
            k = counters[kernel_key]
            wf = k["lds_wavefronts_per_node_test"] * tests            # shared-memory wavefronts of the launch
            peak_wf = n_sm * sm_clock * 1e6                            # one wavefront per SM and clock
            dram = k["dram_bytes_per_face"] * F
            return {"bound": "l1/shared data pipe (LSU wavefronts: 63 % of them bank conflicts between diverged lanes) + texture pipe (node records); not HBM",
                    "lds_wavefronts_per_s": wf / (t_ms * 1e-3), "peak_wavefronts_per_s": peak_wf, "frac": wf / (t_ms * 1e-3) / peak_wf,
                    "lds_wavefronts_per_load": k.get("lds_wavefronts_per_load"), "issue_active_pct": k.get("issue_active_pct"),
                    "long_scoreboard_stall_pct": k.get("long_scoreboard_stall_pct"),
                    "dram_bytes_per_launch": dram, "hbm_frac": dram / (t_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                    "source": f"profiles/{counters_src} (ncu --set full of this build at git {counters.get('git_head', '?')}), per-unit figures x live counts"}

        phys = physical("k_traverse_win_ffd", work["ffd_node_tests"], ffd_ms)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+int32",
            "data": dtag + "; " + mtag,
            "config": {"workload": WORKLOAD, "faces_per_gpu": F, "hp_stride": 1, "ffd_stride": 1, "chunk": args.chunk, "ms_mode": "fast (library default; landmarks within 0.5 px, see tests)",
                       "l2": "inputs larger than L2: 123 MB of crops and ~5 GB of integral stacks / Gabor scratch stream through per step"},
            "p50_ms_per_face": None,
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": cnt["h2d_bytes"] // args.steps, "d2h_bytes_per_step": cnt["d2h_bytes"] // args.steps,
                    "ms_per_step": 1e3 * e2e_s / args.steps},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"kernel": "k_traverse_win2<20,2> (FFD forest, stride 1, shared-memory window, pipelined two-walk loop)", "bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": achieved / peaks["hbm_gbs"], "traffic": phys["dram_bytes_per_launch"] / launches_ffd if phys else None, "peak_kind": peak_kind,
                         "label": "HBM-EQUIVALENT of the SURVEY 8(d) algorithmic bytes (48 B per node test + 4 B per leaf), not a DRAM roofline: the gathers are served "
                                  "from a shared-memory window, so it exceeds 1; see `physical`",
                         "alg_bytes_per_launch": alg_bytes / launches_ffd, "launches_per_step": launches_ffd, "ms_per_step": ffd_ms, "physical": phys},
            "stages_ms_per_step": per_step,
            "kernels": [
                {"kernel": "k_traverse_win2<15,2> (head-pose forest)", "ms_per_step": hp_ms,
                 "hbm_equivalent_gbs": (48 * work["hp_node_tests"] + 4 * work["hp_traversals"]) / (hp_ms * 1e-3) / 1e9 if hp_ms > 0 else 0.0,
                 "physical": physical("k_traverse_win_hp", work["hp_node_tests"], hp_ms)},
                {"kernel": "k_gabor_sep<9..25> + k_gabor_mag<7> + quantise/integral", "bound": "fp32 issue (non-tensor FFMA) + shared-memory operands", "ms_per_step": gabor_ms,
                 "achieved": GABOR_EXECUTED_FLOP_PER_PIXEL * 125 * 125 * F / (gabor_ms * 1e-3) / 1e12 if gabor_ms > 0 else 0.0,
                 "peak": n_sm * 128 * 2 * sm_clock * 1e6 / 1e12, "unit": "TFLOP/s",
                 "note": f"EXECUTED flops: {GABOR_EXECUTED_FLOP_PER_PIXEL:.0f} per pixel (separable 9..25 kernels incl. the halo rows of every 32-row band, direct 7x7), "
                         "not the 35 980 of the direct form"},
                {"kernel": "k_votes_count / offsets / emit", "bound": "hbm (latency / divergence limited)", "ms_per_step": per_step["votes"],
                 "achieved": (8 * work["ffd_traversals"] + 8 * work["votes"]) / (per_step["votes"] * 1e-3) / 1e9 if per_step["votes"] > 0 else 0.0, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                 "note": "leaf ids read twice (count, emit) + votes written"},
                {"kernel": "k_meanshift_fast", "bound": "hbm for the first pass, L2 for the rest", "ms_per_step": per_step["meanshift"],
                 "achieved": 8 * work["vote_passes"] / (per_step["meanshift"] * 1e-3) / 1e9 if per_step["meanshift"] > 0 else 0.0, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                 "note": "8 B per vote and pass; a chain's list stays L2-resident between its passes"},
            ],
            "work_per_step": {k: work[k] for k in ("hp_node_tests", "ffd_node_tests", "hp_traversals", "ffd_traversals", "votes", "vote_passes")},
            "strong": strong,
        }
        for k in line["kernels"]:
            if k.get("achieved") is not None and k.get("peak"):
                k["frac"] = k["achieved"] / k["peak"]
        # host-side p50 latency of single-face crf_analyze_crops calls: at the strides of this workload (comparable with the
        # CPU sample's p50) and at the reference's default strides 4 / 3
        try:
            def p50_single(c):
                lat, one = [], np.zeros(1, crf.FACE_DTYPE)
                for i in range(40):
                    t0 = time.perf_counter()
                    c.analyze_crops_ptr(h_crops.data_ptr() + i * CROP * CROP * 3, 1, CROP, CROP, one)
                    lat.append((time.perf_counter() - t0) * 1e3)
                return float(np.median(lat[8:]))
            line["p50_ms_per_face"] = p50_single(ctx)
            ctx_lat = crf.Context(gm, local_rank, crf._options(None))
            line["p50_ms_per_face_default_strides"] = p50_single(ctx_lat)
            line["config"]["p50"] = "single-face crf_analyze_crops calls with host buffers: stride 1 (this workload) / reference default strides 4,3"
            ctx_lat.close()
        except Exception as e:  # noqa: BLE001
            line["p50_error"] = str(e)
        items = [(c, (0, 0, CROP, CROP)) for c in crops[:64]]
        if om is not None:
            line["cpu_baseline"] = cpu_baseline(om, items, 1, 1, args.cpu_seconds, 64, "the same batch")
        if not args.no_extra:
            line["other_workloads"] = other_workloads(crf, wl, torch, gm, om, local_rank, dev, crops, args)
            line["single_caller"] = single_caller(crf, torch, gm, crops, args)
        print_line(json.dumps(line))
    if dist is not None:
        # The other ranks wait for rank 0's extra measurements on the HOST (gloo): an NCCL barrier would park a spinning kernel on their
        # GPUs, and the single-caller pass above runs on every GPU of the box (its persistent traversal CTAs would queue behind it).
        dist.barrier(group=host_group)
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--faces", type=int, default=4096)
    ap.add_argument("--chunk", type=int, default=0)
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip other_workloads / single_caller")
    ap.add_argument("--strong-faces", type=int, default=32768, help="total crops of the strong-scaling pass (0 = skip)")
    ap.add_argument("--c3-frames", type=int, default=64)
    ap.add_argument("--c5-images", type=int, default=64)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the records of the last timed step (rank 0's batch) as DIR/<field>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the records of the b200 path; the reference arm times bounded CPU samples and returns none")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly one JSON line: library banners written to fd 1 meanwhile (NCCL prints its version there) go to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    out = os.fdopen(real_stdout, "w")
    global print_line
    print_line = lambda line: (out.write(line + "\n"), out.flush())  # noqa: E731
    if args.impl == "reference":
        return run_reference(args, rank, world)
    return run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    sys.exit(main())
