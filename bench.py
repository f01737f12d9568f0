#!/usr/bin/env python
"""bench.py -- stereo pairs/sec (detect + describe + match) on synthetic rectified 1280x720 pairs,
FAST thr 15 + setpoint 5000 + ORB-256, ratio (band mask, kNN-2, Lowe 0.8) AND cross-check matching.

One "step" = one pass of the whole hot path over one batch of stereo pairs.

  value  : pairs/s, kernels only, inputs already resident in HBM (fe_batch_run), CUDA events on the
           library's stream, max over ranks.
  e2e    : pairs/s through the C-ABI call a user makes (fe_pipeline_batch) with pinned HOST buffers:
           H2D of the images and D2H of keypoints + descriptors + both match lists inside the timed
           region, every step.
  roofline / stages : per-kernel CUDA-event durations over the timed region (the library brackets every
           stage with events on its stream) against the measured HBM copy bandwidth
           (MEASURED_PEAKS.json) or, for the Hamming matcher, against a POPC-pipe peak measured in
           this run by a register-only microbenchmark kernel (fe_measure_popc_peak); `traffic` comes from the
           committed ncu --set full summary of this same command (profiles/).
  e2e_steady : the same end-to-end loop run for >= 1 s (the K-step window of `e2e` is ~0.1 s and pays for filling and
           draining the copy pipeline once).
  fabric : host <-> device copy bandwidth of THIS box measured in this run with all ranks copying at once (H2D alone,
           D2H alone, both directions together); `e2e.frac_of_fabric` = e2e / the rate at which that fabric could move
           the step's bytes.  End to end the pipeline is bound by these copies, not by the kernels.
  results_agree (N > 1) : every rank also runs one common probe batch; the SHA-256 digests of its keypoints, descriptors
           and matches are all-gathered (NCCL) and must be identical on all ranks.
  cpu_baseline : the reference's OpenCV call sequence (cv2) on the box's host cores on a bounded
           sample of the same workload (rank 0, N=1 only).
  --impl reference : the same CPU path as its own arm.
  --dump-outputs DIR : after the timed steps, what the timed path returned for its last step is written as DIR/<name>.npy
           (see dump_outputs); the inputs are seeded, so two builds run with the same arguments can be compared file by file.
  --workload c5_1024_sharded : BASELINE config 5 as written -- ONE global batch of 1024 pairs of 1920x1200 / N=10000
           partitioned frame-wise with front_end_b200.shard.shard_range over the N ranks ("scaling": "strong").

Launch: python bench.py --gpus 1 --steps K --warmup W, or under torchrun for N > 1 (one rank per GPU,
pairs sharded frame-wise, no data-path collective -- SURVEY.md section 8e).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (height, width, n_features, default pairs per GPU per step)
    "c2_1280x720_orb5000": (720, 1280, 5000, 96),
    "c1_640x480_orb5000": (480, 640, 5000, 256),
    "c5_1920x1200_orb10000": (1200, 1920, 10000, 48),
    # BASELINE config 5 as written: one GLOBAL batch of 1024 pairs, frame-sharded over the ranks (strong scaling)
    "c5_1024_sharded": (1200, 1920, 10000, 1024),
    # BASELINE config 4: WindowMatcher over 10-frame windows of ORB stereo features (src/WindowMatcher.cpp:75-231): 9 sequences
    # of 10 consecutive frames per step; stereo ratio matching per frame, then box-mask kNN-2 + Lowe between consecutive frames
    "c4_window10_orb5000": (720, 1280, 5000, 90),
    # BASELINE config 3: FAST keypoints (size 7) + SURF_EXTENDED upright (bin/detect_node:33-36), L2 matching
    "c3_1280x720_surf128": (720, 1280, 5000, 96),
}
METRIC = "stereo pairs/sec (detect+describe+match) @1280x720 ORB-5000"


def _ncu_summary(workload):
    import csv
    import glob
    tag = "c3" if "surf" in workload else "c2"
    paths = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_%s_ncu_full_summary*.csv" % tag)))
    if not paths:
        return None, None
    return list(csv.reader(open(paths[-1]))), paths[-1]


def ncu_pipes(kernel_prefix, workload):
    """ALU / XU (POPC) / issue utilisation of the named kernel (% of peak while active) from the committed ncu summary."""
    try:
        rows, path = _ncu_summary(workload)
        hdr = rows[0]
        for r in rows[1:]:
            if r[0].startswith(kernel_prefix):
                out = {k: float(r[[i for i, c in enumerate(hdr) if c.startswith(k)][0]]) for k in ("alu_pct", "xu_pct", "issue_pct")}
                out["source"] = os.path.relpath(path, ROOT)
                return out
    except Exception:
        pass
    return None


def ncu_traffic(kernel_prefix, workload):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the named kernel, from the committed summary of
    the `ncu --set full` capture of this same bench command (profiles/, produced by tools/ncu_summary.py)."""
    try:
        rows, path = _ncu_summary(workload)
        hdr = rows[0]
        ird = [i for i, c in enumerate(hdr) if c.startswith("dram_rd")][0]
        iwr = [i for i, c in enumerate(hdr) if c.startswith("dram_wr")][0]
        scale = {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}
        urd, uwr = hdr[ird].split("[")[1].rstrip("]"), hdr[iwr].split("[")[1].rstrip("]")
        for r in rows[1:]:
            if r[0].startswith(kernel_prefix):
                return float(r[ird]) * scale[urd] + float(r[iwr]) * scale[uwr], os.path.relpath(path, ROOT)
    except Exception:
        pass
    return None, None


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1):
        rows = [r for t, r in self.rows if t0 <= t <= t1 and len(r) >= 8] or [r for _, r in self.rows if len(r) >= 8]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(float(r[1]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[4 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][2]), "reasons": reasons, "samples": len(rows),
                "power_w_max": max(float(r[3]) for r in rows)}


DUMP_BUDGET = 64_000_000       # bytes of --dump-outputs files


def dump_outputs(path, res, cap, tracks=None, seed=0):
    """Writes the batch results of one step (FrontEnd.batch_download's dict; `tracks` = window_batch's (tracks, n_tracks) for
    the window workload) as float32 / float64 .npy files under `path`, at most DUMP_BUDGET bytes in all.  The counts of every
    pair are written in full; keypoints, descriptors and match lists for a sample of pairs fixed by `seed` and the batch shape,
    as many as the budget holds.  Each image's / pair's list is zero-padded to `cap` rows, so the file shapes do not depend on
    the results.  Returns {name: array}."""
    n_kps = np.minimum(res["n_kps"], cap)
    P = len(res["n_a"])
    dw = res["desc"].shape[-1]
    per_pair = 2 * cap * (7 + dw) * 4 + 2 * cap * 4 * 8 + (cap * 4 * 8 if tracks is not None else 0)
    pool = P - 1 if tracks is not None else P            # window tracks exist for the P - 1 consecutive frame pairs
    fixed = (4 * P + 2 * pool) * 8 + 16 * 1024            # counts, pair indices, .npy headers
    S = int(min(pool, max(DUMP_BUDGET - fixed, 0) // per_pair))
    pairs = np.sort(np.random.default_rng(seed).choice(pool, S, replace=False))
    imgs = np.stack([2 * pairs, 2 * pairs + 1], 1).reshape(-1)
    rows = np.arange(cap)

    def records(a, n, dtype):        # structured (..., cap) slab -> (..., cap, fields), rows past each count zeroed
        v = np.stack([a[k].astype(dtype) for k in a.dtype.names], -1)
        return np.where((rows[None, :] < n[:, None])[..., None], v, 0).astype(dtype)

    out = {"n_kps": res["n_kps"].astype(np.float64), "n_a": res["n_a"].astype(np.float64),
           "n_b": res["n_b"].astype(np.float64), "pairs": pairs.astype(np.float64),
           "kps": records(res["kps"][imgs, :cap], n_kps[imgs], np.float32).reshape(S, 2, cap, 7),
           "desc": np.where((rows[None, :] < n_kps[imgs][:, None])[..., None], res["desc"][imgs, :cap], 0)
                     .astype(np.float32).reshape(S, 2, cap, dw)}
    for k, n in (("matches_a", "n_a"), ("matches_b", "n_b")):
        out[k] = records(res[k][pairs, :cap], np.minimum(res[n][pairs], cap), np.float64)
    if tracks is not None:
        t, nt = tracks
        out["n_tracks"] = nt[:pool].astype(np.float64)
        out["tracks"] = records(t[pairs, :cap], np.minimum(nt[pairs], cap), np.float64)
    os.makedirs(path, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(path, k + ".npy"), v)
    return out


# ---- CPU arm: the reference's OpenCV call sequence ----------------------------------------------------------
def cpu_pair(L, R, n_features, cv2):
    """One stereo pair through the reference's CPU path (BASELINE.md section 2): ORB detectAndCompute L+R,
    path A (numpy band mask -> knnMatch k=2 -> ratio 0.8) and path B (crossCheck match -> |dy| <= 0.7)."""
    if cv2 is not None:
        o = cv2.ORB_create(nfeatures=n_features, scaleFactor=1.2, nlevels=1, edgeThreshold=31, firstLevel=0, WTA_K=2,
                           scoreType=cv2.ORB_FAST_SCORE, patchSize=31, fastThreshold=15)
        kl, dl = o.detectAndCompute(L, None)
        kr, dr = o.detectAndCompute(R, None)
        ly = np.array([k.pt[1] for k in kl], np.float32)
        ry = np.array([k.pt[1] for k in kr], np.float32)
        mask = (np.abs(ly[:, None] - ry[None, :]) <= np.float32(2.0)).astype(np.uint8)
        knn = cv2.BFMatcher(cv2.NORM_HAMMING, False).knnMatch(dl, dr, 2, mask)
        a = [m[0] for m in knn if len(m) == 1 or (len(m) == 2 and m[0].distance < 0.8 * m[1].distance)]
        cc = cv2.BFMatcher(cv2.NORM_HAMMING, True).match(dl, dr)
        b = [m for m in cc if abs(ly[m.queryIdx] - ry[m.trainIdx]) <= 0.7]
        return len(kl), len(kr), len(a), len(b)
    from oracle import match as omatch
    from oracle import orb as oorb
    l, r = oorb.orb_detect_and_compute(L, n_features, 15), oorb.orb_detect_and_compute(R, n_features, 15)
    qa = omatch.stereo_match_ratio(l["y"], r["y"], l["desc"], r["desc"], 2.0, 0.8)[0]
    qb = omatch.stereo_match_crosscheck(l["y"], r["y"], l["desc"], r["desc"], 0.7)[0]
    return len(l["x"]), len(r["x"]), len(qa), len(qb)


def cpu_pair_surf_seconds(L, R, n_features, cv2, sample=192):
    """BASELINE config 3 on the CPU (SURVEY section 8d: restated SURF + BFMatcher(NORM_L2)): FAST / top-N keypoints through cv2,
    SURF_EXTENDED descriptors through the numpy restatement of src/surf.cpp (oracle/surf.py, ~2.4 ms per keypoint: a full pair
    would take ~25 s), ratio + cross-check matching through cv2's BFMatcher(NORM_L2).  Bounded: the descriptor stage is TIMED ON
    `sample` KEYPOINTS PER EYE AND SCALED to the keypoint count (its cost is per keypoint); the matcher is timed in full on
    unit-norm random 128-d rows of the real counts (its time does not depend on the values).  Returns seconds per pair."""
    from oracle import surf as osurf
    o = cv2.ORB_create(nfeatures=n_features, scaleFactor=1.2, nlevels=1, edgeThreshold=31, firstLevel=0, WTA_K=2,
                       scoreType=cv2.ORB_FAST_SCORE, patchSize=31, fastThreshold=15)
    t0 = time.perf_counter()
    kl, kr = o.detect(L, None), o.detect(R, None)
    t_det = time.perf_counter() - t0
    t_desc = 0.0
    for img, kps in ((L, kl), (R, kr)):
        n = min(sample, len(kps))
        xs = np.array([k.pt[0] for k in kps[:n]], np.float32)
        ys = np.array([k.pt[1] for k in kps[:n]], np.float32)
        t0 = time.perf_counter()
        osurf.surf_compute(img, xs, ys, np.full(n, 7.0, np.float32), True, True)
        t_desc += (time.perf_counter() - t0) * (len(kps) / max(n, 1))
    rng = np.random.default_rng(0)
    dl = rng.standard_normal((len(kl), 128)).astype(np.float32)
    dr = rng.standard_normal((len(kr), 128)).astype(np.float32)
    dl /= np.linalg.norm(dl, axis=1, keepdims=True)
    dr /= np.linalg.norm(dr, axis=1, keepdims=True)
    ly = np.array([k.pt[1] for k in kl], np.float32)
    ry = np.array([k.pt[1] for k in kr], np.float32)
    t0 = time.perf_counter()
    mask = (np.abs(ly[:, None] - ry[None, :]) <= np.float32(2.0)).astype(np.uint8)
    knn = cv2.BFMatcher(cv2.NORM_L2, False).knnMatch(dl, dr, 2, mask)
    a = [m[0] for m in knn if len(m) == 1 or (len(m) == 2 and m[0].distance < 0.8 * m[1].distance)]
    cc = cv2.BFMatcher(cv2.NORM_L2, True).match(dl, dr)
    b = [m for m in cc if abs(ly[m.queryIdx] - ry[m.trainIdx]) <= 0.7]
    t_match = time.perf_counter() - t0
    return t_det + t_desc + t_match, (t_det, t_desc, t_match, len(kl), len(kr), len(a), len(b))


def cpu_arm_surf(h, w, n_features, steps, warmup):
    from oracle import synth
    import cv2
    cv2.setNumThreads(os.cpu_count() or 1)
    Ls, Rs = synth.stereo_batch(h, w, 1, seed0=0, n_scenes=1)
    times, parts = [], None
    for s in range(warmup + steps):
        dt, parts = cpu_pair_surf_seconds(Ls[0], Rs[0], n_features, cv2)
        if s >= warmup:
            times.append(dt)
    per_pair = sum(times) / len(times)
    return {"value": 1.0 / per_pair, "unit": "pairs/s", "cores": os.cpu_count() or 1, "kind": "port",
            "sample": "1 pair of the same synthetic %dx%d workload x %d steps; keypoints through cv2 %s, SURF_EXTENDED through the numpy "
                      "restatement of src/surf.cpp TIMED ON 192 KEYPOINTS PER EYE AND SCALED to the %d + %d found (descriptor time per pair "
                      "%.1f s of %.1f s), BFMatcher(NORM_L2) knnMatch + crossCheck in full on random unit rows of the real counts (%.2f s); "
                      "cv2.setNumThreads(%d)" % (w, h, len(times), cv2.__version__, parts[3], parts[4], parts[1], per_pair, parts[2],
                                                  os.cpu_count() or 1),
            "ms_per_pair": 1e3 * per_pair, "extrapolated": True}, per_pair


def cpu_window_frames(frames, n_features, cv2):
    """BASELINE config 4 on the CPU: per frame ORB L+R, band mask, knnMatch, Lowe 0.8 -> stereo landmarks; consecutive
    frames: WindowMatcher's 100 x 100 box mask on the left coordinates + knnMatch(k=2) + Lowe 0.8 (WindowMatcher.cpp:104-231)."""
    o = cv2.ORB_create(nfeatures=n_features, scaleFactor=1.2, nlevels=1, edgeThreshold=31, firstLevel=0, WTA_K=2,
                       scoreType=cv2.ORB_FAST_SCORE, patchSize=31, fastThreshold=15)
    prev = None
    n_tracks = 0
    for L, R in frames:
        kl, dl = o.detectAndCompute(L, None)
        kr, dr = o.detectAndCompute(R, None)
        lxy = np.array([k.pt for k in kl], np.float32)
        ry = np.array([k.pt[1] for k in kr], np.float32)
        mask = (np.abs(lxy[:, 1][:, None] - ry[None, :]) <= np.float32(2.0)).astype(np.uint8)
        knn = cv2.BFMatcher(cv2.NORM_HAMMING, False).knnMatch(dl, dr, 2, mask)
        a = [m[0].queryIdx for m in knn if len(m) == 1 or (len(m) == 2 and m[0].distance < 0.8 * m[1].distance)]
        cur = (lxy[a], dl[a])
        if prev is not None:
            wm = ((np.abs(cur[0][:, 0][:, None] - prev[0][:, 0][None, :]) < 50) &
                  (np.abs(cur[0][:, 1][:, None] - prev[0][:, 1][None, :]) < 50)).astype(np.uint8)
            kk = cv2.BFMatcher(cv2.NORM_HAMMING, False).knnMatch(cur[1], prev[1], 2, wm)
            n_tracks += sum(1 for m in kk if len(m) == 1 or (len(m) == 2 and m[0].distance < 0.8 * m[1].distance))
        prev = cur
    return n_tracks


def cpu_arm(h, w, n_features, n_pairs, steps, warmup, window=False):
    from oracle import synth
    try:
        import cv2
        cv2.setNumThreads(os.cpu_count() or 1)
        impl = "cv2 %s (OpenCV C++ inside; the reference's call sequence, glue in numpy)" % cv2.__version__
    except Exception:
        cv2 = None
        impl = "numpy oracle (cv2 not importable)"
    if window and cv2 is not None:
        frames = synth.stereo_sequence(h, w, 0, n_pairs)
        impl += "; stereo ratio matching per frame + WindowMatcher box-mask kNN-2 between consecutive frames"
    else:
        Ls, Rs = synth.stereo_batch(h, w, n_pairs, seed0=0, n_scenes=min(2, n_pairs))
    times = []
    for s in range(warmup + steps):
        t0 = time.perf_counter()
        if window and cv2 is not None:
            cpu_window_frames(frames, n_features, cv2)
        for p in range(0 if window and cv2 is not None else n_pairs):
            cpu_pair(Ls[p], Rs[p], n_features, cv2)
        dt = time.perf_counter() - t0
        if s >= warmup:
            times.append(dt)
    total = sum(times)
    return {"value": n_pairs * len(times) / total, "unit": "pairs/s", "cores": os.cpu_count() or 1, "kind": "port",
            "sample": "%d pairs/step x %d steps of the same synthetic %dx%d workload; %s; all host threads offered "
                      "(cv2.setNumThreads(%d)); FAST/ORB in cv2 are single-threaded, BFMatcher is parallel"
                      % (n_pairs, len(times), w, h, impl, os.cpu_count() or 1),
            "ms_per_pair": 1e3 * total / (n_pairs * len(times))}, total / len(times)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2_1280x720_orb5000", choices=sorted(WORKLOADS))
    ap.add_argument("--pairs", type=int, default=0, help="stereo pairs per GPU per step (default: workload's)")
    ap.add_argument("--cpu-pairs", type=int, default=0, help="pairs in the bounded CPU-baseline sample")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--e2e-workers", type=int, default=3, help="host threads (one fe_ctx each) issuing the e2e steps")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computes; the reference arm keeps only counts")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    h, w, n_features, def_pairs = WORKLOADS[args.workload]
    P = args.pairs or def_pairs
    sharded = args.workload == "c5_1024_sharded"
    G = P                                   # global batch (sharded workload only)
    shard_start = 0
    if sharded and args.impl != "reference":
        from front_end_b200 import shard as fe_shard
        shard_start, shard_stop = fe_shard.shard_range(G, rank, world)
        P = shard_stop - shard_start        # this rank's contiguous block of the global batch
    elif sharded:
        P = -(-G // max(args.gpus, 1))      # rank 0's block size (the CPU arm touches nothing of the GPU package)
    metric = METRIC if args.workload.startswith("c2") else "stereo pairs/sec (detect+describe+match) " + args.workload
    config = {"workload": args.workload, "width": w, "height": h, "fast_threshold": 15, "n_features": n_features,
              "descriptor": "ORB rBRIEF-256", "matching": "ratio(band |dy|<=2, kNN-2, 0.8) + cross-check(|dy|<=0.7)",
              "pairs_per_gpu_per_step": P, "sharding": "frame-wise, no collective",
              **({"global_pairs_per_step": G, "sharding": "front_end_b200.shard.shard_range(%d, rank, world): contiguous blocks of ONE "
                  "global batch, no collective" % G} if sharded else {}),
              "l2_policy": "inputs larger than L2 (%.0f MB of images per step per GPU vs 126 MB L2)" % (2 * P * w * h / 1e6)}

    if "surf" in args.workload:          # both arms carry the same config (the driver compares them)
        config["descriptor"] = "SURF_EXTENDED 128 x f32, upright, on FAST keypoints (size 7)"
        config["matching"] = "L2: ratio(band |dy|<=2, kNN-2, 0.8) + cross-check(|dy|<=0.7); exact: FP32 band candidates, ONE tcgen05 GEMM with a threshold epilogue, FP32 evaluation of the flagged elements"

    # ---- reference arm: the CPU path, rank 0 only ----------------------------------------------------------
    if args.impl == "reference":
        if rank != 0:
            return
        # each step is a BOUNDED sample of the workload's step (cpu_baseline.sample_pairs of its pairs_per_gpu_per_step
        # pairs): the CPU path needs ~0.11 s per pair, a full 96-pair step would take 11 s
        n = args.cpu_pairs or 4
        if "surf" in args.workload:
            n = 1
            cb, step_s = cpu_arm_surf(h, w, n_features, max(args.steps, 1), args.warmup)
        else:
            cb, step_s = cpu_arm(h, w, n_features, n, max(args.steps, 1), args.warmup, args.workload.startswith("c4"))
        cb["sample_pairs"] = n
        print(json.dumps({"impl": "reference", "metric": metric, "value": cb["value"], "unit": "pairs/s",
                          "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": 1e3 * step_s, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "u8", "data": "synthetic", "config": config, "cpu_baseline": cb,
                          "e2e": {"value": cb["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0,
                                  "d2h_bytes_per_step": 0}, "gpu_launches": 0}))
        return

    import torch
    import torch.distributed as dist

    import front_end_b200 as fe
    from front_end_b200 import synth  # seeded synthetic inputs (numpy); nothing under oracle/ is touched by this arm

    torch.cuda.set_device(local_rank)
    if os.environ.get("NCCL_DEBUG", "VERSION").upper() in ("VERSION", "WARN"):
        os.environ["NCCL_DEBUG"] = "NONE"      # NCCL logs to stdout: keep stdout to the one JSON line
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    window = args.workload.startswith("c4")
    if window:
        seqs = [synth.stereo_sequence(h, w, 1000 * rank + s, 10) for s in range(P // 10)]
        Ls = np.stack([fr[0] for sq in seqs for fr in sq])
        Rs = np.stack([fr[1] for sq in seqs for fr in sq])
        config["matching"] = "per frame: ratio(band |dy|<=2, kNN-2, 0.8); consecutive frames: 100x100 box kNN-2 + ratio (WindowMatcher)"
        config["sequences_x_frames"] = [P // 10, 10]
    elif sharded:
        # pairs [shard_start, shard_start + P) of the global batch; at most 128 distinct pairs are generated per rank and
        # tiled (numpy noise generation costs ~0.1 s per 1920x1200 pair), which the config states
        uniq = min(P, 128)
        Lu, Ru = synth.stereo_batch(h, w, uniq, seed0=0, n_scenes=4, first=shard_start)
        reps = -(-P // uniq)
        Ls, Rs = np.concatenate([Lu] * reps)[:P], np.concatenate([Ru] * reps)[:P]
        config["distinct_pairs_per_rank"] = uniq
    else:
        Ls, Rs = synth.stereo_batch(h, w, P, seed0=1000 * rank, n_scenes=4)
    cap = 8192 if n_features <= 5000 else 16384
    surf = "surf" in args.workload
    fe_kwargs = dict(device=local_rank, max_width=w, max_height=h, max_pairs=P, max_keypoints=cap,
                     n_features=n_features, fast_threshold=15, orientation=not surf, surf_upright=True)
    norm = fe.NORM_L2 if surf else fe.NORM_HAMMING
    f = fe.FrontEnd(**fe_kwargs)
    if surf:
        f.set_batch_descriptor(fe.DESC_SURF128)
    cfg_a = fe.match_cfg(mode=fe.MATCH_RATIO, mask=fe.MASK_EPIPOLAR, epi_threshold=2.0, ratio=0.8, norm=norm)
    cfg_b = None if window else fe.match_cfg(mode=fe.MATCH_CROSSCHECK, mask=fe.MASK_NONE, max_dy=0.7, norm=norm)

    def window_out(fw):
        return (fw.pinned((P, cap), fe.MATCH), np.zeros(P, np.int32)) if window else None
    wout = window_out(f)
    hL, hR = f.pinned(Ls.shape, np.uint8), f.pinned(Rs.shape, np.uint8)
    hL[...] = Ls
    hR[...] = Rs
    out = f.alloc_batch_outputs(P, pinned=True)
    stream = torch.cuda.ExternalStream(f.stream, device=torch.device("cuda", local_rank))

    # ---- value: kernels only, inputs resident in HBM ------------------------------------------------------
    f.batch_upload(hL, hR)
    for _ in range(max(args.warmup, 3)):
        f.batch_run(cfg_a, cfg_b, sync=True)
        if window:
            f.window_batch(cap=cap, out=wout)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    f.profile(True)
    f.profile_reset()
    l0 = f.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_start = time.perf_counter()
    e0.record(stream)
    for _ in range(args.steps):
        f.batch_run(cfg_a, cfg_b, sync=False)
        if window:
            f.window_batch(cap=cap, out=wout)     # tracks of the F-1 consecutive frame pairs (includes their D2H)
    e1.record(stream)
    f.sync()
    barrier()
    t_end = time.perf_counter()
    ms = e0.elapsed_time(e1)
    launches = f.kernel_launches() - l0
    stages = f.stage_times()
    f.profile(False)
    popc_peak = f.measure_popc_peak()       # Gpopc/s, register-only probe on this device (roofline denominator)
    res = f.batch_download(out)
    n_kps = res["n_kps"].copy()
    n_a, n_b = res["n_a"].copy(), res["n_b"].copy()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, cap, wout)

    # ---- cross-rank verification: one probe batch every rank runs, digests all-gathered over NCCL ------------------
    results_agree = None
    if world > 1:
        import hashlib
        pL, pR = synth.stereo_batch(h, w, 2, seed0=424242, n_scenes=1)
        po = f.pipeline_batch(pL, pR, cfg_a, cfg_b)
        hsh = hashlib.sha256()
        hsh.update(po["n_kps"][:4].tobytes()); hsh.update(po["n_a"][:2].tobytes()); hsh.update(po["n_b"][:2].tobytes())
        for i in range(4):
            m_ = int(min(po["n_kps"][i], cap))
            hsh.update(po["kps"][i][:m_].tobytes()); hsh.update(po["desc"][i][:m_].tobytes())
        for pi in range(2):
            hsh.update(po["matches_a"][pi][:int(min(po["n_a"][pi], cap))].tobytes())
            hsh.update(po["matches_b"][pi][:int(min(po["n_b"][pi], cap))].tobytes())
        mine_d = torch.tensor(list(hsh.digest()), dtype=torch.uint8, device="cuda")
        all_d = [torch.empty_like(mine_d) for _ in range(world)]
        dist.all_gather(all_d, mine_d)
        results_agree = bool(all(torch.equal(all_d[0], d_) for d_ in all_d))
        if int(po["n_kps"][0]) < 1000:
            results_agree = False           # an empty result on every rank is not agreement
        f.batch_upload(hL, hR)              # the probe replaced the resident batch

    # ---- e2e: the C-ABI call with host buffers, H2D + D2H inside -------------------------------------------
    # Every step is one synchronous fe_pipeline_batch call on pinned host buffers.  Like the reference's
    # StereoCamera (three worker threads, StereoCamera.cpp:5-31) the steps are issued by E2E_WORKERS host
    # threads, each owning its own fe_ctx (one ctx = one stream; ctypes releases the GIL), so one worker's
    # copies overlap the other's kernels.
    workers = [f]
    outs = [out]
    wouts = [wout]
    for _ in range(args.e2e_workers - 1):
        fw = fe.FrontEnd(**fe_kwargs)
        if surf:
            fw.set_batch_descriptor(fe.DESC_SURF128)
        workers.append(fw)
        outs.append(fw.alloc_batch_outputs(P, pinned=True))
        wouts.append(window_out(fw))
    for fw, ow, wo in zip(workers, outs, wouts):
        for _ in range(2):
            fw.pipeline_batch(hL, hR, cfg_a, cfg_b, out=ow)
            if window:
                fw.window_batch(cap=cap, out=wo)
    barrier()
    tb0 = [fw.transfer_bytes() for fw in workers]

    import itertools
    take_lock = threading.Lock()

    def make_work(n_steps):
        # the workers draw step numbers from one counter (a static split would leave one worker with the last step(s) alone)
        counter = itertools.count()

        def work(i):
            while True:
                with take_lock:
                    step = next(counter)
                if step >= n_steps:
                    return
                workers[i].pipeline_batch(hL, hR, cfg_a, cfg_b, out=outs[i])
                if window:
                    workers[i].window_batch(cap=cap, out=wouts[i])
        return work

    work = make_work(args.steps)

    threads = [threading.Thread(target=work, args=(i,)) for i in range(1, len(workers))]
    w0 = time.perf_counter()
    for t_ in threads:
        t_.start()
    work(0)
    for t_ in threads:
        t_.join()
    barrier()
    e2e_s = time.perf_counter() - w0
    t_e2e_end = time.perf_counter()
    tb1 = [fw.transfer_bytes() for fw in workers]
    tb0 = (sum(t_[0] for t_ in tb0), sum(t_[1] for t_ in tb0))
    tb1 = (sum(t_[0] for t_ in tb1), sum(t_[1] for t_ in tb1))

    # ---- e2e_steady: the same loop for >= 1 s of wall clock (same step count on every rank) ------------------------------
    per_step = torch.tensor([e2e_s / max(args.steps, 1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(per_step, op=dist.ReduceOp.MAX)
    steady_steps = int(min(max(np.ceil(1.0 / max(float(per_step[0]), 1e-6)), args.steps), 4000))
    steady_steps = -(-steady_steps // len(workers)) * len(workers)

    work_steady = make_work(steady_steps)

    threads = [threading.Thread(target=work_steady, args=(i,)) for i in range(1, len(workers))]
    barrier()
    w0 = time.perf_counter()
    for t_ in threads:
        t_.start()
    work_steady(0)
    for t_ in threads:
        t_.join()
    barrier()
    steady_s = time.perf_counter() - w0

    # ---- direction-phased schedule (front_end_b200.shard.phased_steps): all ranks copy host->device together, then all
    # device->host together; the kernels of step i overlap the downloads of step i - 1.  It pays where the host fabric
    # delivers less when the two directions compete (the 8-GPU boxes); measured beside the overlapped pipeline whenever
    # several ranks share a host, and the better of the two is reported as `e2e` (both stay in `e2e_schedules`).
    phased_s = phased_steady_s = None
    if (world > 1 or os.environ.get("FE_BENCH_PHASED") == "1") and not window and len(workers) >= 2:
        from front_end_b200 import shard as fe_shard
        hb_name = os.environ.get("MASTER_PORT", "0") + "_" + str(os.getppid() if world > 1 else os.getpid())
        hb = fe_shard.HostBarrier(hb_name, rank, world, create=True) if rank == 0 else None
        barrier()
        if hb is None:
            hb = fe_shard.HostBarrier(hb_name, rank, world, create=False)

        def run_phased(n):
            fe_shard.phased_steps(
                n,
                lambda i: (workers[i & 1].batch_upload(hL, hR), workers[i & 1].sync()),
                lambda i: workers[i & 1].batch_run(cfg_a, cfg_b, sync=False),
                lambda i: workers[i & 1].batch_download(outs[i & 1]),
                hb.wait)
        run_phased(2)
        barrier()
        w0 = time.perf_counter()
        run_phased(args.steps)
        barrier()
        phased_s = time.perf_counter() - w0
        barrier()
        w0 = time.perf_counter()
        run_phased(steady_steps)
        barrier()
        phased_steady_s = time.perf_counter() - w0
        hb.wait()
        hb.close()
    t_e2e_end = time.perf_counter()

    # ---- fabric: what the host <-> device copies of THIS box deliver with all ranks copying at once ------------------
    def measure_fabric(nbytes=128 << 20, reps=4):
        hp0 = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
        hp1 = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
        d0 = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        d1 = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()

        def up():
            with torch.cuda.stream(s1):
                d0.copy_(hp0, non_blocking=True)

        def down():
            with torch.cuda.stream(s2):
                hp1.copy_(d1, non_blocking=True)

        def timed(fn):
            fn()
            barrier()
            t0_ = time.perf_counter()
            for _ in range(reps):
                fn()
            barrier()                                   # all ranks finished: the common window
            dt_ = torch.tensor([time.perf_counter() - t0_], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(dt_, op=dist.ReduceOp.MAX)
            return world * nbytes * reps / float(dt_[0]) / 1e9      # aggregate GB/s over the box

        a = timed(up)
        b = timed(down)
        c = timed(lambda: (up(), down()))
        return {"h2d_gbs": a, "d2h_gbs": b, "duplex_gbs_each_way": c, "ranks_copying": world,
                "how": "every rank copies %d MiB x %d from / to pinned host memory at the same time; aggregate over ranks, wall clock, max over ranks" % (nbytes >> 20, reps)}

    fabric = measure_fabric()
    if rank == 0:
        time.sleep(0.2)
        sampler.stop()

    t = torch.tensor([ms, e2e_s * 1e3, steady_s * 1e3, (phased_s or 0.0) * 1e3, (phased_steady_s or 0.0) * 1e3],
                     dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max, e2e_ms_max, steady_ms_max = float(t[0]), float(t[1]), float(t[2])
    e2e_schedules = {"overlapped": {"ms": e2e_ms_max, "steady_ms": steady_ms_max,
                                    "how": "%d host threads per rank, one fe_ctx each, synchronous fe_pipeline_batch calls (chunked "
                                           "copy-in / compute / copy-out streams inside)" % len(workers)}}
    schedule = "overlapped"
    if phased_s is not None:
        e2e_schedules["phased"] = {"ms": float(t[3]), "steady_ms": float(t[4]),
                                   "how": "shard.phased_steps: per step all ranks fe_batch_upload together, fe_batch_run (async), then all "
                                          "ranks fe_batch_download the previous step together; two fe_ctx per rank; phases separated by "
                                          "shard.HostBarrier"}
        if float(t[4]) < steady_ms_max:                  # the same decision on every rank: t is the max over ranks
            schedule = "phased"
            e2e_ms_max, steady_ms_max = float(t[3]), float(t[4])
    pairs_all = torch.tensor([float(P)], dtype=torch.float64, device="cuda")     # pairs per step over all ranks
    if world > 1:
        dist.all_reduce(pairs_all, op=dist.ReduceOp.SUM)
    pairs_per_step_all = float(pairs_all[0])
    h2d = (tb1[0] - tb0[0]) // max(args.steps, 1)      # counted by the library from the copies it issued
    d2h = (tb1[1] - tb0[1]) // max(args.steps, 1)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    hbm_peak, peak_kind = measured_peaks()
    try:
        tensor_peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops_sustained"])
    except Exception:
        tensor_peak = 1400.0
    steps = args.steps
    total_pairs = pairs_per_step_all * steps
    value = total_pairs / (ms_max * 1e-3)
    # fabric ceiling of the end-to-end rate: both directions run together at the duplex rate until the smaller transfer is
    # done, the rest of the larger one at its one-way rate (bytes per step over ALL ranks)
    H_all, D_all = float(h2d) * world, float(d2h) * world
    dup = fabric["duplex_gbs_each_way"] * 1e9
    t_h, t_d = H_all / dup, D_all / dup
    if t_d <= t_h:
        t_fab = t_d + (H_all - dup * t_d) / (fabric["h2d_gbs"] * 1e9)
    else:
        t_fab = t_h + (D_all - dup * t_h) / (fabric["d2h_gbs"] * 1e9)
    fabric["pairs_per_s_ceiling"] = pairs_per_step_all / max(t_fab, 1e-12)
    # per-stage accounting (rank 0's stream; all ranks run the same shapes)
    img_bytes = 2.0 * P * w * h
    kp_total = float(np.minimum(n_kps, cap).sum())
    pair_ops = float(sum(int(min(n_kps[2 * p], cap)) * int(min(n_kps[2 * p + 1], cap)) for p in range(P))) * 8.0
    desc_bytes = 512 if surf else 32
    alg_bytes = {
        "surf_describe": kp_total * (361 + 512),             # 19 x 19 window + 128 floats
        "fast": img_bytes,                                   # one u8 read of every pixel
        "select": 0.0,
        "orient_pack": kp_total * ((0 if surf else 709) + 28),  # radius-15 disc reads (ORB mode) + wire keypoint
        "gauss7": 2.0 * img_bytes,                           # read u8, write u8
        "rbrief": kp_total * (512 + 32),                     # 512 blurred samples + 32-byte descriptor
    }
    stage_rows = []
    for name, (sms, n_l) in stages.items():
        if n_l == 0 or sms <= 0:
            continue
        per_step_ms = sms / steps
        row = {"kernel": name, "ms_per_step": per_step_ms, "launches_per_step": n_l / steps,
               "share": sms / max(ms, 1e-9)}
        if name == "hamming_cross":
            row.update(bound="int(POPC)", achieved=pair_ops / (per_step_ms * 1e-3) / 1e9, unit="Gword-popc/s")
        elif name == "l2_tensor":
            # algorithmic FLOPs of the named contraction: 2 * Nl * Nr * 128 per pair.  The kernel runs it ONCE (rows = left,
            # columns = right; the column side is verified from the same accumulators), with K = 128 + 16 (the split norms ride
            # in one extra K = 16 step whose A and B operands point at different augmentation columns) on 256 x 128 padded tiles: `executed` is what the tensor pipe did
            fl = pair_ops / 8.0 * 2.0 * 128.0
            a = fl / (per_step_ms * 1e-3) / 1e12
            pad = float(sum((-(-int(min(n_kps[2 * p], cap)) // 256) * 256) * (-(-int(min(n_kps[2 * p + 1], cap)) // 128) * 128)
                            for p in range(P)))
            ex = pad * 2.0 * 144.0 / (per_step_ms * 1e-3) / 1e12
            row.update(bound="tensor", achieved=a, unit="TFLOP/s", frac=a / tensor_peak, executed_tflops=ex,
                       executed_frac=ex / tensor_peak)
        elif name in alg_bytes and alg_bytes[name] > 0:
            a = alg_bytes[name] / (per_step_ms * 1e-3) / 1e9
            row.update(bound="hbm", achieved=a, unit="GB/s", frac=a / hbm_peak)
        stage_rows.append(row)
    stage_rows.sort(key=lambda r: -r["ms_per_step"])
    # the dominant KERNEL (longest single launch): a stage of several launches (the cross-check runs eleven kernels of at most
    # 0.22 ms) is not a kernel; its own roofline object is `roofline_matching` below
    top = max(stage_rows, key=lambda r: r["ms_per_step"] / max(r["launches_per_step"], 1.0)) if stage_rows else None
    # SURVEY section 8(d): detect+describe algorithmic bytes per step = 2*W*H per pair + sum N_out*(28 + 32)
    dd_bytes = img_bytes + kp_total * (28.0 + desc_bytes)
    dd_ms = sum(r["ms_per_step"] for r in stage_rows
                if r["kernel"] in ("fast", "select", "orient_pack", "gauss7", "rbrief", "surf_describe"))
    def matching_roofline(row):
        tr, src = ncu_traffic("hamming_verify_kernel<1", args.workload)
        if tr is None:
            tr, src = ncu_traffic("hamming_cross_kernel", args.workload)
        pruned = os.environ.get("FE_CROSS_PRUNE", "1") != "0"
        return {"kernel": "hamming_verify_kernel<LB4 / LB8 / full> (+ classify, multi-index join, finalize)" if pruned
                else "hamming_cross_kernel", "bound": "int(ALU + POPC pipes)", "achieved": row["achieved"],
                "peak": popc_peak, "unit": "Gword-popc/s", "frac": row["achieved"] / popc_peak,
                "traffic": tr, "traffic_source": src, "algorithmic_bytes": kp_total * 32.0,
                "pipe_utilisation": ncu_pipes("hamming_verify_kernel<0" if pruned else "hamming_cross_kernel", args.workload),
                "peak_kind": "measured in this run: register-only POPC probe kernel (fe_measure_popc_peak)",
                "note": "integer-pipe bound, not HBM/tensor.  `achieved` counts the ALGORITHMIC work of the reference's "
                        "cross-check -- Nl*Nr*8 32-bit XOR+POPC per pair -- over the stage's time.  The stage does not "
                        "execute all of it: band candidates + a multi-index join + one- and two-POPC lower bounds prove ~99% of the pair "
                        "distances irrelevant, the rest use carry-save adders (5 POPC per 8 words); that is why `frac` reads far "
                        "above the POPC issue rate.  pipe_utilisation is that of the full-evaluation passes (class D), which sit at "
                        "the XU / ALU co-saturation point.  Results are identical to the all-pairs kernel (FE_CROSS_PRUNE=0)."}

    def tensor_roofline(row):
        tr, src = ncu_traffic("l2v_gemm_kernel", args.workload)
        return {"kernel": "l2v_gemm_kernel", "bound": "tensor", "achieved": row["achieved"],
                "peak": tensor_peak, "unit": "TFLOP/s", "frac": row["frac"], "executed": row["executed_tflops"],
                "executed_frac": row["executed_frac"], "traffic": tr, "traffic_source": src,
                "peak_kind": "measured bf16 sustained",
                "note": "achieved = 2*Nl*Nr*128 FLOP per pair (the named contraction) / the GEMM kernel's time; it runs once "
                        "per pair (fp16 operands, fp32 accumulate, K = 144 with both norms folded in, padded tiles: `executed`); "
                        "the result is exact: band candidates + threshold epilogue + FP32 evaluation of the flagged elements"}

    roofline = None
    if top is not None:
        if top["kernel"] == "l2_tensor":
            roofline = tensor_roofline(top)
        elif top["kernel"] == "hamming_cross":
            roofline = matching_roofline(top)
        else:
            kernels = {"fast": ["fast16_strip_kernel"], "rbrief": ["rbrief_kernel"],
                       "gauss7": ["gauss7_roll_kernel"], "orient_pack": ["orient_pack_kernel"],
                       "surf_describe": ["surf_describe_kernel"]}.get(top["kernel"], [top["kernel"]])
            trs = [ncu_traffic(k, args.workload) for k in kernels]
            tr = sum(t[0] for t in trs) if all(t[0] is not None for t in trs) else None
            roofline = {"kernel": " + ".join(kernels), "bound": "hbm", "achieved": top.get("achieved"), "peak": hbm_peak,
                        "unit": "GB/s", "frac": top.get("frac"), "traffic": tr, "traffic_source": trs[0][1],
                        "algorithmic_bytes": alg_bytes.get(top["kernel"]), "peak_kind": peak_kind,
                        "pipe_utilisation": ncu_pipes(kernels[0], args.workload),
                        "note": "achieved = algorithmic bytes of the stage / its CUDA-event time.  FAST-9_16 needs 72 packed 16x2 min/max "
                                "operations per pixel pair even in the sliding-window form, all of them on the ALU pipe (VIMNMX, VIMNMX3 and "
                                "HMNMX2 issue at 64 lanes/clk/SM: profiles/r2_pipe_probe.log), so the stage is bound by instruction issue / the "
                                "ALU pipe (pipe_utilisation, from the committed ncu --set full summary), not by HBM.  `traffic` = the image "
                                "read once + the candidate list (the response map round trip of round 1 is gone): 1.23x the algorithmic bytes."
                                if top["kernel"] == "fast" else "achieved = algorithmic bytes of the stage / its CUDA-event time"}
    clocks = sampler.summary(t_start, t_e2e_end)     # kernel-only and end-to-end regions (both under load)

    cpu_baseline = None
    if world == 1 and not args.no_cpu and surf:
        cpu_baseline, _ = cpu_arm_surf(h, w, n_features, 2, 0)
    elif world == 1 and not args.no_cpu:
        cpu_baseline, _ = cpu_arm(h, w, n_features, args.cpu_pairs or 4, 3, 1, window)

    line = {"metric": metric, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_max / steps, "higher_is_better": True, "scaling": "strong" if sharded else "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic", "config": config,
            "e2e": {"value": total_pairs / (e2e_ms_max * 1e-3), "unit": "pairs/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "frac_of_fabric": total_pairs / (e2e_ms_max * 1e-3) / fabric["pairs_per_s_ceiling"],
                    "schedule": schedule,
                    "timing": "wall clock around K steps through the C-ABI with pinned host buffers (schedule: see e2e_schedules), max over ranks"},
            "e2e_steady": {"value": pairs_per_step_all * steady_steps / (steady_ms_max * 1e-3), "unit": "pairs/s", "steps": steady_steps,
                           "seconds": steady_ms_max * 1e-3,
                           "frac_of_fabric": pairs_per_step_all * steady_steps / (steady_ms_max * 1e-3) / fabric["pairs_per_s_ceiling"]},
            "e2e_schedules": e2e_schedules, "fabric": fabric, "results_agree": results_agree,
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
            "roofline_matching": next((matching_roofline(r) if r["kernel"] == "hamming_cross" else tensor_roofline(r)
                                       for r in stage_rows if r["kernel"] in ("hamming_cross", "l2_tensor")), None),
            "detect_describe": {"algorithmic_bytes_per_step": dd_bytes, "ms_per_step": dd_ms,
                                "achieved_gbs": dd_bytes / max(dd_ms * 1e-3, 1e-12) / 1e9,
                                "frac_of_hbm": dd_bytes / max(dd_ms * 1e-3, 1e-12) / 1e9 / hbm_peak, "peak_kind": peak_kind},
            "stages": stage_rows, "cpu_baseline": cpu_baseline,
            "counts": {"keypoints_per_image_mean": float(n_kps.mean()), "ratio_matches_per_pair_mean": float(n_a.mean()),
                       "crosscheck_matches_per_pair_mean": float(n_b.mean())}}
    if window:
        nt = wout[1][:P - 1].astype(np.float64)
        same = np.array([(i + 1) % 10 != 0 for i in range(P - 1)])        # frame pairs inside one sequence
        line["counts"]["tracks_per_consecutive_frame_pair_mean"] = float(nt[same].mean())
    print(json.dumps(line))
    sys.stdout.flush()
    f.close()
    if results_agree is False:
        sys.stderr.write("bench.py: the ranks' results for the common probe batch differ\n")
        sys.exit(3)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
