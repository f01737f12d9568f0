#!/usr/bin/env python
"""The SURF service chain on the device: Fast-Hessian detection in the batched pipeline (fe_set_batch_detector).

usage: python tools/surf_service_time.py [--out FILE.json] [--repeats 3] [--min-seconds 1.0]

Workload: 96 pairs of 1280x720 (synth.stereo_batch), cv::SURF with hessianThreshold 100, 4 octaves, 2 layers, SURF-128
oriented; stereo mode A (|dy| <= 2, Lowe 0.8) and mode B (cross-check + |dy| <= 0.7), both FE_NORM_L2.

Reported, in one JSON:
  - kernel-only: fe_batch_run on the resident batch, CUDA events on the ctx stream over windows of at least --min-seconds
    after warm-up, --repeats repeats;
  - the stage split (fe_stage_times, the library's own event pairs) and the launches per step, in a separate window;
  - end to end: fe_pipeline_batch (H2D + kernels + D2H into pinned host arrays), host clock around synchronous calls;
  - for scale, the download-and-reupload recipe the batch replaces: fe_surf_detect_batch on the 192 images, then one
    fe_stereo_match per pair and mode on the downloaded keypoints and rows (host clock).
The device name, power limit and the SM clock sampled during the timed windows go into the same JSON.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def smi(query):
    r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + query, "--format=csv,noheader,nounits"],
                       capture_output=True, text=True, timeout=30)
    return [v.strip() for v in r.stdout.strip().split(",")] if r.returncode == 0 else None


class ClockSampler:
    """SM clock (MHz) every 0.2 s while running."""

    def __init__(self):
        self.samples, self._stop = [], threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            v = smi("clocks.sm")
            if v:
                self.samples.append(float(v[0]))
            self._stop.wait(0.2)

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--pairs", type=int, default=96)
    args = ap.parse_args()

    import torch

    import front_end_b200 as fe
    from front_end_b200 import synth

    h, w, P = 720, 1280, args.pairs
    surf = dict(hessian_threshold=100.0, n_octaves=4, n_octave_layers=2, extended=True, upright=False)
    Ls, Rs = synth.stereo_batch(h, w, P)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    ca = fe.match_cfg(mode=fe.MATCH_RATIO, mask=fe.MASK_EPIPOLAR, epi_threshold=2.0, ratio=0.8, norm=fe.NORM_L2)
    cb = fe.match_cfg(mode=fe.MATCH_CROSSCHECK, mask=fe.MASK_NONE, norm=fe.NORM_L2, max_dy=0.7)

    f = fe.FrontEnd(max_width=w, max_height=h, max_pairs=P)
    f.set_batch_detector(surf)
    stream = torch.cuda.ExternalStream(f.stream, device=dev)

    def events(step, n_steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f.sync()
        e0.record(stream)
        for _ in range(n_steps):
            step()
        e1.record(stream)
        f.sync()
        return e0.elapsed_time(e1) / n_steps

    def host(step, n_steps):
        f.sync()
        t0 = time.perf_counter()
        for _ in range(n_steps):
            step()
        f.sync()
        return (time.perf_counter() - t0) * 1e3 / n_steps

    def measure(step, clock):
        for _ in range(2):
            step()
        n = max(2, int(np.ceil(args.min_seconds / (clock(step, 2) / 1000.0))))
        reps, clocks = [], []
        for _ in range(args.repeats):
            with ClockSampler() as cs:
                reps.append(clock(step, n))
            clocks += cs.samples
        med = statistics.median(reps)
        return dict(ms_per_step=[round(v, 4) for v in reps], ms_per_step_median=round(med, 4),
                    pairs_per_s_median=round(P / (med / 1000.0), 1), steps_per_window=n,
                    window_s=round(min(reps) * n / 1000.0, 3), sm_clock_mhz_median=statistics.median(clocks) if clocks else None)

    name, power_limit, max_sm = smi("name,power.limit,clocks.max.sm") or (None, None, None)
    result = dict(tool="tools/surf_service_time.py", device=name, power_limit_w=power_limit, sm_clock_max_mhz=max_sm,
                  workload=dict(pairs=P, width=w, height=h, surf=surf, kp_cap=f.max_keypoints,
                                mode_a="ratio 0.8 on |dy| <= 2 (L2)", mode_b="cross-check + |dy| <= 0.7 (L2)"),
                  timing="kernel-only: CUDA events on the ctx stream; end to end and the recipe: host clock around "
                         "synchronous calls; %d repeats of >= %.1f s windows after warm-up" % (args.repeats, args.min_seconds))
    arms = {}

    # kernel-only on the resident batch
    f.batch_upload(Ls, Rs)
    run = lambda: f.batch_run(ca, cb)                                        # noqa: E731
    arms["kernel_only"] = measure(run, events)
    f.profile(True)
    f.profile_reset()
    launches0 = f.kernel_launches()
    n = arms["kernel_only"]["steps_per_window"]
    for _ in range(n):
        run()
    st = f.stage_times()
    f.profile(False)
    arms["kernel_only"]["stage_ms_per_step"] = {k: round(v[0] / n, 4) for k, v in st.items() if v[1]}
    arms["kernel_only"]["stage_launches_per_step"] = {k: v[1] // n for k, v in st.items() if v[1]}
    arms["kernel_only"]["launches_per_step"] = (f.kernel_launches() - launches0) // n
    out = f.batch_download()
    arms["kernel_only"]["keypoints_per_image_mean"] = float(out["n_kps"].mean())
    arms["kernel_only"]["keypoints_per_image_max"] = int(out["n_kps"].max())
    arms["kernel_only"]["mode_a_matches_per_pair_mean"] = float(out["n_a"].mean())
    arms["kernel_only"]["mode_b_matches_per_pair_mean"] = float(out["n_b"].mean())

    # end to end: one fe_pipeline_batch call per step into pinned outputs
    pout = f.alloc_batch_outputs(P, pinned=True)
    arms["end_to_end_pipeline_batch"] = measure(lambda: f.pipeline_batch(Ls, Rs, ca, cb, out=pout), host)
    h2d, d2h = f.transfer_bytes()

    # the recipe the batch replaces: detect every image, download, re-upload one pair and mode at a time
    kind = fe.DESC_SURF128
    imgs = np.stack([im for p in range(P) for im in (Ls[p], Rs[p])])

    def recipe():
        kps, desc = f.surf_detect_batch(imgs, **surf)
        for p in range(P):
            f.stereo_match(kps[2 * p], desc[2 * p], kps[2 * p + 1], desc[2 * p + 1], ca, kind=kind)
            f.stereo_match(kps[2 * p], desc[2 * p], kps[2 * p + 1], desc[2 * p + 1], cb, kind=kind)

    arms["recipe_surf_detect_batch_plus_stereo_match"] = measure(recipe, host)
    f.close()
    for k in ("end_to_end_pipeline_batch", "recipe_surf_detect_batch_plus_stereo_match"):
        arms[k]["vs_kernel_only"] = round(arms[k]["ms_per_step_median"] / arms["kernel_only"]["ms_per_step_median"], 2)
    result["arms"] = arms
    result["transfer_bytes_total"] = dict(h2d=h2d, d2h=d2h)
    line = json.dumps(result, indent=1)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
