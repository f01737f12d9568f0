#!/usr/bin/env python
"""Kernel-only time of config 4's shape with SURF-128 features: fe_window_batch over a resident SURF sequence.

usage: python tools/window_surf_time.py [--out FILE.json] [--repeats 3] [--min-seconds 1.0]

Workload: 9 sequences x 10 frames of 1280x720 (synth.stereo_sequence, one resident batch of 90 pairs as bench.py's c4),
N = 5000 FAST keypoints, cap 8192, upright SURF_EXTENDED, stereo ratio matching on the |dy| <= 2 band (config 3's cfg_a);
then fe_window_batch in WindowMatcher mode (100x100 box kNN-2 + Lowe 0.8) and in liveGraph mode (left and right all-pairs
FP32 cross-checks, no |dy| filter).  For scale, the ORB-256 config-4 step of the same sequences in the same run.

Every arm is timed with CUDA events on the context's stream over windows of at least --min-seconds after warm-up, three
repeats; per-stage kernel times come from fe_stage_times (the library's own event pairs) in a separate profiled window of
the same length.  The device name, power limit and the SM clock sampled during the timed windows go into the same JSON.
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
    args = ap.parse_args()

    import torch

    import front_end_b200 as fe
    from front_end_b200 import synth

    h, w, N, cap, S, F = 720, 1280, 5000, 8192, 9, 10
    P = S * F
    seqs = [synth.stereo_sequence(h, w, s, F) for s in range(S)]
    Ls = np.stack([fr[0] for sq in seqs for fr in sq])
    Rs = np.stack([fr[1] for sq in seqs for fr in sq])
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)

    def arm(surf):
        f = fe.FrontEnd(max_width=w, max_height=h, max_pairs=P, max_keypoints=cap, n_features=N, fast_threshold=15,
                        orientation=not surf, surf_upright=True)
        norm = fe.NORM_L2 if surf else fe.NORM_HAMMING
        if surf:
            f.set_batch_descriptor(fe.DESC_SURF128)
        ca = fe.match_cfg(mode=fe.MATCH_RATIO, mask=fe.MASK_EPIPOLAR, epi_threshold=2.0, ratio=0.8, norm=norm)
        f.batch_upload(Ls, Rs)
        return f, ca, norm

    wout = None

    def timed(f, step, n_steps):
        """ms per step over n_steps steps: CUDA events on the ctx stream, profiling off."""
        stream = torch.cuda.ExternalStream(f.stream, device=dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f.sync()
        e0.record(stream)
        for _ in range(n_steps):
            step()
        e1.record(stream)
        f.sync()
        return e0.elapsed_time(e1) / n_steps

    def stages(f, step, n_steps):
        f.profile(True)
        f.profile_reset()
        for _ in range(n_steps):
            step()
        st = f.stage_times()
        f.profile(False)
        return {k: round(v[0] / n_steps, 4) for k, v in st.items() if v[1]}, {k: v[1] // n_steps for k, v in st.items() if v[1]}

    def measure(f, step):
        for _ in range(3):
            step()
        n = max(3, int(np.ceil(args.min_seconds / (timed(f, step, 3) / 1000.0))))
        reps, clocks = [], []
        for _ in range(args.repeats):
            with ClockSampler() as cs:
                reps.append(timed(f, step, n))
            clocks += cs.samples
        st_ms, st_launch = stages(f, step, n)
        return dict(ms_per_step=[round(v, 4) for v in reps], ms_per_step_median=round(statistics.median(reps), 4),
                    steps_per_window=n, window_s=round(min(reps) * n / 1000.0, 3),
                    sm_clock_mhz_median=statistics.median(clocks) if clocks else None,
                    stage_ms_per_step=st_ms, stage_launches_per_step=st_launch)

    name, power_limit, max_sm = smi("name,power.limit,clocks.max.sm") or (None, None, None)
    result = dict(tool="tools/window_surf_time.py", device=name, power_limit_w=power_limit, sm_clock_max_mhz=max_sm,
                  workload=dict(sequences=S, frames=F, width=w, height=h, n_features=N, kp_cap=cap,
                                stereo="SURF-128 upright, ratio 0.8 on |dy| <= 2 (L2)"),
                  timing="CUDA events on the ctx stream, %d repeats of >= %.1f s windows after warm-up; stages: fe_stage_times"
                         % (args.repeats, args.min_seconds))
    arms = {}

    f, ca, norm = arm(True)
    wout = (np.zeros((P, cap), fe.MATCH), np.zeros(P, np.int32))
    ratio_cfg = fe.match_cfg(mask=fe.MASK_WINDOW, norm=norm)
    live_cfg = fe.match_cfg(mode=fe.MATCH_CROSSCHECK, mask=fe.MASK_NONE, norm=norm)
    arms["surf128_stereo_only"] = measure(f, lambda: f.batch_run(ca, None))
    arms["surf128_window_matcher"] = measure(f, lambda: (f.batch_run(ca, None), f.window_batch(ratio_cfg, cap=cap, out=wout)))
    arms["surf128_window_matcher"]["tracks_per_frame_pair_mean"] = float(wout[1][:P - 1].mean())
    arms["surf128_live_graph"] = measure(f, lambda: (f.batch_run(ca, None), f.window_batch(live_cfg, cap=cap, out=wout)))
    arms["surf128_live_graph"]["tracks_per_frame_pair_mean"] = float(wout[1][:P - 1].mean())
    f.close()
    f, ca, norm = arm(False)
    arms["orb256_c4_window_matcher"] = measure(f, lambda: (f.batch_run(ca, None), f.window_batch(cap=cap, out=wout)))
    arms["orb256_c4_window_matcher"]["tracks_per_frame_pair_mean"] = float(wout[1][:P - 1].mean())
    f.close()
    for k in ("surf128_window_matcher", "surf128_live_graph"):
        arms[k]["window_ms_per_step"] = round(arms[k]["ms_per_step_median"] - arms["surf128_stereo_only"]["ms_per_step_median"], 4)
    result["arms"] = arms
    line = json.dumps(result, indent=1)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
