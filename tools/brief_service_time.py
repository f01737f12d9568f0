#!/usr/bin/env python
"""The BRIEF service chain on the device: BRIEF-32 / BRIEF-16 in the batched pipeline (fe_set_batch_descriptor).

usage: python tools/brief_service_time.py [--out FILE.json] [--parent-root DIR] [--repeats 3] [--min-seconds 1.0]

Workload: 96 pairs of 1280x720 (synth.stereo_batch), ORB detector with n_features 5000, described with BRIEF-32 and then
BRIEF-16 (seeded random test tables, oriented); stereo mode A (|dy| <= 2, Lowe 0.8) and mode B (cross-check + |dy| <= 0.7).

Reported per width, in one JSON:
  - kernel-only: fe_batch_run on the resident batch, CUDA events on the ctx stream over windows of at least --min-seconds
    after warm-up, --repeats repeats; the stage split (fe_stage_times) in a separate window; brief_border_kernel and
    brief_tile_kernel on their own from torch.profiler's CUDA activity in a third window;
  - end to end: fe_pipeline_batch (H2D + kernels + D2H into pinned host arrays), host clock around synchronous calls;
  - the host recipe the batch replaces: the batch's keypoints downloaded, fe_describe per image, fe_stereo_match per pair
    and mode (host clock).
And, for BRIEF-16 rows: the hamming_cross stage of host fe_stereo_match cross-checks over the 96 pairs of the batch's rows,
with this build's 8-half join and, given --parent-root (a built tree of the parent commit), the parent's 16-half join,
alternating the two builds in child processes.  The device name, power limit and SM clock go into the same JSON.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


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


def cross_child(rows_npz, reps):
    """Child process: the hamming_cross stage (ms) of one host cross-check per pair over the saved BRIEF-16 rows, with the
    front_end_b200 found first on sys.path (this build or the parent's)."""
    import front_end_b200 as fe
    d = np.load(rows_npz)
    P = int(d["P"])
    cb = fe.match_cfg(mode=fe.MATCH_CROSSCHECK, mask=fe.MASK_NONE, max_dy=0.7)
    out = []
    with fe.FrontEnd(max_width=1280, max_height=720, max_pairs=1) as f:
        f.profile(True)
        for r in range(reps + 1):                     # the first pass is warm-up
            f.profile_reset()
            for p in range(P):
                nl, nr = int(d["n"][2 * p]), int(d["n"][2 * p + 1])
                f.stereo_match(d["kps"][2 * p][:nl], d["desc"][2 * p][:nl], d["kps"][2 * p + 1][:nr], d["desc"][2 * p + 1][:nr],
                               cb, kind=fe.DESC_BRIEF16)
            st = f.stage_times()["hamming_cross"]
            if r:
                out.append(dict(ms=st[0], launches=st[1]))
    print(json.dumps(dict(runs=out)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--pairs", type=int, default=96)
    ap.add_argument("--parent-root", default=None, help="a built tree of the parent commit (its front_end_b200 and .so)")
    ap.add_argument("--cross-child", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.cross_child:
        cross_child(args.cross_child, args.repeats)
        return
    sys.path.insert(0, ROOT)

    import torch

    import front_end_b200 as fe
    from front_end_b200 import synth
    from oracle import brief as obrief

    h, w, P = 720, 1280, args.pairs
    Ls, Rs = synth.stereo_batch(h, w, P)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    ca = fe.match_cfg()
    cb = fe.match_cfg(mode=fe.MATCH_CROSSCHECK, mask=fe.MASK_NONE, max_dy=0.7)

    def measure(f, step, clock):
        for _ in range(2):
            step()
        n = max(2, int(np.ceil(args.min_seconds / (clock(f, step, 2) / 1000.0))))
        reps, clocks = [], []
        for _ in range(args.repeats):
            with ClockSampler() as cs:
                reps.append(clock(f, step, n))
            clocks += cs.samples
        med = statistics.median(reps)
        return dict(ms_per_step=[round(v, 4) for v in reps], ms_per_step_median=round(med, 4),
                    pairs_per_s_median=round(P / (med / 1000.0), 1), steps_per_window=n,
                    window_s=round(min(reps) * n / 1000.0, 3), sm_clock_mhz_median=statistics.median(clocks) if clocks else None)

    def events(f, step, n_steps):
        stream = torch.cuda.ExternalStream(f.stream, device=dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f.sync()
        e0.record(stream)
        for _ in range(n_steps):
            step()
        e1.record(stream)
        f.sync()
        return e0.elapsed_time(e1) / n_steps

    def host(f, step, n_steps):
        f.sync()
        t0 = time.perf_counter()
        for _ in range(n_steps):
            step()
        f.sync()
        return (time.perf_counter() - t0) * 1e3 / n_steps

    name, power_limit, max_sm = smi("name,power.limit,clocks.max.sm") or (None, None, None)
    result = dict(tool="tools/brief_service_time.py", device=name, power_limit_w=power_limit, sm_clock_max_mhz=max_sm,
                  workload=dict(pairs=P, width=w, height=h, detector="ORB n_features 5000, edge 31, FAST-9_16",
                                tables="oracle.brief.random_tests(bytes, seed 7 / 8), use_orientation",
                                mode_a="ratio 0.8 on |dy| <= 2", mode_b="cross-check + |dy| <= 0.7"),
                  timing="kernel-only: CUDA events on the ctx stream; end to end and the recipe: host clock around "
                         "synchronous calls; %d repeats of >= %.1f s windows after warm-up" % (args.repeats, args.min_seconds))
    widths = {}
    rows16 = None
    for n_bytes, kind, seed in ((32, fe.DESC_BRIEF32, 8), (16, fe.DESC_BRIEF16, 7)):
        arms = {}
        f = fe.FrontEnd(max_width=w, max_height=h, max_pairs=P)
        f.set_brief_pattern(obrief.random_tests(n_bytes, seed), use_orientation=True)
        f.set_batch_descriptor(kind)
        f.batch_upload(Ls, Rs)
        run = lambda: f.batch_run(ca, cb)                                    # noqa: E731
        arms["kernel_only"] = measure(f, run, events)
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
        # the two BRIEF kernels on their own: torch.profiler's CUDA activity over steps of their own (profiling slows the host,
        # so this window is not one of the timed ones)
        from torch.profiler import ProfilerActivity, profile
        n_prof = 20
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(n_prof):
                run()
            f.sync()
        kernels = {}
        for e in prof.key_averages():
            for name in ("brief_border_kernel", "brief_tile_kernel"):
                if name in e.key:
                    us = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
                    kernels[name] = round(kernels.get(name, 0.0) + us / 1000.0 / n_prof, 4)
        arms["kernel_only"]["kernel_ms_per_step_profiler"] = kernels
        out = f.batch_download()
        arms["kernel_only"]["keypoints_per_image_mean"] = float(out["n_kps"].mean())
        arms["kernel_only"]["mode_a_matches_per_pair_mean"] = float(out["n_a"].mean())
        arms["kernel_only"]["mode_b_matches_per_pair_mean"] = float(out["n_b"].mean())
        if n_bytes == 16:
            rows16 = dict(P=P, n=out["n_kps"].copy(), kps=out["kps"].copy(), desc=out["desc"].copy())

        pout = f.alloc_batch_outputs(P, pinned=True)
        arms["end_to_end_pipeline_batch"] = measure(f, lambda: f.pipeline_batch(Ls, Rs, ca, cb, out=pout), host)

        # the recipe the batch replaces: the batch's keypoints downloaded, fe_describe per image, fe_stereo_match per pair
        # and mode (the batch's own detection is not part of it)
        kps = [out["kps"][i][:out["n_kps"][i]].copy() for i in range(2 * P)]
        imgs = [im for p in range(P) for im in (Ls[p], Rs[p])]
        g = fe.FrontEnd(max_width=w, max_height=h, max_pairs=1)
        g.set_brief_pattern(obrief.random_tests(n_bytes, seed), use_orientation=True)

        def recipe():
            d = [g.compute(imgs[i], kps[i], kind) for i in range(2 * P)]
            for p in range(P):
                (lk, ld), (rk, rd) = d[2 * p], d[2 * p + 1]
                g.stereo_match(lk, ld, rk, rd, ca, kind=kind)
                g.stereo_match(lk, ld, rk, rd, cb, kind=kind)

        arms["recipe_download_describe_stereo_match"] = measure(g, recipe, host)
        g.close()
        f.close()
        for k in ("end_to_end_pipeline_batch", "recipe_download_describe_stereo_match"):
            arms[k]["vs_kernel_only"] = round(arms[k]["ms_per_step_median"] / arms["kernel_only"]["ms_per_step_median"], 2)
        widths["brief%d" % n_bytes] = arms
    result["widths"] = widths

    # the cross-check stage on BRIEF-16 rows: this build (8-half join) and the parent (16-half join), alternating
    with tempfile.TemporaryDirectory() as tmp:
        npz = os.path.join(tmp, "rows16.npz")
        np.savez(npz, **rows16)
        roots = [("this_build_8_half_join", ROOT)] + ([("parent_16_half_join", os.path.abspath(args.parent_root))]
                                                     if args.parent_root else [])
        cross = {k: [] for k, _ in roots}
        for _ in range(2):
            for k, root in roots:
                env = dict(os.environ, PYTHONPATH=root)
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--cross-child", npz, "--repeats", "3"],
                                   capture_output=True, text=True, env=env, cwd=tmp, timeout=3600)
                if r.returncode != 0:
                    raise RuntimeError("cross-check child failed (%s): %s" % (k, r.stderr[-2000:]))
                cross[k].append(json.loads(r.stdout.strip().splitlines()[-1]))
        result["brief16_host_cross_check_stage"] = dict(
            what="hamming_cross stage ms summed over one host fe_stereo_match cross-check (|dy| <= 0.7) per pair of the "
                 "BRIEF-16 batch's rows (%d pairs), per pass; each child process runs a warm-up pass and 3 timed passes" % P,
            runs=cross,
            ms_median={k: statistics.median(r["ms"] for c in v for r in c["runs"]) for k, v in cross.items()})
    line = json.dumps(result, indent=1)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
