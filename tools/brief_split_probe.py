"""Input of tools/brief_split_probe.cu: one bench batch (c2 by default) detected by the library, written as
  int32 n_images, w, h, kp_cap | u8 images | u32 counts | f32 kx | f32 ky | f32x2 (cos, sin)
then the probe (built by the nvcc command in its header) is run on it.
  python tools/brief_split_probe.py [--height 720 --width 1280 --pairs 96 --n-features 5000]"""
import argparse
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--height", type=int, default=720)
    ap.add_argument("--width", type=int, default=1280)
    ap.add_argument("--pairs", type=int, default=96)
    ap.add_argument("--n-features", type=int, default=5000)
    ap.add_argument("--probe", default=os.path.join(ROOT, "tools", "brief_split_probe"))
    args = ap.parse_args()
    import front_end_b200 as fe
    from front_end_b200 import synth

    h, w, P, cap = args.height, args.width, args.pairs, 8192
    Ls, Rs = synth.stereo_batch(h, w, P, seed0=0, n_scenes=4)      # bench.py's c2 inputs (rank 0)
    with fe.FrontEnd(device=0, max_width=w, max_height=h, max_pairs=P, max_keypoints=cap, n_features=args.n_features) as f:
        f.batch_upload(Ls, Rs)
        f.batch_run(fe.match_cfg(), None, sync=True)
        res = f.batch_download()
    imgs = np.empty((2 * P, h, w), np.uint8)
    imgs[0::2], imgs[1::2] = Ls, Rs                                  # image 2p = left of pair p, as the library holds them
    n = np.minimum(res["n_kps"], cap).astype(np.uint32)
    kps = res["kps"]
    th = kps["angle"].astype(np.float32) * np.float32(np.pi / 180.0)
    cs = np.stack([np.cos(th.astype(np.float64)).astype(np.float32), np.sin(th.astype(np.float64)).astype(np.float32)], -1)
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "batch.bin")
        with open(path, "wb") as fo:
            np.array([2 * P, w, h, cap], np.int32).tofile(fo)
            imgs.tofile(fo)
            n.tofile(fo)
            np.ascontiguousarray(kps["x"], np.float32).tofile(fo)
            np.ascontiguousarray(kps["y"], np.float32).tofile(fo)
            np.ascontiguousarray(cs, np.float32).tofile(fo)
        sys.exit(subprocess.call([args.probe, path]))


if __name__ == "__main__":
    main()
