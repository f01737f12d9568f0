"""The batched detect-and-describe path describes keypoints per image tile (orb_describe_tile_kernel); the single-image
entry points keep the per-keypoint kernels: FrontEnd.detect() runs orient_pack_kernel and FrontEnd.compute() runs
rbrief_kernel on caller-supplied keypoints.  The two paths must agree bit for bit: every keypoint record (angle bits
included) and all 256 bits of every descriptor."""
import ctypes as C

import numpy as np
import pytest

from oracle import synth

pytestmark = pytest.mark.gpu

TILE_W, TILE_H = 256, 64          # orb_describe_tile_kernel's tile of keypoint centres


def _tile_edge_image(h, w, seed):
    """Isolated bright dots (each one FAST corner) on both sides of every tile boundary and at the tile corners, on a faint
    texture that gives the dots distinct orientations."""
    rng = np.random.default_rng(seed)
    img = (100 + rng.integers(0, 8, size=(h, w))).astype(np.uint8)
    for ty in range(0, h + TILE_H, TILE_H):
        for tx in range(0, w + TILE_W, TILE_W):
            for dx, dy in ((-1, -1), (0, 3), (-5, 0), (4, -4)):
                x, y = tx + dx, ty + dy
                if 0 <= x < w and 0 <= y < h:
                    img[y, x] = 255
                    ex, ey = x + int(rng.integers(-1, 2)), y + int(rng.integers(-1, 2))
                    if 0 <= ex < w and 0 <= ey < h and (ex, ey) != (x, y):
                        img[ey, ex] = 180
    return img


def _check_image(f, img, kps, desc, n):
    ref = f.detect(img)
    assert len(ref) == n
    assert kps.tobytes() == ref.tobytes()
    if n:
        kk, dd = f.compute(img, kps)
        assert kk.tobytes() == kps.tobytes()
        assert np.array_equal(dd, desc)


@pytest.mark.parametrize("h, w, n_features, cap", [(720, 1280, 5000, 8192), (1200, 1920, 10000, 16384),
                                                    (480, 640, 5000, 8192), (562, 1000, 5000, 8192)])
def test_batch_tiles_equal_per_keypoint_kernels(fe, h, w, n_features, cap):
    L, R = synth.stereo_pair(h, w, 7)
    flat = np.full((h, w), 128, np.uint8)
    edges = _tile_edge_image(h, w, 11)
    lefts, rights = np.stack([L, flat]), np.stack([R, edges])
    with fe.FrontEnd(max_width=w, max_height=h, max_pairs=2, max_keypoints=cap, n_features=n_features) as f:
        f.batch_upload(lefts, rights)
        f.batch_run(fe.match_cfg(), None, sync=True)
        out = f.batch_download()
        out = {k: v.copy() for k, v in out.items()}
        imgs = [L, R, flat, edges]                  # image 2p = left of pair p, 2p + 1 = right
        counts = [int(out["n_kps"][i]) for i in range(4)]
        assert counts[0] > 1000 and counts[1] > 1000 and counts[2] == 0
        k = out["kps"][3][:counts[3]]
        xs, ys = k["x"].astype(np.int32), k["y"].astype(np.int32)
        # keypoints on both sides of a tile's left / top edge, and on a tile corner
        assert np.any(xs % TILE_W == 0) and np.any(xs % TILE_W == TILE_W - 1)
        assert np.any(ys % TILE_H == 0) and np.any(ys % TILE_H == TILE_H - 1)
        assert np.any((xs % TILE_W == TILE_W - 1) & (ys % TILE_H == TILE_H - 1))
        for i, img in enumerate(imgs):
            n = counts[i]
            _check_image(f, img, out["kps"][i][:n], out["desc"][i][:n], n)


def test_batch_tiles_with_keypoints_clipped_by_capacity(fe):
    h, w, cap = 480, 640, 1000
    L, R = synth.stereo_pair(h, w, 5)
    with fe.FrontEnd(max_width=w, max_height=h, max_pairs=1, max_keypoints=cap, n_features=5000) as f:
        f.batch_upload(L[None], R[None])
        f.batch_run(fe.match_cfg(), None, sync=True)
        out = f.alloc_batch_outputs(1)
        with pytest.raises(fe.FeError) as err:       # the batch found more keypoints than max_keypoints
            f.batch_download(out)
        assert err.value.code == fe.lib.FE_ERR_CAPACITY
        for i, img in enumerate((L, R)):
            assert out["n_kps"][i] > cap
            kps, desc = out["kps"][i].copy(), out["desc"][i].copy()
            ref = np.zeros(cap, fe.KPOINT)
            n = C.c_int32()
            st = f.lib.fe_detect(f.h, img.ctypes.data_as(C.c_void_p), w, h, w, ref.ctypes.data_as(C.c_void_p), cap,
                                 C.byref(n))
            assert st == fe.lib.FE_ERR_CAPACITY and n.value == out["n_kps"][i]
            assert kps.tobytes() == ref.tobytes()
            kk, dd = f.compute(img, kps)
            assert kk.tobytes() == kps.tobytes() and np.array_equal(dd, desc)
