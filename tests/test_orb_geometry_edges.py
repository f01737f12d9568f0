"""ORB at the default 31-px patch around the edgeThresholds where the kernel choice changes (orb.cu): the intensity-centroid
disc fits the fast orientation kernel from edge 16, bit_pattern_31_ fits the staged rBRIEF kernel and the tile kernel from
edge 19.  Below those the general kernels read cv::ORB's bordered image (raw reflect-101 pixels outside the image).
Every path must equal the oracle assembled from its parts, and the detect-and-describe path must be the tile kernel exactly
from edge 19 on."""
import numpy as np
import pytest

from oracle import fast as ofast
from oracle import orb as oorb
from oracle import synth

pytestmark = pytest.mark.gpu

H, W, N_FEATURES, THRESHOLD = 240, 320, 5000, 15
TILE_FROM_EDGE = 19


def _oracle(img, edge):
    xs, ys, resp = ofast.fast_detect(img, THRESHOLD, 16, True)
    xs, ys, resp = oorb.border_and_retain_best(xs, ys, resp, img.shape, N_FEATURES, edge)
    ang, _, _ = oorb.ic_angle(img, xs, ys)
    # raw=img: below edge 19 the steered pattern leaves the image
    desc = oorb.rbrief256(oorb.gaussian_blur_7x7(img), xs, ys, ang, raw=img)
    return xs, ys, resp, ang, desc


def _check(k, d, ref, edge, what):
    xs, ys, resp, ang, desc = ref
    assert np.array_equal(k["x"], xs.astype(np.float32)) and np.array_equal(k["y"], ys.astype(np.float32)), what
    assert np.array_equal(k["response"], resp.astype(np.float32)), what
    assert np.array_equal(k["angle"], ang), what
    assert np.all(k["size"] == 31) and np.all(k["octave"] == 0), what
    assert np.array_equal(d, desc), what


def _took_tiles(f):
    """The tile kernel describes without an orientation launch of its own."""
    return f.stage_times()["orient_pack"][1] == 0


@pytest.mark.parametrize("edge", [15, 16, 18, 19, 20])
def test_orb_edge_threshold_paths_vs_oracle(fe, edge):
    L, R = synth.stereo_pair(H, W, 13)
    refs = [_oracle(img, edge) for img in (L, R)]
    for xs, ys, _, _, _ in refs:         # keypoints exactly on the border filter's edge, on all four sides
        assert np.any(xs == edge) and np.any(xs == W - 1 - edge) and np.any(ys == edge) and np.any(ys == H - 1 - edge)
    with fe.FrontEnd(max_width=W, max_height=H, max_pairs=1, max_keypoints=8192, n_features=N_FEATURES,
                     fast_threshold=THRESHOLD, edge_threshold=edge) as f:
        f.profile_reset()
        lk, ld, rk, rd, _ = f.stereo_features(L, R)
        assert _took_tiles(f) == (edge >= TILE_FROM_EDGE)
        _check(lk, ld, refs[0], edge, "stereo_features left")
        _check(rk, rd, refs[1], edge, "stereo_features right")

        f.profile_reset()
        f.batch_upload(L[None], R[None])
        f.batch_run(fe.match_cfg(), None, sync=True)
        assert _took_tiles(f) == (edge >= TILE_FROM_EDGE)
        out = f.batch_download()
        for i, ref in enumerate(refs):
            n = int(out["n_kps"][i])
            _check(out["kps"][i][:n], out["desc"][i][:n], ref, edge, "batch image %d" % i)

        for img, k, ref in ((L, lk, refs[0]), (R, rk, refs[1])):
            k2, d2 = f.compute(img, k)
            assert k2.tobytes() == k.tobytes()
            assert np.array_equal(d2, ref[4])
