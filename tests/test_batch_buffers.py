"""The batched pipeline's two host paths share one batch body and one download: fe_batch_run / fe_batch_download on the
whole resident batch, and fe_pipeline_batch chunk by chunk on views of the same buffers (abi.cu).

Transfer accounting: the d2h bytes a download reports follow from the counts it returns, at the descriptor's real row
width (32 bytes for ORB-256, 256 / 512 bytes for SURF-64 / SURF-128), on both paths.

Chunked equals whole batch, bit for bit, for configurations whose buffers only exist in some contexts: the Harris
responses (HARRIS_SCORE), NORM_HAMMING2 rows of ORB WTA_K 3 with its all-pairs cross-check, and a context whose lazily
allocated cross-check scratch is first used by the whole-batch path and then viewed chunk by chunk, with a chunk size that
does not divide the pair count.
"""
import numpy as np
import pytest

from oracle import synth

pytestmark = pytest.mark.gpu

H, W, P, N, CAP = 240, 320, 10, 300, 1024


@pytest.fixture(scope="module")
def FE(fe):
    return fe


def _expected_d2h(FE, out, dim_bytes, chunk):
    """Bytes a download of `out` copies, `chunk` pairs at a time: the counts, then the longest used prefix of every array
    of the chunk, for every row of the chunk."""
    total = 0
    for p0 in range(0, len(out["n_a"]), chunk):
        n_kps, n_a, n_b = out["n_kps"][2 * p0:2 * (p0 + chunk)], out["n_a"][p0:p0 + chunk], out["n_b"][p0:p0 + chunk]
        ni, npairs = len(n_kps), len(n_a)
        max_kp, max_a, max_b = (int(np.minimum(v, CAP).max()) for v in (n_kps, n_a, n_b))
        total += (4 * (ni + 2 * npairs) + FE.KPOINT.itemsize * max_kp * ni + dim_bytes * max_kp * ni +
                  FE.MATCH.itemsize * (max_a + max_b) * npairs)
    return total


def _assert_same(out, ref):
    for k in ("n_kps", "n_a", "n_b"):
        assert np.array_equal(out[k], ref[k]), k
    for i in range(len(out["n_kps"])):
        n = out["n_kps"][i]
        assert np.array_equal(out["kps"][i][:n], ref["kps"][i][:n]), i
        assert np.array_equal(out["desc"][i][:n], ref["desc"][i][:n]), i
    for p in range(len(out["n_a"])):
        assert np.array_equal(out["matches_a"][p][:out["n_a"][p]], ref["matches_a"][p][:ref["n_a"][p]]), p
        assert np.array_equal(out["matches_b"][p][:out["n_b"][p]], ref["matches_b"][p][:ref["n_b"][p]]), p


@pytest.mark.parametrize("kind,dim_bytes", [("DESC_SURF128", 512), ("DESC_SURF64", 256), ("DESC_ORB256", 32)])
def test_download_reports_descriptor_bytes_at_their_width(FE, kind, dim_bytes):
    """fe_batch_download, and the chunked fe_pipeline_batch chunk by chunk, add exactly the bytes implied by the counts they
    return."""
    Ls, Rs = synth.stereo_batch(H, W, P, seed0=230, n_scenes=3)
    surf = kind != "DESC_ORB256"
    norm = FE.NORM_L2 if surf else FE.NORM_HAMMING
    ca = FE.match_cfg(norm=norm)
    cb = FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, norm=norm)
    with FE.FrontEnd(max_width=W, max_height=H, max_pairs=P, max_keypoints=CAP, n_features=N, orientation=not surf) as f:
        f.set_batch_descriptor(getattr(FE, kind))
        f.batch_upload(Ls, Rs)
        f.batch_run(ca, cb, sync=True)
        d0 = f.transfer_bytes()[1]
        ref = f.batch_download()
        d1 = f.transfer_bytes()[1]
        assert ref["n_kps"].min() > 100 and ref["n_b"].min() > 0
        assert d1 - d0 == _expected_d2h(FE, ref, dim_bytes, P)
        f.set_chunk_pairs(3)
        out = f.pipeline_batch(Ls, Rs, ca, cb)
        assert f.transfer_bytes()[1] - d1 == _expected_d2h(FE, out, dim_bytes, 3)
    _assert_same(out, ref)


@pytest.mark.parametrize("case", ["harris_score", "wta3_hamming2", "whole_batch_first"])
def test_chunked_pipeline_equals_whole_batch(FE, case):
    """fe_pipeline_batch in 4 chunks of 3, 3, 3 and 1 pairs equals upload / run / download bit for bit."""
    Ls, Rs = synth.stereo_batch(H, W, P, seed0=250, n_scenes=3)
    norm = FE.NORM_HAMMING2 if case == "wta3_hamming2" else FE.NORM_HAMMING
    ca = FE.match_cfg(norm=norm)
    cb = FE.match_cfg(mode=FE.MATCH_CROSSCHECK, mask=FE.MASK_NONE, norm=norm)
    with FE.FrontEnd(max_width=W, max_height=H, max_pairs=P, max_keypoints=CAP, n_features=N) as f:
        if case == "harris_score":
            f.setScoreType(0)
        if case == "wta3_hamming2":
            f.setWTA_K(3)
        f.set_chunk_pairs(3)

        def whole():
            f.batch_upload(Ls, Rs)
            f.batch_run(ca, cb, sync=True)
            return f.batch_download()

        if case == "whole_batch_first":
            ref = whole()
            out = f.pipeline_batch(Ls, Rs, ca, cb)
        else:
            out = f.pipeline_batch(Ls, Rs, ca, cb)
            ref = whole()
    assert out["n_kps"].min() > 100 and out["n_b"].min() > 0
    _assert_same(out, ref)
