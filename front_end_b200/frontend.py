"""Host-side handle on one fe_ctx (one GPU, one stream).

Method names follow the reference's call sites: ``detect`` / ``compute`` are what
bin/feature_node:50-66 calls on its OpenCV detector / extractor objects, ``knnMatch`` / ``match`` are
the BFMatcher calls of src/front_end/algorithm.py:848-853 and features.py:724, ``stereo_match`` is
stereoMatching (bin/stereo_node:20) and ``window_match`` is WindowMatcher::newStereo's matching
stage (src/WindowMatcher.cpp:104-231).  All arithmetic happens in libfe_b200.so.
"""
import ctypes as C

import numpy as np

from . import lib as L

_lib = None
_SURF_DIM = {L.DESC_SURF64: 64, L.DESC_SURF128: 128}       # float row width of the SURF descriptor kinds
# (width, dtype) of one descriptor row on the host, per descriptor kind
_ROW = {L.DESC_ORB256: (32, np.uint8), L.DESC_SURF64: (64, np.float32), L.DESC_SURF128: (128, np.float32),
        L.DESC_BRIEF16: (16, np.uint8), L.DESC_BRIEF32: (32, np.uint8), L.DESC_BRIEF64: (64, np.uint8), L.DESC_FREAK: (64, np.uint8)}


def get_lib():
    global _lib
    if _lib is None:
        _lib = L.load()
    return _lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _u8img(img):
    img = np.asarray(img)
    if img.dtype != np.uint8 or img.ndim != 2:
        raise ValueError("expected a 2-D uint8 (mono8) image")
    return np.ascontiguousarray(img)


class FrontEnd:
    def __init__(self, device=0, max_width=1920, max_height=1200, max_pairs=1, max_keypoints=16384,
                 fast_threshold=15, fast_type=L.FAST_9_16, nonmax=True, n_features=5000, edge_threshold=31,
                 orientation=True, surf_upright=True, stream=None):
        self.lib = get_lib()
        cfg = L.Config(device, max_width, max_height, 2 * max_pairs, max_keypoints, fast_threshold,
                       fast_type, int(nonmax), n_features, edge_threshold, int(orientation), int(surf_upright), stream)
        h = C.c_void_p()
        st = self.lib.fe_create(C.byref(cfg), C.byref(h))
        if st != L.FE_OK:
            raise L.FeError(st, (self.lib.fe_last_error(None) or b"").decode())
        self.h = h
        self.max_keypoints = max_keypoints
        self.max_pairs = max_pairs
        self._pinned = []

    # -- lifecycle ------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "h", None):
            self.lib.fe_destroy(self.h)
            self.h = None
        for p in self._pinned:
            p.close()
        self._pinned = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, st, allow_capacity=False):
        if st == L.FE_OK or (allow_capacity and st == L.FE_ERR_CAPACITY):
            return st
        raise L.FeError(st, (self.lib.fe_last_error(self.h) or b"").decode())

    def pinned(self, shape, dtype):
        p = L.PinnedArray(self.lib, shape, dtype)
        self._pinned.append(p)
        return p.array

    # -- srv/controlDetection.srv ---------------------------------------------------------------------
    def control_detection(self, threshold, set_point):
        out = C.c_int32()
        self._check(self.lib.fe_set_detection(self.h, threshold, set_point, C.byref(out)))
        return out.value

    # -- FeatureDetector::detect ----------------------------------------------------------------------
    def detect(self, img, cap=None):
        img = _u8img(img)
        cap = cap or self.max_keypoints
        out = np.zeros(cap, L.KPOINT)
        n = C.c_int32()
        self._check(self.lib.fe_detect(self.h, _ptr(img), img.shape[1], img.shape[0], img.strides[0],
                                       _ptr(out), cap, C.byref(n)))
        return out[:n.value]

    # -- cv2.cornerSubPix(img, pts, (5, 5), (-1, -1), (EPS | COUNT, 40, 0.001)) --------------------------------
    def corner_subpix(self, img, kps):
        img = _u8img(img)
        kps = np.ascontiguousarray(kps, dtype=L.KPOINT).copy()
        self._check(self.lib.fe_corner_subpix(self.h, _ptr(img), img.shape[1], img.shape[0], img.strides[0],
                                              _ptr(kps), len(kps)))
        return kps

    # -- gridDetector.detect (features.py:609-641) / live_stereo.cpp:277-352, one eye -------------------------
    def grid_detect(self, img, thresholds, set_point, roi=None, rows=2, cols=3, variant=0, fast_type=L.FAST_7_12,
                    subpix=True, update=True, cap=None):
        """Returns (keypoints, per-cell counts (rows, cols), new thresholds (rows, cols))."""
        img = _u8img(img)
        cap = cap or self.max_keypoints
        thr = np.ascontiguousarray(np.asarray(thresholds, np.int32).reshape(rows * cols)).copy()
        counts = np.zeros(rows * cols, np.int32)
        x, y, w, h = roi if roi is not None else (0, 0, 0, 0)
        cfg = L.GridCfg(x, y, w, h, rows, cols, variant, fast_type, set_point, 0, 0, int(subpix), int(update))
        out = np.zeros(cap, L.KPOINT)
        n = C.c_int32()
        self._check(self.lib.fe_grid_detect(self.h, _ptr(img), img.shape[1], img.shape[0], img.strides[0],
                                            C.byref(cfg), _ptr(thr), _ptr(out), cap, C.byref(n), _ptr(counts)))
        return out[:n.value], counts.reshape(rows, cols), thr.reshape(rows, cols)

    # -- cv::SURF::operator()(img, mask, kps, desc) : Fast-Hessian detect + describe (src/surf.cpp:896-980) -------
    def surf_detect_and_compute(self, img, hessian_threshold=100.0, n_octaves=4, n_octave_layers=2, extended=False,
                                upright=False, cap=None, want_desc=True):
        img = _u8img(img)
        cap = cap or self.max_keypoints
        sp = L.SurfParams(hessian_threshold, n_octaves, n_octave_layers, int(extended), int(upright))
        kps = np.zeros(cap, L.KPOINT)
        dim = 128 if extended else 64
        desc = np.zeros((cap, dim), np.float32) if want_desc else None
        n = C.c_int32()
        self._check(self.lib.fe_surf_detect_and_compute(self.h, _ptr(img), img.shape[1], img.shape[0], img.strides[0],
                                                        C.byref(sp), _ptr(kps), _ptr(desc), cap, C.byref(n)))
        return kps[:n.value], (desc[:n.value] if want_desc else None)

    def surf_detect_batch(self, imgs, hessian_threshold=100.0, n_octaves=4, n_octave_layers=2, extended=False, upright=False,
                          cap=None, want_desc=True):
        """cv::SURF::operator() on a stack of images, device resident: returns (list of kps, list of desc)."""
        imgs = self._u8stack(imgs)
        cap = cap or self.max_keypoints
        sp = L.SurfParams(hessian_threshold, n_octaves, n_octave_layers, int(extended), int(upright))
        n_img = imgs.shape[0]
        kps = np.zeros((n_img, cap), L.KPOINT)
        dim = 128 if extended else 64
        desc = np.zeros((n_img, cap, dim), np.float32) if want_desc else None
        n = np.zeros(n_img, np.int32)
        self._check(self.lib.fe_surf_detect_batch(self.h, n_img, _ptr(imgs), imgs.shape[2], imgs.shape[1], C.byref(sp), _ptr(kps),
                                                  _ptr(desc), cap, _ptr(n)))
        return [kps[i][:n[i]] for i in range(n_img)], ([desc[i][:n[i]] for i in range(n_img)] if want_desc else None)

    # -- DescriptorExtractor::compute -----------------------------------------------------------------
    def compute(self, img, kps, kind=L.DESC_ORB256):
        img = _u8img(img)
        kps = np.ascontiguousarray(kps, dtype=L.KPOINT).copy()
        n = C.c_int32(len(kps))
        width = _ROW[kind]
        desc = np.zeros((max(len(kps), 1), width[0]), width[1])
        self._check(self.lib.fe_describe(self.h, _ptr(img), img.shape[1], img.shape[0], img.strides[0],
                                         _ptr(kps), C.byref(n), _ptr(desc), kind))
        return kps[:n.value], desc[:n.value]

    # -- BFMatcher::knnMatch(q, t, 2, mask) ---------------------------------------------------------------
    def knnMatch(self, q_kps, q_desc, t_kps, t_desc, cfg, kind=L.DESC_ORB256):
        q_kps = np.ascontiguousarray(q_kps, dtype=L.KPOINT)
        t_kps = np.ascontiguousarray(t_kps, dtype=L.KPOINT)
        q_desc, t_desc = np.ascontiguousarray(q_desc), np.ascontiguousarray(t_desc)
        idx = np.zeros((max(len(q_kps), 1), 2), np.int32)
        dist = np.zeros((max(len(q_kps), 1), 2), np.float32)
        self._check(self.lib.fe_knn2(self.h, _ptr(q_kps), _ptr(q_desc), len(q_kps), _ptr(t_kps), _ptr(t_desc),
                                     len(t_kps), kind, C.byref(cfg), _ptr(idx), _ptr(dist)))
        return idx[:len(q_kps)], dist[:len(q_kps)]

    def _match(self, fn, q_kps, q_desc, t_kps, t_desc, cfg, kind):
        q_kps = np.ascontiguousarray(q_kps, dtype=L.KPOINT)
        t_kps = np.ascontiguousarray(t_kps, dtype=L.KPOINT)
        q_desc, t_desc = np.ascontiguousarray(q_desc), np.ascontiguousarray(t_desc)
        cap = max(len(q_kps), 1)
        out = np.zeros(cap, L.MATCH)
        n = C.c_int32()
        self._check(fn(self.h, _ptr(q_kps), _ptr(q_desc), len(q_kps), _ptr(t_kps), _ptr(t_desc), len(t_kps),
                       kind, C.byref(cfg), _ptr(out), cap, C.byref(n)))
        return out[:n.value]

    # -- stereoMatching / live match stage ---------------------------------------------------------------
    def stereo_match(self, l_kps, l_desc, r_kps, r_desc, cfg, kind=L.DESC_ORB256):
        return self._match(self.lib.fe_stereo_match, l_kps, l_desc, r_kps, r_desc, cfg, kind)

    # -- WindowMatcher::newStereo matching stage ---------------------------------------------------------
    def window_match(self, cur_kps, cur_desc, prev_kps, prev_desc, cfg=None, kind=L.DESC_ORB256):
        cfg = cfg or L.match_cfg(mask=L.MASK_WINDOW)
        return self._match(self.lib.fe_window_match, cur_kps, cur_desc, prev_kps, prev_desc, cfg, kind)

    # -- srv/windowMatching.srv: the stateful window (WindowMatcher.cpp:92-102 / the Python window service) ----------
    def window_update(self, l_kps=None, l_desc=None, r_desc=None, cfg=None, reset=False, length=0, variant=0, kind=L.DESC_ORB256):
        """Returns (tracks, frames_in_window).  cfg: ratio + MASK_WINDOW (WindowMatcher) or cross-check + MASK_NONE
        (liveGraph: needs r_desc); its norm defaults to NORM_L2 for DESC_SURF64 / DESC_SURF128 rows ((n, 64) / (n, 128)
        float32), Hamming otherwise.  Switching between binary, SURF-64 and SURF-128 rows needs a reset first.
        reset=True clears the window."""
        nt, fr = C.c_int32(), C.c_int32()
        wc = L.WindowCfg(length, variant)
        if reset:
            self._check(self.lib.fe_window_update(self.h, 1, None, None, None, 0, kind, None, C.byref(wc), None, 0, C.byref(nt), C.byref(fr)))
            return np.zeros(0, L.MATCH), 0
        dim = _SURF_DIM.get(kind, 0)
        cfg = cfg or L.match_cfg(mask=L.MASK_WINDOW, norm=L.NORM_L2 if dim else L.NORM_HAMMING)
        l_kps = np.ascontiguousarray(l_kps, dtype=L.KPOINT)
        l_desc = np.ascontiguousarray(l_desc)
        r_desc = np.ascontiguousarray(r_desc) if r_desc is not None else None
        if dim:
            for d in (l_desc, r_desc):
                if d is not None and (d.dtype != np.float32 or d.shape != (len(l_kps), dim)):
                    raise ValueError("SURF-%d rows: expected a (%d, %d) float32 array" % (dim, len(l_kps), dim))
        cap = max(len(l_kps), 1)
        out = np.zeros(cap, L.MATCH)
        self._check(self.lib.fe_window_update(self.h, 0, _ptr(l_kps), _ptr(l_desc), _ptr(r_desc), len(l_kps), kind, C.byref(cfg),
                                              C.byref(wc), _ptr(out), cap, C.byref(nt), C.byref(fr)))
        return out[:nt.value], fr.value

    # -- getStereoFeatures --------------------------------------------------------------------------------
    def stereo_features(self, left, right, kind=L.DESC_ORB256, cap=None):
        """getStereoFeatures: detect on both eyes and describe with kind (DESC_ORB256, DESC_SURF64 / 128, or DESC_BRIEF16 / 32 /
        64 with the table of set_brief_pattern, after BRIEF's 28-px border).  Returns (l_kps, l_desc, r_kps, r_desc, proc)."""
        left, right = _u8img(left), _u8img(right)
        if left.shape != right.shape or left.strides != right.strides:
            raise ValueError("left/right geometry differs")
        cap = cap or self.max_keypoints
        lk, rk = np.zeros(cap, L.KPOINT), np.zeros(cap, L.KPOINT)
        dw, dt = _ROW[kind]
        ld, rd = np.zeros((cap, dw), dt), np.zeros((cap, dw), dt)
        nl, nr = C.c_int32(), C.c_int32()
        proc = (C.c_double * 4)()
        self._check(self.lib.fe_stereo_features(self.h, _ptr(left), _ptr(right), left.shape[1], left.shape[0],
                                                left.strides[0], kind, _ptr(lk), _ptr(ld), C.byref(nl), _ptr(rk),
                                                _ptr(rd), C.byref(nr), cap, proc))
        return (lk[:nl.value], ld[:nl.value], rk[:nr.value], rd[:nr.value], list(proc))

    def window_batch(self, cfg=None, Q=None, cap=None, out=None):
        """WindowMatcher over the resident sequence (call after batch_run / pipeline_batch with a ratio cfg_a on
        consecutive frames; the default cfg matches SURF batches with NORM_L2).  Returns (tracks [F-1][cap],
        n_tracks [F-1], xyz [F][cap][3] or None)."""
        surf = getattr(self, "_batch_kind", L.DESC_ORB256) in _SURF_DIM
        cfg = cfg or L.match_cfg(mask=L.MASK_WINDOW, norm=L.NORM_L2 if surf else L.NORM_HAMMING)
        cap = cap or self.max_keypoints
        F = self._n_pairs
        if out is not None:                       # caller-owned (e.g. pinned) result buffers: (tracks [>= F-1][cap], n [>= F-1])
            tracks, n = out
        else:
            tracks = np.zeros((max(F - 1, 1), cap), L.MATCH)
            n = np.zeros(max(F - 1, 1), np.int32)
        xyz = np.zeros((F, cap, 3), np.float64) if Q is not None else None
        q = np.ascontiguousarray(Q, np.float64).reshape(16) if Q is not None else None
        self._check(self.lib.fe_window_batch(self.h, C.byref(cfg), _ptr(q), cap, _ptr(tracks), _ptr(n), _ptr(xyz)))
        return tracks[:F - 1], n[:F - 1], xyz

    def set_pyramid(self, nlevels, scale_factor=1.2):
        """nlevels / scaleFactor of cv2.ORB_create (features.py:378-387)."""
        self._check(self.lib.fe_set_orb_pyramid(self.h, nlevels, scale_factor))

    def setWTA_K(self, wta_k):
        """cv2.ORB.setWTA_K: 3 / 4 -> two-bit symbols, match with NORM_HAMMING2."""
        self._check(self.lib.fe_set_orb_wta_k(self.h, wta_k))

    def setScoreType(self, score_type):
        """cv2.ORB.setScoreType: 0 = ORB_HARRIS_SCORE, 1 = ORB_FAST_SCORE."""
        self._check(self.lib.fe_set_orb_score_type(self.h, int(score_type)))

    def set_brief_pattern(self, tests, use_orientation=False):
        """cv2.xfeatures2d.BriefDescriptorExtractor_create(bytes, use_orientation) / cv::BriefDescriptorExtractor(bytes)
        (src/live_stereo.cpp:238): tests = (bytes * 8, 4) int8 rows (y1, x1, y2, x2), bytes in {16, 32, 64}."""
        tests = np.ascontiguousarray(tests, np.int8)
        if tests.ndim != 2 or tests.shape[1] != 4 or tests.shape[0] not in (128, 256, 512):
            raise ValueError("expected (bytes * 8, 4) tests with bytes in {16, 32, 64}")
        self._check(self.lib.fe_set_brief_pattern(self.h, tests.shape[0] // 8, _ptr(tests), int(use_orientation)))

    def set_freak(self, selected_pairs, orientation_normalized=True, scale_normalized=True, pattern_scale=22.0, n_octaves=4):
        """cv2.xfeatures2d.FREAK_create(orientationNormalized, scaleNormalized, patternScale, nOctaves, selectedPairs)
        (bin/detect_node:43-45): selected_pairs = 512 indices into the 903 field pairs (OpenCV's default table is not shipped)."""
        sel = np.ascontiguousarray(selected_pairs, np.int32)
        if sel.shape != (512,):
            raise ValueError("expected 512 selected pair indices")
        self._check(self.lib.fe_set_freak(self.h, int(orientation_normalized), int(scale_normalized), float(pattern_scale),
                                          int(n_octaves), _ptr(sel)))

    def setPatchSize(self, patch_size):
        """cv2.ORB.setPatchSize for the rBRIEF descriptor (bin/detect_node:51)."""
        self._check(self.lib.fe_set_orb_patch_size(self.h, patch_size))

    def batch_landmarks(self, which=0, cap=None):
        """stereoLandmarks of every resident pair (algorithm.py:893-913): dict(l_kps, l_desc, r_kps, r_desc, matches, n).
        Descriptor rows: (P, cap, 32) uint8 for ORB-256 and BRIEF-32 batches, (P, cap, 16) uint8 for BRIEF-16, (P, cap, 64 / 128)
        float32 for SURF-64 / SURF-128."""
        cap = cap or self.max_keypoints
        P = self._n_pairs
        dw, dt = _ROW[getattr(self, "_batch_kind", L.DESC_ORB256)]
        out = dict(l_kps=np.zeros((P, cap), L.KPOINT), r_kps=np.zeros((P, cap), L.KPOINT),
                   l_desc=np.zeros((P, cap, dw), dt), r_desc=np.zeros((P, cap, dw), dt),
                   matches=np.zeros((P, cap), L.MATCH), n=np.zeros(P, np.int32))
        self._check(self.lib.fe_batch_landmarks(self.h, which, cap, _ptr(out["l_kps"]), _ptr(out["l_desc"]), _ptr(out["r_kps"]),
                                                _ptr(out["r_desc"]), _ptr(out["matches"]), _ptr(out["n"])))
        return out

    def set_chunk_pairs(self, pairs):
        """Pairs per chunk of pipeline_batch's overlapped copy / compute path (tuning knob; 0 = default)."""
        self._check(self.lib.fe_set_chunk_pairs(self.h, pairs))

    def set_batch_descriptor(self, kind):
        """Descriptor of the batched pipeline: DESC_ORB256 (default), DESC_SURF64 / DESC_SURF128 (matched with NORM_L2), or
        DESC_BRIEF16 / DESC_BRIEF32 (set_brief_pattern of that width first; the table and use_orientation current at batch_run /
        pipeline_batch apply; keypoints nearer than 28 px to the border are removed after detection; NORM_HAMMING)."""
        self._check(self.lib.fe_set_batch_descriptor(self.h, kind))
        self._desc_kind = self._batch_kind = kind

    def set_batch_detector(self, surf=None):
        """Detector of the batched pipeline (fe_set_batch_detector).  surf=None: FAST / ORB (the default), described with
        set_batch_descriptor's choice.  Otherwise cv::SURF's Fast-Hessian detector: a dict of surf_detect_batch's keywords
        (hessian_threshold=100.0, n_octaves=4, n_octave_layers=2, extended=False, upright=False; {} = all defaults).  Its
        batches hold the surviving keypoints in raster order with SURF-64 / SURF-128 float rows, matched with NORM_L2."""
        if surf is None:
            self._check(self.lib.fe_set_batch_detector(self.h, None))
            self._batch_kind = getattr(self, "_desc_kind", L.DESC_ORB256)
            return
        p = dict(hessian_threshold=100.0, n_octaves=4, n_octave_layers=2, extended=False, upright=False)
        unknown = set(surf) - set(p)
        if unknown:
            raise ValueError("unknown SURF parameters: %s" % sorted(unknown))
        p.update(surf)
        sp = L.SurfParams(p["hessian_threshold"], p["n_octaves"], p["n_octave_layers"], int(p["extended"]), int(p["upright"]))
        self._check(self.lib.fe_set_batch_detector(self.h, C.byref(sp)))
        self._batch_kind = L.DESC_SURF128 if p["extended"] else L.DESC_SURF64

    # -- batched pipeline -----------------------------------------------------------------------------------
    @staticmethod
    def _u8stack(a):
        a = np.asarray(a)
        if a.dtype != np.uint8 or a.ndim != 3:
            raise ValueError("expected an (n_pairs, height, width) uint8 stack")
        return np.ascontiguousarray(a)       # the C-ABI takes dense row-major images (stride = width)

    def batch_upload(self, left, right):
        left, right = self._u8stack(left), self._u8stack(right)
        if left.shape != right.shape:
            raise ValueError("left/right geometry differs")
        self._check(self.lib.fe_batch_upload(self.h, left.shape[0], _ptr(left), _ptr(right), left.shape[2],
                                             left.shape[1]))
        self._n_pairs = left.shape[0]

    def batch_run(self, cfg_a=None, cfg_b=None, sync=False):
        self._check(self.lib.fe_batch_run(self.h, C.byref(cfg_a) if cfg_a else None,
                                          C.byref(cfg_b) if cfg_b else None, int(sync)))

    def batch_download(self, out=None, want=("kps", "desc", "a", "b")):
        """Returns dict(kps, desc, n_kps, matches_a, n_a, matches_b, n_b) of slab arrays."""
        P, cap = self._n_pairs, self.max_keypoints
        if out is None:
            out = self.alloc_batch_outputs(P)
        st = self.lib.fe_batch_download(
            self.h, cap, _ptr(out["kps"]) if "kps" in want else None, _ptr(out["desc"]) if "desc" in want else None,
            _ptr(out["n_kps"]), _ptr(out["matches_a"]) if "a" in want else None, _ptr(out["n_a"]),
            _ptr(out["matches_b"]) if "b" in want else None, _ptr(out["n_b"]))
        self._check(st)
        return out

    def alloc_batch_outputs(self, n_pairs, pinned=False):
        cap = self.max_keypoints
        mk = self.pinned if pinned else (lambda shape, dt: np.zeros(shape, dt))
        dw, dt = _ROW[getattr(self, "_batch_kind", L.DESC_ORB256)]
        return dict(kps=mk((2 * n_pairs, cap), L.KPOINT), desc=mk((2 * n_pairs, cap, dw), dt),
                    n_kps=mk((2 * n_pairs,), np.int32), matches_a=mk((n_pairs, cap), L.MATCH),
                    n_a=mk((n_pairs,), np.int32), matches_b=mk((n_pairs, cap), L.MATCH), n_b=mk((n_pairs,), np.int32))

    def pipeline_batch(self, left, right, cfg_a=None, cfg_b=None, out=None):
        """One C-ABI call: H2D + detect + describe + match + D2H (fe_pipeline_batch)."""
        left, right = self._u8stack(left), self._u8stack(right)
        if left.shape != right.shape:
            raise ValueError("left/right geometry differs")
        P, cap = left.shape[0], self.max_keypoints
        if out is None:
            out = self.alloc_batch_outputs(P)
        self._n_pairs = P
        self._check(self.lib.fe_pipeline_batch(
            self.h, P, _ptr(left), _ptr(right), left.shape[2], left.shape[1],
            C.byref(cfg_a) if cfg_a else None, C.byref(cfg_b) if cfg_b else None, cap, _ptr(out["kps"]),
            _ptr(out["desc"]), _ptr(out["n_kps"]), _ptr(out["matches_a"]), _ptr(out["n_a"]),
            _ptr(out["matches_b"]), _ptr(out["n_b"])))
        return out

    # -- utilities ----------------------------------------------------------------------------------------------
    def sync(self):
        self._check(self.lib.fe_sync(self.h))

    @property
    def stream(self):
        return self.lib.fe_stream(self.h)

    def profile(self, on=True):
        self._check(self.lib.fe_profile_enable(self.h, int(on)))

    def profile_reset(self):
        self._check(self.lib.fe_profile_reset(self.h))

    def stage_times(self):
        n = 16
        names = (C.c_char_p * n)()
        ms = (C.c_double * n)()
        launches = (C.c_int64 * n)()
        cnt = C.c_int32()
        self._check(self.lib.fe_stage_times(self.h, n, names, ms, launches, C.byref(cnt)))
        return {names[i].decode(): (ms[i], launches[i]) for i in range(cnt.value)}

    def measure_popc_peak(self):
        """Measured POPC-pipe issue rate of this device in Gpopc/s (register-only probe kernel)."""
        v = C.c_double()
        self._check(self.lib.fe_measure_popc_peak(self.h, C.byref(v)))
        return v.value

    def kernel_launches(self):
        return int(self.lib.fe_kernel_launches(self.h))

    def transfer_bytes(self):
        """(h2d, d2h) bytes copied by the batched entry points since creation."""
        a, b = C.c_int64(), C.c_int64()
        self._check(self.lib.fe_transfer_bytes(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value
