"""The front end's image and detection stage (CLAHE, padded pyramid, ORB blur, Shi-Tomasi corners) against cv2 at the batch size the
benchmark launches per sub-batch (16 distinct sequences), at an image size that is not a multiple of the stage's tiles, and on a
scene whose corner responses crowd one bin of the detector's candidate histogram."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MIN_DIST = 20        # configs/euroc_mono.yaml min_distance


def _textured(n, H, W, seed):
    """Smooth random texture plus pixel noise: many corners of widely spread strength."""
    import cv2
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        coarse = rng.integers(0, 256, (H // 8 + 1, W // 8 + 1)).astype(np.float32)
        img = cv2.resize(coarse, (W, H), interpolation=cv2.INTER_CUBIC) + rng.normal(0, 4, (H, W))
        out.append(np.clip(img, 0, 255).astype(np.uint8))
    return np.stack(out)


def _check_stage(b, imgs):
    import cv2
    clahe, l1, l2, blur = b.k_pyramid(imgs)
    cl = cv2.createCLAHE(3.0, (8, 8))
    for i in range(len(imgs)):
        ref = cl.apply(imgs[i]); r1 = cv2.pyrDown(ref); r2 = cv2.pyrDown(r1)
        assert np.array_equal(ref, clahe[i]), i
        assert np.array_equal(r1, l1[i]) and np.array_equal(r2, l2[i]), i
        assert np.array_equal(cv2.GaussianBlur(ref, (7, 7), 2, sigmaY=2, borderType=cv2.BORDER_REFLECT_101), blur[i]), i
    for level, ref_level in enumerate((clahe, l1, l2)):
        padded = b.k_pyramid_padded(imgs, level)
        for i in range(len(imgs)):
            ref = cv2.copyMakeBorder(ref_level[i], 24, 24, 24, 24, cv2.BORDER_REFLECT_101)
            assert np.array_equal(ref, padded[i]), (level, i)
    want = min(b.cap, 200)
    det = b.k_detect(clahe, None, want)
    for i in range(len(imgs)):
        ref = cv2.goodFeaturesToTrack(clahe[i], want, 0.01, MIN_DIST).reshape(-1, 2)
        assert np.array_equal(ref, det[i]), i                      # same corners, same order


def test_stage_at_bench_batch(cfg, lib_built):
    from larvio_b200 import api
    b = api.Batch(cfg, n_seq=16)
    try:
        _check_stage(b, _textured(16, 480, 752, 11))
    finally:
        b.close()


def test_stage_at_untiled_size(cfg, lib_built):
    """616x360: neither a multiple of the detector's 64x16 tile nor of 16 bytes per row."""
    from larvio_b200 import api
    b = api.Batch(cfg.with_overrides(resolution_width=616, resolution_height=360), n_seq=3)
    try:
        _check_stage(b, _textured(3, 360, 616, 12))
    finally:
        b.close()


def test_detector_crowded_histogram_bin(cfg, lib_built):
    """A lattice of equal blobs with pixel noise: ~10 000 corners whose responses lie within a few percent, more than 4 096 in one
    bin of the candidate histogram, so the selection has to split that bin."""
    import cv2
    from larvio_b200 import api
    rng = np.random.default_rng(0)
    img = np.zeros((480, 752), np.float32)
    img[3::6, 3::6] = 720.0
    img = cv2.GaussianBlur(img, (0, 0), 1.0) + rng.integers(0, 4, img.shape) + 60
    img = np.clip(img, 0, 255).astype(np.uint8)
    e = cv2.cornerMinEigenVal(img, 3, ksize=3)
    peak = (e == cv2.dilate(e, None)) & (e > np.float32(0.01 * e.max()))
    assert np.bincount(e[peak].view(np.int32) >> 19).max() > 4096          # the premise of this test
    b = api.Batch(cfg, n_seq=2)
    try:
        for want in (200, 37):
            det = b.k_detect(np.stack([img, img[::-1].copy()]), None, want)
            for i, im in enumerate((img, img[::-1])):
                ref = cv2.goodFeaturesToTrack(np.ascontiguousarray(im), want, 0.01, MIN_DIST).reshape(-1, 2)
                assert np.array_equal(ref, det[i]), (want, i)
    finally:
        b.close()
