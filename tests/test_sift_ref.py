"""tests/sift_ref.py is OpenCV's SIFT: the float64 restatement against cv2.SIFT_create(2500, 3, 0.04, 5, 1.2) on small
rendered, noise and blob images (CPU only).  The GPU stage tests (test_gpu_sift.py) rest on this."""
import cv2
import numpy as np
import pytest

import sift_ref as R
from conftest import render_clip


def _rendered(texture_small, W, H, start):
    return cv2.cvtColor(render_clip(texture_small, W, H, 1, start=start)[0], cv2.COLOR_BGR2GRAY)


def _blobs(W, H, period=16, seed=3):
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float64)
    rng = np.random.default_rng(seed)
    img = 60 + 25 * rng.random((H, W))
    for cy in range(period // 2, H, period):
        for cx in range(period // 2, W, period):
            img += 140 * np.exp(-((yy - cy) ** 2 + (xx - cx) ** 2) / (2 * (1.5 + (cx * 7 + cy) % 3) ** 2))
    return np.clip(img, 0, 255).astype(np.uint8)


def _agreement(gray):
    kps, desc = R.detect_and_compute(gray)
    ck, cd = cv2.SIFT_create(2500, 3, 0.04, 5, 1.2).detectAndCompute(gray, None)
    pos = np.stack([kps["x"], kps["y"]], 1).astype(np.float64)
    hit, used, worst = 0, set(), 0
    for i, k in enumerate(ck):
        near = np.abs(pos - np.array(k.pt)).max(1) < 1e-3
        dang = np.abs((kps["angle"].astype(np.float64) - k.angle + 180) % 360 - 180)
        j = np.nonzero(near & (kps["octave"] == k.octave) & (dang < 0.01))[0]
        j = [x for x in j if x not in used]
        if j:
            hit += 1
            used.add(j[0])
            worst = max(worst, int(np.abs(R.quantize(desc[j[0]]).astype(int) - cd[i].astype(int)).max()))
    return len(kps), len(ck), hit, worst


@pytest.mark.parametrize("kind", ["rendered", "noise", "blobs"])
def test_reference_is_opencv_sift(texture_small, kind):
    if kind == "rendered":
        gray = _rendered(texture_small, 320, 180, 2)
    elif kind == "noise":
        gray = np.random.default_rng(11).integers(0, 256, (90, 121), dtype=np.uint8)
    else:
        gray = _blobs(150, 100)
    n, nc, hit, worst = _agreement(gray)
    print(f"{kind}: reference {n}, cv2 {nc}, matched {hit} (same octave word, <= 1e-3 px, <= 0.01 deg), "
          f"max |desc diff| {worst}")
    assert nc > 30
    assert hit >= 0.99 * nc and hit >= 0.99 * n
    assert worst <= 1


def test_kernels_equal_opencv():
    init, inc = R.sigmas()
    taps = R.all_taps()
    assert [len(t) // 2 for t in taps] == [3, 4, 5, 6, 8, 10]
    for s, t in zip([init] + inc, taps):
        k = cv2.getGaussianKernel(R.kernel_size(s), s, cv2.CV_32F).ravel()
        assert np.array_equal(k.astype(np.float64), t), s


def test_blur_border_and_geometry():
    """REFLECT_101 reflected again for kernels wider than the image (cv2.GaussianBlur on float), the octave sizes, the
    nearest decimation."""
    rng = np.random.default_rng(2)
    for h, w in [(3, 6), (7, 12), (15, 24), (40, 33)]:
        img = (rng.random((h, w)) * 255).astype(np.float32)
        for t in R.all_taps():
            s = float(np.sqrt(-1 / (2 * np.log(t[len(t) // 2 + 1] / t[len(t) // 2]))))   # sigma back from the taps
            want = cv2.GaussianBlur(img, (len(t), len(t)), s, s, borderType=cv2.BORDER_REFLECT_101)
            assert np.abs(R.blur64(img, t) - want).max() < 1e-3
        assert np.array_equal(R.blur64(img, R.all_taps()[5], rows=slice(1, h - 1)), R.blur64(img, R.all_taps()[5])[1:h - 1])
    g3 = rng.random((33, 27))
    assert np.array_equal(R.next_octave_base(g3), cv2.resize(g3, (13, 16), interpolation=cv2.INTER_NEAREST))
    assert R.octave_shapes(61, 97) == [(122, 194), (61, 97), (30, 48), (15, 24), (7, 12), (3, 6)]
    assert R.n_octaves(2160, 3840) == 11
    g = rng.integers(0, 256, (9, 14), dtype=np.uint8)
    assert np.array_equal(R.upsample2x(g), cv2.resize(g.astype(np.float32), (28, 18), interpolation=cv2.INTER_LINEAR))


def test_selection_rules():
    """removeDuplicatedSorted (exact equality), retainBest keeps every tie of the threshold, the octave -1 rescale and
    the relative-size filter."""
    k = np.zeros(6, R.KP_DTYPE)
    k["x"] = [4, 4, 4, 2, 8, 8]
    k["y"] = [2, 2, 2, 6, 1, 1]
    k["size"] = [3, 3, 5, 40, 3, 3]
    k["angle"] = [10, 10, 10, 0, 30, 20]
    k["response"] = [0.5, 0.5, 0.5, 0.7, 0.5, 0.1]
    k["octave"] = [0 + (1 << 8)] * 6
    s = R.select(k, 100, nfeatures=3)
    assert len(s) == 4                                   # one duplicate gone, the three responses tied at 0.5 all kept
    assert list(s["x"]) == [1, 2, 2, 4] and list(s["size"]) == [20, 2.5, 1.5, 1.5]
    assert np.all((s["octave"] & 255) == 255) and np.all((s["octave"] >> 8) == 1)
    assert len(R.select(k, 100)) == 5 and len(R.select(k, 100, size_ratio=0.05)) == 4     # size 20 >= 5 goes
    assert len(R.select(k, 400, size_ratio=0.05)) == 4   # 20 < 400 * 0.05 = 20 is false
    assert len(R.select(k, 401, size_ratio=0.05)) == 5
