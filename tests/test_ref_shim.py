"""The CPU mock of OpenCV that oracle/_ref is built against (oracle/ref_shim/w2x_cvshim.hpp), checked against the REAL OpenCV
(cv2 4.x CPU build, present in the image) through the reference functions that use each op: copyMakeBorder (padRoi), flip /
rotate (applyAugmentation, reverseAugmentation), multiply (applyWeights), split + convertTo (blobFromImages), add + convertTo +
cvtColor (render).  cv::cuda::rotate has no CPU twin with the same signature: it is checked against cv2.rotate's quarter
turns (nppiRotate with the reference's shifts is a counter-clockwise turn for angle 90)."""
import numpy as np
import pytest

import refcases
from oracle import ref

cv2 = pytest.importorskip("cv2")
pytestmark = pytest.mark.skipif(not ref.available(), reason="oracle/_ref is not built: needs the upstream waifu2x-tensorrt sources "
                                "(make -C oracle REF=<checkout>)")


def test_copy_make_border_replicate():
    img = refcases.frame(33, 21, 1)
    for x, y, w, h in [(-7, -4, 24, 24), (20, 10, 24, 24), (-3, 5, 40, 8), (5, -6, 8, 40)]:
        l, t = max(0, -x), max(0, -y)
        r, b = max(0, x + w - img.shape[1]), max(0, y + h - img.shape[0])
        inner = img[max(y, 0):min(y + h, img.shape[0]), max(x, 0):min(x + w, img.shape[1])]
        want = cv2.copyMakeBorder(inner, t, b, l, r, cv2.BORDER_REPLICATE)
        assert np.array_equal(ref.pad_roi(img, (x, y, w, h)), want)


def test_flip_and_rotate():
    t = refcases.frame(10, 10, 2)
    want = {0: t, 1: cv2.flip(t, 0), 2: cv2.flip(t, 1), 3: cv2.rotate(t, cv2.ROTATE_90_COUNTERCLOCKWISE), 4: cv2.rotate(t, cv2.ROTATE_180),
            5: cv2.rotate(t, cv2.ROTATE_90_CLOCKWISE), 6: cv2.rotate(cv2.flip(t, 0), cv2.ROTATE_90_COUNTERCLOCKWISE),
            7: cv2.rotate(cv2.flip(t, 1), cv2.ROTATE_90_COUNTERCLOCKWISE)}
    for k in range(8):
        assert np.array_equal(ref.apply_augmentation(t, k), want[k]), k


def test_multiply_f32():
    rng = np.random.default_rng(3)
    size, ov = 16, 4
    t = rng.uniform(-1, 2, size=(size, size, 3)).astype(np.float32)
    w = ref.create_tile_weights(ov, ov, size, size)
    got = ref.apply_weights(t, ov, ov, (5, 5, size, size), 100, 100)  # interior tile: left, top, right, bottom
    want = t
    for i in (3, 0, 1, 2):
        want = cv2.multiply(want, w[i])
    assert np.array_equal(got, want)


def test_split_and_convert_scale():
    tiles = np.stack([refcases.frame(8, 8, 4 + i) for i in range(2)])
    ref.set_pitch_align(1)
    try:
        blob = ref.blob_from_images(tiles)
    finally:
        ref.set_pitch_align(512)
    for i in range(2):
        for c, plane in enumerate(cv2.split(tiles[i])):
            want = plane.astype(np.float32) * np.float32(1.0 / 255.0)  # cv::cuda convertTo works in float: float(alpha) * src
            assert np.array_equal(blob[i, c], want)


def test_render_pack_rounds_half_to_even_and_saturates():
    """convertTo(CV_8UC3, 255) at the end of render(): saturate_cast<uchar>(float) == cvRound (half to even) + clamp."""
    vals = np.array([0.5, 1.5, 2.5, 3.5, 254.5, 255.5, 300.0, -3.0, 126.5, 127.5], np.float32) / np.float32(255.0)
    tile = np.zeros((1, 56, 56, 3), np.float16)
    exact = vals.astype(np.float16).astype(np.float32)  # the values the mock sees
    tile[0, 0, :len(vals), 0] = exact
    out = ref.render(np.zeros((20, 20, 3), np.uint8), refcases.replay_model(tile, 56), 64, 56, 2, 1 / 16, batch=1)
    want = cv2.multiply(exact.reshape(1, -1), np.float64(255.0), dtype=cv2.CV_8U).ravel()  # real OpenCV saturate_cast
    assert np.array_equal(out[0, :len(vals), 2], want)  # R channel of the tile lands in BGR index 2
