"""CPU: oracle/preproc_oracle.py (SURVEY.md section 8 row f1) against the fixtures the UNMODIFIED reference produced
(oracle/make_golden_frames.py, oracle/make_golden_ref_calls.py), including what cv2.resize returns."""
import hashlib
import os

import numpy as np
import pytest

from oracle import preproc_oracle as P


def _sha256(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), np.uint8)


def _case(golden_dir, name):
    g = np.load(os.path.join(golden_dir, f"{name}.npz"))
    fh, fw, fseed = (int(v) for v in g["meta"][:3])
    rows = g["rows"].astype(np.float64)
    boxes = rows[rows[:, 4] > 0.35, :4].round().astype(int)            # easy_ViTPose/inference.py:240,253
    return g, P.make_frame(fh, fw, fseed), boxes


@pytest.mark.parametrize("name", ["frame_a", "frame_b"])
def test_preprocess_matches_reference_fixture(golden_dir, name):
    g, frame, boxes = _case(golden_dir, name)
    crops, org_wh, offs = P.preprocess_frame(frame, boxes)
    assert np.array_equal(P.normalise_lut(), g["lut"])
    assert np.array_equal(org_wh, g["org_wh"]) and np.array_equal(offs, g["offs_yx"])
    for i in range(len(boxes)):
        canvas, _ = P.crop_canvas(frame, boxes[i])
        assert np.array_equal(P.resize_linear_u8(canvas), g["resized"][i])
        want = np.stack([g["lut"][c][g["resized"][i][..., c]] for c in range(3)], 0)
        assert np.array_equal(crops[i], want)


def test_pad_geometry_is_the_reference_rule():
    """pad_image decides with floats (w / h < 3 / 4, int(0.75 * h), int(w / 0.75)); the oracle with integers."""
    for w in range(1, 140):
        for h in range(1, 140):
            ar = w / h
            if ar < 3 / 4:
                tw = int(3 / 4 * h); want = (tw, h, (tw - w) // 2, 0)
            else:
                th = int(w / (3 / 4)); want = (w, th, 0, (th - h) // 2)
            assert P.pad_geometry(w, h) == want, (w, h)
    with pytest.raises(ValueError):
        P.pad_geometry(0, 5)


def test_padded_box_clips_to_frame():
    assert P.padded_box((5, 3, 50, 40), 100, 200) == (0, 0, 60, 50)
    assert P.padded_box((150, 80, 260, 130), 100, 200) == (140, 70, 200, 100)
    assert P.padded_box((300, 300, 310, 310), 100, 200) == (200, 100, 200, 100)      # empty: the reference raises later


def test_resize_matches_cv2_on_random_sizes(golden_dir):
    """cv2.resize(img, (192, 256), INTER_LINEAR) outputs, pinned by their SHA-256 digests (tests/golden/resize_cv2.npz)."""
    g = np.load(os.path.join(golden_dir, "resize_cv2.npz"))
    rs = np.random.RandomState(0)
    sizes = [(rs.randint(1, 700), rs.randint(1, 600)) for _ in range(25)] + [(256, 192), (512, 384), (1, 1), (2, 3), (1080, 810)]
    assert np.array_equal(np.array(sizes), g["sizes"])
    for (h, w), want in zip(sizes, g["sha256"]):
        img = rs.randint(0, 256, size=(h, w, 3), dtype=np.uint8)
        r = P.resize_linear_u8(img)
        assert r.dtype == np.uint8 and r.shape == (256, 192, 3) and np.array_equal(_sha256(r), want), (h, w)


def test_to_frame_coords_is_one_rounding():
    rs = np.random.RandomState(1)
    kp = (rs.rand(4, 17, 3) * 400).astype(np.float32)
    offs = rs.randint(-50, 2000, size=(4, 2)).astype(np.int32)
    out = P.to_frame_coords(kp, offs)
    assert np.array_equal(out[..., :2], kp[..., :2] + offs[:, None, :].astype(np.float32))     # float32 add == f64 add then cast
    assert np.array_equal(out[..., 2], kp[..., 2])


def test_against_reference_pad_image_and_pre_img(golden_dir):
    """The reference's pad_image and VitInference.pre_img on seeded boxes (oracle/make_golden_ref_calls.py): canvas and
    network input are pinned bit for bit through their SHA-256 digests."""
    g = np.load(os.path.join(golden_dir, "pad_pre_img.npz"))
    fh, fw, fseed = (int(v) for v in g["meta"][:3])
    frame = P.make_frame(fh, fw, fseed)
    assert len(g["boxes"]) == 12
    for n, box in enumerate(g["boxes"]):
        bx0, by0, _, _ = P.padded_box(box, fh, fw)
        left, top = (int(v) for v in g["left_top"][n])
        canvas, off = P.crop_canvas(frame, box)
        assert canvas.shape == tuple(g["canvas_shape"][n]) and np.array_equal(_sha256(canvas), g["canvas_sha256"][n])
        assert off == (by0 - top, bx0 - left)
        x = P.pre_img(canvas)
        assert x.dtype == np.float32 and x.shape == tuple(g["x_shape"][n]) and np.array_equal(_sha256(x), g["x_sha256"][n])
        assert tuple(g["org_hw"][n]) == canvas.shape[:2]
