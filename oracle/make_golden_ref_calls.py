"""Generate tests/golden/{decode_postprocess,pad_pre_img,resize_cv2}.npz from the UNMODIFIED reference  --  TEST INFRASTRUCTURE ONLY.

Run where the reference is importable (oracle/ref_import.py):   python oracle/make_golden_ref_calls.py

What is pinned (inputs regenerate from seeds on both sides; only the reference's answers are stored):
  decode_postprocess.npz  VitInference.postprocess (easy_ViTPose/inference.py:187-205) on make_decode_maps(2, 17, 999),
                          one crop per call with org (200 + i, 300 + i): the keypoints [2, 1, 17, 3] it returns
  pad_pre_img.npz         pad_image + VitInference.pre_img (inference.py:259-265, 314-318) on 12 seeded boxes of
                          make_frame(200, 260, 5): the boxes, pad offsets, org sizes, and SHA-256 digests of the padded
                          uint8 canvas and of the float32 network input (the full arrays would not fit a small fixture).
                          The +-10 px pad and clip in front of pad_image is written inline in VitInference.inference
                          (:259-261), so the crop handed to pad_image is cut with the oracle's padded_box; that step is
                          pinned by test_padded_box_clips_to_frame and end to end by the frame_*.npz fixtures.
  resize_cv2.npz          cv2.resize(img, (192, 256), INTER_LINEAR) as pre_img calls it, on the 30 seeded uint8 images of
                          test_resize_matches_cv2_on_random_sizes: their sizes and SHA-256 digests of the outputs
"""
from __future__ import annotations

import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import preproc_oracle as P, ref_import, vitpose_oracle as O  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
DECODE = (2, 17, 999)
FRAME = (200, 260, 5)
BOX_SEED, BOX_DRAWS = 2, 12


def sha256(a: np.ndarray) -> np.ndarray:
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), np.uint8)


def seeded_boxes():
    """The boxes test_preproc_oracle.py draws: RandomState(2), 12 draws, those left empty by the +-10 px pad and clip skipped."""
    fh, fw, _ = FRAME
    rs = np.random.RandomState(BOX_SEED)
    for _ in range(BOX_DRAWS):
        x0, y0 = rs.randint(-20, 240), rs.randint(-20, 180)
        box = np.array([x0, y0, x0 + rs.randint(1, 150), y0 + rs.randint(1, 150)])
        bx0, by0, bx1, by1 = P.padded_box(box, fh, fw)
        if bx1 > bx0 and by1 > by0:
            yield box, (bx0, by0, bx1, by1)


def main() -> None:
    ns = ref_import.load()
    inf = ref_import.load_vitinference()
    os.makedirs(OUT, exist_ok=True)

    N, K, seed = DECODE
    maps = O.make_decode_maps(N, K, seed)
    org_wh = np.array([[200 + i, 300 + i] for i in range(N)], np.int64)
    kp = np.stack([ref_import.postprocess(ns, maps[i:i + 1], int(org_wh[i, 0]), int(org_wh[i, 1])) for i in range(N)], 0)
    np.savez_compressed(os.path.join(OUT, "decode_postprocess.npz"), kpts=kp, org_wh=org_wh, meta=np.array(DECODE, np.int64))
    print("decode_postprocess", kp.shape, kp.dtype)

    frame = P.make_frame(*FRAME)
    stub = type("S", (), {"target_size": (192, 256)})()
    rows = {k: [] for k in ("boxes", "left_top", "org_hw", "canvas_shape", "canvas_sha256", "x_shape", "x_sha256")}
    for box, (bx0, by0, bx1, by1) in seeded_boxes():
        padded, (left, top) = inf.pad_image(frame[by0:by1, bx0:bx1], 3 / 4)
        x, org_h, org_w = inf.VitInference.pre_img(stub, padded)
        assert padded.dtype == np.uint8 and x.dtype == np.float32
        # the oracle must agree before the answers are stored
        canvas, off = P.crop_canvas(frame, box)
        assert np.array_equal(canvas, padded) and off == (by0 - top, bx0 - left)
        assert np.array_equal(P.pre_img(canvas), x)
        for k, v in (("boxes", box), ("left_top", (left, top)), ("org_hw", (org_h, org_w)), ("canvas_shape", padded.shape),
                     ("canvas_sha256", sha256(padded)), ("x_shape", x.shape), ("x_sha256", sha256(x))):
            rows[k].append(np.asarray(v))
    out = {k: np.stack(v, 0).astype(np.uint8 if k.endswith("sha256") else np.int64) for k, v in rows.items()}
    np.savez_compressed(os.path.join(OUT, "pad_pre_img.npz"), meta=np.array([*FRAME, BOX_SEED, BOX_DRAWS], np.int64), **out)
    print("pad_pre_img", len(out["boxes"]), "boxes")

    import cv2
    rs = np.random.RandomState(0)
    sizes = [(rs.randint(1, 700), rs.randint(1, 600)) for _ in range(25)] + [(256, 192), (512, 384), (1, 1), (2, 3), (1080, 810)]
    digests = []
    for h, w in sizes:
        img = rs.randint(0, 256, size=(h, w, 3), dtype=np.uint8)
        r = cv2.resize(img, (192, 256), interpolation=cv2.INTER_LINEAR)
        assert r.dtype == np.uint8 and r.shape == (256, 192, 3) and np.array_equal(P.resize_linear_u8(img), r)
        digests.append(sha256(r))
    np.savez_compressed(os.path.join(OUT, "resize_cv2.npz"), sizes=np.array(sizes, np.int64), sha256=np.stack(digests, 0))
    print("resize_cv2", len(sizes), "images, cv2", cv2.__version__)


if __name__ == "__main__":
    main()
