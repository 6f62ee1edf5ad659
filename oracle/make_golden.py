"""Generate tests/golden/*.npz from the UNMODIFIED reference  --  TEST INFRASTRUCTURE ONLY.

Run here (the container that has /root/reference):   python oracle/make_golden.py
Only some cases:   python oracle/make_golden.py h_wholebody decode_crop
The reference is a Python package and cannot travel to the GPU box, so its outputs on seeded
inputs are committed as small fixtures.  Inputs and weights are NOT stored: both sides
regenerate them from the seeds with oracle.vitpose_oracle.make_state_dict / make_crops /
make_decode_maps (np.random.RandomState is a frozen stream).

What is pinned:
  fwd_<size>_<dataset>.npz  reference ViTPose(cfg).forward heatmaps (vit_models/model.py:23-24)
                            + VitInference.postprocess keypoints (easy_ViTPose/inference.py:187-205);
                            heatmaps too large for one file below 1 MB continue in fwd_<...>.part<i>.npz (oracle/golden_io.py)
  decode_crop.npz           keypoints_from_heatmaps called per crop (N=1), as VitInference does
  decode_batch.npz          keypoints_from_heatmaps called once on an [N,K,H,W] batch
  blur_check                asserted here: oracle blur == cv2.GaussianBlur bit for bit
"""
from __future__ import annotations

import os
import sys
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import golden_io, ref_import, vitpose_oracle as O  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")

# name -> (size letter, dataset module, K, batch, weight seed, crop seed, org_wh per crop, peaky)
FORWARD_CASES = {
    "s_coco": ("s", "coco", 17, 1, 101, 201, [(192, 256)], 0.1),
    "b_coco": ("b", "coco", 17, 2, 102, 202, [(192, 256), (151, 211)], 0.1),
    "l_coco_25": ("l", "coco_25", 25, 1, 103, 203, [(96, 128)], 0.1),
    "h_wholebody": ("h", "wholebody", 133, 1, 104, 204, [(333, 444)], 0.1),
}
DECODE_CASES = {"decode_crop": (6, 17, 301), "decode_batch": (3, 25, 302)}


def main(only: list[str]) -> None:
    import cv2
    import torch
    torch.set_grad_enabled(False)
    ns = ref_import.load()
    os.makedirs(OUT, exist_ok=True)

    # blur order check: the oracle's point-wise blur against cv2 on every pixel of a few maps
    taps = O.gaussian_taps(11)
    assert np.array_equal(taps, cv2.getGaussianKernel(11, 0).astype(np.float32).ravel())
    maps = O.make_decode_maps(1, 10, 7)[0]
    ys, xs = np.mgrid[0:O.HM_H, 0:O.HM_W]
    for m in maps:
        g = cv2.GaussianBlur(m.copy(), (11, 11), 0)
        mine = O.blur_at(m, xs.ravel(), ys.ravel(), taps).reshape(O.HM_H, O.HM_W)
        assert np.array_equal(g, mine), float(np.abs(g - mine).max())
    print("blur order: bit-exact vs cv2", cv2.__version__)

    for name, (size, dataset, K, B, wseed, xseed, org, peaky) in FORWARD_CASES.items():
        if only and name not in only:
            continue
        D, depth, heads = O.MODEL_DIMS[size]
        cfg = ns.dyn_model_import(dataset, size)
        model = ns.ViTPose(cfg).eval()
        sd = O.make_state_dict(D, depth, K, wseed, peaky=peaky, bumps=True)
        model.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}, strict=True)
        x = O.make_crops(B, xseed)
        hm = model(torch.from_numpy(x)).numpy().astype(np.float32)
        org_wh = np.array(org, np.int32)
        kp = np.concatenate([ref_import.postprocess(ns, hm[i:i + 1], int(org_wh[i, 0]), int(org_wh[i, 1]))
                             for i in range(B)], 0).astype(np.float32)
        golden_io.save(os.path.join(OUT, f"fwd_{name}.npz"), dict(heatmaps=hm, kpts=kp, org_wh=org_wh,
                       meta=np.array([D, depth, heads, K, B, wseed, xseed], np.int64), peaky=np.float64(peaky)), split_key="heatmaps")
        print(name, "heatmap range", float(hm.min()), float(hm.max()),
              "positive maxima", int((hm.reshape(B, K, -1).max(-1) > 0).sum()), "/", B * K)

    for name, (N, K, seed) in DECODE_CASES.items():
        if only and name not in only:
            continue
        maps = O.make_decode_maps(N, K, seed)
        rs = np.random.RandomState(seed + 1)
        org_wh = np.stack([rs.randint(64, 513, size=N), rs.randint(64, 513, size=N)], 1).astype(np.int32)
        if name == "decode_crop":
            kp = np.concatenate([ref_import.postprocess(ns, maps[i:i + 1], int(org_wh[i, 0]), int(org_wh[i, 1]))
                                 for i in range(N)], 0)
        else:
            # one call on the whole batch with per-crop centre/scale (what keypoints_from_heatmaps supports)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore", DeprecationWarning)
                pts, prob = ns.keypoints_from_heatmaps(
                    heatmaps=maps, center=np.stack([org_wh[:, 0] // 2, org_wh[:, 1] // 2], 1),
                    scale=org_wh.astype(np.int64), unbiased=True, use_udp=True)
            kp = np.concatenate([pts[:, :, ::-1], prob], 2)
        idx = np.argmax(maps.reshape(N, K, -1), -1).astype(np.int32)
        np.savez_compressed(os.path.join(OUT, f"{name}.npz"), kpts=kp.astype(np.float32), idx=idx,
                            org_wh=org_wh, meta=np.array([N, K, seed], np.int64))
        print(name, "written")


if __name__ == "__main__":
    main(sys.argv[1:])
