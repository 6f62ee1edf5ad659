"""CPU: oracle/vitpose_oracle.py against the reference outputs committed in tests/golden/
(made by oracle/make_golden.py from the unmodified reference).  This is what pins the oracle."""
import os

import numpy as np
import pytest

from oracle import golden_io, vitpose_oracle as O

FWD = ["s_coco", "b_coco", "l_coco_25", "h_wholebody"]


def _load(golden_dir, name):
    return golden_io.load(os.path.join(golden_dir, name + ".npz"))


@pytest.mark.parametrize("name", FWD)
def test_forward_matches_reference_heatmaps(golden_dir, name):
    g = _load(golden_dir, "fwd_" + name)
    D, depth, heads, K, B, wseed, xseed = (int(v) for v in g["meta"])
    sd = O.make_state_dict(D, depth, K, wseed, peaky=float(g["peaky"]), bumps=True)
    hm = O.forward_heatmaps(O.make_crops(B, xseed), sd, depth, heads)
    ref = g["heatmaps"]
    assert hm.shape == ref.shape == (B, K, O.HM_H, O.HM_W)
    # fp32 on both sides, different GEMM blocking: 1e-4 of a +-13 range
    assert np.abs(hm - ref).max() < 2e-4 * np.abs(ref).max()
    assert np.array_equal(hm.reshape(B, K, -1).argmax(-1), ref.reshape(B, K, -1).argmax(-1))


@pytest.mark.parametrize("name", FWD)
def test_decode_of_reference_heatmaps(golden_dir, name):
    g = _load(golden_dir, "fwd_" + name)
    kp, idx = O.decode_maps(g["heatmaps"], g["org_wh"], wrap="crop")
    assert np.array_equal(kp[..., 2], g["kpts"][..., 2])          # score = raw max, exact
    # the blur is bit-exact vs cv2; only np.log's SIMD path can differ between hosts
    assert np.abs(kp[..., :2] - g["kpts"][..., :2]).max() < 2e-3


@pytest.mark.parametrize("name,wrap", [("decode_crop", "crop"), ("decode_batch", "batch")])
def test_decode_edge_cases(golden_dir, name, wrap):
    g = _load(golden_dir, name)
    N, K, seed = (int(v) for v in g["meta"])
    maps = O.make_decode_maps(N, K, seed)
    kp, idx = O.decode_maps(maps, g["org_wh"], wrap=wrap)
    assert np.array_equal(idx, g["idx"])                            # integer argmax: bit-exact
    assert np.array_equal(kp[..., 2], g["kpts"][..., 2])
    ref = g["kpts"][..., :2]
    err = np.abs(kp[..., :2] - ref)
    kinds = (np.arange(N * K) % 10).reshape(N, K)
    well = np.isin(kinds, [0, 1, 2, 3, 5, 7])                       # real peaks: tight
    assert err[well].max() < 1e-3
    # sentinel / flat / noise maps have (near-)singular Hessians: relative agreement
    assert np.all(err[~well] <= 1e-3 + 1e-3 * np.abs(ref[~well]))


def test_reference_postprocess_matches_oracle(golden_dir):
    """VitInference.postprocess of the unmodified reference, one crop per call (oracle/make_golden_ref_calls.py)."""
    g = _load(golden_dir, "decode_postprocess")
    N, K, seed = (int(v) for v in g["meta"])
    maps = O.make_decode_maps(N, K, seed)
    for i in range(N):
        ref = g["kpts"][i]
        kp, _ = O.decode_maps(maps[i:i + 1], g["org_wh"][i:i + 1], wrap="crop")
        assert np.array_equal(kp[..., 2], ref[..., 2])
        assert np.abs(kp - ref).max() < 1e-3 + 1e-3 * np.abs(ref).max()


@pytest.mark.parametrize("name", ["s_coco", "b_coco"])
def test_torch_restatement_matches_reference(golden_dir, name):
    """oracle/torch_ref.py (the torch-ops restatement bench.py times as the CPU / torch-CUDA baselines) against the
    reference outputs: same library ops as the reference modules -> agreement to fp32 round-off."""
    import torch

    from oracle import torch_ref as T
    g = _load(golden_dir, "fwd_" + name)
    D, depth, heads, K, B, wseed, xseed = (int(v) for v in g["meta"])
    sd = T.to_device(O.make_state_dict(D, depth, K, wseed, peaky=float(g["peaky"]), bumps=True), "cpu", torch.float32)
    with torch.no_grad():
        hm = T.forward(torch.from_numpy(O.make_crops(B, xseed)), sd, depth, heads).numpy()
    assert np.abs(hm - g["heatmaps"]).max() < 1e-5 * np.abs(g["heatmaps"]).max()


def test_outlier_fixture_pins_the_oracle_too(golden_dir):
    """Real-ViT-like outliers (residual channels at +-100, pre-GELU +-13 / +-26; oracle.add_outliers): the oracle follows the
    reference there as well, and the fixture really contains what it claims."""
    g = _load(golden_dir, "outlier_b_coco")
    D, depth, heads, K, B, wseed, xseed, oseed = (int(v) for v in g["meta"])
    sd = O.add_outliers(O.make_state_dict(D, depth, K, wseed, peaky=0.1, bumps=True), oseed)
    tok_outliers = np.abs(sd["backbone.pos_embed"][0, 1:]).max(0)
    assert int((tok_outliers > 70).sum()) >= 4                    # four stream channels beyond +-70 on every token
    assert float(np.abs(sd["backbone.blocks.3.mlp.fc1.bias"]).max()) >= 25.0
    hm = O.forward_heatmaps(O.make_crops(B, xseed), sd, depth, heads)
    ref = g["heatmaps"]
    assert np.abs(hm - ref).max() < 5e-4 * (ref.max() - ref.min())
    assert np.array_equal(hm.reshape(B, K, -1).argmax(-1), g["idx"])


@pytest.mark.parametrize("name", ["batch_b_coco_64", "batch_h_wholebody_32", "batch_l_coco_25_64"])
def test_batch_fixtures_are_self_consistent(golden_dir, name):
    """The batch-size fixtures store reference keypoints for every crop but heatmaps only for a sample: the oracle's decode of
    the sampled reference maps must reproduce the stored keypoints of those crops / keypoints (scores exactly)."""
    g = _load(golden_dir, name)
    hm = g["sample_hm"]                                              # [4 crops, 8 keypoints, 64, 48]
    org = g["org_wh"][g["crop_ids"]]
    kp, idx = O.decode_maps(hm, org, wrap="crop")
    ref = g["kpts"][g["crop_ids"]][:, g["kp_ids"]]
    assert np.array_equal(idx, g["idx"][g["crop_ids"]][:, g["kp_ids"]])
    assert np.array_equal(kp[..., 2], ref[..., 2])
    # the reference decodes a crop's K maps in one call; a sentinel map (max <= 0) reads its neighbour map there, so compare
    # coordinates only where the map has a real peak
    ok = ref[..., 2] > 0.05
    assert np.abs(kp[..., :2] - ref[..., :2])[ok].max() < 2e-3 * max(1.0, float(org.max()) / 48.0)
