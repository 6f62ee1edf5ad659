"""CPU: the C-ABI library loads and exports every symbol include/vitpose_b200.h declares; host-side
mirror of the reference interface behaves (no GPU compute here)."""
import ctypes
import os
import re
import subprocess
import sys
import textwrap

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from easy_vitpose_b200 import _lib
    from easy_vitpose_b200.build import LIB, build
    build()
    hdr = open(os.path.join(ROOT, "include", "vitpose_b200.h")).read()
    declared = set(re.findall(r"\b(vpb_[a-z_]+)\s*\(", hdr))
    assert declared, "header declares nothing?"
    lib = ctypes.CDLL(LIB)
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    _lib.lib()


def test_no_cpu_fallback_without_gpu():
    """Runs in a child process with every GPU hidden (CUDA_VISIBLE_DEVICES=""), so a machine with a GPU checks it too."""
    code = textwrap.dedent("""
        import torch
        assert not torch.cuda.is_available()
        from easy_vitpose_b200 import ViTPose, decode_heatmaps, model_cfg
        m = ViTPose(model_cfg("b", 17))
        for call in (lambda: m.to("cpu"), lambda: decode_heatmaps(torch.zeros(1, 17, 64, 48), torch.tensor([[192, 256]]))):
            try:
                call()
            except RuntimeError:
                continue
            raise AssertionError("no RuntimeError without a GPU")
        print("raised")
    """)
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and out.stdout.split() == ["raised"], out.stdout + out.stderr[-2000:]


def test_configs_match_reference_shapes():
    from easy_vitpose_b200 import dyn_model_import
    from easy_vitpose_b200.model import _expected_shapes
    from oracle import vitpose_oracle as O
    for size, ds, K in [("s", "coco", 17), ("b", "ap10k", 17), ("l", "coco_25", 25), ("h", "wholebody", 133)]:
        cfg = dyn_model_import(ds, size)
        D, depth, heads = O.MODEL_DIMS[size]
        assert (cfg["backbone"]["embed_dim"], cfg["backbone"]["depth"], cfg["backbone"]["num_heads"]) == (D, depth, heads)
        assert cfg["keypoint_head"]["out_channels"] == K
        sd = O.make_state_dict(D, 1, K, 0)
        exp = _expected_shapes(D, 1, K)
        assert set(sd) == set(exp)
        for k in sd:
            assert tuple(np.asarray(sd[k]).shape) == tuple(exp[k]), k


def test_state_dict_contract_is_strict():
    import torch
    from easy_vitpose_b200 import ViTPose, model_cfg
    from oracle import vitpose_oracle as O
    m = ViTPose(model_cfg("s", 17))
    sd = {k: torch.from_numpy(np.asarray(v)) for k, v in O.make_state_dict(384, 12, 17, 0).items()}
    extra = dict(sd); extra["backbone.cls_token"] = torch.zeros(1)
    with pytest.raises(RuntimeError):
        m.load_state_dict(extra)
    wrong = dict(sd); wrong["backbone.pos_embed"] = torch.zeros(1, 197, 384)
    with pytest.raises(RuntimeError):
        m.load_state_dict(wrong)
    m.load_state_dict({"state_dict": sd})                     # both checkpoint layouts (inference.py:162-166)
    out = m.state_dict()
    assert set(out) == set(sd) and torch.equal(out["backbone.pos_embed"], sd["backbone.pos_embed"])


def test_synthetic_weights_follow_the_state_dict_contract():
    """easy_vitpose_b200.synthetic (what bench.py's GPU arm loads: it must not import oracle/) produces exactly the reference's
    state_dict keys and shapes (SURVEY.md section 8b), and a strict load accepts them without a GPU."""
    import numpy as np
    import torch

    from easy_vitpose_b200 import ViTPose, model_cfg
    from easy_vitpose_b200.synthetic import random_crops, random_state_dict
    from oracle import vitpose_oracle as O
    for size, K in (("s", 17), ("b", 25)):
        D, depth, heads = O.MODEL_DIMS[size]
        mine = random_state_dict(size, K, seed=3)
        ref = {k: v.shape for k, v in O.make_state_dict(D, depth, K, 3).items() if not k.endswith("num_batches_tracked")}
        assert {k: v.shape for k, v in mine.items()} == ref
        assert all(v.dtype == np.float32 for v in mine.values())
        ViTPose(model_cfg(size, K)).load_state_dict({k: torch.from_numpy(v) for k, v in mine.items()})      # strict, CPU side only
    assert random_crops(2, 1).shape == (2, 3, 256, 192) and np.array_equal(random_crops(2, 1), random_crops(2, 1))


def test_decode_api_fails_loudly_without_cuda_and_checks_its_config():
    """No CPU fallback anywhere on the product path: decode entry points refuse CPU tensors; the reference's config conflicts
    (vit_utils/top_down_eval.py:548-553) and the combinations that are not built raise before any device work."""
    import numpy as np
    import pytest
    import torch

    from easy_vitpose_b200 import decode_heatmaps, keypoints_from_heatmaps
    hm = np.zeros((1, 17, 64, 48), np.float32)
    c = np.array([[96, 128]]); s = np.array([[192, 256]])
    with pytest.raises(RuntimeError):
        decode_heatmaps(torch.zeros(1, 17, 64, 48), torch.tensor([[192, 256]]))
    with pytest.raises(AssertionError):
        keypoints_from_heatmaps(hm, c, s, post_process="megvii", use_udp=True)
    with pytest.raises(AssertionError):
        keypoints_from_heatmaps(hm, c, s, unbiased=True, post_process="megvii")
    with pytest.raises(ValueError):                                   # 17 maps are not triples (reference: reshape fails, :590)
        keypoints_from_heatmaps(hm, c, s, use_udp=True, target_type="CombinedTarget")
    with pytest.raises(ValueError):                                   # N > 1: the reference's index arithmetic does not broadcast (:589)
        keypoints_from_heatmaps(np.zeros((2, 18, 64, 48), np.float32), np.tile(c, (2, 1)), np.tile(s, (2, 1)), use_udp=True,
                                target_type="CombinedTarget")
    with pytest.raises(ValueError):
        keypoints_from_heatmaps(hm, c, s, use_udp=True, target_type="nonsense")
    with pytest.raises(NotImplementedError):                          # even / oversized modulation kernels
        keypoints_from_heatmaps(hm, c, s, post_process="unbiased", kernel=8)
    with pytest.raises(NotImplementedError):
        keypoints_from_heatmaps(hm, c, s, post_process="megvii", kernel=37)
    with pytest.raises(ValueError):                                   # kernel = 1: the reference's _gaussian_blur raises (zero-width border)
        keypoints_from_heatmaps(hm, c, s, post_process="unbiased", kernel=1)
    with pytest.raises(NotImplementedError):                          # CombinedTarget blurs with 2 * kernel + 1 <= 35
        keypoints_from_heatmaps(hm[:, :15], c, s, use_udp=True, kernel=19, target_type="CombinedTarget")
    with pytest.raises(ValueError):
        keypoints_from_heatmaps(hm, c, s, post_process="fancy")
