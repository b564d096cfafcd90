"""CPU: the drop-in model keeps the reference's API and state-dict names."""
import json
import os

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_feature_aligner_state_dict_matches_reference_names():
    from modules.modules import Feature_Aligner

    want = json.load(open(os.path.join(ROOT, "tests", "golden", "feature_aligner_state_dict.json")))
    fa = Feature_Aligner(in_channel=768, mid_channel=256, out_channel=32, n_heads=4, depth=4)
    got = {k: list(v.shape) for k, v in fa.state_dict().items()}
    assert got == want
    for k in ("feature_embedding_2d.0.weight", "feature_embedding_2d.2.weight", "feature_embedding_2d.2.bias"):
        assert k in got


def test_forward_2d3d_shapes_and_determinism():
    from modules.modules import Feature_Aligner

    torch.manual_seed(0)
    fa = Feature_Aligner(768, 256, 32, 4, 4).eval()
    with torch.no_grad():
        a, b = torch.randn(2, 768, 8, 8), torch.randn(2, 768, 8, 8)
        s1, t1 = fa.forward_2d3d(a, b, random_mask=False, mask_ratio=0.0)
        s2, t2 = fa.forward_2d3d(a, b, random_mask=False, mask_ratio=0.0)
    assert s1.shape == t1.shape == (2, 16, 8, 8, 8)
    assert torch.equal(s1, s2) and torch.equal(t1, t2)


def test_forward_2d3d_matches_reference_module(golden):
    """Same initialisation -> same volumes as the reference's own Feature_Aligner.  oracle/make_golden.py built the
    reference's Feature_Aligner(768, 256, 32, 4, 4) under seed 0, stored its head weights in weights.npz and the
    volumes its forward_2d3d made from two seeded [3, 768, 8, 8] inputs in shared_n3000_b3.npz; the same recipe is
    rerun here on this implementation."""
    from modules.modules import Feature_Aligner

    torch.manual_seed(0)
    fa = Feature_Aligner(in_channel=768, mid_channel=256, out_channel=32, n_heads=4, depth=4).eval()
    sd, w = fa.state_dict(), golden["weights"]
    assert np.array_equal(sd["feature_embedding_2d.0.weight"].reshape(32, 384).numpy(), w["W1"])
    assert np.array_equal(sd["feature_embedding_2d.2.weight"].reshape(32, 32).numpy(), w["W2"])
    assert np.array_equal(sd["feature_embedding_2d.2.bias"].numpy(), w["b2"])
    with torch.no_grad():
        src, tgt = fa.forward_2d3d(torch.randn(3, 768, 8, 8), torch.randn(3, 768, 8, 8), random_mask=False, mask_ratio=0.0)
    g = golden["shared_n3000_b3"]
    err = max(float(np.abs(src.numpy() - g["vol_src"]).max()), float(np.abs(tgt.numpy() - g["vol_tgt"]).max()))
    assert err < 5e-5, err


class _TinyBackbone(torch.nn.Module):
    def forward(self, img):
        return torch.nn.functional.adaptive_avg_pool2d(img, 8).repeat(1, 256, 1, 1)


def _cfg():
    return {"DATA": {"NUM_ROTA": 64, "BG": False, "SIZE_THR": 10, "ACC_THR": 15}}


def test_estimator_api_surface():
    from modules.model import Estimator
    from modules.model_co3d import Estimator as EstimatorCo3d

    m = Estimator(_cfg(), feature_extractor=_TinyBackbone()).eval()
    for attr in ("cfg", "num_rota", "feature_extractor", "feature_aligner", "step_outputs", "gt_dis", "pred_Rs"):
        assert hasattr(m, attr)
    for fn in ("feature_extraction", "forward", "validation_step", "test_step", "training_step", "configure_optimizers",
               "infoNCE_loss", "predict"):
        assert callable(getattr(m, fn))
    img = torch.rand(2, 3, 64, 64)
    mask = torch.ones(2, 1, 64, 64)
    with torch.no_grad():
        vs, vt = m(img, mask, img, mask)
    assert vs.shape == vt.shape == (2, 16, 8, 8, 8)
    assert any(k.startswith("feature_aligner.feature_embedding_2d.0.weight") for k in m.state_dict())
    c = EstimatorCo3d(_cfg(), feature_extractor=_TinyBackbone()).eval()
    with torch.no_grad():
        vs, vt = c(img, img)
    assert vs.shape == (2, 16, 8, 8, 8) and c.mid_channel == 256
    # the hot path itself refuses to run without a GPU (no CPU fallback)
    with pytest.raises(RuntimeError):
        m.predict_rotation(vs, vt)


def test_named_backbone_architecture_shape():
    from modules._backbone import build_backbone

    bb = build_backbone().eval()
    n = sum(p.numel() for p in bb.parameters())
    assert 27e6 < n < 29e6                      # SwinV2-T
    with torch.no_grad():
        out = bb(torch.randn(1, 3, 256, 256))
    assert out.shape == (1, 768, 8, 8)


def test_reference_shaped_checkpoint_loads():
    """A checkpoint with the reference's key layout (feature_aligner.* + the MiDaS/timm wrapper's
    feature_extractor.pretrained.model.* + the unused DPT decoder feature_extractor.scratch.*) loads into the
    drop-in Estimator: aligner strictly by name, backbone through the timm -> torchvision mapping."""
    import re

    from modules._backbone import load_reference_state_dict
    from modules.model_co3d import Estimator

    torch.manual_seed(0)
    src = Estimator(_cfg()).eval()
    ref_sd = {"feature_aligner." + k: v.clone() for k, v in src.feature_aligner.state_dict().items()}
    for k, v in src.feature_extractor.model.state_dict().items():       # torchvision -> timm names (inverse mapping)
        m = re.match(r"features\.(\d)\.(.+)$", k)
        if not m:                                                        # final norm.*: same name in timm
            ref_sd["feature_extractor.pretrained.model." + k] = v.clone()
            continue
        i, rest = int(m.group(1)), m.group(2)
        if i == 0:
            name = ("patch_embed.proj." if rest.startswith("0.") else "patch_embed.norm.") + rest.split(".", 1)[1]
        elif i % 2 == 1:
            j, tail = rest.split(".", 1)
            tail = tail.replace("mlp.0.", "mlp.fc1.").replace("mlp.3.", "mlp.fc2.")
            if tail == "attn.qkv.bias":
                c = v.shape[0] // 3
                ref_sd[f"feature_extractor.pretrained.model.layers.{i // 2}.blocks.{j}.attn.q_bias"] = v[:c].clone()
                ref_sd[f"feature_extractor.pretrained.model.layers.{i // 2}.blocks.{j}.attn.v_bias"] = v[2 * c:].clone()
                continue
            name = f"layers.{i // 2}.blocks.{j}.{tail}"
        else:
            name = f"layers.{i // 2 - 1}.downsample.{rest}"
        ref_sd["feature_extractor.pretrained.model." + name] = v.clone()
    ref_sd["feature_extractor.scratch.output_conv.0.weight"] = torch.zeros(4, 4)       # DPT decoder: never executed
    torch.manual_seed(1)
    dst = Estimator(_cfg()).eval()
    rep = load_reference_state_dict(dst, {"state_dict": ref_sd})
    assert rep["skipped"] == ["feature_extractor.scratch.output_conv.0.weight"] and rep["backbone_missing"] == []
    img = torch.randn(1, 3, 256, 256)
    with torch.no_grad():
        a, b = src(img, img.flip(-1)), dst(img, img.flip(-1))
    # qkv.bias carries a k-bias in torchvision that timm does not have: the stand-in zeroes it at construction
    assert torch.allclose(a[0], b[0], atol=1e-5) and torch.allclose(a[1], b[1], atol=1e-5)
    # the call the reference's scripts make (test_co3d.py:218): Estimator.load_from_checkpoint(path, cfg=cfg)
    import os
    import tempfile

    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "checkpoint_co3d.ckpt")
        torch.save({"state_dict": ref_sd, "hyper_parameters": {"cfg": _cfg()}, "epoch": 3}, path)
        torch.manual_seed(2)
        loaded = Estimator.load_from_checkpoint(path, cfg=_cfg()).eval()
        assert loaded.load_report["backbone_missing"] == []
        with torch.no_grad():
            c = loaded(img, img.flip(-1))
        assert torch.allclose(a[0], c[0], atol=1e-5)
        assert Estimator.load_from_checkpoint(path).num_rota == _cfg()["DATA"]["NUM_ROTA"]    # cfg from hyper_parameters

