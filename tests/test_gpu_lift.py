"""GPU: the step upstream of the path (SURVEY.md §8f-2) - ResNetBlock_3D(32->16) as one cluster launch
(`ahv_resblock3d`), `Feature_Aligner.forward_2d3d` using it, and the whole post-backbone tail under one CUDA graph."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)


def test_resblock3d_vs_reference_fixture(ahv, golden_lift, oracle):
    g = golden_lift
    T = lambda a: torch.from_numpy(a).to(DEV)
    out = ahv.ops.resblock3d(T(g["x"]), T(g["conv1_w"]), T(g["conv2_w"]), T(g["down_w"])).cpu().numpy()
    np.testing.assert_allclose(out, g["out"], atol=3e-6, rtol=0)          # the reference's own module, fp32 CPU
    # ragged batch sizes against the restatement (clusters of 8 CTAs per volume, one CTA per SM: 1, 2 and one more
    # volume than there are resident clusters)
    gen = torch.Generator().manual_seed(1)
    resident = max(torch.cuda.get_device_properties(DEV).multi_processor_count // 8, 1)
    for m in (1, 2, resident + 1):
        x = torch.randn(m, 32, 8, 8, 8, generator=gen)
        want = oracle.resblock3d_np(x.numpy(), g["conv1_w"], g["conv2_w"], g["down_w"])
        got = ahv.ops.resblock3d(x.to(DEV), T(g["conv1_w"]), T(g["conv2_w"]), T(g["down_w"])).cpu().numpy()
        np.testing.assert_allclose(got, want, atol=1e-5, rtol=0)


def test_forward_2d3d_uses_the_kernel_and_matches_pytorch(ahv):
    from modules.modules import Feature_Aligner, _ResNetBlock

    torch.manual_seed(0)
    fa = Feature_Aligner(768, 256, 32, 4, 2).to(DEV).eval()
    a, b = torch.randn(3, 768, 8, 8, device=DEV), torch.randn(3, 768, 8, 8, device=DEV)
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False                              # cuDNN convolutions in fp32 for the comparison
    try:
        with torch.no_grad():
            vs, vt = fa.forward_2d3d(a, b, random_mask=False, mask_ratio=0.0)      # 3D block: ahv_resblock3d
            blk = fa.feature_embedding_3d
            x = torch.randn(4, 32, 8, 8, 8, device=DEV)
            fused, eager = blk(x), _ResNetBlock.forward(blk, x)
        assert vs.shape == vt.shape == (3, 16, 8, 8, 8)
        assert torch.allclose(fused, eager, atol=2e-5, rtol=0)
        # under autograd the block stays differentiable PyTorch
        xg = x.clone().requires_grad_(True)
        assert blk(xg).requires_grad
    finally:
        torch.backends.cudnn.allow_tf32 = tf32


def test_graphed_tail_equals_eager(ahv):
    from modules.modules import Feature_Aligner

    torch.manual_seed(1)
    fa = Feature_Aligner(768, 256, 32, 4, 2).to(DEV).eval()
    B, N = 2, 1000
    gt = ahv.GraphedTail(fa, B, N, k=4, device=DEV)
    for seed in (0, 1):
        g = torch.Generator().manual_seed(seed)
        a, b = torch.randn(B, 768, 8, 8, generator=g).to(DEV), torch.randn(B, 768, 8, 8, generator=g).to(DEV)
        R = ahv.so3.sample_rotations(N, seed=seed, device=DEV)
        out = gt(a, b, R)
        with torch.no_grad():
            vs, vt = fa.forward_2d3d(a, b, random_mask=False, mask_ratio=0.0)
            ref = ahv.HypothesisVerifier.from_feature_aligner(fa).score(vs, vt, R, k=4, return_scores=False)
        assert torch.equal(out.topk_idx, ref.topk_idx) and torch.equal(out.topk_val, ref.topk_val)
        assert torch.equal(out.R_best, ref.R_best) and torch.equal(gt.vol_src, vs)
