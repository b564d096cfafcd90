"""GPU: `ahv_resblock3d` (ResNetBlock_3D 32->16 on 8^3, one cluster of 8 CTAs per volume, persistent over volumes)
against F.conv3d in float64 on the CPU, and the identities its fp32 FFMA chain must keep bit for bit.

Gate: |out - ref| <= C * 2^-24 * A, where A is the same chain on |x| and |W|, |W2| * (|W1| * |x|) + |Wd| * |x|: the
bound on every product the kernel rounds.  Where A = 0 (outside an impulse's reach, a zero volume) the output must
be exactly 0.  `_check` prints the largest err / (2^-24 A) of each case.  On an NVIDIA B200 (1000 W) the largest
over this module is 1.33 (the impulses; 0.02-0.35 elsewhere).  C = 4 leaves room for rounding that accumulates
coherently, while a wrong tap, channel or neighbour slab is off by O(A), millions of times the gate."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
C = 4.0
U = 2.0 ** -24


def _weights(seed, scale1=0.06, scale2=0.08, scaled=0.15, mean1=0.0):
    g = torch.Generator().manual_seed(seed)
    w1 = torch.randn(16, 32, 3, 3, 3, generator=g) * scale1 + mean1
    w2 = torch.randn(16, 16, 3, 3, 3, generator=g) * scale2
    wd = torch.randn(16, 32, 1, 1, 1, generator=g) * scaled
    return w1, w2, wd


def reference(x, w1, w2, wd):
    """fp64 output and the error scale A, on the CPU."""
    x, w1, w2, wd = (t.detach().cpu().double() for t in (x, w1, w2, wd))
    out = F.conv3d(F.relu(F.conv3d(x, w1, padding=1)), w2, padding=1) + F.conv3d(x, wd)
    a = F.conv3d(F.conv3d(x.abs(), w1.abs(), padding=1), w2.abs(), padding=1) + F.conv3d(x.abs(), wd.abs())
    return out, a


def _kernel(ahv, x, w1, w2, wd):
    return ahv.ops.resblock3d(x.to(DEV), w1.to(DEV), w2.to(DEV), wd.to(DEV)).cpu()


def _check(got, x, w1, w2, wd, what=""):
    ref, a = reference(x, w1, w2, wd)
    err = (got.double() - ref).abs()
    bad = err > C * U * a
    ratio = float((err / (U * a).clamp_min(1e-300)).max())
    assert not bad.any(), (what, int(bad.sum()), ratio)
    print(f"resblock3d {what}: max err / (2^-24 A) = {ratio:.3f}")


def _resident():
    """Clusters of 8 CTAs that the launch keeps resident: one CTA per SM (154 KB of shared memory each)."""
    return max(torch.cuda.get_device_properties(DEV).multi_processor_count // 8, 1)


# ---- batches around the persistent loop ---------------------------------------------------------------------------

def test_batches_around_the_persistent_loop_and_batch_invariance(ahv):
    """M in {1, R-1, R, R+1, 2R+1, 8R+5} for R resident clusters: fewer volumes than clusters, exactly one pass, a
    second pass for one cluster, and many passes.  Every volume's output in a batch of M equals, bit for bit, its
    output computed alone: the per-volume arithmetic depends on neither the cluster nor the pass, so any difference
    is state left over from an earlier volume."""
    R = _resident()
    sizes = sorted({1, max(R - 1, 1), R, R + 1, 2 * R + 1, 8 * R + 5})
    g = torch.Generator().manual_seed(0)
    pool = torch.randn(sizes[-1], 32, 8, 8, 8, generator=g) * torch.rand(sizes[-1], 1, 1, 1, 1, generator=g) * 2
    assert len({float(v.sum()) for v in pool}) == len(pool)              # every volume distinct
    w1, w2, wd = _weights(1)
    alone = torch.cat([_kernel(ahv, pool[i:i + 1], w1, w2, wd) for i in range(len(pool))])
    _check(alone, pool, w1, w2, wd, "alone")
    for m in sizes:
        got = _kernel(ahv, pool[:m], w1, w2, wd)
        assert torch.equal(got, alone[:m]), (m, R)
    _check(_kernel(ahv, pool, w1, w2, wd), pool, w1, w2, wd, f"M={len(pool)}")


# ---- power-of-two symmetries --------------------------------------------------------------------------------------

@pytest.mark.parametrize("e", [-20, -8, 8, 20])
def test_power_of_two_scales_are_exact(ahv, e):
    """No bias and no constant in the chain, so (away from overflow and subnormals) scaling x by 2^e scales the
    output by 2^e exactly; so does scaling (W1, Wd), and (W2, Wd)."""
    g = torch.Generator().manual_seed(3)
    x = torch.randn(5, 32, 8, 8, 8, generator=g)
    w1, w2, wd = _weights(4)
    base = _kernel(ahv, x, w1, w2, wd)
    s = 2.0 ** e
    assert torch.equal(_kernel(ahv, x * s, w1, w2, wd), base * s)
    assert torch.equal(_kernel(ahv, x, w1 * s, w2, wd * s), base * s)
    assert torch.equal(_kernel(ahv, x, w1, w2 * s, wd * s), base * s)


# ---- impulses at the slab boundaries ------------------------------------------------------------------------------

def test_impulses_in_every_slab(ahv):
    """A unit impulse at interior, face, edge and corner positions of every depth slab d = 0..7 (CTA d of the
    cluster), in several input channels.  conv2 reads slabs d-1 and d+1 from the neighbouring CTAs through DSMEM and
    zeros beyond the volume, so a swapped or stale neighbour slab, or a read through the halo, shows as a wrong value
    or as a non-zero outside the impulse's 5x5x5 reach."""
    hw = [(3, 4), (0, 4), (7, 3), (0, 0), (7, 7), (4, 0)]
    cases = [(d, h, w, c) for d in range(8) for (h, w) in hw for c in (0, 13, 31)]
    x = torch.zeros(len(cases), 32, 8, 8, 8)
    for i, (d, h, w, c) in enumerate(cases):
        x[i, c, d, h, w] = 1.0
    w1, w2, wd = _weights(5)
    got = _kernel(ahv, x, w1, w2, wd)
    _check(got, x, w1, w2, wd, "impulses")
    idx = torch.arange(8)
    for i, (d, h, w, c) in enumerate(cases):
        near = ((idx - d).abs() <= 2)[:, None, None] & ((idx - h).abs() <= 2)[None, :, None] & ((idx - w).abs() <= 2)[None, None, :]
        assert (got[i][:, ~near] == 0).all(), (d, h, w, c)
        assert (got[i][:, near] != 0).any(), (d, h, w, c)


# ---- input and weight regimes -------------------------------------------------------------------------------------

def test_regimes(ahv):
    """Positive offset (conv1 mostly active), negative offset (ReLU kills almost everything: out ~ down(x) alone),
    heavy-tailed Student-t inputs, and trained-like weights: log-uniform per-output-channel scales over four decades
    with dead (all-zero) channels."""
    g = torch.Generator().manual_seed(7)
    rng = np.random.default_rng(7)
    base = torch.randn(6, 32, 8, 8, 8, generator=g)
    w1, w2, wd = _weights(8, mean1=0.02)                                  # conv1 weights lean positive
    for name, x, frac in (("positive offset", base + 3.0, lambda f: f > 0.9),
                          ("negative offset", base - 3.0, lambda f: f < 0.05)):
        h = F.conv3d(x.double(), w1.double(), padding=1)
        f = float((h > 0).double().mean())
        assert frac(f), (name, f)
        _check(_kernel(ahv, x, w1, w2, wd), x, w1, w2, wd, name)
    t = torch.from_numpy(rng.standard_t(2.0, (6, 32, 8, 8, 8)).astype(np.float32))
    assert float(t.abs().max()) > 50.0
    _check(_kernel(ahv, t, w1, w2, wd), t, w1, w2, wd, "student-t")
    # trained-like weights
    s1 = torch.from_numpy(10.0 ** rng.uniform(-3, 1, (16, 1, 1, 1, 1))).float()
    s2 = torch.from_numpy(10.0 ** rng.uniform(-3, 1, (16, 1, 1, 1, 1))).float()
    tw1, tw2, twd = w1 * s1, w2 * s2, wd * s2
    tw1[[2, 9]] = 0.0                                                     # dead conv1 channels
    tw2[:, [2, 5]] = 0.0
    twd[[11]] = 0.0
    _check(_kernel(ahv, base, tw1, tw2, twd), base, tw1, tw2, twd, "trained-like weights")


def test_zero_volume_gives_exact_zero(ahv):
    w1, w2, wd = _weights(9)
    x = torch.zeros(3, 32, 8, 8, 8)
    x[1] = torch.randn(32, 8, 8, 8, generator=torch.Generator().manual_seed(9))
    got = _kernel(ahv, x, w1, w2, wd)
    assert (got[0] == 0).all() and (got[2] == 0).all()
    _check(got, x, w1, w2, wd, "zero volume")


# ---- layouts ------------------------------------------------------------------------------------------------------

def test_layouts_give_the_same_bits(ahv):
    """channels_last_3d, a strided slice and a buffer whose data pointer is 4 bytes past a 16-byte boundary give the
    bits of the contiguous copy."""
    g = torch.Generator().manual_seed(10)
    w1, w2, wd = (t.to(DEV) for t in _weights(11))
    big = torch.randn(8, 32, 8, 8, 8, generator=g).to(DEV)
    run = lambda v: ahv.ops.resblock3d(v, w1, w2, wd)
    x = big[:4].contiguous()
    want = run(x)
    cl = x.to(memory_format=torch.channels_last_3d)
    assert not cl.is_contiguous()
    assert torch.equal(run(cl), want)
    sl = big[::2]
    assert not sl.is_contiguous()
    assert torch.equal(run(sl), run(sl.contiguous()))
    flat = torch.empty(x.numel() + 1, device=DEV)
    off = flat[1:].view_as(x)
    off.copy_(x)
    assert off.data_ptr() % 16 == 4
    assert torch.equal(run(off), want)
    # weights from a 4-byte-offset buffer too
    wf = torch.empty(w1.numel() + 1, device=DEV)
    w1o = wf[1:].view_as(w1)
    w1o.copy_(w1)
    assert torch.equal(ahv.ops.resblock3d(x, w1o, w2, wd), want)


# ---- ResNetBlock_3D: which path runs ------------------------------------------------------------------------------

def test_block_keeps_gradients_of_trainable_weights(ahv):
    """conv1 frozen, conv2 and the downsample trainable: the block must take the differentiable path, and their
    gradients match fp64 autograd on the CPU.  Everything frozen: the fused kernel runs (no grad_fn) and gives the
    bits of ops.resblock3d."""
    from modules.modules import ResNetBlock_3D

    torch.manual_seed(12)
    blk = ResNetBlock_3D(32, 16).to(DEV)
    x = torch.randn(3, 32, 8, 8, 8, generator=torch.Generator().manual_seed(13))
    gout = torch.randn(3, 16, 8, 8, 8, generator=torch.Generator().manual_seed(14))
    blk.conv1.weight.requires_grad_(False)
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False                              # cuDNN convolutions in fp32 for the comparison
    try:
        out = blk(x.to(DEV))
        assert out.grad_fn is not None
        (out * gout.to(DEV)).sum().backward()
    finally:
        torch.backends.cudnn.allow_tf32 = tf32
    assert blk.conv1.weight.grad is None
    w1, w2, wd = (p.detach().cpu().double() for p in (blk.conv1.weight, blk.conv2.weight, blk.downsample[0].weight))
    w2.requires_grad_(True)
    wd.requires_grad_(True)
    xd = x.double()
    ref = F.conv3d(F.relu(F.conv3d(xd, w1, padding=1)), w2, padding=1) + F.conv3d(xd, wd)
    (ref * gout.double()).sum().backward()
    for name, got, want in (("conv2", blk.conv2.weight.grad, w2.grad), ("downsample", blk.downsample[0].weight.grad, wd.grad)):
        assert got is not None, name
        err = (got.cpu().double() - want).abs().max().item()
        assert err <= 1e-5 * want.abs().max().item(), (name, err, want.abs().max().item())
    for p in blk.parameters():
        p.requires_grad_(False)
    out = blk(x.to(DEV))
    assert out.grad_fn is None
    direct = ahv.ops.resblock3d(x.to(DEV), blk.conv1.weight, blk.conv2.weight, blk.downsample[0].weight)
    assert torch.equal(out, direct)
