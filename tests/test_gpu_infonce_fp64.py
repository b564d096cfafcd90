"""GPU: `ahv_infonce` (loss and d loss / d scores in one launch) against a float64 reference of the fp32 inputs,
across shapes, score regimes, temperatures and rotations placed at the positive threshold.

The reference evaluates the mask, the exponentials and both sums in fp64 and never forms a difference of nearly
equal terms: the loss is log1p(sn/sp) and a positive's coefficient is -sn/(sa*sp), sn being the negatives' mass.
Its error is far below the gates, so the gates measure the kernel alone.  They follow from the kernel's arithmetic:
s*(1/T) rounded to fp32 (relative error of exp(s/T) up to |s/T| * 2^-24, 1.2e-6 at |s/T| = 20; exact where 1/T is
a power of two), fp32 expf (2 ulp) and double sums:
  loss      |d| <= 5e-6 * ref                                (relative at every size, including losses << 1)
  gradient  |d| <= 1e-5 * |ref| + 1e-7 * max_row |ref|      (elementwise)
"""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
THR = 15.0
LOSS_RTOL = 5e-6
GRAD_RTOL, GRAD_ROW = 1e-5, 1e-7


# ---- inputs -------------------------------------------------------------------------------------------------------

def _random_rotations(rng, n):
    q = rng.standard_normal((n, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    w, x, y, z = q.T
    return np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                     2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                     2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], -1).reshape(n, 3, 3)


def _rodrigues(axis, theta):
    """[..., 3] unit axes, [...] angles in radians -> [..., 3, 3], fp64."""
    k = np.zeros(axis.shape[:-1] + (3, 3))
    k[..., 0, 1], k[..., 0, 2], k[..., 1, 2] = -axis[..., 2], axis[..., 1], -axis[..., 0]
    k = k - np.swapaxes(k, -1, -2)
    s, c = np.sin(theta)[..., None, None], np.cos(theta)[..., None, None]
    return np.eye(3) + s * k + (1 - c) * (k @ k)


def _offsets(rng, gt, deg):
    """Rotations gt[b] @ exp(theta * axis) at `deg` [B,N] degrees from gt[b] about random axes, rounded to fp32."""
    axis = rng.standard_normal(deg.shape + (3,))
    axis /= np.linalg.norm(axis, axis=-1, keepdims=True)
    return (gt[:, None].astype(np.float64) @ _rodrigues(axis, np.radians(deg))).astype(np.float32)


def _angle_deg(R, gt):
    """fp64 angle [B,N] of the fp32 matrices, as the reference writes it: 180/pi * arccos((clamp(<R,G>,-1,3) - 1)/2)."""
    dot = np.einsum("bnij,bij->bn" if R.ndim == 4 else "nij,bij->bn", R.astype(np.float64), gt.astype(np.float64))
    return 180.0 * np.arccos((np.clip(dot, -1.0, 3.0) - 1.0) / 2.0) / math.pi


def _away_from_threshold(R, gt, thr=THR):
    """Replace hypotheses within 1e-4 deg of the threshold by a ground truth: there fp32 and fp64 may round
    180*acos/pi to different sides (the kernel and the eager formula also round it in different orders), which is
    not a bug.  Such hypotheses must be rare.  A shared R takes gt[0], which callers keep within a few degrees of
    every pair's ground truth."""
    near = np.abs(_angle_deg(R, gt) - thr) <= 1e-4
    assert near.mean() <= 1e-4, near.mean()
    if near.any():
        R = R.copy()
        if R.ndim == 4:
            R[near] = np.broadcast_to(gt[:, None], R.shape)[near]
        else:
            R[near.any(0)] = gt[0]
        assert not (np.abs(_angle_deg(R, gt) - thr) <= 1e-4).any()
    return R


# ---- reference ----------------------------------------------------------------------------------------------------

def reference(s, R, gt, thr, T):
    """fp64 loss [B], gradient [B,N] and positive mask of modules/model.py:43-63 at the fp32 inputs."""
    T = float(np.float32(T))                 # the temperature the kernel receives
    pos = _angle_deg(R, gt) <= np.float32(thr)
    e = np.exp(s.astype(np.float64) / T)
    sp, sn = (e * pos).sum(-1), (e * ~pos).sum(-1)
    sa = sp + sn
    live = sa > 1e-8                          # .clamp(min=1e-8) inactive
    with np.errstate(divide="ignore", invalid="ignore"):
        loss = np.where(live, np.log1p(sn / sp), -np.log(sp / 1e-8))
        c_pos = np.where(live, -sn / (sa * sp), -1.0 / sp)
        c_neg = np.where(live, 1.0 / sa, 0.0)
        grad = np.where(pos, e / T * c_pos[:, None], e / T * c_neg[:, None])
    return loss, grad, pos


def _run(ahv, s, R, gt, thr=THR, T=0.1):
    loss, grad = ahv.ops.infonce(torch.from_numpy(s).to(DEV), torch.from_numpy(R).to(DEV), torch.from_numpy(gt).to(DEV),
                                 thr, T)
    return loss.cpu().numpy().astype(np.float64), grad.cpu().numpy().astype(np.float64)


def _check(ahv, s, R, gt, thr=THR, T=0.1, what=""):
    """Kernel vs reference under the module's gates."""
    ref_l, ref_g, _ = reference(s, R, gt, thr, T)
    got_l, got_g = _run(ahv, s, R, gt, thr, T)
    inf = np.isinf(ref_l)
    assert np.array_equal(np.isinf(got_l), inf) and (got_l[inf] > 0).all(), (what, got_l[inf])
    fin = ~inf
    assert (ref_l[fin] >= 0).all()
    dl = np.abs(got_l[fin] - ref_l[fin])
    assert (dl <= LOSS_RTOL * ref_l[fin]).all(), (what, "loss", ref_l[fin][dl > LOSS_RTOL * ref_l[fin]],
                                                  got_l[fin][dl > LOSS_RTOL * ref_l[fin]])
    assert np.isfinite(got_g).all(), what
    row = np.abs(ref_g).max(-1, keepdims=True)
    gate = GRAD_RTOL * np.abs(ref_g) + GRAD_ROW * row
    dg = np.abs(got_g - ref_g)
    bad = dg > gate
    assert not bad.any(), (what, "grad", int(bad.sum()), float((dg / np.where(row > 0, row, 1)).max()))


# ---- shapes -------------------------------------------------------------------------------------------------------

SHAPES = [(1, 1), (3, 1), (1000, 1), (3, 2), (150, 2), (1, 255), (150, 255), (3, 256), (1000, 256), (3, 257),
          (150, 257), (1, 3000), (150, 3000), (3, 50_001), (1, 1 << 20), (3, 1 << 20)]


@pytest.mark.parametrize("per_pair", [True, False])
@pytest.mark.parametrize("B,N", SHAPES)
def test_shapes_against_fp64(ahv, B, N, per_pair):
    """Fewer hypotheses than threads, ragged tails (255/256/257) and long per-thread loops (2^20 = 4096 per thread),
    the existing uniform score band, hypotheses spread over 0..60 deg so that about a quarter are positive."""
    rng = np.random.default_rng(B * 7919 + N + per_pair)
    if per_pair:
        gt = _random_rotations(rng, B).astype(np.float32)
        R = _offsets(rng, gt, rng.uniform(0.0, 60.0, (B, N)))
    else:                                      # every pair's ground truth within 3 deg of the rotations' centre
        g0 = _random_rotations(rng, 1).astype(np.float32)
        gt = _offsets(rng, g0, rng.uniform(0.0, 3.0, (1, B)))[0]
        R = _offsets(rng, g0, rng.uniform(0.0, 60.0, (1, N)))[0]
    R = _away_from_threshold(R, gt)
    s = rng.uniform(0.2, 0.6, (B, N)).astype(np.float32)
    _check(ahv, s, R, gt, what=(B, N, per_pair))


# ---- score regimes ------------------------------------------------------------------------------------------------

def _pair(rng, N, n_pos, B=1, hi=60.0):
    """B pairs whose first n_pos hypotheses lie within THR - 1 deg and the rest at least THR + 1 deg away."""
    gt = _random_rotations(rng, B).astype(np.float32)
    deg = np.concatenate([rng.uniform(0.0, THR - 1.0, (B, n_pos)), rng.uniform(THR + 1.0, hi, (B, N - n_pos))], 1)
    R = _offsets(rng, gt, deg)
    ref_pos = _angle_deg(R, gt) <= THR
    assert ref_pos[:, :n_pos].all() and not ref_pos[:, n_pos:].any()
    return R, gt


# confident pairs: (N, positives, positive score, negative score).  The first two are the cases where the kernel
# used to lose the loss to fp32 rounding of sp and sa (relative errors ~1e-3 and ~1e-2); the others are stronger.
CONFIDENT = [(3000, 30, 1.0, -0.5), (3000, 30, 0.95, -0.9), (3000, 300, 1.0, -1.0), (50_001, 1, 1.0, -1.0),
             (3000, 2999, 0.9, -0.2), (256, 3, 0.8, -0.4)]


@pytest.mark.parametrize("N,n_pos,s_pos,s_neg", CONFIDENT)
def test_confident_pairs(ahv, N, n_pos, s_pos, s_neg):
    """Positives hold almost all of the softmax mass (a trained model): losses from ~1e-4 down to ~5e-9, where
    -log(fp32(sp)/fp32(sa)) and 1/sa - 1/sp in fp32 cancel.  Scores jitter by 0.01 around the two levels."""
    rng = np.random.default_rng(N + n_pos)
    B = 3
    R, gt = _pair(rng, N, n_pos, B)
    s = np.where(np.arange(N) < n_pos, s_pos, s_neg) + rng.uniform(-0.01, 0.01, (B, N))
    s = s.astype(np.float32)
    ref_l, _, _ = reference(s, R, gt, THR, 0.1)
    assert (ref_l < 1e-3).all() and (ref_l > 0).all(), ref_l
    _check(ahv, s, R, gt, what=(N, n_pos, s_pos, s_neg))


def test_near_uniform_scores(ahv):
    rng = np.random.default_rng(5)
    B, N = 150, 3000
    R, gt = _pair(rng, N, 40, B)
    s = (0.3 + 1e-4 * rng.standard_normal((B, N))).astype(np.float32)
    _check(ahv, s, R, gt)


@pytest.mark.parametrize("N", [1, 2, 257, 3000])
def test_every_hypothesis_positive(ahv, N):
    """sn = 0: the loss is exactly 0 and so is every gradient."""
    rng = np.random.default_rng(N)
    R, gt = _pair(rng, N, N, 3)
    s = rng.uniform(-1.0, 1.0, (3, N)).astype(np.float32)
    loss, grad = _run(ahv, s, R, gt)
    assert (loss == 0).all() and (grad == 0).all(), (loss, np.abs(grad).max())


@pytest.mark.parametrize("N", [1, 2, 257, 3000])
def test_no_positive(ahv, N):
    """sp = 0: the reference's -log(0) = +inf, and finite gradients e/T / sa on every hypothesis."""
    rng = np.random.default_rng(N + 1)
    R, gt = _pair(rng, N, 0, 3)
    s = rng.uniform(-1.0, 1.0, (3, N)).astype(np.float32)
    loss, grad = _run(ahv, s, R, gt)
    assert np.isposinf(loss).all() and np.isfinite(grad).all()
    _check(ahv, s, R, gt)


def test_single_hypothesis(ahv):
    """N = 1: a positive gives loss 0 and gradient 0, a negative +inf and e/T / e = 1/T."""
    rng = np.random.default_rng(1)
    R_pos, gt = _pair(rng, 1, 1, 4)
    R_neg = _offsets(rng, gt, np.full((4, 1), 40.0))
    s = rng.uniform(-1.0, 1.0, (4, 1)).astype(np.float32)
    loss, grad = _run(ahv, s, R_pos, gt)
    assert (loss == 0).all() and (grad == 0).all()
    loss, grad = _run(ahv, s, R_neg, gt)
    assert np.isposinf(loss).all()
    np.testing.assert_allclose(grad, 10.0, rtol=2e-7)


# ---- temperatures -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("T", [0.05, 0.1, 0.5, 1.0, 2.0])
@pytest.mark.parametrize("regime", ["spread", "confident"])
def test_temperatures(ahv, T, regime):
    """|s|/T up to 80.  Spread: at T = 0.05 and 0.1 the scores stay in [-1, 1] (means of cosines, as the model
    produces), so |s/T| <= 20; at T = 0.5, 1 and 2, where 1/T is a power of two and s*(1/T) is exact, they reach 40,
    80 and 160.  Confident: s/T = +-(9.5..10), losses ~1e-7 (far enough from fp32's smallest normal that the fp32
    loss keeps its relative accuracy)."""
    rng = np.random.default_rng(int(T * 100) + (regime == "confident"))
    B, N = 8, 3000
    R, gt = _pair(rng, N, 100, B)
    top = 1.0 if T < 0.5 else 80.0 * T
    if regime == "spread":
        s = rng.uniform(-top, top, (B, N))
    else:                                      # positives at s/T in [9.5, 10], negatives in [-10, -9.5]
        s = np.where(np.arange(N) < 100, 1.0, -1.0) * rng.uniform(9.5, 10.0, (B, N)) * T
    s = s.astype(np.float32)
    assert (np.abs(s.astype(np.float64)) / T <= 80.0 + 1e-9).all()
    _check(ahv, s, R, gt, T=T, what=(T, regime))


@pytest.mark.parametrize("N,n_pos", [(1, 1), (2, 1), (4, 2), (4, 4), (3, 0)])
def test_clamped_total_mass(ahv, N, n_pos):
    """T = 0.05 and every score at -1: sa = N e^-20 <= 8.3e-9 < 1e-8, so the reference's clamp(min=1e-8) is active.
    The loss is -log(sp / 1e-8), the negatives get no gradient (none flows through the clamped sum) and the
    positives get -e/T / sp."""
    rng = np.random.default_rng(N * 10 + n_pos)
    R, gt = _pair(rng, N, n_pos, 2)
    s = np.full((2, N), -1.0, np.float32)
    ref_l, ref_g, pos = reference(s, R, gt, THR, 0.05)
    assert np.exp(-1.0 / 0.05) * N < 1e-8
    assert (ref_g[~pos] == 0).all()
    loss, grad = _run(ahv, s, R, gt, T=0.05)
    assert (grad[~pos] == 0).all()
    assert (np.isposinf(loss) == (n_pos == 0)).all()
    _check(ahv, s, R, gt, T=0.05)


# ---- the positive mask at the threshold ---------------------------------------------------------------------------

@pytest.mark.parametrize("thr", [5.0, 15.0, 30.0, 90.0])
def test_mask_at_threshold(ahv, thr):
    """Rotations at thr +- 1e-3 deg (fp64 Rodrigues, rounded to fp32, the angle recomputed from the fp32 matrix):
    the kernel's positive set, read from the sign of its gradient, equals the fp64 mask."""
    rng = np.random.default_rng(int(thr))
    B, N = 4, 2000
    gt = _random_rotations(rng, B).astype(np.float32)
    side = rng.integers(0, 2, (B, N)) * 2 - 1
    R = _offsets(rng, gt, thr + 1e-3 * side)
    ang = _angle_deg(R, gt)
    assert np.array_equal(ang <= thr, side < 0), "fp32 rounding moved a rotation across the threshold"
    s = rng.uniform(0.2, 0.6, (B, N)).astype(np.float32)
    _, grad = _run(ahv, s, R, gt, thr=thr)
    assert np.array_equal(grad < 0, ang <= thr) and (grad != 0).all()
    _check(ahv, s, R, gt, thr=thr)


# ---- through autograd ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("per_pair", [True, False])
def test_weighted_upstream_gradient(ahv, per_pair):
    """training.infonce_loss under autograd with a weighted upstream gradient (confident and spread pairs mixed),
    and the inference call (want_grad=False) gives the very same losses."""
    rng = np.random.default_rng(11 + per_pair)
    B, N = 6, 3000
    if per_pair:
        R, gt = _pair(rng, N, 30, B)
    else:
        R1, gt1 = _pair(rng, N, 30, 1)
        R, gt = R1[0], np.repeat(gt1, B, 0)
    s = np.where(np.arange(N) < 30, 0.95, -0.9) + rng.uniform(-0.01, 0.01, (B, N))
    s[B // 2:] = rng.uniform(0.2, 0.6, (B - B // 2, N))
    s = s.astype(np.float32)
    w = rng.uniform(-2.0, 2.0, B).astype(np.float32)
    ref_l, ref_g, _ = reference(s, R, gt, THR, 0.1)
    st = torch.from_numpy(s).to(DEV).requires_grad_(True)
    Rt, gtt = torch.from_numpy(R).to(DEV), torch.from_numpy(gt).to(DEV)
    loss = ahv.training.infonce_loss(st, Rt, gtt, THR)
    (loss * torch.from_numpy(w).to(DEV)).sum().backward()
    got_l = loss.detach().cpu().numpy().astype(np.float64)
    assert (np.abs(got_l - ref_l) <= LOSS_RTOL * ref_l).all(), (got_l, ref_l)
    want = ref_g * w.astype(np.float64)[:, None]
    got = st.grad.cpu().numpy().astype(np.float64)
    # one more fp32 rounding (grad * weight) than the kernel's own output: 2^-24 relative, inside the gate
    gate = GRAD_RTOL * np.abs(want) + GRAD_ROW * np.abs(want).max(-1, keepdims=True)
    assert (np.abs(got - want) <= gate).all()
    l2, g2 = ahv.ops.infonce(torch.from_numpy(s).to(DEV), Rt, gtt, THR, want_grad=False)
    assert g2 is None and torch.equal(l2, loss.detach())
