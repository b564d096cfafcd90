"""GPU (B200): the fp32 CUDA-core kernels bit for bit against a numpy model of their own arithmetic (tests/fp32_model.py).

The fp32 scorer (AHV_MATH_FP32) was held to 2e-5 of the C oracle, about 70 times its real error, and the target
features to 2e-6: a tap summed in another order, a coordinate FMA reassociated, a bias added first or a division in
place of a reciprocal multiply moves results by 1e-7 to 1e-6 and passes such gates.  The model restates every fp32
operation in the kernels' order, so here the outputs must be identical to it:

  - AHV_MATH_FP32 scores on every case of tests/tc_model.py, fp32 volumes and bf16 volumes (against the model of the
    bf16 values), shared and per-pair rotations;
  - the target features of ahv_forward_3d2d (and HypothesisVerifier.target_features) at m = 1 .. 9000, on both sides
    of the 4096 volumes where the launcher once switched kernels;
  - rotate_volume, shared and per rotation, through ops and refcompat, on lattice, beyond-volume, shrunk and sheared
    matrices and on the tails of the 8-rotations-per-CTA split.

The backward of rotate_volume adds with float atomics in no fixed order; it is held to the model's per-element bound
on any order of its own rounded terms.  A mismatch reports where it is and how many ulps it is off."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import fp32_model as F  # noqa: E402  (tests/fp32_model.py)
import kernel_arith as K  # noqa: E402
import tc_model as M  # noqa: E402  (the cases)

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
f32 = np.float32


def _T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _head(case):
    return [_T(case[k]) for k in ("W1", "W2", "b2")]


def _bits_report(got, want, where):
    """'' when got and want are bit-identical, else the first mismatches as (where, ulps) and the largest distance."""
    got, want = np.asarray(got, f32), np.asarray(want, f32)
    same = got.view(np.uint32) == want.view(np.uint32)
    if same.all():
        return ""
    bad = np.argwhere(~same)
    ulps = K.ulp_distance(got, want)
    return (f"{len(bad)} of {same.size} differ, at most {int(ulps.max())} ulps; first: "
            + ", ".join(f"{where(tuple(int(i) for i in b))} {int(ulps[tuple(b)])} ulp" for b in bad[:6]))


_CASES = {}


@pytest.fixture(scope="module")
def case(golden, request):
    name = request.param
    if name not in _CASES:
        _CASES.clear()
        _CASES[name] = dict(M.make_case(name, golden), name=name)
    return _CASES[name]


# ---- the scorer -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", M.CASES, indirect=True)
@pytest.mark.parametrize("voldt", ["f32", "bf16"])
def test_fp32_scores_bit_identical_to_the_model(ahv, case, voldt):
    """ahv_score under AHV_MATH_FP32 runs the whole case; the model scores the golden set's first 200 hypotheses of
    each pair, or at most 48 items of any other case (the first and last included)."""
    vs = case["vs"]
    v = _T(vs)
    if voldt == "bf16":
        v, vs = v.bfloat16(), K.bf16_round(vs)
    R = case["R"]
    B, N = vs.shape[0], R.shape[-3]
    s, _, _ = ahv.ops.score(v, _T(case["tgt"]), _T(R), *_head(case), k=min(4, N), math=ahv.MATH_FP32)
    items = F.case_items(case["name"], B, N, cap=48)
    model = F.score(vs, case["tgt"], R, case["W1"], case["W2"], case["b2"], items=items)
    got = s.cpu().numpy().reshape(-1)[items]
    msg = _bits_report(got, model, lambda i: f"(pair {items[i[0]] // N}, hypothesis {items[i[0]] % N})")
    assert not msg, (case["name"], voldt, msg)


# ---- target features ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def many_volumes():
    rng = np.random.default_rng(2024)
    return (rng.standard_normal((9000, 16, 8, 8, 8), dtype=f32) * f32(1.1) - f32(0.2)).astype(f32)


@pytest.mark.parametrize("m", [1, 3, 4096, 4097, 9000])
def test_target_features_bit_identical_to_the_model(ahv, golden, many_volumes, m):
    """ahv_forward_3d2d at m volumes: the sampled rows (the first, last and both sides of 4096 included) equal the
    model; HypothesisVerifier.target_features gives the same bits, and so does a call on the first 4096 volumes alone."""
    w = golden["weights"]
    W = [_T(w[k]) for k in ("W1", "W2", "b2")]
    V = many_volumes[:m]
    Vd = _T(V)
    feat = ahv.ops.forward_3d2d(Vd, *W)
    rows = np.unique(np.concatenate([[0, m - 1], np.arange(4094, 4098),
                                     np.random.default_rng(m).choice(m, min(m, 48), replace=False)]))
    rows = rows[rows < m]
    model = F.target_features(V[rows], w["W1"], w["W2"], w["b2"])
    got = feat.cpu().numpy()
    msg = _bits_report(got[rows], model, lambda i: f"(volume {rows[i[0]]}, channel {i[1]}, position {i[2]})")
    assert not msg, (m, msg)
    assert torch.equal(ahv.HypothesisVerifier(*W).target_features(Vd), feat)
    if m > 4096:
        assert torch.equal(ahv.ops.forward_3d2d(Vd[:4096], *W), feat[:4096])


# ---- rotate_volume --------------------------------------------------------------------------------------------------
def _rotations(kind: str, n: int, seed: int) -> np.ndarray:
    rng = np.random.default_rng(seed)
    R = K.random_rotations(rng, n)
    if kind == "lattice":
        L = K.lattice_rotations()
        R = L[np.arange(n) % len(L)]
    elif kind == "beyond_volume":                            # most samples land outside the volume
        R = R * f32(2.5)
    elif kind == "shrunk":                                   # a zoom into the centre
        R = R * f32(0.35)
    elif kind == "sheared":                                  # not orthonormal
        R = R @ np.array([[1.0, 0.3, 0.0], [0.0, 1.0, -0.2], [0.1, 0.0, 0.9]], f32)
    return np.ascontiguousarray(R, f32)


KINDS = ["random", "lattice", "beyond_volume", "shrunk", "sheared"]
NS = [1, 7, 8, 9, 17, 300]                                   # the tails of the 8-rotations-per-CTA split


def _vol(seed, *shape):
    return (np.random.default_rng(seed).normal(size=shape + (16, 8, 8, 8)) * 1.1 - 0.2).astype(f32)


def _where5(i):
    return f"(rotation {i[0]}, channel {i[1]}, voxel d{i[2]} h{i[3]} w{i[4]})"


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", NS)
def test_rotate_volume_shared_bit_identical(ahv, n, kind):
    vol, R = _vol(n), _rotations(kind, n, seed=n + 17)
    got = ahv.ops.rotate_volume(_T(vol), _T(R)).cpu().numpy()
    msg = _bits_report(got, F.rotate_volume(vol, R), _where5)
    assert not msg, (n, kind, msg)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", [1, 9, 300])
def test_rotate_volume_per_rotation_bit_identical(ahv, n, kind):
    vol, R = _vol(n + 1, n), _rotations(kind, n, seed=n + 29)
    got = ahv.ops.rotate_volume(_T(vol), _T(R)).cpu().numpy()
    msg = _bits_report(got, F.rotate_volume(vol, R), _where5)
    assert not msg, (n, kind, msg)


@pytest.mark.parametrize("n", [1, 9, 300])
def test_refcompat_rotate_volume_bit_identical(ahv, n):
    """The reference idiom passes a stride-0 expand or a [1,...] volume once (a shared volume)."""
    vol, R = _vol(n + 2), _rotations("random", n, seed=n + 41)
    want = F.rotate_volume(vol, R)
    for v in (_T(vol)[None].expand(n, 16, 8, 8, 8), _T(vol)[None]):
        got = ahv.refcompat.rotate_volume(v, _T(R)).cpu().numpy()
        msg = _bits_report(got, want, _where5)
        assert not msg, (n, tuple(v.shape), v.stride(0), msg)


# largest |kernel - exact| / bound seen by the backward tests (scripts/fp32_model_residual.py records it per case)
@pytest.mark.parametrize("per_rotation", [False, True])
@pytest.mark.parametrize("n", NS)
def test_rotate_volume_backward_within_the_bound(ahv, n, per_rotation):
    """Every element of the volume gradient within gamma_(count+1) sum |RN(w g)| of the exact sum of the kernel's own
    terms, for n matrices drawn from the random, lattice, beyond-volume, shrunk and sheared kinds together."""
    pool = np.concatenate([_rotations(k, n, seed=n + 53) for k in KINDS])
    R = np.ascontiguousarray(pool[np.random.default_rng(n).permutation(len(pool))[:n]])
    g = (np.random.default_rng(n + 7).normal(size=(n, 16, 8, 8, 8))).astype(f32)
    got = ahv.ops.rotate_volume_backward(_T(g), _T(R), per_rotation).cpu().numpy().astype(np.float64)
    exact, cnt, bound = F.rotate_volume_adjoint(g, R, per_rotation)
    err = np.abs(got - exact)
    far = np.argwhere(err > bound)
    ratio = float(np.max(np.where(bound > 0, err / np.where(bound > 0, bound, 1.0), np.where(err > 0, np.inf, 0.0))))
    print(f"rotate_volume_backward n={n} per_rotation={per_rotation}: largest error / bound {ratio:.3g}")
    assert len(far) == 0, (n, per_rotation, "beyond the bound at", far[:6].tolist(), ratio)
