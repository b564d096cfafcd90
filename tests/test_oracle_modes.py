"""CPU: modes_oracle (the selection steps of ahv_search_modes) against brute-force restatements of its definitions, on the
nested Hopf grid with tied scores, empty (NaN) centres, slots with fewer than w cells, min_sep = 180 and no levels."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import distinct_oracle  # noqa: E402  (tests/distinct_oracle.py)
import hopf_oracle as h  # noqa: E402  (tests/hopf_oracle.py)
import modes_oracle as mo  # noqa: E402  (tests/modes_oracle.py)
from posterior_oracle import trace_threshold_np  # noqa: E402

f = np.float32


def _trace(a, c):
    t = f(a[0]) * f(c[0])
    for q in range(1, 9):
        t = f(t + f(a[q]) * f(c[q]))
    return t


def brute_slots(G, first_idx, first_R, theta):
    c = trace_threshold_np(theta)
    B, k = first_idx.shape
    out = np.full((B, len(G)), -1)
    for b in range(B):
        for n in range(len(G)):
            wins = [j for j in range(k) if first_idx[b, j] == n]
            if wins:
                out[b, n] = wins[0]
                continue
            for j in range(k):
                if first_idx[b, j] >= 0 and _trace(G[n].reshape(9), first_R[b, j].reshape(9)) >= c:
                    out[b, n] = j
                    break
    return out


def brute_beams(S0, slot, k, w):
    B = S0.shape[0]
    out = np.full((B, k, w), -1)
    for b in range(B):
        for j in range(k):
            cells = sorted((n for n in range(S0.shape[1]) if slot[b, n] == j), key=lambda n: (-float(S0[b, n]), n))[:w]
            out[b, j, : len(cells)] = sorted(cells)
    return out


def brute_level(scores, kids, par, last):
    B, k, w = par.shape
    nc = 8 * w
    nxt = np.full((B, k, w), -1)
    modes = []
    for b in range(B):
        mb = []
        for j in range(k):
            ts = [t for t in range(nc) if par[b, j, t // 8] >= 0]
            ts = sorted(ts, key=lambda t: (-float(scores[b, nc * j + t]), t))[:w]
            nxt[b, j, : len(ts)] = sorted(int(kids[b, nc * j + t]) for t in ts)
            if ts:
                mb.append((-float(scores[b, nc * j + ts[0]]), int(kids[b, nc * j + ts[0]])))
        modes.append(sorted(mb))
    return nxt, modes


def _base(level, B, k, theta, seed, decimals=1):
    rng = np.random.default_rng(seed)
    G = h.hopf_grid_np(level)
    S0 = np.round(rng.standard_normal((B, len(G))).astype(f), decimals)          # many ties
    fv, fi, fR = distinct_oracle.select_distinct_np(S0, G, k, theta)
    return G, S0, fv, fi, fR


@pytest.mark.parametrize("theta", (5.0, 30.0, 60.0, 120.0, 180.0))
@pytest.mark.parametrize("k,w", ((1, 1), (4, 4), (8, 3), (32, 8)))
def test_slots_and_beams_equal_brute_force(theta, k, w):
    G, S0, fv, fi, fR = _base(0, 3, k, theta, seed=k + w)
    slot = mo.slots_np(G, fi, fR, theta)
    assert np.array_equal(slot, brute_slots(G, fi, fR, theta))
    par = mo.beams_np(S0, slot, k, w)
    assert np.array_equal(par, brute_beams(S0, slot, k, w))
    for b in range(3):
        for j in range(k):
            if fi[b, j] < 0:                                                          # an empty slot holds nothing
                assert (slot[b] != j).all() and (par[b, j] == -1).all()
            else:                                                                     # the winner leads its slot
                assert fi[b, j] in par[b, j]
                members = np.flatnonzero(slot[b] == j)
                best = sorted(members, key=lambda n: (-float(S0[b, n]), n))[0]
                assert best == fi[b, j]


def test_the_winner_is_its_slots_whatever_the_trace_says():
    G = h.hopf_grid_np(0)
    fi = np.array([[5, -1]])
    fR = np.stack([G[5], np.full((3, 3), np.nan, f)])[None]
    # min_sep so small that c rounds to 3.0: no cell, not even the winner, passes the trace test
    assert trace_threshold_np(1e-5) == f(3.0)
    slot = mo.slots_np(G, fi, fR, 1e-5)
    assert slot[0, 5] == 0 and (np.delete(slot[0], 5) == -1).all()
    S0 = np.zeros((1, len(G)), f)
    assert np.array_equal(mo.beams_np(S0, slot, 2, 4), [[[5, -1, -1, -1], [-1, -1, -1, -1]]])


def test_nan_centres_hold_no_cell():
    G = h.hopf_grid_np(0)
    fi = np.array([[3, -1, 40]])
    fR = np.stack([G[3], np.full((3, 3), np.nan, f), G[40]])[None]
    slot = mo.slots_np(G, fi, fR, 90.0)
    assert (slot != 1).all() and slot[0, 3] == 0 and slot[0, 40] == 2
    assert np.array_equal(slot, brute_slots(G, fi, fR, 90.0))


def test_a_slot_with_fewer_cells_than_the_beam_is_padded_at_the_end():
    G, S0, fv, fi, fR = _base(0, 2, 32, 10.0, seed=1)                                # 10 deg: about one cell a slot
    slot = mo.slots_np(G, fi, fR, 10.0)
    par = mo.beams_np(S0, slot, 32, 8)
    sizes = (par >= 0).sum(-1)
    assert (sizes[fi >= 0] < 8).any()
    for row in par.reshape(-1, 8):
        n = (row >= 0).sum()
        assert (row[n:] == -1).all() and (np.diff(row[:n]) > 0).all()


def test_min_sep_180_is_one_mode_holding_every_cell():
    G, S0, fv, fi, fR = _base(1, 2, 8, 180.0, seed=2)
    assert (fi[:, 0] >= 0).all() and (fi[:, 1:] == -1).all()
    slot = mo.slots_np(G, fi, fR, 180.0)
    assert (slot == 0).all()
    par = mo.beams_np(S0, slot, 8, 4)
    keys = distinct_oracle._topk_keys_np(S0)
    for b in range(2):
        assert np.array_equal(par[b, 0], np.sort(np.argsort(keys[b])[::-1][:4])) and (par[b, 1:] == -1).all()


def _landscape(R, peaks, weights):
    """A multi-modal score: the weighted best of trace(R P^T) over the peaks, in fp32."""
    Rs = R.reshape(-1, 9).astype(f)
    s = np.max([f(wt) * mo.trace_np(Rs, P.reshape(9).astype(f)) for P, wt in zip(peaks, weights)], axis=0)
    return s.reshape(R.shape[:-2])


@pytest.mark.parametrize("levels", (0, 1, 3))
@pytest.mark.parametrize("k,w", ((1, 4), (4, 2), (8, 4), (5, 8)))
def test_levels_equal_brute_force_and_keep_their_slots(levels, k, w):
    B, base, theta = 2, 1, 30.0
    rng = np.random.default_rng(levels * 10 + k)
    peaks = h.hopf_rotations_np(4, rng.integers(0, h.cells(4), (3,)))
    G = h.hopf_grid_np(base)
    S0 = np.stack([_landscape(G, peaks, (1.0, 0.97, 0.9)), np.round(_landscape(G, peaks[::-1], (1.0, 1.0, 0.5)), 2)])
    fv, fi, fR = distinct_oracle.select_distinct_np(S0, G, k, theta)
    slot = mo.slots_np(G, fi, fR, theta)
    seen = []

    def children(lev, gen):
        kids = h.hopf_children_np(gen).reshape(B, -1)
        return kids, h.hopf_rotations_np(base + lev + 1, kids)

    def score(R):
        s = np.stack([_landscape(R[b], peaks, (1.0, 0.97, 0.9)) for b in range(B)])
        s[:, ::7] = s[:, ::7].max()                                                   # ties, some on children of pads
        seen.append(s)
        return s

    val, idx, R = mo.search_modes_np(S0, G, fv, fi, fR, theta, w, levels, children, score)
    if levels == 0:
        assert val is fv and idx is fi and R is fR
        return
    # replay the levels with the brute-force definitions
    par = brute_beams(S0, slot, k, w)
    for lev in range(levels):
        kids, _ = children(lev, mo.generator_parents_np(par))
        nxt, modes = brute_level(seen[lev], kids, par, lev == levels - 1)
        assert np.array_equal(nxt, mo.level_np(seen[lev], kids, par, False))
        par = nxt
    for b in range(B):
        n = len(modes[b])
        assert [(-float(v), int(i)) for v, i in zip(val[b, :n], idx[b, :n])] == modes[b]
        assert (idx[b, n:] == -1).all() and np.isneginf(val[b, n:]).all() and np.isnan(R[b, n:]).all()
        assert n == (fi[b] >= 0).sum()
        np.testing.assert_array_equal(R[b, :n], h.hopf_rotations_np(base + levels, idx[b, :n]))
        # every mode descends from a base cell of the slot it came from, and the modes come from distinct slots
        origin = slot[b, idx[b, :n] // 8 ** levels]
        assert (origin >= 0).all() and len(set(origin.tolist())) == n
