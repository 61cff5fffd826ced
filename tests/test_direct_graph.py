"""k_direct_graph (direct.cuh): with one read length, no forced cuts and the shared-memory histogram,
one look-back pass builds the bundles, node records, CSR rows, components and in-arcs.  Every case
runs through the C ABI with verification and must equal the oracle's replay bit for bit, and the
profile must show the one kernel in place of the chain it replaces."""
import numpy as np
import pytest

from conftest import PRM
from test_gpu_parity import assert_parity, assert_sweep_parity

pytestmark = pytest.mark.gpu

NOSEG = 0xffffffff
REPLACED = ("direct_count", "direct_bundles", "node_finalize", "comp_write", "in_src")


def solve_direct(solver, s, e, Ls, M, off, R, prm=PRM):
    solver.kernel_profile_reset()
    r = solver.solve(s, e, Ls, M, read_off=off, params=prm, verify=True, want_vectors=True,
                     len_hint=(R, R), profile=True)
    names = {k["name"] for k in solver.kernel_profile()}
    assert r.bundle_path == 1
    assert "direct_graph" in names and not names & set(REPLACED), names
    return r


def reads_in(rng, n, lo, hi, R):
    """n reads of length R that lie in [lo, hi)"""
    s = rng.integers(lo, hi - R + 1, size=n).astype(np.uint32)
    return s, (s + np.uint32(R - 1)).astype(np.uint32)


def batch(parts):
    s = np.concatenate([p[0] for p in parts]).astype(np.uint32)
    e = np.concatenate([p[1] for p in parts]).astype(np.uint32)
    off = np.cumsum([0] + [len(p[0]) for p in parts]).astype(np.uint64)
    return s, e, off


def holes_batch(seed, ns, L, R):
    # islands of reads with uncovered stretches between them: several components per sample, and
    # component indices that run across the 4096-node tiles
    rng = np.random.default_rng(seed)
    parts = []
    for _ in range(ns):
        cuts = np.sort(rng.choice(np.arange(1, L // 500), size=10, replace=False)) * 500
        ss, ee = [], []
        for a, b in zip(cuts[0::2], cuts[1::2]):
            x, y = reads_in(rng, int(rng.integers(500, 3000)), int(a), int(b), R)
            ss.append(x)
            ee.append(y)
        parts.append((np.concatenate(ss), np.concatenate(ee)))
    return batch(parts)


def test_components_across_tiles(solver, O):
    ns, L, R, M = 6, 30_000, 100, 40
    s, e, off = holes_batch(1, ns, L, R)
    r = solve_direct(solver, s, e, [L] * ns, M, off, R)
    assert r.n_components >= 4 * ns
    assert_parity(O, r, s, e, [L] * ns, off, M)


def test_ragged_lengths_empty_samples_and_edges(solver, O):
    # ref_len values that are not multiples of 32 and differ within the batch; a sample without
    # reads, one shorter than a read; reads on position 0 and on the last position
    rng = np.random.default_rng(2)
    R, M = 90, 30
    Ls = [30_001, 12_345, 7, 777, 29_999, 5_000]
    parts = []
    for k, L in enumerate(Ls):
        if L < R or k == 5:
            parts.append((np.zeros(0, np.uint32), np.zeros(0, np.uint32)))
            continue
        s, e = reads_in(rng, 40 * L // R, 0, L, R)
        edge = np.array([0] * 3 + [L - R] * 5, np.uint32)
        s = np.concatenate([edge, s, edge]).astype(np.uint32)
        parts.append((s, (s + np.uint32(R - 1)).astype(np.uint32)))
    s, e, off = batch(parts)
    r = solve_direct(solver, s, e, Ls, M, off, R)
    assert r.demand[0] < 0 and r.cov_capped[sum(L + 1 for L in Ls[:1]) - 2] > 0
    assert_parity(O, r, s, e, Ls, off, M)


def test_sample_at_the_key_limit(solver, O):
    # L + 1 slots: exactly the shared-memory histogram.  The default rule would cut a reference this
    # long into segments (the global-memory histogram), so the call asks for it whole.
    L, R, M = 48 * 1024 - 1, 150, 60
    prm = PRM + (NOSEG,)
    s, e, _, _ = O.gen_reads(3, 60_000, L, R)
    off = np.array([0, len(s)], np.uint64)
    r = solve_direct(solver, s, e, [L], M, off, R, prm)
    assert r.n_components >= 1 and r.seg_len == NOSEG
    assert_parity(O, r, s, e, [L], off, M, prm)


def test_one_sample_and_the_same_sample_in_a_batch_of_512(solver, O):
    # alone: k_maxflow_sm (the in-arc goes into the node records); among 512 samples: k_maxflow
    R, M = 120, 50
    sx, ex, _, _ = O.gen_reads(4, 20_000, 9_000, R)
    one = solve_direct(solver, sx, ex, [9_000], M, np.array([0, len(sx)], np.uint64), R)
    assert_parity(O, one, sx, ex, [9_000], [0, len(sx)], M)
    rng = np.random.default_rng(5)
    parts, Ls = [], []
    for k in range(512):
        if k == 300:
            parts.append((sx, ex))
            Ls.append(9_000)
        else:
            L = int(rng.integers(1_000, 3_000))
            parts.append(reads_in(rng, int(rng.integers(0, 2_500)), 0, L, R))
            Ls.append(L)
    s, e, off = batch(parts)
    r = solve_direct(solver, s, e, Ls, M, off, R)
    assert_parity(O, r, s, e, Ls, off, M)
    mask = O.bitmap_to_mask(r.kept_bitmap, len(s))
    lo, hi = int(off[300]), int(off[301])
    assert np.array_equal(O.bitmap_to_mask(one.kept_bitmap, len(sx)), mask[lo:hi])


def test_minimum_cardinality_sweep_reads_the_fused_arrays(solver, O):
    # the sweep reads excl, diff and outdeg; its K3 needs no in-arcs
    ns, L, R, M = 4, 30_000, 100, 40
    s, e, off = holes_batch(6, ns, L, R)
    prm = (64, 150, 1, 0, NOSEG, 0, 1)
    r = solve_direct(solver, s, e, [L] * ns, M, off, R, prm)
    assert_sweep_parity(O, r, s, e, [L] * ns, off, M, prm)
