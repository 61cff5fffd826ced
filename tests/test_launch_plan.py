"""K3's launch plan (plan_maxflow_sm, csrc/gds_api.cu: whether k_maxflow_sm runs, with how much
shared memory, which queue size, whether the out-CSR cache fits) is a function of the whole call,
above all of its longest possible component.  A component's schedule and kept reads are a function
of the component alone (include/gds.h, gds_params.schedule; the oracle's express_component).  These
tests put components next to others that move the plan across its branches — a sample too long for
one SM, explicit segment lengths on both sides of each branch — and compare every call bit for bit
with the oracle's replay of the same parameters."""
import numpy as np
import pytest

from conftest import PRM
from test_gpu_parity import COUNTERS, _solve_with_env, assert_parity

gpu = pytest.mark.gpu

NOCUT = 0xffffffff
R = 150


def dev_params(seg, schedule=0):
    return (64, 150, 1, 0, seg, 0, 0, schedule)


def oracle_params(seg, schedule=0):
    return (64, 150, 1, 0, seg, schedule)


def batch(parts):
    """[(start, end, ref_len)] -> start, end, ref_lens, read_off of one call"""
    s = np.concatenate([p[0] for p in parts]).astype(np.uint32)
    e = np.concatenate([p[1] for p in parts]).astype(np.uint32)
    off = np.cumsum([0] + [len(p[0]) for p in parts]).astype(np.uint64)
    return s, e, [p[2] for p in parts], off


def reads(O, seed, L, cov, shape):
    s, e, _, _ = O.gen_reads(seed, L * cov // (2 * R), L, R, shape)
    return s, e, L


def companion_parts(O):
    """The 30 kb uniform sample at coverage 1000 (test_express_schedule_parity's whole sample), and
    a 90 kb uniform sample that stays one ~90 000-node component when nothing is cut: at M = 500 the
    first is one express component, the second is too long for the express schedule and for one SM."""
    small = reads(O, 10, 30_000, 1000, "uniform")
    big = reads(O, 11, 90_000, 1000, "uniform")
    return small, big


def solve(solver, O, s, e, Ls, off, M, seg, schedule=0, env=None):
    """One profiled call, checked against the oracle; returns (result, oracle stats, launches by name)."""
    solver.kernel_profile_reset()
    r = _solve_with_env(solver, env or {}, s, e, Ls, M, read_off=off, params=dev_params(seg, schedule),
                        verify=True, want_vectors=True, profile=True)
    launches = {k["name"]: k["launches"] for k in solver.kernel_profile()}
    st = assert_parity(O, r, s, e, Ls, off, M, oracle_params(seg, schedule))
    return r, st, launches


def assert_same_call(a, b):
    for key in COUNTERS + ("verify_violations",):
        assert a[key] == b[key], key
    assert np.array_equal(a.kept_bitmap, b.kept_bitmap)
    assert np.array_equal(a.demand, b.demand) and np.array_equal(a.cov_capped, b.cov_capped)


def test_oracle_companion_keeps_the_schedule_and_the_kept_reads(O):
    # the expectation the device is held to below: next to a sample too long for one SM, the 30 kb
    # sample is solved with the same schedule and keeps the same reads as alone
    small, big = companion_parts(O)
    s1, e1, Ls1, off1 = batch([small])
    bm1, st1 = O.sync_solve(s1, e1, Ls1, off1, 500, params=oracle_params(NOCUT))
    s2, e2, Ls2, off2 = batch([big, small])
    bm2, st2 = O.sync_solve(s2, e2, Ls2, off2, 500, params=oracle_params(NOCUT))
    assert st1.n_express == st2.n_express == 1
    assert st1.n_components == 1 and st2.n_components == 2
    n_big = len(big[0])
    mask2 = O.bitmap_to_mask(bm2, len(s2))
    assert np.array_equal(O.bitmap_to_mask(bm1, len(s1)), mask2[n_big:])
    assert 0 < int(mask2[n_big:].sum()) < len(s1)


@gpu
def test_companion_too_long_for_one_sm_keeps_the_express_schedule(solver, O):
    # the 30 kb sample alone, then after a 90 001-node sample in one call that cuts nothing: the
    # call's longest component no longer fits one SM, the 30 kb sample's component still does and
    # must run in k_maxflow_sm with the express schedule; the 90 kb one goes to k_maxflow
    small, big = companion_parts(O)
    s1, e1, Ls1, off1 = batch([small])
    r1, st1, _ = solve(solver, O, s1, e1, Ls1, off1, 500, NOCUT)
    s2, e2, Ls2, off2 = batch([big, small])
    r2, st2, launches = solve(solver, O, s2, e2, Ls2, off2, 500, NOCUT)
    assert st1.n_express > 0 and st2.n_express > 0
    assert launches["maxflow"] == 2, launches  # k_maxflow_sm, then k_maxflow for its fallback list
    n_big = len(big[0])
    assert np.array_equal(O.bitmap_to_mask(r1.kept_bitmap, len(s1)),
                          O.bitmap_to_mask(r2.kept_bitmap, len(s2))[n_big:])


@gpu
def test_companion_with_the_global_memory_kernel_requested(solver, O):
    # GDS_MF=global asks for k_maxflow only; express components exist only in k_maxflow_sm, so it
    # still runs for them (everything else goes to k_maxflow) and nothing about the answer changes
    small, big = companion_parts(O)
    s, e, Ls, off = batch([big, small])
    a, st, _ = solve(solver, O, s, e, Ls, off, 500, NOCUT)
    b, _, launches = solve(solver, O, s, e, Ls, off, 500, NOCUT, env={"GDS_MF": "global"})
    assert st.n_express > 0
    assert launches["maxflow"] == 2, launches
    assert_same_call(a, b)


# (ref_len, seg_len, M, schedule, coverage) -> the plan's branch for the call's longest component
# (one CTA of 512 threads per SM in all of them; header 320 B, queues of 16 B per entry)
SWEEP = {
    "whole_40961": (40_960, NOCUT, 500, 0, 1000),    # queues of 256, no out-CSR cache: 189 KB
    "whole_40962": (40_961, NOCUT, 500, 0, 1000),    # one node beyond the largest express component
    "whole_51001": (51_000, NOCUT, 500, 0, 1000),    # beyond 50 672 nodes: clamped to 227 KB
    "whole_65520": (65_519, NOCUT, 500, 0, 1000),    # kMf2MaxNodes: still clamped
    "whole_65521": (65_520, NOCUT, 500, 0, 1000),    # beyond kMf2MaxNodes: clamped, longest on fb_list
    "whole_90001": (90_000, NOCUT, 500, 0, 1000),
    "seg_32760": (75_520, 32_760, 500, 0, 1000),     # queues of 1024 with the out-CSR cache
    "seg_40000": (90_000, 40_000, 500, 0, 1000),     # the cache dropped
    "seg_60000": (130_000, 60_000, 500, 0, 1000),    # clamped
    "seg_65520": (141_040, 65_520, 500, 0, 1000),    # segments beyond kMf2MaxNodes
    "schedule2_m60": (90_000, NOCUT, 60, 2, 120),    # express at any supply
    "schedule3_m100": (90_000, NOCUT, 100, 3, 200),  # forced cuts, classic schedule only
}


@gpu
@pytest.mark.parametrize("case", list(SWEEP))
def test_plan_branches_keep_parity(solver, O, case):
    # the "hole" shape: the coverage dips to ~0.4x in the middle, so the forced cuts at cov <= M
    # leave pieces that take the express schedule next to the call's long components
    L, seg, M, schedule, cov = SWEEP[case]
    s, e, Ls, off = batch([reads(O, 100, L, cov, "hole")])
    r, st, launches = solve(solver, O, s, e, Ls, off, M, seg, schedule)
    assert (st.n_express > 0) == (schedule != 3), st.n_express
    if st.n_express:
        assert launches["maxflow"] == 2, launches  # k_maxflow_sm and its fallback k_maxflow


@gpu
def test_context_history_does_not_leak_into_a_call(pkg, solver, O):
    # one context through calls of every kind: long and short, with and without forced cuts
    # (fmult, written per call for the bundles of candidate nodes only, is never cleared), one or
    # several samples.  Each call must equal the same call on a context of its own.
    small, big = companion_parts(O)
    ex = O.SMALL_EXAMPLE
    tiny = (ex["start"], ex["end"], ex["L"])
    three = [reads(O, 20 + k, L, 600, "low_sides") for k, L in enumerate((9_000, 20_000, 4_000))]
    calls = [  # (parts, M, seg_len, schedule)
        ([big, small], 500, NOCUT, 0),
        ([tiny], ex["M"], 0, 0),
        ([reads(O, 30, 65_520, 1000, "hole")], 500, NOCUT, 0),
        ([reads(O, 31, 3_000, 400, "uniform")], 30, 0, 0),
        ([reads(O, 32, 90_000, 1000, "hole")], 500, 40_000, 0),
        ([small], 500, NOCUT, 0),
        (three, 200, 0, 0),
        ([reads(O, 33, 90_000, 200, "hole")], 100, NOCUT, 3),
        (three, 20, 4_096, 0),
        ([reads(O, 34, 90_000, 120, "hole")], 60, NOCUT, 2),
        ([small], 500, NOCUT, 0),
    ]
    shared = pkg.Solver(0)
    try:
        for parts, M, seg, schedule in calls:
            s, e, Ls, off = batch(parts)
            kw = dict(read_off=off, params=dev_params(seg, schedule), verify=True, want_vectors=True)
            r = shared.solve(s, e, Ls, M, **kw)
            assert_parity(O, r, s, e, Ls, off, M, oracle_params(seg, schedule))
            fresh = pkg.Solver(0)
            try:
                assert_same_call(r, fresh.solve(s, e, Ls, M, **kw))
            finally:
                fresh.close()
    finally:
        shared.close()
