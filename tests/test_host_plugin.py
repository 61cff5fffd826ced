"""The C++ host mirror: reads-gen streams equal the reference's, the SolverManager registry knows
the new algorithm, and (on a GPU) the plugin path solve(max_coverage, BamApi&) returns ascending
kept indices that satisfy the reference's coverage invariant."""
import hashlib

import numpy as np
import pytest


@pytest.fixture(scope="module")
def hostlib(pkg):
    from genome_downsampler_b200 import hostlib
    hostlib.load()
    return hostlib


def test_host_reads_gen_matches_oracle_and_reference_streams(hostlib, O):
    for shape in ("uniform", "low_sides", "hole", "zero_sides"):
        s = np.empty(20_000, np.uint32); e = np.empty(20_000, np.uint32)
        q = np.empty(20_000, np.uint8); l = np.empty(20_000, np.uint32)
        hostlib.gen_reads_into(4242, 10_000, 30_000, 150, s, e, q, l, shape=shape)
        s0, e0, q0, l0 = O.gen_reads(4242, 10_000, 30_000, 150, shape)
        assert np.array_equal(s, s0) and np.array_equal(e, e0)
        assert np.array_equal(q, q0.astype(np.uint8)) and np.array_equal(l, l0)


def test_host_reads_gen_matches_reference_build(hostlib, golden):
    # the reference's own stream for these parameters, as stored in golden.json
    g = golden["generators"]["c3"]
    s = np.empty(2 * g["pairs"], np.uint32); e = np.empty(2 * g["pairs"], np.uint32)
    hostlib.gen_reads_into(g["seed"], g["pairs"], g["L"], g["R"], s, e)
    assert hashlib.sha256(s.tobytes()).hexdigest() == g["start"]
    assert hashlib.sha256(e.tobytes()).hexdigest() == g["end"]


def test_gen_batch_threads_equal_serial(hostlib):
    n = 2 * 5_000
    s = np.empty(4 * n, np.uint32); e = np.empty(4 * n, np.uint32)
    hostlib.gen_batch([7, 8, 9, 10], 5_000, 30_000, 150, s, e, threads=4)
    s1 = np.empty(n, np.uint32); e1 = np.empty(n, np.uint32)
    hostlib.gen_reads_into(9, 5_000, 30_000, 150, s1, e1)
    assert np.array_equal(s[2 * n:3 * n], s1) and np.array_equal(e[2 * n:3 * n], e1)


def test_unknown_algorithm_is_rejected(hostlib):
    with pytest.raises(KeyError):
        hostlib.plugin_solve("quasi-mcp-nope", np.zeros(2, np.uint32), np.ones(2, np.uint32), 10, 1)


@pytest.mark.gpu
def test_plugin_solve_through_solver_manager(hostlib, O):
    # SolverManager.get("quasi-mcp-b200").solve(M, BamApi(reads)) exactly as src/app.cpp:130-135
    ex = O.SMALL_EXAMPLE
    ids = hostlib.plugin_solve("quasi-mcp-b200", ex["start"], ex["end"], ex["L"], ex["M"])
    assert len(ids) == 14 and np.all(np.diff(ids.astype(np.int64)) > 0)
    s, e, q, l = O.gen_reads(12345, 50_000, 30_000, 150)
    ids = hostlib.plugin_solve("quasi-mcp-b200", s, e, 30_000, 100)
    mask = np.zeros(len(s), np.uint8); mask[ids] = 1
    cin = O.coverage_fast(s, e, 30_000); cout = O.coverage_fast(s, e, 30_000, mask)
    assert np.array_equal(np.minimum(cin, 100), np.minimum(cout, 100))
    bm, st = O.sync_solve(s, e, [30_000], [0, len(s)], 100, params=(64, 150, 1, 0))
    assert np.array_equal(O.bitmap_to_mask(bm, len(s)), mask)


@pytest.mark.gpu
def test_mcp_b200_plugin_returns_the_minimum_cover(hostlib, O):
    # SolverManager.get("mcp-b200"): the fewest reads with min(coverage, M) kept everywhere — what
    # mcp-cpu's min-cost flow (unit read costs) reports as its optimal cost
    for seed, pairs, L, M, shape in ((5, 40_000, 30_000, 100, "uniform"), (6, 20_000, 9_000, 700, "hole")):
        s, e, q, l = O.gen_reads(seed, pairs, L, 150, shape)
        ids = hostlib.plugin_solve("mcp-b200", s, e, L, M)
        mask = np.zeros(len(s), np.uint8); mask[ids] = 1
        cin = O.coverage_fast(s, e, L); cout = O.coverage_fast(s, e, L, mask)
        assert np.all(np.minimum(cin, M) <= cout)
        _, nopt = O.greedy_multicover(s, e, L, M)
        assert len(ids) == nopt and len(ids) <= len(hostlib.plugin_solve("quasi-mcp-b200", s, e, L, M))


@pytest.mark.gpu
def test_plugin_solve_batch_equals_one_by_one(hostlib, O):
    # QuasiMcpB200MaxFlowSolver::solve_batch: ragged samples (different sizes, shapes and read
    # lengths, so the batch travels as 32-bit columns) and a fixed-length batch (compact transport);
    # every sample's index list equals solve() on that sample alone and the oracle's bitmap
    parts = [O.gen_reads(300 + k, 20_000 + 37 * k, 30_000, 150, sh)
             for k, sh in enumerate(["uniform", "hole", "uniform", "low_sides", "uniform"])]
    rng = np.random.default_rng(4)
    s5 = rng.integers(0, 29_000, size=30_001).astype(np.uint32)   # odd count, variable lengths
    e5 = (s5 + rng.integers(80, 200, size=30_001)).astype(np.uint32)
    for extra in ([], [(s5, e5)]):
        ps = [(p[0], p[1]) for p in parts] + extra
        s = np.concatenate([p[0] for p in ps]); e = np.concatenate([p[1] for p in ps])
        off = np.cumsum([0] + [len(p[0]) for p in ps]).astype(np.uint64)
        per, counts, secs = hostlib.plugin_solve_batch(s, e, off, 30_000, 60, repeats=2)
        assert secs > 0 and len(per) == len(ps)
        bm, st = O.sync_solve(s, e, [30_000] * len(ps), off, 60, params=(64, 150, 1, 0))
        mask = O.bitmap_to_mask(bm, len(s))
        for k, (sk, ek) in enumerate(ps):
            one = hostlib.plugin_solve("quasi-mcp-b200", sk, ek, 30_000, 60)
            assert np.array_equal(per[k], one) and counts[k] == len(one)
            assert np.array_equal(np.flatnonzero(mask[int(off[k]):int(off[k + 1])]), per[k].astype(np.int64))


@pytest.mark.gpu
def test_reference_coverage_tester_runs_against_the_cuda_path(pkg, solver, coverage_tester):
    # the reference's CoverageTester::test (src/tests/coverage_tester.cpp:28-43, restated in
    # conftest.py on its own inputs) drives the CUDA solver through a callback:
    # 5 cases, each solve re-enters the same context like the reference's registry does
    calls = []

    def solve(M, L, s, e):
        r = solver.solve(s, e, L, M, verify=True)
        assert r.verify_violations == 0 and r.flow_value == r.fstar
        calls.append((M, L, len(s), int(r.n_kept)))
        return pkg.Solver.bitmap_to_indices(r.kept_bitmap, len(s))
    assert coverage_tester(solve) == 5
    assert [c[0] for c in calls] == [4, 1000, 8000, 8000, 8000]


@pytest.mark.gpu
def test_host_test_binary_runs_the_five_cases_through_the_plugin(pkg):
    # gds_host_test = the reference's `test` subcommand for this path, C++ end to end:
    # SolverManager -> qmcp::Solver::solve(M, BamApi&) -> C ABI -> device
    import os
    import subprocess
    exe = os.path.join(os.path.dirname(pkg.lib_path()), "gds_host_test")
    out = subprocess.run([exe, "-a", "quasi-mcp-b200", "-b", "4"], capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "solve_batch 4 samples" in out.stdout and "ALL PASSED" in out.stdout


@pytest.mark.gpu
def test_same_capped_coverage_as_the_references_own_cuda_solver(solver, O, tmp_path):
    # quasi-mcp-cuda itself (libs/qmcp-solver/src/quasi_mcp_cuda_max_flow_solver.cu compiled
    # unmodified for sm_100a into oracle/_ref/libgds_refcuda.so) on the same box and input: kept
    # sets may differ (SURVEY finding 3), the M-capped output coverage may not.
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    runner = os.path.join(root, "oracle", "run_refcuda.py")
    if not os.path.exists(os.path.join(root, "oracle", "_ref", "libgds_refcuda.so")):
        pytest.skip("oracle/_ref/libgds_refcuda.so not built (needs /root/reference + nvcc)")
    ex = O.SMALL_EXAMPLE
    cases = [(ex["start"], ex["end"], ex["L"], ex["M"])]
    s, e, _, _ = O.gen_reads(12345, 50_000, 30_000, 150)   # config 3
    cases.append((s, e, 30_000, 100))
    for i, (s, e, L, M) in enumerate(cases):
        inp = tmp_path / ("in%d.npz" % i)
        outp = tmp_path / ("out%d.npy" % i)
        np.savez(inp, s=s, e=e, L=L)
        subprocess.run([sys.executable, runner, "npy", str(inp), str(outp), str(M)], check=True,
                       timeout=300, capture_output=True)
        ids = np.load(outp)
        ref_mask = np.zeros(len(s), np.uint8); ref_mask[ids] = 1
        r = solver.solve(s, e, L, M, verify=True)
        ours = O.bitmap_to_mask(r.kept_bitmap, len(s))
        cin = O.coverage_fast(s, e, L)
        c_ref = O.coverage_fast(s, e, L, ref_mask); c_us = O.coverage_fast(s, e, L, ours)
        assert np.all(np.minimum(cin, M) <= c_ref)          # the reference's own invariant
        assert np.array_equal(np.minimum(c_ref, M), np.minimum(c_us, M))
        assert np.array_equal(np.minimum(c_us, M), np.minimum(cin, M))


def test_host_amplicon_generator_matches_oracle(hostlib, O):
    bed, tsv = O.artic_scheme()
    a0, a1 = O.parse_amplicons(bed, tsv)
    h0, h1 = hostlib.artic_amplicons()
    assert np.array_equal(np.sort(a0), h0) and np.array_equal(np.sort(a1), h1)
    n = 40_000
    s = np.empty(n, np.uint32); e = np.empty(n, np.uint32)
    q = np.empty(n, np.uint8); l = np.empty(n, np.uint32)
    hostlib.gen_reads_amplicon_into(777, n // 2, 30_000, a0, a1, s, e, q, l)
    s0, e0, q0, l0 = O.gen_reads_amplicon(777, n // 2, 30_000, a0, a1)
    assert np.array_equal(s, s0) and np.array_equal(e, e0)
    assert np.array_equal(q, q0.astype(np.uint8)) and np.array_equal(l, l0)
