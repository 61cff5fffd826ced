"""GPU parity tests proper: every call goes through the C ABI (include/gds.h) and is compared
with the CPU oracle on the same seeded inputs — bit-exact for F*, demand vector, capped coverage,
kept bitmap (deterministic schedule) and even the round count."""
import hashlib

import numpy as np
import pytest

from conftest import PRM

pytestmark = pytest.mark.gpu


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def assert_parity(O, r, s, e, ref_lens, read_off, M, prm=PRM):
    bm, st, dem, cov = O.sync_solve(s, e, ref_lens, read_off, M, params=prm, want_vectors=True)
    assert r.fstar == st.fstar == r.flow_value == st.flow_value
    assert np.array_equal(r.demand, dem)
    assert np.array_equal(r.cov_capped, np.minimum(cov, M))
    assert r.n_bundles == st.n_bundles and r.n_components == st.n_components
    assert r.n_kept == st.n_kept
    assert np.array_equal(r.kept_bitmap, bm), "kept bitmap differs from the oracle"
    assert r.rounds_total == st.rounds_total and r.relabels == st.relabels
    assert r.pushes == st.pushes and r.bfs_levels == st.bfs_levels
    assert r.verify_violations == 0
    return st


def test_small_example(solver, O):
    ex = O.SMALL_EXAMPLE
    r = solver.solve(ex["start"], ex["end"], ex["L"], ex["M"], params=PRM, verify=True,
                     want_vectors=True)
    assert r.fstar == 5 and r.n_kept == 14
    assert r.demand.tolist() == [-3, -1, 0, 0, 0, 1, -1, 0, 0, 0, 1, 3]
    assert r.cov_capped.tolist() == [3, 4, 4, 4, 4, 3, 4, 4, 4, 4, 3, 0]
    assert_parity(O, r, ex["start"], ex["end"], [ex["L"]], [0, 16], ex["M"])


def test_fuzz_ragged_batches(solver, O):
    rng = np.random.default_rng(7)
    for it in range(120):
        ns = int(rng.integers(1, 6))
        Ls = rng.integers(1, 400, size=ns).astype(np.uint32)
        ss, ee, off = [], [], [0]
        for L in Ls:
            n = 2 * int(rng.integers(0, 300))  # empty samples happen
            mode = int(rng.integers(0, 3))
            if mode == 0:
                s = rng.integers(0, L, size=n); ln = rng.integers(1, max(2, L // 2 + 1), size=n)
            elif mode == 1:
                s = rng.integers(0, max(1, L // 3), size=n); ln = rng.integers(1, 6, size=n)
            else:
                s = rng.integers(0, L, size=n); ln = np.full(n, rng.integers(1, 30))
            e = np.minimum(s + ln - 1, L - 1)
            ss.append(s); ee.append(e); off.append(off[-1] + n)
        s = np.concatenate(ss).astype(np.uint32); e = np.concatenate(ee).astype(np.uint32)
        M = int(rng.integers(1, 12))
        # every third case also cuts the references into short segments (reads crossing a cut are
        # truncated into one arc per segment); seg_len below the longest read disables the split
        seg = int(rng.integers(1, 120)) if it % 3 == 0 else 0
        prm = (int(rng.integers(1, 100)), int(rng.integers(0, 300)), int(rng.integers(0, 5)), 0, seg)
        off = np.array(off, np.uint64)
        # both ways of finding the bundles (gds_params.bundle_mode: radix sort / direct histogram)
        for bmode in (1, 2):
            r = solver.solve(s, e, Ls, M, read_off=off, params=prm + (bmode,), verify=True,
                             want_vectors=True)
            assert_parity(O, r, s, e, Ls, off, M, prm)
            assert bmode == 2 or r.sort_passes > 0 or len(s) == 0


def test_segmented_reference_matches_oracle_and_unsplit_invariants(solver, O):
    # one 200 kb reference cut into 4 kb segments: F*, demand and capped coverage must equal the
    # unsplit solve bit for bit, the kept set must equal the oracle's replay of the same split
    s, e, q, l = O.gen_reads(777, 300_000, 200_000, 150)
    M = 40
    prm = (64, 150, 1, 0, 4096)
    r = solver.solve(s, e, 200_000, M, params=prm, verify=True, want_vectors=True)
    assert r.n_components >= 49 and r.n_arc_items > len(s)
    assert_parity(O, r, s, e, [200_000], [0, len(s)], M, prm)
    r0 = solver.solve(s, e, 200_000, M, params=(64, 150, 1, 0, 0xffffffff), verify=True,
                      want_vectors=True)
    assert r0.n_components == 1 and r0.n_arc_items == len(s)
    assert r.fstar == r0.fstar == r.flow_value == r0.flow_value
    assert np.array_equal(r.demand, r0.demand) and np.array_equal(r.cov_capped, r0.cov_capped)
    assert r0.n_kept <= r.n_kept <= 1.03 * r0.n_kept  # <= M extra reads per cut
    mask = O.bitmap_to_mask(r.kept_bitmap, len(s))
    assert int(mask.sum()) == r.n_kept
    cin = O.coverage_fast(s, e, 200_000); cout = O.coverage_fast(s, e, 200_000, mask)
    assert np.array_equal(np.minimum(cin, M), np.minimum(cout, M))


@pytest.mark.parametrize("name,pairs,M,shape", [
    ("c3", 50_000, 100, "uniform"), ("c1", 500_000, 100, "uniform"),
    ("ref_uniform", 1_000_000, 1000, "uniform"), ("ref_low_sides", 1_000_000, 8000, "low_sides"),
    ("ref_hole", 1_000_000, 8000, "hole"), ("ref_zero_sides", 1_000_000, 8000, "zero_sides")])
def test_configs_and_reference_shapes_full_size(solver, O, name, pairs, M, shape):
    # BASELINE configs C1, C3 and the reference's own 4 random cases (coverage_tester.cpp:120-175)
    s, e, q, l = O.gen_reads(12345, pairs, 30_000, 150, shape)
    r = solver.solve(s, e, 30_000, M, params=PRM, verify=True, want_vectors=True)
    st = assert_parity(O, r, s, e, [30_000], [0, len(s)], M)
    # the reference's only assertion (is_out_cover_valid), from the bitmap on the host
    mask = O.bitmap_to_mask(r.kept_bitmap, len(s))
    cin = O.coverage_fast(s, e, 30_000); cout = O.coverage_fast(s, e, 30_000, mask)
    assert np.all(np.minimum(cin, M) <= cout)
    if name == "c3":  # optimality vs the mcp-cpu objective (greedy multicover == min-cost optimum)
        _, nopt = O.greedy_multicover(s, e, 30_000, M)
        assert nopt <= r.n_kept <= 1.05 * nopt
    assert st.fstar == {"c3": 100, "c1": 100, "ref_uniform": 1000}.get(name, st.fstar)


def test_variable_lengths_64bit_keys_and_wide_nodes(solver, O):
    # lengths spread over 20 bits + 2^21 nodes -> key wider than 32 bits (u64 sort path)
    rng = np.random.default_rng(5)
    L = 2_000_000
    n = 40_000
    s = rng.integers(0, L - 1_000_001, size=n).astype(np.uint32)
    ln = rng.integers(1, 1_000_000, size=n)
    e = (s + ln - 1).astype(np.uint32)
    r = solver.solve(s, e, L, 7, params=PRM, verify=True, want_vectors=True)
    assert r.key_bits > 32
    assert_parity(O, r, s, e, [L], [0, n], 7)


def test_batch_of_samples(solver, O):
    parts = [O.gen_reads(12345 + k, 100_000, 30_000, 150) for k in range(6)]
    s = np.concatenate([p[0] for p in parts]); e = np.concatenate([p[1] for p in parts])
    off = np.arange(7, dtype=np.uint64) * 200_000
    r = solver.solve(s, e, [30_000] * 6, 100, read_off=off, params=PRM, verify=True,
                     want_vectors=True)
    assert r.n_components == 6
    assert_parity(O, r, s, e, [30_000] * 6, off, 100)
    # each sample's slice equals its stand-alone solve (sharding never changes results)
    mask = O.bitmap_to_mask(r.kept_bitmap, len(s))
    r0 = solver.solve(parts[3][0], parts[3][1], 30_000, 100, params=PRM)
    assert np.array_equal(O.bitmap_to_mask(r0.kept_bitmap, 200_000), mask[600_000:800_000])


def test_zero_coverage_cuts_make_components(solver, O):
    # three islands of reads separated by uncovered stretches -> 3 components (K4)
    parts = []
    for lo in (0, 10_000, 25_000):
        s, e, q, l = O.gen_reads(lo + 1, 4_000, 4_000, 100)
        parts.append((s + lo, e + lo))
    s = np.concatenate([p[0] for p in parts]).astype(np.uint32)
    e = np.concatenate([p[1] for p in parts]).astype(np.uint32)
    r = solver.solve(s, e, 30_000, 50, params=PRM, verify=True, want_vectors=True)
    assert r.n_components == 3
    assert_parity(O, r, s, e, [30_000], [0, len(s)], 50)


def test_filter_path_c2_small(solver, O):
    # config 2 at reduced size: -l 90 -q 30 + synthetic ARTIC BED/TSV, FILTER mode
    bed, tsv = O.artic_scheme()
    a0, a1 = O.parse_amplicons(bed, tsv)
    s, e, q, l = O.gen_reads_amplicon(12345, 250_000, 30_000, a0, a1)
    for filt in (dict(min_len=90, min_mapq=30, amp_start=a0, amp_end=a1),
                 dict(min_len=90, min_mapq=30), dict(min_len=0, min_mapq=0, amp_start=a0, amp_end=a1)):
        r = solver.solve(s, e, 30_000, 100, mapq=q.astype(np.uint8), seq_len=l, filt=filt,
                         params=PRM, verify=True, want_vectors=True)
        pp, kept = O.filter_pairs(s, e, q, l, filt["min_len"], filt["min_mapq"],
                                  filt.get("amp_start"), filt.get("amp_end"))
        assert np.array_equal(r.pair_pass, pp) and r.n_filtered == kept
        assert r.filt_off.tolist() == [0, kept]
        mask = np.repeat(pp, 2).astype(bool)
        fs, fe = s[mask].copy(), e[mask].copy()
        # a call with an amplicon table gets the graph reduction at every M (gds_params.schedule:
        # like 3), one without gets it from M = 128 on; schedule 1 is round 1's graph either way
        AMP = (64, 150, 1, 0, 0, 3)
        assert_parity(O, r, fs, fe, [30_000], [0, kept], 100, AMP if "amp_start" in filt else PRM)
        for M, prm, oprm in ((400, PRM, PRM), (100, (64, 150, 1, 0, 0, 0, 0, 3), AMP),
                             (100, (64, 150, 1, 0, 0, 0, 0, 1), (64, 150, 1, 0, 0, 1))):
            r = solver.solve(s, e, 30_000, M, mapq=q.astype(np.uint8), seq_len=l, filt=filt,
                             params=prm, verify=True, want_vectors=True)
            assert_parity(O, r, fs, fe, [30_000], [0, kept], M, oprm)


def test_c2_full_size_filter_and_solve(solver, O, golden):
    # BASELINE config 2 at full size: 10M reads, -l 90 -q 30, synthetic ARTIC BED/TSV, M=100.
    # The device filter must equal the oracle's AND the reference's own read_bam filter (golden.json
    # holds its output for the first 20k pairs of this stream); the solve is checked bit for bit.
    bed, tsv = O.artic_scheme()
    a0, a1 = O.parse_amplicons(bed, tsv)
    s, e, q, l = O.gen_reads_amplicon(12345, 5_000_000, 30_000, a0, a1)
    filt = dict(min_len=90, min_mapq=30, amp_start=a0, amp_end=a1)
    r = solver.solve(s, e, 30_000, 100, mapq=q.astype(np.uint8), seq_len=l, filt=filt, params=PRM,
                     verify=True, want_vectors=True)
    pp, kept = O.filter_pairs(s, e, q, l, 90, 30, a0, a1)
    assert np.array_equal(r.pair_pass, pp) and r.n_filtered == kept and 0 < kept < len(s)
    mask = np.repeat(pp, 2).astype(bool)
    assert_parity(O, r, s[mask].copy(), e[mask].copy(), [30_000], [0, kept], 100, (64, 150, 1, 0, 0, 3))
    gf = golden["filter"]
    ref = gf["cases"]["l90_q30_tsv"]
    assert (gf["seed"], gf["L"], gf["bed"], gf["tsv"]) == (12345, 30_000, bed, tsv)
    assert (ref["min_len"], ref["min_mapq"], ref["use_bed"], ref["use_tsv"]) == (90, 30, True, True)
    n_ref = 2 * gf["pairs"]
    dev = np.repeat(r.pair_pass[:n_ref // 2], 2).astype(bool)
    assert int(dev.sum()) == ref["n_kept"]
    assert sha(np.nonzero(dev)[0].astype(np.uint64)) == ref["bam_id"]
    assert sha(s[:n_ref][dev]) == ref["start"] and sha(e[:n_ref][dev]) == ref["end"]


def test_filter_on_batches_keeps_sample_offsets(solver, O):
    bed, tsv = O.artic_scheme()
    a0, a1 = O.parse_amplicons(bed, tsv)
    parts = [O.gen_reads_amplicon(50 + k, 20_000 + 1000 * k, 30_000, a0, a1) for k in range(3)]
    s, e, q, l = [np.concatenate([p[i] for p in parts]) for i in range(4)]
    off = np.cumsum([0] + [len(p[0]) for p in parts]).astype(np.uint64)
    filt = dict(min_len=90, min_mapq=30, amp_start=a0, amp_end=a1)
    r = solver.solve(s, e, [30_000] * 3, 40, read_off=off, mapq=q.astype(np.uint8), seq_len=l,
                     filt=filt, params=PRM, verify=True, want_vectors=True)
    pp, kept = O.filter_pairs(s, e, q, l, 90, 30, a0, a1)
    mask = np.repeat(pp, 2).astype(bool)
    foff = [0] + [int(mask[:int(o)].sum()) for o in off[1:]]
    assert r.filt_off.tolist() == foff
    assert_parity(O, r, s[mask].copy(), e[mask].copy(), [30_000] * 3, np.array(foff, np.uint64), 40,
                  (64, 150, 1, 0, 0, 3))


def test_edge_cases(solver, O, pkg):
    # no reads at all
    z = np.zeros(0, np.uint32)
    r = solver.solve(z, z, 100, 5, params=PRM, verify=True, want_vectors=True)
    assert r.n_kept == 0 and r.fstar == 0 and r.n_components == 0 and not r.demand.any()
    # one read, M larger than any coverage: keep everything
    s = np.array([3, 3, 3, 7], np.uint32); e = np.array([9, 9, 9, 7], np.uint32)
    r = solver.solve(s, e, 12, 1000, params=PRM, verify=True, want_vectors=True)
    assert r.n_kept == 4
    assert_parity(O, r, s, e, [12], [0, 4], 1000)
    # M = 0: nothing is required, nothing is kept
    r = solver.solve(s, e, 12, 0, params=PRM, verify=True)
    assert r.n_kept == 0 and r.fstar == 0
    # read touching both ends of the reference; L = 1
    r = solver.solve(np.array([0], np.uint32), np.array([0], np.uint32), 1, 1, params=PRM,
                     verify=True, want_vectors=True)
    assert r.n_kept == 1 and r.demand.tolist() == [-1, 1]
    # all reads identical (one bundle of multiplicity 5000), M = 17 -> lowest 17 indices kept
    s = np.full(5000, 10, np.uint32); e = np.full(5000, 60, np.uint32)
    r = solver.solve(s, e, 100, 17, params=PRM, verify=True)
    assert r.n_bundles == 1 and pkg.Solver.bitmap_to_indices(r.kept_bitmap, 5000).tolist() == \
        list(range(17))
    # out-of-range coordinates are rejected, not clamped (reference would write out of bounds)
    with pytest.raises(pkg.GdsError) as ei:
        solver.solve(np.array([5], np.uint32), np.array([100], np.uint32), 100, 3)
    assert ei.value.code == 2
    with pytest.raises(pkg.GdsError):
        solver.solve(np.array([9], np.uint32), np.array([4], np.uint32), 100, 3)
    # the context survives an error
    ex = O.SMALL_EXAMPLE
    assert solver.solve(ex["start"], ex["end"], ex["L"], ex["M"]).fstar == 5


def test_determinism_and_reuse(solver, O):
    # same instance re-entered (coverage_tester.cpp:28-43 calls solve 5x on one solver): identical
    s, e, q, l = O.gen_reads(99, 200_000, 30_000, 150, "hole")
    ref = None
    for i in range(4):
        r = solver.solve(s, e, 30_000, 1500, params=PRM)
        if ref is None:
            ref = r.kept_bitmap.copy()
        assert np.array_equal(ref, r.kept_bitmap)
        ex = O.SMALL_EXAMPLE  # interleave a different problem size
        assert solver.solve(ex["start"], ex["end"], ex["L"], ex["M"]).n_kept == 14


def test_find_pairs_flag(solver, O):
    s, e, q, l = O.gen_reads(4, 50_000, 30_000, 150)
    r1 = solver.solve(s, e, 30_000, 60, params=PRM)
    r2 = solver.solve(s, e, 30_000, 60, params=PRM, find_pairs=True)
    assert np.array_equal(O.find_pairs_bitmap(r1.kept_bitmap, len(s)), r2.kept_bitmap)


def test_c4_full_size_properties(solver, O):
    # BASELINE config 4: 50M reads / 5 Mb / M=500.  Size-independent properties at full size:
    # F* closed form, sink inflow == F*, on-device recomputed capped coverage equals the input's,
    # n_kept == total bundle flow; plus bit-exact bitmap against the oracle's replay.
    s, e, q, l = O.gen_reads(12345, 25_000_000, 5_000_000, 150)
    r = solver.solve(s, e, 5_000_000, 500, params=PRM, verify=True, want_vectors=True)
    assert r.fstar == 500 == r.flow_value and r.verify_violations == 0
    assert int(np.maximum(0, -r.demand.astype(np.int64)).sum()) == 500
    assert int(r.demand.astype(np.int64).sum()) == 0
    # the default segment rule (include/gds.h gds_params.seg_len): 295 segments of 16 950 positions
    # (113 reads) — all resident at once on a B200 — instead of 306 of 16 384
    assert r.seg_len == 16950 and r.n_components == 295
    # quality (SURVEY §8c P4): every read covers R positions, so no valid answer keeps fewer than
    # M*L/R reads; each of the 295 cuts may cost up to M more.  Within 1 % of that lower bound.
    lower = 500 * 5_000_000 / 150
    assert 0 <= r.n_kept - lower < 1000 + 294 * 500
    assert r.n_kept <= 1.01 * lower
    mask_bits = int(np.unpackbits(r.kept_bitmap.view(np.uint8)).sum())
    assert mask_bits == r.n_kept
    bm, st = O.sync_solve(s, e, [5_000_000], [0, len(s)], 500, params=PRM)
    assert np.array_equal(bm, r.kept_bitmap) and st.rounds_total == r.rounds_total


def test_chunked_host_pipeline_equals_one_call(pkg, solver, O):
    # two contexts, chunks of 2 samples: same bitmap as one gds_solve over the whole batch
    import torch
    parts = [O.gen_reads(500 + k, 16_000, 30_000, 150) for k in range(7)]
    s = np.concatenate([p[0] for p in parts]); e = np.concatenate([p[1] for p in parts])
    n_per = 32_000
    off = np.arange(8, dtype=np.uint64) * n_per
    r = solver.solve(s, e, [30_000] * 7, 40, read_off=off, params=PRM)
    hs = torch.from_numpy(s.view(np.int32)).pin_memory()
    he = torch.from_numpy(e.view(np.int32)).pin_memory()
    bm = torch.zeros(len(s) // 32 + 4, dtype=torch.int32, device="cuda")
    ch = pkg.ChunkedSolver(0)
    try:
        rs = ch.solve_host_batch(hs.data_ptr(), he.data_ptr(), off, [30_000] * 7, 40,
                                 bm.data_ptr(), chunk_samples=2, params=PRM)
    finally:
        ch.close()
    assert len(rs) == 4 and sum(int(x.n_kept) for x in rs) == r.n_kept
    got = bm[:len(s) // 32].cpu().numpy().view(np.uint32)
    assert np.array_equal(got, r.kept_bitmap)


def test_length_hints_fold_validation_into_the_sort(pkg, solver, O):
    # gds_reads.len_min/len_max: same answer as the stand-alone validation pass, one kernel fewer
    parts = [O.gen_reads(900 + k, 20_000, 30_000, 150) for k in range(3)]
    s = np.concatenate([p[0] for p in parts]); e = np.concatenate([p[1] for p in parts])
    off = np.arange(4, dtype=np.uint64) * 40_000
    r0 = solver.solve(s, e, [30_000] * 3, 30, read_off=off, params=PRM, verify=True)
    r1 = solver.solve(s, e, [30_000] * 3, 30, read_off=off, params=PRM, verify=True,
                      len_hint=(150, 150))
    assert np.array_equal(r0.kept_bitmap, r1.kept_bitmap) and r0.rounds_total == r1.rounds_total
    assert r1.kernel_launches < r0.kernel_launches and r1.verify_violations == 0
    # variable lengths with exact hints, single sample
    rng = np.random.default_rng(3)
    s2 = rng.integers(0, 29_000, size=50_000).astype(np.uint32)
    e2 = (s2 + rng.integers(59, 200, size=50_000)).astype(np.uint32)
    lens = e2 - s2 + 1
    ra = solver.solve(s2, e2, 30_000, 25, params=PRM)
    rb = solver.solve(s2, e2, 30_000, 25, params=PRM, len_hint=(int(lens.min()), int(lens.max())))
    assert np.array_equal(ra.kept_bitmap, rb.kept_bitmap)
    # a long reference (segmented path) honours hints too
    s3, e3, _, _ = O.gen_reads(5, 100_000, 100_000, 150)
    rc = solver.solve(s3, e3, 100_000, 40, params=(64, 150, 1, 0, 8192))
    rd = solver.solve(s3, e3, 100_000, 40, params=(64, 150, 1, 0, 8192), len_hint=(150, 150))
    assert np.array_equal(rc.kept_bitmap, rd.kept_bitmap) and rc.n_components == rd.n_components
    # hints that do not hold, and bad coordinates under hints, fail loudly
    with pytest.raises(pkg.GdsError) as ei:
        solver.solve(s2, e2, 30_000, 25, len_hint=(100, 120))
    assert ei.value.code == 1  # GDS_ERR_ARG
    bad = e.copy(); bad[77] = 30_000
    with pytest.raises(pkg.GdsError) as ei:
        solver.solve(s, bad, [30_000] * 3, 30, read_off=off, len_hint=(150, 151))
    assert ei.value.code == 2  # GDS_ERR_RANGE
    assert solver.solve(s, e, [30_000] * 3, 30, read_off=off, params=PRM).n_kept == r0.n_kept


def test_direct_histogram_path_equals_sort_path(solver, O):
    # gds_params.bundle_mode: 30 kb samples with one read length take the sort-free histogram by
    # default (sort_passes == 0); forcing the radix sort must give the same graph and kept set
    parts = [O.gen_reads(4242 + k, 150_000 + 7 * k, 30_000, 150, sh)
             for k, sh in enumerate(["uniform", "hole", "low_sides"])]
    s = np.concatenate([p[0] for p in parts]); e = np.concatenate([p[1] for p in parts])
    off = np.cumsum([0] + [len(p[0]) for p in parts]).astype(np.uint64)
    res = {}
    for bmode in (0, 1, 2):
        res[bmode] = solver.solve(s, e, [30_000] * 3, 300, read_off=off, params=PRM + (0, bmode),
                                  verify=True, want_vectors=True)
    assert res[0].sort_passes == 0 and res[2].sort_passes == 0 and res[1].sort_passes > 0
    for bmode in (0, 2):
        for key in ("fstar", "flow_value", "n_bundles", "n_components", "n_kept", "rounds_total",
                    "pushes", "relabels", "bfs_levels"):
            assert res[bmode][key] == res[1][key], key
        assert np.array_equal(res[bmode].kept_bitmap, res[1].kept_bitmap)
        assert np.array_equal(res[bmode].demand, res[1].demand)
        assert np.array_equal(res[bmode].cov_capped, res[1].cov_capped)
    assert_parity(O, res[0], s, e, [30_000] * 3, off, 300)
    # K5 of the histogram path has two implementations (parallel mark + partial-bundle ranking,
    # and the ordered walk it falls back to): same kept set
    import os
    os.environ["GDS_DIRECT_SELECT"] = "walk"
    try:
        rw = solver.solve(s, e, [30_000] * 3, 300, read_off=off, params=PRM + (0, 2), verify=True)
    finally:
        del os.environ["GDS_DIRECT_SELECT"]
    assert rw.sort_passes == 0 and rw.n_kept == res[1].n_kept and rw.verify_violations == 0
    assert np.array_equal(rw.kept_bitmap, res[1].kept_bitmap)
    # a few read lengths (key = start x #lengths + length) still fit in shared memory
    rng = np.random.default_rng(11)
    s2 = rng.integers(0, 9_000, size=400_000).astype(np.uint32)
    e2 = (s2 + rng.integers(148, 152, size=400_000)).astype(np.uint32)
    ra = solver.solve(s2, e2, 9_200, 200, params=PRM + (0, 2), verify=True, want_vectors=True)
    rb = solver.solve(s2, e2, 9_200, 200, params=PRM + (0, 1), verify=True, want_vectors=True)
    assert ra.sort_passes == 0 and rb.sort_passes > 0
    assert np.array_equal(ra.kept_bitmap, rb.kept_bitmap) and ra.rounds_total == rb.rounds_total
    assert_parity(O, ra, s2, e2, [9_200], [0, len(s2)], 200)
    assert ra.bundle_path == 1 and rb.bundle_path == 0
    # a key space beyond shared memory keeps its counters in global memory (L2): same answer again
    e3 = (s2 + rng.integers(100, 300, size=400_000)).astype(np.uint32)
    rc = solver.solve(s2, e3, 9_400, 50, params=PRM + (0, 0), verify=True, want_vectors=True)
    rd = solver.solve(s2, e3, 9_400, 50, params=PRM + (0, 1), verify=True)
    assert rc.bundle_path == 2 and rc.sort_passes == 0 and rd.bundle_path == 0
    assert np.array_equal(rc.kept_bitmap, rd.kept_bitmap) and rc.rounds_total == rd.rounds_total
    assert rc.n_bundles == rd.n_bundles and rc.verify_violations == 0
    assert_parity(O, rc, s2, e3, [9_400], [0, len(s2)], 50)
    # and so does a segmented reference (reads crossing a cut count twice), batched with a short one
    s4, e4, _, _ = O.gen_reads(77, 120_000, 150_000, 150)
    s5, e5, _, _ = O.gen_reads(78, 30_000, 20_000, 150)
    sb = np.concatenate([s4, s5]); eb = np.concatenate([e4, e5])
    offb = np.array([0, len(s4), len(s4) + len(s5)], np.uint64)
    prm_seg = (64, 150, 1, 0, 8192)
    re = solver.solve(sb, eb, [150_000, 20_000], 60, read_off=offb, params=prm_seg + (0,), verify=True,
                      want_vectors=True)
    rf = solver.solve(sb, eb, [150_000, 20_000], 60, read_off=offb, params=prm_seg + (1,), verify=True)
    assert re.bundle_path == 2 and rf.bundle_path == 0 and re.n_arc_items == rf.n_arc_items > len(sb)
    assert np.array_equal(re.kept_bitmap, rf.kept_bitmap) and re.n_kept == rf.n_kept
    assert re.n_components == rf.n_components and re.pushes == rf.pushes
    assert_parity(O, re, sb, eb, [150_000, 20_000], offb, 60, prm_seg)


def test_direct_selection_walk_many_tiles_and_duplicates(solver, O):
    # the ordered walk of K5 (direct path): tiny key spaces so that every 4096-read tile holds many
    # reads of one key, quotas that run out in the middle of a tile or span several tiles, ragged
    # sample offsets (unaligned 16-byte loads at part boundaries)
    rng = np.random.default_rng(23)
    for it in range(40):
        ns = int(rng.integers(1, 4))
        Ls = rng.integers(2, 60, size=ns).astype(np.uint32)
        ss, ee, off = [], [], [0]
        for L in Ls:
            n = int(rng.integers(0, 30_000))
            nl = int(rng.integers(1, 4))
            s = rng.integers(0, L, size=n)
            e = np.minimum(s + rng.integers(1, 1 + nl, size=n) * int(rng.integers(1, 8)) - 1, L - 1)
            ss.append(s); ee.append(e); off.append(off[-1] + n)
        s = np.concatenate(ss).astype(np.uint32); e = np.concatenate(ee).astype(np.uint32)
        M = int(rng.choice([1, 3, 50, 700, 5000, 20000]))
        off = np.array(off, np.uint64)
        r = solver.solve(s, e, Ls, M, read_off=off, params=PRM + (0, 2), verify=True,
                         want_vectors=True)
        assert r.sort_passes == 0 or len(s) == 0
        assert_parity(O, r, s, e, Ls, off, M)
        if it % 4 == 0:  # and the ordered walk on the same input
            import os
            os.environ["GDS_DIRECT_SELECT"] = "walk"
            try:
                rw = solver.solve(s, e, Ls, M, read_off=off, params=PRM + (0, 2), verify=True)
            finally:
                del os.environ["GDS_DIRECT_SELECT"]
            assert np.array_equal(rw.kept_bitmap, r.kept_bitmap) and rw.n_kept == r.n_kept


def test_compact_transport_start16_and_implied_end(pkg, solver, O):
    # gds_reads.start16 / end == NULL: same answer as the 32-bit columns, 2 bytes per read over PCIe
    parts = [O.gen_reads(7000 + k, 30_000 + 16 * k, 30_000, 150) for k in range(3)]
    s = np.concatenate([p[0] for p in parts]); e = np.concatenate([p[1] for p in parts])
    off = np.cumsum([0] + [len(p[0]) for p in parts]).astype(np.uint64)
    Ls = [30_000] * 3
    r0 = solver.solve(s, e, Ls, 40, read_off=off, params=PRM, verify=True, want_vectors=True)
    r1 = solver.solve(s, None, Ls, 40, read_off=off, params=PRM, verify=True, want_vectors=True,
                      len_hint=(150, 150))
    r2 = solver.solve(s.astype(np.uint16), None, Ls, 40, read_off=off, params=PRM, verify=True,
                      want_vectors=True, len_hint=(150, 150))
    r3 = solver.solve(s.astype(np.uint16), e, Ls, 40, read_off=off, params=PRM + (0, 1), verify=True)
    for r in (r1, r2, r3):
        assert np.array_equal(r.kept_bitmap, r0.kept_bitmap) and r.n_kept == r0.n_kept
        assert r.verify_violations == 0 and r.fstar == r0.fstar
    assert np.array_equal(r2.cov_capped, r0.cov_capped) and np.array_equal(r2.demand, r0.demand)
    assert_parity(O, r2, s, e, Ls, off, 40)
    # odd sizes (the widening kernel's scalar tail) and a long reference with implied ends
    s4, e4, _, _ = O.gen_reads(5, 50_003, 100_000, 150)
    s4, e4 = s4[:100_003].copy(), e4[:100_003].copy()
    ra = solver.solve(s4, e4, 100_000, 40, params=PRM)
    rb = solver.solve(s4, None, 100_000, 40, params=PRM, len_hint=(150, 150))
    assert np.array_equal(ra.kept_bitmap, rb.kept_bitmap)
    # errors: end omitted without a fixed length, 16-bit starts on a long reference, bad range
    with pytest.raises(pkg.GdsError) as ei:
        solver.solve(s, None, Ls, 40, read_off=off)
    assert ei.value.code == 1
    with pytest.raises(pkg.GdsError) as ei:
        solver.solve(s4.astype(np.uint16), None, 100_000, 40, len_hint=(150, 150))
    assert ei.value.code == 1
    bad = s.astype(np.uint16); bad[5] = 29_990
    with pytest.raises(pkg.GdsError) as ei:
        solver.solve(bad, None, Ls, 40, read_off=off, len_hint=(150, 150))
    assert ei.value.code == 2
    # chunked host pipeline with the compact columns
    import torch
    n32 = (len(s) // 32) * 32
    parts = [O.gen_reads(8100 + k, 16_000, 30_000, 150) for k in range(5)]
    s5 = np.concatenate([p[0] for p in parts]); e5 = np.concatenate([p[1] for p in parts])
    off5 = np.arange(6, dtype=np.uint64) * 32_000
    r5 = solver.solve(s5, e5, [30_000] * 5, 40, read_off=off5, params=PRM)
    h16 = torch.from_numpy(s5.astype(np.uint16).view(np.int16)).pin_memory()
    bm = torch.zeros(len(s5) // 32 + 4, dtype=torch.int32, device="cuda")
    ch = pkg.ChunkedSolver(0)
    try:
        rs = ch.solve_host_batch(None, None, off5, [30_000] * 5, 40, bm.data_ptr(), chunk_samples=2,
                                 params=PRM, len_hint=(150, 150), start16_ptr=h16.data_ptr())
    finally:
        ch.close()
    assert sum(int(x.n_kept) for x in rs) == r5.n_kept
    assert np.array_equal(bm[:len(s5) // 32].cpu().numpy().view(np.uint32), r5.kept_bitmap)


def test_c5_shape_batch_parity(solver, O):
    # BASELINE config 5 at its real per-sample shape: 8 samples x 2 M reads / 30 kb / M=100, seeds
    # 12345+k (what bench.py's default workload runs 512 of), one gds_solve, bit-exact against the
    # oracle's replay; every sample's slice equals its stand-alone solve
    ns, pairs = 8, 1_000_000
    parts = [O.gen_reads(12345 + k, pairs, 30_000, 150) for k in range(ns)]
    s = np.concatenate([p[0] for p in parts]); e = np.concatenate([p[1] for p in parts])
    off = np.arange(ns + 1, dtype=np.uint64) * (2 * pairs)
    r = solver.solve(s, e, [30_000] * ns, 100, read_off=off, params=PRM, verify=True,
                     want_vectors=True, len_hint=(150, 150))
    assert r.n_components == ns and r.fstar == 100 * ns and r.bundle_path == 1
    assert_parity(O, r, s, e, [30_000] * ns, off, 100)
    mask = O.bitmap_to_mask(r.kept_bitmap, len(s))
    for k in (0, 5, 7):
        rk = solver.solve(parts[k][0], parts[k][1], 30_000, 100, params=PRM)
        lo = k * 2 * pairs
        assert np.array_equal(O.bitmap_to_mask(rk.kept_bitmap, 2 * pairs), mask[lo:lo + 2 * pairs])
    # the compact transport bench.py's e2e leg uses (16-bit starts, implied ends): same bits
    rc = solver.solve(s.astype(np.uint16), None, [30_000] * ns, 100, read_off=off, params=PRM,
                      len_hint=(150, 150))
    assert np.array_equal(rc.kept_bitmap, r.kept_bitmap)


def _solve_with_env(solver, env, *a, **kw):
    import os
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        return solver.solve(*a, **kw)
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v


COUNTERS = ("fstar", "flow_value", "n_bundles", "n_components", "n_kept", "rounds_total", "pushes",
            "relabels", "bfs_levels", "global_relabels", "max_frontier")


def test_maxflow_kernels_agree(solver, O):
    # K3 exists twice: state in shared memory (maxflow_sm.cuh, default) and state in global memory
    # (maxflow.cuh: GDS_MF=global, and the fallback for components the first cannot take).  Same
    # deterministic schedule: every counter and the bitmap must be identical, and equal the oracle.
    cases = []
    s, e, _, _ = O.gen_reads(31, 150_000, 30_000, 150, "hole")
    cases.append((s, e, [30_000], np.array([0, len(s)], np.uint64), 3000, PRM))
    rng = np.random.default_rng(17)
    s2 = rng.integers(0, 29_000, size=300_000).astype(np.uint32)
    e2 = (s2 + rng.integers(60, 200, size=300_000)).astype(np.uint32)  # heavy nodes: warp mode
    cases.append((s2, e2, [30_000], np.array([0, len(s2)], np.uint64), 80, PRM))
    s3, e3, _, _ = O.gen_reads(32, 200_000, 120_000, 150)  # 8 kb segments: many small components
    cases.append((s3, e3, [120_000], np.array([0, len(s3)], np.uint64), 60, (16, 50, 1, 0, 8192)))
    for s, e, Ls, off, M, prm in cases:
        a = solver.solve(s, e, Ls, M, read_off=off, params=prm, verify=True, want_vectors=True)
        b = _solve_with_env(solver, {"GDS_MF": "global"}, s, e, Ls, M, read_off=off, params=prm,
                            verify=True)
        c = _solve_with_env(solver, {"GDS_MF_OPTR": "0"}, s, e, Ls, M, read_off=off, params=prm)
        # heavy components stay in the shared-memory kernel (its warp passes) instead of k_maxflow
        d = _solve_with_env(solver, {"GDS_MF_WARP": "1", "GDS_SYNC": "1"}, s, e, Ls, M, read_off=off,
                            params=prm)
        for key in COUNTERS:
            assert a[key] == b[key] == c[key] == d[key], key
        assert np.array_equal(a.kept_bitmap, d.kept_bitmap)
        assert np.array_equal(a.kept_bitmap, b.kept_bitmap)
        assert np.array_equal(a.kept_bitmap, c.kept_bitmap)
        assert_parity(O, a, s, e, Ls, off, M, prm)


def test_express_schedule_parity(solver, O):
    # segments of a cut reference run the express schedule in k_maxflow_sm (zero-length back arcs,
    # walks past saturated nodes, closed BFS levels): bit-exact against the oracle's replay, for the
    # default rule, for "classic only", and next to whole samples in the same batch
    L, M = 200_000, 500
    s, e, _, _ = O.gen_reads(7, int(L * 1500 / 150 / 2), L, 150)
    off = np.array([0, len(s)], np.uint64)
    res = {}
    for sched in (0, 1):
        prm = (64, 150, 1, 0, 0, 0, 0, sched)
        r = solver.solve(s, e, [L], M, read_off=off, params=prm, verify=True, want_vectors=True)
        st = assert_parity(O, r, s, e, [L], off, M, (64, 150, 1, 0, 0, sched))
        assert (st.n_express > 0) == (sched == 0)
        res[sched] = r
    assert res[0].rounds_total * 2 < res[1].rounds_total and res[0].n_kept != 0
    # a hole inside some segments (classic there), a whole sample next to the cut one, M = 1000
    s3, e3, _, _ = O.gen_reads(9, 400_000, 100_000, 150, "hole")
    s4, e4, _, _ = O.gen_reads(10, 100_000, 30_000, 150)
    sb = np.concatenate([s3, s4]); eb = np.concatenate([e3, e4])
    offb = np.array([0, len(s3), len(sb)], np.uint64)
    r = solver.solve(sb, eb, [100_000, 30_000], 1000, read_off=offb, params=PRM, verify=True,
                     want_vectors=True)
    st = assert_parity(O, r, sb, eb, [100_000, 30_000], offb, 1000)
    assert 0 < st.n_express < st.n_components
    # the whole sample's bits do not depend on the company it keeps
    alone = solver.solve(s4, e4, [30_000], 1000, params=PRM)
    n3 = len(s3)
    assert n3 % 32 == 0
    assert np.array_equal(r.kept_bitmap[n3 // 32:], alone.kept_bitmap)
    # short segments, variable read lengths (heavy cut nodes, several bundles per node)
    rng = np.random.default_rng(23)
    s5 = rng.integers(0, 59_000, size=400_000).astype(np.uint32)
    e5 = (s5 + rng.integers(100, 160, size=400_000)).astype(np.uint32)
    for prm in ((16, 50, 1, 0, 4096), (64, 150, 1, 0, 8192, 0, 0, 2)):
        r = solver.solve(s5, e5, [60_000], 300, params=prm, verify=True, want_vectors=True)
        oprm = prm[:5] + ((prm[7],) if len(prm) > 5 else ())
        assert_parity(O, r, s5, e5, [60_000], [0, len(s5)], 300, oprm)


def test_forced_reads_out_and_cuts(solver, O):
    # from M = 128 on, bundles that cover a position with cov <= M leave the network with their
    # flow fixed and the components are cut at those positions (graph.cuh); what remains runs the
    # express schedule.  Bit-exact against the oracle; the reference's hard shapes need hops.
    for shape, M, max_rounds in (("hole", 8000, 400), ("zero_sides", 8000, 300), ("low_sides", 8000, 600)):
        s, e, _, _ = O.gen_reads(12345, 1_000_000, 30_000, 150, shape)
        off = np.array([0, len(s)], np.uint64)
        r = solver.solve(s, e, [30_000], M, read_off=off, params=PRM, verify=True, want_vectors=True)
        st = assert_parity(O, r, s, e, [30_000], off, M)
        assert st.n_express >= 1 and r.rounds_max < max_rounds, (shape, r.rounds_max)
        # schedule 1 = round 1's graph and schedule: the same F*, demand, capped coverage; a valid
        # answer of (nearly) the same size, thousands of rounds
        r1 = solver.solve(s, e, [30_000], M, read_off=off, params=(64, 150, 1, 0, 0, 0, 0, 1), verify=True,
                          want_vectors=True)
        assert_parity(O, r1, s, e, [30_000], off, M, (64, 150, 1, 0, 0, 1))
        assert r1.fstar == r.fstar and np.array_equal(r1.demand, r.demand)
        assert r1.rounds_max > 4 * r.rounds_max and abs(int(r1.n_kept) - int(r.n_kept)) <= 0.001 * r.n_kept
    # schedule 3: the reduction below M = 128 too (classic schedule there): amplicon-like dips
    s, e, _, _ = O.gen_reads(21, 300_000, 30_000, 150, "hole")
    r3 = solver.solve(s, e, [30_000], 100, params=(64, 150, 1, 0, 0, 0, 0, 3), verify=True, want_vectors=True)
    st3 = assert_parity(O, r3, s, e, [30_000], [0, len(s)], 100, (64, 150, 1, 0, 0, 3))
    r0 = solver.solve(s, e, [30_000], 100, params=PRM, verify=True, want_vectors=True)
    assert st3.n_express == 0 and r3.n_components >= r0.n_components and r3.fstar == r0.fstar
    # M above the coverage everywhere: every read is forced, nothing is left to solve
    s, e, _, _ = O.gen_reads(5, 50_000, 30_000, 150)
    r = solver.solve(s, e, [30_000], 5000, params=PRM, verify=True, want_vectors=True)
    assert r.n_components == 0 and r.n_kept == len(s) and r.rounds_total == 0
    assert_parity(O, r, s, e, [30_000], [0, len(s)], 5000)
    # a cut reference with a hole, short segments, next to a whole sample, several read lengths
    rng = np.random.default_rng(3)
    s2, e2, _, _ = O.gen_reads(9, 300_000, 90_000, 150, "hole")
    e2 = np.maximum(s2, e2 - rng.integers(0, 30, size=len(e2)).astype(np.uint32))
    s3, e3, _, _ = O.gen_reads(10, 100_000, 30_000, 150, "low_sides")
    sb = np.concatenate([s2, s3]); eb = np.concatenate([e2, e3])
    offb = np.array([0, len(s2), len(sb)], np.uint64)
    for prm in (PRM, (64, 150, 1, 0, 8192), (16, 50, 1, 0, 8192, 0, 0, 2)):
        r = solver.solve(sb, eb, [90_000, 30_000], 400, read_off=offb, params=prm, verify=True,
                         want_vectors=True)
        oprm = prm[:5] + ((prm[7],) if len(prm) > 5 else ())
        assert_parity(O, r, sb, eb, [90_000, 30_000], offb, 400, oprm)


def test_maxflow_fallback_list(solver, O):
    # components the shared-memory kernel cannot take go to k_maxflow through a device-side list:
    # (a) supply beyond 16 bits (M above the coverage: every rise of the coverage is a source);
    # (b) a component too long for one SM next to ones that fit
    s, e, _, _ = O.gen_reads(41, 1_000_000, 30_000, 150)
    sa, ea, _, _ = O.gen_reads(42, 100_000, 30_000, 150)
    sb = np.concatenate([s, sa]); eb = np.concatenate([e, ea])
    off = np.array([0, len(s), len(sb)], np.uint64)
    r = solver.solve(sb, eb, [30_000, 30_000], 100_000, read_off=off, params=PRM, verify=True,
                     want_vectors=True)
    assert r.fstar > 65535 and r.n_kept == len(sb)  # M above every coverage: everything is kept
    assert_parity(O, r, sb, eb, [30_000, 30_000], off, 100_000)
    s2, e2, _, _ = O.gen_reads(43, 150_000, 90_000, 150)
    s3, e3, _, _ = O.gen_reads(44, 50_000, 20_000, 150)
    sc = np.concatenate([s2, s3]); ec = np.concatenate([e2, e3])
    offc = np.array([0, len(s2), len(sc)], np.uint64)
    prm = (64, 150, 1, 0, 0xffffffff)  # no segmentation: a 90 001-node component
    r2 = solver.solve(sc, ec, [90_000, 20_000], 30, read_off=offc, params=prm, verify=True,
                      want_vectors=True)
    assert r2.n_components == 2
    assert_parity(O, r2, sc, ec, [90_000, 20_000], offc, 30, prm)


def test_zero_length_reads_are_accepted_and_never_kept(solver, O, pkg):
    # a read that consumes no reference (end == start - 1: CIGAR '*', an unmapped mate placed at its
    # mate's position) is legal in the reference (read.cpp:5-14; its arc is a self-loop without
    # flow).  Every bundle path must take it, cover nothing with it and never keep it.
    rng = np.random.default_rng(29)
    s, e, _, _ = O.gen_reads(77, 40_000, 9_000, 150)
    s = s.copy(); e = e.copy()
    idx = rng.choice(len(s), size=600, replace=False)
    e[idx] = s[idx] - np.uint32(1)            # includes wrap-around when a start is 0
    s[idx[0]] = 0; e[idx[0]] = np.uint32(0xffffffff)
    for prm in (PRM + (0, 0), PRM + (0, 1), PRM + (0, 2), (64, 150, 1, 0, 2048, 0), (64, 150, 1, 0, 2048, 1)):
        r = solver.solve(s, e, 9_000, 30, params=prm, verify=True, want_vectors=True)
        assert_parity(O, r, s, e, [9_000], [0, len(s)], 30, prm[:5])
        mask = O.bitmap_to_mask(r.kept_bitmap, len(s))
        assert not mask[idx].any()
        cov = O.coverage_fast(s, e, 9_000)
        assert np.array_equal(r.cov_capped[:9_000], np.minimum(cov, 30))
    # only such reads: nothing to cover, nothing kept
    z = np.array([5, 7], np.uint32)
    r = solver.solve(z, z - np.uint32(1), 100, 3, params=PRM, verify=True)
    assert r.n_kept == 0 and r.fstar == 0
    # still out of range: a zero-length read at or beyond the end, and end < start - 1
    with pytest.raises(pkg.GdsError) as ei:
        solver.solve(np.array([100], np.uint32), np.array([99], np.uint32), 100, 3)
    assert ei.value.code == 2
    with pytest.raises(pkg.GdsError):
        solver.solve(np.array([9], np.uint32), np.array([7], np.uint32), 100, 3)


def assert_sweep_parity(O, r, s, e, ref_lens, read_off, M, prm):
    bm, st, dem, cov = O.sweep_solve(s, e, ref_lens, read_off, M, params=prm[:5], want_vectors=True)
    assert r.fstar == st.fstar == r.flow_value
    assert np.array_equal(r.demand, dem) and np.array_equal(r.cov_capped, np.minimum(cov, M))
    assert r.n_bundles == st.n_bundles and r.n_components == st.n_components
    assert r.n_kept == st.n_kept and np.array_equal(r.kept_bitmap, bm), "kept set differs from the oracle's sweep"
    assert r.verify_violations == 0 and r.rounds_total == 0
    return st


def test_minimum_cardinality_sweep(solver, O):
    # gds_params.algorithm = 1: mcp-cpu's objective (fewest reads) by the device sweep.  Bit-exact
    # against the oracle's restatement of the sweep; the kept count equals the greedy-multicover
    # optimum (== network-simplex optimum, tests/test_oracle.py) whenever nothing is segmented; same
    # F*, demand and capped coverage as the push-relabel solve; never more reads than it keeps.
    NOSEG = 0xffffffff
    cases = []
    for seed, (pairs, L, R, M, shape) in enumerate([(50_000, 30_000, 150, 100, "uniform"),
                                                    (200_000, 30_000, 150, 3000, "hole"),
                                                    (30_000, 9_000, 60, 17, "low_sides")]):
        s, e, _, _ = O.gen_reads(500 + seed, pairs, L, R, shape)
        cases.append((s, e, [L], np.array([0, len(s)], np.uint64), M))
    rng = np.random.default_rng(71)
    s2 = rng.integers(0, 29_000, size=300_000).astype(np.uint32)
    e2 = (s2 + rng.integers(60, 200, size=300_000)).astype(np.uint32)  # 140 read lengths
    cases.append((s2, e2, [30_000], np.array([0, len(s2)], np.uint64), 80))
    s3 = rng.integers(0, 5_000, size=60_000).astype(np.uint32)
    e3 = np.minimum(s3 + rng.integers(1, 900, size=60_000) - 1, 4_999).astype(np.uint32)  # ring 1024
    cases.append((s3, e3, [5_000], np.array([0, len(s3)], np.uint64), 25))
    for s, e, Ls, off, M in cases:
        for bmode in (0, 1):
            prm = (64, 150, 1, 0, NOSEG, bmode, 1)
            r = solver.solve(s, e, Ls, M, read_off=off, params=prm, verify=True, want_vectors=True)
            st = assert_sweep_parity(O, r, s, e, Ls, off, M, prm)
        _, nopt = O.greedy_multicover(s, e, Ls[0], M)
        assert r.n_kept == nopt
        r0 = solver.solve(s, e, Ls, M, read_off=off, params=(64, 150, 1, 0, NOSEG), verify=True,
                          want_vectors=True)
        assert r0.fstar == r.fstar and np.array_equal(r0.demand, r.demand) and r.n_kept <= r0.n_kept
    # a batch of samples, zero-length reads, and a segmented reference (every segment swept alone)
    parts = [O.gen_reads(900 + k, 30_000 + 64 * k, 30_000, 150) for k in range(5)]
    s = np.concatenate([p[0] for p in parts]).copy(); e = np.concatenate([p[1] for p in parts]).copy()
    e[::997] = s[::997] - np.uint32(1)
    off = np.cumsum([0] + [len(p[0]) for p in parts]).astype(np.uint64)
    prm = (64, 150, 1, 0, NOSEG, 0, 1)
    r = solver.solve(s, e, [30_000] * 5, 60, read_off=off, params=prm, verify=True, want_vectors=True,
                     len_hint=None)
    assert_sweep_parity(O, r, s, e, [30_000] * 5, off, 60, prm)
    s4, e4, _, _ = O.gen_reads(33, 150_000, 150_000, 150)
    prm = (64, 150, 1, 0, 8192, 0, 1)
    r = solver.solve(s4, e4, 150_000, 40, params=prm, verify=True, want_vectors=True, len_hint=(150, 150))
    st = assert_sweep_parity(O, r, s4, e4, [150_000], [0, len(s4)], 40, prm)
    _, nopt = O.greedy_multicover(s4, e4, 150_000, 40)
    assert nopt <= r.n_kept <= nopt + 40 * (st.n_components - 1)  # at most M reads per cut
    # too long a read for the shared-memory ring: refused, not mis-solved
    import pytest as _pt
    from __graft_entry__ import load_package
    with _pt.raises(load_package().GdsError):
        solver.solve(np.array([0], np.uint32), np.array([4999], np.uint32), 6000, 1,
                     params=(64, 150, 1, 0, NOSEG, 0, 1))
