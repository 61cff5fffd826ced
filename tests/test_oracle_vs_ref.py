"""The project's restatements against the REFERENCE'S OWN outputs: tests/golden/make_golden.py
froze them in tests/golden/golden.json from a build of the reference's unmodified sources.
tests/test_oracle.py checks the oracle's generator and filter against the same entries; the tests
here check the host mirror's generators and BAM reader, the exact per-read coverage routine,
find_pairs on a bitmap, and the reference's CoverageTester against the oracle's solver."""
import hashlib

import numpy as np
import pytest

from conftest import PRM


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


SHAPE_NAMES = ["uniform", "low_sides", "hole", "zero_sides"]


@pytest.fixture(scope="module")
def hostlib(pkg):
    from genome_downsampler_b200 import hostlib
    hostlib.load()
    return hostlib


def test_generators_bit_exact(hostlib, golden):
    # the C++ host mirror of reads_gen.cpp, every stored stream and all four columns
    for name, g in sorted(golden["generators"].items()):
        n = 2 * g["pairs"]
        s = np.empty(n, np.uint32); e = np.empty(n, np.uint32)
        q = np.empty(n, np.uint8); l = np.empty(n, np.uint32)
        hostlib.gen_reads_into(g["seed"], g["pairs"], g["L"], g["R"], s, e, q, l,
                               shape=SHAPE_NAMES[g["shape"]])
        assert [sha(s), sha(e), sha(q.astype(np.uint32)), sha(l)] == \
            [g["start"], g["end"], g["quality"], g["seq_len"]], name


def test_cover_helpers_bit_exact(O, golden):
    # the exact per-read coverage (not coverage_fast) against BamApi::find_input_cover
    for name in ("small_uniform", "small_hole", "c3"):
        g = golden["generators"][name]
        s, e, q, l = O.gen_reads(g["seed"], g["pairs"], g["L"], g["R"], SHAPE_NAMES[g["shape"]])
        cov = O.coverage(s, e, g["L"])
        assert sha(cov) == g["cover"] and cov[:8].tolist() == g["cover_head"], name
        assert int(cov.sum()) == g["cover_sum"], name


def test_filter_matches_read_bam(hostlib, golden, tmp_path):
    # the host BAM reader's pair filter (BamApi(input_filepath, config)) on a BAM of the stored
    # input against the reference's BamApi::read_bam
    gf = golden["filter"]
    bedp, tsvp, path = tmp_path / "scheme.bed", tmp_path / "pairs.tsv", tmp_path / "in.bam"
    bedp.write_text(gf["bed"]); tsvp.write_text(gf["tsv"])
    a0, a1 = hostlib.artic_amplicons(gf["L"])
    n = 2 * gf["pairs"]
    s = np.empty(n, np.uint32); e = np.empty(n, np.uint32)
    q = np.empty(n, np.uint8); l = np.empty(n, np.uint32)
    hostlib.gen_reads_amplicon_into(gf["seed"], gf["pairs"], gf["L"], a0, a1, s, e, q, l)
    hostlib.write_synthetic_bam(path, gf["L"], s, e, q, l, coordinate_sorted=False, threads=2)
    for name, c in sorted(gf["cases"].items()):
        b = hostlib.BamFile(path, min_len=c["min_len"], min_mapq=c["min_mapq"],
                            bed=bedp if c["use_bed"] else None,
                            tsv=tsvp if c["use_bed"] and c["use_tsv"] else None, threads=2)
        got, out = b.reads(), b.filtered_out()
        b.close()
        assert len(got["bam_id"]) == c["n_kept"], name
        assert sha(got["bam_id"]) == c["bam_id"] and got["bam_id"][:10].tolist() == c["first_ids"], name
        assert sha(got["start"].astype(np.uint32)) == c["start"], name
        assert sha(got["end"].astype(np.uint32)) == c["end"], name
        assert sha(out) == c["filtered_out"], name


def test_find_pairs_bitmap_equals_reference_set(O, golden):
    ids = golden["small16"]["filtered_cover_ids"]
    bm = np.zeros(1, np.uint32)
    for i in ids:
        bm[0] |= np.uint32(1 << int(i))
    got = np.nonzero(O.bitmap_to_mask(O.find_pairs_bitmap(bm, 16), 16))[0]
    assert sorted(golden["small16"]["find_pairs"]) == got.tolist()


def test_reference_coverage_tester_accepts_oracle_solvers(O, coverage_tester):
    # CoverageTester::test (5 cases) through qmcp::Solver
    def sync(M, L, s, e):
        bm, st = O.sync_solve(s, e, [L], [0, len(s)], M, params=PRM)
        return np.nonzero(O.bitmap_to_mask(bm, len(s)))[0]
    assert coverage_tester(sync) == 5
