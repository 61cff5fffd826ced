"""gds_kernel_profile (bench.py's roofline reads it): on every solve path each kernel launch is
profiled under a name, the profile accounts for every launch gds_result.kernel_launches counts,
and profiling does not change the answer."""
import os

import numpy as np
import pytest

from conftest import PRM

pytestmark = pytest.mark.gpu


def _cases(O):
    parts = [O.gen_reads(610 + k, 20_000, 30_000, 150) for k in range(3)]
    s = np.concatenate([p[0] for p in parts]); e = np.concatenate([p[1] for p in parts])
    off = np.arange(4, dtype=np.uint64) * 40_000
    batch = dict(start=s, end=e, ref_len=[30_000] * 3, read_off=off)
    sl, el, _, _ = O.gen_reads(620, 120_000, 150_000, 150)
    seg = dict(start=sl, end=el, ref_len=150_000)
    # reads of 150, 151 and 152 positions: several lengths take the global-memory histogram, which
    # reads the bundle count and the input verdict back in the middle of the call
    sv, ev, _, _ = O.gen_reads(640, 40_000, 15_000, 150)
    ev = np.where(ev + 2 < 15_000, ev + np.arange(len(ev)) % 3, ev).astype(np.uint32)
    several = dict(start=sv, end=ev, ref_len=15_000)
    bed, tsv = O.artic_scheme()
    a0, a1 = O.parse_amplicons(bed, tsv)
    sf, ef, q, ln = O.gen_reads_amplicon(630, 50_000, 30_000, a0, a1)
    filt = dict(start=sf, end=ef, ref_len=30_000, mapq=q.astype(np.uint8), seq_len=ln,
                filt=dict(min_len=90, min_mapq=30, amp_start=a0, amp_end=a1))
    # name: (inputs, M, solve keywords, environment)
    return {
        "radix_sort": (batch, 60, dict(params=PRM + (0, 1)), {}),
        "direct_one_length": (batch, 60, dict(params=PRM + (0, 2), len_hint=(150, 150)), {}),
        "global_several_lengths": (several, 60, dict(params=PRM + (0, 2), len_hint=(150, 152)), {}),
        "global_hist_segmented": (seg, 60, dict(params=(64, 150, 1, 0, 8192, 0)), {}),
        "pair_filter": (filt, 100, dict(params=PRM), {}),
        "maxflow_global": (batch, 60, dict(params=PRM), {"GDS_MF": "global"}),
        "express": (batch, 400, dict(params=PRM), {}),
        "min_cardinality": (batch, 60, dict(params=PRM + (0, 0, 1)), {}),
    }


PATHS = ["radix_sort", "direct_one_length", "global_several_lengths", "global_hist_segmented",
         "pair_filter", "maxflow_global", "express", "min_cardinality"]


@pytest.mark.parametrize("path", PATHS)
def test_profile_accounts_for_every_launch(solver, O, path):
    inputs, M, kw, env = _cases(O)[path]
    inputs = dict(inputs)
    args = (inputs.pop("start"), inputs.pop("end"), inputs.pop("ref_len"), M)
    os.environ.update(env)
    try:
        plain = solver.solve(*args, verify=True, **inputs, **kw)
        solver.kernel_profile_reset()
        prof = solver.solve(*args, verify=True, profile=True, **inputs, **kw)
        stats = solver.kernel_profile()
    finally:
        for k in env:
            del os.environ[k]
    assert prof.kernel_launches > 0
    # (the two calls' launch counts may differ: a histogram path repeats its selection once when the
    # context's candidate buffer is still smaller than the call needs)
    assert sum(k["launches"] for k in stats) == prof.kernel_launches
    assert all(k["name"] for k in stats)
    assert np.array_equal(prof.kept_bitmap, plain.kept_bitmap)
    for key in ("n_kept", "fstar", "flow_value", "n_bundles", "n_components", "bundle_path",
                "sort_passes", "verify_violations"):
        assert prof[key] == plain[key], key
    assert plain.verify_violations == 0
    if path.startswith("direct_"):
        assert plain.bundle_path == 1
    if path.startswith("global_"):
        assert plain.bundle_path == 2
    if path == "pair_filter":
        assert np.array_equal(prof.pair_pass, plain.pair_pass)
