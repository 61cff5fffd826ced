import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

PRM = (64, 150, 1, 0)  # default deterministic-schedule knobs (include/gds.h gds_params)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def O():
    import pyoracle
    pyoracle.lib()
    return pyoracle


@pytest.fixture(scope="session")
def R():
    import pyref
    if not pyref.available():
        pytest.skip("oracle/_ref not built (needs /root/reference at build time)")
    pyref.lib()
    return pyref


@pytest.fixture(scope="session")
def pkg():
    from __graft_entry__ import load_package
    return load_package()


@pytest.fixture(scope="session")
def solver(pkg):
    s = pkg.Solver(0)  # raises without a GPU: no CPU fallback
    yield s
    s.close()


@pytest.fixture(scope="session")
def golden():
    import json
    return json.load(open(os.path.join(ROOT, "tests", "golden", "golden.json")))


@pytest.fixture(scope="session")
def coverage_tester(O, golden):
    """The reference's CoverageTester::test (src/tests/coverage_tester.cpp:28-43) restated: its five
    cases in its order, on inputs that must hash to the reference's own streams in golden.json, and
    its one assertion, is_out_cover_valid (:101-107): min(cov_in, M) <= cov_out everywhere.
    run(solve_fn), solve_fn(M, L, start, end) -> kept indices, returns the number of solve calls."""
    import hashlib

    import numpy as np

    def sha(a):
        return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()

    def cases():
        ex = O.SMALL_EXAMPLE
        assert O.coverage(ex["start"], ex["end"], ex["L"]).tolist() == golden["small16"]["cover"]
        yield ex["M"], ex["L"], ex["start"], ex["end"]
        shape_names = {v: k for k, v in O.SHAPES.items()}
        for name, M in (("test_uniform", 1000), ("test_low_sides", 8000), ("test_hole", 8000),
                        ("test_zero_sides", 8000)):
            g = golden["generators"][name]
            s, e, _, _ = O.gen_reads(g["seed"], g["pairs"], g["L"], g["R"], shape_names[g["shape"]])
            assert sha(s) == g["start"] and sha(e) == g["end"]
            yield M, g["L"], s, e

    def run(solve_fn):
        calls = 0
        for M, L, s, e in cases():
            mask = np.zeros(len(s), np.uint8)
            mask[np.asarray(solve_fn(M, L, s, e), np.int64)] = 1
            cin = O.coverage_fast(s, e, L)
            assert np.all(np.minimum(cin, M) <= O.coverage_fast(s, e, L, mask))
            calls += 1
        return calls
    return run
