"""A context owns its device buffers: destroying it gives all of them back."""
import numpy as np
import pytest

from conftest import PRM

pytestmark = pytest.mark.gpu


def test_create_solve_destroy_returns_device_memory(pkg, O):
    import torch

    # 200k reads on a 30 kb reference through the radix sort (gds_params.bundle_mode = 1): both the
    # node-array scans and the sort's histogram scans take the multi-tile path, which allocates the
    # scan's status and ticket buffers
    s, e, _, _ = O.gen_reads(2024, 100_000, 30_000, 150)
    sort_path = PRM + (0, 1)

    def cycle():
        solver = pkg.Solver(0)
        try:
            r_sort = solver.solve(s, e, 30_000, 100, params=sort_path, verify=True)
            r_default = solver.solve(s, e, 30_000, 100, params=PRM, verify=True)
        finally:
            solver.close()
        assert r_sort.sort_passes > 0 and r_sort.verify_violations == 0
        assert r_default.verify_violations == 0
        assert np.array_equal(r_sort.kept_bitmap, r_default.kept_bitmap)
        return int(r_sort.n_kept)

    n_kept = cycle()  # loads the kernels and sets up the CUDA context before the first reading
    torch.cuda.synchronize()
    free_before, _ = torch.cuda.mem_get_info()
    for _ in range(50):
        assert cycle() == n_kept
    torch.cuda.synchronize()
    free_after, _ = torch.cuda.mem_get_info()
    assert abs(free_after - free_before) <= 2 << 20, (free_before, free_after)


def test_contexts_on_one_device_leave_each_others_launches_alone(pkg, O):
    # How much shared memory a kernel may take is a property of the kernel on the device, not of a
    # context.  Context `a` solves large components first; context `b` then solves small ones, whose
    # K3 launches need less.  `b` must not lower the limit under `a`: a's next solve of the same input
    # must run and give the same answer.  Both K3 kernels: the shared-memory one (default) and
    # k_maxflow (GDS_MF=global).
    import os

    parts = [O.gen_reads(610 + k, 20_000, 30_000, 150) for k in range(3)]
    big = (np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts]), [30_000] * 3, 60)
    big_kw = dict(read_off=np.arange(4, dtype=np.uint64) * 40_000, params=PRM, verify=True)
    ex = O.SMALL_EXAMPLE
    small = [(ex["start"], ex["end"], ex["L"], ex["M"]),
             (np.full(5000, 10, np.uint32), np.full(5000, 60, np.uint32), 100, 17)]
    for env in ({}, {"GDS_MF": "global"}):
        os.environ.update(env)
        a, b = pkg.Solver(0), pkg.Solver(0)
        try:
            first = a.solve(*big, **big_kw)
            for args in small:
                assert b.solve(*args, params=PRM, verify=True).verify_violations == 0
            again = a.solve(*big, **big_kw)
        finally:
            a.close()
            b.close()
            for k in env:
                del os.environ[k]
        assert first.rounds_total > 0 and again.verify_violations == 0
        assert np.array_equal(again.kept_bitmap, first.kept_bitmap) and again.n_kept == first.n_kept
