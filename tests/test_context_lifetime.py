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
