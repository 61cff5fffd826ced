"""Randomised parity campaign (GPU vs oracle replay), wider than the pytest fuzz: batches, ragged and
empty samples, variable lengths (heavy nodes), short segments, read-length hints, the bundle paths
(radix sort / shared-memory or global-memory histogram) and the compact transport (16-bit starts,
implied ends).
Run from the repo root on a GPU box:  python tools/gpu_fuzz.py [N_CASES] [SEED]"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from __graft_entry__ import load_oracle, load_package  # noqa: E402


def main():
    n_cases = int(sys.argv[1]) if len(sys.argv) > 1 else 500
    rng = np.random.default_rng(int(sys.argv[2]) if len(sys.argv) > 2 else 1)
    pkg, O = load_package(), load_oracle()
    solver = pkg.Solver(0)
    bad = 0
    n_express = 0
    for it in range(n_cases):
        ns = int(rng.integers(1, 6))
        Ls = rng.integers(1, int(rng.choice([50, 400, 5000, 40000])), size=ns).astype(np.uint32)
        ss, ee, off = [], [], [0]
        for L in Ls:
            n = 2 * int(rng.integers(0, int(rng.choice([10, 300, 5000, 30000]))))
            mode = int(rng.integers(0, 4))
            if mode == 0:
                s = rng.integers(0, L, size=n); ln = rng.integers(1, max(2, L // 2 + 1), size=n)
            elif mode == 1:
                s = rng.integers(0, max(1, L // 3), size=n); ln = rng.integers(1, 6, size=n)
            elif mode == 2:
                s = rng.integers(0, L, size=n); ln = np.full(n, rng.integers(1, 200))
            else:  # clustered starts, lengths 60..160: many bundles per node
                c = rng.integers(0, L, size=max(1, n // 50 + 1))
                s = np.clip(c[rng.integers(0, len(c), size=n)] + rng.integers(-20, 20, size=n), 0, L - 1)
                ln = rng.integers(60, 160, size=n)
            e = np.minimum(s + ln - 1, L - 1)
            ss.append(s); ee.append(e); off.append(off[-1] + n)
        s = np.concatenate(ss).astype(np.uint32); e = np.concatenate(ee).astype(np.uint32)
        off = np.array(off, np.uint64)
        M = int(rng.choice([1, 3, 10, 50, 400]))
        seg = int(rng.choice([0, 0, 37, 150, 1000, 0xffffffff]))
        prm = (int(rng.integers(1, 100)), int(rng.integers(0, 300)), int(rng.integers(0, 5)), 0, seg)
        # gds_params.schedule: express where eligible / classic only / express for every component
        # that is structurally eligible (not only segments of cut references)
        sched = int(rng.choice([0, 0, 1, 2, 2]))
        hint = None
        lens = e - s + 1
        if len(s) and rng.integers(0, 2):
            hint = (int(lens.min()), int(lens.max()))
        bmode = int(rng.integers(0, 3))  # gds_params.bundle_mode: choose / sort / histogram
        s_in, e_in = s, e
        if len(s) and lens.min() == lens.max() and rng.integers(0, 2):  # compact transport
            hint = (int(lens.min()), int(lens.max()))
            e_in = None
            if Ls.max() <= 65536 and rng.integers(0, 2):
                s_in = s.astype(np.uint16)
        try:
            r = solver.solve(s_in, e_in, Ls, M, read_off=off, params=prm + (bmode, 0, sched), verify=True,
                             want_vectors=True, len_hint=hint)
            bm, st, dem, cov = O.sync_solve(s, e, Ls, off, M, params=prm + (sched,), want_vectors=True)
            n_express += st.n_express
            ok = (r.fstar == st.fstar == r.flow_value == st.flow_value and
                  np.array_equal(r.demand, dem) and np.array_equal(r.cov_capped, np.minimum(cov, M))
                  and r.n_kept == st.n_kept and np.array_equal(r.kept_bitmap, bm)
                  and r.rounds_total == st.rounds_total and r.pushes == st.pushes
                  and r.relabels == st.relabels and r.bfs_levels == st.bfs_levels
                  and r.n_bundles == st.n_bundles and r.n_components == st.n_components
                  and r.verify_violations == 0)
        except Exception as ex:  # noqa: BLE001
            ok = False
            print("case %d raised %r" % (it, ex))
        if not ok:
            bad += 1
            print("MISMATCH case %d: ns=%d n=%d Ls=%s M=%d prm=%s hint=%s bundle_mode=%d "
                  "compact=%s schedule=%d" % (it, ns, len(s), Ls.tolist(), M, prm, hint, bmode,
                                              (e_in is None, s_in.dtype.name), sched), flush=True)
            if bad > 5:
                break
    print("fuzz: %d cases, %d mismatches, %d components on the express schedule" % (it + 1, bad, n_express))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
