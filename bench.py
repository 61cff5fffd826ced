#!/usr/bin/env python
"""bench.py — throughput of the quasi-MCP downsampling hot path on B200 (one JSON line on stdout).

    python bench.py --gpus N --steps K --warmup W [--workload c5|c4|c2|c1] [--impl reference]
                    [--dump-outputs DIR]

A "step" is one pass of the whole hot path (validate -> bundle sort -> coverage/demand/CSR ->
component split -> push-relabel max-flow -> kept-read bitmap) over one batch of synthetic reads.

Workloads (BASELINE.json `configs`, SURVEY.md §8d):
  c5 (default)  config[4]: batch of independent 30 kb samples, 2 M reads each
                (reads-gen uniform law, mt19937 seed 12345+k, R=150), MAX_COVERAGE=100.
                512 samples per GPU; ranks own disjoint sample blocks, no data-path collective,
                per-sample bitmaps all-gathered over NCCL at the end of every step (weak scaling;
                the gather of step i overlaps the kernels of step i+1, double-buffered).
  c2            config[1]: 10 M reads over 30 kb with the device pair filter (-l 90 -q 30 + ARTIC-style
                amplicons); `value` counts PRE-filter reads.
  c4            config[3]: 50 M reads over one 5 Mb reference, MAX_COVERAGE=500 (single GPU; N>1
                runs independent replicas with different seeds).
  c1            config[0]: 1 M reads over 30 kb, MAX_COVERAGE=100.

`value`  = reads/s with the reads already resident in HBM (device-timed with CUDA events on the
           stream the kernels are launched on, max over ranks).
`e2e`    = the same metric through the C-ABI call with HOST (pinned) buffers: H2D of start/end and
           D2H of the kept bitmap inside the timed region.
`roofline` = the dominant kernel's algorithmic bytes / its CUDA-event duration, measured live in the
           timed steps (GDS_PROFILE_KERNELS), against MEASURED_PEAKS.json.
`cpu_baseline` = the oracle port of quasi-mcp-cpu (oracle/, single thread) on a bounded sample.

--impl reference times the reference's CPU algorithm (oracle port; OR-Tools is absent so the
reference solver itself cannot be built — DESIGN.md §3) on all host threads, same metric/config.
No part of the product path touches oracle/; there is no CPU fallback (Solver() raises without a GPU).
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "c5": dict(L=30_000, R=150, pairs=1_000_000, M=100, samples=512, seed=12345,
               name="config[4]: batch of independent 30 kb samples x 2M reads (reads-gen uniform, "
                    "seed 12345+k, R=150), MAX_COVERAGE=100"),
    "c4": dict(L=5_000_000, R=150, pairs=25_000_000, M=500, samples=1, seed=12345,
               name="config[3]: 50M reads over a 5 Mb reference (reads-gen uniform, seed 12345, "
                    "R=150), MAX_COVERAGE=500"),
    "c2": dict(L=30_000, R=150, pairs=5_000_000, M=100, samples=1, seed=12345,
               filter=dict(min_len=90, min_mapq=30), min_len=60, p_inside=0.9,
               name="config[1]: 10M reads over a 30 kb reference with the pair filter -l 90 -q 30 + "
                    "synthetic ARTIC-style amplicons (98 x 400 bp, 98 bp overlap; mates inside one "
                    "amplicon with p=0.9, seq_length U{60..150}, MAPQ U{0..100}), MAX_COVERAGE=100"),
    "c1": dict(L=30_000, R=150, pairs=500_000, M=100, samples=1, seed=12345,
               name="config[0]: 1M reads over a 30 kb reference (reads-gen uniform, seed 12345, "
                    "R=150), MAX_COVERAGE=100"),
}
# the reference's own random test cases (src/tests/coverage_tester.cpp:120-175): 2 M reads over 30 kb,
# M = 1000 (uniform law) or 8000 (three density shapes) — thousands of sources and sinks, F* = 12-30 k
for _name, _shape, _m in (("ref_uniform", "uniform", 1000), ("ref_low_sides", "low_sides", 8000),
                          ("ref_hole", "hole", 8000), ("ref_zero_sides", "zero_sides", 8000)):
    WORKLOADS[_name] = dict(L=30_000, R=150, pairs=1_000_000, M=_m, samples=1, seed=12345, shape=_shape,
                            name="reference test case %s (coverage_tester.cpp:120-175): 2M reads over "
                                 "30 kb, reads-gen law '%s', seed 12345, R=150, MAX_COVERAGE=%d"
                                 % (_name, _shape, _m))
METRIC = "reads/sec downsampled (device-timed)"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


ALGORITHM = "quasi-mcp"   # --algorithm: "quasi-mcp" (push-relabel max flow) or "mcp" (minimum cardinality)


SEG_LEN = 0
SCHEDULE = 0


def solver_params():
    """gds_params for the chosen algorithm and segment length (None = library defaults)."""
    if ALGORITHM != "mcp" and not SEG_LEN and not SCHEDULE:
        return None
    return (0, 0, 0, 0, SEG_LEN, 0, 1 if ALGORITHM == "mcp" else 0, SCHEDULE)


def config_for(wname, wl):
    """The workload both arms run — the SAME dict in the B200 line and in the --impl reference line
    (how many samples of it an arm takes per step is the arm's business: config['...'] never holds
    it; see 'shard' / cpu_baseline.sample)."""
    return {"workload": wname + " — " + wl["name"], "samples": wl["samples"],
            "reads_per_sample": 2 * wl["pairs"], "ref_len": wl["L"], "read_len": wl["R"],
            "max_coverage": wl["M"], "seed": wl["seed"],
            "pair_filter": wl.get("filter"), "law": wl.get("shape", "uniform"),
            "algorithm": "quasi-MCP (maximum flow)" if ALGORITHM == "quasi-mcp"
            else "MCP (minimum number of reads, mcp-cpu's objective)",
            **({"seg_len": SEG_LEN} if SEG_LEN else {}),
            **({"schedule": SCHEDULE} if SCHEDULE else {})}


def host_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def bind_to_gpu_numa(device_index):
    """Pin this rank to the CPUs NVML reports as local to its GPU, BEFORE any pinned host buffer is
    allocated, so the end-to-end leg's host->device copies do not cross the socket interconnect
    (8 ranks x 8 GB per step).  Best effort: keeps the inherited affinity otherwise (on this
    pool's single-NUMA VMs it is a no-op)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        local = {i * 64 + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1}
        use = local & os.sched_getaffinity(0)
        if use:
            os.sched_setaffinity(0, use)
            return len(use)
    except Exception:
        pass
    return 0


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def traffic_for(kernel, alg_bytes_per_launch, workload=None):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel`, from the committed
    ncu --set full capture (profiles/traffic.json holds measured DRAM bytes per sorted item; the
    scatter kernels' algorithmic bytes are 16 per item), or None when no capture covers it."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None
    t = json.load(open(p))
    per_item = t.get("per_item", {}).get(kernel)
    if per_item is not None:
        return int(per_item * alg_bytes_per_launch / 16.0)
    ratio = t.get("per_alg_byte", {}).get(kernel)  # measured DRAM bytes per algorithmic byte
    ratio = t.get("per_alg_byte_by_workload", {}).get(workload or "", {}).get(kernel, ratio)
    return None if ratio is None else int(ratio * alg_bytes_per_launch)


# ------------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clocks and throttle reasons of the GPUs in use DURING a timed region (NVML)."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown",
               0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown",
               0x2: "applications_clocks_setting", 0x10: "sync_boost"}
    BAD = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown")

    def __init__(self, devices, period=0.01):
        self.devices, self.period = list(devices), period
        self.sm, self.reasons, self.sm_max = [], set(), 0
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = [pynvml.nvmlDeviceGetHandleByIndex(i) for i in self.devices]
            self.sm_max = max(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
                              for h in self.h)
            for h in self.h:  # prime the queries: the first call of each is slow
                pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                try:
                    pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        except Exception as ex:  # no NVML: report it, do not fake numbers
            self.nv, self.h = None, []
            self.err = repr(ex)

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            for h in self.h:
                try:
                    self.sm.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                    try:
                        r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                    except Exception:
                        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for bit, name in self.REASONS.items():
                        if r & bit:
                            self.reasons.add(name)
                except Exception:
                    pass
            self._stop.wait(self.period)

    def start(self):
        if self.nv:
            self._stop.clear()
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def stop(self):
        if self._t:
            self._stop.set()
            self._t.join()
            self._t = None

    def summary(self):
        if not self.nv:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"]}
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None,
                "sm_max_mhz": int(self.sm_max), "reasons": sorted(self.reasons),
                "samples": len(self.sm)}

    def rejected(self):
        return any(r in self.BAD for r in self.reasons)


# ------------------------------------------------------------------------------- inputs
def generate(wl, sample_ids, pinned):
    """start/end of the given samples, concatenated, as int32 torch tensors on the host (the bits
    are uint32).  Uses the host mirror's reads-gen (libgds_host.so) on all host threads."""
    import torch
    from __graft_entry__ import load_package
    pkg = load_package()
    from genome_downsampler_b200 import hostlib
    n_per = 2 * wl["pairs"]
    n = n_per * len(sample_ids)
    pin = pinned
    try:
        st = torch.empty(n, dtype=torch.int32, pin_memory=pin)
        en = torch.empty(n, dtype=torch.int32, pin_memory=pin)
    except RuntimeError as ex:
        log("pinned allocation of %.1f GB failed (%s); using pageable host memory" % (8e-9 * n, ex))
        pin = False
        st = torch.empty(n, dtype=torch.int32)
        en = torch.empty(n, dtype=torch.int32)
    s_np = st.numpy().view(np.uint32)
    e_np = en.numpy().view(np.uint32)
    if "filter" in wl:  # config 2: one sample, amplicon-aware law, MAPQ and seq_length too
        mq = torch.empty(n, dtype=torch.uint8, pin_memory=pin)
        sl = torch.empty(n, dtype=torch.int32, pin_memory=pin)
        a0, a1 = hostlib.artic_amplicons(wl["L"])
        hostlib.gen_reads_amplicon_into(wl["seed"] + sample_ids[0], wl["pairs"], wl["L"], a0, a1,
                                        s_np, e_np, mq.numpy(), sl.numpy().view(np.uint32),
                                        p_inside=wl["p_inside"], min_len=wl["min_len"],
                                        max_len=wl["R"])
        return st, en, pin, dict(mapq=mq, seq_len=sl, amp_start=a0, amp_end=a1)
    if wl.get("shape", "uniform") != "uniform":
        for j, k in enumerate(sample_ids):
            hostlib.gen_reads_into(wl["seed"] + k, wl["pairs"], wl["L"], wl["R"],
                                   s_np[j * n_per:(j + 1) * n_per], e_np[j * n_per:(j + 1) * n_per],
                                   shape=wl["shape"])
        return st, en, pin, None
    hostlib.gen_batch([wl["seed"] + k for k in sample_ids], wl["pairs"], wl["L"], wl["R"], s_np,
                      e_np, threads=host_threads())
    return st, en, pin, None


# ------------------------------------------------------------------------------- reference arm
def cpu_sample_spec(wl):
    """One CPU solve of the bounded sample: (pairs, L).  c5/c1: one whole sample; c4: a 1/10 scale
    cut of the same law (same coverage depth and M), because one full 50M-read solve takes minutes."""
    if wl["pairs"] > 2_000_000 and "filter" not in wl:
        return wl["pairs"] // 10, wl["L"] // 10
    return wl["pairs"], wl["L"]


def cpu_make_input(O, wl, k, pairs, L):
    """Input k of the CPU legs (same laws and seeds as the B200 arm)."""
    if "filter" in wl:
        bed, tsv = O.artic_scheme(L)
        a0, a1 = O.parse_amplicons(bed, tsv)
        s, e, q, l = O.gen_reads_amplicon(wl["seed"] + k, pairs, L, a0, a1, wl["p_inside"],
                                          wl["min_len"], wl["R"])
        return (s, e, q, l, a0, a1)
    return O.gen_reads(wl["seed"] + k, pairs, L, wl["R"], wl.get("shape", "uniform"))[:2]


def cpu_solve_one(O, wl, inp, L):
    """The reference's CPU path on one input: (filter,) coverage, graph, max-flow, selection.
    Returns (flow value, kept count, kept flag of every (post-filter) read)."""
    if "filter" in wl:
        s, e, q, l, a0, a1 = inp
        pp, kept = O.filter_pairs(s, e, q, l, wl["filter"]["min_len"], wl["filter"]["min_mapq"],
                                  a0, a1)
        m = np.repeat(pp, 2).astype(bool)
        s, e = np.ascontiguousarray(s[m]), np.ascontiguousarray(e[m])
    else:
        s, e = inp
    if ALGORITHM == "mcp":  # mcp-cpu's objective: greedy interval multicover (== min-cost optimum)
        cov = O.coverage_fast(s, e, L)
        fstar = int(np.maximum(0, np.diff(np.minimum(np.concatenate([[0], cov]), wl["M"]).astype(np.int64))).sum())
        kept, nk = O.greedy_multicover(s, e, L, wl["M"])
        return fstar, int(nk), kept
    kept, st = O.ref_solve(s, e, L, wl["M"])
    return int(st.flow_value), int(st.n_kept), kept


def run_reference(args, wl, wname):
    """The reference's CPU algorithm (oracle port of quasi-mcp-cpu) on all host threads."""
    from concurrent.futures import ThreadPoolExecutor
    from __graft_entry__ import load_oracle
    O = load_oracle()
    O.lib()
    cores = host_threads()
    pairs, L = cpu_sample_spec(wl)
    M = wl["M"]
    inputs = [cpu_make_input(O, wl, k, pairs, L) for k in range(cores)]

    def one(k):
        return cpu_solve_one(O, wl, inputs[k], L)

    def step():
        with ThreadPoolExecutor(max_workers=cores) as ex:
            return list(ex.map(one, range(cores)))
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = step()
    dt = time.perf_counter() - t0
    if args.dump_outputs:  # solve 0: the same input whatever the number of host threads
        flow, n_kept, kept = res[0]
        idx = sample_index(len(kept))
        save_npy(args.dump_outputs, "kept_sample_index", idx)
        save_npy(args.dump_outputs, "kept_sample", kept[idx], np.float32)
        save_npy(args.dump_outputs, "flow_value", [flow])
        save_npy(args.dump_outputs, "n_kept", [n_kept])
    reads = 2 * pairs * cores * args.steps
    value = reads / dt
    sample = "%d independent solves per step (one per host thread), each %d reads over %d bp, M=%d" \
             % (cores, 2 * pairs, L, M)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "reads/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": config_for(wname, wl),
        "cpu_baseline": {"value": value, "unit": "reads/s", "cores": cores, "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": "reads/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "flow_value": res[0][0], "n_kept": res[0][1],
    }
    emit(line)


def cpu_baseline(wl, budget_s=12.0, max_solves=32):
    """Single-thread oracle port on a bounded sample (rank 0, N=1 only)."""
    from __graft_entry__ import load_oracle
    O = load_oracle()
    O.lib()
    pairs, L = cpu_sample_spec(wl)
    done, t_solve = 0, 0.0
    while done < max_solves and t_solve < budget_s:
        inp = cpu_make_input(O, wl, done, pairs, L)
        t0 = time.perf_counter()
        cpu_solve_one(O, wl, inp, L)
        t_solve += time.perf_counter() - t0
        done += 1
    return {"value": done * 2 * pairs / t_solve, "unit": "reads/s", "cores": 1, "kind": "port",
            "sample": "%d sequential solves of %d reads over %d bp, M=%d (%.1f s)"
                      % (done, 2 * pairs, L, wl["M"], t_solve)}


def reference_cuda_baseline(wl, timeout_s=180):
    """The reference's OWN GPU backend (quasi-mcp-cuda, compiled unmodified for sm_100a into
    oracle/_ref/libgds_refcuda.so) on one sample of the workload, on this box's GPU, in its own
    process under a timeout (it has no iteration bound and terminates on CUDA errors).  A reported
    baseline — "the thing to beat" of SURVEY §2.2 — never part of the product path."""
    import subprocess
    runner = os.path.join(ROOT, "oracle", "run_refcuda.py")
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libgds_refcuda.so")):
        return {"unavailable": "oracle/_ref/libgds_refcuda.so not built"}
    if "filter" in wl:
        return {"unavailable": "the runner has no pair-filter stage (config 2)"}
    pairs, L = cpu_sample_spec(wl)
    try:
        out = subprocess.run([sys.executable, runner, "gen", str(wl["seed"]), str(pairs), str(L),
                              str(wl["R"]), str(wl["M"]), "2"], capture_output=True, text=True,
                             timeout=timeout_s)
        if out.returncode != 0:
            return {"unavailable": "quasi-mcp-cuda exited %d" % out.returncode}
        d = json.loads(out.stdout.strip().splitlines()[-1])
    except subprocess.TimeoutExpired:
        return {"unavailable": "quasi-mcp-cuda did not finish in %d s" % timeout_s}
    except Exception as ex:
        return {"unavailable": repr(ex)}
    return {"value": d["reads"] / d["best_s"], "unit": "reads/s", "kind": "reference",
            "what": "reference's quasi-mcp-cuda (unmodified .cu, sm_100a) on this GPU, whole solve() "
                    "incl. its host graph build and copies, best of 2 calls",
            "sample": "1 solve of %d reads over %d bp, M=%d" % (d["reads"], d["L"], d["M"]),
            "seconds": d["best_s"], "n_kept": d["n_kept"], "coverage_invariant_ok": d["invariant_ok"]}


# ------------------------------------------------------------------------------- B200 arm
def run_b200(args, wl, wname):
    import torch
    import torch.distributed as dist
    from __graft_entry__ import load_package
    pkg = load_package()
    from genome_downsampler_b200 import sharding

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node %d" % args.gpus)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 path has no CPU fallback")
    if world > 1:
        bind_to_gpu_numa(local_rank)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    # Default = the stated batch (BASELINE config[4]: ONE batch of 512 samples) sharded over the
    # ranks with sharding.shard_samples — strong scaling.  --weak: every rank gets the whole
    # workload's sample count (different seeds).  Single-sample workloads cannot be sharded
    # (DESIGN.md §7): N > 1 runs independent replicas with different seeds ("weak").
    S_total = args.samples if args.samples else wl["samples"]
    shardable = S_total >= world and S_total % world == 0 and S_total > 1
    strong = shardable and not args.weak
    if strong:
        sample_ids = sharding.shard_samples(S_total, world, rank)
    else:
        sample_ids = list(range(rank * S_total, (rank + 1) * S_total))
    S = len(sample_ids)
    n_per = 2 * wl["pairs"]
    n = n_per * S
    t0 = time.time()
    h_st, h_en, pinned, fx = generate(wl, sample_ids, pinned=True)
    log("[rank %d] generated %d reads (%d samples) in %.1f s, pinned=%s" %
        (rank, n, S, time.time() - t0, pinned))
    ref_len = np.full(S, wl["L"], np.uint32)
    read_off = (np.arange(S + 1, dtype=np.uint64) * np.uint64(n_per))
    words = (n + 31) // 32

    stream = torch.cuda.Stream(device=dev)
    solver = pkg.Solver(local_rank)   # raises without a usable GPU
    with torch.cuda.stream(stream):
        solver.set_stream(stream.cuda_stream)
        d_st = h_st.to(dev, non_blocking=True)
        d_en = h_en.to(dev, non_blocking=True)
        # config 2: MAPQ / seq_length columns, the amplicon table and the per-pair verdicts
        filt = d_mq = d_sl = pair_pass = h_pair_pass = None
        if fx is not None:
            d_mq = fx["mapq"].to(dev, non_blocking=True)
            d_sl = fx["seq_len"].to(dev, non_blocking=True)
            pair_pass = torch.zeros(n // 2, dtype=torch.uint8, device=dev)
            h_pair_pass = torch.empty(n // 2, dtype=torch.uint8, pin_memory=True)
            filt = dict(wl["filter"], amp_start=fx["amp_start"], amp_end=fx["amp_end"])

        def fkw(on_device):
            if fx is None:
                return {}
            return dict(mapq_ptr=(d_mq if on_device else fx["mapq"]).data_ptr(),
                        seq_len_ptr=(d_sl if on_device else fx["seq_len"]).data_ptr(), filt=filt,
                        pair_pass_ptr=pair_pass.data_ptr())
        bitmap = torch.zeros(words + 4, dtype=torch.int32, device=dev)
        h_bitmap = torch.empty(words, dtype=torch.int32, pin_memory=True)
        h_gathered = torch.empty((world, words), dtype=torch.int32, pin_memory=True) \
            if world > 1 and rank == 0 else None
        # N > 1: every step ends with an NCCL gather of the ranks' kept bitmaps ON RANK 0 (grouped
        # send/recv: the other ranks receive nothing — sharding.gather_bitmaps_to_root).  Two bitmap
        # / gather buffers alternate so that the gather of step i (NCCL's own stream) runs under the
        # kernels of step i+1; the timed region ends only when the last gather has landed.
        gathered = bitmaps2 = None
        pending = [None, None]
        step_no = [0]
        if world > 1:
            gathered = [torch.empty((world, words), dtype=torch.int32, device=dev) if rank == 0
                        else None for _ in range(2)]
            bitmaps2 = [bitmap, torch.zeros(words + 4, dtype=torch.int32, device=dev)]
            gathered_all = [torch.empty(world * words, dtype=torch.int32, device=dev)
                            for _ in range(2)] if args.gather == "all" else None

        gl = [list(g.unbind(0)) if g is not None else None for g in gathered] if world > 1 else None

        def gather_async(buf_idx):
            if args.gather == "none":      # measurement only: what the collective costs
                return
            if args.gather == "all":       # round 1: every rank receives every bitmap
                pending[buf_idx] = dist.all_gather_into_tensor(
                    gathered_all[buf_idx], bitmaps2[buf_idx][:words], async_op=True)
                return
            pending[buf_idx] = dist.gather(bitmaps2[buf_idx][:words], gl[buf_idx], dst=0, async_op=True)

        def gather_wait(buf_idx=None):
            for i in ([buf_idx] if buf_idx is not None else [0, 1]):
                if pending[i] is not None:
                    pending[i].wait()   # stream-level wait, the host does not block
                    pending[i] = None
        stream.synchronize()

        # exact read-length bounds, as the C++ adapter passes them (it gets them for free while
        # narrowing the reference's size_t arrays): reads-gen emits fixed-length reads
        hint = (wl["R"], wl["R"]) if fx is None else None  # config 2 has variable lengths

        def step_device(profile):
            b = step_no[0] % 2 if world > 1 else 0
            step_no[0] += 1
            if world > 1:
                gather_wait(b)  # the gather that read this buffer two steps ago
            out_bm = bitmaps2[b] if world > 1 else bitmap
            r = solver.solve_device(d_st.data_ptr(), d_en.data_ptr(), n, ref_len, wl["M"],
                                    out_bm.data_ptr(), read_off=read_off, profile=profile,
                                    len_hint=hint, params=solver_params(), **fkw(True))
            if world > 1:
                gather_async(b)
            return r

        # e2e: HOST buffers in (the 32-bit SoA columns the C ABI defines, pinned), kept bitmap back on
        # the host, everything inside the timed region — including, for the headline figure, the
        # narrowing to the compact transport (include/gds.h gds_reads.start16 / end == NULL: 16-bit
        # starts, ends implied by the one read length; 2 bytes per read cross PCIe instead of 8).
        # Round 1 prepared that column outside the timed region; now it happens inside, chunk by
        # chunk ahead of the transfers (hostlib.encode_compact, what the C++ adapter's narrowing loop
        # does; pipeline.py).  "e2e_u32" is the same call with the 32-bit columns sent as they are, and
        # "e2e_preencoded" the round-1 figure (a producer that writes 16-bit starts itself).
        # A batch of many samples goes through the package's chunked host API (two contexts: H2D of
        # chunk c+1 overlaps kernels of chunk c).
        chunked = pkg.ChunkedSolver(local_rank) if S >= 2 * args.chunk_samples else None
        compact_ok = hint is not None and hint[0] == hint[1] and wl["L"] <= 65536
        h_st16 = torch.empty(n, dtype=torch.int16, pin_memory=True) if compact_ok else None
        n_extra = (5 if fx is not None else 0) * n
        # the narrowing runs ahead of the device on its own host threads (pipeline.py); four threads
        # stay free for the two chunk workers, the driver and this interpreter
        enc_threads = args.encode_threads or max(2, (host_threads() - 4) // max(1, min(world, 8)))

        def make_e2e(mode):
            """mode: 'encode' (u32 columns in, narrowed inside the step), 'u32', 'preencoded'."""
            def step():
                if mode == "preencoded":
                    kw = dict(start_ptr=None, end_ptr=None, start16_ptr=h_st16.data_ptr(), len_hint=hint)
                else:
                    # the read length is the generator's parameter (reads_gen's read_length), i.e.
                    # known to the caller like a sequencing run's cycle count: passed as the hint
                    kw = dict(start_ptr=h_st.data_ptr(), end_ptr=h_en.data_ptr(), start16_ptr=None,
                              len_hint=hint)
                if chunked is not None:
                    rs = chunked.solve_host_batch(kw["start_ptr"], kw["end_ptr"], read_off, ref_len,
                                                  wl["M"], bitmap.data_ptr(),
                                                  chunk_samples=args.chunk_samples, params=solver_params(),
                                                  len_hint=kw["len_hint"], start16_ptr=kw["start16_ptr"],
                                                  encode16_ptr=h_st16.data_ptr() if mode == "encode" else None,
                                                  encode_threads=enc_threads)
                    r = rs[-1]
                    r["kernel_launches"] = sum(int(x.kernel_launches) for x in rs)
                else:
                    if mode == "encode":
                        from genome_downsampler_b200 import hostlib
                        fits, lo_, hi_ = hostlib.encode_compact(h_st.data_ptr(), None, n,
                                                                h_st16.data_ptr(), threads=enc_threads)
                        if fits:
                            kw = dict(start_ptr=None, end_ptr=None, start16_ptr=h_st16.data_ptr(),
                                      len_hint=hint)
                    r = solver.solve_device(kw["start_ptr"], kw["end_ptr"], n, ref_len, wl["M"],
                                            bitmap.data_ptr(), read_off=read_off,
                                            input_on_device=False, len_hint=kw["len_hint"],
                                            params=solver_params(),
                                            start16_ptr=kw["start16_ptr"], **fkw(False))
                    if fx is not None:
                        h_pair_pass.copy_(pair_pass, non_blocking=True)
                if world > 1:
                    gather_wait()
                    sharding.gather_bitmaps_to_root(bitmap[:words].view(1, words), out=gathered[0], dst=0)
                    if rank == 0:  # the root hands the whole batch's bitmaps to the host
                        h_gathered.copy_(gathered[0], non_blocking=True)
                else:
                    h_bitmap.copy_(bitmap[:words], non_blocking=True)
                stream.synchronize()
                torch.cuda.current_stream(dev).synchronize()
                return r
            return step

        def barrier():
            stream.synchronize()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        def max_over_ranks(x):
            if world == 1:
                return x
            t = torch.tensor([x], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())

        # correctness gate (untimed): the device re-derives coverage from the kept bitmap
        rv = solver.solve_device(d_st.data_ptr(), d_en.data_ptr(), n, ref_len, wl["M"],
                                 bitmap.data_ptr(), read_off=read_off, verify=True, len_hint=hint,
                                 params=solver_params(), **fkw(True))
        assert rv.verify_violations == 0 and rv.flow_value == rv.fstar, \
            "device verification failed: %r" % dict(rv)

        def timed(step_fn):
            for _ in range(args.warmup):
                step_fn()
            sampler = ClockSampler(range(world) if rank == 0 else [])
            barrier()
            solver.kernel_profile_reset()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            sampler.start()
            e0.record(stream)
            launches, last = 0, None
            for _ in range(args.steps):
                last = step_fn()
                launches += int(last.kernel_launches)
            gather_wait()  # N > 1: the stream waits for the gathers still in flight
            e1.record(stream)
            barrier()
            sampler.stop()
            ms = max_over_ranks(e0.elapsed_time(e1))
            return ms, launches, last, sampler

        for attempt in range(2):
            ms_dev, launches, r_last, clk = timed(lambda: step_device(True))
            if not clk.rejected():
                break
            log("clock record shows %s — measuring once more" % sorted(clk.reasons))
        if args.dump_outputs and rank == 0:  # before the e2e legs reuse the bitmap
            dump_outputs(args.dump_outputs, bitmaps2[(step_no[0] - 1) % 2] if world > 1 else bitmap,
                         r_last["filt_off"] if fx is not None else read_off, r_last, pair_pass)
        prof = solver.kernel_profile()
        e2e_runs = {}
        if compact_ok:
            h_st16.zero_()
            e2e_runs["encode"] = timed(make_e2e("encode"))
            enc_check = h_st16.numpy().view(np.uint16)[:min(n, 1 << 20)].astype(np.uint32)
            assert np.array_equal(enc_check, h_st.numpy().view(np.uint32)[:len(enc_check)])
        e2e_runs["u32"] = timed(make_e2e("u32"))
        if compact_ok:
            e2e_runs["preencoded"] = timed(make_e2e("preencoded"))
        head = "encode" if compact_ok and e2e_runs["encode"][0] <= e2e_runs["u32"][0] else "u32"
        ms_e2e, _, _, clk2 = e2e_runs[head]
        # correctness of the e2e path's own output: the bitmap the host received equals the device one
        if world == 1:
            assert torch.equal(h_bitmap, bitmap[:words].cpu()), "e2e bitmap differs"

    # quality of the answer (SURVEY §8c P4), outside every timed region: kept reads of sample 0 against
    # a lower bound on ANY valid answer — every kept read covers at most R positions, so at least
    # ceil(sum_i min(cov_i, M) / R) reads are needed (for the uniform law the bound is the optimum
    # up to a few reads).  Segmented references (config 4) pay at most M reads per cut on top.
    quality = None
    if fx is None:
        with torch.cuda.stream(stream):
            s0 = d_st[:n_per].long()
            e0_ = d_en[:n_per].long()
            dcov = torch.zeros(wl["L"] + 2, dtype=torch.int64, device=dev)
            dcov.scatter_add_(0, s0, torch.ones_like(s0))
            dcov.scatter_add_(0, e0_ + 1, -torch.ones_like(e0_))
            need = int(torch.clamp(torch.cumsum(dcov[:wl["L"]], 0), max=wl["M"]).sum().item())
            bits0 = bitmap[:n_per // 32].view(torch.uint8)
            kept0 = int(torch.tensor([bin(i).count("1") for i in range(256)], device=dev)[bits0.long()]
                        .sum().item())
        lb = -(-need // wl["R"])
        quality = {"sample": 0, "n_kept": kept0, "lower_bound": lb,
                   "kept_over_lower_bound": round(kept0 / max(lb, 1), 5)}
    total_reads = n * world
    value = total_reads * args.steps / (ms_dev * 1e-3)
    e2e_value = total_reads * args.steps / (ms_e2e * 1e-3)

    def e2e_entry(mode):
        ms = e2e_runs[mode][0]
        compact = mode in ("encode", "preencoded")
        return {"value": total_reads * args.steps / (ms * 1e-3), "unit": "reads/s",
                "ms_per_step": ms / args.steps,
                "h2d_bytes_per_step": (2 * n if compact else 8 * n) + n_extra,
                "d2h_bytes_per_step": 4 * words + (n // 2 if fx is not None else 0),
                "host_input": "pinned uint32 start/end columns (the C ABI's gds_reads), read length known "
                              "to the caller (reads_gen's parameter)" + (
                    " + mapq u8, seq_len u32" if fx is not None else "") if mode != "preencoded"
                else "pinned uint16 start column written by the producer, ends implied",
                "transport": "start u16, end implied by the one read length" if compact
                else "start u32, end u32",
                "encode_in_timed_region": mode != "preencoded",
                "pinned": bool(pinned),
                "api": ("ChunkedSolver.solve_host_batch, %d samples per chunk, 2 contexts"
                        % args.chunk_samples) if chunked is not None else "Solver.solve_device(host)"}
    peak, peak_src = peaks()
    kernels = []
    for k in sorted(prof, key=lambda k: -k["ms"]):
        if k["launches"] == 0 or k["ms"] <= 0:
            continue
        gbs = k["bytes"] / (k["ms"] * 1e-3) / 1e9
        kernels.append({"name": k["name"], "ms_per_step": k["ms"] / args.steps,
                        "launches_per_step": k["launches"] / args.steps,
                        "alg_bytes_per_step": k["bytes"] // args.steps,
                        "gbs": round(gbs, 1), "frac": round(gbs / peak, 4)})
    roofline = None
    if kernels:
        top = kernels[0]
        per_launch = int(top["alg_bytes_per_step"] / max(top["launches_per_step"], 1))
        roofline = {"bound": "hbm", "kernel": top["name"], "achieved": top["gbs"], "peak": peak,
                    "unit": "GB/s", "frac": top["frac"],
                    "traffic": traffic_for(top["name"], per_launch, args.workload),
                    "peak_source": peak_src, "alg_bytes_per_launch": per_launch,
                    "note": ("K3 is bound by the latency of its dependent rounds (rounds x us, see "
                             "result.k3), not by HBM; the streaming kernels are listed in kernels[]")
                    if top["name"] == "maxflow" else None,
                    "ms_per_launch": top["ms_per_step"] / max(top["launches_per_step"], 1)}
        stream_k = [k for k in kernels if k["name"] != "maxflow"]
        if stream_k:
            b = sum(k["alg_bytes_per_step"] for k in stream_k)
            t = sum(k["ms_per_step"] for k in stream_k)
            roofline["streaming_kernels"] = {"gbs": round(b / (t * 1e-3) / 1e9, 1),
                                             "frac": round(b / (t * 1e-3) / 1e9 / peak, 4),
                                             "ms_per_step": t}
        # whole-step figure from SURVEY §8d: B_alg = 8.125*P + 4*(L+1) per sample
        b_alg = (13.125 if fx is not None else 8.125) * n + 4.0 * (wl["L"] + 1) * S
        roofline["step_alg_gbs"] = round(b_alg / (ms_dev / args.steps * 1e-3) / 1e9, 1)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    line = {
        "metric": METRIC, "value": value, "unit": "reads/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev / args.steps,
        "higher_is_better": True, "scaling": "strong" if strong and world > 1 else "weak",
        "vs_baseline": None, "dtype": "u32",
        "data": "synthetic (reads-gen uniform law, mt19937 seed %d+k, generated on the host)"
                % wl["seed"],
        "config": config_for(wname, wl),
        "shard": {"samples_total": S * world if not strong else S_total, "samples_per_gpu": S,
                  "reads_per_gpu": n,
                  "l2": "inputs (%.0f MB per GPU) larger than the 126 MB L2; no flush needed"
                        % (8e-6 * n) if 8 * n > 252e6 else
                        "inputs fit L2: every step re-reads them after >126 MB of other traffic",
                  "parallelism": ("the batch of %d samples block-partitioned over %d ranks "
                                  "(sharding.shard_samples), no data-path collective, kept bitmaps "
                                  "gathered on rank 0 over NCCL (grouped send/recv)" % (S_total, world)
                                  if strong else "%d samples per rank (independent replicas), kept "
                                  "bitmaps gathered on rank 0 over NCCL" % S)
                  if world > 1 else "single GPU"},
        "e2e": e2e_entry(head),
        "gpu_launches": launches,
        "clocks": clk.summary(), "clocks_e2e": clk2.summary(),
        "roofline": roofline, "kernels": kernels[:12],
        "result": {"fstar": int(r_last.fstar), "flow_value": int(r_last.flow_value),
                   "n_filtered": int(r_last.n_filtered),
                   "n_kept": int(r_last.n_kept), "quality": quality, "n_bundles": int(r_last.n_bundles),
                   "n_components": int(r_last.n_components), "rounds_total": int(r_last.rounds_total),
                   "rounds_max": int(r_last.rounds_max), "bfs_levels": int(r_last.bfs_levels),
                   "sort_passes": int(r_last.sort_passes),
                   "bundle_path": ["radix sort", "histogram in shared memory",
                                   "histogram in global memory"][int(r_last.bundle_path)],
                   "partial_bundles": int(r_last.partial_bundles),
                   "partial_candidates": int(r_last.partial_candidates),
                   # K3 is latency-bound, not HBM-bound: its own figures (SURVEY §8d iii)
                   "k3": {"pushes": int(r_last.pushes), "relabels": int(r_last.relabels),
                          "global_relabels": int(r_last.global_relabels),
                          "max_frontier": int(r_last.max_frontier),
                          "steps_per_component": (int(r_last.rounds_total) + int(r_last.bfs_levels))
                          / max(int(r_last.n_components), 1),
                          "us_per_step": 1e3 * r_last.ms_maxflow * max(int(r_last.n_components), 1)
                          / max(int(r_last.rounds_total) + int(r_last.bfs_levels), 1),
                          "pushes_relabels_per_s": (int(r_last.pushes) + int(r_last.relabels))
                          / max(r_last.ms_maxflow * 1e-3, 1e-9)},
                   "phase_ms": {"graph": r_last.ms_graph, "maxflow": r_last.ms_maxflow,
                                "select": r_last.ms_select, "total": r_last.ms_total}},
    }
    for mode in e2e_runs:
        if mode != head:
            line["e2e_" + mode] = e2e_entry(mode)
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(wl)
        line["reference_cuda_baseline"] = reference_cuda_baseline(wl)
    if world > 1:
        dist.destroy_process_group()
    emit(line)


DUMP_READS = 1 << 21   # --dump-outputs: flags of at most this many reads (and pairs), < 64 MB in all


def save_npy(out_dir, name, values, dtype=np.float64):
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), np.asarray(values, dtype=dtype))


def sample_index(n):
    """Every index below n when n <= DUMP_READS, else an ascending fixed seeded sample of them."""
    if n <= DUMP_READS:
        return np.arange(n, dtype=np.int64)
    return np.unique(np.random.default_rng(0).integers(0, n, size=DUMP_READS, dtype=np.int64))


def dump_outputs(out_dir, bitmap, off, r, pair_pass=None):
    """What a caller of the timed path receives from its last step, as .npy files: the kept-read
    count of every sample, the kept flags of a sample of reads (sample_index), with the pair filter
    the verdicts of a sample of pairs, and the result's counters.  off holds the offsets of the
    samples' reads in the bitmap (post-filter offsets with the pair filter: the bitmap indexes the
    reads that passed).  Comparable between builds: the inputs depend only on the workload's seeds."""
    import torch
    off = [int(x) for x in off]
    words = bitmap[:(off[-1] + 31) // 32]
    shifts = torch.arange(32, dtype=torch.int32, device=words.device)
    per_sample = []
    for lo, hi in zip(off[:-1], off[1:]):
        w0 = lo // 32
        flags = ((words[w0:(hi + 31) // 32].unsqueeze(1) >> shifts) & 1).flatten()[lo - 32 * w0:hi - 32 * w0]
        per_sample.append(int(flags.sum().item()))
    save_npy(out_dir, "kept_per_sample", per_sample)
    idx = sample_index(off[-1])
    d_idx = torch.from_numpy(idx).to(words.device)
    save_npy(out_dir, "kept_sample_index", idx)
    save_npy(out_dir, "kept_sample", ((words[d_idx >> 5] >> (d_idx & 31).int()) & 1).cpu().numpy(),
             np.float32)
    if pair_pass is not None:
        idx = sample_index(len(pair_pass))
        save_npy(out_dir, "pair_pass_sample_index", idx)
        save_npy(out_dir, "pair_pass_sample",
                 pair_pass[torch.from_numpy(idx).to(pair_pass.device)].cpu().numpy(), np.float32)
    for k in ("fstar", "flow_value", "n_filtered", "n_kept"):
        save_npy(out_dir, k, [int(getattr(r, k))])


def emit(line):
    """The ONE JSON line goes to the real stdout; everything else (NCCL's version banner, library
    chatter) was redirected to stderr by main()."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)  # C-level writes to stdout (e.g. "NCCL version ...") must not pollute the JSON
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c5", choices=sorted(WORKLOADS))
    ap.add_argument("--samples", type=int, default=0, help="samples per GPU (default: workload's)")
    ap.add_argument("--chunk-samples", type=int, default=64,
                    help="samples per chunk of the end-to-end (host buffer) leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--encode-threads", type=int, default=0,
                    help="host threads of the e2e leg's narrowing (default: host threads - 4, per rank)")
    ap.add_argument("--gather", default="root", choices=["root", "all", "none"],
                    help="N > 1: kept bitmaps gathered on rank 0 (default), all-gathered (round 1), or "
                         "not at all (measures what the collective costs)")
    ap.add_argument("--weak", action="store_true",
                    help="N > 1: every rank takes the workload's full sample count (weak scaling) "
                         "instead of a share of the one batch (default, strong scaling)")
    ap.add_argument("--seg-len", type=int, default=0,
                    help="gds_params.seg_len (0 = the library's default rule); an experiment knob: the "
                         "config line then says so")
    ap.add_argument("--schedule", type=int, default=0, choices=[0, 1, 2, 3],
                    help="gds_params.schedule (include/gds.h); an experiment knob like --seg-len")
    ap.add_argument("--algorithm", default="quasi-mcp", choices=["quasi-mcp", "mcp"],
                    help="quasi-mcp: maximum flow by push-relabel (the north-star path, default); mcp: the "
                         "minimum-cardinality solve (gds_params.algorithm = 1, plugin mcp-b200)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy "
                         "(rank 0's samples when N > 1)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    global ALGORITHM, SEG_LEN, SCHEDULE
    ALGORITHM = args.algorithm
    SEG_LEN = args.seg_len
    SCHEDULE = args.schedule
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) != 0:
            return 0
        run_reference(args, wl, args.workload)
        return 0
    args.warmup = max(args.warmup, 3)  # timing hygiene: never fewer than 3 warm-up steps
    run_b200(args, wl, args.workload)
    return 0


if __name__ == "__main__":
    sys.exit(main())
