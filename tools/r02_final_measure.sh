#!/bin/bash
# One GPU call: tests, smoke, the bench lines of every config, the sweep, K3 probes.
# usage (through gpurun): bash tools/r02_final_measure.sh <tag>
T=${1:-r02z7}
O=gpurun_out
mkdir -p $O
nvidia-smi --query-gpu=name,memory.total --format=csv > $O/${T}_box.txt; nproc >> $O/${T}_box.txt
timeout 1500 python -m pytest tests -m gpu -x -q > $O/${T}_pytest.txt 2>&1; echo "pytest rc=$?" >> $O/${T}_pytest.txt
tail -3 $O/${T}_pytest.txt
timeout 300 python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" > $O/${T}_smoke.txt 2>&1; tail -1 $O/${T}_smoke.txt
timeout 900 python bench.py > $O/${T}_BENCH_c5.json 2> $O/${T}_BENCH_c5.err; echo "c5 rc=$?"
timeout 900 python bench.py --impl reference > $O/${T}_BENCH_reference.json 2> $O/${T}_BENCH_reference.err; echo "ref rc=$?"
for w in c4 c1 c2 ref_uniform ref_low_sides ref_hole ref_zero_sides; do
  timeout 600 python bench.py --workload $w --no-cpu-baseline > $O/${T}_bench_$w.json 2> $O/${T}_bench_$w.err; echo "$w rc=$?"
done
timeout 600 python bench.py --workload c4 --schedule 1 --no-cpu-baseline > $O/${T}_bench_c4_classic.json 2>/dev/null; echo "c4 classic rc=$?"
for w in c1 c4; do
  timeout 600 python bench.py --workload $w --algorithm mcp --no-cpu-baseline > $O/${T}_bench_mcp_$w.json 2> $O/${T}_bench_mcp_$w.err; echo "mcp $w rc=$?"
done
timeout 300 python tools/k3_probe.py c4 1 > $O/${T}_k3_probe_c4.txt 2>&1
timeout 300 ./genome-downsampler_b200/gds_host_test -b 64 > $O/${T}_host_test_batch64.txt 2>&1; tail -2 $O/${T}_host_test_batch64.txt
python - <<PY
import json,glob
for f in sorted(glob.glob("$O/${T}_*.json")):
    try:
        d=json.loads(open(f).read().strip().splitlines()[-1])
        e=d.get("e2e",{})
        print(f, "ms/step %.3f"%d["ms_per_step"], "value %.4g"%d["value"], "e2e %.4g"%e.get("value",0), "e2e ms", e.get("ms_per_step"))
    except Exception as ex:
        print(f, "ERR", ex)
PY
