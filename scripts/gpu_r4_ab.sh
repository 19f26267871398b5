#!/bin/bash
# round 4: padded grid images.  New GPU tests; parent build (geneface_b200/variants/libgfrender_parent.so, built from the parent commit's
# sources) vs this build on the headline frame, 3 alternated pairs; May configurations once per build; output dumps of both builds;
# the whole GPU suite and smoke() on this build.  Usage: scripts/gpu_r4_ab.sh OUTDIR (logs, bench lines and output dumps go there).
O=${1:?usage: scripts/gpu_r4_ab.sh OUTDIR}
mkdir -p "$O"
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks_event_reasons.active --format=csv > $O/card.csv 2>&1; cat $O/card.csv
use() { if [ "$1" = parent ]; then export GF_LIBGFRENDER=geneface_b200/variants/libgfrender_parent.so; else unset GF_LIBGFRENDER; fi; }
echo "== new tests"; timeout 600 python -m pytest tests/test_grid_pad_gpu.py -q -s > $O/pytest_pad.log 2>&1; echo "rc=$?"
grep -E "pad |worst|tc sigma|passed|failed|Error" $O/pytest_pad.log | tail -60
for rep in 1 2 3; do
  for b in parent pr; do
    use $b
    timeout 400 python bench.py --steps 50 --no-cpu-baseline --no-ref-cuda --no-may > $O/t_${b}_$rep.json 2> $O/t_${b}_$rep.err; echo "t_${b}_$rep rc=$?"
  done
done
for b in parent pr; do
  use $b
  for C in may_head may_torso; do
    timeout 300 python bench.py --config $C --no-cpu-baseline --no-ref-cuda > $O/${C}_$b.json 2> $O/${C}_$b.err; echo "${C}_$b rc=$?"
  done
  timeout 300 python bench.py --steps 30 --no-cpu-baseline --no-ref-cuda --no-may --dump-outputs $O/dump_$b > $O/dump_$b.json 2> $O/dump_$b.err; echo "dump_$b rc=$?"
done
unset GF_LIBGFRENDER
python - "$O" <<'PY'
import json, sys, numpy as np
O = sys.argv[1]
for b in ("parent", "pr"):
    for r in (1, 2, 3):
        try:
            d = json.loads(open(f"{O}/t_{b}_{r}.json").read().strip().splitlines()[-1])
            print(b, r, d["ms_per_step"], d["roofline"]["kernel_ms_per_frame"], d["roofline"].get("frac_of_gather_ceiling"))
        except Exception as e: print(b, r, "parse failed", e)
for n in ("rgb8", "counters"):
    try: print(n, "equal:", np.array_equal(np.load(f"{O}/dump_parent/{n}.npy"), np.load(f"{O}/dump_pr/{n}.npy")))
    except Exception as e: print(n, "compare failed", e)
PY
echo "== pytest gpu"; timeout 1500 python -m pytest tests -m gpu -q > $O/pytest_gpu.log 2>&1; echo "rc=$?"; grep -E "passed|failed|FAILED|ERROR" $O/pytest_gpu.log | tail -12
echo "== smoke"; timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $O/smoke.log 2>&1; echo "rc=$?"; tail -1 $O/smoke.log
