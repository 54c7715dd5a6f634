#!/bin/bash
# N-GPU validation run (N = $1, default 2): multi-GPU pytest cases, sharded parity tools, bench at N (headline, c4, c5).
N=${1:-2}
mkdir -p gpurun_out
O=gpurun_out
TR="python -m torch.distributed.run --nnodes=1 --master-addr 127.0.0.1 --nproc-per-node $N"
echo "== multi-GPU pytest"; timeout 600 python -m pytest -q -p no:cacheprovider --timeout=500 tests/test_gpu_full_size.py -k "sharded" tests/test_gpu_search.py -k "sharded or non_current" 2>&1 | tail -6
echo "== check_sharded"
timeout 300 $TR --master-port 29511 tools/check_sharded.py 10000000 384 4096 100 2>&1 | grep -v "^W\|^\*\*\*" | tail -4 | tee $O/r02j_check_sharded_n$N.log
timeout 300 $TR --master-port 29515 tools/check_sharded.py 10000000 768 4096 100 2>&1 | grep -v "^W\|^\*\*\*" | tail -4 | tee -a $O/r02j_check_sharded_n$N.log
timeout 200 $TR --master-port 29513 tools/check_sharded.py 3000 64 50 1000 2>&1 | grep -v "^W\|^\*\*\*" | tail -3 | tee -a $O/r02j_check_sharded_n$N.log
echo "== check_sharded_retrieve"; timeout 300 $TR --master-port 29514 tools/check_sharded_retrieve.py 4000000 384 256 50 100 2>&1 | grep -v "^W\|^\*\*\*" | tail -6 | tee -a $O/r02j_check_sharded_n$N.log
echo "== bench N=$N"
for W in headline c4 c5; do
  timeout 500 $TR --master-port $((29560 + RANDOM % 300)) bench.py --gpus $N --workload $W --steps 20 --warmup 4 > $O/r02j_bench_n${N}_$W.log 2> $O/r02j_bench_n${N}_$W.err; echo "$W rc=$?"; grep -v "^W\|^\*\*\*\|^$" $O/r02j_bench_n${N}_$W.err | tail -5
  python - <<PY
import json
try:
    r=json.loads([l for l in open("gpurun_out/r02j_bench_n${N}_$W.log") if l.startswith("{")][-1])
    rf=r["roofline"] or {}
    print("$W", r["metric"], "value", round(r["value"]), "e2e", round(r["e2e"]["value"]), "ms", round(r["ms_per_step"],3), {k:(round(rf[k],4) if isinstance(rf.get(k),float) else rf.get(k)) for k in ("frac","kernel_ms","kernel_share_of_step")}, "parity", r["parity"]["ok_all_ranks"], "unc", r["uncertified_queries"], r.get("latency_batch1_ms"), r["clocks"])
except Exception as e:
    print("$W bench parse failed", e)
PY
done
timeout 200 $TR --master-port 29541 tools/phase_times.py 2>&1 | grep -v "^W\|^\*\*\*" | tail -12 | tee $O/r02j_phase_times_n$N.log
timeout 300 $TR --master-port 29551 bench.py --impl reference --gpus $N --steps 3 --warmup 1 2>/dev/null | tail -1 | cut -c1-600 | tee $O/r02j_reference_n$N.log
