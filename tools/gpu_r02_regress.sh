#!/bin/bash
# HEAD vs the final tree of round 1 (worktree _r01) at N GPUs on the same box: headline bench, 40 steps
N=${1:-4}
TR="python -m torch.distributed.run --nnodes=1 --master-addr 127.0.0.1 --nproc-per-node $N"
P='
import sys,json
for l in sys.stdin:
    if l.startswith("{"):
        r=json.loads(l); rf=r["roofline"]; print(sys.argv[1], "value", round(r["value"]), "ms", round(r["ms_per_step"],3), "scan_ms", round(rf["kernel_ms"],3), "nonscan_ms", round(r["ms_per_step"]-rf["kernel_ms"],3), "e2e", round(r["e2e"]["value"]), r["clocks"], "launches/step", r["gpu_launches"]/r["steps"])'
for rep in 1 2; do
(cd _r01 && timeout 300 $TR --master-port $((29560 + RANDOM % 300)) bench.py --gpus $N --steps 40 --warmup 5 2>/dev/null | python -c "$P" r01)
timeout 300 $TR --master-port $((29560 + RANDOM % 300)) bench.py --gpus $N --steps 40 --warmup 5 2>/dev/null | python -c "$P" HEAD
done
