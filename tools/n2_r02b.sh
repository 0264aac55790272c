#!/bin/bash
# 2 GPUs: default bench line (strong + weak + train sub-records) on the final tree, and the training step alone (bucketed all-reduce
# hooks join the weight-gradient side stream per bucket)
cd $GRAFT_REPO_ROOT
O=gpurun_out
R="python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1"
timeout -k 5 600 $R --master-port 29517 bench.py --gpus 2 --steps 20 --warmup 3 > $O/r02z_bench_2gpu.json 2> $O/r02z_bench_2gpu.err
tail -c 1200 $O/r02z_bench_2gpu.json; tail -3 $O/r02z_bench_2gpu.err
timeout -k 5 300 $R --master-port 29521 bench.py --gpus 2 --workload train --steps 20 --warmup 5 > $O/r02z_train_2gpu_w1.json 2> $O/r02z_train_2gpu_w1.err
python - <<'PY'
import json
for f in ("r02z_train_2gpu_w1",):
    try:
        d=json.load(open("gpurun_out/%s.json"%f)); print(f, round(d["ms_per_step"],3), d["value"], d.get("loss"), {k:d[k] for k in d if "allreduce" in k or "noar" in k})
    except Exception as e: print(f, "no result", e)
PY
