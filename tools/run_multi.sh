#!/bin/bash
# multi-GPU legs of BASELINE.json (one box, N GPUs): usage  bash tools/run_multi.sh N TAG [ab]
# humanoid-9 update + rollout sweep, cwhh set sharded over the ranks (packed); "ab": also the flat all-reduce for comparison
N=$1; TAG=$2; AB=$3
RUN="python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29511"
mkdir -p gpurun_out
timeout 600 $RUN bench.py --gpus $N --steps 60 --warmup 6 --no-cpu-baseline --no-bf16 --check-replicas --rollout-sweep 1024,4096,16384,65536 \
  > gpurun_out/${TAG}_n${N}.json 2> gpurun_out/${TAG}_n${N}.err; tail -c 300 gpurun_out/${TAG}_n${N}.json; echo
if [ "$AB" = "ab" ]; then
  timeout 600 $RUN bench.py --gpus $N --steps 60 --warmup 6 --no-cpu-baseline --no-bf16 --no-rollout \
    > gpurun_out/${TAG}_n${N}_flat.json 2> gpurun_out/${TAG}_n${N}_flat.err; tail -c 200 gpurun_out/${TAG}_n${N}_flat.json; echo
fi
timeout 600 $RUN bench.py --gpus $N --set 3d_cwhh --packed --batch 100 --steps 30 --warmup 4 \
  > gpurun_out/${TAG}_cwhh_n${N}.json 2> gpurun_out/${TAG}_cwhh_n${N}.err; tail -c 400 gpurun_out/${TAG}_cwhh_n${N}.json; echo
python - <<PY
import json
for f in ["${TAG}_n${N}", "${TAG}_n${N}_flat", "${TAG}_cwhh_n${N}"]:
    try:
        d = json.loads(open("gpurun_out/%s.json" % f).read().strip().splitlines()[-1])
        print(f, d.get("ms_per_step"), d.get("value"), d.get("e2e", {}).get("value"), d.get("replicas"), [round(x["value"] / 1e6, 2) for x in d.get("rollout_sweep", [])])
    except Exception as e:
        print(f, "ERR", e)
PY
