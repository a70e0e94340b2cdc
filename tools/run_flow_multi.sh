#!/bin/bash
# Weak scaling of the IAN.py graph in bf16 at 512 images per GPU, every gather form, at 1 GPU and then at N GPUs in the
# same run, so the scaling ratio comes from one box.
# Usage: [OUT=dir] bash tools/run_flow_multi.sh N [extra bench_flow_multi args]   (JSON lines + logs go to $OUT,
# default flow_multi_out/)
N=${1:-2}
shift
OUT=${OUT:-flow_multi_out}
mkdir -p "$OUT"
for n in $(echo 1 $N | tr ' ' '\n' | sort -nu); do
  for g in p2p_async p2p nccl; do
    python -m torch.distributed.run --standalone --nproc-per-node $n tools/bench_flow_multi.py --graph IAN.py --precision bf16 \
      --per-gpu 512 --gather $g --steps 20 --warmup 5 "$@" > "$OUT/flow_multi_n${n}_${g}.json" 2> "$OUT/flow_multi_n${n}_${g}.err"
    echo "n=$n $g rc=$? $(tail -n 1 "$OUT/flow_multi_n${n}_${g}.json")"
  done
done
