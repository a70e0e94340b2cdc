#!/bin/bash
# full GPU test suite (with recorded parity numbers) + default bench line
mkdir -p gpurun_out/rec
export IAN_TEST_RECORD=$PWD/gpurun_out/rec
(timeout 2400 python -m pytest tests -x -q -m gpu 2>&1 | tail -25) > gpurun_out/pytest_gpu.log
cat gpurun_out/pytest_gpu.log | cut -c1-500
timeout 900 python bench.py --steps 30 --warmup 5 --no-cpu-baseline > gpurun_out/bench_all.json 2> gpurun_out/bench_all.err
tail -2 gpurun_out/bench_all.err
python - <<'PY'
import json
d = json.loads(open("gpurun_out/bench_all.json").read().strip().splitlines()[-1])
print(round(d["value"]), d["ms_per_step"], d["roofline"]["frac_burst"], d["roofline"]["layer_ms"], d["roofline"]["edge_kernel_ms"])
f = d["full_ian"]
print(" full bf16", f["bf16"]["value"], f["bf16"]["ms_per_step"], f["bf16"]["frac_burst"], f["bf16"]["layer_ms"]); print(" fp32", f["fp32_split"]["value"], f["fp32_split"]["layer_ms"])
print(" bf16 vs fp32", f["bf16_vs_fp32_max_abs"], f["bf16_vs_fp32_mean_abs"], f["bf16_vs_fp32_psnr_db"])
print(" edit", d["edit"]); print(" config5", d["config5"]["value"]); print(" e2e", d["e2e"]["value"], d["e2e"]["sync_value"], d["e2e"]["pageable_value"]); print(d["single_image_latency"])
PY
