timeout 100 python -m pytest tests/test_gemm_gpu.py -k "segments" -x -q 2>&1 | tail -2
timeout 200 python -m pytest tests/test_block_gpu.py -x -q 2>&1 | tail -2
run() { n=$1; shift; env "$@" timeout 200 python bench.py --steps 8 --warmup 3 --workload text --no-cpu-baseline --no-int8-peak > gpurun_out/r2_ab_$n.json 2> gpurun_out/r2_ab_$n.err; python - <<PY
import json
d=json.loads(open("gpurun_out/r2_ab_$n.json").read().strip().splitlines()[-1])
k=d["kernels"]
print("$n", d["value"], d["ms_per_step"], d["clocks"]["sm_mhz"], "int8", k["int8_gemm"], "attn_fwd", k["attn_fwd"]["ms_per_step"])
PY
}
run qkv1 A=1
run qkv3 LLAMAX_QKV_ONE_LAUNCH=0
run qkv1b A=1
