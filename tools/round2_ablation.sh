#!/bin/bash
# First GPU call of round 2: validate and measure every opt-in path that was written without a GPU, one JSON line each,
# plus the per-layer cuDNN table the convolution kernels have to beat.
#   gpurun --timeout 1200 -- bash tools/round2_ablation.sh
# Output: gpurun_out/ablation_*.json (+ .err), gpurun_out/conv_layers.{log,json}, gpurun_out/test_optin.log
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
O=gpurun_out
B="python bench.py --gpus 1 --steps 40 --warmup 8 --skip_e2e"
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv > $O/ablation_smi.txt 2>&1
echo "== GEMM rasterisation tests"; timeout 420 python -m pytest tests/test_gpu_gemm_raster.py -m gpu -q --timeout 120 > $O/test_optin.log 2>&1; echo "rc=$?"; tail -n 15 $O/test_optin.log
echo "== per-layer conv table (cuDNN bar + our GEMM route for 1x1 / the 3x3 draft)"; timeout 420 python bench/conv_layers.py --out $O/conv_layers.json > $O/conv_layers.log 2>&1; echo "rc=$?"; cat $O/conv_layers.log
run() {  # name, env...
  local name=$1; shift
  echo "== $name"
  env "$@" timeout 150 $B > $O/ablation_$name.json 2> $O/ablation_$name.err; echo "rc=$?"
  python - "$O/ablation_$name.json" <<'PY'
import json, sys
try:
    d = json.loads(open(sys.argv[1]).read().strip().splitlines()[-1])
    print(f"   {d['value']:.0f} {d['unit']}  {d['ms_per_step']:.3f} ms/step  opt_in={d['config'].get('opt_in')}")
except Exception as e:
    print("   no result:", e)
PY
}
run base A=0
run stem_pad8 B200DDP_STEM_PAD=8
run conv1x1_tc B200DDP_CONV1X1_TC=1
run conv1x1_tc_tmastore B200DDP_CONV1X1_TC=1 B200DDP_GEMM_TMA_STORE=1
run conv1x1_tc_tmastore_bnfuse B200DDP_CONV1X1_TC=1 B200DDP_GEMM_TMA_STORE=1 B200DDP_CONV_BN_FUSE=1
run conv3x3_tc B200DDP_CONV3X3_TC=1
run all_conv_tc B200DDP_STEM_PAD=8 B200DDP_CONV1X1_TC=1 B200DDP_GEMM_TMA_STORE=1 B200DDP_CONV_BN_FUSE=1 B200DDP_CONV3X3_TC=1
echo "== GEMM sweep (raster / TMA store variants)"; timeout 300 python bench/kernel_bench.py --only gemm --out $O/kernels_groupm.json > $O/kernels_groupm.log 2>&1; echo "rc=$?"; grep -i "gemm" $O/kernels_groupm.log | tail -n 60
