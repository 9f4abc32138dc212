#!/bin/bash
# A short, hang-proof check (every step under its own tight timeout): default paths first, then the encoder switches.
# (r2o ran this with the 16-warp GEMM epilogue as well; that variant measured slower and is gone.)
#     gpurun --timeout 480 -- 'bash tools/gpu_quick.sh <tag>'
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
export PYTHONPATH=$PWD TRANSFORMERS_OFFLINE=1 HF_HUB_OFFLINE=1 TOKENIZERS_PARALLELISM=false
O=gpurun_out/${1:-quick}
echo "== default: pair GEMM / attention / GELU op tests"
timeout 150 python -m pytest tests/test_ops_gpu.py -q -p no:cacheprovider -m gpu -x -k "pair or attn_enc or gelu" 2>&1 | tail -2 | tee ${O}_ops.log
echo "== default: encoder parity at large-v3 dims"
timeout 200 python -m pytest tests/test_large_gpu.py -q -p no:cacheprovider -m gpu -s -k "encoder" 2>&1 | grep -E "^\[|passed|failed" | cut -c1-200 | tee ${O}_large_encoder.log
echo "== encoder switches: B = 1 and B = 64"
for spec in "graph+pdl:1:BW_ENC_PDL=1" "graph+pdl:64:BW_ENC_PDL=1" "default:1:" "default:64:" "no graph:1:BW_ENC_GRAPH=0"; do
  IFS=: read -r name a envs <<< "$spec"
  echo "-- $name A=$a" | tee -a ${O}_times.log
  env $envs BW_A=$a BW_G=1 BW_CHUNK_S=30 BW_TIME=1 BW_STEPS=2 timeout 75 python tools/profile_decode.py 2>&1 | grep -E "encode|decode step|rror" | cut -c1-120 | tee -a ${O}_times.log
done
