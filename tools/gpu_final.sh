#!/bin/bash
# Last check of a round: the suites that exercise bw_encode's graph replay (several batch sizes, seek-loop re-encodes) + smoke().
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
export PYTHONPATH=$PWD TRANSFORMERS_OFFLINE=1 HF_HUB_OFFLINE=1 TOKENIZERS_PARALLELISM=false
O=gpurun_out/${1:-final}
timeout 100 python -m pytest tests/test_pipeline_gpu.py -q -p no:cacheprovider -m gpu 2>&1 | tail -2 | tee ${O}_pipeline.log
timeout 90 python -m pytest tests/test_model_gpu.py -q -p no:cacheprovider -m gpu -x 2>&1 | tail -2 | tee ${O}_model.log
timeout 100 python -m pytest tests/test_large_gpu.py -q -p no:cacheprovider -m gpu -s -k "encoder" 2>&1 | grep -E "^\[|passed|failed" | cut -c1-200 | tee ${O}_large_encoder.log
timeout 60 python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" 2>&1 | tail -2 | tee ${O}_smoke.log
