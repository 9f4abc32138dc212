#!/bin/bash
# The gpurun calls of a round, as named sections of ONE script (round 1 left 14 one-off scripts behind):
#     gpurun --timeout 2400 -- 'bash tools/gpu_evidence.sh <tag> <section> [<section> ...]'
# Every section writes gpurun_out/<tag>_*; the summaries worth keeping are copied into profiles/ afterwards.
#   tests        GPU parity tests (-m gpu), per-test durations (PYTEST_K='expr with spaces' selects tests)
#   bench        the bench line (python bench.py), plus the --impl reference arm when REF=1
#   launches     ncu launch list (gpu__time_duration.sum) of a short bench run
#   ncu_mega     ncu --set full of the persistent decoder-step kernel
#   trace        barrier timeline of one decoder step
#   ncu_encoder  ncu --set full of log-mel / tcgen05 GEMM / tcgen05 attention / LayerNorm
#   configs      tools/bench_configs.py C3 C5 C4 (BASELINE.json configs bench.py does not time)
#   ncu_batched  launch list + ncu --set full of the batched decoder step (A = 64)
#   steptime     CUDA-event time of one decoder step at several (audios, beams, chunk length) shapes
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
export PYTHONPATH=$PWD TRANSFORMERS_OFFLINE=1 HF_HUB_OFFLINE=1 TOKENIZERS_PARALLELISM=false
TAG=${1:-r2}; shift
O=gpurun_out/${TAG}
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv > ${O}_gpu.csv
summ() {  # one line per kernel launch of an .ncu-rep: the metrics the judge asks for
  ncu -i "$1" --page raw --csv 2>/dev/null | python tools/ncu_summary.py
}
for sec in "$@"; do
  echo "=================== section $sec ($(date +%H:%M:%S))"
  case $sec in
  tests)
    # one pytest process per file: a trapped kernel poisons only its own process.  The CTA-pair GEMM goes first; if it fails the
    # rest of the call runs the encoder on the first-generation kernel (BW_GEMM2=0) so one bug does not cost the whole call
    timeout 300 python -m pytest tests/test_ops_gpu.py -q -p no:cacheprovider -m gpu -k "pair" --tb=short > ${O}_tests_pair.log 2>&1
    tail -3 ${O}_tests_pair.log
    if ! grep -q " passed" ${O}_tests_pair.log || grep -q "failed\|error" ${O}_tests_pair.log; then export BW_GEMM2=0; echo "!! gemm_tc2 failed: BW_GEMM2=0 for the rest"; fi
    : > ${O}_tests.log
    for f in tests/test_ops_gpu.py tests/test_model_gpu.py tests/test_pipeline_gpu.py tests/test_large_gpu.py; do
      n=$(basename $f .py)
      timeout ${TEST_TIMEOUT:-600} python -m pytest $f -q -p no:cacheprovider -m gpu -s --durations=8 --tb=short ${PYTEST_ARGS} ${PYTEST_K:+-k "$PYTEST_K"} > ${O}_${n}_full.log 2>&1
      grep -E "^\[|passed|failed|FAILED|ERROR|Error" ${O}_${n}_full.log | tail -40 | tee -a ${O}_tests.log
    done ;;
  bench)
    timeout 900 python bench.py --steps 10 --warmup 3 2> ${O}_bench.err | tee ${O}_bench.json | cut -c1-1500
    tail -2 ${O}_bench.err | cut -c1-300
    if [ -n "$REF" ]; then timeout 900 python bench.py --impl reference --steps 3 --warmup 1 2>/dev/null | tee ${O}_bench_ref.json | cut -c1-600; fi ;;
  launches)
    BW_NO_HF_CUDA=1 timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file ${O}_launches.csv \
      python bench.py --steps 2 --warmup 3 --no-cpu-baseline > ${O}_bench_under_ncu.log 2>&1
    python tools/ncu_summary.py --launch-list ${O}_launches.csv | tee ${O}_launches_summary.txt | head -40 ;;
  ncu_mega)
    BW_STEPS=8 timeout 600 ncu --set full --clock-control none --import-source on -k regex:decode_mega -s 20 -c 1 \
      -o ${O}_mega python tools/profile_decode.py > ${O}_ncu_mega.log 2>&1
    tail -1 ${O}_ncu_mega.log; summ ${O}_mega.ncu-rep | tee ${O}_mega_summary.txt ;;
  trace)
    timeout 300 python tools/mega_trace.py 2>&1 | tee ${O}_trace.log | tail -30 ;;
  ncu_encoder)
    for spec in "gemm_tc:40:4" "attn_enc_tc:8:2" "logmel:2:2" "layernorm_rows:8:2"; do
      IFS=: read -r pat skip cnt <<< "$spec"
      BW_STEPS=2 timeout 600 ncu --set full --clock-control none --import-source on -k regex:$pat -s $skip -c $cnt \
        -o ${O}_$pat python tools/profile_decode.py > ${O}_ncu_$pat.log 2>&1
      tail -1 ${O}_ncu_$pat.log; summ ${O}_$pat.ncu-rep | tee ${O}_${pat}_summary.txt
    done
    BW_TIME=1 BW_STEPS=2 timeout 300 python tools/profile_decode.py 2>&1 | tail -4 | tee ${O}_encoder_times.log ;;
  configs)
    for c in ${CONFIGS:-C3 C5 C4}; do
      timeout ${CONFIG_TIMEOUT:-420} python tools/bench_configs.py $c ${CONFIG_ARGS} 2> ${O}_config_$c.err | tee ${O}_config_$c.json | cut -c1-900
      tail -2 ${O}_config_$c.err | cut -c1-300
    done ;;
  ncu_batched)
    BW_A=${BW_A:-64} BW_STEPS=2 BW_NO_GRAPH=1 timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file ${O}_batched_launches.csv \
      python tools/profile_decode.py > ${O}_ncu_batched_list.log 2>&1
    tail -1 ${O}_ncu_batched_list.log; python tools/ncu_summary.py --launch-list ${O}_batched_launches.csv | tee ${O}_batched_launches_summary.txt | head -40
    for spec in ${BATCHED_KERNELS:-"cross_attn:40:2" "gemm_tc_kernel:10:8" "gemm_tc2:20:6" "resid_ln:100:2" "self_attn:40:2"}; do
      IFS=: read -r pat skip cnt <<< "$spec"
      BW_A=${BW_A:-64} BW_STEPS=2 BW_NO_GRAPH=1 timeout 600 ncu --set full --clock-control none --import-source on -k regex:$pat -s $skip -c $cnt \
        -o ${O}_b_$pat python tools/profile_decode.py > ${O}_ncu_b_$pat.log 2>&1
      tail -1 ${O}_ncu_b_$pat.log; summ ${O}_b_$pat.ncu-rep | tee ${O}_b_${pat}_summary.txt
    done ;;
  steptime)
    # CUDA-event time of one decoder step at several batch shapes (+ algorithmic GB/s), encoder and log-mel times
    for spec in ${STEP_SPECS:-"1:1:30" "64:1:30" "32:1:15" "64:5:30" "8:1:30"}; do
      IFS=: read -r a g c <<< "$spec"
      BW_A=$a BW_G=$g BW_CHUNK_S=$c BW_TIME=1 BW_STEPS=2 timeout 240 python tools/profile_decode.py 2>&1 | grep -E "decode step|encode|logmel|Error|error" | tee -a ${O}_steptime.log
    done ;;
  driver)
    # exactly what the driver runs at round end: the whole GPU suite in ONE process, then smoke()
    timeout 1800 python -m pytest tests/ -x -q -m gpu > ${O}_driver_pytest.log 2>&1; tail -4 ${O}_driver_pytest.log
    timeout 600 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2 | tee ${O}_smoke.log ;;
  pdl)
    for v in 1 0; do
      for spec in "32:1:15" "64:1:30"; do
        IFS=: read -r a g c <<< "$spec"
        echo "BW_PDL=$v A=$a" | tee -a ${O}_pdl.log
        BW_PDL=$v BW_A=$a BW_G=$g BW_CHUNK_S=$c BW_TIME=1 BW_STEPS=2 timeout 240 python tools/profile_decode.py 2>&1 | grep -E "decode step|programmatic" | tee -a ${O}_pdl.log
      done
    done ;;
  *) echo "unknown section $sec" ;;
  esac
done
ls -la gpurun_out | head -60
