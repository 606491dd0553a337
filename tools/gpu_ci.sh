#!/bin/bash
# Runs on the GPU box under gpurun.  Each stage has its own timeout so a deadlocked kernel cannot eat the whole lease.
# usage: tools/gpu_ci.sh [stages...]   stages: gemm norm sla mb bench
mkdir -p gpurun_out
STAGES=${@:-"gemm norm sla mb"}
for s in $STAGES; do
  case $s in
    probe) timeout 120 python -m pytest tests/test_gpu_umma_probe.py -x -q -m gpu > gpurun_out/t_probe.log 2>&1 ;;
    gemm)  timeout 300 python -m pytest tests/test_gpu_quant_gemm.py -x -q -m gpu > gpurun_out/t_gemm.log 2>&1 ;;
    norm)  timeout 200 python -m pytest tests/test_gpu_norm.py -q -m gpu > gpurun_out/t_norm.log 2>&1 ;;
    slaprep) timeout 200 python -m pytest tests/test_gpu_sla.py -q -m gpu -k "quant_qk or block_map" > gpurun_out/t_slaprep.log 2>&1 ;;
    slamom) timeout 120 python -m pytest tests/test_gpu_sla.py -x -q -m gpu -k "linear_moments" > gpurun_out/t_slamom.log 2>&1 ;;
    slaattn) timeout 300 python -m pytest tests/test_gpu_sla.py -x -q -m gpu -k "forward" > gpurun_out/t_slaattn.log 2>&1 ;;
    mb)    timeout 400 python tools/microbench.py --iters 10 > gpurun_out/mb.log 2>&1 ;;
    bench) timeout 900 python bench.py > gpurun_out/bench.log 2>&1 ;;
    all)   timeout 1200 python -m pytest tests -x -q -m gpu > gpurun_out/t_all.log 2>&1 ;;
  esac
  echo "== stage $s rc=$?"
done
for f in gpurun_out/t_*.log; do echo "#### $f"; tail -n 25 $f; done
[ -f gpurun_out/mb.log ] && cat gpurun_out/mb.log
true
