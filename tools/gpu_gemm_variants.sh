#!/bin/bash
# GEMM variant matrix (round 2): TMA ring depth x cross-K-block TMEM prefetch mode.  Rebuilds gemm_w8a8.cu per variant on the
# GPU machine, runs the bit-exactness tests and the GEMM microbench lines.  Output: OUT_DIR/gemmvar_<name>.jsonl
OUT=${1:?usage: tools/gpu_gemm_variants.sh OUT_DIR}
mkdir -p "$OUT"
variant() {
  local name=$1 defs=$2
  touch turbodiffusion_b200/csrc/gemm_w8a8.cu
  TDB200_NVCC_DEFINES="$defs" python -m turbodiffusion_b200._build > "$OUT"/gemmvar_${name}_build.log 2>&1 || { echo "$name: build failed"; tail -5 "$OUT"/gemmvar_${name}_build.log; return; }
  timeout 200 python -m pytest tests/test_gpu_quant_gemm.py -x -q -m gpu > "$OUT"/gemmvar_${name}_tests.log 2>&1
  echo "== $name tests rc=$? $(tail -n 1 "$OUT"/gemmvar_${name}_tests.log)"
  timeout 300 python tools/microbench.py --filter "gemm_w8a8" --iters 10 --out "$OUT"/gemmvar_${name}.jsonl 2>/dev/null | grep '^{' | grep -v rowwise | python -c "
import sys,json
print('   ', ' | '.join(f\"{json.loads(l)['name'].split('/')[0][9:]}{json.loads(l)['name'].split('/')[1]}:{json.loads(l)['name'].split('/')[2][:6]} {json.loads(l)['tflops']:.0f}\" for l in sys.stdin))
"
}
variant s3_xpf2 "-DTDB_GEMM_STAGES=3 -DTDB_GEMM_XPF=2"
variant s3_xpf0 "-DTDB_GEMM_STAGES=3 -DTDB_GEMM_XPF=0"
variant s3_xpf1 "-DTDB_GEMM_STAGES=3 -DTDB_GEMM_XPF=1"
variant s4_xpf0 "-DTDB_GEMM_STAGES=4 -DTDB_GEMM_XPF=0"
variant s4_xpf2 "-DTDB_GEMM_STAGES=4 -DTDB_GEMM_XPF=2"
touch turbodiffusion_b200/csrc/gemm_w8a8.cu
python -m turbodiffusion_b200._build > "$OUT"/gemmvar_restore.log 2>&1 && echo "default build restored"
