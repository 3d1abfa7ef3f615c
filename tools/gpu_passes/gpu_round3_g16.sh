#!/bin/bash
# in_group_size 16 GEMM / transposed GEMM: the whole gpu suite (incl. tests/test_gpu_gemm_g16.py), then the probe on the Llama-3-8B shapes with the GEMV passes
# (AQLM_B200_DISABLE_TCGEN05=1) and the tensor-core path alternating per (shape, batch), both ops; the g = 8 kernel on the
# same shapes as context (each probe file starts with the device line: name, power limit, SM clocks); smoke and bench last.
# Usage: bash tools/gpu_passes/gpu_round3_g16.sh OUT_DIR   (from the repo root; every result file goes to OUT_DIR)
set -x
OUT=${1:?usage: gpu_round3_g16.sh OUT_DIR}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm --format=csv > "$OUT"/smi_g16.txt
timeout 1200 python -m pytest tests -m gpu -q > "$OUT"/pytest_gpu_g16.log 2>&1; echo "pytest rc=$?" >> "$OUT"/pytest_gpu_g16.log
tail -25 "$OUT"/pytest_gpu_g16.log
B=7,8,12,16,64,256
for op in matmat_dequant matmat_dequant_transposed; do
  timeout 600 python tools/probe_gemm.py --in-group 16 --batches $B --op $op --settings "DISABLE_TCGEN05=1;" \
    > "$OUT"/probe_gemm_g16_$op.jsonl 2>&1
  timeout 600 python tools/probe_gemm.py --in-group 8 --batches $B --op $op > "$OUT"/probe_gemm_g16_context_g8_$op.jsonl 2>&1
done
cat "$OUT"/probe_gemm_g16_*.jsonl | cut -c1-400
timeout 200 python -c "import __graft_entry__ as g; g.smoke()" > "$OUT"/smoke_g16.log 2>&1; echo "smoke rc=$?" >> "$OUT"/smoke_g16.log
tail -3 "$OUT"/smoke_g16.log
timeout 600 python bench.py --gpus 1 --skip-cpu --skip-reference-gpu > "$OUT"/bench_n1_g16.json 2> "$OUT"/bench_n1_g16.err; echo "bench rc=$?"
tail -3 "$OUT"/bench_n1_g16.err
cut -c1-600 "$OUT"/bench_n1_g16.json
