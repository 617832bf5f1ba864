#!/bin/bash
# Runs the GPU parity suites in separate processes (a faulting kernel poisons only its own
# process), then smoke and a short bench.  Logs land in gpurun_out/.
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,driver_version,memory.total --format=csv > gpurun_out/gpu.txt 2>&1
run() { # name, timeout, cmd...
  local name=$1; local to=$2; shift 2
  timeout $to "$@" > gpurun_out/$name.log 2>&1
  echo "$name exit=$?" | tee -a gpurun_out/summary.txt
  tail -n 15 gpurun_out/$name.log
}
: > gpurun_out/summary.txt
run attn 300 python -m pytest tests/test_gpu_ops.py -m gpu -q --tb=short -k "attention_16bit or peaked"
run ops_simt 600 python -m pytest tests/test_gpu_ops.py -m gpu -q --tb=short -k "fp32 or temporal or norm or upsample or resize or pyramid or cubic"
run ops_tc 600 python -m pytest tests/test_gpu_ops.py -m gpu -q --tb=short -k "16bit or bitwise or peaked"
run head 600 python -m pytest tests/test_gpu_head.py -m gpu -q --tb=short
run gemm_ln 600 python -m pytest tests/test_gpu_gemm_ln.py -m gpu -q --tb=short
run fwd_fp32 900 python -m pytest tests/test_gpu_forward.py -m gpu -q --tb=short -k "fp32 or video or order or preprocessing"
run fwd_16 900 python -m pytest tests/test_gpu_forward.py -m gpu -q --tb=short -k "16bit or determ or repacked or full_size or sweep"
run smoke 600 python -c "import __graft_entry__ as g; g.smoke()"
run bench 900 python bench.py --steps 5 --warmup 3 --kernels-out gpurun_out/bench_kernels.json
cat gpurun_out/summary.txt
