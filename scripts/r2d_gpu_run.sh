#!/bin/bash
# Evidence call with the final defaults: whole GPU suite, VQ / LBS stand-alone timings,
# the bench line (1 stream vs 4 streams), smoke(), ncu --set full of the SMPL blend GEMM and the skinning kernel.
cd "${GRAFT_REPO_ROOT:-/root/repo}"
export PYTHONPATH=.
export THMR_BENCH_WATCHDOG=300
O=gpurun_out; mkdir -p $O
T0=$(date +%s)
el() { echo "[t+$(( $(date +%s) - T0 ))s] $*"; }
timeout 400 python -m pytest tests -m gpu -q > $O/r2d_pytest_gpu.log 2>&1
el "full pytest rc=$?"; tail -4 $O/r2d_pytest_gpu.log
timeout 120 python scripts/dev_vq_lbs.py > $O/r2d_vq_lbs.log 2>&1; el "vq/lbs rc=$?"; cat $O/r2d_vq_lbs.log
timeout 420 python bench.py --steps 20 --warmup 5 > $O/r2d_bench_b200_n1.json 2> $O/r2d_bench_b200_n1.err
el "bench rc=$?"; grep early $O/r2d_bench_b200_n1.err | head -3
timeout 120 python -c "import __graft_entry__ as g; g.smoke()" > $O/r2d_smoke.log 2>&1
el "smoke rc=$?"; tail -2 $O/r2d_smoke.log
timeout 150 ncu --set full --clock-control none --import-source on -k "regex:gemm_f16_tn_kernel|smpl_skin_kernel" -s 16 -c 2 -f -o $O/r2d_prof_lbs \
    python scripts/dev_vq_lbs.py lbs > $O/r2d_ncu_lbs.log 2>&1
el "ncu lbs full rc=$?"
