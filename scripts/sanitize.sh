# compute-sanitizer passes over the kernels (GPU box): racecheck / synccheck on the shared-memory kernels, memcheck on the host
# pipelines.  The summary lines of every pass are collected in gpurun_out/${TAG}_sanitizer.log (copied to profiles/ when kept).
TAG=${1:-r2}
LOG=gpurun_out/${TAG}_sanitizer.log
mkdir -p gpurun_out; : > $LOG
run() { echo "== compute-sanitizer --tool $1 :: pytest $2 -k \"$3\"" >> $LOG
  timeout 900 compute-sanitizer --tool $1 --print-limit 10 python -m pytest $2 -x -q -k "$3" 2>&1 | grep -vE "Host Frame|^\s*$" | tail -6 >> $LOG; }
run racecheck "tests/test_gpu_parity.py" "test_plan_golden and not wide and (blobs or adversarial or wall)"
run racecheck "tests/test_gpu_parity.py" "test_plan_golden_wide and (blobs or wall)"
# the bucket form of K7 (plan_grid.cuh), forced for the golden plans (n = 40 .. 1000: by-index scan and bucket scan) and at cfg3's shape
RRTK_PLAN_IMPL=grid run racecheck "tests/test_gpu_parity.py" "test_plan_golden and not wide and not informed and (blobs or adversarial or wall or cfg1)"
RRTK_PLAN_IMPL=grid run synccheck "tests/test_gpu_parity.py" "test_plan_golden and not wide and not informed and (blobs or cfg1)"
RRTK_PLAN_IMPL=grid run memcheck "tests/test_gpu_parity.py" "test_plan_golden and not wide and not informed"
run memcheck "tests/test_gpu_parity.py" "cfg3_batch_vs_oracle and star"
run memcheck "tests/test_gpu_rewire.py tests/test_gpu_clearance.py" "informed_plans_bit_exact and 96x96 or directional or pipelined_worlds"
run racecheck "tests/test_gpu_clearance.py" "fields_are_capped_cone_depths"
run racecheck "tests/test_gpu_rewire.py" "96x96_n500 or 96x96_n600 or several_plans"
run racecheck "tests/test_gpu_parity.py" "sample_stream or rejection_path"
run synccheck "tests/test_gpu_rewire.py tests/test_gpu_parity.py" "96x96_n500 or 96x96_n600 or several_plans or (test_plan_golden and blobs)"
run memcheck "tests/test_gpu_parity.py tests/test_gpu_replan.py tests/test_gpu_rewire.py tests/test_gpu_clearance.py" "pipelined or packed_grids or path_records or carry or inflate or edge_cases or 96x96 or dubins_collision or dubins_sample or clearance"
# the path shortcut (csrc/shortcut.cu): rows staged in shared memory, rewritten in place, on the host entry and in the pipeline
run memcheck "tests/test_gpu_shortcut.py" "random_polylines or host_entry or fused_flag or device_records"
run racecheck "tests/test_gpu_shortcut.py" "hand_made or random_polylines"
cat $LOG
