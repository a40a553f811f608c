#!/bin/bash
# compute-sanitizer over the hot path (SURVEY.md section 5: race detection / sanitizers hook).
#   memcheck  : out-of-bounds / misaligned global and shared accesses, leaks of device memory
#   racecheck : shared-memory hazards (k_linear_memories_band staging, k_coarse_packed task tables + bit-planes,
#               k_refine<true> / k_refine_bits partial sums, block scans)
#   synccheck : barrier / mbarrier misuse (the TMA staging of k_coarse_packed, __syncthreads in divergent code)
# on (a) __graft_entry__.smoke() -- one full match checked against the oracle -- and (b) the fused multi-GPU exchange
# with three handles in one process (peer stores, ticket counters, frame flags, the collector's spin wait), and
# (c) memcheck on the matches that take the fallback kernels: byte-wise refinement without the filter, unsafe templates
# next to eligible ones (filter + k_refine<true>, H-planes derived by k_refine_prep), three pyramid levels, and
# (d) memcheck on template extraction (lm_extract_templates: tests/test_gpu_training.py).
# Usage (on a GPU box):  bash tools/sanitize.sh [outdir]      -> <outdir>/summary.txt, one log per tool x case
set -u
OUT=${1:-gpurun_out/sanitize}
mkdir -p "$OUT"
export LINEMOD_B200_PEER_TIMEOUT_MS=600000   # kernels run 10-100x slower under the sanitizer: no false peer timeouts
CS=${CS:-compute-sanitizer}
: > "$OUT/summary.txt"
run() {  # tool case command...
  local tool=$1 name=$2; shift 2
  local log="$OUT/${tool}_${name}.log"
  timeout 900 $CS --tool "$tool" --error-exitcode 7 --print-limit 20 --log-file "$log" "$@" > "$OUT/${tool}_${name}.out" 2>&1
  local rc=$?
  local errs
  errs=$(grep -E "ERROR SUMMARY|RACECHECK SUMMARY" "$log" | tail -1)
  echo "$tool $name rc=$rc :: ${errs:-no summary line}" | tee -a "$OUT/summary.txt"
}
for tool in memcheck racecheck synccheck; do
  run "$tool" smoke python -c "import __graft_entry__ as g; g.smoke()"
  run "$tool" exchange3 python -m pytest "tests/test_gpu_dist.py::test_fused_exchange_three_handles_one_process" -x -q -p no:cacheprovider
done
P=tests/test_gpu_match_parity.py
run memcheck fallbacks python -m pytest -x -q -p no:cacheprovider "$P::test_two_levels_without_filter_bit_exact" \
  "$P::test_unsafe_templates_take_the_byte_path_next_to_the_bit_sliced_one" "$P::test_match_bit_exact_synthetic[T6-640-512-96-35-70.0]"
run memcheck training python -m pytest -x -q -p no:cacheprovider tests/test_gpu_training.py
echo "done: $(cat "$OUT/summary.txt" | wc -l) runs" | tee -a "$OUT/summary.txt"
