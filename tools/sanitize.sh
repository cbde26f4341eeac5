#!/bin/bash
# The library's own sanitizer run.  compute-sanitizer is not available on the GPU machines (the refusal is kept in
# profiles/sanitizer/compute_sanitizer_refused.txt), so the checks are compiled in:
#   1. build/variants/checks.so = the library with -DRT_CHECKS=1: every dynamically indexed device access (BVH nodes,
#      leaf references, primitive / material / texture / texel arrays, both traversal stacks, accumulator pixels) is
#      bounds-checked on the device; a failure surfaces as RT_ERR_CUDA from the next rt_synchronize
#      (build it here first:  python tools/ab_variants.py build "checks:-DRT_CHECKS=1")
#   2. tools/sanitize_target.py drives every kernel of the library through it on small inputs — parity queries, random
#      closest hits, renders with all four render kernels + instrumented variants, push / adopt / peer paths with two
#      contexts — and asserts that the kernels still produce identical accumulators (a race would show up there)
#   3. the same target on the product build, 3 times: bit-identical accumulators across repeats = no data race visible
# usage (under gpurun):  bash tools/sanitize.sh        logs -> gpurun_out/sanitizer/
cd "$(dirname "$0")/.."
OUT=gpurun_out/sanitizer
mkdir -p $OUT
rc=0
RT_B200_LIB=build/variants/checks.so RT_B200_DEBUG=1 python tools/sanitize_target.py > $OUT/checks_build.log 2>&1 || rc=1
echo "checks build: rc=$rc, $(grep -c 'device-side checks evaluated' $OUT/checks_build.log) synchronisations reported, failures: $(grep -c 'worst failing site [1-9]' $OUT/checks_build.log)"
# the checks themselves must fire: one planted out-of-range sphere reference -> rt_synchronize reports site 5 (CHK_SPHERE)
RT_B200_LIB=build/variants/checks.so RT_B200_CHECK_SELFTEST=1 SAN_SELFTEST=1 python tools/sanitize_target.py > $OUT/checks_selftest.log 2>&1
if grep -q "device-side bounds check failed at site 5" $OUT/checks_selftest.log; then echo "checks self-test: the planted bad reference was reported (site 5 = CHK_SPHERE)"; else echo "checks self-test: NOT reported"; rc=1; fi
for i in 1 2 3; do
  SAN_HASH=1 python tools/sanitize_target.py > $OUT/product_run$i.log 2>&1 || rc=1
done
if cmp -s <(grep HASH $OUT/product_run1.log) <(grep HASH $OUT/product_run2.log) && cmp -s <(grep HASH $OUT/product_run1.log) <(grep HASH $OUT/product_run3.log); then
  echo "product build: 3 runs, $(grep -c HASH $OUT/product_run1.log) accumulator hashes identical across runs"
else
  echo "product build: accumulator hashes DIFFER between runs"; rc=1
fi
exit $rc
