#!/bin/bash
# compute-sanitizer over the round-2 kernels (BPTT tcgen05 / TMA tensor-map kernels, SIMT policy variants, halting
# rollout tail, stat reduction).  bash profiles/run_sanitizer_r2.sh  (under gpurun, one GPU)
OUT=gpurun_out/r2_compute_sanitizer.txt
T1="tests/test_gpu_grad.py::test_run_batch_boundary_and_gradient_match_the_reference tests/test_gpu_variants.py::test_variant_forward_matches_reference"
T2="tests/test_gpu_grad.py::test_run_batch_boundary_and_gradient_match_the_reference[grad_pp_easy_ic3net-auto] tests/test_gpu_grad.py::test_run_batch_boundary_and_gradient_match_the_reference[grad_tj_medium_ic3net-auto]"
echo "# compute-sanitizer, round 2: $T1" > $OUT
echo "## memcheck" >> $OUT
timeout 900 compute-sanitizer --tool memcheck python -m pytest $T1 -q --timeout 800 -p no:cacheprovider 2>&1 | grep -v "^$" | tail -6 >> $OUT
echo "## racecheck ($T2)" >> $OUT
timeout 900 compute-sanitizer --tool racecheck python -m pytest $T2 -q --timeout 800 -p no:cacheprovider 2>&1 | grep -v "^$" | tail -6 >> $OUT
cat $OUT
