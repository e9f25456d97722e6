#!/bin/bash
# compute-sanitizer passes over the hand-synchronised kernels (mbarrier ring of the row smoother, tag-polling chain
# smoother, look-back of the Field.sum tables).  Run on the GPU box: gpurun -- tools/sanitize.sh ; logs land in gpurun_out/.
# Eager launches (RLFC_NO_GRAPH=1): the sanitizer tracks kernels launched from graphs with conditional nodes poorly.
out=gpurun_out
mkdir -p $out
CS=/usr/local/cuda/bin/compute-sanitizer
run() {  # name tool env... -- args
  name=$1; tool=$2; shift 2
  envs=(); while [ "$1" != "--" ]; do envs+=("$1"); shift; done; shift
  echo "=== $name: compute-sanitizer --tool $tool ${envs[*]} python tools/sanitize_run.py $*" > $out/san_$name.txt
  env RLFC_NO_GRAPH=1 "${envs[@]}" timeout 900 $CS --tool $tool --print-limit 20 python tools/sanitize_run.py "$@" >> $out/san_$name.txt 2>&1
  echo "exit code $?" >> $out/san_$name.txt
  grep -E "ERROR SUMMARY|RACECHECK SUMMARY|exit code|^ok" $out/san_$name.txt | tail -3
}
run memcheck_default memcheck --
run memcheck_chain memcheck RLFC_SMOOTHER=chain --
run memcheck_wave memcheck RLFC_SMOOTHER=wave -- --small
run initcheck_default initcheck --
run initcheck_chain initcheck RLFC_SMOOTHER=chain --
run racecheck_default racecheck -- --small
run racecheck_wave racecheck RLFC_SMOOTHER=wave -- --small
run racecheck_chain racecheck RLFC_SMOOTHER=chain -- --small
run synccheck_default synccheck -- --small
