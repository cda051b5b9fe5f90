#!/bin/bash
# compute-sanitizer summaries for profiles/ (run under gpurun): memcheck + racecheck of three training steps and an evaluation pass
# through (a) the default kernels, (b) the tcgen05 path of wide models, and memcheck of the catalog scorer / samplers.
out=gpurun_out/r02_sanitizer.txt
: > $out
run() { # name, tool, env..., cmd
  name=$1; tool=$2; shift; shift
  echo "== $name ($tool)" >> $out
  timeout 900 env "$@" > gpurun_out/_san_raw.txt 2>&1
  grep -aE "ERROR SUMMARY|RACECHECK SUMMARY|hazard|Invalid|========= [A-Z]" gpurun_out/_san_raw.txt | cut -c1-200 | head -20 >> $out
  grep -aqE "ERROR SUMMARY|RACECHECK SUMMARY" gpurun_out/_san_raw.txt || { echo "(no summary line; exit tail follows)" >> $out; grep -av "^{" gpurun_out/_san_raw.txt | tail -5 | cut -c1-300 >> $out; }
}
run "train steps + eval, default kernels (bf16)" memcheck ADT_SEQ_FUSED=1 compute-sanitizer --tool memcheck --print-limit 5 python tools/seq_ab.py 2 50
run "train steps + eval, default kernels (bf16)" racecheck ADT_SEQ_FUSED=1 compute-sanitizer --tool racecheck --print-limit 5 python tools/seq_ab.py 2 50
run "wide model (H 128): tcgen05 forward / backward path, MN-major + split-K GEMMs, row kernels" memcheck X=1 compute-sanitizer --tool memcheck --print-limit 5 python tools/seq_ab.py 2 40 128
run "wide model (H 128): same" racecheck X=1 compute-sanitizer --tool racecheck --print-limit 5 python tools/seq_ab.py 2 40 128
run "catalog scorer 100k x 64 (two-pass tcgen05 + re-score), samplers" memcheck X=1 compute-sanitizer --tool memcheck --print-limit 5 python tools/sanitize_misc.py
rm -f gpurun_out/_san_raw.txt
cat $out
