#!/bin/bash
# compute-sanitizer (memcheck, initcheck, racecheck, synccheck) over the GPU parity tests that reach every kernel.
# usage: scripts/gpu_sanitize.sh <out-file>
OUT=${1:-gpurun_out/sanitizer.txt}
SEL='golden or text_batch or empty or odd or pairing or random_programs or synthetic or homopolymer or gz or bgzf or inflate or deflate'
# the aligner at its limits: reads of CSQ_MAX_READ_LEN bases first and last in their batches (the 16-byte read fetches
# and the reversed walk of RightmostFront reach into the pool padding) with adapters of CSQ_MAX_ADAPTER bases
MATRIX_SEL='m128 or packed_cell or read_length_limit'
# hand-built programs: 65 535-byte headers, UMI parts of up to 895 bases and REVCOMP - the long-header, bytewise and
# tail paths of both emitters
PROGRAMS_SEL='header_limit or umi_parts or revcomp'
echo "# compute-sanitizer, 1x B200: python -m pytest tests/test_gpu_parity.py tests/test_gpu_gz.py -m gpu -k '$SEL'" \
     "and tests/test_gpu_align_matrix.py -m gpu -k '$MATRIX_SEL'" \
     "and tests/test_gpu_programs.py -m gpu -k '$PROGRAMS_SEL' under each tool" > $OUT
for tool in memcheck initcheck racecheck synccheck; do
  echo "== $tool" >> $OUT
  timeout 420 compute-sanitizer --tool $tool --error-exitcode 99 python -m pytest tests/test_gpu_parity.py tests/test_gpu_gz.py -m gpu -q -x -k "$SEL" 2>&1 \
    | grep -E "passed|failed|error|ERROR SUMMARY|RACECHECK SUMMARY|hazard|Invalid|Uninitialized|at 0x|by thread" | head -40 >> $OUT
  echo "== $tool, tests/test_gpu_align_matrix.py" >> $OUT
  timeout 420 compute-sanitizer --tool $tool --error-exitcode 99 python -m pytest tests/test_gpu_align_matrix.py -m gpu -q -x -k "$MATRIX_SEL" 2>&1 \
    | grep -E "passed|failed|error|ERROR SUMMARY|RACECHECK SUMMARY|hazard|Invalid|Uninitialized|at 0x|by thread" | head -40 >> $OUT
  echo "== $tool, tests/test_gpu_programs.py" >> $OUT
  timeout 420 compute-sanitizer --tool $tool --error-exitcode 99 python -m pytest tests/test_gpu_programs.py -m gpu -q -x -k "$PROGRAMS_SEL" 2>&1 \
    | grep -E "passed|failed|error|ERROR SUMMARY|RACECHECK SUMMARY|hazard|Invalid|Uninitialized|at 0x|by thread" | head -40 >> $OUT
done
# the TMA engine's writes (cp.async.bulk shared -> global in k_emit_stage) are not tracked by initcheck: the same
# tests with the direct emitter (plain st.global) show what the tool says about everything else
echo "== initcheck, CSQ_PLAN_FLAGS=256 (CSQ_PLAN_EMIT_G16: output written by st.global instead of cp.async.bulk)" >> $OUT
CSQ_PLAN_FLAGS=256 timeout 420 compute-sanitizer --tool initcheck --error-exitcode 99 python -m pytest tests/test_gpu_parity.py tests/test_gpu_gz.py -m gpu -q -x -k "$SEL" 2>&1 \
  | grep -E "passed|failed|error|ERROR SUMMARY|Uninitialized|at 0x" | head -20 >> $OUT
cat $OUT
