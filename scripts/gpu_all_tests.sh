# round-end checks: every test file that carries the `gpu` marker, one pytest process per file (a faulting kernel poisons only its
# own CUDA context), then smoke()
set +e
mkdir -p gpurun_out
rm -f gpurun_out/summary.txt
run() { name=$1; shift; timeout 1200 python -m pytest "$@" -q -m gpu --timeout 600 -p no:cacheprovider > gpurun_out/$name.log 2>&1; echo "$name exit $?" >> gpurun_out/summary.txt; tail -4 gpurun_out/$name.log; }
for f in $(grep -l "pytest.mark.gpu" tests/test_*.py); do
  run "$(basename "$f" .py)" "$f"
done
python -c "import __graft_entry__ as g; g.smoke()" > gpurun_out/smoke.log 2>&1; echo "smoke exit $?" >> gpurun_out/summary.txt; tail -2 gpurun_out/smoke.log
cat gpurun_out/summary.txt
