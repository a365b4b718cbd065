#!/bin/bash
# Collects the round's evidence on one B200 (run under gpurun from the repo root): tests, bench lines, ncu launch list and
# full capture of the step's kernels, the public detect_orfs() timing, sanitizer runs.  Usage: collect.sh <tag>
tag=${1:-r2v}
out=gpurun_out
python -m pytest tests -x -q -m gpu > $out/${tag}_tests.log 2>&1; tail -2 $out/${tag}_tests.log
python bench.py --steps 20 --warmup 3 > $out/${tag}_bench_n1.json 2> $out/${tag}_bench_n1.err
python bench.py --impl reference --steps 20 --warmup 3 > $out/${tag}_bench_reference_arm.json 2> $out/${tag}_bench_reference_arm.err
python bench.py --steps 10 --warmup 3 --no-cpu-baseline --reads-format columns > $out/${tag}_bench_n1_columns.json 2> $out/${tag}_bench_n1_columns.err
python bench.py --steps 10 --warmup 3 --no-cpu-baseline --k1 red > $out/${tag}_bench_n1_k1red.json 2> $out/${tag}_bench_n1_k1red.err
python bench.py --steps 10 --warmup 3 --no-cpu-baseline --min-reads-per-codon 1 > $out/${tag}_bench_n1_minreads1.json 2> $out/${tag}_bench_n1_minreads1.err
python bench.py --steps 10 --warmup 3 --no-cpu-baseline --layout dense > $out/${tag}_bench_n1_dense.json 2> $out/${tag}_bench_n1_dense.err
python bench.py --config C5 --steps 10 --warmup 3 --no-cpu-baseline > $out/${tag}_bench_C5_fullsize.json 2> $out/${tag}_bench_C5.err
python bench.py --config C4 --libraries 64 > $out/${tag}_bench_C4_n1.json 2> $out/${tag}_bench_C4_n1.err
python bench.py --config C3 --steps 10 --warmup 3 --no-cpu-baseline > $out/${tag}_bench_C3_n1.json 2> $out/${tag}_bench_C3_n1.err
ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $out/${tag}_launches.csv python bench.py --steps 8 --warmup 1 --no-cpu-baseline > $out/${tag}_b_under_ncu.log 2>&1
ncu --set full --import-source on --clock-control none -k regex:"bin_stream|atom_pass|compose_refs" -s 3 -c 3 -o $out/${tag}_step_kernels -f python bench.py --steps 2 --warmup 1 --no-cpu-baseline > $out/${tag}_ncu_full.log 2>&1
python profiles/e2e_detect_orfs.py > $out/${tag}_e2e_detect_orfs.json 2> $out/${tag}_e2e_detect_orfs.err
python profiles/e2e_probe.py > $out/${tag}_e2e_probe.txt 2>&1
python profiles/tools/k1_time.py > $out/${tag}_k1_fresh_vs_red.txt 2>&1
compute-sanitizer --tool memcheck python -m pytest tests/test_gpu_parity.py -x -q -m gpu -k "stream or edge or golden_pipeline or sparse_clear" > $out/${tag}_sanitizer_memcheck.log 2>&1; tail -3 $out/${tag}_sanitizer_memcheck.log
compute-sanitizer --tool racecheck python -m pytest tests/test_gpu_parity.py -x -q -m gpu -k "stream or edge_cases_compact" > $out/${tag}_sanitizer_racecheck.log 2>&1; tail -3 $out/${tag}_sanitizer_racecheck.log
ls $out | grep ${tag}_
