#!/bin/bash
# Round-2 evaluation on one B200 (run under gpurun): tests, bench lines, ncu launch list + full captures.
# Everything lands in gpurun_out/r02_eval/.
O=gpurun_out/r02_eval; mkdir -p $O
python -m pytest tests -m gpu -x -q > $O/pytest.log 2>&1; tail -3 $O/pytest.log
python bench.py > $O/bench_default.jsonl 2> $O/bench_default.err || tail -5 $O/bench_default.err
python bench.py --impl reference --steps 2 --warmup 1 > $O/bench_reference.jsonl 2> $O/bench_reference.err
for wl in ml1m_item_pearson_k40 ml20m_user_msd_k100 ml20m_item_cosine_k40 ml20m_item_msd_k40 ml20m_item_pearson_baseline_k40 netflix_item_cosine_k50; do
  python bench.py --workload $wl --steps 3 --warmup 3 --no-cpu-baseline >> $O/bench_other.jsonl 2>> $O/bench_other.err
done
python tools/i8_peak.py --out $O/int8_peak.json > $O/i8.log 2>&1
python bench.py --steps 2 --warmup 3 --no-cpu-baseline > $O/pre.log 2>&1 && \
ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $O/launches_default.csv \
    python bench.py --steps 2 --warmup 3 --no-cpu-baseline > $O/ncu_list.log 2>&1
ncu --set full --clock-control none --import-source on -k regex:'sim_stream_kernel|predict_select_kernel' -s 6 -c 3 \
    -o $O/r02_default_full -f python bench.py --steps 2 --warmup 3 --no-cpu-baseline > $O/ncu_full.log 2>&1
ls -la $O
