#!/bin/bash
# final evidence of round 2: full GPU suite, bench lines (cfg2 default, reference arm, cfg4), cfg4 / LSTM profiles, sanitizer
cd "$GRAFT_REPO_ROOT" 2>/dev/null || true
O=gpurun_out
timeout 1800 python -m pytest -q -p no:cacheprovider tests -m gpu > $O/r02fin_pytest.log 2>&1
echo "pytest rc=$?"; tail -6 $O/r02fin_pytest.log
timeout 900 python bench.py --steps 20 --warmup 5 > $O/r02fin_bench_n1.json 2> $O/r02fin_bench_n1.err
echo "bench rc=$?"; tail -2 $O/r02fin_bench_n1.err
timeout 600 python bench.py --impl reference --steps 2 --warmup 1 > $O/r02fin_bench_ref.json 2> $O/r02fin_bench_ref.err
echo "ref rc=$?"
timeout 600 python bench.py --steps 20 --warmup 5 --no-cpu-baseline --no-train-block > $O/r02fin_bench_reverse.json 2> /dev/null
timeout 600 python bench.py --config cfg4 --steps 10 --warmup 3 > $O/r02fin_cfg4.json 2> $O/r02fin_cfg4.err
python - <<'PY'
import json
for n in ('bench_n1', 'bench_ref', 'bench_reverse', 'cfg4'):
    try:
        d = json.loads(open(f'gpurun_out/r02fin_{n}.json').read().strip().splitlines()[-1])
        print(n, {k: d.get(k) for k in ('value', 'ms_per_step', 'gpu_launches')}, (d.get('e2e') or {}).get('ms_per_step'), (d.get('cpu_baseline') or {}).get('value'))
    except Exception as e:
        print(n, 'failed', e)
PY
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 1200 --csv --log-file $O/r02fin_launches_cfg4.csv \
  python bench.py --config cfg4 --steps 1 --warmup 3 --no-cpu-baseline --no-lib-ab > $O/r02fin_prof_a.log 2>&1
python tools/summarize_launches.py $O/r02fin_launches_cfg4.csv > $O/r02fin_launches_cfg4_summary.md; head -16 $O/r02fin_launches_cfg4_summary.md
timeout 900 ncu --set full --clock-control none --import-source on -k regex:k_bilstm --launch-skip 12 --launch-count 2 -o $O/r02fin_lstm \
  python bench.py --config cfg4 --steps 1 --warmup 1 --no-cpu-baseline --no-lib-ab > $O/r02fin_prof_b.log 2>&1
python tools/ncu_summary.py $O/r02fin_lstm.ncu-rep lstm > $O/r02fin_lstm.md 2>&1; cat $O/r02fin_lstm.md
python tools/ncu_roles.py $O/r02fin_lstm.ncu-rep 0 > $O/r02fin_lstm_roles.txt 2>&1
for tool in memcheck racecheck synccheck; do
  timeout 900 compute-sanitizer --tool $tool --print-limit 3 python tools/sanitize.py f16x3 > $O/r02fin_san_$tool.log 2>&1
  echo "$tool: $(grep -E 'ERROR SUMMARY|RACECHECK SUMMARY' $O/r02fin_san_$tool.log | tail -1)"
done
du -sm $O
