#!/bin/bash
# round 2 re-entry: parity tests, default bench, single-image sizes, launch lists (image + batch pass)
mkdir -p gpurun_out
nproc > gpurun_out/r2a_nproc.txt
timeout 1500 python -m pytest tests -m gpu -x -q > gpurun_out/r2a_pytest.log 2>&1; echo "pytest rc=$?" >> gpurun_out/r2a_pytest.log
tail -5 gpurun_out/r2a_pytest.log
timeout 900 python bench.py --steps 50 --warmup 5 > gpurun_out/r2a_bench.json 2> gpurun_out/r2a_bench.err; echo "bench rc=$?"
tail -c 600 gpurun_out/r2a_bench.err
python - <<'PY'
import json
d=json.load(open('gpurun_out/r2a_bench.json'))
print({k:d[k] for k in ('value','ms_per_step','stage_ms','gpu_launches')})
print(d['e2e'])
b=d['extra']['batch1080p']
print(d['roofline']['frac'], b.get('resident'), b.get('files_returned'), b.get('e2e'), b.get('error'))
print(d['extra'].get('frame4k'), d['extra'].get('dct_microbench'))
print(d.get('cpu_baseline'))
PY
python tools/one_image.py 16384 16384 50
python tools/one_image.py 3840 2160 200
python tools/one_image.py 1920 1080 200
python tools/one_image.py 512 512 200
python tools/one_image.py 16384 16384 2 > /dev/null 2>&1 &&
ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file gpurun_out/r2a_launches16k.csv python tools/one_image.py 16384 16384 1 > gpurun_out/r2a_ncu16k.log 2>&1
python tools/one_batch.py 128 2 &&
ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file gpurun_out/r2a_launches_batch.csv python tools/one_batch.py 128 1 > gpurun_out/r2a_ncubatch.log 2>&1
tail -30 gpurun_out/r2a_launches16k.csv | cut -c1-200
