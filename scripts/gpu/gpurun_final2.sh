set -x
python -m pytest tests -m gpu -x -q 2>&1 | tail -4
python bench.py --impl reference --steps 3 --warmup 1 > gpurun_out/bench_ref_j.json 2> gpurun_out/bench_j.err
python bench.py --steps 5 --warmup 3 > gpurun_out/bench_j.json 2>> gpurun_out/bench_j.err; tail -c 400 gpurun_out/bench_j.err
ncu --metrics gpu__time_duration.sum --clock-control none -c 90 --csv --log-file gpurun_out/r01_v2h_launches.csv python bench.py --steps 2 --warmup 1 --no-cpu-baseline --no-e2e --no-per-residue --no-extras > /dev/null 2>&1
PLAAC_FUZZ_N=300 python -m pytest tests/test_gpu_fuzz.py -m gpu -q 2>&1 | tail -2
python -c "
import json; d=json.load(open('gpurun_out/bench_j.json')); print(d['value'], d['ms_per_step'], d['roofline']['frac'], d['clocks'], d['gpu_launches']); print(d['e2e']); print(d['extras']['long_sequences']); print(d['extras']['ranking']); print(d['per_residue_mode']['batch_200k'])"
