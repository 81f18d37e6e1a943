mkdir -p gpurun_out
timeout 900 python -m pytest tests -m gpu -x -q > gpurun_out/s2_gputests8.log 2>&1; echo "tests rc=$?"; tail -3 gpurun_out/s2_gputests8.log
B="python bench.py --steps 20 --warmup 5 --no-decode --no-cpu-baseline --no-gpu-eager"
run() { name=$1; shift; env "$@" $B > gpurun_out/s2_exp_$name.json 2> gpurun_out/s2_exp_$name.err; python - <<PY
import json
try:
    d=json.loads(open('gpurun_out/s2_exp_$name.json').read().strip().splitlines()[-1])
    print('$name', round(d['ms_per_step'],3), 'rb', d['kernels'].get('recurrent_bwd',{}).get('ms_per_step'), 'rf', d['kernels'].get('recurrent_fwd',{}).get('ms_per_step'), 'prep', d['kernels'].get('image_prep',{}).get('ms_per_step'))
except Exception as e: print('$name', 'FAILED', e)
PY
}
run k1 X=1
