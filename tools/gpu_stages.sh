# stage times of the many-chain configurations; args: extra bench flags
for cfg in "64 64 lcc" "64 1024 ssd" "128 64 lcc" "128 1 lcc"; do set -- $cfg
for mode in reference per_chain; do
python bench.py --size $1 --chains $2 --data $3 --hyper-mode $mode --steps 10 --warmup 3 --e2e-steps 3 --no-cpu-baseline --no-aten-gpu-baseline --no-configs 2>&1 | tail -1 | python -c "
import json,sys
d=json.loads(sys.stdin.read())
print('$cfg $mode', 'ms/step', round(d['ms_per_step'],3), 'G', round(d['value']/1e9,3), 'mixture', round(d['stage_ms']['mixture_step'],3), 'launches', d['gpu_launches']//10)"
done; done
