out=${1:?usage: tools/gpu_iter.sh OUT_DIR   (logs and bench JSON go to OUT_DIR)}
set -x
mkdir -p "$out"
timeout 600 python -m pytest tests/test_gpu_parity.py -x -q -m gpu > "$out/t_parity.log" 2>&1; echo "parity rc=$?"
tail -15 "$out/t_parity.log"
for cfg in ${CFGS:-c2 c3}; do
timeout 300 python bench.py --config $cfg --steps 3 --warmup 3 --no-cpu-baseline > "$out/b_$cfg.json" 2> "$out/b_$cfg.err"; echo "$cfg rc=$?"
python -c "import json; d=json.load(open('$out/b_$cfg.json')); s=d['stage_ms_per_step']; print('$cfg', 'step ms', round(d['ms_per_step'],2), 'kdecoy', round(s['kernel_decoy_attempts'],2), 'decoys', round(s['decoys'],2), 'kscore', round(d['roofline']['launch_ms'],3), 'frac', round(d['roofline']['frac'],4), 'e2e', round(d['e2e']['value']))"
done
