# usage (on the GPU box): bash tools/ab_bench.sh <workload> <flags...>   e.g.  bash tools/ab_bench.sh c2 0 2 32 128
# One compact line per cbev debug-flag value (A/B timing probes, tools/README.md): ms/step, kernel times, roofline, e2e.
wl="$1"; shift
for v in "$@"; do
  timeout 300 python bench.py --workload "$wl" --steps 300 --warmup 60 --no-cpu-baseline --no-extras --pool 512 --debug-flags "$v" 2>/dev/null | python -c "
import json,sys
d=json.loads(sys.stdin.read().strip().splitlines()[-1]); r=d['roofline']
print('$wl flags $v', 'ms %.4f'%d['ms_per_step'], 'render %.4f move %.4f judge %.4f'%(r['kernel_ms'],r['sim_kernel_ms'],r['judge_kernel_ms']), 'frac %.3f step %.3f'%(r['frac'],r['step_frac']), 'e2e %.3e venv %.3e'%(d['e2e']['value'], d['e2e_vector_env']['value']), 'blocks', ['%.2f'%b for b in d['blocks_ms']])"
done
