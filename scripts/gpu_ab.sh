# A/B timing on the C2 bench of library builds (BMO_LIB=path) and of the wave path (BMO_PERSIST=0).  Usage: bash scripts/gpu_ab.sh TAG "ENV1=.. ENV2=..;ENV..."
TAG=${1:-ab}; SPECS=$2
mkdir -p gpurun_out
IFS=';' read -ra ARR <<< "$SPECS"
for rep in 1 2; do
for spec in "${ARR[@]}"; do
  name=$(echo "$spec" | tr ' /=' '___')
  env $spec python bench.py --steps 10 --warmup 3 --no-cpu-baseline --no-detector --no-extras 2> gpurun_out/${TAG}_${name}.err > gpurun_out/${TAG}_${name}.json
  echo "== [$spec] rc=$?"
  python -c "import json,sys; d=json.loads(open(sys.argv[1]).read()); c=d.get('roofline_compaction') or {}; print('value %.4g e2e %.4g ms/step %.4f  k1 ms/launch %.4f sdf/step %.4g launches %d  compaction %.0f GB/s (%.3f)' % (d['value'], d['e2e']['value'], d['ms_per_step'], d['roofline']['ms_per_launch'], d['roofline']['counted']['sdf_evals_per_step'], d['gpu_launches'], c.get('achieved') or 0, c.get('frac') or 0))" gpurun_out/${TAG}_${name}.json
done
done
