mkdir -p gpurun_out
for g in 1 2 4 8 16; do
  v=$(RLFC_GROUPS=$g timeout 120 python bench.py --no-cpu-baseline --steps 4 --warmup 3 --profile-steps 0 2>/dev/null | python -c "import sys,json; d=json.loads(sys.stdin.read().strip().splitlines()[-1]); print(round(d['value'],1), round(d['e2e']['value'],1))")
  echo "groups=$g -> $v"
done
