cd "$(dirname "$0")/.."
for ns in 2048 4096 8192 16384 65536; do
  for k in 3 4 2; do
    out=$(timeout 300 python bench.py --streams $ns --seconds 20 --steps 3 --warmup 3 --no-cpu --no-e2e --no-config4 --kernel $k 2>&1 | grep '^{' | python -c "
import sys,json
for l in sys.stdin:
    d=json.loads(l); print(d['roofline']['kernel_ms_per_launch'], d['value'])")
    echo "streams=$ns kernel=$k => $out"
  done
done
