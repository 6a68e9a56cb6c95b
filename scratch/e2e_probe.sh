for g in 16 37 148 592; do echo "egress grid $g"; GOFR_EGRESS_GRID=$g python bench.py --steps 8 --warmup 3 2>&1 | python -c "
import json,sys;d=json.loads(sys.stdin.read().strip().splitlines()[-1]);print(d['e2e']['ms_per_step'])"; done
for c in 16384 32768 131072 262144; do echo "chunk $c"; python bench.py --steps 8 --warmup 3 --chunk $c 2>&1 | python -c "
import json,sys;d=json.loads(sys.stdin.read().strip().splitlines()[-1]);print(d['e2e']['ms_per_step'])"; done
