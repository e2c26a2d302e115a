timeout 200 python -m pytest tests/test_gpu_chains.py -x -q -m gpu > gpurun_out/t_chains.log 2>&1; tail -5 gpurun_out/t_chains.log
run() { timeout 120 python bench.py --no-cpu-baseline --no-extra --steps 8 --warmup 3 "$@" 2>/dev/null | python -c "
import json,sys;d=json.loads(sys.stdin.read());print('  ',round(d['value']),round(d['roofline']['frac'],4),round(d['ms_per_step'],3),'e2e',round(d['e2e']['value']),'acc',round(d['acceptance_rate'],4))"; }
echo "dynamic 256 chunk1 wpc7"; run
echo "dynamic 256 chunk2"; IPMCMC_SCHED_CHUNK=2 run
echo "dynamic 256 chunk5"; IPMCMC_SCHED_CHUNK=5 run
echo "dynamic 256 wpc8"; IPMCMC_SCHED_WPC=8 run
echo "dynamic 1024"; run --workload burgers_pcn_1024 --steps 3
