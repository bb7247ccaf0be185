# On a machine with N GPUs: VARIANT=trace EXTRA="" bash scripts/gpu_multi.sh N   (VARIANT: a library from scripts/build_variants.py, optional)
cd $GRAFT_REPO_ROOT
N=$1
mkdir -p gpurun_out
if [ -n "$VARIANT" ]; then cp localexpstereo_b200/liblexp_cuda.so /tmp/orig.so; cp variants/liblexp_cuda_$VARIANT.so localexpstereo_b200/liblexp_cuda.so; fi
timeout 240 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29517 bench.py --gpus $N --steps 5 --warmup 3 $EXTRA > gpurun_out/bench_n$N.json 2> gpurun_out/bench_n$N.err
if [ -n "$VARIANT" ]; then cp /tmp/orig.so localexpstereo_b200/liblexp_cuda.so; fi
tail -3 gpurun_out/bench_n$N.err | cut -c1-300
python - <<PY
import json
try:
    d=json.loads(open('gpurun_out/bench_n$N.json').read().strip().splitlines()[-1])
    print('N=$N value %.3e ms/step %.2f e2e %.3e frac %.3f'%(d['value'],d['ms_per_step'],d['e2e']['value'],d['roofline']['frac']), d['roofline']['ms_by_layer'])
except Exception as e: print('parse fail',e)
PY
