#!/bin/bash
# e2e of dcb_decombine_ascii at N ranks of one host with the chunk sharing off (DCB_HOST_SHARE=0: the device packs every
# chunk of bench.py's page-locked text) and on (1: two-ended).  usage (on a host with N GPUs): bash tools/e2e_scale.sh N
N=$1
for hs in 0 1; do
DCB_HOST_SHARE=$hs timeout 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 2951$hs bench.py --gpus $N --steps 20 --no-workloads --no-cpu-baseline 2>/dev/null | python -c "
import json,sys
d=json.loads(sys.stdin.read().strip().splitlines()[-1])
print('N=$N DCB_HOST_SHARE=$hs: e2e %.0f M reads/s' % (d['e2e']['value']/1e6), d['e2e'].get('chunks_packed_by'), 'ceiling GB/s per GPU %.1f' % d['e2e']['h2d_ceiling']['GBps_per_gpu'])
"
done
