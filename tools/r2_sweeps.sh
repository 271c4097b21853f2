#!/bin/bash
# round-2 sweeps at the full 8.8M-document corpus on one GPU: k=1000 warm-start variants, MRL widths
mkdir -p gpurun_out/sw
run() {  # name, env..., -- bench args
  name=$1; shift
  envs=()
  while [ "$1" != "--" ]; do envs+=("$1"); shift; done
  shift
  env "${envs[@]}" timeout 900 python bench.py "$@" --no-cpu-baseline > gpurun_out/sw/$name.json 2> gpurun_out/sw/$name.err
  echo "$name rc=$? $(python -c "
import json
d=json.load(open('gpurun_out/sw/$name.json'))
r=d['roofline']
print(round(d['ms_per_step'],2),'ms; main',round(r['kernel_ms'],2),'ms frac',round(r['frac'],3),'whole',round(r.get('whole_step',{}).get('frac',0),3),'parity',d['parity']['ok'],'passes',[(p['tiles'],p['splits']) for p in r.get('passes',[])])
" 2>&1 | tail -1) $(tail -1 gpurun_out/sw/$name.err | cut -c1-160)"
}
for w in ${SWEEPS:-k1000 mrl}; do
  if [ $w = k1000 ]; then
    run k1000_default X=1 -- --config c2k1000 --steps 4 --warmup 3
    run k1000_p128k_r LR_FLATIP_PREFIX_DOCS=131072 LR_FLATIP_REFRESH=1 -- --config c2k1000 --steps 4 --warmup 3
    run k1000_p64k_r LR_FLATIP_PREFIX_DOCS=65536 LR_FLATIP_REFRESH=1 -- --config c2k1000 --steps 4 --warmup 3
    run k1000_p32k_r LR_FLATIP_PREFIX_DOCS=32768 LR_FLATIP_REFRESH=1 -- --config c2k1000 --steps 4 --warmup 3
    run k1000_p128k LR_FLATIP_PREFIX_DOCS=131072 -- --config c2k1000 --steps 4 --warmup 3
  fi
  if [ $w = mrl ]; then
    for m in 128 256 512 1024; do run c3m$m X=1 -- --config c3m$m --steps 5 --warmup 3; done
  fi
done
