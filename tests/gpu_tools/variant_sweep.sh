#!/bin/bash
# forward / backward variant A/B per workload (MLSTM_FORCE_VARIANT = <fwd><bwd>: forward 1 = single pass, 2 = two-phase;
# backward 2 = chunk parallel, 3 = fused walk)
for w in ${@:-cfg2_B32_NH4_S400_DH64 cfg2alt_B32_NH4_S400_DH128 cfg3_B32_NH4_S1600_DH128 ddp_B8_NH4_S1600_DH128}; do
  for v in 12 22 13 23; do
    MLSTM_FORCE_VARIANT=$v timeout 200 python bench.py --workload $w --steps 30 --warmup 5 --no-cpu-baseline | python -c "import json,sys; d=json.load(sys.stdin); r=d['roofline']; print('$w'[:8], '$v', round(d['value']/1e6,1), round(d['ms_per_step'],4), {k:round(v,4) for k,v in r['per_kernel_ms'].items()})"
  done
done
