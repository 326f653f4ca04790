# A/B of kernel variants on the GPU box: build variants/libdtr_<name>.so (from edited sources), then
# `gpurun -- bash tools/ab_variants.sh <name>...`; the library under test is selected with DTR_B200_LIB.
# Every line is parity checked by bench.py itself (a wrong frame exits non-zero and prints PARITY FAILURE).
cd /root/repo
WL=${WL:-"views1080_tex mesh1080 fill4k"}
run() { # name lib
  for w in $WL; do
  DTR_B200_LIB=$2 python bench.py --workload $w --views 64 --steps 50 --warmup 5 --e2e-steps 2 --no-cpu-baseline --no-others 2>gpurun_out/ab_$1_$w.err | python -c "
import sys,json
t=sys.stdin.read().strip()
try:
    d=json.loads(t.splitlines()[-1]); r=d['roofline']
    print('$1 $w', 'value',round(d['value'],2),'ms/step',round(d['ms_per_step'],4),'raster',round(r['stage_ms_per_step']['raster'],4), 'iso', round(r.get('stage_ms_isolated',{}).get('raster',0),4), 'frac', round(r['frac'],4), 'parity', d.get('parity_checked'))
except Exception as e:
    print('$1 $w FAILED', e, open('gpurun_out/ab_$1_$w.err').read()[-400:])
"
  done
}
run base /root/repo/dtrenderer_b200/libdtr_b200.so
for v in "$@"; do run $v /root/repo/variants/libdtr_$v.so; done
