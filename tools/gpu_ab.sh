q() { timeout 600 python bench.py --steps 5 --warmup 3 --no-cpu --no-sharded --no-e2e --no-latency > gpurun_out/ab.json 2> gpurun_out/ab.err; python -c "
import json; d=json.load(open('gpurun_out/ab.json')); k=d['kernel_ms']; print('$1', round(d['value']), round(d['ms_per_step'],1), d['clocks']['sm_mhz'], 'resid', k['gemm_resid'], 'swiglu', k['gemm_swiglu'], 'ratio', round(k['gemm_resid']/k['gemm_swiglu'],4), 'attn_full', k['attn_full'], 'k1', k['k1_hpass'], k['k1_vpass'])"; }
mkdir -p gpurun_out
q shipped
ZV_NVCC_EXTRA="-DZV_ATTN_POLY_EVERY=3" python -m zoomearth_b200.build --force > /dev/null 2>&1; q poly3
ZV_NVCC_EXTRA="-DZV_ATTN_POLY_EVERY=0" python -m zoomearth_b200.build --force > /dev/null 2>&1; q poly0
python -m zoomearth_b200.build --force > /dev/null 2>&1; q shipped_again
