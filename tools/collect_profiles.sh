#!/bin/bash
# Collect the evidence bench.py's numbers are explained by (run under gpurun, 1 GPU):
#   1. bench.py line (value / e2e / roofline / cpu_baseline / extra) and the reference arm
#   2. ncu launch list of one mid-sequence decode step (per-launch device time, cold-cache, serialised)
#   3. ncu --set full of the dominant kernels (decode attention, decode contractions)
#   4. prefill + VQ launch list, ncu --set full of the prefill contractions (tensor-pipe utilisation)
#   5. mmu front-end: launch list of the SigLIP tower, ncu --set full of its attention and contractions
set -x
R=${1:-r02}
mkdir -p gpurun_out
timeout 900 python bench.py --steps 5 --warmup 3 > gpurun_out/${R}_bench.json 2> gpurun_out/${R}_bench.err
tail -c 400 gpurun_out/${R}_bench.err
KREG='^(gemm_tc|gemm_swiglu_sk|gemm_simt|attn_|resid_rmsnorm|swiglu|bias_act|cfg_sample|qkv_rope|embed_gather|prefill_|gather_last|kv_broadcast)'
PG_STEPS=300 PG_GRAPH=0 timeout 400 ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum --clock-control none \
  -k regex:"$KREG" -s 43300 -c 180 --csv --log-file gpurun_out/${R}_launches_decode_step.csv python tools/profile_step.py > gpurun_out/p_a.log 2>&1
PG_STEPS=300 PG_GRAPH=0 timeout 400 ncu --set full --clock-control none --import-source on -k regex:"attn_decode_v5" -s 7000 -c 1 \
  -o gpurun_out/${R}_attn_decode python tools/profile_step.py > gpurun_out/p_b.log 2>&1
PG_STEPS=300 PG_GRAPH=0 timeout 400 ncu --set full --clock-control none --import-source on -k regex:"gemm_tc_kernel" -s 28900 -c 4 \
  -o gpurun_out/${R}_gemm_tc python tools/profile_step.py > gpurun_out/p_c.log 2>&1
PG_STEPS=2 PG_GRAPH=0 PG_VQ=1 timeout 400 ncu --metrics gpu__time_duration.sum --clock-control none \
  -k regex:"^(gemm_tc|gemm_simt|im2col|gn_|conv_epilogue|softmax_rows|vq_codebook|attn_prefill|qkv_rope|resid_rmsnorm|swiglu|prefill_|gather_last|kv_broadcast)" -c 2000 \
  --csv --log-file gpurun_out/${R}_launches_prefill_vq.csv python tools/profile_step.py > gpurun_out/p_d.log 2>&1
PG_STEPS=2 PG_GRAPH=0 timeout 400 ncu --set full --clock-control none --import-source on -k regex:"gemm_tc2_kernel" -s 1 -c 4 \
  -o gpurun_out/${R}_gemm_prefill python tools/profile_step.py > gpurun_out/p_e.log 2>&1
PG_B=32 PG_ITERS=1 timeout 400 ncu --metrics gpu__time_duration.sum --clock-control none -k regex:"^(gemm_tc|vit_|bias_act|to_f32)" -c 900 \
  --csv --log-file gpurun_out/${R}_launches_siglip.csv python tools/siglip_time.py > gpurun_out/p_f.log 2>&1
PG_B=32 PG_ITERS=1 timeout 400 ncu --set full --clock-control none --import-source on -k regex:"vit_attn_tc|gemm_tc_kernel" -s 40 -c 6 \
  -o gpurun_out/${R}_siglip python tools/siglip_time.py > gpurun_out/p_g.log 2>&1
timeout 300 python tools/siglip_time.py > gpurun_out/${R}_siglip_time.json 2>/dev/null
# post-process on the box (gpurun copies back at most 64 MiB: the .ncu-rep files stay behind)
for k in decode_step prefill_vq siglip; do python tools/summarize_launches.py gpurun_out/${R}_launches_$k.csv > gpurun_out/${R}_launches_$k.txt; done
for k in attn_decode gemm_tc gemm_prefill siglip; do python tools/extract_ncu.py gpurun_out/${R}_$k.ncu-rep > gpurun_out/${R}_$k.full.txt; done
rm -f gpurun_out/*.ncu-rep
ls -la gpurun_out | tail -24
# afterwards, where ncu is installed:
#   python tools/summarize_launches.py gpurun_out/${R}_launches_decode_step.csv > profiles/${R}_launches_decode_step.txt   (same for prefill_vq, siglip)
#   python tools/extract_ncu.py gpurun_out/${R}_attn_decode.ncu-rep > profiles/${R}_attn_decode.full.txt   (same for gemm_tc, gemm_prefill, siglip)
#   python tools/sass_summary.py > profiles/${R}_sass_opcodes.txt
# scaling: gpurun --gpus N -- tools/scale_sweep.sh N [--model janus-pro-7b --batch 32]
