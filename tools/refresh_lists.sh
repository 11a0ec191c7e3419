#!/bin/bash
# Launch lists of the prefill + VQ decode and of the SigLIP tower, and the ncu --set full extract of the tower kernels, post-processed
# on the box (run under gpurun; results land in gpurun_out/).
R=r02
PG_STEPS=2 PG_GRAPH=0 PG_VQ=1 timeout 400 ncu --metrics gpu__time_duration.sum --clock-control none \
  -k regex:"^(gemm_tc|gemm_simt|im2col|gn_|conv_epilogue|softmax_rows|vq_codebook|attn_prefill|qkv_rope|resid_rmsnorm|swiglu|prefill_|gather_last|kv_broadcast)" -c 2000 \
  --csv --log-file gpurun_out/${R}_launches_prefill_vq.csv python tools/profile_step.py > gpurun_out/p_d.log 2>&1
PG_B=32 PG_ITERS=1 timeout 400 ncu --metrics gpu__time_duration.sum --clock-control none -k regex:"^(gemm_tc|vit_|bias_act|to_f32)" -c 900 \
  --csv --log-file gpurun_out/${R}_launches_siglip.csv python tools/siglip_time.py > gpurun_out/p_f.log 2>&1
PG_B=32 PG_ITERS=1 timeout 400 ncu --set full --clock-control none --import-source on -k regex:"vit_attn_tc|gemm_tc" -s 40 -c 6 \
  -o gpurun_out/${R}_siglip python tools/siglip_time.py > gpurun_out/p_g.log 2>&1
for k in prefill_vq siglip; do python tools/summarize_launches.py gpurun_out/${R}_launches_$k.csv > gpurun_out/${R}_launches_$k.txt; done
python tools/extract_ncu.py gpurun_out/${R}_siglip.ncu-rep > gpurun_out/${R}_siglip.full.txt
rm -f gpurun_out/*.ncu-rep
head -8 gpurun_out/${R}_launches_siglip.txt
