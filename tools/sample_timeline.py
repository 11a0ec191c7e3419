"""In-kernel timeline of the fused CFG + softmax + multinomial + embed kernel inside the decode graph.
PG_TOP_P (default 1.0 = off) sets the sampler's top-p."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from plangen_b200 import JANUS_1P3B, synthetic
from plangen_b200.engine import FastJanus
B = 16; dims = JANUS_1P3B; dev = torch.device("cuda", 0)
sd = synthetic.random_state_dict(dims, dev, seed=0, with_vq=False)
eng = FastJanus(sd, dims, mode="bf16", max_batch=B, max_prompt=512, with_vq=False)
del sd
cond, neg = synthetic.layoutsam_prompts(dims, B, seed=1234)
ids, mask = synthetic.collate_cfg_batch(cond, neg, dims.pad_id, dims.n_img_tokens)
emb = eng.language_model.get_input_embeddings()(ids.to(dev))
dbg = torch.zeros(256 * 16, dtype=torch.int64, device=dev)
eng.set_option("sample_dbg_ptr", dbg.data_ptr())
eng.sample_image(emb, B, 40, mask.to(dev), 5.0, 1.0, generator=0, top_p=float(os.environ.get("PG_TOP_P", "1.0")))
torch.cuda.synchronize()
eng.set_option("sample_dbg_ptr", 0)
t = dbg.cpu().numpy().reshape(-1, 16).astype(np.float64)
t = t[t[:, 0] > 0]
t0 = t[:, 0].min()
names = ["entry", "past wait", "logits loaded + CFG", "exp done", "philox/argmax done", "token known", "embed row gathered", "exit"]
for k, nm in enumerate(names):
    v = (t[:, k] - t0) / 1e3
    print(f"  {nm:22s} min {v.min():6.2f}  p50 {np.median(v):6.2f}  max {v.max():6.2f} us")
