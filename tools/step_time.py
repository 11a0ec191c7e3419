"""Decode-loop timing sweeps over engine options (one engine, graph re-captured per setting).

PG_TOP_P=1.0,0.9 times the sampler's top-p settings instead, alternated three times in this one process."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from plangen_b200 import JANUS_1P3B, synthetic
from plangen_b200.engine import FastJanus

B = int(os.environ.get("PG_B", "16"))
dims = JANUS_1P3B
dev = torch.device("cuda", 0)
sd = synthetic.random_state_dict(dims, dev, seed=0, with_vq=False)
eng = FastJanus(sd, dims, mode="bf16", max_batch=B, max_prompt=512, with_vq=False)
del sd
cond, neg = synthetic.layoutsam_prompts(dims, B, seed=1234)
ids, mask = synthetic.collate_cfg_batch(cond, neg, dims.pad_id, dims.n_img_tokens)
ids, mask = ids.to(dev), mask.to(dev)
emb = eng.language_model.get_input_embeddings()(ids)
st = torch.cuda.current_stream(dev)
DEFAULTS = {"use_pdl": 1, "use_graph": 1, "use_tc": 1, "attn_impl": 3}


def loop_ms(n=576, top_p=1.0):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    eng.sample_image(emb, B, n, mask, 5.0, 1.0, generator=0, top_p=top_p)   # warm (captures the graph)
    eng.sample_image(emb, B, 1, mask, 5.0, 1.0, generator=0, top_p=top_p)   # warm the 1-token path too (its first run is
    torch.cuda.synchronize()                                        # ~90 ms slower, which used to deflate the first ms/step by 0.16 ms)
    ev[0].record(st)
    eng.sample_image(emb, B, 1, mask, 5.0, 1.0, generator=0, top_p=top_p)
    ev[1].record(st)
    eng.sample_image(emb, B, n, mask, 5.0, 1.0, generator=0, top_p=top_p)
    ev[2].record(st)
    torch.cuda.synchronize()
    pre = ev[0].elapsed_time(ev[1])
    return round(pre, 2), round((ev[1].elapsed_time(ev[2]) - pre) / (n - 1), 4)


top_ps = [float(x) for x in os.environ.get("PG_TOP_P", "").split(",") if x]
if top_ps:
    for rep in range(3):
        for p in top_ps:
            print(f"top_p={p} (prefill ms, ms/decode step)", loop_ms(top_p=p), flush=True)
    sys.exit(0)
sweeps = [s for s in os.environ.get("PG_SWEEP", "").split(";") if s]
print("baseline (prefill ms, ms/decode step)", loop_ms(), flush=True)
for s in sweeps:
    kv = dict(x.split("=") for x in s.split(","))
    for k, v in kv.items():
        eng.set_option(k, int(v))
    print(s, loop_ms(), flush=True)
    for k in kv:
        eng.set_option(k, DEFAULTS.get(k, 0))
