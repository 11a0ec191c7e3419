"""In-situ timeline of ONE decode step (plain launches + PDL): per-kernel begin/end from %globaltimer."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from plangen_b200 import JANUS_1P3B, synthetic
from plangen_b200.engine import FastJanus
B = int(os.environ.get("PG_B", "16")); dims = JANUS_1P3B; dev = torch.device("cuda", 0)
sd = synthetic.random_state_dict(dims, dev, seed=0, with_vq=False)
eng = FastJanus(sd, dims, mode="bf16", max_batch=B, max_prompt=512, with_vq=False, options={"use_graph": int(os.environ.get("PG_GRAPH", "1"))})
del sd
cond, neg = synthetic.layoutsam_prompts(dims, B, seed=1234)
ids, mask = synthetic.collate_cfg_batch(cond, neg, dims.pad_id, dims.n_img_tokens)
emb = eng.language_model.get_input_embeddings()(ids.to(dev))
step = int(os.environ.get("PG_STEP", "300"))
NS = 256
prof = torch.zeros(4 * NS, dtype=torch.int64, device=dev)
eng.set_option("prof_ptr", prof.data_ptr()); eng.set_option("prof_step", step)
eng.sample_image(emb, B, step + 3, mask.to(dev), 5.0, 1.0, generator=0)
torch.cuda.synchronize()
snap = prof[2 * NS:].cpu()
t = torch.stack([snap[:NS], snap[NS:]], 1)
used = (t[:, 1] > 0).nonzero().flatten().tolist()
t0 = int(t[used, 0].min())
names = []
# launch order of instrumented kernels in a step: head gemm, head gemm, then per layer: qkv, attn, o, norm, gu, down, norm
per_layer = ["qkv", "attn", "o", "norm1", "gu", "down", "norm2"]
labels = ["head0", "head1"] + [f"L{l}.{n}" for l in range(dims.L) for n in per_layer]
rows = [(labels[i] if i < len(labels) else str(i), (int(t[i, 0]) - t0) / 1e3, (int(t[i, 1]) - t0) / 1e3) for i in used]
print("slots used", len(used), "step span us", rows[-1][2] - rows[0][1])
import collections
dur = collections.defaultdict(list); gap = collections.defaultdict(list); excl = collections.defaultdict(list)
prev_end = None
for name, b, e in rows:
    k = name.split(".")[-1]
    dur[k].append(e - b)
    if prev_end is not None:
        gap[k].append(b - prev_end)            # negative = overlap with predecessor
        excl[k].append(e - max(b, prev_end))   # time this kernel adds to the critical path
    prev_end = max(prev_end, e) if prev_end is not None else e
print(f"{'kernel':8s} {'dur us':>8s} {'start-prev_end':>15s} {'adds to path':>13s}")
for k in ["head0", "head1"] + per_layer:
    if dur[k]:
        f = lambda v: sum(v) / max(len(v), 1)
        print(f"{k:8s} {f(dur[k]):8.2f} {f(gap[k]):15.2f} {f(excl[k]):13.2f}")
npl = len(per_layer)
for name, b, e in rows[2 + npl * 10: 2 + npl * 11]:
    print(f"  {name:12s} begin {b:9.2f} end {e:9.2f} dur {e-b:7.2f}")
print("first rows of the step (head gemms, then layer 0):")
for name, b, e in rows[:6]:
    print(f"  {name:12s} begin {b:9.2f} end {e:9.2f} dur {e-b:7.2f}")
print("last rows:")
for name, b, e in rows[-3:]:
    print(f"  {name:12s} begin {b:9.2f} end {e:9.2f} dur {e-b:7.2f}")
