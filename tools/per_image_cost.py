"""Decode-loop cost of per-image sampling settings at configs[1] (Janus-1.3B architecture, bf16, B = 16, bench prompts).

Times, alternated three times in this one process (ms per decode step = (n-token loop - 1-token loop) / (n - 1), CUDA
events, decode graph):
  scalar          scalar Python arguments, CFG 5, T 1 (the op layer passes them as a uniform settings array)
  uniform         one-value-per-image lists with every image at CFG 5, T 1 and one batch-wide seed (same graph as
                  `scalar`)
  mixed           mixed CFG / T / top-k, top-p 0.9 on half the images, one generator per image
  scalar_top_p    scalar arguments with top-p 0.9 on every image
  scalar_filters  scalar arguments with top-k 50 and top-p 0.9 on every image (the filter work `mixed` asks for)
"""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from plangen_b200 import JANUS_1P3B, synthetic
from plangen_b200.engine import FastJanus

B, N = 16, int(os.environ.get("PG_STEPS", "576"))
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

MIXED = dict(cfg_weight=[(1.0, 3.0, 5.0, 7.5)[b % 4] for b in range(B)],
             temperature=[(1.0, 0.7, 1.3)[b % 3] for b in range(B)],
             top_k=[(0, 50, 1000)[b % 3] for b in range(B)],
             top_p=[0.9 if b % 2 else 1.0 for b in range(B)])
VARIANTS = {
    "scalar": lambda: dict(cfg_weight=5.0, temperature=1.0, generator=0),
    "uniform": lambda: dict(cfg_weight=[5.0] * B, temperature=[1.0] * B, generator=0),
    "mixed": lambda: dict(MIXED, generator=[torch.Generator(device=dev).manual_seed(100 + b) for b in range(B)]),
    "scalar_top_p": lambda: dict(cfg_weight=5.0, temperature=1.0, generator=0, top_p=0.9),
    "scalar_filters": lambda: dict(cfg_weight=5.0, temperature=1.0, generator=0, top_k=50, top_p=0.9),
}


def run(n, kw):
    kw = dict(kw)
    return eng.sample_image(emb, B, n, mask, kw.pop("cfg_weight"), kw.pop("temperature"), **kw)


def loop_ms(name):
    mk = VARIANTS[name]
    run(N, mk()); run(1, mk())                     # warm: graph capture and the 1-token path
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    a, b = mk(), mk()
    ev[0].record(st)
    run(1, a)
    ev[1].record(st)
    run(N, b)
    ev[2].record(st)
    torch.cuda.synchronize()
    pre = ev[0].elapsed_time(ev[1])
    return (ev[1].elapsed_time(ev[2]) - pre) / (N - 1)


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
print(f"device: {torch.cuda.get_device_name(0)}; nvidia-smi (name, power limit, max SM clock): {smi[0] if smi else 'n/a'}")
print(f"configs[1]: B = {B}, P = {ids.shape[1]}, {N} tokens")
res = {k: [] for k in VARIANTS}
for rep in range(3):
    for k in VARIANTS:
        res[k].append(loop_ms(k))
        print(f"rep {rep} {k:14s} {res[k][-1]:.4f} ms/step", flush=True)
mean = {k: sum(v) / len(v) for k, v in res.items()}
for k in VARIANTS:
    d = mean[k] - mean["scalar"]
    print(f"{k:14s} mean {mean[k]:.4f} ms/step  vs scalar {d:+.4f} ms ({100 * d / mean['scalar']:+.2f} %)")
for ref in ("scalar_top_p", "scalar_filters"):
    d = mean["mixed"] - mean[ref]
    print(f"mixed vs {ref} {d:+.4f} ms ({100 * d / mean[ref]:+.2f} %)")
print(f"graph captures: {eng.counter('graph_captures')}")
