"""Decode-loop cost of guidance schedules at configs[1] (Janus-1.3B architecture, bf16, B = 16, bench prompts).

Times, alternated three times in this one process (ms per decode step = (n-token loop - 1-token loop) / (n - 1), CUDA
events):
  scalar      scalar Python arguments, CFG 5, T 1 (passed on as a uniform settings array), decode graph
  uniform     one-value-per-image lists with every image at CFG 5, T 1 and one batch-wide seed, the same decode graph
  ramp        a linear-ramp schedule, 1 -> w over the steps (w = 1 / 3 / 5 / 7.5 by image), decode graph
  const       the schedule with every entry 5 (its tokens are compared with `uniform`'s: they must be identical)
  stepwise    what a caller has to do without schedules: the loop in Python, one language_model.model(...) decode
              step, gen_head and cfg_sample_embed with that step's weights per token (plain launches), PG_STEPWISE
              tokens (default 256)
"""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from plangen_b200 import JANUS_1P3B, synthetic
from plangen_b200.engine import FastJanus

B, N = 16, int(os.environ.get("PG_STEPS", "576"))
N_SW = int(os.environ.get("PG_STEPWISE", "256"))
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
W = torch.tensor([(1.0, 3.0, 5.0, 7.5)[b % 4] for b in range(B)])[:, None]


def ramp(n):
    return 1.0 + (W - 1.0) * torch.linspace(0, 1, n)


VARIANTS = {
    "scalar": lambda n: dict(cfg_weight=5.0),
    "uniform": lambda n: dict(cfg_weight=[5.0] * B),
    "ramp": lambda n: dict(cfg_weight=ramp(n)),
    "const": lambda n: dict(cfg_weight=torch.full((B, n), 5.0)),
}


def run(n, name):
    return eng.sample_image(emb, B, n, mask, VARIANTS[name](n)["cfg_weight"], 1.0, generator=0)


def stepwise(n):
    """The Python loop over language_model.model / gen_head / cfg_sample_embed, weights of column i at step i."""
    sched = ramp(n)
    lm = eng.language_model.model
    tokens = torch.zeros(B, n, dtype=torch.int32, device=dev)
    per_step = eng.philox_offset_per_step(B)
    out = lm(inputs_embeds=emb, attention_mask=mask, use_cache=True)
    h = out.last_hidden_state[:, -1, :]
    for i in range(n):
        logits = eng.gen_head(h)
        x = eng.cfg_sample_embed(logits, sched[:, i].tolist(), 1.0, 0, per_step * i, i, n, tokens)
        if i + 1 < n:
            out = lm(inputs_embeds=x.view(2 * B, 1, -1), past_key_values=out.past_key_values)
            h = out.last_hidden_state[:, -1, :]
    return tokens


def per_step_ms(fn, n):
    fn(n); fn(1)                                   # warm: graph capture and the 1-token path
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    ev[0].record(st)
    fn(1)
    ev[1].record(st)
    fn(n)
    ev[2].record(st)
    torch.cuda.synchronize()
    return (ev[1].elapsed_time(ev[2]) - ev[0].elapsed_time(ev[1])) / (n - 1)


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
print(f"device: {torch.cuda.get_device_name(0)}; nvidia-smi (name, power limit, max SM clock): {smi[0] if smi else 'n/a'}")
print(f"configs[1]: B = {B}, P = {ids.shape[1]}, {N} tokens (stepwise: {N_SW} tokens)")
names = list(VARIANTS) + ["stepwise"]
res = {k: [] for k in names}
for rep in range(3):
    for k in names:
        res[k].append(per_step_ms(stepwise, N_SW) if k == "stepwise" else per_step_ms(lambda n, k=k: run(n, k), N))
        print(f"rep {rep} {k:9s} {res[k][-1]:.4f} ms/step", flush=True)
mean = {k: sum(v) / len(v) for k, v in res.items()}
for k in names:
    d = mean[k] - mean["scalar"]
    print(f"{k:9s} mean {mean[k]:.4f} ms/step  vs scalar {d:+.4f} ms ({100 * d / mean['scalar']:+.2f} %)  "
          f"range {min(res[k]):.4f}-{max(res[k]):.4f}")
d = mean["ramp"] - mean["uniform"]
print(f"ramp vs uniform {d:+.4f} ms ({100 * d / mean['uniform']:+.2f} %)")
same = torch.equal(run(N, "const"), run(N, "uniform"))
print(f"const schedule tokens == uniform tokens ({B} x {N}): {same}")
print(f"graph captures: {eng.counter('graph_captures')}")
