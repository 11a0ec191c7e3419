"""Cost of image-token log-probabilities at configs[1] (Janus-1.3B architecture, bf16, B = 16, bench prompts).

Alternated three times in this one process, CUDA events:
  1. ms per decode step = (n-token loop - 1-token loop) / (n - 1), decode graph:
       uniform / uniform_lp   one value per image, every image at CFG 5, T 1, one batch-wide seed; log-probs off / on
       mixed / mixed_lp       mixed CFG / T / top-k, top-p 0.9 on half the images, one generator per image; off / on
  2. ms per batch of scoring 576 given tokens per image: the teacher-forced scorer (one prefill over prompt + image
     tokens, one wide gen_head) against the teacher-forced decode loop (edit_region all 0) with log-probs, on the same
     prompts and tokens, on an engine built with max_prompt >= P + 575.
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
cond, neg = synthetic.layoutsam_prompts(dims, B, seed=1234)
ids, mask = synthetic.collate_cfg_batch(cond, neg, dims.pad_id, dims.n_img_tokens)
ids, mask = ids.to(dev), mask.to(dev)
P = ids.shape[1]
eng_long = FastJanus(sd, dims, mode="bf16", max_batch=B, max_prompt=P + dims.n_img_tokens, with_vq=False)
del sd
emb = eng.language_model.get_input_embeddings()(ids)
st = torch.cuda.current_stream(dev)

MIXED = dict(cfg_weight=[(1.0, 3.0, 5.0, 7.5)[b % 4] for b in range(B)],
             temperature=[(1.0, 0.7, 1.3)[b % 3] for b in range(B)],
             top_k=[(0, 50, 1000)[b % 3] for b in range(B)],
             top_p=[0.9 if b % 2 else 1.0 for b in range(B)])
VARIANTS = {
    "uniform": lambda: dict(cfg_weight=[5.0] * B, temperature=[1.0] * B, generator=0),
    "uniform_lp": lambda: dict(cfg_weight=[5.0] * B, temperature=[1.0] * B, generator=0, return_logprobs=True),
    "mixed": lambda: dict(MIXED, generator=[torch.Generator(device=dev).manual_seed(100 + b) for b in range(B)]),
    "mixed_lp": lambda: dict(MIXED, generator=[torch.Generator(device=dev).manual_seed(100 + b) for b in range(B)],
                             return_logprobs=True),
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


# tokens to score: the engine's own samples
tokens = run(N, dict(cfg_weight=5.0, temperature=1.0, generator=0))
forced = {"edit_region": torch.zeros(B, N, dtype=torch.int32)}


def score_ms():
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record(st)
    lp = eng_long.score_image_tokens(tokens=ids, mask=mask[:, : P + N], image_tokens=tokens, cfg_weight=5.0)
    ev[1].record(st)
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]), lp


def forced_loop_ms():
    e2 = eng_long.language_model.get_input_embeddings()(ids)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record(st)
    _, lp = eng_long.sample_image(e2, B, N, mask, 5.0, 1.0, generator=0, batch=forced, gt_labels=tokens,
                                  use_teacher_forcing=True, return_logprobs=True)
    ev[1].record(st)
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]), lp


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
print(f"device: {torch.cuda.get_device_name(0)}; nvidia-smi (name, power limit, max SM clock): {smi[0] if smi else 'n/a'}")
print(f"configs[1]: B = {B}, P = {P}, {N} tokens; scorer engine max_prompt = {P + dims.n_img_tokens}")
score_ms(); forced_loop_ms()                        # warm both paths
res = {k: [] for k in list(VARIANTS) + ["scorer", "forced_loop"]}
for rep in range(3):
    for k in VARIANTS:
        res[k].append(loop_ms(k))
        print(f"rep {rep} {k:12s} {res[k][-1]:.4f} ms/step", flush=True)
    t_s, lp_s = score_ms()
    t_l, lp_l = forced_loop_ms()
    res["scorer"].append(t_s); res["forced_loop"].append(t_l)
    print(f"rep {rep} scorer {t_s:.2f} ms/batch  teacher-forced loop {t_l:.2f} ms/batch", flush=True)
mean = {k: sum(v) / len(v) for k, v in res.items()}
for off, on in (("uniform", "uniform_lp"), ("mixed", "mixed_lp")):
    d = mean[on] - mean[off]
    print(f"{on:12s} mean {mean[on]:.4f} ms/step vs {off} {mean[off]:.4f}: {d:+.4f} ms ({100 * d / mean[off]:+.2f} %)")
print(f"scorer mean {mean['scorer']:.2f} ms/batch, teacher-forced loop {mean['forced_loop']:.2f} ms/batch: "
      f"{mean['forced_loop'] / mean['scorer']:.1f}x")
diff = (lp_s - lp_l).abs()
print(f"scorer vs loop log-probs (two bf16 evaluations): max |diff| {diff.max().item():.4f}, mean {diff.mean().item():.5f}; "
      f"all finite: {bool(torch.isfinite(lp_s).all())}")
