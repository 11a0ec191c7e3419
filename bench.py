#!/usr/bin/env python
"""Benchmark of the PlanGen CFG image-token decode path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

One "step" = one batch through the hot path: prompt embed + prefill + 576 x (gen_head, CFG, Philox
sample, embed, KV-cached decode step) + VQ decode_code, for BASELINE.json configs[1]
(layout2image, Janus-1.3B architecture, random-init weights, bf16, batch 16 = 32 rows with the
cond/uncond pair, synthetic LayoutSAM-shaped prompts with 4-8 boxes).  Prints ONE JSON line.

  value     images/s, whole job, inputs already resident in HBM (CUDA-event timed, max over ranks)
  e2e       same metric through the public host-buffer API (pinned-host ids/mask -> uint8 images in
            host memory; H2D and D2H inside the timed region)
  roofline  the dominant kernel (TMA-staged KV-cache decode attention) timed alone with CUDA events
  cpu_baseline  the oracle port of the reference PyTorch path on the box's host cores (bounded sample)
  extra     the other BASELINE.json configurations (uni_2stage, mmu, Janus-Pro-7B), measured after the timed region

`--impl reference` times the reference's own CPU implementation of the path: the oracle restatement
of System.t2i / sample_image (oracle/janus_oracle.py; the reference itself cannot be imported here,
see DESIGN.md) on all host threads: one full 576-token image per step, wall clock, nothing extrapolated.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "images/sec/box (576-tok CFG decode, layout2image bf16 batch 16)"
UNIT = "images/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--model", default="janus-1.3b", choices=["janus-1.3b", "janus-pro-7b"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the bounded configs[2]/[3]/[4] measurements after the timed region")
    ap.add_argument("--option", action="append", default=[], help="engine option key=value")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (uint8 images, image tokens) and "
                         "which batch rows they are as DIR/<name>.npy in float32, at most 64 MB in all, so that two builds "
                         "can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    return args


# ----------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        # under load = upper half of the samples (idle gaps between steps pull the clock down)
        load = sm[len(sm) // 2:] if sm else []
        med = load[len(load) // 2] if load else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------- reference arm (CPU)
def cpu_reference_sample(model_name: str, threads: int, prompt_len: int = 256, rows_b: int = 1, n_decode: int = 24,
                         vq: bool = True, sd=None):
    """Oracle port of the reference path on host cores: prefill + n_decode decode steps (+ VQ decode of
    one image), extrapolated to a 576-token image.  Returns a dict incl. images/s."""
    import torch
    from oracle import janus_oracle as O
    torch.set_num_threads(threads)
    d = O.PRESETS[model_name]
    if sd is None:
        sd = O.init_state_dict(d, seed=0, with_vq=vq)
    cond, neg = O.synthetic_prompts(d, rows_b, seed=1234, lo=prompt_len, hi=prompt_len)
    ids, mask = O.t2i_infer_collate_batch(cond, neg, d.pad_id, d.n_img_tokens)
    times = []

    def timed_forward(**kw):
        t0 = time.perf_counter()
        out = O.llama_model_forward(sd, d, **kw)
        times.append(time.perf_counter() - t0)
        return out

    g = torch.Generator().manual_seed(0)
    t0 = time.perf_counter()
    with torch.inference_mode():
        emb = O.embed_tokens(sd, ids)
        toks = O.sample_image(sd, d, emb, rows_b, n_decode + 1, mask, 5.0, 1.0, O.make_torch_sampler(g), mode="fp32",
                              lm_forward=timed_forward)
    loop_s = time.perf_counter() - t0
    prefill_s = times[0]
    dec = sorted(times[1:])
    step_s = dec[len(dec) // 2]
    other_s = max(loop_s - sum(times), 0.0) / (n_decode + 1)        # head + CFG + sample + embed per token
    vq_s = 0.0
    if vq:
        codes = torch.randint(0, d.img_vocab, (1, d.n_img_tokens), dtype=torch.int32)
        t0 = time.perf_counter()
        with torch.inference_mode():
            O.decode_code(sd, d, codes, [1, d.code_dim, d.grid, d.grid])
        vq_s = time.perf_counter() - t0
    n = d.n_img_tokens
    per_batch = prefill_s + (n - 1) * step_s + n * other_s + rows_b * vq_s
    return {"images_per_s": rows_b / per_batch, "prefill_s": prefill_s, "ms_per_decode_step": 1e3 * step_s,
            "vq_decode_s_per_image": vq_s, "rows": 2 * rows_b, "prompt_len": prompt_len, "n_decode_timed": n_decode,
            "sample_wall_s": loop_s + vq_s}


def cpu_reference_full_image(model_name: str, threads: int, prompt_len: int = 256, sd=None, images: int = 1,
                             warmup: int = 1):
    """`images` full images, one after the other, through the oracle port of System.t2i on host cores, nothing
    extrapolated: each is embed + prefill + 575 decode steps (each LlamaModel.forward timed) + gen_head / CFG /
    sampling / embed per token + VQ decode_code.  `warmup` untimed short passes (prefill + 2 tokens) page the weights
    in first.  BASELINE configs[0]: B=1 (R=2 rows with the CFG pair), P=256, fp32.  wall_s and loop_s cover all the
    images; prefill_s and vq_s are per image (median, mean)."""
    import torch
    from oracle import janus_oracle as O
    torch.set_num_threads(threads)
    d = O.PRESETS[model_name]
    if sd is None:
        sd = O.init_state_dict(d, seed=0, with_vq=True)
    cond, neg = O.synthetic_prompts(d, 1, seed=1234, lo=prompt_len, hi=prompt_len)
    ids, mask = O.t2i_infer_collate_batch(cond, neg, d.pad_id, d.n_img_tokens)
    times = []

    def timed_forward(**kw):
        t0 = time.perf_counter()
        out = O.llama_model_forward(sd, d, **kw)
        times.append(time.perf_counter() - t0)
        return out

    for _ in range(warmup):
        g = torch.Generator().manual_seed(0)
        with torch.inference_mode():
            O.sample_image(sd, d, O.embed_tokens(sd, ids), 1, 3, mask, 5.0, 1.0, O.make_torch_sampler(g), mode="fp32")
    prefill, dec, loop_s, vq_s = [], [], 0.0, 0.0
    t0 = time.perf_counter()
    for _ in range(images):
        times.clear()
        g = torch.Generator().manual_seed(0)
        ta = time.perf_counter()
        with torch.inference_mode():
            emb = O.embed_tokens(sd, ids)
            toks = O.sample_image(sd, d, emb, 1, d.n_img_tokens, mask, 5.0, 1.0, O.make_torch_sampler(g), mode="fp32",
                                  lm_forward=timed_forward)
            tb = time.perf_counter()
            O.decode_code(sd, d, toks.to(torch.int32), [1, d.code_dim, d.grid, d.grid])
        tc = time.perf_counter()
        loop_s, vq_s = loop_s + tb - ta, vq_s + tc - tb
        prefill.append(times[0])
        dec += times[1:]
    wall_s = time.perf_counter() - t0
    prefill.sort()
    dec.sort()
    return {"wall_s": wall_s, "images": images, "loop_s": loop_s, "vq_s": vq_s / images,
            "prefill_s": prefill[len(prefill) // 2],
            "ms_per_decode_step_median": 1e3 * dec[len(dec) // 2], "ms_per_decode_step_p90": 1e3 * dec[int(0.9 * len(dec))],
            "decode_steps_timed": len(dec), "rows": 2, "prompt_len": prompt_len}


def cpu_b16_estimate(model_name: str, threads: int, sd, vq_s_per_image: float):
    """What the same CPU path would do at the B200 arm's batch (B=16, R=32): a bounded measurement - prefill of 32 rows
    at P=64 scaled linearly in tokens to the bench's P, 4 decode steps at R=32 (weight streaming dominates a CPU step,
    the context length barely matters), VQ decode at the measured per-image cost - labelled an ESTIMATE."""
    import torch
    from oracle import janus_oracle as O
    torch.set_num_threads(threads)
    d = O.PRESETS[model_name]
    B, P_meas, P_bench = 16, 64, 354
    cond, neg = O.synthetic_prompts(d, B, seed=99, lo=P_meas, hi=P_meas)
    ids, mask = O.t2i_infer_collate_batch(cond, neg, d.pad_id, d.n_img_tokens)
    times = []

    def timed_forward(**kw):
        t0 = time.perf_counter()
        out = O.llama_model_forward(sd, d, **kw)
        times.append(time.perf_counter() - t0)
        return out

    g = torch.Generator().manual_seed(0)
    t0 = time.perf_counter()
    with torch.inference_mode():
        O.sample_image(sd, d, O.embed_tokens(sd, ids), B, 5, mask, 5.0, 1.0, O.make_torch_sampler(g), mode="fp32",
                       lm_forward=timed_forward)
    loop = time.perf_counter() - t0
    other = max(loop - sum(times), 0.0) / 5
    step = sorted(times[1:])[len(times[1:]) // 2]
    n = d.n_img_tokens
    per_batch = times[0] * P_bench / P_meas + (n - 1) * step + n * other + B * vq_s_per_image
    return {"images_per_s_estimate": B / per_batch, "rows": 2 * B, "prefill_s_at_P64": times[0], "ms_per_decode_step_r32": 1e3 * step,
            "how": "prefill(R=32, P=64) x 354/64 + 575 x median of 4 decode steps at R=32 + 576 x head/CFG/sample/embed + 16 x VQ"}


def run_reference_arm(args):
    """Reference arm: the reference's CPU PyTorch path (oracle port; the reference itself cannot be imported, DESIGN.md)
    on all host threads.  One step is one full 576-token image of BASELINE configs[0] (B=1, R=2, P=256, fp32): embed +
    prefill + 575 decode steps + VQ decode, wall clock, nothing extrapolated; the timed region is --steps K such images
    (~25-30 s each).  --warmup W: W short untimed passes (prefill + 2 tokens) page the weights in."""
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    from oracle import janus_oracle as O
    d = O.PRESETS[args.model]
    sd = O.init_state_dict(d, seed=0, with_vq=True)
    r = cpu_reference_full_image(args.model, threads, prompt_len=256, sd=sd, images=args.steps, warmup=args.warmup)
    ips = args.steps / r["wall_s"]
    b16 = cpu_b16_estimate(args.model, threads, sd, r["vq_s"])
    line = {
        "metric": METRIC, "value": ips, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * r["wall_s"] / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[0] layout2image (task_type=uni), Janus-1.3B-arch random init, B=1 (R=2 rows with the CFG "
                               "pair), P=256, 576 VQ tokens, CFG 5, fp32 on CPU; reference arm = oracle port of System.t2i / "
                               "sample_image (the reference cannot be imported here); timed region = --steps full images, one "
                               "per step (embed + prefill + 575 decode steps + VQ decode), wall clock, no extrapolation",
                   "same_config_as_b200_arm": False,
                   "note": "the B200 arm runs configs[1] (B=16 per GPU, bf16); cpu_baseline_b16 below estimates this CPU path at B=16"},
        "timed": {"images": r["images"], "wall_s": r["wall_s"], "prefill_s": r["prefill_s"], "decode_steps": r["decode_steps_timed"],
                  "ms_per_decode_step_median": r["ms_per_decode_step_median"], "ms_per_decode_step_p90": r["ms_per_decode_step_p90"],
                  "vq_decode_s_per_image": r["vq_s"]},
        "cpu_baseline": {"value": ips, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": "--steps full images: R=2 rows, P=256: prefill + 575 decode steps + VQ decode (nothing extrapolated)",
                         "ms_per_decode_step": r["ms_per_decode_step_median"], "ms_per_decode_step_p90": r["ms_per_decode_step_p90"],
                         "prefill_s": r["prefill_s"], "vq_decode_s_per_image": r["vq_s"], "torch": torch.__version__},
        "cpu_baseline_b16": b16,
        "e2e": {"value": ips, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- B200 arm
def kernel_roofline(eng, kv_start, lens, P: int, peaks: dict, iters: int = 6):
    """Dominant kernel of the decode step timed alone (29 % of a mid-sequence step in the ncu launch list, 44 % of the
    in-graph critical path, profiles/): the KV-cache
    decode attention `attn_decode_v5_kernel`, one launch per layer, rotating over all L layers so the K/V
    tiles come from HBM (L x ~130 MB >> 126 MB L2).  Position = the middle of the 576-token loop.
    achieved = algorithmic K+V bytes per launch / CUDA-event time per launch on the launching stream."""
    import ctypes as C
    import torch
    from plangen_b200 import _lib
    d = eng.dims
    R = len(lens)
    pos = P + d.n_img_tokens // 2
    st = torch.cuda.current_stream(eng.device)
    sp = C.c_void_p(st.cuda_stream)
    _lib.check(eng._lib.pg_debug_zero_part(eng._h, R * 3 * d.H * d.head_dim * 4, sp))
    eng.set_option("attn_test_alias_p", P)                 # as in the real step: repeated prompt rows read their source row's strips

    def one_pass():
        for l in range(d.L):
            _lib.check(eng._lib.pg_test_attn_decode(eng._h, C.c_void_p(kv_start.data_ptr()), R, pos, l, sp))

    for _ in range(3):
        one_pass()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(iters):
        one_pass()
    e1.record(st)
    torch.cuda.synchronize()
    per_launch_s = e0.elapsed_time(e1) / 1e3 / (iters * d.L)
    eng.set_option("attn_test_alias_p", 0)
    kv_tok = 2 * d.H * d.head_dim * 2                      # K and V bytes per cached token per row per layer (bf16)
    alg_bytes = sum((ln + d.n_img_tokens // 2) * kv_tok for ln in lens) + R * kv_tok
    achieved = alg_bytes / per_launch_s / 1e9
    peak = peaks.get("hbm_gbs")
    which = "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    if not peak:
        peak, which = 6650.0, "fallback (B200_PROFILING.md)"
    return {"bound": "hbm", "kernel": "attn_decode_v5_kernel (KV-cache decode attention, paired CFG batch, 1 launch/layer)",
            "achieved": achieved, "peak": peak, "peak_source": which, "unit": "GB/s", "frac": achieved / peak,
            "traffic": _ncu_traffic_bytes(), "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum of one launch, ncu --set full "
            "at step ~290 of the same workload (profiles/r02_attn_decode.full.txt); algorithmic K+V bytes there ~129 MB.  Below 1x: the "
            "16 unconditional rows repeat one negative prompt and read its K/V from the first copy's strips, served by L2 "
            "(1.03x with that switched off, 1.14x in round 1 before the first / last tile of a row were trimmed to their valid tokens)",
            "algorithmic_bytes_per_launch": alg_bytes, "us_per_launch": per_launch_s * 1e6, "position": pos}


def _ncu_traffic_bytes():
    """DRAM bytes of one attention launch from the committed ncu extract (None if the file is missing)."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r02_attn_decode.full.txt")
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    total, seen = 0.0, 0
    try:
        with open(path) as f:
            for line in f:
                parts = line.split()
                if len(parts) == 3 and parts[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum") and parts[2] in scale:
                    total += float(parts[1]) * scale[parts[2]]
                    seen += 1
    except OSError:
        return None
    return int(total) if seen == 2 else None


DUMP_BYTES = 64 << 20


def dump_outputs(path: str, images, tokens):
    """Write one step's (B, 3, H, W) uint8 images and (B, n) image tokens, and the batch rows they are, as float32 .npy
    files.  When the batch does not fit DUMP_BYTES, the rows are a fixed seeded sample of whole images."""
    import numpy as np
    import torch
    n = images.shape[0]
    per_row = 4 * (images[0].numel() + tokens[0].numel() + 1)
    keep = min(n, DUMP_BYTES // per_row)
    rows = torch.arange(n)
    if keep < n:
        rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:keep].sort().values
    out = {"images": images[rows.to(images.device)], "tokens": tokens[rows.to(tokens.device)], "rows": rows}
    os.makedirs(path, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy().astype(np.float32))


def _timed(st, fn):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    out = fn()
    e1.record(st)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def extra_configs(dev, peaks):
    """The other BASELINE.json configurations, measured AFTER the timed region of the headline config (rank 0, one GPU,
    bounded: one warm + one timed pass each, CUDA events on the launching stream).  Not part of `value`.
      configs[2]  uni_2stage per-GPU share: stage-1 greedy layout-text decode of 64 rows (prompts 80-160 tokens, 200 new
                  tokens, eos never hit) + stage-2 CFG image decode at B=64 (R=128 rows)
      configs[3]  mmu per-GPU share: SigLIP-L tower + aligner on 128 images, scatter into 620-token prompts, prefill +
                  64 greedy tokens for 128 rows
      configs[4]  Janus-Pro-7B architecture, layout2image B=32 per GPU (R=64 rows)"""
    import gc
    import torch
    from plangen_b200 import JANUS_1P3B, JANUS_7B, synthetic
    from plangen_b200.engine import FastJanus
    peak = peaks.get("hbm_gbs") or 6650.0
    tpeak = peaks.get("bf16_tflops_sustained") or 1369.6
    st = torch.cuda.current_stream(dev)
    out = {}

    def loop_bytes(eng, dims, lens, n_new, head_bytes):
        kvb = 2 * dims.L * dims.D * 2
        return eng.weight_bytes_per_step + head_bytes + len(lens) * (sum(lens) / len(lens) + n_new / 2) * kvb + len(lens) * kvb

    def text_batch(dims, rows, P, seed):
        g = torch.Generator().manual_seed(seed)
        lens = torch.randint(P // 2, P + 1, (rows,), generator=g).tolist()
        lens[0] = P
        ids = torch.full((rows, P), dims.pad_id, dtype=torch.int32)
        mask = torch.zeros(rows, P, dtype=torch.int32)
        for r, n in enumerate(lens):
            ids[r, P - n:] = torch.randint(0, dims.pad_id, (n,), generator=g, dtype=torch.int32)
            mask[r, P - n:] = 1
        return ids.to(dev), mask.to(dev), lens

    # ---- configs[2] and configs[3] on one Janus-1.3B engine (64 images / 128 text rows per GPU, vision tower built)
    dims = JANUS_1P3B
    sd = synthetic.random_state_dict(dims, dev, seed=0, with_vq=True, with_lm_head=True, with_vision=True)
    eng = FastJanus(sd, dims, mode="bf16", max_batch=64, max_prompt=640, device=str(dev), max_images=128)
    del sd
    ids, mask, lens = text_batch(dims, 64, 160, 5)
    emb = eng.language_model.get_input_embeddings()(ids)
    eos, N = dims.vocab - 1, 200
    gen = lambda n: eng.language_model.generate(inputs_embeds=emb, attention_mask=mask, pad_token_id=eos, eos_token_id=eos, max_new_tokens=n)
    gen(N)
    t1, _ = _timed(st, lambda: gen(1))
    tn, _ = _timed(st, lambda: gen(N))
    step1 = (tn - t1) / (N - 1)
    lm_head_extra = dims.vocab * dims.D * 2 - (dims.img_embed * dims.D + dims.img_vocab * dims.img_embed) * 2
    cond, neg = synthetic.layoutsam_prompts(dims, 64, seed=77)
    ids2, mask2 = synthetic.collate_cfg_batch(cond, neg, dims.pad_id, dims.n_img_tokens)
    ids2, mask2 = ids2.to(dev), mask2.to(dev)
    P2 = ids2.shape[1]
    lens2 = (mask2[:, :P2] != 0).sum(1).tolist()
    run2 = lambda: eng.images_to_uint8(eng.t2i(tokens=ids2, mask=mask2, cfg_weight=5.0, temperature=1.0)[0])
    run2()
    t2, _ = _timed(st, run2)
    e2 = eng.language_model.get_input_embeddings()(ids2)
    tp, _ = _timed(st, lambda: eng.sample_image(e2, 64, 1, mask2, 5.0, 1.0, generator=0))
    tl, _ = _timed(st, lambda: eng.sample_image(e2, 64, dims.n_img_tokens, mask2, 5.0, 1.0, generator=0))
    step2 = (tl - tp) / (dims.n_img_tokens - 1)
    out["configs[2] uni_2stage, 64 prompts per GPU"] = {
        "images_per_s": 64 / ((tn + t2) / 1e3), "stage1_ms": tn, "stage1_ms_per_greedy_step": step1, "stage1_tokens_per_s": 64 / step1 * 1e3,
        "stage1_step_frac_of_hbm_peak": loop_bytes(eng, dims, lens, N, lm_head_extra) / (step1 / 1e3) / 1e9 / peak,
        "stage2_ms": t2, "stage2_images_per_s": 64 / (t2 / 1e3), "stage2_ms_per_decode_step": step2,
        "stage2_step_frac_of_hbm_peak": loop_bytes(eng, dims, lens2, dims.n_img_tokens, 0) / (step2 / 1e3) / 1e9 / peak,
        "shape": f"stage 1: 64 rows, prompts 80-160 tokens, {N} greedy tokens (lm_head 102400); stage 2: B=64 (R=128 rows), P={P2}, 576 tokens + VQ decode"}
    # mmu: 128 rows, one image each: tower + aligner + scatter, then prefill + greedy tokens
    nI, T, n_new = 128, 620, 64
    g = torch.Generator().manual_seed(9)
    pix = (torch.rand(nI, 1, 3, dims.sig_image, dims.sig_image, generator=g) * 2 - 1).to(dev)
    idm = torch.randint(1, dims.pad_id, (nI, T), generator=g, dtype=torch.int32).to(dev)
    seq = torch.zeros(nI, T, dtype=torch.bool, device=dev)
    seq[:, 8:8 + dims.sig_patches] = True
    embm = torch.ones(nI, 1, dims.sig_patches, dtype=torch.bool, device=dev)
    am = torch.ones(nI, T, dtype=torch.int32, device=dev)
    front = lambda: eng.prepare_inputs_embeds(idm, pix, seq, embm)
    front()
    tf, xm = _timed(st, front)
    genm = lambda n: eng.language_model.generate(inputs_embeds=xm, attention_mask=am, pad_token_id=eos, eos_token_id=eos, max_new_tokens=n)
    genm(2)
    tg1, _ = _timed(st, lambda: genm(1))
    tgn, _ = _timed(st, lambda: genm(n_new))
    W, L, NP, F = dims.sig_width, dims.sig_layers, dims.sig_patches, dims.sig_mlp
    flop_img = 2 * (L * (4 * W * W + 2 * W * F) + 3 * dims.sig_patch ** 2 * W + W * dims.D + dims.D * dims.D) * NP + L * 4 * NP * NP * W
    out["configs[3] mmu, 128 images per GPU"] = {
        "images_per_s": nI / ((tf + tgn) / 1e3), "front_end_ms": tf, "front_end_images_per_s": nI / (tf / 1e3),
        "front_end_tflops": flop_img * nI / (tf / 1e3) / 1e12, "front_end_frac_of_sustained_bf16_peak": flop_img * nI / (tf / 1e3) / 1e12 / tpeak,
        "prefill_plus_first_token_ms": tg1, "ms_per_greedy_step": (tgn - tg1) / (n_new - 1),
        "shape": f"128 x (3,384,384) images -> SigLIP-L/16 + aligner + scatter into T={T} prompts; prefill + {n_new} greedy tokens, 128 rows"}
    del eng, emb, e2, xm, pix
    gc.collect()
    torch.cuda.empty_cache()
    # ---- configs[4]: Janus-Pro-7B architecture, B=32 per GPU
    dims = JANUS_7B
    sd = synthetic.random_state_dict(dims, dev, seed=0, with_vq=True)
    eng = FastJanus(sd, dims, mode="bf16", max_batch=32, max_prompt=512, device=str(dev))
    del sd
    torch.cuda.empty_cache()
    cond, neg = synthetic.layoutsam_prompts(dims, 32, seed=1234)
    ids7, mask7 = synthetic.collate_cfg_batch(cond, neg, dims.pad_id, dims.n_img_tokens)
    ids7, mask7 = ids7.to(dev), mask7.to(dev)
    P7 = ids7.shape[1]
    lens7 = (mask7[:, :P7] != 0).sum(1).tolist()
    run7 = lambda: eng.images_to_uint8(eng.t2i(tokens=ids7, mask=mask7, cfg_weight=5.0, temperature=1.0)[0])
    e7 = eng.language_model.get_input_embeddings()(ids7)
    eng.sample_image(e7, 32, 8, mask7, 5.0, 1.0, generator=0)                                  # warm (graph capture)
    tp7, _ = _timed(st, lambda: eng.sample_image(e7, 32, 1, mask7, 5.0, 1.0, generator=0))
    t7, _ = _timed(st, run7)
    tl7, _ = _timed(st, lambda: eng.sample_image(e7, 32, dims.n_img_tokens, mask7, 5.0, 1.0, generator=0))
    step7 = (tl7 - tp7) / (dims.n_img_tokens - 1)
    out["configs[4] Janus-Pro-7B-arch layout2image, B=32 per GPU"] = {
        "images_per_s": 32 / (t7 / 1e3), "ms_per_batch": t7, "prefill_ms": tp7, "ms_per_decode_step": step7,
        "decode_step_frac_of_hbm_peak": loop_bytes(eng, dims, lens7, dims.n_img_tokens, 0) / (step7 / 1e3) / 1e9 / peak,
        "shape": f"R=64 rows, P={P7}, 576 tokens, CFG 5 + VQ decode"}
    del eng
    gc.collect()
    torch.cuda.empty_cache()
    return out


def run_b200_arm(args):
    import torch
    import torch.distributed as dist
    from plangen_b200 import JANUS_1P3B, JANUS_7B
    from plangen_b200.engine import FastJanus
    from plangen_b200 import synthetic, dp

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: plangen_b200 has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"        # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
        dist.init_process_group("nccl", device_id=dev)
    dims = JANUS_1P3B if args.model == "janus-1.3b" else JANUS_7B
    B = args.batch
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass

    sd = synthetic.random_state_dict(dims, dev, seed=0, with_vq=True)
    opts = {}
    for kv in args.option:
        k, v = kv.split("=")
        opts[k] = int(v)
    eng = FastJanus(sd, dims, mode="bf16", max_batch=B, max_prompt=512, device=str(dev), options=opts)
    sd_cpu_needed = (rank == 0 and world == 1 and not args.no_cpu_baseline)
    if not sd_cpu_needed:
        del sd
    torch.cuda.empty_cache()

    # each rank decodes its own batches (weak scaling): batch index = step * world + rank
    def batch_for(step):
        cond, neg = synthetic.layoutsam_prompts(dims, B, seed=1234 + step * world + rank)
        return synthetic.collate_cfg_batch(cond, neg, dims.pad_id, dims.n_img_tokens)

    total = args.warmup + args.steps
    host = [batch_for(i) for i in range(total)]
    dev_batches = [(i.to(dev), m.to(dev)) for i, m in host]
    pinned = [(i.pin_memory(), m.pin_memory()) for i, m in host]
    out_host = torch.empty(B, 3, dims.img_size, dims.img_size, dtype=torch.uint8, pin_memory=True)

    def step_resident(k):
        ids, mask = dev_batches[k]
        dec, _ = eng.t2i(tokens=ids, mask=mask, cfg_weight=5.0, temperature=1.0)
        return eng.images_to_uint8(dec)

    def run_resident(ks):
        # every rank decodes its own batches back to back (no collective in the data path, SURVEY §8e); the images
        # of all ranks are gathered ONCE at the end of the job, inside the timed region
        imgs = [step_resident(k) for k in ks]
        return dp.gather_images(torch.cat(imgs, 0), world)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    run_resident(range(args.warmup))
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    eng.set_option("reset_launches", 0)
    st = torch.cuda.current_stream(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(st)
    images_out = run_resident(range(args.warmup, total))
    e1.record(st)
    barrier()
    elapsed = dp.max_over_ranks(e0.elapsed_time(e1) / 1e3, dev)
    launches = eng.counter("launches")
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # the gathered images are rank-major: rank 0's last batch sits at the end of its own steps
        dump_outputs(args.dump_outputs, images_out[(args.steps - 1) * B:args.steps * B], eng.last_tokens)
    del images_out

    # decode-step time alone (graph replays), for the roofline of the step
    P = dev_batches[args.warmup][0].shape[1]
    lens = (dev_batches[args.warmup][1][:, :P] != 0).sum(1).tolist()

    # end-to-end through the host-buffer API
    barrier()
    t0 = time.perf_counter()
    for k in range(args.warmup, total):
        ids, mask = pinned[k]
        eng.generate_from_host(ids, mask, out_host=out_host)
    barrier()
    e2e_elapsed = dp.max_over_ranks(time.perf_counter() - t0, dev)

    # per-phase timing of one batch (prefill / decode loop / VQ), events on the launching stream
    phases = {}
    if rank == 0:
        ids, mask = dev_batches[args.warmup]
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        emb = eng.language_model.get_input_embeddings()(ids)
        torch.cuda.synchronize()
        ev[0].record(st)
        toks1 = eng.sample_image(emb, B, 1, mask, 5.0, 1.0, generator=0)          # prefill + 1 token
        ev[1].record(st)
        toks = eng.sample_image(emb, B, dims.n_img_tokens, mask, 5.0, 1.0, generator=0)
        ev[2].record(st)
        eng.gen_vision_model.decode_code(toks, shape=[B, dims.code_dim, dims.grid, dims.grid])
        ev[3].record(st)
        torch.cuda.synchronize()
        prefill_ms = ev[0].elapsed_time(ev[1])
        loop_ms = ev[1].elapsed_time(ev[2]) - prefill_ms
        phases = {"prefill_ms": prefill_ms, "decode_loop_ms": loop_ms, "vq_decode_ms": ev[2].elapsed_time(ev[3]),
                  "ms_per_decode_step": loop_ms / (dims.n_img_tokens - 1)}
        kvb = 2 * dims.L * dims.D * 2
        mean_T = sum(lens) / len(lens) + dims.n_img_tokens / 2
        step_bytes = eng.weight_bytes_per_step + len(lens) * mean_T * kvb + len(lens) * kvb
        peak = peaks.get("hbm_gbs") or 6650.0
        phases["decode_step_algorithmic_GB"] = step_bytes / 1e9
        phases["decode_step_GBps"] = step_bytes / (phases["ms_per_decode_step"] / 1e3) / 1e9
        phases["decode_step_frac_of_hbm_peak"] = phases["decode_step_GBps"] / peak

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    images = B * world * args.steps
    line = {
        "metric": METRIC, "value": images / elapsed, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * elapsed / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "impl": "b200",
        "config": {"workload": f"configs[1] layout2image (task_type=uni), {dims.name}-arch random init, batch {B} per GPU "
                               f"(R={2 * B} rows with the cond/uncond pair), padded prompt P={P}, 576 VQ tokens, CFG 5, T 1, "
                               "prefill + 576-step decode loop + VQ decode_code; prompts sharded per rank",
                   "l2": "working set per decode step (2.5 GB weights + KV) >> 126 MB L2, no explicit flush",
                   "parallelism": f"dp{world}"},
        "clocks": clk,
        "e2e": {"value": images / e2e_elapsed, "unit": UNIT,
                "h2d_bytes_per_step": int(sum(t.numel() * t.element_size() for t in pinned[0])),
                "d2h_bytes_per_step": int(out_host.numel())},
        "gpu_launches": int(launches),
        "phases": phases,
    }
    if not args.no_roofline:
        kvs = (dev_batches[args.warmup][1][:, :P] == 0).sum(1).to(torch.int32).contiguous()
        line["roofline"] = kernel_roofline(eng, kvs, lens, P, peaks)
    if world == 1 and not args.no_extra and args.model == "janus-1.3b" and args.batch == 16:
        del eng
        eng = None
        torch.cuda.empty_cache()
        try:
            line["extra"] = extra_configs(dev, peaks)
        except Exception as ex:                      # the headline line must still be printed
            line["extra"] = {"error": repr(ex)[:400]}
    if world == 1 and not args.no_cpu_baseline:
        del eng
        torch.cuda.empty_cache()
        threads = os.cpu_count() or 1
        cb = cpu_reference_sample(args.model, threads, prompt_len=256, rows_b=1, n_decode=24, vq=True,
                                  sd={k: v.cpu() for k, v in sd.items()})
        line["cpu_baseline"] = {"value": cb["images_per_s"], "unit": UNIT, "cores": threads, "kind": "port",
                                "sample": "BASELINE configs[0]: R=2 rows (B=1 + CFG pair), P=256, fp32 oracle port: prefill + 24 "
                                          "decode steps + VQ decode of 1 image, extrapolated to 576 tokens",
                                "ms_per_decode_step": cb["ms_per_decode_step"], "prefill_s": cb["prefill_s"],
                                "vq_decode_s_per_image": cb["vq_decode_s_per_image"], "torch": torch.__version__}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
