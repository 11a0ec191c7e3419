"""Torch reference for image-token log-probabilities.

log p(tok) is log_softmax of the filtered scaled CFG logits (tests/per_image_ref.py: CFG rounded per op in the engine
dtype, /temperature, top-k then top-p per row) gathered at the emitted token - HF compute_transition_scores(...,
normalize_logits=True) on the processed scores.  A removed token is exactly -inf; a kept one far below the maximum keeps
its finite value.  score_ref is the teacher-forced scorer's reference: ONE uncached forward over prompt + image tokens,
gen_head at the positions that predict each image token; loop_ref is the cached decode loop with every step recorded."""
from typing import Optional, Sequence

import torch

from oracle import janus_oracle as O
from tests import per_image_ref as PR


def logprobs_of(filtered: torch.Tensor, tok: torch.Tensor) -> torch.Tensor:
    """(B, V) filtered scaled logits, (B,) tokens -> (B,) fp32 log-probs."""
    return torch.log_softmax(filtered.float(), dim=-1).gather(1, tok.long().view(-1, 1)).squeeze(1)


def step_logprobs(logits: torch.Tensor, mode: str, tok: torch.Tensor, cfg_weight: Sequence[float],
                  temperature: Sequence[float], top_k: Sequence[int], top_p: Sequence[float]) -> torch.Tensor:
    t = PR.filter_rows(PR.scaled_cfg(logits, mode, cfg_weight, temperature), top_k, top_p)
    return logprobs_of(t, tok)


@torch.inference_mode()
def loop_ref(sd, d, tokens: torch.Tensor, mask: torch.Tensor, n_tok: int, cfg_weight, temperature, top_k, top_p,
             generator=None, forced: Optional[torch.Tensor] = None):
    """fp32 cached decode loop: tokens (B, n_tok) and their log-probs.  forced (B, n_tok): every token is forced
    (teacher forcing with edit_region all 0); otherwise the tokens are drawn with `generator` as PR.draw does."""
    x = O.embed_tokens(sd, tokens)
    B = x.shape[0] // 2
    toks = torch.zeros(B, n_tok, dtype=torch.int, device=tokens.device)
    lps = torch.zeros(B, n_tok, dtype=torch.float32, device=tokens.device)
    outputs = None
    for i in range(n_tok):
        outputs = O.llama_model_forward(sd, d, inputs_embeds=x, attention_mask=mask, use_cache=True,
                                        past_key_values=outputs.past_key_values if i != 0 else None)
        logits = O.gen_head(sd, outputs.last_hidden_state[:, -1, :])
        t = PR.filter_rows(PR.scaled_cfg(logits, "fp32", cfg_weight, temperature), top_k, top_p)
        tok = forced[:, i].to(tokens.device) if forced is not None else PR.draw(t, generator)
        toks[:, i] = tok.int()
        lps[:, i] = logprobs_of(t, tok)
        pair = torch.stack([tok, tok], dim=1).view(-1)
        x = O.prepare_gen_img_embeds(sd, pair).unsqueeze(1)
    return toks, lps


@torch.inference_mode()
def score_ref(sd, d, tokens: torch.Tensor, mask: torch.Tensor, image_tokens: torch.Tensor, cfg_weight, temperature,
              top_k, top_p, mode: str = "fp32") -> torch.Tensor:
    """One uncached forward over prompt + image tokens (the reference's full-sequence forward; `mode` "fp32" or
    "autocast"), gen_head at columns P-1 .. P+n-2, CFG, filters, log_softmax at the given tokens -> (B, n)."""
    dev = tokens.device
    B, n = image_tokens.shape
    P = tokens.shape[1]
    with O._autocast_ctx(mode, dev):
        x = O.embed_tokens(sd, tokens)
        pair = torch.repeat_interleave(image_tokens.long().to(dev), 2, dim=0)           # rows 2b, 2b+1 <- image b
        img = O.prepare_gen_img_embeds(sd, pair[:, : n - 1].reshape(-1)).reshape(2 * B, n - 1, -1)
        seq = torch.cat([x.float(), img.float()], dim=1)                                  # fp32 residual stream
        out = O.llama_model_forward(sd, d, inputs_embeds=seq, attention_mask=mask[:, : P + n - 1], use_cache=False)
        logits = O.gen_head(sd, out.last_hidden_state[:, P - 1: P + n - 1, :])        # (2B, n, V)
    lg = logits.float().permute(1, 0, 2).reshape(n * 2 * B, -1)                          # step-major pairs
    k = list(top_k) * n
    p = list(top_p) * n
    w = list(cfg_weight) * n
    tt = list(temperature) * n
    bf = "bf16" if mode == "autocast" else "fp32"
    t = PR.filter_rows(PR.scaled_cfg(lg, bf, w, tt), k, p)
    lp = logprobs_of(t, image_tokens.to(dev).t().reshape(-1))
    return lp.view(n, B).t().contiguous()
