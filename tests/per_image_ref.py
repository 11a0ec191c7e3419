"""Torch reference for per-image sampling settings (cfg_weight, temperature, top_k, top_p, generator per image).

The per-row twin of tests/top_p_ref.py: every row of a batch is treated with its own scalars exactly as the scalar path
treats a whole batch, then drawn with torch.multinomial on the row alone with its own generator (per-image RNG), or on
the whole batch with one generator (batch-wide RNG)."""
from typing import Optional, Sequence, Union

import numpy as np
import torch

from oracle import janus_oracle as O
from tests import top_p_ref as TP

Gen = Union[torch.Generator, Sequence[torch.Generator]]


def scaled_cfg(logits: torch.Tensor, mode: str, cfg_weight: Sequence[float], temperature: Sequence[float]) -> torch.Tensor:
    """The kernel's t per row: the CFG combine rounded per op in the engine's dtype (the product in fp32, as torch computes
    a low-precision tensor times a scalar), then a correctly rounded division by the row's temperature (a tensor divisor:
    torch divides by a Python scalar through its reciprocal), rounded to the engine's dtype."""
    dt = torch.bfloat16 if mode == "bf16" else torch.float32
    lg = logits.to(dt)
    c, u = lg[0::2], lg[1::2]
    w = torch.tensor(cfg_weight, dtype=torch.float32, device=logits.device)[:, None]
    temp = torch.tensor(temperature, dtype=torch.float32, device=logits.device)[:, None]
    t = u + ((c - u).float() * w).to(dt)
    return (t.float() / temp).to(dt).float()


def filter_rows(t: torch.Tensor, top_k: Sequence[int], top_p: Sequence[float]) -> torch.Tensor:
    """top_p_ref.top_k_top_p_filter applied to each row with that row's top_k and top_p."""
    return torch.cat([TP.top_k_top_p_filter(t[b:b + 1], int(top_k[b]), float(top_p[b])) for b in range(t.shape[0])])


def draw(filtered: torch.Tensor, generator: Gen) -> torch.Tensor:
    """softmax, then torch.multinomial: per row with generator[b], or over the whole batch with one generator."""
    probs = torch.softmax(filtered, dim=-1)
    if isinstance(generator, torch.Generator):
        return torch.multinomial(probs, 1, generator=generator).squeeze(-1)
    return torch.cat([torch.multinomial(probs[b:b + 1], 1, generator=g) for b, g in enumerate(generator)]).squeeze(-1)


def ambiguous_rows(t: torch.Tensor, top_k: Sequence[int], top_p: Sequence[float], tol: float = 1e-6) -> torch.Tensor:
    """Rows whose fp64 cumulative mass, in the ascending order, comes within tol of fp32(1 - top_p) before the last: there
    torch's fp32 cumsum order legitimately decides the nucleus (rows with top_p = 1 never are)."""
    out = torch.zeros(t.shape[0], dtype=torch.bool, device=t.device)
    for b in range(t.shape[0]):
        if float(top_p[b]) >= 1.0:
            continue
        r = TP.top_k_top_p_filter(t[b:b + 1], int(top_k[b]), 1.0).double()
        s = torch.sort(r, dim=-1).values.softmax(-1).cumsum(-1)[:, :-1]
        out[b] = bool(((s - float(np.float32(1.0 - float(top_p[b])))).abs() < tol).any())
    return out


@torch.inference_mode()
def t2i_tokens(sd, d, tokens: torch.Tensor, mask: torch.Tensor, n_tok: int, cfg_weight: Sequence[float],
               temperature: Sequence[float], top_k: Sequence[int], top_p: Sequence[float], generator: Gen,
               edit_region: Optional[torch.Tensor] = None, gt_labels: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Image tokens (B, n_tok) of the oracle's fp32 decode loop (as top_p_ref.t2i_tokens) with per-row settings."""
    x = O.embed_tokens(sd, tokens)
    num_gen = x.shape[0] // 2
    out = torch.zeros(num_gen, n_tok, dtype=torch.int, device=tokens.device)
    outputs = None
    for i in range(n_tok):
        outputs = O.llama_model_forward(sd, d, inputs_embeds=x, attention_mask=mask, use_cache=True,
                                        past_key_values=outputs.past_key_values if i != 0 else None)
        logits = O.gen_head(sd, outputs.last_hidden_state[:, -1, :])
        t = filter_rows(scaled_cfg(logits, "fp32", cfg_weight, temperature), top_k, top_p)
        tok = draw(t, generator)[:, None]
        if edit_region is not None:
            for bid in range(len(edit_region)):
                if edit_region[bid, i].item() == 0:
                    tok[bid, 0] = gt_labels[bid, i]
        out[:, i] = tok.squeeze(dim=-1)
        tok = torch.cat([tok.unsqueeze(dim=1), tok.unsqueeze(dim=1)], dim=1).view(-1)
        x = O.prepare_gen_img_embeds(sd, tok).unsqueeze(dim=1)
    return out
