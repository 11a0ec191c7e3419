"""Torch reference for guidance schedules: a guidance weight per image and per step.

At step i image b is treated exactly as tests/per_image_ref.py treats it with cfg_weight[b] = schedule[b][i] (CFG rounded
per op, /temperature, top-k then top-p per row, torch.multinomial on the row's generator), and its log-prob is
tests/logprob_ref.py's under that distribution.  The scorer's reference is logprob_ref.score_ref with one weight column
per position: entry (b, i) of a scorer run with cfg_weight = schedule[:, i] depends on that column only."""
from typing import Optional, Sequence

import torch

from oracle import janus_oracle as O
from tests import logprob_ref as LR
from tests import per_image_ref as PR


def column(schedule, i: int):
    """The per-image weights of step i."""
    return [float(row[i]) for row in schedule]


@torch.inference_mode()
def loop_ref(sd, d, tokens: torch.Tensor, mask: torch.Tensor, n_tok: int, schedule, temperature: Sequence[float],
             top_k: Sequence[int], top_p: Sequence[float], generator=None, edit_region: Optional[torch.Tensor] = None,
             gt_labels: Optional[torch.Tensor] = None, greedy: bool = False):
    """The oracle's fp32 cached decode loop (per_image_ref.t2i_tokens, logprob_ref.loop_ref) with step i's weights taken
    from column i of `schedule` (num_gen, n_tok): tokens (num_gen, n_tok) and their log-probs.  greedy: the arg-max of the
    top-k-filtered distribution (top-p does not apply), as the engine's greedy mode.  Teacher forcing as the reference's
    override loop (plangen_base.py:593-598)."""
    x = O.embed_tokens(sd, tokens)
    B = x.shape[0] // 2
    toks = torch.zeros(B, n_tok, dtype=torch.int, device=tokens.device)
    lps = torch.zeros(B, n_tok, dtype=torch.float32, device=tokens.device)
    kp = [1.0] * B if greedy else top_p
    outputs = None
    for i in range(n_tok):
        outputs = O.llama_model_forward(sd, d, inputs_embeds=x, attention_mask=mask, use_cache=True,
                                        past_key_values=outputs.past_key_values if i != 0 else None)
        logits = O.gen_head(sd, outputs.last_hidden_state[:, -1, :])
        t = PR.filter_rows(PR.scaled_cfg(logits, "fp32", column(schedule, i), temperature), top_k, kp)
        tok = torch.softmax(t, dim=-1).argmax(-1) if greedy else PR.draw(t, generator)
        if edit_region is not None:
            for bid in range(len(edit_region)):
                if edit_region[bid, i].item() == 0:
                    tok[bid] = gt_labels[bid, i]
        toks[:, i] = tok.int()
        lps[:, i] = LR.logprobs_of(t, tok)
        pair = torch.stack([tok, tok], dim=1).view(-1)
        x = O.prepare_gen_img_embeds(sd, pair).unsqueeze(1)
    return toks, lps


@torch.inference_mode()
def score_ref(sd, d, tokens: torch.Tensor, mask: torch.Tensor, image_tokens: torch.Tensor, schedule, temperature,
              top_k, top_p, mode: str = "fp32") -> torch.Tensor:
    """logprob_ref.score_ref (one uncached full-sequence forward) with position i scored under column i of `schedule`
    (B, n) -> (B, n) log-probs."""
    n = image_tokens.shape[1]
    out = torch.empty(image_tokens.shape, dtype=torch.float32, device=tokens.device)
    for i in range(n):
        out[:, i] = LR.score_ref(sd, d, tokens, mask, image_tokens, column(schedule, i), temperature, top_k, top_p,
                                 mode=mode)[:, i]
    return out
