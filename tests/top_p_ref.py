"""Torch reference for top-k / top-p filtering of the image-token sampler (the reference model has neither).

top_k_top_p_filter is HF's TopKLogitsWarper then TopPLogitsWarper (min_tokens_to_keep = 1, filter value -inf), the
order GenerationMixin._get_logits_processor applies them in.  t2i_tokens is oracle.janus_oracle.t2i's decode loop
(fp32, `tokens` branch, no VQ decode) built from the oracle's pieces, with the filter between /temperature and the
softmax."""
from typing import Optional

import torch

from oracle import janus_oracle as O


def top_k_top_p_filter(scores: torch.Tensor, top_k: int = 0, top_p: float = 1.0) -> torch.Tensor:
    """top_k = 0 and top_p = 1 are off, as in transformers."""
    if top_k > 0:
        k = min(top_k, scores.shape[-1])
        scores = scores.masked_fill(scores < torch.topk(scores, k)[0][..., -1, None], float("-inf"))
    if top_p < 1.0:
        sorted_logits, sorted_idx = torch.sort(scores, descending=False)
        cum = sorted_logits.softmax(dim=-1).cumsum(dim=-1)
        remove = cum <= (1 - top_p)
        remove[..., -1:] = False
        scores = scores.masked_fill(remove.scatter(1, sorted_idx, remove), float("-inf"))
    return scores


@torch.inference_mode()
def t2i_tokens(sd, d, tokens: torch.Tensor, mask: torch.Tensor, n_tok: int, top_k: int = 0, top_p: float = 1.0,
               cfg_weight: float = 5.0, temperature: float = 1.0, seed: int = 0, sampler: Optional[O.Sampler] = None,
               edit_region: Optional[torch.Tensor] = None, gt_labels: Optional[torch.Tensor] = None,
               trace: Optional[list] = None) -> torch.Tensor:
    """Image tokens (B, n_tok) of O.t2i(sd, d, tokens, mask, ...) with the filter applied; `trace` collects the
    filtered scaled logits of each step."""
    dev = tokens.device
    if sampler is None:
        sampler = O.make_torch_sampler(torch.Generator(device=dev).manual_seed(seed))
    x = O.embed_tokens(sd, tokens)
    num_gen = x.shape[0] // 2
    out = torch.zeros(num_gen, n_tok, dtype=torch.int, device=dev)
    outputs = None
    for i in range(n_tok):
        outputs = O.llama_model_forward(sd, d, inputs_embeds=x, attention_mask=mask, use_cache=True,
                                        past_key_values=outputs.past_key_values if i != 0 else None)
        logits = O.gen_head(sd, outputs.last_hidden_state[:, -1, :])
        c, u = logits[0::2, :], logits[1::2, :]
        t = top_k_top_p_filter((u + cfg_weight * (c - u)) / temperature, top_k, top_p)
        if trace is not None:
            trace.append(t)
        tok = sampler(torch.softmax(t, dim=-1), i)
        if edit_region is not None:
            for bid in range(len(edit_region)):
                if edit_region[bid, i].item() == 0:
                    tok[bid, 0] = gt_labels[bid, i]
        out[:, i] = tok.squeeze(dim=-1)
        tok = torch.cat([tok.unsqueeze(dim=1), tok.unsqueeze(dim=1)], dim=1).view(-1)
        x = O.prepare_gen_img_embeds(sd, tok).unsqueeze(dim=1)
    return out
