"""Text-to-semantic infilling as a test oracle, composed from oracle/t2s.py (which it leaves unchanged): the reference decode loop of
TextToSemanticWLen.infer (modeling_text_to_semantic.py:184-267) on [text] bytes [sep] [speech] s_1 .. s_N [sep], started from a
full_mask that holds only the speech positions to regenerate. Those start as [mask]; the known ones hold semantic token + offset,
the form every iteration writes back for a sampled id (:256-257), and like the text rows they keep it (:258) and enter re-masking with
confidence +inf (:250). mask_len counts the regenerated positions only: the reference's initial = mask.sum(). With every position
regenerated this is oracle.t2s.infer exactly."""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

from oracle import s2a as os2a
from oracle import t2s as ot2s


def build_infill_sequence(cfg, text_tokens, semantic_tokens, regenerate):
    """[text] bytes [sep] [speech] s_1 .. s_N [sep] with s_k = [mask] where regenerate[k], else semantic_tokens[k] + offset, and
    full_mask = the regenerated speech positions. -> input_ids [1, L], full_mask [1, L]"""
    input_ids, speech = ot2s.build_sequence(cfg, text_tokens, regenerate.numel())
    start = text_tokens.numel() + 3
    regen = regenerate.to(input_ids.device).bool()
    known = semantic_tokens.to(input_ids.device).long() + cfg.num_special + cfg.text_vocab
    input_ids[0, start:start + regen.numel()] = torch.where(regen, input_ids[0, start:start + regen.numel()], known)
    full_mask = torch.zeros_like(speech)
    full_mask[0, start:start + regen.numel()] = regen
    return input_ids, full_mask


def infer_infill(sd, cfg, text, semantic_tokens, regenerate, pred_iters=10, temperature=1.0, cat_gumbel=None, remask_gumbel=None,
                 mode="fp32", forced_ids=None, forced_masks=None, trace=None, device="cpu"):
    """oracle.t2s.infer's loop from the masked start -> the regenerated tokens [T] (semantic vocabulary), in time order. Noise,
    forcing and trace as in oracle.t2s.infer over L = n_text + N + 4 positions; trace["step_sampled"] also receives the running
    sampled tokens after every iteration."""
    text_tokens = text if torch.is_tensor(text) else ot2s.text_tokens_of(text, cfg, device)
    input_ids, full_mask = build_infill_sequence(cfg, text_tokens, semantic_tokens, regenerate)
    offset = cfg.num_special + cfg.text_vocab
    sampled = input_ids.clone()
    if trace is not None:
        trace.update(step_logits=[], step_ids=[], step_masks=[], step_conf=[], step_cut=[], step_sampled=[], input_ids=input_ids,
                     full_mask=full_mask)
    ratios = [math.cos(math.pi / 2.0 * ((t + 1) / pred_iters)) for t in range(pred_iters)]
    mask = full_mask.clone()
    initial = mask.sum(dim=-1)
    emb = sd["input_embedding.weight"]
    for i, ratio in enumerate(ratios):
        logits = ot2s.embeddings_to_logits(sd, cfg, F.embedding(sampled, emb), mode)
        if i == pred_iters - 1:
            ids = logits.argmax(dim=-1)
            if trace is not None:
                trace["step_logits"].append(logits)
                trace["step_ids"].append(ids)
            if forced_ids is not None:
                ids = forced_ids[i]
            sampled = torch.where(full_mask, ids, input_ids)
        else:
            ids = (logits + cat_gumbel[i].view(1, -1, logits.shape[-1]).to(logits.device)).argmax(dim=-1)
            if trace is not None:
                trace["step_logits"].append(logits)
                trace["step_ids"].append(ids)
            if forced_ids is not None:
                ids = forced_ids[i]
            mask_len = torch.floor(initial.float() * ratio).long()
            mask_len = torch.maximum(torch.tensor(1, device=logits.device), torch.minimum(mask_len, initial))
            probs = F.softmax(logits, dim=-1)
            sel = torch.take_along_dim(probs, ids.unsqueeze(-1), -1).squeeze(-1)
            sel = torch.where(mask, sel, torch.inf)
            next_mask = os2a.random_topk_mask(mask_len, sel, remask_gumbel[i].to(sel.device), temperature * ratio, trace)
            if trace is not None:
                trace["step_masks"].append(next_mask)
            if forced_masks is not None:
                next_mask = forced_masks[i]
            sampled = torch.where(next_mask, torch.tensor(ot2s.MASK, device=ids.device), ids + offset)
            sampled = torch.where(full_mask, sampled, input_ids)
            mask = next_mask
        if trace is not None:
            trace["step_sampled"].append(sampled)
    return sampled[full_mask]
