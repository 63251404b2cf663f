"""Oracle of S2A infilling (test infrastructure): infer_special with the known frames anywhere in the utterance.

Composed from oracle/s2a.py's functions, which it leaves as they are. The target rows are picked by a boolean mask `target` [B, N]
with the same count T in every row, as the reference's masked_select(...).view(b, ...) does (injection_conformer_wrapper.py:85-88,
:135-141); every other row is a known row and is treated exactly as a prompt row (modeling_injection_conformer.py:157-168): input
sem + LN(Linear(level-0 feature)), never sampled or re-masked, injected with the cumulative ground-truth features of its levels
(:124-125). With the known rows as a prefix each function below computes what its oracle/s2a.py counterpart computes for that prompt.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

from oracle import s2a as os2a


def _sel(t, target):
    """The target rows of t [B, N, ...] in time order -> [B, T, ...]."""
    return t[target].view(t.shape[0], -1, *t.shape[2:])


def _put(t, target, v):
    """Writes v [B, T, ...] to the rows _sel(t, target) reads."""
    t[target] = v.reshape(-1, *v.shape[2:])


def build_infill_input(sd, cfg, semantic_tokens, acoustic_tokens, target, mode="fp32"):
    """semantic_tokens [B, N], acoustic_tokens [B, q, N] (ignored where target), target bool [B, N] -> encoder input x [B, N, d], the
    semantic embedding of the target rows [B, T, d] and the prompt injections ([B, N, latent] per level, zeros on target rows; None when
    no row is known). Known rows are built as os2a.build_encoder_input builds prompt rows, at their own positions."""
    sem = F.embedding(semantic_tokens, sd["semantic_embedding.weight"])
    u = os2a.codes_to_features_unreduced(sd, cfg, torch.where(target[:, None], 0, acoustic_tokens), mode)   # [B, q, latent, N]
    ac = os2a._ln(os2a._linear(u[:, 0].transpose(1, 2), sd["acoustic_feat_proj.0.weight"], sd["acoustic_feat_proj.0.bias"], mode),
                  sd["acoustic_feat_proj.1.weight"], sd["acoustic_feat_proj.1.bias"])
    t3 = target[:, :, None]
    x = torch.where(t3, sem + sd["mask_token"].expand(sem.shape[0], sem.shape[1], -1), sem + ac)
    prompt_inj = None
    if not bool(target.all()):
        prompt_inj = []
        for i in range(min(len(cfg.injection_layers), acoustic_tokens.shape[1])):
            s = u[:, 0]
            for j in range(1, i + 1):
                s = os2a._r(s + u[:, j], mode)
            prompt_inj.append(torch.where(t3, 0.0, s.transpose(1, 2)))
    return x, _sel(sem, target), prompt_inj


def forward_first_level(sd, cfg, x, target, mode="fp32"):
    """os2a.forward_first_level on the rows of `target` -> [B, T, codes]."""
    freqs = os2a.rotary_freqs(x.shape[-2], cfg.dim_head, x.device)
    for i in range(cfg.depth):
        out = os2a.conformer_block(sd, i, x, cfg, freqs, mode)
        if i in cfg.injection_layers:
            return _sel(os2a.single_to_logits(sd, out, cfg.injection_layers.index(i), mode), target)
        x = out
    raise ValueError("no injection layer")


def forward_full(sd, cfg, x, target, prompt_injections=None, mode="fp32", forced_coarse=None, trace=None):
    """os2a.forward_full with the target rows of `target` (forced_coarse [B, n_inj, T]) -> logits [B, Q, T, codes]; the other rows
    receive prompt_injections."""
    freqs = os2a.rotary_freqs(x.shape[-2], cfg.dim_head, x.device)
    coarse_outs, coarse_logits = [], []
    for i in range(cfg.depth):
        out = os2a.conformer_block(sd, i, x, cfg, freqs, mode)
        if i in cfg.injection_layers:
            k = cfg.injection_layers.index(i)
            residual = coarse_outs[-1] if (coarse_outs and cfg.residual) else 0
            coarse_outs.append(out)
            if cfg.use_injection:
                coarse_logits.append(os2a.single_to_logits(sd, out, k, mode))
                tokens = torch.stack([l.argmax(dim=-1) for l in coarse_logits], dim=1)      # [B, k+1, N]
                if forced_coarse is not None:
                    tokens = tokens.clone()
                    _put(tokens.transpose(1, 2), target, forced_coarse[:, : k + 1].transpose(1, 2))
                inj = os2a.codes_to_features(sd, cfg, tokens, mode).transpose(1, 2)        # [B, N, latent]
                if prompt_injections is not None:
                    inj = torch.where(target[:, :, None], inj, prompt_injections[k])
                out = out + os2a.project_injection(sd, k, inj, mode) + residual
            else:
                out = out + residual
        x = out
    x_t = _sel(x, target)
    coarse_t = [_sel(c, target) for c in coarse_outs]
    n_fine = cfg.n_codebooks - len(cfg.injection_layers)
    fine = os2a._linear(x_t, sd["encoder.fine_head.0.weight"], sd["encoder.fine_head.0.bias"], mode)
    fine = fine.view(*x_t.shape[:2], n_fine, cfg.hidden)
    allo = torch.cat([c[:, :, None, :] for c in coarse_t] + [fine], dim=-2)
    h = os2a._ln(allo, sd["encoder.to_logits.0.weight"], sd["encoder.to_logits.0.bias"])
    w, bias = sd["encoder.to_logits.1.weight"], sd["encoder.to_logits.1.bias"][0, 0]
    r = lambda t: os2a._r(t, mode)
    if mode == "bf16":
        logits = r(r(torch.einsum("bnqd,qdl->bnql", r(h), r(w))) + bias)
    else:
        logits = torch.einsum("bnqd,qdl->bnql", h, w) + bias
    if trace is not None:
        trace["coarse_logits"] = [_sel(l, target) for l in coarse_logits]
    return logits.permute(0, 2, 1, 3)


def infer_infill(sd, cfg, semantic_tokens, acoustic_tokens, regenerate, steps=1, temperature=1.0, cat_gumbel=None, remask_gumbel=None,
                 mode="fp32", forced_ids=None, forced_masks=None, forced_coarse=None, trace=None):
    """os2a.infer_special's decode loop (modeling_injection_conformer.py:170-230) on the regenerated frames: semantic_tokens [B, N],
    acoustic_tokens [B, q, N], regenerate bool [B, N] (same count T per row). Noise, forcing and trace are per regenerated frame, as in
    infer_special. Returns the codes of the regenerated frames in time order [B, Q, T]."""
    target = regenerate.bool()
    x, sem, prompt_inj = build_infill_input(sd, cfg, semantic_tokens, acoustic_tokens, target, mode)
    B, T = sem.shape[:2]
    mask_token = sd["mask_token"].expand(B, T, -1)
    if trace is not None:
        trace.update(step_logits=[], step_ids=[], step_masks=[], step_conf=[], step_cut=[], x0=x.clone())
    if steps > 1:
        ratios = [math.cos(math.pi / 2.0 * ((t + 1) / steps)) for t in range(steps)]
        mask = torch.ones(B, T, dtype=torch.bool, device=x.device)
        initial = mask.sum(dim=-1)
        for i, ratio in enumerate(ratios):
            logits = forward_first_level(sd, cfg, x.clone(), target, mode)
            if i == steps - 1:
                ids = logits.argmax(dim=-1)
            else:
                ids = (logits + cat_gumbel[i].view(B, T, -1).to(logits.device)).argmax(dim=-1)
            if trace is not None:
                trace["step_logits"].append(logits)
                trace["step_ids"].append(ids)
            if forced_ids is not None:
                ids = forced_ids[i]
            feats = os2a.feat_proj(sd, cfg, ids, mode)
            _put(x, target, torch.where(mask[..., None], sem + feats, _sel(x, target)))
            if i < steps - 1:
                mask_len = torch.floor(initial * ratio)
                mask_len = torch.maximum(torch.ones_like(mask_len), torch.minimum(torch.sum(mask, dim=-1) - 1, mask_len))
                probs = F.softmax(logits, dim=-1)
                sel = torch.take_along_dim(probs, ids.unsqueeze(-1), -1).squeeze(-1)
                sel = torch.where(mask, sel, torch.inf)
                next_mask = os2a.random_topk_mask(mask_len, sel, remask_gumbel[i].to(sel.device), temperature * ratio, trace)
                if trace is not None:
                    trace["step_masks"].append(next_mask)
                if forced_masks is not None:
                    next_mask = forced_masks[i]
                _put(x, target, torch.where(next_mask[..., None], sem + mask_token, _sel(x, target)))
                mask = next_mask
    if trace is not None:
        trace["x_final"] = x.clone()
    all_logits = forward_full(sd, cfg, x, target, prompt_inj, mode, forced_coarse, trace)
    if trace is not None:
        trace["all_logits"] = all_logits
    return all_logits.argmax(dim=-1)
