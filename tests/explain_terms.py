"""Float64 restatement of the per-history-item terms of a pair score (the explanations of include/nais_b200.h
nais_pairs_explain), built from the same formulas as oracle.nais_oracle.attention_network (model.py:246-297 and siblings).

For branch b, row r and history position h:  E_bh = exp(a_bh) * [hist_h != tgt],  S_b = sum_h E_bh,  s_bh = sum_d x_bhd,
w_bh * s_bh = E_bh * s_bh / S_b^beta.  The contribution of h is c_h = sum_b w_bh s_bh; sum_h c_h is the score."""
from __future__ import annotations

from typing import Dict, Optional

import torch

from oracle import nais_oracle as orc


def attention_terms(sd: Dict[str, torch.Tensor], variant: str, beta: float, hist: torch.Tensor, tgt: torch.Tensor,
                    hreg: Optional[torch.Tensor] = None, treg: Optional[torch.Tensor] = None, aux: Optional[torch.Tensor] = None,
                    dtype: torch.dtype = torch.float64) -> Dict[str, torch.Tensor]:
    """Dense layout ([B,H] rows).  Returns E, ws (= w * s), s: [n_branch, B, H]; S: [n_branch, B]; mask: [B, H] (True = the
    cell takes part); contrib: [B, H] = ws summed over the branches; attn: [n_branch, B, H] = E / S."""
    v = orc.VARIANTS[variant]
    P = {k: t.to(dtype) for k, t in sd.items()}
    q = P["embed_history.weight"][hist]
    p = P["embed_target.weight"][tgt]
    mask = hist != tgt[:, None]
    if variant == "disentangled":
        bias = aux.to(dtype) * P["embed_distance.weight"][0].sum()
        x = q * p[:, None, :]
        xr = P["embed_region.weight"][hreg] * P["embed_region.weight"][treg][:, None, :]
        a = torch.relu(x @ P["attn_layer1.weight"].T + P["attn_layer1.bias"]) @ P["attn_layer2.weight"][0] + bias
        ar = torch.relu(xr @ P["region_attn_layer1.weight"].T + P["region_attn_layer1.bias"]) @ P["region_attn_layer2.weight"][0] + bias
        logits, sims = [a, ar], [x.sum(-1), xr.sum(-1)]
    else:
        if v["has_region"]:
            q = torch.cat((q, P["embed_region.weight"][hreg]), -1)
            p = torch.cat((p, P["embed_region.weight"][treg]), -1)
        x = q * p[:, None, :]
        sim = x.sum(-1)
        if v["dist"] == "latlon":
            g = torch.sigmoid((aux.to(dtype) * v["scale"]) @ P["dist_layer.weight"].T + P["dist_layer.bias"])
            x = torch.cat((x, g), -1)
        logits, sims = [torch.relu(x @ P["attn_layer1.weight"].T + P["attn_layer1.bias"]) @ P["attn_layer2.weight"][0]], [sim]
    E = torch.stack([torch.exp(a) * mask.to(dtype) for a in logits])
    s = torch.stack(sims)
    S = E.sum(-1)
    ws = E / torch.pow(S, beta)[..., None] * s
    return dict(E=E, ws=ws, s=s, S=S, mask=mask, contrib=ws.sum(0), attn=E / S[..., None])
