"""Oracle restatement of SASRec (reference: genrec/models/sasrec.py).
TEST INFRASTRUCTURE - see oracle/__init__.py.

``drop(name, t)`` stands for the reference's nn.Dropout (None = eval mode; see oracle.hstu.Drop): ``emb`` (sasrec.py:110),
``{block}attn`` on the attention weights (:236), ``{block}ffn_hid`` and ``{block}ffn_out`` (:264, :265 - the reference's
PointWiseFeedForward calls its one nn.Dropout twice), with ``{block}`` = ``blocks.{i}.``.
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch
import torch.nn.functional as F

from .hstu import Drop, _ln, _no_drop

Params = Dict[str, torch.Tensor]


def sasrec_attention_forward(query, key_value, mask, p: Params, prefix: str, num_heads: int, drop: Optional[Drop] = None,
                             drop_name: str = "attn"):
    """MultiHeadAttention.forward.  Follows genrec/models/sasrec.py:192-246.

    query: LayerNorm'ed input [B,L,D]; key_value: raw input [B,L,D]; mask [B,L,1] float (1 = valid).
    """
    B, L, D = query.shape
    H, dh = num_heads, D // num_heads
    g = lambda k: p[prefix + k]
    Q = query @ g("q_proj.weight").T + g("q_proj.bias")                          # :201
    K = key_value @ g("k_proj.weight").T + g("k_proj.bias")                      # :202
    V = key_value @ g("v_proj.weight").T + g("v_proj.bias")                      # :203
    Q = Q.reshape(B, L, H, dh).transpose(1, 2)
    K = K.reshape(B, L, H, dh).transpose(1, 2)
    V = V.reshape(B, L, H, dh).transpose(1, 2)
    S = (Q @ K.transpose(-2, -1)) * (dh ** -0.5)                                  # :211
    key_mask = mask.squeeze(-1)[:, None, None, :]                                 # :217
    S = S.masked_fill(key_mask == 0, -1e9)                                        # :220-221
    causal = torch.triu(torch.ones(L, L), diagonal=1).bool()
    S = S.masked_fill(causal[None, None], -1e9)                                   # :224-225
    A = F.softmax(S, dim=-1)                                                      # :228
    A = A * mask.squeeze(-1)[:, None, :, None]                                    # :232-233 (query mask AFTER softmax)
    A = (drop or _no_drop)(drop_name, A)                                          # :236
    out = (A @ V).transpose(1, 2).reshape(B, L, D)                                # :239-240
    return out + query                                                            # :244 (residual = normalised query)


def sasrec_block_forward(x, mask, p: Params, prefix: str, num_heads: int, drop: Optional[Drop] = None):
    """SASRecBlock.forward.  Follows genrec/models/sasrec.py:152-165, :258-266."""
    drop = drop or _no_drop
    g = lambda k: p[prefix + k]
    q = _ln(x, g("norm1.weight"), g("norm1.bias"), 1e-8)
    x = sasrec_attention_forward(q, x, mask, p, prefix + "attention.", num_heads, drop, prefix + "attn")   # :160
    h = _ln(x, g("norm2.weight"), g("norm2.bias"), 1e-8)
    hid = drop(prefix + "ffn_hid", F.relu(h @ g("ffn.fc1.weight").T + g("ffn.fc1.bias")))             # :264
    f = drop(prefix + "ffn_out", hid @ g("ffn.fc2.weight").T + g("ffn.fc2.bias"))                     # :265
    return f + x                                                                                       # :266


def sasrec_forward(input_ids, targets, p: Params, num_heads: int, num_blocks: int, drop: Optional[Drop] = None
                   ) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """SASRec.forward.  Follows genrec/models/sasrec.py:79-130."""
    drop = drop or _no_drop
    B, L = input_ids.shape
    E = p["item_embedding.weight"]
    D = E.shape[1]
    mask = (input_ids != 0).unsqueeze(-1).to(E.dtype)                             # :100
    x = F.embedding(input_ids, E, padding_idx=0) * (D ** 0.5)                     # :103 (+ :45 padding_idx)
    x = x + p["position_embedding.weight"][:L].unsqueeze(0)                       # :106-107
    x = drop("emb", x)                                                            # :110
    x = x * mask                                                                  # :111
    for i in range(num_blocks):
        x = sasrec_block_forward(x, mask, p, f"blocks.{i}.", num_heads, drop)     # :115
        x = x * mask                                                              # :116
    x = _ln(x, p["final_norm.weight"], p["final_norm.bias"], 1e-8)               # :118
    logits = x @ E.T                                                              # :121
    loss = None
    if targets is not None:
        loss = F.cross_entropy(logits.reshape(-1, E.shape[0]), targets.reshape(-1), ignore_index=0)
    return logits, loss
