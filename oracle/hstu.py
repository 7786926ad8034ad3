"""Oracle restatement of the HSTU model (reference: genrec/models/hstu.py).

Functional style: every function takes a ``state_dict``-shaped mapping of
tensors (same key names as the reference module, SURVEY.md Appendix C) so the
same checkpoint drives the reference, the oracle and the CUDA path.
Runs on CPU in whatever dtype the parameters / activations carry (fp32, fp64).
TEST INFRASTRUCTURE - see oracle/__init__.py.
"""
from __future__ import annotations

import math
from typing import Callable, Dict, Optional, Tuple

import torch
import torch.nn.functional as F

Params = Dict[str, torch.Tensor]
# drop(name, t) -> t': a dropout site of the reference, by name.  Tests pass one that multiplies by a known mask (kept elements
# scaled, dropped ones 0) so the oracle reproduces a training-mode forward; None is eval mode.
Drop = Callable[[str, torch.Tensor], torch.Tensor]


def _no_drop(name: str, t: torch.Tensor) -> torch.Tensor:
    return t


# --------------------------------------------------------------------------- buckets
def temporal_bucket(time_diff: torch.Tensor, num_buckets: int = 64) -> torch.Tensor:
    """|dt| -> log bucket.  Follows genrec/models/hstu.py:368-384.

    fp32 log, true division by the literal 0.693 (not ln 2), truncation, clamp.
    """
    mag = torch.clamp(torch.abs(time_diff), min=1).float()      # hstu.py:376
    b = (torch.log(mag) / 0.693).long()                          # hstu.py:381
    return torch.clamp(b, min=0, max=num_buckets - 1)            # hstu.py:382


def position_bucket(rel: torch.Tensor, num_buckets: int = 32, max_distance: int = 128) -> torch.Tensor:
    """T5-style log bucket of clamp(rel, 0).  Follows genrec/models/hstu.py:300-328."""
    rel = torch.clamp(rel, min=0)                                # hstu.py:312
    max_exact = num_buckets // 2                                 # hstu.py:315
    small = rel < max_exact                                      # hstu.py:316
    large = max_exact + (
        torch.log(rel.float() / max_exact) / math.log(max_distance / max_exact) * (num_buckets - max_exact)
    ).long()                                                     # hstu.py:319-323
    large = torch.clamp(large, max=num_buckets - 1)              # hstu.py:325
    return torch.where(small, rel, large)                        # hstu.py:327


def position_bias(table: torch.Tensor, L: int, num_buckets: int = 32, max_distance: int = 128) -> torch.Tensor:  # noqa: E302
    """[H, L, L] bias.  Follows genrec/models/hstu.py:330-349.

    NOTE the reference builds ``pos[None,:] - pos[:,None]`` = (j - i) for cell
    (i, j) (hstu.py:340) - the opposite sign of its comment - then clamps at 0,
    so every causal cell (j <= i) lands in bucket 0 (SURVEY.md section 0).
    """
    pos = torch.arange(L, device=table.device)
    rel = pos.unsqueeze(0) - pos.unsqueeze(1)                    # [i, j] = j - i
    bkt = position_bucket(rel, num_buckets, max_distance)
    return F.embedding(bkt, table).permute(2, 0, 1)              # [H, L, L]   (nn.Embedding lookup, hstu.py:346-347)


def temporal_bias(table: torch.Tensor, timestamps: torch.Tensor) -> torch.Tensor:
    """[B, H, L, L] bias.  Follows genrec/models/hstu.py:386-409."""
    diff = timestamps.unsqueeze(2) - timestamps.unsqueeze(1)     # [b,i,j] = ts_i - ts_j  (:400)
    bkt = temporal_bucket(diff, table.shape[0])
    return F.embedding(bkt, table).permute(0, 3, 1, 2)           # nn.Embedding lookup (:406-407)


# --------------------------------------------------------------------------- layer
def _ln(x: torch.Tensor, w: torch.Tensor, b: torch.Tensor, eps: float) -> torch.Tensor:
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    return (x - mu) / torch.sqrt(var + eps) * w + b


def hstu_layer_forward(
    x: torch.Tensor,                       # [B, L, D]
    padding_mask: torch.Tensor,            # [B, L] bool, True = padded key
    timestamps: Optional[torch.Tensor],    # [B, L] int64 or None
    p: Params,
    prefix: str,
    num_heads: int,
    use_temporal_bias: bool = True,
    num_position_buckets: int = 32,
    max_position_distance: int = 128,
    return_intermediates: bool = False,
    drop: Optional[Drop] = None,
):
    """One HSTU block.  Follows genrec/models/hstu.py:222-280 (SURVEY Appendix A).

    ``drop(name, t)`` stands for the reference's nn.Dropout at the three places it sits in a block (None = eval mode):
    ``{prefix}gate`` (:275), ``{prefix}ffn_hid`` (:212) and ``{prefix}ffn_out`` (:214)."""
    drop = drop or _no_drop
    B, L, D = x.shape
    H, dh = num_heads, D // num_heads
    g = lambda k: p[prefix + k]

    proj = F.silu(x @ g("projection.weight").T + g("projection.bias"))          # :234
    U, V, Q, K = proj.chunk(4, dim=-1)                                            # :235
    Q = Q.reshape(B, L, H, dh).transpose(1, 2)                                    # :238
    K = K.reshape(B, L, H, dh).transpose(1, 2)
    V = V.reshape(B, L, H, dh).transpose(1, 2)

    S = Q @ K.transpose(-2, -1)                                                   # :244 (no scaling)
    S = S + position_bias(g("position_bias.relative_attention_bias.weight"), L,
                          num_position_buckets, max_position_distance).unsqueeze(0)   # :247-248
    if use_temporal_bias and timestamps is not None:                              # :251
        S = S + temporal_bias(g("temporal_bias.temporal_attention_bias.weight"), timestamps)

    causal = torch.triu(torch.ones(L, L, device=x.device), diagonal=1).bool()    # hstu.py:121
    S = S.masked_fill(causal[None, None], -1e9)                                   # :256
    S = S.masked_fill(padding_mask[:, None, None, :], -1e9)                       # :259
    A = F.silu(S)                                                                 # :263
    O = (A @ V).transpose(1, 2).reshape(B, L, D)                                  # :266-267

    N = _ln(O, g("attn_norm.weight"), g("attn_norm.bias"), 1e-5)                 # :271
    x1 = x + drop(prefix + "gate", N * U)                                         # :272-275
    xn = _ln(x1, g("ffn_norm.weight"), g("ffn_norm.bias"), 1e-5)                 # :278
    hid = drop(prefix + "ffn_hid", F.silu(xn @ g("ffn.0.weight").T + g("ffn.0.bias")))   # :210-212
    y = x1 + drop(prefix + "ffn_out", hid @ g("ffn.3.weight").T + g("ffn.3.bias"))     # :213-214, :278
    if return_intermediates:
        return y, dict(P=proj, S=S, A=A, O=O, N=N, x1=x1, xn=xn, hid=hid)
    return y


def hstu_forward(
    input_ids: torch.Tensor,               # [B, L] int64, 0 = pad
    timestamps: Optional[torch.Tensor],
    targets: Optional[torch.Tensor],
    p: Params,
    num_heads: int,
    num_blocks: int,
    use_temporal_bias: bool = True,
    num_position_buckets: int = 32,
    max_position_distance: int = 128,
    drop: Optional[Drop] = None,
) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """Whole model.  Follows genrec/models/hstu.py:99-148.  ``drop``: see ``hstu_layer_forward``; the embedding's is ``emb`` (:128)."""
    drop = drop or _no_drop
    padding_mask = input_ids == 0                                                 # :124
    E = p["item_embedding.weight"]
    x = F.embedding(input_ids, E, padding_idx=0)      # :127 (+ :62 padding_idx: no gather-grad into row 0)
    x = drop("emb", x)                                                            # :128
    for i in range(num_blocks):                                                   # :131-132
        x = hstu_layer_forward(x, padding_mask, timestamps, p, f"layers.{i}.", num_heads,
                               use_temporal_bias, num_position_buckets, max_position_distance, drop=drop)
    x = _ln(x, p["final_norm.weight"], p["final_norm.bias"], 1e-5)               # :134
    logits = x @ E.T                                                              # :137
    loss = None
    if targets is not None:                                                       # :141-146
        loss = F.cross_entropy(logits.reshape(-1, E.shape[0]), targets.reshape(-1), ignore_index=0)
    return logits, loss


def hstu_predict(input_ids, timestamps, p, num_heads, num_blocks, top_k=10, **kw) -> torch.Tensor:
    """Follows genrec/models/hstu.py:150-157."""
    logits, _ = hstu_forward(input_ids, timestamps, None, p, num_heads, num_blocks, **kw)
    last = logits[:, -1, :].clone()
    last[:, 0] = float("-inf")
    return torch.topk(last, top_k, dim=-1).indices


def recall_ndcg(top_items: torch.Tensor, targets: torch.Tensor, ks=(1, 5, 10)) -> Dict[str, float]:
    """Sums (not means) of Recall@k / NDCG@k.  Follows genrec/trainers/hstu_trainer.py:62-70."""
    out = {}
    for k in ks:
        hit = top_items[:, :k] == targets[:, None]
        rank = hit.float().argmax(-1) + 1
        anyhit = hit.any(-1)
        out[f"Recall@{k}"] = float(anyhit.sum())
        out[f"NDCG@{k}"] = float((anyhit.float() / torch.log2(rank.float() + 1.0)).sum())
    return out


def time_bucket_thresholds(num_buckets: int = 64) -> torch.Tensor:
    """thr[k] = smallest |dt| >= 1 whose reference bucket is >= k (k = 0..num_buckets-1).

    Found by bisection on ``temporal_bucket`` itself (monotone in |dt|), so integer
    compares against ``thr`` reproduce the fp32 log/0.693 expression bit-exactly.
    """
    thr = torch.empty(num_buckets, dtype=torch.int64)
    thr[0] = 0
    hi_cap = (1 << 62)
    for k in range(1, num_buckets):
        lo, hi = 1, hi_cap
        if int(temporal_bucket(torch.tensor([hi]), 1 << 20)) < k:
            thr[k] = torch.iinfo(torch.int64).max
            continue
        while lo < hi:
            mid = (lo + hi) // 2
            if int(temporal_bucket(torch.tensor([mid]), 1 << 20)) >= k:
                hi = mid
            else:
                lo = mid + 1
        thr[k] = lo
    return thr
