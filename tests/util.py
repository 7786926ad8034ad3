from typing import Optional

import torch


def relerr(a: torch.Tensor, ref: torch.Tensor) -> float:
    """max-norm relative error: |a - ref|_inf / |ref|_inf (SURVEY.md section 7 'autocast semantics')."""
    a, ref = a.detach().float().cpu(), ref.detach().float().cpu()
    d = ref.abs().max().item()
    return ((a - ref).abs().max().item() / d) if d > 0 else (a - ref).abs().max().item()


def budget(golden_ac: torch.Tensor, golden: torch.Tensor, slack: float = 1.5, floor: float = 4e-3) -> float:
    """bf16 tolerance = slack x the reference's OWN bf16-autocast error on this tensor (+ a small floor)."""
    return slack * relerr(golden_ac, golden) + floor


HSTU_LAYER_KEYS = {
    "projection.weight": "proj_w", "projection.bias": "proj_b",
}


def make_batch(B, L, V, seed, pad=True, device="cpu"):
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(1, V + 1, (B, L), generator=g)
    gaps = torch.randint(1, 3 * 86400, (B, L), generator=g)
    gaps[:, ::5] = torch.randint(1, 50, (B, (L + 4) // 5), generator=g)
    ts = 1_300_000_000 + torch.cumsum(gaps, 1)
    tg = torch.roll(ids, -1, 1)
    tg[:, -1] = torch.randint(1, V + 1, (B,), generator=g)
    if pad and B >= 3 and L >= 3:
        n1 = max(1, L // 3)
        ids[1, :n1] = 0; ts[1, :n1] = 0; tg[1, : n1 - 1] = 0
        ids[2, :] = 0; ts[2, :] = 0; tg[2, :] = 0
        tg[2, -1] = 7
    return ids.to(device), ts.to(device), tg.to(device)


def close(a: torch.Tensor, ref: torch.Tensor, rel: float, floor: float = 1e-4) -> bool:
    """|a - ref|_inf <= rel * max(|ref|_inf, floor)  (floor: gradients that are analytically zero, e.g. the key-projection
    bias under a softmax, are pure rounding noise in both implementations)."""
    a, ref = a.detach().float().cpu(), ref.detach().float().cpu()
    return (a - ref).abs().max().item() <= rel * max(ref.abs().max().item(), floor)


def drop_thresh_scale(p: float):
    """(thresh, keep scale) of csrc/common.cuh make_dropout: an element is dropped when its 16 random bits are < thresh =
    round(p * 2^16) (p as the float32 the C ABI receives), a kept one is scaled by the float32 65536 / (65536 - thresh) - the
    reciprocal of the realised keep probability, not exactly 1 / (1 - p)."""
    import numpy as np
    t = float(np.float32(p)) * 65536.0 + 0.5
    thresh = 0 if p <= 0 else min(int(t), 65536)
    scale = 0.0 if thresh >= 65536 else float(np.float32(65536.0) / np.float32(65536 - thresh))
    return thresh, scale


def drop_mask(rows, cols, p: float, seed: int, site: int, seed_dev: Optional[int] = None):
    """numpy restatement of csrc/common.cuh Dropout: bool [len(rows), len(cols)], True = dropped, for the elements at (row, column)
    of the operand a kernel addresses its mask by.  The kernel's seed is ``seed + *seed_dev`` (uint64, wrapping, so a carry into
    the high word counts); rows and columns are uint32 (a column pair shares one hash: low 16 bits for even, high for odd)."""
    import numpy as np
    u = np.uint32
    thresh, _ = drop_thresh_scale(p)
    s = (int(seed) + int(seed_dev or 0)) & 0xFFFFFFFFFFFFFFFF
    k0 = u((s & 0xFFFFFFFF) ^ ((int(site) * 0x9E3779B1) & 0xFFFFFFFF))
    k1 = u(((s >> 32) + 0x7F4A7C15) & 0xFFFFFFFF)
    row = (np.asarray(rows, dtype=np.int64) & 0xFFFFFFFF).astype(np.uint32)[:, None]
    col = (np.asarray(cols, dtype=np.int64) & 0xFFFFFFFF).astype(np.uint32)[None, :]
    with np.errstate(over="ignore"):
        ka = (row ^ k1) * u(0x9E3779B1)
        ka = ka ^ (ka >> u(16))
        b = ka * u(0x846CA68B)
        kb = k0 ^ (b ^ (b >> u(15)))
        x = ((col >> u(1)) ^ kb) * u(0x7FEB352D)
        x = x ^ (x >> u(15))
        x = (x ^ ka) * u(0x846CA68B)
        x = x ^ (x >> u(16))
    bits = np.where((col & u(1)) != 0, x >> u(16), x & u(0xFFFF))
    return bits < thresh


def keep_scale(rows, cols, p: float, seed: int, site: int, seed_dev: Optional[int] = None, dtype=torch.float64) -> torch.Tensor:
    """What the kernel multiplies each element by: 0 where ``drop_mask`` drops, the keep scale elsewhere."""
    _, scale = drop_thresh_scale(p)
    return torch.from_numpy(~drop_mask(rows, cols, p, seed, site, seed_dev)).to(dtype) * scale


def frob_relerr(a: torch.Tensor, ref: torch.Tensor) -> float:
    a, ref = a.detach().double().cpu(), ref.detach().double().cpu()
    d = ref.norm().item()
    return (a - ref).norm().item() / d if d > 0 else (a - ref).norm().item()
