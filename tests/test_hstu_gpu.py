"""GPU parity of the HSTU path (through the C ABI) against the golden fixtures of the reference and against the oracle."""
import pytest
import torch

from tests.util import budget, make_batch, relerr

pytestmark = pytest.mark.gpu


def _load_layer(g, dev):
    from genrec_b200.hstu import HSTULayer
    cfg = g["cfg"]
    layer = HSTULayer(cfg["embed_dim"], cfg["num_heads"], 0.0, 32, 64, 128, True)
    layer.load_state_dict(g["state_dict"])
    return layer.to(dev)


@pytest.mark.parametrize("name", ["hstu_layer_d64h2_L70.pt", "hstu_layer_d64h2_L1.pt"])
def test_layer_vs_reference_golden(golden, name):
    g = golden(name)
    dev = torch.device("cuda:0")
    layer = _load_layer(g, dev).train()
    x = g["x"].to(dev).requires_grad_(True)
    L = x.shape[1]
    causal = torch.triu(torch.ones(L, L, device=dev), diagonal=1).bool()
    y = layer(x, causal, g["padding_mask"].to(dev), g["timestamps"].to(dev))
    y.backward(g["dy"].to(dev))
    ac = g["autocast"]
    assert relerr(y, g["y"]) <= budget(ac["y"], g["y"]), relerr(y, g["y"])
    assert relerr(x.grad, g["dx"]) <= budget(ac["dx"], g["dx"]), relerr(x.grad, g["dx"])
    for n, p in layer.named_parameters():
        e, b = relerr(p.grad, g["grads"][n]), budget(ac["grads"][n], g["grads"][n])
        assert e <= b, f"{n}: {e} > {b}"
    # degenerate position bias (SURVEY section 0): only row 0 of the table receives gradient
    gp = layer.position_bias.relative_attention_bias.weight.grad
    assert gp[0].abs().sum() > 0 and gp[1:].abs().sum() == 0


@pytest.mark.parametrize("name", ["hstu_model_d64h2.pt", "hstu_model_d128h4_nots.pt", "hstu_model_notime.pt"])
def test_model_vs_reference_golden(golden, name):
    from genrec_b200.hstu import HSTU
    g = golden(name)
    cfg = g["cfg"]
    dev = torch.device("cuda:0")
    m = HSTU(cfg["num_items"], 64, cfg["embed_dim"], cfg["num_heads"], cfg["num_blocks"], dropout=0.0,
             use_temporal_bias=cfg["use_temporal_bias"])
    m.load_state_dict(g["state_dict"])
    m = m.to(dev).train()
    m.return_train_logits = True
    ids, tg = g["input_ids"].to(dev), g["targets"].to(dev)
    ts = g["timestamps"].to(dev) if cfg["pass_ts"] else None
    logits, loss = m(ids, ts, tg)
    loss.backward()
    ac = g["autocast"]
    assert logits.shape == g["logits"].shape and logits.dtype == torch.float32
    assert relerr(logits[:, -1], g["logits"][:, -1]) <= budget(ac["logits_last"], g["logits"][:, -1])
    assert abs(loss.item() - g["loss"].item()) <= 3 * abs(ac["loss"].item() - g["loss"].item()) + 5e-3
    for n, p in m.named_parameters():
        ref = g["grads"][n]
        got = p.grad if p.grad is not None else torch.zeros_like(p)
        if ref.abs().max() == 0:
            assert got.abs().max() == 0, n
            continue
        e, b = relerr(got, ref), budget(ac["grads"][n], ref, slack=2.0, floor=8e-3)
        assert e <= b, f"{n}: {e} > {b}"
    # padding_idx: no gather-gradient into row 0 beyond what the tied logits give (checked through the golden grads above)
    m.eval()
    top = m.predict(ids, ts, top_k=10)
    ref_top = g["top10"]
    overlap = sum(len(set(a.tolist()) & set(b.tolist())) for a, b in zip(top.cpu(), ref_top)) / ref_top.numel()
    assert overlap >= 0.9, overlap


@pytest.mark.parametrize("B,L,D,H", [(2, 7, 128, 4), (3, 50, 128, 4), (2, 200, 128, 4), (2, 257, 128, 4), (2, 130, 256, 8),
                                     (2, 64, 128, 2)])
def test_layer_vs_oracle_shapes(B, L, D, H):
    """Oracle (fp32, CPU) vs CUDA on seeded inputs across tile-boundary lengths, incl. padded and fully padded rows."""
    from genrec_b200.hstu import HSTULayer
    from oracle import hstu as oh
    dev = torch.device("cuda:0")
    torch.manual_seed(L * 131 + D)
    layer = HSTULayer(D, H, 0.0, 32, 64, 128, True)
    with torch.no_grad():
        for n, p in layer.named_parameters():
            if "attention_bias" in n:
                p.normal_(0, 0.5)
            elif n.endswith("bias"):
                p.normal_(0, 0.1)
            elif "norm" in n:
                p.add_(0.1 * torch.randn_like(p))
            else:
                p.normal_(0, 0.08)
    ids, ts, _ = make_batch(max(B, 3), L, 50, seed=L)
    ids, ts = ids[:B] if B < 3 else ids, ts[:B] if B < 3 else ts
    Bn = ids.shape[0]
    x = torch.randn(Bn, L, D)
    dy = torch.randn(Bn, L, D)
    sd = {k: v.detach().clone().requires_grad_(True) for k, v in layer.state_dict().items()}
    xo = x.clone().requires_grad_(True)
    yo = oh.hstu_layer_forward(xo, ids == 0, ts, sd, "", H)
    yo.backward(dy)
    layer = layer.to(dev).train()
    xg = x.to(dev).requires_grad_(True)
    yg = layer(xg, None, (ids == 0).to(dev), ts.to(dev))
    yg.backward(dy.to(dev))
    assert relerr(yg, yo) < 2.5e-2, relerr(yg, yo)
    assert relerr(xg.grad, xo.grad) < 2.5e-2, relerr(xg.grad, xo.grad)
    for n, p in layer.named_parameters():
        ref = sd[n].grad
        e = relerr(p.grad, ref)
        assert e < 4e-2, f"{n}: {e}"


def test_full_size_properties():
    """BASELINE cfg-2 shape (B=128, L=200, D=128, H=4): size-independent properties of the block."""
    from genrec_b200.hstu import HSTULayer
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    B, L, D, H = 128, 200, 128, 4
    layer = HSTULayer(D, H, 0.0, 32, 64, 128, True).to(dev).eval()
    with torch.no_grad():
        for n, p in layer.named_parameters():
            if "attention_bias" in n:
                p.normal_(0, 0.3)
    ids, ts, _ = make_batch(B, L, 12101, seed=1, pad=True, device=dev)
    x = torch.randn(B, L, D, device=dev)
    pad = ids == 0
    with torch.no_grad():
        y = layer(x, None, pad, ts)
        assert torch.isfinite(y).all()
        # determinism
        assert torch.equal(y, layer(x, None, pad, ts))
        # causality: perturbing positions >= 120 leaves outputs < 120 bit-identical
        x2 = x.clone(); x2[:, 120:] += 1.0
        ts2 = ts.clone(); ts2[:, 120:] += 999
        y2 = layer(x2, None, pad, ts2)
        assert torch.equal(y[:, :120], y2[:, :120]) and not torch.equal(y[:, 120:], y2[:, 120:])
        # padded keys are invisible: changing x at padded positions changes only those rows
        x3 = x.clone(); x3[pad] = 7.0
        y3 = layer(x3, None, pad, ts)
        assert torch.equal(y[~pad], y3[~pad])
        # batch independence: a sequence alone gives the same rows
        y1 = layer(x[5:6].contiguous(), None, pad[5:6], ts[5:6].contiguous())
        assert torch.equal(y1[0], y[5])
        # fully padded row: attention output is 0 -> finite, equals the no-attention path
        assert torch.isfinite(y[2]).all()
    # time-shift invariance: adding a constant to every timestamp leaves the result unchanged (bias depends on |dt| only)
    with torch.no_grad():
        tsh = ts.clone(); tsh[~pad] += 12345
        ysh = layer(x, None, pad, tsh)
        assert torch.equal(y[~pad], ysh[~pad])


def test_dropout_statistics_and_reseed():
    from genrec_b200.hstu import HSTU
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    m = HSTU(500, 50, 64, 2, 1, dropout=0.2).to(dev).train()
    ids, ts, tg = make_batch(8, 50, 500, seed=3, pad=False, device=dev)
    import genrec_b200.functional as Fn
    seed, sd = m._seeds(dev)
    x, _ = Fn.EmbedFn.apply(ids, m.item_embedding.weight, None, 1.0, 0, 0.2, seed, sd)
    frac = (x == 0).float().mean().item()
    assert 0.17 < frac < 0.23, frac
    kept = x[x != 0] / m.item_embedding.weight[ids][x != 0]
    assert torch.allclose(kept, torch.full_like(kept, 1.25), atol=1e-5)
    _, l1 = m(ids, ts, tg)
    _, l2 = m(ids, ts, tg)
    assert abs(l1.item() - l2.item()) > 1e-4   # device seed counter advanced -> different masks
    m.eval()
    _, e1 = m(ids, ts, tg)
    _, e2 = m(ids, ts, tg)
    assert abs(e1.item() - e2.item()) < 1e-5   # (float atomics in the loss reduction: not bit-deterministic)
    # gradient flows with dropout on and is finite
    m.train()
    _, l = m(ids, ts, tg)
    l.backward()
    assert all(torch.isfinite(p.grad).all() for p in m.parameters() if p.grad is not None)


def test_cpu_tensors_raise():
    from genrec_b200.hstu import HSTU
    m = HSTU(50, 20, 64, 2, 1, dropout=0.0)
    with pytest.raises(RuntimeError):
        m(torch.randint(1, 50, (2, 5)))
