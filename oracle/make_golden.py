"""Generate tests/golden/*.pt from the UNMODIFIED reference modules (build container only).

    python -m oracle.make_golden          # needs /root/reference

Every fixture holds seeded inputs, the reference ``state_dict`` and the reference's own outputs
(forward values and autograd gradients, fp32 unless noted).  The oracle restatement and the CUDA
path are both checked against these files; the files are small (< 2 MB together) and committed.
TEST INFRASTRUCTURE - see oracle/__init__.py.
"""
from __future__ import annotations

import io
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import ref_loader  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def _perturb(model, seed):
    """Reference init leaves biases 0 / LN = identity; perturb so every term is exercised."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for n, p in model.named_parameters():
            if n.endswith("norm.weight") or ".norm" in n and n.endswith("weight"):
                p.add_(0.1 * torch.randn(p.shape, generator=g))
            elif n.endswith("bias") and p.dim() == 1:
                p.copy_(0.1 * torch.randn(p.shape, generator=g))
            elif "attention_bias" in n:
                p.copy_(0.5 * torch.randn(p.shape, generator=g))
            elif "projection.weight" in n or "ffn" in n and n.endswith("weight"):
                p.copy_(0.15 * torch.randn(p.shape, generator=g))
            elif "item_embedding" in n:
                p.copy_(0.5 * torch.randn(p.shape, generator=g))
                p[0].zero_()


def _batch(B, L, V, seed, pad_rows=True):
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(1, V + 1, (B, L), generator=g)
    gaps = torch.randint(1, 3 * 86400, (B, L), generator=g)
    gaps[:, ::5] = torch.randint(1, 50, (B, (L + 4) // 5), generator=g)     # some near-simultaneous events
    ts = 1_300_000_000 + torch.cumsum(gaps, 1)
    tg = torch.roll(ids, -1, 1)
    tg[:, -1] = torch.randint(1, V + 1, (B,), generator=g)
    if pad_rows and B >= 3:
        n1 = L // 3
        ids[1, :n1] = 0; ts[1, :n1] = 0; tg[1, : n1 - 1] = 0               # left-padded, like hstu_collate_fn
        ids[2, :] = 0; ts[2, :] = 0; tg[2, :] = 0                           # fully padded row
        tg[2, -1] = 7                                                       # last pad position still has a target
    return ids, ts, tg


def golden_hstu(name, V, D, H, blocks, B, L, seed, use_time=True, pass_ts=True):
    R = ref_loader.ref_hstu()
    torch.manual_seed(seed)
    m = R.HSTU(num_items=V, max_seq_len=L, embed_dim=D, num_heads=H, num_blocks=blocks, dropout=0.0,
               use_temporal_bias=use_time)
    _perturb(m, seed + 1)
    m.train()
    ids, ts, tg = _batch(B, L, V, seed + 2)
    logits, loss = m(ids, ts if pass_ts else None, tg)
    loss.backward()
    grads = {n: (p.grad.clone() if p.grad is not None else torch.zeros_like(p)) for n, p in m.named_parameters()}
    m.zero_grad()
    with torch.autocast("cpu", dtype=torch.bfloat16):       # yardstick: the reference's own bf16-autocast error
        logits_ac, loss_ac = m(ids, ts if pass_ts else None, tg)
    loss_ac.float().backward()
    grads_ac = {n: (p.grad.clone() if p.grad is not None else torch.zeros_like(p)) for n, p in m.named_parameters()}
    m.eval()
    top = m.predict(ids, ts if pass_ts else None, top_k=10)
    _save(dict(autocast=dict(loss=loss_ac.detach().float(), grads=grads_ac, logits_last=logits_ac.detach().float()[:, -1]),
               cfg=dict(num_items=V, embed_dim=D, num_heads=H, num_blocks=blocks, use_temporal_bias=use_time,
                        pass_ts=pass_ts),
               state_dict={k: v.clone() for k, v in m.state_dict().items()},
               input_ids=ids, timestamps=ts, targets=tg,
               logits=logits.detach(), loss=loss.detach(), grads=grads, top10=top),
          name, parts=("grads", "autocast"))


def _save(d, name, parts=()):
    """torch.save ``d`` as tests/golden/<name>.  Fixture files stay under 1 MB: a larger one keeps each key in ``parts`` in its own
    file <stem>.<key>.pt (tests/conftest.py's ``golden`` loader puts them back)."""
    buf = io.BytesIO()
    torch.save(d, buf)
    if buf.tell() > 1_000_000 and parts:
        for key in parts:
            torch.save(d.pop(key), os.path.join(OUT, f"{name[:-3]}.{key}.pt"))
        d["_parts"] = list(parts)
    torch.save(d, os.path.join(OUT, name))


def golden_hstu_fp64(name, seed=3):
    """The reference HSTU in fp64 (default init, no dropout) on a padded batch with timestamps: logits and loss, for the oracle's
    1e-12 agreement check.  The parameters are initialised in fp32 and converted, so they are stored in fp32 exactly."""
    R = ref_loader.ref_hstu()
    torch.manual_seed(seed)
    m = R.HSTU(num_items=60, max_seq_len=40, embed_dim=64, num_heads=2, num_blocks=2, dropout=0.0).double()
    B, L = 3, 37
    ids = torch.randint(1, 61, (B, L)); ids[0, :11] = 0
    ts = torch.cumsum(torch.randint(1, 10 ** 6, (B, L)), 1) + 1_300_000_000; ts[ids == 0] = 0
    tg = torch.randint(1, 61, (B, L))
    with torch.no_grad():
        logits, loss = m(ids, ts, tg)
    sd = {k: v.float() for k, v in m.state_dict().items()}
    assert all(torch.equal(sd[k].double(), v) for k, v in m.state_dict().items())
    _save(dict(cfg=dict(num_heads=2, num_blocks=2), state_dict=sd, input_ids=ids, timestamps=ts, targets=tg, logits=logits,
               loss=loss), name)


def golden_hstu_layer(name, D, H, B, L, seed):
    R = ref_loader.ref_hstu()
    torch.manual_seed(seed)
    layer = R.HSTULayer(embed_dim=D, num_heads=H, dropout=0.0, num_position_buckets=32, num_time_buckets=64,
                        max_position_distance=128, use_temporal_bias=True)
    _perturb(layer, seed + 1)
    g = torch.Generator().manual_seed(seed + 3)
    ids, ts, _ = _batch(B, L, 100, seed + 2)
    x = torch.randn(B, L, D, generator=g).requires_grad_(True)
    dy = torch.randn(B, L, D, generator=g)
    causal = torch.triu(torch.ones(L, L), diagonal=1).bool()
    y = layer(x, causal, ids == 0, ts)
    y.backward(dy)
    ref = dict(y=y.detach().clone(), dx=x.grad.clone(), grads={n: p.grad.clone() for n, p in layer.named_parameters()})
    layer.zero_grad(); x.grad = None
    with torch.autocast("cpu", dtype=torch.bfloat16):
        y_ac = layer(x, causal, ids == 0, ts)
    y_ac.float().backward(dy)
    ac = dict(y=y_ac.detach().float(), dx=x.grad.clone(), grads={n: p.grad.clone() for n, p in layer.named_parameters()})
    layer.zero_grad(); x.grad = None
    y = layer(x, causal, ids == 0, ts)
    y.backward(dy)
    torch.save(dict(autocast=ac, cfg=dict(embed_dim=D, num_heads=H),
                    state_dict={k: v.clone() for k, v in layer.state_dict().items()},
                    x=x.detach(), dy=dy, padding_mask=(ids == 0), timestamps=ts, y=y.detach(), dx=x.grad.clone(),
                    grads={n: p.grad.clone() for n, p in layer.named_parameters()}),
               os.path.join(OUT, name))


def golden_sasrec(name, V, D, H, blocks, F_, B, L, seed):
    S = ref_loader.ref_sasrec()
    torch.manual_seed(seed)
    m = S.SASRec(num_items=V, max_seq_len=L + 3, embed_dim=D, num_heads=H, num_blocks=blocks, ffn_dim=F_, dropout=0.0)
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for n, p in m.named_parameters():
            if n.endswith("bias"):
                p.copy_(0.1 * torch.randn(p.shape, generator=g))
            elif "norm" in n:
                p.add_(0.1 * torch.randn(p.shape, generator=g))
    m.train()
    ids, _, tg = _batch(B, L, V, seed + 2)
    logits, loss = m(ids, tg)
    loss.backward()
    # attention module alone (block 0), with a gradient probe
    attn = m.blocks[0].attention
    xq = torch.randn(B, L, D, generator=g).requires_grad_(True)
    xkv = torch.randn(B, L, D, generator=g).requires_grad_(True)
    mask = (ids != 0).unsqueeze(-1).float()
    dout = torch.randn(B, L, D, generator=g)
    grads_model = {n: p.grad.clone() for n, p in m.named_parameters()}
    m.zero_grad()
    out = attn(xq, xkv, mask)
    out.backward(dout)
    torch.save(dict(cfg=dict(num_items=V, embed_dim=D, num_heads=H, num_blocks=blocks, ffn_dim=F_, max_seq_len=L + 3),
                    state_dict={k: v.clone() for k, v in m.state_dict().items()},
                    input_ids=ids, targets=tg, logits=logits.detach(), loss=loss.detach(), grads=grads_model,
                    attn=dict(query=xq.detach(), key_value=xkv.detach(), mask=mask, dout=dout, out=out.detach(),
                              dquery=xq.grad.clone(), dkey_value=xkv.grad.clone(),
                              grads={n: p.grad.clone() for n, p in attn.named_parameters()})),
               os.path.join(OUT, name))


def _pin_dropout(model, sites, seed, p):
    """Replace the output of every nn.Dropout of ``model`` by ``input * mask`` through forward hooks (the reference source stays
    untouched).  ``sites(module_name, call_index) -> oracle site name``: a module that runs more than once per forward (SASRec's
    PointWiseFeedForward) is told apart by call order.  The keep masks are drawn once per site name (first forward) and replayed
    afterwards; returns (masks, reset) - call reset() before each forward."""
    g = torch.Generator().manual_seed(seed)
    masks, calls = {}, {}

    def hook(mod_name):
        def f(mod, inp, out):
            k = calls.get(mod_name, 0)
            calls[mod_name] = k + 1
            site = sites(mod_name, k)
            if site not in masks:
                masks[site] = torch.rand(inp[0].shape, generator=g) >= p
            return inp[0] * (masks[site].to(inp[0].dtype) / (1 - p))
        return f

    for n, mod in model.named_modules():
        if isinstance(mod, torch.nn.Dropout):
            mod.register_forward_hook(hook(n))
    return masks, calls.clear


def golden_hstu_dropout(name, V=50, D=64, H=2, blocks=2, B=3, L=20, p=0.2, seed=110):
    """The reference HSTU in train mode with every nn.Dropout pinned to a recorded mask: loss, logits and every gradient, plus the
    masks (bool, True = kept; a kept element is scaled by 1 / (1 - p)) under the oracle's site names."""
    R = ref_loader.ref_hstu()
    torch.manual_seed(seed)
    m = R.HSTU(num_items=V, max_seq_len=L, embed_dim=D, num_heads=H, num_blocks=blocks, dropout=p)
    _perturb(m, seed + 1)
    m.train()
    names = {"emb_dropout": "emb"}
    for i in range(blocks):
        names.update({f"layers.{i}.dropout": f"layers.{i}.gate", f"layers.{i}.ffn.2": f"layers.{i}.ffn_hid",
                      f"layers.{i}.ffn.4": f"layers.{i}.ffn_out"})
    masks, reset = _pin_dropout(m, lambda n, k: names[n], seed + 3, p)
    ids, ts, tg = _batch(B, L, V, seed + 2)
    reset()
    logits, loss = m(ids, ts, tg)
    loss.backward()
    assert sorted(masks) == sorted(names.values())
    _save(dict(cfg=dict(num_heads=H, num_blocks=blocks, p=p), state_dict={k: v.clone() for k, v in m.state_dict().items()},
               input_ids=ids, timestamps=ts, targets=tg, masks=masks, logits=logits.detach(), loss=loss.detach(),
               grads={n: q.grad.clone() for n, q in m.named_parameters()}), name)


def golden_sasrec_dropout(name, V=50, D=64, H=2, blocks=2, F_=128, B=3, L=20, p=0.2, seed=120):
    """As golden_hstu_dropout, for SASRec: embedding, attention weights, and the two calls of each block's FFN dropout."""
    S = ref_loader.ref_sasrec()
    torch.manual_seed(seed)
    m = S.SASRec(num_items=V, max_seq_len=L, embed_dim=D, num_heads=H, num_blocks=blocks, ffn_dim=F_, dropout=p)
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for n, q in m.named_parameters():
            if n.endswith("bias"):
                q.copy_(0.1 * torch.randn(q.shape, generator=g))
            elif "norm" in n:
                q.add_(0.1 * torch.randn(q.shape, generator=g))
    m.train()

    def site(n, k):
        if n == "emb_dropout":
            return "emb"
        blk = n.split(".attention.")[0].split(".ffn.")[0] + "."
        return blk + ("attn" if n.endswith("attention.dropout") else ("ffn_hid", "ffn_out")[k])

    masks, reset = _pin_dropout(m, site, seed + 3, p)
    ids, _, tg = _batch(B, L, V, seed + 2)
    reset()
    logits, loss = m(ids, tg)
    loss.backward()
    assert len(masks) == 1 + 3 * blocks
    _save(dict(cfg=dict(num_heads=H, num_blocks=blocks, p=p), state_dict={k: v.clone() for k, v in m.state_dict().items()},
               input_ids=ids, targets=tg, masks=masks, logits=logits.detach(), loss=loss.detach(),
               grads={n: q.grad.clone() for n, q in m.named_parameters()}), name)


def golden_rqvae(name, seed, N=300, levels=3, K=256, D=32):
    ns = ref_loader.ref_genrec_package()
    rq = ns.rqvae
    torch.manual_seed(seed)
    m = rq.RqVae(input_dim=96, embed_dim=D, hidden_dims=[64, 48], codebook_size=K,
                 codebook_kmeans_init=False, codebook_mode=rq.QuantizeForwardMode.STE,
                 codebook_last_layer_mode=rq.QuantizeForwardMode.STE, n_layers=levels, n_cat_features=0)
    m.eval()
    g = torch.Generator().manual_seed(seed + 1)
    x = torch.randn(N, 96, generator=g)
    x = x / x.norm(dim=1, keepdim=True)
    with torch.no_grad():
        # spread the latent so that all three levels see non-trivial residuals
        for i, l in enumerate(m.layers):
            l.embedding.weight.copy_((torch.rand(K, D, generator=g) - 0.5) * (0.4 / (2 ** i)))
        # exact ties: duplicate a code so the first-index rule is exercised
        m.layers[0].embedding.weight[200] = m.layers[0].embedding.weight[17]
        m.layers[1].embedding.weight[3] = m.layers[1].embedding.weight[250]
        out = m.get_semantic_ids(x)
        latent = m.encode(x)
    torch.save(dict(cfg=dict(levels=levels, K=K, D=D, input_dim=96, hidden_dims=[64, 48]),
                    state_dict={k: v.clone() for k, v in m.state_dict().items() if not k.startswith("decoder")},
                    x=x, latent=latent, embeddings=out.embeddings, residuals=out.residuals, sem_ids=out.sem_ids,
                    quantize_loss=out.quantize_loss),
               os.path.join(OUT, name))


def golden_kats(name):
    R = ref_loader.ref_hstu()
    ns = ref_loader.ref_genrec_package()
    tb = R.TemporalBias(64, 2)
    pb = R.RelativePositionBias(32, 128, 2)
    thr = [2, 4, 8, 16, 32, 64, 128, 256, 512, 1023, 2045, 4089, 8177, 16351, 32696, 65382, 130745, 261451, 522824,
           1045495, 2090681, 4180745, 8360257, 16718042, 33431190, 66852590, 133685356, 267331576, 534583856,
           1069011233, 2137709504, 4274784897, 8548302081]
    near = torch.tensor([t + o for t in thr for o in (-2, -1, 0, 1, 2)])
    d = torch.cat([torch.arange(0, 3000), near, torch.tensor([86400, 522823, 522824, 522825, 2 ** 24 + 1, 10 ** 8, 2 ** 31 - 1,
                                                          2 ** 31, 2 ** 31 + 129, 1_700_000_000, 2 ** 40, 2 ** 62])])
    g = torch.Generator().manual_seed(5)
    d = torch.cat([d, torch.randint(1, 2 ** 31, (4000,), generator=g)])
    pos = torch.arange(150)
    rel = pos.unsqueeze(0) - pos.unsqueeze(1)
    col = ns.amazon_hstu.hstu_collate_fn(
        [dict(history=[1, 2, 3], timestamps=[10, 20, 30], target=4), dict(history=[5], timestamps=[7], target=6)], 50)
    ecol = ns.amazon_hstu.hstu_eval_collate_fn(
        [dict(history=[1, 2, 3], timestamps=[10, 20, 30], target=4), dict(history=[5], timestamps=[7], target=6)], 2)
    scol = ns.amazon_sasrec.sasrec_collate_fn(
        [dict(history=[1, 2, 3], target=4), dict(history=[5], target=6)], 50) if hasattr(ns.amazon_sasrec, "sasrec_collate_fn") else None
    torch.save(dict(dt=d, dt_bucket=tb._temporal_bucket(d).to(torch.int8), dt_bucket_neg=tb._temporal_bucket(-d).to(torch.int8),
                    rel_bucket_150=pb._relative_position_bucket(rel).to(torch.int8),
                    rel_bucket_raw=pb._relative_position_bucket(torch.arange(-5, 400)),
                    silu_m1e9_f32=torch.nn.functional.silu(torch.tensor([-1e9])),
                    silu_m1e9_bf16=torch.nn.functional.silu(torch.tensor([-1e9], dtype=torch.bfloat16)).float(),
                    hstu_collate=col, hstu_eval_collate=ecol, sasrec_collate=scol),
               os.path.join(OUT, name))


def golden_tiger_decode(name, seed, B=3, K=4, num_emb=8, sem_dim=3, use_trie=True):
    """Tiger.generate of the unmodified reference on a tiny random model; records what the decode loop consumed (per-step logits,
    the torch.multinomial draws) and produced (final beams), so the post-processing can be replayed without the model."""
    tg = ref_loader.ref_tiger()
    torch.manual_seed(seed)
    m = tg.Tiger(embedding_dim=32, attn_dim=48, dropout=0.0, num_heads=2, n_layers=2, num_item_embeddings=num_emb,
                 num_user_embeddings=10, sem_id_dim=sem_dim).eval()
    g = torch.Generator().manual_seed(seed + 1)
    # a small item set with shared prefixes, a duplicate item and a first level with fewer than K distinct tokens
    valid = torch.tensor([[1, 2, 3], [1, 2, 5], [1, 4, 0], [6, 0, 0], [6, 0, 7], [6, 3, 3], [2, 2, 2], [2, 2, 2], [1, 4, 1]])
    N = 6
    users = torch.randint(0, 10, (B, 1), generator=g)
    items = torch.randint(0, num_emb, (B, N), generator=g)
    types = torch.arange(N).remainder(sem_dim).unsqueeze(0).expand(B, -1).contiguous()
    mask = torch.ones(B, N, dtype=torch.long)
    mask[1, 4:] = 0
    step_logits, draws = [], []
    orig_step, orig_multi = m._decode_step, torch.multinomial

    def rec_step(*a, **k):
        out = orig_step(*a, **k)
        step_logits.append(out.detach().clone())
        return out

    def rec_multi(*a, **k):
        out = orig_multi(*a, **k)
        draws.append(out.clone())
        return out

    m._decode_step = rec_step
    torch.multinomial = rec_multi
    try:
        with torch.no_grad():
            out = m.generate(users, items, types, mask, temperature=0.2, n_top_k_candidates=K, valid_item_ids=valid, use_trie=use_trie)
    finally:
        torch.multinomial = orig_multi
    torch.save(dict(cfg=dict(B=B, K=K, num_emb=num_emb, sem_dim=sem_dim, temperature=0.2, use_trie=use_trie), valid_item_ids=valid,
                    step_logits=step_logits, draws=draws, sem_ids=out.sem_ids.clone(), log_probas=out.log_probas.detach().clone()),
               os.path.join(OUT, name))


def golden_t5_attention(name, seed, D=64, H=2, B=3, Lq=37, Lk=21):
    """T5Attention of the unmodified reference: encoder self-attention with key padding, decoder self-attention with the causal mask,
    cross-attention with memory padding - outputs and every gradient, fp32."""
    tr = ref_loader.ref_transformer()
    torch.manual_seed(seed)
    g = torch.Generator().manual_seed(seed + 1)
    cases = {}
    for case, cross, q_len, k_len, causal in (("encoder", False, Lq, Lq, False), ("decoder", False, 9, 9, True), ("cross", True, 9, Lk, False)):
        heads = 1 if case == "decoder" else H          # head_dim 64 in the decoder case, 32 in the others
        m = tr.T5Attention(D, heads, dropout=0.0, is_cross_attention=cross).eval()
        with torch.no_grad():
            for p in m.parameters():
                p.copy_(torch.randn(p.shape, generator=g) * (0.5 if p.shape[-1] == 1 else 0.09))
        x = torch.randn(B, q_len, D, generator=g, requires_grad=True)
        ctx = torch.randn(B, k_len, D, generator=g, requires_grad=True) if cross else None
        pad = torch.zeros(B, k_len, dtype=torch.bool)
        pad[1, k_len - 5:] = True
        if case == "encoder":
            pad[2, :] = True                     # a fully padded sequence: the reference's softmax is uniform there
        if case == "decoder":
            pad = None
        mask = torch.nn.Transformer.generate_square_subsequent_mask(q_len) if causal else None
        out, _ = m(x, ctx, ctx, attn_mask=mask, key_padding_mask=pad)
        dy = torch.randn(out.shape, generator=g)
        out.backward(dy)
        cases[case] = dict(cross=cross, causal=causal, heads=heads, state_dict={k: v.detach().clone() for k, v in m.state_dict().items()}, x=x.detach().clone(),
                           ctx=ctx.detach().clone() if cross else None, pad=pad, dy=dy, out=out.detach().clone(), dx=x.grad.clone(),
                           dctx=ctx.grad.clone() if cross else None, grads={n: p.grad.clone() for n, p in m.named_parameters()})
    torch.save(dict(cfg=dict(D=D, H=H), cases=cases), os.path.join(OUT, name))


def main():
    assert ref_loader.available(), "reference tree not found"
    os.makedirs(OUT, exist_ok=True)
    golden_hstu("hstu_model_d64h2.pt", V=50, D=64, H=2, blocks=2, B=4, L=24, seed=10)
    golden_hstu("hstu_model_d128h4_nots.pt", V=40, D=128, H=4, blocks=1, B=3, L=17, seed=20, use_time=True, pass_ts=False)
    golden_hstu("hstu_model_notime.pt", V=40, D=64, H=2, blocks=1, B=3, L=9, seed=30, use_time=False)
    golden_hstu_fp64("hstu_model_fp64.pt")
    golden_hstu_layer("hstu_layer_d64h2_L70.pt", D=64, H=2, B=3, L=70, seed=40)
    golden_hstu_layer("hstu_layer_d64h2_L1.pt", D=64, H=2, B=3, L=1, seed=50)
    golden_sasrec("sasrec_d64h2.pt", V=50, D=64, H=2, blocks=2, F_=256, B=4, L=21, seed=60)
    golden_hstu_dropout("hstu_dropout.pt")
    golden_sasrec_dropout("sasrec_dropout.pt")
    golden_rqvae("rqvae_3x256x32.pt", seed=70)
    golden_kats("kats.pt")
    golden_t5_attention("t5_attention.pt", seed=100)
    golden_tiger_decode("tiger_decode_trie.pt", seed=80)
    golden_tiger_decode("tiger_decode_notrie.pt", seed=90, use_trie=False)
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
