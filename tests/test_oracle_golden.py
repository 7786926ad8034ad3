"""The oracle restatement vs the fixtures produced by the UNMODIFIED reference (oracle/make_golden.py)."""
import numpy as np
import pytest
import torch

from oracle import hstu as oh
from oracle import rqvae as orq
from oracle import sasrec as osr


def _req(t):
    return {k: v.clone().requires_grad_(v.is_floating_point()) for k, v in t.items()}


@pytest.mark.parametrize("name", ["hstu_model_d64h2.pt", "hstu_model_d128h4_nots.pt", "hstu_model_notime.pt"])
def test_hstu_model_forward_backward(golden, name):
    g = golden(name)
    cfg = g["cfg"]
    p = _req(g["state_dict"])
    ts = g["timestamps"] if cfg["pass_ts"] else None
    logits, loss = oh.hstu_forward(g["input_ids"], ts, g["targets"], p, cfg["num_heads"], cfg["num_blocks"],
                                   use_temporal_bias=cfg["use_temporal_bias"])
    torch.testing.assert_close(logits, g["logits"], rtol=1e-5, atol=2e-5)
    torch.testing.assert_close(loss, g["loss"], rtol=1e-6, atol=1e-6)
    loss.backward()
    for n, gr in g["grads"].items():
        got = p[n].grad if p[n].grad is not None else torch.zeros_like(p[n])
        torch.testing.assert_close(got, gr, rtol=2e-4, atol=2e-6, msg=lambda m: f"{n}: {m}")
    top = oh.hstu_predict(g["input_ids"], ts, g["state_dict"], cfg["num_heads"], cfg["num_blocks"],
                          use_temporal_bias=cfg["use_temporal_bias"])
    assert torch.equal(top, g["top10"])


@pytest.mark.parametrize("name", ["hstu_layer_d64h2_L70.pt", "hstu_layer_d64h2_L1.pt"])
def test_hstu_layer(golden, name):
    g = golden(name)
    p = _req(g["state_dict"])
    x = g["x"].clone().requires_grad_(True)
    y = oh.hstu_layer_forward(x, g["padding_mask"], g["timestamps"], p, "", g["cfg"]["num_heads"])
    torch.testing.assert_close(y, g["y"], rtol=1e-5, atol=2e-5)
    y.backward(g["dy"])
    torch.testing.assert_close(x.grad, g["dx"], rtol=1e-4, atol=5e-5)
    for n, gr in g["grads"].items():
        torch.testing.assert_close(p[n].grad, gr, rtol=2e-4, atol=1e-4, msg=lambda m: f"{n}: {m}")


def test_degenerate_position_bias_known_answer(golden):
    """SURVEY section 0: every causal cell uses bucket 0; rows 1.. of the table get zero gradient."""
    g = golden("hstu_layer_d64h2_L70.pt")
    gr = g["grads"]["position_bias.relative_attention_bias.weight"]
    assert gr[0].abs().sum() > 0 and gr[1:].abs().sum() == 0
    k = golden("kats.pt")
    rb = k["rel_bucket_150"]
    L = rb.shape[0]
    causal = torch.tril(torch.ones(L, L)).bool()
    assert int(rb[causal].max()) == 0
    pos = torch.arange(L)
    assert torch.equal(oh.position_bucket(pos[None] - pos[:, None]).to(torch.int8), rb)
    assert torch.equal(oh.position_bucket(torch.arange(-5, 400)), k["rel_bucket_raw"])


def test_temporal_bucket_known_answers(golden):
    k = golden("kats.pt")
    assert torch.equal(oh.temporal_bucket(k["dt"]).to(torch.int8), k["dt_bucket"])
    assert torch.equal(oh.temporal_bucket(-k["dt"]).to(torch.int8), k["dt_bucket_neg"])
    got = oh.temporal_bucket(torch.tensor([0, 1, 2, 3, 4, 1023, 1024, 86400, 2 ** 31])).tolist()
    assert got == [0, 0, 1, 1, 2, 10, 10, 16, 31]
    # integer-threshold form (what the CUDA kernel uses) == the fp32-log form
    thr = oh.time_bucket_thresholds(64)
    d = k["dt"].clamp(min=1)
    e = torch.floor(torch.log2(d.double())).long()
    e = torch.where((1 << e.clamp(max=62)) > d, e - 1, e)
    b = e + (d >= thr[(e + 1).clamp(max=63)]).long()
    assert torch.equal(b.clamp(0, 63).to(torch.int8), k["dt_bucket"])
    assert float(k["silu_m1e9_f32"]) == 0.0 and float(k["silu_m1e9_bf16"]) == 0.0


def test_sasrec(golden):
    g = golden("sasrec_d64h2.pt")
    cfg = g["cfg"]
    p = _req(g["state_dict"])
    logits, loss = osr.sasrec_forward(g["input_ids"], g["targets"], p, cfg["num_heads"], cfg["num_blocks"])
    torch.testing.assert_close(logits, g["logits"], rtol=1e-5, atol=5e-5)
    torch.testing.assert_close(loss, g["loss"], rtol=1e-6, atol=1e-6)
    loss.backward()
    for n, gr in g["grads"].items():
        got = p[n].grad if p[n].grad is not None else torch.zeros_like(p[n])
        torch.testing.assert_close(got, gr, rtol=5e-4, atol=5e-6, msg=lambda m: f"{n}: {m}")
    a = g["attn"]
    p = _req(g["state_dict"])
    q = a["query"].clone().requires_grad_(True)
    kv = a["key_value"].clone().requires_grad_(True)
    out = osr.sasrec_attention_forward(q, kv, a["mask"], p, "blocks.0.attention.", cfg["num_heads"])
    torch.testing.assert_close(out, a["out"], rtol=1e-5, atol=1e-5)
    out.backward(a["dout"])
    torch.testing.assert_close(q.grad, a["dquery"], rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(kv.grad, a["dkey_value"], rtol=1e-4, atol=1e-5)
    for n, gr in a["grads"].items():
        torch.testing.assert_close(p["blocks.0.attention." + n].grad, gr, rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("name", ["hstu_dropout.pt", "sasrec_dropout.pt"])
def test_dropout_sites_vs_reference_golden(golden, name):
    """Training mode: the unmodified reference with every nn.Dropout pinned to a recorded mask (oracle/make_golden.py) against the
    oracle's ``drop`` hook fed the same masks - each hook sits where the reference applies its dropout, and every site is used."""
    g = golden(name)
    cfg = g["cfg"]
    p = _req(g["state_dict"])
    used = []

    def drop(site, t):
        used.append(site)
        return t * (g["masks"][site].to(t.dtype) / (1 - cfg["p"]))

    if name.startswith("hstu"):
        logits, loss = oh.hstu_forward(g["input_ids"], g["timestamps"], g["targets"], p, cfg["num_heads"], cfg["num_blocks"], drop=drop)
    else:
        logits, loss = osr.sasrec_forward(g["input_ids"], g["targets"], p, cfg["num_heads"], cfg["num_blocks"], drop=drop)
    assert sorted(used) == sorted(g["masks"])
    torch.testing.assert_close(logits, g["logits"], rtol=1e-5, atol=5e-5)
    torch.testing.assert_close(loss, g["loss"], rtol=1e-6, atol=1e-6)
    loss.backward()
    for n, gr in g["grads"].items():
        got = p[n].grad if p[n].grad is not None else torch.zeros_like(p[n])
        torch.testing.assert_close(got, gr, rtol=5e-4, atol=5e-6, msg=lambda m: f"{n}: {m}")
    # the masks really drop: without them the oracle is far from the recording
    lo0, _ = (oh.hstu_forward(g["input_ids"], g["timestamps"], None, g["state_dict"], cfg["num_heads"], cfg["num_blocks"])
              if name.startswith("hstu") else osr.sasrec_forward(g["input_ids"], None, g["state_dict"], cfg["num_heads"], cfg["num_blocks"]))
    assert (lo0 - g["logits"]).abs().max() > 1e-2 * g["logits"].abs().max()


def test_rqvae(golden):
    g = golden("rqvae_3x256x32.pt")
    sd = g["state_dict"]
    enc = [sd[k] for k in sorted(k for k in sd if k.startswith("encoder.mlp"))]
    latent = orq.mlp_encoder(g["x"], enc)
    torch.testing.assert_close(latent, g["latent"], rtol=1e-6, atol=1e-6)
    cbs = [sd[f"layers.{i}.embedding.weight"] for i in range(g["cfg"]["levels"])]
    out = orq.residual_quantize(g["latent"], cbs)
    assert torch.equal(out.sem_ids, g["sem_ids"])
    torch.testing.assert_close(out.embeddings, g["embeddings"], rtol=0, atol=0)
    torch.testing.assert_close(out.residuals, g["residuals"], rtol=0, atol=0)
    torch.testing.assert_close(out.quantize_loss, g["quantize_loss"], rtol=1e-6, atol=1e-7)
    # duplicated codes (exact ties) resolve to the first index
    assert 200 not in out.sem_ids[:, 0].tolist() and 250 not in out.sem_ids[:, 1].tolist()
    # the C restatement agrees except where the torch GEMM's rounding flips a near-tie
    ids_c, _ = orq.residual_quantize_c(g["latent"].numpy(), torch.stack(cbs).numpy())
    agree = (torch.from_numpy(ids_c) == g["sem_ids"]).all(dim=1).float().mean()
    assert agree > 0.98


def test_collate_known_answers(golden):
    k = golden("kats.pt")
    c = k["hstu_collate"]
    assert c["input_ids"].tolist() == [[1, 2, 3], [0, 0, 5]]
    assert c["targets"].tolist() == [[2, 3, 4], [0, 5, 6]]
    assert c["timestamps"].tolist() == [[10, 20, 30], [0, 0, 7]]


def test_oracle_vs_reference_fp64(golden):
    """The oracle restatement in fp64 reproduces the logits and loss of the unmodified reference HSTU run in fp64."""
    g = golden("hstu_model_fp64.pt")
    sd = {k: v.double() for k, v in g["state_dict"].items()}
    lo, ls = oh.hstu_forward(g["input_ids"], g["timestamps"], g["targets"], sd, g["cfg"]["num_heads"], g["cfg"]["num_blocks"])
    assert lo.dtype == g["logits"].dtype == torch.float64
    assert (lo - g["logits"]).abs().max() < 1e-12 and (ls - g["loss"]).abs() < 1e-12


@pytest.mark.parametrize("name", ["tiger_decode_trie.pt", "tiger_decode_notrie.pt"])
def test_tiger_decode_oracle_vs_reference_recording(golden, name):
    """The oracle's restatement of Tiger.generate's post-processing replays the recorded logits and multinomial draws of the unmodified
    reference to the same beams (tiger.py:364-441)."""
    from oracle import tiger_decode as od
    g = golden(name)
    c = g["cfg"]
    s, l = od.replay(g["step_logits"], g["draws"], g["valid_item_ids"], c["B"], c["K"], c["num_emb"], c["temperature"], c["use_trie"])
    assert torch.equal(s, g["sem_ids"])
    assert torch.equal(l, g["log_probas"])


def test_trie_csr_equals_the_dict_trie():
    """Host-side data format: the CSR trie holds exactly the nodes and edges of the reference's dict trie (tiger.py:49-69)."""
    from genrec_b200.tiger_decode import TrieCSR
    from oracle import tiger_decode as od
    g = torch.Generator().manual_seed(0)
    valid = torch.randint(0, 12, (300, 3), generator=g)
    valid[10] = valid[3]
    root = od.build_trie(valid)
    t = TrieCSR.build(valid)
    off, tok, child = t.child_off.tolist(), t.child_tok.tolist(), t.child_node.tolist()
    seen = 0
    stack = [(root, 0)]
    while stack:
        nd, i = stack.pop()
        seen += 1
        kids = sorted(nd.keys())
        assert tok[off[i]:off[i + 1]] == kids
        for e, k in zip(range(off[i], off[i + 1]), kids):
            stack.append((nd[k], child[e]))
    assert seen == t.n_nodes
    assert TrieCSR.build(valid.view(100, 3, 3)).child_tok.tolist() == tok          # (B, T, C) input, tiger.py:58-60


def test_t5_attention_oracle_vs_reference_golden(golden):
    """oracle/t5_attention.py reproduces the unmodified reference's T5Attention (outputs, every gradient) exactly, and the bucket map of
    the product's host code equals the reference formula (transformer.py:13-41)."""
    from oracle import t5_attention as ot
    from genrec_b200.t5_attention import relative_position_buckets
    g = golden("t5_attention.pt")
    for name, c in g["cases"].items():
        x = c["x"].clone().requires_grad_(True)
        sd = {k: v.clone().requires_grad_(True) for k, v in c["state_dict"].items()}
        ctx = c["ctx"].clone().requires_grad_(True) if c["cross"] else None
        mask = torch.nn.Transformer.generate_square_subsequent_mask(x.shape[1]) if c["causal"] else None
        out = ot.t5_attention_forward(x, ctx, ctx, sd, c["heads"], c["cross"], mask, c["pad"])
        out.backward(c["dy"])
        assert torch.equal(out, c["out"]) and torch.equal(x.grad, c["dx"]), name
        for k in sd:
            assert torch.equal(sd[k].grad, c["grads"][k]), (name, k)
    for lq, lk in ((37, 37), (9, 21), (200, 300), (1, 5)):
        i = torch.arange(lq)[:, None]; j = torch.arange(lk)[None, :]
        assert torch.equal(ot.bucket_of(j - i), relative_position_buckets(lq, lk).long()[(j - i) + lq - 1])


def test_trie_csr_edge_shapes():
    """One item, a 1-D item, items sharing every prefix: node and edge counts of the CSR trie (tiger.py:49-69 semantics)."""
    from genrec_b200.tiger_decode import TrieCSR
    t = TrieCSR.build(torch.tensor([4, 2, 9]))                       # 1-D: one sequence (tiger.py:61-62)
    assert t.n_nodes == 4 and t.child_tok.tolist() == [4, 2, 9] and t.child_off.tolist() == [0, 1, 2, 3, 3]
    t = TrieCSR.build(torch.tensor([[1, 1, 1], [1, 1, 1], [1, 1, 2]]))
    assert t.n_nodes == 5 and t.child_off.tolist() == [0, 1, 2, 4, 4, 4] and t.child_tok.tolist() == [1, 1, 1, 2]
    t = TrieCSR.build(torch.tensor([[0, 5], [3, 5], [0, 4]]))
    assert t.child_tok.tolist() == [0, 3, 4, 5, 5] and t.child_node.tolist() == [1, 2, 3, 4, 5]
