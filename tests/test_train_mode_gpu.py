"""Training mode against fp64 references: dropout through every kernel that applies or re-derives a mask, and the fused Adam step.

The dropout masks are restated on the host (tests/util.py ``drop_mask``) at each kernel's own addressing and fed to the oracle
through its ``drop`` hook, so a backward kernel that addresses its mask differently from its forward, a mask applied one op early
or late, a wrong keep scale or an ignored device seed counter all show up as a parity failure.
"""
import math

import numpy as np
import pytest
import torch

from tests.util import frob_relerr, keep_scale, make_batch, relerr

pytestmark = pytest.mark.gpu

SITE_GATE, SITE_FFN_HID, SITE_FFN_OUT, SITE_ATTN, SITE_EMBED = 0, 1, 2, 3, 250    # csrc/api.cu; a layer's site is layer * 8 + which
HSTU_SITE = {"gate": SITE_GATE, "ffn_hid": SITE_FFN_HID, "ffn_out": SITE_FFN_OUT}
# (seed, device counter): a seed below 2^32 and no counter; a seed just under 2^32 whose sum with the counter carries into the high word
SEEDS = {"lo": (0x5EED1234, None), "carry": (0xFFFFFFF0, 3 * 0x9E3779B1)}


def _seed_dev(sd, dev):
    return None if sd is None else torch.tensor([sd], dtype=torch.int64, device=dev)


# ------------------------------------------------------------------------------------------------ HSTU block
def _hstu_drop(B, L, p, seed, sd, layer, wrong=None):
    """The oracle's drop hook for one block: every site masked as the kernels address it (row = token, column = feature).
    ``wrong`` names a site whose mask is drawn from seed + 1 instead (negative control)."""
    def drop(name, t):
        which = name.rsplit(".", 1)[-1]
        s = seed + (1 if which == wrong else 0)
        m = keep_scale(range(B * L), range(t.shape[-1]), p, s, layer * 8 + HSTU_SITE[which], sd)
        return t * m.view(B, L, -1).to(t.dtype)
    return drop


def _hstu_block_case(B, L, D, H, p, layer_index, seed_kind, wrong=None):
    """-> list of (tensor name, relative error vs the fp64 oracle, bound of test_hstu_gpu.py::test_layer_vs_oracle_shapes)."""
    from genrec_b200.hstu import HSTULayer
    from oracle import hstu as oh
    dev = torch.device("cuda:0")
    torch.manual_seed(L * 131 + D + layer_index)
    layer = HSTULayer(D, H, p, 32, 64, 128, True)
    layer.layer_index = layer_index
    with torch.no_grad():
        for n, q in layer.named_parameters():
            if "attention_bias" in n:
                q.normal_(0, 0.5)
            elif n.endswith("bias"):
                q.normal_(0, 0.1)
            elif "norm" in n:
                q.add_(0.1 * torch.randn_like(q))
            else:
                q.normal_(0, 0.08)
    ids, ts, _ = make_batch(3, L, 50, seed=L)          # row 1 left-padded, row 2 fully padded
    if B == 2:
        ids, ts = ids[1:], ts[1:]
    elif B > 3:
        ids2, ts2, _ = make_batch(B - 3, L, 50, seed=L + 1, pad=False)
        ids, ts = torch.cat([ids, ids2]), torch.cat([ts, ts2])
    x = torch.randn(B, L, D)
    dy = torch.randn(B, L, D)
    seed, sd = SEEDS[seed_kind]
    sd64 = {k: v.detach().double().requires_grad_(True) for k, v in layer.state_dict().items()}
    xo = x.double().requires_grad_(True)
    yo = oh.hstu_layer_forward(xo, ids == 0, ts, sd64, "", H, drop=_hstu_drop(B, L, p, seed, sd, layer_index, wrong))
    yo.backward(dy.double())
    layer = layer.to(dev).train()
    xg = x.to(dev).requires_grad_(True)
    yg = layer(xg, None, (ids == 0).to(dev), ts.to(dev), _seed=seed, _seed_dev=_seed_dev(sd, dev))
    yg.backward(dy.to(dev))
    rows = [("y", relerr(yg, yo), 2.5e-2), ("dx", relerr(xg.grad, xo.grad), 2.5e-2)]
    rows += [(n, relerr(q.grad, sd64[n].grad), 4e-2) for n, q in layer.named_parameters()]
    return rows


@pytest.mark.parametrize("seed_kind", ["lo", "carry"])
@pytest.mark.parametrize("layer_index", [0, 3])
@pytest.mark.parametrize("p", [0.2, 0.5])
@pytest.mark.parametrize("B,L,D,H", [(3, 50, 128, 4), (4, 200, 128, 4), (2, 300, 128, 4), (2, 130, 256, 8)])
def test_hstu_block_dropout_vs_oracle_fp64(B, L, D, H, p, layer_index, seed_kind):
    """One block in training mode (gate, FFN hidden and FFN output dropout) against the fp64 oracle with the same masks: y, dx and
    every parameter gradient.  L = 200 runs the mma.sync attention kernels, L = 300 the tcgen05 ones."""
    bad = [r for r in _hstu_block_case(B, L, D, H, p, layer_index, seed_kind) if not r[1] < r[2]]
    assert not bad, bad


def test_hstu_block_dropout_negative_control():
    """The comparison above can see a wrong mask: with the FFN hidden mask drawn from seed + 1 in the oracle, the worst tensor
    misses its bound by far more than 5x (measured on a B200 at 1000 W: 25.5x, on the hidden-layer bias gradient)."""
    rows = _hstu_block_case(3, 50, 128, 4, 0.2, 3, "carry", wrong="ffn_hid")
    worst = max(rows, key=lambda r: r[1] / r[2])
    print("negative control, HSTU block:", worst, f"margin {worst[1] / worst[2]:.1f}x")
    assert worst[1] >= 5 * worst[2], worst


# ------------------------------------------------------------------------------------------------ SASRec attention core
def _sasrec_core_case(L, dh, wrong=False):
    import genrec_b200.functional as Fn
    dev = torch.device("cuda:0")
    B, H, p, layer = 4, 2, 0.3, 2
    D = H * dh
    g = torch.Generator().manual_seed(L * 5 + dh)
    q, k, v = [(torch.randn(B, L, D, generator=g)).to(torch.bfloat16) for _ in range(3)]
    dout = torch.randn(B, L, D, generator=g).to(torch.bfloat16)
    pad = torch.zeros(B, L, dtype=torch.bool)
    pad[1, : L // 3] = True                       # left padding
    pad[2, 3::7] = True                           # scattered padded queries and keys
    pad[3, :] = True                              # fully padded sequence
    seed, sd = SEEDS["carry"]
    out, lse = Fn.sasrec_attention_fwd(q.to(dev), k.to(dev), v.to(dev), pad.to(torch.uint8).to(dev), H, p, seed, _seed_dev(sd, dev), layer)
    dq, dk, dv = Fn.sasrec_attention_bwd(q.to(dev), k.to(dev), v.to(dev), pad.to(torch.uint8).to(dev), out, lse, dout.to(dev), H, p, seed,
                                         _seed_dev(sd, dev), layer)
    # fp64 restatement of sasrec.py:206-240 on the same bf16 operands; the attention-weight mask is addressed by
    # row (b * H + h) * L + i, column j in all three kernels
    keep = keep_scale(range(B * H * L), range(L), p, seed + (1 if wrong else 0), layer * 8 + SITE_ATTN, sd).view(B, H, L, L)
    Q, K, V = [t.double().view(B, L, H, dh).transpose(1, 2).requires_grad_(True) for t in (q, k, v)]
    S = (Q @ K.transpose(-2, -1)) * dh ** -0.5
    S = S.masked_fill(pad[:, None, None, :], -1e9)
    S = S.masked_fill(torch.triu(torch.ones(L, L, dtype=torch.bool), diagonal=1), -1e9)
    A = torch.softmax(S, -1) * (~pad).double()[:, None, :, None]
    O = ((A * keep) @ V).transpose(1, 2).reshape(B, L, D)
    O.backward(dout.double())
    grad = lambda t: t.grad.transpose(1, 2).reshape(B, L, D)
    valid = ~pad
    assert out.float()[pad.to(dev)].abs().max() == 0 if pad.any() else True
    return [("out", relerr(out.float().cpu()[valid], O.detach()[valid]), 8e-3), ("dq", relerr(dq, grad(Q)), 1.5e-2),
            ("dk", relerr(dk, grad(K)), 1.5e-2), ("dv", relerr(dv, grad(V)), 1.5e-2)]


@pytest.mark.parametrize("dh", [32, 64])
@pytest.mark.parametrize("L", [1, 50, 64, 65, 130, 200])
def test_sasrec_attention_core_dropout_vs_fp64(L, dh):
    """Fn.sasrec_attention_fwd / _bwd with attention-weight dropout p = 0.3 (seed carrying into the high word, layer 2) against an
    fp64 restatement with the same mask, within the bounds of test_attn_tc_gpu.py::test_attention_core_vs_torch_fp32."""
    bad = [r for r in _sasrec_core_case(L, dh) if not r[1] < r[2]]
    assert not bad, bad


def test_sasrec_attention_core_dropout_negative_control():
    """With the reference's attention mask drawn from seed + 1 the worst tensor misses its bound by more than 5x (measured on a
    B200 at 1000 W: 131x, on out)."""
    rows = _sasrec_core_case(130, 64, wrong=True)
    worst = max(rows, key=lambda r: r[1] / r[2])
    print("negative control, SASRec attention core:", worst, f"margin {worst[1] / worst[2]:.1f}x")
    assert worst[1] >= 5 * worst[2], worst


# ------------------------------------------------------------------------------------------------ whole models at dropout 0.2
def _yardstick(rows, small):
    """The cfg-2 rule of test_cfg2_parity_gpu.py: rows = (name, ours Frobenius, reference autocast Frobenius, ours max-norm, reference
    autocast max-norm) against the fp32 oracle run with the same masks."""
    for r in rows:
        print(f"| {r[0]} | {r[1]:.2e} | {r[2]:.2e} | {r[1] / max(r[2], 1e-12):.2f} | {r[3]:.2e} | {r[4]:.2e} |")
    big_r = [a / b for n, a, b, c, d in rows if n not in small and n != "loss" and b > 0]
    small_r = [a / b for n, a, b, c, d in rows if n in small and b > 0]
    gm = lambda v: math.exp(sum(math.log(max(x, 1e-6)) for x in v) / max(len(v), 1))
    print(f"geometric mean of ours / reference-autocast: matrices {gm(big_r):.3f} ({len(big_r)}), small vectors {gm(small_r):.3f}")
    bad = [r for r in rows if r[1] > (3.0 if r[0] in small else 1.1) * r[2] + 5e-4 or r[3] > 3.0 * r[4] + 1e-3]
    assert not bad, bad
    assert gm(big_r) <= 1.0 and gm(small_r) <= 1.25, (gm(big_r), gm(small_r))


def _compare_grads(rows, small, named_params, gref, gac):
    for n, q in named_params:
        ref = gref[n]
        got = q.grad if q.grad is not None else torch.zeros_like(q)
        if ref.abs().max() == 0:
            assert got.abs().max() == 0, n
            continue
        rows.append((n + ".grad", frob_relerr(got, ref), frob_relerr(gac[n], ref), relerr(got, ref), relerr(gac[n], ref)))
        if ref.numel() < 4096:
            small.add(n + ".grad")


def _oracle_grads(forward, sd, spy_module, spy_name, spy_prefix_arg, prefix, autocast):
    """forward(p) -> loss with the oracle; returns the loss, every parameter gradient and the gradient entering block ``prefix``."""
    p = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    grabbed = {}
    orig = getattr(spy_module, spy_name)

    def spy(x, *a, **kw):
        if a[spy_prefix_arg] == prefix:
            x.retain_grad(); grabbed["x"] = x
        return orig(x, *a, **kw)

    setattr(spy_module, spy_name, spy)
    try:
        if autocast:
            with torch.autocast("cpu", dtype=torch.bfloat16):
                lo = forward(p)
        else:
            lo = forward(p)
        lo.float().backward()
    finally:
        setattr(spy_module, spy_name, orig)
    return float(lo), {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in p.items()}, grabbed["x"].grad.float()


def _patch_seeds(m, seed, sd):
    m._seeds = lambda device: (seed, _seed_dev(sd, device))


def test_hstu_cfg2_model_dropout_vs_oracle():
    """The headline HSTU configuration (4 blocks, d = 128, h = 4, L = 200, V = 12,101; B = 8 as in test_cfg2_full_model_vs_oracle) in
    training mode at dropout 0.2: loss, dX into the last block and every gradient against the fp32 oracle with the same embedding,
    gate and FFN masks, held to the oracle's own bf16-autocast error with those masks."""
    from oracle import hstu as oh
    from tests.test_cfg2_parity_gpu import H, L, NB, V, _cfg2_model
    dev = torch.device("cuda:0")
    B, p = 8, 0.2
    seed, sd = SEEDS["carry"]
    m = _cfg2_model(dropout=p)
    state = {k: v.clone() for k, v in m.state_dict().items()}
    ids, ts, tg = make_batch(B, L, V, seed=5, pad=True)
    ids[3, :57] = 0; ts[3, :57] = 0; tg[3, :56] = 0
    T = B * L
    masks = {}

    def drop(name, t):
        if name not in masks:
            if name == "emb":
                site = SITE_EMBED
            else:
                i, which = name.split(".")[1:]
                site = int(i) * 8 + HSTU_SITE[which]
            masks[name] = keep_scale(range(T), range(t.shape[-1]), p, seed, site, sd, torch.float32).view(B, L, -1)
        return t * masks[name].to(t.dtype)

    fwd = lambda q: oh.hstu_forward(ids, ts, tg, q, H, NB, drop=drop)[1]
    lo, gref, dxref = _oracle_grads(fwd, state, oh, "hstu_layer_forward", 3, f"layers.{NB - 1}.", False)
    la, gac, dxac = _oracle_grads(fwd, state, oh, "hstu_layer_forward", 3, f"layers.{NB - 1}.", True)
    m = m.to(dev).train()
    _patch_seeds(m, seed, sd)
    got = {}
    hook = m.layers[NB - 1].register_forward_pre_hook(lambda mod, args: args[0].register_hook(lambda g: got.__setitem__("dx", g.clone())) and None)
    _, loss = m(ids.to(dev), ts.to(dev), tg.to(dev))
    loss.backward()
    hook.remove()
    el, ea = abs(loss.item() - lo) / abs(lo), abs(la - lo) / abs(lo)
    rows = [("loss", el, ea, el, ea),
            ("dX into the last block", frob_relerr(got["dx"], dxref), frob_relerr(dxac, dxref), relerr(got["dx"], dxref), relerr(dxac, dxref))]
    small = set()
    _compare_grads(rows, small, m.named_parameters(), gref, gac)
    _yardstick(rows, small)


def test_sasrec_cfg1_model_dropout_vs_oracle():
    """SASRec at the cfg-1 shape (B = 128, L = 50, d = 64, 2 blocks, 1k items) in training mode at dropout 0.2: loss, dX into the
    last block and every gradient against the fp32 oracle with the same embedding, attention-weight and FFN masks; same yardstick as
    the HSTU model above."""
    from genrec_b200.sasrec import SASRec
    from oracle import sasrec as osr
    dev = torch.device("cuda:0")
    B, L, D, H, NB, Fd, V, p = 128, 50, 64, 2, 2, 256, 1000, 0.2
    seed, sd = SEEDS["lo"]
    torch.manual_seed(L + D)
    m = SASRec(V, L, D, H, NB, Fd, dropout=p)
    g = torch.Generator().manual_seed(3)
    with torch.no_grad():
        for n, q in m.named_parameters():
            if n.endswith("bias"):
                q.copy_(0.1 * torch.randn(q.shape, generator=g))
            elif "norm" in n:
                q.add_(0.1 * torch.randn(q.shape, generator=g))
    state = {k: v.clone() for k, v in m.state_dict().items()}
    ids, _, tg = make_batch(B, L, V, seed=L)
    T = B * L
    masks = {}

    def drop(name, t):
        if name not in masks:
            if name == "emb":
                mk = keep_scale(range(T), range(D), p, seed, SITE_EMBED, sd, torch.float32).view(B, L, D)
            else:
                _, i, which = name.split(".")
                if which == "attn":
                    mk = keep_scale(range(B * H * L), range(L), p, seed, int(i) * 8 + SITE_ATTN, sd, torch.float32).view(B, H, L, L)
                else:
                    mk = keep_scale(range(T), range(t.shape[-1]), p, seed, int(i) * 8 + HSTU_SITE[which], sd, torch.float32).view(B, L, -1)
            masks[name] = mk
        return t * masks[name].to(t.dtype)

    fwd = lambda q: osr.sasrec_forward(ids, tg, q, H, NB, drop=drop)[1]
    lo, gref, dxref = _oracle_grads(fwd, state, osr, "sasrec_block_forward", 2, f"blocks.{NB - 1}.", False)
    la, gac, dxac = _oracle_grads(fwd, state, osr, "sasrec_block_forward", 2, f"blocks.{NB - 1}.", True)
    assert sorted(masks) == sorted(["emb"] + [f"blocks.{i}.{w}" for i in range(NB) for w in ("attn", "ffn_hid", "ffn_out")])
    m = m.to(dev).train()
    _patch_seeds(m, seed, sd)
    got = {}
    hook = m.blocks[NB - 1].register_forward_pre_hook(lambda mod, args: args[0].register_hook(lambda g: got.__setitem__("dx", g.clone())) and None)
    _, loss = m(ids.to(dev), tg.to(dev))
    loss.backward()
    hook.remove()
    el, ea = abs(loss.item() - lo) / abs(lo), abs(la - lo) / abs(lo)
    rows = [("loss", el, ea, el, ea),
            ("dX into the last block", frob_relerr(got["dx"], dxref), frob_relerr(dxac, dxref), relerr(got["dx"], dxref), relerr(dxac, dxref))]
    small = set()
    # the key-projection bias has an analytically zero gradient under the softmax: both sides are rounding noise
    _compare_grads(rows, small, [(n, q) for n, q in m.named_parameters() if not n.endswith("k_proj.bias")], gref, gac)
    _yardstick(rows, small)


# ------------------------------------------------------------------------------------------------ Adam
def adam_ref_step(p, g, m, v, step, lr, beta1, beta2, eps, weight_decay):
    """torch.optim.Adam's single-tensor step (amsgrad = maximize = False), in place, in whatever dtype the tensors carry."""
    if weight_decay != 0:
        g = g + weight_decay * p
    m.lerp_(g, 1 - beta1)
    v.mul_(beta2).addcmul_(g, g, value=1 - beta2)
    bc1, bc2 = 1 - beta1 ** step, 1 - beta2 ** step
    denom = (v.sqrt() / math.sqrt(bc2)).add_(eps)
    p.addcdiv_(m, denom, value=-lr / bc1)


ADAM_CFGS = {"default": (1e-3, (0.9, 0.999), 1e-8, 0.0, 1.0), "wd": (3e-3, (0.9, 0.98), 1e-8, 1e-2, 1.0),
             "scaled": (1e-2, (0.8, 0.99), 1e-6, 0.0, 0.125)}


@pytest.mark.parametrize("cfg", list(ADAM_CFGS))
def test_adam_restatement_is_torch_adam(cfg):
    """The restatement the kernel is checked against is torch.optim.Adam(foreach=False) in fp64."""
    lr, betas, eps, wd, _ = ADAM_CFGS[cfg]
    g = torch.Generator().manual_seed(1)
    p0 = torch.randn(300, generator=g, dtype=torch.float64)
    tp = p0.clone().requires_grad_(True)
    opt = torch.optim.Adam([tp], lr=lr, betas=betas, eps=eps, weight_decay=wd, foreach=False)
    p, m, v = p0.clone(), torch.zeros_like(p0), torch.zeros_like(p0)
    for k in range(1, 31):
        gr = torch.randn(300, generator=g, dtype=torch.float64) * 10 ** (6 * torch.rand(300, generator=g, dtype=torch.float64) - 4)
        tp.grad = gr.clone()
        opt.step()
        adam_ref_step(p, gr, m, v, k, lr, betas[0], betas[1], eps, wd)
        torch.testing.assert_close(p, tp.detach(), rtol=1e-13, atol=1e-15)


def _grads(n, k, gen, dev):
    """Heavy-tailed magnitudes (1e-5 .. 1e3, Cauchy-like), exact zeros, constant-sign elements, and a block that is zero on some steps."""
    mag = 10 ** (8 * torch.rand(n, generator=gen, device=dev) - 5)
    sign = torch.where(torch.rand(n, generator=gen, device=dev) < 0.5, -1.0, 1.0)
    cls = torch.arange(n, device=dev) % 5
    g = sign * mag
    g = torch.where(cls == 1, torch.zeros_like(g), g)                  # always zero
    g = torch.where(cls == 2, mag, g)                                  # constant sign
    if k % 4 == 0:
        g = torch.where(cls == 3, torch.zeros_like(g), g)              # intermittently zero
    return g.float()


@pytest.mark.parametrize("n", [1, 255, 257, 2 * 148 * 16 * 256 + 7])
@pytest.mark.parametrize("cfg", list(ADAM_CFGS))
def test_adam_step_vs_torch_adam_fp64(cfg, n):
    """Fn.adam_step over 100 steps against the fp64 restatement of torch.optim.Adam, with the hyperparameters as the float32 values the C
    ABI receives.  Every step: the device (step, 1 - beta1^step, 1 - beta2^step) triple against double; p, m and v against one fp64 step
    from the kernel's own previous state (so one step's error cannot hide in the accumulated rounding); p against an independent fp64
    run, |dp| <= 1e-5 lr k + 2^-22 max|p| sqrt(k) (the second term: the float32 rounding of p, a random walk over k steps); the bf16
    mirror equal to p.bfloat16() bit for bit, or untouched when it is None; the gradient zeroed or kept as asked.
    n = 2 * 148 * 16 * 256 + 7 exceeds one pass of the grid (sm_count * 16 blocks of 256 threads) on a B200."""
    import genrec_b200.functional as Fn
    dev = torch.device("cuda:0")
    lr, (b1, b2), eps, wd, gs = ADAM_CFGS[cfg]
    f = lambda x: float(np.float32(x))
    lr32, b132, b232, eps32, wd32 = f(lr), f(b1), f(b2), f(eps), f(wd)
    gen = torch.Generator(device=dev).manual_seed(n + len(cfg))
    p = torch.randn(n, generator=gen, device=dev)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    mirror = torch.zeros(n, dtype=torch.bfloat16, device=dev)
    state = torch.zeros(4, dtype=torch.float32, device=dev)
    pr, mr, vr = p.double(), torch.zeros_like(p, dtype=torch.float64), torch.zeros_like(p, dtype=torch.float64)
    pmax = p.abs().max().item()
    for k in range(1, 101):
        g = _grads(n, k, gen, dev)
        gk = g.clone()
        zero_grad, with_mirror = k % 2 == 1, k % 3 != 0
        p_prev, m_prev, v_prev, mirror0 = p.double(), m.double(), v.double(), mirror.clone()
        Fn.adam_step(p, gk, m, v, mirror if with_mirror else None, state, lr, b1, b2, eps, wd, gs, zero_grad)
        st = state.double().cpu()
        assert st[0].item() == k
        for j, b in ((1, b132), (2, b232)):
            want = 1 - b ** k
            assert abs(st[j].item() - want) <= 2 ** -23 * want, (k, j, st[j].item(), want)
        # one fp64 step from the kernel's previous state
        ge = g.double() * gs
        p0, m0, v0 = p_prev.clone(), m_prev.clone(), v_prev.clone()
        adam_ref_step(p0, ge, m0, v0, k, lr32, b132, b232, eps32, wd32)
        # rounding scales: the weight-decay term can cancel the gradient, so they use |g| + |wd p|
        gabs = ge.abs() + wd32 * p_prev.abs()
        mscale = b132 * m_prev.abs() + (1 - b132) * gabs
        vscale = b232 * v_prev + (1 - b232) * gabs * gabs
        assert ((m.double() - m0).abs() <= 2 ** -21 * mscale + 1e-30).all(), (k, (m.double() - m0).abs().max().item())
        assert ((v.double() - v0).abs() <= 2 ** -21 * vscale + 1e-30).all(), (k, (v.double() - v0).abs().max().item())
        dp1 = (p.double() - p0).abs()
        assert (dp1 <= 1e-5 * lr + 2 ** -23 * p0.abs()).all(), (k, dp1.max().item())
        # an independent fp64 run
        adam_ref_step(pr, ge, mr, vr, k, lr32, b132, b232, eps32, wd32)
        dp = (p.double() - pr).abs().max().item()
        assert dp <= 1e-5 * lr * k + 2 ** -22 * pmax * math.sqrt(k), (k, dp)
        if with_mirror:
            assert torch.equal(mirror, p.bfloat16())
        else:
            assert torch.equal(mirror, mirror0)
        assert torch.equal(gk, torch.zeros_like(g)) if zero_grad else torch.equal(gk, g)


def test_flat_adam_matches_torch_adam_and_resumes_bit_for_bit():
    """FlatAdam on a plain multi-layer module with odd parameter sizes against torch.optim.Adam (fp64) on a twin fed the same
    gradients, with the learning rate changed mid-run; a state_dict round trip mid-run continues bit-identically to the
    uninterrupted run; the padding slots of the flat buffers stay exactly 0.  The hyperparameters are powers of two, so the float32
    values the kernel receives are the twin's."""
    import copy
    from genrec_b200.optim import FlatAdam
    dev = torch.device("cuda:0")
    lr0, lr1, betas, eps, wd = 2 ** -9, 2 ** -11, (0.875, 1 - 2 ** -7), 2 ** -27, 2 ** -7

    def net():
        torch.manual_seed(0)
        mod = torch.nn.Sequential(torch.nn.Linear(37, 61), torch.nn.Tanh(), torch.nn.Linear(61, 5), torch.nn.Linear(5, 3, bias=False))
        mod.register_parameter("odd", torch.nn.Parameter(torch.randn(3, 7)))
        return mod

    g = torch.Generator().manual_seed(2)
    grads = [[torch.randn(q.shape, generator=g) * 10 ** (4 * torch.rand(q.shape, generator=g) - 2) for q in net().parameters()]
             for _ in range(30)]
    twin = copy.deepcopy(net()).double()
    topt = torch.optim.Adam(twin.parameters(), lr=lr0, betas=betas, eps=eps, weight_decay=wd, foreach=False)

    def run(model, opt, steps, twin_too=False):
        for k in steps:
            if k == 15:
                opt.lr = lr1
                if twin_too:
                    topt.param_groups[0]["lr"] = lr1
            for q, gr in zip(model.parameters(), grads[k]):
                q.grad.copy_(gr)
            opt.step()
            if twin_too:
                for q, gr in zip(twin.parameters(), grads[k]):
                    q.grad = gr.double()
                topt.step()
                for (n, q), tq in zip(model.named_parameters(), twin.parameters()):
                    d = (q.detach().double().cpu() - tq.detach()).abs().max().item()
                    assert d <= 1e-5 * lr0 * (k + 1) + 2 ** -22 * tq.abs().max().item() * math.sqrt(k + 1), (k, n, d)

    m1 = net().to(dev)
    o1 = FlatAdam(m1, lr=lr0, betas=betas, eps=eps, weight_decay=wd)
    run(m1, o1, range(10), twin_too=True)
    ck_model = {k: v.clone() for k, v in m1.state_dict().items()}
    ck_opt = {k: (v.clone() if torch.is_tensor(v) else v) for k, v in o1.state_dict().items()}
    run(m1, o1, range(10, 30), twin_too=True)
    torch.cuda.synchronize()
    used = torch.zeros(o1.n, dtype=torch.bool)
    for q, o in zip(o1.params, o1.buffers.offsets):
        used[o:o + q.numel()] = True
    pad = ~used.to(dev)
    assert pad.any()
    for t in (o1.flat, o1.grad, o1.m, o1.v, o1.mirror.float()):
        assert t[pad].abs().max().item() == 0
    m2 = net().to(dev)
    o2 = FlatAdam(m2, lr=lr0, betas=betas, eps=eps, weight_decay=wd)
    m2.load_state_dict(ck_model)
    o2.load_state_dict(ck_opt)
    run(m2, o2, range(10, 30))
    for a, b in ((o2.flat, o1.flat), (o2.m, o1.m), (o2.v, o1.v), (o2.state, o1.state), (o2.mirror, o1.mirror)):
        assert torch.equal(a, b)
