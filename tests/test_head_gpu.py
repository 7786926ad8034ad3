"""Fused tied-embedding cross-entropy head (genrec/models/hstu.py:137-146) against a plain fp32 torch restatement of the same lines:
loss, d loss / d x, the tied-table gradient and the final-LayerNorm gradients, over every D the kernels are compiled for, ragged token /
class counts (partial tiles on both axes, a single class tile, class halves of unequal length) and ignored rows (target 0)."""
import os
import subprocess
import sys

import pytest
import torch

from tests.util import relerr

pytestmark = pytest.mark.gpu


def _case(B, L, D, C, seed, frac_ignored=0.3):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, L, D, generator=g)
    ln_g = 1 + 0.1 * torch.randn(D, generator=g)
    ln_b = 0.1 * torch.randn(D, generator=g)
    table = 0.5 * torch.randn(C, D, generator=g)
    tg = torch.randint(1, C, (B, L), generator=g)
    tg[torch.rand(B, L, generator=g) < frac_ignored] = 0
    tg[0, :] = 0                                    # one fully ignored sequence
    return x, ln_g, ln_b, table, tg


def _reference(x, ln_g, ln_b, table, tg):
    x = x.clone().requires_grad_(True); ln_g = ln_g.clone().requires_grad_(True); ln_b = ln_b.clone().requires_grad_(True)
    table = table.clone().requires_grad_(True)
    xf = torch.nn.functional.layer_norm(x, (x.shape[-1],), ln_g, ln_b, 1e-5)
    # the product path rounds LN(x) and the table to bf16 before the logits GEMM (as the reference's autocast does)
    logits = xf @ table.t()
    loss = torch.nn.functional.cross_entropy(logits.view(-1, table.shape[0]), tg.view(-1), ignore_index=0)
    loss.backward()
    return loss.detach(), x.grad, ln_g.grad, ln_b.grad, table.grad


def _ours(x, ln_g, ln_b, table, tg):
    from genrec_b200 import functional as Fn
    dev = torch.device("cuda:0")
    x = x.to(dev).requires_grad_(True); ln_g = ln_g.to(dev).requires_grad_(True); ln_b = ln_b.to(dev).requires_grad_(True)
    table = table.to(dev).requires_grad_(True)
    tb = Fn.cast_bf16(table.detach())
    loss = Fn.HeadLossFn.apply(x, ln_g, ln_b, table, tb, tg.to(dev), 1e-5)
    loss.backward()
    torch.cuda.synchronize()
    return loss.detach().cpu(), x.grad.cpu(), ln_g.grad.cpu(), ln_b.grad.cpu(), table.grad.cpu()


SHAPES = [(3, 50, 64, 97), (2, 200, 128, 1203), (5, 77, 128, 12102), (2, 130, 256, 1000), (2, 64, 128, 128), (4, 64, 64, 129)]


@pytest.mark.parametrize("B,L,D,C", SHAPES)
def test_head_loss_and_gradients_vs_torch_fp32(B, L, D, C):
    case = _case(B, L, D, C, seed=B * 1000 + C)
    ref = _reference(*case)
    got = _ours(*case)
    assert abs(got[0].item() - ref[0].item()) < 2e-3 * abs(ref[0].item()) + 1e-4, (got[0].item(), ref[0].item())
    for name, a, b in zip(("dx", "dln_g", "dln_b", "dtable"), got[1:], ref[1:]):
        assert torch.isfinite(a).all(), name
        assert relerr(a, b) < 2e-2, (name, relerr(a, b))
    # ignored rows receive no gradient at all, and row 0 of the table only what the softmax sends there
    assert got[1][0].abs().max() == 0


def test_head_all_rows_ignored_is_nan_like_the_reference():
    x, ln_g, ln_b, table, tg = _case(2, 16, 128, 300, seed=1)
    tg[:] = 0
    got = _ours(x, ln_g, ln_b, table, tg)
    assert torch.isnan(got[0])                       # F.cross_entropy: 0 / 0 valid targets (hstu.py:141-146)


def test_head_schedules_agree(tmp_path):
    """GRB_CE=store keeps the G' tensor and the TN GEMM for dE (the only schedule at D = 256); GRB_CE=exact is the two-sweep kernel without
    any [T, C] tensor; the default is the one-sweep kernel.  All three must agree at D = 128."""
    code = (
        "import torch, sys; sys.path.insert(0, %r)\n"
        "from tests.test_head_gpu import _case, _ours\n"
        "out = _ours(*_case(3, 90, 128, 2500, seed=9))\n"
        "torch.save(out, sys.argv[1])\n" % os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    outs = []
    for mode in ("store", "exact", ""):
        path = str(tmp_path / f"head_{mode or 'default'}.pt")
        env = dict(os.environ, GRB_CE=mode)
        if not mode:
            env.pop("GRB_CE")
        subprocess.run([sys.executable, "-c", code, path], check=True, env=env, timeout=300)
        outs.append(torch.load(path))
    for other in outs[1:]:
        assert abs(outs[0][0].item() - other[0].item()) < 1e-5
        for a, b in zip(outs[0][1:], other[1:]):
            assert relerr(a, b) < 1e-2, relerr(a, b)


def test_head_wide_logit_range():
    """Logits spread over +-60 nats, the target far from the row maximum for most rows: the one-sweep kernel's shift (probe tile / target
    logit) sits well below the true maximum and the result must still be the exact softmax."""
    g = torch.Generator().manual_seed(4)
    x, ln_g, ln_b, table, tg = _case(3, 70, 128, 3000, seed=21)
    table = table * 3.0                                   # |logit| up to ~ 60
    table[2000:2100] *= 1.6                               # the largest logits live far from the probe tile (classes 0..127)
    ref = _reference(x, ln_g, ln_b, table, tg)
    got = _ours(x, ln_g, ln_b, table, tg)
    assert torch.isfinite(got[0]) and abs(got[0].item() - ref[0].item()) < 3e-3 * abs(ref[0].item()), (got[0].item(), ref[0].item())
    for name, a, b in zip(("dx", "dln_g", "dln_b", "dtable"), got[1:], ref[1:]):
        assert torch.isfinite(a).all(), name
        assert relerr(a, b) < 3e-2, (name, relerr(a, b))


def _overflow_case():
    """Every row's logit for class 2500 sits ~190 nats above everything else (LayerNorm bias = 1 along a table row of 1.5s), far from
    the probe tile (classes 0..127) and - for all but a handful of rows - not the target."""
    x, ln_g, ln_b, table, tg = _case(2, 40, 128, 3000, seed=33, frac_ignored=0.0)
    ln_g = torch.ones(128); ln_b = torch.ones(128)
    table = 0.01 * table
    table[2500] = 1.5
    tg[tg == 2500] = 7
    return x, ln_g, ln_b, table, tg


def test_one_sweep_range_limit_is_loud_and_exact_mode_has_none(tmp_path):
    """DESIGN 3.3: the one-sweep kernel's exponent shift is max(probe tile, target logit); a class beating both by more than ~98 nats
    overflows that row - the loss comes out non-finite, never silently wrong - and GRB_CE=exact computes the same case exactly."""
    code = (
        "import torch, sys; sys.path.insert(0, %r)\n"
        "from tests.test_head_gpu import _overflow_case, _ours\n"
        "out = _ours(*_overflow_case())\n"
        "torch.save(out, sys.argv[1])\n" % os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    res = {}
    for mode in ("", "exact"):
        path = str(tmp_path / f"head_overflow_{mode or 'default'}.pt")
        env = dict(os.environ, GRB_CE=mode)
        if not mode:
            env.pop("GRB_CE")
        subprocess.run([sys.executable, "-c", code, path], check=True, env=env, timeout=300)
        res[mode] = torch.load(path)
    assert not torch.isfinite(res[""][0])                            # loud
    ref = _reference(*_overflow_case())
    got = res["exact"]
    assert torch.isfinite(got[0]) and abs(got[0].item() - ref[0].item()) < 2e-3 * abs(ref[0].item())
    assert relerr(got[1], ref[1]) < 3e-2 and relerr(got[4], ref[4]) < 3e-2
