"""GEMM building blocks through the C ABI (tcgen05/TMA kernels) vs torch."""
import pytest
import torch

from tests.util import drop_mask

pytestmark = pytest.mark.gpu


def _ref_linear(x, w, b):
    return x.float() @ w.float().T + b


@pytest.mark.parametrize("T,N,K", [(128, 128, 64), (210, 512, 128), (25600, 512, 128), (1000, 128, 512), (77, 64, 64), (300, 256, 1024)])
@pytest.mark.parametrize("act", [0, 1, 2])
def test_linear_forward(T, N, K, act):
    import genrec_b200.functional as Fn
    dev = torch.device("cuda:0")
    g = torch.Generator(device="cpu").manual_seed(T + N + K)
    x = torch.randn(T, K, generator=g).to(dev).bfloat16()
    w = (torch.randn(N, K, generator=g) * 0.1).to(dev).bfloat16()
    b = torch.randn(N, generator=g).to(dev)
    z, a = Fn.linear_fwd(x, w, b, act)
    ref = _ref_linear(x, w, b)
    torch.testing.assert_close(z.float(), ref, rtol=1e-2, atol=2e-2)
    if act == 1:
        torch.testing.assert_close(a.float(), torch.nn.functional.silu(z.float()), rtol=1e-2, atol=1e-2)
    if act == 2:
        torch.testing.assert_close(a.float(), torch.relu(z.float()), rtol=1e-2, atol=1e-2)


@pytest.mark.parametrize("T,N,K", [(128, 128, 128), (210, 512, 128), (25600, 512, 128), (25600, 128, 512), (77, 64, 64), (1000, 12102, 128)])
def test_linear_backward(T, N, K):
    import genrec_b200.functional as Fn
    dev = torch.device("cuda:0")
    g = torch.Generator(device="cpu").manual_seed(T + N + K + 1)
    dy = (torch.randn(T, N, generator=g) * 0.1).to(dev).bfloat16()
    if N % 8:
        pytest.skip("N must be a multiple of 8 for a contiguous bf16 operand")
    x = torch.randn(T, K, generator=g).to(dev).bfloat16()
    w = (torch.randn(N, K, generator=g) * 0.1).to(dev).bfloat16()
    res = torch.randn(T, K, generator=g).to(dev)
    dx, dw, db = Fn.linear_bwd(dy, w, x, dx_residual=res)
    torch.testing.assert_close(dx, res + dy.float() @ w.float(), rtol=1e-2, atol=1e-2 * (N ** 0.5) * 0.1)
    ref_dw = dy.float().T @ x.float()
    assert ((dw - ref_dw).abs().max() / ref_dw.abs().max()).item() < 2e-3
    ref_db = dy.float().sum(0)
    assert ((db - ref_db).abs().max() / ref_db.abs().max()).item() < 2e-3


def test_linear_residual_and_rowscale():
    import genrec_b200.functional as Fn
    dev = torch.device("cuda:0")
    g = torch.Generator(device="cpu").manual_seed(5)
    T, N, K = 333, 128, 512
    x = torch.randn(T, K, generator=g).to(dev).bfloat16()
    w = (torch.randn(N, K, generator=g) * 0.05).to(dev).bfloat16()
    b = torch.randn(N, generator=g).to(dev)
    res = torch.randn(T, N, generator=g).to(dev)
    rs = (torch.rand(T, generator=g) > 0.3).float().to(dev)
    y = Fn.linear_residual_fwd(x, w, b, res, rs)
    torch.testing.assert_close(y, (res + _ref_linear(x, w, b)) * rs[:, None], rtol=1e-2, atol=2e-2)


@pytest.mark.parametrize("p", [0.2, 0.5])
def test_dropout_masks_agree_between_forward_and_backward(p):
    """The backward kernels re-derive the forward dropout mask from (seed, site, row, column): the zero pattern of the
    forward output must equal the zero pattern the matching backward kernel applies, for every kernel pair that shares
    a site, and the realised drop rate must be p."""
    import genrec_b200.functional as Fn
    dev = torch.device("cuda:0")
    g = torch.Generator(device="cpu").manual_seed(11)
    T, K, N = 777, 128, 512
    seed, site = 1234567, 5
    x = torch.randn(T, K, generator=g).to(dev).bfloat16()
    w = (torch.randn(N, K, generator=g) * 0.1).to(dev).bfloat16()
    b = torch.randn(N, generator=g).to(dev)
    # hidden-activation dropout: forward GEMM epilogue vs the d-activation GEMM epilogue
    z, a = Fn.linear_fwd(x, w, b, 1, p=p, seed=seed, site=site)
    z0, a0 = Fn.linear_fwd(x, w, b, 1)
    assert torch.equal(z, z0)
    fwd_drop = (a == 0) & (a0 != 0)
    kept = (a != 0)
    torch.testing.assert_close(a[kept].float(), a0[kept].float() / (1 - p), rtol=2e-2, atol=1e-3)
    dyb = (torch.randn(T, K, generator=g).abs() + 0.5).to(dev).bfloat16()     # strictly positive
    wpos = (torch.rand(K, N, generator=g) + 0.1).to(dev).bfloat16()          # dy @ w > 0 everywhere
    gz = Fn.linear_dact_bwd(dyb, wpos, z.float().abs().add(0.5).bfloat16(), 1, p=p, seed=seed, site=site)   # silu'(z>0) > 0
    bwd_drop = gz == 0
    assert torch.equal(fwd_drop | (a0 == 0), bwd_drop | (a0 == 0))
    assert abs(bwd_drop.float().mean().item() - p) < 0.01
    # output dropout: residual GEMM epilogue vs the row cast kernel
    res = torch.zeros(T, K, device=dev)
    w2 = (torch.randn(K, N, generator=g) * 0.1).to(dev).bfloat16()
    b2 = (torch.rand(K, generator=g) + 5.0).to(dev)      # outputs far from zero
    y = Fn.linear_residual_fwd(a0, w2, b2, res, p=p, seed=seed, site=site + 1)
    c = Fn.cast_rows_bf16(torch.ones(T, K, device=dev), p=p, seed=seed, site=site + 1)
    assert torch.equal(y == 0, c == 0)
    assert abs((c == 0).float().mean().item() - p) < 0.01
    # a different site or seed gives a different mask
    c2 = Fn.cast_rows_bf16(torch.ones(T, K, device=dev), p=p, seed=seed, site=site + 2)
    c3 = Fn.cast_rows_bf16(torch.ones(T, K, device=dev), p=p, seed=seed + 1, site=site + 1)
    assert not torch.equal(c2 == 0, c == 0) and not torch.equal(c3 == 0, c == 0)
    # the mask is the documented pure function of (seed, site, row, column): bit-exact against the numpy restatement
    assert torch.equal((c == 0).cpu(), torch.from_numpy(drop_mask(range(T), range(K), p, seed, site + 1)))
    # rows and columns are decorrelated: cross-correlations are those of an ideal generator
    Tm, Dm = 512, 1024
    m = (Fn.cast_rows_bf16(torch.ones(Tm, Dm, device=dev), p=p, seed=seed, site=9) == 0).double()
    assert abs(m.mean().item() - p) < 0.005
    zc = (m - p) / (p * (1 - p)) ** 0.5
    cr = zc @ zc.T / Dm
    cc = zc.T @ zc / Tm
    cr.fill_diagonal_(0)
    cc.fill_diagonal_(0)
    assert cr.abs().max().item() < 6.5 / Dm ** 0.5 and abs(cr.std().item() * Dm ** 0.5 - 1) < 0.05    # sigma = 1/sqrt(n)
    assert cc.abs().max().item() < 6.5 / Tm ** 0.5 and abs(cc.std().item() * Tm ** 0.5 - 1) < 0.05
    assert abs((m[1:] * m[:-1]).mean().item() - p * p) < 0.005
    assert abs((m[:, 1:] * m[:, :-1]).mean().item() - p * p) < 0.005

