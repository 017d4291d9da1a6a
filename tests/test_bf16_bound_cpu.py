"""How sensitive is the half-ulp bound of oracle/bf16_bound.py?  A CPU emulation of the conv kernels' arithmetic as a
matmul: bf16 operands, fp32 accumulation in 16-wide K blocks (one tcgen05 MMA step each), fp32 bias and bf16 residual
added in fp32, one round to bf16.  Round-to-nearest-even must satisfy the bound on every element; truncating the
result, or rounding to bf16 before the bias and again before the residual, must each break it on more than 20 % of
the elements — while the former 2e-2 relative bar accepts both broken variants."""
import pytest
import torch

from oracle.bf16_bound import assert_bf16_close, bf16_tolerance, ulp_bf16


def _truncate_bf16(f32):
    return (f32.view(torch.int32) & ~0xFFFF).view(torch.float32)


@pytest.mark.parametrize("K", [32, 576, 4608, 9072])
def test_bound_accepts_rne_and_rejects_truncation_and_double_rounding(K):
    g = torch.Generator().manual_seed(K)
    M, N = 4096, 128
    x = torch.randn((M, K), generator=g).bfloat16()
    w = (torch.randn((N, K), generator=g) / K ** 0.5).bfloat16()
    b = torch.randn((N,), generator=g)
    res = torch.randn((M, N), generator=g).bfloat16()
    xd, wd = x.double(), w.double()
    ref = xd @ wd.T + b.double() + res.double()
    S = xd.abs() @ wd.abs().T + b.double().abs() + res.double().abs()
    acc = torch.zeros((M, N), dtype=torch.float32)
    xf, wf = x.float(), w.float()
    for k0 in range(0, K, 16):
        acc += xf[:, k0:k0 + 16] @ wf[:, k0:k0 + 16].T
    f = acc + b + res.float()
    rne = f.bfloat16()
    worst = assert_bf16_close(rne, ref, S, f"K={K} round-to-nearest-even")
    assert worst > 0.5, "the bound is far looser than the rounding it is meant to check"
    tol = bf16_tolerance(ref, S)
    loose = 2e-2 * ref.abs().clamp(min=1.0)
    broken = {
        "truncate": _truncate_bf16(f),
        "double-round": ((acc.bfloat16().float() + b).bfloat16().float() + res.float()).bfloat16().float(),
    }
    for name, y in broken.items():
        err = (y.double() - ref).abs()
        frac = (err > tol).double().mean().item()
        print(f"K={K} {name}: {100 * frac:.1f} % of elements outside the half-ulp bound "
              f"(worst err/tol {(err / tol).max().item():.2f}), {int((err > loose).sum())} outside the 2e-2 bar; "
              f"round-to-nearest worst err/tol {worst:.3f}")
        assert frac > 0.2, (name, frac)
        assert int((err > loose).sum()) == 0
        with pytest.raises(AssertionError, match="outside the half-ulp bound"):
            assert_bf16_close(y, ref, S, name)


def test_ulp_bf16_and_nan():
    v = torch.tensor([1.0, 1.5, 2.0, -3.0, 0.0, 6.0, 2.0 ** -20])
    want = torch.tensor([2.0 ** -7, 2.0 ** -7, 2.0 ** -6, 2.0 ** -6, 2.0 ** -133, 2.0 ** -5, 2.0 ** -27],
                        dtype=torch.float64)
    assert torch.equal(ulp_bf16(v), want)
    # the spacing really is the distance to the next bf16 number
    nxt = (v.bfloat16().view(torch.int16) + 1).view(torch.bfloat16).double()
    assert torch.equal((nxt.abs() - v.double().abs())[:4], want[:4])
    with pytest.raises(AssertionError, match="1 of 2"):
        assert_bf16_close(torch.tensor([1.0, float("nan")]), torch.ones(2, dtype=torch.float64), torch.ones(2))
