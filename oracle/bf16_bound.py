"""The accuracy bound a bf16-output convolution kernel is held to.

The conv kernels multiply bf16 operands exactly, accumulate in fp32, add the fp32 bias (and the bf16 residual) in
fp32 and round once to bf16 (round-to-nearest-even).  Against the exact result `ref64` of the same operation on the
same bf16 operands, every output element y therefore satisfies

    |y - ref64| <= 0.5 * ulp_bf16(ref64) + 2^-17 * S

where S is the same operation on |x|, |w| plus |bias| + |residual|: the half ulp is the final rounding, 2^-17 * S
covers the fp32 accumulation (2^-24 per addition, with room for the sum's depth; see tests/test_bf16_bound_cpu.py for
the emulation that sizes it).  ReLU / ReLU6 are applied to ref64 in fp64: clamping at 0 and 6 (both exact in bf16)
commutes with round-to-nearest and never increases a distance.

A kernel that truncates instead of rounding, or rounds an intermediate (the accumulator before the bias or the
residual is added) to bf16, breaks this bound on a large fraction of elements, while a relative bar of 2e-2 accepts
both."""
import torch
import torch.nn.functional as F

ACC_REL = 2.0 ** -17


def ulp_bf16(v):
    """The spacing of bf16 numbers at |v| (8 significant bits; normal range only, as bf16 subnormals sit below
    every value these tests produce)."""
    a = v.abs().double().clamp(min=2.0 ** -126)
    _, e = torch.frexp(a)                  # a = m * 2^e, m in [0.5, 1): the leading bit is 2^(e-1)
    return torch.ldexp(torch.ones_like(a), (e - 8).to(torch.int32))


def bf16_tolerance(ref64, S):
    return 0.5 * ulp_bf16(ref64) + ACC_REL * S.double()


def assert_bf16_close(y, ref64, S, msg=""):
    """Assert |y - ref64| <= 0.5 ulp_bf16(ref64) + 2^-17 S element-wise (NaN in y fails).  Returns the worst
    err / tol so that callers can report how close to the bound the kernel runs."""
    ref64 = ref64.double()
    err = (y.double() - ref64).abs()
    ratio = err / bf16_tolerance(ref64, S)
    bad = ~(ratio <= 1.0)
    flat = torch.where(torch.isnan(ratio), torch.full_like(ratio, float("inf")), ratio).flatten()
    i = int(flat.argmax())
    worst = flat[i].item()
    if bool(bad.any()):
        where = list(torch.unravel_index(torch.tensor(i), ratio.shape))
        raise AssertionError(
            f"{msg}: {int(bad.sum())} of {ratio.numel()} elements outside the half-ulp bound; worst err/tol {worst:.3f} "
            f"at {[int(t) for t in where]} (y={y.flatten()[i].item():.8g}, ref={ref64.flatten()[i].item():.8g}, "
            f"S={S.flatten()[i].item():.6g})")
    return worst


def conv_ref64(x, w, bias=None, stride=1, pad=0, groups=1, residual=None, relu=0, images=None):
    """fp64 reference of a kernel conv and its magnitude sum S, NHWC like the kernel's output.

    x NHWC bf16 (exactly the kernel's input); w [Cout, Cin/groups, KH, KW] in any float type, rounded to bf16 here as
    the packing does; bias fp32 [Cout] or None; residual NHWC bf16 or None; relu 0 none, 1 ReLU, 2 ReLU6.
    `images` selects batch entries (the reference runs on those only, to bound memory); None means all."""
    if images is not None:
        idx = torch.as_tensor(list(images), device=x.device)
        x = x.index_select(0, idx)
        residual = residual.index_select(0, idx) if residual is not None else None
    xd = x.double().permute(0, 3, 1, 2)
    wd = w.to(x.device).to(torch.bfloat16).double()
    ref = F.conv2d(xd, wd, None, stride=stride, padding=pad, groups=groups)
    S = F.conv2d(xd.abs(), wd.abs(), None, stride=stride, padding=pad, groups=groups)
    if bias is not None:
        bd = bias.to(x.device).double().view(1, -1, 1, 1)
        ref = ref + bd
        S = S + bd.abs()
    if residual is not None:
        rd = residual.double().permute(0, 3, 1, 2)
        ref = ref + rd
        S = S + rd.abs()
    if relu:
        ref = ref.clamp(min=0.0, max=6.0 if relu == 2 else None)
    return ref.permute(0, 2, 3, 1), S.permute(0, 2, 3, 1)
