"""Parity of the conv kernels AT THE SHAPES bench.py TIMES: SSD-ResNet50 512x512 at 64 images per GPU (cfg2), the
SSD-MobileNetV2 300x300 layers at 64 images (cfg3) and the SSDBiFPN-RegNetX032 1280x1280 grouped convolutions at 4
images (cfg5) — the multi-way (interleaved accumulator) and weight-resident instantiations of conv_igemm_kernel,
partial groups with ghost tiles, multi-group persistence, the chunked grouped conv, conv_pair_kernel, mbconv_kernel
on a persistent grid and the row-streaming depthwise kernel at full size.

Every case asserts (through ssdsb_conv_last_launch / ssdsb_mbconv_last_launch) WHICH instantiation the launch
heuristics picked, so a change of the heuristics cannot silently move a case back onto the WAYS=1 path.

Tolerance: bf16 outputs within half a bf16 ulp plus the fp32 accumulation error of an fp64 reference on the same bf16
operands (oracle/bf16_bound.py), over the whole batch; WAYS / residency / pairing / fusion must not change a single bit
(checked against the WAYS=1 launch, the separate launches, the per-output depthwise kernel)."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle.bf16_bound import ACC_REL, assert_bf16_close, conv_ref64

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def K():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    from ssds_pytorch_b200 import conv
    return conv


def check_batch(y, x, w, b, stride, pad, msg, chunk=8, **kw):
    """assert_bf16_close against conv_ref64 over the whole batch, `chunk` images at a time (bounded memory);
    returns the worst err / tol"""
    worst = 0.0
    for n0 in range(0, x.shape[0], chunk):
        img = range(n0, min(n0 + chunk, x.shape[0]))
        ref, S = conv_ref64(x, w, b, stride, pad, images=img, **kw)
        worst = max(worst, assert_bf16_close(y[n0:n0 + chunk], ref, S, f"{msg}, images {n0}+"))
    return worst


# N, H, W, Cin, Cout, k, stride, pad, relu, residual, expect (subset of last_launch() that must hold)
CASES = [
    # layer1 3x3 64->64 @128x128: BLOCK_N=64, 4 ways (the 72 KiB weight slab does not fit next to 4-way stages)
    (64, 128, 128, 64, 64, 3, 1, 1, True, False, dict(block_n=64, ways=4, b_resident=0, ghost=0)),
    # layer1 conv1 1x1 64->64 @128x128: 4 ways, resident
    (64, 128, 128, 64, 64, 1, 1, 0, True, False, dict(block_n=64, ways=4, b_resident=1)),
    # layer1 conv3 1x1 64->256 + identity @128x128: BLOCK_N=256 (1 way), resident weights, residual prefetch
    (64, 128, 128, 64, 256, 1, 1, 0, True, True, dict(block_n=256, ways=1, b_resident=1)),
    # layer2 3x3 128->128 @64x64: BLOCK_N=128, 2 ways, weights streamed (288 KiB)
    (64, 64, 64, 128, 128, 3, 1, 1, True, False, dict(block_n=128, ways=2, b_resident=0, ghost=0)),
    # layer2.0 conv2 3x3/s2 128->128 @128x128 -> 64x64
    (64, 128, 128, 128, 128, 3, 2, 1, True, False, dict(block_n=128, ways=2)),
    # layer2.0 downsample 1x1/s2 256->512 @128x128 -> 64x64 (no ReLU)
    (64, 128, 128, 256, 512, 1, 2, 0, False, False, dict(block_n=256, ways=1)),
    # layer3 3x3 256->256 @32x32 and layer3 conv3 1x1 256->1024 + identity
    (64, 32, 32, 256, 256, 3, 1, 1, True, False, dict(block_n=256, ways=1)),
    (64, 32, 32, 256, 1024, 1, 1, 0, True, True, dict(block_n=256, ways=1)),
    # layer4 1x1 2048->512 @16x16 (long K) and 512->2048 + identity
    (64, 16, 16, 2048, 512, 1, 1, 0, True, False, dict(block_n=256, ways=1)),
    (64, 16, 16, 512, 2048, 1, 1, 0, True, True, dict(block_n=256, ways=1)),
    # partial last group (ghost tiles): 37 x (5 x 9) = 1665 M-tiles, 4 ways -> 417 groups, 1 real + 3 ghosts
    (37, 72, 80, 64, 64, 3, 1, 1, True, False, dict(block_n=64, ways=4, ghost=1)),
    # same with 2 ways: 21 x 45 = 945 M-tiles -> 473 groups, the last one half empty
    (21, 72, 80, 128, 128, 3, 1, 1, True, False, dict(block_n=128, ways=2, ghost=1)),
    # ghost tiles + residual (staged epilogue must skip nothing and clip everything; 6 staging slots -> 2 ways)
    (37, 72, 80, 64, 64, 1, 1, 0, True, True, dict(block_n=64, ways=2, ghost=1)),
    # 4 ways + resident weights + ghost tiles, no residual
    (37, 72, 80, 64, 64, 1, 1, 0, True, False, dict(block_n=64, ways=4, b_resident=1, ghost=1)),
    # cfg3 (SSD-MobileNetV2 300x300, B=64; relu 2 = ReLU6).  Project 144(160) -> 24(32) of the stride-2 block at
    # 38x38: 960 M-tiles are too few for 4 ways -> <64,32,2>
    (64, 38, 38, 160, 32, 1, 1, 0, 0, False, dict(block_n=64, block_k=32, ways=2, ghost=0)),
    # expand 24(32) -> 144(160) at 75x75: <256,32,1> with resident weights on a full grid
    (64, 75, 75, 32, 160, 1, 1, 0, 2, False, dict(block_n=256, block_k=32, ways=1, b_resident=1, grid=148)),
]


@pytest.mark.parametrize("case", CASES, ids=lambda c: "x".join(str(v) for v in c[:8]))
def test_conv_at_baseline_shape(K, case, monkeypatch):
    N, H, W, Cin, Cout, k, stride, pad, relu, use_res, expect = case
    g = torch.Generator(device="cuda").manual_seed(sum(case[:8]))
    x = torch.randn((N, H, W, Cin), generator=g, device="cuda").to(torch.bfloat16)
    w = torch.randn((Cout, Cin, k, k), generator=g, device="cuda") * (1.0 / np.sqrt(Cin * k * k))
    b = torch.randn((Cout,), generator=g, device="cuda")
    Ho, Wo = (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1
    res = torch.randn((N, Ho, Wo, Cout), generator=g, device="cuda").to(torch.bfloat16) if use_res else None
    wp = K.pack_weight(w.cpu()).cuda()
    y = torch.full((N, Ho, Wo, Cout), float("nan"), dtype=torch.bfloat16, device="cuda")
    K.conv2d(x, wp, b, k, k, stride, pad, relu, res, out=y)
    got = K.last_launch()
    torch.cuda.synchronize()
    for key, v in expect.items():
        assert got[key] == v, f"launch heuristics changed: {got} (expected {expect})"
    assert got["groups"] > got["grid"], f"not persistent over several groups: {got}"
    # (1) bit-identical to the 1-way, non-interleaved launch of the same kernel family
    monkeypatch.setenv("SSDSB_WAYS", "1")
    y1 = K.conv2d(x, wp, b, k, k, stride, pad, relu, res)
    assert K.last_launch()["ways"] == 1
    monkeypatch.delenv("SSDSB_WAYS")
    torch.cuda.synchronize()
    assert torch.equal(y, y1), "multi-way / resident launch differs from the 1-way launch"
    del y1
    # (2) vs fp64 on the same bf16 operands
    worst = check_batch(y, x, w, b, stride, pad, f"{case[:10]} {got}", residual=res, relu=int(relu))
    print(f"conv {case[:10]} {got}: worst err/tol {worst:.3f}")
    assert torch.isfinite(y.float()).all()


def test_stem_at_baseline_shape(K):
    """resnet.py:42-44 conv1 7x7/s2 at 512x512, B=64 through the windowed s2d stem (BLOCK_N=64, 4 ways)."""
    g = torch.Generator().manual_seed(5)
    N, H, W = 64, 512, 512
    w = torch.randn((64, 3, 7, 7), generator=g) * 0.1
    b = torch.randn((64,), generator=g) * 0.1
    img = torch.randint(0, 256, (N, H, W, 3), generator=g, dtype=torch.uint8).cuda()
    packed = K.pack_image_s2d(img, 0.0, 255.0, padded=True)
    y = K.conv2d(packed, K.pack_stem_weight_s2d(w).cuda(), b.cuda(), 4, 4, 1, 2, True,
                 Ho=H // 2, Wo=W // 2, x_kind=1, x_width=W // 2)
    got = K.last_launch()
    torch.cuda.synchronize()
    assert got["block_n"] == 64 and got["ways"] == 4, got
    wr, br = w.to(torch.bfloat16).float().cuda(), b.cuda()
    worst = 0.0
    for n0 in range(0, N, 8):
        xr = (img[n0:n0 + 8].float() / 255.0).to(torch.bfloat16).float().permute(0, 3, 1, 2)
        ref = F.conv2d(xr, wr, br, stride=2, padding=3).relu().permute(0, 2, 3, 1)
        err = (y[n0:n0 + 8].float() - ref).abs() / ref.abs().clamp(min=1.0)
        worst = max(worst, err.max().item())
    assert worst <= 2e-2, worst


@pytest.mark.parametrize("shape", [(64, 64, 64, 512), (64, 32, 32, 1024)])
def test_head_at_baseline_shape(K, shape):
    """multibox head 3x3 Cin->(24 loc + 480 conf) at the cfg-2 level sizes (ssd.py:100-103), fp32 NCHW out."""
    N, H, W, Cin = shape
    g = torch.Generator(device="cuda").manual_seed(H)
    x = torch.randn((N, H, W, Cin), generator=g, device="cuda").to(torch.bfloat16)
    w = torch.randn((504, Cin, 3, 3), generator=g, device="cuda") * (1.0 / np.sqrt(Cin * 9))
    b = torch.cat([torch.zeros(24), torch.full((480,), -4.595)]).cuda()
    loc, conf = K.conv2d_head(x, K.pack_weight(w.cpu()).cuda(), b, 24, True)
    got = K.last_launch()
    torch.cuda.synchronize()
    assert got["block_n"] == 256 and got["groups"] > got["grid"], got
    # loc is fp32: the fp32 accumulation error only; conf (sigmoid with __expf) keeps 1e-4
    wl, wc = 0.0, 0.0
    for n0 in range(0, N, 8):
        ref, S = conv_ref64(x, w, b, 1, 1, images=range(n0, n0 + 8))
        ref, S = ref.permute(0, 3, 1, 2), S.permute(0, 3, 1, 2)
        wl = max(wl, ((loc[n0:n0 + 8].double() - ref[:, :24]).abs() / (ACC_REL * S[:, :24])).max().item())
        wc = max(wc, (conf[n0:n0 + 8].double() - ref[:, 24:].sigmoid()).abs().max().item())
    print(f"head {shape}: loc worst err/(2^-17 S) {wl:.3f}, conf max err {wc:.2e}")
    assert wl <= 1.0 and wc <= 1e-4, (wl, wc)


PAIR_CASES = [
    (64, 128, 128, 64, 256, 64),     # layer1: conv3 64->256 (+identity) -> next conv1 256->64
    (64, 128, 128, 64, 256, 128),    # layer1 -> layer2 transition
    (64, 64, 64, 128, 512, 128),     # layer2
    (64, 64, 64, 128, 512, 256),     # layer2 -> layer3 transition
]


@pytest.mark.parametrize("case", PAIR_CASES, ids=lambda c: "x".join(str(v) for v in c))
def test_conv_pair_at_baseline_shape(K, case):
    """conv_pair_kernel at the sizes model.py pairs at B=64 (>= 8 M-tiles per SM): bit-identical to two
    conv2d launches, and y1 vs torch fp32."""
    N, H, W, Cin, Cmid, Cout2 = case
    g = torch.Generator(device="cuda").manual_seed(sum(case))
    x = torch.randn((N, H, W, Cin), generator=g, device="cuda").to(torch.bfloat16)
    w1f = torch.randn((Cmid, Cin, 1, 1), generator=g, device="cuda") / np.sqrt(Cin)
    w2f = torch.randn((Cout2, Cmid, 1, 1), generator=g, device="cuda") / np.sqrt(Cmid)
    w1, w2 = K.pack_weight(w1f.cpu()).cuda(), K.pack_weight(w2f.cpu()).cuda()
    b1 = torch.randn((Cmid,), generator=g, device="cuda")
    b2 = torch.randn((Cout2,), generator=g, device="cuda")
    res = torch.randn((N, H, W, Cmid), generator=g, device="cuda").to(torch.bfloat16)
    r1 = K.conv2d(x, w1, b1, 1, 1, 1, 0, True, res)
    r2 = K.conv2d(r1, w2, b2, 1, 1, 1, 0, True)
    for _ in range(2):
        y1 = torch.full_like(r1, float("nan"))
        y2 = torch.full_like(r2, float("nan"))
        K.conv1x1_pair(x, w1, b1, True, res, w2, b2, True, out1=y1, out2=y2)
        torch.cuda.synchronize()
        assert torch.equal(y1, r1)
        assert torch.equal(y2, r2)
    worst = check_batch(y1, x, w1f, b1, 1, 0, f"pair y1 {case}", residual=res, relu=1)
    print(f"pair y1 {case}: worst err/tol {worst:.3f}")


# N, H_in, channels (unpadded), stride, expect — the SSDBiFPN-RegNetX032 3x3 grouped convs (group width 48) at
# 1280x1280, B=4 (cfg5): one chunk of 96 channels (two groups) per 128-row weight slab, two interleaved accumulators
# and the direct (un-staged) epilogue walking 96 of the accumulator's 128 columns
GROUPED_CASES = [
    (4, 320, 96, 1, dict(ghost=0)),          # stage 1 @320x320
    (4, 160, 192, 1, dict(ghost=0)),         # stage 2 @160x160
    (4, 80, 432, 1, dict(ghost=0)),          # stage 3 @80x80, 432 -> 480 channels
    (4, 40, 1008, 1, dict(ghost=0)),         # stage 4 @40x40, 1008 -> 1056 channels
    (4, 320, 192, 2, dict(ghost=0)),         # first (stride 2) blocks of stages 2-4
    (4, 160, 432, 2, dict(ghost=0)),
    (4, 80, 1008, 2, dict(ghost=0)),
    (5, 40, 1008, 1, dict(ghost=1)),         # off-benchmark: 75 M-tiles, the last group's second tile is a ghost
]


@pytest.mark.parametrize("case", GROUPED_CASES, ids=lambda c: "x".join(str(v) for v in c[:4]))
def test_grouped_conv_at_cfg5_shape(K, case, monkeypatch):
    N, H, Cc, stride, expect = case
    gw, chunk = 48, 96
    c_pad = (Cc + chunk - 1) // chunk * chunk
    g = torch.Generator(device="cuda").manual_seed(Cc * 10 + stride + N)
    x = torch.zeros((N, H, H, c_pad), dtype=torch.bfloat16, device="cuda")
    x[..., :Cc] = torch.randn((N, H, H, Cc), generator=g, device="cuda").to(torch.bfloat16)
    w = torch.randn((Cc, gw, 3, 3), generator=g, device="cuda") * (1.0 / np.sqrt(gw * 9))
    b = torch.zeros(c_pad, device="cuda")
    b[:Cc] = torch.randn((Cc,), generator=g, device="cuda") * 0.2
    wp = K.pack_grouped_weight(w.cpu(), chunk, c_pad).cuda()
    ho = (H - 1) // stride + 1
    y = torch.full((N, ho, ho, c_pad), float("nan"), dtype=torch.bfloat16, device="cuda")
    K.conv2d(x, wp, b, 3, 3, stride, 1, True, out=y, chunk=chunk)
    got = K.last_launch()
    torch.cuda.synchronize()
    want = dict(block_n=128, block_k=32, ways=2, **expect)
    for key, v in want.items():
        assert got[key] == v, f"launch heuristics changed: {got} (expected {want})"
    assert got["groups"] > got["grid"], got
    monkeypatch.setenv("SSDSB_WAYS", "1")
    y1 = K.conv2d(x, wp, b, 3, 3, stride, 1, True, chunk=chunk)
    assert K.last_launch()["ways"] == 1
    monkeypatch.delenv("SSDSB_WAYS")
    torch.cuda.synchronize()
    assert torch.equal(y, y1), "2-way grouped launch differs from the 1-way launch"
    del y1
    assert (y[..., Cc:] == 0).all(), "padded channels must stay exactly 0"
    worst = check_batch(y[..., :Cc], x[..., :Cc], w, b[:Cc], stride, 1, f"grouped {case[:4]} {got}", chunk=1,
                        groups=Cc // gw, relu=1)
    print(f"grouped {case[:4]} {got}: worst err/tol {worst:.3f}")


# N, H, W, C, stride — every depthwise 3x3 of SSD-MobileNetV2 300x300 at B=64 (cfg3; channels padded to 32).  Which
# of them the plan runs as separate launches depends on its per-block timing, so all are covered.
DW_CFG3 = [
    (64, 150, 150, 32, 1), (64, 150, 150, 96, 2), (64, 75, 75, 160, 1), (64, 75, 75, 160, 2),
    (64, 38, 38, 192, 1), (64, 38, 38, 192, 2), (64, 19, 19, 384, 1), (64, 19, 19, 576, 1),
    (64, 19, 19, 576, 2), (64, 10, 10, 960, 1),
]


@pytest.mark.parametrize("case", DW_CFG3, ids=lambda c: "x".join(str(v) for v in c))
def test_dwconv3x3_at_cfg3_shape(K, case, monkeypatch):
    """the row-streaming depthwise kernel with the chunking its heuristic picks at B=64: bit-identical to the
    per-output kernel (SSDSB_DW_SIMPLE=1) and within the half-ulp bound of fp64 (+ folded BN bias + ReLU6)."""
    N, H, W, Cc, stride = case
    g = torch.Generator(device="cuda").manual_seed(sum(case))
    x = torch.randn((N, H, W, Cc), generator=g, device="cuda").to(torch.bfloat16)
    wf = torch.randn((Cc, 1, 3, 3), generator=g, device="cuda") * 0.4
    b = torch.randn((Cc,), generator=g, device="cuda") * 0.3
    w = K.pack_dw_weight(wf.cpu()).cuda()
    monkeypatch.delenv("SSDSB_DW_ROWS", raising=False)
    monkeypatch.setenv("SSDSB_DW_SIMPLE", "1")
    want = K.dwconv3x3(x, w, b, stride, 2)
    monkeypatch.delenv("SSDSB_DW_SIMPLE")
    y = K.dwconv3x3(x, w, b, stride, 2)
    torch.cuda.synchronize()
    assert torch.equal(y, want), "row-streaming depthwise kernel differs from the per-output kernel"
    assert (y.float() == 6.0).any() and (y.float() == 0.0).any()
    worst = check_batch(y, x, wf, b, stride, 1, str(case), groups=Cc, relu=2)
    print(f"dwconv3x3 {case}: worst err/tol {worst:.3f}")
