"""tcgen05 implicit-GEMM convolution vs an fp64 reference of the same op on the kernel's bf16 operands (the kernel
multiplies bf16 x bf16 exactly and accumulates in fp32, so the only differences are fp32 summation order and the final
bf16 rounding of the output).
Tolerance: bf16 outputs within half a bf16 ulp plus the fp32 accumulation error (oracle/bf16_bound.py).  The stems
keep |err| <= 2e-2 * max(1, |ref|): their reference normalises the image itself instead of consuming the bf16 tensor
pack_image_s2d produces.  The fp32 head: loc within 2^-17 * S, the sigmoid-ed conf (computed with __expf) 1e-4."""
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


CASES = [
    # N, H, W, Cin, Cout, k, stride, pad, relu, residual
    (2, 16, 16, 64, 64, 1, 1, 0, True, False),      # 1x1, BLOCK_N=64
    (2, 16, 16, 64, 256, 1, 1, 0, False, True),     # 1x1 + residual, BLOCK_N=256
    (2, 32, 32, 64, 64, 3, 1, 1, True, False),      # 3x3 halo, 2 x 4 tiles
    (3, 16, 16, 128, 128, 3, 2, 1, True, False),    # 3x3 stride 2, BLOCK_N=128
    (2, 16, 16, 256, 512, 1, 2, 0, False, False),   # 1x1 stride 2 (downsample)
    (4, 8, 8, 128, 256, 3, 1, 1, True, False),      # 8x8 map: BN=2 images per tile
    (8, 4, 4, 64, 128, 3, 2, 1, True, False),       # 4x4 -> 2x2: many images per tile
    (5, 2, 2, 64, 64, 3, 1, 1, True, False),        # tiny map, ragged batch (5 of 32)
    (3, 1, 1, 64, 64, 1, 1, 0, True, False),        # 1x1 map
    (2, 19, 19, 64, 96, 3, 1, 1, True, False),      # 19x19 (MobileNet-SSD level): ragged tile rows
    (1, 40, 24, 192, 320, 3, 1, 1, True, True),     # non-pow2 channels, several K blocks, edges
    (2, 64, 64, 512, 64, 1, 1, 0, True, False),     # long K
    (2, 38, 38, 32, 192, 1, 1, 0, 2, False),        # MobileNetV2 expand: Cin=32 (64B K-blocks), ReLU6
    (2, 19, 19, 576, 96, 1, 1, 0, False, True),     # MobileNetV2 project + residual, Cout=96 (direct path)
    (2, 19, 19, 96, 64, 3, 1, 1, True, False),      # Cin=96 = 3 x 32
    (3, 10, 10, 160, 160, 3, 1, 1, 2, False),       # Cin=160 (32-blocks), 10x10 ragged tile, ReLU6
    (2, 75, 75, 160, 32, 1, 1, 0, False, False),    # Cout=32 (padded 24-channel layer)
]


@pytest.mark.parametrize("case", CASES)
def test_conv_nhwc(K, case):
    N, H, W, Cin, Cout, k, stride, pad, relu, use_res = case
    g = torch.Generator().manual_seed(hash(case) % (2 ** 31))
    x = torch.randn((N, H, W, Cin), generator=g).to(torch.bfloat16).cuda()
    w = torch.randn((Cout, Cin, k, k), generator=g) * (1.0 / np.sqrt(Cin * k * k))
    b = torch.randn((Cout,), generator=g)
    Ho, Wo = (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1
    res = torch.randn((N, Ho, Wo, Cout), generator=g).to(torch.bfloat16).cuda() if use_res else None
    y = K.conv2d(x, K.pack_weight(w).cuda(), b.cuda(), k, k, stride, pad, relu, res)
    torch.cuda.synchronize()
    ref, S = conv_ref64(x, w, b, stride, pad, residual=res, relu=int(relu))
    worst = assert_bf16_close(y, ref, S, str(case))
    print(f"conv {case}: worst err/tol {worst:.3f}")


def test_conv_head_split_sigmoid(K):
    """multibox head (ssd.py:100-103): loc 24 + conf 480 channels fused, fp32 NCHW, sigmoid on conf."""
    g = torch.Generator().manual_seed(3)
    N, H, W, Cin, A, Cc = 3, 16, 16, 128, 6, 80
    x = torch.randn((N, H, W, Cin), generator=g).to(torch.bfloat16).cuda()
    w = torch.randn((A * 4 + A * Cc, Cin, 3, 3), generator=g) * 0.02
    b = torch.cat([torch.zeros(A * 4), torch.full((A * Cc,), -4.595)])
    for sig in (True, False):
        loc, conf = K.conv2d_head(x, K.pack_weight(w).cuda(), b.cuda(), A * 4, sig)
        torch.cuda.synchronize()
        ref, S = conv_ref64(x, w, b, 1, 1)
        ref, S = ref.permute(0, 3, 1, 2), S.permute(0, 3, 1, 2)
        rl, rc = ref[:, :A * 4], ref[:, A * 4:]
        if sig:
            rc = rc.sigmoid()
        assert loc.shape == rl.shape and conf.shape == rc.shape
        # fp32 outputs: fp32 accumulation error only (no bf16 rounding)
        assert ((loc.double() - rl).abs() <= ACC_REL * S[:, :A * 4]).all(), ((loc.double() - rl).abs().max().item())
        if sig:
            assert (conf.double() - rc).abs().max().item() <= 1e-4
        else:
            assert ((conf.double() - rc).abs() <= ACC_REL * S[:, A * 4:]).all()


def test_stem_s2d_equals_7x7s2(K):
    """resnet.py:42-44 conv1 7x7/s2/p3 on a 3-channel image == 4x4/s1 conv on the space-to-depth
    packing, through pack_image_s2d for both fp32 NCHW and uint8 NHWC inputs."""
    g = torch.Generator().manual_seed(5)
    N, H, W = 2, 64, 96
    w = torch.randn((64, 3, 7, 7), generator=g) * 0.1
    b = torch.randn((64,), generator=g) * 0.1
    img_u8 = torch.randint(0, 256, (N, H, W, 3), generator=g, dtype=torch.uint8)
    for fmt in ("f32", "u8"):
        if fmt == "f32":
            src = (img_u8.float() / 255.0).permute(0, 3, 1, 2).contiguous().cuda()
            packed = K.pack_image_s2d(src, 0.0, 1.0)
        else:
            packed = K.pack_image_s2d(img_u8.cuda(), 0.0, 255.0)
        y = K.conv2d(packed, K.pack_stem_weight_s2d(w).cuda(), b.cuda(), 4, 4, 1, 2, True,
                     Ho=H // 2, Wo=W // 2)
        # windowed variant: left-padded rows, 4 taps x 16 ch fetched as one 128-byte K-block
        src_p = src if fmt == "f32" else img_u8.cuda()
        packed_p = K.pack_image_s2d(src_p, 0.0, 1.0 if fmt == "f32" else 255.0, padded=True)
        y2 = K.conv2d(packed_p, K.pack_stem_weight_s2d(w).cuda(), b.cuda(), 4, 4, 1, 2, True,
                      Ho=H // 2, Wo=W // 2, x_kind=1, x_width=W // 2)
        torch.cuda.synchronize()
        assert torch.equal(y, y2), "windowed stem differs from the per-tap stem"
        xr = (img_u8.float() / 255.0).to(torch.bfloat16).float().permute(0, 3, 1, 2).cuda()
        ref = F.conv2d(xr, w.to(torch.bfloat16).float().cuda(), b.cuda(), stride=2, padding=3).relu()
        ref = ref.permute(0, 2, 3, 1)
        err = (y.float() - ref).abs() / ref.abs().clamp(min=1.0)
        assert err.max().item() <= 2e-2, (fmt, err.max().item())


def test_stem_3x3s2_mobilenet(K):
    """MobileNetV2 conv1 (mobilenet.py:78: ConvBNReLU(3, 32, stride=2), 3x3/p1) on the same s2d path."""
    g = torch.Generator().manual_seed(6)
    N, H, W = 2, 60, 84
    w = torch.randn((32, 3, 3, 3), generator=g) * 0.2
    b = torch.randn((32,), generator=g) * 0.1
    img = torch.rand((N, 3, H, W), generator=g)
    packed = K.pack_image_s2d(img.cuda(), 0.0, 1.0, padded=True)
    y = K.conv2d(packed, K.pack_stem_weight_s2d(w).cuda(), b.cuda(), 4, 4, 1, 2, 2,
                 Ho=H // 2, Wo=W // 2, x_kind=1, x_width=W // 2)
    torch.cuda.synchronize()
    ref = F.conv2d(img.to(torch.bfloat16).float().cuda(), w.to(torch.bfloat16).float().cuda(), b.cuda(),
                   stride=2, padding=1).clamp(0, 6).permute(0, 2, 3, 1)
    err = (y.float() - ref).abs() / ref.abs().clamp(min=1.0)
    assert err.max().item() <= 2e-2, err.max().item()


@pytest.mark.parametrize("case", [(2, 38, 38, 192, 1, 2), (2, 38, 38, 192, 2, 2), (1, 75, 75, 160, 2, 1),
                                  (3, 10, 10, 960, 1, 2), (2, 19, 19, 96, 2, 0), (2, 3, 3, 32, 1, 2)])
def test_dwconv3x3(K, case):
    """depthwise 3x3 + folded BN + ReLU6 (torchvision InvertedResidual) vs F.conv2d(groups=C)."""
    N, H, W, Cc, stride, relu = case
    g = torch.Generator().manual_seed(sum(case))
    x = torch.randn((N, H, W, Cc), generator=g).to(torch.bfloat16).cuda()
    w = torch.randn((Cc, 1, 3, 3), generator=g) * 0.3
    b = torch.randn((Cc,), generator=g) * 0.2
    y = K.dwconv3x3(x, K.pack_dw_weight(w).cuda(), b.cuda(), stride, relu)
    torch.cuda.synchronize()
    ref, S = conv_ref64(x, w, b, stride, 1, groups=Cc, relu=relu)
    assert y.shape == ref.shape
    worst = assert_bf16_close(y, ref, S, str(case))
    print(f"dwconv3x3 {case}: worst err/tol {worst:.3f}")


RAGGED = [
    # N, H, W, Cin, Cout, k, stride, relu, residual — Cout % 64 == 32: the last 64-column chunk of the staged
    # TMA-store epilogue is half full (clipped by the store's tensor map)
    (2, 75, 75, 32, 160, 1, 1, 2, False),     # MobileNetV2 expand 24(32) -> 144(160), 1 n-tile of 256, 3 chunks
    (2, 75, 75, 160, 32, 1, 1, 0, True),      # project + residual, 4-way BLOCK_N = 64 with half a chunk per tile
    (3, 38, 38, 192, 32, 1, 1, 0, False),
    (2, 19, 19, 384, 96, 1, 1, 0, True),      # BLOCK_N = 128, 2 chunks, residual TMA load clipped too
    (2, 20, 20, 96, 288, 3, 1, 1, False),     # two n-tiles: 256 + 32
    (1, 40, 24, 64, 480, 1, 2, 1, True),      # RegNet width 432 padded to 480, stride 2 + residual
    (5, 3, 3, 64, 96, 3, 1, 2, False),        # tiny map, several images per tile
]


@pytest.mark.parametrize("case", RAGGED)
def test_conv_ragged_cout_staged_equals_direct(K, case, monkeypatch):
    """[r2] Cout % 64 != 0 layers now take the staged epilogue (full-line TMA stores) instead of per-lane 16-byte
    stores: same arithmetic, so the two paths must agree bit for bit — and with the torch reference within the
    file's tolerance.  The output is a channel slice of a wider buffer (concat-style stride): the clipped TMA store
    must not touch the neighbouring channels."""
    N, H, W, Cin, Cout, k, stride, relu, use_res = case
    pad = k // 2
    g = torch.Generator().manual_seed(Cout * 7 + Cin)
    x = torch.randn((N, H, W, Cin), generator=g).to(torch.bfloat16).cuda()
    w = torch.randn((Cout, Cin, k, k), generator=g) * (1.0 / np.sqrt(Cin * k * k))
    b = (torch.randn((Cout,), generator=g) * 0.2).cuda()
    ho, wo = (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1
    res = torch.randn((N, ho, wo, Cout), generator=g).to(torch.bfloat16).cuda() if use_res else None
    wp = K.pack_weight(w).cuda()
    outs = []
    for direct in (False, True):
        if direct:
            monkeypatch.setenv("SSDSB_DIRECT_RAGGED", "1")
        else:
            monkeypatch.delenv("SSDSB_DIRECT_RAGGED", raising=False)
        wide = torch.full((N, ho, wo, Cout + 32), 7.0, dtype=torch.bfloat16, device="cuda")
        y = K.conv2d(x, wp, b, k, k, stride, pad, relu, residual=res, out=wide[..., :Cout])
        torch.cuda.synchronize()
        assert torch.all(wide[..., Cout:] == 7.0), "store touched the neighbouring channels"
        outs.append(y.clone())
    monkeypatch.delenv("SSDSB_DIRECT_RAGGED", raising=False)
    assert torch.equal(outs[0], outs[1])
    ref, S = conv_ref64(x, w, b, stride, pad, residual=res, relu=relu)
    worst = assert_bf16_close(outs[0], ref, S, str(case))
    print(f"ragged {case}: worst err/tol {worst:.3f}")


@pytest.mark.parametrize("case", [(2, 75, 75, 160, 1, 2), (1, 150, 150, 96, 2, 2), (2, 19, 19, 384, 1, 2),
                                  (3, 10, 10, 960, 1, 2), (2, 21, 13, 64, 2, 1), (1, 7, 9, 32, 1, 0)])
def test_dwconv3x3_stream_any_chunking(K, case, monkeypatch):
    """[r2] the software-pipelined row-streaming depthwise kernel is bit-identical to the per-output kernel
    (same fp32 tap order) however the launch cuts the rows into chunks: the heuristic's own choice, 1-row chunks,
    chunks shorter / longer than the prefetch ring, one chunk for the whole map."""
    N, H, W, Cc, stride, relu = case
    g = torch.Generator().manual_seed(sum(case) + 1)
    x = torch.randn((N, H, W, Cc), generator=g).to(torch.bfloat16).cuda()
    w = K.pack_dw_weight(torch.randn((Cc, 1, 3, 3), generator=g) * 0.3).cuda()
    b = (torch.randn((Cc,), generator=g) * 0.2).cuda()
    monkeypatch.setenv("SSDSB_DW_SIMPLE", "1")
    want = K.dwconv3x3(x, w, b, stride, relu).clone()
    monkeypatch.delenv("SSDSB_DW_SIMPLE")
    for rows in (None, 1, 2, 3, 5, 7, 11, 1000):
        if rows is None:
            monkeypatch.delenv("SSDSB_DW_ROWS", raising=False)
        else:
            monkeypatch.setenv("SSDSB_DW_ROWS", str(rows))
        got = K.dwconv3x3(x, w, b, stride, relu)
        torch.cuda.synchronize()
        assert torch.equal(got, want), (case, rows)
    monkeypatch.delenv("SSDSB_DW_ROWS", raising=False)


@pytest.mark.parametrize("case", [(2, 10, 12, 64), (1, 4, 5, 256), (3, 20, 20, 32), (1, 1, 1, 8)])
def test_maxpool5x5s1_spp_cascade(K, case):
    """[r2] YOLOv4's SPP block (yolo.py:161-184): x | maxpool5 | maxpool9 | maxpool13 concatenated = three cascaded
    5x5 / stride-1 pools between channel slices of one buffer; exact (max of bf16 values)."""
    N, H, W, Cc = case
    g = torch.Generator().manual_seed(sum(case))
    x = torch.randn((N, H, W, Cc), generator=g).to(torch.bfloat16).cuda()
    cat = torch.full((N, H, W, 4 * Cc), 9.0, dtype=torch.bfloat16, device="cuda")
    cat[..., :Cc] = x
    for k in range(3):
        K.maxpool5x5s1(cat[..., k * Cc:(k + 1) * Cc], cat[..., (k + 1) * Cc:(k + 2) * Cc])
    torch.cuda.synchronize()
    xn = x.float().permute(0, 3, 1, 2)
    ref = torch.cat([xn] + [F.max_pool2d(xn, kernel_size=kk, stride=1, padding=kk // 2) for kk in (5, 9, 13)], dim=1)
    assert torch.equal(cat.float(), ref.permute(0, 2, 3, 1))


MBCONV = [
    # N, H, W, Cin, hid, Cout, stride, residual — the MobileNetV2-SSD 300x300 block shapes (channels padded to 32
    # as the plan stores them; hid == Cin and no expand layer for the first block) + ragged odd cases
    (2, 150, 150, 32, 32, 32, 1, False),
    (2, 150, 150, 32, 96, 32, 2, False),
    (2, 75, 75, 32, 160, 32, 1, True),
    (2, 75, 75, 32, 160, 32, 2, False),
    (3, 38, 38, 32, 192, 32, 1, True),
    (2, 38, 38, 32, 192, 64, 2, False),
    (2, 19, 19, 64, 384, 64, 1, True),
    (2, 19, 19, 64, 384, 96, 1, False),
    (2, 19, 19, 96, 576, 96, 1, True),
    (2, 19, 19, 96, 576, 160, 2, False),
    (3, 10, 10, 160, 960, 160, 1, True),
    (1, 21, 13, 32, 64, 32, 1, True),
    (1, 7, 9, 64, 128, 96, 2, False),
    (70, 5, 5, 64, 128, 64, 1, True),        # more tiles than SMs would hold at once is not needed: many images
]
# the eleven MobileNetV2 block shapes again at the cfg3 batch (64 images): one CTA per SM, each working through several
# output tiles — except the two 10x10-output blocks, whose 128 tiles are fewer than the SMs
MBCONV += [(64,) + c[1:] for c in MBCONV[:11]]


@pytest.mark.parametrize("case", MBCONV)
def test_mbconv_fused_equals_three_launches(K, case):
    """[r2] ssdsb_mbconv_bf16 (expand -> depthwise -> project [+x] in one launch, the expanded tensor never
    leaves the SM) is bit-identical to conv2d -> dwconv3x3 -> conv2d: same bf16 rounding points, same fp32
    accumulation order.  Activations are scaled so that ReLU6 clips on both sides."""
    N, H, W, Cin, hid, Cout, stride, res = case
    g = torch.Generator().manual_seed(sum(case))
    x = torch.randn((N, H, W, Cin), generator=g).to(torch.bfloat16).cuda()
    has_expand = hid != Cin or Cin != 32 or stride != 1 or res
    if has_expand:
        we = K.pack_weight(torch.randn((hid, Cin, 1, 1), generator=g) * (2.0 / np.sqrt(Cin))).cuda()
        be = (torch.randn((hid,), generator=g) * 0.5).cuda()
    else:
        we = be = None
    wd = K.pack_dw_weight(torch.randn((hid, 1, 3, 3), generator=g) * 0.4).cuda()
    bd = (torch.randn((hid,), generator=g) * 0.3).cuda()
    wp = K.pack_weight(torch.randn((Cout, hid, 1, 1), generator=g) * (1.0 / np.sqrt(hid))).cuda()
    bp = (torch.randn((Cout,), generator=g) * 0.2).cuda()
    h = K.conv2d(x, we, be, 1, 1, 1, 0, 2) if has_expand else x
    d = K.dwconv3x3(h, wd, bd, stride, 2)
    want = K.conv2d(d, wp, bp, 1, 1, 1, 0, 0, residual=x if res else None)
    got = K.mbconv(x, we, be, wd, bd, wp, bp, stride, res, (2, 2, 0))
    torch.cuda.synchronize()
    info = K.mbconv_last_launch()
    assert got.shape == want.shape
    if N == 64:
        ho, wo = got.shape[1:3]
        tiles = N * -(-ho // info["tile_h"]) * -(-wo // info["tile_w"])
        assert info["grid"] == min(tiles, K.sm_count()), f"{info}, {tiles} tiles"
        assert info["grid"] < tiles or ho == 10, f"not persistent: {info}, {tiles} tiles"
    if not torch.equal(got, want):
        diff = (got.float() - want.float()).abs()
        bad = (diff > 0).nonzero()
        raise AssertionError(f"{case} {info}: {bad.shape[0]} of {diff.numel()} differ, max {diff.max().item():.4g}, "
                             f"first at {bad[0].tolist()}, last at {bad[-1].tolist()}")
    assert (d.float() == 0.0).any() and d.float().max().item() >= 3.0
    if has_expand:                      # both clamp bounds of both ReLU6 stages are exercised
        assert (h.float() == 6.0).any() and (h.float() == 0.0).any() and (d.float() == 6.0).any()


def test_mbconv_unsupported_is_loud(K):
    x = torch.zeros((1, 10, 10, 160), dtype=torch.bfloat16, device="cuda")
    we = torch.zeros((960, 1, 160), dtype=torch.bfloat16, device="cuda")
    wd = torch.zeros((9, 960), dtype=torch.bfloat16, device="cuda")
    wp = torch.zeros((320, 1, 960), dtype=torch.bfloat16, device="cuda")
    z = lambda n: torch.zeros(n, device="cuda")
    with pytest.raises(NotImplementedError):
        K.mbconv(x, we, z(960), wd, z(960), wp, z(320))


@pytest.mark.parametrize("case", [(2, 20, 20, 432, 1), (2, 20, 20, 192, 2), (1, 40, 24, 96, 1), (3, 10, 10, 1008, 1)])
def test_grouped_conv_regnet(K, case):
    """RegNet 3x3 grouped conv (group width 48; regnet.py:69) as a block-diagonal chunked igemm:
    channels padded to a multiple of 96 (two groups per chunk), padded channels stay 0."""
    N, H, W, Cc, stride = case
    gw, chunk = 48, 96
    c_pad = (Cc + chunk - 1) // chunk * chunk
    g = torch.Generator().manual_seed(Cc + stride)
    x = torch.zeros((N, H, W, c_pad), dtype=torch.bfloat16)
    x[..., :Cc] = torch.randn((N, H, W, Cc), generator=g).to(torch.bfloat16)
    w = torch.randn((Cc, gw, 3, 3), generator=g) * (1.0 / np.sqrt(gw * 9))
    b = torch.zeros(c_pad)
    b[:Cc] = torch.randn((Cc,), generator=g) * 0.2
    y = K.conv2d(x.cuda(), K.pack_grouped_weight(w, chunk, c_pad).cuda(), b.cuda(), 3, 3, stride, 1, True,
                 chunk=chunk)
    torch.cuda.synchronize()
    ref, S = conv_ref64(x[..., :Cc].cuda(), w, b[:Cc], stride, 1, groups=Cc // gw, relu=1)
    assert y.shape[-1] == c_pad
    worst = assert_bf16_close(y[..., :Cc], ref, S, str(case))
    print(f"grouped {case}: worst err/tol {worst:.3f}")
    assert (y[..., Cc:] == 0).all()


def test_bifpn_fuse(K):
    """BiFPN weighted fusion (bifpn.py:41-62) vs the torch expressions of the reference."""
    g = torch.Generator().manual_seed(15)
    a = torch.randn((2, 10, 14, 256), generator=g).to(torch.bfloat16).cuda()
    coarse = torch.randn((2, 5, 7, 256), generator=g).to(torch.bfloat16).cuda()
    fine = torch.randn((2, 20, 28, 256), generator=g).to(torch.bfloat16).cuda()
    c = torch.randn((2, 10, 14, 256), generator=g).to(torch.bfloat16).cuda()
    nchw = lambda t: t.float().permute(0, 3, 1, 2)
    w0, w1, w2 = 0.37, 0.41, 0.22
    up = K.bifpn_fuse(a, coarse, w0, w1, mode=0)
    ref = (w0 * nchw(a) + w1 * F.interpolate(nchw(coarse), scale_factor=2, mode="nearest")).permute(0, 2, 3, 1)
    assert (up.float() - ref).abs().max().item() <= 2e-2
    dn = K.bifpn_fuse(a, fine, w0, w1, c=c, w2=w2, mode=1)
    ref = (w0 * nchw(a) + w1 * F.max_pool2d(nchw(fine), kernel_size=2) + w2 * nchw(c)).permute(0, 2, 3, 1)
    assert (dn.float() - ref).abs().max().item() <= 2e-2
    dn2 = K.bifpn_fuse(a, fine, w0, w1, mode=1)
    ref = (w0 * nchw(a) + w1 * F.max_pool2d(nchw(fine), kernel_size=2)).permute(0, 2, 3, 1)
    assert (dn2.float() - ref).abs().max().item() <= 2e-2


def test_upsample2x_add(K):
    g = torch.Generator().manual_seed(12)
    coarse = torch.randn((2, 5, 7, 256), generator=g).to(torch.bfloat16).cuda()
    fine = torch.randn((2, 10, 14, 256), generator=g).to(torch.bfloat16).cuda()
    ref = (F.interpolate(coarse.float().permute(0, 3, 1, 2), scale_factor=2, mode="nearest") +
           fine.float().permute(0, 3, 1, 2)).permute(0, 2, 3, 1).to(torch.bfloat16)
    K.upsample2x_add(coarse, fine)
    assert torch.equal(fine, ref)


def test_maxpool(K):
    g = torch.Generator().manual_seed(9)
    for (N, H, W, Cc) in [(2, 32, 32, 64), (1, 15, 17, 8), (2, 7, 9, 16), (1, 2, 2, 8), (3, 33, 20, 24), (1, 1, 1, 8)]:
        x = torch.randn((N, H, W, Cc), generator=g).to(torch.bfloat16).cuda()
        y = K.maxpool3x3s2(x)
        ref = F.max_pool2d(x.float().permute(0, 3, 1, 2), 3, 2, 1).permute(0, 2, 3, 1)
        assert torch.equal(y.float(), ref)


PAIR_CASES = [
    # N, H, W, Cin, Cmid, Cout2, residual      (conv3 of one bottleneck -> conv1 of the next)
    (4, 32, 32, 64, 256, 64, True),      # layer1 geometry: 1 K-block, 4 chunks, N2 = 64
    (2, 32, 32, 128, 512, 128, True),    # layer2: two 256-wide n-tiles for y1
    (2, 16, 16, 256, 1024, 256, True),   # layer3
    (2, 16, 16, 512, 2048, 512, True),   # layer4: Cout2 = 512 -> two n-tiles for y2 as well
    (3, 32, 32, 64, 256, 128, True),     # stage transition: next block is twice as wide
    (1, 16, 8, 64, 64, 64, False),       # ONE tile per CTA, one chunk per tile (flush path), no residual
    (2, 19, 19, 64, 128, 64, True),      # ragged tile rows
    (40, 16, 16, 64, 256, 64, True),     # 320 tiles on 148 CTAs: CTAs with 2 and 3 tiles
]


@pytest.mark.parametrize("case", PAIR_CASES)
def test_conv1x1_pair_bit_identical_to_two_launches(K, case):
    """conv_pair.cu: conv3(+residual+ReLU) and the next conv1(+ReLU) fused; y1 and y2 must be the very
    same bf16 values two separate launches produce (same K-block order, y1 round-trips through bf16)."""
    N, H, W, Cin, Cmid, Cout2, use_res = case
    g = torch.Generator().manual_seed(hash(case) % (2 ** 31))
    x = torch.randn((N, H, W, Cin), generator=g).to(torch.bfloat16).cuda()
    w1 = K.pack_weight(torch.randn((Cmid, Cin, 1, 1), generator=g) / np.sqrt(Cin)).cuda()
    w2 = K.pack_weight(torch.randn((Cout2, Cmid, 1, 1), generator=g) / np.sqrt(Cmid)).cuda()
    b1 = torch.randn((Cmid,), generator=g).cuda()
    b2 = torch.randn((Cout2,), generator=g).cuda()
    res = torch.randn((N, H, W, Cmid), generator=g).to(torch.bfloat16).cuda() if use_res else None
    r1 = K.conv2d(x, w1, b1, 1, 1, 1, 0, True, res)
    r2 = K.conv2d(r1, w2, b2, 1, 1, 1, 0, True)
    for _ in range(3):                      # repeated: a stale-read race would show up as flakiness
        y1 = torch.full_like(r1, float("nan"))
        y2 = torch.full_like(r2, float("nan"))
        K.conv1x1_pair(x, w1, b1, True, res, w2, b2, True, out1=y1, out2=y2)
        torch.cuda.synchronize()
        assert torch.equal(y1, r1)
        assert torch.equal(y2, r2)
