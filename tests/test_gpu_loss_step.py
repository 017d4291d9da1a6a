"""The one-launch training-step loss (csrc/loss_step.cu, `pipeline.fused_loss_step`) vs
  (a) the reference-pinned oracle run the long way (oracle/box_oracle.py: extract_targets per level + the
      criterion + the caller's masks / normalisation, pipeline_anchor_basic.py:62-97),
  (b) the per-level kernels it replaces (ssdsb_match_iou + ssdsb_multibox_loss_sum / focal / loc sums), and
  (c) itself: determinism, CUDA-graph capture, optional depth / box_target outputs.
Bars: depth and positive counts bit-exact (integer-valued matching); box_target to the match kernel's own bar
(bit-identical: same code); loss scalars 3e-4 relative vs the oracle (fp32 sums of ~1e5 terms; the GPU BCE uses a
log1p polynomial with 2.3e-7 relative error — hard negatives at the selection cut may swap, which moves the sum
by < 1e-7 relative)."""
from collections import OrderedDict

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def P():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    from ssds_pytorch_b200 import pipeline
    return pipeline


def make_targets(rng, B_, T, ncls, img):
    tg = np.full((B_, T, 5), -1, np.float32)
    for b_ in range(B_):
        n = int(rng.integers(1, T + 1))
        tg[b_, :n, :2] = rng.uniform(0, img * 0.75, (n, 2))
        tg[b_, :n, 2:4] = rng.uniform(16, 256, (n, 2))
        tg[b_, :n, 4] = rng.integers(0, ncls, n)
    return tg


def setup(seed, Bn, C, levels, T, img, scales=(4.0, 5.04, 6.35)):
    from oracle import box_oracle as O
    rng = np.random.default_rng(seed)
    anchors = OrderedDict((s, O.generate_anchors(s, [1, 2, 0.5], list(scales))) for s, _ in levels)
    A = len(scales) * 3
    tg = make_targets(rng, Bn, T, C, img)
    conf = [rng.normal(-4.6, 1.0, (Bn, A * C, hw, hw)).astype(np.float32) for _, hw in levels]
    loc = [rng.normal(0, 0.5, (Bn, A * 4, hw, hw)).astype(np.float32) for _, hw in levels]
    tanc = OrderedDict((s, torch.from_numpy(a).cuda()) for s, a in anchors.items())
    return rng, anchors, tanc, tg, conf, loc, A


def oracle_step(O, anchors, levels, tg, conf, loc, Bn, A, C, cls, ty, ratio=3):
    ecs = els = 0.0
    efg = 0
    per = []
    for (s, hw), c, l in zip(levels, conf, loc):
        cls_t, box_t, dep = O.extract_targets(tg, anchors, C, s, (hw, hw), [0.5, 0.4])
        if cls == "MultiBoxLoss":
            sums, npos = O.multibox_loss_reduced(c.reshape(Bn, A, C, hw, hw), cls_t, dep, ratio)
            lsum = np.zeros(Bn)
            if ty is not None:
                lv = O.loc_loss(l.reshape(Bn, A, 4, hw, hw), box_t, ty)
                _, lsum, _ = O.masked_loss_sums(np.zeros_like(cls_t), lv, dep)
        else:
            f = O.focal_loss(c.reshape(Bn, A, C, hw, hw), cls_t)
            lv = O.loc_loss(l.reshape(Bn, A, 4, hw, hw), box_t, ty or "smoothl1")
            sums, lsum, npos = O.masked_loss_sums(f, lv, dep)
            if ty is None:
                lsum = np.zeros(Bn)
        ecs += sums.sum()
        els += lsum.sum()
        efg += max(int(npos.sum()), 1)
        per.append((sums, lsum, npos, dep, box_t))
    return ecs / efg, els / efg, efg, per


@pytest.mark.parametrize("cls,ty", [("MultiBoxLoss", None), ("MultiBoxLoss", "smoothl1"), ("FocalLoss", "smoothl1"),
                                    ("FocalLoss", "giou"), ("MultiBoxLoss", "ciou"), ("FocalLoss", "diou"),
                                    ("FocalLoss", "iou")])
def test_fused_step_vs_oracle_pipeline(P, cls, ty):
    from oracle import box_oracle as O
    Bn, C = 3, 20
    levels = [(8, 20), (16, 10), (32, 5)]
    _, anchors, tanc, tg, conf, loc, A = setup(77, Bn, C, levels, 12, 160)
    tg[1, 2:] = -1                                     # an image with two targets only
    names = {None: None, "smoothl1": "SmoothL1Loss", "iou": "IOULoss", "giou": "GIOULoss", "diou": "DIOULoss",
             "ciou": "CIOULoss"}
    sc, parts = P.fused_loss_step([torch.from_numpy(x).cuda() for x in loc], [torch.from_numpy(x).cuda() for x in conf],
                                  torch.from_numpy(tg).cuda(), tanc, C, cls, names[ty], with_targets=True)
    torch.cuda.synchronize()
    ecl, ell, efg, per = oracle_step(O, anchors, levels, tg, conf, loc, Bn, A, C, cls, ty)
    sc = sc.cpu().numpy()
    assert efg > 3 and sc[2] == efg
    np.testing.assert_allclose(sc[0], ecl, rtol=3e-4)
    if ty is not None:
        np.testing.assert_allclose(sc[1], ell, rtol=3e-4)
    else:
        assert sc[1] == 0.0
    for li, (sums, lsum, npos, dep, box_t) in enumerate(per):
        np.testing.assert_array_equal(parts["num_pos"][li].cpu().numpy(), npos.astype(np.float32))
        np.testing.assert_array_equal(parts["depth"][li].cpu().numpy(), dep)
        np.testing.assert_allclose(parts["box_target"][li].cpu().numpy(), box_t, rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(parts["cls_sum"][li].cpu().numpy(), sums, rtol=3e-4, atol=1e-5)
        if ty is not None:
            np.testing.assert_allclose(parts["loc_sum"][li].cpu().numpy(), lsum, rtol=3e-4, atol=1e-5)


def test_fused_step_cfg4_geometry_vs_per_level_kernels(P):
    """SSDFPN-ResNet50 640^2 geometry (5 levels, A=9, C=80, 76 725 anchors per image, T=32), 4 images, one of
    them without targets and one with a single target: vs extract_targets + MultiBoxLoss.forward_sum per level
    (the kernels parity-tested against the reference goldens in test_gpu_box_ops.py)."""
    import ssds_pytorch_b200 as S
    Bn, C = 4, 80
    levels = [(8, 80), (16, 40), (32, 20), (64, 10), (128, 5)]
    _, anchors, tanc, tg, conf, loc, A = setup(4321, Bn, C, levels, 32, 640)
    tg[2, :, :] = -1                                   # empty image: depth 0 everywhere, no positives -> no negatives
    tg[3, 1:] = -1
    tgc = torch.from_numpy(tg).cuda()
    confc = [torch.from_numpy(x).cuda() for x in conf]
    locc = [torch.from_numpy(x).cuda() for x in loc]
    sc, parts = P.fused_loss_step(locc, confc, tgc, tanc, C, "MultiBoxLoss", "SmoothL1Loss", with_targets=True)
    crit, lcrit = S.MultiBoxLoss(3), S.SmoothL1Loss(0.11)
    tot = ltot = 0.0
    fg = 0.0
    for li, ((s, hw), c, l) in enumerate(zip(levels, confc, locc)):
        _, box_t, dep = S.extract_targets(tgc, tanc, C, s, (hw, hw), [0.5, 0.4], with_cls_target=False)
        ls, npos = crit.forward_sum(c.view(Bn, A, C, hw, hw), dep)
        lsum = lcrit.forward_sum(l.view(Bn, A, 4, hw, hw), box_t, dep)
        assert torch.equal(parts["depth"][li], dep)
        assert torch.equal(parts["box_target"][li], box_t)
        assert torch.equal(parts["num_pos"][li], npos)
        np.testing.assert_allclose(parts["cls_sum"][li].cpu().numpy(), ls.cpu().numpy(), rtol=2e-5, atol=1e-6)
        np.testing.assert_allclose(parts["loc_sum"][li].cpu().numpy(), lsum.cpu().numpy(), rtol=2e-5, atol=1e-6)
        assert parts["cls_sum"][li][2].item() == 0.0 and parts["num_pos"][li][2].item() == 0.0
        tot += ls.double().sum().item()
        ltot += lsum.double().sum().item()
        fg += max(npos.sum().item(), 1.0)
    sc = sc.cpu().numpy()
    np.testing.assert_allclose(sc[0], tot / fg, rtol=2e-5)
    np.testing.assert_allclose(sc[1], ltot / fg, rtol=2e-5)
    assert sc[2] == fg
    # deterministic: a second launch gives the same bits; CUDA-graph capture replays the same bits
    sc2, _ = P.fused_loss_step(locc, confc, tgc, tanc, C, "MultiBoxLoss", "SmoothL1Loss")
    assert torch.equal(sc2.cpu(), torch.from_numpy(sc))
    out = torch.zeros(3, device="cuda")
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        P.fused_loss_step(locc, confc, tgc, tanc, C, "MultiBoxLoss", "SmoothL1Loss", out=out)     # warm-up on st
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=st):
            P.fused_loss_step(locc, confc, tgc, tanc, C, "MultiBoxLoss", "SmoothL1Loss", out=out)
    out.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out.cpu(), torch.from_numpy(sc))


def test_fused_step_many_targets_and_negpos_clamp(P):
    """T = 150 (second staging chunk) and a negpos_ratio so large that ratio * num_pos exceeds N - 1 (the clamp of
    criterion.py:65: every anchor but one ranks as a hard negative, zeros included, in index order)."""
    from oracle import box_oracle as O
    Bn, C = 2, 6
    levels = [(16, 12)]
    rng, anchors, tanc, tg, conf, loc, A = setup(5, Bn, C, levels, 150, 192, scales=(2.0, 2.828))
    tg[:, :, 2:4] = np.where(tg[:, :, 2:4] > 0, np.minimum(tg[:, :, 2:4], 64.0), tg[:, :, 2:4])
    for ratio in (3, 60):
        sc, parts = P.fused_loss_step([torch.from_numpy(x).cuda() for x in loc], [torch.from_numpy(x).cuda() for x in conf],
                                      torch.from_numpy(tg).cuda(), tanc, C, "MultiBoxLoss", None, negpos_ratio=ratio,
                                      with_targets=True)
        ecl, _, efg, per = oracle_step(O, anchors, levels, tg, conf, loc, Bn, A, C, "MultiBoxLoss", None, ratio)
        np.testing.assert_array_equal(parts["depth"][0].cpu().numpy(), per[0][3])
        np.testing.assert_array_equal(parts["num_pos"][0].cpu().numpy(), per[0][2].astype(np.float32))
        N = A * 12 * 12
        if ratio == 60:
            assert (ratio * per[0][2] > N - 1).all() and (per[0][2] > 0).all(), "case must exercise the num_neg clamp"
        np.testing.assert_allclose(parts["cls_sum"][0].cpu().numpy(), per[0][0], rtol=3e-4)
        np.testing.assert_allclose(sc.cpu().numpy()[0], ecl, rtol=3e-4)


def test_loss_step_host_api_matches_device_path(P):
    """pipeline.LossStep: pinned host batch -> loss scalars on the host == fused_loss_step on the model's own
    training-mode outputs."""
    from ssds_pytorch_b200 import synth
    fl = [[3, 4, 5, "Conv:S"], [128, 256, 512, 256]]
    cfg = {"MODEL": {"SSDS": "SSD", "NETS": "ResNet18", "IMAGE_SIZE": [160, 160], "NUM_CLASSES": 20,
                     "FEATURE_LAYER": fl, "SIZES": [[2.0, 2.828]] * 4, "ASPECT_RATIOS": [[1, 2, 0.5]] * 4},
           "DATASET": {"PREPROC": {"MEAN": 0, "STD": 255}}}
    sd = synth.synthetic_state_dict("ResNet18", fl, [6] * 4, 20, seed=3, style="test")
    step = P.LossStep(cfg, sd, use_graph=False, cls_criterion="FocalLoss", loc_criterion="SmoothL1Loss")
    g = torch.Generator().manual_seed(9)
    x = torch.randint(0, 256, (3, 160, 160, 3), generator=g, dtype=torch.uint8)
    tg = synth.synthetic_targets(3, T=8, seed=2)
    tg[..., :4] *= 0.25
    out = step.loss_host(x.pin_memory(), tg.pin_memory())
    step.sync()
    got = out.clone()
    loc, conf = step.model(x.cuda())
    sc, _ = P.fused_loss_step(loc, conf, tg.cuda(), step.anchors, 20, "FocalLoss", "SmoothL1Loss")
    assert torch.equal(got, sc.cpu()) and got[2] >= 4 and torch.isfinite(got).all()


@pytest.mark.parametrize("pinned", [True, False])
def test_loss_step_host_api_pipelined_batches(P, pinned):
    """[r2] loss_host overlaps the H2D copy of call i with the step of call i-1 (copy stream, two staging sets):
    five different batches issued back to back without a sync give exactly the per-batch results of the synchronous
    device path, from pinned and from pageable host buffers (the caller reuses ONE pageable buffer: the call must not
    return before that source has been consumed)."""
    from ssds_pytorch_b200 import synth
    fl = [[3, 4, 5, "Conv:S"], [128, 256, 512, 256]]
    cfg = {"MODEL": {"SSDS": "SSD", "NETS": "ResNet18", "IMAGE_SIZE": [160, 160], "NUM_CLASSES": 20,
                     "FEATURE_LAYER": fl, "SIZES": [[2.0, 2.828]] * 4, "ASPECT_RATIOS": [[1, 2, 0.5]] * 4},
           "DATASET": {"PREPROC": {"MEAN": 0, "STD": 255}}}
    sd = synth.synthetic_state_dict("ResNet18", fl, [6] * 4, 20, seed=3, style="test")
    step = P.LossStep(cfg, sd, use_graph=True)
    g = torch.Generator().manual_seed(10)
    xs = [torch.randint(0, 256, (3, 160, 160, 3), generator=g, dtype=torch.uint8) for _ in range(5)]
    tgs = []
    for i in range(5):
        t = synth.synthetic_targets(3, T=8, seed=20 + i)
        t[..., :4] *= 0.25
        tgs.append(t)
    want = []
    for x, t in zip(xs, tgs):
        want.append(step.loss_device(x.cuda(), t.cuda()).cpu().clone())
    outs = []
    if pinned:
        for x, t in zip(xs, tgs):
            outs.append(step.loss_host(x.pin_memory(), t.pin_memory()))
            if len(outs) >= 2:                      # the result tensors alternate between two pinned buffers
                step.sync()
                outs[-2] = outs[-2].clone()
    else:
        hx, ht = torch.empty_like(xs[0]), torch.empty_like(tgs[0])
        for x, t in zip(xs, tgs):
            hx.copy_(x)
            ht.copy_(t)
            outs.append(step.loss_host(hx, ht))
            step.sync()
            outs[-1] = outs[-1].clone()
    step.sync()
    for o, w in zip(outs, want):
        assert torch.equal(o.clone(), w)
    assert len({tuple(w.tolist()) for w in want}) == 5


def test_fused_step_at_cfg4_bench_shape(P):
    """What bench.py times for cfg4: LossStep(cfg4) at B=16 on the init-style weights (logits clustered around the
    -4.595 prior bias), the engine's own training-mode logits, the bench targets.  vs extract_targets +
    MultiBoxLoss.forward_sum per level (depth and num_pos bit-exact, cls_sum 2e-5) and, for one image, vs the numpy
    oracle (the file's 3e-4 bar)."""
    import bench
    import ssds_pytorch_b200 as S
    from oracle import box_oracle as O
    from ssds_pytorch_b200 import synth
    from ssds_pytorch_b200.model import number_box_from_cfg
    cfg = bench.cfg_dict("cfg4")
    m = cfg["MODEL"]
    Bn, C = 16, m["NUM_CLASSES"]
    nb = number_box_from_cfg(m)
    assert nb == [9] * 5
    sd = synth.synthetic_state_dict(m["NETS"], m["FEATURE_LAYER"], nb, C, seed=0, style="init", ssds=m["SSDS"])
    step = P.LossStep(cfg, sd, use_graph=False)
    H, W = m["IMAGE_SIZE"]
    x = torch.randint(0, 256, (Bn, H, W, 3), generator=torch.Generator().manual_seed(1234), dtype=torch.uint8).cuda()
    tg = synth.synthetic_targets(Bn, seed=4321).cuda()
    loc, conf = step.model(x)
    sc, parts = P.fused_loss_step(loc, conf, tg, step.anchors, C, "MultiBoxLoss", None, with_targets=True)
    torch.cuda.synchronize()
    assert torch.equal(sc, step.loss_device(x, tg)), "LossStep.loss_device differs from fused_loss_step"
    crit = S.MultiBoxLoss(3)
    tot, fg = 0.0, 0.0
    for li, ((s, anc), c) in enumerate(zip(step.anchors.items(), conf)):
        hh, ww = c.shape[-2:]
        A = anc.shape[0]
        _, _, dep = S.extract_targets(tg, step.anchors, C, s, (hh, ww), [0.5, 0.4], with_cls_target=False)
        ls, npos = crit.forward_sum(c.view(Bn, A, C, hh, ww), dep)
        assert torch.equal(parts["depth"][li], dep)
        assert torch.equal(parts["num_pos"][li], npos)
        np.testing.assert_allclose(parts["cls_sum"][li].cpu().numpy(), ls.cpu().numpy(), rtol=2e-5, atol=1e-6)
        tot += ls.double().sum().item()
        fg += max(npos.sum().item(), 1.0)
    sc = sc.cpu().numpy()
    print(f"cfg4 loss step B={Bn}: cls_loss {sc[0]:.6f}, fg {sc[2]:.0f}, logits in "
          f"[{min(c.min().item() for c in conf):.3f}, {max(c.max().item() for c in conf):.3f}]")
    assert sc[2] == fg and fg > Bn
    np.testing.assert_allclose(sc[0], tot / fg, rtol=2e-5)
    # one image through the numpy oracle
    i = 5
    anchors = OrderedDict((s, a.cpu().numpy()) for s, a in step.anchors.items())
    tgi = tg[i:i + 1].cpu().numpy()
    for li, ((s, anc), c) in enumerate(zip(anchors.items(), conf)):
        hh, ww = c.shape[-2:]
        A = anc.shape[0]
        cls_t, _, dep = O.extract_targets(tgi, anchors, C, s, (hh, ww), [0.5, 0.4])
        sums, npos = O.multibox_loss_reduced(c[i:i + 1].cpu().numpy().reshape(1, A, C, hh, ww), cls_t, dep, 3)
        np.testing.assert_array_equal(parts["depth"][li][i:i + 1].cpu().numpy(), dep)
        assert parts["num_pos"][li][i].item() == npos[0]
        np.testing.assert_allclose(parts["cls_sum"][li][i].item(), sums[0], rtol=3e-4)


# 16 well-separated values for a negative anchor's largest logit: equal values make exact ties in the hard-negative
# rank key (max over classes of BCE(x, 0) = softplus(max x)); every other logit of the anchor lies 0.5 - 6 below it,
# so tied anchors have different CE sums and which of them the cut takes changes the loss
TIE_LEVELS = np.arange(16, dtype=np.float32) * np.float32(0.25) - np.float32(3.0)


def tie_case(seed):
    """(anchors, levels, targets, conf, depth per level, cls target per level) with the max logits drawn from TIE_LEVELS"""
    from oracle import box_oracle as O
    Bn, C = 2, 20
    levels = [(8, 20), (16, 10), (32, 5)]
    rng, anchors, tanc, tg, _, loc, A = setup(seed, Bn, C, levels, 6, 160)
    for b in range(Bn):                    # two boxes per image at the anchor size of each level: positives everywhere
        for k, (s, _) in enumerate(levels * 2):
            wh = s * rng.uniform(3.5, 4.6, 2)
            tg[b, k, :2] = rng.uniform(0, 160 - wh)
            tg[b, k, 2:4] = wh
            tg[b, k, 4] = rng.integers(0, C)
    conf, deps, clss = [], [], []
    for s, hw in levels:
        top = rng.choice(TIE_LEVELS, size=(Bn, A, 1, hw, hw))
        other = top - rng.uniform(0.5, 6.0, (Bn, A, C, hw, hw)).astype(np.float32)
        arg = rng.integers(0, C, (Bn, A, 1, hw, hw))
        c = np.where(np.arange(C).reshape(1, 1, C, 1, 1) == arg, top, other).astype(np.float32)
        conf.append(c.reshape(Bn, A * C, hw, hw))
        cls_t, _, dep = O.extract_targets(tg, anchors, C, s, (hw, hw), [0.5, 0.4])
        deps.append(dep)
        clss.append(cls_t)
    return anchors, tanc, levels, tg, conf, loc, deps, clss, Bn, A, C


def reduced_with_tiebreak(c5, dep, ratio, reverse):
    """O.multibox_loss_reduced's per-image sums with the rank ties broken by ascending (the criterion's stable sort)
    or descending index; also the size of the tie group at the cut and how many of it are taken."""
    from oracle import box_oracle as O
    ce = O.bce_with_logits(c5, np.zeros_like(c5))          # negatives only carry the key; positives are added below
    out = []
    for b in range(c5.shape[0]):
        key = ce[b].max(axis=1).reshape(-1).copy()
        d = dep[b].reshape(-1)
        key[d != 0] = 0
        idx = np.arange(key.size)
        order = np.lexsort((-idx if reverse else idx, -key.astype(np.float64)))
        num_neg = min(ratio * int((d > 0).sum()), key.size - 1)
        neg = np.zeros(key.size, bool)
        neg[order[:num_neg]] = True
        cut = key[order[num_neg - 1]]
        group = int((key == cut).sum())
        taken = int((key[order[:num_neg]] == cut).sum())
        out.append((neg, cut, group, taken, key[order[num_neg]]))
    return out


def test_hard_negative_selection_breaks_ties_by_index(P):
    """The hard-negative cut falls INSIDE a group of exactly equal rank keys in every (image, level): which of the tied
    anchors are taken (the lower indices, criterion.py's stable descending sort) decides the loss.
      * MultiBoxLoss.forward's mask (out != 0) == O.multibox_loss's mask, exactly;
      * the fused step's per-pair cls_sum and MultiBoxLoss.forward_sum == O.multibox_loss_reduced within 5e-6: the
        fast softplus has 2.3e-7 relative error per term and fp32 partial sums of a few thousand positive terms
        add < 1e-6, so 5e-6 is ample for a correct kernel;
      * the oracle with the REVERSED tie-break (higher index first) is at least 10x that tolerance away in every
        pair, so a kernel that cuts the tie group at the wrong end cannot pass."""
    import ssds_pytorch_b200 as S
    from oracle import box_oracle as O
    rtol = 5e-6
    anchors, tanc, levels, tg, conf, loc, deps, clss, Bn, A, C = tie_case(1)
    sc, parts = P.fused_loss_step([torch.from_numpy(x).cuda() for x in loc], [torch.from_numpy(x).cuda() for x in conf],
                                  torch.from_numpy(tg).cuda(), tanc, C, "MultiBoxLoss", None, with_targets=True)
    crit = S.MultiBoxLoss(3)
    for li, ((s, hw), c, dep, cls_t) in enumerate(zip(levels, conf, deps, clss)):
        c5 = c.reshape(Bn, A, C, hw, hw)
        want, npos = O.multibox_loss_reduced(c5, cls_t, dep, 3)
        ce = O.bce_with_logits(c5, cls_t)
        cuts = reduced_with_tiebreak(c5, dep, 3, reverse=False)
        cuts_r = reduced_with_tiebreak(c5, dep, 3, reverse=True)
        for b in range(Bn):
            neg, cut, group, taken, nxt = cuts[b]
            assert nxt == cut and 0 < taken < group, f"level {li} image {b}: the cut is not inside a tie group"
            m_r = (dep[b] > 0) | cuts_r[b][0].reshape(dep[b].shape)
            sum_r = (ce[b] * m_r * (dep[b] >= 0)).astype(np.float64).sum()
            margin = abs(sum_r - want[b]) / abs(want[b])
            print(f"level {li} image {b}: num_pos {npos[b]}, tie group of {group} at key {cut:.6f}, {taken} taken; "
                  f"reversed tie-break moves the sum by {margin:.2e} (tolerance {rtol:.0e})")
            assert margin >= 10 * rtol
        # the unreduced drop-in: same mask
        mask_o = O.multibox_loss(c5, cls_t, dep, 3) != 0
        out = crit(torch.from_numpy(c5).cuda(), torch.from_numpy(cls_t).cuda(), torch.from_numpy(dep).cuda())
        mask_g = (out != 0).cpu().numpy()
        assert (mask_g == mask_o).all(), f"level {li}: {int((mask_g != mask_o).sum())} mask elements differ"
        ls, npos_g = crit.forward_sum(torch.from_numpy(c5).cuda(), torch.from_numpy(dep).cuda())
        np.testing.assert_array_equal(npos_g.cpu().numpy(), npos.astype(np.float32))
        np.testing.assert_array_equal(parts["depth"][li].cpu().numpy(), dep)
        np.testing.assert_allclose(ls.cpu().numpy(), want, rtol=rtol)
        np.testing.assert_allclose(parts["cls_sum"][li].cpu().numpy(), want, rtol=rtol)
