"""Drop-in checks against what the unmodified reference package computes, stored by
tests/golden/make_golden_reference.py in tests/golden/reference_dropin.npz (inputs and weights are rebuilt here
from their seeds):

  1. the seam: the reference's `Decoder` call sequence (ssds/modeling/layers/decoder.py:25-49: per-level decode,
     concatenation, nms) with `box.decode` / `box.nms` routed through `ssds._C` exactly as INTEGRATION.md's
     two-line patch does (box.py:419-421, :483-485), on GPU tensors, vs the reference's own Decoder on the CPU:
     classes / keep order bit-exact, scores 2e-6, boxes 1e-4;
  2. experiments/cfgs/tests/test.yml AS SHIPPED (YOLOV3 + ResNet18 @320, BASELINE configs[0] plumbing) end to end:
     `ssds_pytorch_b200.SSDDetector` from the yml + a state_dict in the reference's layout vs the reference's
     `create_model` + `Decoder` on the same weights and image (bf16 conv stack: detections matched noise-aware);
  3. cfg 1b (SSD + MobileNetV2 @300, the other plumbing config) and YOLOV4, same way;
  4. checkpoint -> detector -> mAP, scored like the reference's `MeanAveragePrecision`.
"""
import os
from collections import OrderedDict

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

SEAM_DECODER = (0.05, 0.6, 100, 300, True, True)    # conf thr, nms thr, top_n, top_n per level, rescore, DIoU
PLUMBING = ["test.yml", "cfg1b", "yolov4"]
ROUND_TRIP_MODEL = dict(SSDS="SSD", NETS="ResNet18", IMAGE_SIZE=[192, 192], NUM_CLASSES=20,
                        FEATURE_LAYER=[[3, 4, 5, "Conv:S"], [128, 256, 512, 256]],
                        SIZES=[[2.0, 2.828]] * 4, ASPECT_RATIOS=[[1, 2, 0.5]] * 4)
MAP_ARGS = (20, 0.01, 0.5)                            # classes, conf threshold, IoU threshold
N_MAP_PINS = 4


def seam_inputs():
    return 3, 6, 80, [(8, 20, 24), (16, 10, 12), (32, 5, 6)], np.random.default_rng(7)


def seam_tensors(B, A, C, levels, rng):
    conf, loc = [], []
    for s, h, w in levels:
        n = B * A * C * h * w
        conf.append(torch.from_numpy(((rng.permutation(n) + 0.5) / n * 0.3).astype(np.float32).reshape(B, A * C, h, w)))
        loc.append(torch.from_numpy(rng.normal(0, 0.5, (B, A * 4, h, w)).astype(np.float32)))
    return conf, loc


def plumbing_cfg(which):
    if which == "test.yml":
        import yaml
        with open(os.path.join(GOLDEN_DIR, "reference_test.yml")) as f:
            return yaml.safe_load(f)
    if which == "yolov4":
        # [r2] the SPP + PAN neck (yolo.py:161-392) with one 'Conv:S' extra level
        return {"MODEL": dict(SSDS="YOLOV4", NETS="ResNet18", IMAGE_SIZE=[256, 320], NUM_CLASSES=20,
                              FEATURE_LAYER=[[3, 4, 5, "Conv:S"], [128, 256, 512, 256]],
                              SIZES=[[2.0, 2.828]] * 4, ASPECT_RATIOS=[[1, 2, 0.5]] * 4)}
    return {"MODEL": dict(SSDS="SSD", NETS="MobileNetV2", IMAGE_SIZE=[300, 300], NUM_CLASSES=80,
                          FEATURE_LAYER=[[5, 7, "Conv:S", "Conv:S", "Conv:S", "Conv:S"], [96, 320, 512, 256, 256, 128]],
                          SIZES=[[2.0, 2.828]] * 6, ASPECT_RATIOS=[[1, 2, 0.5]] * 6)}


def _weights(model_cfg, seed, style):
    from ssds_pytorch_b200 import synth
    from ssds_pytorch_b200.model import number_box_from_cfg
    return synth.synthetic_state_dict(model_cfg["NETS"], model_cfg["FEATURE_LAYER"], number_box_from_cfg(model_cfg),
                                      model_cfg["NUM_CLASSES"], seed=seed, style=style, ssds=model_cfg["SSDS"])


def plumbing_weights_and_images(model_cfg, init_mean, init_std):
    """A state_dict in the reference's layout, each tensor drawn at the mean and spread the reference's own
    initialisation gives it (`init_mean` / `init_std`, one per key, stored with the golden data), with non-trivial
    BN statistics so that folding is exercised; two uint8 NHWC images."""
    from ssds_pytorch_b200 import synth
    from ssds_pytorch_b200.model import number_box_from_cfg
    shapes = synth.model_shapes(model_cfg["SSDS"], model_cfg["NETS"], model_cfg["FEATURE_LAYER"],
                                number_box_from_cfg(model_cfg), model_cfg["NUM_CLASSES"])
    assert len(shapes) == len(init_mean) == len(init_std)
    g = torch.Generator().manual_seed(5)
    sd = OrderedDict()
    for (k, shape), m, sd_k in zip(shapes, init_mean.tolist(), init_std.tolist()):
        if k.endswith("num_batches_tracked"):
            sd[k] = torch.tensor(0, dtype=torch.long)
        elif k.endswith("running_mean"):
            sd[k] = torch.randn(shape, generator=g) * 0.1
        elif k.endswith("running_var"):
            sd[k] = torch.rand(shape, generator=g) + 0.5
        else:
            sd[k] = m + sd_k * torch.randn(shape, generator=g)
    H, W = model_cfg["IMAGE_SIZE"]
    return sd, torch.randint(0, 256, (2, H, W, 3), generator=g, dtype=torch.uint8)


def round_trip_weights_and_images():
    sd = _weights(ROUND_TRIP_MODEL, 3, "init")
    g = torch.Generator().manual_seed(8)
    for k in sd:
        if k.endswith("running_mean"):
            sd[k] = torch.randn(sd[k].shape, generator=g) * 0.1
        elif k.endswith("running_var"):
            sd[k] = torch.rand(sd[k].shape, generator=g) + 0.5
        elif k.startswith("conf.") and k.endswith("weight"):
            sd[k] = torch.randn(sd[k].shape, generator=g) * 0.012     # spread the scores: a non-trivial ranking
        elif k.startswith("loc.") and k.endswith("weight"):
            sd[k] = torch.randn(sd[k].shape, generator=g) * 0.0005    # small deltas: boxes stay inside the image
    return sd, torch.randint(0, 256, (4, 192, 192, 3), generator=g, dtype=torch.uint8)


def round_trip_targets(dets):
    """The reference's 12 most confident detections per image play the annotated objects."""
    return [np.concatenate([dets[1][i, :12], dets[2][i, :12, None]], 1) for i in range(dets[0].shape[0])]


@pytest.fixture(scope="module")
def gold():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    return np.load(os.path.join(GOLDEN_DIR, "reference_dropin.npz"))


def test_reference_decoder_through_the_C_seam(gold):
    import sys
    import types
    import ssds_pytorch_b200 as S
    B, A, C, levels, rng = seam_inputs()
    anchors = OrderedDict((s, torch.from_numpy(gold[f"seam_anchors{i}"])) for i, (s, _, _) in enumerate(levels))
    conf, loc = seam_tensors(B, A, C, levels, rng)

    # INTEGRATION.md: `from ssds._C import decode as decode_cuda, nms as nms_cuda` + the two call sites
    pkg = types.ModuleType("ssds")                            # stands in for the reference package
    try:
        _C = S.install(pkg)
        assert pkg._C is _C and sys.modules["ssds._C"] is _C  # export.py:134-139 feature flag
    finally:
        sys.modules.pop("ssds._C", None)

    def decode_patched(all_cls_head, all_box_head, stride=1, threshold=0.05, top_n=1000, anchors=None, rescore=True):
        return _C.decode(all_cls_head.float(), all_box_head.float(), anchors.view(-1).tolist(), stride, threshold,
                         top_n, rescore)

    def nms_patched(all_scores, all_boxes, all_classes, nms=0.5, ndetections=100, using_diou=True):
        return _C.nms(all_scores.float(), all_boxes.float(), all_classes.float(), nms, ndetections, using_diou)

    thr, nms_thr, top_n, per_level, rescore, diou = SEAM_DECODER
    decoded = [decode_patched(c.cuda(), l.cuda(), s, thr, per_level, a, rescore=rescore)
               for l, c, (s, a) in zip(loc, conf, anchors.items())]
    decoded = [torch.cat(t, 1) for t in zip(*decoded)]
    got = nms_patched(*decoded, nms_thr, top_n, using_diou=diou)
    torch.cuda.synchronize()
    gs, gb, gc = [t.cpu().numpy() for t in got]
    want = gold["seam_scores"], gold["seam_boxes"], gold["seam_classes"]
    assert (want[0] > 0).sum() > 50
    np.testing.assert_array_equal(gc, want[2])
    np.testing.assert_allclose(gs, want[0], rtol=0, atol=2e-6)
    np.testing.assert_allclose(gb, want[1], rtol=0, atol=1e-4)


def _match(s, b, c, rs, rb, rc, px=1.5, rel=0.05):
    found = total = 0
    for i in range(rs.shape[0]):
        for j in range(rs.shape[1]):
            if rs[i, j] <= 0:
                continue
            total += 1
            m = (c[i] == rc[i, j]) & (np.abs(b[i] - rb[i, j]).max(axis=1) <= px) & \
                (np.abs(s[i] - rs[i, j]) <= rel * rs[i, j] + 1e-5)
            found += bool(m.any())
    return found, total


@pytest.mark.parametrize("which", PLUMBING)
def test_plumbing_config_end_to_end_vs_reference(gold, which):
    """BASELINE configs[0]: the reference's CPU plumbing config.  The state_dict has the reference's keys, shapes
    and init statistics and goes into SSDDetector unchanged; the reference ran its own create_model + Decoder on
    the same weights and images."""
    from ssds_pytorch_b200.ssds import SSDDetector
    cfg = plumbing_cfg(which)
    sd, img = plumbing_weights_and_images(cfg["MODEL"], gold[f"{which}_init_mean"], gold[f"{which}_init_std"])
    rs, rb, rc = gold[f"{which}_scores"], gold[f"{which}_boxes"], gold[f"{which}_classes"]
    cfg["DATASET"] = {"PREPROC": {"MEAN": 0, "STD": 255}}
    det = SSDDetector(cfg, sd)
    assert list(det.anchors.keys()) == gold[f"{which}_strides"].tolist()
    for i, a in enumerate(det.anchors.values()):
        np.testing.assert_array_equal(a.cpu().numpy(), gold[f"{which}_anchors{i}"])
    s, b, c = det(img.numpy())                                 # the reference facade: numpy uint8 NHWC in, numpy out
    found, total = _match(s, b.astype(np.float32), c.astype(np.float32), rs, np.trunc(rb), rc)
    print(f"{which}: {found}/{total} reference detections reproduced by the bf16 engine")
    assert total > 20 and found >= 0.9 * total


def test_checkpoint_to_map_round_trip(gold, tmp_path):
    """SURVEY 8f-2's end-to-end check: a checkpoint as the reference's `save_checkpoints` writes it
    (ssds/core/checkpoint.py:18-34: the state_dict + one line in checkpoint_list.txt) ->
    `ssds_pytorch_b200.checkpoint.detector_from_checkpoint` -> detections -> mAP as the reference's
    `MeanAveragePrecision` (ssds/core/evaluation_metrics.py:5-142) scores them, next to the reference model +
    Decoder on the same weights, scored by the reference metric on the same synthetic ground truth.  The restated
    metric must reproduce the reference metric on the stored detection sets first.  bf16 conv stack: the two mAPs
    must agree within 0.05."""
    from oracle.box_oracle import mean_average_precision
    from ssds_pytorch_b200.checkpoint import detector_from_checkpoint, find_previous_checkpoint
    sd, img = round_trip_weights_and_images()
    d = str(tmp_path)
    path = os.path.join(d, "ssd_resnet18_synth_epoch_7.pth")
    torch.save(sd, path)
    with open(os.path.join(d, "checkpoint_list.txt"), "w") as f:
        f.write(str(gold["rt_index"]).replace("{dir}", d))
    cfg = {"MODEL": ROUND_TRIP_MODEL, "DATASET": {"PREPROC": {"MEAN": 0, "STD": 255}}}
    epochs, files = find_previous_checkpoint(d)                # the reference's checkpoint_list.txt index
    assert epochs == [7] and files == [path]
    det, report = detector_from_checkpoint(cfg, files[-1])
    assert report["resumed"] == len(sd) and not report["unresumed"]
    rdet = gold["rt_scores"], gold["rt_boxes"], gold["rt_classes"]
    targets = round_trip_targets(rdet)
    for p in ["rt"] + [f"pin{j}" for j in range(N_MAP_PINS)]:
        dets = gold[f"{p}_scores"], gold[f"{p}_boxes"], gold[f"{p}_classes"]
        assert mean_average_precision(dets, targets, *MAP_ARGS) == pytest.approx(float(gold[f"{p}_map"]), abs=1e-12), p
    s, b, c = det.detect_device(img.cuda())
    ours = s.cpu().numpy(), b.cpu().numpy(), c.cpu().numpy()
    maps = [float(gold["rt_map"]), mean_average_precision(ours, targets, *MAP_ARGS)]
    print(f"mAP (reference metric) of the reference detections {maps[0]:.4f} vs the B200 engine's {maps[1]:.4f}")
    assert maps[0] > 0.5 and abs(maps[0] - maps[1]) <= 0.05
