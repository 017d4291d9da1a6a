"""Golden data for the tests that compare with the reference package as a whole: its model builder, its
checkpoint files, its Decoder and its mAP metric.  Runs the reference's own code (CPU, fp32) where its source
tree is available; the tests only read what this script stores.

    SSDS_REFERENCE=<reference source tree> python tests/golden/make_golden_reference.py

Weights are seeded (`synth.synthetic_state_dict`, or drawn at the per-tensor statistics of the reference's own
init, which are stored too) and loaded into the reference's own `create_model`, so that the tests can rebuild them
without the reference.  Writes
  reference_state_dicts.json.gz  create_model(cfg).state_dict() keys + shapes per engine combination
                                 (tests/test_model_shapes_vs_reference_cpu.py), and what the reference's
                                 save_checkpoints / find_previous_checkpoint / resume_checkpoint do
                                 (tests/test_checkpoint_cpu.py)
  reference_dropin.npz           the reference's Decoder and end-to-end detections, and its mAP on stored
                                 detection sets (tests/test_gpu_dropin_vs_reference.py)
"""
import gzip
import json
import os
import sys
import tempfile
import warnings
from collections import OrderedDict

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(1, os.path.dirname(HERE))
warnings.filterwarnings("ignore")

from oracle import ref_runner                                 # noqa: E402
import test_checkpoint_cpu as TC                              # noqa: E402
import test_gpu_dropin_vs_reference as TD                     # noqa: E402
import test_model_shapes_vs_reference_cpu as TS               # noqa: E402

ref_runner.REF_DIR = os.environ.get("SSDS_REFERENCE", ref_runner.REF_DIR)
R = ref_runner.shim()
if not hasattr(np, "float"):
    np.float = float                  # numpy >= 1.24 removed the aliases evaluation_metrics.py:91,123 uses
if not hasattr(np, "NAN"):
    np.NAN = np.nan
from ssds.core import checkpoint as RCK                       # noqa: E402
from ssds.core.evaluation_metrics import MeanAveragePrecision  # noqa: E402
from ssds.modeling.layers import box as rbox                  # noqa: E402
from ssds.modeling.layers import decoder as rdec              # noqa: E402


def state_dict_tables():
    out = {}
    for name, (ssds, nets, fl) in TS.CASES.items():
        L = len(fl[0])
        model_cfg = dict(SSDS=ssds, NETS=nets, IMAGE_SIZE=[128, 128], NUM_CLASSES=20, FEATURE_LAYER=fl,
                         SIZES=[[2.0, 2.828]] * L, ASPECT_RATIOS=[[1, 2, 0.5]] * L)
        model = ref_runner.build_reference_model(model_cfg)[0]
        out[name] = [[k, list(v.shape)] for k, v in model.state_dict().items()]
    return out


def checkpoint_semantics():
    """save_checkpoints of a DataParallel model (`module.` keys), then resume_checkpoint into a fresh model per
    scope: which value each key of the result took (the checkpoint's, the fresh model's, or both when equal)."""
    model_cfg = TC.CFG["MODEL"]
    model = ref_runner.build_reference_model(model_cfg)[0]
    model.load_state_dict(TC._sd(TC.CKPT_SEED))
    out = {"scopes": {}}
    with tempfile.TemporaryDirectory() as d:
        RCK.save_checkpoints(torch.nn.DataParallel(model), d, TC.CKPT_PREFIX, TC.CKPT_EPOCH)
        out["index"] = open(os.path.join(d, "checkpoint_list.txt")).read().replace(d, "{dir}")
        epochs, files = RCK.find_previous_checkpoint(d)
        out["found"] = [epochs, [f.replace(d, "{dir}") for f in files]]
        saved = torch.load(files[-1])
        out["saved_keys"] = list(saved)
        for scope in TC.SCOPES:
            fresh = ref_runner.build_reference_model(model_cfg)[0]
            fresh.load_state_dict(TC._sd(TC.BASE_SEED))
            base = OrderedDict((k, v.clone()) for k, v in fresh.state_dict().items())
            RCK.resume_checkpoint(fresh, files[-1], scope)
            res = fresh.state_dict()
            src = {}
            for k, v in res.items():
                c, b = torch.equal(v, saved["module." + k]), torch.equal(v, base[k])
                assert c or b, k
                src[k] = "both" if c and b else "checkpoint" if c else "base"
            out["scopes"][scope] = {"keys": list(res), "source": src}
    return out


def seam_decoder(G):
    B, A, C, levels, rng = TD.seam_inputs()
    anchors = OrderedDict((s, rbox.generate_anchors(s, [1, 2, 0.5], [2.0, 2.828])) for s, _, _ in levels)
    conf, loc = TD.seam_tensors(B, A, C, levels, rng)
    want = rdec.Decoder(*TD.SEAM_DECODER)(loc, conf, anchors)
    for i, a in enumerate(anchors.values()):
        G[f"seam_anchors{i}"] = a.numpy()
    G["seam_scores"], G["seam_boxes"], G["seam_classes"] = [t.numpy() for t in want]
    print("seam: detections", int((want[0] > 0).sum()))


def plumbing(G):
    for which in TD.PLUMBING:
        model_cfg = TD.plumbing_cfg(which)["MODEL"]
        model, anchors, decoder, m = ref_runner.build_reference_model(model_cfg)
        init = [v.double() for v in model.state_dict().values()]          # the reference's own init, seed 0
        G[f"{which}_init_mean"] = np.asarray([float(v.mean()) for v in init])
        G[f"{which}_init_std"] = np.asarray([float(v.std()) if v.numel() > 1 else 0.0 for v in init])
        sd, img = TD.plumbing_weights_and_images(model_cfg, G[f"{which}_init_mean"], G[f"{which}_init_std"])
        model.load_state_dict(sd)
        model.eval()
        x = (img.float() / 255.0).permute(0, 3, 1, 2).contiguous()
        with torch.no_grad():
            rs, rb, rc = decoder(*model(x), anchors)
        G[f"{which}_strides"] = np.asarray(list(anchors.keys()))
        for i, a in enumerate(anchors.values()):
            G[f"{which}_anchors{i}"] = a.numpy()
        G[f"{which}_scores"], G[f"{which}_boxes"], G[f"{which}_classes"] = rs.numpy(), rb.numpy(), rc.numpy()
        print(which, "detections", int((rs > 0).sum()))


def reference_map(dets, targets):
    metric = MeanAveragePrecision(*TD.MAP_ARGS)
    metric([torch.as_tensor(d) for d in dets], [torch.as_tensor(t) for t in targets])
    return float(metric.get_results()[0])


def round_trip(G):
    model_cfg = TD.ROUND_TRIP_MODEL
    model, anchors, decoder, m = ref_runner.build_reference_model(model_cfg)
    sd, img = TD.round_trip_weights_and_images()
    model.load_state_dict(sd)
    model.eval()
    x = (img.float() / 255.0).permute(0, 3, 1, 2).contiguous()
    with torch.no_grad():
        rdet = [t.numpy() for t in decoder(*model(x), anchors)]
    with tempfile.TemporaryDirectory() as d:
        RCK.save_checkpoints(model, d, "ssd_resnet18_synth", 7)
        G["rt_index"] = np.asarray(open(os.path.join(d, "checkpoint_list.txt")).read().replace(d, "{dir}"))
    G["rt_scores"], G["rt_boxes"], G["rt_classes"] = rdet
    targets = TD.round_trip_targets(rdet)
    G["rt_map"] = np.float64(reference_map(rdet, targets))
    # the reference metric on perturbed copies (shifted boxes, reshuffled scores, relabelled classes, dropped
    # detections): pins the restated metric the test scores the B200 detections with
    rng = np.random.default_rng(17)
    for j in range(TD.N_MAP_PINS):
        s, b, c = (a.copy() for a in rdet)
        b += rng.normal(0, 4.0 * (j + 1), b.shape).astype(np.float32)
        s = np.where(s > 0, rng.permutation(s.ravel()).reshape(s.shape) if j % 2 else s * rng.uniform(0.5, 1.5, s.shape),
                     s).astype(np.float32)
        relabel = rng.random(c.shape) < 0.1 * (j + 1)
        c = np.where(relabel, rng.integers(0, 20, c.shape), c).astype(np.float32)
        s[rng.random(s.shape) < 0.1] = 0
        G[f"pin{j}_scores"], G[f"pin{j}_boxes"], G[f"pin{j}_classes"] = s, b, c
        G[f"pin{j}_map"] = np.float64(reference_map((s, b, c), targets))
    print("round trip: reference mAP", float(G["rt_map"]), "pins", [float(G[f"pin{j}_map"]) for j in range(TD.N_MAP_PINS)])


def main():
    tables = {"state_dicts": state_dict_tables(), "checkpoint": checkpoint_semantics()}
    with gzip.GzipFile(os.path.join(HERE, "reference_state_dicts.json.gz"), "wb", mtime=0) as f:
        f.write(json.dumps(tables, separators=(",", ":"), sort_keys=True).encode())
    G = {}
    seam_decoder(G)
    plumbing(G)
    round_trip(G)
    out = os.path.join(HERE, "reference_dropin.npz")
    np.savez_compressed(out, **G)
    print("wrote", out, os.path.getsize(out) // 1024, "KiB")


if __name__ == "__main__":
    main()
