"""Weight import (SURVEY 8f rank 2): ssds_pytorch_b200.checkpoint against the reference's own
ssds/core/checkpoint.py — a checkpoint laid out as the reference's `save_checkpoints` writes it, read back by our
`find_previous_checkpoint` / `load_checkpoint` and compared key by key with what the reference's
`resume_checkpoint` made of the same file (tests/golden/reference_state_dicts.json.gz, written by
tests/golden/make_golden_reference.py).
"""
import gzip
import json
import os
from collections import OrderedDict

import pytest
import torch

from ssds_pytorch_b200 import checkpoint as CK
from ssds_pytorch_b200 import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_state_dicts.json.gz")
FL = [[3, 4, 5, "Conv:S"], [128, 256, 512, 256]]
CFG = {"MODEL": {"SSDS": "SSD", "NETS": "ResNet18", "IMAGE_SIZE": [96, 160], "NUM_CLASSES": 20, "FEATURE_LAYER": FL,
                 "SIZES": [[2.0, 2.828]] * 4, "ASPECT_RATIOS": [[1, 2, 0.5]] * 4}}
# the reference round trip: weights of seed CKPT_SEED saved from a DataParallel model (`module.` keys) as
# <prefix>_epoch_<epoch>.pth, resumed into a model holding the weights of seed BASE_SEED under each scope
CKPT_SEED, BASE_SEED, CKPT_PREFIX, CKPT_EPOCH = 0, 1, "ssd_resnet18_x", 3
SCOPES = ("", "backbone,extras")


def _sd(seed):
    return synth.synthetic_state_dict("ResNet18", FL, [6] * 4, 20, seed=seed, style="test")


def test_index_module_prefix_scope_and_validation(tmp_path):
    sd = _sd(1)
    f1, f2 = str(tmp_path / "m_epoch_1.pth"), str(tmp_path / "m_epoch_7.pth")
    torch.save(sd, f1)
    torch.save({"state_dict": OrderedDict(("module." + k, v) for k, v in _sd(2).items())}, f2)   # DDP-style wrapper
    with open(tmp_path / "checkpoint_list.txt", "w") as f:
        f.write(f"epoch 1: {f1}\nepoch 7: {f2}\n")
    assert CK.find_previous_checkpoint(str(tmp_path)) == ([1, 7], [f1, f2])
    assert CK.find_previous_checkpoint(str(tmp_path / "nope")) is False
    got, rep = CK.load_checkpoint(f2)
    assert list(got) == list(sd) and rep["resumed"] == len(sd)
    assert all(torch.equal(got[k], v) for k, v in _sd(2).items())
    assert CK.check_state_dict(CFG, got)["ok"]
    # scope: only matching keys are taken, everything else keeps the base values (checkpoint.py:110-131)
    base = _sd(3)
    got, rep = CK.load_checkpoint(f2, "backbone.layer1,loc", base)
    for k in base:
        src = _sd(2)[k] if ("backbone.layer1" in k or "loc" in k) else base[k]
        assert torch.equal(got[k], src), k
    assert set(rep["unresumed"]) == {k for k in base if "backbone.layer1" not in k and "loc" not in k}
    # validation catches a foreign checkpoint before anything is packed
    bad = OrderedDict(sd)
    bad["backbone.conv1.weight"] = torch.zeros(32, 3, 7, 7)
    del bad["loc.0.weight"]
    bad["something.else"] = torch.zeros(1)
    chk = CK.check_state_dict(CFG, bad)
    assert not chk["ok"] and chk["missing"] == ["loc.0.weight"] and chk["unexpected"] == ["something.else"]
    assert chk["mismatched"] == [("backbone.conv1.weight", (32, 3, 7, 7), (64, 3, 7, 7))]
    with pytest.raises(FileNotFoundError):
        CK.load_checkpoint(str(tmp_path / "missing.pth"))
    assert CK.main(["--cfg", _write_cfg(tmp_path), "--checkpoint", str(tmp_path), "--dry-run"]) == 0


def _write_cfg(tmp_path):
    import yaml
    p = str(tmp_path / "cfg.yml")
    with open(p, "w") as f:
        yaml.safe_dump(CFG, f)
    return p


def test_against_reference_save_and_resume(tmp_path):
    with gzip.open(GOLDEN, "rt") as f:
        ref = json.load(f)["checkpoint"]
    d = str(tmp_path)
    saved = _sd(CKPT_SEED)
    assert sorted(ref["saved_keys"]) == sorted("module." + k for k in saved)
    torch.save(OrderedDict((k, saved[k[len("module."):]]) for k in ref["saved_keys"]),
               os.path.join(d, f"{CKPT_PREFIX}_epoch_{CKPT_EPOCH}.pth"))
    with open(os.path.join(d, "checkpoint_list.txt"), "w") as f:
        f.write(ref["index"].replace("{dir}", d))
    epochs, files = CK.find_previous_checkpoint(d)
    assert [epochs, files] == [ref["found"][0], [p.replace("{dir}", d) for p in ref["found"][1]]]
    for scope in SCOPES:
        want = ref["scopes"][scope]
        base = _sd(BASE_SEED)
        got, rep = CK.load_checkpoint(files[-1], scope, OrderedDict((k, v.clone()) for k, v in base.items()))
        assert list(got) == want["keys"]
        for k in got:
            src = want["source"][k]
            if src in ("checkpoint", "both"):
                assert torch.equal(got[k], saved[k]), (scope, k)
            if src in ("base", "both"):
                assert torch.equal(got[k], base[k]), (scope, k)
        assert CK.check_state_dict(CFG, got)["ok"]
        if scope:
            assert rep["unresumed"] and all("backbone" not in k and "extras" not in k for k in rep["unresumed"])
