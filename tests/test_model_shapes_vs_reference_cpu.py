"""`synth.model_shapes` (the layer table checkpoint validation and the synthetic weights rely on) against the
reference's own `create_model(cfg).state_dict()` for every engine combination model.ENGINES offers, as stored in
tests/golden/reference_state_dicts.json.gz by tests/golden/make_golden_reference.py."""
import gzip
import json
import os

import pytest

from ssds_pytorch_b200 import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_state_dicts.json.gz")

FPN = [[3, 4, 5, "Conv:S", "Conv:S"], [512, 1024, 2048, 2048, 256]]
CASES = {
    "SSD-ResNet50": ("SSD", "ResNet50", [[3, 4, 5, "Conv:S", "Conv:S", "Conv:S"], [512, 1024, 2048, 512, 256, 256]]),
    "SSD-ResNet18": ("SSD", "ResNet18", [[3, 4, 5, "Conv:S"], [128, 256, 512, 256]]),
    "SSD-MobileNetV2": ("SSD", "MobileNetV2", [[5, 7, "Conv:S", "Conv:S", "Conv:S", "Conv:S"],
                                               [96, 320, 512, 256, 256, 128]]),
    "SSDFPN-ResNet50": ("SSDFPN", "ResNet50", FPN),
    "SSDBiFPN-ResNet50": ("SSDBiFPN", "ResNet50", FPN),
    "SSDBiFPN-RegNetX032": ("SSDBiFPN", "RegNetX032", [[2, 3, 4, "Conv:S", "Conv:S"], [192, 432, 1008, 1008, 256]]),
    "SSDFPN-RegNetX032": ("SSDFPN", "RegNetX032", [[2, 3, 4, "Conv:S", "Conv:S"], [192, 432, 1008, 1008, 256]]),
    "YOLOV3-ResNet18": ("YOLOV3", "ResNet18", [[3, 4, 5], [128, 256, 512]]),            # experiments/cfgs/tests/test.yml
    "YOLOV3-ResNet50+extras": ("YOLOV3", "ResNet50", [[3, 4, 5, "Conv:S"], [512, 1024, 2048, 512]]),
    "YOLOV3-ResNet18 [in,out] depth pairs": ("YOLOV3", "ResNet18", [[3, 4, 5, "Conv:S"],
                                                                     [[128, 128], [256, 128], [512, 256], 256]]),
    "YOLOV4-ResNet18+extras": ("YOLOV4", "ResNet18", [[3, 4, 5, "Conv:S"], [128, 256, 512, 256]]),
    "YOLOV4-ResNet50": ("YOLOV4", "ResNet50", [[3, 4, 5], [512, 1024, 2048]]),
}


@pytest.fixture(scope="module")
def ref():
    with gzip.open(GOLDEN, "rt") as f:
        return json.load(f)["state_dicts"]


@pytest.mark.parametrize("name", list(CASES))
def test_layer_table_equals_reference_state_dict(ref, name):
    ssds, nets, fl = CASES[name]
    L = len(fl[0])
    want = [(k, tuple(s)) for k, s in ref[name]]
    got = [(k, tuple(s)) for k, s in synth.model_shapes(ssds, nets, fl, [6] * L, 20)]
    assert [k for k, _ in got] == [k for k, _ in want]                 # same keys, same ORDER
    assert got == want
