"""The plans bench.py times for cfg3 (SSD-MobileNetV2 300x300, B=64), cfg4 (SSDFPN-ResNet50 640x640, B=16, training
mode: raw logits) and cfg5 (SSDBiFPN-RegNetX032 1280x1280, B=4), each at its benchmark batch, against
  (a) the launch record: the multi-way conv_igemm instantiations these plans are known to run must be launched;
  (b) the same model planned with every optimisation off (SSDSB_WAYS=1 SSDSB_NO_PAIR=1 SSDSB_NO_MBFUSE=1
      SSDSB_DW_SIMPLE=1) and run without a CUDA graph: the graph-replayed outputs must be bit-identical;
  (c) the model oracle under the bf16 policy on sampled images (images are independent): the tolerance of
      test_gpu_model.test_conv_stack_vs_oracle_bf16_policy, loc |err| <= 2e-2 * (1 + max|loc|) and
      conf |err| <= 5e-4 + 4e-2 * conf (training-mode logits are compared through the sigmoid); for cfg5 at most
      1.5x the distance between the bf16-policy and the fp32 oracle where that is larger.
The distance of the bf16-policy oracle from the fp32 oracle is printed beside each result."""
import pytest
import torch

pytestmark = pytest.mark.gpu

# (block_n, block_k, ways) each plan must launch
MULTIWAY = {"cfg3": {(64, 32, 2)}, "cfg4": {(128, 64, 2), (64, 64, 2), (64, 64, 4)},
            "cfg5": {(128, 32, 2), (64, 64, 2)}}
ORACLE = {"cfg3": "ssd_mobilenetv2_forward", "cfg4": "ssdfpn_resnet_forward", "cfg5": "ssdbifpn_forward"}
SAMPLED = {"cfg3": (0, 37, 63), "cfg4": (0, 9, 15), "cfg5": (0, 3)}
# the cfg3 <64,32,2> launch is the project 144(160) -> 24(32) of the stride-2 block at 38x38; the plan may instead run
# that block as one fused mbconv launch if that measures faster when the plan is built
CFG3_64x32x2_LAYER = "conv1x1s1 160->32 @38x38"
PLAIN = {"SSDSB_WAYS": "1", "SSDSB_NO_PAIR": "1", "SSDSB_NO_MBFUSE": "1", "SSDSB_DW_SIMPLE": "1"}


@pytest.fixture(scope="module")
def env():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    import ssds_pytorch_b200 as S
    return S


def _build(name):
    import bench
    from ssds_pytorch_b200 import synth
    from ssds_pytorch_b200.model import engine_for, number_box_from_cfg
    cfg = bench.cfg_dict(name)
    m, pre = cfg["MODEL"], cfg["DATASET"]["PREPROC"]
    nb = number_box_from_cfg(m)
    sd = synth.synthetic_state_dict(m["NETS"], m["FEATURE_LAYER"], nb, m["NUM_CLASSES"], seed=0, style="test",
                                    ssds=m["SSDS"])
    model = engine_for(m["SSDS"], m["NETS"])(sd, m["FEATURE_LAYER"], m["NUM_CLASSES"], nb, device="cuda",
                                             mean=float(pre["MEAN"]), std=float(pre["STD"]))
    model.train(bench.CONFIGS[name]["kind"] == "loss")
    return sd, m, model


def _dist(loc, conf, rloc, rconf, training):
    """(max |loc err| / (1 + max|loc|), max conf err / (5e-4 + 4e-2 conf)) over the levels"""
    wl = wc = 0.0
    for l, c, rl, rc in zip(loc, conf, rloc, rconf):
        assert l.shape == rl.shape and c.shape == rc.shape
        if training:
            c, rc = c.sigmoid(), rc.sigmoid()
        wl = max(wl, (l - rl).abs().max().item() / (1.0 + rl.abs().max().item()))
        wc = max(wc, ((c - rc).abs() / (5e-4 + 4e-2 * rc)).max().item())
    return wl, wc


@pytest.mark.parametrize("name", ["cfg3", "cfg4", "cfg5"])
def test_timed_plan_vs_plain_plan_and_oracle(env, name, monkeypatch):
    import bench
    from oracle import model_oracle as M
    from ssds_pytorch_b200 import conv as K
    for k in PLAIN:
        monkeypatch.delenv(k, raising=False)
    B = bench.CONFIGS[name]["batch"]
    sd, m, model = _build(name)
    H, W = m["IMAGE_SIZE"]
    xg = torch.randint(0, 256, (B, H, W, 3), generator=torch.Generator().manual_seed(1234), dtype=torch.uint8).cuda()
    loc, conf = model(xg, use_graph=True)
    torch.cuda.synchronize()
    got = [t.clone() for t in loc + conf]
    L = len(loc)
    plan = model.plan_for(xg)
    kinds = [v["kind"] for v in plan["info"].values()]
    # (a) replay the plan un-graphed, reading the launch record after every step
    seen = set()
    for s in plan["steps"]:
        s()
        ll = K.last_launch()
        seen.add((ll["block_n"], ll["block_k"], ll["ways"]))
    torch.cuda.synchronize()
    want = set(MULTIWAY[name])
    note = ""
    if name == "cfg3" and CFG3_64x32x2_LAYER not in kinds:
        assert any(k.startswith("mbconv s2 32->160->32 @38x38") for k in kinds), kinds
        want.discard((64, 32, 2))
        note = " (the 38x38 stride-2 block runs fused: no <64,32,2> launch)"
    print(f"{name} B={B}: {len(plan['steps'])} launches, conv instantiations (block_n, block_k, ways) "
          f"{sorted(seen)}{note}")
    assert want <= seen, f"{name}: expected {sorted(want)} among {sorted(seen)}"
    for a, b in zip(got, loc + conf):
        assert torch.equal(a, b), "graph replay differs from eager replay"
    # (b) every optimisation off, no graph
    for k, v in PLAIN.items():
        monkeypatch.setenv(k, v)
    _, _, plain = _build(name)
    loc1, conf1 = plain(xg, use_graph=False)
    torch.cuda.synchronize()
    plain_kinds = [v["kind"] for v in plain.plan_for(xg)["info"].values()]
    assert not any(k.startswith(("pair1x1", "mbconv")) for k in plain_kinds)
    for k in PLAIN:
        monkeypatch.delenv(k)
    for i, (a, b) in enumerate(zip(got, loc1 + conf1)):
        assert torch.equal(a, b), f"{name}: output {i} of the timed plan differs from the plain plan"
    del plain, loc1, conf1
    # (c) the bf16-policy oracle on sampled images, and its own distance from the fp32 oracle
    fwd = getattr(M, ORACLE[name])
    sd_gpu = {k: v.cuda() for k, v in sd.items()}
    training = model.training
    worst_l = worst_c = noise_l = noise_c = 0.0
    for i in SAMPLED[name]:
        xi = (xg[i:i + 1].float() / 255.0).permute(0, 3, 1, 2).contiguous()
        with torch.no_grad():
            rloc, rconf = fwd(sd_gpu, xi, m["FEATURE_LAYER"], training=training, policy="bf16")
            floc, fconf = fwd(sd_gpu, xi, m["FEATURE_LAYER"], training=training, policy="fp32")
        wl, wc = _dist([t[i:i + 1] for t in got[:L]], [t[i:i + 1] for t in got[L:]], rloc, rconf, training)
        nl, nc = _dist(rloc, rconf, floc, fconf, training)
        worst_l, worst_c = max(worst_l, wl), max(worst_c, wc)
        noise_l, noise_c = max(noise_l, nl), max(noise_c, nc)
    print(f"{name} {H}x{W} B={B} images {SAMPLED[name]}: vs bf16-policy oracle max |loc err|/(1+max|loc|) "
          f"{worst_l:.3e}, max conf err / tol {worst_c:.3f}; bf16-policy vs fp32 oracle: loc {noise_l:.3e}, "
          f"conf {noise_c:.3f} x tol")
    limit_l, limit_c = 2e-2, 1.0
    if name == "cfg5":
        # RegNetX032 + 5 BiFPN levels at 1280x1280 with synthetic weights: the bf16-policy oracle is itself ~1.7x the
        # conf tolerance away from the fp32 oracle (B200, 1000 W), and a different fp32 summation order moves the bf16
        # roundings as much; bound the kernel by 1.5x that measured distance, as test_gpu_model does for yolo4_50
        limit_l, limit_c = max(limit_l, 1.5 * noise_l), max(limit_c, 1.5 * noise_c)
    assert worst_l <= limit_l and worst_c <= limit_c, (worst_l, worst_c, limit_l, limit_c)
