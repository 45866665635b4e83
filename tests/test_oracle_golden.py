"""Pins the oracle (oracle/crf_oracle.py) against golden vectors produced by the unmodified reference
(tests/golden/make_golden.py): bit-exact index maps, fp32 forward outputs and every gradient."""
import numpy as np
import pytest
import torch

from oracle import crf_oracle as O
from tests.helpers import HEAD_CASES, LAYER_CASES, golden_layer_inputs, golden_rel_l2, load_golden, rel_l2


def test_index_maps_bit_exact():
    g = load_golden("index_maps")
    for H, W, s in g["cases"]:
        H, W, s = int(H), int(W), int(s)
        tag = f"{H}x{W}s{s}"
        x = torch.arange(1, 2 * H * W * 3 + 1, dtype=torch.float32).reshape(2, H, W, 3)
        win = O.window_gather(x, 7, s)
        assert np.array_equal(win.numpy(), g["gather." + tag]), tag
        wv = torch.arange(1, win.numel() + 1, dtype=torch.float32).reshape(win.shape)
        back = O.window_scatter(wv, 2, H, W, 7, s)
        assert np.array_equal(back.numpy(), g["scatter." + tag]), tag
        if s == 3:
            assert np.array_equal(O.shift_mask(H, W, 7, s), g["mask." + tag]), tag
            assert np.array_equal(O.window_region_ids(H, W, 7, s), g["region." + tag]), tag


def test_known_answer_facts():
    """SURVEY.md 8c known-answer facts established on the reference."""
    g = load_golden("index_maps")
    idx = O.relative_position_index(7)
    assert np.array_equal(idx, g["relative_position_index"])
    assert idx[0, :10].tolist() == [84, 83, 82, 81, 80, 79, 78, 71, 70, 69]
    assert abs(float(g["scale_hd32"][0]) - 32 ** -0.5) < 1e-12
    rid = O.window_region_ids(15, 20, 7, 3)
    sets = [sorted(set(r.tolist())) for r in rid]
    assert sets == [[0], [0], [1, 2], [0], [0], [1, 2], [3, 6], [3, 6], [4, 5, 7, 8]]
    assert O.padded_size(120, 7) == 126 and O.padded_size(160, 7) == 161


@pytest.mark.parametrize("name", LAYER_CASES + HEAD_CASES)
def test_layer_forward_backward_matches_reference(name):
    g = load_golden(name)
    (B, H, W, C, nH, depth), x, v, blocks = golden_layer_inputs(g)
    x = x.detach().requires_grad_(True)
    v = v.detach().requires_grad_(True)
    for p in blocks:
        for t in p.values():
            t.requires_grad_(True)
    y = O.basic_crf_layer(x, v, H, W, blocks, nH)
    y.backward(torch.from_numpy(g["dy"]))
    assert rel_l2(y.detach(), g["y"]) < 1e-5
    assert rel_l2(x.grad, g["dx"]) < 1e-5
    assert rel_l2(v.grad, g["dv"]) < 1e-5
    for i, p in enumerate(blocks):
        for k, t in p.items():
            assert golden_rel_l2(g, f"grad.blocks.{i}.{k}", t.grad) < 2e-5, (i, k)


def test_loss_matches_reference_golden():
    """oracle.model_oracle.ssim_l1_loss (and the host-side composition in training.py) against the value and gradient
    the unmodified reference loss produced (loss.SSIM + nn.L1Loss as combined at train.py:94-100)."""
    import torch
    from monocular_depth_estimation_b200 import training as TR
    from oracle import model_oracle as MO
    g = load_golden("loss_ssim_l1")
    for tag in ("a", "b", "c"):
        for fn in (MO.ssim_l1_loss, TR.depth_loss):
            pred = torch.from_numpy(g[f"pred.{tag}"]).requires_grad_(True)
            val = fn(pred, torch.from_numpy(g[f"target.{tag}"]))
            val.backward()
            assert abs(float(val.detach()) - float(g[f"loss.{tag}"][0])) < 1e-6
            assert rel_l2(pred.grad, g[f"dpred.{tag}"]) < 1e-5


def test_full_model_oracle_matches_reference_model():
    """oracle.model_oracle.OraclePTModel (the CPU baseline / reference arm of bench.py and the checker of the whole-model
    GPU test) against the UNMODIFIED reference model (src/model_mobileV3_large_newCRFs.py PTModel, executed in the build
    container by tests/golden/make_golden.py): same name-seeded weights, eval mode, 2 x 3 x 64 x 96 image -- depth map,
    loss, image gradient and a dozen parameter gradients spread over encoder, bridge, the four stages and the head."""
    from oracle import model_oracle as MO
    from tests.helpers import MODEL_GRAD_KEYS, fill_by_name
    g = load_golden("model_64x96")
    model = fill_by_name(MO.OraclePTModel()).eval()
    assert sorted(model.state_dict().keys()) == g["keys"].tolist()          # one checkpoint fits both
    image = torch.from_numpy(g["image"]).requires_grad_(True)
    pred = model(image)
    loss = MO.ssim_l1_loss(pred, MO.depth_norm(torch.from_numpy(g["depth"])))
    loss.backward()
    assert rel_l2(pred.detach(), g["pred"]) < 1e-5
    assert abs(float(loss.detach()) - float(g["loss"][0])) < 1e-6
    assert rel_l2(image.grad, g["dimage"]) < 1e-4
    params = dict(model.named_parameters())
    for k in MODEL_GRAD_KEYS:
        assert rel_l2(params[k].grad, g["grad." + k]) < 1e-4, k


def test_product_model_state_dict_matches_reference_model():
    """The product model's module tree takes the reference model's checkpoint as-is (keys and shapes)."""
    from monocular_depth_estimation_b200.model import PTModel
    from oracle import model_oracle as MO
    g = load_golden("model_64x96")
    ours, ref = PTModel().state_dict(), MO.OraclePTModel().state_dict()
    assert sorted(ours.keys()) == g["keys"].tolist()
    for k, t in ours.items():
        assert tuple(t.shape) == tuple(ref[k].shape) and t.dtype == ref[k].dtype, k
