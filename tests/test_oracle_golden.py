"""Pins oracle/segtran_oracle.py against the committed golden fixtures produced by the real reference
(oracle/gen_golden.py)."""
import pytest
import torch

from oracle import segtran_oracle as O
from tests.helpers import load_golden, oracle_encoder, rel_err

ENC_CASES = ["enc3d_small", "enc2d_compress", "enc3d_clamp", "enc3d_ragged", "enc2d_nosqueeze", "enc3d_sqffn", "enc3d_sharedout"]
TOL = 2e-5          # fp32 CPU vs fp32 CPU, different op order


@pytest.mark.parametrize("name", ENC_CASES)
def test_encoder_forward_matches_golden(name):
    fx = load_golden(name)
    col = {}
    y, _ = oracle_encoder(fx, collect=col)
    assert y.shape == fx["out"].shape
    assert rel_err(y, fx["out"]) < TOL
    # the attention-score maxima the reference tracked (segtran_shared.py:569-573); order: per layer in-squeeze, squeeze-out
    L = len(fx["dims"]) - 1
    ref = fx["max_attn"]
    got = col["max_attn"]
    if not fx.get("use_squeezed_transformer", True):
        assert all(abs(g - r) <= 1e-3 * max(1.0, abs(r)) for g, r in zip(got, ref))
        return
    for i in range(L):
        assert abs(got[2 * i] - ref[i]) <= 1e-3 * max(1.0, abs(ref[i]))
        assert abs(got[2 * i + 1] - ref[L + i]) <= 1e-3 * max(1.0, abs(ref[L + i]))


@pytest.mark.parametrize("name", ENC_CASES)
def test_encoder_grads_match_golden(name):
    fx = load_golden(name)
    x = fx["x"].clone().requires_grad_(True)
    p = {"voxel_fusion." + k: v.clone().requires_grad_(True) for k, v in fx["state_dict"].items()}
    from tests.helpers import variant_kwargs
    y = O.fusion_encoder(p, "voxel_fusion.", x, fx["voxels_pos"], fx["vmask"], fx["dims"], fx["num_modes"],
                         **variant_kwargs(fx))
    (y * fx["G"]).sum().backward()
    assert rel_err(x.grad, fx["grad_x"]) < 5e-5
    gscale = max(float(g.abs().max()) for g in fx["grad_params"].values())
    for k, g in fx["grad_params"].items():
        got = p["voxel_fusion." + k].grad
        if k.endswith("query.weight") or k.endswith("query.bias"):          # tied: key.* is the same Parameter
            kk = "voxel_fusion." + k.replace("query.", "key.")
            got = got + (p[kk].grad if p[kk].grad is not None else 0)
        assert got is not None, k
        # gradients that are zero / pure cancellation noise in exact arithmetic (softmax shift invariance,
        # 1-mode soft-aggregate) are compared on the scale of the largest parameter gradient
        assert float((got - g).abs().max()) <= 2e-4 * float(g.abs().max()) + 1e-6 * gscale, k


def _oracle_seg(fx, dims, grad=False):
    p = {k: v.clone().requires_grad_(grad) for k, v in fx["state_dict"].items()}
    feats = [f.clone().requires_grad_(grad) for f in fx["feats"]]
    return p, feats


def test_seg3d_shell_matches_golden():
    """Oracle hot path fed with the in-FPN / out-FPN tensors recomputed in plain torch from the stored
    backbone features (FPN pyramids are out of the hot path; stock ops, segtran3d.py:299-323, 347-359)."""
    import torch.nn.functional as F
    fx = load_golden("seg3d_tiny")
    p = fx["state_dict"]
    f = fx["feats"]
    # in-FPN '34' (AN scheme) + depth pooling
    cur = F.conv3d(f[3], p["in_fpn34_conv.weight"], p["in_fpn34_conv.bias"])
    cur = cur + F.interpolate(f[4], size=cur.shape[2:], mode="trilinear", align_corners=False)
    cur = F.group_norm(cur, 8, p["in_gn4b.weight"], p["in_gn4b.bias"])
    sz = list(cur.shape[2:]); sz[0] //= 2
    feat_fpn = F.interpolate(cur, size=sz, mode="trilinear", align_corners=False)
    # out-FPN '12' -> curr_feat
    c = F.conv3d(f[1], p["out_fpn12_conv3d.weight"], p["out_fpn12_conv3d.bias"])
    c = F.group_norm(c + F.interpolate(f[2], size=c.shape[2:], mode="trilinear", align_corners=False), 8,
                     p["out_gn2b.weight"], p["out_gn2b.bias"])
    c2 = F.conv3d(c, p["out_fpn23_conv3d.weight"], p["out_fpn23_conv3d.bias"])
    c2 = F.group_norm(c2 + F.interpolate(f[3], size=c2.shape[2:], mode="trilinear", align_corners=False), 8,
                      p["out_gn3b.weight"], p["out_gn3b.bias"])
    B = feat_fpn.shape[0]
    N = feat_fpn[0, 0].numel()
    vmask = torch.ones(B, N, dtype=torch.long)      # 3-D mask is all ones (bias of in_bridge_to3, SURVEY §3.2)
    y = O.hot_path_3d(p, feat_fpn, c2, vmask, (32, 32, 32), [48, 48], 4, 2)
    assert rel_err(y, fx["out"]) < TOL


def test_seg2d_shell_matches_golden():
    import torch.nn.functional as F
    fx = load_golden("seg2d_tiny")
    p = fx["state_dict"]
    f = fx["feats"]
    cur = F.conv2d(f[3], p["in_fpn34_conv.weight"], p["in_fpn34_conv.bias"])
    cur = cur + F.interpolate(f[4], size=cur.shape[2:], mode="bilinear", align_corners=False)
    feat_fpn = F.group_norm(cur, 8, p["in_gn4b.weight"], p["in_gn4b.bias"])
    c = F.conv2d(f[1], p["out_fpn12_conv.weight"], p["out_fpn12_conv.bias"])
    c = F.group_norm(c + F.interpolate(f[2], size=c.shape[2:], mode="bilinear", align_corners=False), 8,
                     p["out_gn2b.weight"], p["out_gn2b.bias"])
    c2 = F.conv2d(c, p["out_fpn23_conv.weight"], p["out_fpn23_conv.bias"])
    c2 = F.group_norm(c2 + F.interpolate(f[3], size=c2.shape[2:], mode="bilinear", align_corners=False), 8,
                      p["out_gn3b.weight"], p["out_gn3b.bias"])
    # 2-D mask: AvgPool2d(8)(|x|).sum(1) > 0 on the raw image (segtran2d.py:229-233, pool_stride = 2**3)
    vmask = (F.avg_pool2d(fx["batch"].abs(), 8).sum(1) > 0).reshape(2, -1)
    assert 0 < int(vmask.sum()) < vmask.numel()
    y = O.hot_path_2d(p, feat_fpn, c2, vmask, (64, 64), [48, 48, 24], 4)
    assert rel_err(y, fx["out"]) < TOL


def test_oracle_matches_live_reference_train_mode_shapes():
    """A fresh config (not one of the encoder fixtures) run by the reference in train() mode; dropout=0 so train() ==
    eval() numerically.  Weights, inputs and output recorded by oracle/gen_golden.py construction."""
    fx = load_golden("enc_train")
    p = {"voxel_fusion." + k: v for k, v in fx["state_dict"].items()}
    y = O.fusion_encoder(p, "voxel_fusion.", fx["x"], fx["voxels_pos"], fx["vmask"], fx["dims"], fx["num_modes"])
    assert y.shape == fx["out"].shape
    assert rel_err(y, fx["out"]) < TOL


def test_dice_and_indices():
    idx = O.gen_all_indices((2, 3))
    assert idx.tolist() == [[[0, 0], [0, 1], [0, 2]], [[1, 0], [1, 1], [1, 2]]]
    a = torch.tensor([1, 1, 0, 0]); b = torch.tensor([1, 0, 0, 0])
    assert abs(O.dice_hard(a, b) - 2 / 3) < 1e-12
    assert O.dice_hard(torch.zeros(3), torch.zeros(3)) == 1.0
