"""Generate tests/golden/*.pt by running the REAL reference (askerlee/segtran @ /root/reference).

TEST INFRASTRUCTURE ONLY.  Run in the build container:  python -m oracle.gen_golden
Each fixture holds seeded inputs, the reference module's state_dict (backbone weights dropped),
the reference outputs, and the gradients of ``loss = (out * G).sum()`` w.r.t. inputs and
parameters.  The fixtures pin oracle/segtran_oracle.py (CPU tests) and the CUDA path (GPU tests);
they are deliberately small (tens to hundreds of KB).
"""
from __future__ import annotations

import os
import sys
from argparse import Namespace

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle import ref_import as R                      # noqa: E402
from oracle import segtran_oracle as O                  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")


def _grads(module, loss, inputs):
    params = [(n, p) for n, p in module.named_parameters() if p.requires_grad]
    gs = torch.autograd.grad(loss, [p for _, p in params] + list(inputs), allow_unused=True)
    gp = {n: g for (n, _), g in zip(params, gs[:len(params)]) if g is not None}
    gi = list(gs[len(params):])
    return gp, gi


def gen_encoder(name, dims, M, A, pd, qkb, grid, B, seed, wscale=1.0, mask_p=0.2, squeeze=True, sq_ffn=False,
                out_type="private"):
    ns = R.load()
    cfg = R.encoder_config(ns.shared, dims=dims, num_modes=M, num_attractors=A, pos_dim=pd, qk_have_bias=qkb)
    cfg.use_squeezed_transformer = squeeze               # --nosqueeze: plain N x N cross attention per layer
    cfg.has_FFN_in_squeeze = sq_ffn                      # --squeezeuseffn
    cfg.trans_output_type = out_type
    enc = R.build_encoder(cfg, seed=seed).eval()
    if wscale != 1.0:                       # push the scores past attn_clip=500 (segtran_shared.py:578-580)
        with torch.no_grad():
            for n, p in enc.named_parameters():
                if n.endswith("query.weight"):
                    p.mul_(wscale)
    N = 1
    for g in grid:
        N *= g
    torch.manual_seed(seed + 100)
    x = torch.randn(B, N, dims[0], requires_grad=True)
    pos = O.voxels_pos_for_grid(grid, (8,) * pd, B)
    mask = (torch.rand(B, N, 1) > mask_p).long()
    G = torch.randn(B, N, dims[-1])
    with R.quiet():
        y = enc(x, pos, mask, torch.Size(grid))
    gp, gi = _grads(enc, (y * G).sum(), [x])
    if squeeze:
        max_attn = [float(t.in_ator_trans.max_attn) for t in enc.translayers] + \
                   [float(t.ator_out_trans.max_attn) for t in enc.translayers]
    else:
        max_attn = [float(t.max_attn) for t in enc.translayers]
    fx = dict(kind="encoder", dims=list(dims), num_modes=M, num_attractors=A, pos_dim=pd, qk_have_bias=qkb,
              grid=list(grid), use_squeezed_transformer=squeeze, has_FFN_in_squeeze=sq_ffn,
              trans_output_type=out_type, x=x.detach(), voxels_pos=pos, vmask=mask, G=G, out=y.detach(),
              state_dict={k: v.clone() for k, v in enc.state_dict().items()},
              grad_params=gp, grad_x=gi[0], max_attn=max_attn)
    torch.save(fx, os.path.join(OUT, name + ".pt"))
    print(name, "out", tuple(y.shape), "max|out|", float(y.abs().max()), "max_attn", max_attn)


class FixedFeatBackbone3d(torch.nn.Module):
    """Stands in for InceptionI3d.extract_features (aj_i3d.py:325-333): returns stored feature maps."""

    def __init__(self, feats):
        super().__init__()
        self.feats = feats

    def extract_features(self, x):
        keys = ["MaxPool3d_2a_3x3", "Conv3d_2c_3x3", "Mixed_3c", "Mixed_4f", "Mixed_5c"]
        return dict(zip(keys, self.feats))


def gen_seg3d(name, seed=3):
    ns = R.load()
    ns.shared.bb2feat_dims["i3d-tiny"] = [8, 16, 24, 32, 48]
    args = Namespace(num_classes=4, backbone_type="i3d-tiny", use_pretrained=False, num_attractors=12,
                     num_translayers=1, num_modes=4, trans_output_type="private", mid_type="shared",
                     orig_in_channels=4, D_pool_K=2, inchan_to3_scheme="bridgeconv", D_groupsize=1, device="cpu",
                     in_fpn_layers="34", out_fpn_layers="1234", in_fpn_scheme="AN", out_fpn_scheme="AN",
                     translayer_compress_ratios=[1, 1], dropout_prob=0.0, tie_qk_scheme="shared",
                     qk_have_bias=True, use_squeezed_transformer=True, pos_code_type="lsinu")
    torch.manual_seed(seed)
    with R.quiet():
        ns.seg3d.CONFIG.update_config(args)
        net = ns.seg3d.Segtran3d(ns.seg3d.CONFIG)
    net.eval()
    B, S = 2, 32
    c = ns.shared.bb2feat_dims["i3d-tiny"]
    torch.manual_seed(seed + 1)
    batch = torch.randn(B, 4, S, S, S)
    batch[:, :, :, :, :8] = 0                                  # a zero slab (mask is still all-ones in 3-D, SURVEY §3.2)
    feats = [torch.randn(B, c[0], 16, 16, 16), torch.randn(B, c[1], 16, 16, 16), torch.randn(B, c[2], 16, 8, 8),
             torch.randn(B, c[3], 8, 4, 4), torch.randn(B, c[4], 4, 2, 2)]
    feats = [f.requires_grad_(True) for f in feats]
    net.backbone = FixedFeatBackbone3d(feats)
    G = torch.randn(B, 4, S, S, S)
    with R.quiet(), R.cuda_literal_to_cpu():
        y = net(batch)
    gp, gi = _grads(net, (y * G).sum(), feats[1:])
    sd = {k: v.clone() for k, v in net.state_dict().items() if not k.startswith("backbone.")}
    fx = dict(kind="seg3d", args=vars(args), bb_feat_dims=c, batch=batch, feats=[f.detach() for f in feats], G=G,
              out=y.detach(), state_dict=sd, grad_params=gp, grad_feats=[None] + gi)
    torch.save(fx, os.path.join(OUT, name + ".pt"))
    print(name, "out", tuple(y.shape), "max|out|", float(y.abs().max()))


class FixedFeatBackbone2d(torch.nn.Module):
    """Stands in for ResNet.ext_features (resnet.py:186-200)."""

    def __init__(self, feats):
        super().__init__()
        self.feats = feats

    def ext_features(self, x):
        return tuple(self.feats)


def gen_seg2d(name, seed=4):
    ns = R.load()
    ns.shared.bb2feat_dims["resnet-tiny"] = [8, 16, 24, 32, 48]
    args = Namespace(num_classes=3, backbone_type="resnet-tiny", use_pretrained=False, num_attractors=10,
                     num_translayers=2, num_modes=4, trans_output_type="private", mid_type="shared",
                     device="cpu", in_fpn_layers="34", out_fpn_layers="1234", in_fpn_scheme="AN",
                     out_fpn_scheme="AN", translayer_compress_ratios=[1, 1, 2], dropout_prob=0.0,
                     tie_qk_scheme="shared", qk_have_bias=False, use_squeezed_transformer=True,
                     pos_code_type="lsinu", use_global_bias=False, num_modalities=0)
    import resnet as ref_resnet
    ref_resnet.__dict__["resnet-tiny"] = lambda pretrained=False, do_pool1=True: torch.nn.Identity()
    torch.manual_seed(seed)
    with R.quiet():
        ns.seg2d.CONFIG.update_config(args)
        net = ns.seg2d.Segtran2d(ns.seg2d.CONFIG)
    net.eval()
    B, S = 2, 64
    c = ns.shared.bb2feat_dims["resnet-tiny"]
    torch.manual_seed(seed + 1)
    batch = torch.randn(B, 3, S, S)
    batch[:, :, :16, :] = 0                                    # true zero padding -> masked tokens (segtran2d.py:339)
    feats = [torch.randn(B, c[0], 32, 32), torch.randn(B, c[1], 32, 32), torch.randn(B, c[2], 16, 16),
             torch.randn(B, c[3], 8, 8), torch.randn(B, c[4], 4, 4)]
    feats = [f.requires_grad_(True) for f in feats]
    net.backbone = FixedFeatBackbone2d(feats)
    G = torch.randn(B, 3, S, S)
    with R.quiet():
        y = net(batch)
    gp, gi = _grads(net, (y * G).sum(), feats[1:])
    sd = {k: v.clone() for k, v in net.state_dict().items() if not k.startswith("backbone.")}
    fx = dict(kind="seg2d", args=vars(args), bb_feat_dims=c, batch=batch, feats=[f.detach() for f in feats], G=G,
              out=y.detach(), state_dict=sd, grad_params=gp, grad_feats=[None] + gi)
    torch.save(fx, os.path.join(OUT, name + ".pt"))
    print(name, "out", tuple(y.shape), "max|out|", float(y.abs().max()))


def gen_train():
    """Loss (train3d.py:731-756) and optimiser (optimization.py BertAdam + train3d.py:760 global clip) fixtures, produced by
    the reference's own functions."""
    R.load()
    from utils import losses as ref_losses            # /root/reference/code/utils/losses.py
    import optimization as ref_opt                    # /root/reference/code/optimization.py
    from oracle import train_oracle as T
    torch.manual_seed(11)
    B, K, sp = 2, 4, (6, 5, 8)
    logits = (torch.randn(B, K, *sp) * 2.5).requires_grad_(True)
    mask = (torch.rand(B, K, *sp) > 0.6).float()
    pos_weight = T.normalised_bce_weight([0., 3, 1, 1.75], K)            # BraTS default (train3d.py:223, :517-518)
    class_weights = T.default_class_weights(K)
    dice_w = 0.5
    bce = torch.nn.BCEWithLogitsLoss(pos_weight=pos_weight)
    ce = bce(logits.permute([0, 2, 3, 4, 1]), mask.permute([0, 2, 3, 4, 1]))
    soft = torch.sigmoid(logits)
    dice = 0
    for cls in range(1, K):
        dice = dice + ref_losses.dice_loss_indiv(soft[:, cls], mask[:, cls]) * class_weights[cls]
    loss = (1 - dice_w) * ce + dice_w * dice
    (g,) = torch.autograd.grad(loss, [logits])
    torch.save(dict(kind="train_loss", logits=logits.detach(), mask=mask, pos_weight=pos_weight,
                    class_weights=class_weights, dice_w=dice_w, loss=loss.detach(), ce=ce.detach(), dice=dice.detach(),
                    dlogits=g), os.path.join(OUT, "train_loss_tiny.pt"))
    print("train_loss_tiny loss", float(loss), "ce", float(ce), "dice", float(dice))

    # optimiser: 5 parameters in 3 groups, one of them never receives a gradient; 4 steps
    torch.manual_seed(12)
    shapes = [(33, 17), (64,), (5, 7, 3), (1,), (40, 9)]
    params = [torch.nn.Parameter(torch.randn(*s) * 0.3) for s in shapes]
    init = [p.detach().clone() for p in params]
    lr, decay = 2e-3, 1e-2
    groups = [{"params": [params[0], params[2], params[4]], "weight_decay": decay, "lr": lr},
              {"params": [params[1]], "weight_decay": decay * 0.1, "lr": lr},
              {"params": [params[3]], "weight_decay": 0.0, "lr": lr * 100}]
    per_lr = [lr, lr, lr, lr * 100, lr]
    per_wd = [decay, decay * 0.1, decay, 0.0, decay]
    t_total, warm = 8, 0.25
    opt = ref_opt.BertAdam(groups, warmup=warm, t_total=t_total, weight_decay=decay)
    grads, after = [], []
    for step in range(4):
        gs = [torch.randn(*s) * (10.0 if step == 1 else 0.02) for s in shapes]      # step 1 trips both clips
        gs[4] = None                                                                    # never-used parameter
        grads.append([None if g is None else g.clone() for g in gs])
        opt.zero_grad()
        for p, g in zip(params, gs):
            p.grad = None if g is None else g.clone()
        torch.nn.utils.clip_grad_norm_(params, 0.1)                                     # train3d.py:760-761
        opt.step()
        after.append([p.detach().clone() for p in params])
    torch.save(dict(kind="train_bertadam", shapes=shapes, init=init, grads=grads, after=after, lr=per_lr,
                    weight_decay=per_wd, t_total=t_total, warmup=warm, grad_clip=0.1, max_grad_norm=0.05),
               os.path.join(OUT, "train_bertadam_tiny.pt"))
    print("train_bertadam_tiny: 4 steps, |p0| after", float(after[-1][0].abs().max()))


def gen_poly(name="poly2d_tiny", seed=31):
    """Reference Polyformer layer (code/networks/polyformer.py): output and gradients on a small feature map."""
    R.load()
    import networks.polyformer as ref_poly                      # /root/reference/code/networks/polyformer.py
    args = Namespace(num_attractors=8, num_modes=4, tie_qk_scheme="loose", qk_have_bias=True, pos_code_type="lsinu")
    torch.manual_seed(seed)
    with R.quiet():
        net = ref_poly.Polyformer(32, chan_axis=1, args=args)
    net.eval()
    torch.manual_seed(seed + 1)
    x = torch.randn(2, 32, 12, 10).requires_grad_()
    G = torch.randn(2, 32, 12, 10)
    with R.quiet():
        y = net(x)
    gp, gi = _grads(net, (y * G).sum(), [x])
    torch.save(dict(kind="poly", args=vars(args), feat_dim=32, x=x.detach(), G=G, out=y.detach(),
                    state_dict={k: v.clone() for k, v in net.state_dict().items()}, grad_params=gp, grad_x=gi[0]),
               os.path.join(OUT, name + ".pt"))
    print(name, "out", tuple(y.shape), "max|out|", float(y.abs().max()))


INIT_CASES = [([64, 64], 4, 16, 3, True), ([64, 64, 32], 4, 8, 2, False)]


def gen_construction():
    """What the construction tests compare against, recorded from the reference modules (digests where the test needs
    exact equality, values where it needs numbers):
      init_seed3.pt     encoders of INIT_CASES built with seed 3: state_dict order and digests, named_parameters order;
      seg3d_init.pt     the Segtran3d shell of seg3d_tiny's args built with seed 3: every state_dict name, the backbone's
                        tensor shapes, the CPU RNG state before (digest) and after (value) the backbone's construction,
                        and the digests of every non-backbone tensor;
      enc_train.pt      a fresh encoder config in train() mode (dropout 0): weights, inputs and output."""
    from tests.helpers import state_digests, tensor_digest
    ns = R.load()
    cases = {}
    for dims, M, A, pd, qkb in INIT_CASES:
        cfg = R.encoder_config(ns.shared, dims=dims, num_modes=M, num_attractors=A, pos_dim=pd, qk_have_bias=qkb)
        enc = R.build_encoder(cfg, seed=3)
        cases[repr((dims, M, A, pd, qkb))] = dict(state_digests=state_digests(enc.state_dict()),
                                                  param_names=[n for n, _ in enc.named_parameters()])
    torch.save(dict(kind="init", seed=3, cases=cases), os.path.join(OUT, "init_seed3.pt"))
    print("init_seed3", list(cases))

    ns.shared.bb2feat_dims["i3d-tiny"] = [8, 16, 24, 32, 48]
    args = Namespace(**torch.load(os.path.join(OUT, "seg3d_tiny.pt"), weights_only=False)["args"])
    rng = {}
    i3d = ns.seg3d.InceptionI3d

    def recording_i3d(*a, **kw):
        rng["before"] = torch.get_rng_state()
        net = i3d(*a, **kw)
        rng["after"] = torch.get_rng_state()
        return net

    ns.seg3d.InceptionI3d = recording_i3d
    try:
        torch.manual_seed(3)
        with R.quiet():
            ns.seg3d.CONFIG.update_config(args)
            net = ns.seg3d.Segtran3d(ns.seg3d.CONFIG)
    finally:
        ns.seg3d.InceptionI3d = i3d
    sd = net.state_dict()
    torch.save(dict(kind="seg3d_init", seed=3, names=list(sd),
                    backbone_shapes={k: tuple(v.shape) for k, v in sd.items() if k.startswith("backbone.")},
                    rng_before_backbone=tensor_digest(rng["before"]), rng_after_backbone=rng["after"],
                    state_digests=state_digests({k: v for k, v in sd.items() if not k.startswith("backbone.")})),
               os.path.join(OUT, "seg3d_init.pt"))
    print("seg3d_init", len(sd), "tensors")

    dims = [32, 32, 16]
    cfg = R.encoder_config(ns.shared, dims=dims, num_modes=2, num_attractors=5, pos_dim=2, qk_have_bias=True)
    enc = R.build_encoder(cfg, seed=11).train()
    torch.manual_seed(12)
    x = torch.randn(3, 20, 32)
    pos = O.voxels_pos_for_grid((4, 5), (8, 8), 3)
    mask = torch.ones(3, 20, 1, dtype=torch.bool)
    with R.quiet():
        y = enc(x, pos, mask, torch.Size((4, 5)))
    torch.save(dict(kind="enc_train", dims=dims, num_modes=2, grid=[4, 5], x=x, voxels_pos=pos, vmask=mask,
                    state_dict=dict(enc.state_dict()), out=y.detach()),
               os.path.join(OUT, "enc_train.pt"))
    print("enc_train out", tuple(y.shape))


def gen_infer():
    """Sliding-window inference fixtures produced by the reference's own test_util3d.test_single_case (un-padded volumes:
    the reference's padding branch hands F.pad the pads in the wrong dimension order, test_util3d.py:119-120, and cannot run)."""
    import types
    R.load()
    for name in ("h5py", "nibabel", "medpy", "medpy.metric", "common_util", "tqdm"):
        if name not in sys.modules:
            m = types.ModuleType(name)
            sys.modules[name] = m
    sys.modules["medpy"].metric = sys.modules["medpy.metric"]
    sys.modules["common_util"].get_filename = lambda p: p
    sys.modules["tqdm"].tqdm = lambda x, **k: x
    import test_util3d as T3                                    # /root/reference/code/test_util3d.py
    from tests.helpers import AffinePickNet
    zeros = torch.zeros

    def zeros_cpu(*a, **kw):
        if kw.get("device") == "cuda":
            kw["device"] = "cpu"
        return zeros(*a, **kw)

    cases = {}
    specs = [("brats_same", "brats", 4, (4, 40, 36, 30), (24, 24, 16), (24, 24, 16), 3, 12, 8),
             ("brats_resized", "brats", 4, (4, 33, 41, 27), (24, 20, 16), (16, 16, 12), 4, 10, 8),
             ("argmax", "other", 3, (2, 30, 30, 20), (16, 16, 12), (16, 16, 12), 5, 8, 6)]
    for key, task, K, shp, ops_, ips, bs, sxy, szz in specs:
        torch.manual_seed(len(key))
        image = torch.randn(*shp) * 2.0
        a = [1.0 + 0.5 * k for k in range(K)]
        b = [-0.3 + 0.2 * k for k in range(K)]
        ch = [k % shp[0] for k in range(K)]
        net = AffinePickNet(a, b, ch)
        torch.zeros = zeros_cpu
        try:
            hard, soft = T3.test_single_case(net, image, ops_, ips, bs, sxy, szz, task, "segtran", K)
        finally:
            torch.zeros = zeros
        cases[key] = dict(task=task, K=K, image=image, orig_patch=ops_, input_patch=ips, batch_size=bs, stride_xy=sxy,
                          stride_z=szz, a=a, b=b, ch=ch, hard=hard, soft=soft)
        print("infer", key, tuple(hard.shape), tuple(soft.shape), float(soft.mean()))
    torch.save(dict(kind="infer", cases=cases), os.path.join(OUT, "infer_sw.pt"))


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(4)
    if len(sys.argv) > 1 and sys.argv[1] == "train":
        gen_train()
        return
    if len(sys.argv) > 1 and sys.argv[1] == "infer":
        gen_infer()
        return
    if len(sys.argv) > 1 and sys.argv[1] == "poly":
        gen_poly()
        return
    if len(sys.argv) > 1 and sys.argv[1] == "construction":
        gen_construction()
        return
    if len(sys.argv) > 1 and sys.argv[1] == "variants":
        gen_encoder("enc2d_nosqueeze", [64, 64], 4, 8, 2, True, (6, 7), 2, seed=21, squeeze=False)
        gen_encoder("enc3d_sqffn", [64, 64], 4, 16, 3, True, (3, 4, 5), 2, seed=22, sq_ffn=True)
        gen_encoder("enc3d_sharedout", [64, 64], 4, 16, 3, True, (3, 4, 5), 2, seed=23, out_type="shared")
        return
    gen_encoder("enc3d_small", [64, 64], 4, 16, 3, True, (3, 4, 5), 2, seed=1)
    gen_encoder("enc2d_compress", [64, 64, 32], 4, 8, 2, False, (6, 7), 2, seed=2)
    gen_encoder("enc3d_clamp", [64, 64], 4, 16, 3, True, (3, 4, 5), 1, seed=7, wscale=60.0)
    gen_encoder("enc3d_ragged", [96, 96], 4, 24, 3, True, (5, 3, 7), 3, seed=9)       # N=105: not a tile multiple
    gen_seg3d("seg3d_tiny")
    gen_seg2d("seg2d_tiny")
    gen_infer()
    gen_poly()


if __name__ == "__main__":
    main()
