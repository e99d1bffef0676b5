"""CPU oracle for the Segtran Squeeze-and-Expansion hot path.

TEST INFRASTRUCTURE ONLY.  Nothing in ``segtran_b200/`` may import this module; only
``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / ``--impl reference``
legs use it, and only as the checker (or as the timed CPU baseline), never as the product path.

This is a functional restatement (plain PyTorch on CPU, fp32 by default, fp64 if the inputs are
fp64) of the reference algorithm in askerlee/segtran, written against the reference's
*state_dict key names* so that a reference checkpoint / ``state_dict()`` can be fed in unchanged.
Every function cites the reference file:line it follows (paths relative to the reference root,
``code/networks/...``).

Parity pinning: the reference ships no golden vectors or unit tests (SURVEY.md §4), so this
restatement is pinned against the reference *itself*, imported in the build container:
``oracle/gen_golden.py`` runs the real ``SegtranFusionEncoder`` / ``Segtran3d`` / ``Segtran2d``
modules on seeded inputs and stores inputs, weights, outputs and gradients under ``tests/golden/``;
``tests/test_oracle_golden.py`` checks this file against those fixtures.

The restatement deliberately keeps the reference's formulation (no algebraic shortcuts): separate
K/V projections of all tokens, the un-collapsed segmentation head, etc.  The CUDA path is free to
restructure; the parity tests then prove the restructuring is value-preserving.
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Sequence

import torch
import torch.nn.functional as F

Tensor = torch.Tensor
Params = Dict[str, Tensor]

LN_EPS = 1e-12          # every LayerNorm on the path: segtran_shared.py:263,288,371,885,888,984


# ----------------------------------------------------------------------------------------------
# helpers
# ----------------------------------------------------------------------------------------------
def gen_all_indices(shape: Sequence[int], device="cpu") -> Tensor:
    """Integer coordinates of every cell of a grid, row-major: [*shape, len(shape)].
    Follows segtran_shared.py:28-36."""
    axes = [torch.arange(s, device=device) for s in shape]
    return torch.stack(torch.meshgrid(*axes, indexing="ij"), dim=len(shape))


def layer_norm(x: Tensor, g: Optional[Tensor] = None, b: Optional[Tensor] = None) -> Tensor:
    """LayerNorm over the last dim, biased variance, eps=1e-12 (nn.LayerNorm semantics)."""
    mu = x.mean(dim=-1, keepdim=True)
    var = ((x - mu) ** 2).mean(dim=-1, keepdim=True)
    y = (x - mu) * torch.rsqrt(var + LN_EPS)
    if g is not None:
        y = y * g + b
    return y


def gelu_erf(x: Tensor) -> Tensor:
    """Exact (erf) GELU == F.gelu default; config.act_fun, segtran_shared.py:107."""
    return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))


def _dropout(x: Tensor, p: float, training: bool) -> Tensor:
    return F.dropout(x, p, training) if (training and p > 0) else x


# ----------------------------------------------------------------------------------------------
# positional code  (segtran_shared.py:979-998, 1228-1238)
# ----------------------------------------------------------------------------------------------
def pos_lsinu(voxels_pos: Tensor, w: Tensor, b: Tensor) -> Tensor:
    """Learnable-sinusoid positional code.
    voxels_pos [B,N,pd] -> [B,N,C0].  pos/pos.max() (global scalar max, :1231); Linear(pd->C0)
    (:991); sin on even output columns, cos on odd ones, interleaved (:992-995); LayerNorm without
    affine (:996)."""
    pos_n = voxels_pos / voxels_pos.max()
    e = pos_n @ w.t() + b
    pe = torch.empty_like(e)
    pe[..., 0::2] = torch.sin(e[..., 0::2])
    pe[..., 1::2] = torch.cos(e[..., 1::2])
    return layer_norm(pe)


# ----------------------------------------------------------------------------------------------
# CrossAttFeatTrans + ExpandedFeatTrans   (segtran_shared.py:404-476, 553-610)
# ----------------------------------------------------------------------------------------------
def cross_att(p: Params, pre: str, in_query: Tensor, in_key: Tensor, num_modes: int, feat_dim: int,
              has_ffn: bool, *, attn_clip: float = 500.0, att_drop: float = 0.0,
              hid_drop: float = 0.0, training: bool = False, trans_output_type: str = "private",
              stats: Optional[dict] = None) -> Tensor:
    """One CrossAttFeatTrans.forward (:553-610) followed by its ExpandedFeatTrans (:404-476).

    in_query [B,U1,C], in_key [B,U2,C].  Q and K share one weight/bias (tie_qk 'shared',
    :528-531; the state_dict carries both names, we read ``query``).  Returns [B,U1,feat_dim].
    """
    M = num_modes
    Wq = p[pre + "query.weight"]
    bq = p.get(pre + "query.bias")
    Wk = p.get(pre + "key.weight", Wq)
    bk = p.get(pre + "key.bias", bq)
    B, U1, C = in_query.shape
    U2 = in_key.shape[1]
    d = C // M                                                       # attention_mode_dim :484
    q = F.linear(in_query, Wq, bq).view(B, U1, M, d).permute(0, 2, 1, 3)     # :559,:548-551
    k = F.linear(in_key, Wk, bk).view(B, U2, M, d).permute(0, 2, 1, 3)       # :560
    s = torch.matmul(q, k.transpose(-1, -2)) / math.sqrt(d)          # :566-567
    smax = float(s.detach().max())                                            # :570
    if stats is not None:
        stats.setdefault("max_attn", []).append(smax)
    if smax > attn_clip:                                             # :578-580
        s = torch.clamp(s, -attn_clip, attn_clip)
    if stats is not None:
        stats.setdefault("scores", []).append(s)
    probs = _dropout(torch.softmax(s, dim=-1), att_drop, training)   # :601-605

    # ---- ExpandedFeatTrans.forward(in_key, probs) ----
    Fd = feat_dim
    Wv = p[pre + "out_trans.first_linear.weight"]                    # [M*F, C], no bias (v_has_bias False)
    bv = p.get(pre + "out_trans.first_linear.bias")
    v = F.linear(in_key, Wv, bv)                                     # :414   [B,U2,M*F], channel = m*F+f
    v = v.view(B, U2, M, Fd).permute(0, 2, 1, 3)                     # :416-419  [B,M,U2,F]
    u = torch.matmul(probs, v)                                       # :447   [B,M,U1,F]
    if not has_ffn:                                                  # :452-457
        w = torch.softmax(F.linear(u, p[pre + "out_trans.feat_softaggr.feat2score.weight"],
                                   p[pre + "out_trans.feat_softaggr.feat2score.bias"]), dim=1)
        z = (u * w).sum(dim=1)                                       # :318-325 (identity when M == 1)
        return layer_norm(z, p[pre + "out_trans.first_norm_layer.weight"],
                          p[pre + "out_trans.first_norm_layer.bias"])
    # MMSharedMid :232-251 — one Linear(F->F) shared by all modes, erf-GELU, dropout
    g = gelu_erf(F.linear(u, p[pre + "out_trans.intermediate.shared_linear.weight"],
                          p[pre + "out_trans.intermediate.shared_linear.bias"]))
    g = _dropout(g, hid_drop, training)
    if trans_output_type == "private":
        # MMPrivateOutput :266-275 — grouped 1x1 Conv1d == per-mode Linear; the residual is computed
        # and then DISCARDED (:269-272), so no shortcut here.
        Wo = p[pre + "out_trans.output.group_linear.weight"].view(M, Fd, Fd)       # [M*F, F, 1]
        bo = p[pre + "out_trans.output.group_linear.bias"].view(M, 1, Fd)
        y = torch.einsum("bmnf,mof->bmno", g, Wo) + bo
    else:
        # MMSharedOutput :291-308 — shared Linear, residual kept (:305)
        y = F.linear(g, p[pre + "out_trans.output.shared_linear.weight"],
                     p[pre + "out_trans.output.shared_linear.bias"]) + u
    y = _dropout(y, hid_drop, training)
    y = layer_norm(y, p[pre + "out_trans.output.resout_norm_layer.weight"],
                   p[pre + "out_trans.output.resout_norm_layer.bias"])          # :274
    # LearnedSoftAggregate :318-325
    w = torch.softmax(F.linear(y, p[pre + "out_trans.feat_softaggr.feat2score.weight"],
                               p[pre + "out_trans.feat_softaggr.feat2score.bias"]), dim=1)
    return (y * w).sum(dim=1)


def squeezed_layer(p: Params, pre: str, h: Tensor, num_modes: int, feat_dim: int, sq_ffn: bool = False, **kw) -> Tensor:
    """SqueezedAttFeatTrans.forward (:809-816): attractors attend to tokens (1 mode; FFN only with
    --squeezeuseffn, config1 :796-799), then tokens attend to the updated attractors (M modes, full FFN)."""
    B, N, C = h.shape
    att = p[pre + "attractors"].expand(B, -1, -1)
    a = cross_att(p, pre + "in_ator_trans.", att, h, 1, C, sq_ffn, **kw)
    return cross_att(p, pre + "ator_out_trans.", h, a, num_modes, feat_dim, True, **kw)


def fusion_encoder(p: Params, pre: str, vfeat: Tensor, voxels_pos: Tensor, vmask: Tensor,
                   translayer_dims: Sequence[int], num_modes: int = 4, *, pos_code_weight: float = 1.0,
                   hid_drop: float = 0.0, att_drop: float = 0.0, training: bool = False,
                   attn_clip: float = 500.0, trans_output_type: str = "private",
                   collect: Optional[dict] = None, use_squeezed_transformer: bool = True,
                   has_FFN_in_squeeze: bool = False) -> Tensor:
    """SegtranFusionEncoder.forward (:907-975) with squeezed attention, pos_code_type 'lsinu'.
    vfeat [B,N,C0], voxels_pos [B,N,pd], vmask [B,N,1] (int/bool/float), returns [B,N,C_last]."""
    pe = pos_lsinu(voxels_pos.to(vfeat.dtype), p[pre + "pos_code_layer.pos_coder.pos_fc.weight"],
                   p[pre + "pos_code_layer.pos_coder.pos_fc.bias"])
    x = vfeat
    layers = []
    for i in range(len(translayer_dims) - 1):
        C, Fd = translayer_dims[i], translayer_dims[i + 1]
        h = layer_norm(x, p[pre + f"vfeat_norm_layers.{i}.weight"],
                       p[pre + f"vfeat_norm_layers.{i}.bias"])                   # :916
        h = layer_norm(h + pos_code_weight * pe[:, :, :C])                      # :930-934
        if i == 0:
            h = _dropout(h, hid_drop, training)                                 # :944-945
        h = h * vmask.to(h.dtype)                                               # :946
        kw = dict(attn_clip=attn_clip, att_drop=att_drop, hid_drop=hid_drop, training=training,
                  trans_output_type=trans_output_type, stats=collect)
        if use_squeezed_transformer:
            x = squeezed_layer(p, pre + f"translayers.{i}.", h, num_modes, Fd, sq_ffn=has_FFN_in_squeeze, **kw)
        else:                                     # --nosqueeze (:877-878): plain self cross-attention over all tokens
            x = cross_att(p, pre + f"translayers.{i}.", h, h, num_modes, Fd, True, **kw)
        layers.append(x)
    if collect is not None:
        collect["layers_vfeat"] = layers
    return x


# ----------------------------------------------------------------------------------------------
# flatten / scatter / segmentation head  (segtran3d.py:326-332, 364-386, 478-496;
#                                          segtran2d.py:264-269, 304-306, 421-436)
# ----------------------------------------------------------------------------------------------
def flatten_tokens(feat: Tensor) -> Tensor:
    """[B,C,*grid] channels-first -> [B,N,C] token-major (segtran3d.py:328-330 / segtran2d.py:264-267)."""
    B, C = feat.shape[:2]
    return feat.reshape(B, C, -1).transpose(1, 2).contiguous()


def scatter_tokens(tok: Tensor, grid: Sequence[int]) -> Tensor:
    """[B,N,F] -> [B,F,*grid] (segtran3d.py:478-480 / segtran2d.py:421-423)."""
    B, N, Fd = tok.shape
    return tok.transpose(1, 2).reshape(B, Fd, *grid)


def seg_head_3d(p: Params, curr_feat: Tensor, vfeat_fused: Tensor, grid: Sequence[int],
                out_size: Sequence[int], D_pool_K: int = 2) -> Tensor:
    """Voxel-wise head, reference formulation.
    curr_feat [B,Cf,D1,H1,W1] (output of the out-FPN pyramid, segtran3d.py:347-359),
    vfeat_fused [B,N,F] tokens on ``grid`` = (D2,H2,W2), out_size = (H,W,D) of the input volume.
    :364-367 trilinear upsample of the fused tokens + out_fpn_bridgeconv3d(curr_feat);
    :381-386 trilinear depth x D_pool_K; :488-490 permute to (H,W,D), out_conv3d 1x1;
    :495 trilinear to the input size."""
    vf = scatter_tokens(vfeat_fused, grid)
    up = F.interpolate(vf, size=curr_feat.shape[2:], mode="trilinear", align_corners=False)
    x = F.conv3d(curr_feat, p["out_fpn_bridgeconv3d.weight"], p["out_fpn_bridgeconv3d.bias"]) + up
    if D_pool_K > 1:
        sz = list(x.shape[2:])
        sz[0] *= D_pool_K
        x = F.interpolate(x, size=sz, mode="trilinear", align_corners=False)
    x = x.permute(0, 1, 3, 4, 2)
    s = F.conv3d(x, p["out_conv3d.weight"], p["out_conv3d.bias"])
    return F.interpolate(s, size=tuple(out_size), mode="trilinear", align_corners=False)


def seg_head_2d(p: Params, curr_feat: Tensor, vfeat_fused: Tensor, grid: Sequence[int],
                out_size: Sequence[int]) -> Tensor:
    """2-D head (segtran2d.py:304-306 bridgeconv + bilinear upsample of fused tokens; :427 out_conv
    1x1; :435-436 bilinear to the input size)."""
    vf = scatter_tokens(vfeat_fused, grid)
    up = F.interpolate(vf, size=curr_feat.shape[2:], mode="bilinear", align_corners=False)
    if "out_fpn_bridgeconv.weight" in p:                 # nn.Identity when dims agree (segtran2d.py:177-180)
        x = F.conv2d(curr_feat, p["out_fpn_bridgeconv.weight"], p["out_fpn_bridgeconv.bias"]) + up
    else:
        x = curr_feat + up
    s = F.conv2d(x, p["out_conv.weight"], p["out_conv.bias"])
    return F.interpolate(s, size=tuple(out_size), mode="bilinear", align_corners=False)


def voxels_pos_for_grid(grid: Sequence[int], scales: Sequence[float], B: int, dtype=torch.float32,
                        device="cpu") -> Tensor:
    """Pixel coordinates of the token grid: gen_all_indices(grid) * per-axis model scale, repeated over
    the batch (segtran3d.py:442-470, segtran2d.py:364-382)."""
    idx = gen_all_indices(tuple(grid), device=device).reshape(-1, len(grid)).to(dtype)
    idx = idx * torch.tensor([list(scales)], dtype=dtype, device=device)
    return idx.unsqueeze(0).repeat(B, 1, 1)


def hot_path_3d(p: Params, feat_fpn: Tensor, curr_feat: Tensor, vmask: Tensor, out_size: Sequence[int],
                translayer_dims: Sequence[int], num_modes: int = 4, D_pool_K: int = 2, **kw) -> Tensor:
    """flatten -> fusion encoder -> scatter -> head, i.e. segtran3d.py:326-332 + :442-498 with the
    backbone / FPN pyramids factored out.
    feat_fpn [B,C0,D2,H2,W2] (in-FPN output after depth pooling), curr_feat [B,Cf,D1,H1,W1],
    vmask [B,N] in {0,1}, out_size = (H,W,D).  Parameter names as in Segtran3d.state_dict()."""
    B = feat_fpn.shape[0]
    grid = tuple(feat_fpn.shape[2:])
    H, W, D = out_size
    scales = (D // grid[0], H // grid[1], W // grid[2])                      # segtran3d.py:446-456
    pos = voxels_pos_for_grid(grid, scales, B, feat_fpn.dtype, feat_fpn.device)
    tok = flatten_tokens(feat_fpn)
    fused = fusion_encoder(p, "voxel_fusion.", tok, pos, vmask.reshape(B, -1, 1), translayer_dims,
                           num_modes, **kw)
    return seg_head_3d(p, curr_feat, fused, grid, out_size, D_pool_K)


def hot_path_2d(p: Params, feat_fpn: Tensor, curr_feat: Tensor, vmask: Tensor, out_size: Sequence[int],
                translayer_dims: Sequence[int], num_modes: int = 4, **kw) -> Tensor:
    """2-D counterpart (segtran2d.py:264-269 + :362-436)."""
    B = feat_fpn.shape[0]
    grid = tuple(feat_fpn.shape[2:])
    H, W = out_size
    pos = voxels_pos_for_grid(grid, (H // grid[0], W // grid[1]), B, feat_fpn.dtype, feat_fpn.device)
    tok = flatten_tokens(feat_fpn)
    fused = fusion_encoder(p, "voxel_fusion.", tok, pos, vmask.reshape(B, -1, 1), translayer_dims,
                           num_modes, **kw)
    return seg_head_2d(p, curr_feat, fused, grid, out_size)


def polyformer_layer(p: Params, pre: str, in_feat: Tensor, num_modes: int = 4, **kw) -> Tensor:
    """PolyformerLayer.forward (code/networks/polyformer.py:35-60, chan_axis = 1, poly_do_layernorm False):
    2x2 average pooling (:39), channels swapped with the LAST dim and flattened to tokens (:41, :46), attractors attend
    to the tokens and the tokens to the updated attractors — both CrossAttFeatTrans WITHOUT the FFN, M modes soft-aggregated
    (segtran_shared.py:452-457) — then back to the map layout, bilinear up-sampling (:56-57) and the residual (:58)."""
    B, C = in_feat.shape[:2]
    half0 = F.avg_pool2d(in_feat, 2)
    half = half0.transpose(1, -1)
    vfeat = half.reshape(B, -1, C)
    att = p[pre + "attractors"].expand(B, -1, -1)
    a = cross_att(p, pre + "in_ator_trans.", att, vfeat, num_modes, C, False, **kw)
    out = cross_att(p, pre + "ator_out_trans.", vfeat, a, num_modes, C, False, **kw)
    out = out.transpose(1, -1).reshape(half0.shape)
    up = F.interpolate(out, size=in_feat.shape[2:], mode="bilinear", align_corners=False)
    return in_feat + up


def dice_hard(a: Tensor, b: Tensor) -> float:
    """2|A∩B| / (|A|+|B|) on boolean masks (test_util2d.py:229-237 restated; 1.0 when both empty)."""
    a = a.bool()
    b = b.bool()
    den = int(a.sum()) + int(b.sum())
    return 1.0 if den == 0 else 2.0 * int((a & b).sum()) / den
