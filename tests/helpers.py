"""Shared test helpers (tolerances, fixture loading, oracle drivers)."""
import hashlib
import os

import torch

from oracle import segtran_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    return torch.load(os.path.join(GOLDEN, name + ".pt"), map_location="cpu", weights_only=False)


def rel_err(a, b):
    """max|a-b| / max|b| — the '1e-3 rel' of BASELINE.json's north_star, as used in every parity test."""
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def tensor_digest(t):
    """SHA-256 of a tensor's dtype, shape and bytes: two tensors have the same digest iff they are bit-identical, so a
    fixture can pin exact values without storing them."""
    t = t.detach().cpu().contiguous()
    h = hashlib.sha256(("%s %s" % (t.dtype, tuple(t.shape))).encode())
    h.update(t.reshape(-1).view(torch.uint8).numpy().tobytes())
    return h.hexdigest()


def state_digests(sd):
    """name -> tensor_digest, in state_dict order."""
    return {k: tensor_digest(v) for k, v in sd.items()}


def rms_rel(a, b):
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    return float((a - b).pow(2).mean().sqrt() / b.pow(2).mean().sqrt().clamp_min(1e-30))


def oracle_encoder(fx, x=None, dtype=torch.float32, collect=None):
    p = {"voxel_fusion." + k: v.to(dtype) for k, v in fx["state_dict"].items()}
    x = fx["x"] if x is None else x
    return O.fusion_encoder(p, "voxel_fusion.", x.to(dtype), fx["voxels_pos"].to(dtype), fx["vmask"], fx["dims"],
                            fx["num_modes"], collect=collect, **variant_kwargs(fx)), p


def variant_kwargs(fx):
    return dict(use_squeezed_transformer=fx.get("use_squeezed_transformer", True),
                has_FFN_in_squeeze=fx.get("has_FFN_in_squeeze", False),
                trans_output_type=fx.get("trans_output_type", "private"))


def encoder_config(cfg_cls, *, dims, num_modes=4, num_attractors=16, pos_dim=3, qk_have_bias=True, dropout=0.0):
    """SegtranConfig (reference's or ours) with what Segtran{2d,3d}Config.update_config would derive."""
    cfg = cfg_cls()
    cfg.num_translayers = len(dims) - 1
    cfg.translayer_dims = list(dims)
    cfg.translayer_compress_ratios = [1] * len(dims)
    cfg.trans_in_dim, cfg.trans_out_dim, cfg.min_feat_dim = dims[0], dims[-1], min(dims)
    cfg.num_modes, cfg.num_attractors, cfg.pos_dim, cfg.qk_have_bias = num_modes, num_attractors, pos_dim, qk_have_bias
    cfg.hidden_dropout_prob = cfg.attention_probs_dropout_prob = dropout
    return cfg


def build_b200_encoder(fx, device="cuda", dropout=0.0):
    import segtran_b200.networks.segtran_shared as S
    cfg = encoder_config(S.SegtranConfig, dims=fx["dims"], num_modes=fx["num_modes"],
                         num_attractors=fx["num_attractors"], pos_dim=fx["pos_dim"], qk_have_bias=fx["qk_have_bias"],
                         dropout=dropout)
    cfg.use_squeezed_transformer = fx.get("use_squeezed_transformer", True)
    cfg.has_FFN_in_squeeze = fx.get("has_FFN_in_squeeze", False)
    cfg.trans_output_type = fx.get("trans_output_type", "private")
    enc = S.SegtranFusionEncoder(cfg, "Fusion")
    init = S.SegtranInitWeights(cfg)
    enc.apply(init.tie_qk)
    enc.load_state_dict(fx["state_dict"], strict=True)
    return enc.to(device)


class AffinePickNet(torch.nn.Module):
    """Stand-in segmentation net for the inference-path fixtures: class k's score = a[k] * x[:, ch[k]] + b[k] — element-wise, so
    it is reproducible to the last ulp on any device (the sliding-window logic is what the fixtures pin, not a network)."""

    def __init__(self, a, b, ch):
        super().__init__()
        self.a, self.b, self.ch = [float(v) for v in a], [float(v) for v in b], [int(c) for c in ch]

    def forward(self, x):
        return torch.stack([x[:, c] * a + b for a, b, c in zip(self.a, self.b, self.ch)], dim=1)
