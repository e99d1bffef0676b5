#!/usr/bin/env python
"""Benchmark of the Segtran hot path on B200 (contract: see the task statement / DESIGN.md §Measurement).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config 1..5] [--scaling weak|strong]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
         bench.py --gpus N --steps K --warmup W

Workloads = the five BASELINE.json configs (SURVEY.md §8a table).  The default (`--config 4`) is the one the metric is
quoted on: Segtran3d BraTS 112^3 x 4ch, translayers=1, attractors=1024, modes=4, per-GPU batch 4, training mode
(dropout 0.2, reference default train3d.py:213).  One step = one training step of the hot path
    token flatten -> Squeeze-and-Expansion stack -> scatter -> voxel/pixel-wise head -> BCE + Dice loss (train3d.py:731-756)
    -> backward -> (N>1: NCCL all-reduce of the flat gradient bucket) -> BertAdam update (optimization.py, --gradclip 0.1)
on synthetic feature tensors of the shapes the backbone / FPN pyramids produce at that config and synthetic n-hot masks;
gradients flow to both feature tensors and to every parameter.  metric = voxels/s (pixels/s in 2-D) = global batch *
prod(input size) / step time.  `--impl reference` times the CPU oracle of the same step at the same batch size; the
`cuda_eager_baseline` object of the N=1 line is the same reference formulation (oracle/, plain functional PyTorch) run on
the GPU — the "reference PyTorch-CUDA" figure BASELINE.json's >=10x target refers to.
"""
from __future__ import annotations

import argparse
import contextlib
import json
import os
import subprocess
import sys
import threading
import time
from argparse import Namespace

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# SURVEY.md §8a: per-config shapes probed from the reference.  `Cf`/`sp1`: channels / resolution of the out-FPN feature map
# that enters the head; `ref_gflop`: forward FLOPs per sample of the fusion stack in the reference's formulation (§8d).
CONFIGS = {
    1: dict(kind="2d", title="Segtran2d fundus 288^2 eff-b4 translayers=1 bs=2", backbone="eff-b4", B=2, S=288, grid=(36, 36),
            dims=[1792, 1792], compress=[1, 1], Cf=160, sp1=(144, 144), classes=3, attractors=256, modes=4, qk_bias=True,
            ref_gflop=109.7, precision="tf32"),
    2: dict(kind="2d", title="Segtran2d fundus 576^2 eff-b4 translayers=3 layercompress=1,1,2,2 bs=6 --noqkbias",
            backbone="eff-b4", B=6, S=576, grid=(72, 72), dims=[1792, 1792, 896, 448], compress=[1, 1, 2, 2], Cf=160,
            sp1=(288, 288), classes=3, attractors=256, modes=4, qk_bias=False, ref_gflop=661.4, precision="tf32"),
    3: dict(kind="2d", title="Segtran2d polyp 352^2 resnet50 translayers=2 bs=16", backbone="resnet50", B=16, S=352,
            grid=(44, 44), dims=[2048, 2048, 2048], compress=[1, 1, 1], Cf=1024, sp1=(176, 176), classes=2, attractors=256,
            modes=4, qk_bias=True, ref_gflop=411.5, precision="tf32"),
    4: dict(kind="3d", title="Segtran3d BraTS 112^3x4ch translayers=1 attractors=1024 bs=4", backbone="i3d", B=4, S=112,
            grid=(14, 14, 14), dims=[1024, 1024], compress=[1, 1], Cf=832, sp1=(56, 56, 56), classes=4, attractors=1024,
            modes=4, qk_bias=True, ref_gflop=116.5, precision="tf32"),
    5: dict(kind="3d", title="Segtran3d BraTS 144^3x4ch translayers=2 attractors=2048 bs=2/GPU", backbone="i3d", B=2, S=144,
            grid=(18, 18, 18), dims=[1024, 1024, 1024], compress=[1, 1, 1], Cf=832, sp1=(72, 72, 72), classes=4,
            attractors=2048, modes=4, qk_bias=True, ref_gflop=663.1, precision="tf32"),
}
DROPOUT = 0.2
# training-step settings of the reference for --net segtran on BraTS (train3d.py:211-212, :223, :61, :73)
TRAIN = dict(lr=2e-4, decay=1e-4, grad_clip=0.1, dice_w=0.5, bce_weight=[0., 3., 1., 1.75], warmup=0.05, t_total=10000)


def metric_name(c):
    if c["kind"] == "3d":
        return "voxels/sec fwd+bwd Segtran3d BraTS %d^3 bs=%d hot path" % (c["S"], c["B"])
    return "pixels/sec fwd+bwd Segtran2d %d^2 bs=%d hot path" % (c["S"], c["B"])


def unit_name(c):
    return "voxels/s" if c["kind"] == "3d" else "pixels/s"


def units_per_sample(c):
    return c["S"] ** (3 if c["kind"] == "3d" else 2)


def workload_name(c, B):
    return ("%s (per-GPU batch %d): hot path = flatten + squeeze-expansion stack + %s-wise head, fwd + BCE/Dice loss + bwd + "
            "BertAdam step, dropout %.1f" % (c["title"], B, "voxel" if c["kind"] == "3d" else "pixel", DROPOUT))


def model_args(c, device, dropout):
    a = Namespace(num_classes=c["classes"], backbone_type=c["backbone"], use_pretrained=False,
                  num_attractors=c["attractors"], num_translayers=len(c["dims"]) - 1, num_modes=c["modes"],
                  trans_output_type="private", mid_type="shared", device=device, in_fpn_layers="34",
                  out_fpn_layers="1234", in_fpn_scheme="AN", out_fpn_scheme="AN",
                  translayer_compress_ratios=list(c["compress"]), dropout_prob=dropout, tie_qk_scheme="shared",
                  qk_have_bias=c["qk_bias"], use_squeezed_transformer=True, pos_code_type="lsinu")
    if c["kind"] == "3d":
        a.orig_in_channels, a.D_pool_K, a.inchan_to3_scheme, a.D_groupsize = 4, 2, "bridgeconv", 1
    else:
        a.use_global_bias, a.num_modalities = False, 0
    return a


def build_net(c, device, dropout=DROPOUT, seed=1337):
    """The drop-in shell (Identity backbone: the bench feeds the FPN outputs directly) with seed-defined weights."""
    torch.manual_seed(seed)
    with contextlib.redirect_stdout(open(os.devnull, "w")):
        if c["kind"] == "3d":
            from segtran_b200.networks import segtran3d as S
            cfg = S.Segtran3dConfig()
            cfg.update_config(model_args(c, device, dropout))
            net = S.Segtran3d(cfg, backbone=torch.nn.Identity())
        else:
            from segtran_b200.networks import segtran2d as S
            cfg = S.Segtran2dConfig()
            cfg.update_config(model_args(c, device, dropout))
            net = S.Segtran2d(cfg, backbone=torch.nn.Identity())
    assert [int(d) for d in cfg.translayer_dims] == list(c["dims"]), (cfg.translayer_dims, c["dims"])
    net.scales_printed = True
    return net


def hot_params(net, c):
    head = [net.out_fpn_bridgeconv3d, net.out_conv3d] if c["kind"] == "3d" else [net.out_fpn_bridgeconv, net.out_conv]
    ps = list(net.voxel_fusion.parameters())
    for m in head:
        ps += list(m.parameters())
    return ps


def hot_state(net, c):
    """name -> tensor of the hot-path parameters, keyed like the reference's state_dict (what the oracle consumes)."""
    pre = ("out_fpn_bridgeconv3d.", "out_conv3d.") if c["kind"] == "3d" else ("out_fpn_bridgeconv.", "out_conv.")
    return {k: v for k, v in net.state_dict().items() if k.startswith("voxel_fusion.") or k.startswith(pre)}


def loss_weights(c, device):
    K = c["classes"]
    if c["kind"] == "3d":
        pw = torch.tensor(TRAIN["bce_weight"][:K], device=device)
        pw = pw * (K - 1) / pw.sum()                                       # train3d.py:517-518
    else:
        pw = torch.ones(K, device=device)                                  # 2-D drivers: unweighted BCE
    cw = torch.ones(K, device=device)
    cw[0] = 0
    cw = cw / cw.sum()                                                     # train3d.py:686-690
    return pw, cw


def synthetic_batch(c, B, device, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    sp = (c["S"],) * (3 if c["kind"] == "3d" else 2)
    feat = torch.randn(B, c["dims"][0], *c["grid"], generator=g)
    curr = torch.randn(B, c["Cf"], *c["sp1"], generator=g)
    Y = (torch.rand(B, c["classes"], *sp, generator=g) > 0.7)              # synthetic n-hot masks (SURVEY 8d)
    return feat.to(device), curr.to(device), Y.to(device)


# ----------------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md recipe)
# ----------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [t.strip() for t in out.strip().split(",")]
                if len(f) >= 6:
                    self.samples.append(f)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        mhz = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": mhz[len(mhz) // 2] if mhz else None,
                "sm_max_mhz": int(self.samples[0][1]) if self.samples[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.samples)}


# ----------------------------------------------------------------------------------------------------------
# reference formulation (oracle/): CPU arm, cpu_baseline, and the PyTorch-CUDA eager baseline
# ----------------------------------------------------------------------------------------------------------
def oracle_step_factory(c, B, device="cpu"):
    """One training step (fwd + loss + bwd + clip + BertAdam) of the reference FORMULATION on `device` for B samples of
    config c, with the same seed-defined initial weights as the B200 arm (the shell's own state_dict feeds the oracle)."""
    from oracle import segtran_oracle as O
    from oracle import train_oracle as T
    net = build_net(c, "cpu")
    p = {k: v.detach().clone().to(device).requires_grad_() for k, v in hot_state(net, c).items()
         if ".key." not in k}                                        # key.* aliases query.* (tie_qk 'shared')
    del net
    feat, curr, Y = synthetic_batch(c, B, device, 4242)
    feat.requires_grad_()
    curr.requires_grad_()
    Y = Y.float()
    pw, cw = loss_weights(c, device)
    N = 1
    for s in c["grid"]:
        N *= s
    vmask = torch.ones(B, N, device=device)
    sp = (c["S"],) * (3 if c["kind"] == "3d" else 2)
    params = list(p.values())
    leaves = params + [feat, curr]
    state = {}

    def step():
        for v in leaves:
            v.grad = None
        if c["kind"] == "3d":
            y = O.hot_path_3d(p, feat, curr, vmask, sp, c["dims"], c["modes"], 2, hid_drop=DROPOUT, att_drop=DROPOUT,
                              training=True)
        else:
            y = O.hot_path_2d(p, feat, curr, vmask, sp, c["dims"], c["modes"], hid_drop=DROPOUT, att_drop=DROPOUT,
                              training=True)
        loss, _, _ = T.seg_loss(y, Y, pw, cw, TRAIN["dice_w"])             # train3d.py:731-756
        loss.backward()
        with torch.no_grad():                                              # train3d.py:760-762
            gs = [v.grad for v in params]
            T.clip_grad_norm([gg for gg in gs if gg is not None], TRAIN["grad_clip"])
            T.bert_adam_step([v.data for v in params], gs, state, lr=[TRAIN["lr"]] * len(params),
                             weight_decay=[TRAIN["decay"]] * len(params), warmup=TRAIN["warmup"], t_total=TRAIN["t_total"])
        return loss.detach()

    desc = "B=%d of config (%s), full fwd + BCE/Dice loss + bwd + clip + BertAdam step, reference formulation, dropout %.1f" % (
        B, c["title"], DROPOUT)
    return step, B * units_per_sample(c), desc


def time_oracle_cpu(c, B, steps, warmup, budget_s):
    """Times the CPU oracle at the workload's own per-GPU batch (same config as the B200 arm).  The number of warm-up /
    timed steps is cut to fit the budget, down to timing a single step; only if even one full-size step does not fit is
    the batch reduced (and the line says so).  On many-core hosts PyTorch's CPU kernels can be slower with every core
    than with a few dozen threads, so a second thread count is probed and the faster one kept (`cores` = threads used)."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    same = True
    step, units, desc = oracle_step_factory(c, B)
    t0 = time.time()
    step()
    probe = time.time() - t0
    if probe > budget_s and B > 1:                                  # bounded sample: fall back to one sample
        same = False
        step, units, desc = oracle_step_factory(c, 1)
        t0 = time.time()
        step()
        probe = time.time() - t0
    used, spent = cores, probe
    if cores > 32 and spent + probe <= budget_s:                  # probe a moderate thread count as well
        torch.set_num_threads(32)
        t0 = time.time()
        step()
        p32 = time.time() - t0
        spent += p32
        if p32 < probe:
            used, probe = 32, p32
        else:
            torch.set_num_threads(cores)
    left = budget_s - spent
    timed = int(min(steps, left // max(probe, 1e-9)))
    if timed < 1:
        return units / probe, probe, used, desc + ", the probe step is the timed one", same
    for _ in range(int(min(max(0, warmup - 1), max(0, left // probe - timed)))):
        step()
    t0 = time.time()
    for _ in range(timed):
        step()
    dt = (time.time() - t0) / timed
    return units / dt, dt, used, desc + ", %d timed step%s" % (timed, "" if timed == 1 else "s"), same


def time_oracle_cuda(c, B, steps=3, warmup=2):
    """The reference formulation as plain PyTorch ops on the GPU (fp32; matmul TF32 off as the reference leaves it, and
    a second figure with allow_tf32) — SURVEY 8d(i).  CUDA events, device-resident inputs."""
    out = {}
    desc = ""
    prev = torch.backends.cuda.matmul.allow_tf32
    try:
        for tf32 in (False, True):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            step, units, desc = oracle_step_factory(c, B, device="cuda")
            for _ in range(warmup):
                step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out["fp32_matmul_tf32" if tf32 else "fp32"] = {"ms_per_step": ms, "value": units / ms * 1e3}
            del step
            torch.cuda.empty_cache()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    out["unit"] = unit_name(c)
    out["sample"] = desc
    out["note"] = "oracle/ (functional PyTorch restatement of the reference, un-collapsed head) on cuda, eager, CUDA events"
    return out


def local_batch(c, args, world):
    if args.scaling == "strong":                                  # train3d.py:495: batch_size //= world_size
        if c["B"] % world:
            raise SystemExit("--scaling strong: global batch %d is not divisible by %d GPUs" % (c["B"], world))
        return c["B"] // world
    return c["B"]


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    c = CONFIGS[args.config]
    B = local_batch(c, args, int(os.environ.get("WORLD_SIZE", "1")))
    v, dt, cores, desc, same = time_oracle_cpu(c, B, args.steps, args.warmup,
                                               float(os.environ.get("SEGTRAN_REF_BUDGET_S", "200")))
    line = {"metric": metric_name(c), "value": v, "unit": unit_name(c), "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": workload_name(c, B), "baseline_config": args.config, "reference_sample": desc,
                       "same_batch_as_b200_arm": same},
            "cpu_baseline": {"value": v, "unit": unit_name(c), "cores": cores, "kind": "port", "sample": desc},
            "e2e": {"value": v, "unit": unit_name(c), "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------
# B200 arm
# ----------------------------------------------------------------------------------------------------------
class KernelTimer:
    """CUDA-event timing of individual C-ABI calls on the launching stream (for the roofline of the dominant kernel)."""

    def __init__(self):
        self.records = []                       # (name, info, ev0, ev1)
        self.shapes = []
        self.gemm_bytes = []
        self.enabled = False

    @contextlib.contextmanager
    def __call__(self, name, cargs):
        if not self.enabled:
            yield
            return
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        info = None
        if name == "sx_gemm":
            g = cargs[0]._obj
            info = 2.0 * g.M * g.N * g.K * g.Z0 * g.Z1
            es = 2.0 if g.op_dtype == 1 else 4.0
            za = (g.Z0 if g.A.stride_z0 else 1) * (g.Z1 if g.A.stride_z1 else 1)      # broadcast operands are read once
            zb = (g.Z0 if g.B.stride_z0 else 1) * (g.Z1 if g.B.stride_z1 else 1)
            zc = (g.Z0 if g.c_stride_z0 or g.Z0 == 1 else 1) * (g.Z1 if g.c_stride_z1 or g.Z1 == 1 else 1)
            cs = 2.0 if g.c_dtype == 1 else 4.0
            self.gemm_bytes.append(es * (g.M * g.K * za + g.N * g.K * zb) + cs * g.M * g.N * zc * (2 if g.preact else 1))
            self.shapes.append("%dx%dx%d z%d %s%s sk%d%s" % (g.M, g.N, g.K, g.Z0 * g.Z1, "kM"[g.A.major], "kM"[g.B.major],
                                                            g.split_k, " bf16" if g.op_dtype == 1 else ""))
        elif name == "sx_attn_probs_fwd":
            a = cargs[0]._obj
            info = 2.0 * a.B * a.M * a.U1 * a.U2 * a.d * (2 if a.U2 > 256 else 1)      # executed (two passes when keys > 256)
        elif name.startswith("sx_head_contract"):
            B, Cf, V = (cargs[3], cargs[4], cargs[5]) if name.endswith("fwd") else (cargs[2], cargs[3], cargs[4])
            info = 4.0 * B * Cf * V
        e0.record()
        yield
        e1.record()
        self.records.append((name, info, e0, e1))

    def gemm_shapes(self):
        out, i = {}, 0
        for name, info, e0, e1 in self.records:
            if name == "sx_gemm":
                a = out.setdefault(self.shapes[i], [0.0, 0.0, 0])
                a[0] += e0.elapsed_time(e1)
                a[1] += info
                a[2] += 1
                i += 1
        return {k: {"ms": v[0] / v[2], "tflops": v[1] / v[0] / 1e9, "n": v[2]} for k, v in
                sorted(out.items(), key=lambda kv: -kv[1][0])}

    def gemm_roofline(self, peak_tflops, peak_gbs):
        """Per-launch roofline: bound_i = max(flops_i / tensor peak, algorithmic bytes_i / HBM peak).  Returns the sum of
        the bounds over the sum of the measured times, and the time split between tensor-bound and HBM-bound launches."""
        i, tb, tt, hb, ht = 0, 0.0, 0.0, 0.0, 0.0
        for name, info, e0, e1 in self.records:
            if name != "sx_gemm":
                continue
            ms = e0.elapsed_time(e1)
            t_f = info / (peak_tflops * 1e12) * 1e3
            t_b = self.gemm_bytes[i] / (peak_gbs * 1e9) * 1e3
            if t_f >= t_b:
                tb, tt = tb + t_f, tt + ms
            else:
                hb, ht = hb + t_b, ht + ms
            i += 1
        return {"frac_of_bound": (tb + hb) / max(tt + ht, 1e-9),
                "tensor_bound_launches": {"ms": tt, "frac": tb / max(tt, 1e-9)},
                "hbm_bound_launches": {"ms": ht, "frac": hb / max(ht, 1e-9)}}

    def summarize(self):
        agg = {}
        for name, info, e0, e1 in self.records:
            ms = e0.elapsed_time(e1)
            a = agg.setdefault(name, [0.0, 0.0, 0])
            a[0] += ms
            a[1] += info or 0.0
            a[2] += 1
        return agg


DUMP_MAX_ELEMS = 1 << 21        # 8 MB of float32 per array: the six arrays of a dump stay under 64 MB
DUMP_SEED = 20240917


def dump_outputs(out_dir, arrays):
    """Writes every array as out_dir/<name>.npy in float32.  An array of more than DUMP_MAX_ELEMS elements is written as a
    flat sample of DUMP_MAX_ELEMS elements at sorted positions drawn with a fixed seed from its size, so two runs of the
    same config sample the same positions.  The inputs and weights of a run are fixed by its arguments, but the kernels
    reduce with floating-point atomics and every step trains on the last one's update, so two runs agree to rounding
    amplified over the steps, not bit for bit: compare dumps with a tolerance."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        v = t.detach()
        if v.numel() > DUMP_MAX_ELEMS:
            g = torch.Generator().manual_seed(DUMP_SEED)
            idx = torch.randint(v.numel(), (DUMP_MAX_ELEMS,), generator=g).sort().values
            v = v.reshape(-1)[idx.to(v.device)]
        np.save(os.path.join(out_dir, name + ".npy"), v.float().cpu().numpy())


def bucket_checksum(params):
    """Integer checksum of the parameter bits (identical on every rank iff the parameters are)."""
    acc = torch.zeros(2, dtype=torch.int64, device=params[0].device)
    for p in params:
        v = p.detach().contiguous().view(torch.int32).to(torch.int64)
        acc[0] += v.sum()
        acc[1] += (v * v & 0xFFFFF).sum()
    return acc


def run_b200(args):
    import torch.distributed as dist
    from segtran_b200 import _lib as L
    from segtran_b200 import ops
    from segtran_b200.parallel import GradBucket
    from segtran_b200.train import FlatBertAdam, seg_loss

    c = CONFIGS[args.config]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    precision = args.precision or c["precision"]
    ops.set_precision(precision)
    if os.environ.get("SEGTRAN_GEMM_MAX_CTAS"):            # bring-up knob: cap the persistent GEMM grids (SMs left to NCCL)
        L.call("sx_gemm_debug_set", b"max_ctas", int(os.environ["SEGTRAN_GEMM_MAX_CTAS"]))
    if args.no_fused_attn:
        ops.set_attn_fusion(False)
    B = local_batch(c, args, world)
    net = build_net(c, "cuda").to(dev).train()   # the same initial weights on every rank (data parallelism) ...
    torch.manual_seed(1337 + rank)               # ... different synthetic data and dropout masks per rank
    hp = hot_params(net, c)
    use_graph = not args.no_graph
    # N>1: the gradient all-reduce is issued from inside the step (and captured with it) at layer milestones, so most of
    # the bucket travels over NVLink while the rest of backward is still running
    bucket = GradBucket(hp, direct_accumulate=True, milestones=world > 1 and not args.no_overlap)
    feat, curr, Yb = synthetic_batch(c, B, dev, 4242 + rank)
    feat.requires_grad_()
    curr.requires_grad_()
    Y = Yb.float()
    pw, cw = loss_weights(c, dev)
    sp = (c["S"],) * (3 if c["kind"] == "3d" else 2)
    # the reference's optimiser on the hot-path parameters: BertAdam + --gradclip (train3d.py:334-355, :760-762); it
    # re-points the parameters into one flat buffer, so it is built before the step is captured
    opt = None if args.no_optimizer else FlatBertAdam(
        [{"params": hp, "lr": TRAIN["lr"], "weight_decay": TRAIN["decay"]}], warmup=TRAIN["warmup"],
        t_total=TRAIN["t_total"], grad_clip=TRAIN["grad_clip"], bucket=bucket)

    last = {}

    def compute():
        bucket.zero()
        feat.grad = None
        curr.grad = None
        logits = net.hot_path(feat, curr, None, sp)
        if args.dump_outputs:
            last["logits"] = logits             # in a captured step: the graph's buffer, rewritten by every replay
        loss, _, _ = seg_loss(logits, Y, pw, cw, TRAIN["dice_w"])         # train3d.py:731-756
        loss.backward()
        if world > 1 and not args.no_overlap:
            bucket.allreduce_async()            # what no milestone covered; joins the side stream (graph-capturable)
            bucket.wait()
        return loss

    if use_graph:
        from segtran_b200.graph import CapturedStep
        compute_fn = CapturedStep(compute, warmup=3)       # one cudaGraphLaunch per step instead of ~115 launches
    else:
        compute_fn = compute

    def step():
        loss = compute_fn()
        if world > 1 and args.no_overlap:
            bucket.allreduce_async()
            bucket.wait()
        if opt is not None:
            opt.step()                          # after the gradient exchange; 3 launches + 1 memset, all on the device
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    # ---- timed region: exactly K steps, device events, barrier + synchronize on both sides ----
    l0 = L.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    h0 = time.perf_counter()
    for _ in range(args.steps):
        loss = step()
    host_ms = (time.perf_counter() - h0) * 1e3 / args.steps        # host time to ENQUEUE a step (no sync inside)
    e1.record()
    barrier()
    launches = L.launch_count - l0
    if use_graph:
        launches = compute_fn.kernel_launches * args.steps      # kernels inside the replayed graph
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t) / args.steps
    value = world * B * units_per_sample(c) / (ms_step * 1e-3)
    # data-parallel sanity: every rank must hold bit-identical parameters after the same number of steps
    checksum_agree = None
    if world > 1 and opt is not None:
        cs = bucket_checksum(hp)
        lo, hi = cs.clone(), cs.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        checksum_agree = bool(torch.equal(lo, hi))
    if args.dump_outputs and rank == 0:
        # what the last timed step hands its caller: loss, logits, gradients of both feature tensors and of every
        # hot-path parameter, and the parameters after the update
        dump_outputs(args.dump_outputs, {
            "loss": loss, "logits": last["logits"], "grad_feat": feat.grad, "grad_curr": curr.grad,
            "param_grads": torch.cat([(torch.zeros_like(p) if p.grad is None else p.grad).reshape(-1) for p in hp]),
            "params": torch.cat([p.detach().reshape(-1) for p in hp])})

    # ---- the same K steps again with a CUDA-event pair around every C-ABI call (per-kernel durations for the
    #      roofline; the extra event records cost host time, so this pass is not the headline number) ----
    timer = KernelTimer()
    L.set_hook(timer)
    timer.enabled = True
    i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    i0.record()
    for _ in range(args.steps):
        compute()                                      # eager: the hook sees every C-ABI call
    i1.record()
    barrier()
    timer.enabled = False
    L.set_hook(None)
    ms_instr = i0.elapsed_time(i1) / args.steps

    # ---- end-to-end: host (pinned) feature buffers -> H2D every step (double-buffered) -> step -> D2H loss ----
    hfeat = [torch.randn(feat.shape).pin_memory() for _ in range(2)]
    hcurr = [torch.randn(curr.shape).pin_memory() for _ in range(2)]
    dfeat = [torch.empty_like(feat) for _ in range(2)]
    dcurr = [torch.empty_like(curr) for _ in range(2)]
    hmask = [(torch.rand(Y.shape) > 0.7).to(torch.uint8).pin_memory() for _ in range(2)]   # n-hot labels, 1 B/voxel
    dmask = [torch.empty(Y.shape, dtype=torch.uint8, device=dev) for _ in range(2)]
    hloss = torch.zeros(1).pin_memory()
    copy_stream = torch.cuda.Stream(device=dev)
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]

    def upload(i):
        s = i & 1
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[s])
            dfeat[s].copy_(hfeat[s], non_blocking=True)
            dcurr[s].copy_(hcurr[s], non_blocking=True)
            dmask[s].copy_(hmask[s], non_blocking=True)
            ready[s].record(copy_stream)

    def e2e_step(i):
        s = i & 1
        torch.cuda.current_stream().wait_event(ready[s])
        f = dfeat[s].detach().requires_grad_()
        cc = dcurr[s].detach().requires_grad_()
        bucket.zero()
        logits = net.hot_path(f, cc, None, sp)
        loss, _, _ = seg_loss(logits, dmask[s].float(), pw, cw, TRAIN["dice_w"])
        loss.backward()
        bucket.allreduce_async()
        bucket.wait()
        if opt is not None:
            opt.step()
        consumed[s].record()
        hloss.copy_(loss.detach(), non_blocking=True)

    e2e_steps = max(2, min(args.steps, 10))
    for s in range(2):
        consumed[s].record()
    upload(0)
    e2e_step(0)                                                    # warm
    barrier()
    upload(0)
    t0e, t1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0e.record()
    for i in range(e2e_steps):
        if i + 1 < e2e_steps:
            upload(i + 1)                                          # prefetch next step's inputs during this step
        e2e_step(i)
    t1e.record()
    barrier()
    sampler.stop_flag = True
    te = torch.tensor([t0e.elapsed_time(t1e)], device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_ms = float(te) / e2e_steps
    h2d = (hfeat[0].numel() + hcurr[0].numel()) * 4 + hmask[0].numel()

    if rank == 0:
        agg = timer.summarize()
        total_ms = sum(a[0] for a in agg.values())
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        top = max(agg.items(), key=lambda kv: kv[1][0])
        kname, (kms, kwork, kcount) = top
        bf16 = precision == "bf16"
        if kname == "sx_gemm":
            # TF32 operands: the tensor-core peak is half the measured dense bf16 figure
            src = "measured" if "bf16_tflops_sustained" in peaks else "fallback"
            peak = peaks.get("bf16_tflops_sustained", 1400.0) / (1.0 if bf16 else 2.0)
            ach = kwork / (kms * 1e-3) / 1e12
            # the executed count is lower than the reference formulation's (SURVEY §8d: ref_gflop per sample forward, x3
            # for fwd+bwd) because of the re-associated in-squeeze and mid Linear (DESIGN §4.5)
            ref_flops = c["ref_gflop"] * 1e9 * 3 * B * args.steps
            roof = {"bound": "tensor", "kernel": "sx_gemm_kernel (tcgen05 kind::%s)" % ("f16/bf16" if bf16 else "tf32"),
                    "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": None,
                    "achieved_reference_formulation": ref_flops / (kms * 1e-3) / 1e12,
                    "executed_tflop_per_step": kwork / args.steps / 1e12,
                    "peak_source": "%s bf16 sustained%s" % (src, "" if bf16 else " / 2 (tf32 rate)"), "launches": kcount,
                    "share_of_step": kms / total_ms}
            hbm_peak = peaks.get("hbm_gbs", 6570.0)
            pl = timer.gemm_roofline(peak, hbm_peak)
            for v in pl.values():
                if isinstance(v, dict):
                    v["ms"] /= args.steps
            roof["per_launch"] = pl
            roof["algorithmic_bytes_per_launch"] = sum(timer.gemm_bytes) / max(len(timer.gemm_bytes), 1)
            try:        # DRAM bytes of the GEMM launches of a step from an ncu capture of this command (profiles/, per launch)
                tr = json.load(open(os.path.join(ROOT, "profiles", "gemm_dram_traffic.json")))
                if args.config == 4 and not bf16:
                    roof["traffic"] = tr["dram_bytes_per_launch"]
                    roof["traffic_source"] = tr.get("source", "profiles/gemm_dram_traffic.json")
            except Exception:
                pass
        else:
            src = "measured" if "hbm_gbs" in peaks else "fallback"
            peak = peaks.get("hbm_gbs", 6650.0)
            ach = kwork / (kms * 1e-3) / 1e9
            roof = {"bound": "hbm", "kernel": kname, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": None, "peak_source": src, "launches": kcount, "share_of_step": kms / total_ms}
        breakdown = {k: {"ms_per_step": v[0] / args.steps, "calls_per_step": v[2] / args.steps}
                     for k, v in sorted(agg.items(), key=lambda kv: -kv[1][0])}
        N = 1
        for s in c["grid"]:
            N *= s
        line = {"metric": metric_name(c), "value": value, "unit": unit_name(c), "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": args.scaling,
                "vs_baseline": None, "dtype": precision, "data": "synthetic",
                "config": {"workload": workload_name(c, B), "baseline_config": args.config,
                           "global_batch": world * B, "tokens_per_sample": N, "parallelism": "dp%d" % world,
                           "l2": "inputs (%.2f GB/step) exceed the 126 MB L2; no explicit flush" % (
                               (feat.numel() + curr.numel() + Y.numel()) * 4 / 1e9),
                           "grad_bucket_bytes": bucket.bytes(),
                           "launch": "cuda-graph replay of fwd+loss+bwd" if use_graph else "eager",
                           "allreduce": None if world == 1 else (
                               "one NCCL all-reduce after the step" if args.no_overlap else
                               "NCCL all-reduce of bucket ranges issued at layer milestones inside the (captured) step"),
                           "attention": "unfused (GEMM + softmax kernels)" if args.no_fused_attn else
                                        "fused tcgen05 scores+softmax kernel (sx_attn)",
                           "loss": "BCEWithLogits(pos_weight) + per-class Dice on the full-size logits (train3d.py:731-756)",
                           "optimizer": None if opt is None else "FlatBertAdam on the hot-path parameters incl. --gradclip "
                                                                 "0.1 (optimization.py:90-164, train3d.py:760-762), in the step"},
                "clocks": sampler.summary(),
                "e2e": {"value": world * B * units_per_sample(c) / (e2e_ms * 1e-3), "unit": unit_name(c),
                        "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "steps": e2e_steps,
                        "note": "pinned host feature tensors + uint8 n-hot labels, double-buffered H2D on a copy stream, loss read back"},
                "gpu_launches": launches, "roofline": roof, "kernel_breakdown": breakdown,
                "ms_per_step_instrumented": ms_instr, "host_enqueue_ms_per_step": host_ms, "kernel_ms_per_step": total_ms / args.steps,
                "loss": float(hloss)}
        if checksum_agree is not None:
            line["dp_param_checksums_agree"] = checksum_agree
        if world == 1 and precision == "tf32" and not args.no_fp32_equivalent:
            # the same step with every contraction as an error-compensated 3-pass TF32 product (fp32-grade results,
            # 1e-7 .. 1e-5 against the fp32 oracle): what the default mode's TF32 trade buys.  Eager launches (no graph).
            ops.set_precision("tf32x3")
            try:
                fe_fn, fe_launch = compute, "eager"
                if use_graph:
                    try:                                   # replayed as a CUDA graph like the headline step ...
                        from segtran_b200.graph import CapturedStep
                        fe_fn, fe_launch = CapturedStep(compute, warmup=2), "cuda-graph replay of fwd+loss+bwd"
                    except Exception as ex:                # ... or launched eagerly (host-bound: an upper bound)
                        torch.cuda.synchronize()
                        fe_fn, fe_launch = compute, "eager (graph capture failed: %s)" % repr(ex)[:120]
                for _ in range(2):
                    fe_fn()
                    if opt is not None:
                        opt.step()
                f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                nf = max(2, min(args.steps, 5))
                torch.cuda.synchronize()
                f0.record()
                for _ in range(nf):
                    fe_fn()
                    if opt is not None:
                        opt.step()
                f1.record()
                torch.cuda.synchronize()
                fms = f0.elapsed_time(f1) / nf
                line["fp32_equivalent"] = {"precision": "tf32x3", "ms_per_step": fms, "steps": nf, "launch": fe_launch,
                                           "value": B * units_per_sample(c) / (fms * 1e-3), "unit": unit_name(c)}
                fe_fn = None
            except Exception as ex:                        # never lose the headline line over the extra figure
                line["fp32_equivalent"] = {"unavailable": repr(ex)[:200]}
            finally:
                ops.set_precision(precision)
        if world == 1 and not args.no_eager_baseline:
            compute_fn = None
            torch.cuda.empty_cache()
            try:
                eb = time_oracle_cuda(c, B)
                eb["speedup_vs_fp32"] = eb["fp32"]["ms_per_step"] / ms_step
                eb["speedup_vs_fp32_matmul_tf32"] = eb["fp32_matmul_tf32"]["ms_per_step"] / ms_step
                line["cuda_eager_baseline"] = eb
            except Exception as ex:               # e.g. out of memory for the un-collapsed head
                line["cuda_eager_baseline"] = {"unavailable": repr(ex)[:200]}
        if world == 1 and not args.no_cpu_baseline:
            v, dt, cores, desc, same = time_oracle_cpu(c, B, 1, 1, float(os.environ.get("SEGTRAN_CPU_BUDGET_S", "150")))
            line["cpu_baseline"] = {"value": v, "unit": unit_name(c), "cores": cores, "kind": "port", "sample": desc,
                                    "same_batch_as_b200_arm": same}
        print(json.dumps(line))
        if os.environ.get("SEGTRAN_BENCH_VERBOSE"):
            for k, v in timer.gemm_shapes().items():
                print("GEMM %-40s %8.3f ms %8.1f TF/s x%d" % (k, v["ms"], v["tflops"], v["n"]), file=sys.stderr)
    if world > 1:
        # a CUDA graph that captured NCCL work keeps the communicator busy: destroy_process_group() then never returns
        # (observed: both ranks stuck there after the result line was printed).  Drop the graph, drain the device, make sure
        # every rank got here, and leave without the collective teardown.
        compute_fn = None
        import gc
        gc.collect()
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=4, choices=sorted(CONFIGS), help="BASELINE.json config number (1-5)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: per-GPU batch fixed; strong: the config's batch is the GLOBAL batch (train3d.py:495)")
    ap.add_argument("--precision", default=None, choices=["tf32", "tf32x3", "bf16"])
    ap.add_argument("--no-optimizer", action="store_true", help="leave the BertAdam update out of the step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--no-fp32-equivalent", action="store_true",
                    help="skip the extra tf32x3 (fp32-grade) timing of the same step")
    ap.add_argument("--no-fused-attn", action="store_true", help="squeeze-out attention as separate GEMM + softmax kernels")
    ap.add_argument("--no-overlap", action="store_true", help="N>1: one all-reduce of the whole bucket after the step")
    ap.add_argument("--no-graph", action="store_true", help="enqueue every kernel from Python instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (loss, logits, feature and parameter "
                         "gradients, updated parameters) as DIR/<name>.npy in float32; arrays of more than %d elements "
                         "as a fixed seeded sample" % DUMP_MAX_ELEMS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the b200 step")
    wd = float(os.environ.get("SEGTRAN_BENCH_WATCHDOG_S", "0"))
    if wd == 0 and args.impl != "reference" and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        wd = 900.0                                 # a multi-rank run takes ~1 min: a stalled collective must not hang the launcher
    if wd > 0:                                     # dump every thread's Python stack and exit if the run stalls
        import faulthandler
        faulthandler.dump_traceback_later(wd, exit=True)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
