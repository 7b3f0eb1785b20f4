"""TEST INFRASTRUCTURE (like mock_ops.py): the distinct GEMM-layer geometries the training steps issue on the VC2 models.

`census()` lists, for a [batch, 4, frames, h, w] latent, every distinct (kind, point grid, cin, cout, has_bias, pad_in, pad_out, role)
of the VC2 `UNetModel` (built on the meta device: no weights, well under a second):

    kind      linear | conv2d | conv3d (the tensor-core layer kinds of lora_train._base_op; 1x1 convolutions are per-point Linears)
    points    the channels-last point grid the layer runs on: (M,) | (n, h, w) | (b, t, hw)
    pad_in / pad_out   the zero-padded channel counts of the 4-channel conv_in / out (0 = none), as train_unet / full_train run them
    role      lora    a LoRA target on the tensor-core path (`unet_lora_workload` kind != skip)
              down    a Downsample `op`: the stride-1 conv at the PRE-down grid, followed by resample2x "sub"
              up      an Upsample `conv`: at the 2x grid, after upsample_nearest2x
              pad     conv_in / out, zero-padded to 64 channels
              frozen  a GEMM layer that is not a LoRA target (init_attn's Conv1d proj_in / proj_out): frozen in the v1 LoRA step,
                      trained by the v2 full fine-tune (full_train.FullUNet)

`decoder_census()` lists the same for the conv / 1x1 layers of `vae_train.DecoderGrad` decoding one frame (VC2 VAE config).
"""
from __future__ import annotations

from collections import namedtuple

import torch
import torch.nn as nn

Geo = namedtuple("Geo", "kind points cin cout has_bias pad_in pad_out role")


def geo_id(g: Geo) -> str:
    pts = "x".join(str(p) for p in g.points)
    pad = (f"-pin{g.pad_in}" if g.pad_in else "") + (f"-pout{g.pad_out}" if g.pad_out else "")
    return f"{g.role}-{g.kind}-{pts}-{g.cin}to{g.cout}{'-b' if g.has_bias else ''}{pad}"


def _unet(cfg=None):
    from t2v_turbo_b200.configs import VC2_UNET
    from t2v_turbo_b200.unet import UNetModel
    with torch.device("meta"):
        return UNetModel(**(cfg or VC2_UNET))


def _gemm_modules(model):
    return [(n, m) for n, m in model.named_modules() if isinstance(m, (nn.Linear, nn.Conv1d, nn.Conv2d, nn.Conv3d))]


def _resample_grids(unet, h, w):
    """{Downsample / Upsample module: the (h, w) grid of its INPUT} by the traversal order of train_unet._build."""
    from t2v_turbo_b200 import unet as U
    grids = {}

    def walk(seq, hh, ww):
        for layer in seq:
            if isinstance(layer, U.Downsample):
                grids[layer] = (hh, ww)
                hh, ww = hh // 2, ww // 2
            elif isinstance(layer, U.Upsample):
                grids[layer] = (hh, ww)
                hh, ww = hh * 2, ww * 2
        return hh, ww
    hh, ww = h, w
    for blk in list(unet.input_blocks) + [unet.middle_block] + list(unet.output_blocks):
        hh, ww = walk(blk, hh, ww)
    return grids


def unet_layer_map(batch=1, frames=16, h=40, w=64, unet=None):
    """{qualified module name: Geo} for every weight-bearing Linear / Conv module of the VC2 UNetModel."""
    from t2v_turbo_b200 import unet as U
    from t2v_turbo_b200.lora_train import unet_lora_workload
    unet = unet if unet is not None else _unet()
    n = batch * frames
    mods = dict(_gemm_modules(unet))
    owner = {}
    for g, (gh, gw) in _resample_grids(unet, h, w).items():
        sub = g.op if isinstance(g, U.Downsample) else g.conv
        owner[sub] = (g, gh, gw)
    out = {}
    for name, kind, pts, cin, cout in unet_lora_workload(unet, batch, frames, h, w):
        m = mods[name]
        bias = m.bias is not None
        if kind != "skip":
            out[name] = Geo(kind, tuple(pts), cin, cout, bias, 0, 0, "lora")
        elif m in owner:
            g, gh, gw = owner[m]
            if isinstance(g, U.Downsample):
                out[name] = Geo("conv2d", (n, gh, gw), cin, cout, bias, 0, 0, "down")
            else:
                out[name] = Geo("conv2d", (n, 2 * gh, 2 * gw), cin, cout, bias, 0, 0, "up")
        elif isinstance(m, nn.Conv2d) and m.kernel_size == (3, 3) and (cin < 64 or cout < 64):   # conv_in / out.2 at the full grid
            out[name] = Geo("conv2d", (n, h, w), cin, cout, bias, 64 if cin < 64 else 0, 64 if cout < 64 else 0, "pad")
        else:
            raise AssertionError(f"{name}: a skipped LoRA layer the census does not resolve")
    for name, m in mods.items():       # GEMM layers that are not LoRA targets: init_attn's Conv1d proj_in / proj_out
        if name in out:
            continue
        if isinstance(m, nn.Conv1d) and m.kernel_size == (1,) and name.startswith("init_attn."):
            out[name] = Geo("linear", (n * h * w,), m.in_channels, m.out_channels, m.bias is not None, 0, 0, "frozen")
        else:
            raise AssertionError(f"{name}: a GEMM layer the census does not know")
    return out


def census(batch=1, frames=16, h=40, w=64):
    """Distinct Geo entries of the VC2 UNet (first-appearance order)."""
    return list(dict.fromkeys(unet_layer_map(batch, frames, h, w).values()))


def decoder_layer_map(h=40, w=64, ddconfig=None):
    """{qualified module name under `decoder`: Geo} for DecoderGrad decoding ONE frame from an h x w latent."""
    from t2v_turbo_b200.configs import VC2_VAE_DDCONFIG
    from t2v_turbo_b200.vae import Decoder
    with torch.device("meta"):
        d = Decoder(**(ddconfig or VC2_VAE_DDCONFIG))
    out = {}

    def conv(name, m, gh, gw, role="conv", pad_in=0, pad_out=0):
        out[name] = Geo("conv2d", (1, gh, gw), m.in_channels, m.out_channels, True, pad_in, pad_out, role)

    def lin(name, m, gh, gw):
        out[name] = Geo("linear", (gh * gw,), m.in_channels, m.out_channels, True, 0, 0, "conv1x1")

    def res(prefix, rb, gh, gw):
        conv(prefix + ".conv1", rb.conv1, gh, gw)
        conv(prefix + ".conv2", rb.conv2, gh, gw)
        if rb.in_channels != rb.out_channels:
            lin(prefix + ".nin_shortcut", rb.nin_shortcut, gh, gw)

    conv("conv_in", d.conv_in, h, w, "pad", pad_in=64)          # DecoderGrad.conv_in: the adjoint runs 64-channel padded
    res("mid.block_1", d.mid.block_1, h, w)
    for p in ("q", "k", "v", "proj_out"):
        lin(f"mid.attn_1.{p}", getattr(d.mid.attn_1, p), h, w)
    res("mid.block_2", d.mid.block_2, h, w)
    gh, gw = h, w
    for i in reversed(range(d.num_resolutions)):
        for j, rb in enumerate(d.up[i].block):
            res(f"up.{i}.block.{j}", rb, gh, gw)
        if i != 0:
            gh, gw = 2 * gh, 2 * gw
            conv(f"up.{i}.upsample.conv", d.up[i].upsample.conv, gh, gw, "up")
    conv("conv_out", d.conv_out, gh, gw, "pad", pad_out=64)      # 3 output channels, padded
    return out, d


def decoder_census(h=40, w=64):
    return list(dict.fromkeys(decoder_layer_map(h, w)[0].values()))
