"""The layer census (tests/layer_census.py) and a CPU rehearsal of the layer-adjoint tests (tests/test_layer_adjoints_gpu.py).

Coverage: every weight-bearing Linear / Conv module of the VC2 UNet and of its VAE decoder maps to one census entry, and the LoRA
subset reproduces the step's counts (575 LoRA layers, 51 tensor-core geometries) — when the model changes, this fails until the
census is updated.  Self-check: the GPU test bodies run here through tests/mock_ops.py (bf16 activations) at small geometries, one
per layer kind plus a padded layer and a down / up pair, which proves the references, rounding points, tap bookkeeping and
guard checks before any GPU time is spent.
"""
import pytest
import torch
import torch.nn as nn

import mock_ops
from layer_census import Geo, census, decoder_census, decoder_layer_map, unet_layer_map, _gemm_modules, _unet


def test_unet_census_covers_every_gemm_layer():
    unet = _unet()
    lmap = unet_layer_map(unet=unet)
    names = [n for n, _ in _gemm_modules(unet)]
    assert sorted(lmap) == sorted(names)
    entries = set(census())
    assert all(g in entries for g in lmap.values())
    from t2v_turbo_b200.lora import lora_target_layers
    lora_names = {n for n, _ in lora_target_layers(unet)}
    lora = {n: g for n, g in lmap.items() if n in lora_names}
    tc = {(g.kind, g.points, g.cin, g.cout) for g in lora.values() if g.role == "lora"}
    print(f"\n[census] {len(lmap)} GEMM layers, {len(lora)} LoRA layers, {len(tc)} LoRA tensor-core geometries, "
          f"{len(entries)} distinct census entries")
    assert len(lora) == 575 and len(tc) == 51
    roles = sorted(g.role for n, g in lmap.items() if g.role != "lora")
    assert roles == ["down"] * 3 + ["frozen"] * 2 + ["pad"] * 2 + ["up"] * 3, roles
    assert {n for n, g in lmap.items() if g.role == "frozen"} == {"init_attn.0.proj_in", "init_attn.0.proj_out"}
    # the resolved layers run where train_unet runs them: conv_in / out at the latent grid, padded to 64 channels;
    # the Downsample convs at the grid BEFORE subsampling, the Upsample convs at the grid AFTER upsampling
    assert lmap["input_blocks.0.0"] == Geo("conv2d", (16, 40, 64), 4, 320, True, 64, 0, "pad")
    assert lmap["out.2"] == Geo("conv2d", (16, 40, 64), 320, 4, True, 0, 64, "pad")
    assert [lmap[f"input_blocks.{i}.0.op"].points for i in (3, 6, 9)] == [(16, 40, 64), (16, 20, 32), (16, 10, 16)]
    assert [lmap[n].points for n in ("output_blocks.2.1.conv", "output_blocks.5.3.conv", "output_blocks.8.3.conv")] == \
        [(16, 10, 16), (16, 20, 32), (16, 40, 64)]
    # the edge geometries: M = 1 embedding rows (wgrad's < 16-point padding), the 16 x 77 context rows (a ragged last tile),
    # Cin = 960 / 1920 / 2560 (half-empty 128-channel wgrad blocks), the 5 x 8 level (3x3 taps on a grid smaller than a tile)
    pts = {g.points for g in entries}
    assert {(1,), (1232,), (16, 5, 8)} <= pts
    assert {960, 1920, 2560} <= {g.cin for g in entries if g.kind == "conv2d"}


def test_decoder_census_covers_every_gemm_layer():
    lmap, dec = decoder_layer_map()
    names = [n for n, m in dec.named_modules() if isinstance(m, (nn.Linear, nn.Conv2d, nn.Conv3d))]
    assert sorted(lmap) == sorted(names)
    assert set(lmap.values()) == set(decoder_census())
    assert lmap["conv_in"] == Geo("conv2d", (1, 40, 64), 4, 512, True, 64, 0, "pad")
    assert lmap["conv_out"] == Geo("conv2d", (1, 320, 512), 128, 3, True, 0, 64, "pad")
    print(f"\n[census] decoder: {len(lmap)} GEMM layers, {len(set(lmap.values()))} distinct geometries")


# ----------------------------------------------------------------------------- CPU rehearsal of the GPU bodies
_SMALL_LORA = [Geo("linear", (40,), 64, 128, True, 0, 0, "lora"), Geo("linear", (1,), 128, 64, True, 0, 0, "lora"),
               Geo("conv2d", (2, 5, 8), 128, 64, True, 0, 0, "lora"), Geo("conv3d", (2, 4, 10), 64, 64, False, 0, 0, "lora")]
_SMALL_FULL = _SMALL_LORA + [Geo("conv2d", (2, 8, 8), 4, 64, True, 64, 0, "pad"), Geo("conv2d", (2, 8, 8), 64, 4, True, 0, 64, "pad")]
_SMALL_RESAMPLE = [Geo("conv2d", (2, 8, 12), 64, 64, True, 0, 0, "down"), Geo("conv2d", (2, 8, 12), 64, 64, True, 0, 0, "up")]


@pytest.fixture
def mocked(monkeypatch):
    mock_ops.install(monkeypatch, act=torch.bfloat16)
    import test_layer_adjoints_gpu as T
    return T


@pytest.mark.parametrize("geo", _SMALL_LORA, ids=lambda g: f"{g.kind}-{'x'.join(map(str, g.points))}")
def test_selfcheck_lora(mocked, geo):
    mocked.check_lora(geo, torch.device("cpu"))


@pytest.mark.parametrize("geo", _SMALL_FULL, ids=lambda g: f"{g.kind}-{'x'.join(map(str, g.points))}-{g.cin}to{g.cout}")
def test_selfcheck_full(mocked, geo):
    mocked.check_full(geo, torch.device("cpu"))


@pytest.mark.parametrize("geo", _SMALL_RESAMPLE, ids=lambda g: g.role)
def test_selfcheck_resample(mocked, geo):
    mocked.check_resample(geo, torch.device("cpu"))


@pytest.mark.parametrize("kind,grid", [("conv2d", (4, 5, 8)), ("conv2d", (4, 10, 16)), ("conv3d", (2, 16, 6))])
def test_selfcheck_impulse(mocked, kind, grid):
    mocked.check_impulse(kind, grid, 64, torch.device("cpu"))


@pytest.mark.parametrize("geo", [Geo("conv2d", (1, 6, 8), 4, 64, True, 64, 0, "pad"), Geo("conv2d", (1, 6, 8), 64, 3, True, 0, 64, "pad"),
                                 Geo("linear", (48,), 128, 64, True, 0, 0, "conv1x1")], ids=lambda g: f"{g.kind}-{g.cin}to{g.cout}")
def test_selfcheck_decoder(mocked, geo):
    mocked.check_decoder(geo, torch.device("cpu"))


def test_selfcheck_guard_band_catches_stray_write(mocked):
    """The guard bands detect a write one element past a gradient view."""
    A = mocked.GuardedArena({"w": (3, 5), "b": (3,)}, torch.device("cpu"))
    A.check_guards("untouched")
    o, s = A.layout["w"]
    A.grads[o + 15] += 1.0
    with pytest.raises(AssertionError, match="guard-band"):
        A.check_guards("stray write")
