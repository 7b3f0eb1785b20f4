"""Layer adjoints of the training steps on B200, at every GEMM-layer geometry the VC2 steps issue (tests/layer_census.py).

Both training steps take their gradients from two kernels used in ways the forward suite does not reach: the input gradients
re-run the forward implicit GEMM (t2v_gemm) on transposed, tap-reversed weights (for LoRA layers over the K-concatenated
[W^T | D^T] with the dual-source A operand (dy | dt)), and every weight gradient is t2v_wgrad (conv taps = TMA coordinate
offsets, padding = TMA zero fill, fp32 red.add into the gradient arena).  Each test runs the real host code of one layer kind
(lora_train.lora_forward / lora_backward, full_train._FullLayer, vae_train._Conv / _Lin) and compares it with an fp64 reference
computed from the same bf16-rounded operands:

    a  LoRA layer, one case per LoRA geometry: y, dx (2 bf16 ulps of the element + 1 of the output scale, assert_close) and
       d lora_up / d lora_down accumulated into prefilled arena views (the fp32 accumulation bound below)
    b  full fine-tune layer, one case per census geometry: y, dx, dW, db against autograd of F.linear / conv2d / conv3d; gradient
       views prefilled (the kernels must accumulate) and surrounded by sentinel guard bands (no write may land outside them)
    c  Downsample / Upsample compositions (conv + resample2x "sub" / "stuff"; upsample_nearest2x + conv / "pool") against autograd
       of F.conv2d(stride 2) and F.interpolate(nearest) + F.conv2d at the three down and three up levels
    d  impulse tests, exact: dy one-hot in point and channel at the corners / edges of frames and the first / last frame of both
       videos, so that every output element is at most one bf16 product: dx is the tap-reversed weight entry, dW the shifted input
    e  the VAE decoder's frozen conv / 1x1 layers (DecoderGrad): y and dx

fp32 accumulation bound (dW, db): |err| <= 1e-5 * S + 1e-7 * max|ref| elementwise, where S is the per-element sum of the absolute
values of every summand (the prefilled value and each product), i.e. the fp64 reference evaluated on |operands|.

The check_* bodies take the device as an argument: tests/test_layer_census.py runs them on CPU through tests/mock_ops.py at small
geometries, which proves the references, rounding points and guard checks without a GPU.
"""
from __future__ import annotations

import contextlib
import math
import types

import pytest
import torch
import torch.nn.functional as F

from layer_census import Geo, census, decoder_census, geo_id
from test_kernels_gpu import assert_close

BF16 = torch.bfloat16
KSHAPE = {"linear": (), "conv2d": (3, 3), "conv3d": (3, 1, 1)}
R = 64                      # LoRA rank of the steps (every VC2 target has cin, cout >= 64)


# ----------------------------------------------------------------------------- helpers
def _bf(t):
    """fp32 tensor holding bf16 values: what the kernels see after their bf16 cast, exactly."""
    return t.to(BF16).float()


def _randn(g, *shape, scale=1.0):
    return torch.randn(*shape, generator=g, device=g.device) * scale


def _ref_op(kind, x, w, b=None):
    """The layer's forward in torch on channels-last x ([M, K] | [n, h, w, C] | [b, t, hw, C]), w in torch's weight layout."""
    if kind == "linear":
        return F.linear(x, w.reshape(w.shape[0], -1), b)
    if kind == "conv2d":
        return F.conv2d(x.permute(0, 3, 1, 2), w, b, padding=1).permute(0, 2, 3, 1)
    y = F.conv3d(x.permute(0, 3, 1, 2).unsqueeze(-1), w, b, padding=(1, 0, 0))        # [b, C, t, hw, 1]
    return y.squeeze(-1).permute(0, 2, 3, 1)


def _ref_grads(f, x, w, b, dy):
    """fp64 autograd of y = f(x, w, b) -> (y, dx, dw, db)."""
    x = x.double().requires_grad_(True)
    w = w.double().requires_grad_(True)
    leaves = [x, w]
    if b is not None:
        b = b.double().requires_grad_(True)
        leaves.append(b)
    with torch.enable_grad():
        y = f(x, w, b)
        grads = torch.autograd.grad(y, leaves, dy.double())
    return (y.detach(),) + tuple(grads) + ((None,) if b is None else ())


def assert_accum(got, ref, s, what):
    """The fp32-accumulation bound: |got - ref| <= 1e-5 * S + 1e-7 * max|ref| (S: the reference on |summands|)."""
    got, ref, s = got.double(), ref.double(), s.double()
    err = (got - ref).abs()
    tol = 1e-5 * s + 1e-7 * ref.abs().max()
    bad = err > tol
    print(f"[tol] {what}: worst err/tol {(err / tol).max().item():.3f}, max err {err.max().item():.3e}, "
          f"scale {ref.abs().max().item():.3e}")
    assert not bad.any(), (f"{what}: {int(bad.sum())}/{bad.numel()} outside the fp32 accumulation bound, max err "
                           f"{err.max().item():.4g}, first bad idx {bad.nonzero()[0].tolist()}")


class GuardedArena:
    """Stand-in for the gradient arenas (lora_train.LoraArena / full_train.FullArena): named fp32 views into one parameter buffer
    and one gradient buffer, every gradient view surrounded by GUARD sentinel values (a NaN bit pattern) that must stay
    bit-unchanged: a kernel writing outside the view it was given shows up in `check_guards`."""
    GUARD = 256
    SENTINEL = 0x7FA5A5A5

    def __init__(self, shapes: dict, device):
        self.layout, off = {}, self.GUARD
        for name, s in shapes.items():
            self.layout[name] = (off, tuple(s))
            off += (math.prod(s) + 3) // 4 * 4 + self.GUARD
        self.params = torch.zeros(off, device=device, dtype=torch.float32)
        self.grads = torch.full((off,), self.SENTINEL, device=device, dtype=torch.int32).view(torch.float32)
        self.guard = torch.ones(off, device=device, dtype=torch.bool)
        for o, s in self.layout.values():
            self.guard[o:o + math.prod(s)] = False

    def _view(self, buf, name):
        o, s = self.layout[name]
        return buf[o:o + math.prod(s)].view(s)

    def param(self, name):
        return self._view(self.params, name)

    def grad(self, name):
        return self._view(self.grads, name)

    def check_guards(self, what):
        g = self.grads.view(torch.int32)[self.guard]
        n_bad = int((g != self.SENTINEL).sum())
        assert n_bad == 0, f"{what}: {n_bad} guard-band values around the gradient views were overwritten"


@contextlib.contextmanager
def _recording(mod, *names):
    """Wrap mod.<name> so that every call's (first argument, output) is recorded."""
    calls = {n: [] for n in names}
    orig = {n: getattr(mod, n) for n in names}

    def wrap(n):
        def f(*a, **k):
            out = orig[n](*a, **k)
            calls[n].append((a[0], out))
            return out
        return f
    try:
        for n in names:
            setattr(mod, n, wrap(n))
        yield calls
    finally:
        for n in names:
            setattr(mod, n, orig[n])


def _output_of(calls, first_arg):
    """The output of the one recorded call whose first operand is (a view of) first_arg."""
    outs = [o for a, o in calls if torch.is_tensor(a) and a.data_ptr() == first_arg.data_ptr()]
    assert len(outs) == 1, f"{len(outs)} recorded calls read that operand"
    return outs[0]


# ----------------------------------------------------------------------------- a. LoRA layer
def check_lora(geo: Geo, dev, seed=0, scale=0.7, p=0.1):
    """lora_forward / lora_backward of one LoRA layer (explicit keep-mask, p = 0.1) against fp64 on the path's own bf16
    intermediates.  t is returned by lora_forward; u, the scaled branch, du and dt are the outputs of the ops calls the path made
    (recorded, not recomputed: a split-K GEMM accumulates with fp32 atomics, so a second call may round differently) and are
    checked against fp64 themselves, so every rounding point of the path is pinned."""
    from t2v_turbo_b200 import lora_train as lt
    from t2v_turbo_b200 import ops
    kind, pts, cin, cout = geo.kind, tuple(geo.points), geo.cin, geo.cout
    ks = KSHAPE[kind]
    taps = math.prod(ks)
    g = torch.Generator(device=dev).manual_seed(seed)
    w = _bf(_randn(g, cout, cin, *ks, scale=(cin * taps) ** -0.5))
    b = _randn(g, cout, scale=0.5) if geo.has_bias else None
    A = GuardedArena({"up": (cout, R), "down": (R, cin) + ks}, dev)
    A.param("up").copy_(_bf(_randn(g, cout, R, scale=0.5 * R ** -0.5)))
    A.param("down").copy_(_bf(_randn(g, R, cin, *ks, scale=(cin * taps) ** -0.5)))
    pre_up, pre_down = _randn(g, cout, R, scale=0.5), _randn(g, R, cin, *ks, scale=0.5)
    A.grad("up").copy_(pre_up)
    A.grad("down").copy_(pre_down)
    pk = lt._PackedLora(kind, w.reshape(cout, -1) if kind == "linear" else w, b, A.param("up"), A.param("down"), scale)
    m = math.prod(pts)
    mask = torch.empty((m, cout), device=dev, dtype=torch.float32).bernoulli_(1.0 - p, generator=g).to(torch.uint8)
    ms = 1.0 / (1.0 - p)
    x = _randn(g, *pts, cin).to(BF16)
    dy = _randn(g, *pts, cout).to(BF16)

    with _recording(ops, "linear", "scale_mask") as fwd:
        y, t, _, _ = lt.lora_forward(pk, x, mask, ms)
    with _recording(ops, "linear", "scale_mask") as bwd:
        dx = lt.lora_backward(pk, x, t, mask, ms, dy, A.grad("up"), A.grad("down"))
    u = _output_of(fwd["linear"], t)
    (_, branch), = fwd["scale_mask"]
    (_, du), = bwd["scale_mask"]
    dt = _output_of(bwd["linear"], du)

    tag = f"lora {geo_id(geo)}"
    U, D, mk = A.param("up").double(), A.param("down").double(), mask.double()
    x64, t64, u64, du64, dt64 = x.double(), t.double().reshape(m, R), u.double(), du.double(), dt.double()
    assert_close(t, _ref_op(kind, x64, D), what=f"{tag} t")
    assert_close(u, t64 @ U.t(), what=f"{tag} u")
    assert_close(branch, u64 * (scale * ms) * mk, what=f"{tag} branch")
    assert_close(du, dy.double().reshape(m, cout) * (scale * ms) * mk, what=f"{tag} du")
    assert_close(dt, du64 @ U, what=f"{tag} dt")
    y_base, dx_base, _, _ = _ref_grads(lambda a, ww, bb: _ref_op(kind, a, ww, bb), x64, w, b, dy)
    assert_close(y, y_base + branch.double().view(y_base.shape), what=f"{tag} y")
    dt_pts = dt64.view(*pts, R)
    _, dx_down, d_down, _ = _ref_grads(lambda a, ww, bb: _ref_op(kind, a, ww), x64, D, None, dt_pts)
    assert_close(dx, dx_base + dx_down, what=f"{tag} dx")
    assert_accum(A.grad("up"), pre_up.double() + du64.t() @ t64,
                 pre_up.double().abs() + du64.abs().t() @ t64.abs(), f"{tag} d_up")
    _, _, s_down, _ = _ref_grads(lambda a, ww, bb: _ref_op(kind, a, ww), x64.abs(), D, None, dt_pts.abs())
    assert_accum(A.grad("down"), pre_down.double() + d_down, pre_down.double().abs() + s_down, f"{tag} d_down")
    A.check_guards(tag)


# ----------------------------------------------------------------------------- b. full fine-tune layer
def _full_layer(geo: Geo, dev, g, prefill=True):
    """A full_train._FullLayer over a GuardedArena holding its weight (bf16 values), bias and prefilled gradients."""
    from t2v_turbo_b200 import full_train
    ks = KSHAPE[geo.kind]
    shapes = {"L.weight": (geo.cout, geo.cin) + ks}
    if geo.has_bias:
        shapes["L.bias"] = (geo.cout,)
    A = GuardedArena(shapes, dev)
    A.param("L.weight").copy_(_bf(_randn(g, *shapes["L.weight"], scale=(geo.cin * math.prod(ks)) ** -0.5)))
    if geo.has_bias:
        A.param("L.bias").copy_(_randn(g, geo.cout, scale=0.5))
    pre = {n: (_randn(g, *s, scale=0.5) if prefill else torch.zeros(s, device=dev)) for n, s in shapes.items()}
    for n, v in pre.items():
        A.grad(n).copy_(v)
    lay = full_train._FullLayer("L", types.SimpleNamespace(bias=True if geo.has_bias else None), geo.kind, A,
                                pad_in=geo.pad_in, pad_out=geo.pad_out)
    lay.pack()
    return lay, A, pre


def _check_param_grads(geo, A, pre, dw, db, sw, sb, tag):
    assert_accum(A.grad("L.weight"), pre["L.weight"].double() + dw, pre["L.weight"].double().abs() + sw, f"{tag} dW")
    if geo.has_bias:
        assert_accum(A.grad("L.bias"), pre["L.bias"].double() + db, pre["L.bias"].double().abs() + sb, f"{tag} db")
    A.check_guards(tag)


def check_full(geo: Geo, dev, seed=1):
    """_FullLayer forward + backward: y, dx, dW, db against fp64 autograd.  Padded layers (conv_in / out) get non-zero values in
    their padding channels: the padded weight rows / columns must ignore them and the gradient fold must drop them."""
    kind, pts, cin, cout = geo.kind, tuple(geo.points), geo.cin, geo.cout
    g = torch.Generator(device=dev).manual_seed(seed)
    lay, A, pre = _full_layer(geo, dev, g)
    params0 = A.params.clone()
    pc_in, pc_out = geo.pad_in or cin, geo.pad_out or cout
    x = _randn(g, *pts, pc_in).to(BF16)
    dy = _randn(g, *pts, pc_out).to(BF16)
    y, saved = lay.forward(x, True)
    dx = lay.backward(saved, dy)

    tag = f"full {geo_id(geo)}"
    w, b = A.param("L.weight"), (A.param("L.bias") if geo.has_bias else None)

    def f(a, ww, bb):
        return _ref_op(kind, a, ww, bb)
    y64, dx64, dw64, db64 = _ref_grads(f, x[..., :cin], w, b, dy[..., :cout])
    _, _, sw, sb = _ref_grads(f, x[..., :cin].double().abs(), w, b, dy[..., :cout].double().abs())
    assert_close(y[..., :cout], y64, what=f"{tag} y")
    assert_close(dx[..., :cin], dx64, what=f"{tag} dx")
    if pc_out > cout:
        assert not y[..., cout:].any(), f"{tag}: padding output channels are not zero"
    if pc_in > cin:
        assert not dx[..., cin:].any(), f"{tag}: padding input-gradient channels are not zero"
        assert not lay._gw_p.any(), f"{tag}: the padded gradient buffer was not cleared after the fold"
    _check_param_grads(geo, A, pre, dw64, db64, sw, sb, tag)
    assert torch.equal(A.params, params0), f"{tag}: the backward wrote into the parameters"


# ----------------------------------------------------------------------------- c. Downsample / Upsample compositions
def check_resample(geo: Geo, dev, seed=2):
    """role down: the stride-1 conv at the pre-down grid + resample2x "sub" (forward), "stuff" + the layer's backward (adjoint),
    as train_unet._seq_fwd / _seq_bwd run a Downsample, against autograd of F.conv2d(stride=2, padding=1).
    role up: upsample_nearest2x + conv, the layer's backward + "pool", against autograd of F.interpolate(nearest) + F.conv2d."""
    from t2v_turbo_b200 import ops
    assert geo.kind == "conv2d" and geo.role in ("down", "up") and geo.cin == geo.cout
    n, hh, ww = geo.points
    c = geo.cin
    g = torch.Generator(device=dev).manual_seed(seed)
    lay, A, pre = _full_layer(geo, dev, g)
    w, b = A.param("L.weight"), (A.param("L.bias") if geo.has_bias else None)
    tag = f"resample {geo_id(geo)}"
    if geo.role == "down":
        x = _randn(g, n, hh, ww, c).to(BF16)
        dy = _randn(g, n, hh // 2, ww // 2, c).to(BF16)
        y_full, saved = lay.forward(x, True)
        y = ops.resample2x(y_full, "sub")
        dx = lay.backward(saved, ops.resample2x(dy.contiguous(), "stuff"))

        def f(a, k, bb):
            return F.conv2d(a.permute(0, 3, 1, 2), k, bb, stride=2, padding=1).permute(0, 2, 3, 1)
    else:
        x = _randn(g, n, hh // 2, ww // 2, c).to(BF16)
        dy = _randn(g, n, hh, ww, c).to(BF16)
        y, saved = lay.forward(ops.upsample_nearest2x(x), True)
        dx = ops.resample2x(lay.backward(saved, dy), "pool")

        def f(a, k, bb):
            up = F.interpolate(a.permute(0, 3, 1, 2), scale_factor=2, mode="nearest")
            return F.conv2d(up, k, bb, padding=1).permute(0, 2, 3, 1)
    y64, dx64, dw64, db64 = _ref_grads(f, x, w, b, dy)
    _, _, sw, sb = _ref_grads(f, x.double().abs(), w, b, dy.double().abs())
    assert_close(y, y64, what=f"{tag} y")
    assert_close(dx, dx64, what=f"{tag} dx")
    _check_param_grads(geo, A, pre, dw64, db64, sw, sb, tag)


# ----------------------------------------------------------------------------- d. impulse (border) tests
def _sites_2d(n, h, w):
    """Corners, edge midpoints and the centre of frames 0, 1 and n - 1, kept >= 3 points apart (Chebyshev) within a frame so
    that no two 3x3 neighbourhoods overlap; frame 2 (n >= 4) carries none."""
    cands = [(0, 0), (0, w - 1), (h - 1, 0), (h - 1, w - 1), (0, w // 2), (h - 1, w // 2), (h // 2, 0), (h // 2, w - 1), (h // 2, w // 2)]
    keep = []
    for q in cands:
        if all(max(abs(q[0] - p[0]), abs(q[1] - p[1])) >= 3 for p in keep):
            keep.append(q)
    return [(f, qy, qx) for f in sorted({0, 1, n - 1}) for qy, qx in keep]


def check_impulse(kind, grid, c, dev, seed=4):
    """dy one-hot in point and channel (impulse k at site q_k, output channel j_k): every dx / dW element is at most one bf16 x 1
    product, so the results are exact.  dx[q_k + off(tap)] == W[j_k, :, tap] and zero everywhere else (neighbouring frames, the
    other video, the padding); dW[j_k, :, tap] == x[q_k + off(tap)] or 0 where the tap lands in the padding; db[j_k] == 1."""
    geo = Geo(kind, tuple(grid), c, c, True, 0, 0, "impulse")
    g = torch.Generator(device=dev).manual_seed(seed)
    lay, A, _ = _full_layer(geo, dev, g, prefill=False)
    w = A.param("L.weight")
    x = _randn(g, *grid, c).to(BF16)
    _, saved = lay.forward(x, True)
    if kind == "conv2d":
        n, h, wd = grid
        sites = _sites_2d(n, h, wd)
        # tap (ky, kx) of output point (f, y, x) reads input point (f, y + ky - 1, x + kx - 1)
        reads = [[((f, qy + ky - 1, qx + kx - 1), (ky, kx)) for ky in range(3) for kx in range(3)
                  if 0 <= qy + ky - 1 < h and 0 <= qx + kx - 1 < wd] for f, qy, qx in sites]
    else:
        b, t, hw = grid
        sites = [(v, q, 0) for v in range(b) for q in (0, t // 2, t - 1)]
        sites = [(v, q, (7 * k + 3) % hw) for k, (v, q, _) in enumerate(sites)]      # distinct pixels: no shared neighbourhood
        reads = [[((v, q + kt - 1, s), (kt, 0, 0)) for kt in range(3) if 0 <= q + kt - 1 < t] for v, q, s in sites]
    assert len(sites) <= c
    js = [(5 * k) % c for k in range(len(sites))]                  # distinct output channels, spread over the 64-column slices
    dy = torch.zeros(*grid, c, device=dev, dtype=BF16)
    for (site, j) in zip(sites, js):
        dy[site + (j,)] = 1.0
    dx = lay.backward(saved, dy)
    exp_dx = torch.zeros(*grid, c, device=dev, dtype=torch.float32)
    exp_dw = torch.zeros_like(w)
    for rd, j in zip(reads, js):
        for pt, tap in rd:
            exp_dx[pt] = w[(j, slice(None)) + tap]
            exp_dw[(j, slice(None)) + tap] = x[pt].float()
    exp_db = torch.zeros(c, device=dev)
    exp_db[js] = 1.0
    tag = f"impulse {kind} {'x'.join(map(str, grid))}"
    bad = (dx.float() != exp_dx).nonzero()
    assert torch.equal(dx, exp_dx.to(BF16)), f"{tag} dx: {len(bad)} elements differ, first {bad[:4].tolist()}"
    bad = (A.grad("L.weight") != exp_dw).nonzero()
    assert torch.equal(A.grad("L.weight"), exp_dw), f"{tag} dW: {len(bad)} elements differ, first {bad[:4].tolist()}"
    assert torch.equal(A.grad("L.bias"), exp_db), f"{tag} db"
    A.check_guards(tag)
    print(f"[exact] {tag}: {len(sites)} impulses, dx / dW / db bit-exact")


# ----------------------------------------------------------------------------- e. VAE decoder layers
def check_decoder(geo: Geo, dev, seed=5):
    """vae_train._Conv (3x3, padded conv_in / conv_out included) and _Lin (1x1) of DecoderGrad: y = fwd(x), dx = bwd(dy)."""
    from t2v_turbo_b200 import vae_train
    kind, pts, cin, cout = geo.kind, tuple(geo.points), geo.cin, geo.cout
    ks = (3, 3) if kind == "conv2d" else (1, 1)
    g = torch.Generator(device=dev).manual_seed(seed)
    w = _bf(_randn(g, cout, cin, *ks, scale=(cin * math.prod(ks)) ** -0.5))
    b = _randn(g, cout, scale=0.5)
    mod = types.SimpleNamespace(weight=w, bias=b)
    S = vae_train._Conv(mod, pad_in=geo.pad_in, pad_out=geo.pad_out) if kind == "conv2d" else vae_train._Lin(mod)
    pc_in, pc_out = geo.pad_in or cin, geo.pad_out or cout
    x = _randn(g, *pts, pc_in).to(BF16)
    dy = _randn(g, *pts, pc_out).to(BF16)
    y = S.fwd(x)
    dx = S.bwd(dy)
    y64, dx64, _, _ = _ref_grads(lambda a, ww, bb: _ref_op(kind, a, ww, bb), x[..., :cin], w, b, dy[..., :cout])
    tag = f"decoder {geo_id(geo)}"
    assert_close(y[..., :cout], y64, what=f"{tag} y")
    assert_close(dx[..., :cin], dx64, what=f"{tag} dx")
    if pc_out > cout:
        assert not y[..., cout:].any(), f"{tag}: padding output channels are not zero"
    if pc_in > cin:
        assert not dx[..., cin:].any(), f"{tag}: padding input-gradient channels are not zero"


# ----------------------------------------------------------------------------- the B200 tests
_UNET = census()
_LORA = list({(g.kind, g.points, g.cin, g.cout): g for g in _UNET if g.role in ("lora", "down", "up")}.values())
_FULL = list({g[:7]: g for g in _UNET}.values())
_RESAMPLE = [g for g in _UNET if g.role in ("down", "up")]
_DECODER = decoder_census()


@pytest.mark.gpu
@pytest.mark.parametrize("geo", _LORA, ids=geo_id)
def test_lora_layer_adjoint(cuda_device, geo):
    check_lora(geo, cuda_device)


@pytest.mark.gpu
@pytest.mark.parametrize("geo", _FULL, ids=geo_id)
def test_full_layer_adjoint(cuda_device, geo):
    check_full(geo, cuda_device)


@pytest.mark.gpu
@pytest.mark.parametrize("geo", _RESAMPLE, ids=geo_id)
def test_resample_composition(cuda_device, geo):
    check_resample(geo, cuda_device)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,grid", [("conv2d", (4, 5, 8)), ("conv2d", (4, 10, 16)), ("conv2d", (4, 40, 64)),
                                       ("conv3d", (2, 16, 40))], ids=lambda v: v if isinstance(v, str) else "x".join(map(str, v)))
def test_impulse_exact(cuda_device, kind, grid):
    check_impulse(kind, grid, 128, cuda_device)


@pytest.mark.gpu
@pytest.mark.parametrize("geo", _DECODER, ids=geo_id)
def test_decoder_layer_adjoint(cuda_device, geo):
    check_decoder(geo, cuda_device)
