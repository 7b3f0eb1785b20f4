"""GPU parity of the v2 full fine-tune step (t2v_turbo_b200/full_train.py, distill_v2.py, csrc/train_full.cu).

STATUS.  Written after the round's GPU budget was all but spent; the last 1.7 GPU-minutes bought two short runs on a B200
(`profiles/r02_v2_gpu_kernel_tests.log`, `profiles/r02_v2_gpu_step_tests.log`):
  * every kernel-contract test below (GroupNorm / LayerNorm affine gradients, EMA, `wgrad_wide` incl. the in-place 64-column B
    slices against copied slices) PASSED (20 tests) — they are ordinary tests now;
  * the self-target step (+ a training-mode optimizer step) PASSED — ordinary test;
  * the step against the reference composition ran end to end: model_pred / target rel-L2 6.7e-3 / 6.4e-3, x_prev 1.3e-6, loss
    0.99671 vs 0.99582, every gradient finite, norm ratios 0.870 .. 1.113, stored tensors rel-L2 median 0.20 / worst 0.26 — the
    same noise-dominated picture as the v1 step (the pseudo-Huber gradient is sign-like: a fraction f of flipped signs costs
    2 sqrt(f) in rel-L2; tests/test_student_gpu.py observed 0.29 - 0.33 and 0.90 .. 1.17 there).  My first-guess bound (8e-2) was
    wrong, not the step; the assertions that run reached are ordinary now with the v1 test's sanity bounds, the ones it did NOT
    reach (clip norm, AdamW deltas, EMA) and the new LINEAR-loss test that pins the backward itself against the reference's
    autograd (the v1 suite's approach) have never executed and stay NON-STRICT xfail: they run, XPASS is evidence, a failure
    does not redden the suite.  Each of them (and the ones added later for the decoder gradient, the motion-prior score and the
    mid-size student) runs in ITS OWN PROCESS with a timeout (`test_never_run_in_its_own_process`), so a hang or a sticky CUDA error
    in never-executed device code cannot stall or poison anything else; what they measure is appended to
    gpurun_out/r02_never_run_observed.jsonl and their logs to gpurun_out/r02_never_run_child_logs.txt.  The file sorts last.

Kernel contracts are checked against tests/mock_ops.py evaluated on the CPU in fp32 on the same bf16-rounded inputs.
"""
import os

import pytest
import torch

import mock_ops
from test_kernels_gpu import BF16, _ops, assert_close, rnd

pytestmark = pytest.mark.gpu
_CHILD = bool(os.environ.get("T2V_ZZ_CHILD"))
NEVER_RUN = []


def never_run(fn):
    """A test whose device code has never executed.  It runs in ITS OWN PROCESS (test_never_run_in_its_own_process below spawns
    `pytest this_file::name --runxfail` with a timeout), so a hang, an illegal address or a sticky CUDA error in one of them can neither
    stall the suite nor poison the tests that run after it; in the parent process the body is skipped."""
    NEVER_RUN.append(fn.__name__)
    return pytest.mark.skipif(not _CHILD, reason="never-run device code: executed in a child process by test_never_run_in_its_own_process")(fn)
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _rel(got, ref):
    got, ref = got.double().cpu(), ref.double().cpu()
    return ((got - ref).norm() / (ref.norm() + 1e-30)).item()


def _observe(test, **values):
    """Append what a never-run test measured to gpurun_out/r02_never_run_observed.jsonl (the -q log drops the prints of xfailed tests)."""
    import json
    try:
        d = os.path.join(os.environ.get("GRAFT_REPO_ROOT", os.path.dirname(os.path.dirname(os.path.abspath(__file__)))), "gpurun_out")
        os.makedirs(d, exist_ok=True)
        with open(os.path.join(d, "r02_never_run_observed.jsonl"), "a") as f:
            f.write(json.dumps({"test": test, **{k: (float(v) if not isinstance(v, (str, list, tuple)) else v) for k, v in values.items()}}) + "\n")
    except OSError:
        pass


def _mock(dtype=torch.float32):
    mock_ops.ACT = dtype
    return mock_ops


# ----------------------------------------------------------------------------- the new kernels
@pytest.mark.parametrize("n,hw,c,silu", [(4, 640, 320, True), (2, 2560, 640, True), (3, 160, 1280, False), (16, 40, 128, True),
                                          (2, 1000, 64, False), (1, 320, 2560, True)])
def test_groupnorm_affine_grad(cuda_device, n, hw, c, silu):
    ops = _ops()
    x = (rnd(n * hw, c, scale=1.5, seed=1) + 0.7).to(BF16)
    dy = rnd(n * hw, c, seed=2).to(BF16)
    gamma, beta = (1.0 + 0.3 * rnd(c, seed=3)).float(), (0.2 * rnd(c, seed=4)).float()
    dg = torch.full((c,), 0.5, device="cuda")          # accumulated INTO
    db = torch.full((c,), -0.25, device="cuda")
    ws = []
    ops.groupnorm_bwd(x, dy, gamma, beta, rows_per_sample=hw, eps=1e-5, silu=silu, keep_ws=ws)
    ops.groupnorm_affine_grad(x, dy, gamma, beta, ws[0], dg, db, rows_per_sample=hw, eps=1e-5, silu=silu)
    m = _mock()
    rg, rb = torch.full((c,), 0.5), torch.full((c,), -0.25)
    xs = x.float().cpu()
    m.groupnorm_affine_grad(xs, dy.float().cpu(), gamma.cpu(), beta.cpu(), ("gn-stats", xs.data_ptr(), hw, 32), rg, rb,
                            rows_per_sample=hw, eps=1e-5, silu=silu)
    assert_close(dg.cpu(), rg, rtol=2e-3, atol_scale=1e-3, what=f"gn dgamma n={n} hw={hw} c={c}")     # fp32 sums: tighter than bf16 outputs
    assert_close(db.cpu(), rb, rtol=2e-3, atol_scale=1e-3, what=f"gn dbeta n={n} hw={hw} c={c}")


@pytest.mark.parametrize("rows,c", [(4096, 320), (2560, 640), (1000, 1280), (77, 64), (5, 1024)])
def test_layernorm_affine_grad(cuda_device, rows, c):
    ops = _ops()
    x = (rnd(rows, c, scale=2.0, seed=5) - 0.3).to(BF16)
    dy = rnd(rows, c, seed=6).to(BF16)
    dg, db = torch.ones(c, device="cuda"), torch.zeros(c, device="cuda")
    ops.layernorm_affine_grad(x, dy, dg, db, 1e-5)
    rg, rb = torch.ones(c), torch.zeros(c)
    _mock().layernorm_affine_grad(x.float().cpu(), dy.float().cpu(), rg, rb, 1e-5)
    assert_close(dg.cpu(), rg, rtol=2e-3, atol_scale=1e-3, what=f"ln dgamma rows={rows} c={c}")
    assert_close(db.cpu(), rb, rtol=2e-3, atol_scale=1e-3, what=f"ln dbeta rows={rows} c={c}")


@pytest.mark.parametrize("n,offset", [(1 << 20, 0), (1000003, 0), (4099, 1), (3, 0)])
def test_ema_update(cuda_device, n, offset):
    ops = _ops()
    tgt = rnd(n + offset, seed=7)[offset:]           # offset 1: a 4-byte-aligned slice takes the scalar path
    src = rnd(n + offset, seed=8)[offset:]
    ref = tgt.clone().mul_(0.95).add_(src, alpha=0.05)
    ops.ema_update(tgt, src, 0.95)
    assert torch.allclose(tgt, ref, rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("kind,shape,cout", [("linear", (4096, 320), 320), ("linear", (616, 1024), 640), ("linear", (2, 256), 320),
                                             ("conv2d", (4, 16, 24, 128), 192), ("conv3d", (2, 8, 160, 64), 128)])
def test_wgrad_wide_base_weight_gradient(cuda_device, kind, shape, cout):
    """dW of a whole layer through 64-column slices of dy read in place == the contract (and == wgrad on copied slices)."""
    ops = _ops()
    x = rnd(*shape, seed=9).to(BF16)
    dy = rnd(*shape[:-1], cout, seed=10).to(BF16)
    cin = shape[-1]
    taps = None if kind == "linear" else (ops._TAPS_3X3 if kind == "conv2d" else ops._TAPS_T3)
    nt = 1 if taps is None else len(taps)
    out = torch.zeros(cout, cin, nt, device="cuda")
    ops.wgrad_wide(x, dy, out, taps=taps, out_strides=(cin * nt, nt, 1))
    ref = torch.zeros(cout, cin, nt)
    _mock().wgrad_wide(x.float().cpu(), dy.float().cpu(), ref, taps=taps, out_strides=(cin * nt, nt, 1))
    assert_close(out.cpu(), ref, rtol=4e-3, atol_scale=2e-3, what=f"wgrad_wide {kind} {shape} -> {cout}")
    if shape[0] >= 16:
        out2 = torch.zeros_like(out)
        for j0 in range(0, cout, 64):
            ops.wgrad(x, dy[..., j0:j0 + 64].contiguous(), out2[j0:j0 + 64], taps=taps, out_strides=(cin * nt, nt, 1))
        assert_close(out, out2, rtol=1e-3, atol_scale=1e-4, what="wgrad_wide vs wgrad on copied slices")   # fp32 atomics: order only


# ----------------------------------------------------------------------------- the whole step
def _setup(with_ema=True):
    from oracle.configs import UNET_CONFIGS
    from oracle.weights import seeded_state_dict
    from t2v_turbo_b200.distill_v2 import V2Step
    from t2v_turbo_b200.full_train import FullUNet
    from t2v_turbo_b200.scheduler import T2VTurboScheduler
    from t2v_turbo_b200.unet import UNetModel
    g = torch.load(os.path.join(GOLD, "v2_step_small_motion.pt"))
    spec = UNET_CONFIGS["small_motion"]
    m = UNetModel(**spec["cfg"])
    sd = seeded_state_dict(m.state_dict(), spec["weight_seed"])
    m.load_state_dict(sd, strict=True)
    m = m.cuda().eval()
    s = FullUNet(m, with_target=with_ema).eval()
    s.pack()
    target = None
    if with_ema:
        gq = torch.Generator().manual_seed(g["target_perturb_seed"])
        for n, p in m.named_parameters():
            s.arena.view(s.arena.target, s.arena.index[n]).copy_(sd[n] * (1.0 + 0.02 * torch.randn(p.shape, generator=gq)))
        target = UNetModel(**spec["cfg"])
        target.load_state_dict(sd, strict=True)
        from t2v_turbo_b200.distill_v2 import attach_ema_target
        target = attach_ema_target(s, target.cuda(), dtype=torch.float32)     # the EMA network's parameters ARE the target arena
    h = g["hyper"]
    step = V2Step(s, T2VTurboScheduler(linear_start=0.00085, linear_end=0.012), target_unet=target, num_ddim_timesteps=h["n_ddim"],
                  topk=h["topk"], motion_gs=h["motion_gs"], percentage=h["percentage"], use_motion_cond=True,
                  timestep_scaling_factor=h["ts_scale"])
    return g, s, step, sd


def _run_reference_step():
    from t2v_turbo_b200.distill_v2 import train_step_v2
    g, s, step, sd = _setup(with_ema=True)
    inp, h = g["inputs"], g["hyper"]
    batch = {k: inp[k].cuda() for k in ("index", "z_t", "cond_teacher_out", "uncond_teacher_out", "score", "use_motion_guide", "prompt_emb")}
    p0 = s.arena.params.clone()
    out = train_step_v2(step, batch, lr=h["lr"], temporal_lr_scale=h["temporal_lr_scale"], ema_decay=h["ema_decay"],
                        max_grad_norm=h["max_grad_norm"], weight_decay=h["weight_decay"], fixed=dict(w=inp["w"]))
    torch.cuda.synchronize()
    return g, s, out, p0          # (the optimizer folds clip / mean into its grad_scale: arena.grads still holds the raw gradients)


def test_v2_step_vs_reference_composition(cuda_device):
    """Forward quantities, loss and the gradient's direction (observed on B200: see the file header)."""
    g, s, out, p0 = _run_reference_step()
    assert out["start_timesteps"].tolist() == g["start_timesteps"].tolist() and out["timesteps"].tolist() == g["timesteps"].tolist()
    e = {k: _rel(out[k], g[k]) for k in ("model_pred", "x_prev", "target")}
    loss, loss_ref = float(out["loss"]), float(g["loss"])
    print(f"\n[v2 small] loss {loss:.6f} vs reference {loss_ref:.6f}; rel-L2 {e}")
    assert e["x_prev"] < 1e-5 and e["model_pred"] < 1.4e-2 and e["target"] < 1.3e-2, e          # observed 1.3e-6 / 6.7e-3 / 6.4e-3
    # The loss is the pseudo-Huber mean of OUR model_pred - target (fp64 recomputation), and it departs from the reference loss
    # by no more than the forward departures above allow: the pseudo-Huber function is 1-Lipschitz, so |loss - loss_ref| <=
    # mean |(p - t) - (p_ref - t_ref)|.  A fixed bound on |loss - loss_ref| is not a property of the code: the fp32 atomics make
    # each run a different bf16 rounding pattern, and on these 2 048 elements the loss moved by 8.9e-4 and by 2.2e-3 between runs.
    d, d_ref = (out["model_pred"] - out["target"]).double().cpu(), (g["model_pred"] - g["target"]).double()
    c = 0.001                                                                                  # V2Step's default huber_c
    own = float(((d * d + c * c).sqrt() - c).mean())
    assert abs(loss - own) < 1e-5 * own, (loss, own)
    assert abs(loss - loss_ref) <= float((d - d_ref).abs().mean()) + 1e-6, (loss, loss_ref, float((d - d_ref).abs().mean()))
    assert abs(loss - loss_ref) < 1e-2 * loss_ref, (loss, loss_ref)
    names = s.arena.names
    gv = s.arena.grad
    assert torch.isfinite(s.arena.grads).all()
    ratio = torch.tensor([gv(n).double().norm().item() / max(g["grad_norms"][n], 1e-30) for n in names])
    print(f"[v2 small] grad-norm ratio ours/reference: min {ratio.min():.4f} max {ratio.max():.4f} over {len(names)} tensors")
    rels = {n: _rel(gv(n), sc * t.float()) for n, (sc, t) in g["grads_full"].items()}
    wn = max(rels, key=rels.get)
    print(f"[v2 small] full-tensor rel-L2 over {len(rels)} tensors: median {sorted(rels.values())[len(rels) // 2]:.3e}, worst {rels[wn]:.3e} ({wn})")
    # sign-like loss gradient: noise-dominated (header).  Observed 0.870 .. 1.113 and 0.20 / 0.26; the v1 step's sanity bounds.
    assert (ratio - 1).abs().max() < 0.25 and rels[wn] < 0.45, (ratio.min(), ratio.max(), wn, rels[wn])


def test_v2_step_self_target_and_second_step(cuda_device):
    from t2v_turbo_b200.distill_v2 import train_step_v2
    g, s, step, _ = _setup(with_ema=False)
    inp = g["inputs"]
    batch = {k: inp[k].cuda() for k in ("index", "z_t", "cond_teacher_out", "uncond_teacher_out", "score", "prompt_emb")}
    s.arena.zero_grad()
    out = step(batch, fixed=dict(w=inp["w"]))
    assert _rel(out["target"], g["target_self"]) < 3e-2
    assert abs(float(out["loss"]) - float(g["loss_self_target"])) < 3e-2 * float(g["loss_self_target"])
    s.train()                                        # dropouts on: finite gradients, and a step changes the prediction
    out1 = train_step_v2(step, batch, lr=1e-4, fixed=dict(w=inp["w"]))
    assert torch.isfinite(s.arena.grads).all() and float(s.arena.grad_norm()) > 0
    s.eval()
    s.arena.zero_grad()
    out2 = step(batch, fixed=dict(w=inp["w"]))
    assert _rel(out2["model_pred"], out["model_pred"]) > 1e-5, "the optimizer step did not change the student's prediction"
    assert torch.isfinite(out1["loss"]).all()


@never_run
def test_v2_step_clip_optimizer_and_ema(cuda_device):
    g, s, out, p0 = _run_reference_step()
    h = g["hyper"]
    gn = float(s.arena.grad_norm())
    _observe("v2_step_clip_optimizer_and_ema", grad_norm=gn, grad_norm_ref=g["total_norm"])
    assert abs(gn - g["total_norm"]) < 6e-2 * g["total_norm"], (gn, g["total_norm"])
    # the first AdamW step moves each weight by ~lr * sign(grad) (+ weight decay): bounded by lr per group, 3x larger in the temporal group
    moved = (s.arena.params - p0).abs()
    tmask = torch.zeros_like(moved, dtype=torch.bool)
    for lo, hi, temporal in s.arena.runs:
        tmask[lo:hi] = temporal
    bound = h["lr"] * (1 + h["weight_decay"] * float(p0.abs().max()))
    assert float(moved[~tmask].max()) <= 1.05 * bound + 1e-9 and float(moved[tmask].max()) <= 1.05 * bound * h["temporal_lr_scale"] + 1e-9
    assert float(moved[tmask].mean()) > 2.0 * float(moved[~tmask].mean()), "temporal group must step with lr * temporal_lr_scale"
    for n, t in g["ema_after"].items():
        assert _rel(s.arena.view(s.arena.target, s.arena.index[n]), t) < 1e-4, n


@never_run
def test_full_unet_backward_vs_reference_autograd_linear_loss(cuda_device):
    """The backward itself, pinned the way the v1 suite pins its student: a LINEAR loss sum(eps * g) (no sign-like gradient), every
    one of the 629 parameter gradients against the unmodified reference's fp32 autograd (tests/golden/full_grads_small_motion.pt),
    with the reference's OWN bf16 forward + backward as the yardstick (stored in the fixture: output 1.9e-2, gradients median
    4.0e-2 / worst 6.5e-2 / concatenated 3.8e-2, norm ratios 0.986 .. 1.020).  Bounds = up to 2x that yardstick (the v1 student test holds 1.3x / 1.15x; bias and
    norm-affine gradients are small tensors, so this one is looser); never observed for this model."""
    from oracle.configs import UNET_CONFIGS, unet_inputs
    from oracle.weights import seeded_state_dict
    from t2v_turbo_b200.full_train import FullUNet
    from t2v_turbo_b200.unet import UNetModel
    g = torch.load(os.path.join(GOLD, "full_grads_small_motion.pt"))
    spec = UNET_CONFIGS["small_motion"]
    m = UNetModel(**spec["cfg"])
    m.load_state_dict(seeded_state_dict(m.state_dict(), spec["weight_seed"]), strict=True)
    s = FullUNet(m.cuda().eval()).eval()
    s.pack()
    inp = unet_inputs(spec, g["timestep"])
    y = s(inp["x"].cuda(), inp["timesteps"].cuda(), context=inp["context"].cuda(), fps=16, timestep_cond=inp["timestep_cond"].cuda(),
          motion_cond=inp["motion_cond"].cuda())
    e_y = _rel(y, g["output"])
    s.arena.zero_grad()
    s.backward(g["d_out"].cuda())
    torch.cuda.synchronize()
    assert torch.isfinite(s.arena.grads).all()
    names = g["names"]
    ratio = torch.tensor([s.arena.grad(n).double().norm().item() / max(g["grad_norms"][n], 1e-30) for n in names])
    rels = {n: _rel(s.arena.grad(n), sc * t.float()) for n, (sc, t) in g["grads_full"].items()}
    wn = max(rels, key=rels.get)
    total = _rel(torch.cat([s.arena.grad(n).flatten() for n in rels]), torch.cat([(sc * t.float()).flatten() for sc, t in g["grads_full"].values()]))
    rb = g["ref_bf16"]
    print(f"\n[full small] forward rel-L2 {e_y:.3e}; grad-norm ratio {ratio.min():.4f} .. {ratio.max():.4f} over {len(names)} tensors; stored tensors "
          f"median {sorted(rels.values())[len(rels) // 2]:.3e} worst {rels[wn]:.3e} ({wn}) concatenated {total:.3e}; reference bf16: {rb}")
    _observe("full_unet_backward_linear_loss", forward_rel=e_y, ratio_min=ratio.min(), ratio_max=ratio.max(), worst_rel=rels[wn], worst_name=wn,
             concat_rel=total)
    assert e_y <= 1.15 * rb["output_rel"], (e_y, rb["output_rel"])
    assert (ratio - 1).abs().max() < 6e-2, (ratio.min(), ratio.max())
    assert rels[wn] <= 2.0 * rb["grad_rel_worst"] and total <= 1.5 * rb["grad_rel_concat"], (wn, rels[wn], total)


# ----------------------------------------------------------------------------- vae.decode WITH grad (never run on a GPU)
@never_run
@pytest.mark.parametrize("n,hw,scale", [(2, 256, 128 ** -0.5), (1, 2560, 512 ** -0.5)])
def test_softmax_bwd_rows(cuda_device, n, hw, scale):
    ops = _ops()
    s = (rnd(n, hw, hw, seed=30) * 3.0).to(BF16)
    p = s.clone()
    ops.softmax_rows_(p, scale)
    dp = rnd(n, hw, hw, seed=31).to(BF16)
    ds = dp.clone()
    ops.softmax_bwd_rows_(ds, p, scale)
    ref = p.float().cpu().clone()
    _mock().softmax_bwd_rows_(dpr := dp.float().cpu().clone(), ref, scale)
    assert_close(ds.cpu(), dpr, what=f"softmax_bwd_rows {n}x{hw}x{hw}")


@never_run
def test_decoder_grad_vs_oracle_autograd(cuda_device):
    """vae_train.decode_with_grad on B200 vs autograd through the VAE oracle (fp32, CPU): image and the latent gradient under a
    clamp + non-linear score, the reference's frame call form.  Bounds: the VAE decode test's (2.0e-2) for the image, 4x that for the
    gradient through ~30 bf16 layers and a clamp; never observed."""
    from oracle.configs import VAE_CONFIGS
    from oracle.vae_oracle import decode_first_stage_2dae
    from oracle.weights import vae_state_dict
    from t2v_turbo_b200.vae import AutoencoderKL
    from t2v_turbo_b200.vae_train import decode_with_grad
    spec = VAE_CONFIGS["small"]
    v = AutoencoderKL(spec["ddconfig"], spec["embed_dim"])
    sd = vae_state_dict(v.state_dict(), spec["weight_seed"])
    v.load_state_dict(sd)
    v = v.cuda().eval()
    z = torch.randn(spec["z_shape"], generator=torch.Generator().manual_seed(3))
    side = 16 * 2 ** (len(spec["ddconfig"]["ch_mult"]) - 1)
    probe = torch.randn(1, 3, 4, side, side, generator=torch.Generator().manual_seed(5))

    def reward(img, pr):
        x = (img / 2 + 0.5).clamp(0, 1)
        return (x * pr).sum() + (x ** 2).mean()
    z1 = z.clone().cuda().requires_grad_(True)
    img = decode_with_grad(v, z1, scale=1.0 / 0.18215)
    reward(img, probe.cuda()).backward()
    torch.cuda.synchronize()
    z2 = z.clone().requires_grad_(True)
    ref = decode_first_stage_2dae(sd, spec["ddconfig"], z2)
    reward(ref, probe).backward()
    e_img, e_g = _rel(img.detach(), ref.detach()), _rel(z1.grad, z2.grad)
    print(f"\n[decoder grad small] image rel-L2 {e_img:.3e}, latent-gradient rel-L2 {e_g:.3e}")
    _observe("decoder_grad", image_rel=e_img, latent_grad_rel=e_g)
    assert e_img < 2.0e-2 and e_g < 8.0e-2, (e_img, e_g)


# ----------------------------------------------------------------------------- the motion-prior score (never run on a GPU)
@never_run
@pytest.mark.parametrize("b,t,hw,heads", [(2, 4, 64, 2), (1, 16, 160, 5)])
def test_attention_temporal_probs_bwd(cuda_device, b, t, hw, heads):
    ops = _ops()
    inner = heads * 64
    qkv = rnd(b * t * hw, 3 * inner, seed=32).to(BF16)
    q, k = qkv[:, :inner], qkv[:, inner:2 * inner]                      # views of a fused projection
    dp = rnd(b * hw * heads, t, t, seed=35)
    dq, dk = ops.attention_temporal_probs_bwd(q, k, dp, b=b, t=t, hw=hw, heads=heads, scale=0.125)
    rq, rk = _mock().attention_temporal_probs_bwd(q.float().cpu().contiguous(), k.float().cpu().contiguous(), dp.cpu(), b=b, t=t, hw=hw,
                                                   heads=heads, scale=0.125)
    assert_close(dq.cpu(), rq, what=f"probs_bwd dq b={b} t={t} hw={hw} H={heads}")
    assert_close(dk.cpu(), rk, what=f"probs_bwd dk b={b} t={t} hw={hw} H={heads}")


@never_run
def test_motion_prior_score_vs_reference(cuda_device):
    """get_motion_prior_score on B200 vs the unmodified reference's autograd (fp32 fixture).  The score is a gradient through ~40 bf16
    layers of a loss on softmax outputs; bound: 2x the student-gradient yardstick (worst 6e-2), never observed."""
    from oracle.configs import UNET_CONFIGS
    from oracle.weights import seeded_state_dict
    from t2v_turbo_b200.motion_prior import ScoreUNet, get_motion_prior_score
    from t2v_turbo_b200.unet import UNetModel
    g = torch.load(os.path.join(GOLD, "motion_score_small.pt"))
    m = UNetModel(**g["cfg"])
    m.load_state_dict(seeded_state_dict(m.state_dict(), UNET_CONFIGS["small"]["weight_seed"]), strict=True)
    view = ScoreUNet(m.cuda().eval())
    view.pack()
    score, eps = get_motion_prior_score(view, g["latents"].cuda(), g["ts"].cuda(), g["example"].cuda(), {"context": g["ctx_orig"].cuda(), "fps": 16},
                                        {"context": g["ctx_inf"].cuda(), "fps": 16}, g["temp_loss_scale"])
    torch.cuda.synchronize()
    e_eps, e_s = _rel(eps, g["cond_teacher_output"]), _rel(score, g["score"])
    print(f"\n[motion score small] eps rel-L2 {e_eps:.3e}, score rel-L2 {e_s:.3e}")
    _observe("motion_prior_score", eps_rel=e_eps, score_rel=e_s)
    assert e_eps < 3e-2 and e_s < 1.5e-1, (e_eps, e_s)


@never_run
def test_student_unet_vc2_topology_vs_reference_lora_gradients(cuda_device):
    """The v1 student on the FULL VC2 topology at 128 base channels (575 LoRA layers; 2x2-pixel frames at the deepest level — GEMM
    geometries no other GPU test reaches) against the unmodified reference's autograd, yardstick = the reference's own bf16 backward
    (stored in the fixture: median 4.8e-2 / worst 7.6e-2 / concatenated 4.2e-2).  The same comparison passes on CPU at 2e-4
    (tests/test_train_composition_cpu.py); never run on a GPU."""
    from oracle.configs import UNET_CONFIGS, student_loras, unet_inputs
    from oracle.weights import seeded_state_dict
    from t2v_turbo_b200.train_unet import StudentUNet
    from t2v_turbo_b200.unet import UNetModel
    g = torch.load(os.path.join(GOLD, "student_grads_mid.pt"))
    spec = {**UNET_CONFIGS["mid"], "x_shape": tuple(g["x_shape"])}
    m = UNetModel(**spec["cfg"])
    m.load_state_dict(seeded_state_dict(m.state_dict(), spec["weight_seed"]), strict=True)
    s = StudentUNet(m.cuda().eval(), r=64).eval()
    s.arena.load_list(student_loras(g["shapes"]))
    s.pack()
    inp = unet_inputs(spec, g["timestep"])
    y = s(inp["x"].cuda(), inp["timesteps"].cuda(), context=inp["context"].cuda(), fps=16, timestep_cond=inp["timestep_cond"].cuda())
    e_y = _rel(y, g["output"])
    s.arena.zero_grad()
    s.backward(g["d_out"].cuda())
    torch.cuda.synchronize()
    n = len(s.arena.shapes)
    ratio = torch.tensor([s.arena.grad(i).double().norm().item() / max(g["grad_norms"][i].item(), 1e-30) for i in range(n)])
    rels = {j: _rel(s.arena.grad(j), sc * t.float()) for j, (sc, t) in g["grads_full"].items()}
    total = _rel(torch.cat([s.arena.grad(j).flatten() for j in rels]), torch.cat([(sc * t.float()).flatten() for sc, t in g["grads_full"].values()]))
    rb = g["ref_bf16"]
    print(f"\n[student mid] forward {e_y:.3e}; grad-norm ratio {ratio.min():.4f} .. {ratio.max():.4f}; stored tensors worst {max(rels.values()):.3e} "
          f"concatenated {total:.3e}; reference bf16: {rb}")
    _observe("student_unet_vc2_topology", forward_rel=e_y, ratio_min=ratio.min(), ratio_max=ratio.max(), worst_rel=max(rels.values()), concat_rel=total)
    assert e_y <= 1.15 * rb["output_rel"] and (ratio - 1).abs().max() < 4e-2
    assert max(rels.values()) <= 1.5 * rb["grad_rel_worst"] and total <= 1.3 * rb["grad_rel_concat"]


@never_run
def test_graphed_v2_step_matches_eager(cuda_device):
    """GraphedV2Step (the device side of the self-target step as a chain of CUDA graphs cut at the gradient-arena hooks) reproduces the
    eager step: same loss and gradients for the same draws (eval mode), replayed with a different batch in between (the static buffers
    really are re-read), cuts at descending arena offsets.  The v1 twin of this test passes on B200; this one never ran."""
    from t2v_turbo_b200.distill_v2 import GraphedV2Step
    g, s, step, _ = _setup(with_ema=False)
    inp = g["inputs"]
    batch = {k: inp[k].cuda() for k in ("index", "z_t", "cond_teacher_out", "uncond_teacher_out", "score", "use_motion_guide", "prompt_emb")}
    other = {k: (v.flip(0) if torch.is_tensor(v) and v.dim() > 0 else v) for k, v in batch.items()}
    fixed = dict(w=inp["w"])
    s.arena.zero_grad()
    out_e = step(batch, fixed=fixed)
    grads_e, loss_e = s.arena.grads.clone(), float(out_e["loss"])
    gs = GraphedV2Step(step, batch)
    offs = [o for _, o in gs.segments]
    assert offs == sorted(offs, reverse=True) and offs[-1] == 0 and len(offs) >= 3, offs
    s.arena.zero_grad()
    gs(other, fixed=dict(w=inp["w"].flip(0)))
    s.arena.zero_grad()
    out_g = gs(batch, fixed=fixed)
    torch.cuda.synchronize()
    e_l, e_g = abs(float(out_g["loss"]) - loss_e) / loss_e, _rel(s.arena.grads, grads_e)
    _observe("graphed_v2_step", loss_rel=e_l, grads_rel=e_g, segments=len(offs))
    assert e_l < 1e-5 and e_g < 2e-2, (e_l, e_g)              # fp32 atomics reorder between runs: the v1 test's run-to-run bound


# ----------------------------------------------------------------------------- the isolation harness for everything marked @never_run
@pytest.mark.xfail(strict=False, reason="device code that never ran on a GPU (round-2 budget exhausted): an XPASS here is the first evidence, "
                                        "a failure is recorded but does not redden the suite; host composition CPU-verified")
@pytest.mark.parametrize("name", NEVER_RUN)
def test_never_run_in_its_own_process(cuda_device, name):
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "pytest", f"{os.path.abspath(__file__)}::{name}", "-m", "gpu", "--runxfail", "-q", "-s", "-p", "no:cacheprovider"]
    try:
        r = subprocess.run(cmd, cwd=root, env={**os.environ, "T2V_ZZ_CHILD": "1"}, capture_output=True, text=True, timeout=900)
        rc, out = r.returncode, r.stdout[-6000:] + r.stderr[-2000:]
    except subprocess.TimeoutExpired as e:
        rc, out = -9, f"TIMEOUT after 900 s\n{(e.stdout or b'')[-3000:]!r}"
    try:
        d = os.path.join(os.environ.get("GRAFT_REPO_ROOT", root), "gpurun_out")
        os.makedirs(d, exist_ok=True)
        with open(os.path.join(d, "r02_never_run_child_logs.txt"), "a") as f:
            f.write(f"===== {name}: rc={rc}\n{out}\n")
    except OSError:
        pass
    import re
    assert rc == 0, f"{name} failed in its child process (rc={rc}):\n{out[-1500:]}"
    assert re.search(r"\b\d+ passed", out) and not re.search(r"\b\d+ skipped", out), f"{name}: the child did not actually run it:\n{out[-600:]}"
