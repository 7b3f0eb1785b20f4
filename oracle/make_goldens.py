"""Generate the parity fixtures under tests/golden/ by executing the UNMODIFIED reference
(/root/reference, read-only) in the authoring container.  Test infrastructure; run once:

    python oracle/make_goldens.py [--full]

Each fixture stores the config, the seeds, the inputs and the reference's fp32 output.  Weights are
NOT stored: they are regenerated from (sorted key, shape, seed) by oracle/weights.seeded_state_dict,
identically here (loaded into the reference modules) and on the GPU box (loaded into the B200 modules).
`--full` additionally runs BASELINE config 1 (full VC2 UNet, 1x4x16x40x64, fp32; ~2-3 min of CPU)
and one full-resolution VAE frame.
"""
import argparse
import os
import sys
import time

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = "/root/reference"
sys.path.insert(0, os.path.join(HERE, "shim"))
sys.path.insert(0, REF)
sys.path.insert(0, ROOT)

from oracle.configs import UNET_CONFIGS, VAE_CONFIGS, student_loras, unet_inputs  # noqa: E402
from oracle.weights import seeded_state_dict  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def ref_unet(cfg, seed):
    from lvdm.modules.networks.openaimodel3d import UNetModel
    m = UNetModel(**cfg).eval()
    sd = seeded_state_dict(m.state_dict(), seed)
    m.load_state_dict(sd, strict=True)
    return m


def gen_unet(name, full=False):
    spec = UNET_CONFIGS[name]
    cfg = spec["cfg"]
    t0 = time.time()
    m = ref_unet(cfg, spec["weight_seed"])
    outs = []
    for ts in spec["timesteps"]:
        inp = unet_inputs(spec, ts)
        with torch.no_grad():
            y = m(inp["x"], inp["timesteps"], context=inp["context"], fps=inp["fps"], timestep_cond=inp["timestep_cond"],
                  motion_cond=inp.get("motion_cond"))
        outs.append(y.clone())
        print(f"  {name} t={ts}: out std {y.std():.4f} absmax {y.abs().max():.4f} ({time.time()-t0:.1f}s)")
    torch.save({"name": name, "timesteps": spec["timesteps"], "outputs": outs,
                "n_params": sum(p.numel() for p in m.parameters())}, os.path.join(GOLD, f"unet_{name}.pt"))


def gen_vae(name):
    from lvdm.modules.networks.ae_modules import Decoder
    spec = VAE_CONFIGS[name]
    dd = spec["ddconfig"]
    dec = Decoder(**dd).eval()
    pq = torch.nn.Conv2d(spec["embed_dim"], dd["z_channels"], 1)
    template = {f"decoder.{k}": v for k, v in dec.state_dict().items()}
    template.update({f"post_quant_conv.{k}": v for k, v in pq.state_dict().items()})
    sd = seeded_state_dict(template, spec["weight_seed"])
    dec.load_state_dict({k[len("decoder."):]: v for k, v in sd.items() if k.startswith("decoder.")})
    pq.load_state_dict({k[len("post_quant_conv."):]: v for k, v in sd.items() if k.startswith("post_quant_conv.")})
    g = torch.Generator().manual_seed(spec["input_seed"])
    z = torch.randn(spec["z_shape"], generator=g)
    with torch.no_grad():
        # ddpm3d.py:666-679 decode_first_stage_2DAE semantics, frame by frame
        zz = 1.0 / 0.18215 * z
        frames = [dec(pq(zz[:, :, i])).unsqueeze(2) for i in range(zz.shape[2])]
        out = torch.cat(frames, dim=2)
    print(f"  vae {name}: out std {out.std():.4f} absmax {out.abs().max():.4f}")
    torch.save({"name": name, "z": z, "output": out}, os.path.join(GOLD, f"vae_{name}.pt"))


def gen_vae_enc(name):
    """Encode path (SURVEY §8 a21): reference Encoder + quant_conv + DiagonalGaussianDistribution.sample with a seeded
    noise tensor (the reference draws it on the CPU, distributions.py:38-41), times scale_factor (ddpm3d.py:558-567)."""
    from lvdm.modules.networks.ae_modules import Encoder
    from lvdm.distributions import DiagonalGaussianDistribution
    spec = VAE_CONFIGS[name]
    dd = spec["ddconfig"]
    enc = Encoder(**dd).eval()
    qc = torch.nn.Conv2d(2 * dd["z_channels"], 2 * spec["embed_dim"], 1)
    template = {f"encoder.{k}": v for k, v in enc.state_dict().items()}
    template.update({f"quant_conv.{k}": v for k, v in qc.state_dict().items()})
    sd = seeded_state_dict(template, spec["weight_seed"] + 100)
    enc.load_state_dict({k[len("encoder."):]: v for k, v in sd.items() if k.startswith("encoder.")})
    qc.load_state_dict({k[len("quant_conv."):]: v for k, v in sd.items() if k.startswith("quant_conv.")})
    g = torch.Generator().manual_seed(spec["input_seed"] + 100)
    b, _, t, hz, wz = spec["z_shape"]
    f = 2 ** (len(dd["ch_mult"]) - 1)   # spatial reduction of the encoder
    x = torch.randn((b, 3, t, hz * f, wz * f), generator=g)
    noise = torch.randn((b * t, spec["embed_dim"], hz, wz), generator=g)
    with torch.no_grad():
        frames = x.permute(0, 2, 1, 3, 4).reshape(b * t, 3, hz * f, wz * f)
        post = DiagonalGaussianDistribution(qc(enc(frames)))
        z = 0.18215 * post.sample(noise=noise)
        zm = 0.18215 * post.mode()
        back = lambda v: v.reshape(b, t, *v.shape[1:]).permute(0, 2, 1, 3, 4).contiguous()
    print(f"  vae_enc {name}: z std {z.std():.4f} absmax {z.abs().max():.4f}; moments absmax {post.parameters.abs().max():.3f}")
    torch.save({"name": name, "x": x, "noise": noise, "z_sample": back(z), "z_mode": back(zm)}, os.path.join(GOLD, f"vae_enc_{name}.pt"))


def gen_lora(name="small"):
    """LoRA wire format + merge (SURVEY §8 a23 / (f) rank 2): the reference injects LoRA below the UNetModel
    (utils/lora.py:387-486), the flat [up, down, ...] list is filled with seeded values, collapse_lora (:793-830) merges
    it.  Stored: per target layer its name, the shapes of up / down and a digest (sum, abs-sum) of the merged weight."""
    from utils import lora as rlora
    spec = UNET_CONFIGS[name]
    m = ref_unet(spec["cfg"], spec["weight_seed"])
    rlora.inject_trainable_lora_extended(m, target_replace_module={"UNetModel"}, r=64)
    g = torch.Generator().manual_seed(4242)
    ups_downs = list(rlora.extract_lora_ups_down(m, target_replace_module={"UNetModel"}))
    flat = []
    for up, down in ups_downs:
        up.weight.data = torch.randn(up.weight.shape, generator=g) * 0.05
        down.weight.data = torch.randn(down.weight.shape, generator=g) * 0.05
        flat += [up.weight.data.clone(), down.weight.data.clone()]
    rlora.collapse_lora(m, {"UNetModel"})
    rlora.monkeypatch_remove_lora(m)
    layers = [(n, mod) for n, mod in m.named_modules() if mod.__class__ in (torch.nn.Linear, torch.nn.Conv2d, torch.nn.Conv3d)]
    assert len(layers) * 2 == len(flat)
    rec = [dict(name=n, up=tuple(flat[2 * i].shape), down=tuple(flat[2 * i + 1].shape),
                sum=mod.weight.double().sum().item(), abs=mod.weight.double().abs().sum().item())
           for i, (n, mod) in enumerate(layers)]
    print(f"  lora {name}: {len(layers)} layers, {sum(t.numel() for t in flat)} LoRA parameters")
    torch.save({"name": name, "seed": 4242, "layers": rec}, os.path.join(GOLD, f"lora_{name}.pt"))


def gen_unet_probs():
    """Attention-probability export (SURVEY §8f rank 4): the reference UNet built with record_attn_probs=True keeps
    softmax(q k^T) of the decoder's temporal self-attentions (attention.py:124-126; read by motion_prior_sample.py:40-56)."""
    spec = UNET_CONFIGS["small"]
    m = ref_unet({**spec["cfg"], "record_attn_probs": True}, spec["weight_seed"])
    inp = unet_inputs(spec, 519)
    with torch.no_grad():
        y = m(inp["x"], inp["timesteps"], context=inp["context"], fps=inp["fps"], timestep_cond=inp["timestep_cond"])
    probs = {n: mod.attention_probs.clone() for n, mod in m.named_modules()
             if n.endswith("transformer_blocks.0.attn1") and getattr(mod, "attention_probs", None) is not None}
    print("  recorded:", {k: tuple(v.shape) for k, v in probs.items()})
    torch.save({"timestep": 519, "output": y, "probs": probs}, os.path.join(GOLD, "unet_small_probs.pt"))


LORA_LAYER_CASES = {
    # kind: (ctor kwargs of the reference module, input shape in the reference layout)
    "linear": (dict(in_features=128, out_features=192, bias=True), (3, 100, 128)),
    "conv2d": (dict(in_channels=64, out_channels=128, kernel_size=3, padding=1), (2, 64, 12, 16)),
    "conv3d": (dict(in_channels=64, out_channels=64, kernel_size=(3, 1, 1), padding=(1, 0, 0)), (1, 64, 4, 6, 8)),
}


def gen_lora_layers():
    """Forward + backward of the reference's LoraInjectedLinear / Conv2d / Conv3d (utils/lora.py:19-230), r = 64, dropout 0,
    scale 0.7, seeded weights / input / upstream gradient: y, dx, d lora_up.weight, d lora_down.weight."""
    from utils import lora as rlora
    out = {}
    g = torch.Generator().manual_seed(777)
    for kind, (kw, xs) in LORA_LAYER_CASES.items():
        cls = dict(linear=rlora.LoraInjectedLinear, conv2d=rlora.LoraInjectedConv2d, conv3d=rlora.LoraInjectedConv3d)[kind]
        m = cls(**kw, r=64, dropout_p=0.0, scale=0.7)
        base = m.linear if kind == "linear" else m.conv
        with torch.no_grad():
            for prm in (base.weight, base.bias, m.lora_up.weight, m.lora_down.weight):
                if prm is not None:
                    fan = prm[0].numel() if prm.dim() > 1 else 1
                    prm.copy_(torch.randn(prm.shape, generator=g) * (0.3 if prm.dim() == 1 else 0.8 / fan ** 0.5))
        x = torch.randn(xs, generator=g).requires_grad_(True)
        y = m(x)
        dy = torch.randn(y.shape, generator=g)
        y.backward(dy)
        out[kind] = dict(w=base.weight.detach().clone(), b=base.bias.detach().clone() if base.bias is not None else None,
                         up=m.lora_up.weight.detach().clone(), down=m.lora_down.weight.detach().clone(), x=x.detach().clone(), dy=dy,
                         y=y.detach().clone(), dx=x.grad.clone(), d_up=m.lora_up.weight.grad.clone(), d_down=m.lora_down.weight.grad.clone(),
                         scale=0.7)
        print(f"  lora layer {kind}: y std {y.std():.3f}, dx std {x.grad.std():.3f}, d_up std {m.lora_up.weight.grad.std():.3f}, "
              f"d_down std {m.lora_down.weight.grad.std():.3f}")
    torch.save(out, os.path.join(GOLD, "lora_layers.pt"))


def gen_student_grads(name="small", every=5, x_shape=None, with_bf16=True):
    """The student forward + backward of train_t2v_turbo_v1_lora.py:640-656,1040-1048,1190 on the UNMODIFIED reference: the UNet
    with LoRA injected by the reference's own `inject_trainable_lora_extended` (r = 64, target {"UNetModel"}), seeded LoRA
    weights (both up and down non-zero so every gradient is exercised), eval mode (all dropouts off: deterministic), fp32.
    loss = sum(eps_pred * g) for a seeded g.  Stores the LoRA list (wire order), g, the output and every LoRA gradient."""
    from utils.lora import extract_lora_ups_down, inject_trainable_lora_extended
    spec = dict(UNET_CONFIGS[name])
    if x_shape is not None:
        spec["x_shape"] = x_shape
    m = ref_unet(spec["cfg"], spec["weight_seed"])
    m.requires_grad_(False)
    params, _ = inject_trainable_lora_extended(m, target_replace_module={"UNetModel"}, r=64)
    m.eval()
    ups_downs = list(extract_lora_ups_down(m, target_replace_module={"UNetModel"}))
    shapes = []
    for up, down in ups_downs:
        shapes += [tuple(up.weight.shape), tuple(down.weight.shape)]
    loras = student_loras(shapes)
    with torch.no_grad():
        for i, (up, down) in enumerate(ups_downs):
            up.weight.copy_(loras[2 * i])
            down.weight.copy_(loras[2 * i + 1])
            up.weight.requires_grad_(True)
            down.weight.requires_grad_(True)
    inp = unet_inputs(spec, spec["timesteps"][0])
    y = m(inp["x"], inp["timesteps"], context=inp["context"], fps=inp["fps"], timestep_cond=inp["timestep_cond"])
    d_out = torch.randn(y.shape, generator=torch.Generator().manual_seed(4243))
    (y * d_out).sum().backward()
    grads = []
    for up, down in ups_downs:
        grads += [up.weight.grad.clone(), down.weight.grad.clone()]
    norms = torch.tensor([x.double().norm().item() for x in grads], dtype=torch.float64)
    # yardstick for the tolerance: the reference's OWN bf16 forward + backward (weights, inputs and autograd in bfloat16, the
    # precision the training script's autocast runs the student in) against its fp32 gradients above
    m16 = m.bfloat16()
    m16.dtype = torch.bfloat16      # app.py:143 sets the attribute the reference casts its embeddings to
    for up, down in ups_downs:
        up.weight.grad = None
        down.weight.grad = None
    y16 = m16(inp["x"].bfloat16(), inp["timesteps"], context=inp["context"].bfloat16(), fps=inp["fps"], timestep_cond=inp["timestep_cond"].bfloat16())
    (y16 * d_out.bfloat16()).sum().backward()
    g16 = []
    for up, down in ups_downs:
        g16 += [up.weight.grad.float(), down.weight.grad.float()]
    rel16 = [((a.double() - b.double()).norm() / (b.double().norm() + 1e-30)).item() for a, b in zip(g16, grads)]
    cat16 = ((torch.cat([a.flatten() for a in g16]).double() - torch.cat([b.flatten() for b in grads]).double()).norm()
             / torch.cat([b.flatten() for b in grads]).double().norm()).item()
    ref_bf16 = dict(output_rel=((y16.float() - y.detach()).norm() / y.detach().norm()).item(), grad_rel_median=sorted(rel16)[len(rel16) // 2],
                    grad_rel_worst=max(rel16), grad_rel_concat=cat16,
                    norm_ratio=(min(a.norm().item() / (b.norm().item() + 1e-30) for a, b in zip(g16, grads)),
                                max(a.norm().item() / (b.norm().item() + 1e-30) for a, b in zip(g16, grads))))
    print("  reference bf16 vs its fp32:", ref_bf16)
    # the fixture keeps every norm and, to stay small, the full tensors of a fixed subset of layers (first / last three and
    # every fifth), each as fp16 scaled by its max (5e-4 of the tensor's scale: far below the parity tolerance)
    n_layers = len(grads) // 2
    keep = sorted(set(range(3)) | set(range(n_layers - 3, n_layers)) | set(range(0, n_layers, every)))
    full = {}
    for li in keep:
        for j in (2 * li, 2 * li + 1):
            sc = grads[j].abs().max().item() + 1e-30
            full[j] = (sc, (grads[j] / sc).half())
    print(f"  student grads {name}: {n_layers} LoRA layers, out std {y.std():.4f}, grad norm {norms.pow(2).sum().sqrt():.4f}, "
          f"{len(keep)} layers stored in full")
    torch.save({"name": name, "timestep": spec["timesteps"][0], "x_shape": tuple(spec["x_shape"]), "shapes": shapes, "d_out": d_out,
                "output": y.detach().clone(), "grad_norms": norms, "grads_full": full, "ref_bf16": ref_bf16},
               os.path.join(GOLD, f"student_grads_{name}.pt"))


def distill_inputs(spec, bsz=2):
    """Seeded inputs of the distillation-step fixture (shared with tests/test_student_gpu.py through the saved file)."""
    g = torch.Generator().manual_seed(5151)
    shape = (bsz,) + tuple(spec["x_shape"][1:])
    cd = spec["cfg"]["context_dim"]
    return dict(latents=torch.randn(shape, generator=g) * 0.8, prompt=torch.randn(bsz, spec["ctx_len"], cd, generator=g),
                uncond=torch.randn(bsz, spec["ctx_len"], cd, generator=g) * 0.5, index=torch.tensor([37, 4][:bsz]),
                noise=torch.randn(shape, generator=g), w=torch.tensor([6.5, 13.0][:bsz]))


def gen_distill_step(name="small"):
    """One consistency-distillation step (train_t2v_turbo_v1_lora.py:976-1190 with the reward terms off) composed from the
    UNMODIFIED reference pieces: T2VTurboScheduler.add_noise, the LoRA-injected student, the teacher UNet (the same weights
    without time_cond_proj, as :636-639 loads them), scalings_for_boundary_conditions / get_predicted_original_sample /
    get_predicted_noise / guidance_scale_embedding / huber_loss (utils/common_utils.py) and DDIMSolver.ddim_step — fp32, eval
    mode (dropouts off), fixed random draws.  Stores the loss, the intermediate latents and the LoRA gradients."""
    from lvdm.modules.networks.openaimodel3d import UNetModel
    from ode_solver.ddim_solver import DDIMSolver
    from scheduler.t2v_turbo_scheduler import T2VTurboScheduler
    from utils.common_utils import (append_dims, get_predicted_noise, get_predicted_original_sample, guidance_scale_embedding, huber_loss,
                                    scalings_for_boundary_conditions)
    from utils.lora import extract_lora_ups_down, inject_trainable_lora_extended
    spec = UNET_CONFIGS[name]
    unet = ref_unet(spec["cfg"], spec["weight_seed"])
    tcfg = dict(spec["cfg"])
    tcfg["time_cond_proj_dim"] = None
    teacher = UNetModel(**tcfg).eval()
    teacher.load_state_dict({k: v for k, v in unet.state_dict().items() if not k.startswith("time_cond_proj")}, strict=True)
    teacher.requires_grad_(False)
    unet.requires_grad_(False)
    inject_trainable_lora_extended(unet, target_replace_module={"UNetModel"}, r=64)
    unet.eval()
    ups_downs = list(extract_lora_ups_down(unet, target_replace_module={"UNetModel"}))
    shapes = []
    for up, down in ups_downs:
        shapes += [tuple(up.weight.shape), tuple(down.weight.shape)]
    loras = student_loras(shapes)
    with torch.no_grad():
        for i, (up, down) in enumerate(ups_downs):
            up.weight.copy_(loras[2 * i])
            down.weight.copy_(loras[2 * i + 1])
            up.weight.requires_grad_(True)
            down.weight.requires_grad_(True)
    noise_scheduler = T2VTurboScheduler(linear_start=0.00085, linear_end=0.012)
    alpha_schedule = torch.sqrt(noise_scheduler.alphas_cumprod)
    sigma_schedule = torch.sqrt(1 - noise_scheduler.alphas_cumprod)
    solver = DDIMSolver(noise_scheduler.alphas_cumprod.numpy(), ddim_timesteps=50, use_scale=False)
    inp = distill_inputs(spec)
    latents, index, noise, w = inp["latents"], inp["index"], inp["noise"], inp["w"]
    bsz = latents.shape[0]
    topk, ts_scale, fps = 20, 10.0, 16
    # ---- :976-1021
    start_timesteps = solver.ddim_timesteps[index]
    timesteps = start_timesteps - topk
    timesteps = torch.where(timesteps < 0, torch.zeros_like(timesteps), timesteps)
    c_skip_start, c_out_start = [append_dims(x, latents.ndim) for x in scalings_for_boundary_conditions(start_timesteps, timestep_scaling=ts_scale)]
    c_skip, c_out = [append_dims(x, latents.ndim) for x in scalings_for_boundary_conditions(timesteps, timestep_scaling=ts_scale)]
    noisy_model_input = noise_scheduler.add_noise(latents, noise, start_timesteps)
    w_embedding = guidance_scale_embedding(w, embedding_dim=256)
    wv = w.reshape(bsz, 1, 1, 1, 1)
    context = {"context": inp["prompt"].float(), "fps": fps}
    # ---- :1023-1039
    noise_pred = unet(noisy_model_input, start_timesteps, **context, timestep_cond=w_embedding)
    pred_x_0 = get_predicted_original_sample(noise_pred, start_timesteps, noisy_model_input, "epsilon", alpha_schedule, sigma_schedule)
    model_pred = c_skip_start * noisy_model_input + c_out_start * pred_x_0
    # ---- :1102-1181
    with torch.no_grad():
        cond_teacher_output = teacher(noisy_model_input, start_timesteps, **context)
        cond_pred_x0 = get_predicted_original_sample(cond_teacher_output, start_timesteps, noisy_model_input, "epsilon", alpha_schedule, sigma_schedule)
        cond_pred_noise = get_predicted_noise(cond_teacher_output, start_timesteps, noisy_model_input, "epsilon", alpha_schedule, sigma_schedule)
        uncond_teacher_output = teacher(noisy_model_input, start_timesteps, context=inp["uncond"])
        uncond_pred_x0 = get_predicted_original_sample(uncond_teacher_output, start_timesteps, noisy_model_input, "epsilon", alpha_schedule, sigma_schedule)
        uncond_pred_noise = get_predicted_noise(uncond_teacher_output, start_timesteps, noisy_model_input, "epsilon", alpha_schedule, sigma_schedule)
        pred_x0 = cond_pred_x0 + wv * (cond_pred_x0 - uncond_pred_x0)
        pred_noise = cond_pred_noise + wv * (cond_pred_noise - uncond_pred_noise)
        x_prev = solver.ddim_step(pred_x0, pred_noise, index)
        target_noise_pred = unet(x_prev.float(), timesteps, **context, timestep_cond=w_embedding)
        pred_x_0_t = get_predicted_original_sample(target_noise_pred, timesteps, x_prev, "epsilon", alpha_schedule, sigma_schedule)
        target = c_skip * x_prev + c_out * pred_x_0_t
    distill_loss = huber_loss(model_pred, target, 0.001)
    distill_loss.backward()
    grads = []
    for up, down in ups_downs:
        grads += [up.weight.grad.clone(), down.weight.grad.clone()]
    norms = torch.tensor([x.double().norm().item() for x in grads], dtype=torch.float64)
    n_layers = len(grads) // 2
    keep = sorted(set(range(2)) | set(range(n_layers - 2, n_layers)) | set(range(0, n_layers, 12)))
    full = {}
    for li in keep:
        for j in (2 * li, 2 * li + 1):
            sc = grads[j].abs().max().item() + 1e-30
            full[j] = (sc, (grads[j] / sc).half())
    print(f"  distill step {name}: loss {distill_loss.item():.6f}, start t {start_timesteps.tolist()}, t {timesteps.tolist()}, "
          f"grad norm {norms.pow(2).sum().sqrt():.5f}, x_prev std {x_prev.std():.4f}")
    torch.save({"name": name, "inputs": inp, "shapes": shapes, "loss": distill_loss.detach().clone(), "noisy": noisy_model_input,
                "model_pred": model_pred.detach().clone(), "x_prev": x_prev, "target": target, "start_timesteps": start_timesteps,
                "timesteps": timesteps, "grad_norms": norms, "grads_full": full}, os.path.join(GOLD, f"distill_step_{name}.pt"))


def gen_full_grads(name="small_motion"):
    """The v2 student's forward + backward (train_latent_t2v_turbo_v2.py:1043-1050,1264) on the UNMODIFIED reference with EVERY
    parameter trainable, for a LINEAR loss sum(eps_pred * g) with a seeded g (the distillation loss's sign-like gradient makes any
    bf16 run noise-dominated, see the step fixtures; this one pins the backward itself), eval mode, fp32 — plus the yardstick for
    the tolerance: the reference's OWN bf16 forward + backward against these fp32 gradients."""
    spec = UNET_CONFIGS[name]
    m = ref_unet(spec["cfg"], spec["weight_seed"])
    m.requires_grad_(True)
    inp = unet_inputs(spec, spec["timesteps"][0])
    kw = dict(context=inp["context"], fps=inp["fps"], timestep_cond=inp["timestep_cond"], motion_cond=inp.get("motion_cond"))
    y = m(inp["x"], inp["timesteps"], **kw)
    d_out = torch.randn(y.shape, generator=torch.Generator().manual_seed(4244))
    (y * d_out).sum().backward()
    names = [n for n, _ in m.named_parameters()]
    grads = {n: p.grad.clone() for n, p in m.named_parameters()}
    norms = {n: g.double().norm().item() for n, g in grads.items()}
    m16 = m.bfloat16()
    m16.dtype = torch.bfloat16
    for p in m16.parameters():
        p.grad = None
    kw16 = {k: (v.bfloat16() if torch.is_tensor(v) else v) for k, v in kw.items()}
    y16 = m16(inp["x"].bfloat16(), inp["timesteps"], **kw16)
    (y16 * d_out.bfloat16()).sum().backward()
    g16 = {n: p.grad.float() for n, p in m16.named_parameters()}
    rel = lambda a, b: ((a.double() - b.double()).norm() / (b.double().norm() + 1e-30)).item()      # noqa: E731
    rel16 = {n: rel(g16[n], grads[n]) for n in names}
    cat = lambda d: torch.cat([d[n].flatten() for n in names])                                      # noqa: E731
    ratios = [g16[n].norm().item() / (grads[n].norm().item() + 1e-30) for n in names]
    ref_bf16 = dict(output_rel=rel(y16.float(), y.detach()), grad_rel_median=sorted(rel16.values())[len(names) // 2],
                    grad_rel_worst=max(rel16.values()), grad_rel_worst_name=max(rel16, key=rel16.get), grad_rel_concat=rel(cat(g16), cat(grads)),
                    norm_ratio=(min(ratios), max(ratios)))
    print("  reference bf16 vs its fp32:", ref_bf16)
    keep = [n for i, n in enumerate(names) if (i % 13 == 0 or n.startswith(("motion_cond_proj", "combine_proj", "time_cond_proj", "out.", "input_blocks.0.0")))
            and grads[n].numel() <= 150000]
    full = {}
    for n in keep:
        sc = grads[n].abs().max().item() + 1e-30
        full[n] = (sc, (grads[n] / sc).half())
    print(f"  full grads {name}: {len(names)} parameter tensors, out std {y.std():.4f}, grad norm {sum(v * v for v in norms.values()) ** 0.5:.4f}, "
          f"{len(keep)} tensors stored in full")
    torch.save({"name": name, "timestep": spec["timesteps"][0], "names": names, "d_out": d_out, "output": y.detach().clone(), "grad_norms": norms,
                "grads_full": full, "ref_bf16": ref_bf16}, os.path.join(GOLD, f"full_grads_{name}.pt"))


def gen_motion_score(name="small"):
    """The motion-prior score of the v2 preprocessing (motion_prior_sample.py:40-84) on the UNMODIFIED reference: the teacher UNet built
    with record_attn_probs=True (no time_cond_proj), `get_temp_attn_prob` restated over EVERY recording module (the reference hard-codes
    output_blocks.3-11, which are exactly the recording ones of the VC2 UNet; the small config has fewer output blocks),
    utils.common_utils.compute_temp_loss, torch.autograd.grad w.r.t. the latents — fp32."""
    from utils.common_utils import compute_temp_loss
    spec = UNET_CONFIGS[name]
    cfg = {**spec["cfg"], "time_cond_proj_dim": None, "record_attn_probs": True}
    from lvdm.modules.networks.openaimodel3d import UNetModel
    m = UNetModel(**cfg).eval()
    sd = seeded_state_dict(m.state_dict(), spec["weight_seed"])
    m.load_state_dict(sd, strict=True)
    m.requires_grad_(False)
    g = torch.Generator().manual_seed(7171)
    shape = spec["x_shape"]
    cd = spec["cfg"]["context_dim"]
    latents, example = torch.randn(shape, generator=g), torch.randn(shape, generator=g)
    ctx_inf, ctx_orig = torch.randn(shape[0], spec["ctx_len"], cd, generator=g), torch.randn(shape[0], spec["ctx_len"], cd, generator=g)
    ts = torch.tensor([699])
    temp_loss_scale = 20.0

    def get_temp_attn_prob(unet, latent, ts, context):          # motion_prior_sample.py:40-56
        out = unet(latent, ts, **context)
        probs = {n: mod.attention_probs for n, mod in unet.named_modules()
                 if n.endswith("blocks.0.attn1") and getattr(mod, "record_attn_probs", False)}
        return out, probs
    with torch.no_grad():
        _, probs_example = get_temp_attn_prob(m, example, ts, {"context": ctx_orig, "fps": 16})
        probs_example = {k: v.clone() for k, v in probs_example.items()}
    with torch.set_grad_enabled(True):                           # :73-83
        latents.requires_grad_(True)
        cond_teacher_output, probs = get_temp_attn_prob(m, latents, ts, {"context": ctx_inf, "fps": 16})
        loss = temp_loss_scale * compute_temp_loss(probs, probs_example)
        score = torch.autograd.grad(loss, latents)[0].detach()
    print(f"  motion score {name}: {len(probs)} recording layers {list(probs)}, loss {loss.item():.6f}, score std {score.std():.4e}")
    torch.save({"name": name, "cfg": cfg, "latents": latents.detach(), "example": example, "ctx_inf": ctx_inf, "ctx_orig": ctx_orig, "ts": ts,
                "temp_loss_scale": temp_loss_scale, "layers": list(probs), "loss": loss.detach(), "score": score,
                "cond_teacher_output": cond_teacher_output.detach(), "probs": {k: v.detach().half() for k, v in probs.items()}},
               os.path.join(GOLD, f"motion_score_{name}.pt"))


def gen_preprocess_sample(name="small"):
    """preprocess_scripts/preprocess_with_motion_prior.py:326-401 for one video, composed from the UNMODIFIED reference pieces: the teacher
    UNet (record_attn_probs=True), T2VTurboScheduler.add_noise, DDIMSolver.ddim_reverse_step in the script's reverse_ddim_loop, the
    unconditional forward, get_motion_prior_score restated as in gen_motion_score — fp32; the record as the script pickles it (before
    the fp16 cast)."""
    from lvdm.modules.networks.openaimodel3d import UNetModel
    from ode_solver.ddim_solver import DDIMSolver
    from scheduler.t2v_turbo_scheduler import T2VTurboScheduler
    from utils.common_utils import compute_temp_loss
    spec = UNET_CONFIGS[name]
    cfg = {**spec["cfg"], "time_cond_proj_dim": None, "record_attn_probs": True}
    m = UNetModel(**cfg).eval()
    m.load_state_dict(seeded_state_dict(m.state_dict(), spec["weight_seed"]), strict=True)
    m.requires_grad_(False)
    ns = T2VTurboScheduler(linear_start=0.00085, linear_end=0.012)
    solver = DDIMSolver(ns.alphas_cumprod.numpy(), ddim_timesteps=50, use_scale=False)
    g = torch.Generator().manual_seed(8181)
    shape = spec["x_shape"]
    cd = spec["cfg"]["context_dim"]
    latents, noise = torch.randn(shape, generator=g) * 0.8, torch.randn(shape, generator=g)
    prompt, uncond = torch.randn(1, spec["ctx_len"], cd, generator=g), torch.randn(1, spec["ctx_len"], cd, generator=g) * 0.5
    index = torch.tensor([2])
    temp_loss_scale, fps = 20.0, 16
    context, uncond_context = {"context": prompt, "fps": fps}, {"context": uncond, "fps": fps}

    def probs_of(unet):
        return {n: mod.attention_probs for n, mod in unet.named_modules() if n.endswith("blocks.0.attn1") and getattr(mod, "record_attn_probs", False)}
    with torch.no_grad():
        start_timesteps = solver.ddim_timesteps[index]
        z_ts = ns.add_noise(latents, noise, start_timesteps)
        inter, cur = [], latents
        for i in range(index.item() + 1):                       # reverse_ddim_loop, motion_prior_sample.py:27-37
            ts = solver.ddim_timesteps[torch.full((1,), i, dtype=torch.long)].long()
            cur = solver.ddim_reverse_step(cur, m(cur, ts, **context), ts)
            inter.append(cur)
        z_examples, z_examples_prev = inter[-1], (inter[-2] if index.item() > 0 else latents)
        uncond_teacher_output = m(z_ts, start_timesteps, **uncond_context)
        m(z_examples, start_timesteps, **context)
        probs_example = {k: v.clone() for k, v in probs_of(m).items()}
    with torch.set_grad_enabled(True):
        z = z_ts.clone().requires_grad_(True)
        cond_teacher_output = m(z, start_timesteps, **context)
        loss = temp_loss_scale * compute_temp_loss(probs_of(m), probs_example)
        scores = torch.autograd.grad(loss, z)[0].detach()
    print(f"  preprocess sample {name}: index {index.item()}, t {start_timesteps.tolist()}, loss {loss.item():.5f}, score std {scores.std():.4e}")
    rec = dict(index=index[0], z_t=z_ts[0], cond_teacher_out=cond_teacher_output.detach()[0], uncond_teacher_out=uncond_teacher_output[0],
               score=scores[0], z_example=z_examples[0], z_example_prev=z_examples_prev[0], prompt_emb=prompt[0])
    torch.save({"name": name, "cfg": cfg, "latents": latents, "noise": noise, "prompt": prompt, "uncond": uncond, "temp_loss_scale": temp_loss_scale,
                "record": rec}, os.path.join(GOLD, f"preprocess_sample_{name}.pt"))


def v2_inputs(spec, bsz=2):
    """Seeded batch of the v2 latent dataset (preprocess_with_motion_prior.py:392-401 keys) for the v2-step fixture."""
    g = torch.Generator().manual_seed(6161)
    shape = (bsz,) + tuple(spec["x_shape"][1:])
    cd = spec["cfg"]["context_dim"]
    return dict(index=torch.tensor([171, 63][:bsz]), z_t=torch.randn(shape, generator=g), cond_teacher_out=torch.randn(shape, generator=g),
                uncond_teacher_out=torch.randn(shape, generator=g), score=torch.randn(shape, generator=g) * 2.0,
                use_motion_guide=torch.tensor([True, True][:bsz]), prompt_emb=torch.randn(bsz, spec["ctx_len"], cd, generator=g),
                w=torch.tensor([6.5, 13.0][:bsz]))


def gen_v2_step(name="small_motion"):
    """One full fine-tune step of train_latent_t2v_turbo_v2.py:945-1276 (reward terms off, --use_motion_cond, --use_target_unet)
    composed from the UNMODIFIED reference pieces — UNetModel with EVERY parameter trainable, the parameter grouping of :799-815
    executed on the reference's own module tree, guidance_scale_embedding / scalings_for_boundary_conditions /
    get_predicted_original_sample / get_predicted_noise / extract_into_tensor / huber_loss / update_ema (utils/common_utils.py),
    DDIMSolver.ddim_step, torch.optim.AdamW over the two groups, clip_grad_norm_ — fp32, eval mode (dropouts off), fixed draws.
    Sample 0 has index >= (1 - percentage) * N (motion guidance on), sample 1 below it (off)."""
    import copy

    from lvdm.common import extract_into_tensor
    from lvdm.modules.attention import TemporalTransformer
    from ode_solver.ddim_solver import DDIMSolver
    from scheduler.t2v_turbo_scheduler import T2VTurboScheduler
    from utils.common_utils import (append_dims, get_predicted_noise, get_predicted_original_sample, guidance_scale_embedding, huber_loss,
                                    scalings_for_boundary_conditions, update_ema)
    spec = UNET_CONFIGS[name]
    unet = ref_unet(spec["cfg"], spec["weight_seed"])
    unet.requires_grad_(True)
    target_unet = copy.deepcopy(unet).requires_grad_(False)
    # the EMA network starts from different values than the student here, so that the target branch and update_ema are exercised
    with torch.no_grad():
        gq = torch.Generator().manual_seed(99)
        for p in target_unet.parameters():
            p.mul_(1.0 + 0.02 * torch.randn(p.shape, generator=gq))
    target_sd0 = {k: v.clone() for k, v in target_unet.state_dict().items()}
    # ---- :799-815, verbatim logic on the reference modules
    temporal_params, other_params, temporal_names = [], [], []
    named_modules_dict = dict(unet.named_modules())
    for n, p in unet.named_parameters():
        if n.startswith("init_attn.0"):
            temporal_params.append(p); temporal_names.append(n)
        elif len(n.split(".")) > 2:
            module_name = ".".join(n.split(".")[:3])
            if module_name in named_modules_dict and isinstance(named_modules_dict[module_name], TemporalTransformer):
                temporal_params.append(p); temporal_names.append(n)
            else:
                other_params.append(p)
        else:
            other_params.append(p)
    lr, temporal_lr_scale, wd, ema_decay, max_grad_norm = 1e-5, 3.0, 0.01, 0.95, 1.0
    optimizer = torch.optim.AdamW([{"params": other_params}, {"params": temporal_params, "lr": lr * temporal_lr_scale}], lr=lr,
                                  betas=(0.9, 0.999), weight_decay=wd, eps=1e-8)
    noise_scheduler = T2VTurboScheduler(linear_start=0.00085, linear_end=0.012)
    alpha_schedule = torch.sqrt(noise_scheduler.alphas_cumprod)
    sigma_schedule = torch.sqrt(1 - noise_scheduler.alphas_cumprod)
    n_ddim, topk, ts_scale, fps, motion_gs_arg, percentage = 200, 5, 10.0, 16, 0.05, 0.5
    solver = DDIMSolver(noise_scheduler.alphas_cumprod.numpy(), ddim_timesteps=n_ddim, use_scale=False)
    inp = v2_inputs(spec)
    index, w = inp["index"], inp["w"]
    noisy_model_input, cond_teacher_output, uncond_teacher_output = inp["z_t"], inp["cond_teacher_out"], inp["uncond_teacher_out"]
    score, use_motion_guide = inp["score"], inp["use_motion_guide"]
    bsz = index.shape[0]
    index_reshape = index.reshape(bsz, 1, 1, 1, 1)
    # ---- :985-1039
    start_timesteps = solver.ddim_timesteps[index]
    timesteps = start_timesteps - topk
    timesteps = torch.where(timesteps < 0, torch.zeros_like(timesteps), timesteps)
    c_skip_start, c_out_start = [append_dims(x, noisy_model_input.ndim) for x in scalings_for_boundary_conditions(start_timesteps, timestep_scaling=ts_scale)]
    c_skip, c_out = [append_dims(x, noisy_model_input.ndim) for x in scalings_for_boundary_conditions(timesteps, timestep_scaling=ts_scale)]
    w_embedding = guidance_scale_embedding(w, 256)
    wv = w.reshape(bsz, 1, 1, 1, 1)
    motion_gs = motion_gs_arg * torch.ones((bsz,))
    condition = torch.logical_and(use_motion_guide, index >= (1 - percentage) * n_ddim)
    motion_gs = torch.where(condition, motion_gs, torch.zeros_like(motion_gs))
    motion_gs_embedding = guidance_scale_embedding(motion_gs, 256)
    motion_gs_host = motion_gs.clone()
    motion_gs = motion_gs.reshape(bsz, 1, 1, 1, 1)
    context = {"context": inp["prompt_emb"], "fps": fps}
    # ---- :1043-1060
    noise_pred = unet(noisy_model_input, start_timesteps, **context, timestep_cond=w_embedding, motion_cond=motion_gs_embedding)
    pred_x_0 = get_predicted_original_sample(noise_pred, start_timesteps, noisy_model_input, "epsilon", alpha_schedule, sigma_schedule)
    model_pred = c_skip_start * noisy_model_input + c_out_start * pred_x_0
    # ---- :1168-1256
    with torch.no_grad():
        cond_pred_x0 = get_predicted_original_sample(cond_teacher_output, start_timesteps, noisy_model_input, "epsilon", alpha_schedule, sigma_schedule)
        cond_pred_noise = get_predicted_noise(cond_teacher_output, start_timesteps, noisy_model_input, "epsilon", alpha_schedule, sigma_schedule)
        uncond_pred_x0 = get_predicted_original_sample(uncond_teacher_output, start_timesteps, noisy_model_input, "epsilon", alpha_schedule, sigma_schedule)
        uncond_pred_noise = get_predicted_noise(uncond_teacher_output, start_timesteps, noisy_model_input, "epsilon", alpha_schedule, sigma_schedule)
        pred_x0 = cond_pred_x0 + wv * (cond_pred_x0 - uncond_pred_x0)
        pred_noise = cond_pred_noise + wv * (cond_pred_noise - uncond_pred_noise)
        alphas = extract_into_tensor(alpha_schedule, start_timesteps, score.shape)
        condition5 = torch.logical_and(use_motion_guide.reshape(bsz, 1, 1, 1, 1), index_reshape >= (1 - percentage) * n_ddim)
        alphas = torch.where(condition5, alphas, torch.ones_like(alphas))
        pred_noise -= motion_gs * (1 - alphas) ** (0.5) * score
        x_prev = solver.ddim_step(pred_x0, pred_noise, index)
        out_t = {}
        for tag, net in (("ema", target_unet), ("self", unet)):
            target_noise_pred = net(x_prev.float(), timesteps, **context, timestep_cond=w_embedding, motion_cond=motion_gs_embedding)
            pred_x_0_t = get_predicted_original_sample(target_noise_pred.to(torch.float32), timesteps, x_prev, "epsilon", alpha_schedule, sigma_schedule)
            out_t[tag] = c_skip * x_prev + c_out * pred_x_0_t
    target = out_t["ema"]
    distill_loss = huber_loss(model_pred, target, 0.001)
    loss_self = huber_loss(model_pred.detach(), out_t["self"], 0.001)
    distill_loss.backward()
    names = [n for n, _ in unet.named_parameters()]
    grads = {n: p.grad.clone() for n, p in unet.named_parameters()}
    norms = {n: g.double().norm().item() for n, g in grads.items()}
    total_norm = float(torch.nn.utils.clip_grad_norm_(unet.parameters(), max_grad_norm))
    optimizer.step()
    update_ema(target_unet.parameters(), unet.parameters(), ema_decay)
    # kept in full (fp16 scaled by the max): a fixed subset of gradients; after the step: the same subset of student / EMA parameters
    keep = [n for i, n in enumerate(names) if (i % 17 == 0 or n.startswith(("motion_cond_proj", "combine_proj", "time_cond_proj", "out.2", "input_blocks.0.0")))
            and grads[n].numel() <= 150000]
    full = {}
    for n in keep:
        sc = grads[n].abs().max().item() + 1e-30
        full[n] = (sc, (grads[n] / sc).half())
    sd1 = dict(unet.named_parameters())
    sd_t1 = dict(target_unet.named_parameters())
    sd0 = seeded_state_dict(unet.state_dict(), spec["weight_seed"])
    stepped = {}                                                                         # parameter DELTAS of the AdamW step
    for n in keep:
        d = sd1[n].detach() - sd0[n]
        sc = d.abs().max().item() + 1e-30
        stepped[n] = (sc, (d / sc).half())
    ema_after = {n: sd_t1[n].detach().clone() for n in [k for k in keep if grads[k].numel() <= 70000][:12]}
    print(f"  v2 step {name}: loss {distill_loss.item():.6f} (self-target {loss_self.item():.6f}), start t {start_timesteps.tolist()}, "
          f"t {timesteps.tolist()}, motion_gs {motion_gs_host.tolist()}, grad norm {total_norm:.5f}, {len(temporal_names)} temporal / "
          f"{len(names) - len(temporal_names)} other parameters, {len(keep)} tensors stored in full")
    torch.save({"name": name, "inputs": inp, "hyper": dict(lr=lr, temporal_lr_scale=temporal_lr_scale, weight_decay=wd, ema_decay=ema_decay,
                                                          max_grad_norm=max_grad_norm, n_ddim=n_ddim, topk=topk, motion_gs=motion_gs_arg,
                                                          percentage=percentage, ts_scale=ts_scale),
                "target_perturb_seed": 99, "temporal_names": temporal_names, "names": names,
                "loss": distill_loss.detach().clone(), "loss_self_target": loss_self.detach().clone(),
                "model_pred": model_pred.detach().clone(), "x_prev": x_prev, "target": target, "target_self": out_t["self"],
                "start_timesteps": start_timesteps, "timesteps": timesteps, "motion_gs": motion_gs_host,
                "grad_norms": norms, "total_norm": total_norm, "grads_full": full, "param_delta": stepped, "ema_after": ema_after},
               os.path.join(GOLD, f"v2_step_{name}.pt"))


def gen_distill_tables():
    """Host-side tables / closed forms of the distillation step straight from the reference: DDIMSolver (ode_solver/ddim_solver.py),
    scalings_for_boundary_conditions and guidance_scale_embedding (utils/common_utils.py), and one tensor-level composition of
    the per-sample algebra (:1030-1039, :1108-1181) on random latents in fp64 for the coefficient-folding test."""
    from ode_solver.ddim_solver import DDIMSolver
    from scheduler.t2v_turbo_scheduler import T2VTurboScheduler
    from utils.common_utils import (append_dims, get_predicted_noise, get_predicted_original_sample, guidance_scale_embedding,
                                    scalings_for_boundary_conditions)
    ns = T2VTurboScheduler(linear_start=0.00085, linear_end=0.012)
    solver = DDIMSolver(ns.alphas_cumprod.numpy(), ddim_timesteps=50, use_scale=False)
    ts = torch.tensor([0, 19, 99, 499, 759, 999])
    cs, co = scalings_for_boundary_conditions(ts, timestep_scaling=10.0)
    w = torch.tensor([5.0, 7.5, 14.25])
    out = dict(ddim_timesteps=solver.ddim_timesteps.clone(), ddim_alpha_cumprods=solver.ddim_alpha_cumprods.clone(),
               ddim_alpha_cumprods_prev=solver.ddim_alpha_cumprods_prev.clone(), scal_t=ts, c_skip=cs, c_out=co, w=w,
               w_emb=guidance_scale_embedding(w, embedding_dim=256))
    # tensor-level composition in fp64
    g = torch.Generator().manual_seed(77)
    alpha, sigma = torch.sqrt(ns.alphas_cumprod).double(), torch.sqrt(1 - ns.alphas_cumprod).double()
    solver.ddim_alpha_cumprods_prev = solver.ddim_alpha_cumprods_prev.double()
    index = torch.tensor([49, 7, 0])
    start = solver.ddim_timesteps[index]
    tn = torch.where(start - 20 < 0, torch.zeros_like(start), start - 20)
    lat, noise, e_s, e_c, e_u, e_t = (torch.randn(3, 4, 2, 3, 3, generator=g, dtype=torch.float64) for _ in range(6))
    z = ns.add_noise(lat, noise, start)
    css, cos_ = [append_dims(x.double(), 5) for x in scalings_for_boundary_conditions(start, timestep_scaling=10.0)]
    csn, con = [append_dims(x.double(), 5) for x in scalings_for_boundary_conditions(tn, timestep_scaling=10.0)]
    model_pred = css * z + cos_ * get_predicted_original_sample(e_s, start, z, "epsilon", alpha, sigma)
    wv = w.double().reshape(3, 1, 1, 1, 1)
    cx0, cn = get_predicted_original_sample(e_c, start, z, "epsilon", alpha, sigma), get_predicted_noise(e_c, start, z, "epsilon", alpha, sigma)
    ux0, un = get_predicted_original_sample(e_u, start, z, "epsilon", alpha, sigma), get_predicted_noise(e_u, start, z, "epsilon", alpha, sigma)
    x_prev = solver.ddim_step(cx0 + wv * (cx0 - ux0), cn + wv * (cn - un), index)
    target = csn * x_prev + con * get_predicted_original_sample(e_t, tn, x_prev, "epsilon", alpha, sigma)
    out["compose"] = dict(index=index, w=w, lat=lat, noise=noise, e_s=e_s, e_c=e_c, e_u=e_u, e_t=e_t, z=z, model_pred=model_pred, x_prev=x_prev,
                          target=target, start=start, tn=tn)
    # DDIM inversion step (inverse_ddim.py / motion_prior_sample.py:27-37 -> DDIMSolver.ddim_reverse_step), fp64
    solver.alpha_cumprods = solver.alpha_cumprods.double() if torch.is_tensor(solver.alpha_cumprods) else torch.from_numpy(solver.alpha_cumprods).double()
    rts = torch.tensor([999, 499, 19, 4])
    rx, re = (torch.randn(4, 4, 2, 3, 3, generator=g, dtype=torch.float64) for _ in range(2))
    out["reverse"] = dict(ts=rts, x_prev=rx, eps=re, x_t=solver.ddim_reverse_step(rx, re, rts), step_ratio=int(solver.step_ratio))
    torch.save(out, os.path.join(GOLD, "distill_tables.pt"))
    print("  distill tables: ddim_timesteps", solver.ddim_timesteps[:4].tolist(), "...", solver.ddim_timesteps[-2:].tolist())


def gen_scheduler():
    from scheduler.t2v_turbo_scheduler import T2VTurboScheduler
    s = T2VTurboScheduler(linear_start=0.00085, linear_end=0.012)
    table = {}
    for n, o in [(4, 50), (8, 50), (16, 50), (4, 200), (8, 200), (16, 200), (1, 50)]:
        s.set_timesteps(n, o)
        table[(n, o)] = s.timesteps.clone()
    g = torch.Generator().manual_seed(11)
    x = torch.randn(1, 4, 4, 8, 8, generator=g)
    eps = torch.randn(1, 4, 4, 8, 8, generator=g)
    s.set_timesteps(4, 50)
    steps = []
    for i, t in enumerate(s.timesteps):
        gen = torch.Generator().manual_seed(100 + i)
        noise = torch.randn(x.shape, generator=torch.Generator().manual_seed(100 + i))
        prev, den = s.step(eps, i, t, x, generator=gen, return_dict=False)
        steps.append({"i": i, "t": int(t), "noise": noise, "prev": prev, "den": den})
    # add_noise (:470-495), fp32 and bf16, per-sample timesteps
    an_x, an_n = torch.randn(3, 4, 2, 5, 5, generator=g), torch.randn(3, 4, 2, 5, 5, generator=g)
    an_t = torch.tensor([0, 519, 999])
    add_noise = {"x": an_x, "noise": an_n, "t": an_t, "out_f32": s.add_noise(an_x, an_n, an_t),
                 "out_bf16": s.add_noise(an_x.bfloat16(), an_n.bfloat16(), an_t)}
    # bf16 steps (what the bf16 pipeline executes: every tensor op rounds to bf16)
    steps_bf16 = []
    for i, t in enumerate(s.timesteps):
        # the reference draws its own noise (randn_tensor in the sample dtype from the generator; variance_noise is ignored)
        noise = torch.randn(x.shape, generator=torch.Generator().manual_seed(100 + i), dtype=torch.bfloat16)
        prev, den = s.step(eps.bfloat16(), i, t, x.bfloat16(), generator=torch.Generator().manual_seed(100 + i), return_dict=False)
        steps_bf16.append({"i": i, "t": int(t), "noise": noise, "prev": prev, "den": den})
    torch.save({"alphas_cumprod": s.alphas_cumprod.clone(), "timesteps": table, "x": x, "eps": eps, "steps": steps,
                "add_noise": add_noise, "steps_bf16": steps_bf16,
                "scalings": {t: tuple(float(v) for v in s.get_scalings_for_boundary_condition_discrete(t)) for t in (0, 279, 999)}},
               os.path.join(GOLD, "scheduler.pt"))
    print("  scheduler: alphas_cumprod[0], [999] =", float(s.alphas_cumprod[0]), float(s.alphas_cumprod[999]))


def gen_scheduler_bf16_cuda():
    """The reference scheduler's bf16 steps EXECUTED ON A CUDA DEVICE (run where one is): torch's CUDA kernels keep the 0-dim
    fp32 coefficients in fp32, so these differ from the CPU `steps_bf16` of scheduler.pt by a few ulps and are what the fused
    step kernel reproduces bit for bit.  Needs a copy of the reference (oracle/_ref/ or the source tree) and a GPU."""
    from oracle import ref_loader
    assert ref_loader.enable() is not None, "no copy of the reference"
    from scheduler.t2v_turbo_scheduler import T2VTurboScheduler
    assert torch.cuda.is_available(), "the CUDA arithmetic of the reference needs a GPU"
    g = torch.load(os.path.join(GOLD, "scheduler.pt"))
    s = T2VTurboScheduler(linear_start=0.00085, linear_end=0.012)
    s.set_timesteps(4, 50)
    xb, eb = g["x"].bfloat16().cuda(), g["eps"].bfloat16().cuda()
    steps = []
    for st in g["steps_bf16"]:
        prev, den = s.step(eb, st["i"], s.timesteps[st["i"]], xb, generator=torch.Generator().manual_seed(100 + st["i"]), return_dict=False)
        steps.append({"i": st["i"], "t": int(s.timesteps[st["i"]]), "prev": prev.cpu(), "den": den.cpu()})
    torch.save({"device": torch.cuda.get_device_name(0), "torch": str(torch.__version__), "steps": steps},
               os.path.join(GOLD, "scheduler_bf16_cuda.pt"))
    print("  scheduler bf16 on", torch.cuda.get_device_name(0))


def gen_lora_traversal():
    """(name, weight shape) of every Linear / Conv2d / Conv3d of the reference UNetModel on the `mid` config, in
    named_modules() order: the order utils/lora.py injects LoRA layers in."""
    import json
    from lvdm.modules.networks.openaimodel3d import UNetModel
    cfg = UNET_CONFIGS["mid"]["cfg"]
    m = UNetModel(**cfg)
    rows = [[n, list(mod.weight.shape)] for n, mod in m.named_modules()
            if mod.__class__ in (torch.nn.Linear, torch.nn.Conv2d, torch.nn.Conv3d)]
    with open(os.path.join(GOLD, "lora_traversal_mid.json"), "w") as f:
        f.write('{"config": "mid", "layers": [\n' + ",\n".join(json.dumps(r) for r in rows) + "\n]}\n")
    print(f"  lora traversal: {len(rows)} layers")


def _ref_pipeline(unet_name):
    """The unmodified reference pipeline around a small UNet / VAE (the attributes it touches: pipeline:27-29,144,216)."""
    from pipeline.t2v_turbo_vc2_pipeline import T2VTurboVC2Pipeline
    from scheduler.t2v_turbo_scheduler import T2VTurboScheduler
    from lvdm.modules.networks.ae_modules import Decoder
    uspec, vspec = UNET_CONFIGS[unet_name], VAE_CONFIGS["small"]
    unet = ref_unet(uspec["cfg"], uspec["weight_seed"])
    dd = vspec["ddconfig"]
    dec = Decoder(**dd).eval()
    pq = torch.nn.Conv2d(vspec["embed_dim"], dd["z_channels"], 1)
    template = {f"decoder.{k}": v for k, v in dec.state_dict().items()}
    template.update({f"post_quant_conv.{k}": v for k, v in pq.state_dict().items()})
    sd = seeded_state_dict(template, vspec["weight_seed"])
    dec.load_state_dict({k[len("decoder."):]: v for k, v in sd.items() if k.startswith("decoder.")})
    pq.load_state_dict({k[len("post_quant_conv."):]: v for k, v in sd.items() if k.startswith("post_quant_conv.")})

    class FakeVAE(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.decoder, self.post_quant_conv = dec, pq

        def decode(self, z, **kw):
            return self.decoder(self.post_quant_conv(z))

    class FakeT2V(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.first_stage_model = FakeVAE()
            self.model = torch.nn.Module()
            self.model.diffusion_model = unet
            self.cond_stage_model = torch.nn.Identity()
            self.temporal_length = 4
            self.scale_factor = 0.18215

        def decode_first_stage_2DAE(self, z, **kw):   # ddpm3d.py:666-679
            z = 1.0 / self.scale_factor * z
            return torch.cat([self.first_stage_model.decode(z[:, :, i]).unsqueeze(2) for i in range(z.shape[2])], dim=2)

    pipe = T2VTurboVC2Pipeline(FakeT2V(), T2VTurboScheduler(linear_start=0.00085, linear_end=0.012),
                               {"params": {"unet_config": {"params": uspec["cfg"]}}})
    return pipe, uspec


def _run_pipeline_cases(pipe, prompt_embeds, cases):
    res = {}
    for key, kw in cases.items():
        out = {}
        for otype, name in (("latent", "latent"), ("pt", "video")):
            gen = torch.Generator().manual_seed(1234)
            out[name] = pipe(prompt_embeds=prompt_embeds, height=64, width=64, frames=4, fps=16, guidance_scale=7.5,
                             generator=gen, output_type=otype, **kw)
        res[key] = out
        print(f"  pipeline {key} {kw}: latent std {out['latent'].std():.4f} video std {out['video'].std():.4f}")
    return res


def gen_pipeline():
    """4- and 8-step T2VTurboVC2Pipeline on CPU with the small UNet/VAE through the unmodified reference classes."""
    pipe, uspec = _ref_pipeline("small")
    g = torch.Generator().manual_seed(5)
    prompt_embeds = torch.randn(1, 77, uspec["cfg"]["context_dim"], generator=g)
    res = _run_pipeline_cases(pipe, prompt_embeds, {s: dict(num_inference_steps=s, lcm_origin_steps=50) for s in (4, 8)})
    torch.save({"prompt_embeds": prompt_embeds, "results": res}, os.path.join(GOLD, "pipeline_small.pt"))


def gen_pipeline_v2():
    """BASELINE config 3 (the v2 sampling path): 16 steps, lcm_origin_steps=200 (what app.py / predict.py pass), and the
    motion-conditioned UNet with use_motion_cond=True, motion_gs=0.05, percentage=0.5 (pipeline:191-204: the motion
    embedding switches to the embedding of 0 below t = 500), batch 2.  Each case stores its kwargs."""
    cases_plain = {"s16_o200": dict(num_inference_steps=16, lcm_origin_steps=200),
                   "s4_o200": dict(num_inference_steps=4, lcm_origin_steps=200)}
    pipe, uspec = _ref_pipeline("small")
    g = torch.Generator().manual_seed(6)
    pe = torch.randn(1, 77, uspec["cfg"]["context_dim"], generator=g)
    out = {"plain": {"prompt_embeds": pe, "cases": cases_plain, "results": _run_pipeline_cases(pipe, pe, cases_plain)}}
    cases_motion = {"s16_o200_motion": dict(num_inference_steps=16, lcm_origin_steps=200, use_motion_cond=True, motion_gs=0.05,
                                            percentage=0.5),
                    "s8_o50_motion": dict(num_inference_steps=8, lcm_origin_steps=50, use_motion_cond=True, motion_gs=0.05,
                                          percentage=0.5)}
    pipe, uspec = _ref_pipeline("small_motion")
    pe2 = torch.randn(2, 77, uspec["cfg"]["context_dim"], generator=g)
    out["motion"] = {"prompt_embeds": pe2, "cases": cases_motion, "results": _run_pipeline_cases(pipe, pe2, cases_motion)}
    torch.save(out, os.path.join(GOLD, "pipeline_small_v2.pt"))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--full", action="store_true")
    ap.add_argument("--only", default="")
    a = ap.parse_args()
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(os.cpu_count())
    todo = a.only.split(",") if a.only else ["scheduler", "unet_small", "unet_mid", "vae_small", "vae_enc_small", "lora_small", "pipeline", "unet_small_motion", "pipeline_v2", "lora_layers", "unet_probs", "student_grads", "distill_step", "distill_tables", "v2_step", "full_grads", "motion_score", "preprocess_sample", "student_grads_mid", "lora_traversal"] + (["unet_full", "vae_full", "vae_enc_full", "unet_full_t", "unet_full_b2"] if a.full else [])
    for item in todo:
        print("generating", item)
        if item == "scheduler":
            gen_scheduler()
        elif item == "scheduler_bf16_cuda":    # not in the default list: needs a GPU
            gen_scheduler_bf16_cuda()
        elif item == "lora_traversal":
            gen_lora_traversal()
        elif item.startswith("unet_") and item != "unet_probs":
            gen_unet(item[5:])
        elif item == "lora_layers":
            gen_lora_layers()
        elif item == "student_grads":
            gen_student_grads()
        elif item == "student_grads_mid":      # the full VC2 topology (575 LoRA layers) at 128 base channels, a small latent
            gen_student_grads("mid", every=40, x_shape=(1, 4, 8, 16, 16))
        elif item == "distill_step":
            gen_distill_step()
        elif item == "distill_tables":
            gen_distill_tables()
        elif item == "v2_step":
            gen_v2_step()
        elif item == "full_grads":
            gen_full_grads()
        elif item == "motion_score":
            gen_motion_score()
        elif item == "preprocess_sample":
            gen_preprocess_sample()
        elif item == "unet_probs":
            gen_unet_probs()
        elif item.startswith("lora_"):
            gen_lora(item[5:])
        elif item.startswith("vae_enc_"):
            gen_vae_enc(item[8:])
        elif item.startswith("vae_"):
            gen_vae(item[4:])
        elif item == "pipeline":
            gen_pipeline()
        elif item == "pipeline_v2":
            gen_pipeline_v2()
        elif item == "lora_layers":
            gen_lora_layers()
