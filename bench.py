#!/usr/bin/env python
"""bench.py — BASELINE.json headline metric on B200: 4-step T2VTurboVC2Pipeline, one 16-frame 320x512
video per call (BASELINE config[1]: "T2VTurboVC2Pipeline 4-step inference, 16x320x512, bf16, 1xB200").

A "step" is one full pipeline call (4 UNet forwards + 4 scheduler steps + batched VAE decode) on
synthetic inputs (random prompt embeddings, random-init weights of the VC2 architecture).
  value : frames/s, whole job (all ranks), CUDA-event timed, inputs resident in HBM.
  e2e   : same metric through the public pipeline call with HOST buffers — prompt embeddings in pinned
          host memory (H2D each step) and the decoded video copied back to pinned host memory (D2H).
  roofline     : tensor-core roofline of the dominant kernel family (gemm_tc: every Linear / conv),
                 algorithmic FLOPs / CUDA-event time of those launches, measured live in an eager pass.
  cpu_baseline : the unmodified reference UNetModel + Decoder timed on the host cores on a bounded sample of the
                 same config (one full UNet forward + one decoded frame; video = 4 forwards + 16 frames).
`--impl reference` runs only that CPU arm: the UNMODIFIED reference modules from the git-ignored snapshot
oracle/_ref/ (made by oracle/build_ref.py; it travels to the GPU box), full config, or the oracle port if absent.
Multi-GPU (torchrun): replicas only — each rank samples its own videos; no data-path collective.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FRAMES, HEIGHT, WIDTH, STEPS = 16, 320, 512, 4
# videos per pipeline call per GPU.  Measured on B200 (profiles/r02_batch_sweep.json): 156 / 164 / 180 / 189 / 194 / 195
# frames/s at bs 1 / 2 / 4 / 8 / 12 / 16 — the UNet's level-2/3 layers and the ~8 us fixed cost of each of its ~1 000 launches
# amortise over the batch, and under the 1 kW power cap a fuller tensor pipe is the cheaper way to buy frames.  The metric is
# throughput (frames/s per GPU), so the headline runs at the batch where it saturates (activations ~70 GB of the 180 GB);
# `--batch 1` gives the latency configuration.
DEFAULT_BATCH = 16
# BASELINE.md §3 (hooked reference forward): algorithmic FLOPs
UNET_TFLOP, VAE_TFLOP = 12.581, 25.016
PIPE_TFLOP = STEPS * UNET_TFLOP + VAE_TFLOP   # 75.34


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tflops=d["bf16_tflops_sustained"], hbm=d["hbm_gbs"], src="measured (MEASURED_PEAKS.json, sustained)")
    return dict(tflops=1400.0, hbm=6650.0, src="fallback (B200_PROFILING.md)")


def ncu_gemm_traffic():
    """DRAM bytes (read + write) per gemm_tc launch, averaged over the launches of one pipeline step, from the committed
    ncu capture of scripts/profile_step.py (profiles/README.md); None when the summary is absent."""
    p = os.path.join(ROOT, "profiles", "r02_launches_step_summary.json")
    if not os.path.exists(p):
        p = os.path.join(ROOT, "profiles", "r01_launches_step_final_summary.json")
    if not os.path.exists(p):
        return None
    d = json.load(open(p))
    rows = [v for k, v in d.items() if "gemm_tc_kernel" in k]
    n = sum(v["launches"] for v in rows)
    return sum(v["dram_read_bytes"] + v["dram_write_bytes"] for v in rows) / n if n else None


def ncu_traffic_batch():
    """videos per call of the step the ncu capture above was taken on (the per-launch traffic scales with it)"""
    p = os.path.join(ROOT, "profiles", "r02_launches_step_summary.json")
    try:
        return json.load(open(p)).get("_meta", {}).get("batch")
    except OSError:
        return None


class ClockSampler:
    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        if not sm:
            return None
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 6 and r[2 + i].lower().startswith("active") for r in self.rows)]
        return dict(sm_mhz=statistics.median(sm), sm_max_mhz=float(self.rows[0][1]), reasons=reasons, samples=len(sm))


def build_ms_pipeline(device, use_graph=True):
    """BASELINE configs[4]: ModelScope UNet3DConditionModel + diffusers KL-VAE names over the same kernels, random-init weights."""
    import torch
    from t2v_turbo_b200.ms_adapter import DiffusersAutoencoderKL, T2VTurboMSPipeline, UNet3DConditionModel
    from t2v_turbo_b200.scheduler import T2VTurboScheduler
    with torch.device(device):
        unet = UNet3DConditionModel(time_cond_proj_dim=256)
        vae = DiffusersAutoencoderKL()
    g = torch.Generator(device=device).manual_seed(0)
    with torch.no_grad():
        for mod in (unet, vae):
            for name, p in mod.named_parameters():
                if p.dim() >= 2:
                    p.copy_(torch.randn(p.shape, generator=g, device=device) * (0.6 / p[0].numel() ** 0.5))
                elif name.endswith("weight"):
                    p.copy_(1.0 + 0.05 * torch.randn(p.shape, generator=g, device=device))
                else:
                    p.copy_(0.02 * torch.randn(p.shape, generator=g, device=device))
    return T2VTurboMSPipeline(unet.eval().half(), vae.eval().half(), scheduler=T2VTurboScheduler(linear_start=0.00085, linear_end=0.012),
                              use_cuda_graph=use_graph)


def build_pipeline(device, use_graph=True, motion=False):
    import torch
    from t2v_turbo_b200.configs import VC2_UNET, VC2_VAE_DDCONFIG
    if motion:   # BASELINE configs[2]: the v2 checkpoints add the motion-guidance embedding (predict.py:60-77)
        VC2_UNET = {**VC2_UNET, "motion_cond_proj_dim": 256}
    from t2v_turbo_b200.pipeline import LatentVideoModel, T2VTurboVC2Pipeline
    from t2v_turbo_b200.scheduler import T2VTurboScheduler
    from t2v_turbo_b200.unet import UNetModel
    from t2v_turbo_b200.vae import AutoencoderKL
    with torch.device(device):
        unet = UNetModel(**VC2_UNET)
        vae = AutoencoderKL(VC2_VAE_DDCONFIG, 4)
    g = torch.Generator(device=device).manual_seed(0)
    with torch.no_grad():
        for mod in (unet, vae):
            for name, p in mod.named_parameters():
                if p.dim() >= 2:
                    fan_in = p[0].numel()
                    p.copy_(torch.randn(p.shape, generator=g, device=device) * (0.6 / fan_in ** 0.5))
                elif name.endswith("weight"):
                    p.copy_(1.0 + 0.05 * torch.randn(p.shape, generator=g, device=device))
                else:
                    p.copy_(0.02 * torch.randn(p.shape, generator=g, device=device))
    unet.eval()
    vae.eval()
    unet.dtype = torch.bfloat16     # what app.py:143 does for bf16 inference
    t2v = LatentVideoModel(unet, vae, temporal_length=FRAMES)
    pipe = T2VTurboVC2Pipeline(t2v, T2VTurboScheduler(linear_start=0.00085, linear_end=0.012),
                               {"params": {"unet_config": {"params": VC2_UNET}}}, use_cuda_graph=use_graph)
    return pipe


WORKLOAD = "T2VTurboVC2Pipeline 4-step, 16x320x512, VC2 UNet (1.41B) + KL-VAE decode, bs=%d per GPU"


def _fill_random(module, seed=0):
    """Random-init weights of the bench (same recipe as build_pipeline) for a module created on the meta device."""
    import torch
    module.to_empty(device="cpu")
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in module.named_parameters():
            if p.dim() >= 2:
                p.normal_(0, 0.6 / p[0].numel() ** 0.5, generator=g)
            elif name.endswith("weight"):
                p.fill_(1.0)
            else:
                p.zero_()
    return module.eval()


def reference_sample():
    """The UNMODIFIED reference (oracle/_ref snapshot made by oracle/build_ref.py; /root/reference in the authoring
    container) on the host cores, full BASELINE config: one step = ONE `UNetModel.forward` on the full 1x4x16x40x64
    latent + 77x1024 context (naive attention: xformers is not installed, attention.py:128-144) and ONE decoded 320x512
    frame through `Decoder`; a 4-step 16-frame video costs 4 * t_unet + 16 * t_frame (the reference decodes frame by
    frame, ddpm3d.py:671-677).  dtype and thread count are whichever is fastest on this host (probed on the frame
    decode before the timed region).  Returns None when no copy of the reference is available."""
    import torch
    from oracle import ref_loader
    if ref_loader.enable() is None:
        return None
    from t2v_turbo_b200.configs import VC2_UNET, VC2_VAE_DDCONFIG
    from lvdm.modules.networks.openaimodel3d import UNetModel as RefUNet
    from lvdm.modules.networks.ae_modules import Decoder as RefDecoder
    with torch.device("meta"):
        unet, dec = RefUNet(**VC2_UNET), RefDecoder(**VC2_VAE_DDCONFIG)
    unet, dec = _fill_random(unet, 0), _fill_random(dec, 1)
    g = torch.Generator().manual_seed(0)
    z = torch.randn(1, 4, HEIGHT // 8, WIDTH // 8, generator=g)
    ncpu = os.cpu_count() or 1
    forced_t, forced_d = os.environ.get("T2V_REF_THREADS"), os.environ.get("T2V_REF_DTYPE")
    cands_t = [int(forced_t)] if forced_t else sorted({min(ncpu, n) for n in (16, 32, 64, ncpu)})
    cands_d = [dict(f32=torch.float32, bf16=torch.bfloat16)[forced_d]] if forced_d else [torch.float32, torch.bfloat16]
    best, probe = None, {}
    for dt in cands_d:
        dec.to(dt)
        zz = z.to(dt)
        for nt in cands_t:
            torch.set_num_threads(nt)
            with torch.no_grad():
                dec(zz)   # warm (allocator, oneDNN primitive cache)
                t0 = time.perf_counter()
                dec(zz)
                dtm = time.perf_counter() - t0
            probe[f"{str(dt).split('.')[-1]}/{nt}"] = round(dtm, 2)
            if best is None or dtm < best[0]:
                best = (dtm, dt, nt)
    _, dt, nt = best
    torch.set_num_threads(nt)
    unet.to(dt)
    unet.dtype = dt            # what app.py:143 does
    dec.to(dt)
    x = torch.randn(1, 4, FRAMES, HEIGHT // 8, WIDTH // 8, generator=g).to(dt)
    ctx = torch.randn(1, 77, 1024, generator=g).to(dt)
    from oracle.unet_oracle import guidance_scale_embedding
    w = guidance_scale_embedding(torch.tensor([7.5]), 256).to(dt)
    ts = torch.tensor([999])
    zz = z.to(dt)

    def run():
        with torch.no_grad():
            t0 = time.perf_counter()
            unet(x, ts, context=ctx, fps=16, timestep_cond=w)
            t1 = time.perf_counter()
            dec(zz)
            t2 = time.perf_counter()
        return STEPS * (t1 - t0) + FRAMES * (t2 - t1), (t1 - t0, t2 - t1)
    desc = (f"unmodified reference UNetModel.forward (1x4x16x40x64, 77x1024 context, naive attention) + Decoder on one 320x512 "
            f"frame per step, {str(dt).split('.')[-1]}, {nt} threads of {ncpu}; video time = 4*t_unet + 16*t_frame; "
            f"probe (frame decode s per dtype/threads): {probe}")
    return run, "reference", nt, str(dt).split(".")[-1].replace("float32", "f32").replace("bfloat16", "bf16"), desc


def port_sample():
    """Fallback when no copy of the reference travels with the repo: the oracle port of UNetModel.forward (fp32)."""
    import torch
    from t2v_turbo_b200.configs import VC2_UNET, VC2_VAE_DDCONFIG
    from oracle.unet_oracle import unet_forward, guidance_scale_embedding
    from oracle.vae_oracle import decode_first_stage_2dae
    from t2v_turbo_b200.unet import UNetModel
    from t2v_turbo_b200.vae import AutoencoderKL
    nt = min(os.cpu_count() or 1, 16)
    torch.set_num_threads(nt)

    def rand_sd(shapes, seed):
        g = torch.Generator().manual_seed(seed)
        sd = {}
        for k, shp in shapes.items():
            if len(shp) >= 2:
                fan_in = 1
                for v in shp[1:]:
                    fan_in *= v
                sd[k] = torch.empty(shp).normal_(0, 0.6 / fan_in ** 0.5, generator=g)
            else:
                sd[k] = torch.ones(shp) if k.endswith("weight") else torch.zeros(shp)
        return sd
    with torch.device("meta"):
        ushapes = {k: v.shape for k, v in UNetModel(**VC2_UNET).state_dict().items()}
        vshapes = {k: v.shape for k, v in AutoencoderKL(VC2_VAE_DDCONFIG, 4).state_dict().items()}
    usd, vsd = rand_sd(ushapes, 0), rand_sd(vshapes, 1)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(1, 4, FRAMES, HEIGHT // 8, WIDTH // 8, generator=g)
    ctx = torch.randn(1, 77, 1024, generator=g)
    w = guidance_scale_embedding(torch.tensor([7.5]), 256)
    ts = torch.tensor([999])

    def run():
        with torch.no_grad():
            t0 = time.perf_counter()
            unet_forward(usd, VC2_UNET, x, ts, ctx, fps=16, timestep_cond=w)
            t1 = time.perf_counter()
            decode_first_stage_2dae(vsd, VC2_VAE_DDCONFIG, x[:, :, :1])
            t2 = time.perf_counter()
        return STEPS * (t1 - t0) + FRAMES * (t2 - t1), (t1 - t0, t2 - t1)
    desc = (f"oracle PORT (oracle/_ref absent) of UNetModel.forward (full 1x4x16x40x64) + one decoded frame per step, fp32, "
            f"{nt} threads; video time = 4*t_unet + 16*t_frame")
    return run, "port", nt, "f32", desc


def cpu_arm():
    return reference_sample() or port_sample()


def run_reference(args, rank, world):
    """`--impl reference`: the reference's own CPU implementation of the path, on this arm's config / metric / unit.
    Rank 0 alone runs; K timed steps after W warm-ups, each step one bounded sample (see reference_sample)."""
    if rank != 0:
        return
    run, kind, threads, dtype, desc = cpu_arm()
    for _ in range(args.warmup):
        run()
    recs = [run() for _ in range(args.steps)]
    t_video = sum(r[0] for r in recs) / len(recs)
    t_unet = sum(r[1][0] for r in recs) / len(recs)
    t_frame = sum(r[1][1] for r in recs) / len(recs)
    fps = FRAMES / t_video
    line = dict(impl="reference", metric="4-step 16x320x512 frames/sec", value=fps, unit="frames/s", n_gpus=args.gpus,
                steps=args.steps, warmup=args.warmup, ms_per_step=(t_unet + t_frame) * 1e3, higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype=dtype, data="synthetic", config=dict(workload=WORKLOAD % args.batch, videos_per_step=args.batch),
                cpu_baseline=dict(value=fps, unit="frames/s", cores=threads, kind=kind,
                                  sample=desc + f"; measured t_unet {t_unet:.2f} s, t_frame {t_frame:.2f} s per step "
                                                f"(ms_per_step = t_unet + t_frame, the wall time of one step; value = 16 frames / "
                                                f"(4*t_unet + 16*t_frame) = {t_video:.1f} s per video)"),
                e2e=dict(value=fps, unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    _emit(line)


_RESULT_FD = None


def _reserve_stdout():
    """Contract: exactly ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner on
    stdout when NCCL_DEBUG is set), so file descriptor 1 is pointed at stderr for the whole run and the result line is
    written to the saved descriptor at the end."""
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def _emit(line):
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    os.write(_RESULT_FD if _RESULT_FD is not None else 1, data)


DUMP_BYTES = 64 * 10 ** 6      # --dump-outputs: every .npy file together, headers included, stays under this


def snapshot_outputs(arrays, budget=DUMP_BYTES - 64 * 1024):
    """Host copies of the arrays one timed step returned, for --dump-outputs: float64 stays float64 and so do integer
    tensors (exact below 2**53), every other dtype becomes float32.  The arrays are taken smallest first, each whole if it
    fits its even share of what is left of the budget; a larger one is replaced by a fixed sample of k of its flattened
    elements, `np.random.default_rng(0).choice(numel, k, replace=False)` in ascending order, so the same shapes always
    yield the same positions.  Taken right after the timed loop: graph replays write into the same output buffers, so
    later work would overwrite them."""
    import numpy as np
    import torch
    ts = {name: torch.as_tensor(t).detach() for name, t in arrays.items()}
    out, left = {}, budget
    for i, name in enumerate(sorted(ts, key=lambda n: ts[n].numel())):
        t = ts[name]
        dt = torch.float32 if t.is_floating_point() and t.dtype != torch.float64 else torch.float64
        k = left // (len(ts) - i) // dt.itemsize
        if t.numel() > k:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), size=k, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        out[name] = t.to(dt).cpu().numpy()
        left -= out[name].nbytes
    return {name: out[name] for name in arrays}


def write_outputs(directory, arrays):
    """--dump-outputs: DIR/<name>.npy for every array snapshot_outputs() kept."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def run_train_step(args, rank, local_rank, world):
    """`--workload train-step` (BASELINE config 4, SURVEY section 8 a22 + e): one v1 consistency-distillation step per rank on one
    16x320x512 sample (latents 1x4x16x40x64, 77x1024 prompt embeddings): add_noise, the LoRA-injected student forward
    (training mode: LoRA + temporal-conv dropouts), two teacher forwards (conditional / unconditional) + CFG + one DDIM step,
    the gradient-free target forward, the pseudo-Huber loss, the hand-written backward through all 575 LoRA layers and every
    GroupNorm / LayerNorm / attention / GEGLU between them, the bucketed NCCL all-reduce of the 117 142 176-value fp32 gradient
    arena overlapped with that backward, global-norm clipping and ONE fused AdamW launch
    (train_t2v_turbo_v1_lora.py:976-1194 without the reward models; random-init weights, synthetic latents)."""
    import torch
    from t2v_turbo_b200 import dist as t2v_dist, ops
    from t2v_turbo_b200.configs import VC2_UNET
    from t2v_turbo_b200.distill import DistillStep, train_step
    from t2v_turbo_b200.scheduler import T2VTurboScheduler
    from t2v_turbo_b200.train_unet import StudentUNet
    from t2v_turbo_b200.unet import UNetModel
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    t2v_dist.init_replicas("nccl", device)
    torch.manual_seed(1234 + rank)
    with torch.device(device):
        base = UNetModel(**{**VC2_UNET, "time_cond_proj_dim": 256})
        teacher = UNetModel(**VC2_UNET)
    with torch.no_grad():      # zero-initialised output convs would make the gradients vanish: give every parameter a value
        for m in (base, teacher):
            for prm in m.parameters():
                if prm.dim() > 1 and float(prm.abs().max()) == 0.0:
                    prm.normal_(0, 0.02)
    base, teacher = base.eval(), teacher.eval()
    teacher.dtype = torch.bfloat16
    student = StudentUNet(base, r=64, dropout_p=0.1).train()
    with torch.no_grad():
        for i in range(0, len(student.arena.shapes), 2):
            student.arena.param(i).normal_(0, 0.02)
    student.pack()
    red = t2v_dist.ArenaReducer(student.arena.grads, n_buckets=8)
    student.on_grads_final = red.ready
    dstep = DistillStep(student, teacher, T2VTurboScheduler(linear_start=0.00085, linear_end=0.012))
    g = torch.Generator(device=device).manual_seed(99 + rank)
    latents = torch.randn(1, 4, FRAMES, HEIGHT // 8, WIDTH // 8, device=device, generator=g)
    prompt = torch.randn(1, 77, 1024, device=device, generator=g)
    uncond = torch.randn(1, 77, 1024, device=device, generator=g) * 0.5

    use_graph = not args.no_graph
    if use_graph:      # the whole device side of the step as a chain of CUDA graphs cut at the reducer's bucket boundaries
        from t2v_turbo_b200.distill import GraphedDistillStep
        student.on_grads_final = None
        n_a = ops.LAUNCHES
        step = GraphedDistillStep(dstep, latents, prompt, uncond, reducer=red)      # runs the device step twice: warm-up + capture
        launches_per_step = (ops.LAUNCHES - n_a) // 2
        student.graph_refresh()
    else:
        step = dstep

    def one():
        return train_step(step, latents, prompt, uncond, lr=1e-5, reducer=red, world=world)
    for _ in range(max(args.warmup, 2)):
        out = one()
    torch.cuda.synchronize()
    n0 = ops.LAUNCHES
    sampler = ClockSampler(local_rank)
    t2v_dist.barrier(device)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = one()
    e1.record()
    t2v_dist.barrier(device)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:     # what train_step returned for the last timed step
        write_outputs(args.dump_outputs, snapshot_outputs(out))
    ms = e0.elapsed_time(e1)
    launches = ops.LAUNCHES - n0
    finite = bool(torch.isfinite(out["loss"]).all()) and bool(torch.isfinite(student.arena.params).all())
    # GPU time of the phases (each captured as its own CUDA graph and replayed; not part of the timed region)
    z = dstep.scheduler.add_noise(latents, torch.randn_like(latents), torch.tensor([499], device=device))
    zb = z.bfloat16()
    ts = torch.tensor([499], device=device)
    w_emb = torch.zeros(1, 256, device=device)
    d_eps = torch.randn_like(z)
    student.on_grads_final = None

    def graph_ms(fn, reps=3):
        g_ = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g_, capture_error_mode="thread_local"):
            fn()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g_.replay()
        a.record()
        for _ in range(reps):
            g_.replay()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps, g_
    student.arena.zero_grad()
    fwd_ms, g_f = graph_ms(lambda: student(z, ts, context=prompt, fps=16, timestep_cond=w_emb), reps=1)   # (keeps its tapes for the backward)
    bwd_ms, g_b = graph_ms(lambda: student.backward(d_eps), reps=1)
    tea_ms, g_t = graph_ms(lambda: teacher(zb, ts, context=prompt, fps=16))
    phases = dict(student_forward_ms=fwd_ms, student_backward_ms=bwd_ms, teacher_forward_ms=tea_ms)
    del g_f, g_b, g_t
    ar = [torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)]
    ar[0].record()
    for _ in range(5):
        red.ready(0)
        red.finish()
    ar[1].record()
    torch.cuda.synchronize()
    ar_ms = ar[0].elapsed_time(ar[1]) / 5
    ms, ar_ms = t2v_dist.max_over_ranks([ms, ar_ms], device)
    if rank == 0:
        per = ms / args.steps
        _emit(dict(metric="v1 consistency-distillation steps/sec (one 16x320x512 sample per rank; student fwd+bwd, 2 teacher fwd, target fwd, "
                          "all-reduce, AdamW)", value=world * args.steps / (ms * 1e-3), unit="samples/s", n_gpus=world, steps=args.steps,
                   warmup=max(args.warmup, 2), ms_per_step=per, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16",
                   data="synthetic",
                   config=dict(workload="train_t2v_turbo_v1_lora.py:976-1194 without the reward models: VC2 UNet (1.41B) student with 575 LoRA "
                                        "layers (r=64, dropout 0.1) + frozen teacher, bs=1 per rank, fp32 gradient arena 117142176 values, "
                                        "8-bucket NCCL all-reduce overlapped with the backward, fused AdamW", parallelism=f"dp{world}",
                               cuda_graph=use_graph, graph_segments=len(step.segments) if use_graph else 0, finite=finite),
                   gpu_launches=launches if not use_graph else launches_per_step * args.steps, phases=phases,
                   allreduce=dict(bytes=student.arena.grads.numel() * 4, ms_alone=ar_ms, share_of_step=ar_ms / per if world > 1 else 0.0,
                                  gb_per_s=(student.arena.grads.numel() * 4 / (ar_ms * 1e-3) / 1e9) if world > 1 else None, buckets=8),
                   loss=float(out["loss"]), clocks=clocks))


def run_v2_step(args, rank, local_rank, world):
    """`--workload v2-step` (SURVEY section 8 f1; train_latent_t2v_turbo_v2.py:945-1276 without the reward models): one v2 FULL
    fine-tune step per rank on one 16x320x512 sample with stored teacher outputs — motion-conditioned student forward (training
    mode), motion-prior guidance + DDIM step, the EMA network's target forward, pseudo-Huber loss, the hand-written backward with
    weight / bias / norm-affine gradients for all 1.41 B parameters, the bucketed NCCL all-reduce of the 5.65 GB fp32 gradient
    arena overlapped with that backward, global-norm clip, fused AdamW over the two lr groups (33 launches), operand refresh (and, with
    --no-graph, the EMA target + its update).  Default: the self-target step as a chain of CUDA graphs; --no-graph: eager + EMA target.
    NOT part of the default bench and — the round's GPU budget having run out first — this WORKLOAD has never been executed
    (the step it times has: tests/test_zz_full_train_gpu.py on a small UNet): the line is unmeasured until someone runs it."""
    import torch
    from t2v_turbo_b200 import dist as t2v_dist, ops
    from t2v_turbo_b200.configs import VC2_UNET
    from t2v_turbo_b200.distill_v2 import V2Step, attach_ema_target, train_step_v2
    from t2v_turbo_b200.full_train import FullUNet
    from t2v_turbo_b200.scheduler import T2VTurboScheduler
    from t2v_turbo_b200.unet import UNetModel
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    t2v_dist.init_replicas("nccl", device)
    torch.manual_seed(1234)                     # identical initial weights on every rank, like DDP's broadcast
    cfg = {**VC2_UNET, "time_cond_proj_dim": 256, "motion_cond_proj_dim": 256}
    with torch.device(device):
        base, target = UNetModel(**cfg), UNetModel(**cfg)
    with torch.no_grad():
        for prm in base.parameters():
            if prm.dim() > 1 and float(prm.abs().max()) == 0.0:
                prm.normal_(0, 0.02)
    use_graph = not args.no_graph            # graphs: the self-target step (the script's default, --use_target_unet off); --no-graph: eager + EMA target
    student = FullUNet(base.eval(), with_target=not use_graph).train()
    student.pack()
    target = None if use_graph else attach_ema_target(student, target)
    red = t2v_dist.ArenaReducer(student.arena.grads, n_buckets=16)
    step = V2Step(student, T2VTurboScheduler(linear_start=0.00085, linear_end=0.012), target_unet=target)
    g = torch.Generator(device=device).manual_seed(99 + rank)
    shape = (1, 4, FRAMES, HEIGHT // 8, WIDTH // 8)
    batch = dict(index=torch.tensor([150]), use_motion_guide=torch.tensor([True]),
                 prompt_emb=torch.randn(1, 77, 1024, device=device, generator=g),
                 **{k: torch.randn(shape, device=device, generator=g) for k in ("z_t", "cond_teacher_out", "uncond_teacher_out", "score")})

    launches_per_step = None
    if use_graph:
        from t2v_turbo_b200.distill_v2 import GraphedV2Step
        n_a = ops.LAUNCHES
        step = GraphedV2Step(step, batch, reducer=red)       # runs the device step twice: warm-up + capture
        launches_per_step = (ops.LAUNCHES - n_a) // 2
        student.graph_refresh()                              # the per-step operand refresh (~600 layers) as one graph replay

    def one():
        return train_step_v2(step, batch, lr=1e-5, temporal_lr_scale=1.0, ema_decay=0.95, reducer=red, world=world)
    for _ in range(max(args.warmup, 2)):
        out = one()
    torch.cuda.synchronize()
    n0 = ops.LAUNCHES
    sampler = ClockSampler(local_rank)
    t2v_dist.barrier(device)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = one()
    e1.record()
    t2v_dist.barrier(device)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:     # what train_step_v2 returned for the last timed step
        write_outputs(args.dump_outputs, snapshot_outputs(out))
    ms = t2v_dist.max_over_ranks([e0.elapsed_time(e1)], device)[0]
    finite = bool(torch.isfinite(out["loss"]).all()) and bool(torch.isfinite(student.arena.params).all())
    launches = (ops.LAUNCHES - n0) + (launches_per_step * args.steps if use_graph else 0)
    if rank == 0:
        _emit(dict(metric="v2 full fine-tune steps/sec (one 16x320x512 sample per rank; student fwd+bwd over all 1.41B parameters, EMA target "
                          "fwd, all-reduce, AdamW, EMA)", value=world * args.steps / (ms * 1e-3), unit="samples/s", n_gpus=world,
                   steps=args.steps, warmup=max(args.warmup, 2), ms_per_step=ms / args.steps, higher_is_better=True, scaling="weak",
                   vs_baseline=None, dtype="bf16", data="synthetic",
                   config=dict(workload="train_latent_t2v_turbo_v2.py:945-1276 without the reward models: VC2 UNet (1.41B, motion-conditioned), "
                                        "every parameter trains, bs=1 per rank, fp32 gradient arena %d values, 16-bucket NCCL all-reduce overlapped "
                                        "with the backward, two-group fused AdamW" % student.arena.padded, parallelism=f"dp{world}",
                               cuda_graph=use_graph, target="self" if use_graph else "ema", finite=finite),
                   gpu_launches=launches, loss=float(out["loss"]), clocks=clocks))
    t2v_dist.shutdown()


def run_lora_step(args, rank, local_rank, world):
    """`--workload lora-step` (supplementary; BASELINE config 4's data-parallel exchange): per rank, the 567 LoRA-injected
    layers of the VC2 UNet that are on the tensor-core training path (utils/lora.py:19-230, r = 64) run forward and backward
    at the activation geometry of one 16x320x512 sample — base GEMM + LoRA down / up in the forward; dgrad (base and LoRA)
    and the two weight-gradient GEMMs per layer in the backward, written straight into the 117 142 176-value fp32 arena —
    then the bucketed NCCL sum all-reduce of the arena (overlapped with the backward, reverse layer order), global-norm
    clipping and ONE fused AdamW launch.  Layer inputs / upstream gradients are independent random tensors per shape: the
    non-GEMM layers between the LoRA layers (GroupNorm, LayerNorm, attention, GEGLU) have no backward kernels yet, so this
    is the LoRA-layer + exchange + optimizer part of train_t2v_turbo_v1_lora.py:1190-1194, not the whole student step."""
    import math
    import torch
    from t2v_turbo_b200 import dist as t2v_dist, lora_train as lt, ops
    from t2v_turbo_b200.configs import VC2_UNET
    from t2v_turbo_b200.unet import UNetModel
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    t2v_dist.init_replicas("nccl", device)
    with torch.device("meta"):
        unet = UNetModel(**VC2_UNET)
    work = lt.unet_lora_workload(unet)
    arena = lt.arena_for_unet(unet, device, r=64)
    gen = torch.Generator(device=device).manual_seed(7 + rank)
    layers, acts, flops = [], {}, 0
    from t2v_turbo_b200.lora import lora_target_layers
    mods = dict(lora_target_layers(unet))
    for i, (name, kind, pts, cin, cout) in enumerate(work):
        if kind == "skip":
            continue
        m = mods[name]
        wshape = tuple(m.weight.shape)
        w = torch.randn(wshape, device=device, generator=gen) * (0.6 / math.prod(wshape[1:]) ** 0.5)
        arena.param(2 * i).normal_(0, 0.02, generator=gen)             # lora_up (non-zero so that every GEMM does real work)
        arena.param(2 * i + 1).normal_(0, 1.0 / 64, generator=gen)     # lora_down ~ N(0, 1/r)
        pk = lt._PackedLora(kind, w, None, arena.param(2 * i), arena.param(2 * i + 1), 1.0)
        del w
        for key, ch in (("x", cin), ("dy", cout)):
            if (key, pts, ch) not in acts:
                acts[(key, pts, ch)] = torch.randn(*pts, ch, device=device, generator=gen).to(torch.bfloat16)
        taps = dict(linear=1, conv2d=9, conv3d=3)[kind]
        mm = math.prod(pts)
        flops += 2 * mm * (2 * taps * cin * cout + 2 * (taps * cin * 64 + 64 * cout) + taps * cin * 64 + cout * 64)
        layers.append((i, pk, acts[("x", pts, cin)], acts[("dy", pts, cout)]))
    red = t2v_dist.ArenaReducer(arena.grads, n_buckets=8)
    saved = [None] * len(layers)

    def forward_all():
        for k, (i, pk, x, dy) in enumerate(layers):                     # arena order
            _, saved[k], _, _ = lt.lora_forward(pk, x, None, 1.0)

    def backward_range(k_hi, k_lo):                                     # layers k_hi-1 .. k_lo, reverse order
        for k in range(k_hi - 1, k_lo - 1, -1):
            i, pk, x, dy = layers[k]
            lt.lora_backward(pk, x, saved[k], None, 1.0, dy, arena.grad(2 * i), arena.grad(2 * i + 1))

    # The backward is cut where the gradients cross a bucket boundary of the reducer: after segment s every gradient of
    # bucket s is final and its all-reduce is issued while the next segment's GEMMs run.  Each segment (and the forward)
    # is ONE CUDA graph — the step is ~5 700 small launches, host-bound when issued one by one through ctypes.
    cuts, k_hi = [], len(layers)
    for a, _ in reversed(red.bounds):
        k_lo = min(next((k for k, (i, *_r) in enumerate(layers) if arena.offsets[2 * i] >= a), len(layers)), k_hi)
        # after this segment every gradient at or above the first parameter of layer k_lo is final
        cuts.append((k_hi, k_lo, arena.offsets[2 * layers[k_lo][0]] if k_lo < len(layers) else arena.padded))
        k_hi = k_lo
    use_graph = not args.no_graph

    def capture(fn):
        fn()                                                            # warm-up: lazy allocations, kernel attributes
        torch.cuda.synchronize()
        if not use_graph:
            return fn
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            fn()
        return g.replay
    fwd = capture(forward_all)
    segs = [(capture(lambda hi=hi, lo=lo: backward_range(hi, lo)), a) for hi, lo, a in cuts]

    def step():
        fwd()
        arena.zero_grad()
        for run, a in segs:
            run()
            red.ready(a)
        red.finish()
        arena.adamw_step(lr=1e-5, grad_scale=1.0 / world, max_grad_norm=1.0)

    for _ in range(max(args.warmup, 2)):
        step()
    n0 = ops.LAUNCHES
    sampler = ClockSampler(local_rank)
    t2v_dist.barrier(device)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    t2v_dist.barrier(device)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:     # the step returns nothing: its results are the updated LoRA parameters and their gradients
        write_outputs(args.dump_outputs, snapshot_outputs(dict(params=arena.params, grads=arena.grads)))
    ms = e0.elapsed_time(e1)
    launches = ops.LAUNCHES - n0
    # the exchange alone (same buffer, no overlap), for the all-reduce share
    ar = [torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)]
    torch.cuda.synchronize()
    ar[0].record()
    for _ in range(5):
        red.ready(0)
        red.finish()
    ar[1].record()
    torch.cuda.synchronize()
    ar_ms = ar[0].elapsed_time(ar[1]) / 5
    ms, ar_ms = t2v_dist.max_over_ranks([ms, ar_ms], device)
    if rank == 0:
        per = ms / args.steps
        _emit(dict(metric="LoRA-layer forward+backward + gradient all-reduce + AdamW, steps/sec (one 16x320x512 sample per rank)",
                   value=world * args.steps / (ms * 1e-3), unit="samples/s", n_gpus=world, steps=args.steps, warmup=max(args.warmup, 2),
                   ms_per_step=per, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16", data="synthetic",
                   config=dict(workload="567 LoRA-injected layers of the VC2 UNet (r=64), fwd+bwd at bs=1 per rank, fp32 gradient arena "
                                        "117142176 values, bucketed NCCL all-reduce, fused AdamW", parallelism=f"dp{world}",
                               cuda_graph=use_graph, not_included="backward of GroupNorm / LayerNorm / attention / GEGLU (not built)"),
                   gpu_launches=launches, tflop_per_step=flops / 1e12, tflops=flops / (per * 1e-3) / 1e12,
                   allreduce=dict(bytes=arena.padded * 4, ms_alone=ar_ms, share_of_step=ar_ms / per if world > 1 else 0.0,
                                  gb_per_s=(arena.padded * 4 / (ar_ms * 1e-3) / 1e9) if world > 1 else None, buckets=8),
                   clocks=clocks))
    t2v_dist.shutdown()


def main():
    _reserve_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=DEFAULT_BATCH, help="videos per pipeline call per GPU")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sample-steps", type=int, default=STEPS, help="num_inference_steps of the pipeline workloads (BASELINE configs[2]: 8, 16)")
    ap.add_argument("--motion-cond", action="store_true", help="VC2 pipeline with the v2 motion conditioning (BASELINE configs[2])")
    ap.add_argument("--workload", default="pipeline", choices=["pipeline", "ms-pipeline", "lora-step", "train-step", "v2-step"],
                    help="pipeline = the headline metric; lora-step = the data-parallel LoRA training exchange (supplementary)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (float32 / float64, at most "
                         "64 MB in all: larger outputs as a fixed seeded sample); the inputs depend only on the arguments")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm only times a bounded sample of the workload and returns no outputs")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.workload == "train-step":
        return run_train_step(args, rank, local_rank, world)
    if args.workload == "v2-step":
        return run_v2_step(args, rank, local_rank, world)
    if args.workload == "lora-step":
        run_lora_step(args, rank, local_rank, world)
        return
    args.warmup = max(args.warmup, 3)

    import torch
    from t2v_turbo_b200 import dist as t2v_dist
    from t2v_turbo_b200 import ops
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    t2v_dist.init_replicas("nccl", device)
    ms_model = args.workload == "ms-pipeline"
    n_sample = args.sample_steps
    H, W = (256, 256) if ms_model else (HEIGHT, WIDTH)
    headline = not ms_model and n_sample == STEPS and not args.motion_cond      # the BASELINE configs[1] line
    pipe = build_ms_pipeline(device, use_graph=not args.no_graph) if ms_model else \
        build_pipeline(device, use_graph=not args.no_graph, motion=args.motion_cond)
    gen = torch.Generator(device=device).manual_seed(1234 + rank)
    bs = args.batch
    pe_dev = torch.randn(bs, 77, 1024, device=device, dtype=torch.float16 if ms_model else torch.bfloat16, generator=gen)

    def call(pe):
        if ms_model:
            return pipe(prompt_embeds=pe, height=H, width=W, frames=FRAMES, guidance_scale=7.5, num_inference_steps=n_sample,
                        lcm_origin_steps=50, generator=gen, output_type="pt")
        extra = dict(use_motion_cond=True, motion_gs=0.05, percentage=0.5, lcm_origin_steps=200) if args.motion_cond else \
            dict(lcm_origin_steps=50)
        return pipe(prompt_embeds=pe, height=H, width=W, frames=FRAMES, fps=16, guidance_scale=7.5,
                    num_inference_steps=n_sample, generator=gen, output_type="pt", **extra)

    def barrier():
        t2v_dist.barrier(device)

    # ---------------- device-resident arm
    for _ in range(args.warmup):
        vid = call(pe_dev)
    assert tuple(vid.shape) == (bs, 3, FRAMES, H, W)
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        vid = call(pe_dev)
    e1.record()
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:     # the decoded videos of the last timed call
        write_outputs(args.dump_outputs, snapshot_outputs(dict(video=vid)))
    ms = e0.elapsed_time(e1)
    finite = bool(torch.isfinite(vid.float()).all())

    # ---------------- end-to-end arm: host buffers in, host buffers out
    pe_host = pe_dev.cpu().pin_memory()
    out_host = torch.empty((bs, 3, FRAMES, H, W), dtype=vid.dtype).pin_memory()
    for _ in range(2):
        out_host.copy_(call(pe_host), non_blocking=True)
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(args.steps):
        out_host.copy_(call(pe_host), non_blocking=True)   # H2D inside the pipeline call, D2H of the video here
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)

    ms, ms_e2e = t2v_dist.max_over_ranks([ms, ms_e2e], device)   # the slowest replica defines the job time

    # ---------------- UNet forward alone (graph replay), part of the headline metric triple: at the bench batch and at bs = 1
    def unet_ms(nb):
        lat = torch.randn(nb, 4, FRAMES, HEIGHT // 8, WIDTH // 8, device=device, dtype=torch.bfloat16, generator=gen)
        ts = torch.full((nb,), 999, device=device, dtype=torch.long)
        wemb = pipe.get_w_embedding(torch.tensor([7.5]).repeat(nb), 256).to(device).to(torch.bfloat16)
        pe = pe_dev[:nb].contiguous()
        for _ in range(2):
            pipe._unet_call(lat, ts, pe, wemb, None, 16)
        u0, u1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        u0.record()
        for _ in range(10):
            pipe._unet_call(lat, ts, pe, wemb, None, 16)
        u1.record()
        torch.cuda.synchronize()
        return u0.elapsed_time(u1) / 10
    if ms_model or args.motion_cond:      # the UNet-alone latency belongs to the headline configuration only
        unet_ms_batch = unet_ms_1 = None
    else:
        unet_ms_batch = unet_ms(bs)
        unet_ms_1 = unet_ms(1) if bs > 1 else unet_ms_batch

    # ---------------- launches per step + roofline of the dominant kernel family (eager pass, CUDA events per call)
    pipe.use_cuda_graph = False
    call(pe_dev)
    torch.cuda.synchronize()
    n0 = ops.LAUNCHES
    ops.start_profile()
    call(pe_dev)
    prof = ops.stop_profile()
    launches_per_step = ops.LAUNCHES - n0
    pk = peaks()
    gemm = prof.get("gemm", dict(ms=0.0, flops=0, calls=0))
    tot_ms = sum(v["ms"] for v in prof.values()) or 1.0
    achieved = gemm["flops"] / (gemm["ms"] * 1e-3) / 1e12 if gemm["ms"] > 0 else 0.0
    roofline = dict(bound="tensor", kernel="gemm_tc_kernel (all Linear / Conv2d / Conv3d launches of one pipeline call)",
                    achieved=achieved, peak=pk["tflops"], unit="TFLOP/s", frac=achieved / pk["tflops"], peak_source=pk["src"],
                    traffic=ncu_gemm_traffic(), traffic_unit="DRAM bytes per launch (ncu, avg over one step)", traffic_batch=ncu_traffic_batch(),
                    algorithmic_bytes_per_launch=gemm.get("bytes", 0) / max(1, gemm["calls"]),
                    algorithmic_bytes_note="per launch: input activation once + weights once + output (+ residual), bf16; conv taps re-read the input through L2",
                    launches=gemm["calls"], avg_launch_us=gemm["ms"] * 1e3 / max(1, gemm["calls"]),
                    share_of_step=gemm["ms"] / tot_ms,
                    families={k: dict(calls=v["calls"], ms=round(v["ms"], 3), tflops=round(v["flops"] / max(v["ms"], 1e-9) / 1e9, 1))
                              for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])})

    if rank == 0:
        frames_total = FRAMES * bs * args.steps * world
        value = frames_total / (ms * 1e-3)
        pipe_tflop = None if ms_model else n_sample * UNET_TFLOP + VAE_TFLOP      # SURVEY §8d: 75.34 / 125.67 / 226.32 for 4 / 8 / 16 steps
        if ms_model:
            workload = (f"T2VTurboMSPipeline {n_sample}-step, 16x256x256, ModelScope UNet3DConditionModel + diffusers KL-VAE (fp16 at the "
                        f"boundary, bf16 inside), bs={bs} per GPU")
        elif headline:
            workload = WORKLOAD % bs
        else:
            workload = (f"T2VTurboVC2Pipeline {n_sample}-step, 16x320x512, VC2 UNet (1.41B"
                        + (" + motion_cond_proj, use_motion_cond, motion_gs 0.05, percentage 0.5, lcm_origin_steps 200" if args.motion_cond else "")
                        + f") + KL-VAE decode, bs={bs} per GPU")
        line = dict(metric=f"{n_sample}-step 16x{H}x{W} frames/sec", value=value, unit="frames/s", n_gpus=world, steps=args.steps,
                    warmup=args.warmup, ms_per_step=ms / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype="bf16", data="synthetic",
                    config=dict(workload=workload, videos_per_step=bs,
                                parallelism=f"replicas x{world} (no data-path collective)", cuda_graph=not args.no_graph,
                                l2="working set per step (2.83 GB weights per UNet forward + activations) >> 126 MB L2; no flush needed",
                                batch_note="throughput configuration: bs videos per pipeline call (bs=1 latency numbers: unet_fwd_ms, "
                                           "profiles/r02_batch_sweep.json)",
                                output_finite=finite),
                    clocks=clocks,
                    e2e=dict(value=frames_total / (ms_e2e * 1e-3), unit="frames/s", h2d_bytes_per_step=pe_host.numel() * 2,
                             d2h_bytes_per_step=out_host.numel() * 2),
                    gpu_launches=launches_per_step * args.steps, roofline=roofline)
        if pipe_tflop is not None:
            line["config"]["algorithmic_tflop_per_step"] = pipe_tflop * bs
            line["tensor_frac_of_step"] = pipe_tflop * bs / (ms / args.steps * 1e-3) / pk["tflops"]
        if unet_ms_1 is not None:
            line.update(unet_fwd_ms=unet_ms_1, unet_fwd_ms_per_video_at_batch=unet_ms_batch / bs,
                        unet_fwd_tflops=UNET_TFLOP * bs / (unet_ms_batch * 1e-3))
        if world == 1 and not args.no_cpu_baseline and headline:
            torch.cuda.synchronize()
            run, kind, threads, cdt, desc = cpu_arm()
            tv, (tu, tf) = run()
            line["cpu_baseline"] = dict(value=FRAMES / tv, unit="frames/s", cores=threads, kind=kind, dtype=cdt,
                                        sample=desc + f"; one sample: t_unet {tu:.1f} s, t_frame {tf:.1f} s")
        _emit(line)
    t2v_dist.shutdown()


if __name__ == "__main__":
    main()
