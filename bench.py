#!/usr/bin/env python
"""bench.py -- BASELINE.json metric: UNet denoising steps/sec @ 768x768, 4 images (UNet batch 8 under CFG),
Kandinsky-2.2 decoder configuration (1.22 B-parameter UNet, 32 context tokens, guidance 4, DDPM learned-range).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

One "step" = one classifier-free-guidance-doubled UNet forward + guidance combine + scheduler update for the
batch (SURVEY.md 8d).  Own arm: the C-ABI kernels of libk2b200.so replayed as a CUDA graph; one process per
GPU, each rank denoises its own 4 images (weak scaling, the only collective is one NCCL broadcast of the
conditioning embeddings before step 0).  `value` times K steps with the latents resident in HBM; `e2e` times
the same K steps through the module boundary with the latents coming from / returning to pinned host memory
every step.  `--dump-outputs DIR` writes the latents of the last timed step to DIR/latent.npy (float32), so that two
builds run with the same arguments (hence the same seeded weights, embeddings, noise and latents) can be compared output
for output.  `--impl reference` times the reference algorithm's CPU path (the oracle port of the reference
modules; the reference itself is Python and not part of this repository) on the host cores.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "kandinsky-2_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

METRIC = "unet_denoising_steps_per_sec"
UNIT = "steps/s"
UNET_CFG = dict(model_dim=768, image_encoder_in_dim=1280, text_encoder_in_dim1=1024, text_encoder_in_dim2=768,
                num_image_embs=32, pooling_type="from_model", in_channels=4, model_channels=384, out_channels=8,
                num_res_blocks=3, attention_resolutions=(2, 4, 8), channel_mult=(1, 2, 3, 4), use_fp16=True,
                num_heads=1, num_head_channels=64, use_scale_shift_norm=True, resblock_updown=True,
                cond_version="2.2")


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return dict(tflops_burst=d.get("bf16_tflops"), tflops_sustained=d.get("bf16_tflops_sustained"),
                    hbm_gbs=d.get("hbm_gbs"), source="MEASURED_PEAKS.json")
    return dict(tflops_burst=1590.0, tflops_sustained=1400.0, hbm_gbs=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.f = None

    def start(self):
        try:
            self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.f.name)
        if not sm:
            return None
        return dict(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), samples=len(sm), reasons=sorted(reasons))


def dist_setup(n_gpus):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"  # keep stdout to the one JSON line (NCCL prints its version banner there)
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return world, rank, local


def cpu_oracle_sample(images, lat_h, lat_w, threads, reps=1, warm=0, budget_s=200.0):
    """Times the oracle (torch fp32 restatement of the reference modules) on the host: one CFG-doubled UNet
    forward of `images` of the 4 images at full model size.  Returns seconds per forward (list)."""
    from oracle import unet_oracle as uo
    torch.set_num_threads(threads)
    cfg = uo.CONFIG_2_2
    g = torch.Generator().manual_seed(0)
    sd = {}
    for k, shape in uo.unet_param_spec(cfg):  # cheap init: values do not change the arithmetic cost
        t = torch.empty(shape)
        if len(shape) == 1:
            t.fill_(1.0 if k.endswith("weight") else 0.0)
        else:
            fan = 1
            for d in shape[1:]:
                fan *= d
            t.uniform_(-1.0, 1.0, generator=g).mul_((3.0 / fan) ** 0.5)
        sd[k] = t
    N = 2 * images
    x = torch.randn(N, 4, lat_h, lat_w, generator=g)
    t = torch.full((N,), 980.0)
    img = torch.randn(N, cfg["image_encoder_in_dim"], generator=g)
    times = []
    t_begin = time.perf_counter()
    with torch.no_grad():
        for i in range(warm + reps):
            t0 = time.perf_counter()
            uo.unet_forward(sd, cfg, x, t, image_emb=img)
            dt = time.perf_counter() - t0
            if i >= warm:
                times.append(dt)
            if times and time.perf_counter() - t_begin > budget_s:
                break  # keep the whole run within a few minutes (reported as steps_timed)
    return times


def run_reference(args):
    """Reference arm: the reference algorithm's CPU implementation on this box's host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = int(os.environ.get('K2_CPU_THREADS', 0)) or min(os.cpu_count() or 1, 32)
    lat_h, lat_w = args.height // 8, args.width // 8
    # bounded sample: 1 of the 4 images (UNet batch 2 of 8) per step; a full step is 4 such forwards
    times = cpu_oracle_sample(1, lat_h, lat_w, threads, reps=args.steps, warm=args.warmup)
    per_fwd = sum(times) / len(times)
    ms_per_step = per_fwd * args.batch * 1e3
    value = 1e3 / ms_per_step
    sample = (f"EXTRAPOLATED: each timed step = one CFG-doubled fp32 forward of 1 of the {args.batch} images (UNet batch 2 "
              f"of {2 * args.batch}) at {lat_h}x{lat_w}, full 1.22B model, oracle port of the reference modules (the reference "
              f"itself is Python and is not on this box); step time = that forward x{args.batch}")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, 1),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "steps_timed": len(times)}))


def run_torch_gpu(args):
    """Side baseline (SURVEY.md 8d last row): the reference ALGORITHM on this GPU in the reference's own fp16 mode through
    plain PyTorch -- the oracle restatement of the reference modules (oracle/unet_oracle.py, fp16=True: cuDNN convolutions,
    torch.einsum attention with an fp32 softmax, GroupNorm32 in fp32) + the CFG combine and DDPM update in torch.  Same step,
    same geometry, weights of the same architecture; NOT the product and not part of any parity claim."""
    from oracle import unet_oracle as uo
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    dev = torch.device("cuda", 0)
    B, H, W = args.batch, args.height // 8, args.width // 8
    cfg = uo.CONFIG_2_2
    g = torch.Generator(device=dev).manual_seed(0)
    sd = {}
    for k, shape in uo.unet_param_spec(cfg):
        if len(shape) == 1:
            sd[k] = torch.full(shape, 1.0 if k.endswith("weight") else 0.0, device=dev)
        else:
            fan = 1
            for d in shape[1:]:
                fan *= d
            sd[k] = torch.randn(shape, device=dev, generator=g) / fan ** 0.5
    sd = uo.to_reference_fp16(sd)
    x = torch.randn(B, 4, H, W, device=dev, generator=g)
    img = torch.randn(2 * B, 1280, device=dev, generator=g)

    def one_step(n):
        nonlocal x
        t = torch.full((2 * B,), 980.0 - 20 * (n % 49), device=dev)
        out = uo.unet_forward(sd, cfg, torch.cat([x, x]), t, image_emb=img, fp16=True)
        eps, _ = out.split(4, dim=1)
        eu, ec = eps.chunk(2)
        e = eu + 4.0 * (ec - eu)
        x0 = (1.02 * x - 0.2 * e).clamp(-2, 2)
        x = 0.5 * x0 + 0.5 * x + 0.01 * torch.randn_like(x)

    with torch.no_grad():
        for n in range(max(args.warmup, 3)):
            one_step(n)
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for n in range(args.steps):
            one_step(n)
        e.record()
        torch.cuda.synchronize()
    ms = s.elapsed_time(e) / args.steps
    print(json.dumps({
        "impl": "torch_gpu", "metric": METRIC, "value": 1e3 / ms, "unit": UNIT, "n_gpus": 1, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16", "data": "synthetic", "config": workload_config(args, 1),
        "note": "PyTorch-eager fp16 side baseline (cuDNN conv + einsum attention), oracle restatement of the reference modules"}))


def _init_pipe_with_model(pipe, config, dev, model):
    """Kandinsky2_2 around an already-built UNet (the 1.22B synthetic model of the step benchmark)."""
    from kandinsky2.pipelines import SyntheticEmbedder
    from kandinsky2.vqgan import MOVQ
    pipe.config = config
    pipe.device = dev
    pipe.task_type = "text2img"
    pipe.use_fp16 = True
    pipe.model = model
    ie = config["image_enc_params"]
    pipe.scale = ie["scale"]
    pipe.image_encoder = MOVQ(**ie["params"], device=dev, param_dtype=torch.float16).init_synthetic_(1)
    pipe.embedder = SyntheticEmbedder(1280)
    pipe.base_seed = 1234


def workload_config(args, world):
    return {"workload": f"Kandinsky-2.2 text2img {args.height}x{args.width}, batch {args.batch} per GPU, 50-step "
                        f"DDPM schedule, CFG 4 (BASELINE configs[1])",
            "latent": [args.height // 8, args.width // 8], "images_per_gpu": args.batch,
            "unet_batch_per_gpu": 2 * args.batch, "global_images": args.batch * world, "context_tokens": 32,
            "unet_params": 1228661768 + 0, "parallelism": f"dp{world} (replicas, one conditioning broadcast)",
            "l2": "per-step working set (2.5 GB weights + activations) exceeds the 126 MB L2; no explicit flush"}


# BASELINE.json configs other than the metric config, as per-GPU step geometries (name, images per GPU, latent H, W, inpaint)
OTHER_CONFIGS = [
    ("cfg-2p text2img 512x768 (north_star's 4x64x96 latents), batch 4", 4, 64, 96, False),
    ("cfg-3 text2img 1024x1024, batch 16 over 8 GPUs = 2 images per GPU (BASELINE configs[2])", 2, 128, 128, False),
    ("cfg-4 inpainting 768x768, batch 4, 9-channel masked-latent stem (BASELINE configs[3])", 4, 96, 96, True),
    ("cfg-5 ControlNet-depth 768x768, batch 8 over 4 GPUs = 2 images per GPU, 8-channel stem = latent + hint features "
     "(BASELINE configs[4]; the hint stem runs once per generation, outside the step)", 2, 96, 96, "hint"),
]


def build_unet(dev, inpaint=False):
    from kandinsky2.model.unet import InpaintText2ImUNet, Text2ImUNet
    if inpaint == "hint":
        model = Text2ImUNet(**dict(UNET_CFG, in_channels=8), hint_channels=4, device=dev, param_dtype=torch.float16)
    else:
        model = (InpaintText2ImUNet if inpaint else Text2ImUNet)(**UNET_CFG, device=dev, param_dtype=torch.float16)
    model.init_synthetic_(seed=0)
    model.finalize(release_params=True)
    return model


def step_roofline(plan, ms_per_step, n_unet, H, W, peaks, reps=2):
    """Per-kernel-family CUDA-event times of one eager pass of the step's launch plan -> the `roofline` object."""
    from oracle import unet_oracle as uo  # FLOP accounting of the reference graph only (checker-side helper)
    prof = plan.profile(reps=reps)
    total_ms = sum(v["ms"] for v in prof.values())
    conv = prof["conv_gemm"]
    achieved = conv["flops"] / (conv["ms"] * 1e-3) / 1e12
    peak = peaks["tflops_sustained"] or peaks["tflops_burst"]
    step_flops = uo.algorithmic_flops(uo.CONFIG_2_2, n_unet, H, W, 32)
    return {
        "bound": "tensor", "kernel": "conv_gemm_kernel (3x3 / 1x1 / Conv1d implicit GEMM, tcgen05)",
        "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
        "frac_of_burst": achieved / peaks["tflops_burst"] if peaks["tflops_burst"] else None, "traffic": None,
        "peak_source": f"{peaks['source']} bf16_tflops_sustained (kernel timed inside a long step); burst "
                       f"{peaks['tflops_burst']}",
        "flops_note": "algorithmic FLOPs of the REFERENCE graph; the three up-ResBlock convs execute 4/9 of theirs (3x3 over a "
                      "nearest-2x upsampling = four 2x2 phase convolutions, DESIGN.md section 3)",
        "launches_per_step": conv["launches"], "kernel_ms_per_step": conv["ms"],
        "share_of_step": conv["ms"] / total_ms,
        "step_algorithmic_tflop": step_flops / 1e12,
        "step_tflops_achieved": step_flops / (ms_per_step * 1e-3) / 1e12,
        "step_frac_of_peak": step_flops / (ms_per_step * 1e-3) / 1e12 / peak,
        "step_frac_of_burst": step_flops / (ms_per_step * 1e-3) / 1e12 / peaks["tflops_burst"] if peaks["tflops_burst"] else None,
        "per_kind_ms": {k: round(v["ms"], 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])},
        "attention_tflops": prof["attention"]["flops"] / (prof["attention"]["ms"] * 1e-3) / 1e12,
    }


DUMP_LIMIT_BYTES = (64 << 20) - 4096  # 64 MB in all, less room for the .npy header


def dump_latent(out_dir, x, world, rank):
    """--dump-outputs: the latents the timed path returned after its last step, every rank's rows in rank order, as
    out_dir/latent.npy (float32).  Above the size limit a fixed, seeded sample of the flattened elements is written."""
    import numpy as np
    if world > 1:
        import torch.distributed as dist
        parts = [torch.empty_like(x) for _ in range(world)]
        dist.all_gather(parts, x.contiguous())
        x = torch.cat(parts)
    if rank != 0:
        return
    a = x.float().cpu().numpy()
    if a.nbytes > DUMP_LIMIT_BYTES:
        keep = np.random.default_rng(0).choice(a.size, DUMP_LIMIT_BYTES // a.itemsize, replace=False)
        a = a.reshape(-1)[np.sort(keep)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "latent.npy"), a)


def run_k2(args):
    from kandinsky2 import ops
    from kandinsky2.model.gaussian_diffusion import FusedStep, create_ddpm_v22
    world, rank, local = dist_setup(args.gpus)
    ops.set_tuning(4, 0 if os.environ.get("K2_PDL", "1") == "0" else 1)  # programmatic dependent launch of the step's kernels
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    B, H, W = args.batch, args.height // 8, args.width // 8

    model = build_unet(dev, inpaint=args.inpaint)

    # conditioning: rank 0 draws the image embeddings for the whole job, ONE broadcast, each rank keeps its rows
    emb = torch.empty(world, 2 * B, 1280, device=dev)
    if rank == 0:
        emb.copy_(torch.randn(world, 2 * B, 1280, generator=torch.Generator().manual_seed(1234)).to(dev))
    if world > 1:
        import torch.distributed as dist
        dist.broadcast(emb, src=0)
    image_emb = emb[rank].contiguous()

    diffusion = create_ddpm_v22(50)
    coef, ts = diffusion._tables(dev)
    g = torch.Generator(device=dev).manual_seed(1234 + rank)

    def make_step(mdl, b, h, w, emb_rows, inpaint):
        kw, extra = dict(image_emb=emb_rows), {}
        if inpaint == "hint":  # ControlNet-depth: a depth map at image resolution feeds the hint stem once per generation
            kw["hint"] = torch.rand(1, 3, 8 * h, 8 * w, device=dev, generator=g).expand(2 * b, -1, -1, -1).contiguous()
        elif inpaint:  # masked-latent path: the stem sees [x, image*mask, mask]; x0 is blended with the clean latent in the step
            init = torch.randn(1, 4, h, w, device=dev, generator=g)
            mask = (torch.rand(1, 1, h, w, device=dev, generator=g) > 0.5).float()
            kw["inpaint_image"] = (init * mask).repeat(2 * b, 1, 1, 1)
            kw["inpaint_mask"] = mask.repeat(2 * b, 1, 1, 1)
            extra = dict(inpaint_init=init.repeat(b, 1, 1, 1), inpaint_mask=mask.repeat(b, 1, 1, 1))
        return FusedStep(mdl, b, h, w, kw, guidance_scale=4.0, cond_first=False, clip_range=2.0, threshold_mode=0, **extra)

    order = list(range(diffusion.num_timesteps))[::-1]
    oidx = torch.tensor(order, device=dev, dtype=torch.long)

    def schedule(st, b, h, w):
        """The 50-step DDPM schedule + the run's per-step noise staged on the device (what the pipeline's loop does): a step
        is then ONE graph launch (k2_step_begin + UNet + k2_sampler_step + k2_step_end), nothing else."""
        st.set_schedule(ts[oidx], coef[oidx], torch.randn(len(order), b, 4, h, w, device=dev, generator=g))
        xs = st.latent()
        xs.copy_(torch.randn(b, 4, h, w, device=dev, generator=g))
        return xs

    step = make_step(model, B, H, W, image_emb, args.inpaint)
    x = schedule(step, B, H, W)

    def one_step(n):
        step.advance(x)

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for n in range(k):
            fn(n)
        e.record()
        barrier()
        ms = torch.tensor([s.elapsed_time(e)], device=dev)
        if world > 1:
            import torch.distributed as dist
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    # kernels per step, counted by the library during one eager (un-graphed) step
    model.use_cuda_graph = False
    ops.reset_launch_count()
    one_step(0)
    torch.cuda.synchronize()
    launches_per_step = int(ops.launch_count())
    model.use_cuda_graph = True
    x.copy_(torch.randn(B, 4, H, W, device=dev, generator=g))

    for n in range(max(args.warmup, 3)):
        one_step(n)
    sampler = ClockSampler(local)
    sampler.start()
    ms = timed(one_step, args.steps)
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_latent(args.dump_outputs, x, world, rank)  # before the e2e steps below overwrite x from host memory
    ms_per_step = ms / args.steps
    value = world * 1e3 / ms_per_step

    # e2e: same steps through the module boundary with HOST latents (pinned), H2D + D2H every step
    x_host = torch.randn(B, 4, H, W).pin_memory()
    out_host = torch.empty(B, 4, H, W).pin_memory()

    def e2e_step(n):
        x.copy_(x_host, non_blocking=True)
        one_step(n)
        out_host.copy_(x, non_blocking=True)

    for n in range(3):
        e2e_step(n)
    e2e_ms = timed(e2e_step, args.steps) / args.steps
    nbytes = x_host.numel() * 4

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f16", "data": "synthetic (random-init 1.22B UNet, N(0,1) latents/embeddings)",
        "config": workload_config(args, world),
        "e2e": {"value": world * 1e3 / e2e_ms, "unit": UNIT, "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": nbytes,
                "ms_per_step": e2e_ms},
        "gpu_launches": launches_per_step * args.steps,
        "clocks": clocks,
    }

    peaks = measured_peaks()
    if rank == 0 and not args.no_profile:
        if args.detail:
            det = step.plan.profile_detail(reps=3)
            with open(args.detail, "w") as f:
                json.dump([dict(i=i, kind=k, gflop=fl / 1e9, us=ms * 1e3, tflops=(fl / (ms * 1e-3) / 1e12 if ms > 0 else 0))
                           for i, (k, fl, ms) in enumerate(det)], f)
        line["roofline"] = step_roofline(step.plan, ms_per_step, 2 * B, H, W, peaks)
        # DRAM traffic of the dominant kernel comes from an ncu launch list of this same step (it cannot be measured inside
        # an un-profiled run): profiles/conv_traffic_r2.json carries the commit it was measured at
        traffic_file = os.path.join(ROOT, "profiles", "conv_traffic_r2.json")
        if os.path.exists(traffic_file):
            with open(traffic_file) as f:
                tf = json.load(f)
            line["roofline"]["traffic"] = tf["dram_bytes_per_launch"]
            line["roofline"]["traffic_note"] = tf["note"]
            line["roofline"]["traffic_measured_at_commit"] = tf.get("commit")
    if rank == 0 and world == 1 and not args.no_configs:
        # the other BASELINE configs' per-GPU step geometry: steps/s (graph replay, latents resident) + the same roofline object
        cfgs = {}
        for name, b, h, w, inp in OTHER_CONFIGS:
            mdl = model if inp == args.inpaint else build_unet(dev, inpaint=inp)
            emb_c = torch.randn(2 * b, 1280, device=dev, generator=g)
            mdl.del_cache()  # new conditioning (the UNet caches it per generation, like the reference)
            st = make_step(mdl, b, h, w, emb_c, inp)
            xc = schedule(st, b, h, w)

            def stepc(n, st=st, xc=xc):
                st.advance(xc)
            for n in range(3):
                stepc(n)
            ms_c = timed(stepc, 10) / 10
            cfgs[name] = {"steps_per_s": 1e3 / ms_c, "ms_per_step": ms_c, "images_per_gpu": b, "latent": [h, w],
                          "unet_batch": 2 * b}
            if not args.no_profile:
                r = step_roofline(st.plan, ms_c, 2 * b, h, w, peaks, reps=1)
                cfgs[name].update(step_algorithmic_tflop=r["step_algorithmic_tflop"], step_tflops_achieved=r["step_tflops_achieved"],
                                  step_frac_of_peak=r["step_frac_of_peak"], conv_gemm_tflops=r["achieved"],
                                  conv_gemm_frac=r["frac"], per_kind_ms=r["per_kind_ms"])
            del st, xc
            if mdl is not model:
                del mdl
            torch.cuda.empty_cache()
        line["configs"] = cfgs
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = int(os.environ.get('K2_CPU_THREADS', 0)) or min(os.cpu_count() or 1, 32)
        t = cpu_oracle_sample(1, H, W, threads, reps=1, warm=0)[0]
        v = 1.0 / (t * B)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                                "sample": f"EXTRAPOLATED: one CFG-doubled fp32 oracle forward of 1 of the {B} images at "
                                          f"{H}x{W} ({t:.1f} s), step time = that x{B}"}
    if not args.no_images:
        # BASELINE's second figure: images/s of the whole decoder call (50 denoising steps + MoVQ decode + uint8), through
        # the public pipeline API, each rank generating its own `batch` images.
        from kandinsky2.configs import CONFIG_2_2
        from kandinsky2.pipelines import Kandinsky2_2
        del step
        model.del_cache()
        pipe = Kandinsky2_2.__new__(Kandinsky2_2)
        _init_pipe_with_model(pipe, CONFIG_2_2, dev, model)
        calls = []
        for it in range(4):  # call 0 builds the plans / graphs / MoVQ packing; 1..3 are steady state
            barrier()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            s.record()
            imgs = pipe.generate_text2img("bench", batch_size=B * world, decoder_steps=50, decoder_guidance_scale=4,
                                          h=args.height, w=args.width)
            e.record()
            barrier()
            wall_ms = (time.perf_counter() - t0) * 1e3
            ms_img = torch.tensor([s.elapsed_time(e), wall_ms], device=dev)
            if world > 1:
                import torch.distributed as dist
                dist.all_reduce(ms_img, op=dist.ReduceOp.MAX)
            if it > 0:
                calls.append(ms_img.tolist())
        dev_ms = sorted(c[0] for c in calls)
        med = dev_ms[len(dev_ms) // 2]
        line["images"] = {"value": B * world / (med * 1e-3), "unit": "images/s", "decoder_steps": 50,
                          "ms_per_call": med, "ms_per_call_min": dev_ms[0], "ms_per_call_all": [round(c[0], 1) for c in calls],
                          "host_wall_ms_all": [round(c[1], 1) for c in calls], "images_per_rank": len(imgs),
                          "statistic": "median of 3 steady-state calls (CUDA events, max over ranks); call 0 (plan / graph "
                                       "build) excluded",
                          "includes": "latent init, 50 x (UNet + scheduler), MoVQ decode, uint8 + D2H + PIL"}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="k2", choices=["k2", "reference", "torch_gpu"])
    ap.add_argument("--batch", type=int, default=4)
    ap.add_argument("--height", type=int, default=768)
    ap.add_argument("--width", type=int, default=768)
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--detail", default=None, help="write per-launch timings of one eager step to this JSON file")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-images", action="store_true", help="skip the whole-call images/s measurement")
    ap.add_argument("--no-configs", action="store_true", help="skip the other BASELINE configs' step geometries (N=1 only)")
    ap.add_argument("--inpaint", action="store_true", help="main workload = the inpainting UNet (9-channel stem)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the latents of the last timed step to DIR/latent.npy (float32)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "k2":
        ap.error("--dump-outputs writes the outputs of the k2 step (--impl k2)")
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "torch_gpu":
        run_torch_gpu(args)
    else:
        run_k2(args)


if __name__ == "__main__":
    main()
