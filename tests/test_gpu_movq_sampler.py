"""GPU parity: MoVQ decode, VQ indices (bit-exact), the fused sampler loop against the reference trajectory golden,
and the pipelines' public surface.  fp16-storage tolerances are stated per test."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def _load(name):
    return torch.load(os.path.join(GOLD, name + ".pt"), weights_only=False)


def test_movq_decode_golden():
    from kandinsky2.vqgan import MOVQ
    from oracle import movq_oracle as mo, synth
    fx = _load("movq_tiny")
    sd = synth.synth_state_dict(mo.movq_param_spec(fx["dd"], 4, fx["n_embed"]), seed=fx["weight_seed"])
    m = MOVQ(fx["dd"], fx["n_embed"], 4)
    m.load_state_dict(sd)
    m.to("cuda")
    y = m.decode(fx["z"].cuda())
    ref = fx["out"].cuda()
    rel = ((y - ref).norm() / ref.norm()).item()
    err = (y - ref).abs().max().item()
    # fp16 activations through 2 levels of SpatialNorm/conv/attention: 6e-3 relative L2, 4e-2 max-abs on O(1) pixels
    assert rel < 6e-3 and err < 4e-2, (rel, err)
    # VQ code indices: integer output, must be bit-exact with the reference's argmin
    idx = m.quantize_indices(fx["z"].cuda())
    assert torch.equal(idx.cpu(), fx["indices"])
    # uint8 tail equals the reference's process_images arithmetic applied to OUR fp32 image
    u8 = m.decode_to_uint8(fx["z"].cuda(), crop_h=14, crop_w=15)
    assert torch.equal(u8, mo.process_images(y)[:, :14, :15])
    # encoder (image -> latent) vs the reference's MOVQ.encode
    ze = m.encode(fx["image"].cuda())
    relz = ((ze - fx["latent"].cuda()).norm() / fx["latent"].cuda().norm()).item()
    assert ze.shape == fx["latent"].shape and relz < 6e-3, relz


def test_movq_decode_mid_vs_oracle():
    """ch=64, 3 levels, attention at the lowest level with T=1024 tokens, against the fp32 oracle on the GPU."""
    from kandinsky2.vqgan import MOVQ
    from oracle import movq_oracle as mo, synth
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    dd = dict(mo.DDCONFIG_2_1, ch=64, ch_mult=(1, 2, 4), resolution=128)
    sd = synth.synth_state_dict(mo.movq_param_spec(dd, 4, 128), seed=9)
    m = MOVQ(dd, 128, 4)
    m.load_state_dict(sd)
    m.to("cuda")
    z = torch.randn(2, 4, 32, 32, generator=torch.Generator().manual_seed(1)).cuda()
    y = m.decode(z)
    with torch.no_grad():
        ref = mo.movq_decode({k: v.cuda() for k, v in sd.items()}, dd, z)
    rel = ((y - ref).norm() / ref.norm()).item()
    assert y.shape == (2, 3, 128, 128) and rel < 8e-3, rel


def test_movq_decode_full_size_vs_oracle():
    """The real decoder (DDCONFIG_2_1: ch 128, mult (1,2,2,4), 4 attention blocks of ONE head of width 512) on a 96x96 latent
    -> 768x768 image, T = 9216 attention tokens (BASELINE configs[1..3] decode geometry), against the fp32 oracle on the GPU;
    also graph replay == eager, a batch of 2 == the two images decoded alone (no cross-image coupling in the batched
    attention GEMMs), and decode_to_uint8 == the reference's process_images arithmetic on our fp32 image."""
    from kandinsky2.vqgan import MOVQ
    from oracle import movq_oracle as mo, synth
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    dd = dict(mo.DDCONFIG_2_1)
    sd = synth.synth_state_dict(mo.movq_param_spec(dd, 4, 16384), seed=10)
    m = MOVQ(dd, 16384, 4)
    m.load_state_dict(sd)
    m.to("cuda")
    z = torch.randn(2, 4, 96, 96, generator=torch.Generator().manual_seed(2)).cuda()
    m.use_cuda_graph = False
    y_eager = m.decode(z)
    m.use_cuda_graph = True
    y = m.decode(z)
    assert torch.equal(y, y_eager) and torch.equal(y, m.decode(z)), "graph replay must be bit-identical to the eager plan"
    assert y.shape == (2, 3, 768, 768)
    sdc = {k: v.cuda() for k, v in sd.items()}
    with torch.no_grad():
        ref = mo.movq_decode(sdc, dd, z[:1])
    rel = ((y[:1] - ref).norm() / ref.norm()).item()
    err = (y[:1] - ref).abs().max().item()
    print(f"MoVQ decode 96x96 -> 768x768: rel L2 {rel:.3e} max abs {err:.3e} (image rms {ref.pow(2).mean().sqrt().item():.3f})")
    assert rel < 8e-3, rel
    y1 = m.decode(z[1:])
    rel1 = ((y1 - y[1:]).norm() / y[1:].norm()).item()
    assert rel1 < 1e-3, rel1   # different tile shapes at batch 1 may change fp32 summation order, nothing more
    # decode_to_uint8 against the reference's process_images arithmetic on the very fp32 image it converted (the plan's static
    # output buffer), and that image against the replay further up, after another plan has run (a race in the epilogue of the
    # fused d = 512 attention once made this later replay drift, DESIGN.md section 4).
    u8 = m.decode_to_uint8(z, crop_h=760, crop_w=768)
    y_now = m._plan("decode", 2, 96, 96).out.clone()
    assert torch.equal(u8, mo.process_images(y_now)[:, :760, :768])
    drift = (y_now - y).abs().max().item()
    print(f"MoVQ decode: max abs difference between the replay above and this one: {drift:.3e}")
    assert drift <= 1e-3, drift   # (an fp16 rounding flip inside the decoder moves an output value by up to ~1e-4)


def test_sampler_trajectory_golden():
    """5 reference p_sampler steps (CFG 4, clamp +-2, dynamic threshold, injected noise) on the tiny UNet."""
    from kandinsky2.model.gaussian_diffusion import create_gaussian_diffusion
    from oracle import synth, unet_oracle as uo
    from tests.test_gpu_unet import _build
    fx = _load("traj_tiny")
    sd = synth.synth_state_dict(uo.unet_param_spec(fx["cfg"]), seed=fx["weight_seed"])
    m = _build(fx["cfg"], sd)
    d = create_gaussian_diffusion(steps=1000, learn_sigma=True, noise_schedule="linear", rescale_timesteps=True,
                                  rescale_learned_sigmas=True, timestep_respacing=str(fx["steps"]), linear_start=0.00085,
                                  linear_end=0.012)
    x_T = fx["x_T"].cuda()
    B = x_T.shape[0]
    kw = {k: v.cuda() for k, v in fx["cond"].items()}
    out = d.p_sample_loop(m, (2 * B, 4, 16, 16), noise=torch.cat([x_T, x_T]), model_kwargs=kw, guidance_scale=fx["guidance"],
                          cond_first=True, clip_denoised=True, step_noise=fx["step_noise"].cuda())[:B]
    ref = fx["out"].cuda()
    err = (out - ref).abs().max().item()
    rel = ((out - ref).norm() / ref.norm()).item()
    # CFG scale 4 amplifies the UNet's fp16 error ~4x per step; 5 steps: 3e-2 max-abs on O(1) latents, 1e-2 relative
    assert err < 3e-2 and rel < 1e-2, (err, rel)


@pytest.mark.parametrize("inpaint", [False, True])
def test_ddpm_v22_loop_vs_restated_diffusers(inpaint):
    """Kandinsky 2.2 decoder loop (create_ddpm_v22 + the fused step, unconditional rows first, +-2 clip, learned-range
    variance from the text half) and its inpainting variant (known region re-noised to the next timestep with the initial
    noise, final blend with the clean latent) against oracle/diffusion_oracle.py: ddpm_v22_loop -- the restatement of
    diffusers' DDPMScheduler.step + KandinskyV22[Inpaint]Pipeline (PARITY UNPINNED: diffusers is not in /root/reference).
    The UNet is the tiny reference-pinned one; 6 steps, guidance 4, injected step noise."""
    from kandinsky2.model.gaussian_diffusion import create_ddpm_v22
    from oracle import diffusion_oracle as do, synth, unet_oracle as uo
    from tests.test_gpu_unet import _build
    cfg = dict(uo.CONFIG_TINY, inpainting=inpaint)
    sd = synth.synth_state_dict(uo.unet_param_spec(cfg), seed=4)
    m = _build(cfg, sd)
    g = torch.Generator().manual_seed(8)
    B, H, W, steps = 2, 16, 16, 6
    x_T = torch.randn(B, 4, H, W, generator=g)
    noise = torch.randn(steps, B, 4, H, W, generator=g)
    kw = dict(full_emb=torch.randn(2 * B, 7, 96, generator=g), pooled_emb=torch.randn(2 * B, 48, generator=g),
              image_emb=torch.randn(2 * B, 48, generator=g))
    extra, okw = {}, {}
    if inpaint:
        init = torch.randn(1, 4, H, W, generator=g)
        mask = (torch.rand(1, 1, H, W, generator=g) > 0.4).float()
        kw["inpaint_image"] = (init * mask).repeat(2 * B, 1, 1, 1)
        kw["inpaint_mask"] = mask.repeat(2 * B, 1, 1, 1)
        extra = dict(inpaint_init=init.repeat(B, 1, 1, 1).cuda(), inpaint_mask=mask.repeat(B, 1, 1, 1).cuda(),
                     inpaint_renoise=True)
        okw = dict(inpaint_init=init, inpaint_mask=mask)
    d = create_ddpm_v22(steps)
    out = d.p_sample_loop(m, (2 * B, 4, H, W), noise=torch.cat([x_T, x_T]).cuda(), model_kwargs={k: v.cuda() for k, v in kw.items()},
                          guidance_scale=4.0, cond_first=False, clip_denoised=False, step_noise=noise.cuda(), **extra)[:B]
    with torch.no_grad():
        ref = do.ddpm_v22_loop(lambda xx, tt: uo.unet_forward(sd, cfg, xx, tt, **kw), x_T, steps, 4.0, noise, **okw)
    err = (out.cpu() - ref).abs().max().item()
    rel = ((out.cpu() - ref).norm() / ref.norm()).item()
    # measured on the B200: rel L2 6e-3, max-abs 8e-2 (guidance 4 x sqrt(1/ac - 1) ~ 5 at the first steps amplifies the UNet's
    # fp16 error; no dynamic-threshold renormalisation on this path, unlike the 2.1 trajectory test)
    assert err < 2e-1 and rel < 1e-2, (err, rel)
    if inpaint:  # the known region of the result IS the clean latent
        keep = mask.bool().expand(B, 4, H, W)
        assert torch.allclose(out.cpu()[keep], init.expand(B, 4, H, W)[keep], atol=1e-6)


def _tiny_overrides():
    return {"model_config": dict(num_channels=64, num_res_blocks=1, model_dim=128, channel_mult="1,2",
                                 attention_resolutions="32"),
            "image_enc_params": dict(params=dict(embed_dim=4, n_embed=64, ddconfig=dict(
                double_z=False, z_channels=4, resolution=256, in_channels=3, out_ch=3, ch=32, ch_mult=[1, 1, 2, 2],
                num_res_blocks=1, attn_resolutions=[32], dropout=0.0)))}


@pytest.mark.parametrize("version", ["2.1", "2.2"])
def test_pipeline_surface(version):
    from kandinsky2 import get_kandinsky2
    pipe = get_kandinsky2("cuda", task_type="text2img", model_version=version, cache_dir="/nonexistent",
                          config_overrides=_tiny_overrides())
    if version == "2.1":
        imgs = pipe.generate_text2img("a red cat", num_steps=4, batch_size=2, guidance_scale=4, h=70, w=100, sampler="p_sampler")
        again = pipe.generate_text2img("a red cat", num_steps=4, batch_size=2, guidance_scale=4, h=70, w=100, sampler="p_sampler")
        mixed = pipe.mix_images(["a cat", "a dog"], [0.3, 0.7], num_steps=3, batch_size=1, h=64, w=64, sampler="p_sampler")
        ddim = pipe.generate_text2img("a red cat", num_steps=10, batch_size=1, h=64, w=64)  # default sampler = ddim_sampler
        assert len(ddim) == 1 and ddim[0].size == (64, 64)
        plms = pipe.generate_text2img("a red cat", num_steps=10, batch_size=1, h=64, w=64, sampler="plms_sampler")
        assert len(plms) == 1 and plms[0].size == (64, 64)
        with pytest.raises(ValueError):
            pipe.generate_text2img("x", num_steps=4, sampler="euler")
    else:
        imgs = pipe.generate_text2img("a red cat", batch_size=2, decoder_steps=4, h=70, w=100)
        again = pipe.generate_text2img("a red cat", batch_size=2, decoder_steps=4, h=70, w=100)
        mixed = pipe.mix_images(["a cat", "a dog"], [0.3, 0.7], batch_size=1, decoder_steps=3, h=64, w=64)
    assert len(imgs) == 2 and len(mixed) == 1
    want = (100, 70) if version == "2.1" else (128, 128)   # 2.1 crops to (h, w); 2.2 rounds up to x64 (kandinsky2_2_model.py:68)
    assert imgs[0].size == want and imgs[0].mode == "RGB"
    assert all(a.tobytes() == b.tobytes() for a, b in zip(imgs, again)), "same prompt + seeds -> identical images"
    assert imgs[0].tobytes() != imgs[1].tobytes()


def test_pipeline_inpainting_21():
    from kandinsky2 import get_kandinsky2
    pipe = get_kandinsky2("cuda", task_type="inpainting", model_version="2.1", cache_dir="/nonexistent",
                          config_overrides=_tiny_overrides())
    lat = torch.randn(1, 4, 8, 8, generator=torch.Generator().manual_seed(0))
    mask = torch.ones(64, 64)
    mask[:, 40:] = 0
    imgs = pipe.generate_inpainting("a hat", lat, mask.numpy(), num_steps=3, batch_size=1, guidance_scale=4, h=64, w=64,
                                    sampler="p_sampler")
    assert len(imgs) == 1 and imgs[0].size == (64, 64)
    # PIL input goes through the MoVQ encoder; default sampler (DDIM)
    imgs2 = pipe.generate_inpainting("a hat", imgs[0], mask.numpy(), num_steps=5, batch_size=1, h=64, w=64)
    assert imgs2[0].size == (64, 64)


def test_pipeline_inpainting_22():
    """Kandinsky2_2.generate_inpainting (kandinsky2_2_model.py:143-173 -> diffusers KandinskyV22InpaintPipeline): surface, determinism,
    and the defining property of the diffusers rule -- the kept region (mask = 1) of the decoded image does not depend on the
    prompt, because its latent is exactly the encoded input."""
    from kandinsky2 import get_kandinsky2
    pipe = get_kandinsky2("cuda", task_type="inpainting", model_version="2.2", cache_dir="/nonexistent",
                          config_overrides=_tiny_overrides())
    lat = torch.randn(1, 4, 8, 8, generator=torch.Generator().manual_seed(0))
    mask = torch.ones(64, 64)
    mask[:, 40:] = 0
    a = pipe.generate_inpainting("a hat", lat, mask.numpy(), batch_size=2, decoder_steps=4, h=64, w=64)
    b = pipe.generate_inpainting("a hat", lat, mask.numpy(), batch_size=2, decoder_steps=4, h=64, w=64)
    c = pipe.generate_inpainting("a dog", lat, mask.numpy(), batch_size=2, decoder_steps=4, h=64, w=64)
    assert len(a) == 2 and a[0].size == (64, 64) and a[0].mode == "RGB"
    assert all(x.tobytes() == y.tobytes() for x, y in zip(a, b))
    assert a[0].tobytes() != c[0].tobytes()
    # PIL input goes through the MoVQ encoder
    d = pipe.generate_inpainting("a hat", a[0], mask.numpy(), batch_size=1, decoder_steps=3, h=64, w=64)
    assert d[0].size == (64, 64)


def test_pipeline_img2img_pil():
    from kandinsky2 import get_kandinsky2
    from PIL import Image
    import numpy as np
    src = Image.fromarray((np.random.default_rng(0).random((70, 90, 3)) * 255).astype("uint8"))
    for version in ("2.1", "2.2"):
        pipe = get_kandinsky2("cuda", task_type="img2img", model_version=version, cache_dir="/nonexistent",
                              config_overrides=_tiny_overrides())
        if version == "2.1":
            out = pipe.generate_img2img("a dog", src, strength=0.6, num_steps=10, batch_size=1, h=64, w=64)
        else:
            out = pipe.generate_img2img("a dog", src, strength=0.5, batch_size=1, decoder_steps=6, h=64, w=64)
        assert len(out) == 1 and out[0].size == (64, 64)


def test_ddim_loop_matches_oracle_rule():
    """DDIM (eta 0) through the fused step kernel vs the oracle's restatement of p_sample_ddim driven by the oracle UNet."""
    from kandinsky2.model.gaussian_diffusion import DDIMSampler, create_gaussian_diffusion
    from oracle import diffusion_oracle as do, synth, unet_oracle as uo
    from tests.test_gpu_unet import _build
    fx = _load("traj_tiny")
    cfg = fx["cfg"]
    sd = synth.synth_state_dict(uo.unet_param_spec(cfg), seed=fx["weight_seed"])
    m = _build(cfg, sd)
    d = create_gaussian_diffusion(steps=1000, learn_sigma=True, noise_schedule="linear", rescale_timesteps=True,
                                  rescale_learned_sigmas=True, timestep_respacing="", linear_start=0.00085, linear_end=0.012)
    x_T = fx["x_T"].cuda()
    B = x_T.shape[0]
    kw = {k: v.cuda() for k, v in fx["cond"].items()}
    S, gscale = 4, 3.0
    out, _ = DDIMSampler(m, d).sample(S, 2 * B, (4, 16, 16), conditioning=kw, x_T=torch.cat([x_T, x_T]), guidance_scale=gscale)
    tt, al, alp = do.ddim_schedule(S)
    sdc = {k: v.cuda() for k, v in sd.items()}
    x = x_T.clone()
    with torch.no_grad():
        for i in range(len(tt))[::-1]:
            mo = uo.unet_forward(sdc, cfg, torch.cat([x, x]), torch.full((2 * B,), float(tt[i]), device="cuda"), **kw)
            eps = mo[B:, :4] + gscale * (mo[:B, :4] - mo[B:, :4])
            x = do.ddim_step(x, eps, float(al[i]), float(alp[i]))
    err = (out[:B] - x).abs().max().item()
    rel = ((out[:B] - x).norm() / x.norm()).item()
    # 4 DDIM steps from t = 751: 1/sqrt(a_t) up to ~6 and guidance 3 amplify the UNet's fp16 error per step
    assert rel < 2e-2 and err < 0.15 * x.abs().max().item(), (err, rel, x.abs().max().item())


def test_plms_loop_matches_oracle_rule():
    """PLMS (samplers.py:571-637: improved-Euler first step with two UNet calls, then Adams-Bashforth 2/3/4 over the CFG
    epsilon history) through k2_plms_step vs the same rule evaluated with the fp32 oracle UNet."""
    from kandinsky2.model.gaussian_diffusion import PLMSSampler, create_gaussian_diffusion
    from oracle import diffusion_oracle as do, synth, unet_oracle as uo
    from tests.test_gpu_unet import _build
    fx = _load("traj_tiny")
    cfg = fx["cfg"]
    sd = synth.synth_state_dict(uo.unet_param_spec(cfg), seed=fx["weight_seed"])
    m = _build(cfg, sd)
    d = create_gaussian_diffusion(steps=1000, learn_sigma=True, noise_schedule="linear", rescale_timesteps=True,
                                  rescale_learned_sigmas=True, timestep_respacing="", linear_start=0.00085, linear_end=0.012)
    x_T = fx["x_T"].cuda()
    B = x_T.shape[0]
    kw = {k: v.cuda() for k, v in fx["cond"].items()}
    S, gscale = 5, 2.0
    out, _ = PLMSSampler(m, d).sample(S, 2 * B, (4, 16, 16), conditioning=kw, x_T=torch.cat([x_T, x_T]), guidance_scale=gscale)
    tt, al, alp = do.ddim_schedule(S)
    sdc = {k: v.cuda() for k, v in sd.items()}

    def eps_at(x, t):
        mo = uo.unet_forward(sdc, cfg, torch.cat([x, x]), torch.full((2 * B,), float(t), device="cuda"), **kw)
        return mo[B:, :4] + gscale * (mo[:B, :4] - mo[B:, :4])

    x, old = x_T.clone(), []
    with torch.no_grad():
        for i in range(len(tt))[::-1]:
            e_t = eps_at(x, tt[i])
            if len(old) == 0:
                e_next = eps_at(do.ddim_step(x, e_t, float(al[i]), float(alp[i])), tt[max(i - 1, 0)])
                ep = (e_t + e_next) / 2
            elif len(old) == 1:
                ep = (3 * e_t - old[-1]) / 2
            elif len(old) == 2:
                ep = (23 * e_t - 16 * old[-1] + 5 * old[-2]) / 12
            else:
                ep = (55 * e_t - 59 * old[-1] + 37 * old[-2] - 9 * old[-3]) / 24
            x = do.ddim_step(x, ep, float(al[i]), float(alp[i]))
            old = (old + [e_t])[-3:]
    rel = ((out[:B] - x).norm() / x.norm()).item()
    assert rel < 3e-2, rel



def test_pipeline_controlnet_22():
    """Kandinsky2_2(task_type="controlnet").generate_controlnet (BASELINE configs[4]): surface, determinism, and the hint
    actually steering the result."""
    from kandinsky2 import get_kandinsky2
    pipe = get_kandinsky2("cuda", task_type="controlnet", model_version="2.2", cache_dir="/nonexistent",
                          config_overrides=_tiny_overrides())
    g = torch.Generator().manual_seed(3)
    hint = torch.rand(1, 3, 64, 64, generator=g)
    a = pipe.generate_controlnet("a red cat", hint, batch_size=2, decoder_steps=3, h=64, w=64)
    b = pipe.generate_controlnet("a red cat", hint, batch_size=2, decoder_steps=3, h=64, w=64)
    c = pipe.generate_controlnet("a red cat", 1.0 - hint, batch_size=2, decoder_steps=3, h=64, w=64)
    assert len(a) == 2 and a[0].size == (64, 64)
    assert all(x.tobytes() == y.tobytes() for x, y in zip(a, b))
    assert a[0].tobytes() != c[0].tobytes()
    with pytest.raises(ValueError):
        get_kandinsky2("cuda", task_type="controlnet", model_version="2.1", cache_dir="/nonexistent")
