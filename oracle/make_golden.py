"""Writes tests/golden/*.pt by EXECUTING THE REFERENCE (build container only: needs /root/reference).

    python -m oracle.make_golden

Every fixture holds the config, the weight seed (weights are re-synthesised from oracle/synth.py), the
inputs and the reference's outputs in fp32.  The same script asserts that the oracle restatement
(oracle/*_oracle.py) reproduces the reference on each fixture -- this is what pins the oracle.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_shim, synth  # noqa: E402
from oracle import unet_oracle as uo  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def build_ref_unet(cfg):
    with ref_shim.reference_modules() as R:
        m21 = R.load("model.text2im_model2_1")
        cls = m21.InpaintText2ImUNet if cfg.get("inpainting") else m21.Text2ImUNet
        model = cls(model_dim=cfg["model_dim"], image_encoder_in_dim=cfg["image_encoder_in_dim"],
                    text_encoder_in_dim1=cfg["text_encoder_in_dim1"], text_encoder_in_dim2=cfg["text_encoder_in_dim2"],
                    num_image_embs=cfg["num_image_embs"], pooling_type="from_model", in_channels=cfg["in_channels"],
                    model_channels=cfg["model_channels"], out_channels=cfg["out_channels"],
                    num_res_blocks=cfg["num_res_blocks"], attention_resolutions=tuple(cfg["attention_ds"]), dropout=0,
                    channel_mult=cfg["channel_mult"], use_fp16=False, num_heads=1,
                    num_head_channels=cfg["num_head_channels"], num_heads_upsample=-1, use_scale_shift_norm=True,
                    resblock_updown=True, cache_text_emb=True)
    return model.eval()


def unet_inputs(cfg, B, H, W, ntext, seed):
    g = torch.Generator().manual_seed(seed)
    d = dict(x=torch.randn(B, cfg["in_channels"], H, W, generator=g),
             t=torch.tensor([999.0, 500.0, 20.0, 0.0][:B]),
             full_emb=torch.randn(B, ntext, cfg["text_encoder_in_dim1"], generator=g),
             pooled_emb=torch.randn(B, cfg["text_encoder_in_dim2"], generator=g),
             image_emb=torch.randn(B, cfg["image_encoder_in_dim"], generator=g))
    if cfg.get("inpainting"):
        d["inpaint_image"] = torch.randn(B, cfg["in_channels"], H, W, generator=g)
        d["inpaint_mask"] = (torch.rand(B, 1, H, W, generator=g) > 0.5).float()
    return d


def golden_unet(name, cfg, B, H, W, ntext, wseed, iseed):
    model = build_ref_unet(cfg)
    spec = uo.unet_param_spec(cfg)
    ref_keys = [(k, tuple(v.shape)) for k, v in model.state_dict().items()]
    assert ref_keys == [(k, tuple(s)) for k, s in spec], "oracle parameter spec != reference state_dict"
    sd = synth.synth_state_dict(spec, seed=wseed)
    model.load_state_dict(sd, strict=True)
    inp = unet_inputs(cfg, B, H, W, ntext, iseed)
    kw = {k: v for k, v in inp.items() if k not in ("x", "t")}
    with torch.no_grad():
        y_ref = model(inp["x"], inp["t"], **kw)
        y_orc = uo.unet_forward(sd, cfg, inp["x"], inp["t"], **kw)
    err = (y_ref - y_orc).abs().max().item()
    assert err <= 1e-5, f"{name}: oracle deviates from the reference by {err}"
    # the reference in ITS OWN fp16 mode (Text2ImUNet.convert_to_fp16, text2im_model2_1.py:49-55; the pipelines feed fp16
    # embeddings): pins the oracle's fp16 mode, which calibrates the product's deviation on the GPU (tests/test_gpu_unet.py)
    model.del_cache()
    model.dtype = torch.float16
    model.convert_to_fp16()
    with torch.no_grad():
        y_ref16 = model(inp["x"], inp["t"], **{k: (v.half() if k.endswith("_emb") else v) for k, v in kw.items()})
        y_orc16 = uo.unet_forward(uo.to_reference_fp16(sd), cfg, inp["x"], inp["t"], fp16=True, **kw)
    err16 = (y_ref16 - y_orc16).abs().max().item()
    assert err16 <= 1e-5, f"{name}: oracle fp16 mode deviates from the reference's fp16 mode by {err16}"
    print(f"{name}: reference fp16 mode vs fp32 mode max abs {(y_ref16 - y_ref).abs().max():.2e}; oracle fp16 vs it {err16:.2e}")
    torch.save(dict(cfg=cfg, weight_seed=wseed, inputs=inp, out=y_ref, out_ref_fp16=y_ref16, shape=(B, H, W), ntext=ntext,
                    weight_checksum=float(sum(v.double().sum() for v in sd.values()))),
               os.path.join(GOLD, name + ".pt"))
    print(f"{name}: reference out std {y_ref.std():.4f}, oracle-vs-reference max abs {err:.2e}")


def golden_fp16_probe():
    """The fp16 CPU arithmetic of the host that wrote the `out_ref_fp16` outputs above (unet_oracle.fp16_cpu_probe): a host
    that reproduces it computes the reference's fp16 mode bit for bit like this one."""
    probe = uo.fp16_cpu_probe()
    torch.save(probe, os.path.join(GOLD, "fp16_cpu_probe.pt"))
    print("fp16_cpu_probe:", probe["cpu_capability"])


def main():
    os.makedirs(GOLD, exist_ok=True)
    torch.manual_seed(0)
    golden_unet("unet_tiny", uo.CONFIG_TINY, 2, 16, 16, 7, wseed=1, iseed=5)
    golden_unet("unet_tiny_inpaint", dict(uo.CONFIG_TINY, inpainting=True), 2, 16, 16, 7, wseed=2, iseed=6)
    golden_fp16_probe()
    for extra in EXTRA:
        extra()


def golden_movq(name, dd, B, h, w, wseed, iseed, n_embed=64):
    import contextlib
    import io
    from oracle import movq_oracle as mo
    with ref_shim.reference_modules() as R:
        ae = R.load("vqgan.autoencoder")
        with contextlib.redirect_stdout(io.StringIO()):  # the reference ctor prints (movq_modules.py:261-265)
            m = ae.MOVQ(dict(dd, double_z=False, dropout=0.0), n_embed=n_embed, embed_dim=4).eval()
    dd = dict(dd, double_z=False)
    spec = mo.movq_param_spec(dd, 4, n_embed)
    ref = [(k, tuple(v.shape)) for k, v in m.state_dict().items()]
    assert ref == [(k, tuple(s)) for k, s in spec], "oracle MoVQ parameter spec != reference state_dict"
    sd = synth.synth_state_dict(spec, seed=wseed)
    m.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(iseed)
    z = torch.randn(B, 4, h, w, generator=g)
    scale = 2 ** (len(dd["ch_mult"]) - 1)
    image = torch.rand(B, 3, h * scale, w * scale, generator=g) * 2 - 1
    with torch.no_grad():
        y_ref = m.decode(z)
        y_orc = mo.movq_decode(sd, dd, z)
        lat_ref = m.encode(image)
        lat_orc = mo.movq_encode(sd, dd, image)
        zf = z.permute(0, 2, 3, 1).reshape(-1, 4)
        # VectorQuantizer.forward's distance/argmin lines (quntize.py:89-98) on the same z
        emb = m.quantize.embedding.weight
        d = torch.sum(zf ** 2, dim=1, keepdim=True) + torch.sum(emb ** 2, dim=1) - 2 * torch.einsum("bd,dn->bn", zf, emb.t())
        idx_ref = torch.argmin(d, dim=1)
        idx_orc = mo.vq_indices(zf, sd["quantize.embedding.weight"])
    assert (lat_ref - lat_orc).abs().max().item() <= 1e-5, "MoVQ encoder oracle deviates"
    err = (y_ref - y_orc).abs().max().item()
    assert err <= 1e-5 and torch.equal(idx_ref, idx_orc), f"{name}: MoVQ oracle deviates ({err})"
    torch.save(dict(dd=dd, n_embed=n_embed, weight_seed=wseed, z=z, out=y_ref, indices=idx_ref, image=image, latent=lat_ref),
               os.path.join(GOLD, name + ".pt"))
    print(f"{name}: reference out std {y_ref.std():.4f}, oracle-vs-reference max abs {err:.2e}")


def golden_trajectory(name, cfg, B, H, W, ntext, steps, guidance, wseed, iseed):
    """Reference SpacedDiffusion.p_sample_loop (p_sampler path of Kandinsky2_1.generate_img) on the tiny reference
    UNet with the CFG closure of kandinsky2_1_model.py:222-233 and injected noise."""
    from oracle import diffusion_oracle as do
    model = build_ref_unet(cfg)
    spec = uo.unet_param_spec(cfg)
    sd = synth.synth_state_dict(spec, seed=wseed)
    model.load_state_dict(sd, strict=True)
    inp = unet_inputs(cfg, 2 * B, H, W, ntext, iseed)
    g = torch.Generator().manual_seed(iseed + 100)
    x_T = torch.randn(2 * B, 4, H, W, generator=g)
    step_noise = torch.randn(steps, 2 * B, 4, H, W, generator=g)
    kw = dict(full_emb=inp["full_emb"], pooled_emb=inp["pooled_emb"], image_emb=inp["image_emb"])
    with ref_shim.reference_modules() as R:
        mc = R.load("model.model_creation")
        gdm = R.load("model.gaussian_diffusion")
        diffusion = mc.create_gaussian_diffusion(steps=1000, learn_sigma=True, sigma_small=False, noise_schedule="linear",
                                                 use_kl=False, predict_xstart=False, rescale_timesteps=True,
                                                 rescale_learned_sigmas=True, timestep_respacing=str(steps),
                                                 linear_start=0.00085, linear_end=0.012)

        def model_fn(x_t, ts, **kwargs):  # kandinsky2_1_model.py:222-233, sampler == "p_sampler"
            half = x_t[: len(x_t) // 2]
            combined = torch.cat([half, half], dim=0)
            model_out = model(combined, ts, **kwargs)
            eps, rest = model_out[:, :4], model_out[:, 4:]
            cond_eps, uncond_eps = torch.split(eps, len(eps) // 2, dim=0)
            half_eps = uncond_eps + guidance * (cond_eps - uncond_eps)
            eps = torch.cat([half_eps, half_eps], dim=0)
            return torch.cat([eps, rest], dim=1)

        it = iter(step_noise)
        orig = gdm.th.randn_like
        gdm.th.randn_like = lambda x: next(it)
        try:
            model.del_cache()
            with torch.no_grad():
                out = diffusion.p_sample_loop(model_fn, (2 * B, 4, H, W), device="cpu", noise=x_T, progress=False,
                                              model_kwargs=kw, denoised_fn=lambda x: x.clamp(-2, 2))[:B]
        finally:
            gdm.th.randn_like = orig
        tables = dict(betas=diffusion.betas.copy(), timestep_map=list(diffusion.timestep_map),
                      post_logvar=diffusion.posterior_log_variance_clipped.copy(),
                      coef1=diffusion.posterior_mean_coef1.copy(), coef2=diffusion.posterior_mean_coef2.copy())
    # the oracle restatement on the same inputs
    tab = do.Tables(do.linear_betas(), do.space_timesteps(1000, steps))
    assert tab.timestep_map == tables["timestep_map"] and np.allclose(tab.betas, tables["betas"], rtol=0, atol=0)
    assert np.array_equal(tab.post_logvar, tables["post_logvar"]) and np.array_equal(tab.coef1, tables["coef1"])
    with torch.no_grad():
        orc = do.p_sample_loop(lambda xx, tt: uo.unet_forward(sd, cfg, xx, tt, **kw), tab, x_T[:B], step_noise[:, :B], guidance)
    err = (out - orc).abs().max().item()
    assert err <= 1e-4, f"{name}: oracle trajectory deviates from the reference by {err}"
    torch.save(dict(cfg=cfg, weight_seed=wseed, cond=kw, x_T=x_T[:B].clone(), step_noise=step_noise[:, :B].clone(),
                    steps=steps, guidance=guidance, out=out, tables=tables), os.path.join(GOLD, name + ".pt"))
    print(f"{name}: final latent std {out.std():.4f}, oracle-vs-reference max abs {err:.2e}")


def golden_sampler(name, which, cfg, B, H, W, ntext, steps, guidance, wseed, iseed):
    """Reference DDIMSampler / PLMSSampler (model/samplers.py, the non-p_sampler branch of Kandinsky2_1.generate_img,
    kandinsky2_1_model.py:222-281) on the tiny reference UNet.  The classes hard-code "cuda"; ref_shim.cuda_as_cpu maps
    that device to the CPU without touching the reference source."""
    from oracle import diffusion_oracle as do
    model = build_ref_unet(cfg)
    sd = synth.synth_state_dict(uo.unet_param_spec(cfg), seed=wseed)
    model.load_state_dict(sd, strict=True)
    inp = unet_inputs(cfg, 2 * B, H, W, ntext, iseed)
    g = torch.Generator().manual_seed(iseed + 200)
    x_T = torch.randn(B, 4, H, W, generator=g)
    kw = dict(full_emb=inp["full_emb"], pooled_emb=inp["pooled_emb"], image_emb=inp["image_emb"])
    with ref_shim.reference_modules() as R, ref_shim.cuda_as_cpu():
        mc = R.load("model.model_creation")
        sm = R.load("model.samplers")
        diffusion = mc.create_gaussian_diffusion(steps=1000, learn_sigma=True, sigma_small=False, noise_schedule="linear",
                                                 use_kl=False, predict_xstart=False, rescale_timesteps=True,
                                                 rescale_learned_sigmas=True, timestep_respacing="",
                                                 linear_start=0.00085, linear_end=0.012)

        def model_fn(x_t, ts, **kwargs):  # kandinsky2_1_model.py:222-233, sampler != "p_sampler"
            half = x_t[: len(x_t) // 2]
            combined = torch.cat([half, half], dim=0)
            model_out = model(combined, ts, **kwargs)
            eps = model_out[:, :4]
            cond_eps, uncond_eps = torch.split(eps, len(eps) // 2, dim=0)
            half_eps = uncond_eps + guidance * (cond_eps - uncond_eps)
            return torch.cat([half_eps, half_eps], dim=0)

        cls = sm.DDIMSampler if which == "ddim" else sm.PLMSSampler
        sampler = cls(model=model_fn, old_diffusion=diffusion, schedule="linear")
        model.del_cache()
        with torch.no_grad():
            out, _ = sampler.sample(steps, 2 * B, (4, H, W), conditioning=kw, x_T=torch.cat([x_T, x_T]), verbose=False)
        out = out[:B].clone()
        ddim_t = np.asarray(sampler.ddim_timesteps).copy()
    loop = do.ddim_sample_loop if which == "ddim" else do.plms_sample_loop
    with torch.no_grad():
        orc = loop(lambda xx, tt: uo.unet_forward(sd, cfg, xx, tt, **kw), x_T, steps, guidance)
    err = (out - orc).abs().max().item()
    assert np.array_equal(ddim_t, do.ddim_schedule(steps)[0]), "DDIM timesteps differ"
    assert err <= 1e-4, f"{name}: oracle {which} loop deviates from the reference by {err}"
    torch.save(dict(cfg=cfg, weight_seed=wseed, cond=kw, x_T=x_T.clone(), steps=steps, guidance=guidance, out=out,
                    sampler=which), os.path.join(GOLD, name + ".pt"))
    print(f"{name}: final latent std {out.std():.4f}, oracle-vs-reference max abs {err:.2e}")


def golden_host_utils():
    """Reference host pre-processing of the img2img / inpainting entry points (`kandinsky2/utils.py:11-54`): prepare_mask
    (python-loop erosion), prepare_image (PIL bicubic + scaling) and q_sample, on seeded inputs."""
    from PIL import Image
    g = torch.Generator().manual_seed(77)
    mask = (torch.rand(1, 1, 24, 20, generator=g) > 0.3).float()
    mask[:, :, 5:9, 4:12] = 0
    img = (torch.rand(37, 53, 3, generator=g) * 255).to(torch.uint8).numpy()
    x0 = torch.randn(2, 4, 8, 8, generator=g)
    noise = torch.randn(2, 4, 8, 8, generator=g)
    t = torch.tensor([10, 700])
    with ref_shim.reference_modules() as R:
        ut = R.load("utils")
        out = dict(mask_in=mask.clone(), mask_out=ut.prepare_mask(mask.clone()), img_in=img,
                   img_out=ut.prepare_image(Image.fromarray(img), w=64, h=48), x0=x0, noise=noise, t=t,
                   q_out=ut.q_sample(x0, t, noise=noise))
    torch.save(out, os.path.join(GOLD, "host_utils.pt"))
    print("host_utils: mask kept", float(out["mask_out"].mean()), "q_sample std", float(out["q_out"].std()))


def golden_prior(name, cfg, B, steps, guidance, wseed, iseed):
    """Reference PriorTransformer.forward and PriorDiffusionModel.forward (`model/prior.py:159-384`) on synthetic weights.
    `clip` (tokenizer only) is stubbed; the config is a SimpleNamespace with the fields prior.py reads."""
    import types
    from oracle import prior_oracle as po
    spec = po.prior_param_spec(cfg)
    sd = synth.synth_state_dict(spec, seed=wseed)
    g = torch.Generator().manual_seed(iseed)
    D, n_txt = cfg["clip_dim"], cfg["text_ctx"]
    x = torch.randn(2 * B, D, generator=g)
    t = torch.tensor([999.0, 500.0, 20.0, 0.0][:2 * B])
    text_emb = torch.randn(2 * B, D, generator=g)
    text_enc = torch.randn(2 * B, n_txt, cfg["clip_xf_width"], generator=g)
    mask = torch.ones(2 * B, n_txt, dtype=torch.bool)
    mask[0, 3:] = False
    mask[B:, 1:] = False                                   # the unconditional rows: only the start token is real
    x_T = torch.randn(B, D, generator=g)
    step_noise = torch.randn(steps, B, D, generator=g)
    clip_mean, clip_std = torch.randn(D, generator=g), torch.rand(D, generator=g) + 0.5
    saved = {k: sys.modules.get(k) for k in ("clip", "clip.simple_tokenizer")}
    clip_stub, tok_stub = types.ModuleType("clip"), types.ModuleType("clip.simple_tokenizer")
    tok_stub.SimpleTokenizer = object
    tok_stub.default_bpe = lambda: None
    sys.modules["clip"], sys.modules["clip.simple_tokenizer"] = clip_stub, tok_stub
    try:
        with ref_shim.reference_modules() as R:
            pr = R.load("model.prior")
            gdm = R.load("model.gaussian_diffusion")
            ns = types.SimpleNamespace
            conf = ns(model=ns(hparams=ns(**cfg)),
                      diffusion=ns(steps=1000, learn_sigma=False, sigma_small=True, noise_schedule="cosine", use_kl=False,
                                   predict_xstart=True, rescale_learned_sigmas=False, timestep_respacing=""))
            tok = ns(padded_tokens_and_mask=lambda texts, n: (torch.zeros(1, n, dtype=torch.long), torch.zeros(1, n, dtype=torch.bool)))
            pdm = pr.PriorDiffusionModel(conf, tok, clip_mean, clip_std).eval()
            assert [(k, tuple(v.shape)) for k, v in pdm.model.state_dict().items()] == [(k, tuple(s_)) for k, s_ in spec], \
                "oracle prior parameter spec != reference state_dict"
            pdm.model.load_state_dict(sd, strict=True)
            with torch.no_grad():
                y_ref = pdm.model(x, t, text_emb=text_emb, text_enc=text_enc, mask=mask, causal_mask=pdm.causal_mask)
            # sampling loop with injected noise: first th.randn = x_T (both halves), th.randn_like = the per-step noise
            it = iter(step_noise)
            o_randn, o_like = gdm.th.randn, gdm.th.randn_like
            gdm.th.randn = lambda *a, **k: torch.cat([x_T, x_T])
            gdm.th.randn_like = lambda v: (lambda nz: torch.cat([nz, nz]))(next(it))
            try:
                with torch.no_grad():
                    s_ref = pdm(text_emb, text_enc, mask, cf_guidance_scales=torch.full((B,), guidance),
                                timestep_respacing=str(steps))
            finally:
                gdm.th.randn, gdm.th.randn_like = o_randn, o_like
            rs = R.load("model.respace")
            use_steps = sorted(rs.space_timesteps(1000, str(steps)))
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    with torch.no_grad():
        y_orc = po.prior_forward(sd, cfg, x, t, text_emb, text_enc, mask)
        s_orc = po.prior_sample(lambda xx, tt: po.prior_forward(sd, cfg, xx, tt, text_emb, text_enc, mask), x_T, step_noise,
                                use_steps, guidance, clip_mean, clip_std)
    e1, e2 = (y_ref - y_orc).abs().max().item(), (s_ref - s_orc).abs().max().item()
    assert e1 <= 1e-4 and e2 <= 1e-4, f"{name}: oracle prior deviates from the reference: forward {e1}, sample {e2}"
    torch.save(dict(cfg=cfg, weight_seed=wseed, x=x, t=t, text_emb=text_emb, text_enc=text_enc, mask=mask, out=y_ref,
                    x_T=x_T, step_noise=step_noise, use_steps=use_steps, guidance=guidance, clip_mean=clip_mean,
                    clip_std=clip_std, sample=s_ref), os.path.join(GOLD, name + ".pt"))
    print(f"{name}: forward std {y_ref.std():.4f} (oracle err {e1:.2e}), sample std {s_ref.std():.4f} (oracle err {e2:.2e})")


def golden_schedule():
    """Known-answer constants of the reference schedule code (SURVEY.md 8c)."""
    with ref_shim.reference_modules() as R:
        mc = R.load("model.model_creation")
        rs = R.load("model.respace")
        nn_ = R.load("model.nn")
        d50 = mc.create_gaussian_diffusion(steps=1000, learn_sigma=True, noise_schedule="linear", rescale_timesteps=True,
                                           rescale_learned_sigmas=True, timestep_respacing="50", linear_start=0.00085,
                                           linear_end=0.012)
        kat = dict(space50=sorted(rs.space_timesteps(1000, "50")), space20=sorted(rs.space_timesteps(1000, "20")),
                   betas50=d50.betas.copy(), post_logvar50=d50.posterior_log_variance_clipped.copy(),
                   coef1_50=d50.posterior_mean_coef1.copy(), coef2_50=d50.posterior_mean_coef2.copy(),
                   sqrt_recip50=d50.sqrt_recip_alphas_cumprod.copy(), sqrt_recipm1_50=d50.sqrt_recipm1_alphas_cumprod.copy(),
                   temb=nn_.timestep_embedding(torch.tensor([999.0, 0.0, 500.5]), 384))
        sm = R.load("model.samplers")  # pure-numpy schedule helpers of the DDIM sampler (the class itself needs CUDA)
        d1000 = mc.create_gaussian_diffusion(steps=1000, learn_sigma=True, noise_schedule="linear", rescale_timesteps=True,
                                             rescale_learned_sigmas=True, timestep_respacing="", linear_start=0.00085,
                                             linear_end=0.012)
        for S in (50, 30):
            t = sm.make_ddim_timesteps("uniform", S, 1000, verbose=False)
            sig, al, alp = sm.make_ddim_sampling_parameters(d1000.alphas_cumprod, t, 0.0, verbose=False)
            kat[f"ddim{S}"] = dict(t=t.copy(), alphas=np.asarray(al).copy(), alphas_prev=np.asarray(alp).copy(),
                                   sigmas=np.asarray(sig).copy())
    torch.save(kat, os.path.join(GOLD, "schedule_kat.pt"))
    print("schedule_kat: betas50[:3]", kat["betas50"][:3])


EXTRA = [
    lambda: golden_movq("movq_tiny", __import__("oracle.movq_oracle", fromlist=["x"]).DDCONFIG_TINY, 2, 8, 8, wseed=4, iseed=3),
    lambda: golden_trajectory("traj_tiny", uo.CONFIG_TINY, 2, 16, 16, 7, steps=5, guidance=4.0, wseed=1, iseed=21),
    golden_schedule,
    golden_host_utils,
    lambda: golden_prior("prior_tiny", __import__("oracle.prior_oracle", fromlist=["x"]).CONFIG_PRIOR_TINY, 2, steps=4,
                         guidance=4.0, wseed=5, iseed=31),
    lambda: golden_sampler("ddim_tiny", "ddim", uo.CONFIG_TINY, 2, 16, 16, 7, steps=4, guidance=3.0, wseed=1, iseed=21),
    lambda: golden_sampler("plms_tiny", "plms", uo.CONFIG_TINY, 2, 16, 16, 7, steps=5, guidance=2.0, wseed=1, iseed=21),
]

if __name__ == "__main__":
    main()
