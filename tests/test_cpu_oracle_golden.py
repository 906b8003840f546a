"""CPU: the oracle restatement against the committed golden vectors (written by oracle/make_golden.py from the
reference's own code), the schedule known-answer constants, and the host-side schedule code of the product."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def _load(name):
    return torch.load(os.path.join(GOLD, name + ".pt"), weights_only=False)


@pytest.mark.parametrize("name", ["unet_tiny", "unet_tiny_inpaint"])
def test_unet_oracle_matches_reference_golden(name):
    from oracle import synth, unet_oracle as uo
    fx = _load(name)
    sd = synth.synth_state_dict(uo.unet_param_spec(fx["cfg"]), seed=fx["weight_seed"])
    assert abs(float(sum(v.double().sum() for v in sd.values())) - fx["weight_checksum"]) < 1e-6
    inp = fx["inputs"]
    kw = {k: v for k, v in inp.items() if k not in ("x", "t")}
    with torch.no_grad():
        y = uo.unet_forward(sd, fx["cfg"], inp["x"], inp["t"], **kw)
    assert (y - fx["out"]).abs().max().item() <= 1e-5


@pytest.mark.parametrize("name", ["unet_tiny", "unet_tiny_inpaint"])
def test_unet_oracle_fp16_mode_matches_reference_fp16_mode(name):
    """The oracle's fp16 mode (to_reference_fp16 + fp16=True) against the reference's own fp16 mode
    (Text2ImUNet.convert_to_fp16()).  It is the comparator of the GPU calibration test
    (tests/test_gpu_unet.py::test_unet_full_size_fp16_calibration).

    fp16 convolutions on a CPU depend on the CPU (AVX512-FP16 / AVX512 / AVX2 paths accumulate differently: the same fixture
    re-run on another host moves by ~4e-3), so the pin has two parts: (1) on a host whose fp16 arithmetic matches that of
    the host that wrote the fixture (tests/golden/fp16_cpu_probe.pt, bit for bit) the oracle must reproduce the reference's
    stored fp16 output to 1e-5 -- same code path, same kernels; (2) everywhere, the oracle stays within 3x the reference's
    own fp16-vs-fp32 gap of the committed fixture (oracle/make_golden.py)."""
    from oracle import synth, unet_oracle as uo
    fx = _load(name)
    sd = synth.synth_state_dict(uo.unet_param_spec(fx["cfg"]), seed=fx["weight_seed"])
    inp = fx["inputs"]
    kw = {k: v for k, v in inp.items() if k not in ("x", "t")}
    with torch.no_grad():
        y = uo.unet_forward(uo.to_reference_fp16(sd), fx["cfg"], inp["x"], inp["t"], fp16=True, **kw)
    assert y.dtype == torch.float32
    gap = (fx["out_ref_fp16"] - fx["out"]).abs().max().item()
    # the reference's fp16 mode itself is ~5e-3 away from its fp32 mode at this size: the north_star's 1e-3 is not a property
    # of the reference
    assert gap > 1e-3
    assert (y - fx["out_ref_fp16"]).abs().max().item() <= 3 * gap
    assert (y - fx["out"]).abs().max().item() <= 3 * gap
    if uo.fp16_cpu_probe() == _load("fp16_cpu_probe"):
        assert (y - fx["out_ref_fp16"]).abs().max().item() <= 1e-5


def test_movq_oracle_matches_reference_golden():
    from oracle import movq_oracle as mo, synth
    fx = _load("movq_tiny")
    sd = synth.synth_state_dict(mo.movq_param_spec(fx["dd"], 4, fx["n_embed"]), seed=fx["weight_seed"])
    with torch.no_grad():
        y = mo.movq_decode(sd, fx["dd"], fx["z"])
    assert (y - fx["out"]).abs().max().item() <= 1e-5
    zf = fx["z"].permute(0, 2, 3, 1).reshape(-1, 4)
    assert torch.equal(mo.vq_indices(zf, sd["quantize.embedding.weight"]), fx["indices"])  # bit-exact indices
    with torch.no_grad():
        ze = mo.movq_encode(sd, fx["dd"], fx["image"])
    assert (ze - fx["latent"]).abs().max().item() <= 1e-5


def test_trajectory_oracle_matches_reference_golden():
    from oracle import diffusion_oracle as do, synth, unet_oracle as uo
    fx = _load("traj_tiny")
    sd = synth.synth_state_dict(uo.unet_param_spec(fx["cfg"]), seed=fx["weight_seed"])
    tab = do.Tables(do.linear_betas(), do.space_timesteps(1000, fx["steps"]))
    with torch.no_grad():
        out = do.p_sample_loop(lambda xx, tt: uo.unet_forward(sd, fx["cfg"], xx, tt, **fx["cond"]), tab, fx["x_T"],
                               fx["step_noise"], fx["guidance"])
    assert (out - fx["out"]).abs().max().item() <= 1e-4


@pytest.mark.parametrize("name", ["ddim_tiny", "plms_tiny"])
def test_ddim_plms_oracle_matches_reference_golden(name):
    """The oracle's DDIM / PLMS loops vs the output of the reference's own DDIMSampler / PLMSSampler classes
    (model/samplers.py, executed by oracle/make_golden.py through the cuda->cpu device shim)."""
    from oracle import diffusion_oracle as do, synth, unet_oracle as uo
    fx = _load(name)
    cfg = fx["cfg"]
    sd = synth.synth_state_dict(uo.unet_param_spec(cfg), seed=fx["weight_seed"])
    loop = do.ddim_sample_loop if fx["sampler"] == "ddim" else do.plms_sample_loop
    with torch.no_grad():
        out = loop(lambda xx, tt: uo.unet_forward(sd, cfg, xx, tt, **fx["cond"]), fx["x_T"], fx["steps"], fx["guidance"])
    assert (out - fx["out"]).abs().max().item() <= 1e-4


def test_schedule_known_answers():
    """Constants obtained by running the reference (SURVEY.md 8c) + the product's host schedule code."""
    from oracle import diffusion_oracle as do
    kat = _load("schedule_kat")
    b = do.linear_betas()
    assert b[0] == 0.00085 and abs(b[999] - 0.012) < 1e-15
    ac = np.cumprod(1 - b)
    assert abs(ac[0] - 0.99915) < 1e-12 and abs(ac[499] - 0.1618121459134018) < 1e-12
    assert abs(ac[999] - 0.0015789629305514416) < 1e-14
    assert do.space_timesteps(1000, 50) == kat["space50"] and do.space_timesteps(1000, 20) == kat["space20"]
    assert kat["space20"][:6] == [0, 53, 105, 158, 210, 263] and kat["space50"][-3:] == [958, 979, 999]
    tab = do.Tables(b, kat["space50"])
    assert np.array_equal(tab.betas, kat["betas50"]) and np.array_equal(tab.post_logvar, kat["post_logvar50"])
    assert np.allclose(kat["betas50"][:3], [0.00085, 0.01916717422017, 0.02481784056427294], rtol=1e-12)
    assert abs(kat["post_logvar50"][0] + 7.1128514473284525) < 1e-12
    # product host code (no GPU needed: numpy tables only)
    from kandinsky2.model.gaussian_diffusion import create_gaussian_diffusion, create_ddpm_v22, space_timesteps
    assert sorted(space_timesteps(1000, "50")) == kat["space50"]
    d = create_gaussian_diffusion(steps=1000, learn_sigma=True, noise_schedule="linear", rescale_timesteps=True,
                                  rescale_learned_sigmas=True, timestep_respacing="50", linear_start=0.00085,
                                  linear_end=0.012)
    assert np.array_equal(d.betas, kat["betas50"])
    coef = d.coef_table()
    assert np.array_equal(coef[:, 0], kat["sqrt_recip50"].astype(np.float32))
    assert np.array_equal(coef[:, 1], kat["sqrt_recipm1_50"].astype(np.float32))
    assert np.array_equal(coef[:, 2], kat["coef1_50"].astype(np.float32))
    assert np.array_equal(coef[:, 3], kat["coef2_50"].astype(np.float32))
    assert np.array_equal(coef[:, 4], kat["post_logvar50"].astype(np.float32))
    assert d.model_timestep(49) == 999.0 and d.model_timestep(1) == 20.0
    v22 = create_ddpm_v22(50)
    assert v22.timestep_map[:3] == [0, 20, 40] and v22.timestep_map[-1] == 980 and v22.num_timesteps == 50
    # DDIM schedule helpers (samplers.py:21-55) -- oracle restatement and the product's coefficient table
    from kandinsky2.model.gaussian_diffusion import DDIMSampler
    d1000 = create_gaussian_diffusion(steps=1000, learn_sigma=True, noise_schedule="linear", rescale_timesteps=True,
                                      rescale_learned_sigmas=True, timestep_respacing="", linear_start=0.00085,
                                      linear_end=0.012)
    for S in (50, 30):
        ref = kat[f"ddim{S}"]
        tt, al, alp = do.ddim_schedule(S)
        assert np.array_equal(tt, ref["t"]) and np.array_equal(al, ref["alphas"]) and np.array_equal(alp, ref["alphas_prev"])
        assert not ref["sigmas"].any()
        s = DDIMSampler(None, d1000)
        s.make_schedule(S)
        assert np.array_equal(s.ddim_timesteps, ref["t"]) and np.array_equal(s.ddim_alphas, ref["alphas"])
        # the fused-step coefficients reproduce the reference's two-line update on random data
        g = np.random.default_rng(0)
        x, e = g.standard_normal(64), g.standard_normal(64)
        c = s.coef_table().astype(np.float64)
        for i in (0, S // 2, len(tt) - 1):
            x0 = c[i, 0] * x - c[i, 1] * e
            assert np.allclose(c[i, 2] * x0 + c[i, 3] * x, do.ddim_step(x, e, al[i], alp[i]), rtol=2e-5, atol=2e-5)
    # timestep embedding known answers (cos first)
    from oracle import unet_oracle as uo
    te = uo.timestep_embedding(torch.tensor([999.0, 0.0, 500.5]), 384)
    assert torch.equal(te, kat["temb"])
    assert abs(te[0, 0].item() - 0.99964982) < 1e-6 and abs(te[0, 192].item() + 0.02646075) < 1e-6


def test_param_counts_and_flops():
    from oracle import movq_oracle as mo, unet_oracle as uo
    n = sum(int(np.prod(s)) for _, s in uo.unet_param_spec(uo.CONFIG_2_1))
    assert n == 1228661768  # SURVEY.md 8c: CONFIG_2_1 UNet parameter count
    f = uo.algorithmic_flops(uo.CONFIG_2_2, 8, 96, 96, 32)
    assert abs(f / 1e12 - 15.940) < 0.02  # BASELINE.md: 15.940 TFLOP per cfg-2 step
    assert abs(uo.algorithmic_flops(uo.CONFIG_2_1, 2, 32, 32, 87) / 1e12 - 0.433) < 0.002
    fm = mo.decode_flops(mo.DDCONFIG_2_1, 4, 96, 96)
    assert abs(fm / 1e12 - 19.54) < 0.3  # BASELINE.md: 19.542 TFLOP per B=4 768^2 decode


def test_host_preprocessing_matches_reference_golden():
    """kandinsky2/utils.py of the product (prepare_mask, prepare_image, q_sample -- the host side of generate_img2img /
    generate_inpainting) against the outputs of the reference's own functions (`utils.py:11-54`, host_utils.pt)."""
    from PIL import Image
    sys.path.insert(0, os.path.join(ROOT, "kandinsky-2_b200"))
    from kandinsky2 import utils as ku
    fx = _load("host_utils")
    assert torch.equal(ku.prepare_mask(fx["mask_in"].clone()), fx["mask_out"])
    assert torch.equal(ku.prepare_image(Image.fromarray(fx["img_in"]), w=64, h=48), fx["img_out"])
    got = ku.q_sample(fx["x0"], fx["t"], noise=fx["noise"])
    assert torch.allclose(got, fx["q_out"], rtol=0, atol=1e-6)


def test_prior_oracle_matches_reference_golden():
    """Groundwork for SURVEY.md 8f rank 3: the oracle's restatement of the diffusion prior (transformer forward and the
    predict-x0 / cosine-schedule sampling loop with classifier-free guidance) against the outputs of the reference's own
    PriorTransformer / PriorDiffusionModel classes (prior_tiny.pt)."""
    from oracle import prior_oracle as po, synth
    fx = _load("prior_tiny")
    cfg = fx["cfg"]
    sd = synth.synth_state_dict(po.prior_param_spec(cfg), seed=fx["weight_seed"])
    with torch.no_grad():
        y = po.prior_forward(sd, cfg, fx["x"], fx["t"], fx["text_emb"], fx["text_enc"], fx["mask"])
        s = po.prior_sample(lambda xx, tt: po.prior_forward(sd, cfg, xx, tt, fx["text_emb"], fx["text_enc"], fx["mask"]),
                            fx["x_T"], fx["step_noise"], fx["use_steps"], fx["guidance"], fx["clip_mean"], fx["clip_std"])
    assert (y - fx["out"]).abs().max().item() <= 1e-5
    assert (s - fx["sample"]).abs().max().item() <= 1e-4
    # full-size parameter count of the 2.1 prior (20 layers, width 2048)
    n = sum(int(np.prod(shape)) for _, shape in po.prior_param_spec(po.CONFIG_PRIOR))
    assert 1.0e9 < n < 1.1e9, n
