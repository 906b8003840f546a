"""The fused sampler-step kernels (k2_sampler_step, k2_plms_step, k2_step_begin / k2_step_end) against float64 numpy
restatements computed from the same float32 inputs and the same float32 coefficient rows, at the latent sizes the pipelines
run (4 x 96 x 96 = 36 864 values per sample, 4 x 128 x 128 = 65 536).

The dynamic threshold's percentile is exact, so it is checked bit for bit against _percentile995, a restatement of numpy >= 2's
np.percentile(v, 99.5) that test_percentile995_matches_numpy pins to the installed numpy.  Everything else is checked per
element within ROUNDOFFS fp32 unit roundoffs of the sum of the absolute values of the terms that produce it (see _step_ref):
the kernels are built with nvcc's default FMA contraction, so bit equality is not expected there, but any wrong term (a
swapped CFG half, a misplaced blend, a wrong coefficient) is off by many orders of magnitude more."""
import numpy as np
import pytest
import torch

F32 = np.float32
UNIT = 2.0 ** -24   # fp32 unit roundoff
ROUNDOFFS = 16


# ------------------------------------------------------------------------------------------------
# numpy >= 2 percentile, restated
# ------------------------------------------------------------------------------------------------
def _percentile995(v):
    """np.percentile(v, 99.5) for float32 v as numpy >= 2 computes it (numpy/lib/_function_base_impl.py).  Under NEP 50 the
    arithmetic stays in float32: percentile divides q by float32(100); the 'linear' method's virtual index is (n - 1) * q;
    _get_indexes takes floor and floor + 1, both moved to the last element when the index reaches n - 1; _get_gamma subtracts
    the intp floor (in float64, exact) and casts back to float32; _lerp rounds each operation to float32 and switches to
    b - (b - a) * (1 - t) for t >= 0.5."""
    v = np.sort(np.asarray(v, dtype=F32).ravel())
    n = v.size
    q = F32(99.5) / F32(100)
    pos = F32(n - 1) * q
    if pos >= n - 1:
        lo = hi = n - 1
    else:
        lo = int(np.floor(pos))
        hi = lo + 1
    t = F32(np.float64(pos) - np.float64(lo))
    a, b = v[lo], v[hi]
    d = F32(b - a)
    if t >= F32(0.5):
        return F32(b - F32(d * F32(F32(1) - t)))
    return F32(a + F32(d * t))


def _threshold(x0_sample0):
    """The dynamic threshold s = max(percentile_99.5(|x0 of sample 0|), 1) in float32."""
    return max(_percentile995(np.abs(x0_sample0)), F32(1.0))


def _bits(a):
    return np.asarray(a, dtype=F32).view(np.uint32)


@pytest.mark.skipif(np.lib.NumpyVersion(np.__version__) < "2.0.0",
                    reason="_percentile995 restates numpy >= 2; numpy 1.x interpolates in float64")
def test_percentile995_matches_numpy():
    rng = np.random.default_rng(995)
    checked = 0
    for n in (1, 2, 256, 4 * 13 * 17, 1024, 24576, 36864, 65536):
        for k in range(45):
            v = rng.standard_normal(n, dtype=F32) * F32((1e-3, 0.25, 1.0, 2.0, 8.0, 100.0)[k % 6])
            # signed data, |data|, and |data| clamped at 2.0 (many values tie at the top, as after the x0 clamp)
            for arr in (v, np.abs(v), np.minimum(np.abs(v), F32(2.0))):
                ref = np.percentile(arr, 99.5)
                assert ref.dtype == np.float32
                got = _percentile995(arr)
                assert _bits(got) == _bits(ref), (n, k, got, ref)
                checked += 1
    assert checked >= 1000


# ------------------------------------------------------------------------------------------------
# inputs and coefficient rows
# ------------------------------------------------------------------------------------------------
def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=F32)).cuda()


def _host(t):
    return t.detach().cpu().numpy()


def _model_out(rng, B, C2, H, W, cond_first):
    """[2B, C2, H, W] with the conditional and unconditional halves drawn differently (so a swapped half cannot pass) and
    the variance channels in [-1, 1]."""
    cond = np.empty((B, C2, H, W), F32)
    unc = np.empty((B, C2, H, W), F32)
    cond[:, :4] = rng.standard_normal((B, 4, H, W))
    unc[:, :4] = 0.6 * rng.standard_normal((B, 4, H, W)) + 0.25
    if C2 > 4:
        cond[:, 4:] = rng.uniform(-1, 1, (B, C2 - 4, H, W))
        unc[:, 4:] = rng.uniform(-1, 0, (B, C2 - 4, H, W))
    return np.concatenate([cond, unc] if cond_first else [unc, cond]).astype(F32)


def _mask(rng, B, H, W):
    """[B, 1, H, W]: about a quarter exactly 1 (known), a quarter exactly 0, the rest fractional (a resized mask's edge)."""
    return np.clip(rng.uniform(-0.5, 1.5, (B, 1, H, W)), 0, 1).astype(F32)


def _diffusion_config():
    from kandinsky2.configs import _DIFFUSION
    return dict(_DIFFUSION)


def _rows_21():
    from kandinsky2.model.gaussian_diffusion import create_gaussian_diffusion
    return create_gaussian_diffusion(**dict(_diffusion_config(), timestep_respacing="50")).coef_table()


def _rows_22():
    from kandinsky2.model.gaussian_diffusion import create_ddpm_v22
    return create_ddpm_v22(50).coef_table()


def _ddim():
    from kandinsky2.model.gaussian_diffusion import DDIMSampler, create_gaussian_diffusion
    s = DDIMSampler(None, create_gaussian_diffusion(**_diffusion_config()))
    s.make_schedule(50)
    return s


def _rows_ddim():
    return _ddim().coef_table()


# the sampling loops run the table backwards: the first step is the last row, the last step is row 0 (coef[6] = 0, coef[7] = 1)
STEPS = {"first": -1, "middle": 25, "last": 0}

# (cond_first, threshold_mode, clip, guidance, rows, 2.1 inpainting, 2.2 inpainting, noise) of each product configuration
PATHS = {
    "p21": (1, 1, 2.0, 7.0, _rows_21, False, False, True),
    "p21_inpaint": (1, 1, 2.0, 7.0, _rows_21, True, False, True),
    "ddpm22": (0, 0, 2.0, 4.0, _rows_22, False, False, True),
    "ddpm22_inpaint": (0, 0, 2.0, 4.0, _rows_22, False, True, True),
    "ddim": (1, 0, 1e30, 7.0, _rows_ddim, False, False, False),
}

SHAPES = [(4, 96, 96), (4, 64, 96), (2, 128, 128), (1, 96, 96), (2, 16, 16)]


# ------------------------------------------------------------------------------------------------
# float64 restatement of k2_sampler_step
# ------------------------------------------------------------------------------------------------
def _step_ref(mo, x, noise, coef, g, cond_first, clip, s=None, init=None, mask=None, rnoise=None):
    """-> (x0, bound of x0, x_{t-1}, bound of x_{t-1}) in float64.  x0 is the kernel's work value (after the clamp and the
    2.1 blend, before the dynamic threshold).  s: the threshold to apply (None = threshold off).  Each bound is the sum of
    the absolute values of the terms that produce the value; the variance comes from the conditional rows in both orderings
    (for 2.2 that is diffusers' variance_pred_text)."""
    B = x.shape[0]
    mo, x, noise = mo.astype(np.float64), x.astype(np.float64), noise.astype(np.float64)
    c = coef.astype(np.float64)
    cond, unc = (mo[:B], mo[B:]) if cond_first else (mo[B:], mo[:B])
    ec, eu = cond[:, :4], unc[:, :4]
    eps = eu + g * (ec - eu)
    a_eps = np.abs(eu) + g * np.abs(ec - eu)
    x0 = np.clip(c[0] * x - c[1] * eps, -clip, clip)
    a_x0 = np.abs(c[0] * x) + abs(c[1]) * a_eps
    if mask is not None and rnoise is None:  # Kandinsky 2.1: the known region replaces x0 after the clamp
        m, init = mask.astype(np.float64), init.astype(np.float64)
        x0 = x0 * (1 - m) + init * m
        a_x0 = a_x0 * (1 - m) + np.abs(init) * m
    work_x0, a_work_x0 = x0, a_x0
    if s is not None:
        s = float(s)
        x0 = np.clip(x0, -s, s) / s
        a_x0 = a_x0 / s
    mean = c[2] * x0 + c[3] * x
    a_mean = abs(c[2]) * a_x0 + np.abs(c[3] * x)
    frac = (cond[:, 4:8] + 1) / 2
    logvar = frac * c[5] + (1 - frac) * c[4]
    term = c[6] * np.exp(0.5 * logvar) * noise
    # exp turns logvar's absolute rounding error (at most a few roundoffs of |c4| + |c5|) into a relative one
    a_term = np.abs(term) * (1 + abs(c[4]) + abs(c[5]))
    xn, a_xn = mean + term, a_mean + a_term
    if mask is not None and rnoise is not None:  # Kandinsky 2.2: the known region is the clean latent re-noised with coef[7]
        m, init, rn = mask.astype(np.float64), init.astype(np.float64), rnoise.astype(np.float64)
        sg = np.sqrt(max(0.0, 1 - c[7] * c[7]))
        known = c[7] * init + sg * rn
        # sqrt(1 - c^2) carries the rounding of c * c amplified by c^2 / (2 sqrt(1 - c^2))
        a_known = np.abs(c[7] * init) + np.abs(rn) * (sg + (c[7] ** 2 / (2 * sg) if sg > 0 else 0.0))
        xn = m * known + (1 - m) * xn
        a_xn = m * a_known + (1 - m) * a_xn
    return work_x0, a_work_x0, xn, a_xn


def _assert_close(got, ref, bound, what):
    err = np.abs(got.astype(np.float64) - ref)
    lim = ROUNDOFFS * UNIT * bound
    bad = err > lim
    assert not bad.any(), (f"{what}: {int(bad.sum())} of {bad.size} elements exceed {ROUNDOFFS} roundoffs of their terms; "
                           f"worst excess {float((err / np.maximum(lim, 1e-300)).max()):.3g}x")


# ------------------------------------------------------------------------------------------------
# 1. the percentile, bit-exact
# ------------------------------------------------------------------------------------------------
IDENTITY_ROW = np.array([1, 0, 0, 0, 0, 0, 0, 0], F32)   # x0 = clamp(1 * x - 0 * eps) = clamp(x) exactly, FMA or not


def _x0_and_threshold(x, clip=2.0, seed=0):
    """Mode 2 (x0 and the percentile, no update) with the identity row: -> (x after the call, work x0, work s)."""
    from kandinsky2 import ops
    B, _, H, W = x.shape
    n = B * 4 * H * W
    rng = np.random.default_rng(seed)
    xd = _dev(x)
    work = torch.full((n + 4096,), float("nan"), device="cuda")
    ops.sampler_step(_dev(_model_out(rng, B, 8, H, W, 1)), xd, _dev(np.zeros_like(x)), _dev(IDENTITY_ROW), 7.0, 1, clip=clip,
                     threshold_mode=2, work=work)
    w = _host(work)
    return _host(xd), w[:n].reshape(x.shape), w[n]


def _shared_top_bytes(rng, shape, nbytes):
    """|values| whose bit patterns share their top `nbytes` bytes with 1.5 (0x3FC00000), random below, random signs: every
    radix pass up to that one sees a single bin."""
    low = 8 * (4 - nbytes)
    base = np.uint32(0x3FC00000) & ~np.uint32((1 << low) - 1)
    u = base | rng.integers(0, 1 << low, size=shape, dtype=np.uint32)
    v = u.view(F32)
    return np.where(rng.random(shape) < 0.5, -v, v).astype(F32)


def _zeros_and_subnormals(rng, shape, top_fraction):
    u = rng.integers(0, 1 << 23, size=shape, dtype=np.uint32)                 # subnormals (and a few +0)
    u = np.where(rng.random(shape) < 0.3, np.uint32(0), u)                    # many exact zeros
    u = u | np.where(rng.random(shape) < 0.5, np.uint32(1 << 31), np.uint32(0))  # +-0 and +-subnormal
    v = u.view(F32)
    big = rng.random(shape) < top_fraction
    return np.where(big, F32(1.0) + rng.random(shape, dtype=F32), v).astype(F32)


def _percentile_case(name, rng):
    if name.startswith("gauss"):
        B, H, W = {"gauss_96x96": (4, 96, 96), "gauss_64x96": (4, 64, 96), "gauss_128x128": (4, 128, 128),
                   "gauss_16x16": (2, 16, 16), "gauss_13x17": (1, 13, 17)}[name]
        return (0.6 * rng.standard_normal((B, 4, H, W))).astype(F32)
    shape = (4, 4, 96, 96)
    if name == "saturated":       # about 18 % of sample 0 at +-clip: ranks lo and hi both inside the tie, s = clip
        return (1.5 * rng.standard_normal(shape)).astype(F32)
    if name == "below_one":       # all |x0| < 1: s = 1
        return np.clip(0.3 * rng.standard_normal(shape), -0.999, 0.999).astype(F32)
    if name.startswith("top_bytes"):
        return _shared_top_bytes(rng, shape, int(name[-1]))
    if name == "zeros_subnormals":
        return _zeros_and_subnormals(rng, shape, 0.0)
    if name == "zeros_subnormals_top":  # 1.5 % above 1: the ranks fall among them, with +-0 / subnormals below
        return _zeros_and_subnormals(rng, shape, 0.015)
    raise KeyError(name)


PERCENTILE_CASES = ["gauss_96x96", "gauss_64x96", "gauss_128x128", "gauss_16x16", "gauss_13x17", "saturated", "below_one",
                    "top_bytes_1", "top_bytes_2", "top_bytes_3", "zeros_subnormals", "zeros_subnormals_top"]


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [0, 1, 2])
@pytest.mark.parametrize("case", PERCENTILE_CASES)
def test_percentile_bit_exact(case, seed):
    rng = np.random.default_rng([seed, PERCENTILE_CASES.index(case)])
    x = _percentile_case(case, rng)
    clip = 2.0
    x_after, x0, s = _x0_and_threshold(x, clip=clip, seed=seed)
    assert np.array_equal(_bits(x_after), _bits(x)), "mode 2 must not update x"
    assert np.array_equal(x0, np.clip(x, -clip, clip)), "the identity row must place x0 = clamp(x) exactly"
    want = _threshold(x0[0])
    assert _bits(s) == _bits(want), (case, float(s), float(want))
    if case == "saturated":
        assert s == F32(clip)
    if case in ("below_one", "zeros_subnormals"):
        assert s == F32(1.0)
    if case.startswith("top_bytes") or case == "zeros_subnormals_top":
        assert s > 1.0


@pytest.mark.gpu
def test_percentile_reads_sample_zero_only():
    rng = np.random.default_rng(7)
    x = (0.6 * rng.standard_normal((4, 4, 96, 96))).astype(F32)
    _, x0, s = _x0_and_threshold(x)
    assert _bits(s) == _bits(_threshold(x0[0]))
    other = x.copy()
    other[1:] = (1.2 * rng.standard_normal(other[1:].shape)).astype(F32)
    assert _bits(_x0_and_threshold(other)[2]) == _bits(s), "samples 1..B-1 must not move the threshold"
    first = x.copy()
    first[0] *= F32(1.1)
    _, x0f, sf = _x0_and_threshold(first)
    assert sf != s and _bits(sf) == _bits(_threshold(x0f[0]))


# ------------------------------------------------------------------------------------------------
# 2. the full step against float64, every configuration the pipelines launch
# ------------------------------------------------------------------------------------------------
def _step_inputs(path, B, H, W, seed):
    cond_first, mode, clip, g, rows, inp21, inp22, has_noise = PATHS[path]
    rng = np.random.default_rng(seed)
    mo = _model_out(rng, B, 8, H, W, cond_first)
    x = rng.standard_normal((B, 4, H, W)).astype(F32)
    noise = rng.standard_normal((B, 4, H, W)).astype(F32) if has_noise else np.zeros((B, 4, H, W), F32)
    init = (0.8 * rng.standard_normal((B, 4, H, W))).astype(F32) if inp21 or inp22 else None
    mask = _mask(rng, B, H, W) if inp21 or inp22 else None
    rnoise = rng.standard_normal((B, 4, H, W)).astype(F32) if inp22 else None
    return mo, x, noise, init, mask, rnoise


@pytest.mark.gpu
@pytest.mark.parametrize("step", list(STEPS))
@pytest.mark.parametrize("B,H,W", SHAPES)
@pytest.mark.parametrize("path", list(PATHS))
def test_sampler_step_vs_float64(path, B, H, W, step):
    from kandinsky2 import ops
    cond_first, mode, clip, g, rows, inp21, inp22, _ = PATHS[path]
    coef = rows()[STEPS[step]]
    mo, x, noise, init, mask, rnoise = _step_inputs(path, B, H, W, seed=B * 1000 + H + W)
    n = B * 4 * H * W
    xd = _dev(x)
    work = torch.full((n + 4096,), float("nan"), device="cuda")
    dv = lambda a: None if a is None else _dev(a)
    ops.sampler_step(_dev(mo), xd, _dev(noise), _dev(coef), g, cond_first, clip=clip, threshold_mode=mode,
                     inpaint_init=dv(init), inpaint_mask=dv(mask), work=work, inpaint_noise=dv(rnoise))
    got, w = _host(xd), _host(work)
    x0_k = w[:n].reshape(x.shape)
    s = None
    if mode == 1:
        s = w[n]
        assert _bits(s) == _bits(_threshold(x0_k[0])), "the threshold must be the exact percentile of the kernel's x0"
    x0_ref, a_x0, ref, bound = _step_ref(mo, x, noise, coef, g, cond_first, clip, s, init, mask, rnoise)
    _assert_close(x0_k, x0_ref, a_x0, "x0")
    _assert_close(got, ref, bound, "x_{t-1}")
    if inp22:
        known = np.broadcast_to(mask == 1, x.shape)
        c = np.float64(coef[7])
        want = c * init.astype(np.float64) + np.sqrt(max(0.0, 1 - c * c)) * rnoise.astype(np.float64)
        _assert_close(got[known], want[known], bound[known], "2.2 known region")
        if step == "last":
            assert coef[7] == 1 and np.array_equal(_bits(got[known]), _bits(init[known])), \
                "the last step must return the clean latent in the known region"
    if step == "last" and path != "ddim":
        assert coef[6] == 0


# ------------------------------------------------------------------------------------------------
# 3. the split threshold modes of the sharded 2.1 path, on one GPU
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("inpaint", [False, True])
@pytest.mark.parametrize("B,H,W", [(4, 96, 96), (2, 16, 16)])
def test_split_threshold_modes(B, H, W, inpaint):
    from kandinsky2 import ops
    path = "p21_inpaint" if inpaint else "p21"
    cond_first, _, clip, g, rows, _, _, _ = PATHS[path]
    coef = _dev(rows()[STEPS["middle"]])
    mo, x, noise, init, mask, _ = _step_inputs(path, B, H, W, seed=11)
    n = B * 4 * H * W
    mo, noise = _dev(mo), _dev(noise)
    init, mask = (_dev(init), _dev(mask)) if inpaint else (None, None)

    def run(mode, work, xd=None):
        xd = _dev(x) if xd is None else xd
        ops.sampler_step(mo, xd, noise, coef, g, cond_first, clip=clip, threshold_mode=mode, inpaint_init=init,
                         inpaint_mask=mask, work=work)
        return xd

    def fresh():
        return torch.full((n + 4096,), float("nan"), device="cuda")

    w1 = fresh()
    x1 = _host(run(1, w1))
    w1 = _host(w1)
    # rank 0 of a sharded run: mode 2 then mode 3 on the same work buffer
    w23 = fresh()
    x23 = run(3, w23, run(2, w23))
    assert np.array_equal(_bits(_host(x23)), _bits(x1))
    assert np.array_equal(_bits(_host(w23)[:n + 1]), _bits(w1[:n + 1]))
    # the other ranks: mode 4 computes x0 only and leaves work[n] alone; the broadcast s then drives mode 3
    w4 = fresh()
    w4[n] = 12345.0
    x4 = run(4, w4)
    assert np.array_equal(_bits(_host(x4)), _bits(x)), "mode 4 must not update x"
    assert _host(w4)[n] == F32(12345.0), "mode 4 must not write the threshold"
    assert np.array_equal(_bits(_host(w4)[:n]), _bits(w1[:n]))
    w2 = fresh()
    run(2, w2)
    w4[n] = w2[n]
    x43 = run(3, w4, x4)
    assert np.array_equal(_bits(_host(x43)), _bits(x1))


# ------------------------------------------------------------------------------------------------
# 4. k2_plms_step
# ------------------------------------------------------------------------------------------------
def _plms_row(i, w):
    """PLMSSampler.sample's coefficient row for step i (DDIM schedule) with epsilon weights w."""
    s = _ddim()
    a_t, a_p = s.ddim_alphas[i], s.ddim_alphas_prev[i]
    return np.array([1.0 / np.sqrt(a_t), np.sqrt(1.0 - a_t) / np.sqrt(a_t), np.sqrt(a_p), np.sqrt(1.0 - a_p)] + list(w), F32)


def _plms_ref(mo, x, hist, coef, g, cond_first):
    """-> (e_t, its bound, x', its bound) in float64; None history entries contribute nothing."""
    B = x.shape[0]
    mo, x = mo.astype(np.float64), x.astype(np.float64)
    c = coef.astype(np.float64)
    cond, unc = (mo[:B], mo[B:]) if cond_first else (mo[B:], mo[:B])
    ec, eu = cond[:, :4], unc[:, :4]
    e_t = eu + g * (ec - eu)
    a_et = np.abs(eu) + g * np.abs(ec - eu)
    ep, a_ep = c[4] * e_t, abs(c[4]) * a_et
    for j, h in enumerate(hist):
        if h is not None:
            ep = ep + c[5 + j] * h.astype(np.float64)
            a_ep = a_ep + np.abs(c[5 + j] * h.astype(np.float64))
    x0 = c[0] * x - c[1] * ep
    a_x0 = np.abs(c[0] * x) + abs(c[1]) * a_ep
    return e_t, a_et, c[2] * x0 + c[3] * ep, abs(c[2]) * a_x0 + abs(c[3]) * a_ep


def _check_plms(hist_np, w, C2, cond_first, alias, store, B=2, H=96, W=96, seed=0):
    from kandinsky2 import ops
    rng = np.random.default_rng(seed)
    g = 7.0
    mo = _model_out(rng, B, C2, H, W, cond_first)
    x = rng.standard_normal((B, 4, H, W)).astype(F32)
    coef = _plms_row(30, w)
    xd = _dev(x)
    out = xd if alias else torch.full_like(xd, float("nan"))
    st = torch.full_like(xd, float("nan")) if store else None
    ops.plms_step(_dev(mo), xd, out, [None if h is None else _dev(h) for h in hist_np], st, _dev(coef), g, cond_first)
    e_t, a_et, ref, bound = _plms_ref(mo, x, hist_np, coef, g, cond_first)
    _assert_close(_host(out), ref, bound, "plms x'")
    if store:
        _assert_close(_host(st), e_t, a_et, "stored e_t")
    if not alias:
        assert np.array_equal(_bits(_host(xd)), _bits(x)), "x must be left alone when out is a separate buffer"


@pytest.mark.gpu
@pytest.mark.parametrize("cond_first", [0, 1])
@pytest.mark.parametrize("C2", [8, 4])
@pytest.mark.parametrize("depth", [0, 1, 2, 3, "euler"])
def test_plms_step_vs_float64(depth, C2, cond_first):
    """The calls PLMSSampler.sample makes: the first step's e_t into a separate output with the history slot stored, the
    improved-Euler (0.5, 0.5) row in place without a store, and Adams-Bashforth 2/3/4 in place storing e_t."""
    from kandinsky2.model.gaussian_diffusion import PLMSSampler
    rng = np.random.default_rng([C2, cond_first, 0 if depth == "euler" else depth + 1])
    hist = [(0.7 * rng.standard_normal((2, 4, 96, 96)) + 0.1 * j).astype(F32) for j in range(3)]
    if depth == 0:
        _check_plms([], (1.0, 0.0, 0.0, 0.0), C2, cond_first, alias=False, store=True)
    elif depth == "euler":
        _check_plms(hist[:1], (0.5, 0.5, 0.0, 0.0), C2, cond_first, alias=True, store=False)
    else:
        _check_plms(hist[:depth], PLMSSampler._AB[depth], C2, cond_first, alias=True, store=True)


@pytest.mark.gpu
def test_plms_step_skips_missing_history():
    from kandinsky2.model.gaussian_diffusion import PLMSSampler
    rng = np.random.default_rng(5)
    hist = [(0.7 * rng.standard_normal((2, 4, 96, 96))).astype(F32) for _ in range(3)]
    _check_plms([hist[0], None, hist[2]], PLMSSampler._AB[3], 8, 1, alias=True, store=True)
    _check_plms([None, hist[1], None], PLMSSampler._AB[3], 8, 0, alias=False, store=True)


# ------------------------------------------------------------------------------------------------
# 5. k2_step_begin / k2_step_end inside one captured CUDA graph
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("with_noise", [True, False])
def test_step_begin_end_graph_wraps(with_noise):
    from kandinsky2 import ops
    rng = np.random.default_rng(3)
    B, H, W, n_steps = 2, 16, 24, 5
    shape = (B, 4, H, W)
    # the tables are longer than the schedule (as FusedStep's are): a counter that did not wrap would read other values
    rows = n_steps + 3
    ts_seq = _dev(rng.uniform(0, 1000, rows))
    coef_seq = _dev(rng.standard_normal((rows, 8)))
    noise_seq = _dev(rng.standard_normal((rows,) + shape)) if with_noise else None
    x = _dev(rng.standard_normal(shape))
    x_in = torch.full((2 * B, 4, H, W), float("nan"), device="cuda")
    t_in = torch.full((2 * B,), float("nan"), device="cuda")
    coef_out = torch.full((8,), float("nan"), device="cuda")
    noise = torch.full(shape, -7.0, device="cuda")
    counter = torch.tensor([0, n_steps], dtype=torch.int32, device="cuda")

    def launch():
        ops.step_begin(x, x_in, t_in, coef_out, ts_seq, coef_seq, noise_seq, noise, counter)
        ops.step_end(counter)

    launch()  # warm-up outside the capture (one-time launch attributes)
    torch.cuda.synchronize()
    noise.fill_(-7.0)
    counter.copy_(torch.tensor([0, n_steps], dtype=torch.int32))
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        launch()
    torch.cuda.synchronize()
    assert _host(counter)[0] == 0, "capturing must not run the step"
    ts_h, coef_h = _host(ts_seq), _host(coef_seq)
    noise_h = _host(noise_seq) if with_noise else None
    for r in range(n_steps + 2):
        x.copy_(_dev(rng.standard_normal(shape)))
        graph.replay()
        torch.cuda.synchronize()
        k = r % n_steps
        xh = _host(x)
        assert np.array_equal(_bits(_host(x_in)), _bits(np.concatenate([xh, xh]))), r
        assert np.array_equal(_bits(_host(t_in)), _bits(np.full(2 * B, ts_h[k], F32))), r
        assert np.array_equal(_bits(_host(coef_out)), _bits(coef_h[k])), r
        if with_noise:
            assert np.array_equal(_bits(_host(noise)), _bits(noise_h[k])), r
        else:
            assert (_host(noise) == F32(-7.0)).all(), "without a noise table the noise buffer is left alone"
    assert _host(counter).tolist() == [n_steps + 2, n_steps]
