"""GPU parity of the non-conv kernels (attention, GroupNorm, small dense layers, MoVQ helpers) against plain torch fp32
on the same inputs (the sampler-step kernels are in test_gpu_sampler_step.py).  Tolerances are the fp16-storage
tolerances stated per test."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _ref_attention(qkv, enc, heads):
    """unet.py:286-340 restated on [B, T, heads*192] / [B, Tc, heads*128] rows (fp32)."""
    B, T, _ = qkv.shape
    q, k, v = qkv.float().reshape(B, T, heads, 3, 64).unbind(3)
    if enc is not None:
        ek, ev = enc.float().reshape(B, enc.shape[1], heads, 2, 64).unbind(3)
        k = torch.cat([ek, k], 1)
        v = torch.cat([ev, v], 1)
    w = torch.einsum("bthd,bshd->bhts", q, k) / 8.0
    w = torch.softmax(w, -1)
    return torch.einsum("bhts,bshd->bthd", w, v).reshape(B, T, heads * 64)


ATTN_DEFAULT_LAYOUT = 1  # k2_api.cu g_attn_half
ATTN_DEFAULT_STAGGER = 1200  # k2_api.cu g_attn_stagger


@pytest.mark.parametrize("B,heads,T,Tc", [
    (2, 2, 64, 17),      # golden tiny config: one partial block each
    (1, 3, 144, 32),     # level-3 geometry: 2 query tiles, ragged key tail
    (2, 12, 576, 87),    # level-2 geometry, 2.1 context length
    (1, 2, 2304, 32),    # level-1 geometry: 18 query tiles x 19 key blocks
    (1, 1, 256, 0),      # no encoder tokens
    (1, 1, 130, 200),    # encoder longer than one block
])
@pytest.mark.parametrize("half_rows", [0, 1])
def test_attention_d64(B, heads, T, Tc, half_rows):
    """both softmax layouts of k2_attention_d64 (tuning key 9: one thread per score row / half a row per thread) and, for the
    level-1 geometry, the MUFU-free exp2 on 2/8 of the scores (key 6)"""
    from kandinsky2 import ops
    g = torch.Generator(device="cuda").manual_seed(0)
    qkv = torch.randn(B, T, heads * 192, device="cuda", generator=g).half()
    enc = torch.randn(B, Tc, heads * 128, device="cuda", generator=g).half() if Tc else None
    ops.set_tuning(9, half_rows)
    ops.set_tuning(6, 2 if T == 2304 else 0)
    try:
        out = ops.attention_d64(qkv, heads, enc)
        torch.cuda.synchronize()
    finally:
        ops.set_tuning(9, ATTN_DEFAULT_LAYOUT)
        ops.set_tuning(6, 0)
    ref = _ref_attention(qkv, enc, heads)
    err = (out.float() - ref).abs().max().item()
    # P is rounded to fp16 before PV (as in the reference's fp16 mode, unet.py:338): abs tol 4e-3 on O(1) values
    assert err < 4e-3, err
    rel = ((out.float() - ref).norm() / ref.norm()).item()
    assert rel < 2e-3, rel


@pytest.mark.parametrize("half_rows", [0, 1])
def test_attention_d64_modes_bit_identical(half_rows):
    """The start-up offset of the second query tile (tuning key 5; each tile has its own MMA issuer) only moves work in time,
    and the packed FFMA2 / FADD2 softmax arithmetic (key 6 + 10 / + 30) rounds exactly like the scalar instructions: the
    output must not change by a bit.  T = 600 gives two full query tiles per CTA plus a ragged third CTA."""
    from kandinsky2 import ops
    g = torch.Generator(device="cuda").manual_seed(3)
    B, heads, T, Tc = 2, 3, 600, 32
    qkv = torch.randn(B, T, heads * 192, device="cuda", generator=g).half()
    enc = torch.randn(B, Tc, heads * 128, device="cuda", generator=g).half()
    ops.set_tuning(9, half_rows)
    outs = {}
    try:
        for mode, stagger in ((0, 1200), (0, 0), (0, 5000), (10, 1200), (30, 1200), (1, 1200), (31, 300)):
            ops.set_tuning(6, mode)
            ops.set_tuning(5, stagger)
            outs[(mode, stagger)] = ops.attention_d64(qkv, heads, enc)
        torch.cuda.synchronize()
    finally:
        ops.set_tuning(9, ATTN_DEFAULT_LAYOUT)
        ops.set_tuning(6, 0)
        ops.set_tuning(5, ATTN_DEFAULT_STAGGER)
    ref = _ref_attention(qkv, enc, heads)
    assert (outs[(0, 1200)].float() - ref).abs().max().item() < 4e-3
    for key in ((0, 0), (0, 5000), (10, 1200), (30, 1200)):
        assert torch.equal(outs[key], outs[(0, 1200)]), key
    assert torch.equal(outs[(31, 300)], outs[(1, 1200)])
    assert (outs[(1, 1200)].float() - ref).abs().max().item() < 4e-3


@pytest.mark.parametrize("half_rows", [0, 1])
def test_attention_large_logits(half_rows):
    """online-softmax rescaling: strongly peaked rows whose maximum moves between key blocks."""
    from kandinsky2 import ops
    g = torch.Generator(device="cuda").manual_seed(1)
    B, heads, T = 1, 2, 512
    qkv = (torch.randn(B, T, heads * 192, device="cuda", generator=g) * 3).half()
    ops.set_tuning(9, half_rows)
    try:
        out = ops.attention_d64(qkv, heads, None)
    finally:
        ops.set_tuning(9, ATTN_DEFAULT_LAYOUT)
    ref = _ref_attention(qkv, None, heads)
    assert torch.isfinite(out).all()
    assert (out.float() - ref).abs().max().item() < 3e-2


@pytest.mark.parametrize("NB,H,W,C0,C1", [(2, 16, 16, 64, 0), (3, 12, 12, 128, 64), (1, 96, 96, 384, 0), (8, 4, 4, 1536, 1536)])
def test_gn_stats_apply(NB, H, W, C0, C1):
    from kandinsky2 import ops
    g = torch.Generator(device="cuda").manual_seed(2)
    C = C0 + C1
    buf = (torch.randn(NB, H, W, C + 8, device="cuda", generator=g) * 2 + 0.5).half()
    x0 = buf[..., :C0]
    x1 = buf[..., C0:C] if C1 else None
    gamma = torch.randn(C, device="cuda", generator=g)
    beta = torch.randn(C, device="cuda", generator=g)
    film = torch.randn(NB, 2 * C, device="cuda", generator=g) * 0.3
    st = ops.gn_stats(x0, x1, groups=32, eps=1e-5)
    xcat = buf[..., :C].float().permute(0, 3, 1, 2)
    xg = xcat.reshape(NB, 32, -1)
    assert torch.allclose(st[..., 0], xg.mean(-1), atol=1e-4)
    assert torch.allclose(st[..., 1], 1 / torch.sqrt(xg.var(-1, unbiased=False) + 1e-5), rtol=1e-4)
    ref_n = F.group_norm(xcat, 32, gamma, beta, 1e-5)
    # plain GN + SiLU
    y = ops.gn_apply(x0, x1, st, gamma, beta, act=1)
    assert (y.float().permute(0, 3, 1, 2) - F.silu(ref_n)).abs().max().item() < 2e-2
    # FiLM + SiLU
    sc, sh = film[:, :C, None, None], film[:, C:, None, None]
    y = ops.gn_apply(x0, x1, st, gamma, beta, film=film, act=1)
    assert (y.float().permute(0, 3, 1, 2) - F.silu(ref_n * (1 + sc) + sh)).abs().max().item() < 3e-2
    # no activation (attention norm)
    y = ops.gn_apply(x0, x1, st, gamma, beta, act=0)
    assert (y.float().permute(0, 3, 1, 2) - ref_n).abs().max().item() < 2e-2
    # down / up resampling of both branches
    y, xr = ops.gn_apply(x0, x1, st, gamma, beta, act=1, resample=1, want_xres=True)
    assert (y.float().permute(0, 3, 1, 2) - F.avg_pool2d(F.silu(ref_n), 2)).abs().max().item() < 2e-2
    assert (xr.float().permute(0, 3, 1, 2) - F.avg_pool2d(xcat, 2)).abs().max().item() < 1e-2
    y, xr = ops.gn_apply(x0, x1, st, gamma, beta, act=1, resample=2, want_xres=True)
    assert (y.float().permute(0, 3, 1, 2) - F.interpolate(F.silu(ref_n), scale_factor=2)).abs().max().item() < 2e-2
    assert (xr.float().permute(0, 3, 1, 2) - F.interpolate(xcat, scale_factor=2)).abs().max().item() == 0


def test_spatial_norm():
    from kandinsky2 import ops
    g = torch.Generator(device="cuda").manual_seed(3)
    NB, H, W, C = 2, 16, 16, 64
    x = torch.randn(NB, H, W, C, device="cuda", generator=g).half()
    zq = torch.randn(NB, 4, 8, 8, device="cuda", generator=g)
    gamma = torch.randn(C, device="cuda", generator=g); beta = torch.randn(C, device="cuda", generator=g)
    wy = torch.randn(C, 4, device="cuda", generator=g); by = torch.randn(C, device="cuda", generator=g)
    wb = torch.randn(C, 4, device="cuda", generator=g); bb = torch.randn(C, device="cuda", generator=g)
    st = ops.gn_stats(x, None, groups=32, eps=1e-6)
    sn_w = torch.cat([wy, by[:, None], wb, bb[:, None]], 1).contiguous()
    y = ops.gn_apply(x, None, st, gamma, beta, act=1, zq=ops.nchw_to_nhwc_f32(zq), sn_w=sn_w)
    xc = x.float().permute(0, 3, 1, 2)
    z = F.interpolate(zq, size=(H, W), mode="nearest")
    ref = F.group_norm(xc, 32, gamma, beta, 1e-6) * F.conv2d(z, wy[:, :, None, None], by) + F.conv2d(z, wb[:, :, None, None], bb)
    ref = ref * torch.sigmoid(ref)
    assert (y.float().permute(0, 3, 1, 2) - ref).abs().max().item() < 5e-2


def test_linear_layernorm_temb():
    from kandinsky2 import ops
    g = torch.Generator(device="cuda").manual_seed(4)
    M, K, N = 8, 1536, 3072
    x = torch.randn(M, K, device="cuda", generator=g)
    W = (torch.randn(N, K, device="cuda", generator=g) / K ** 0.5)
    b = torch.randn(N, device="cuda", generator=g)
    y = ops.linear(x, W, b, silu_in=True)
    assert torch.allclose(y, F.linear(F.silu(x), W, b), atol=2e-4, rtol=1e-4)
    y = ops.linear(x, W.half(), b, silu_out=True)
    assert torch.allclose(y, F.silu(F.linear(x, W.half().float(), b)), atol=2e-4, rtol=1e-4)
    x2 = torch.randn(5, 100, device="cuda", generator=g)
    W2 = torch.randn(37, 100, device="cuda", generator=g)
    add = torch.randn(5, 37, device="cuda", generator=g)
    assert torch.allclose(ops.linear(x2, W2, None, add=add), F.linear(x2, W2) + add, atol=1e-4, rtol=1e-4)
    ga = torch.randn(N, device="cuda", generator=g); be = torch.randn(N, device="cuda", generator=g)
    xx = torch.randn(M, N, device="cuda", generator=g) * 3 + 1
    assert torch.allclose(ops.layernorm(xx, ga, be), F.layer_norm(xx, (N,), ga, be), atol=1e-4, rtol=1e-4)
    t = torch.tensor([999.0, 0.0, 500.5, 20.0], device="cuda")
    emb = ops.timestep_embedding(t, 384)
    half = 192
    freqs = torch.exp(-math.log(10000) * torch.arange(half, dtype=torch.float32, device="cuda") / half)
    ref = torch.cat([torch.cos(t[:, None] * freqs), torch.sin(t[:, None] * freqs)], -1)
    assert (emb - ref).abs().max().item() < 2e-4
    # known-answer constants from the reference (SURVEY.md section 8c)
    assert abs(emb[0, 0].item() - 0.99964982) < 1e-4 and abs(emb[0, 192].item() + 0.02646075) < 2e-4


def test_stem_im2col_matches_conv():
    from kandinsky2 import ops
    g = torch.Generator(device="cuda").manual_seed(5)
    NB, H, W = 2, 12, 10
    x = torch.randn(NB, 4, H, W, device="cuda", generator=g)
    img = torch.randn(NB, 4, H, W, device="cuda", generator=g)
    mask = (torch.rand(NB, 1, H, W, device="cuda", generator=g) > 0.5).float()
    w = torch.randn(64, 9, 3, 3, device="cuda", generator=g) / 9
    bias = torch.randn(64, device="cuda", generator=g)
    patches = ops.stem_im2col(x, img, mask, mul23=True)
    y = ops.gemm_rows(patches, ops.pack_stem_weight(w), 64, bias=bias)
    ref = F.conv2d(torch.cat([x, img * mask, mask], 1).half().float(), w.half().float(), bias, padding=1)
    assert (y.float().permute(0, 3, 1, 2) - ref).abs().max().item() < 2e-2


def test_vq_argmin_bit_exact():
    from kandinsky2 import ops
    g = torch.Generator(device="cuda").manual_seed(7)
    cb = torch.randn(16384, 4, device="cuda", generator=g)
    z = torch.randn(4096, 4, device="cuda", generator=g)
    idx = ops.vq_argmin(z, cb)
    # same operation order as the kernel, evaluated densely in fp32 without fused multiply-adds
    zz = ((z[:, 0] * z[:, 0] + z[:, 1] * z[:, 1]) + z[:, 2] * z[:, 2]) + z[:, 3] * z[:, 3]
    best = torch.cdist(z.double(), cb.double()).argmin(1)
    # the fp32 argmin may differ from the fp64 one only on near-ties: check distance optimality instead
    d_k = (z - cb[idx]).double().pow(2).sum(1)
    d_b = (z - cb[best]).double().pow(2).sum(1)
    assert ((d_k - d_b) <= 1e-5 * (1 + d_b)).all()
    assert (idx == best).float().mean().item() > 0.999


def test_images_to_u8():
    from kandinsky2 import ops
    x = torch.linspace(-1.2, 1.2, 2 * 3 * 8 * 8, device="cuda").reshape(2, 3, 8, 8)
    out = ops.images_to_u8(x, 6, 7)
    ref = ((x + 1) * 127.5).round().clamp(0, 255).to(torch.uint8)[:, :, :6, :7].permute(0, 2, 3, 1)
    assert torch.equal(out, ref)


@pytest.mark.parametrize("NB,H,W,C0,C1,resample", [(8, 24, 24, 1152, 0, 0), (2, 48, 48, 768, 384, 0), (8, 12, 12, 1536, 0, 2),
                                                   (2, 24, 24, 256, 0, 1)])
def test_gn_apply_fold_matches_finalize_plus_apply(NB, H, W, C0, C1, resample):
    """k2_gn_apply_fold (statistics folded from the producers' partial sums inside the apply kernel) against the
    k2_gn_finalize + k2_gn_apply pair."""
    from kandinsky2 import ops
    g = torch.Generator(device="cuda").manual_seed(11)
    outs, parts, rgs = [], [], []
    for cout in [C0] + ([C1] if C1 else []):
        x = torch.randn(NB, H, W, 64, device="cuda", generator=g).half()
        w = torch.randn(cout, 64, 3, 3, device="cuda", generator=g) / 24
        part = torch.zeros(ops.gn_part_floats(NB, H, W, cout), device="cuda")
        info = [0] * 7
        outs.append(ops.conv_gemm([(x, 9)], ops.pack_conv_weight(w), cout, gn_part=part, info=info))
        assert info[5] in (1, 2), info
        parts.append(part)
        rgs.append(info[6] // NB)
    C = C0 + C1
    gamma, beta = torch.randn(C, device="cuda", generator=g), torch.randn(C, device="cuda", generator=g)
    film = torch.randn(NB, 2 * C, device="cuda", generator=g)
    st = torch.empty(NB, 32, 2, device="cuda")
    ops.gn_finalize(parts[0], C0, parts[1] if C1 else None, C1, NB, rgs[0], H * W, st, rg1=rgs[1] if C1 else None)
    ref = ops.gn_apply(outs[0], outs[1] if C1 else None, st, gamma, beta, film=film, act=1, resample=resample)
    got = ops.gn_apply_fold(outs[0], outs[1] if C1 else None, parts[0], rgs[0], parts[1] if C1 else None,
                            rgs[1] if C1 else 0, gamma, beta, film=film, act=1, resample=resample)
    torch.cuda.synchronize()
    assert (got.float() - ref.float()).abs().max().item() <= 2e-3 * max(1.0, ref.float().abs().max().item())


@pytest.mark.parametrize("NB,H,W,C,zs,act", [(2, 16, 16, 512, 1, 0), (2, 32, 48, 256, 2, 1), (1, 64, 64, 128, 8, 1), (3, 24, 40, 128, 4, 1)])
def test_sn_apply(NB, H, W, C, zs, act):
    """k2_sn_apply (MoVQ SpatialNorm + swish, movq_modules.py:61-68,21-23) against torch fp32 on the same fp16 activations."""
    from kandinsky2 import ops
    g = torch.Generator(device="cuda").manual_seed(31)
    x = (torch.randn(NB, H, W, C, device="cuda", generator=g) * 1.5 + 0.3).half()
    zq = torch.randn(NB, H // zs, W // zs, 4, device="cuda", generator=g)
    gamma = 1 + 0.1 * torch.randn(C, device="cuda", generator=g)
    beta = 0.1 * torch.randn(C, device="cuda", generator=g)
    wy, by = torch.randn(C, 4, device="cuda", generator=g) / 2, torch.randn(C, device="cuda", generator=g) / 4 + 1
    wb, bb = torch.randn(C, 4, device="cuda", generator=g) / 2, torch.randn(C, device="cuda", generator=g) / 4
    sn_w = torch.cat([wy, by[:, None], wb, bb[:, None]], 1).contiguous()
    st = ops.gn_stats(x, None, eps=1e-6)
    y = ops.sn_apply(x, st, gamma, beta, zq, sn_w, act=act)
    torch.cuda.synchronize()
    xn = F.group_norm(x.float().permute(0, 3, 1, 2), 32, gamma, beta, eps=1e-6)
    zu = F.interpolate(zq.permute(0, 3, 1, 2), size=(H, W), mode="nearest")
    ref = xn * (F.conv2d(zu, wy[:, :, None, None], by)) + F.conv2d(zu, wb[:, :, None, None], bb)
    if act:
        ref = ref * torch.sigmoid(ref)
    ref = ref.permute(0, 2, 3, 1)
    err = (y.float() - ref).abs().max().item()
    assert err <= 3e-3 * max(1.0, ref.abs().max().item()), err


def test_transpose_and_batched_gemm():
    """k2_transpose_f16 and the batched k2_conv_gemm_cfg (w_batch_stride): the MoVQ AttnBlock's scores = q k^T and out = P v
    for all images in one launch each (movq_modules.py:209-219)."""
    from kandinsky2 import ops
    g = torch.Generator(device="cuda").manual_seed(32)
    B, T, C = 3, 320, 128   # T / 128 = 2.5 boxes per image: odd box count, the pair kernel must not straddle images
    qkv = torch.randn(B, T, 3 * C, device="cuda", generator=g).half()
    vT = ops.transpose_f16(qkv[:, :, 2 * C:])
    assert torch.equal(vT, qkv[:, :, 2 * C:].transpose(1, 2).contiguous())
    scores = torch.empty(B, T, T, device="cuda", dtype=torch.float16)
    ops.conv_gemm([(qkv[:, :, :C].unsqueeze(1), 1)], qkv[0, :, C:2 * C], T, out=scores.view(B, 1, T, T), w_batch_stride=T * 3 * C)
    ref = torch.einsum("btc,bsc->bts", qkv[:, :, :C].float(), qkv[:, :, C:2 * C].float())
    assert ((scores.float() - ref).norm() / ref.norm()).item() < 1e-3
    p = torch.softmax(ref * C ** -0.5, -1).half()
    o = torch.empty(B, T, C, device="cuda", dtype=torch.float16)
    ops.conv_gemm([(p.view(B, 1, T, T), 1)], vT[0], C, out=o.view(B, 1, T, C), w_batch_stride=C * T)
    torch.cuda.synchronize()
    ref_o = torch.einsum("bts,bsc->btc", p.float(), qkv[:, :, 2 * C:].float())
    assert ((o.float() - ref_o).norm() / ref_o.norm()).item() < 1e-3


@pytest.mark.parametrize("B,T", [(2, 384), (1, 1152), (2, 320)])
def test_attention_d512(B, T):
    """k2_attention_d512 (the MoVQ AttnBlock's softmax(q k^T / sqrt(512)) v, one head of width 512, fused) against torch fp32 on
    the same fp16 q / k / v; T = 320 exercises a ragged last key block and query tile."""
    from kandinsky2 import ops
    g = torch.Generator(device="cuda").manual_seed(41)
    qkv = torch.randn(B, T, 1536, device="cuda", generator=g).half()
    qkv[:, :, :512] *= 2.0   # sharper softmax: exercises the running-maximum logic
    out = ops.attention_d512(qkv, 512 ** -0.5)
    torch.cuda.synchronize()
    q, k, v = qkv.float().split(512, dim=-1)
    ref = torch.softmax(torch.einsum("btc,bsc->bts", q, k) * 512 ** -0.5, dim=-1) @ v
    err = (out.float() - ref).abs().max().item()
    rel = ((out.float() - ref).norm() / ref.norm()).item()
    assert rel < 3e-3 and err < 2e-2 * max(1.0, ref.abs().max().item()), (rel, err)
