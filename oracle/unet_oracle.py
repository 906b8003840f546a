"""Oracle: torch-fp32 restatement of the reference UNet denoiser (TEST INFRASTRUCTURE -- see oracle/__init__.py).

Follows, function by function (paths relative to /root/reference/kandinsky2/model):
  topology / parameter names   unet.py:372-563 (UNetModel.__init__), text2im_model2_1.py:14-47
  timestep_embedding           nn.py:101-121
  ResBlock.forward             unet.py:193-220   (GroupNorm32 nn.py:31-37; Upsample :67-77; Downsample :105-107)
  AttentionBlock.forward       unet.py:260-269
  QKVAttention.forward         unet.py:286-340   (non-flash branch :333-340)
  Text2ImUNet.get_text_emb     text2im_model2_1.py:57-80
  Text2ImUNet.forward          text2im_model2_1.py:85-103
  InpaintText2ImUNet.forward   text2im_model2_1.py:146-155
It is written against a flat state dict with the reference's key names, so the same synthetic weights
drive the reference (oracle/make_golden.py), this oracle, and the CUDA product.

cond == "2.2" swaps the conditioning head for the Kandinsky-2.2 one (diffusers ImageProjection +
ImageTimeEmbedding; NOT in /root/reference -> that head is "parity unpinned", restated from the published
diffusers algorithm: image_embeds -> Linear(1280, 32*768) -> LayerNorm(768) tokens; Linear(1280,1536) ->
LayerNorm -> added to the time embedding).  The backbone is identical.
"""
import math

import torch
import torch.nn.functional as F

CONFIG_2_1 = dict(  # configs.py:125-149 resolved through model_creation.py:33-48
    in_channels=4, model_channels=384, out_channels=8, num_res_blocks=3, attention_ds=(2, 4, 8),
    channel_mult=(1, 2, 3, 4), num_head_channels=64, model_dim=768, image_encoder_in_dim=768,
    text_encoder_in_dim1=1024, text_encoder_in_dim2=768, num_image_embs=10, inpainting=False, cond="2.1")

CONFIG_2_2 = dict(CONFIG_2_1, image_encoder_in_dim=1280, num_image_embs=32, cond="2.2")

CONFIG_TINY = dict(  # small enough for committed golden vectors; exercises every layer kind
    in_channels=4, model_channels=64, out_channels=8, num_res_blocks=1, attention_ds=(2,),
    channel_mult=(1, 2), num_head_channels=64, model_dim=128, image_encoder_in_dim=48,
    text_encoder_in_dim1=96, text_encoder_in_dim2=48, num_image_embs=3, inpainting=False, cond="2.1")


def unet_topology(cfg):
    """Layer list of the three stages. Each block is a list of ('conv'|'res'|'attn', ...) tuples.
    res = ('res', cin, cout, updown) with updown in {None, 'down', 'up'}.  (unet.py:421-557)"""
    mc, mult, nrb = cfg["model_channels"], cfg["channel_mult"], cfg["num_res_blocks"]
    cin = cfg["in_channels"] * 2 + 1 if cfg.get("inpainting") else cfg["in_channels"]
    ch = mult[0] * mc
    inp = [[("conv", cin, ch)]]
    chans = [ch]
    ds = 1
    for level, m in enumerate(mult):
        for _ in range(nrb):
            blk = [("res", ch, m * mc, None)]
            ch = m * mc
            if ds in cfg["attention_ds"]:
                blk.append(("attn", ch))
            inp.append(blk)
            chans.append(ch)
        if level != len(mult) - 1:
            inp.append([("res", ch, ch, "down")])
            chans.append(ch)
            ds *= 2
    mid = [("res", ch, ch, None), ("attn", ch), ("res", ch, ch, None)]
    out = []
    for level, m in list(enumerate(mult))[::-1]:
        for i in range(nrb + 1):
            ich = chans.pop()
            blk = [("res", ch + ich, m * mc, None)]
            ch = m * mc
            if ds in cfg["attention_ds"]:
                blk.append(("attn", ch))
            if level and i == nrb:
                blk.append(("res", ch, ch, "up"))
                ds //= 2
            out.append(blk)
    return inp, mid, out


def _res_spec(p, cin, cout, spec, temb):
    spec += [(p + "in_layers.0.weight", (cin,)), (p + "in_layers.0.bias", (cin,)),
             (p + "in_layers.2.weight", (cout, cin, 3, 3)), (p + "in_layers.2.bias", (cout,)),
             (p + "emb_layers.1.weight", (2 * cout, temb)), (p + "emb_layers.1.bias", (2 * cout,)),
             (p + "out_layers.0.weight", (cout,)), (p + "out_layers.0.bias", (cout,)),
             (p + "out_layers.3.weight", (cout, cout, 3, 3)), (p + "out_layers.3.bias", (cout,))]
    if cin != cout:
        spec += [(p + "skip_connection.weight", (cout, cin, 1, 1)), (p + "skip_connection.bias", (cout,))]


def _attn_spec(p, ch, enc, spec):
    spec += [(p + "norm.weight", (ch,)), (p + "norm.bias", (ch,)),
             (p + "qkv.weight", (3 * ch, ch, 1)), (p + "qkv.bias", (3 * ch,)),
             (p + "encoder_kv.weight", (2 * ch, enc, 1)), (p + "encoder_kv.bias", (2 * ch,)),
             (p + "proj_out.weight", (ch, ch, 1)), (p + "proj_out.bias", (ch,))]


def unet_param_spec(cfg):
    """[(state_dict key, shape)] in the reference's registration order."""
    mc = cfg["model_channels"]
    temb = 4 * mc
    md = cfg["model_dim"]
    spec = [("time_embed.0.weight", (temb, mc)), ("time_embed.0.bias", (temb,)),
            ("time_embed.2.weight", (temb, temb)), ("time_embed.2.bias", (temb,))]
    inp, mid, out = unet_topology(cfg)

    def stage(prefix, blocks):
        for bi, blk in enumerate(blocks):
            for li, layer in enumerate(blk):
                p = f"{prefix}.{bi}.{li}." if prefix != "middle_block" else f"{prefix}.{li}."
                if layer[0] == "conv":
                    spec.extend([(p + "weight", (layer[2], layer[1], 3, 3)), (p + "bias", (layer[2],))])
                elif layer[0] == "res":
                    _res_spec(p, layer[1], layer[2], spec, temb)
                else:
                    _attn_spec(p, layer[1], md, spec)

    stage("input_blocks", inp)
    stage("middle_block", [mid])
    stage("output_blocks", out)
    ch0 = cfg["channel_mult"][0] * mc
    spec += [("out.0.weight", (ch0,)), ("out.0.bias", (ch0,)),
             ("out.2.weight", (cfg["out_channels"], ch0, 3, 3)), ("out.2.bias", (cfg["out_channels"],))]
    ie = cfg["image_encoder_in_dim"]
    if cfg.get("cond", "2.1") == "2.1":
        spec += [("clip_to_seq.weight", (md * cfg["num_image_embs"], ie)), ("clip_to_seq.bias", (md * cfg["num_image_embs"],)),
                 ("to_model_dim_n.weight", (md, cfg["text_encoder_in_dim1"])), ("to_model_dim_n.bias", (md,)),
                 ("proj_n.weight", (temb, cfg["text_encoder_in_dim2"])), ("proj_n.bias", (temb,)),
                 ("ln_model_n.weight", (temb,)), ("ln_model_n.bias", (temb,)),
                 ("img_layer.weight", (temb, ie)), ("img_layer.bias", (temb,))]
    else:
        spec += [("encoder_hid_proj.image_embeds.weight", (md * cfg["num_image_embs"], ie)),
                 ("encoder_hid_proj.image_embeds.bias", (md * cfg["num_image_embs"],)),
                 ("encoder_hid_proj.norm.weight", (md,)), ("encoder_hid_proj.norm.bias", (md,)),
                 ("add_embedding.image_proj.weight", (temb, ie)), ("add_embedding.image_proj.bias", (temb,)),
                 ("add_embedding.image_norm.weight", (temb,)), ("add_embedding.image_norm.bias", (temb,))]
    return spec


# ------------------------------------------------------------------------------------------------
def timestep_embedding(t, dim, max_period=10000):  # nn.py:101-121 (cos first)
    half = dim // 2
    freqs = torch.exp(-math.log(max_period) * torch.arange(half, dtype=torch.float32, device=t.device) / half)
    args = t[:, None].float() * freqs[None]
    emb = torch.cat([torch.cos(args), torch.sin(args)], dim=-1)
    if dim % 2:
        emb = torch.cat([emb, torch.zeros_like(emb[:, :1])], dim=-1)
    return emb


def _gn(x, sd, p, swish):  # GroupNorm32, 32 groups, eps 1e-5
    y = F.group_norm(x.float(), 32, sd[p + "weight"].float(), sd[p + "bias"].float(), 1e-5).to(x.dtype)
    return F.silu(y) if swish else y


def _res(x, emb, sd, p, updown):
    h = _gn(x, sd, p + "in_layers.0.", True)
    if updown == "up":
        h = F.interpolate(h, scale_factor=2, mode="nearest")
        x = F.interpolate(x, scale_factor=2, mode="nearest")
    elif updown == "down":
        h = F.avg_pool2d(h, 2, 2)
        x = F.avg_pool2d(x, 2, 2)
    h = F.conv2d(h, sd[p + "in_layers.2.weight"], sd[p + "in_layers.2.bias"], padding=1)
    e = F.linear(F.silu(emb), sd[p + "emb_layers.1.weight"], sd[p + "emb_layers.1.bias"]).to(h.dtype)
    scale, shift = e[:, :, None, None].chunk(2, dim=1)
    h = _gn(h, sd, p + "out_layers.0.", False) * (1 + scale) + shift
    h = F.conv2d(F.silu(h), sd[p + "out_layers.3.weight"], sd[p + "out_layers.3.bias"], padding=1)
    if (p + "skip_connection.weight") in sd:
        x = F.conv2d(x, sd[p + "skip_connection.weight"], sd[p + "skip_connection.bias"])
    return x + h


def qkv_attention(qkv, enc_kv, heads):  # unet.py:286-340
    bs, width, length = qkv.shape
    ch = width // (3 * heads)
    q, k, v = qkv.reshape(bs * heads, ch * 3, length).split(ch, dim=1)
    if enc_kv is not None:
        ek, ev = enc_kv.reshape(bs * heads, ch * 2, -1).split(ch, dim=1)
        k = torch.cat([ek, k], dim=-1)
        v = torch.cat([ev, v], dim=-1)
    scale = 1 / math.sqrt(math.sqrt(ch))
    w = torch.einsum("bct,bcs->bts", q * scale, k * scale)
    w = torch.softmax(w.float(), dim=-1).type(w.dtype)
    a = torch.einsum("bts,bcs->bct", w, v)
    return a.reshape(bs, -1, length)


def _attn(x, xf_out, sd, p, head_ch):
    b, c, hh, ww = x.shape
    qkv = F.conv1d(_gn(x, sd, p + "norm.", False).view(b, c, -1), sd[p + "qkv.weight"], sd[p + "qkv.bias"])
    enc = F.conv1d(xf_out, sd[p + "encoder_kv.weight"], sd[p + "encoder_kv.bias"])
    h = qkv_attention(qkv, enc, c // head_ch)
    h = F.conv1d(h, sd[p + "proj_out.weight"], sd[p + "proj_out.bias"])
    return x + h.reshape(b, c, hh, ww)


def conditioning(sd, cfg, full_emb=None, pooled_emb=None, image_emb=None):
    """-> (xf_proj [N, 4*mc], xf_out [N, model_dim, ctx])"""
    md = cfg["model_dim"]
    if cfg.get("cond", "2.1") == "2.1":  # text2im_model2_1.py:57-80, pooling_type 'from_model'
        clip_seq = F.linear(image_emb, sd["clip_to_seq.weight"], sd["clip_to_seq.bias"]).reshape(
            image_emb.shape[0], cfg["num_image_embs"], md)
        xf_proj = F.linear(pooled_emb, sd["proj_n.weight"], sd["proj_n.bias"])
        xf_proj = F.layer_norm(xf_proj, xf_proj.shape[-1:], sd["ln_model_n.weight"], sd["ln_model_n.bias"])
        xf_proj = xf_proj + F.linear(image_emb, sd["img_layer.weight"], sd["img_layer.bias"])
        xf_out = torch.cat((clip_seq, F.linear(full_emb, sd["to_model_dim_n.weight"], sd["to_model_dim_n.bias"])), dim=1)
        return xf_proj, xf_out.permute(0, 2, 1)
    tok = F.linear(image_emb, sd["encoder_hid_proj.image_embeds.weight"], sd["encoder_hid_proj.image_embeds.bias"])
    tok = tok.reshape(image_emb.shape[0], cfg["num_image_embs"], md)
    tok = F.layer_norm(tok, (md,), sd["encoder_hid_proj.norm.weight"], sd["encoder_hid_proj.norm.bias"])
    add = F.linear(image_emb, sd["add_embedding.image_proj.weight"], sd["add_embedding.image_proj.bias"])
    add = F.layer_norm(add, add.shape[-1:], sd["add_embedding.image_norm.weight"], sd["add_embedding.image_norm.bias"])
    return add, tok.permute(0, 2, 1)


def to_reference_fp16(sd):
    """State dict as the reference holds it after convert_to_fp16() (unet.py:566-571 + fp16_util.py:9-16): the Conv1d / Conv2d
    weights and biases of input_blocks / middle_block / output_blocks in fp16, everything else (GroupNorm gains, emb_layers
    and time_embed Linears, the `out` head) fp32; Text2ImUNet.convert_to_fp16 (text2im_model2_1.py:49-55) also halves the
    2.1 conditioning head, whose inputs the pipeline passes in fp16."""
    out = {}
    head = ("clip_to_seq.", "proj_n.", "to_model_dim_n.", "ln_model_n.", "img_layer.")
    for k, v in sd.items():
        torso = k.startswith(("input_blocks.", "middle_block.", "output_blocks."))
        is_conv = torso and (v.dim() >= 3 or (k.endswith(".bias") and sd[k[:-4] + "weight"].dim() >= 3))
        out[k] = v.half() if is_conv or k.startswith(head) else v.float()
    return out


def fp16_cpu_probe():
    """Fingerprint of this host's fp16 CPU arithmetic: seeded fp16 conv2d / conv1d / bmm, GroupNorm and SiLU on fp16 data,
    fp32 softmax, plus ATen's CPU capability.  oneDNN's fp16 kernels (AVX512-FP16 / AMX vs AVX512 / AVX2) and ATen's
    vectorised kernels sum in different orders, so the fp16 mode's outputs differ between hosts by ~5e-3 at the tiny UNet's
    size; hosts that agree on this probe bit for bit reproduce each other's fp16 forwards exactly.  Tensors are returned as
    SHA-256 digests of their bytes."""
    import hashlib
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 64, 16, 16, generator=g).half()
    w = (torch.randn(128, 64, 3, 3, generator=g) / 24).half()
    b = torch.randn(128, generator=g).half()
    w1 = (torch.randn(192, 128, 1, generator=g) / 11).half()
    y = F.conv2d(x, w, b, padding=1)
    q = F.conv1d(y.reshape(2, 128, 256), w1)
    a = torch.bmm(q[:, :64].transpose(1, 2), q[:, 64:128])
    n = F.group_norm(y.float(), 32).half()
    out = dict(conv2d=y, conv1d=q, bmm=a, group_norm=n, silu=F.silu(n), softmax=torch.softmax(a.float() * 0.125, dim=-1).half())
    out = {k: hashlib.sha256(v.contiguous().numpy().tobytes()).hexdigest() for k, v in out.items()}
    out["cpu_capability"] = torch.backends.cpu.get_cpu_capability()
    return out


def unet_forward(sd, cfg, x, timesteps, full_emb=None, pooled_emb=None, image_emb=None, inpaint_image=None,
                 inpaint_mask=None, taps=None, fp16=False):
    """fp32 forward. `taps` (optional dict) receives intermediate activations keyed by block name.
    fp16=True: the reference's own fp16 mode (use_fp16, text2im_model2_1.py:94,100): sd from to_reference_fp16, the torso
    runs on h = x.half() (fp16 storage between all ops; GroupNorm32 and softmax upcast internally, nn.py:31-37,
    unet.py:338), time_embed / emb_layers / the `out` head stay fp32.  Used to CALIBRATE the product's deviation."""
    if cfg.get("inpainting"):
        if inpaint_image is None:
            inpaint_image = torch.zeros_like(x)
        if inpaint_mask is None:
            inpaint_mask = torch.zeros_like(x[:, :1])
        x = torch.cat([x, inpaint_image * inpaint_mask, inpaint_mask], dim=1)
    mc = cfg["model_channels"]
    emb = timestep_embedding(timesteps, mc)
    emb = F.linear(F.silu(F.linear(emb, sd["time_embed.0.weight"], sd["time_embed.0.bias"])),
                   sd["time_embed.2.weight"], sd["time_embed.2.bias"])
    if fp16 and cfg.get("cond", "2.1") == "2.1":  # the pipeline feeds the (halved) head fp16 embeddings
        full_emb, pooled_emb, image_emb = full_emb.half(), pooled_emb.half(), image_emb.half()
    xf_proj, xf_out = conditioning(sd, cfg, full_emb, pooled_emb, image_emb)
    emb = emb + xf_proj.to(emb)
    inp, mid, out = unet_topology(cfg)
    hc = cfg["num_head_channels"]

    def run(prefix, blk, h):
        for li, layer in enumerate(blk):
            p = f"{prefix}.{li}."
            if layer[0] == "conv":
                h = F.conv2d(h, sd[p + "weight"], sd[p + "bias"], padding=1)
            elif layer[0] == "res":
                h = _res(h, emb, sd, p, layer[3])
            else:
                h = _attn(h, xf_out, sd, p, hc)
        if taps is not None:
            taps[prefix] = h
        return h

    hs = []
    h = x
    if fp16:
        h = x.half()
        xf_out = xf_out.half()
    for bi, blk in enumerate(inp):
        h = run(f"input_blocks.{bi}", blk, h)
        hs.append(h)
    h = run("middle_block", mid, h)
    for bi, blk in enumerate(out):
        h = torch.cat([h, hs.pop()], dim=1)
        h = run(f"output_blocks.{bi}", blk, h)
    h = h.to(x.dtype)
    h = _gn(h, sd, "out.0.", True)
    return F.conv2d(h, sd["out.2.weight"], sd["out.2.bias"], padding=1)


def algorithmic_flops(cfg, B, H, W, ctx):
    """2*MAC over convs / GEMMs / QK^T / PV of one forward (SURVEY.md section 8d numerator)."""
    inp, mid, out = unet_topology(cfg)
    md = cfg["model_dim"]
    total = 0
    h, w = H, W

    def layer_flops(layer, h, w):
        f = 0
        if layer[0] == "conv":
            f += 2 * B * h * w * layer[2] * layer[1] * 9
        elif layer[0] == "res":
            _, cin, cout, ud = layer
            if ud == "up":
                h, w = h * 2, w * 2
            elif ud == "down":
                h, w = h // 2, w // 2
            f += 2 * B * h * w * cout * (cin * 9 + cout * 9 + (cin if cin != cout else 0))
            f += 2 * B * 2 * cout * 4 * cfg["model_channels"]
        else:
            c = layer[1]
            T = h * w
            f += 2 * B * T * c * (3 * c + c) + 2 * B * ctx * md * 2 * c
            f += 2 * 2 * B * T * (T + ctx) * c
        return f, h, w

    for blk in inp + [mid] + out:
        for layer in blk:
            f, h, w = layer_flops(layer, h, w)
            total += f
    total += 2 * B * H * W * cfg["out_channels"] * cfg["channel_mult"][0] * cfg["model_channels"] * 9
    return total
