"""Lowering of the CelebA-HQ DDPM UNet (SDEdit checkpoint family) to the engine program.

Mirrors ddpm/unet_ddpm.py:200-345: ResnetBlock (L85-142, additive temb, no output rescale), AttnBlock (L145-197,
single head of width C, 1x1-conv projections), conv resampling (Downsample = pad (0,1,0,1) + 3x3 stride 2, L63-82;
Upsample = nearest x2 + 3x3, L44-60), GroupNorm(32, eps 1e-6), [sin | cos] timestep embedding (L14-32).
State-dict names are the reference's.
"""
from types import SimpleNamespace

from .lowering_common import Act, AttnBlock, ResBlock, act_seg, lower_attn_block, lower_input_conv, lower_output_head, \
    lower_resblock, lower_time_embedding, new_act, pack_conv1x1, pack_conv3x3
from .program import Program, view

EPS = 1e-6


def celeba_cfg():
    return SimpleNamespace(image_size=256, ch=128, out_ch=3, ch_mult=(1, 1, 2, 2, 4, 4), num_res_blocks=2,
                           attn_resolutions=(16,), in_channels=3)


def cfg_from_reference(config):
    m = config.model
    assert m.resamp_with_conv and m.in_channels == 3, "unsupported DDPM UNet variant"
    return SimpleNamespace(image_size=config.data.image_size, ch=m.ch, out_ch=m.out_ch, ch_mult=tuple(m.ch_mult),
                           num_res_blocks=m.num_res_blocks, attn_resolutions=tuple(m.attn_resolutions), in_channels=3)


def block_list(cfg):
    """Every ResnetBlock in execution order: (prefix, cin, cout) -- shared by the temb GEMM and the walk."""
    ch, nres = cfg.ch, len(cfg.ch_mult)
    in_mult = (1,) + tuple(cfg.ch_mult)
    blocks = []
    block_in = None
    for lvl in range(nres):
        block_in, block_out = ch * in_mult[lvl], ch * cfg.ch_mult[lvl]
        for b in range(cfg.num_res_blocks):
            blocks.append((f"down.{lvl}.block.{b}.", block_in, block_out))
            block_in = block_out
    blocks.append(("mid.block_1.", block_in, block_in))
    blocks.append(("mid.block_2.", block_in, block_in))
    for lvl in reversed(range(nres)):
        block_out = ch * cfg.ch_mult[lvl]
        skip_in = ch * cfg.ch_mult[lvl]
        for b in range(cfg.num_res_blocks + 1):
            if b == cfg.num_res_blocks:
                skip_in = ch * in_mult[lvl]
            blocks.append((f"up.{lvl}.block.{b}.", block_in + skip_in, block_out))
            block_in = block_out
    return blocks


def param_shapes(cfg):
    sh = {}
    ch, temb = cfg.ch, cfg.ch * 4
    sh["temb.dense.0.weight"], sh["temb.dense.0.bias"] = (temb, ch), (temb,)
    sh["temb.dense.1.weight"], sh["temb.dense.1.bias"] = (temb, temb), (temb,)
    sh["conv_in.weight"], sh["conv_in.bias"] = (ch, 3, 3, 3), (ch,)
    for p, cin, cout in block_list(cfg):
        sh[p + "norm1.weight"], sh[p + "norm1.bias"] = (cin,), (cin,)
        sh[p + "conv1.weight"], sh[p + "conv1.bias"] = (cout, cin, 3, 3), (cout,)
        sh[p + "temb_proj.weight"], sh[p + "temb_proj.bias"] = (cout, temb), (cout,)
        sh[p + "norm2.weight"], sh[p + "norm2.bias"] = (cout,), (cout,)
        sh[p + "conv2.weight"], sh[p + "conv2.bias"] = (cout, cout, 3, 3), (cout,)
        if cin != cout:
            sh[p + "nin_shortcut.weight"], sh[p + "nin_shortcut.bias"] = (cout, cin, 1, 1), (cout,)
    nres = len(cfg.ch_mult)
    res = cfg.image_size
    in_mult = (1,) + tuple(cfg.ch_mult)

    def attn(p, c):
        sh[p + "norm.weight"], sh[p + "norm.bias"] = (c,), (c,)
        for n in ("q", "k", "v", "proj_out"):
            sh[p + n + ".weight"], sh[p + n + ".bias"] = (c, c, 1, 1), (c,)

    for lvl in range(nres):
        c = ch * cfg.ch_mult[lvl]
        if res in cfg.attn_resolutions:
            for b in range(cfg.num_res_blocks):
                attn(f"down.{lvl}.attn.{b}.", c)
        if lvl != nres - 1:
            sh[f"down.{lvl}.downsample.conv.weight"], sh[f"down.{lvl}.downsample.conv.bias"] = (c, c, 3, 3), (c,)
            res //= 2
    attn("mid.attn_1.", ch * cfg.ch_mult[-1])
    for lvl in reversed(range(nres)):
        c = ch * cfg.ch_mult[lvl]
        if res in cfg.attn_resolutions:
            for b in range(cfg.num_res_blocks + 1):
                attn(f"up.{lvl}.attn.{b}.", c)
        if lvl != 0:
            sh[f"up.{lvl}.upsample.conv.weight"], sh[f"up.{lvl}.upsample.conv.bias"] = (c, c, 3, 3), (c,)
            res *= 2
    sh["norm_out.weight"], sh["norm_out.bias"] = (ch * cfg.ch_mult[0],), (ch * cfg.ch_mult[0],)
    sh["conv_out.weight"], sh["conv_out.bias"] = (cfg.out_ch, ch * cfg.ch_mult[0], 3, 3), (cfg.out_ch,)
    return sh


def lower(cfg, sd, B):
    S = cfg.image_size
    prog = Program(B, S, S)
    nres = len(cfg.ch_mult)

    def P(name):
        return sd[name].detach().float().cpu()

    def pair(p, a="weight", b="bias"):
        return P(p + a), P(p + b)

    # ---- timestep embedding MLP (L14-32) + all temb_proj(swish(temb)) in one GEMM --------------------------------
    blocks = block_list(cfg)
    temb_all, offs, temb_ld = lower_time_embedding(prog, B, pair("temb.dense.0."), pair("temb.dense.1."),
                                                   [pair(p + "temb_proj.") for p, _, _ in blocks], cos_first=0,
                                                   half_minus_1=1)
    temb_off = {p: off for (p, _, _), off in zip(blocks, offs)}

    def resblock(p, x0: Act, x1: Act = None):
        """ResnetBlock.forward, unet_ddpm.py:123-142."""
        cin = x0.C + (x1.C if x1 else 0)
        cout = P(p + "conv1.weight").shape[0]
        blk = ResBlock(p[:-1], cin, cout, gn0=pair(p + "norm1."), conv0=pair(p + "conv1."), gn1=pair(p + "norm2."),
                       conv1=pair(p + "conv2."), skip=pair(p + "nin_shortcut.") if cin != cout else None,
                       temb=view(temb_all, temb_off[p]), temb_ld=temb_ld, film=False, groups0=32, groups1=32, eps=EPS)
        return lower_resblock(prog, blk, B, x0, x1)

    def attnblock(p, x: Act):
        """AttnBlock.forward, unet_ddpm.py:172-197."""
        q, k, v, o = ((pack_conv1x1(P(p + n + ".weight")), P(p + n + ".bias")) for n in ("q", "k", "v", "proj_out"))
        blk = AttnBlock(p[:-1], pair(p + "norm."), q, k, v, o, heads=1, scale=int(x.C) ** (-0.5), groups=32, eps=EPS)
        return lower_attn_block(prog, blk, B, x)

    def resample_conv(p, x: Act, mode):
        """Downsample (pad right/bottom + 3x3 stride 2) / Upsample (nearest x2 + 3x3) on the raw stream."""
        C = x.C
        if mode == "down":
            xb = prog.tensor(p + "xb", B * x.H * x.W * C, "bf16")
            prog.cast(src=x.t, C=C, B=B, H=x.H, W=x.W, out_bf16=xb)
            Ho, Wo = x.H // 2, x.W // 2
            seg = act_seg(xb, C, taps=9, stride=2)
        else:
            Ho, Wo = x.H * 2, x.W * 2
            xb = prog.tensor(p + "xb", B * Ho * Wo * C, "bf16")
            prog.cast(src=x.t, C=C, B=B, H=x.H, W=x.W, out_bf16=xb, resample=1)
            seg = act_seg(xb, C, taps=9)
        out = new_act(prog, p + "out", B, C, Ho, Wo)
        prog.gemm([seg], prog.const_bf16(p + "w", pack_conv3x3(P(p + "conv.weight"))), C, 9 * C, B, Ho, Wo, C,
                  bias=prog.const_f32(p + "b", P(p + "conv.bias")), out_f32=out.t, stats=out.stats)
        return out

    # ---- Model.forward, unet_ddpm.py:305-345 -------------------------------------------------------------
    h0 = lower_input_conv(prog, pair("conv_in."), B)
    hs = [h0]
    res = S
    for lvl in range(nres):
        for b in range(cfg.num_res_blocks):
            h = resblock(f"down.{lvl}.block.{b}.", hs[-1])
            if res in cfg.attn_resolutions:
                h = attnblock(f"down.{lvl}.attn.{b}.", h)
            hs.append(h)
        if lvl != nres - 1:
            hs.append(resample_conv(f"down.{lvl}.downsample.", hs[-1], "down"))
            res //= 2
    h = hs[-1]
    h = resblock("mid.block_1.", h)
    h = attnblock("mid.attn_1.", h)
    h = resblock("mid.block_2.", h)
    for lvl in reversed(range(nres)):
        for b in range(cfg.num_res_blocks + 1):
            h = resblock(f"up.{lvl}.block.{b}.", h, hs.pop())
            if res in cfg.attn_resolutions:
                h = attnblock(f"up.{lvl}.attn.{b}.", h)
        if lvl != 0:
            h = resample_conv(f"up.{lvl}.upsample.", h, "up")
            res *= 2
    assert not hs
    lower_output_head(prog, h, pair("norm_out."), 32, EPS, pair("conv_out."), B)
    prog.meta.update(model="ddpm", out_channels=cfg.out_ch, cond="timestep")
    return prog
