"""Lowering of the guided_diffusion (ADM) UNet to the engine program.

Mirrors guided_diffusion/unet.py:404-671 for DiffPure's ImageNet configuration (configs/imagenet.yml:5-19):
ResBlock with scale-shift norm and resblock_updown (L151-264), AttentionBlock + QKVAttentionLegacy (L267-362:
head-major q|k|v packing, scale ch^-1/4 on q and k), GroupNorm32 (nn.py:25-27, eps 1e-5, fp32 compute),
[cos | sin] timestep embedding (nn.py:111-129), learn_sigma -> 6 output channels.
The reference's fp16 torso (unet.py:626-632) becomes bf16 tensor-core operands with fp32 accumulation and an fp32
residual stream (more accurate than the reference's fp16 adds; SURVEY appendix C, P6).
State-dict names are the reference's.
"""
from types import SimpleNamespace

from .lowering_common import Act, AttnBlock, ResBlock, lower_attn_block, lower_data_gradient, lower_input_conv, \
    lower_output_head, lower_resblock, lower_time_embedding, pack_conv1x1
from .program import Program, view

EPS = 1e-5


def imagenet_cfg():
    return SimpleNamespace(image_size=256, model_channels=256, out_channels=6, num_res_blocks=2,
                           channel_mult=(1, 1, 2, 2, 4, 4), attention_ds=(8, 16, 32), num_head_channels=64)


def cfg_from_reference(config):
    """config.model as in configs/imagenet.yml merged over script_util.model_and_diffusion_defaults()."""
    m = config.model
    image_size = m.image_size
    cm = getattr(m, "channel_mult", "")
    if cm == "" or cm is None:
        cm = {512: (0.5, 1, 1, 2, 2, 4, 4), 256: (1, 1, 2, 2, 4, 4), 128: (1, 1, 2, 3, 4), 64: (1, 2, 3, 4)}[image_size]
    elif isinstance(cm, str):
        cm = tuple(int(c) for c in cm.split(","))
    ar = m.attention_resolutions
    ar = [int(r) for r in ar.split(",")] if isinstance(ar, str) else list(ar)
    assert getattr(m, "use_scale_shift_norm", True) and getattr(m, "resblock_updown", False) and \
        getattr(m, "learn_sigma", False) and not getattr(m, "class_cond", False), "unsupported ADM variant"
    return SimpleNamespace(image_size=image_size, model_channels=m.num_channels, out_channels=6,
                           num_res_blocks=m.num_res_blocks, channel_mult=tuple(cm),
                           attention_ds=tuple(image_size // r for r in ar), num_head_channels=m.num_head_channels)


def block_plan(cfg):
    """input_blocks / middle_block / output_blocks as lists of (kind, kwargs) (unet.py:486-606)."""
    mc = cfg.model_channels
    ch = int(cfg.channel_mult[0] * mc)
    inp = [[("conv_in", dict(cout=ch))]]
    chans = [ch]
    ds = 1
    for level, mult in enumerate(cfg.channel_mult):
        for _ in range(cfg.num_res_blocks):
            layers = [("res", dict(cin=ch, cout=int(mult * mc), mode=0))]
            ch = int(mult * mc)
            if ds in cfg.attention_ds:
                layers.append(("attn", dict(c=ch)))
            inp.append(layers)
            chans.append(ch)
        if level != len(cfg.channel_mult) - 1:
            inp.append([("res", dict(cin=ch, cout=ch, mode=2))])
            chans.append(ch)
            ds *= 2
    mid = [("res", dict(cin=ch, cout=ch, mode=0)), ("attn", dict(c=ch)), ("res", dict(cin=ch, cout=ch, mode=0))]
    out = []
    for level, mult in list(enumerate(cfg.channel_mult))[::-1]:
        for i in range(cfg.num_res_blocks + 1):
            ich = chans.pop()
            layers = [("res", dict(cin=ch + ich, cout=int(mc * mult), mode=0))]
            ch = int(mc * mult)
            if ds in cfg.attention_ds:
                layers.append(("attn", dict(c=ch)))
            if level and i == cfg.num_res_blocks:
                layers.append(("res", dict(cin=ch, cout=ch, mode=1)))
                ds //= 2
            out.append(layers)
    return inp, mid, out, ch


def _all_layers(cfg):
    inp, mid, out, ch = block_plan(cfg)
    for i, layers in enumerate(inp):
        for j, (k, kw) in enumerate(layers):
            yield f"input_blocks.{i}.{j}.", k, kw
    for j, (k, kw) in enumerate(mid):
        yield f"middle_block.{j}.", k, kw
    for i, layers in enumerate(out):
        for j, (k, kw) in enumerate(layers):
            yield f"output_blocks.{i}.{j}.", k, kw


def param_shapes(cfg):
    emb = cfg.model_channels * 4
    sh = {"time_embed.0.weight": (emb, cfg.model_channels), "time_embed.0.bias": (emb,),
          "time_embed.2.weight": (emb, emb), "time_embed.2.bias": (emb,)}
    for p, kind, kw in _all_layers(cfg):
        if kind == "conv_in":
            sh[p + "weight"], sh[p + "bias"] = (kw["cout"], 3, 3, 3), (kw["cout"],)
        elif kind == "res":
            cin, cout = kw["cin"], kw["cout"]
            sh[p + "in_layers.0.weight"], sh[p + "in_layers.0.bias"] = (cin,), (cin,)
            sh[p + "in_layers.2.weight"], sh[p + "in_layers.2.bias"] = (cout, cin, 3, 3), (cout,)
            sh[p + "emb_layers.1.weight"], sh[p + "emb_layers.1.bias"] = (2 * cout, emb), (2 * cout,)
            sh[p + "out_layers.0.weight"], sh[p + "out_layers.0.bias"] = (cout,), (cout,)
            sh[p + "out_layers.3.weight"], sh[p + "out_layers.3.bias"] = (cout, cout, 3, 3), (cout,)
            if cin != cout:
                sh[p + "skip_connection.weight"], sh[p + "skip_connection.bias"] = (cout, cin, 1, 1), (cout,)
        else:
            c = kw["c"]
            sh[p + "norm.weight"], sh[p + "norm.bias"] = (c,), (c,)
            sh[p + "qkv.weight"], sh[p + "qkv.bias"] = (3 * c, c, 1), (3 * c,)
            sh[p + "proj_out.weight"], sh[p + "proj_out.bias"] = (c, c, 1), (c,)
    ch = block_plan(cfg)[3]
    sh["out.0.weight"], sh["out.0.bias"] = (ch,), (ch,)
    sh["out.2.weight"], sh["out.2.bias"] = (cfg.out_channels, ch, 3, 3), (cfg.out_channels,)
    return sh


def lower(cfg, sd, B, tape=None):
    """tape: a list -> every block appends the tensors its data-gradient needs and the program stops in front of the output
    GroupNorm / conv (`lower_vjp` appends the backward ops)."""
    S = cfg.image_size
    prog = Program(B, S, S)
    inp, mid, out, _ = block_plan(cfg)

    def P(name):
        return sd[name].detach().float().cpu()

    def pair(p, a="weight", b="bias"):
        return P(p + a), P(p + b)

    # ---- time embedding MLP (nn.py:111-129) + every ResBlock's FiLM projection Linear(SiLU(emb)) in one GEMM -----------
    res_p = [p for p, kind, _ in _all_layers(cfg) if kind == "res"]
    film_all, offs, film_ld = lower_time_embedding(prog, B, pair("time_embed.0."), pair("time_embed.2."),
                                                   [pair(p + "emb_layers.1.") for p in res_p], cos_first=1, half_minus_1=0)
    film_off = dict(zip(res_p, offs))

    def resblock(p, kw, x0: Act, x1: Act = None):
        """ResBlock._forward, unet.py:244-264 (scale-shift norm; up/down applied after norm+act, before the conv)."""
        cin, cout = kw["cin"], kw["cout"]
        blk = ResBlock(p[:-1], cin, cout, gn0=pair(p + "in_layers.0."), conv0=pair(p + "in_layers.2."),
                       gn1=pair(p + "out_layers.0."), conv1=pair(p + "out_layers.3."),
                       skip=pair(p + "skip_connection.") if cin != cout else None, temb=view(film_all, film_off[p]),
                       temb_ld=film_ld, film=True, groups0=32, groups1=32, eps=EPS, resample=kw["mode"])
        return lower_resblock(prog, blk, B, x0, x1, tape=tape)

    def attnblock(p, x: Act):
        """AttentionBlock._forward + QKVAttentionLegacy, unet.py:307-313,345-362."""
        C = x.C
        d = cfg.num_head_channels
        heads = C // d
        # legacy packing: output channel h*3d + {0,1,2}*d + c  ->  head-major q | k | v blocks
        wqkv = P(p + "qkv.weight").reshape(heads, 3, d, C)
        bqkv = P(p + "qkv.bias").reshape(heads, 3, d)
        q, k, v = ((wqkv[:, j].reshape(C, C).contiguous(), bqkv[:, j].reshape(C).contiguous()) for j in range(3))
        blk = AttnBlock(p[:-1], pair(p + "norm."), q, k, v, (pack_conv1x1(P(p + "proj_out.weight")), P(p + "proj_out.bias")),
                        heads=heads, scale=float(d) ** (-0.5), groups=32, eps=EPS)
        return lower_attn_block(prog, blk, B, x, tape=tape)

    def run(prefix, layers, x0, x1=None):
        h = x0
        for j, (kind, kw) in enumerate(layers):
            p = f"{prefix}{j}."
            if kind == "res":
                h = resblock(p, kw, h, x1)
                x1 = None
            else:
                h = attnblock(p, h)
        return h

    # ---- UNetModel.forward, unet.py:642-671 ---------------------------------------------------------------
    h = lower_input_conv(prog, pair("input_blocks.0.0."), B, tape)
    hs = [h]
    for i, layers in enumerate(inp[1:], start=1):
        h = run(f"input_blocks.{i}.", layers, h)
        hs.append(h)
    h = run("middle_block.", mid, h)
    for i, layers in enumerate(out):
        h = run(f"output_blocks.{i}.", layers, h, hs.pop())
    assert not hs
    lower_output_head(prog, h, pair("out.0."), 32, EPS, pair("out.2."), B, tape)
    prog.meta.update(model="adm", out_channels=cfg.out_channels, cond="timestep")
    return prog


def lower_vjp(cfg, sd, B, g_channels=3):
    """Forward (with a tape) followed by the data-gradient ops: the program of `dp_unet_vjp`, gx = J(x, t)^T g with g the
    gradient wrt the first `g_channels` output channels (3 = the eps half, all the VP-SDE path of
    runners/diffpure_sde.py:96-122 reads; 6 = eps and the learned-variance half).

    The reference differentiates this network through torchsde's adjoint for the ImageNet white-box attacks
    (run_scripts/imagenet/run_in_rand_inf.sh -> eval_sde_adv.py:126-128 -> runners/diffpure_sde.py:233-239). The
    per-sample scale-shift rows fold into gn_bwd's gamma / beta; attention is multi-head at T = 1024 / 256 / 64. Held
    against torch.autograd on the reference-pinned oracle forward (tests/test_vjp_lowering_cpu.py)."""
    tape = []
    prog = lower(cfg, sd, B, tape=tape)
    return lower_data_gradient(prog, tape, B, g_channels)
