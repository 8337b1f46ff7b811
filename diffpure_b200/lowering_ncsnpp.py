"""Lowering of the DDPM++ / NCSN++ score network to the engine program.

Mirrors score_sde/models/ncsnpp.py:35-381 for DiffPure's CIFAR-10 configuration (configs/cifar10.yml:18-40):
biggan res-blocks (layerspp.py:212-274), AttnBlockpp (layerspp.py:62-91), NIN (layers.py:546-555),
positional timestep embedding (layers.py:515-529), naive 2x up / 2x2-mean down (up_or_down_sampling.py:67-77).
The state_dict uses the reference's parameter names (`all_modules.<i>.<...>`).

Fusions per res-block (reference: 2 GroupNorm + 2 SiLU + 2-3 conv + Linear + adds + optional resample/cat
= ~14 ATen ops) -> 3 kernels:
  gn_apply(GN0+SiLU [+up/down] [+concat] [+bf16 copy of x for the 1x1 shortcut])
  gemm(Conv_0 3x3 + bias + Dense_0(SiLU(temb)) add + GroupNorm_1 + SiLU: statistics and normalisation in the epilogue,
       the sample's accumulators resident in TMEM -> the conv result never reaches HBM)
  gemm(Conv_1 3x3 [+ Conv_2 1x1 as extra K] + biases + residual + 1/sqrt(2) + next block's GN statistics)
All per-block Dense_0(SiLU(temb)) projections are one GEMM per step.
"""
import os
from types import SimpleNamespace

from .lowering_common import INV_SQRT2, Act, AttnBlock, ResBlock, const_pair, lower_attn_block, lower_data_gradient, \
    lower_input_conv, lower_output_head, lower_resblock, lower_time_embedding, pack_dgrad3x3  # noqa: F401 (re-export)
from .program import Program, view

EPS = 1e-6


def cifar10_cfg():
    return SimpleNamespace(image_size=32, num_channels=3, nf=128, ch_mult=(1, 2, 2, 2), num_res_blocks=8,
                           attn_resolutions=(16,))


def cfg_from_reference(config):
    """Accepts the reference's yaml namespace (config.model.*, config.data.*)."""
    m, d = config.model, config.data
    assert m.name == "ncsnpp" and m.resblock_type.lower() == "biggan" and not m.fir and m.skip_rescale \
        and m.progressive == "none" and m.progressive_input == "none" and m.embedding_type == "positional" \
        and m.conditional and m.nonlinearity.lower() == "swish", "unsupported NCSN++ variant"
    return SimpleNamespace(image_size=d.image_size, num_channels=d.num_channels, nf=m.nf, ch_mult=tuple(m.ch_mult),
                           num_res_blocks=m.num_res_blocks, attn_resolutions=tuple(m.attn_resolutions))


def _groups(c):
    return min(c // 4, 32)


def module_plan(cfg):
    """(kind, kwargs) per `all_modules` index, in the reference's construction order (ncsnpp.py:68-230)."""
    nf, ch_mult, nrb = cfg.nf, cfg.ch_mult, cfg.num_res_blocks
    nres = len(ch_mult)
    res_at = [cfg.image_size // (2 ** i) for i in range(nres)]
    plan = [("lin0", {}), ("lin1", {}), ("conv_in", {})]
    skips = [nf]
    c = nf
    for lvl in range(nres):
        for _ in range(nrb):
            co = nf * ch_mult[lvl]
            plan.append(("res", dict(cin=c, cout=co, mode=0, role="down")))
            c = co
            if res_at[lvl] in cfg.attn_resolutions:
                plan.append(("attn", dict(c=c)))
            skips.append(c)
        if lvl != nres - 1:
            plan.append(("res", dict(cin=c, cout=c, mode=2, role="downsample")))
            skips.append(c)
    plan += [("res", dict(cin=c, cout=c, mode=0, role="mid")), ("attn", dict(c=c)),
             ("res", dict(cin=c, cout=c, mode=0, role="mid"))]
    for lvl in reversed(range(nres)):
        for _ in range(nrb + 1):
            co = nf * ch_mult[lvl]
            plan.append(("res", dict(cin=c + skips.pop(), cout=co, mode=0, role="up")))
            c = co
        if res_at[lvl] in cfg.attn_resolutions:
            plan.append(("attn", dict(c=c)))
        if lvl != 0:
            plan.append(("res", dict(cin=c, cout=c, mode=1, role="upsample")))
    assert not skips
    plan += [("gn_out", dict(c=c)), ("conv_out", dict(c=c))]
    return plan


def param_shapes(cfg):
    """name -> shape of every parameter in the reference's state_dict order (ncsnpp.py:68-230, layerspp.py:212-240)."""
    shapes = {}
    temb = 4 * cfg.nf
    for i, (kind, kw) in enumerate(module_plan(cfg)):
        p = f"all_modules.{i}."
        if kind == "lin0":
            shapes[p + "weight"], shapes[p + "bias"] = (temb, cfg.nf), (temb,)
        elif kind == "lin1":
            shapes[p + "weight"], shapes[p + "bias"] = (temb, temb), (temb,)
        elif kind == "conv_in":
            shapes[p + "weight"], shapes[p + "bias"] = (cfg.nf, cfg.num_channels, 3, 3), (cfg.nf,)
        elif kind == "gn_out":
            shapes[p + "weight"], shapes[p + "bias"] = (kw["c"],), (kw["c"],)
        elif kind == "conv_out":
            shapes[p + "weight"], shapes[p + "bias"] = (cfg.num_channels, kw["c"], 3, 3), (cfg.num_channels,)
        elif kind == "res":
            cin, cout = kw["cin"], kw["cout"]
            shapes[p + "GroupNorm_0.weight"], shapes[p + "GroupNorm_0.bias"] = (cin,), (cin,)
            shapes[p + "Conv_0.weight"], shapes[p + "Conv_0.bias"] = (cout, cin, 3, 3), (cout,)
            shapes[p + "Dense_0.weight"], shapes[p + "Dense_0.bias"] = (cout, temb), (cout,)
            shapes[p + "GroupNorm_1.weight"], shapes[p + "GroupNorm_1.bias"] = (cout,), (cout,)
            shapes[p + "Conv_1.weight"], shapes[p + "Conv_1.bias"] = (cout, cout, 3, 3), (cout,)
            if cin != cout or kw["mode"] != 0:
                shapes[p + "Conv_2.weight"], shapes[p + "Conv_2.bias"] = (cout, cin, 1, 1), (cout,)
        elif kind == "attn":
            c = kw["c"]
            shapes[p + "GroupNorm_0.weight"], shapes[p + "GroupNorm_0.bias"] = (c,), (c,)
            for j in range(4):
                shapes[p + f"NIN_{j}.W"], shapes[p + f"NIN_{j}.b"] = (c, c), (c,)
    return shapes


def lower(cfg, sd, B, tape=None, fuse_attn=True):
    """Build the engine program for batch size B. `sd`: name -> fp32 torch tensor (CPU).
    Every res-block's GroupNorm_1 + act runs in the epilogue of its Conv_0 GEMM, and a block's output GroupNorm + act is
    written by its producer's epilogue wherever `consumer_gn` allows it.
    fuse_attn: an attention block of T = 256 tokens x C = 256 channels (the 16x16 level of the CIFAR-10 model) as ONE
    kernel (`attn_block`, dp_attn.cu) instead of five GEMM launches; DP_FUSE_ATTN=0 in the environment turns it off (A/B).
    tape: a list -> every block appends the tensors its data-gradient needs, no fusion, and the program stops in front
    of the output GroupNorm / conv (`lower_vjp` appends the backward ops)."""
    S = cfg.image_size
    prog = Program(B, S, S)
    plan = module_plan(cfg)
    fuse = tape is None
    fuse_attn = fuse and fuse_attn and os.environ.get("DP_FUSE_ATTN", "1") != "0"

    def P(i, name):
        return sd[f"all_modules.{i}.{name}"].detach().float().cpu()

    def pair(i, a, b):
        return P(i, a), P(i, b)

    # ---- time embedding MLP + all per-block Dense_0 projections in one GEMM (layers.py:515-529, ncsnpp.py:252-254;
    # every consumer applies act(temb), layerspp.py:263) -------------------------------------------------------------
    res_idx = [i for i, (kind, _) in enumerate(plan) if kind == "res"]
    temb_all, offs, temb_ld = lower_time_embedding(
        prog, B, pair(0, "weight", "bias"), pair(1, "weight", "bias"),
        [pair(i, "Dense_0.weight", "Dense_0.bias") for i in res_idx], cos_first=0, half_minus_1=1)
    temb_off = dict(zip(res_idx, offs))

    def consumer_gn(j, C):
        """If the op after plan entry j-1 normalises the WHOLE incoming tensor (C channels) on its own -- a plain res-block
        (no up / down resample in front of Conv_0, no channel concat), an attention block or the output GroupNorm -- return
        what the producer's epilogue needs to emit that operand itself (`gn_epilogue_args`)."""
        if not fuse or j >= len(plan):
            return None
        kind, kw = plan[j]
        if kind == "res" and kw["mode"] == 0 and kw["role"] in ("down", "mid") and kw["cin"] == C:
            gamma, beta = const_pair(prog, f"m{j}.gn0", pair(j, "GroupNorm_0.weight", "GroupNorm_0.bias"))
            return dict(gamma=gamma, beta=beta, groups=_groups(C), eps=EPS, silu=1, raw16=kw["cin"] != kw["cout"])
        if kind == "attn" and kw["c"] == C:
            gamma, beta = const_pair(prog, f"m{j}.gn", pair(j, "GroupNorm_0.weight", "GroupNorm_0.bias"))
            return dict(gamma=gamma, beta=beta, groups=_groups(C), eps=EPS, silu=0, raw16=False)
        if kind == "gn_out" and kw["c"] == C:
            gamma, beta = const_pair(prog, "out.gn", pair(j, "weight", "bias"))
            return dict(gamma=gamma, beta=beta, groups=_groups(C), eps=EPS, silu=1, raw16=False)
        return None

    def resblock(i, x0: Act, x1: Act = None):
        """ResnetBlockBigGANpp.forward, layerspp.py:242-274."""
        kw = plan[i][1]
        cin, cout, mode = kw["cin"], kw["cout"], kw["mode"]
        skip = pair(i, "Conv_2.weight", "Conv_2.bias") if cin != cout or mode != 0 else None
        blk = ResBlock(f"m{i}", cin, cout, gn0=pair(i, "GroupNorm_0.weight", "GroupNorm_0.bias"),
                       conv0=pair(i, "Conv_0.weight", "Conv_0.bias"), gn1=pair(i, "GroupNorm_1.weight", "GroupNorm_1.bias"),
                       conv1=pair(i, "Conv_1.weight", "Conv_1.bias"), skip=skip, temb=view(temb_all, temb_off[i]),
                       temb_ld=temb_ld, film=False, groups0=_groups(cin), groups1=_groups(cout), eps=EPS,
                       alpha=INV_SQRT2, resample=mode)
        return lower_resblock(prog, blk, B, x0, x1, fuse_gn1=fuse, next_gn=consumer_gn(i + 1, cout), tape=tape)

    def attnblock(i, x: Act):
        """AttnBlockpp.forward, layerspp.py:75-91 (single head of width C, scale C^-1/2, skip_rescale).
        NIN: y = x.W + b with W [in, out]."""
        q, k, v, o = ((P(i, f"NIN_{j}.W").t().contiguous(), P(i, f"NIN_{j}.b")) for j in range(4))
        blk = AttnBlock(f"m{i}", pair(i, "GroupNorm_0.weight", "GroupNorm_0.bias"), q, k, v, o, heads=1,
                        scale=x.C ** -0.5, groups=_groups(x.C), eps=EPS, alpha=INV_SQRT2)
        # the whole block behind the GroupNorm as one kernel (dp_attn.cu): q, k, v^T, the logits, P and o stay on chip
        one_kernel = fuse_attn and x.H * x.W == 256 and x.C == 256
        return lower_attn_block(prog, blk, B, x, one_kernel=one_kernel,
                                next_gn=None if one_kernel else consumer_gn(i + 1, x.C), tape=tape)

    # ---- walk the module list exactly as NCSNpp.forward does (ncsnpp.py:263-381) ----------------------
    h0 = lower_input_conv(prog, pair(2, "weight", "bias"), B, tape)
    idx = 3
    hs = [h0]
    nres = len(cfg.ch_mult)
    for lvl in range(nres):
        for _ in range(cfg.num_res_blocks):
            h = resblock(idx, hs[-1])
            idx += 1
            if h.H in cfg.attn_resolutions:
                h = attnblock(idx, h)
                idx += 1
            hs.append(h)
        if lvl != nres - 1:
            hs.append(resblock(idx, hs[-1]))
            idx += 1
    h = hs[-1]
    h = resblock(idx, h); idx += 1
    h = attnblock(idx, h); idx += 1
    h = resblock(idx, h); idx += 1
    for lvl in reversed(range(nres)):
        for _ in range(cfg.num_res_blocks + 1):
            h = resblock(idx, h, hs.pop())
            idx += 1
        if h.H in cfg.attn_resolutions:
            h = attnblock(idx, h)
            idx += 1
        if lvl != 0:
            h = resblock(idx, h)
            idx += 1
    assert not hs and idx + 2 == len(plan)
    lower_output_head(prog, h, pair(idx, "weight", "bias"), _groups(h.C), EPS, pair(idx + 1, "weight", "bias"), B, tape)
    prog.meta.update(model="ncsnpp", out_channels=cfg.num_channels, cond="999*t")
    return prog


def lower_vjp(cfg, sd, B):
    """Forward (with a tape) followed by the data-gradient ops: the program of `dp_unet_vjp`, gx = J(x, t)^T g.

    Mirrors oracle/ncsnpp_vjp.py (held to torch.autograd on the reference-identical forward). The reference reaches this
    through torchsde's adjoint (runners/diffpure_sde.py:233-239); here the runner differentiates the discrete Euler loop
    it actually runs."""
    tape = []
    prog = lower(cfg, sd, B, tape=tape)
    return lower_data_gradient(prog, tape, B, g_channels=cfg.num_channels)
