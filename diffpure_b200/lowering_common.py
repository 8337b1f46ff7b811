"""The blocks the three UNet lowerings share, each emitted in one place: time embedding, res-block, attention block,
input conv, output head and the data-gradient walk over a forward's tape. A model lowering reads its state dict into
`ResBlock` / `AttnBlock` records and walks its network in the reference's order; everything here sees only records."""
import math
from dataclasses import dataclass
from typing import Optional, Tuple

import torch

from .program import ASeg, Program, Tensor, View, stats_rows, view

INV_SQRT2 = 1.0 / math.sqrt(2.0)


@dataclass
class Act:
    """An fp32 NHWC residual-stream tensor with its per-channel GroupNorm partial statistics."""
    t: Tensor
    C: int
    H: int
    W: int
    stats: Optional[Tensor]
    P: int  # partials per sample
    pre: Optional[Tensor] = None    # bf16 act(GroupNorm(x)) already produced for the next block by the producer's epilogue
    raw16: Optional[Tensor] = None  # bf16 copy of x written next to it (operand of the next block's 1x1 shortcut)


def pack_conv3x3(w):
    """[Cout, Cin, 3, 3] -> [Cout, 9*Cin] with K index = (ky*3+kx)*Cin + ci (tap-major, matches the TMA tap loop)."""
    co, ci = w.shape[0], w.shape[1]
    return w.permute(0, 2, 3, 1).reshape(co, 9 * ci).contiguous()


def pack_conv1x1(w):
    """[Cout, Cin, 1, 1] or [Cout, Cin] -> [Cout, Cin]."""
    return w.reshape(w.shape[0], -1).contiguous()


def pad_rows(w, mult=128):
    """Zero-pad the leading (output) dimension to a multiple of `mult`."""
    n = w.shape[0]
    n2 = (n + mult - 1) // mult * mult
    if n2 == n:
        return w
    pad = torch.zeros((n2 - n,) + tuple(w.shape[1:]), dtype=w.dtype)
    return torch.cat([w, pad], dim=0)


def new_act(prog: Program, name, B, C, H, W, with_stats=True, dtype="f32"):
    t = prog.tensor(name, B * H * W * C, dtype)
    if with_stats:
        rows, P = stats_rows(B, H * W)
        st = prog.tensor(name + ".stats", rows * C * 2, "f32")
    else:
        st, P = None, 0
    return Act(t, C, H, W, st, P)


def act_seg(t, C, taps=1, stride=1, c_total=None, offset=0):
    return ASeg(view(t, offset), C, C if c_total is None else c_total, taps, stride, 1 if (taps == 9 and stride == 1) else 0)


def lower_attention(prog, name, hn, wq, wk, wv, bq, bk, bv, B, T, C, heads, scale, rec=None):
    """Self-attention core on a normalised bf16 input hn [B*T, C]: returns o bf16 [B*T, C] with channel h*d + c.

    wq/wk/wv: [C, C] (out, in) with output rows ordered head-major; b*: [C].
      T <= 64        : one GEMM for q|k|v, then the whole-sequence smem kernel
      T in {128,256} : q|k GEMM, V^T GEMM (weights as A operand), tcgen05 S GEMM with the softmax epilogue
                       (numerator + row sums), tcgen05 O GEMM scaled by 1/rowsum
      longer T       : fp32 logits to HBM, row-softmax kernel, O GEMM
    """
    d = C // heads
    o = prog.tensor(name + ".o", B * T * C, "bf16")
    if T <= 64:
        qkv = prog.tensor(name + ".qkv", B * T * 3 * C, "bf16")
        prog.gemm([act_seg(hn, C)], prog.const_bf16(name + ".wqkv", torch.cat([wq, wk, wv], 0)), 3 * C, C, 1, 1, B * T,
                  3 * C, bias=prog.const_f32(name + ".bqkv", torch.cat([bq, bk, bv])), out_bf16=qkv)
        prog.attn_small(qkv, o, B, T, heads, d, scale)
        if rec is not None:
            rec.update(qkv=qkv)
        return o
    assert T % 128 == 0 and d % 64 == 0, "tensor-core attention needs T % 128 == 0 and head dim % 64 == 0"
    qk = prog.tensor(name + ".qk", B * T * 2 * C, "bf16")
    prog.gemm([act_seg(hn, C)], prog.const_bf16(name + ".wqk", torch.cat([wq, wk], 0)), 2 * C, C, 1, 1, B * T, 2 * C,
              bias=prog.const_f32(name + ".bqk", torch.cat([bq, bk])), out_bf16=qk)
    # V^T per sample (all heads stacked): [C, T] = Wv[C, C] . hn_b[T, C]^T  (weights as the A operand, bias along M)
    vt = prog.tensor(name + ".vt", B * C * T, "bf16")
    prog.gemm([act_seg(prog.const_bf16(name + ".wv", wv), C)], hn, B * T, C, 1, 1, C, T, batch=B, a_batch_rows=0,
              b_batch_rows=T, out_batch_stride=C * T, bias=prog.const_f32(name + ".bv", bv), bias_along_m=1,
              out_bf16=vt, ldc=T)
    pm = prog.tensor(name + ".p", B * heads * T * T, "bf16")
    s_args = dict(batch=B * heads, inner=heads, a_batch_rows=T, a_inner_k=d, b_batch_rows=T, b_inner_k=d, w_cols=C,
                  out_batch_stride=heads * T * T, out_inner_stride=T * T, ldc=T)
    a_q = [act_seg(qk, d, c_total=2 * C)]
    if T <= 256:
        rs = prog.tensor(name + ".rowsum", B * heads * T, "f32")
        prog.gemm(a_q, view(qk, C), B * T, 2 * C, 1, 1, T, T, out_bf16=pm, softmax=1, softmax_scale=scale,
                  rowsum_out=rs, **s_args)
    else:
        rs = None
        logits = prog.tensor(name + ".s", B * heads * T * T, "f32")
        prog.gemm(a_q, view(qk, C), B * T, 2 * C, 1, 1, T, T, out_f32=logits, alpha=scale, **s_args)
        prog.softmax_rows(logits, pm, B * heads * T, T)
    prog.gemm([act_seg(pm, T)], vt, B * C, T, 1, 1, T, d, batch=B * heads, inner=heads, a_batch_rows=heads * T,
              a_inner_rows=T, b_batch_rows=C, b_inner_rows=d, out_batch_stride=T * C, out_inner_stride=d, rowscale=rs,
              out_bf16=o, ldc=C)
    if rec is not None:      # what the data-gradient of this block reads (lower_attention_bwd)
        rec.update(qk=qk, vt=vt, pm=pm, rs=rs)
    return o


def pack_dgrad3x3(w):
    """Conv2d weight [Cout, Cin, 3, 3] -> the B operand of its data-gradient GEMM (the same implicit 3x3 GEMM with the
    taps flipped and in / out swapped): [Cin, 9*Cout] with K index = (ky*3+kx)*Cout + co reading w[co, ci, 2-ky, 2-kx]."""
    co, ci = w.shape[0], w.shape[1]
    return w.flip(2, 3).permute(1, 2, 3, 0).reshape(ci, 9 * co).contiguous()


def transposed(prog, name, src, rows, cols, ld_in, in_batch_stride, batch):
    """bf16 [batch][rows][cols] (row pitch ld_in) -> new tensor [batch][cols][rows]."""
    out = prog.tensor(name, batch * rows * cols, "bf16")
    prog.transpose(src, out, rows, cols, ld_in, rows, batch, in_batch_stride, rows * cols)
    return out


def lower_attention_bwd(prog, name, rec, go, B, T, C, heads, scale):
    """Data-gradient of `lower_attention`: go = dL/d(o) bf16 [B*T, C] -> dq | dk | dv bf16 [B*T, 3C] (head-major columns
    inside each third, as the forward q | k | v). Per (sample, head): dV = P^T dO, dP = dO V^T, dS = P (dP - rowsum(dP P)),
    dQ = scale dS K, dK = scale dS^T Q -- tcgen05 GEMMs over bf16 transposes + the row-wise `softmax_bwd` kernel
    (`attn_small_bwd` for T <= 64)."""
    d = C // heads
    dqkv = prog.tensor(name + ".dqkv", B * T * 3 * C, "bf16")
    if T <= 64:
        prog.attn_small_bwd(rec["qkv"], go, dqkv, B, T, heads, d, scale)
        return dqkv
    qk, vt, pm, rs = rec["qk"], rec["vt"], rec["pm"], rec["rs"]
    v = transposed(prog, name + ".v", vt, C, T, T, C * T, B)                          # [B][T][C]
    qT = transposed(prog, name + ".qT", view(qk, 0), T, C, 2 * C, T * 2 * C, B)       # [B][C][T]
    kT = transposed(prog, name + ".kT", view(qk, C), T, C, 2 * C, T * 2 * C, B)
    goT = transposed(prog, name + ".goT", go, T, C, C, T * C, B)
    BH = B * heads
    # dP[b,h] = dO[b,:,h] . V[b,:,h]^T   (fp32 [B][heads][T][T])
    dp = prog.tensor(name + ".dp", BH * T * T, "f32")
    prog.gemm([act_seg(go, d, c_total=C)], v, B * T, C, 1, 1, T, T, batch=BH, inner=heads, a_batch_rows=T, a_inner_k=d,
              b_batch_rows=T, b_inner_k=d, w_cols=C, out_batch_stride=heads * T * T, out_inner_stride=T * T, out_f32=dp,
              ldc=T)
    ds = prog.tensor(name + ".ds", BH * T * T, "bf16")
    pn = prog.tensor(name + ".pn", BH * T * T, "bf16")
    prog.softmax_bwd(pm, rs, dp, ds, pn, BH * T, T)            # rs None: pm is the normalised softmax already
    dsT = transposed(prog, name + ".dsT", ds, T, T, T, T * T, BH)
    pnT = transposed(prog, name + ".pnT", pn, T, T, T, T * T, BH)
    # [T, d] results into the head's columns of the q / k / v third of dqkv
    bat = dict(batch=BH, inner=heads, a_batch_rows=heads * T, a_inner_rows=T, b_batch_rows=C, b_inner_rows=d,
               out_batch_stride=T * 3 * C, out_inner_stride=d, ldc=3 * C)
    prog.gemm([act_seg(ds, T)], kT, B * C, T, 1, 1, T, d, alpha=scale, out_bf16=view(dqkv, 0), **bat)
    prog.gemm([act_seg(dsT, T)], qT, B * C, T, 1, 1, T, d, alpha=scale, out_bf16=view(dqkv, C), **bat)
    prog.gemm([act_seg(pnT, T)], goT, B * C, T, 1, 1, T, d, out_bf16=view(dqkv, 2 * C), **bat)
    return dqkv


# ---- block records ----------------------------------------------------------------------------------------------------
Pair = Tuple[torch.Tensor, torch.Tensor]     # (weight, bias) or (gamma, beta), fp32 host tensors


@dataclass
class ResBlock:
    """One residual block, read by the model adapter from its state dict. Conv weights are [Cout, Cin, kh, kw].
    out = alpha * (skip(x') + conv1(act(GN1(conv0(act(GN0(x))') + temb)))), ' = the optional 2x up / down resample;
    skip = the 1x1 conv, or identity when `skip` is None."""
    name: str
    cin: int
    cout: int
    gn0: Pair
    conv0: Pair
    gn1: Pair
    conv1: Pair
    skip: Optional[Pair]
    temb: View            # this block's columns of the time-embedding projection
    temb_ld: int
    film: bool            # temb is a per-sample scale | shift applied in GN1 (ADM), else a bias on conv0's output
    groups0: int
    groups1: int
    eps: float
    alpha: float = 1.0
    resample: int = 0     # between GN0 + act and conv0: 0 none, 1 nearest 2x up, 2 2x2-mean down


@dataclass
class AttnBlock:
    """One self-attention block: out = alpha * (x + proj(attention(q, k, v of GN(x)))). Weights are [out, in] with the
    q / k / v output rows head-major."""
    name: str
    gn: Pair
    q: Pair
    k: Pair
    v: Pair
    proj: Pair
    heads: int
    scale: float
    groups: int
    eps: float
    alpha: float = 1.0


def const_pair(prog, name, pair):
    return prog.const_f32(name + ".w", pair[0]), prog.const_f32(name + ".b", pair[1])


def gn_epilogue_args(prog, out: Act, spec, name, B):
    """gemm() keyword arguments that make the producer of `out` also write its consumer's normalised operand.
    spec: None, or dict(gamma, beta, groups, eps, silu, raw16) of the consumer's GroupNorm."""
    if spec is None:
        return {}
    out.pre = prog.tensor(name + ".next_a0", B * out.H * out.W * out.C, "bf16")
    kw = dict(gn_out=out.pre, gn_gamma=spec["gamma"], gn_beta=spec["beta"], gn_groups=spec["groups"],
              gn_eps=spec["eps"], gn_silu=spec["silu"])
    if spec["raw16"]:
        out.raw16 = prog.tensor(name + ".next_xb", B * out.H * out.W * out.C, "bf16")
        kw["out_bf16"] = out.raw16
    return kw


# ---- forward emitters ---------------------------------------------------------------------------------------------------
def lower_time_embedding(prog, B, dense0: Pair, dense1: Pair, projs, cos_first, half_minus_1):
    """Sinusoidal embedding -> Linear + SiLU -> Linear + SiLU -> every block's projection of it as ONE GEMM (every
    consumer applies SiLU to the embedding first, so the second layer stores it after its SiLU).
    projs: (weight, bias) per block. Returns the fp32 projections [B, ld], each block's first column, and ld."""
    dim, emb_dim = dense0[0].shape[1], dense0[0].shape[0]
    offs, n = [], 0
    for w, _ in projs:
        offs.append(n)
        n += w.shape[0]
    ld = (n + 127) // 128 * 128
    w_all = pad_rows(torch.cat([w for w, _ in projs], 0))
    b_all = torch.cat([b for _, b in projs] + [torch.zeros(ld - n)], 0)
    emb = prog.tensor("temb.emb", B * dim, "bf16")
    prog.embed(emb, B, dim, cos_first=cos_first, half_minus_1=half_minus_1)
    t1 = prog.tensor("temb.h1", B * emb_dim, "bf16")
    prog.gemm([act_seg(emb, dim)], prog.const_bf16("temb.w0", dense0[0]), emb_dim, dim, 1, 1, B, emb_dim,
              bias=prog.const_f32("temb.b0", dense0[1]), silu=1, out_bf16=t1)
    t2 = prog.tensor("temb.h2", B * emb_dim, "bf16")
    prog.gemm([act_seg(t1, emb_dim)], prog.const_bf16("temb.w1", dense1[0]), emb_dim, emb_dim, 1, 1, B, emb_dim,
              bias=prog.const_f32("temb.b1", dense1[1]), silu=1, out_bf16=t2)
    out = prog.tensor("temb.all", B * ld, "f32")
    prog.gemm([act_seg(t2, emb_dim)], prog.const_bf16("temb.wall", w_all), ld, emb_dim, 1, 1, B, ld,
              bias=prog.const_f32("temb.ball", b_all), out_f32=out)
    return out, offs, ld


def lower_input_conv(prog, conv: Pair, B, tape=None):
    """The 3 -> C input conv (`Program.conv_in_gemm`)."""
    S, cout = prog.H, conv[0].shape[0]
    h0 = new_act(prog, "conv_in.out", B, cout, S, S)
    prog.conv_in_gemm("conv_in", conv[0], conv[1], h0.t, h0.stats, B, S, S, cout)
    if tape is not None:
        tape.append(dict(kind="conv_in", out=h0, w=conv[0]))
    return h0


def lower_resblock(prog, blk: ResBlock, B, x0: Act, x1: Act = None, fuse_gn1=False, next_gn=None, tape=None):
    """GN0 + act (+ resample, + concat of x1) -> conv0 (+ temb) -> GN1 (+ FiLM) + act -> conv1 (+ the 1x1 shortcut as
    extra K, or the residual) as 3-4 launches. x0.pre: GN0 + act already came out of the producer's epilogue.
    fuse_gn1: GN1 + act in conv0's epilogue (the conv result never leaves TMEM; needs a bias temb).
    next_gn: the consumer's GroupNorm emitted by conv1's epilogue (`gn_epilogue_args`).
    tape: a list -> append what the data-gradient of the block reads (`lower_data_gradient`)."""
    cin, cout, mode, name = blk.cin, blk.cout, blk.resample, blk.name
    assert cin == x0.C + (x1.C if x1 else 0)
    H, W = x0.H, x0.W
    Ho, Wo = (H * 2, W * 2) if mode == 1 else ((H // 2, W // 2) if mode == 2 else (H, W))
    shortcut = blk.skip is not None
    gn0 = gn1 = h = None
    if x0.pre is not None:
        assert x1 is None and mode == 0 and (x0.raw16 is not None) == shortcut
        a0, xb, xr = x0.pre, x0.raw16, None
    else:
        a0 = prog.tensor(name + ".a0", B * Ho * Wo * cin, "bf16")
        xb = prog.tensor(name + ".xb", B * Ho * Wo * cin, "bf16") if shortcut else None
        xr = prog.tensor(name + ".xr", B * Ho * Wo * cin, "f32") if (mode != 0 and not shortcut) else None
        gn0 = const_pair(prog, name + ".gn0", blk.gn0)
        prog.gn_apply(src0=x0.t, stats0=x0.stats, C0=x0.C, P0=x0.P, src1=x1.t if x1 else None,
                      stats1=x1.stats if x1 else None, C1=x1.C if x1 else 0, P1=x1.P if x1 else 0, gamma=gn0[0],
                      beta=gn0[1], B=B, H=H, W=W, groups=blk.groups0, eps=blk.eps, silu=1, resample=mode, out_bf16=a0,
                      raw_bf16=xb, raw_f32=xr)
    a1 = prog.tensor(name + ".a1", B * Ho * Wo * cout, "bf16")
    w0 = prog.const_bf16(name + ".w0", pack_conv3x3(blk.conv0[0]))
    b0 = prog.const_f32(name + ".b0", blk.conv0[1])
    gn1 = const_pair(prog, name + ".gn1", blk.gn1)
    rowvec = {} if blk.film else dict(rowvec=blk.temb, rowvec_ld=blk.temb_ld, rowvec_rows_per_sample=Ho * Wo)
    if fuse_gn1:
        assert not blk.film
        prog.gemm([act_seg(a0, cin, taps=9)], w0, cout, 9 * cin, B, Ho, Wo, cout, bias=b0, **rowvec, gn_out=a1,
                  gn_gamma=gn1[0], gn_beta=gn1[1], gn_groups=blk.groups1, gn_eps=blk.eps, gn_silu=1)
    else:
        # conv0's result is only read by GN1: stored in bf16 (the statistics come from the fp32 accumulators)
        h = new_act(prog, name + ".h", B, cout, Ho, Wo, dtype="bf16")
        prog.gemm([act_seg(a0, cin, taps=9)], w0, cout, 9 * cin, B, Ho, Wo, cout, bias=b0, **rowvec, out_bf16=h.t,
                  stats=h.stats)
        film = dict(film=blk.temb, film_ld=blk.temb_ld) if blk.film else {}
        prog.gn_apply(src0=h.t, stats0=h.stats, C0=cout, P0=h.P, gamma=gn1[0], beta=gn1[1], **film, B=B, H=Ho, W=Wo,
                      groups=blk.groups1, eps=blk.eps, silu=1, out_bf16=a1)
    out = new_act(prog, name + ".out", B, cout, Ho, Wo)
    nxt = gn_epilogue_args(prog, out, next_gn, name, B)
    segs, w1, b1, resid = [act_seg(a1, cout, taps=9)], pack_conv3x3(blk.conv1[0]), blk.conv1[1], None
    if shortcut:
        segs.append(act_seg(xb, cin))
        w1, b1 = torch.cat([w1, pack_conv1x1(blk.skip[0])], dim=1), b1 + blk.skip[1]
    else:
        resid = xr if xr is not None else x0.t
    prog.gemm(segs, prog.const_bf16(name + ".w1", w1), cout, w1.shape[1], B, Ho, Wo, cout,
              bias=prog.const_f32(name + ".b1", b1), resid=resid, alpha=blk.alpha, out_f32=out.t, stats=out.stats, **nxt)
    if tape is not None:
        assert shortcut or x1 is None, "an identity residual over a channel concat has no data-gradient here"
        tape.append(dict(kind="res", blk=blk, x0=x0, x1=x1, h=h, out=out, gn0=gn0, gn1=gn1))
    return out


def lower_attn_block(prog, blk: AttnBlock, B, x: Act, one_kernel=False, next_gn=None, tape=None):
    """GN (or x.pre) -> `lower_attention` -> output projection + residual (+ the consumer's GroupNorm, `next_gn`).
    one_kernel: everything behind the GroupNorm as the `attn_block` kernel (single head, T = C = 256)."""
    C, H, W, name = x.C, x.H, x.W, blk.name
    T = H * W
    gn = None
    if x.pre is not None:
        hn = x.pre
    else:
        gn = const_pair(prog, name + ".gn", blk.gn)
        hn = prog.tensor(name + ".hn", B * T * C, "bf16")
        prog.gn_apply(src0=x.t, stats0=x.stats, C0=C, P0=x.P, gamma=gn[0], beta=gn[1], B=B, H=H, W=W, groups=blk.groups,
                      eps=blk.eps, silu=0, out_bf16=hn)
    (wq, bq), (wk, bk), (wv, bv), (wo, bo) = blk.q, blk.k, blk.v, blk.proj
    if one_kernel:
        assert blk.heads == 1 and next_gn is None and tape is None
        out = new_act(prog, name + ".out", B, C, H, W)
        prog.attn_block(hn, prog.const_bf16(name + ".wqkv3", torch.cat([wq, wk, wv, wo], 0)),
                        prog.const_f32(name + ".bqkv3", torch.cat([bq, bk, bv, bo])), x.t, out.t, out.stats,
                        B, T, C, blk.scale, blk.alpha)
        return out
    rec = dict(kind="attn", blk=blk, x=x, gn=gn) if tape is not None else None
    o = lower_attention(prog, name, hn, wq, wk, wv, bq, bk, bv, B, T, C, blk.heads, blk.scale, rec=rec)
    out = new_act(prog, name + ".out", B, C, H, W)
    nxt = gn_epilogue_args(prog, out, next_gn, name, B)
    prog.gemm([act_seg(o, C)], prog.const_bf16(name + ".w3", wo), C, C, B, H, W, C,
              bias=prog.const_f32(name + ".b3", bo), resid=x.t, alpha=blk.alpha, out_f32=out.t, stats=out.stats, **nxt)
    if tape is not None:
        rec["out"] = out
        tape.append(rec)
    return out


def lower_output_head(prog, x: Act, gn: Pair, groups, eps, conv: Pair, B, tape=None):
    """GroupNorm + SiLU (or x.pre) -> the output conv + the per-step update (`Program.conv_out_gemm`). With a tape the
    program stops in front of it: the data-gradient walk starts here."""
    S = prog.H
    if tape is not None:
        tape.append(dict(kind="out", x=x, gn=gn, groups=groups, eps=eps, w=conv[0]))
        return
    if x.pre is not None:
        a = x.pre
    else:
        a = prog.tensor("out.a", B * S * S * x.C, "bf16")
        gamma, beta = const_pair(prog, "out.gn", gn)
        prog.gn_apply(src0=x.t, stats0=x.stats, C0=x.C, P0=x.P, gamma=gamma, beta=beta, B=B, H=S, W=S, groups=groups,
                      eps=eps, silu=1, out_bf16=a)
    prog.conv_out_gemm("out", a, conv[0], conv[1], B, S, S, x.C, conv[0].shape[0])


# ---- data gradient ------------------------------------------------------------------------------------------------------
def lower_data_gradient(prog, tape, B, g_channels):
    """Appends gx = J(x, t)^T g to a forward lowered with `tape` (the program of `dp_unet_vjp`), g the gradient wrt the
    first `g_channels` output channels. Every conv is the same tcgen05 implicit GEMM with flipped / transposed weights,
    GroupNorm (+SiLU, +FiLM, +resample, +concat) the two-pass `gn_bwd` op, attention `lower_attention_bwd`. The gradient
    stream is fp32 (like the residual stream), GEMM operands bf16. Everything is read from the tape records."""
    S = prog.H
    grad = {}        # tensor index -> (fp32 gradient, bf16 copy) of a residual-stream tensor
    skip_grad = {}   # tensor index -> fp32 gradient that reached the tensor through its skip connection

    def gpair(name, n):
        return prog.tensor(name + ".g32", n, "f32"), prog.tensor(name + ".g16", n, "bf16")

    # ---- output conv (the first g_channels output channels) + output GroupNorm ----------------------------------------
    head = tape[-1]
    hl = head["x"]
    C = hl.C
    gin = prog.tensor("bwd.gin", B * S * S * 64, "bf16")
    prog.grad_in(gin, B, S, S, g_channels, 64)
    wout = torch.zeros(64, C, 3, 3)
    wout[:g_channels] = head["w"][:g_channels]
    ga = prog.tensor("bwd.out.ga", B * S * S * C, "f32")
    prog.gemm([act_seg(gin, 64, taps=9)], prog.const_bf16("bwd.out.w", pack_dgrad3x3(wout)), C, 9 * 64, B, S, S, C,
              out_f32=ga)
    g32, g16 = gpair("bwd.out", B * S * S * C)
    gamma, beta = const_pair(prog, "bwd.out.gn", head["gn"])
    prog.gn_bwd(src0=hl.t, stats0=hl.stats, C0=C, P0=hl.P, gamma=gamma, beta=beta, B=B, H=S, W=S, groups=head["groups"],
                eps=head["eps"], silu=1, g=ga, d0_f32=g32, d0_bf16=g16)
    grad[hl.t.index] = (g32, g16)

    def res_bwd(r):
        blk, x0, x1, h = r["blk"], r["x0"], r["x1"], r["h"]
        cin, cout, Ho, Wo = blk.cin, blk.cout, h.H, h.W
        H, W = x0.H, x0.W
        name = "bwd." + blk.name
        g32, g16 = grad.pop(r["out"].t.index)
        ga1 = prog.tensor(name + ".ga1", B * Ho * Wo * cout, "f32")
        prog.gemm([act_seg(g16, cout, taps=9)], prog.const_bf16(name + ".w1", pack_dgrad3x3(blk.conv1[0])),
                  cout, 9 * cout, B, Ho, Wo, cout, alpha=blk.alpha, out_f32=ga1)
        gc0 = prog.tensor(name + ".gc0", B * Ho * Wo * cout, "bf16")
        film = dict(film=blk.temb, film_ld=blk.temb_ld) if blk.film else {}
        prog.gn_bwd(src0=h.t, stats0=h.stats, C0=cout, P0=h.P, gamma=r["gn1"][0], beta=r["gn1"][1], **film, B=B, H=Ho,
                    W=Wo, groups=blk.groups1, eps=blk.eps, silu=1, g=ga1, d0_bf16=gc0)
        ga0 = prog.tensor(name + ".ga0", B * Ho * Wo * cin, "f32")
        prog.gemm([act_seg(gc0, cout, taps=9)], prog.const_bf16(name + ".w0", pack_dgrad3x3(blk.conv0[0])),
                  cin, 9 * cout, B, Ho, Wo, cin, out_f32=ga0)
        if blk.skip is not None:
            gxs = prog.tensor(name + ".gxs", B * Ho * Wo * cin, "f32")
            prog.gemm([act_seg(g16, cout)], prog.const_bf16(name + ".w2", pack_conv1x1(blk.skip[0]).t().contiguous()),
                      cin, cout, B, Ho, Wo, cin, alpha=blk.alpha, out_f32=gxs)
            add0, scale = gxs, 1.0
        else:
            add0, scale = g32, blk.alpha
        d32, d16 = gpair(name + ".dx", B * H * W * x0.C)
        d1 = prog.tensor(name + ".dskip", B * H * W * x1.C, "f32") if x1 else None
        prog.gn_bwd(src0=x0.t, stats0=x0.stats, C0=x0.C, P0=x0.P, src1=x1.t if x1 else None,
                    stats1=x1.stats if x1 else None, C1=x1.C if x1 else 0, P1=x1.P if x1 else 0, gamma=r["gn0"][0],
                    beta=r["gn0"][1], B=B, H=H, W=W, groups=blk.groups0, eps=blk.eps, silu=1, resample=blk.resample,
                    g=ga0, add0=add0, add0_scale=scale, add1=skip_grad.pop(x0.t.index, None), d0_f32=d32, d0_bf16=d16,
                    d1_f32=d1)
        grad[x0.t.index] = (d32, d16)
        if x1:
            skip_grad[x1.t.index] = d1

    def attn_bwd(r):
        blk, x = r["blk"], r["x"]
        C, H, W = x.C, x.H, x.W
        T = H * W
        name = "bwd." + blk.name
        g32, g16 = grad.pop(r["out"].t.index)
        go = prog.tensor(name + ".go", B * T * C, "bf16")
        prog.gemm([act_seg(g16, C)], prog.const_bf16(name + ".w3", blk.proj[0].t().contiguous()), C, C, 1, 1, B * T, C,
                  alpha=blk.alpha, out_bf16=go)
        dqkv = lower_attention_bwd(prog, name, r, go, B, T, C, blk.heads, blk.scale)
        ghn = prog.tensor(name + ".ghn", B * T * C, "f32")
        wqkv = torch.cat([blk.q[0], blk.k[0], blk.v[0]], 0).t().contiguous()       # [C_in, 3 C_out]
        prog.gemm([act_seg(dqkv, 3 * C)], prog.const_bf16(name + ".wqkv", wqkv), C, 3 * C, 1, 1, B * T, C, out_f32=ghn)
        d32, d16 = gpair(name + ".dx", B * T * C)
        prog.gn_bwd(src0=x.t, stats0=x.stats, C0=C, P0=x.P, gamma=r["gn"][0], beta=r["gn"][1], B=B, H=H, W=W,
                    groups=blk.groups, eps=blk.eps, silu=0, g=ghn, add0=g32, add0_scale=blk.alpha,
                    add1=skip_grad.pop(x.t.index, None), d0_f32=d32, d0_bf16=d16)
        grad[x.t.index] = (d32, d16)

    for r in reversed(tape[1:-1]):
        (res_bwd if r["kind"] == "res" else attn_bwd)(r)
    h0, w_in = tape[0]["out"], tape[0]["w"]
    _, g16 = grad.pop(h0.t.index)
    assert not grad and not skip_grad, (list(grad), list(skip_grad))
    ncol = w_in.shape[1]
    gx8 = prog.tensor("bwd.gx8", B * S * S * 8, "f32")
    prog.gemm([act_seg(g16, h0.C, taps=9)], prog.const_bf16("bwd.conv_in.w", pack_dgrad3x3(w_in)), ncol, 9 * h0.C,
              B, S, S, 8, out_f32=gx8, ldc=8)
    prog.update(gx8, 8, B, S, S, ncol)
    prog.meta.update(vjp=True)
    return prog
