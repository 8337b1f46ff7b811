"""Generate the committed golden vectors from the REFERENCE's own modules (build container only).

    python oracle/make_golden.py            # writes tests/golden/*.npz

Needs /root/reference (read-only) and a writable TORCH_EXTENSIONS_DIR: importing score_sde.models.ncsnpp
JIT-builds the reference's two StyleGAN2 ops (~2-4 min the first time, no GPU needed). Weights come from the
seeded factory oracle/weights.py; inputs and noise from seeded torch generators, so the GPU box regenerates
identical operands without the reference.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ncsnpp as O, ref_import, sde as OS, weights  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def inputs(seed, B, S):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(B, 3, S, S, generator=g) * 2 - 1
    t = torch.rand(B, generator=g) * 0.2 + 0.001
    return x, t


def euler_shim(sde, y0, ts, method="euler", bm=None, dt=1e-3, **kw):
    """Fixed-step Ito Euler with torchsde's step grid; `bm(ta, tb)` must return the Brownian increment."""
    assert method == "euler"
    t, y = ts[0], y0
    while t < ts[-1]:
        tn = torch.minimum(t + dt, ts[-1])
        y = y + sde.f(t, y) * (tn - t) + sde.g(t, y) * bm(t, tn)
        t = tn
    return torch.stack([y0, y])


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.set_grad_enabled(False)
    # ---- 1. full CIFAR-10 DDPM++ (configs/cifar10.yml), one UNet evaluation --------------------------------
    model, cfg = ref_import.build_ncsnpp()
    sd = weights.make_state_dict(O.param_shapes(O.CIFAR10_CFG), seed=0)
    missing = model.load_state_dict(sd, strict=False)
    assert set(missing.missing_keys) <= {"sigmas"} and not missing.unexpected_keys, missing
    x, t = inputs(100, 2, 32)
    y = model(x, t * 999)
    np.savez_compressed(os.path.join(OUT, "ncsnpp_cifar10_eval.npz"), x=x.numpy(), labels=(t * 999).numpy(),
                        y=y.numpy(), seed=0)
    print("cifar10 eval: |y| mean", y.abs().mean().item())

    # ---- 2. reduced configurations (same block types) -----------------------------------------------------
    for name, ov, cfg_o in [
        ("tinyA", dict(nf=64, ch_mult=[1, 2], num_res_blocks=1, attn_resolutions=[8], **{"data.image_size": 16}),
         O.tiny_cfg(64, (1, 2), 1, (8,), 16)),
        ("tinyB", dict(nf=64, ch_mult=[1, 2, 2], num_res_blocks=1, attn_resolutions=[16], **{"data.image_size": 32}),
         O.tiny_cfg(64, (1, 2, 2), 1, (16,), 32)),
    ]:
        m, c = ref_import.build_ncsnpp(ov)
        sdt = weights.make_state_dict(O.param_shapes(cfg_o), seed=1)
        r = m.load_state_dict(sdt, strict=False)
        assert set(r.missing_keys) <= {"sigmas"} and not r.unexpected_keys, r
        S = cfg_o.image_size
        x, t = inputs(200, 3, S)
        y = m(x, t * 999)
        # reference RevVPSDE driven by the Euler shim with injected noise (runners/diffpure_sde.py:50-147)
        ref_import.install(euler_shim)
        from runners.diffpure_sde import RevVPSDE
        rev = RevVPSDE(model=m, score_type="score_sde", img_shape=(3, S, S))
        t_star = 4
        g = torch.Generator().manual_seed(300)
        x0 = torch.rand(3, 3, S, S, generator=g) * 2 - 1
        e0 = torch.randn(3, 3, S, S, generator=g)
        steps = OS.num_steps(t_star)
        z = torch.randn(steps, 3, 3, S, S, generator=g)
        xs = OS.forward_diffuse(x0, e0, t_star)
        grid = OS.time_grid(t_star)
        ts = torch.stack([grid[0], grid[-1]])
        k = {"i": 0}

        def bm(ta, tb):
            dw = z[k["i"]].reshape(3, -1) * torch.sqrt(tb - ta)
            k["i"] += 1
            return dw

        out = euler_shim(rev, xs.reshape(3, -1), ts, bm=bm)[-1].reshape(3, 3, S, S)
        f0 = rev.f(grid[0], xs.reshape(3, -1)).reshape(3, 3, S, S)
        g0 = rev.g(grid[0], xs.reshape(3, -1))[:, 0]
        np.savez_compressed(os.path.join(OUT, f"ncsnpp_{name}.npz"), x=x.numpy(), labels=(t * 999).numpy(),
                            y=y.numpy(), x0=x0.numpy(), e0=e0.numpy(), z=z.numpy(), t_star=t_star,
                            loop_out=out.numpy(), f0=f0.numpy(), g0=g0.numpy(), seed=1)
        print(name, "eval |y|", y.abs().mean().item(), "loop |x|", out.abs().mean().item(), "steps", steps)




def golden_adm_and_celeba():
    """ADM (guided_diffusion) and CelebA-HQ DDPM: reference UNet evaluations and the reference's own reverse steps."""
    from oracle import adm as A, ddpm_unet as D, ddpm_loops as OL
    torch.set_grad_enabled(False)
    # ---- ADM, reduced width/size, all three attention regimes (T = 1024, 256, 64) ------------------------
    m, diffusion, mc = ref_import.build_adm(num_channels=64, image_size=64, num_res_blocks=1)
    oc = A.tiny_cfg(64, 64, (1, 2, 3, 4), 1, (32, 16, 8))
    sd = weights.make_state_dict(A.param_shapes(oc), seed=5)
    m.load_state_dict(sd)
    g = torch.Generator().manual_seed(400)
    x = torch.rand(2, 3, 64, 64, generator=g) * 2 - 1
    t = torch.tensor([7, 130])
    y = m(x, t)
    m16, _, _ = ref_import.build_adm(num_channels=64, image_size=64, num_res_blocks=1, use_fp16=True)
    m16.load_state_dict(sd)
    m16.convert_to_fp16()
    y16 = m16(x, t)
    # reference p_sample chain (runners/diffpure_guided.py:59-75), t = 3, noise replayed from the torch RNG stream
    t_levels = 3
    x0 = torch.rand(2, 3, 64, 64, generator=g) * 2 - 1
    betas = torch.from_numpy(diffusion.betas).float()
    torch.manual_seed(77)
    e = torch.randn_like(x0)
    a = (1 - betas).cumprod(dim=0)
    xx = x0 * a[t_levels - 1].sqrt() + e * (1.0 - a[t_levels - 1]).sqrt()
    for i in reversed(range(t_levels)):
        xx = diffusion.p_sample(m, xx, torch.tensor([i] * 2), clip_denoised=True, denoised_fn=None, cond_fn=None,
                                model_kwargs=None)["sample"]
    torch.manual_seed(77)
    e2 = torch.randn_like(x0)
    z = torch.stack([torch.randn_like(x0) for _ in range(t_levels)])
    assert torch.equal(e, e2)
    np.savez_compressed(os.path.join(OUT, "adm_tiny.npz"), x=x.numpy(), t=t.numpy(), y=y.numpy(), y_fp16=y16.numpy(),
                        x0=x0.numpy(), e0=e.numpy(), z=z.numpy(), t_levels=t_levels, loop_out=xx.numpy(), seed=5)
    print("adm tiny |y|", y.abs().mean().item(), "fp16-torso rel", ((y16 - y).norm() / y.norm()).item())

    # ---- CelebA-HQ DDPM, reduced ------------------------------------------------------------------------------
    m, cfg = ref_import.build_celeba({"ch": 64, "ch_mult": [1, 2, 2], "num_res_blocks": 1, "attn_resolutions": [16],
                                      "data.image_size": 32})
    oc = D.tiny_cfg(32, 64, (1, 2, 2), 1, (16,))
    sd = weights.make_state_dict(D.param_shapes(oc), seed=4)
    m.load_state_dict(sd)
    x = torch.rand(2, 3, 32, 32, generator=g) * 2 - 1
    t = torch.tensor([5, 400])
    y = m(x, t)
    from runners.diffpure_ddpm import image_editing_denoising_step_flexible_mask, get_beta_schedule
    betas64 = get_beta_schedule(beta_start=1e-4, beta_end=2e-2, num_diffusion_timesteps=1000)
    ac = np.cumprod(1.0 - betas64)
    logvar = np.log(np.maximum(betas64 * (1.0 - np.append(1.0, ac[:-1])) / (1.0 - ac), 1e-20))
    betas = torch.from_numpy(betas64).float()
    t_levels = 4
    x0 = torch.rand(2, 3, 32, 32, generator=g) * 2 - 1
    torch.manual_seed(78)
    e = torch.randn_like(x0)
    a = (1 - betas).cumprod(dim=0)
    xx = x0 * a[t_levels - 1].sqrt() + e * (1.0 - a[t_levels - 1]).sqrt()
    for i in reversed(range(t_levels)):
        xx = image_editing_denoising_step_flexible_mask(xx, t=torch.tensor([i] * 2), model=m, logvar=logvar, betas=betas)
    torch.manual_seed(78)
    e2 = torch.randn_like(x0)
    z = torch.stack([torch.randn_like(x0) for _ in range(t_levels)])
    np.savez_compressed(os.path.join(OUT, "celeba_tiny.npz"), x=x.numpy(), t=t.numpy(), y=y.numpy(), x0=x0.numpy(),
                        e0=e.numpy(), z=z.numpy(), t_levels=t_levels, loop_out=xx.numpy(), seed=4)
    print("celeba tiny |y|", y.abs().mean().item())


if __name__ == "__main__" and not ({"--siblings", "--adm-vpsde", "--checkpoint-keys", "--guided-schedules",
                                    "--reference-interfaces"} & set(sys.argv)):
    if "--adm-celeba" not in sys.argv:
        main()
    if "--ncsnpp" not in sys.argv:
        golden_adm_and_celeba()


def golden_siblings():
    """Reference VPODE.ode_fn (runners/diffpure_ode.py:90-125) and LDSDE.f/g (runners/diffpure_ldsde.py:92-148) on the
    reduced DDPM++ (tinyB) -- pins oracle/sde.py:vpode_f / ldsde_f."""
    torch.set_grad_enabled(False)
    ref_import.install()
    m, c = ref_import.build_ncsnpp(dict(nf=64, ch_mult=[1, 2, 2], num_res_blocks=1, attn_resolutions=[16],
                                        **{"data.image_size": 32}))
    cfg_o = O.tiny_cfg(64, (1, 2, 2), 1, (16,), 32)
    sdt = weights.make_state_dict(O.param_shapes(cfg_o), seed=1)
    m.load_state_dict(sdt, strict=False)
    from runners.diffpure_ode import VPODE
    from runners.diffpure_ldsde import LDSDE
    g = torch.Generator().manual_seed(500)
    x = torch.rand(2, 3, 32, 32, generator=g) * 2 - 1
    x_init = torch.rand(2, 3, 32, 32, generator=g) * 2 - 1
    t = torch.tensor(0.07)
    ode = VPODE(model=m, score_type="score_sde", img_shape=(3, 32, 32))
    dx = ode(t, (x.reshape(2, -1),))[0].reshape(2, 3, 32, 32)
    ld = LDSDE(model=m, x_init=x_init.reshape(2, -1), score_type="score_sde", img_shape=(3, 32, 32), sigma2=1e-3,
               lambda_ld=1e-2, eta=5)
    f = ld.f(torch.tensor(0.95), x.reshape(2, -1)).reshape(2, 3, 32, 32)
    gg = ld.g(torch.tensor(0.95), x.reshape(2, -1))[:, 0]
    np.savez_compressed(os.path.join(OUT, "siblings_tinyB.npz"), x=x.numpy(), x_init=x_init.numpy(), t_ode=0.07,
                        ode_dx=dx.numpy(), ld_f=f.numpy(), ld_g=gg.numpy(), seed=1)
    print("siblings: |dx|", dx.abs().mean().item(), "|f|", f.abs().mean().item(), "g", gg)


if __name__ == "__main__" and "--siblings" in sys.argv:
    golden_siblings()


def golden_adm_vpsde():
    """The canonical ImageNet configuration (run_scripts/imagenet/run_in_rand_inf.sh:12-24: --diffusion_type sde with the
    default score_type 'guided_diffusion'): the reference's RevVPSDE (runners/diffpure_sde.py:50-147, L101-112 eps -> score
    with integer timesteps, first 3 of 6 output channels) around the reduced ADM UNet, driven by the Euler shim with
    injected Brownian increments."""
    from oracle import adm as A
    torch.set_grad_enabled(False)
    m, diffusion, mc = ref_import.build_adm(num_channels=64, image_size=64, num_res_blocks=1)
    oc = A.tiny_cfg(64, 64, (1, 2, 3, 4), 1, (32, 16, 8))
    sd = weights.make_state_dict(A.param_shapes(oc), seed=5)
    m.load_state_dict(sd)
    ref_import.install(euler_shim)
    from runners.diffpure_sde import RevVPSDE
    S, B, t_star = 64, 2, 4
    rev = RevVPSDE(model=m, score_type="guided_diffusion", img_shape=(3, S, S), model_kwargs={})
    g = torch.Generator().manual_seed(600)
    x0 = torch.rand(B, 3, S, S, generator=g) * 2 - 1
    e0 = torch.randn(B, 3, S, S, generator=g)
    steps = OS.num_steps(t_star)
    z = torch.randn(steps, B, 3, S, S, generator=g)
    xs = OS.forward_diffuse(x0, e0, t_star)
    grid = OS.time_grid(t_star)
    ts = torch.stack([grid[0], grid[-1]])
    k = {"i": 0}

    def bm(ta, tb):
        dw = z[k["i"]].reshape(B, -1) * torch.sqrt(tb - ta)
        k["i"] += 1
        return dw

    out = euler_shim(rev, xs.reshape(B, -1), ts, bm=bm)[-1].reshape(B, 3, S, S)
    f0 = rev.f(grid[0], xs.reshape(B, -1)).reshape(B, 3, S, S)
    g0 = rev.g(grid[0], xs.reshape(B, -1))[:, 0]
    # x0 / e0 / z are regenerated by the tests from the same seeded generator (adm_vpsde_inputs below)
    np.savez_compressed(os.path.join(OUT, "adm_tiny_vpsde.npz"), t_star=t_star, loop_out=out.numpy(), f0=f0.numpy(),
                        g0=g0.numpy(), seed=5, input_seed=600)
    print("adm tiny VP-SDE: loop |x|", out.abs().mean().item(), "steps", steps, "|f0|", f0.abs().mean().item())


if __name__ == "__main__" and "--adm-vpsde" in sys.argv:
    golden_adm_vpsde()


def golden_checkpoint_keys():
    """The key sets (ordered names + shapes) of the three real checkpoints the reference loads with strict load_state_dict:
    pretrained/score_sde/checkpoint_8.pth['model'] (runners/diffpure_sde.py:178-182), pretrained/guided_diffusion/
    256x256_diffusion_uncond.pt (diffpure_guided.py:31) and celeba_hq.ckpt (diffpure_ddpm.py:72-74) -- i.e. the
    state_dict() of the reference modules built from the shipped yaml configs. The files themselves do not exist offline."""
    import json
    out = {}
    m, _ = ref_import.build_ncsnpp()
    out["score_sde/checkpoint_8.pth:model (configs/cifar10.yml)"] = [[k, list(v.shape)] for k, v in m.state_dict().items()]
    with torch.device("meta"):
        adm, _, _ = ref_import.build_adm()
    out["guided_diffusion/256x256_diffusion_uncond.pt (configs/imagenet.yml)"] = \
        [[k, list(v.shape)] for k, v in adm.state_dict().items()]
    with torch.device("meta"):
        cel, _ = ref_import.build_celeba()
    out["celeba_hq.ckpt (configs/celeba.yml)"] = [[k, list(v.shape)] for k, v in cel.state_dict().items()]
    with open(os.path.join(OUT, "checkpoint_keys.json"), "w") as f:
        json.dump(out, f)
    for k, v in out.items():
        print(k, len(v), "tensors", sum(int(np.prod(s)) for _, s in v), "elements")


if __name__ == "__main__" and "--checkpoint-keys" in sys.argv:
    golden_checkpoint_keys()


GUIDED_SCHEDULE_CASES = [  # (diffusion_steps, noise_schedule, timestep_respacing, rescale_timesteps)
    (1000, "linear", "1000", True),      # configs/imagenet.yml
    (1000, "linear", "250", True),
    (1000, "linear", "100,50,25", False),
    (1000, "cosine", "ddim50", True),
    (500, "cosine", "", False),
]


def golden_guided_schedules():
    """The reference's SpacedDiffusion tables (guided_diffusion/script_util.py:create_gaussian_diffusion ->
    respace.py:63-99) for non-default timestep_respacing / noise_schedule / rescale_timesteps, and one learned-range
    p_sample chain of the reduced ADM under timestep_respacing='100,50,25' (runners/diffpure_guided.py:59-75)."""
    ref_import.install()
    from guided_diffusion.script_util import create_gaussian_diffusion, create_model_and_diffusion, \
        model_and_diffusion_defaults
    from oracle import adm as A
    torch.set_grad_enabled(False)
    out = {}
    for ci, (n, ns, tr, rs) in enumerate(GUIDED_SCHEDULE_CASES):
        d = create_gaussian_diffusion(steps=n, learn_sigma=True, noise_schedule=ns, timestep_respacing=tr,
                                      rescale_timesteps=rs)
        out[f"c{ci}_timestep_map"] = np.array(d.timestep_map, dtype=np.int64)
        for k in ("betas", "sqrt_recip_alphas_cumprod", "sqrt_recipm1_alphas_cumprod", "posterior_mean_coef1",
                  "posterior_mean_coef2", "posterior_log_variance_clipped"):
            out[f"c{ci}_{k}"] = np.asarray(getattr(d, k), dtype=np.float64)
    # chain: reduced ADM through the reference's own SpacedDiffusion.p_sample (model wrapped by _WrappedModel)
    cfg = ref_import.load_config("imagenet.yml")
    mc = model_and_diffusion_defaults()
    mc.update(vars(cfg.model))
    mc.update(num_channels=64, image_size=64, num_res_blocks=1, attention_resolutions="32,16,8", use_fp16=False,
              timestep_respacing="100,50,25")
    m, diffusion = create_model_and_diffusion(**mc)
    m.eval()
    oc = A.tiny_cfg(64, 64, (1, 2, 3, 4), 1, (32, 16, 8))
    m.load_state_dict(weights.make_state_dict(A.param_shapes(oc), seed=5))
    t_levels, B, S = 3, 2, 64
    g = torch.Generator().manual_seed(700)
    x0 = torch.rand(B, 3, S, S, generator=g) * 2 - 1
    e0 = torch.randn(B, 3, S, S, generator=g)
    betas = torch.from_numpy(diffusion.betas).float()
    a = (1 - betas).cumprod(dim=0)
    xx = x0 * a[t_levels - 1].sqrt() + e0 * (1.0 - a[t_levels - 1]).sqrt()
    torch.manual_seed(79)
    for i in reversed(range(t_levels)):
        xx = diffusion.p_sample(m, xx, torch.tensor([i] * B), clip_denoised=True, denoised_fn=None, cond_fn=None,
                                model_kwargs=None)["sample"]
    torch.manual_seed(79)
    z = torch.stack([torch.randn_like(x0) for _ in range(t_levels)])
    np.savez_compressed(os.path.join(OUT, "guided_schedules.npz"), chain_respacing="100,50,25", chain_t_levels=t_levels,
                        chain_seed=5, chain_input_seed=700, chain_z=z.numpy(), chain_out=xx.numpy(), **out)
    print("guided schedules:", len(GUIDED_SCHEDULE_CASES), "cases; respaced chain |x|", xx.abs().mean().item(),
          "model timesteps", [diffusion.timestep_map[i] for i in reversed(range(t_levels))])


if __name__ == "__main__" and "--guided-schedules" in sys.argv:
    golden_guided_schedules()


def golden_reference_interfaces():
    """What four CPU tests compare against, recorded from the reference so that they need only the repository:
      reference_checkpoints.npz   two score_sde checkpoints (plain and DataParallel 'module.' keys) written by the
                                  reference's own NCSNpp + optimizer + ExponentialMovingAverage, and the state dict its
                                  restore_checkpoint + ema.copy_to produce from them (runners/diffpure_sde.py:42-47,178-182)
      reference_interfaces.json   the state_dict() names / shapes / dtypes of the reduced ADM (after convert_to_fp16) and
                                  CelebA modules with the configs that built them; the runner classes eval_sde_adv.py
                                  imports and the calls its SDE_Adv_Model (L34-93) makes on them, with configs/cifar10.yml
      spaced_timesteps.npz        guided_diffusion/respace.py:space_timesteps on seeded random section specs, every 'ddimN'
                                  of a 300-step chain, and the specs it rejects"""
    import contextlib
    import io
    import json
    import tempfile
    import types
    from types import SimpleNamespace as NS
    torch.set_grad_enabled(False)
    ref_import.install()

    # ---- checkpoints through the reference's loader -------------------------------------------------------------
    from score_sde.models.ema import ExponentialMovingAverage
    from score_sde.losses import get_optimizer
    from runners.diffpure_sde import restore_checkpoint
    over = dict(nf=8, ch_mult=[1, 2], num_res_blocks=1, attn_resolutions=[8], **{"data.image_size": 16})
    ck, want = {}, None
    for wrap in (False, True):
        model, cfg = ref_import.build_ncsnpp(over)
        if wrap:
            model = torch.nn.DataParallel(model)
        for i, p in enumerate(model.parameters()):   # every tensor distinct (offset i) and varying inside (a period-7
            p.data.copy_(i + (torch.arange(p.numel()) % 7 - 3).reshape(p.shape) / 8)  # ramp): exposes ordering mistakes
        ema = ExponentialMovingAverage(model.parameters(), decay=0.5)
        for p in model.parameters():                 # the weights move away from the EMA shadow
            p.data.add_(0.5)
        opt = get_optimizer(cfg, model.parameters())
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "checkpoint_8.pth")
            torch.save({"optimizer": opt.state_dict(), "model": model.state_dict(), "ema": ema.state_dict(), "step": 3},
                       path)
            with open(path, "rb") as f:
                ck["wrapped" if wrap else "plain"] = np.frombuffer(f.read(), dtype=np.uint8)
            model2, cfg2 = ref_import.build_ncsnpp(over)
            if wrap:
                model2 = torch.nn.DataParallel(model2)
            ema2 = ExponentialMovingAverage(model2.parameters(), decay=cfg2.model.ema_rate)
            state = dict(step=0, optimizer=get_optimizer(cfg2, model2.parameters()), model=model2, ema=ema2)
            restore_checkpoint(path, state, "cpu")
            ema2.copy_to(model2.parameters())
        got = (model2.module if wrap else model2).state_dict()
        if want is None:
            want = got
        assert list(got) == list(want) and all(torch.equal(got[k], want[k]) for k in want)
    buf = io.BytesIO()
    torch.save(want, buf)
    np.savez_compressed(os.path.join(OUT, "reference_checkpoints.npz"), ckpt_plain=ck["plain"], ckpt_wrapped=ck["wrapped"],
                        want=np.frombuffer(buf.getvalue(), dtype=np.uint8))
    print("checkpoints:", len(want), "tensors,", {k: v.size for k, v in ck.items()}, "bytes")

    # ---- module state dicts and the configs behind them ------------------------------------------------------------
    def listing(sd):
        return [[k, list(v.shape), str(v.dtype).replace("torch.", "")] for k, v in sd.items()]

    def plain(ns):
        return {k: plain(v) for k, v in vars(ns).items()} if isinstance(ns, NS) else ns

    out = {}
    m, _, mc = ref_import.build_adm(num_channels=64, image_size=64, num_res_blocks=1, use_fp16=True)
    out["adm"] = {"model_config": dict(mc), "state_dict": listing(m.state_dict())}
    mc_, ccfg = ref_import.build_celeba({"ch": 64, "ch_mult": [1, 2, 2], "num_res_blocks": 1, "attn_resolutions": [16],
                                        "data.image_size": 32})
    out["celeba"] = {"config": plain(ccfg), "state_dict": listing(mc_.state_dict())}

    # ---- eval_sde_adv.SDE_Adv_Model on a recording stand-in for the runners package ---------------------------------
    rec = {"imports": {}, "constructions": []}
    args = NS(classifier_name="x", domain="cifar10", t=5, rand_t=False, t_delta=15, use_bm=False, score_type="score_sde",
              sample_step=1, log_dir="unused", verbose=False)
    config = ref_import.load_config("cifar10.yml")
    cifar10_yml = plain(config)
    config.device = torch.device("cpu")
    names = {id(args): "args", id(config): "config", id(config.device): "config.device"}

    def recording_module(modname):
        mod = types.ModuleType(modname)

        def getattr_(cls_name):
            if cls_name.startswith("__"):                # the import system's own probes (__path__, ...)
                raise AttributeError(cls_name)
            if cls_name not in rec["imports"].setdefault(modname, []):
                rec["imports"][modname].append(cls_name)

            class Runner:
                def __init__(self, *a, **kw):
                    rec["constructions"].append({"diffusion_type": args.diffusion_type, "module": modname,
                                                 "class": cls_name, "args": [names[id(v)] for v in a],
                                                 "kwargs": {k: names[id(v)] for k, v in kw.items()}})
            return Runner
        mod.__getattr__ = getattr_
        return mod

    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "runners" or k.startswith("runners.")}
    try:
        sys.modules["runners"] = types.ModuleType("runners")
        for sub in ("diffpure_ddpm", "diffpure_guided", "diffpure_sde", "diffpure_ode", "diffpure_ldsde"):
            sys.modules["runners." + sub] = recording_module("runners." + sub)
        sys.modules.pop("eval_sde_adv", None)
        import eval_sde_adv
        eval_sde_adv.get_image_classifier = lambda name: torch.nn.Identity()
        for dt in ("ddpm", "sde", "ode", "ldsde", "celebahq-ddpm"):
            args.diffusion_type = dt
            with contextlib.redirect_stdout(io.StringIO()):
                eval_sde_adv.SDE_Adv_Model(args, config)
    finally:
        for k in [k for k in sys.modules if k == "runners" or k.startswith("runners.") or k == "eval_sde_adv"]:
            sys.modules.pop(k)
        sys.modules.update(saved)
    out["sde_adv_model"] = dict(rec, cifar10_yml=cifar10_yml)
    with open(os.path.join(OUT, "reference_interfaces.json"), "w") as f:
        json.dump(out, f)
    print("interfaces:", len(out["adm"]["state_dict"]), "ADM tensors,", len(out["celeba"]["state_dict"]),
          "CelebA tensors,", len(rec["constructions"]), "runner constructions")

    # ---- respace.space_timesteps -------------------------------------------------------------------------------------
    from guided_diffusion.respace import space_timesteps
    rng = np.random.default_rng(7)
    rn, rspec, rkept = [], [], []
    for _ in range(300):
        n = int(rng.integers(8, 1200))
        k = int(rng.integers(1, 6))
        size = n // k
        counts = [int(rng.integers(1, max(2, min(size, 60)))) for _ in range(k)]
        rn.append(n)
        rspec.append(",".join(str(c) for c in counts))
        rkept.append(sorted(space_timesteps(n, rspec[-1])))
    dn, dkept, rejected = [], [], []
    for want_n in range(1, 301):
        try:
            dkept.append(sorted(space_timesteps(300, f"ddim{want_n}")))
            dn.append(want_n)
        except ValueError:
            rejected.append((300, f"ddim{want_n}"))
    for bad in ("400", "10,200"):
        try:
            space_timesteps(300, bad)
        except ValueError:
            rejected.append((300, bad))
    np.savez_compressed(os.path.join(OUT, "spaced_timesteps.npz"), random_n=np.array(rn), random_spec=np.array(rspec),
                        random_len=np.array([len(v) for v in rkept]), random_kept=np.concatenate(rkept).astype(np.int16),
                        ddim_n=np.array(dn), ddim_len=np.array([len(v) for v in dkept]),
                        ddim_kept=np.concatenate(dkept).astype(np.int16),
                        rejected_n=np.array([r[0] for r in rejected]), rejected_spec=np.array([r[1] for r in rejected]))
    print("spaced timesteps:", len(rn), "random specs,", len(dn), "feasible ddimN,", len(rejected), "rejected specs")


if __name__ == "__main__" and "--reference-interfaces" in sys.argv:
    golden_reference_interfaces()
