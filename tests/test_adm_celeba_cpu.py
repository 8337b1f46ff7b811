"""CPU: ADM (guided_diffusion) and CelebA-HQ DDPM -- oracles vs the golden vectors generated from the reference's
own modules / reverse steps, lowerings vs oracles through the program interpreter, schedule tables vs oracle loops."""
import os

import numpy as np
import pytest
import torch

from diffpure_b200 import lowering_adm as LA, lowering_ddpm as LD, schedule
from oracle import adm as A, ddpm_loops as OL, ddpm_unet as D, weights
from golden_inputs import adm_vpsde_inputs, respaced_chain_inputs
from oracle import sde as OS
from program_interp import Interp

G = os.path.join(os.path.dirname(__file__), "golden")
ADM_TINY = A.tiny_cfg(64, 64, (1, 2, 3, 4), 1, (32, 16, 8))
CELEBA_TINY = D.tiny_cfg(32, 64, (1, 2, 2), 1, (16,))


def load(name):
    return {k: torch.from_numpy(v) if v.ndim else v for k, v in np.load(os.path.join(G, name)).items()}


def rel(a, b):
    return ((a - b).norm() / b.norm()).item()


def test_adm_oracle_matches_reference_golden():
    d = load("adm_tiny.npz")
    sd = weights.make_state_dict(A.param_shapes(ADM_TINY), seed=int(d["seed"]))
    unet = lambda x, t: A.forward(ADM_TINY, sd, x, t)  # noqa: E731
    assert (unet(d["x"], d["t"]) - d["y"]).abs().max().item() < 1e-5
    out = OL.purify_guided(unet, d["x0"], int(d["t_levels"]), d["e0"], d["z"])
    assert (out - d["loop_out"]).abs().max().item() < 1e-4
    # the reference's fp16-torso mode differs from fp32 by ~2e-3: the bound our bf16 path is judged against
    assert 5e-4 < rel(d["y_fp16"], d["y"]) < 1e-2


def test_celeba_oracle_matches_reference_golden():
    d = load("celeba_tiny.npz")
    sd = weights.make_state_dict(D.param_shapes(CELEBA_TINY), seed=int(d["seed"]))
    unet = lambda x, t: D.forward(CELEBA_TINY, sd, x, t)  # noqa: E731
    assert (unet(d["x"], d["t"]) - d["y"]).abs().max().item() < 1e-5
    out = OL.purify_celeba(unet, d["x0"], int(d["t_levels"]), d["e0"], d["z"])
    assert (out - d["loop_out"]).abs().max().item() < 1e-5


def test_adm_lowering_matches_oracle():
    d = load("adm_tiny.npz")
    sd = weights.make_state_dict(A.param_shapes(ADM_TINY), seed=int(d["seed"]))
    assert set(LA.param_shapes(ADM_TINY).items()) == {(k, tuple(v)) for k, v in A.param_shapes(ADM_TINY).items()}
    prog = LA.lower(ADM_TINY, sd, 2)
    y32 = Interp(prog, emulate_bf16=False).run(d["x"], d["t"].float())
    assert rel(y32, d["y"]) < 1e-5
    assert rel(Interp(prog, emulate_bf16=True).run(d["x"], d["t"].float()), d["y"]) < 2e-2
    kinds = {o.kind for o in prog.ops}
    assert {"softmax_rows", "attn_small", "gemm", "gn_apply"} <= kinds   # T = 1024 / 256 / 64 attention paths


def test_celeba_lowering_matches_oracle():
    d = load("celeba_tiny.npz")
    sd = weights.make_state_dict(D.param_shapes(CELEBA_TINY), seed=int(d["seed"]))
    assert set(LD.param_shapes(CELEBA_TINY).items()) == {(k, tuple(v)) for k, v in D.param_shapes(CELEBA_TINY).items()}
    prog = LD.lower(CELEBA_TINY, sd, 2)
    assert rel(Interp(prog, emulate_bf16=False).run(d["x"], d["t"].float()), d["y"]) < 1e-5
    assert rel(Interp(prog, emulate_bf16=True).run(d["x"], d["t"].float()), d["y"]) < 2e-2


def test_full_size_parameter_tables():
    n = lambda sh: sum(int(np.prod(v)) for v in sh.values())  # noqa: E731
    assert n(LA.param_shapes(LA.imagenet_cfg())) == 552814086     # SURVEY.md section 0
    assert n(LD.param_shapes(LD.celeba_cfg())) == 113673219


def test_ddpm_schedules_reproduce_oracle_steps():
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 3, 8, 8, generator=g)
    e6 = torch.randn(2, 6, 8, 8, generator=g)
    z = torch.randn(2, 3, 8, 8, generator=g)
    tab = OL.GuidedTables()
    cond, coef, sx, se = schedule.guided_tables(150)
    assert len(cond) == 150 and cond[0] == 149 and cond[-1] == 0
    for k in (0, 70, 148, 149):
        ref = OL.guided_p_sample(lambda xx, tt: e6, tab, x, 149 - k, z)
        c = coef[k]
        eps, v = e6[:, :3], e6[:, 3:]
        x0 = (c[0] * x - c[1] * eps).clamp(-1, 1)
        frac = (v + 1) / 2
        mine = c[2] * x0 + c[3] * x + c[6] * torch.exp(0.5 * (frac * c[4] + (1 - frac) * c[5])) * z
        assert (ref - mine).abs().max().item() < 1e-6
    e3 = e6[:, :3]
    ref = OL.purify_celeba(lambda xx, tt: e3, x, 3, z, torch.stack([z, z, z]))
    _, cf, sx3, se3 = schedule.ddpm_tables(3)
    xx = sx3 * x + se3 * z
    for k in range(3):
        xx = cf[k, 0] * xx + cf[k, 1] * e3 + cf[k, 2] * z
    assert (ref - xx).abs().max().item() < 1e-5


def test_adm_on_the_vpsde_path_oracle_and_tables_match_reference_golden():
    """The canonical ImageNet configuration (--diffusion_type sde, score_type 'guided_diffusion'): the fixture was produced
    by the reference's RevVPSDE around its own ADM UNet (runners/diffpure_sde.py:101-112,131-147)."""
    d = load("adm_tiny_vpsde.npz")
    t_star = int(d["t_star"])
    sd = weights.make_state_dict(A.param_shapes(ADM_TINY), seed=int(d["seed"]))
    unet = lambda x, t: A.forward(ADM_TINY, sd, x, t)  # noqa: E731
    x0, e0, z = adm_vpsde_inputs(d["input_seed"], t_star)
    with torch.no_grad():
        out = OS.purify_sde(unet, x0, t_star, e0, z, score_type="guided_diffusion")
        xs = OS.forward_diffuse(x0, e0, t_star)
        grid = OS.time_grid(t_star)
        f0 = OS.rev_vpsde_f(unet, "guided_diffusion", grid[0], xs)
    assert (out - d["loop_out"]).abs().max().item() < 1e-4
    assert (f0 - d["f0"]).abs().max().item() < 1e-4
    assert (OS.rev_vpsde_g(grid[0], 2) - d["g0"]).abs().max().item() < 1e-6
    # the engine's per-step tables (cond = floor(fp32(s * 1000)), c0, c1, c2) replay the same trajectory
    cond, coef = schedule.vpsde_tables(t_star, "guided_diffusion")
    assert cond.tolist() == [float(int(v)) for v in cond.tolist()] and len(cond) == OS.num_steps(t_star)
    xx = xs
    with torch.no_grad():
        for k in range(len(cond)):
            eps = unet(xx, torch.full((2,), int(cond[k])))[:, :3]
            xx = float(coef[k, 0]) * xx + float(coef[k, 1]) * eps + float(coef[k, 2]) * z[k]
    assert (xx - d["loop_out"]).abs().max().item() < 1e-4
    # ... and the 150-step ImageNet grid starts at 149 with one duplicate (SURVEY appendix A.5)
    c150, _ = schedule.vpsde_tables(150, "guided_diffusion")
    assert len(c150) == 150 and c150[0] == 149 and c150[-1] == 1 and len(set(c150.tolist())) == 149


GUIDED_CASES = [(1000, "linear", "1000", True), (1000, "linear", "250", True), (1000, "linear", "100,50,25", False),
                (1000, "cosine", "ddim50", True), (500, "cosine", "", False)]   # oracle/make_golden.py:GUIDED_SCHEDULE_CASES


def test_respaced_guided_chains_match_reference_golden():
    """timestep_respacing / noise_schedule / rescale_timesteps (configs/imagenet.yml invites changing them): the product's
    host tables (schedule.GuidedChain) and the oracle's (ddpm_loops.GuidedTables) are bit-identical to the reference's
    create_gaussian_diffusion -> SpacedDiffusion (fixture tests/golden/guided_schedules.npz), and the oracle chain under
    '100,50,25' reproduces the reference's own p_sample chain."""
    d = np.load(os.path.join(G, "guided_schedules.npz"))
    names = ("betas", "sqrt_recip_alphas_cumprod", "sqrt_recipm1_alphas_cumprod", "posterior_mean_coef1",
             "posterior_mean_coef2", "posterior_log_variance_clipped")
    for ci, (n, ns, tr, rs) in enumerate(GUIDED_CASES):
        ch = schedule.GuidedChain(n, ns, tr, rs)
        tab = OL.GuidedTables(n, ns, tr, rs)
        assert ch.timestep_map.tolist() == d[f"c{ci}_timestep_map"].tolist() == list(tab.timestep_map)
        mine = (ch.betas, ch.sqrt_recip_ac, ch.sqrt_recipm1_ac, ch.c1, ch.c2, ch.post_logvar_clipped)
        orac = (tab.betas, tab.sqrt_recip_ac, tab.sqrt_recipm1_ac, tab.c1, tab.c2, tab.post_logvar_clipped)
        for k, a, b in zip(names, mine, orac):
            assert np.array_equal(a, d[f"c{ci}_{k}"]) and np.array_equal(b, d[f"c{ci}_{k}"]), (ci, k)
        # the device tables: rows t-1 ... 0 of the chain, the UNet conditioned on the mapped (and rescaled) timestep
        t = min(7, ch.num_timesteps)
        cond, coef, sx, se = schedule.guided_tables(t, n, ns, tr, rs)
        idx = np.arange(t - 1, -1, -1)
        want = ch.timestep_map[idx].astype(np.float32) * (np.float32(1000.0 / n) if rs else np.float32(1))
        assert np.array_equal(cond, want) and coef.shape == (t, 8)
        assert np.array_equal(coef[:, 4], np.log(d[f"c{ci}_betas"])[idx].astype(np.float32))
    # chain through the oracle ADM
    sd = weights.make_state_dict(A.param_shapes(ADM_TINY), seed=int(d["chain_seed"]))
    unet = lambda x, t: A.forward(ADM_TINY, sd, x, t)  # noqa: E731
    x0, e0 = respaced_chain_inputs(int(d["chain_input_seed"]))
    out = OL.purify_guided(unet, x0, int(d["chain_t_levels"]), e0, torch.from_numpy(d["chain_z"]),
                           timestep_respacing=str(d["chain_respacing"]))
    assert (out - torch.from_numpy(d["chain_out"])).abs().max().item() < 1e-4
    # ... and it is a different chain from the full one (the fixture would not notice a ignored respacing otherwise)
    full = OL.purify_guided(unet, x0, int(d["chain_t_levels"]), e0, torch.from_numpy(d["chain_z"]))
    assert (full - torch.from_numpy(d["chain_out"])).abs().max().item() > 1e-2
    with np.testing.assert_raises(ValueError):
        schedule.guided_tables(51, 1000, "cosine", "ddim50")


def test_spaced_timesteps_equals_the_reference_on_random_specs():
    """schedule.spaced_timesteps / oracle _kept_steps vs the reference's own space_timesteps (respace.py:7-60) on seeded random
    section specs and every feasible 'ddimN' of a 300-step chain; infeasible specs raise ValueError in all three. The
    reference's answers are recorded in spaced_timesteps.npz (oracle/make_golden.py --reference-interfaces)."""
    d = np.load(os.path.join(G, "spaced_timesteps.npz"))
    rejected = [str(s) for s in d["rejected_spec"]]
    assert len(d["random_n"]) == 300 and len(d["ddim_n"]) + sum(s.startswith("ddim") for s in rejected) == 300
    assert {"400", "10,200"} <= set(rejected)
    for key, specs in (("random", d["random_spec"]), ("ddim", [f"ddim{k}" for k in d["ddim_n"]])):
        ns = d["random_n"] if key == "random" else [300] * len(specs)
        kept = np.split(d[key + "_kept"], np.cumsum(d[key + "_len"])[:-1])
        for n, spec, want in zip(ns, specs, kept):
            n, spec, want = int(n), str(spec), want.tolist()
            assert schedule.spaced_timesteps(n, spec) == want == OL._kept_steps(n, spec), (n, spec)
    for n, bad in zip(d["rejected_n"], d["rejected_spec"]):
        for fn in (schedule.spaced_timesteps, OL._kept_steps):
            with pytest.raises(ValueError):
                fn(int(n), str(bad))
