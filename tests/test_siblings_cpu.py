"""CPU: ODE / LDSDE sibling loops -- oracle integrands vs the reference's VPODE / LDSDE (golden), schedules vs oracle loops,
and the drop-in: the reference's unmodified eval_sde_adv.SDE_Adv_Model constructed on top of diffpure_b200.runners."""
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from diffpure_b200 import schedule
from oracle import ncsnpp as O, sde as OS, weights

G = os.path.join(os.path.dirname(__file__), "golden")


def test_sibling_integrands_match_reference():
    d = {k: torch.from_numpy(v) if v.ndim else v for k, v in np.load(os.path.join(G, "siblings_tinyB.npz")).items()}
    cfg = O.tiny_cfg(64, (1, 2, 2), 1, (16,), 32)
    sd = weights.make_state_dict(O.param_shapes(cfg), seed=int(d["seed"]))
    unet = lambda x, t: O.forward(cfg, sd, x, t)  # noqa: E731
    dx = OS.vpode_f(unet, "score_sde", torch.tensor(float(d["t_ode"])), d["x"])
    assert (dx - d["ode_dx"]).abs().max().item() < 1e-4 * max(1.0, d["ode_dx"].abs().max().item())
    f = OS.ldsde_f(unet, "score_sde", d["x"], d["x_init"], 1e-3, 1e-2)
    assert (f - d["ld_f"]).abs().max().item() < 1e-4 * max(1.0, d["ld_f"].abs().max().item())
    assert abs(float(d["ld_g"][0]) - float(np.sqrt(1e-2) * 5)) < 1e-6


def test_sibling_schedules_reproduce_oracle_loops():
    g = torch.Generator().manual_seed(0)
    x0 = torch.rand(2, 3, 8, 8, generator=g) * 2 - 1
    e = torch.randn(2, 3, 8, 8, generator=g)
    eps = torch.randn(2, 3, 8, 8, generator=g)
    unet = lambda xx, tt: eps  # noqa: E731
    for step in (1e-3, 1e-2):
        ref = OS.purify_ode(unet, x0, 100, e, step_size=step)
        cond, coef = schedule.vpode_tables(100, step)
        x = OS.forward_diffuse(x0, e, 100)
        for k in range(len(cond)):
            x = coef[k, 0] * x + coef[k, 1] * eps
        assert (ref - x).abs().max().item() < 1e-5 and (coef[:, 2] == 0).all()
    n = OS.num_steps_ldsde(100)
    z = torch.randn(n, 2, 3, 8, 8, generator=g)
    ref = OS.purify_ldsde(unet, x0, 100, z)
    cond, coef = schedule.ldsde_tables(100)
    assert len(cond) == n == 10 and abs(cond[0] - 9.99) < 1e-4
    x = x0.clone()
    for k in range(n):
        x = coef[k, 0] * x + coef[k, 1] * eps + coef[k, 2] * z[k] + coef[k, 3] * x0
    assert (ref - x).abs().max().item() < 1e-5


def test_reference_sde_adv_model_is_a_drop_in():
    """What the reference's own SDE_Adv_Model (eval_sde_adv.py:34-93) asks of its runners, asked of this package's: the
    runner classes it imports and the constructor calls it makes for each diffusion_type, recorded from the reference with
    configs/cifar10.yml (golden: oracle/make_golden.py --reference-interfaces), replayed on diffpure_b200.runners."""
    import importlib
    import inspect
    import json
    import diffpure_b200.runners.diffpure_sde as rs
    with open(os.path.join(G, "reference_interfaces.json")) as f:
        rec = json.load(f)["sde_adv_model"]
    runners = lambda mod: importlib.import_module("diffpure_b200." + mod)  # noqa: E731  ('runners.x' -> ours)
    assert len(rec["imports"]) == 5
    for mod, names in rec["imports"].items():
        for name in names:
            assert hasattr(runners(mod), name), (mod, name)
    assert sorted(c["diffusion_type"] for c in rec["constructions"]) == ["celebahq-ddpm", "ddpm", "ldsde", "ode", "sde"]
    for c in rec["constructions"]:
        inspect.signature(getattr(runners(c["module"]), c["class"])).bind(*c["args"], **c["kwargs"])

    c = next(c for c in rec["constructions"] if c["diffusion_type"] == "sde")
    cfg = O.tiny_cfg(64, (1, 2, 2), 1, (16,), 32)
    sd = weights.make_state_dict(O.param_shapes(cfg), seed=1)
    args = SimpleNamespace(classifier_name="x", diffusion_type="sde", domain="cifar10", t=5, rand_t=False,
                           t_delta=15, use_bm=False, score_type="score_sde", sample_step=1, log_dir="/tmp/dp_dropin",
                           verbose=False)
    config = json.loads(json.dumps(rec["cifar10_yml"]), object_hook=lambda o: SimpleNamespace(**o))
    config.model.nf, config.model.ch_mult, config.model.num_res_blocks = 64, [1, 2, 2], 1
    config.model.attn_resolutions = [16]
    config.device = torch.device("cpu")
    value = {"args": args, "config": config, "config.device": config.device}
    rs_load = rs._load_score_sde_state
    rs._load_score_sde_state = lambda path, device="cpu": sd
    try:
        runner = getattr(runners(c["module"]), c["class"])(*[value[a] for a in c["args"]],
                                                            **{k: value[v] for k, v in c["kwargs"].items()})
    finally:
        rs._load_score_sde_state = rs_load
    assert type(runner).__module__ == "diffpure_b200.runners.diffpure_sde"
    assert runner.model.kind == "ncsnpp" and hasattr(runner, "rev_vpsde")
