"""CPU: checkpoint ingest (SURVEY.md section 8f-3). The score_sde checkpoint layout -- DataParallel 'module.' keys, the
'sigmas' buffer, EMA shadow parameters that replace the weights -- is loaded by diffpure_b200 exactly as the reference's
restore_checkpoint + ExponentialMovingAverage.copy_to do (runners/diffpure_sde.py:42-47,175-182; score_sde/models/ema.py:61-72)."""
import io
import json
import os
from types import SimpleNamespace as NS

import numpy as np
import pytest
import torch

G = os.path.join(os.path.dirname(__file__), "golden")


def _fake_checkpoint(tmp_path):
    """A checkpoint in the reference's on-disk layout, written by hand (no reference code needed)."""
    from diffpure_b200 import lowering_ncsnpp as L, synthetic
    from types import SimpleNamespace
    cfg = SimpleNamespace(image_size=16, num_channels=3, nf=64, ch_mult=(1, 2), num_res_blocks=1, attn_resolutions=(8,))
    shapes = L.param_shapes(cfg)
    model_sd = {"module." + k: v for k, v in synthetic.random_state_dict(shapes, seed=3).items()}
    model_sd["module.sigmas"] = torch.linspace(50.0, 0.01, 1000)
    ema_sd = synthetic.random_state_dict(shapes, seed=4)
    state = {"optimizer": {}, "model": model_sd, "step": 7,
             "ema": {"decay": 0.9999, "num_updates": 7, "shadow_params": [ema_sd[k] for k in shapes]}}
    path = os.path.join(tmp_path, "checkpoint_8.pth")
    torch.save(state, path)
    return path, ema_sd


def test_score_sde_checkpoint_layout(tmp_path):
    from diffpure_b200.runners.diffpure_sde import _load_score_sde_state
    path, ema_sd = _fake_checkpoint(str(tmp_path))
    sd = _load_score_sde_state(path)
    assert "sigmas" in sd and not any(k.startswith("module.") for k in sd)
    for k, v in ema_sd.items():
        assert torch.equal(sd[k], v), k                  # EMA shadow replaced every weight, in parameter order


@pytest.mark.parametrize("wrap", [False, True])
def test_score_sde_checkpoint_matches_reference_loader(tmp_path, wrap):
    """A file written by the reference's own classes (NCSNpp + DataParallel + optimizer + EMA) through ours, against what
    the reference's restore_checkpoint + ema.copy_to make of it (golden: oracle/make_golden.py --reference-interfaces)."""
    d = np.load(os.path.join(G, "reference_checkpoints.npz"))
    path = os.path.join(str(tmp_path), "checkpoint_8.pth")
    with open(path, "wb") as f:
        f.write(d["ckpt_wrapped" if wrap else "ckpt_plain"].tobytes())
    want = torch.load(io.BytesIO(d["want"].tobytes()))
    from diffpure_b200.runners.diffpure_sde import _load_score_sde_state
    got = _load_score_sde_state(path)
    assert set(got) == set(want)
    for k, v in want.items():
        assert torch.equal(got[k], v), k


def _ref_yaml(name):
    """The shipped yaml files' model sections, restated (configs/*.yml) -- what the runners receive as `config`."""
    from types import SimpleNamespace as NS
    if name == "cifar10":
        return NS(data=NS(dataset="CIFAR10", image_size=32, num_channels=3),
                  model=NS(name="ncsnpp", resblock_type="biggan", fir=False, skip_rescale=True, progressive="none",
                           progressive_input="none", embedding_type="positional", conditional=True, nonlinearity="swish",
                           nf=128, ch_mult=[1, 2, 2, 2], num_res_blocks=8, attn_resolutions=[16]))
    if name == "imagenet":
        return NS(data=NS(dataset="ImageNet"),
                  model=NS(attention_resolutions="32,16,8", class_cond=False, diffusion_steps=1000, rescale_timesteps=True,
                           timestep_respacing="1000", image_size=256, learn_sigma=True, noise_schedule="linear",
                           num_channels=256, num_head_channels=64, num_res_blocks=2, resblock_updown=True, use_fp16=True,
                           use_scale_shift_norm=True))
    return NS(data=NS(dataset="CelebA_HQ", image_size=256),
              model=NS(ch=128, out_ch=3, ch_mult=[1, 1, 2, 2, 4, 4], num_res_blocks=2, attn_resolutions=[16], in_channels=3,
                       resamp_with_conv=True, var_type="fixedsmall"))


def test_real_checkpoint_key_sets():
    """The three real checkpoints are loaded by the reference with strict load_state_dict, so their key sets are the
    state_dict() of the reference modules built from the shipped configs (fixture: oracle/make_golden.py
    --checkpoint-keys). The lowerings must consume exactly those names and shapes (plus nothing else)."""
    import json
    from diffpure_b200 import lowering_adm as LA, lowering_ddpm as LD, lowering_ncsnpp as LN
    with open(os.path.join(os.path.dirname(__file__), "golden", "checkpoint_keys.json")) as f:
        keys = json.load(f)
    want = {k: {n: tuple(s) for n, s in v} for k, v in keys.items()}
    ck = want["score_sde/checkpoint_8.pth:model (configs/cifar10.yml)"]
    got = LN.param_shapes(LN.cfg_from_reference(_ref_yaml("cifar10")))
    assert ck.pop("sigmas") == (1000,)                      # the one buffer the score network never reads (ncsnpp.py:59)
    assert {k: tuple(v) for k, v in got.items()} == ck and list(got) == list(ck)   # same order: the EMA shadow list is positional
    ck = want["guided_diffusion/256x256_diffusion_uncond.pt (configs/imagenet.yml)"]
    got = LA.param_shapes(LA.cfg_from_reference(_ref_yaml("imagenet")))
    assert {k: tuple(v) for k, v in got.items()} == ck
    ck = want["celeba_hq.ckpt (configs/celeba.yml)"]
    got = LD.param_shapes(LD.cfg_from_reference(_ref_yaml("celeba")))
    assert {k: tuple(v) for k, v in got.items()} == ck


def test_reference_module_state_dicts_load_directly():
    """state_dict() of the reference's own (reduced) ADM -- after convert_to_fp16, as GuidedDiffusion holds it
    (diffpure_guided.py:31-35) -- and CelebA modules go straight into the runners: names, shapes and dtypes are accepted
    and the lowered programs reproduce the reference modules through the CPU interpreter. The modules' state-dict listings
    and configs are recorded from the reference (golden: oracle/make_golden.py --reference-interfaces); their outputs for
    the seeded factory weights are adm_tiny.npz (fp16 torso) and celeba_tiny.npz."""
    from program_interp import Interp
    from diffpure_b200 import lowering_adm as LA, lowering_ddpm as LD
    from oracle import adm as A, ddpm_unet as D, weights
    with open(os.path.join(G, "reference_interfaces.json")) as f:
        rec = json.load(f)
    ns = lambda d: json.loads(json.dumps(d), object_hook=lambda o: NS(**o))  # noqa: E731

    def rel(a, b):
        return ((a - b).norm() / b.norm()).item()

    listing = rec["adm"]["state_dict"]
    assert any(dt == "float16" for _, _, dt in listing)
    cfg = LA.cfg_from_reference(ns({"model": rec["adm"]["model_config"]}))
    assert {k: tuple(v) for k, v in LA.param_shapes(cfg).items()} == {k: tuple(s) for k, s, _ in listing}
    d = np.load(os.path.join(G, "adm_tiny.npz"))
    factory = weights.make_state_dict(A.param_shapes(A.tiny_cfg(64, 64, (1, 2, 3, 4), 1, (32, 16, 8))), seed=int(d["seed"]))
    sd = {k: factory[k].to(getattr(torch, dt)) for k, _, dt in listing}     # the dtypes the reference module holds
    sd32 = {k: v.float() for k, v in sd.items()}
    got = Interp(LA.lower(cfg, sd32, 2), emulate_bf16=False).run(torch.from_numpy(d["x"]), torch.from_numpy(d["t"]).float())
    assert rel(got, torch.from_numpy(d["y_fp16"])) < 2e-2                # the reference ran its torso in fp16

    listing = rec["celeba"]["state_dict"]
    lcfg = LD.cfg_from_reference(ns(rec["celeba"]["config"]))
    assert {k: tuple(v) for k, v in LD.param_shapes(lcfg).items()} == {k: tuple(s) for k, s, _ in listing}
    d = np.load(os.path.join(G, "celeba_tiny.npz"))
    factory = weights.make_state_dict(D.param_shapes(D.tiny_cfg(32, 64, (1, 2, 2), 1, (16,))), seed=int(d["seed"]))
    sdc = {k: factory[k].to(getattr(torch, dt)) for k, _, dt in listing}
    gotc = Interp(LD.lower(lcfg, sdc, 2), emulate_bf16=False).run(torch.from_numpy(d["x"]), torch.from_numpy(d["t"]).float())
    assert rel(gotc, torch.from_numpy(d["y"])) < 1e-4
