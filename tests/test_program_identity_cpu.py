"""CPU: every lowering still emits the program recorded in tests/golden/program_fingerprints.json.

The engine's launches follow from the `Program` alone, so two lowerings that produce the same canonical program run the
same kernels on the same operands. The canonical form takes the ops in order with every argument; an activation becomes
(first-use number, dtype, numel, offset), so tensor names and creation order do not count, and a constant becomes
(dtype, numel, sha256 of the bytes it is uploaded as), so constants are compared by value. Two GEMM fields the kernel
provably never reads are normalised: with `inner == 1` the per-head strides are only ever multiplied by head index 0, and
`w_cols` equal to the A segments' total K is what `dp_op_gemm` uses for 0.

Pooled activation bytes and constant bytes may shrink (a shared constant, a tighter pool) but never grow.
`python tests/test_program_identity_cpu.py` rewrites the fixture."""
import functools
import hashlib
import json
import os
import sys

import pytest
import torch

from diffpure_b200 import lowering_adm as LA, lowering_ddpm as LD, lowering_ncsnpp as LN, synthetic
from diffpure_b200.engine import Engine, _align
from diffpure_b200.program import ASeg, View
from oracle import adm as A, ddpm_unet as D, ncsnpp as O

FIXTURE = os.path.join(os.path.dirname(__file__), "golden", "program_fingerprints.json")

NCSNPP_TINY = {"small-attn": O.tiny_cfg(64, (1, 2), 1, (8,), 16),               # T = 64: attn_small
               "tc-attn-updown": O.tiny_cfg(64, (1, 2, 2), 2, (16,), 32),      # T = 256: GEMM attention, up / down
               "fused-attn-block": O.tiny_cfg(128, (1, 2), 1, (16,), 32)}      # T = C = 256: the one-kernel block
MODELS = {"ncsnpp-" + k: (LN, cfg) for k, cfg in NCSNPP_TINY.items()}
MODELS.update({"ncsnpp-cifar10": (LN, LN.cifar10_cfg()),
               "adm-tiny": (LA, A.tiny_cfg(64, 64, (1, 2, 3, 4), 1, (32, 16, 8))),
               "celeba-tiny": (LD, D.tiny_cfg(32, 64, (1, 2, 2), 1, (16,))),
               "adm-imagenet": (LA, LA.imagenet_cfg()),
               "celeba-full": (LD, LD.celeba_cfg())})

CASES = [(f"{m}/{v}", m, v, B) for m, B in (("ncsnpp-small-attn", 2), ("ncsnpp-tc-attn-updown", 2),
                                            ("ncsnpp-fused-attn-block", 2), ("ncsnpp-cifar10", 2))
         for v in ("lower", "lower-unfused-attn", "lower_vjp")]
CASES += [("adm-tiny/lower", "adm-tiny", "lower", 2), ("adm-tiny/lower_vjp", "adm-tiny", "lower_vjp", 2),
          ("celeba-tiny/lower", "celeba-tiny", "lower", 2),
          ("adm-imagenet/lower", "adm-imagenet", "lower", 1), ("adm-imagenet/lower_vjp", "adm-imagenet", "lower_vjp", 1),
          ("celeba-full/lower", "celeba-full", "lower", 1)]

GEMM_HEAD_FIELDS = ("a_inner_k", "a_inner_rows", "b_inner_k", "b_inner_rows", "out_inner_stride")


@functools.lru_cache(maxsize=1)
def _state_dict(model):
    mod, cfg = MODELS[model]
    return synthetic.random_state_dict(mod.param_shapes(cfg), seed=0)


def build(model, variant, B):
    mod, cfg = MODELS[model]
    sd = _state_dict(model)
    if variant == "lower_vjp":
        return mod.lower_vjp(cfg, sd, B)
    if variant == "lower-unfused-attn":
        return mod.lower(cfg, sd, B, fuse_attn=False)
    return mod.lower(cfg, sd, B)


def _const_digest(t):
    v = t.init.detach().cpu().contiguous().reshape(-1)
    raw = v.to(torch.bfloat16).view(torch.int16) if t.dtype == "bf16" else v.to(torch.float32)
    return hashlib.sha256(raw.numpy().tobytes()).hexdigest()


def fingerprint(prog):
    """Canonical SHA-256 of a program (see the module docstring)."""
    act_no, digests = {}, {}

    def canon(v):
        if isinstance(v, View):
            t = v.tensor
            if t.init is None:
                return ["act", act_no.setdefault(t.index, len(act_no)), t.dtype, t.numel, v.offset]
            if t.index not in digests:
                digests[t.index] = _const_digest(t)
            return ["const", t.dtype, t.numel, digests[t.index], v.offset]
        if isinstance(v, ASeg):
            return ["aseg", canon(v.act), v.C, v.c_total, v.taps, v.stride, v.pad]
        if isinstance(v, (list, tuple)):
            return [canon(x) for x in v]
        if isinstance(v, float):
            return ["f", v.hex()]
        assert v is None or isinstance(v, (int, str)), type(v)
        return v

    h = hashlib.sha256()
    for op in prog.ops:
        args = dict(op.args)
        if op.kind == "gemm":
            if args["inner"] == 1:
                args.update({k: 0 for k in GEMM_HEAD_FIELDS})
            if args["w_cols"] == sum(s.taps * s.C for s in args["a"]):
                args["w_cols"] = 0
        h.update(json.dumps([op.kind, sorted((k, canon(v)) for k, v in args.items())]).encode())
        h.update(b"\n")
    return h.hexdigest()


def pooled_activation_bytes(prog):
    e = Engine.__new__(Engine)                         # no CUDA library: only the placement logic runs
    e.program, e._ptr, e._loc, e.act_bytes = prog, {}, {}, 0
    top = [0]

    def alloc(nbytes):
        top[0] += nbytes
        return len(e._loc), top[0] - nbytes
    e._alloc = alloc
    e._place_activations(True)
    return e.act_bytes


def measure(model, variant, B):
    prog = build(model, variant, B)
    return dict(hash=fingerprint(prog), ops=len(prog.ops), act_bytes=pooled_activation_bytes(prog),
                const_bytes=sum(_align(t.nbytes) for t in prog.tensors if t.init is not None))


@pytest.fixture(autouse=True)
def _default_attention(monkeypatch):
    monkeypatch.delenv("DP_FUSE_ATTN", raising=False)


@pytest.mark.parametrize("case,model,variant,B", CASES, ids=[c[0] for c in CASES])
def test_program_is_unchanged(case, model, variant, B):
    with open(FIXTURE) as f:
        want = json.load(f)[case]
    got = measure(model, variant, B)
    assert (got["hash"], got["ops"]) == (want["hash"], want["ops"])
    assert got["act_bytes"] <= want["act_bytes"]
    assert got["const_bytes"] <= want["const_bytes"]


def test_fingerprint_sees_a_changed_constant_and_ignores_names():
    mod, cfg = MODELS["ncsnpp-small-attn"]
    sd = _state_dict("ncsnpp-small-attn")
    prog = mod.lower(cfg, sd, 2)
    ref = fingerprint(prog)
    for t in prog.tensors:
        t.name = "renamed." + t.name
    assert fingerprint(prog) == ref
    sd2 = dict(sd, **{"all_modules.3.Conv_0.bias": sd["all_modules.3.Conv_0.bias"] + 1e-3})
    assert fingerprint(mod.lower(cfg, sd2, 2)) != ref


if __name__ == "__main__":
    os.environ.pop("DP_FUSE_ATTN", None)
    out = {}
    for case, model, variant, B in CASES:
        out[case] = measure(model, variant, B)
        print(case, out[case], file=sys.stderr)
    with open(FIXTURE, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
