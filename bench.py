#!/usr/bin/env python
"""bench.py -- purified images/sec of the DiffPure reverse-SDE hot path on B200 (BASELINE.json metric).

Headline workload (configs[1]): CIFAR-10 32x32 DDPM++ (score_sde NCSN++, configs/cifar10.yml), VP-SDE t*=0.1 ->
100 Euler-Maruyama steps, batch 512 per GPU, random-init weights (seeded factory), synthetic images.
One "step" of this benchmark = one whole purification of one batch (100 UNet evaluations + fused updates).

  value      images/s with inputs resident in HBM (dp_purify through the C ABI), max-over-ranks device time
  e2e        the same through the reference-facing runner API (`<Runner>.image_editing_sample`)
             from pinned host memory and back (H2D + D2H inside the timed region)
  roofline   dominant kernel = the tcgen05 implicit-GEMM kernel: executed GEMM FLOPs / CUDA-event time of its
             launches (per-op events on the engine stream) vs the measured bf16 peak
  cpu_baseline  the oracle (CPU restatement of the reference loop) on a bounded sample
  gpu_eager_baseline  the same restatement as plain PyTorch eager kernels (cuDNN / cuBLAS) on this GPU: the
             "reference PyTorch eager on the same B200" bar of BASELINE.md section 3.2 (bounded sample)
  secondary  configs[2] on one GPU: ImageNet 256x256 ADM on the canonical VP-SDE path
             (run_scripts/imagenet/run_in_rand_inf.sh:12-24, --diffusion_type sde, t=150 -> 150 Euler steps),
             batch 32, 1 warm-up + 1 timed purification, with its own roofline / e2e

`--config adm|celeba|adm-guided` make configs[2] / configs[3] / the guided_diffusion ancestral chain the main line.
`--impl reference` times the reference's algorithm on the host cores (oracle port; the reference itself is
Python + an unvendored torchsde and cannot travel to the GPU box).
N > 1: one process per GPU (torchrun), the packed weight blob broadcast once over NCCL, batch sharded, one
all_gather of the purified images per step; no collective inside the SDE loop. Scaling is weak (fixed images per GPU).
"""
import argparse
import contextlib
import io
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402,F401
import torch  # noqa: E402

T_STAR = 100

# BASELINE.json configs. `cifar10` (configs[1]) is the headline workload and the default.
WORKLOADS = {
    "cifar10": dict(desc="CIFAR-10 32x32 DDPM++ VP-SDE t*=0.1, 100 Euler steps", size=32, batch=512, flops=37.09e9,
                    metric="purified images/sec (100-step VP-SDE)", steps=100),
    "adm": dict(desc="ImageNet 256x256 guided_diffusion ADM, VP-SDE t*=0.15, 150 Euler steps (score_type guided_diffusion)",
                size=256, batch=32, flops=2239.67e9, metric="purified images/sec (150-step VP-SDE, ADM)", steps=150),
    "adm-guided": dict(desc="ImageNet 256x256 guided_diffusion ADM, 150 ancestral steps (learned-range p_sample)",
                       size=256, batch=32, flops=2239.67e9, metric="purified images/sec (150-step ADM chain)",
                       steps=150),
    "celeba": dict(desc="CelebA-HQ 256x256 ddpm/unet_ddpm, 100 ancestral steps", size=256, batch=16, flops=497.03e9,
                   metric="purified images/sec (100-step DDPM chain)", steps=100),
}


def ref_config(name, cfg):
    """(runner class, args, config) in the reference's own yaml / argparse shape for a workload."""
    if name == "cifar10":
        from diffpure_b200.runners.diffpure_sde import RevGuidedDiffusion as R
        args = SimpleNamespace(t=T_STAR, rand_t=False, t_delta=15, use_bm=False, score_type="score_sde", sample_step=1,
                               log_dir="/tmp/diffpure_b200_bench", save_images=False)
        config = SimpleNamespace(data=SimpleNamespace(dataset="CIFAR10", image_size=32, num_channels=3),
                                 model=SimpleNamespace(name="ncsnpp", resblock_type="biggan", fir=False,
                                                       skip_rescale=True, progressive="none", progressive_input="none",
                                                       embedding_type="positional", conditional=True,
                                                       nonlinearity="swish", nf=cfg.nf, ch_mult=list(cfg.ch_mult),
                                                       num_res_blocks=cfg.num_res_blocks,
                                                       attn_resolutions=list(cfg.attn_resolutions)))
    elif name in ("adm", "adm-guided"):
        model = SimpleNamespace(attention_resolutions="32,16,8", class_cond=False, diffusion_steps=1000,
                                rescale_timesteps=True, timestep_respacing="1000", image_size=256, learn_sigma=True,
                                noise_schedule="linear", num_channels=256, num_head_channels=64, num_res_blocks=2,
                                resblock_updown=True, use_fp16=True, use_scale_shift_norm=True)
        config = SimpleNamespace(data=SimpleNamespace(dataset="ImageNet"), model=model)
        if name == "adm":
            from diffpure_b200.runners.diffpure_sde import RevGuidedDiffusion as R
            args = SimpleNamespace(t=150, rand_t=False, t_delta=15, use_bm=False, score_type="guided_diffusion",
                                   sample_step=1, log_dir="/tmp/diffpure_b200_bench", save_images=False)
        else:
            from diffpure_b200.runners.diffpure_guided import GuidedDiffusion as R
            args = SimpleNamespace(t=150, sample_step=1, log_dir="/tmp/diffpure_b200_bench", save_images=False)
    else:
        from diffpure_b200.runners.diffpure_ddpm import Diffusion as R
        args = SimpleNamespace(t=100, sample_step=1, log_dir="/tmp/diffpure_b200_bench", save_images=False)
        config = SimpleNamespace(data=SimpleNamespace(dataset="CelebA_HQ", image_size=256),
                                 model=SimpleNamespace(ch=128, out_ch=3, ch_mult=[1, 1, 2, 2, 4, 4], num_res_blocks=2,
                                                       attn_resolutions=[16], in_channels=3, resamp_with_conv=True,
                                                       var_type="fixedsmall"),
                                 diffusion=SimpleNamespace(beta_start=1e-4, beta_end=2e-2, num_diffusion_timesteps=1000))
    return R, args, config


def make_workload(name, seed=0, real_weights=True):
    """(lowering module, cfg, state_dict, cond, coef, sx, se, update_kind) for a BASELINE config, random-init weights.
    real_weights=False: zeros of the right shapes (ranks that receive the packed blob by broadcast)."""
    from diffpure_b200 import lib, schedule, synthetic
    if name == "cifar10":
        from diffpure_b200 import lowering_ncsnpp as L
        cfg = L.cifar10_cfg()
        cond, coef = schedule.vpsde_tables(T_STAR)
        sx, se = schedule.vpsde_forward_scales(T_STAR)
        kind = lib.DP_UPDATE_LINEAR
    elif name == "adm":
        from diffpure_b200 import lowering_adm as L
        cfg = L.imagenet_cfg()
        cond, coef = schedule.vpsde_tables(150, "guided_diffusion")       # runners/diffpure_sde.py:101-112
        sx, se = schedule.vpsde_forward_scales(150)
        kind = lib.DP_UPDATE_LINEAR
    elif name == "adm-guided":
        from diffpure_b200 import lowering_adm as L
        cfg = L.imagenet_cfg()
        cond, coef, sx, se = schedule.guided_tables(150)
        kind = lib.DP_UPDATE_LEARNED_RANGE
    else:
        from diffpure_b200 import lowering_ddpm as L
        cfg = L.celeba_cfg()
        cond, coef, sx, se = schedule.ddpm_tables(100)
        kind = lib.DP_UPDATE_LINEAR
    shapes = L.param_shapes(cfg)
    sd = synthetic.random_state_dict(shapes, seed=seed) if real_weights else {k: torch.zeros(v) for k, v in shapes.items()}
    return L, cfg, sd, cond, coef, sx, se, kind


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return p.get("bf16_tflops_sustained", p.get("bf16_tflops")), p.get("hbm_gbs"), "measured (MEASURED_PEAKS.json, sustained bf16)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md: 1.4 PF/s sustained, 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        hot = [v for v in sm if v > 500] or sm
        return {"sm_mhz": statistics.median(hot) if hot else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------
# CPU / same-GPU eager baselines: the oracle restatement of the reference loop (bench-only use of oracle/)
# ------------------------------------------------------------------------------------------------------------
_CPU_THREADS = None


def _best_cpu_threads(unet, x, t):
    """The reference sets no thread count (torch default = all cores); on many-core hosts the 32x32 convs scale
    badly, so give the reference its best case: time one UNet eval per candidate and keep the fastest."""
    global _CPU_THREADS
    if _CPU_THREADS is not None:
        return _CPU_THREADS
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (16, 32, 64) if c <= ncpu} | {min(ncpu, 8)}) or [ncpu]
    best, best_dt = cands[0], 1e30
    for c in cands:
        torch.set_num_threads(c)
        unet(x, t)                                  # warm
        t0 = time.perf_counter()
        unet(x, t)
        dt = time.perf_counter() - t0
        if dt < best_dt:
            best, best_dt = c, dt
    _CPU_THREADS = best
    return best


def _oracle_euler_steps(unet, x, grid, steps, gen, sync=None):
    from oracle import sde as OS
    B = x.shape[0]
    t0 = time.perf_counter()
    for k in range(steps):
        t, tn = grid[k], grid[k + 1]
        h = tn - t
        f = OS.rev_vpsde_f(unet, "score_sde", t, x)
        gk = OS.rev_vpsde_g(t, B)[:, None, None, None]
        x = x + f * h + gk * torch.randn(x.shape, generator=gen, device=x.device) * torch.sqrt(h)
    if sync:
        sync()
    return time.perf_counter() - t0


def cpu_reference_rate(batch, steps, threads=None):
    """Oracle (CPU port of the reference loop) on a bounded sample: `batch` images, `steps` of the 100 Euler steps."""
    from oracle import ncsnpp as O, sde as OS, weights
    cfg = O.CIFAR10_CFG
    sd = weights.make_state_dict(O.param_shapes(cfg), seed=0)
    g = torch.Generator().manual_seed(0)
    x0 = torch.rand(batch, 3, 32, 32, generator=g) * 2 - 1
    e0 = torch.randn(batch, 3, 32, 32, generator=g)
    grid = OS.time_grid(T_STAR)
    x = OS.forward_diffuse(x0, e0, T_STAR)
    unet = lambda xx, tt: O.forward(cfg, sd, xx, tt)  # noqa: E731
    with torch.no_grad():
        threads = threads or _best_cpu_threads(unet, x, torch.full((batch,), 99.0))
        torch.set_num_threads(threads)
        dt = _oracle_euler_steps(unet, x, grid, steps, g)
    full = dt * (len(grid) - 1) / steps
    return batch / full, dt, threads


def gpu_eager_rate(dev, batch=512, steps=5):
    """The same restatement run as plain PyTorch eager ops on this GPU (cuDNN convs, ~1,100 ATen kernels per evaluation,
    SURVEY section 0): fp32 (the reference's dtype for DDPM++; TF32 convolutions as torch defaults) and bf16 autocast.
    `steps` of the 100 Euler steps at the benchmark batch, extrapolated linearly."""
    from oracle import ncsnpp as O, sde as OS, weights
    cfg = O.CIFAR10_CFG
    sd = {k: v.to(dev) for k, v in weights.make_state_dict(O.param_shapes(cfg), seed=0).items()}
    g = torch.Generator(device=dev).manual_seed(0)
    x0 = torch.rand(batch, 3, 32, 32, generator=g, device=dev) * 2 - 1
    e0 = torch.randn(batch, 3, 32, 32, generator=g, device=dev)
    grid = OS.time_grid(T_STAR).to(dev)
    x = OS.forward_diffuse(x0.cpu(), e0.cpu(), T_STAR).to(dev)
    unet = lambda xx, tt: O.forward(cfg, sd, xx, tt)  # noqa: E731
    out = {}
    torch.backends.cudnn.benchmark = True
    sync = lambda: torch.cuda.synchronize(dev)  # noqa: E731
    with torch.no_grad():
        for name, ctx in (("fp32", contextlib.nullcontext()),
                          ("bf16_autocast", torch.autocast("cuda", dtype=torch.bfloat16))):
            with ctx:
                _oracle_euler_steps(unet, x, grid, 2, g, sync)       # warm-up (cuDNN autotune)
                sync()
                dt = _oracle_euler_steps(unet, x, grid, steps, g, sync)
            out[name] = batch / (dt * (len(grid) - 1) / steps)
    return {"value": out["fp32"], "value_bf16_autocast": out["bf16_autocast"], "unit": "images/s",
            "kind": "oracle port as PyTorch eager ops on the same GPU (cuDNN / cuBLAS, cudnn.benchmark)",
            "sample": f"batch {batch}, {steps} of 100 Euler steps, extrapolated linearly"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals = []
    batch, sub = 16, 10                                        # each step: ~4 s of CPU work
    for i in range(args.warmup + args.steps):
        rate, dt, threads = cpu_reference_rate(batch, sub)
        if i >= args.warmup:
            vals.append((rate, dt))
    rate = statistics.mean(v[0] for v in vals)
    ms = statistics.mean(v[1] for v in vals) * 1e3 * (100 / sub)
    sample = (f"oracle CPU port of the reference loop, batch {batch} (configs[0]), {sub} of 100 Euler steps, "
              f"extrapolated linearly, {threads} threads (fastest of 8/16/32/64)")
    line = {"impl": "reference", "metric": WORKLOADS["cifar10"]["metric"], "value": rate, "unit": "images/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "CIFAR-10 32x32 DDPM++ VP-SDE t*=0.1, 100 Euler steps (CPU sample: batch 16, "
                                   f"{sub} of 100 steps timed, EXTRAPOLATED linearly to 100)",
                       "weights": "random-init (seeded)"},
            "cpu_baseline": {"value": rate, "unit": "images/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": rate, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------
def measure(name, B, steps, warmup, rank, world, local, dev, dist, want_e2e=True, sample_clocks=True):
    """Build the engine of a workload (packed blob broadcast under NCCL), time `steps` purifications, then the same
    through the runner API from pinned host memory, then the per-op roofline. Returns the fields of a bench line."""
    from diffpure_b200.engine import Engine, WeightBlob
    wl = WORKLOADS[name]
    S = wl["size"]
    L, cfg, sd, cond, coef, sx, se, update_kind = make_workload(name, seed=0, real_weights=(rank == 0 or world == 1))
    prog = L.lower(cfg, sd, B)
    blob = WeightBlob(prog, local, upload=(rank == 0))       # rank 0 packs + uploads; the others only lay out
    if world > 1:
        blob.broadcast(src=0)                                 # ONE NCCL broadcast of the packed bytes
    eng = Engine(prog, device=local, blob=blob)
    nsteps = len(cond)
    assert nsteps == wl["steps"]
    g = torch.Generator(device="cpu").manual_seed(1234 + rank)
    x_host = (torch.rand(B, 3, S, S, generator=g) * 2 - 1).pin_memory()
    x_dev = x_host.to(dev)
    gathered = [torch.empty_like(x_dev) for _ in range(world)] if world > 1 else None
    last = {}

    def one_step(seed):
        out = eng.purify(x_dev, cond, coef, sx, se, update_kind=update_kind, seed=seed, sample_offset=rank * B)
        if world > 1:
            dist.all_gather(gathered, out)
        last["purified"] = out
        return out

    def timed(fn, k):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(k):
            fn(1000 + i)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.barrier()
            ms = float(t.item())
        return ms

    for i in range(warmup):
        one_step(i)
    sampler = ClockSampler(local) if (rank == 0 and sample_clocks) else None
    if sampler:
        sampler.start()
    ms_total = timed(one_step, steps)
    clocks = sampler.stop() if sampler else None
    value = world * B * steps / (ms_total / 1e3)
    # the images the last timed step returned (every rank's, in rank order), before the runs below reuse the engine
    purified = (torch.cat(gathered) if world > 1 else last["purified"]).float().cpu()

    # ---- e2e through the runner API from pinned host memory ----------------------------------------------
    e2e = None
    if want_e2e:
        R, rargs, rconfig = ref_config(name, cfg)
        with contextlib.redirect_stdout(io.StringIO()):
            runner = R(rargs, rconfig, device=dev, state_dict=sd)
        runner.model.adopt_engine(eng)            # share the engine (and blob) already built for this batch size
        runner.sample_offset = rank * B
        out_host = torch.empty(B, 3, S, S).pin_memory()

        def e2e_step(seed):
            with torch.no_grad():
                out = runner.image_editing_sample(x_host.to(dev, non_blocking=True), bs_id=2, tag="bench", seed=seed)
            out_host.copy_(out, non_blocking=True)
            torch.cuda.current_stream().synchronize()

        if name == "cifar10":
            e2e_step(0)
        ms_e2e = timed(e2e_step, steps)
        e2e = {"value": world * B * steps / (ms_e2e / 1e3), "unit": "images/s",
               "h2d_bytes_per_step": B * 3 * S * S * 4, "d2h_bytes_per_step": B * 3 * S * S * 4,
               "api": f"{R.__module__}.{R.__name__}.image_editing_sample"}

    res = {"value": value, "ms_per_step": ms_total / steps, "clocks": clocks, "e2e": e2e, "nsteps": nsteps,
           "launches": steps * (nsteps * eng.launches_per_step + 2), "B": B, "purified": purified}
    if rank == 0:
        res["roofline"] = roofline_of(eng, wl, B, value / world, nsteps)
    res["engine"] = eng
    return res


def roofline_of(eng, wl, B, value_per_gpu, nsteps):
    """Per-op CUDA events on the engine's stream (dp_profile_ops): the tcgen05 GEMM kernel's executed FLOPs over its
    summed launch time vs the measured sustained bf16 peak; the whole-loop algorithmic fraction beside it."""
    peak_tf, peak_gbs, peak_src = load_peaks()
    prof = None
    for _ in range(3):
        prof = eng.profile_ops(mode=1)
    by_kind = {}
    for kind, ms, fl in prof:
        d = by_kind.setdefault(kind, [0, 0.0, 0.0])
        d[0] += 1
        d[1] += ms
        d[2] += fl
    gemm_n, gemm_ms, gemm_fl = by_kind["gemm"]
    eval_ms = sum(v[1] for v in by_kind.values())
    achieved_tf = gemm_fl / (gemm_ms / 1e3) / 1e12            # executed GEMM FLOPs only (conv_in / attn_small excluded)
    roofline = {"bound": "tensor",
                "kernel": "dp::gemm_kernel<BN, EPI, CG> (tcgen05 implicit GEMM, CG=2: cta_group::2 CTA pairs)",
                "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf,
                "traffic": None, "peak_source": peak_src, "launches_per_eval": gemm_n,
                "avg_launch_ms": gemm_ms / gemm_n, "alg_flops_per_launch": gemm_fl / gemm_n,
                "alg_flops_per_image_eval": wl["flops"], "executed_gemm_flops_per_eval": gemm_fl,
                "kernel_share_of_eval": gemm_ms / eval_ms, "cta_pair_launches_per_eval": eng.pair_gemms,
                "launches_per_eval_all_kernels": eng.launches_per_eval,
                "eval_ms_by_kind": {k: round(v[1], 4) for k, v in by_kind.items()},
                "eval_launches_by_kind": {k: v[0] for k, v in by_kind.items()},
                "whole_loop_frac_of_peak": value_per_gpu * nsteps * wl["flops"] / 1e12 / peak_tf}
    ab = by_kind.get("attn_block")
    if ab:   # the one-kernel attention blocks (dp_attn.cu): six 256^3 GEMMs per sample each, also on the tcgen05 pipe
        roofline["attn_block"] = {"kernel": "dp::attn_block_kernel (cta_group::2, q/k/v/logits/P on chip)",
                                  "launches_per_eval": ab[0], "ms_per_eval": round(ab[1], 4),
                                  "achieved": ab[2] / (ab[1] / 1e3) / 1e12, "unit": "TFLOP/s"}
        roofline["tensor_kernels_frac"] = (gemm_fl + ab[2]) / ((gemm_ms + ab[1]) / 1e3) / 1e12 / peak_tf
    traffic_path = os.path.join(ROOT, "profiles", "gemm_dram_bytes_per_launch.json")
    if os.path.exists(traffic_path):                           # DRAM bytes need ncu: taken from the committed capture
        with open(traffic_path) as f:
            t = json.load(f)
        roofline["traffic"] = t.get("dram_bytes_per_launch")
        roofline["traffic_source"] = "ncu --set full capture committed under profiles/ (" + str(t.get("source", "r01")) + "), not this run"
    return roofline


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, purified):
    """Save what the timed path returned so that two builds run with the same arguments (same seeded weights, images
    and noise) can be compared output for output. Above DUMP_LIMIT, a seeded sample of whole images is kept."""
    n = purified.shape[0]
    keep = max(1, DUMP_LIMIT // (purified[0].numel() * 4))
    if keep < n:
        idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:keep].sort().values
        purified = purified[idx]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "purified.npy"), purified.numpy().astype(np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cifar10", choices=list(WORKLOADS), help="BASELINE workload (default: headline)")
    ap.add_argument("--batch", type=int, default=0, help="images per GPU (0 = the config's BASELINE batch)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the embedded ADM (configs[2]) measurement")
    ap.add_argument("--no-gpu-eager", action="store_true", help="skip the same-GPU PyTorch-eager baseline")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the images the last timed step returned to DIR/purified.npy (float32; at most "
                         f"{DUMP_LIMIT >> 20} MB: beyond that a fixed, seeded sample of whole images in batch order)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a B200 GPU (use --impl reference for the CPU arm)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    wl = WORKLOADS[args.config]
    B = args.batch or wl["batch"]
    big = wl["size"] > 32
    steps, warmup = args.steps, args.warmup
    main_res = measure(args.config, B, steps, warmup, rank, world, local, dev, dist, want_e2e=not args.no_e2e)
    main_res.pop("engine").close()
    purified = main_res.pop("purified")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, purified)

    secondary = None
    if args.config == "cifar10" and world == 1 and not args.no_secondary:
        # configs[2]: ImageNet ADM on the VP-SDE path, 1 warm-up + 1 timed purification (~12 s each at B=32)
        torch.cuda.empty_cache()
        r = measure("adm", WORKLOADS["adm"]["batch"], 1, 1, rank, world, local, dev, dist, want_e2e=not args.no_e2e)
        r.pop("engine").close()
        w2 = WORKLOADS["adm"]
        secondary = {"metric": w2["metric"], "value": r["value"], "unit": "images/s", "n_gpus": 1, "steps": 1, "warmup": 1,
                     "ms_per_step": r["ms_per_step"], "dtype": "bf16", "data": "synthetic",
                     "config": {"workload": "%s, batch %d per GPU" % (w2["desc"], r["B"]),
                                "weights": "random-init (seeded factory)"},
                     "clocks": r["clocks"], "e2e": r["e2e"], "gpu_launches": r["launches"], "roofline": r["roofline"]}

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    cpu = None
    if not args.no_cpu_baseline and args.config == "cifar10" and world == 1:   # the contract: rank 0 at N=1 only
        rate, dt, threads = cpu_reference_rate(16, 30)         # ~10-15 s of CPU work
        cpu = {"value": rate, "unit": "images/s", "cores": threads, "kind": "port",
               "sample": f"oracle CPU port of the reference loop, batch 16 (configs[0]), 30 of 100 Euler steps "
                         f"({dt:.1f} s), extrapolated linearly; threads = fastest of 8/16/32/64"}
    gpu_eager = None
    if not args.no_gpu_eager and args.config == "cifar10" and world == 1:
        torch.cuda.empty_cache()
        try:
            gpu_eager = gpu_eager_rate(dev)
        except Exception as ex:                                 # a baseline leg must never take the bench line down
            gpu_eager = {"unavailable": repr(ex)[:200]}

    line = {"metric": wl["metric"], "value": main_res["value"], "unit": "images/s", "n_gpus": world,
            "steps": steps, "warmup": warmup, "ms_per_step": main_res["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "%s, batch %d per GPU" % (wl["desc"], B),
                       "weights": "random-init (seeded factory)", "global_batch": world * B,
                       "parallelism": "dp%d" % world,
                       "l2": "per-step working set (>= 2 GB of activations) exceeds the 126 MB L2"},
            "clocks": main_res["clocks"], "e2e": main_res["e2e"], "gpu_launches": main_res["launches"],
            "roofline": main_res["roofline"], "cpu_baseline": cpu, "gpu_eager_baseline": gpu_eager,
            "secondary": secondary}
    if big:
        line["config"]["l2"] = "per-step working set (>= 10 GB of activations) exceeds the 126 MB L2"
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
