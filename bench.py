#!/usr/bin/env python
"""Benchmark of the Asyrp hot path: 256x256 images/sec for a complete 40-step Asyrp edit trajectory.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--batch B] [--workload NAME]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One "step" = one pass of the hot path over one batch: x_T -> x_0 through all 40 reverse steps (20 of them with the
Δh injection and the second decoder pass, 8 with injected noise; t_edit=500, t_addnoise=200).  Workload at N=1 is
BASELINE.json configs[1] (DDPM CelebA-HQ 256x256, batch 16, the shipped 'smiling' DeltaBlock); every rank runs the same
per-GPU batch (weak scaling, each sample's trajectory is independent; the only collective is the one-time weight
broadcast).

Prints ONE JSON line (rank 0):
  value          device-timed (CUDA events, inputs resident in HBM), whole job
  e2e            through Asyrp.edit_batch with pinned host buffers (H2D of x_T, D2H of x_0 inside the timed region)
  roofline       the tcgen05 conv kernel: algorithmic conv FLOPs of one edit-step UNet evaluation / (device time of the
                 captured evaluation minus that of its non-conv launches; CUDA graphs, CUDA events), vs the measured
                 sustained bf16 cuBLAS peak; `traffic` is read from the committed ncu capture under profiles/
  parity         engine vs the REFERENCE's own output (tests/golden/, written by tests/golden/make_golden.py) on the
                 same weights / x_T / noise, for this workload
  cpu_baseline   the reference's own CPU code (oracle/_ref, staged by oracle/stage_reference.py; falls back to the
                 restatement oracle/ = kind "port") on a bounded sample, on the host's cores
  eager_gpu_baseline  the reference's own modules + denoising_step in eager PyTorch (TF32 default) on the same B200

`--dump-outputs DIR` writes what the device-timed path computed in its last step: DIR/x0.npy, the float32 x_0 of the
whole job (every rank's batch shard, in rank order, gathered to rank 0).  Weights, x_T and the pre-drawn noise are
seeded, so two builds run with the same arguments can be compared output for output.

`--impl reference` times the reference's CPU implementation: a "step" there is a bounded sample (one edit reverse step
+ one non-edit reverse step at B=1, scaled x n_edit / x n_plain to a trajectory), `ms_per_step` is the measured time of
that sample, and one full B=1 trajectory is run in the warm-up to validate the scaling.
"""
import argparse
import csv
import glob
import json
import os
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
GOLD = os.path.join(ROOT, "tests", "golden")

METRIC = "256x256 images/sec, 40-step Asyrp edit"
WORKLOADS = {
    # name: (family, config key, per-GPU batch, steps in trajectory, DeltaBlock checkpoint, golden trajectory)
    "ddpm_celeba_b16": ("ddpm", "celeba", 16, 40, "smiling_LC_CelebA_HQ_t999_ninv40_ngen40_0.pth",
                        "ddpm_celeba_smiling_traj40_b16.npz"),
    "iddpm_afhq_b8": ("adm", "afhq", 8, 40, "dog_happy_LC_dog_t999_ninv40_ngen40_0.pth", "adm_afhq_happy_traj40.npz"),
    "ddpm_church_b32": ("ddpm", "church", 32, 40, "church_gothic_LC_church_outdoor_t999_ninv40_ngen40_0.pth",
                        "ddpm_church_gothic_traj40.npz"),
    "adm_imagenet_b4": ("adm", "imagenet", 4, 50, None, "adm_imagenet_traj50.npz"),
}
# algorithmic GFLOP per image per UNet pass (2*MAC), SURVEY.md §8(d): encoder, decoder, delta block
FLOPS = {"celeba": (135.1, 361.9, 0.07), "church": (135.1, 361.9, 0.07), "afhq": (78.9, 309.0, 0.07),
         "imagenet": (580.4, 1659.3, 0.27)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["bf16_tflops_sustained"], d["hbm_gbs"], d.get("bf16_tflops"), \
            "measured (MEASURED_PEAKS.json: sustained bf16 cuBLAS for a kernel timed inside a long step)"
    return 1400.0, 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons during the timed region (pynvml, 100 ms period)"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag = index, [], set(), False
        self.max_mhz = None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                     nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
            while not self.stop_flag:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
                time.sleep(0.1)
        except Exception as e:  # noqa: BLE001
            self.reasons.add(f"sampler_error:{type(e).__name__}")

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def load_delta_block(model, ckpt):
    """the shipped DeltaBlock of SURVEY §8(d) (tests/golden/checkpoint/, format {"0": layer_0.state_dict()},
    diffusion_latent.py:674-676); seeded random where the reference ships none (ImageNet)"""
    p = os.path.join(GOLD, "checkpoint", ckpt) if ckpt else None
    if p and os.path.exists(p):
        model.layer_0.load_state_dict(torch.load(p, map_location="cpu", weights_only=True)["0"])
        return ckpt
    return "seeded random DeltaBlock"


def build_model(family, key, device, ckpt=None, seed=1234):
    from asyrp_official_b200 import arch, modules, synthetic
    from asyrp_official_b200.configs import load_config
    if family == "ddpm":
        model = modules.DDPM(load_config(key))
    else:
        model = modules._create_adm({"afhq": arch.AFHQ_HP, "imagenet": arch.IMAGENET_HP}[key])
    model.setattr_layers(1)
    synthetic.randomize_(model, seed=seed)  # UNet and DeltaBlock: seeded random init, never zeroed
    delta = load_delta_block(model, ckpt)
    return model.to(device), delta


def dump_outputs(d, arrays, max_bytes=64 * 10**6, seed=1234):
    """--dump-outputs: each tensor as d/<name>.npy in float32, max_bytes in all; a tensor over its share keeps a seeded
    sample of its leading-axis rows (ascending), the same rows in every run with the same arguments"""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    share = max_bytes // len(arrays)
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        if a.nbytes > share:
            rows = max(1, share // (a.nbytes // a.shape[0]))
            a = a[np.sort(np.random.default_rng(seed).choice(a.shape[0], rows, replace=False))]
        np.save(os.path.join(d, f"{name}.npy"), a)


def f_img(key, steps, n_edit):
    e, d, dl = FLOPS[key]
    return (steps * (e + d) + n_edit * (d + dl)) * 1e9


# ---------------------------------------------------------------------------------------------------------------
# the reference itself (oracle/_ref): CPU arm, CPU baseline, eager-GPU baseline
# ---------------------------------------------------------------------------------------------------------------
def reference_model(family, key, state_dict, device):
    """the reference's own UNet class (models/ddpm/diffusion.py:327, improved_ddpm/script_util.py:102) holding
    `state_dict`; None when oracle/_ref has not been staged"""
    if not os.path.isdir(os.path.join(REF_DIR, "models")):
        return None, None
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    import importlib
    du = importlib.import_module("utils.diffusion_utils")
    if family == "ddpm":
        from asyrp_official_b200.configs import load_config
        m = importlib.import_module("models.ddpm.diffusion").DDPM(load_config(key))
    else:
        m = importlib.import_module("models.improved_ddpm.script_util").i_DDPM({"afhq": "AFHQ", "imagenet": "IMAGENET"}[key])
    m.setattr_layers(1)
    res = m.load_state_dict(state_dict, strict=False)
    assert not res.unexpected_keys and not [k for k in res.missing_keys if "label_emb" not in k], res
    return m.eval().to(device), du


def reference_trajectory(model, du, x, seq, seq_next, betas, logvar, learn_sigma, t_edit=500, t_addnoise=200,
                         only=None):
    """the loop of Asyrp.save_image (diffusion_latent.py:499-520) around the reference's denoising_step; `only`: a list
    of step indices to run (bounded sample) -> per-step wall times"""
    times = []
    dev = x.device
    bs = x.shape[0]
    with torch.no_grad():
        for k, (i, j) in enumerate(zip(reversed(seq), reversed(seq_next))):
            if only is not None and k not in only:
                continue
            t = (torch.ones(bs) * i).to(dev)
            t_next = (torch.ones(bs) * j).to(dev)
            t0 = time.perf_counter()
            x, _, _, _ = du.denoising_step(x, t=t, t_next=t_next, models=model, logvars=logvar, sampling_type="ddim",
                                           b=betas, learn_sigma=learn_sigma, index=0,
                                           eta=1.0 if i < t_addnoise else 0.0, t_edit=t_edit, hs_coeff=(1.0, 1.0),
                                           delta_h=None, ignore_timestep=False, dt_lambda=1)
            if dev.type == "cuda":
                torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
    return x, times


def cpu_setup(family, key, ckpt, traj_steps):
    mirror, delta = build_model(family, key, "cpu", ckpt)
    sd = {k: v.float() for k, v in mirror.state_dict().items()}
    from asyrp_official_b200.schedule import make_sequences
    from asyrp_official_b200.utils.diffusion_utils import get_beta_schedule
    import numpy as np
    b64 = get_beta_schedule(beta_start=1e-4, beta_end=0.02, num_diffusion_timesteps=1000)
    betas = torch.from_numpy(b64).float()
    ac = np.cumprod(1.0 - b64)
    logvar = np.log(np.maximum(b64 * (1.0 - np.append(1.0, ac[:-1])) / (1.0 - ac), 1e-20))
    seq, seq_next = make_sequences(999, traj_steps)
    g = torch.Generator().manual_seed(1234)
    x = torch.randn(1, 3, 256, 256, generator=g)
    ref, du = reference_model(family, key, sd, torch.device("cpu"))
    if ref is not None:
        def run(only):
            return reference_trajectory(ref, du, x, seq, seq_next, betas, logvar, family == "adm", only=only)[1]
        kind = "reference"
    else:  # oracle/_ref not staged: the restatement (oracle/) — the one other place bench.py may execute oracle/
        from oracle import adm as oa, ddpm as od, sampler as osmp
        if family == "ddpm":
            fwd = lambda *a, **k: od.ddpm_forward(sd, od.CELEBA_CFG, *a, **k)  # noqa: E731
        else:
            hp = {"afhq": oa.AFHQ_HP, "imagenet": oa.IMAGENET_HP}[key]
            fwd = lambda *a, **k: oa.adm_forward(sd, hp, *a, **k)  # noqa: E731

        def run(only):
            ts = []
            for k, (i, j) in enumerate(zip(reversed(seq), reversed(seq_next))):
                if only is not None and k not in only:
                    continue
                t0 = time.perf_counter()
                osmp.denoising_step(x, torch.ones(1) * i, torch.ones(1) * j, model=fwd, b=betas,
                                    learn_sigma=family == "adm", index=0, t_edit=500, hs_coeff=(1.0, 1.0),
                                    logvars=logvar)
                ts.append(time.perf_counter() - t0)
            return ts
        kind = "port"
    return run, kind, seq, delta


def sample_indices(seq, t_edit=500):
    """one edit step (the first, t=999) and one non-edit step (first with t < t_edit) of the reversed sequence"""
    rs = list(reversed(seq))
    return 0, next(k for k, t in enumerate(rs) if t < t_edit), sum(1 for t in rs if t >= t_edit)


def pick_threads(run, k_e, k_p):
    """torch's CPU conv does not scale to every core of a large host: try all cores and 32, keep the faster"""
    best, best_thr = float("inf"), os.cpu_count()
    for thr in sorted({os.cpu_count(), min(32, os.cpu_count())}):
        torch.set_num_threads(thr)
        t = sum(run([k_e, k_p]))
        if t < best:
            best, best_thr = t, thr
    torch.set_num_threads(best_thr)
    return best_thr


def cpu_sample(run, kind, seq, traj_steps, reps=1):
    k_e, k_p, n_edit = sample_indices(seq)
    best = (float("inf"), float("inf"))
    for _ in range(reps):
        te, tp = run([k_e, k_p])
        if te + tp < sum(best):
            best = (te, tp)
    traj_s = n_edit * best[0] + (traj_steps - n_edit) * best[1]
    what = "the reference's own denoising_step + UNet (oracle/_ref)" if kind == "reference" else \
        "fp32 torch CPU restatement of the reference (oracle/)"
    return {"value": 1.0 / traj_s, "unit": "img/s", "cores": torch.get_num_threads(), "kind": kind,
            "sample": f"B=1: 1 edit reverse step ({best[0]:.2f}s) + 1 non-edit reverse step ({best[1]:.2f}s) of the "
                      f"{traj_steps}-step trajectory, scaled x{n_edit}/x{traj_steps - n_edit}; {what}, "
                      f"{torch.get_num_threads()} threads"}, best


def eager_gpu(family, key, ckpt, batch, traj_steps, dev, reps=2, golden=None):
    """the reference's modules + denoising_step, eager PyTorch on the B200 (cuDNN/cuBLAS, TF32 convs as torch's
    default): full trajectories at the bench batch"""
    mirror, _ = build_model(family, key, "cpu", ckpt)
    sd = {k: v.float() for k, v in mirror.state_dict().items()}
    ref, du = reference_model(family, key, sd, dev)
    if ref is None:
        return None
    import numpy as np
    from asyrp_official_b200.schedule import make_sequences
    from asyrp_official_b200.utils.diffusion_utils import get_beta_schedule
    b64 = get_beta_schedule(beta_start=1e-4, beta_end=0.02, num_diffusion_timesteps=1000)
    betas = torch.from_numpy(b64).float().to(dev)
    ac = np.cumprod(1.0 - b64)
    logvar = np.log(np.maximum(b64 * (1.0 - np.append(1.0, ac[:-1])) / (1.0 - ac), 1e-20))
    seq, seq_next = make_sequences(999, traj_steps)
    g = torch.Generator().manual_seed(1234)
    x = torch.randn(batch, 3, 256, 256, generator=g).to(dev)
    best = float("inf")
    for r in range(reps + 1):  # first pass = warm-up (cuDNN autotune off by default; lazy init)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        reference_trajectory(ref, du, x, seq, seq_next, betas, logvar, family == "adm")
        torch.cuda.synchronize()
        if r:
            best = min(best, time.perf_counter() - t0)
    ref_parity = None
    gp = os.path.join(GOLD, golden) if golden else None
    if gp and os.path.exists(gp):
        # how far the reference's OWN GPU path (cuDNN TF32 convs, torch's default) lands from its CPU fp32 output on
        # the golden inputs of this workload: the yardstick for the engine's `parity` (same fixture, same noise)
        gd = np.load(gp)
        gb = int(gd["batch"])
        g = torch.Generator().manual_seed(int(gd["x_seed"]))
        xg = torch.randn(gb, 3, 256, 256, generator=g)
        gn = torch.Generator().manual_seed(int(gd["noise_seed"]))
        noises = {i: torch.randn(xg.shape, generator=gn).to(dev) for i in gd["seq"].tolist()}
        order = [i for i in reversed(seq) if i < int(gd["t_addnoise"])]  # the stochastic steps (eta = 1 below t_addnoise), in loop order
        orig = torch.randn_like
        it = iter(order)
        torch.randn_like = lambda ten, *a, **k: noises[next(it)]
        try:
            xr, _ = reference_trajectory(ref, du, xg.to(dev), seq, seq_next, betas, logvar, family == "adm")
        finally:
            torch.randn_like = orig
        gref = torch.from_numpy(gd["x0_sub"])
        err = (xr.cpu()[..., ::4, ::4] - gref).abs().max().item()
        m = float(gd["x0_absmax"])
        ref_parity = {"max_abs": round(err, 5), "max_ref": round(m, 3), "rel": round(err / max(m, 1.0), 7), "batch": gb,
                      "what": f"{golden}: the reference's eager GPU run (TF32 convs) vs the reference's CPU fp32 run"}
    del ref
    torch.cuda.empty_cache()
    return {"value": round(batch / best, 3), "unit": "img/s", "batch": batch, "s_per_trajectory": round(best, 3),
            "parity_vs_cpu_reference": ref_parity,
            "how": "oracle/_ref modules + utils.diffusion_utils.denoising_step in the save_image loop "
                   "(diffusion_latent.py:499-520), eager PyTorch on cuda:0, fp32 tensors, "
                   f"cudnn.allow_tf32={torch.backends.cudnn.allow_tf32}, matmul.allow_tf32="
                   f"{torch.backends.cuda.matmul.allow_tf32}; the reference always runs both decoders (34.4 vs the "
                   "27.1 TFLOP/img the engine executes)"}


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant conv instantiation, from the newest
    committed ncu --set full summary under profiles/ (bytes), or None"""
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_conv_ncu_full.csv")))
    for f in reversed(files):
        try:
            rows = list(csv.reader(open(f)))
            hdr, units = rows[0], rows[1]
            ir, iw = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
            mult = {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}[units[ir]]
            r = rows[2]
            return (float(r[ir]) + float(r[iw])) * mult, os.path.relpath(f, ROOT), r[0]
        except Exception:  # noqa: BLE001
            continue
    return None, None, None


def parity_check(model, runner, sch_kw, golden, dev):
    """engine vs the reference's own output on the golden inputs of this workload (tests/golden/<golden>)"""
    import numpy as np
    p = os.path.join(GOLD, golden) if golden else None
    if not p or not os.path.exists(p):
        return None
    from asyrp_official_b200.schedule import Schedule
    gd = np.load(p)
    B = int(gd["batch"])
    g = torch.Generator().manual_seed(int(gd["x_seed"]))
    x = torch.randn(B, 3, 256, 256, generator=g)
    sch = Schedule(**sch_kw)
    gn = torch.Generator().manual_seed(int(gd["noise_seed"]))
    noises = {i: torch.randn(x.shape, generator=gn) for i in gd["seq"].tolist()}
    noise = torch.stack([noises[s.t] for s in sch.steps if s.stochastic]) if sch.n_stochastic else None
    x0 = runner.edit_batch(model, x, sch, noise=noise)
    ref = torch.from_numpy(gd["x0_sub"])
    err = (x0[..., ::4, ::4] - ref).abs().max().item()
    m = float(gd["x0_absmax"])
    return {"max_abs": round(err, 5), "max_ref": round(m, 3), "rel": round(err / max(m, 1.0), 7), "batch": B,
            "config": f"{golden}: reference's own modules + denoising_step on CPU fp32 vs the engine, same weights, "
                      "x_T and pre-drawn noise (stride-4 subsample of x_0)",
            "note": "random-init UNets are not denoisers: x0_t = (x_t - e*sqrt(1-abar))/sqrt(abar) amplifies e by "
                    "160 at t=999, so |x_0| ~ 8e2; rel = max_abs / max|x_0|"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="ddpm_celeba_b16", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=None, help="per-GPU batch override")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write x_0 of the last timed step as DIR/x0.npy (float32, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the b200 arm")
    family, key, batch, traj_steps, ckpt, golden = WORKLOADS[args.workload]
    batch = args.batch or batch
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    from asyrp_official_b200.schedule import Schedule, make_sequences
    from asyrp_official_b200.utils.diffusion_utils import get_beta_schedule
    betas = torch.from_numpy(get_beta_schedule(beta_start=1e-4, beta_end=0.02, num_diffusion_timesteps=1000)).float()
    seq, seq_next = make_sequences(999, traj_steps)
    sch_kw = dict(betas=betas, seq=seq, seq_next=seq_next, t_edit=500, t_addnoise=200, hs_coeff=(1.0, 1.0))
    sch = Schedule(**sch_kw)
    config = {"workload": f"{args.workload}: {family.upper()} {key} UNet 256x256, per-GPU batch {batch}, "
                          f"{traj_steps}-step Asyrp edit (t_edit=500 -> {sch.n_edit} edit steps, t_addnoise=200 -> "
                          f"{sch.n_stochastic} stochastic steps), DeltaBlock index 0 "
                          f"({ckpt or 'seeded random'}), hs_coeff (1,1)",
              "per_gpu_batch": batch, "global_batch": batch * args.gpus, "trajectory_steps": traj_steps,
              "parallelism": f"batch-sharded x{args.gpus} (one process per GPU, no per-step collective)",
              "cache": "per-step working set (GBs of activations) exceeds the 126 MB L2; no explicit flush needed"}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        t_wall = time.perf_counter()
        run, kind, seq_, _ = cpu_setup(family, key, ckpt, traj_steps)
        k_e, k_p, n_edit = sample_indices(seq_)
        pick_threads(run, k_e, k_p)  # warm-up leg 1: thread count
        full_s = None
        if args.warmup >= 1:         # warm-up leg 2: ONE full B=1 trajectory, validates the scaled sample
            t0 = time.perf_counter()
            run(None)
            full_s = time.perf_counter() - t0
        samples = []
        t0 = time.perf_counter()
        for _ in range(args.steps):
            samples.append(run([k_e, k_p]))
        timed = time.perf_counter() - t0
        te = sum(s[0] for s in samples) / len(samples)
        tp = sum(s[1] for s in samples) / len(samples)
        traj_s = n_edit * te + (traj_steps - n_edit) * tp
        value = 1.0 / traj_s
        cb = {"value": value, "unit": "img/s", "cores": torch.get_num_threads(), "kind": kind,
              "sample": f"each step = 1 edit reverse step ({te:.2f}s) + 1 non-edit reverse step ({tp:.2f}s) at B=1, "
                        f"scaled x{n_edit}/x{traj_steps - n_edit} to the {traj_steps}-step trajectory; "
                        f"{'the reference own code from oracle/_ref' if kind == 'reference' else 'oracle/ port'}, "
                        f"{torch.get_num_threads()} threads"}
        line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "img/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * timed / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config, "cpu_baseline": cb,
                "e2e": {"value": value, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "full_trajectory_check": None if full_s is None else {
                    "measured_s": round(full_s, 2), "scaled_sample_s": round(traj_s, 2),
                    "what": "one complete B=1 40-step trajectory of the reference (run in the warm-up) vs the "
                            "per-step sample scaled to a trajectory"},
                "note": "ms_per_step is the measured time of one bounded sample step (2 of the trajectory's reverse "
                        "steps), not of a trajectory; value scales it to images/sec",
                "wall_s": time.perf_counter() - t_wall}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ B200 arm
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 arm has no CPU fallback (use --impl reference)")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from asyrp_official_b200 import _lib
    from asyrp_official_b200.configs import load_config
    from asyrp_official_b200.diffusion_latent import Asyrp, broadcast_weights
    model, delta = build_model(family, key, dev, ckpt)
    if dist is not None:
        broadcast_weights(model)  # the path's one collective (NCCL over NVLink)
    cfg_ns = load_config("celeba" if family == "ddpm" else "afhq")
    runner = Asyrp(argparse.Namespace(user_defined_t_edit=500, user_defined_t_addnoise=200), cfg_ns, device=dev)
    runner.t_edit, runner.t_addnoise = 500, 200
    eng = model.engine
    g = torch.Generator().manual_seed(1234 + rank)
    x_host = torch.randn(batch, 3, 256, 256, generator=g).pin_memory()
    out_host = torch.empty_like(x_host).pin_memory()
    x_dev = x_host.to(dev)
    # seeded like x_T, on a generator of its own: the same noise in every run, whatever else draws random numbers
    noise = torch.randn(sch.n_stochastic, batch, 3, 256, 256, device=dev,
                        generator=torch.Generator(device=dev).manual_seed(1234 + rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-timed throughput: inputs resident in HBM, graph replay
    for _ in range(max(args.warmup, 1)):
        eng.sample(x_dev, sch, noise=noise, out=x_dev.new_empty(x_dev.shape))
    out_dev = torch.empty_like(x_dev)
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        eng.sample(x_dev, sch, noise=noise, out=out_dev)
    e1.record()
    barrier()
    sampler.stop_flag = True
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if dist is not None:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_per_step = ms.item() / args.steps
    value = batch * args.gpus / (ms_per_step / 1000.0)
    launches = eng.last_launches * args.steps
    if args.dump_outputs:
        x0 = out_dev
        if dist is not None:  # what a caller of the batch-sharded job receives: every rank's shard, in rank order
            shards = [torch.empty_like(out_dev) for _ in range(world)]
            dist.all_gather(shards, out_dev)
            x0 = torch.cat(shards)
        if rank == 0:
            dump_outputs(args.dump_outputs, {"x0": x0})

    # ---- end to end through the runner API: pinned host x_T -> device -> trajectory -> pinned host x_0
    for _ in range(2):
        runner.edit_batch(model, x_host, sch, out=out_host)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        runner.edit_batch(model, x_host, sch, out=out_host)
        torch.cuda.synchronize()
    t_e2e = torch.tensor([time.perf_counter() - t0], device=dev)
    if dist is not None:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    e2e = {"value": batch * args.gpus / (t_e2e.item() / args.steps), "unit": "img/s",
           "h2d_bytes_per_step": x_host.numel() * 4, "d2h_bytes_per_step": out_host.numel() * 4,
           "api": "Asyrp.edit_batch(model, x_T pinned host, schedule, out=pinned host)"}

    if rank != 0:
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return
    # ---- roofline of the dominant kernel (tcgen05 implicit-GEMM conv), timed inside the captured evaluation:
    # eval_ms   = device time of a CUDA graph holding ALL launches of one edit-step UNet evaluation (valid data flow,
    #             the clocks / power state of the real trajectory), replayed back to back, CUDA events around the replays
    # other_ms  = the same for a graph holding every NON-conv launch of that evaluation
    # conv_ms   = eval_ms - other_ms (launch gaps are charged to the conv kernel)
    # A graph of the conv launches alone is NOT used: without the GroupNorm finalise launches between them the
    # activations degenerate to NaN within a few replays, the board draws less power, clocks rise from ~1.57 to
    # 1.97 GHz and the kernel reads 25-30 % faster than it runs on real data (measured: 10.1 vs 13.1 ms).
    peak_tf, peak_gbs, burst_tf, peak_src = peaks()
    P = eng.plan(batch)
    seq_l = P.launches(True, temb=False)
    convs = [L for L in seq_l if L.kind == "conv"]
    others = [L for L in seq_l if L.kind != "conv"]
    ms_eval = P.graph_time(seq_l)
    ms_other = P.graph_time(others)
    ms_conv = ms_eval - ms_other
    conv_flops = sum(L.flops for L in convs)
    conv_tf = conv_flops / (ms_conv * 1e-3) / 1e12
    conv_exec_tf = sum(L.exec_flops for L in convs) / (ms_conv * 1e-3) / 1e12
    step_tf = value / args.gpus * f_img(key, traj_steps, sch.n_edit) / 1e12
    kinds = {}
    for L in others:
        kinds.setdefault(L.kind, []).append(L)
    kern = {}
    for k, ls in kinds.items():
        ms_k = P.graph_time(ls, reps=10, warm=2)
        nb = sum(L.nbytes for L in ls)
        kern[k] = {"ms": round(ms_k, 3), "launches": len(ls), "gbs": round(nb / (ms_k * 1e-3) / 1e9, 1) if nb else None}
    P.graph_time(seq_l, reps=1, warm=0)  # leave valid activations behind
    traffic, traffic_src, traffic_kernel = ncu_traffic()
    roofline = {"bound": "tensor", "kernel": "conv_gemm_kernel (tcgen05 implicit GEMM, fp16 operands, fp32 accumulate)",
                "achieved": round(conv_tf, 1), "peak": peak_tf, "unit": "TFLOP/s", "frac": round(conv_tf / peak_tf, 4),
                "traffic": traffic,
                "traffic_note": None if traffic is None else
                f"dram read+write bytes per launch of {traffic_kernel} from {traffic_src} (ncu --set full)",
                "peak_source": peak_src,
                "frac_of_burst_peak": (round(conv_tf / burst_tf, 4) if burst_tf else None),
                "executed_tflops": round(conv_exec_tf, 1),
                "executed_note": "the Upsample.conv launches issue 4/9 of their algorithmic MACs (sub-pixel phases); "
                                 "every other conv launch executes exactly its algorithmic FLOPs",
                "how": f"algorithmic conv FLOPs ({conv_flops / 1e12:.2f} TFLOP) of the {len(convs)} conv launches of one "
                       f"edit-step UNet evaluation at batch {batch} / (device time of the captured evaluation, "
                       f"{ms_eval:.3f} ms, minus that of its {len(others)} non-conv launches, {ms_other:.3f} ms); CUDA "
                       "graphs replayed 20x back to back, CUDA events around the replays",
                "conv_ms": round(ms_conv, 3), "eval_ms": round(ms_eval, 3), "other_ms": round(ms_other, 3),
                "conv_share_of_step": round(ms_conv / ms_eval, 4), "launches_per_edit_eval": len(seq_l),
                "whole_step": {"achieved": round(step_tf, 1), "frac": round(step_tf / peak_tf, 4),
                               "f_img_tflop": round(f_img(key, traj_steps, sch.n_edit) / 1e12, 2)},
                "other_kernels": kern}
    parity = None if args.no_parity else parity_check(model, runner, sch_kw, golden, dev)
    cb = None
    if not args.no_cpu_baseline:
        run, kind, seq_, _ = cpu_setup(family, key, ckpt, traj_steps)
        k_e, k_p, _ = sample_indices(seq_)
        pick_threads(run, k_e, k_p)
        cb, _ = cpu_sample(run, kind, seq_, traj_steps, reps=2)
    eager = None
    if not args.no_eager_baseline:
        try:
            eager = eager_gpu(family, key, ckpt, batch, traj_steps, dev, golden=golden)
        except Exception as e:  # noqa: BLE001
            eager = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
    line = {"metric": METRIC, "value": round(value, 3), "unit": "img/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms_per_step, 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16", "data": f"synthetic (seeded random UNet weights, {delta}, "
            "Gaussian x_T)", "config": config, "roofline": roofline, "cpu_baseline": cb, "e2e": e2e,
            "gpu_launches": launches, "clocks": sampler.summary(), "parity": parity, "eager_gpu_baseline": eager,
            "pdl": bool(_lib.load().asyrp_get_pdl())}
    print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
