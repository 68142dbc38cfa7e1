"""Generate the golden fixtures under tests/golden/ by running the REFERENCE'S OWN modules (imported from the
reference checkout, oracle/stage_reference.reference_dir()) on the synthetic weights of oracle/synth.py.

    python tests/golden/make_golden.py [--full] [--traj celeba16,afhq,imagenet]

The fixtures pin the oracle (tests/test_oracle.py, CPU) and are what the CUDA engine is compared with on the GPU,
where the tests never read the reference itself.  Nothing here is imported by the product package.

Fixtures (npz, fp32):
  ddpm_mini.npz / adm_mini.npz      full tensors of reduced configurations: plain forward, Asyrp forward
                                    (t >= t_edit and t < t_edit), 10-step edit trajectory with a stochastic tail
  ddpm_celeba_fwd.npz               CelebA-HQ config, 256x256, B=1, Asyrp forward at t=999 (stride-4 subsample)
  ddpm_celeba_traj40.npz            40-step Asyrp edit trajectory, B=1 (stride-4 subsample of x_0 + per-step |x0_t| max)
  adm_afhq_fwd.npz, adm_imagenet_fwd.npz   one Asyrp forward each (stride-4 subsample)
  checkpoint/*.pth                  the three shipped DeltaBlocks SURVEY §8(d) names, key "0" only
                                    ({"0": layer_0.state_dict()}, the part diffusion_latent.py:674-676 loads)
  ddpm_celeba_smiling_traj40_b16.npz   BASELINE configs[1] in full: B=16, 40-step edit, 'smiling' DeltaBlock
  adm_afhq_happy_traj40.npz            configs[2] at B=1: iDDPM-AFHQ, 'dog_happy' DeltaBlock, 40 steps
  ddpm_church_gothic_traj40.npz        configs[3] at B=1: DDPM LSUN-Church (same UNet as CelebA), 'church_gothic' block
  adm_imagenet_traj50.npz              configs[4] at B=1: ADM-ImageNet, seeded DeltaBlock, 50 steps
  ddpm_celeba_bounded_t400.npz         the pipeline in the image range (|x| < 2 throughout): inversion of a synthetic image
                                    + 40-step edit at --t_0 400 with conv_out scaled by 0.03; full x_T and x_0 (--traj bounded)
                                    (trajectory fixtures: stride-4 subsample of x_0, |x_0| max, seeds, sequence)
"""
import argparse
import os
import sys
import time
from types import SimpleNamespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle.stage_reference import reference_dir  # noqa: E402
REF = reference_dir()
sys.path.insert(0, REF)

from oracle import adm as o_adm, ddpm as o_ddpm, sampler as o_smp, synth  # noqa: E402

from models.ddpm.diffusion import DDPM  # noqa: E402  (reference)
from models.improved_ddpm.unet import UNetModel  # noqa: E402  (reference)
from models.improved_ddpm.script_util import i_DDPM  # noqa: E402  (reference)
import utils.diffusion_utils as ref_du  # noqa: E402  (reference)


def ref_ddpm(cfg, n_delta):
    c = SimpleNamespace(model=SimpleNamespace(ch=cfg["ch"], out_ch=cfg["out_ch"], ch_mult=list(cfg["ch_mult"]),
                                              num_res_blocks=cfg["num_res_blocks"],
                                              attn_resolutions=list(cfg["attn_resolutions"]), dropout=0.0,
                                              in_channels=cfg["in_channels"], resamp_with_conv=True),
                        data=SimpleNamespace(image_size=cfg["image_size"]))
    m = DDPM(c)
    m.setattr_layers(n_delta)
    return m.eval()


def ref_adm(hp, n_delta):
    ds = tuple(hp["image_size"] // r for r in hp["attention_resolutions"])
    m = UNetModel(image_size=hp["image_size"], in_channels=3, model_channels=hp["model_channels"],
                  out_channels=hp["out_channels"], num_res_blocks=hp["num_res_blocks"], attention_resolutions=ds,
                  dropout=0.0, channel_mult=hp["channel_mult"], num_classes=None, use_checkpoint=False,
                  use_fp16=False, num_heads=4, num_head_channels=hp["num_head_channels"], num_heads_upsample=-1,
                  use_scale_shift_norm=True, resblock_updown=True, use_new_attention_order=False)
    m.setattr_layers(n_delta)
    return m.eval()


def load_checked(model, shapes, sd, ignore=()):
    """the oracle's parameter inventory must equal the reference module's state_dict (names and shapes)"""
    ref_sd = {k: tuple(v.shape) for k, v in model.state_dict().items() if not k.startswith(tuple(ignore))}
    mine = {k: tuple(v) for k, v in shapes.items()}
    assert ref_sd == mine, (sorted(set(ref_sd) ^ set(mine))[:10],
                            [(k, ref_sd[k], mine[k]) for k in ref_sd if k in mine and ref_sd[k] != mine[k]][:10])
    res = model.load_state_dict(sd, strict=False)
    assert not res.unexpected_keys and all(k.startswith(tuple(ignore)) for k in res.missing_keys), res


def ref_trajectory(model, x_T, betas, seq, seq_next, t_edit, t_addnoise, learn_sigma, noises, rec):
    """diffusion_latent.py:499-520 with the reference denoising_step; randn_like replaced by the pre-drawn noise"""
    x = x_T.clone()
    bs = x.shape[0]
    for i, j in zip(reversed(seq), reversed(seq_next)):
        t = torch.ones(bs) * i
        t_next = torch.ones(bs) * j
        orig = torch.randn_like
        ref_du.torch.randn_like = lambda ten, _i=i: noises[_i]
        try:
            x, x0_t, _, _ = ref_du.denoising_step(x, t=t, t_next=t_next, models=model, logvars=None if learn_sigma else
                                                  o_smp.make_logvar(o_smp.get_beta_schedule(
                                                      beta_start=1e-4, beta_end=0.02, num_diffusion_timesteps=1000)),
                                                  sampling_type="ddim", b=betas, learn_sigma=learn_sigma, index=0,
                                                  eta=1.0 if i < t_addnoise else 0.0, t_edit=t_edit,
                                                  hs_coeff=(1.0, 1.0), delta_h=None, ignore_timestep=False,
                                                  dt_lambda=1, warigari=False)
        finally:
            ref_du.torch.randn_like = orig
        rec.append((i, x0_t))
    return x


def sub(t, s=4):
    return t[..., ::s, ::s].contiguous().numpy()


@torch.no_grad()
def mini(family):
    if family == "ddpm":
        cfg = o_ddpm.MINI_CFG
        shapes = o_ddpm.ddpm_param_shapes(cfg, 1)
        model = ref_ddpm(cfg, 1)
        fwd = lambda sd, *a, **k: o_ddpm.ddpm_forward(sd, cfg, *a, **k)  # noqa: E731
        learn_sigma = False
    else:
        cfg = o_adm.MINI_HP
        shapes = o_adm.adm_param_shapes(cfg, 1)
        model = ref_adm(cfg, 1)
        fwd = lambda sd, *a, **k: o_adm.adm_forward(sd, cfg, *a, **k)  # noqa: E731
        learn_sigma = True
    sd = synth.synth_state_dict(shapes, seed=1234, style="jittered")
    load_checked(model, shapes, sd)
    B, S = 2, cfg["image_size"]
    x = synth.synth_noise((B, 3, S, S), seed=1234)
    out = {}
    # plain forward (index=None), Asyrp forward above and below t_edit
    cases = {"plain": dict(t=999.0), "edit": dict(t=600.0, index=0, t_edit=500, hs_coeff=(1.0, 0.7)),
             "pass": dict(t=300.0, index=0, t_edit=500, hs_coeff=(1.0, 0.7))}
    for name, kw in cases.items():
        kw = dict(kw)
        t = torch.ones(B) * kw.pop("t")
        r = model(x, t, **kw)
        o = fwd(sd, x, t, **kw)
        for key, a, b in zip(("et", "et_mod", "delta_h", "middle_h"), r, o):
            if a is None:
                assert b is None
                continue
            assert torch.equal(a, b), f"oracle != reference: {family} {name} {key} {(a - b).abs().max()}"
            out[f"{name}_{key}"] = a.numpy()
    # 10-step trajectory, t_edit=500, stochastic (eta=1) below t_addnoise=300
    betas = o_smp.make_betas()
    seq, seq_next = o_smp.make_sequences(999, 10)
    g = torch.Generator().manual_seed(4321)
    noises = {i: torch.randn(x.shape, generator=g) for i in seq}
    rec = []
    xf = ref_trajectory(model, x, betas, seq, seq_next, 500, 300, learn_sigma, noises, rec)
    rec_o = []
    xo = o_smp.run_trajectory(lambda *a, **k: fwd(sd, *a, **k), x, betas=betas, seq=seq, seq_next=seq_next,
                              t_edit=500, t_addnoise=300, index=0, hs_coeff=(1.0, 1.0), learn_sigma=learn_sigma,
                              noises=noises, record=rec_o)
    assert torch.equal(xf, xo), (xf - xo).abs().max()
    out["traj_x0"] = xf.numpy()
    out["traj_x0t"] = np.stack([r[1].numpy() for r in rec])
    out["traj_noise_seed"] = np.array(4321)
    # DDIM inversion x_0 -> x_T and deterministic reconstruction with the plain UNet (precompute_pairs,
    # diffusion_latent.py:1032-1072): reference denoising_step with t < t_next, index=None
    x0img = torch.tanh(synth.synth_noise((B, 3, S, S), seed=77))
    logv = None if learn_sigma else o_smp.make_logvar(o_smp.get_beta_schedule(beta_start=1e-4, beta_end=0.02,
                                                                             num_diffusion_timesteps=1000))
    xr, xo_ = x0img.clone(), x0img.clone()
    for i, j in zip(seq_next[1:], seq[1:]):
        t, tn = torch.ones(B) * i, torch.ones(B) * j
        xr = ref_du.denoising_step(xr, t=t, t_next=tn, models=model, logvars=logv, sampling_type="ddim", b=betas, eta=0,
                                   learn_sigma=learn_sigma)[0]
        xo_ = o_smp.denoising_step(xo_, t, tn, model=lambda *a, **k: fwd(sd, *a, **k), logvars=logv, b=betas, eta=0.0,
                                   learn_sigma=learn_sigma)[0]
    assert torch.equal(xr, xo_), (xr - xo_).abs().max()
    out["inv_x0"], out["inv_xT"] = x0img.numpy(), xr.numpy()
    for i, j in zip(reversed(seq), reversed(seq_next)):
        t, tn = torch.ones(B) * i, torch.ones(B) * j
        xr = ref_du.denoising_step(xr, t=t, t_next=tn, models=model, logvars=logv, sampling_type="ddim", b=betas,
                                   learn_sigma=learn_sigma)[0]
    out["inv_rec"] = xr.numpy()
    np.savez_compressed(os.path.join(HERE, f"{family}_mini.npz"), **out)
    print(f"{family}_mini ok: |x_final|max={xf.abs().max():.3f}")


@torch.no_grad()
def full_forward(name, family, cfg, t_val=999.0):
    t0 = time.time()
    if family == "ddpm":
        shapes = o_ddpm.ddpm_param_shapes(cfg, 1)
        model = ref_ddpm(cfg, 1)
        fwd = lambda sd, *a, **k: o_ddpm.ddpm_forward(sd, cfg, *a, **k)  # noqa: E731
        ignore = ()
    else:
        shapes = o_adm.adm_param_shapes(cfg, 1)
        model = ref_adm(cfg, 1)
        fwd = lambda sd, *a, **k: o_adm.adm_forward(sd, cfg, *a, **k)  # noqa: E731
        ignore = ()
    sd = synth.synth_state_dict(shapes, seed=1234, style="torch_default")
    load_checked(model, shapes, sd, ignore)
    x = synth.synth_noise((1, 3, 256, 256), seed=1234)
    t = torch.ones(1) * t_val
    r = model(x, t, index=0, t_edit=500, hs_coeff=(1.0, 1.0))
    o = fwd(sd, x, t, index=0, t_edit=500, hs_coeff=(1.0, 1.0))
    out = {}
    for key, a, b in zip(("et", "et_mod", "delta_h", "middle_h"), r, o):
        assert torch.equal(a, b), f"oracle != reference: {name} {key} {(a - b).abs().max()}"
        out[key] = sub(a) if a.shape[-1] == 256 else a.numpy()
        out[key + "_absmax"] = np.array(a.abs().max().item())
        out[key + "_mean"] = np.array(a.double().mean().item())
        out[key + "_std"] = np.array(a.double().std().item())
    np.savez_compressed(os.path.join(HERE, f"{name}_fwd.npz"), **out)
    print(f"{name}_fwd ok ({time.time() - t0:.1f}s): |et|max={r[0].abs().max():.3f} |et_mod|max={r[1].abs().max():.3f}")
    return model, sd


@torch.no_grad()
def full_trajectory(model, sd, cfg):
    """BASELINE config 2 restricted to B=1: DDPM CelebA-HQ 256x256, 40-step Asyrp edit, t_edit=500, t_addnoise=200"""
    t0 = time.time()
    x = synth.synth_noise((1, 3, 256, 256), seed=1234)
    betas = o_smp.make_betas()
    seq, seq_next = o_smp.make_sequences(999, 40)
    g = torch.Generator().manual_seed(4321)
    noises = {i: torch.randn(x.shape, generator=g) for i in seq}
    rec = []
    xf = ref_trajectory(model, x, betas, seq, seq_next, 500, 200, False, noises, rec)
    out = {"x0": sub(xf), "x0_absmax": np.array(xf.abs().max().item()), "x0_std": np.array(xf.double().std().item()),
           "x0t_absmax": np.array([r[1].abs().max().item() for r in rec]),
           "x0_full_f16": xf.to(torch.float16).numpy()}
    np.savez_compressed(os.path.join(HERE, "ddpm_celeba_traj40.npz"), **out)
    print(f"ddpm_celeba_traj40 ok ({time.time() - t0:.1f}s): |x_0|max={xf.abs().max():.2f}")


SHIPPED = {"celeba": "smiling_LC_CelebA_HQ_t999_ninv40_ngen40_0.pth", "afhq": "dog_happy_LC_dog_t999_ninv40_ngen40_0.pth",
           "church": "church_gothic_LC_church_outdoor_t999_ninv40_ngen40_0.pth"}


def shipped_delta_block(key):
    """copy the DeltaBlock weights of a shipped checkpoint (checkpoint/<name>.pth, key "0") into tests/golden/checkpoint/"""
    src = torch.load(os.path.join(REF, "checkpoint", SHIPPED[key]), map_location="cpu", weights_only=True)
    os.makedirs(os.path.join(HERE, "checkpoint"), exist_ok=True)
    blk = {k: v.clone() for k, v in src["0"].items()}
    torch.save({"0": blk}, os.path.join(HERE, "checkpoint", SHIPPED[key]))
    return blk


@torch.no_grad()
def trajectory_fixture(name, family, cfg, key, B, n_step, chunk=4):
    """BASELINE workload `name`: the reference's own modules + denoising_step, synthetic seeded UNet weights
    (torch_default style), the shipped DeltaBlock where one exists, x_T = randn(B,3,256,256; seed 1234), pre-drawn noise
    (seed 4321, one draw per sequence entry in ascending order), t_edit=500, t_addnoise=200, hs_coeff (1,1)"""
    t0 = time.time()
    if family == "ddpm":
        shapes = o_ddpm.ddpm_param_shapes(cfg, 1)
        model = ref_ddpm(cfg, 1)
        fwd = lambda sd, *a, **k: o_ddpm.ddpm_forward(sd, cfg, *a, **k)  # noqa: E731
    else:
        shapes = o_adm.adm_param_shapes(cfg, 1)
        model = ref_adm(cfg, 1)
        fwd = lambda sd, *a, **k: o_adm.adm_forward(sd, cfg, *a, **k)  # noqa: E731
    sd = synth.synth_state_dict(shapes, seed=1234, style="torch_default")
    if key in SHIPPED:
        for k, v in shipped_delta_block(key).items():
            assert sd["layer_0." + k].shape == v.shape, k
            sd["layer_0." + k] = v
    load_checked(model, shapes, sd)
    g = torch.Generator().manual_seed(1234)
    x = torch.randn(B, 3, 256, 256, generator=g)
    betas = o_smp.make_betas()
    seq, seq_next = o_smp.make_sequences(999, n_step)
    gn = torch.Generator().manual_seed(4321)
    noises = {i: torch.randn(x.shape, generator=gn) for i in seq}
    outs = []
    for c0 in range(0, B, chunk):
        sl = slice(c0, min(B, c0 + chunk))
        nz = {i: v[sl] for i, v in noises.items()}
        rec = []
        xf = ref_trajectory(model, x[sl], betas, seq, seq_next, 500, 200, family == "adm", nz, rec)
        if c0 == 0:  # the oracle restatement must reproduce the reference bit for bit (first sample)
            xo = o_smp.run_trajectory(lambda *a, **k: fwd(sd, *a, **k), x[:1], betas=betas, seq=seq, seq_next=seq_next,
                                      t_edit=500, t_addnoise=200, index=0, hs_coeff=(1.0, 1.0),
                                      learn_sigma=family == "adm", noises={i: v[:1] for i, v in noises.items()})
            # bit-equal at equal batch size (checked by mini() / full_trajectory()); here the reference ran a chunk of
            # `chunk` samples and oneDNN blocks a B=4 conv differently from a B=1 one: ~1e-6 relative
            assert (xo - xf[:1]).abs().max() <= 2e-5 * xf[:1].abs().max(), (xo - xf[:1]).abs().max()
        outs.append(xf)
        print(f"  {name}: samples {sl.start}..{sl.stop - 1} done ({time.time() - t0:.0f}s)", flush=True)
    xf = torch.cat(outs)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), x0_sub=sub(xf), x0_absmax=np.array(xf.abs().max().item()),
                        x0_absmax_per_sample=xf.abs().amax(dim=(1, 2, 3)).numpy(), x0_std=np.array(xf.double().std().item()),
                        batch=np.array(B), x_seed=np.array(1234), noise_seed=np.array(4321), seq=np.array(seq),
                        t_edit=np.array(500), t_addnoise=np.array(200))
    print(f"{name} ok ({time.time() - t0:.1f}s): |x_0|max={xf.abs().max():.2f}")


@torch.no_grad()
def bounded_fixture(gamma=0.03, t_0=400, n_step=40, t_edit=200, t_addnoise=80):
    """The Asyrp pipeline in the IMAGE range, at full size: DDPM CelebA-HQ 256x256, synthetic seeded weights + the shipped
    'smiling' DeltaBlock, conv_out (weight and bias) scaled by `gamma`, --t_0 400 (a flag of the reference,
    1/sqrt(alpha-bar_400) = 2.2 instead of 160): precompute_pairs' inversion of a synthetic image in [-1, 1]
    (diffusion_latent.py:922-933), then save_image's edit loop (:499-520) from that x_T.  Everything stays within
    |x| < 2 (the UNet sees ordinary O(1) inputs at every step), so the engine-vs-reference error of this fixture is
    an ABSOLUTE number on an O(1)-range image.  Reference's own modules + denoising_step; oracle must agree bit for bit."""
    t0 = time.time()
    cfg = o_ddpm.CELEBA_CFG
    shapes = o_ddpm.ddpm_param_shapes(cfg, 1)
    model = ref_ddpm(cfg, 1)
    sd = synth.synth_state_dict(shapes, seed=1234, style="torch_default")
    for k, v in shipped_delta_block("celeba").items():
        sd["layer_0." + k] = v
    sd["conv_out.weight"] = sd["conv_out.weight"] * gamma
    sd["conv_out.bias"] = sd["conv_out.bias"] * gamma
    load_checked(model, shapes, sd)
    fwd = lambda *a, **k: o_ddpm.ddpm_forward(sd, cfg, *a, **k)  # noqa: E731
    x0 = synth.synth_image((1, 3, 256, 256), seed=77).to(torch.float16).float()  # stored as fp16: exactly representable
    betas = o_smp.make_betas()
    seq, seq_next = o_smp.make_sequences(t_0, n_step)
    logv = o_smp.make_logvar(o_smp.get_beta_schedule(beta_start=1e-4, beta_end=0.02, num_diffusion_timesteps=1000))
    xr, xo = x0.clone(), x0.clone()
    for i, j in zip(seq_next[1:], seq[1:]):
        t, tn = torch.ones(1) * i, torch.ones(1) * j
        xr = ref_du.denoising_step(xr, t=t, t_next=tn, models=model, logvars=logv, sampling_type="ddim", b=betas, eta=0,
                                   learn_sigma=False)[0]
        xo = o_smp.denoising_step(xo, t, tn, model=fwd, logvars=logv, b=betas, eta=0.0)[0]
    assert torch.equal(xr, xo), (xr - xo).abs().max()
    x_T = xr
    gn = torch.Generator().manual_seed(4321)
    noises = {i: torch.randn(x0.shape, generator=gn) for i in seq}
    rec = []
    xf = ref_trajectory(model, x_T, betas, seq, seq_next, t_edit, t_addnoise, False, noises, rec)
    xo = o_smp.run_trajectory(fwd, x_T, betas=betas, seq=seq, seq_next=seq_next, t_edit=t_edit, t_addnoise=t_addnoise,
                              index=0, hs_coeff=(1.0, 1.0), noises=noises, logvars=logv)
    assert torch.equal(xf, xo), (xf - xo).abs().max()
    np.savez_compressed(os.path.join(HERE, "ddpm_celeba_bounded_t400.npz"), x0_in=x0.to(torch.float16).numpy(),
                        x_T=x_T.numpy(), x0_out=xf.numpy(), gamma=np.array(gamma), t_0=np.array(t_0), seq=np.array(seq),
                        t_edit=np.array(t_edit), t_addnoise=np.array(t_addnoise), noise_seed=np.array(4321),
                        x0t_absmax=np.array([r[1].abs().max().item() for r in rec]))
    print(f"ddpm_celeba_bounded_t400 ok ({time.time() - t0:.0f}s): |x_0 in| {x0.abs().max():.3f} |x_T| {x_T.abs().max():.3f} "
          f"|x_0 out| {xf.abs().max():.3f} |x_0 out - x_0 in| {(xf - x0).abs().max():.3f} (rms {(xf - x0).pow(2).mean().sqrt():.3f}) "
          f"max_t |x0_t| {max(r[1].abs().max().item() for r in rec):.3f}")


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--full", action="store_true", help="also the 256x256 fixtures (minutes of CPU time)")
    ap.add_argument("--traj", default="", help="comma list of trajectory fixtures: celeba16, afhq, imagenet, church, bounded")
    ap.add_argument("--skip-mini", action="store_true")
    args = ap.parse_args()
    torch.set_num_threads(os.cpu_count())
    for t in [t for t in args.traj.split(",") if t]:
        if t == "celeba16":
            trajectory_fixture("ddpm_celeba_smiling_traj40_b16", "ddpm", o_ddpm.CELEBA_CFG, "celeba", 16, 40)
        elif t == "afhq":
            trajectory_fixture("adm_afhq_happy_traj40", "adm", o_adm.AFHQ_HP, "afhq", 1, 40)
        elif t == "imagenet":
            trajectory_fixture("adm_imagenet_traj50", "adm", o_adm.IMAGENET_HP, "imagenet", 1, 50)
        elif t == "church":
            trajectory_fixture("ddpm_church_gothic_traj40", "ddpm", o_ddpm.CELEBA_CFG, "church", 1, 40)
        elif t == "bounded":
            bounded_fixture()
        else:
            raise SystemExit(f"unknown trajectory fixture {t}")
    if args.skip_mini:
        sys.exit(0)
    mini("ddpm")
    mini("adm")
    if args.full:
        m, sd = full_forward("ddpm_celeba", "ddpm", o_ddpm.CELEBA_CFG)
        full_trajectory(m, sd, o_ddpm.CELEBA_CFG)
        del m, sd
        full_forward("adm_afhq", "adm", o_adm.AFHQ_HP)
        full_forward("adm_imagenet", "adm", o_adm.IMAGENET_HP)
