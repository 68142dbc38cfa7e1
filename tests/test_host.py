"""Host-side logic and the C-ABI surface (no GPU): library loads and exports every declared symbol, state-dict /
checkpoint compatibility of the module mirrors, schedule coefficients, config / CLI surface, loud failure without
a CUDA device."""
import argparse
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from asyrp_official_b200 import _lib
    from asyrp_official_b200.build import build_library
    build_library()
    hdr = open(os.path.join(ROOT, "include", "asyrp_b200.h")).read()
    declared = set(re.findall(r"\b(asyrp_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 15
    lib = _lib.load()
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/asyrp_b200.h but not exported"
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    assert lib.asyrp_last_error() is not None
    # pure host helper (no device): tile bookkeeping for the GroupNorm partial sums
    assert lib.asyrp_conv_stats_tiles(256, 256, 256, 0) == 512  # 128x256 tiles
    lib.asyrp_set_pair128(0)
    assert lib.asyrp_conv_stats_tiles(256, 256, 128, 1) == 512  # swapped 128x256 tiles, two slots each
    assert lib.asyrp_conv_tile_config(256, 256, 128, 1) == 128 * 16 + 2
    lib.asyrp_set_pair128(1)
    assert lib.asyrp_conv_stats_tiles(256, 256, 128, 1) == 256  # CTA pairs, 256 px x 128 ch per CTA: one slot per tile
    assert lib.asyrp_conv_tile_config(256, 256, 128, 1) == 128 * 16 + 2 + (1 << 16)
    lib.asyrp_set_pair128(-1)
    assert lib.asyrp_conv_stats_tiles(8, 8, 512, 1) == 4        # 2 samples per tile, one slot per lane quarter


def test_no_cpu_fallback():
    from asyrp_official_b200 import modules
    from asyrp_official_b200._lib import AsyrpError
    from asyrp_official_b200.configs import load_config
    cfg = load_config("celeba")
    cfg.model.ch, cfg.model.ch_mult, cfg.data.image_size = 64, [1, 2], 32
    m = modules.DDPM(cfg)
    if not torch.cuda.is_available():
        with pytest.raises(AsyrpError):
            m(torch.zeros(1, 3, 32, 32), torch.zeros(1))


def test_param_inventory_matches_oracle_inventory():
    from asyrp_official_b200 import arch
    from oracle import adm as oa, ddpm as od
    pairs = [(arch.ddpm_arch(**od.CELEBA_CFG), od.ddpm_param_shapes(od.CELEBA_CFG, 2)),
             (arch.ddpm_arch(**od.MINI_CFG), od.ddpm_param_shapes(od.MINI_CFG, 2)),
             (arch.adm_arch(**oa.AFHQ_HP), oa.adm_param_shapes(oa.AFHQ_HP, 2)),
             (arch.adm_arch(**oa.IMAGENET_HP), oa.adm_param_shapes(oa.IMAGENET_HP, 2)),
             (arch.adm_arch(**oa.MINI_HP), oa.adm_param_shapes(oa.MINI_HP, 2))]
    for a, o in pairs:
        mine = {k: tuple(v) for k, v in arch.param_shapes(a, 2).items()}
        assert mine == {k: tuple(v) for k, v in o.items()}


def test_module_state_dict_and_delta_checkpoint_format():
    """same keys as the reference modules; a Δh checkpoint {"0": layer_0.state_dict()} loads with all keys matched
    (diffusion_latent.py:674-676).  Uses the reference's shipped 'smiling' DeltaBlock (tests/golden/checkpoint/: its
    "0" entry, tensor for tensor)."""
    from asyrp_official_b200 import modules, synthetic
    from asyrp_official_b200.configs import load_config
    m = modules.DDPM(load_config("celeba.yml"))
    m.setattr_layers(1)
    keys = set(m.layer_0.state_dict())
    assert keys == {"conv1.weight", "conv1.bias", "temb_proj.weight", "temb_proj.bias", "norm2.weight", "norm2.bias",
                    "conv2.weight", "conv2.bias"}
    v0 = m._version
    ck = os.path.join(ROOT, "tests", "golden", "checkpoint", "smiling_LC_CelebA_HQ_t999_ninv40_ngen40_0.pth")
    sd = torch.load(ck, map_location="cpu", weights_only=True)["0"]
    res = m.layer_0.load_state_dict(sd)
    assert not res.missing_keys and not res.unexpected_keys
    assert torch.equal(m.layer_0.conv1.weight, sd["conv1.weight"])
    assert m._version > v0  # engine weights are re-packed after any load_state_dict
    a = modules.i_DDPM("AFHQ")
    a.setattr_layers(1)
    assert set(a.layer_0.state_dict()) == {"in_layers.0.weight", "in_layers.0.bias", "in_layers.2.weight",
                                           "in_layers.2.bias", "emb_layers.1.weight", "emb_layers.1.bias",
                                           "out_layers.0.weight", "out_layers.0.bias", "out_layers.3.weight",
                                           "out_layers.3.bias"}
    # zero_module() layers of the ADM family start at zero like the reference's (unet.py:252-254,336,657)
    assert a.state_dict()["out.2.weight"].abs().max() == 0 and a.state_dict()["input_blocks.1.0.out_layers.3.weight"].abs().max() == 0
    synthetic.randomize_(a, 7)
    assert a.state_dict()["out.2.weight"].abs().max() > 0
    with pytest.raises(ValueError):
        modules.i_DDPM("LSUN")
    assert modules.guided_Diffusion("MetFACE").arch.mid_ch == 512 and modules.i_DDPM("IMAGENET").arch.mid_ch == 1024


def test_schedule_coefficients_match_oracle_step():
    """Schedule's host-side coefficients reproduce the oracle's denoising_step update bit-for-bit (fp32)"""
    from asyrp_official_b200.schedule import Schedule, make_sequences
    from oracle import sampler as osmp
    betas = osmp.make_betas()
    seq, nxt = make_sequences(999, 40)
    assert (seq, nxt) == osmp.make_sequences(999, 40)
    sch = Schedule(betas, seq, nxt, t_edit=500, t_addnoise=200, hs_coeff=(1.0, 0.5))
    # 8 steps have t < t_addnoise, but the last one (t_next = -1, alpha-bar_next = 1) has a zero noise coefficient
    assert sch.n_edit == 20 and sch.n_stochastic == 7 and len(sch.steps) == 40
    assert sch.steps[0].t == 999 and sch.steps[-1].t_next == -1 and sch.steps[-1].an == 1.0
    g = torch.Generator().manual_seed(0)
    x, e, em, z = (torch.randn(1, 3, 4, 4, generator=g) for _ in range(4))
    for s in (sch.steps[0], sch.steps[25], sch.steps[-1]):
        model = lambda xt, t, **k: (e, em, None, None)  # noqa: E731
        eta = 1.0 if s.c1 != 0.0 else 0.0
        ref, x0, _, _ = osmp.denoising_step(x, torch.ones(1) * s.t, torch.ones(1) * s.t_next, model=model, b=betas,
                                            eta=eta, index=0, t_edit=500, hs_coeff=(1.0, 0.5), noise=z)
        at, an = torch.tensor(s.at), torch.tensor(s.an)
        x0_mine = (x - em * (1 - at).sqrt()) / at.sqrt()
        mine = an.sqrt() * x0_mine + torch.tensor(s.c2) * e
        if s.c1 != 0.0:
            mine = mine + torch.tensor(s.c1) * z
        assert torch.equal(x0, x0_mine) and torch.allclose(ref, mine, rtol=0, atol=1e-6)


def test_config_and_cli_surface(tmp_path, monkeypatch):
    from asyrp_official_b200 import main as cli
    from asyrp_official_b200.configs import load_config
    c = load_config("afhq.yml")
    assert c.data.dataset == "AFHQ" and c.model.ch_mult == [1, 1, 2, 2, 4, 4] and c.diffusion.beta_end == 0.02
    y = tmp_path / "my.yml"
    y.write_text("data:\n  dataset: LSUN\n  category: church_outdoor\n  image_size: 256\n  channels: 3\n"
                 "model:\n  ch: 128\n  var_type: fixedsmall\ndiffusion:\n  beta_start: 0.0001\n  beta_end: 0.02\n"
                 "  num_diffusion_timesteps: 1000\n")
    assert load_config(str(y)).data.category == "church_outdoor"
    with pytest.raises(FileNotFoundError):
        load_config("nope.yml")
    monkeypatch.chdir(tmp_path)
    args, cfg = cli.parse_args_and_config(["--run_test", "--config", "celeba.yml", "--exp", "./runs/smiling",
                                           "--n_train_step", "40", "--user_defined_t_edit", "500"])
    assert args.exp == "./runs/smiling_LC_CelebA_HQ_t999_ninv40_ngen40"  # main.py:235
    assert args.lpips_edit_th == 0.33 and args.n_test_step == 40 and args.bs_train == 1 and args.seed == 1234
    assert os.path.isdir(args.test_image_folder)


def test_runner_host_logic():
    """sequences, hs_coeff scaling (diffusion_latent.py:626,654,659) and LPIPS-table t_edit lookup on the CelebA-HQ
    tables the reference ships (utils/celeba_LPIPS_distance_{x0_t,x}.tsv, stored under tests/golden/lpips/)"""
    from asyrp_official_b200.configs import load_config
    from asyrp_official_b200.diffusion_latent import Asyrp
    a = argparse.Namespace(user_defined_t_edit=None, user_defined_t_addnoise=None, clip_cosine=0.8, config="celeba.yml",
                           lpips_table_dir=os.path.join(ROOT, "tests", "golden", "lpips"), add_noise_from_xt=True)
    r = Asyrp(a, load_config("celeba"), device="cpu")
    assert r.betas.dtype == torch.float32 and r.logvar.shape == (1000,)
    r.set_t_edit_t_addnoise(LPIPS_th=0.33, LPIPS_addnoise_th=1.2)
    assert 400 <= r.t_edit <= 560 and r.t_addnoise == 167  # SURVEY.md Appendix D
    a2 = argparse.Namespace(user_defined_t_edit=500, user_defined_t_addnoise=200)
    r2 = Asyrp(a2, load_config("celeba"), device="cpu")
    r2.set_t_edit_t_addnoise()
    sch = r2.make_schedule(*__import__("asyrp_official_b200.schedule", fromlist=["x"]).make_sequences(999, 40),
                           hs_coeff=(1.0, 1.0))
    assert (r2.t_edit, r2.t_addnoise, sch.n_edit, sch.n_stochastic) == (500, 200, 20, 7)
    with pytest.raises(ValueError):
        Asyrp(argparse.Namespace(user_defined_t_edit=None, user_defined_t_addnoise=None), load_config("celeba"),
              device="cpu").set_t_edit_t_addnoise()


def test_weight_packing_layout():
    """pack_weights is pure tensor reshuffling: check the K layouts the kernels rely on, on the CPU"""
    from asyrp_official_b200 import arch, modules, synthetic
    from asyrp_official_b200.engine import pack_weights
    from oracle import adm as oa, ddpm as od
    for a, make in ((arch.ddpm_arch(**od.MINI_CFG), None), (arch.adm_arch(**oa.MINI_HP), None)):
        shapes = arch.param_shapes(a, 1)
        from oracle import synth
        sd = synth.synth_state_dict(shapes, 1234, "jittered")
        W, emb_off, emb_total = pack_weights(a, sd, "cpu", 1)
        assert emb_total == W["emb_cat.w"].shape[0] == W["emb_cat.b"].shape[0] and emb_total % 64 == 0
        for stage in a.enc + [a.mid] + a.dec:
            for layer in stage:
                if isinstance(layer, arch.Res):
                    p = layer.name
                    assert W[p + ".w1"].shape == (layer.cout, 9 * layer.cin) and W[p + ".w1"].dtype == torch.float16
                    # conv2: 9*cout columns, then the 1x1 shortcut (cin columns) or the identity skip (cout columns)
                    assert W[p + ".w2"].shape == (layer.cout, 9 * layer.cout + layer.cin)
                    if layer.cin == layer.cout:
                        assert torch.equal(W[p + ".w2"][:, 9 * layer.cout:].float(), torch.eye(layer.cout))
                    if layer.split:  # decoder: segment-major K (h columns of every tap, then skip columns of every tap)
                        c0 = layer.split[0]
                        key = p + (".conv1.weight" if a.family == "ddpm" else ".in_layers.2.weight")
                        w = sd[key]
                        assert torch.equal(W[p + ".w1"][:, :9 * c0].float().reshape(layer.cout, 3, 3, c0),
                                           w[:, :c0].permute(0, 2, 3, 1).to(torch.float16).float())
        assert W["conv_in.w"].shape[1] == 9 * 64 and W["conv_out.w"].shape[0] == 16


def test_upconv_subpixel_weights():
    """pack_upconv_weight: conv3x3(nearest-x2(x)) == four 2x2 phase convs on x (reference: Upsample.forward,
    models/ddpm/diffusion.py:77-87).  Checked in fp64 with the packed layout the kernel consumes."""
    import torch.nn.functional as F
    from asyrp_official_b200 import ops
    torch.manual_seed(0)
    n, ci, co, h, w = 2, 5, 3, 6, 4
    x = torch.randn(n, ci, h, w, dtype=torch.float64)
    wt = torch.randn(co, ci, 3, 3, dtype=torch.float64)
    ref = F.conv2d(F.interpolate(x, scale_factor=2.0, mode="nearest"), wt, padding=1)
    # packed rows: (a*2+b)*co + o ; columns: (dy*2+dx)*ci + i ; source pixel (y-1+a+dy, x-1+b+dx)
    # (computed in fp32 by the packer; compare against an fp64 re-evaluation with a matching tolerance)
    pk = ops.pack_upconv_weight(wt.float()).double().reshape(2, 2, co, 2, 2, ci)
    xp = F.pad(x, (1, 1, 1, 1))
    out = torch.zeros(n, co, 2 * h, 2 * w, dtype=torch.float64)
    for a in (0, 1):
        for b in (0, 1):
            acc = torch.zeros(n, co, h, w, dtype=torch.float64)
            for dy in (0, 1):
                for dx in (0, 1):
                    patch = xp[:, :, a + dy:a + dy + h, b + dx:b + dx + w]
                    acc += torch.einsum("oi,nihw->nohw", pk[a, b, :, dy, dx, :], patch)
            out[:, :, a::2, b::2] = acc
    assert (out - ref).abs().max() < 2e-2 * ref.abs().max()  # fp16 rounding of the packed weights
    pk32 = ops.pack_upconv_weight(wt.float())
    assert pk32.shape == (4 * co, 4 * ci) and pk32.dtype == torch.float16


@pytest.mark.parametrize("mode", ["ddpm", "dt_lambda", "ignore"])
def test_schedule_sample_type_dt_lambda_and_key(mode):
    """Schedule carries what save_image forwards to denoising_step on every step (diffusion_latent.py:507-520):
    'ddpm' ancestral coefficients, the dt_lambda override at t >= 999, ignore_timestep; the coefficients reproduce the
    oracle's step; hs_coeff VALUES are not part of the graph key (they are device-side parameters)"""
    from asyrp_official_b200.schedule import Schedule, make_sequences
    from oracle import sampler as osmp
    betas = osmp.make_betas()
    logvar = osmp.make_logvar(osmp.get_beta_schedule(beta_start=1e-4, beta_end=0.02, num_diffusion_timesteps=1000))
    seq, nxt = make_sequences(999, 10)
    base = Schedule(betas, seq, nxt, t_edit=500, t_addnoise=0, hs_coeff=(1.0, 1.0))
    assert base.key() == Schedule(betas, seq, nxt, t_edit=500, t_addnoise=0, hs_coeff=(0.3, 2.0)).key()
    g = torch.Generator().manual_seed(0)
    x, e, z = (torch.randn(1, 3, 4, 4, generator=g) for _ in range(3))
    model = lambda xt, t, **k: (e, e, None, None)  # noqa: E731
    if mode == "ignore":
        s2 = Schedule(betas, seq, nxt, t_edit=500, t_addnoise=0, hs_coeff=(1.0, 1.0), ignore_timestep=True)
        assert s2.key() != base.key() and s2.ignore_timestep
        return
    if mode == "ddpm":
        sch = Schedule(betas, seq, nxt, t_edit=500, t_addnoise=0, hs_coeff=(1.0, 1.0), sample_type="ddpm", logvars=logvar)
        assert sch.n_stochastic == 10 and sch.key() != base.key() and sch.steps[-1].mask == 0.0
        for s in (sch.steps[0], sch.steps[-1]):
            ref = osmp.denoising_step(x, torch.ones(1) * s.t, torch.ones(1) * s.t_next, model=model, b=betas,
                                      logvars=logvar, sampling_type="ddpm", noise=z)[0]
            at, bt = torch.tensor(s.at), torch.tensor(s.bt)
            mine = 1 / torch.sqrt(1.0 - bt) * (x - bt / torch.sqrt(1 - at) * e) + s.mask * torch.exp(
                torch.tensor(0.5 * s.logvar)) * z
            assert torch.allclose(ref, mine, rtol=0, atol=1e-6)
        with pytest.raises(ValueError):
            Schedule(betas, seq, nxt, t_edit=500, sample_type="ddpm", dt_lambda=0.5, logvars=logvar)
        return
    sch = Schedule(betas, seq, nxt, t_edit=500, t_addnoise=0, hs_coeff=(1.0, 1.0), dt_lambda=0.7)
    assert sch.key() != base.key() and sch.steps[1] == base.steps[1]  # only t >= dt_end = 999 is affected
    s = sch.steps[0]
    ref = osmp.denoising_step(x, torch.ones(1) * s.t, torch.ones(1) * s.t_next, model=model, b=betas, dt_lambda=0.7)[0]
    at, an = torch.tensor(s.at), torch.tensor(s.an)
    mine = an.sqrt() * ((x - e * (1 - at).sqrt()) / at.sqrt()) + torch.tensor(s.c2) * e
    assert torch.allclose(ref, mine, rtol=0, atol=1e-6) and s.c1 == 0.0


def test_reference_staging_script(tmp_path, monkeypatch):
    """oracle/stage_reference.py copies the reference's hot-path sources verbatim into a git-ignored directory, on a
    stand-in checkout with the reference's layout; the checkout is $ASYRP_REFERENCE_DIR, else the default location"""
    from oracle import stage_reference as mod
    assert "oracle/_ref/" in open(os.path.join(ROOT, ".gitignore")).read()
    assert mod.DST == os.path.join(ROOT, "oracle", "_ref")
    monkeypatch.delenv("ASYRP_REFERENCE_DIR", raising=False)
    monkeypatch.setattr(mod, "REFERENCE", str(tmp_path / "missing"))
    assert mod.stage(None, str(tmp_path / "x"), quiet=True) is False
    assert mod.stage(str(tmp_path / "missing"), str(tmp_path / "x"), quiet=True) is False
    assert not (tmp_path / "x").exists()
    src = tmp_path / "src"
    files = {rel: f"{rel}\n".encode() * 3 for rel in (
        "utils/diffusion_utils.py", "models/ddpm/diffusion.py", "models/improved_ddpm/unet.py",
        "models/guided_diffusion/unet.py", "configs/celeba.yml", *(f"checkpoint/{c}" for c in mod.CKPTS))}
    skipped = ("utils/celeba_LPIPS_distance_x.tsv", "models/__pycache__/m.cpython-312.pyc", "checkpoint/other_0.pth",
               "main.py")
    for rel in (*files, *skipped):
        (src / rel).parent.mkdir(parents=True, exist_ok=True)
        (src / rel).write_bytes(files.get(rel, b"x"))
    for how in ("default", "env"):
        dst = tmp_path / f"ref_{how}"
        (dst / "models").mkdir(parents=True)
        (dst / "models" / "stale.py").write_text("")  # an earlier staging's leftovers are replaced
        if how == "default":
            monkeypatch.setattr(mod, "REFERENCE", str(src))
        else:
            monkeypatch.setattr(mod, "REFERENCE", str(tmp_path / "missing"))
            monkeypatch.setenv("ASYRP_REFERENCE_DIR", str(src))
        assert mod.stage(dst=str(dst), quiet=True)
        staged = {os.path.relpath(os.path.join(d, f), dst) for d, _, fs in os.walk(dst) for f in fs}
        assert staged == set(files)
        for rel, data in files.items():
            assert (dst / rel).read_bytes() == data, rel


def test_engine_numerics_emulation_switches():
    """oracle/emulate.py with every rounding switched off is the fp32 oracle; switched on it differs at the fp16 level"""
    from oracle import ddpm as od, emulate as em, synth
    cfg = od.MINI_CFG
    sd = synth.synth_state_dict(od.ddpm_param_shapes(cfg, 1), 1234, "jittered")
    x, t = synth.synth_noise((1, 3, 32, 32), 1234), torch.ones(1) * 700
    ref = od.ddpm_forward(sd, cfg, x, t, index=0, t_edit=500, hs_coeff=(1.0, 0.7))
    off = em.ddpm_forward(sd, cfg, x, t, index=0, t_edit=500, hs_coeff=(1.0, 0.7), flags=em.NONE)
    on = em.ddpm_forward(sd, cfg, x, t, index=0, t_edit=500, hs_coeff=(1.0, 0.7), flags=em.ALL)
    for a, b, c in zip(ref, off, on):
        scale = a.abs().max().item()
        assert (a - b).abs().max().item() <= 2e-5 * scale
        assert 1e-5 * scale < (a - c).abs().max().item() < 1e-2 * scale


def test_shipped_delta_block_fixtures_load():
    """tests/golden/checkpoint/*.pth: the DeltaBlocks SURVEY §8(d) names, in the {"0": state_dict} format run_test loads"""
    from asyrp_official_b200 import modules
    from asyrp_official_b200.configs import load_config
    d = os.path.join(ROOT, "tests", "golden", "checkpoint")
    m = modules.DDPM(load_config("celeba"))
    m.setattr_layers(1)
    for name in ("smiling_LC_CelebA_HQ_t999_ninv40_ngen40_0.pth", "church_gothic_LC_church_outdoor_t999_ninv40_ngen40_0.pth"):
        ck = torch.load(os.path.join(d, name), map_location="cpu", weights_only=True)
        res = m.layer_0.load_state_dict(ck["0"])
        assert not res.missing_keys and not res.unexpected_keys
    a = modules.i_DDPM("AFHQ")
    a.setattr_layers(1)
    ck = torch.load(os.path.join(d, "dog_happy_LC_dog_t999_ninv40_ngen40_0.pth"), map_location="cpu", weights_only=True)
    res = a.layer_0.load_state_dict(ck["0"])
    assert not res.missing_keys and not res.unexpected_keys
