"""Every kernel launch of the four benchmark plans, replayed in isolation against a float64 reference.

The whole-UNet tests (test_model_gpu.py) compare ~100-layer networks within 4e-3 of max|ref|, and the kernel tests
(test_kernels_gpu.py) use hand-picked shapes.  A wrong tile class, a bad batch tail or a stale statistics slot in one
layer can hide inside the first and be missed by the second.  This file closes that gap:

  1. For each bench workload (ddpm_celeba_b16, ddpm_church_b32, iddpm_afhq_b8, adm_imagenet_b4) the UNet is built with
     synthetic weights and one DeltaBlock at the bench's per-GPU batch, and every launch the plan makes is recorded
     (metadata only: shapes, strides, storage offsets, dtypes, scalars, GNSpec fields, the tile class) during one edit
     forward and one explicit-delta_h forward, once with the affine-table GroupNorm and once with ASYRP_GN_FOLD.
  2. Each unique launch is replayed on fresh random operands laid out with the recorded strides and offsets, and
     compared with a float64 evaluation of the C-ABI semantics documented in include/asyrp_b200.h (the ref_* helpers
     below; the unmarked tests at the bottom pin them against composed torch.nn.functional ops on the CPU).
  3. Every conv is rebuilt at N = 1 on its first and last sample; output and statistics must be bit-identical to the
     batched run (a sample's result may not depend on its batch neighbours: multi-GPU sharding relies on it).
  4. The sampler updates run at each workload's shape, out of place and with x_next aliasing x.

Bounds (max-abs error over max|ref|, the figures test_kernels_gpu.py states for the same kernels):
  conv, raw fp16 operand 1.5e-3; affine-table operand (+SiLU) 2.5e-3; in-kernel GroupNorm or transformed up2 3e-3;
  fp32 logits and raw planar output 2e-5; GroupNorm statistics 2e-3*max + 1e-3 (3e-3 for up2).  The up2 reference
  uses the packed sub-pixel weights themselves, so a raw up2 conv gets the raw-operand bound.
"""
import inspect
import math
import time
from collections import namedtuple
from types import SimpleNamespace as NS

import pytest
import torch
import torch.nn.functional as F

from asyrp_official_b200 import ops
from asyrp_official_b200.ops import MODE_1x1, MODE_3x3, MODE_3x3_S2, STAT_SCALE, GNSpec

WORKLOADS = {  # bench.py WORKLOADS: family, per-GPU batch (church has CelebA's architecture)
    "ddpm_celeba_b16": ("ddpm", "celeba", 16),
    "ddpm_church_b32": ("ddpm", "church", 32),
    "iddpm_afhq_b8": ("adm", "afhq", 8),
    "adm_imagenet_b4": ("adm", "imagenet", 4),
}
TOL_RAW, TOL_TABLE, TOL_GN, TOL_F32 = 1.5e-3, 2.5e-3, 3e-3, 2e-5


def h16(x):
    """fp16 rounding, kept in x's dtype"""
    return x.to(torch.float16).to(x.dtype)


def silu(x):
    return x * torch.sigmoid(x)


def _at(t, shape, stride, extra):
    """view of t's storage at t's offset + extra elements"""
    return t.as_strided(shape, stride, t.storage_offset() + extra)


# ============================================================================ float64 references of the C ABI
def conv_geometry(segs, out=None, out_shape=None, out_heads=1, up2=False, **_):
    """(N, H, W, Cout) of the descriptor, as ConvOp derives it (up2: the source image)"""
    if out is not None:
        N, H, W, Cout = out.shape
        if out_heads > 1:
            N, Cout = N * out_heads, Cout // out_heads
    else:
        N, H, W, Cout = out_shape
    if up2:
        H, W = H // 2, W // 2
    return N, H, W, Cout


def gn_affine_from_sums(spec, e, off, C):
    """(a, b) of channels [off, off + C) of the concatenated GroupNorm input for batch entry e, from the int64
    (sum, sum of squares) * 2^18 accumulators: GroupNorm(32, eps) [* (1 + scale) + shift]"""
    Ct = sum(spec.C)
    cpg = Ct // 32
    pairs = torch.cat([s[e].double() for s in spec.sums], 0) / STAT_SCALE  # [Ct/2][2]
    g = pairs.reshape(32, cpg // 2, 2).sum(1)
    cnt = float(spec.hw * cpg)
    mean = g[:, 0] / cnt
    rstd = 1.0 / torch.sqrt((g[:, 1] / cnt - mean * mean).clamp_min(0.0) + spec.eps)
    ch = torch.arange(off, off + C, device=pairs.device)
    grp = ch // cpg
    a = spec.gamma.double()[ch] * rstd[grp]
    b = spec.beta.double()[ch] - mean[grp] * a
    if spec.ss is not None:
        row = _at(spec.ss, (2 * Ct,), (1,), e * spec.ss_stride).double()
        sc = 1.0 + row[ch]
        a, b = a * sc, b * sc + row[Ct + ch]
    return a, b


def _taps(x, mode, H, W, phase=None):
    """tap-ordered [H][W][C] operand views of the transformed source x (zero padding applied after the transform)"""
    if mode == MODE_1x1:
        return [x]
    if mode == MODE_3x3_S2:  # source [2H][2W][C], pad right / bottom by 1, stride 2
        xp = F.pad(x, (0, 0, 0, 1, 0, 1))
        return [xp[ky:ky + 2 * H:2, kx:kx + 2 * W:2] for ky in range(3) for kx in range(3)]
    xp = F.pad(x, (0, 0, 1, 1, 1, 1))
    if phase is None:
        return [xp[ky:ky + H, kx:kx + W] for ky in range(3) for kx in range(3)]
    a, b = phase  # sub-pixel phase (2i+a, 2j+b): 2x2 taps on source pixels (i-1+a+dy, j-1+b+dx)
    return [xp[a + dy:a + dy + H, b + dx:b + dx + W] for dy in range(2) for dx in range(2)]


def ref_conv(segs, weight, out=None, ebias=None, ebias_stride=0, residual=None, res_scale=1.0, acc_scale=1.0,
             stats=None, out_planar=None, out_shape=None, weight_batched=False, a_heads=1, b_heads=1, out_heads=1,
             up2=False, scales=None, res_mode=0, sums_out=None, entries=None):
    """asyrp_conv_create + asyrp_conv_launch in float64, with ConvOp's arguments.  Returns the pre-rounding output
    [E][Ho][Wo][Cout] and the per-(entry, channel pair) (sum, sum of squares) [E][Cout/2][2] of the batch entries
    `entries` (default: all).  An entry is a (sample, head) pair when heads > 1."""
    segs = [tuple(sg) + (None, 0, 0) * (len(sg) == 2) for sg in segs]
    N, H, W, Cout = conv_geometry(segs, out, out_shape, out_heads, up2)
    entries = range(N) if entries is None else entries
    if scales is not None:
        acc_scale, res_scale = float(scales[0]), float(scales[1])
    ktot = sum((1 if m == MODE_1x1 else (4 if up2 else 9)) * s.shape[-1] for s, m, *_ in segs)
    rows = Cout * (4 if up2 else 1)
    outs = []
    for e in entries:
        xs = []
        for i, (src, mode, aff, off, act) in enumerate(segs):
            C = src.shape[-1]
            hs, ws = (2 * H, 2 * W) if mode == MODE_3x3_S2 else (H, W)
            if i == 0 and a_heads > 1:  # [N/heads][H][W][ld], head h reads channels [h*C, (h+1)*C)
                x = _at(src, (hs, ws, C), (src.stride(1), src.stride(2), 1),
                        (e // a_heads) * src.stride(0) + (e % a_heads) * C)
            else:
                x = src[e]
            x = x.double()
            if aff is not None:
                if isinstance(aff, GNSpec):
                    a, b = gn_affine_from_sums(aff, e, off, C)
                else:
                    ab = _at(aff, (C, 2), (2, 1), e * aff.shape[1] * 2 + off * 2).double()
                    a, b = ab[:, 0], ab[:, 1]
                x = x * a + b
                if act:
                    x = silu(x)
                x = h16(x)  # the transformed operand is rounded to fp16 before the MMA
            xs.append((x, mode))
        if weight_batched and b_heads > 1:  # [N/heads][Cout][ld], head h reads columns [h*K, (h+1)*K)
            w = _at(weight, (rows, ktot), (weight.stride(-2), 1), (e // b_heads) * weight.stride(0) + (e % b_heads) * ktot)
        elif weight_batched:
            w = weight[e][:, :ktot]
        else:
            w = weight[:, :ktot]
        w = w.double()

        def gemm(phase, wrows):
            acc, k = None, 0
            for x, mode in xs:
                C = x.shape[-1]
                for tap in _taps(x, mode, H, W, phase):
                    t = tap.reshape(-1, C) @ wrows[:, k:k + C].t()
                    acc = t if acc is None else acc + t
                    k += C
            return acc.reshape(H, W, -1)

        if up2:
            v = torch.empty(2 * H, 2 * W, Cout, dtype=torch.float64, device=w.device)
            for a_ in (0, 1):
                for b_ in (0, 1):
                    ph = a_ * 2 + b_
                    v[a_::2, b_::2] = gemm((a_, b_), w[ph * Cout:(ph + 1) * Cout])
        else:
            v = gemm(None, w)
        if ebias is not None:
            v = v + _at(ebias, (Cout,), (1,), e * ebias_stride).double()
        v = v * acc_scale
        if residual is not None:
            r = residual[e].double()
            if res_mode == 1:
                r = r.repeat_interleave(2, 0).repeat_interleave(2, 1)
            elif res_mode == 2:
                r = r.reshape(H, 2, W, 2, Cout).mean(dim=(1, 3))
            v = v + res_scale * r
        outs.append(v)
    v = torch.stack(outs)
    pr = v.reshape(v.shape[0], -1, Cout // 2, 2)
    st = torch.stack([pr.sum(dim=(1, 3)), (pr * pr).sum(dim=(1, 3))], -1)
    return v, st


def ref_gn_finalize(stats_a, Ca, stats_b, Cb, gamma, beta, eps, N, HW, scale_shift=None, ss_stride=0):
    """affine [N][C][2] of asyrp_gn_finalize in float64, and the magnitude of the terms each entry is made of"""
    pairs = stats_a.double().sum(1)
    if stats_b is not None and Cb:
        pairs = torch.cat([pairs, stats_b.double().sum(1)], 1)
    C = Ca + Cb
    cpg = C // 32
    g = pairs.reshape(N, 32, cpg // 2, 2).sum(2)
    cnt = float(HW * cpg)
    mean = g[..., 0] / cnt
    rstd = 1.0 / torch.sqrt((g[..., 1] / cnt - mean * mean).clamp_min(0.0) + eps)
    mean_c, rstd_c = mean.repeat_interleave(cpg, 1), rstd.repeat_interleave(cpg, 1)
    a = gamma.double()[None] * rstd_c
    b = beta.double()[None] - mean_c * a
    mag_b = beta.double().abs()[None] + (mean_c * a).abs()
    if scale_shift is not None:
        ss = _at(scale_shift, (N, 2 * C), (ss_stride, 1), 0).double()
        sc = 1.0 + ss[:, :C]
        a, b = a * sc, b * sc + ss[:, C:]
        mag_b = mag_b * sc.abs() + ss[:, C:].abs()
    return torch.stack([a, b], -1), torch.stack([a.abs(), mag_b], -1)


def ref_apply(src_a, src_b, affine, act, resample, affine_offset=0):
    """asyrp_apply in float64: resample(act(a*x + b)) over the channel concat, NHWC"""
    x = src_a.double() if src_b is None else torch.cat([src_a.double(), src_b.double()], -1)
    N, Hi, Wi, C = x.shape
    if affine is not None:
        ab = _at(affine, (N, C, 2), (affine.shape[1] * 2, 2, 1), affine_offset * 2).double()
        x = x * ab[:, None, None, :, 0] + ab[:, None, None, :, 1]
    if act:
        x = silu(x)
    if resample == 1:
        x = x.reshape(N, Hi // 2, 2, Wi // 2, 2, C).mean(dim=(2, 4))
    elif resample == 2:
        x = x.repeat_interleave(2, 1).repeat_interleave(2, 2)
    return x


def ref_linear(inp, weight, bias, O, act_in=False, act_out=False):
    """asyrp_linear in float64, and the Higham bound (I + 8) u sum|w f(x)| of an fp32 evaluation"""
    x = inp.double()
    if act_in:
        x = silu(x)
    w = weight.double()[:O]
    y = x @ w.t()
    mag = x.abs() @ w.abs().t()
    if bias is not None:
        y = y + bias.double()[:O]
        mag = mag + bias.double()[:O].abs()
    bound = (inp.shape[1] + 8) * 2.0 ** -24 * mag
    if act_out:
        y = silu(y)
        bound = 1.1 * bound
    return y, bound + 1e-7


def ref_slerp_h(h, dh, t, use_mask):
    """asyrp_slerp_h in float64: h [N][H][W][C], dh [N][C][H][W] -> h2 [N][H][W][C] (pre-rounding)"""
    N, H, W, C = h.shape
    a = h.double().permute(0, 3, 1, 2)
    d = dh.double().expand(N, C, H, W)
    m = torch.ones(H, W, dtype=torch.float64, device=h.device)
    if use_mask:
        m = torch.zeros_like(m)
        m[4:H - 1, 3:5] = 1.0
    am, dm = a * m, d * m
    nh, nd = am.flatten(1).norm(dim=1), dm.flatten(1).norm(dim=1)
    th = torch.acos((am * dm).flatten(1).sum(1) / (nh * nd))
    s0, s1 = torch.sin(th - th * t) / torch.sin(th), torch.sin(th * t) / torch.sin(th)
    scale = torch.ones_like(nh) if use_mask else nh / nd
    v = s0[:, None, None, None] * a + (s1 * scale)[:, None, None, None] * d
    v = torch.where(m.bool(), v, a)
    return v.permute(0, 2, 3, 1)


def ref_timestep_embedding(t, dim, variant):
    half = dim // 2
    i = torch.arange(half, dtype=torch.float32, device=t.device)
    fr = torch.exp(i * -(math.log(10000) / (half - 1))) if variant == 0 else torch.exp(-math.log(10000) * i / half)
    e = t.double()[:, None] * fr.double()[None]
    return torch.cat([torch.sin(e), torch.cos(e)] if variant == 0 else [torch.cos(e), torch.sin(e)], 1)


def pair_stats(v):
    """[E][..][C] -> per channel pair (sum, sum of squares) [E][C/2][2]"""
    pr = v.reshape(v.shape[0], -1, v.shape[-1] // 2, 2)
    return torch.stack([pr.sum(dim=(1, 3)), (pr * pr).sum(dim=(1, 3))], -1)


# ============================================================================ recording the plans
Meta = namedtuple("Meta", "shape stride offset dtype")
SpecMeta = namedtuple("SpecMeta", "sid sums C eps hw ss ss_stride")


def _meta(t):
    return Meta(tuple(t.shape), tuple(t.stride()), t.storage_offset(), t.dtype)


def _key(v):
    """dedup key: storage offsets only by their alignment class (they differ from layer to layer, e.g. the
    emb_all column slice each ResBlock reads, without changing what the kernel does)"""
    if isinstance(v, Meta):
        return Meta(v.shape, v.stride, v.offset % 128, v.dtype)
    if isinstance(v, (tuple, list)):  # SpecMeta and the table tuples included
        return tuple(_key(x) for x in v)
    return v


def _tile_shape(H, W, halo):
    """mirror of conv_tile_shape (csrc/conv_gemm.cu): (TW, TH, NB)"""
    if halo:
        return 8, 16, 1
    if H == 1:
        tw, th = min(W, 128), 1
    else:
        tw = min(W, 16)
        th = min(128 // tw, 8, H)
    while 128 % (tw * th):
        th -= 1
    return tw, th, 128 // (tw * th)


def _tile_config(H, W, Cout, halo, phases):
    """mirror of conv_config (csrc/conv_gemm.cu): (BN, MT); checked against asyrp_conv_tile_config below"""
    tw, th, nb = _tile_shape(H, W, halo)
    if Cout == 16:
        return 16, (2 if nb == 1 and H > 1 and H % (2 * th) == 0 and W % tw == 0 else 1)
    tiles_x, tiles_n = -(-W // tw), -(-16 // nb)
    best, best_tiles = None, -1
    for bn, mt in ((256, 1), (128, 2), (128, 1), (64, 2), (64, 1)):
        if Cout % bn or (mt == 2 and not (nb == 1 and H > 1 and H % (2 * th) == 0 and W % tw == 0)):
            continue
        tiles = tiles_x * -(-H // (th * mt)) * tiles_n * (Cout // bn) * phases
        if tiles >= 120:
            return bn, mt
        if tiles > best_tiles:
            best, best_tiles = (bn, mt), tiles
    return best


class Recorder:
    def __init__(self):
        self.convs, self.calls = [], []

    def conv(self, op, segs, weight, kw):
        segs = [tuple(sg) + (None, 0, 0) * (len(sg) == 2) for sg in segs]
        specs, tables = {}, {}
        sm = []
        for src, mode, aff, off, act in segs:
            if isinstance(aff, GNSpec):
                sid = specs.setdefault(id(aff), len(specs))
                am = SpecMeta(sid, tuple(_meta(s) for s in aff.sums), tuple(aff.C), aff.eps, aff.hw,
                              _meta(aff.ss) if aff.ss is not None else None, aff.ss_stride)
            elif aff is not None:
                am = ("table", tables.setdefault(id(aff), len(tables)), _meta(aff))
            else:
                am = None
            sm.append((_meta(src), mode, am, off, act))
        km = {k: (_meta(v) if torch.is_tensor(v) else v) for k, v in kw.items()}
        N, H, W, Cout = conv_geometry(segs, **kw)
        has3 = any(sg[1] == MODE_3x3 for sg in segs)
        halo = has3 and H % 16 == 0 and W % 8 == 0
        up2 = bool(kw.get("up2", False))
        bn, mt = _tile_config(H, W, Cout, halo, 4 if up2 else 1)
        lib_cfg = ops.conv_tile_config(H, W, Cout, has3)
        if not up2:  # the mirror must agree with the library
            assert (bn, mt) == lib_cfg[:2], ((N, H, W, Cout, has3), (bn, mt), lib_cfg)
        kinds = ["gn" if isinstance(a[2], SpecMeta) else ("table" if a[2] else "raw") for a in sm]
        variant = "pair" if op.cta2 else ("swap" if (bn, mt) == (128, 2) else "one")
        cls = (bn, mt, variant, halo, up2, "+".join(sorted(set(kinds))), len(segs))
        rec = dict(segs=sm, weight=_meta(weight), kw=km, N=N, H=H, W=W, Cout=Cout, cta2=op.cta2, tile_config=lib_cfg,
                   nb=_tile_shape(H, W, halo)[2], cls=cls, desc=None)
        rec["sig"] = _key((rec["segs"], rec["weight"], tuple(sorted(km.items())), op.cta2))
        op._asyrp_rec = rec
        self.convs.append(rec)

    def call(self, name, fn, args, kwargs):
        b = inspect.signature(fn).bind(*args, **kwargs)
        b.apply_defaults()
        a = {k: (_meta(v) if torch.is_tensor(v) else v) for k, v in b.arguments.items()}
        self.calls.append(dict(name=name, args=a, sig=_key((name, tuple(sorted(a.items()))))))


WRAPPED = ["gn_finalize", "apply", "linear", "timestep_embedding", "pack_input", "unpack_nchw", "slerp_h", "attention",
           "softmax_rows", "transpose_tc"]


def _record_plans(mp, rec, model, N, fold):
    """build the plan for batch N with engine.GN_FOLD = fold and run the edit and explicit-delta_h forwards"""
    from asyrp_official_b200 import engine
    mp.setattr(engine, "GN_FOLD", fold)
    eng = model.engine
    eng.plans.clear()
    eng.graphs.clear()
    dev = eng.device
    g = torch.Generator().manual_seed(7)
    S = eng.arch.image_size
    x = torch.randn(N, 3, S, S, generator=g).to(dev)
    t = torch.full((N,), 800.0, device=dev)
    model(x, t, index=0, t_edit=500, hs_coeff=(1.0, 0.8))
    P = eng.plans[N]
    dh = torch.randn(*P.dh_user.shape[1:], generator=g).to(dev)
    model(x, t, index=0, t_edit=500, hs_coeff=(0.7, 1.0), delta_h=dh)
    torch.cuda.synchronize()
    for L in P.temb_ops + P.enc_ops + P.delta_ops + P.slerp_ops + P.dec_mod_ops + P.dec_ops:
        op = getattr(L.fn, "__self__", None)
        if op is not None and getattr(op, "_asyrp_rec", None) is not None:
            op._asyrp_rec["desc"] = L.desc
    eng.plans.clear()
    eng.graphs.clear()


def _build_model(family, key, dev):
    from asyrp_official_b200 import modules, synthetic
    from oracle import adm as oa, ddpm as od
    if family == "ddpm":
        cfg = od.CELEBA_CFG
        ns = NS(model=NS(**{**cfg, "dropout": 0.0, "resamp_with_conv": True}), data=NS(image_size=cfg["image_size"]))
        m = modules.DDPM(ns)
    else:
        m = modules._create_adm({"afhq": oa.AFHQ_HP, "imagenet": oa.IMAGENET_HP}[key])
    m.setattr_layers(1)
    return synthetic.randomize_(m, 1234, "torch_default").to(dev)


def record_workload(name, dev):
    """{fold: (conv records, other-launch records)} of one bench workload, all launches (not yet deduplicated)"""
    family, key, N = WORKLOADS[name]
    model = _build_model(family, key, dev)
    out = {}
    base_conv = ops.ConvOp
    for fold in (False, True):
        rec = Recorder()

        class RecordingConvOp(base_conv):
            def __init__(self, segs, weight, **kw):
                super().__init__(segs, weight, **kw)
                rec.conv(self, segs, weight, kw)

        with pytest.MonkeyPatch.context() as mp:
            mp.setattr(ops, "ConvOp", RecordingConvOp)
            for fn_name in WRAPPED:
                orig = getattr(ops, fn_name)

                def wrapper(*a, _n=fn_name, _f=orig, **k):
                    rec.call(_n, _f, a, k)
                    return _f(*a, **k)

                mp.setattr(ops, fn_name, wrapper)
            _record_plans(mp, rec, model, N, fold)
        out[fold] = (rec.convs, rec.calls)
    del model
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return out


def dedup(recs):
    seen = {}
    for r in recs:
        seen.setdefault(r["sig"], r)
    return list(seen.values())


# ============================================================================ replay
class Fresh:
    """fresh random tensors laid out like the recorded ones (as_strided on a new base tensor)"""

    def __init__(self, dev, seed):
        self.dev = dev
        self.g = torch.Generator(device=dev).manual_seed(seed)

    def base(self, m, fill):
        n = m.offset + 1 + sum((s - 1) * st for s, st in zip(m.shape, m.stride))
        n += m.stride[-2] if len(m.stride) > 1 else 0  # heads read past the view's last row (channel slices of qkv)
        if fill == "nan":
            b = torch.full((n,), float("nan"), dtype=m.dtype, device=self.dev)
        elif fill == "zero":
            b = torch.zeros(n, dtype=m.dtype, device=self.dev)
        else:
            scale, shift = fill
            b = (torch.randn(n, generator=self.g, device=self.dev) * scale + shift).to(m.dtype)
        return b.as_strided(m.shape, m.stride, m.offset)

    def randn(self, shape, scale=1.0, shift=0.0, dtype=torch.float32):
        return (torch.randn(shape, generator=self.g, device=self.dev) * scale + shift).to(dtype)


def _sums_of(x):
    """int64 (sum, sum of squares) * 2^18 per (sample, channel pair) of an NHWC tensor"""
    v = x.double()
    return torch.round(pair_stats(v) * STAT_SCALE).to(torch.int64)


class ConvReplay:
    """the fresh operands of one recorded conv and the ConvOp arguments built from them (all samples, or one)"""

    def __init__(self, r, fr):
        self.r = r
        kw = r["kw"]
        transformed = [sg[2] is not None for sg in r["segs"]]
        self.srcs = [fr.base(sg[0], (1.5, 0.3) if tr else (1.0, 0.0)) for sg, tr in zip(r["segs"], transformed)]
        self.tables, self.specs = {}, {}
        for sg, src in zip(r["segs"], self.srcs):
            am = sg[2]
            if isinstance(am, SpecMeta) and am.sid not in self.specs:
                Ct = sum(am.C)
                sums = [fr.base(m, "zero") for m in am.sums]
                ss = fr.base(am.ss, (0.3, 0.0)) if am.ss is not None else None
                self.specs[am.sid] = dict(sums=sums, C=list(am.C), gamma=fr.randn((Ct,), 0.3, 1.0),
                                          beta=fr.randn((Ct,), 0.3), eps=am.eps, hw=am.hw, ss=ss, ss_stride=am.ss_stride)
            elif am is not None and not isinstance(am, SpecMeta) and am[1] not in self.tables:
                t = fr.base(am[2], (0.5, 0.0))
                t[..., 0] += 1.0
                self.tables[am[1]] = t
        # GroupNorm sums of the replayed sources: channels [off, off + C) of the concat are this segment's source
        for sg, src in zip(r["segs"], self.srcs):
            am = sg[2]
            if isinstance(am, SpecMeta):
                sp = self.specs[am.sid]
                k = 0 if sg[3] < am.C[0] else 1
                assert sg[3] == (0 if k == 0 else am.C[0]) and src.shape[-1] == am.C[k], "GNSpec source mismatch"
                sp["sums"][k].copy_(_sums_of(src))
        for sp in self.specs.values():  # a GroupNorm source that is no segment of this conv: synthetic statistics
            for k, s in enumerate(sp["sums"]):
                if not s.any():
                    hw = sp["hw"]
                    m_, v_ = fr.randn(s.shape[:2], 0.5).double(), fr.randn(s.shape[:2], 0.3, 1.0).double().abs()
                    s.copy_(torch.round(torch.stack([2 * hw * m_, 2 * hw * (m_ * m_ + v_)], -1) * STAT_SCALE).long())
        up2 = bool(kw.get("up2", False))
        if up2:  # 3x3 weights through the sub-pixel packing the engine uses
            C = self.srcs[0].shape[-1]
            w3 = fr.randn((r["Cout"], C, 3, 3), 1.0 / math.sqrt(9 * C))
            self.weight = fr.base(r["weight"], "zero")
            self.weight.copy_(ops.pack_upconv_weight(w3))
        else:
            self.weight = fr.base(r["weight"], (1.0 / math.sqrt(r["weight"].shape[-1]), 0.0))
        self.kw = {}
        for k, v in kw.items():
            if not isinstance(v, Meta):
                self.kw[k] = v
            elif k in ("out", "out_planar", "stats"):
                self.kw[k] = fr.base(v, "nan")
            elif k == "sums_out":
                self.kw[k] = fr.base(v, "zero")
            elif k == "scales":
                s = fr.base(v, "zero")
                s[0], s[1] = 0.7, 1.25
                self.kw[k] = s
            elif k == "ebias":
                self.kw[k] = fr.base(v, (1.0, 0.0))
            else:  # residual
                self.kw[k] = fr.base(v, (1.0, 0.0))
        heads = max(kw.get("a_heads", 1), kw.get("b_heads", 1), kw.get("out_heads", 1))
        self.samples = r["N"] // heads

    def args(self, n=None):
        """ConvOp arguments over all samples, or sliced to sample n (every batch-indexed tensor)"""
        S = self.samples

        def cut(t):
            if n is None or t is None:
                return t
            k = t.shape[0] // S
            return t[n * k:(n + 1) * k]

        specs = {sid: GNSpec([cut(s) for s in sp["sums"]], sp["C"], sp["gamma"], sp["beta"], sp["eps"], sp["hw"],
                             cut(sp["ss"]), sp["ss_stride"]) for sid, sp in self.specs.items()}
        segs = []
        for sg, src in zip(self.r["segs"], self.srcs):
            am = sg[2]
            aff = None if am is None else (specs[am.sid] if isinstance(am, SpecMeta) else cut(self.tables[am[1]]))
            segs.append((cut(src), sg[1], aff, sg[3], sg[4]))
        kw = dict(self.kw)
        for k in ("out", "out_planar", "stats", "sums_out", "residual"):
            if kw.get(k) is not None:
                kw[k] = cut(kw[k])
        if kw.get("ebias") is not None and kw.get("ebias_stride", 0):
            kw["ebias"] = cut(kw["ebias"])
        if kw.get("weight_batched"):
            weight = cut(self.weight)
        else:
            weight = self.weight
        if n is not None and kw.get("out") is None:
            kw["out_shape"] = (1,) + tuple(kw["out_shape"][1:])
        return segs, weight, kw

    def fresh_outputs(self, kw):
        """N = 1 rebuild: new output buffers (NaN / zero) of the sliced shapes"""
        kw = dict(kw)
        for k in ("out", "out_planar", "stats"):
            if kw.get(k) is not None:
                kw[k] = torch.full_like(kw[k], float("nan"))
        if kw.get("sums_out") is not None:
            kw["sums_out"] = torch.zeros_like(kw["sums_out"])
        return kw


def conv_label(r):
    bn, mt, var, halo, up2, kinds, nseg = r["cls"]
    segs = " + ".join(f"{'1x1 3x3 s2'.split()[sg[1]]}{'' if sg[2] is None else ('*gn' if isinstance(sg[2], SpecMeta) else '*')}"
                      f":{sg[0].shape[-1]}{'' if sg[0].stride[2] == sg[0].shape[-1] else f'(ld {sg[0].stride[2]})'}"
                      for sg in r["segs"])
    return (f"[{r['desc'] or 'conv'}] {segs} -> {r['Cout']} @{r['H']}x{r['W']} N={r['N']} "
            f"BN={bn} MT={mt} {var}{' halo' if halo else ''}{' up2' if up2 else ''} NB={r['nb']}")


def conv_tolerance(r):
    kinds = r["cls"][5]
    kw = r["kw"]
    if kw.get("out") is not None and kw["out"].dtype == torch.float32:
        return TOL_F32
    if "gn" in kinds or (r["cls"][4] and kinds != "raw"):
        return TOL_GN
    if "table" in kinds:
        return TOL_TABLE
    return TOL_F32 if kw.get("out_planar") is not None else TOL_RAW


def replay_conv(r, dev, seed, fails):
    fr = Fresh(dev, seed)
    R = ConvReplay(r, fr)
    segs, weight, kw = R.args()
    op = ops.ConvOp(segs, weight, **kw)
    assert op.cta2 == r["cta2"], conv_label(r)
    op.launch()
    torch.cuda.synchronize()
    label = conv_label(r)
    N, S = r["N"], R.samples
    heads = N // S
    out, planar, stats, sums = kw.get("out"), kw.get("out_planar"), kw.get("stats"), kw.get("sums_out")
    if stats is not None and not torch.isfinite(stats).all():
        fails.append(f"{label}: statistics slots left unwritten")
    check = range(S) if N * r["H"] * r["W"] * r["Cout"] <= (1 << 22) else sorted({0, S - 1})
    entries = [s * heads + h for s in check for h in range(heads)]
    v, st = ref_conv(segs, weight, entries=entries, **kw)
    ou = kw.get("out_heads", 1)
    for i, e in enumerate(entries):
        if planar is not None:
            got = planar[e].double().permute(1, 2, 0)
            ref = v[i][..., :planar.shape[1]]
        elif ou > 1:
            got = out[e // ou, ..., (e % ou) * r["Cout"]:(e % ou + 1) * r["Cout"]].double()
            ref = v[i]
        else:
            got, ref = out[e].double(), v[i]
        got = got.reshape(ref.shape)
        err, mag = (got - ref).abs().max().item(), ref.abs().max().item()
        tol = conv_tolerance(r)
        if not err <= tol * mag + 1e-6:
            fails.append(f"{label}: entry {e} max-abs err {err:.3e} > {tol} * max|ref| {mag:.3e}")
        if stats is not None:
            tol_s = 3e-3 if r["cls"][4] else 2e-3
            got_s = stats[e].double().sum(0)
            es = (got_s - st[i]).abs().max().item()
            if not es <= tol_s * st[i].abs().max().item() + 1e-3:
                fails.append(f"{label}: entry {e} statistics err {es:.3e} (max {st[i].abs().max().item():.3e})")
            if sums is not None:
                es = (sums[e].double() / STAT_SCALE - st[i]).abs().max().item()
                if not es <= tol_s * st[i].abs().max().item() + 1e-3:
                    fails.append(f"{label}: entry {e} int64 sums err {es:.3e}")
    # batch invariance: the same conv at N = 1 on the first and last sample
    for n in sorted({0, S - 1}):
        s1, w1, k1 = R.args(n)
        k1 = R.fresh_outputs(k1)
        op1 = ops.ConvOp(s1, w1, **k1)
        op1.launch()
        torch.cuda.synchronize()
        del op1
        sl = slice(n * heads, (n + 1) * heads) if out is None or out.shape[0] == N else slice(n, n + 1)
        for k in ("out", "out_planar"):
            if kw.get(k) is not None:
                full = kw[k][slice(n, n + 1) if kw[k].shape[0] == S else sl]
                if not torch.equal(full, k1[k]):
                    fails.append(f"{label}: sample {n} of {S} alone != inside the batch ({k})")
        if stats is not None:
            a, b = stats[n], k1["stats"][0]
            if r["nb"] > 1:  # a tile spans NB samples: alone, the sample may sit in other slots of its tile
                a, b = a.sort(dim=0).values, b.sort(dim=0).values
            if not torch.equal(a, b):
                fails.append(f"{label}: sample {n} statistics alone != inside the batch")
            if sums is not None and not torch.equal(sums[n], k1["sums_out"][0]):
                fails.append(f"{label}: sample {n} int64 sums alone != inside the batch")
    del op, R


def replay_call(c, dev, seed, fails):
    """one non-conv launch on fresh operands against its float64 reference"""
    fr = Fresh(dev, seed)
    a = c["args"]
    name = c["name"]
    label = f"{name}(" + ", ".join(f"{k}={list(v.shape) if isinstance(v, Meta) else v}" for k, v in a.items()) + ")"

    def bad(msg):
        fails.append(f"{label}: {msg}")

    if name == "gn_finalize":
        N, HW = a["N"], a["HW"]
        st = []
        for m, Cs in ((a["stats_a"], a["Ca"]), (a["stats_b"], a["Cb"])):
            if m is None:
                st.append(None)
                continue
            T = m.shape[1]
            pix = 2.0 * HW / T  # values per (slot, channel pair)
            mu, var = fr.randn(m.shape[:-1], 0.5).double(), fr.randn(m.shape[:-1], 0.3, 1.0).double().abs()
            s = fr.base(m, "zero")
            s.copy_(torch.stack([pix * mu, pix * (mu * mu + var)], -1))
            st.append(s)
        C = a["Ca"] + a["Cb"]
        gamma, beta = fr.randn((C,), 0.3, 1.0), fr.randn((C,), 0.3)
        ss = fr.base(a["scale_shift"], (0.3, 0.0)) if a["scale_shift"] is not None else None
        aff = fr.base(a["affine"], "nan")
        ops.gn_finalize(st[0], a["Ca"], st[1], a["Cb"], gamma, beta, a["eps"], N, HW, aff, ss, a["ss_stride"])
        torch.cuda.synchronize()
        ref, mag = ref_gn_finalize(st[0], a["Ca"], st[1], a["Cb"], gamma, beta, a["eps"], N, HW, ss, a["ss_stride"])
        # fp32 products of fp64 statistics: <= 8 fp32 ulps of the largest term
        err = (aff.double() - ref).abs() - 2.0 ** -20 * mag
        if not err.max().item() <= 0:
            bad(f"affine off by {err.max().item():.3e} beyond 8 ulps")
    elif name == "apply":
        src_a = fr.base(a["src_a"], (1.5, 0.3))
        src_b = fr.base(a["src_b"], (1.5, 0.3)) if a["src_b"] is not None else None
        aff = None
        if a["affine"] is not None:
            aff = fr.base(a["affine"], (0.5, 0.0))
            aff[..., 0] += 1.0
        out = fr.base(a["out"], "nan")
        ops.apply(src_a, src_b, aff, out, a["act"], a["resample"], a["affine_offset"])
        torch.cuda.synchronize()
        ref = ref_apply(src_a, src_b, aff, a["act"], a["resample"], a["affine_offset"])
        err, mag = (out.double() - ref).abs().max().item(), ref.abs().max().item()
        if not err <= 2e-3 * mag:
            bad(f"max-abs err {err:.3e} of max|ref| {mag:.3e}")
    elif name == "linear":
        w = fr.base(a["weight"], (1.0 / math.sqrt(a["weight"].shape[1]), 0.0))
        b = fr.base(a["bias"], (0.5, 0.0)) if a["bias"] is not None else None
        O = a["weight"].shape[0]
        runs = [(fr.base(a["inp"], (1.0, 0.0)), fr.base(a["out"], "nan"))]
        I = a["weight"].shape[1]
        if I in (128, 256, 512, 1024):  # also several staging passes of the fast path (N > 32 KB / (4 I) samples)
            nc = 32768 // (4 * I)
            runs.append((fr.randn((2 * nc + 1, I)), torch.full((2 * nc + 1, O), float("nan"), device=dev)))
        for inp, out in runs:
            ops.linear(inp, w, b, out, a["act_in"], a["act_out"])
            torch.cuda.synchronize()
            ref, bound = ref_linear(inp, w, b, O, a["act_in"], a["act_out"])
            err = ((out[:, :O].double() - ref).abs() - bound).max().item()
            if not err <= 0:
                bad(f"N={inp.shape[0]}: exceeds the fp32 summation bound by {err:.3e}")
    elif name == "timestep_embedding":
        t = torch.rand(a["t"].shape, generator=fr.g, device=dev) * 1000.0
        out = fr.base(a["out"], "nan")
        ops.timestep_embedding(t, out, a["variant"])
        torch.cuda.synchronize()
        err = (out.double() - ref_timestep_embedding(t, out.shape[1], a["variant"])).abs().max().item()
        if not err < 2e-4:  # sin / cos of fp32 arguments up to ~1e3
            bad(f"max-abs err {err:.3e}")
    elif name == "pack_input":
        x = fr.base(a["x"], (1.0, 0.0))
        out = fr.base(a["out"], "nan")
        ops.pack_input(x, out)
        torch.cuda.synchronize()
        ref = torch.zeros(out.shape, dtype=torch.float16, device=dev)
        ref[..., :x.shape[1]] = x.permute(0, 2, 3, 1).to(torch.float16)
        if not torch.equal(out, ref):
            bad("not the fp16 NHWC copy")
    elif name == "unpack_nchw":
        x = fr.base(a["inp"], (1.0, 0.0))
        out = fr.base(a["out"], "nan")
        ops.unpack_nchw(x, out)
        torch.cuda.synchronize()
        if not torch.equal(out, x.permute(0, 3, 1, 2).float()):
            bad("not the fp32 NCHW copy")
    elif name == "transpose_tc":
        x = fr.base(a["inp"], (1.0, 0.0))
        out = fr.base(a["out"], "nan")
        ops.transpose_tc(x, out)
        torch.cuda.synchronize()
        if not torch.equal(out, x.transpose(1, 2)):
            bad("not the transpose")
    elif name == "softmax_rows":
        S = fr.base(a["S"], (4.0, 0.0))
        P = fr.base(a["P"], "nan")
        ops.softmax_rows(S, P, a["scale"])
        torch.cuda.synchronize()
        ref = torch.softmax(S.double() * a["scale"], dim=-1)
        err = (P.double() - ref).abs().max().item()
        if not err < 6e-4:
            bad(f"max-abs err {err:.3e}")
    elif name == "attention":
        qkv = fr.base(a["qkv"], (1.0, 0.0))
        out = fr.base(a["out"], "nan")
        heads, d = a["heads"], a["head_dim"]
        ops.attention(qkv, out, heads, d, a["scale"])
        torch.cuda.synchronize()
        Nn, T, _ = qkv.shape
        Cc = heads * d
        q, k, v = [qkv[..., i * Cc:(i + 1) * Cc].double().reshape(Nn, T, heads, d).permute(0, 2, 1, 3) for i in range(3)]
        ref = (torch.softmax(q @ k.transpose(-1, -2) * a["scale"], -1) @ v).permute(0, 2, 1, 3).reshape(Nn, T, Cc)
        err, mag = (out.double() - ref).abs().max().item(), ref.abs().max().item()
        if not err <= 1.5e-3 * mag:
            bad(f"max-abs err {err:.3e} of max|ref| {mag:.3e}")
    elif name == "slerp_h":
        h = fr.base(a["h"], (1.0, 0.0))
        N, H, W, C = h.shape
        variants = [(fr.base(a["dh"], (1.0, 0.0)), a["t"] or 0.3, a["use_mask"])]
        shared = fr.randn((C, H, W))  # one delta_h for every sample (dh_sample_stride 0)
        variants += [(shared, 0.3, False), (shared, 0.3, True)]
        for dh, t, use_mask in variants:
            h2 = torch.full(h.shape, float("nan"), dtype=torch.float16, device=dev)
            stats = fr.base(a["stats"], "nan")
            ops.slerp_h(h, dh, h2, stats, t, use_mask)
            torch.cuda.synchronize()
            ref = ref_slerp_h(h, dh if dh.dim() == 4 else dh[None], t, use_mask)
            what = f"dh {list(dh.shape)} t={t} mask={use_mask}"
            err, mag = (h2.double() - ref).abs().max().item(), ref.abs().max().item()
            if not err <= 2e-3 * mag:
                bad(f"{what}: h2 max-abs err {err:.3e} of max|ref| {mag:.3e}")
            sref = pair_stats(ref)
            es = (stats[:, 0].double() - sref).abs().max().item()
            if not es <= 2e-3 * sref.abs().max().item() + 1e-3:
                bad(f"{what}: slot-0 statistics err {es:.3e}")
            if stats.shape[1] > 1 and not torch.equal(stats[:, 1:], torch.zeros_like(stats[:, 1:])):
                bad(f"{what}: statistics slots 1..{stats.shape[1] - 1} not zeroed")
    else:
        raise AssertionError(name)


# ============================================================================ GPU tests
_T0 = {}


@pytest.fixture(scope="module", autouse=True)
def _wall_time():
    _T0["t"] = time.time()
    yield
    print(f"\n[plan replay] wall time of tests/test_plan_replay_gpu.py: {time.time() - _T0['t']:.1f} s")


@pytest.mark.gpu
@pytest.mark.parametrize("workload", list(WORKLOADS))
def test_plan_launches_replay_against_fp64_reference(cuda_device, workload):
    """every unique launch of the workload's plan (GN_FOLD off and on) against the float64 reference, and every conv
    bit-identical at N = 1 on its first and last sample"""
    t0 = time.time()
    rec = record_workload(workload, cuda_device)
    convs, calls = [], []
    for fold, (cv, cl) in rec.items():
        uc, ul = dedup(cv), dedup(cl)
        print(f"\n[plan replay] {workload} GN_FOLD={'on' if fold else 'off'}: {len(uc)} unique conv launches "
              f"(of {len(cv)} created), {len(ul)} unique other launches (of {len(cl)} calls)")
        convs += cv
        calls += cl
    convs, calls = dedup(convs), dedup(calls)
    names = sorted({c["name"] for c in calls})
    for want in ("gn_finalize", "apply", "linear", "timestep_embedding", "pack_input", "unpack_nchw", "slerp_h",
                 "softmax_rows", "transpose_tc"):
        assert want in names, f"{workload}: the plan never called {want}"
    fails, replayed = [], {}
    for i, r in enumerate(convs):
        replay_conv(r, cuda_device, 1000 + i, fails)
        replayed[r["cls"]] = replayed.get(r["cls"], 0) + 1
    for i, c in enumerate(calls):
        replay_call(c, cuda_device, 5000 + i, fails)
    torch.cuda.empty_cache()
    recorded = {r["cls"] for fold in rec.values() for r in fold[0]}
    print(f"[plan replay] {workload}: {len(convs)} unique convs, {len(calls)} unique other launches replayed "
          f"in {time.time() - t0:.1f} s; conv classes:")
    print("    BN  MT  variant  halo   up2    operand   segs  replayed")
    for cls in sorted(replayed, key=str):
        bn, mt, var, halo, up2, kinds, nseg = cls
        print(f"    {bn:<4}{mt:<4}{var:<9}{str(halo):<7}{str(up2):<7}{kinds:<10}{nseg:<6}{replayed[cls]}")
    assert recorded == set(replayed), f"conv classes recorded but not replayed: {recorded - set(replayed)}"
    assert not fails, f"{workload}: {len(fails)} failing launches:\n" + "\n".join(fails)


@pytest.mark.gpu
@pytest.mark.parametrize("workload", list(WORKLOADS))
def test_sampler_updates_in_place_at_workload_shape(cuda_device, workload):
    """asyrp_ddpm_update / asyrp_ddim_update at the workload's (N, Cx, Ce, HW) with x_next aliasing x, as the captured
    trajectory calls them: bitwise equal to the out-of-place call.  DDIM: bitwise equal to the fp32 formula in the
    reference's operation order.  DDPM: exp goes through expf (<= 2 ulps), so the bound is 4 fp32 ulps of the two
    terms it adds, 2^-21 * (|mean| + |sigma z|)."""
    family, _, N = WORKLOADS[workload]
    dev = cuda_device
    Cx, Ce, S = 3, (6 if family == "adm" else 3), 256
    g = torch.Generator().manual_seed(11)
    x = torch.randn(N, Cx, S, S, generator=g)
    et = torch.randn(N, Ce, S, S, generator=g)
    if Ce == 2 * Cx:  # learned log-variance channels in a realistic range
        et[:, Cx:] = torch.rand(N, Cx, S, S, generator=g) * -6.0
    em = et + 0.1 * torch.randn(N, Ce, S, S, generator=g)
    z = torch.randn(N, Cx, S, S, generator=g)
    xd, etd, emd, zd = (t.to(dev) for t in (x, et, em, z))
    f32 = lambda v: torch.tensor(v, dtype=torch.float32)  # noqa: E731
    # DDPM ancestral step
    at, bt, logvar = 0.35, 0.012, -4.2
    for mask in (0.0, 1.0):
        oop = torch.full_like(xd, float("nan"))
        ops.ddpm_update(xd, etd, zd, oop, at, bt, logvar, Ce == 2 * Cx, mask)
        inp = xd.clone()
        ops.ddpm_update(inp, etd, zd, inp, at, bt, logvar, Ce == 2 * Cx, mask)
        torch.cuda.synchronize()
        assert torch.equal(inp, oop), f"{workload}: ddpm_update with x_next is x differs (mask {mask})"
        weight = f32(bt) / torch.sqrt(1 - f32(at))
        inv = 1 / torch.sqrt(1 - f32(bt))
        mean = inv * (x - weight * et[:, :Cx])
        lv = et[:, Cx:2 * Cx] if Ce == 2 * Cx else f32(logvar)
        noise = (f32(mask) * torch.exp(0.5 * lv)) * z
        ref = mean + noise
        excess = ((oop.cpu() - ref).abs() - 2.0 ** -21 * (mean.abs() + noise.abs())).max().item()
        assert excess <= 0, f"{workload}: ddpm_update beyond 4 ulps by {excess:.3e} (mask {mask})"
    # DDIM step, deterministic and with noise, with the x0 output
    at, an = 0.3, 0.6
    c1 = math.sqrt((1 - at / an) * (1 - an) / (1 - at))
    c2 = math.sqrt((1 - an) - c1 ** 2)
    x0 = (x - em[:, :Cx] * torch.sqrt(1 - f32(at))) / torch.sqrt(f32(at))
    for zz, cc1, cc2 in ((None, 0.0, math.sqrt(1 - an)), (zd, c1, c2)):
        oop, x0o = torch.full_like(xd, float("nan")), torch.full_like(xd, float("nan"))
        ops.ddim_update(xd, etd, emd, zz, oop, x0o, at, an, cc1, cc2)
        inp, x0i = xd.clone(), torch.full_like(xd, float("nan"))
        ops.ddim_update(inp, etd, emd, zz, inp, x0i, at, an, cc1, cc2)
        torch.cuda.synchronize()
        ref = torch.sqrt(f32(an)) * x0 + f32(cc2) * et[:, :Cx]
        if zz is not None:
            ref = ref + f32(cc1) * z
        what = f"{workload}: ddim_update ({'eta > 0' if zz is not None else 'eta = 0'})"
        assert torch.equal(inp, oop) and torch.equal(x0i, x0o), f"{what} with x_next is x differs"
        assert torch.equal(oop.cpu(), ref) and torch.equal(x0o.cpu(), x0), f"{what} != the fp32 formula"


# ============================================================================ CPU checks of the references
def _g(seed):
    return torch.Generator().manual_seed(seed)


def _nchw(t):
    return t.double().permute(0, 3, 1, 2)


def _nhwc16(x):
    return x.permute(0, 2, 3, 1).contiguous().to(torch.float16)


def test_ref_conv_segments_bias_residual_stats_vs_torch():
    """1x1 + 3x3 + 3x3-s2-free segments into one accumulator, per-sample ebias rows of a strided table, residual with
    host and device scales, statistics and 2^18 sums"""
    g = _g(1)
    N, H, W, C1, C2, Co = 2, 6, 5, 64, 64, 64
    x1, x2 = torch.randn(N, C1, H, W, generator=g), torch.randn(N, C2, H, W, generator=g)
    w3, w1 = torch.randn(Co, C1, 3, 3, generator=g), torch.randn(Co, C2, 1, 1, generator=g)
    table = torch.randn(N, 3 * Co, generator=g)
    eb = table[:, Co:2 * Co]  # a column slice of a wider per-sample table, stride 3*Co
    res = torch.randn(N, Co, H, W, generator=g)
    wp = torch.cat([ops.pack_conv_weight(w3), ops.pack_conv_weight(w1)], 1)
    want = F.conv2d(h16(x1.double()), h16(w3.double()), padding=1) + F.conv2d(h16(x2.double()), h16(w1.double()))
    want = 0.75 * (want + eb.double()[:, :, None, None]) + 1.5 * h16(res.double())
    segs = [(_nhwc16(x1), MODE_3x3), (_nhwc16(x2), MODE_1x1)]
    for scales, kw in ((None, dict(acc_scale=0.75, res_scale=1.5)), (torch.tensor([0.75, 1.5]), {})):
        v, st = ref_conv(segs, wp, out_shape=(N, H, W, Co), ebias=eb, ebias_stride=3 * Co, residual=_nhwc16(res),
                         scales=scales, **kw)
        assert torch.allclose(_nchw(v), want, rtol=0, atol=1e-9)
        assert torch.allclose(st, pair_stats(want.permute(0, 2, 3, 1)), rtol=1e-12, atol=1e-9)
    v1, _ = ref_conv(segs, wp, out_shape=(N, H, W, Co), ebias=eb, ebias_stride=3 * Co, entries=[1])
    assert torch.allclose(v1[0], (want[1] - 1.5 * h16(res.double())[1]).permute(1, 2, 0) / 0.75, atol=1e-9)
    # stride-2 segment: source [N][2H][2W][C], pad right / bottom by 1; shared ebias row
    xs = torch.randn(N, C1, 2 * H, 2 * W, generator=g)
    b = torch.randn(Co, generator=g)
    v, _ = ref_conv([(_nhwc16(xs), MODE_3x3_S2)], ops.pack_conv_weight(w3), out_shape=(N, H, W, Co), ebias=b)
    want = F.conv2d(F.pad(h16(xs.double()), (0, 1, 0, 1)), h16(w3.double()), stride=2) + b.double()[None, :, None, None]
    assert torch.allclose(_nchw(v), want, atol=1e-9)


def test_ref_conv_operand_transforms_vs_torch():
    """affine table with SiLU and GNSpec (+ scale/shift rows of a wider table): the transform comes before the zero
    padding, its result is rounded to fp16"""
    g = _g(2)
    N, H, W, Ca, Cb, Co = 2, 4, 4, 64, 64, 64
    # multiples of 2^-9: their squares are multiples of 2^-18, so the int64 sums below are exact
    xa, xb = (torch.round((torch.randn(N, c, H, W, generator=g) * 1.5 + 0.3) * 512) / 512 for c in (Ca, Cb))
    w = torch.randn(Co, Ca + Cb, 3, 3, generator=g) / 30
    wp = torch.cat([ops.pack_conv_weight(w[:, :Ca]), ops.pack_conv_weight(w[:, Ca:])], 1)
    xs = torch.cat([h16(xa.double()), h16(xb.double())], 1)
    # affine table, rows [N][Ca+Cb][2]
    aff = torch.stack([torch.randn(N, Ca + Cb, generator=g) * 0.5 + 1, torch.randn(N, Ca + Cb, generator=g) * 0.5], -1)
    y = h16(silu(xs * aff[..., 0].double()[:, :, None, None] + aff[..., 1].double()[:, :, None, None]))
    want = F.conv2d(y, h16(w.double()), padding=1)
    v, _ = ref_conv([(_nhwc16(xa), MODE_3x3, aff, 0, 1), (_nhwc16(xb), MODE_3x3, aff, Ca, 1)], wp,
                    out_shape=(N, H, W, Co))
    assert torch.allclose(_nchw(v), want, atol=1e-9)
    # in-kernel GroupNorm from 2^18 sums of the two sources
    sums = [torch.round(pair_stats(t.permute(0, 2, 3, 1)) * STAT_SCALE).long() for t in (h16(xa.double()), h16(xb.double()))]
    gamma, beta = torch.randn(Ca + Cb, generator=g) * 0.3 + 1, torch.randn(Ca + Cb, generator=g) * 0.3
    wide = torch.randn(N, 2 * (Ca + Cb) + 5, generator=g) * 0.3
    ss = wide[:, 3:3 + 2 * (Ca + Cb)]
    spec = GNSpec(sums, [Ca, Cb], gamma, beta, 1e-5, H * W, ss, wide.shape[1])
    y = F.group_norm(xs, 32, gamma.double(), beta.double(), eps=1e-5)
    y = y * (1 + ss[:, :Ca + Cb].double()[:, :, None, None]) + ss[:, Ca + Cb:].double()[:, :, None, None]
    want = F.conv2d(h16(silu(y)), h16(w.double()), padding=1)
    v, _ = ref_conv([(_nhwc16(xa), MODE_3x3, spec, 0, 1), (_nhwc16(xb), MODE_3x3, spec, Ca, 1)], wp,
                    out_shape=(N, H, W, Co))
    assert (_nchw(v) - want).abs().max().item() <= 1e-9


def test_ref_conv_up2_residual_modes_planar_vs_torch():
    """up2 phases with the packed sub-pixel weights, nearest-x2 / avg-pool residuals, planar output"""
    g = _g(3)
    N, H, W, C = 2, 4, 6, 64
    x = torch.randn(N, C, H, W, generator=g)
    w = torch.randint(-8, 9, (C, C, 3, 3), generator=g).float() / 64  # pre-summed taps stay exact in fp16
    want = F.conv2d(F.interpolate(h16(x.double()), scale_factor=2, mode="nearest"), w.double(), padding=1)
    v, st = ref_conv([(_nhwc16(x), MODE_3x3)], ops.pack_upconv_weight(w), out_shape=(N, 2 * H, 2 * W, C), up2=True)
    assert torch.allclose(_nchw(v), want, atol=1e-9)
    assert torch.allclose(st, pair_stats(want.permute(0, 2, 3, 1)), rtol=1e-12, atol=1e-9)
    a = torch.randn(N, C, H, W, generator=g)
    w3 = torch.randn(C, C, 3, 3, generator=g) / 24
    base = F.conv2d(h16(a.double()), h16(w3.double()), padding=1)
    for mode, rs in ((1, (H // 2, W // 2)), (2, (2 * H, 2 * W))):
        r = torch.randn(N, C, *rs, generator=g)
        skip = F.interpolate(h16(r.double()), scale_factor=2, mode="nearest") if mode == 1 else F.avg_pool2d(h16(r.double()), 2)
        v, _ = ref_conv([(_nhwc16(a), MODE_3x3)], ops.pack_conv_weight(w3), out_shape=(N, H, W, C),
                        residual=_nhwc16(r), res_mode=mode)
        assert torch.allclose(_nchw(v), base + skip, atol=1e-9)
    outp = torch.zeros(N, 3, H, W)
    v, _ = ref_conv([(_nhwc16(a), MODE_3x3)], ops.pack_conv_weight(w3), out_shape=(N, H, W, C), out_planar=outp)
    assert torch.allclose(_nchw(v)[:, :3], base[:, :3], atol=1e-9)


def test_ref_conv_batched_heads_vs_einsum():
    """weight_batched GEMMs of the attention: q k^T per (sample, head) on channel slices of one qkv tensor, and
    P v^T written into the head's channel slice"""
    g = _g(4)
    N, T, heads, d = 2, 16, 2, 64
    C = heads * d
    qkv = torch.randn(N, T, 3 * C, generator=g).to(torch.float16)
    q, k, v = (qkv[..., i * C:(i + 1) * C].double().reshape(N, T, heads, d).permute(0, 2, 1, 3) for i in range(3))
    S = torch.zeros(N * heads, 1, T, T)
    got, _ = ref_conv([(qkv.view(N, 1, T, 3 * C)[..., :d], MODE_1x1)], qkv[:, :, C:C + d], out=S, weight_batched=True,
                      a_heads=heads, b_heads=heads)
    assert torch.allclose(got.reshape(N, heads, T, T), q @ k.transpose(-1, -2), atol=1e-9)
    P = torch.softmax(got, -1).to(torch.float16).reshape(N * heads, 1, T, T)
    vT = qkv[:, :, 2 * C:].transpose(1, 2).contiguous()
    O = torch.zeros(N, 1, T, C, dtype=torch.float16)
    got, _ = ref_conv([(P, MODE_1x1)], vT.view(N * heads, d, T), out=O, weight_batched=True, out_heads=heads)
    want = P.double().reshape(N, heads, T, T) @ v
    assert torch.allclose(got.reshape(N, heads, T, d), want, atol=1e-9)
    # single head: per-sample weight matrices [N][Cout][K]
    got, _ = ref_conv([(qkv.view(N, 1, T, 3 * C)[..., :C], MODE_1x1)], qkv[:, :, C:2 * C], out=torch.zeros(N, 1, T, T),
                      weight_batched=True)
    qq, kk = qkv[..., :C].double(), qkv[..., C:2 * C].double()
    assert torch.allclose(got.reshape(N, T, T), qq @ kk.transpose(1, 2), atol=1e-9)


def test_ref_pointwise_helpers_vs_torch():
    """gn_finalize / apply / linear / slerp references against torch GroupNorm, pooling and the slerp formula"""
    g = _g(5)
    N, H, W, Ca, Cb = 2, 4, 4, 64, 128
    x = torch.randn(N, Ca + Cb, H, W, generator=g) * 1.5 + 0.3
    gamma, beta = torch.randn(Ca + Cb, generator=g) + 1, torch.randn(Ca + Cb, generator=g)
    ss = torch.randn(N, 2 * (Ca + Cb), generator=g) * 0.3
    T = 4  # tile slots: split the pixels into 4 partial sums
    xs = x.double().permute(0, 2, 3, 1).reshape(N, T, -1, Ca + Cb)
    st = torch.stack([pair_stats(xs[:, i]) for i in range(T)], 1)
    aff, _ = ref_gn_finalize(st[..., :Ca // 2, :], Ca, st[..., Ca // 2:, :], Cb, gamma, beta, 1e-6, N, H * W, ss, 2 * (Ca + Cb))
    y = F.group_norm(x.double(), 32, gamma.double(), beta.double(), eps=1e-6)
    y = y * (1 + ss[:, :Ca + Cb].double()[:, :, None, None]) + ss[:, Ca + Cb:].double()[:, :, None, None]
    got = x.double() * aff[..., 0][:, :, None, None] + aff[..., 1][:, :, None, None]
    assert torch.allclose(got, y, atol=1e-9)
    # apply: concat of two sources, table offset, SiLU, both resamples
    sa, sb = _nhwc16(x[:, :Ca]), _nhwc16(x[:, Ca:])
    aff32 = aff.float()
    wide = torch.cat([torch.randn(N, 8, 2, generator=g), aff32], 1)
    a32, b32 = aff32[..., 0].double()[:, :, None, None], aff32[..., 1].double()[:, :, None, None]
    for resample in (0, 1, 2):
        got = ref_apply(sa, sb, wide.contiguous(), 1, resample, affine_offset=8)
        ref = F.silu(torch.cat([_nchw(sa), _nchw(sb)], 1) * a32 + b32)
        ref = F.avg_pool2d(ref, 2) if resample == 1 else (F.interpolate(ref, scale_factor=2) if resample == 2 else ref)
        assert torch.allclose(_nchw(got), ref, atol=1e-9)
    # linear
    inp, w, b = torch.randn(3, 40, generator=g), torch.randn(24, 40, generator=g), torch.randn(24, generator=g)
    y, bound = ref_linear(inp, w, b, 24, act_in=True, act_out=True)
    assert torch.allclose(y, F.silu(F.linear(F.silu(inp.double()), w.double(), b.double())), atol=1e-12)
    assert (bound > 0).all() and bound.max() < 1e-3
    # slerp: t = 0 keeps h, t = 1 gives |h| dh / |dh|; the mask keeps h outside rows 4..H-2, columns 3..4
    h = torch.randn(2, 8, 8, 64, generator=g).to(torch.float16)
    dh = torch.randn(2, 64, 8, 8, generator=g)
    assert torch.allclose(ref_slerp_h(h, dh, 0.0, False), h.double(), atol=1e-9)
    v = ref_slerp_h(h, dh, 1.0, False).permute(0, 3, 1, 2)
    nh = h.double().flatten(1).norm(dim=1)
    assert torch.allclose(v, dh.double() * (nh / dh.double().flatten(1).norm(dim=1))[:, None, None, None], atol=1e-9)
    vm = ref_slerp_h(h, dh, 0.4, True)
    keep = torch.ones(8, 8, dtype=torch.bool)
    keep[4:7, 3:5] = False
    assert torch.equal(vm[:, keep], h.double()[:, keep]) and not torch.allclose(vm[:, ~keep], h.double()[:, ~keep])
    e = ref_timestep_embedding(torch.tensor([0.0, 10.0]), 8, 1)
    assert torch.equal(e[0], torch.tensor([1.0] * 4 + [0.0] * 4, dtype=torch.float64))


def test_tile_class_mirror_examples():
    """the Python mirror of conv_tile_shape / conv_config on the geometries the header documents"""
    assert _tile_shape(32, 32, True) == (8, 16, 1)
    assert _tile_shape(8, 8, False) == (8, 8, 2)
    assert _tile_shape(4, 4, False) == (4, 4, 8)
    assert _tile_shape(1, 256, False) == (128, 1, 1)
    assert _tile_config(256, 256, 16, True, 1) == (16, 2)
    assert _tile_config(8, 8, 512, False, 1)[1] == 1  # NB > 1: never two stacked sub-tiles
