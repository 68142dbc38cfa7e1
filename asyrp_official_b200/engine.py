"""UNet kernel plans and the trajectory engine.

A `UNetEngine` owns, for one UNet (arch.Arch + a state dict in the reference's naming):
  * the packed device weights (fp16 [Cout][K] conv matrices, fp32 biases / norm parameters, fused 1x1 shortcut
    columns, concatenated timestep-embedding projections);
  * one static kernel plan per batch size: pre-created conv ops (TMA descriptors), pooled activation buffers and
    an ordered list of kernel launches for the shared encoder, the Δh injection, and the two decoder passes
    (reference forward: models/ddpm/diffusion.py:473-580, models/improved_ddpm/unet.py:676-752);
  * `forward()` — the reference's per-call semantics — and `sample()` — the whole N-step Asyrp trajectory
    (diffusion_latent.py:499-520 + utils/diffusion_utils.py:24-109) captured once into a CUDA graph and replayed
    with no host synchronisation between steps.

Everything computed here is a kernel of libasyrp_b200.so; torch provides device memory, streams and graphs.
"""
import math
import os

import torch

from . import ops
from .arch import Arch, Attn, Res, Resample
from .ops import MODE_1x1, MODE_3x3, MODE_3x3_S2, RESAMPLE_AVGPOOL2, RESAMPLE_NONE, RESAMPLE_UP2


# ASYRP_DUAL_STREAM=0: run the two decoder passes of an edit step one after the other (A/B measurements)
DUAL_STREAM = os.environ.get("ASYRP_DUAL_STREAM", "1") != "0"
# layers narrower than this keep a pointwise GroupNorm-apply launch instead of the in-kernel operand transform
# (ASYRP_FUSE_MIN_H=8 fuses the 8x8 layers too: 28 launches fewer per edit evaluation)
FUSE_MIN_H = int(os.environ.get("ASYRP_FUSE_MIN_H", "16"))
# ASYRP_GN_FOLD=1: GroupNorm finalised inside the consuming conv kernel from integer-atomic per-sample sums the
# producers' epilogues accumulate (no gn_finalize launch, no affine table) for every layer of at least 16x16: 226 instead
# of 315 launches per edit evaluation, non-conv time 1.04 -> 0.68 ms — but the conv kernels pay more than that back
# (per-tile group statistics on the transform warps' critical path, 64-bit atomics in every epilogue): measured
# 34.2 -> 32.0 img/s (DDPM b16), 35.8 -> 33.7 (AFHQ b8), 5.45 -> 5.17 (ImageNet b4).  Off by default; the path is
# complete and covered by tests (test_groupnorm_finalised_inside_the_consumer_conv, and tests/test_plan_replay_gpu.py
# replays every launch of the four bench plans built with it on).
GN_FOLD = os.environ.get("ASYRP_GN_FOLD", "0") in ("1", "2")
GN_FOLD_PRODUCERS_ONLY = os.environ.get("ASYRP_GN_FOLD", "0") == "2"  # diagnostic: atomics on, consumers use tables
# ResBlock identity skips x + h ride conv2's K loop as an identity weight block (C extra MACs per output, exact: fp16 x
# times 1.0 into the fp32 accumulator).  ASYRP_SKIP_AS_K=0 reads x in the epilogue instead.  A/B on one B200 (round 2,
# ABAB order): 35.57 / 35.51 img/s with the K columns vs 34.39 / 34.30 with the epilogue read — the scattered fp16
# residual loads of the swapped-operand epilogue cost more than 11 % extra MMAs on those convs.
SKIP_AS_K = os.environ.get("ASYRP_SKIP_AS_K", "1") != "0"


class Act:
    """NHWC fp16 activation + the partial GroupNorm sums its producer wrote (per-tile fp32 slots, and — for layers whose
    consumers finalise the GroupNorm in-kernel — per-sample int64 accumulators)"""
    __slots__ = ("t", "stats", "sums")

    def __init__(self, t, stats=None, sums=None):
        self.t, self.stats, self.sums = t, stats, sums

    @property
    def C(self):
        return self.t.shape[3]

    @property
    def H(self):
        return self.t.shape[1]

    @property
    def W(self):
        return self.t.shape[2]


class Launch:
    __slots__ = ("fn", "kind", "flops", "nbytes", "desc", "has_res", "exec_flops")

    def __init__(self, fn, kind, flops, nbytes):
        self.fn, self.kind, self.flops, self.nbytes, self.desc, self.has_res = fn, kind, flops, nbytes, kind, False
        self.exec_flops = flops  # FLOPs the kernel issues; differs from the algorithmic count for sub-pixel up-convs

    def __call__(self):
        self.fn()


class GN:
    """One GroupNorm over the channel concat of `srcs`, in whichever form its consumers need: `spec()` for convs that
    finalise it in-kernel, `table()` (emits the asyrp_gn_finalize launch, once) for the pointwise apply kernel."""

    def __init__(self, plan, srcs, gamma, beta, scale_shift=None, ss_stride=0):
        self.plan, self.srcs, self.gamma, self.beta, self.ss, self.ss_stride = plan, srcs, gamma, beta, scale_shift, ss_stride
        self._table = None

    def spec(self):
        if not GN_FOLD or GN_FOLD_PRODUCERS_ONLY or any(s_.sums is None for s_ in self.srcs):
            return None
        a = self.srcs[0]
        return ops.GNSpec([s_.sums for s_ in self.srcs], [s_.C for s_ in self.srcs], self.gamma, self.beta,
                          self.plan.eng.arch.gn_eps, a.H * a.W, self.ss, self.ss_stride)

    def operand(self):
        """what a fused conv segment takes: the in-kernel spec when available, else the affine table"""
        sp = self.spec()
        return sp if sp is not None else self.table()

    def table(self):
        if self._table is None:
            self._table = self.plan._gn_table(self.srcs, self.gamma, self.beta, self.ss, self.ss_stride)
        return self._table

    def release(self):
        if self._table is not None:
            self.plan.pool.release(self._table)
            self._table = None


class Pool:
    """Exact-size free lists of device buffers.  The plan is a fixed launch sequence on one stream, so a buffer
    released after the last op that reads it can be handed to any later op."""

    def __init__(self, device):
        self.device = device
        self.free = {}
        self.total = 0

    def alloc(self, shape, dtype):
        n = math.prod(shape) * torch.empty((), dtype=dtype).element_size()
        n = (n + 255) // 256 * 256
        lst = self.free.get(n)
        if lst:
            raw = lst.pop()
        else:
            raw = torch.empty(n, dtype=torch.uint8, device=self.device)
            self.total += n
        t = raw[: math.prod(shape) * torch.empty((), dtype=dtype).element_size()].view(dtype).view(shape)
        t._asyrp_raw = raw
        return t

    def release(self, t):
        raw = t._asyrp_raw
        self.free.setdefault(raw.numel(), []).append(raw)


def pack_weights(arch: Arch, sd, device, n_delta):
    """reference-named fp32 state dict -> device tensors the plan consumes"""
    W = {}
    f32 = lambda t: t.detach().to(device=device, dtype=torch.float32).contiguous()  # noqa: E731
    pk = lambda t: ops.pack_conv_weight(t.detach().float()).to(device)  # noqa: E731
    ddpm = arch.family == "ddpm"

    # timestep MLP
    for n in arch.temb_names:
        W[n + ".weight"], W[n + ".bias"] = f32(sd[n + ".weight"]), f32(sd[n + ".bias"])

    # conv_in: input channels padded to one 64-channel K chunk
    w = sd[arch.conv_in + ".weight"].detach().float()
    wpad = torch.zeros(w.shape[0], 64, 3, 3)
    wpad[:, : w.shape[1]] = w.cpu()
    W["conv_in.w"], W["conv_in.b"] = pk(wpad), f32(sd[arch.conv_in + ".bias"])

    emb_w, emb_b, emb_off = [], [], {}
    off = 0

    def add_emb(name, w_, b_):
        nonlocal off
        emb_w.append(w_.detach().float().cpu())
        emb_b.append(b_.detach().float().cpu())
        emb_off[name] = off
        off += w_.shape[0]

    def res(layer):
        p = layer.name
        if ddpm:
            n1, c1, n2, c2, sc = ".norm1", ".conv1", ".norm2", ".conv2", ".nin_shortcut"
            # conv1 bias folded into the timestep projection row: h = conv1(..) + b1 + temb_proj(swish(temb))
            add_emb(p, sd[p + ".temb_proj.weight"], sd[p + ".temb_proj.bias"] + sd[p + c1 + ".bias"])
        else:
            n1, c1, n2, c2, sc = ".in_layers.0", ".in_layers.2", ".out_layers.0", ".out_layers.3", ".skip_connection"
            add_emb(p, sd[p + ".emb_layers.1.weight"], sd[p + ".emb_layers.1.bias"])
            W[p + ".b1"] = f32(sd[p + c1 + ".bias"])
        W[p + ".g1"], W[p + ".be1"] = f32(sd[p + n1 + ".weight"]), f32(sd[p + n1 + ".bias"])
        W[p + ".g2"], W[p + ".be2"] = f32(sd[p + n2 + ".weight"]), f32(sd[p + n2 + ".bias"])
        # K layout is segment-major: a concatenated input (decoder) is two K-segments, each tap-major over its own
        # channels, because the conv reads the two source tensors separately (the concat is never materialised)
        w1 = sd[p + c1 + ".weight"].detach().float()
        parts, o = [], 0
        for c_ in (layer.split or (layer.cin,)):
            parts.append(ops.pack_conv_weight(w1[:, o:o + c_]))
            o += c_
        W[p + ".w1"] = torch.cat(parts, dim=1).contiguous().to(device)
        w2 = ops.pack_conv_weight(sd[p + c2 + ".weight"].detach().float())
        b2 = sd[p + c2 + ".bias"].detach().float().cpu()
        if layer.resample != "none":
            # ADM up / down ResBlock (channels unchanged): the skip branch is x resampled, added by the epilogue through
            # an index-mapped residual read; conv1 of an up block runs on the source image as sub-pixel phases
            assert layer.cin == layer.cout and not layer.split
            W[p + ".w2r"] = w2.contiguous().to(device)
            if layer.resample == "up":
                W[p + ".w1_up"] = ops.pack_upconv_weight(w1).to(device)
        if layer.cin != layer.cout:
            # 1x1 shortcut on the raw (possibly concatenated) input: extra K columns of the same GEMM
            w2 = torch.cat([w2, ops.pack_conv_weight(sd[p + sc + ".weight"].detach().float())], dim=1)
            b2 = b2 + sd[p + sc + ".bias"].detach().float().cpu()
        else:
            # identity skip x + h: a residual read in conv2's epilogue (W[".w2r"]); or (ASYRP_SKIP_AS_K=1) K columns with
            # an identity weight block (exact: fp16 x times 1.0 into the fp32 accumulator), the residual then rides the
            # TMA / tensor-core pipeline at the price of C extra MACs per output
            if layer.resample == "none":
                W[p + ".w2r"] = w2.contiguous().to(device)
            w2 = torch.cat([w2, torch.eye(layer.cout, dtype=w2.dtype, device=w2.device)], dim=1)
        W[p + ".w2"], W[p + ".b2"] = w2.contiguous().to(device), f32(b2)

    def attn(layer):
        p, c = layer.name, layer.c
        W[p + ".g"], W[p + ".be"] = f32(sd[p + ".norm.weight"]), f32(sd[p + ".norm.bias"])
        if ddpm:
            wq = torch.cat([sd[p + f".{n}.weight"].detach().float().reshape(c, c) for n in ("q", "k", "v")], 0)
            bq = torch.cat([sd[p + f".{n}.bias"].detach().float() for n in ("q", "k", "v")], 0)
        else:
            # reference channel order [head][q|k|v][ch] (QKVAttentionLegacy, unet.py:386-388) -> [q|k|v][head][ch]
            d = arch.head_ch
            heads = c // d
            wq = sd[p + ".qkv.weight"].detach().float().reshape(heads, 3, d, c).permute(1, 0, 2, 3).reshape(3 * c, c)
            bq = sd[p + ".qkv.bias"].detach().float().reshape(heads, 3, d).permute(1, 0, 2).reshape(3 * c)
        W[p + ".wqkv"], W[p + ".bqkv"] = pk(wq), f32(bq)
        W[p + ".wproj"] = pk(sd[p + ".proj_out.weight"].detach().float().reshape(c, c))
        W[p + ".bproj"] = f32(sd[p + ".proj_out.bias"])

    def resample(layer):
        p = layer.name
        W[p + ".w"], W[p + ".b"] = pk(sd[p + ".conv.weight"]), f32(sd[p + ".conv.bias"])
        if layer.kind == "up":  # sub-pixel form of conv3x3(nearest-x2(x)): 4 phase kernels of 2x2 taps
            W[p + ".w_up"] = ops.pack_upconv_weight(sd[p + ".conv.weight"].detach().float()).to(device)

    for stage in arch.enc + [arch.mid] + arch.dec:
        for layer in stage:
            {Res: res, Attn: attn, Resample: resample}[type(layer)](layer)

    # conv_out: output channels padded to one 16-wide N tile; only [0, out_ch) is stored (fp32 planar)
    w = sd[arch.conv_out + ".weight"].detach().float().cpu()
    wpad = torch.zeros(16, *w.shape[1:])
    wpad[: w.shape[0]] = w
    bpad = torch.zeros(16)
    bpad[: w.shape[0]] = sd[arch.conv_out + ".bias"].detach().float().cpu()
    W["conv_out.w"], W["conv_out.b"] = pk(wpad), f32(bpad)
    W["norm_out.g"], W["norm_out.be"] = f32(sd[arch.norm_out + ".weight"]), f32(sd[arch.norm_out + ".bias"])

    # DeltaBlocks  (ddpm/diffusion.py:228-263, improved_ddpm/unet.py:776-853)
    for i in range(n_delta):
        p = f"layer_{i}"
        if ddpm:
            W[p + ".w1"] = pk(sd[p + ".conv1.weight"])
            W[p + ".b1"] = f32(sd[p + ".conv1.bias"])
            add_emb(p, sd[p + ".temb_proj.weight"], sd[p + ".temb_proj.bias"] + sd[p + ".conv1.bias"])
            W[p + ".g2"], W[p + ".be2"] = f32(sd[p + ".norm2.weight"]), f32(sd[p + ".norm2.bias"])
            W[p + ".w2"], W[p + ".b2"] = pk(sd[p + ".conv2.weight"]), f32(sd[p + ".conv2.bias"])
        else:
            W[p + ".g1"], W[p + ".be1"] = f32(sd[p + ".in_layers.0.weight"]), f32(sd[p + ".in_layers.0.bias"])
            W[p + ".w1"] = pk(sd[p + ".in_layers.2.weight"])
            W[p + ".b1"] = f32(sd[p + ".in_layers.2.bias"])
            add_emb(p, sd[p + ".emb_layers.1.weight"], sd[p + ".emb_layers.1.bias"] + sd[p + ".in_layers.2.bias"])
            W[p + ".g2"], W[p + ".be2"] = f32(sd[p + ".out_layers.0.weight"]), f32(sd[p + ".out_layers.0.bias"])
            W[p + ".w2"], W[p + ".b2"] = pk(sd[p + ".out_layers.3.weight"]), f32(sd[p + ".out_layers.3.bias"])

    W["emb_cat.w"] = torch.cat(emb_w, 0).to(device).contiguous()
    W["emb_cat.b"] = torch.cat(emb_b, 0).to(device).contiguous()
    return W, emb_off, off


class Plan:
    """Static launch sequence for one batch size"""

    def __init__(self, eng, N):
        self.eng, self.N = eng, N
        a, dev = eng.arch, eng.device
        S = a.image_size
        self.pool = Pool(dev)
        self.x = torch.zeros(N, a.in_ch, S, S, dtype=torch.float32, device=dev)  # sampler state / UNet input
        self.t = torch.zeros(N, dtype=torch.float32, device=dev)
        self.et = torch.zeros(N, a.out_ch, S, S, dtype=torch.float32, device=dev)
        self.et_mod = torch.zeros(N, a.out_ch, S, S, dtype=torch.float32, device=dev)
        self.temb_ops, self.enc_ops, self.delta_ops, self.dec_ops, self.dec_mod_ops = [], [], [], [], []
        # DeltaBlock coefficients (acc_scale, res_scale) of the h2 = c0*h + sum_i c_{i+1}*delta_h_i epilogues live in
        # device memory: one captured graph serves every hs_coeff tuple
        self.coef = torch.ones(max(eng.n_delta, 1), 2, dtype=torch.float32, device=dev)
        # int64 (sum, sum of squares) accumulators of every >= 16x16 conv output, one arena zeroed by ONE memset at the
        # start of an evaluation (a buffer is never reused: two producers must not add into the same sums)
        self.sums_arena = torch.zeros(max(1 << 20, N * 98304), dtype=torch.int64, device=dev) if GN_FOLD else None
        self.sums_used = 0
        self._temps = []     # materialised operands to release after the next conv launch is recorded
        self._cur = self.enc_ops
        self._build()

    # ------------------------------------------------------------------ builder primitives
    def _emit(self, fn, kind="misc", flops=0.0, nbytes=0.0):
        """append one kernel launch; kind / algorithmic flops / algorithmic HBM bytes feed bench.py's roofline"""
        self._cur.append(Launch(fn, kind, flops, nbytes))

    def _act(self, H, W, C, stats=False, has_3x3=False, tiles=None):
        t = self.pool.alloc((self.N, H, W, C), torch.float16)
        st, sums = None, None
        if stats:
            tiles = tiles if tiles is not None else ops.conv_stats_tiles(H, W, C, has_3x3)
            st = self.pool.alloc((self.N, tiles, C // 2, 2), torch.float32)
            if GN_FOLD and H >= 16 and W >= 16:  # tiles lie inside one sample: the epilogue can add per-sample sums
                n = self.N * C
                assert self.sums_used + n <= self.sums_arena.numel(), "sums arena exhausted"
                sums = self.sums_arena[self.sums_used:self.sums_used + n].view(self.N, C // 2, 2)
                self.sums_used += n
        return Act(t, st, sums)

    def _free(self, act):
        self.pool.release(act.t)
        if act.stats is not None:
            self.pool.release(act.stats)

    def _gn(self, srcs, gamma, beta, scale_shift=None, ss_stride=0):
        return GN(self, srcs, gamma, beta, scale_shift, ss_stride)

    def _gn_table(self, srcs, gamma, beta, scale_shift=None, ss_stride=0):
        N = self.N
        C = sum(s.C for s in srcs)
        aff = self.pool.alloc((N, C, 2), torch.float32)
        a, b = srcs[0], (srcs[1] if len(srcs) > 1 else None)
        HW = a.H * a.W
        eps = self.eng.arch.gn_eps
        self._emit(lambda: ops.gn_finalize(a.stats, a.C, b.stats if b else None, b.C if b else 0, gamma, beta, eps, N,
                                           HW, aff, scale_shift, ss_stride), "gn_finalize",
                   nbytes=4.0 * (a.stats.numel() + (b.stats.numel() if b else 0) + aff.numel()))
        return aff

    def _apply(self, srcs, affine, act, resample=RESAMPLE_NONE, affine_offset=0):
        a, b = srcs[0], (srcs[1] if len(srcs) > 1 else None)
        C = sum(s.C for s in srcs)
        H = a.H // 2 if resample == RESAMPLE_AVGPOOL2 else (a.H * 2 if resample == RESAMPLE_UP2 else a.H)
        Wd = a.W // 2 if resample == RESAMPLE_AVGPOOL2 else (a.W * 2 if resample == RESAMPLE_UP2 else a.W)
        out = self._act(H, Wd, C, stats=False)
        n_in = out.t.numel() * (4 if resample == RESAMPLE_AVGPOOL2 else (0.25 if resample == RESAMPLE_UP2 else 1))
        self._emit(lambda: ops.apply(a.t, b.t if b else None, affine, out.t, act, resample, affine_offset), "apply",
                   nbytes=2.0 * (n_in + out.t.numel()))
        return out

    def _conv(self, segs, weight, Cout, H, W, ebias=None, ebias_stride=0, residual=None, res_scale=1.0,
              acc_scale=1.0, stats=True, planar=None, algo_flops=None, up2=False, scales=None, res_mode=0):
        """H, W: output geometry (for up2 = twice the source's)"""
        out = None
        if planar is None:
            out = self._act(H, W, Cout, stats=stats, has_3x3=any(sg[1] == MODE_3x3 for sg in segs),
                            tiles=ops.conv_stats_tiles_up2(H // 2, W // 2, Cout) if up2 else None)
        segs = [tuple(sg) + (None, 0, 0) * (len(sg) == 2) for sg in segs]
        op = ops.ConvOp([(sg[0].t,) + sg[1:] for sg in segs], weight, out=out.t if out else None, ebias=ebias,
                        ebias_stride=ebias_stride, residual=residual.t if residual is not None else None,
                        res_scale=res_scale, acc_scale=acc_scale, stats=out.stats if out else None,
                        out_planar=planar, out_shape=(self.N, H, W, Cout), up2=up2, scales=scales, res_mode=res_mode,
                        sums_out=out.sums if out else None)
        ktot = weight.shape[-1]
        flops = algo_flops if algo_flops is not None else 2.0 * self.N * H * W * Cout * ktot
        nbytes = 2.0 * (sum(sg[0].t.numel() for sg in segs) + weight.numel() + self.N * H * W * Cout
                        + (residual.t.numel() if residual is not None else 0))
        self._emit(op.launch, "conv", flops, nbytes)
        self._cur[-1].exec_flops = 2.0 * self.N * H * W * Cout * ktot if up2 else flops
        self._cur[-1].desc = ("up2 " if up2 else "") + " + ".join(
            f"{'1x1 3x3 s2'.split()[sg[1]]}{'*' if sg[2] is not None else ''}:{sg[0].C}" for sg in segs) + \
            f" -> {Cout} @{H}x{W}"
        self._cur[-1].has_res = residual is not None
        return out, op

    # ------------------------------------------------------------------ blocks
    def _fused(self, srcs, mode, aff, act):
        """conv segments over the channel concat of `srcs` with the GroupNorm affine (+SiLU) fused into the operand.
        Layers smaller than 16x16 keep the pointwise kernel: their K loop is a chain of short stages, and the in-kernel
        transform (one stage at a time) would sit on the critical path; the tensors are ~1 MB."""
        segs, off = [], 0
        small = srcs[0].H < FUSE_MIN_H
        for s_ in srcs:
            if small:
                a_ = self._apply([s_], aff.table(), act, affine_offset=off)
                self._temps.append(a_)
                segs.append((a_, mode))
            else:
                segs.append((s_, mode, aff.operand(), off, act))
            off += s_.C
        return segs

    def _drop_temps(self):
        for a_ in self._temps:
            self._free(a_)
        self._temps = []

    def _res_block(self, layer: Res, srcs):
        """ResnetBlock (ddpm/diffusion.py:151-170) / ResBlock (improved_ddpm/unet.py:278-298): two fused
        GN-apply+SiLU+conv3x3 launches; the 1x1 shortcut is extra K of the second; the block input is read raw."""
        eng, W = self.eng, self.eng.W
        p, ddpm = layer.name, self.eng.arch.family == "ddpm"
        eoff = eng.emb_off[p]
        mode = {"none": RESAMPLE_NONE, "up": RESAMPLE_UP2, "down": RESAMPLE_AVGPOOL2}[layer.resample]
        aff1 = self._gn(srcs, W[p + ".g1"], W[p + ".be1"])
        xr, a1, res_mode, up_fused = None, None, 0, False
        if mode != RESAMPLE_NONE:
            # ADM up/down block: the resample sits between SiLU and the conv, and the skip branch is resampled too
            # (unet.py:279-284).  The skip branch is never materialised: conv2's epilogue reads x through the resample
            # index map (res_mode).  Up: conv1 = conv(nearest-x2(silu(GN(x)))) runs on the source image as four
            # sub-pixel phases with the GN-apply + SiLU fused into the operand.  Down: the pooled activation is
            # materialised (a quarter of the input's size).
            src = srcs[0]
            res_mode = 1 if mode == RESAMPLE_UP2 else 2
            Ho = src.H * 2 if mode == RESAMPLE_UP2 else src.H // 2
            if ops.conv_tile_config(Ho, Ho * src.W // src.H, layer.cout, True) == (128, 2):
                # swapped-operand tile: its epilogue owns one channel per lane, a resampled residual is 32 scattered
                # 2-byte loads per chunk (measured 260 vs 121 us at 256^2) -> materialise x_upd(x) and add it as
                # identity K columns like every other skip
                res_mode = 0
                xr = self._apply(srcs, None, 0, mode)
            up_fused = mode == RESAMPLE_UP2 and src.H >= 16 and ops.conv_stats_tiles_up2(src.H, src.W, layer.cout) > 0
            if up_fused:
                H, Wd = 2 * src.H, 2 * src.W
                segs1 = [(src, MODE_3x3, aff1.operand(), 0, 1)]
            else:
                a1 = self._apply(srcs, aff1.table(), 1, mode)
                segs1, H, Wd = [(a1, MODE_3x3)], a1.H, a1.W
        else:
            segs1, H, Wd = self._fused(srcs, MODE_3x3, aff1, 1), srcs[0].H, srcs[0].W
        if ddpm:
            h, _ = self._conv(segs1, W[p + ".w1"], layer.cout, H, Wd,
                              ebias=self.emb_all[:, eoff:eoff + layer.cout], ebias_stride=eng.emb_total)
            aff2 = self._gn([h], W[p + ".g2"], W[p + ".be2"])
        else:
            if up_fused:
                h, _ = self._conv(segs1, W[p + ".w1_up"], layer.cout, H, Wd, ebias=W[p + ".b1"], up2=True,
                                  algo_flops=2.0 * self.N * H * Wd * layer.cout * 9 * layer.cin)
            else:
                h, _ = self._conv(segs1, W[p + ".w1"], layer.cout, H, Wd, ebias=W[p + ".b1"])
            # GN(h)*(1+scale)+shift, [scale | shift] = Linear(SiLU(emb))  (unet.py:287-294)
            aff2 = self._gn([h], W[p + ".g2"], W[p + ".be2"], self.emb_all[:, eoff:eoff + 2 * layer.cout],
                            eng.emb_total)
        aff1.release()
        if a1 is not None:
            self._free(a1)
        segs2 = self._fused([h], MODE_3x3, aff2, 1)
        if res_mode:
            out, _ = self._conv(segs2, W[p + ".w2r"], layer.cout, H, Wd, ebias=W[p + ".b2"], residual=srcs[0],
                                res_mode=res_mode)
        elif layer.cin != layer.cout:
            out, _ = self._conv(segs2 + [(s_, MODE_1x1) for s_ in srcs], W[p + ".w2"], layer.cout, H, Wd,
                                ebias=W[p + ".b2"])
        elif SKIP_AS_K or xr is not None:
            out, _ = self._conv(segs2 + [(xr if xr is not None else srcs[0], MODE_1x1)], W[p + ".w2"], layer.cout, H, Wd,
                                ebias=W[p + ".b2"],
                                algo_flops=2.0 * self.N * H * Wd * layer.cout * 9 * layer.cout)
        else:
            out, _ = self._conv(segs2, W[p + ".w2r"], layer.cout, H, Wd, ebias=W[p + ".b2"], residual=srcs[0])
        aff2.release()
        self._free(h)
        if xr is not None:
            self._free(xr)
        self._drop_temps()
        return out

    def _attn_block(self, layer: Attn, x):
        a_, W = self.eng.arch, self.eng.W
        p, C = layer.name, layer.c
        d = a_.head_ch if a_.head_ch else C
        heads = C // d
        aff = self._gn([x], W[p + ".g"], W[p + ".be"])
        qkv, _ = self._conv(self._fused([x], MODE_1x1, aff, 0), W[p + ".wqkv"], 3 * C, x.H, x.W, ebias=W[p + ".bqkv"],
                            stats=False)
        aff.release()
        self._drop_temps()
        att = self._act(x.H, x.W, C, stats=False)
        N, T = self.N, x.H * x.W
        scale = float(d) ** -0.5  # C^-0.5 (ddpm/diffusion.py:213) == (d^-1/4)^2 (improved_ddpm/unet.py:389-392)
        if heads == 1 and T % 128 == 0 and T <= 1024:
            # tensor-core path: S = q k^T and O = P v are batched GEMMs on the conv kernel (per-sample "weights" k / v^T)
            qkv3 = qkv.t.view(N, T, 3 * C)
            q4 = qkv.t.view(N, 1, T, 3 * C)[..., :C]
            S = self.pool.alloc((N, 1, T, T), torch.float32)  # logits stay fp32 for the softmax
            Pm = self.pool.alloc((N, 1, T, T), torch.float16)
            vT = self.pool.alloc((N, C, T), torch.float16)
            op_s = ops.ConvOp([(q4, MODE_1x1)], qkv3[:, :, C:2 * C], out=S, weight_batched=True)
            self._emit(op_s.launch, "attention", flops=2.0 * N * T * T * C)
            self._emit(lambda: ops.transpose_tc(qkv3[:, :, 2 * C:], vT), "attention")
            self._emit(lambda: ops.softmax_rows(S, Pm, scale), "attention")
            op_o = ops.ConvOp([(Pm, MODE_1x1)], vT, out=att.t.view(N, 1, T, C), weight_batched=True)
            self._emit(op_o.launch, "attention", flops=2.0 * N * T * T * C)
            for buf in (S, Pm, vT):
                self.pool.release(buf)
        elif d == 64 and T % 128 == 0 and T <= 1024:
            # multi-head (QKVAttentionLegacy): the same two GEMMs batched over (sample, head); q_h / k_h are 64-channel
            # slices of the qkv tensor (head dimension in the TMA maps), O_h is written into its channel slice
            qkv3 = qkv.t.view(N, T, 3 * C)
            q4 = qkv.t.view(N, 1, T, 3 * C)[..., :d]
            S = self.pool.alloc((N * heads, 1, T, T), torch.float32)
            Pm = self.pool.alloc((N * heads, 1, T, T), torch.float16)
            vT = self.pool.alloc((N, C, T), torch.float16)
            op_s = ops.ConvOp([(q4, MODE_1x1)], qkv3[:, :, C:C + d], out=S, weight_batched=True, a_heads=heads,
                              b_heads=heads)
            self._emit(op_s.launch, "attention", flops=2.0 * N * T * T * C)
            self._emit(lambda: ops.transpose_tc(qkv3[:, :, 2 * C:], vT), "attention")
            self._emit(lambda: ops.softmax_rows(S, Pm, scale), "attention")
            op_o = ops.ConvOp([(Pm, MODE_1x1)], vT.view(N * heads, d, T), out=att.t.view(N, 1, T, C),
                              weight_batched=True, out_heads=heads)
            self._emit(op_o.launch, "attention", flops=2.0 * N * T * T * C)
            for buf in (S, Pm, vT):
                self.pool.release(buf)
        else:
            self._emit(lambda: ops.attention(qkv.t.view(N, T, 3 * C), att.t.view(N, T, C), heads, d, scale),
                       "attention", flops=4.0 * N * T * T * C, nbytes=2.0 * N * T * 4 * C)
        out, _ = self._conv([(att, MODE_1x1)], W[p + ".wproj"], C, x.H, x.W, ebias=W[p + ".bproj"], residual=x)
        self._free(qkv)
        self._free(att)
        return out

    def _resample_block(self, layer: Resample, x):
        W = self.eng.W
        p = layer.name
        if layer.kind == "down":
            out, _ = self._conv([(x, MODE_3x3_S2)], W[p + ".w"], layer.c, x.H // 2, x.W // 2, ebias=W[p + ".b"])
            return out
        if ops.conv_stats_tiles_up2(x.H, x.W, layer.c) > 0:
            # Upsample.conv on the source image as four sub-pixel phases (4/9 of the MACs, nothing materialised);
            # algorithmic FLOPs = the reference's 9-tap conv on the 2H x 2W image, executed = 4 taps
            out, _ = self._conv([(x, MODE_3x3)], W[p + ".w_up"], layer.c, 2 * x.H, 2 * x.W, ebias=W[p + ".b"], up2=True,
                                algo_flops=2.0 * self.N * 4 * x.H * x.W * layer.c * 9 * x.C)
            return out
        up = self._apply([x], None, 0, RESAMPLE_UP2)
        out, _ = self._conv([(up, MODE_3x3)], W[p + ".w"], layer.c, up.H, up.W, ebias=W[p + ".b"])
        self._free(up)
        return out

    def _run_stage(self, stage, h, skip=None, keep_input=False):
        """apply the layers of one stage; intermediate tensors are returned to the pool"""
        first = True
        for layer in stage:
            if isinstance(layer, Res):
                srcs = [h, skip] if (first and skip is not None) else [h]
                nh = self._res_block(layer, srcs)
            elif isinstance(layer, Attn):
                nh = self._attn_block(layer, h)
            else:
                nh = self._resample_block(layer, h)
            if not (first and keep_input):
                self._free(h)
            h, first = nh, False
        return h

    # ------------------------------------------------------------------ whole network
    def _build(self):
        eng, a, N, dev = self.eng, self.eng.arch, self.N, self.eng.device
        W = eng.W
        S = a.image_size
        # ---- timestep embedding MLP + every per-block projection in one launch each.  They depend on t only:
        # sample() evaluates them once per schedule step before the loop (a table) and the graph copies one row per step
        self._cur = self.temb_ops
        e0 = torch.zeros(N, a.base_ch, dtype=torch.float32, device=dev)
        e1 = torch.zeros(N, a.temb_ch, dtype=torch.float32, device=dev)
        self.temb = torch.zeros(N, a.temb_ch, dtype=torch.float32, device=dev)
        self.emb_all = torch.zeros(N, eng.emb_total, dtype=torch.float32, device=dev)
        variant = 0 if a.family == "ddpm" else 1
        n0, n1 = a.temb_names
        self._emit(lambda: ops.timestep_embedding(self.t, e0, variant), "temb")
        self._emit(lambda: ops.linear(e0, W[n0 + ".weight"], W[n0 + ".bias"], e1, act_out=True), "temb")
        self._emit(lambda: ops.linear(e1, W[n1 + ".weight"], W[n1 + ".bias"], self.temb), "temb")
        self._emit(lambda: ops.linear(self.temb, W["emb_cat.w"], W["emb_cat.b"], self.emb_all, act_in=True), "temb",
                   nbytes=4.0 * W["emb_cat.w"].numel())
        # ---- encoder
        self._cur = self.enc_ops
        if GN_FOLD:  # zero every int64 statistics accumulator of the evaluation (encoder and both decoder passes) at once
            self._emit(lambda: self.sums_arena[:self.sums_used].zero_(), "memset")
        xin = self._act(S, S, 64, stats=False)
        self._emit(lambda: ops.pack_input(self.x, xin.t), "pack_input", nbytes=4.0 * self.x.numel() + 2.0 * xin.t.numel())
        first_ch = a.enc[1][0].cin
        h, _ = self._conv([(xin, MODE_3x3)], W["conv_in.w"], first_ch, S, S, ebias=W["conv_in.b"],
                          algo_flops=2.0 * N * S * S * first_ch * 9 * a.in_ch)
        self._free(xin)
        hs = [h]
        for stage in a.enc[1:]:
            h = self._run_stage(stage, hs[-1], keep_input=True)
            hs.append(h)
        h = self._run_stage(a.mid, hs[-1], keep_input=True)
        self.middle_h = h
        self.hs = hs
        # ---- Δh injection: h2 = c0*h + sum_i c_{i+1} * layer_i(h, temb)
        self._cur = self.delta_ops
        self.delta_h = None
        h2 = h
        for i in range(eng.n_delta):
            h2 = self._delta_block(i, h, h2, last=(i == eng.n_delta - 1))
        if h2 is h:  # no DeltaBlocks: h2 is only ever produced by the explicit-delta_h path
            h2 = self._act(h.H, h.W, a.mid_ch, stats=True)
        self.h2 = h2
        # explicit delta_h (DiffStyle / raw delta_h checkpoints): h2 = slerp(1-c0, h, |h| dh/|dh|), written into the same
        # h2 buffer (+ its GroupNorm partial sums) the DeltaBlock path produces, so the decoder plan is shared
        self.dh_user = torch.zeros(N, a.mid_ch, h.H, h.W, dtype=torch.float32, device=dev)
        self.slerp_ops = []
        self._cur = self.slerp_ops
        st = eng.state
        self._emit(lambda: ops.slerp_h(self.middle_h.t, self.dh_user, self.h2.t, self.h2.stats, st["slerp_t"],
                                       st["use_mask"]), "slerp")
        # ---- decoders: (h2 -> et_mod) and (h -> et); same weights, same skip tensors.  The second pass allocates from
        # its own pool: in an edit step the two passes are independent and run CONCURRENTLY on two streams
        # (run_edit_and_decoder) — a persistent conv kernel leaves SMs idle in its last wave (512 tiles on 148 SMs =
        # 3.46 rounds), and the other pass's kernel fills them
        self._cur = self.dec_mod_ops
        self._decoder(self.h2, self.et_mod)
        self._cur = self.dec_ops
        main_pool, self.pool = self.pool, Pool(dev)
        self._decoder(self.middle_h, self.et)
        self.side_pool, self.pool = self.pool, main_pool
        self.side_stream = torch.cuda.Stream(device=dev)
        self.mid_f32 = torch.zeros(N, a.mid_ch, h.H, h.W, dtype=torch.float32, device=dev)
        self.delta_f32 = torch.zeros_like(self.mid_f32)

    def _delta_block(self, i, h, h2_prev, last):
        eng, a, W = self.eng, self.eng.arch, self.eng.W
        p, C = f"layer_{i}", a.mid_ch
        eoff = eng.emb_off[p]
        seg1 = [(h, MODE_1x1)]
        aff1 = None
        if a.family == "adm":  # GN, SiLU before the first 1x1 conv (improved_ddpm/unet.py:821-825)
            aff1 = self._gn([h], W[p + ".g1"], W[p + ".be1"])
            seg1 = self._fused([h], MODE_1x1, aff1, 1)
        # two variants of the first conv: with the timestep projection (default) and without (ignore_timestep)
        d1, op_t = self._conv(seg1, W[p + ".w1"], C, h.H, h.W, ebias=self.emb_all[:, eoff:eoff + C],
                              ebias_stride=eng.emb_total)
        self._cur.pop()
        op_nt = ops.ConvOp([(sg[0].t,) + tuple(sg[1:]) for sg in seg1], W[p + ".w1"], out=d1.t, ebias=W[p + ".b1"],
                           stats=d1.stats)
        st = self.eng.state
        self._emit(lambda: (op_nt if st["ignore_timestep"] else op_t).launch(), "conv",
                   2.0 * self.N * h.H * h.W * C * C)
        if aff1 is not None:
            aff1.release()
        aff = self._gn([d1], W[p + ".g2"], W[p + ".be2"])
        seg2 = self._fused([d1], MODE_1x1, aff, 1)
        if last:  # API-visible delta_h = output of the last DeltaBlock
            dh, _ = self._conv(seg2, W[p + ".w2"], C, h.H, h.W, ebias=W[p + ".b2"], stats=False)
            self.delta_h = dh
        # h2 = c_{i+1} * (conv2(a2) + b2) + (c0*h | 1*h2_prev), with GroupNorm partial sums for the decoder
        h2, op = self._conv(seg2, W[p + ".w2"], C, h.H, h.W, ebias=W[p + ".b2"], residual=h2_prev,
                            scales=self.coef[i])
        aff.release()
        self._free(d1)
        self._drop_temps()
        if h2_prev is not h:
            self._free(h2_prev)
        return h2

    def _decoder(self, h_in, out_planar):
        a, W = self.eng.arch, self.eng.W
        h = h_in
        idx = -1
        for si, stage in enumerate(a.dec):
            h = self._run_stage(stage, h, skip=self.hs[idx], keep_input=(si == 0))
            idx -= 1
        aff = self._gn([h], W["norm_out.g"], W["norm_out.be"])
        self._conv(self._fused([h], MODE_3x3, aff, 1), W["conv_out.w"], 16, h.H, h.W, ebias=W["conv_out.b"],
                   stats=False, planar=out_planar, algo_flops=2.0 * self.N * h.H * h.W * a.out_ch * 9 * h.C)
        aff.release()
        self._free(h)
        self._drop_temps()

    # ------------------------------------------------------------------ execution
    def set_coeffs(self, hs_coeff):
        """hs_coeff = (c0, c1, ..): DeltaBlock i's epilogue computes c_{i+1}*(conv + bias) + (c0 if i == 0 else 1)*prev;
        written to device memory (stream-ordered), so it also takes effect for an already captured graph"""
        n = self.eng.n_delta
        if n == 0 or len(hs_coeff) < n + 1:
            return  # schedules without edit steps (origin pass, inversion) carry no DeltaBlock coefficients
        host = torch.tensor([[float(hs_coeff[i + 1]), float(hs_coeff[0]) if i == 0 else 1.0] for i in range(n)],
                            dtype=torch.float32)
        self.coef.copy_(host, non_blocking=False)

    def launches(self, edit, temb=True):
        """kernel launches of one UNet evaluation"""
        ops_ = (self.temb_ops if temb else []) + self.enc_ops + (self.delta_ops + self.dec_mod_ops if edit else []) \
            + self.dec_ops
        return ops_

    def profile(self, edit=True, reps=3):
        """CUDA-event time of every launch of one UNet evaluation (eager, serialised): list of
        (kind, ms, algorithmic flops, algorithmic bytes).  Used by bench.py for the per-kernel roofline."""
        seq = self.launches(edit)
        best = [float("inf")] * len(seq)
        for _ in range(reps):
            evs = []
            for L in seq:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                L()
                e1.record()
                evs.append((e0, e1))
            torch.cuda.synchronize()
            for i, (e0, e1) in enumerate(evs):
                best[i] = min(best[i], e0.elapsed_time(e1))
        return [(L.kind, ms, L.flops, L.nbytes) for L, ms in zip(seq, best)]

    def run_temb(self):
        for f in self.temb_ops:
            f()

    def run_encoder(self):
        for f in self.enc_ops:
            f()

    def graph_time(self, launches, reps=20, warm=5):
        """average device time (ms) of one pass over `launches`, captured as a CUDA graph and replayed back to back:
        the launch gaps, clocks and power state of the real trajectory graph rather than eager per-launch events"""
        st = torch.cuda.Stream(device=self.eng.device)
        st.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(st):
            for L in launches:
                L()
        torch.cuda.current_stream().wait_stream(st)
        torch.cuda.synchronize(self.eng.device)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for L in launches:
                L()
        for _ in range(warm):
            g.replay()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            g.replay()
        e1.record()
        torch.cuda.synchronize(self.eng.device)
        return e0.elapsed_time(e1) / reps

    def run_edit(self, explicit=False):
        for f in (self.slerp_ops if explicit else self.delta_ops):
            f()
        for f in self.dec_mod_ops:
            f()

    def run_decoder(self):
        for f in self.dec_ops:
            f()

    def run_edit_and_decoder(self, explicit=False):
        """edit step: Δh injection + decoder(h2) on the current stream, decoder(h) concurrently on the side stream
        (fork / join by events; inside a stream capture this becomes two parallel branches of the graph)"""
        if not DUAL_STREAM:
            self.run_edit(explicit)
            self.run_decoder()
            return
        cur = torch.cuda.current_stream()
        self.side_stream.wait_stream(cur)
        with torch.cuda.stream(self.side_stream):
            self.run_decoder()
        self.run_edit(explicit)
        cur.wait_stream(self.side_stream)


class UNetEngine:
    """Device weights + plans for one UNet."""

    def __init__(self, arch: Arch, state_dict, device, n_delta=0):
        if not torch.cuda.is_available():
            raise ops._lib.AsyrpError("UNetEngine needs a CUDA device (sm_100a); there is no CPU path")
        ops._lib.load()
        self.arch, self.device, self.n_delta = arch, torch.device(device), n_delta
        self.state = {"ignore_timestep": False, "slerp_t": 0.0, "use_mask": False}
        with torch.cuda.device(self.device):
            self.W, self.emb_off, self.emb_total = pack_weights(arch, state_dict, self.device, n_delta)
        self.plans = {}
        self.graphs = {}

    def plan(self, N) -> Plan:
        if N not in self.plans:
            with torch.cuda.device(self.device):
                self.plans[N] = Plan(self, N)
        return self.plans[N]

    # ---- reference forward() semantics -------------------------------------------------------------
    def forward(self, x, t, index=None, t_edit=400, hs_coeff=(1.0, 1.0), ignore_timestep=False, delta_h=None,
                use_mask=False):
        """(et, et_modified | None, delta_h | None, middle_h) as fp32 NCHW tensors (new tensors, like the reference).
        delta_h given: the explicit-Δh branch, h2 = slerp(1 - hs_coeff[0], h, |h| Δh / |Δh|) (ddpm/diffusion.py:518-539)."""
        N = x.shape[0]
        P = self.plan(N)
        with torch.cuda.device(self.device):
            P.x.copy_(x)
            P.t.copy_(t.to(torch.float32))
            edit = index is not None and float(t[0]) >= t_edit  # host decision, ddpm/diffusion.py:510
            explicit = delta_h is not None
            if index is not None and index + 1 > self.n_delta and edit and not explicit:
                raise ops._lib.AsyrpError(f"index={index} needs {index + 1} DeltaBlocks; engine packed {self.n_delta}")
            self.state["ignore_timestep"] = bool(ignore_timestep)
            P.run_temb()
            P.run_encoder()
            delta = None
            if edit and explicit:
                dh = delta_h.detach().to(self.device, torch.float32)
                P.dh_user.copy_(dh if dh.dim() == 4 else dh[None].expand_as(P.dh_user))
                self.state["slerp_t"], self.state["use_mask"] = 1.0 - float(hs_coeff[0]), bool(use_mask)
                P.run_edit(explicit=True)
                delta = delta_h  # the reference returns the tensor it was given
            elif edit:
                if index + 1 != self.n_delta:
                    raise ops._lib.AsyrpError("forward(index=i) requires i+1 == number of packed DeltaBlocks")
                P.set_coeffs(hs_coeff)
                P.run_edit()
                ops.unpack_nchw(P.delta_h.t, P.delta_f32)
                delta = P.delta_f32.clone()
            P.run_decoder()
            ops.unpack_nchw(P.middle_h.t, P.mid_f32)
            et = P.et.clone()
            if index is None:
                et_mod = None
            elif edit:
                et_mod = P.et_mod.clone()
            else:
                et_mod = et.clone()  # h2 = h below t_edit: the reference's second decoder pass is bit-identical
                if explicit:
                    delta = delta_h
            return et, et_mod, delta, P.mid_f32.clone()

    # ---- whole trajectory --------------------------------------------------------------------------
    MAX_GRAPHS = 4  # captured trajectory graphs kept per engine (least recently used is dropped)

    def _build_trajectory(self, P, schedule, use_graph, explicit, record_dh, record_process):
        """per-(batch, schedule) state: the timestep-embedding table, the noise buffer, the step loop and its graph"""
        steps = schedule.steps
        n_sto = schedule.n_stochastic
        zbuf = torch.zeros((max(n_sto, 1), *P.x.shape), dtype=torch.float32, device=self.device)
        # timestep MLP + every per-block projection depend on t only: evaluate them once per step here (4 launches
        # each, outside the graph); inside the graph a step just copies its row into the buffer the convs read
        emb_table = torch.empty((len(steps), *P.emb_all.shape), dtype=torch.float32, device=self.device)
        for k, s in enumerate(steps):
            P.t.fill_(float(s.t))
            P.run_temb()
            emb_table[k].copy_(P.emb_all)
        learned_sigma = self.arch.out_ch == 2 * self.arch.in_ch

        def is_edit(s):  # 'ddpm' steps use e_t only (utils/diffusion_utils.py:74-82): the edit pass cannot change x
            return s.edit and s.kind == "ddim" and (explicit or self.n_delta > 0)

        n_edit = sum(1 for s in steps if is_edit(s))
        rec = {}
        if explicit:   # per-edit-step explicit delta_h rows (raw-Δh checkpoints / mean Δh), filled before each replay
            rec["dh_in"] = torch.zeros((max(n_edit, 1), *P.dh_user.shape), dtype=torch.float32, device=self.device)
        if record_dh:  # DeltaBlock outputs per edit step (get_delta_hs, diffusion_latent.py:528-532)
            rec["delta_h"] = torch.zeros((max(n_edit, 1), *P.delta_f32.shape), dtype=torch.float32, device=self.device)
        if record_process:  # x_t and x0_t after every step (save_process_*, :485-491,523-527)
            rec["x"] = torch.zeros((len(steps), *P.x.shape), dtype=torch.float32, device=self.device)
            rec["x0_t"] = torch.zeros((len(steps), *P.x.shape), dtype=torch.float32, device=self.device)

        def body():
            zi = ei = 0
            for k, s in enumerate(steps):
                P.emb_all.copy_(emb_table[k])
                P.run_encoder()
                edit = is_edit(s)
                if edit:
                    if explicit:
                        P.dh_user.copy_(rec["dh_in"][ei])
                    P.run_edit_and_decoder(explicit=explicit)
                    if record_dh:
                        ops.unpack_nchw(P.delta_h.t, rec["delta_h"][ei])
                    ei += 1
                else:
                    P.run_decoder()
                z = None
                if s.stochastic:
                    z = zbuf[zi]
                    zi += 1
                if s.kind == "ddpm":
                    ops.ddpm_update(P.x, P.et, z, P.x, s.at, s.bt, s.logvar, learned_sigma, s.mask)
                else:
                    ops.ddim_update(P.x, P.et, P.et_mod if edit else P.et, z, P.x,
                                    rec["x0_t"][k] if record_process else None, s.at, s.an, s.c1, s.c2)
                if record_process:
                    rec["x"][k].copy_(P.x)

        n_launch = sum(len(P.launches(False, temb=False)) + 1 for s in steps)
        n_launch += n_edit * ((len(P.slerp_ops) if explicit else len(P.delta_ops)) + len(P.dec_mod_ops) + int(record_dh))
        g = {"zbuf": zbuf, "emb_table": emb_table, "body": body, "graph": None, "launches": n_launch, "rec": rec,
             "n_edit": n_edit}
        if use_graph:
            s_ = torch.cuda.Stream(device=self.device)
            s_.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s_):
                # warm-up launch outside capture (lazy function attributes, first-touch)
                P.emb_all.copy_(emb_table[0])
                P.run_encoder()
                if explicit or self.n_delta:
                    P.run_edit_and_decoder(explicit=explicit)
                else:
                    P.run_decoder()
            torch.cuda.current_stream().wait_stream(s_)
            torch.cuda.synchronize(self.device)
            cg = torch.cuda.CUDAGraph()
            with torch.cuda.graph(cg):
                body()
            g["graph"] = cg
        return g

    def sample(self, x_T, schedule, noise=None, use_graph=True, out=None, delta_hs=None, use_mask=False,
               record_dh=False, record_process=False):
        """Run the reverse trajectory of `schedule` (sampler.Schedule) from x_T; returns x_0 (fp32 NCHW).

        The step list, the edit/plain/stochastic phase of every step and all sampler coefficients are host-side
        integers / floats fixed before launch, so the whole loop is one CUDA graph: per step a copy of the step's
        timestep-embedding row, the UNet kernels, and the fused DDIM (or ancestral 'ddpm') update that writes x_t in
        place.  The DeltaBlock coefficients hs_coeff are device-side values: every coefficient tuple replays the same
        graph.  noise: [n_stochastic_steps][N][C][H][W] (pre-drawn N(0,1)).

        delta_hs: explicit Δh for the edit steps, [n_edit][C][h][w] (or [n_edit][N][C][h][w]) — the reference's
        forward(delta_h=...) branch: h2 = slerp(1 - hs_coeff[0], h, |h| Δh/|Δh|) (ddpm/diffusion.py:518-539).
        record_dh / record_process: keep the DeltaBlock output of every edit step / (x_t, x0_t) of every step in
        `self.last_records` (device tensors owned by the cached trajectory; clone before the next call)."""
        N = x_T.shape[0]
        P = self.plan(N)
        explicit = delta_hs is not None
        slerp_t = 1.0 - float(schedule.hs_coeff[0]) if explicit else 0.0
        key = (N, bool(use_graph), schedule.key(), explicit, slerp_t, bool(use_mask) if explicit else False,
               bool(record_dh), bool(record_process))
        with torch.cuda.device(self.device):
            n_sto = schedule.n_stochastic
            if n_sto:
                assert noise is not None and noise.shape[0] == n_sto, "pre-drawn noise required for stochastic steps"
            # kernel variants / parameters baked at capture time (all part of `key`)
            self.state["ignore_timestep"] = schedule.ignore_timestep
            self.state["slerp_t"], self.state["use_mask"] = slerp_t, bool(use_mask)
            if record_dh and (explicit or self.n_delta == 0):
                raise ops._lib.AsyrpError("record_dh needs the DeltaBlock path")
            g = self.graphs.pop(key, None)
            if g is None:
                g = self._build_trajectory(P, schedule, use_graph, explicit, record_dh, record_process)
                while len(self.graphs) >= self.MAX_GRAPHS:
                    self.graphs.pop(next(iter(self.graphs)))
            self.graphs[key] = g  # most recently used last
            self.last_launches = g["launches"]
            self.last_records = g["rec"]
            P.set_coeffs(schedule.hs_coeff)
            if explicit and g["n_edit"]:
                dh = delta_hs.to(self.device, torch.float32)
                assert dh.shape[0] == g["n_edit"], f"delta_hs has {dh.shape[0]} rows, schedule has {g['n_edit']} edit steps"
                g["rec"]["dh_in"].copy_(dh if dh.dim() == 5 else dh[:, None].expand_as(g["rec"]["dh_in"]))
            P.x.copy_(x_T, non_blocking=True)
            if n_sto:
                g["zbuf"].copy_(noise, non_blocking=True)
            if g["graph"] is not None:
                g["graph"].replay()
            else:
                g["body"]()
            if out is None:
                return P.x.clone()
            out.copy_(P.x)
            return out
