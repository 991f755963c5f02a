"""B200-native UNet for the SD-v1 denoising loop: drop-in for the reference's
`ldm.modules.diffusionmodules.openaimodel.UNetModel` (constructor kwargs openaimodel.py:443-469,
`forward(x, timesteps, context)` openaimodel.py:710-742, state-dict keys unchanged).

Nothing here computes with torch: forward() only sequences the hand-written sm_100a kernels of libsdb200.so
(ops.py). torch provides device memory and the current stream. nn.Module is used solely so that the reference's
`load_state_dict` / `instantiate_from_config` plumbing (ldm/util.py:78-93, scripts/txt2img.py:49-66) sees this
object; there are no nn layers and no parameters.

Data layout: activations NHWC; the residual stream is fp32, tensor-core operands are fp16 (fp32 accumulate);
GroupNorm/LayerNorm statistics, softmax, FiLM and residual adds are fp32 (SURVEY.md §7.3-1).
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops
from .arch import unet_param_shapes, unet_plan
from .ops import ACT_GEGLU, ACT_SILU
from .util import adopt_state_dict


def _dpad(d):
    return (d + 63) // 64 * 64


def _pack_conv3(w):  # [Cout, Cin, 3, 3] -> [Cout, 9*Cin], k = (ky*3+kx)*Cin + c
    return w.permute(0, 2, 3, 1).reshape(w.shape[0], -1).contiguous().half()


def _pack_conv3_padk(w, kpad):  # small-Cin convs through im2col: K zero-padded to kpad
    p = torch.zeros((w.shape[0], kpad), dtype=torch.float16, device=w.device)
    p[:, : 9 * w.shape[1]] = _pack_conv3(w)
    return p


def _pack_heads(w, heads, d, dpad):  # [heads*d, K] -> [heads*dpad, K], zero rows between heads
    K = w.shape[1]
    p = torch.zeros((heads, dpad, K), dtype=torch.float16, device=w.device)
    p[:, :d] = w.reshape(heads, d, K).half()
    return p.reshape(heads * dpad, K).contiguous()


def _hilo(w):
    hi = w.half()
    return hi, (w - hi.float()).half()


def _pack_hilo_1x1(w):  # [N, K] fp32 -> [N, 3K] = [W_hi | W_hi | W_lo], multiplied by A = [A_hi | A_lo | A_hi]
    hi, lo = _hilo(w)
    return torch.cat([hi, hi, lo], dim=1).contiguous()


def _pack_hilo_conv3(w):  # [N, C, 3, 3] fp32 -> [N, 9 * 3C], per tap [W_hi | W_hi | W_lo]
    wk = w.permute(0, 2, 3, 1).reshape(w.shape[0], 9, w.shape[1])
    hi, lo = _hilo(wk)
    return torch.cat([hi, hi, lo], dim=2).reshape(w.shape[0], -1).contiguous()


def _geglu_tile(inner):
    """Accumulator tile width of the GEGLU GEMM: 256 ([128 value | 128 gate], CTA-pair tiles) when the inner width
    allows, else 128."""
    return 256 if inner % 128 == 0 else 128


def _pack_geglu(w, b):  # [8C, C]: rows [0,4C) value, [4C,8C) gate -> per accumulator tile [half value | half gate]
    inner = w.shape[0] // 2
    half = _geglu_tile(inner) // 2
    assert inner % half == 0
    idx = torch.arange(inner, device=w.device).reshape(-1, half)
    perm = torch.cat([idx, idx + inner], dim=1).reshape(-1)
    return w[perm].contiguous().half(), b[perm].contiguous().float()


class UNetModel(nn.Module):
    # The 1x1 convs that act on the raw residual stream (ResBlock skip_connection, SpatialTransformer proj_in /
    # proj_out) and the final 320->4 conv run with hi/lo-split fp16 operands (three tensor-core passes, ~fp32 operand
    # precision); everything else is single-pass fp16. These few layers (5% of the FLOPs) carry ~60% of the fp16
    # operand-rounding error of eps (DESIGN.md, numerics).

    def __init__(self, image_size, in_channels, model_channels, out_channels, num_res_blocks, attention_resolutions,
                 dropout=0, channel_mult=(1, 2, 4, 8), conv_resample=True, dims=2, num_classes=None,
                 use_checkpoint=False, use_fp16=False, num_heads=-1, num_head_channels=-1, num_heads_upsample=-1,
                 use_scale_shift_norm=False, resblock_updown=False, use_new_attention_order=False,
                 use_spatial_transformer=False, transformer_depth=1, context_dim=None, n_embed=None, legacy=True):
        super().__init__()
        # same argument checks as the reference (openaimodel.py:471-489)
        if use_spatial_transformer:
            assert context_dim is not None, "Fool!! You forgot to include the dimension of your cross-attention conditioning..."
        if context_dim is not None:
            assert use_spatial_transformer, "Fool!! You forgot to use the spatial transformer for your cross-attention conditioning..."
            context_dim = list(context_dim) if isinstance(context_dim, (list, tuple)) else context_dim
        if num_heads == -1:
            assert num_head_channels != -1, "Either num_heads or num_head_channels has to be set"
        # the B200 path covers the configuration SD v1 ships (v1-inference.yaml:29-44)
        unsupported = dict(dims=dims != 2, num_classes=num_classes is not None, resblock_updown=resblock_updown,
                           use_scale_shift_norm=use_scale_shift_norm, n_embed=n_embed is not None,
                           no_spatial_transformer=not use_spatial_transformer, transformer_depth=transformer_depth != 1,
                           num_head_channels=num_head_channels != -1, dropout=dropout != 0,
                           conv_resample=not conv_resample)
        bad = [k for k, v in unsupported.items() if v]
        if bad:
            raise NotImplementedError(f"sdb200.UNetModel supports the SD-v1 UNet configuration only; unsupported: {bad}")
        self.cfg = dict(image_size=image_size, in_channels=in_channels, model_channels=model_channels,
                        out_channels=out_channels, num_res_blocks=num_res_blocks,
                        attention_resolutions=list(attention_resolutions), channel_mult=list(channel_mult),
                        num_heads=num_heads, use_spatial_transformer=True, transformer_depth=1,
                        context_dim=context_dim, legacy=legacy)
        self.in_channels, self.model_channels, self.out_channels = in_channels, model_channels, out_channels
        self.num_heads = num_heads
        self.context_dim = context_dim
        self.dtype = torch.float32
        self.plan = unet_plan(self.cfg)
        self.shapes = unet_param_shapes(self.cfg)
        # channels per fused GroupNorm-statistics entry: every channel count of the UNet (and of its skip concats) is a
        # multiple of model_channels, so the 32 groups always tile into entries of model_channels / 32 channels
        self._sg = model_channels // 32 if model_channels % 32 == 0 else 1
        self.W = None           # packed weights (device)
        self._ctx_ref = None    # the context tensor whose cross-attention K/V are cached (strong reference)
        self._ctx_ver = -1
        self._ctx_kv = None
        self._kv_static = {}
        self._graphs = {}
        self._arena = None
        self._side = None       # side stream of the FiLM chain (forked / joined inside every forward, graph-capturable)
        self.use_cuda_graph = False   # replay one captured graph per UNet evaluation (set by the pipeline / bench)
        self.autotune = True          # graph mode: pick (block_n, split-K) per GEMM problem by measurement before capture

    # ------------------------------------------------------------------ weights
    def _load_from_state_dict(self, state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys,
                              error_msgs):
        sd = adopt_state_dict(self, state_dict, prefix, missing_keys, unexpected_keys, error_msgs)
        if sd is None:
            return
        self._host_sd = sd
        if self.W is not None:
            self.pack_weights(self.W["device"])

    def load_weights(self, sd, device):
        """sd: UNetModel.state_dict()-style mapping (reference key names). Packs to kernel-native fp16 layouts."""
        for k, shape in self.shapes.items():
            assert k in sd, f"missing key {k}"
            assert tuple(sd[k].shape) == tuple(shape), (k, tuple(sd[k].shape), shape)
        self._host_sd = {k: sd[k] for k in self.shapes}
        self.pack_weights(torch.device(device))
        return self

    def _apply(self, fn, *a, **k):  # .cuda()/.to(device) triggers packing, like moving an nn.Module's parameters
        r = super()._apply(fn, *a, **k)
        probe = fn(torch.empty(0))
        if probe.is_cuda and getattr(self, "_host_sd", None) is not None and (self.W is None or self.W["device"] != probe.device):
            self.pack_weights(probe.device)
        return r

    @torch.no_grad()
    def pack_weights(self, device):
        sd = {k: v.detach().to(device=device, dtype=torch.float32) for k, v in self._host_sd.items()}
        W = {"device": device}
        f32 = lambda k: sd[k].contiguous()
        f16 = lambda k: sd[k].half().contiguous()
        heads = self.num_heads
        mc = self.model_channels
        W["te0_w"], W["te0_b"] = f16("time_embed.0.weight"), f32("time_embed.0.bias")
        W["te2_w"], W["te2_b"] = f16("time_embed.2.weight"), f32("time_embed.2.bias")
        emb_w, emb_b, emb_off = [], [], {}
        off = 0

        def pack_res(pre, a):
            nonlocal off
            r = {"cin": a["cin"], "cout": a["cout"]}
            r["gn1"] = (f32(pre + ".in_layers.0.weight"), f32(pre + ".in_layers.0.bias"))
            r["w1"], r["b1"] = _pack_conv3(sd[pre + ".in_layers.2.weight"]), f32(pre + ".in_layers.2.bias")
            r["gn2"] = (f32(pre + ".out_layers.0.weight"), f32(pre + ".out_layers.0.bias"))
            r["w2"], r["b2"] = _pack_conv3(sd[pre + ".out_layers.3.weight"]), f32(pre + ".out_layers.3.bias")
            if a["cin"] != a["cout"]:
                r["ws"] = _pack_hilo_1x1(sd[pre + ".skip_connection.weight"].reshape(a["cout"], a["cin"]))
                r["bs"] = f32(pre + ".skip_connection.bias")
            emb_w.append(sd[pre + ".emb_layers.1.weight"].half())
            emb_b.append(sd[pre + ".emb_layers.1.bias"])
            r["film_off"] = off
            off += a["cout"]
            return r

        def pack_st(pre, a):
            ch, d = a["ch"], a["dhead"]
            dp = _dpad(d)
            tb = pre + ".transformer_blocks.0"
            s = {"ch": ch, "d": d, "dpad": dp, "heads": heads}
            s["gn"] = (f32(pre + ".norm.weight"), f32(pre + ".norm.bias"))
            s["w_in"], s["b_in"] = _pack_hilo_1x1(sd[pre + ".proj_in.weight"].reshape(ch, ch)), f32(pre + ".proj_in.bias")
            s["w_out"], s["b_out"] = _pack_hilo_1x1(sd[pre + ".proj_out.weight"].reshape(ch, ch)), f32(pre + ".proj_out.bias")
            for i in (1, 2, 3):
                s[f"ln{i}"] = (f32(f"{tb}.norm{i}.weight"), f32(f"{tb}.norm{i}.bias"))
            s["w_qk1"] = torch.cat([_pack_heads(sd[tb + ".attn1.to_q.weight"], heads, d, dp),
                                    _pack_heads(sd[tb + ".attn1.to_k.weight"], heads, d, dp)], 0).contiguous()
            s["w_v1"] = _pack_heads(sd[tb + ".attn1.to_v.weight"], heads, d, dp)
            s["w_o1"], s["b_o1"] = f16(tb + ".attn1.to_out.0.weight"), f32(tb + ".attn1.to_out.0.bias")
            s["w_q2"] = _pack_heads(sd[tb + ".attn2.to_q.weight"], heads, d, dp)
            s["w_k2"] = _pack_heads(sd[tb + ".attn2.to_k.weight"], heads, d, dp)
            s["w_v2"] = _pack_heads(sd[tb + ".attn2.to_v.weight"], heads, d, dp)
            s["w_o2"], s["b_o2"] = f16(tb + ".attn2.to_out.0.weight"), f32(tb + ".attn2.to_out.0.bias")
            s["w_ff1"], s["b_ff1"] = _pack_geglu(sd[tb + ".ff.net.0.proj.weight"], sd[tb + ".ff.net.0.proj.bias"])
            s["w_ff2"], s["b_ff2"] = f16(tb + ".ff.net.2.weight"), f32(tb + ".ff.net.2.bias")
            return s

        def pack_layers(layers):
            out = []
            for kind, pre, a in layers:
                if kind == "conv_in":
                    out.append((kind, {"w": _pack_conv3_padk(sd[pre + ".weight"], 64), "b": f32(pre + ".bias"),
                                       "cout": a["cout"]}))
                elif kind == "res":
                    out.append((kind, pack_res(pre, a)))
                elif kind == "st":
                    out.append((kind, pack_st(pre, a)))
                elif kind == "down":
                    out.append((kind, {"w": _pack_conv3(sd[pre + ".op.weight"]), "b": f32(pre + ".op.bias"), "ch": a["ch"]}))
                elif kind == "up":
                    out.append((kind, {"w": _pack_conv3(sd[pre + ".conv.weight"]), "b": f32(pre + ".conv.bias"), "ch": a["ch"]}))
            return out

        W["input"] = [pack_layers(l) for l in self.plan["input"]]
        W["middle"] = pack_layers(self.plan["middle"])
        W["output"] = [pack_layers(l) for l in self.plan["output"]]
        W["gn_out"] = (f32("out.0.weight"), f32("out.0.bias"))
        W["w_out"] = _pack_hilo_conv3(sd["out.2.weight"])
        W["b_out"] = f32("out.2.bias")
        W["emb_w"] = torch.cat(emb_w, 0).contiguous()
        W["emb_b"] = torch.cat(emb_b, 0).float().contiguous()
        W["st_list"] = [p for grp in W["input"] + [W["middle"]] + W["output"] for k, p in grp if k == "st"]
        self.W = W
        self._ctx_ref = None
        self._kv_static = {}
        self._graphs = {}

    # ------------------------------------------------------------------ blocks
    def _film(self, t):
        """time_embed MLP + all 22 emb_layers in three weight-streaming launches (fp32 activations)."""
        W = self.W
        te = ops.timestep_embedding_f32(t, self.model_channels)
        h = ops.linear_small(te, W["te0_w"], W["te0_b"], act=ACT_SILU)
        # ResBlocks only ever consume SiLU(emb) (openaimodel.py:217-218), so apply it in this epilogue
        h = ops.linear_small(h, W["te2_w"], W["te2_b"], act=ACT_SILU)
        return ops.linear_small(h, W["emb_w"], W["emb_b"])          # [N, sum(Cout)] fp32

    def _res(self, r, h, skip, film, emit_f16=False):
        """ResBlock._forward (openaimodel.py:255-275); `skip` is the UNet skip tensor concatenated along C.
        emit_f16: the last GEMM also writes an fp16 copy of the block output (operand of a following stride-2 conv)."""
        nb, H, Wd, _ = h.shape
        if "ws" in r:
            hn, raw, _, raw_lo = ops.groupnorm(h, *r["gn1"], x1=skip, eps=1e-5, silu=True, want_raw_lo=True)
        else:
            hn, _ = ops.groupnorm(h, *r["gn1"], x1=skip, eps=1e-5, silu=True)
        fv = film[:, r["film_off"]: r["film_off"] + r["cout"]]
        _, h1 = ops.gemm(hn, r["w1"], taps=9, bias=r["b1"], film=fv, want_f32=True, splits=-1, want_stats=True, stats_group=self._sg)
        h1 = h1.view(nb, H, Wd, r["cout"])
        hn2, _ = ops.groupnorm(h1, *r["gn2"], eps=1e-5, silu=True)
        if "ws" in r:    # skip 1x1 conv on the raw stream: [x_hi | x_lo | x_hi] . [W_hi | W_hi | W_lo]
            _, res = ops.gemm(raw, r["ws"], a1=raw_lo, a2=raw, bias=r["bs"], want_f32=True, splits=-1)
        else:
            assert skip is None
            res = h.view(-1, r["cout"])
        o16, out = ops.gemm(hn2, r["w2"], taps=9, bias=r["b2"], residual=res, want_f32=True, want_f16=emit_f16, splits=-1,
                            want_stats=True, stats_group=self._sg)
        out = out.view(nb, H, Wd, r["cout"])
        if emit_f16:
            out._sdb_f16 = o16.view(nb, H, Wd, r["cout"])
        return out

    def _st(self, s, x, kv, emit_f16=False):
        """SpatialTransformer.forward (attention.py:250-261) with one BasicTransformerBlock (:211-215)."""
        nb, H, Wd, ch = x.shape
        ntok = H * Wd
        heads, d, dp = s["heads"], s["d"], s["dpad"]
        hd = heads * dp
        scale = d ** -0.5
        xn, _, xn_lo, _ = ops.groupnorm(x, *s["gn"], eps=1e-6, silu=False, want_lo=True)
        _, t0 = ops.gemm(xn, s["w_in"], a1=xn_lo, a2=xn, bias=s["b_in"], want_f32=True, splits=-1)   # tokens [M, ch] fp32
        # --- self attention
        y = ops.layernorm(t0, *s["ln1"])
        qk, _ = ops.gemm(y, s["w_qk1"], want_f16=True)                                     # [M, 2*hd]
        qk3 = qk.view(nb, ntok, 2 * hd)
        if ntok % 8 == 0:
            # V^T straight out of the tensor cores by swapping the operand roles: [hd, M] = Wv . y^T
            vt, _ = ops.gemm(s["w_v1"], y, want_f16=True, b_dynamic=True)
            vt3 = vt.view(hd, nb, ntok).permute(1, 0, 2)                                   # [nb, hd, ntok] (strided view)
        else:  # TMA needs 16-byte aligned strides: tiny token counts go through an explicit transpose
            v, _ = ops.gemm(y, s["w_v1"], want_f16=True)
            vt3 = ops.transpose_f16(v.view(nb, ntok, hd))
        o = ops.attention(qk3[:, :, :hd], qk3[:, :, hd:], vt3, heads=heads, d=d, dpad=dp, nq=ntok, nkv=ntok, scale=scale)
        _, t1 = ops.gemm(o.view(-1, ch), s["w_o1"], bias=s["b_o1"], residual=t0, want_f32=True, splits=-1)
        # --- cross attention (K / V^T of the context are precomputed per prompt)
        y = ops.layernorm(t1, *s["ln2"])
        q, _ = ops.gemm(y, s["w_q2"], want_f16=True)
        k2, vt2, nkv = kv
        o = ops.attention(q.view(nb, ntok, hd), k2, vt2, heads=heads, d=d, dpad=dp, nq=ntok, nkv=nkv, scale=scale)
        _, t2 = ops.gemm(o.view(-1, ch), s["w_o2"], bias=s["b_o2"], residual=t1, want_f32=True, splits=-1)
        # --- GEGLU feed-forward
        y = ops.layernorm(t2, *s["ln3"])
        g, _ = ops.gemm(y, s["w_ff1"], bias=s["b_ff1"], act=ACT_GEGLU, want_f16=True,
                        block_n=_geglu_tile(s["w_ff1"].shape[0] // 2))
        t3, _, t3_lo = ops.gemm(g, s["w_ff2"], bias=s["b_ff2"], residual=t2, want_lo=True, splits=-1)
        o16, out = ops.gemm(t3, s["w_out"], a1=t3_lo, a2=t3, bias=s["b_out"], residual=x.view(-1, ch), want_f32=True,
                            want_f16=emit_f16, splits=-1, rows_per_sample=ntok, want_stats=True, stats_group=self._sg)
        out = out.view(nb, H, Wd, ch)
        if emit_f16:
            out._sdb_f16 = o16.view(nb, H, Wd, ch)
        return out

    def context_kv(self, context, static=False):
        """Cross-attention K and V^T for all SpatialTransformers (x/t independent: once per prompt).
        static=True writes into persistent per-shape buffers so captured CUDA graphs stay valid across prompts."""
        nb, nkv, cd = context.shape
        ctx16 = ops.cast_f16(context.contiguous().float().view(nb * nkv, cd))
        bufs = self._kv_static.setdefault((nb, nkv), {}) if static else {}
        ld = (nkv + 7) // 8 * 8
        out = []
        for i, s in enumerate(self.W["st_list"]):
            hd = s["heads"] * s["dpad"]
            if i not in bufs:
                bufs[i] = (torch.empty((nb * nkv, hd), dtype=torch.float16, device=context.device),
                           torch.empty((nb * nkv, hd), dtype=torch.float16, device=context.device),
                           torch.empty((nb, hd, ld), dtype=torch.float16, device=context.device))
            kb, vb, vtb = bufs[i]
            ops.gemm(ctx16, s["w_k2"], out_f16=kb)
            ops.gemm(ctx16, s["w_v2"], out_f16=vb)
            ops.transpose_f16(vb.view(nb, nkv, hd), out=vtb)
            out.append((kb.view(nb, nkv, hd), vtb, nkv))
        return out

    def set_context(self, context):
        """Cache the cross-attention K/V for `context` ([uncond; cond] batch). forward() reuses them for the same
        tensor object (unmodified since) or for a tensor with equal contents; the cached tensor is kept alive, so a new
        prompt can never alias it through a recycled allocation."""
        self._ctx_kv = self.context_kv(context, static=True)
        self._ctx_ref, self._ctx_ver = context, context._version
        return self._ctx_kv

    def _context_cached(self, context):
        ref = self._ctx_ref
        if ref is None or self._ctx_kv is None:
            return False
        if context is ref:
            return context._version == self._ctx_ver
        # a different tensor object (the reference samplers build torch.cat([uc, c]) every step, plms.py:182-185):
        # compare contents - a 2x77x768 compare is far cheaper than 32 projection GEMMs
        return (ref._version == self._ctx_ver and context.shape == ref.shape and context.dtype == ref.dtype
                and context.device == ref.device and bool(torch.equal(context, ref)))

    def _run_layers(self, layers, h, skip, film, kvs, st_idx, emit_f16=False):
        """emit_f16: the block's output feeds a Downsample next, whose stride-2 conv reads an fp16 copy through TMA."""
        for li, (kind, p) in enumerate(layers):
            last = emit_f16 and li == len(layers) - 1
            if kind == "res":
                h = self._res(p, h, skip, film, emit_f16=last)
                skip = None
            elif kind == "st":
                h = self._st(p, h, kvs[st_idx[0]], emit_f16=last)
                st_idx[0] += 1
            elif kind == "down":
                # Downsample (openaimodel.py:149-153): 3x3, stride 2, pad 1, straight from the NHWC activation through
                # strided TMA boxes (element strides {1,2,2,1}); no im2col buffer
                nb, H, Wd, c = h.shape
                h16 = getattr(h, "_sdb_f16", None)
                if h16 is None:
                    h16 = ops.cast_f16(h)
                _, o = ops.gemm(h16, p["w"], taps=9, conv_stride=2, bias=p["b"], want_f32=True, splits=-1, want_stats=True, stats_group=self._sg)
                h = o.view(nb, (H + 1) // 2, (Wd + 1) // 2, c)
            elif kind == "up":
                nb, H, Wd, c = h.shape
                up = ops.upsample2x(h)
                _, o = ops.gemm(up, p["w"], taps=9, bias=p["b"], want_f32=True, splits=-1, want_stats=True, stats_group=self._sg)
                h = o.view(nb, 2 * H, 2 * Wd, c)
            elif kind == "conv_in":
                nb, H, Wd, c = h.shape
                col = ops.im2col3x3(h, 64)
                _, o = ops.gemm(col, p["w"], bias=p["b"], want_f32=True, rows_per_sample=H * Wd, want_stats=True, stats_group=self._sg)
                h = o.view(nb, H, Wd, p["cout"])
        return h

    # ------------------------------------------------------------------ forward
    def _forward_impl(self, x, t, kvs):
        """x NCHW fp32, t fp32 [nb], kvs from context_kv -> eps NCHW fp32. Pure kernel sequence (graph-capturable)."""
        nb, _, H, Wd = x.shape
        if self._arena is None:
            self._arena = ops.StatsArena(x.device)
        self._arena.reset()          # one memset for all fused GroupNorm statistics of this evaluation
        ops.ARENA = self._arena
        try:
            return self._forward_body(x, t, kvs)
        finally:
            ops.ARENA = None

    def _forward_body(self, x, t, kvs):
        nb, _, H, Wd = x.shape
        # The FiLM chain (timestep embedding -> time_embed MLP -> all emb_layers, three weight-streaming launches, ~37 us)
        # depends on t only: it runs on a side stream next to nchw->nhwc / conv_in and joins before the first ResBlock.
        cur = torch.cuda.current_stream()
        if self._side is None:
            self._side = torch.cuda.Stream()
        side = self._side
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            film = self._film(t)
        film.record_stream(cur)
        h, _ = ops.nchw_to_nhwc(x)
        W = self.W
        hs = []
        st_idx = [0]
        joined = False
        for bi, layers in enumerate(W["input"]):
            if not joined and any(kind != "conv_in" for kind, _ in layers):
                cur.wait_stream(side)
                joined = True
            nxt = W["input"][bi + 1] if bi + 1 < len(W["input"]) else None
            h = self._run_layers(layers, h, None, film, kvs, st_idx, emit_f16=bool(nxt) and nxt[0][0] == "down")
            hs.append(h)
        if not joined:
            cur.wait_stream(side)
        h = self._run_layers(W["middle"], h, None, film, kvs, st_idx)
        for layers in W["output"]:
            h = self._run_layers(layers, h, hs.pop(), film, kvs, st_idx)
        hn, _, hn_lo, _ = ops.groupnorm(h, *W["gn_out"], eps=1e-5, silu=True, want_lo=True)
        _, o = ops.gemm(hn, W["w_out"], a1=hn_lo, a2=hn, taps=9, bias=W["b_out"], want_f32=True)
        return ops.nhwc_to_nchw(o.view(nb, H, Wd, self.out_channels))

    def _graph_for(self, shape, kvs):
        """Capture one UNet evaluation (~400 kernels) as a CUDA graph with static x / t / eps / K,V buffers."""
        g = self._graphs.get(shape)
        if g is None:
            dev = self.W["device"]
            sx = torch.zeros(shape, dtype=torch.float32, device=dev)
            st = torch.zeros((shape[0],), dtype=torch.float32, device=dev)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):      # warm-up outside capture: cudaFuncSetAttribute, allocator pools,
                ops.AUTOTUNE = self.autotune   # and one-time (block_n, split-K) selection per GEMM problem
                try:
                    self._forward_impl(sx, st, kvs)
                finally:
                    ops.AUTOTUNE = False
                self._forward_impl(sx, st, kvs)
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            n0 = ops.launch_count()
            with torch.cuda.graph(graph):
                out = self._forward_impl(sx, st, kvs)
            g = {"graph": graph, "x": sx, "t": st, "out": out, "launches": ops.launch_count() - n0, "kvs": kvs}
            self._graphs[shape] = g
        return g

    # ------------------------------------------------------------------ handle-level C entry (include/sdb200.h)
    @torch.no_grad()
    def c_handle(self, shape, context):
        """Build the C-side handle of one guided evaluation for latents of `shape` = (n, c, h, w) and the given context:
        walks the model once between sdb_plan_begin / sdb_plan_end (every launch is recorded with its arguments; the
        pass doubles as warm-up), then wraps the plan and its static x / t / eps buffers in an sdb_unet. Afterwards
        `sdb_unet_forward(handle, x, t, eps, stream)` and `sdb_sample_plms` run without any Python on the hot path.
        All intermediates of the recorded pass live in a private memory pool owned by the returned object."""
        import ctypes as C
        from . import lib as _l
        lib = _l.load()
        dev = self.W["device"]
        kvs = self.set_context(context)
        x = torch.zeros(shape, dtype=torch.float32, device=dev)
        t = torch.zeros((shape[0],), dtype=torch.float32, device=dev)
        ops.AUTOTUNE = self.autotune
        try:
            self._forward_impl(x, t, kvs)       # (block_n, split-K) selection happens outside the recording
        finally:
            ops.AUTOTUNE = False
        torch.cuda.synchronize()
        pool = torch.cuda.MemPool()
        plan = C.c_void_p()
        with torch.cuda.use_mem_pool(pool):
            _l.check(lib.sdb_plan_begin(C.byref(plan)), "sdb_plan_begin")
            try:
                eps = self._forward_impl(x, t, kvs)
            finally:
                _l.check(lib.sdb_plan_end(plan), "sdb_plan_end")
        torch.cuda.synchronize()
        h = C.c_void_p()
        _l.check(lib.sdb_unet_create(plan, C.c_void_p(x.data_ptr()), C.c_void_p(t.data_ptr()), C.c_void_p(eps.data_ptr()),
                                     shape[0], shape[1], eps.shape[1], shape[2], shape[3], C.byref(h)), "sdb_unet_create")
        return CUNet(h, plan, pool, (x, t, eps, kvs, context), int(lib.sdb_plan_size(plan)))

    @torch.no_grad()
    def forward(self, x, timesteps=None, context=None, y=None, **kwargs):
        assert y is None, "must specify y if and only if the model is class-conditional"
        assert self.W is not None, "weights not loaded (load_state_dict / load_weights, then .cuda())"
        if not x.is_cuda:
            raise RuntimeError("sdb200.UNetModel runs on CUDA (sm_100a) only; there is no CPU fallback")
        assert x.dim() == 4 and x.shape[1] == self.in_channels
        assert context is not None and context.shape[0] == x.shape[0] and context.shape[2] == self.context_dim
        nb, _, H, Wd = x.shape
        lv = len(self.cfg["channel_mult"]) - 1
        assert H % (1 << lv) == 0 and Wd % (1 << lv) == 0, "latent size must be divisible by 2^(levels-1)"
        cached = self._context_cached(context)
        if self.use_cuda_graph:
            if not cached:
                self.set_context(context)
            g = self._graph_for(tuple(x.shape), self._ctx_kv)
            assert g["kvs"] is self._ctx_kv or all(a[0].data_ptr() == b[0].data_ptr() for a, b in zip(g["kvs"], self._ctx_kv))
            if x.data_ptr() != g["x"].data_ptr():
                g["x"].copy_(x)
            g["t"].copy_(timesteps)
            g["graph"].replay()
            ops.add_graph_launches(g["launches"])
            # a fresh tensor, as the reference returns: callers may keep eps across evaluations (the reference's PLMS
            # history does when guidance is off, plms.py:159-162), the graph's static output buffer is overwritten
            return g["out"].clone() if x.dtype == torch.float32 else g["out"].to(x.dtype)
        kvs = self._ctx_kv if cached else self.context_kv(context)
        t = timesteps.to(torch.float32).contiguous()
        eps = self._forward_impl(x.contiguous().float(), t, kvs)
        return eps.to(x.dtype)


class CUNet:
    """Owner of an sdb_unet handle (include/sdb200.h): the C plan, its CUDA graph and the memory pool holding every
    intermediate buffer of the recorded evaluation."""

    def __init__(self, handle, plan, pool, keep, n_launches):
        self.handle, self.plan, self.pool, self.keep, self.n_launches = handle, plan, pool, keep, n_launches
        self.x, self.t, self.eps = keep[0], keep[1], keep[2]

    def forward(self, x, t, out=None):
        """eps = UNet(x, t) through sdb_unet_forward on the current stream (x, t: fp32 cuda tensors)."""
        import ctypes as C
        from . import lib as _l
        lib = _l.load()
        if out is None:
            out = torch.empty_like(self.eps)
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        _l.check(lib.sdb_unet_forward(self.handle, C.c_void_p(x.data_ptr()), C.c_void_p(t.data_ptr()),
                                      C.c_void_p(out.data_ptr()), st), "sdb_unet_forward")
        return out

    def sample_plms(self, x_T, sampler, scale, guided=True):
        """Whole PLMS trajectory in C (sdb_sample_plms) with the schedule of an sdb200 PLMSSampler on which
        make_schedule() has been called. Returns (x_0 latent, pred_x0)."""
        import ctypes as C
        import numpy as np
        from . import lib as _l
        lib = _l.load()
        b = x_T.shape[0]
        rep = 2 if guided else 1
        per = x_T.numel()
        work = torch.empty((5 + 2 * rep) * per, dtype=torch.float32, device=x_T.device)
        x_out, p0 = torch.empty_like(x_T), torch.empty_like(x_T)
        arr = lambda a: np.ascontiguousarray(np.asarray(a, dtype=np.float32))
        ts, al, ap = arr(sampler.ddim_timesteps), arr(sampler.ddim_alphas), arr(sampler.ddim_alphas_prev)
        sq, sg = arr(sampler.ddim_sqrt_one_minus_alphas), arr(sampler.ddim_sigmas)
        fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))
        d = _l.PlmsDesc()
        d.unet, d.x, d.x_out, d.pred_x0_out, d.work = self.handle, x_T.data_ptr(), x_out.data_ptr(), p0.data_ptr(), work.data_ptr()
        d.batch, d.n_steps, d.guided, d.scale = b, len(ts), 1 if guided else 0, float(scale)
        d.timesteps, d.alphas, d.alphas_prev, d.sqrt_one_minus_alphas, d.sigmas = fp(ts), fp(al), fp(ap), fp(sq), fp(sg)
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        _l.check(lib.sdb_sample_plms(C.byref(d), st), "sdb_sample_plms")
        torch.cuda.current_stream().synchronize()   # the host schedule arrays and `work` must outlive the enqueued work
        return x_out, p0

    def close(self):
        from . import lib as _l
        if self.handle is not None:
            lib = _l.load()
            lib.sdb_unet_destroy(self.handle)
            lib.sdb_plan_destroy(self.plan)
            self.handle = self.plan = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
