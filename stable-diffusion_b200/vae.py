"""B200-native AutoencoderKL (SD first stage): drop-in for `ldm.models.autoencoder.AutoencoderKL`
(`encode(x) -> posterior`, `decode(z) -> image`; autoencoder.py:285-333) over the VAE Encoder/Decoder of
ldm/modules/diffusionmodules/model.py:368-568. State-dict keys unchanged (`encoder.*`, `decoder.*`, `quant_conv.*`,
`post_quant_conv.*`). Same kernels as the UNet: tcgen05 implicit-GEMM convs, fp32 GroupNorm (eps 1e-6) + SiLU
producing the fp16 operand, fp32 residual stream. The single-head mid-block attention (c=512, N=h*w;
model.py:178-202) runs as QK^T GEMM -> fp32 row softmax -> PV GEMM per image (head dim 512 exceeds the flash
kernel's TMEM budget), with the value bias folded through proj_out (softmax rows sum to 1).
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops
from .arch import vae_param_shapes
from .unet import _pack_conv3, _pack_conv3_padk
from .util import adopt_state_dict


def _sg(c):
    """Channels per fused-statistics entry for a c-channel tensor that feeds GroupNorm(32): one entry per group."""
    return c // 32 if c % 32 == 0 and c >= 32 else 1


class DiagonalGaussianDistribution:
    """distributions.py:24-62 on device tensors: parameters NCHW = [mean | logvar]."""

    def __init__(self, moments_nhwc, nb, h, w, zc):
        self._m = moments_nhwc  # fp32 [nb*h*w, 2*zc]
        self.nb, self.h, self.w, self.zc = nb, h, w, zc
        assert zc == 4, "SD first stage has 4 latent channels"

    @property
    def parameters(self):
        return ops.nhwc_to_nchw(self._m.view(self.nb, self.h, self.w, 2 * self.zc))

    @property
    def mean(self):
        return self.parameters[:, : self.zc]

    @property
    def logvar(self):
        return torch.clamp(self.parameters[:, self.zc:], -30.0, 20.0)

    def sample(self, noise=None, scale=1.0):
        if noise is None:  # the reference draws on the CPU generator then moves (distributions.py:36)
            noise = torch.randn((self.nb, self.zc, self.h, self.w)).to(self._m.device)
        z = ops.vae_sample(self._m, noise.contiguous().float(), self.nb, self.h * self.w, scale)
        return z.view(self.nb, self.zc, self.h, self.w)

    def mode(self):
        return self.mean


class AutoencoderKL(nn.Module):
    def __init__(self, ddconfig, lossconfig=None, embed_dim=4, ckpt_path=None, ignore_keys=(), image_key="image",
                 colorize_nlabels=None, monitor=None):
        super().__init__()
        assert ddconfig["double_z"], "AutoencoderKL needs double_z"
        assert not ddconfig.get("attn_resolutions"), "SD-v1 VAE: attention only in the mid block"
        self.cfg = dict(embed_dim=embed_dim, ddconfig=dict(ddconfig))
        self.embed_dim = embed_dim
        self.shapes = vae_param_shapes(self.cfg)
        self.W = None
        self._host_sd = None

    # ------------------------------------------------------------------ weights
    def _load_from_state_dict(self, state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys,
                              error_msgs):
        sd = adopt_state_dict(self, state_dict, prefix, missing_keys, unexpected_keys, error_msgs, ignore=("loss.",))
        if sd is None:
            return
        self._host_sd = sd
        if self.W is not None:
            self.pack_weights(self.W["device"])

    def load_weights(self, sd, device):
        for k, shape in self.shapes.items():
            assert k in sd and tuple(sd[k].shape) == tuple(shape), k
        self._host_sd = {k: sd[k] for k in self.shapes}
        self.pack_weights(torch.device(device))
        return self

    def _apply(self, fn, *a, **k):
        r = super()._apply(fn, *a, **k)
        probe = fn(torch.empty(0))
        if probe.is_cuda and self._host_sd is not None and (self.W is None or self.W["device"] != probe.device):
            self.pack_weights(probe.device)
        return r

    @torch.no_grad()
    def pack_weights(self, device):
        sd = {k: v.detach().to(device=device, dtype=torch.float32) for k, v in self._host_sd.items()}
        f32 = lambda k: sd[k].contiguous()
        W = {"device": device}

        def conv3(pre):
            w = sd[pre + ".weight"]
            if w.shape[1] % 64:
                return {"w": _pack_conv3_padk(w, (9 * w.shape[1] + 63) // 64 * 64), "b": f32(pre + ".bias"), "col": True,
                        "cout": w.shape[0], "cin": w.shape[1]}
            return {"w": _pack_conv3(w), "b": f32(pre + ".bias"), "col": False, "cout": w.shape[0], "cin": w.shape[1]}

        def resnet(pre):
            r = {"gn1": (f32(pre + ".norm1.weight"), f32(pre + ".norm1.bias")), "c1": conv3(pre + ".conv1"),
                 "gn2": (f32(pre + ".norm2.weight"), f32(pre + ".norm2.bias")), "c2": conv3(pre + ".conv2")}
            if pre + ".nin_shortcut.weight" in sd:
                w = sd[pre + ".nin_shortcut.weight"]
                r["ws"], r["bs"] = w.reshape(w.shape[0], w.shape[1]).half().contiguous(), f32(pre + ".nin_shortcut.bias")
            return r

        def attn(pre):
            c = sd[pre + ".q.weight"].shape[0]
            m = lambda n: sd[f"{pre}.{n}.weight"].reshape(c, c)
            wo = m("proj_out")
            return {"c": c, "gn": (f32(pre + ".norm.weight"), f32(pre + ".norm.bias")),
                    "w_q": m("q").half().contiguous(), "b_q": f32(pre + ".q.bias"),
                    "w_k": m("k").half().contiguous(), "b_k": f32(pre + ".k.bias"),
                    "w_v": m("v").half().contiguous(), "w_o": wo.half().contiguous(),
                    # softmax rows sum to 1: P (V + 1 b_v^T) W_o^T = P V W_o^T + W_o b_v
                    "b_o": (sd[pre + ".proj_out.bias"] + wo @ sd[pre + ".v.bias"]).contiguous()}

        def levels(pre, kind):
            out = []
            lvl = 0
            while f"{pre}.{lvl}.block.0.norm1.weight" in sd:
                blocks = []
                b = 0
                while f"{pre}.{lvl}.block.{b}.norm1.weight" in sd:
                    blocks.append(resnet(f"{pre}.{lvl}.block.{b}"))
                    b += 1
                rs = conv3(f"{pre}.{lvl}.{kind}.conv") if f"{pre}.{lvl}.{kind}.conv.weight" in sd else None
                out.append({"blocks": blocks, "resample": rs})
                lvl += 1
            return out

        for side in ("encoder", "decoder"):
            W[side] = {"conv_in": conv3(side + ".conv_in"), "mid1": resnet(side + ".mid.block_1"),
                       "attn": attn(side + ".mid.attn_1"), "mid2": resnet(side + ".mid.block_2"),
                       "gn_out": (f32(side + ".norm_out.weight"), f32(side + ".norm_out.bias")),
                       "conv_out": conv3(side + ".conv_out")}
        W["encoder"]["levels"] = levels("encoder.down", "downsample")
        W["decoder"]["levels"] = levels("decoder.up", "upsample")
        W["quant_w"] = sd["quant_conv.weight"].reshape(sd["quant_conv.weight"].shape[0], -1).contiguous()
        W["quant_b"] = f32("quant_conv.bias")
        W["pq_w"] = sd["post_quant_conv.weight"].reshape(sd["post_quant_conv.weight"].shape[0], -1).contiguous()
        W["pq_b"] = f32("post_quant_conv.bias")
        self.W = W

    # ------------------------------------------------------------------ blocks
    @staticmethod
    def _conv3(c, x16=None, x32=None, **epi):
        """3x3 conv pad 1: TMA implicit GEMM when C_in % 64 == 0, else explicit im2col (3/4-channel inputs)."""
        if c["col"]:
            nb, H, Wd, _ = x32.shape
            col = ops.im2col3x3(x32, c["w"].shape[1])
            _, o = ops.gemm(col, c["w"], bias=c["b"], want_f32=True, rows_per_sample=H * Wd, want_stats=True,
                            stats_group=_sg(c["cout"]), **epi)
            return o.view(nb, H, Wd, c["cout"])
        nb, H, Wd, _ = x16.shape
        # every conv output here feeds a GroupNorm next: let the epilogue store its statistics partials
        _, o = ops.gemm(x16, c["w"], taps=9, bias=c["b"], want_f32=True, splits=-1, want_stats=True,
                        stats_group=_sg(c["cout"]), **epi)
        return o.view(nb, H, Wd, c["cout"])

    def _resnet(self, r, x):
        """ResnetBlock.forward with temb=None (model.py:121-141)."""
        nb, H, Wd, cin = x.shape
        hn, raw = ops.groupnorm(x, *r["gn1"], eps=1e-6, silu=True, want_raw="ws" in r)
        h1 = self._conv3(r["c1"], x16=hn)
        hn2, _ = ops.groupnorm(h1, *r["gn2"], eps=1e-6, silu=True)
        if "ws" in r:
            _, res = ops.gemm(raw, r["ws"], bias=r["bs"], want_f32=True)
        else:
            res = x.view(-1, cin)
        return self._conv3(r["c2"], x16=hn2, residual=res)

    def _attn(self, a, x):
        """AttnBlock.forward (model.py:178-202)."""
        nb, H, Wd, c = x.shape
        n = H * Wd
        hn, _ = ops.groupnorm(x, *a["gn"], eps=1e-6, silu=False)
        q_all, _ = ops.gemm(hn, a["w_q"], bias=a["b_q"], want_f16=True)           # [nb*n, c]
        k_all, _ = ops.gemm(hn, a["w_k"], bias=a["b_k"], want_f16=True)
        if c == 512 and n % 8 == 0:
            # d = 512 flash kernel: the N x N logits stay on the SM (sdb_attention, dpad 512); V^T for the whole batch comes
            # straight out of the tensor cores (operand roles swapped), one strided view per image
            vt, _ = ops.gemm(a["w_v"], hn.view(nb * n, c), want_f16=True, b_dynamic=True)      # [c, nb*n]
            vt3 = vt.view(c, nb, n).permute(1, 0, 2)
            o = ops.attention(q_all.view(nb, n, c), k_all.view(nb, n, c), vt3, heads=1, d=c, dpad=c, nq=n, nkv=n,
                              scale=float(int(c) ** -0.5))
            _, out = ops.gemm(o.view(-1, c), a["w_o"], bias=a["b_o"], residual=x.view(-1, c), want_f32=True,
                              rows_per_sample=n, want_stats=True, stats_group=_sg(c))
            return out.view(nb, H, Wd, c)
        # other widths (test configurations): logits through the GEMM kernel, one image at a time
        o = torch.empty((nb, n, c), dtype=torch.float16, device=x.device)
        npad = (n + 7) // 8 * 8
        for b in range(nb):
            hb = hn.view(nb, n, c)[b]
            q = q_all.view(nb, n, c)[b]
            k = k_all.view(nb, n, c)[b]
            if n % 8 == 0:
                vt, _ = ops.gemm(a["w_v"], hb, want_f16=True, b_dynamic=True)      # V^T [c, n]
            else:
                v, _ = ops.gemm(hb, a["w_v"], want_f16=True)
                vt = ops.transpose_f16(v.view(1, n, c))[0]
            _, s = ops.gemm(q, k, want_f32=True, b_dynamic=True)                   # [n, n] fp32 logits
            p = ops.softmax_rows(s, float(int(c) ** -0.5))
            if npad != n:
                raise NotImplementedError("VAE attention needs h*w % 8 == 0")
            ops.gemm(p, vt.contiguous(), out_f16=o[b], b_dynamic=True)
        _, out = ops.gemm(o.view(-1, c), a["w_o"], bias=a["b_o"], residual=x.view(-1, c), want_f32=True,
                          rows_per_sample=n, want_stats=True, stats_group=_sg(c))
        return out.view(nb, H, Wd, c)

    # ------------------------------------------------------------------ public API
    @torch.no_grad()
    def decode(self, z, scale=1.0, nhwc=False):
        """AutoencoderKL.decode (autoencoder.py:330-333) on z*scale; NCHW fp32 in / out (nhwc=True keeps the
        kernels' native NHWC output, which is what the image writer wants: txt2img.py:322)."""
        assert self.W is not None and z.is_cuda, "sdb200.AutoencoderKL runs on CUDA only (no CPU fallback)"
        W, D = self.W, self.W["decoder"]
        zh, _ = ops.nchw_to_nhwc(z.contiguous().float())
        h = ops.pointwise_small(zh, W["pq_w"], W["pq_b"], alpha=float(scale))
        h = self._conv3(D["conv_in"], x32=h)
        h = self._resnet(D["mid1"], h)
        h = self._attn(D["attn"], h)
        h = self._resnet(D["mid2"], h)
        for lvl in reversed(D["levels"]):
            for r in lvl["blocks"]:
                h = self._resnet(r, h)
            if lvl["resample"] is not None:   # Upsample: nearest 2x + conv (model.py:42-57)
                h = self._conv3(lvl["resample"], x16=ops.upsample2x(h))
        hn, _ = ops.groupnorm(h, *D["gn_out"], eps=1e-6, silu=True)
        out = self._conv3(D["conv_out"], x16=hn)
        return out if nhwc else ops.nhwc_to_nchw(out)

    @torch.no_grad()
    def encode(self, x):
        """AutoencoderKL.encode (autoencoder.py:324-328): returns the diagonal Gaussian posterior."""
        assert self.W is not None and x.is_cuda, "sdb200.AutoencoderKL runs on CUDA only (no CPU fallback)"
        W, E = self.W, self.W["encoder"]
        xh, _ = ops.nchw_to_nhwc(x.contiguous().float())
        h = self._conv3(E["conv_in"], x32=xh)
        for lvl in E["levels"]:
            for r in lvl["blocks"]:
                h = self._resnet(r, h)
            if lvl["resample"] is not None:   # Downsample: pad (0,1,0,1) + conv stride 2 pad 0 (model.py:60-79)
                # straight from the NHWC activation through strided TMA boxes (conv_shift 1 = pad right / bottom only)
                nb, H, Wd, c = h.shape
                rs = lvl["resample"]
                _, o = ops.gemm(ops.cast_f16(h), rs["w"], taps=9, conv_stride=2, conv_shift=1, bias=rs["b"], want_f32=True,
                                splits=-1, want_stats=True, stats_group=_sg(c))
                h = o.view(nb, H // 2, Wd // 2, c)
        h = self._resnet(E["mid1"], h)
        h = self._attn(E["attn"], h)
        h = self._resnet(E["mid2"], h)
        hn, _ = ops.groupnorm(h, *E["gn_out"], eps=1e-6, silu=True)
        m = self._conv3(E["conv_out"], x16=hn)
        nb, H, Wd, c2 = m.shape
        moments = ops.pointwise_small(m, W["quant_w"], W["quant_b"])
        return DiagonalGaussianDistribution(moments.view(nb * H * Wd, c2), nb, H, Wd, c2 // 2)

    def forward(self, input, sample_posterior=True):
        posterior = self.encode(input)
        z = posterior.sample() if sample_posterior else posterior.mode()
        return self.decode(z), posterior
