"""B200-native safety checker: drop-in for what `scripts/txt2img.py:26-29, 88-95` builds from third-party packages -
transformers' CLIPFeatureExtractor (`safety_feature_extractor`) and diffusers' StableDiffusionSafetyChecker
(`safety_checker`): `check_safety(x_image)` -> (x_checked_image, has_nsfw_concept).

Everything runs on the GPU, on the same kernel family as the UNet: PIL's 8-bit bicubic resample restated in its own
fixed-point arithmetic (sdb_resample_u8; the coefficient tables are computed on the host as PIL's precompute_coeffs
does), normalisation, ViT patch extraction, the CLIP ViT-L/14 vision tower (fp32 LayerNorm -> fp16 operands, tcgen05
GEMMs with fused bias / quick-GELU / residual epilogues, tcgen05 attention), the visual projection and the concept
decision (sdb_safety_scores). State-dict keys are diffusers' (`vision_model.vision_model.*`, `visual_projection.weight`,
`concept_embeds`, `special_care_embeds`, `*_weights`). There is no CPU fallback.
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn as nn

from . import lib as _l
from . import ops
from .arch import CLIP_IMAGE_MEAN, CLIP_IMAGE_STD, SD_V1_SAFETY, safety_param_shapes
from .ops import ACT_QUICK_GELU, _ptr, _stream
from .util import adopt_state_dict


def _bicubic(x):
    a = -0.5
    x = abs(x)
    if x < 1.0:
        return ((a + 2.0) * x - (a + 3.0)) * x * x + 1
    if x < 2.0:
        return (((x - 5) * x + 8) * x - 4) * a
    return 0.0


def pil_resample_coeffs(in_size, out_size, support=2.0, filt=_bicubic, precision_bits=22):
    """PIL Resample.c precompute_coeffs + normalize_coeffs_8bpc: per output position the first source index, the tap
    count and the 22-bit fixed-point weights. Returns (bounds int32 [out, 2], coefs int32 [out, ksize], ksize)."""
    scale = filterscale = in_size / out_size
    if filterscale < 1.0:
        filterscale = 1.0
    sup = support * filterscale
    ksize = int(math.ceil(sup)) * 2 + 1
    bounds = np.zeros((out_size, 2), dtype=np.int32)
    coefs = np.zeros((out_size, ksize), dtype=np.int32)
    ss = 1.0 / filterscale
    for xx in range(out_size):
        center = (xx + 0.5) * scale
        xmin = int(center - sup + 0.5)
        if xmin < 0:
            xmin = 0
        xmax = int(center + sup + 0.5)
        if xmax > in_size:
            xmax = in_size
        xmax -= xmin
        k = [filt((x + xmin - center + 0.5) * ss) for x in range(xmax)]
        ww = sum(k)
        if ww != 0.0:
            k = [v / ww for v in k]
        for x, v in enumerate(k):
            coefs[xx, x] = int(-0.5 + v * (1 << precision_bits)) if v < 0 else int(0.5 + v * (1 << precision_bits))
        bounds[xx] = (xmin, xmax)
    return bounds, coefs, ksize


class CLIPImagePreprocessor:
    """CLIPFeatureExtractor (resize shorter side to `size` with PIL bicubic, centre crop, 1/255, normalise) on the GPU."""

    def __init__(self, size=224, mean=CLIP_IMAGE_MEAN, std=CLIP_IMAGE_STD):
        self.size, self.mean, self.std = size, tuple(mean), tuple(std)
        self._tables = {}

    def _table(self, in_size, out_size, device):
        key = (in_size, out_size, str(device))
        if key not in self._tables:
            b, c, k = pil_resample_coeffs(in_size, out_size)
            self._tables[key] = (torch.from_numpy(b).to(device), torch.from_numpy(c).to(device), k)
        return self._tables[key]

    @torch.no_grad()
    def __call__(self, images):
        """images: fp32 cuda [B, H, W, 3] in [0, 1] (or uint8) -> pixel_values fp32 [B, 3, size, size]."""
        if not images.is_cuda:
            raise RuntimeError("sdb200.CLIPImagePreprocessor runs on CUDA only (no CPU fallback)")
        B, H, W, _ = images.shape
        images = images.contiguous()
        lib = _l.load()
        short, long = (W, H) if W <= H else (H, W)
        new_long = int(self.size * long / short)
        nw, nh = (self.size, new_long) if W <= H else (new_long, self.size)
        src8 = images if images.dtype == torch.uint8 else None
        src32 = None if src8 is not None else images.float()
        cur_w = W
        if nw != W:   # horizontal pass first, into an 8-bit intermediate, as ImagingResample does
            bnd, cf, k = self._table(W, nw, images.device)
            tmp = torch.empty((B, H, nw, 3), dtype=torch.uint8, device=images.device)
            _l.check(lib.sdb_resample_u8(_ptr(src8), _ptr(src32), B, H, W, nw, k, _ptr(bnd), _ptr(cf), 0, 0, _ptr(tmp),
                                         _stream()), "sdb_resample_u8")
            src8, src32, cur_w = tmp, None, nw
        if nh != H:
            bnd, cf, k = self._table(H, nh, images.device)
            tmp = torch.empty((B, nh, cur_w, 3), dtype=torch.uint8, device=images.device)
            _l.check(lib.sdb_resample_u8(_ptr(src8), _ptr(src32), B, cur_w, H, nh, k, _ptr(bnd), _ptr(cf), 1, cur_w,
                                         _ptr(tmp), _stream()), "sdb_resample_u8")
            src8, src32 = tmp, None
        if src8 is None:   # no resize at all: still the numpy_to_pil rounding
            src8 = (src32 * 255).round().clamp(0, 255).to(torch.uint8)
        out = torch.empty((B, 3, self.size, self.size), dtype=torch.float32, device=images.device)
        _l.check(lib.sdb_clip_normalize(_ptr(src8), B, src8.shape[1], src8.shape[2], self.size, *self.mean, *self.std,
                                        _ptr(out), _stream()), "sdb_clip_normalize")
        return out


class _VisionModel(nn.Module):
    """Holds the `vision_model.*` keys of the checkpoint (diffusers nests a CLIPVisionModel there)."""

    def __init__(self):
        super().__init__()


class StableDiffusionSafetyChecker(nn.Module):
    def __init__(self, config=None, device="cuda"):
        super().__init__()
        self.cfg = dict(config or SD_V1_SAFETY)
        self.device = device
        self.shapes = safety_param_shapes(self.cfg)
        self.W = None
        self._host_sd = None
        self.feature_extractor = CLIPImagePreprocessor(self.cfg["image_size"])

    def _load_from_state_dict(self, state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys,
                              error_msgs):
        sd = adopt_state_dict(self, state_dict, prefix, missing_keys, unexpected_keys, error_msgs,
                              ignore=("vision_model.vision_model.embeddings.position_ids",))
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
        f16 = lambda k: sd[k].half().contiguous()
        cfg = self.cfg
        h, P = cfg["hidden_size"], cfg["patch_size"]
        v = "vision_model.vision_model"
        kpad = (3 * P * P + 63) // 64 * 64
        wp = torch.zeros((h, kpad), dtype=torch.float16, device=device)
        wp[:, : 3 * P * P] = sd[f"{v}.embeddings.patch_embedding.weight"].reshape(h, -1).half()
        pos = f32(f"{v}.embeddings.position_embedding.weight")
        W = {"device": device, "w_patch": wp, "kpad": kpad, "pos_patches": pos[1:].contiguous(),
             "cls_pos": (sd[f"{v}.embeddings.class_embedding"] + pos[0]).contiguous(),
             "ln_pre": (f32(f"{v}.pre_layrnorm.weight"), f32(f"{v}.pre_layrnorm.bias")),
             "ln_post": (f32(f"{v}.post_layernorm.weight"), f32(f"{v}.post_layernorm.bias")), "layers": []}
        for i in range(cfg["num_hidden_layers"]):
            p = f"{v}.encoder.layers.{i}"
            wo = sd[p + ".self_attn.out_proj.weight"]
            W["layers"].append({
                "ln1": (f32(p + ".layer_norm1.weight"), f32(p + ".layer_norm1.bias")),
                "ln2": (f32(p + ".layer_norm2.weight"), f32(p + ".layer_norm2.bias")),
                "w_qk": torch.cat([sd[p + ".self_attn.q_proj.weight"], sd[p + ".self_attn.k_proj.weight"]], 0).half().contiguous(),
                "b_qk": torch.cat([sd[p + ".self_attn.q_proj.bias"], sd[p + ".self_attn.k_proj.bias"]]).contiguous(),
                "w_v": f16(p + ".self_attn.v_proj.weight"),
                "w_o": wo.half().contiguous(),
                # softmax rows sum to 1: the value bias passes through the attention unchanged -> fold it through out_proj
                "b_o": (sd[p + ".self_attn.out_proj.bias"] + wo @ sd[p + ".self_attn.v_proj.bias"]).contiguous(),
                "w_fc1": f16(p + ".mlp.fc1.weight"), "b_fc1": f32(p + ".mlp.fc1.bias"),
                "w_fc2": f16(p + ".mlp.fc2.weight"), "b_fc2": f32(p + ".mlp.fc2.bias")})
        W["w_proj"] = f16("visual_projection.weight")
        W["concept"], W["special"] = f32("concept_embeds"), f32("special_care_embeds")
        W["concept_w"], W["special_w"] = f32("concept_embeds_weights"), f32("special_care_embeds_weights")
        self.W = W

    @torch.no_grad()
    def image_embeds(self, pixel_values):
        """pixel_values fp32 cuda [B, 3, S, S] -> image_embeds fp32 [B, projection_dim] (vision tower + visual_projection)."""
        assert self.W is not None and pixel_values.is_cuda, "sdb200.StableDiffusionSafetyChecker runs on CUDA only"
        W, cfg = self.W, self.cfg
        lib = _l.load()
        B = pixel_values.shape[0]
        S, P, h = cfg["image_size"], cfg["patch_size"], cfg["hidden_size"]
        heads = cfg["num_attention_heads"]
        d = h // heads
        assert d == 64, "CLIP vision heads are 64 wide"
        eps = cfg["layer_norm_eps"]
        g = S // P
        n = g * g + 1
        pix = pixel_values.contiguous().float()
        patches = torch.empty((B * g * g, W["kpad"]), dtype=torch.float16, device=pix.device)
        _l.check(lib.sdb_patchify(_ptr(pix), B, S, P, W["kpad"], _ptr(patches), _stream()), "sdb_patchify")
        x = torch.empty((B, n, h), dtype=torch.float32, device=pix.device)
        for b in range(B):   # token 0 = class + pos[0]; tokens 1.. = patch embedding + pos (residual of the GEMM)
            ops.axpby(W["cls_pos"], 1.0, 0.0, out=x[b, 0])
            ops.gemm(patches[b * g * g:(b + 1) * g * g], W["w_patch"], residual=W["pos_patches"], out_f32=x[b, 1:])
        _, x = ops.layernorm(x.view(B * n, h), *W["ln_pre"], eps=eps, want_f32=True)
        for L in W["layers"]:
            y = ops.layernorm(x, *L["ln1"], eps=eps)
            qk, _ = ops.gemm(y, L["w_qk"], bias=L["b_qk"], want_f16=True)
            v, _ = ops.gemm(y, L["w_v"], want_f16=True)
            qk3 = qk.view(B, n, 2 * h)
            vt = ops.transpose_f16(v.view(B, n, h))
            o = ops.attention(qk3[:, :, :h], qk3[:, :, h:], vt, heads=heads, d=d, dpad=d, nq=n, nkv=n, scale=d ** -0.5)
            _, x = ops.gemm(o.view(-1, h), L["w_o"], bias=L["b_o"], residual=x, want_f32=True)
            y = ops.layernorm(x, *L["ln2"], eps=eps)
            gq, _ = ops.gemm(y, L["w_fc1"], bias=L["b_fc1"], act=ACT_QUICK_GELU, want_f16=True)
            _, x = ops.gemm(gq, L["w_fc2"], bias=L["b_fc2"], residual=x, want_f32=True)
        cls = torch.empty((B, h), dtype=torch.float32, device=pix.device)
        xv = x.view(B, n, h)
        for b in range(B):
            ops.axpby(xv[b, 0], 1.0, 0.0, out=cls[b])
        _, pooled = ops.layernorm(cls, *W["ln_post"], eps=eps, want_f32=True)
        return ops.linear_small(pooled, W["w_proj"])

    @torch.no_grad()
    def forward(self, clip_input, images):
        """StableDiffusionSafetyChecker.forward: images fp32 cuda [B, H, W, 3]; flagged images are blanked in place.
        Returns (images, has_nsfw_concept list[bool])."""
        W = self.W
        lib = _l.load()
        emb = self.image_embeds(clip_input)
        B, dim = emb.shape
        ns, nc = W["special"].shape[0], W["concept"].shape[0]
        scores = torch.empty((B, ns + nc), dtype=torch.float32, device=emb.device)
        flagged = torch.empty((B,), dtype=torch.int32, device=emb.device)
        _l.check(lib.sdb_safety_scores(_ptr(emb), B, dim, _ptr(W["special"]), _ptr(W["special_w"]), ns, _ptr(W["concept"]),
                                       _ptr(W["concept_w"]), nc, _ptr(scores), _ptr(flagged), _stream()), "sdb_safety_scores")
        if images is not None:
            assert images.is_cuda and images.dtype == torch.float32 and images.is_contiguous()
            _l.check(lib.sdb_blank_flagged(_ptr(images), images[0].numel(), B, _ptr(flagged), _stream()), "sdb_blank_flagged")
        self.last_scores = scores
        return images, [bool(v) for v in flagged.cpu().tolist()]

    @torch.no_grad()
    def check_safety(self, x_image, replacement=None):
        """scripts/txt2img.py:88-95: x_image fp32 [B, H, W, 3] in [0, 1] on the GPU. Flagged images are replaced by
        `replacement` ([H, W, 3], the script's assets/rick.jpeg resized) when given, else left blank."""
        clip_input = self.feature_extractor(x_image)
        x_checked, has = self.forward(clip_input, x_image)
        if replacement is not None:
            for i, bad in enumerate(has):
                if bad and tuple(replacement.shape) == tuple(x_checked[i].shape):
                    x_checked[i].copy_(replacement)
        return x_checked, has


class WatermarkEncoder:
    """`imwatermark.WatermarkEncoder` as scripts/txt2img.py:261-264 uses it (`set_watermark('bytes', b"StableDiffusionV1")`,
    `encode(img, 'dwtDct')`), on the GPU: uint8 RGB cuda tensors [H, W, 3] or [B, H, W, 3] in, watermarked uint8 RGB out
    (the script's RGB -> BGR -> encode -> RGB round trip folded into the kernels)."""

    def __init__(self):
        self._bits = None

    def set_watermark(self, wm_type="bytes", content=b""):
        if wm_type != "bytes":
            raise NotImplementedError("only the 'bytes' watermark of scripts/txt2img.py is implemented")
        self._bits = np.unpackbits(np.frombuffer(bytes(content), dtype=np.uint8)).astype(np.uint8)
        self._dev = {}

    def encode(self, img, method="dwtDct"):
        if method != "dwtDct":
            raise NotImplementedError("only the 'dwtDct' method of scripts/txt2img.py is implemented")
        if self._bits is None or len(self._bits) == 0:
            raise RuntimeError("set_watermark() first")
        if not (img.is_cuda and img.dtype == torch.uint8):
            raise RuntimeError("sdb200.WatermarkEncoder takes uint8 CUDA tensors (no CPU fallback)")
        single = img.dim() == 3
        x = (img[None] if single else img).contiguous()
        B, H, W, _ = x.shape
        bits = self._dev.get(str(x.device))
        if bits is None:
            bits = self._dev[str(x.device)] = torch.from_numpy(self._bits).to(x.device)
        scratch = torch.empty_like(x)
        out = torch.empty_like(x)
        _l.check(_l.load().sdb_watermark_dwtdct(_ptr(x), B, H, W, _ptr(bits), int(bits.numel()), 36.0, _ptr(scratch), _ptr(out),
                                                _stream()), "sdb_watermark_dwtdct")
        return out[0] if single else out


def put_watermark(img, wm_encoder=None):
    """scripts/txt2img.py:69-74 for uint8 RGB cuda tensors."""
    return img if wm_encoder is None else wm_encoder.encode(img, "dwtDct")
