"""ORACLE tooling: generate tests/golden/*.pt by running the UNMODIFIED reference (/root/reference) on CPU fp32.

Run in the build container:  python oracle/make_golden.py
Inputs are seeded; weights come from stable-diffusion_b200/arch.random_state_dict (seeded, every tensor drawn —
the reference's zero_module init would make eps identically 0), loaded with load_state_dict(strict=True) into the
reference modules. Only inputs + reference outputs are stored (weights are regenerated from the seed by the tests).
The script also evaluates oracle/ldm_oracle.py against every vector it writes and prints the error.
"""
from __future__ import annotations

import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import ldm_oracle as O  # noqa: E402
import ref_harness as R  # noqa: E402
import sdb200  # noqa: E402,F401
from sdb200 import arch  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
UNET_SEED, VAE_SEED, CLIP_SEED, SAFETY_SEED = 11, 12, 13, 14


def rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


def save(name, obj):
    path = os.path.join(OUT, name)
    torch.save(obj, path)
    print(f"  wrote {name} ({os.path.getsize(path) / 1024:.0f} KiB)")


def gen(shape, seed, scale=1.0):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed)) * scale


def drawn(kind, shape, seed):
    """A seeded input stored as its draw (no file over 1 MB): tests/helpers.golden() draws it again, bit for bit."""
    return {kind: tuple(shape), "seed": seed}


@torch.no_grad()
def unet_goldens():
    cases = []
    for tag, cfg, shapes in (
        ("tiny", arch.TINY_UNET, [((2, 4, 16, 16), [981, 1]), ((3, 4, 8, 8), [500, 500, 21])]),
        ("sdv1", arch.SD_V1_UNET, [((2, 4, 16, 16), [981, 981]), ((2, 4, 64, 64), [981, 981]), ((1, 4, 32, 32), [261])]),
    ):
        sd = arch.random_state_dict(arch.unet_param_shapes(cfg), UNET_SEED)
        net = R.build_unet(cfg)
        net.load_state_dict(sd, strict=True)
        for i, (xs, ts) in enumerate(shapes):
            x = gen(xs, 100 + i)
            t = torch.tensor(ts, dtype=torch.long)
            ctx = gen((xs[0], 77, cfg["context_dim"]), 200 + i)
            t0 = time.time()
            eps = net(x, t, context=ctx)
            dt = time.time() - t0
            mine = O.unet_forward(sd, x, t, ctx, num_heads=cfg["num_heads"])
            print(f"unet {tag} {xs} t={ts}: ref {dt:.1f}s  eps std {float(eps.std()):.3f} absmax {float(eps.abs().max()):.2f}"
                  f"  oracle rel-L2 {rel(mine, eps):.2e}")
            cases.append(dict(cfg=tag, x=x, t=t, ctx=drawn("randn", ctx.shape, 200 + i), eps=eps, seed=UNET_SEED))
        del net
    save("unet.pt", cases)


@torch.no_grad()
def vae_goldens():
    cases = []
    for tag, cfg, zshape, ishape in (("tiny", arch.TINY_VAE, (2, 4, 8, 8), (2, 3, 32, 32)),
                                     ("sdv1", arch.SD_V1_VAE, (1, 4, 8, 8), (1, 3, 64, 64))):
        sd = arch.random_state_dict(arch.vae_param_shapes(cfg), VAE_SEED)
        vae = R.build_vae(cfg)
        vae.load_state_dict(sd, strict=True)
        z = gen(zshape, 300)
        img = gen(ishape, 301).clamp(-1, 1)
        dec = vae.decode(z)
        post = vae.encode(img)
        moments = torch.cat([post.mean, post.logvar], 1)  # logvar already clamped (distributions.py:28)
        raw_moments = vae.quant_conv(vae.encoder(img))
        print(f"vae {tag}: decode oracle rel {rel(O.vae_decode(sd, z), dec):.2e}; "
              f"encode oracle rel {rel(O.vae_encode_moments(sd, img), raw_moments):.2e}; dec std {float(dec.std()):.3f}")
        cases.append(dict(cfg=tag, z=z, img=img, dec=dec, moments=raw_moments, mean=post.mean, logvar=post.logvar,
                          seed=VAE_SEED))
    save("vae.pt", cases)


@torch.no_grad()
def pipeline_goldens():
    """Samplers + LatentDiffusion facade of the reference on a tiny model (real apply_model / DiffusionWrapper /
    register_schedule / decode_first_stage / get_first_stage_encoding code paths)."""
    ld = R.build_latent_diffusion(arch.TINY_UNET, arch.TINY_VAE)
    usd = arch.random_state_dict(arch.unet_param_shapes(arch.TINY_UNET), UNET_SEED)
    vsd = arch.random_state_dict(arch.vae_param_shapes(arch.TINY_VAE), VAE_SEED)
    ld.model.diffusion_model.load_state_dict(usd, strict=True)
    ld.first_stage_model.load_state_dict(vsd, strict=True)
    plms, ddim = R.build_samplers(ld)
    B, shape = 2, [4, 16, 16]
    c = gen((B, 77, 64), 400)
    uc = gen((B, 77, 64), 401)
    x_T = gen((B, *shape), 402)
    out = dict(c=c, uc=uc, x_T=x_T, unet_seed=UNET_SEED, vae_seed=VAE_SEED)

    model_fn = lambda x, t, cc: O.unet_forward(usd, x, t, cc, num_heads=arch.TINY_UNET["num_heads"])
    import contextlib
    import io
    buf = io.StringIO()
    for S in (50, 10):
        preds = []
        with contextlib.redirect_stdout(buf), contextlib.redirect_stderr(buf):
            s_plms, _ = plms.sample(S=S, conditioning=c, batch_size=B, shape=shape, verbose=False,
                                    unconditional_guidance_scale=7.5, unconditional_conditioning=uc, eta=0.0,
                                    x_T=x_T, img_callback=lambda p, i: preds.append(p.clone()))
        out[f"plms{S}"] = s_plms
        out[f"plms{S}_pred_x0"] = torch.stack([preds[0], preds[1], preds[len(preds) // 2], preds[-1]])
        out[f"plms{S}_timesteps"] = torch.tensor(np.array(plms.ddim_timesteps))
        out[f"plms{S}_alphas"] = torch.as_tensor(np.array(plms.ddim_alphas, dtype=np.float64))
        out[f"plms{S}_alphas_prev"] = torch.as_tensor(np.array(plms.ddim_alphas_prev, dtype=np.float64))
        out[f"plms{S}_sqrt_one_minus_alphas"] = torch.as_tensor(np.array(plms.ddim_sqrt_one_minus_alphas, dtype=np.float64))
        out[f"plms{S}_sigmas"] = torch.as_tensor(np.array(plms.ddim_sigmas, dtype=np.float64))
        mine = O.plms_sample(model_fn, x_T, c, uc, 7.5, S=S)
        print(f"plms S={S}: sample std {float(s_plms.std()):.3f}; oracle rel {rel(mine, s_plms):.2e}")
        with contextlib.redirect_stdout(buf), contextlib.redirect_stderr(buf):
            s_ddim, _ = ddim.sample(S=S, conditioning=c, batch_size=B, shape=shape, verbose=False,
                                    unconditional_guidance_scale=7.5, unconditional_conditioning=uc, eta=0.0, x_T=x_T)
        out[f"ddim{S}"] = s_ddim
        print(f"ddim S={S}: oracle rel {rel(O.ddim_sample(model_fn, x_T, c, uc, 7.5, S=S), s_ddim):.2e}")
    # guidance off (scale 1.0 -> batch not doubled, plms.py:179-180)
    with contextlib.redirect_stdout(buf), contextlib.redirect_stderr(buf):
        s1, _ = plms.sample(S=10, conditioning=c, batch_size=B, shape=shape, verbose=False,
                            unconditional_guidance_scale=1.0, unconditional_conditioning=None, eta=0.0, x_T=x_T)
    out["plms10_noguidance"] = s1
    print(f"plms S=10 no guidance: oracle rel {rel(O.plms_sample(model_fn, x_T, c, None, 1.0, S=10), s1):.2e}")
    # img2img: encode_first_stage -> get_first_stage_encoding (samples!) -> stochastic_encode -> decode (img2img.py:235-264)
    img = gen((B, 3, 32, 32), 403).clamp(-1, 1)
    torch.manual_seed(1234)
    z0 = ld.get_first_stage_encoding(ld.encode_first_stage(img))
    torch.manual_seed(1234)
    enc_noise = torch.randn(z0.shape)  # the draw DiagonalGaussianDistribution.sample made (distributions.py:36)
    with contextlib.redirect_stdout(buf), contextlib.redirect_stderr(buf):
        ddim.make_schedule(ddim_num_steps=50, ddim_eta=0.0, verbose=False)
    t_enc = 37
    se_noise = gen(z0.shape, 404)
    z_enc = ddim.stochastic_encode(z0, torch.tensor([t_enc] * B), noise=se_noise)
    with contextlib.redirect_stdout(buf), contextlib.redirect_stderr(buf):
        z_dec = ddim.decode(z_enc, c, t_enc, unconditional_guidance_scale=5.0, unconditional_conditioning=uc)
    x_dec = ld.decode_first_stage(z_dec)
    out.update(img=img, enc_noise=enc_noise, z0=z0, se_noise=se_noise, z_enc=z_enc, t_enc=t_enc, z_dec=z_dec, x_dec=x_dec)
    mz0 = O.get_first_stage_encoding(O.vae_encode_moments(vsd, img), enc_noise)
    mzenc = O.stochastic_encode(mz0, t_enc, se_noise)
    mzdec = O.ddim_sample(model_fn, mzenc, c, uc, 5.0, S=50, t_start=t_enc)
    print(f"img2img: z0 rel {rel(mz0, z0):.2e}; z_enc rel {rel(mzenc, z_enc):.2e}; z_dec rel {rel(mzdec, z_dec):.2e}; "
          f"x_dec rel {rel(O.decode_first_stage(vsd, mzdec), x_dec):.2e}")
    # apply_model facade (ddpm.py:891-992 plain path)
    t = torch.tensor([981, 21])
    out["apply_model_t"] = t
    out["apply_model_eps"] = ld.apply_model(x_T, t, c)
    # schedule buffers (ddpm.py:117-169)
    for k in ("betas", "alphas_cumprod", "alphas_cumprod_prev", "sqrt_alphas_cumprod", "sqrt_one_minus_alphas_cumprod"):
        out["sched_" + k] = getattr(ld, k).clone()
    save("pipeline_tiny.pt", out)


@torch.no_grad()
def samplers_ext_goldens():
    """SURVEY 8(f) rows on the tiny model, run by the reference's own code: DPMSolverSampler
    (dpm_solver/sampler.py + dpm_solver.py, multistep order 2, data prediction) and the mask (inpainting) branch
    of PLMSSampler / DDIMSampler (plms.py:147-150, ddim.py:144-147) with the q_sample draws recorded."""
    import contextlib
    import io
    ld = R.build_latent_diffusion(arch.TINY_UNET, arch.TINY_VAE)
    usd = arch.random_state_dict(arch.unet_param_shapes(arch.TINY_UNET), UNET_SEED)
    ld.model.diffusion_model.load_state_dict(usd, strict=True)
    plms, ddim = R.build_samplers(ld)
    from ldm.models.diffusion.dpm_solver import DPMSolverSampler
    DPMSolverSampler.register_buffer = lambda s, n, a: setattr(s, n, a)
    dpm = DPMSolverSampler(ld)
    B, shape = 2, [4, 16, 16]
    c, uc, x_T = gen((B, 77, 64), 400), gen((B, 77, 64), 401), gen((B, *shape), 402)
    out = dict(c=c, uc=uc, x_T=x_T, unet_seed=UNET_SEED)
    model_fn = lambda x, t, cc: O.unet_forward(usd, x, t, cc, num_heads=arch.TINY_UNET["num_heads"])
    buf = io.StringIO()
    for S, scale in ((20, 7.5), (10, 7.5), (15, 1.0)):
        with contextlib.redirect_stdout(buf), contextlib.redirect_stderr(buf):
            s_ref, _ = dpm.sample(S=S, conditioning=c, batch_size=B, shape=shape, verbose=False,
                                  unconditional_guidance_scale=scale,
                                  unconditional_conditioning=uc if scale != 1.0 else None, eta=0.0, x_T=x_T)
        out[f"dpm{S}_s{scale}"] = s_ref
        mine = O.dpm_solver_sample(model_fn, x_T, c, uc if scale != 1.0 else None, scale, S=S)
        print(f"dpm-solver S={S} scale={scale}: sample std {float(s_ref.std()):.3f}; oracle rel {rel(mine, s_ref):.2e}")
    # inpainting: mask (B,1,H,W) of 0/1 blocks, x0 = the latent to keep where mask == 1
    mask = (gen((B, 1, 16, 16), 410) > 0).float()
    x0 = gen((B, *shape), 411)
    out.update(mask=mask, x0=x0)
    real_randn_like = torch.randn_like
    for name, smp, fn in (("plms", plms, O.masked_plms_sample), ("ddim", ddim, O.masked_ddim_sample)):
        draws = []

        def rec_randn_like(t, *a, **k):
            r = real_randn_like(t, *a, **k)
            draws.append(r.clone())
            return r
        torch.manual_seed(77)
        torch.randn_like = rec_randn_like
        try:
            with contextlib.redirect_stdout(buf), contextlib.redirect_stderr(buf):
                s_ref, _ = smp.sample(S=10, conditioning=c, batch_size=B, shape=shape, verbose=False,
                                      unconditional_guidance_scale=7.5, unconditional_conditioning=uc, eta=0.0,
                                      x_T=x_T, mask=mask, x0=x0)
        finally:
            torch.randn_like = real_randn_like
        assert len(draws) == 10, len(draws)
        out[f"masked_{name}10"] = s_ref
        out[f"masked_{name}10_qnoise"] = torch.stack(draws)
        mine = fn(model_fn, x_T, c, uc, 7.5, mask, x0, draws, S=10)
        print(f"masked {name} S=10: oracle rel {rel(mine, s_ref):.2e}")
    save("samplers_ext.pt", out)


@torch.no_grad()
def clip_goldens():
    """Third-party arithmetic (transformers CLIPTextModel): pinned against the installed transformers, random weights."""
    from transformers import CLIPTextConfig, CLIPTextModel
    cases = []
    for tag, cfg in (("tiny", arch.TINY_CLIP), ("sdv1", arch.SD_V1_CLIP)):
        hf_cfg = CLIPTextConfig(vocab_size=cfg["vocab_size"], hidden_size=cfg["hidden_size"],
                                intermediate_size=cfg["intermediate_size"], num_hidden_layers=cfg["num_hidden_layers"],
                                num_attention_heads=cfg["num_attention_heads"],
                                max_position_embeddings=cfg["max_position_embeddings"], hidden_act="quick_gelu",
                                layer_norm_eps=cfg["layer_norm_eps"], bos_token_id=cfg["vocab_size"] - 2,
                                eos_token_id=cfg["vocab_size"] - 1, pad_token_id=cfg["vocab_size"] - 1)
        model = CLIPTextModel(hf_cfg).eval()
        sd = arch.random_state_dict(arch.clip_param_shapes(cfg), CLIP_SEED)
        missing, unexpected = model.load_state_dict(sd, strict=False)
        assert not unexpected and all("position_ids" in m for m in missing), (missing, unexpected)
        g = torch.Generator().manual_seed(500)
        ids = torch.randint(0, cfg["vocab_size"] - 2, (2, 77), generator=g)
        ids[:, 0] = cfg["vocab_size"] - 2          # BOS
        ids[0, 9:] = cfg["vocab_size"] - 1         # EOS + pad (max_length padding, modules.py:153-154)
        ids[1, 30:] = cfg["vocab_size"] - 1
        z = model(input_ids=ids).last_hidden_state
        mine = O.clip_text(sd, ids, cfg["num_attention_heads"], cfg["layer_norm_eps"])
        print(f"clip {tag}: z std {float(z.std()):.3f}; oracle rel {rel(mine, z):.2e}")
        cases.append(dict(cfg=tag, ids=ids, z=z, seed=CLIP_SEED))
    save("clip.pt", cases)


def safety_goldens():
    """Third-party arithmetic (CLIP vision tower + projection): pinned against the installed transformers
    CLIPVisionModelWithProjection on random weights; preprocessing against PIL through the oracle."""
    from transformers import CLIPVisionConfig, CLIPVisionModelWithProjection
    cases = []
    for tag, cfg in (("tiny", arch.TINY_SAFETY), ("sdv1", arch.SD_V1_SAFETY)):
        hf_cfg = CLIPVisionConfig(hidden_size=cfg["hidden_size"], intermediate_size=cfg["intermediate_size"],
                                  num_hidden_layers=cfg["num_hidden_layers"], num_attention_heads=cfg["num_attention_heads"],
                                  image_size=cfg["image_size"], patch_size=cfg["patch_size"],
                                  projection_dim=cfg["projection_dim"], hidden_act="quick_gelu",
                                  layer_norm_eps=cfg["layer_norm_eps"])
        model = CLIPVisionModelWithProjection(hf_cfg).eval()
        sd = arch.random_state_dict(arch.safety_param_shapes(cfg), SAFETY_SEED)
        hf_sd = {k[len("vision_model."):]: v for k, v in sd.items() if k.startswith("vision_model.")}
        hf_sd["visual_projection.weight"] = sd["visual_projection.weight"]
        missing, unexpected = model.load_state_dict(hf_sd, strict=False)
        assert not unexpected and all("position_ids" in m for m in missing), (missing, unexpected)
        g = torch.Generator().manual_seed(600)
        # a smooth-ish random image in [0, 1] at twice the tower's input size, through the real preprocessing
        img = torch.rand(2, cfg["image_size"] * 2 + 6, cfg["image_size"] * 2, 3, generator=g)
        pix = O.clip_image_preprocess(img.numpy(), size=cfg["image_size"])
        with torch.no_grad():
            emb = model(pixel_values=pix).image_embeds
        mine = O.clip_vision_embeds(sd, pix, cfg["num_attention_heads"], cfg["layer_norm_eps"])
        print(f"safety {tag}: embeds std {float(emb.std()):.3f}; oracle rel {rel(mine, emb):.2e}")
        images = drawn("rand", img.shape, 600) if tag == "tiny" else None
        cases.append(dict(cfg=tag, images=images, pixel_values=pix.half() if tag != "tiny" else pix,
                          image_embeds=emb, seed=SAFETY_SEED))   # (sdv1: fp16 pixels keep the fixture small; the
        if tag != "tiny":                                          #  embeds below are those OF the rounded pixels)
            with torch.no_grad():
                cases[-1]["image_embeds"] = model(pixel_values=pix.half().float()).image_embeds
    save("safety.pt", cases)


def _sub(t, stride=4, off=1):
    """Strided pixel subset of an NCHW image (full-size decodes are megabytes; rel-L2 over a regular 1/16 sample of the
    pixels plus the whole-tensor norm pins the same arithmetic)."""
    return t[..., off::stride, off::stride].contiguous()


@torch.no_grad()
def fullsize_goldens():
    """BASELINE-size fixtures from the UNMODIFIED reference (VERDICT r01 item 2): SD-v1 UNet at the C5 latent
    (2,4,96,96), C1 (2,4,64,64) with a SECOND weight seed, and the SD-v1 VAE at the sizes the benchmarks decode /
    encode (64x64 -> 512^2 and 96x96 -> 768^2). Inputs are regenerated from the stored seeds by the tests."""
    out = dict(unet=[], vae=[])
    cfg = arch.SD_V1_UNET
    for wseed, xs, ts, xseed in ((UNET_SEED, (2, 4, 96, 96), [981, 981], 110), (21, (2, 4, 64, 64), [501, 21], 111)):
        sd = arch.random_state_dict(arch.unet_param_shapes(cfg), wseed)
        net = R.build_unet(cfg)
        net.load_state_dict(sd, strict=True)
        x = gen(xs, xseed)
        t = torch.tensor(ts, dtype=torch.long)
        ctx = gen((xs[0], 77, cfg["context_dim"]), xseed + 100)
        t0 = time.time()
        eps = net(x, t, context=ctx)
        dt = time.time() - t0
        mine = O.unet_forward(sd, x, t, ctx, num_heads=cfg["num_heads"])
        print(f"unet sdv1 seed {wseed} {xs} t={ts}: ref {dt:.1f}s eps std {float(eps.std()):.3f}  oracle rel-L2 {rel(mine, eps):.2e}")
        out["unet"].append(dict(cfg="sdv1", seed=wseed, x_shape=xs, x_seed=xseed, ctx_seed=xseed + 100, t=t, eps=eps))
        del net, sd
    vcfg = arch.SD_V1_VAE
    sd = arch.random_state_dict(arch.vae_param_shapes(vcfg), VAE_SEED)
    vae = R.build_vae(vcfg)
    vae.load_state_dict(sd, strict=True)
    for lat, zseed in ((64, 310), (96, 311)):
        z = gen((1, 4, lat, lat), zseed)
        img = gen((1, 3, 8 * lat, 8 * lat), zseed + 10).clamp(-1, 1)
        t0 = time.time()
        dec = vae.decode(z)
        raw_moments = vae.quant_conv(vae.encoder(img))
        dt = time.time() - t0
        o_dec = O.vae_decode(sd, z)
        o_mom = O.vae_encode_moments(sd, img)
        print(f"vae sdv1 latent {lat}: ref {dt:.1f}s; decode oracle rel {rel(o_dec, dec):.2e}; encode oracle rel "
              f"{rel(o_mom, raw_moments):.2e}; dec std {float(dec.std()):.3f}")
        out["vae"].append(dict(cfg="sdv1", seed=VAE_SEED, latent=lat, z_seed=zseed, img_seed=zseed + 10,
                               dec_sub=_sub(dec), dec_norm=float(dec.double().norm()), dec_mean=float(dec.double().mean()),
                               dec_crop=dec[..., 100:164, 200:264].contiguous(), moments=raw_moments))
    save("fullsize_unet.pt", out["unet"])
    for v in out["vae"]:
        save(f"fullsize_vae_{v['latent']}.pt", v)


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(os.cpu_count())
    which = sys.argv[1:] or ["unet", "vae", "pipeline", "clip", "samplers_ext", "safety"]
    if "unet" in which:
        unet_goldens()
    if "vae" in which:
        vae_goldens()
    if "pipeline" in which:
        pipeline_goldens()
    if "clip" in which:
        clip_goldens()
    if "safety" in which:
        safety_goldens()
    if "samplers_ext" in which:
        samplers_ext_goldens()
    if "fullsize" in which:   # slow (minutes, ~20 GB of host memory): not part of the default set
        fullsize_goldens()
