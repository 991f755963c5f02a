"""The oracle (oracle/ldm_oracle.py) against the golden vectors produced by the UNMODIFIED reference
(oracle/make_golden.py). CPU only. This is the pin that lets the GPU tests trust the oracle."""
import numpy as np
import pytest
import torch

from helpers import CFGS, golden, rel_l2, weights
import ldm_oracle as O


@pytest.mark.parametrize("idx", range(5))
def test_unet_oracle_matches_reference(idx):
    case = golden("unet.pt")[idx]
    if case["cfg"] == "sdv1" and case["x"].shape[-1] == 64:
        pytest.skip("C1 full-size case is covered by test_unet_c1_oracle (slow)")
    sd = weights("unet", case["cfg"], case["seed"])
    eps = O.unet_forward(sd, case["x"], case["t"], case["ctx"], num_heads=CFGS["unet"][case["cfg"]]["num_heads"])
    assert rel_l2(eps, case["eps"]) < 1e-5


@pytest.mark.slow
def test_unet_c1_oracle():
    """BASELINE config C1: (2,4,64,64) latent + (2,77,768) context, fp32 CPU."""
    case = [c for c in golden("unet.pt") if c["cfg"] == "sdv1" and c["x"].shape[-1] == 64][0]
    sd = weights("unet", "sdv1", case["seed"])
    eps = O.unet_forward(sd, case["x"], case["t"], case["ctx"])
    assert rel_l2(eps, case["eps"]) < 1e-5


@pytest.mark.parametrize("idx", range(2))
def test_vae_oracle_matches_reference(idx):
    case = golden("vae.pt")[idx]
    sd = weights("vae", case["cfg"], case["seed"])
    assert rel_l2(O.vae_decode(sd, case["z"]), case["dec"]) < 1e-5
    m = O.vae_encode_moments(sd, case["img"])
    assert rel_l2(m, case["moments"]) < 1e-5
    mean, logvar = m.chunk(2, 1)
    assert rel_l2(mean, case["mean"]) < 1e-5 and rel_l2(logvar.clamp(-30, 20), case["logvar"]) < 1e-5


@pytest.mark.parametrize("idx", range(2))
def test_clip_oracle_matches_transformers(idx):
    case = golden("clip.pt")[idx]
    cfg = CFGS["clip"][case["cfg"]]
    sd = weights("clip", case["cfg"], case["seed"])
    z = O.clip_text(sd, case["ids"], cfg["num_attention_heads"], cfg["layer_norm_eps"])
    assert rel_l2(z, case["z"]) < 1e-5


def test_schedule_tables():
    g = golden("pipeline_tiny.pt")
    sched = O.register_schedule()
    for k in ("betas", "alphas_cumprod", "alphas_cumprod_prev", "sqrt_alphas_cumprod", "sqrt_one_minus_alphas_cumprod"):
        assert torch.equal(sched[k], g["sched_" + k]), k
    assert abs(float(sched["alphas_cumprod"][0]) - 0.99915) < 1e-6
    assert abs(float(sched["alphas_cumprod"][999]) - 0.0046601) < 1e-7
    for S in (50, 10):
        sc = O.sampler_schedule(S)
        assert np.array_equal(sc["timesteps"], g[f"plms{S}_timesteps"].numpy())
        f32 = lambda t: t.to(torch.float32)
        assert torch.equal(torch.tensor(sc["alphas"]), f32(g[f"plms{S}_alphas"]))
        assert torch.equal(torch.tensor(sc["alphas_prev"]), f32(g[f"plms{S}_alphas_prev"]))
        assert torch.equal(torch.tensor(sc["sqrt_one_minus_alphas"]), f32(g[f"plms{S}_sqrt_one_minus_alphas"]))
        assert torch.equal(torch.tensor(sc["sigmas"]), f32(g[f"plms{S}_sigmas"]))
    assert list(O.make_ddim_timesteps(50)[:3]) == [1, 21, 41] and O.make_ddim_timesteps(50)[-1] == 981


def test_samplers_oracle_match_reference():
    g = golden("pipeline_tiny.pt")
    usd = weights("unet", "tiny", g["unet_seed"])
    evals = []

    def model_fn(x, t, c):
        evals.append(x.shape[0])
        return O.unet_forward(usd, x, t, c, num_heads=CFGS["unet"]["tiny"]["num_heads"])

    assert rel_l2(model_fn(g["x_T"], g["apply_model_t"], g["c"]), g["apply_model_eps"]) < 1e-5
    evals.clear()
    s = O.plms_sample(model_fn, g["x_T"], g["c"], g["uc"], 7.5, S=10)
    assert evals == [4] * 11, "PLMS makes S+1 evaluations on a CFG-doubled batch"
    assert rel_l2(s, g["plms10"]) < 1e-4
    assert rel_l2(O.ddim_sample(model_fn, g["x_T"], g["c"], g["uc"], 7.5, S=10), g["ddim10"]) < 1e-4
    evals.clear()
    assert rel_l2(O.plms_sample(model_fn, g["x_T"], g["c"], None, 1.0, S=10), g["plms10_noguidance"]) < 1e-4
    assert evals == [2] * 11, "scale 1.0 does not double the batch"


@pytest.mark.slow
def test_samplers_oracle_50_steps_and_img2img():
    g = golden("pipeline_tiny.pt")
    usd = weights("unet", "tiny", g["unet_seed"])
    vsd = weights("vae", "tiny", g["vae_seed"])
    model_fn = lambda x, t, c: O.unet_forward(usd, x, t, c, num_heads=CFGS["unet"]["tiny"]["num_heads"])
    assert rel_l2(O.plms_sample(model_fn, g["x_T"], g["c"], g["uc"], 7.5, S=50), g["plms50"]) < 1e-4
    assert rel_l2(O.ddim_sample(model_fn, g["x_T"], g["c"], g["uc"], 7.5, S=50), g["ddim50"]) < 1e-4
    z0 = O.get_first_stage_encoding(O.vae_encode_moments(vsd, g["img"]), g["enc_noise"])
    assert rel_l2(z0, g["z0"]) < 1e-5
    z_enc = O.stochastic_encode(z0, g["t_enc"], g["se_noise"])
    assert rel_l2(z_enc, g["z_enc"]) < 1e-5
    z_dec = O.ddim_sample(model_fn, z_enc, g["c"], g["uc"], 5.0, S=50, t_start=g["t_enc"])
    assert rel_l2(z_dec, g["z_dec"]) < 1e-4
    assert rel_l2(O.decode_first_stage(vsd, z_dec), g["x_dec"]) < 1e-4


def test_oracle_matches_reference_fullsize_fixtures():
    """BASELINE-size fixtures (tests/golden/fullsize_*.pt, written by the unmodified reference): the oracle reproduces the
    second-weight-seed C1 eps to fp32 round-off (bit-exactly on the host that wrote the fixtures; MKL / oneDNN pick their
    blocking and reduction order from the core count, so another host differs in the last bits: 2.4e-6 on an 8-core
    container) and the 512^2 VAE decode likewise (the 96x96 cases need ~20 GB and half a minute each; make_golden.py
    prints their oracle error when the fixtures are made)."""
    import ldm_oracle as O
    case = golden("fullsize_unet.pt")[1]
    g = lambda shape, seed: torch.randn(shape, generator=torch.Generator().manual_seed(seed))
    x, ctx = g(case["x_shape"], case["x_seed"]), g((case["x_shape"][0], 77, 768), case["ctx_seed"])
    eps = O.unet_forward(weights("unet", "sdv1", case["seed"]), x, case["t"], ctx)
    assert torch.equal(eps, case["eps"]) or rel_l2(eps, case["eps"]) < 1e-5
    v = golden("fullsize_vae_64.pt")
    dec = O.vae_decode(weights("vae", "sdv1", v["seed"]), g((1, 4, v["latent"], v["latent"]), v["z_seed"]))
    assert rel_l2(dec[..., 1::4, 1::4], v["dec_sub"]) < 5e-6 and abs(float(dec.double().norm()) / v["dec_norm"] - 1) < 1e-6
