"""Parity at BASELINE.json sizes against fixtures made by the UNMODIFIED reference (oracle/make_golden.py fullsize):
SD-v1 UNet at the C5 latent (2,4,96,96) and at C1 with a second weight seed, the bench path (CUDA graph + autotuned
tiles) against the C1 golden, SD-v1 VAE decode / encode at 64x64 (512^2) and 96x96 (768^2) latents, and the C3 batch
(N_s = 64) against its own N_s = 2 evaluation. Tolerances are written here and the measured values are printed."""
import pytest
import torch

from helpers import CFGS, golden, rel_l2, weights

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]
TOL_EPS = 1e-3    # north_star: eps within 1e-3 rel-L2 of the reference (fp16 operands, fp32 accumulate)
TOL_VAE = 2e-3    # ~30 conv layers with fp16 operands; same bound as the small-size VAE tests


def _gen(shape, seed):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed))


def _sub(t, stride=4, off=1):
    return t[..., off::stride, off::stride]


@pytest.mark.parametrize("idx", range(2))
def test_unet_fullsize_vs_reference(cuda_dev, idx):
    import sdb200
    case = golden("fullsize_unet.pt")[idx]
    m = sdb200.UNetModel(**CFGS["unet"]["sdv1"]).load_weights(weights("unet", "sdv1", case["seed"]), cuda_dev)
    x = _gen(case["x_shape"], case["x_seed"])
    ctx = _gen((case["x_shape"][0], 77, 768), case["ctx_seed"])
    eps = m(x.to(cuda_dev), case["t"].to(cuda_dev), context=ctx.to(cuda_dev))
    err = rel_l2(eps, case["eps"])
    print(f"unet sdv1 weight-seed {case['seed']} {tuple(case['x_shape'])}: eps rel-L2 {err:.3e} (tol {TOL_EPS})")
    assert eps.shape == case["eps"].shape and err < TOL_EPS, err


def test_unet_graph_autotune_path_vs_reference_c1(cuda_dev):
    """The path bench.py times (CUDA graph replay, measured tile choice) against the reference's C1 golden."""
    import sdb200
    case = golden("unet.pt")[3]
    assert tuple(case["x"].shape) == (2, 4, 64, 64) and case["cfg"] == "sdv1"
    m = sdb200.UNetModel(**CFGS["unet"]["sdv1"]).load_weights(weights("unet", "sdv1", case["seed"]), cuda_dev)
    m.use_cuda_graph = True
    x, t, ctx = case["x"].to(cuda_dev), case["t"].to(cuda_dev), case["ctx"].to(cuda_dev)
    first = m(x, t, context=ctx).clone()      # autotune + capture + first replay
    again = m(x, t, context=ctx).clone()      # pure replay
    e1, e2 = rel_l2(first, case["eps"]), rel_l2(again, case["eps"])
    print(f"unet sdv1 C1 graph+autotune: eps rel-L2 {e1:.3e} / replay {e2:.3e} (tol {TOL_EPS})")
    assert e1 < TOL_EPS and e2 < TOL_EPS


def test_unet_c3_batch_rows_equal_their_ns2_evaluation(cuda_dev):
    """C3 (batch 32 -> N_s = 64): every sample of the big batch equals the same sample evaluated at N_s = 2
    (different tile shapes / split-K change the fp32 summation order, which flips fp16 roundings of intermediate
    operands here and there: agreement to a fraction of the parity tolerance, printed)."""
    import sdb200
    m = sdb200.UNetModel(**CFGS["unet"]["sdv1"]).load_weights(weights("unet", "sdv1", 11), cuda_dev)
    x2 = _gen((2, 4, 64, 64), 120).to(cuda_dev)
    c2 = _gen((2, 77, 768), 121).to(cuda_dev)
    t2 = torch.tensor([981, 981], device=cuda_dev)
    small = m(x2, t2, context=c2)
    big = m(x2.repeat(32, 1, 1, 1), t2.repeat(32), context=c2.repeat(32, 1, 1))
    assert big.shape == (64, 4, 64, 64)
    worst = max(rel_l2(big[i:i + 2], small) for i in range(0, 64, 2))
    print(f"unet sdv1 N_s=64 rows vs N_s=2: worst rel-L2 {worst:.3e}")
    assert worst < 7e-4


@pytest.mark.parametrize("idx", range(2))
def test_vae_fullsize_vs_reference(cuda_dev, idx):
    import sdb200
    case = golden(f"fullsize_vae_{(64, 96)[idx]}.pt")
    lat = case["latent"]
    vae = sdb200.AutoencoderKL(**CFGS["vae"]["sdv1"]).load_weights(weights("vae", "sdv1", case["seed"]), cuda_dev)
    z = _gen((1, 4, lat, lat), case["z_seed"])
    dec = vae.decode(z.to(cuda_dev))
    assert dec.shape == (1, 3, 8 * lat, 8 * lat)
    e_sub = rel_l2(_sub(dec), case["dec_sub"])
    e_crop = rel_l2(dec[..., 100:164, 200:264], case["dec_crop"])
    norm = float(dec.double().norm())
    print(f"vae sdv1 decode {lat}x{lat} -> {8 * lat}^2: rel-L2 {e_sub:.3e} (1/16 pixel sample) {e_crop:.3e} (64x64 crop); "
          f"|dec| {norm:.3f} vs {case['dec_norm']:.3f} (tol {TOL_VAE})")
    assert e_sub < TOL_VAE and e_crop < 2 * TOL_VAE and abs(norm / case["dec_norm"] - 1) < 1e-3
    img = _gen((1, 3, 8 * lat, 8 * lat), case["img_seed"]).clamp(-1, 1)
    post = vae.encode(img.to(cuda_dev))
    mean, logvar = case["moments"][:, :4], case["moments"][:, 4:].clamp(-30.0, 20.0)
    e_mean, e_lv = rel_l2(post.mean, mean), rel_l2(post.logvar, logvar)
    print(f"vae sdv1 encode {8 * lat}^2: mean {e_mean:.3e} logvar {e_lv:.3e}")
    assert e_mean < TOL_VAE and e_lv < TOL_VAE
