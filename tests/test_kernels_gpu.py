"""GPU unit parity of each hand-written kernel against a plain PyTorch fp32 restatement of the same op.
(Whole-model parity against the oracle lives in test_unet_gpu.py etc.)"""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(300)]


def rel_l2(a, b):
    a = a.double().flatten()
    b = b.double().flatten()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


@pytest.fixture(scope="module")
def S(cuda_dev):
    import sdb200
    return sdb200


def _rand16(shape, dev, gen, scale=1.0):
    return (torch.randn(shape, generator=gen, device="cpu") * scale).to(dev).half()


@pytest.mark.parametrize("M,N,K,bn", [
    (128, 128, 64, 128), (256, 128, 128, 128), (154, 320, 768, 0), (8192, 320, 320, 160), (1000, 96, 192, 32),
    (512, 64, 1280, 64), (384, 512, 256, 256), (128, 1280, 1280, 0), (300, 4, 320, 0),
])
def test_gemm_plain(S, cuda_dev, M, N, K, bn):
    g = torch.Generator().manual_seed(M * 7 + N)
    a = _rand16((M, K), cuda_dev, g)
    b = _rand16((N, K), cuda_dev, g, K ** -0.5)
    bias = torch.randn(N, generator=g).to(cuda_dev)
    res = torch.randn(M, N, generator=g).to(cuda_dev)
    o16, o32 = S.ops.gemm(a, b, bias=bias, residual=res, want_f16=True, want_f32=True, block_n=bn)
    torch.cuda.synchronize()
    ref = a.double() @ b.double().t() + bias + res
    assert rel_l2(o32, ref) < 1e-5, rel_l2(o32, ref)
    assert rel_l2(o16.float(), ref) < 6e-4


@pytest.mark.parametrize("nb,h,w,c,n", [
    (2, 16, 16, 64, 128), (2, 8, 8, 128, 64), (3, 8, 8, 64, 32), (1, 64, 64, 320, 320), (2, 32, 32, 640, 640),
    (1, 12, 12, 64, 64), (2, 24, 24, 128, 96), (1, 128, 128, 128, 128), (2, 64, 64, 320, 4),
])
def test_conv3x3(S, cuda_dev, nb, h, w, c, n):
    g = torch.Generator().manual_seed(nb * 131 + h + c)
    x = _rand16((nb, h, w, c), cuda_dev, g)
    wt = _rand16((n, c, 3, 3), cuda_dev, g, (9 * c) ** -0.5)
    bias = torch.randn(n, generator=g).to(cuda_dev)
    film = torch.randn(nb, n, generator=g).to(cuda_dev)
    wk = wt.permute(0, 2, 3, 1).reshape(n, 9 * c).contiguous()  # [n, (ky,kx,c)]
    _, o32 = S.ops.gemm(x, wk, taps=9, bias=bias, film=film, want_f32=True)
    torch.cuda.synchronize()
    ref = F.conv2d(x.double().permute(0, 3, 1, 2), wt.double(), bias.double(), padding=1) + film[:, :, None, None]
    ref = ref.permute(0, 2, 3, 1).reshape(nb * h * w, n)
    assert rel_l2(o32, ref) < 1e-5, rel_l2(o32, ref)


@pytest.mark.parametrize("nb,h,w,c,n,shift", [
    (2, 64, 64, 320, 320, 0), (2, 32, 32, 640, 640, 0), (2, 16, 16, 1280, 1280, 0), (1, 24, 24, 64, 96, 0),
    (1, 64, 64, 128, 128, 1), (2, 16, 16, 64, 64, 1), (1, 34, 34, 64, 32, 1),
])
def test_conv3x3_stride2_through_strided_tma(S, cuda_dev, nb, h, w, c, n, shift):
    """Downsample convs without im2col: shift 0 = symmetric zero pad 1 (openaimodel.py:149-153), shift 1 = the VAE's
    pad-right/bottom-only variant (model.py:72-76)."""
    g = torch.Generator().manual_seed(nb * 17 + h + c + shift)
    x = _rand16((nb, h, w, c), cuda_dev, g)
    wt = _rand16((n, c, 3, 3), cuda_dev, g, (9 * c) ** -0.5)
    bias = torch.randn(n, generator=g).to(cuda_dev)
    wk = wt.permute(0, 2, 3, 1).reshape(n, 9 * c).contiguous()
    _, o32 = S.ops.gemm(x, wk, taps=9, conv_stride=2, conv_shift=shift, bias=bias, want_f32=True, splits=-1)
    torch.cuda.synchronize()
    xin = x.double().permute(0, 3, 1, 2)
    if shift:
        ref = F.conv2d(F.pad(xin, (0, 1, 0, 1)), wt.double(), bias.double(), stride=2, padding=0)
    else:
        ref = F.conv2d(xin, wt.double(), bias.double(), stride=2, padding=1)
    ho, wo = ref.shape[2], ref.shape[3]
    assert o32.shape == (nb * ho * wo, n)
    ref = ref.permute(0, 2, 3, 1).reshape(nb * ho * wo, n)
    assert rel_l2(o32, ref) < 1e-5, rel_l2(o32, ref)


def test_conv3x3_concat_and_skip(S, cuda_dev):
    g = torch.Generator().manual_seed(5)
    nb, h, w, c0, c1, n = 2, 16, 16, 128, 64, 128
    x0 = _rand16((nb, h, w, c0), cuda_dev, g)
    x1 = _rand16((nb, h, w, c1), cuda_dev, g)
    wt = _rand16((n, c0 + c1, 3, 3), cuda_dev, g, (9 * (c0 + c1)) ** -0.5)
    wk = wt.permute(0, 2, 3, 1).reshape(n, -1).contiguous()
    _, o32 = S.ops.gemm(x0, wk, a1=x1, taps=9, want_f32=True)
    xc = torch.cat([x0, x1], -1).double().permute(0, 3, 1, 2)
    ref = F.conv2d(xc, wt.double(), padding=1).permute(0, 2, 3, 1).reshape(-1, n)
    assert rel_l2(o32, ref) < 1e-5
    # 1x1 skip over the concat
    w1 = _rand16((n, c0 + c1), cuda_dev, g, (c0 + c1) ** -0.5)
    _, s32 = S.ops.gemm(x0, w1, a1=x1, want_f32=True, residual=o32)
    ref2 = torch.cat([x0, x1], -1).double().reshape(-1, c0 + c1) @ w1.double().t() + ref
    assert rel_l2(s32, ref2) < 1e-5


def _check_stats(o32, nb, rps, n):
    """Per-tile statistics partials attached by gemm(want_stats=True): summed over the tile slots they must equal the
    per-(sample, channel group) sum / sum of squares of the fp32 output."""
    st, T, sg = o32._sdb_stats
    assert st.shape == (nb, T, n // sg, 2) and st.dtype == torch.float32
    got = st.double().sum(1)
    x = o32.double().view(nb, rps, n // sg, sg)
    ref = torch.stack([x.sum((1, 3)), (x * x).sum((1, 3))], -1)
    assert rel_l2(got, ref) < 1e-5, rel_l2(got, ref)


@pytest.mark.parametrize("M,N,K,bn,sg", [
    (8192, 320, 320, 160, 10), (2048, 640, 1280, 160, 10), (512, 1280, 640, 160, 10), (1000, 256, 192, 128, 4),
    (256, 512, 128, 256, 1), (4096, 320, 960, 160, 10), (384, 320, 64, 160, 2),
])
def test_gemm_cta_pair(S, cuda_dev, M, N, K, bn, sg):
    """cta_group::2: two CTAs per 256 x block_n tile, each loading half of the weight tile (odd tile counts included)."""
    g = torch.Generator().manual_seed(M + N + K)
    a = _rand16((M, K), cuda_dev, g)
    b = _rand16((N, K), cuda_dev, g, K ** -0.5)
    bias = torch.randn(N, generator=g).to(cuda_dev)
    res = torch.randn(M, N, generator=g).to(cuda_dev)
    rps = M if M % 128 == 0 else 0
    o16, o32 = S.ops.gemm(a, b, bias=bias, residual=res, want_f16=True, want_f32=True, block_n=bn, pair=2,
                          rows_per_sample=rps, want_stats=bool(rps), stats_group=sg)
    torch.cuda.synchronize()
    ref = a.double() @ b.double().t() + bias + res
    assert rel_l2(o32, ref) < 1e-5, rel_l2(o32, ref)
    assert rel_l2(o16.float(), ref) < 6e-4
    if rps:
        _check_stats(o32, 1, rps, N)


@pytest.mark.parametrize("nb,h,w,c,n,bn,pair,sp", [
    (2, 64, 64, 320, 320, 160, 2, 1), (2, 32, 32, 640, 640, 160, 2, 2), (2, 16, 16, 1280, 1280, 160, 2, 4),
    (2, 8, 8, 1280, 1280, 160, 1, 4), (2, 16, 16, 640, 1280, 128, 1, 2), (3, 32, 32, 64, 256, 256, 2, 2),
    (2, 8, 8, 320, 640, 160, 1, 2), (1, 16, 16, 128, 64, 64, 1, 4),
])
def test_conv3x3_pair_and_cluster_splitk(S, cuda_dev, nb, h, w, c, n, bn, pair, sp):
    """3x3 convs on CTA pairs and with split-K reduced inside the cluster through distributed shared memory: fused
    epilogue (bias, FiLM, residual, fp16 + fp32 outputs) and the per-tile statistics partials."""
    g = torch.Generator().manual_seed(nb * 131 + h + c + sp)
    x = _rand16((nb, h, w, c), cuda_dev, g)
    wt = _rand16((n, c, 3, 3), cuda_dev, g, (9 * c) ** -0.5)
    bias = torch.randn(n, generator=g).to(cuda_dev)
    film = torch.randn(nb, n, generator=g).to(cuda_dev)
    res = torch.randn(nb * h * w, n, generator=g).to(cuda_dev)
    wk = wt.permute(0, 2, 3, 1).reshape(n, 9 * c).contiguous()
    sg = 10 if n % 10 == 0 and bn % 10 == 0 else 2
    o16, o32 = S.ops.gemm(x, wk, taps=9, bias=bias, film=film, residual=res, want_f32=True, want_f16=True, block_n=bn,
                          pair=pair, splits=sp, splitk_mode=2 if sp > 1 else 0, want_stats=True, stats_group=sg)
    torch.cuda.synchronize()
    ref = F.conv2d(x.double().permute(0, 3, 1, 2), wt.double(), bias.double(), padding=1) + film[:, :, None, None]
    ref = ref.permute(0, 2, 3, 1).reshape(nb * h * w, n) + res
    assert rel_l2(o32, ref) < 1e-5, rel_l2(o32, ref)
    assert rel_l2(o16.float(), ref) < 6e-4
    _check_stats(o32, nb, h * w, n)
    # bit-reproducible: fixed-order reduction, no atomics anywhere
    o16b, o32b = S.ops.gemm(x, wk, taps=9, bias=bias, film=film, residual=res, want_f32=True, want_f16=True, block_n=bn,
                            pair=pair, splits=sp, splitk_mode=2 if sp > 1 else 0, want_stats=True, stats_group=sg)
    assert torch.equal(o32, o32b) and torch.equal(o32._sdb_stats[0], o32b._sdb_stats[0])


@pytest.mark.parametrize("M,N,K,sp,pair", [(128, 1280, 5120, 4, 1), (512, 1280, 5120, 4, 2), (2048, 640, 2560, 2, 2),
                                            (512, 320, 1280, 2, 1), (640, 1280, 1920, 2, 2)])
def test_gemm_cluster_splitk_plain(S, cuda_dev, M, N, K, sp, pair):
    g = torch.Generator().manual_seed(M + K + sp)
    a = _rand16((M, K), cuda_dev, g)
    b = _rand16((N, K), cuda_dev, g, K ** -0.5)
    bias = torch.randn(N, generator=g).to(cuda_dev)
    res = torch.randn(M, N, generator=g).to(cuda_dev)
    o16, o32, lo = S.ops.gemm(a, b, bias=bias, residual=res, want_f32=True, want_lo=True, block_n=160 if N % 160 == 0 else 128,
                              pair=pair, splits=sp, splitk_mode=2)
    ref = a.double() @ b.double().t() + bias + res
    assert rel_l2(o32, ref) < 1e-5, rel_l2(o32, ref)
    assert rel_l2(o16.float() + lo.float(), ref) < 2e-6


def test_gemm_workspace_splitk_statistics(S, cuda_dev):
    """Workspace split-K (second kernel) also writes the per-block statistics partials."""
    g = torch.Generator().manual_seed(21)
    nb, h, w, c, n = 2, 8, 8, 640, 1280
    x = _rand16((nb, h, w, c), cuda_dev, g)
    wk = _rand16((n, 9 * c), cuda_dev, g, (9 * c) ** -0.5)
    _, o32 = S.ops.gemm(x, wk, taps=9, want_f32=True, splits=6, splitk_mode=1, want_stats=True, stats_group=10)
    wt = wk.reshape(n, 3, 3, c).permute(0, 3, 1, 2).double()
    ref = F.conv2d(x.double().permute(0, 3, 1, 2), wt, padding=1).permute(0, 2, 3, 1).reshape(-1, n)
    assert rel_l2(o32, ref) < 1e-5
    _check_stats(o32, nb, h * w, n)


def test_gemm_geglu_wide_tile_on_cta_pairs(S, cuda_dev):
    """GEGLU with 256-wide accumulator tiles ([128 value | 128 gate]) on CTA pairs and on single CTAs."""
    g = torch.Generator().manual_seed(12)
    K, inner = 320, 1280
    wfull = _rand16((2 * inner, K), cuda_dev, g, K ** -0.5)
    bfull = torch.randn(2 * inner, generator=g).to(cuda_dev)
    idx = []
    for t in range(inner // 128):
        idx += list(range(t * 128, t * 128 + 128)) + list(range(inner + t * 128, inner + t * 128 + 128))
    idx = torch.tensor(idx, device=cuda_dev)
    wp, bp = wfull[idx].contiguous(), bfull[idx].contiguous()
    for M, pair in ((1000, 2), (128, 1), (8192, 2)):
        a = _rand16((M, K), cuda_dev, g)
        o16, _ = S.ops.gemm(a, wp, bias=bp, act=S.ops.ACT_GEGLU, want_f16=True, block_n=256, pair=pair)
        y = a.float() @ wfull.float().t() + bfull
        ref = y[:, :inner] * F.gelu(y[:, inner:])
        assert o16.shape == (M, inner)
        assert rel_l2(o16.float(), ref) < 8e-4, (M, pair, rel_l2(o16.float(), ref))


@pytest.mark.parametrize("splits", [2, 5, 9])
def test_gemm_splitk(S, cuda_dev, splits):
    g = torch.Generator().manual_seed(splits)
    nb, h, w, c, n = 2, 8, 8, 320, 1280
    x = _rand16((nb, h, w, c), cuda_dev, g)
    wk = _rand16((n, 9 * c), cuda_dev, g, (9 * c) ** -0.5)
    bias = torch.randn(n, generator=g).to(cuda_dev)
    res = torch.randn(nb * h * w, n, generator=g).to(cuda_dev)
    o16, o32 = S.ops.gemm(x, wk, taps=9, bias=bias, residual=res, want_f32=True, want_f16=True, splits=splits)
    wt = wk.reshape(n, 3, 3, c).permute(0, 3, 1, 2).double()
    ref = F.conv2d(x.double().permute(0, 3, 1, 2), wt, bias.double(), padding=1).permute(0, 2, 3, 1).reshape(-1, n) + res
    assert rel_l2(o32, ref) < 1e-5
    assert rel_l2(o16.float(), ref) < 6e-4


def test_gemm_geglu_and_acts(S, cuda_dev):
    g = torch.Generator().manual_seed(11)
    M, K, inner = 300, 320, 1280
    a = _rand16((M, K), cuda_dev, g)
    wfull = _rand16((2 * inner, K), cuda_dev, g, K ** -0.5)   # rows [0,inner) = x, [inner, 2inner) = gate
    bfull = torch.randn(2 * inner, generator=g).to(cuda_dev)
    # pack: tile t holds rows x[t*64:(t+1)*64] then gate[t*64:(t+1)*64]
    idx = []
    for t in range(inner // 64):
        idx += list(range(t * 64, t * 64 + 64)) + list(range(inner + t * 64, inner + t * 64 + 64))
    idx = torch.tensor(idx, device=cuda_dev)
    o16, _ = S.ops.gemm(a, wfull[idx].contiguous(), bias=bfull[idx].contiguous(), act=S.ops.ACT_GEGLU, want_f16=True)
    y = a.float() @ wfull.float().t() + bfull
    ref = y[:, :inner] * F.gelu(y[:, inner:])
    assert o16.shape == (M, inner)
    assert rel_l2(o16.float(), ref) < 8e-4, rel_l2(o16.float(), ref)
    for act, fn in [(S.ops.ACT_SILU, F.silu), (S.ops.ACT_QUICK_GELU, lambda v: v * torch.sigmoid(1.702 * v))]:
        _, o32 = S.ops.gemm(a, wfull[:256].contiguous(), bias=bfull[:256].contiguous(), act=act, want_f32=True)
        ref = fn(a.float() @ wfull[:256].float().t() + bfull[:256])
        assert rel_l2(o32, ref) < 1e-5


def _attn_ref(q, k, v, scale, causal=False):
    s = torch.einsum("bhid,bhjd->bhij", q, k) * scale
    if causal:
        n = s.shape[-1]
        mask = torch.triu(torch.ones(s.shape[-2], n, device=s.device, dtype=torch.bool), 1)
        s = s.masked_fill(mask, float("-inf"))
    return torch.einsum("bhij,bhjd->bhid", s.softmax(-1), v)


@pytest.mark.parametrize("B,H,nq,nkv,d,dpad,causal,amp", [
    (2, 8, 256, 256, 40, 64, False, 1.0), (2, 8, 4096, 4096, 40, 64, False, 1.0), (2, 8, 1024, 1024, 80, 128, False, 1.0),
    (2, 8, 256, 256, 160, 192, False, 1.0), (2, 8, 64, 64, 160, 192, False, 1.0), (2, 8, 4096, 77, 40, 64, False, 1.0),
    (3, 8, 1024, 77, 80, 128, False, 1.0), (2, 12, 77, 77, 64, 64, True, 1.0), (1, 8, 1024, 1024, 40, 64, False, 6.0),
    (1, 2, 200, 333, 64, 64, False, 3.0),
    # split-state kernel (dpad 64, d < 64): a fully masked column half, ragged tiles, small / large head dims
    (1, 2, 100, 20, 40, 64, False, 1.0), (1, 2, 130, 45, 56, 64, False, 2.0), (1, 4, 64, 64, 8, 64, False, 1.0),
    (1, 2, 300, 97, 40, 64, True, 1.0),
])
def test_attention(S, cuda_dev, B, H, nq, nkv, d, dpad, causal, amp):
    g = torch.Generator().manual_seed(nq + nkv + d)
    q = (torch.randn(B, H, nq, d, generator=g) * amp).half()
    k = (torch.randn(B, H, nkv, d, generator=g) * amp).half()
    v = torch.randn(B, H, nkv, d, generator=g).half()
    scale = d ** -0.5
    ref = _attn_ref(q.float(), k.float(), v.float(), scale, causal)          # [B,H,nq,d]
    ref = ref.permute(0, 2, 1, 3).reshape(B, nq, H * d)

    def pad_tokens(t):  # [B,H,n,d] -> [B,n,H*dpad]
        tp = F.pad(t, (0, dpad - d))
        return tp.permute(0, 2, 1, 3).reshape(B, t.shape[2], H * dpad).contiguous().to(cuda_dev)

    qp, kp = pad_tokens(q), pad_tokens(k)
    ld = (nkv + 7) // 8 * 8
    vt = torch.zeros(B, H * dpad, ld, dtype=torch.float16)
    vt[:, :, :nkv] = F.pad(v, (0, dpad - d)).permute(0, 1, 3, 2).reshape(B, H * dpad, nkv)
    vt = vt.to(cuda_dev)
    out = S.ops.attention(qp, kp, vt, heads=H, d=d, dpad=dpad, nq=nq, nkv=nkv, scale=scale, causal=causal)
    torch.cuda.synchronize()
    err = rel_l2(out.float().cpu(), ref)
    assert err < 2e-3, err


@pytest.mark.parametrize("B,n,amp", [(1, 4096, 1.0), (2, 1024, 3.0), (1, 200, 1.0), (3, 64, 1.0)])
def test_attention_wide_d512(S, cuda_dev, B, n, amp):
    """Single-head d = 512 flash kernel (AutoencoderKL AttnBlock, model.py:178-202) against the materialised softmax."""
    c = 512
    g = torch.Generator().manual_seed(n)
    q = (torch.randn(B, n, c, generator=g) * amp).half()
    k = (torch.randn(B, n, c, generator=g) * amp).half()
    v = torch.randn(B, n, c, generator=g).half()
    scale = c ** -0.5
    ref = torch.softmax(torch.einsum("bid,bjd->bij", q.float(), k.float()) * scale, -1) @ v.float()
    ld = (n + 7) // 8 * 8
    vt = torch.zeros(B, c, ld, dtype=torch.float16)
    vt[:, :, :n] = v.transpose(1, 2)
    out = S.ops.attention(q.to(cuda_dev), k.to(cuda_dev), vt.to(cuda_dev), heads=1, d=c, dpad=c, nq=n, nkv=n, scale=scale)
    torch.cuda.synchronize()
    err = rel_l2(out.float().cpu(), ref)
    assert err < 2e-3, err


@pytest.mark.parametrize("nb,h,w,c0,c1,silu,eps", [
    (2, 16, 16, 320, 0, True, 1e-5), (2, 8, 8, 1280, 1280, True, 1e-5), (2, 32, 32, 640, 320, False, 1e-6),
    (1, 64, 64, 128, 0, True, 1e-6), (2, 16, 16, 1280, 640, True, 1e-5),
])
def test_groupnorm(S, cuda_dev, nb, h, w, c0, c1, silu, eps):
    g = torch.Generator().manual_seed(c0 + c1)
    x0 = (torch.randn(nb, h, w, c0, generator=g) * 2 + 0.5).to(cuda_dev)
    x1 = (torch.randn(nb, h, w, c1, generator=g) - 1.0).to(cuda_dev) if c1 else None
    C = c0 + c1
    gamma = (1 + 0.1 * torch.randn(C, generator=g)).to(cuda_dev)
    beta = (0.1 * torch.randn(C, generator=g)).to(cuda_dev)
    out, raw = S.ops.groupnorm(x0, gamma, beta, x1=x1, eps=eps, silu=silu, want_raw=True)
    xc = x0 if x1 is None else torch.cat([x0, x1], -1)
    ref = F.group_norm(xc.permute(0, 3, 1, 2), 32, gamma, beta, eps)
    if silu:
        ref = F.silu(ref)
    ref = ref.permute(0, 2, 3, 1)
    assert rel_l2(out.float(), ref) < 5e-4
    assert rel_l2(raw.float(), xc) < 5e-4


def test_layernorm_softmax(S, cuda_dev):
    g = torch.Generator().manual_seed(3)
    for c in (320, 640, 1280, 768):
        x = (torch.randn(77 * 3, c, generator=g) * 3 + 1).to(cuda_dev)
        gamma = (1 + 0.1 * torch.randn(c, generator=g)).to(cuda_dev)
        beta = (0.1 * torch.randn(c, generator=g)).to(cuda_dev)
        out = S.ops.layernorm(x, gamma, beta, 1e-5)
        assert rel_l2(out.float(), F.layer_norm(x, (c,), gamma, beta, 1e-5)) < 5e-4
    x = torch.randn(100, 4096, generator=g).to(cuda_dev) * 4
    p = S.ops.softmax_rows(x, 0.3)
    assert rel_l2(p.float(), (x * 0.3).softmax(-1)) < 1e-3


def test_elementwise(S, cuda_dev):
    g = torch.Generator().manual_seed(4)
    x = torch.randn(2, 8, 8, 8, generator=g).to(cuda_dev)
    o32, o16 = S.ops.nchw_to_nhwc(x, want_f16=True)
    assert torch.equal(o32, x.permute(0, 2, 3, 1).contiguous())
    assert torch.equal(S.ops.nhwc_to_nchw(o32), x)
    # im2col: 3x3, stride 1, pad 1
    xi = torch.randn(2, 9, 9, 4, generator=g).to(cuda_dev)
    col = S.ops.im2col3x3(xi, 64)
    un = F.unfold(xi.permute(0, 3, 1, 2), 3, padding=1)
    # unfold: [nb, c*9, L] with index c*9 + tap -> ours tap*c + ch
    un = un.reshape(2, 4, 9, -1).permute(0, 3, 2, 1).reshape(-1, 36)
    assert torch.allclose(col[:, :36].float(), un, atol=2e-3)
    assert float(col[:, 36:].abs().max()) == 0.0
    up = S.ops.upsample2x(o32)
    assert torch.allclose(up.float(), F.interpolate(x, scale_factor=2, mode="nearest").permute(0, 2, 3, 1), atol=2e-3)
    t = torch.tensor([981.0, 1.0, 500.5], device=cuda_dev)
    te = S.ops.timestep_embedding_f32(t, 320)
    half = 160
    freqs = torch.exp(-math.log(10000) * torch.arange(half, dtype=torch.float32, device=cuda_dev) / half)
    args = t[:, None] * freqs[None]
    ref = torch.cat([torch.cos(args), torch.sin(args)], -1)
    assert te.dtype == torch.float32 and float((te - ref).abs().max()) < 2e-3
    tr = S.ops.transpose_f16(o16.reshape(2, 64, 8))
    assert tr.shape == (2, 8, 64) and torch.equal(tr, o16.reshape(2, 64, 8).transpose(1, 2))


def test_gemm_hilo_split_recovers_fp32_operands(S, cuda_dev):
    """[A_hi | A_lo | A_hi] . [W_hi | W_hi | W_lo]: three fp16 passes reproduce the fp32-operand product."""
    g = torch.Generator().manual_seed(21)
    M, K, N = 512, 640, 320
    a = torch.randn(M, K, generator=g).to(cuda_dev) * 3
    w = (torch.randn(N, K, generator=g) * K ** -0.5).to(cuda_dev)
    a_hi = a.half()
    a_lo = (a - a_hi.float()).half()
    w_hi = w.half()
    w_lo = (w - w_hi.float()).half()
    wk = torch.cat([w_hi, w_hi, w_lo], 1).contiguous()
    _, o3 = S.ops.gemm(a_hi, wk, a1=a_lo, a2=a_hi, want_f32=True)
    _, o1 = S.ops.gemm(a_hi, w_hi, want_f32=True)
    ref = a.double() @ w.double().t()
    assert rel_l2(o3, ref) < 5e-6, rel_l2(o3, ref)
    assert rel_l2(o1, ref) > 1e-4          # single pass carries the fp16 operand rounding
    # epilogue hi/lo outputs
    hi, f32, lo = S.ops.gemm(a_hi, w_hi, want_f32=True, want_lo=True)
    assert torch.equal(hi, f32.half())
    assert rel_l2(hi.float() + lo.float(), f32) < 2e-6
    # groupnorm hi/lo
    x = torch.randn(2, 8, 8, 128, generator=g).to(cuda_dev)
    gamma = torch.ones(128, device=cuda_dev)
    beta = torch.zeros(128, device=cuda_dev)
    out, raw, out_lo, raw_lo = S.ops.groupnorm(x, gamma, beta, want_lo=True, want_raw_lo=True)
    ref_n = F.group_norm(x.permute(0, 3, 1, 2), 32, gamma, beta, 1e-5).permute(0, 2, 3, 1)
    assert rel_l2(out.float() + out_lo.float(), ref_n) < 5e-6
    assert rel_l2(raw.float() + raw_lo.float(), x) < 1e-6


def test_gemm_many_tiles_persistent(S, cuda_dev):
    """More tiles than SMs: every persistent CTA walks several tiles through both TMEM accumulators."""
    g = torch.Generator().manual_seed(22)
    for (M, N, K, bn) in [(128 * 40, 1280, 192, 128), (128 * 37 + 5, 640, 320, 64), (128 * 9, 2560, 128, 256),
                          (4096, 4096, 512, 0)]:
        a = _rand16((M, K), cuda_dev, g)
        b = _rand16((N, K), cuda_dev, g, K ** -0.5)
        bias = torch.randn(N, generator=g).to(cuda_dev)
        o16, o32 = S.ops.gemm(a, b, bias=bias, want_f16=True, want_f32=True, block_n=bn)
        ref = a.double() @ b.double().t() + bias
        assert rel_l2(o32, ref) < 1e-5, (M, N, K, bn, rel_l2(o32, ref))
        assert rel_l2(o16.float(), ref) < 6e-4


def test_gemm_narrow_tiles_many_per_cta(S, cuda_dev):
    """block_n 32/64 with more than two tiles per persistent CTA (accumulator hand-off with idle epilogue warps)."""
    g = torch.Generator().manual_seed(23)
    for (M, N, K, bn) in [(128 * 500, 32, 128, 32), (128 * 300, 96, 64, 32), (128 * 450, 64, 192, 64), (128 * 700, 3, 128, 0)]:
        a = _rand16((M, K), cuda_dev, g)
        b = _rand16((N, K), cuda_dev, g, K ** -0.5)
        _, o32 = S.ops.gemm(a, b, want_f32=True, block_n=bn)
        ref = a.double() @ b.double().t()
        assert rel_l2(o32, ref) < 1e-5, (M, N, K, bn)


def test_gemm_fused_groupnorm_stats_and_inkernel_splitk(S, cuda_dev):
    """Per-tile statistics partials stored by the GEMM epilogue (any split-K mode, entries of 1 / 2 / 10 channels) feed
    groupnorm() without a reduction pass, also across a channel concat and through the large-image fold kernel."""
    g = torch.Generator().manual_seed(31)
    for (nb, h, w, c, n, splits, sg) in [(2, 16, 16, 128, 320, 0, 10), (2, 8, 8, 320, 640, 4, 10), (3, 8, 8, 64, 64, -1, 2),
                                         (2, 32, 32, 64, 128, 0, 1), (1, 128, 128, 64, 128, 0, 4), (2, 24, 24, 64, 320, 0, 10), (3, 24, 24, 128, 160, 2, 10)]:
        x = _rand16((nb, h, w, c), cuda_dev, g)
        wk = _rand16((n, 9 * c), cuda_dev, g, (9 * c) ** -0.5)
        bias = torch.randn(n, generator=g).to(cuda_dev)
        res = (torch.randn(nb * h * w, n, generator=g) * 2 + 0.7).to(cuda_dev)
        _, o32 = S.ops.gemm(x, wk, taps=9, bias=bias, residual=res, want_f32=True, splits=splits, want_stats=True,
                            stats_group=sg)
        wt = wk.reshape(n, 3, 3, c).permute(0, 3, 1, 2).double()
        ref = F.conv2d(x.double().permute(0, 3, 1, 2), wt, bias.double(), padding=1).permute(0, 2, 3, 1).reshape(-1, n) + res
        assert rel_l2(o32, ref) < 1e-5, (nb, h, w, c, n, splits, rel_l2(o32, ref))
        assert S.ops.channel_stats(o32) is not None
        _check_stats(o32, nb, h * w, n)
        gamma = (1 + 0.1 * torch.randn(n, generator=g)).to(cuda_dev)
        beta = (0.1 * torch.randn(n, generator=g)).to(cuda_dev)
        y, _ = S.ops.groupnorm(o32.view(nb, h, w, n), gamma, beta, eps=1e-5, silu=True)   # uses the fused stats
        yr = F.silu(F.group_norm(ref.float().reshape(nb, h, w, n).permute(0, 3, 1, 2), 32, gamma, beta, 1e-5)).permute(0, 2, 3, 1)
        assert rel_l2(y.float(), yr) < 6e-4
    # concat of two stat-carrying tensors (groups straddle the boundary: 192 + 64 channels, 8 per group)
    xa = _rand16((2, 8, 8, 64), cuda_dev, g)
    wa = _rand16((192, 9 * 64), cuda_dev, g, 0.05)
    wb = _rand16((64, 9 * 64), cuda_dev, g, 0.05)
    _, a32 = S.ops.gemm(xa, wa, taps=9, want_f32=True, want_stats=True, stats_group=2)
    _, b32 = S.ops.gemm(xa, wb, taps=9, want_f32=True, want_stats=True, stats_group=2, splits=2, splitk_mode=2)
    gam = torch.ones(256, device=cuda_dev)
    bet = torch.zeros(256, device=cuda_dev)
    y, _ = S.ops.groupnorm(a32.view(2, 8, 8, 192), gam, bet, x1=b32.view(2, 8, 8, 64), eps=1e-6)
    cat = torch.cat([a32.view(2, 8, 8, 192), b32.view(2, 8, 8, 64)], -1)
    yr = F.group_norm(cat.permute(0, 3, 1, 2), 32, gam, bet, 1e-6).permute(0, 2, 3, 1)
    assert rel_l2(y.float(), yr) < 6e-4


def test_c_abi_rejects_bad_arguments(S, cuda_dev):
    """Error behaviour of the boundary: non-zero return + message, surfaced as RuntimeError (never a silent fallback)."""
    a = torch.zeros(128, 64, dtype=torch.float16, device=cuda_dev)
    b = torch.zeros(64, 64, dtype=torch.float16, device=cuda_dev)
    with pytest.raises(RuntimeError, match="taps"):
        d = S.lib.GemmDesc()
        d.a0, d.b, d.c0, d.nb, d.h, d.w, d.taps, d.n = a.data_ptr(), b.data_ptr(), 64, 1, 1, 128, 5, 64
        d.out_f32 = torch.empty(128, 64, device=cuda_dev).data_ptr()
        S.lib.check(S.lib.load().sdb_gemm(d, None), "sdb_gemm")
    with pytest.raises(RuntimeError, match="multiple of 64"):
        S.ops.gemm(torch.zeros(128, 40, dtype=torch.float16, device=cuda_dev),
                   torch.zeros(64, 40, dtype=torch.float16, device=cuda_dev), want_f32=True)
    with pytest.raises(RuntimeError, match="dpad"):
        q = torch.zeros(1, 64, 96, dtype=torch.float16, device=cuda_dev)
        S.ops.attention(q, q, torch.zeros(1, 96, 64, dtype=torch.float16, device=cuda_dev), heads=1, d=96, dpad=96,
                        nq=64, nkv=64, scale=1.0)
    with pytest.raises(RuntimeError, match="GEGLU"):
        S.ops.gemm(a, torch.zeros(96, 64, dtype=torch.float16, device=cuda_dev), act=S.ops.ACT_GEGLU, want_f16=True)
