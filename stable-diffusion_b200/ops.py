"""Tensor-level wrappers over the C ABI: PyTorch tensors in/out (device memory + current stream only).

Every function enqueues hand-written sm_100a kernels from libsdb200.so on the current CUDA stream; none of
them computes with torch. Shapes follow the engine's layouts: activations NHWC, fp32 residual stream,
fp16 tensor-core operands.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import lib as _l
from .lib import ACT_GEGLU, ACT_NONE, ACT_QUICK_GELU, ACT_SILU, AttnDesc, GemmDesc  # noqa: F401

_GRAPH_LAUNCHES = 0  # kernels replayed from CUDA graphs (counted at capture time, added per replay)
PROFILE = None      # when a list: gemm()/attention() append (kind, flops, start_event, end_event)
RECORD = None       # when a list: gemm() appends (desc, algorithmic_flops, keepalive) so bench.py can replay the launches
AUTOTUNE = False    # when True, gemm() times the (block_n, split-K) candidates of an unseen problem once and caches the best
TUNED = {}          # problem key -> (block_n, splits)


def launch_count():
    """Kernels launched from libsdb200.so: direct launches (counted in C) + kernels replayed inside CUDA graphs."""
    return int(_l.load().sdb_launch_count()) + _GRAPH_LAUNCHES


def add_graph_launches(n):
    global _GRAPH_LAUNCHES
    _GRAPH_LAUNCHES += int(n)



def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _chk16(t, name):
    assert t.dtype == torch.float16 and t.is_cuda and t.is_contiguous(), f"{name}: need contiguous cuda fp16"


def _chk32(t, name):
    assert t.dtype == torch.float32 and t.is_cuda and t.is_contiguous(), f"{name}: need contiguous cuda fp32"


def gemm(a0, b, *, a1=None, a2=None, a3=None, nb=None, h=None, w=None, taps=1, bias=None, film=None,
         rows_per_sample=0, residual=None, act=ACT_NONE, alpha=1.0, out_f16=None, out_f32=None, out_f16_lo=None,
         want_f16=False, want_f32=False, want_lo=False, n=None, block_n=0, splits=0, workspace=None,
         want_stats=False, stats_group=1, b_dynamic=False, conv_stride=1, conv_shift=0, pair=0, splitk_mode=0):
    """acc = A @ B^T with fused epilogue (see sdb_gemm in include/sdb200.h).

    a0 (, a1, a2, a3): fp16 [..., c_i] NHWC activations or plain [rows, c_i] matrices, concatenated along K.
    b: fp16 [n, taps*sum(c_i)].
    Returns (out_f16, out_f32), or (out_f16, out_f32, out_f16_lo) when the hi/lo pair is requested.
    block_n / pair / splits / splitk_mode: explicit tile width, CTA pairs (2) or single CTAs (1), split-K factor and how
    its partials meet (1 workspace + second kernel, 2 thread-block cluster); 0 = let the library (or the autotuner) pick.
    want_stats: the epilogue also stores per-tile GroupNorm partial sums of the fp32 output (entries of `stats_group`
    channels); they are attached to the output tensor (see channel_stats()) so the following groupnorm() skips its
    reduction pass.
    """
    _chk16(a0, "a0")
    _chk16(b, "b")
    srcs = [a0]
    for t_ in (a1, a2, a3):
        if t_ is None:
            break
        _chk16(t_, "a_i")
        assert t_.shape[:-1] == a0.shape[:-1]
        srcs.append(t_)
    chans = [t_.shape[-1] for t_ in srcs]
    c0 = chans[0]
    in_h = in_w = 0
    if taps == 9:
        assert a0.dim() == 4, "3x3 conv needs NHWC input"
        nb, h, w = a0.shape[0], a0.shape[1], a0.shape[2]
        if conv_stride == 2:      # output size of a 3x3 / stride-2 conv: symmetric pad 1 (shift 0) or pad right/bottom (shift 1)
            in_h, in_w = h, w
            h, w = (in_h + 1 - conv_shift) // 2, (in_w + 1 - conv_shift) // 2
    else:
        rows = a0.numel() // c0
        nb, h, w = 1, 1, rows
    n = b.shape[0] if n is None else n
    assert b.shape[1] == taps * sum(chans), (b.shape, taps, chans)
    M = nb * h * w
    n_out = n // 2 if act == ACT_GEGLU else n
    if out_f16 is None and (want_f16 or want_lo):
        out_f16 = torch.empty((M, n_out), dtype=torch.float16, device=a0.device)
    if out_f16_lo is None and want_lo:
        out_f16_lo = torch.empty((M, n_out), dtype=torch.float16, device=a0.device)
    if out_f32 is None and want_f32:
        out_f32 = torch.empty((M, n_out), dtype=torch.float32, device=a0.device)
    assert out_f16 is not None or out_f32 is not None
    lib = _l.load()
    d = GemmDesc()
    ptrs = [_ptr(t_) for t_ in srcs] + [None] * (4 - len(srcs))
    cs = chans + [0] * (4 - len(chans))
    d.a0, d.a1, d.a2, d.a3 = ptrs
    d.c0, d.c1, d.c2, d.c3 = cs
    d.nb, d.h, d.w, d.taps = nb, h, w, taps
    d.b, d.n, d.alpha = _ptr(b), n, alpha
    d.bias = _ptr(bias)
    d.film = _ptr(film)
    d.ldf = film.stride(0) if film is not None else 0
    d.rows_per_sample = rows_per_sample
    d.residual = _ptr(residual)
    d.ldr = residual.shape[-1] if residual is not None else 0
    d.act = act
    d.out_f16, d.out_f32, d.out_f16_lo = _ptr(out_f16), _ptr(out_f32), _ptr(out_f16_lo)
    d.ldo = 0
    d.block_n, d.pair, d.splitk_mode = block_n, pair, splitk_mode
    d.b_dynamic = 1 if b_dynamic else 0   # b produced by the previous kernel: no early (pre-dependency) prefetch
    d.conv_stride, d.conv_shift, d.in_h, d.in_w = conv_stride, conv_shift, in_h, in_w
    d.splits = splits
    if splits and (splits > 1 or splits == -1) and splitk_mode != 2:
        if workspace is None:
            workspace = splitk_workspace(a0.device)
        d.workspace = _ptr(workspace)
        d.workspace_floats = workspace.numel()
    rps = rows_per_sample if rows_per_sample else h * w
    stats_ok = want_stats and out_f32 is not None and act != ACT_GEGLU and (taps == 9 or rows_per_sample) and \
        M % rps == 0 and n % stats_group == 0
    d.stats_group = stats_group
    if stats_ok:
        d.stats_out = C.c_void_p(16)     # placeholder: the plan only needs to know that statistics are wanted
    plan = (C.c_int32 * 5)()
    tunable = block_n == 0 and pair == 0 and splitk_mode == 0 and splits in (0, -1) and act != ACT_GEGLU
    if tunable:
        key = (M, n, b.shape[1], taps, len(srcs), bias is not None, film is not None, residual is not None, act,
               out_f16 is not None, out_f32 is not None, out_f16_lo is not None, stats_ok, stats_group, conv_stride)
        choice = TUNED.get(key)
        if choice is None and AUTOTUNE:
            choice = TUNED[key] = _tune_gemm(d, M, n, rps, stats_ok, stats_group)
        if choice is not None:
            d.block_n, d.pair, d.splits, d.splitk_mode = choice
    rc = lib.sdb_gemm_plan(C.byref(d), plan)
    if rc != 0 and stats_ok:             # this problem / tile shape cannot produce fused statistics: plain GEMM, the
        stats_ok = False                 # consumer falls back to its own reduction pass
        d.stats_out = None
        rc = lib.sdb_gemm_plan(C.byref(d), plan)
    _l.check(rc, "sdb_gemm_plan")
    d.block_n, d.pair, d.splits, d.splitk_mode = plan[0], plan[1], plan[2], plan[3]
    stats = None
    if stats_ok:
        shape = (M // rps, plan[4], n // stats_group, 2)
        stats = ARENA.take(shape) if ARENA is not None else None
        if stats is None:
            stats = torch.empty(shape, dtype=torch.float32, device=a0.device)
        d.stats_out = _ptr(stats)
        out_f32._sdb_stats = (stats, plan[4], stats_group)   # travels with the tensor object (and, through ._base, its views)
    if RECORD is not None:
        # operand-split passes ([A_hi|A_lo|A_hi]) are overhead, not algorithmic work: count K once
        k_alg = b.shape[1] // 3 if (len(srcs) == 3 and srcs[0] is srcs[2]) else b.shape[1]
        RECORD.append((d, 2.0 * M * n * k_alg, (srcs, b, bias, film, residual, out_f16, out_f32, out_f16_lo, workspace, stats)))
    if PROFILE is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    _l.check(lib.sdb_gemm(C.byref(d), _stream()), "sdb_gemm")
    if PROFILE is not None:
        e1.record()
        PROFILE.append(("gemm", 2.0 * M * n * b.shape[1], e0, e1, (M, n, b.shape[1], taps)))
    if out_f16_lo is not None:
        return out_f16, out_f32, out_f16_lo
    return out_f16, out_f32


class StatsArena:
    """One fp32 bump buffer per forward pass for all fused GroupNorm statistics. The GEMM epilogues STORE their per-tile
    partial sums (every slot has exactly one writer), so nothing is zeroed: reset() only rewinds the bump pointer;
    gemm(want_stats=True) carves its [samples, T, n / group, 2] slice."""

    def __init__(self, device, n_floats=4 * 1024 * 1024):
        self.buf = torch.empty(n_floats, dtype=torch.float32, device=device)
        self.off = 0

    def reset(self):
        self.off = 0

    def take(self, shape):
        n = 1
        for s_ in shape:
            n *= s_
        if self.off + n > self.buf.numel():
            return None
        v = self.buf[self.off: self.off + n].view(shape)
        self.off += (n + 3) // 4 * 4
        return v


ARENA = None   # set by the model around a forward pass (UNetModel._forward_impl)


def channel_stats(x):
    """Fused GroupNorm statistics (partials tensor, slots per sample, channels per entry) attached to `x` (or the tensor
    it is a view of) by the gemm() that produced it."""
    st = getattr(x, "_sdb_stats", None)
    if st is None and x._base is not None and x._base.numel() == x.numel():
        st = getattr(x._base, "_sdb_stats", None)
    return st


def _tune_gemm(d, M, n, rps, stats_ok, stats_group):
    """Time the (tile width, CTA pair, split-K) candidates of one GEMM problem on its real operands (CUDA events, GPU
    kept busy by a leading spin so host launch gaps do not enter) and return the fastest
    (block_n, pair, splits, splitk_mode)."""
    lib = _l.load()
    st = _stream()
    keep = (d.block_n, d.pair, d.splits, d.splitk_mode, d.stats_out)
    scratch = None
    if stats_ok:
        d.stats_out = C.c_void_p(16)     # placeholder while the candidates are planned (sized below)
    plan = (C.c_int32 * 5)()
    cands = []
    max_slots = 1
    for bn in (64, 128, 160, 256):
        pad = (n + bn - 1) // bn * bn - n
        if bn > 64 and pad >= bn // 2:
            continue
        for cg in (1, 2):
            for sp, mode in ((1, 0), (2, 2), (4, 2), (2, 1), (3, 1), (4, 1), (6, 1), (8, 1), (12, 1), (16, 1)):
                if mode == 1 and not d.workspace:
                    continue
                tiles = ((M + 127) // 128) * ((n + bn - 1) // bn) * sp
                if sp > 1 and tiles > 3 * 148:
                    continue
                d.block_n, d.pair, d.splits, d.splitk_mode = bn, cg, sp, mode
                if lib.sdb_gemm_plan(C.byref(d), plan) != 0:
                    continue
                if (plan[0], plan[1], plan[2], plan[3]) != (bn, cg, sp, mode if sp > 1 else 0):
                    continue
                cands.append((bn, cg, sp, mode))
                max_slots = max(max_slots, int(plan[4]))
    if stats_ok:
        # the statistics slots per sample depend on the candidate (tiles x cluster splits, or one per 32 rows with the
        # workspace epilogue): size the scratch for the largest one - a smaller buffer is overrun by the epilogues
        scratch = torch.empty((M // rps) * max_slots * (n // stats_group) * 2 + 16, dtype=torch.float32,
                              device=torch.device("cuda", torch.cuda.current_device()))
        d.stats_out = _ptr(scratch)
    best, best_t = None, float("inf")
    for cand in cands:
        d.block_n, d.pair, d.splits, d.splitk_mode = cand
        if lib.sdb_gemm(C.byref(d), st) != 0:      # warm-up / validity
            continue
        t = float("inf")
        for _ in range(3):      # best of three short bursts: one noisy burst must not decide the captured tile shape
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda._sleep(400_000)
            e0.record()
            for _ in range(4):
                lib.sdb_gemm(C.byref(d), st)
            e1.record()
            e1.synchronize()
            t = min(t, e0.elapsed_time(e1))
        if t < best_t:
            best, best_t = cand, t
    d.block_n, d.pair, d.splits, d.splitk_mode, d.stats_out = keep
    del scratch
    return best


_WS = {}
WS_FLOATS = 16 * 1024 * 1024


def splitk_workspace(device):
    """Persistent fp32 scratch for split-K partials (stream-ordered reuse: one GEMM at a time per stream)."""
    key = (device.type, device.index)
    if key not in _WS:
        _WS[key] = torch.empty(WS_FLOATS, dtype=torch.float32, device=device)
    return _WS[key]


def attention(q, k, vt, *, heads, d, dpad, nq, nkv, scale, causal=False, out=None):
    """q [B, nq, heads*dpad], k [B, nkv, heads*dpad], vt [B, heads*dpad, ldvt] fp16 -> out [B, nq, heads*d] fp16."""
    for name, t_ in (("q", q), ("k", k), ("vt", vt)):
        assert t_.dtype == torch.float16 and t_.is_cuda and t_.dim() == 3 and t_.stride(2) == 1, f"{name}: bad layout"
    B = q.shape[0]
    if out is None:
        out = torch.empty((B, nq, heads * d), dtype=torch.float16, device=q.device)
    a = AttnDesc()
    a.q, a.k, a.vt, a.out = _ptr(q), _ptr(k), _ptr(vt), _ptr(out)
    a.batch, a.heads, a.nq, a.nkv, a.d, a.dpad = B, heads, nq, nkv, d, dpad
    a.ldq, a.ldk, a.ldvt, a.ldo = q.stride(1), k.stride(1), vt.stride(1), out.stride(1)
    a.q_batch_stride, a.k_batch_stride = q.stride(0), k.stride(0)
    a.vt_batch_stride, a.o_batch_stride = vt.stride(0), out.stride(0)
    a.scale, a.causal = scale, 1 if causal else 0
    if PROFILE is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    _l.check(_l.load().sdb_attention(C.byref(a), _stream()), "sdb_attention")
    if PROFILE is not None:
        e1.record()
        PROFILE.append(("attention", 4.0 * B * heads * nq * nkv * d, e0, e1, (B, heads, nq, nkv, d)))
    return out


def groupnorm(x0, gamma, beta, *, x1=None, groups=32, eps=1e-5, silu=False, want_raw=False, want_lo=False,
              want_raw_lo=False):
    """x0 (, x1): fp32 NHWC [nb, h, w, c]; returns (normalised fp16 NHWC [nb,h,w,c0+c1], raw fp16 or None), plus the
    low halves (out_lo, raw_lo) of the hi/lo split when requested: (out, raw, out_lo, raw_lo)."""
    _chk32(x0, "x0")
    nb, h, w, c0 = x0.shape
    c1 = 0
    if x1 is not None:
        _chk32(x1, "x1")
        c1 = x1.shape[-1]
    out = torch.empty((nb, h, w, c0 + c1), dtype=torch.float16, device=x0.device)
    raw = torch.empty_like(out) if (want_raw or want_raw_lo) else None
    out_lo = torch.empty_like(out) if want_lo else None
    raw_lo = torch.empty_like(out) if want_raw_lo else None
    ws = torch.empty(nb * (128 * groups * 2 + groups * 2 + 1), dtype=torch.float32, device=x0.device)
    cs0 = channel_stats(x0)
    cs1 = channel_stats(x1) if x1 is not None else None
    sg = cs0[2] if cs0 is not None else 1
    cpg = (c0 + c1) // groups
    if cs0 is None or (x1 is not None and (cs1 is None or cs1[2] != sg)) or cpg % sg or c0 % sg or c1 % sg:
        cs0 = cs1 = None     # no (compatible) fused statistics: the kernel pair below computes them
    t0, t1 = (cs0[1] if cs0 else 0), (cs1[1] if cs1 else 0)
    _l.check(_l.load().sdb_groupnorm(_ptr(x0), _ptr(x1), c0, c1, nb, h * w, groups, _ptr(gamma), _ptr(beta),
                                     eps, 1 if silu else 0, _ptr(out), _ptr(raw), _ptr(out_lo), _ptr(raw_lo), _ptr(ws),
                                     _ptr(cs0[0]) if cs0 else None, _ptr(cs1[0]) if cs1 else None, t0, t1, sg,
                                     _stream()), "sdb_groupnorm")
    if want_lo or want_raw_lo:
        return out, raw, out_lo, raw_lo
    return out, raw


def layernorm(x, gamma, beta, eps=1e-5, want_f32=False):
    """x fp32 [rows, c] -> fp16 [rows, c]."""
    _chk32(x, "x")
    c = x.shape[-1]
    rows = x.numel() // c
    out = torch.empty(x.shape, dtype=torch.float16, device=x.device)
    out32 = torch.empty_like(x) if want_f32 else None
    _l.check(_l.load().sdb_layernorm(_ptr(x), rows, c, _ptr(gamma), _ptr(beta), eps, _ptr(out), _ptr(out32),
                                     _stream()), "sdb_layernorm")
    return (out, out32) if want_f32 else out


def softmax_rows(x, scale):
    _chk32(x, "x")
    cols = x.shape[-1]
    rows = x.numel() // cols
    out = torch.empty(x.shape, dtype=torch.float16, device=x.device)
    _l.check(_l.load().sdb_softmax_rows(_ptr(x), rows, cols, scale, _ptr(out), _stream()), "sdb_softmax_rows")
    return out


def nchw_to_nhwc(x, want_f32=True, want_f16=False):
    _chk32(x, "x")
    nb, c, h, w = x.shape
    o32 = torch.empty((nb, h, w, c), dtype=torch.float32, device=x.device) if want_f32 else None
    o16 = torch.empty((nb, h, w, c), dtype=torch.float16, device=x.device) if want_f16 else None
    _l.check(_l.load().sdb_nchw_to_nhwc(_ptr(x), nb, c, h * w, _ptr(o32), _ptr(o16), _stream()), "sdb_nchw_to_nhwc")
    return o32, o16


def nhwc_to_nchw(x, out=None):
    _chk32(x, "x")
    nb, h, w, c = x.shape
    if out is None:
        out = torch.empty((nb, c, h, w), dtype=torch.float32, device=x.device)
    _l.check(_l.load().sdb_nhwc_to_nchw(_ptr(x), nb, c, h * w, _ptr(out), _stream()), "sdb_nhwc_to_nchw")
    return out


def im2col3x3(x, kpad):
    """x fp32 NHWC [nb, h, w, c] -> fp16 [nb*h*w, kpad]: the 3x3 / stride-1 / pad-1 patches, K zero-padded to kpad."""
    _chk32(x, "x")
    nb, h, w, c = x.shape
    out = torch.empty((nb * h * w, kpad), dtype=torch.float16, device=x.device)
    _l.check(_l.load().sdb_im2col3x3(_ptr(x), nb, h, w, c, kpad, _ptr(out), _stream()), "sdb_im2col3x3")
    return out


def upsample2x(x):
    _chk32(x, "x")
    nb, h, w, c = x.shape
    out = torch.empty((nb, 2 * h, 2 * w, c), dtype=torch.float16, device=x.device)
    _l.check(_l.load().sdb_upsample2x(_ptr(x), nb, h, w, c, _ptr(out), _stream()), "sdb_upsample2x")
    return out


def cast_f16(x):
    _chk32(x, "x")
    out = torch.empty(x.shape, dtype=torch.float16, device=x.device)
    _l.check(_l.load().sdb_cast_f16(_ptr(x), x.numel(), _ptr(out), _stream()), "sdb_cast_f16")
    return out


def transpose_f16(x, ldo=None, out=None):
    """x fp16 [B, rows, cols] -> [B, cols, ldo] (rows valid, ldo >= rows, multiple of 8 for TMA)."""
    _chk16(x, "x")
    B, rows, cols = x.shape
    if ldo is None:
        ldo = (rows + 7) // 8 * 8
    if out is None:
        out = torch.empty((B, cols, ldo), dtype=torch.float16, device=x.device)  # pad columns are never read
    assert out.shape == (B, cols, ldo) and out.is_contiguous()
    _l.check(_l.load().sdb_transpose_f16(_ptr(x), B, rows, cols, cols, _ptr(out), ldo, _stream()),
             "sdb_transpose_f16")
    return out


def timestep_embedding_f32(t, dim, max_period=10000.0):
    _chk32(t, "t")
    out = torch.empty((t.numel(), dim), dtype=torch.float32, device=t.device)
    _l.check(_l.load().sdb_timestep_embedding_f32(_ptr(t), t.numel(), dim, max_period, _ptr(out), _stream()),
             "sdb_timestep_embedding_f32")
    return out


def linear_small(x, w, bias=None, act=ACT_NONE, want_f16=False):
    """x fp32 [m, k] (m small), w fp16 [n, k] -> fp32 [m, n] (fp32 activations end to end)."""
    _chk32(x, "x")
    _chk16(w, "w")
    m, k = x.shape
    n = w.shape[0]
    out = torch.empty((m, n), dtype=torch.float32, device=x.device)
    out16 = torch.empty((m, n), dtype=torch.float16, device=x.device) if want_f16 else None
    _l.check(_l.load().sdb_linear_small(_ptr(x), m, k, _ptr(w), n, _ptr(bias), act, _ptr(out), _ptr(out16),
                                        _stream()), "sdb_linear_small")
    return (out, out16) if want_f16 else out


def sampler_step(x, eps2, *, guided, scale, order, hist, noise, a_t, a_prev, sigma_t, sqrt_one_minus_a_t,
                 x_prev=None, pred_x0=None, e_out=None, dup=False, eps_cond=None):
    """One fused CFG + PLMS/DDIM update. x: [b,...] fp32; eps2: [2b,...] if guided else [b,...].
    dup: x_prev is a [2b,...] buffer and both halves receive the new latent (the next step's doubled batch)."""
    _chk32(x, "x")
    _chk32(eps2, "eps2")
    n = x.numel()
    if x_prev is None:
        x_prev = torch.empty((2,) + tuple(x.shape), dtype=torch.float32, device=x.device).flatten(0, 1) if dup \
            else torch.empty_like(x)
    if pred_x0 is None:
        pred_x0 = torch.empty_like(x)
    xp2 = None
    if dup:
        assert x_prev.numel() == 2 * n and x_prev.is_contiguous()
        xp2 = C.c_void_p(x_prev.data_ptr() + 4 * n)
    h = list(hist) + [None] * (3 - len(hist))
    _l.check(_l.load().sdb_sampler_step(_ptr(x), _ptr(eps2), _ptr(eps_cond), 1 if guided else 0, scale, order, _ptr(h[0]),
                                        _ptr(h[1]), _ptr(h[2]), _ptr(noise), a_t, a_prev, sigma_t,
                                        sqrt_one_minus_a_t, n, _ptr(x_prev), xp2, _ptr(pred_x0), _ptr(e_out),
                                        _stream()), "sdb_sampler_step")
    return x_prev, pred_x0, e_out


def dpm_solver_step(x, eps2, *, guided, scale, sigma_s, alpha_s, order, m_prev, c_x, c_m, inv_r0, x_out, dup=False,
                    eps_cond=None):
    """One fused CFG + data-prediction + DPM-Solver++ (2M) update; returns (x_out, m0). dup as in sampler_step."""
    _chk32(x, "x")
    _chk32(eps2, "eps2")
    n = x.numel()
    m_out = torch.empty_like(x)
    xo2 = None
    if dup:
        assert x_out.numel() == 2 * n and x_out.is_contiguous()
        xo2 = C.c_void_p(x_out.data_ptr() + 4 * n)
    _l.check(_l.load().sdb_dpm_solver_step(_ptr(x), _ptr(eps2), _ptr(eps_cond), 1 if guided else 0, scale, sigma_s, alpha_s, order,
                                           _ptr(m_prev), c_x, c_m, inv_r0, n, _ptr(m_out), _ptr(x_out), xo2,
                                           _stream()), "sdb_dpm_solver_step")
    return x_out, m_out


def mask_blend(img_orig, mask, img, b, dup=False):
    """img[:b] = img_orig * mask + (1 - mask) * img[:b], in place; dup also writes the result to img[b:2b]."""
    _chk32(img_orig, "img_orig")
    _chk32(mask, "mask")
    _chk32(img, "img")
    nb, c = img_orig.shape[0], img_orig.shape[1]
    hw = img_orig[0, 0].numel()
    assert nb == b and mask.shape[0] == nb and mask[0, 0].numel() == hw, (img_orig.shape, mask.shape)
    i2 = C.c_void_p(img.data_ptr() + 4 * img_orig.numel()) if dup else None
    _l.check(_l.load().sdb_mask_blend(_ptr(img_orig), _ptr(mask), mask.shape[1], nb, c, hw, _ptr(img), i2, _stream()),
             "sdb_mask_blend")
    return img


def axpby2(x, y, a, b):
    _chk32(x, "x")
    _chk32(y, "y")
    out = torch.empty_like(x)
    _l.check(_l.load().sdb_axpby2(_ptr(x), _ptr(y), a, b, x.numel(), _ptr(out), _stream()), "sdb_axpby2")
    return out


def vae_sample(moments, noise, nb, hw, scale_factor):
    _chk32(moments, "moments")
    z = torch.empty((nb, 4, hw), dtype=torch.float32, device=moments.device)
    _l.check(_l.load().sdb_vae_sample(_ptr(moments), _ptr(noise), nb, hw, scale_factor, _ptr(z), _stream()),
             "sdb_vae_sample")
    return z


def to_uint8(x):
    _chk32(x, "x")
    out = torch.empty(x.shape, dtype=torch.uint8, device=x.device)
    _l.check(_l.load().sdb_to_uint8(_ptr(x), x.numel(), _ptr(out), _stream()), "sdb_to_uint8")
    return out


def axpby(x, a, b=0.0, out=None):
    _chk32(x, "x")
    if out is None:
        out = torch.empty_like(x)
    else:
        _chk32(out, "out")
        assert out.numel() == x.numel()
    _l.check(_l.load().sdb_axpby(_ptr(x), a, b, x.numel(), _ptr(out), _stream()), "sdb_axpby")
    return out


def pointwise_small(x, w, b=None, alpha=1.0):
    """x fp32 [..., cin] NHWC, w fp32 [cout, cin] -> fp32 [..., cout]."""
    _chk32(x, "x")
    _chk32(w, "w")
    cout, cin = w.shape
    assert x.shape[-1] == cin
    out = torch.empty(tuple(x.shape[:-1]) + (cout,), dtype=torch.float32, device=x.device)
    _l.check(_l.load().sdb_pointwise_small(_ptr(x), x.numel() // cin, cin, cout, _ptr(w), _ptr(b), alpha, _ptr(out),
                                           _stream()), "sdb_pointwise_small")
    return out


def embed_tokens(ids, tok, pos):
    """ids int64 [B, n] -> fp32 [B*n, dim]."""
    assert ids.dtype == torch.int64 and ids.is_cuda and ids.is_contiguous()
    B, n = ids.shape
    dim = tok.shape[1]
    out = torch.empty((B * n, dim), dtype=torch.float32, device=ids.device)
    _l.check(_l.load().sdb_embed_tokens(_ptr(ids), B * n, n, dim, tok.shape[0], _ptr(tok), _ptr(pos), _ptr(out),
                                        _stream()), "sdb_embed_tokens")
    return out
