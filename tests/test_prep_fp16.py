"""Kernel 0 and the fused Ulysses exchange in fp16: the fused pre-attention path for half-precision models
(CogVideoX-2B: 30 heads x 64, LayerNorm(64) with bias, FP16 inference).

diffusers rounds at the same points in fp16 as in bf16 -- RMSNorm rounds x * rsqrt(mean(x^2) + eps) to the weight's
dtype and the product with the weight again, LayerNorm rounds once, the rotary embedding rounds its fp32 sum once -- so
the fp16 restatement below keeps the oracle's order (oracle/prep_oracle.py) and rounds with f16_round, and kernel 0's
kF16 forms round with
cvt.rn.f16x2.f32: overflow becomes +-inf, results below 2^-14 stay subnormal.  The bar is assert_prep_close with fp16's
unit roundoff: |got - ref| <= 2^-10 * |pair| + 2^-24 and at least 99.9 % of the elements identical."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from fake_attention import FakeAttention
from helpers import cos_sim
from oracle import make_golden as MG
from oracle import prep_oracle as PO
from rsa_b200 import geometry as G
from rsa_b200 import native as N
from rsa_b200 import ops, parallel

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F16 = torch.float16


def assert_prep_close_f16(got, ref, what="", ulps=1):
    """assert_prep_close (helpers.py) with fp16's ulp: |got - ref| <= ulps * 2^-10 * |pair| + 2^-24 (one subnormal
    step), and >= 99.9 % of the elements identical.  Infinities must sit at the same places with the same sign.
    ulps = 2 for RMSNorm between implementations with different rsqrt: RMSNorm rounds twice, and in fp16 (11 bits) the
    fp32-ulp difference of rsqrt flips the first rounding often enough (1.28 x the one-ulp bound on the GPU) that the
    flipped ulp, multiplied by the weight and rounded again, shows as up to two at the output."""
    got = np.asarray(got, dtype=np.float32)
    ref = np.asarray(ref, dtype=np.float32)
    inf = np.isinf(ref)
    assert np.array_equal(np.isinf(got), inf) and np.array_equal(got[inf], ref[inf]), f"{what}: infinities differ"
    assert not np.isnan(got).any(), f"{what}: NaN"
    g, r = np.where(inf, 0, got), np.where(inf, 0, ref)
    pair = np.sqrt(r[..., 0::2].astype(np.float64) ** 2 + r[..., 1::2] ** 2).repeat(2, axis=-1)
    tol = pair * ulps * 2.0 ** -10 + 2.0 ** -24
    worst = float(np.max(np.abs(g.astype(np.float64) - r) / tol))
    assert worst <= 1.0, f"{what}: worst deviation {worst:.2f} x the bound"
    same = float(np.mean(got == ref))
    assert same >= 0.999, f"{what}: only {same:.5f} of the elements identical"


# ------------------------------------------------------------------------------------------- fp16 restatements
# oracle/prep_oracle.py restates the sequence in bf16; these are the same functions in kernel 0's order with every
# rounding to fp16 (its reduction helpers are reused unchanged).
def f16_round(x):
    """fp32 -> nearest-even float16, returned as fp32: overflow gives +-inf (as .to(torch.float16)), and values below
    2^-14 become fp16 subnormals, not zeros."""
    with np.errstate(over="ignore"):
        return np.asarray(x, dtype=np.float32).astype(np.float16).astype(np.float32)


def _rms_apply(x, rinv, weight):
    """diffusers RMSNorm after the statistic: x * rinv rounded to the weight's dtype, times the weight, rounded."""
    xn = f16_round((np.asarray(x, np.float32) * rinv[..., None]).astype(np.float32))
    return f16_round((xn * np.asarray(weight, np.float32)).astype(np.float32))


def _rinv(var, eps):
    return (1.0 / np.sqrt(var.astype(np.float64) + np.float64(np.float32(eps)))).astype(np.float32)


def rms_norm_f16(x, weight, eps):
    """RMSNorm(128) per head: mean(x^2) in kernel 0's order (prep_oracle.mean_square_kernel_order)."""
    return _rms_apply(x, _rinv(PO.mean_square_kernel_order(x), eps), weight)


def rms_norm_across_heads_f16(x, weight, eps):
    """Wan: RMSNorm over all heads*128 channels of a token, in row_rms_kernel's order."""
    return _rms_apply(x, _rinv(PO.mean_square_row_kernel_order(x), eps), weight)


def layer_norm_f16(x, weight, bias, eps):
    """torch.nn.LayerNorm(D), D = 128 or 64, in kernel 0's order (per lane a sequential sum of its 8 columns, a butterfly
    over the D / 8 lanes of the head; two-pass variance), statistics and affine in fp32, one rounding."""
    x = np.asarray(x, dtype=np.float32)
    d_ = x.shape[-1]
    n = d_ // 8
    lanes = x.reshape(*x.shape[:-1], n, 8)
    sm = np.zeros(lanes.shape[:-1], dtype=np.float32)
    for c in range(8):
        sm = (sm + lanes[..., c]).astype(np.float32)
    o = 1
    while o < n:
        sm = (sm + sm[..., np.arange(n) ^ o]).astype(np.float32)
        o <<= 1
    mean = (sm[..., 0] * np.float32(1.0 / d_)).astype(np.float32)
    d = (lanes - mean[..., None, None]).astype(np.float32)
    ss = np.zeros(lanes.shape[:-1], dtype=np.float32)
    for c in range(8):
        ss = PO._fma32(d[..., c], d[..., c], ss)
    o = 1
    while o < n:
        ss = (ss + ss[..., np.arange(n) ^ o]).astype(np.float32)
        o <<= 1
    var = (ss[..., 0] * np.float32(1.0 / d_)).astype(np.float32)
    t = (d.reshape(x.shape) * _rinv(var, eps)[..., None]).astype(np.float32)
    return f16_round(PO._fma32(np.broadcast_to(np.asarray(weight, np.float32), x.shape), t,
                               np.broadcast_to(np.asarray(bias, np.float32), x.shape)))


def rotary_f16(x, cos, sin):
    """x [..., S, D], cos / sin [S, D] fp32: two fp32 products and a sum, rounded once to fp16."""
    x = np.asarray(x, np.float32)
    rot = np.empty_like(x)
    rot[..., 0::2] = -x[..., 1::2]
    rot[..., 1::2] = x[..., 0::2]
    return f16_round(((x * cos).astype(np.float32) + (rot * sin).astype(np.float32)).astype(np.float32))


def prep_f16(src, heads, hd=128, weight=None, eps=1e-6, cos=None, sin=None, rope_rows=0, bias=None):
    """src [B, rows, heads*hd] -> [B, heads, rows, hd]: RMSNorm across heads (weight [heads*128], before the split), head
    split, per-head RMSNorm (weight [hd]) or LayerNorm (weight and bias), rotary embedding on the first rope_rows rows."""
    b, rows, _ = src.shape
    src = np.asarray(src, np.float32)
    if weight is not None and np.asarray(weight).size == heads * 128 and bias is None:
        src = rms_norm_across_heads_f16(src, weight, eps)
        weight = None
    x = src.reshape(b, rows, heads, hd).transpose(0, 2, 1, 3)
    if weight is not None and bias is not None:
        x = layer_norm_f16(x, weight, bias, eps)
    elif weight is not None:
        x = rms_norm_f16(x, weight, eps)
    if rope_rows:
        x = x.copy()
        x[:, :, :rope_rows] = rotary_f16(x[:, :, :rope_rows], cos[:rope_rows], sin[:rope_rows])
    return x


FORMS = ["none", "rms", "wan_complex", "wan_cos_sin", "layer128", "layer64"]


def _case(form, batch, heads, rows, n_rope, seed, device="cpu"):
    """fp16 sources, fp16 norm parameters and rotary tables of one form.  Returns a dict: src (3 tensors
    [B, rows, H*D]), hd, the qkv_prep keyword arguments (kw), and per tensor the oracle's and PyTorch's q / k."""
    hd = 64 if form == "layer64" else 128
    g = torch.Generator().manual_seed(seed)
    src = [torch.randn(batch, rows, heads * hd, generator=g).mul(1.5).to(F16) for _ in range(3)]
    wan = form.startswith("wan")
    nw = heads * 128 if wan else hd
    w = [(1 + 0.1 * torch.randn(nw, generator=g)).to(F16) for _ in range(2)]
    bias = [(0.05 * torch.randn(hd, generator=g)).to(F16) for _ in range(2)]
    if wan:
        n_rope = rows
    ang = torch.outer(torch.arange(n_rope, dtype=torch.float64), 1.0 / (256.0 ** (torch.arange(0, hd, 2) / hd)))
    cos = ang.cos().float().repeat_interleave(2, dim=1)
    sin = ang.sin().float().repeat_interleave(2, dim=1)
    kw = dict(eps=1e-6)
    if form == "wan_complex":                       # Wan2.1: complex freqs, multiplied in float64
        emb = torch.polar(torch.ones_like(ang), ang)[None, None]
        kw.update(rope=(cos, sin))
    elif form == "wan_cos_sin":                     # Wan2.2: interleaved cos / sin tables [1, S, 1, 128]
        emb = (cos[None, :, None], sin[None, :, None])
        kw.update(rope=(cos, sin))
    else:
        emb = None
        kw.update(rope=(cos, sin), rope_rows=n_rope)
    out = dict(src=src, hd=hd, kw=kw, oracle=[], torch=[])
    for i in range(2):
        x = src[i]
        xn = x.float().numpy()
        o = prep_f16(xn, heads, hd, None if form == "none" else w[i].float().numpy(), 1e-6, cos.numpy(), sin.numpy(),
                     n_rope, bias[i].float().numpy() if form.startswith("layer") else None)
        out["oracle"].append(o)
        xd, wd, bd = x.to(device), w[i].to(device), bias[i].to(device)
        cd, sd = cos.to(device), sin.to(device)
        if form in ("none", "rms"):
            t = MG.torch_prep(xd, heads, None if form == "none" else wd, 1e-6, cd, sd, n_rope)
        elif form.startswith("layer"):
            t = MG.torch_prep_cog(xd, heads, wd, bd, 1e-6, cd, sd, n_rope)
        elif form == "wan_complex":
            t = MG.torch_prep_wan(xd, heads, wd, 1e-6, emb.to(device))
        else:
            from rectified_spaattn import _processors as P
            var = xd.to(torch.float32).pow(2).mean(-1, keepdim=True)
            y = (xd * torch.rsqrt(var + 1e-6)).to(wd.dtype) * wd
            t = P.rope_cos_sin(y.unflatten(2, (heads, -1)), *(e.to(device) for e in emb)).transpose(1, 2)
        out["torch"].append(t.float().cpu().numpy())
    if form != "none":
        kw.update(q_weight=w[0], k_weight=w[1])
    if form.startswith("layer"):
        kw.update(q_bias=bias[0], k_bias=bias[1])
    return out


# ------------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("form", FORMS)
def test_f16_restatement_matches_torch(form):
    """The fp16 restatement (prep_f16) against the literal PyTorch op sequence run in fp16 on the CPU: no norm,
    RMSNorm(128), Wan's RMSNorm across heads with both rotary forms, LayerNorm(128), LayerNorm(64); the rotary
    embedding on the first rows (Wan: all rows)."""
    c = _case(form, 2, 2, 300, 220, 61)
    for i in range(2):
        assert c["oracle"][i].shape == (2, 2, 300, c["hd"])
        assert_prep_close_f16(c["oracle"][i], c["torch"][i], f"{form} tensor {i}")


def test_f16_round_keeps_infinities_and_subnormals():
    x = np.array([65504.0, 65520.0, -1e6, 2.0 ** -20, 2.0 ** -25, 2.0 ** -24 * 1.5, 1.0 + 2.0 ** -11], np.float32)
    want = torch.from_numpy(x).to(F16).float().numpy()
    assert np.array_equal(f16_round(x), want)
    assert np.isinf(want[1]) and want[3] == 2.0 ** -20 and want[5] == 2.0 ** -23


def _desc(heads, seq, hd, dtype, geo):
    d = N.AttnDesc()
    d.batch, d.heads, d.seq, d.head_dim, d.dtype = 1, heads, seq, hd, dtype
    for name in ("q_stride", "k_stride", "v_stride", "o_stride"):
        arr = getattr(d, name)
        arr[0], arr[1], arr[2] = heads * seq * hd, seq * hd, hd
    d.family, d.n_blocks, d.nq_blocks, d.text_keys = geo.family, geo.n_blocks, geo.nq_blocks, geo.text_keys
    d.kv_len, d.kv_zero_from, d.text_end_block = geo.kv_len, geo.kv_zero_from, geo.text_end_block
    d.text_q_valid, d.top_k, d.p_remain, d.first_frame_blocks = geo.text_q_valid, 2, 0.3, geo.first_frame_blocks
    d.vis_len = geo.vis_len
    return d


def test_cabi_fp16_refusals():
    """Before any device call: an unknown dtype is refused by name (rsa_qkv_prep, rsa_qkv_prep_gather,
    rsa_row_rms_dtype); norms 0-2 at head_dim 64 are refused in fp16 with the message bf16 gets; the fp16 gather at 64
    columns refuses norm 1."""
    lib = N.lib()
    geo = G.cogvideo(1250, 226)
    p = N.PrepDesc()
    p.rows, p.dst_row = geo.seq, 0
    for t in range(3):
        p.src_stride[t][0], p.src_stride[t][1] = geo.seq * 128, 128
    r = N.PeerRoute()
    r.n_ranks, r.rank, r.rows_per_rank, r.heads_total, r.head0 = 2, 0, 625, 4, 0
    r.src_table = 16                                               # never read on the host
    r.src_stride[0], r.src_stride[1] = 625 * 4 * 64, 4 * 64
    d = _desc(2, geo.seq, 64, 7, geo)
    p.norm = 3
    assert lib.rsa_qkv_prep(C.byref(p), C.byref(d), 16, 16, 16, 16, 16, 16, 0, None, 0, None) == -2
    assert b"dtype 7" in lib.rsa_last_error_string()
    assert lib.rsa_qkv_prep_gather(C.byref(p), C.byref(d), C.byref(r), 16, 16, 16, 0, None, 0, None) == -2
    assert b"dtype 7" in lib.rsa_last_error_string()
    st = (C.c_int64 * 2)(1024, 1024)
    assert lib.rsa_row_rms_dtype(16, 16, 1, 8, 1024, st, st, 1e-6, 16, 16, 7, None) == -2
    assert b"dtype 7" in lib.rsa_last_error_string()
    for norm in (0, 1, 2):
        p.norm = norm
        msgs = []
        for dt in (N.DTYPE_BF16, N.DTYPE_F16):
            d = _desc(2, geo.seq, 64, dt, geo)
            assert lib.rsa_qkv_prep(C.byref(p), C.byref(d), 16, 16, 16, 16, 16, 16, 0, None, 0, None) == -2
            msgs.append(lib.rsa_last_error_string())
        assert msgs[0] == msgs[1] and b"head_dim 64" in msgs[1] and f"norm {norm}".encode() in msgs[1], msgs
    p.norm = 1
    d = _desc(2, geo.seq, 64, N.DTYPE_F16, geo)
    assert lib.rsa_qkv_prep_gather(C.byref(p), C.byref(d), C.byref(r), 16, 16, 16, 0, None, 0, None) == -2
    msg = lib.rsa_last_error_string()
    assert b"norm 1" in msg and b"dtype" not in msg, msg


def test_fused_ulysses_refuses_other_dtypes():
    """FusedUlysses takes bf16 or fp16; any other dtype is refused before any collective or CUDA call."""
    geo = G.wan(1000)
    for dt in (torch.float32, torch.float64, torch.int16):
        with pytest.raises(ValueError, match="dtype"):
            parallel.FusedUlysses(1, 2, geo, 2, 0.3, dtype=dt)


# ------------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


@pytest.mark.gpu
@pytest.mark.parametrize("compact", [True, False])
@pytest.mark.parametrize("form", FORMS)
def test_kernel0_fp16_against_oracle_and_torch(dev, monkeypatch, form, compact):
    """Kernel 0 in fp16, every norm form, both rotary-table forms: batch 2, 3 heads (odd: at 64 columns the last head
    pair is half empty), 1000 rows (not a multiple of 128), rotary embedding on the first 870 (Wan: all).  q and k meet
    the fp16 bar against the fp16 oracle and against PyTorch's sequence on the GPU; v is copied bit for bit."""
    monkeypatch.setattr(ops, "COMPACT_ROPE", compact)
    b, heads, rows = 2, 3, 1000
    c = _case(form, b, heads, rows, 870, 71, dev)
    hd = c["hd"]
    q, k, v = (torch.full((b, heads, rows, hd), float("nan"), dtype=F16, device=dev) for _ in range(3))
    plan = ops.Plan(q, k, v, G.wan(rows), 1, 0.3, None)
    kw = {n: (tuple(t.to(dev) for t in x) if isinstance(x, tuple) else (x.to(dev) if torch.is_tensor(x) else x))
          for n, x in c["kw"].items()}
    src = [t.to(dev) for t in c["src"]]
    with pytest.raises(RuntimeError, match="allow_fp16"):              # opt-in: without it an fp16 plan is refused
        plan.qkv_prep(*src, pool=False, **kw)
    with pytest.raises(RuntimeError, match="torch.bfloat16 but the plan is torch.float16"):
        plan.qkv_prep(src[0].to(torch.bfloat16), *src[1:], pool=False, allow_fp16=True, **kw)
    plan.qkv_prep(*src, pool=False, allow_fp16=True, **kw)
    torch.cuda.synchronize()
    ulps = 2 if form in ("rms", "wan_complex", "wan_cos_sin") else 1
    for i, (name, got) in enumerate((("q", q), ("k", k))):
        g = got.float().cpu().numpy()
        assert_prep_close_f16(g, c["oracle"][i], f"{form} {name} vs oracle", ulps)
        assert_prep_close_f16(g, c["torch"][i], f"{form} {name} vs torch", ulps)
    want_v = src[2].view(b, rows, heads, hd).transpose(1, 2)
    assert torch.equal(v.view(torch.int16), want_v.contiguous().view(torch.int16))


@pytest.mark.gpu
def test_kernel0_fp16_overflow_is_inf(dev):
    """Norm 0 with the rotary embedding on inputs near 6.5e4: x cos - y sin leaves fp16's range for many pairs, and
    kernel 0 stores +-inf exactly where PyTorch's .to(torch.float16) does (no saturation); every finite value equal."""
    heads, rows = 2, 256
    g = torch.Generator(device=dev).manual_seed(5)
    src = [((torch.rand(1, rows, heads * 128, generator=g, device=dev) * 2 - 1) * 65504).to(F16) for _ in range(3)]
    ang = torch.full((rows, 64), 0.7, device=dev) + 0.1 * torch.rand(rows, 64, generator=g, device=dev)
    cos, sin = ang.cos().repeat_interleave(2, 1).contiguous(), ang.sin().repeat_interleave(2, 1).contiguous()
    q, k, v = (torch.empty(1, heads, rows, 128, dtype=F16, device=dev) for _ in range(3))
    plan = ops.Plan(q, k, v, G.wan(rows), 1, 0.3, None)
    plan.qkv_prep(*src, rope=(cos, sin), rope_rows=rows, pool=False, allow_fp16=True)
    want = MG.torch_prep(src[0], heads, None, 1e-6, cos, sin, rows)
    torch.cuda.synchronize()
    assert torch.isinf(want).sum().item() > 1000
    assert torch.equal(torch.isinf(q), torch.isinf(want)) and not torch.isnan(q).any()
    assert torch.equal(q.view(torch.int16), want.contiguous().view(torch.int16))


@pytest.mark.gpu
@pytest.mark.parametrize("hd", [128, 64])
def test_kernel0_fp16_layer_norm_keeps_subnormals(dev, hd):
    """LayerNorm with a weight of 2^-16 (itself an fp16 subnormal): outputs fall below 2^-14 and are stored as fp16
    subnormals, identical to PyTorch's within one subnormal step and never flushed to zero."""
    heads, rows = 2, 512
    g = torch.Generator(device=dev).manual_seed(9)
    src = [torch.randn(1, rows, heads * hd, generator=g, device=dev).to(F16) for _ in range(3)]
    w = torch.full((hd,), 2.0 ** -16, device=dev).to(F16)
    bias = torch.zeros(hd, device=dev).to(F16)
    q, k, v = (torch.empty(1, heads, rows, hd, dtype=F16, device=dev) for _ in range(3))
    plan = ops.Plan(q, k, v, G.wan(rows), 1, 0.3, None)
    plan.qkv_prep(*src, q_weight=w, k_weight=w, q_bias=bias, k_bias=bias, eps=1e-6, pool=False, allow_fp16=True)
    want = MG.torch_prep_cog(src[0], heads, w, bias, 1e-6, None, None, 0)
    torch.cuda.synchronize()
    got, ref = q.float().cpu().numpy(), want.float().cpu().numpy()
    sub = (ref != 0) & (np.abs(ref) < 2.0 ** -14)
    assert sub.mean() > 0.9
    assert not ((got == 0) & (ref != 0)).any(), "subnormal results flushed to zero"
    assert_prep_close_f16(got, ref, f"LayerNorm({hd}) subnormals")


def _walk_sources(b, heads, s, hd, dev, seed):
    """fp16 projection outputs with video-like block structure (a random walk of block means under iid noise)."""
    g = torch.Generator(device=dev).manual_seed(seed)
    nb = (s + 127) // 128
    out = []
    for i in range(3):
        x = torch.randn(b, nb * 128, heads * hd, generator=g, device=dev)
        if i < 2:
            mu = torch.cumsum(torch.randn(b, nb, heads * hd, generator=g, device=dev) * 0.35, dim=1)
            x += mu.repeat_interleave(128, dim=1)
        out.append(x[:, :s].to(F16).contiguous())
    return out


def _params(n, dev, seed, bias=False):
    g = torch.Generator(device=dev).manual_seed(seed)
    w = [(1 + 0.1 * torch.randn(n, generator=g, device=dev)).to(F16) for _ in range(2)]
    if not bias:
        return dict(q_weight=w[0], k_weight=w[1], eps=1e-6)
    b = [(0.05 * torch.randn(n, generator=g, device=dev)).to(F16) for _ in range(2)]
    return dict(q_weight=w[0], k_weight=w[1], q_bias=b[0], k_bias=b[1], eps=1e-6)


def _rope(n, hd, dev):
    ang = torch.outer(torch.arange(n, dtype=torch.float32, device=dev), 1.0 / (256.0 ** (torch.arange(0, hd, 2, device=dev) / hd)))
    return ang.cos().repeat_interleave(2, 1).contiguous(), ang.sin().repeat_interleave(2, 1).contiguous()


def _pools_like_kernel2(plan, hd):
    """The statistics kernel 0 left (workspace NaN-filled first), then run_pooled; then Plan.run, whose kernel 2 pools
    the stored rows: statistics and outputs bit-identical."""
    names = ("q_pool", "q_mad", "k_cat", "k_mad", "v_pool")
    fused = {n: plan.view()[n].clone() for n in names}
    out_pooled = plan.run_pooled().clone()
    out_whole = plan.run().clone()
    torch.cuda.synchronize()
    separate = plan.view()
    for n in names:
        assert torch.equal(fused[n].view(torch.int32), separate[n].view(torch.int32)), n
        if hd == 64:
            assert not fused[n][..., 64:].any(), n
    assert torch.equal(out_pooled.view(torch.int16), out_whole.view(torch.int16))
    assert out_whole.float().abs().max().item() > 0 and not torch.isnan(out_whole).any()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["hunyuan", "hunyuan_ragged", "wan", "cog_small", "cogvideox-2b"])
def test_kernel0_fp16_pools_like_kernel2(dev, shape):
    """Kernel 0's fp16 pooled statistics are kernel 2's on the stored fp16 rows, bit for bit, and Plan.run_pooled
    after it equals Plan.run: HunyuanVideo form (RMSNorm, latent rows at dst_row 0, text rows at the visual token
    count), its ragged form (1000 visual tokens: two calls), Wan (RMSNorm across heads), CogVideoX small and
    CogVideoX-2B's full shape (13 x 30 x 45 + 226 = 17 776 tokens, 30 heads x 64, LayerNorm, no rotary embedding;
    pooled as one segment: the CogVideoX block geometry has no layout for 17 550 visual tokens in front of the text).
    The stored q of the HunyuanVideo forms meets the bar against the fp16 oracle."""
    if shape.startswith("hunyuan"):
        nv, text, heads, hd = (1024 if shape == "hunyuan" else 1000), 256, 3, 128
        s = nv + text
        geo, nbr, top_k = G.hunyuan(s, nv + 200, text), None, 2
    elif shape == "wan":
        s, heads, hd = 1035, 3, 128
        geo, nbr, top_k = G.wan(s, 2), None, 2
    else:
        (t, h, w), heads, top_k = ((4, 16, 16), 3, 2) if shape == "cog_small" else ((13, 30, 45), 30, 30)
        nv, text, hd = t * h * w, 226, 64
        s = nv + text
        geo = G.cogvideo(s, text) if shape == "cog_small" else G.wan(s)
        nbr = ops.gilbert_block_neighbors(t, h, w) if shape == "cog_small" else None
    src = _walk_sources(1, heads, s, hd, dev, 5)
    q, k, v = (torch.empty(1, heads, s, hd, dtype=F16, device=dev) for _ in range(3))
    plan = ops.Plan(q, k, v, geo, top_k, 0.3, nbr, private_workspace=True)
    plan.ws.view(torch.uint8).fill_(0xff)
    if shape.startswith("hunyuan"):
        prm = _params(128, dev, 6)
        rope = _rope(nv, 128, dev)
        plan.qkv_prep(*(x[:, :nv] for x in src), dst_row=0, rope=rope, allow_fp16=True, **prm)
        plan.qkv_prep(*(x[:, nv:] for x in src), dst_row=nv, allow_fp16=True, **prm)
        _pools_like_kernel2(plan, hd)
        w = prm["q_weight"].float().cpu().numpy()
        sn = src[0].float().cpu().numpy()
        cos, sin = (x.cpu().numpy() for x in rope)
        want = np.concatenate([prep_f16(sn[:, :nv], heads, 128, w, 1e-6, cos, sin, nv),
                               prep_f16(sn[:, nv:], heads, 128, w, 1e-6)], axis=2)
        assert_prep_close_f16(q.float().cpu().numpy(), want, shape, ulps=2)
    elif shape == "wan":
        plan.qkv_prep(*src, rope=_rope(s, 128, dev), allow_fp16=True, **_params(heads * 128, dev, 6))
        _pools_like_kernel2(plan, hd)
    else:
        rope = _rope(nv, 64, dev) if shape == "cog_small" else None     # CogVideoX-2B has no rotary embedding
        plan.qkv_prep(*src, rope=rope, rope_rows=nv if rope else None, allow_fp16=True, **_params(64, dev, 6, bias=True))
        _pools_like_kernel2(plan, hd)


# ------------------------------------------------------------------------------------- processors on the GPU
def _close(a, b):
    a, b = a.float().cpu().numpy(), b.float().cpu().numpy()
    assert np.isfinite(a).all()
    assert cos_sim(a, b) >= 0.999 and abs(a - b).max() <= 4e-2 * max(1.0, abs(b).max())


def _mk(dev, *a, **kw):
    torch.manual_seed(0)
    return FakeAttention(*a, **kw).to(dev).to(F16)


@pytest.fixture
def prep_calls(monkeypatch):
    """Counts kernel-0 calls on fp16 plans: a processor test must see the fused path taken, not the op-by-op one."""
    n = [0]
    orig = ops.Plan.qkv_prep

    def counted(self, *a, **kw):
        if self.q.dtype == F16:
            n[0] += 1
        return orig(self, *a, **kw)

    monkeypatch.setattr(ops.Plan, "qkv_prep", counted)
    return n


def _families(dev):
    """(name, make(mode, dense_call) -> processor, call(processor) -> output, reference processor for SDPA) of every
    family on small fp16 layers; top_k 99 puts the sparse calls in the dense limit."""
    from rectified_spaattn import rectified_cogvideo_attn as cog
    from rectified_spaattn import rectified_flux_attn as flux
    from rectified_spaattn import rectified_hunyuan_attn as hun
    from rectified_spaattn import rectified_wan21_attn as wan21
    from rectified_spaattn import rectified_wan22_attn as wan22
    dim, heads, s, nv = 256, 2, 1000, 1024
    g = torch.Generator(device=dev).manual_seed(1)
    ang = torch.rand(nv + 512, 64, generator=g, device=dev) * 6.28
    cos, sin = ang.cos().repeat_interleave(2, 1), ang.sin().repeat_interleave(2, 1)
    x_w = torch.randn(1, s, dim, generator=g, device=dev).to(F16)
    x = torch.randn(1, nv, dim, generator=g, device=dev).to(F16)
    out = []
    a_w = _mk(dev, dim, heads, norm="inner")
    emb21 = torch.polar(torch.ones_like(ang[:s], dtype=torch.float64), ang[:s].double())[None, None]
    def wan(cls):
        def make(mode, dense):                      # step 0 is a warm-up (dense) call, step 20 a sparse one
            pr = cls(mode, 99, None, 0.3, processor_id=5, first_frame_blocks=2)
            pr.current_step = 0 if dense else 20
            return pr
        return make
    out.append(("wan2.1", wan(wan21.RectifiedWanT2VSpaAttnProcessor2_0), lambda pr: pr(a_w, x_w, None, None, emb21)))
    emb22 = (cos[None, :s, None], sin[None, :s, None])
    out.append(("wan2.2", wan(wan22.RectifiedWanTI2VSpaAttnProcessor2_0), lambda pr: pr(a_w, x_w, None, None, emb22)))
    a_h = _mk(dev, dim, heads, added=True)
    txt = torch.randn(1, 256, dim, generator=g, device=dev).to(F16)

    def make_hun(mode, dense):
        pr = hun.RectifiedHunyuanVideoSpaAttnProcessor2_0("flash" if dense and mode != "torch" else mode, 99, None, 0.3)
        pr.num_true = nv + 200
        return pr
    mask = (torch.arange(nv + 256, device=dev) < nv + 200).view(1, 1, 1, -1)
    out.append(("hunyuan", make_hun, lambda pr: pr(a_h, x, txt, mask if pr.mode != "torch" else
                                                   mask.expand(1, 1, nv + 256, nv + 256), (cos[:nv], sin[:nv]))))
    txt5 = torch.randn(1, 512, dim, generator=g, device=dev).to(F16)
    out.append(("flux", lambda mode, dense: flux.RectifiedFluxSpaAttnProcessor2_0(
        mode, 99, None, 0.3, processor_id=40 if dense else 1, text_length=512),
        lambda pr: pr(a_h, x, txt5, None, (cos, sin))))
    a_c = _mk(dev, dim, 4, head_dim=64, norm="layer")
    txt_c = torch.randn(1, 226, dim, generator=g, device=dev).to(F16)
    cos64, sin64 = ang[:nv, :32].cos().repeat_interleave(2, 1), ang[:nv, :32].sin().repeat_interleave(2, 1)

    def make_cog(mode, dense):
        pr = cog.RectifiedCogVideoXVideoSpaAttnProcessor2_0(mode, 99, None, 0.3)
        pr.current_step = 0 if dense else 5
        return pr
    out.append(("cogvideox", make_cog, lambda pr: pr(a_c, x, txt_c, None, (cos64, sin64))))
    return out


def _outputs(o):
    return o if isinstance(o, tuple) else (o,)


@pytest.mark.gpu
@pytest.mark.parametrize("dense", [False, True])
def test_processors_fp16_fused(dev, prep_calls, dense):
    """All five families on fp16 layers with fuse_prep_fp16 (and fuse_prep_dense for the dense calls: Wan warm-up,
    HunyuanVideo mode "flash", Flux block 40, CogVideoX call 0): kernel 0 runs, and the layer agrees with the same
    processor op by op and with SDPA through the same modules.  With the switch off, the output is bit-identical to
    fuse_prep = False: fp16 models keep the op-by-op path by default."""
    for name, make, call in _families(dev):
        outs = {}
        for variant in ("fp16", "default", "unfused", "sdpa"):
            pr = make("torch" if variant == "sdpa" else "sparse", dense)
            pr.fuse_prep = variant != "unfused"
            pr.fuse_prep_dense = dense and variant != "unfused"
            pr.fuse_prep_fp16 = variant == "fp16"
            before = prep_calls[0]
            with torch.no_grad():
                outs[variant] = _outputs(call(pr))
            assert (prep_calls[0] > before) == (variant == "fp16"), (name, variant)
        for a, b, c, d in zip(outs["fp16"], outs["default"], outs["unfused"], outs["sdpa"]):
            n_ok = 200 if name == "hunyuan" and a.shape[1] == 256 else a.shape[1]    # padded text rows: undefined
            assert a.dtype == F16
            _close(a[:, :n_ok], c[:, :n_ok])
            _close(a[:, :n_ok], d[:, :n_ok])
            assert torch.equal(b.view(torch.int16), c.view(torch.int16)), name


@pytest.mark.gpu
def test_bf16_norm_weights_under_fp16_activations_stay_op_by_op(dev):
    """Norm parameters must have the activations' dtype: diffusers rounds a bf16 weight's product elsewhere, so an fp16
    layer with bf16 norm weights is not fused even with fuse_prep_fp16 (the gates return None)."""
    from rectified_spaattn import _processors as P
    from rectified_spaattn import rectified_wan21_attn as wan21
    attn = _mk(dev, 256, 2, head_dim=64, norm="layer")
    attn.norm_q.to(torch.bfloat16)
    hs = torch.randn(1, 1250, 256, device=dev).to(F16)
    with torch.no_grad():
        assert P.fused_prep_attention(attn, hs, None, G.cogvideo(1250, 226), 2, 0.3, None, None, rope_text=False,
                                      fp16=True) is None
        attn.norm_q.to(F16)
        assert P.fused_prep_attention(attn, hs, None, G.cogvideo(1250, 226), 2, 0.3, None, None, rope_text=False,
                                      fp16=True) is not None
        assert P.fused_prep_attention(attn, hs, None, G.cogvideo(1250, 226), 2, 0.3, None, None,
                                      rope_text=False) is None                      # the switch off: not fused
        a_w = _mk(dev, 256, 2, norm="inner")
        a_w.norm_k.to(torch.bfloat16)
        pr = wan21.RectifiedWanT2VSpaAttnProcessor2_0("sparse", 2, None, 0.3, processor_id=3)
        x = torch.randn(1, 1000, 256, device=dev).to(F16)
        assert pr._fused(a_w, x, None, None, fp16=True) is None
        a_w.norm_k.to(F16)
        assert pr._fused(a_w, x, None, None, fp16=True) is not None


@pytest.mark.gpu
def test_fp16_cogvideox_layer_records_into_a_cuda_graph(dev):
    """A whole fp16 CogVideoX attention layer through kernel 0 at 64 columns (sparse, top_k 2) records into one CUDA
    graph and replays on new inputs with the eager result, bit for bit."""
    from rectified_spaattn import rectified_cogvideo_attn as cog
    attn = _mk(dev, 256, 4, head_dim=64, norm="layer")
    pr = cog.RectifiedCogVideoXVideoSpaAttnProcessor2_0("sparse", 2, None, 0.3)
    pr.current_step, pr.fuse_prep_fp16 = 5, True
    nv = 1024
    rope = _rope(nv, 64, dev)
    g = torch.Generator(device=dev).manual_seed(3)
    mu = torch.cumsum(torch.randn(nv // 128, 256, generator=g, device=dev) * 0.35, dim=0).repeat_interleave(128, dim=0)
    xs = [(torch.randn(nv, 256, generator=g, device=dev) + mu)[None].to(F16) for _ in range(2)]
    ts = [torch.randn(1, 226, 256, generator=g, device=dev).to(F16) for _ in range(2)]
    with torch.no_grad():
        eager = [pr(attn, x, t, None, rope) for x, t in zip(xs, ts)]
        x_in, t_in = xs[0].clone(), ts[0].clone()
        stream = torch.cuda.Stream()
        stream.wait_stream(torch.cuda.current_stream())
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.stream(stream):
            pr(attn, x_in, t_in, None, rope)
            stream.synchronize()
            with torch.cuda.graph(graph, stream=stream):
                h_out, e_out = pr(attn, x_in, t_in, None, rope)
        for x, t, ref in zip(xs, ts, eager):
            x_in.copy_(x)
            t_in.copy_(t)
            graph.replay()
            torch.cuda.synchronize()
            assert torch.equal(h_out, ref[0]) and torch.equal(e_out, ref[1])


# ------------------------------------------------------------------------------------------ fused Ulysses in fp16
def _ulysses(n, workload, dense, port):
    args = [workload, "--dtype", "float16"] + (["--dense"] if dense else [])
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n),
                        "--master-addr", "127.0.0.1", "--master-port", str(port),
                        os.path.join(REPO, "tools", "check_fused_ulysses.py")] + args,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["dtype"] == "float16" and line["dense"] is dense and line["n_gpus"] == n
    return line


@pytest.mark.gpu
@pytest.mark.parametrize("dense", [False, True])
@pytest.mark.parametrize("workload", ["cog", "odd"])
def test_fused_ulysses_fp16_one_rank(dev, workload, dense):
    """FusedUlysses(dtype=torch.float16) on one rank: the gather inside kernel 0 and the scatter inside kernel 4's
    epilogue run over the (own) peer buffers, and the result is bit-identical to the single-GPU kernel 0 + attention
    call, sparse and dense: CogVideoX form (64-column heads, LayerNorm) and Wan form (RMSNorm across heads)."""
    port = {("cog", False): 29611, ("cog", True): 29612, ("odd", False): 29613, ("odd", True): 29614}[workload, dense]
    line = _ulysses(1, workload, dense, port)
    assert line["fused_equals_single_gpu_bitwise_checked_ranks"] == [True]


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["cog", "odd"])
def test_fused_ulysses_fp16_two_gpus(dev, workload):
    """The fp16 fused exchange on 2 GPUs, uneven token and head shards: every rank's rows bit-identical to the
    single-GPU call (CogVideoX form; Wan form with the statistic across heads from rsa_row_rms_dtype)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    line = _ulysses(2, workload, False, {"cog": 29615, "odd": 29616}[workload])
    assert line["fused_equals_single_gpu_bitwise_checked_ranks"] == [True, True]
