"""Kernel 4 (`attn_tc5_kernel`, csrc/attn_tc5.cu) against a float64 reference with a per-element error bound derived
from the kernel's arithmetic, at the inputs where a flash-attention kernel goes wrong: one-hot rows, row maxima that grow
by more than the lazy-rescale threshold at every block (and by so much that the rescale factor underflows), a first
block that makes every later weight underflow, exact ties, and keys at or past kv_len that would win their row.

The kernel computes, per 128-key block of a row, S = q^ k^T in fp32 (log2 units), p = 2^(S - m) with the running maximum
m raised lazily, P = dtype(p), l += p (unrounded), O += P V in fp32, and at the end dtype(O / l).  Relative to the float64
result ref = sum p v / sum p that gives, for element (i, c),

    |out - ref| <= u_o |ref| + (2 u_P + e_exp + 2 delta_i) A_ic + 2^-24,     A_ic = sum_j p_ij |v_jc| / sum_j p_ij

u_o, u_P: unit roundoff of the output / P dtype (2^-8 bf16, 2^-11 fp16); e_exp: relative error of the exponential
(2^-21 for MUFU ex2, 7.5e-5 for the FMA-pipe polynomial exp2_poly2); delta_i = ln2 * D * 2^-24 * max_j sum_d |q^_id k_jd|:
the fp32 accumulation of S, turned into a relative error of p.  The numerator and l each see e_exp and delta once; the
second u_P covers what is left: fp32 rounding of s * scale - m (|x| <= thr for every weight that is not negligible:
<= 2^-18 relative), of the rescale factor and of O's accumulation over at most a few thousand keys, all below 2^-12,
and P values that underflow (2^-24 absolute for fp16, under 2^-125 for bf16).

q^ is the query as the kernel multiplies it: q~ = dtype(fp32(q * sigma)) on the masked entry's default path (q_round = 1,
the reference Triton kernel's rounding), sigma * q with the fp32 scores scaled instead (fp32_scale=True and
dense_attention, flash-attn's arithmetic); sigma = fp32(D^-1/2 * 1.44269504).

The instantiations that only RSA_TC5_POLY / RSA_TC5_THR select run in a child process (`python <this file> --leg NAME`)
that runs the same matrix and prints one JSON line.  Which instantiation ran is read from the CUDA kernel names in
torch.profiler, not inferred from the dispatch code."""
import json
import math
import os
import re
import subprocess
import sys
import time
import zlib

import numpy as np
import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if __name__ == "__main__":   # a leg: the child process is not started by pytest, so set the path conftest.py sets
    for _p in (REPO, os.path.join(REPO, "rectified-spaattn_b200"), os.path.join(REPO, "tests")):
        if _p not in sys.path:
            sys.path.insert(0, _p)

BF16, FP16 = torch.bfloat16, torch.float16
UNIT = {BF16: 2.0 ** -8, FP16: 2.0 ** -11}
E_MUFU, E_POLY = 2.0 ** -21, 7.5e-5
LN2 = math.log(2.0)


def sigma(d):
    """The kernel's scale_log2 (rsa_api.cu): fp32(D^-1/2 * 1.44269504)."""
    return float(np.float32((1.0 / math.sqrt(d)) * 1.44269504))


def rescale_threshold(dtype):
    """The lazy-rescale threshold kernel 4 runs with (attention_rescale_threshold, rsa_api.cu): RSA_TC5_THR in [0, 64],
    else 32; at most 8 for fp16, whose P must stay below 2^16."""
    e = os.environ.get("RSA_TC5_THR")
    try:
        v = float(e) if e is not None else 32.0
    except ValueError:
        v = 32.0
    if not 0.0 <= v <= 64.0:
        v = 32.0
    return min(v, 8.0) if dtype == FP16 else v


# ------------------------------------------------------------------------------------------------ reference
def allowed_keys(b, h, s, skv, kv_len, keep, device):
    """bool [B, H, S, S_kv]: key j is attended by row i (j < kv_len and, with a block mask, block (i/128, j/128) kept)."""
    a = (torch.arange(skv, device=device) < kv_len).expand(b, h, s, skv)
    if keep is not None:
        a = a & keep.to(device).repeat_interleave(128, 2)[:, :, :s].repeat_interleave(128, 3)[:, :, :, :skv]
    return a


def reference(q, k, v, kv_len, q_round, keep=None):
    """float64 attention with the kernel's scale and query rounding -> (ref, A, delta), each float64 on q's device; ref
    and A are [B, H, S, D], delta [B, H, S, 1].  Rows without an attended key are zero (the kernel writes zeros)."""
    b, h, s, d = q.shape
    skv = k.shape[2]
    sg = sigma(d)
    qh = (q.float() * sg).to(q.dtype).double() if q_round else q.double() * sg
    kd, vd = k.double(), v.double()
    ok = allowed_keys(b, h, s, skv, kv_len, keep, q.device)
    t = (qh @ kd.transpose(-1, -2)).masked_fill(~ok, -math.inf)
    m = t.amax(-1, keepdim=True)
    p = torch.exp2(t - torch.where(torch.isfinite(m), m, torch.zeros_like(m)))
    p = torch.where(ok, p, torch.zeros_like(p))
    lsum = p.sum(-1, keepdim=True)
    inv = torch.where(lsum > 0, 1.0 / lsum.clamp_min(1e-300), torch.zeros_like(lsum))
    ref = (p @ vd) * inv
    A = (p @ vd.abs()) * inv
    mag = (qh.abs() @ kd.abs().transpose(-1, -2)).masked_fill(~ok, 0.0)
    delta = LN2 * d * 2.0 ** -24 * mag.amax(-1, keepdim=True)
    return ref, A, delta


def error_bound(ref, A, delta, dtype, e_exp):
    u = UNIT[dtype]
    return u * ref.abs() + (2 * u + e_exp + 2 * delta) * A + 2.0 ** -24


def worst_ratio(out, ref, A, delta, dtype, e_exp):
    """max |out - ref| / bound over the elements (inf when out is not finite)."""
    o = out.double()
    if not torch.isfinite(o).all():
        return math.inf
    return float(((o - ref).abs() / error_bound(ref, A, delta, dtype, e_exp)).max())


# ------------------------------------------------------------------------------------------------ regimes
REGIMES = ("diffuse", "peaked", "rising", "rising126", "falling", "ties", "pad")


def make_inputs(regime, b, h, s, skv, d, kv_len, dtype, seed, device, strided=False):
    """q [B,H,S,D], k / v [B,H,S_kv,D] in `dtype`, from a fixed seed.  strided: [B,S,H,D] storage viewed as [B,H,S,D]."""
    g = torch.Generator(device=device).manual_seed(seed)
    q = torch.randn(b, h, s, d, generator=g, device=device)
    k = torch.randn(b, h, skv, d, generator=g, device=device)
    v = torch.randn(b, h, skv, d, generator=g, device=device)
    sg, half = sigma(d), d // 2
    if regime == "peaked":
        # t = sigma q.k has standard deviation 1.4427 c^2 when q and k are N(0, c^2): c^2 = 69 spans about +-300
        q, k = q * 8.3, k * 8.3
    elif regime in ("rising", "rising126"):
        # even rows: q = e_c, c = (row / 2) mod D/2; in key block j the keys at even in-block positions are g_j e_c, so the
        # row maximum grows by `step` per block (thr + 8, or 130 so that the rescale factor 2^-130 underflows).  Odd rows
        # and the other keys live on the other half of the columns: diffuse, and orthogonal to the aligned keys.
        step = rescale_threshold(dtype) + 8.0 if regime == "rising" else 130.0
        rows = torch.arange(s, device=device)
        q[..., :half] = 0.0
        even = rows % 2 == 0
        q[:, :, even] = 0.0
        q[:, :, even, (rows[even] // 2) % half] = 1.0
        k[..., :half] = 0.0
        keys = torch.arange(skv, device=device)
        al = (keys % 128) % 2 == 0
        k[:, :, al] = 0.0
        gain = (keys[al] // 128).double() * step / sg
        k[:, :, al, ((keys[al] % 128) // 2) % half] = gain.float()
    elif regime == "falling":
        # every row's block-0 scores are > 140 above every later score: all later p are below 2^-130
        a = math.sqrt(145.0 / sg)
        q[..., 0] = a
        k[..., 0] = 0.0
        k[:, :, :128, 0] = a
    elif regime == "ties":
        q.zero_()
    elif regime == "pad":
        # keys past kv_len would win every row and carry the largest finite value
        idx = torch.arange(kv_len, skv, device=device) % s
        k[:, :, kv_len:] = 50.0 * q[:, :, idx]
        v[:, :, kv_len:] = torch.finfo(dtype).max
    q, k, v = (t.to(dtype) for t in (q, k, v))
    if strided:
        q, k, v = (t.permute(0, 2, 1, 3).contiguous().permute(0, 2, 1, 3) for t in (q, k, v))
    return q, k, v


# ------------------------------------------------------------------------------------------------ CPU emulation
def _f32(x):
    return np.asarray(x, dtype=np.float32)


def _fma32(a, b, c):
    """fp32 fma: the product of two floats is exact in float64, so one rounding after the add (double rounding of the
    float64 sum is the only deviation, at most one fp32 ulp on a handful of inputs)."""
    return _f32(np.asarray(a, np.float64) * np.asarray(b, np.float64) + np.asarray(c, np.float64))


POLY_C3, POLY_C2, POLY_C1, POLY_C0 = (np.float32(c) for c in (0.05517587438225746, 0.24261151254177094,
                                                               0.6932601928710938, 0.9999279975891113))


def exp2_poly2_emulated(x):
    """csrc/attn_tc5.cu exp2_poly2 step by step in fp32."""
    x = _f32(x)
    magic = np.float32(12582912.0)
    with np.errstate(invalid="ignore", over="ignore"):
        t = _f32(x + magic)
        r = _f32(t - magic)
        f = _fma32(r, -1.0, x)
        p = _fma32(f, POLY_C3, POLY_C2)
        p = _fma32(p, f, POLY_C1)
        p = _fma32(p, f, POLY_C0)
        bits = p.view(np.uint32) + (t.view(np.uint32) << np.uint32(23))
    return np.where(x < -125.0, np.float32(0.0), bits.view(np.float32))


def _exp2_mufu(x):
    """ex2.approx.ftz: 2^x, results below 2^-126 flushed to +0 (the 2^-22 approximation error is not modelled)."""
    y = torch.exp2(x)
    return torch.where(x < -126.0, torch.zeros_like(y), y)


def emulate(q, k, v, kv_len, q_round, thr, poly_pairs=0, keep=None, scale_error=1.0):
    """Kernel 4's arithmetic on the CPU in fp32, block by block in ascending order: lazy rescale of O and l, P rounded
    to the input dtype for the P V product while l sums the unrounded p, output dtype(O * (1 / l)).  Of every 8 score
    columns, the last 2 * poly_pairs take the polynomial exp2."""
    dtype = q.dtype
    b, h, s, d = q.shape
    skv = k.shape[2]
    sg = np.float32(sigma(d) * scale_error)
    if q_round:
        qh, scale = (q.float() * float(sg)).to(dtype).float(), np.float32(1.0)
    else:
        qh, scale = q.float(), sg
    ok = allowed_keys(b, h, s, skv, kv_len, keep, "cpu")
    m_ref = torch.full((b, h, s, 1), -math.inf)
    l = torch.zeros(b, h, s, 1)
    O = torch.zeros(b, h, s, d)
    poly_col = torch.tensor([(c % 8) // 2 >= 4 - poly_pairs for c in range(128)])
    for j0 in range(0, (kv_len + 127) // 128 * 128, 128):
        kb, vb, okb = k[:, :, j0:j0 + 128].float(), v[:, :, j0:j0 + 128].float(), ok[..., j0:j0 + 128]
        row_on = okb.any(-1, keepdim=True)
        sc = (qh @ kb.transpose(-1, -2)).masked_fill(~okb, -math.inf)
        mx = torch.from_numpy(_f32(sc.amax(-1, keepdim=True).numpy() * scale))
        first = torch.isinf(m_ref) & (m_ref < 0)
        need = ~first & (mx > m_ref + thr)
        alpha = torch.where(need, _exp2_mufu(m_ref - mx), torch.ones_like(mx))
        alpha = torch.where(row_on, alpha, torch.ones_like(alpha))
        m_ref = torch.where(row_on & (first | need), mx, m_ref)
        l, O = l * alpha, O * alpha
        x = torch.from_numpy(_fma32(sc.numpy(), scale, -m_ref.numpy()))
        p = _exp2_mufu(x)
        if poly_pairs:
            pp = torch.from_numpy(exp2_poly2_emulated(x.numpy()))
            p = torch.where(poly_col[:kb.shape[2]], pp, p)
        p = torch.where(row_on, p, torch.zeros_like(p))
        l = l + p.sum(-1, keepdim=True)
        O = O + p.to(dtype).float() @ vb
    inv = torch.where(l > 0, 1.0 / l, torch.zeros_like(l))
    return (O * inv).to(dtype)


# ------------------------------------------------------------------------------------------------ CPU tests
def test_reference_equals_float64_sdpa():
    """On fp32-scale inputs (q_round = 0) the reference is attention in float64: equal to float64 SDPA over the
    attended keys, with the kv_len cut."""
    F = torch.nn.functional
    for dtype in (BF16, FP16):
        for d in (64, 128):
            q, k, v = make_inputs("diffuse", 2, 2, 130, 300, d, 257, dtype, 3, "cpu")
            ref, _, _ = reference(q, k, v, 257, 0)
            want = F.scaled_dot_product_attention(q.double(), k[:, :, :257].double(), v[:, :, :257].double(),
                                                  scale=sigma(d) * LN2)
            assert torch.allclose(ref, want, rtol=1e-9, atol=1e-12), float((ref - want).abs().max())


def test_exp2_poly2_emulation_error_and_underflow():
    """exp2_poly2 (restated step by step in fp32) is within 7.5e-5 of 2^x relative over [-125, 64], and exactly +0 below
    -125 -- -inf, the score of a key past kv_len, included (where it once returned 2^-125)."""
    x = np.concatenate([np.linspace(-125.0, 64.0, 400001), -125.0 + np.linspace(0, 1, 1001) ** 2]).astype(np.float32)
    got = exp2_poly2_emulated(x).astype(np.float64)
    rel = np.abs(got / np.exp2(x.astype(np.float64)) - 1.0)
    assert rel.max() <= E_POLY, (float(rel.max()), float(x[np.argmax(rel)]))
    low = np.array([-np.inf, -3e38, -1e6, -200.0, -126.0, -125.5, np.nextafter(np.float32(-125), np.float32(-126))],
                   dtype=np.float32)
    out = exp2_poly2_emulated(low)
    assert np.all(out == 0.0) and not np.any(np.signbit(out)), out


EMU_SHAPE = (1, 2, 130, 300, 64)   # b, h, s, s_kv, d: two query tiles (one partial), three key blocks (one partial)


def _emu_check(regime, dtype, q_round, poly, kv_len, keep=None, **ablation):
    b, h, s, skv, d = EMU_SHAPE
    thr = rescale_threshold(dtype)
    q, k, v = make_inputs(regime, b, h, s, skv, d, kv_len, dtype, zlib.crc32(regime.encode()), "cpu")
    ref, A, delta = reference(q, k, v, kv_len, q_round, keep)
    emu_kv = kv_len + ablation.get("kv_shift", 0)
    out = emulate(q, k, v, emu_kv, q_round, thr, poly, keep, ablation.get("scale_error", 1.0))
    return worst_ratio(out, ref, A, delta, dtype, E_POLY if poly else E_MUFU)


@pytest.mark.parametrize("regime", REGIMES)
def test_emulated_kernel_meets_the_bound(regime):
    """The fp32 emulation of the kernel (bf16 / fp16 P, l from unrounded p, lazy rescale, output rounding) is within
    the bound in every regime, both query paths, with MUFU and with the polynomial, at kv_len inside a block and at
    S_kv, and with a block mask."""
    g = torch.Generator().manual_seed(5)
    keep = torch.rand(1, 2, 2, 3, generator=g) < 0.6
    keep[..., 0] = True
    for dtype in (BF16, FP16):
        for q_round in (1, 0):
            for poly in (0, 2):
                for kv_len, km in ((200, None), (300, None), (257, keep)):
                    r = _emu_check(regime, dtype, q_round, poly, kv_len, km)
                    assert r <= 1.0, (regime, dtype, q_round, poly, kv_len, km is not None, r)


def test_bound_fails_a_wrong_kernel():
    """The bound is not vacuous: the same emulation fails it with one key dropped (kv_len - 1), with the scale off by
    1 %, and with the first key past kv_len attended at full weight."""
    for dtype in (BF16, FP16):
        for q_round in (1, 0):
            assert _emu_check("ties", dtype, q_round, 0, 65, kv_shift=-1) > 1.0
            assert _emu_check("diffuse", dtype, q_round, 0, 65, scale_error=1.01) > 1.0
            assert _emu_check("pad", dtype, q_round, 0, 200, kv_shift=1) > 1.0


# ------------------------------------------------------------------------------------------------ GPU matrix
# entry -> (kind, q_round, random mask)
ENTRIES = {
    "masked_ones": ("masked", 1, False),
    "masked_random": ("masked", 1, True),
    "masked_ones_fp32": ("masked", 0, False),
    "masked_random_fp32": ("masked", 0, True),
    "dense_bhsd": ("dense", 0, False),
    "dense_bshd": ("dense", 0, False),
}
# (head_dim, attention flags): 64 with flag 4 runs the 128-column form on the same tensors
FORMS = ((128, 0), (64, 0), (64, 4))
# name -> (batch, heads, S, S_kv, kv_len, q_valid, strided)
SHAPES = {
    "1x1": (1, 1, 1, 1, 1, 1, False),
    "129": (1, 1, 129, 129, 129, 129, False),
    "383": (1, 1, 383, 383, 383, 383, False),
    "130x1000": (1, 1, 130, 1000, 1000, 130, False),
    "4224x512": (1, 1, 4224, 512, 512, 4224, False),
    **{f"kv{n}": (1, 1, 300, 300, n, 300, False) for n in (1, 63, 64, 65, 127, 128, 129, 300)},
    **{f"qv{n}": (1, 1, 300, 300, 300, n, False) for n in (1, 127, 128, 129)},
    "batch2_strided": (2, 2, 300, 300, 257, 290, True),
}
# the fourteen product instantiations of attn_tc5_kernel: (kPolyPairs, kF16, kD, kDense); the debug ones are excluded
INSTANTIATIONS = ([(p, False, 128, False) for p in range(5)] + [(0, True, 128, False)]
                  + [(p, False, 64, False) for p in range(3)] + [(1, True, 64, False)]
                  + [(0, False, 128, True), (0, True, 128, True), (1, False, 64, True), (1, True, 64, True)])
# environment-only legs: (environment, dtypes, entries, forms) -- each runs only what its variable changes
MASKED = tuple(e for e in ENTRIES if ENTRIES[e][0] == "masked")
LEGS = {
    "poly0": ({"RSA_TC5_POLY": "0"}, (BF16,), MASKED, ((64, 0),)),
    "poly1": ({"RSA_TC5_POLY": "1"}, (BF16,), MASKED, ((128, 0), (64, 4))),
    "poly2": ({"RSA_TC5_POLY": "2"}, (BF16,), MASKED, FORMS),
    "poly3": ({"RSA_TC5_POLY": "3"}, (BF16,), MASKED, ((128, 0), (64, 4))),
    "poly4": ({"RSA_TC5_POLY": "4"}, (BF16,), MASKED, ((128, 0), (64, 4))),
    "thr0": ({"RSA_TC5_THR": "0"}, (BF16, FP16), tuple(ENTRIES), FORMS),
}


def _parse_kernel(name):
    """(kPolyPairs, kF16, kD, kDense) from a demangled or mangled attn_tc5_kernel name, None for another kernel."""
    m = re.search(r"attn_tc5_kernel<([^>]*)>", name)
    if m:
        a = [x.strip().replace("(bool)", "").replace("(int)", "") for x in m.group(1).split(",")]
        tf = lambda x: x in ("true", "1")
        return None if tf(a[0]) else (int(a[1]), tf(a[2]), int(a[3]), tf(a[4]) if len(a) > 4 else False)
    m = re.search(r"attn_tc5_kernelILb(\d)ELi(\d+)ELb(\d)ELi(\d+)E(?:Lb(\d)E)?", name)
    if m:
        return None if m.group(1) == "1" else (int(m.group(2)), m.group(3) == "1", int(m.group(4)), m.group(5) == "1")
    return None


def _kernels_of(fn):
    """Runs fn under torch.profiler and returns the attn_tc5_kernel instantiations it launched."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {x for x in (_parse_kernel(e.name) for e in prof.events()) if x is not None}


def _random_keep(b, h, nq, nb, kv_len, seed, device):
    """Random block mask that keeps >= 1 attendable block per row; the partial kv_len block is kept by tiles 0 and 1
    and block 0 by tile 0 only, so the pair schedule walks the partial block first for those tiles."""
    g = torch.Generator().manual_seed(seed)
    nvalid = (kv_len + 127) // 128
    keep = torch.rand(b, h, nq, nb, generator=g) < 0.5
    keep[..., nvalid:] = False
    pick = torch.randint(0, nvalid, (b, h, nq), generator=g)
    keep.scatter_(3, pick.unsqueeze(-1), True)
    keep[:, :, :2, nvalid - 1] = True
    if nvalid > 1 and nq > 1:
        keep[:, :, 0, 0], keep[:, :, 1, 0] = True, False
    return keep.to(device)


def _call(entry, q, k, v, kv_len, q_valid, keep, pad_rows=5):
    """Kernel 4 through `entry`, with `out` a slice of a larger NaN-filled buffer -> (output [B,H,S,D], tail rows)."""
    from rsa_b200 import ops
    kind, q_round, _ = ENTRIES[entry]
    b, h, s, d = q.shape
    if entry == "dense_bshd":
        buf = torch.full((b, s + pad_rows, h, d), math.nan, dtype=q.dtype, device=q.device)
        ops.dense_attention(q, k, v, q_valid, kv_len, out=buf[:, :s])
        return buf[:, :s].permute(0, 2, 1, 3), buf[:, s:]
    buf = torch.full((b, h, s + pad_rows, d), math.nan, dtype=q.dtype, device=q.device)
    if kind == "dense":
        ops.dense_attention(q, k, v, q_valid, kv_len, out=buf[:, :, :s])
    else:
        ops.masked_attention(q, k, v, keep, kv_len, out=buf[:, :, :s], fp32_scale=q_round == 0)
    return buf[:, :, :s], buf[:, :, s:]


def _e_exp(entry, dtype, d, flags):
    """Error of the exponential for the instantiation the call reaches: any polynomial pairs -> 7.5e-5."""
    poly = os.environ.get("RSA_TC5_POLY", "")
    d_inst = 64 if d == 64 and not flags & 4 else 128
    if ENTRIES[entry][0] == "dense" or dtype == FP16:
        return E_POLY if d_inst == 64 else E_MUFU
    if d_inst == 64:
        return E_MUFU if poly in ("0", "3", "4") else E_POLY
    return E_POLY if poly in ("1", "2", "3", "4") else E_MUFU


def run_matrix(dtypes=(BF16, FP16), entries=tuple(ENTRIES), forms=FORMS, device="cuda:0"):
    """Every entry x dtype x form x shape x regime against the bound; the pad regime also against the same call with
    the padding rows of K and V zeroed (bit-identical).  -> dict of counts, failures and reached instantiations."""
    from rsa_b200 import ops
    res = {"cases": 0, "bound_failures": [], "pad_failures": [], "layout_failures": [], "kernels": set()}
    for entry in entries:
        kind, q_round, rnd = ENTRIES[entry]
        for dtype in dtypes:
            for d, flags in forms:
                ops.set_attention_flags(flags)
                try:
                    e_exp = _e_exp(entry, dtype, d, flags)
                    first = True
                    for sname, (b, h, s, skv, kv_len, q_valid, strided) in SHAPES.items():
                        if kind == "masked":
                            if sname.startswith("qv"):
                                continue        # masked_attention writes every row: q_valid is S
                            q_valid = s
                        nq, nb = (s + 127) // 128, (skv + 127) // 128
                        seed = zlib.crc32(f"{sname}/{d}".encode())
                        keep = (_random_keep(b, h, nq, nb, kv_len, seed, device) if rnd else
                                torch.ones(b, h, nq, nb, dtype=torch.bool, device=device) if kind == "masked" else None)
                        for regime in REGIMES:
                            q, k, v = make_inputs(regime, b, h, s, skv, d, kv_len, dtype, seed, device, strided)
                            tag = f"{entry}/{str(dtype)[6:]}/d{d}f{flags}/{sname}/{regime}"
                            if first:
                                res["kernels"] |= _kernels_of(lambda: _call(entry, q, k, v, kv_len, q_valid, keep))
                                first = False
                            out, tail = _call(entry, q, k, v, kv_len, q_valid, keep)
                            res["cases"] += 1
                            if not (torch.isnan(tail).all() and not out[:, :, q_valid:].any()):
                                res["layout_failures"].append(tag)
                            ref, A, delta = reference(q, k, v, kv_len, q_round, keep if kind == "masked" else None)
                            r = worst_ratio(out[:, :, :q_valid], ref[:, :, :q_valid], A[:, :, :q_valid],
                                            delta[:, :, :q_valid], dtype, e_exp)
                            if r > 1.0:
                                res["bound_failures"].append(f"{tag}: {r:.3g} x bound")
                            if regime == "pad" and kv_len < skv:
                                k0, v0 = k.clone(), v.clone()
                                k0[:, :, kv_len:], v0[:, :, kv_len:] = 0, 0
                                out0, _ = _call(entry, q, k0, v0, kv_len, q_valid, keep)
                                if not torch.equal(out.view(torch.int16), out0.view(torch.int16)):
                                    n = int((out.view(torch.int16) != out0.view(torch.int16)).sum())
                                    res["pad_failures"].append(f"{tag}: {n} elements differ")
                finally:
                    ops.set_attention_flags(0)
    torch.cuda.synchronize()
    res["kernels"] = sorted(res["kernels"])
    return res


def _summary(res, limit=20):
    return {k: (v[:limit] if isinstance(v, list) and k != "kernels" else v) for k, v in res.items()} | {
        "n_" + k: len(res[k]) for k in ("bound_failures", "pad_failures", "layout_failures")}


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def main_matrix(dev):
    t0 = time.time()
    res = run_matrix(device=dev)
    res["seconds"] = time.time() - t0
    return res


_LEG_RESULTS = {}


def _leg(name):
    """Runs one environment leg in a child process (once per session) -> its JSON summary."""
    if name not in _LEG_RESULTS:
        env = {k: v for k, v in os.environ.items() if k not in ("RSA_TC5_POLY", "RSA_TC5_THR")}
        env.update(LEGS[name][0])
        cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), "--leg", name]
        r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900, cwd=REPO)
        lines = [x for x in r.stdout.splitlines() if x.startswith("{")]
        assert r.returncode == 0 and lines, f"leg {name} exited with {r.returncode}:\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}"
        res = json.loads(lines[-1])
        res["kernels"] = [tuple(x) for x in res["kernels"]]
        _LEG_RESULTS[name] = res
    return _LEG_RESULTS[name]


@pytest.mark.gpu
def test_matrix_within_float64_bound(main_matrix):
    """Masked (all-ones and random mask, both query paths) and dense (both out layouts) entries, bf16 and fp16, 128 and
    64 columns and 64 through the 128-column form, every shape and regime: within the bound of the float64 reference;
    rows >= q_valid zero, rows past S of the out buffer untouched."""
    assert main_matrix["cases"] > 3000
    assert not main_matrix["layout_failures"], main_matrix["layout_failures"][:20]
    assert not main_matrix["bound_failures"], (len(main_matrix["bound_failures"]), main_matrix["bound_failures"][:20])


@pytest.mark.gpu
def test_keys_past_kv_len_have_exactly_zero_weight(main_matrix):
    """Keys at or past kv_len that would win their row (K = 50 x the query, V = the dtype's largest value) change no
    bit of the output: the same call with those rows of K and V zeroed is bit-identical."""
    assert not main_matrix["pad_failures"], (len(main_matrix["pad_failures"]), main_matrix["pad_failures"][:20])


@pytest.mark.gpu
@pytest.mark.parametrize("leg", list(LEGS))
def test_environment_selected_instantiations(dev, leg):
    """RSA_TC5_POLY = 0..4 and RSA_TC5_THR = 0 (every increase of a row maximum rescales) select instantiations and a
    code path no default call reaches: the same matrix, bound and pad contract in a child process."""
    res = _leg(leg)
    assert res["cases"] > 0 and res["kernels"]
    assert not res["layout_failures"], res["layout_failures"]
    assert not res["bound_failures"], (res["n_bound_failures"], res["bound_failures"])
    assert not res["pad_failures"], (res["n_pad_failures"], res["pad_failures"])


@pytest.mark.gpu
def test_every_instantiation_is_reached(main_matrix):
    """Each of the fourteen product instantiations of attn_tc5_kernel ran in at least one case (kernel names from the
    profiler); the environment legs reach the RSA_TC5_POLY ones."""
    reached = set(main_matrix["kernels"])
    for name in LEGS:
        reached |= set(_leg(name)["kernels"])
    assert set(INSTANTIATIONS) <= reached, sorted(set(INSTANTIATIONS) - reached)
    assert reached <= set(INSTANTIATIONS), sorted(reached - set(INSTANTIATIONS))


# ------------------------------------------------------------------------------------ dense at production head counts
@pytest.mark.gpu
@pytest.mark.parametrize("b,h,s,d,dtype", [(1, 24, 4224, 128, BF16), (1, 48, 2048 + 97, 64, FP16),
                                           (2, 20, 4096, 128, BF16)], ids=["24h_33tiles", "48h_fp16_d64", "b2_20h"])
def test_dense_production_head_counts(dev, b, h, s, d, dtype):
    """The dense form past the first few CTAs (in-order grid decode, cluster partners sharing every block): bit-identical
    to masked_attention(all-ones, fp32_scale=True), and within the bound on the first and the last (b, h)."""
    from rsa_b200 import ops
    q, k, v = make_inputs("diffuse", b, h, s, s, d, s, dtype, 17 + h, dev)
    got = ops.dense_attention(q, k, v, s, s)
    want = ops.masked_attention(q, k, v, torch.ones(b, h, (s + 127) // 128, (s + 127) // 128, dtype=torch.bool,
                                                    device=dev), s, fp32_scale=True)
    torch.cuda.synchronize()
    assert torch.equal(got.view(torch.int16), want.view(torch.int16))
    e_exp = E_POLY if d == 64 else E_MUFU
    for bi, hi in ((0, 0), (b - 1, h - 1)):
        sl = lambda t: t[bi:bi + 1, hi:hi + 1]
        ref, A, delta = reference(sl(q), sl(k), sl(v), s, 0)
        assert worst_ratio(sl(got), ref, A, delta, dtype, e_exp) <= 1.0, (bi, hi)


if __name__ == "__main__":
    if len(sys.argv) == 3 and sys.argv[1] == "--leg" and sys.argv[2] in LEGS:
        _, dtypes, entries, forms = LEGS[sys.argv[2]]
        t0 = time.time()
        out = run_matrix(dtypes, entries, forms)
        out["seconds"] = time.time() - t0
        out["leg"] = sys.argv[2]
        print(json.dumps(_summary(out)), flush=True)
        sys.exit(0)
    sys.exit(f"usage: {sys.argv[0]} --leg {{{','.join(LEGS)}}}")
