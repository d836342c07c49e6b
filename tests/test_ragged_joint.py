"""Ragged visual segments of Flux and CogVideoX: the padded layout of geometry.flux / geometry.cogvideo.

Flux at 1360x768 (4 080 image tokens) and CogVideoX-2B / -5B at 49 frames of 480x720 (17 550 video tokens + 226 text)
are shapes the reference cannot lay out.  The geometry completes the last visual block with `gap` zero rows that exist
nowhere in memory (pooled as zeros with divisor 128, never attended as keys, never written as queries) and puts the text
blocks block-aligned behind them -- the extension HunyuanVideo's 129-frame shape already takes.

No reference output exists for these shapes.  The oracle's geometry functions (oracle/rsa_oracle.py) restate the
reference's rules; the extension they lack is restated here (_oracle_flux, _oracle_cogvideo) the way geometry_hunyuan
restates HunyuanVideo's, and the small cases below are oracle-only.  The strongest check needs no reference at all: insert the gap zero rows into the tensors
explicitly and run the aligned geometry the reference rule gives for them.  Every mask-building stage must then be
bit-identical, and so must every visual query tile whose kept list does not hold the last visual block; the other tiles
differ only by the pad keys, which the aligned call attends as zero keys, and are held to the oracle."""
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
from oracle import cases as CS
from oracle import gilbert_oracle as GO
from oracle import rsa_oracle as O
from rsa_b200 import geometry as G
from rsa_b200 import native as N
from rsa_b200 import ops

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ATOL_OUT, COS_OUT = 2e-2, 0.999
DTYPES = {"bf16": torch.bfloat16, "fp16": torch.float16}


# ------------------------------------------------------------------------------------------------ geometry (CPU)
def _flux_parent(seq, text_length, kv_len=None):
    """geometry.flux as it was before the padded layout (frozen copy)."""
    if seq % 128:
        raise RuntimeError("needs S % 128 == 0")
    kv_len = seq if kv_len is None else int(kv_len)
    nb = seq // 128
    nq = nb - text_length // 128
    if nq <= 0 or text_length < 1:
        raise ValueError("inconsistent")
    return G.BlockGeometry(1, seq, nb, nq, text_length, kv_len, seq, -(-kv_len // 128), seq - nq * 128)


def _cogvideo_parent(seq, text_length):
    """geometry.cogvideo as it was before the padded layout (frozen copy)."""
    nb = -(-seq // 128)
    pad = nb * 128 - seq
    nq = nb - (text_length + pad) // 128
    if nq <= 0 or text_length < 1 or nq * 128 + text_length > nb * 128:
        raise ValueError("inconsistent")
    return G.BlockGeometry(1, seq, nb, nq, text_length, seq, seq, nb, seq - nq * 128)


# ------------------------------------------------------------------------------ oracle: the padded layout, restated
def _oracle_padded_joint(seq, text_length, top_k, p_remain, kv_len=None):
    """Ragged visual segment of Flux / CogVideoX: the extension of O.geometry_hunyuan -- `seq - text_length` visual
    tokens completed with `gap` zero rows to whole blocks, the text blocks aligned behind them, kv_len / kv_zero_from
    shifted into the padded layout; every text token is a text key and a valid text query."""
    nv = seq - text_length
    nq = (nv + 127) // 128
    gap = nq * 128 - nv
    nb = nq + (text_length + 127) // 128
    kv = (seq if kv_len is None else kv_len) + gap
    return O.Geometry("joint", seq, nb * 128, nb, nq, text_length, kv, seq + gap, (kv + 127) // 128, top_k, p_remain,
                      0, text_length, gap)


def _oracle_flux(seq, text_length, top_k, p_remain, kv_len=None):
    """O.geometry_flux (the reference's rule, S % 128 == 0), else the padded layout."""
    if seq % 128:
        return _oracle_padded_joint(seq, text_length, top_k, p_remain, kv_len)
    return O.geometry_flux(seq, text_length, top_k, p_remain, kv_len)


def _oracle_cogvideo(seq, text_length, top_k, p_remain):
    """O.geometry_cogvideo where the reference's rule has a layout (NQ*128 + text <= NB*128), else the padded layout."""
    nb = (seq + 127) // 128
    nq = nb - (text_length + nb * 128 - seq) // 128
    if nq * 128 + text_length > nb * 128:
        return _oracle_padded_joint(seq, text_length, top_k, p_remain)
    return O.geometry_cogvideo(seq, text_length, top_k, p_remain)


# Oracle-only small cases (no reference fixture can exist: the reference raises at these shapes).
#   name: (family, grid(t,h,w), text_len, heads, top_k, p, regime, seed, head_dim)
RAGGED_JOINT_CASES = {
    "flux_ragged_127": ("flux", (1, 25, 41), 512, 2, 3, 0.3, "walk", 51, 128),      # 1 025 + 512 tokens, gap 127
    "flux_ragged_4": ("flux", (1, 30, 34), 512, 2, 3, 0.3, "walk", 52, 128),        # 1 020 + 512 tokens, gap 4
    "cog_ragged": ("cogvideo", (3, 10, 35), 226, 2, 3, 0.3, "walk", 53, 128),       # 1 050 + 226 tokens, gap 102
    "cog_ragged_d64": ("cogvideo", (3, 10, 35), 226, 2, 3, 0.3, "walk", 54, 64),
}


def _key(g):
    return (g.n_blocks, g.nq_blocks, g.vis_len, g.gap, g.kv_len)


def test_geometry_values():
    assert _key(G.cogvideo(17550 + 226, 226)) == (140, 138, 17550, 114, 17890)        # CogVideoX-2B / -5B, 49 frames
    assert _key(G.flux(4080 + 512, 512)) == (36, 32, 4080, 16, 4608)                   # Flux 1360x768
    for nv in (3600, 3952, 8160):                                                      # 1280x720, 832x1216, 1920x1088
        g = G.flux(nv + 512, 512)
        assert g.vis_len == nv and g.gap == g.nq_blocks * 128 - nv > 0 and g.n_blocks == g.nq_blocks + 4
        assert g.kv_len == g.kv_zero_from == g.nq_blocks * 128 + 512 and g.text_end_block == g.n_blocks
        assert g.text_keys == g.text_q_valid == 512
    g = G.cogvideo(17550 + 226, 226)
    assert g.text_keys == g.text_q_valid == 226 and g.kv_zero_from == g.kv_len and g.text_end_block == g.n_blocks
    assert G.flux(4592, 512, 4592) == G.flux(4592, 512)
    assert G.flux(4592, 512, 4500).kv_len == 4500 + 16                               # a shorter kv_len is shifted too
    for bad in ((100, 226), (226, 226), (300, 0)):           # no visual token, or no text token
        for f in (G.cogvideo, G.flux):
            with pytest.raises(ValueError):
                f(*bad)


@pytest.mark.parametrize("text", [226, 256, 512])
def test_existing_shapes_keep_their_geometry(text):
    """For every visual count 128 m + r: where the earlier function returned a geometry, the same one; where it raised,
    the padded layout (or, for Flux with a block-aligned visual segment, the aligned layout it implies)."""
    padded = 0
    for m in range(0, 150):
        for r in range(128):
            nv = 128 * m + r
            if nv == 0:
                continue
            s = nv + text
            for new, old in ((G.flux, _flux_parent), (G.cogvideo, _cogvideo_parent)):
                try:
                    want = old(s, text)
                except (RuntimeError, ValueError):
                    want = None
                if want is not None:
                    assert new(s, text) == want, (new.__name__, s, text)
                    continue
                g = new(s, text)
                nq = -(-nv // 128)
                assert (g.nq_blocks, g.n_blocks, g.gap) == (nq, nq + -(-text // 128), nq * 128 - nv)
                assert g.vis_len == (nv if g.gap else 0) and g.text_keys == g.text_q_valid == text
                assert g.kv_len == g.kv_zero_from == nq * 128 + text and g.text_end_block == -(-g.kv_len // 128)
                padded += g.gap > 0
    assert padded > 0
    if text != 226:                                                  # the reference's CogVideoX rule lays out every such shape
        assert all(G.cogvideo(128 * m + r + text, text) == _cogvideo_parent(128 * m + r + text, text)
                   for m in range(1, 40) for r in range(128))


def test_product_and_oracle_geometry_agree():
    fields = lambda g: (g.n_blocks, g.nq_blocks, g.text_keys, g.kv_len, g.kv_zero_from, g.text_end_block,
                        g.text_q_valid, g.gap)
    for text in (226, 256, 512):
        for nv in list(range(900, 1300)) + [3600, 3952, 4080, 8160, 17550]:
            s = nv + text
            assert fields(G.flux(s, text)) == fields(_oracle_flux(s, text, 2, 0.3)), (s, text)
            assert fields(G.cogvideo(s, text)) == fields(_oracle_cogvideo(s, text, 2, 0.3)), (s, text)
            og = _oracle_flux(s, text, 2, 0.3)
            assert og.seq_pad == og.n_blocks * 128


def test_oracle_cases():
    """The oracle-only ragged cases have the gaps they are named for, and the oracle lays them out."""
    want = {"flux_ragged_127": 127, "flux_ragged_4": 4, "cog_ragged": 102, "cog_ragged_d64": 102}
    assert set(RAGGED_JOINT_CASES) == set(want)
    for name, gap in want.items():
        case = _case(name)
        assert case["ogeo"].gap == gap == case["geo"].gap
        assert case["q"].shape[-1] == RAGGED_JOINT_CASES[name][8]
        assert not (set(RAGGED_JOINT_CASES) & set(CS.CASES))         # no golden file is expected for them


def _desc(heads, geo, hd):
    return ops._fill_desc(N.AttnDesc(), (1, heads, geo.seq, hd),
                          [(heads * geo.seq * hd, geo.seq * hd, hd)] * 3 + [(geo.seq * heads * hd, hd, heads * hd)],
                          geo, 2, 0.3, None)


def test_workspace_bytes_for_padded_descriptors():
    lib = N.lib()
    for geo, hd in ((G.cogvideo(17776, 226), 64), (G.cogvideo(1276, 226), 128), (G.flux(4592, 512), 128),
                    (G.flux(1537, 512), 128), (G.flux(8672, 512), 128)):
        d = _desc(2, geo, hd)
        d.dtype = N.DTYPE_BF16
        assert lib.rsa_attn_workspace_bytes(C.byref(d)) > 0, lib.rsa_last_error_string()
        d.dtype = N.DTYPE_F16
        assert lib.rsa_attn_workspace_bytes(C.byref(d)) > 0, lib.rsa_last_error_string()


@pytest.mark.parametrize("dtype", [N.DTYPE_BF16, N.DTYPE_F16])
def test_gather_two_call_form_at_64_columns(dtype):
    """rsa_qkv_prep_gather at head_dim 64 takes the visual tokens and the text tokens in two calls (it gets as far as the
    workspace, which is left out here), and still refuses rows that name neither segment."""
    lib = N.lib()
    geo = G.cogvideo(1276, 226)
    nv = geo.vis_len
    d = _desc(3, geo, 64)
    d.dtype = dtype
    r = N.PeerRoute()
    r.n_ranks, r.rank, r.rows_per_rank, r.heads_total, r.head0 = 2, 0, 638, 3, 0
    r.src_table = 16                                                   # never read on the host
    r.src_stride[0], r.src_stride[1] = 638 * 3 * 64, 3 * 64
    p = N.PrepDesc()
    p.norm, p.q_weight, p.k_weight, p.q_bias, p.k_bias, p.eps = 3, 16, 16, 16, 16, 1e-6

    def call(rows, dst_row):
        p.rows, p.dst_row = rows, dst_row
        rc = lib.rsa_qkv_prep_gather(C.byref(p), C.byref(d), C.byref(r), 16, 16, 16, 1, None, 0, None)
        return rc, lib.rsa_last_error_string()

    for rows, dst in ((nv, 0), (geo.seq - nv, nv)):
        rc, msg = call(rows, dst)
        assert rc != 0 and b"workspace is null" in msg, msg
    for rows, dst in ((geo.seq, 0), (nv - 1, 0), (geo.seq - nv, 0), (100, nv), (geo.seq - nv, nv - 128)):
        rc, msg = call(rows, dst)
        assert rc != 0
        assert b"must name the whole sequence, the visual tokens or the text tokens" in msg, msg


# ------------------------------------------------------------------------------------------------ GPU
def _case(name):
    fam, (t, h, w), text_len, heads, top_k, p, regime, seed, hd = RAGGED_JOINT_CASES[name]
    nv = t * h * w
    s = nv + text_len
    q, k, v = O.synth_qkv(heads, s, hd, regime, seed)
    if fam == "flux":
        geo, ogeo = G.flux(s, text_len), _oracle_flux(s, text_len, top_k, p)
    else:
        geo, ogeo = G.cogvideo(s, text_len), _oracle_cogvideo(s, text_len, top_k, p)
    return dict(fam=fam, nv=nv, s=s, text=text_len, heads=heads, top_k=top_k, p=p, q=q, k=k, v=v, hd=hd, geo=geo,
                ogeo=ogeo, nbr=GO.gilbert_block_neighbors(t, h, w))


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    assert N.lib().rsa_device_ok() == 1, "not an sm_100 device"
    return torch.device("cuda:0")


def _rounded(x, dt):
    """numpy fp32 [..] -> (the values the GPU holds as fp32 numpy, the device tensor)."""
    t = torch.from_numpy(np.ascontiguousarray(x)).to(dt)
    return t.float().numpy(), t


def _aligned_geometry(fam, s, text):
    """The reference rule's own layout of the explicitly padded sequence (S + gap tokens): no gap of its own."""
    g = G.flux(s, text) if fam == "flux" else G.cogvideo(s, text)
    assert g.gap == 0
    return g


def _pad_rows(x, nv, gap):
    """[B, H, S, D] -> [B, H, S + gap, D] with gap zero rows at token nv."""
    z = torch.zeros(*x.shape[:2], gap, x.shape[3], dtype=x.dtype, device=x.device)
    return torch.cat([x[:, :, :nv], z, x[:, :, nv:]], dim=2).contiguous()


STAGES = ("q_pool", "q_mad", "k_cat", "k_mad", "v_pool", "scores", "nogapr", "probs", "w_skip", "n_needed", "kept_cnt",
          "R", "C")


def _staged(q, k, v, geo, top_k, p, nbr):
    plan = ops.Plan(q, k, v, geo, top_k, p, torch.from_numpy(np.asarray(nbr)), debug_dump_probs=True,
                    private_workspace=True)
    plan.pool_stats()
    plan.block_scores()
    plan.block_select()
    plan.rect_c()
    out = plan.sparse_attention()
    torch.cuda.synchronize()
    return plan, out


def _padding_equivalence(q, k, v, geo, fam, text, top_k, p, nbr, oracle_out, what):
    """q, k, v: device [1, H, S, D].  The ragged call against the aligned call on the explicitly padded tensors."""
    nv, gap, nq = geo.vis_len, geo.gap, geo.nq_blocks
    pr, out_r = _staged(q, k, v, geo, top_k, p, nbr)
    qp, kp, vp = (_pad_rows(x, nv, gap) for x in (q, k, v))
    pp, out_p = _staged(qp, kp, vp, _aligned_geometry(fam, geo.seq + gap, text), top_k, p, nbr)
    vr, vpd = pr.view(), pp.view()
    for key in STAGES:
        a, b = vr[key], vpd[key]
        assert a.shape == b.shape, f"{what}: {key} shapes differ"
        assert torch.equal(a.contiguous().view(torch.uint8), b.contiguous().view(torch.uint8)), f"{what}: {key} differs"
    mask = pr.dense_mask()
    assert torch.equal(mask, pp.dense_mask()), f"{what}: kept blocks differ"
    cnt = vr["kept_cnt"].cpu()
    ki_r, ki_p = (x["kept_idx"].cpu() for x in (vr, vpd))
    for bh in range(cnt.shape[0]):
        for i in range(cnt.shape[1]):
            assert torch.equal(ki_r[bh, i, : cnt[bh, i]], ki_p[bh, i, : cnt[bh, i]]), f"{what}: kept list {bh}, {i}"
    out_p = torch.cat([out_p[:, :nv], out_p[:, nv + gap:]], dim=1)                   # the pad rows are never written
    o_r, o_p = out_r[0].float().cpu().numpy(), out_p[0].float().cpu().numpy()       # [S, H, D]
    keeps_last = mask[:, :nq, nq - 1].cpu().numpy()                                  # [H, NQ]
    same_tiles = 0
    for h in range(o_r.shape[1]):
        for i in range(nq):
            rows = slice(128 * i, min(128 * (i + 1), nv))
            if not keeps_last[h, i]:
                assert np.array_equal(o_r[rows, h].view(np.uint32), o_p[rows, h].view(np.uint32)), f"{what}: tile {i}"
                same_tiles += 1
            else:       # only the pad keys differ: the aligned call attends them as zero keys
                _bar(o_r[rows, h], oracle_out[rows, h], f"{what}: head {h} tile {i}")
        _bar(o_r[nv:, h], oracle_out[nv:, h], f"{what}: head {h} text rows")
    assert same_tiles > 0, f"{what}: every tile keeps the last visual block -- nothing compared bit for bit"
    return pr, out_r


def _bar(got, ref, what):
    err = float(np.abs(got - ref).max())
    assert err <= ATOL_OUT, f"{what}: max-abs-err {err}"
    assert cos_sim(got, ref) >= COS_OUT, what


def _oracle_out(q, k, v, ogeo, nbr, dname):
    """fp32 numpy [H, S, D] inputs -> oracle output [S, H, D]."""
    return O.forward(q[None], k[None], v[None], ogeo, nbr, q_dtype=dname).reshape(q.shape[1], q.shape[0], q.shape[2])


def _check_stages_vs_oracle(plan, hi, q, k, v, ogeo, nbr, what, max_flips=2):
    """Kernels 2, 3a bit-exact; 3b's P within fp32 rounding of expf and the selection exact given the kernel's P; R, C
    within fp32 tolerance (the bars of test_gpu_parity / test_gpu_fullsize_stages)."""
    vw = plan.view()
    st, _, _, _ = O.mask_stages(q, k, v, ogeo, nbr)
    nq = ogeo.nq_blocks
    for key, name in (("q_pool", "qp"), ("q_mad", "dq"), ("k_mad", "dk"), ("v_pool", "vp")):
        got = vw[key][hi].cpu().numpy()
        assert np.array_equal(got[..., : q.shape[1]], st[name][..., : q.shape[1]]), f"{what}: {key}"
    assert np.array_equal(vw["k_cat"][hi, :nq, : q.shape[1]].cpu().numpy(), st["kp"][:, : q.shape[1]]), what
    assert np.array_equal(vw["k_cat"][hi, nq:, : q.shape[1]].cpu().numpy(), st["ktext"]), f"{what}: text keys"
    assert np.array_equal(vw["scores"][hi].cpu().numpy(), st["scores"]), f"{what}: scores"
    assert np.array_equal(vw["nogapr"][hi].cpu().numpy().astype(bool), st["nogapr"]), f"{what}: GAPR bytes"
    p_gpu = vw["probs"][hi].cpu().numpy()
    np.testing.assert_allclose(p_gpu, st["probs"], rtol=3e-5, atol=1e-9, err_msg=what)
    m, n = O.select_blocks(p_gpu, ogeo, nbr)
    assert np.array_equal(vw["n_needed"][hi].cpu().numpy(), n), f"{what}: n_needed"
    mask = plan.dense_mask()[hi].cpu().numpy()
    assert np.array_equal(mask[:nq], m), f"{what}: mask"
    assert int((m != st["mask"]).sum()) <= max_flips, f"{what}: mask against the pure oracle"
    r, c, _, w = O.rectify_factors(p_gpu, m, st["nogapr"], st["vp"], ogeo)
    np.testing.assert_allclose(vw["R"][hi, :nq].cpu().numpy(), r, rtol=0, atol=2e-6, err_msg=what)
    assert np.array_equal(vw["w_skip"][hi].cpu().numpy(), w), f"{what}: W"
    c_gpu = vw["C"][hi, :nq].cpu().numpy()                  # 128 columns; a 64-column head leaves 64..127 zero
    np.testing.assert_allclose(c_gpu[:, : q.shape[1]], c, rtol=1e-4, atol=2e-6, err_msg=what)
    assert not c_gpu[:, q.shape[1]:].any(), what


def _device_case(case, dname, dev):
    dt = DTYPES[dname]
    qn, q = _rounded(case["q"][0], dt)
    kn, k = _rounded(case["k"][0], dt)
    vn, v = _rounded(case["v"][0], dt)
    return (qn, kn, vn), tuple(x[None].to(dev) for x in (q, k, v))


@pytest.mark.gpu
@pytest.mark.parametrize("dname", ["bf16", "fp16"])
@pytest.mark.parametrize("name", list(RAGGED_JOINT_CASES))
def test_small_case_against_oracle(dev, name, dname):
    """Every stage and the output of the ragged call against the oracle's restatement of the padded layout."""
    case = _case(name)
    (qn, kn, vn), (q, k, v) = _device_case(case, dname, dev)
    plan, out = _staged(q, k, v, case["geo"], case["top_k"], case["p"], case["nbr"])
    for hi in range(case["heads"]):
        _check_stages_vs_oracle(plan, hi, qn[hi], kn[hi], vn[hi], case["ogeo"], case["nbr"], f"{name} {dname} head {hi}")
    ref = _oracle_out(qn, kn, vn, case["ogeo"], case["nbr"], dname)
    _bar(out[0].float().cpu().numpy(), ref, f"{name} {dname}")
    whole = ops.Plan(q, k, v, case["geo"], case["top_k"], case["p"], torch.from_numpy(case["nbr"])).run()
    assert torch.equal(whole.view(torch.int16), out.view(torch.int16))                  # the one-call form


@pytest.mark.gpu
@pytest.mark.parametrize("dname", ["bf16", "fp16"])
@pytest.mark.parametrize("name", list(RAGGED_JOINT_CASES))
def test_padding_equivalence(dev, name, dname):
    case = _case(name)
    (qn, kn, vn), (q, k, v) = _device_case(case, dname, dev)
    ref = _oracle_out(qn, kn, vn, case["ogeo"], case["nbr"], dname)
    _padding_equivalence(q, k, v, case["geo"], case["fam"], case["text"], case["top_k"], case["p"], case["nbr"], ref,
                         f"{name} {dname}")


@pytest.mark.gpu
@pytest.mark.parametrize("dname", ["bf16", "fp16"])
@pytest.mark.parametrize("name", list(RAGGED_JOINT_CASES))
def test_dense_limit_against_sdpa(dev, name, dname):
    """top_k >= NQ keeps every block: the ragged call is dense attention over the tensors as the caller holds them
    (SDPA on the un-padded memory tensors) -- no gap row is ever attended."""
    case = _case(name)
    _, (q, k, v) = _device_case(case, dname, dev)
    geo = case["geo"]
    out = ops.Plan(q, k, v, geo, geo.nq_blocks + 1, case["p"], torch.from_numpy(case["nbr"])).run()
    ref = torch.nn.functional.scaled_dot_product_attention(q.float(), k.float(), v.float()).transpose(1, 2)
    _close(out, ref, f"{name} {dname}")


FULL = {
    # name: (family, visual tokens, text tokens, heads of the model, head_dim, dtype, drop)
    "cogvideox-2b": ("cogvideo", 13 * 30 * 45, 226, 30, 64, "fp16", 0.75),
    "cogvideox-5b": ("cogvideo", 13 * 30 * 45, 226, 48, 64, "bf16", 0.9),
    "flux-1360x768": ("flux", 85 * 48, 512, 24, 128, "bf16", 0.75),
    "flux-1920x1088": ("flux", 120 * 68, 512, 24, 128, "bf16", 0.9),
}
FULL_GRID = {"cogvideox-2b": (13, 30, 45), "cogvideox-5b": (13, 30, 45), "flux-1360x768": (1, 48, 85),
             "flux-1920x1088": (1, 68, 120)}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FULL))
def test_full_shape_one_head(dev, name):
    """One head at the model's own token count: stages bit-exact against the oracle (a handful of near-tie flips
    against the pure oracle allowed, as at the other full sizes), the output at the usual bar, and padding
    equivalence.  top_k = int((1 - drop) * visual blocks) as in the reference's scripts."""
    fam, nv, text, _, hd, dname, drop = FULL[name]
    s = nv + text
    geo = G.flux(s, text) if fam == "flux" else G.cogvideo(s, text)
    assert geo.gap > 0
    top_k = O.select_block_num(drop, nv // 128)
    ogeo = (_oracle_flux if fam == "flux" else _oracle_cogvideo)(s, text, top_k, 0.3)
    nbr = GO.gilbert_block_neighbors(*FULL_GRID[name])
    qa, ka, va = O.synth_qkv(1, s, hd, "walk", 61)
    (qn, kn, vn), (q, k, v) = _device_case(dict(q=qa, k=ka, v=va), dname, dev)
    ref = _oracle_out(qn, kn, vn, ogeo, nbr, dname)
    plan, out = _padding_equivalence(q, k, v, geo, fam, text, top_k, 0.3, nbr, ref, name)
    _check_stages_vs_oracle(plan, 0, qn[0], kn[0], vn[0], ogeo, nbr, name, max_flips=8)
    _bar(out[0].float().cpu().numpy(), ref, name)


# ------------------------------------------------------------------------------------------ processors
def _rope(n, hd, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    ang = torch.rand(n, hd // 2, generator=g, device=dev) * 6.28
    return ang.cos().repeat_interleave(2, 1).contiguous(), ang.sin().repeat_interleave(2, 1).contiguous()


def _layers(dev):
    """(name, make(top_k, dense_call) -> processor, call(processor) -> output) at ragged shapes: Flux dual- and
    single-stream (1 025 image + 512 text tokens, gap 127), CogVideoX at 128 and 64 columns (1 050 + 226, gap 102;
    the 64-column layer in fp16 with fuse_prep_fp16)."""
    from rectified_spaattn import rectified_cogvideo_attn as cog
    from rectified_spaattn import rectified_flux_attn as flux
    dim, nv_f, nv_c = 256, 1025, 1050
    g = torch.Generator(device=dev).manual_seed(7)
    rnd = lambda n, dt: torch.randn(1, n, dim, generator=g, device=dev).to(dt)
    bf = torch.bfloat16
    torch.manual_seed(0)
    a_dual = FakeAttention(dim, 2, added=True).to(dev).to(bf)
    a_single = FakeAttention(dim, 2).to(dev).to(bf)
    a_c128 = FakeAttention(dim, 2, head_dim=128, norm="layer").to(dev).to(bf)
    a_c64 = FakeAttention(dim, 4, head_dim=64, norm="layer").to(dev).to(torch.float16)
    x_f, t_f = rnd(nv_f, bf), rnd(512, bf)
    joint = torch.cat([x_f, t_f], dim=1)
    rope_f = _rope(nv_f + 512, 128, dev, 1)
    x_c, t_c = rnd(nv_c, bf), rnd(226, bf)
    x_c16, t_c16 = rnd(nv_c, torch.float16), rnd(226, torch.float16)
    rope_c128, rope_c64 = _rope(nv_c, 128, dev, 2), _rope(nv_c, 64, dev, 3)

    def mk_flux(pid_sparse):
        def make(top_k, dense):
            return flux.RectifiedFluxSpaAttnProcessor2_0("sparse", top_k, None, 0.3,
                                                         processor_id=40 if dense else pid_sparse, text_length=512)
        return make

    def mk_cog(fp16):
        def make(top_k, dense):
            pr = cog.RectifiedCogVideoXVideoSpaAttnProcessor2_0("sparse", top_k, None, 0.3)
            pr.current_step = 0 if dense else 5
            pr.fuse_prep_fp16 = fp16
            return pr
        return make

    return [
        ("flux dual-stream", mk_flux(1), lambda pr: pr(a_dual, x_f, t_f, None, rope_f)),
        ("flux single-stream", mk_flux(60), lambda pr: pr(a_single, joint, None, None, rope_f)),
        ("cogvideox 128", mk_cog(False), lambda pr: pr(a_c128, x_c, t_c, None, rope_c128)),
        ("cogvideox 64 fp16", mk_cog(True), lambda pr: pr(a_c64, x_c16, t_c16, None, rope_c64)),
    ]


@pytest.fixture
def prep_calls(monkeypatch):
    n = [0]
    orig = ops.Plan.qkv_prep

    def counted(self, *a, **kw):
        n[0] += 1
        return orig(self, *a, **kw)

    monkeypatch.setattr(ops.Plan, "qkv_prep", counted)
    return n


def _close(a, b, what):
    a, b = a.float().cpu().numpy(), b.float().cpu().numpy()
    assert np.isfinite(a).all(), what
    assert cos_sim(a, b) >= 0.999 and abs(a - b).max() <= 4e-2 * max(1.0, abs(b).max()), what


@pytest.mark.gpu
@pytest.mark.parametrize("dense", [False, True])
def test_processors_fused_and_op_by_op(dev, prep_calls, dense):
    """Both routes run at ragged shapes: the fused one (kernel 0 in two calls, visual and text; fuse_prep_dense for
    the dense calls) and the op-by-op one, sparse (top_k 3) and dense calls; in the dense limit (top_k 99) they agree."""
    for name, make, call in _layers(dev):
        for top_k in (3, 99):
            outs = {}
            for fused in (True, False):
                pr = make(top_k, dense)
                pr.fuse_prep, pr.fuse_prep_dense = fused, fused and dense
                before = prep_calls[0]
                with torch.no_grad():
                    o = call(pr)
                outs[fused] = o if isinstance(o, tuple) else (o,)
                assert (prep_calls[0] - before == 2) == fused, (name, fused, prep_calls[0] - before)
                assert all(torch.isfinite(x).all() for x in outs[fused]), name
            if top_k == 99 or dense:
                for a, b in zip(outs[True], outs[False]):
                    _close(a, b, f"{name} dense={dense} top_k={top_k}")


# ------------------------------------------------------------------------------- mask re-use, host buffers
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["flux_ragged_127", "cog_ragged_d64"])
def test_mask_reuse_and_host_call(dev, name):
    """At a ragged shape: a call that re-uses the cached selection on the same inputs equals a rebuild, bit for bit
    (keep "lists" and "all"), and the host-buffer call equals the device call."""
    case = _case(name)
    _, (q, k, v) = _device_case(case, "bf16", dev)
    geo, nbr = case["geo"], torch.from_numpy(case["nbr"])
    ref = ops.rectified_attention(q, k, v, geo, case["top_k"], case["p"], nbr).clone()
    for keep in ("lists", "all"):
        cache = ops.MaskCache(2, keep)
        outs = [ops.rectified_attention(q, k, v, geo, case["top_k"], case["p"], nbr, mask_cache=cache).clone()
                for _ in range(3)]
        assert cache.calls == 3
        for o in outs:
            assert torch.equal(o.view(torch.int16), ref.view(torch.int16)), keep
    host = ops.rectified_attention(*(x.cpu().pin_memory() for x in (q, k, v)), geo, case["top_k"], case["p"], nbr)
    torch.cuda.synchronize()
    assert not host.is_cuda and torch.equal(host.view(torch.int16), ref.cpu().view(torch.int16))


# ------------------------------------------------------------------------------------------ fused Ulysses
def _ulysses(n, workload, dense, dname, port):
    args = [workload, "--dtype", {"bf16": "bfloat16", "fp16": "float16"}[dname]] + (["--dense"] if dense else [])
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n),
                        "--master-addr", "127.0.0.1", "--master-port", str(port),
                        os.path.join(REPO, "tools", "check_fused_ulysses.py")] + args,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["dense"] is dense and line["n_gpus"] == n
    return line


ULYSSES = [("cog_ragged", False, "fp16"), ("cog_ragged", True, "bf16"), ("flux_ragged", False, "bf16"),
           ("flux_ragged", True, "fp16")]


@pytest.mark.gpu
@pytest.mark.parametrize("workload,dense,dname", ULYSSES)
def test_fused_ulysses_one_rank(dev, workload, dense, dname):
    """FusedUlysses on one rank at a ragged shape (two gathers: visual and text tokens; Flux rotates its text tokens
    with table rows [nv, S)): bit-identical to the single-GPU kernel 0 + attention call.  CogVideoX form at 64 columns,
    Flux form at 128; sparse and dense, bf16 and fp16."""
    port = 29631 + ULYSSES.index((workload, dense, dname))
    line = _ulysses(1, workload, dense, dname, port)
    assert line["fused_equals_single_gpu_bitwise_checked_ranks"] == [True]


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["cog_ragged", "flux_ragged"])
def test_fused_ulysses_two_gpus(dev, workload):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    line = _ulysses(2, workload, False, "bf16", {"cog_ragged": 29641, "flux_ragged": 29642}[workload])
    assert line["fused_equals_single_gpu_bitwise_checked_ranks"] == [True, True]
