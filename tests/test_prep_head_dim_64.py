"""Kernel 0 and the fused Ulysses exchange at head_dim 64 (CogVideoX1.5: 48 heads x 64, LayerNorm(64) on q / k).

The 64-column form works on pairs of adjacent heads (h, h + 1): a source row's two 64-column slices are one 256-byte
copy, lanes 0-7 of a half-warp take head h and lanes 8-15 head h + 1.  LayerNorm(64) reduces over the 8 lanes that
share a (row, head) with a fixed butterfly (xor 1, 2, 4); `prep64` below restates that order.  Pooled statistics keep
kernel 2's summation order, so they are bit-identical to pooling the stored rows, with columns 64..127 exactly zero."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from fake_attention import FakeAttention
from helpers import assert_prep_close, cos_sim
from oracle import make_golden as MG
from oracle import prep_oracle as PO
from rsa_b200 import geometry as G
from rsa_b200 import native as N
from rsa_b200 import ops

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------- 64-column oracle
def layer_norm64(x, weight, bias, eps):
    """torch.nn.LayerNorm(64) on bf16 values in kernel 0's order: per lane a sequential sum of its 8 columns, a butterfly
    over the 8 lanes of the head (xor 1, 2, 4); two-pass variance (fma chain of the centred values, same butterfly);
    statistics and affine in fp32, one rounding to bf16."""
    x = np.asarray(x, dtype=np.float32)
    lanes = x.reshape(*x.shape[:-1], 8, 8)
    sm = np.zeros(lanes.shape[:-1], dtype=np.float32)
    for c in range(8):
        sm = (sm + lanes[..., c]).astype(np.float32)
    for o in (1, 2, 4):
        sm = (sm + sm[..., np.arange(8) ^ o]).astype(np.float32)
    mean = (sm[..., 0] * np.float32(1.0 / 64.0)).astype(np.float32)
    d = (lanes - mean[..., None, None]).astype(np.float32)
    ss = np.zeros(lanes.shape[:-1], dtype=np.float32)
    for c in range(8):
        ss = PO._fma32(d[..., c], d[..., c], ss)
    for o in (1, 2, 4):
        ss = (ss + ss[..., np.arange(8) ^ o]).astype(np.float32)
    var = (ss[..., 0] * np.float32(1.0 / 64.0)).astype(np.float32)
    rstd = (1.0 / np.sqrt(var.astype(np.float64) + np.float64(np.float32(eps)))).astype(np.float32)
    t = (d.reshape(x.shape) * rstd[..., None]).astype(np.float32)
    return PO.bf16_round(PO._fma32(np.broadcast_to(np.asarray(weight, np.float32), x.shape), t,
                                   np.broadcast_to(np.asarray(bias, np.float32), x.shape)))


def prep64(src, heads, weight, bias, eps, cos, sin, rope_rows):
    """src [B, rows, heads*64] -> [B, heads, rows, 64]: head split, LayerNorm(64), rotary embedding on the first
    rope_rows tokens (cos / sin [>= rope_rows, 64])."""
    b, rows, _ = src.shape
    x = np.asarray(src, np.float32).reshape(b, rows, heads, 64).transpose(0, 2, 1, 3)
    x = layer_norm64(x, weight, bias, eps)
    if rope_rows:
        x = x.copy()
        x[:, :, :rope_rows] = PO.rotary(x[:, :, :rope_rows], cos[:rope_rows], sin[:rope_rows])
    return x


def _inputs(batch, heads, rows, n_rope, seed, scale=1.5):
    g = torch.Generator().manual_seed(seed)
    src = [torch.randn(batch, rows, heads * 64, generator=g).mul(scale).to(torch.bfloat16) for _ in range(3)]
    w = [(1 + 0.1 * torch.randn(64, generator=g)).to(torch.bfloat16) for _ in range(2)]
    bias = [(0.05 * torch.randn(64, generator=g)).to(torch.bfloat16) for _ in range(2)]
    ang = torch.outer(torch.arange(n_rope, dtype=torch.float32), 1.0 / (256.0 ** (torch.arange(0, 64, 2) / 64)))
    cos, sin = ang.cos().repeat_interleave(2, dim=1), ang.sin().repeat_interleave(2, dim=1)      # [n_rope, 64]
    return src, w, bias, cos, sin


# ------------------------------------------------------------------------------------------------------ CPU
def test_oracle_matches_torch_prep_cog_at_64_columns():
    """The 64-column oracle against the PyTorch op sequence of the CogVideoX processor (LayerNorm(64) then the rotary
    embedding on the video tokens), two heads, batch 2, text rows past rope_rows."""
    heads, rows, n_rope = 2, 300, 220
    src, w, bias, cos, sin = _inputs(2, heads, rows, n_rope, 41)
    for i in range(2):
        want = MG.torch_prep_cog(src[i], heads, w[i], bias[i], 1e-6, cos, sin, n_rope)
        got = prep64(src[i].float().numpy(), heads, w[i].float().numpy(), bias[i].float().numpy(), 1e-6, cos.numpy(),
                     sin.numpy(), n_rope)
        assert got.shape == (2, heads, rows, 64)
        assert_prep_close(got, want.float().numpy(), f"tensor {i}")


def _desc64(geo, heads, b=1):
    d = N.AttnDesc()
    d.batch, d.heads, d.seq, d.head_dim = b, heads, geo.seq, 64
    for name in ("q_stride", "k_stride", "v_stride", "o_stride"):
        arr = getattr(d, name)
        arr[0], arr[1], arr[2] = heads * geo.seq * 64, geo.seq * 64, 64
    d.family, d.n_blocks, d.nq_blocks, d.text_keys = geo.family, geo.n_blocks, geo.nq_blocks, geo.text_keys
    d.kv_len, d.kv_zero_from, d.text_end_block = geo.kv_len, geo.kv_zero_from, geo.text_end_block
    d.text_q_valid, d.top_k, d.p_remain, d.first_frame_blocks = geo.text_q_valid, 2, 0.3, geo.first_frame_blocks
    d.vis_len = geo.vis_len
    return d


def test_cabi_refuses_other_norms_at_64_columns():
    """Kernel 0 has a 64-column form for LayerNorm (norm 3) only: the C ABI refuses norms 0-2 at head_dim 64 before it
    touches the device, naming the norm, and a route whose rows are heads_total * 64 channels passes the stride check."""
    lib = N.lib()
    geo = G.cogvideo(1250, 226)
    d = _desc64(geo, 2)
    p = N.PrepDesc()
    p.rows, p.dst_row = geo.seq, 0
    for t in range(3):
        p.src_stride[t][0], p.src_stride[t][1] = geo.seq * 128, 128
    for norm in (0, 1, 2):
        p.norm = norm
        assert lib.rsa_qkv_prep(C.byref(p), C.byref(d), 16, 16, 16, 16, 16, 16, 0, None, 0, None) == -2
        msg = lib.rsa_last_error_string()
        assert b"head_dim 64" in msg and f"norm {norm}".encode() in msg, msg
    r = N.PeerRoute()
    r.n_ranks, r.rank, r.rows_per_rank, r.heads_total, r.head0 = 2, 0, 625, 4, 0
    r.src_table = 16                                               # never read on the host
    r.src_stride[0], r.src_stride[1] = 625 * 4 * 64, 4 * 64        # a 64-column row: heads_total * 64 channels
    p.norm = 1
    assert lib.rsa_qkv_prep_gather(C.byref(p), C.byref(d), C.byref(r), 16, 16, 16, 0, None, 0, None) == -2
    msg = lib.rsa_last_error_string()
    assert b"norm 1" in msg and b"strides" not in msg, msg
    r.src_stride[1] = 4 * 64 - 8                                   # shorter than a row: refused for its strides
    assert lib.rsa_qkv_prep_gather(C.byref(p), C.byref(d), C.byref(r), 16, 16, 16, 0, None, 0, None) == -1
    assert b"strides" in lib.rsa_last_error_string()


# ------------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


@pytest.mark.gpu
@pytest.mark.parametrize("compact", [True, False])
def test_kernel0_64_columns_against_oracle_and_torch(dev, monkeypatch, compact):
    """Kernel 0 at 64 columns: 3 heads (the last pair half empty), batch 2, 1000 rows (not a multiple of 128), the
    rotary embedding on the first 870 rows only; the compact (cos, sin)-pair table and the two-table form."""
    monkeypatch.setattr(ops, "COMPACT_ROPE", compact)
    heads, rows, n_rope, b = 3, 1000, 870, 2
    src, w, bias, cos, sin = _inputs(b, heads, rows, n_rope, 43)
    q, k, v = (torch.full((b, heads, rows, 64), float("nan"), dtype=torch.bfloat16, device=dev) for _ in range(3))
    plan = ops.Plan(q, k, v, G.wan(rows), 1, 0.3, None)
    plan.qkv_prep(*(t.to(dev) for t in src), q_weight=w[0], k_weight=w[1], q_bias=bias[0], k_bias=bias[1], eps=1e-6,
                  rope=(cos.to(dev), sin.to(dev)), rope_rows=n_rope, pool=False)
    torch.cuda.synchronize()
    for i, (name, got) in enumerate((("q", q), ("k", k))):
        want = prep64(src[i].float().numpy(), heads, w[i].float().numpy(), bias[i].float().numpy(), 1e-6, cos.numpy(),
                      sin.numpy(), n_rope)
        tref = MG.torch_prep_cog(src[i].to(dev), heads, w[i].to(dev), bias[i].to(dev), 1e-6, cos.to(dev), sin.to(dev),
                                 n_rope)
        g = got.float().cpu().numpy()
        assert_prep_close(g, want, f"{name} vs oracle")
        assert_prep_close(g, tref.float().cpu().numpy(), f"{name} vs torch on GPU")
    want_v = src[2].view(b, rows, heads, 64).transpose(1, 2)
    assert torch.equal(v.cpu().view(torch.int16), want_v.contiguous().view(torch.int16))


def _walk_sources(b, heads, s, dev, seed):
    """Projection outputs with the block structure of video (neighbouring blocks similar): a random walk of block
    means under iid noise, so the pooled scores are not near-ties."""
    g = torch.Generator(device=dev).manual_seed(seed)
    nb = (s + 127) // 128
    out = []
    for i in range(3):
        x = torch.randn(b, nb * 128, heads * 64, generator=g, device=dev)
        if i < 2:
            mu = torch.cumsum(torch.randn(b, nb, heads * 64, generator=g, device=dev) * 0.35, dim=1)
            x += mu.repeat_interleave(128, dim=1)
        out.append(x[:, :s].to(torch.bfloat16).contiguous())
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["small", "cogvideox1.5"])
def test_kernel0_64_columns_pools_like_kernel2(dev, shape):
    """Kernel 0's pooled statistics at 64 columns are those kernel 2 computes from the stored rows, bit for bit, with
    columns 64..127 of every statistics row exactly zero (the workspace is filled with NaN first), and the pooled call
    equals the whole call.  Small CogVideoX geometry (3 heads, 4x16x16 + 226 text) and CogVideoX1.5's full shape
    (48 heads, 11x48x80 + 226 text = 42 466 tokens)."""
    (t, h, w), heads, top_k = ((4, 16, 16), 3, 2) if shape == "small" else ((11, 48, 80), 48, 82)
    text = 226
    nv = t * h * w
    s = nv + text
    geo = G.cogvideo(s, text)
    nbr = ops.gilbert_block_neighbors(t, h, w)
    src = _walk_sources(1, heads, s, dev, 5)
    g = torch.Generator(device=dev).manual_seed(6)
    w_, b_ = ([(1 + 0.1 * torch.randn(64, generator=g, device=dev)).to(torch.bfloat16) for _ in range(2)],
              [(0.05 * torch.randn(64, generator=g, device=dev)).to(torch.bfloat16) for _ in range(2)])
    ang = torch.outer(torch.arange(nv, dtype=torch.float32, device=dev), 1.0 / (256.0 ** (torch.arange(0, 64, 2, device=dev) / 64)))
    rope = (ang.cos().repeat_interleave(2, 1).contiguous(), ang.sin().repeat_interleave(2, 1).contiguous())
    q, k, v = (torch.empty(1, heads, s, 64, dtype=torch.bfloat16, device=dev) for _ in range(3))
    plan = ops.Plan(q, k, v, geo, top_k, 0.3, nbr, private_workspace=True)
    plan.ws.view(torch.uint8).fill_(0xff)
    plan.qkv_prep(*src, q_weight=w_[0], k_weight=w_[1], q_bias=b_[0], k_bias=b_[1], eps=1e-6, rope=rope, rope_rows=nv)
    names = ("q_pool", "q_mad", "k_cat", "k_mad", "v_pool")
    fused = {n: plan.view()[n].clone() for n in names}
    out_pooled = plan.run_pooled().clone()
    out_whole = plan.run().clone()           # kernel 2 pools the stored rows, then the same kernels 3a-4
    torch.cuda.synchronize()
    separate = plan.view()
    for n in names:
        assert torch.equal(fused[n].view(torch.int32), separate[n].view(torch.int32)), n
        assert not fused[n][..., 64:].any(), n
    assert torch.equal(out_pooled.view(torch.int16), out_whole.view(torch.int16))
    assert out_whole.float().abs().max().item() > 0


def _close(a, b):
    a, b = a.float().cpu().numpy(), b.float().cpu().numpy()
    assert cos_sim(a, b) >= 0.999 and abs(a - b).max() <= 4e-2 * max(1.0, abs(b).max())


def _cog_layer(dev, heads=4, dim=256, nv=1024, n_txt=226, seed=0):
    from rectified_spaattn import _processors as P
    torch.manual_seed(seed)
    attn = FakeAttention(dim, heads, head_dim=64, norm="layer").to(dev).to(torch.bfloat16)
    g = torch.Generator(device=dev).manual_seed(seed + 1)
    mu = torch.cumsum(torch.randn(nv // 128, dim, generator=g, device=dev) * 0.35, dim=0).repeat_interleave(128, dim=0)
    x = (torch.randn(nv, dim, generator=g, device=dev) + mu)[None].to(torch.bfloat16)
    txt = torch.randn(1, n_txt, dim, generator=g, device=dev).to(torch.bfloat16)
    ang = torch.outer(torch.arange(nv, dtype=torch.float32, device=dev), 1.0 / (256.0 ** (torch.arange(0, 64, 2, device=dev) / 64)))
    rope = (ang.cos().repeat_interleave(2, 1).contiguous(), ang.sin().repeat_interleave(2, 1).contiguous())
    return P, attn, x, txt, rope


@pytest.mark.gpu
def test_cogvideox_processor_takes_kernel0(dev):
    """The CogVideoX processor on a 64-dimensional-head module (LayerNorm(64) with bias) runs kernel 0: the fused section
    returns a tensor, and the layer agrees with the op-by-op path (fuse_prep = False) and, in the dense limit, with
    SDPA through the same module."""
    from rectified_spaattn import rectified_cogvideo_attn as cog
    P, attn, x, txt, rope = _cog_layer(dev)
    nv, n_txt, heads = x.shape[1], txt.shape[1], attn.heads
    with torch.no_grad():
        hs = torch.cat([x, txt], dim=1)
        fused = P.fused_prep_attention(attn, hs, None, G.cogvideo(hs.shape[1], n_txt), 99, 0.3, None, rope,
                                       rope_text=False)
        assert fused is not None and fused.shape == (1, nv + n_txt, heads * 64)
        outs = {}
        for fuse in (True, False):
            pr = cog.RectifiedCogVideoXVideoSpaAttnProcessor2_0("sparse", 99, None, 0.3)
            pr.fuse_prep = fuse
            pr.current_step = 5
            outs[fuse] = pr(attn, x, txt, None, rope)
        q, k, v = (P.heads_first(f(hs), heads) for f in (attn.to_q, attn.to_k, attn.to_v))
        q, k = attn.norm_q(q), attn.norm_k(k)
        q = torch.cat([P.rope_real(q[:, :, :nv], rope), q[:, :, nv:]], dim=2)
        k = torch.cat([P.rope_real(k[:, :, :nv], rope), k[:, :, nv:]], dim=2)
        o = torch.nn.functional.scaled_dot_product_attention(q, k, v).transpose(1, 2).flatten(2, 3)
        o = attn.to_out[1](attn.to_out[0](o))
        via_fused = attn.to_out[1](attn.to_out[0](fused))
    for i in range(2):
        _close(outs[True][i], outs[False][i])
    _close(outs[True][0], o[:, :nv])
    _close(outs[True][1], o[:, nv:])
    # the processor's attention section is the fused one
    assert torch.equal(via_fused[:, :nv], outs[True][0]) and torch.equal(via_fused[:, nv:], outs[True][1])


@pytest.mark.gpu
def test_cogvideox_layer_records_into_a_cuda_graph(dev):
    """A whole CogVideoX attention layer through kernel 0 at 64 columns (sparse: top_k 2) records into one CUDA graph
    and replays on new inputs with the eager result, bit for bit."""
    from rectified_spaattn import rectified_cogvideo_attn as cog
    P, attn, x0, t0, rope = _cog_layer(dev)
    pr = cog.RectifiedCogVideoXVideoSpaAttnProcessor2_0("sparse", 2, None, 0.3)
    pr.current_step = 5
    g = torch.Generator(device=dev).manual_seed(3)
    xs = [x0] + [torch.randn(x0.shape, device=dev, generator=g).to(torch.bfloat16) for _ in range(1)]
    ts = [t0] + [torch.randn(t0.shape, device=dev, generator=g).to(torch.bfloat16) for _ in range(1)]
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


@pytest.mark.gpu
def test_fused_ulysses_cogvideox_two_gpus(dev):
    """The fused Ulysses exchange in CogVideoX form (64-column heads, LayerNorm with bias, rotary embedding on the video
    tokens) on 2 GPUs through torchrun: 3 heads (2 + 1) and 611 tokens (306 + 305); every rank's rows are
    bit-identical to the single-GPU call."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29580",
                        os.path.join(REPO, "tools", "check_fused_ulysses.py"), "cog"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["head_dim"] == 64 and line["rows_last_rank"] < line["rows_per_rank"] and line["heads_rank0"] == 2
    assert line["fused_equals_single_gpu_bitwise_checked_ranks"] == [True, True]
