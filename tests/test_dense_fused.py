"""Dense attention calls on the fused path: kernel 4's list-free dense form (rsa_dense_attention /
rsa_dense_attention_scatter, ABI 108), `fullattn(mode="flash")` on it, `ProcessorBase.fuse_prep_dense` (kernel 0 without
pooling, then the dense form) and `FusedUlysses.run(dense=True)`.

The dense form walks every key block of every query tile in the order pair_schedule_kernel gives all-ones lists, so it
is bit-identical to kernel 4 on an all-ones mask with flash-attn's arithmetic (masked_attention(fp32_scale=True))."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from fake_attention import FakeAttention
from helpers import cos_sim
from rsa_b200 import native as N
from rsa_b200 import ops, parallel

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARG, UNSUPPORTED = -1, -2


# ------------------------------------------------------------------------------------------------------ CPU
def _desc(b=1, h=2, s=1000, d=128, dtype=N.DTYPE_BF16):
    x = N.AttnDesc()
    x.batch, x.heads, x.seq, x.head_dim, x.dtype = b, h, s, d, dtype
    for name in ("q_stride", "k_stride", "v_stride", "o_stride"):
        arr = getattr(x, name)
        arr[0], arr[1], arr[2] = h * s * d, s * d, d
    x.family, x.n_blocks, x.kv_len = 9, -3, -1          # geometry fields: neither read nor validated
    return x


def _route(n_ranks=2, rank=0, rows=500, heads_total=4, head0=0, hd=128):
    r = N.PeerRoute()
    r.n_ranks, r.rank, r.rows_per_rank, r.heads_total, r.head0 = n_ranks, rank, rows, heads_total, head0
    r.out_table = 16                                  # never read on the host
    r.out_stride[0], r.out_stride[1] = rows * heads_total * hd, heads_total * hd
    return r


def _dense(d, q=16, k=16, v=16, out=16, seq_kv=1000, q_valid=1000, kv_len=1000):
    return N.lib().rsa_dense_attention(None if d is None else C.byref(d), q, k, v, out, seq_kv, q_valid, kv_len, None)


def _scatter(d, route, q=16, k=16, v=16, q_valid=1000, kv_len=1000):
    return N.lib().rsa_dense_attention_scatter(None if d is None else C.byref(d), q, k, v,
                                               None if route is None else C.byref(route), q_valid, kv_len, None)


def _refused(rc, code, *words):
    msg = N.lib().rsa_last_error_string().decode()
    assert rc == code, (rc, msg)
    for w in words:
        assert w in msg, (w, msg)


def test_dense_entry_points_refuse_bad_arguments():
    """Every refusal of rsa_dense_attention returns RSA_ERR_ARG / RSA_ERR_UNSUPPORTED with a message naming the cause,
    before any CUDA call (this runs without a device)."""
    _refused(_dense(None), ARG, "null")
    for kw in (dict(q=None), dict(k=None), dict(v=None), dict(out=None)):
        _refused(_dense(_desc(), **kw), ARG, "null")
    _refused(_dense(_desc(d=96)), UNSUPPORTED, "head_dim", "96")
    _refused(_dense(_desc(dtype=7)), UNSUPPORTED, "dtype 7")
    _refused(_dense(_desc(b=0)), ARG, "positive")
    _refused(_dense(_desc(), seq_kv=0), ARG, "positive")
    _refused(_dense(_desc(b=300, h=300)), UNSUPPORTED, "batch*heads")
    for qv in (0, 1001):
        _refused(_dense(_desc(), q_valid=qv), ARG, f"q_valid={qv}")
    for kl in (0, 513):
        _refused(_dense(_desc(), seq_kv=512, kv_len=kl), ARG, f"kv_len={kl}", "seq_kv=512")
    for name in ("q_stride", "k_stride", "v_stride", "o_stride"):
        d = _desc()
        getattr(d, name)[1] = 1004
        _refused(_dense(d), UNSUPPORTED, "strides")
        getattr(d, name)[1] = -8
        _refused(_dense(d), UNSUPPORTED, "strides")
    for kw in (dict(q=24), dict(k=40), dict(v=8), dict(out=1032)):
        _refused(_dense(_desc(), **kw), UNSUPPORTED, "16-byte aligned")


def test_dense_scatter_refuses_bad_arguments():
    """rsa_dense_attention_scatter: the same checks (seq_kv = seq), the route validated as for the pooled scatter, and
    head_dim 64 refused under attention flag 4 (the 128-column instantiation would place heads 128 columns apart)."""
    d = _desc()
    _refused(_scatter(None, _route()), ARG, "null")
    _refused(_scatter(d, _route(), q=None), ARG, "null")
    _refused(_scatter(d, None), ARG, "route is null")
    _refused(_scatter(d, _route(), q_valid=0), ARG, "q_valid=0")
    _refused(_scatter(d, _route(), kv_len=1001), ARG, "kv_len=1001", "seq_kv=1000")
    _refused(_scatter(_desc(d=64), _route(hd=64), k=24), UNSUPPORTED, "16-byte aligned")
    _refused(_scatter(d, _route(n_ranks=9)), ARG, "rank 0 of 9")
    _refused(_scatter(d, _route(rows=400)), ARG, "do not tile seq 1000")
    _refused(_scatter(d, _route(head0=3)), ARG, "heads [3, 5)")
    r = _route()
    r.out_stride[1] = 4 * 128 - 8
    _refused(_scatter(d, r), ARG, "result table / strides")
    r.out_table = None
    r.out_stride[1] = 4 * 128
    _refused(_scatter(d, r), ARG, "result table / strides")
    try:
        N.lib().rsa_debug_set_attention_flags(4)
        _refused(_scatter(_desc(d=64), _route(hd=64)), UNSUPPORTED, "head_dim 64", "64-column")
    finally:
        N.lib().rsa_debug_set_attention_flags(0)


def test_fused_ulysses_dense_argument_checks():
    """FusedUlysses.run(dense=...) takes a bool, and the 64-column form still needs the LayerNorm parameters; both are
    refused before any collective or CUDA call."""
    fu = object.__new__(parallel.FusedUlysses)
    fu.plan, fu.head_dim = None, 128
    with pytest.raises(TypeError, match="dense"):
        fu.run(dense="yes")
    with pytest.raises(TypeError, match="dense"):
        fu.run(dense=1)
    fu.head_dim = 64
    with pytest.raises(RuntimeError, match="LayerNorm"):
        fu.run(dense=True)


def test_dense_ops_refuse_bad_tensors():
    """ops.dense_attention has no CPU implementation and refuses a CPU tensor before touching the library."""
    q = torch.zeros(1, 2, 128, 128, dtype=torch.bfloat16)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        ops.dense_attention(q, q, q, 128, 128)


# ------------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


# (batch, heads, seq, seq_kv, q_valid, kv_len, dtype, head_dim, strided, out layout)
CASES = {
    "s1000": (1, 3, 1000, 1000, 1000, 1000, torch.bfloat16, 128, False, "bhsd"),
    "s1250": (1, 3, 1250, 1250, 1250, 1250, torch.bfloat16, 128, False, "bshd"),
    "kv_len_lt_s": (1, 2, 1250, 1250, 1250, 1100, torch.bfloat16, 128, False, "bhsd"),
    "q_valid_lt_s": (1, 2, 1250, 1250, 1057, 1250, torch.bfloat16, 128, False, "bshd"),
    "batch2_strided": (2, 3, 1000, 1000, 950, 990, torch.bfloat16, 128, True, "bshd"),
    "fp16": (2, 3, 1250, 1250, 1200, 1130, torch.float16, 128, True, "bhsd"),
    "hd64": (1, 5, 1250, 1250, 1250, 1250, torch.bfloat16, 64, False, "bshd"),
    "hd64_fp16_strided": (2, 3, 1000, 1000, 999, 870, torch.float16, 64, True, "bhsd"),
    "seq_kv_512": (1, 4, 4096, 512, 4096, 512, torch.bfloat16, 128, False, "bshd"),
    "seq_kv_512_hd64": (1, 3, 4096, 512, 4000, 500, torch.bfloat16, 64, True, "bhsd"),
}


def _qkv(b, h, s, skv, d, dtype, strided, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    if strided:     # [B, S, H, D] storage viewed as [B, H, S, D]: token stride H*D, head stride D
        mk = lambda n: torch.randn(b, n, h, d, generator=g, device=dev).to(dtype).permute(0, 2, 1, 3)
    else:
        mk = lambda n: torch.randn(b, h, n, d, generator=g, device=dev).to(dtype)
    return mk(s), mk(skv), mk(skv)


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_dense_bit_identical_to_masked_all_ones(dev, case):
    """dense_attention equals masked_attention(all-ones mask, fp32_scale=True) with rows >= q_valid zeroed, bit for bit,
    and SDPA over the valid rows / keys within 2e-2 max-abs and cosine 0.999."""
    b, h, s, skv, qv, kl, dtype, d, strided, layout = CASES[case]
    q, k, v = _qkv(b, h, s, skv, d, dtype, strided, dev, 7)
    mask = torch.ones(b, h, (s + 127) // 128, (skv + 127) // 128, dtype=torch.bool, device=dev)
    want = ops.masked_attention(q, k, v, mask, kl, fp32_scale=True)
    want[:, :, qv:] = 0
    out = None
    if layout == "bshd":
        out = torch.full((b, s, h, d), float("nan"), dtype=dtype, device=dev)
    got = ops.dense_attention(q, k, v, qv, kl, out=out)
    if layout == "bshd":
        assert got is out
        got = out.permute(0, 2, 1, 3)
    torch.cuda.synchronize()
    assert torch.equal(got.contiguous().view(torch.int16), want.contiguous().view(torch.int16))
    ref = F.scaled_dot_product_attention(q[:, :, :qv].float(), k[:, :, :kl].float(), v[:, :, :kl].float())
    a, r = got[:, :, :qv].float().cpu().numpy(), ref.cpu().numpy()
    assert np.abs(a - r).max() <= 2e-2 and cos_sim(a, r) >= 0.999
    assert not got[:, :, qv:].any()


@pytest.mark.gpu
def test_plan_run_dense_writes_plan_output(dev):
    """Plan.run_dense writes the plan's [B, S, H, D] output, equal to ops.dense_attention on the same tensors."""
    from rsa_b200 import geometry as G
    q, k, v = _qkv(1, 3, 1250, 1250, 128, torch.bfloat16, False, dev, 11)
    plan = ops.Plan(q, k, v, G.hunyuan(1250, 1150), 2, 0.3)
    o = plan.run_dense(1150, 1150)
    assert o is plan.out and o.shape == (1, 1250, 3, 128)
    want = ops.dense_attention(q, k, v, 1150, 1150)
    torch.cuda.synchronize()
    assert torch.equal(o.permute(0, 2, 1, 3).contiguous().view(torch.int16), want.view(torch.int16))


# ------------------------------------------------------------------------------------- processors on the GPU
def _close(a, b):
    a, b = a.float().cpu().numpy(), b.float().cpu().numpy()
    assert cos_sim(a, b) >= 0.999 and abs(a - b).max() <= 4e-2 * max(1.0, abs(b).max())


def _mk(dev, *a, **kw):
    torch.manual_seed(0)
    return FakeAttention(*a, **kw).to(dev).to(torch.bfloat16)


def _rope_tables(n, d, dev):
    ang = torch.rand(n, d // 2, device=dev) * 6.28
    return ang.cos().repeat_interleave(2, dim=1), ang.sin().repeat_interleave(2, dim=1), ang


@pytest.fixture
def dense_calls(monkeypatch):
    """Counts Plan.run_dense calls: a processor test must see the fused dense path taken, not the op-by-op fallback."""
    n = [0]
    orig = ops.Plan.run_dense

    def counted(self, *a, **kw):
        n[0] += 1
        return orig(self, *a, **kw)

    monkeypatch.setattr(ops.Plan, "run_dense", counted)
    return n


def _both(make, call, dense_calls):
    """Runs call(processor) with fuse_prep_dense True and False; returns both outputs and checks the fused one took
    the dense kernel and that both advanced current_step the same way."""
    outs, steps = {}, {}
    for fuse in (True, False):
        pr = make()
        pr.fuse_prep_dense = fuse
        before = dense_calls[0]
        step0 = pr.current_step
        with torch.no_grad():
            outs[fuse] = call(pr)
        assert (dense_calls[0] - before) == (1 if fuse else 0)
        steps[fuse] = pr.current_step - step0
    assert steps[True] == steps[False] == 1
    return outs[True], outs[False]


@pytest.mark.gpu
def test_wan_dense_calls_fused(dev, dense_calls):
    """Wan2.1 T2V warm-up call, Wan2.1 I2V on a module with image projections (dense layer 0), Wan2.2 TI2V warm-up and
    A14B dense layer 40 (cos / sin tables), and mode "flash": fused dense == op-by-op, both == SDPA.  The I2V call passes
    no context: a self-attention call with one is never fused (its keys would come from the context, as on the sparse
    path), so the image cross-attention of the fused section is covered by the direct _fused(dense=True) test below."""
    from rectified_spaattn import rectified_wan21_attn as wan21
    from rectified_spaattn import rectified_wan22_attn as wan22
    dim, heads, s = 256, 2, 1000
    x = torch.randn(1, s, dim, device=dev).to(torch.bfloat16)
    cos, sin, ang = _rope_tables(s, 128, dev)
    for cls, rope, kw, pid, step, mode in (
            (wan21.RectifiedWanT2VSpaAttnProcessor2_0, "complex", {}, 3, 0, "sparse"),
            (wan21.RectifiedWanI2VSpaAttnProcessor2_0, "complex", dict(image_ctx=True), 0, 30, "sparse"),
            (wan22.RectifiedWanTI2VSpaAttnProcessor2_0, "cos_sin", {}, 5, 4, "sparse"),
            (wan22.RectifiedWanT2VSpaAttnProcessor2_0, "cos_sin", {}, 40, 60, "sparse"),
            (wan21.RectifiedWanT2VSpaAttnProcessor2_0, "complex", {}, 7, 50, "flash")):
        attn = _mk(dev, dim, heads, norm="inner", **kw)
        emb = torch.polar(torch.ones_like(ang, dtype=torch.float64), ang.double())[None, None] if rope == "complex" \
            else (cos[None, :, None], sin[None, :, None])

        def make():
            pr = cls(mode, 99, None, 0.3, processor_id=pid, first_frame_blocks=2)
            pr.current_step = step
            return pr

        fused, unfused = _both(make, lambda pr: pr(attn, x, None, None, emb), dense_calls)
        with torch.no_grad():
            want = cls("torch", 99, None, 0.3, processor_id=pid)(attn, x, None, None, emb)
        _close(fused, unfused)
        _close(fused, want)


@pytest.mark.gpu
def test_wan_i2v_dense_adds_image_cross_attention(dev):
    """The I2V image cross-attention is added to the dense fused section exactly as to the sparse one: _fused(dense=True)
    with an image context equals the same call without it plus image_cross_attention on kernel 0's q."""
    from rectified_spaattn import _processors as P
    from rectified_spaattn import rectified_wan21_attn as wan21
    dim, heads, s = 256, 2, 1000
    attn = _mk(dev, dim, heads, norm="inner", image_ctx=True)
    x = torch.randn(1, s, dim, device=dev).to(torch.bfloat16)
    img = torch.randn(1, 257, dim, device=dev).to(torch.bfloat16)
    _, _, ang = _rope_tables(s, 128, dev)
    emb = torch.polar(torch.ones_like(ang, dtype=torch.float64), ang.double())[None, None]
    pr = wan21.RectifiedWanI2VSpaAttnProcessor2_0("sparse", 99, None, 0.3, processor_id=0)
    with torch.no_grad():
        plain = pr._fused(attn, x, emb, None, dense=True).clone()
        with_img = pr._fused(attn, x, emb, img, dense=True)
        q = P.heads_first(attn.norm_q(attn.to_q(x)), heads)
        q = P.rope_complex(q, emb)
        extra = P.image_cross_attention(attn, q, img)
    _close(with_img, plain + extra)
    assert not torch.equal(with_img, plain)


@pytest.mark.gpu
def test_hunyuan_flash_mode_fused(dev, dense_calls):
    """HunyuanVideo mode="flash": dual-stream, single-stream and a ragged visual segment (1000 video tokens), 200 of 256
    text tokens valid (q_valid = kv_len = num_true): fused dense == op-by-op, both == SDPA on the valid rows."""
    from rectified_spaattn import rectified_hunyuan_attn as hun
    dim, heads = 256, 2
    for nv in (1024, 1000):
        x = torch.randn(1, nv, dim, device=dev).to(torch.bfloat16)
        txt = torch.randn(1, 256, dim, device=dev).to(torch.bfloat16)
        cos, sin, _ = _rope_tables(nv, 128, dev)
        mask = (torch.arange(nv + 256, device=dev) < nv + 200).view(1, 1, 1, -1)
        for added in (True, False):
            attn = _mk(dev, dim, heads, added=added)
            make = lambda: hun.RectifiedHunyuanVideoSpaAttnProcessor2_0("flash", 99, None, 0.3)
            fused, unfused = _both(make, lambda pr: pr(attn, x, txt, mask, (cos, sin)), dense_calls)
            with torch.no_grad():
                hr, er = hun.RectifiedHunyuanVideoSpaAttnProcessor2_0("torch", 99, None, 0.3)(
                    attn, x, txt, mask.expand(1, 1, nv + 256, nv + 256), (cos, sin))
            _close(fused[0], unfused[0])
            _close(fused[1][:, :200], unfused[1][:, :200])
            _close(fused[0], hr)
            _close(fused[1][:, :200], er[:, :200])
            if not added:     # no output projections on a single-stream module: the padded text rows are zeros
                assert not fused[1][:, 200:].any()


@pytest.mark.gpu
def test_flux_dense_single_stream_layer_fused(dev, dense_calls):
    """A Flux single-stream block in the dense range (processor_id 40): fused dense == op-by-op == SDPA."""
    from rectified_spaattn import _processors as P
    from rectified_spaattn import rectified_flux_attn as flux
    dim, heads, nv = 256, 2, 1024
    hs = torch.randn(1, nv + 512, dim, device=dev).to(torch.bfloat16)
    cos, sin, _ = _rope_tables(nv + 512, 128, dev)
    attn = _mk(dev, dim, heads)
    make = lambda: flux.RectifiedFluxSpaAttnProcessor2_0("sparse", 99, None, 0.3, processor_id=40, text_length=512)
    fused, unfused = _both(make, lambda pr: pr(attn, hs, None, None, (cos, sin)), dense_calls)
    with torch.no_grad():
        q, k, v = (P.heads_first(f(hs), heads) for f in (attn.to_q, attn.to_k, attn.to_v))
        q, k = P.rope_real(attn.norm_q(q), (cos, sin)), P.rope_real(attn.norm_k(k), (cos, sin))
        want = F.scaled_dot_product_attention(q, k, v).transpose(1, 2).flatten(2, 3)
    _close(fused, unfused)
    _close(fused, want)


def _cog_inputs(dev, heads=4, dim=256, nv=1024, n_txt=226, seed=0):
    torch.manual_seed(seed)
    attn = FakeAttention(dim, heads, head_dim=64, norm="layer").to(dev).to(torch.bfloat16)
    g = torch.Generator(device=dev).manual_seed(seed + 1)
    x = torch.randn(1, nv, dim, generator=g, device=dev).to(torch.bfloat16)
    txt = torch.randn(1, n_txt, dim, generator=g, device=dev).to(torch.bfloat16)
    ang = torch.outer(torch.arange(nv, dtype=torch.float32, device=dev),
                      1.0 / (256.0 ** (torch.arange(0, 64, 2, device=dev) / 64)))
    rope = (ang.cos().repeat_interleave(2, 1).contiguous(), ang.sin().repeat_interleave(2, 1).contiguous())
    return attn, x, txt, rope


@pytest.mark.gpu
def test_cogvideox_call0_fused_64_columns(dev, dense_calls):
    """CogVideoX call 0 (dense) with 64-dimensional heads and LayerNorm(64): fused dense == op-by-op == SDPA."""
    from rectified_spaattn import _processors as P
    from rectified_spaattn import rectified_cogvideo_attn as cog
    attn, x, txt, rope = _cog_inputs(dev)
    nv, heads = x.shape[1], attn.heads
    make = lambda: cog.RectifiedCogVideoXVideoSpaAttnProcessor2_0("sparse", 99, None, 0.3)
    fused, unfused = _both(make, lambda pr: pr(attn, x, txt, None, rope), dense_calls)
    with torch.no_grad():
        hs = torch.cat([x, txt], dim=1)
        q, k, v = (P.heads_first(f(hs), heads) for f in (attn.to_q, attn.to_k, attn.to_v))
        q, k = attn.norm_q(q), attn.norm_k(k)
        q = torch.cat([P.rope_real(q[:, :, :nv], rope), q[:, :, nv:]], dim=2)
        k = torch.cat([P.rope_real(k[:, :, :nv], rope), k[:, :, nv:]], dim=2)
        o = F.scaled_dot_product_attention(q, k, v).transpose(1, 2).flatten(2, 3)
        o = attn.to_out[1](attn.to_out[0](o))
    for i in range(2):
        _close(fused[i], unfused[i])
    _close(fused[0], o[:, :nv])
    _close(fused[1], o[:, nv:])


@pytest.mark.gpu
def test_fused_dense_layer_records_into_a_cuda_graph(dev):
    """A HunyuanVideo attention layer in mode "flash" with fuse_prep_dense (num_true given: no host synchronisation)
    records into one CUDA graph and replays on new inputs with the eager result, bit for bit."""
    from rectified_spaattn import rectified_hunyuan_attn as hun
    dim, heads, nv = 256, 2, 1024
    attn = _mk(dev, dim, heads, added=True)
    cos, sin, _ = _rope_tables(nv, 128, dev)
    pr = hun.RectifiedHunyuanVideoSpaAttnProcessor2_0("flash", 2, None, 0.3)
    pr.num_true, pr.fuse_prep_dense = nv + 200, True
    g = torch.Generator(device=dev).manual_seed(3)
    xs = [torch.randn(1, nv, dim, device=dev, generator=g).to(torch.bfloat16) for _ in range(2)]
    ts = [torch.randn(1, 256, dim, device=dev, generator=g).to(torch.bfloat16) for _ in range(2)]
    with torch.no_grad():
        eager = [pr(attn, x, t, None, (cos, sin)) for x, t in zip(xs, ts)]
        x_in, t_in = xs[0].clone(), ts[0].clone()
        stream = torch.cuda.Stream()
        stream.wait_stream(torch.cuda.current_stream())
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.stream(stream):
            pr(attn, x_in, t_in, None, (cos, sin))
            stream.synchronize()
            with torch.cuda.graph(graph, stream=stream):
                h_out, e_out = pr(attn, x_in, t_in, None, (cos, sin))
        for x, t, ref in zip(xs, ts, eager):
            x_in.copy_(x)
            t_in.copy_(t)
            graph.replay()
            torch.cuda.synchronize()
            assert torch.equal(h_out, ref[0]) and torch.equal(e_out, ref[1])


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["odd", "c3b", "cog"])
def test_fused_ulysses_dense_two_gpus(dev, workload):
    """FusedUlysses.run(dense=True) on 2 GPUs through torchrun: every rank's rows bit-identical to the single-GPU kernel 0
    (no pooling) + Plan.run_dense.  Wan form with 3 heads on 2 ranks and 1035 tokens, the ragged HunyuanVideo form
    (129 frames), and the CogVideoX form (64-column heads)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    port = {"odd": 29591, "c3b": 29592, "cog": 29593}[workload]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port),
                        os.path.join(REPO, "tools", "check_fused_ulysses.py"), workload, "--dense"],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["dense"] is True
    checked = line["fused_equals_single_gpu_bitwise_checked_ranks"]
    assert checked and all(checked)
