"""The eight Rectified*SpaAttnProcessor2_0 classes keep the reference's constructor arguments, attributes, gates,
step counters and return values (SURVEY.md 3.4, 8b).  CPU tests cover the host logic; the GPU tests run every
processor on a fake `Attention` module and check the sparse path in its dense limit (select_block_num >= NB =>
every block kept, R = 1, C = 0) against the same processor in mode "torch" (plain SDPA through the same projections)."""
import math

import pytest
import torch

from fake_attention import FakeAttention
from helpers import cos_sim
from rectified_spaattn import rectified_cogvideo_attn as cog
from rectified_spaattn import rectified_flux_attn as flux
from rectified_spaattn import rectified_hunyuan_attn as hun
from rectified_spaattn import rectified_wan21_attn as wan21
from rectified_spaattn import rectified_wan22_attn as wan22


# ------------------------------------------------------------------------------------------------ host logic
def test_constructors_and_attributes():
    p = wan21.RectifiedWanT2VSpaAttnProcessor2_0("sparse", 64, None, 0.3, processor_id=5, first_frame_blocks=12)
    assert (p.mode, p.select_block_num, p.p_remain_rates, p.current_step, p.processor_id, p.first_frame_blocks) == \
        ("sparse", 64, 0.3, 0, 5, 12)
    p = wan22.RectifiedWanT2VSpaAttnProcessor2_0("sparse", 147, None, 0.3, 7, 28, warm_steps=10)
    assert p.warm_steps == 10 and p.steps_per_cycle == 80
    p = flux.RectifiedFluxSpaAttnProcessor2_0("sparse", 51, None, 0.3, processor_id=3, text_length=512)
    assert p.text_length == 512
    for cls in (hun.RectifiedHunyuanVideoSpaAttnProcessor2_0, cog.RectifiedCogVideoXVideoSpaAttnProcessor2_0):
        q = cls("sparse", 179, None, 0.3, processor_id=1)
        assert q.block_neighbor_list is None and q.current_step == 0


def test_warmup_gates_match_reference():
    t2v = wan21.RectifiedWanT2VSpaAttnProcessor2_0("sparse", 1, None, 0.3, processor_id=2)
    assert not t2v.sparse_now()
    t2v.current_step = 10
    assert t2v.sparse_now()
    t2v.processor_id = 1
    assert not t2v.sparse_now()                                          # first two layers stay dense
    i2v = wan21.RectifiedWanI2VSpaAttnProcessor2_0("sparse", 1, None, 0.3, processor_id=2)
    assert i2v.sparse_now()                                              # no step warm-up for I2V
    a14 = wan22.RectifiedWanI2VSpaAttnProcessor2_0("sparse", 1, None, 0.3, processor_id=40, warm_steps=4)
    a14.current_step = 50
    assert not a14.sparse_now()                                          # layers 0, 1, 40, 41 stay dense
    a14.processor_id = 42
    assert a14.sparse_now()
    a14.current_step = 3
    assert not a14.sparse_now()
    for _ in range(77):
        a14._tick()
    assert a14.current_step == 0                                         # 3 + 77 = 80 -> wraps


def test_rope_helpers_agree():
    from rectified_spaattn import _processors as P
    g = torch.Generator().manual_seed(0)
    x = torch.randn(1, 2, 8, 16, generator=g)
    ang = torch.rand(8, 8, generator=g) * 6.28
    cos, sin = ang.cos().repeat_interleave(2, dim=1), ang.sin().repeat_interleave(2, dim=1)
    a = P.rope_real(x, (cos, sin))
    b = P.rope_complex(x, torch.polar(torch.ones(8, 8, dtype=torch.float64), ang.double())[None, None])
    c = P.rope_cos_sin(x.transpose(1, 2), cos[None, :, None], sin[None, :, None]).transpose(1, 2)
    assert torch.allclose(a, b, atol=1e-5) and torch.allclose(a, c, atol=1e-5)


# ------------------------------------------------------------------------------------------------ on the GPU
def _mk(dev, *a, **kw):
    torch.manual_seed(0)
    return FakeAttention(*a, **kw).to(dev).to(torch.bfloat16)


def _rope_tables(n, d, dev):
    ang = torch.rand(n, d // 2, device=dev) * 6.28
    return ang.cos().repeat_interleave(2, dim=1), ang.sin().repeat_interleave(2, dim=1), ang


def _close(a, b):
    a, b = a.float().cpu().numpy(), b.float().cpu().numpy()
    assert cos_sim(a, b) >= 0.999 and abs(a - b).max() <= 4e-2 * max(1.0, abs(b).max())


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


@pytest.mark.gpu
def test_wan_processors_dense_limit(dev):
    dim, heads, s = 256, 2, 1000
    x = torch.randn(1, s, dim, device=dev).to(torch.bfloat16)
    cos, sin, ang = _rope_tables(s, 128, dev)
    for cls, rope, kw in ((wan21.RectifiedWanT2VSpaAttnProcessor2_0, "complex", {}),
                          (wan21.RectifiedWanI2VSpaAttnProcessor2_0, "complex", dict(image_ctx=True)),
                          (wan22.RectifiedWanTI2VSpaAttnProcessor2_0, "cos_sin", {}),
                          (wan22.RectifiedWanT2VSpaAttnProcessor2_0, "cos_sin", {})):
        attn = _mk(dev, dim, heads, norm="inner", **kw)
        emb = torch.polar(torch.ones_like(ang, dtype=torch.float64), ang.double())[None, None] if rope == "complex" \
            else (cos[None, :, None], sin[None, :, None])
        enc = torch.randn(1, 257 + 512, dim, device=dev).to(torch.bfloat16) if kw else None
        sp = cls("sparse", 99, None, 0.3, processor_id=3, first_frame_blocks=2)
        ref = cls("torch", 99, None, 0.3, processor_id=3, first_frame_blocks=2)
        sp.current_step = 20
        with torch.no_grad():
            if kw:   # I2V: self-attention keys come from hidden_states only when no text context is passed
                out, want = sp(attn, x, None, None, emb), ref(attn, x, None, None, emb)
            else:
                out, want = sp(attn, x, None, None, emb), ref(attn, x, None, None, emb)
        assert out.shape == (1, s, dim) and sp.current_step == 21
        _close(out, want)
        # warm-up call (dense through kernel 4 as "flash") gives the same answer
        warm = cls("sparse", 99, None, 0.3, processor_id=0, first_frame_blocks=2)
        with torch.no_grad():
            _close(warm(attn, x, None, None, emb), want)
    with pytest.raises(ImportError):
        wan21.RectifiedWanT2VSpaAttnProcessor2_0("bogus", 1, None, 0.3)(attn, x, None, None, None)


@pytest.mark.gpu
def test_joint_text_processors_dense_limit(dev):
    dim, heads, nv = 256, 2, 1024
    x = torch.randn(1, nv, dim, device=dev).to(torch.bfloat16)
    cos, sin, _ = _rope_tables(nv, 128, dev)
    # HunyuanVideo dual-stream block: 256 text tokens, 200 valid
    attn = _mk(dev, dim, heads, added=True)
    txt = torch.randn(1, 256, dim, device=dev).to(torch.bfloat16)
    mask = (torch.arange(nv + 256, device=dev) < nv + 200).view(1, 1, 1, -1)
    sp = hun.RectifiedHunyuanVideoSpaAttnProcessor2_0("sparse", 99, None, 0.3)
    ref = hun.RectifiedHunyuanVideoSpaAttnProcessor2_0("torch", 99, None, 0.3)
    with torch.no_grad():
        h, e = sp(attn, x, txt, mask, (cos, sin))
        hr, er = ref(attn, x, txt, mask.expand(1, 1, nv + 256, nv + 256), (cos, sin))
    assert h.shape == (1, nv, dim) and e.shape == (1, 256, dim) and sp.current_step == 1
    _close(h, hr)
    _close(e[:, :200], er[:, :200])            # padded text rows are undefined in the reference, zeros here
    # Flux dual-stream block, 512 text tokens, RoPE over the joint sequence
    cos2, sin2, _ = _rope_tables(nv + 512, 128, dev)
    txt = torch.randn(1, 512, dim, device=dev).to(torch.bfloat16)
    sp = flux.RectifiedFluxSpaAttnProcessor2_0("sparse", 99, None, 0.3, processor_id=1, text_length=512)
    dn = flux.RectifiedFluxSpaAttnProcessor2_0("sparse", 99, None, 0.3, processor_id=40, text_length=512)  # dense layer
    with torch.no_grad():
        h, e = sp(attn, x, txt, None, (cos2, sin2))
        hd, ed = dn(attn, x, txt, None, (cos2, sin2))
    _close(h, hd)
    _close(e, ed)
    # CogVideoX: 226 text tokens (ragged: 1024 + 226 = 1250 tokens), sparse from call 5 on
    attn = _mk(dev, dim, heads)
    txt = torch.randn(1, 226, dim, device=dev).to(torch.bfloat16)
    sp = cog.RectifiedCogVideoXVideoSpaAttnProcessor2_0("sparse", 99, None, 0.3)
    with torch.no_grad():
        hd, ed = sp(attn, x, txt, None, (cos, sin))      # call 0: dense
        sp.current_step = 5
        h, e = sp(attn, x, txt, None, (cos, sin))        # sparse, dense limit
    assert h.shape == (1, nv, dim) and e.shape == (1, 226, dim)
    _close(h, hd)
    _close(e, ed)


@pytest.mark.gpu
def test_fused_prep_processors_match_unfused(dev):
    """HunyuanVideo / Flux processors with kernel 0 (head split + QK RMSNorm + RoPE + pooling fused, the default) against
    the same processors running those steps op by op (`fuse_prep = False`): dual-stream, single-stream and a ragged
    visual segment.  (torch.nn.RMSNorm rounds once where diffusers' RMSNorm -- which kernel 0 follows -- rounds twice,
    so rows differ by at most a bf16 ulp before the attention; the dense limit keeps the block choice out of it.)"""
    dim, heads = 256, 2
    for nv in (1024, 1000):
        x = torch.randn(1, nv, dim, device=dev).to(torch.bfloat16)
        txt = torch.randn(1, 256, dim, device=dev).to(torch.bfloat16)
        cos, sin, _ = _rope_tables(nv, 128, dev)
        mask = (torch.arange(nv + 256, device=dev) < nv + 200).view(1, 1, 1, -1)
        for added in (True, False):                      # dual-stream / single-stream block
            attn = _mk(dev, dim, heads, added=added)
            outs = []
            for fuse in (True, False):
                if not fuse and nv % 128:
                    continue                              # the op-by-op path is the reference's: aligned only
                pr = hun.RectifiedHunyuanVideoSpaAttnProcessor2_0("sparse", 99, None, 0.3)
                pr.fuse_prep = fuse
                with torch.no_grad():
                    outs.append(pr(attn, x, txt, mask, (cos, sin)))
            if len(outs) == 2:
                _close(outs[0][0], outs[1][0])
                _close(outs[0][1][:, :200], outs[1][1][:, :200])
            else:                                         # ragged: against dense SDPA through the same modules
                ref = hun.RectifiedHunyuanVideoSpaAttnProcessor2_0("torch", 99, None, 0.3)
                with torch.no_grad():
                    hr, er = ref(attn, x, txt, mask.expand(1, 1, nv + 256, nv + 256), (cos, sin))
                _close(outs[0][0], hr)
                _close(outs[0][1][:, :200], er[:, :200])
    # Flux: dual-stream (text appended, rotated) and single-stream (one joint tensor)
    nv = 1024
    x = torch.randn(1, nv, dim, device=dev).to(torch.bfloat16)
    txt = torch.randn(1, 512, dim, device=dev).to(torch.bfloat16)
    cos2, sin2, _ = _rope_tables(nv + 512, 128, dev)
    for added, args in ((True, (x, txt)), (False, (torch.cat([x, txt], dim=1), None))):
        attn = _mk(dev, dim, heads, added=added)
        outs = []
        for fuse in (True, False):
            pr = flux.RectifiedFluxSpaAttnProcessor2_0("sparse", 99, None, 0.3, processor_id=1, text_length=512)
            pr.fuse_prep = fuse
            with torch.no_grad():
                outs.append(pr(attn, args[0], args[1], None, (cos2, sin2)))
        if added:
            _close(outs[0][0], outs[1][0])
            _close(outs[0][1], outs[1][1])
        else:
            _close(outs[0], outs[1])
    # CogVideoX: LayerNorm(head_dim) with bias, 226 text tokens (ragged end), sparse from call 5 on
    attn = _mk(dev, dim, heads, norm="layer")
    txt = torch.randn(1, 226, dim, device=dev).to(torch.bfloat16)
    cos, sin, _ = _rope_tables(nv, 128, dev)
    outs = []
    for fuse in (True, False):
        pr = cog.RectifiedCogVideoXVideoSpaAttnProcessor2_0("sparse", 99, None, 0.3)
        pr.fuse_prep, pr.current_step = fuse, 5
        with torch.no_grad():
            outs.append(pr(attn, x, txt, None, (cos, sin)))
    _close(outs[0][0], outs[1][0])
    _close(outs[0][1], outs[1][1])


@pytest.mark.gpu
def test_whole_layer_records_into_a_cuda_graph(dev):
    """SURVEY 8f rank 3, last clause: with the host synchronisations gone (the caller supplies `num_true`), a whole
    attention layer through the processor protocol -- projections, kernel 0, kernels 3a-4, output projections --
    records into one CUDA graph and replays on new inputs with the eager result, bit for bit."""
    dim, heads, nv = 256, 2, 1024
    attn = _mk(dev, dim, heads, added=True)
    cos, sin, _ = _rope_tables(nv, 128, dev)
    pr = hun.RectifiedHunyuanVideoSpaAttnProcessor2_0("sparse", 2, None, 0.3)
    pr.num_true = nv + 200
    g = torch.Generator(device=dev).manual_seed(3)
    xs = [torch.randn(1, nv, dim, device=dev, generator=g).to(torch.bfloat16) for _ in range(2)]
    ts = [torch.randn(1, 256, dim, device=dev, generator=g).to(torch.bfloat16) for _ in range(2)]
    with torch.no_grad():
        eager = [pr(attn, x, t, None, (cos, sin)) for x, t in zip(xs, ts)]      # also warms up every lazy allocation
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
def test_processor_mask_refresh_interval(dev):
    """`mask_refresh_interval = 2`: the second call of a layer keeps the first call's block selection (fused and
    op-by-op paths); on unchanged inputs that is bit-identical to rebuilding, and the third call rebuilds."""
    dim, heads, nv = 256, 2, 2048
    attn = _mk(dev, dim, heads, added=True)
    cos, sin, _ = _rope_tables(nv, 128, dev)
    x = torch.randn(1, nv, dim, device=dev).to(torch.bfloat16)
    txt = torch.randn(1, 256, dim, device=dev).to(torch.bfloat16)
    for fuse in (True, False):
        plain = hun.RectifiedHunyuanVideoSpaAttnProcessor2_0("sparse", 2, None, 0.3)
        cached = hun.RectifiedHunyuanVideoSpaAttnProcessor2_0("sparse", 2, None, 0.3)
        plain.fuse_prep = cached.fuse_prep = fuse
        plain.num_true = cached.num_true = nv + 200
        cached.mask_refresh_interval = 2
        with torch.no_grad():
            ref = plain(attn, x, txt, None, (cos, sin))
            outs = [cached(attn, x, txt, None, (cos, sin)) for _ in range(3)]
        torch.cuda.synchronize()
        c = cached._mask_cache()
        assert c.calls == 3 and c.valid
        for o in outs:
            assert torch.equal(o[0], ref[0]) and torch.equal(o[1], ref[1])


@pytest.mark.gpu
def test_cogvideox_processor_with_64_dim_heads(dev):
    """CogVideoX1.5's real geometry: 64-dimensional heads, LayerNorm(64) on q/k, 226 text tokens.  Kernel 0 does not
    apply (it is built for 128 columns), so the processor runs the reference's op sequence and the attention goes
    through kernels 2-4 with head_dim 64 (missing columns read as zeros); dense warm-up call (kernel 4, all blocks) and
    sparse call in the dense limit must agree with each other and with PyTorch SDPA through the same module."""
    from rectified_spaattn import _processors as P
    dim, heads, nv = 256, 4, 1024
    attn = FakeAttention(dim, heads, head_dim=64, norm="layer").to(dev).to(torch.bfloat16)
    x = torch.randn(1, nv, dim, device=dev).to(torch.bfloat16)
    txt = torch.randn(1, 226, dim, device=dev).to(torch.bfloat16)
    cos, sin, _ = _rope_tables(nv, 64, dev)
    sp = cog.RectifiedCogVideoXVideoSpaAttnProcessor2_0("sparse", 99, None, 0.3)
    with torch.no_grad():
        hd, ed = sp(attn, x, txt, None, (cos, sin))      # call 0: dense (warm-up), kernel 4 with every block kept
        sp.current_step = 5
        h, e = sp(attn, x, txt, None, (cos, sin))        # sparse, dense limit
        # the same layer by hand with SDPA
        hs = torch.cat([x, txt], dim=1)                  # the processor moves the text tokens last
        q, k, v = (P.heads_first(f(hs), heads) for f in (attn.to_q, attn.to_k, attn.to_v))
        q, k = attn.norm_q(q), attn.norm_k(k)
        q = torch.cat([P.rope_real(q[:, :, :nv], (cos, sin)), q[:, :, nv:]], dim=2)
        k = torch.cat([P.rope_real(k[:, :, :nv], (cos, sin)), k[:, :, nv:]], dim=2)
        o = torch.nn.functional.scaled_dot_product_attention(q, k, v).transpose(1, 2).flatten(2, 3)
        o = attn.to_out[1](attn.to_out[0](o))
    assert h.shape == (1, nv, dim) and e.shape == (1, 226, dim)
    _close(h, hd)
    _close(e, ed)
    _close(h, o[:, :nv])
    _close(e, o[:, nv:])


def test_wan_rope_cache_is_keyed_by_tensor_identity():
    """ADVICE r1: diffusers rebuilds rotary_emb on every forward and the allocator re-uses addresses, so (pointer, shape,
    version) alone can name two different tables.  A hit needs the SAME tensor object; anything else is recomputed."""
    import torch
    from rectified_spaattn import _processors as P
    n = 16
    ang = torch.rand(1, 1, n, 64)
    emb = torch.polar(torch.ones_like(ang), ang)
    cos1, sin1 = P.wan_rope_tables(emb, n)
    assert P.wan_rope_tables(emb, n)[0] is cos1                      # same object: cached
    other = torch.polar(torch.ones_like(ang), ang + 0.5)
    emb.data.copy_(other)                                            # same pointer, shape AND version, new contents
    alias = emb.view(emb.shape)                                      # ... seen through another tensor object
    assert alias.data_ptr() == emb.data_ptr() and alias._version == emb._version
    cos2, _ = P.wan_rope_tables(alias, n)
    assert cos2 is not cos1
    assert torch.allclose(cos2[:, 0::2], other.real.reshape(n, 64).float())
