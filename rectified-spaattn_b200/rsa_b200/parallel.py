"""Multi-GPU host logic for the rectified sparse-attention path: one process per GPU (torch.distributed, NCCL over
NVLink 5 / NVSwitch on the B200 box; gloo in the CPU tests).

The path is independent per (batch, head) end to end -- pooling, scoring, selection, attention and rectification
all run per head (reference grid axis B*H, rectified_wan21_attn.py:138) -- so the natural sharding is
HEAD-PARALLEL with no collective on the data path: every rank runs the same call on its own contiguous slice of
heads.  The reference itself has no multi-GPU path for one attention call (it only fans prompts out over GPUs,
eval/video/experiments/multigpu_hunyuan.py:287-298); its `shape_xfuse` flag (rectified_wan21_attn.py:290,
:353-357) is the hook an Ulysses-style sequence-parallel wrapper would use, and that wrapper is what
`ulysses_attention` provides: one all-to-all turns sequence-sharded Q/K/V into head-sharded full sequences, the
local call runs unchanged, one all-to-all brings the output back.
"""
from __future__ import annotations

import torch
import torch.distributed as dist


def shard_heads(heads: int, world: int, rank: int):
    """(first_head, n_local_heads) of `rank`: contiguous, remainder heads go to the lowest ranks."""
    if world < 1 or not 0 <= rank < world:
        raise ValueError(f"bad rank/world {rank}/{world}")
    base, rem = divmod(heads, world)
    n = base + (1 if rank < rem else 0)
    first = rank * base + min(rank, rem)
    return first, n


def seq_to_head_shard(x: torch.Tensor, group=None) -> torch.Tensor:
    """[B, H, S/P, D] on every rank (sequence-sharded, all heads) -> [B, H/P, S, D] (all tokens, own heads).

    One all_to_all_single: rank r sends its tokens of head-group g to rank g.  H must divide by P and every rank
    must hold the same number of tokens (pad the sequence before sharding, as the Wan/CogVideoX paths do)."""
    world = dist.get_world_size(group)
    if world == 1:
        return x
    b, h, s_loc, d = x.shape
    if h % world:
        raise ValueError(f"{h} heads do not split over {world} ranks")
    hl = h // world
    # send buffer ordered by destination rank: [P, B, H/P, S/P, D]
    send = x.reshape(b, world, hl, s_loc, d).permute(1, 0, 2, 3, 4).contiguous()
    recv = torch.empty_like(send)
    dist.all_to_all_single(recv, send, group=group)
    # recv[src] = tokens of rank src's sequence slice for my heads -> concatenate along the sequence
    return recv.permute(1, 2, 0, 3, 4).reshape(b, hl, world * s_loc, d)


def head_to_seq_shard(o: torch.Tensor, group=None) -> torch.Tensor:
    """[B, S, H/P, D] (all tokens, own heads; the `shape_xfuse=True` layout) -> [B, S/P, H, D] (own tokens, all
    heads).  Inverse exchange of seq_to_head_shard for the attention output."""
    world = dist.get_world_size(group)
    if world == 1:
        return o
    b, s, hl, d = o.shape
    if s % world:
        raise ValueError(f"{s} tokens do not split over {world} ranks")
    s_loc = s // world
    send = o.reshape(b, world, s_loc, hl, d).permute(1, 0, 2, 3, 4).contiguous()  # [P(dst), B, S/P, H/P, D]
    recv = torch.empty_like(send)
    dist.all_to_all_single(recv, send, group=group)
    # recv[src] = my tokens for rank src's heads -> concatenate along the head axis in rank order
    return recv.permute(1, 2, 0, 3, 4).reshape(b, s_loc, world * hl, d)


def ulysses_attention(q, k, v, attention_fn, group=None):
    """Sequence-parallel wrapper: q, k, v are [B, H, S/P, D] shards; `attention_fn(q, k, v)` takes [B, H/P, S, D]
    and returns [B, S, H/P, D] (call the per-model entry point with shape_xfuse=True).  Returns [B, S/P, H*D]."""
    ql, kl, vl = (seq_to_head_shard(t, group) for t in (q, k, v))
    o = attention_fn(ql, kl, vl)
    o = head_to_seq_shard(o, group)
    b, s_loc, h, d = o.shape
    return o.reshape(b, s_loc, h * d)


# ------------------------------------------------------------------------------------------ fused exchange
class _RawDevice:
    """Exposes a raw device pointer to torch.as_tensor through __cuda_array_interface__."""

    def __init__(self, ptr, shape, typestr="<u2"):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 3}


def _peer_tensor(ptr, shape, dtype=torch.bfloat16):
    return torch.as_tensor(_RawDevice(ptr, shape), device="cuda").view(dtype)


class FusedUlysses:
    """Ulysses sequence parallelism without data collectives (one process per GPU of one NVSwitch box).

    Rank r owns the consecutive tokens [r * rows, min((r + 1) * rows, S)), rows = ceil(S / P) (`self.local_rows` of
    them: the last rank may hold fewer).  It writes its Q/K/V projection outputs [B, local_rows, H*D] into
    peer-visible buffers (`self.q_src`, `self.k_src`, `self.v_src`); `run()` then
      1. barrier (one-element all_reduce: every rank's sources are written),
      2. kernel 0 in gather form: reads, for this rank's H/P heads, every token's rows straight from the owning rank's
         buffer over NVLink, applies head split / RMSNorm or LayerNorm / rotary embedding, stores local [B, H/P, S, D]
         and pools,
      3. kernels 3a-3c, kernel 4 with the scatter epilogue: every output row is stored straight into the owning rank's
         result buffer [B, rows, H, D],
      4. barrier (every rank's scatter has landed),
    and returns this rank's rows of the result, [B, rows, H*D] -- what `ulysses_attention` computes with two
    all-to-alls (233 + 78 MB per GPU at C3a, P = 8) and two staging copies around the call.
    run(dense=True) is the form for calls that attend densely (warm-up steps, dense layers): kernel 0 gathers without
    pooling and kernel 4's list-free dense form scatters, between the same two barriers.
    D = head_dim: 128, or 64 (CogVideoX; run() then needs the LayerNorm parameters q_weight, k_weight, q_bias, k_bias).
    dtype: torch.bfloat16 or torch.float16, the dtype of the peer buffers, of the plan's tensors and of the norm
    parameters (converted to it in run()); kernel 0 rounds where diffusers rounds, in that format."""

    def __init__(self, batch, heads_total, geo, top_k, p_remain, nbr=None, group=None, head_dim=128,
                 dtype=torch.bfloat16):
        from . import native as N
        from . import ops
        import ctypes as C
        if dtype not in (torch.bfloat16, torch.float16):
            raise ValueError(f"dtype must be torch.bfloat16 or torch.float16 (got {dtype})")
        self.group = group
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        if self.world > 8:
            raise ValueError("at most 8 ranks (one NVSwitch box)")
        if heads_total < self.world:
            raise ValueError("every rank must compute at least one head")
        if head_dim not in (128, 64):
            raise ValueError("head_dim must be 128 or 64")
        self.head_dim = hd = head_dim
        self.dtype = dtype
        # heads need not divide by the ranks: the first (H mod P) ranks take one head more (12 heads on 8 ranks:
        # 2,2,2,2,1,1,1,1); this rank computes heads [head0, head0 + heads)
        base, extra = divmod(heads_total, self.world)
        self.batch, self.heads_total = batch, heads_total
        self.heads = base + (1 if self.rank < extra else 0)
        self.head0 = self.rank * base + min(self.rank, extra)
        self.seq = geo.seq
        self.rows = -(-geo.seq // self.world)           # rows per rank the buffers are laid out for
        if self.rows * (self.world - 1) >= geo.seq:
            raise ValueError("every rank must own at least one token")
        self.local_rows = min(self.rows, geo.seq - self.rank * self.rows)
        self.device = torch.device("cuda", torch.cuda.current_device())
        L = N.lib()
        self._lib, self._own, self._opened = L, [], []
        n_elems = batch * self.rows * heads_total * hd
        ptrs = []
        # q, k, v sources, the result, and the per-token RMS statistics of q and k (Wan's norm across heads: every rank
        # computes them from the full rows of ITS tokens, the gathering ranks read them over NVLink)
        sizes = [n_elems * 2] * 4 + [batch * self.rows * 4] * 2
        for nbytes in sizes:
            ptr = C.c_void_p()
            N.check(L.rsa_peer_alloc(nbytes, C.byref(ptr)), "rsa_peer_alloc")
            self._own.append(ptr.value)
            h = (C.c_char * 64)()
            N.check(L.rsa_peer_export(ptr, h), "rsa_peer_export")
            ptrs.append(bytes(h))
        everyone = [None] * self.world
        dist.all_gather_object(everyone, ptrs, group=group)
        table = torch.empty(6, self.world, dtype=torch.int64)
        for r in range(self.world):
            for t in range(6):
                if r == self.rank:
                    table[t, r] = self._own[t]
                else:
                    pp = C.c_void_p()
                    N.check(L.rsa_peer_open(C.create_string_buffer(everyone[r][t], 64), C.byref(pp)), "rsa_peer_open")
                    self._opened.append(pp.value)
                    table[t, r] = pp.value
        self._table = table.to(self.device)
        shape = (batch, self.rows, heads_total * hd)
        # views of this rank's own rows (the buffers themselves hold `rows` rows on every rank)
        self.q_src, self.k_src, self.v_src, self.out = (_peer_tensor(p, shape, dtype)[:, :self.local_rows]
                                                        for p in self._own[:4])
        self._flag = torch.zeros(1, device=self.device)
        q, k, v = (torch.empty(batch, self.heads, self.seq, hd, dtype=dtype, device=self.device)
                   for _ in range(3))
        self.plan = ops.Plan(q, k, v, geo, top_k, p_remain, nbr, private_workspace=True)
        route = N.PeerRoute()
        route.n_ranks, route.rank, route.rows_per_rank, route.heads_total = self.world, self.rank, self.rows, heads_total
        route.head0 = self.head0
        route.src_table = self._table[:3].data_ptr()
        route.out_table = self._table[3].data_ptr()
        route.src_stride[0], route.src_stride[1] = self.rows * heads_total * hd, heads_total * hd
        route.out_stride[0], route.out_stride[1] = self.rows * heads_total * hd, heads_total * hd
        route.rinv_table = self._table[4:6].data_ptr()
        self.route = route

    def _barrier(self):
        dist.all_reduce(self._flag, group=self.group)       # stream-ordered, one element: nothing but a barrier

    def run(self, q_weight=None, k_weight=None, eps=1e-6, rope=None, rope_rows=None, q_bias=None, k_bias=None,
            dense=False):
        """q_weight / k_weight: RMSNorm weights ([128] per head, or [heads_total*128] across heads); with q_bias /
        k_bias: LayerNorm over head_dim (CogVideoX), the only norm at head_dim 64.  dense=True: dense attention over the
        geometry's valid tokens (memory rows: num_true for HunyuanVideo, S otherwise) instead of the sparse call."""
        from . import native as N
        from . import ops
        import ctypes as C
        if not isinstance(dense, bool):
            raise TypeError("dense must be True or False")
        plan = self.plan
        hd = self.head_dim
        if hd == 64 and (q_weight is None or q_bias is None):
            raise RuntimeError("head_dim 64 is built for CogVideoX's LayerNorm: q_weight, k_weight, q_bias, k_bias")
        p = N.PrepDesc()
        p.rows, p.dst_row = self.seq, 0
        keep = []
        if q_weight is not None:
            ws_ = [w.detach().to(device=self.device, dtype=self.dtype).contiguous() for w in (q_weight, k_weight)]
            keep += ws_
            p.norm, p.eps, p.q_weight, p.k_weight = 1, float(eps), ws_[0].data_ptr(), ws_[1].data_ptr()
            if q_bias is not None or k_bias is not None:    # LayerNorm over head_dim (CogVideoX)
                bs_ = [x.detach().to(device=self.device, dtype=self.dtype).contiguous() for x in (q_bias, k_bias)]
                if any(x.numel() != hd for x in ws_ + bs_):
                    raise RuntimeError("LayerNorm weights and biases must have head_dim elements")
                keep += bs_
                p.norm, p.q_bias, p.k_bias = 3, bs_[0].data_ptr(), bs_[1].data_ptr()
            elif all(w.numel() == self.heads_total * 128 for w in ws_):
                # RMSNorm over all heads*128 channels of a token (Wan, rectified_wan21_attn.py:423-426): the statistic
                # needs whole rows, which only the owning rank holds -> computed here, before the barrier
                p.norm = 2
                st2 = (C.c_int64 * 2)(self.rows * self.heads_total * 128, self.heads_total * 128)
                with torch.cuda.device(self.device):
                    # the statistics buffers are [batch, rows] like every peer buffer; rsa_row_rms packs its output as
                    # [batch, its row count], so a short last shard is done one batch element at a time
                    even = self.local_rows == self.rows
                    dtc = N.DTYPE_F16 if self.dtype == torch.float16 else N.DTYPE_BF16
                    for b in range(1 if even else self.batch):
                        off = b * self.rows
                        N.check(self._lib.rsa_row_rms_dtype(self._own[0] + off * self.heads_total * 256,
                                                            self._own[1] + off * self.heads_total * 256,
                                                            self.batch if even else 1, self.local_rows,
                                                            self.heads_total * 128, st2, st2, float(eps),
                                                            self._own[4] + off * 4, self._own[5] + off * 4, dtc,
                                                            ops._stream(self.device)), "rsa_row_rms_dtype")
            elif any(w.numel() != 128 for w in ws_):
                raise RuntimeError("norm weights must have 128 (per head) or heads*128 (across heads) elements")
        if rope is not None:
            cos, sin = (t.detach().to(device=self.device, dtype=torch.float32).contiguous() for t in rope)
            keep += [cos, sin]
            p.rope_rows = cos.shape[0] if rope_rows is None else int(rope_rows)
            p.cos, p.sin = cos.data_ptr(), sin.data_ptr()
        self._barrier()
        st = ops._stream(self.device)
        gap = plan.desc.vis_len and plan.desc.nq_blocks * 128 - plan.desc.vis_len
        pool = 0 if dense else 1
        with torch.cuda.device(self.device):
            if gap:     # ragged visual segment: the block structure restarts at the text tokens -> two gathers
                nv = plan.desc.vis_len
                n_rope = p.rope_rows
                p.rows, p.dst_row = nv, 0
                p.rope_rows = min(n_rope, nv)
                N.check(self._lib.rsa_qkv_prep_gather(C.byref(p), C.byref(plan.desc), C.byref(self.route),
                                                      plan.q.data_ptr(), plan.k.data_ptr(), plan.v.data_ptr(), pool,
                                                      plan.ws.data_ptr(), plan.ws_bytes, st), "rsa_qkv_prep_gather")
                # text tokens: rotated with table rows [nv, rope_rows) when the tables reach past the visual tokens (Flux)
                p.rows, p.dst_row, p.rope_rows = self.seq - nv, nv, max(0, n_rope - nv)
                if p.rope_rows:
                    p.cos, p.sin = p.cos + nv * hd * 4, p.sin + nv * hd * 4
            N.check(self._lib.rsa_qkv_prep_gather(C.byref(p), C.byref(plan.desc), C.byref(self.route), plan.q.data_ptr(),
                                                  plan.k.data_ptr(), plan.v.data_ptr(), pool, plan.ws.data_ptr(),
                                                  plan.ws_bytes, st), "rsa_qkv_prep_gather")
            if dense:
                n_valid = plan.desc.kv_len - gap    # the geometry's kv_len counts the gap rows of a ragged segment
                N.check(self._lib.rsa_dense_attention_scatter(
                    C.byref(plan.desc), plan.q.data_ptr(), plan.k.data_ptr(), plan.v.data_ptr(), C.byref(self.route),
                    n_valid, n_valid, st), "rsa_dense_attention_scatter")
            else:
                N.check(self._lib.rsa_rectified_attention_pooled_scatter(
                    C.byref(plan.desc), plan.q.data_ptr(), plan.k.data_ptr(), plan.v.data_ptr(), C.byref(self.route),
                    plan.ws.data_ptr(), plan.ws_bytes, st), "rsa_rectified_attention_pooled_scatter")
        self._barrier()
        self._keep = keep
        return self.out

    def close(self):
        torch.cuda.synchronize()
        dist.barrier(group=self.group)
        for p in self._opened:
            self._lib.rsa_peer_close(p)
        for p in self._own:
            self._lib.rsa_peer_free(p)
        self._opened, self._own = [], []
