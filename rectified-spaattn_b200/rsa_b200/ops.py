"""Host-side plumbing over the C ABI: PyTorch supplies device memory and the current CUDA stream, nothing else.

Every function here fails loudly (RsaError / RuntimeError) when the native library is missing or a tensor is
not on a CUDA device -- there is no eager-PyTorch fallback for the hot path."""
from __future__ import annotations

import ctypes as C
import math
import os

import torch

from . import geometry as G
from . import native as N

BLOCK = 128


# --------------------------------------------------------------------------------------------- host geometry
def gilbert_mapping(t, h, w, axis_order=("w", "h", "t")):
    """(linear_to_hilbert, hilbert_to_linear) as CPU int64 tensors (utils/jenga_gilbert.py:458-504)."""
    n = t * h * w
    l2h = torch.empty(n, dtype=torch.int64)
    h2l = torch.empty(n, dtype=torch.int64)
    ao = None if axis_order is None else "".join(axis_order).encode()
    N.check(N.lib().rsa_gilbert_map(t, h, w, ao, l2h.data_ptr(), h2l.data_ptr()), "rsa_gilbert_map")
    return l2h, h2l


def gilbert_block_neighbors(t, h, w, block_size=128, axis_order=("w", "h", "t")):
    """bool [NB, NB] CPU tensor (utils/jenga_gilbert.py:613-693)."""
    nb = (t * h * w + block_size - 1) // block_size
    out = torch.empty(nb, nb, dtype=torch.uint8)
    ao = None if axis_order is None else "".join(axis_order).encode()
    N.check(N.lib().rsa_gilbert_block_neighbors(t, h, w, block_size, ao, out.data_ptr()),
            "rsa_gilbert_block_neighbors")
    return out.bool()


# --------------------------------------------------------------------------------------------------- permute
def _need_cuda(x, name):
    if not (isinstance(x, torch.Tensor) and x.is_cuda):
        raise RuntimeError(f"{name} must be a CUDA tensor: this path has no CPU implementation")


def _stream(dev):
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def permute_rows(x, index, out=None):
    """out[b, i, :] = x[b, index[i], :]; x is [B, N, ...] (rows contiguous) or [N, ...]; index int64 on device.
    Replaces hidden_states[:, self.hilbert_order] (scripts/main_hunyuan.py:88-89, :183)."""
    _need_cuda(x, "x")
    squeeze = False
    if x.dim() == 2:
        x = x.unsqueeze(0)
        squeeze = True
    if x.dim() < 3:
        raise ValueError("permute_rows expects [B, N, C] or [N, C]")
    if index.dtype != torch.int64 or not index.is_cuda:
        index = index.to(device=x.device, dtype=torch.int64)
    index = index.contiguous()
    b, n = x.shape[0], x.shape[1]
    row_shape = x.shape[2:]
    row_elems = math.prod(row_shape)
    if x[0].is_contiguous() is False:
        x = x.contiguous()
    row_bytes = row_elems * x.element_size()
    n_out = index.numel()
    if out is None:
        out = torch.empty((b, n_out) + tuple(row_shape), dtype=x.dtype, device=x.device)
    sb = x.stride(0) * x.element_size() if b > 1 else n * row_bytes
    db = out.stride(0) * out.element_size() if b > 1 else n_out * row_bytes
    with torch.cuda.device(x.device):
        N.check(N.lib().rsa_permute_rows(x.data_ptr(), out.data_ptr(), index.data_ptr(), b, n_out, n, row_bytes, sb,
                                         db, _stream(x.device)), "rsa_permute_rows")
    return out[0] if squeeze else out


# ------------------------------------------------------------------------------------------------- attention
_nbr_cache = {}
_ws_cache = {}


def _device_neighbors(nbr, device):
    """uint8 [rows, cols] device copy of block_neighbor_list, cached (the reference re-uploads it every call,
    rectified_wan21_attn.py:261-262)."""
    if nbr is None:
        return None
    key = (nbr.data_ptr(), tuple(nbr.shape), nbr.device.type, str(device), nbr._version)
    hit = _nbr_cache.get(key)
    if hit is not None and hit[0] is nbr:
        return hit[1]
    dev = nbr.to(device=device, dtype=torch.bool).contiguous().view(torch.uint8)
    if len(_nbr_cache) > 16:
        _nbr_cache.clear()
    _nbr_cache[key] = (nbr, dev)
    return dev


def _workspace(device, nbytes):
    """Scratch shared by the short-lived Plans of one (device, CUDA stream): calls enqueued on one stream run one after
    the other and may re-use it; calls on different streams of a device (cond / uncond on parallel streams, threads) each
    get their own, so kernels of one call never overwrite scores, lists, R or C of another.  A buffer that is outgrown is
    kept alive until its stream has drained (record_stream) instead of being freed under kernels still using it."""
    stream = torch.cuda.current_stream(device)
    key = (str(device), stream.cuda_stream)
    ws = _ws_cache.get(key)
    if ws is None or ws.numel() < nbytes:
        if ws is not None:
            ws.record_stream(stream)
        ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=device)
        _ws_cache[key] = ws
    return ws


def _strides3(t):
    # [B, H, S, D] view -> (batch, head, token) element strides; D must be contiguous
    if t.stride(3) != 1:
        raise RuntimeError("head_dim must be the contiguous dimension")
    return (t.stride(0), t.stride(1), t.stride(2))


_rope_cache = {}
COMPACT_ROPE = os.environ.get("RSA_COMPACT_ROPE", "1") != "0"     # tests switch this off to compare the two table layouts


def _compact_rope(cos_in, sin_in, cos, sin):
    """diffusers builds its real rotary tables with repeat_interleave(2): both elements of a pair see the same cos and
    the same sin.  When that holds (checked ONCE per table pair -- one host sync -- and remembered; the tables are
    constants of a generation) the kernel is given one [rows, head_dim / 2] table of (cos_i, sin_i) pairs instead of
    two [rows, head_dim] tables.  Returns None for tables of any other form."""
    if not COMPACT_ROPE:
        return None
    # Keyed by storage, offset and version, and the entry keeps the caller's tensors (hence their storage) alive, so
    # a pointer can never come back as a different table; per-call slices of one table hit the same entry.
    key = (cos_in.untyped_storage().data_ptr(), cos_in.storage_offset(), sin_in.untyped_storage().data_ptr(),
           sin_in.storage_offset(), tuple(cos_in.shape), tuple(cos_in.stride()), cos_in._version, sin_in._version,
           str(cos.device))
    hit = _rope_cache.get(key)
    if hit is not None:
        return hit[2]
    packed = None
    if bool((cos[:, 0::2] == cos[:, 1::2]).all() & (sin[:, 0::2] == sin[:, 1::2]).all()):
        packed = torch.stack([cos[:, 0::2], sin[:, 0::2]], dim=-1).reshape(cos.shape[0], cos.shape[1]).contiguous()
    if len(_rope_cache) > 8:
        _rope_cache.clear()
    _rope_cache[key] = (cos_in, sin_in, packed)
    return packed


class Plan:
    """One call's descriptor + workspace; build once per (shape, geometry) and reuse across layers/steps."""

    def __init__(self, q, k, v, geo: G.BlockGeometry, top_k, p_remain, nbr=None, debug_dump_probs=False, out=None,
                 private_workspace=False, mask_cache=None):
        for t, n in ((q, "query"), (k, "key"), (v, "value")):
            _need_cuda(t, n)
            if t.dtype not in (torch.bfloat16, torch.float16) or t.dtype != q.dtype:
                raise RuntimeError(f"{n} must be bfloat16 or float16 like the query (got {t.dtype})")
        b, h, s, d = q.shape
        if k.shape != q.shape or v.shape != q.shape:
            raise RuntimeError("query/key/value shapes differ")
        if d not in (64, 128):
            # same precondition family as the reference's `assert Lk in {16, 32, 64, 128}` (wan21 :121); 128 is what
            # every BASELINE model has, 64 is CogVideoX (the kernels read the missing 64 columns as zeros)
            raise AssertionError("head_dim must be 128 or 64")
        if s != geo.seq:
            raise ValueError("geometry was built for a different sequence length")
        self.device = q.device
        self.shape = (b, h, s, d)
        self.out = out if out is not None else torch.empty((b, s, h, d), dtype=q.dtype, device=q.device)
        if self.out.dtype != q.dtype:
            raise RuntimeError("out must have the dtype of query/key/value")
        o4 = self.out.view(b, s, h, d).permute(0, 2, 1, 3)
        self.nbr_dev = _device_neighbors(nbr, q.device)
        desc = _fill_desc(N.AttnDesc(), (b, h, s, d), [_strides3(t) for t in (q, k, v, o4)], geo, top_k, p_remain,
                          self.nbr_dev, debug_dump_probs)
        desc.dtype = N.DTYPE_F16 if q.dtype == torch.float16 else N.DTYPE_BF16
        self.desc = desc
        L = N.lib()
        self.ws_bytes = L.rsa_attn_workspace_bytes(C.byref(desc))
        if self.ws_bytes == 0:
            raise N.RsaError("invalid attention descriptor: " + L.rsa_last_error_string().decode())
        # one workspace per device is shared by short-lived plans (a call's stages run back to back on one stream);
        # a plan that is kept across other calls (FusedUlysses) owns its own
        self.mask_mode = N.MASK_BUILD
        self.mask_cache = mask_cache
        if mask_cache is not None:    # the cache owns the workspace (it survives this plan) and says what to re-use
            # the neighbour matrix is a constant of the latent grid: identified by the caller's storage, not its bytes
            key = (self.shape, geo, int(top_k), float(p_remain), str(q.dtype),
                   None if nbr is None else (nbr.data_ptr(), tuple(nbr.shape), nbr._version))
            self.mask_mode, self.ws = mask_cache.next_mode(key, q.device, self.ws_bytes)
        else:
            self.ws = (torch.empty(self.ws_bytes, dtype=torch.uint8, device=q.device) if private_workspace
                       else _workspace(q.device, self.ws_bytes))
        self.q, self.k, self.v = q, k, v

    # --- stages (each enqueues on the current stream; no host sync)
    def _call(self, fn, *args):
        L = N.lib()
        with torch.cuda.device(self.device):
            N.check(getattr(L, fn)(C.byref(self.desc), *args, self.ws.data_ptr(), self.ws_bytes,
                                   _stream(self.device)), fn)

    def pool_stats(self):
        self._call("rsa_pool_stats", self.q.data_ptr(), self.k.data_ptr(), self.v.data_ptr())

    def block_scores(self):
        self._call("rsa_block_scores")

    def block_select(self):
        self._call("rsa_block_select")

    def rect_c(self):
        self._call("rsa_rect_c")

    def sparse_attention(self):
        self._call("rsa_sparse_attention", self.q.data_ptr(), self.k.data_ptr(), self.v.data_ptr(),
                   self.out.data_ptr())
        return self.out

    def run(self, mask_mode=None):
        """The whole call.  mask_mode (enum rsa_mask_mode; default: what the plan's MaskCache asked for, else
        MASK_BUILD): MASK_KEEP_LISTS / MASK_KEEP_ALL re-use the selection an earlier MASK_BUILD run left in this
        plan's workspace (which must then be private or owned by a MaskCache)."""
        mask_mode = self.mask_mode if mask_mode is None else mask_mode
        if mask_mode == N.MASK_BUILD:
            self._call("rsa_rectified_attention", self.q.data_ptr(), self.k.data_ptr(), self.v.data_ptr(),
                       self.out.data_ptr())
        else:
            self._reuse(mask_mode, 0)
        if self.mask_cache is not None:
            self.mask_cache.ran(mask_mode)
        return self.out

    def run_pooled(self, mask_mode=None):
        """Kernels 3a-4 on the pooled statistics qkv_prep(..., pool=True) left in this plan's workspace."""
        mask_mode = self.mask_mode if mask_mode is None else mask_mode
        if mask_mode == N.MASK_BUILD:
            self._call("rsa_rectified_attention_pooled", self.q.data_ptr(), self.k.data_ptr(), self.v.data_ptr(),
                       self.out.data_ptr())
        else:
            self._reuse(mask_mode, 1)
        if self.mask_cache is not None:
            self.mask_cache.ran(mask_mode)
        return self.out

    def run_dense(self, q_valid, kv_len):
        """Dense attention over this plan's q, k, v into its [B, S, H, D] output (rsa_dense_attention): query rows
        >= q_valid are zeros, keys >= kv_len are not attended.  No block selection, no workspace."""
        with torch.cuda.device(self.device):
            N.check(N.lib().rsa_dense_attention(C.byref(self.desc), self.q.data_ptr(), self.k.data_ptr(),
                                                self.v.data_ptr(), self.out.data_ptr(), self.shape[2], int(q_valid),
                                                int(kv_len), _stream(self.device)), "rsa_dense_attention")
        return self.out

    def _reuse(self, mask_mode, pooled):
        L = N.lib()
        with torch.cuda.device(self.device):
            N.check(L.rsa_rectified_attention_reuse(C.byref(self.desc), self.q.data_ptr(), self.k.data_ptr(),
                                                    self.v.data_ptr(), self.out.data_ptr(), self.ws.data_ptr(),
                                                    self.ws_bytes, int(mask_mode), int(pooled), _stream(self.device)),
                    "rsa_rectified_attention_reuse")

    def qkv_prep(self, q_src, k_src, v_src, dst_row=0, q_weight=None, k_weight=None, eps=1e-6, rope=None,
                 rope_rows=None, pool=True, q_bias=None, k_bias=None, allow_fp16=False):
        """Kernel 0: fills rows [dst_row, dst_row + rows) of this plan's q, k, v from projection outputs
        [B, rows, H*head_dim] (head split, per-head RMSNorm or LayerNorm, rotary embedding on the first `rope_rows`
        tokens, re-layout) and, with pool=True, the pooled statistics of those blocks.  head_dim 128 takes every norm;
        head_dim 64 (CogVideoX) takes LayerNorm only (q_weight, k_weight, q_bias, k_bias).
        The sources have the plan's dtype and the norm parameters are converted to it: kernel 0 rounds where diffusers
        rounds, in bf16 or fp16.  An fp16 plan takes kernel 0 only with allow_fp16=True (the switch
        ProcessorBase.fuse_prep_fp16 sets), so that an fp16 caller keeps the op-by-op sequence unless it opts in."""
        b, h, s, d = self.shape
        dt = self.q.dtype
        if dt == torch.float16 and not allow_fp16:
            raise RuntimeError("kernel 0 in float16 is opt-in: pass allow_fp16=True")
        if dt not in (torch.bfloat16, torch.float16) or d not in (128, 64):
            raise RuntimeError("kernel 0 follows diffusers' rounding points and is built for bfloat16 or float16 with "
                               "head_dim 128 or 64")
        if d == 64 and (q_weight is None or q_bias is None):
            raise RuntimeError("kernel 0 at head_dim 64 is built for CogVideoX's LayerNorm: q_weight, k_weight, "
                               "q_bias and k_bias are needed")
        for t, n in ((q_src, "q_src"), (k_src, "k_src"), (v_src, "v_src")):
            _need_cuda(t, n)
            if t.dtype != dt:
                raise RuntimeError(f"{n} is {t.dtype} but the plan is {dt}: kernel 0 reads its sources in the plan's dtype")
            if t.dim() != 3 or t.shape[0] != b or t.shape[2] != h * d or t.stride(2) != 1:
                raise RuntimeError(f"{n} must be a [B, rows, H*{d}] tensor with contiguous channels")
        rows = q_src.shape[1]
        if k_src.shape[1] != rows or v_src.shape[1] != rows:
            raise RuntimeError("q/k/v sources differ in length")
        p = N.PrepDesc()
        p.rows, p.dst_row = rows, int(dst_row)
        for i, t in enumerate((q_src, k_src, v_src)):
            p.src_stride[i][0], p.src_stride[i][1] = t.stride(0), t.stride(1)
        keep = []
        if q_weight is not None or k_weight is not None:
            if q_weight is None or k_weight is None:
                raise RuntimeError("both norm weights are needed")
            ws_ = [w.detach().to(device=self.device, dtype=dt).contiguous() for w in (q_weight, k_weight)]
            if q_bias is not None or k_bias is not None:    # LayerNorm over head_dim (CogVideoX)
                bs_ = [x.detach().to(device=self.device, dtype=dt).contiguous() for x in (q_bias, k_bias)]
                if any(w.numel() != d for w in ws_ + bs_):
                    raise RuntimeError("LayerNorm weights and biases must have head_dim elements")
                keep += bs_
                p.norm, p.q_bias, p.k_bias = 3, bs_[0].data_ptr(), bs_[1].data_ptr()
            elif all(w.numel() == d for w in ws_):
                p.norm = 1                                  # RMSNorm over head_dim
            elif all(w.numel() == h * d for w in ws_):
                p.norm = 2                                  # RMSNorm across heads (Wan)
                scratch = torch.empty(2 * b * rows, dtype=torch.float32, device=self.device)
                keep.append(scratch)
                p.row_scratch = scratch.data_ptr()
            else:
                raise RuntimeError("RMSNorm weights must have head_dim or heads*head_dim elements")
            keep += ws_
            p.eps = float(eps)
            p.q_weight, p.k_weight = ws_[0].data_ptr(), ws_[1].data_ptr()
        if rope is not None:
            cos, sin = (t.detach().to(device=self.device, dtype=torch.float32).contiguous() for t in rope)
            n_rope = cos.shape[0] if rope_rows is None else int(rope_rows)
            if cos.shape != sin.shape or cos.dim() != 2 or cos.shape[1] != d or cos.shape[0] < n_rope:
                raise RuntimeError("rotary tables must be (cos, sin) of shape [rope_rows, head_dim]")
            packed = _compact_rope(rope[0], rope[1], cos, sin)
            if packed is not None:      # one [rows, 64] table of (cos_i, sin_i) pairs: half the bytes per row
                keep.append(packed)
                p.rope_rows, p.rope_compact, p.cos = n_rope, 1, packed.data_ptr()
            else:
                keep += [cos, sin]
                p.rope_rows, p.cos, p.sin = n_rope, cos.data_ptr(), sin.data_ptr()
        L = N.lib()
        with torch.cuda.device(self.device):
            N.check(L.rsa_qkv_prep(C.byref(p), C.byref(self.desc), q_src.data_ptr(), k_src.data_ptr(),
                                   v_src.data_ptr(), self.q.data_ptr(), self.k.data_ptr(), self.v.data_ptr(),
                                   1 if pool else 0, self.ws.data_ptr(), self.ws_bytes, _stream(self.device)),
                    "rsa_qkv_prep")
        self._keep = keep   # the kernel reads them asynchronously

    # --- workspace views for the parity tests
    def view(self):
        v = N.WsView()
        N.check(N.lib().rsa_attn_workspace_view(C.byref(self.desc), self.ws.data_ptr(), self.ws_bytes, C.byref(v)),
                "rsa_attn_workspace_view")
        b, h, _, _ = self.shape
        bh = b * h
        g = self.desc
        base = self.ws.data_ptr()

        def t(ptr, shape, dtype):
            if not ptr:
                return None
            n = math.prod(shape) * torch.empty((), dtype=dtype).element_size()
            off = ptr - base
            return self.ws[off: off + n].view(dtype).view(shape)

        nq, nb = g.nq_blocks, g.n_blocks
        return dict(
            q_pool=t(v.q_pool, (bh, nq, 128), torch.float32), q_mad=t(v.q_mad, (bh, nq, 128), torch.float32),
            k_cat=t(v.k_cat, (bh, v.nkc, 128), torch.float32), k_mad=t(v.k_mad, (bh, nq, 128), torch.float32),
            v_pool=t(v.v_pool, (bh, nb, 128), torch.float32),
            scores=t(v.scores, (bh, nq, v.score_ld), torch.float32)[:, :, : v.nkc],
            nogapr=t(v.nogapr, (bh, nq, v.nogapr_ld), torch.uint8)[:, :, :nq],
            probs=None if not v.probs else t(v.probs, (bh, nq, v.ent_ld), torch.float32)[:, :, : v.n_entries],
            w_skip=t(v.w_skip, (bh, nq, v.ent_ld), torch.float32)[:, :, : v.n_entries],
            mask_bits=t(v.mask_bits, (bh, v.nqt, v.mask_words), torch.int32),
            kept_idx=t(v.kept_idx, (bh, v.nqt, nb), torch.int16),
            kept_cnt=t(v.kept_cnt, (bh, v.nqt), torch.int32),
            n_needed=t(v.n_needed, (bh, max(nq, 1)), torch.int32),
            R=t(v.R, (bh, v.nqt), torch.float32), C=t(v.C, (bh, v.nqt, 128), torch.float32),
            sched_idx=t(v.sched_idx, (bh, v.nqt, nb), torch.int16),
            pair_shared=t(v.pair_shared, (bh, (v.nqt + 1) // 2), torch.int32),
            quad_shared=t(v.quad_shared, (bh, (v.nqt + 1) // 2), torch.int32))

    def dense_mask(self):
        """bool [BH, NQT, NB] reconstructed from the kept-block bitmask (the reference's one_hot layout)."""
        vw = self.view()
        bits = vw["mask_bits"]
        nb = self.desc.n_blocks
        j = torch.arange(nb, device=bits.device)
        words = bits[:, :, (j >> 5)]
        return ((words >> (j & 31)) & 1).bool()


def _fill_desc(desc, shape, strides, geo, top_k, p_remain, nbr_dev, debug_dump_probs=False):
    b, h, s, d = shape
    desc.batch, desc.heads, desc.seq, desc.head_dim = b, h, s, d
    for name, st in zip(("q_stride", "k_stride", "v_stride", "o_stride"), strides):
        arr = getattr(desc, name)
        for i in range(3):
            arr[i] = st[i]
    desc.family = geo.family
    desc.n_blocks, desc.nq_blocks, desc.text_keys = geo.n_blocks, geo.nq_blocks, geo.text_keys
    desc.kv_len, desc.kv_zero_from = geo.kv_len, geo.kv_zero_from
    desc.text_end_block, desc.text_q_valid = geo.text_end_block, geo.text_q_valid
    desc.top_k, desc.p_remain = int(top_k), float(p_remain)
    desc.first_frame_blocks = geo.first_frame_blocks
    desc.vis_len = geo.vis_len
    if nbr_dev is not None:
        desc.nbr_rows, desc.nbr_cols = nbr_dev.shape
        desc.nbr = nbr_dev.data_ptr()
    desc.debug_dump_probs = 1 if debug_dump_probs else 0
    return desc


_host_scratch = {}
HOST_HEADS_PER_CHUNK = None   # None: 2 heads per chunk from 8 heads up, else 1 (a head-parallel rank may hold only 3)


def rectified_attention_host(q, k, v, geo, top_k, p_remain, nbr=None, shape_xfuse=False, heads_per_chunk=None,
                             out=None, device=None):
    """The same call for PAGE-LOCKED HOST tensors (rsa_rectified_attention_host): chunks of heads stream through
    H2D -> kernels -> D2H on three CUDA streams of `device` (default: the current device).  Returns a pinned host
    tensor in the reference's layout; it is complete once the current stream of `device` is synchronised."""
    if not torch.cuda.is_available():
        raise RuntimeError("no CUDA device: this path has no CPU implementation")
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    for t, n in ((q, "query"), (k, "key"), (v, "value")):
        if t.is_cuda or t.dtype not in (torch.bfloat16, torch.float16) or t.dtype != q.dtype:
            raise RuntimeError(f"{n} must be a bfloat16 (or float16) host tensor")
        if not t.is_pinned():
            raise RuntimeError(f"{n} must be page-locked (tensor.pin_memory()): the copies run asynchronously")
    b, h, s, d = q.shape
    if k.shape != q.shape or v.shape != q.shape:
        raise RuntimeError("query/key/value shapes differ")
    if d not in (64, 128):
        raise AssertionError("head_dim must be 128 or 64")
    if s != geo.seq:
        raise ValueError("geometry was built for a different sequence length")
    if out is None:
        out = torch.empty((b, s, h, d), dtype=q.dtype, pin_memory=True)
    elif out.is_cuda or not out.is_pinned() or out.numel() != b * s * h * d or out.dtype != q.dtype:
        raise RuntimeError("out must be a pinned host tensor of B*S*H*D elements with the inputs' dtype")
    o4 = out.view(b, s, h, d).permute(0, 2, 1, 3)
    nbr_dev = _device_neighbors(nbr, device)
    desc = _fill_desc(N.AttnDesc(), (b, h, s, d), [_strides3(t) for t in (q, k, v, o4)], geo, top_k, p_remain,
                      nbr_dev)
    desc.dtype = N.DTYPE_F16 if q.dtype == torch.float16 else N.DTYPE_BF16
    hc = int(heads_per_chunk or HOST_HEADS_PER_CHUNK or (2 if h >= 8 else 1))
    L = N.lib()
    need = L.rsa_host_call_scratch_bytes(C.byref(desc), hc)
    if need == 0:
        raise N.RsaError("invalid attention descriptor: " + L.rsa_last_error_string().decode())
    scratch = _host_scratch.get(str(device))
    if scratch is None or scratch.numel() < need:
        scratch = torch.empty(need, dtype=torch.uint8, device=device)
        _host_scratch[str(device)] = scratch
    with torch.cuda.device(device):
        N.check(L.rsa_rectified_attention_host(C.byref(desc), q.data_ptr(), k.data_ptr(), v.data_ptr(),
                                               out.data_ptr(), hc, scratch.data_ptr(), scratch.numel(),
                                               _stream(device)), "rsa_rectified_attention_host")
    out = out.view(b, s, h, d)
    return out if shape_xfuse else out.view(b, s, h * d)


class MaskCache:
    """Block selection kept across calls (SURVEY 8f rank 4): one per attention layer.  The reference rebuilds its
    mask in every layer of every denoising step (rectified_hunyuan_attn.py:334-346); with a cache the selection is
    rebuilt every `refresh_every`-th call and re-used in between -- `keep="lists"`: P, the GAPR test, R and C are still
    recomputed from the current tensors (RSA_MASK_KEEP_LISTS), `keep="all"`: only kernel 4 runs (RSA_MASK_KEEP_ALL).
    The cache IS the call's workspace (kept lists, pair schedule, R, C), owned here instead of shared per device.
    refresh_every = 1 is the reference's behaviour."""

    def __init__(self, refresh_every=1, keep="lists"):
        if keep not in ("lists", "all"):
            raise ValueError("keep must be 'lists' or 'all'")
        self.refresh_every = max(1, int(refresh_every))
        self.keep = keep
        self.calls = 0
        self.valid = False      # the workspace holds a selection built by an earlier call
        self._ws = None
        self._key = None

    def reset(self):
        """Forget the cached selection (new prompt / new generation)."""
        self.calls = 0
        self._key = None
        self.valid = False

    def next_mode(self, key, device, ws_bytes):
        """(mask_mode, workspace) for the next call whose geometry is `key`.  A query: the schedule only advances when
        a call has actually been enqueued (`ran`), so a plan that is built and then abandoned changes nothing."""
        if self._key != key or self._ws is None or self._ws.device != device or self._ws.numel() < ws_bytes:
            if self._ws is None or self._ws.device != device or self._ws.numel() < ws_bytes:
                self._ws = torch.empty(ws_bytes, dtype=torch.uint8, device=device)
            self._key = key
            self.calls = 0
            self.valid = False
        mode = N.MASK_BUILD
        if self.valid and self.calls % self.refresh_every != 0:
            mode = N.MASK_KEEP_LISTS if self.keep == "lists" else N.MASK_KEEP_ALL
        return mode, self._ws

    def ran(self, mode):
        """A call in `mode` has been enqueued on this cache's workspace."""
        if mode == N.MASK_BUILD:
            self.valid = True
        self.calls += 1


def rectified_attention(q, k, v, geo, top_k, p_remain, nbr=None, shape_xfuse=False, mask_cache=None):
    """[B,H,S,D] bf16 -> [B,S,H*D] (or [B,S,H,D] with shape_xfuse) -- the reference's return layout
    (rectified_wan21_attn.py:353-357).  Host (pinned) tensors take the pipelined host-buffer entry point and come
    back as a pinned host tensor; the arithmetic runs on the GPU either way.  mask_cache: an optional MaskCache."""
    if isinstance(q, torch.Tensor) and not q.is_cuda and torch.cuda.is_available():
        if mask_cache is not None:
            raise RuntimeError("mask re-use needs device-resident tensors (the host-buffer call owns no lasting workspace)")
        return rectified_attention_host(q, k, v, geo, top_k, p_remain, nbr, shape_xfuse)
    out = Plan(q, k, v, geo, top_k, p_remain, nbr, mask_cache=mask_cache).run()
    b, s, h, d = out.shape
    return out if shape_xfuse else out.view(b, s, h * d)


def masked_attention(q, k, v, block_mask, kv_len, sm_scale=None, out=None, fp32_scale=False):
    """Kernel 4 alone on a dense block mask: the surface of _triton_block_sparse_attention_onehot
    (rectified_wan21_attn.py:108-117).  q,k,v [B,H,S,D] bf16 (any batch / head / token strides with D contiguous -- the
    ABI takes strides, nothing is copied), block_mask bool [B,H,NQ,NB] -> [B,H,S,D].  Like that kernel, the query is
    pre-scaled by sm_scale * log2(e) and ROUNDED to the input dtype (:61-62); fp32_scale=True scales the fp32 scores
    instead, which is what flash-attn does (the mirror's dense `fullattn`)."""
    _need_cuda(q, "q")
    if q.dtype not in (torch.bfloat16, torch.float16) or k.dtype != q.dtype or v.dtype != q.dtype:
        raise RuntimeError("q, k, v must all be bfloat16 or all float16")
    if sm_scale is not None and abs(sm_scale - q.shape[-1] ** -0.5) > 1e-7:
        raise ValueError("only sm_scale = head_dim ** -0.5 is supported")
    b, h, s, d = q.shape
    if d not in (64, 128):
        raise AssertionError("head_dim must be 128 or 64")
    skv = k.shape[2]
    nqb, nkb = (s + 127) // 128, (skv + 127) // 128
    if tuple(block_mask.shape[-2:]) != (nqb, nkb):
        raise ValueError("block_mask shape does not match the sequence lengths")
    m = block_mask.reshape(b * h, nqb, nkb).to(device=q.device, dtype=torch.bool).contiguous().view(torch.uint8)
    if out is None:
        out = torch.zeros_like(q, memory_format=torch.contiguous_format)
    elif out.shape != q.shape or out.dtype != q.dtype or out.stride(3) != 1:
        raise RuntimeError("out must have the shape and dtype of q with a contiguous head_dim")
    L = N.lib()

    def flat(t):
        """[B,H,S,D] view -> (tensor, (bh stride, token stride)) for a [B*H, S, D] addressing; copies only when batch and
        head do not collapse into one stride and the strides are not multiples of 8."""
        if t.stride(3) != 1 or any(x % 8 for x in t.stride()[:3]):
            t = t.contiguous()
        if t.shape[0] == 1 or t.stride(0) == t.shape[1] * t.stride(1):
            return t, (t.stride(1), t.stride(2))
        t = t.contiguous()
        return t, (t.stride(1), t.stride(2))

    (q3, qs), (k3, ks), (v3, vs) = flat(q), flat(k), flat(v)
    o3, os_ = flat(out)
    if o3.data_ptr() != out.data_ptr():
        raise RuntimeError("out must be addressable as [B*H, S, D] with strides that are multiples of 8")
    nbytes = L.rsa_masked_attention_workspace_bytes(b * h, nqb, nkb)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=q.device)
    mk = lambda st: (C.c_int64 * 2)(*st)
    with torch.cuda.device(q.device):
        N.check(L.rsa_masked_attention(q3.data_ptr(), k3.data_ptr(), v3.data_ptr(), o3.data_ptr(), b * h, s, skv,
                                       int(kv_len), mk(qs), mk(ks), mk(vs), mk(os_), m.data_ptr(), nqb, nkb,
                                       ws.data_ptr(), nbytes, _stream(q.device),
                                       (N.DTYPE_F16 if q.dtype == torch.float16 else N.DTYPE_BF16)
                                       | (N.ATTN_FP32_SCALE if fp32_scale else 0), d),
                "rsa_masked_attention")
    return out


def dense_attention(q, k, v, q_valid, kv_len, out=None):
    """Dense attention on kernel 4 without lists (rsa_dense_attention): q [B,H,S,D], k / v [B,H,S_kv,D] views with any
    strides (D contiguous), bf16 or fp16, D = 128 or 64.  Query rows >= q_valid are zeros, keys >= kv_len are not
    attended; flash-attn's arithmetic.  `out`: a [B,H,S,D] tensor or view, or a [B,S,H,D] tensor written through its
    permuted view (the processors' layout); returned as given (a new contiguous [B,H,S,D] tensor when None)."""
    _need_cuda(q, "q")
    if q.dtype not in (torch.bfloat16, torch.float16) or k.dtype != q.dtype or v.dtype != q.dtype:
        raise RuntimeError("q, k, v must all be bfloat16 or all float16")
    b, h, s, d = q.shape
    if d not in (64, 128):
        raise AssertionError("head_dim must be 128 or 64")
    skv = k.shape[2]
    if k.shape != (b, h, skv, d) or v.shape != k.shape:
        raise RuntimeError("key/value must be [B, H, S_kv, D] with the query's B, H and D")

    def ready(t):       # the kernel reads through TMA: strides multiples of 8 elements, 16-byte aligned base
        if t.stride(3) != 1 or any(x % 8 for x in t.stride()[:3]) or t.data_ptr() % 16:
            t = t.contiguous()
        return t

    q, k, v = ready(q), ready(k), ready(v)
    if out is None:
        out = torch.empty((b, h, s, d), dtype=q.dtype, device=q.device)
    if out.dtype != q.dtype or out.device != q.device:
        raise RuntimeError("out must have the dtype and device of q")
    if tuple(out.shape) == (b, h, s, d):
        o4 = out
    elif tuple(out.shape) == (b, s, h, d):
        o4 = out.permute(0, 2, 1, 3)
    else:
        raise RuntimeError("out must be [B, H, S, D] or [B, S, H, D]")
    if o4.stride(3) != 1:
        raise RuntimeError("out must have a contiguous head_dim")
    desc = N.AttnDesc()
    desc.batch, desc.heads, desc.seq, desc.head_dim = b, h, s, d
    for name, t in zip(("q_stride", "k_stride", "v_stride", "o_stride"), (q, k, v, o4)):
        arr = getattr(desc, name)
        for i in range(3):
            arr[i] = t.stride(i)
    desc.dtype = N.DTYPE_F16 if q.dtype == torch.float16 else N.DTYPE_BF16
    with torch.cuda.device(q.device):
        N.check(N.lib().rsa_dense_attention(C.byref(desc), q.data_ptr(), k.data_ptr(), v.data_ptr(), o4.data_ptr(), skv,
                                            int(q_valid), int(kv_len), _stream(q.device)), "rsa_dense_attention")
    return out


def set_attention_flags(flags):
    """Bring-up / cross-check switches of kernel 4 (rsa_debug_set_attention_flags); bit 2 = head_dim 64 through the
    128-column instantiation."""
    N.lib().rsa_debug_set_attention_flags(int(flags))
