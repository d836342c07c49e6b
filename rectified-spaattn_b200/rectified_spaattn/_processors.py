"""Shared pieces of the eight `Rectified*SpaAttnProcessor2_0` classes (not part of the reference's surface).

The processors follow the diffusers `AttnProcessor` protocol exactly like the reference's (same constructor arguments,
attributes, `__call__` signature, return values, warm-up gates and step counters -- SURVEY.md 3.4); what surrounds the
hot path (QKV / output projections of the caller's `attn` module, QK norms, RoPE) stays plain PyTorch on the caller's
modules, and the attention itself goes through the per-family `rectified_block_sparse_attention` /
`fullattn(mode="flash")`, i.e. the sm_100a kernels.  diffusers is not imported: the three RoPE conventions the
reference takes from it (or defines inline) are restated here.
"""
from typing import Optional

import torch
import torch.nn.functional as F


def heads_first(x, heads):
    """[B, S, H*D] -> [B, H, S, D] (reference: `unflatten(2, (heads, -1)).transpose(1, 2)`)."""
    return x.unflatten(2, (heads, -1)).transpose(1, 2)


def rope_real(x, freqs):
    """diffusers.models.embeddings.apply_rotary_emb with use_real=True, use_real_unbind_dim=-1 (what
    rectified_hunyuan_attn.py:460-478, rectified_flux_attn.py:483-486 and rectified_cogvideo_attn.py:460-469 call):
    x [B, H, S, D], freqs = (cos, sin) each [S, D]; pairs are (x[2i], x[2i+1])."""
    cos, sin = freqs
    cos, sin = cos[None, None].to(x.device), sin[None, None].to(x.device)
    xr, xi = x.reshape(*x.shape[:-1], -1, 2).unbind(-1)
    rot = torch.stack([-xi, xr], dim=-1).flatten(3)
    return (x.float() * cos + rot.float() * sin).to(x.dtype)


def rope_complex(x, freqs):
    """The inline helper of rectified_wan21_attn.py:433-438: complex multiply in float64, x [B, H, S, D]."""
    dtype = torch.float32 if x.device.type == "mps" else torch.float64
    xc = torch.view_as_complex(x.to(dtype).unflatten(3, (-1, 2)))
    return torch.view_as_real(xc * freqs).flatten(3, 4).type_as(x)


def rope_cos_sin(x, freqs_cos, freqs_sin):
    """The inline helper of rectified_wan22_attn.py:52-64 (x [B, S, H, D], interleaved cos/sin tables)."""
    x1, x2 = x.unflatten(-1, (-1, 2)).unbind(-1)
    cos, sin = freqs_cos[..., 0::2], freqs_sin[..., 1::2]
    out = torch.empty_like(x)
    out[..., 0::2] = x1 * cos - x2 * sin
    out[..., 1::2] = x1 * sin + x2 * cos
    return out.type_as(x)


def kv_valid(attention_mask, s_k):
    """`attention_mask.sum().item() if attention_mask else S_k` of the reference (one host sync when a mask is given)."""
    if attention_mask is None:
        return int(s_k)
    return int(attention_mask.sum().item())


def image_cross_attention(attn, query, encoder_hidden_states_img):
    """Wan I2V: dense attention of all queries over the 257 CLIP image tokens (rectified_wan21_attn.py:445-458).
    Dense, tiny KV: not part of the sparse path, left to PyTorch SDPA.  query is [B, H, S, D]."""
    key_img = attn.norm_added_k(attn.add_k_proj(encoder_hidden_states_img))
    value_img = attn.add_v_proj(encoder_hidden_states_img)
    key_img, value_img = heads_first(key_img, attn.heads), heads_first(value_img, attn.heads)
    out = F.scaled_dot_product_attention(query, key_img, value_img, attn_mask=None, dropout_p=0.0, is_causal=False)
    return out.transpose(1, 2).flatten(2, 3).type_as(query)


def split_wan_context(attn, encoder_hidden_states):
    """(image part, text part) of the Wan cross-attention context; 512 = text encoder context length, hard-coded
    in the reference (rectified_wan21_attn.py:411-416)."""
    if getattr(attn, "add_k_proj", None) is None or encoder_hidden_states is None:
        return None, encoder_hidden_states
    n_img = encoder_hidden_states.shape[1] - 512
    return encoder_hidden_states[:, :n_img], encoder_hidden_states[:, n_img:]


def dense(fullattn, query, key, value, mode, attention_mask, s_k):
    """The reference's dense branch: fullattn(...) then `.transpose(1, 2).reshape(B, S_q, -1)`."""
    b, _, s_q, _ = query.shape
    cu_q = [0, s_q, s_q]
    cu_kv = [0, s_k, key.shape[2]]
    out = fullattn(query, key, value, mode=mode, drop_rate=0.0, attn_mask=attention_mask, causal=False,
                   cu_seqlens_q=cu_q, cu_seqlens_kv=cu_kv, max_seqlen_q=s_q, max_seqlen_kv=key.shape[2],
                   batch_size=b)
    return out.transpose(1, 2).reshape(b, s_q, -1)


def rms_params(mod, dtype=torch.bfloat16):
    """(weight, eps) if `mod` is an RMSNorm over head_dim = 128 with a weight of `dtype` (the activations' dtype: a
    weight of another dtype rounds elsewhere in diffusers) and no bias -- the form kernel 0 fuses (diffusers RMSNorm of
    HunyuanVideo / Flux `norm_q`, `norm_k`, `norm_added_q`, `norm_added_k`); else None."""
    w, eps = getattr(mod, "weight", None), getattr(mod, "eps", None)
    if mod is None or w is None or eps is None or getattr(mod, "bias", None) is not None:
        return None
    if "RMSNorm" not in type(mod).__name__ or w.dtype != dtype or w.numel() != 128 or not w.is_cuda:
        return None
    return w, float(eps)


def wan_rms_params(mod, heads, dtype=torch.bfloat16):
    """(weight, eps) if `mod` is an RMSNorm over all heads*128 channels with a weight of `dtype` (Wan norm_q / norm_k)."""
    w, eps = getattr(mod, "weight", None), getattr(mod, "eps", None)
    if mod is None or w is None or eps is None or getattr(mod, "bias", None) is not None:
        return None
    if "RMSNorm" not in type(mod).__name__ or w.dtype != dtype or w.numel() != heads * 128 or not w.is_cuda:
        return None
    return w, float(eps)


_wan_rope_cache = {}


def wan_rope_tables(emb, n):
    """fp32 (cos, sin) [n, 128] tables from either Wan rotary form: Wan2.1's complex `freqs` [1, 1, S, 64]
    (rectified_wan21_attn.py:433-438) or Wan2.2's (freqs_cos, freqs_sin) [1, S, 1, 128] (rectified_wan22_attn.py:52-64,
    which reads cos[..., 0::2] and sin[..., 1::2]).  Cached per tensor: the tables are constants of a generation."""
    src = tuple(emb) if isinstance(emb, (tuple, list)) else (emb,)
    key = tuple((t.data_ptr(), tuple(t.shape), t._version) for t in src) + (n,)
    hit = _wan_rope_cache.get(key)
    # the entry keeps the source tensors alive and is honoured only for the SAME tensor objects: diffusers rebuilds
    # rotary_emb on every transformer forward and the caching allocator hands the same address back, so another latent
    # grid with the same token count would otherwise hit a stale table (ADVICE r1)
    if hit is not None and len(hit[0]) == len(src) and all(a is b for a, b in zip(hit[0], src)):
        return hit[1]
    if isinstance(emb, torch.Tensor) and emb.is_complex() and emb.shape[-1] == 64 and emb.shape[-2] >= n:
        f = emb.reshape(-1, 64)[-emb.shape[-2]:][:n]
        cos, sin = f.real.float().repeat_interleave(2, dim=1), f.imag.float().repeat_interleave(2, dim=1)
    elif isinstance(emb, (tuple, list)) and len(emb) == 2 and all(t.shape[-1] == 128 and t.numel() >= n * 128 for t in emb):
        c, s_ = (t.reshape(-1, 128)[:n].float() for t in emb)
        cos, sin = c[:, 0::2].repeat_interleave(2, dim=1), s_[:, 1::2].repeat_interleave(2, dim=1)
    else:
        return None
    if len(_wan_rope_cache) > 8:
        _wan_rope_cache.clear()
    _wan_rope_cache[key] = (src, (cos.contiguous(), sin.contiguous()))
    return _wan_rope_cache[key][1]


def head_norm_params(mod, head_dim=128, dtype=torch.bfloat16):
    """dict(q_weight-style kwargs) for a per-head norm kernel 0 fuses: RMSNorm(128) (HunyuanVideo / Flux) or
    LayerNorm(head_dim) with bias (CogVideoX: head_dim 128 or 64), parameters of `dtype`; else None.  Returns (weight,
    bias or None, eps)."""
    r = rms_params(mod, dtype) if head_dim == 128 else None     # kernel 0 has no RMSNorm at 64 columns
    if r is not None:
        return r[0], None, r[1]
    w, b, eps = getattr(mod, "weight", None), getattr(mod, "bias", None), getattr(mod, "eps", None)
    if mod is None or w is None or b is None or eps is None or "LayerNorm" not in type(mod).__name__:
        return None
    if (w.dtype != dtype or b.dtype != dtype or w.numel() != head_dim or b.numel() != head_dim
            or not w.is_cuda):
        return None
    return w, b, float(eps)


def rope_tables(emb, n, head_dim=128):
    """(cos, sin) fp32 [>= n, head_dim] tables as diffusers passes them (`image_rotary_emb`), or None if `emb` has
    another form."""
    if not (isinstance(emb, (tuple, list)) and len(emb) == 2):
        return None
    cos, sin = emb
    ok = all(isinstance(t, torch.Tensor) and t.dim() == 2 and t.shape[1] == head_dim and t.shape[0] >= n
             for t in (cos, sin))
    return (cos, sin) if ok else None


def prep_dtype_ok(x, fp16):
    """Kernel 0 runs on bf16 activations, and on fp16 ones when the processor's fuse_prep_fp16 switch is set."""
    return x.dtype == torch.bfloat16 or (fp16 and x.dtype == torch.float16)


def fused_prep_attention(attn, hidden_states, encoder_hidden_states, geo, top_k, p_remain, nbr, image_rotary_emb,
                         rope_text, mask_cache=None, dense=False, fp16=False):
    """The fused form of a joint-text processor's middle section (kernel 0 + kernels 3a-4): projections ->
    rsa_qkv_prep (head split, RMSNorm / LayerNorm, RoPE, re-layout, pooling) -> rsa_rectified_attention_pooled.  Returns
    [B, S, H*D], or None when this layer does not have the shape kernel 0 fuses (the caller then runs the op-by-op path).
    D (head_dim) is read from `to_q`'s output width: 128, or 64 (CogVideoX, LayerNorm only).
    `rope_text`: Flux rotates the text tokens too (their table rows follow the image rows); HunyuanVideo does not.
    `dense`: the call the op-by-op path sends to fullattn(mode="flash") -- kernel 0 without pooling, then dense
    attention over the first `geo.kv_len - geo.gap` memory rows (num_true for HunyuanVideo, S otherwise) as queries
    and keys; top_k, p_remain, nbr and mask_cache are not used.
    `fp16`: fp16 activations take kernel 0 too (ProcessorBase.fuse_prep_fp16); the norm parameters must then be fp16."""
    from rsa_b200 import ops
    heads = attn.heads
    if not hidden_states.is_cuda or not prep_dtype_ok(hidden_states, fp16):
        return None
    dt = hidden_states.dtype
    inner = getattr(attn.to_q, "out_features", None)
    hd = inner // heads if isinstance(inner, int) and inner % heads == 0 else 0
    if hd not in (128, 64):
        return None
    dual = getattr(attn, "add_q_proj", None) is not None and encoder_hidden_states is not None
    def pair(nq, nk):
        a, c = head_norm_params(getattr(attn, nq, None), hd, dt), head_norm_params(getattr(attn, nk, None), hd, dt)
        if a is None or c is None or a[2] != c[2] or (a[1] is None) != (c[1] is None):
            return None
        return dict(q_weight=a[0], k_weight=c[0], q_bias=a[1], k_bias=c[1], eps=a[2])

    lat_norm = pair("norm_q", "norm_k")
    if lat_norm is None:
        return None
    enc_norm = None
    if dual:
        enc_norm = pair("norm_added_q", "norm_added_k")
        if enc_norm is None:
            return None
    b, s = hidden_states.shape[0], geo.seq
    nv = geo.vis_len or geo.nq_blocks * 128
    rope = None
    if image_rotary_emb is not None:
        rope = rope_tables(image_rotary_emb, s if rope_text else nv, hd)
        if rope is None:
            return None
    lat = [f(hidden_states) for f in (attn.to_q, attn.to_k, attn.to_v)]
    if lat[0].shape[2] != heads * hd:
        return None
    enc = None
    if dual:
        enc = [f(encoder_hidden_states) for f in (attn.add_q_proj, attn.add_k_proj, attn.add_v_proj)]
        if lat[0].shape[1] != nv or enc[0].shape[1] != s - nv:
            return None
    elif lat[0].shape[1] != s:
        return None
    # every "this layer does not fit" exit is above: from here on the call is made
    q, k, v = (torch.empty(b, heads, s, hd, dtype=dt, device=hidden_states.device) for _ in range(3))
    plan = ops.Plan(q, k, v, geo, top_k, p_remain, nbr, mask_cache=None if dense else mask_cache)
    cut = lambda r, a, z: None if r is None else (r[0][a:z], r[1][a:z])
    pool = not dense
    lat_norm, enc_norm = (None if n is None else dict(n, allow_fp16=fp16) for n in (lat_norm, enc_norm))
    if dual:
        plan.qkv_prep(*lat, dst_row=0, rope=cut(rope, 0, nv), pool=pool, **lat_norm)
        plan.qkv_prep(*enc, dst_row=nv, rope=cut(rope, nv, s) if rope_text else None, pool=pool, **enc_norm)
    else:
        n_rope = 0 if rope is None else (s if rope_text else nv)
        if geo.gap:     # ragged visual segment: the two segments are separate block ranges
            plan.qkv_prep(*(t[:, :nv] for t in lat), dst_row=0, rope=cut(rope, 0, nv), pool=pool, **lat_norm)
            plan.qkv_prep(*(t[:, nv:] for t in lat), dst_row=nv, rope=cut(rope, nv, s) if rope_text else None,
                          pool=pool, **lat_norm)
        else:
            plan.qkv_prep(*lat, dst_row=0, rope=rope, rope_rows=n_rope, pool=pool, **lat_norm)
    if dense:
        n_valid = geo.kv_len - geo.gap      # memory rows: kv_len counts the gap rows of a ragged visual segment
        return plan.run_dense(n_valid, n_valid).view(b, s, heads * hd)
    return plan.run_pooled().view(b, s, heads * hd)


class ProcessorBase:
    """Constructor arguments and mutable per-layer state shared by every reference processor
    (e.g. rectified_wan21_attn.py:390-401)."""

    steps_per_cycle = 50  # `current_step` wraps to 0 after this many calls
    fuse_prep = True      # joint-text processors: run head split / QK norm / RoPE / pooling as kernel 0 when the layer allows
    # the same for the calls that go to fullattn(mode="flash") (warm-up calls, dense layers, mode "flash"): kernel 0
    # without pooling, then kernel 4's list-free dense form.  Off by default: the op-by-op route stays the reference's.
    fuse_prep_dense = False
    # kernel 0 for fp16 layers too (fp16 models such as CogVideoX-2B): with fuse_prep on their sparse calls, with
    # fuse_prep_dense on their dense calls as well.  The norm parameters must be fp16 like the activations.  Off by
    # default: until it is switched on, an fp16 model runs its pre-attention op by op exactly as before.
    fuse_prep_fp16 = False

    def __init__(self, mode, select_block_num, block_neighbor_list, p_remain_rates, processor_id=0):
        self.mode = mode
        self.select_block_num = select_block_num
        self.block_neighbor_list = block_neighbor_list
        self.p_remain_rates = p_remain_rates
        self.current_step = 0
        self.processor_id = processor_id
        if not hasattr(F, "scaled_dot_product_attention"):
            raise ImportError(f"{type(self).__name__} requires PyTorch 2.0. To use it, please upgrade PyTorch to 2.0.")

    # Extension (SURVEY 8f rank 4), off by default: rebuild the block selection only every `mask_refresh_interval`-th
    # sparse call of this layer and re-use it in between (`mask_keep` = "lists": R and C are still recomputed from the
    # current tensors; "all": only kernel 4 runs).  1 = the reference's behaviour (a new mask per call).  The cache is
    # dropped whenever `current_step` wraps, i.e. at the start of every generation.
    # A pipeline that runs classifier-free guidance as two forwards per denoising step calls the processor
    # `calls_per_step` = 2 times per step (the Wan pipelines: that is why their counter wraps at 100 for 50 steps): every
    # branch then has its own cache, so the interval counts denoising steps and the unconditional pass is never handed a
    # selection built from the conditional pass's Q / K.
    mask_refresh_interval = 1
    mask_keep = "lists"
    calls_per_step = 1
    _caches = None

    def _mask_cache(self):
        if self.mask_refresh_interval <= 1:
            return None
        if self._caches is None or len(self._caches) != self.calls_per_step:
            self._caches = [None] * self.calls_per_step
        branch = self.current_step % self.calls_per_step
        c = self._caches[branch]
        if c is None or c.refresh_every != self.mask_refresh_interval or c.keep != self.mask_keep:
            from rsa_b200 import ops
            c = self._caches[branch] = ops.MaskCache(self.mask_refresh_interval, self.mask_keep)
        return c

    def _tick(self):
        self.current_step += 1
        if self.current_step == self.steps_per_cycle:
            self.current_step = 0
            for c in self._caches or ():
                if c is not None:
                    c.reset()


class WanProcessorBase(ProcessorBase):
    """Wan2.1 T2V / I2V and Wan2.2 TI2V / T2V / I2V self-attention processors; they differ only in the warm-up gate,
    the RoPE convention and the step wrap."""

    steps_per_cycle = 100
    calls_per_step = 2  # conditional + unconditional forward per denoising step
    rope = "complex"  # "complex" (Wan2.1) | "cos_sin" (Wan2.2)

    def __init__(self, mode, select_block_num, block_neighbor_list, p_remain_rates, processor_id=0,
                 first_frame_blocks=0):
        super().__init__(mode, select_block_num, block_neighbor_list, p_remain_rates, processor_id)
        self.first_frame_blocks = first_frame_blocks

    def sparse_now(self) -> bool:
        raise NotImplementedError

    def _fused(self, attn, hidden_states, rotary_emb, enc_img, dense=False, fp16=False):
        """Kernel 0 form of the middle section (reference rectified_wan21_attn.py:419-470): projections -> RMSNorm across
        heads + rotary embedding + head split + pooling in one pass -> kernels 3a-4.  None when the layer does not have
        the shape kernel 0 fuses.  `dense`: a warm-up call or dense layer -- kernel 0 without pooling, then dense
        attention over all S tokens.  `fp16`: fp16 activations (and fp16 norm weights) take kernel 0 too."""
        from rsa_b200 import geometry as G
        from rsa_b200 import ops
        heads = attn.heads
        if not hidden_states.is_cuda or not prep_dtype_ok(hidden_states, fp16):
            return None
        dt = hidden_states.dtype
        nq_ = wan_rms_params(getattr(attn, "norm_q", None), heads, dt)
        nk_ = wan_rms_params(getattr(attn, "norm_k", None), heads, dt)
        if nq_ is None or nk_ is None or nq_[1] != nk_[1]:
            return None
        b, s, _ = hidden_states.shape
        rope = None
        if rotary_emb is not None:
            rope = wan_rope_tables(rotary_emb, s)
            if rope is None:
                return None
        src = [f(hidden_states) for f in (attn.to_q, attn.to_k, attn.to_v)]
        if src[0].shape[2] != heads * 128:
            return None
        q, k, v = (torch.empty(b, heads, s, 128, dtype=dt, device=hidden_states.device) for _ in range(3))
        plan = ops.Plan(q, k, v, G.wan(s, self.first_frame_blocks), self.select_block_num, self.p_remain_rates,
                        self.block_neighbor_list, mask_cache=None if dense else self._mask_cache())
        plan.qkv_prep(*src, dst_row=0, q_weight=nq_[0], k_weight=nk_[0], eps=nq_[1], rope=rope, pool=not dense,
                      allow_fp16=fp16)
        out = (plan.run_dense(s, s) if dense else plan.run_pooled()).view(b, s, heads * 128)
        if enc_img is not None:
            out = out + image_cross_attention(attn, q, enc_img)
        return out

    def __call__(self, attn, hidden_states: torch.Tensor, encoder_hidden_states: Optional[torch.Tensor] = None,
                 attention_mask: Optional[torch.Tensor] = None, rotary_emb=None) -> torch.Tensor:
        from .attn import fullattn
        from .rectified_wan21_attn import rectified_block_sparse_attention

        enc_img, encoder_hidden_states = split_wan_context(attn, encoder_hidden_states)
        if encoder_hidden_states is None:
            encoder_hidden_states = hidden_states
        if self.mode == "sparse" and self.sparse_now() and self.fuse_prep and encoder_hidden_states is hidden_states:
            fused = self._fused(attn, hidden_states, rotary_emb, enc_img, fp16=self.fuse_prep_fp16)
            if fused is not None:
                self._tick()
                return attn.to_out[1](attn.to_out[0](fused))
        if (self.mode == "flash" or (self.mode == "sparse" and not self.sparse_now())) and self.fuse_prep_dense \
                and encoder_hidden_states is hidden_states and attention_mask is None:
            fused = self._fused(attn, hidden_states, rotary_emb, enc_img, dense=True, fp16=self.fuse_prep_fp16)
            if fused is not None:
                self._tick()
                return attn.to_out[1](attn.to_out[0](fused))
        query = attn.to_q(hidden_states)
        key = attn.to_k(encoder_hidden_states)
        value = attn.to_v(encoder_hidden_states)
        if getattr(attn, "norm_q", None) is not None:
            query = attn.norm_q(query)
        if getattr(attn, "norm_k", None) is not None:
            key = attn.norm_k(key)
        if self.rope == "cos_sin":
            query, key, value = (t.unflatten(2, (attn.heads, -1)) for t in (query, key, value))
            if rotary_emb is not None:
                query, key = rope_cos_sin(query, *rotary_emb), rope_cos_sin(key, *rotary_emb)
            query, key, value = query.transpose(1, 2), key.transpose(1, 2), value.transpose(1, 2)
        else:
            query, key, value = (heads_first(t, attn.heads) for t in (query, key, value))
            if rotary_emb is not None:
                query, key = rope_complex(query, rotary_emb), rope_complex(key, rotary_emb)
        hidden_img = image_cross_attention(attn, query, enc_img) if enc_img is not None else None

        s_k = kv_valid(attention_mask, key.shape[2])
        if self.mode == "sparse" and self.sparse_now():
            hidden_states = rectified_block_sparse_attention(
                query, key, value, attn_mask=attention_mask, top_k=self.select_block_num,
                max_seqlen_q=query.shape[2], max_seqlen_kv=key.shape[2], block_neighbor_list=self.block_neighbor_list,
                p_remain_rates=self.p_remain_rates, first_frame_blocks=self.first_frame_blocks,
                mask_cache=self._mask_cache())
        elif self.mode == "sparse":
            hidden_states = dense(fullattn, query, key, value, "flash", attention_mask, s_k)
        elif self.mode in ("flash", "torch", "vanilla"):
            hidden_states = dense(fullattn, query, key, value, self.mode, attention_mask, s_k)
        else:
            raise ImportError("Undefined Attention Processor! Just support sparse, flash, torch, vanilla.")
        hidden_states = hidden_states.type_as(query)
        self._tick()
        if hidden_img is not None:
            hidden_states = hidden_states + hidden_img
        hidden_states = attn.to_out[0](hidden_states)
        hidden_states = attn.to_out[1](hidden_states)
        return hidden_states
