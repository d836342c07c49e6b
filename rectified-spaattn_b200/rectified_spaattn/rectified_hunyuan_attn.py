"""Drop-in mirror of the reference rectified_spaattn/rectified_hunyuan_attn.py (HunyuanVideo joint text+video
attention: video tokens first, 256 text tokens last).  See rectified_wan21_attn.py for the symbol map; the
text-row flash-attn call (reference :371-380) and the K/V masked_fill_ (:307-308) are folded into the kernels
(dense query tiles, kv_len bound) -- key/value are NOT modified in place.
"""
import torch

from rsa_b200 import geometry as _G
from rsa_b200 import ops as _ops

from . import _common
from .attn import fullattn  # noqa: F401
from .gapr_mask import estimate_pr_gain  # noqa: F401
from .rectified_wan21_attn import _triton_block_sparse_attention_onehot  # noqa: F401  (identical kernel)


def _geometry(seq, cu_seqlens_q, num_true):
    if num_true is None:
        cu = _common.host_ints(cu_seqlens_q)
        if cu is None:
            raise RuntimeError("HunyuanVideo path needs cu_seqlens_q = [0, num_true, S] (the reference's "
                               "no-cu_seqlens branch leaves `attenable` undefined, rectified_hunyuan_attn.py:318-323)")
        num_true = cu[1]
        if cu[2] != seq:
            raise ValueError("cu_seqlens_q[2] must equal the sequence length")
    return _G.hunyuan(seq, int(num_true))


def _build_block_index_with_importance_optimized(query, key, top_k, block_size_M=128, block_size_N=128,
                                                 text_start_block=None, text_end_block=None, num_blocks=None,
                                                 prob_threshold=0.7, block_neighbor_list=None, attenable=None):
    _common.check_blocks(block_size_M, block_size_N)
    s = key.shape[2]
    a = int(attenable)
    geo = _G.hunyuan(s, s - 256 + a)
    return _common.build_index(query, key, geo, top_k, prob_threshold, block_neighbor_list)


def block_sparse_attention_combined(query, key, value, attn_mask, top_k, block_size_M=128, block_size_N=128,
                                    cu_seqlens_q=None, cu_seqlens_kv=None, max_seqlen_q=None, max_seqlen_kv=None,
                                    prob_threshold=0.5, block_neighbor_list=None, shape_xfuse=False, num_true=None,
                                    mask_cache=None):
    _common.check_blocks(block_size_M, block_size_N)
    geo = _geometry(query.shape[2], cu_seqlens_q, num_true)
    return _common.run(query, key, value, geo, top_k, prob_threshold, block_neighbor_list, shape_xfuse,
                       mask_cache)


def rectified_block_sparse_attention(query, key, value, attn_mask, top_k, block_size_M=128, block_size_N=128,
                                     cu_seqlens_q=None, cu_seqlens_kv=None, max_seqlen_q=None, max_seqlen_kv=None,
                                     block_neighbor_list=None, shape_xfuse=False, p_remain_rates=0.5, num_true=None,
                                     mask_cache=None):
    """`num_true` (host int) is an optional extension: it avoids reading cu_seqlens_q back from the device."""
    return block_sparse_attention_combined(
        query, key, value, attn_mask, top_k, block_size_M, block_size_N, cu_seqlens_q, cu_seqlens_kv,
        max_seqlen_q, max_seqlen_kv, block_neighbor_list=block_neighbor_list, shape_xfuse=shape_xfuse,
        prob_threshold=p_remain_rates, num_true=num_true, mask_cache=mask_cache)


from . import _processors as _P  # noqa: E402


class RectifiedHunyuanVideoSpaAttnProcessor2_0(_P.ProcessorBase):
    """HunyuanVideo joint text+video processor (reference :419-545): text tokens are appended LAST, RoPE on the video
    tokens only, sparse at every layer and step when mode == "sparse"; returns (hidden_states,
    encoder_hidden_states).  `num_true` (valid tokens = video + unpadded text) is read from `attention_mask` with one
    host sync per call exactly like the reference (:502) unless the caller sets `self.num_true`."""

    num_true = None

    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None, image_rotary_emb=None):
        single_stream = getattr(attn, "add_q_proj", None) is None and encoder_hidden_states is not None
        if single_stream:
            hidden_states = torch.cat([hidden_states, encoder_hidden_states], dim=1)
        sparse = self.mode == "sparse"
        if ((sparse and self.fuse_prep) or (self.mode == "flash" and self.fuse_prep_dense)) \
                and encoder_hidden_states is not None:
            # kernel 0: everything between the projections and the attention in one pass (reference :448-498)
            s = hidden_states.shape[1] + (0 if single_stream else encoder_hidden_states.shape[1])
            num_true = self.num_true if self.num_true is not None else _P.kv_valid(attention_mask, s)
            fused = _P.fused_prep_attention(attn, hidden_states, None if single_stream else encoder_hidden_states,
                                            _G.hunyuan(s, int(num_true), encoder_hidden_states.shape[1]),
                                            self.select_block_num, self.p_remain_rates, self.block_neighbor_list,
                                            image_rotary_emb, rope_text=False,
                                            mask_cache=self._mask_cache() if sparse else None, dense=not sparse, fp16=self.fuse_prep_fp16)
            if fused is not None:
                n_txt = encoder_hidden_states.shape[1]
                hidden_states, encoder_hidden_states = fused[:, :-n_txt], fused[:, -n_txt:]
                if getattr(attn, "to_out", None) is not None:
                    hidden_states = attn.to_out[1](attn.to_out[0](hidden_states))
                if getattr(attn, "to_add_out", None) is not None:
                    encoder_hidden_states = attn.to_add_out(encoder_hidden_states)
                self._tick()
                return hidden_states, encoder_hidden_states
        query, key, value = (_P.heads_first(f(hidden_states), attn.heads) for f in (attn.to_q, attn.to_k, attn.to_v))
        if getattr(attn, "norm_q", None) is not None:
            query = attn.norm_q(query)
        if getattr(attn, "norm_k", None) is not None:
            key = attn.norm_k(key)
        if image_rotary_emb is not None:
            if single_stream:
                n_txt = encoder_hidden_states.shape[1]
                query = torch.cat([_P.rope_real(query[:, :, :-n_txt], image_rotary_emb), query[:, :, -n_txt:]], dim=2)
                key = torch.cat([_P.rope_real(key[:, :, :-n_txt], image_rotary_emb), key[:, :, -n_txt:]], dim=2)
            else:
                query, key = _P.rope_real(query, image_rotary_emb), _P.rope_real(key, image_rotary_emb)
        if getattr(attn, "add_q_proj", None) is not None and encoder_hidden_states is not None:
            eq, ek, ev = (_P.heads_first(f(encoder_hidden_states), attn.heads)
                          for f in (attn.add_q_proj, attn.add_k_proj, attn.add_v_proj))
            if getattr(attn, "norm_added_q", None) is not None:
                eq = attn.norm_added_q(eq)
            if getattr(attn, "norm_added_k", None) is not None:
                ek = attn.norm_added_k(ek)
            query, key, value = (torch.cat([a, b], dim=2) for a, b in ((query, eq), (key, ek), (value, ev)))

        b, _, s, _ = query.shape
        num_true = self.num_true if self.num_true is not None else _P.kv_valid(attention_mask, s)
        if self.mode == "sparse":
            hidden_states = rectified_block_sparse_attention(
                query, key, value, attn_mask=attention_mask, top_k=self.select_block_num, max_seqlen_q=s,
                max_seqlen_kv=s, block_neighbor_list=self.block_neighbor_list, p_remain_rates=self.p_remain_rates,
                num_true=num_true,
                mask_cache=self._mask_cache())
        elif self.mode in ("flash", "torch", "vanilla"):
            cu = [0, num_true, s]
            hidden_states = fullattn(query, key, value, mode=self.mode, drop_rate=0.0, attn_mask=attention_mask,
                                     causal=False, cu_seqlens_q=cu, cu_seqlens_kv=cu, max_seqlen_q=s, max_seqlen_kv=s,
                                     batch_size=b)
            hidden_states = hidden_states.transpose(1, 2).reshape(b, s, -1)
        if encoder_hidden_states is not None:
            n_txt = encoder_hidden_states.shape[1]
            hidden_states, encoder_hidden_states = hidden_states[:, :-n_txt], hidden_states[:, -n_txt:]
            if getattr(attn, "to_out", None) is not None:
                hidden_states = attn.to_out[1](attn.to_out[0](hidden_states))
            if getattr(attn, "to_add_out", None) is not None:
                encoder_hidden_states = attn.to_add_out(encoder_hidden_states)
        self._tick()
        return hidden_states, encoder_hidden_states
