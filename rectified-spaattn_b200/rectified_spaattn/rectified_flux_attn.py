"""Drop-in mirror of the reference rectified_spaattn/rectified_flux_attn.py (Flux.1-dev joint attention: image
tokens first, `text_length` text tokens last; image token counts that do not fill whole blocks -- 1360x768, 1280x720,
832x1216, 1920x1088 -- take the padded layout of geometry.flux, which the reference does not have).  See rectified_wan21_attn.py for the symbol map."""
import torch

from rsa_b200 import geometry as _G
from rsa_b200 import ops as _ops

from . import _common
from .attn import fullattn  # noqa: F401
from .gapr_mask import estimate_pr_gain  # noqa: F401
from .rectified_wan21_attn import _triton_block_sparse_attention_onehot  # noqa: F401


def _build_block_index_with_importance_optimized(query, key, top_k, block_size_M=128, block_size_N=128,
                                                 text_start_block=None, text_end_block=None, num_blocks=None,
                                                 prob_threshold=0.7, block_neighbor_list=None, attenable=None):
    _common.check_blocks(block_size_M, block_size_N)
    geo = _G.flux(key.shape[2], int(attenable))
    return _common.build_index(query, key, geo, top_k, prob_threshold, block_neighbor_list)


def block_sparse_attention_combined(query, key, value, attn_mask, top_k, block_size_M=128, block_size_N=128,
                                    cu_seqlens_q=None, cu_seqlens_kv=None, max_seqlen_q=None, max_seqlen_kv=None,
                                    prob_threshold=0.5, block_neighbor_list=None, text_length=256, shape_xfuse=False,
                                    mask_cache=None):
    _common.check_blocks(block_size_M, block_size_N)
    cu = _common.host_ints(cu_seqlens_kv)
    kv_len = cu[1] if cu is not None else None     # seqlens = cu_seqlens_kv[1:2]  (reference :307)
    geo = _G.flux(query.shape[2], int(text_length), kv_len)
    return _common.run(query, key, value, geo, top_k, prob_threshold, block_neighbor_list, shape_xfuse,
                       mask_cache)


def rectified_block_sparse_attention(query, key, value, attn_mask, top_k, block_size_M=128, block_size_N=128,
                                     cu_seqlens_q=None, cu_seqlens_kv=None, max_seqlen_q=None, max_seqlen_kv=None,
                                     block_neighbor_list=None, shape_xfuse=False, p_remain_rates=0.5, text_length=256,
                                     mask_cache=None):
    return block_sparse_attention_combined(
        query, key, value, attn_mask, top_k, block_size_M, block_size_N, cu_seqlens_q, cu_seqlens_kv,
        max_seqlen_q, max_seqlen_kv, block_neighbor_list=block_neighbor_list, shape_xfuse=shape_xfuse,
        prob_threshold=p_remain_rates, text_length=text_length, mask_cache=mask_cache)


from . import _processors as _P  # noqa: E402
from .attn import fullattn as _fullattn  # noqa: E402


class RectifiedFluxSpaAttnProcessor2_0(_P.ProcessorBase):
    """Flux.1-dev processor (reference :408-542): text tokens moved LAST ("Jenga attention"), RoPE over the whole
    joint sequence, sparse except in single-stream blocks 37..56 (the last 20), which stay dense."""

    def __init__(self, mode, select_block_num, block_neighbor_list, p_remain_rates, processor_id=0, text_length=256):
        super().__init__(mode, select_block_num, block_neighbor_list, p_remain_rates, processor_id)
        self.text_length = text_length

    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None, image_rotary_emb=None):
        sparse = self.mode == "sparse" and (self.processor_id < 37 or self.processor_id >= 57)
        # every call that is not sparse goes to fullattn(mode="flash") below: single-stream blocks 37-56, other modes
        if (self.fuse_prep if sparse else self.fuse_prep_dense) and attention_mask is None:
            # kernel 0: everything between the projections and the attention in one pass (reference :431-486)
            s = hidden_states.shape[1] + (encoder_hidden_states.shape[1] if encoder_hidden_states is not None else 0)
            fused = None
            if s > self.text_length:    # a ragged S takes the padded layout of _G.flux (two kernel-0 calls)
                fused = _P.fused_prep_attention(attn, hidden_states, encoder_hidden_states, _G.flux(s, self.text_length),
                                                self.select_block_num, self.p_remain_rates, self.block_neighbor_list,
                                                image_rotary_emb, rope_text=True,
                                                mask_cache=self._mask_cache() if sparse else None, dense=not sparse, fp16=self.fuse_prep_fp16)
            if fused is not None:
                self._tick()
                if encoder_hidden_states is None:
                    return fused
                n_txt = encoder_hidden_states.shape[1]
                hidden_states, encoder_hidden_states = fused[:, :-n_txt], fused[:, -n_txt:]
                return attn.to_out[1](attn.to_out[0](hidden_states)), attn.to_add_out(encoder_hidden_states)
        query, key, value = (_P.heads_first(f(hidden_states), attn.heads) for f in (attn.to_q, attn.to_k, attn.to_v))
        if getattr(attn, "norm_q", None) is not None:
            query = attn.norm_q(query)
        if getattr(attn, "norm_k", None) is not None:
            key = attn.norm_k(key)
        if encoder_hidden_states is not None:  # dual-stream block: context projections, appended last
            eq, ek, ev = (_P.heads_first(f(encoder_hidden_states), attn.heads)
                          for f in (attn.add_q_proj, attn.add_k_proj, attn.add_v_proj))
            if getattr(attn, "norm_added_q", None) is not None:
                eq = attn.norm_added_q(eq)
            if getattr(attn, "norm_added_k", None) is not None:
                ek = attn.norm_added_k(ek)
            query, key, value = (torch.cat([a, b], dim=2) for a, b in ((query, eq), (key, ek), (value, ev)))
        if image_rotary_emb is not None:
            query, key = _P.rope_real(query, image_rotary_emb), _P.rope_real(key, image_rotary_emb)

        s_k = _P.kv_valid(attention_mask, key.shape[2])
        if self.mode == "sparse" and (self.processor_id < 37 or self.processor_id >= 57):
            cu = [0, s_k, key.shape[2]]
            hidden_states = rectified_block_sparse_attention(
                query, key, value, attn_mask=attention_mask, top_k=self.select_block_num, cu_seqlens_q=cu,
                cu_seqlens_kv=cu, max_seqlen_q=query.shape[2], max_seqlen_kv=key.shape[2],
                block_neighbor_list=self.block_neighbor_list, p_remain_rates=self.p_remain_rates,
                text_length=self.text_length,
                mask_cache=self._mask_cache())
        else:
            hidden_states = _P.dense(_fullattn, query, key, value, "flash", attention_mask, s_k)
        hidden_states = hidden_states.to(query.dtype)
        self._tick()
        if encoder_hidden_states is not None:
            n_txt = encoder_hidden_states.shape[1]
            hidden_states, encoder_hidden_states = hidden_states[:, :-n_txt], hidden_states[:, -n_txt:]
            hidden_states = attn.to_out[1](attn.to_out[0](hidden_states))
            encoder_hidden_states = attn.to_add_out(encoder_hidden_states)
            return hidden_states, encoder_hidden_states
        return hidden_states
