"""Drop-in mirror of the reference rectified_spaattn/rectified_cogvideo_attn.py (CogVideoX1.5 joint attention:
video tokens first, text last, zero-padded to a multiple of 128).  See rectified_wan21_attn.py for the symbol map."""
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
    s = key.shape[2]
    nq = int(text_start_block) if text_start_block is not None else (s // 128 - (int(attenable) + 127) // 128)
    a = int(attenable)
    geo = _G.BlockGeometry(1, s, (s + 127) // 128, nq, a, s, s, (s + 127) // 128, s - nq * 128)
    return _common.build_index(query, key, geo, top_k, prob_threshold, block_neighbor_list)


def block_sparse_attention_combined(query, key, value, attn_mask, top_k, block_size_M=128, block_size_N=128,
                                    cu_seqlens_q=None, cu_seqlens_kv=None, max_seqlen_q=None, max_seqlen_kv=None,
                                    prob_threshold=0.5, block_neighbor_list=None, text_length=256, shape_xfuse=False,
                                    mask_cache=None):
    _common.check_blocks(block_size_M, block_size_N)
    geo = _G.cogvideo(query.shape[2], int(text_length))
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


class RectifiedCogVideoXVideoSpaAttnProcessor2_0(_P.ProcessorBase):
    """CogVideoX1.5 processor (reference :410-523): text tokens moved LAST, RoPE on the video tokens only, sparse from
    call 5 on; returns (hidden_states, encoder_hidden_states) split after the output projection."""

    def __call__(self, attn, hidden_states, encoder_hidden_states, attention_mask=None, image_rotary_emb=None):
        n_txt = encoder_hidden_states.size(1)
        hidden_states = torch.cat([hidden_states, encoder_hidden_states], dim=1)
        b, s, _ = hidden_states.shape
        if attention_mask is not None:
            attention_mask = attn.prepare_attention_mask(attention_mask, s, b)
            attention_mask = attention_mask.view(b, attn.heads, -1, attention_mask.shape[-1])
        sparse = self.mode == "sparse" and self.current_step >= 5     # otherwise fullattn(mode="flash") below
        if ((self.fuse_prep if sparse else self.fuse_prep_dense) and attention_mask is None
                and not getattr(attn, "is_cross_attention", False)):
            # kernel 0: head split + LayerNorm + RoPE + pooling in one pass (reference :443-469), then kernels 3a-4
            fused = _P.fused_prep_attention(attn, hidden_states, None, _G.cogvideo(s, n_txt), self.select_block_num,
                                            self.p_remain_rates, self.block_neighbor_list, image_rotary_emb,
                                            rope_text=False, mask_cache=self._mask_cache() if sparse else None,
                                            dense=not sparse, fp16=self.fuse_prep_fp16)
            if fused is not None:
                self._tick()
                hidden_states = attn.to_out[1](attn.to_out[0](fused))
                return hidden_states.split([hidden_states.size(1) - n_txt, n_txt], dim=1)
        query, key, value = (_P.heads_first(f(hidden_states), attn.heads) for f in (attn.to_q, attn.to_k, attn.to_v))
        if getattr(attn, "norm_q", None) is not None:
            query = attn.norm_q(query)
        if getattr(attn, "norm_k", None) is not None:
            key = attn.norm_k(key)
        if image_rotary_emb is not None:
            query = torch.cat([_P.rope_real(query[:, :, :-n_txt], image_rotary_emb), query[:, :, -n_txt:]], dim=2)
            if not getattr(attn, "is_cross_attention", False):
                key = torch.cat([_P.rope_real(key[:, :, :-n_txt], image_rotary_emb), key[:, :, -n_txt:]], dim=2)

        s_k = _P.kv_valid(attention_mask, key.shape[2])
        if self.mode == "sparse" and self.current_step >= 5:
            cu = [0, s_k, key.shape[2]]
            hidden_states = rectified_block_sparse_attention(
                query, key, value, attn_mask=attention_mask, top_k=self.select_block_num, cu_seqlens_q=cu,
                cu_seqlens_kv=cu, max_seqlen_q=s, max_seqlen_kv=key.shape[2],
                block_neighbor_list=self.block_neighbor_list, p_remain_rates=self.p_remain_rates, text_length=n_txt,
                mask_cache=self._mask_cache())
        else:
            hidden_states = _P.dense(_fullattn, query, key, value, "flash", attention_mask, s_k)
        hidden_states = hidden_states.to(query.dtype)
        self._tick()
        hidden_states = attn.to_out[1](attn.to_out[0](hidden_states))
        return hidden_states.split([hidden_states.size(1) - n_txt, n_txt], dim=1)
