"""Mirror of the reference rectified_spaattn/attn.py (dense attention helper).

`fullattn(..., mode="flash")` -- the only mode on the sparse path (text rows, warm-up layers/steps; reference
attn.py:107-120 calls flash_attn_varlen_func) -- runs on kernel 4's list-free dense form (rsa_dense_attention), so the
package has no flash-attn dependency.  Modes "torch" and "vanilla" are the reference's A/B-comparison switches
(scripts --mode), not part of the hot path; they are kept as plain PyTorch for completeness.
"""
import math

import torch
import torch.nn.functional as F

from rsa_b200 import ops as _ops

MEMORY_LAYOUT = {
    "flash": (lambda x: x, lambda x: x),  # kernel 4 reads [b,a,s,d] through strides: no varlen repacking
    "torch": (lambda x: x, lambda x: x),
    "vanilla": (lambda x: x, lambda x: x),
}


def get_cu_seqlens(img_seq_len, txt_seq_len, text_len, device="cuda"):
    """cu_seqlens = [0, img+text_len[0], max_len, ...] as int32 (reference attn.py:34-57)."""
    batch_size = len(text_len)
    max_len = img_seq_len + txt_seq_len
    cu = [0] * (2 * batch_size + 1)
    for i in range(batch_size):
        cu[2 * i + 1] = i * max_len + int(text_len[i]) + img_seq_len
        cu[2 * i + 2] = (i + 1) * max_len
    return torch.tensor(cu, dtype=torch.int32, device=device)


def _flash_like(q, k, v, cu_seqlens_q, cu_seqlens_kv, batch_size):
    """Dense attention with the varlen semantics the reference relies on: query rows below cu_seqlens_q[1] attend
    keys below cu_seqlens_kv[1]; the remaining (padding) rows are defined as zeros.  q,k,v are [B,H,S,D]."""
    b, h, sq, d = q.shape
    skv = k.shape[2]
    q_valid, kv_len = sq, skv
    if cu_seqlens_q is not None:
        cq = cu_seqlens_q.tolist() if isinstance(cu_seqlens_q, torch.Tensor) else list(cu_seqlens_q)
        q_valid = min(sq, int(cq[1]))
    if cu_seqlens_kv is not None:
        ck = cu_seqlens_kv.tolist() if isinstance(cu_seqlens_kv, torch.Tensor) else list(cu_seqlens_kv)
        kv_len = min(skv, int(ck[1]))
    if q_valid < 1:
        return torch.zeros_like(q, memory_format=torch.contiguous_format)
    # kernel 4 walking every block without lists: bit-identical to the masked form on an all-ones mask with
    # fp32_scale=True (flash-attn's arithmetic), with no mask, no workspace and rows >= q_valid written as zeros
    return _ops.dense_attention(q, k, v, q_valid, kv_len)


def fullattn(q, k, v, mode="flash", drop_rate=0, attn_mask=None, causal=False, cu_seqlens_q=None,
             cu_seqlens_kv=None, max_seqlen_q=None, max_seqlen_kv=None, batch_size=1):
    """q [b,a,s,d], k/v [b,a,s1,d] -> [b,a,s,d] in every mode, like the reference (attn.py:60-154: the flash
    branch views the varlen result as [b, s, a, d] and its post-layout transposes it back)."""
    if mode == "flash":
        if causal or drop_rate:
            raise NotImplementedError("causal / dropout are unused on this path")
        if batch_size != 1 and cu_seqlens_q is not None:
            raise NotImplementedError("varlen batches > 1 are not used by any reference script")
        return _flash_like(q, k, v, cu_seqlens_q, cu_seqlens_kv, batch_size)
    if mode == "torch":
        if attn_mask is not None and attn_mask.dtype != torch.bool:
            attn_mask = attn_mask.to(q.dtype)
        return F.scaled_dot_product_attention(q, k, v, attn_mask=attn_mask, dropout_p=drop_rate, is_causal=causal)
    if mode == "vanilla":
        s = (q @ k.transpose(-2, -1)) * (1 / math.sqrt(q.size(-1)))
        if causal:
            s = s.masked_fill(~torch.ones(s.shape[-2:], dtype=torch.bool, device=q.device).tril(), float("-inf"))
        if attn_mask is not None:
            s = s.masked_fill(~attn_mask, float("-inf")) if attn_mask.dtype == torch.bool else s + attn_mask
        return torch.dropout(s.softmax(dim=-1), p=drop_rate, train=True) @ v
    raise NotImplementedError(f"Unsupported attention mode: {mode}")


def get_attn_mask(img_seq_len, txt_seq_len, text_len, device="cuda"):
    batch_size = len(text_len)
    m = torch.zeros(batch_size, img_seq_len + txt_seq_len, device=device, dtype=torch.bool)
    for i in range(batch_size):
        m[i, : img_seq_len + int(text_len[i])] = True
    return m.unsqueeze(1).unsqueeze(1)


def get_flash_attn_params(img_seq_len, txt_seq_len, text_len, device="cuda"):
    cu = get_cu_seqlens(img_seq_len, txt_seq_len, text_len, device)
    s = img_seq_len + txt_seq_len
    return cu, cu, s, s
