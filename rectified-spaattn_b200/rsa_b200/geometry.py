"""Per-model block geometry of one attention call, reduced to the integers rsa_attn_desc carries.

Mirrors how each reference family derives seqlens / attenable / normal_blocks / text_end_block / padding:
  wan       rectified_wan21_attn.py:299-313
  hunyuan   rectified_hunyuan_attn.py:313-332   (the reference needs S % 128 == 0 and raises otherwise, :356; here a
            ragged visual segment -- 129 frames = 118 800 tokens -- is completed with zero rows, see hunyuan())
  flux      rectified_flux_attn.py:307-317     (the reference needs S % 128 == 0 and raises otherwise; here a ragged
            visual segment -- 1360x768 = 4 080 image tokens -- is completed with zero rows, see flux())
  cogvideo  rectified_cogvideo_attn.py:307-322 (the reference's rule has no layout when the visual tokens end 1-30 tokens
            past a block boundary with 226 text tokens -- 49 frames at 480x720 = 17 550 tokens; those are completed with
            zero rows, see cogvideo())
"""
from __future__ import annotations

from dataclasses import dataclass

BLOCK = 128


@dataclass(frozen=True)
class BlockGeometry:
    family: int            # native.FAMILY_WAN / FAMILY_JOINT
    seq: int
    n_blocks: int
    nq_blocks: int
    text_keys: int
    kv_len: int
    kv_zero_from: int
    text_end_block: int
    text_q_valid: int
    first_frame_blocks: int = 0
    vis_len: int = 0       # joint family: visual tokens when they do not fill whole blocks (0 = nq_blocks * 128)

    @property
    def gap(self):
        """Zero rows that complete the last visual block in the padded layout (not present in memory)."""
        return self.nq_blocks * BLOCK - self.vis_len if self.vis_len else 0


def _ceil_blocks(n):
    return (n + BLOCK - 1) // BLOCK


def wan(seq, first_frame_blocks=0):
    nb = _ceil_blocks(seq)
    return BlockGeometry(0, seq, nb, nb, 0, seq, seq, nb, 0, int(first_frame_blocks or 0))


def hunyuan(seq, num_true, text_len=256):
    """HunyuanVideo: `text_len` (256) text tokens last, `num_true` = visual + valid text tokens.

    Block-aligned visual segment (S % 128 == 0): exactly the reference's live branch (:313-332).
    Ragged visual segment (the 129-frame shape, 118 800 + 256): the reference raises (:356).  Extension, following the
    rule its Wan/CogVideoX paths use for ragged inputs (wan21 :299-302): the last visual block is completed with
    zero rows -- pooled as zeros with divisor 128, never attended as keys, never written as queries -- and the text
    blocks follow block-aligned.  kv_len / kv_zero_from / text_end_block are positions in that padded layout."""
    nv = seq - text_len
    attenable = text_len - (seq - num_true)
    if nv <= 0 or attenable < 1 or num_true > seq:
        raise ValueError(f"inconsistent HunyuanVideo geometry: S={seq}, num_true={num_true}")
    nq = _ceil_blocks(nv)
    gap = nq * BLOCK - nv
    nb = nq + _ceil_blocks(text_len)
    valid_v = num_true + gap                      # end of the valid keys in the padded layout
    return BlockGeometry(1, seq, nb, nq, attenable, valid_v, valid_v, _ceil_blocks(valid_v), num_true - nv,
                         vis_len=nv if gap else 0)


def _padded_joint(seq, text_length, kv_len=None):
    """Joint layout [visual | gap zero rows | text] of a ragged visual segment (the extension hunyuan() describes):
    `seq - text_length` visual tokens in ceil(/128) blocks, the text blocks block-aligned behind them, and kv_len /
    kv_zero_from shifted by the gap into the padded layout.  Every text token is a text key and a valid text query."""
    nv = seq - text_length
    if nv <= 0 or text_length < 1:
        raise ValueError(f"inconsistent joint geometry: S={seq}, text_length={text_length}")
    nq = _ceil_blocks(nv)
    gap = nq * BLOCK - nv
    nb = nq + _ceil_blocks(text_length)
    kv = (seq if kv_len is None else int(kv_len)) + gap
    return BlockGeometry(1, seq, nb, nq, text_length, kv, seq + gap, _ceil_blocks(kv), text_length,
                         vis_len=nv if gap else 0)


def flux(seq, text_length, kv_len=None):
    """Flux.1-dev: `text_length` text tokens last.  S % 128 == 0: exactly the reference's rule (:307-317).  Ragged S
    (1360x768: 4 080 + 512 tokens): the reference raises; extension as in hunyuan() -- the last visual block is
    completed with zero rows, pooled as zeros with divisor 128, never attended as keys, never written as queries, and
    the text blocks follow block-aligned (_padded_joint)."""
    if seq % BLOCK:
        return _padded_joint(seq, text_length, kv_len)
    kv_len = seq if kv_len is None else int(kv_len)
    nb = seq // BLOCK
    nq = nb - text_length // BLOCK
    if nq <= 0 or text_length < 1:
        raise ValueError(f"inconsistent Flux geometry: S={seq}, text_length={text_length}")
    return BlockGeometry(1, seq, nb, nq, text_length, kv_len, seq, _ceil_blocks(kv_len), seq - nq * BLOCK)


def cogvideo(seq, text_length):
    """CogVideoX: `text_length` (226) text tokens last.  Wherever the reference's rule (:307-322) lays the sequence out
    it is used as is -- including when it counts the first text tokens as visual (visual tokens 31-127 past a block
    boundary with 226 text tokens).  Where it has no layout (nq * 128 + text_length > n_blocks * 128: CogVideoX-2B / -5B
    at 49 frames, 17 550 + 226 tokens) the reference raises; extension as in hunyuan() -- the last visual block is
    completed with zero rows, pooled as zeros with divisor 128, never attended as keys, never written as queries, and
    the text blocks follow block-aligned (_padded_joint)."""
    nb = _ceil_blocks(seq)
    pad = nb * BLOCK - seq
    nq = nb - (text_length + pad) // BLOCK
    if nq <= 0 or text_length < 1:
        raise ValueError(f"inconsistent CogVideoX geometry: S={seq}, text_length={text_length}")
    if nq * BLOCK + text_length > nb * BLOCK:
        return _padded_joint(seq, text_length)
    return BlockGeometry(1, seq, nb, nq, text_length, seq, seq, nb, seq - nq * BLOCK)
