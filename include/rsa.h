/* rsa.h -- C ABI of librsa_b200.so: the rectified block-sparse attention hot path for NVIDIA B200 (sm_100a).
 *
 * Drop-in boundary for the hot path of BienLuky/Rectified-SpaAttn (reference paths relative to its root).
 * The reference has no native code; what it runs as PyTorch eager ops + a Triton JIT kernel + flash-attn calls
 * is exported here as plain C entry points (raw device pointers, explicit sizes/strides, a cudaStream_t passed
 * as void*, caller-owned workspace, int status codes, no exceptions, no allocation, no host synchronisation).
 * Each entry point cites the reference interface it replaces.  The Python mirror of the reference modules
 * (rectified-spaattn_b200/rectified_spaattn/*.py) binds these with ctypes; INTEGRATION.md shows the stub a
 * maintainer of the reference would add.
 *
 * Conventions: all tensors are bf16 unless stated (query/key/value/out may be fp16: rsa_attn_desc.dtype), head_dim
 * 128 or 64 (CogVideoX; see rsa_attn_desc.head_dim and the entry points), block size == 128 tokens.
 * "BH" = batch * heads (heads are independent end to end).  Strides are in ELEMENTS of the tensor's dtype.
 */
#ifndef RSA_H_
#define RSA_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RSA_VERSION 110 /* 110: rsa_qkv_prep_gather takes the visual / text two-call form at head_dim 64 too */
#define RSA_BLOCK 128
#define RSA_HEAD_DIM 128
#define RSA_MAX_ENTRIES 2048 /* max sortable entries per query block: NQ (+1 for the text aggregate) */

enum rsa_status {
  RSA_OK = 0,
  RSA_ERR_ARG = -1,         /* null pointer, negative size, inconsistent geometry */
  RSA_ERR_UNSUPPORTED = -2, /* head_dim / norm form not built, too many blocks, misaligned strides */
  RSA_ERR_CUDA = -3,        /* a CUDA runtime/driver call failed; see rsa_last_error_string() */
  RSA_ERR_WORKSPACE = -4    /* workspace pointer null or smaller than rsa_attn_workspace_bytes() */
};

enum rsa_dtype {
  RSA_DTYPE_BF16 = 0, /* every reference script runs its transformer in bf16 */
  RSA_DTYPE_F16 = 1   /* the reference kernel is dtype-generic (p.to(q.dtype), rectified_wan21_attn.py:97): fp16 too */
};

enum rsa_family {
  RSA_FAMILY_WAN = 0,  /* video tokens only            (rectified_wan21_attn.py:276-357) */
  RSA_FAMILY_JOINT = 1 /* video tokens first, text last (rectified_{hunyuan,flux,cogvideo}_attn.py) */
};

/* Thread-local description of the last failure returned by any rsa_* call on this thread. */
const char* rsa_last_error_string(void);
int rsa_version(void);
/* 1 if the library was built with the tcgen05/TMEM/TMA attention kernel and the current device is sm_100. */
int rsa_device_ok(void);

/* The reference's recursion gilbert_xyz2d_r (utils/jenga_gilbert.py:84-288): index, counted from cur_idx, of the point
 * (x_dst, y_dst, z_dst) on the generalised Hilbert curve through the box with origin (x, y, z) spanned by the major, mid
 * and minor vectors a, b, c (axis-parallel, signed).  -1 if the point is outside the box or the box is degenerate. */
int64_t rsa_gilbert_xyz2d_r(int64_t cur_idx, int64_t x_dst, int64_t y_dst, int64_t z_dst, int64_t x, int64_t y, int64_t z,
                            int64_t ax, int64_t ay, int64_t az, int64_t bx, int64_t by, int64_t bz, int64_t cx,
                            int64_t cy, int64_t cz);

/* ------------------------------------------------------------------------------------------------------
 * Host geometry (pure CPU).  Replaces utils/jenga_gilbert.py:
 *   gilbert_mapping(t,h,w,axis_order)                 :458-504  -> rsa_gilbert_map
 *   gilbert_block_neighbor_mapping(t,h,w,block_size)  :613-693  -> rsa_gilbert_block_neighbors
 * axis_order is a 3-character string over {'w','h','t'} (major, mid, minor), e.g. "wht"; NULL selects the
 * reference's size-based default (gilbert_xyz2d :34-54).  linear index = z*h*w + y*w + x.
 * out is a row-major [NB, NB] byte matrix (0/1), NB = ceil(t*h*w / block_size). */
int rsa_gilbert_map(int t, int h, int w, const char* axis_order, int64_t* linear_to_hilbert,
                    int64_t* hilbert_to_linear);
int rsa_gilbert_block_neighbors(int t, int h, int w, int block_size, const char* axis_order, uint8_t* out);

/* ------------------------------------------------------------------------------------------------------
 * Kernel 1: token permute / unpermute.  Replaces the advanced-index gathers in the patched transformer forward
 *   hidden_states[:, self.hilbert_order], hidden_states[:, self.linear_to_hilbert]  (scripts/main_hunyuan.py:88-89, :183)
 * dst[b, i, :] = src[b, index[i], :] for i < n_out.  index: device int64 (the reference keeps torch.long).
 * row_bytes must be a multiple of 16; src/dst 16-byte aligned; batch strides in bytes. */
int rsa_permute_rows(const void* src, void* dst, const int64_t* index, int batch, int64_t n_out, int64_t n_src,
                     int64_t row_bytes, int64_t src_batch_stride_bytes, int64_t dst_batch_stride_bytes,
                     void* stream);

/* ------------------------------------------------------------------------------------------------------
 * The attention path.  One descriptor describes one call of the reference's inner surface
 *   rectified_block_sparse_attention(query, key, value, attn_mask, top_k, ..., block_neighbor_list,
 *                                    p_remain_rates, first_frame_blocks | text_length)
 *   (rectified_wan21_attn.py:361-386, rectified_hunyuan_attn.py:393-417, rectified_flux_attn.py:380-405,
 *    rectified_cogvideo_attn.py:382-407)
 * after the per-family geometry (hunyuan :313-332, flux :307-317, cogvideo :307-322, wan21 :299-313) has been
 * reduced to integers by the caller. */
typedef struct rsa_attn_desc {
  int32_t batch, heads, seq, head_dim; /* query/key/value are [batch, heads, seq, head_dim] views; head_dim */
                                       /* 128, or 64 (CogVideoX): the kernels work on 128 columns and read the  */
                                       /* missing ones as zeros (no copy), which changes neither q.k, the pooled */
                                       /* statistics nor the GAPR test; the scale is head_dim^-1/2 either way    */
  int64_t q_stride[3];                 /* element strides of (batch, head, token); head_dim is contiguous  */
  int64_t k_stride[3];
  int64_t v_stride[3];
  int64_t o_stride[3];                 /* output viewed as [batch, heads, seq, head_dim]; the reference's   */
                                       /* [B, S, H*D] result is strides (S*H*D, D, H*D)                     */
  int32_t family;                      /* enum rsa_family                                                   */
  int32_t n_blocks;                    /* NB  = ceil(seq/128): KV blocks (pad rows count as zeros)          */
  int32_t nq_blocks;                   /* NQ  = query blocks on the sparse path (= visual blocks)           */
  int32_t text_keys;                   /* a   = text keys scored as single tokens (`attenable`), 0 for WAN  */
  int32_t kv_len;                      /* Lkv = keys >= kv_len are never attended (`seqlens`)               */
  int32_t kv_zero_from;                /* K,V rows >= this pool as zeros (hunyuan masked_fill_ :307-308)    */
  int32_t text_end_block;              /* first KV block that is never kept                                 */
  int32_t text_q_valid;                /* text query rows with a defined result; later rows are zero-filled */
  int32_t top_k;                       /* select_block_num                                                  */
  float p_remain;                      /* p_remain_rates (compared as fp32)                                 */
  int32_t first_frame_blocks;          /* WAN only, 0 = none                                                */
  int32_t nbr_rows, nbr_cols;          /* block_neighbor_list shape; both 0 = None                          */
  const uint8_t* nbr;                  /* DEVICE pointer, row-major bytes (torch.bool storage)              */
  int32_t debug_dump_probs;            /* !=0: stage 3b also writes P to the workspace (parity tests)       */
  int32_t vis_len;                     /* JOINT: visual tokens; text token i lives at memory row vis_len+i. */
                                       /* 0 = nq_blocks*128 (block-aligned visual segment, the only case    */
                                       /* the reference runs, hunyuan :356).  Otherwise nq_blocks =         */
                                       /* ceil(vis_len/128): the last visual block is completed with        */
                                       /* gap = nq_blocks*128 - vis_len zero rows (the Wan/CogVideoX rule,  */
                                       /* wan21 :299-302: pooled as zeros, never attended, never written),  */
                                       /* n_blocks = nq_blocks + ceil((seq - vis_len)/128), and kv_len,     */
                                       /* kv_zero_from, text_end_block refer to that PADDED layout (visual  */
                                       /* token t at t, text token i at nq_blocks*128 + i).  seq and the    */
                                       /* strides always describe the tensors as they lie in memory.        */
  int32_t dtype;                       /* enum rsa_dtype of query / key / value / out (kernels 2 and 4; pooled   */
                                       /* statistics, scores and selection are fp32 either way).  Kernel 0       */
                                       /* (rsa_qkv_prep*) follows diffusers' rounding points in this dtype.      */
} rsa_attn_desc;

/* Pointers into the caller's workspace (all device memory, fp32 unless noted). */
typedef struct rsa_ws_view {
  float* q_pool;      /* [BH, NQ, 128]   block means of Q                  (wan21 :189-190)                 */
  float* q_mad;       /* [BH, NQ, 128]   mean |Q - Qp| per block           (gapr_mask.py:19,23)             */
  float* k_cat;       /* [BH, NKC, 128]  rows [0,NQ) = block means of K, rows [NQ,NQ+a) = text keys         */
  float* k_mad;       /* [BH, NQ, 128]                                     (gapr_mask.py:20,30)             */
  float* v_pool;      /* [BH, NB, 128]   block means of V                  (wan21 :337)                     */
  float* scores;      /* [BH, NQ, score_ld]  unscaled Qp.[Kp;Kt]^T         (wan21 :203)                     */
  uint8_t* nogapr;    /* [BH, NQ, nogapr_ld] bytes, columns [0,NQ)         (gapr_mask.py:42)                */
  float* probs;       /* [BH, NQ, ent_ld]  P (only if debug_dump_probs)    (wan21 :213 / hunyuan :223)      */
  float* w_skip;      /* [BH, NQ, ent_ld]  P where not(part) else 0        (wan21 :336)                     */
  uint32_t* mask_bits;/* [BH, NQT, mask_words] kept-block bitmask, bit j of word j/32 = block j             */
  uint16_t* kept_idx; /* [BH, NQT, NB] ascending kept block indices (u16)                                    */
  int32_t* kept_cnt;  /* [BH, NQT]                                                                           */
  int32_t* n_needed;  /* [BH, NQ]  n_i = max(#{cumsum <= p} + 1, top_k)    (wan21 :224-229)                 */
  float* R;           /* [BH, NQT]  (1 for text query blocks)              (wan21 :332)                     */
  float* C;           /* [BH, NQT, 128] (0 for text query blocks)          (wan21 :338)                     */
  int32_t nkc, score_ld, n_entries, ent_ld, mask_words, nqt, nogapr_ld, reserved;
  uint16_t* sched_idx;   /* [BH, NQT, NB] the order kernel 4 walks each list in: for the pair of query tiles (2p, 2p+1)  */
                         /* first the blocks both keep (ascending; K/V tiles loaded once for both), then the rest       */
  int32_t* pair_shared;  /* [BH, ceil(NQT/2)] length of that common prefix                                              */
  int32_t* quad_shared;  /* [BH, ceil(NQT/2)] how many of those blocks the PARTNER pair of kernel 4's 2-CTA cluster keeps  */
                         /* as well (they lead the prefix; one K/V tile per cluster, TMA multicast); 0 = no partner       */
} rsa_ws_view;

/* sizeof(rsa_attn_desc) / sizeof(rsa_prep_desc) / sizeof(rsa_peer_route) as THIS library was compiled: a binding written in
 * another language (INTEGRATION.md section 2) checks its own struct against these before the first call. */
size_t rsa_attn_desc_size(void);
size_t rsa_prep_desc_size(void);
size_t rsa_peer_route_size(void);

size_t rsa_attn_workspace_bytes(const rsa_attn_desc* d);
int rsa_attn_workspace_view(const rsa_attn_desc* d, void* workspace, size_t workspace_bytes, rsa_ws_view* out);

/* Kernel 2: block mean pooling of Q, K, V + GAPR deviation statistics in one pass per tensor.
 * Replaces Q_blocks.mean / K_blocks.mean (wan21 :189-192), value_pool (:337) and delta_q/delta_k abs().mean()
 * (gapr_mask.py:19-30).  Fills q_pool, q_mad, k_cat, k_mad, v_pool. */
int rsa_pool_stats(const rsa_attn_desc* d, const void* q, const void* k, const void* v, void* workspace,
                   size_t workspace_bytes, void* stream);

/* Kernel 3a: pooled score products + GAPR test.  Replaces torch.bmm (wan21 :203) and estimate_pr_gain
 * (gapr_mask.py:26-42).  Fills scores, nogapr. */
int rsa_block_scores(const rsa_attn_desc* d, void* workspace, size_t workspace_bytes, void* stream);

/* Kernel 3b: softmax, IPAR re-allocation, sort / cumulative threshold / top-k, neighbour + first-frame + text
 * unions, R, skipped-block weights; emits the per-row kept-block index lists.  Replaces wan21 :206-271 /
 * hunyuan :208-277 and the R half of wan21 :329-333.  Tie-break: probability descending, index ascending;
 * cumulative sum sequential in fp32.  Fills probs (optional), mask_bits, kept_idx, kept_cnt, n_needed, R, w_skip. */
int rsa_block_select(const rsa_attn_desc* d, void* workspace, size_t workspace_bytes, void* stream);

/* Kernel 3c: C = W_skip . Vp.  Replaces torch.matmul(attn_pool_novalid, value_pool) (wan21 :336-338). */
int rsa_rect_c(const rsa_attn_desc* d, void* workspace, size_t workspace_bytes, void* stream);

/* Kernel 4: block-sparse attention over the kept lists with the rectification epilogue O = Os*R + C fused into
 * the output write, text query blocks handled as dense rows.  Replaces _triton_block_sparse_attention_onehot
 * (wan21 :108-168, kernel :16-105), the epilogue (wan21 :346), the flash-attn call for text rows
 * (hunyuan :371-380) and the cat/permute/reshape (hunyuan :383-387).  Reads kept_idx, kept_cnt, R, C; writes the
 * pair schedule (sched_idx, pair_shared) it walks. */
int rsa_sparse_attention(const rsa_attn_desc* d, const void* q, const void* k, const void* v, void* out,
                         void* workspace, size_t workspace_bytes, void* stream);

/* All of the above in order on one stream (no host synchronisation; CUDA-graph capturable). */
int rsa_rectified_attention(const rsa_attn_desc* d, const void* q, const void* k, const void* v, void* out,
                            void* workspace, size_t workspace_bytes, void* stream);

/* Mask re-use across calls (SURVEY 8f rank 4; the reference rebuilds its mask in every layer of every step,
 * rectified_hunyuan_attn.py:334-346, although the selections of adjacent denoising steps are highly correlated).  The
 * workspace of an earlier RSA_MASK_BUILD call on the same descriptor geometry is the cache:
 *   RSA_MASK_BUILD       same as rsa_rectified_attention (pooled = 0) / rsa_rectified_attention_pooled (pooled = 1)
 *   RSA_MASK_KEEP_LISTS  kernels 2 (unless pooled), 3a, 3b without its sort / threshold / scatter, 3c, 4: the kept-block
 *                        lists (and the pair schedule) stay; P, the GAPR test, R and C are recomputed from the CURRENT
 *                        q, k, v, so the rectification O = Os*R + C is exact for the cached selection
 *   RSA_MASK_KEEP_ALL    kernel 4 only: lists, R and C of the earlier call are applied to the current q, k, v
 * The caller decides when a cached selection is still good (same layer, adjacent step); nothing here checks it. */
enum rsa_mask_mode { RSA_MASK_BUILD = 0, RSA_MASK_KEEP_LISTS = 1, RSA_MASK_KEEP_ALL = 2 };
int rsa_rectified_attention_reuse(const rsa_attn_desc* d, const void* q, const void* k, const void* v, void* out,
                                  void* workspace, size_t workspace_bytes, int mask_mode, int pooled, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Kernel 0 (SURVEY 8f rank 1): what the reference's processors do between the QKV projections and the attention call,
 * fused into one pass over the projection outputs: head split, per-head QK RMSNorm, rotary embedding, re-layout
 * [B, rows, H*D] -> [B, H, S, D] (D = head_dim), and (pool != 0) kernel 2's block pooling of the rows just produced, so Q, K, V
 * are written once and never read back before kernel 4.  Replaces rectified_hunyuan_attn.py:448-479 and the same
 * sequence in rectified_flux_attn.py:
 *   query.unflatten(2, (heads, -1)).transpose(1, 2)                                   :448-450
 *   attn.norm_q / attn.norm_k = diffusers RMSNorm(head_dim, eps, elementwise_affine)   :453-456
 *       (x * rsqrt(mean(x^2) + eps) in fp32, rounded to bf16, times the bf16 weight, rounded to bf16)
 *   diffusers apply_rotary_emb(x, (cos, sin), use_real=True, use_real_unbind_dim=-1)   :459-478
 *       (x * cos + rotate_pairs(x) * sin in fp32, rounded to bf16; only the first rope_rows tokens)
 * and the Wan form of the same steps (rectified_wan21_attn.py:419-441, rectified_wan22_attn.py:44-64): RMSNorm over
 * all heads*128 channels before the head split (norm = 2), then the rotary embedding -- Wan2.1 multiplies complex pairs
 * in float64, Wan2.2 uses cos/sin tables; both are the same real arithmetic, done here in fp32 (the bf16 result
 * differs from the float64 route only when a value sits within 2^-24 of a rounding boundary).
 * diffusers 0.34.0 (requirements.txt:18) is not vendored in the reference; the two functions are restated from its
 * published source (oracle/prep_oracle.py).
 * One call handles the `rows` tokens of ONE source: the latent stream (dst_row = 0) or, for a dual-stream block, the
 * encoder stream (dst_row = visual token count; rope_rows = 0).  Destination tensors, their strides and the block
 * geometry come from the attention descriptor the rows are produced for.  With pool != 0 the workspace must be that
 * descriptor's workspace and every visual / text block must be produced by such calls before
 * rsa_rectified_attention_pooled runs.
 * head_dim 128 takes every norm; head_dim 64 (CogVideoX1.5: 48 heads x 64) takes norm 3 only (RSA_ERR_UNSUPPORTED
 * otherwise), with the pooled statistics' columns 64..127 written as zeros, as rsa_pool_stats computes them.
 * The 16-bit tensors -- sources, destinations, norm weights and biases -- are all in the descriptor's dtype, bf16 or fp16
 * (an fp16 model, e.g. CogVideoX-2B, runs the same diffusers sequence in fp16).  Every rounding point rounds to that
 * format to nearest even: in fp16 an overflow becomes +-inf, as .to(torch.float16) gives, and results below 2^-14 stay
 * subnormal.  The same norms and head dims are built in both dtypes. */
typedef struct rsa_prep_desc {
  int32_t rows;             /* tokens in the source tensors                                                   */
  int32_t dst_row;          /* memory row of the destination the first source token goes to: 0 or the visual  */
                            /* token count                                                                    */
  int64_t src_stride[3][2]; /* q, k, v sources [batch, rows, heads*head_dim]: (batch, token) element strides   */
  int32_t norm;             /* 0 = none, 1 = RMSNorm over head_dim (HunyuanVideo, Flux), 2 = RMSNorm over all  */
                            /* heads*128 channels of a token (Wan2.1 / Wan2.2, rectified_wan21_attn.py:423-426)*/
                            /* 3 = LayerNorm over head_dim with weight and bias (CogVideoX, cogvideo :452-455) */
  float eps;
  const void* q_weight;     /* DEVICE [head_dim] (norms 1, 3) or [heads*128] (norm 2), in the descriptor's      */
                            /* dtype: norm_q.weight                                                            */
  const void* k_weight;     /* likewise norm_k.weight                                                          */
  int32_t rope_rows;        /* source tokens [0, rope_rows) are rotated; 0 = no rotary embedding               */
  int32_t rope_compact;     /* 0: cos and sin are two tables.  1: `cos` is ONE table [rope_rows, head_dim/2] of */
                            /* (cos_i, sin_i) pairs and `sin` is ignored -- diffusers' tables repeat every value  */
                            /* for the two elements of a pair (repeat_interleave(2)), so this holds the same      */
                            /* numbers in half the bytes; the caller vouches for cos[2i] == cos[2i+1] and         */
                            /* sin[2i] == sin[2i+1] (rsa_b200/ops.py checks once per table).  Same arithmetic.    */
  const float* cos;         /* DEVICE fp32 [rope_rows, head_dim] (diffusers' repeat-interleaved cos table)     */
  const float* sin;
  float* row_scratch;       /* norm 2 only: DEVICE scratch of 2*batch*rows floats for the per-token statistics  */
  const void* q_bias;       /* norm 3 only: DEVICE [head_dim] in the descriptor's dtype (norm_q.bias)           */
  const void* k_bias;
} rsa_prep_desc;

int rsa_qkv_prep(const rsa_prep_desc* p, const rsa_attn_desc* d, const void* q_src, const void* k_src,
                 const void* v_src, void* q, void* k, void* v, int pool, void* workspace, size_t workspace_bytes,
                 void* stream);

/* Kernels 3a, 3b, 3c, 4 on pooled statistics that rsa_qkv_prep(pool = 1) has left in the workspace. */
int rsa_rectified_attention_pooled(const rsa_attn_desc* d, const void* q, const void* k, const void* v, void* out,
                                   void* workspace, size_t workspace_bytes, void* stream);

/* The whole call on HOST buffers: query/key/value/out are host pointers (page-locked memory gives the full PCIe rate;
 * pageable memory is correct but serialises), described by the same descriptor (strides = the host tensors').  Heads
 * are independent, so the call is cut into chunks of heads_per_chunk heads and pipelined on three streams: H2D of
 * chunk c+1 | kernels 2-4 of chunk c (on `stream`) | D2H of chunk c-1, over double-buffered staging carved from
 * device_scratch (rsa_host_call_scratch_bytes).  desc->nbr stays a DEVICE pointer.  Only enqueues work; the result is
 * complete when `stream` reaches the point of return.  The two copy streams and six events per device are created on
 * first use and kept (the only global state besides the error string).  Replaces, for a caller holding host tensors,
 * `q.cuda(); k.cuda(); v.cuda(); rectified_block_sparse_attention(...).cpu()` around hunyuan :393-417. */
size_t rsa_host_call_scratch_bytes(const rsa_attn_desc* d, int heads_per_chunk);
int rsa_rectified_attention_host(const rsa_attn_desc* d, const void* q, const void* k, const void* v, void* out,
                                 int heads_per_chunk, void* device_scratch, size_t scratch_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Peer memory (one process per GPU on one NVSwitch box).  rsa_peer_alloc returns zero-filled device memory that can
 * be exported to the other ranks (CUDA IPC): rsa_peer_export fills a 64-byte handle to send through any host channel
 * (torch.distributed.all_gather_object in rsa_b200/parallel.py), rsa_peer_open maps a received handle and returns a
 * device pointer valid in this process.  Used by the fused Ulysses exchange below; the reference has no counterpart
 * (it never splits one attention call over GPUs, SURVEY 8e). */
#define RSA_PEER_HANDLE_BYTES 64
#define RSA_MAX_PEERS 8
int rsa_peer_alloc(size_t bytes, void** ptr);
int rsa_peer_free(void* ptr);
int rsa_peer_export(const void* ptr, void* handle64);
int rsa_peer_open(const void* handle64, void** ptr);
int rsa_peer_close(void* ptr);

/* Fused Ulysses exchange (sequence-parallel host model; SURVEY 8e "fusion target", 8f rank 3).  Every rank owns
 * rows_per_rank consecutive tokens of all heads_total heads before the attention and must own the same tokens of the
 * result after it; in between, rank r computes heads [r*H, (r+1)*H) (H = desc->heads) over ALL tokens.  Instead of two
 * all-to-alls around the call,
 *   rsa_qkv_prep_gather      kernel 0 reads each token's projection rows straight from the owning rank's peer-mapped
 *                            buffer over NVLink (head split + norm + rotary embedding + re-layout + pooling as usual),
 *   rsa_rectified_attention_pooled_scatter   kernel 4's epilogue stores each output row straight into the owning
 *                            rank's result buffer.
 * The caller provides the barriers: every rank's sources written before the gather, every rank's scatter finished
 * before the results are read (a zero-byte collective on the stream; rsa_b200/parallel.py uses an all_reduce of one
 * element).  Rank i owns tokens [i * rows_per_rank, min((i + 1) * rows_per_rank, seq)): rows_per_rank = ceil(seq / n_ranks)
 * when the tokens do not divide (every rank must own at least one; all buffers are laid out for rows_per_rank rows).
 * This rank computes heads [head0, head0 + desc->heads) of the heads_total heads; the shards need not be even (12 heads
 * on 8 ranks: 2,2,2,2,1,1,1,1), every rank states its own first head and its own count.  Prep norm 0, 1, or 2 (2 needs
 * rinv_table) at head_dim 128; norm 3 (LayerNorm, CogVideoX) at head_dim 64.  A ragged visual segment (HunyuanVideo 129
 * frames, Flux 1360x768, CogVideoX 49 frames at 480x720) takes two gather calls like rsa_qkv_prep, at either head_dim:
 * the visual tokens (dst_row 0) and the text tokens (dst_row = visual token count); the source token of row r is
 * dst_row + r in both. */
typedef struct rsa_peer_route {
  int32_t n_ranks, rank;
  int32_t rows_per_rank;
  int32_t heads_total;          /* heads of the host model = channels / head_dim of the source and result rows     */
  int32_t head0;                /* this rank's first head: it computes heads [head0, head0 + desc->heads)          */
  int32_t reserved;             /* 0                                                                               */
  const void* const* src_table; /* DEVICE array [3][n_ranks] (q, k, v): every rank's projection output,           */
                                /* [batch, rows_per_rank, heads_total*head_dim] in the descriptor's dtype, as      */
                                /* mapped in THIS process                                                           */
  int64_t src_stride[2];        /* (batch, token) element strides of those buffers                                 */
  void* const* out_table;       /* DEVICE array [n_ranks]: every rank's result buffer [batch, rows_per_rank,       */
                                /* heads_total, head_dim] in the descriptor's dtype, as mapped in this process      */
  int64_t out_stride[2];        /* (batch, token) element strides of those buffers                                 */
  const float* const* rinv_table; /* prep norm 2 (Wan: RMSNorm over all heads_total*128 channels of a token) only:  */
                                /* DEVICE array [2][n_ranks] (q, k): every rank's per-token statistics              */
                                /* rsqrt(mean(x^2) + eps), [batch, rows_per_rank] fp32, which the OWNING rank computes */
                                /* from its full rows with rsa_row_rms before the barrier; NULL otherwise            */
} rsa_peer_route;

/* Per-token RMS statistic of the q and k projection rows over all `channels` (= heads_total * 128) channels:
 * rinv[b * rows + r] = rsqrt(mean(x[b, r, :]^2) + eps), the fp32 value diffusers' RMSNorm multiplies by (Wan's norm_q /
 * norm_k span all heads, rectified_wan21_attn.py:423-426).  rsa_qkv_prep (norm 2) runs this itself; under the fused
 * Ulysses exchange every rank runs it on the tokens it owns so that the gathering ranks need not see whole rows. */
int rsa_row_rms(const void* q_src, const void* k_src, int batch, int rows, int channels, const int64_t q_stride[2],
                const int64_t k_stride[2], float eps, float* rinv_q, float* rinv_k, void* stream);
/* The same for rows in `dtype` (enum rsa_dtype: bf16 or fp16; the statistic is fp32 either way).  rsa_row_rms reads bf16. */
int rsa_row_rms_dtype(const void* q_src, const void* k_src, int batch, int rows, int channels, const int64_t q_stride[2],
                      const int64_t k_stride[2], float eps, float* rinv_q, float* rinv_k, int dtype, void* stream);

int rsa_qkv_prep_gather(const rsa_prep_desc* p, const rsa_attn_desc* d, const rsa_peer_route* route, void* q, void* k,
                        void* v, int pool, void* workspace, size_t workspace_bytes, void* stream);
int rsa_rectified_attention_pooled_scatter(const rsa_attn_desc* d, const void* q, const void* k, const void* v,
                                           const rsa_peer_route* route, void* workspace, size_t workspace_bytes,
                                           void* stream);

/* The reference's Triton kernel rounds the pre-scaled query to the input dtype before Q.K^T (q = (q * sm_scale *
 * 1.44269504).to(dtype), rectified_wan21_attn.py:61-62); flash-attn, which the reference calls for text rows and for its
 * dense "flash" mode (attn.py:107-120), scales the fp32 scores instead.  Kernel 4 does the former on visual query tiles
 * and the latter on text tiles.  OR-ed into the `dtype` argument of rsa_masked_attention, this flag selects flash-attn's
 * arithmetic for the whole call (the dense mode of the mirror's fullattn). */
#define RSA_ATTN_FP32_SCALE 256

/* Kernel 4 alone on a caller-supplied dense block mask (bytes, [BH, n_q_blocks, n_kv_blocks]) -- the literal
 * surface of _triton_block_sparse_attention_onehot(q, k, v, seqlens, block_mask, sm_scale) (wan21 :108-117).
 * q/k/v/out are [BH, seq, head_dim] with the given token strides; R = 1, C = 0.  workspace must hold
 * rsa_masked_attention_workspace_bytes(). */
size_t rsa_masked_attention_workspace_bytes(int bh, int n_q_blocks, int n_kv_blocks);
int rsa_masked_attention(const void* q, const void* k, const void* v, void* out, int bh, int seq_q, int seq_kv,
                         int kv_len, const int64_t q_stride[2], const int64_t k_stride[2],
                         const int64_t v_stride[2], const int64_t o_stride[2], const uint8_t* block_mask,
                         int n_q_blocks, int n_kv_blocks, void* workspace, size_t workspace_bytes, void* stream,
                         int dtype /* enum rsa_dtype */, int head_dim /* 128 or 64 */);

/* Dense attention: kernel 4 walking every key block of every query tile, without lists, mask or workspace.  Replaces
 * fullattn(mode="flash") (attn.py:107-120, flash_attn_varlen_func) with the cu_seqlens the processors pass,
 * [0, q_valid, S] for the queries and [0, kv_len, S] for the keys: query rows >= q_valid are written as zeros, keys
 * >= kv_len are never attended.  Flash-attn's arithmetic (the fp32 scores are scaled; what RSA_ATTN_FP32_SCALE selects
 * in rsa_masked_attention), and the result is bit-identical to rsa_masked_attention on an all-ones mask with that flag
 * (rows >= q_valid zeroed): the walk is the pair schedule of all-ones lists in closed form.
 * Reads only batch, heads, seq (= query rows), head_dim (128 or 64), the four stride triples and dtype (bf16 or fp16)
 * of `d`; the block-geometry fields are neither read nor validated.  q is [batch, heads, seq, head_dim], k and v are
 * [batch, heads, seq_kv, head_dim] (seq_kv may differ from seq), out is [batch, heads, seq, head_dim], all through the
 * descriptor's strides (multiples of 8 elements, 16-byte aligned bases).  Needs 1 <= q_valid <= seq and
 * 1 <= kv_len <= seq_kv.  RSA_TC5_POLY and the debug dump do not apply to this form. */
int rsa_dense_attention(const rsa_attn_desc* d, const void* q, const void* k, const void* v, void* out, int seq_kv,
                        int q_valid, int kv_len, void* stream);
/* The same with the fused Ulysses scatter epilogue of rsa_rectified_attention_pooled_scatter: every output row is stored
 * into the owning rank's result buffer (route->out_table); seq_kv = seq (q, k, v come from rsa_qkv_prep_gather with
 * pool = 0).  The route is validated as there, and head_dim 64 is refused under the debug dump or attention flag 4. */
int rsa_dense_attention_scatter(const rsa_attn_desc* d, const void* q, const void* k, const void* v,
                                const rsa_peer_route* route, int q_valid, int kv_len, void* stream);

/* Bring-up hook (tests only): while non-null, the tcgen05 kernel's CTA for query tile 0 of batch*head 0 writes, as
 * fp32, S of its first kept block [128x128], the un-normalised O [128x128], the row sums l [128] and the row
 * maxima m [128] (log2 domain), then from offset 33024 a clock trace (64 steps x 16 slots, cycles since CTA start) to
 * this DEVICE buffer of >= 34048 floats. */
void rsa_debug_set_attention_dump(float* device_buffer);
/* Bring-up ablations, honoured only while a dump buffer is set: bit 0 = skip the softmax arithmetic (results are
 * garbage; measures the TMA + tensor pipeline alone), bit 1 = no K/V loads after the first ring fill.  Bit 2 is
 * honoured without a dump buffer: head_dim 64 runs through the 128-column instantiation (second granule = TMA zero
 * fill) instead of the 64-column one -- the cross-check and the A/B timing of the two forms; bit 4 likewise: kernel 4's
 * grid in its former order (head by head, no re-pairing of the tail) for A/B timing; bit 5 (32) likewise: kernel 4
 * launched without thread-block clusters and without the multicast prefix (the round-1 skeleton; the kept lists are then
 * walked in another order, so results agree within the output bar, not bit for bit), for A/B timing of the clusters.  The environment variable RSA_ATTN_FLAGS holds bits for the whole
 * process (OR-ed into whatever this call sets). */
void rsa_debug_set_attention_flags(int flags);
/* Host-side views of kernel 4's grid order (tests): the (batch*head, pair, tile0, tile1, repaired) CTA `id` of a launch
 * over n_bh heads works on, given the number of last heads whose text pairs go first -- the same inline function the
 * kernel calls -- and that number as the library computes it for a descriptor (-1: invalid descriptor). */
void rsa_debug_attention_grid_slot(int id, int n_q_tiles, int nq_vis, int n_bh, int front_heads, int former_order,
                                   int out[5]);
int rsa_debug_front_text_heads(const rsa_attn_desc* d);

#ifdef __cplusplus
}
#endif
#endif /* RSA_H_ */
