// rsa_common.cuh -- shared host/device helpers for librsa_b200.so (sm_100a only).
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "rsa.h"

namespace rsa {

void set_error(const char* fmt, ...);

#define RSA_FAIL(code, ...)       \
  do {                            \
    ::rsa::set_error(__VA_ARGS__);\
    return (code);                \
  } while (0)

#define RSA_CUDA_CHECK(expr)                                                            \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess) RSA_FAIL(RSA_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(_e)); \
  } while (0)

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Workspace carve-up shared by every stage (offsets in bytes from a 256-B aligned base).
struct WsLayout {
  int bh, nq, nb, nqt, a, nkc, score_ld, n_entries, ent_ld, mask_words, nogapr_ld;
  // transposed copies [bh][128][ldq | ldk] of q_pool, q_mad, k_cat, k_mad: what kernel 3a stages from (coalesced)
  size_t off_q_pool_t, off_q_mad_t, off_k_cat_t, off_k_mad_t;
  int ldq, ldk;
  size_t off_q_pool, off_q_mad, off_k_cat, off_k_mad, off_v_pool, off_scores, off_nogapr, off_probs, off_w,
      off_mask, off_kidx, off_kcnt, off_nneed, off_R, off_C, off_sched, off_pshared, off_qshared, total;
};

// Padded ("virtual") layout <-> memory rows.  Visual token t sits at row t in both; the last visual block is completed
// with `gap` zero rows that exist nowhere in memory; text token i is memory row vis_len + i and padded row
// nq_vis*128 + i.  WAN: everything is visual, gap = 0.
struct RowMap {
  int vis_len;  // visual tokens in memory
  int nq_vis;   // visual blocks = ceil(vis_len / 128)
  int gap;      // nq_vis*128 - vis_len for JOINT (0 when aligned); 0 for WAN (its ragged tail is the end of the tensor)
};
inline RowMap row_map(const rsa_attn_desc* d) {
  RowMap m;
  if (d->family == RSA_FAMILY_JOINT) {
    m.vis_len = d->vis_len > 0 ? d->vis_len : d->nq_blocks * RSA_BLOCK;
    if (m.vis_len > d->seq) m.vis_len = d->seq;
    m.nq_vis = (m.vis_len + RSA_BLOCK - 1) / RSA_BLOCK;
    m.gap = m.nq_vis * RSA_BLOCK - m.vis_len;
  } else {
    m.vis_len = d->seq;
    m.nq_vis = (d->seq + RSA_BLOCK - 1) / RSA_BLOCK;
    m.gap = 0;
  }
  return m;
}

float attention_rescale_threshold(bool f16);
// Kernel 4's 1-D grid: which pair of query tiles CTA `id` works on.
// Pairs of adjacent query tiles.  The pairs that hold the dense (text) tiles are several times longer than the others
// (C3b: 931 rounds against ~200, Flux: 516 against ~65).  The grid walks the heads in order, each head's text pairs first
// and then its visual pairs (K/V of one head stay L2-resident and are read from HBM once) -- except that the text pairs
// of the LAST front_text_heads heads are moved to the very start of the grid: where they stood, they ran on after
// everything else had finished (a text pair lasts as long as several heads' worth of visual pairs).
// Tiles of a pair: (2 pair, 2 pair + 1).  With an odd number of visual tiles and an even number of text tiles
// (HunyuanVideo 129 frames: 929 + 2) that rule would pair the last visual tile with a text tile and leave the other text
// tile alone -- two CTAs running a 931-block list mostly single-slot.  The tail is re-paired instead: the odd visual tile
// alone, the text tiles with each other (`repaired`: such tiles walk their original ascending lists, kept_idx, because
// the pair schedule was computed for the (2p, 2p+1) rule; text lists are all "every block with valid keys", so the whole
// list is common to both slots).  former_order (attention flag 16, A/B): head by head, no re-pairing.
struct GridSlot {
  int bh, pair, tile0, tile1;  // tile1 >= nqt: the pair has one tile
  bool repaired;
};
__host__ __device__ inline GridSlot attention_grid_slot(int id, int nqt, int nq_vis, int n_bh, int front_text_heads,
                                                        bool former_order) {
  GridSlot g;
  const int n_pairs = (nqt + 1) / 2;
  const int nqv = nq_vis < nqt ? nq_vis : nqt;  // visual tiles (rsa_masked_attention passes "all of them" as 2^20)
  const int vis_pairs = nqv / 2;                // pairs made of visual tiles only
  const int txt_pairs = n_pairs - vis_pairs;    // pairs with a text tile (or the odd last tile)
  int front = front_text_heads < 0 ? 0 : front_text_heads;
  if (front > n_bh) front = n_bh;
  if (former_order) front = 0;
  const int n_front = front * txt_pairs;
  const int n_inline = (n_bh - front) * n_pairs;
  if (id < n_front) {  // text pairs of the last `front` heads
    g.bh = n_bh - front + id / txt_pairs;
    g.pair = n_pairs - 1 - id % txt_pairs;
  } else if (id - n_front < n_inline) {  // the other heads: text pairs, then visual pairs
    id -= n_front;
    g.bh = id / n_pairs;
    g.pair = n_pairs - 1 - id % n_pairs;
  } else {  // visual pairs of the last `front` heads
    id -= n_front + n_inline;
    g.bh = n_bh - front + id / vis_pairs;
    g.pair = vis_pairs - 1 - id % vis_pairs;
  }
  const int n_txt_tiles = nqt - nqv;
  g.repaired = (nqv & 1) && n_txt_tiles >= 2 && !(n_txt_tiles & 1) && g.pair >= vis_pairs && !former_order;
  g.tile0 = 2 * g.pair;
  g.tile1 = 2 * g.pair + 1;
  if (g.repaired) {
    const int q = g.pair - vis_pairs;  // 0: the odd visual tile; q >= 1: text tiles (nq_vis + 2q - 2, nq_vis + 2q - 1)
    g.tile0 = q == 0 ? nqv - 1 : nqv + 2 * q - 2;
    g.tile1 = q == 0 ? nqt : g.tile0 + 1;
  }
  return g;
}

int validate_desc(const rsa_attn_desc* d);
WsLayout make_layout(const rsa_attn_desc* d);
int check_ws(const rsa_attn_desc* d, const void* ws, size_t bytes, WsLayout* out);

// stage launchers (defined in the .cu files)
int launch_pool_stats(const rsa_attn_desc* d, const void* q, const void* k, const void* v, char* ws,
                      const WsLayout& L, cudaStream_t s);
int launch_qkv_prep(const rsa_prep_desc* p, const rsa_attn_desc* d, const void* q_src, const void* k_src,
                    const void* v_src, const rsa_peer_route* route, void* q, void* k, void* v, char* ws,
                    const WsLayout* L, cudaStream_t s);
int launch_row_rms(const void* q_src, const void* k_src, int batch, int rows, int channels, const int64_t* qs,
                   const int64_t* ks, float eps, float* rq, float* rk, bool f16, cudaStream_t s);
int launch_block_scores(const rsa_attn_desc* d, char* ws, const WsLayout& L, cudaStream_t s);
int launch_block_select(const rsa_attn_desc* d, char* ws, const WsLayout& L, cudaStream_t s, bool keep_lists = false);
int launch_rect_c(const rsa_attn_desc* d, char* ws, const WsLayout& L, cudaStream_t s);

// Attention kernel arguments common to both implementations.  q/k/v/o are addressed as [bh][token][128].
struct AttnArgs {
  const __nv_bfloat16 *q, *k, *v;
  __nv_bfloat16* o;
  int batch, heads;         // bh = batch*heads; head index = bh % heads, batch index = bh / heads
  int64_t qs[3], ks[3], vs[3], os[3];  // element strides (batch, head, token)
  int seq_q;                // query rows that exist (rows >= seq_q are neither read nor written)
  int seq_kv;               // key rows that exist in memory
  int kv_len;               // keys >= kv_len masked to -inf
  int q_valid;              // query rows >= q_valid are written as zeros
  int vis_len, nq_vis, gap; // RowMap: blocks/tiles < nq_vis read memory rows [128 i, ..) bounded by vis_len, the others
                            // read memory rows vis_len + 128 (i - nq_vis); kv_len and q_valid are PADDED-layout rows
  int nqt;                  // query tiles per head
  int nb;                   // kv blocks per head (row length of kept_idx)
  const uint16_t* kept_idx; // [bh, nqt, nb]
  const int32_t* kept_cnt;  // [bh, nqt]
  uint16_t* sched_idx;      // [bh, nqt, nb]  pair schedule written by launch_pair_schedule, walked by kernel 4
  int32_t* pair_shared;     // [bh, ceil(nqt/2)]
  int32_t* quad_shared;     // [bh, ceil(nqt/2)]  blocks the partner pair of the 2-CTA cluster keeps too (lead the prefix)
  const float* R;           // [bh, nqt]  or nullptr (=1)
  const float* C;           // [bh, nqt, 128] or nullptr (=0)
  __nv_bfloat16* const* o_table;  // fused Ulysses scatter: result buffer of every rank (device array) or nullptr
  int peer_rows, peer_head0;      // tokens per rank; first head of this rank inside a token of the result buffers
  int64_t peer_os[2];             // (batch, token) element strides of the result buffers
  float scale_log2;         // head_dim^-0.5 * log2(e)
  int front_text_heads;     // kernel 4's grid: the text pairs of this many last heads are scheduled before everything else
  float rescale_thr;        // kernel 4: O and l are rescaled only when a row maximum grows by more than 2^rescale_thr
  int head_dim;             // 128 or 64: columns that exist in q/k/v/o (the rest of the 128-column tiles reads as zeros)
  int q_round;              // 1: visual query tiles use q~ = dtype(q * sm_scale * log2 e) like the reference's Triton kernel
                            // (wan21 :61-62); 0: S is scaled in fp32 everywhere (flash-attn's arithmetic, attn.py:107-120)
  int f16;                  // q/k/v/o hold fp16 instead of bf16 (the pointer types above are nominal: 2-byte elements)
  int dbg_flags;            // bring-up ablations (rsa_debug_set_attention_flags), only read by the debug kernel
  float* dbg;               // bring-up dump of tile 0 / bh 0 (rsa_debug_set_attention_dump), normally null
};

int launch_attention_mma(const AttnArgs& a, cudaStream_t s);      // mma.sync cross-check kernel: tests/xcheck only, not in the product library
// tcgen05 / TMEM / TMA kernel; dense = true: the list-free form (every tile walks blocks 0 .. ceil(kv_len/128) - 1;
// kept_idx, kept_cnt, sched_idx, pair_shared, quad_shared, R and C are not read)
int launch_attention_tc5(const AttnArgs& a, cudaStream_t s, bool dense = false);
int launch_pair_schedule(const AttnArgs& a, cudaStream_t s);  // kept lists -> sched_idx / pair_shared
int launch_mask_to_lists(const uint8_t* mask, int bh, int nq, int nkv, int kv_blocks_valid, uint16_t* kept_idx,
                         int32_t* kept_cnt, cudaStream_t s);

extern float* g_attention_dbg;
extern int g_attention_dbg_flags;

}  // namespace rsa
