// rsa_api.cu -- the C ABI of librsa_b200.so (declared in include/rsa.h): argument validation, workspace
// carve-up and stage sequencing.  No allocation, no host synchronisation, everything on the caller's stream.
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include "rsa_common.cuh"

namespace rsa {

static thread_local char g_err[512] = "";
float* g_attention_dbg = nullptr;
// RSA_ATTN_FLAGS: switches that stay set for the whole process (A/B runs of the test suite), OR-ed into whatever
// rsa_debug_set_attention_flags sets
static int env_attention_flags() {
  const char* e = getenv("RSA_ATTN_FLAGS");
  return e ? atoi(e) : 0;
}
static const int g_env_attention_flags = env_attention_flags();
int g_attention_dbg_flags = g_env_attention_flags;

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// Lazy rescale threshold of kernel 4 in log2 units: O and l are rescaled only when a row maximum grows by more than
// 2^thr, so P <= 2^thr and l, O <= S * 2^thr * max|v| -- far inside fp32 for thr = 32; P is bf16 (fp32's exponent range)
// or fp16, where it must stay below 2^16: 8 there.  C3b, same box: kernel 4 31.44 / 31.41 / 31.29 ms for 8 / 16 / 32.
float attention_rescale_threshold(bool f16) {
  static float v = -1.f;
  if (v < 0.f) {
    const char* e = getenv("RSA_TC5_THR");
    v = e ? (float)atof(e) : 32.f;
    if (!(v >= 0.f && v <= 64.f)) v = 32.f;
  }
  return f16 && v > 8.f ? 8.f : v;
}

int validate_desc(const rsa_attn_desc* d) {
  if (!d) RSA_FAIL(RSA_ERR_ARG, "descriptor is null");
  if (d->head_dim != RSA_HEAD_DIM && d->head_dim != 64)
    RSA_FAIL(RSA_ERR_UNSUPPORTED, "head_dim must be 128 or 64 (got %d); the reference asserts Lk in {16,32,64,128}", d->head_dim);
  if (d->batch <= 0 || d->heads <= 0 || d->seq <= 0) RSA_FAIL(RSA_ERR_ARG, "batch/heads/seq must be positive");
  if (d->dtype != RSA_DTYPE_BF16 && d->dtype != RSA_DTYPE_F16) RSA_FAIL(RSA_ERR_UNSUPPORTED, "dtype %d is not one of rsa_dtype (bf16, fp16)", d->dtype);
  if ((int64_t)d->batch * d->heads > 65535) RSA_FAIL(RSA_ERR_UNSUPPORTED, "batch*heads > 65535");
  if (d->family != RSA_FAMILY_WAN && d->family != RSA_FAMILY_JOINT) RSA_FAIL(RSA_ERR_ARG, "unknown family %d", d->family);
  if (d->vis_len < 0 || d->vis_len > d->seq) RSA_FAIL(RSA_ERR_ARG, "vis_len=%d out of [0, seq]", d->vis_len);
  const RowMap rm = row_map(d);
  const int nb = rm.nq_vis + (d->seq - rm.vis_len + RSA_BLOCK - 1) / RSA_BLOCK;
  if (d->n_blocks != nb)
    RSA_FAIL(RSA_ERR_ARG, "n_blocks=%d but the layout has %d (visual %d + text %d)", d->n_blocks, nb, rm.nq_vis, nb - rm.nq_vis);
  if (d->nq_blocks < 0 || d->nq_blocks > nb) RSA_FAIL(RSA_ERR_ARG, "nq_blocks=%d out of [0,%d]", d->nq_blocks, nb);
  const int seq_v = d->seq + rm.gap;  // length of the padded layout
  if (d->family == RSA_FAMILY_WAN) {
    if (d->nq_blocks != nb || d->text_keys != 0) RSA_FAIL(RSA_ERR_ARG, "WAN family needs nq_blocks == n_blocks and text_keys == 0");
    if (d->vis_len != 0 && d->vis_len != d->seq) RSA_FAIL(RSA_ERR_ARG, "WAN family: vis_len must be 0 or seq");
  } else {
    if (d->nq_blocks >= nb) RSA_FAIL(RSA_ERR_ARG, "JOINT family needs at least one text block");
    if (d->vis_len != 0 && d->nq_blocks != (d->vis_len + RSA_BLOCK - 1) / RSA_BLOCK)
      RSA_FAIL(RSA_ERR_ARG, "nq_blocks=%d but ceil(vis_len/128)=%d", d->nq_blocks, (d->vis_len + RSA_BLOCK - 1) / RSA_BLOCK);
    if (d->text_keys < 1 || d->text_keys > d->seq - rm.vis_len)
      RSA_FAIL(RSA_ERR_ARG, "text_keys=%d must be in [1, seq - vis_len]", d->text_keys);
  }
  const int n_ent = d->nq_blocks + (d->family == RSA_FAMILY_JOINT ? 1 : 0);
  if (n_ent > RSA_MAX_ENTRIES) RSA_FAIL(RSA_ERR_UNSUPPORTED, "more than %d sortable blocks per row", RSA_MAX_ENTRIES);
  // kernel 3b keeps a row's kept-block bitmask in shared memory: RSA_MAX_ENTRIES / 32 + 1 words (block_select.cu)
  if ((nb + 31) / 32 > RSA_MAX_ENTRIES / 32 + 1)
    RSA_FAIL(RSA_ERR_UNSUPPORTED, "more than %d KV blocks (visual + text)", (RSA_MAX_ENTRIES / 32 + 1) * 32);
  if (d->kv_len < 1 || d->kv_len > seq_v) RSA_FAIL(RSA_ERR_ARG, "kv_len=%d out of [1, %d]", d->kv_len, seq_v);
  if (d->kv_zero_from < 0) RSA_FAIL(RSA_ERR_ARG, "kv_zero_from < 0");
  if (d->text_end_block < d->nq_blocks || d->text_end_block > nb) RSA_FAIL(RSA_ERR_ARG, "text_end_block out of range");
  if (d->top_k < 0 || d->first_frame_blocks < 0) RSA_FAIL(RSA_ERR_ARG, "top_k / first_frame_blocks negative");
  if (!(d->p_remain >= 0.f)) RSA_FAIL(RSA_ERR_ARG, "p_remain must be >= 0");
  if (d->text_q_valid < 0 ||
      (d->family == RSA_FAMILY_JOINT && d->text_q_valid > d->seq - rm.vis_len))
    RSA_FAIL(RSA_ERR_ARG, "text_q_valid out of range");
  if ((d->nbr_rows > 0) != (d->nbr_cols > 0) || (d->nbr_rows > 0 && !d->nbr)) RSA_FAIL(RSA_ERR_ARG, "neighbour matrix inconsistent");
  const int64_t* st[4] = {d->q_stride, d->k_stride, d->v_stride, d->o_stride};
  for (int t = 0; t < 4; ++t)
    for (int i = 0; i < 3; ++i)
      if (st[t][i] < 0 || st[t][i] % 8) RSA_FAIL(RSA_ERR_UNSUPPORTED, "strides must be non-negative multiples of 8 elements (16 bytes)");
  return RSA_OK;
}

WsLayout make_layout(const rsa_attn_desc* d) {
  WsLayout L;
  L.bh = d->batch * d->heads;
  L.nq = d->nq_blocks;
  L.nb = d->n_blocks;
  L.nqt = d->n_blocks;  // every 128-row query tile (visual + text) gets a list
  L.a = d->text_keys;
  L.nkc = L.nq + L.a;
  L.score_ld = (int)align_up(L.nkc, 4);
  L.n_entries = L.nq + (d->family == RSA_FAMILY_JOINT ? 1 : 0);
  L.ent_ld = (int)align_up(L.n_entries, 4);
  L.mask_words = (L.nb + 31) / 32;
  L.nogapr_ld = (int)align_up(L.nq > 0 ? L.nq : 1, 4);
  size_t o = 0;
  auto take = [&](size_t bytes) {
    size_t at = o;
    o = align_up(o + bytes, 256);
    return at;
  };
  const size_t f = sizeof(float);
  L.off_q_pool = take((size_t)L.bh * L.nq * 128 * f);
  L.off_q_mad = take((size_t)L.bh * L.nq * 128 * f);
  L.off_k_cat = take((size_t)L.bh * L.nkc * 128 * f);
  L.off_k_mad = take((size_t)L.bh * L.nq * 128 * f);
  L.off_v_pool = take((size_t)L.bh * L.nb * 128 * f);
  L.off_scores = take((size_t)L.bh * L.nq * L.score_ld * f);
  L.off_nogapr = take((size_t)L.bh * L.nq * L.nogapr_ld);
  L.off_probs = take(d->debug_dump_probs ? (size_t)L.bh * L.nq * L.ent_ld * f : 0);
  L.off_w = take((size_t)L.bh * L.nq * L.ent_ld * f);
  L.off_mask = take((size_t)L.bh * L.nqt * L.mask_words * 4);
  L.off_kidx = take((size_t)L.bh * L.nqt * L.nb * 2);
  L.off_kcnt = take((size_t)L.bh * L.nqt * 4);
  L.off_nneed = take((size_t)L.bh * (L.nq > 0 ? L.nq : 1) * 4);
  L.off_R = take((size_t)L.bh * L.nqt * f);
  L.off_C = take((size_t)L.bh * L.nqt * 128 * f);
  L.off_sched = take((size_t)L.bh * L.nqt * L.nb * 2);
  L.off_pshared = take((size_t)L.bh * ((L.nqt + 1) / 2) * 4);
  L.off_qshared = take((size_t)L.bh * ((L.nqt + 1) / 2) * 4);
  L.ldq = (int)align_up(L.nq > 0 ? L.nq : 1, 4);
  L.ldk = (int)align_up(L.nkc > 0 ? L.nkc : 1, 4);
  L.off_q_pool_t = take((size_t)L.bh * 128 * L.ldq * f);
  L.off_q_mad_t = take((size_t)L.bh * 128 * L.ldq * f);
  L.off_k_cat_t = take((size_t)L.bh * 128 * L.ldk * f);
  L.off_k_mad_t = take((size_t)L.bh * 128 * L.ldq * f);
  L.total = o;
  return L;
}

int check_ws(const rsa_attn_desc* d, const void* ws, size_t bytes, WsLayout* out) {
  int rc = validate_desc(d);
  if (rc != RSA_OK) return rc;
  *out = make_layout(d);
  if (!ws) RSA_FAIL(RSA_ERR_WORKSPACE, "workspace is null");
  if ((uintptr_t)ws % 256) RSA_FAIL(RSA_ERR_WORKSPACE, "workspace must be 256-byte aligned");
  if (bytes < out->total) RSA_FAIL(RSA_ERR_WORKSPACE, "workspace too small: %zu < %zu", bytes, out->total);
  return RSA_OK;
}

// Kernel 4's grid (attention_grid_slot): how many of the last heads have their text pairs moved to the front.  A text
// pair walks all n_blocks blocks; one head's visual pairs take about vis_pairs * kept / SMs rounds per SM, with
// kept >= top_k.  The text pairs of the heads whose batch would start less than one text pair before the end go first.
static int front_text_heads(const WsLayout& L, int top_k) {
  if (L.nq < 2) return L.bh;    // no visual pairs at all: every pair is in the front set
  if (L.nqt <= L.nq) return 0;  // no text tiles
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) {
      (void)cudaGetLastError();
      sms = 148;
    }
  }
  const double per_head = (double)(L.nq / 2) * (double)(top_k > 0 ? top_k : 1) / (double)sms;
  const double f = (double)L.nb / per_head;
  return f >= (double)L.bh ? L.bh : ((int)f + 2 > L.bh ? L.bh : (int)f + 2);
}

static int fill_attn_args(const rsa_attn_desc* d, const void* q, const void* k, const void* v, void* out, char* ws,
                          const WsLayout& L, AttnArgs* a) {
  a->q = (const __nv_bfloat16*)q;
  a->k = (const __nv_bfloat16*)k;
  a->v = (const __nv_bfloat16*)v;
  a->o = (__nv_bfloat16*)out;
  a->batch = d->batch;
  a->heads = d->heads;
  for (int i = 0; i < 3; ++i) {
    a->qs[i] = d->q_stride[i];
    a->ks[i] = d->k_stride[i];
    a->vs[i] = d->v_stride[i];
    a->os[i] = d->o_stride[i];
  }
  a->seq_q = d->seq;
  a->seq_kv = d->seq;
  a->kv_len = d->kv_len;
  const RowMap rm = row_map(d);
  a->vis_len = rm.vis_len;
  a->nq_vis = rm.nq_vis;
  a->gap = rm.gap;
  a->q_valid = d->family == RSA_FAMILY_JOINT ? d->nq_blocks * RSA_BLOCK + d->text_q_valid : d->seq;
  if (a->q_valid > d->seq + rm.gap) a->q_valid = d->seq + rm.gap;
  a->nqt = L.nqt;
  a->nb = L.nb;
  a->kept_idx = (const uint16_t*)(ws + L.off_kidx);
  a->kept_cnt = (const int32_t*)(ws + L.off_kcnt);
  a->sched_idx = (uint16_t*)(ws + L.off_sched);
  a->pair_shared = (int32_t*)(ws + L.off_pshared);
  a->quad_shared = (int32_t*)(ws + L.off_qshared);
  a->R = (const float*)(ws + L.off_R);
  a->C = (const float*)(ws + L.off_C);
  a->o_table = nullptr;
  a->peer_rows = a->peer_head0 = 0;
  a->peer_os[0] = a->peer_os[1] = 0;
  a->scale_log2 = (float)((1.0 / sqrt((double)d->head_dim)) * 1.44269504);  // the reference's qk_scale (wan21 :145)
  a->head_dim = d->head_dim;
  a->rescale_thr = attention_rescale_threshold(d->dtype == RSA_DTYPE_F16);
  a->front_text_heads = front_text_heads(L, d->top_k);
  a->f16 = d->dtype == RSA_DTYPE_F16;
  a->q_round = 1;
  a->dbg = g_attention_dbg;
  a->dbg_flags = g_attention_dbg_flags;
  return RSA_OK;
}

// reschedule = false: the kept lists have not changed since the last launch on this workspace, so neither has the
// pair schedule kernel 4 walks (mask re-use)
static int launch_attention(const AttnArgs& a, cudaStream_t s, bool reschedule = true) {
  int rc = reschedule ? launch_pair_schedule(a, s) : RSA_OK;
  return rc != RSA_OK ? rc : launch_attention_tc5(a, s);
}

// Schedule for kernel 4.  One CTA of kernel 4 works on a pair of query tiles (2p, 2p+1) of a head; pairs p and p ^ 1 --
// four adjacent tiles -- are PARTNERS when both consist of whole visual tiles.  Attention over a set of kept blocks does
// not depend on the order they are visited in, so each tile's list is re-ordered as
//   [blocks all FOUR tiles of the two partner pairs keep, ascending]   quad_shared counts them: where kernel 4's grid puts
//                                                 the partners into one 2-CTA cluster, one K / V tile is fetched per
//                                                 cluster (each CTA loads one 64-column granule and multicasts it)
//   [other blocks both tiles of the pair keep, ascending]    one K / V tile per CTA serves both of its tiles (pair_shared
//                                                 counts these and the quad blocks)
//   [the rest, ascending].
// The order depends on the head's own lists only -- not on how many heads a call holds or where kernel 4's grid puts the
// pair -- so a head's result is bit-identical however the heads are split over calls, chunks or GPUs.
__global__ void __launch_bounds__(128) pair_schedule_kernel(const uint16_t* __restrict__ kept_idx,
                                                            const int32_t* __restrict__ kept_cnt, int nqt, int nb,
                                                            int vis_pairs, int quads_off, uint16_t* __restrict__ sched_idx,
                                                            int32_t* __restrict__ pair_shared,
                                                            int32_t* __restrict__ quad_shared) {
  __shared__ uint32_t bm[4][2048];  // one bit per KV block (nb <= 65535): own tiles 0, 1; partner tiles 2, 3
  __shared__ int warp_tot[3][4];
  __shared__ int n_common[2];
  const int pair = blockIdx.x, bh = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int npairs = (nqt + 1) / 2;
  const bool partner = !quads_off && pair < vis_pairs && (pair ^ 1) < vis_pairs;
  const int64_t row0 = (int64_t)bh * nqt + 2 * pair;
  const bool has1 = 2 * pair + 1 < nqt;
  const int64_t prow0 = (int64_t)bh * nqt + 2 * (pair ^ 1);
  const int cnt[4] = {kept_cnt[row0], has1 ? kept_cnt[row0 + 1] : 0, partner ? kept_cnt[prow0] : 0,
                      partner ? kept_cnt[prow0 + 1] : 0};
  const int words = (nb + 31) / 32;
  for (int w = tid; w < words; w += 128) bm[0][w] = bm[1][w] = bm[2][w] = bm[3][w] = 0u;
  if (tid < 2) n_common[tid] = 0;
  __syncthreads();
  for (int t = 0; t < 4; ++t) {
    const uint16_t* src = kept_idx + ((t < 2 ? row0 : prow0) + (t & 1)) * nb;
    for (int i = tid; i < cnt[t]; i += 128) {
      const int x = src[i];
      atomicOr(&bm[t][x >> 5], 1u << (x & 31));
    }
  }
  __syncthreads();
  int c2 = 0, c4 = 0;
  for (int w = tid; w < words; w += 128) {
    const uint32_t m2 = bm[0][w] & bm[1][w];
    c2 += __popc(m2);
    c4 += __popc(m2 & bm[2][w] & bm[3][w]);
  }
  for (int o = 16; o > 0; o >>= 1) {
    c2 += __shfl_xor_sync(0xffffffffu, c2, o);
    c4 += __shfl_xor_sync(0xffffffffu, c4, o);
  }
  if (lane == 0) {
    if (c2) atomicAdd(&n_common[0], c2);
    if (c4) atomicAdd(&n_common[1], c4);
  }
  __syncthreads();
  const int ncom = n_common[0], nquad = partner ? n_common[1] : 0;
  if (tid == 0) {
    pair_shared[(int64_t)bh * npairs + pair] = ncom;
    quad_shared[(int64_t)bh * npairs + pair] = nquad;
  }
  for (int t = 0; t < 2; ++t) {
    const uint16_t* src = kept_idx + (row0 + t) * nb;
    uint16_t* dst = sched_idx + (row0 + t) * nb;
    int base[3] = {0, nquad, ncom};  // next output slot of: quad blocks, other pair-common blocks, the rest
    for (int i0 = 0; i0 < cnt[t]; i0 += 128) {
      const int i = i0 + tid;
      const bool ok = i < cnt[t];
      const int x = ok ? (int)src[i] : 0;
      const uint32_t bit = 1u << (x & 31);
      const bool com = ok && (bm[t ^ 1][x >> 5] & bit);
      const bool quad = com && partner && (bm[2][x >> 5] & bm[3][x >> 5] & bit);
      const int cls = !ok ? -1 : (quad ? 0 : (com ? 1 : 2));
      uint32_t bal[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) bal[c] = __ballot_sync(0xffffffffu, cls == c);
      if (lane == 0) {
#pragma unroll
        for (int c = 0; c < 3; ++c) warp_tot[c][warp] = __popc(bal[c]);
      }
      __syncthreads();
      const uint32_t below = (1u << lane) - 1u;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        int before = 0, tot = 0;
        for (int w = 0; w < 4; ++w) {
          if (w < warp) before += warp_tot[c][w];
          tot += warp_tot[c][w];
        }
        if (cls == c) dst[base[c] + before + __popc(bal[c] & below)] = (uint16_t)x;
        base[c] += tot;
      }
      __syncthreads();
    }
  }
}

int launch_pair_schedule(const AttnArgs& a, cudaStream_t s) {
  if (a.nqt == 0) return RSA_OK;
  const int nqv = a.nq_vis < a.nqt ? a.nq_vis : a.nqt;
  // attention flag 32 (A/B): no quad prefix at all, i.e. the schedule and the kernel of round 1
  const int quads_off = (a.dbg_flags & 32) ? 1 : 0;
  dim3 grid((a.nqt + 1) / 2, a.batch * a.heads);
  pair_schedule_kernel<<<grid, 128, 0, s>>>(a.kept_idx, a.kept_cnt, a.nqt, a.nb, nqv / 2, quads_off, a.sched_idx,
                                            a.pair_shared, a.quad_shared);
  RSA_CUDA_CHECK(cudaGetLastError());
  return RSA_OK;
}

// dense byte mask [bh, nq, nkv] -> ascending u16 lists (one warp per row)
__global__ void mask_to_lists_kernel(const uint8_t* __restrict__ mask, int rows, int nkv, int kv_blocks_valid,
                                     uint16_t* __restrict__ kept_idx, int32_t* __restrict__ kept_cnt) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const uint8_t* m = mask + (int64_t)row * nkv;
  uint16_t* out = kept_idx + (int64_t)row * nkv;
  int base = 0;
  for (int j0 = 0; j0 < nkv; j0 += 32) {
    const int j = j0 + lane;
    const bool on = j < nkv && j < kv_blocks_valid && m[j] != 0;
    const uint32_t bal = __ballot_sync(0xffffffffu, on);
    if (on) out[base + __popc(bal & ((1u << lane) - 1u))] = (uint16_t)j;
    base += __popc(bal);
  }
  if (lane == 0) kept_cnt[row] = base;
}

int launch_mask_to_lists(const uint8_t* mask, int bh, int nq, int nkv, int kv_blocks_valid, uint16_t* kept_idx,
                         int32_t* kept_cnt, cudaStream_t s) {
  const int rows = bh * nq;
  if (rows == 0) return RSA_OK;
  mask_to_lists_kernel<<<(rows + 7) / 8, 256, 0, s>>>(mask, rows, nkv, kv_blocks_valid, kept_idx, kept_cnt);
  RSA_CUDA_CHECK(cudaGetLastError());
  return RSA_OK;
}

}  // namespace rsa

using namespace rsa;

extern "C" const char* rsa_last_error_string(void) { return g_err; }
extern "C" int rsa_version(void) { return RSA_VERSION; }
extern "C" size_t rsa_attn_desc_size(void) { return sizeof(rsa_attn_desc); }
extern "C" size_t rsa_prep_desc_size(void) { return sizeof(rsa_prep_desc); }
extern "C" size_t rsa_peer_route_size(void) { return sizeof(rsa_peer_route); }

extern "C" int rsa_device_ok(void) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  cudaDeviceProp p;
  if (cudaGetDeviceProperties(&p, dev) != cudaSuccess) return 0;
  return p.major == 10 ? 1 : 0;
}

extern "C" void rsa_debug_set_attention_dump(float* device_buffer) { g_attention_dbg = device_buffer; }
extern "C" void rsa_debug_attention_grid_slot(int id, int n_q_tiles, int nq_vis, int n_bh, int front_heads,
                                              int former_order, int out[5]) {
  const GridSlot g = attention_grid_slot(id, n_q_tiles, nq_vis, n_bh, front_heads, former_order != 0);
  out[0] = g.bh, out[1] = g.pair, out[2] = g.tile0, out[3] = g.tile1, out[4] = g.repaired ? 1 : 0;
}
extern "C" int rsa_debug_front_text_heads(const rsa_attn_desc* d) {
  if (validate_desc(d) != RSA_OK) return -1;
  return front_text_heads(make_layout(d), d->top_k);
}
extern "C" void rsa_debug_set_attention_flags(int flags) { g_attention_dbg_flags = flags | g_env_attention_flags; }

extern "C" size_t rsa_attn_workspace_bytes(const rsa_attn_desc* d) {
  if (validate_desc(d) != RSA_OK) return 0;
  return make_layout(d).total;
}

extern "C" int rsa_attn_workspace_view(const rsa_attn_desc* d, void* workspace, size_t bytes, rsa_ws_view* out) {
  WsLayout L;
  int rc = check_ws(d, workspace, bytes, &L);
  if (rc != RSA_OK) return rc;
  if (!out) RSA_FAIL(RSA_ERR_ARG, "view pointer is null");
  char* ws = (char*)workspace;
  out->q_pool = (float*)(ws + L.off_q_pool);
  out->q_mad = (float*)(ws + L.off_q_mad);
  out->k_cat = (float*)(ws + L.off_k_cat);
  out->k_mad = (float*)(ws + L.off_k_mad);
  out->v_pool = (float*)(ws + L.off_v_pool);
  out->scores = (float*)(ws + L.off_scores);
  out->nogapr = (uint8_t*)(ws + L.off_nogapr);
  out->probs = d->debug_dump_probs ? (float*)(ws + L.off_probs) : nullptr;
  out->w_skip = (float*)(ws + L.off_w);
  out->mask_bits = (uint32_t*)(ws + L.off_mask);
  out->kept_idx = (uint16_t*)(ws + L.off_kidx);
  out->kept_cnt = (int32_t*)(ws + L.off_kcnt);
  out->n_needed = (int32_t*)(ws + L.off_nneed);
  out->R = (float*)(ws + L.off_R);
  out->C = (float*)(ws + L.off_C);
  out->nkc = L.nkc;
  out->score_ld = L.score_ld;
  out->n_entries = L.n_entries;
  out->ent_ld = L.ent_ld;
  out->mask_words = L.mask_words;
  out->nqt = L.nqt;
  out->nogapr_ld = L.nogapr_ld;
  out->reserved = 0;
  out->sched_idx = (uint16_t*)(ws + L.off_sched);
  out->pair_shared = (int32_t*)(ws + L.off_pshared);
  out->quad_shared = (int32_t*)(ws + L.off_qshared);
  return RSA_OK;
}

extern "C" int rsa_pool_stats(const rsa_attn_desc* d, const void* q, const void* k, const void* v, void* workspace,
                              size_t bytes, void* stream) {
  WsLayout L;
  int rc = check_ws(d, workspace, bytes, &L);
  if (rc != RSA_OK) return rc;
  if (!q || !k || !v) RSA_FAIL(RSA_ERR_ARG, "rsa_pool_stats: null tensor");
  return launch_pool_stats(d, q, k, v, (char*)workspace, L, (cudaStream_t)stream);
}

extern "C" int rsa_block_scores(const rsa_attn_desc* d, void* workspace, size_t bytes, void* stream) {
  WsLayout L;
  int rc = check_ws(d, workspace, bytes, &L);
  if (rc != RSA_OK) return rc;
  return launch_block_scores(d, (char*)workspace, L, (cudaStream_t)stream);
}

extern "C" int rsa_block_select(const rsa_attn_desc* d, void* workspace, size_t bytes, void* stream) {
  WsLayout L;
  int rc = check_ws(d, workspace, bytes, &L);
  if (rc != RSA_OK) return rc;
  return launch_block_select(d, (char*)workspace, L, (cudaStream_t)stream);
}

extern "C" int rsa_rect_c(const rsa_attn_desc* d, void* workspace, size_t bytes, void* stream) {
  WsLayout L;
  int rc = check_ws(d, workspace, bytes, &L);
  if (rc != RSA_OK) return rc;
  return launch_rect_c(d, (char*)workspace, L, (cudaStream_t)stream);
}

extern "C" int rsa_sparse_attention(const rsa_attn_desc* d, const void* q, const void* k, const void* v, void* out,
                                    void* workspace, size_t bytes, void* stream) {
  WsLayout L;
  int rc = check_ws(d, workspace, bytes, &L);
  if (rc != RSA_OK) return rc;
  if (!q || !k || !v || !out) RSA_FAIL(RSA_ERR_ARG, "rsa_sparse_attention: null tensor");
  AttnArgs a;
  fill_attn_args(d, q, k, v, out, (char*)workspace, L, &a);
  return launch_attention(a, (cudaStream_t)stream);
}

extern "C" int rsa_rectified_attention(const rsa_attn_desc* d, const void* q, const void* k, const void* v, void* out,
                                       void* workspace, size_t bytes, void* stream) {
  WsLayout L;
  int rc = check_ws(d, workspace, bytes, &L);
  if (rc != RSA_OK) return rc;
  if (!q || !k || !v || !out) RSA_FAIL(RSA_ERR_ARG, "rsa_rectified_attention: null tensor");
  char* ws = (char*)workspace;
  cudaStream_t s = (cudaStream_t)stream;
  if ((rc = launch_pool_stats(d, q, k, v, ws, L, s)) != RSA_OK) return rc;
  if ((rc = launch_block_scores(d, ws, L, s)) != RSA_OK) return rc;
  if ((rc = launch_block_select(d, ws, L, s)) != RSA_OK) return rc;
  if ((rc = launch_rect_c(d, ws, L, s)) != RSA_OK) return rc;
  AttnArgs a;
  fill_attn_args(d, q, k, v, out, ws, L, &a);
  return launch_attention(a, s);
}

extern "C" int rsa_qkv_prep(const rsa_prep_desc* p, const rsa_attn_desc* d, const void* q_src, const void* k_src,
                            const void* v_src, void* q, void* k, void* v, int pool, void* workspace, size_t bytes,
                            void* stream) {
  int rc = validate_desc(d);
  if (rc != RSA_OK) return rc;
  if (!p) RSA_FAIL(RSA_ERR_ARG, "rsa_qkv_prep: descriptor is null");
  // diffusers' rounding points in the descriptor's dtype: bf16 or fp16 (validate_desc has refused any other)
  if (d->dtype != RSA_DTYPE_BF16 && d->dtype != RSA_DTYPE_F16)
    RSA_FAIL(RSA_ERR_UNSUPPORTED, "rsa_qkv_prep: dtype %d is not bf16 or fp16", d->dtype);
  if (d->head_dim != RSA_HEAD_DIM && d->head_dim != 64) RSA_FAIL(RSA_ERR_UNSUPPORTED, "rsa_qkv_prep: head_dim must be 128 or 64 (got %d)", d->head_dim);
  if (d->head_dim == 64 && p->norm != 3)
    RSA_FAIL(RSA_ERR_UNSUPPORTED, "rsa_qkv_prep: head_dim 64 is built for norm 3 (LayerNorm, CogVideoX) only, not norm %d", p->norm);
  if (!q_src || !k_src || !v_src || !q || !k || !v) RSA_FAIL(RSA_ERR_ARG, "rsa_qkv_prep: null tensor");
  const RowMap rm = row_map(d);
  if (p->rows < 1) RSA_FAIL(RSA_ERR_ARG, "rsa_qkv_prep: rows must be positive");
  if (p->dst_row != 0 && !(d->family == RSA_FAMILY_JOINT && p->dst_row == rm.vis_len))
    RSA_FAIL(RSA_ERR_ARG, "rsa_qkv_prep: dst_row must be 0 or the visual token count (%d)", rm.vis_len);
  const int room = p->dst_row == 0 ? (d->family == RSA_FAMILY_JOINT && pool ? rm.vis_len : d->seq) : d->seq - rm.vis_len;
  if (p->rows > d->seq - p->dst_row) RSA_FAIL(RSA_ERR_ARG, "rsa_qkv_prep: %d rows do not fit behind row %d of %d", p->rows, p->dst_row, d->seq);
  if (pool && p->rows != room && !(p->dst_row == 0 && p->rows == d->seq && rm.gap == 0))
    RSA_FAIL(RSA_ERR_ARG, "rsa_qkv_prep: pooling needs whole segments (%d rows here, segment has %d)", p->rows, room);
  if (p->norm < 0 || p->norm > 3) RSA_FAIL(RSA_ERR_UNSUPPORTED, "rsa_qkv_prep: norm must be 0, 1 (RMSNorm over head_dim), 2 (across heads) or 3 (LayerNorm)");
  if (p->norm == 3 && (!p->q_bias || !p->k_bias || (uintptr_t)p->q_bias % 16 || (uintptr_t)p->k_bias % 16))
    RSA_FAIL(RSA_ERR_ARG, "rsa_qkv_prep: norm 3 needs 16-byte aligned biases");
  if (p->norm == 2 && (!p->row_scratch || (uintptr_t)p->row_scratch % 4)) RSA_FAIL(RSA_ERR_ARG, "rsa_qkv_prep: norm 2 needs row_scratch (2*batch*rows floats)");
  if (p->norm && (!p->q_weight || !p->k_weight)) RSA_FAIL(RSA_ERR_ARG, "rsa_qkv_prep: norm weights are null");
  if (p->rope_rows < 0 || p->rope_rows > p->rows) RSA_FAIL(RSA_ERR_ARG, "rsa_qkv_prep: rope_rows out of range");
  if (p->rope_rows > 0 && (!p->cos || (!p->sin && !p->rope_compact))) RSA_FAIL(RSA_ERR_ARG, "rsa_qkv_prep: rotary tables are null");
  for (int t = 0; t < 3; ++t)
    for (int i = 0; i < 2; ++i)
      if (p->src_stride[t][i] < 0 || p->src_stride[t][i] % 8) RSA_FAIL(RSA_ERR_UNSUPPORTED, "rsa_qkv_prep: source strides must be multiples of 8 elements");
  const void* ptrs[8] = {q_src, k_src, v_src, q, k, v, p->q_weight, p->k_weight};
  for (int i = 0; i < 8; ++i)
    if ((uintptr_t)ptrs[i] % 16) RSA_FAIL(RSA_ERR_UNSUPPORTED, "rsa_qkv_prep: tensors must be 16-byte aligned");
  if (p->rope_rows > 0 && (((uintptr_t)p->cos % 16) || (!p->rope_compact && (uintptr_t)p->sin % 16))) RSA_FAIL(RSA_ERR_UNSUPPORTED, "rsa_qkv_prep: rotary tables must be 16-byte aligned");
  WsLayout L;
  if (pool && (rc = check_ws(d, workspace, bytes, &L)) != RSA_OK) return rc;
  return launch_qkv_prep(p, d, q_src, k_src, v_src, nullptr, q, k, v, (char*)workspace, pool ? &L : nullptr,
                         (cudaStream_t)stream);
}

static int validate_route(const rsa_attn_desc* d, const rsa_peer_route* r, bool need_src, bool need_out) {
  if (!r) RSA_FAIL(RSA_ERR_ARG, "peer route is null");
  if (r->n_ranks < 1 || r->n_ranks > RSA_MAX_PEERS || r->rank < 0 || r->rank >= r->n_ranks)
    RSA_FAIL(RSA_ERR_ARG, "peer route: rank %d of %d", r->rank, r->n_ranks);
  // rank i owns tokens [i * rows_per_rank, min((i + 1) * rows_per_rank, seq)): every rank at least one, the last one possibly fewer
  if (r->rows_per_rank < 1 || (int64_t)r->rows_per_rank * r->n_ranks < d->seq ||
      (int64_t)r->rows_per_rank * (r->n_ranks - 1) >= d->seq)
    RSA_FAIL(RSA_ERR_ARG, "peer route: %d ranks x %d rows do not tile seq %d (every rank must own a token)", r->n_ranks,
             r->rows_per_rank, d->seq);
  if (r->head0 < 0 || d->heads < 1 || r->head0 + d->heads > r->heads_total)
    RSA_FAIL(RSA_ERR_ARG, "peer route: heads [%d, %d) outside the %d heads of a row", r->head0, r->head0 + d->heads, r->heads_total);
  const int64_t row = (int64_t)r->heads_total * d->head_dim;  // channels of a source / result row
  if (need_src && (!r->src_table || r->src_stride[0] < 0 || r->src_stride[1] < row || r->src_stride[0] % 8 || r->src_stride[1] % 8))
    RSA_FAIL(RSA_ERR_ARG, "peer route: source table / strides");
  if (need_out && (!r->out_table || r->out_stride[0] < 0 || r->out_stride[1] < row || r->out_stride[0] % 8 || r->out_stride[1] % 8))
    RSA_FAIL(RSA_ERR_ARG, "peer route: result table / strides");
  return RSA_OK;
}

extern "C" int rsa_qkv_prep_gather(const rsa_prep_desc* p, const rsa_attn_desc* d, const rsa_peer_route* route,
                                   void* q, void* k, void* v, int pool, void* workspace, size_t bytes, void* stream) {
  int rc = validate_desc(d);
  if (rc != RSA_OK) return rc;
  if ((rc = validate_route(d, route, true, false)) != RSA_OK) return rc;
  if (!p || !q || !k || !v) RSA_FAIL(RSA_ERR_ARG, "rsa_qkv_prep_gather: null pointer");
  if (d->dtype != RSA_DTYPE_BF16 && d->dtype != RSA_DTYPE_F16)
    RSA_FAIL(RSA_ERR_UNSUPPORTED, "rsa_qkv_prep_gather: dtype %d is not bf16 or fp16", d->dtype);
  if (d->head_dim != RSA_HEAD_DIM && d->head_dim != 64)
    RSA_FAIL(RSA_ERR_UNSUPPORTED, "rsa_qkv_prep_gather: head_dim must be 128 or 64 (got %d)", d->head_dim);
  // like rsa_qkv_prep: the whole sequence in one call, or -- ragged visual segment -- the visual tokens (dst_row 0) and
  // the text tokens (dst_row = visual token count) in two; source token = dst_row + row either way
  const RowMap rm = row_map(d);
  const bool whole = p->dst_row == 0 && p->rows == d->seq && rm.gap == 0;
  const bool vis = p->dst_row == 0 && p->rows == rm.vis_len && d->family == RSA_FAMILY_JOINT;
  const bool txt = p->dst_row == rm.vis_len && p->rows == d->seq - rm.vis_len && d->family == RSA_FAMILY_JOINT;
  if (!whole && !vis && !txt)
    RSA_FAIL(RSA_ERR_ARG, "rsa_qkv_prep_gather: rows / dst_row must name the whole sequence, the visual tokens or the text tokens");
  // head_dim 128: norms 0-2; head_dim 64 (CogVideoX): LayerNorm (norm 3), in the same one- or two-call forms
  if (d->head_dim == 64) {
    if (p->norm != 3)
      RSA_FAIL(RSA_ERR_UNSUPPORTED, "rsa_qkv_prep_gather: head_dim 64 is built for norm 3 (LayerNorm, CogVideoX) only, not norm %d", p->norm);
    if (!p->q_bias || !p->k_bias || (uintptr_t)p->q_bias % 16 || (uintptr_t)p->k_bias % 16)
      RSA_FAIL(RSA_ERR_ARG, "rsa_qkv_prep_gather: norm 3 needs 16-byte aligned biases");
  } else if (p->norm < 0 || p->norm > 2) {
    RSA_FAIL(RSA_ERR_UNSUPPORTED, "rsa_qkv_prep_gather: norm must be 0, 1 or 2 at head_dim 128 (got %d)", p->norm);
  }
  if (p->norm == 2 && !route->rinv_table)
    RSA_FAIL(RSA_ERR_ARG, "rsa_qkv_prep_gather: norm 2 needs route->rinv_table (rsa_row_rms on every owning rank)");
  if (p->norm && (!p->q_weight || !p->k_weight)) RSA_FAIL(RSA_ERR_ARG, "rsa_qkv_prep_gather: norm weights are null");
  if (p->rope_rows < 0 || p->rope_rows > p->rows) RSA_FAIL(RSA_ERR_ARG, "rsa_qkv_prep_gather: rope_rows out of range");
  if (p->rope_rows > 0 && (!p->cos || (!p->sin && !p->rope_compact))) RSA_FAIL(RSA_ERR_ARG, "rsa_qkv_prep_gather: rotary tables are null");
  WsLayout L;
  if (pool && (rc = check_ws(d, workspace, bytes, &L)) != RSA_OK) return rc;
  return launch_qkv_prep(p, d, nullptr, nullptr, nullptr, route, q, k, v, (char*)workspace, pool ? &L : nullptr,
                         (cudaStream_t)stream);
}

extern "C" int rsa_row_rms_dtype(const void* q_src, const void* k_src, int batch, int rows, int channels,
                                 const int64_t q_stride[2], const int64_t k_stride[2], float eps, float* rinv_q,
                                 float* rinv_k, int dtype, void* stream) {
  if (!q_src || !k_src || !rinv_q || !rinv_k || !q_stride || !k_stride) RSA_FAIL(RSA_ERR_ARG, "rsa_row_rms: null pointer");
  if (dtype != RSA_DTYPE_BF16 && dtype != RSA_DTYPE_F16) RSA_FAIL(RSA_ERR_UNSUPPORTED, "rsa_row_rms: dtype %d is not bf16 or fp16", dtype);
  if (batch < 1 || rows < 1 || channels < 8 || channels % 8) RSA_FAIL(RSA_ERR_ARG, "rsa_row_rms: bad sizes");
  if (((uintptr_t)q_src | (uintptr_t)k_src) % 16 || q_stride[1] % 8 || k_stride[1] % 8 || q_stride[0] % 8 || k_stride[0] % 8)
    RSA_FAIL(RSA_ERR_UNSUPPORTED, "rsa_row_rms: rows must be 16-byte aligned");
  return launch_row_rms(q_src, k_src, batch, rows, channels, q_stride, k_stride, eps, rinv_q, rinv_k,
                        dtype == RSA_DTYPE_F16, (cudaStream_t)stream);
}

extern "C" int rsa_row_rms(const void* q_src, const void* k_src, int batch, int rows, int channels,
                           const int64_t q_stride[2], const int64_t k_stride[2], float eps, float* rinv_q, float* rinv_k,
                           void* stream) {
  return rsa_row_rms_dtype(q_src, k_src, batch, rows, channels, q_stride, k_stride, eps, rinv_q, rinv_k, RSA_DTYPE_BF16,
                           stream);
}

extern "C" int rsa_rectified_attention_pooled_scatter(const rsa_attn_desc* d, const void* q, const void* k,
                                                      const void* v, const rsa_peer_route* route, void* workspace,
                                                      size_t bytes, void* stream) {
  WsLayout L;
  int rc = check_ws(d, workspace, bytes, &L);
  if (rc != RSA_OK) return rc;
  if ((rc = validate_route(d, route, false, true)) != RSA_OK) return rc;
  // result rows are [heads_total, head_dim]: the epilogue places head h at (head0 + h) * head_dim of the kernel
  // instantiation, so 64-column heads must run the 64-column one (not the debug dump or attention flag 4)
  if (d->head_dim == 64 && (g_attention_dbg || (g_attention_dbg_flags & 4)))
    RSA_FAIL(RSA_ERR_UNSUPPORTED, "rsa_rectified_attention_pooled_scatter: head_dim 64 runs the 64-column kernel 4 only");
  if (!q || !k || !v) RSA_FAIL(RSA_ERR_ARG, "rsa_rectified_attention_pooled_scatter: null tensor");
  char* ws = (char*)workspace;
  cudaStream_t s = (cudaStream_t)stream;
  if ((rc = launch_block_scores(d, ws, L, s)) != RSA_OK) return rc;
  if ((rc = launch_block_select(d, ws, L, s)) != RSA_OK) return rc;
  if ((rc = launch_rect_c(d, ws, L, s)) != RSA_OK) return rc;
  AttnArgs a;
  fill_attn_args(d, q, k, v, nullptr, ws, L, &a);
  a.o_table = (__nv_bfloat16* const*)route->out_table;
  a.peer_rows = route->rows_per_rank;
  a.peer_head0 = route->head0;
  a.peer_os[0] = route->out_stride[0];
  a.peer_os[1] = route->out_stride[1];
  return launch_attention(a, s);
}

extern "C" int rsa_rectified_attention_pooled(const rsa_attn_desc* d, const void* q, const void* k, const void* v,
                                              void* out, void* workspace, size_t bytes, void* stream) {
  WsLayout L;
  int rc = check_ws(d, workspace, bytes, &L);
  if (rc != RSA_OK) return rc;
  if (!q || !k || !v || !out) RSA_FAIL(RSA_ERR_ARG, "rsa_rectified_attention_pooled: null tensor");
  char* ws = (char*)workspace;
  cudaStream_t s = (cudaStream_t)stream;
  if ((rc = launch_block_scores(d, ws, L, s)) != RSA_OK) return rc;
  if ((rc = launch_block_select(d, ws, L, s)) != RSA_OK) return rc;
  if ((rc = launch_rect_c(d, ws, L, s)) != RSA_OK) return rc;
  AttnArgs a;
  fill_attn_args(d, q, k, v, out, ws, L, &a);
  return launch_attention(a, s);
}

extern "C" int rsa_rectified_attention_reuse(const rsa_attn_desc* d, const void* q, const void* k, const void* v,
                                             void* out, void* workspace, size_t bytes, int mask_mode, int pooled,
                                             void* stream) {
  WsLayout L;
  int rc = check_ws(d, workspace, bytes, &L);
  if (rc != RSA_OK) return rc;
  if (!q || !k || !v || !out) RSA_FAIL(RSA_ERR_ARG, "rsa_rectified_attention_reuse: null tensor");
  if (mask_mode < RSA_MASK_BUILD || mask_mode > RSA_MASK_KEEP_ALL)
    RSA_FAIL(RSA_ERR_ARG, "rsa_rectified_attention_reuse: mask_mode %d is not one of rsa_mask_mode", mask_mode);
  char* ws = (char*)workspace;
  cudaStream_t s = (cudaStream_t)stream;
  if (mask_mode != RSA_MASK_KEEP_ALL) {
    if (!pooled && (rc = launch_pool_stats(d, q, k, v, ws, L, s)) != RSA_OK) return rc;
    if ((rc = launch_block_scores(d, ws, L, s)) != RSA_OK) return rc;
    if ((rc = launch_block_select(d, ws, L, s, mask_mode == RSA_MASK_KEEP_LISTS)) != RSA_OK) return rc;
    if ((rc = launch_rect_c(d, ws, L, s)) != RSA_OK) return rc;
  }
  AttnArgs a;
  fill_attn_args(d, q, k, v, out, ws, L, &a);
  return launch_attention(a, s, mask_mode == RSA_MASK_BUILD);
}

extern "C" size_t rsa_masked_attention_workspace_bytes(int bh, int nq, int nkv) {
  if (bh <= 0 || nq <= 0 || nkv <= 0) return 0;
  // kept lists + counts + pair schedule + common-prefix lengths
  return 2 * align_up((size_t)bh * nq * nkv * 2, 256) + align_up((size_t)bh * nq * 4, 256) +
         2 * align_up((size_t)bh * ((nq + 1) / 2) * 4, 256);
}

extern "C" int rsa_masked_attention(const void* q, const void* k, const void* v, void* out, int bh, int seq_q,
                                    int seq_kv, int kv_len, const int64_t q_stride[2], const int64_t k_stride[2],
                                    const int64_t v_stride[2], const int64_t o_stride[2], const uint8_t* block_mask,
                                    int n_q_blocks, int n_kv_blocks, void* workspace, size_t bytes, void* stream,
                                    int dtype, int head_dim) {
  if (!q || !k || !v || !out || !block_mask) RSA_FAIL(RSA_ERR_ARG, "rsa_masked_attention: null pointer");
  const int q_round = (dtype & RSA_ATTN_FP32_SCALE) ? 0 : 1;
  dtype &= ~RSA_ATTN_FP32_SCALE;
  if (dtype != RSA_DTYPE_BF16 && dtype != RSA_DTYPE_F16) RSA_FAIL(RSA_ERR_UNSUPPORTED, "rsa_masked_attention: dtype %d", dtype);
  if (head_dim != RSA_HEAD_DIM && head_dim != 64) RSA_FAIL(RSA_ERR_UNSUPPORTED, "rsa_masked_attention: head_dim must be 128 or 64 (got %d)", head_dim);
  if (bh <= 0 || bh > 65535 || seq_q <= 0 || seq_kv <= 0 || kv_len < 1 || kv_len > seq_kv)
    RSA_FAIL(RSA_ERR_ARG, "rsa_masked_attention: bad sizes");
  if (n_q_blocks != (seq_q + 127) / 128 || n_kv_blocks != (seq_kv + 127) / 128)
    RSA_FAIL(RSA_ERR_ARG, "rsa_masked_attention: block counts do not match the sequence lengths");
  const size_t need = rsa_masked_attention_workspace_bytes(bh, n_q_blocks, n_kv_blocks);
  if (!workspace || bytes < need || (uintptr_t)workspace % 256) RSA_FAIL(RSA_ERR_WORKSPACE, "rsa_masked_attention: workspace");
  const int64_t* st[4] = {q_stride, k_stride, v_stride, o_stride};
  for (int t = 0; t < 4; ++t)
    for (int i = 0; i < 2; ++i)
      if (st[t][i] < 0 || st[t][i] % 8) RSA_FAIL(RSA_ERR_UNSUPPORTED, "strides must be multiples of 8 elements");
  char* ws = (char*)workspace;
  const size_t list_bytes = align_up((size_t)bh * n_q_blocks * n_kv_blocks * 2, 256);
  uint16_t* kidx = (uint16_t*)ws;
  uint16_t* sched = (uint16_t*)(ws + list_bytes);
  int32_t* kcnt = (int32_t*)(ws + 2 * list_bytes);
  int32_t* pshared = (int32_t*)(ws + 2 * list_bytes + align_up((size_t)bh * n_q_blocks * 4, 256));
  int32_t* qshared = (int32_t*)((char*)pshared + align_up((size_t)bh * ((n_q_blocks + 1) / 2) * 4, 256));
  cudaStream_t s = (cudaStream_t)stream;
  int rc = launch_mask_to_lists(block_mask, bh, n_q_blocks, n_kv_blocks, (kv_len + 127) / 128, kidx, kcnt, s);
  if (rc != RSA_OK) return rc;
  AttnArgs a;
  a.q = (const __nv_bfloat16*)q;
  a.k = (const __nv_bfloat16*)k;
  a.v = (const __nv_bfloat16*)v;
  a.o = (__nv_bfloat16*)out;
  a.batch = 1;
  a.heads = bh;
  a.qs[0] = a.ks[0] = a.vs[0] = a.os[0] = 0;
  a.qs[1] = q_stride[0], a.qs[2] = q_stride[1];
  a.ks[1] = k_stride[0], a.ks[2] = k_stride[1];
  a.vs[1] = v_stride[0], a.vs[2] = v_stride[1];
  a.os[1] = o_stride[0], a.os[2] = o_stride[1];
  a.seq_q = seq_q;
  a.seq_kv = seq_kv;
  a.kv_len = kv_len;
  a.q_valid = seq_q;
  a.vis_len = 1 << 30;  // no text segment: every block is "visual", nothing is shifted
  a.nq_vis = 1 << 20;
  a.gap = 0;
  a.nqt = n_q_blocks;
  a.nb = n_kv_blocks;
  a.kept_idx = kidx;
  a.kept_cnt = kcnt;
  a.sched_idx = sched;
  a.pair_shared = pshared;
  a.quad_shared = qshared;
  a.R = nullptr;
  a.C = nullptr;
  a.o_table = nullptr;
  a.peer_rows = a.peer_head0 = 0;
  a.peer_os[0] = a.peer_os[1] = 0;
  a.scale_log2 = (float)((1.0 / sqrt((double)head_dim)) * 1.44269504);  // the reference's qk_scale (wan21 :145)
  a.head_dim = head_dim;
  a.rescale_thr = attention_rescale_threshold(dtype == RSA_DTYPE_F16);
  a.front_text_heads = 0;
  a.f16 = dtype == RSA_DTYPE_F16;
  a.q_round = q_round;
  a.dbg = g_attention_dbg;
  a.dbg_flags = g_attention_dbg_flags;
  return launch_attention(a, s);
}

// Dense attention without lists (kernel 4's kDense form): only batch, heads, seq, head_dim, the strides and dtype of the
// descriptor are read.  Every refusal happens here, before any CUDA call.
static int validate_dense(const rsa_attn_desc* d, const void* q, const void* k, const void* v, const void* out,
                          bool scatter, int seq_kv, int q_valid, int kv_len, const char* fn) {
  if (!d || !q || !k || !v || (!scatter && !out)) RSA_FAIL(RSA_ERR_ARG, "%s: null pointer", fn);
  if (d->head_dim != RSA_HEAD_DIM && d->head_dim != 64)
    RSA_FAIL(RSA_ERR_UNSUPPORTED, "%s: head_dim must be 128 or 64 (got %d)", fn, d->head_dim);
  if (d->dtype != RSA_DTYPE_BF16 && d->dtype != RSA_DTYPE_F16)
    RSA_FAIL(RSA_ERR_UNSUPPORTED, "%s: dtype %d is not one of rsa_dtype (bf16, fp16)", fn, d->dtype);
  if (d->batch <= 0 || d->heads <= 0 || d->seq <= 0 || seq_kv <= 0)
    RSA_FAIL(RSA_ERR_ARG, "%s: batch/heads/seq/seq_kv must be positive", fn);
  if ((int64_t)d->batch * d->heads > 65535) RSA_FAIL(RSA_ERR_UNSUPPORTED, "%s: batch*heads > 65535", fn);
  if (q_valid < 1 || q_valid > d->seq) RSA_FAIL(RSA_ERR_ARG, "%s: q_valid=%d out of [1, seq=%d]", fn, q_valid, d->seq);
  if (kv_len < 1 || kv_len > seq_kv) RSA_FAIL(RSA_ERR_ARG, "%s: kv_len=%d out of [1, seq_kv=%d]", fn, kv_len, seq_kv);
  const int64_t* st[4] = {d->q_stride, d->k_stride, d->v_stride, d->o_stride};
  for (int t = 0; t < (scatter ? 3 : 4); ++t)
    for (int i = 0; i < 3; ++i)
      if (st[t][i] < 0 || st[t][i] % 8)
        RSA_FAIL(RSA_ERR_UNSUPPORTED, "%s: strides must be non-negative multiples of 8 elements (16 bytes)", fn);
  if (((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)(scatter ? nullptr : out)) % 16)
    RSA_FAIL(RSA_ERR_UNSUPPORTED, "%s: q/k/v/out must be 16-byte aligned", fn);
  return RSA_OK;
}

static void fill_dense_args(const rsa_attn_desc* d, const void* q, const void* k, const void* v, void* out, int seq_kv,
                            int q_valid, int kv_len, AttnArgs* a) {
  memset(a, 0, sizeof(*a));
  a->q = (const __nv_bfloat16*)q;
  a->k = (const __nv_bfloat16*)k;
  a->v = (const __nv_bfloat16*)v;
  a->o = (__nv_bfloat16*)out;
  a->batch = d->batch;
  a->heads = d->heads;
  for (int i = 0; i < 3; ++i) {
    a->qs[i] = d->q_stride[i];
    a->ks[i] = d->k_stride[i];
    a->vs[i] = d->v_stride[i];
    a->os[i] = d->o_stride[i];
  }
  a->seq_q = d->seq;
  a->seq_kv = seq_kv;
  a->kv_len = kv_len;
  a->q_valid = q_valid;
  a->vis_len = 1 << 30;  // no text segment: every block is "visual", nothing is shifted (as rsa_masked_attention)
  a->nq_vis = 1 << 20;
  a->gap = 0;
  a->nqt = (d->seq + RSA_BLOCK - 1) / RSA_BLOCK;
  a->nb = (seq_kv + RSA_BLOCK - 1) / RSA_BLOCK;
  a->scale_log2 = (float)((1.0 / sqrt((double)d->head_dim)) * 1.44269504);
  a->head_dim = d->head_dim;
  a->rescale_thr = attention_rescale_threshold(d->dtype == RSA_DTYPE_F16);
  a->front_text_heads = 0;
  a->f16 = d->dtype == RSA_DTYPE_F16;
  a->q_round = 0;        // flash-attn's arithmetic: the fp32 scores are scaled, q is not rounded
  a->dbg = nullptr;      // the dense form has no debug dump
  a->dbg_flags = g_attention_dbg_flags;
}

extern "C" int rsa_dense_attention(const rsa_attn_desc* d, const void* q, const void* k, const void* v, void* out,
                                   int seq_kv, int q_valid, int kv_len, void* stream) {
  int rc = validate_dense(d, q, k, v, out, false, seq_kv, q_valid, kv_len, "rsa_dense_attention");
  if (rc != RSA_OK) return rc;
  AttnArgs a;
  fill_dense_args(d, q, k, v, out, seq_kv, q_valid, kv_len, &a);
  return launch_attention_tc5(a, (cudaStream_t)stream, true);
}

extern "C" int rsa_dense_attention_scatter(const rsa_attn_desc* d, const void* q, const void* k, const void* v,
                                           const rsa_peer_route* route, int q_valid, int kv_len, void* stream) {
  int rc = validate_dense(d, q, k, v, nullptr, true, d ? d->seq : 0, q_valid, kv_len, "rsa_dense_attention_scatter");
  if (rc != RSA_OK) return rc;
  if ((rc = validate_route(d, route, false, true)) != RSA_OK) return rc;
  // as rsa_rectified_attention_pooled_scatter: the epilogue places head h at (head0 + h) * head_dim of the instantiation
  if (d->head_dim == 64 && (g_attention_dbg || (g_attention_dbg_flags & 4)))
    RSA_FAIL(RSA_ERR_UNSUPPORTED, "rsa_dense_attention_scatter: head_dim 64 runs the 64-column kernel 4 only");
  AttnArgs a;
  fill_dense_args(d, q, k, v, nullptr, d->seq, q_valid, kv_len, &a);
  a.o_table = (__nv_bfloat16* const*)route->out_table;
  a.peer_rows = route->rows_per_rank;
  a.peer_head0 = route->head0;
  a.peer_os[0] = route->out_stride[0];
  a.peer_os[1] = route->out_stride[1];
  return launch_attention_tc5(a, (cudaStream_t)stream, true);
}
