// block_select.cu -- kernel 3b: per query block, turn pooled scores into the kept-block list and the
// rectification weights.  One CTA (256 threads) per (head, query block); everything stays in shared memory.
// Replaces (reference paths relative to the reference root):
//   softmax(A * D^-1/2)                                            rectified_wan21_attn.py:206-213
//   IPAR re-allocation (joint family)                              rectified_hunyuan_attn.py:218-223
//   sort(desc) / cumsum / (cumsum <= p).sum()+1 / max(.., top_k)   rectified_wan21_attn.py:220-229
//   one-hot scatter through four expanded int64 index tensors      rectified_wan21_attn.py:232-256 (host sync)
//   neighbour / first-frame / text-block unions                    wan21 :259-271, hunyuan :265-277
//   part = one_hot | nogapr; R = sum(part * P); P masked by ~part  wan21 :329-336, hunyuan :348-355
// Defined where the reference is not (SURVEY.md 0.5/0.6): ties sort by (probability desc, index asc); the
// cumulative sum is sequential fp32 in sorted order; the threshold is compared as fp32.
// Outputs: kept-block bitmask, ascending u16 kept-block index list + count (what kernel 4 walks), n_needed, R,
// W = P*(1-part) for kernel 3c, optionally P itself for the parity tests.
#include <math.h>

#include "rsa_common.cuh"

namespace rsa {
namespace {

constexpr int kThreads = 256;
constexpr int kMaxEnt = RSA_MAX_ENTRIES;
constexpr int kMaxWords = kMaxEnt / 32 + 1;

struct SelectArgs {
  const float* scores;    // [BH,NQ,score_ld]
  const uint8_t* nogapr;  // [BH,NQ,nogapr_ld]
  float* probs;           // optional
  float* w_skip;          // [BH,NQ,ent_ld]
  uint32_t* mask_bits;    // [BH,NQT,mask_words]
  uint16_t* kept_idx;     // [BH,NQT,NB]
  int32_t* kept_cnt;      // [BH,NQT]
  int32_t* n_needed;      // [BH,NQ]
  float* R;               // [BH,NQT]
  float* C;               // [BH,NQT,128] (text rows zeroed here)
  const uint8_t* nbr;
  int nbr_rows, nbr_cols;
  int nq, nqt, nb, nkc, score_ld, nogapr_ld, n_ent, ent_ld, mask_words;
  int joint, top_k, first_frame_blocks, text_end_block, kv_blocks_valid;
  int keep_lists;  // mask re-use: the kept-block bitmask / lists of an earlier call on this workspace stay as they are;
                   // only P, R and W are recomputed from the current scores and GAPR bytes
  float p_remain, scale;
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// block-wide reductions with a fixed combination order (warp tree, then warps 0..7 sequentially)
__device__ float block_sum(float v, float* scratch) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = scratch[0];
#pragma unroll
  for (int w = 1; w < kThreads / 32; ++w) t += scratch[w];
  return t;
}
__device__ float block_max(float v, float* scratch) {
  v = warp_max(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = scratch[0];
#pragma unroll
  for (int w = 1; w < kThreads / 32; ++w) t = fmaxf(t, scratch[w]);
  return t;
}

// Emits the ascending index list of the set bits of s_mask[0..words) restricted to blocks < limit.
__device__ void emit_list(const uint32_t* s_mask, int words, int limit, uint16_t* out, int32_t* out_cnt,
                          int* s_scan) {
  const int tid = threadIdx.x;
  // words <= 65 -> one warp scans (up to 3 words per lane)
  if (tid < 32) {
    int cnt[3], tot = 0;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const int w = tid * 3 + r;
      uint32_t m = 0;
      if (w < words) {
        m = s_mask[w];
        const int lo = w * 32;
        if (lo + 32 > limit) m = (lo >= limit) ? 0u : (m & ((1u << (limit - lo)) - 1u));
      }
      cnt[r] = __popc(m);
      tot += cnt[r];
    }
    int incl = tot;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int n = __shfl_up_sync(0xffffffffu, incl, o);
      if (tid >= o) incl += n;
    }
    int excl = incl - tot;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const int w = tid * 3 + r;
      if (w < words) s_scan[w] = excl;
      excl += cnt[r];
    }
    if (tid == 31) *out_cnt = incl;
  }
  __syncthreads();
  for (int w = tid; w < words; w += kThreads) {
    uint32_t m = s_mask[w];
    const int lo = w * 32;
    if (lo + 32 > limit) m = (lo >= limit) ? 0u : (m & ((1u << (limit - lo)) - 1u));
    int o = s_scan[w];
    while (m) {
      const int b = __ffs(m) - 1;
      m &= m - 1;
      out[o++] = (uint16_t)(lo + b);
    }
  }
}

// Descending bitonic sort of n_sort = kThreads * EPT probabilities, as their bit patterns (p >= +0, so unsigned
// integer order = float order; one min/max instruction per compare).  Only the sorted VALUES are needed: the
// cumulative sum runs over them, and the selected set is recovered from the value of the n-th entry (see the kernel).
// Thread t holds elements [EPT*t, EPT*t + EPT) in registers: partners at distance j < EPT are in the same thread, at
// distance j < 32*EPT in the same warp (shuffle), and only the few stages with j >= 32*EPT go through shared memory
// (6 of the 55 stages for 1024 entries).  K and J are template parameters so every x[] index is a compile-time
// constant and the values stay in registers.
template <int EPT, int K, int J>
__device__ __forceinline__ void sort_steps(uint32_t (&x)[EPT], uint32_t* s_val, int tid) {
  if constexpr (J >= 32 * EPT) {
    __syncthreads();
#pragma unroll
    for (int r = 0; r < EPT; ++r) s_val[r * kThreads + tid] = x[r];  // [r][tid]: conflict-free
    __syncthreads();
#pragma unroll
    for (int r = 0; r < EPT; ++r) {
      const int e = tid * EPT + r;
      const int pt = tid ^ (J / EPT);  // partner element e ^ J = (pt, r)
      const uint32_t y = s_val[r * kThreads + pt];
      const bool take_max = ((e & K) == 0) != ((e & J) != 0);
      x[r] = take_max ? max(x[r], y) : min(x[r], y);
    }
  } else if constexpr (J >= EPT) {
#pragma unroll
    for (int r = 0; r < EPT; ++r) {
      const int e = tid * EPT + r;
      const uint32_t y = __shfl_xor_sync(0xffffffffu, x[r], J / EPT);
      const bool take_max = ((e & K) == 0) != ((e & J) != 0);
      x[r] = take_max ? max(x[r], y) : min(x[r], y);
    }
  } else {
#pragma unroll
    for (int r = 0; r < EPT; ++r) {
      if ((r & J) == 0) {  // r is the lower element of the pair (r, r | J)
        const int e = tid * EPT + r;
        const bool desc = (e & K) == 0;
        const uint32_t hi = max(x[r], x[r | J]), lo = min(x[r], x[r | J]);
        x[r] = desc ? hi : lo;
        x[r | J] = desc ? lo : hi;
      }
    }
  }
  if constexpr (J > 1) sort_steps<EPT, K, J / 2>(x, s_val, tid);
  else if constexpr (K < kThreads * EPT) sort_steps<EPT, 2 * K, K>(x, s_val, tid);
}

// s_p[0..n_net) -> s_val sorted descending (entries >= n_net count as +0).  The joint family's text aggregate
// (entry n_net, the highest index, n_ent = n_net + 1) is not put through the network: in (value desc, index asc) order
// it comes after every visual entry >= it, so it is inserted at position #{visual entries >= it} while the sorted values
// are written out.  That keeps the network at the next power of two above the number of VISUAL blocks -- Flux at
// 4096^2 has 512 of them, and 513 entries would double the network to 1024.
template <int EPT>
__device__ void sort_desc(const float* s_p, int n_net, int n_ent, uint32_t* s_val, int* s_pos, int tid) {
  uint32_t x[EPT];
#pragma unroll
  for (int r = 0; r < EPT; ++r) {
    const int e = tid * EPT + r;
    x[r] = e < n_net ? __float_as_uint(s_p[e]) : 0u;
  }
  if (tid == 0) *s_pos = 0;
  sort_steps<EPT, 2, 1>(x, s_val, tid);
  __syncthreads();
  if (n_ent > n_net) {
    const uint32_t extra = __float_as_uint(s_p[n_net]);
    int ge = 0;
#pragma unroll
    for (int r = 0; r < EPT; ++r) ge += (tid * EPT + r < n_net && x[r] >= extra) ? 1 : 0;
    if (ge) atomicAdd(s_pos, ge);
    __syncthreads();
    const int pos = *s_pos;
#pragma unroll
    for (int r = 0; r < EPT; ++r) {
      const int e = tid * EPT + r;
      if (e < n_net) s_val[e + (e >= pos ? 1 : 0)] = x[r];
    }
    if (tid == 0) s_val[pos] = extra;
  } else {
#pragma unroll
    for (int r = 0; r < EPT; ++r) s_val[tid * EPT + r] = x[r];
  }
  __syncthreads();
}

// Held to 8 CTAs per SM: the kernel is issue-bound with long barrier waits; without a bound ptxas drifted from 48 to 64
// registers = 4 CTAs per SM and the kernel lost 11 %.  At 5 / 6 / 8 CTAs per SM: C3b 0.69 / 0.63 / 0.62 ms, Flux
// 0.23 / 0.22 / 0.21, C4 0.51 / 0.47 / 0.45 (profiles/r01_block_select_occupancy_ab.txt).
__global__ void __launch_bounds__(kThreads, 8) block_select_kernel(const SelectArgs a) {
  __shared__ float s_p[kMaxEnt + 1];
  __shared__ uint32_t s_val[kMaxEnt + 1];  // sorted probability bit patterns
  __shared__ uint32_t s_thr;           // bit pattern of the n-th largest probability
  __shared__ int s_ties_needed, s_ties_total;
  __shared__ uint32_t s_mask[kMaxWords];
  __shared__ int s_scan[kMaxWords];
  __shared__ float s_red[kThreads / 32];
  __shared__ int s_n;

  const int bh = blockIdx.y, i = blockIdx.x, tid = threadIdx.x;
  const int words = a.mask_words;
  const int64_t orow = (int64_t)bh * a.nqt + i;

  if (i >= a.nq) {
    if (a.keep_lists) return;  // dense list, R = 1 and C = 0 are already in place
    // text query block: dense row (all valid KV blocks), R = 1, C = 0
    for (int w = tid; w < words; w += kThreads) {
      const int lo = w * 32;
      uint32_t m = 0xffffffffu;
      if (lo + 32 > a.kv_blocks_valid) m = (lo >= a.kv_blocks_valid) ? 0u : ((1u << (a.kv_blocks_valid - lo)) - 1u);
      s_mask[w] = m;
      a.mask_bits[orow * words + w] = m;
    }
    if (tid < 128) a.C[orow * 128 + tid] = 0.f;
    if (tid == 0) a.R[orow] = 1.f;
    __syncthreads();
    emit_list(s_mask, words, a.kv_blocks_valid, a.kept_idx + orow * a.nb, a.kept_cnt + orow, s_scan);
    return;
  }

  const int nq = a.nq, n_in = a.nkc, n_ent = a.n_ent;
  const float* srow = a.scores + ((int64_t)bh * nq + i) * a.score_ld;

  // ---- softmax over all n_in columns (visual pooled keys + single text keys)
  float lm = -INFINITY;
  for (int j = tid; j < n_in; j += kThreads) lm = fmaxf(lm, __fmul_rn(srow[j], a.scale));
  const float mx = block_max(lm, s_red);
  float ls = 0.f;
  for (int j = tid; j < n_in; j += kThreads) {
    const float e = expf(__fsub_rn(__fmul_rn(srow[j], a.scale), mx));
    if (j < nq) s_p[j] = e;
    ls += e;
  }
  const float tot = block_sum(ls, s_red);
  if (!a.joint) {
    for (int j = tid; j < nq; j += kThreads) s_p[j] = __fdiv_rn(s_p[j], tot);
  } else {
    // IPAR: visual blocks stand for 128 keys each, text keys for one (hunyuan :218-223)
    float lns = 0.f, lts = 0.f;
    for (int j = tid; j < n_in; j += kThreads) {
      if (j < nq) {
        const float p0 = __fdiv_rn(s_p[j], tot);
        s_p[j] = p0;
        lns += p0;
      } else {
        lts += __fdiv_rn(expf(__fsub_rn(__fmul_rn(srow[j], a.scale), mx)), tot);
      }
    }
    const float ns = block_sum(lns, s_red);
    const float ts = block_sum(lts, s_red);
    const float den = __fadd_rn(__fmul_rn(ns, 128.f), ts);
    for (int j = tid; j < nq; j += kThreads) s_p[j] = __fdiv_rn(__fmul_rn(s_p[j], 128.f), den);
    if (tid == 0) s_p[nq] = __fdiv_rn(ts, den);
  }
  __syncthreads();
  if (a.probs) {
    float* prow = a.probs + ((int64_t)bh * nq + i) * a.ent_ld;
    for (int j = tid; j < n_ent; j += kThreads) prow[j] = s_p[j];
  }

  if (a.keep_lists) {
    // ---- mask re-use (SURVEY 8f rank 4): the selection of an earlier call stands; rectify it with the current P
    for (int w = tid; w < words; w += kThreads) s_mask[w] = a.mask_bits[orow * words + w];
    __syncthreads();
    const uint8_t* grow = a.nogapr + ((int64_t)bh * nq + i) * a.nogapr_ld;
    float* wrow = a.w_skip + ((int64_t)bh * nq + i) * a.ent_ld;
    float lr = 0.f;
    for (int j = tid; j < n_ent; j += kThreads) {
      bool part = (s_mask[j >> 5] >> (j & 31)) & 1u;
      if (j < nq && grow[j]) part = true;
      const float p = s_p[j];
      lr += part ? p : 0.f;
      wrow[j] = part ? 0.f : p;
    }
    const float r = block_sum(lr, s_red);
    if (tid == 0) a.R[orow] = r;
    return;
  }

  // ---- sort the probabilities (descending); ties are resolved below by index, ascending
  // entries that go through the sorting network: all of them, unless leaving the text aggregate out halves the network
  // (the visual blocks alone fill a power of two: Flux at 4096^2 / 2048^2); it is then inserted afterwards
  int n_sort = kThreads;
  while (n_sort < nq) n_sort <<= 1;
  const int n_net = (a.joint && n_sort == nq) ? nq : n_ent;
  while (n_sort < n_net) n_sort <<= 1;
  if (n_sort == kThreads) sort_desc<1>(s_p, n_net, n_ent, s_val, &s_ties_total, tid);
  else if (n_sort == 2 * kThreads) sort_desc<2>(s_p, n_net, n_ent, s_val, &s_ties_total, tid);
  else if (n_sort == 4 * kThreads) sort_desc<4>(s_p, n_net, n_ent, s_val, &s_ties_total, tid);
  else sort_desc<8>(s_p, n_net, n_ent, s_val, &s_ties_total, tid);

  // ---- sequential fp32 cumulative sum over the sorted probabilities (wan21 :221-229)
  if (tid == 0) {
    // probabilities are >= 0, so c never decreases: count in chunks of 8 (independent loads, one dependent add
    // chain) and stop after the first chunk that crosses the threshold
    float c = 0.f;
    int cnt = 0;
    for (int k0 = 0; k0 < n_ent; k0 += 8) {
      float pk[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) pk[u] = k0 + u < n_ent ? __uint_as_float(s_val[k0 + u]) : INFINITY;
      int ok = 0;
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        c = __fadd_rn(c, pk[u]);
        ok += (c <= a.p_remain) ? 1 : 0;
      }
      cnt += ok;
      if (ok < 8) break;
    }
    int n = cnt + 1;
    if (n < a.top_k) n = a.top_k;
    if (n > n_ent) n = n_ent;
    s_n = n;
    a.n_needed[(int64_t)bh * nq + i] = n;
    // The n selected entries in (probability desc, index asc) order are: every entry above the n-th value, plus the
    // first `ties_needed` entries (by index) equal to it.
    uint32_t thr = 0u;
    int above = 0;
    if (n > 0) {
      thr = s_val[n - 1];
      above = n - 1;
      while (above > 0 && s_val[above - 1] == thr) --above;
    }
    s_thr = thr;
    s_ties_needed = n - above;
    s_ties_total = 0;
  }
  for (int w = tid; w < words; w += kThreads) s_mask[w] = 0u;
  __syncthreads();
  const int n = s_n;
  const uint32_t thr = s_thr;

  // ---- scatter the n best entries, then the constant unions
  if (n > 0) {
    int my_ties = 0;
    for (int j = tid; j < n_ent; j += kThreads) {
      const uint32_t v = __float_as_uint(s_p[j]);
      if (v > thr) atomicOr(&s_mask[j >> 5], 1u << (j & 31));
      my_ties += v == thr ? 1 : 0;
    }
    if (my_ties) atomicAdd(&s_ties_total, my_ties);
    __syncthreads();
    if (s_ties_total == s_ties_needed) {  // the usual case: one entry holds the n-th value
      for (int j = tid; j < n_ent; j += kThreads)
        if (__float_as_uint(s_p[j]) == thr) atomicOr(&s_mask[j >> 5], 1u << (j & 31));
    } else if (tid == 0) {                // several equal probabilities straddle the cut: lowest indices first
      int left = s_ties_needed;
      for (int j = 0; j < n_ent && left > 0; ++j)
        if (__float_as_uint(s_p[j]) == thr) {
          s_mask[j >> 5] |= 1u << (j & 31);
          --left;
        }
    }
    __syncthreads();
  }
  if (a.nbr != nullptr && i < a.nbr_rows) {
    const int cols = a.nbr_cols < nq ? a.nbr_cols : nq;
    const uint8_t* nrow = a.nbr + (int64_t)i * a.nbr_cols;
    for (int j = tid; j < cols; j += kThreads)
      if (nrow[j]) atomicOr(&s_mask[j >> 5], 1u << (j & 31));
  }
  if (!a.joint) {
    if (i < a.first_frame_blocks)
      for (int j = tid; j < a.first_frame_blocks && j < a.nb; j += kThreads) atomicOr(&s_mask[j >> 5], 1u << (j & 31));
  } else {
    for (int j = nq + tid; j < a.text_end_block && j < a.nb; j += kThreads) atomicOr(&s_mask[j >> 5], 1u << (j & 31));
  }
  __syncthreads();

  // ---- rectification weights: part = kept | nogapr over the n_ent probability columns
  const uint8_t* grow = a.nogapr + ((int64_t)bh * nq + i) * a.nogapr_ld;
  float* wrow = a.w_skip + ((int64_t)bh * nq + i) * a.ent_ld;
  float lr = 0.f;
  for (int j = tid; j < n_ent; j += kThreads) {
    bool part = (s_mask[j >> 5] >> (j & 31)) & 1u;
    if (j < nq && grow[j]) part = true;
    const float p = s_p[j];
    lr += part ? p : 0.f;
    wrow[j] = part ? 0.f : p;
  }
  const float r = block_sum(lr, s_red);
  if (tid == 0) a.R[orow] = r;
  for (int w = tid; w < words; w += kThreads) a.mask_bits[orow * words + w] = s_mask[w];
  emit_list(s_mask, words, a.kv_blocks_valid < a.nb ? a.kv_blocks_valid : a.nb, a.kept_idx + orow * a.nb,
            a.kept_cnt + orow, s_scan);
}

}  // namespace

int launch_block_select(const rsa_attn_desc* d, char* ws, const WsLayout& L, cudaStream_t s, bool keep_lists) {
  SelectArgs a;
  a.keep_lists = keep_lists ? 1 : 0;
  a.scores = (const float*)(ws + L.off_scores);
  a.nogapr = (const uint8_t*)(ws + L.off_nogapr);
  a.probs = d->debug_dump_probs ? (float*)(ws + L.off_probs) : nullptr;
  a.w_skip = (float*)(ws + L.off_w);
  a.mask_bits = (uint32_t*)(ws + L.off_mask);
  a.kept_idx = (uint16_t*)(ws + L.off_kidx);
  a.kept_cnt = (int32_t*)(ws + L.off_kcnt);
  a.n_needed = (int32_t*)(ws + L.off_nneed);
  a.R = (float*)(ws + L.off_R);
  a.C = (float*)(ws + L.off_C);
  a.nbr = (d->nbr_rows > 0 && d->nbr_cols > 0) ? d->nbr : nullptr;
  a.nbr_rows = d->nbr_rows;
  a.nbr_cols = d->nbr_cols;
  a.nq = L.nq;
  a.nqt = L.nqt;
  a.nb = L.nb;
  a.nkc = L.nkc;
  a.score_ld = L.score_ld;
  a.nogapr_ld = L.nogapr_ld;
  a.n_ent = L.n_entries;
  a.ent_ld = L.ent_ld;
  a.mask_words = L.mask_words;
  a.joint = d->family == RSA_FAMILY_JOINT;
  a.top_k = d->top_k;
  a.first_frame_blocks = d->first_frame_blocks;
  a.text_end_block = d->text_end_block;
  a.kv_blocks_valid = (d->kv_len + 127) / 128;
  a.p_remain = d->p_remain;
  a.scale = (float)(1.0 / sqrt((double)d->head_dim));  // == float32(head_dim ** -0.5)
  if (L.nqt == 0) return RSA_OK;
  dim3 grid(L.nqt, L.bh);
  block_select_kernel<<<grid, kThreads, 0, s>>>(a);
  RSA_CUDA_CHECK(cudaGetLastError());
  return RSA_OK;
}

}  // namespace rsa
