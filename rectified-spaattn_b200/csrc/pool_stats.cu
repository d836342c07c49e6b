// pool_stats.cu -- kernel 2: block mean pooling of Q, K, V and the GAPR deviation statistics in ONE read.
// Replaces, per 128-token block (reference paths relative to the reference root):
//   query_pool / key_pool / value_pool = X_blocks.mean(dim=-2)    rectified_wan21_attn.py:189-192, :337
//   delta = X_blocks - pool; delta.abs().mean(dim=-2)             rectified_spaattn/gapr_mask.py:19-30
//   key_text = key[:, :, NQ*128 : NQ*128 + attenable]             rectified_hunyuan_attn.py:193-194
// The reference re-reads Q and K four times and materialises two full-size temporaries; here every element of
// Q, K, V is read from HBM exactly once (algorithmic bytes = 3*S*H*D*2) and stays in registers for the
// second (deviation) sweep.
//
// The 256 threads of a CTA reduce one (block, head, tensor) at a time.  Within a block, thread (warp w, lane l) owns
// rows 16w + 2*it + (l>>4), it = 0..7, and the eight columns 8*(l&15) .. +7.  Summation order per block (the oracle
// replicates it bit for bit):
//   lane chain over it = 0..7 (sequential fp32) -> half-warp pair (shfl xor 16) -> warps 0..7 (sequential).
// Rows >= valid_rows contribute zeros; the divisor is always 128 (the reference zero-pads, wan21 :299-302).
// Rows are counted in the padded layout (rsa_common.cuh RowMap): a visual block reads memory rows below vis_len and
// zeros above, a text block reads memory rows shifted down by the gap.
//
// Kernel 0 is a second front end of the same reduction ("prep"): instead of loading finished Q/K/V rows it builds them from
// the projection outputs [B, S, H*D] -- per-head RMSNorm, rotary embedding, re-layout to [B, H, S, D] -- stores
// them, and pools the values it has just rounded to bf16, so the pooled statistics are bit-identical to pooling the
// stored rows and Q, K, V are never read back.  Replaces rectified_hunyuan_attn.py:448-479 (and the same sequence
// in rectified_flux_attn.py): unflatten/transpose, attn.norm_q / attn.norm_k (diffusers RMSNorm(head_dim, eps):
// x * rsqrt(mean(x^2) + eps) in fp32 -> bf16 -> * weight -> bf16) and diffusers apply_rotary_emb(use_real=True,
// use_real_unbind_dim=-1): out = x * cos + rotate_pairs(x) * sin in fp32 (two products and a sum, each rounded) -> bf16.
// An fp16 model runs the same sequence in fp16 (diffusers rounds at the same points in either format): kernel 0's kF16
// forms round with cvt.rn.f16x2.f32 -- no .satfinite, so an overflow becomes +-inf as in .to(torch.float16), and results
// below 2^-14 stay fp16 subnormals -- and pool the fp16 rows they store, exactly as kernel 2's fp16 form reads them.
#include <cuda_fp16.h>

#include "ptx_sm100.cuh"
#include "rsa_common.cuh"

namespace rsa {
namespace {

constexpr int kThreads = 256;

struct PrepArgs {  // 16-bit tensors are in the descriptor's dtype (bf16, or fp16 in the kF16 forms)
  const __nv_bfloat16* src[3];  // q, k, v projection outputs [B, rows, H*D], D = head_dim (128, or 64 with LayerNorm)
  int64_t src_stride[3][2];     // (batch, token) element strides
  __nv_bfloat16* dst[3];        // [B, H, S, D] views
  int64_t dst_stride[3][3];     // (batch, head, token)
  const __nv_bfloat16* w[2];    // norm weights of q, k ([D], or [H*128] with w_head_stride = 128) or nullptr
  const __nv_bfloat16* bias[2]; // LayerNorm biases of q, k ([D]) -- kNorm = 3 only
  int w_head_stride;            // 0: one weight vector per tensor (norm over head_dim); 128: norm across heads (Wan)
  const float* row_rinv[2];     // norm across heads: rsqrt(mean(x^2) + eps) per (batch, source row), from row_rms_kernel
  float eps;
  const float *cos, *sin;       // fp32 [rope_rows, D]
  int rope_compact;             // cos = [rope_rows, D / 2] pairs (cos_i, sin_i), sin unused: half the table bytes per row
  int rope_rows;                // source rows below this are rotated
  int rows;                     // source rows
  int dst_row0;                 // memory row of source row 0 in the destination
  int blk0;                     // padded-layout block of source row 0
  int pool;                     // also pool the produced rows
  // fused Ulysses gather: source row r lives on rank r / src_rows (peer-mapped buffers), head h is head src_head0 + h there
  const __nv_bfloat16* const* src_table;  // device array [3][n_src] or nullptr
  const float* const* rinv_table;         // gather with the norm across heads: device array [2][n_src] of [B, src_rows] fp32
  int n_src, src_rows, src_head0;
};

struct PoolArgs {
  const __nv_bfloat16* x[3];  // q, k, v
  int64_t stride[3][3];       // (batch, head, token) element strides
  int valid_rows[3];          // padded-layout rows >= this are zeros
  int vis_len, nq_vis, gap;   // RowMap
  int n_blk[3];               // blocks to pool per tensor (NQ, NQ, NB)
  float* mean[3];             // q_pool, k_cat, v_pool
  float* mad[3];              // q_mad, k_mad, nullptr
  int out_rows[3];            // rows per head of the mean arrays (NQ, NKC, NB)
  int heads;
  int head_dim;               // 128 or 64: columns >= head_dim do not exist in x and pool as zeros
  // text keys copied as fp32 rows behind the pooled keys
  int text_keys, text_from;   // a, memory row of the first text token (= vis_len)
};

template <bool kF16 = false>
__device__ __forceinline__ void unpack8(const uint4& u, float* f) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t;
    if constexpr (kF16) t = __half22float2(reinterpret_cast<const __half2*>(&u)[i]);
    else t = __bfloat1622float2(reinterpret_cast<const __nv_bfloat162*>(&u)[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}

// Kernel 0's rounding points: two fp32 values rounded to the 16-bit format as one packed pair.  fp16 takes
// cvt.rn.f16x2.f32 without .satfinite (overflow -> +-inf, as .to(torch.float16)); neither form flushes subnormals.
template <bool kF16>
struct Pair16 {
  using T = __nv_bfloat162;
  static __device__ __forceinline__ T pack(float a, float b) { return __floats2bfloat162_rn(a, b); }
};
template <>
struct Pair16<true> {
  using T = __half2;
  static __device__ __forceinline__ T pack(float a, float b) {
    uint32_t u;
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(u) : "f"(b), "f"(a));  // a -> low half, b -> high half
    return *reinterpret_cast<const __half2*>(&u);
  }
};
template <bool kF16>
__device__ __forceinline__ float2 round2(float a, float b) {
  if constexpr (kF16) return __half22float2(Pair16<true>::pack(a, b));
  else return __bfloat1622float2(__floats2bfloat162_rn(a, b));
}

// Kernel 0's row transform (process_rows below): rows of one 128-token block of one head, normalised / rotated / rounded
// to the 16-bit format, stored to the destination and left in the register layout the pooling sweep uses.  The source
// rows arrive through the shared-memory ring of qkv_prep_stream_kernel; the rotary-table row of step it + 1 is requested
// before step it is computed.  Without loads issued ahead the kernel is latency-bound (first version, loads issued row
// by row: 2.1 ms at C3b, 26 % of DRAM throughput).
struct RopeRow {
  float4 c0, c1, s0, s1;
};
template <bool kCompact, int kD = 128>
__device__ __forceinline__ RopeRow load_rope(const PrepArgs& p, int r, int col, bool on) {
  RopeRow t;
  t.c0 = t.c1 = t.s0 = t.s1 = make_float4(0.f, 0.f, 0.f, 0.f);
  if (on) {
    const float4* cp = reinterpret_cast<const float4*>(p.cos + (int64_t)r * kD + col);
    if constexpr (kCompact) {
      // the thread's 8 columns are 4 pairs: (cos, sin) x 4 = 8 floats at the same offset of the kD-float row
      const float4 a = __ldg(cp), b = __ldg(cp + 1);
      t.c0 = make_float4(a.x, a.x, a.z, a.z), t.c1 = make_float4(b.x, b.x, b.z, b.z);
      t.s0 = make_float4(a.y, a.y, a.w, a.w), t.s1 = make_float4(b.y, b.y, b.w, b.w);
    } else {
      const float4* sp = reinterpret_cast<const float4*>(p.sin + (int64_t)r * kD + col);
      t.c0 = __ldg(cp), t.c1 = __ldg(cp + 1), t.s0 = __ldg(sp), t.s1 = __ldg(sp + 1);
    }
  }
  return t;
}

// kNorm: 0 none, 1 RMSNorm over head_dim, 2 RMSNorm across heads (row statistic precomputed), 3 LayerNorm over head_dim.
// kGather: rows come from peer-mapped buffers.  kCompact: one (cos, sin)-pair table.  Compile-time so that each form
// carries only its own code and registers (with all of them behind run-time flags the HunyuanVideo form lost 40 %).
// kD: head_dim.  At 64 (CogVideoX, LayerNorm only) a thread's 8 columns belong to one of two adjacent heads h, h + 1
// (see qkv_prep_stream_kernel); `heads` tells whether head h + 1 exists.  kF16: the rows, weights and biases are fp16.
// raw[it] = source row jblk * 128 + 16 warp + 2 it + (lane >> 4), columns 8 (lane & 15) .. +7 of head h (kD = 64:
// columns 8 (lane & 7) .. +7 of head h + ((lane >> 3) & 1)), zeros beyond the source: normalise / rotate / round, store
// to the destination, and leave the rounded values in raw (zeros for the lanes of a head that does not exist).
template <int kNorm, bool kCompact, bool kGather, int kD, bool kF16>
__device__ __forceinline__ void process_rows(const PrepArgs& p, int which, int b, int h, int jblk, int warp, int lane,
                                             uint4 (&raw)[8], int heads) {
  static_assert(kD == 128 || (kD == 64 && kNorm == 3), "the 64-column form is built for LayerNorm (CogVideoX) only");
  const int col = kD == 128 ? 8 * (lane & 15) : 8 * (lane & 7);
  const int hh = kD == 128 ? h : h + ((lane >> 3) & 1);
  const bool head_live = kD == 128 || hh < heads;
  __nv_bfloat16* dst = p.dst[which] + b * p.dst_stride[which][0] + hh * p.dst_stride[which][1] + col;
  const int r0 = jblk * 128 + 16 * warp + (lane >> 4);
  if (which == 2) {  // V: re-layout only
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int r = r0 + 2 * it;
      if (r < p.rows && head_live) *reinterpret_cast<uint4*>(dst + (int64_t)(p.dst_row0 + r) * p.dst_stride[which][2]) = raw[it];
    }
    return;
  }
  float wgt[8];
  // (src_head0: under the fused Ulysses gather this rank's head h is head src_head0 + h of the token's row; else 0)
  if constexpr (kNorm != 0)
    unpack8<kF16>(__ldg(reinterpret_cast<const uint4*>(p.w[which] + (p.src_head0 + h) * p.w_head_stride + col)), wgt);
  const float* rinv_rows = (kNorm == 2 && !kGather) ? p.row_rinv[which] + (int64_t)b * p.rows : nullptr;
  float bia[8];
  if constexpr (kNorm == 3) unpack8<kF16>(__ldg(reinterpret_cast<const uint4*>(p.bias[which] + col)), bia);
  RopeRow next = load_rope<kCompact, kD>(p, r0, col, r0 < p.rows && r0 < p.rope_rows);
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    const int r = r0 + 2 * it;
    const bool live = r < p.rows;
    const bool rot = live && r < p.rope_rows;
    const RopeRow t = next;
    if (it < 7) next = load_rope<kCompact, kD>(p, r + 2, col, r + 2 < p.rows && r + 2 < p.rope_rows);
    float f[8];
    unpack8<kF16>(raw[it], f);
    if constexpr (kNorm == 3) {
      // torch.nn.LayerNorm(head_dim) on a bf16 / fp16 tensor: statistics and affine in fp32, ONE rounding
      // (cogvideo :452-455; two-pass variance, fixed butterfly order over the kD / 8 lanes that share the (row, head))
      float sm = 0.f;
#pragma unroll
      for (int c = 0; c < 8; ++c) sm = __fadd_rn(sm, f[c]);
#pragma unroll
      for (int o = 1; o < kD / 8; o <<= 1) sm = __fadd_rn(sm, __shfl_xor_sync(0xffffffffu, sm, o));
      const float mean = __fmul_rn(sm, 1.0f / kD);
      float ss = 0.f;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        f[c] = __fsub_rn(f[c], mean);
        ss = __fmaf_rn(f[c], f[c], ss);
      }
#pragma unroll
      for (int o = 1; o < kD / 8; o <<= 1) ss = __fadd_rn(ss, __shfl_xor_sync(0xffffffffu, ss, o));
      const float rstd = rsqrtf(__fadd_rn(__fmul_rn(ss, 1.0f / kD), p.eps));
#pragma unroll
      for (int c = 0; c < 8; c += 2) {
        const float2 y = round2<kF16>(__fmaf_rn(wgt[c], __fmul_rn(rstd, f[c]), bia[c]),
                                      __fmaf_rn(wgt[c + 1], __fmul_rn(rstd, f[c + 1]), bia[c + 1]));
        f[c] = y.x;
        f[c + 1] = y.y;
      }
    } else if constexpr (kNorm != 0) {
      float rinv;
      if constexpr (kNorm == 2) {  // norm across heads: the row statistic was computed over all H*128 channels beforehand
        if constexpr (kGather) {  // the owning rank computed the statistic from its full rows (rsa_row_rms)
          const int tok = p.dst_row0 + r, owner = live ? tok / p.src_rows : 0;
          rinv = live ? __ldg(p.rinv_table[which * p.n_src + owner] + (int64_t)b * p.src_rows + (tok - owner * p.src_rows)) : 0.f;
        } else {
          rinv = live ? __ldg(rinv_rows + r) : 0.f;
        }
      } else {
        // mean(x^2) over the 128 channels of this head: 8 per lane, then a fixed butterfly over the 16 lanes
        float ss = 0.f;
#pragma unroll
        for (int c = 0; c < 8; ++c) ss = __fmaf_rn(f[c], f[c], ss);
#pragma unroll
        for (int o = 1; o < 16; o <<= 1) ss = __fadd_rn(ss, __shfl_xor_sync(0xffffffffu, ss, o));
        rinv = rsqrtf(__fadd_rn(__fmul_rn(ss, 1.0f / 128.0f), p.eps));
      }
#pragma unroll
      for (int c = 0; c < 8; c += 2) {  // packed conversions: one F2FP per pair, the scalar cvt runs on the XU pipe
        const float2 xn = round2<kF16>(__fmul_rn(f[c], rinv), __fmul_rn(f[c + 1], rinv));
        const float2 y = round2<kF16>(__fmul_rn(xn.x, wgt[c]), __fmul_rn(xn.y, wgt[c + 1]));
        f[c] = y.x;
        f[c + 1] = y.y;
      }
    }
    if (rot) {
      const float cs[8] = {t.c0.x, t.c0.y, t.c0.z, t.c0.w, t.c1.x, t.c1.y, t.c1.z, t.c1.w};
      const float sn[8] = {t.s0.x, t.s0.y, t.s0.z, t.s0.w, t.s1.x, t.s1.y, t.s1.z, t.s1.w};
      float g[8];
#pragma unroll
      for (int c = 0; c < 8; c += 2) {  // rotate_pairs(x)[2i] = -x[2i+1], [2i+1] = x[2i]
        g[c] = __fadd_rn(__fmul_rn(f[c], cs[c]), __fmul_rn(-f[c + 1], sn[c]));
        g[c + 1] = __fadd_rn(__fmul_rn(f[c + 1], cs[c + 1]), __fmul_rn(f[c], sn[c + 1]));
      }
#pragma unroll
      for (int c = 0; c < 8; ++c) f[c] = g[c];
    }
    typename Pair16<kF16>::T o2[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) o2[c] = Pair16<kF16>::pack(f[2 * c], f[2 * c + 1]);
    const uint4 u = *reinterpret_cast<const uint4*>(o2);
    if (live && head_live) *reinterpret_cast<uint4*>(dst + (int64_t)(p.dst_row0 + r) * p.dst_stride[which][2]) = u;
    raw[it] = live && head_live ? u : make_uint4(0, 0, 0, 0);
  }
}

// RMSNorm across heads (Wan: attn.norm_q / norm_k = RMSNorm(heads*head_dim), rectified_wan21_attn.py:423-426): one warp
// per source row computes rsqrt(mean(x^2) + eps) over all H*128 channels.  Order (replicated by the oracle): lane l
// runs one fma chain over its columns 8(l + 32 j) .. +7, j = 0, 1, ..; then a butterfly over the lanes.  kF16: fp16 rows
// (the statistic is fp32 either way).
template <bool kF16>
__global__ void __launch_bounds__(256) row_rms_kernel(const __nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ k,
                                                      int64_t qsb, int64_t qst, int64_t ksb, int64_t kst, int rows,
                                                      int inner, float eps, float* __restrict__ rq, float* __restrict__ rk) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  const int b = blockIdx.y, which = blockIdx.z;
  if (row >= rows) return;
  const __nv_bfloat16* x = which ? k + b * ksb + (int64_t)row * kst : q + b * qsb + (int64_t)row * qst;
  float ss = 0.f;
  for (int c0 = 8 * lane; c0 < inner; c0 += 256) {
    float f[8];
    unpack8<kF16>(__ldg(reinterpret_cast<const uint4*>(x + c0)), f);
#pragma unroll
    for (int c = 0; c < 8; ++c) ss = __fmaf_rn(f[c], f[c], ss);
  }
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) ss = __fadd_rn(ss, __shfl_xor_sync(0xffffffffu, ss, o));
  if (lane == 0) (which ? rk : rq)[(int64_t)b * rows + row] = rsqrtf(__fadd_rn(__fdiv_rn(ss, (float)inner), eps));
}

// ---------------------------------------------------------------------------------------------------------------
// Kernel 2 (what rsa_pool_stats launches), streaming: a CTA that requests one block, waits for it, reduces it across
// three barriers and leaves has nothing in flight for the SM while it reduces (one CTA per block reached 0.77 of the
// measured copy bandwidth at C3b).  So a persistent grid (2 CTAs per SM) walks contiguous ranges of (tensor, head,
// block) items; an otherwise idle warp keeps kPoolStages blocks in flight with bulk copies (cp.async.bulk, no tensor
// map: each row is head_dim * 2 contiguous bytes; rows of a [B, H, S, D] tensor with token stride D are one 32 KB copy)
// into a shared-memory ring, and the 256 threads reduce block i from shared memory with the thread <-> row mapping and
// summation order given at the top of this file while blocks i + 1, i + 2 land.
constexpr int kPoolStages = 3;
constexpr int kPoolStageBytes = 128 * 256;
constexpr int kPoolSmem = kPoolStages * kPoolStageBytes + 64;

// One block's statistics from its values held in registers (thread (warp, lane): rows 16 warp + 2 i + (lane >> 4),
// columns 8 (lane & 15) .. +7 as four pairs), in the summation order documented at the top of this file.  Packed fp32
// instructions (add.rn.f32x2: two independent IEEE additions per instruction, so the order per column -- the contract
// with the oracle -- is untouched): at the SM clock the part sustains under its power cap these kernels are bound by
// issue slots, not by HBM (ncu: 57 % of the issue slots at 5.8 TB/s and 1.9 GHz before this diet).
// `after_first_barrier` runs once every thread of the CTA holds its part of the block in registers.  Three barriers per
// block (two without deviations); s_part has one buffer per sweep, which saves the barrier between blocks: the next
// block writes s_part[0] (last read two barriers ago) and s_mean / s_part[1] only after its own first / second
// barrier, which every reader reaches first.
// kD = 64 (kernel 0's head pairs): columns [0, 64) are head bh's, [64, 128) head bh + 1's, which exists only when
// live_cols == 128; each head's statistics row gets exact zeros in its columns [64, 128), as kernel 2 computes them for
// 64-column heads.
template <int kD = 128, class F>
__device__ __forceinline__ void pool_block(const PoolArgs& a, const float2 (&f)[8][4], int which, int bh, int blk,
                                           float (*s_part)[8][128], float* s_mean, int tid, int warp, int lane,
                                           F&& after_first_barrier, int live_cols = 128) {
  const int col = 8 * (lane & 15);
  float2 acc[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) acc[c] = make_float2(0.f, 0.f);
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[c] = __fadd2_rn(acc[c], f[i][c]);
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    acc[c].x = __fadd_rn(acc[c].x, __shfl_xor_sync(0xffffffffu, acc[c].x, 16));
    acc[c].y = __fadd_rn(acc[c].y, __shfl_xor_sync(0xffffffffu, acc[c].y, 16));
  }
  if (lane < 16) {
    reinterpret_cast<float4*>(&s_part[0][warp][col])[0] = make_float4(acc[0].x, acc[0].y, acc[1].x, acc[1].y);
    reinterpret_cast<float4*>(&s_part[0][warp][col])[1] = make_float4(acc[2].x, acc[2].y, acc[3].x, acc[3].y);
  }
  __syncthreads();
  after_first_barrier();
  if (tid < 128) {
    float t = s_part[0][0][tid];
#pragma unroll
    for (int w = 1; w < 8; ++w) t = __fadd_rn(t, s_part[0][w][tid]);
    const float m = __fmul_rn(t, 1.0f / 128.0f);
    s_mean[tid] = m;
    if constexpr (kD == 128) {
      a.mean[which][((int64_t)bh * a.out_rows[which] + blk) * 128 + tid] = m;
    } else if (tid < live_cols) {
      float* row = a.mean[which] + ((int64_t)(bh + (tid >> 6)) * a.out_rows[which] + blk) * 128 + (tid & 63);
      row[0] = m;
      row[64] = 0.f;
    }
  }
  __syncthreads();
  if (a.mad[which] == nullptr) return;  // V: means only (uniform over the CTA)
  const float4 m0 = reinterpret_cast<const float4*>(&s_mean[col])[0], m1 = reinterpret_cast<const float4*>(&s_mean[col])[1];
  const float2 negm[4] = {make_float2(-m0.x, -m0.y), make_float2(-m0.z, -m0.w), make_float2(-m1.x, -m1.y),
                          make_float2(-m1.z, -m1.w)};
  float dev[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) dev[c] = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const float2 d2 = __fadd2_rn(f[i][c], negm[c]);  // x - mean == x + (-mean) exactly
      dev[2 * c] = __fadd_rn(dev[2 * c], fabsf(d2.x));
      dev[2 * c + 1] = __fadd_rn(dev[2 * c + 1], fabsf(d2.y));
    }
#pragma unroll
  for (int c = 0; c < 8; ++c) dev[c] = __fadd_rn(dev[c], __shfl_xor_sync(0xffffffffu, dev[c], 16));
  if (lane < 16) {
    reinterpret_cast<float4*>(&s_part[1][warp][col])[0] = make_float4(dev[0], dev[1], dev[2], dev[3]);
    reinterpret_cast<float4*>(&s_part[1][warp][col])[1] = make_float4(dev[4], dev[5], dev[6], dev[7]);
  }
  __syncthreads();
  if (tid < 128) {
    float t = s_part[1][0][tid];
#pragma unroll
    for (int w = 1; w < 8; ++w) t = __fadd_rn(t, s_part[1][w][tid]);
    if constexpr (kD == 128) {
      a.mad[which][((int64_t)bh * a.n_blk[which] + blk) * 128 + tid] = __fmul_rn(t, 1.0f / 128.0f);
    } else if (tid < live_cols) {
      float* row = a.mad[which] + ((int64_t)(bh + (tid >> 6)) * a.n_blk[which] + blk) * 128 + (tid & 63);
      row[0] = __fmul_rn(t, 1.0f / 128.0f);
      row[64] = 0.f;
    }
  }
}

template <bool kF16>
__device__ __forceinline__ void unpack_row(const uint4& u, float2 (&f)[4]) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    if constexpr (kF16) f[c] = __half22float2(*reinterpret_cast<const __half2*>(&w[c]));
    else f[c] = make_float2(__uint_as_float(w[c] << 16), __uint_as_float(w[c] & 0xffff0000u));
  }
}

struct StreamCursor {  // (tensor, head, block) walked in order without divisions
  int which, bh, blk;
  __device__ __forceinline__ void advance(const int (&per_head)[3], int n_bh) {
    const int ph = which == 0 ? per_head[0] : (which == 1 ? per_head[1] : per_head[2]);
    if (++blk == ph) {
      blk = 0;
      if (++bh == n_bh) {
        bh = 0;
        ++which;
      }
    }
  }
};

template <bool kF16>
__global__ void __launch_bounds__(kThreads, 2) pool_stats_stream_kernel(const PoolArgs a, const int n_items) {
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ __align__(16) float s_part[2][8][128];  // [sweep]: two buffers save the barrier between blocks
  __shared__ __align__(16) float s_mean[128];
  using namespace ptx;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar0 = sbase + kPoolStages * kPoolStageBytes;
  // contiguous, balanced range of items for this CTA
  const int lo = (int)((int64_t)n_items * blockIdx.x / gridDim.x), hi = (int)((int64_t)n_items * (blockIdx.x + 1) / gridDim.x);
  const int per_head[3] = {a.n_blk[0], a.n_blk[1], a.n_blk[2]};
  const int n_bh = n_items / (per_head[0] + per_head[1] + per_head[2]);
  StreamCursor cur;
  {
    const int t0 = n_bh * per_head[0], t1 = t0 + n_bh * per_head[1];
    cur.which = lo < t0 ? 0 : (lo < t1 ? 1 : 2);
    const int r = lo - (cur.which == 0 ? 0 : (cur.which == 1 ? t0 : t1));
    const int ph = cur.which == 0 ? per_head[0] : (cur.which == 1 ? per_head[1] : per_head[2]);
    cur.bh = r / ph;
    cur.blk = r - cur.bh * ph;
  }
  StreamCursor nxt = cur;  // warp 0: the next item to request
  if (tid == 0) {
    for (int s = 0; s < kPoolStages; ++s) mbar_init(bar0 + 8 * s, 1);
    fence_barrier_init();
  }
  __syncthreads();

  const int row_bytes = a.head_dim * 2;
  // rows of a block that hold data (the others pool as zeros): visual blocks end at vis_len, K / V at kv_zero_from
  auto rows_of = [&](const StreamCursor& it) {
    const int valid = it.blk < a.nq_vis ? min(a.valid_rows[it.which], a.vis_len) : a.valid_rows[it.which];
    return max(0, min(128, valid - it.blk * 128));
  };
  // warp 0 requests item `nxt` into stage n % kPoolStages
  auto issue = [&](int n) {
    const StreamCursor it = nxt;
    nxt.advance(per_head, n_bh);
    const int st = n % kPoolStages;
    const int rows = rows_of(it);
    const int shift = it.blk < a.nq_vis ? 0 : a.gap;
    const int b = it.bh / a.heads, h = it.bh - b * a.heads;
    const int64_t ts = a.stride[it.which][2];
    const __nv_bfloat16* src = a.x[it.which] + b * a.stride[it.which][0] + h * a.stride[it.which][1] +
                               (int64_t)(it.blk * 128 - shift) * ts;
    const uint32_t dst = sbase + st * kPoolStageBytes, bar = bar0 + 8 * st;
    if (lane == 0) {
      if (rows > 0) mbar_arrive_expect_tx(bar, (uint32_t)(rows * row_bytes));
      else mbar_arrive(bar);
    }
    __syncwarp();
    if (ts == 128 && a.head_dim == 128) {
      if (lane == 0 && rows > 0) bulk_load_1d(dst, src, (uint32_t)(rows * 256), bar);
    } else {
      for (int r = lane; r < rows; r += 32) bulk_load_1d(dst + r * 256, src + (int64_t)r * ts, (uint32_t)row_bytes, bar);
    }
  };
  const int n_mine = hi - lo;
  // The requests are issued by warp 7, which has nothing to do while warps 0-3 finish a block's means: after the first
  // barrier of block n every thread holds that block in registers, so its stage is free for block n + kPoolStages.
  constexpr int kIssuer = 7;
  if (warp == kIssuer)
    for (int n = 0; n < kPoolStages && n < n_mine; ++n) issue(n);

  const int col = 8 * (lane & 15);
  const int rloc = 16 * warp + (lane >> 4);  // this thread's first row inside a block; then every second row
  for (int n = 0; n < n_mine; ++n) {
    const int which = cur.which, bh = cur.bh, blk = cur.blk;
    const int nrows = rows_of(cur);
    cur.advance(per_head, n_bh);
    const int st = n % kPoolStages;
    mbar_wait(bar0 + 8 * st, (n / kPoolStages) & 1);
    const uint4* tp = reinterpret_cast<const uint4*>(smem + st * kPoolStageBytes + rloc * 256 + col * 2);
    float2 f[8][4];  // the block's values stay unpacked in registers for both sweeps
    if (nrows == 128 && a.head_dim == 128) {  // the common case: a whole block, nothing to predicate
#pragma unroll
      for (int i = 0; i < 8; ++i) unpack_row<kF16>(tp[i * 32], f[i]);
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        uint4 u = make_uint4(0, 0, 0, 0);
        if (rloc + 2 * i < nrows && col < a.head_dim) u = tp[i * 32];
        unpack_row<kF16>(u, f[i]);
      }
    }
    pool_block(a, f, which, bh, blk, s_part, s_mean, tid, warp, lane, [&]() {
      if (warp == kIssuer && n + kPoolStages < n_mine) issue(n + kPoolStages);
    });
  }
  __syncthreads();

  // text keys scored as single tokens -> fp32 rows [NQ, NQ + a) of k_cat (hunyuan :193-194): one 16-lane group per row
  const int64_t text_rows = (int64_t)n_bh * a.text_keys;
  for (int64_t t = (int64_t)blockIdx.x * (kThreads / 16) + (tid >> 4); t < text_rows; t += (int64_t)gridDim.x * (kThreads / 16)) {
    const int bh = (int)(t / a.text_keys), tk = (int)(t - (int64_t)bh * a.text_keys);
    const int b = bh / a.heads, h = bh % a.heads;
    const int tok = a.text_from + tk;
    const __nv_bfloat16* src = a.x[1] + b * a.stride[1][0] + h * a.stride[1][1] + (int64_t)tok * a.stride[1][2];
    float f[8];
    uint4 u = make_uint4(0, 0, 0, 0);
    if (tok + a.gap < a.valid_rows[1] && 8 * (tid & 15) < a.head_dim) u = *reinterpret_cast<const uint4*>(src + 8 * (tid & 15));
    unpack8<kF16>(u, f);
    float* dst = a.mean[1] + ((int64_t)bh * a.out_rows[1] + a.n_blk[1] + tk) * 128 + 8 * (tid & 15);
    reinterpret_cast<float4*>(dst)[0] = make_float4(f[0], f[1], f[2], f[3]);
    reinterpret_cast<float4*>(dst)[1] = make_float4(f[4], f[5], f[6], f[7]);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Kernel 0 (what rsa_qkv_prep / rsa_qkv_prep_gather launch).  Same structure as kernel 2:
// a persistent grid, the source rows of the next blocks in flight as 256-byte bulk copies (one per token row and head:
// the projection output is [B, rows, H*128]) into a shared-memory ring, issued by the otherwise idle warp 7; the 256
// threads take block n from shared memory into the register layout of process_rows (normalise / rotate / round /
// store) and pool the rounded values with pool_block.  For the fused Ulysses gather the sources are the peer-mapped
// buffers of the owning ranks: the copies cross NVLink with three blocks (96 KB) in flight per CTA instead of exposing
// one NVLink round trip (~4 us) per block.
// Items are ordered block-major, then tensor, then head: the 3 * B * H items of one token block read the same source
// rows (all heads of a token are contiguous) and the same rotary-table rows, which therefore stay in L1 / L2 instead
// of being streamed from HBM once per head (the table alone is as large as L2 at the HunyuanVideo size).
// kD = 64 (CogVideoX): an item is a pair of adjacent heads (h, h + 1) of one batch element, whose two 64-column slices
// are one 256-byte run of the source row -- the same copies into the same stage rows as at 128 columns.  Lanes 0-7 of
// each half-warp take head h, lanes 8-15 head h + 1; an odd head count leaves the last pair half empty (128-byte
// copies, nothing stored for the missing head).  Every lane stays busy: the kernel is bound by issue slots, and one
// head per item would idle half of them.  n_bh counts pairs then (B * ceil(H / 2)).
// kF16: fp16 rows (every form above has one); the rounding points, the copies and the pooling order are the same.
template <int kNorm, bool kGather, bool kCompact, int kD, bool kF16>
__global__ void __launch_bounds__(kThreads, 2) qkv_prep_stream_kernel(const PoolArgs a, const PrepArgs p, const int n_blocks,
                                                                      const int n_bh) {
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ __align__(16) float s_part[2][8][128];
  __shared__ __align__(16) float s_mean[128];
  using namespace ptx;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar0 = sbase + kPoolStages * kPoolStageBytes;
  const int per_blk = 3 * n_bh;
  const int n_items = n_blocks * per_blk;
  const int lo = (int)((int64_t)n_items * blockIdx.x / gridDim.x), hi = (int)((int64_t)n_items * (blockIdx.x + 1) / gridDim.x);
  struct Cursor {
    int jblk, which, bh;
  };
  auto advance = [&](Cursor& c) {
    if (++c.bh == n_bh) {
      c.bh = 0;
      if (++c.which == 3) {
        c.which = 0;
        ++c.jblk;
      }
    }
  };
  Cursor cur;
  cur.jblk = lo / per_blk;
  cur.which = (lo - cur.jblk * per_blk) / n_bh;
  cur.bh = lo - cur.jblk * per_blk - cur.which * n_bh;
  Cursor nxt = cur;
  if (tid == 0) {
    for (int s = 0; s < kPoolStages; ++s) mbar_init(bar0 + 8 * s, 1);
    fence_barrier_init();
  }
  __syncthreads();

  // Every warp requests its own 16 rows of item `nxt` (one 256-byte copy per lane 0..15) into stage n % kPoolStages;
  // thread 0 arms the barrier with the byte count of the whole block.
  auto issue = [&](int n) {
    const Cursor it = nxt;
    advance(nxt);
    const int st = n % kPoolStages;
    const int rows = max(0, min(128, p.rows - it.jblk * 128));
    const int per_b = kD == 128 ? a.heads : (a.heads + 1) >> 1;  // items per (block, tensor, batch element)
    const int b = it.bh / per_b, u = it.bh - b * per_b;
    const int h = kD == 128 ? u : 2 * u;  // (first) head of the item
    const uint32_t row_bytes = (kD == 128 || h + 1 < a.heads) ? 256u : 128u;
    const uint32_t dst = sbase + st * kPoolStageBytes, bar = bar0 + 8 * st;
    if (tid == 0) {
      if (rows > 0) mbar_arrive_expect_tx(bar, (uint32_t)rows * row_bytes);
      else mbar_arrive(bar);
    }
    const int r = 16 * warp + lane;
    if (lane < 16 && r < rows) {
      const int64_t ts = p.src_stride[it.which][1];
      const int row = it.jblk * 128 + r;
      if constexpr (!kGather) {
        bulk_load_1d(dst + r * 256, p.src[it.which] + b * p.src_stride[it.which][0] + (int64_t)h * kD + (int64_t)row * ts, row_bytes, bar);
      } else {
        const int tok = p.dst_row0 + row;  // the peer buffers hold the tokens in memory order, like the destination
        const int owner = tok / p.src_rows;
        const __nv_bfloat16* base = p.src_table[it.which * p.n_src + owner];
        bulk_load_1d(dst + r * 256, base + b * p.src_stride[it.which][0] + (int64_t)(p.src_head0 + h) * kD +
                                        (int64_t)(tok - owner * p.src_rows) * ts, row_bytes, bar);
      }
    }
  };
  const int n_mine = hi - lo;
  for (int n = 0; n < kPoolStages && n < n_mine; ++n) issue(n);

  const int col = 8 * (lane & 15);
  const int rloc = 16 * warp + (lane >> 4);
  for (int n = 0; n < n_mine; ++n) {
    const int which = cur.which, bh = cur.bh, jblk = cur.jblk;
    advance(cur);
    const int blk = p.blk0 + jblk;
    const int per_b = kD == 128 ? a.heads : (a.heads + 1) >> 1;
    const int b = bh / per_b, u = bh - b * per_b;
    const int h = kD == 128 ? u : 2 * u;
    const int bh0 = kD == 128 ? bh : b * a.heads + h;          // (first) head's row of the statistics
    const int live_cols = (kD == 128 || h + 1 < a.heads) ? 128 : 64;  // 64: head h + 1 does not exist
    const bool lane_live = kD == 128 || col < live_cols;
    const int st = n % kPoolStages;
    mbar_wait(bar0 + 8 * st, (n / kPoolStages) & 1);
    const uint4* tp = reinterpret_cast<const uint4*>(smem + st * kPoolStageBytes + rloc * 256 + col * 2);
    const int rows = p.rows - jblk * 128;  // source rows of this block (>= 1)
    uint4 raw[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      raw[i] = make_uint4(0, 0, 0, 0);
      if (rloc + 2 * i < rows && lane_live) raw[i] = tp[i * 32];
    }
    process_rows<kNorm, kCompact, kGather, kD, kF16>(p, which, b, h, jblk, warp, lane, raw, a.heads);
    const bool visual = blk < a.nq_vis;
    bool pooled = false;
    if (p.pool) {
      const int valid = visual ? min(a.valid_rows[which], a.vis_len) : a.valid_rows[which];
      const int row0 = blk * 128 + rloc;
      // rows the pooling counts as zeros (K, V rows >= kv_zero_from; hunyuan masked_fill_ :307-308) stay stored as they are
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if (row0 + 2 * i >= valid) raw[i] = make_uint4(0, 0, 0, 0);
      if (which == 1 && !visual) {
        // text keys scored as single tokens: fp32 rows [NQ, NQ + a) of k_cat (hunyuan :193-194)
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int t = (blk - a.nq_vis) * 128 + rloc + 2 * i;  // text token index
          if (t < a.text_keys && lane_live) {
            float f[8];
            unpack8<kF16>(raw[i], f);
            // kD = 64: head bh0 + (col >> 6), its columns (col & 63) .. +7, and zeros in the 64 columns it lacks
            const int row_bh = kD == 128 ? bh : bh0 + (col >> 6), row_col = kD == 128 ? col : col & 63;
            float* dstk = a.mean[1] + ((int64_t)row_bh * a.out_rows[1] + a.n_blk[1] + t) * 128 + row_col;
            reinterpret_cast<float4*>(dstk)[0] = make_float4(f[0], f[1], f[2], f[3]);
            reinterpret_cast<float4*>(dstk)[1] = make_float4(f[4], f[5], f[6], f[7]);
            if constexpr (kD == 64) {
              reinterpret_cast<float4*>(dstk + 64)[0] = make_float4(0.f, 0.f, 0.f, 0.f);
              reinterpret_cast<float4*>(dstk + 64)[1] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
          }
        }
      }
      pooled = blk < a.n_blk[which];  // uniform over the CTA
    }
    if (pooled) {
      float2 f[8][4];
#pragma unroll
      for (int i = 0; i < 8; ++i) unpack_row<kF16>(raw[i], f[i]);
      pool_block<kD>(a, f, which, bh0, blk, s_part, s_mean, tid, warp, lane, [&]() {
        if (n + kPoolStages < n_mine) issue(n + kPoolStages);
      }, live_cols);
    } else {
      __syncthreads();  // every thread has taken its rows out of the stage
      if (n + kPoolStages < n_mine) issue(n + kPoolStages);
    }
  }
}

}  // namespace

static PoolArgs pool_args(const rsa_attn_desc* d, const void* q, const void* k, const void* v, char* ws,
                          const WsLayout& L) {
  PoolArgs a;
  a.x[0] = (const __nv_bfloat16*)q;
  a.x[1] = (const __nv_bfloat16*)k;
  a.x[2] = (const __nv_bfloat16*)v;
  for (int i = 0; i < 3; ++i) {
    a.stride[0][i] = d->q_stride[i];
    a.stride[1][i] = d->k_stride[i];
    a.stride[2][i] = d->v_stride[i];
  }
  const RowMap rm = row_map(d);
  const int seq_v = d->seq + rm.gap;
  const int kvz = d->kv_zero_from < seq_v ? d->kv_zero_from : seq_v;
  a.vis_len = rm.vis_len;
  a.nq_vis = rm.nq_vis;
  a.gap = rm.gap;
  a.valid_rows[0] = seq_v;
  a.valid_rows[1] = kvz;
  a.valid_rows[2] = kvz;
  a.n_blk[0] = L.nq;
  a.n_blk[1] = L.nq;
  a.n_blk[2] = L.nb;
  a.mean[0] = (float*)(ws + L.off_q_pool);
  a.mean[1] = (float*)(ws + L.off_k_cat);
  a.mean[2] = (float*)(ws + L.off_v_pool);
  a.mad[0] = (float*)(ws + L.off_q_mad);
  a.mad[1] = (float*)(ws + L.off_k_mad);
  a.mad[2] = nullptr;
  a.out_rows[0] = L.nq;
  a.out_rows[1] = L.nkc;
  a.out_rows[2] = L.nb;
  a.heads = d->heads;
  a.head_dim = d->head_dim;
  a.text_keys = L.a;
  a.text_from = rm.vis_len;
  return a;
}

// SMs of the current device, queried once: the persistent grids of kernels 0 and 2 are two CTAs per SM.
static int sm_count(int* sms) {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    RSA_CUDA_CHECK(cudaGetDevice(&dev));
    RSA_CUDA_CHECK(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
  }
  *sms = n;
  return RSA_OK;
}

int launch_pool_stats(const rsa_attn_desc* d, const void* q, const void* k, const void* v, char* ws,
                      const WsLayout& L, cudaStream_t s) {
  const PoolArgs a = pool_args(d, q, k, v, ws, L);
  static bool configured = false;
  if (!configured) {
    RSA_CUDA_CHECK(cudaFuncSetAttribute(pool_stats_stream_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPoolSmem));
    RSA_CUDA_CHECK(cudaFuncSetAttribute(pool_stats_stream_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPoolSmem));
    // two CTAs of 100 KB each per SM: without the hint the driver may pick a smaller shared-memory carve-out that holds one
    RSA_CUDA_CHECK(cudaFuncSetAttribute(pool_stats_stream_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    RSA_CUDA_CHECK(cudaFuncSetAttribute(pool_stats_stream_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    configured = true;
  }
  int sms = 0;
  if (const int rc = sm_count(&sms); rc != RSA_OK) return rc;
  const int64_t items = (int64_t)L.bh * (2 * (int64_t)L.nq + L.nb);
  if (items == 0) return RSA_OK;
  if (items > 0x7fffffffLL) RSA_FAIL(RSA_ERR_UNSUPPORTED, "rsa_pool_stats: too many blocks");
  const int grid = (int)(items < 2 * sms ? items : 2 * sms);
  if (d->dtype == RSA_DTYPE_F16) pool_stats_stream_kernel<true><<<grid, kThreads, kPoolSmem, s>>>(a, (int)items);
  else pool_stats_stream_kernel<false><<<grid, kThreads, kPoolSmem, s>>>(a, (int)items);
  RSA_CUDA_CHECK(cudaGetLastError());
  return RSA_OK;
}

int launch_row_rms(const void* q_src, const void* k_src, int batch, int rows, int channels, const int64_t* qs,
                   const int64_t* ks, float eps, float* rq, float* rk, bool f16, cudaStream_t s) {
  dim3 g((rows + 7) / 8, batch, 2);
  auto kernel = f16 ? row_rms_kernel<true> : row_rms_kernel<false>;
  kernel<<<g, 256, 0, s>>>((const __nv_bfloat16*)q_src, (const __nv_bfloat16*)k_src, qs[0], qs[1], ks[0], ks[1], rows,
                           channels, eps, rq, rk);
  RSA_CUDA_CHECK(cudaGetLastError());
  return RSA_OK;
}

// One form of kernel 0.  Its shared-memory attributes are set on its first launch: two CTAs of 100 KB each per SM, as
// for kernel 2.
template <int kNorm, bool kGather, bool kCompact, int kD, bool kF16>
static int launch_prep_stream(const PoolArgs& a, const PrepArgs& pa, int grid, int blocks, int n_bh, cudaStream_t s) {
  auto kernel = qkv_prep_stream_kernel<kNorm, kGather, kCompact, kD, kF16>;
  static bool configured = false;
  if (!configured) {
    RSA_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPoolSmem));
    RSA_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    configured = true;
  }
  kernel<<<grid, kThreads, kPoolSmem, s>>>(a, pa, blocks, n_bh);
  RSA_CUDA_CHECK(cudaGetLastError());
  return RSA_OK;
}

// The forms of kernel 0 that are built, for each rotary-table form (kCompact) and dtype (kF16): 128 columns with norms
// 0-3 locally and norms 0-2 in gather form, 64 columns with norm 3 (LayerNorm, CogVideoX) in both.  rsa_qkv_prep and
// rsa_qkv_prep_gather (rsa_api.cu) refuse every other norm and head_dim.
template <bool kCompact, bool kF16>
static int launch_prep_form(int norm, bool gather, int head_dim, const PoolArgs& a, const PrepArgs& pa, int grid,
                            int blocks, int n_bh, cudaStream_t s) {
  if (head_dim == 64) {
    if (gather) return launch_prep_stream<3, true, kCompact, 64, kF16>(a, pa, grid, blocks, n_bh, s);
    return launch_prep_stream<3, false, kCompact, 64, kF16>(a, pa, grid, blocks, n_bh, s);
  }
  if (gather) {
    switch (norm) {
      case 1: return launch_prep_stream<1, true, kCompact, 128, kF16>(a, pa, grid, blocks, n_bh, s);
      case 2: return launch_prep_stream<2, true, kCompact, 128, kF16>(a, pa, grid, blocks, n_bh, s);
      default: return launch_prep_stream<0, true, kCompact, 128, kF16>(a, pa, grid, blocks, n_bh, s);
    }
  }
  switch (norm) {
    case 1: return launch_prep_stream<1, false, kCompact, 128, kF16>(a, pa, grid, blocks, n_bh, s);
    case 2: return launch_prep_stream<2, false, kCompact, 128, kF16>(a, pa, grid, blocks, n_bh, s);
    case 3: return launch_prep_stream<3, false, kCompact, 128, kF16>(a, pa, grid, blocks, n_bh, s);
    default: return launch_prep_stream<0, false, kCompact, 128, kF16>(a, pa, grid, blocks, n_bh, s);
  }
}

int launch_qkv_prep(const rsa_prep_desc* p, const rsa_attn_desc* d, const void* q_src, const void* k_src,
                    const void* v_src, const rsa_peer_route* route, void* q, void* k, void* v, char* ws,
                    const WsLayout* L, cudaStream_t s) {
  const RowMap rm = row_map(d);
  PrepArgs pa;
  pa.src[0] = (const __nv_bfloat16*)q_src, pa.src[1] = (const __nv_bfloat16*)k_src, pa.src[2] = (const __nv_bfloat16*)v_src;
  pa.dst[0] = (__nv_bfloat16*)q, pa.dst[1] = (__nv_bfloat16*)k, pa.dst[2] = (__nv_bfloat16*)v;
  for (int t = 0; t < 3; ++t) {
    pa.src_stride[t][0] = p->src_stride[t][0];
    pa.src_stride[t][1] = p->src_stride[t][1];
  }
  for (int i = 0; i < 3; ++i) {
    pa.dst_stride[0][i] = d->q_stride[i];
    pa.dst_stride[1][i] = d->k_stride[i];
    pa.dst_stride[2][i] = d->v_stride[i];
  }
  pa.w[0] = p->norm ? (const __nv_bfloat16*)p->q_weight : nullptr;
  pa.w[1] = p->norm ? (const __nv_bfloat16*)p->k_weight : nullptr;
  pa.w_head_stride = p->norm == 2 ? 128 : 0;
  pa.bias[0] = (const __nv_bfloat16*)p->q_bias;
  pa.bias[1] = (const __nv_bfloat16*)p->k_bias;
  pa.row_rinv[0] = pa.row_rinv[1] = nullptr;
  const bool f16 = d->dtype == RSA_DTYPE_F16;
  if (p->norm == 2 && !route) {
    float* rq = p->row_scratch;
    float* rk = rq + (int64_t)d->batch * p->rows;
    const int rc = launch_row_rms(q_src, k_src, d->batch, p->rows, d->heads * 128, p->src_stride[0], p->src_stride[1],
                                  p->eps, rq, rk, f16, s);
    if (rc != RSA_OK) return rc;
    pa.row_rinv[0] = rq;
    pa.row_rinv[1] = rk;
  }
  pa.eps = p->eps;
  pa.cos = p->cos;
  pa.sin = p->sin;
  pa.rope_compact = p->rope_compact != 0;
  pa.rope_rows = p->rope_rows;
  pa.rows = p->rows;
  pa.dst_row0 = p->dst_row;
  // destination row -> block of the padded layout: visual rows start block 0, text rows start block nq_vis
  pa.blk0 = p->dst_row == 0 ? 0 : rm.nq_vis;
  pa.pool = L != nullptr;
  pa.src_table = nullptr;
  pa.rinv_table = nullptr;
  pa.n_src = pa.src_rows = pa.src_head0 = 0;
  if (route) {
    pa.src_table = (const __nv_bfloat16* const*)route->src_table;
    pa.rinv_table = route->rinv_table;
    pa.n_src = route->n_ranks;
    pa.src_rows = route->rows_per_rank;
    pa.src_head0 = route->head0;
    for (int t = 0; t < 3; ++t) {
      pa.src_stride[t][0] = route->src_stride[0];
      pa.src_stride[t][1] = route->src_stride[1];
    }
  }
  PoolArgs a;
  if (L) {
    a = pool_args(d, q, k, v, ws, *L);
  } else {
    a = PoolArgs{};
    a.heads = d->heads;
    a.head_dim = d->head_dim;
    a.nq_vis = rm.nq_vis;
    a.vis_len = rm.vis_len;
    a.gap = rm.gap;
  }
  const int blocks = (p->rows + 127) / 128;
  const bool compact = pa.rope_compact && pa.rope_rows > 0;
  const bool hd64 = d->head_dim == 64;  // items are head pairs (qkv_prep_stream_kernel)
  const int n_bh = d->batch * (hd64 ? (d->heads + 1) / 2 : d->heads);
  const int64_t items = (int64_t)blocks * 3 * n_bh;
  if (items > 0x7fffffffLL) RSA_FAIL(RSA_ERR_UNSUPPORTED, "rsa_qkv_prep: too many blocks");
  int sms = 0;
  if (const int rc = sm_count(&sms); rc != RSA_OK) return rc;
  const int grid = (int)(items < 2 * sms ? items : 2 * sms);
  const bool gather = route != nullptr;
  if (f16) {
    if (compact) return launch_prep_form<true, true>(p->norm, gather, d->head_dim, a, pa, grid, blocks, n_bh, s);
    return launch_prep_form<false, true>(p->norm, gather, d->head_dim, a, pa, grid, blocks, n_bh, s);
  }
  if (compact) return launch_prep_form<true, false>(p->norm, gather, d->head_dim, a, pa, grid, blocks, n_bh, s);
  return launch_prep_form<false, false>(p->norm, gather, d->head_dim, a, pa, grid, blocks, n_bh, s);
}

}  // namespace rsa
