// attn_tc5.cu -- kernel 4, the product path: block-sparse attention over per-row kept-block lists on the
// 5th-generation tensor cores (tcgen05.mma, accumulators in TMEM), operands fed by TMA, with the rectification
// epilogue O = Os * R + C fused into the output write.
//
// Replaces (reference paths): _triton_block_sparse_attention_onehot + kernel (rectified_wan21_attn.py:16-168),
// the epilogue `output_normal * R + C` (:346), the flash-attn call for text query rows
// (rectified_hunyuan_attn.py:371-380; text tiles simply carry a dense list with R = 1, C = 0) and the final
// cat / permute / reshape (:383-387; the output is written straight into [B, S, H, D]).
//
// One CTA per SM works on TWO adjacent 128-row query tiles of one (batch, head) -- "slots" 0 and 1 -- each with
// its own kept-block list, its own S/P and O accumulators in TMEM (4 x 128 columns = all 512) and its own softmax
// warpgroup.  A single MMA-issuing thread alternates between the slots, so the tensor pipe runs slot 1's MMAs
// while slot 0's softmax warpgroup is busy and vice versa (two co-resident single-tile CTAs lock into phase and
// halve the throughput: measured, see DESIGN.md).  Per kept block j of a slot's list:
//     warp 0 (TMA)      K_j, V_j tiles -> 16 KB shared-memory granules (128 rows x 64 bf16, 128-byte swizzle),
//                       (two per tile = one ring stage; 5 stages shared by both slots, filled in the order the
//                       MMA warp consumes them)
//     warps 4-7 / 8-11  once per tile: q~ = dtype(q * head_dim^-1/2 * log2 e) in place in shared memory -- the
//                       reference kernel rounds the pre-scaled query to the input dtype (wan21 :61-62), and at
//                       HunyuanVideo sizes that rounding is most of what separates two correct kernels
//     warp 1 (MMA)      S = q~ K_j^T           8 x tcgen05.mma 128x128x16, A and B from shared memory
//     warps 4-7 / 8-11  S (TMEM) -> registers, running max with lazy rescale of O, p = exp2(s*c - m), row sums,
//                       P (bf16) -> TMEM over the S columns, handed over in two halves of 64 keys
//     warp 1 (MMA)      O += P V_j             8 x tcgen05.mma 128x128x16, A = P from TMEM, B = V_j (MN-major)
// and at the end of a list the slot's warpgroup reads O from TMEM, applies 1/l, R and C and stores bf16 rows.
//
// Two CTAs with consecutive grid ids form a CLUSTER (two adjacent pairs of query tiles = four adjacent tiles of a head).
// The blocks all four tiles keep lead every list (pair_schedule_kernel, rsa_api.cu); over that prefix each K / V tile is
// fetched from L2 once per cluster: CTA rank r loads the 64-column granule r and MULTICASTS it into both CTAs' rings
// (cp.async.bulk.tensor ... .multicast::cluster), both CTAs walk the prefix at the same ring positions, and a stage of
// the prefix is refilled only after both CTAs' MMAs have released it (tcgen05.commit ... .multicast::cluster onto both
// "empty" barriers).  Behind the prefix the two CTAs are independent again.
#include <cuda.h>
#include <math.h>
#include <stdlib.h>

#include "ptx_sm100.cuh"
#include "rsa_common.cuh"

namespace rsa {
namespace {

using namespace ptx;

constexpr int kThreads = 384;    // warp 0 TMA, warp 1 MMA, warp 2 TMEM alloc, warp 3 idle, warps 4-7 / 8-11 softmax
constexpr int kGranule = 16384;  // 128 rows x 64 bf16
constexpr int kStages = 5;       // K/V tiles (2 granules each) in flight, shared by both slots
constexpr int kOffQ = 0;         // Q: [slot][head_dim half] granules
constexpr int kOffRing = 4 * kGranule;
constexpr int kOffBar = kOffRing + kStages * 2 * kGranule;
constexpr int kSmemBytes = kOffBar + 256;
constexpr uint32_t kTmemCols = 512;       // S/P of slot s at [128 s, +128), O of slot s at [256 + 128 s, +128)
// Of every 4 float2 pairs of exponentials, this many are evaluated on the FMA pipe (Cody-Waite range reduction +
// degree-3 polynomial, max relative error 7.5e-5, far below the bf16 rounding of P) instead of MUFU.EX2.  On B200
// the FMA pipe turned out to be the scarcer resource for this loop, so the default is 0.
constexpr int kDefaultPolyPairs = 0;  // measured best on B200 (0: 1209, 1: 1180, 2: 1159, 3: 1066 TFLOP/s); RSA_TC5_POLY overrides

// barrier slots (8 bytes each) inside the kOffBar region
enum {
  B_QFULL = 0,   // [2]  TMA -> MMA: Q tile of the slot landed
  B_SFULL = 2,   // [2]  MMA -> softmax: S = Q K^T complete
  B_PHALF = 4,   // [2][2]  softmax -> MMA: P columns of key half 0 / 1 written (and O rescaled)
  B_OFULL = 8,   // [2]  MMA -> softmax: last P V complete
  B_QSCALED = 10,  // [2]  softmax -> MMA: Q tile of the slot pre-scaled and rounded in place (q~)
  B_KVFULL = 12,
  B_KVEMPTY = 12 + kStages,
  B_COUNT = 12 + 2 * kStages
};
static_assert(B_COUNT * 8 + 4 <= 256, "barrier region");
static_assert(kSmemBytes <= 232448, "shared memory per CTA");

// head_dim 64 instantiation: share of the exponentials on the FMA pipe (see kDefaultPolyPairs); that form has 640
// tensor-pipe cycles per kept pair against 1024 MUFU cycles, so unlike the 128-column form it is MUFU-bound
constexpr int kDefaultPolyPairs64 = 1;  // CogVideoX1.5 shape, kernel 4: 8.30 / 8.09 / 8.30 ms for 0 / 1 / 2; RSA_TC5_POLY overrides

__device__ __forceinline__ float u2f(uint32_t u) { return __uint_as_float(u); }
__device__ __forceinline__ uint32_t f2u(float f) { return __float_as_uint(f); }

// 2^x for x <= ~8 on the FMA pipe, two lanes at a time: x = n + f, n = round(x), f in [-0.5, 0.5];
// 2^f ~ c0 + f (c1 + f (c2 + f c3)); the integer n is added into the exponent field.
__device__ __forceinline__ float2 exp2_poly2(float2 x) {
  const float kMagic = 12582912.f;  // 1.5 * 2^23: adding it leaves round(x) in the low mantissa bits
  x.x = fmaxf(x.x, -125.f);
  x.y = fmaxf(x.y, -125.f);
  const float2 t = __fadd2_rn(x, make_float2(kMagic, kMagic));
  const float2 r = __fadd2_rn(t, make_float2(-kMagic, -kMagic));
  const float2 f = __ffma2_rn(r, make_float2(-1.f, -1.f), x);
  float2 p = __ffma2_rn(f, make_float2(0.05517587438225746f, 0.05517587438225746f),
                        make_float2(0.24261151254177094f, 0.24261151254177094f));
  p = __ffma2_rn(p, f, make_float2(0.6932601928710938f, 0.6932601928710938f));
  p = __ffma2_rn(p, f, make_float2(0.9999279975891113f, 0.9999279975891113f));
  p.x = __int_as_float(__float_as_int(p.x) + (__float_as_int(t.x) << 23));
  p.y = __int_as_float(__float_as_int(p.y) + (__float_as_int(t.y) << 23));
  return p;
}

// kDebug: bring-up instantiation that also dumps S / O / l / m and a clock trace of one CTA (rsa.h,
// rsa_debug_set_attention_dump); the product instantiation carries none of that code.
constexpr int kTraceBase = 33024, kTraceSteps = 64, kTraceSlots = 16;
#define RSA_TRACE(cond, step, slot)                                                                  \
  do {                                                                                               \
    if (kDebug && (cond) && (step) >= 0 && (step) < kTraceSteps)                                       \
      a.dbg[kTraceBase + (step) * kTraceSlots + (slot)] = (float)(clock64() - t0);                     \
  } while (0)

// kD: head_dim the instantiation is built for.  128: two 64-column granules per Q/K/V tile (a tensor whose head_dim is
// 64 can still run here: its tensor maps zero-fill the second granule).  64 (CogVideoX): one granule per tile, S = Q K^T
// over 4 k-steps instead of 8, O = P V as N = 64 MMAs into 64 TMEM columns -- 640 instead of 1024 tensor-pipe cycles
// per kept pair, half the K/V bytes; the softmax side is the same, so this form is MUFU-bound rather than tensor-bound.
// kDense: every query tile walks key blocks 0 .. ceil(kv_len/128) - 1 and no list, schedule, R or C is read (dense
// attention, rsa_dense_attention).  The walk is what pair_schedule_kernel makes of all-ones lists, in closed form: the
// lists are ascending, a pair of two tiles shares all of them (nsh), and partner pairs share all of them too (nq4), so
// the result is bit-identical to the listed form on an all-ones mask.
template <bool kDebug, int kPolyPairs, bool kF16 = false, int kD = 128, bool kDense = false>
__global__ void __launch_bounds__(kThreads, 1)
attn_tc5_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmQt,
                const __grid_constant__ CUtensorMap tmKt, const __grid_constant__ CUtensorMap tmVt, const AttnArgs a) {
  // tmQ/tmK/tmV cover the visual rows [0, vis_len) (rows past the end read as zeros = the padding of the last visual
  // block); tmQt/tmKt/tmVt cover the text rows, which start at memory row vis_len (RowMap, rsa_common.cuh).
  extern __shared__ __align__(1024) uint8_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // which pair of query tiles this CTA works on: attention_grid_slot (rsa_common.cuh) explains the order
  const int n_pairs = (a.nqt + 1) / 2;
  const int total_ctas = n_pairs * a.batch * a.heads;
  if ((int)blockIdx.x >= total_ctas) return;  // the grid is rounded up to whole clusters
  const GridSlot gs = attention_grid_slot((int)blockIdx.x, a.nqt, a.nq_vis, a.batch * a.heads, a.front_text_heads,
                                          (a.dbg_flags & 16) != 0);
  const int pair = gs.pair, bh = gs.bh, tile0 = gs.tile0, tile1 = gs.tile1;
  const bool repair = gs.repaired;
  const int b = bh / a.heads, h = bh % a.heads;
  const int64_t lrow0 = (int64_t)bh * a.nqt + tile0;
  // counts and prefix length are clamped so that a workspace that never saw a build (mask re-use misused) yields
  // garbage values, not an unbounded walk; out-of-range block numbers read as zero tiles through TMA
  const int ndense = kDense ? (a.kv_len + 127) / 128 : 0;
  const int cnt0 = kDense ? ndense : min(max(a.kept_cnt[lrow0], 0), a.nb);
  const int cnt1 = tile1 < a.nqt ? (kDense ? ndense : min(max(a.kept_cnt[lrow0 + 1], 0), a.nb)) : 0;
  // the pair schedule (rsa_api.cu: pair_schedule_kernel): both lists start with the nsh blocks the two tiles have in
  // common, in the same order, so over rounds [0, nsh) one K tile and one V tile serve both slots
  const uint16_t* __restrict__ list0 = kDense ? nullptr : (repair ? a.kept_idx : a.sched_idx) + lrow0 * a.nb;
  const uint16_t* __restrict__ list1 = kDense ? nullptr : list0 + a.nb;
  const int nsh = (kDense || repair) ? min(cnt0, cnt1)
                         : min(max(a.pair_shared[(int64_t)bh * n_pairs + pair], 0), min(cnt0, cnt1));
  const int rounds = max(cnt0, cnt1);
  // The common prefix of the two partner pairs (pair, pair ^ 1; see the header) is walked by every pair, but only a
  // cluster that actually holds both partners shares its K / V tiles.  Both CTAs evaluate the SAME expression on the same
  // words of the workspace -- both pairs' quad counts, pair counts and list lengths -- so they agree on nq4 whatever
  // those words hold.  (The 64-column and debug instantiations never share.)
  int nq4 = 0;
  const int vis_pairs = min(a.nq_vis, a.nqt) / 2;
  if (kD == 128 && !kDebug && !(a.dbg_flags & 32) && !repair && pair < vis_pairs && (pair ^ 1) < vis_pairs && ((int)blockIdx.x ^ 1) < total_ctas) {
    const GridSlot gp = attention_grid_slot((int)blockIdx.x ^ 1, a.nqt, a.nq_vis, a.batch * a.heads, a.front_text_heads,
                                            (a.dbg_flags & 16) != 0);
    if (kDense && !gp.repaired && gp.bh == bh && gp.pair == (pair ^ 1)) {
      nq4 = ndense;  // both pairs have two tiles (pair, pair ^ 1 < vis_pairs), so every block is common to all four
    } else if (!kDense && !gp.repaired && gp.bh == bh && gp.pair == (pair ^ 1)) {
      const int64_t prow = (int64_t)bh * a.nqt + gp.tile0;
      const int pc0 = min(max(a.kept_cnt[prow], 0), a.nb), pc1 = min(max(a.kept_cnt[prow + 1], 0), a.nb);
      const int pnsh = min(max(a.pair_shared[(int64_t)bh * n_pairs + gp.pair], 0), min(pc0, pc1));
      const int qa = a.quad_shared[(int64_t)bh * n_pairs + pair], qb = a.quad_shared[(int64_t)bh * n_pairs + gp.pair];
      if (qa == qb && qa > 0 && qa <= min(nsh, pnsh)) nq4 = qa;
    }
  }
  const int n_quad_tiles = 2 * nq4;  // ring positions [0, 2 nq4): K0, V0, K1, V1, ... of the common prefix
  const uint32_t cta_rank = nq4 > 0 ? cluster_ctarank() : 0u;

  constexpr int kG = kD / 64;                       // granules per Q/K/V tile
  constexpr uint32_t kTileBytes = kG * kGranule;
  constexpr uint32_t kIdQK = kF16 ? umma_idesc_f16(128, 128, false) : umma_idesc_bf16(128, 128, false);
  constexpr uint32_t kIdPV = kF16 ? umma_idesc_f16(128, kD, true) : umma_idesc_bf16(128, kD, true);
  const long long t0 = kDebug ? clock64() : 0;
  const bool dbg = kDebug && a.dbg != nullptr && lrow0 == 0;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar0 = sbase + kOffBar;
  auto bar = [&](int i) { return bar0 + 8u * (uint32_t)i; };
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + kOffBar + B_COUNT * 8);

  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&tmQ);
    prefetch_tensormap(&tmK);
    prefetch_tensormap(&tmV);
    if (a.nq_vis < a.nb) {
      prefetch_tensormap(&tmKt);
      prefetch_tensormap(&tmVt);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(bar(B_QFULL + s), 1);
      mbar_init(bar(B_SFULL + s), 1);
      mbar_init(bar(B_PHALF + 2 * s), 128);
      mbar_init(bar(B_PHALF + 2 * s + 1), 128);
      mbar_init(bar(B_OFULL + s), 1);
      mbar_init(bar(B_QSCALED + s), 128);
    }
    for (int i = 0; i < kStages; ++i) {
      mbar_init(bar(B_KVFULL + i), 1);
      mbar_init(bar(B_KVEMPTY + i), 2);  // two releases per use: this CTA's and the cluster partner's, or this CTA's twice
    }
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc(smem_u32((const void*)tmem_slot), kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  if (nq4 > 0) cluster_sync_all();  // the partner's barriers exist before anything of this CTA can signal them

  if (warp < 4) {
    setmaxnreg_dec<56>();
    if (warp == 0 && rounds > 0) {
      // ------------------------------------------------------------------------------------ TMA producer
      // Same deterministic order as the MMA warp: round r, slot s: V_s(r-1) then K_s(r); one ring stage = one
      // whole 128 x 128 tile (two granules, one barrier).
      if (lane == 0) {
#pragma unroll
        for (int s = 0; s < 2; ++s) {
          const int tile = s ? tile1 : tile0;
          if ((s ? cnt1 : cnt0) > 0) {
            const bool txt = tile >= a.nq_vis;
            const void* map = txt ? (const void*)&tmQt : (const void*)&tmQ;
            const int row = (txt ? tile - a.nq_vis : tile) * 128;
            mbar_arrive_expect_tx(bar(B_QFULL + s), kTileBytes);
            tma_load_4d(sbase + kOffQ + 2 * s * kGranule, map, bar(B_QFULL + s), 0, row, h, b);
            if (kG == 2) tma_load_4d(sbase + kOffQ + (2 * s + 1) * kGranule, map, bar(B_QFULL + s), 64, row, h, b);
          }
        }
      }
      int n = 0;  // stage counter: ring stage n % kStages, use n / kStages
      int mine0 = 0, mine1 = 0, prev0 = 0, prev1 = 0;
      for (int r = 0; r <= rounds; ++r) {
        if ((r & 31) == 0) {
          mine0 = (r + lane < cnt0) ? (kDense ? r + lane : (int)list0[r + lane]) : 0;
          mine1 = (r + lane < cnt1) ? (kDense ? r + lane : (int)list1[r + lane]) : 0;
        }
        const int cur0 = __shfl_sync(0xffffffffu, mine0, r & 31);
        const int cur1 = __shfl_sync(0xffffffffu, mine1, r & 31);
        if (lane == 0) {
#pragma unroll
          for (int s = 0; s < 2; ++s) {
            const int cnt = s ? cnt1 : cnt0;
#pragma unroll
            for (int t = 0; t < 2; ++t) {  // t = 0: V tile of block r-1; t = 1: K tile of block r
              const bool shared = s == 1 && (t == 0 ? r - 1 < nsh : r < nsh);  // slot 0 already loaded this tile
              if ((t == 0 ? (r >= 1 && r <= cnt) : (r < cnt)) && !shared) {
                const int blk = t == 0 ? (s ? prev1 : prev0) : (s ? cur1 : cur0);
                const bool txt = blk >= a.nq_vis;
                const int row = (txt ? blk - a.nq_vis : blk) * 128;
                const void* map = t == 0 ? (txt ? (const void*)&tmVt : (const void*)&tmV)
                                         : (txt ? (const void*)&tmKt : (const void*)&tmK);
                const int st = n % kStages;
                const uint32_t dst = sbase + kOffRing + st * 2 * kGranule;
                mbar_wait(bar(B_KVEMPTY + st), ((n / kStages) & 1) ^ 1);
                if (kDebug && (a.dbg_flags & 2) && n >= kStages) {  // ablation: no K/V traffic after the first fill
                  mbar_arrive(bar(B_KVFULL + st));
                } else if (n < n_quad_tiles) {
                  // common prefix of the cluster: this CTA fetches granule `cta_rank` for BOTH CTAs, the partner the other
                  mbar_arrive_expect_tx(bar(B_KVFULL + st), kTileBytes);
                  tma_load_4d_multicast(dst + cta_rank * kGranule, map, bar(B_KVFULL + st), 64 * (int)cta_rank, row, h, b,
                                        (uint16_t)3);
                } else {
                  mbar_arrive_expect_tx(bar(B_KVFULL + st), kTileBytes);
                  tma_load_4d(dst, map, bar(B_KVFULL + st), 0, row, h, b);
                  if (kG == 2) tma_load_4d(dst + kGranule, map, bar(B_KVFULL + st), 64, row, h, b);
                }
                ++n;
              }
            }
          }
        }
        prev0 = cur0;
        prev1 = cur1;
        __syncwarp();
      }
    } else if (warp == 1 && rounds > 0) {
      // -------------------------------------------------------------------------------------- MMA issuer
      // The whole warp walks the schedule (so every descriptor is warp-uniform); one elected lane issues.
      const bool leader = elect_one();
      int n = 0;
      int st_v0 = 0, par_v0 = 0, st_k0 = 0, par_k0 = 0;  // slot 0's stages of this round (slot 1 re-uses them when shared)
      int pos_v0 = 0, pos_k0 = 0;                        // ... and their ring positions
      // Frees the stage used at ring position `pos`: two arrivals complete a phase of its "empty" barrier.  If the stage's
      // NEXT use (pos + kStages) is a tile of the cluster's common prefix, the partner writes into it too and needs this
      // CTA's release: one arrival on each CTA's barrier; otherwise the next writer is this CTA alone: both arrivals here.
      auto release_stage = [&](int st, int pos) {
        if (pos + kStages < n_quad_tiles) {
          umma_commit_multicast(bar(B_KVEMPTY + st), (uint16_t)3);
        } else {
          umma_commit(bar(B_KVEMPTY + st));
          umma_commit(bar(B_KVEMPTY + st));
        }
      };
      for (int r = 0; r <= rounds; ++r) {
#pragma unroll
        for (int s = 0; s < 2; ++s) {
          const int cnt = s ? cnt1 : cnt0;
          const uint32_t tS = tmem + 128 * s, tO = tmem + 256 + 128 * s;
          const bool do_pv = r >= 1 && r <= cnt, do_qk = r < cnt;
          if (do_pv) {
            // O += P V for block r-1; key halves (P columns) in the order the softmax warpgroup releases them.
            // V's head_dim halves are the two granules of the stage: one N = 128 MN-major descriptor, LBO 16 KB.
            const bool reuse = s == 1 && r - 1 < nsh;  // V tile shared with slot 0
            const int st = reuse ? st_v0 : n % kStages;
            const int par = reuse ? par_v0 : (n / kStages) & 1;
            const int pos = reuse ? pos_v0 : n;
            if (!reuse) ++n;
            if (s == 0) st_v0 = st, par_v0 = par, pos_v0 = pos;
            const bool release = !(s == 0 && r - 1 < nsh);  // the last user frees the stage
            const uint64_t vd = smem_desc_sw128(sbase + kOffRing + st * 2 * kGranule, kGranule);
            RSA_TRACE(dbg && s == 0 && leader, r - 1, 10);
            mbar_wait(bar(B_KVFULL + st), par);
            RSA_TRACE(dbg && s == 0 && leader, r - 1, 13);
            mbar_wait(bar(B_PHALF + 2 * s), (r - 1) & 1);
            tc_fence_after();
            RSA_TRACE(dbg && s == 0 && leader, r - 1, 9);
            if (leader) {
#pragma unroll
              for (int ks = 0; ks < 4; ++ks)  // 16 keys = 16 rows of 128 B; P: 16 bf16 = 8 TMEM columns
                umma_ts(tO, tS + ks * 8, vd + 128 * ks, kIdPV, (r > 1 || ks > 0) ? 1u : 0u);
            }
            mbar_wait(bar(B_PHALF + 2 * s + 1), (r - 1) & 1);
            tc_fence_after();
            if (leader) {
#pragma unroll
              for (int ks = 4; ks < 8; ++ks) umma_ts(tO, tS + ks * 8, vd + 128 * ks, kIdPV, 1u);
              if (release) release_stage(st, pos);
              if (r == cnt) umma_commit(bar(B_OFULL + s));
            }
            RSA_TRACE(dbg && s == 0 && leader, r - 1, 11);
          }
          if (do_qk) {
            // S = Q K^T for block r: head_dim halves 0 / 1 = granules 0 / 1 of the stage (and of Q)
            const bool reuse = s == 1 && r < nsh;  // K tile shared with slot 0
            const int st = reuse ? st_k0 : n % kStages;
            const int par = reuse ? par_k0 : (n / kStages) & 1;
            const int pos = reuse ? pos_k0 : n;
            if (!reuse) ++n;
            if (s == 0) st_k0 = st, par_k0 = par, pos_k0 = pos;
            const bool release = !(s == 0 && r < nsh);
            const uint64_t kd = smem_desc_sw128(sbase + kOffRing + st * 2 * kGranule);
            const uint64_t qd = smem_desc_sw128(sbase + kOffQ + 2 * s * kGranule);
            if (r == 0) mbar_wait(bar(B_QSCALED + s), 0);
            RSA_TRACE(dbg && s == 0 && leader, r, 14);
            mbar_wait(bar(B_KVFULL + st), par);
            tc_fence_after();
            RSA_TRACE(dbg && s == 0 && leader, r, 12);
            if (leader) {
#pragma unroll
              for (int ks = 0; ks < kD / 16; ++ks) {  // 16 head_dim elements = 32 bytes inside the swizzle atom
                const uint32_t off = (ks >> 2) * (kGranule >> 4) + 2 * (ks & 3);
                umma_ss(tS, qd + off, kd + off, kIdQK, ks != 0);
              }
              if (release) release_stage(st, pos);
              umma_commit(bar(B_SFULL + s));
            }
            RSA_TRACE(dbg && s == 0 && leader, r, 8);
          }
          __syncwarp();
        }
      }
    }
  } else {
    // ------------------------------------------------------------------- softmax + epilogue warpgroups
    setmaxnreg_inc<224>();
    const int s = (warp - 4) >> 2;  // slot
    const int quarter = warp & 3;   // TMEM lanes [32*quarter, +32) belong to this warp
    const int row = quarter * 32 + lane;
    const int tile = s ? tile1 : tile0;
    const int cnt = s ? cnt1 : cnt0;
    const uint16_t* __restrict__ list = s ? list1 : list0;
    const int64_t lrow = lrow0 + s;
    const uint32_t tS = tmem + 128 * s + ((uint32_t)(quarter * 32) << 16);
    const uint32_t tO = tS + 256;
    float m_ref = -INFINITY, l = 0.f;
    const bool tr = dbg && s == 0 && row == 0;
    // Visual tiles follow the reference's Triton kernel, which rounds the pre-scaled query to the input dtype
    // (q~ = dtype(q * sm_scale * log2 e), wan21 :61-62) so that S leaves the tensor core in the log2 domain; text tiles
    // follow its flash-attn call (hunyuan :371-380), which scales S in fp32 instead.
    const bool prescale = a.q_round != 0 && tile < a.nq_vis;
    const float scale = prescale ? 1.f : a.scale_log2;
    const float2 scale2 = make_float2(scale, scale);

    if (tile < a.nqt) {
      if (cnt > 0) {
        mbar_wait(bar(B_QFULL + s), 0);
        if (prescale) {
          // in place in shared memory; element-wise, so the swizzle does not matter: 128 threads x 16 bytes per step
          uint4* qt = reinterpret_cast<uint4*>(smem + kOffQ + 2 * s * kGranule) + (threadIdx.x - 128 - 128 * s);
#pragma unroll 4
          for (int i = 0; i < (int)(kTileBytes / 2048); ++i) {
            uint4 x = qt[i * 128];
            x.x = scale_x2<kF16>(x.x, a.scale_log2);
            x.y = scale_x2<kF16>(x.y, a.scale_log2);
            x.z = scale_x2<kF16>(x.z, a.scale_log2);
            x.w = scale_x2<kF16>(x.w, a.scale_log2);
            qt[i * 128] = x;
          }
          fence_proxy_async_smem();
        }
        mbar_arrive(bar(B_QSCALED + s));
      }
      for (int i = 0; i < cnt; ++i) {
        RSA_TRACE(tr, i, 0);
        // valid keys in this block (the schedule is not ascending): the end of the valid keys, and the end of the
        // visual tokens inside the last visual block (zero rows that pad it are never attended)
        const int blk = kDense ? i : (int)list[i];
        int lim = a.kv_len - blk * 128;
        if (blk < a.nq_vis) lim = min(lim, a.vis_len - blk * 128);
        mbar_wait(bar(B_SFULL + s), i & 1);
        tc_fence_after();
        RSA_TRACE(tr, i, 1);
        if (kDebug && (a.dbg_flags & 1)) {  // ablation: no softmax work, hand P (garbage) straight back
          tc_fence_before();
          mbar_arrive(bar(B_PHALF + 2 * s));
          mbar_arrive(bar(B_PHALF + 2 * s + 1));
          continue;
        }
        uint32_t sr[128];
        tmem_ld32(tS + 0, sr + 0);
        tmem_ld32(tS + 32, sr + 32);
        tmem_wait_ld();
        tmem_ld32(tS + 64, sr + 64);  // in flight while the first half is reduced
        tmem_ld32(tS + 96, sr + 96);
        const bool partial = lim < 128;  // keys >= kv_len -> -inf (wan21 :75-87); at most two blocks of a list
        if (partial) {
#pragma unroll
          for (int c = 0; c < 64; ++c)
            if (c >= lim) sr[c] = 0xff800000u;
        }
        float mx0 = u2f(sr[0]), mx1 = u2f(sr[1]), mx2 = u2f(sr[2]), mx3 = u2f(sr[3]);
#pragma unroll
        for (int c = 4; c < 64; c += 4) {
          mx0 = fmaxf(mx0, u2f(sr[c]));
          mx1 = fmaxf(mx1, u2f(sr[c + 1]));
          mx2 = fmaxf(mx2, u2f(sr[c + 2]));
          mx3 = fmaxf(mx3, u2f(sr[c + 3]));
        }
        tmem_wait_ld();
        RSA_TRACE(tr, i, 2);
        if (kDebug && dbg && s == 0 && i == 0) {
#pragma unroll
          for (int c = 0; c < 128; ++c) a.dbg[row * 128 + c] = u2f(sr[c]);
        }
        if (partial) {
#pragma unroll
          for (int c = 64; c < 128; ++c)
            if (c >= lim) sr[c] = 0xff800000u;
        }
#pragma unroll
        for (int c = 64; c < 128; c += 4) {
          mx0 = fmaxf(mx0, u2f(sr[c]));
          mx1 = fmaxf(mx1, u2f(sr[c + 1]));
          mx2 = fmaxf(mx2, u2f(sr[c + 2]));
          mx3 = fmaxf(mx3, u2f(sr[c + 3]));
        }
        const float mx_s = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3)) * scale;
        if (i == 0) {
          m_ref = mx_s;
        } else {
          const bool need = mx_s > m_ref + a.rescale_thr;
          if (__any_sync(0xffffffffu, need)) {  // tcgen05.ld/st are warp-collective: rescale the warp's 32 rows
            const float alpha = need ? ex2(m_ref - mx_s) : 1.f;
            const float2 alpha2 = make_float2(alpha, alpha);
            if (need) m_ref = mx_s;
            l *= alpha;
#pragma unroll
            for (int c4 = 0; c4 < kD / 32; ++c4) {
              uint32_t o[32];
              tmem_ld32(tO + c4 * 32, o);
              tmem_wait_ld();
#pragma unroll
              for (int j = 0; j < 32; j += 2) {
                const float2 v = __fmul2_rn(make_float2(u2f(o[j]), u2f(o[j + 1])), alpha2);
                o[j] = f2u(v.x);
                o[j + 1] = f2u(v.y);
              }
              tmem_st32(tO + c4 * 32, o);
            }
          }
        }
        RSA_TRACE(tr, i, 3);
        const float2 negm2 = make_float2(-m_ref, -m_ref);
        float2 la = make_float2(0.f, 0.f), lb = make_float2(0.f, 0.f);
#pragma unroll
        for (int c16 = 0; c16 < 4; ++c16) {  // 32 S columns -> 16 packed P columns
          uint32_t pk[16];
#pragma unroll
          for (int j = 0; j < 32; j += 8) {
            float2 x[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int c = c16 * 32 + j + 2 * e;
              x[e] = __ffma2_rn(make_float2(u2f(sr[c]), u2f(sr[c + 1])), scale2, negm2);
            }
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              if (e >= 4 - kPolyPairs) {
                x[e] = exp2_poly2(x[e]);
              } else {
                x[e].x = ex2(x[e].x);
                x[e].y = ex2(x[e].y);
              }
            }
            la = __fadd2_rn(la, __fadd2_rn(x[0], x[1]));
            lb = __fadd2_rn(lb, __fadd2_rn(x[2], x[3]));
#pragma unroll
            for (int e = 0; e < 4; ++e) pk[j / 2 + e] = pack_x2<kF16>(x[e].x, x[e].y);
          }
          tmem_st16(tS + c16 * 16, pk);
          if (c16 & 1) {  // 64 keys done: hand this half of P to the MMA thread
            tmem_wait_st();
            tc_fence_before();
            mbar_arrive(bar(B_PHALF + 2 * s + (c16 >> 1)));
            if (c16 == 1) RSA_TRACE(tr, i, 4);
          }
        }
        la = __fadd2_rn(la, lb);
        l += la.x + la.y;
        RSA_TRACE(tr, i, 5);
      }

      // ---------------------------------------------------------------------------------------- epilogue
      const float R = a.R ? a.R[lrow] : 1.f;
      const float inv = l > 0.f ? R / l : 0.f;
      const float* __restrict__ crow = a.C ? a.C + lrow * 128 : nullptr;
      const int grow = tile * 128 + row;                            // row in the padded layout
      const int mrow = tile < a.nq_vis ? grow : grow - a.gap;       // row in memory
      const bool store = tile < a.nq_vis ? grow < min(a.vis_len, a.seq_q) : mrow < a.seq_q;
      const bool zero = grow >= a.q_valid;
      __nv_bfloat16* orow;
      if (a.o_table == nullptr) {
        orow = a.o + b * a.os[0] + h * a.os[1] + (int64_t)mrow * a.os[2];
      } else {  // fused Ulysses scatter: the row belongs to rank mrow / peer_rows; store into its buffer over NVLink
        const int owner = store ? mrow / a.peer_rows : 0;  // rows that are not stored must not index past the table
        orow = a.o_table[owner] + b * a.peer_os[0] +
               (int64_t)(mrow - owner * a.peer_rows) * a.peer_os[1] + (a.peer_head0 + h) * kD;
      }
      if (cnt > 0) {
        mbar_wait(bar(B_OFULL + s), 0);
        tc_fence_after();
      }
#pragma unroll
      for (int c4 = 0; c4 < kD / 32; ++c4) {
        uint32_t o[32];
        if (cnt > 0) {
          tmem_ld32(tO + c4 * 32, o);
          tmem_wait_ld();
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) o[j] = 0u;
        }
        if (kDebug && dbg && s == 0) {
#pragma unroll
          for (int j = 0; j < 32; ++j) a.dbg[16384 + row * 128 + c4 * 32 + j] = u2f(o[j]);
          if (c4 == 0) {
            a.dbg[32768 + row] = l;
            a.dbg[32768 + 128 + row] = m_ref;
          }
        }
        if (store && c4 * 32 < a.head_dim) {
#pragma unroll
          for (int j = 0; j < 32; j += 8) {
            uint32_t w[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int c = c4 * 32 + j + 2 * e;
              const float c0 = crow ? crow[c] : 0.f, c1 = crow ? crow[c + 1] : 0.f;
              w[e] = zero ? 0u : pack_x2<kF16>(fmaf(u2f(o[j + 2 * e]), inv, c0), fmaf(u2f(o[j + 2 * e + 1]), inv, c1));
            }
            *reinterpret_cast<uint4*>(orow + c4 * 32 + j) = make_uint4(w[0], w[1], w[2], w[3]);
          }
        }
      }
    }
    tc_fence_before();
  }

  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem, kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

// [batch, heads, rows, 128] bf16 view with element strides st = (batch, head, row) -> 4-D tensor map whose box is
// one granule: 64 head_dim elements x 128 rows, 128-byte swizzle; rows past the end read as zeros (the
// reference zero-pads to a multiple of 128, rectified_wan21_attn.py:299-302).
// cuTensorMapEncodeTiled costs ~10 us on the host and a launch needs up to six maps: at C1 sizes that was most of the
// call.  A tensor map is a pure function of (base, shape, strides, dtype), so the encoded maps are kept in a small
// per-thread table keyed by exactly those values (SURVEY 8b: "a TMA-descriptor cache keyed by (ptr, shape)"); a layer
// that calls with the same tensors or the same allocator addresses every step never encodes again.
struct MapKey {
  const void* base;
  int batch, heads, rows, head_dim, f16;
  int64_t st[3];
  bool operator==(const MapKey& o) const {
    return base == o.base && batch == o.batch && heads == o.heads && rows == o.rows && head_dim == o.head_dim &&
           f16 == o.f16 && st[0] == o.st[0] && st[1] == o.st[1] && st[2] == o.st[2];
  }
};
constexpr int kMapCacheSize = 32;
struct MapCache {
  MapKey key[kMapCacheSize];
  CUtensorMap map[kMapCacheSize];
  int used = 0, next = 0;
};

int make_map(CUtensorMap* m, const __nv_bfloat16* base, int batch, int heads, int rows, const int64_t* st, bool f16,
             int head_dim) {
  static thread_local MapCache cache;
  const MapKey key{base, batch, heads, rows, head_dim, f16 ? 1 : 0, {st[0], st[1], st[2]}};
  for (int i = 0; i < cache.used; ++i)
    if (cache.key[i] == key) {
      *m = cache.map[i];
      return RSA_OK;
    }
  EncodeTiledFn fn = encode_fn();
  if (!fn) RSA_FAIL(RSA_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
  if ((uintptr_t)base % 16) RSA_FAIL(RSA_ERR_UNSUPPORTED, "q/k/v must be 16-byte aligned");
  // head_dim 64: the second 64-column granule of every tile lies outside the tensor and is zero-filled by TMA
  cuuint64_t dims[4] = {(cuuint64_t)head_dim, (cuuint64_t)rows, (cuuint64_t)heads, (cuuint64_t)batch};
  int64_t sr = st[2], sh = st[1], sb = st[0];
  if (sr < head_dim) RSA_FAIL(RSA_ERR_UNSUPPORTED, "token stride must be >= head_dim");
  if (heads == 1 && sh == 0) sh = sr * rows;  // a size-1 dimension's stride is never used but must be valid
  if (batch == 1 && sb == 0) sb = sh * heads > sr * rows ? sh * heads : sr * rows;
  if (sh <= 0 || sb <= 0) RSA_FAIL(RSA_ERR_UNSUPPORTED, "head/batch strides must be positive");
  cuuint64_t strides[3] = {(cuuint64_t)sr * 2, (cuuint64_t)sh * 2, (cuuint64_t)sb * 2};
  cuuint32_t box[4] = {64, 128, 1, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = fn(m, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, (void*)base, dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) RSA_FAIL(RSA_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  const int slot = cache.used < kMapCacheSize ? cache.used++ : (cache.next++ % kMapCacheSize);
  cache.key[slot] = key;
  cache.map[slot] = *m;
  return RSA_OK;
}

struct Maps {
  CUtensorMap q, k, v, qt, kt, vt;
};

template <bool kDebug, int kPolyPairs, bool kF16 = false, int kD = 128, bool kDense = false>
int launch(dim3 grid, cudaStream_t s, const Maps& m, const AttnArgs& a) {
  static bool configured = false;  // one flag per instantiation
  if (!configured) {
    RSA_CUDA_CHECK(cudaFuncSetAttribute(attn_tc5_kernel<kDebug, kPolyPairs, kF16, kD, kDense>,
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    configured = true;
  }
  // clusters of two CTAs (consecutive ids): the grid is rounded up to a whole number of them
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((grid.x + 1) / 2 * 2);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = kSmemBytes;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (a.dbg_flags & 32) ? 1 : 2;  // flag 32 (A/B): no clusters, no quad prefix = the round-1 kernel
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  RSA_CUDA_CHECK(cudaLaunchKernelEx(&cfg, attn_tc5_kernel<kDebug, kPolyPairs, kF16, kD, kDense>, m.q, m.k, m.v, m.qt, m.kt, m.vt, a));
  return RSA_OK;
}

int poly_pairs(int dflt = kDefaultPolyPairs) {
  static int v = -2;
  if (v == -2) {
    const char* e = getenv("RSA_TC5_POLY");
    v = (e && e[0] >= '0' && e[0] <= '4' && !e[1]) ? e[0] - '0' : -1;
  }
  return v >= 0 ? v : dflt;
}

// The list-free dense form (kDense): flash-attn's arithmetic (q_round = 0), default polynomial setting, no debug dump.
// With attention flag 4 a 64-column tensor runs the 128-column form, as in launch_attention_tc5.
static int launch_dense(const Maps& m, const AttnArgs& a, cudaStream_t s) {
  const dim3 grid((unsigned)((a.nqt + 1) / 2) * (unsigned)(a.batch * a.heads));
  if (a.head_dim == 64 && !(a.dbg_flags & 4))
    return a.f16 ? launch<false, kDefaultPolyPairs64, true, 64, true>(grid, s, m, a)
                 : launch<false, kDefaultPolyPairs64, false, 64, true>(grid, s, m, a);
  return a.f16 ? launch<false, kDefaultPolyPairs, true, 128, true>(grid, s, m, a)
               : launch<false, kDefaultPolyPairs, false, 128, true>(grid, s, m, a);
}

}  // namespace

int launch_attention_tc5(const AttnArgs& a, cudaStream_t s, bool dense) {
  if (a.nqt == 0) return RSA_OK;
  Maps m;
  int rc;
  // visual rows [0, vis) and text rows [vis, seq) of each tensor (RowMap); without a text segment the text maps are
  // never used and simply repeat the visual ones
  const int vis_q = a.vis_len < a.seq_q ? a.vis_len : a.seq_q, vis_kv = a.vis_len < a.seq_kv ? a.vis_len : a.seq_kv;
  if ((rc = make_map(&m.q, a.q, a.batch, a.heads, vis_q, a.qs, a.f16 != 0, a.head_dim)) != RSA_OK) return rc;
  if ((rc = make_map(&m.k, a.k, a.batch, a.heads, vis_kv, a.ks, a.f16 != 0, a.head_dim)) != RSA_OK) return rc;
  if ((rc = make_map(&m.v, a.v, a.batch, a.heads, vis_kv, a.vs, a.f16 != 0, a.head_dim)) != RSA_OK) return rc;
  m.qt = m.q, m.kt = m.k, m.vt = m.v;
  if (a.seq_q > vis_q && (rc = make_map(&m.qt, a.q + (int64_t)vis_q * a.qs[2], a.batch, a.heads, a.seq_q - vis_q, a.qs, a.f16 != 0, a.head_dim)) != RSA_OK) return rc;
  if (a.seq_kv > vis_kv) {
    if ((rc = make_map(&m.kt, a.k + (int64_t)vis_kv * a.ks[2], a.batch, a.heads, a.seq_kv - vis_kv, a.ks, a.f16 != 0, a.head_dim)) != RSA_OK) return rc;
    if ((rc = make_map(&m.vt, a.v + (int64_t)vis_kv * a.vs[2], a.batch, a.heads, a.seq_kv - vis_kv, a.vs, a.f16 != 0, a.head_dim)) != RSA_OK) return rc;
  }
  if (dense) return launch_dense(m, a, s);
  const dim3 grid((unsigned)((a.nqt + 1) / 2) * (unsigned)(a.batch * a.heads));
  if (a.head_dim == 64 && !a.dbg && !(a.dbg_flags & 4)) {  // the 64-column instantiations (the debug kernel stays 128 wide)
    if (a.f16) return launch<false, kDefaultPolyPairs64, true, 64>(grid, s, m, a);
    switch (poly_pairs(kDefaultPolyPairs64)) {
      case 1: return launch<false, 1, false, 64>(grid, s, m, a);
      case 2: return launch<false, 2, false, 64>(grid, s, m, a);
      default: return launch<false, 0, false, 64>(grid, s, m, a);
    }
  }
  if (a.f16) return a.dbg ? launch<true, kDefaultPolyPairs, true>(grid, s, m, a) : launch<false, kDefaultPolyPairs, true>(grid, s, m, a);
  if (a.dbg) return poly_pairs() == 1 ? launch<true, 1>(grid, s, m, a) : poly_pairs() == 2 ? launch<true, 2>(grid, s, m, a) : launch<true, kDefaultPolyPairs>(grid, s, m, a);
  switch (poly_pairs()) {
    case 1: return launch<false, 1>(grid, s, m, a);
    case 3: return launch<false, 3>(grid, s, m, a);
    case 4: return launch<false, 4>(grid, s, m, a);
    case 2: return launch<false, 2>(grid, s, m, a);
    default: return launch<false, 0>(grid, s, m, a);
  }
}

}  // namespace rsa
