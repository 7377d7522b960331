// Full-vocabulary evaluation on the 5th-gen tensor cores with the [R, V] score matrix never written
// (ADER.py:99-103 `pred_last = argsort(argsort(-test_logits))` + util.py:323-339: the metrics only read
// rank(gt) = #{j : s_j > s_gt} + #{j < gt : s_j == s_gt}).
//
// Filter and refine -- ranks come out IDENTICAL to the exact fp32 path (ader_eval_rank_topk):
//   1. exact anchor: s_gt[i] = the fp32 score of the ground-truth item, computed with the very fmaf chain of the exact
//      logits kernel (sgemm.cu: acc = fmaf(a_k, b_k, acc), k ascending), one thread per row;
//   2. tcgen05 pass: approximate scores S~ = rep . E^T from a two-term bf16 split of both operands
//      (x = x_hi + x_lo + r, |r| <= 2^-18 |x|) as three products hi.hi + hi.lo + lo.hi accumulated in one TMEM tile:
//      |S~_ij - s_ij| <= eps_i := C_ERR * ||rep_i|| * max_j ||E_j||  (split remainder 1.2e-5, fp32 accumulation of 480
//      terms and the exact path's own rounding together stay below 1e-4 of sum |a_k b_k| <= ||a|| ||b||; C_ERR = 2^-12);
//      the epilogue counts  S~_ij > s_gt + eps_i  (certainly above) and appends the few columns with
//      |S~_ij - s_gt| <= eps_i to a per-row candidate list;
//   3. refine: candidates are re-scored with the exact fmaf chain and compared exactly (ties -> lower index first).
// A row whose candidate list overflows (CAP entries) raises the overflow flag; the host then takes the exact path.
//
// Operands: hi | lo halves side by side in one row-major bf16 matrix [rows][320] (320 = 5 swizzle spans of 64: the
// span that holds hi[128..159] also holds lo[0..31], so a tile is 5 regions instead of 6).  Tiles reach shared memory by
// TMA (SWIZZLE_128B) and are K-major UMMA operands; a k-step of either half is addressed by its column.
//   X (stationary): 128 rows of rep      = 5 regions x 16 KB = 80 KB
//   Y (streamed)  :  64 rows of the table = 5 regions x  8 KB = 40 KB, ring of 3
//   S tile 128 x 64 fp32 in TMEM (2 buffers x 64 columns), 30 MMAs (M = 128, N = 64, K = 16) per tile.
// Work: CTA = (row tile, vocabulary chunk); counts are merged with integer atomics (order independent).
//
// Log-sum-exp (the normaliser of the next-item softmax, ADER.py:91-93): the same pass keeps a running (max, sum exp) of
// its row per (chunk, column half) over the approximate scores of items 1..V, and k_lse_merge combines a row's slots in a
// fixed order.  Every S~ is within eps_i of s, so |lse~ - lse| <= eps_i plus the rounding of the sums.
#include "tc_common.cuh"
#include <limits.h>
#include <stdlib.h>

namespace ader {
namespace ev {
using namespace ader::tc;

constexpr int D2 = 320;                 // hi | lo columns of the operand matrices
constexpr int HALF = 160;               // column of lo[0]
static_assert(HALF == PATH_TC_MAX_D, "ADER_PATH_EVAL_TC: rows of d <= HALF columns");
constexpr int NREG = 5;
constexpr int XREG = 128 * 128, YREG = 64 * 128;
constexpr int XBYTES = NREG * XREG, YBYTES = NREG * YREG;
constexpr int NST = 3;
constexpr int TM = 128, TN = 64;
constexpr int NTHREADS = 320, NEPI = 256;
constexpr int SMEM_EVAL = 1024 + XBYTES + NST * YBYTES + 256;
constexpr float C_ERR = 1.0f / 4096.0f;

struct EvalArgs {
  int R, V, n_mtiles, n_vtiles, n_chunks;
  const float* lo_thr;       // [R] s_gt - eps
  const float* hi_thr;       // [R] s_gt + eps
  int* above;                // [R] certainly-above count (atomicAdd)
  int* cand_cnt;             // [R]
  int* cand;                 // [R][cap]
  int cap;
  int* flags;                // [0] candidate overflow, [1] pipeline timeout
  // top-k
  float* maxbuf;             // MS: [n_chunks * 2 * MS][R] the MS largest approximate scores of each (chunk, column half) of a row
  const float* lo_topk;      // CAND: [R] columns with S~ >= lo_topk[i] are top-k candidates
  int* tk_cnt;               // [R]
  int* tk_cand;              // [R][cap]
  // EXCL: columns never scored for a row (a recommended session's own items)
  const int* excl;           // [R][EXCL_W] ascending, distinct
  const int* excl_cnt;       // [R]
};
constexpr int EXCL_W = 64;              // a session holds at most maxlen <= 64 items

// fp32 rows -> [rows_pad][320] bf16 (hi | lo), optional row norms and their maximum (as int bits of a non-negative float)
__global__ void __launch_bounds__(256) k_pack_hilo(const float* __restrict__ src, long long ld, int n_rows, int d, int rows_pad,
                                                   __nv_bfloat16* __restrict__ out, float* __restrict__ norm, int* __restrict__ max_norm) {
  const int row = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (row >= rows_pad) return;
  float ss = 0.f;
  for (int c = lane; c < HALF; c += 32) {
    float x = 0.f;
    if (row < n_rows && c < d) x = src[(long long)row * ld + c];
    const __nv_bfloat16 h = __float2bfloat16_rn(x);
    const __nv_bfloat16 l = __float2bfloat16_rn(x - __bfloat162float(h));
    out[(long long)row * D2 + c] = h;
    out[(long long)row * D2 + HALF + c] = l;
    ss = fmaf(x, x, ss);
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  if (lane == 0 && row < n_rows) {
    const float nrm = sqrtf(ss) * 1.0001f;            // rounding of the norm itself must not shrink the bound
    if (norm) norm[row] = nrm;
    if (max_norm) atomicMax(max_norm, __float_as_int(nrm));
  }
}

// exact score of the ground-truth item (the fmaf chain of sgemm.cu) and the certainty band around it
__global__ void __launch_bounds__(256) k_gt_band(const float* __restrict__ table1, const float* __restrict__ rep, const int* __restrict__ gt,
                                                 int R, int d, const float* __restrict__ rnorm, const int* __restrict__ max_norm,
                                                 float* __restrict__ sg, float* __restrict__ lo_thr, float* __restrict__ hi_thr) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= R) return;
  const float* a = rep + (long long)i * d;
  const float* b = table1 + (long long)(gt[i] - 1) * d;
  float acc = 0.f;
  for (int k = 0; k < d; ++k) acc = fmaf(a[k], b[k], acc);
  const float eps = C_ERR * rnorm[i] * __int_as_float(*max_norm);
  sg[i] = acc; lo_thr[i] = acc - eps; hi_thr[i] = acc + eps;
}

// K-major SW128 descriptor of the 16-column k-step that starts at matrix column `col` of a tile whose regions are `reg` bytes
__device__ __forceinline__ uint64_t desc_col(uint32_t base, int col, int reg) {
  return make_desc_sw128(base + (col >> 6) * reg + (col & 63) * 2, 16, 1024);
}

// One pass over the [R, V] approximate scores; its epilogue does what the template parameters ask of each eligible column:
//   RANK: count the columns certainly above the row's anchor (S~ > hi_thr) and append those in [lo_thr, hi_thr] to cand;
//   CAND: append the columns with S~ >= lo_topk to tk_cand;
//   MS:   keep the MS largest scores of every (chunk, column half) of a row, sorted in registers, in maxbuf (0: none);
//   EXCL: the row's excl list is left out (a column is eligible when it is an item and not excluded);
//   LSE:  keep (max, sum exp(S~ - max)) of every (chunk, column half) of a row in lse_part [n_chunks * 2][R].
// lse_part is a parameter of its own behind the tensor maps, so EvalArgs and the maps sit at the same offsets in every
// instance.
template <bool RANK, bool CAND, int MS, bool EXCL, bool LSE>
__global__ void __launch_bounds__(NTHREADS, 1) k_eval_tc(EvalArgs a, const __grid_constant__ CUtensorMap tm_x,
                                                         const __grid_constant__ CUtensorMap tm_y, float2* __restrict__ lse_part) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sX = smem;
  uint8_t* sY = smem + XBYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + XBYTES + NST * YBYTES);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 16);
  const uint32_t bar0 = smem_u32(bars);
  auto BAR = [&](int i) { return bar0 + 8u * i; };
  constexpr int B_XFULL = 0, B_YFULL = 1, B_YEMPTY = 4, B_TFULL = 7, B_TEMPTY = 9;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int* err = a.flags + 1;

  const int x_tile = blockIdx.x % a.n_mtiles, chunk = blockIdx.x / a.n_mtiles;
  const int y_lo = (int)((long long)chunk * a.n_vtiles / a.n_chunks);
  const int y_hi = (int)((long long)(chunk + 1) * a.n_vtiles / a.n_chunks);
  const int n_it = max(0, y_hi - y_lo);

  if (threadIdx.x == 0) {
    mbar_init(BAR(B_XFULL), 1);
    for (int s = 0; s < NST; ++s) { mbar_init(BAR(B_YFULL + s), 1); mbar_init(BAR(B_YEMPTY + s), 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(BAR(B_TFULL + s), 1); mbar_init(BAR(B_TEMPTY + s), NEPI); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_x) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_y) : "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(128u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    if (lane == 0 && n_it > 0) {
      mbar_expect_tx(BAR(B_XFULL), XBYTES);
#pragma unroll
      for (int j = 0; j < NREG; ++j) tma_load_2d(smem_u32(sX) + j * XREG, &tm_x, 64 * j, x_tile * TM, BAR(B_XFULL));
      for (int it = 0; it < n_it; ++it) {
        const int ys = it % NST; const uint32_t yph = (it / NST) & 1;
        mbar_wait(BAR(B_YEMPTY + ys), yph ^ 1, err);
        mbar_expect_tx(BAR(B_YFULL + ys), YBYTES);
#pragma unroll
        for (int j = 0; j < NREG; ++j)
          tma_load_2d(smem_u32(sY + ys * YBYTES) + j * YREG, &tm_y, 64 * j, (y_lo + it) * TN, BAR(B_YFULL + ys));
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane == 0 && n_it > 0) {
      constexpr uint32_t IDESC = make_idesc(TM, TN, 0, 0);
      const uint32_t xa = smem_u32(sX);
      mbar_wait(BAR(B_XFULL), 0, err);
      for (int it = 0; it < n_it; ++it) {
        const int s = it & 1; const uint32_t ph = (it >> 1) & 1;
        const int ys = it % NST; const uint32_t yph = (it / NST) & 1;
        mbar_wait(BAR(B_YFULL + ys), yph, err);
        mbar_wait(BAR(B_TEMPTY + s), ph ^ 1, err);
        tc_fence_after();
        const uint32_t ya = smem_u32(sY + ys * YBYTES);
        // hi.hi + hi.lo + lo.hi (lo.lo is below the error bound): 3 x 10 k-steps into one accumulator
#pragma unroll
        for (int p = 0; p < 3; ++p) {
          const int ac = (p == 2) ? HALF : 0, bc = (p == 1) ? HALF : 0;
#pragma unroll
          for (int k = 0; k < 10; ++k)
            umma_bf16(tmem + s * TN, desc_col(xa, ac + 16 * k, XREG), desc_col(ya, bc + 16 * k, YREG), IDESC, (p | k) != 0);
        }
        umma_commit(BAR(B_YEMPTY + ys));
        umma_commit(BAR(B_TFULL + s));
      }
    }
    __syncwarp();
  } else {
    const int q = warp & 3, half = (warp - 2) >> 2;      // TMEM lane quarter, which 32 of the tile's 64 columns
    const int row = q * 32 + lane, gi = x_tile * TM + row;
    const uint32_t tlane = (uint32_t)(q * 32) << 16;
    const bool live = gi < a.R;
    const float lo = (live && RANK) ? a.lo_thr[gi] : INFINITY, hi = (live && RANK) ? a.hi_thr[gi] : INFINITY;
    const float lo_k = (live && CAND) ? a.lo_topk[gi] : INFINITY;
    const int* xl = a.excl + (long long)gi * EXCL_W;
    const int nx = (EXCL && live) ? a.excl_cnt[gi] : 0;
    int cur = 0;                                  // cursor into the row's sorted exclusion list
    float top[MS > 0 ? MS : 1];                   // descending; each entry is a different column
#pragma unroll
    for (int s = 0; s < MS; ++s) top[s] = -INFINITY;
    int above = 0;
    float lmax = -INFINITY, lsum = 0.f;           // LSE: running max and sum exp(S~ - lmax) of the slot
    for (int it = 0; it < n_it; ++it) {
      const int s = it & 1; const uint32_t ph = (it >> 1) & 1;
      mbar_wait(BAR(B_TFULL + s), ph, err);
      tc_fence_after();
      uint32_t r[32];
      tmem_ld32(tmem + tlane + s * TN + half * 32, r);
      tc_fence_before();
      mbar_arrive(BAR(B_TEMPTY + s));
      const int j0 = (y_lo + it) * TN + half * 32;
      if (!live) continue;
      unsigned ex = 0u;
      if constexpr (EXCL) {
        // windows come in ascending column order, so one forward walk of the list serves the whole pass
        while (cur < nx && xl[cur] < j0) ++cur;
        for (int c = cur; c < nx && xl[c] < j0 + 32; ++c) ex |= 1u << (xl[c] - j0);
      }
      const bool whole = j0 + 32 <= a.V;          // else: zero padding rows of the table matrix are not items
      unsigned unsure = 0u, topc = 0u;
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const float v = __uint_as_float(r[i]);
        const bool ok = (whole || j0 + i < a.V) && !((ex >> i) & 1u);
        if constexpr (RANK) {
          above += (ok && v > hi) ? 1 : 0;
          unsure |= (ok && v >= lo && v <= hi) ? (1u << i) : 0u;
        }
        if constexpr (CAND) topc |= (ok && v >= lo_k) ? (1u << i) : 0u;
        if constexpr (MS == 1) {
          if (ok) top[0] = fmaxf(top[0], v);
        } else if constexpr (MS > 1) {
          if (ok && v > top[MS - 1]) {            // insert v into the sorted list, dropping the smallest
#pragma unroll
            for (int t = MS - 1; t > 0; --t) top[t] = fmaxf(fminf(v, top[t - 1]), top[t]);
            top[0] = fmaxf(v, top[0]);
          }
        }
      }
      if constexpr (LSE) {
        // window max first, so each score takes one exp; the window's 32 terms are summed before they join the slot's sum
        constexpr float LOG2E = 1.4426950408889634f;
        float wm = -INFINITY;
#pragma unroll
        for (int i = 0; i < 32; ++i) if (whole || j0 + i < a.V) wm = fmaxf(wm, __uint_as_float(r[i]));
        if (wm > lmax) { lsum *= exp2f((lmax - wm) * LOG2E); lmax = wm; }
        float ws = 0.f;
#pragma unroll
        for (int i = 0; i < 32; ++i) ws += (whole || j0 + i < a.V) ? exp2f((__uint_as_float(r[i]) - lmax) * LOG2E) : 0.f;
        lsum += ws;
      }
      while (unsure) {                            // rare: a handful of columns per row in the whole pass
        const int i = __ffs(unsure) - 1; unsure &= unsure - 1;
        const int pos = atomicAdd(a.cand_cnt + gi, 1);
        if (pos < a.cap) a.cand[(long long)gi * a.cap + pos] = j0 + i; else atomicExch(a.flags, 1);
      }
      while (topc) {
        const int i = __ffs(topc) - 1; topc &= topc - 1;
        const int pos = atomicAdd(a.tk_cnt + gi, 1);
        if (pos < a.cap) a.tk_cand[(long long)gi * a.cap + pos] = j0 + i; else atomicExch(a.flags, 1);
      }
    }
    if (live) {
#pragma unroll
      for (int t = 0; t < MS; ++t) a.maxbuf[(long long)((chunk * 2 + half) * MS + t) * a.R + gi] = top[t];
      if constexpr (LSE) lse_part[(long long)(chunk * 2 + half) * a.R + gi] = make_float2(lmax, lsum);
    }
    if (live && RANK && above) atomicAdd(a.above + gi, above);
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(128u) : "memory");
  }
}

// exact re-score of the candidates of a row (warp per row, lane per candidate): rank = certainly-above + exactly-above
__global__ void __launch_bounds__(256) k_refine(const float* __restrict__ table1, const float* __restrict__ rep, const int* __restrict__ gt,
                                                int R, int d, const float* __restrict__ sg, const int* __restrict__ above,
                                                const int* __restrict__ cand_cnt, const int* __restrict__ cand, int cap,
                                                int* __restrict__ rank) {
  const int i = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (i >= R) return;
  const int n = min(cand_cnt[i], cap), g = gt[i] - 1;
  const float s0 = sg[i];
  const float* a = rep + (long long)i * d;
  int c = 0;
  for (int t = lane; t < n; t += 32) {
    const int j = cand[(long long)i * cap + t];
    if (j == g) continue;
    const float* b = table1 + (long long)j * d;
    float acc = 0.f;
    for (int k = 0; k < d; ++k) acc = fmaf(a[k], b[k], acc);
    c += (acc > s0) || (acc == s0 && j < g);
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if (lane == 0) rank[i] = above[i] + c;
}

// tau = the k-th largest of a row's local maxima (each belongs to a different item, so at least k items score >= tau - eps);
// every top-k item then has an approximate score >= tau - 2 eps.  Warp per row.
__global__ void __launch_bounds__(256) k_topk_threshold(const float* __restrict__ maxbuf, int n_slots, int R, int k,
                                                        const float* __restrict__ rnorm, const int* __restrict__ max_norm,
                                                        float* __restrict__ lo_topk) {
  const int i = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (i >= R) return;
  float v[8];                                     // n_slots <= 256
#pragma unroll
  for (int q = 0; q < 8; ++q) { const int sidx = lane + 32 * q; v[q] = sidx < n_slots ? maxbuf[(long long)sidx * R + i] : -INFINITY; }
  float kth = -INFINITY;
  for (int round = 0; round < k; ++round) {       // k rounds of "remove the current maximum"
    float best = -INFINITY; int bq = -1;
#pragma unroll
    for (int q = 0; q < 8; ++q) if (v[q] > best) { best = v[q]; bq = q; }
    float wb = best;
#pragma unroll
    for (int o = 16; o; o >>= 1) wb = fmaxf(wb, __shfl_xor_sync(0xffffffffu, wb, o));
    const unsigned who = __ballot_sync(0xffffffffu, best == wb && bq >= 0);
    if (who && lane == __ffs(who) - 1) {
#pragma unroll
      for (int q = 0; q < 8; ++q) if (q == bq) v[q] = -INFINITY;
    }
    kth = wb;
  }
  if (lane == 0) lo_topk[i] = kth - 2.f * C_ERR * rnorm[i] * __int_as_float(*max_norm);
}

// exact re-score of the top-k candidates of a row and selection of the k best (score descending, ties -> lower index):
// warp per row, up to 8 candidates per lane (cap = 256)
__global__ void __launch_bounds__(256) k_topk_refine(const float* __restrict__ table1, const float* __restrict__ rep, int R, int d,
                                                     const int* __restrict__ tk_cnt, const int* __restrict__ tk_cand, int cap, int k,
                                                     int* __restrict__ topk_item, float* __restrict__ topk_score) {
  const int i = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (i >= R) return;
  const int n = min(tk_cnt[i], cap);
  const float* a = rep + (long long)i * d;
  float sc[8]; int id[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const int t = lane + 32 * q;
    sc[q] = -INFINITY; id[q] = 0x7fffffff;
    if (t < n) {
      const int j = tk_cand[(long long)i * cap + t];
      const float* b = table1 + (long long)j * d;
      float acc = 0.f;
      for (int c = 0; c < d; ++c) acc = fmaf(a[c], b[c], acc);
      sc[q] = acc; id[q] = j;
    }
  }
  for (int round = 0; round < k; ++round) {
    float bs = -INFINITY; int bi = 0x7fffffff, bq = -1;
#pragma unroll
    for (int q = 0; q < 8; ++q) if (id[q] != 0x7fffffff && (sc[q] > bs || (sc[q] == bs && id[q] < bi))) { bs = sc[q]; bi = id[q]; bq = q; }
    float ws = bs; int wi = bi;
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      const float os = __shfl_xor_sync(0xffffffffu, ws, o); const int oi = __shfl_xor_sync(0xffffffffu, wi, o);
      if (os > ws || (os == ws && oi < wi)) { ws = os; wi = oi; }
    }
    if (bq >= 0 && bi == wi) {
#pragma unroll
      for (int q = 0; q < 8; ++q) if (q == bq) id[q] = 0x7fffffff;
    }
    if (lane == 0) {
      const bool ok = wi != 0x7fffffff;
      topk_item[(long long)i * k + round] = ok ? wi + 1 : 0;
      topk_score[(long long)i * k + round] = ok ? ws : -INFINITY;
    }
  }
}

// lse[i] = log sum over the row's n_slots (max, sum) pairs, combined in a fixed order (lane-strided, then a butterfly), in
// fp64; nll[i] = lse[i] - sg[i] when sg is given.  Warp per row; a slot without items is (-inf, 0).
__global__ void __launch_bounds__(256) k_lse_merge(const float2* __restrict__ part, int n_slots, int R, const float* __restrict__ sg,
                                                   float* __restrict__ lse, float* __restrict__ nll) {
  const int i = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (i >= R) return;
  double m = -INFINITY, s = 0.0;
  auto join = [&](double m2, double s2) {         // (m, s) <- (m, s) + (m2, s2); -inf maxima carry a zero sum
    const double mx = fmax(m, m2);
    if (mx == -INFINITY) return;
    s = (m == mx ? s : s * exp(m - mx)) + (m2 == mx ? s2 : s2 * exp(m2 - mx));
    m = mx;
  };
  for (int t = lane; t < n_slots; t += 32) {
    const float2 p = part[(long long)t * R + i];
    join(p.x, p.y);
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    const double m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, s, o);
    join(m2, s2);
  }
  if (lane == 0) {
    const float l = (float)(m + log(s));
    lse[i] = l;
    if (sg) nll[i] = l - sg[i];
  }
}

// ids [R, L] (left-padded, 0 = empty) -> the row's columns id - 1 < V, ascending and distinct, in excl [R][EXCL_W] + excl_cnt [R].
// Warp per row, two ids per lane: an id is kept at its first position; its slot is the number of distinct smaller ids.
__global__ void __launch_bounds__(256) k_excl_lists(const int* __restrict__ ids, int R, int L, int V, int* __restrict__ excl,
                                                    int* __restrict__ excl_cnt) {
  const int i = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (i >= R) return;
  int v[2]; bool first[2]; int less[2];
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int c = lane + 32 * h;
    const int id = c < L ? ids[(long long)i * L + c] : 0;
    v[h] = (id >= 1 && id <= V) ? id - 1 : INT_MAX;
    first[h] = v[h] != INT_MAX; less[h] = 0;
  }
  for (int p = 0; p < 64; ++p) {
    const int x = __shfl_sync(0xffffffffu, p < 32 ? v[0] : v[1], p & 31);
#pragma unroll
    for (int h = 0; h < 2; ++h) if (x == v[h] && p < lane + 32 * h) first[h] = false;
  }
  for (int p = 0; p < 64; ++p) {
    const int x = __shfl_sync(0xffffffffu, p < 32 ? v[0] : v[1], p & 31);
    const bool fx = __shfl_sync(0xffffffffu, p < 32 ? first[0] : first[1], p & 31);
#pragma unroll
    for (int h = 0; h < 2; ++h) less[h] += (fx && x < v[h]) ? 1 : 0;
  }
#pragma unroll
  for (int h = 0; h < 2; ++h) if (first[h]) excl[(long long)i * EXCL_W + less[h]] = v[h];
  const int n = __popc(__ballot_sync(0xffffffffu, first[0])) + __popc(__ballot_sync(0xffffffffu, first[1]));
  if (lane == 0) excl_cnt[i] = n;
}

static int eval_chunks(int R, int V) {
  const int n_mtiles = cdiv(R, TM), n_vtiles = cdiv(V, TN);
  int best = 1; double best_eff = 0.0;
  const int cmax = n_vtiles / 8 > 1 ? (n_vtiles / 8 < 128 ? n_vtiles / 8 : 128) : 1;      // >= 8 streamed tiles per CTA, <= 256 top-k slots per row
  for (int c = 1; c <= cmax; ++c) {
    const long long ctas = (long long)n_mtiles * c;
    const long long waves = (ctas + 147) / 148;
    const double eff = (double)ctas / (148.0 * waves);
    if (eff > best_eff + 1e-9) { best_eff = eff; best = c; }
  }
  return best;
}

struct EvalWs {
  __nv_bfloat16 *x16, *y16;
  float *rnorm, *sg, *lo, *hi;
  int *max_norm, *above, *cand_cnt, *cand, *flags, *tk_cnt, *tk_cand;
  float *lo_topk, *maxbuf;
  int *excl, *excl_cnt;
  float2* lse_part;
  size_t bytes;
};
// excl: append the exclusion lists (recommendation); lse: append the (max, sum) slots of the log-sum-exp pass.  The layout
// before them is the same either way.
static EvalWs carve(int R, int V, bool excl, bool lse, char* base) {
  EvalWs w; size_t o = 0;
  auto take = [&](size_t n) { char* p = base ? base + o : nullptr; o += align_up(n); return p; };
  const int nm = cdiv(R, TM), nv = cdiv(V, TN), cap = ADER_EVAL_CAND_CAP;
  w.x16 = (__nv_bfloat16*)take((size_t)nm * TM * D2 * 2);
  w.y16 = (__nv_bfloat16*)take((size_t)nv * TN * D2 * 2);
  w.rnorm = (float*)take(sizeof(float) * R);
  w.sg = (float*)take(sizeof(float) * R);
  w.lo = (float*)take(sizeof(float) * R);
  w.hi = (float*)take(sizeof(float) * R);
  // zeroed per call in one memset: [max_norm(4 ints) | flags(4 ints) | above R | cand_cnt R]
  w.max_norm = (int*)take(sizeof(int) * (8 + 2 * (size_t)R));
  w.flags = w.max_norm + 4; w.above = w.max_norm + 8; w.cand_cnt = w.above + R;
  w.cand = (int*)take(sizeof(int) * (size_t)R * cap);
  w.tk_cnt = (int*)take(sizeof(int) * (size_t)R);
  w.tk_cand = (int*)take(sizeof(int) * (size_t)R * cap);
  w.lo_topk = (float*)take(sizeof(float) * (size_t)R);
  w.maxbuf = (float*)take(sizeof(float) * (size_t)R * 2 * 128);
  w.excl = excl ? (int*)take(sizeof(int) * (size_t)R * EXCL_W) : nullptr;
  w.excl_cnt = excl ? (int*)take(sizeof(int) * (size_t)R) : nullptr;
  w.lse_part = lse ? (float2*)take(sizeof(float2) * (size_t)R * 2 * eval_chunks(R, V)) : nullptr;
  w.bytes = o;
  return w;
}

template <bool RANK, bool CAND, int MS, bool EXCL, bool LSE = false>
static int eval_pass(const EvalArgs& a, const CUtensorMap& tx, const CUtensorMap& ty, cudaStream_t st,
                     float2* lse_part = nullptr) {
  if (int e = kernel_ready<k_eval_tc<RANK, CAND, MS, EXCL, LSE>>(SMEM_EVAL, "k_eval_tc")) return e;
  k_eval_tc<RANK, CAND, MS, EXCL, LSE><<<a.n_mtiles * a.n_chunks, NTHREADS, SMEM_EVAL, st>>>(a, tx, ty, lse_part);
  return 0;
}

template <bool EXCL>
static int maxima_pass(int ms, const EvalArgs& a, const CUtensorMap& tx, const CUtensorMap& ty, cudaStream_t st) {
  switch (ms) {
    case 1: return eval_pass<false, false, 1, EXCL>(a, tx, ty, st);
    case 2: return eval_pass<false, false, 2, EXCL>(a, tx, ty, st);
    case 4: return eval_pass<false, false, 4, EXCL>(a, tx, ty, st);
    default: return eval_pass<false, false, 8, EXCL>(a, tx, ty, st);
  }
}

}  // namespace ev
}  // namespace ader

using namespace ader;
using namespace ader::ev;

// The pipeline behind the tensor-core entries.  gt (or NULL): the exact score of the ground truth (k_gt_band); with rank, the
// rank of the ground truth from it, the counting pass and k_refine.  k > 0: top-k, from a maxima pass, tau (k_topk_threshold),
// a candidate pass and k_topk_refine.  ids (or NULL, never with gt): each row's own items are left out of the maxima and the
// candidates.  lse (or NULL): the log-sum-exp pass over items 1..V and k_lse_merge, and with gt nll = lse - s_gt.
// overflow may be NULL when no candidate list is collected.
// The maxima pass keeps m scores per (chunk, column half), m = the smallest of 1, 2, 4, 8 with 2 * nc * m >= k (the eval
// entries admit only 2 * nc >= k, so they run with m = 1; 2 * nc * m <= 256, the slot count k_topk_threshold takes).  All
// kept scores belong to different eligible items, so at least k eligible items score >= tau - eps and every eligible item
// whose exact score reaches the k-th one has S~ >= tau - 2 eps.
static int topk_tc_run(const AderModel* m, const float* theta, const float* rep, const int32_t* gt, const int32_t* ids, int R,
                       int V, int k, void* ws, int32_t* rank, int32_t* topk_item, float* topk_score, int32_t* overflow,
                       float* lse, float* nll, cudaStream_t st) {
  const int d = m->d, cap = ADER_EVAL_CAND_CAP;
  EvalWs w = carve(R, V, ids != nullptr, lse != nullptr, (char*)ws);
  const int nm = cdiv(R, TM), nv = cdiv(V, TN), nc = eval_chunks(R, V);
  int ms = 1;
  while (ms < 8 && 2 * nc * ms < k) ms *= 2;
  CUtensorMap tx, ty;
  if (int e = make_map2d(&tx, w.x16, D2, (uint64_t)nm * TM, D2 * 2, TM)) return e;
  if (int e = make_map2d(&ty, w.y16, D2, (uint64_t)nv * TN, D2 * 2, TN)) return e;
  const float* table1 = theta + d;                       // item 1 = table row 1 (ADER.py:90-91)
  cudaMemsetAsync(w.max_norm, 0, sizeof(int) * (8 + (rank ? 2 * (size_t)R : 0)), st);
  if (k > 0) cudaMemsetAsync(w.tk_cnt, 0, sizeof(int) * (size_t)R, st);
  k_pack_hilo<<<cdiv((long long)nv * TN * 32, 256), 256, 0, st>>>(table1, d, V, d, nv * TN, w.y16, nullptr, w.max_norm);
  k_pack_hilo<<<cdiv((long long)nm * TM * 32, 256), 256, 0, st>>>(rep, d, R, d, nm * TM, w.x16, w.rnorm, nullptr);
  if (gt) k_gt_band<<<cdiv(R, 256), 256, 0, st>>>(table1, rep, gt, R, d, w.rnorm, w.max_norm, w.sg, w.lo, w.hi);
  if (ids) k_excl_lists<<<cdiv((long long)R * 32, 256), 256, 0, st>>>(ids, R, m->maxlen, V, w.excl, w.excl_cnt);
  EvalArgs a = {};
  a.R = R; a.V = V; a.n_mtiles = nm; a.n_vtiles = nv; a.n_chunks = nc;
  a.lo_thr = w.lo; a.hi_thr = w.hi; a.above = w.above; a.cand_cnt = w.cand_cnt; a.cand = w.cand; a.cap = cap; a.flags = w.flags;
  a.maxbuf = w.maxbuf; a.lo_topk = w.lo_topk; a.tk_cnt = w.tk_cnt; a.tk_cand = w.tk_cand;
  a.excl = w.excl; a.excl_cnt = w.excl_cnt;
  if (k > 0) {
    if (int e = ids ? maxima_pass<true>(ms, a, tx, ty, st) : maxima_pass<false>(ms, a, tx, ty, st)) return e;
    k_topk_threshold<<<cdiv((long long)R * 32, 256), 256, 0, st>>>(w.maxbuf, 2 * nc * ms, R, k, w.rnorm, w.max_norm, w.lo_topk);
  }
  if (rank) {
    if (int e = k > 0 ? eval_pass<true, true, 0, false>(a, tx, ty, st) : eval_pass<true, false, 0, false>(a, tx, ty, st)) return e;
  } else if (k > 0) {
    if (int e = ids ? eval_pass<false, true, 0, true>(a, tx, ty, st) : eval_pass<false, true, 0, false>(a, tx, ty, st)) return e;
  }
  if (k > 0)
    k_topk_refine<<<cdiv((long long)R * 32, 256), 256, 0, st>>>(table1, rep, R, d, w.tk_cnt, w.tk_cand, cap, k, topk_item, topk_score);
  if (rank) k_refine<<<cdiv((long long)R * 32, 256), 256, 0, st>>>(table1, rep, gt, R, d, w.sg, w.above, w.cand_cnt, w.cand, cap, rank);
  if (lse) {
    if (int e = eval_pass<false, false, 0, false, true>(a, tx, ty, st, w.lse_part)) return e;
    k_lse_merge<<<cdiv((long long)R * 32, 256), 256, 0, st>>>(w.lse_part, 2 * nc, R, gt ? w.sg : nullptr, lse, nll);
  }
  if (overflow) cudaMemcpyAsync(overflow, w.flags, sizeof(int), cudaMemcpyDeviceToDevice, st);
  ADER_CHECK_LAUNCH(lse ? "logsumexp_tc" : gt ? "eval_rank_tc" : "recommend_topk_tc");
  return 0;
}

extern "C" size_t ader_eval_rank_tc_ws_bytes(const AderModel* m, int32_t R, int32_t V) {
  if (check_model(m) || R <= 0 || V <= 0 || path_check(m, ADER_PATH_EVAL_TC)) return 0;
  return carve(R, V, false, false, nullptr).bytes;
}

extern "C" int32_t ader_eval_rank_tc(const AderModel* m, const float* theta, const float* rep, const int32_t* gt, int32_t R,
                                     int32_t V, void* ws, int32_t* rank, int32_t* overflow, void* stream) {
  if (int e = check_model(m)) return e;
  if (int e = path_check(m, ADER_PATH_EVAL_TC)) return e;
  ADER_CHECK_ARG(theta && rep && gt && ws && rank && overflow, "eval_rank_tc: NULL pointer");
  ADER_CHECK_ARG(R > 0 && V >= 1 && V < m->v_tab, "eval_rank_tc: bad sizes");
  return topk_tc_run(m, theta, rep, gt, nullptr, R, V, 0, ws, rank, nullptr, nullptr, overflow, nullptr, nullptr, (cudaStream_t)stream);
}

extern "C" int32_t ader_eval_topk_chunks(const AderModel* m, int32_t R, int32_t V) {
  if (check_model(m) || R <= 0 || V <= 0) return 0;
  return eval_chunks(R, V);
}

extern "C" int32_t ader_eval_rank_topk_tc(const AderModel* m, const float* theta, const float* rep, const int32_t* gt, int32_t R,
                                          int32_t V, int32_t k, void* ws, int32_t* rank, int32_t* topk_item, float* topk_score,
                                          int32_t* overflow, void* stream) {
  if (int e = check_model(m)) return e;
  if (int e = path_check(m, ADER_PATH_EVAL_TC)) return e;
  ADER_CHECK_ARG(theta && rep && gt && ws && rank && overflow && topk_item && topk_score, "eval_rank_topk_tc: NULL pointer");
  ADER_CHECK_ARG(R > 0 && V >= 1 && V < m->v_tab && k >= 1 && k <= 32, "eval_rank_topk_tc: bad sizes");
  const int nc = eval_chunks(R, V);
  ADER_CHECK_ARG(2 * nc >= k && 2 * nc <= 256, "eval_rank_tc: top-%d needs %d..128 vocabulary chunks per row tile (have %d): use ader_eval_rank_topk", k, (k + 1) / 2, nc);
  return topk_tc_run(m, theta, rep, gt, nullptr, R, V, k, ws, rank, topk_item, topk_score, overflow, nullptr, nullptr,
                     (cudaStream_t)stream);
}

extern "C" size_t ader_recommend_tc_ws_bytes(const AderModel* m, int32_t R, int32_t V) {
  if (check_model(m) || R <= 0 || V <= 0 || path_check(m, ADER_PATH_EVAL_TC)) return 0;
  return carve(R, V, true, false, nullptr).bytes;
}

extern "C" int32_t ader_recommend_topk_tc(const AderModel* m, const float* theta, const float* rep, const int32_t* ids, int32_t R,
                                          int32_t V, int32_t k, void* ws, int32_t* topk_item, float* topk_score,
                                          int32_t* overflow, void* stream) {
  if (int e = check_model(m)) return e;
  if (int e = path_check(m, ADER_PATH_EVAL_TC)) return e;
  ADER_CHECK_ARG(theta && rep && ws && topk_item && topk_score && overflow, "recommend_topk_tc: NULL pointer");
  ADER_CHECK_ARG(R > 0 && V >= 1 && V < m->v_tab && k >= 1 && k <= 100, "recommend_topk_tc: bad sizes");
  const int nc = eval_chunks(R, V);
  ADER_CHECK_ARG(2 * nc * 8 >= k, "recommend_topk_tc: top-%d needs %d vocabulary chunks per row tile (have %d): use ader_recommend_topk",
                 k, (k + 15) / 16, nc);
  return topk_tc_run(m, theta, rep, nullptr, ids, R, V, k, ws, nullptr, topk_item, topk_score, overflow, nullptr, nullptr,
                     (cudaStream_t)stream);
}

extern "C" size_t ader_logsumexp_tc_ws_bytes(const AderModel* m, int32_t R, int32_t V) {
  if (check_model(m) || R <= 0 || V <= 0 || path_check(m, ADER_PATH_EVAL_TC)) return 0;
  return carve(R, V, false, true, nullptr).bytes;
}

extern "C" int32_t ader_logsumexp_tc(const AderModel* m, const float* theta, const float* rep, const int32_t* gt, int32_t R,
                                     int32_t V, void* ws, float* lse, float* nll, void* stream) {
  if (int e = check_model(m)) return e;
  if (int e = path_check(m, ADER_PATH_EVAL_TC)) return e;
  if (int e = check_lse_args(m, theta, rep, gt, R, V, ws, lse, nll, "logsumexp_tc")) return e;
  return topk_tc_run(m, theta, rep, gt, nullptr, R, V, 0, ws, nullptr, nullptr, nullptr, nullptr, lse, nll, (cudaStream_t)stream);
}
