// Segmented herding exemplar selection (util.py:401-434; SURVEY A.6).  One CTA per label item.
// All arithmetic is fp32 in the order NumPy uses where that order is defined:
//   norm_j = sqrt(pairwise_sum(x*x))   (np.linalg.norm axis reduce over the contiguous axis)
//   D_j    = x / norm_j ;  mu = (sequential sum over candidates) / n ;  w <- (w + mu) - D[:, i]
// The 150-term dot w.D_j is a BLAS call in the reference (summation order unspecified); here
// it is a lane-strided sum + butterfly.  Picks can therefore differ only at near-ties.
#include "common.cuh"
#include <stdlib.h>

namespace ader {

// NumPy pairwise_sum for a contiguous float32 vector of squares (numpy/core/src/umath/loops_utils.h):
// n < 8: sequential; n <= 128: 8 accumulators; else split at n/2 rounded down to a multiple of 8.
__device__ float np_pairwise_sq(const float* __restrict__ x, int n) {
  if (n < 8) {
    float r = 0.f;
    for (int i = 0; i < n; ++i) r = __fadd_rn(r, __fmul_rn(x[i], x[i]));
    return r;
  }
  if (n <= 128) {
    float r[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) r[k] = __fmul_rn(x[k], x[k]);
    int i;
    for (i = 8; i < n - (n % 8); i += 8) {
#pragma unroll
      for (int k = 0; k < 8; ++k) r[k] = __fadd_rn(r[k], __fmul_rn(x[i + k], x[i + k]));
    }
    float res = __fadd_rn(__fadd_rn(__fadd_rn(r[0], r[1]), __fadd_rn(r[2], r[3])),
                          __fadd_rn(__fadd_rn(r[4], r[5]), __fadd_rn(r[6], r[7])));
    for (; i < n; ++i) res = __fadd_rn(res, __fmul_rn(x[i], x[i]));
    return res;
  }
  int n2 = n / 2; n2 -= n2 % 8;
  return __fadd_rn(np_pairwise_sq(x, n2), np_pairwise_sq(x + n2, n - n2));
}

__global__ void __launch_bounds__(256) k_herding(const float* __restrict__ rep, int d, const int* __restrict__ cand,
                                                 const int* __restrict__ seg_off, const int* __restrict__ quota,
                                                 const int* __restrict__ max_steps, float* __restrict__ Dn,
                                                 int* __restrict__ selected, int* __restrict__ picks,
                                                 int* __restrict__ n_picked, const int* __restrict__ list, const int* __restrict__ list_n) {
  __shared__ float w[256], mu[256];
  __shared__ float bestv[8]; __shared__ int bestj[8];
  __shared__ int pick_s, cnt_s;
  if (list && (int)blockIdx.x >= *list_n) return;
  const int s = list ? list[blockIdx.x] : blockIdx.x;
  const int off = seg_off[s], n = seg_off[s + 1] - off;
  const int m = min(quota[s], n);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (n <= 0 || m <= 0) { if (tid == 0) n_picked[s] = 0; return; }

  // D = rep^T / ||rep^T||_2, one thread per candidate for the norm (NumPy's summation order)
  for (int j = tid; j < n; j += blockDim.x) {
    const float* x = rep + (long long)cand[off + j] * d;
    float nrm = sqrtf(np_pairwise_sq(x, d));
    float* o = Dn + (long long)(off + j) * d;
    for (int c = 0; c < d; ++c) o[c] = __fdiv_rn(x[c], nrm);
    selected[off + j] = 0;
  }
  __syncthreads();
  if (tid < d) {
    float acc = 0.f;
    for (int j = 0; j < n; ++j) acc = __fadd_rn(acc, Dn[(long long)(off + j) * d + tid]);
    float mval = __fdiv_rn(acc, (float)n);
    mu[tid] = mval; w[tid] = mval;
  }
  if (tid == 0) cnt_s = 0;
  __syncthreads();

  const int steps = max_steps[s];
  for (int step = 0; step < steps; ++step) {
    float bv = -INFINITY; int bj = 0x7fffffff;
    for (int j = warp; j < n; j += 8) {
      const float* D = Dn + (long long)(off + j) * d;
      float acc = 0.f;
      for (int c = lane; c < d; c += 32) acc = fmaf(w[c], D[c], acc);
#pragma unroll
      for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if (acc > bv) { bv = acc; bj = j; }          // j ascending inside a warp: first max kept
    }
    if (lane == 0) { bestv[warp] = bv; bestj[warp] = bj; }
    __syncthreads();
    if (tid == 0) {
      float fv = bestv[0]; int fj = bestj[0];
      for (int q = 1; q < 8; ++q)
        if (bestv[q] > fv || (bestv[q] == fv && bestj[q] < fj)) { fv = bestv[q]; fj = bestj[q]; }
      // every dot product NaN (a zero-norm rep row: 0/0 in the normalisation): no comparison succeeded; np.argmax
      // returns index 0 for an all-NaN vector (util.py:426), and the index must stay inside the segment
      if (fj < 0 || fj >= n) fj = 0;
      pick_s = fj;
      if (!selected[off + fj]) { selected[off + fj] = 1; picks[off + cnt_s] = fj; cnt_s = cnt_s + 1; }
    }
    __syncthreads();
    const int pk = pick_s;
    if (tid < d) w[tid] = __fsub_rn(__fadd_rn(w[tid], mu[tid]), Dn[(long long)(off + pk) * d + tid]);
    const bool done = (cnt_s == m);
    __syncthreads();
    if (done) break;
  }
  if (tid == 0) n_picked[s] = cnt_s;
}


// =====================================================================================================================
// Second generation: the same arithmetic, element for element (norm by NumPy's pairwise order, sequential mean, the dot
// as a lane-strided fmaf chain + xor butterfly, first-max arg-max, (w + mu) - D), so the picks are bit-identical to
// k_herding -- but the normalised candidates D live ON CHIP for the whole selection instead of being re-read from global
// memory at every arg-max step, and the launch shape follows the segment size (YOOCHOOSE: median 3 candidates, p99 ~350,
// max 3 342; DIGINETICA: median 2, max 98):
//   n <= 16   one WARP per segment, D and w in registers (5 values per lane and row): no shared memory, no barriers;
//   n <= 350  one CTA per segment, D in shared memory (<= 210 KB);
//   larger    one CLUSTER of 8 CTAs per segment, D split over their shared memories (8 x 350 rows; a segment beyond 2 800
//             keeps the remainder of each CTA's slice in global memory / L2); per step the 8 local arg-maxima meet
//             in CTA 0 (DSMEM), the owner of the pick broadcasts its row into every CTA (DSMEM), two cluster barriers;
//   > 16 384  k_herding (D in global memory / L2).
// A prologue kernel sorts the segment ids into the four classes.
constexpr int HS_MAX = 16, HM_MAX = 350, HB_CTAS = 8, HB_PER = 350, HB_MAX = HB_CTAS * HB_PER;
constexpr int HB_NMAX = 16384, HB_BM_WORDS = HB_NMAX / 32;      // largest segment of the cluster form (picked-candidate bitmap)
constexpr int HD = 150;                        // rows are padded to 5 x 32 lanes; d <= 160
constexpr int HREG = 5;

__global__ void k_herding_classify(const int* __restrict__ seg_off, const int* __restrict__ quota, int n_seg, int* __restrict__ cnt,
                                   int* __restrict__ l_small, int* __restrict__ l_mid, int* __restrict__ l_big, int* __restrict__ l_huge,
                                   int* __restrict__ n_picked) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_seg) return;
  const int n = seg_off[s + 1] - seg_off[s];
  if (n <= 0 || min(quota[s], n) <= 0) { n_picked[s] = 0; return; }
  if (n <= HS_MAX) l_small[atomicAdd(cnt + 0, 1)] = s;
  else if (n <= HM_MAX) l_mid[atomicAdd(cnt + 1, 1)] = s;
  else if (n <= HB_NMAX) l_big[atomicAdd(cnt + 2, 1)] = s;     // > 2800: the rows beyond 8 x 350 spill to global memory
  else l_huge[atomicAdd(cnt + 3, 1)] = s;
}

__device__ __forceinline__ float warp_dot(const float (&w)[HREG], const float (&D)[HREG]) {
  float acc = 0.f;
#pragma unroll
  for (int i = 0; i < HREG; ++i) acc = fmaf(w[i], D[i], acc);          // c = lane, lane + 32, ...: ascending c per lane
#pragma unroll
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  return acc;
}

// ---- n <= 16: warp per segment, everything in registers -----------------------------------------------------------------
__global__ void __launch_bounds__(256) k_herding_small(const float* __restrict__ rep, int d, const int* __restrict__ cand,
                                                       const int* __restrict__ seg_off, const int* __restrict__ quota,
                                                       const int* __restrict__ max_steps, const int* __restrict__ list,
                                                       const int* __restrict__ cnt, int* __restrict__ picks, int* __restrict__ n_picked) {
  const int wi = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (wi >= cnt[0]) return;
  const int s = list[wi];
  const int off = seg_off[s], n = seg_off[s + 1] - off;
  const int m = min(quota[s], n);
  float D[HS_MAX][HREG];
  // norm of candidate j by lane j (NumPy's summation order), broadcast; rows loaded coalesced
  float nrm_l = 1.f;
  if (lane < n) nrm_l = sqrtf(np_pairwise_sq(rep + (long long)cand[off + lane] * d, d));
#pragma unroll
  for (int j = 0; j < HS_MAX; ++j) {
    const float nrm = __shfl_sync(0xffffffffu, nrm_l, j);
    if (j < n) {
      const float* x = rep + (long long)cand[off + j] * d;
#pragma unroll
      for (int i = 0; i < HREG; ++i) { const int c = lane + 32 * i; D[j][i] = c < d ? __fdiv_rn(x[c], nrm) : 0.f; }
    } else {
#pragma unroll
      for (int i = 0; i < HREG; ++i) D[j][i] = 0.f;
    }
  }
  float mu[HREG], w[HREG];
#pragma unroll
  for (int i = 0; i < HREG; ++i) {
    float acc = 0.f;
#pragma unroll
    for (int j = 0; j < HS_MAX; ++j) if (j < n) acc = __fadd_rn(acc, D[j][i]);
    mu[i] = __fdiv_rn(acc, (float)n); w[i] = mu[i];
  }
  unsigned sel = 0u; int cnt_p = 0;
  const int steps = max_steps[s];
  for (int step = 0; step < steps; ++step) {
    float bv = -INFINITY; int bj = 0;
#pragma unroll
    for (int j = 0; j < HS_MAX; ++j) {
      if (j < n) { const float a = warp_dot(w, D[j]); if (a > bv) { bv = a; bj = j; } }
    }
    if (!(sel >> bj & 1u)) { sel |= 1u << bj; if (lane == 0) picks[off + cnt_p] = bj; ++cnt_p; }
#pragma unroll
    for (int j = 0; j < HS_MAX; ++j)
      if (j == bj) {
#pragma unroll
        for (int i = 0; i < HREG; ++i) w[i] = __fsub_rn(__fadd_rn(w[i], mu[i]), D[j][i]);
      }
    if (cnt_p == m) break;
  }
  if (lane == 0) n_picked[s] = cnt_p;
}

// ---- shared by the CTA and cluster forms: rows [j0, j0 + nl) of the segment normalised into shared memory ---------------
// rows beyond `cap_s` (only in segments larger than the cluster's shared memories) go to the global spill gD [*, 160]
__device__ __forceinline__ void load_norm_rows(const float* __restrict__ rep, int d, const int* __restrict__ cand, int off, int j0, int nl,
                                               float* __restrict__ sD, float* __restrict__ snrm, int cap_s = 0x7fffffff,
                                               float* __restrict__ gD = nullptr) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int b0 = 0; b0 < nl; b0 += cap_s) {             // norms staged cap_s rows at a time (snrm holds cap_s entries)
    const int nb = min(cap_s, nl - b0);
    for (int j = threadIdx.x; j < nb; j += blockDim.x) snrm[j] = sqrtf(np_pairwise_sq(rep + (long long)cand[off + j0 + b0 + j] * d, d));
    __syncthreads();
    for (int j = warp; j < nb; j += nw) {
      const float* x = rep + (long long)cand[off + j0 + b0 + j] * d;
      const float nrm = snrm[j];
      float* o = (b0 + j < cap_s) ? sD + (b0 + j) * 160 : gD + (long long)(b0 + j - cap_s) * 160;
      for (int c = lane; c < 160; c += 32) o[c] = c < d ? __fdiv_rn(x[c], nrm) : 0.f;
    }
    __syncthreads();
  }
}
// local first-max over rows [0, nl) of sD against w (shared): result (value, local index) of this CTA
__device__ __forceinline__ void local_argmax(const float* __restrict__ sD, const float* __restrict__ sw, int nl, float* bestv, int* bestj,
                                             float& fv, int& fj, int cap_s = 0x7fffffff, const float* __restrict__ gD = nullptr) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  float wv[HREG];
#pragma unroll
  for (int i = 0; i < HREG; ++i) wv[i] = sw[lane + 32 * i];
  float bv = -INFINITY; int bj = 0x7fffffff;
  for (int j = warp; j < nl; j += nw) {                // j ascending per warp, warps merged below by (value, index): first max
    const float* row = j < cap_s ? sD + j * 160 : gD + (long long)(j - cap_s) * 160;
    float Dv[HREG];
#pragma unroll
    for (int i = 0; i < HREG; ++i) Dv[i] = row[lane + 32 * i];
    const float a = warp_dot(wv, Dv);
    if (a > bv) { bv = a; bj = j; }
  }
  if (lane == 0) { bestv[warp] = bv; bestj[warp] = bj; }
  __syncthreads();
  fv = bestv[0]; fj = bestj[0];
  for (int q = 1; q < nw; ++q)
    if (bestv[q] > fv || (bestv[q] == fv && bestj[q] < fj)) { fv = bestv[q]; fj = bestj[q]; }
}

// ---- 16 < n <= 350: CTA per segment, D in shared memory -------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_herding_mid(const float* __restrict__ rep, int d, const int* __restrict__ cand,
                                                     const int* __restrict__ seg_off, const int* __restrict__ quota,
                                                     const int* __restrict__ max_steps, const int* __restrict__ list,
                                                     const int* __restrict__ cnt, int* __restrict__ selected, int* __restrict__ picks,
                                                     int* __restrict__ n_picked) {
  extern __shared__ float hs[];
  if ((int)blockIdx.x >= cnt[1]) return;
  float* sD = hs;                                  // [HM_MAX][160]
  float* sw = hs + HM_MAX * 160;                   // [160]
  float* smu = sw + 160;
  float* snrm = smu + 160;                         // [HM_MAX]
  __shared__ float bestv[8]; __shared__ int bestj[8];
  __shared__ int cnt_s;
  const int s = list[blockIdx.x];
  const int off = seg_off[s], n = seg_off[s + 1] - off;
  const int m = min(quota[s], n), tid = threadIdx.x;
  load_norm_rows(rep, d, cand, off, 0, n, sD, snrm);
  for (int j = tid; j < n; j += blockDim.x) selected[off + j] = 0;
  if (tid < 160) {
    float acc = 0.f;
    for (int j = 0; j < n; ++j) acc = __fadd_rn(acc, sD[j * 160 + tid]);
    const float mv = tid < d ? __fdiv_rn(acc, (float)n) : 0.f;
    smu[tid] = mv; sw[tid] = mv;
  }
  if (tid == 0) cnt_s = 0;
  __syncthreads();
  const int steps = max_steps[s];
  for (int step = 0; step < steps; ++step) {
    float fv; int fj;
    local_argmax(sD, sw, n, bestv, bestj, fv, fj);
    if (fj < 0 || fj >= n) fj = 0;
    if (tid == 0 && !selected[off + fj]) { selected[off + fj] = 1; picks[off + cnt_s] = fj; cnt_s = cnt_s + 1; }
    __syncthreads();
    if (tid < 160) sw[tid] = __fsub_rn(__fadd_rn(sw[tid], smu[tid]), sD[fj * 160 + tid]);
    const bool done = (cnt_s == m);
    __syncthreads();
    if (done) break;
  }
  if (tid == 0) n_picked[s] = cnt_s;
}

// ---- 350 < n <= 2800: cluster of 8 CTAs per segment, D split over their shared memories (DSMEM) ----------------------------
__device__ __forceinline__ uint32_t cluster_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t map_to_cta(const void* p, uint32_t cta) {       // shared::cluster address of `p` in CTA `cta`
  uint32_t a = (uint32_t)__cvta_generic_to_shared(p), r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(cta));
  return r;
}
__device__ __forceinline__ void st_cluster_f32(uint32_t addr, float v) { asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory"); }
__device__ __forceinline__ void st_cluster_s32(uint32_t addr, int v) { asm volatile("st.shared::cluster.s32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }

__global__ void __cluster_dims__(HB_CTAS, 1, 1) __launch_bounds__(256)
k_herding_big(const float* __restrict__ rep, int d, const int* __restrict__ cand, const int* __restrict__ seg_off,
              const int* __restrict__ quota, const int* __restrict__ max_steps, const int* __restrict__ list,
              const int* __restrict__ cnt, float* __restrict__ Dn, int* __restrict__ picks, int* __restrict__ n_picked) {
  extern __shared__ float hs[];
  const int ci = blockIdx.x / HB_CTAS;
  if (ci >= cnt[2]) return;                        // uniform over the cluster
  const uint32_t cr = cluster_rank();
  float* sD = hs;                                  // [HB_PER][160] this CTA's candidates
  float* sw = hs + HB_PER * 160;
  float* smu = sw + 160;
  float* srow = smu + 160;                         // [160] row of the pick, written by its owner (DSMEM)
  float* spart = srow + 160;                       // [160] running mean partial handed from CTA r-1 to r
  float* snrm = spart + 160;                       // [HB_PER]
  unsigned* bm = reinterpret_cast<unsigned*>(snrm + HB_PER);         // picked-candidate bitmap, replicated in every CTA
  __shared__ float bestv[8]; __shared__ int bestj[8];
  __shared__ float gv[HB_CTAS]; __shared__ int gj[HB_CTAS];          // CTA 0 collects the local maxima here
  __shared__ int cnt_s;
  const int s = list[ci];
  const int off = seg_off[s], n = seg_off[s + 1] - off;
  const int m = min(quota[s], n), tid = threadIdx.x;
  const int per = (n + HB_CTAS - 1) / HB_CTAS;     // candidates per CTA, contiguous ranges in candidate order; the first HB_PER
  const int j0 = min(n, (int)cr * per), nl = min(n, j0 + per) - j0;   // of them sit in shared memory, the rest (segments > 2800) in gD
  float* gD = Dn + (long long)(off + j0) * 160;    // this CTA's slice of the spill (row stride 160)
  load_norm_rows(rep, d, cand, off, j0, nl, sD, snrm, HB_PER, gD);
  for (int q = tid; q < HB_BM_WORDS; q += blockDim.x) bm[q] = 0u;
  if (tid == 0) cnt_s = 0;
  // mean: ONE sequential sum over the candidates in order (D.mean(axis=1) adds candidate by candidate): CTA r continues
  // the partial of CTA r-1, the last one divides and hands mu (= the initial w) to everybody
  if (cr == 0 && tid < 160) spart[tid] = 0.f;
  cluster_sync_all();
  for (uint32_t r = 0; r < HB_CTAS; ++r) {
    if (cr == r && tid < 160) {
      float acc = spart[tid];
      for (int j = 0; j < nl; ++j) acc = __fadd_rn(acc, j < HB_PER ? sD[j * 160 + tid] : gD[(long long)(j - HB_PER) * 160 + tid]);
      if (r + 1 < HB_CTAS) st_cluster_f32(map_to_cta(spart + tid, r + 1), acc);
      else {
        const float mv = tid < d ? __fdiv_rn(acc, (float)n) : 0.f;
        for (uint32_t q = 0; q < HB_CTAS; ++q) { st_cluster_f32(map_to_cta(smu + tid, q), mv); st_cluster_f32(map_to_cta(sw + tid, q), mv); }
      }
    }
    cluster_sync_all();
  }
  const int steps = max_steps[s];
  const uint32_t av = map_to_cta(gv, 0), aj = map_to_cta(gj, 0);
  for (int step = 0; step < steps; ++step) {
    float fv; int fj;
    local_argmax(sD, sw, nl, bestv, bestj, fv, fj, HB_PER, gD);
    if (tid == 0) {                                // (value, GLOBAL candidate index) of this CTA -> CTA 0
      st_cluster_f32(av + 4u * cr, nl > 0 ? fv : -INFINITY);
      st_cluster_s32(aj + 4u * cr, nl > 0 ? j0 + fj : 0x7fffffff);
    }
    cluster_sync_all();
    float bvv = -INFINITY; int bjj = 0x7fffffff;   // every CTA takes the first maximum of the eight (lower index wins ties)
    for (int q = 0; q < HB_CTAS; ++q) {
      float v; int jx;
      asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(av + 4u * q) : "memory");
      asm volatile("ld.shared::cluster.s32 %0, [%1];" : "=r"(jx) : "r"(aj + 4u * q) : "memory");
      if (v > bvv || (v == bvv && jx < bjj)) { bvv = v; bjj = jx; }
    }
    if (bjj < 0 || bjj >= n) bjj = 0;              // all-NaN dots: index 0, like np.argmax
    const bool is_new = !(bm[bjj >> 5] >> (bjj & 31) & 1u);
    if (bjj >= j0 && bjj < j0 + nl) {              // owner: record the pick, broadcast its row into every CTA
      if (tid == 0 && is_new) picks[off + cnt_s] = bjj;
      if (tid < 160) {
        const int lj = bjj - j0;
        const float v = lj < HB_PER ? sD[lj * 160 + tid] : gD[(long long)(lj - HB_PER) * 160 + tid];
        for (uint32_t q = 0; q < HB_CTAS; ++q) st_cluster_f32(map_to_cta(srow + tid, q), v);
      }
    }
    cluster_sync_all();                            // srow has landed everywhere; everyone has read gv / gj and the bitmap
    if (tid < 160) sw[tid] = __fsub_rn(__fadd_rn(sw[tid], smu[tid]), srow[tid]);
    if (tid == 0 && is_new) { bm[bjj >> 5] |= 1u << (bjj & 31); cnt_s = cnt_s + 1; }
    __syncthreads();
    if (cnt_s == m) break;                         // replicated count: every CTA of the cluster leaves at the same step
  }
  if (cr == 0 && tid == 0) n_picked[s] = cnt_s;
  cluster_sync_all();                              // no CTA exits while a peer may still address its shared memory
}

}  // namespace ader

using namespace ader;

// Dn: rows of stride 160 (spill of k_herding_big) or d (k_herding, the only form of hidden_units > 160)
static size_t dn_floats(const AderModel* m, int32_t N) { return (size_t)N * (m->d > 160 ? m->d : 160); }

extern "C" size_t ader_herding_ws_bytes(const AderModel* m, int32_t N) {
  if (check_model(m) || N <= 0) return 0;
  // [Dn fp32 (global-memory fallback for segments > 2800)] [selected N] [class lists 4 x N] [counters]
  return align_up(sizeof(float) * dn_floats(m, N)) + align_up(sizeof(int) * (size_t)N) + 4 * align_up(sizeof(int) * (size_t)N) + 256;
}

extern "C" int32_t ader_herding_segmented(const AderModel* m, const float* rep, int32_t N, const int32_t* cand,
                                          const int32_t* seg_off, int32_t n_seg, const int32_t* quota,
                                          const int32_t* max_steps, void* ws, int32_t* picks, int32_t* n_picked,
                                          void* stream) {
  if (int e = check_model(m)) return e;
  ADER_CHECK_ARG(rep && cand && seg_off && quota && max_steps && ws && picks && n_picked, "herding: NULL pointer");
  ADER_CHECK_ARG(N > 0 && n_seg > 0, "herding: empty input");
  cudaStream_t st = (cudaStream_t)stream;
  char* base = (char*)ws; size_t o = 0;
  auto take = [&](size_t n) { char* p = base + o; o += align_up(n); return p; };
  float* Dn = (float*)take(sizeof(float) * dn_floats(m, N));
  int* selected = (int*)take(sizeof(int) * (size_t)N);
  int* lists[4];
  for (int k = 0; k < 4; ++k) lists[k] = (int*)take(sizeof(int) * (size_t)N);
  int* cnt = (int*)take(256);
  static const bool v1 = [] { const char* e = getenv("ADER_B200_HERDING"); return e && e[0] == '1'; }();
  if (v1 || path_check(m, ADER_PATH_HERDING_ONCHIP, false)) {   // first generation: CTA per segment, D in global memory
    k_herding<<<n_seg, 256, 0, st>>>(rep, m->d, cand, seg_off, quota, max_steps, Dn, selected, picks, n_picked, nullptr, nullptr);
    ADER_CHECK_LAUNCH("herding");
    return 0;
  }
  constexpr int SMEM_MID = (HM_MAX * 160 + 2 * 160 + HM_MAX) * 4;
  constexpr int SMEM_BIG = (HB_PER * 160 + 4 * 160 + HB_PER) * 4 + HB_BM_WORDS * 4;
  if (int e = kernel_ready<k_herding_mid>(SMEM_MID, "k_herding_mid")) return e;
  if (int e = kernel_ready<k_herding_big>(SMEM_BIG, "k_herding_big")) return e;
  cudaMemsetAsync(cnt, 0, 256, st);
  k_herding_classify<<<cdiv(n_seg, 256), 256, 0, st>>>(seg_off, quota, n_seg, cnt, lists[0], lists[1], lists[2], lists[3], n_picked);
  // grids are upper bounds of the class sizes (a class-c segment has more than its lower size bound of candidates);
  // CTAs beyond the device-side count leave at once
  const int g_small = n_seg, g_mid = N / (HS_MAX + 1) + 1, g_big = N / (HM_MAX + 1) + 1, g_huge = N / (HB_NMAX + 1) + 1;
  k_herding_small<<<cdiv((long long)g_small * 32, 256), 256, 0, st>>>(rep, m->d, cand, seg_off, quota, max_steps, lists[0], cnt, picks, n_picked);
  k_herding_mid<<<g_mid < n_seg ? g_mid : n_seg, 256, SMEM_MID, st>>>(rep, m->d, cand, seg_off, quota, max_steps, lists[1], cnt, selected, picks, n_picked);
  k_herding_big<<<(g_big < n_seg ? g_big : n_seg) * HB_CTAS, 256, SMEM_BIG, st>>>(rep, m->d, cand, seg_off, quota, max_steps, lists[2], cnt, Dn, picks, n_picked);
  k_herding<<<g_huge < n_seg ? g_huge : n_seg, 256, 0, st>>>(rep, m->d, cand, seg_off, quota, max_steps, Dn, selected, picks, n_picked, lists[3], cnt + 3);
  ADER_CHECK_LAUNCH("herding");
  return 0;
}
