// SASRec encoder over PACKED real tokens (modules.py:23-271, ADER.py:25-85), forward and
// backward, exact fp32.  Packing is exact w.r.t. the reference's dense-over-padding graph
// (SURVEY A.1 / A.10): padded keys get exactly zero attention weight for real queries and
// padded rows never reach `rep`, so only the T = sum(len) real tokens are computed.
//
// Layout in HBM: every activation is a [T, d] fp32 matrix in row order of (session row, position);
// row r owns tokens row_off[r] .. row_off[r+1).  T lives on the device (row_off[M]) so the whole
// step is stream-ordered with no host synchronisation; grids are sized for the capacity Tcap and
// surplus CTAs exit at once.
#include "common.cuh"

namespace ader {

constexpr int NSLOT = 8;          // per-block [Tcap,d] activation slots
constexpr int SPLITS = 21;        // split-K partials for weight / LN / bias gradients (21 x 7 problems = 147 CTAs: one wave of 148 SMs)
constexpr int PG_LANES = 6;       // token lanes per column in the LN / position gradient reductions (160 x 6 = 960 threads)
constexpr int PG_LANES_WIDE = 4;  // the same for hidden_units > 160 (256 x 4 = 1024 threads)

// workspace flag words: packing / overflow flags.  k_row_len (first kernel of every forward) zeroes them.
constexpr int N_WS_FLAGS = 4;

struct EncWs {
  int *row_len, *row_off, *tok_row, *tok_id, *flags;
  float* slot[8][NSLOT];           // [block][slot]
  float *mean1[8], *rstd1[8], *mean2[8], *rstd2[8], *probs[8];
  float* xfinal; float *meanf, *rstdf;
  void* wshadow;                   // fused path: bf16 weight shadows, NB x 10 x [160][168]
  size_t bytes;
};

static EncWs carve_enc(const AderModel* m, int M, int Tcap, char* base) {
  EncWs w; size_t o = 0;
  auto take = [&](size_t n) { char* p = base ? base + o : nullptr; o += align_up(n); return p; };
  const size_t d = m->d;
  w.row_len = (int*)take(sizeof(int) * M);
  w.row_off = (int*)take(sizeof(int) * (M + 1));
  w.tok_row = (int*)take(sizeof(int) * Tcap);
  w.tok_id  = (int*)take(sizeof(int) * Tcap);
  w.flags   = (int*)take(sizeof(int) * N_WS_FLAGS);
  for (int b = 0; b < m->num_blocks; ++b) {
    for (int s = 0; s < NSLOT; ++s) w.slot[b][s] = (float*)take(sizeof(float) * Tcap * d);
    w.mean1[b] = (float*)take(sizeof(float) * Tcap); w.rstd1[b] = (float*)take(sizeof(float) * Tcap);
    w.mean2[b] = (float*)take(sizeof(float) * Tcap); w.rstd2[b] = (float*)take(sizeof(float) * Tcap);
    w.probs[b] = (float*)take(sizeof(float) * (size_t)m->num_heads * Tcap * m->maxlen);
  }
  w.xfinal = (float*)take(sizeof(float) * Tcap * d);
  w.meanf = (float*)take(sizeof(float) * M); w.rstdf = (float*)take(sizeof(float) * M);
  w.wshadow = take((size_t)m->num_blocks * 10 * 160 * 168 * 2);
  w.bytes = o;
  return w;
}

struct BwdWs {
  float* g[11];          // gX, gXin, gO, gH, gZ, gY, gQ, gK, gV, gQ1, spare
  float* partial;        // [SPLITS][dense_count]
  int *keys[2], *vals[2], *hist;
  float* Dv;             // fused path: per-token softmax-backward row dots
  float* spart; int* scount;   // windowed scatter: partial slots [windows][2][SPAD], arrival counters [windows]
  int2* sbounds;               // [windows] segment head of a window's first run / segment end of its last run (scatter plan)
  float* g2[8];          // fused path: second set of gO..gQ1 (blocks alternate sets, so the weight-gradient kernel of
                         // block b may still read its set while block b-1's data-gradient kernels write the other)
  size_t bytes;
};
static int sort_tiles(int Tcap) { return cdiv(Tcap, 2048); }
static BwdWs carve_bwd(const AderModel* m, int M, int Tcap, char* base) {
  BwdWs w; size_t o = 0;
  auto take = [&](size_t n) { char* p = base ? base + o : nullptr; o += align_up(n); return p; };
  Layout l = make_layout(m);
  for (int i = 0; i < 11; ++i) w.g[i] = (float*)take(sizeof(float) * (size_t)Tcap * m->d);
  w.partial = (float*)take(sizeof(float) * (size_t)SPLITS * l.dense_count());
  for (int i = 0; i < 2; ++i) { w.keys[i] = (int*)take(sizeof(int) * Tcap); w.vals[i] = (int*)take(sizeof(int) * Tcap); }
  w.hist = (int*)take(sizeof(int) * 256 * (size_t)sort_tiles(Tcap));
  w.Dv = (float*)take(sizeof(float) * Tcap);
  for (int i = 0; i < 8; ++i) w.g2[i] = (float*)take(sizeof(float) * (size_t)Tcap * m->d);
  w.spart = (float*)take(sizeof(float) * (size_t)cdiv(Tcap, 16) * 2 * 256);
  w.scount = (int*)take(sizeof(int) * (size_t)cdiv(Tcap, 16));
  w.sbounds = (int2*)take(sizeof(int2) * (size_t)cdiv(Tcap, 16));
  w.bytes = o;
  return w;
}

// ------------------------------------------------------------------------------------------
// packing
// ------------------------------------------------------------------------------------------
__global__ void k_row_len(const int* __restrict__ ids, int M, int L, int* __restrict__ row_len, int* __restrict__ flags) {
  if (blockIdx.x == 0) for (int i = threadIdx.x; i < N_WS_FLAGS; i += blockDim.x) flags[i] = 0;   // (a memset node costs ~10 us in a graph)
  int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (r >= M) return;
  int c = 0;
  for (int j = lane; j < L; j += 32) c += (ids[(long long)r * L + j] != 0);
#pragma unroll
  for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if (lane == 0) row_len[r] = c;
}

// single CTA exclusive scan; row_off[M] = T (clamped to Tcap, overflow flagged)
__global__ void __launch_bounds__(1024) k_scan_rows(const int* __restrict__ row_len, int M, int Tcap,
                                                    int* __restrict__ row_off, int* __restrict__ flags) {
  __shared__ int warp_sum[32];
  __shared__ int carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int base = 0; base < M; base += 1024) {
    int i = base + threadIdx.x;
    int v = (i < M) ? row_len[i] : 0;
    int x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) warp_sum[wid] = x;
    __syncthreads();
    if (wid == 0) {
      int s = warp_sum[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += y; }
      warp_sum[lane] = s;
    }
    __syncthreads();
    int excl = carry + (wid ? warp_sum[wid - 1] : 0) + x - v;
    if (i < M) row_off[i] = excl;
    __syncthreads();
    if (threadIdx.x == 1023) carry = excl + v;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    int T = carry;
    if (T > Tcap) { flags[0] = T; T = Tcap; }   // overflow: host checks flags[0] lazily
    row_off[M] = T;
  }
}

__global__ void k_fill_tok(const int* __restrict__ ids, const int* __restrict__ row_len,
                           const int* __restrict__ row_off, int M, int L, int Tcap,
                           int* __restrict__ tok_row, int* __restrict__ tok_id) {
  int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (r >= M) return;
  int n = row_len[r], off = row_off[r];
  for (int i = lane; i < n; i += 32) {
    if (off + i < Tcap) {
      tok_row[off + i] = r;
      tok_id[off + i] = ids[(long long)r * L + (L - n + i)];   // real tokens are the suffix (util.py:161-169)
    }
  }
}

// ------------------------------------------------------------------------------------------
// embedding: x = (E0[id]*sqrt(d) + P[pos]) * dropout     (modules.py:124-130, ADER.py:41-60)
// ------------------------------------------------------------------------------------------
__global__ void k_embed(const float* __restrict__ table, const float* __restrict__ pos_table,
                        const int* __restrict__ tok_row, const int* __restrict__ tok_id,
                        const int* __restrict__ row_len, const int* __restrict__ row_off,
                        const int* __restrict__ dT, int d, int L, float sqrt_d,
                        float drop_p, uint64_t seed, float* __restrict__ x) {
  long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  int T = *dT;
  if (e >= (long long)T * d) return;
  int t = (int)(e / d), c = (int)(e % d);
  int r = tok_row[t];
  int p = L - row_len[r] + (t - row_off[r]);
  int id = tok_id[t];
  float v = table[(long long)id * d + c] * sqrt_d + pos_table[p * d + c];
  if (drop_p > 0.f) v *= drop_scale(seed, 0u, (uint64_t)e, drop_p);
  x[e] = v;
}

// ------------------------------------------------------------------------------------------
// LayerNorm (modules.py:44-48): population variance, eps inside the sqrt.  Warp per token.
// ------------------------------------------------------------------------------------------
constexpr int LN_MAXE = 8;  // d <= 256
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ void ln_row_fwd(const float* __restrict__ x, float* __restrict__ out,
                                           const float* __restrict__ beta, const float* __restrict__ gamma,
                                           int d, int lane, float& mean_o, float& rstd_o) {
  float v[LN_MAXE]; float s = 0.f;
#pragma unroll
  for (int i = 0; i < LN_MAXE; ++i) { int c = lane + 32 * i; v[i] = (c < d) ? x[c] : 0.f; s += v[i]; }
  float mean = warp_sum(s) / (float)d;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < LN_MAXE; ++i) { int c = lane + 32 * i; if (c < d) { float t = v[i] - mean; q += t * t; } }
  float var = warp_sum(q) / (float)d;
  float rstd = 1.0f / sqrtf(var + 1e-8f);
#pragma unroll
  for (int i = 0; i < LN_MAXE; ++i) { int c = lane + 32 * i; if (c < d) out[c] = gamma[c] * ((v[i] - mean) * rstd) + beta[c]; }
  mean_o = mean; rstd_o = rstd;
}

__global__ void k_ln_fwd(const float* __restrict__ x, float* __restrict__ out, float* __restrict__ mean,
                         float* __restrict__ rstd, const float* __restrict__ beta,
                         const float* __restrict__ gamma, const int* __restrict__ dT, int d) {
  int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (t >= *dT) return;
  float mu, rs;
  ln_row_fwd(x + (long long)t * d, out + (long long)t * d, beta, gamma, d, lane, mu, rs);
  if (lane == 0) { mean[t] = mu; rstd[t] = rs; }
}

// final LN on the last token of every row only (ADER.py:82-85): rep[r] = LN(x[last(r)])
__global__ void k_ln_last_fwd(const float* __restrict__ x, const int* __restrict__ row_len,
                              const int* __restrict__ row_off, int M, float* __restrict__ rep,
                              float* __restrict__ mean, float* __restrict__ rstd,
                              const float* __restrict__ beta, const float* __restrict__ gamma, int d) {
  pdl_wait(); pdl_go();
  int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (r >= M) return;
  int n = row_len[r];
  if (n == 0) {   // empty row (no usable session): defined as zeros, carries no gradient
    for (int c = lane; c < d; c += 32) rep[(long long)r * d + c] = 0.f;
    if (lane == 0) { mean[r] = 0.f; rstd[r] = 0.f; }
    return;
  }
  int t = row_off[r] + n - 1;
  float mu, rs;
  ln_row_fwd(x + (long long)t * d, rep + (long long)r * d, beta, gamma, d, lane, mu, rs);
  if (lane == 0) { mean[r] = mu; rstd[r] = rs; }
}

// dx (+)= LN backward.  g = dout*gamma; dx = rstd*(g - mean(g) - xhat*mean(g*xhat))
__device__ __forceinline__ void ln_row_bwd(const float* __restrict__ dout, const float* __restrict__ x,
                                           float mean, float rstd, const float* __restrict__ gamma,
                                           float* __restrict__ dx, int d, int lane, bool accumulate) {
  float g[LN_MAXE], xh[LN_MAXE]; float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int i = 0; i < LN_MAXE; ++i) {
    int c = lane + 32 * i;
    if (c < d) { xh[i] = (x[c] - mean) * rstd; g[i] = dout[c] * gamma[c]; s1 += g[i]; s2 += g[i] * xh[i]; }
    else { xh[i] = 0.f; g[i] = 0.f; }
  }
  s1 = warp_sum(s1) / (float)d; s2 = warp_sum(s2) / (float)d;
#pragma unroll
  for (int i = 0; i < LN_MAXE; ++i) {
    int c = lane + 32 * i;
    if (c < d) { float v = rstd * (g[i] - s1 - xh[i] * s2); dx[c] = accumulate ? dx[c] + v : v; }
  }
}

__global__ void k_ln_bwd(const float* __restrict__ dout, const float* __restrict__ x,
                         const float* __restrict__ mean, const float* __restrict__ rstd,
                         const float* __restrict__ gamma, float* __restrict__ dx,
                         const int* __restrict__ dT, int d, int accumulate) {
  int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (t >= *dT) return;
  long long o = (long long)t * d;
  ln_row_bwd(dout + o, x + o, mean[t], rstd[t], gamma, dx + o, d, lane, accumulate != 0);
}

// gX[t] = LNf backward of d_rep[row] when t is the last token of its row, else 0.
__global__ void k_lnf_bwd(const float* __restrict__ d_rep, const float* __restrict__ x,
                          const float* __restrict__ mean, const float* __restrict__ rstd,
                          const float* __restrict__ gamma, const int* __restrict__ tok_row,
                          const int* __restrict__ row_off, float* __restrict__ gx,
                          const int* __restrict__ dT, int d) {
  pdl_wait(); pdl_go();
  int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (t >= *dT) return;
  int r = tok_row[t];
  long long o = (long long)t * d;
  if (t != row_off[r + 1] - 1) { for (int c = lane; c < d; c += 32) gx[o + c] = 0.f; return; }
  ln_row_bwd(d_rep + (long long)r * d, x + o, mean[r], rstd[r], gamma, gx + o, d, lane, false);
}

// The same with the d_rep reduction of the loss group folded in (fused step): warp t < Tcap is token t as above, but the
// warp of a row's last token first sums the row's split partials (the left-to-right sum of tc::k_reduce_drep, all loads of
// a trip in flight together) and writes d_rep[row]; warps Tcap.. cover the rows without tokens (d_rep only).  One launch
// and one L2 round trip less on the critical chain, bit-identical values.
__global__ void k_lnf_bwd_drep(const DrepFuse df, float* d_rep, const float* __restrict__ x,
                               const float* __restrict__ mean, const float* __restrict__ rstd,
                               const float* __restrict__ gamma, const int* __restrict__ tok_row,
                               const int* __restrict__ row_off, const int* __restrict__ row_len, float* __restrict__ gx,
                               const int* __restrict__ dT, int M, int Tcap, int d) {
  pdl_wait(); pdl_go();
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  int r; long long o = 0; bool do_ln;
  if (w < Tcap) {
    if (w >= *dT) return;
    r = tok_row[w];
    o = (long long)w * d;
    if (w != row_off[r + 1] - 1) { for (int c = lane; c < d; c += 32) gx[o + c] = 0.f; return; }
    do_ln = true;
  } else {
    r = w - Tcap;
    if (r >= M || row_len[r] != 0) return;
    do_ln = false;
  }
  const size_t cs = (size_t)df.rows_pad * df.kp;
  const float* p0 = df.part + (size_t)r * df.kp + lane;
  float s[LN_MAXE];
#pragma unroll
  for (int e = 0; e < LN_MAXE; ++e) s[e] = 0.f;
  int k = 0;
  for (; k + 8 <= df.n_chunks; k += 8) {          // eight chunks x all columns of the row in flight per trip
    float v[LN_MAXE][8];
#pragma unroll
    for (int e = 0; e < LN_MAXE; ++e)
#pragma unroll
      for (int j = 0; j < 8; ++j) v[e][j] = (lane + 32 * e < d) ? __ldcg(p0 + 32 * e + (size_t)(k + j) * cs) : 0.f;
#pragma unroll
    for (int e = 0; e < LN_MAXE; ++e)
#pragma unroll
      for (int j = 0; j < 8; ++j) s[e] += v[e][j];
  }
  for (; k < df.n_chunks; ++k) {
#pragma unroll
    for (int e = 0; e < LN_MAXE; ++e) if (lane + 32 * e < d) s[e] += __ldcg(p0 + 32 * e + (size_t)k * cs);
  }
#pragma unroll
  for (int e = 0; e < LN_MAXE; ++e) {
    const int c = lane + 32 * e;
    if (c < d) {
      float t = s[e];
      if (df.u && r >= df.n_train) t -= df.u[(size_t)(r - df.u_row0) * df.kp + c];
      d_rep[(long long)r * d + c] = t;
    }
  }
  if (!do_ln) return;
  __threadfence_block();        // the row below is read back by the lanes that wrote it
  ln_row_bwd(d_rep + (long long)r * d, x + o, mean[r], rstd[r], gamma, gx + o, d, lane, false);
}

// partial LN parameter gradients: dbeta[c] = sum_t dout[t,c]; dgamma[c] = sum_t dout[t,c]*xhat[t,c]
// split s sums tokens [s*chunk, (s+1)*chunk) sequentially -> deterministic.
// rows != nullptr: "last token" mode (dout indexed by row, x by last token of the row, count = M).
template <int LANES>
__global__ void k_ln_param_grad(const float* __restrict__ dout, const float* __restrict__ x,
                                const float* __restrict__ mean, const float* __restrict__ rstd,
                                const int* __restrict__ dT, int count_host,
                                const int* __restrict__ row_len, const int* __restrict__ row_off,
                                int d, float* __restrict__ pbeta, float* __restrict__ pgamma,
                                long long split_stride) {
  // blockDim = (ceil32(d), LANES): thread (c, k) sums tokens lo+k, lo+k+LANES, ... ; the
  // LANES partial sums are then added in lane order -> deterministic.
  __shared__ float sb_s[LANES][256], sg_s[LANES][256];
  const int c = threadIdx.x, k = threadIdx.y;
  const int s = blockIdx.x;
  const int count = row_off ? count_host : *dT;
  const int chunk = (count + gridDim.x - 1) / gridDim.x;
  const int lo = s * chunk, hi = min(count, lo + chunk);
  float sb = 0.f, sg = 0.f;
  if (c < d) {
    for (int i = lo + k; i < hi; i += LANES) {
      long long xo, go; float mu, rs;
      if (row_off) {
        if (row_len[i] == 0) continue;
        xo = (long long)(row_off[i + 1] - 1) * d; go = (long long)i * d; mu = mean[i]; rs = rstd[i];
      } else { xo = go = (long long)i * d; mu = mean[i]; rs = rstd[i]; }
      float g = dout[go + c];
      sb += g; sg += g * ((x[xo + c] - mu) * rs);
    }
  }
  sb_s[k][c] = sb; sg_s[k][c] = sg;
  __syncthreads();
  if (k == 0 && c < d) {
    float tb = 0.f, tg = 0.f;
#pragma unroll
    for (int q = 0; q < LANES; ++q) { tb += sb_s[q][c]; tg += sg_s[q][c]; }
    pbeta[(long long)s * split_stride + c] = tb;
    pgamma[(long long)s * split_stride + c] = tg;
  }
}

// ------------------------------------------------------------------------------------------
// causal self-attention per session row (modules.py:177-223).  CTA per row, 4 warps.
// ------------------------------------------------------------------------------------------
// ---- shared-memory staging helpers (d even; rows are contiguous [n, d] in global memory) ------
// row-major copy: dst[i*d + c]
__device__ __forceinline__ void stage_rows(const float* __restrict__ src, float* __restrict__ dst, int n, int d) {
  const int n2 = (n * d) >> 1;
  const float2* s2 = reinterpret_cast<const float2*>(src);
  float2* d2 = reinterpret_cast<float2*>(dst);
  for (int base = threadIdx.x; base < n2; base += 4 * blockDim.x) {
    float2 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) { int idx = base + u * blockDim.x; if (idx < n2) v[u] = s2[idx]; }
#pragma unroll
    for (int u = 0; u < 4; ++u) { int idx = base + u * blockDim.x; if (idx < n2) d2[idx] = v[u]; }
  }
}
// transposed copy: dst[c*LP + i]; columns i in [n, LP) are zero-filled
__device__ __forceinline__ void stage_rows_t(const float* __restrict__ src, float* __restrict__ dst, int n, int d, int LP) {
  const int n2 = (n * d) >> 1;
  const float2* s2 = reinterpret_cast<const float2*>(src);
  for (int base = threadIdx.x; base < n2; base += 4 * blockDim.x) {
    float2 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) { int idx = base + u * blockDim.x; if (idx < n2) v[u] = s2[idx]; }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      int idx = base + u * blockDim.x;
      if (idx < n2) { int e = idx * 2; int i = e / d, c = e - i * d; dst[c * LP + i] = v[u].x; dst[(c + 1) * LP + i] = v[u].y; }
    }
  }
  const int pad = LP - n;
  for (int idx = threadIdx.x; idx < d * pad; idx += blockDim.x) { int c = idx / pad, i = n + idx % pad; dst[c * LP + i] = 0.f; }
}

// Attention kernels: one CTA (8 warps) per session row.  A warp owns a block of 4 queries (or 4 keys in
// the transposed products); operands are staged so that the per-k inner step is one conflict-free LDS
// (lanes over keys / features) + one broadcast LDS.128 (the 4 queries) feeding 4 independent FMA chains.
// Tile sizes and shared-memory budgets: common.cuh (attn_fwd_smem / attn_bwd_smem).

__global__ void __launch_bounds__(ATT_THREADS) k_attn_fwd(const float* __restrict__ Q, const float* __restrict__ K,
                                                          const float* __restrict__ V, const float* __restrict__ Q1,
                                                          const int* __restrict__ row_len, const int* __restrict__ row_off,
                                                          int d, int nh, int L, int Tcap, float drop_p, uint64_t seed,
                                                          uint32_t site, float* __restrict__ probs, float* __restrict__ Y) {
  extern __shared__ __align__(16) float sm[];
  const int r = blockIdx.x;
  const int n = row_len[r];
  if (n == 0) return;
  const int off = row_off[r];
  const int LP = att_lp(L);
  float* Qt = sm;                    // [d][LP]
  float* Kt = Qt + d * LP;           // [d][LP]
  float* Vs = Kt + d * LP;           // [L][d]
  float* Pt = Vs + al4(L * d);       // [ATT_WARPS][64][4]
  stage_rows_t(Q + (long long)off * d, Qt, n, d, LP);
  stage_rows_t(K + (long long)off * d, Kt, n, d, LP);
  stage_rows(V + (long long)off * d, Vs, n, d);
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int dh = d / nh;
  const float denom = sqrtf((float)dh);
  float* pw = Pt + warp * 256;
  const int nblk = (n + 3) >> 2;
  for (int h = 0; h < nh; ++h) {
    const int hc = h * dh;
    for (int blk = warp; blk < nblk; blk += ATT_WARPS) {
      const int i0 = blk * 4;
      const int imax = min(i0 + 3, n - 1);
      float s[2][4];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int j = lane + 32 * u;
#pragma unroll
        for (int q = 0; q < 4; ++q) s[u][q] = -INFINITY;
        if (32 * u > imax) continue;                     // warp-uniform
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        const int jj = min(j, LP - 1);
#pragma unroll 4
        for (int k = 0; k < dh; ++k) {
          const float kv = Kt[(hc + k) * LP + jj];
          const float4 q4 = *reinterpret_cast<const float4*>(&Qt[(hc + k) * LP + i0]);
          acc[0] = fmaf(q4.x, kv, acc[0]); acc[1] = fmaf(q4.y, kv, acc[1]);
          acc[2] = fmaf(q4.z, kv, acc[2]); acc[3] = fmaf(q4.w, kv, acc[3]);
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) if (j <= i0 + q && i0 + q < n) s[u][q] = acc[q] / denom;
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int i = i0 + q;
        if (i >= n) break;                               // warp-uniform
        const float mx = warp_max(fmaxf(s[0][q], s[1][q]));
        const float e0 = (lane <= i) ? expf(s[0][q] - mx) : 0.f;
        const float e1 = (lane + 32 <= i) ? expf(s[1][q] - mx) : 0.f;
        const float sum = warp_sum(e0 + e1);
        const float p[2] = {e0 / sum, e1 / sum};
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int j = lane + 32 * u;
          float pd = 0.f;
          if (j < L) {
            const long long po = ((long long)h * Tcap + off + i) * L + j;
            probs[po] = p[u];
            pd = p[u];
            if (drop_p > 0.f) pd *= drop_scale(seed, site, (uint64_t)po, drop_p);
          }
          pw[j * 4 + q] = pd;
        }
      }
      for (int q = imax - i0 + 1; q < 4; ++q) { pw[lane * 4 + q] = 0.f; pw[(lane + 32) * 4 + q] = 0.f; }
      __syncwarp();
      for (int c = lane; c < dh; c += 32) {
        float o[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
        for (int j = 0; j <= imax; ++j) {
          const float v = Vs[j * d + hc + c];
          const float4 p4 = *reinterpret_cast<const float4*>(&pw[j * 4]);
          o[0] = fmaf(p4.x, v, o[0]); o[1] = fmaf(p4.y, v, o[1]); o[2] = fmaf(p4.z, v, o[2]); o[3] = fmaf(p4.w, v, o[3]);
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          if (i0 + q < n) {
            const long long g = (long long)(off + i0 + q) * d + hc + c;
            Y[g] = o[q] + Q1[g];                  // residual on the NORMALISED queries (modules.py:223)
          }
        }
      }
      __syncwarp();
    }
  }
}

__global__ void __launch_bounds__(ATT_THREADS) k_attn_bwd(const float* __restrict__ Q, const float* __restrict__ K,
                                                          const float* __restrict__ V, const float* __restrict__ probs,
                                                          const float* __restrict__ gY, const int* __restrict__ row_len,
                                                          const int* __restrict__ row_off, int d, int nh, int L, int Tcap,
                                                          float drop_p, uint64_t seed, uint32_t site,
                                                          float* __restrict__ gQ, float* __restrict__ gK,
                                                          float* __restrict__ gV) {
  extern __shared__ __align__(16) float sm[];
  const int r = blockIdx.x;
  const int n = row_len[r];
  if (n == 0) return;
  const int off = row_off[r];
  const int LP = att_lp(L);
  float* Gt = sm;                    // gY transposed [d][LP]
  float* Vt = Gt + d * LP;           // V transposed  [d][LP]
  float* Qs = Vt + d * LP;           // [L][d]
  float* Ks = Qs + al4(L * d);       // [L][d]
  float* Gs = Ks + al4(L * d);       // [L][d]
  float* dSs = Gs + al4(L * d);      // [L][LP]   dS[i][j]
  float* dSt = dSs + L * LP;         // [L][LP]   dS^T[j][i]
  float* Pds = dSt + L * LP;         // [L][LP]   dropped probs [i][j]
  stage_rows_t(gY + (long long)off * d, Gt, n, d, LP);
  stage_rows_t(V + (long long)off * d, Vt, n, d, LP);
  stage_rows(Q + (long long)off * d, Qs, n, d);
  stage_rows(K + (long long)off * d, Ks, n, d);
  stage_rows(gY + (long long)off * d, Gs, n, d);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int dh = d / nh;
  const float denom = sqrtf((float)dh);
  const int nblk = (n + 3) >> 2;
  for (int h = 0; h < nh; ++h) {
    const int hc = h * dh;
    // zero dS / dS^T / Pd (entries above the diagonal and the LP padding must read as 0)
    for (int idx = threadIdx.x; idx < 3 * L * LP; idx += blockDim.x) dSs[idx] = 0.f;
    __syncthreads();
    // phase 1: dP = gY . V^T (block of 4 queries x 32 keys), softmax backward
    for (int blk = warp; blk < nblk; blk += ATT_WARPS) {
      const int i0 = blk * 4;
      const int imax = min(i0 + 3, n - 1);
      float dp[2][4];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
#pragma unroll
        for (int q = 0; q < 4; ++q) dp[u][q] = 0.f;
        if (32 * u > imax) continue;
        const int jj = min(lane + 32 * u, LP - 1);
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
        for (int k = 0; k < dh; ++k) {
          const float vv = Vt[(hc + k) * LP + jj];
          const float4 g4 = *reinterpret_cast<const float4*>(&Gt[(hc + k) * LP + i0]);
          acc[0] = fmaf(g4.x, vv, acc[0]); acc[1] = fmaf(g4.y, vv, acc[1]);
          acc[2] = fmaf(g4.z, vv, acc[2]); acc[3] = fmaf(g4.w, vv, acc[3]);
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) dp[u][q] = acc[q];
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int i = i0 + q;
        if (i >= n) break;
        float P[2], dP[2], scl[2];
        float rowdot = 0.f;
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int j = lane + 32 * u;
          P[u] = 0.f; dP[u] = 0.f; scl[u] = 1.f;
          if (j <= i) {
            const long long po = ((long long)h * Tcap + off + i) * L + j;
            P[u] = probs[po];
            if (drop_p > 0.f) scl[u] = drop_scale(seed, site, (uint64_t)po, drop_p);
            dP[u] = dp[u][q] * scl[u];
            rowdot += dP[u] * P[u];
          }
        }
        rowdot = warp_sum(rowdot);
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int j = lane + 32 * u;
          if (j <= i) {
            const float ds = P[u] * (dP[u] - rowdot) / denom;
            dSs[i * LP + j] = ds; dSt[j * LP + i] = ds; Pds[i * LP + j] = P[u] * scl[u];
          }
        }
      }
    }
    __syncthreads();
    // phase 2a: gQ[i] = sum_{j<=i} dS[i][j] K[j]  (block of 4 queries, lanes over features)
    for (int blk = warp; blk < nblk; blk += ATT_WARPS) {
      const int i0 = blk * 4;
      const int imax = min(i0 + 3, n - 1);
      for (int c = lane; c < dh; c += 32) {
        float o[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
        for (int j = 0; j <= imax; ++j) {
          const float kv = Ks[j * d + hc + c];
          const float4 s4 = *reinterpret_cast<const float4*>(&dSt[j * LP + i0]);
          o[0] = fmaf(s4.x, kv, o[0]); o[1] = fmaf(s4.y, kv, o[1]); o[2] = fmaf(s4.z, kv, o[2]); o[3] = fmaf(s4.w, kv, o[3]);
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) if (i0 + q < n) gQ[(long long)(off + i0 + q) * d + hc + c] = o[q];
      }
    }
    // phase 2b: gK[j] = sum_{i>=j} dS[i][j] Q[i],  gV[j] = sum_{i>=j} Pd[i][j] gY[i]  (block of 4 keys)
    for (int blk = warp; blk < nblk; blk += ATT_WARPS) {
      const int j0 = blk * 4;
      for (int c = lane; c < dh; c += 32) {
        float ok[4] = {0.f, 0.f, 0.f, 0.f}, ov[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
        for (int i = j0; i < n; ++i) {
          const float qv = Qs[i * d + hc + c], gv = Gs[i * d + hc + c];
          const float4 s4 = *reinterpret_cast<const float4*>(&dSs[i * LP + j0]);
          const float4 p4 = *reinterpret_cast<const float4*>(&Pds[i * LP + j0]);
          ok[0] = fmaf(s4.x, qv, ok[0]); ok[1] = fmaf(s4.y, qv, ok[1]); ok[2] = fmaf(s4.z, qv, ok[2]); ok[3] = fmaf(s4.w, qv, ok[3]);
          ov[0] = fmaf(p4.x, gv, ov[0]); ov[1] = fmaf(p4.y, gv, ov[1]); ov[2] = fmaf(p4.z, gv, ov[2]); ov[3] = fmaf(p4.w, gv, ov[3]);
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          if (j0 + q < n) {
            gK[(long long)(off + j0 + q) * d + hc + c] = ok[q];
            gV[(long long)(off + j0 + q) * d + hc + c] = ov[q];
          }
        }
      }
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------
// small elementwise helpers
// ------------------------------------------------------------------------------------------
// out[e] = in[e] * dropmask(site, e)   (gradient of an output-dropout site)
__global__ void k_apply_drop(const float* in, float* out, const int* __restrict__ dT,
                             int d, float p, uint64_t seed, uint32_t site) {
  long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (long long)(*dT) * d) return;
  out[e] = in[e] * drop_scale(seed, site, (uint64_t)e, p);
}

// fused-step form of k_reduce_partials over the whole dense range: the reduced gradient is stored AND the TF1-Adam
// update of that element (optim.cu: adam_update_elem, the very expression k_adam evaluates) is applied in place;
// thread 0 bumps the step counter (every reader of it has finished by now)
__global__ void k_reduce_partials_adam(const float* __restrict__ partial, long long stride, int splits, long long n,
                                       float* __restrict__ gout, float* __restrict__ theta, float* __restrict__ am,
                                       float* __restrict__ av, int* __restrict__ state, float beta1, float beta2, float eps,
                                       float ewc_lambda, const float* __restrict__ fisher, const float* __restrict__ theta_star) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float lr_t = __int_as_float(state[1]);
  float th = theta[i], m1 = am[i], v1 = av[i];        // in flight with the partials
  float s = 0.f;
  int k = 0;
  for (; k + 8 <= splits; k += 8) {                   // left-to-right sum, eight loads in flight per trip
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = partial[(long long)(k + j) * stride + i];
#pragma unroll
    for (int j = 0; j < 8; ++j) s += v[j];
  }
  for (; k < splits; ++k) s += partial[(long long)k * stride + i];
  gout[i] = s;
  adam_update_elem(s, th, m1, v1, lr_t, beta1, beta2, eps, ewc_lambda, fisher ? fisher[i] : 0.f, theta_star ? theta_star[i] : 0.f);
  theta[i] = th; am[i] = m1; av[i] = v1;
  if (i == 0) state[0] += 1;
}

// grad_dense[i] = sum_s partial[s][i] for i in [lo, hi)
__global__ void k_reduce_partials(const float* __restrict__ partial, long long stride, int splits,
                                  long long lo, long long hi, float* __restrict__ out) {
  long long i = lo + (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= hi) return;
  float s = 0.f;
  for (int k = 0; k < splits; ++k) s += partial[(long long)k * stride + i];
  out[i] = s;
}

// position-table gradient: dP[p,c] = sum over rows having position p of dx0[token(r,p), c]
template <int LANES>
__global__ void k_pos_grad(const float* __restrict__ gx, const int* __restrict__ row_len,
                           const int* __restrict__ row_off, int M, int L, int d,
                           float drop_p, uint64_t seed0, const int* __restrict__ d_step, float* __restrict__ gpos,
                           long long split_stride) {
  const uint64_t seed = seed0 + (d_step ? (uint64_t)(uint32_t)__ldg(d_step) : 0ull);
  // grid (L, splits): CTA (p, s) sums the rows of chunk s that have position p into partial slot s.
  // blockDim = (ceil32(d), LANES): thread (c, k) sums rows lo+k, lo+k+LANES, ...; lanes reduced in fixed order.
  // (Round 2 tried eight rows per trip and ten positions per CTA with the row lengths fetched once: 23 us and 34 us in the
  // step against 16-19 us for this form -- the tail kernels run beside the last weight-gradient CTAs, and what a variant
  // gains in dependent trips it loses to registers / shared memory that no longer fit beside them.)
  __shared__ float part[LANES][256];
  const int p = blockIdx.x, c = threadIdx.x, k = threadIdx.y;
  const int chunk = (M + gridDim.y - 1) / gridDim.y;
  const int lo = blockIdx.y * chunk, hi = min(M, lo + chunk);
  gpos += (long long)blockIdx.y * split_stride;
  float s = 0.f;
  if (c < d) {
    for (int r = lo + k; r < hi; r += LANES) {
      int n = row_len[r];
      if (n >= L - p) {
        long long e = (long long)(row_off[r] + p - (L - n)) * d + c;
        float v = gx[e];
        if (drop_p > 0.f) v *= drop_scale(seed, 0u, (uint64_t)e, drop_p);
        s += v;
      }
    }
  }
  part[k][c] = s;
  __syncthreads();
  if (k == 0 && c < d) {
    float t = 0.f;
#pragma unroll
    for (int q = 0; q < LANES; ++q) t += part[q][c];
    gpos[p * d + c] = t;
  }
}

// block (ceil32(d) columns, token lanes) of the two reductions above: PG_LANES lanes up to d = 160, PG_LANES_WIDE above
template <typename... Args>
static void launch_ln_param_grad(dim3 grid, int d, cudaStream_t st, Args... args) {
  const int cols = ((d + 31) / 32) * 32;
  if (cols * PG_LANES <= 1024) k_ln_param_grad<PG_LANES><<<grid, dim3(cols, PG_LANES), 0, st>>>(args...);
  else k_ln_param_grad<PG_LANES_WIDE><<<grid, dim3(cols, PG_LANES_WIDE), 0, st>>>(args...);
}
template <typename... Args>
static void launch_pos_grad(dim3 grid, int d, cudaStream_t st, Args... args) {
  const int cols = ((d + 31) / 32) * 32;
  if (cols * PG_LANES <= 1024) k_pos_grad<PG_LANES><<<grid, dim3(cols, PG_LANES), 0, st>>>(args...);
  else k_pos_grad<PG_LANES_WIDE><<<grid, dim3(cols, PG_LANES_WIDE), 0, st>>>(args...);
}

// ------------------------------------------------------------------------------------------
// embedding-gradient scatter (subsystem 3): stable LSD radix sort of (item id, token) (the "plan", depends on the
// packed ids only) + windowed segmented reduction (k_scatter_apply).  Deterministic: every table row is a fixed
// function of the sorted order; the only float reductions to memory have exactly one contributor per address.
// ------------------------------------------------------------------------------------------
constexpr int SORT_TILE = 2048;

// start of the plan: arrival counters back to zero (a memset node costs ~10 us in a graph)
__global__ void k_plan_zero(int* __restrict__ scount, int n_count) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_count) scount[i] = 0;
}

__global__ void __launch_bounds__(256) k_sort_hist(const int* __restrict__ keys, const int* __restrict__ dT,
                                                   int shift, int ntiles, int* __restrict__ hist) {
  __shared__ int h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  const int T = *dT;
  const int base = blockIdx.x * SORT_TILE;
  for (int r = 0; r < SORT_TILE / 256; ++r) {
    int i = base + r * 256 + threadIdx.x;
    if (i < T) atomicAdd(&h[(keys[i] >> shift) & 255], 1);    // integer atomics: order-independent result
  }
  __syncthreads();
  hist[threadIdx.x * ntiles + blockIdx.x] = h[threadIdx.x];
}

// exclusive scan of hist (digit-major) in place; single CTA
__global__ void __launch_bounds__(1024) k_sort_scan(int* __restrict__ hist, int n) {
  __shared__ int warp_sum_s[32];
  __shared__ int carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int base = 0; base < n; base += 1024) {
    int i = base + threadIdx.x;
    int v = (i < n) ? hist[i] : 0;
    int x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) warp_sum_s[wid] = x;
    __syncthreads();
    if (wid == 0) {
      int s = warp_sum_s[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += y; }
      warp_sum_s[lane] = s;
    }
    __syncthreads();
    int excl = carry + (wid ? warp_sum_s[wid - 1] : 0) + x - v;
    if (i < n) hist[i] = excl;
    __syncthreads();
    if (threadIdx.x == 1023) carry = excl + v;
    __syncthreads();
  }
}

__global__ void __launch_bounds__(256) k_sort_scatter(const int* __restrict__ keys_in, const int* __restrict__ vals_in,
                                                      const int* __restrict__ dT, int shift, int ntiles,
                                                      const int* __restrict__ hist, int first_pass,
                                                      int* __restrict__ keys_out, int* __restrict__ vals_out) {
  __shared__ int running[256];
  __shared__ int cnt[8][256];
  const int T = *dT;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  running[tid] = hist[tid * ntiles + blockIdx.x];
  const int base = blockIdx.x * SORT_TILE;
  for (int r = 0; r < SORT_TILE / 256; ++r) {
#pragma unroll
    for (int w = 0; w < 8; ++w) cnt[w][tid] = 0;
    __syncthreads();
    int i = base + r * 256 + tid;
    bool valid = i < T;
    int key = valid ? keys_in[i] : 0;
    int val = valid ? (first_pass ? i : vals_in[i]) : 0;
    int digit = valid ? ((key >> shift) & 255) : 256 + lane;      // invalid lanes match nobody
    unsigned mask = __match_any_sync(0xffffffffu, digit);
    int rank_in_warp = __popc(mask & ((1u << lane) - 1u));
    if (valid && rank_in_warp == 0) cnt[warp][digit] = __popc(mask);
    __syncthreads();
    if (valid) {
      int pre = 0;
      for (int w = 0; w < warp; ++w) pre += cnt[w][digit];
      int dst = running[digit] + pre + rank_in_warp;
      keys_out[dst] = key; vals_out[dst] = val;
    }
    __syncthreads();
    int tot = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) tot += cnt[w][tid];
    running[tid] += tot;
    __syncthreads();
  }
}

// Segmented reduction over the sorted pairs, windowed: the (item id, token) pairs are radix-sorted OFF the
// critical path (the ids are known as soon as the batch is packed), so the part that has to wait for the gradient is
// one launch with no serial tail.  One warp per window of SW consecutive sorted positions: its SW gradient rows are
// fetched in one batch, runs of equal ids are summed in sorted (= token) order, and
//   * a run that is a whole segment goes to its table row with one reduction per element (the row has exactly one
//     contributor, so the result does not depend on any ordering),
//   * a run that is a PIECE of a longer segment (a hot item spanning several windows) is parked in a partial slot;
//     the last piece to arrive (per-segment arrival counter) adds the pieces in window order and writes the row.
// Every row is therefore a fixed function of the sorted order: deterministic, and a 230-occurrence item costs two
// dependent batches instead of fifteen.
constexpr int SW = 16;
static_assert(SW == 16, "k_seg_bounds (scatter plan) is written for windows of 16 positions");
constexpr int SPAD = 160 > LN_MAXE * 32 ? 160 : LN_MAXE * 32;      // floats per partial slot
// Plan: for every window of SW sorted positions, where the segment of its FIRST run starts (if that run continues from the
// previous window) and where the segment of its LAST run ends (if it continues into the next window).  Warp per window.
__global__ void __launch_bounds__(256) k_seg_bounds(const int* __restrict__ keys, const int* __restrict__ dT, int2* __restrict__ bounds) {
  const int T = *dT;
  const int w = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  const int p0 = w * 16;
  if (p0 >= T) return;
  const int n = min(16, T - p0);
  const int kf = keys[p0], kl = keys[p0 + n - 1];
  int head = p0, end = p0 + n;
  if (p0 > 0 && keys[p0 - 1] == kf) {                            // last position before p0 with another id, + 1
    for (int base = p0 - 32;; base -= 32) {
      const int q = base + lane;
      const unsigned m = __ballot_sync(0xffffffffu, q < 0 || keys[q] != kf);
      if (m) { head = base + (31 - __clz(m)) + 1; break; }
    }
  }
  if (p0 + n < T && keys[p0 + n] == kl) {                        // segment end (exclusive)
    for (int base = p0 + n;; base += 32) {
      const int q = base + lane;
      const unsigned m = __ballot_sync(0xffffffffu, q >= T || keys[q] != kl);
      if (m) { end = base + __ffs(m) - 1; break; }
    }
  }
  if (lane == 0) bounds[w] = make_int2(head, end);
}

// A run that is a PIECE of a longer segment (a hot item spanning several windows): rare, and kept out of line -- inlined
// into the 16-fold unrolled window loop it made the kernel 139 KB of code, most of which was only ever jumped over.
template <int NEL>
__device__ __noinline__ void scatter_piece(int p0, int w, int lane, int ku, int run_start, int u,
                                           bool cont_before, bool cont_after, const float (&acc)[NEL], float* __restrict__ gtable, int d,
                                           float scale, float* __restrict__ part, int* __restrict__ counter, const int2* __restrict__ bounds) {
          float* mine = part + ((long long)w * 2 + (cont_before ? 0 : 1)) * SPAD;
#pragma unroll
          for (int i = 0; i < NEL; ++i) mine[lane + 32 * i] = acc[i];
          // where the segment starts / ends was worked out by the plan (k_seg_bounds, off the critical path): a hot item of
          // 230 occurrences used to cost every one of its windows ~8 dependent key loads in each direction here
          int head = p0 + run_start, end = p0 + u + 1;
          if (cont_before) head = bounds[w].x;
          if (cont_after) end = bounds[w].y;
          const int w1 = head / SW, w2 = (end - 1) / SW;
          __threadfence();
          __syncwarp();
          int old = 0;
          if (lane == 0) old = atomicAdd(counter + w1, 1);
          old = __shfl_sync(0xffffffffu, old, 0);
          if (old == w2 - w1) {                                    // last piece to arrive: add the pieces in window order
            __threadfence();
            float tot[NEL];
#pragma unroll
            for (int i = 0; i < NEL; ++i) tot[i] = 0.f;
            for (int pw = w1; pw <= w2; pw += 8) {
              float t[8][NEL];
#pragma unroll
              for (int x = 0; x < 8; ++x) {
                const bool ok = pw + x <= w2;
                const float* src = part + ((long long)(ok ? pw + x : w1) * 2 + ((pw + x == w1) ? 1 : 0)) * SPAD;
#pragma unroll
                for (int i = 0; i < NEL; ++i) t[x][i] = ok ? __ldcg(src + lane + 32 * i) : 0.f;
              }
#pragma unroll
              for (int x = 0; x < 8; ++x)
#pragma unroll
                for (int i = 0; i < NEL; ++i) tot[i] += t[x][i];
            }
#pragma unroll
            for (int i = 0; i < NEL; ++i) { const int c = lane + 32 * i; if (c < d) atomicAdd(gtable + (long long)ku * d + c, scale * tot[i]); }
            if (lane == 0) counter[w1] = 0;                        // ready for the next step
          }
}

template <int NEL>
__global__ void __launch_bounds__(256) k_scatter_apply(const int* __restrict__ keys, const int* __restrict__ vals,
                                                       const int* __restrict__ dT, const float* __restrict__ gx, int d, float scale,
                                                       float* __restrict__ gtable, float* __restrict__ part, int* __restrict__ counter,
                                                       const int2* __restrict__ bounds) {
  const int T = *dT;
  const int w = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  const int p0 = w * SW;
  if (p0 >= T) return;
  const int n = min(SW, T - p0);
  const int key_l = (lane < n) ? keys[p0 + lane] : -1;
  const int val_l = (lane < n) ? vals[p0 + lane] : 0;
  const int key_prev = (p0 > 0) ? keys[p0 - 1] : -1;
  const int key_next = (p0 + n < T) ? keys[p0 + n] : -1;
  float v[SW][NEL];
#pragma unroll
  for (int u = 0; u < SW; ++u) {
    const int tu = __shfl_sync(0xffffffffu, val_l, u);
    const long long o = (long long)tu * d;
#pragma unroll
    for (int i = 0; i < NEL; ++i) { const int c = lane + 32 * i; v[u][i] = (u < n && c < d) ? gx[o + c] : 0.f; }
  }
  float acc[NEL];
#pragma unroll
  for (int i = 0; i < NEL; ++i) acc[i] = 0.f;
  int run_start = 0;
#pragma unroll
  for (int u = 0; u < SW; ++u) {
    const int ku = __shfl_sync(0xffffffffu, key_l, u);
    const int kn = __shfl_sync(0xffffffffu, key_l, (u + 1) & 31);
    if (u < n) {                                                   // warp-uniform
#pragma unroll
      for (int i = 0; i < NEL; ++i) acc[i] += v[u][i];
      const bool last_in_window = (u + 1 == n);
      if (last_in_window || kn != ku) {                            // the run [run_start, u] of item ku ends here
        const bool cont_after = last_in_window && key_next == ku;
        const bool cont_before = run_start == 0 && key_prev == ku;
        if (!cont_after && !cont_before) {
#pragma unroll
          for (int i = 0; i < NEL; ++i) { const int c = lane + 32 * i; if (c < d) atomicAdd(gtable + (long long)ku * d + c, scale * acc[i]); }
        } else {
          scatter_piece<NEL>(p0, w, lane, ku, run_start, u, cont_before, cont_after, acc, gtable, d, scale, part, counter, bounds);
        }
#pragma unroll
        for (int i = 0; i < NEL; ++i) acc[i] = 0.f;
        run_start = u + 1;
      }
    }
  }
}

static int key_bits(int v_tab) { int b = 1; while ((1LL << b) < v_tab) ++b; return b; }

}  // namespace ader
#include "encoder_fused.cuh"
namespace ader {

// ------------------------------------------------------------------------------------------
// group entry points
// ------------------------------------------------------------------------------------------
// packed token lists of a batch (row_len, row_off, tok_row, tok_id): three small launches
static void launch_pack_tokens(const int32_t* ids, int M, int L, int Tcap, const EncWs& w, cudaStream_t st) {
  k_row_len<<<cdiv((long long)M * 32, 256), 256, 0, st>>>(ids, M, L, w.row_len, w.flags);
  k_scan_rows<<<1, 1024, 0, st>>>(w.row_len, M, Tcap, w.row_off, w.flags);
  k_fill_tok<<<cdiv((long long)M * 32, 256), 256, 0, st>>>(ids, w.row_len, w.row_off, M, L, Tcap, w.tok_row, w.tok_id);
}
static int run_dense(cudaStream_t st, const float* A, const float* W, const float* bias, float* C,
                     int Tcap, const int* dT, int d, bool transW, int relu, const float* resid,
                     const float* relu_mask, int accumulate, float alpha,
                     float drop_p, uint64_t seed, uint32_t site) {
  GemmArgs g; gemm_defaults(g);
  g.A = A; g.a_rs = d; g.a_cs = 1;
  g.B = W; if (!transW) { g.b_rs = d; g.b_cs = 1; } else { g.b_rs = 1; g.b_cs = d; }
  g.C = C; g.c_rs = d; g.c_cs = 1;
  g.M = Tcap; g.N = d; g.K = d; g.dM = dT;
  g.bias = bias; g.resid = resid; g.resid_ld = d; g.relu_mask = relu_mask; g.mask_ld = d;
  g.relu = relu; g.accumulate = accumulate; g.alpha = alpha;
  g.drop_p = drop_p; g.drop_seed = seed; g.drop_site = site;
  return launch_gemm(g, st);
}

// dW partial[s] = act^T . grad over token split s, db partial[s] = colsum(grad)
static GemmArgs wgrad_args(const float* act, const float* grad, float* pW, float* pb,
                           long long split_stride, int Tcap, const int* dT, int d) {
  GemmArgs g; gemm_defaults(g);
  g.A = act; g.a_rs = 1; g.a_cs = d;       // A(m=c_in, k=t) = act[t*d + c_in]
  g.B = grad; g.b_rs = d; g.b_cs = 1;      // B(k=t, n=c_out)
  g.C = pW; g.c_rs = d; g.c_cs = 1;
  g.M = d; g.N = d; g.K = Tcap; g.dK = dT;
  g.splits = SPLITS; g.split_stride = split_stride; g.colsum = pb;
  return g;
}
static int run_wgrad(cudaStream_t st, const float* act, const float* grad, float* pW, float* pb,
                     long long split_stride, int Tcap, const int* dT, int d) {
  return launch_gemm(wgrad_args(act, grad, pW, pb, split_stride, Tcap, dT, d), st);
}

static int run_table_scatter(const AderModel* m, const Layout& l, const EncWs& w, const BwdWs& g, const float* gX,
                             int M, int Tcap, float* grad, cudaStream_t st);
// Tail shared by both encoder paths: split-K partials -> dense gradients, position table, item-table scatter.
// gX must already carry the embedding-dropout mask (site 0): the callers apply it once when they produce gX, so
// the position-table reduction and the scatter do not re-hash every element.
static int run_embedding_grads(const AderModel* m, const Layout& l, const EncWs& w, const BwdWs& g, const float* gX,
                               int M, int Tcap, float* grad, cudaStream_t st) {
  const float p = 0.f; const uint64_t seed = 0; const int* d_step = nullptr;
  const int d = m->d, L = m->maxlen;
  const int* dT = w.row_off + M;
  const long long PS = l.dense_count();
  // position table (ADER.py:41-52): per-row-chunk partials into the first L*d entries of the split slots
  launch_pos_grad(dim3(L, SPLITS), d, st, gX, w.row_len, w.row_off, M, L, d, p, seed, d_step, g.partial, PS);
  // dense parameter gradients (position table included): reduce the split partials in fixed order
  k_reduce_partials<<<cdiv(PS, 256), 256, 0, st>>>(g.partial, PS, SPLITS, 0, PS, grad + l.off_pos);
  return run_table_scatter(m, l, w, g, gX, M, Tcap, grad, st);
}

// ---- item-table scatter (modules.py:127-130) ------------------------------------------------------------------
static int sort_passes(const AderModel* m) { return (key_bits(m->v_tab) + 7) / 8; }
// plan: stable LSD radix sort of (item id, token); depends on the packed ids only
static int run_scatter_plan(const AderModel* m, const EncWs& w, const BwdWs& g, int M, int Tcap, cudaStream_t st) {
  const int* dT = w.row_off + M;
  const int ntiles = sort_tiles(Tcap);
  const int bits = key_bits(m->v_tab);
  const int n_count = cdiv(Tcap, SW);
  k_plan_zero<<<cdiv(n_count, 256), 256, 0, st>>>(g.scount, n_count);
  int cur = 0;
  const int* kin = w.tok_id; const int* vin = nullptr;
  int pass = 0;
  for (int shift = 0; shift < bits; shift += 8, ++pass) {
    k_sort_hist<<<ntiles, 256, 0, st>>>(kin, dT, shift, ntiles, g.hist);
    k_sort_scan<<<1, 1024, 0, st>>>(g.hist, 256 * ntiles);
    k_sort_scatter<<<ntiles, 256, 0, st>>>(kin, vin, dT, shift, ntiles, g.hist, pass == 0, g.keys[cur], g.vals[cur]);
    kin = g.keys[cur]; vin = g.vals[cur]; cur ^= 1;
  }
  k_seg_bounds<<<cdiv((long long)n_count * 32, 256), 256, 0, st>>>(kin, dT, g.sbounds);
  ADER_CHECK_LAUNCH("scatter plan");
  return 0;
}
static int run_scatter_apply(const AderModel* m, const Layout& l, const EncWs& w, const BwdWs& g, const float* gX,
                             int M, int Tcap, float* grad, cudaStream_t st) {
  const int d = m->d;
  const int* dT = w.row_off + M;
  const int fin = (sort_passes(m) - 1) & 1;
  const int grid = cdiv((long long)cdiv(Tcap, SW) * 32, 256);
  if (d <= 160)
    k_scatter_apply<5><<<grid, 256, 0, st>>>(g.keys[fin], g.vals[fin], dT, gX, d, sqrtf((float)d), grad + l.off_table, g.spart, g.scount, g.sbounds);
  else
    k_scatter_apply<LN_MAXE><<<grid, 256, 0, st>>>(g.keys[fin], g.vals[fin], dT, gX, d, sqrtf((float)d), grad + l.off_table, g.spart, g.scount, g.sbounds);
  ADER_CHECK_LAUNCH("scatter apply");
  return 0;
}
static int run_table_scatter(const AderModel* m, const Layout& l, const EncWs& w, const BwdWs& g, const float* gX,
                             int M, int Tcap, float* grad, cudaStream_t st) {
  if (int e = run_scatter_plan(m, w, g, M, Tcap, st)) return e;
  return run_scatter_apply(m, l, w, g, gX, M, Tcap, grad, st);
}

}  // namespace ader

using namespace ader;

extern "C" size_t ader_encoder_ws_bytes(const AderModel* m, int32_t M, int32_t Tcap) {
  if (check_model(m) || M <= 0 || Tcap <= 0) return 0;
  return carve_enc(m, M, Tcap, nullptr).bytes;
}
extern "C" size_t ader_encoder_bwd_ws_bytes(const AderModel* m, int32_t M, int32_t Tcap) {
  if (check_model(m) || M <= 0 || Tcap <= 0) return 0;
  return carve_bwd(m, M, Tcap, nullptr).bytes;
}
extern "C" int64_t ader_encoder_ws_slot(const AderModel* m, int32_t M, int32_t Tcap, int32_t slot, int32_t block) {
  if (check_model(m) || M <= 0 || Tcap <= 0 || block < 0 || block >= m->num_blocks) return -1;
  EncWs w = carve_enc(m, M, Tcap, (char*)0x1000);   // fake base to turn pointers into offsets
  const char* base = (const char*)0x1000;
  auto off = [&](const void* p) { return (int64_t)((const char*)p - base); };
  switch (slot) {
    case -1: return off(w.row_len);
    case -2: return off(w.row_off);
    case -3: return off(w.tok_row);
    case -4: return off(w.flags);
    case 8: return off(w.xfinal);
    case 9: return off(w.probs[block]);
    default:
      if (slot >= 0 && slot < NSLOT) return off(w.slot[block][slot]);
  }
  return -1;
}

extern "C" int32_t ader_encoder_fwd(const AderModel* m, const float* theta, const int32_t* ids, int32_t M,
                                    int32_t Tcap, void* ws, float* rep, float dropout_rate, uint64_t seed,
                                    void* stream) {
  if (int e = check_model(m)) return e;
  if (int e = path_check(m, ADER_PATH_ENCODER_FWD)) return e;
  ADER_CHECK_ARG(theta && ids && ws && rep, "encoder_fwd: NULL pointer");
  ADER_CHECK_ARG(M > 0 && Tcap > 0 && (long long)Tcap <= (long long)M * m->maxlen, "encoder_fwd: bad M/Tcap (%d, %d)", M, Tcap);
  ADER_CHECK_ARG(dropout_rate >= 0.f && dropout_rate < 1.f, "encoder_fwd: dropout_rate out of range");
  cudaStream_t st = (cudaStream_t)stream;
  if (int e = kernel_ready<k_attn_fwd>((int)ATTN_FWD_SMEM_MAX, "k_attn_fwd")) return e;
  const Layout l = make_layout(m);
  const int d = m->d, L = m->maxlen;
  EncWs w = carve_enc(m, M, Tcap, (char*)ws);
  const int* dT = w.row_off + M;

  launch_pack_tokens(ids, M, L, Tcap, w, st);
  k_embed<<<cdiv((long long)Tcap * d, 256), 256, 0, st>>>(theta + l.off_table, theta + l.off_pos, w.tok_row, w.tok_id,
                                                           w.row_len, w.row_off, dT, d, L, sqrtf((float)d),
                                                           dropout_rate, seed, w.slot[0][0]);
  ADER_CHECK_LAUNCH("encoder_fwd/pack+embed");

  const size_t attn_smem = attn_fwd_smem(d, L);
  const int ln_grid = cdiv((long long)Tcap * 32, 256);

  for (int b = 0; b < m->num_blocks; ++b) {
    const float* P = theta + l.block(b);
    float* X = w.slot[b][0]; float* Q1 = w.slot[b][1]; float* Qp = w.slot[b][2]; float* Kp = w.slot[b][3];
    float* Vp = w.slot[b][4]; float* Y = w.slot[b][5]; float* Z = w.slot[b][6]; float* H = w.slot[b][7];
    float* Xn = (b + 1 < m->num_blocks) ? w.slot[b + 1][0] : w.xfinal;
    k_ln_fwd<<<ln_grid, 256, 0, st>>>(X, Q1, w.mean1[b], w.rstd1[b], P + l.ln1b, P + l.ln1g, dT, d);
    if (int e = run_dense(st, Q1, P + l.wq, P + l.bq, Qp, Tcap, dT, d, false, 0, nullptr, nullptr, 0, 1.f, 0.f, 0, 0)) return e;
    if (int e = run_dense(st, X, P + l.wk, P + l.bk, Kp, Tcap, dT, d, false, 0, nullptr, nullptr, 0, 1.f, 0.f, 0, 0)) return e;
    if (int e = run_dense(st, X, P + l.wv, P + l.bv, Vp, Tcap, dT, d, false, 0, nullptr, nullptr, 0, 1.f, 0.f, 0, 0)) return e;
    k_attn_fwd<<<M, ATT_THREADS, attn_smem, st>>>(Qp, Kp, Vp, Q1, w.row_len, w.row_off, d, m->num_heads, L, Tcap,
                                          dropout_rate, seed, 1u + 3u * b, w.probs[b], Y);
    k_ln_fwd<<<ln_grid, 256, 0, st>>>(Y, Z, w.mean2[b], w.rstd2[b], P + l.ln2b, P + l.ln2g, dT, d);
    if (int e = run_dense(st, Z, P + l.w1, P + l.b1, H, Tcap, dT, d, false, 1, nullptr, nullptr, 0, 1.f,
                          dropout_rate, seed, 2u + 3u * b)) return e;
    if (int e = run_dense(st, H, P + l.w2, P + l.b2, Xn, Tcap, dT, d, false, 0, Z, nullptr, 0, 1.f,
                          dropout_rate, seed, 3u + 3u * b)) return e;
    ADER_CHECK_LAUNCH("encoder_fwd/block");
  }
  k_ln_last_fwd<<<cdiv((long long)M * 32, 256), 256, 0, st>>>(w.xfinal, w.row_len, w.row_off, M, rep, w.meanf, w.rstdf,
                                                               theta + l.off_lnf, theta + l.off_lnf + d, d);
  ADER_CHECK_LAUNCH("encoder_fwd/final_ln");
  return 0;
}

// ---- batched EWC Fisher diagonal (EWC.py:126-164) ---------------------------------------------------------------------
// The reference runs one forward + backward PER SAMPLE and squares the dense 26 MB gradient each time.  Here ONE batched
// exact forward / data-gradient backward serves all S samples, and wherever the ordinary backward would SUM a weight
// gradient over the tokens of the batch, the hook below sums over the tokens of ONE sample, squares (fp32, np.square on
// float32) and accumulates over samples in fp64 (F_accum is float64):
//   linear layers   g_s[i][j] = sum_{t in s} x[t][i] dy[t][j]          (k_fisher_linear, + bias = sum_t dy)
//   LayerNorm       dbeta_s = sum_t dout[t], dgamma_s = sum_t dout[t] xhat[t]   (k_fisher_ln)
//   position table  row p receives dx0 of the one token of s at p     (k_fisher_pos)
//   item table      g_s[v] = dl_s[v] rep_s  (+ sqrt(d) sum of dx0 over the tokens of s with id v):
//                   sum_s (dl_s[v] rep_s[f])^2 for all v by k_fisher_table over row chunks of dl = softmax - onehot,
//                   the few (s, v) with an input occurrence corrected by k_fisher_scatter_fix.
struct FisherHook {
  double* acc;                 // flat fp64, theta layout
  const int* tok_row;          // sample of each packed token
  const float* rep;            // [S, d]
  const float* lse;            // [S] log-sum-exp of the sample's logits
  const int* pos;              // [S] labels
  const float* theta;
  int S, V;
};

struct FLMat { const float* X; const float* G; double* accW; double* accb; };
struct FLArgs { FLMat p[3]; const int* tok_row; const int* dT; int d; };
constexpr int FL_TT = 32, FL_IB = 8;
// grid (ceil(d / 8), n_mat), 160 threads: thread j owns entries (i0 .. i0+7, j) of W (in-major [i][j]) -- exclusive, no atomics
__global__ void __launch_bounds__(160) k_fisher_linear(FLArgs a) {
  __shared__ float sG[FL_TT][160];
  __shared__ float sX[FL_TT][FL_IB];
  __shared__ int sRow[FL_TT];
  const FLMat P = a.p[blockIdx.y];
  const int d = a.d, i0 = blockIdx.x * FL_IB, j = threadIdx.x, T = *a.dT;
  double acc[FL_IB], accb = 0.0;
  float gs[FL_IB], gb = 0.f;
#pragma unroll
  for (int ii = 0; ii < FL_IB; ++ii) { acc[ii] = 0.0; gs[ii] = 0.f; }
  int cur = -1;
  for (int t0 = 0; t0 < T; t0 += FL_TT) {
    const int nt = min(FL_TT, T - t0);
    for (int e = threadIdx.x; e < nt * d; e += 160) sG[e / d][e % d] = P.G[(long long)t0 * d + e];
    for (int e = threadIdx.x; e < nt * FL_IB; e += 160) {
      const int tt = e / FL_IB, ii = e % FL_IB;
      sX[tt][ii] = (i0 + ii < d) ? P.X[(long long)(t0 + tt) * d + i0 + ii] : 0.f;
    }
    if (threadIdx.x < nt) sRow[threadIdx.x] = a.tok_row[t0 + threadIdx.x];
    __syncthreads();
    if (j < d) {
      for (int tt = 0; tt < nt; ++tt) {
        const int r = sRow[tt];
        if (r != cur) {
          if (cur >= 0) {
#pragma unroll
            for (int ii = 0; ii < FL_IB; ++ii) { acc[ii] += (double)__fmul_rn(gs[ii], gs[ii]); gs[ii] = 0.f; }
            accb += (double)__fmul_rn(gb, gb); gb = 0.f;
          }
          cur = r;
        }
        const float g = sG[tt][j];
#pragma unroll
        for (int ii = 0; ii < FL_IB; ++ii) gs[ii] = fmaf(sX[tt][ii], g, gs[ii]);
        gb += g;
      }
    }
    __syncthreads();
  }
  if (j < d && cur >= 0) {
#pragma unroll
    for (int ii = 0; ii < FL_IB; ++ii) acc[ii] += (double)__fmul_rn(gs[ii], gs[ii]);
    accb += (double)__fmul_rn(gb, gb);
  }
  if (j < d) {
#pragma unroll
    for (int ii = 0; ii < FL_IB; ++ii) if (i0 + ii < d) P.accW[(long long)(i0 + ii) * d + j] += acc[ii];
    if (blockIdx.x == 0) P.accb[j] += accb;
  }
}

// one CTA, 160 threads (feature c): per-sample LayerNorm parameter gradients.  rows == nullptr: token mode (dout, x, mean,
// rstd per token); else "last token" mode of the final LayerNorm (dout, mean, rstd per row, x at the row's last token).
__global__ void __launch_bounds__(160) k_fisher_ln(const float* __restrict__ dout, const float* __restrict__ x,
                                                   const float* __restrict__ mean, const float* __restrict__ rstd,
                                                   const int* __restrict__ tok_row, const int* __restrict__ dT, int M,
                                                   const int* __restrict__ row_len, const int* __restrict__ row_off, int d,
                                                   double* __restrict__ acc_beta, double* __restrict__ acc_gamma) {
  const int c = threadIdx.x;
  if (c >= d) return;
  double ab = 0.0, ag = 0.0;
  if (row_off) {
    for (int r = 0; r < M; ++r) {
      if (row_len[r] == 0) continue;
      const float g = dout[(long long)r * d + c];
      const float xh = (x[(long long)(row_off[r + 1] - 1) * d + c] - mean[r]) * rstd[r];
      const float gg = g * xh;
      ab += (double)__fmul_rn(g, g); ag += (double)__fmul_rn(gg, gg);
    }
  } else {
    const int T = *dT;
    float sb = 0.f, sg = 0.f; int cur = -1;
    for (int t0 = 0; t0 < T; t0 += 8) {                      // eight tokens' loads in flight, then the ordered accumulation
      float g8[8], x8[8], mu8[8], rs8[8]; int r8[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int t = min(t0 + k, T - 1);
        g8[k] = dout[(long long)t * d + c]; x8[k] = x[(long long)t * d + c]; mu8[k] = mean[t]; rs8[k] = rstd[t]; r8[k] = tok_row[t];
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        if (t0 + k >= T) break;
        if (r8[k] != cur) {
          if (cur >= 0) { ab += (double)__fmul_rn(sb, sb); ag += (double)__fmul_rn(sg, sg); sb = 0.f; sg = 0.f; }
          cur = r8[k];
        }
        sb += g8[k]; sg += g8[k] * ((x8[k] - mu8[k]) * rs8[k]);
      }
    }
    if (cur >= 0) { ab += (double)__fmul_rn(sb, sb); ag += (double)__fmul_rn(sg, sg); }
  }
  acc_beta[c] += ab; acc_gamma[c] += ag;
}

// grid L (position p), 160 threads: acc_pos[p][c] += sum over samples holding position p of dx0^2
__global__ void __launch_bounds__(160) k_fisher_pos(const float* __restrict__ gx, const int* __restrict__ row_len,
                                                    const int* __restrict__ row_off, int M, int L, int d, double* __restrict__ acc_pos) {
  const int p = blockIdx.x, c = threadIdx.x;
  if (c >= d) return;
  double a = 0.0;
  for (int r0 = 0; r0 < M; r0 += 8) {
    float v8[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int r = min(r0 + k, M - 1);
      const int n = row_len[r];
      v8[k] = (r0 + k < M && n >= L - p) ? gx[(long long)(row_off[r] + p - (L - n)) * d + c] : 0.f;
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) a += (double)__fmul_rn(v8[k], v8[k]);
  }
  acc_pos[(long long)p * d + c] += a;
}

// dl = softmax(logits) - onehot in place over a chunk of rows (CTA per row), lse out
__global__ void __launch_bounds__(256) k_fisher_softmax(float* __restrict__ lg, long long ld, int V, const int* __restrict__ pos,
                                                        float* __restrict__ lse) {
  __shared__ float sh[8];
  float* s = lg + (long long)blockIdx.x * ld;
  float mx = -INFINITY;
  for (int j = threadIdx.x; j < V; j += 256) mx = fmaxf(mx, s[j]);
#pragma unroll
  for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = mx;
  __syncthreads();
  mx = sh[0];
  for (int w = 1; w < 8; ++w) mx = fmaxf(mx, sh[w]);
  __syncthreads();
  float sum = 0.f;
  for (int j = threadIdx.x; j < V; j += 256) sum += expf(s[j] - mx);
#pragma unroll
  for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = sum;
  __syncthreads();
  float tot = 0.f;
  for (int w = 0; w < 8; ++w) tot += sh[w];
  const float l = mx + logf(tot);
  const int g = pos[blockIdx.x] - 1;
  for (int j = threadIdx.x; j < V; j += 256) s[j] = expf(s[j] - l) - (j == g ? 1.f : 0.f);
  if (threadIdx.x == 0) lse[blockIdx.x] = l;
}

// acc_tab[v][f] += sum over the chunk's samples of (dl[s][v] * rep[s][f])^2.  CTA = 64 items x all features, 256 threads:
// thread (v = t / 4, fq = t % 4) owns features fq, fq + 4, ...; samples staged 16 at a time.
constexpr int FT_V = 64, FT_S = 16, FT_F = 40;
__global__ void __launch_bounds__(256) k_fisher_table(const float* __restrict__ dl, long long ld, const float* __restrict__ rep,
                                                      int n_rows, int V, int d, double* __restrict__ acc_tab) {
  __shared__ float sD[FT_S][FT_V];
  __shared__ float sR[FT_S][160];
  const int v0 = blockIdx.x * FT_V, vl = threadIdx.x >> 2, fq = threadIdx.x & 3;
  double acc[FT_F];
#pragma unroll
  for (int k = 0; k < FT_F; ++k) acc[k] = 0.0;
  for (int s0 = 0; s0 < n_rows; s0 += FT_S) {
    const int ns = min(FT_S, n_rows - s0);
    for (int e = threadIdx.x; e < ns * FT_V; e += 256) {
      const int ss = e / FT_V, vv = e % FT_V;
      sD[ss][vv] = (v0 + vv < V) ? dl[(long long)(s0 + ss) * ld + v0 + vv] : 0.f;
    }
    for (int e = threadIdx.x; e < ns * d; e += 256) sR[e / d][e % d] = rep[(long long)s0 * d + e];
    __syncthreads();
    for (int ss = 0; ss < ns; ++ss) {
      const float x = sD[ss][vl];
#pragma unroll
      for (int k = 0; k < FT_F; ++k) {
        const int f = fq + 4 * k;
        if (f < d) { const float g = __fmul_rn(x, sR[ss][f]); acc[k] += (double)__fmul_rn(g, g); }
      }
    }
    __syncthreads();
  }
  if (v0 + vl < V) {
#pragma unroll
    for (int k = 0; k < FT_F; ++k) { const int f = fq + 4 * k; if (f < d) acc_tab[(long long)(v0 + vl) * d + f] += acc[k]; }
  }
}

// CTA per sample, 160 threads: rows of the item table that also receive the sample's input-lookup scatter get
// (dl rep + sc)^2 instead of (dl rep)^2.  Different samples may share an item: fp64 atomics (order changes the sum by ~1e-16).
__global__ void __launch_bounds__(160) k_fisher_scatter_fix(FisherHook h, const float* __restrict__ gx0, const int* __restrict__ tok_id,
                                                            const int* __restrict__ row_len, const int* __restrict__ row_off, int d,
                                                            float sqrt_d, double* __restrict__ acc_tab) {
  __shared__ float red[8];
  const int r = blockIdx.x, c = threadIdx.x;
  const int n = row_len[r], off = row_off[r];
  if (n == 0) return;
  const float l = h.lse[r];
  const int g = h.pos[r];
  const float rp = c < d ? h.rep[(long long)r * d + c] : 0.f;
  for (int t = 0; t < n; ++t) {
    const int id = tok_id[off + t];
    bool first = true;
    for (int u = 0; u < t; ++u) if (tok_id[off + u] == id) { first = false; break; }
    if (!first) continue;                                     // uniform over the CTA
    float sc = 0.f;
    for (int u = t; u < n; ++u) if (tok_id[off + u] == id && c < d) sc += gx0[(long long)(off + u) * d + c];
    sc *= sqrt_d;
    float part = c < d ? rp * h.theta[(long long)id * d + c] : 0.f;      // logit of item `id` for this sample
#pragma unroll
    for (int o = 16; o; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    __syncthreads();
    if ((c & 31) == 0) red[c >> 5] = part;
    __syncthreads();
    float logit = 0.f;
    for (int w = 0; w < 5; ++w) logit += red[w];
    const float dlv = expf(logit - l) - (id == g ? 1.f : 0.f);
    if (c < d && id <= h.V) {
      const float a0 = __fmul_rn(dlv, rp);
      const float a1 = __fadd_rn(a0, sc);
      atomicAdd(acc_tab + (long long)id * d + c, (double)__fmul_rn(a1, a1) - (double)__fmul_rn(a0, a0));
    }
  }
}

static int fisher_linear(const FisherHook& fh, cudaStream_t st, int n, const float* const* X, const float* const* G,
                         const long long* offW, const long long* offb, const int* dT, int d) {
  FLArgs a; a.tok_row = fh.tok_row; a.dT = dT; a.d = d;
  for (int k = 0; k < n; ++k) a.p[k] = {X[k], G[k], fh.acc + offW[k], fh.acc + offb[k]};
  k_fisher_linear<<<dim3(cdiv(d, FL_IB), n), 160, 0, st>>>(a);
  return 0;
}

static int enc_bwd_exact(const AderModel* m, const float* theta, const int32_t* ids, int32_t M, int32_t Tcap, const void* ws,
                         void* bwd_ws, const float* d_rep, float* grad, float dropout_rate, uint64_t seed, cudaStream_t st,
                         const FisherHook* fh);

extern "C" int32_t ader_encoder_bwd(const AderModel* m, const float* theta, const int32_t* ids, int32_t M,
                                    int32_t Tcap, const void* ws, void* bwd_ws, const float* d_rep, float* grad,
                                    float dropout_rate, uint64_t seed, void* stream) {
  if (int e = check_model(m)) return e;
  if (int e = path_check(m, ADER_PATH_ENCODER_BWD)) return e;
  ADER_CHECK_ARG(theta && ids && ws && bwd_ws && d_rep && grad, "encoder_bwd: NULL pointer");
  ADER_CHECK_ARG(M > 0 && Tcap > 0, "encoder_bwd: bad M/Tcap");
  ADER_CHECK_ARG(dropout_rate >= 0.f && dropout_rate < 1.f, "encoder_bwd: dropout_rate out of range");
  return enc_bwd_exact(m, theta, ids, M, Tcap, ws, bwd_ws, d_rep, grad, dropout_rate, seed, (cudaStream_t)stream, nullptr);
}

static int enc_bwd_exact(const AderModel* m, const float* theta, const int32_t* ids, int32_t M, int32_t Tcap, const void* ws,
                         void* bwd_ws, const float* d_rep, float* grad, float dropout_rate, uint64_t seed, cudaStream_t st,
                         const FisherHook* fh) {
  if (int e = kernel_ready<k_attn_bwd>((int)ATTN_BWD_SMEM_MAX, "k_attn_bwd")) return e;
  const Layout l = make_layout(m);
  const int d = m->d, L = m->maxlen;
  const float p = dropout_rate;
  EncWs w = carve_enc(m, M, Tcap, (char*)ws);
  BwdWs g = carve_bwd(m, M, Tcap, (char*)bwd_ws);
  const int* dT = w.row_off + M;
  const long long PS = l.dense_count();                 // split stride of the partial workspace
  auto part = [&](long long param_off) { return g.partial + (param_off - l.off_pos); };
  float *gX = g.g[0], *gXin = g.g[1], *gO = g.g[2], *gH = g.g[3], *gZ = g.g[4], *gY = g.g[5],
        *gQ = g.g[6], *gK = g.g[7], *gV = g.g[8], *gQ1 = g.g[9];
  const int ln_grid = cdiv((long long)Tcap * 32, 256);
  const int el_grid = cdiv((long long)Tcap * d, 256);

  const size_t attn_smem = attn_bwd_smem(d, L);      // within ATTN_BWD_SMEM_MAX: the entries ran path_check

  // final LayerNorm (ADER.py:82): only the last token of each row carries gradient
  k_lnf_bwd<<<ln_grid, 256, 0, st>>>(d_rep, w.xfinal, w.meanf, w.rstdf, theta + l.off_lnf + d, w.tok_row, w.row_off, gX, dT, d);
  if (fh) k_fisher_ln<<<1, 160, 0, st>>>(d_rep, w.xfinal, w.meanf, w.rstdf, w.tok_row, dT, M, w.row_len, w.row_off, d,
                                         fh->acc + l.off_lnf, fh->acc + l.off_lnf + d);
  else launch_ln_param_grad(dim3(SPLITS), d, st, d_rep, w.xfinal, w.meanf, w.rstdf, dT, M, w.row_len, w.row_off, d,
                                                 part(l.off_lnf), part(l.off_lnf + d), PS);
  ADER_CHECK_LAUNCH("encoder_bwd/final_ln");

  for (int b = m->num_blocks - 1; b >= 0; --b) {
    const long long bo = l.block(b);
    const float* P = theta + bo;
    const float* X = w.slot[b][0]; const float* Q1 = w.slot[b][1]; const float* Qp = w.slot[b][2];
    const float* Kp = w.slot[b][3]; const float* Vp = w.slot[b][4]; const float* Y = w.slot[b][5];
    const float* Z = w.slot[b][6]; const float* H = w.slot[b][7];
    const float* gOut = gX;
    if (p > 0.f) {   // x_out = drop(h.W2 + b2) + z  (modules.py:259-266)
      k_apply_drop<<<el_grid, 256, 0, st>>>(gX, gO, dT, d, p, seed, 3u + 3u * b);
      gOut = gO;
    }
    if (fh) { const float* Xs[1] = {H}; const float* Gs[1] = {gOut}; const long long ow[1] = {bo + l.w2}, ob[1] = {bo + l.b2};
              fisher_linear(*fh, st, 1, Xs, Gs, ow, ob, dT, d); }
    else if (int e = run_wgrad(st, H, gOut, part(bo + l.w2), part(bo + l.b2), PS, Tcap, dT, d)) return e;
    // gH = (gOut . W2^T) * [h > 0] * 1/(1-p)   (h is stored post-dropout)
    if (int e = run_dense(st, gOut, P + l.w2, nullptr, gH, Tcap, dT, d, true, 0, nullptr, H, 0,
                          p > 0.f ? 1.f / (1.f - p) : 1.f, 0.f, 0, 0)) return e;
    if (fh) { const float* Xs[1] = {Z}; const float* Gs[1] = {gH}; const long long ow[1] = {bo + l.w1}, ob[1] = {bo + l.b1};
              fisher_linear(*fh, st, 1, Xs, Gs, ow, ob, dT, d); }
    else if (int e = run_wgrad(st, Z, gH, part(bo + l.w1), part(bo + l.b1), PS, Tcap, dT, d)) return e;
    // gZ = gH . W1^T + gX   (residual z -> x_out)
    if (int e = run_dense(st, gH, P + l.w1, nullptr, gZ, Tcap, dT, d, true, 0, gX, nullptr, 0, 1.f, 0.f, 0, 0)) return e;
    k_ln_bwd<<<ln_grid, 256, 0, st>>>(gZ, Y, w.mean2[b], w.rstd2[b], P + l.ln2g, gY, dT, d, 0);
    if (fh) k_fisher_ln<<<1, 160, 0, st>>>(gZ, Y, w.mean2[b], w.rstd2[b], w.tok_row, dT, 0, nullptr, nullptr, d,
                                           fh->acc + bo + l.ln2b, fh->acc + bo + l.ln2g);
    else launch_ln_param_grad(dim3(SPLITS), d, st, gZ, Y, w.mean2[b], w.rstd2[b], dT, 0, nullptr, nullptr, d,
                                                   part(bo + l.ln2b), part(bo + l.ln2g), PS);
    k_attn_bwd<<<M, ATT_THREADS, attn_smem, st>>>(Qp, Kp, Vp, w.probs[b], gY, w.row_len, w.row_off, d, m->num_heads, L, Tcap,
                                          p, seed, 1u + 3u * b, gQ, gK, gV);
    ADER_CHECK_LAUNCH("encoder_bwd/attn");
    if (fh) {
      const float* Xs[3] = {Q1, X, X}; const float* Gs[3] = {gQ, gK, gV};
      const long long ow[3] = {bo + l.wq, bo + l.wk, bo + l.wv}, ob[3] = {bo + l.bq, bo + l.bk, bo + l.bv};
      fisher_linear(*fh, st, 3, Xs, Gs, ow, ob, dT, d);
    } else {
      if (int e = run_wgrad(st, Q1, gQ, part(bo + l.wq), part(bo + l.bq), PS, Tcap, dT, d)) return e;
      if (int e = run_wgrad(st, X, gK, part(bo + l.wk), part(bo + l.bk), PS, Tcap, dT, d)) return e;
      if (int e = run_wgrad(st, X, gV, part(bo + l.wv), part(bo + l.bv), PS, Tcap, dT, d)) return e;
    }
    // gQ1 = gQ . Wq^T + gY   (y = attn + q)
    if (int e = run_dense(st, gQ, P + l.wq, nullptr, gQ1, Tcap, dT, d, true, 0, gY, nullptr, 0, 1.f, 0.f, 0, 0)) return e;
    if (int e = run_dense(st, gK, P + l.wk, nullptr, gXin, Tcap, dT, d, true, 0, nullptr, nullptr, 0, 1.f, 0.f, 0, 0)) return e;
    if (int e = run_dense(st, gV, P + l.wv, nullptr, gXin, Tcap, dT, d, true, 0, nullptr, nullptr, 1, 1.f, 0.f, 0, 0)) return e;
    k_ln_bwd<<<ln_grid, 256, 0, st>>>(gQ1, X, w.mean1[b], w.rstd1[b], P + l.ln1g, gXin, dT, d, 1);
    if (fh) k_fisher_ln<<<1, 160, 0, st>>>(gQ1, X, w.mean1[b], w.rstd1[b], w.tok_row, dT, 0, nullptr, nullptr, d,
                                           fh->acc + bo + l.ln1b, fh->acc + bo + l.ln1g);
    else launch_ln_param_grad(dim3(SPLITS), d, st, gQ1, X, w.mean1[b], w.rstd1[b], dT, 0, nullptr, nullptr, d,
                                                   part(bo + l.ln1b), part(bo + l.ln1g), PS);
    ADER_CHECK_LAUNCH("encoder_bwd/block");
    float* t = gX; gX = gXin; gXin = t;
  }

  if (p > 0.f) k_apply_drop<<<el_grid, 256, 0, st>>>(gX, gX, dT, d, p, seed, 0u);   // x0 = drop(emb) (ADER.py:55)
  if (fh) {
    k_fisher_pos<<<L, 160, 0, st>>>(gX, w.row_len, w.row_off, M, L, d, fh->acc + l.off_pos);
    k_fisher_scatter_fix<<<M, 160, 0, st>>>(*fh, gX, w.tok_id, w.row_len, w.row_off, d, sqrtf((float)d), fh->acc + l.off_table);
  } else if (int e = run_embedding_grads(m, l, w, g, gX, M, Tcap, grad, st)) return e;
  ADER_CHECK_LAUNCH("encoder_bwd/embedding");
  return 0;
}

// workspace of ader_fisher_batched: rep [S, d], d_rep [S, d], lse [S], a chunk of logits / dl [FISHER_CHUNK, ld(V)]
constexpr int FISHER_CHUNK = 256;
static long long fisher_ld(int V) { return ((long long)V + 3) / 4 * 4; }
extern "C" size_t ader_fisher_batched_ws_bytes(const AderModel* m, int32_t S, int32_t V) {
  if (check_model(m) || S <= 0 || V <= 0 || path_check(m, ADER_PATH_FISHER_BATCHED)) return 0;
  return 2 * align_up(sizeof(float) * (size_t)S * m->d) + align_up(sizeof(float) * (size_t)S) +
         align_up(sizeof(float) * (size_t)FISHER_CHUNK * fisher_ld(V));
}

extern "C" int32_t ader_fisher_batched(const AderModel* m, const float* theta, const int32_t* ids, const int32_t* pos, int32_t S,
                                       int32_t Tcap, int32_t V, void* enc_ws, void* bwd_ws, void* ws, double* acc, void* stream) {
  if (int e = check_model(m)) return e;
  if (int e = path_check(m, ADER_PATH_FISHER_BATCHED)) return e;
  ADER_CHECK_ARG(theta && ids && pos && enc_ws && bwd_ws && ws && acc, "fisher_batched: NULL pointer");
  ADER_CHECK_ARG(S > 0 && Tcap > 0 && V >= 1 && V < m->v_tab, "fisher_batched: bad sizes");
  cudaStream_t st = (cudaStream_t)stream;
  const int d = m->d;
  const Layout l = make_layout(m);
  char* base = (char*)ws; size_t o = 0;
  auto take = [&](size_t n) { char* p = base + o; o += align_up(n); return p; };
  float* rep = (float*)take(sizeof(float) * (size_t)S * d);
  float* d_rep = (float*)take(sizeof(float) * (size_t)S * d);
  float* lse = (float*)take(sizeof(float) * (size_t)S);
  float* lg = (float*)take(sizeof(float) * (size_t)FISHER_CHUNK * fisher_ld(V));
  const long long ld = fisher_ld(V);
  if (int e = ader_encoder_fwd(m, theta, ids, S, Tcap, enc_ws, rep, 0.f, 0, stream)) return e;      // eval mode (EWC.py:151-152)
  for (int r0 = 0; r0 < S; r0 += FISHER_CHUNK) {
    const int nr = (S - r0 < FISHER_CHUNK) ? S - r0 : FISHER_CHUNK;
    if (int e = ader_logits(m, theta, rep + (size_t)r0 * d, nr, V, lg, ld, stream)) return e;
    k_fisher_softmax<<<nr, 256, 0, st>>>(lg, ld, V, pos + r0, lse + r0);
    GemmArgs g; gemm_defaults(g);                            // d_rep = dl . E[1..V]   (K = V)
    g.A = lg; g.a_rs = ld; g.a_cs = 1;
    g.B = theta + d; g.b_rs = d; g.b_cs = 1;
    g.C = d_rep + (size_t)r0 * d; g.c_rs = d; g.c_cs = 1;
    g.M = nr; g.N = d; g.K = V;
    if (int e = launch_gemm(g, st)) return e;
    k_fisher_table<<<cdiv(V, FT_V), 256, 0, st>>>(lg, ld, rep + (size_t)r0 * d, nr, V, d, acc + l.off_table + d);
    ADER_CHECK_LAUNCH("fisher_batched/table");
  }
  EncWs w = carve_enc(m, S, Tcap, (char*)enc_ws);
  FisherHook fh;
  fh.acc = acc; fh.tok_row = w.tok_row; fh.rep = rep; fh.lse = lse; fh.pos = pos; fh.theta = theta; fh.S = S; fh.V = V;
  return enc_bwd_exact(m, theta, ids, S, Tcap, enc_ws, bwd_ws, d_rep, nullptr, 0.f, 0, st, &fh);
}

// ------------------------------------------------------------------------------------------
// fused tensor-core path (encoder_fused.cuh): same contract, same workspace slots
// ------------------------------------------------------------------------------------------
namespace ader {
static_assert(PATH_TC_MAX_D == fz::KP, "the fused encoder pads features to KP columns");
// SMs of the current device (a cached query of the runtime): the tile kernels launch at most one CTA per SM
static int sm_count() {
  int dev = 0, n = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
  return n;
}
static int fused_ready() {
  if (int e = kernel_ready<fz::k_qkv_fwd>((int)fz::QKV_FWD_SMEM, "k_qkv_fwd")) return e;
  if (int e = kernel_ready<fz::k_ffn_fwd>((int)fz::FFN_FWD_SMEM, "k_ffn_fwd")) return e;
  if (int e = kernel_ready<fz::k_ffn_bwd>((int)fz::FFN_BWD_SMEM, "k_ffn_bwd")) return e;
  if (int e = kernel_ready<fz::k_qkv_bwd>((int)fz::QKV_BWD_SMEM, "k_qkv_bwd")) return e;
  if (int e = kernel_ready<fz::k_wgrad2>((int)fz::WGRAD2_SMEM, "k_wgrad2")) return e;
  if (int e = kernel_ready<fz::k_attn_ln_fwd>(2 * fz::att_rows_cap(64) * fz::KP * 4, "k_attn_ln_fwd")) return e;
  return kernel_ready<fz::k_attn_bwd_s1>(fz::att_bwd_smem(64, fz::KP), "k_attn_bwd_s1");
}
static const fz::op_t* shadow_of(const EncWs& w, int b, int which, int orient) {
  return (const fz::op_t*)w.wshadow + (size_t)((b * 5 + which) * 2 + orient) * (fz::KP * fz::LDS);
}
}  // namespace ader

#ifdef ADER_TC_TIMELINE
extern "C" int32_t ader_debug_fz_timeline(long long* out) {
  cudaDeviceSynchronize();
  return (int32_t)cudaMemcpyFromSymbol(out, fz::g_fz_tl, sizeof(fz::g_fz_tl));
}
#endif

extern "C" int32_t ader_encoder_fwd_tc(const AderModel* m, const float* theta, const int32_t* ids, int32_t M,
                                       int32_t Tcap, void* ws, float* rep, float dropout_rate, uint64_t seed,
                                       const int32_t* d_step, void* stream) {
  Fork f = Fork::serial((cudaStream_t)stream);
  return enc_fwd_tc_run(m, theta, ids, M, Tcap, ws, rep, dropout_rate, seed, d_step, f);
}

int ader::enc_fwd_tc_run(const AderModel* m, const float* theta, const int32_t* ids, int M, int Tcap, void* ws, float* rep,
                         float dropout_rate, uint64_t seed, const int32_t* d_step, Fork& f) {
  if (int e = check_model(m)) return e;
  if (int e = path_check(m, ADER_PATH_ENCODER_TC)) return e;
  ADER_CHECK_ARG(theta && ids && ws && rep, "encoder_fwd_tc: NULL pointer");
  ADER_CHECK_ARG(M > 0 && Tcap > 0 && (long long)Tcap <= (long long)M * m->maxlen, "encoder_fwd_tc: bad M/Tcap (%d, %d)", M, Tcap);
  ADER_CHECK_ARG(dropout_rate >= 0.f && dropout_rate < 1.f, "encoder_fwd_tc: dropout_rate out of range");
  if (int e = fused_ready()) return e;
  cudaStream_t st = f.main;
  const Layout l = make_layout(m);
  const int d = m->d, L = m->maxlen;
  EncWs w = carve_enc(m, M, Tcap, (char*)ws);
  const int* dT = w.row_off + M;

  // weight shadows depend on theta only: off the packing chain (joined before the first tile kernel)
  f.edge(st, f.a);
  fz::k_pack_weights<<<dim3(m->num_blocks * 5, fz::KP / fz::PACK_BAND), 256, 0, f.a>>>(theta, l, (fz::op_t*)w.wshadow);
  launch_pack_tokens(ids, M, L, Tcap, w, st);
  ADER_CHECK_LAUNCH("encoder_fwd_tc/pack");
  if (f.parallel()) { f.tok_ready = f.take(); cudaEventRecord(f.tok_ready, st); f.has_tok_ready = true; }
  f.edge(f.a, st);

  const int tile_grid = min(cdiv(Tcap, fz::TM), sm_count());
  const int warp_grid = cdiv(Tcap, fz::ATT_TOK);
  const size_t att_smem = sizeof(float) * 2 * (size_t)fz::att_rows_cap(L) * d;
  for (int b = 0; b < m->num_blocks; ++b) {
    const float* P = theta + l.block(b);
    float* X = w.slot[b][0]; float* Q1 = w.slot[b][1]; float* Qp = w.slot[b][2]; float* Kp = w.slot[b][3];
    float* Vp = w.slot[b][4]; float* Y = w.slot[b][5]; float* Z = w.slot[b][6]; float* H = w.slot[b][7];
    float* Xn = (b + 1 < m->num_blocks) ? w.slot[b + 1][0] : w.xfinal;
    fz::QkvFwdArgs qa;
    qa.X = X; qa.Xw = X; qa.embed = (b == 0);
    qa.table = theta + l.off_table; qa.pos_table = theta + l.off_pos;
    qa.tok_row = w.tok_row; qa.tok_id = w.tok_id; qa.row_len = w.row_len; qa.row_off = w.row_off;
    qa.sqrt_d = sqrtf((float)d); qa.drop_p = dropout_rate; qa.seed = seed; qa.d_step = d_step;
    qa.ln_b = P + l.ln1b; qa.ln_g = P + l.ln1g; qa.Q1 = Q1; qa.mean = w.mean1[b]; qa.rstd = w.rstd1[b];
    qa.Wq = shadow_of(w, b, 0, 0); qa.Wk = shadow_of(w, b, 1, 0); qa.Wv = shadow_of(w, b, 2, 0);
    qa.bq = P + l.bq; qa.bk = P + l.bk; qa.bv = P + l.bv;
    qa.Q = Qp; qa.K = Kp; qa.V = Vp; qa.dT = dT; qa.d = d; qa.L = L;

    fz::AttnFwdArgs aa;
    aa.Q = Qp; aa.K = Kp; aa.V = Vp; aa.Q1 = Q1; aa.tok_row = w.tok_row; aa.row_off = w.row_off;
    aa.probs = w.probs[b]; aa.Y = Y; aa.Z = Z; aa.mean2 = w.mean2[b]; aa.rstd2 = w.rstd2[b];
    aa.ln_b = P + l.ln2b; aa.ln_g = P + l.ln2g; aa.dT = dT; aa.d = d; aa.nh = m->num_heads; aa.L = L; aa.Tcap = Tcap;
    aa.drop_p = dropout_rate; aa.seed = seed; aa.d_step = d_step; aa.site = 1u + 3u * b;

    fz::FfnFwdArgs fa;
    fa.Z = Z; fa.H = H; fa.Xn = Xn; fa.W1 = shadow_of(w, b, 3, 0); fa.W2 = shadow_of(w, b, 4, 0);
    fa.b1 = P + l.b1; fa.b2 = P + l.b2; fa.dT = dT; fa.d = d;
    fa.drop_p = dropout_rate; fa.seed = seed; fa.d_step = d_step; fa.site1 = 2u + 3u * b; fa.site2 = 3u + 3u * b;
    launch_chain(fz::k_qkv_fwd, dim3(tile_grid), dim3(fz::NTHR), fz::QKV_FWD_SMEM, st, f.pdl && b > 0, qa);
    launch_chain(fz::k_attn_ln_fwd, dim3(warp_grid), dim3(256), att_smem, st, f.pdl, aa);
    launch_chain(fz::k_ffn_fwd, dim3(tile_grid), dim3(fz::NTHR), fz::FFN_FWD_SMEM, st, f.pdl, fa);
    ADER_CHECK_LAUNCH("encoder_fwd_tc/block");
  }
  launch_chain(k_ln_last_fwd, dim3(cdiv((long long)M * 32, 256)), dim3(256), 0, st, f.pdl, (const float*)w.xfinal, (const int*)w.row_len,
               (const int*)w.row_off, M, rep, w.meanf, w.rstdf, theta + l.off_lnf, theta + l.off_lnf + d, d);
  ADER_CHECK_LAUNCH("encoder_fwd_tc/final_ln");
  return 0;
}

// weight / LayerNorm-parameter gradient launch: two 4-warp CTAs per GEMM problem and split, one per LayerNorm problem
static void launch_wgrad(const fz::WgradArgs& wa, cudaStream_t st) {
  fz::k_wgrad2<<<dim3(SPLITS, 2 * wa.n_gemm + wa.n_ln), fz::WG2_THR, fz::WGRAD2_SMEM, st>>>(wa);
}

int ader::enc_scatter_plan_run(const AderModel* m, int M, int Tcap, const void* ws, void* bwd_ws, Fork& f) {
  if (!f.parallel() || !f.has_tok_ready) return 0;
  EncWs w = carve_enc(m, M, Tcap, (char*)ws);
  BwdWs g = carve_bwd(m, M, Tcap, (char*)bwd_ws);
  cudaStreamWaitEvent(f.c, f.tok_ready, 0);
  if (int e = run_scatter_plan(m, w, g, M, Tcap, f.c)) return e;
  f.plan_ready = f.take();
  cudaEventRecord(f.plan_ready, f.c);
  f.plan_done = true;
  return 0;
}

extern "C" int32_t ader_encoder_bwd_tc(const AderModel* m, const float* theta, const int32_t* ids, int32_t M,
                                       int32_t Tcap, const void* ws, void* bwd_ws, const float* d_rep, float* grad,
                                       float dropout_rate, uint64_t seed, const int32_t* d_step, void* stream) {
  Fork f = Fork::serial((cudaStream_t)stream);
  return enc_bwd_tc_run(m, theta, ids, M, Tcap, ws, bwd_ws, d_rep, grad, dropout_rate, seed, d_step, f);
}

// Launch plan (f.parallel()): the data-gradient chain lnf_bwd -> per block (ffn_bwd, attn_bwd, qkv_bwd) -> scatter stays on
// f.main; the weight-gradient kernel of each block, the LayerNorm-parameter / position-table reductions and the fixed-order
// reduction of the split partials run beside it on f.a / f.c.  Blocks alternate between two sets of gradient buffers and
// the block-to-block gradient rotates over three, so a weight-gradient kernel never reads a buffer the chain is rewriting.
int ader::enc_bwd_tc_run(const AderModel* m, const float* theta, const int32_t* ids, int M, int Tcap, const void* ws, void* bwd_ws,
                         const float* d_rep, float* grad, float dropout_rate, uint64_t seed, const int32_t* d_step, Fork& f) {
  if (int e = check_model(m)) return e;
  if (int e = path_check(m, ADER_PATH_ENCODER_TC)) return e;
  ADER_CHECK_ARG(theta && ids && ws && bwd_ws && d_rep && grad, "encoder_bwd_tc: NULL pointer");
  ADER_CHECK_ARG(M > 0 && Tcap > 0, "encoder_bwd_tc: bad M/Tcap");
  ADER_CHECK_ARG(dropout_rate >= 0.f && dropout_rate < 1.f, "encoder_bwd_tc: dropout_rate out of range");
  if (int e = fused_ready()) return e;
  cudaStream_t st = f.main;
  const Layout l = make_layout(m);
  const int d = m->d, L = m->maxlen;
  const float p = dropout_rate;
  EncWs w = carve_enc(m, M, Tcap, (char*)ws);
  BwdWs g = carve_bwd(m, M, Tcap, (char*)bwd_ws);
  const int* dT = w.row_off + M;
  const long long PS = l.dense_count();
  auto part = [&](long long param_off) { return g.partial + (param_off - l.off_pos); };
  float* chain[3] = {g.g[0], g.g[1], g.g[10]};
  int ci = 0;
  const int ln_grid = cdiv((long long)Tcap * 32, 256);
  const int ln_threads = ((d + 31) / 32) * 32;
  const int tile_grid = min(cdiv(Tcap, fz::TM), sm_count());

  // final LayerNorm: data gradient on the chain, parameter gradient beside it
  auto ln_params = [&] {
    f.edge(st, f.c);
    k_ln_param_grad<PG_LANES><<<SPLITS, dim3(ln_threads, PG_LANES), 0, f.c>>>(d_rep, w.xfinal, w.meanf, w.rstdf, dT, M, w.row_len, w.row_off, d,
                                                   part(l.off_lnf), part(l.off_lnf + d), PS);
  };
  if (f.has_drep) {                           // the loss group left the d_rep reduction to the kernel below
    launch_chain(k_lnf_bwd_drep, dim3(cdiv((long long)(Tcap + M) * 32, 256)), dim3(256), 0, st, f.pdl, f.drep, const_cast<float*>(d_rep),
                 (const float*)w.xfinal, (const float*)w.meanf, (const float*)w.rstdf, theta + l.off_lnf + d, (const int*)w.tok_row,
                 (const int*)w.row_off, (const int*)w.row_len, chain[0], dT, M, Tcap, d);
    ADER_CHECK_LAUNCH("encoder_bwd_tc/final_ln+d_rep");
    ln_params();
  } else {
    ln_params();
    // directly behind the d_rep reduction on f.main in the fused step (f.pdl is only set there)
    launch_chain(k_lnf_bwd, dim3(ln_grid), dim3(256), 0, st, f.pdl, d_rep, (const float*)w.xfinal, (const float*)w.meanf, (const float*)w.rstdf,
                 theta + l.off_lnf + d, (const int*)w.tok_row, (const int*)w.row_off, chain[0], dT, d);
    ADER_CHECK_LAUNCH("encoder_bwd_tc/final_ln");
  }

  cudaEvent_t wg_done[8][3];                // weight-gradient pieces of block b finished (f.wg[k]), parallel plans only
  for (int b = m->num_blocks - 1; b >= 0; --b) {
    const long long bo = l.block(b);
    const float* P = theta + bo;
    const float* X = w.slot[b][0]; const float* Q1 = w.slot[b][1]; const float* Qp = w.slot[b][2];
    const float* Kp = w.slot[b][3]; const float* Vp = w.slot[b][4]; const float* Y = w.slot[b][5];
    const float* Z = w.slot[b][6]; const float* H = w.slot[b][7];
    float* const* gs = (b & 1) ? g.g2 : g.g + 2;
    float *gO = gs[0], *gH = gs[1], *gZ = gs[2], *gY = gs[3], *gQ = gs[4], *gK = gs[5], *gV = gs[6], *gQ1 = gs[7];
    float* gX = chain[ci % 3]; float* gXin = chain[(ci + 1) % 3]; ++ci;
    // this block rewrites the buffer set (and chain buffer) last read by the weight-gradient kernel of block b + 2
    const bool joined = f.parallel() && b + 2 < m->num_blocks;
    if (joined) for (int k = 0; k < 3; ++k) cudaStreamWaitEvent(st, wg_done[b + 2][k], 0);
    fz::FfnBwdArgs fa;
    fa.gX = gX; fa.gO = gO; fa.H = H; fa.Y = Y; fa.Q1 = Q1; fa.mean2 = w.mean2[b]; fa.rstd2 = w.rstd2[b];
    fa.ln_g = P + l.ln2g; fa.W2b = shadow_of(w, b, 4, 1); fa.W1b = shadow_of(w, b, 3, 1);
    fa.gH = gH; fa.gZ = gZ; fa.gY = gY; fa.D = g.Dv; fa.dT = dT; fa.d = d;
    fa.drop_p = p; fa.seed = seed; fa.d_step = d_step; fa.site2 = 3u + 3u * b;
    fz::AttnBwdArgs ab;
    ab.Q = Qp; ab.K = Kp; ab.V = Vp; ab.probs = w.probs[b]; ab.gY = gY; ab.D = g.Dv;
    ab.tok_row = w.tok_row; ab.row_off = w.row_off; ab.gQ = gQ; ab.gK = gK; ab.gV = gV;
    ab.dT = dT; ab.d = d; ab.nh = m->num_heads; ab.L = L; ab.Tcap = Tcap; ab.drop_p = p; ab.seed = seed; ab.d_step = d_step; ab.site = 1u + 3u * b;
    fz::QkvBwdArgs qb;
    qb.gQ = gQ; qb.gK = gK; qb.gV = gV; qb.gY = gY; qb.X = X; qb.mean1 = w.mean1[b]; qb.rstd1 = w.rstd1[b];
    qb.ln_g = P + l.ln1g; qb.Wqb = shadow_of(w, b, 0, 1); qb.Wkb = shadow_of(w, b, 1, 1); qb.Wvb = shadow_of(w, b, 2, 1);
    qb.gQ1 = gQ1; qb.gXin = gXin; qb.dT = dT; qb.d = d;
    qb.drop_p = (b == 0) ? p : 0.f; qb.seed = seed; qb.d_step = d_step;       // block 0: x0 = drop(emb) (ADER.py:55)
    // weight / bias / LayerNorm-parameter gradients (TF32 tensor cores, fp32 accumulate, split partials) in three pieces
    const float* gOut = (p > 0.f) ? gO : gX;
    fz::WgradArgs wa[3];
    wa[0].p[0] = {H, gOut, nullptr, nullptr, part(bo + l.w2), part(bo + l.b2)};
    wa[0].p[1] = {Z, gH, nullptr, nullptr, part(bo + l.w1), part(bo + l.b1)};
    wa[0].p[2] = {Y, gZ, w.mean2[b], w.rstd2[b], part(bo + l.ln2b), part(bo + l.ln2g)};
    wa[0].n_gemm = 2; wa[0].n_ln = 1;
    wa[1].p[0] = {Q1, gQ, nullptr, nullptr, part(bo + l.wq), part(bo + l.bq)};
    wa[1].p[1] = {X, gK, nullptr, nullptr, part(bo + l.wk), part(bo + l.bk)};
    wa[1].p[2] = {X, gV, nullptr, nullptr, part(bo + l.wv), part(bo + l.bv)};
    wa[1].n_gemm = 3; wa[1].n_ln = 0;
    wa[2].p[0] = {X, gQ1, w.mean1[b], w.rstd1[b], part(bo + l.ln1b), part(bo + l.ln1g)};
    wa[2].n_gemm = 0; wa[2].n_ln = 1;
    for (int k = 0; k < 3; ++k) { wa[k].dT = dT; wa[k].d = d; wa[k].split_stride = PS; }
    // each weight-gradient piece is launched on its own stream as soon as its gradients exist, so
    // most of that work is done while the data-gradient chain is still running
    launch_chain(fz::k_ffn_bwd, dim3(tile_grid), dim3(fz::NTHR), fz::FFN_BWD_SMEM, st, f.pdl && !joined, fa);
    f.edge(st, f.wg[0]);
    launch_wgrad(wa[0], f.wg[0]);
    if (m->num_heads == 1) launch_chain(fz::k_attn_bwd_s1, dim3(cdiv(Tcap, fz::ATT_TOK)), dim3(256), (size_t)fz::att_bwd_smem(L, d), st, f.pdl, ab);
    else fz::k_attn_bwd_w<<<ln_grid, 256, 0, st>>>(ab);
    f.edge(st, f.wg[1]);
    launch_wgrad(wa[1], f.wg[1]);
    launch_chain(fz::k_qkv_bwd, dim3(tile_grid), dim3(fz::NTHR), fz::QKV_BWD_SMEM, st, f.pdl, qb);
    ADER_CHECK_LAUNCH("encoder_bwd_tc/dgrad");
    f.edge(st, f.wg[2]);
    launch_wgrad(wa[2], f.wg[2]);
    ADER_CHECK_LAUNCH("encoder_bwd_tc/wgrad");
    if (f.parallel())
      for (int k = 0; k < 3; ++k) { wg_done[b][k] = f.take(); cudaEventRecord(wg_done[b][k], f.wg[k]); }
  }
  const float* gX0 = chain[ci % 3];          // gradient w.r.t. the (dropout-masked) embedding output

  // Issue order of the tail = launch order of the graph nodes that become ready together when the chain ends: the
  // latency-bound scatter first, the bulk kernels (table Adam, position-table reduction) behind it -- a 5 000-CTA grid
  // issued first would sit in front of the scatter's 30 CTAs in the block scheduler.
  cudaEvent_t chain_end = nullptr;           // the data-gradient chain has produced gX0 (side work below waits for this, not
  if (f.parallel()) { chain_end = f.take(); cudaEventRecord(chain_end, st); }   // for the scatter issued in front of it)
  // item-table scatter (modules.py:127-130): adds to the rows the dE kernel wrote
  if (f.has_table_ready) cudaStreamWaitEvent(st, f.table_ready, 0);
  if (f.plan_done) {
    cudaStreamWaitEvent(st, f.plan_ready, 0);
    if (int e = run_scatter_apply(m, l, w, g, gX0, M, Tcap, grad, st)) return e;
  } else if (int e = run_table_scatter(m, l, w, g, gX0, M, Tcap, grad, st)) return e;
  if (f.adam) {                              // ... and the item-table rows here
    cudaStreamWaitEvent(st, f.adam->prep_ready, 0);
    if (int e = adam_table_part(m, *f.adam, st)) return e;
  }
  // position table (ADER.py:41-52) beside the scatter; then all split partials -> dense gradients in fixed order
  if (chain_end) cudaStreamWaitEvent(f.c, chain_end, 0);
  k_pos_grad<PG_LANES><<<dim3(L, SPLITS), dim3(ln_threads, PG_LANES), 0, f.c>>>(gX0, w.row_len, w.row_off, M, L, d, 0.f, 0, nullptr, g.partial, PS);
  f.edge(f.c, f.a);
  f.edge(f.wg[1], f.a);
  f.edge(f.wg[2], f.a);
  if (f.adam) {                              // fused step: reduce the partials and update the dense parameters in one launch
    const AdamPlan& ap = *f.adam;
    cudaStreamWaitEvent(f.a, ap.prep_ready, 0);
    k_reduce_partials_adam<<<cdiv(PS, 256), 256, 0, f.a>>>(g.partial, PS, SPLITS, PS, grad + l.off_pos, ap.theta + l.off_pos,
                                                           ap.m + l.off_pos, ap.v + l.off_pos, ap.state, ap.a.beta1, ap.a.beta2, ap.a.eps,
                                                           ap.a.ewc_lambda, ap.a.fisher ? ap.a.fisher + l.off_pos : nullptr,
                                                           ap.a.theta_star ? ap.a.theta_star + l.off_pos : nullptr);
  } else {
    k_reduce_partials<<<cdiv(PS, 256), 256, 0, f.a>>>(g.partial, PS, SPLITS, 0, PS, grad + l.off_pos);
  }
  f.edge(f.a, st);
  ADER_CHECK_LAUNCH("encoder_bwd_tc/embedding");
  return 0;
}

extern "C" int32_t ader_gather_rows_i32(const int32_t* src, const int32_t* idx, int32_t n, int32_t width,
                                        int32_t* out, void* stream);
__global__ void k_gather_rows(const int* __restrict__ src, const int* __restrict__ idx, int n, int width, int* __restrict__ out) {
  long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (long long)n * width) return;
  int i = (int)(e / width), c = (int)(e % width);
  out[e] = src[(long long)idx[i] * width + c];
}
extern "C" int32_t ader_gather_rows_i32(const int32_t* src, const int32_t* idx, int32_t n, int32_t width,
                                        int32_t* out, void* stream) {
  ADER_CHECK_ARG(src && idx && out && n >= 0 && width > 0, "gather_rows: bad argument");
  if (n == 0) return 0;
  k_gather_rows<<<cdiv((long long)n * width, 256), 256, 0, (cudaStream_t)stream>>>(src, idx, n, width, out);
  ADER_CHECK_LAUNCH("gather_rows");
  return 0;
}

// Batch assembly in one launch: rows ti[] of the train matrix (+ their labels) followed by rows ei[] of the exemplar
// matrix (+ their aux word: teacher row or label) -> ids [n_train + n_ex, width], pos [n_train], aux [n_ex].
__global__ void k_gather_batch(const int* __restrict__ t_ids, const int* __restrict__ t_lab, const int* __restrict__ ti, int n_train,
                               const int* __restrict__ e_ids, const int* __restrict__ e_aux, const int* __restrict__ ei, int n_ex,
                               int width, int* __restrict__ ids, int* __restrict__ pos, int* __restrict__ aux) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int w1 = width + 1;
  if (e >= (long long)(n_train + n_ex) * w1) return;
  const int row = (int)(e / w1), c = (int)(e % w1);
  if (row < n_train) {
    const long long src = ti[row];
    if (c < width) ids[(long long)row * width + c] = t_ids[src * width + c];
    else pos[row] = t_lab[src];
  } else {
    const int r = row - n_train;
    const long long src = ei[r];
    if (c < width) ids[(long long)row * width + c] = e_ids[src * width + c];
    else if (aux) aux[r] = e_aux ? e_aux[src] : 0;
  }
}
extern "C" int32_t ader_gather_batch(const int32_t* t_ids, const int32_t* t_lab, const int32_t* ti, int32_t n_train,
                                     const int32_t* e_ids, const int32_t* e_aux, const int32_t* ei, int32_t n_ex,
                                     int32_t width, int32_t* ids, int32_t* pos, int32_t* aux, void* stream) {
  ADER_CHECK_ARG(n_train >= 0 && n_ex >= 0 && width > 0 && ids, "gather_batch: bad argument");
  ADER_CHECK_ARG(n_train == 0 || (t_ids && t_lab && ti && pos), "gather_batch: NULL train pointer");
  ADER_CHECK_ARG(n_ex == 0 || (e_ids && ei), "gather_batch: NULL exemplar pointer");
  if (n_train + n_ex == 0) return 0;
  k_gather_batch<<<cdiv((long long)(n_train + n_ex) * (width + 1), 256), 256, 0, (cudaStream_t)stream>>>(
      t_ids, t_lab, ti, n_train, e_ids, e_aux, ei, n_ex, width, ids, pos, aux);
  ADER_CHECK_LAUNCH("gather_batch");
  return 0;
}

// The same batch assembly fed from an epoch-resident index queue (SURVEY 8(f): the host leaves the training loop): `q`
// holds the row indices of every step of the epoch back to back ([train indices | exemplar indices] per step), q_off[s]
// is where step s starts, *counter is the running step.  A captured step graph replays with no host-to-device traffic at
// all; ader_queue_advance (stream-ordered behind the gather) moves to the next step.
__global__ void k_gather_batch_q(const int* __restrict__ t_ids, const int* __restrict__ t_lab, int n_train,
                                 const int* __restrict__ e_ids, const int* __restrict__ e_aux, int n_ex,
                                 const int* __restrict__ q, const long long* __restrict__ q_off, const int* __restrict__ counter,
                                 int width, int* __restrict__ ids, int* __restrict__ pos, int* __restrict__ aux) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int w1 = width + 1;
  if (e >= (long long)(n_train + n_ex) * w1) return;
  const int* ti = q + q_off[*counter];
  const int* ei = ti + n_train;
  const int row = (int)(e / w1), c = (int)(e % w1);
  if (row < n_train) {
    const long long src = ti[row];
    if (c < width) ids[(long long)row * width + c] = t_ids[src * width + c];
    else pos[row] = t_lab[src];
  } else {
    const int r = row - n_train;
    const long long src = ei[r];
    if (c < width) ids[(long long)row * width + c] = e_ids[src * width + c];
    else if (aux) aux[r] = e_aux ? e_aux[src] : 0;
  }
}
__global__ void k_queue_advance(int* counter) { *counter += 1; }

extern "C" int32_t ader_gather_batch_q(const int32_t* t_ids, const int32_t* t_lab, int32_t n_train, const int32_t* e_ids,
                                       const int32_t* e_aux, int32_t n_ex, const int32_t* q, const int64_t* q_off,
                                       const int32_t* counter, int32_t width, int32_t* ids, int32_t* pos, int32_t* aux,
                                       void* stream) {
  ADER_CHECK_ARG(n_train >= 0 && n_ex >= 0 && width > 0 && ids && q && q_off && counter, "gather_batch_q: bad argument");
  ADER_CHECK_ARG(n_train == 0 || (t_ids && t_lab && pos), "gather_batch_q: NULL train pointer");
  ADER_CHECK_ARG(n_ex == 0 || e_ids, "gather_batch_q: NULL exemplar pointer");
  if (n_train + n_ex == 0) return 0;
  k_gather_batch_q<<<cdiv((long long)(n_train + n_ex) * (width + 1), 256), 256, 0, (cudaStream_t)stream>>>(
      t_ids, t_lab, n_train, e_ids, e_aux, n_ex, q, (const long long*)q_off, counter, width, ids, pos, aux);
  ADER_CHECK_LAUNCH("gather_batch_q");
  return 0;
}
extern "C" int32_t ader_queue_advance(int32_t* counter, void* stream) {
  ADER_CHECK_ARG(counter, "queue_advance: NULL pointer");
  k_queue_advance<<<1, 1, 0, (cudaStream_t)stream>>>(counter);
  ADER_CHECK_LAUNCH("queue_advance");
  return 0;
}
