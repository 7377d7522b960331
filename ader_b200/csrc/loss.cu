// Output projection + softmax cross-entropy + ADER distillation (ADER.py:88-93, 108-138),
// exact-fp32 reference mode: logits are produced by the strided SGEMM, a row kernel turns them
// into the loss and dS in place, two more GEMMs give d_rep and the dense item-table gradient.
// (The tcgen05 fused kernel in logits_tc.cu is the fast path; this file is the exact one and
// also serves eval scoring, teacher-logit export and the Fisher path.)
#include "common.cuh"

namespace ader {

constexpr int DR_SPLITS = 16;

__device__ __forceinline__ float block_reduce(float v, bool is_max, float* sh) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    float y = __shfl_xor_sync(0xffffffffu, v, o);
    v = is_max ? fmaxf(v, y) : v + y;
  }
  __syncthreads();                 // protect sh from the previous call
  if (lane == 0) sh[wid] = v;
  __syncthreads();
  float r = is_max ? -INFINITY : 0.f;
  for (int w = 0; w < nw; ++w) r = is_max ? fmaxf(r, sh[w]) : r + sh[w];   // fixed order
  return r;
}

// one CTA per row; logits row -> row_loss, and dS written in place.
__global__ void __launch_bounds__(256) k_ce_kd_rows(float* __restrict__ S, long long ld, AderLossArgs a,
                                                    float* __restrict__ row_loss) {
  __shared__ float sh[32];
  const int i = blockIdx.x;
  float* s = S + (long long)i * ld;
  const int V = a.V;
  const bool is_train = i < a.n_train;
  if (is_train || a.mode == 2) {
    const int label = is_train ? a.pos[i] : a.ex_pos[i - a.n_train];
    const float coef = is_train ? 1.0f / (float)(a.n_train_global > 0 ? a.n_train_global : a.n_train)
                                : a.lambda_ / (float)(a.n_ex_global > 0 ? a.n_ex_global : a.n_ex);
    float mx = -INFINITY;
    for (int j = threadIdx.x; j < V; j += blockDim.x) mx = fmaxf(mx, s[j]);
    mx = block_reduce(mx, true, sh);
    float sum = 0.f;
    for (int j = threadIdx.x; j < V; j += blockDim.x) sum += expf(s[j] - mx);
    sum = block_reduce(sum, false, sh);
    const float lse = mx + logf(sum);
    const float sl = s[label - 1];
    __syncthreads();
    if (threadIdx.x == 0) row_loss[i] = lse - sl;
    for (int j = threadIdx.x; j < V; j += blockDim.x) {
      float p = expf(s[j] - lse);
      s[j] = coef * (p - (j == label - 1 ? 1.f : 0.f));
    }
  } else {   // KD: student softmax over the first V_prev columns only (ADER.py:134)
    const int Vp = a.V_prev;
    const long long trow = a.teacher_row ? a.teacher_row[i - a.n_train] : (i - a.n_train);
    const float* t = a.teacher + trow * a.teacher_ld;
    const float coef = a.lambda_ / (float)(a.n_ex_global > 0 ? a.n_ex_global : a.n_ex);
    float mx = -INFINITY, mt = -INFINITY;
    for (int j = threadIdx.x; j < Vp; j += blockDim.x) { mx = fmaxf(mx, s[j]); mt = fmaxf(mt, t[j]); }
    mx = block_reduce(mx, true, sh);
    mt = block_reduce(mt, true, sh);
    float sum = 0.f, sumt = 0.f;
    for (int j = threadIdx.x; j < Vp; j += blockDim.x) { sum += expf(s[j] - mx); sumt += expf(t[j] - mt); }
    sum = block_reduce(sum, false, sh);
    sumt = block_reduce(sumt, false, sh);
    const float lse = mx + logf(sum), lset = mt + logf(sumt);
    float dot = 0.f;
    for (int j = threadIdx.x; j < Vp; j += blockDim.x) dot += expf(t[j] - lset) * s[j];
    dot = block_reduce(dot, false, sh);
    if (threadIdx.x == 0) row_loss[i] = lse - dot;
    for (int j = threadIdx.x; j < V; j += blockDim.x)
      s[j] = (j < Vp) ? coef * (expf(s[j] - lse) - expf(t[j] - lset)) : 0.f;
  }
}

__global__ void __launch_bounds__(256) k_loss_reduce(const float* __restrict__ row_loss, int n_train, int n_ex,
                                                     float lambda_, float* __restrict__ loss, int den_train, int den_ex) {
  __shared__ float sh[32];
  float a = 0.f, b = 0.f;
  for (int i = threadIdx.x; i < n_train; i += blockDim.x) a += row_loss[i];
  for (int i = threadIdx.x; i < n_ex; i += blockDim.x) b += row_loss[n_train + i];
  a = block_reduce(a, false, sh);
  b = block_reduce(b, false, sh);
  if (threadIdx.x == 0) {
    float v = n_train > 0 ? a / (float)den_train : 0.f;
    if (n_ex > 0) v += lambda_ * (b / (float)den_ex);
    loss[0] = v;
  }
}

__global__ void k_reduce_splits(const float* __restrict__ partial, long long stride, int splits, long long n,
                                float* __restrict__ out) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s = 0.f;
  for (int k = 0; k < splits; ++k) s += partial[(long long)k * stride + i];
  out[i] = s;
}

int launch_loss_reduce(const float* row_loss, int n_train, int n_ex, float lambda_, float* loss, cudaStream_t st,
                       int den_train, int den_ex) {
  k_loss_reduce<<<1, 256, 0, st>>>(row_loss, n_train, n_ex, lambda_, loss, den_train > 0 ? den_train : n_train,
                                   den_ex > 0 ? den_ex : n_ex);
  ADER_CHECK_LAUNCH("loss_reduce");
  return 0;
}

static long long logits_ld(int V) { return ((long long)V + 3) / 4 * 4; }

// rows = fp32 row of item 1 (theta + d, or a frozen teacher_table), row stride d
static int run_logits_rows(const AderModel* m, const float* rows, const float* rep, int M, int V, float* out,
                           long long ld, cudaStream_t st) {
  GemmArgs g; gemm_defaults(g);
  const int d = m->d;
  g.A = rep; g.a_rs = d; g.a_cs = 1;
  g.B = rows; g.b_rs = 1; g.b_cs = d;             // B(k=c, n=v) = E[(v+1)*d + c]  (ADER.py:90-91)
  g.C = out; g.c_rs = ld; g.c_cs = 1;
  g.M = M; g.N = V; g.K = d;
  return launch_gemm(g, st);
}
static int run_logits(const AderModel* m, const float* theta, const float* rep, int M, int V, float* out,
                      long long ld, cudaStream_t st) {
  return run_logits_rows(m, theta + m->d, rep, M, V, out, ld, st);
}

// frozen teacher: out[e, :] = src[teacher_row[e], :] (identity when teacher_row is NULL)
__global__ void k_gather_rep(const float* __restrict__ src, const int* __restrict__ row, int n, int d, float* __restrict__ out) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)n * d) return;
  const int e = (int)(idx / d), c = (int)(idx % d);
  out[idx] = src[(long long)(row ? row[e] : e) * d + c];
}

// ---- evaluation rows: rank of the ground truth + top-k (ADER.py:103, util.py:323-339) -------
struct ValIdx { float v; int j; };
__device__ __forceinline__ bool better(float v, int j, float bv, int bj) { return v > bv || (v == bv && j < bj); }

__global__ void __launch_bounds__(256) k_rank_topk_rows(const float* __restrict__ S, long long ld, int V,
                                                        const int* __restrict__ gt, int k,
                                                        int* __restrict__ rank, int* __restrict__ topk_item,
                                                        float* __restrict__ topk_score) {
  __shared__ float shv[8]; __shared__ int shj[8]; __shared__ int shc[8];
  __shared__ float pv_s; __shared__ int pj_s;
  const int i = blockIdx.x;
  const float* s = S + (long long)i * ld;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (gt) {
    const int g = gt[i] - 1;
    const float sg = s[g];
    int c = 0;
    for (int j = threadIdx.x; j < V; j += blockDim.x) { float v = s[j]; c += (v > sg) || (v == sg && j < g); }
#pragma unroll
    for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if (lane == 0) shc[wid] = c;
    __syncthreads();
    if (threadIdx.x == 0) { int t = 0; for (int w = 0; w < 8; ++w) t += shc[w]; rank[i] = t; }
  }
  if (k <= 0) return;
  if (threadIdx.x == 0) { pv_s = INFINITY; pj_s = -1; }
  __syncthreads();
  for (int it = 0; it < k; ++it) {
    const float pv = pv_s; const int pj = pj_s;
    float bv = -INFINITY; int bj = 0x7fffffff;
    for (int j = threadIdx.x; j < V; j += blockDim.x) {
      float v = s[j];
      bool eligible = (v < pv) || (v == pv && j > pj);
      if (eligible && better(v, j, bv, bj)) { bv = v; bj = j; }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      float ov = __shfl_xor_sync(0xffffffffu, bv, o); int oj = __shfl_xor_sync(0xffffffffu, bj, o);
      if (better(ov, oj, bv, bj)) { bv = ov; bj = oj; }
    }
    if (lane == 0) { shv[wid] = bv; shj[wid] = bj; }
    __syncthreads();
    if (threadIdx.x == 0) {
      float fv = shv[0]; int fj = shj[0];
      for (int w = 1; w < 8; ++w) if (better(shv[w], shj[w], fv, fj)) { fv = shv[w]; fj = shj[w]; }
      bool ok = fj != 0x7fffffff;
      topk_item[(long long)i * k + it] = ok ? fj + 1 : 0;
      topk_score[(long long)i * k + it] = ok ? fv : -INFINITY;
      pv_s = fv; pj_s = ok ? fj : 0x7fffffff;
    }
    __syncthreads();
  }
}

}  // namespace ader

using namespace ader;

static bool frozen_kd(const AderLossArgs* a) { return a->mode == 1 && a->n_ex > 0 && a->teacher_rep; }

extern "C" size_t ader_loss_ws_bytes(const AderModel* m, const AderLossArgs* a) {
  if (check_model(m) || !a || a->M <= 0 || a->V <= 0) return 0;
  size_t o = align_up(sizeof(float) * (size_t)a->M * logits_ld(a->V));
  o += align_up(sizeof(float) * (size_t)DR_SPLITS * a->M * m->d);
  if (frozen_kd(a) && a->V_prev > 0) {      // gathered exemplar reps + their teacher logits [n_ex, V_prev]
    o += align_up(sizeof(float) * (size_t)a->n_ex * m->d);
    o += align_up(sizeof(float) * (size_t)a->n_ex * logits_ld(a->V_prev));
  }
  return o;
}

extern "C" int32_t ader_loss_fwd_bwd(const AderModel* m, const float* theta, const float* rep,
                                     const AderLossArgs* a, void* ws, float* loss, float* row_loss,
                                     float* d_rep, float* grad, void* stream) {
  if (int e = check_model(m)) return e;
  ADER_CHECK_ARG(theta && rep && a && ws && loss && row_loss, "loss_fwd_bwd: NULL pointer");
  ADER_CHECK_ARG(a->M == a->n_train + a->n_ex && a->M > 0, "loss_fwd_bwd: M (%d) != n_train + n_ex (%d + %d)", a->M, a->n_train, a->n_ex);
  ADER_CHECK_ARG(a->V >= 1 && a->V < m->v_tab, "loss_fwd_bwd: max_item %d outside table of %d rows", a->V, m->v_tab);
  ADER_CHECK_ARG(a->mode >= 0 && a->mode <= 2, "loss_fwd_bwd: bad mode %d", a->mode);
  ADER_CHECK_ARG(a->n_train == 0 || a->pos, "loss_fwd_bwd: pos is NULL");
  if (a->n_ex > 0) {
    ADER_CHECK_ARG(a->mode != 0, "loss_fwd_bwd: exemplar rows given in vanilla mode");
    if (a->mode == 1) { if (int e = check_teacher(a, "loss_fwd_bwd", false)) return e; }
    if (a->mode == 2) ADER_CHECK_ARG(a->ex_pos, "loss_fwd_bwd: exemplar_pos is NULL");
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int d = m->d, M = a->M, V = a->V;
  const long long ld = logits_ld(V);
  float* S = (float*)ws;
  float* part = (float*)((char*)ws + align_up(sizeof(float) * (size_t)M * ld));
  AderLossArgs ka = *a;
  if (frozen_kd(a)) {
    // teacher logits of the exemplar rows from the snapshot, by the same SGEMM as ader_logits (each element is a
    // sequential k-sum independent of M and of the row's position), so the rows match stored logits bit for bit
    char* p = (char*)part + align_up(sizeof(float) * (size_t)DR_SPLITS * M * d);
    float* trep = (float*)p;
    float* tl = (float*)(p + align_up(sizeof(float) * (size_t)a->n_ex * d));
    const long long tld = logits_ld(a->V_prev);
    k_gather_rep<<<cdiv((long long)a->n_ex * d, 256), 256, 0, st>>>(a->teacher_rep, a->teacher_row, a->n_ex, d, trep);
    ADER_CHECK_LAUNCH("gather teacher reps");
    if (int e = run_logits_rows(m, a->teacher_table, trep, a->n_ex, a->V_prev, tl, tld, st)) return e;
    ka.teacher = tl; ka.teacher_row = nullptr; ka.teacher_ld = tld;
  }
  if (int e = run_logits(m, theta, rep, M, V, S, ld, st)) return e;
  k_ce_kd_rows<<<M, 256, 0, st>>>(S, ld, ka, row_loss);
  if (int e = launch_loss_reduce(row_loss, a->n_train, a->n_ex, a->lambda_, loss, st, a->n_train_global, a->n_ex_global)) return e;
  ADER_CHECK_LAUNCH("loss rows");
  if (d_rep) {   // d_rep = dS . E[1..V]   (split-K over the vocabulary, fixed-order reduce)
    GemmArgs g; gemm_defaults(g);
    g.A = S; g.a_rs = ld; g.a_cs = 1;
    g.B = theta + d; g.b_rs = d; g.b_cs = 1;
    g.C = part; g.c_rs = d; g.c_cs = 1;
    g.M = M; g.N = d; g.K = V; g.splits = DR_SPLITS; g.split_stride = (long long)M * d;
    if (int e = launch_gemm(g, st)) return e;
    k_reduce_splits<<<cdiv((long long)M * d, 256), 256, 0, st>>>(part, (long long)M * d, DR_SPLITS, (long long)M * d, d_rep);
    ADER_CHECK_LAUNCH("d_rep reduce");
  }
  if (grad) {    // dE[1..V] = dS^T . rep
    GemmArgs g; gemm_defaults(g);
    g.A = S; g.a_rs = 1; g.a_cs = ld;
    g.B = rep; g.b_rs = d; g.b_cs = 1;
    g.C = grad + d; g.c_rs = d; g.c_cs = 1;
    g.M = V; g.N = d; g.K = M;
    if (int e = launch_gemm(g, st)) return e;
  }
  return 0;
}

extern "C" int32_t ader_logits(const AderModel* m, const float* theta, const float* rep, int32_t M, int32_t V,
                               float* logits, int64_t ld, void* stream) {
  if (int e = check_model(m)) return e;
  ADER_CHECK_ARG(theta && rep && logits && M > 0 && V >= 1 && V < m->v_tab && ld >= V, "logits: bad argument");
  return run_logits(m, theta, rep, M, V, logits, ld, (cudaStream_t)stream);
}

extern "C" size_t ader_eval_ws_bytes(const AderModel* m, int32_t M, int32_t V) {
  if (check_model(m) || M <= 0 || V <= 0) return 0;
  return align_up(sizeof(float) * (size_t)M * logits_ld(V));
}

extern "C" int32_t ader_eval_rank_topk(const AderModel* m, const float* theta, const float* rep, const int32_t* gt,
                                       int32_t M, int32_t V, int32_t k, void* ws, int32_t* rank,
                                       int32_t* topk_item, float* topk_score, void* stream) {
  if (int e = check_model(m)) return e;
  ADER_CHECK_ARG(theta && rep && ws && M > 0 && V >= 1 && V < m->v_tab, "eval_rank_topk: bad argument");
  ADER_CHECK_ARG(k >= 0 && k <= 32 && (k == 0 || (topk_item && topk_score)), "eval_rank_topk: bad k");
  ADER_CHECK_ARG(!gt || rank, "eval_rank_topk: rank is NULL");
  cudaStream_t st = (cudaStream_t)stream;
  const long long ld = logits_ld(V);
  float* S = (float*)ws;
  if (int e = run_logits(m, theta, rep, M, V, S, ld, st)) return e;
  k_rank_topk_rows<<<M, 256, 0, st>>>(S, ld, V, gt, k, rank, topk_item, topk_score);
  ADER_CHECK_LAUNCH("rank_topk_rows");
  return 0;
}
