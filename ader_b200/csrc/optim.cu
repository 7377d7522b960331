// TF1 Adam (tf.train.AdamOptimizer, ADER.py:96; SURVEY S10 / A.3) fused with the EWC penalty
// gradient (EWC.py:115-124), and the Fisher-diagonal accumulators (EWC.py:126-164).
// HBM-bound: 24 B/param (theta, m, v read+write) + 4 B/param gradient read.
#include "common.cuh"

namespace ader {

// state[0] = step t (int), state[1] = bits of lr_t (float)
__global__ void k_adam_prep(int* __restrict__ state, float lr, float beta1, float beta2) {
  int t = state[0] + 1;
  state[0] = t;
  double lr_t = (double)lr * sqrt(1.0 - pow((double)beta2, (double)t)) / (1.0 - pow((double)beta1, (double)t));
  state[1] = __float_as_int((float)lr_t);
}

// early form for the fused step: the step size of step t + 1 without touching the counter (the dropout streams of the
// running step still read state[0]); the dense update (encoder.cu: k_reduce_partials_adam) bumps the counter when it is done
__global__ void k_adam_prep_early(int* __restrict__ state, float lr, float beta1, float beta2) {
  const int t = state[0] + 1;
  double lr_t = (double)lr * sqrt(1.0 - pow((double)beta2, (double)t)) / (1.0 - pow((double)beta1, (double)t));
  state[1] = __float_as_int((float)lr_t);
}

__global__ void __launch_bounds__(256) k_adam(float* __restrict__ theta, float* __restrict__ am, float* __restrict__ av,
                                              const float* __restrict__ grad, const int* __restrict__ state,
                                              long long n_table, long long table_lo, long long dense_lo, long long n_total,
                                              float beta1, float beta2, float eps, float ewc_lambda,
                                              const float* __restrict__ fisher, const float* __restrict__ theta_star) {
  const float lr_t = __int_as_float(state[1]);
  // two elements per thread (both ranges start on even offsets because d is even)
  long long i2 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 2;
  if (i2 >= n_total) return;
  long long e = (i2 < n_table) ? table_lo + i2 : dense_lo + (i2 - n_table);
  float2 g = *reinterpret_cast<const float2*>(grad + e);
  float2 th = *reinterpret_cast<const float2*>(theta + e);
  float2 m = *reinterpret_cast<const float2*>(am + e);
  float2 v = *reinterpret_cast<const float2*>(av + e);
  float2 f = make_float2(0.f, 0.f), ts = make_float2(0.f, 0.f);
  if (ewc_lambda != 0.f) {
    f = *reinterpret_cast<const float2*>(fisher + e);
    ts = *reinterpret_cast<const float2*>(theta_star + e);
  }
  adam_update_elem(g.x, th.x, m.x, v.x, lr_t, beta1, beta2, eps, ewc_lambda, f.x, ts.x);
  adam_update_elem(g.y, th.y, m.y, v.y, lr_t, beta1, beta2, eps, ewc_lambda, f.y, ts.y);
  *reinterpret_cast<float2*>(theta + e) = th;
  *reinterpret_cast<float2*>(am + e) = m;
  *reinterpret_cast<float2*>(av + e) = v;
}

__global__ void __launch_bounds__(256) k_fisher_acc(const float* __restrict__ grad, double* __restrict__ acc,
                                                    long long n_table, long long table_lo, long long dense_lo,
                                                    long long n_total) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_total) return;
  long long e = (i < n_table) ? table_lo + i : dense_lo + (i - n_table);
  float g = grad[e];
  float sq = __fmul_rn(g, g);          // np.square on float32 stays float32 (EWC.py:161)
  acc[e] += (double)sq;                // accumulated in float64 (EWC.py:136-137)
}

__global__ void __launch_bounds__(256) k_fisher_fin(const double* __restrict__ acc, float* __restrict__ fisher,
                                                    long long n_table, long long table_lo, long long dense_lo,
                                                    long long n_total, double inv_n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_total) return;
  long long e = (i < n_table) ? table_lo + i : dense_lo + (i - n_table);
  fisher[e] = (float)(acc[e] * inv_n);
}

}  // namespace ader

using namespace ader;

extern "C" int32_t ader_adam_step(const AderModel* m, float* theta, float* adam_m, float* adam_v,
                                  const float* grad, int32_t* state, const AderAdamArgs* a, void* stream) {
  if (int e = check_model(m)) return e;
  ADER_CHECK_ARG(theta && adam_m && adam_v && grad && state && a, "adam_step: NULL pointer");
  ADER_CHECK_ARG(a->V >= 1 && a->V < m->v_tab, "adam_step: max_item %d outside table", a->V);
  ADER_CHECK_ARG(a->ewc_lambda == 0.f || (a->fisher && a->theta_star), "adam_step: EWC needs fisher and theta_star");
  const Layout l = make_layout(m);
  const long long n_table = (long long)a->V * m->d;
  const long long n_total = n_table + l.dense_count();
  cudaStream_t st = (cudaStream_t)stream;
  k_adam_prep<<<1, 1, 0, st>>>(state, a->lr, a->beta1, a->beta2);
  k_adam<<<cdiv(n_total / 2 + 1, 256), 256, 0, st>>>(theta, adam_m, adam_v, grad, state, n_table, (long long)m->d,
                                                     l.off_pos, n_total, a->beta1, a->beta2, a->eps, a->ewc_lambda,
                                                     a->fisher, a->theta_star);
  ADER_CHECK_LAUNCH("adam");
  return 0;
}

int ader::adam_prep_early(const AdamPlan& p, cudaStream_t st) {
  k_adam_prep_early<<<1, 1, 0, st>>>(p.state, p.a.lr, p.a.beta1, p.a.beta2);
  ADER_CHECK_LAUNCH("adam prep");
  return 0;
}
int ader::adam_table_part(const AderModel* m, const AdamPlan& p, cudaStream_t st) {
  const Layout l = make_layout(m);
  const long long n_table = (long long)p.a.V * m->d;
  k_adam<<<cdiv(n_table / 2 + 1, 256), 256, 0, st>>>(p.theta, p.m, p.v, p.grad, p.state, n_table, (long long)m->d, l.off_pos, n_table,
                                                     p.a.beta1, p.a.beta2, p.a.eps, p.a.ewc_lambda, p.a.fisher, p.a.theta_star);
  ADER_CHECK_LAUNCH("adam table");
  return 0;
}
extern "C" int32_t ader_fisher_accumulate(const AderModel* m, const float* grad, double* acc, int32_t V, void* stream) {
  if (int e = check_model(m)) return e;
  ADER_CHECK_ARG(grad && acc && V >= 1 && V < m->v_tab, "fisher_accumulate: bad argument");
  const Layout l = make_layout(m);
  const long long n_table = (long long)V * m->d, n_total = n_table + l.dense_count();
  k_fisher_acc<<<cdiv(n_total, 256), 256, 0, (cudaStream_t)stream>>>(grad, acc, n_table, (long long)m->d, l.off_pos, n_total);
  ADER_CHECK_LAUNCH("fisher_acc");
  return 0;
}

extern "C" int32_t ader_fisher_finalize(const AderModel* m, const double* acc, float* fisher, int32_t V,
                                        int32_t n_data, void* stream) {
  if (int e = check_model(m)) return e;
  ADER_CHECK_ARG(acc && fisher && V >= 1 && V < m->v_tab && n_data > 0, "fisher_finalize: bad argument");
  const Layout l = make_layout(m);
  const long long n_table = (long long)V * m->d, n_total = n_table + l.dense_count();
  cudaStream_t st = (cudaStream_t)stream;
  cudaMemsetAsync(fisher, 0, sizeof(float) * l.total, st);
  k_fisher_fin<<<cdiv(n_total, 256), 256, 0, st>>>(acc, fisher, n_table, (long long)m->d, l.off_pos, n_total, 1.0 / (double)n_data);
  ADER_CHECK_LAUNCH("fisher_fin");
  return 0;
}
