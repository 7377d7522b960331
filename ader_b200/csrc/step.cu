// One training pass as a fork/join DAG: encoder forward, logits + CE + distillation forward/backward, encoder
// backward and the embedding scatter (everything of `train_op` before the optimiser, main.py:233-256).
//
// The three tensor-core groups are latency chains of 3-25 us kernels; a third of the launches of a step is not on
// the critical path (teacher products, table-tile packing, dE, weight / LayerNorm / position gradients, partial
// reductions).  This entry issues the same kernels as
//     ader_encoder_fwd_tc -> ader_loss_fwd_bwd_tc -> ader_encoder_bwd_tc
// with the same arguments -- results are bit-identical -- but puts the off-path work on five library-owned streams
// joined by events, and launches the kernel-to-kernel links of the chain as programmatic dependent launches.
// Captured by a CUDA graph the side streams become parallel branches of the graph.  ader_train_step_tc adds the
// optimiser to the same DAG.
#include "common.cuh"

namespace ader {

struct StreamPool {
  cudaStream_t s[5];     // side streams, lowest priority (3 general + 2 more for weight-gradient pieces)
  cudaEvent_t ev[128];
  bool ok;
  StreamPool() : ok(false) {}
  int init() {
    if (ok) return 0;
    int least = 0, greatest = 0;
    cudaDeviceGetStreamPriorityRange(&least, &greatest);
    for (int i = 0; i < 5; ++i)
      if (cudaStreamCreateWithPriority(&s[i], cudaStreamNonBlocking, least) != cudaSuccess) return fail(-3, "train_fwd_bwd_tc: cannot create a stream");
    for (int i = 0; i < 128; ++i)
      if (cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming) != cudaSuccess) return fail(-3, "train_fwd_bwd_tc: cannot create an event");
    ok = true;
    return 0;
  }
};
// one pool per host thread and device (streams belong to the device that was current at creation)
static thread_local StreamPool g_pool[16];

}  // namespace ader

using namespace ader;

static int run_step(const AderModel* m, const float* theta, const int32_t* ids, int32_t M, int32_t Tcap,
                    const AderLossArgs* a, void* enc_ws, void* bwd_ws, void* loss_ws, float* rep,
                    float* loss, float* row_loss, float* d_rep, float* grad, float dropout_rate,
                    uint64_t seed, const int32_t* d_step, int32_t serial, cudaStream_t st, AdamPlan* adam,
                    const char* entry) {
  ADER_CHECK_ARG(m && theta && ids && a && enc_ws && bwd_ws && loss_ws && rep && loss && row_loss && d_rep && grad,
                 "train step: NULL pointer");
  ADER_CHECK_ARG(dropout_rate >= 0.f && dropout_rate < 1.f, "%s: dropout_rate out of range", entry);
  ADER_CHECK_ARG(a->M == M, "train step: loss rows (%d) != encoder rows (%d)", a->M, M);
  Fork f = Fork::serial(st);
  if (!serial) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 16) return fail(-3, "train step: bad device");
    StreamPool& p = g_pool[dev];
    if (int e = p.init()) return e;
    f.a = p.s[0]; f.b = p.s[1]; f.c = p.s[2];
    f.wg[0] = f.a; f.wg[1] = p.s[3]; f.wg[2] = p.s[4];
    f.ev = p.ev; f.n_ev = 128; f.next_ev = 0;
  }
  // The chain stays on the caller's stream (a highest-priority chain stream measured slower: the hardware schedules
  // strictly by priority without back-fill, the side streams starve) and its kernel-to-kernel links are programmatic
  // dependent launches (0.343 -> 0.328 ms per step); DESIGN §3.4.
  f.pdl = true;
  f.fuse_drep = f.parallel() && d_rep;
  // teacher products / table tiles need nothing from the encoder: start them first, beside it
  f.edge(f.main, f.b);
  if (int e = loss_tc_run(m, theta, nullptr, a, loss_ws, nullptr, nullptr, nullptr, grad, f, 1)) return e;
  if (adam) {                 // the step size of this update depends on the step counter only
    if (f.parallel()) {
      f.edge(f.main, f.c);
      if (int e = adam_prep_early(*adam, f.c)) return e;
      adam->prep_ready = f.take();
      cudaEventRecord(adam->prep_ready, f.c);
      f.adam = adam;
    }
  }
  if (int e = enc_fwd_tc_run(m, theta, ids, M, Tcap, enc_ws, rep, dropout_rate, seed, d_step, f)) return e;
  if (int e = enc_scatter_plan_run(m, M, Tcap, enc_ws, bwd_ws, f)) return e;
  if (int e = loss_tc_run(m, theta, rep, a, loss_ws, loss, row_loss, d_rep, grad, f, 2)) return e;
  if (int e = enc_bwd_tc_run(m, theta, ids, M, Tcap, enc_ws, bwd_ws, d_rep, grad, dropout_rate, seed, d_step, f)) return e;
  // close the DAG: every side stream is ordered before the tail of the caller's stream
  f.edge(f.a, st);
  f.edge(f.b, st);
  f.edge(f.c, st);
  f.edge(f.wg[1], st);
  f.edge(f.wg[2], st);
  ADER_CHECK_LAUNCH("train step");
  if (adam && !f.adam)        // serial plan: the ordinary optimiser call behind the pass
    return ader_adam_step(m, adam->theta, adam->m, adam->v, adam->grad, adam->state, &adam->a, (void*)st);
  return 0;
}

extern "C" int32_t ader_train_fwd_bwd_tc(const AderModel* m, const float* theta, const int32_t* ids, int32_t M, int32_t Tcap,
                                         const AderLossArgs* a, void* enc_ws, void* bwd_ws, void* loss_ws, float* rep,
                                         float* loss, float* row_loss, float* d_rep, float* grad, float dropout_rate,
                                         uint64_t seed, const int32_t* d_step, int32_t serial, void* stream) {
  return run_step(m, theta, ids, M, Tcap, a, enc_ws, bwd_ws, loss_ws, rep, loss, row_loss, d_rep, grad, dropout_rate, seed,
                  d_step, serial, (cudaStream_t)stream, nullptr, "train_fwd_bwd_tc");
}

extern "C" int32_t ader_train_step_tc(const AderModel* m, float* theta, const int32_t* ids, int32_t M, int32_t Tcap,
                                      const AderLossArgs* a, void* enc_ws, void* bwd_ws, void* loss_ws, float* rep,
                                      float* loss, float* row_loss, float* d_rep, float* grad, float dropout_rate,
                                      uint64_t seed, const int32_t* d_step, float* adam_m, float* adam_v, int32_t* state,
                                      const AderAdamArgs* opt, int32_t serial, void* stream) {
  ADER_CHECK_ARG(m && adam_m && adam_v && state && opt, "train_step_tc: NULL pointer");
  ADER_CHECK_ARG(opt->V >= 1 && opt->V < m->v_tab, "train_step_tc: max_item %d outside table", opt->V);
  ADER_CHECK_ARG(opt->ewc_lambda == 0.f || (opt->fisher && opt->theta_star), "train_step_tc: EWC needs fisher and theta_star");
  AdamPlan plan;
  plan.theta = theta; plan.m = adam_m; plan.v = adam_v; plan.grad = grad; plan.state = state; plan.a = *opt; plan.prep_ready = nullptr;
  return run_step(m, theta, ids, M, Tcap, a, enc_ws, bwd_ws, loss_ws, rep, loss, row_loss, d_rep, grad, dropout_rate, seed,
                  d_step, serial, (cudaStream_t)stream, &plan, "train_step_tc");
}
