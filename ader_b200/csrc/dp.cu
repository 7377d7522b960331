// Data-parallel optimiser step over NVLink peer memory (SURVEY 8e; the reference is single-device:
// main.py:96,120,143, so everything here is new).
//
// One process per GPU; every rank holds a full replica of theta and its own gradient of the step
// (rows of the batch are sharded, loss denominators are the GLOBAL counts, so the wanted gradient is
// the plain SUM over ranks).  Instead of  all-reduce(grad) -> Adam on every rank  (2 x 7/8 of the
// gradient over the links AND the full 28 B/param optimiser traffic on every GPU), ONE kernel does
//
//     reduce-scatter (peer loads)  ->  TF1 Adam on the owned slice  ->  all-gather (peer stores)
//
// Rank r owns a contiguous slice of the update index space [item-table rows 1..V | dense parameters]
// (the same index space k_adam walks).  For its slice it loads the gradient of every rank over NVLink
// (ld.global.cv: peer lines must not be served from a stale L1), adds them in rank order 0..N-1
// (fixed order: run-to-run deterministic, and every replica receives the same bits), applies
// adam_update_elem (the very expression the single-GPU kernels evaluate) with its LOCAL m / v --
// the optimiser state of a slice is only ever touched by its owner -- and stores the new theta
// into every replica.  Link traffic per GPU and step: (N-1)/N of the gradient in, (N-1)/N of theta out.
//
// Synchronisation (no host, graph-capturable): a flag block per rank in peer-mapped memory,
//   flags[src] (src < N): arrival counter written by rank `src` (monotonic epoch numbers),
//   EPOCH: this rank's epoch (2 per step), DONE: CTA completion counter, ERR: timeout marker.
// k_dp_arrive (one warp, directly in front of k_dp_adam): publishes "my gradient is complete" (epoch e+1) to every
// rank and waits until all ranks have published (A); it also prepares the bias-corrected step size.  k_dp_adam works;
// k_dp_publish (one warp, directly behind it: the kernel boundary orders every peer load / store of the update before
// it) publishes e+2 = "I have read your gradients and written your theta" (B).  ader_dp_wait (first kernel of the next
// step) waits for B from every rank before anything overwrites the gradient or reads theta.  Only single-warp kernels
// ever spin (they leave the SMs to whatever the other ranks still have to run -- also when several emulated ranks share
// one GPU in the tests); spins time out (~20 s) and mark ERR instead of hanging the GPU.
#include "common.cuh"
#include <string.h>
#include <stdlib.h>

namespace ader {
namespace dp {

constexpr int F_EPOCH = 32, F_DONE = 33, F_ERR = 34, F_LR = 35;

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float2 ld_cv2(const float* p) {
  float2 v;
  asm volatile("ld.global.cv.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p));
  return v;
}
__device__ __forceinline__ unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ uint32_t ld_relaxed_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// wait until flags[src] >= want (signed distance: epochs wrap after 2^31 steps); false on timeout.  The poll itself is a
// relaxed load of LOCAL memory (the peer wrote the flag over the link); one acquire fence follows the successful poll
// (an acquire load per poll and a 64 ns sleep made each cross-GPU barrier cost ~10 us, measured with the peer traffic off).
__device__ __forceinline__ bool wait_flag(const uint32_t* f, uint32_t want, uint32_t* err) {
  if ((int32_t)(ld_relaxed_sys(f) - want) < 0) {
    const unsigned long long t0 = gtime();
    unsigned spins = 0;
    while ((int32_t)(ld_relaxed_sys(f) - want) < 0) {
      if ((++spins & 1023u) == 0 && gtime() - t0 > 20000000000ull) { atomicExch(err, 1u); return false; }
    }
  }
  asm volatile("fence.acq_rel.sys;" ::: "memory");
  return true;
}

struct DpFlags {
  int rank, world;
  uint32_t* flags[ADER_DP_MAX_RANKS];
};

struct DpArgs {
  int rank, world;
  float* theta[ADER_DP_MAX_RANKS];
  const float* grad[ADER_DP_MAX_RANKS];
  uint32_t* flags[ADER_DP_MAX_RANKS];
  float *m, *v;
  int* state;
  // update index space = two element ranges (item-table rows 1..V, dense parameters), walked in QUADS of four
  // floats so that peer traffic moves in 16-byte accesses.  A range starts on an even element; when its byte offset is
  // 8 mod 16 the first quad holds only its upper float2 (ph = 1), and a range may end with a half quad.
  long long e0[2];            // first element of the range
  long long n2[2];            // float2 units in the range
  int ph[2];                  // 1: unit 0 sits in the upper half of quad 0
  long long q0[2];            // first global quad of the range (q0[0] = 0), q_total = all quads
  long long q_lo, q_hi;       // quads owned by this rank
  float lr, beta1, beta2, eps, ewc_lambda;
  const float *fisher, *theta_star;
  float* mc_theta;            // NVLS multicast views of theta / grad (k_dp_adam_mc), else NULL
  const float* mc_grad;
};

__device__ __forceinline__ float4 ld_cg4(const float* p) {
  float4 v;
  asm volatile("ld.global.cg.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ float2 ld_cg2(const float* p) {
  float2 v;
  asm volatile("ld.global.cg.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p));
  return v;
}

// W = upper bound of the world size (array extents in registers), U = quads per thread and trip: U * W peer loads of
// 16 bytes are in flight per thread before the first add (NVLink round trips are ~2-3 us: the link only fills with
// megabytes outstanding, and only with 16-byte accesses -- 8-byte ones reached ~150 GB/s per direction).
// Peer lines are never in this SM's L1 at kernel start (L1 is invalidated at launch boundaries) and .cg keeps them out.
// One quad (four floats, 16-byte peer accesses) per thread, launched like the single-GPU Adam kernel: tens of thousands of
// resident threads keep megabytes of peer loads in flight (NVLink round trips are 2-3 us), and there is NO in-kernel
// completion protocol -- a first version closed with a system fence + ticket per CTA and ran 2x slower than plain Adam on
// purely local data; now the kernel boundary is the fence and k_dp_publish (one warp, stream-ordered behind this kernel)
// announces "read your gradients, wrote your theta".  W = upper bound of the world size (register array extents).
template <int W>
__global__ void __launch_bounds__(256) k_dp_adam(DpArgs a) {
  const long long q = a.q_lo + (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= a.q_hi) return;
  const float lr_t = __uint_as_float(ld_relaxed_sys(a.flags[a.rank] + F_LR));       // prepared by k_dp_arrive
  const int s = q >= a.q0[1] ? 1 : 0;
  const long long u0 = 2 * (q - a.q0[s]) - a.ph[s];                 // float2 unit of the quad's lower half
  const long long el = a.e0[s] + 2 * u0;                            // 16-byte aligned element
  const int msk = ((u0 >= 0) ? 1 : 0) | ((u0 + 1 < a.n2[s]) ? 2 : 0);
  float4 gr[W];
#pragma unroll
  for (int r = 0; r < W; ++r) {
    if (r < a.world) {
      if (msk == 3) gr[r] = ld_cg4(a.grad[r] + el);
      else {
        const float2 h = ld_cg2(a.grad[r] + el + (msk == 2 ? 2 : 0));
        gr[r] = (msk == 2) ? make_float4(0.f, 0.f, h.x, h.y) : make_float4(h.x, h.y, 0.f, 0.f);
      }
    }
  }
  const int lo = (msk & 1) ? 0 : 2, hi = (msk & 2) ? 4 : 2;
  float th[4], m[4], v[4], f[4] = {0.f, 0.f, 0.f, 0.f}, ts[4] = {0.f, 0.f, 0.f, 0.f};
  const bool ewc = a.ewc_lambda != 0.f;
#pragma unroll
  for (int h = 0; h < 4; h += 2) {
    if (h < lo || h >= hi) continue;
    const long long x = el + h;
    const float2 t2 = *reinterpret_cast<const float2*>(a.theta[a.rank] + x);
    const float2 m2 = *reinterpret_cast<const float2*>(a.m + x);
    const float2 v2 = *reinterpret_cast<const float2*>(a.v + x);
    th[h] = t2.x; th[h + 1] = t2.y; m[h] = m2.x; m[h + 1] = m2.y; v[h] = v2.x; v[h + 1] = v2.y;
    if (ewc) {
      const float2 f2 = *reinterpret_cast<const float2*>(a.fisher + x);
      const float2 s2 = *reinterpret_cast<const float2*>(a.theta_star + x);
      f[h] = f2.x; f[h + 1] = f2.y; ts[h] = s2.x; ts[h + 1] = s2.y;
    }
  }
  float g[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int r = 0; r < W; ++r)
    if (r < a.world) {                                                    // rank order: deterministic
      g[0] = __fadd_rn(g[0], gr[r].x); g[1] = __fadd_rn(g[1], gr[r].y);
      g[2] = __fadd_rn(g[2], gr[r].z); g[3] = __fadd_rn(g[3], gr[r].w);
    }
#pragma unroll
  for (int h = 0; h < 4; h += 2) {
    if (h < lo || h >= hi) continue;
    const long long x = el + h;
    adam_update_elem(g[h], th[h], m[h], v[h], lr_t, a.beta1, a.beta2, a.eps, a.ewc_lambda, f[h], ts[h]);
    adam_update_elem(g[h + 1], th[h + 1], m[h + 1], v[h + 1], lr_t, a.beta1, a.beta2, a.eps, a.ewc_lambda, f[h + 1], ts[h + 1]);
    *reinterpret_cast<float2*>(a.m + x) = make_float2(m[h], m[h + 1]);
    *reinterpret_cast<float2*>(a.v + x) = make_float2(v[h], v[h + 1]);
  }
#pragma unroll
  for (int r = 0; r < W; ++r) {
    if (r >= a.world) continue;
    if (msk == 3) *reinterpret_cast<float4*>(a.theta[r] + el) = make_float4(th[0], th[1], th[2], th[3]);
    else *reinterpret_cast<float2*>(a.theta[r] + el + lo) = make_float2(th[lo], th[lo + 1]);
  }
}

// ---- NVLS variant: the NVSwitch sums and broadcasts ------------------------------------------------------------------
// `mc_grad` / `mc_theta` are multicast addresses bound to every rank's gradient / parameter buffer.  One
// multimem.ld_reduce.add returns the sum of the quad over all ranks (added inside the switch: this rank receives 16 bytes
// instead of 16 x world), one multimem.st delivers the new quad to every replica (sent once instead of world times), so the
// NVLink traffic per rank is 2 x its slice whatever the world size.  The owner still computes and everyone receives the
// same bits, so replicas stay bit-identical; the order of the in-switch sum is the switch's, not rank order.
__device__ __forceinline__ float4 mm_ld_sum4(const float* p) {
  float4 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float2 mm_ld_sum2(const float* p) {
  float2 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void mm_st4(float* p, float a, float b, float c, float d) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ void mm_st2(float* p, float a, float b) {
  asm volatile("multimem.st.relaxed.sys.global.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(a), "f"(b) : "memory");
}

__global__ void __launch_bounds__(256) k_dp_adam_mc(DpArgs a) {
  const long long q = a.q_lo + (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= a.q_hi) return;
  const float lr_t = __uint_as_float(ld_relaxed_sys(a.flags[a.rank] + F_LR));
  const int s = q >= a.q0[1] ? 1 : 0;
  const long long u0 = 2 * (q - a.q0[s]) - a.ph[s];
  const long long el = a.e0[s] + 2 * u0;
  const int msk = ((u0 >= 0) ? 1 : 0) | ((u0 + 1 < a.n2[s]) ? 2 : 0);
  float g[4] = {0.f, 0.f, 0.f, 0.f};
  if (msk == 3) { const float4 t = mm_ld_sum4(a.mc_grad + el); g[0] = t.x; g[1] = t.y; g[2] = t.z; g[3] = t.w; }
  else {
    const int o = (msk == 2) ? 2 : 0;
    const float2 t = mm_ld_sum2(a.mc_grad + el + o);
    g[o] = t.x; g[o + 1] = t.y;
  }
  const int lo = (msk & 1) ? 0 : 2, hi = (msk & 2) ? 4 : 2;
  float th[4] = {0.f, 0.f, 0.f, 0.f};
  const bool ewc = a.ewc_lambda != 0.f;
#pragma unroll
  for (int h = 0; h < 4; h += 2) {
    if (h < lo || h >= hi) continue;
    const long long x = el + h;
    const float2 t2 = *reinterpret_cast<const float2*>(a.theta[a.rank] + x);
    float2 m2 = *reinterpret_cast<const float2*>(a.m + x);
    float2 v2 = *reinterpret_cast<const float2*>(a.v + x);
    float2 f2 = make_float2(0.f, 0.f), s2 = make_float2(0.f, 0.f);
    if (ewc) { f2 = *reinterpret_cast<const float2*>(a.fisher + x); s2 = *reinterpret_cast<const float2*>(a.theta_star + x); }
    th[h] = t2.x; th[h + 1] = t2.y;
    adam_update_elem(g[h], th[h], m2.x, v2.x, lr_t, a.beta1, a.beta2, a.eps, a.ewc_lambda, f2.x, s2.x);
    adam_update_elem(g[h + 1], th[h + 1], m2.y, v2.y, lr_t, a.beta1, a.beta2, a.eps, a.ewc_lambda, f2.y, s2.y);
    *reinterpret_cast<float2*>(a.m + x) = m2;
    *reinterpret_cast<float2*>(a.v + x) = v2;
  }
  if (msk == 3) mm_st4(a.mc_theta + el, th[0], th[1], th[2], th[3]);
  else mm_st2(a.mc_theta + el + lo, th[lo], th[lo + 1]);
}

// B: stream order puts every load / store of k_dp_adam before this kernel (the kernel boundary is the system-wide fence)
__global__ void k_dp_publish(DpFlags a, int* state) {
  uint32_t* myf = a.flags[a.rank];
  const uint32_t e = ld_relaxed_sys(myf + F_EPOCH);
  if (threadIdx.x == 0) {
    state[0] = state[0] + 1;
    state[1] = (int)ld_relaxed_sys(myf + F_LR);
    st_release_sys(myf + F_EPOCH, e + 2);
  }
  if ((int)threadIdx.x < a.world) st_release_sys(a.flags[threadIdx.x] + a.rank, e + 2);
}

// A: stream order puts every gradient write of this rank before this kernel
__global__ void k_dp_arrive(DpFlags a, const int* state, float lr, float beta1, float beta2) {
  uint32_t* myf = a.flags[a.rank];
  const uint32_t e = ld_acquire_sys(myf + F_EPOCH);
  if (threadIdx.x == 31) {                             // bias-corrected step size of this update (TF1 Adam), off the waiting lanes
    const int t = state[0] + 1;
    const double lr_t = (double)lr * sqrt(1.0 - pow((double)beta2, (double)t)) / (1.0 - pow((double)beta1, (double)t));
    myf[F_LR] = __float_as_uint((float)lr_t);
  }
  if ((int)threadIdx.x < a.world) {
    st_release_sys(a.flags[threadIdx.x] + a.rank, e + 1);       // kernel boundary: the gradient is already in device memory
    wait_flag(myf + threadIdx.x, e + 1, myf + F_ERR);
  }
}

__global__ void k_dp_wait(int rank, int world, uint32_t* myf) {
  const uint32_t e = ld_acquire_sys(myf + F_EPOCH);
  if ((int)threadIdx.x < world) wait_flag(myf + threadIdx.x, e, myf + F_ERR);
}

}  // namespace dp
}  // namespace ader

using namespace ader;
using namespace ader::dp;

// CUDA loads kernels lazily, and a first-use load may wait for the context to drain: it must not happen while an
// arrive kernel is already spinning (several emulated ranks in one process would stall until the timeout), so
// every kernel of this file is loaded on the device before the first launch of any of them.
static int check_comm(const AderDpComm* c) {
  ADER_CHECK_ARG(c, "dp: comm is NULL");
  ADER_CHECK_ARG(c->world >= 1 && c->world <= ADER_DP_MAX_RANKS && c->rank >= 0 && c->rank < c->world, "dp: bad rank %d / world %d", c->rank, c->world);
  for (int r = 0; r < c->world; ++r) ADER_CHECK_ARG(c->theta[r] && c->grad[r] && c->flags[r], "dp: NULL pointer for rank %d", r);
  if (int e = kernel_ready<k_dp_adam<2>>(0, "k_dp_adam<2>")) return e;
  if (int e = kernel_ready<k_dp_adam<4>>(0, "k_dp_adam<4>")) return e;
  if (int e = kernel_ready<k_dp_adam<8>>(0, "k_dp_adam<8>")) return e;
  if (int e = kernel_ready<k_dp_adam<16>>(0, "k_dp_adam<16>")) return e;
  if (int e = kernel_ready<k_dp_adam_mc>(0, "k_dp_adam_mc")) return e;
  if (int e = kernel_ready<k_dp_publish>(0, "k_dp_publish")) return e;
  if (int e = kernel_ready<k_dp_arrive>(0, "k_dp_arrive")) return e;
  return kernel_ready<k_dp_wait>(0, "k_dp_wait");
}

extern "C" int32_t ader_dp_wait(const AderDpComm* c, void* stream) {
  if (int e = check_comm(c)) return e;
  k_dp_wait<<<1, 32, 0, (cudaStream_t)stream>>>(c->rank, c->world, c->flags[c->rank]);
  ADER_CHECK_LAUNCH("dp_wait");
  return 0;
}

extern "C" int32_t ader_dp_adam_step(const AderModel* m, const AderDpComm* c, float* adam_m, float* adam_v, int32_t* state,
                                     const AderAdamArgs* a, void* stream) {
  if (int e = check_model(m)) return e;
  if (int e = check_comm(c)) return e;
  ADER_CHECK_ARG(adam_m && adam_v && state && a, "dp_adam_step: NULL pointer");
  ADER_CHECK_ARG(a->V >= 1 && a->V < m->v_tab, "dp_adam_step: max_item %d outside table", a->V);
  ADER_CHECK_ARG(a->ewc_lambda == 0.f || (a->fisher && a->theta_star), "dp_adam_step: EWC needs fisher and theta_star");
  const Layout l = make_layout(m);
  DpArgs d;
  d.rank = c->rank; d.world = c->world;
  for (int r = 0; r < ADER_DP_MAX_RANKS; ++r) {
    d.theta[r] = r < c->world ? c->theta[r] : nullptr;
    d.grad[r] = r < c->world ? c->grad[r] : nullptr;
    d.flags[r] = r < c->world ? c->flags[r] : nullptr;
  }
  d.m = adam_m; d.v = adam_v; d.state = state;
  // two element ranges, both starting and ending on even elements (d is even); quads are 16-byte aligned float4s
  const long long starts[2] = {(long long)m->d, l.off_pos};
  const long long counts[2] = {(long long)a->V * m->d, l.dense_count()};
  long long q = 0;
  for (int s = 0; s < 2; ++s) {
    d.e0[s] = starts[s]; d.n2[s] = counts[s] / 2;
    d.ph[s] = (int)((starts[s] / 2) & 1);                    // byte offset 8 mod 16 <=> odd float2 index
    d.q0[s] = q;
    q += (d.n2[s] + d.ph[s] + 1) / 2;
  }
  const long long q_total = q;
  d.q_lo = q_total * c->rank / c->world;
  d.q_hi = q_total * (c->rank + 1) / c->world;
  d.lr = a->lr; d.beta1 = a->beta1; d.beta2 = a->beta2; d.eps = a->eps; d.ewc_lambda = a->ewc_lambda;
  d.fisher = a->fisher; d.theta_star = a->theta_star;
  d.mc_theta = c->mc_theta; d.mc_grad = c->mc_grad;
  ADER_CHECK_ARG((c->mc_theta == nullptr) == (c->mc_grad == nullptr), "dp_adam_step: mc_theta and mc_grad go together");
  ADER_CHECK_ARG(((uintptr_t)c->mc_theta % 16) == 0 && ((uintptr_t)c->mc_grad % 16) == 0, "dp_adam_step: multicast views must be 16-byte aligned");
  ADER_CHECK_ARG(((uintptr_t)adam_m % 16) == 0 && ((uintptr_t)adam_v % 16) == 0, "dp_adam_step: optimiser slots must be 16-byte aligned");
  for (int r = 0; r < c->world; ++r)
    ADER_CHECK_ARG(((uintptr_t)c->theta[r] % 16) == 0 && ((uintptr_t)c->grad[r] % 16) == 0, "dp_adam_step: theta / grad of rank %d must be 16-byte aligned", r);
  const long long mine = d.q_hi - d.q_lo;
  const int grid = cdiv(mine > 0 ? mine : 1, 256);
  DpFlags fl;
  fl.rank = c->rank; fl.world = c->world;
  for (int r = 0; r < ADER_DP_MAX_RANKS; ++r) fl.flags[r] = d.flags[r];
  cudaStream_t st = (cudaStream_t)stream;
  k_dp_arrive<<<1, 32, 0, st>>>(fl, state, a->lr, a->beta1, a->beta2);
  if (c->mc_theta) k_dp_adam_mc<<<grid, 256, 0, st>>>(d);
  else if (c->world <= 2) k_dp_adam<2><<<grid, 256, 0, st>>>(d);
  else if (c->world <= 4) k_dp_adam<4><<<grid, 256, 0, st>>>(d);
  else if (c->world <= 8) k_dp_adam<8><<<grid, 256, 0, st>>>(d);
  else k_dp_adam<16><<<grid, 256, 0, st>>>(d);
  k_dp_publish<<<1, 32, 0, st>>>(fl, state);
  ADER_CHECK_LAUNCH("dp_adam_step");
  return 0;
}

extern "C" int32_t ader_dp_status(const AderDpComm* c, int32_t* err_out, uint32_t* epoch_out) {
  if (int e = check_comm(c)) return e;
  uint32_t w[3] = {0, 0, 0};
  if (cudaMemcpy(w, c->flags[c->rank] + F_EPOCH, sizeof(w), cudaMemcpyDeviceToHost) != cudaSuccess)
    return fail(-3, "dp_status: %s", cudaGetErrorString(cudaGetLastError()));
  if (epoch_out) *epoch_out = w[0];
  if (err_out) *err_out = (int32_t)w[2];
  return 0;
}

// ---- CUDA IPC plumbing: map another process's device allocation (one process per GPU) -------------------
typedef int (*cuMemGetAddressRange_t)(unsigned long long*, size_t*, unsigned long long);

extern "C" int32_t ader_ipc_export(const void* dev_ptr, void* handle64, int64_t* offset) {
  ADER_CHECK_ARG(dev_ptr && handle64 && offset, "ipc_export: NULL pointer");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qr;
  if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &fn, cudaEnableDefault, &qr) != cudaSuccess || !fn)
    return fail(-3, "ipc_export: cuMemGetAddressRange unavailable");
  unsigned long long base = 0; size_t size = 0;
  if (((cuMemGetAddressRange_t)fn)(&base, &size, (unsigned long long)(uintptr_t)dev_ptr) != 0)
    return fail(-3, "ipc_export: not a device allocation");
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, (void*)(uintptr_t)base);
  if (e != cudaSuccess) { cudaGetLastError(); return fail(-3, "ipc_export: %s", cudaGetErrorString(e)); }
  memcpy(handle64, &h, 64);
  *offset = (int64_t)((unsigned long long)(uintptr_t)dev_ptr - base);
  return 0;
}

extern "C" int32_t ader_ipc_open(const void* handle64, void** base_ptr) {
  ADER_CHECK_ARG(handle64 && base_ptr, "ipc_open: NULL pointer");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  cudaError_t e = cudaIpcOpenMemHandle(base_ptr, h, cudaIpcMemLazyEnablePeerAccess);
  if (e != cudaSuccess) { cudaGetLastError(); return fail(-3, "ipc_open: %s", cudaGetErrorString(e)); }
  return 0;
}

extern "C" int32_t ader_ipc_close(void* base_ptr) {
  if (!base_ptr) return 0;
  cudaError_t e = cudaIpcCloseMemHandle(base_ptr);
  if (e != cudaSuccess) { cudaGetLastError(); return fail(-3, "ipc_close: %s", cudaGetErrorString(e)); }
  return 0;
}
