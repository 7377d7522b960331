// Shared host/device helpers for libader_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <math.h>
#include <atomic>
#include "../../include/ader_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libader_b200 is written for sm_100a (B200) only"
#endif

namespace ader {

int fail(int code, const char* fmt, ...);

#define ADER_CHECK_ARG(cond, ...) do { if (!(cond)) return ::ader::fail(-1, __VA_ARGS__); } while (0)
#define ADER_CHECK_LAUNCH(name) do { cudaError_t e__ = cudaGetLastError(); \
    if (e__ != cudaSuccess) return ::ader::fail(-3, "%s: %s", name, cudaGetErrorString(e__)); } while (0)

// Prepares kernel K for launches on the current device: 0, or -3 with a message naming the kernel.  The first call per
// (kernel, device) sets K's dynamic shared-memory limit to smem_bytes (0 for a kernel that only needs its module loaded
// before the first launch), which also loads K's module; later calls cost one cudaGetDevice and one atomic load, so a
// stream capture after an eager first call reaches no other CUDA call.  Kernel attributes are per device.  Every caller
// of one K passes the same smem_bytes, so threads racing on the first call set the same value.
template <auto K>
int kernel_ready(int smem_bytes, const char* name) {
  static std::atomic<uint64_t> ready{0};                 // bit i: prepared on device i
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(-3, "%s: no current device: %s", name, cudaGetErrorString(e));
  }
  if (dev >= 64) return fail(-3, "%s: device %d is beyond the 64 the library serves", name, dev);
  const uint64_t bit = 1ull << dev;
  if (ready.load(std::memory_order_acquire) & bit) return 0;
  e = cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(-3, "%s: cannot reserve %d B of shared memory on device %d: %s", name, smem_bytes, dev, cudaGetErrorString(e));
  }
  ready.fetch_or(bit, std::memory_order_release);
  return 0;
}

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }
static inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

// ---- flat parameter layout (SURVEY A.2, EWC.py:90) ----------------------------------------
struct Layout {
  int v_tab, d, L, nb, nh;
  long long off_table, off_pos, off_blocks, block_size, off_lnf, total;
  // offsets inside one block
  long long ln1b, ln1g, wq, bq, wk, bk, wv, bv, ln2b, ln2g, w1, b1, w2, b2;
  __host__ __device__ long long block(int b) const { return off_blocks + (long long)b * block_size; }
  long long dense_count() const { return total - off_pos; }
};

static inline Layout make_layout(const AderModel* m) {
  Layout l;
  l.v_tab = m->v_tab; l.d = m->d; l.L = m->maxlen; l.nb = m->num_blocks; l.nh = m->num_heads;
  long long d = m->d, dd = d * d;
  l.off_table = 0;
  l.off_pos = (long long)m->v_tab * d;
  l.off_blocks = l.off_pos + (long long)m->maxlen * d;
  l.ln1b = 0; l.ln1g = d; l.wq = 2 * d; l.bq = 2 * d + dd; l.wk = 3 * d + dd; l.bk = 3 * d + 2 * dd;
  l.wv = 4 * d + 2 * dd; l.bv = 4 * d + 3 * dd; l.ln2b = 5 * d + 3 * dd; l.ln2g = 6 * d + 3 * dd;
  l.w1 = 7 * d + 3 * dd; l.b1 = 7 * d + 4 * dd; l.w2 = 8 * d + 4 * dd; l.b2 = 8 * d + 5 * dd;
  l.block_size = 9 * d + 5 * dd;
  l.off_lnf = l.off_blocks + (long long)m->num_blocks * l.block_size;
  l.total = l.off_lnf + 2 * d;
  return l;
}

static inline int check_model(const AderModel* m) {
  if (!m) return fail(-1, "model is NULL");
  if (m->d <= 0 || m->d > 256 || m->d % 2) return fail(-1, "hidden_units must be even and <= 256 (got %d)", m->d);
  if (m->maxlen <= 0 || m->maxlen > 64) return fail(-1, "maxlen must be in 1..64 (got %d)", m->maxlen);
  if (m->num_heads <= 0 || m->d % m->num_heads) return fail(-1, "num_heads must divide hidden_units");
  if (m->num_blocks <= 0 || m->num_blocks > 8) return fail(-1, "num_blocks must be in 1..8");
  if (m->v_tab < 2) return fail(-1, "v_tab must be >= 2");
  return 0;
}

// ---- shape limits of the kernel paths (ader_path_check) ----------------------------------------
// The exact attention kernels (encoder.cu) hold one whole session row per CTA in shared memory: K^T and V^T
// [d][LP] plus the row's queries (forward) or Q, K, dY and the [L][LP] score tiles (backward).
constexpr int ATT_THREADS = 256, ATT_WARPS = 8;
__host__ __device__ inline int att_lp(int L) { return (L + 3) / 4 * 4; }
__host__ __device__ inline int al4(int x) { return (x + 3) & ~3; }
constexpr size_t ATTN_FWD_SMEM_MAX = 200 * 1024, ATTN_BWD_SMEM_MAX = 220 * 1024;
static inline size_t attn_fwd_smem(int d, int L) {
  return sizeof(float) * (2 * (size_t)d * att_lp(L) + (size_t)al4(L * d) + ATT_WARPS * 256);
}
static inline size_t attn_bwd_smem(int d, int L) {
  return sizeof(float) * (2 * (size_t)d * att_lp(L) + 3 * (size_t)al4(L * d) + 3 * (size_t)L * att_lp(L));
}
// widest model of the fused encoder, the tcgen05 loss / evaluation and the on-chip herding (operands padded to 160 columns)
constexpr int PATH_TC_MAX_D = 160;
// 0 if `path` (ADER_PATH_*) serves the (already checked) model, else -1; the message is set only when `report`
int path_check(const AderModel* m, int path, bool report = true);

// The fields of AderLossArgs (a != NULL), as every logits + CE + distillation entry takes them.  The teacher of a
// distillation (mode 1) call is stored logits (`teacher`) or a frozen snapshot (`teacher_rep` + the table the entry reads:
// fp32 rows for the exact entry, the bf16 shadow for the tcgen05 ones `tc`) -- exactly one of the two.
static inline int check_loss_args(const AderModel* m, const AderLossArgs* a, const char* who, bool tc) {
  if (a->M != a->n_train + a->n_ex || a->M <= 0)
    return fail(-1, "%s: M (%d) != n_train + n_ex (%d + %d)", who, a->M, a->n_train, a->n_ex);
  if (a->V < 1 || a->V >= m->v_tab) return fail(-1, "%s: max_item %d outside table of %d rows", who, a->V, m->v_tab);
  if (a->mode < 0 || a->mode > 2) return fail(-1, "%s: bad mode %d", who, a->mode);
  if (a->n_train > 0 && !a->pos) return fail(-1, "%s: pos is NULL", who);
  if (a->n_ex <= 0) return 0;
  if (a->mode == 0) return fail(-1, "%s: exemplar rows given in vanilla mode", who);
  if (a->mode == 2 && !a->ex_pos) return fail(-1, "%s: exemplar_pos is NULL", who);
  if (a->mode != 1) return 0;
  const bool stored = a->teacher != nullptr, frozen = a->teacher_rep != nullptr;
  if (stored == frozen)
    return fail(-1, "%s: mode 1 takes exactly one teacher source: teacher (stored logits) or teacher_rep (frozen snapshot)", who);
  if (a->V_prev < 1 || a->V_prev > a->V) return fail(-1, "%s: bad teacher (V_prev=%d, V=%d)", who, a->V_prev, a->V);
  if (stored && a->teacher_ld < a->V_prev) return fail(-1, "%s: bad teacher (teacher_ld %lld < V_prev %d)", who, (long long)a->teacher_ld, a->V_prev);
  if (frozen && !tc && !a->teacher_table) return fail(-1, "%s: frozen teacher without teacher_table", who);
  if (frozen && tc && !a->teacher_table16) return fail(-1, "%s: frozen teacher without teacher_table16 (see ader_pack_table16)", who);
  return 0;
}

// The arguments of the two log-sum-exp entries (ader_logsumexp, ader_logsumexp_tc): nll is written exactly when gt is given.
static inline int check_lse_args(const AderModel* m, const float* theta, const float* rep, const int32_t* gt, int R, int V,
                                 const void* ws, const float* lse, const float* nll, const char* who) {
  if (!theta) return fail(-1, "%s: theta is NULL", who);
  if (!rep) return fail(-1, "%s: rep is NULL", who);
  if (!ws) return fail(-1, "%s: ws is NULL", who);
  if (!lse) return fail(-1, "%s: lse is NULL", who);
  if (R <= 0) return fail(-1, "%s: R must be > 0 (got %d)", who, R);
  if (V < 1 || V >= m->v_tab) return fail(-1, "%s: V=%d outside the items 1..%d of the table", who, V, m->v_tab - 1);
  if (gt && !nll) return fail(-1, "%s: gt is given but nll is NULL", who);
  if (!gt && nll) return fail(-1, "%s: nll is given but gt is NULL", who);
  return 0;
}

// ---- programmatic dependent launch (PDL) -----------------------------------------------------------------
// Chain kernels call pdl_wait() before their first access to data of the preceding kernel (a no-op for a normal
// launch) and pdl_go() right behind it; launch_chain() sets the programmatic-stream-serialization attribute when
// `pdl` is on, so the next kernel's CTAs are scheduled and run their prologue (barrier init, bulk copies of the weight
// shadows, LayerNorm parameters) while the previous kernel drains.  ONLY kernels that call pdl_wait() may be launched
// through launch_chain(.., pdl = true).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_go() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_chain(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<Args&&>(args)...);
}

// ---- fork/join plan of one call (step.cu) -----------------------------------------------------
// The fused training entry (ader_train_fwd_bwd_tc) issues its launches as a DAG over a few internal
// streams: `main` carries the critical chain, a / b / c carry work that is off it (weight-shadow packing,
// teacher products, dE, weight gradients, position gradient, partial reductions).  With a == b == c == main
// every edge is a no-op and the launches are issued in the historical serial order, so the single-stream
// entry points run the very same code.  Under stream capture the side streams join the capture through
// the event edges and become parallel branches of the CUDA graph.
// one element of tf.train.AdamOptimizer (ADER.py:96; epsilon outside the bias correction) + EWC penalty gradient
// (EWC.py:115-124); the single definition both optimiser kernels evaluate
__device__ __forceinline__ void adam_update_elem(float g, float& th, float& m, float& v, float lr_t, float beta1, float beta2,
                                                 float eps, float ewc_lambda, float fisher, float theta_star) {
  // explicit rounding intrinsics: the compiler may not re-associate or contract differently in the two kernels
  if (ewc_lambda != 0.f) g = __fmaf_rn(__fmul_rn(ewc_lambda, fisher), __fsub_rn(th, theta_star), g);
  m = __fmaf_rn(beta1, m, __fmul_rn(__fsub_rn(1.f, beta1), g));
  v = __fmaf_rn(beta2, v, __fmul_rn(__fmul_rn(__fsub_rn(1.f, beta2), g), g));
  th = __fsub_rn(th, __fdiv_rn(__fmul_rn(lr_t, m), __fadd_rn(__fsqrt_rn(v), eps)));
}

// optimiser step folded into the fused training entry (single GPU: no gradient all-reduce between backward and Adam)
struct AdamPlan {
  float *theta, *m, *v; const float* grad; int32_t* state; AderAdamArgs a;
  cudaEvent_t prep_ready;       // bias-corrected step size of this step is in state[1]
};
int adam_prep_early(const AdamPlan& p, cudaStream_t st);                       // state[1] = lr_t(state[0] + 1); no increment
int adam_table_part(const AderModel* m, const AdamPlan& p, cudaStream_t st);   // item-table rows 1..V

// d_rep reduction folded into the final-LayerNorm backward (fused step only): the loss group hands its split partials over
// instead of launching k_reduce_drep; part is [n_chunks][rows_pad][kp] fp32, u the [.,kp] teacher term of the distillation rows
struct DrepFuse { const float* part; const float* u; int n_chunks, rows_pad, kp, u_row0, n_train; };

struct Fork {
  const AdamPlan* adam;
  cudaStream_t main, a, b, c;
  cudaStream_t wg[3];                      // the three weight-gradient pieces of a block run beside each other (wg[0] == a)
  cudaEvent_t* ev; int n_ev, next_ev;      // event pool (timing disabled); reuse is safe: every wait is issued right after its record
  cudaEvent_t table_ready;                 // recorded on `b` after the dE kernel: the scatter into the item table waits for it
  bool has_table_ready;
  cudaEvent_t tok_ready;                   // recorded on `main` once the packed token ids exist (the scatter plan needs only them)
  bool has_tok_ready;
  cudaEvent_t plan_ready;                  // recorded on `c` behind the scatter plan (sorted ids)
  bool plan_done;
  bool pdl;                                // launch the kernel-to-kernel chain links of `main` as programmatic dependent launches
  bool fuse_drep, has_drep;                // fused step: the d_rep partials are summed by the final-LayerNorm backward kernel
  DrepFuse drep;
  static Fork serial(cudaStream_t st) {
    Fork f; f.main = f.a = f.b = f.c = st; f.wg[0] = f.wg[1] = f.wg[2] = st; f.ev = nullptr; f.n_ev = f.next_ev = 0; f.pdl = false; f.adam = nullptr;
    f.fuse_drep = f.has_drep = false; f.drep = DrepFuse();
    f.table_ready = f.tok_ready = f.plan_ready = nullptr; f.has_table_ready = f.has_tok_ready = f.plan_done = false;
    return f;
  }
  bool parallel() const { return a != main; }
  cudaEvent_t take() { cudaEvent_t e = ev[next_ev % n_ev]; ++next_ev; return e; }
  // work launched on `to` after this call also waits for everything launched on `from` before it
  void edge(cudaStream_t from, cudaStream_t to) {
    if (from == to) return;
    cudaEvent_t e = take();
    cudaEventRecord(e, from);
    cudaStreamWaitEvent(to, e, 0);
  }
};

// internal forms of the tensor-core entry points (encoder.cu / logits_tc.cu), shared with step.cu
int enc_fwd_tc_run(const AderModel* m, const float* theta, const int32_t* ids, int M, int Tcap, void* ws, float* rep,
                   float dropout_rate, uint64_t seed, const int32_t* d_step, Fork& f);
int enc_bwd_tc_run(const AderModel* m, const float* theta, const int32_t* ids, int M, int Tcap, const void* ws, void* bwd_ws,
                   const float* d_rep, float* grad, float dropout_rate, uint64_t seed, const int32_t* d_step, Fork& f);
// the scatter's sort of (item id, token) pairs on f.c, as soon as the token ids are packed (parallel plans only)
int enc_scatter_plan_run(const AderModel* m, int M, int Tcap, const void* ws, void* bwd_ws, Fork& f);
// phase 0: everything that does not need `rep` (table tiles, teacher statistics / tiles, uc partials) on f.b;
// phase 1: the rest (rep tiles, forward statistics, loss, d_rep on f.main; dE on f.b)
int loss_tc_run(const AderModel* m, const float* theta, const float* rep, const AderLossArgs* a, void* ws, float* loss,
                float* row_loss, float* d_rep, float* grad, Fork& f, int phase_mask);

// ---- generic fp32 GEMM (sgemm.cu) ----------------------------------------------------------
// C(m,n) = epilogue( sum_k A(m,k) * B(k,n) ), element (i,j) of X at X[i*rs + j*cs].
struct GemmArgs {
  const float* A; long long a_rs, a_cs;
  const float* B; long long b_rs, b_cs;
  float* C; long long c_rs, c_cs;
  int M, N, K;
  const int* dM;          // optional device override of M (token count)
  const int* dK;          // optional device override of K
  const float* bias;      // [N] added per column (or NULL)
  const float* resid;     // [M,N] row-major (ld = resid_ld) added (or NULL)
  long long resid_ld;
  const float* relu_mask; // [M,N] row-major (ld = mask_ld): out *= (mask > 0)  (or NULL)
  long long mask_ld;
  int relu;               // out = max(out, 0)
  int accumulate;         // C += out instead of C = out
  float alpha;
  int splits;             // split-K: grid.z; split z writes C + z*split_stride, k-range chunked
  long long split_stride;
  float* colsum;          // optional [N] (+ z*split_stride): column sums of B over this split's k-range
  // dropout applied to the epilogue output (after relu), tf.layers.dropout semantics
  float drop_p; uint64_t drop_seed; uint32_t drop_site;
};
void gemm_defaults(GemmArgs& g);
int launch_gemm(const GemmArgs& g, cudaStream_t st);

// ---- counter-based dropout mask (shared by fwd and bwd) -----------------------------------
// u = fmix32(idx ^ key(seed, site)) / 2^24: a stateless 32-bit hash (murmur3 finaliser) of the element index,
// keyed per (seed + step, site).  ~10 integer instructions per element; key terms are loop invariant.
__host__ __device__ inline uint32_t fmix32(uint32_t h) {
  h ^= h >> 16; h *= 0x85ebca6bu; h ^= h >> 13; h *= 0xc2b2ae35u; h ^= h >> 16;
  return h;
}
// Dropout site: everything that does not depend on the element (hash key of (seed, site), integer drop threshold,
// keep scale 1/(1-p)) is computed ONCE; drop_mul() is then one 32-bit mix, a compare and a select per element.
// u = (r >> 8) * 2^-24 < p  <=>  (r >> 8) < ceil(p * 2^24)   (both sides exact in fp32).
struct DropSite { uint32_t key, thr; float keep; };
__host__ __device__ inline DropSite drop_site(uint64_t seed, uint32_t site, float p) {
  DropSite s;
  s.key = fmix32((uint32_t)seed * 0x9E3779B1u + (uint32_t)(seed >> 32) * 0x7FEB352Du + site * 0x846CA68Bu + 0x5bd1e995u);
  s.thr = p > 0.f ? (uint32_t)ceilf(p * 16777216.0f) : 0u;
  s.keep = 1.0f / (1.0f - p);
  return s;
}
// multiplier (0 or 1/(1-p)) for element `idx` of the site
__host__ __device__ inline float drop_mul(const DropSite& s, uint64_t idx) {
  const uint32_t r = fmix32(((uint32_t)idx ^ s.key) + (uint32_t)(idx >> 32) * 0x27d4eb2fu);
  return (r >> 8) < s.thr ? 0.0f : s.keep;
}
__host__ __device__ inline float drop_scale(uint64_t seed, uint32_t site, uint64_t idx, float p) {
  return drop_mul(drop_site(seed, site, p), idx);
}

}  // namespace ader
