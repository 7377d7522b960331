// Fused tensor-core encoder (subsystem 1 of the north star): the SASRec blocks of modules.py:23-271 /
// ADER.py:25-85 over PACKED real tokens with 16-bit tensor-core operands and fp32 accumulation,
// forward and backward.  Operand type: IEEE fp16 with a per-row power-of-two scale (exactly undone in
// the epilogue) -- the same tensor-core rate and bytes as bf16 but 11 significand bits instead of 8, which
// matters here because parity with the fp32 reference is the first gate (measured: gradient error vs the fp32
// oracle 3-5 % rel-L2 with bf16 operands, see profiles/; the row scale removes fp16's range problem for
// gradients).  Included by encoder.cu (same translation unit: it shares the packing, LayerNorm,
// radix-sort and segmented-reduction kernels of the exact path).
//
// Why these shapes.  At the reference's batch sizes a step holds T ~ 2-6 k real tokens (8-10 % of
// the dense [M,50] grid), so every dense layer is a [T,150] x [150,150] product: ~0.2 GFLOP, far
// below what one launch costs.  The step is bound by launch count and by the dependent chain of small
// kernels, not by the math pipe, so the design is
//   * token tiles of 32 rows (T/32 ~ 110 CTAs spread over the 148 SMs; a 128-row tcgen05 tile
//     would leave 80 % of the SMs idle at these T) on warp-level mma.sync.m16n8k16 (fp16 operands, fp32 accumulate),
//   * the weight matrices as 16-bit shadows [n][k] (row stride 168 -> conflict-free 32-bit fragment
//     loads), one 53 760-byte contiguous block each, staged into shared memory by cp.async.bulk + mbarrier
//     (TMA bulk path) once per CTA, overlapped with the LayerNorm prologue,
//   * whole sub-layers fused in one kernel: [embed] + LN1 + Q/K/V projections; attention + residual +
//     LN2 (warp per query, straight from L1/L2: rows are 1-50 tokens); FFN1 + ReLU + FFN2 + residual;
//     and in backward FFN dgrad + LN2 backward; attention backward (warp per token, flash-style
//     D = gY.(Y - q) so no dS matrix is stored); Q/K/V dgrad + LN1 backward.
//   * weight / bias / LN-parameter gradients stay fp32 (grouped split-K SIMT GEMM over the 5 matrices of a
//     block in ONE launch, fixed reduction order -> deterministic).
// Saved activations stay fp32 in HBM in the same workspace slots as the exact path, so the two paths can
// be compared slot by slot (tests/test_gpu_parity.py).
#pragma once
#include <cuda_fp16.h>

namespace ader {
namespace fz {

using op_t = __half;                    // 16-bit operand type of the tiles and weight shadows
constexpr int KP = 160;                 // feature dim padded to a multiple of 16 (d <= 160 on this path)
constexpr int LDS = 168;                // row stride (op_t elements) of shared-memory operand tiles and weight shadows
constexpr int TM = 32;                  // token rows per tile
constexpr int NTHR = 256;               // 8 warps: (m-tile = warp & 1) x (column group = warp >> 1)
constexpr int NT = 5;                   // n8 tiles per warp (4 column groups x 5 x 8 = 160 columns)
constexpr int WMAT_BYTES = KP * LDS * 2;        // 53 760
constexpr int ATILE_BYTES = TM * LDS * 2;       // 10 752
constexpr int FT_LD = 168;              // row stride (floats) of fp32 staging tiles (168 % 32 == 8: conflict-free float2 stores)
constexpr int FTILE_BYTES = TM * FT_LD * 4;     // 21 504
constexpr int NE = 5;                   // features per lane in the warp-per-token kernels (32 x 5 = 160)

// effective dropout seed: host value + optional device-resident step counter (lets a captured CUDA graph draw
// fresh masks on every replay: the counter is the Adam step the optimiser kernel increments)
__device__ __forceinline__ uint64_t eff_seed(uint64_t seed, const int* d_step) {
  return seed + (d_step ? (uint64_t)(uint32_t)__ldg(d_step) : 0ull);
}

// Optional phase timeline (debug builds: -DADER_TC_TIMELINE): %globaltimer stamps by thread 0 of each CTA.
#ifdef ADER_TC_TIMELINE
__device__ long long g_fz_tl[8][160][16];
__device__ __forceinline__ void fz_tl(int k, int slot) {
  if (threadIdx.x == 0 && blockIdx.x < 160) { long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); g_fz_tl[k][blockIdx.x][slot] = t; }
}
#define FZ_TL(k, slot) fz_tl(k, slot)
#define FZ_TLV(k, slot, v) do { if (threadIdx.x == 0 && blockIdx.x < 160) g_fz_tl[k][blockIdx.x][slot] = (v); } while (0)
#else
#define FZ_TL(k, slot) do { } while (0)
#define FZ_TLV(k, slot, v) do { } while (0)
#endif

// ---- PTX helpers ---------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  for (uint32_t spin = 0; !done; ++spin) {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    if (!done && spin > (1u << 26)) __trap();   // a broken copy must not hang the GPU
  }
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// one weight shadow as 8 bulk copies (several requests in flight), all completing on `bar`
__device__ __forceinline__ void load_wmat(uint32_t dst, const op_t* src, uint32_t bar) {
  constexpr int CH = WMAT_BYTES / 8;    // 6720, multiple of 16
#pragma unroll
  for (int i = 0; i < 8; ++i) bulk_g2s(dst + i * CH, (const char*)src + i * CH, CH, bar);
}
__device__ __forceinline__ void mma_16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3,
                                         uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// acc[j] (+)= A[16 x 160] . W[n0 + 8j .. +8][160]^T for the warp's m-tile / column group.
//   A: first row of the m-tile in a [TM][LDS] op_t tile;  W: row n0 of a [KP][LDS] shadow ([n][k]).
__device__ __forceinline__ void warp_gemm(const op_t* __restrict__ A, const op_t* __restrict__ W, float (&acc)[NT][4], int lane) {
  const int g = lane >> 2, t = lane & 3;
  const uint32_t* a_lo = reinterpret_cast<const uint32_t*>(A + g * LDS) + t;
  const uint32_t* a_hi = reinterpret_cast<const uint32_t*>(A + (g + 8) * LDS) + t;
  const uint32_t* w = reinterpret_cast<const uint32_t*>(W + g * LDS) + t;
#pragma unroll
  for (int ks = 0; ks < KP / 16; ++ks) {
    const uint32_t a0 = a_lo[ks * 8], a1 = a_hi[ks * 8], a2 = a_lo[ks * 8 + 4], a3 = a_hi[ks * 8 + 4];
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      const uint32_t b0 = w[j * 8 * (LDS / 2) + ks * 8], b1 = w[j * 8 * (LDS / 2) + ks * 8 + 4];
      mma_16816(acc[j], a0, a1, a2, a3, b0, b1);
    }
  }
}
__device__ __forceinline__ void zero_acc(float (&acc)[NT][4]) {
#pragma unroll
  for (int j = 0; j < NT; ++j) { acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f; }
}
__device__ __forceinline__ float clamp_h(float v) { return fminf(fmaxf(v, -65504.f), 65504.f); }
__device__ __forceinline__ void st_op2(op_t* p, float a, float b) {
  *reinterpret_cast<__half2*>(p) = __floats2half2_rn(clamp_h(a), clamp_h(b));
}
__device__ __forceinline__ op_t to_op(float v) { return __float2half_rn(clamp_h(v)); }
// power-of-two scale s with max * s in [2^10, 2^11): 16x headroom for the chained product, exact to undo (inv = 1/s).
// Exponent arithmetic on the bit pattern: mx = m * 2^e with m in [0.5, 1)  ->  s = 2^(11 - e), clamped to 2^+-100.
__device__ __forceinline__ float row_scale(float mx, float& inv) {
  if (!(mx > 0.f)) { inv = 1.f; return 1.f; }
  const int e = (int)((__float_as_uint(mx) >> 23) & 0xffu) - 126;      // subnormal (field 0) -> clamps to 2^100 like any tiny value
  const int k = min(max(11 - e, -100), 100);
  inv = __uint_as_float((uint32_t)(127 - k) << 23);
  return __uint_as_float((uint32_t)(127 + k) << 23);
}
// ---- batched row access: every warp owns RPW = 4 consecutive tile rows.  All global loads of a phase are issued
// before the first use (one L2 round trip per phase instead of one per row), reductions of the 4 rows interleave.
constexpr int RPW = TM / 8;
__device__ __forceinline__ void warp_sum_n(float (&v)[RPW]) {
#pragma unroll
  for (int o = 16; o; o >>= 1)
#pragma unroll
    for (int r = 0; r < RPW; ++r) v[r] += __shfl_xor_sync(0xffffffffu, v[r], o);
}
__device__ __forceinline__ void warp_max_n(float (&v)[RPW]) {
#pragma unroll
  for (int o = 16; o; o >>= 1)
#pragma unroll
    for (int r = 0; r < RPW; ++r) v[r] = fmaxf(v[r], __shfl_xor_sync(0xffffffffu, v[r], o));
}
// x[rr][e] = G[t0 + warp*RPW + rr][lane + 32 e]   (0 outside [0,T) x [0,d))
__device__ __forceinline__ void load_rows(float (&x)[RPW][NE], const float* G, int t0, int T, int d, int warp, int lane) {
#pragma unroll
  for (int rr = 0; rr < RPW; ++rr) {
    const int tk = t0 + warp * RPW + rr;
#pragma unroll
    for (int e = 0; e < NE; ++e) { const int c = lane + 32 * e; x[rr][e] = (tk < T && c < d) ? G[(long long)tk * d + c] : 0.f; }
  }
}
// per-lane scalars of the warp's rows (mean / rstd / D ...)
__device__ __forceinline__ void load_row_scalars(float (&v)[RPW], const float* G, int t0, int T, int warp) {
#pragma unroll
  for (int rr = 0; rr < RPW; ++rr) { const int tk = t0 + warp * RPW + rr; v[rr] = (tk < T) ? G[tk] : 0.f; }
}
// registers -> 16-bit operand tile rows with a per-row power-of-two scale (x2, if given, shares the scale: joint max)
__device__ __forceinline__ void put_rows_scaled(op_t* __restrict__ As, float* __restrict__ inv_scale, const float (&x)[RPW][NE],
                                                int warp, int lane, const float (*x2)[NE] = nullptr, op_t* __restrict__ As2 = nullptr) {
  float mx[RPW];
#pragma unroll
  for (int rr = 0; rr < RPW; ++rr) {
    float m = 0.f;
#pragma unroll
    for (int e = 0; e < NE; ++e) { m = fmaxf(m, fabsf(x[rr][e])); if (x2) m = fmaxf(m, fabsf(x2[rr][e])); }
    mx[rr] = m;
  }
  warp_max_n(mx);
#pragma unroll
  for (int rr = 0; rr < RPW; ++rr) {
    const int r = warp * RPW + rr;
    float inv;
    const float sc = row_scale(mx[rr], inv);
#pragma unroll
    for (int e = 0; e < NE; ++e) {
      const int c = lane + 32 * e;
      As[r * LDS + c] = to_op(x[rr][e] * sc);
      if (x2) As2[r * LDS + c] = to_op(x2[rr][e] * sc);
    }
    if (lane == 0) inv_scale[r] = inv;
  }
}
__device__ __forceinline__ void put_rows(op_t* __restrict__ As, const float (&x)[RPW][NE], int warp, int lane) {
#pragma unroll
  for (int rr = 0; rr < RPW; ++rr)
#pragma unroll
    for (int e = 0; e < NE; ++e) As[(warp * RPW + rr) * LDS + lane + 32 * e] = to_op(x[rr][e]);
}
// elements of a [T,d] matrix co-located with this thread's accumulator fragment (row = mt*16 + g + 8h, col pair);
// issued ahead of the GEMM whose epilogue consumes them
__device__ __forceinline__ void load_frag(float2 (&v)[NT][2], const float* G, int t0, int T, int d, int mt, int ng, int lane) {
  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const int c = ng * (NT * 8) + j * 8 + 2 * t;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int tk = t0 + mt * 16 + g + 8 * h;
      v[j][h] = (tk < T && c < d) ? *reinterpret_cast<const float2*>(G + (long long)tk * d + c) : make_float2(0.f, 0.f);
    }
  }
}
__device__ __forceinline__ void load_bias_frag(float2 (&b)[NT], const float* __restrict__ bias, int d, int ng, int lane) {
  const int t = lane & 3;
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const int c = ng * (NT * 8) + j * 8 + 2 * t;
    b[j] = (c < d) ? *reinterpret_cast<const float2*>(bias + c) : make_float2(0.f, 0.f);
  }
}
// visit accumulator elements with their fragment coordinates: f(j, h, tile row, col, v0, v1)
template <typename F>
__device__ __forceinline__ void for_frag(const float (&acc)[NT][4], int mt, int ng, int lane, F f) {
  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const int col = ng * (NT * 8) + j * 8 + 2 * t;
    f(j, 0, mt * 16 + g, col, acc[j][0], acc[j][1]);
    f(j, 1, mt * 16 + g + 8, col, acc[j][2], acc[j][3]);
  }
}

// ---- weight shadows ------------------------------------------------------------------------------
// shadow[(b*5 + w)*2 + 0][n][k] = W_w[k][n]   (forward:  out = in . W,   B(k = in,  n = out))
// shadow[(b*5 + w)*2 + 1][n][k] = W_w[n][k]   (backward: gin = gout . W^T, B(k = out, n = in))
// grid (5 * NB matrices, 5 bands of 32 output rows): CTA stages W[n0:n0+32, :] and W[:, n0:n0+32] and writes rows
// n0..n0+31 of both orientations with coalesced 32-bit stores.
constexpr int PACK_BAND = 32;
__global__ void __launch_bounds__(256) k_pack_weights(const float* __restrict__ theta, Layout l, op_t* __restrict__ shadow) {
  __shared__ float rowband[PACK_BAND][KP + 1];    // rowband[r][k] = W[n0 + r][k]
  __shared__ float colband[KP][PACK_BAND + 1];    // colband[k][r] = W[k][n0 + r]
  const int w = blockIdx.x % 5, b = blockIdx.x / 5;
  const int n0 = blockIdx.y * PACK_BAND;
  const long long rel[5] = {l.wq, l.wk, l.wv, l.w1, l.w2};
  const float* W = theta + l.block(b) + rel[w];
  const int d = l.d;
  for (int idx = threadIdx.x; idx < PACK_BAND * KP; idx += blockDim.x) {
    const int r = idx / KP, k = idx % KP;
    rowband[r][k] = (n0 + r < d && k < d) ? W[(long long)(n0 + r) * d + k] : 0.f;
  }
  for (int idx = threadIdx.x; idx < KP * PACK_BAND; idx += blockDim.x) {
    const int k = idx / PACK_BAND, r = idx % PACK_BAND;
    colband[k][r] = (n0 + r < d && k < d) ? W[(long long)k * d + n0 + r] : 0.f;
  }
  __syncthreads();
  op_t* out0 = shadow + (size_t)(blockIdx.x * 2) * (KP * LDS);
  op_t* out1 = out0 + KP * LDS;
  for (int idx = threadIdx.x; idx < PACK_BAND * (LDS / 2); idx += blockDim.x) {
    const int r = idx / (LDS / 2), k = (idx % (LDS / 2)) * 2;
    if (n0 + r >= KP) continue;
    float a0 = 0.f, a1 = 0.f, b0 = 0.f, b1 = 0.f;
    if (k < KP) { a0 = colband[k][r]; a1 = colband[k + 1][r]; b0 = rowband[r][k]; b1 = rowband[r][k + 1]; }
    st_op2(out0 + (n0 + r) * LDS + k, a0, a1);
    st_op2(out1 + (n0 + r) * LDS + k, b0, b1);
  }
}

// ---- forward: [embed] + LN1 + Q/K/V ---------------------------------------------------------------
struct QkvFwdArgs {
  const float* X;            // [T,d] block input (ignored when embed != 0: computed here and written to Xw)
  float* Xw;
  int embed;
  const float *table, *pos_table; const int *tok_row, *tok_id, *row_len, *row_off;
  float sqrt_d, drop_p; uint64_t seed; const int* d_step;
  const float *ln_b, *ln_g; float *Q1, *mean, *rstd;
  const op_t *Wq, *Wk, *Wv; const float *bq, *bk, *bv;
  float *Q, *K, *V;
  const int* dT; int d, L;
};
constexpr size_t QKV_FWD_SMEM = 3 * WMAT_BYTES + 2 * ATILE_BYTES + TM * 4 + 16;

// One 32-token tile [t0, t0 + TM) of the rows below T: [embedding] + LN1 -> operand tiles, Q / K / V products.  wait_q() /
// wait_kv() block until the Wq / (Wk, Wv) shadows have landed in shared memory (no-ops once they have).
template <class WaitQ, class WaitKV>
__device__ __forceinline__ void qkv_fwd_tile(const QkvFwdArgs& a, int t0, int T, uint64_t seed_eff, op_t* __restrict__ A1, op_t* __restrict__ A2,
                                             float* __restrict__ rs, const op_t* Wq_s, const op_t* Wk_s, const op_t* Wv_s,
                                             const float (&lg)[NE], const float (&lb)[NE], const float2 (&bq)[NT], const float2 (&bk)[NT],
                                             const float2 (&bv)[NT], WaitQ wait_q, WaitKV wait_kv) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int mt = warp & 1, ng = warp >> 1;
  const int d = a.d;
  const DropSite ds0 = drop_site(seed_eff, 0u, a.drop_p);
  FZ_TL(0, 6);
  // ---- prologue: [embedding] + LayerNorm of the warp's 4 rows -> fp32 q1 (HBM) and the two operand tiles
  float x[RPW][NE];
  if (a.embed) {         // x = (E0[id]*sqrt(d) + P[pos]) * dropout   (modules.py:124-130, ADER.py:41-60)
    int rowi[RPW], idv[RPW], pp[RPW];
#pragma unroll
    for (int rr = 0; rr < RPW; ++rr) {
      const int tk = t0 + warp * RPW + rr;
      rowi[rr] = (tk < T) ? a.tok_row[tk] : 0; idv[rr] = (tk < T) ? a.tok_id[tk] : 0;
    }
#pragma unroll
    for (int rr = 0; rr < RPW; ++rr) {
      const int tk = t0 + warp * RPW + rr;
      pp[rr] = (tk < T) ? a.L - a.row_len[rowi[rr]] + (tk - a.row_off[rowi[rr]]) : 0;
    }
#pragma unroll
    for (int rr = 0; rr < RPW; ++rr) {
      const int tk = t0 + warp * RPW + rr;
#pragma unroll
      for (int e = 0; e < NE; ++e) {
        const int c = lane + 32 * e;
        x[rr][e] = (tk < T && c < d) ? a.table[(long long)idv[rr] * d + c] * a.sqrt_d + a.pos_table[pp[rr] * d + c] : 0.f;
      }
    }
#pragma unroll
    for (int rr = 0; rr < RPW; ++rr) {
      const int tk = t0 + warp * RPW + rr;
#pragma unroll
      for (int e = 0; e < NE; ++e) {
        const int c = lane + 32 * e;
        if (tk < T && c < d) {
          if (a.drop_p > 0.f) x[rr][e] *= drop_mul(ds0, (uint64_t)tk * d + c);
          a.Xw[(long long)tk * d + c] = x[rr][e];
        }
      }
    }
  } else {
    load_rows(x, a.X, t0, T, d, warp, lane);
  }
  float sm[RPW], mx[RPW], qv[RPW];
#pragma unroll
  for (int rr = 0; rr < RPW; ++rr) {
    float s = 0.f, m = 0.f;
#pragma unroll
    for (int e = 0; e < NE; ++e) { s += x[rr][e]; m = fmaxf(m, fabsf(x[rr][e])); }
    sm[rr] = s; mx[rr] = m;
  }
  warp_sum_n(sm); warp_max_n(mx);
  FZ_TL(0, 7);
  const float inv_d = 1.0f / (float)d;
#pragma unroll
  for (int rr = 0; rr < RPW; ++rr) {
    sm[rr] *= inv_d;
    float q = 0.f;
#pragma unroll
    for (int e = 0; e < NE; ++e) { const int c = lane + 32 * e; if (c < d) { const float u = x[rr][e] - sm[rr]; q += u * u; } }
    qv[rr] = q;
  }
  warp_sum_n(qv);
#pragma unroll
  for (int rr = 0; rr < RPW; ++rr) {
    const int r = warp * RPW + rr, tk = t0 + r;
    const float mean = sm[rr], rstd = rsqrtf(qv[rr] * inv_d + 1e-8f);
    float sci;
    const float sc = row_scale(mx[rr], sci);
#pragma unroll
    for (int e = 0; e < NE; ++e) {
      const int c = lane + 32 * e;
      float y = 0.f;
      if (tk < T && c < d) { y = lg[e] * ((x[rr][e] - mean) * rstd) + lb[e]; a.Q1[(long long)tk * d + c] = y; }
      A1[r * LDS + c] = to_op(y);
      A2[r * LDS + c] = to_op(x[rr][e] * sc);
    }
    if (lane == 0) { rs[r] = sci; if (tk < T) { a.mean[tk] = mean; a.rstd[tk] = rstd; } }
  }
  __syncthreads();
  FZ_TL(0, 2);
  wait_q();
  FZ_TL(0, 3);
  float acc[NT][4];
  zero_acc(acc);
  warp_gemm(A1 + mt * 16 * LDS, Wq_s + ng * (NT * 8) * LDS, acc, lane);
  for_frag(acc, mt, ng, lane, [&](int j, int h, int r, int c, float v0, float v1) {
    if (t0 + r < T && c < d)
      *reinterpret_cast<float2*>(a.Q + (long long)(t0 + r) * d + c) = make_float2(v0 + bq[j].x, v1 + bq[j].y);
  });
  FZ_TL(0, 4);
  wait_kv();
  zero_acc(acc);
  warp_gemm(A2 + mt * 16 * LDS, Wk_s + ng * (NT * 8) * LDS, acc, lane);
  for_frag(acc, mt, ng, lane, [&](int j, int h, int r, int c, float v0, float v1) {
    if (t0 + r < T && c < d)
      *reinterpret_cast<float2*>(a.K + (long long)(t0 + r) * d + c) = make_float2(v0 * rs[r] + bk[j].x, v1 * rs[r] + bk[j].y);
  });
  FZ_TL(0, 8);
  zero_acc(acc);
  warp_gemm(A2 + mt * 16 * LDS, Wv_s + ng * (NT * 8) * LDS, acc, lane);
  for_frag(acc, mt, ng, lane, [&](int j, int h, int r, int c, float v0, float v1) {
    if (t0 + r < T && c < d)
      *reinterpret_cast<float2*>(a.V + (long long)(t0 + r) * d + c) = make_float2(v0 * rs[r] + bv[j].x, v1 * rs[r] + bv[j].y);
  });
  __syncthreads();
  FZ_TL(0, 5);
}

__global__ void __launch_bounds__(NTHR, 1) k_qkv_fwd(const __grid_constant__ QkvFwdArgs a) {
  FZ_TL(0, 0);
  const uint64_t seed_eff = eff_seed(a.seed, a.d_step);
  extern __shared__ __align__(128) uint8_t smem[];
  op_t* Wsm = reinterpret_cast<op_t*>(smem);
  op_t* A1 = reinterpret_cast<op_t*>(smem + 3 * WMAT_BYTES);      // LN1(x)
  op_t* A2 = A1 + TM * LDS;                                      // x (row-scaled: the residual stream is unbounded)
  float* rs = reinterpret_cast<float*>(smem + 3 * WMAT_BYTES + 2 * ATILE_BYTES);
  const uint32_t bar = smem_u32(smem + 3 * WMAT_BYTES + 2 * ATILE_BYTES + TM * 4);
  const int T = *a.dT, d = a.d;
  const int ntiles = (T + TM - 1) / TM;
  if ((int)blockIdx.x >= ntiles) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) {
    mbar_init(bar, 1);
    mbar_expect_tx(bar, 3 * WMAT_BYTES);
    load_wmat(smem_u32(Wsm), a.Wq, bar);
    load_wmat(smem_u32(Wsm) + WMAT_BYTES, a.Wk, bar);
    load_wmat(smem_u32(Wsm) + 2 * WMAT_BYTES, a.Wv, bar);
  }
  const int ng = warp >> 1;
  float lg[NE], lb[NE];
#pragma unroll
  for (int e = 0; e < NE; ++e) { const int c = lane + 32 * e; lg[e] = (c < d) ? a.ln_g[c] : 0.f; lb[e] = (c < d) ? a.ln_b[c] : 0.f; }
  float2 bq[NT], bk[NT], bv[NT];
  load_bias_frag(bq, a.bq, d, ng, lane); load_bias_frag(bk, a.bk, d, ng, lane); load_bias_frag(bv, a.bv, d, ng, lane);
  pdl_wait(); pdl_go();        // everything above reads step constants only (weights, LN parameters, T)
  __syncthreads();
  FZ_TL(0, 1);
  bool first = true;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
    qkv_fwd_tile(a, tile * TM, T, seed_eff, A1, A2, rs, Wsm, Wsm + KP * LDS, Wsm + 2 * KP * LDS, lg, lb, bq, bk, bv,
                 [&] { if (first) { mbar_wait(bar, 0); first = false; } }, [] {});
}

// ---- warp-per-token attention building blocks -------------------------------------------------------------
// Keys / queries are processed in blocks of 8 rows: all 40 row loads of a block are independent (one L2 round
// trip per block instead of one per key), and the 8 dot products are finished by a reduce-scatter (9 shuffles
// for 8 sums instead of 40): afterwards EVERY lane holds the sum for row (lane & 7) of the block.
constexpr int KB = 8;
__device__ __forceinline__ float reduce_scatter8(float (&v)[KB], int lane) {
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float send = (lane & 4) ? v[k] : v[k + 4];
    const float keep = (lane & 4) ? v[k + 4] : v[k];
    v[k] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
  }
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const float send = (lane & 2) ? v[k] : v[k + 2];
    const float keep = (lane & 2) ? v[k + 2] : v[k];
    v[k] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
  }
  {
    const float send = (lane & 1) ? v[0] : v[1];
    const float keep = (lane & 1) ? v[1] : v[0];
    v[0] = keep + __shfl_xor_sync(0xffffffffu, send, 1);
  }
  float r = v[0];
  r += __shfl_xor_sync(0xffffffffu, r, 8);
  r += __shfl_xor_sync(0xffffffffu, r, 16);
  return r;
}
// every lane <- dot(x[.], rows[(lane & 7) * d + .]) over features [c_lo, c_hi) when (lane & 7) < count, else 0.
__device__ __forceinline__ float block_dots(const float (&x)[NE], const float* __restrict__ rows, int d, int count,
                                            int c_lo, int c_hi, int lane) {
  float part[KB];
#pragma unroll
  for (int u = 0; u < KB; ++u) {
    const float* r = rows + (long long)min(u, count - 1) * d;      // clamped duplicate loads hit L1
    float p = 0.f;
#pragma unroll
    for (int e = 0; e < NE; ++e) { const int c = lane + 32 * e; if (c >= c_lo && c < c_hi) p = fmaf(x[e], r[c], p); }
    part[u] = (u < count) ? p : 0.f;
  }
  return reduce_scatter8(part, lane);
}
// acc[.] += sum_{u < count} w_u * rows[u * d + .], w_u held by lane u (u < 8); features [c_lo, c_hi).  Fixed order.
__device__ __forceinline__ void block_axpy(float (&acc)[NE], float w, const float* __restrict__ rows, int d, int count,
                                           int c_lo, int c_hi, int lane) {
  float v[KB][NE], wu[KB];
#pragma unroll
  for (int u = 0; u < KB; ++u) {
    wu[u] = __shfl_sync(0xffffffffu, w, u);
    if (u >= count) wu[u] = 0.f;
    const float* r = rows + (long long)min(u, count - 1) * d;
#pragma unroll
    for (int e = 0; e < NE; ++e) { const int c = lane + 32 * e; v[u][e] = (c >= c_lo && c < c_hi) ? r[c] : 0.f; }
  }
#pragma unroll
  for (int u = 0; u < KB; ++u)
#pragma unroll
    for (int e = 0; e < NE; ++e) acc[e] = fmaf(wu[u], v[u][e], acc[e]);
}

// ---- forward: causal attention + residual + LN2, warp per query token (modules.py:177-223, 40-48) ---
struct AttnFwdArgs {
  const float *Q, *K, *V, *Q1;
  const int *tok_row, *row_off;
  float *probs, *Y, *Z, *mean2, *rstd2;
  const float *ln_b, *ln_g;
  const int* dT; int d, nh, L, Tcap;
  float drop_p; uint64_t seed; const int* d_step; uint32_t site;
};

// cooperative copy of n2 float2 (rows are contiguous [n, d] in global memory, 8-byte aligned), 8 loads in flight per thread
__device__ __forceinline__ void stage_f2(float* __restrict__ dst, const float* src, int n2) {
  const float2* s2 = reinterpret_cast<const float2*>(src);
  float2* d2 = reinterpret_cast<float2*>(dst);
  for (int base = threadIdx.x; base < n2; base += 8 * blockDim.x) {
    float2 v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) { const int idx = base + u * blockDim.x; if (idx < n2) v[u] = s2[idx]; }
#pragma unroll
    for (int u = 0; u < 8; ++u) { const int idx = base + u * blockDim.x; if (idx < n2) d2[idx] = v[u]; }
  }
}
constexpr int ATT_TOK = 8;          // tokens (= warps) per CTA of the warp-per-token attention kernels
__host__ __device__ constexpr int att_rows_cap(int L) { return L + ATT_TOK - 1; }   // K/V rows a CTA can need

// The 8 consecutive tokens of a CTA belong to at most a few sessions, and a token only attends to earlier tokens of
// its own session, so the union of all keys the CTA needs is ONE contiguous token range [row start of the first
// token, last token of the CTA]: <= L + 7 rows.  K and V of that range are staged in shared memory by a cooperative,
// fully overlapped copy (one L2 round trip for the CTA), and the warps then work out of shared memory.
// One group of ATT_TOK consecutive query tokens [t0, t0 + ATT_TOK) of the rows below T (all threads of the CTA call it:
// cooperative staging + one __syncthreads inside).
__device__ __forceinline__ void attn_fwd_group(const AttnFwdArgs& a, int t0, int T, float* __restrict__ att_sm, uint64_t seed_eff) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int d = a.d, L = a.L;
  const int tk = min(t0 + warp, T - 1);          // surplus warps of the last CTA shadow its last token (no stores)
  const bool live = t0 + warp < T;
  const int row = a.tok_row[tk];
  const int lo = a.row_off[a.tok_row[t0]];
  const int off = a.row_off[row];
  const int hi = min(t0 + ATT_TOK, T);
  float q[NE], o[NE], q1[NE];
#pragma unroll
  for (int e = 0; e < NE; ++e) {
    const int c = lane + 32 * e;
    q[e] = (c < d) ? a.Q[(long long)tk * d + c] : 0.f;
    q1[e] = (c < d) ? a.Q1[(long long)tk * d + c] : 0.f;
    o[e] = 0.f;
  }
  float* Ks = att_sm;
  float* Vs = att_sm + att_rows_cap(L) * d;
  const DropSite dsp = drop_site(seed_eff, a.site, a.drop_p);
  FZ_TL(4, 0);
  stage_f2(Ks, a.K + (long long)lo * d, (hi - lo) * d / 2);
  stage_f2(Vs, a.V + (long long)lo * d, (hi - lo) * d / 2);
  __syncthreads();
  FZ_TL(4, 1);
  if (live) {
    const int i = tk - off;                       // query index inside its session; keys 0..i
    const int dh = d / a.nh;
    const float inv_denom = 1.0f / sqrtf((float)dh);
    const int j8 = lane & 7;
    const float* Krow = Ks + (off - lo) * d;
    const float* Vrow = Vs + (off - lo) * d;
    for (int h = 0; h < a.nh; ++h) {
      const int c_lo = h * dh, c_hi = c_lo + dh;
      const long long po = ((long long)h * a.Tcap + tk) * L;
      // online softmax over key blocks of 8 (running max m, running sum l); raw scores are parked in the probs
      // row and normalised in place afterwards
      float m = -INFINITY, l = 0.f;
      float oh[NE];
  #pragma unroll
      for (int e = 0; e < NE; ++e) oh[e] = 0.f;
      for (int j0 = 0; j0 <= i; j0 += KB) {
        const int cnt = min(KB, i + 1 - j0);
        const float sc = block_dots(q, Krow + (long long)j0 * d, d, cnt, c_lo, c_hi, lane) * inv_denom;
        const bool valid = j8 < cnt;
        float bm = valid ? sc : -INFINITY;
        bm = fmaxf(bm, __shfl_xor_sync(0xffffffffu, bm, 4));
        bm = fmaxf(bm, __shfl_xor_sync(0xffffffffu, bm, 2));
        bm = fmaxf(bm, __shfl_xor_sync(0xffffffffu, bm, 1));
        const float m_new = fmaxf(m, bm);
        const float corr = expf(m - m_new);
        float pj = valid ? expf(sc - m_new) : 0.f;
        float ps = pj;
        ps += __shfl_xor_sync(0xffffffffu, ps, 4);
        ps += __shfl_xor_sync(0xffffffffu, ps, 2);
        ps += __shfl_xor_sync(0xffffffffu, ps, 1);
        l = l * corr + ps;
        m = m_new;
        if (lane < KB && valid) a.probs[po + j0 + j8] = sc;
        if (a.drop_p > 0.f && valid) pj *= drop_mul(dsp, (uint64_t)(po + j0 + j8));
  #pragma unroll
        for (int e = 0; e < NE; ++e) oh[e] *= corr;
        block_axpy(oh, pj, Vrow + (long long)j0 * d, d, cnt, c_lo, c_hi, lane);
      }
      const float inv_l = 1.0f / l;
  #pragma unroll
      for (int e = 0; e < NE; ++e) { const int c = lane + 32 * e; if (c >= c_lo && c < c_hi) o[e] = oh[e] * inv_l; }
      __syncwarp();
  #pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int j = lane + 32 * u;
        if (j < L) a.probs[po + j] = (j <= i) ? expf(a.probs[po + j] - m) * inv_l : 0.f;
      }
    }
    FZ_TL(4, 2);
    // y = attn + q1 (residual on the NORMALISED queries, modules.py:223), z = LN2(y)
    float y[NE]; float sm = 0.f;
    float lg[NE], lb[NE];              // loaded BEFORE the stores below: a load behind a store through an unrelated pointer is not hoisted
  #pragma unroll
    for (int e = 0; e < NE; ++e) { const int c = lane + 32 * e; lg[e] = (c < d) ? a.ln_g[c] : 0.f; lb[e] = (c < d) ? a.ln_b[c] : 0.f; }
  #pragma unroll
    for (int e = 0; e < NE; ++e) {
      const int c = lane + 32 * e;
      y[e] = (c < d) ? o[e] + q1[e] : 0.f;
      if (c < d) a.Y[(long long)tk * d + c] = y[e];
      sm += y[e];
    }
    const float inv_d = 1.0f / (float)d;
    const float mean = warp_sum(sm) * inv_d;
    float qq = 0.f;
  #pragma unroll
    for (int e = 0; e < NE; ++e) { const int c = lane + 32 * e; if (c < d) { const float u = y[e] - mean; qq += u * u; } }
    const float rstd = rsqrtf(warp_sum(qq) * inv_d + 1e-8f);
  #pragma unroll
    for (int e = 0; e < NE; ++e) {
      const int c = lane + 32 * e;
      if (c < d) a.Z[(long long)tk * d + c] = lg[e] * ((y[e] - mean) * rstd) + lb[e];
    }
    if (lane == 0) { a.mean2[tk] = mean; a.rstd2[tk] = rstd; }
  }
  FZ_TL(4, 3);
}

__global__ void __launch_bounds__(256, 3) k_attn_ln_fwd(const __grid_constant__ AttnFwdArgs a) {
  extern __shared__ __align__(16) float att_sm[];
  const uint64_t seed_eff = eff_seed(a.seed, a.d_step);
  const int T = *a.dT;
  const int t0 = blockIdx.x * ATT_TOK;
  if (t0 >= T) return;
  pdl_wait(); pdl_go();
  attn_fwd_group(a, t0, T, att_sm, seed_eff);
}

// ---- forward: FFN1 + ReLU + FFN2 + residual (modules.py:252-271) -----------------------------------
struct FfnFwdArgs {
  const float* Z; float *H, *Xn;
  const op_t *W1, *W2; const float *b1, *b2;
  const int* dT; int d;
  float drop_p; uint64_t seed; const int* d_step; uint32_t site1, site2;
};
constexpr size_t FFN_FWD_SMEM = 2 * WMAT_BYTES + 2 * ATILE_BYTES + 16;

// One 32-token tile: FFN1 + ReLU (+ dropout) -> H, FFN2 (+ dropout) + residual -> Xn.  A2's padding columns must be zero.
template <class WaitW>
__device__ __forceinline__ void ffn_fwd_tile(const FfnFwdArgs& a, int t0, int T, uint64_t seed_eff, op_t* __restrict__ A1, op_t* __restrict__ A2,
                                             const op_t* W1_s, const op_t* W2_s, const float2 (&b1)[NT], const float2 (&b2)[NT], WaitW wait_w) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int mt = warp & 1, ng = warp >> 1;
  const int d = a.d;
  const DropSite ds1 = drop_site(seed_eff, a.site1, a.drop_p), ds2 = drop_site(seed_eff, a.site2, a.drop_p);
  FZ_TL(5, 0);
  float z[RPW][NE];
  load_rows(z, a.Z, t0, T, d, warp, lane);
  float2 zf[NT][2];
  load_frag(zf, a.Z, t0, T, d, mt, ng, lane);          // residual operand of the second epilogue
  put_rows(A1, z, warp, lane);
  __syncthreads();
  FZ_TL(5, 1);
  wait_w();
  FZ_TL(5, 2);
  float acc[NT][4];
  zero_acc(acc);
  warp_gemm(A1 + mt * 16 * LDS, W1_s + ng * (NT * 8) * LDS, acc, lane);
  FZ_TL(5, 5);
  for_frag(acc, mt, ng, lane, [&](int j, int h, int r, int c, float v0, float v1) {
    if (c < d) {
      float h0 = 0.f, h1 = 0.f;
      if (t0 + r < T) {
        const long long e = (long long)(t0 + r) * d + c;
        h0 = fmaxf(v0 + b1[j].x, 0.f); h1 = fmaxf(v1 + b1[j].y, 0.f);
        if (a.drop_p > 0.f) { h0 *= drop_mul(ds1, (uint64_t)e); h1 *= drop_mul(ds1, (uint64_t)e + 1); }
        *reinterpret_cast<float2*>(a.H + e) = make_float2(h0, h1);
      }
      st_op2(A2 + r * LDS + c, h0, h1);
    }
  });
  __syncthreads();
  FZ_TL(5, 3);
  zero_acc(acc);
  warp_gemm(A2 + mt * 16 * LDS, W2_s + ng * (NT * 8) * LDS, acc, lane);
  for_frag(acc, mt, ng, lane, [&](int j, int h, int r, int c, float v0, float v1) {
    if (t0 + r < T && c < d) {
      const long long e = (long long)(t0 + r) * d + c;
      float x0 = v0 + b2[j].x, x1 = v1 + b2[j].y;
      if (a.drop_p > 0.f) { x0 *= drop_mul(ds2, (uint64_t)e); x1 *= drop_mul(ds2, (uint64_t)e + 1); }
      *reinterpret_cast<float2*>(a.Xn + e) = make_float2(x0 + zf[j][h].x, x1 + zf[j][h].y);
    }
  });
  __syncthreads();
  FZ_TL(5, 4);
}

__global__ void __launch_bounds__(NTHR, 1) k_ffn_fwd(const __grid_constant__ FfnFwdArgs a) {
  const uint64_t seed_eff = eff_seed(a.seed, a.d_step);
  extern __shared__ __align__(128) uint8_t smem[];
  op_t* Wsm = reinterpret_cast<op_t*>(smem);
  op_t* A1 = reinterpret_cast<op_t*>(smem + 2 * WMAT_BYTES);
  op_t* A2 = A1 + TM * LDS;
  const uint32_t bar = smem_u32(smem + 2 * WMAT_BYTES + 2 * ATILE_BYTES);
  const int T = *a.dT, d = a.d;
  const int ntiles = (T + TM - 1) / TM;
  if ((int)blockIdx.x >= ntiles) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) {
    mbar_init(bar, 1);
    mbar_expect_tx(bar, 2 * WMAT_BYTES);
    load_wmat(smem_u32(Wsm), a.W1, bar);
    load_wmat(smem_u32(Wsm) + WMAT_BYTES, a.W2, bar);
  }
  // zero the padding columns of the hidden tile once (the epilogue only writes columns < d)
  for (int idx = tid; idx < TM * LDS; idx += NTHR) A2[idx] = to_op(0.f);
  const int ng = warp >> 1;
  float2 b1[NT], b2[NT];
  load_bias_frag(b1, a.b1, d, ng, lane); load_bias_frag(b2, a.b2, d, ng, lane);
  pdl_wait(); pdl_go();
  __syncthreads();
  bool first = true;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
    ffn_fwd_tile(a, tile * TM, T, seed_eff, A1, A2, Wsm, Wsm + KP * LDS, b1, b2, [&] { if (first) { mbar_wait(bar, 0); first = false; } });
}

// ---- LayerNorm backward of the warp's 4 rows (dout in a shared fp32 tile, x / mean / rstd preloaded) ----------
// dx = rstd*(g - mean(g) - xhat*mean(g*xhat)),  g = dout*gamma.
__device__ __forceinline__ void ln_bwd_rows(const float* __restrict__ Ft, const float (&xv)[RPW][NE], const float (&mean)[RPW],
                                            const float (&rstd)[RPW], const float (&gam)[NE], int d, int warp, int lane,
                                            float (&dx)[RPW][NE]) {
  float s1[RPW], s2[RPW];
  float xh[RPW][NE];
#pragma unroll
  for (int rr = 0; rr < RPW; ++rr) {
    const float* dr = Ft + (warp * RPW + rr) * FT_LD;
    float a1 = 0.f, a2 = 0.f;
#pragma unroll
    for (int e = 0; e < NE; ++e) {
      const int c = lane + 32 * e;
      if (c < d) { xh[rr][e] = (xv[rr][e] - mean[rr]) * rstd[rr]; dx[rr][e] = dr[c] * gam[e]; a1 += dx[rr][e]; a2 += dx[rr][e] * xh[rr][e]; }
      else { xh[rr][e] = 0.f; dx[rr][e] = 0.f; }
    }
    s1[rr] = a1; s2[rr] = a2;
  }
  warp_sum_n(s1); warp_sum_n(s2);
  const float inv_d = 1.0f / (float)d;
#pragma unroll
  for (int rr = 0; rr < RPW; ++rr) {
    const float m1 = s1[rr] * inv_d, m2 = s2[rr] * inv_d;
#pragma unroll
    for (int e = 0; e < NE; ++e) dx[rr][e] = rstd[rr] * (dx[rr][e] - m1 - xh[rr][e] * m2);
  }
}

// ---- backward: FFN dgrad + LN2 backward --------------------------------------------------------------
struct FfnBwdArgs {
  const float* gX;           // grad w.r.t. the block output
  float* gO;                 // gX * dropout(site2) (written only when drop_p > 0; the wgrad of W2 reads it)
  const float *H, *Y, *Q1, *mean2, *rstd2, *ln_g;
  const op_t *W2b, *W1b;     // backward-orientation shadows
  float *gH, *gZ, *gY, *D;
  const int* dT; int d;
  float drop_p; uint64_t seed; const int* d_step; uint32_t site2;
};
constexpr size_t FFN_BWD_SMEM = 2 * WMAT_BYTES + 2 * ATILE_BYTES + FTILE_BYTES + TM * 4 + 16;

// One 32-token tile: gOut -> gH -> gZ (two products against the backward-orientation shadows), LN2 backward -> gY, D.
// A2's padding columns must be zero.
template <class WaitW>
__device__ __forceinline__ void ffn_bwd_tile(const FfnBwdArgs& a, int t0, int T, uint64_t seed_eff, op_t* __restrict__ A1, op_t* __restrict__ A2,
                                             float* __restrict__ Ft, float* __restrict__ rs, const op_t* W2_s, const op_t* W1_s,
                                             const float (&gam)[NE], float inv_keep, WaitW wait_w) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int mt = warp & 1, ng = warp >> 1;
  const int d = a.d;
  // gOut = gX * dropout(site2): x_out = drop(h.W2 + b2) + z   (modules.py:259-266)
  float go[RPW][NE];
  load_rows(go, a.gX, t0, T, d, warp, lane);
  float2 hf[NT][2], gxf[NT][2];
  load_frag(hf, a.H, t0, T, d, mt, ng, lane);
  load_frag(gxf, a.gX, t0, T, d, mt, ng, lane);
  if (a.drop_p > 0.f) {
    const DropSite ds2 = drop_site(seed_eff, a.site2, a.drop_p);
#pragma unroll
    for (int rr = 0; rr < RPW; ++rr) {
      const int tk = t0 + warp * RPW + rr;
#pragma unroll
      for (int e = 0; e < NE; ++e) {
        const int c = lane + 32 * e;
        if (tk < T && c < d) {
          const long long el = (long long)tk * d + c;
          go[rr][e] *= drop_mul(ds2, (uint64_t)el);
          a.gO[el] = go[rr][e];
        }
      }
    }
  }
  put_rows_scaled(A1, rs, go, warp, lane);
  __syncthreads();
  FZ_TL(1, 2);
  wait_w();
  FZ_TL(1, 3);
  float acc[NT][4];
  zero_acc(acc);
  warp_gemm(A1 + mt * 16 * LDS, W2_s + ng * (NT * 8) * LDS, acc, lane);
  // gH = (gOut . W2^T) * [h > 0] / (1 - p)   (h is stored post-dropout)
  for_frag(acc, mt, ng, lane, [&](int j, int h, int r, int c, float v0, float v1) {
    if (c < d) {
      float g0 = 0.f, g1 = 0.f;
      if (t0 + r < T) {
        g0 = hf[j][h].x > 0.f ? v0 * inv_keep : 0.f; g1 = hf[j][h].y > 0.f ? v1 * inv_keep : 0.f;   // still carries the row scale
        *reinterpret_cast<float2*>(a.gH + (long long)(t0 + r) * d + c) = make_float2(g0 * rs[r], g1 * rs[r]);
      }
      st_op2(A2 + r * LDS + c, g0, g1);
    }
  });
  // rows of the LayerNorm-backward pass: issue their loads now, they land while the second product runs
  float yv[RPW][NE], q1[RPW][NE], mean[RPW], rstd[RPW];
  load_rows(yv, a.Y, t0, T, d, warp, lane);
  load_rows(q1, a.Q1, t0, T, d, warp, lane);
  load_row_scalars(mean, a.mean2, t0, T, warp);
  load_row_scalars(rstd, a.rstd2, t0, T, warp);
  __syncthreads();
  FZ_TL(1, 4);
  zero_acc(acc);
  warp_gemm(A2 + mt * 16 * LDS, W1_s + ng * (NT * 8) * LDS, acc, lane);
  // gZ = gH . W1^T + gX   (residual z -> x_out)
  for_frag(acc, mt, ng, lane, [&](int j, int h, int r, int c, float v0, float v1) {
    if (c < d) {
      float z0 = 0.f, z1 = 0.f;
      if (t0 + r < T) {
        z0 = v0 * rs[r] + gxf[j][h].x; z1 = v1 * rs[r] + gxf[j][h].y;
        *reinterpret_cast<float2*>(a.gZ + (long long)(t0 + r) * d + c) = make_float2(z0, z1);
      }
      *reinterpret_cast<float2*>(Ft + r * FT_LD + c) = make_float2(z0, z1);
    }
  });
  __syncthreads();
  FZ_TL(1, 5);
  // gY = LN2 backward;  D = gY . (Y - q1)  (= sum_j dP_ij P_ij of the attention softmax backward)
  float dx[RPW][NE], dd[RPW];
  ln_bwd_rows(Ft, yv, mean, rstd, gam, d, warp, lane, dx);
#pragma unroll
  for (int rr = 0; rr < RPW; ++rr) {
    const int tk = t0 + warp * RPW + rr;
    float acc_d = 0.f;
#pragma unroll
    for (int e = 0; e < NE; ++e) {
      const int c = lane + 32 * e;
      if (tk < T && c < d) { a.gY[(long long)tk * d + c] = dx[rr][e]; acc_d = fmaf(dx[rr][e], yv[rr][e] - q1[rr][e], acc_d); }
    }
    dd[rr] = acc_d;
  }
  warp_sum_n(dd);
  if (lane == 0) {
#pragma unroll
    for (int rr = 0; rr < RPW; ++rr) { const int tk = t0 + warp * RPW + rr; if (tk < T) a.D[tk] = dd[rr]; }
  }
  __syncthreads();
  FZ_TL(1, 6);
}

__global__ void __launch_bounds__(NTHR, 1) k_ffn_bwd(const __grid_constant__ FfnBwdArgs a) {
  FZ_TL(1, 0);
  const uint64_t seed_eff = eff_seed(a.seed, a.d_step);
  extern __shared__ __align__(128) uint8_t smem[];
  op_t* Wsm = reinterpret_cast<op_t*>(smem);
  op_t* A1 = reinterpret_cast<op_t*>(smem + 2 * WMAT_BYTES);
  op_t* A2 = A1 + TM * LDS;
  float* Ft = reinterpret_cast<float*>(smem + 2 * WMAT_BYTES + 2 * ATILE_BYTES);
  float* rs = reinterpret_cast<float*>(smem + 2 * WMAT_BYTES + 2 * ATILE_BYTES + FTILE_BYTES);
  const uint32_t bar = smem_u32(smem + 2 * WMAT_BYTES + 2 * ATILE_BYTES + FTILE_BYTES + TM * 4);
  const int T = *a.dT, d = a.d;
  const int ntiles = (T + TM - 1) / TM;
  if ((int)blockIdx.x >= ntiles) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) {
    mbar_init(bar, 1);
    mbar_expect_tx(bar, 2 * WMAT_BYTES);
    load_wmat(smem_u32(Wsm), a.W2b, bar);
    load_wmat(smem_u32(Wsm) + WMAT_BYTES, a.W1b, bar);
  }
  for (int idx = tid; idx < TM * LDS; idx += NTHR) A2[idx] = to_op(0.f);
  float gam[NE];
#pragma unroll
  for (int e = 0; e < NE; ++e) { const int c = lane + 32 * e; gam[e] = (c < d) ? a.ln_g[c] : 0.f; }
  pdl_wait(); pdl_go();
  __syncthreads();
  FZ_TL(1, 1);
  const float inv_keep = a.drop_p > 0.f ? 1.f / (1.f - a.drop_p) : 1.f;
  bool first = true;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
    ffn_bwd_tile(a, tile * TM, T, seed_eff, A1, A2, Ft, rs, Wsm, Wsm + KP * LDS, gam, inv_keep,
                 [&] { if (first) { mbar_wait(bar, 0); first = false; } });
}

// ---- backward: attention, warp per token (query role -> gQ, key role -> gK, gV) ------------------------
struct AttnBwdArgs {
  const float *Q, *K, *V, *probs, *gY, *D;
  const int *tok_row, *row_off;
  float *gQ, *gK, *gV;
  const int* dT; int d, nh, L, Tcap;
  float drop_p; uint64_t seed; const int* d_step; uint32_t site;
};

__global__ void __launch_bounds__(256) k_attn_bwd_w(const __grid_constant__ AttnBwdArgs a) {
  const uint64_t seed_eff = eff_seed(a.seed, a.d_step);
  const int tk = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (tk >= *a.dT) return;
  const int d = a.d, L = a.L;
  const int row = a.tok_row[tk];
  const int off = a.row_off[row];
  const int n = a.row_off[row + 1] - off;
  const int i = tk - off;
  const int dh = d / a.nh;
  const float inv_denom = 1.0f / sqrtf((float)dh);
  float gy[NE], vt[NE], gq[NE], gk[NE], gv[NE];
#pragma unroll
  for (int e = 0; e < NE; ++e) {
    const int c = lane + 32 * e;
    gy[e] = (c < d) ? a.gY[(long long)tk * d + c] : 0.f;
    vt[e] = (c < d) ? a.V[(long long)tk * d + c] : 0.f;
    gq[e] = gk[e] = gv[e] = 0.f;
  }
  const float Di = a.D[tk];
  for (int h = 0; h < a.nh; ++h) {
    const int c_lo = h * dh, c_hi = c_lo + dh;
    // D restricted to this head when nh > 1: D_h = sum_j dP_ij P_ij is recomputed from the head's own columns
    float Dh = Di;
    const long long po_i = ((long long)h * a.Tcap + tk) * L;
    // ---- query role: gQ[i] = sum_{j<=i} dS_ij K[j]
    if (a.nh > 1) {
      float acc = 0.f;
      for (int j = 0; j <= i; ++j) {
        const float* vr = a.V + (long long)(off + j) * d;
        float p = 0.f;
#pragma unroll
        for (int e = 0; e < NE; ++e) { const int c = lane + 32 * e; if (c >= c_lo && c < c_hi) p = fmaf(gy[e], vr[c], p); }
        p = warp_sum(p);
        const float P = a.probs[po_i + j];
        const float scl = a.drop_p > 0.f ? drop_scale(seed_eff, a.site, (uint64_t)(po_i + j), a.drop_p) : 1.f;
        acc = fmaf(p * scl, P, acc);
      }
      Dh = acc;
    }
    for (int j0 = 0; j0 <= i; j0 += 4) {
      float part[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = min(j0 + u, i);
        const float* vr = a.V + (long long)(off + j) * d;
        float p = 0.f;
#pragma unroll
        for (int e = 0; e < NE; ++e) { const int c = lane + 32 * e; if (c >= c_lo && c < c_hi) p = fmaf(gy[e], vr[c], p); }
        part[u] = p;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float dp = warp_sum(part[u]);
        const int j = j0 + u;
        if (j <= i) {
          const float P = a.probs[po_i + j];
          const float scl = a.drop_p > 0.f ? drop_scale(seed_eff, a.site, (uint64_t)(po_i + j), a.drop_p) : 1.f;
          const float ds = P * (dp * scl - Dh) * inv_denom;
          const float* kr = a.K + (long long)(off + j) * d;
#pragma unroll
          for (int e = 0; e < NE; ++e) { const int c = lane + 32 * e; if (c >= c_lo && c < c_hi) gq[e] = fmaf(ds, kr[c], gq[e]); }
        }
      }
    }
    // ---- key role: gK[i] = sum_{i'>=i} dS_i'i Q[i'],  gV[i] = sum_{i'>=i} Pd_i'i gY[i']
    for (int q0 = i; q0 < n; q0 += 4) {
      float part[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int qi = min(q0 + u, n - 1);
        const float* gr = a.gY + (long long)(off + qi) * d;
        float p = 0.f;
#pragma unroll
        for (int e = 0; e < NE; ++e) { const int c = lane + 32 * e; if (c >= c_lo && c < c_hi) p = fmaf(gr[c], vt[e], p); }
        part[u] = p;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float dp = warp_sum(part[u]);
        const int qi = q0 + u;
        if (qi < n) {
          const int tq = off + qi;
          const long long po = ((long long)h * a.Tcap + tq) * L + i;
          const float P = a.probs[po];
          const float scl = a.drop_p > 0.f ? drop_scale(seed_eff, a.site, (uint64_t)po, a.drop_p) : 1.f;
          float Dq = a.D[tq];
          if (a.nh > 1) {      // per-head D of query qi (rare path: num_heads > 1)
            float acc = 0.f;
            const long long pq = ((long long)h * a.Tcap + tq) * L;
            const float* gr = a.gY + (long long)tq * d;
            for (int j = 0; j <= qi; ++j) {
              const float* vr = a.V + (long long)(off + j) * d;
              float p = 0.f;
#pragma unroll
              for (int e = 0; e < NE; ++e) { const int c = lane + 32 * e; if (c >= c_lo && c < c_hi) p = fmaf(gr[c], vr[c], p); }
              p = warp_sum(p);
              const float s2 = a.drop_p > 0.f ? drop_scale(seed_eff, a.site, (uint64_t)(pq + j), a.drop_p) : 1.f;
              acc = fmaf(p * s2, a.probs[pq + j], acc);
            }
            Dq = acc;
          }
          const float ds = P * (dp * scl - Dq) * inv_denom;
          const float pd = P * scl;
          const float* qr = a.Q + (long long)tq * d;
          const float* gr = a.gY + (long long)tq * d;
#pragma unroll
          for (int e = 0; e < NE; ++e) {
            const int c = lane + 32 * e;
            if (c >= c_lo && c < c_hi) { gk[e] = fmaf(ds, qr[c], gk[e]); gv[e] = fmaf(pd, gr[c], gv[e]); }
          }
        }
      }
    }
  }
#pragma unroll
  for (int e = 0; e < NE; ++e) {
    const int c = lane + 32 * e;
    if (c < d) {
      a.gQ[(long long)tk * d + c] = gq[e];
      a.gK[(long long)tk * d + c] = gk[e];
      a.gV[(long long)tk * d + c] = gv[e];
    }
  }
}

// Shared-memory form of the single-head backward kernel (same staging idea as the forward kernel).  Phase 1 (query
// role) stages V and K of [row start of the first token, last token of the CTA]; phase 2 (key role) re-uses the same
// buffers for gY and Q of [first token of the CTA, end of the last token's session]: both ranges are <= L + 7 rows.
// The probabilities a token needs (its own row as a query, its column as a key) and the D values of its later
// queries are fetched into registers up front, so the block loops touch no global memory.
__host__ __device__ constexpr int att_bwd_smem(int L, int d) { return 2 * att_rows_cap(L) * d * 4; }
// One group of ATT_TOK consecutive tokens [t0, t0 + ATT_TOK) of the rows below T (all threads of the CTA call it; the
// caller separates two groups by a __syncthreads: the staging buffers are reused).
__device__ __forceinline__ void attn_bwd_group(const AttnBwdArgs& a, int t0, int T, float* __restrict__ att_sm, uint64_t seed_eff) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int d = a.d, L = a.L;
  const int tk = min(t0 + warp, T - 1);
  const bool live = t0 + warp < T;
  const int row = a.tok_row[tk];
  const int lo = a.row_off[a.tok_row[t0]];
  const int hi = min(t0 + ATT_TOK, T);
  const int hi2 = a.row_off[a.tok_row[hi - 1] + 1];          // end of the session of the CTA's last token
  const int off = a.row_off[row];
  const int n = a.row_off[row + 1] - off;
  const int i = tk - off;
  const float inv_denom = 1.0f / sqrtf((float)d);
  const int j8 = lane & 7;
  float gy[NE], vt[NE], gq[NE], gk[NE], gv[NE];
#pragma unroll
  for (int e = 0; e < NE; ++e) {
    const int c = lane + 32 * e;
    gy[e] = (c < d) ? a.gY[(long long)tk * d + c] : 0.f;
    vt[e] = (c < d) ? a.V[(long long)tk * d + c] : 0.f;
    gq[e] = gk[e] = gv[e] = 0.f;
  }
  const float Di = a.D[tk];
  const DropSite dsp = drop_site(seed_eff, a.site, a.drop_p);
  // probabilities / dropout scales / D: own row (query role: key lane + 32u) and own column (key role: query tk + lane + 32u)
  float pq[2], sq[2], pk[2], sk[2], dk[2];
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const int j = lane + 32 * u;
    pq[u] = 0.f; sq[u] = 1.f; pk[u] = 0.f; sk[u] = 1.f; dk[u] = 0.f;
    if (j <= i) {
      const long long po = (long long)tk * L + j;
      pq[u] = a.probs[po];
      if (a.drop_p > 0.f) sq[u] = drop_mul(dsp, (uint64_t)po);
    }
    if (i + j < n) {
      const int tq = tk + j;
      const long long po = (long long)tq * L + i;
      pk[u] = a.probs[po];
      dk[u] = a.D[tq];
      if (a.drop_p > 0.f) sk[u] = drop_mul(dsp, (uint64_t)po);
    }
  }
  float* As = att_sm;
  float* Bs = att_sm + att_rows_cap(L) * d;
  // ---- phase 1, query role: dS_ij = P_ij (dP_ij - D_i) / sqrt(d),  gQ[i] = sum_{j<=i} dS_ij K[j]
  stage_f2(As, a.V + (long long)lo * d, (hi - lo) * d / 2);
  stage_f2(Bs, a.K + (long long)lo * d, (hi - lo) * d / 2);
  __syncthreads();
  if (live) {
    for (int j0 = 0; j0 <= i; j0 += KB) {
      const int cnt = min(KB, i + 1 - j0);
      const float dp = block_dots(gy, As + (off - lo + j0) * d, d, cnt, 0, d, lane);
      const int j = j0 + j8;
      const float P = __shfl_sync(0xffffffffu, (j < 32) ? pq[0] : pq[1], j & 31);
      const float scl = __shfl_sync(0xffffffffu, (j < 32) ? sq[0] : sq[1], j & 31);
      const float ds = (j8 < cnt) ? P * (dp * scl - Di) * inv_denom : 0.f;
      block_axpy(gq, ds, Bs + (off - lo + j0) * d, d, cnt, 0, d, lane);
    }
  }
  __syncthreads();
  // ---- phase 2, key role: gK[i] = sum_{q>=i} dS_qi Q[q],  gV[i] = sum_{q>=i} Pd_qi gY[q]
  stage_f2(As, a.gY + (long long)t0 * d, (hi2 - t0) * d / 2);
  stage_f2(Bs, a.Q + (long long)t0 * d, (hi2 - t0) * d / 2);
  __syncthreads();
  if (live) {
    for (int q0 = 0; i + q0 < n; q0 += KB) {          // queries tk + q0 .. of the same session
      const int cnt = min(KB, n - i - q0);
      const float dp = block_dots(vt, As + (tk - t0 + q0) * d, d, cnt, 0, d, lane);
      const int u = q0 + j8;
      const float P = __shfl_sync(0xffffffffu, (u < 32) ? pk[0] : pk[1], u & 31);
      const float scl = __shfl_sync(0xffffffffu, (u < 32) ? sk[0] : sk[1], u & 31);
      const float Dq = __shfl_sync(0xffffffffu, (u < 32) ? dk[0] : dk[1], u & 31);
      const float ds = (j8 < cnt) ? P * (dp * scl - Dq) * inv_denom : 0.f;
      const float pd = (j8 < cnt) ? P * scl : 0.f;
      block_axpy(gk, ds, Bs + (tk - t0 + q0) * d, d, cnt, 0, d, lane);
      block_axpy(gv, pd, As + (tk - t0 + q0) * d, d, cnt, 0, d, lane);
    }
  #pragma unroll
    for (int e = 0; e < NE; ++e) {
      const int c = lane + 32 * e;
      if (c < d) {
        a.gQ[(long long)tk * d + c] = gq[e];
        a.gK[(long long)tk * d + c] = gk[e];
        a.gV[(long long)tk * d + c] = gv[e];
      }
    }
  }
}

__global__ void __launch_bounds__(256, 3) k_attn_bwd_s1(const __grid_constant__ AttnBwdArgs a) {
  extern __shared__ __align__(16) float att_sm[];
  const uint64_t seed_eff = eff_seed(a.seed, a.d_step);
  const int T = *a.dT;
  const int t0 = blockIdx.x * ATT_TOK;
  if (t0 >= T) return;
  pdl_wait(); pdl_go();
  attn_bwd_group(a, t0, T, att_sm, seed_eff);
}

// ---- backward: Q/K/V dgrad + LN1 backward --------------------------------------------------------------
struct QkvBwdArgs {
  const float *gQ, *gK, *gV, *gY, *X, *mean1, *rstd1, *ln_g;
  const op_t *Wqb, *Wkb, *Wvb;
  float *gQ1, *gXin;
  const int* dT; int d;
  float drop_p; uint64_t seed; const int* d_step;   // drop_p > 0 (first block only): gXin *= embedding-dropout mask (site 0)
};
constexpr size_t QKV_BWD_SMEM = 3 * WMAT_BYTES + 3 * ATILE_BYTES + FTILE_BYTES + 2 * TM * 4 + 16;
static_assert(3 * ATILE_BYTES >= FTILE_BYTES, "second fp32 tile aliases the operand tiles");

// One 32-token tile: gXin = gK.Wk^T + gV.Wv^T + LN1 backward(gQ.Wq^T + gY).  The K/V products run first, the Q product
// second; wait_kv() / wait_q() run in front of each and block until the shadows it reads have landed.
template <class WaitKV, class WaitQ>
__device__ __forceinline__ void qkv_bwd_tile(const QkvBwdArgs& a, int t0, int T, uint64_t seed_eff, op_t* __restrict__ A1, op_t* __restrict__ A2,
                                             op_t* __restrict__ A3, float* __restrict__ Ft, float* __restrict__ Ft2, float* __restrict__ rsq,
                                             float* __restrict__ rskv, const op_t* Wq_s, const op_t* Wk_s, const op_t* Wv_s,
                                             const float (&gam)[NE], WaitKV wait_kv, WaitQ wait_q) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int mt = warp & 1, ng = warp >> 1;
  const int d = a.d;
  {
    float gq[RPW][NE], gk[RPW][NE], gv[RPW][NE];
    load_rows(gq, a.gQ, t0, T, d, warp, lane);
    load_rows(gk, a.gK, t0, T, d, warp, lane);
    load_rows(gv, a.gV, t0, T, d, warp, lane);
    put_rows_scaled(A1, rsq, gq, warp, lane);
    put_rows_scaled(A2, rskv, gk, warp, lane, gv, A3);
  }
  float2 gyf[NT][2];
  load_frag(gyf, a.gY, t0, T, d, mt, ng, lane);
  __syncthreads();
  wait_kv();
  float acc_kv[NT][4], acc[NT][4];
  zero_acc(acc_kv);
  warp_gemm(A2 + mt * 16 * LDS, Wk_s + ng * (NT * 8) * LDS, acc_kv, lane);
  warp_gemm(A3 + mt * 16 * LDS, Wv_s + ng * (NT * 8) * LDS, acc_kv, lane);
  // rows of the LayerNorm-backward pass: loads in flight during the Q product
  float xv[RPW][NE], mean[RPW], rstd[RPW];
  load_rows(xv, a.X, t0, T, d, warp, lane);
  load_row_scalars(mean, a.mean1, t0, T, warp);
  load_row_scalars(rstd, a.rstd1, t0, T, warp);
  wait_q();
  zero_acc(acc);
  warp_gemm(A1 + mt * 16 * LDS, Wq_s + ng * (NT * 8) * LDS, acc, lane);
  // gQ1 = gQ . Wq^T + gY   (y = attn + q1)
  for_frag(acc, mt, ng, lane, [&](int j, int h, int r, int c, float v0, float v1) {
    if (c < d) {
      float q0 = 0.f, q1 = 0.f;
      if (t0 + r < T) {
        q0 = v0 * rsq[r] + gyf[j][h].x; q1 = v1 * rsq[r] + gyf[j][h].y;
        *reinterpret_cast<float2*>(a.gQ1 + (long long)(t0 + r) * d + c) = make_float2(q0, q1);
      }
      *reinterpret_cast<float2*>(Ft + r * FT_LD + c) = make_float2(q0, q1);
    }
  });
  __syncthreads();                       // every warp is done reading A1..A3 (Ft2 aliases them)
  for_frag(acc_kv, mt, ng, lane, [&](int j, int h, int r, int c, float v0, float v1) {
    if (c < d) *reinterpret_cast<float2*>(Ft2 + r * FT_LD + c) = make_float2(v0 * rskv[r], v1 * rskv[r]);
  });
  __syncthreads();
  // gXin = gK.Wk^T + gV.Wv^T + LN1 backward(gQ1)   [* embedding-dropout mask in the first block]
  float dx[RPW][NE];
  ln_bwd_rows(Ft, xv, mean, rstd, gam, d, warp, lane, dx);
  const DropSite ds0 = drop_site(seed_eff, 0u, a.drop_p);
#pragma unroll
  for (int rr = 0; rr < RPW; ++rr) {
    const int r = warp * RPW + rr, tk = t0 + r;
#pragma unroll
    for (int e = 0; e < NE; ++e) {
      const int c = lane + 32 * e;
      if (tk < T && c < d) {
        float v = dx[rr][e] + Ft2[r * FT_LD + c];
        if (a.drop_p > 0.f) v *= drop_mul(ds0, (uint64_t)tk * d + c);
        a.gXin[(long long)tk * d + c] = v;
      }
    }
  }
  __syncthreads();
}

__global__ void __launch_bounds__(NTHR, 1) k_qkv_bwd(const __grid_constant__ QkvBwdArgs a) {
  const uint64_t seed_eff = eff_seed(a.seed, a.d_step);
  extern __shared__ __align__(128) uint8_t smem[];
  op_t* Wsm = reinterpret_cast<op_t*>(smem);
  op_t* A1 = reinterpret_cast<op_t*>(smem + 3 * WMAT_BYTES);
  op_t* A2 = A1 + TM * LDS;
  op_t* A3 = A2 + TM * LDS;
  float* Ft2 = reinterpret_cast<float*>(smem + 3 * WMAT_BYTES);              // aliases A1..A3 after the GEMMs
  float* Ft = reinterpret_cast<float*>(smem + 3 * WMAT_BYTES + 3 * ATILE_BYTES);
  float* rsq = reinterpret_cast<float*>(smem + 3 * WMAT_BYTES + 3 * ATILE_BYTES + FTILE_BYTES);
  float* rskv = rsq + TM;
  const uint32_t bar = smem_u32(smem + 3 * WMAT_BYTES + 3 * ATILE_BYTES + FTILE_BYTES + 2 * TM * 4);
  const int T = *a.dT, d = a.d;
  const int ntiles = (T + TM - 1) / TM;
  if ((int)blockIdx.x >= ntiles) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) {
    mbar_init(bar, 1);
    mbar_expect_tx(bar, 3 * WMAT_BYTES);
    load_wmat(smem_u32(Wsm), a.Wqb, bar);
    load_wmat(smem_u32(Wsm) + WMAT_BYTES, a.Wkb, bar);
    load_wmat(smem_u32(Wsm) + 2 * WMAT_BYTES, a.Wvb, bar);
  }
  float gam[NE];
#pragma unroll
  for (int e = 0; e < NE; ++e) { const int c = lane + 32 * e; gam[e] = (c < d) ? a.ln_g[c] : 0.f; }
  pdl_wait(); pdl_go();
  __syncthreads();
  bool first = true;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
    qkv_bwd_tile(a, tile * TM, T, seed_eff, A1, A2, A3, Ft, Ft2, rsq, rskv, Wsm, Wsm + KP * LDS, Wsm + 2 * KP * LDS, gam,
                 [&] { if (first) { mbar_wait(bar, 0); first = false; } }, [] {});
}

// ---- backward: weight / bias / LayerNorm-parameter gradients of one block -----------------------------------------
// dW[c_in][c_out] = sum_t act[t][c_in] * grad[t][c_out] is a [150 x T] x [T x 150] product whose contraction
// runs over tokens.  TF32 mma.sync.m16n8k8: both operands are read straight from their natural [t][c] fp32 layout, no
// transposes and no range scaling (8-bit exponent), 10-bit mantissa.  A (split, problem) owns a contiguous range of
// 32-token tiles; the `splits` partials are reduced afterwards in index order (k_reduce_partials) -> deterministic.
// Problems 0..n_gemm-1: weight + bias gradients; problems n_gemm..: LayerNorm (beta, gamma) gradients
// (act = LN input x, grad = dout, xhat rebuilt from mean / rstd).
//   * a tile operand is ONE cp.async.bulk of the contiguous [32 tokens][d] block (19 200 B) completing on an mbarrier, the
//     next tile in flight behind the one being multiplied (ring depth: see WG2_NST).  Staging a tile with one 8-byte
//     cp.async per element pair is issue-bound: 6 us from entry to the first tile (profiles/r2/wgrad_phase_timeline.txt);
//   * shared-memory rows keep the global stride d, and the k slots of a k-step are mapped to tile rows so that the four
//     rows one fragment load touches are 4 apart (4 * 150 = 24 mod 32 banks): conflict-free without padding.  Summation
//     over k does not care which token sits in which slot as long as A and B agree;
//   * a (split, problem) is TWO CTAs of 4 warps, each owning 160 x 80 of the result (the tensor pipe of an SM is saturated by
//     4 warps with 25 independent accumulators each), so a launch of 3 problems x 21 splits covers 126 SMs;
//   * partials leave through shared memory as coalesced 8-byte row stores.
// Bias and LayerNorm-parameter sums run in token order.
constexpr int WG_TK = 32;                     // tokens per staged tile
constexpr int WG_MAXP = 3;                    // problems of one launch (the largest piece: the Q, K and V matrices)
struct WgradProb { const float *act, *grad, *mean, *rstd; float *out0, *out1; };   // GEMM: out0 = pW, out1 = pb; LN: out0 = pbeta, out1 = pgamma
struct WgradArgs { WgradProb p[WG_MAXP]; int n_gemm, n_ln; const int* dT; int d; long long split_stride; };

// fp32 -> tf32, round to nearest with ties away from zero: cvt.rna.tf32.f32 as ONE integer add on the bit pattern (half an
// ulp of the 10-bit mantissa added to the magnitude; the tensor core ignores the low 13 bits, so they need no masking).
// Same operand values as the conversion instruction for every finite input, but on the full-rate integer pipe: the 30
// conversions per 25 mma of a k-step cost as much issue time as the products themselves.
__device__ __forceinline__ uint32_t to_tf32(float v) { return __float_as_uint(v) + 0x1000u; }
__device__ __forceinline__ void mma_tf32(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

constexpr int WG2_THR = 128;
// ring depth (-DADER_WG2_NST=n): measured in the step on one box, 200 graph replays each, two runs per depth
// (profiles/r2b/wgrad2_ring_depth.txt): 5 stages (205 KB) 0.2807 / 0.2804 ms, 3 stages (123 KB) 0.2799 / 0.2801,
// 2 stages (82 KB) 0.2789 / 0.2780 (end to end 0.289 against 0.294).  Small but repeatable: the kernel runs beside the
// data-gradient chain, where a smaller footprint packs better than an earlier first tile
#ifndef ADER_WG2_NST
#define ADER_WG2_NST 2
#endif
constexpr int WG2_NST = ADER_WG2_NST;
constexpr int WG2_OPB = WG_TK * KP * 4;                      // bytes of one operand slot (d <= 160)
constexpr int WG2_STG_LD = 88;                               // staging row stride of the 160 x 80 result block
constexpr size_t WGRAD2_SMEM = (size_t)WG2_NST * 2 * WG2_OPB + 64;
static_assert(160 * WG2_STG_LD * 4 <= WG2_NST * 2 * WG2_OPB, "result staging must fit the ring");    // 56 320 B: two stages suffice

__global__ void __launch_bounds__(WG2_THR) k_wgrad2(const __grid_constant__ WgradArgs a) {
  extern __shared__ __align__(128) float wsm[];
  const int T = *a.dT, d = a.d;
  const int ntiles = (T + WG_TK - 1) / WG_TK;
  const int chunk = (ntiles + gridDim.x - 1) / gridDim.x;
  const int tile_lo = blockIdx.x * chunk, tile_hi = min(ntiles, tile_lo + chunk);
  const int n_my = max(tile_hi - tile_lo, 0);
  const bool is_ln = (int)blockIdx.y >= 2 * a.n_gemm;
  const int prob = is_ln ? a.n_gemm + ((int)blockIdx.y - 2 * a.n_gemm) : ((int)blockIdx.y >> 1);
  const int half = is_ln ? 0 : ((int)blockIdx.y & 1);
  const WgradProb pr = a.p[prob];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t4 = lane & 3;
  const int wm = warp & 1, wn = warp >> 1;           // warp block: rows wm*80.., columns half*80 + wn*40..
  const uint32_t bar0 = smem_u32(reinterpret_cast<char*>(wsm) + (size_t)WG2_NST * 2 * WG2_OPB);
  auto issue = [&](int li) {                         // thread 0: both operands of local tile li into stage li % NST
    const int t0 = (tile_lo + li) * WG_TK;
    const int rv = min(WG_TK, T - t0) & ~1;          // bulk copies move whole 16-byte units: an even number of rows
    const uint32_t bytes = (uint32_t)(rv * d * 4);
    const int s = li % WG2_NST;
    const uint32_t bar = bar0 + 8 * s;
    mbar_expect_tx(bar, 2 * bytes);
    if (bytes) {
      const uint32_t dst = smem_u32(reinterpret_cast<char*>(wsm) + (size_t)s * 2 * WG2_OPB);
      bulk_g2s(dst, pr.act + (long long)t0 * d, bytes, bar);
      bulk_g2s(dst + WG2_OPB, pr.grad + (long long)t0 * d, bytes, bar);
    }
  };
  if (tid == 0) {
    for (int s = 0; s < WG2_NST; ++s) mbar_init(bar0 + 8 * s, 1);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    for (int li = 0; li < n_my && li < WG2_NST; ++li) issue(li);
  }
  float acc[5][5][4];
#pragma unroll
  for (int i = 0; i < 5; ++i)
#pragma unroll
    for (int j = 0; j < 5; ++j) { acc[i][j][0] = acc[i][j][1] = acc[i][j][2] = acc[i][j][3] = 0.f; }
  float cs0[2] = {0.f, 0.f}, cs1[2] = {0.f, 0.f};    // GEMM: [0] = bias column half*80 + tid (tid < 80); LN: columns tid, tid + 128
  __syncthreads();                                   // barrier words initialised before anyone waits on them
#pragma unroll 1
  for (int li = 0; li < n_my; ++li) {
    const int s = li % WG2_NST;
    float* As = reinterpret_cast<float*>(reinterpret_cast<char*>(wsm) + (size_t)s * 2 * WG2_OPB);
    float* Bs = reinterpret_cast<float*>(reinterpret_cast<char*>(As) + WG2_OPB);
    const int t0 = (tile_lo + li) * WG_TK;
    const int rv = min(WG_TK, T - t0);
    if (rv < WG_TK) {                                // last tile of the batch: odd last row by hand, rows beyond T zero
      const int re = rv & ~1;
      for (int idx = tid; idx < (WG_TK - re) * d; idx += WG2_THR) {
        const int r = re + idx / d, c = idx % d;
        const bool ok = r < rv;
        As[r * d + c] = ok ? pr.act[(long long)(t0 + r) * d + c] : 0.f;
        Bs[r * d + c] = ok ? pr.grad[(long long)(t0 + r) * d + c] : 0.f;
      }
      __syncthreads();
    }
    mbar_wait(bar0 + 8 * s, (uint32_t)(li / WG2_NST) & 1u);
    if (!is_ln) {
#pragma unroll
      for (int ks = 0; ks < WG_TK / 8; ++ks) {
        // k slot t4 <-> tile row R + 2q + 4*t4, k slot t4 + 4 <-> the row below it (R = 16 * (ks / 2), q = ks % 2)
        const int row = (ks >> 1) * 16 + (ks & 1) * 2 + 4 * t4;
        const float* ar = As + row * d + wm * 80 + g;
        const float* br = Bs + row * d + half * 80 + wn * 40 + g;
        uint32_t bf[5][2];
#pragma unroll
        for (int j = 0; j < 5; ++j) { bf[j][0] = to_tf32(br[j * 8]); bf[j][1] = to_tf32(br[d + j * 8]); }
#pragma unroll
        for (int i = 0; i < 5; ++i) {
          const uint32_t a0 = to_tf32(ar[i * 16]), a1 = to_tf32(ar[i * 16 + 8]);
          const uint32_t a2 = to_tf32(ar[d + i * 16]), a3 = to_tf32(ar[d + i * 16 + 8]);
#pragma unroll
          for (int j = 0; j < 5; ++j) mma_tf32(acc[i][j], a0, a1, a2, a3, bf[j][0], bf[j][1]);
        }
      }
      const int c = half * 80 + tid;
      if (tid < 80 && c < d) {                        // bias gradient: column sums of grad, token order
#pragma unroll 8
        for (int r = 0; r < WG_TK; ++r) cs0[0] += Bs[r * d + c];
      }
    } else {                                          // LayerNorm parameter gradients (rows beyond T are zero: gq = 0)
#pragma unroll
      for (int r8 = 0; r8 < WG_TK; r8 += 8) {
        float mu[8], rs[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) { const int t = min(t0 + r8 + j, T - 1); mu[j] = __ldg(pr.mean + t); rs[j] = __ldg(pr.rstd + t); }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const int c = tid + q * WG2_THR;
          if (c < d) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float gq = Bs[(r8 + j) * d + c];
              cs0[q] += gq;
              cs1[q] += gq * ((As[(r8 + j) * d + c] - mu[j]) * rs[j]);
            }
          }
        }
      }
    }
    __syncthreads();                                  // every reader of stage s is done: refill it
    if (tid == 0 && li + WG2_NST < n_my) issue(li + WG2_NST);
  }
  const long long so = (long long)blockIdx.x * a.split_stride;
  if (!is_ln) {
    // 160 x 80 block -> shared memory (the ring is idle: every copy was waited for) -> coalesced 8-byte row stores
    float* stg = wsm;
#pragma unroll
    for (int i = 0; i < 5; ++i)
#pragma unroll
      for (int j = 0; j < 5; ++j) {
        const int m = wm * 80 + i * 16 + g, n = wn * 40 + j * 8 + 2 * t4;
        *reinterpret_cast<float2*>(stg + m * WG2_STG_LD + n) = make_float2(acc[i][j][0], acc[i][j][1]);
        *reinterpret_cast<float2*>(stg + (m + 8) * WG2_STG_LD + n) = make_float2(acc[i][j][2], acc[i][j][3]);
      }
    __syncthreads();
    const int ncol2 = min(80, d - half * 80) / 2;     // float2 columns of this half that exist (d is even)
    float* out = pr.out0 + so + half * 80;
    for (int f = tid; f < d * 40; f += WG2_THR) {
      const int m = f / 40, c2 = f % 40;
      if (c2 < ncol2) *reinterpret_cast<float2*>(out + (long long)m * d + 2 * c2) = *reinterpret_cast<const float2*>(stg + m * WG2_STG_LD + 2 * c2);
    }
    const int c = half * 80 + tid;
    if (tid < 80 && c < d) pr.out1[so + c] = cs0[0];
  } else {
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int c = tid + q * WG2_THR;
      if (c < d) { pr.out0[so + c] = cs0[q]; pr.out1[so + c] = cs1[q]; }
    }
  }
}

}  // namespace fz
}  // namespace ader
