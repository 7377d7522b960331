// Generic strided fp32 GEMM with fused epilogues -- the exact-arithmetic workhorse of the
// parity path (encoder dense layers, weight gradients with deterministic split-K, materialised
// logits for the fp32 reference mode).  64x64 tiles, the whole K chunk (160) staged in shared memory by
// cp.async with every load in flight at once, 256 threads, 4x4 register micro-tiles.
// Summation order over k is fixed (sequential inside a split, splits reduced in index order by
// reduce_partials) so results are run-to-run deterministic.
#include "common.cuh"

namespace ader {

void gemm_defaults(GemmArgs& g) {
  g.A = nullptr; g.B = nullptr; g.C = nullptr;
  g.a_rs = g.a_cs = g.b_rs = g.b_cs = g.c_rs = g.c_cs = 0;
  g.M = g.N = g.K = 0; g.dM = nullptr; g.dK = nullptr;
  g.bias = nullptr; g.resid = nullptr; g.resid_ld = 0; g.relu_mask = nullptr; g.mask_ld = 0;
  g.relu = 0; g.accumulate = 0; g.alpha = 1.0f; g.splits = 1; g.split_stride = 0; g.colsum = nullptr;
  g.drop_p = 0.f; g.drop_seed = 0; g.drop_site = 0;
}

constexpr int BM = 64, BN = 64;
constexpr int KC = 160;            // K chunk staged in shared memory at once (covers K = d = 150 in one go)
constexpr int LDK = KC + 4;        // row stride of a k-contiguous tile  ([rows][k]);  164 % 32 == 4
constexpr int LDM = BM + 4;        // row stride of an m/n-contiguous tile ([k][rows])
constexpr int A_FLOATS = (BM * LDK > KC * LDM) ? BM * LDK : KC * LDM;
constexpr size_t SGEMM_SMEM = sizeof(float) * 2 * A_FLOATS;

__device__ __forceinline__ void cp_async8(float* dst, const float* src, int src_bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async4(float* dst, const float* src, int src_bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src), "r"(src_bytes) : "memory");
}

// Stage a [rows x KC] operand tile.  KFAST: k is the contiguous global dimension -> smem [rows][LDK];
// else rows are contiguous -> smem [k][LDM].  Out-of-range elements are zero-filled by cp.async.
template <bool KFAST>
__device__ __forceinline__ void stage_tile(float* sm, const float* __restrict__ G, long long r_stride, long long k_stride,
                                           int r0, int R, int k0, int k_hi, bool vec2) {
  const int tid = threadIdx.x;
  if (vec2) {
    constexpr int PAIRS = BM * KC / 2;
#pragma unroll 4
    for (int idx = tid; idx < PAIRS; idx += 256) {
      int rr, kk;
      if (KFAST) { kk = (idx % (KC / 2)) * 2; rr = idx / (KC / 2); } else { rr = (idx % (BM / 2)) * 2; kk = idx / (BM / 2); }
      const int gr = r0 + rr, gk = k0 + kk;
      int valid;
      if (KFAST) valid = (gr < R) ? max(0, min(2, k_hi - gk)) : 0; else valid = (gk < k_hi) ? max(0, min(2, R - gr)) : 0;
      const float* src = valid ? G + (long long)gr * r_stride + (long long)gk * k_stride : G;
      float* dst = KFAST ? sm + rr * LDK + kk : sm + kk * LDM + rr;
      cp_async8(dst, src, valid * 4);
    }
  } else {
    constexpr int ELEMS = BM * KC;
#pragma unroll 4
    for (int idx = tid; idx < ELEMS; idx += 256) {
      int rr, kk;
      if (KFAST) { kk = idx % KC; rr = idx / KC; } else { rr = idx % BM; kk = idx / BM; }
      const int gr = r0 + rr, gk = k0 + kk;
      const bool ok = gr < R && gk < k_hi;
      const float* src = ok ? G + (long long)gr * r_stride + (long long)gk * k_stride : G;
      float* dst = KFAST ? sm + rr * LDK + kk : sm + kk * LDM + rr;
      cp_async4(dst, src, ok ? 4 : 0);
    }
  }
}

template <bool A_KFAST, bool B_KFAST>
__device__ __forceinline__ void sgemm_body(const GemmArgs& g, int a_vec2, int b_vec2, const int z) {
  extern __shared__ __align__(16) float sg_smem[];
  float* As = sg_smem;
  float* Bs = sg_smem + A_FLOATS;
  const int M = g.dM ? *g.dM : g.M;
  const int K = g.dK ? *g.dK : g.K;
  const int N = g.N;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  if (m0 >= M || n0 >= N) return;
  const int kchunk = ((K + g.splits - 1) / g.splits + 3) / 4 * 4;
  const int k_lo = z * kchunk;
  const int k_hi = min(K, k_lo + kchunk);

  const int tid = threadIdx.x;
  const int ty = tid >> 4, tx = tid & 15;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  float bsum[4] = {0.f, 0.f, 0.f, 0.f};
  const bool do_colsum = (g.colsum != nullptr) && (blockIdx.y == 0) && (ty == 0);

  for (int k0 = k_lo; k0 < k_hi; k0 += KC) {
    // A(m,k): row stride a_rs, k stride a_cs.  B(k,n): "rows" are n (stride b_cs), k stride b_rs.
    stage_tile<A_KFAST>(As, g.A, g.a_rs, g.a_cs, m0, M, k0, k_hi, a_vec2 != 0);
    stage_tile<B_KFAST>(Bs, g.B, g.b_cs, g.b_rs, n0, N, k0, k_hi, b_vec2 != 0);
    asm volatile("cp.async.commit_group;\n cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    const int kc = min(KC, (k_hi - k0 + 3) / 4 * 4);
    for (int kk = 0; kk < kc; kk += 4) {
      float av[4][4], bv[4][4];       // [q = k offset][i / j]
      if (A_KFAST) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float4 a = *reinterpret_cast<const float4*>(&As[(ty * 4 + i) * LDK + kk]);
          av[0][i] = a.x; av[1][i] = a.y; av[2][i] = a.z; av[3][i] = a.w;
        }
      } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float4 a = *reinterpret_cast<const float4*>(&As[(kk + q) * LDM + ty * 4]);
          av[q][0] = a.x; av[q][1] = a.y; av[q][2] = a.z; av[q][3] = a.w;
        }
      }
      if (B_KFAST) {                  // columns tx + 16 j: 8 consecutive rows x 16 B hit distinct banks (LDK % 32 == 4)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float4 b = *reinterpret_cast<const float4*>(&Bs[(tx + 16 * j) * LDK + kk]);
          bv[0][j] = b.x; bv[1][j] = b.y; bv[2][j] = b.z; bv[3][j] = b.w;
        }
      } else {                        // columns tx*4 + j
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float4 b = *reinterpret_cast<const float4*>(&Bs[(kk + q) * LDM + tx * 4]);
          bv[q][0] = b.x; bv[q][1] = b.y; bv[q][2] = b.z; bv[q][3] = b.w;
        }
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[q][i], bv[q][j], acc[i][j]);
        if (do_colsum) {
#pragma unroll
          for (int j = 0; j < 4; ++j) bsum[j] += bv[q][j];
        }
      }
    }
    __syncthreads();
  }

  float* C = g.C + (long long)z * g.split_stride;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int gm = m0 + ty * 4 + i;
    if (gm >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int gn = n0 + (B_KFAST ? tx + 16 * j : tx * 4 + j);
      if (gn >= N) continue;
      float v = g.alpha * acc[i][j];
      if (g.bias) v += g.bias[gn];
      if (g.relu) v = fmaxf(v, 0.f);
      if (g.relu_mask) v = (g.relu_mask[(long long)gm * g.mask_ld + gn] > 0.f) ? v : 0.f;
      if (g.drop_p > 0.f) v *= drop_scale(g.drop_seed, g.drop_site, (uint64_t)gm * N + gn, g.drop_p);
      if (g.resid) v += g.resid[(long long)gm * g.resid_ld + gn];
      long long o = (long long)gm * g.c_rs + (long long)gn * g.c_cs;
      if (g.accumulate) v += C[o];
      C[o] = v;
    }
  }
  if (do_colsum) {
    float* cs = g.colsum + (long long)z * g.split_stride;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int gn = n0 + (B_KFAST ? tx + 16 * j : tx * 4 + j);
      if (gn < N) cs[gn] = bsum[j];
    }
  }
}

template <bool A_KFAST, bool B_KFAST>
__global__ void __launch_bounds__(256, 2) sgemm_kernel(GemmArgs g, int a_vec2, int b_vec2) {
  sgemm_body<A_KFAST, B_KFAST>(g, a_vec2, b_vec2, blockIdx.z);
}

template <bool AK, bool BK_>
static int launch_one(const GemmArgs& g, dim3 grid, int av, int bv, cudaStream_t st) {
  if (int e = kernel_ready<sgemm_kernel<AK, BK_>>((int)SGEMM_SMEM, "sgemm_kernel")) return e;
  sgemm_kernel<AK, BK_><<<grid, 256, SGEMM_SMEM, st>>>(g, av, bv);
  return 0;
}

int launch_gemm(const GemmArgs& g, cudaStream_t st) {
  if (g.M <= 0 || g.N <= 0) return 0;
  dim3 grid(cdiv(g.N, BN), cdiv(g.M, BM), g.splits);
  if (grid.y > 65535u) return fail(-2, "sgemm: M=%d too large for grid.y", g.M);
  const bool ak = (g.a_cs == 1), bk = (g.b_rs == 1);       // k contiguous in A / in B
  // 8-byte cp.async needs: unit stride along the fast dim, even stride along the other, 8 B aligned base
  auto vec_ok = [](const float* p, long long fast, long long other) {
    return fast == 1 && (other % 2 == 0) && ((uintptr_t)p % 8 == 0);
  };
  const int av = ak ? vec_ok(g.A, g.a_cs, g.a_rs) : vec_ok(g.A, g.a_rs, g.a_cs);
  const int bv = bk ? vec_ok(g.B, g.b_rs, g.b_cs) : vec_ok(g.B, g.b_cs, g.b_rs);
  const int e = ak && bk ? launch_one<true, true>(g, grid, av, bv, st)
              : ak       ? launch_one<true, false>(g, grid, av, bv, st)
              : bk       ? launch_one<false, true>(g, grid, av, bv, st)
                         : launch_one<false, false>(g, grid, av, bv, st);
  if (e) return e;
  ADER_CHECK_LAUNCH("sgemm_kernel");
  return 0;
}

}  // namespace ader
