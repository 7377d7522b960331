// tcgen05 / TMEM / TMA / mbarrier building blocks shared by the tensor-core kernels of libader_b200
// (logits_tc.cu: logits + CE + distillation; eval_tc.cu: full-vocabulary scoring with a rank epilogue).
#pragma once
#include "common.cuh"
#include <cuda.h>            // CUtensorMap (types only: the encoder is fetched through cudaGetDriverEntryPoint, no libcuda link)
#include <cuda_bf16.h>

namespace ader {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int* err) {
  uint32_t done = 0;
  for (uint32_t spin = 0; !done; ++spin) {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    if (!done && spin > (1u << 24)) {            // a broken pipeline must not hang the GPU
      if (err) atomicExch(err, 1);
      __trap();
    }
  }
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
               ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// 32 consecutive TMEM columns of this thread's lane
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31]) :: "memory");
}
__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
// wait for outstanding tcgen05.ld; the registers are passed as in/out operands so the compiler cannot
// schedule their first use ahead of the wait
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31]) :: "memory");
}
// 16 consecutive TMEM columns of this thread's lane (no wait) / wait with the registers pinned behind it
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait16(uint32_t (&r)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]) :: "memory");
}
__device__ __forceinline__ float ex2(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

// instruction descriptor (cute::UMMA::InstrDescriptor): c=F32 [4,6), a=BF16 [7,10), b=BF16 [10,13),
// a_major [15], b_major [16], N>>3 [17,23), M>>4 [24,29)
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, int a_mn, int b_mn, int a_neg = 0) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_neg << 13) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
// shared-memory matrix descriptor, SWIZZLE_128B (cute::UMMA::SmemDescriptor): start>>4 [0,14), LBO>>4 [16,30),
// SBO>>4 [32,46), version=1 [46,48), layout_type=2 [61,64)
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | (1ull << 46) | (2ull << 61);
}
}  // namespace tc
}  // namespace ader

// ---- host: TMA tensor maps over row-major bf16 matrices ------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
// bf16 matrix [rows][cols], row pitch in bytes (multiple of 16); box = 64 columns (128 B, one swizzle span) x 128 rows
static inline int make_map2d(CUtensorMap* tm, const void* base, uint64_t cols, uint64_t rows, uint64_t pitch_bytes, uint32_t box_rows = 128) {
  static const EncodeTiledFn enc = [] {          // one lookup per process: the entry point does not depend on the device
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qr) == cudaSuccess) return (EncodeTiledFn)fn;
    cudaGetLastError();
    return (EncodeTiledFn)nullptr;
  }();
  if (!enc) return ::ader::fail(-3, "loss_tc: cuTensorMapEncodeTiled is unavailable (driver too old?)");
  const cuuint64_t gdim[2] = {cols, rows};
  const cuuint64_t gstr[1] = {pitch_bytes};
  const cuuint32_t box[2] = {64, box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return ::ader::fail(-3, "loss_tc: cuTensorMapEncodeTiled failed (%d)", (int)r);
  return 0;
}
