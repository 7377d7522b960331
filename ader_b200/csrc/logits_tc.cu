// Fused output projection + online-softmax CE + ADER distillation on the 5th-gen tensor cores
// (tcgen05.mma, accumulators in TMEM), ADER.py:88-93 / 108-138.  The [M, V] logits never touch HBM.
//
// Operand format in HBM: the bf16 shadows of the item table and of `rep` are plain row-major bf16 matrices [rows][160]
// (d = 150 zero-padded to 160, rows padded to whole 128-row tiles).  Tiles reach shared memory through TMA tensor maps
// (cp.async.bulk.tensor, SWIZZLE_128B) and every MMA operand is a canonical 128-byte-swizzled UMMA layout:
//   a tile = 128 rows x 192 k in shared memory = three "regions" of [128 rows][64 k = 128 B] (16 KB each; the TMA box of
//   region 2 hangs over the 160-column matrix and is zero-filled, so nothing beyond column 159 is ever read from HBM);
//   * K-major operand of  S = rep . E^T : k-step s (16 k) starts at region s/4, byte (s%4)*32; SBO = 1024 (8-row groups);
//   * MN-major operand (N or M = the 64 contiguous elements of a region row, K = tile row) of the gradient products:
//     k-step s (16 rows) starts at byte s*2048; LBO = 16384 (next region = next 64 MN elements), SBO = 1024.
//   The dS tile the epilogue writes ([128 m][128 v] bf16 = two regions, 16-byte chunks XOR-swizzled by row & 7) is the
//   K-major A operand of dRep = dS . E (M = m) and, read MN-major, the A operand of dE = dS^T . rep (M = v).
// Swizzled operands are what make the gradient products cheap: read MN-major out of pre-tiled no-swizzle operands, the
// second product ran at ~1.9 us per tile against ~0.4 us for the first (profiles/r1f).
//
// Kernel roles (320 threads): warp 0 = TMA producer, warp 1 = MMA issuer (one elected lane) +
// TMEM allocator, warps 2..9 = epilogue: TMEM lane quarter = warp % 4, column half = (warp - 2) / 4, so
// two threads share one logits row (64 of the 128 tile columns each).
//   MODE_FWD : per (row-tile, vocab-chunk) CTA: S tiles -> online (max, sumexp), label logit, KD dot
//   MODE_DREP: same loop; dS (bf16) is staged in shared memory and a second MMA accumulates
//              dRep[128, 160] in TMEM across the CTA's vocab tiles
//   MODE_DE  : per vocab-tile CTA, loops over row tiles; second MMA accumulates dE[128, 160]
//
// Distillation rows (ADER.py:133-137) enter by LINEARITY, not inside the S-tile epilogues.  With
// P = softmax(teacher) over the V_prev columns,  KD_i = lse_i(s[:V_prev]) - rep_i . u_i  and
// dS_i = coef * (softmax(s_i[:V_prev]) - P_i),  where  u = P . E  ([M_e, V_prev] x [V_prev, d]).  So in the
// three kernels above a distillation row is a label-free softmax row of width V_prev (no teacher traffic,
// no extra exponentials), and the teacher contributes through two more tensor-core products on bf16 tiles
// of Pc = coef * P (k_teacher_rows16: coalesced one-pass read of the fp32 teacher rows):
//   MODE_TU  : uc = Pc . E partials over a vocabulary chunk (second-MMA datapath of DREP with the "dS" operand
//              loaded instead of computed)   -> loss dot = rep.uc / coef,  d_rep -= uc
//   MODE_DE  : after its row-tile loop the CTA of a vocabulary tile < V_prev runs one more second-MMA per exemplar
//              row tile with the A operand NEGATED in the instruction descriptor: dE[v] -= Pc^T . rep
// A frozen teacher (AderLossArgs.teacher_rep) builds Pc from a snapshot of the previous model instead of stored logits:
// T = trep . E_prev^T tiles go through MODE_FWD on the snapshot's operands (label-free rows of width V_prev: the teacher's
// online (max, sumexp) per chunk, merged into lse_t), then
//   MODE_TP  : recomputes the T tiles and writes Pc = coef * exp(T - lse_t) as bf16 straight into the matrix MODE_TU / MODE_DE read
#include "tc_common.cuh"

namespace ader {
namespace tc {

constexpr int TILE = 128;
constexpr int KP = 160;                       // padded feature dim
static_assert(KP == PATH_TC_MAX_D, "ADER_PATH_LOSS_TC: rows of d <= KP columns");
constexpr int TILE_BYTES = TILE * KP * 2;     // 40960: one 128-row tile of an operand matrix in HBM
constexpr int DS_BYTES = TILE * TILE * 2;     // 32768: one 128 x 128 tile of the teacher-probability matrix in HBM
constexpr int KSTEPS1 = KP / 16;              // 10 MMAs per S tile
constexpr int KSTEPS2 = TILE / 16;            // 8 MMAs per gradient tile
constexpr float LOG2E = 1.4426950408889634f;

enum { MODE_FWD = 0, MODE_DREP = 1, MODE_DE = 2, MODE_TU = 3, MODE_TP = 4 };
__host__ __device__ constexpr bool is_teach(int mode) { return mode == MODE_TU; }
__host__ __device__ constexpr bool fwd_like(int mode) { return mode == MODE_FWD || mode == MODE_TP; }   // S tiles only, no second product

struct TcArgs {
  int M, V, V_total, n_mtiles, n_vtiles, n_chunks;   // V = columns of this shard, V_total = max_item
  // loss description
  int n_train, n_ex, V_prev, mode;
  float coef_train, coef_ex;    // 1/n_train, lambda/n_ex
  const int* pos; const int* ex_pos;
  int v_off;                    // vocab-parallel: global column of local column 0 (multiple of 128); V is the LOCAL width
  const float* lse;             // [M]   (backward)
  const float* lse_t;           // [n_ex] teacher log-sum-exp
  float* stats;                 // FWD: [n_chunks*2][M][4] = (max, sumexp, label logit, kd dot) per column half
  float* drep_part;             // DREP: [n_chunks][n_mtiles*128][160]
  float* grad_table;            // DE: grad + d (row of item 1), row stride d
  int d;
  int* err;                     // device error flag (barrier timeout)
  // teacher products (MODE_TU, teacher tail of MODE_DE)
  int x0_t, n_et, n_vtp, n_chunks_t;   // first row tile holding exemplar rows, their count, teacher vocab tiles, TU chunks
  float* u_part;                // TU: [n_chunks_t][n_et*128][160]
  // MODE_TP (frozen teacher): output Pc matrix [n_mtiles*128][n_vtiles*128] bf16; rows [t_row_lo, t_row_hi) are exemplars
  __nv_bfloat16* pt_out;
  int t_row_lo, t_row_hi;
};

// per-row description of the loss (shared by all modes)
struct RowInfo {
  int kind;           // 0 none (row >= M), 1 softmax row of width vlim (one-hot label, or label = -1 for distillation rows)
  int vlim;           // softmax width
  int label;          // 0-based column of the one-hot label (kind 1), else -1
  float coef;         // dS scale
  float lse2;         // lse * log2(e)  (backward)
};
__device__ __forceinline__ RowInfo row_info(const TcArgs& a, int gm, bool bwd) {
  // all column indices inside the kernel are LOCAL to this vocabulary shard: labels, softmax widths and the
  // teacher row pointer are shifted by v_off here (a label outside the shard simply never matches)
  RowInfo r; r.kind = 0; r.vlim = 0; r.label = -1; r.coef = 0.f; r.lse2 = 0.f;
  if (gm >= a.M) return r;
  int vlim_g;
  if (gm < a.n_train) { r.kind = 1; vlim_g = a.V_total; r.label = a.pos[gm] - 1 - a.v_off; r.coef = a.coef_train; }
  else if (a.mode == 2) { r.kind = 1; vlim_g = a.V_total; r.label = a.ex_pos[gm - a.n_train] - 1 - a.v_off; r.coef = a.coef_ex; }
  else { r.kind = 1; vlim_g = a.V_prev; r.coef = a.coef_ex; }   // distillation row: softmax over V_prev, no label (teacher term: MODE_TU/TG)
  r.vlim = max(0, min(a.V, vlim_g - a.v_off));
  if (bwd) r.lse2 = a.lse[gm] * LOG2E;
  return r;
}

constexpr int NTHREADS = 320, NEPI = 256;
constexpr int DE_LD = 164;     // fp32 row stride of the dE staging tile (164 % 32 == 4: conflict-free 16-byte row writes)

// Optional per-CTA timeline (debug builds only: -DADER_TC_TIMELINE): clock64 stamps of the pipeline roles.
#ifdef ADER_TC_TIMELINE
__device__ long long g_tl[3][192][64];
__device__ __forceinline__ long long gtimer() { long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define TL2(slot) do { if (blockIdx.x < 192 && MODE < 3) g_tl[MODE][blockIdx.x][slot] = gtimer(); } while (0)
#else
#define TL2(slot) do { } while (0)
#endif

constexpr int REG2 = 16384;                  // one region: 128 rows x 128 B
constexpr int TILE2_BYTES = 3 * REG2;        // 49152
constexpr int DS2_BYTES = 2 * REG2;          // 32768
constexpr int ROW16 = KP;                    // bf16 row pitch (elements) of the HBM operand matrices
__host__ __device__ constexpr int n_stages2(int mode) { return 3; }
__host__ __device__ constexpr int n_ds2(int mode) { return fwd_like(mode) ? 0 : 1; }
constexpr int smem_tc2(int mode) { return 1024 + (1 + n_stages2(mode)) * TILE2_BYTES + n_ds2(mode) * DS2_BYTES + 256; }
static_assert(TILE * DE_LD * 4 <= n_stages2(MODE_DREP) * TILE2_BYTES, "dE staging tile must fit the streamed-tile ring");

// 128 rows x 160 (192) k starting at matrix row `row0`
__device__ __forceinline__ void load_tile2(uint32_t dst, const CUtensorMap* tm, int row0, uint32_t bar) {
  mbar_expect_tx(bar, TILE2_BYTES);
#pragma unroll
  for (int j = 0; j < 3; ++j) tma_load_2d(dst + j * REG2, tm, 64 * j, row0, bar);
}
// 128 rows x 128 columns of the teacher-probability matrix starting at (row0, col0)
__device__ __forceinline__ void load_ds2(uint32_t dst, const CUtensorMap* tm, int col0, int row0, uint32_t bar) {
  mbar_expect_tx(bar, DS2_BYTES);
#pragma unroll
  for (int j = 0; j < 2; ++j) tma_load_2d(dst + j * REG2, tm, col0 + 64 * j, row0, bar);
}
__device__ __forceinline__ uint64_t desc_kmajor(uint32_t base, int kstep) {      // 16 k of a K-major tile
  return make_desc_sw128(base + (kstep >> 2) * REG2 + (kstep & 3) * 32, 16, 1024);
}
__device__ __forceinline__ uint64_t desc_mnmajor(uint32_t base, int kstep) {     // 16 rows (= K) of an MN-major tile
  return make_desc_sw128(base + kstep * 2048, REG2, 1024);
}

template <int MODE>
__global__ void __launch_bounds__(NTHREADS, 1) k_tc2(TcArgs a, const __grid_constant__ CUtensorMap tm_rep,
                                                     const __grid_constant__ CUtensorMap tm_e,
                                                     const __grid_constant__ CUtensorMap tm_pt) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);   // SW128 atoms: 1 KB aligned
  constexpr int NST = n_stages2(MODE), ND = n_ds2(MODE);
  uint8_t* sX = smem;
  uint8_t* sY = smem + TILE2_BYTES;
  uint8_t* sD = smem + (1 + NST) * TILE2_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (1 + NST) * TILE2_BYTES + ND * DS2_BYTES);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 24);
  const uint32_t bar0 = smem_u32(bars);
  auto BAR = [&](int i) { return bar0 + 8u * i; };
  constexpr int B_XFULL = 0, B_YFULL = 1, B_YEMPTY = 5, B_TFULL = 9, B_TEMPTY = 11, B_DSFULL = 13, B_DSEMPTY = 15, B_ACC = 17, B_PFULL = 18;
  constexpr int NDS = ND > 0 ? ND : 1;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#ifdef ADER_TC_TIMELINE
  if (threadIdx.x == 0 && blockIdx.x < 192 && MODE < 3) { const long long gt = gtimer(); g_tl[MODE][blockIdx.x][0] = gt; g_tl[MODE][blockIdx.x][1] = gt; }
#endif

  // ---- work assignment ---------------------------------------------------------------------------
  int x_tile, y_lo, y_hi, chunk = 0;    // stationary tile index, streamed tile range, vocabulary chunk
  if (MODE == MODE_DE) { x_tile = blockIdx.x; y_lo = 0; y_hi = a.n_mtiles; }
  else if (MODE == MODE_TU) {
    x_tile = a.x0_t + blockIdx.x % a.n_et; chunk = blockIdx.x / a.n_et;                            // exemplar row tile; vocab chunk
    y_lo = (int)((long long)chunk * a.n_vtp / a.n_chunks_t);
    y_hi = (int)((long long)(chunk + 1) * a.n_vtp / a.n_chunks_t);
  } else {
    x_tile = blockIdx.x % a.n_mtiles; chunk = blockIdx.x / a.n_mtiles;
    y_lo = (int)((long long)chunk * a.n_vtiles / a.n_chunks);           // balanced split of the vocabulary tiles
    y_hi = (int)((long long)(chunk + 1) * a.n_vtiles / a.n_chunks);
  }
  const int n_it = max(0, y_hi - y_lo);
  const CUtensorMap* tmX = (MODE == MODE_DE) ? &tm_e : &tm_rep;
  const CUtensorMap* tmY = (MODE == MODE_DE) ? &tm_rep : &tm_e;
  // DE: teacher iterations appended after the row-tile loop (this vocabulary tile holds teacher columns)
  const int n_tt = (MODE == MODE_DE && x_tile < a.n_vtp) ? a.n_et : 0;

  // ---- setup ---------------------------------------------------------------------------------------
  if (threadIdx.x == 0) {
    mbar_init(BAR(B_XFULL), 1);
    for (int s = 0; s < NST; ++s) { mbar_init(BAR(B_YFULL + s), 1); mbar_init(BAR(B_YEMPTY + s), 1); }
    for (int s = 0; s < 2; ++s) {
      mbar_init(BAR(B_TFULL + s), 1); mbar_init(BAR(B_TEMPTY + s), NEPI);
      mbar_init(BAR(B_DSFULL + s), is_teach(MODE) ? 1 : NEPI); mbar_init(BAR(B_DSEMPTY + s), 1);
    }
    mbar_init(BAR(B_ACC), 1);
    mbar_init(BAR(B_PFULL), 1); mbar_init(BAR(B_PFULL + 1), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(tmX) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(tmY) : "memory");
    if (is_teach(MODE) || MODE == MODE_DE) asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_pt) : "memory");
  }
  constexpr uint32_t TMEM_COLS = fwd_like(MODE) ? 256u : 512u;
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  constexpr uint32_t ACC_COL = 256;
  pdl_wait(); pdl_go();      // barrier init + TMEM allocation above overlap the previous kernel's drain (chain launches)
  if (threadIdx.x == 64) TL2(2);

  if (warp == 0) {
    // ===== producer: one elected lane issues the TMA loads ==========================================
    if (lane == 0 && n_it > 0) {
      if (!is_teach(MODE)) load_tile2(smem_u32(sX), tmX, x_tile * TILE, BAR(B_XFULL));
      TL2(3);
      for (int it = 0; it < n_it; ++it) {
        const int ys = it % NST; const uint32_t yph = (it / NST) & 1;
        mbar_wait(BAR(B_YEMPTY + ys), yph ^ 1, a.err);
        load_tile2(smem_u32(sY + ys * TILE2_BYTES), tmY, (y_lo + it) * TILE, BAR(B_YFULL + ys));
        if (it < 8) TL2(8 + it);
        if (is_teach(MODE)) {               // the "dS" operand is a stored tile of coef * softmax(teacher)
          const int s = it % NDS; const uint32_t ph = (it / NDS) & 1;
          mbar_wait(BAR(B_DSEMPTY + s), ph ^ 1, a.err);
          load_ds2(smem_u32(sD + s * DS2_BYTES), &tm_pt, (y_lo + it) * TILE, (x_tile - a.x0_t) * TILE, BAR(B_DSFULL + s));
        }
      }
      // The dS buffer(s) were cycled by the EPILOGUE during the row-tile loop; this warp has not followed their phases, so a
      // parity wait on DSEMPTY alone could be satisfied by a completion several tiles back.  Every second product also
      // commits to the Y stage it read: wait for the LAST row tile's commit (a phase this warp has not consumed yet), after
      // which the DSEMPTY phase count is exactly n_it and the sequential parity waits below are unambiguous.
      if (n_tt > 0) mbar_wait(BAR(B_YEMPTY + (n_it - 1) % NST), ((n_it - 1) / NST) & 1, a.err);
      for (int jt = 0; jt < n_tt; ++jt) {   // DE: rep tile of exemplar row tile jt + its teacher tile for this vocabulary tile
        const int idx = n_it + jt;
        const int ys = idx % NST; const uint32_t yph = (idx / NST) & 1;
        mbar_wait(BAR(B_YEMPTY + ys), yph ^ 1, a.err);
        load_tile2(smem_u32(sY + ys * TILE2_BYTES), tmY, (a.x0_t + jt) * TILE, BAR(B_YFULL + ys));
        const int s = idx % NDS; const uint32_t ph = (idx / NDS) & 1;
        mbar_wait(BAR(B_DSEMPTY + s), ph ^ 1, a.err);
        load_ds2(smem_u32(sD + s * DS2_BYTES), &tm_pt, x_tile * TILE, jt * TILE, BAR(B_PFULL + s));
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===== MMA issuer ===================================================================================
    if (lane == 0 && n_it > 0) {
      constexpr uint32_t IDESC1 = make_idesc(128, 128, 0, 0);
      constexpr bool DE_LIKE = (MODE == MODE_DE);
      constexpr uint32_t IDESC2 = DE_LIKE ? make_idesc(128, KP, 1, 1) : make_idesc(128, KP, 0, 1);
      const uint32_t xa = smem_u32(sX);
      auto issue_s = [&](int it) {          // S[buf] = rep_tile . e_tile^T  (both operands K-major)
        const int s = it & 1; const uint32_t ph = (it >> 1) & 1;
        const int ys = it % NST; const uint32_t yph = (it / NST) & 1;
        mbar_wait(BAR(B_YFULL + ys), yph, a.err);
        if (it < 8) TL2(48 + it);
        mbar_wait(BAR(B_TEMPTY + s), ph ^ 1, a.err);
        if (it < 8) TL2(16 + it);
        tc_fence_after();
        const uint32_t ya = smem_u32(sY + ys * TILE2_BYTES);
        const uint32_t A = (MODE == MODE_DE) ? ya : xa;     // rows of S = logits rows (rep)
        const uint32_t B = (MODE == MODE_DE) ? xa : ya;
#pragma unroll
        for (int k = 0; k < KSTEPS1; ++k)
          umma_bf16(tmem + s * 128, desc_kmajor(A, k), desc_kmajor(B, k), IDESC1, k > 0);
        if (fwd_like(MODE)) umma_commit(BAR(B_YEMPTY + ys));
        umma_commit(BAR(B_TFULL + s));
      };
      if (!is_teach(MODE)) { mbar_wait(BAR(B_XFULL), 0, a.err); issue_s(0); }
      for (int it = 0; it < n_it; ++it) {
        if (!is_teach(MODE) && it + 1 < n_it) issue_s(it + 1);
        if (!fwd_like(MODE)) {
          const int s = it % NDS; const uint32_t ph = (it / NDS) & 1;
          const int ys = it % NST;
          if (is_teach(MODE)) mbar_wait(BAR(B_YFULL + ys), (it / NST) & 1, a.err);
          mbar_wait(BAR(B_DSFULL + s), ph, a.err);
          if (it < 8) TL2(56 + it);
          tc_fence_after();
          const uint32_t da = smem_u32(sD + s * DS2_BYTES);
          const uint32_t ya = smem_u32(sY + ys * TILE2_BYTES);
#pragma unroll
          for (int k = 0; k < KSTEPS2; ++k) {
            // dS tile [128 m][128 v]: DREP / TU read it K-major (M = m, K = v), DE reads it MN-major (M = v, K = m);
            // the streamed tile is the MN-major B operand (N = feature, K = tile row)
            const uint64_t ad = DE_LIKE ? desc_mnmajor(da, k) : desc_kmajor(da, k);
            umma_bf16(tmem + ACC_COL, ad, desc_mnmajor(ya, k), IDESC2, (it > 0 || k > 0));
          }
          umma_commit(BAR(B_YEMPTY + ys));
          umma_commit(BAR(B_DSEMPTY + s));
        }
      }
      if (MODE == MODE_DE) {                // dE[v] -= Pc^T . rep over the exemplar row tiles (A negated)
        constexpr uint32_t IDESC2N = make_idesc(128, KP, 1, 1, 1);
        uint32_t pph[2] = {0u, 0u};
        for (int jt = 0; jt < n_tt; ++jt) {
          const int idx = n_it + jt;
          const int ys = idx % NST; const int s = idx % NDS;
          mbar_wait(BAR(B_YFULL + ys), (idx / NST) & 1, a.err);
          mbar_wait(BAR(B_PFULL + s), pph[s], a.err); pph[s] ^= 1u;
          tc_fence_after();
          const uint32_t da = smem_u32(sD + s * DS2_BYTES);
          const uint32_t ya = smem_u32(sY + ys * TILE2_BYTES);
#pragma unroll
          for (int k = 0; k < KSTEPS2; ++k)
            umma_bf16(tmem + ACC_COL, desc_mnmajor(da, k), desc_mnmajor(ya, k), IDESC2N, 1u);
          umma_commit(BAR(B_YEMPTY + ys));
          umma_commit(BAR(B_DSEMPTY + s));
        }
      }
      if (!fwd_like(MODE)) umma_commit(BAR(B_ACC));
    }
    __syncwarp();
  } else {
    // ===== epilogue: TMEM lane = logits row ===============================================================
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    const int row = q * 32 + lane;
    const uint32_t tlane = (uint32_t)(q * 32) << 16;
    RowInfo ri, ri_next;
    float mx = -INFINITY, sum = 0.f, lab = 0.f, dot = 0.f;
    if (is_teach(MODE)) { ri = RowInfo(); ri_next = RowInfo(); }
    else if (MODE != MODE_DE) ri = row_info(a, x_tile * TILE + row, MODE != MODE_FWD);
    else ri_next = row_info(a, y_lo * TILE + row, true);
    if (MODE == MODE_TP && (x_tile * TILE + row < a.t_row_lo || x_tile * TILE + row >= a.t_row_hi)) ri.kind = 0;   // zero row
    for (int it = 0; it < (is_teach(MODE) ? 0 : n_it); ++it) {
      const int s = it & 1; const uint32_t ph = (it >> 1) & 1;
      int v0;
      if (MODE == MODE_DE) {
        ri = ri_next;
        if (it + 1 < n_it) ri_next = row_info(a, (y_lo + it + 1) * TILE + row, true);
        v0 = x_tile * TILE;
      } else v0 = (y_lo + it) * TILE;
      mbar_wait(BAR(B_TFULL + s), ph, a.err);
      if (threadIdx.x == 64 && it < 8) TL2(24 + it);
      tc_fence_after();
      // This thread's 64 columns in four chunks of 16: the TMEM load of chunk c+1 is in flight while chunk c goes through
      // the exponentials (a 128x128 fp32 tile is 64 KB of TMEM reads: as long as the MUFU work, so they must overlap);
      // the S buffer goes back to the MMA warp as soon as the last chunk has landed.
      uint32_t rb[2][16];
      const uint32_t tcol = tmem + tlane + s * 128 + half * 64;
      tmem_ld16_nowait(tcol, rb[0]);
      tmem_ld_wait16(rb[0]);
      if (threadIdx.x == 64 && it == 2) TL2(4);
      const int vb0 = v0 + half * 64;
      const bool full = (ri.kind != 0) && (vb0 + 64 <= ri.vlim);
      uint32_t pk[32];                         // BWD: this thread's 64 gradient values as bf16 pairs
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        uint32_t (&cur)[16] = rb[c & 1];
        if (c < 3) tmem_ld16_nowait(tcol + (c + 1) * 16, rb[(c + 1) & 1]);
        const int vb = vb0 + c * 16;
        if (MODE == MODE_FWD) {
          if (full) {
            float cm = __uint_as_float(cur[0]);
#pragma unroll
            for (int i = 1; i < 16; ++i) cm = fmaxf(cm, __uint_as_float(cur[i]));
            const float nm = fmaxf(mx, cm);
            sum *= ex2((mx - nm) * LOG2E);
            mx = nm;
            const float nm2 = nm * LOG2E;
            float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int i = 0; i < 16; ++i) s4[i & 3] += ex2(fmaf(__uint_as_float(cur[i]), LOG2E, -nm2));
            sum += (s4[0] + s4[1]) + (s4[2] + s4[3]);
            if (ri.label >= vb && ri.label < vb + 16) {
#pragma unroll
              for (int i = 0; i < 16; ++i) if (vb + i == ri.label) lab = __uint_as_float(cur[i]);
            }
          } else if (ri.kind != 0 && vb < ri.vlim) {               // boundary chunk: per-element checks
            float cm = -INFINITY;
#pragma unroll
            for (int i = 0; i < 16; ++i) if (vb + i < ri.vlim) cm = fmaxf(cm, __uint_as_float(cur[i]));
            const float nm = fmaxf(mx, cm);
            sum *= ex2((mx - nm) * LOG2E);
            mx = nm;
            const float nm2 = nm * LOG2E;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const int v = vb + i;
              if (v < ri.vlim) {
                const float sv = __uint_as_float(cur[i]);
                sum += ex2(fmaf(sv, LOG2E, -nm2));
                if (v == ri.label) lab = sv;
              }
            }
          }
        } else {
          float g[16];
          if (full) {
#pragma unroll
            for (int i = 0; i < 16; ++i) g[i] = ri.coef * ex2(fmaf(__uint_as_float(cur[i]), LOG2E, -ri.lse2));
            if (ri.label >= vb && ri.label < vb + 16) {
#pragma unroll
              for (int i = 0; i < 16; ++i) if (vb + i == ri.label) g[i] -= ri.coef;
            }
          } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const int v = vb + i;
              float gv = 0.f;
              if (ri.kind != 0 && v < ri.vlim) {
                const float p = ex2(fmaf(__uint_as_float(cur[i]), LOG2E, -ri.lse2));
                gv = ri.coef * (p - (v == ri.label ? 1.f : 0.f));
              }
              g[i] = gv;
            }
          }
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            __nv_bfloat162 h = __floats2bfloat162_rn(g[2 * u], g[2 * u + 1]);
            pk[c * 8 + u] = *reinterpret_cast<uint32_t*>(&h);
          }
        }
        if (c < 3) tmem_ld_wait16(rb[(c + 1) & 1]);
        if (c == 2) {                          // all 64 columns are in registers: hand the S buffer back
          tc_fence_before();
          mbar_arrive(BAR(B_TEMPTY + s));
        }
      }
      if (threadIdx.x == 64 && it == 2) TL2(5);
      if (MODE == MODE_TP) {                   // Pc row segment: 64 bf16 = 128 contiguous bytes of this thread's row
        uint4* o = reinterpret_cast<uint4*>(a.pt_out + (size_t)(x_tile * TILE + row) * ((size_t)a.n_vtiles * TILE) + vb0);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
      } else if (MODE != MODE_FWD) {
        const int sd = it % NDS; const uint32_t dph = (it / NDS) & 1;
        // the exponentials above overlap the second product of the previous tile; only the stores wait for its dS buffer
        mbar_wait(BAR(B_DSEMPTY + sd), dph ^ 1, a.err);
        if (threadIdx.x == 64 && it == 2) TL2(6);
        // region `half` (this thread's 64 columns), row `row`: eight 16-byte chunks, chunk j at position j ^ (row & 7)
        uint8_t* drow = sD + sd * DS2_BYTES + half * REG2 + row * 128;
#pragma unroll
        for (int j = 0; j < 8; ++j)
          *reinterpret_cast<uint4*>(drow + ((j ^ (row & 7)) << 4)) = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
        fence_async_smem();
        mbar_arrive(BAR(B_DSFULL + sd));
      }
      if (threadIdx.x == 64 && it < 8) TL2(32 + it);
    }
    if (MODE == MODE_FWD) {
      const int gm = x_tile * TILE + row;
      if (gm < a.M) {
        float4 o = make_float4(mx, sum, lab, dot);
        *reinterpret_cast<float4*>(a.stats + ((size_t)(chunk * 2 + half) * a.M + gm) * 4) = o;
      }
    } else if (MODE != MODE_TP && n_it > 0) {
      mbar_wait(BAR(B_ACC), 0, a.err);
      tc_fence_after();
      // accumulator [128 rows, 160] -> the (now idle) Y stages, row pitch DE_LD floats (conflict-free 16-byte row writes) ...
#pragma unroll 1
      for (int c4 = half; c4 < KP / 32; c4 += 2) {
        uint32_t r[32];
        tmem_ld32(tmem + tlane + ACC_COL + c4 * 32, r);
        float* stg = reinterpret_cast<float*>(sY) + row * DE_LD + c4 * 32;
#pragma unroll
        for (int i = 0; i < 32; i += 4)
          *reinterpret_cast<float4*>(stg + i) = make_float4(__uint_as_float(r[i]), __uint_as_float(r[i + 1]),
                                                            __uint_as_float(r[i + 2]), __uint_as_float(r[i + 3]));
      }
      asm volatile("bar.sync 1, %0;" ::"n"(NEPI) : "memory");
      const float* stg = reinterpret_cast<const float*>(sY);
      const int ew = warp - 2;
      if (MODE == MODE_DREP || MODE == MODE_TU) {
        // ... and out as ONE contiguous 80 KB block (partials are [rows][160] fp32): fully coalesced 16-byte stores
        float* o = (MODE == MODE_DREP) ? a.drep_part + ((size_t)chunk * a.n_mtiles * TILE + (size_t)x_tile * TILE) * KP
                                       : a.u_part + ((size_t)chunk * a.n_et * TILE + (size_t)(x_tile - a.x0_t) * TILE) * KP;
        for (int f = ew * 32 + lane; f < TILE * (KP / 4); f += NEPI) {
          const int rr = f / (KP / 4), c4 = f % (KP / 4);
          *reinterpret_cast<float4*>(o + (size_t)rr * KP + c4 * 4) = *reinterpret_cast<const float4*>(stg + rr * DE_LD + c4 * 4);
        }
      } else {                                // DE: whole table rows (d floats, contiguous) per warp
        for (int rr = ew; rr < TILE; rr += NEPI / 32) {
          const int v = x_tile * TILE + rr;
          if (v >= a.V) break;
          float2* o = reinterpret_cast<float2*>(a.grad_table + (size_t)v * a.d);
          for (int c2 = lane; c2 < a.d / 2; c2 += 32) o[c2] = *reinterpret_cast<const float2*>(stg + rr * DE_LD + 2 * c2);
        }
      }
      tc_fence_before();
    } else if (MODE == MODE_DREP || MODE == MODE_TU) {
      float* o = (MODE == MODE_DREP) ? a.drep_part + ((size_t)chunk * a.n_mtiles * TILE + (size_t)x_tile * TILE + row) * KP
                                     : a.u_part + ((size_t)chunk * a.n_et * TILE + (size_t)(x_tile - a.x0_t) * TILE + row) * KP;
      for (int i = half * (KP / 2); i < (half + 1) * (KP / 2); ++i) o[i] = 0.f;
    }
  }
  if (threadIdx.x == 64) TL2(40);
  __syncthreads();
  if (threadIdx.x == 0) TL2(41);
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(TMEM_COLS) : "memory");
  }
}

// fp32 rows -> row-major bf16 [rows_pad][160] (rows >= n_rows and columns >= d are zero): the HBM operand of the tc2 kernels
// (zero4: four flag words cleared on the way -- a memset node in front of this kernel costs ~10 us in a graph)
__global__ void k_pack_rows16(const float* __restrict__ src, long long ld, int n_rows, int d, int rows_pad,
                              __nv_bfloat16* __restrict__ out, int* __restrict__ zero4) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (zero4 && idx < 4) zero4[idx] = 0;
  const long long total = (long long)rows_pad * (ROW16 / 8);
  if (idx >= total) return;
  const int kc = (int)(idx % (ROW16 / 8));
  const long long row = idx / (ROW16 / 8);
  uint32_t pk[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float v0 = 0.f, v1 = 0.f;
    const int k = kc * 8 + i * 2;
    if (row < n_rows) {
      if (k < d) v0 = src[row * ld + k];
      if (k + 1 < d) v1 = src[row * ld + k + 1];
    }
    __nv_bfloat162 h = __floats2bfloat162_rn(v0, v1);
    pk[i] = *reinterpret_cast<uint32_t*>(&h);
  }
  *reinterpret_cast<uint4*>(out + row * ROW16 + kc * 8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
}

// frozen teacher: the exemplar rows' snapshot reps as the row-major bf16 [n_et*128][160] operand of the teacher passes, in
// the row convention of Pc (row = step row - x0*128; rows that are not exemplar rows and columns >= d are zero)
__global__ void k_pack_trep16(const float* __restrict__ trep, const int* __restrict__ teacher_row, int n_train, int M, int x0,
                              int d, int rows_pad, __nv_bfloat16* __restrict__ out) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)rows_pad * (ROW16 / 8)) return;
  const int kc = (int)(idx % (ROW16 / 8));
  const int row = (int)(idx / (ROW16 / 8));
  const int e = x0 * TILE + row - n_train;
  const float* src = (e >= 0 && e + n_train < M) ? trep + (long long)(teacher_row ? teacher_row[e] : e) * d : nullptr;
  uint32_t pk[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int k = kc * 8 + i * 2;
    const float v0 = (src && k < d) ? src[k] : 0.f, v1 = (src && k + 1 < d) ? src[k + 1] : 0.f;
    __nv_bfloat162 h = __floats2bfloat162_rn(v0, v1);
    pk[i] = *reinterpret_cast<uint32_t*>(&h);
  }
  *reinterpret_cast<uint4*>(out + (long long)row * ROW16 + kc * 8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
}

// Pc = coef * softmax(teacher) as ONE row-major bf16 matrix [n_et*128][n_vtp*128] (row = step row - x0*128, column = local
// vocabulary column; zeros outside the exemplar rows / beyond V_prev): TMA cuts the dS-layout tiles out of it.
__global__ void __launch_bounds__(256) k_teacher_rows16(const float* __restrict__ teacher, const int* __restrict__ teacher_row,
                                                        long long ld, int vec4, const float* __restrict__ lse_t, int n_train, int M,
                                                        int V_prev, int v_off, int x0, int n_vtp, float coef,
                                                        __nv_bfloat16* __restrict__ out) {
  const int vt = blockIdx.x, et = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long ldo = (long long)n_vtp * TILE;
  const int vl = vt * TILE + lane * 4;
  const int vg = v_off + vl;
  float4 t[16]; float l[16];
#pragma unroll
  for (int rr = 0; rr < 16; ++rr) {
    const int m = warp * 16 + rr;
    const int e = (x0 + et) * TILE + m - n_train;
    t[rr] = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY); l[rr] = 0.f;
    if (e >= 0 && e + n_train < M && vg < V_prev) {
      const float* row = teacher + (long long)(teacher_row ? teacher_row[e] : e) * ld;
      l[rr] = lse_t[e];
      if (vec4 && vg + 3 < V_prev) t[rr] = __ldg(reinterpret_cast<const float4*>(row + vg));
      else {
        t[rr].x = row[vg];
        if (vg + 1 < V_prev) t[rr].y = row[vg + 1];
        if (vg + 2 < V_prev) t[rr].z = row[vg + 2];
        if (vg + 3 < V_prev) t[rr].w = row[vg + 3];
      }
    }
  }
#pragma unroll
  for (int rr = 0; rr < 16; ++rr) {
    const int m = warp * 16 + rr;
    const __nv_bfloat162 a = __floats2bfloat162_rn(coef * expf(t[rr].x - l[rr]), coef * expf(t[rr].y - l[rr]));
    const __nv_bfloat162 b = __floats2bfloat162_rn(coef * expf(t[rr].z - l[rr]), coef * expf(t[rr].w - l[rr]));
    uint2 pk; pk.x = *reinterpret_cast<const uint32_t*>(&a); pk.y = *reinterpret_cast<const uint32_t*>(&b);
    *reinterpret_cast<uint2*>(out + ((long long)et * TILE + m) * ldo + vl) = pk;
  }
}

// teacher log-sum-exp per exemplar row (CTA per row)
__global__ void __launch_bounds__(256) k_teacher_lse(const float* __restrict__ teacher, const int* __restrict__ teacher_row,
                                                     long long ld, int Vp, float* __restrict__ lse_t) {
  __shared__ float sh[8];
  const int e = blockIdx.x;
  const float* t = teacher + (long long)(teacher_row ? teacher_row[e] : e) * ld;
  float mx = -INFINITY;
  for (int j = threadIdx.x; j < Vp; j += 256) mx = fmaxf(mx, t[j]);
#pragma unroll
  for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = mx;
  __syncthreads();
  mx = sh[0];
  for (int w = 1; w < 8; ++w) mx = fmaxf(mx, sh[w]);
  __syncthreads();
  float s = 0.f;
  for (int j = threadIdx.x; j < Vp; j += 256) s += expf(t[j] - mx);
#pragma unroll
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) { float tot = 0.f; for (int w = 0; w < 8; ++w) tot += sh[w]; lse_t[e] = mx + logf(tot); }
}

// uc[n_et*128, 160] = sum over chunks of the MODE_TU partials (fixed order); udot[row] = rep_row . uc_row.
// CTA (KP threads) per row.
__global__ void __launch_bounds__(KP) k_reduce_u(const float* __restrict__ part, int n_chunks, int rows, float* __restrict__ u,
                                                 const float* __restrict__ rep, int x0, int M, int d, float* __restrict__ udot) {
  __shared__ float sh[KP / 32];
  const int r = blockIdx.x, c = threadIdx.x;
  pdl_wait(); pdl_go();
  const float* pp = part + (size_t)r * KP + c;
  const size_t cs = (size_t)rows * KP;
  float s = 0.f;
  int k = 0;
  for (; k + 8 <= n_chunks; k += 8) {
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = pp[(size_t)(k + j) * cs];
#pragma unroll
    for (int j = 0; j < 8; ++j) s += v[j];
  }
  for (; k < n_chunks; ++k) s += pp[(size_t)k * cs];
  u[(size_t)r * KP + c] = s;
  const int gm = x0 * TILE + r;
  float p = (gm < M && c < d) ? s * rep[(size_t)gm * d + c] : 0.f;
#pragma unroll
  for (int o = 16; o; o >>= 1) p += __shfl_xor_sync(0xffffffffu, p, o);
  if ((c & 31) == 0) sh[c >> 5] = p;
  __syncthreads();
  if (c == 0) { float t = 0.f; for (int w = 0; w < KP / 32; ++w) t += sh[w]; udot[r] = t; }
}

// merge the per-chunk online-softmax partials: lse[M], row_loss[M].  Distillation rows: dot = rep_i . u_i.
// Warp per row, lanes over the chunk partials (one L2 round trip instead of a serial walk over the chunks);
// lane partials are combined in a fixed butterfly order.
__global__ void __launch_bounds__(256) k_merge_stats(const float* __restrict__ stats, int M, int n_chunks, int n_train, int mode,
                                                     float* __restrict__ lse, float* __restrict__ row_loss, float* __restrict__ local_out,
                                                     const float* __restrict__ udot, int x0, float coef_ex) {
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  pdl_wait(); pdl_go();
  if (i >= M) return;
  float mx = -INFINITY, lab = 0.f;
  for (int c = lane; c < n_chunks; c += 32) mx = fmaxf(mx, stats[((size_t)c * M + i) * 4]);
#pragma unroll
  for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float sum = 0.f;
  for (int c = lane; c < n_chunks; c += 32) {
    const float4 s = *reinterpret_cast<const float4*>(stats + ((size_t)c * M + i) * 4);
    if (s.x > -INFINITY) sum += s.y * expf(s.x - mx);
    lab += s.z;
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) { sum += __shfl_xor_sync(0xffffffffu, sum, o); lab += __shfl_xor_sync(0xffffffffu, lab, o); }
  if (lane) return;
  float dot = 0.f;
  // distillation rows: sum_j softmax(t)_j s_ij = rep_i . (P.E)_i = rep_i . uc_i / coef  (coef = 0: the term has zero weight)
  if (i >= n_train && mode == 1 && udot && coef_ex != 0.f) dot = udot[i - x0 * TILE] / coef_ex;
  if (local_out) {      // vocab-parallel: hand the shard's (max, sumexp, label logit, kd dot) to the host-side all-reduce
    *reinterpret_cast<float4*>(local_out + (size_t)i * 4) = make_float4(mx, sum, lab, dot);
    return;
  }
  const float l = mx + logf(sum);
  lse[i] = l;
  const bool kd = (i >= n_train) && mode == 1;
  row_loss[i] = kd ? l - dot : l - lab;
}

// frozen teacher: lse_t[r] of every packed exemplar row from the per-chunk (max, sumexp) partials of the MODE_FWD pass over
// the snapshot (k_merge_stats without label, distillation and row-loss terms).  Warp per row, fixed butterfly order.
__global__ void __launch_bounds__(256) k_merge_lse(const float* __restrict__ stats, int rows, int n_chunks, float* __restrict__ lse) {
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (i >= rows) return;
  float mx = -INFINITY;
  for (int c = lane; c < n_chunks; c += 32) mx = fmaxf(mx, stats[((size_t)c * rows + i) * 4]);
#pragma unroll
  for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float sum = 0.f;
  for (int c = lane; c < n_chunks; c += 32) {
    const float2 s = *reinterpret_cast<const float2*>(stats + ((size_t)c * rows + i) * 4);
    if (s.x > -INFINITY) sum += s.y * expf(s.x - mx);
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  if (lane == 0) lse[i] = mx + logf(sum);
}

// d_rep[M, d] = sum over chunks of the padded partials  (- uc = coef_ex * P.E for distillation rows)
__global__ void k_reduce_drep(const float* __restrict__ part, int n_chunks, int rows_pad, int M, int d,
                              float* __restrict__ d_rep, const float* __restrict__ u, int x0, int n_train) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  pdl_wait(); pdl_go();
  if (idx >= (long long)M * d) return;
  const int i = (int)(idx / d), c = (int)(idx % d);
  // same left-to-right sum as a plain loop, but eight independent loads are in flight per trip (the plain loop paid one
  // L2 round trip per chunk: ~20 us for 24 chunks on the critical chain)
  const float* p = part + (size_t)i * KP + c;
  const size_t cs = (size_t)rows_pad * KP;
  float s = 0.f;
  int k = 0;
  for (; k + 8 <= n_chunks; k += 8) {
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = p[(size_t)(k + j) * cs];
#pragma unroll
    for (int j = 0; j < 8; ++j) s += v[j];
  }
  for (; k < n_chunks; ++k) s += p[(size_t)k * cs];
  if (u && i >= n_train) s -= u[(size_t)(i - x0 * TILE) * KP + c];
  d_rep[idx] = s;
}

}  // namespace tc
}  // namespace ader

using namespace ader;
using namespace ader::tc;

// loss_reduce lives in loss.cu
namespace ader { int launch_loss_reduce(const float* row_loss, int n_train, int n_ex, float lambda_, float* loss, cudaStream_t st,
                                        int den_train, int den_ex); }

struct TcWs {
  uint8_t *rep_tiles, *e_tiles, *pt_tiles;
  float *stats, *lse, *lse_t, *drep_part, *u_part, *u, *udot;
  uint8_t* trep16;                         // frozen teacher: packed exemplar reps [n_et*128][160] bf16
  float *tstats, *lse_tt;                  // ... its per-chunk statistics and log-sum-exp per packed row
  int* err;
  int x0_t, n_et, n_vtp, n_chunks_t;       // teacher products (0 tiles when the step has no distillation rows)
  size_t bytes;
};
static int tc_chunks(int n_mtiles, int n_vtiles) {
  // vocabulary chunks per row tile: fill whole waves of 148 SMs (one CTA per SM), keep >= 4 tiles per CTA
  int best = 1; double best_eff = 0.0;
  const int cmax = n_vtiles / 4 > 1 ? (n_vtiles / 4 < 64 ? n_vtiles / 4 : 64) : 1;
  for (int c = 1; c <= cmax; ++c) {
    const long long ctas = (long long)n_mtiles * c;
    const long long waves = (ctas + 147) / 148;
    const double eff = (double)ctas / (148.0 * waves);
    if (eff > best_eff + 1e-9) { best_eff = eff; best = c; }
  }
  return best;
}
// workspace of a call over logits columns [v_lo, v_hi); its teacher columns are the part of [0, V_prev) inside that range
static TcWs carve_tc(const AderLossArgs* a, int v_lo, int v_hi, char* base) {
  TcWs w; size_t o = 0;
  auto take = [&](size_t n) { char* p = base ? base + o : nullptr; o += align_up(n); return p; };
  const int M = a->M, V = v_hi - v_lo, n_ex = a->n_ex;
  const int t_hi = a->V_prev < v_hi ? a->V_prev : v_hi;
  const int Vp_local = n_ex > 0 && a->mode == 1 && t_hi > v_lo ? t_hi - v_lo : 0;
  const int nm = cdiv(M, TILE), nv = cdiv(V, TILE), nc = tc_chunks(nm, nv);
  const bool kd = Vp_local > 0;
  w.x0_t = kd ? (M - n_ex) / TILE : 0;
  w.n_et = kd ? (M - 1) / TILE - w.x0_t + 1 : 0;
  w.n_vtp = kd ? cdiv(Vp_local, TILE) : 0;
  w.n_chunks_t = kd ? tc_chunks(w.n_et, w.n_vtp) : 0;
  w.rep_tiles = (uint8_t*)take((size_t)nm * TILE_BYTES);
  w.e_tiles = (uint8_t*)take((size_t)nv * TILE_BYTES);
  w.stats = (float*)take(sizeof(float) * 4 * (size_t)nc * 2 * M);
  w.lse = (float*)take(sizeof(float) * M);
  w.lse_t = (float*)take(sizeof(float) * (n_ex > 0 ? n_ex : 1));
  w.drep_part = (float*)take(sizeof(float) * (size_t)nc * nm * TILE * KP);
  w.pt_tiles = (uint8_t*)take((size_t)w.n_et * w.n_vtp * DS_BYTES + 16);
  w.u_part = (float*)take(sizeof(float) * ((size_t)w.n_chunks_t * w.n_et * TILE * KP + 4));
  w.u = (float*)take(sizeof(float) * ((size_t)w.n_et * TILE * KP + 4));
  w.udot = (float*)take(sizeof(float) * ((size_t)w.n_et * TILE + 4));
  w.err = (int*)take(sizeof(int) * 4);
  const bool fz = a->teacher_rep && kd;
  w.trep16 = fz ? (uint8_t*)take((size_t)w.n_et * TILE * ROW16 * 2) : nullptr;
  w.tstats = fz ? (float*)take(sizeof(float) * 4 * (size_t)w.n_chunks_t * 2 * w.n_et * TILE) : nullptr;
  w.lse_tt = fz ? (float*)take(sizeof(float) * (size_t)w.n_et * TILE) : nullptr;
  w.bytes = o;
  return w;
}

extern "C" size_t ader_loss_tc_ws_bytes(const AderModel* m, const AderLossArgs* a) {
  if (check_model(m) || !a || a->M <= 0 || a->V <= 0) return 0;
  return carve_tc(a, 0, a->V, nullptr).bytes;
}

extern "C" size_t ader_table16_ws_bytes(const AderModel* m, int32_t V) {
  if (check_model(m) || V <= 0 || path_check(m, ADER_PATH_LOSS_TC)) return 0;
  return (size_t)cdiv(V, TILE) * TILE * ROW16 * 2;
}

static int tc_ready() {
  if (int e = kernel_ready<k_tc2<MODE_FWD>>(smem_tc2(MODE_FWD), "k_tc2<MODE_FWD>")) return e;
  if (int e = kernel_ready<k_tc2<MODE_DREP>>(smem_tc2(MODE_DREP), "k_tc2<MODE_DREP>")) return e;
  if (int e = kernel_ready<k_tc2<MODE_DE>>(smem_tc2(MODE_DE), "k_tc2<MODE_DE>")) return e;
  if (int e = kernel_ready<k_tc2<MODE_TU>>(smem_tc2(MODE_TU), "k_tc2<MODE_TU>")) return e;
  return kernel_ready<k_tc2<MODE_TP>>(smem_tc2(MODE_TP), "k_tc2<MODE_TP>");
}

// TMA tensor maps over the row-major bf16 operand matrices
struct TcMaps { CUtensorMap rep, e, pt, trep, ttab; };     // trep / ttab: frozen teacher only

// The tcgen05 plan of one call over logits columns [v_lo, v_hi) -- the single-GPU loss is the one shard [0, V): workspace,
// kernel arguments and tensor maps.  grad (or NULL) receives dE in item-table rows v_lo+1 .. v_hi.  Host work only.
static int tc_plan(const AderModel* m, const AderLossArgs* a, int v_lo, int v_hi, void* ws, float* grad,
                   TcWs& w, TcArgs& t, TcMaps& mp) {
  const int d = m->d, M = a->M, V = v_hi - v_lo;
  w = carve_tc(a, v_lo, v_hi, (char*)ws);
  const int nm = cdiv(M, TILE), nv = cdiv(V, TILE), nc = tc_chunks(nm, nv);
  if (int e = tc_ready()) return e;

  t.M = M; t.V = V; t.V_total = a->V; t.v_off = v_lo; t.n_mtiles = nm; t.n_vtiles = nv; t.n_chunks = nc;
  t.n_train = a->n_train; t.n_ex = a->n_ex; t.V_prev = a->V_prev; t.mode = a->n_ex > 0 ? a->mode : 0;
  t.coef_train = a->n_train > 0 ? 1.0f / (float)(a->n_train_global > 0 ? a->n_train_global : a->n_train) : 0.f;
  t.coef_ex = a->n_ex > 0 ? a->lambda_ / (float)(a->n_ex_global > 0 ? a->n_ex_global : a->n_ex) : 0.f;
  t.pos = a->pos; t.ex_pos = a->ex_pos;
  t.lse = w.lse; t.lse_t = w.lse_t; t.stats = w.stats; t.drep_part = w.drep_part;
  t.grad_table = grad ? grad + (size_t)(1 + v_lo) * d : nullptr;
  t.d = d; t.err = w.err;
  t.x0_t = w.x0_t; t.n_et = w.n_et; t.n_vtp = w.n_vtp; t.n_chunks_t = w.n_chunks_t; t.u_part = w.u_part;
  t.pt_out = nullptr; t.t_row_lo = t.t_row_hi = 0;

  if (int e = make_map2d(&mp.rep, w.rep_tiles, ROW16, (uint64_t)nm * TILE, ROW16 * 2)) return e;
  if (int e = make_map2d(&mp.e, w.e_tiles, ROW16, (uint64_t)nv * TILE, ROW16 * 2)) return e;
  if (w.n_et > 0 && w.n_vtp > 0) {
    if (int e = make_map2d(&mp.pt, w.pt_tiles, (uint64_t)w.n_vtp * TILE, (uint64_t)w.n_et * TILE, (uint64_t)w.n_vtp * TILE * 2)) return e;
  } else mp.pt = mp.e;       // never dereferenced (no teacher tiles), but the parameter must be a valid map
  if (w.trep16) {            // frozen teacher
    if (int e = make_map2d(&mp.trep, w.trep16, ROW16, (uint64_t)w.n_et * TILE, ROW16 * 2)) return e;
    if (int e = make_map2d(&mp.ttab, a->teacher_table16, ROW16, (uint64_t)w.n_vtp * TILE, ROW16 * 2)) return e;
  }
  return 0;
}

// launches shared by the single-GPU and vocab-parallel entry points -----------------------------------------------
// teacher statistics + tiles + uc partials (rep-independent), then u = sum of partials and udot = rep . u
// frozen teacher: Pc from the snapshot (packed reps -> MODE_FWD statistics of T = trep . E_prev^T -> lse_t -> MODE_TP tiles)
static void launch_teacher_frozen(const AderLossArgs* a, const TcWs& w, const TcArgs& t, int d, cudaStream_t st, const TcMaps& mp) {
  const int rows = w.n_et * TILE;
  k_pack_trep16<<<cdiv((long long)rows * (ROW16 / 8), 256), 256, 0, st>>>(a->teacher_rep, a->teacher_row, a->n_train, a->M, w.x0_t, d,
                                                                         rows, reinterpret_cast<__nv_bfloat16*>(w.trep16));
  TcArgs tt = t;                          // every packed row is a label-free softmax row of width V_prev over the snapshot's table
  tt.M = rows; tt.V = a->V_prev; tt.V_total = a->V_prev; tt.v_off = 0;
  tt.n_mtiles = w.n_et; tt.n_vtiles = w.n_vtp; tt.n_chunks = w.n_chunks_t;
  tt.n_train = 0; tt.mode = 1; tt.stats = w.tstats; tt.lse = w.lse_tt; tt.drep_part = nullptr; tt.grad_table = nullptr;
  tt.pt_out = reinterpret_cast<__nv_bfloat16*>(w.pt_tiles);
  tt.t_row_lo = a->n_train - w.x0_t * TILE; tt.t_row_hi = a->M - w.x0_t * TILE;
  k_tc2<MODE_FWD><<<w.n_et * w.n_chunks_t, NTHREADS, smem_tc2(MODE_FWD), st>>>(tt, mp.trep, mp.ttab, mp.pt);
  k_merge_lse<<<cdiv((long long)rows * 32, 256), 256, 0, st>>>(w.tstats, rows, w.n_chunks_t * 2, w.lse_tt);
  k_tc2<MODE_TP><<<w.n_et * w.n_chunks_t, NTHREADS, smem_tc2(MODE_TP), st>>>(tt, mp.trep, mp.ttab, mp.pt);
}
static void launch_teacher_tu(const AderLossArgs* a, const TcWs& w, const TcArgs& t, int v_off, cudaStream_t st, const TcMaps& mp) {
  if (a->teacher_rep) {                   // frozen teacher (single GPU: v_off == 0)
    launch_teacher_frozen(a, w, t, t.d, st, mp);
  } else {
    // teacher rows 16-byte aligned (ld % 4 == 0, shard offset too): 128-bit loads
    const int vec4 = (a->teacher_ld % 4 == 0 && (uintptr_t)a->teacher % 16 == 0 && v_off % 4 == 0) ? 1 : 0;
    k_teacher_lse<<<a->n_ex, 256, 0, st>>>(a->teacher, a->teacher_row, a->teacher_ld, a->V_prev, w.lse_t);
    k_teacher_rows16<<<dim3(w.n_vtp, w.n_et), 256, 0, st>>>(a->teacher, a->teacher_row, a->teacher_ld, vec4, w.lse_t,
                                                           a->n_train, a->M, a->V_prev, v_off, w.x0_t, w.n_vtp, t.coef_ex,
                                                           reinterpret_cast<__nv_bfloat16*>(w.pt_tiles));
  }
  k_tc2<MODE_TU><<<w.n_et * w.n_chunks_t, NTHREADS, smem_tc2(MODE_TU), st>>>(t, mp.rep, mp.e, mp.pt);
}
static void launch_reduce_u(const AderLossArgs* a, const TcWs& w, const float* rep, int d, cudaStream_t st) {
  k_reduce_u<<<w.n_et * TILE, KP, 0, st>>>(w.u_part, w.n_chunks_t, w.n_et * TILE, w.u, rep, w.x0_t, a->M, d, w.udot);
}
static void launch_teacher_u(const AderLossArgs* a, const TcWs& w, const TcArgs& t, int v_off, const float* rep, int d,
                             cudaStream_t st, const TcMaps& mp) {
  launch_teacher_tu(a, w, t, v_off, st, mp);
  launch_reduce_u(a, w, rep, d, st);
}
// operand packing: fp32 rows -> the row-major bf16 matrix the tensor maps describe
static void launch_pack(const float* src, long long ld, int n_rows, int d, int n_tiles, uint8_t* out, cudaStream_t st, int* zero4 = nullptr) {
  k_pack_rows16<<<cdiv((long long)n_tiles * TILE * (ROW16 / 8), 256), 256, 0, st>>>(src, ld, n_rows, d, n_tiles * TILE,
                                                                                    reinterpret_cast<__nv_bfloat16*>(out), zero4);
}

extern "C" int32_t ader_loss_fwd_bwd_tc(const AderModel* m, const float* theta, const float* rep,
                                        const AderLossArgs* a, void* ws, float* loss, float* row_loss,
                                        float* d_rep, float* grad, void* stream) {
  Fork f = Fork::serial((cudaStream_t)stream);
  return loss_tc_run(m, theta, rep, a, ws, loss, row_loss, d_rep, grad, f, 3);
}

// Measurement hook (bench.py roofline): re-launches ONLY k_tc2<FWD>, <DREP>, <DE> on a workspace that a preceding
// ader_loss_fwd_bwd_tc call with the same arguments prepared (tiles, lse, teacher tiles); outputs are the same values.
extern "C" int32_t ader_debug_loss_tc_kernels(const AderModel* m, const float* theta, const AderLossArgs* a, void* ws,
                                              float* grad, void* stream) {
  Fork f = Fork::serial((cudaStream_t)stream);
  return loss_tc_run(m, theta, nullptr, a, ws, nullptr, nullptr, nullptr, grad, f, 4);
}

// phase_mask bit 0: table tiles + teacher products that do not need `rep`, on f.b;
// bit 1: everything else.  Forward statistics, loss and d_rep stay on f.main; the scalar loss reduction goes to f.c and
// the dE kernel to f.b (f.table_ready is recorded behind it: whoever adds into the item-table gradient waits for it).
int ader::loss_tc_run(const AderModel* m, const float* theta, const float* rep, const AderLossArgs* a, void* ws, float* loss,
                      float* row_loss, float* d_rep, float* grad, Fork& f, int phase_mask) {
  if (int e = check_model(m)) return e;
  if (int e = path_check(m, ADER_PATH_LOSS_TC)) return e;
  ADER_CHECK_ARG(theta && a && ws, "loss_fwd_bwd_tc: NULL pointer");
  ADER_CHECK_ARG(!(phase_mask & 2) || (rep && loss && row_loss), "loss_fwd_bwd_tc: NULL pointer");
  if (int e = check_loss_args(m, a, "loss_fwd_bwd_tc", true)) return e;
  cudaStream_t st = f.main, sb = f.b;
  const int d = m->d, M = a->M, V = a->V;
  const bool kd = a->n_ex > 0 && a->mode == 1;
  TcWs w; TcArgs t; TcMaps mp;
  if (int e = tc_plan(m, a, 0, V, ws, grad, w, t, mp)) return e;
  const int nm = t.n_mtiles, nv = t.n_vtiles, nc = t.n_chunks;
  if (phase_mask == 4) {      // measurement only: the three tensor-core kernels on an already prepared workspace, launched as
                              // in the step: programmatic dependent launches along the chain
    launch_chain(k_tc2<MODE_FWD>, dim3(nm * nc), dim3(NTHREADS), (size_t)smem_tc2(MODE_FWD), st, true, t, mp.rep, mp.e, mp.pt);
    launch_chain(k_tc2<MODE_DREP>, dim3(nm * nc), dim3(NTHREADS), (size_t)smem_tc2(MODE_DREP), st, true, t, mp.rep, mp.e, mp.pt);
    if (grad) launch_chain(k_tc2<MODE_DE>, dim3(nv), dim3(NTHREADS), (size_t)smem_tc2(MODE_DE), st, true, t, mp.rep, mp.e, mp.pt);
    ADER_CHECK_LAUNCH("tc kernels");
    return 0;
  }
  if (phase_mask & 1) {
    launch_pack(theta + d, d, V, d, nv, w.e_tiles, sb, w.err);       // clears the error words on the way
    if (kd) launch_teacher_tu(a, w, t, 0, sb, mp);
    ADER_CHECK_LAUNCH("tc prep");
  }
  if (!(phase_mask & 2)) return 0;

  f.edge(sb, st);
  launch_pack(rep, d, M, d, nm, w.rep_tiles, st);
  // chain links (kernel directly behind a kernel on f.main) may be programmatic dependent launches
  if (kd) launch_chain(k_reduce_u, dim3(w.n_et * TILE), dim3(KP), 0, st, f.pdl, (const float*)w.u_part, w.n_chunks_t, w.n_et * TILE, w.u, rep,
                       w.x0_t, a->M, d, w.udot);
  ADER_CHECK_LAUNCH("tc pack");
  launch_chain(k_tc2<MODE_FWD>, dim3(nm * nc), dim3(NTHREADS), (size_t)smem_tc2(MODE_FWD), st, f.pdl, t, mp.rep, mp.e, mp.pt);
  launch_chain(k_merge_stats, dim3(cdiv((long long)M * 32, 256)), dim3(256), 0, st, f.pdl, (const float*)w.stats, M, nc * 2, a->n_train, t.mode,
               w.lse, row_loss, (float*)nullptr, (const float*)(kd ? w.udot : nullptr), w.x0_t, t.coef_ex);
  cudaEvent_t lse_ready = nullptr;
  if (f.parallel()) { lse_ready = f.take(); cudaEventRecord(lse_ready, st); }
  f.edge(st, f.c);
  if (int e = launch_loss_reduce(row_loss, a->n_train, a->n_ex, a->lambda_, loss, f.c, a->n_train_global, a->n_ex_global)) return e;
  ADER_CHECK_LAUNCH("tc fwd");
  if (d_rep) {
    launch_chain(k_tc2<MODE_DREP>, dim3(nm * nc), dim3(NTHREADS), (size_t)smem_tc2(MODE_DREP), st, f.pdl, t, mp.rep, mp.e, mp.pt);
    if (f.fuse_drep) {        // fused step: the final-LayerNorm backward kernel sums the partials (encoder.cu, k_lnf_bwd_drep)
      f.drep.part = w.drep_part; f.drep.u = kd ? w.u : nullptr; f.drep.n_chunks = nc; f.drep.rows_pad = nm * TILE; f.drep.kp = KP;
      f.drep.u_row0 = w.x0_t * TILE; f.drep.n_train = a->n_train;
      f.has_drep = true;
    } else
      launch_chain(k_reduce_drep, dim3(cdiv((long long)M * d, 256)), dim3(256), 0, st, f.pdl, (const float*)w.drep_part, nc, nm * TILE, M, d, d_rep,
                   (const float*)(kd ? w.u : nullptr), w.x0_t, a->n_train);
    ADER_CHECK_LAUNCH("tc d_rep");
  }
  if (grad) {
    if (f.parallel()) cudaStreamWaitEvent(sb, lse_ready, 0);
    k_tc2<MODE_DE><<<nv, NTHREADS, smem_tc2(MODE_DE), sb>>>(t, mp.rep, mp.e, mp.pt);
    ADER_CHECK_LAUNCH("tc d_table");
    if (f.parallel()) { f.table_ready = f.take(); cudaEventRecord(f.table_ready, sb); f.has_table_ready = true; }
  }
  // f.c (scalar loss) is joined by the caller's closing edges: a join here would sit between d_rep and the backward chain
  return 0;
}


#ifdef ADER_TC_TIMELINE
extern "C" int32_t ader_debug_tc_timeline(long long* out) {
  cudaDeviceSynchronize();
  return (int32_t)cudaMemcpyFromSymbol(out, g_tl, sizeof(g_tl));
}
#endif

// ---- vocab-parallel variant (SURVEY 8e): this rank owns logits columns [v_lo, v_hi) ---------------------
// the arguments of ader_loss_fwd_bwd_tc except a frozen teacher, and a 128-aligned shard inside [0, V)
static int vp_check(const AderModel* m, const AderLossArgs* a, int v_lo, int v_hi) {
  if (int e = check_model(m)) return e;
  if (int e = path_check(m, ADER_PATH_LOSS_TC)) return e;
  ADER_CHECK_ARG(a, "loss_tc_vp: NULL pointer");
  ADER_CHECK_ARG(!a->teacher_rep, "loss_tc_vp: a frozen teacher (teacher_rep) is not supported by the vocab-parallel entries");
  if (int e = check_loss_args(m, a, "loss_tc_vp", true)) return e;
  ADER_CHECK_ARG(v_lo >= 0 && v_lo < v_hi && v_hi <= a->V && v_lo % TILE == 0, "loss_tc_vp: shard [%d,%d) must be 128-aligned inside [0,%d)", v_lo, v_hi, a->V);
  return 0;
}

extern "C" size_t ader_loss_tc_vp_ws_bytes(const AderModel* m, const AderLossArgs* a, int32_t v_lo, int32_t v_hi) {
  if (check_model(m) || !a || a->M <= 0 || v_hi <= v_lo || a->teacher_rep) return 0;
  return carve_tc(a, v_lo, v_hi, nullptr).bytes;
}

extern "C" int32_t ader_loss_tc_vp_fwd(const AderModel* m, const float* theta, const float* rep, const AderLossArgs* a,
                                       int32_t v_lo, int32_t v_hi, void* ws, float* stats, void* stream) {
  if (int e = vp_check(m, a, v_lo, v_hi)) return e;
  ADER_CHECK_ARG(theta && rep && ws && stats, "loss_tc_vp_fwd: NULL pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int d = m->d;
  TcWs w; TcArgs t; TcMaps mp;
  if (int e = tc_plan(m, a, v_lo, v_hi, ws, nullptr, w, t, mp)) return e;
  cudaMemsetAsync(w.err, 0, sizeof(int) * 4, st);
  launch_pack(rep, d, a->M, d, t.n_mtiles, w.rep_tiles, st);
  launch_pack(theta + (size_t)(1 + v_lo) * d, d, t.V, d, t.n_vtiles, w.e_tiles, st);
  if (w.n_et > 0) launch_teacher_u(a, w, t, v_lo, rep, d, st, mp);
  k_tc2<MODE_FWD><<<t.n_mtiles * t.n_chunks, NTHREADS, smem_tc2(MODE_FWD), st>>>(t, mp.rep, mp.e, mp.pt);
  k_merge_stats<<<cdiv((long long)a->M * 32, 256), 256, 0, st>>>(w.stats, a->M, t.n_chunks * 2, a->n_train, t.mode, nullptr, nullptr, stats,
                                                 w.n_et > 0 ? w.udot : nullptr, w.x0_t, t.coef_ex);
  ADER_CHECK_LAUNCH("loss_tc_vp_fwd");
  return 0;
}

extern "C" int32_t ader_loss_tc_vp_bwd(const AderModel* m, const float* theta, const float* rep, const AderLossArgs* a,
                                       int32_t v_lo, int32_t v_hi, void* ws, const float* lse, float* d_rep_partial,
                                       float* grad, void* stream) {
  if (int e = vp_check(m, a, v_lo, v_hi)) return e;
  ADER_CHECK_ARG(theta && rep && ws && lse, "loss_tc_vp_bwd: NULL pointer");
  cudaStream_t st = (cudaStream_t)stream;
  TcWs w; TcArgs t; TcMaps mp;
  if (int e = tc_plan(m, a, v_lo, v_hi, ws, grad, w, t, mp)) return e;     // operands were packed by the forward call
  t.lse = lse;
  if (d_rep_partial) {
    k_tc2<MODE_DREP><<<t.n_mtiles * t.n_chunks, NTHREADS, smem_tc2(MODE_DREP), st>>>(t, mp.rep, mp.e, mp.pt);
    k_reduce_drep<<<cdiv((long long)a->M * m->d, 256), 256, 0, st>>>(w.drep_part, t.n_chunks, t.n_mtiles * TILE, a->M, m->d, d_rep_partial,
                                                                     w.n_et > 0 ? w.u : nullptr, w.x0_t, a->n_train);
  }
  if (grad) k_tc2<MODE_DE><<<t.n_vtiles, NTHREADS, smem_tc2(MODE_DE), st>>>(t, mp.rep, mp.e, mp.pt);
  ADER_CHECK_LAUNCH("loss_tc_vp_bwd");
  return 0;
}

extern "C" int32_t ader_pack_table16(const AderModel* m, const float* rows, int32_t V, void* out, void* stream) {
  if (int e = check_model(m)) return e;
  if (int e = path_check(m, ADER_PATH_LOSS_TC)) return e;
  ADER_CHECK_ARG(rows && out, "pack_table16: NULL pointer");
  ADER_CHECK_ARG(V >= 1 && V < m->v_tab, "pack_table16: V=%d outside the table of %d rows", V, m->v_tab);
  const long long rows_pad = (long long)cdiv(V, TILE) * TILE;
  k_pack_rows16<<<cdiv(rows_pad * (ROW16 / 8), 256), 256, 0, (cudaStream_t)stream>>>(rows, m->d, V, m->d, (int)rows_pad,
                                                                                     reinterpret_cast<__nv_bfloat16*>(out), nullptr);
  ADER_CHECK_LAUNCH("pack_table16");
  return 0;
}
