// Error reporting + introspection entry points of libader_b200.so.
#include "common.cuh"
#include <string.h>

namespace ader {
static thread_local char g_err[512] = "";
int fail(int code, const char* fmt, ...) {
  va_list ap; va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int path_check(const AderModel* m, int path, bool report) {
  const int d = m->d, L = m->maxlen;
  auto refuse = [&](const char* fmt, auto... args) { return report ? fail(-1, fmt, args...) : -1; };
  auto smem = [&](const char* what, size_t need, size_t have) {
    if (need <= have) return 0;
    return refuse("%s: the attention tile of one session needs %zu bytes of shared memory, more than its %zu "
                  "(hidden_units=%d, maxlen=%d)", what, need, have, d, L);
  };
  auto tc = [&](const char* what) {
    if (d <= PATH_TC_MAX_D) return 0;
    return refuse("%s needs hidden_units <= %d (hidden_units=%d, maxlen=%d)", what, PATH_TC_MAX_D, d, L);
  };
  switch (path) {
    case ADER_PATH_ENCODER_FWD: return smem("exact encoder forward", attn_fwd_smem(d, L), ATTN_FWD_SMEM_MAX);
    case ADER_PATH_ENCODER_BWD: return smem("exact encoder backward", attn_bwd_smem(d, L), ATTN_BWD_SMEM_MAX);
    case ADER_PATH_ENCODER_TC: return tc("the fused encoder");
    case ADER_PATH_LOSS_TC: return tc("the tcgen05 loss");
    case ADER_PATH_EVAL_TC: return tc("tcgen05 evaluation");
    case ADER_PATH_FISHER_BATCHED:
      if (int e = tc("the batched Fisher")) return e;
      if (int e = path_check(m, ADER_PATH_ENCODER_FWD, report)) return e;
      return path_check(m, ADER_PATH_ENCODER_BWD, report);
    case ADER_PATH_HERDING_ONCHIP: return tc("on-chip herding");
  }
  return refuse("path_check: unknown path %d", path);
}
}  // namespace ader

using namespace ader;

extern "C" int32_t ader_abi_version(void) { return ADER_ABI_VERSION; }
extern "C" const char* ader_last_error(void) { return g_err; }

extern "C" int32_t ader_path_check(const AderModel* m, int32_t path) {
  if (int e = check_model(m)) return e;
  return path_check(m, path);
}

extern "C" int64_t ader_param_count(const AderModel* m) {
  if (check_model(m)) return -1;
  return make_layout(m).total;
}
extern "C" int64_t ader_dense_count(const AderModel* m) {
  if (check_model(m)) return -1;
  return make_layout(m).dense_count();
}
extern "C" int64_t ader_param_offset(const AderModel* m, int32_t idx) {
  if (check_model(m)) return -1;
  const Layout l = make_layout(m);
  const int n = 2 + 14 * m->num_blocks + 2;
  if (idx < 0 || idx >= n) { fail(-1, "param_offset: index %d out of range (%d tensors)", idx, n); return -1; }
  if (idx == 0) return l.off_table;
  if (idx == 1) return l.off_pos;
  if (idx >= 2 + 14 * m->num_blocks) return l.off_lnf + (long long)(idx - 2 - 14 * m->num_blocks) * m->d;
  const int b = (idx - 2) / 14, k = (idx - 2) % 14;
  const long long rel[14] = {l.ln1b, l.ln1g, l.wq, l.bq, l.wk, l.bk, l.wv, l.bv, l.ln2b, l.ln2g, l.w1, l.b1, l.w2, l.b2};
  return l.block(b) + rel[k];
}
