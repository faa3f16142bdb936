// Error channel, version and launch counter of the saga_b200 C ABI.
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "saga_common.cuh"

namespace saga {
std::atomic<int64_t> g_launches{0};

char* err_buf() {
  static thread_local char buf[512] = "";
  return buf;
}

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(err_buf(), 512, fmt, ap);
  va_end(ap);
  return code;
}
}  // namespace saga

// ---- tuning / A-B options ------------------------------------------------------------------------------------
// Every switch the kernels' launchers consult (previous-generation kernels kept as parity twins, tuning aids) lives
// in this table: initialised ONCE from the environment variable of the same name, changed at run time through
// saga_set_option.  The launchers read an atomic pointer -- there is no getenv on the hot path.
namespace saga {
static const char* const OPT_NAMES[] = {
    "SAGA_DEC_NO_FUSE", "SAGA_DEC_FUSE_MASK", "SAGA_CQT_CONTRACT_V1", "SAGA_UMMA_DEBUG", "SAGA_UMMA_CFG",
    "SAGA_UMMA_NO_SHARED_BANK", "SAGA_STFT_FRAMES", "SAGA_STFT_NO_EO", "SAGA_ISTFT_ONE_WARP", "SAGA_STFT_RING",
    "SAGA_STFT_RING_SHAPE", "SAGA_ISTFT_RING", "SAGA_SUB_CLUSTER_MIN_STEPS", "SAGA_SUB_NO_CLUSTER", "SAGA_SUB_NO_FLAT",
    "SAGA_SUB_FLAT_CHUNKS", "SAGA_DB_LEAN", "SAGA_DB_CHUNKS", "SAGA_CQT_STREAM", "SAGA_DEC_NO_PHASE", "SAGA_ISTFT_RING_RUN", "SAGA_CQT_STREAM_SS", "SAGA_CQT_STREAM_TWO_ISSUERS", "SAGA_CQT_STREAM_NO_UNROLL"};
constexpr int N_OPTS = sizeof(OPT_NAMES) / sizeof(OPT_NAMES[0]);
static std::atomic<const char*> g_opts[N_OPTS];
static std::once_flag g_opts_once;

static void opts_init() {
  std::call_once(g_opts_once, [] {
    for (int i = 0; i < N_OPTS; ++i) {
      const char* e = getenv(OPT_NAMES[i]);
      g_opts[i].store(e ? strdup(e) : nullptr, std::memory_order_relaxed);
    }
  });
}

int opt_id(const char* name) {
  for (int i = 0; i < N_OPTS; ++i)
    if (strcmp(name, OPT_NAMES[i]) == 0) return i;
  return -1;
}

const char* opt_value(int id) {
  if (id < 0 || id >= N_OPTS) return nullptr;
  opts_init();
  return g_opts[id].load(std::memory_order_acquire);
}
}  // namespace saga

extern "C" int saga_set_option(const char* name, const char* value) {
  if (!name) return saga::set_error(SAGA_ERR_INVALID, "set_option: null name");
  const int id = saga::opt_id(name);
  if (id < 0) return saga::set_error(SAGA_ERR_INVALID, "set_option: unknown option %s", name);
  saga::opts_init();
  saga::g_opts[id].store(value ? strdup(value) : nullptr, std::memory_order_release);   // old strings are not freed:
  return SAGA_OK;                                                                       // a launcher may still read them
}

extern "C" const char* saga_get_option(const char* name) { return name ? saga::opt_value(saga::opt_id(name)) : nullptr; }

extern "C" const char* saga_last_error_string(void) { return saga::err_buf(); }
// 2: + saga_short_window_batch_exec, saga_gather_frames_exec, saga_cqt_frames_exec, saga_set/get_option
// 3: + saga_cqt_frames_shared_exec, saga_cqt_frames_shared_multi_exec, saga_istft_rows_exec (additions only)
//    + saga_cqt_peak_workspace_bytes, saga_cqt_peak_exec, saga_window_slide_exec (additions only: existing entries
//    unchanged)
//    + saga_stft_rows_exec (addition only)
extern "C" int saga_abi_version(void) { return 3; }
extern "C" int64_t saga_launch_count(void) { return saga::g_launches.load(); }
