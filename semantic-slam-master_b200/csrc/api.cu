// Library-wide plumbing: thread-local error text, device check, launch counter.
#include <stdarg.h>

#include <mutex>
#include <vector>

#include "common.cuh"

namespace sslam {

static thread_local char g_err[512] = "";
std::atomic<uint64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// ---- optional per-kernel timing: CUDA events recorded around every launch on the launch stream
std::atomic<int> g_profile_on{0};
namespace {
struct ProfRec { int kind; cudaEvent_t beg, end; };
std::mutex g_prof_mu;
std::vector<ProfRec> g_prof_recs;
std::vector<cudaEvent_t> g_prof_pool;
cudaEvent_t prof_event() {
  if (!g_prof_pool.empty()) { cudaEvent_t e = g_prof_pool.back(); g_prof_pool.pop_back(); return e; }
  cudaEvent_t e = nullptr;
  cudaEventCreate(&e);
  return e;
}
}  // namespace

void prof_mark(int kind, cudaStream_t stream, bool begin) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (begin) {
    ProfRec r{kind, prof_event(), nullptr};
    cudaEventRecord(r.beg, stream);
    g_prof_recs.push_back(r);
  } else if (!g_prof_recs.empty() && g_prof_recs.back().end == nullptr) {
    g_prof_recs.back().end = prof_event();
    cudaEventRecord(g_prof_recs.back().end, stream);
  }
}

static int query_device(int* sms) {
  int dev = 0, n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    cudaGetLastError();
    set_error("no CUDA device visible (%s); libsslam_b200 has no CPU fallback",
              e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    return SSLAM_ENODEVICE;
  }
  SSLAM_CHECK_CUDA(cudaGetDevice(&dev));
  int major = 0;
  SSLAM_CHECK_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  SSLAM_CHECK_CUDA(cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev));
  if (major != 10) {
    set_error("device %d has compute capability %d.x; libsslam_b200 is built for sm_100a only", dev,
              major);
    return SSLAM_ENODEVICE;
  }
  return SSLAM_OK;
}

// per-device cache (compute capability and SM count are properties of a device, and one process
// may drive several): state 0 = not queried, 1 = usable, 2 = not usable
constexpr int MAX_DEVICES = 64;
static std::atomic<int> g_dev_state[MAX_DEVICES];
static std::atomic<int> g_dev_sms[MAX_DEVICES];
static std::atomic<int> g_nodevice{0};              // no device visible at all (cached)

int check_device() {
  if (g_nodevice.load(std::memory_order_relaxed)) {
    set_error("no CUDA device visible; libsslam_b200 has no CPU fallback");
    return SSLAM_ENODEVICE;
  }
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); dev = -1; }
  if (dev >= 0 && dev < MAX_DEVICES) {
    const int st = g_dev_state[dev].load(std::memory_order_acquire);
    if (st == 1) return SSLAM_OK;
    if (st == 2) {
      set_error("device %d is not an sm_100 device; libsslam_b200 has no CPU fallback", dev);
      return SSLAM_ENODEVICE;
    }
  }
  int sms = 0;
  const int rc = query_device(&sms);
  if (dev < 0) {
    if (rc == SSLAM_ENODEVICE) g_nodevice.store(1);
    return rc;
  }
  if (dev < MAX_DEVICES && (rc == SSLAM_OK || rc == SSLAM_ENODEVICE)) {
    g_dev_sms[dev].store(sms);
    g_dev_state[dev].store(rc == SSLAM_OK ? 1 : 2, std::memory_order_release);
  }
  return rc;
}

int num_sms() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MAX_DEVICES) return 148;
  const int s = g_dev_sms[dev].load();
  return s > 0 ? s : 148;
}

}  // namespace sslam

extern "C" int sslam_abi_version(void) { return SSLAM_ABI_VERSION; }

extern "C" int sslam_last_error(char* buf, size_t len) {
  size_t n = strlen(sslam::g_err);
  if (buf && len) {
    size_t c = n < len - 1 ? n : len - 1;
    memcpy(buf, sslam::g_err, c);
    buf[c] = 0;
  }
  return (int)n;
}

extern "C" int sslam_device_check(void) { return sslam::check_device(); }

extern "C" uint64_t sslam_launch_count(void) { return sslam::g_launches.load(); }

static const char* const kKindNames[sslam::KK_COUNT] = {
    "decode_scan", "decode_topk", "decode_count", "decode_resolve", "nms", "gather", "l2norm",
    "match_f32", "match_tc", "split_pair", "unpack_cols", "match_finalize", "gemm_f16x3", "layernorm",
    "eval_points", "cell_softmax", "conv_head", "ransac_hyp", "ransac_score", "ransac_refit", "pose",
    "pnp_hyp", "pnp_score", "pnp_refit", "triangulate", "bundle_adjust"};

extern "C" int sslam_profile_enable(int on) {
  std::lock_guard<std::mutex> lk(sslam::g_prof_mu);
  for (auto& r : sslam::g_prof_recs) {
    if (r.beg) sslam::g_prof_pool.push_back(r.beg);
    if (r.end) sslam::g_prof_pool.push_back(r.end);
  }
  sslam::g_prof_recs.clear();
  sslam::g_profile_on.store(on ? 1 : 0);
  return SSLAM_OK;
}

extern "C" int sslam_profile_kinds(void) { return sslam::KK_COUNT; }

extern "C" const char* sslam_profile_kind_name(int kind) {
  return (kind >= 0 && kind < sslam::KK_COUNT) ? kKindNames[kind] : "";
}

extern "C" int sslam_profile_read(int kind, double* total_ms, uint64_t* launches) {
  std::lock_guard<std::mutex> lk(sslam::g_prof_mu);
  double ms = 0.0;
  uint64_t n = 0;
  for (auto& r : sslam::g_prof_recs) {
    if (r.kind != kind || !r.end) continue;
    SSLAM_CHECK_CUDA(cudaEventSynchronize(r.end));
    float t = 0.f;
    SSLAM_CHECK_CUDA(cudaEventElapsedTime(&t, r.beg, r.end));
    ms += t;
    ++n;
  }
  if (total_ms) *total_ms = ms;
  if (launches) *launches = n;
  return SSLAM_OK;
}
