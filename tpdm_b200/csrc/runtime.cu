#include <cstdlib>
// tpdm_b200 -- error reporting, device queries and TMA descriptor encoding shared by the library.
#include <stdarg.h>

#include <atomic>
#include <mutex>
#include <vector>

#include "host.h"

namespace tpdm {

static thread_local std::string g_last_error;

void set_last_error(const std::string& msg) { g_last_error = msg; }

int fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

static thread_local const int* g_skip = nullptr;
void set_skip_flag(const int* f) { g_skip = f; }
const int* skip_flag() { return g_skip; }
static thread_local const int* g_bmask = nullptr;
static thread_local int g_bslots = 1;
void set_batch_mask(const int* m, int slots) {
  g_bmask = m;
  g_bslots = slots > 0 ? slots : 1;
}
const int* batch_mask() { return g_bmask; }
int batch_mask_slots() { return g_bslots; }

static std::atomic<long long> g_launches{0};
bool pdl_enabled() {
  static const bool on = [] {
    const char* e = std::getenv("TPDM_PDL");
    return e == nullptr || e[0] != '0';
  }();
  return on;
}
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
void count_launches(long long n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
long long launches_so_far() { return g_launches.load(std::memory_order_relaxed); }

namespace {
struct Profiler {
  std::vector<cudaEvent_t> ev;
  std::vector<int> cls;
  std::vector<double> flops;
  std::vector<const int*> skip;   // device skip flag the launch was made under (set_skip_flag), or null
  size_t n = 0;
  long long dropped = 0;          // records of the last stop whose launch returned at once because its skip flag was set
  bool on = false;
};
Profiler g_prof;
}  // namespace

bool profiling_active() { return g_prof.on; }

void prof_begin(int cls, double flops, cudaStream_t s) {
  if (!g_prof.on || 2 * (g_prof.n + 1) > g_prof.ev.size()) return;
  g_prof.cls[g_prof.n] = cls;
  g_prof.flops[g_prof.n] = flops;
  g_prof.skip[g_prof.n] = skip_flag();
  cudaEventRecord(g_prof.ev[2 * g_prof.n], s);
}
void prof_end(cudaStream_t s) {
  if (!g_prof.on || 2 * (g_prof.n + 1) > g_prof.ev.size()) return;
  cudaEventRecord(g_prof.ev[2 * g_prof.n + 1], s);
  ++g_prof.n;
}

int num_sms() {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
  }
  return sms;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPointByVersion("cuTensorMapEncodeTiled", &p, 12000, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

int encode_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                     const uint32_t* box) {
  return encode_tmap(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, base, rank, dims, strides_bytes, box);
}

int encode_tmap(CUtensorMap* out, CUtensorMapDataType dtype, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                const uint32_t* box) {
  EncodeTiledFn fn = get_encode_fn();
  TPDM_CHECK(fn != nullptr, TPDM_ERR_CUDA, "cuTensorMapEncodeTiled unavailable (no CUDA driver / device?)");
  TPDM_CHECK((reinterpret_cast<uintptr_t>(base) & 15) == 0, TPDM_ERR_ARG, "TMA base pointer must be 16-byte aligned");
  cuuint64_t gdim[5];
  cuuint64_t gstr[5];
  cuuint32_t bx[5];
  cuuint32_t estr[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bx[i] = box[i];
    estr[i] = 1;
    if (i + 1 < rank) {
      gstr[i] = strides_bytes[i];
      TPDM_CHECK(gstr[i] % 16 == 0, TPDM_ERR_SHAPE, "TMA stride %llu not a multiple of 16 bytes", (unsigned long long)gstr[i]);
    }
  }
  CUresult r = fn(out, dtype, static_cast<cuuint32_t>(rank), const_cast<void*>(base), gdim, gstr, bx, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  TPDM_CHECK(r == CUDA_SUCCESS, TPDM_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d (rank %d, dims %llu %llu, box %u %u)",
             static_cast<int>(r), rank, (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0), box[0],
             rank > 1 ? box[1] : 0);
  return 0;
}

}  // namespace tpdm

extern "C" const char* tpdm_last_error(void) { return tpdm::g_last_error.c_str(); }
extern "C" int tpdm_abi_version(void) { return TPDM_ABI_VERSION; }

extern "C" long long tpdm_launch_count(int reset) {
  long long v = tpdm::g_launches.load();
  if (reset) tpdm::g_launches.store(0);
  return v;
}

extern "C" long long tpdm_profile_dropped(void) { return tpdm::g_prof.dropped; }

extern "C" int tpdm_profile_start(int max_records) {
  using namespace tpdm;
  TPDM_CHECK(max_records > 0, TPDM_ERR_ARG, "tpdm_profile_start: max_records must be positive");
  while (g_prof.ev.size() < static_cast<size_t>(2 * max_records)) {
    cudaEvent_t e;
    TPDM_CUDA_OK(cudaEventCreate(&e));
    g_prof.ev.push_back(e);
  }
  g_prof.cls.assign(max_records, 0);
  g_prof.flops.assign(max_records, 0.0);
  g_prof.skip.assign(max_records, nullptr);
  g_prof.n = 0;
  g_prof.dropped = 0;
  g_prof.on = true;
  return 0;
}

extern "C" int tpdm_profile_stop(double* ms, double* flops, long long* count, int n_classes) {
  using namespace tpdm;
  TPDM_CHECK(ms && flops && count && n_classes > 0, TPDM_ERR_ARG, "tpdm_profile_stop: null argument");
  g_prof.on = false;
  for (int c = 0; c < n_classes; ++c) ms[c] = flops[c] = 0.0, count[c] = 0;
  if (g_prof.n > 0) TPDM_CUDA_OK(cudaEventSynchronize(g_prof.ev[2 * g_prof.n - 1]));
  // A launch made under a skip flag that reads 1 now was a speculatively enqueued step the device skipped (the flags are
  // write-once per trajectory: all_done[k] / idle_flag go 0 -> 1 and stay).  Such records carry no work: they are dropped, so
  // neither their algorithmic FLOPs nor their (~0) time reach the per-class sums.
  const int* last_ptr = nullptr;
  int last_val = 0;
  g_prof.dropped = 0;
  for (size_t i = 0; i < g_prof.n; ++i) {
    if (g_prof.skip[i] != nullptr) {
      if (g_prof.skip[i] != last_ptr) {
        last_ptr = g_prof.skip[i];
        TPDM_CUDA_OK(cudaMemcpy(&last_val, last_ptr, sizeof(int), cudaMemcpyDeviceToHost));
      }
      if (last_val != 0) {
        ++g_prof.dropped;
        continue;
      }
    }
    float t = 0.f;
    TPDM_CUDA_OK(cudaEventElapsedTime(&t, g_prof.ev[2 * i], g_prof.ev[2 * i + 1]));
    const int c = g_prof.cls[i];
    if (c >= 0 && c < n_classes) {
      ms[c] += t;
      flops[c] += g_prof.flops[i];
      count[c] += 1;
    }
  }
  return 0;
}
