// Host-side helpers shared by the translation units of the library (matcher api.cu, extractor superpoint.cu):
// device buffers that only ever grow, fp16-split plane pairs, the PDL-aware kernel launcher, and the host runtime both
// handle types embed (error reporting, device, loaded weights, launch log).
#pragma once
#include <cstdarg>
#include <cstdio>
#include <map>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "../../include/onepose_b200.h"
#include "common.cuh"
#include "gemm_tc.cuh"

namespace opb {

// >= 0: byte value written into every fresh allocation that the algorithm does not require to be zero (opb_debug_set_ws_fill)
int ws_fill_byte();

struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  bool grew = false;      // set by ensure() when it (re)allocated: the caller orders the fill against its stream
  cudaError_t ensure(size_t need, bool zero = false) {
    if (need <= bytes) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
    cudaError_t e = cudaMalloc(&p, need);
    if (e != cudaSuccess) return e;
    bytes = need;
    grew = true;
    if (zero) e = cudaMemset(p, 0, need);                                 // buffers whose untouched parts are read as zero (bd, flags)
    else if (ws_fill_byte() >= 0) e = cudaMemset(p, ws_fill_byte(), need);   // test hook: poison everything else
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
  }
  template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

// A window of rows of a [rows, 256] plane pair (the residual stream of a chunk, the query-only buffer, ...).
struct XView {
  __half* hi;
  __half* lo;
  CPlanes c(int ld) const { return CPlanes{hi, lo, ld}; }
  Planes m(int ld) const { return Planes{hi, lo, ld}; }
};

struct PlaneBuf {
  DevBuf hi, lo;
  cudaError_t ensure(size_t elems, bool zero = false) {
    cudaError_t e = hi.ensure(elems * sizeof(__half), zero);
    if (e != cudaSuccess) return e;
    return lo.ensure(elems * sizeof(__half), zero);
  }
  void release() { hi.release(); lo.release(); }
  CPlanes c(int ld, size_t off_elems = 0) const { return CPlanes{hi.as<__half>() + off_elems, lo.as<__half>() + off_elems, ld}; }
  Planes m(int ld, size_t off_elems = 0) const { return Planes{hi.as<__half>() + off_elems, lo.as<__half>() + off_elems, ld}; }
  XView view(size_t row_off = 0) const { return XView{hi.as<__half>() + row_off * kD, lo.as<__half>() + row_off * kD}; }
};

inline void split_host(const std::vector<double>& w, std::vector<__half>& hi, std::vector<__half>& lo) {
  hi.resize(w.size());
  lo.resize(w.size());
  for (size_t i = 0; i < w.size(); ++i) split_f32((float)w[i], hi[i], lo[i]);
}

// Every kernel of the library begins with griddep_sync() and is launched with programmatic stream serialization (PDL).
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

// Raise the max-dynamic-shared-memory attribute of `kern` on the current device to `bytes`.  The attribute is per device, so
// it is recorded per (kernel, device) and set once for each.
inline cudaError_t ensure_smem_attr(const void* kern, int bytes) {
  static std::mutex mu;
  static std::map<std::pair<const void*, int>, int> set;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  std::lock_guard<std::mutex> lock(mu);
  int& cur = set[{kern, dev}];
  if (cur >= bytes) return cudaSuccess;
  e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) cur = bytes;
  return e;
}

// Host runtime of a handle (opb_matcher, opb_superpoint derive from it).
struct HostState {
  int device = 0;                                        // every entry point makes it current first (ENTER)
  std::string err;                                       // message of the handle's last failed call
  std::map<std::string, std::vector<float>> host_w;      // weights loaded by name, packed by finalize
  // Launch log of the current call: the launch count and, with profiling on, CUDA events on the launch stream: ev[0] before
  // the first launch, ev[i + 1] after launch i (named, with its algorithmic FLOPs), ev_end when the call finished.  Entry i
  // takes ev[i + 1] - ev[i], so its time includes the launch gap in front of it.
  int launches = 0;
  bool profiling = false;
  std::vector<cudaEvent_t> ev;
  size_t ev_used = 0;
  std::vector<std::string> ev_name;
  std::vector<double> ev_flops;
  cudaEvent_t ev_end = nullptr;
  ~HostState() {
    for (auto e : ev) cudaEventDestroy(e);
    if (ev_end) cudaEventDestroy(ev_end);
  }
};

// Message of this thread's last failed call that had no handle (opb_last_error(NULL), opb_sp_last_error(NULL)).
inline thread_local std::string g_last_error;

// Record the message of a failed call on the handle (or, without one, in g_last_error) and return `code`.
__attribute__((format(printf, 3, 4))) inline int fail(HostState* s, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  (s ? s->err : g_last_error) = buf;
  return code;
}

#define CK(s, expr)                                                                                                 \
  do {                                                                                                              \
    cudaError_t _e = (expr);                                                                                        \
    if (_e != cudaSuccess)                                                                                          \
      return opb::fail(s, OPB_E_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__);  \
  } while (0)

// First statement of a handle's entry point: reject a null handle, make the handle's device current.
#define ENTER(h)                                                                                                    \
  do {                                                                                                              \
    if (!(h)) return opb::fail(nullptr, OPB_E_INVALID, "%s: null handle", __func__);                                \
    CK(h, cudaSetDevice((h)->device));                                                                              \
  } while (0)

// Status of the <<<>>> launches a call just made.
inline int launch_status(HostState* s, const char* fn) {
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? OPB_OK : fail(s, OPB_E_CUDA, "%s: launch failed: %s", fn, cudaGetErrorString(e));
}

inline void record_event(HostState* s, cudaStream_t st) {
  if (s->ev_used == s->ev.size()) {
    cudaEvent_t e;
    cudaEventCreate(&e);
    s->ev.push_back(e);
  }
  cudaEventRecord(s->ev[s->ev_used++], st);
}

// Start the launch log of a call.
inline void begin_call(HostState* s, cudaStream_t st) {
  s->launches = 0;
  s->ev_used = 0;
  s->ev_name.clear();
  s->ev_flops.clear();
  if (s->profiling) record_event(s, st);
}

inline void log_launch(HostState* s, cudaStream_t st, const char* name, double flops) {
  s->launches++;
  if (!s->profiling) return;
  record_event(s, st);
  s->ev_name.push_back(name);
  s->ev_flops.push_back(flops);
}

inline void end_call(HostState* s, cudaStream_t st) {
  if (!s->profiling) return;
  if (!s->ev_end) cudaEventCreate(&s->ev_end);
  cudaEventRecord(s->ev_end, st);
}

// Milliseconds of log entry i (the launch and the gap in front of it).
inline int entry_ms(HostState* s, size_t i, float* ms) {
  CK(s, cudaEventElapsedTime(ms, s->ev[i], s->ev[i + 1]));
  return OPB_OK;
}

// Launch a kernel through launch_k and log it; on failure, return from the calling function.
#define LAUNCH(s, st, name, ...)                                                                                    \
  do {                                                                                                              \
    cudaError_t _le = opb::launch_k(__VA_ARGS__);                                                                   \
    if (_le != cudaSuccess) return opb::fail(s, OPB_E_CUDA, "launch of %s failed: %s", name, cudaGetErrorString(_le)); \
    opb::log_launch(s, st, name, 0.0);                                                                              \
  } while (0)

// One launch of the tcgen05 GEMM core, logged as `name` with `flops` algorithmic FLOPs.
inline int run_gemm(HostState* s, const GemmProblem& p, cudaStream_t st, double flops, const char* name) {
  const int rc = launch_gemm_tc(p, st);
  log_launch(s, st, name, flops);
  if (rc != 0)
    return fail(s, rc == -1 ? OPB_E_INVALID : OPB_E_CUDA, "GEMM launch failed (%s, rc=%d): %s", name, rc, cudaGetErrorString(cudaGetLastError()));
  return OPB_OK;
}

// The loaded weight `key`, which must have n elements: OPB_E_STATE when it is missing, OPB_E_INVALID when its size differs.
inline int find_w(HostState* s, const std::string& key, size_t n, const std::vector<float>*& out) {
  auto it = s->host_w.find(key);
  if (it == s->host_w.end()) return fail(s, OPB_E_STATE, "missing weight '%s'", key.c_str());
  if (it->second.size() != n) return fail(s, OPB_E_INVALID, "weight '%s' has %zu elements, expected %zu", key.c_str(), it->second.size(), n);
  out = &it->second;
  return OPB_OK;
}

// Weight uploads are synchronous copies on the legacy stream; finalize ends with a device synchronisation so that they are
// ordered against whatever (non-blocking) stream the caller uses afterwards.
inline int upload_planes(HostState* s, PlaneBuf& dst, const std::vector<double>& w, size_t off_elems = 0, size_t total_elems = 0) {
  std::vector<__half> hi, lo;
  split_host(w, hi, lo);
  CK(s, dst.ensure(total_elems ? total_elems : w.size()));
  CK(s, cudaMemcpy(dst.hi.as<__half>() + off_elems, hi.data(), hi.size() * sizeof(__half), cudaMemcpyHostToDevice));
  CK(s, cudaMemcpy(dst.lo.as<__half>() + off_elems, lo.data(), lo.size() * sizeof(__half), cudaMemcpyHostToDevice));
  return OPB_OK;
}
template <typename T> int upload_f32(HostState* s, DevBuf& dst, const std::vector<T>& w) {
  const std::vector<float> f(w.begin(), w.end());
  CK(s, dst.ensure(f.size() * sizeof(float)));
  CK(s, cudaMemcpy(dst.p, f.data(), f.size() * sizeof(float), cudaMemcpyHostToDevice));
  return OPB_OK;
}

#ifdef __CUDACC__
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
#endif

}  // namespace opb
