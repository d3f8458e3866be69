// Error plumbing, device queries and the host plumbing of host.cuh, shared by every translation unit of libsurgvid.
#include <map>
#include <mutex>
#include <utility>

#include "host.cuh"

namespace sv {

static thread_local std::string g_last_error;

void set_error(const std::string& msg) { g_last_error = msg; }

int fail(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}

int device_sm_count() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  static std::mutex mu;
  static int cached_dev = -1, cached = 0;
  std::lock_guard<std::mutex> lock(mu);
  if (cached_dev == dev) return cached;
  int n = 0;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
  cached_dev = dev;
  cached = n;
  return n;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is a PER-DEVICE attribute: remember which (device, kernel, bytes) were configured and
// never cache a failure, so a handle created on a second GPU of the same process opts its kernels in again.
int ensure_dynamic_smem(const void* fn, int bytes) {
  if (bytes <= 48 * 1024) return SV_OK;
  int dev = 0;
  SV_CUDA_OK(cudaGetDevice(&dev));
  static std::mutex mu;
  static std::map<std::pair<int, const void*>, int> configured;
  std::lock_guard<std::mutex> lock(mu);
  auto key = std::make_pair(dev, fn);
  auto it = configured.find(key);
  if (it != configured.end() && it->second >= bytes) return SV_OK;
  cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) return fail(SV_ERR_CUDA, std::string("cudaFuncSetAttribute(MaxDynamicSharedMemorySize): ") + cudaGetErrorString(e));
  configured[key] = bytes;
  return SV_OK;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const int*,
                                   const int*, cuuint32_t, cuuint32_t, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int encode_failed(const char* fn, const char* what, CUresult r) {
  return fail(SV_ERR_CUDA, std::string(fn) + "(" + what + ") failed, CUresult " + std::to_string(static_cast<int>(r)));
}

int encode_tiled(CUtensorMap* map, CUtensorMapDataType dtype, int rank, const void* base, const cuuint64_t* dims, const cuuint64_t* strides,
                 const cuuint32_t* box, CUtensorMapSwizzle swizzle, CUtensorMapL2promotion l2, const char* what) {
  static const EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    const bool ok = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess;
    return ok ? reinterpret_cast<EncodeTiledFn>(p) : nullptr;
  }();
  if (fn == nullptr) return fail(SV_ERR_CUDA, "cuTensorMapEncodeTiled driver entry point unavailable (no CUDA driver?)");
  const cuuint32_t elem_strides[5] = {1, 1, 1, 1, 1};
  const CUresult r = fn(map, dtype, static_cast<cuuint32_t>(rank), const_cast<void*>(base), dims, strides, box, elem_strides,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, l2, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? SV_OK : encode_failed("cuTensorMapEncodeTiled", what, r);
}

int encode_im2col(CUtensorMap* map, CUtensorMapDataType dtype, int rank, const void* base, const cuuint64_t* dims, const cuuint64_t* strides,
                  const int* lower, const int* upper, cuuint32_t channels, cuuint32_t pixels, const cuuint32_t* elem_strides,
                  CUtensorMapSwizzle swizzle, CUtensorMapL2promotion l2, const char* what) {
  static const EncodeIm2colFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    const bool ok = cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess;
    return ok ? reinterpret_cast<EncodeIm2colFn>(p) : nullptr;
  }();
  if (fn == nullptr) return fail(SV_ERR_CUDA, "cuTensorMapEncodeIm2col driver entry point unavailable (no CUDA driver?)");
  const CUresult r = fn(map, dtype, static_cast<cuuint32_t>(rank), const_cast<void*>(base), dims, strides, lower, upper, channels, pixels,
                        elem_strides, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, l2, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? SV_OK : encode_failed("cuTensorMapEncodeIm2col", what, r);
}

int StateDict::set(const char* name, const float* host_data, const int64_t* shape, int32_t ndim) {
  SV_CHECK(shape != nullptr || ndim == 0, "null argument");
  HostTensor t;
  int64_t n = 1;
  for (int i = 0; i < ndim; ++i) {
    SV_CHECK(shape[i] >= 0, "set_tensor: negative dimension");
    t.shape.push_back(shape[i]);
    n *= shape[i];
  }
  if (host_data) t.data.assign(host_data, host_data + n);
  else t.data.assign(static_cast<size_t>(n), 0.f);
  tensors[name] = std::move(t);
  packed = false;
  return SV_OK;
}

int StateDict::get(const std::string& key, const std::vector<int64_t>& shape, const char* who, const HostTensor** out) const {
  *out = nullptr;
  auto it = tensors.find(key);
  if (it == tensors.end()) return fail(SV_ERR_STATE, std::string(who) + ": missing state_dict key '" + key + "'");
  if (it->second.shape != shape) return fail(SV_ERR_INVALID, std::string(who) + ": wrong shape for '" + key + "'");
  *out = &it->second;
  return SV_OK;
}

int upload_bytes(int device, void** dst, const void* src, size_t bytes) {
  SV_CUDA_OK(cudaSetDevice(device));
  if (*dst) { cudaFree(*dst); *dst = nullptr; }
  SV_CUDA_OK(cudaMalloc(dst, bytes));
  SV_CUDA_OK(cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice));
  return SV_OK;
}

size_t StreamRegistry::counter_bytes(int32_t n_streams) { return (static_cast<size_t>(n_streams) * sizeof(int64_t) + 255) & ~static_cast<size_t>(255); }

static std::string with_prefix(const char* prefix, const char* msg) { return std::string(prefix) + ": " + msg; }

int StreamRegistry::reset(void* state, size_t state_bytes, size_t need, int32_t n_streams, const int32_t* stream_ids, int32_t n_ids,
                          cudaStream_t st) {
  SV_CHECK(n_streams >= 1, with_prefix(prefix_, "n_streams >= 1"));
  SV_CHECK(state_bytes >= need, with_prefix(prefix_, "state too small"));
  SV_CHECK((reinterpret_cast<uintptr_t>(state) & 255) == 0, with_prefix(prefix_, "state must be 256-byte aligned"));
  if (stream_ids == nullptr) {   // every stream: the whole state, so that no stale ring row is left behind
    SV_CUDA_OK(cudaMemsetAsync(state, 0, need, st));
    seen_[state].assign(n_streams, 0);
    return SV_OK;
  }
  auto it = seen_.find(state);
  if (it == seen_.end()) return fail(SV_ERR_STATE, with_prefix(prefix_, "reset every stream of a new state (stream_ids = NULL) first"));
  SV_CHECK(static_cast<int32_t>(it->second.size()) == n_streams, with_prefix(prefix_, "n_streams differs from the state's last full reset"));
  SV_CHECK(n_ids >= 1, with_prefix(prefix_, "n_ids >= 1"));
  std::vector<char> hit(n_streams, 0);
  for (int i = 0; i < n_ids; ++i) {
    SV_CHECK(stream_ids[i] >= 0 && stream_ids[i] < n_streams, with_prefix(prefix_, "stream id out of range"));
    SV_CHECK(!hit[stream_ids[i]], with_prefix(prefix_, "duplicate stream id"));
    hit[stream_ids[i]] = 1;
  }
  for (int i = 0; i < n_ids; ++i) {
    SV_CUDA_OK(cudaMemsetAsync(static_cast<int64_t*>(state) + stream_ids[i], 0, sizeof(int64_t), st));
    it->second[stream_ids[i]] = 0;
  }
  return SV_OK;
}

int StreamRegistry::check_step(const void* state, size_t state_bytes, size_t need, int32_t n_streams, const int32_t* stream_ids,
                               const int64_t* counts, int32_t n_ids, std::vector<int64_t>* out_tab) const {
  SV_CHECK(n_streams >= 1, with_prefix(prefix_, "n_streams >= 1"));
  SV_CHECK(state_bytes >= need, with_prefix(prefix_, "state too small"));
  auto it = seen_.find(state);
  if (it == seen_.end()) return fail(SV_ERR_STATE, with_prefix(prefix_, "the state was not reset through this handle (reset every stream first)"));
  SV_CHECK(static_cast<int32_t>(it->second.size()) == n_streams, with_prefix(prefix_, "n_streams differs from the state's last full reset"));
  SV_CHECK(n_ids >= 1 && n_ids <= n_streams, with_prefix(prefix_, "1 <= n_ids <= n_streams"));
  std::vector<int64_t>& tab = *out_tab;
  tab.assign(2 * static_cast<size_t>(n_ids) + 1, 0);
  std::vector<char> hit(n_streams, 0);
  for (int i = 0; i < n_ids; ++i) {
    const int32_t s = stream_ids[i];
    SV_CHECK(s >= 0 && s < n_streams, with_prefix(prefix_, "stream id out of range"));
    SV_CHECK(!hit[s], with_prefix(prefix_, "duplicate stream id"));
    hit[s] = 1;
    SV_CHECK(counts[i] >= 1, with_prefix(prefix_, "counts must be >= 1"));
    SV_CHECK(counts[i] < (1LL << 31) - it->second[s], with_prefix(prefix_, "a stream position would pass 2^31"));
    tab[i + 1] = tab[i] + counts[i];
    SV_CHECK(tab[i + 1] < (1LL << 31), with_prefix(prefix_, "too many rows in one step"));
    tab[n_ids + 1 + i] = s;
  }
  return SV_OK;
}

void StreamRegistry::advance(const void* state, const int32_t* stream_ids, const int64_t* counts, int32_t n_ids) {
  std::vector<int64_t>& seen = seen_.at(state);
  for (int i = 0; i < n_ids; ++i) seen[stream_ids[i]] += counts[i];
}

}  // namespace sv

extern "C" {
const char* sv_last_error(void) { return sv::g_last_error.c_str(); }
int sv_abi_version(void) { return SV_ABI_VERSION; }
}
