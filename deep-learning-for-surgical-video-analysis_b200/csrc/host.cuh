// Host-only plumbing shared by the handles and ops of libsurgvid: tensor-map encoding, the state-dict store, weight upload and the
// stream-state registry.  Definitions in api.cu.
#pragma once
#include <map>
#include <string>
#include <vector>

#include "common.cuh"

namespace sv {

// ---- tensor maps: one cached driver-entry-point lookup per encoder; `what` names the map in the error message ----------------
// element strides 1, no interleave, no OOB fill value (out-of-bounds elements read as zero)
int encode_tiled(CUtensorMap* map, CUtensorMapDataType dtype, int rank, const void* base, const cuuint64_t* dims, const cuuint64_t* strides,
                 const cuuint32_t* box, CUtensorMapSwizzle swizzle, CUtensorMapL2promotion l2, const char* what);
// no interleave, no OOB fill value
int encode_im2col(CUtensorMap* map, CUtensorMapDataType dtype, int rank, const void* base, const cuuint64_t* dims, const cuuint64_t* strides,
                  const int* lower, const int* upper, cuuint32_t channels, cuuint32_t pixels, const cuuint32_t* elem_strides,
                  CUtensorMapSwizzle swizzle, CUtensorMapL2promotion l2, const char* what);

// ---- state dict: the tensors a handle was given by name (sv_*_set_tensor), checked and converted by its pack_weights -----------
struct HostTensor {
  std::vector<float> data;
  std::vector<int64_t> shape;
};

struct StateDict {
  std::map<std::string, HostTensor> tensors;
  bool packed = false;   // the handle's device weights were built from `tensors` as they are now

  // Stores a copy of host_data (zeros when it is NULL) and clears `packed`.  shape == NULL with ndim > 0, or a negative dimension:
  // SV_ERR_INVALID.
  int set(const char* name, const float* host_data, const int64_t* shape, int32_t ndim);
  // The tensor `key` with exactly `shape`.  Missing: SV_ERR_STATE, "<who>: missing state_dict key '<key>'"; another shape:
  // SV_ERR_INVALID, "<who>: wrong shape for '<key>'".
  int get(const std::string& key, const std::vector<int64_t>& shape, const char* who, const HostTensor** out) const;
};

// ---- weight upload: *dst becomes a device copy of src on `device`; the previous allocation, if any, is freed ----------------------
int upload_bytes(int device, void** dst, const void* src, size_t bytes);
template <class D, class S>
int upload(int device, D** dst, const std::vector<S>& src) {
  static_assert(sizeof(D) == sizeof(S), "upload: element sizes differ");
  return upload_bytes(device, reinterpret_cast<void**>(dst), src.data(), src.size() * sizeof(S));
}

// ---- stream states ---------------------------------------------------------------------------------------------------------------
// A stream state starts with int64 frame counters seen[n_streams], padded to 256 bytes; the module's rings follow.  The handle is the
// only writer of those counters and keeps a host copy per state address, so that a step is refused before launch when the state was
// not reset through the handle or a stream position would pass 2^31.  `prefix` starts every message ("mstcn stream", "trans stream").
class StreamRegistry {
 public:
  explicit StreamRegistry(const char* prefix) : prefix_(prefix) {}
  static size_t counter_bytes(int32_t n_streams);
  // stream_ids == NULL: zero the whole state (state_bytes >= need) and register it; otherwise zero the counters of stream_ids only
  // (ring rows are read at positions [0, seen) alone, and those are rewritten before they are read again)
  int reset(void* state, size_t state_bytes, size_t need, int32_t n_streams, const int32_t* stream_ids, int32_t n_ids, cudaStream_t st);
  // checks a step's (stream_ids, counts) against the host counters and fills tab: chunk row offsets [n_ids + 1], then stream ids [n_ids]
  int check_step(const void* state, size_t state_bytes, size_t need, int32_t n_streams, const int32_t* stream_ids, const int64_t* counts,
                 int32_t n_ids, std::vector<int64_t>* tab) const;
  // after a step checked by check_step was enqueued
  void advance(const void* state, const int32_t* stream_ids, const int64_t* counts, int32_t n_ids);

 private:
  const char* prefix_;
  std::map<const void*, std::vector<int64_t>> seen_;
};

}  // namespace sv
