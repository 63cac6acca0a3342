// The NDArray handle of the flat C ABI, shared by c_api_runtime.cc (NDArray / serializer functions), c_api_extra.cc and c_api_graph.cc
// (executor bindings, imperative invoke, autograd).  Reference role: the NDArrayHandle of include/mxnet/c_api.h:60.
//
// Two kinds of array: a host array keeps its bytes in rec.data; a device array (GXNDArrayCreateEx with dev_type 2) keeps float32 data in
// device memory from the native pool (storage_gpu.cu) on device `dev_id`, and rec.data stays empty.  Every reader of host bytes goes through
// HostBytes(), which refuses device arrays, so no entry point reads a device pointer as host memory.
#pragma once
#include <cstdint>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "params_io.h"

namespace gxrt {
namespace capi {

struct AGNode;                          // autograd history of an array (c_api_graph.cc)

struct HostArray {
  gxrt::NDRec rec;                      // device arrays: shape and dtype only
  std::vector<uint32_t> shape32;        // GetShape hands out a pointer that stays valid until the handle is freed
  std::shared_ptr<AGNode> ag;           // set while the array is a marked variable or the output of a recorded operator
  int ag_out = 0;                       // which output of that operator
  HostArray* grad = nullptr;            // marked variables: where Backward writes (not owned)
  int grad_req = 0;
  int dev_id = -1;                      // >= 0: a device array on this CUDA device
  float* dptr = nullptr;                // its data
  bool owns_dptr = false;               // false: a view of executor memory (GXExecutorOutputs)
  bool device() const { return dev_id >= 0; }
  size_t Bytes() const;                 // payload size, host or device
  ~HostArray();
};

inline HostArray* ND(void* h) {
  if (h == nullptr) throw std::runtime_error("null NDArray handle");
  return static_cast<HostArray*>(h);
}

// the host bytes of `a`; `fn` names the entry point in the error raised for a device array
inline std::string& HostBytes(HostArray* a, const char* fn) {
  if (a->device()) throw std::runtime_error(std::string(fn) + ": device array (this function works on host arrays only)");
  return a->rec.data;
}

// device arrays (c_api_runtime.cc): allocation from the pool of `dev` (zero-filled), and a host copy of the contents as an NDRec
HostArray* NewDeviceArray(const std::vector<int64_t>& shape, int dev);
void ReleaseDevice(HostArray* a);       // gives an owned device buffer back to the pool (the destructor calls it)
gxrt::NDRec HostCopy(const HostArray* a);
void SyncDevice(int dev);               // waits for the library stream of `dev`
void SyncAllDevices();                  // ... of every device an array was created on
// whether [p, p + bytes) lies inside a live device array: raw-pointer entry points (KVStore, predictor) refuse such buffers
bool IsDeviceBuffer(const void* p);

}  // namespace capi
}  // namespace gxrt
