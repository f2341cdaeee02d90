// launch.cuh — host-side launch plumbing shared by the kernel files: the driver's tensor-map encoder, an LRU cache
// of encoded tensor maps, and once-per-device set-up (function attributes, constant memory, SM count).
#pragma once
#include "common.cuh"
#include <cuda.h>
#include <mutex>
#include <vector>

typedef CUresult (*GsEncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// cuTensorMapEncodeTiled, looked up in the driver once per process; nullptr if the driver does not have it
GsEncodeTiledFn gs_encode_tiled_fn();

// What a tensor map is encoded from: the base pointer, which of the owner's map formats, and up to four sizes.
struct GsMapKey {
  const void* base;
  int kind;
  int dims[4];
};

// Tensor maps depend only on their key, and the kernels' callers launch on the same buffers call after call, so the
// driver's encode (1.5-2 us of host time each) is paid once per key.  Most-recently-used table shared by all threads;
// each kernel file owns one, with the encode function of its own map formats.
class GsMapCache {
 public:
  typedef bool (*EncodeFn)(GsEncodeTiledFn enc, const GsMapKey& key, CUtensorMap* out);
  GsMapCache(int slots, EncodeFn encode) : table_(slots), encode_(encode) {}
  // false if the driver has no encoder or rejects the map
  bool get(const GsMapKey& key, CUtensorMap* out);

 private:
  struct Slot { GsMapKey key; CUtensorMap map; unsigned long long stamp; bool used; };
  std::vector<Slot> table_;
  EncodeFn encode_;
  unsigned long long clock_ = 0;
  std::mutex mu_;
};

// Per-device one-time set-up.  Function attributes (opt-in shared memory) and constant memory belong to a device, so
// a process that uses a second GPU must set them there too.
constexpr int kGsMaxDevices = 64;
struct GsDeviceOnce { bool done[kGsMaxDevices] = {}; };

// Runs init(dev) for the current device unless it has succeeded there before; calls are serialised.  Returns GOSLAM_OK,
// GOSLAM_ELAUNCH if init fails (the error is kept for goslam_last_cuda_error and init runs again on the next call), or
// GOSLAM_EINVAL for a device ordinal of kGsMaxDevices or more.
int gs_device_once(GsDeviceOnce& once, cudaError_t (*init)(int dev));

// multiprocessor count of the current device, queried once per device
int gs_sm_count();
