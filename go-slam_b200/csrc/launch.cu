// launch.cu — see launch.cuh.
#include "launch.cuh"

GsEncodeTiledFn gs_encode_tiled_fn() {
  static const GsEncodeTiledFn fn = []() -> GsEncodeTiledFn {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      return nullptr;
    return reinterpret_cast<GsEncodeTiledFn>(p);
  }();
  return fn;
}

bool GsMapCache::get(const GsMapKey& k, CUtensorMap* out) {
  std::lock_guard<std::mutex> lock(mu_);
  int victim = -1;
  for (int i = 0; i < (int)table_.size(); ++i) {
    Slot& s = table_[i];
    if (s.used && s.key.base == k.base && s.key.kind == k.kind && s.key.dims[0] == k.dims[0] &&
        s.key.dims[1] == k.dims[1] && s.key.dims[2] == k.dims[2] && s.key.dims[3] == k.dims[3]) {
      s.stamp = ++clock_;
      *out = s.map;
      return true;
    }
    // victim: a free slot if there is one, else the least recently used
    if (victim < 0 || (table_[victim].used && (!s.used || s.stamp < table_[victim].stamp))) victim = i;
  }
  Slot& v = table_[victim];
  const GsEncodeTiledFn enc = gs_encode_tiled_fn();
  if (!enc || !encode_(enc, k, &v.map)) { v.used = false; return false; }
  v.key = k; v.used = true; v.stamp = ++clock_;
  *out = v.map;
  return true;
}

static std::mutex g_device_mu;

int gs_device_once(GsDeviceOnce& once, cudaError_t (*init)(int dev)) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) { gs_note_cuda_error(e); return GOSLAM_ELAUNCH; }
  if (dev < 0 || dev >= kGsMaxDevices) return GOSLAM_EINVAL;
  std::lock_guard<std::mutex> lock(g_device_mu);
  if (once.done[dev]) return GOSLAM_OK;
  e = init(dev);
  if (e != cudaSuccess) { gs_note_cuda_error(e); return GOSLAM_ELAUNCH; }
  once.done[dev] = true;
  return GOSLAM_OK;
}

static GsDeviceOnce g_sm_once;
static int g_sm_count[kGsMaxDevices];

static cudaError_t sm_count_init(int dev) {
  return cudaDeviceGetAttribute(&g_sm_count[dev], cudaDevAttrMultiProcessorCount, dev);
}

int gs_sm_count() {
  int dev = 0;
  if (gs_device_once(g_sm_once, sm_count_init) != GOSLAM_OK || cudaGetDevice(&dev) != cudaSuccess) return 148;
  return g_sm_count[dev];
}
