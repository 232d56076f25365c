// api.cu — context lifecycle of libgpud_b200.so
#include <stdarg.h>

#include "internal.h"

extern "C" int32_t gpud_abi_version(void) { return GPUD_ABI_VERSION; }

extern "C" int32_t gpud_ctx_create(const int32_t* cuda_devs, int32_t n, gpud_ctx** out) {
  if (!out || n < 1 || n > GPUD_MAX_GPUS || !cuda_devs) return GPUD_E_INVALID;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    cudaGetLastError();
    return GPUD_E_CUDA;   // no CUDA device: there is no CPU fallback on this path
  }
  gpud_ctx* ctx = new gpud_ctx();
  for (int i = 0; i < n; ++i) {
    if (cuda_devs[i] < 0 || cuda_devs[i] >= count) {
      delete ctx;
      return GPUD_E_INVALID;
    }
    ctx->devs.push_back(cuda_devs[i]);
  }
  ctx->scan.assign(n, nullptr);
  ctx->comm.assign(n, nullptr);
  ctx->fabric_tables.assign(n, nullptr);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, ctx->devs[0]) == cudaSuccess) ctx->sm_count = prop.multiProcessorCount;
  // per-call scratch comes from the stream-ordered pool (cudaMallocAsync); keep up to 256 MiB cached across synchronisations,
  // otherwise every call that ends in a sync hands its scratch back to the driver and the next one pays for it again
  for (int i = 0; i < n; ++i) {
    cudaMemPool_t pool;
    unsigned long long keep = 256ull << 20;
    if (cudaDeviceGetDefaultMemPool(&pool, ctx->devs[i]) == cudaSuccess) cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    cudaGetLastError();
  }
  *out = ctx;
  return GPUD_OK;
}

extern "C" int32_t gpud_ctx_destroy(gpud_ctx* ctx) {
  if (!ctx) return GPUD_E_INVALID;
  for (size_t i = 0; i < ctx->devs.size(); ++i) {
    cudaSetDevice(ctx->devs[i]);
    if (ctx->scan[i]) gpud_scan_state_free(ctx->scan[i]);
    if (ctx->comm[i]) gpud_comm_state_free(ctx->comm[i]);
    if (ctx->fabric_tables[i]) cudaFree(ctx->fabric_tables[i]);
  }
  delete ctx;
  return GPUD_OK;
}

extern "C" int32_t gpud_last_error(gpud_ctx* ctx, char* buf, int32_t cap) {
  if (!ctx || !buf || cap < 1) return GPUD_E_INVALID;
  std::lock_guard<std::mutex> g(ctx->mu);
  snprintf(buf, (size_t)cap, "%s", ctx->last_error.c_str());
  return GPUD_OK;
}

extern "C" int32_t gpud_host_alloc(int64_t bytes, void** out) {
  if (!out || bytes <= 0) return GPUD_E_INVALID;
  cudaError_t e = cudaMallocHost(out, (size_t)bytes);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return e == cudaErrorMemoryAllocation ? GPUD_E_NOMEM : GPUD_E_CUDA;
  }
  return GPUD_OK;
}

extern "C" int32_t gpud_host_free(void* p) {
  if (!p) return GPUD_E_INVALID;
  return cudaFreeHost(p) == cudaSuccess ? GPUD_OK : GPUD_E_CUDA;
}

// struct sizes for binding layout checks (ctypes / cgo): 0 hit, 1 fabric_raw, 2 fabric_local, 3 fabric_verdict, 4 ring_cfg,
// 5 kmsg_event, 6 ib_snapshot, 7 ib_verdict, 8 metric, 9 dedup_rule, 10 temperature, 11 poll_counters, 12 event_row, .., 17 drain_info
extern "C" int32_t gpud_sizeof(int32_t which) {
  switch (which) {
    case 0: return (int32_t)sizeof(gpud_xid_hit);
    case 1: return (int32_t)sizeof(gpud_fabric_raw);
    case 2: return (int32_t)sizeof(gpud_fabric_local);
    case 3: return (int32_t)sizeof(gpud_fabric_verdict);
    case 4: return (int32_t)sizeof(gpud_ring_cfg);
    case 5: return (int32_t)sizeof(gpud_kmsg_event);
    case 6: return (int32_t)sizeof(gpud_ib_snapshot);
    case 7: return (int32_t)sizeof(gpud_ib_verdict);
    case 8: return (int32_t)sizeof(gpud_metric);
    case 9: return (int32_t)sizeof(gpud_dedup_rule);
    case 10: return (int32_t)sizeof(gpud_temperature);
    case 11: return (int32_t)sizeof(gpud_poll_counters);
    case 12: return (int32_t)sizeof(gpud_event_row);
    case 13: return (int32_t)sizeof(gpud_nvml_device);
    case 14: return (int32_t)sizeof(gpud_remapped_rows);
    case 15: return (int32_t)sizeof(gpud_ecc_errors);
    case 16: return (int32_t)sizeof(gpud_gpm_metrics);
    case 17: return (int32_t)sizeof(gpud_drain_info);
  }
  return -1;
}
