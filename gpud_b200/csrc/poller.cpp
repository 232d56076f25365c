// poller.cpp — real ingest (SURVEY.md 8f.3): the host poller that reads the NVML gauges of one GPU and feeds K1 with raw
// uint32 poll rows through pinned memory (gpud_ring_push_timed: every row carries the wall-clock ms its getters returned at, which
// the streaming drain turns into the end time of each window).  The getters are the ones the reference's components call
// once per minute and widen with metric.Set(float64(v)):
//   temperature C     dev.GetTemperature(nvml.TEMPERATURE_GPU)        components/accelerator/nvidia/temperature/temperature.go:85
//   power mW          dev.GetPowerUsage()                              components/accelerator/nvidia/power/power.go:46
//   graphics / mem MHz dev.GetClockInfo(CLOCK_GRAPHICS / CLOCK_MEM)    components/accelerator/nvidia/clock-speed/clock_speed.go:41,59
//   SM MHz            nvmlDeviceGetClockInfo(NVML_CLOCK_SM)
//   gpu / mem util %  dev.GetUtilizationRates()                        components/accelerator/nvidia/utilization/utilization.go:44
//   memory used MiB   dev.GetMemoryInfo()                              components/accelerator/nvidia/memory/memory.go:83
// NVML is dlopen'ed (libnvidia-ml.so.1 ships with the driver, not with CUDA).  A getter that fails - unsupported or transient -
// never puts a sentinel into the ring: its column repeats the last good value and the failure is recorded beside the rows
// (gpud_poll_row_hold / gpud_poller_errors), like the reference's "...Supported = false" fields next to an unset gauge.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <time.h>

#include <algorithm>
#include <string>
#include <vector>

#include "internal.h"

namespace {

typedef int nvmlReturn_t;
typedef struct nvmlDevice_st* nvmlDevice_t;
struct nvmlUtilization_t { unsigned int gpu, memory; };
struct nvmlMemory_t { unsigned long long total, free, used; };

struct Nvml {
  void* so = nullptr;
  nvmlReturn_t (*init)() = nullptr;
  nvmlReturn_t (*by_pci)(const char*, nvmlDevice_t*) = nullptr;
  nvmlReturn_t (*temperature)(nvmlDevice_t, int, unsigned int*) = nullptr;
  nvmlReturn_t (*power)(nvmlDevice_t, unsigned int*) = nullptr;
  nvmlReturn_t (*clock)(nvmlDevice_t, int, unsigned int*) = nullptr;
  nvmlReturn_t (*util)(nvmlDevice_t, nvmlUtilization_t*) = nullptr;
  nvmlReturn_t (*memory)(nvmlDevice_t, nvmlMemory_t*) = nullptr;
  const char* (*err)(nvmlReturn_t) = nullptr;
  nvmlReturn_t (*name)(nvmlDevice_t, char*, unsigned int) = nullptr;
  nvmlReturn_t (*link_state)(nvmlDevice_t, unsigned int, int*) = nullptr;
  nvmlReturn_t (*link_errors)(nvmlDevice_t, unsigned int, int, unsigned long long*) = nullptr;
  nvmlReturn_t (*fabric_v)(nvmlDevice_t, void*) = nullptr;
  nvmlReturn_t (*p2p)(nvmlDevice_t, nvmlDevice_t, int, int*) = nullptr;
  nvmlReturn_t (*temp_threshold)(nvmlDevice_t, int, unsigned int*) = nullptr;
  nvmlReturn_t (*margin_temp)(nvmlDevice_t, void*) = nullptr;
  nvmlReturn_t (*clock_reasons)(nvmlDevice_t, unsigned long long*) = nullptr;
  nvmlReturn_t (*ecc_total)(nvmlDevice_t, int, int, unsigned long long*) = nullptr;
  nvmlReturn_t (*ecc_mode)(nvmlDevice_t, int*, int*) = nullptr;
  nvmlReturn_t (*ecc_location)(nvmlDevice_t, int, int, int, unsigned long long*) = nullptr;
  nvmlReturn_t (*remapped_rows)(nvmlDevice_t, unsigned int*, unsigned int*, unsigned int*, unsigned int*) = nullptr;
  nvmlReturn_t (*field_values)(nvmlDevice_t, int, void*) = nullptr;
  nvmlReturn_t (*uuid)(nvmlDevice_t, char*, unsigned int) = nullptr;
  nvmlReturn_t (*count)(unsigned int*) = nullptr;
  nvmlReturn_t (*by_index)(unsigned int, nvmlDevice_t*) = nullptr;
  nvmlReturn_t (*pci_info)(nvmlDevice_t, void*) = nullptr;
  nvmlReturn_t (*driver_version)(char*, unsigned int) = nullptr;
  nvmlReturn_t (*gpm_support)(nvmlDevice_t, void*) = nullptr;
  nvmlReturn_t (*gpm_alloc)(void**) = nullptr;
  nvmlReturn_t (*gpm_free)(void*) = nullptr;
  nvmlReturn_t (*gpm_sample)(nvmlDevice_t, void*) = nullptr;
  nvmlReturn_t (*gpm_metrics)(void*) = nullptr;
};

Nvml* nvml() {
  static Nvml n;
  static bool tried = false;
  if (!tried) {
    tried = true;
    n.so = dlopen("libnvidia-ml.so.1", RTLD_NOW | RTLD_GLOBAL);
    if (n.so) {
      *(void**)&n.init = dlsym(n.so, "nvmlInit_v2");
      *(void**)&n.by_pci = dlsym(n.so, "nvmlDeviceGetHandleByPciBusId_v2");
      *(void**)&n.temperature = dlsym(n.so, "nvmlDeviceGetTemperature");
      *(void**)&n.power = dlsym(n.so, "nvmlDeviceGetPowerUsage");
      *(void**)&n.clock = dlsym(n.so, "nvmlDeviceGetClockInfo");
      *(void**)&n.util = dlsym(n.so, "nvmlDeviceGetUtilizationRates");
      *(void**)&n.memory = dlsym(n.so, "nvmlDeviceGetMemoryInfo");
      *(void**)&n.err = dlsym(n.so, "nvmlErrorString");
      *(void**)&n.name = dlsym(n.so, "nvmlDeviceGetName");
      *(void**)&n.link_state = dlsym(n.so, "nvmlDeviceGetNvLinkState");
      *(void**)&n.link_errors = dlsym(n.so, "nvmlDeviceGetNvLinkErrorCounter");
      *(void**)&n.fabric_v = dlsym(n.so, "nvmlDeviceGetGpuFabricInfoV");           // driver >= 550 (fabric_state.go:262-267); absent symbol = not supported
      *(void**)&n.p2p = dlsym(n.so, "nvmlDeviceGetP2PStatus");
      *(void**)&n.temp_threshold = dlsym(n.so, "nvmlDeviceGetTemperatureThreshold");
      *(void**)&n.margin_temp = dlsym(n.so, "nvmlDeviceGetMarginTemperature");
      *(void**)&n.clock_reasons = dlsym(n.so, "nvmlDeviceGetCurrentClocksEventReasons");
      if (!n.clock_reasons) *(void**)&n.clock_reasons = dlsym(n.so, "nvmlDeviceGetCurrentClocksThrottleReasons");   // the pre-535 name of the same getter
      *(void**)&n.ecc_total = dlsym(n.so, "nvmlDeviceGetTotalEccErrors");
      *(void**)&n.ecc_mode = dlsym(n.so, "nvmlDeviceGetEccMode");
      *(void**)&n.ecc_location = dlsym(n.so, "nvmlDeviceGetMemoryErrorCounter");
      *(void**)&n.remapped_rows = dlsym(n.so, "nvmlDeviceGetRemappedRows");
      *(void**)&n.field_values = dlsym(n.so, "nvmlDeviceGetFieldValues");
      *(void**)&n.uuid = dlsym(n.so, "nvmlDeviceGetUUID");
      *(void**)&n.count = dlsym(n.so, "nvmlDeviceGetCount_v2");
      *(void**)&n.by_index = dlsym(n.so, "nvmlDeviceGetHandleByIndex_v2");
      *(void**)&n.pci_info = dlsym(n.so, "nvmlDeviceGetPciInfo_v3");
      *(void**)&n.driver_version = dlsym(n.so, "nvmlSystemGetDriverVersion");
      *(void**)&n.gpm_support = dlsym(n.so, "nvmlGpmQueryDeviceSupport");     // driver >= 520; absent symbols = not supported
      *(void**)&n.gpm_alloc = dlsym(n.so, "nvmlGpmSampleAlloc");
      *(void**)&n.gpm_free = dlsym(n.so, "nvmlGpmSampleFree");
      *(void**)&n.gpm_sample = dlsym(n.so, "nvmlGpmSampleGet");
      *(void**)&n.gpm_metrics = dlsym(n.so, "nvmlGpmMetricsGet");
      if (!n.init || !n.by_pci || !n.temperature || !n.power || !n.clock || !n.util || !n.memory || n.init() != 0) { dlclose(n.so); n.so = nullptr; }
    }
  }
  return n.so ? &n : nullptr;
}

}  // namespace

struct gpud_poller {
  gpud_ctx* ctx = nullptr;
  gpud_ring* ring = nullptr;
  int dev = 0;
  nvmlDevice_t h = nullptr;
  uint32_t* rows = nullptr;      // pinned [cap_rows][GPUD_POLL_N_FIELDS]
  int64_t cap_rows = 0, n_rows = 0;
  double last_poll_s = 0.0;      // wall time of the last gpud_poller_poll call
  uint32_t held[GPUD_POLL_N_FIELDS] = {0};       // last good value per column (what a failed getter's column repeats)
  uint32_t fail_mask = 0;                        // columns that failed at least once since create
  int32_t last_rc[GPUD_POLL_N_FIELDS] = {0};     // the NVML return code of each column's last failure
  uint64_t n_failed[GPUD_POLL_N_FIELDS] = {0};
  uint64_t* field_rows = nullptr;                // pinned [cap_rows][GPUD_FIELD_ROW_N] (gpud_poller_poll_fields)
  uint64_t field_held[GPUD_FIELD_ROW_N] = {0};
  double gpm_held[GPUD_GPM_N] = {0};
  std::vector<int64_t> row_ms;                   // [cap_rows]: unix ms of each row of the batch being polled
  int64_t last_ms = INT64_MIN;                   // the newest row time handed out (row times never go back, even if the clock does)
};

// CLOCK_REALTIME in ms, taken as soon as a row's getters have returned; clamped so that a clock step back cannot make a row older
// than the one before it (gpud_ring_push_timed refuses that)
static int64_t row_time_ms(gpud_poller* p) {
  timespec ts;
  clock_gettime(CLOCK_REALTIME, &ts);
  p->last_ms = std::max(p->last_ms, (int64_t)ts.tv_sec * 1000 + ts.tv_nsec / 1000000);
  return p->last_ms;
}

extern "C" int32_t gpud_poller_create(gpud_ctx* ctx, int32_t dev, gpud_ring* ring, gpud_poller** out) {
  if (!ctx || !ring || !out) return GPUD_E_INVALID;
  Nvml* N = nvml();
  if (!N) return gpud_fail(ctx, GPUD_E_UNSUPPORTED, "libnvidia-ml.so.1 not available (no driver on this host)");
  if (gpud_ring_n_fields(ring) != GPUD_POLL_N_FIELDS) return gpud_fail(ctx, GPUD_E_INVALID, "the gauge poller needs a ring of %d fields (this one has %d)", GPUD_POLL_N_FIELDS, gpud_ring_n_fields(ring));
  char bus[32];
  GPUD_CUDA(ctx, cudaDeviceGetPCIBusId(bus, sizeof bus, dev));
  nvmlDevice_t h;
  const nvmlReturn_t rc = N->by_pci(bus, &h);
  if (rc != 0) return gpud_fail(ctx, GPUD_E_UNSUPPORTED, "nvmlDeviceGetHandleByPciBusId(%s): %s", bus, N->err ? N->err(rc) : "error");
  gpud_poller* p = new gpud_poller();
  p->ctx = ctx; p->ring = ring; p->dev = dev; p->h = h;
  p->cap_rows = 1 << 14;
  p->row_ms.assign((size_t)p->cap_rows, 0);
  if (cudaMallocHost(&p->rows, (size_t)p->cap_rows * GPUD_POLL_N_FIELDS * sizeof(uint32_t)) != cudaSuccess) {
    delete p;
    return gpud_fail(ctx, GPUD_E_CUDA, "pinned poll buffer");
  }
  *out = p;
  return GPUD_OK;
}

extern "C" void gpud_poller_destroy(gpud_poller* p) {
  if (!p) return;
  if (p->rows) cudaFreeHost(p->rows);
  if (p->field_rows) cudaFreeHost(p->field_rows);
  delete p;
}

// The poller's rule for a getter that fails (oracle/SPEC.md "poll rows"): the column HOLDS its last good value (0 before the first
// good read) and the failure is recorded beside the row - a sentinel must never reach the ring, where it would be aggregated as a
// 4.29e9 reading.  Pure, exported for the CPU tests.
extern "C" int32_t gpud_poll_row_hold(const uint32_t* fresh, const int32_t* nvml_rc, int32_t n_cols, uint32_t* held, uint32_t* row_out, uint32_t* fail_mask) {
  if (!fresh || !nvml_rc || !held || !row_out || n_cols < 0 || n_cols > 32) return GPUD_E_INVALID;
  uint32_t mask = 0;
  for (int32_t c = 0; c < n_cols; ++c) {
    if (nvml_rc[c] == 0) held[c] = fresh[c];
    else mask |= 1u << c;
    row_out[c] = held[c];
  }
  if (fail_mask) *fail_mask = mask;
  return GPUD_OK;
}

// one poll row: eight getters, in GPUD_POLL_* order
static void poll_row(Nvml* N, gpud_poller* p, uint32_t* r) {
  unsigned int v = 0;
  uint32_t fresh[GPUD_POLL_N_FIELDS] = {0};
  int32_t rc[GPUD_POLL_N_FIELDS];
  rc[GPUD_POLL_TEMPERATURE_C] = (int32_t)N->temperature(p->h, 0 /* NVML_TEMPERATURE_GPU */, &v); fresh[GPUD_POLL_TEMPERATURE_C] = v;
  rc[GPUD_POLL_POWER_MW] = (int32_t)N->power(p->h, &v); fresh[GPUD_POLL_POWER_MW] = v;
  rc[GPUD_POLL_CLOCK_GRAPHICS_MHZ] = (int32_t)N->clock(p->h, 0 /* NVML_CLOCK_GRAPHICS */, &v); fresh[GPUD_POLL_CLOCK_GRAPHICS_MHZ] = v;
  rc[GPUD_POLL_CLOCK_SM_MHZ] = (int32_t)N->clock(p->h, 1 /* NVML_CLOCK_SM */, &v); fresh[GPUD_POLL_CLOCK_SM_MHZ] = v;
  rc[GPUD_POLL_CLOCK_MEM_MHZ] = (int32_t)N->clock(p->h, 2 /* NVML_CLOCK_MEM */, &v); fresh[GPUD_POLL_CLOCK_MEM_MHZ] = v;
  nvmlUtilization_t u{};
  rc[GPUD_POLL_UTIL_GPU_PCT] = rc[GPUD_POLL_UTIL_MEM_PCT] = (int32_t)N->util(p->h, &u);
  fresh[GPUD_POLL_UTIL_GPU_PCT] = u.gpu; fresh[GPUD_POLL_UTIL_MEM_PCT] = u.memory;
  nvmlMemory_t m{};
  rc[GPUD_POLL_MEMORY_USED_MIB] = (int32_t)N->memory(p->h, &m); fresh[GPUD_POLL_MEMORY_USED_MIB] = (uint32_t)(m.used >> 20);
  uint32_t mask = 0;
  gpud_poll_row_hold(fresh, rc, GPUD_POLL_N_FIELDS, p->held, r, &mask);
  if (mask) {
    p->fail_mask |= mask;
    for (int c = 0; c < GPUD_POLL_N_FIELDS; ++c) if (mask & (1u << c)) { p->last_rc[c] = rc[c]; ++p->n_failed[c]; }
  }
}

extern "C" int32_t gpud_poller_errors(gpud_poller* p, uint32_t* fail_mask, int32_t* last_nvml_rc, uint64_t* n_failed) {
  if (!p) return GPUD_E_INVALID;
  if (fail_mask) *fail_mask = p->fail_mask;
  for (int c = 0; c < GPUD_POLL_N_FIELDS; ++c) {
    if (last_nvml_rc) last_nvml_rc[c] = p->last_rc[c];
    if (n_failed) n_failed[c] = p->n_failed[c];
  }
  return GPUD_OK;
}

extern "C" int32_t gpud_poller_poll(gpud_poller* p, int64_t n_polls, int64_t interval_us) {
  if (!p || n_polls < 0 || interval_us < 0) return GPUD_E_INVALID;
  Nvml* N = nvml();
  if (!N) return GPUD_E_UNSUPPORTED;
  timespec t0, t1;
  clock_gettime(CLOCK_MONOTONIC, &t0);
  int64_t done = 0;
  while (done < n_polls) {
    const int64_t batch = std::min<int64_t>(p->cap_rows, n_polls - done);
    for (int64_t i = 0; i < batch; ++i) {
      poll_row(N, p, p->rows + i * GPUD_POLL_N_FIELDS);
      p->row_ms[i] = row_time_ms(p);
      if (interval_us) { timespec ts{(time_t)(interval_us / 1000000), (long)(interval_us % 1000000) * 1000L}; nanosleep(&ts, nullptr); }
    }
    p->n_rows = batch;
    const int32_t rc = gpud_ring_push_timed(p->ring, p->rows, batch, GPUD_DT_U32, p->row_ms.data());   // pinned: direct DMA + widening append, synchronous return
    if (rc) return rc;
    done += batch;
  }
  clock_gettime(CLOCK_MONOTONIC, &t1);
  p->last_poll_s = (double)(t1.tv_sec - t0.tv_sec) + 1e-9 * (double)(t1.tv_nsec - t0.tv_nsec);
  return GPUD_OK;
}

extern "C" int32_t gpud_poller_last_rows(gpud_poller* p, uint32_t* rows, int64_t cap_rows, int64_t* n_rows, double* seconds) {
  if (!p) return GPUD_E_INVALID;
  const int64_t n = std::min(cap_rows, p->n_rows);
  if (n > 0 && rows) memcpy(rows, p->rows, (size_t)n * GPUD_POLL_N_FIELDS * sizeof(uint32_t));
  if (n_rows) *n_rows = p->n_rows;
  if (seconds) *seconds = p->last_poll_s;
  return GPUD_OK;
}

// ---- NVLink / fabric record of this poller's GPU, straight from NVML (SURVEY.md 8a rows A3, A13) -------------------------------
namespace {
constexpr nvmlReturn_t kNvmlNotSupported = 3, kNvmlGpuLost = 15, kNvmlResetRequired = 16;     // nvml.h nvmlReturn_t
// nvmlGpuFabricInfo_v3_t (nvml.h): version, clusterUuid[16], status, cliqueId, state, healthMask, healthSummary
struct FabricInfoV3 { unsigned int version; unsigned char cluster_uuid[16]; nvmlReturn_t status; unsigned int clique_id; unsigned char state; unsigned int health_mask;
                      unsigned char health_summary; };
static_assert(sizeof(FabricInfoV3) == 40, "nvmlGpuFabricInfo_v3_t layout");
// pkg/nvidia/errors/error.go:33-92: the code, or the driver's error string saying so (lower-cased, trimmed, substring)
std::string norm(const char* e) {
  std::string h = e ? e : "";
  for (char& c : h) if (c >= 'A' && c <= 'Z') c = (char)(c - 'A' + 'a');
  const size_t a = h.find_first_not_of(" \t\r\n\v\f"), b = h.find_last_not_of(" \t\r\n\v\f");
  return a == std::string::npos ? std::string() : h.substr(a, b - a + 1);
}
bool has(const std::string& h, const char* needle) { return h.find(needle) != std::string::npos; }
bool classify_not_supported(nvmlReturn_t r, const char* errstr) { return r == kNvmlNotSupported || has(norm(errstr), "not supported"); }
bool classify_gpu_lost(nvmlReturn_t r, const char* errstr) {
  if (r == kNvmlGpuLost) return true;
  const std::string e = norm(errstr);
  return has(e, "gpu lost") || has(e, "gpu is lost") || has(e, "gpu_is_lost");
}
bool classify_reset_required(nvmlReturn_t r, const char* errstr) {
  if (r == kNvmlResetRequired) return true;
  const std::string e = norm(errstr);
  return has(e, "gpu requires reset") || has(e, "gpu reset");
}
bool is_not_supported(Nvml* N, nvmlReturn_t r) { return classify_not_supported(r, N->err ? N->err(r) : ""); }
bool is_gpu_lost(Nvml* N, nvmlReturn_t r) { return classify_gpu_lost(r, N->err ? N->err(r) : ""); }
bool is_reset_required(Nvml* N, nvmlReturn_t r) { return classify_reset_required(r, N->err ? N->err(r) : ""); }
}  // namespace

extern "C" int32_t gpud_poller_product_name(gpud_poller* p, char* out, int32_t cap) {
  if (!p || !out || cap <= 0) return GPUD_E_INVALID;
  Nvml* N = nvml();
  if (!N || !N->name) return GPUD_E_UNSUPPORTED;
  const nvmlReturn_t rc = N->name(p->h, out, (unsigned int)cap);
  if (rc != 0) return gpud_fail(p->ctx, GPUD_E_UNSUPPORTED, "nvmlDeviceGetName: %s", N->err ? N->err(rc) : "error");
  return GPUD_OK;
}

// GetNVLink (nvlink/nvlink.go:93-168), GetFabricState's V3 query (pkg/nvidia/nvml/device/fabric_state.go:268-306) and
// getPeerNVLinkP2PStatus (nvlink/p2p.go:21-50) for one GPU.
extern "C" int32_t gpud_poller_fabric_raw(gpud_poller* p, uint32_t gpu_index, const char* const* peer_bus_ids, int32_t n_peers, gpud_fabric_raw* out) {
  if (!p || !out || n_peers < 0 || n_peers > GPUD_MAX_GPUS || (n_peers && !peer_bus_ids) || gpu_index >= GPUD_MAX_GPUS) return GPUD_E_INVALID;
  Nvml* N = nvml();
  if (!N || !N->link_state || !N->link_errors) return gpud_fail(p->ctx, GPUD_E_UNSUPPORTED, "NVML NVLink getters not available");
  memset(out, 0, sizeof *out);
  out->gpu_index = gpu_index;
  out->nvlink_supported = 1;
  for (unsigned int link = 0; link < GPUD_MAX_LINKS; ++link) {
    int active = 0;
    const nvmlReturn_t rc = N->link_state(p->h, link, &active);
    if (is_not_supported(N, rc)) {               // on link 0: no NVLink hardware; later: fewer links than NVML_NVLINK_MAX_LINKS
      if (out->n_links == 0) out->nvlink_supported = 0;
      break;
    }
    if (is_gpu_lost(N, rc)) return gpud_fail(p->ctx, GPUD_E_STATE, "GPU lost");                  // nvmlerrors.ErrGPULost
    if (is_reset_required(N, rc)) return gpud_fail(p->ctx, GPUD_E_STATE, "GPU requires reset");  // nvmlerrors.ErrGPURequiresReset
    if (rc != 0) continue;                       // "failed get nvlink state -- retrying": the link is left out of States
    const uint32_t i = out->n_links++;
    out->link_feature_enabled[i] = active == 1 /* NVML_FEATURE_ENABLED */ ? 1 : 0;
    unsigned long long v = 0;
    if (N->link_errors(p->h, link, 0 /* NVML_NVLINK_ERROR_DL_REPLAY */, &v) == 0) out->link_replay_errors[i] = v;
    if (N->link_errors(p->h, link, 1 /* NVML_NVLINK_ERROR_DL_RECOVERY */, &v) == 0) out->link_recovery_errors[i] = v;
    if (N->link_errors(p->h, link, 2 /* NVML_NVLINK_ERROR_DL_CRC_FLIT */, &v) == 0) out->link_crc_errors[i] = v;
  }
  // fabric state: the V3 structure carries the health mask and summary; anything else = no fabric telemetry for this GPU
  if (N->fabric_v) {
    FabricInfoV3 fi;
    memset(&fi, 0, sizeof fi);
    fi.version = (unsigned int)sizeof(FabricInfoV3) | (3u << 24);             // NVML_STRUCT_VERSION(GpuFabricInfo, 3)
    const nvmlReturn_t rc = N->fabric_v(p->h, &fi);
    if (is_gpu_lost(N, rc)) return gpud_fail(p->ctx, GPUD_E_STATE, "GPU lost");
    if (is_reset_required(N, rc)) return gpud_fail(p->ctx, GPUD_E_STATE, "GPU requires reset");
    if (rc == 0) {
      out->fabric_valid = 1;
      out->fabric_state = fi.state;
      out->fabric_summary = fi.health_summary;
      out->fabric_status = (int32_t)fi.status;
      out->fabric_health_mask = fi.health_mask;
      out->clique_id = fi.clique_id;
    }
  }
  char name[96] = {0};
  if (N->name && N->name(p->h, name, sizeof name) == 0)
    out->system_expected_nvlink = (gpud_product_fm_supported(name) || gpud_product_fabric_state_supported(name)) ? 1u : 0u;   // nvlink/component.go:164-183
  for (int j = 0; j < GPUD_MAX_GPUS; ++j) out->p2p_status[j] = GPUD_P2P_UNPROBED;
  if (N->p2p) {
    for (int32_t j = 0; j < n_peers; ++j) {
      if ((uint32_t)j == gpu_index || !peer_bus_ids[j] || !*peer_bus_ids[j]) continue;
      nvmlDevice_t peer;
      if (N->by_pci(peer_bus_ids[j], &peer) != 0) continue;
      int st = 6;
      if (N->p2p(p->h, peer, 2 /* NVML_P2P_CAPS_INDEX_NVLINK */, &st) != 0) continue;           // a failed probe stays unprobed (component.go:430-447)
      out->p2p_status[j] = (uint8_t)((st >= 0 && st <= 5) ? st : 6);                            // toP2PStatusCode: anything else is "U"
    }
  }
  return GPUD_OK;
}

// GetTemperature (temperature/temperature.go:78-221): current GPU and HBM sensors, the thermal margin, the four thresholds.  A
// getter that fails leaves its field 0 / unsupported like the reference; GPU lost / requires reset end the read.
extern "C" int32_t gpud_poller_temperature(gpud_poller* p, gpud_temperature* out) {
  if (!p || !out) return GPUD_E_INVALID;
  Nvml* N = nvml();
  if (!N) return GPUD_E_UNSUPPORTED;
  memset(out, 0, sizeof *out);
  auto fatal = [&](nvmlReturn_t rc) -> int32_t {
    if (is_gpu_lost(N, rc)) return gpud_fail(p->ctx, GPUD_E_STATE, "GPU lost");
    if (is_reset_required(N, rc)) return gpud_fail(p->ctx, GPUD_E_STATE, "GPU requires reset");
    return GPUD_OK;
  };
  unsigned int v = 0;
  nvmlReturn_t rc = N->temperature(p->h, 0 /* NVML_TEMPERATURE_GPU */, &v);
  if (rc == 0) out->current_gpu_core_c = v; else if (int32_t e = fatal(rc)) return e;
  rc = N->temperature(p->h, 1 /* temperatureSensorMemory, temperature.go:75 */, &v);
  if (rc == 0) { out->current_hbm_c = v; out->hbm_supported = 1; } else if (int32_t e = fatal(rc)) return e;
  if (N->margin_temp) {
    struct { unsigned int version; int margin; } mt = {(unsigned int)(8u | (1u << 24)) /* nvmlMarginTemperature_v1 */, 0};
    rc = N->margin_temp(p->h, &mt);
    if (rc == 0) { out->slowdown_margin_c = mt.margin; out->margin_supported = 1; } else if (int32_t e = fatal(rc)) return e;
  }
  if (N->temp_threshold) {
    uint32_t* dst[4] = {&out->threshold_shutdown_c, &out->threshold_slowdown_c, &out->threshold_mem_max_c, &out->threshold_gpu_max_c};
    for (int t = 0; t < 4; ++t) {                  // NVML_TEMPERATURE_THRESHOLD_SHUTDOWN, _SLOWDOWN, _MEM_MAX, _GPU_MAX = 0..3
      rc = N->temp_threshold(p->h, t, &v);
      if (rc == 0) *dst[t] = v; else if (int32_t e = fatal(rc)) return e;
    }
  }
  return GPUD_OK;
}

// GetClockEvents (hw-slowdown/clock_events.go:111-166: the reasons bitmask, decoded by gpud_clock_event_reasons) and the four ECC
// totals of GetECCErrors (ecc/ecc_errors.go:136-240).
extern "C" int32_t gpud_poller_counters(gpud_poller* p, gpud_poll_counters* out) {
  if (!p || !out) return GPUD_E_INVALID;
  Nvml* N = nvml();
  if (!N) return GPUD_E_UNSUPPORTED;
  memset(out, 0, sizeof *out);
  if (N->clock_reasons) {
    unsigned long long m = 0;
    const nvmlReturn_t rc = N->clock_reasons(p->h, &m);
    if (rc == 0) { out->clock_event_reasons = m; out->clock_events_supported = 1; }
    else if (is_gpu_lost(N, rc)) return gpud_fail(p->ctx, GPUD_E_STATE, "GPU lost");
    else if (is_reset_required(N, rc)) return gpud_fail(p->ctx, GPUD_E_STATE, "GPU requires reset");
    else if (!is_not_supported(N, rc)) return gpud_fail(p->ctx, GPUD_E_STATE, "failed to get device clock event reasons: %s", N->err ? N->err(rc) : "error");
  }
  if (N->ecc_total) {
    // (errorType, counterType): aggregate corrected / uncorrected, volatile corrected / uncorrected -- the reference's order
    const int q[4][2] = {{0, 1}, {1, 1}, {0, 0}, {1, 0}};   // NVML_MEMORY_ERROR_TYPE_CORRECTED 0 / UNCORRECTED 1 ; NVML_VOLATILE_ECC 0 / AGGREGATE_ECC 1
    uint64_t* dst[4] = {&out->ecc_aggregate_corrected, &out->ecc_aggregate_uncorrected, &out->ecc_volatile_corrected, &out->ecc_volatile_uncorrected};
    for (int i = 0; i < 4; ++i) {
      unsigned long long c = 0;
      const nvmlReturn_t rc = N->ecc_total(p->h, q[i][0], q[i][1], &c);
      if (rc == 0) { *dst[i] = c; out->ecc_read_mask |= 1u << i; }
      else if (is_gpu_lost(N, rc)) return gpud_fail(p->ctx, GPUD_E_STATE, "GPU lost");
      else if (is_reset_required(N, rc)) return gpud_fail(p->ctx, GPUD_E_STATE, "GPU requires reset");
    }
  }
  return GPUD_OK;
}

// test entry (not in gpud_b200.h): the error classes of pkg/nvidia/errors for a return code and the text nvmlErrorString gave for it:
// bit 1 not supported, 2 GPU lost, 4 GPU requires reset
extern "C" int32_t gpudh_nvml_error_class(int32_t ret, const char* error_string) {
  return (classify_not_supported(ret, error_string) ? 1 : 0) | (classify_gpu_lost(ret, error_string) ? 2 : 0) | (classify_reset_required(ret, error_string) ? 4 : 0);
}

extern "C" int32_t gpud_nvml_error_strings_from_driver(void) {
  Nvml* N = nvml();
  if (!N || !N->err) return GPUD_E_UNSUPPORTED;
  gpud_set_nvml_error_string((gpud_nvml_error_string_fn)N->err);       // const char* nvmlErrorString(nvmlReturn_t): the same shape
  return GPUD_OK;
}


// ---- rows A3 / A4 of SURVEY.md 8(a): what the reference's nvml.Instance and its ecc / remapped-rows components read ------------------
namespace {
// nvmlPciInfo_t (nvml.h): busIdLegacy[16], domain, bus, device, pciDeviceId, pciSubSystemId, busId[32]
struct PciInfo { char bus_id_legacy[16]; unsigned int domain, bus, device, pci_device_id, pci_subsystem_id; char bus_id[32]; };
static_assert(sizeof(PciInfo) == 68, "nvmlPciInfo_t layout");
// nvmlFieldValue_t (nvml.h:2677)
struct FieldValue { unsigned int field_id, scope_id; long long timestamp, latency_usec; int value_type; nvmlReturn_t nvml_return; union { double d; unsigned int ui; unsigned long ul; unsigned long long ull; long long sll; int si; unsigned short us; } value; };
static_assert(sizeof(FieldValue) == 40, "nvmlFieldValue_t layout");

// go-nvlib's device.GetPCIBusID (v0.8.1 pkg/nvlib/device/device.go): the NVML busId lower-cased, with the first four zeros of the
// eight-digit domain dropped ("00000000:3B:00.0" -> "0000:3b:00.0").
void gonvlib_bus_id(const char* nvml_bus_id, char* out, size_t cap) {
  std::string id;
  for (const char* c = nvml_bus_id; *c; ++c) id.push_back((*c >= 'A' && *c <= 'Z') ? (char)(*c - 'A' + 'a') : *c);
  if (id != "0000" && id.compare(0, 4, "0000") == 0) id.erase(0, 4);
  snprintf(out, cap, "%s", id.c_str());
}
}  // namespace

extern "C" int32_t gpud_nvml_bus_id(const char* nvml_bus_id, char* out, int32_t cap) {
  if (!nvml_bus_id || !out || cap < 1) return GPUD_E_INVALID;
  gonvlib_bus_id(nvml_bus_id, out, (size_t)cap);
  return GPUD_OK;
}

// nvml.New's enumeration (pkg/nvidia/nvml/instance.go:197-273): every device's UUID and PCI bus id (the map key and the value
// device.New keeps, device/device.go:46-70), the product name of device 0 and the driver version; plus the CUDA ordinal of each
// device so the rest of this library can be pointed at it.
extern "C" int32_t gpud_nvml_devices(gpud_nvml_device* out, int32_t cap, int32_t* n_out, char* driver_version, int32_t driver_cap) {
  if (!n_out || cap < 0 || (cap && !out)) return GPUD_E_INVALID;
  Nvml* N = nvml();
  if (!N || !N->count || !N->by_index || !N->uuid || !N->pci_info) return GPUD_E_UNSUPPORTED;
  unsigned int n = 0;
  if (N->count(&n) != 0) return GPUD_E_STATE;
  *n_out = (int32_t)n;
  if (driver_version && driver_cap > 0) { driver_version[0] = 0; if (N->driver_version) N->driver_version(driver_version, (unsigned int)driver_cap); }
  for (unsigned int i = 0; i < n && (int32_t)i < cap; ++i) {
    gpud_nvml_device& d = out[i];
    memset(&d, 0, sizeof d);
    d.index = (int32_t)i;
    d.cuda_device = -1;
    nvmlDevice_t h;
    nvmlReturn_t rc = N->by_index(i, &h);                    // "error getting device handle for index": the errored-instance case (:190-203)
    if (rc != 0) { d.nvml_rc = rc; continue; }
    if ((rc = N->uuid(h, d.uuid, sizeof d.uuid)) != 0) { d.nvml_rc = rc; continue; }
    PciInfo pi;
    memset(&pi, 0, sizeof pi);
    if ((rc = N->pci_info(h, &pi)) != 0) { d.nvml_rc = rc; continue; }
    gonvlib_bus_id(pi.bus_id, d.bus_id, sizeof d.bus_id);
    if (N->name) N->name(h, d.name, sizeof d.name);
    int cd = -1;
    if (cudaDeviceGetByPCIBusId(&cd, pi.bus_id) == cudaSuccess) d.cuda_device = cd; else cudaGetLastError();
  }
  return (int32_t)n > cap ? GPUD_E_CAPACITY : GPUD_OK;
}

// "uuid=bus_id;uuid=bus_id;..." of the enumerated devices: the `devices` argument of gpud_xid_state_from_store
extern "C" int32_t gpud_nvml_devices_arg(char* out, int32_t cap) {
  if (!out || cap < 1) return GPUD_E_INVALID;
  gpud_nvml_device d[GPUD_MAX_GPUS];
  int32_t n = 0;
  const int32_t rc = gpud_nvml_devices(d, GPUD_MAX_GPUS, &n, nullptr, 0);
  if (rc != GPUD_OK && rc != GPUD_E_CAPACITY) return rc;
  std::string s;
  for (int32_t i = 0; i < n && i < GPUD_MAX_GPUS; ++i) {
    if (d[i].nvml_rc != 0) continue;
    if (!s.empty()) s += ";";
    s += d[i].uuid; s += "="; s += d[i].bus_id;
  }
  if ((int32_t)s.size() + 1 > cap) return GPUD_E_CAPACITY;
  memcpy(out, s.c_str(), s.size() + 1);
  return (int32_t)s.size();
}

// GetRemappedRows (remapped-rows/remapped_rows.go:52-86)
extern "C" int32_t gpud_poller_remapped_rows(gpud_poller* p, gpud_remapped_rows* out) {
  if (!p || !out) return GPUD_E_INVALID;
  Nvml* N = nvml();
  if (!N) return GPUD_E_UNSUPPORTED;
  memset(out, 0, sizeof *out);
  out->supported = 1;
  if (!N->remapped_rows) { out->supported = 0; return GPUD_OK; }
  unsigned int corr = 0, unc = 0, pending = 0, failed = 0;
  const nvmlReturn_t rc = N->remapped_rows(p->h, &corr, &unc, &pending, &failed);
  if (is_not_supported(N, rc)) { out->supported = 0; return GPUD_OK; }
  if (is_gpu_lost(N, rc)) return gpud_fail(p->ctx, GPUD_E_STATE, "GPU lost");
  if (is_reset_required(N, rc)) return gpud_fail(p->ctx, GPUD_E_STATE, "GPU requires reset");
  if (rc != 0) return gpud_fail(p->ctx, GPUD_E_STATE, "failed to get device remapped rows: %s", N->err ? N->err(rc) : "error");
  out->remapped_due_to_correctable_errors = (int32_t)corr;
  out->remapped_due_to_uncorrectable_errors = (int32_t)unc;
  out->remapping_pending = pending ? 1 : 0;
  out->remapping_failed = failed ? 1 : 0;
  return GPUD_OK;
}

// The remapped-rows Check over the box's readings (remapped-rows/component.go:197-300): per GPU, in the order given, "<bus id>
// qualifies for RMA (row remapping failed, remapped due to N uncorrectable error(s))" when the failure flag is set and "<bus id>
// needs reset (detected pending row remapping)" when a remapping is pending; Unhealthy with the issues joined by ", ", else
// Healthy "N devices support remapped rows and found no issue".  *action: HardwareInspection once any GPU failed (RMA takes
// precedence), else RebootSystem when one is pending, else 0.
extern "C" int32_t gpud_remapped_rows_check(const gpud_remapped_rows* rows, const char* const* bus_ids, int32_t n, int32_t* health, int32_t* action,
                                            char* reason, int32_t cap) {
  if (n < 0 || (n && (!rows || !bus_ids)) || !health || !reason || cap < 1) return GPUD_E_INVALID;
  std::string issues;
  int act = 0;
  for (int32_t i = 0; i < n; ++i) {
    const gpud_remapped_rows& r = rows[i];
    if (r.remapping_pending && act != GPUD_ACT_HARDWARE_INSPECTION) act = GPUD_ACT_REBOOT_SYSTEM;
    if (r.remapping_failed) act = GPUD_ACT_HARDWARE_INSPECTION;
    char buf[256];
    if (r.remapping_failed) {
      snprintf(buf, sizeof buf, "%s qualifies for RMA (row remapping failed, remapped due to %d uncorrectable error(s))", bus_ids[i] ? bus_ids[i] : "", r.remapped_due_to_uncorrectable_errors);
      if (!issues.empty()) issues += ", ";
      issues += buf;
    }
    if (r.remapping_pending) {
      snprintf(buf, sizeof buf, "%s needs reset (detected pending row remapping)", bus_ids[i] ? bus_ids[i] : "");
      if (!issues.empty()) issues += ", ";
      issues += buf;
    }
  }
  *health = issues.empty() ? 0 : 2;
  if (action) *action = act;
  if (issues.empty()) { char buf[96]; snprintf(buf, sizeof buf, "%d devices support remapped rows and found no issue", n); issues = buf; }
  if ((int32_t)issues.size() + 1 > cap) return -1;
  memcpy(reason, issues.c_str(), issues.size() + 1);
  return (int32_t)issues.size();
}

// GetECCModeEnabled + GetECCErrors (ecc/ecc_mode.go, ecc/ecc_errors.go:136-880): the four totals, then - only with ECC mode on - the
// per-location counters in the reference's order; the first "not supported" ends the read with supported = 0 and what was read so
// far, GPU lost / requires reset fail it.
extern "C" int32_t gpud_poller_ecc_errors(gpud_poller* p, gpud_ecc_errors* out) {
  if (!p || !out) return GPUD_E_INVALID;
  Nvml* N = nvml();
  if (!N || !N->ecc_total) return GPUD_E_UNSUPPORTED;
  memset(out, 0, sizeof *out);
  out->supported = 1;
  int cur = 0, pend = 0;
  if (N->ecc_mode && N->ecc_mode(p->h, &cur, &pend) == 0) { out->ecc_mode_current = cur == 1; out->ecc_mode_pending = pend == 1; }
  auto done = [&](nvmlReturn_t rc, int32_t* fail) -> bool {   // true = stop reading
    *fail = GPUD_OK;
    if (rc == 0) return false;
    if (is_not_supported(N, rc)) { out->supported = 0; return true; }
    if (is_gpu_lost(N, rc)) { *fail = gpud_fail(p->ctx, GPUD_E_STATE, "GPU lost"); return true; }
    if (is_reset_required(N, rc)) { *fail = gpud_fail(p->ctx, GPUD_E_STATE, "GPU requires reset"); return true; }
    *fail = gpud_fail(p->ctx, GPUD_E_STATE, "failed to get ecc errors: %s", N->err ? N->err(rc) : "error");
    return true;
  };
  int32_t fail;
  // totals: (corrected, aggregate), (uncorrected, aggregate), (corrected, volatile), (uncorrected, volatile)  (:148-240)
  if (done(N->ecc_total(p->h, 0, 1, (unsigned long long*)&out->aggregate[GPUD_ECC_TOTAL].corrected), &fail)) return fail;
  if (done(N->ecc_total(p->h, 1, 1, (unsigned long long*)&out->aggregate[GPUD_ECC_TOTAL].uncorrected), &fail)) return fail;
  if (done(N->ecc_total(p->h, 0, 0, (unsigned long long*)&out->volatile_[GPUD_ECC_TOTAL].corrected), &fail)) return fail;
  if (done(N->ecc_total(p->h, 1, 0, (unsigned long long*)&out->volatile_[GPUD_ECC_TOTAL].uncorrected), &fail)) return fail;
  if (!out->ecc_mode_current || !N->ecc_location) return GPUD_OK;                       // :241-245
  // nvml.MEMORY_LOCATION_*: L1 0, L2 1, DRAM / DEVICE_MEMORY 2, REGISTER_FILE 3, TEXTURE_MEMORY 4, TEXTURE_SHM 5, SRAM 7
  static const struct { int slot, loc; } kAgg[] = {{GPUD_ECC_L1, 0}, {GPUD_ECC_L2, 1}, {GPUD_ECC_DRAM, 2}, {GPUD_ECC_SRAM, 7}, {GPUD_ECC_DEVICE_MEMORY, 2},
                                                   {GPUD_ECC_TEXTURE_MEMORY, 4}, {GPUD_ECC_SHARED_MEMORY, 5}};
  for (const auto& a : kAgg) {
    if (done(N->ecc_location(p->h, 0, 1, a.loc, (unsigned long long*)&out->aggregate[a.slot].corrected), &fail)) return fail;
    if (done(N->ecc_location(p->h, 1, 1, a.loc, (unsigned long long*)&out->aggregate[a.slot].uncorrected), &fail)) return fail;
  }
  for (const auto& a : kAgg) {
    if (done(N->ecc_location(p->h, 0, 0, a.loc, (unsigned long long*)&out->volatile_[a.slot].corrected), &fail)) return fail;
    if (done(N->ecc_location(p->h, 1, 0, a.loc, (unsigned long long*)&out->volatile_[a.slot].uncorrected), &fail)) return fail;
  }
  if (done(N->ecc_location(p->h, 0, 0, 3, (unsigned long long*)&out->volatile_[GPUD_ECC_REGISTER_FILE].corrected), &fail)) return fail;
  if (done(N->ecc_location(p->h, 1, 0, 3, (unsigned long long*)&out->volatile_[GPUD_ECC_REGISTER_FILE].uncorrected), &fail)) return fail;
  return GPUD_OK;
}

// One driver round trip for a whole row of counters: nvmlDeviceGetFieldValues over GPUD_FIELD_ROW (SURVEY.md 8f.3).  values[i] is
// the field widened to u64 (doubles truncated), nvml_rc[i] the field's own return code.
static const unsigned int kFieldRow[GPUD_FIELD_ROW_N] = {186 /* POWER_INSTANT mW */, 185 /* POWER_AVERAGE mW */, 82 /* MEMORY_TEMP C */, 83 /* TOTAL_ENERGY mJ */,
                                                         3, 4, 5, 6 /* ECC SBE/DBE volatile, aggregate totals */, 38, 45, 52, 59 /* NVLink CRC flit / CRC data / replay / recovery totals */,
                                                         142, 143, 144, 145 /* remapped rows: correctable, uncorrectable, pending, failure */, 94 /* PCIe replay counter */};
static int32_t field_row(Nvml* N, nvmlDevice_t h, uint64_t* values, int32_t* rcs) {
  FieldValue fv[GPUD_FIELD_ROW_N];
  memset(fv, 0, sizeof fv);
  for (int i = 0; i < GPUD_FIELD_ROW_N; ++i) fv[i].field_id = kFieldRow[i];
  const nvmlReturn_t rc = N->field_values(h, GPUD_FIELD_ROW_N, fv);
  if (rc != 0) return (int32_t)rc;
  for (int i = 0; i < GPUD_FIELD_ROW_N; ++i) {
    if (rcs) rcs[i] = (int32_t)fv[i].nvml_return;
    uint64_t v = 0;
    if (fv[i].nvml_return == 0) {
      switch (fv[i].value_type) {   // nvmlValueType_t: 0 double, 1 uint, 2 ulong, 3 ulonglong, 4 slonglong, 5 sint, 6 ushort
        case 0: v = fv[i].value.d > 0 ? (uint64_t)fv[i].value.d : 0; break;
        case 1: v = fv[i].value.ui; break;
        case 2: v = fv[i].value.ul; break;
        case 3: v = fv[i].value.ull; break;
        case 4: v = (uint64_t)fv[i].value.sll; break;
        case 5: v = (uint64_t)(int64_t)fv[i].value.si; break;
        case 6: v = fv[i].value.us; break;
      }
    }
    values[i] = v;
  }
  return 0;
}

extern "C" int32_t gpud_poller_field_row(gpud_poller* p, uint64_t* values, int32_t* nvml_rc) {
  if (!p || !values) return GPUD_E_INVALID;
  Nvml* N = nvml();
  if (!N || !N->field_values) return GPUD_E_UNSUPPORTED;
  const int32_t rc = field_row(N, p->h, values, nvml_rc);
  return rc == 0 ? GPUD_OK : gpud_fail(p->ctx, GPUD_E_STATE, "nvmlDeviceGetFieldValues: %s", N->err ? N->err(rc) : "error");
}

// n_polls rows of GPUD_FIELD_ROW, one driver call each, appended to `ring` (GPUD_FIELD_ROW_N fields) as raw uint64 rows through
// pinned memory; a field whose read fails holds its last good value, like gpud_poller_poll.
extern "C" int32_t gpud_poller_poll_fields(gpud_poller* p, gpud_ring* ring, int64_t n_polls, int64_t interval_us, double* seconds) {
  if (!p || !ring || n_polls < 0 || interval_us < 0) return GPUD_E_INVALID;
  Nvml* N = nvml();
  if (!N || !N->field_values) return GPUD_E_UNSUPPORTED;
  if (gpud_ring_n_fields(ring) != GPUD_FIELD_ROW_N) return gpud_fail(p->ctx, GPUD_E_INVALID, "the field-row source needs a ring of %d fields (this one has %d)", GPUD_FIELD_ROW_N, gpud_ring_n_fields(ring));
  if (!p->field_rows) {
    if (cudaMallocHost(&p->field_rows, (size_t)p->cap_rows * GPUD_FIELD_ROW_N * sizeof(uint64_t)) != cudaSuccess) return gpud_fail(p->ctx, GPUD_E_CUDA, "pinned field rows");
  }
  timespec t0, t1;
  clock_gettime(CLOCK_MONOTONIC, &t0);
  int64_t done = 0;
  while (done < n_polls) {
    const int64_t batch = std::min<int64_t>(p->cap_rows, n_polls - done);
    for (int64_t i = 0; i < batch; ++i) {
      uint64_t v[GPUD_FIELD_ROW_N];
      int32_t rcs[GPUD_FIELD_ROW_N];
      const int32_t rc = field_row(N, p->h, v, rcs);
      p->row_ms[i] = row_time_ms(p);
      uint64_t* row = p->field_rows + i * GPUD_FIELD_ROW_N;
      for (int c = 0; c < GPUD_FIELD_ROW_N; ++c) {
        if (rc == 0 && rcs[c] == 0) p->field_held[c] = v[c];
        row[c] = p->field_held[c];
      }
      if (interval_us) { timespec ts{(time_t)(interval_us / 1000000), (long)(interval_us % 1000000) * 1000L}; nanosleep(&ts, nullptr); }
    }
    const int32_t rc = gpud_ring_push_timed(ring, p->field_rows, batch, GPUD_DT_U64, p->row_ms.data());
    if (rc) return rc;
    done += batch;
  }
  clock_gettime(CLOCK_MONOTONIC, &t1);
  if (seconds) *seconds = (double)(t1.tv_sec - t0.tv_sec) + 1e-9 * (double)(t1.tv_nsec - t0.tv_nsec);
  return GPUD_OK;
}

// ---- GPM (components/accelerator/nvidia/gpm) ------------------------------------------------------------------------------------
// nvml.h's GPM records (version 1 of both): the metric array is sized like go-nvml's binding ([210]; NVML reads numMetrics of them).
namespace {
struct NvmlGpmSupport { unsigned int version, is_supported; };
struct NvmlGpmMetric { unsigned int metric_id; nvmlReturn_t nvml_return; double value; struct { char* short_name; char* long_name; char* unit; } info; };
struct NvmlGpmMetricsGet { unsigned int version, num_metrics; void* sample1; void* sample2; NvmlGpmMetric metrics[210]; };
// the component's default ids (gpm/component.go:56-64): SM_OCCUPANCY, INTEGER_UTIL, ANY / DFMA / HMMA / IMMA_TENSOR_UTIL, FP64 / FP32 / FP16_UTIL
const unsigned int kGpmIds[GPUD_GPM_N] = {3, 4, 5, 6, 7, 9, 11, 12, 13};
bool is_version_mismatch(Nvml* N, nvmlReturn_t rc) {          // nvmlerrors.IsVersionMismatchError: the return code or its text
  if (rc == 25 /* NVML_ERROR_ARGUMENT_VERSION_MISMATCH */) return true;
  const char* e = N->err ? N->err(rc) : nullptr;
  if (!e) return false;
  std::string t(e);
  for (auto& c : t) c = (char)tolower((unsigned char)c);
  return t.find("version mismatch") != std::string::npos;
}
struct GpmSample {
  Nvml* N; void* h = nullptr;
  explicit GpmSample(Nvml* n) : N(n) {}
  ~GpmSample() { if (h && N->gpm_free) N->gpm_free(h); }
};
}  // namespace

// SupportedByDevice (gpm/gpm.go:17-45): not-supported and version-mismatch answers mean "no", lost / reset-required GPUs are errors
extern "C" int32_t gpud_poller_gpm_supported(gpud_poller* p, int32_t* supported) {
  if (!p || !supported) return GPUD_E_INVALID;
  Nvml* N = nvml();
  if (!N) return GPUD_E_UNSUPPORTED;
  *supported = 0;
  if (!N->gpm_support || !N->gpm_alloc || !N->gpm_free || !N->gpm_sample || !N->gpm_metrics) return GPUD_OK;
  NvmlGpmSupport q{1u, 0u};
  const nvmlReturn_t rc = N->gpm_support(p->h, &q);
  if (is_not_supported(N, rc) || is_version_mismatch(N, rc)) return GPUD_OK;
  if (is_gpu_lost(N, rc)) return gpud_fail(p->ctx, GPUD_E_STATE, "GPU lost");
  if (is_reset_required(N, rc)) return gpud_fail(p->ctx, GPUD_E_STATE, "GPU requires reset");
  if (rc != 0) return gpud_fail(p->ctx, GPUD_E_STATE, "could not query GPM support: %s", N->err ? N->err(rc) : "error");
  *supported = q.is_supported != 0;
  return GPUD_OK;
}

static int32_t gpm_take(gpud_poller* p, Nvml* N, void* sample) {
  const nvmlReturn_t rc = N->gpm_sample(p->h, sample);
  return rc == 0 ? GPUD_OK : gpud_fail(p->ctx, GPUD_E_STATE, "could not get sample: %s", N->err ? N->err(rc) : "error");
}
static int32_t gpm_between(gpud_poller* p, Nvml* N, void* s1, void* s2, gpud_gpm_metrics* out) {
  static thread_local NvmlGpmMetricsGet g;                       // 8.4 KB
  memset(&g, 0, sizeof g);
  g.version = 1;
  g.num_metrics = GPUD_GPM_N;
  g.sample1 = s1;
  g.sample2 = s2;
  for (int i = 0; i < GPUD_GPM_N; ++i) g.metrics[i].metric_id = kGpmIds[i];
  const nvmlReturn_t rc = N->gpm_metrics(&g);
  if (rc != 0) return gpud_fail(p->ctx, GPUD_E_STATE, "failed to get gpm metric: %s", N->err ? N->err(rc) : "error");
  for (int i = 0; i < GPUD_GPM_N; ++i) { out->value[i] = g.metrics[i].value; out->nvml_rc[i] = (int32_t)g.metrics[i].nvml_return; }
  return GPUD_OK;
}

// GetGPMMetrics (gpm/gpm.go:65-149): two samples `sample_ms` apart, one nvmlGpmMetricsGet over the nine ids
extern "C" int32_t gpud_poller_gpm_metrics(gpud_poller* p, int64_t sample_ms, gpud_gpm_metrics* out) {
  if (!p || !out || sample_ms < 0) return GPUD_E_INVALID;
  Nvml* N = nvml();
  if (!N) return GPUD_E_UNSUPPORTED;
  memset(out, 0, sizeof *out);
  if (!N->gpm_support || !N->gpm_alloc || !N->gpm_free || !N->gpm_sample || !N->gpm_metrics) return GPUD_OK;      // supported = 0
  GpmSample s1(N), s2(N);
  nvmlReturn_t rc = N->gpm_alloc(&s1.h);
  if (is_not_supported(N, rc) || is_version_mismatch(N, rc)) return GPUD_OK;
  if (is_gpu_lost(N, rc)) return gpud_fail(p->ctx, GPUD_E_STATE, "GPU lost");
  if (is_reset_required(N, rc)) return gpud_fail(p->ctx, GPUD_E_STATE, "GPU requires reset");
  if (rc != 0) return gpud_fail(p->ctx, GPUD_E_STATE, "could not allocate sample: %s", N->err ? N->err(rc) : "error");
  rc = N->gpm_alloc(&s2.h);
  if (rc != 0) return gpud_fail(p->ctx, GPUD_E_STATE, "could not allocate sample: %s", N->err ? N->err(rc) : "error");
  int32_t r = gpm_take(p, N, s1.h);
  if (r) return r;
  timespec t0, t1;
  clock_gettime(CLOCK_MONOTONIC, &t0);
  if (sample_ms) { timespec ts{(time_t)(sample_ms / 1000), (long)(sample_ms % 1000) * 1000000L}; nanosleep(&ts, nullptr); }
  r = gpm_take(p, N, s2.h);
  if (r) return r;
  clock_gettime(CLOCK_MONOTONIC, &t1);
  r = gpm_between(p, N, s1.h, s2.h, out);
  if (r) return r;
  out->supported = 1;
  out->sample_seconds = (double)(t1.tv_sec - t0.tv_sec) + 1e-9 * (double)(t1.tv_nsec - t0.tv_nsec);
  return GPUD_OK;
}

// The same getter as a field source of the ring (SURVEY.md A3, "GPM f64"): n_polls rows of the nine metrics, one row per sample
// interval - consecutive rows share a sample (n_polls + 1 nvmlGpmSampleGet calls), so the intervals tile the time line without gaps.
extern "C" int32_t gpud_poller_poll_gpm(gpud_poller* p, gpud_ring* ring, int64_t n_polls, int64_t sample_ms, double* seconds) {
  if (!p || !ring || n_polls < 0 || sample_ms < 0) return GPUD_E_INVALID;
  Nvml* N = nvml();
  if (!N || !N->gpm_support || !N->gpm_alloc || !N->gpm_free || !N->gpm_sample || !N->gpm_metrics) return GPUD_E_UNSUPPORTED;
  if (gpud_ring_n_fields(ring) != GPUD_GPM_N) return gpud_fail(p->ctx, GPUD_E_INVALID, "the GPM source needs a ring of %d fields (this one has %d)", GPUD_GPM_N, gpud_ring_n_fields(ring));
  int32_t sup = 0;
  int32_t r = gpud_poller_gpm_supported(p, &sup);
  if (r) return r;
  if (!sup) return gpud_fail(p->ctx, GPUD_E_UNSUPPORTED, "GPM not supported");
  GpmSample a(N), b(N);
  if (N->gpm_alloc(&a.h) != 0 || N->gpm_alloc(&b.h) != 0) return gpud_fail(p->ctx, GPUD_E_STATE, "could not allocate sample");
  timespec t0, t1;
  clock_gettime(CLOCK_MONOTONIC, &t0);
  r = gpm_take(p, N, a.h);
  if (r) return r;
  void* prev = a.h;
  void* next = b.h;
  for (int64_t i = 0; i < n_polls; ++i) {
    if (sample_ms) { timespec ts{(time_t)(sample_ms / 1000), (long)(sample_ms % 1000) * 1000000L}; nanosleep(&ts, nullptr); }
    r = gpm_take(p, N, next);
    if (r) return r;
    gpud_gpm_metrics m;
    r = gpm_between(p, N, prev, next, &m);
    if (r) return r;
    const int64_t ms = row_time_ms(p);
    double row[GPUD_GPM_N];
    for (int c = 0; c < GPUD_GPM_N; ++c) {                                  // a metric NVML could not compute holds its last good value
      if (m.nvml_rc[c] == 0) p->gpm_held[c] = m.value[c];
      row[c] = p->gpm_held[c];
    }
    r = gpud_ring_push_timed(ring, row, 1, GPUD_DT_F64, &ms);
    if (r) return r;
    std::swap(prev, next);
  }
  clock_gettime(CLOCK_MONOTONIC, &t1);
  if (seconds) *seconds = (double)(t1.tv_sec - t0.tv_sec) + 1e-9 * (double)(t1.tv_nsec - t0.tv_nsec);
  return GPUD_OK;
}

// The gpm component's Check over the box's readings (gpm/component.go:196-290): one GPU without GPM -> Healthy "GPM not supported",
// else Healthy "all N GPU(s) were checked, no GPM issue found"; getter errors are the getters' own return codes.
extern "C" int32_t gpud_gpm_check(const gpud_gpm_metrics* m, int32_t n, int32_t* health, char* reason, int32_t cap) {
  if (n < 0 || (n && !m) || !health || !reason || cap < 1) return GPUD_E_INVALID;
  *health = 0;
  char buf[96];
  bool all = true;
  for (int32_t i = 0; i < n; ++i) all = all && m[i].supported != 0;
  if (!all) snprintf(buf, sizeof buf, "GPM not supported");
  else snprintf(buf, sizeof buf, "all %d GPU(s) were checked, no GPM issue found", n);
  const int len = (int)strlen(buf);
  if (len + 1 > cap) return -1;
  memcpy(reason, buf, (size_t)len + 1);
  return len;
}
