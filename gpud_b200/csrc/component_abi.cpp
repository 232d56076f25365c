// component_abi.cpp — the C ABI over the host mirror of components.Component (components/types.go:20-66) for the three paths this
// library replaces: the xid component (scan + event bucket + evolveHealthyState), the temperature component (poll -> ring ->
// windowed aggregates, and the reference's threshold rules over the current reading) and the nvlink component (per-GPU records ->
// peer-store gather -> box verdict).  Conventions kept from the reference (SURVEY.md 8b):
//   * Start() does not block; it spawns the ticker that calls Check() every interval (temperature/component.go:81-104);
//   * Check() takes no context, embeds errors in the result and never throws (types.go:48-53);
//   * LastHealthStates() returns the cached state, or a single Healthy "no data yet" state before the first check (types.go:55-58,
//     temperature/component.go:368-379); results are guarded by a mutex because readers come from other threads;
//   * Events(since) is descending by time, strictly after `since`; Close() stops the ticker.
#include <time.h>

#include <atomic>
#include <condition_variable>
#include <memory>
#include <thread>

#include "host_component.h"
#include "internal.h"
#include "ring_drain.h"

namespace {

using gpud::Health;
using gpud::HealthState;

int64_t now_unix() { return (int64_t)time(nullptr); }

struct DevSlot { int dev = 0; gpud_ring* ring = nullptr; gpud_poller* poller = nullptr; std::string uuid, bus_id; };

// pollers (and the small rings they feed) for every device of the ctx; UUIDs from the NVML enumeration
int32_t open_slots(gpud_ctx* ctx, int n_fields_ring, int64_t cap, int window, std::vector<DevSlot>* out) {
  gpud_nvml_device devs[GPUD_MAX_GPUS];
  int32_t n_nvml = 0;
  gpud_nvml_devices(devs, GPUD_MAX_GPUS, &n_nvml, nullptr, 0);
  for (int dev : ctx->devs) {
    DevSlot s;
    s.dev = dev;
    gpud_ring_cfg cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.n_fields = n_fields_ring; cfg.capacity = cap; cfg.window = window;
    int32_t rc = gpud_ring_create(ctx, dev, &cfg, &s.ring);
    if (rc == GPUD_OK) rc = gpud_poller_create(ctx, dev, s.ring, &s.poller);
    if (rc != GPUD_OK) { if (s.ring) gpud_ring_destroy(s.ring); for (DevSlot& o : *out) { gpud_poller_destroy(o.poller); gpud_ring_destroy(o.ring); } out->clear(); return rc; }
    for (int32_t i = 0; i < n_nvml && i < GPUD_MAX_GPUS; ++i)
      if (devs[i].cuda_device == dev && devs[i].nvml_rc == 0) { s.uuid = devs[i].uuid; s.bus_id = devs[i].bus_id; }
    if (s.uuid.empty()) s.uuid = "GPU-" + std::to_string(dev);
    out->push_back(s);
  }
  return GPUD_OK;
}
void close_slots(std::vector<DevSlot>* slots) {
  for (DevSlot& s : *slots) { if (s.poller) gpud_poller_destroy(s.poller); if (s.ring) gpud_ring_destroy(s.ring); }
  slots->clear();
}

// The poll columns as the reference's gauges name them: component_name = the component that owns the gauge, metric name = SubSystem +
// gauge name (components/accelerator/nvidia/{temperature,power,clock-speed,utilization,memory}/metrics.go).  The reference has no SM
// clock gauge, and its memory gauge counts bytes where this column counts MiB: those two names say what the column holds.
const char* const kPollComponent[GPUD_POLL_N_FIELDS] = {
    "accelerator-nvidia-temperature", "accelerator-nvidia-power", "accelerator-nvidia-clock-speed", "accelerator-nvidia-clock-speed",
    "accelerator-nvidia-clock-speed", "accelerator-nvidia-utilization", "accelerator-nvidia-utilization", "accelerator-nvidia-memory"};
const char* const kPollMetric[GPUD_POLL_N_FIELDS] = {
    "accelerator_nvidia_temperature_current_celsius", "accelerator_nvidia_power_current_usage_milli_watts",
    "accelerator_nvidia_clock_speed_graphics_mhz", "accelerator_nvidia_clock_speed_sm_mhz", "accelerator_nvidia_clock_speed_memory_mhz",
    "accelerator_nvidia_utilization_gpu_util_percent", "accelerator_nvidia_utilization_memory_util_percent", "accelerator_nvidia_memory_used_mib"};

// temperature: one poll row per check into the ring (the windowed aggregates stay available through gpud_component_ring), the
// reference's rules over the current reading (temperature/component.go:190-287); with a metrics store attached, every completed window
// of the ring goes into the store right after the poll (the Syncer's job in the reference, pkg/metrics/syncer/syncer.go:36-82)
class TemperatureComponent : public gpud::Component {
 public:
  static constexpr const char* kName = "accelerator-nvidia-temperature";            // temperature/component.go:27
  TemperatureComponent(gpud_ctx* ctx, int32_t margin_threshold_c) : ctx_(ctx), margin_(margin_threshold_c) {}
  ~TemperatureComponent() override { close_slots(&slots_); }
  int32_t Open() { return open_slots(ctx_, GPUD_POLL_N_FIELDS, 1 << 16, 1000, &slots_); }
  std::string Name() const override { return kName; }
  std::vector<std::string> Tags() const override { return {"accelerator", "gpu", "nvidia", kName}; }
  bool IsSupported() const override { return !slots_.empty(); }
  int32_t Start() override { return 0; }
  gpud::CheckResult Check() override {
    gpud::CheckResult cr;
    cr.component = kName;
    HealthState s;
    s.time_unix = now_unix(); s.name = kName; s.component = kName;
    std::vector<gpud_temperature> ts(slots_.size());
    std::vector<const char*> uuids;
    for (size_t i = 0; i < slots_.size(); ++i) {
      int32_t rc = gpud_poller_poll(slots_[i].poller, 1, 0);                          // the sample sink: one row into the ring
      if (rc == GPUD_OK && store_) sync_metrics(slots_[i]);
      if (rc == GPUD_OK) rc = gpud_poller_temperature(slots_[i].poller, &ts[i]);
      if (rc != GPUD_OK) {                                                            // "error getting temperature" (:196-204)
        char msg[512] = {0};
        gpud_last_error(ctx_, msg, sizeof msg);
        s.health = Health::Unhealthy; s.reason = "error getting temperature"; s.error = msg;
        cr.health = s.health; cr.summary = s.reason; cr.states.push_back(s);
        store(s);
        return cr;
      }
      uuids.push_back(slots_[i].uuid.c_str());
    }
    int32_t health = 0;
    char reason[2048];
    if (gpud_temperature_reason(ts.data(), uuids.data(), (int32_t)ts.size(), margin_, &health, reason, sizeof reason) < 0) snprintf(reason, sizeof reason, "reason too long");
    s.health = health ? Health::Degraded : Health::Healthy;
    s.reason = reason;
    cr.health = s.health; cr.summary = s.reason; cr.states.push_back(s);
    store(s);
    return cr;
  }
  std::vector<HealthState> LastHealthStates() override {
    std::lock_guard<std::mutex> g(mu_);
    if (!checked_) { HealthState s; s.time_unix = now_unix(); s.name = kName; s.component = kName; s.reason = "no data yet"; return {s}; }
    return {last_};
  }
  std::vector<gpud::Event> Events(int64_t) override { return {}; }                    // temperature/component.go:118-120: no events
  int32_t Close() override { return 0; }
  gpud_ring* ring(int slot) { return slot >= 0 && slot < (int)slots_.size() ? slots_[slot].ring : nullptr; }
  // caller holds the component's check lock
  int32_t SetMetricsStore(gpud_store* st, const char* table) {
    if (st) {
      const int32_t rc = gpud_store_metrics_table(st, table);                         // CreateTable (metrics/store/sqlite.go:87-106)
      if (rc != GPUD_OK) return rc;
    }
    store_ = st;
    table_ = table ? table : "";
    return GPUD_OK;
  }
 private:
  // A failed drain leaves the check result alone (the reference Syncer only logs, syncer.go:52-54) and the windows where they are
  void sync_metrics(const DevSlot& s) {
    std::string labels = "{\"uuid\":";
    gpud::jstr(labels, s.uuid);
    labels += "}";
    gpud_drain_info info;
    const int32_t rc = gpud_ring_drain_to_store(s.ring, store_, table_.c_str(), kPollComponent, kPollMetric, labels.c_str(), 0, kMaxDrain, &info,
                                                nullptr, nullptr);
    if (rc != GPUD_OK) {
      char msg[512] = {0};
      gpud_store_last_error(store_, msg, sizeof msg);
      gpud_fail(ctx_, rc, "metrics drain of %s: %s", s.uuid.c_str(), msg);
    }
  }
  static constexpr int64_t kMaxDrain = 128;                                            // > the 66 windows a 64 Ki-sample ring holds
  gpud_store* store_ = nullptr;
  std::string table_;
  void store(const HealthState& s) { std::lock_guard<std::mutex> g(mu_); last_ = s; checked_ = true; }
  gpud_ctx* ctx_;
  int32_t margin_;
  std::vector<DevSlot> slots_;
  std::mutex mu_;
  HealthState last_;
  bool checked_ = false;
};

// nvlink: every GPU's record from NVML, the fused publish + gather over NVLink peer stores, the replicated verdict
// (nvlink/component.go:164-311, evaluate_threshold.go:77-188)
class NvlinkComponent : public gpud::Component {
 public:
  static constexpr const char* kName = "accelerator-nvidia-nvlink";                  // nvlink/component.go:27
  NvlinkComponent(gpud_ctx* ctx, int32_t at_least) : ctx_(ctx), at_least_(at_least) {}
  ~NvlinkComponent() override { close_slots(&slots_); }
  int32_t Open() { return open_slots(ctx_, GPUD_POLL_N_FIELDS, 1024, 16, &slots_); }
  std::string Name() const override { return kName; }
  std::vector<std::string> Tags() const override { return {"accelerator", "gpu", "nvidia", kName}; }
  bool IsSupported() const override { return !slots_.empty(); }
  int32_t Start() override { return 0; }
  gpud::CheckResult Check() override {
    gpud::CheckResult cr;
    cr.component = kName;
    HealthState s;
    s.time_unix = now_unix(); s.name = kName; s.component = kName;
    const int n = (int)slots_.size();
    std::vector<gpud_fabric_raw> raws(n);
    std::vector<std::string> bus(n);
    std::vector<const char*> peers(n), uuids(n);
    for (int i = 0; i < n; ++i) {
      char b[32] = {0};
      cudaDeviceGetPCIBusId(b, sizeof b, slots_[i].dev);
      bus[i] = b; peers[i] = bus[i].c_str(); uuids[i] = slots_[i].uuid.c_str();
    }
    int32_t rc = GPUD_OK;
    for (int i = 0; i < n && rc == GPUD_OK; ++i) rc = gpud_poller_fabric_raw(slots_[i].poller, (uint32_t)i, peers.data(), n, &raws[i]);
    std::vector<gpud_fabric_verdict> verdicts(n);
    if (rc == GPUD_OK) rc = gpud_fabric_gather_p2p(ctx_, raws.data(), at_least_, nullptr, verdicts.data());
    if (rc != GPUD_OK) {
      char msg[512] = {0};
      gpud_last_error(ctx_, msg, sizeof msg);
      s.health = Health::Unhealthy; s.reason = "error getting nvlink"; s.error = msg;
    } else {
      char reason[4096];
      if (gpud_fabric_reason(&verdicts[0], uuids.data(), n, reason, sizeof reason) < 0) snprintf(reason, sizeof reason, "reason too long");
      s.health = verdicts[0].nvlink_health == 2 ? Health::Unhealthy : Health::Healthy;
      s.reason = reason;
      if (gpud_fabric_suggest_reboot(&verdicts[0])) { s.has_actions = true; s.actions.repair_actions = {GPUD_ACT_REBOOT_SYSTEM}; }
    }
    cr.health = s.health; cr.summary = s.reason; cr.states.push_back(s);
    std::lock_guard<std::mutex> g(mu_);
    last_ = s; checked_ = true;
    return cr;
  }
  std::vector<HealthState> LastHealthStates() override {
    std::lock_guard<std::mutex> g(mu_);
    if (!checked_) { HealthState s; s.time_unix = now_unix(); s.name = kName; s.component = kName; s.reason = "no data yet"; return {s}; }
    return {last_};
  }
  std::vector<gpud::Event> Events(int64_t) override { return {}; }                    // nvlink/component.go: no events
  int32_t Close() override { return 0; }
 private:
  gpud_ctx* ctx_;
  int32_t at_least_;
  std::vector<DevSlot> slots_;
  std::mutex mu_;
  HealthState last_;
  bool checked_ = false;
};

std::string event_json(const gpud::Event& e, const std::string& component) {       // apiv1.Event (api/v1/types.go:108-123)
  std::string o = "{";
  if (!component.empty()) { o += "\"component\":"; gpud::jstr(o, component); o += ","; }
  time_t t = (time_t)e.time_unix;
  struct tm tmv;
  gmtime_r(&t, &tmv);
  char tb[48];
  strftime(tb, sizeof tb, "\"time\":\"%Y-%m-%dT%H:%M:%SZ\"", &tmv);
  o += tb;
  if (!e.name.empty()) { o += ",\"name\":"; gpud::jstr(o, e.name); }
  if (!e.type.empty()) { o += ",\"type\":"; gpud::jstr(o, e.type); }
  if (!e.message.empty()) { o += ",\"message\":"; gpud::jstr(o, e.message); }
  o += "}";
  return o;
}

}  // namespace

struct gpud_component {
  std::unique_ptr<gpud::Component> impl;
  gpud::XidComponent* xid = nullptr;             // non-null when impl is the xid component
  TemperatureComponent* temp = nullptr;
  std::thread ticker;
  std::mutex mu;
  std::condition_variable cv;
  bool stop = false, started = false;
  std::atomic<int64_t> checks{0};
  std::mutex check_mu;                           // one Check at a time (the ticker and a caller's own Check share the device state)
};

extern "C" int32_t gpud_component_create(gpud_ctx* ctx, const char* name, const gpud_component_cfg* cfg, gpud_component** out) {
  if (!ctx || !name || !out) return GPUD_E_INVALID;
  gpud_component_cfg c;
  memset(&c, 0, sizeof c);
  if (cfg) c = *cfg;
  std::unique_ptr<gpud_component> h(new gpud_component());
  const std::string nm = name;
  if (nm == gpud::XidComponent::kName) {
    h->xid = new gpud::XidComponent(ctx, ctx->devs[0], c.row_remapping_supported != 0, c.reboot_threshold > 0 ? c.reboot_threshold : 2);
    h->impl.reset(h->xid);
  } else if (nm == TemperatureComponent::kName) {
    h->temp = new TemperatureComponent(ctx, c.margin_threshold_c);
    h->impl.reset(h->temp);
    const int32_t rc = h->temp->Open();
    if (rc != GPUD_OK) return rc;
  } else if (nm == NvlinkComponent::kName) {
    NvlinkComponent* n = new NvlinkComponent(ctx, c.nvlink_at_least);
    h->impl.reset(n);
    const int32_t rc = n->Open();
    if (rc != GPUD_OK) return rc;
  } else {
    return gpud_fail(ctx, GPUD_E_INVALID, "unknown component %s", name);
  }
  *out = h.release();
  return GPUD_OK;
}

extern "C" int32_t gpud_component_name(gpud_component* c, char* out, int32_t cap) {
  if (!c || !out || cap < 1) return GPUD_E_INVALID;
  snprintf(out, (size_t)cap, "%s", c->impl->Name().c_str());
  return GPUD_OK;
}

static void run_check(gpud_component* c, gpud::CheckResult* out) {
  std::lock_guard<std::mutex> g(c->check_mu);
  gpud::CheckResult cr = c->impl->Check();
  if (c->xid && !cr.found.empty()) c->xid->IngestHits(cr.found, now_unix());        // the xid watcher's persist step (component.go:468-577)
  c->checks.fetch_add(1);
  if (out) *out = cr;
}

extern "C" int32_t gpud_component_check(gpud_component* c, int32_t* health, char* reason, int32_t cap) {
  if (!c) return GPUD_E_INVALID;
  gpud::CheckResult cr;
  run_check(c, &cr);
  if (health) *health = (int32_t)cr.health;
  if (reason && cap > 0) snprintf(reason, (size_t)cap, "%s", cr.summary.c_str());
  return GPUD_OK;
}

extern "C" int32_t gpud_component_start(gpud_component* c, int64_t interval_ms) {
  if (!c || interval_ms < 1) return GPUD_E_INVALID;
  std::lock_guard<std::mutex> g(c->mu);
  if (c->started) return GPUD_E_STATE;
  c->started = true;
  c->impl->Start();
  c->ticker = std::thread([c, interval_ms] {                                          // check once at once, then every tick
    for (;;) {
      run_check(c, nullptr);
      std::unique_lock<std::mutex> lk(c->mu);
      if (c->cv.wait_for(lk, std::chrono::milliseconds(interval_ms), [c] { return c->stop; })) return;
    }
  });
  return GPUD_OK;
}

extern "C" int32_t gpud_component_close(gpud_component* c) {
  if (!c) return GPUD_E_INVALID;
  {
    std::lock_guard<std::mutex> g(c->mu);
    c->stop = true;
  }
  c->cv.notify_all();
  if (c->ticker.joinable()) c->ticker.join();
  return c->impl->Close();
}

extern "C" void gpud_component_destroy(gpud_component* c) {
  if (!c) return;
  gpud_component_close(c);
  delete c;
}

extern "C" int64_t gpud_component_checks(gpud_component* c) { return c ? c->checks.load() : 0; }

extern "C" int32_t gpud_component_last_health_states(gpud_component* c, char* json, int32_t cap) {
  if (!c || !json || cap < 1) return GPUD_E_INVALID;
  std::string o = "[";
  bool first = true;
  for (const HealthState& s : c->impl->LastHealthStates()) { if (!first) o += ","; first = false; o += s.to_json(); }
  o += "]";
  if ((int32_t)o.size() + 1 > cap) return GPUD_E_CAPACITY;
  memcpy(json, o.c_str(), o.size() + 1);
  return (int32_t)o.size();
}

extern "C" int32_t gpud_component_events(gpud_component* c, int64_t since_unix, char* json, int32_t cap) {
  if (!c || !json || cap < 1) return GPUD_E_INVALID;
  std::string o = "[";
  bool first = true;
  for (const gpud::Event& e : c->impl->Events(since_unix)) { if (!first) o += ","; first = false; o += event_json(e, c->impl->Name()); }
  o += "]";
  if ((int32_t)o.size() + 1 > cap) return GPUD_E_CAPACITY;
  memcpy(json, o.c_str(), o.size() + 1);
  return (int32_t)o.size();
}

// xid only: the kmsg bytes Check() scans (kmsg.ReadAll's result), SetHealthy (xid/set_healthy.go:14-35), a reboot event of the os bucket
extern "C" int32_t gpud_component_xid_set_source(gpud_component* c, const uint8_t* buf, int64_t len, int32_t raw_kmsg, int64_t boot_unix) {
  if (!c || !c->xid || len < 0 || (len && !buf)) return GPUD_E_INVALID;
  std::lock_guard<std::mutex> g(c->check_mu);
  c->xid->SetKmsgSource(std::string(reinterpret_cast<const char*>(buf), (size_t)len), raw_kmsg != 0, boot_unix);
  return GPUD_OK;
}
extern "C" int32_t gpud_component_xid_set_healthy(gpud_component* c, int64_t now) { return (c && c->xid) ? c->xid->SetHealthy(now) : GPUD_E_INVALID; }
extern "C" int32_t gpud_component_xid_add_reboot(gpud_component* c, int64_t unix_s) {
  if (!c || !c->xid) return GPUD_E_INVALID;
  c->xid->AddRebootEvent(unix_s);
  c->xid->Start();
  return GPUD_OK;
}
extern "C" int32_t gpud_component_xid_set_devices(gpud_component* c, const char* devices /* "uuid=bus_id;..." */) {
  if (!c || !c->xid) return GPUD_E_INVALID;
  gpud::DeviceMap m;
  std::string s = devices ? devices : "";
  size_t p = 0;
  while (p < s.size()) {
    size_t e = s.find(';', p);
    if (e == std::string::npos) e = s.size();
    const std::string kv = s.substr(p, e - p);
    const size_t eq = kv.find('=');
    if (eq != std::string::npos) m[kv.substr(0, eq)] = kv.substr(eq + 1);
    p = e + 1;
  }
  c->xid->SetDevices(m);
  return GPUD_OK;
}
// temperature only: the ring the component's polls land in (device slot of the ctx), for gpud_ring_reduce / gpud_ring_read
extern "C" gpud_ring* gpud_component_ring(gpud_component* c, int32_t slot) { return (c && c->temp) ? c->temp->ring(slot) : nullptr; }
extern "C" int32_t gpud_component_set_metrics_store(gpud_component* c, gpud_store* st, const char* table) {
  if (!c || !c->temp) return GPUD_E_INVALID;
  std::lock_guard<std::mutex> g(c->check_mu);
  return c->temp->SetMetricsStore(st, table);
}
