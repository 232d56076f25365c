/* gpud_b200.h — C ABI of libgpud_b200.so: the B200-native telemetry aggregation / Xid scan hot path of gpud.
 *
 * This is the drop-in boundary a thin cgo file in a gpud `components.Component` would bind
 * (INTEGRATION.md shows the stub).  The reference has no FFI seam of its own (it is 100 % Go,
 * SURVEY.md §0); each entry point names the reference function(s) whose work it replaces.
 *
 * Conventions
 *  - every function returns int32 status: 0 = GPUD_OK, <0 = GPUD_E_*; gpud_last_error() copies the message.
 *  - no exceptions, no callbacks, nothing retains caller memory after return (cgo pointer rule).
 *  - the library owns device memory and pinned staging; the caller owns every buffer it passes.
 *  - callable from any OS thread: each entry does cudaSetDevice itself.  Calls on the same ring / the
 *    same (ctx, dev) scanner must be serialised by the caller (the Go side holds a mutex, like
 *    `lastMu` in components/accelerator/nvidia/temperature/component.go:99-104).
 *  - there is NO CPU fallback: without a CUDA device every compute entry fails with GPUD_E_CUDA.
 */
#ifndef GPUD_B200_H
#define GPUD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GPUD_ABI_VERSION 1

#define GPUD_OK 0
#define GPUD_E_INVALID (-1)  /* bad argument                                   */
#define GPUD_E_CUDA (-2)     /* CUDA runtime error (message has the cudaError)  */
#define GPUD_E_NOMEM (-3)
#define GPUD_E_CAPACITY (-4) /* caller's output buffer too small; *n_* = needed */
#define GPUD_E_NCCL (-5)
#define GPUD_E_STATE (-6)    /* call order (e.g. read before reduce)            */
#define GPUD_E_UNSUPPORTED (-7) /* a host facility is missing (NVML for the poller) */

typedef struct gpud_ctx gpud_ctx;
typedef struct gpud_ring gpud_ring;

int32_t gpud_abi_version(void);
/* sizeof of the ABI structs for binding layout checks (5 gpud_kmsg_event, 6 gpud_ib_snapshot, 7 gpud_ib_verdict, 8 gpud_metric):
 * 0 gpud_xid_hit, 1 gpud_fabric_raw, 2 gpud_fabric_local,
 * 3 gpud_fabric_verdict, 4 gpud_ring_cfg, 9 gpud_dedup_rule .. 12 gpud_event_row, 13 gpud_nvml_device, 14 gpud_remapped_rows, 15 gpud_ecc_errors, 16 gpud_gpm_metrics,
 * 17 gpud_drain_info; -1 otherwise. */
int32_t gpud_sizeof(int32_t which);

/* One context per process; `cuda_devs[n]` are the CUDA ordinals this process drives (one per rank when
 * launched one-process-per-GPU).  Replaces the per-process NVML instance wiring of
 * pkg/nvidia/nvml/instance.go:110-273 for the compute side (NVML itself stays the data source). */
int32_t gpud_ctx_create(const int32_t* cuda_devs, int32_t n, gpud_ctx** out);
int32_t gpud_ctx_destroy(gpud_ctx* ctx);
/* Thread-safe copy of the last error message recorded on this ctx (NUL-terminated, truncated to cap). */
int32_t gpud_last_error(gpud_ctx* ctx, char* buf, int32_t cap);

/* Pinned host memory for sample batches / log buffers a caller wants DMA'd without the staging copy. */
int32_t gpud_host_alloc(int64_t bytes, void** out);
int32_t gpud_host_free(void* p);

/* ------------------------------------------------------------------------------------------------
 * Counter-sample ring + windowed aggregates.
 * Replaces: the gauge -> scrape -> SQLite row path of pkg/metrics (scraper/prometheus.go:28-81,
 * syncer/syncer.go:36-82, store/sqlite.go:108-164) as the sample sink, and adds the windowed
 * min/max/mean/EMA/p99/threshold-count the north star asks for.  The reference has NO implementation
 * of those aggregates: definitions are oracle/SPEC.md ("parity unpinned").  The strict `>` of n_over
 * mirrors components/accelerator/nvidia/temperature/component.go:228,240.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  int32_t n_fields;         /* F: gauges per GPU (api/v1/types.go:136-141 fixes the sample type: f64)   */
  int32_t window;           /* W: tumbling window length in samples, 1..1024                            */
  int64_t capacity;         /* CAP: samples kept per field (even, >= window)                            */
  double ema_alpha;         /* 0 => min(2/(W+1), 0.9999); otherwise in (0, 0.9999]                    */
  int32_t q_num, q_den;     /* order statistic, nearest rank ceil(m*q_num/q_den); 0/0 => 99/100         */
  const double* thresholds; /* [F] or NULL (= +inf: nothing counts)                                     */
} gpud_ring_cfg;

enum { GPUD_OP_MIN = 0, GPUD_OP_MAX = 1, GPUD_OP_MEAN = 2, GPUD_OP_EMA = 3, GPUD_OP_P99 = 4, GPUD_OP_NOVER = 5, GPUD_N_OPS = 6 };

int32_t gpud_ring_create(gpud_ctx* ctx, int32_t dev, const gpud_ring_cfg* cfg, gpud_ring** out);
int32_t gpud_ring_destroy(gpud_ring* ring);
/* Use an existing CUDA stream (cudaStream_t as void*) for every launch/copy of this ring; NULL = the ring's own. */
int32_t gpud_ring_set_stream(gpud_ring* ring, void* cuda_stream);
/* Append n_rows polls.  host_rows is [n_rows][F] row-major f64 in ordinary host memory (one row = one
 * poll of all F gauges, the shape the poll loop produces, temperature/component.go:165-273).  The rows are
 * staged through the library's pinned double buffers, copied with cudaMemcpyAsync and scattered into the
 * field-major ring [F][CAP] by the append kernel.  Returns after the caller's buffer has been consumed. */
int32_t gpud_ring_push(gpud_ring* ring, const double* host_rows, int64_t n_rows);
/* Same, source already in device memory on the ring's device (append kernel only). */
int32_t gpud_ring_push_device(gpud_ring* ring, const double* dev_rows, int64_t n_rows);
/* Same as gpud_ring_push for rows of RAW counter samples in the getter's own type: NVML returns uint32 (temperature C,
 * power mW, clocks MHz, utilisation %: pkg/nvidia/nvml/lib/... getters behind temperature/component.go:252-272,
 * power/component.go, clock-speed/component.go) or uint64 (memory bytes, ECC counts); DCGM fields are int64 or double.
 * The widening the reference does on the host - metric.Set(float64(v)) - happens in the append kernel instead (exact;
 * round-to-nearest-even above 2^53 like Go), so a uint32 poll row crosses PCIe at half the bytes. */
enum { GPUD_DT_F64 = 0, GPUD_DT_U32 = 1, GPUD_DT_I32 = 2, GPUD_DT_F32 = 3, GPUD_DT_I64 = 4, GPUD_DT_U64 = 5,
       GPUD_DT_U16 = 6, GPUD_DT_I16 = 7, GPUD_DT_U8 = 8 };   /* narrow gauges: degrees C, percent, MHz */
int32_t gpud_ring_push_raw(gpud_ring* ring, const void* host_rows, int64_t n_rows, int32_t dtype);

/* getClockEventReasons (hw-slowdown/clock_events.go:151-153,168-264): what the set bits of an
 * nvmlDeviceGetCurrentClocksEventReasons bitmask mean.  hw_out / other_out receive the sorted descriptions, one per line;
 * flags3 = {HWSlowdown, HWSlowdownThermal, HWSlowdownPowerBrake}.  Returns 100 * n_hw + n_other, -1 if a buffer is too small. */
int32_t gpud_clock_event_reasons(uint64_t bitmask, char* hw_out, int32_t hw_cap, char* other_out, int32_t other_cap, int32_t* flags3);
/* ClockEvents.HWSlowdownEvent's Message (hw-slowdown/clock_events.go:87-102,158-161): "<uuid>: <reason>" for every hardware-slowdown
 * reason of the bitmask, sorted, joined by ", ".  Returns the length, 0 when the reading yields no event, -1 if it does not fit. */
int32_t gpud_hw_slowdown_event_message(uint64_t bitmask, const char* gpu_uuid, char* out, int32_t cap);
/* The evaluation half of the hw-slowdown Check (hw-slowdown/component.go:352-407): event times as read back from the bucket (the rule
 * keeps those strictly after now - window, pkg/eventstore/database.go:330), distinct event-minutes / window minutes >= threshold ->
 * health 2 (Unhealthy) with RepairActionTypeHardwareInspection and the reference's reason text; defaults 10 min / 0.6 (:29-35). */
int32_t gpud_hw_slowdown_check(const int64_t* event_unix, int32_t n, int64_t now_unix, int64_t window_seconds, double threshold_per_minute,
                               int32_t* health, double* freq_per_minute, int32_t* hardware_inspection, char* reason, int32_t reason_cap);

/* Real ingest (SURVEY.md 8f.3): a host poller that reads the NVML gauges of CUDA device `dev` - the getters behind the
 * reference's temperature / power / clock-speed / utilization / memory components (temperature/temperature.go:85,
 * power/power.go:46, clock-speed/clock_speed.go:41,59, utilization/utilization.go:44, memory/memory.go:83) - into pinned
 * uint32 poll rows and appends them to `ring` with gpud_ring_push_timed.  The ring must have GPUD_POLL_N_FIELDS fields, in this
 * column order.  NVML is dlopen'ed; GPUD_E_UNSUPPORTED if the host has no driver library.  Every row is pushed with the wall-clock ms its
 * getters returned at (gpud_ring_push_timed), as are the rows of gpud_poller_poll_fields and gpud_poller_poll_gpm. */
enum { GPUD_POLL_TEMPERATURE_C = 0, GPUD_POLL_POWER_MW = 1, GPUD_POLL_CLOCK_GRAPHICS_MHZ = 2, GPUD_POLL_CLOCK_SM_MHZ = 3,
       GPUD_POLL_CLOCK_MEM_MHZ = 4, GPUD_POLL_UTIL_GPU_PCT = 5, GPUD_POLL_UTIL_MEM_PCT = 6, GPUD_POLL_MEMORY_USED_MIB = 7,
       GPUD_POLL_N_FIELDS = 8 };
/* A getter that fails does NOT put a sentinel into the ring: the column holds its last good value (0 before the first good read,
 * oracle/SPEC.md) and the failure is recorded for gpud_poller_errors.  gpud_poll_row_hold is that rule as a pure function:
 * fresh[c] is taken when nvml_rc[c] == 0, otherwise held[c] is repeated and bit c of *fail_mask is set. */
int32_t gpud_poll_row_hold(const uint32_t* fresh, const int32_t* nvml_rc, int32_t n_cols, uint32_t* held, uint32_t* row_out, uint32_t* fail_mask);
typedef struct gpud_poller gpud_poller;
int32_t gpud_poller_create(gpud_ctx* ctx, int32_t dev, gpud_ring* ring, gpud_poller** out);
void gpud_poller_destroy(gpud_poller* poller);
/* Take n_polls poll rows (interval_us apart; 0 = back to back) and append them.  Synchronous. */
int32_t gpud_poller_poll(gpud_poller* poller, int64_t n_polls, int64_t interval_us);
/* The rows of the last push batch (at most 16384) as they went over PCIe, and the wall time of the last poll call. */
int32_t gpud_poller_last_rows(gpud_poller* poller, uint32_t* rows, int64_t cap_rows, int64_t* n_rows, double* seconds);
/* Columns whose getter failed at least once since create (bit c), each column's last NVML return code and failure count
 * ([GPUD_POLL_N_FIELDS] each; any pointer may be NULL). */
int32_t gpud_poller_errors(gpud_poller* poller, uint32_t* fail_mask, int32_t* last_nvml_rc, uint64_t* n_failed);
/* GetTemperature (temperature/temperature.go:78-221) for this poller's GPU, and the per-GPU rules of the temperature component's
 * Check (temperature/component.go:206-248) over such a reading: *bits = 1 GPU core above its max-operating threshold | 2 HBM above
 * the memory max | 4 thermal margin at or below margin_threshold_c (0 = rule off, temperature/threshold.go:13); the component's
 * reason is the first of margin, GPU, HBM (:273-287), its health Degraded when any bit is set. */
typedef struct {
  uint32_t current_gpu_core_c, current_hbm_c;
  uint32_t threshold_shutdown_c, threshold_slowdown_c, threshold_mem_max_c, threshold_gpu_max_c;
  int32_t slowdown_margin_c;
  uint8_t hbm_supported, margin_supported, pad[2];
} gpud_temperature;
int32_t gpud_poller_temperature(gpud_poller* poller, gpud_temperature* out);
int32_t gpud_temperature_check(const gpud_temperature* t, int32_t margin_threshold_c, int32_t* bits);
/* The component's check result over the box's n readings (temperature/component.go:190-287): *health 0 Healthy / 1 Degraded, and the
 * reason text -- the findings of the first non-empty class (margin, GPU, HBM) as "<uuid> ..." joined by ", " in the order given, or
 * "all n GPU(s) were checked, no temperature issue found".  Returns the length, -1 if it does not fit. */
int32_t gpud_temperature_reason(const gpud_temperature* ts, const char* const* gpu_uuids, int32_t n, int32_t margin_threshold_c, int32_t* health,
                                char* out, int32_t cap);
/* GetClockEvents' reasons bitmask (hw-slowdown/clock_events.go:111-166; decode with gpud_clock_event_reasons) and the four ECC
 * totals of ecc/ecc_errors.go:136-240; ecc_read_mask bit 0..3 = aggregate corrected, aggregate uncorrected, volatile corrected,
 * volatile uncorrected were read. */
typedef struct {
  uint64_t clock_event_reasons;
  uint64_t ecc_aggregate_corrected, ecc_aggregate_uncorrected, ecc_volatile_corrected, ecc_volatile_uncorrected;
  uint32_t clock_events_supported, ecc_read_mask;
} gpud_poll_counters;
int32_t gpud_poller_counters(gpud_poller* poller, gpud_poll_counters* out);
/* The fused window reduce runs a persistent grid that fills every CTA slot of the GPU (2 per SM, the whole register file), so a
 * kernel launched meanwhile on another stream - the fabric record's pack / all-gather / verdict - could only start by delaying one of
 * the grid's CTAs, which then finishes a whole kernel-time late.  Leaving n_ctas slots out of the grid (work is divided over whatever
 * grid is launched; each slot costs 1/296 of the throughput) lets such kernels run concurrently.  Default 0.  A collective that runs
 * beside the reduce needs as many slots as it has CTAs: NCCL opens one channel (one CTA) per NVLink between two GPUs unless it is held
 * back (NCCL_MAX_CTAS / ncclConfig_t.maxCTAs = 1 is plenty for the 128-byte fabric record; bench.py does that). */
int32_t gpud_ring_set_cta_reserve(gpud_ring* ring, int32_t n_ctas);
/* Rows A3 / A4 of the hot path's NVML side.
 * gpud_nvml_devices: nvml.New's enumeration (pkg/nvidia/nvml/instance.go:197-273, device/device.go:46-70): per device the UUID, the
 * PCI bus id in go-nvlib's GetPCIBusID form ("0000:3b:00.0"; gpud_nvml_bus_id is that conversion alone), the product name, the CUDA
 * ordinal (-1 if CUDA does not see it) and, when a getter failed, its NVML return code (the "errored instance" case).  *n = devices
 * NVML reports (GPUD_E_CAPACITY if more than cap).  gpud_nvml_devices_arg renders "uuid=bus_id;..." - the `devices` argument of
 * gpud_xid_state_from_store - and returns its length. */
typedef struct { int32_t index, cuda_device, nvml_rc, pad; char uuid[96]; char bus_id[32]; char name[96]; } gpud_nvml_device;
int32_t gpud_nvml_devices(gpud_nvml_device* out, int32_t cap, int32_t* n, char* driver_version, int32_t driver_version_cap);
int32_t gpud_nvml_devices_arg(char* out, int32_t cap);
int32_t gpud_nvml_bus_id(const char* nvml_bus_id, char* out, int32_t cap);
/* GetRemappedRows (remapped-rows/remapped_rows.go:52-86) for the poller's GPU, and the component's Check over the box's readings
 * (remapped-rows/component.go:197-300): *health 0 Healthy / 2 Unhealthy, *action GPUD_ACT_HARDWARE_INSPECTION once any GPU's remapping
 * failed, else GPUD_ACT_REBOOT_SYSTEM when one is pending, else 0; returns the reason's length, -1 if it does not fit. */
typedef struct { int32_t remapped_due_to_correctable_errors, remapped_due_to_uncorrectable_errors; uint8_t remapping_pending, remapping_failed, supported, pad; } gpud_remapped_rows;
int32_t gpud_poller_remapped_rows(gpud_poller* poller, gpud_remapped_rows* out);
int32_t gpud_remapped_rows_check(const gpud_remapped_rows* rows, const char* const* bus_ids, int32_t n, int32_t* health, int32_t* action, char* reason, int32_t cap);
/* GetECCModeEnabled + GetECCErrors (ecc/ecc_mode.go, ecc/ecc_errors.go:136-880): totals and - with ECC mode on - the per-location
 * counters nvmlDeviceGetMemoryErrorCounter reports, in the slots of the reference's AllECCErrorCounts; the first "not supported" ends
 * the read with supported = 0. */
enum { GPUD_ECC_TOTAL = 0, GPUD_ECC_L1 = 1, GPUD_ECC_L2 = 2, GPUD_ECC_DRAM = 3, GPUD_ECC_SRAM = 4, GPUD_ECC_DEVICE_MEMORY = 5, GPUD_ECC_TEXTURE_MEMORY = 6,
       GPUD_ECC_SHARED_MEMORY = 7, GPUD_ECC_REGISTER_FILE = 8, GPUD_ECC_N_LOCATIONS = 9 };
typedef struct { uint64_t corrected, uncorrected; } gpud_ecc_counts;
typedef struct { gpud_ecc_counts aggregate[GPUD_ECC_N_LOCATIONS]; gpud_ecc_counts volatile_[GPUD_ECC_N_LOCATIONS]; uint8_t ecc_mode_current, ecc_mode_pending, supported, pad[5]; } gpud_ecc_errors;
int32_t gpud_poller_ecc_errors(gpud_poller* poller, gpud_ecc_errors* out);
/* One driver round trip per poll row (SURVEY.md 8f.3): nvmlDeviceGetFieldValues over the GPUD_FIELD_ROW_N counters below, widened to
 * uint64.  gpud_poller_field_row reads one row (nvml_rc[i] = that field's own return code, may be NULL); gpud_poller_poll_fields takes
 * n_polls rows and appends them to `ring` (GPUD_FIELD_ROW_N fields) as raw uint64 rows; a field that fails holds its last good value. */
enum { GPUD_FIELD_POWER_INSTANT_MW = 0, GPUD_FIELD_POWER_AVERAGE_MW = 1, GPUD_FIELD_MEMORY_TEMP_C = 2, GPUD_FIELD_TOTAL_ENERGY_MJ = 3,
       GPUD_FIELD_ECC_SBE_VOLATILE = 4, GPUD_FIELD_ECC_DBE_VOLATILE = 5, GPUD_FIELD_ECC_SBE_AGGREGATE = 6, GPUD_FIELD_ECC_DBE_AGGREGATE = 7,
       GPUD_FIELD_NVLINK_CRC_FLIT_TOTAL = 8, GPUD_FIELD_NVLINK_CRC_DATA_TOTAL = 9, GPUD_FIELD_NVLINK_REPLAY_TOTAL = 10, GPUD_FIELD_NVLINK_RECOVERY_TOTAL = 11,
       GPUD_FIELD_REMAPPED_CORRECTABLE = 12, GPUD_FIELD_REMAPPED_UNCORRECTABLE = 13, GPUD_FIELD_REMAPPED_PENDING = 14, GPUD_FIELD_REMAPPED_FAILURE = 15,
       GPUD_FIELD_PCIE_REPLAY = 16, GPUD_FIELD_ROW_N = 17 };
int32_t gpud_poller_field_row(gpud_poller* poller, uint64_t* values, int32_t* nvml_rc);
int32_t gpud_poller_poll_fields(gpud_poller* poller, gpud_ring* ring, int64_t n_polls, int64_t interval_us, double* seconds);
/* GPM (components/accelerator/nvidia/gpm): SupportedByDevice (gpm.go:17-45; "not supported" and "version mismatch" answers, or an NVML
 * without the GPM entry points, mean 0) and GetGPMMetrics (gpm.go:65-149): two nvmlGpmSampleGet `sample_ms` apart (the component: 5000)
 * and one nvmlGpmMetricsGet over the component's nine metric ids (component.go:56-64), in the order of the enum; supported = 0 and
 * zeroes where the device has no GPM.  gpud_poller_poll_gpm is the same getter as a field source: n_polls float64 rows of the nine
 * metrics appended to `ring` (GPUD_GPM_N fields), consecutive rows sharing a sample.  gpud_gpm_check is the component's Check over
 * the box's readings (component.go:196-290): returns the reason's length, -1 if it does not fit; *health 0 Healthy. */
enum { GPUD_GPM_SM_OCCUPANCY = 0, GPUD_GPM_INTEGER_UTIL = 1, GPUD_GPM_ANY_TENSOR_UTIL = 2, GPUD_GPM_DFMA_TENSOR_UTIL = 3, GPUD_GPM_HMMA_TENSOR_UTIL = 4,
       GPUD_GPM_IMMA_TENSOR_UTIL = 5, GPUD_GPM_FP64_UTIL = 6, GPUD_GPM_FP32_UTIL = 7, GPUD_GPM_FP16_UTIL = 8, GPUD_GPM_N = 9 };
typedef struct { double value[GPUD_GPM_N]; int32_t nvml_rc[GPUD_GPM_N]; int32_t supported; double sample_seconds; } gpud_gpm_metrics;
int32_t gpud_poller_gpm_supported(gpud_poller* poller, int32_t* supported);
int32_t gpud_poller_gpm_metrics(gpud_poller* poller, int64_t sample_ms, gpud_gpm_metrics* out);
int32_t gpud_poller_poll_gpm(gpud_poller* poller, gpud_ring* ring, int64_t n_polls, int64_t sample_ms, double* seconds);
int32_t gpud_gpm_check(const gpud_gpm_metrics* metrics, int32_t n, int32_t* health, char* reason, int32_t cap);
int32_t gpud_ring_counts(gpud_ring* ring, int64_t* total_pushed, int64_t* count, int64_t* n_windows);
/* Launch the fused window-reduce (+ EMA carry) over the ring's current content; asynchronous. */
int32_t gpud_ring_reduce(gpud_ring* ring);
int32_t gpud_ring_sync(gpud_ring* ring);
/* Device time of the last reduce's two kernels (CUDA events recorded on the ring's stream around each launch). */
int32_t gpud_ring_kernel_ms(gpud_ring* ring, float* reduce_ms, float* carry_ms);
/* Copy one aggregate to host: [F][n_windows] row-major; f64 for MIN..P99, uint32 for NOVER.  Synchronises. */
int32_t gpud_ring_read(gpud_ring* ring, int32_t op, void* out, int64_t out_bytes);
/* Device pointer of an aggregate (same layout), valid until the next reduce/destroy. */
int32_t gpud_ring_result_ptr(gpud_ring* ring, int32_t op, void** dev_ptr);

/* Whole-range aggregates of the most recent `last_n` samples of every field (last_n = 0 => whole ring, i.e. the W = CAP order
 * statistic of BASELINE configs[3]); exact.  Ranges of >= 64 Ki samples read HBM once (sampled pivots + classification fused into
 * the window pass), shorter ones and any field the sample misjudged use a multi-pass radix select.  out_f64 is [5][F]
 * (MIN,MAX,MEAN,EMA,P99), n_over [F].  Synchronous. */
int32_t gpud_ring_reduce_range(gpud_ring* ring, int64_t last_n, double* out_f64, uint32_t* out_n_over);
/* Device time of the last gpud_ring_reduce_range that took the single-pass route: pivots + fused range pass + EMA carry, and the
 * whole device side (+ finish), and how many fields had to be re-done by the radix select (normally 0) with the reason for each
 * (reasons[GPUD_RANGE_OPEN_*] counts fields; may be NULL). */
enum { GPUD_RANGE_OPEN_SHORT = 1,    /* the range is shorter than the single-pass threshold          */
       GPUD_RANGE_OPEN_NAN = 2,      /* the field holds a +NaN (ordered above +inf, SPEC.md)          */
       GPUD_RANGE_OPEN_PIVOTS = 3,   /* the sample produced NaN pivots                                */
       GPUD_RANGE_OPEN_ABOVE = 4,    /* the wanted rank lies above the upper pivot                    */
       GPUD_RANGE_OPEN_BELOW = 5,    /* ... below the lower pivot                                     */
       GPUD_RANGE_OPEN_OVERFLOW = 6, /* more keys between the pivots than the list holds              */
       GPUD_RANGE_N_OPEN_REASONS = 7 };
int32_t gpud_ring_range_stats(gpud_ring* ring, float* pass_ms, float* total_ms, int32_t* fields_by_histogram, int32_t* reasons);

/* Streaming windows: what a metrics syncer (pkg/metrics/syncer/syncer.go:76-82, which scrapes the gauges of
 * pkg/metrics/scraper/prometheus.go:28-81 on its ticker) reads from the ring instead of the gauges.  Sample i of a field is the i-th
 * sample pushed since gpud_ring_create (rows a push skips because n_rows > CAP still count); window k is samples [kW, (k+1)W), complete
 * once (k+1)W <= total.  The ring keeps a cursor `next` (first window not drained yet, initially 0).  A drain returns complete windows
 * from k0 = max(next, ceil((total - count) / W)) upward, oldest first, each reduced on the GPU exactly once:
 *   n_lost = k0 - next windows were overwritten before they were drained; n_windows = min(floor(total / W) - k0, max_windows) are
 *   returned (window first_window + j); n_pending complete windows remain.  Afterwards next = k0 + n_windows.  max_windows = 0 is a
 *   query: *info is filled and nothing moves.
 * min / max / p<q> / n_over / mean are the aggregates of gpud_ring_reduce over the window's W samples.  The EMA runs over the stream and
 * continues from the last window the previous drain returned, except on the first drain and after a loss, where it starts at the first
 * sample of the first returned window.  Output: out_f64[(op * F + f) * max_windows + j] for op GPUD_OP_MIN .. GPUD_OP_P99,
 * n_over[f * max_windows + j], window_end_unix_ms[j] (may be NULL) = the time of the window's last row when that row came through
 * gpud_ring_push_timed, else 0.  The results of gpud_ring_reduce / gpud_ring_read are not touched.  Synchronous. */
typedef struct { int64_t first_window, n_windows, n_lost, n_pending; } gpud_drain_info;
int32_t gpud_ring_drain(gpud_ring* ring, int64_t max_windows, double* out_f64, uint32_t* out_n_over, int64_t* window_end_unix_ms, gpud_drain_info* info);
/* gpud_ring_push_raw with the time each row was read (unix ms, row_unix_ms[n_rows]): non-decreasing within the call and not earlier
 * than the last timed row, else GPUD_E_INVALID and nothing is appended.  Untimed pushes give the windows they complete time 0. */
int32_t gpud_ring_push_timed(gpud_ring* ring, const void* host_rows, int64_t n_rows, int32_t dtype, const int64_t* row_unix_ms);

/* ------------------------------------------------------------------------------------------------
 * components.Component (components/types.go:20-66) for the three paths this library replaces, as objects: what a Go file that
 * implements the interface forwards to, method by method.
 *   name                                 reference component                           Check()
 *   "accelerator-nvidia-error-xid"       xid/component.go:255-311, 468-611             scan the kmsg bytes on the GPU, persist new hits in the
 *                                                                                      event bucket, evolveHealthyState over bucket + reboots
 *   "accelerator-nvidia-temperature"     temperature/component.go:81-287               one NVML poll row per GPU into its ring (the windowed
 *                                                                                      aggregates stay readable through gpud_component_ring),
 *                                                                                      the threshold rules over the current reading
 *   "accelerator-nvidia-nvlink"          nvlink/component.go:164-311                   every GPU's NVLink / fabric record, gathered over NVLink
 *                                                                                      peer stores, the replicated box verdict
 * Start is non-blocking: it spawns a ticker that runs Check at once and then every interval; Check embeds errors in the state and
 * never fails the call; LastHealthStates is the cached apiv1.HealthStates JSON, a single Healthy "no data yet" state before the first
 * check; Events is apiv1.Events JSON, newest first, strictly after `since`; Close stops the ticker.  Safe to call from any thread.
 * ---------------------------------------------------------------------------------------------- */
typedef struct gpud_component gpud_component;
typedef struct {
  int32_t row_remapping_supported; /* xid: drop Xid 63 / 64, they belong to the remapped-rows component (xid/component.go:290) */
  int32_t reboot_threshold;        /* xid: reboots after which the action becomes HARDWARE_INSPECTION (default 2)               */
  int32_t margin_threshold_c;      /* temperature: thermal-margin rule, 0 = off (temperature/threshold.go:13)                   */
  int32_t nvlink_at_least;         /* nvlink: GPUs that must have every link up, 0 = no threshold (nvlink/threshold.go)         */
} gpud_component_cfg;
int32_t gpud_component_create(gpud_ctx* ctx, const char* name, const gpud_component_cfg* cfg /* NULL = defaults */, gpud_component** out);
void gpud_component_destroy(gpud_component* c);
int32_t gpud_component_name(gpud_component* c, char* out, int32_t cap);
int32_t gpud_component_start(gpud_component* c, int64_t interval_ms);                       /* Start() */
int32_t gpud_component_check(gpud_component* c, int32_t* health, char* reason, int32_t cap); /* Check(): health 0 Healthy / 1 Degraded / 2 Unhealthy */
int32_t gpud_component_last_health_states(gpud_component* c, char* json, int32_t cap);       /* returns the length */
int32_t gpud_component_events(gpud_component* c, int64_t since_unix, char* json, int32_t cap);
int32_t gpud_component_close(gpud_component* c);                                             /* Close() */
int64_t gpud_component_checks(gpud_component* c);                                            /* checks run so far (ticker + direct) */
/* xid: the bytes Check scans (what kmsg.ReadAll returned; raw_kmsg: /dev/kmsg records, event time = boot_unix + usec), SetHealthy
 * (xid/set_healthy.go:14-35), a reboot event of the os bucket, the UUID -> bus id map ("uuid=bus_id;...", gpud_nvml_devices_arg). */
int32_t gpud_component_xid_set_source(gpud_component* c, const uint8_t* buf, int64_t len, int32_t raw_kmsg, int64_t boot_unix);
int32_t gpud_component_xid_set_healthy(gpud_component* c, int64_t now_unix);
int32_t gpud_component_xid_add_reboot(gpud_component* c, int64_t unix_s);
int32_t gpud_component_xid_set_devices(gpud_component* c, const char* devices);
/* temperature: the ring the polls of the ctx's slot-th device land in (NULL otherwise) */
gpud_ring* gpud_component_ring(gpud_component* c, int32_t slot);

/* ------------------------------------------------------------------------------------------------
 * kmsg Xid / SXid scan + classification.
 * Replaces: xid.Match (components/accelerator/nvidia/xid/kmsg.go:202-245 with the regexes at :22,:29,:38,:43),
 * sxid.Match (sxid/kmsg.go:58-73, regexes :17,:20), the catalog lookups GetDetail / detailFromNVLinkInfo
 * (xid/xid.go:74-117, 2954-2995) applied per line of a buffer as in xid/kmsg_test.go:252-267 and
 * xid/component.go:274-299.
 * ---------------------------------------------------------------------------------------------- */
enum { GPUD_SCAN_LINES = 0,   /* units are '\n'-separated lines (strings.Split(buf, "\n"))                  */
       GPUD_SCAN_RAW_KMSG = 1 /* units are /dev/kmsg records "prio,seq,usec,flags;msg" (+ " KEY=val" lines);
                                 Match runs on the message part (pkg/kmsg/watcher.go:292-332)               */ };
/* OR into `mode`: also run the stateless line matchers of the other kmsg-reading components on every unit (SURVEY.md
 * 8f.1), one hit per (unit, pattern); the pattern is the hit's `kind`:
 *   nccl        `.*segfault at.*in libnccl\.so.*`                      components/accelerator/nvidia/nccl/kmsg_matcher.go:12
 *   peermem     `.*ERROR detected invalid context, skipping further processing`      .../peermem/kmsg_matcher.go:14
 *   infiniband  pci power / port module temperature / ACCESS_REG        .../infiniband/kmsg_matcher.go:15,25,57
 *   cpu         blocked too long / soft lockup (capture: "comm:pid")    components/cpu/kmsg_matcher.go:18,30
 *   os          VFS file-max limit reached                              components/os/kmsg_matcher.go:18
 *   disk        the eight patterns of                                   components/disk/kmsg_matcher.go:11-55
 * For these kinds dev_off/dev_len (and device[], truncated) hold the capture the component appends to its message
 * (cpu: process info; infiniband ACCESS_REG: the first PCI BDF of the line; else empty) and `link` the byte offset the
 * match is anchored at.
 * The two STATEFUL matchers (os kernel-panic assembly os/kmsg_matcher.go:60-125, memory OOM parser
 * memory/kmsg_matcher.go:29-109) are split: the scan reports their six line primitives (kinds 19..24) with the capture
 * groups the state machines read as buffer spans -
 *   OS_PANIC_CPU_PID       dev = CPU digits, pid = PID digits, pname = Comm
 *   MEM_OOM_CONTAINER      dev = constraint, unit_name = oom_memcg, inj = task_memcg, pname = task, pid = pid
 *   MEM_OOM_LEGACY_CONTAINER  dev = group 1, unit_name = group 2        MEM_OOM_KILLED_PROCESS  pid, pname
 * - and gpud_kmsg_stateful_feed() runs the reference's two state machines over them. */
#define GPUD_SCAN_EXT_MATCHERS 0x100
enum {
  GPUD_KIND_XID = 1, GPUD_KIND_SXID = 2, GPUD_KIND_NCCL_SEGFAULT = 3, GPUD_KIND_PEERMEM_INVALID_CONTEXT = 4,
  GPUD_KIND_IB_PCI_POWER_INSUFFICIENT = 5, GPUD_KIND_IB_PORT_MODULE_HIGH_TEMPERATURE = 6, GPUD_KIND_IB_ACCESS_REG_FAILED = 7,
  GPUD_KIND_CPU_BLOCKED_TOO_LONG = 8, GPUD_KIND_CPU_SOFT_LOCKUP = 9, GPUD_KIND_OS_VFS_FILE_MAX_LIMIT_REACHED = 10,
  GPUD_KIND_DISK_RAID_ARRAY_FAILURE = 11, GPUD_KIND_DISK_FILESYSTEM_READ_ONLY = 12, GPUD_KIND_DISK_NVME_PATH_FAILURE = 13,
  GPUD_KIND_DISK_NVME_TIMEOUT = 14, GPUD_KIND_DISK_NVME_DEVICE_DISABLED = 15, GPUD_KIND_DISK_BEYOND_END_OF_DEVICE = 16,
  GPUD_KIND_DISK_BUFFER_IO_ERROR = 17, GPUD_KIND_DISK_SUPERBLOCK_WRITE_ERROR = 18,
  /* line primitives of the two stateful matchers: not events by themselves, input of gpud_kmsg_stateful_feed */
  GPUD_KIND_OS_PANIC_START = 19, GPUD_KIND_OS_PANIC_CPU_PID = 20, GPUD_KIND_MEM_OOM_START = 21, GPUD_KIND_MEM_OOM_CONTAINER = 22,
  GPUD_KIND_MEM_OOM_LEGACY_CONTAINER = 23, GPUD_KIND_MEM_OOM_KILLED_PROCESS = 24, GPUD_KIND_COUNT = 25
};
enum { GPUD_EVENT_UNKNOWN = 0, GPUD_EVENT_INFO = 1, GPUD_EVENT_WARNING = 2, GPUD_EVENT_CRITICAL = 3, GPUD_EVENT_FATAL = 4 };
enum { GPUD_ACT_IGNORE_NO_ACTION_REQUIRED = 1, GPUD_ACT_REBOOT_SYSTEM = 2, GPUD_ACT_HARDWARE_INSPECTION = 3,
       GPUD_ACT_CHECK_USER_APP_AND_GPU = 4 };
#define GPUD_HIT_EXTENDED 0x1u      /* matched the NVLink5 extended format (kmsg.go:29)                       */
#define GPUD_HIT_FALLEN_OFF_BUS 0x2u /* xid 79 implied by the fallen-off-the-bus fallbacks (kmsg.go:38,43)    */
#define GPUD_HIT_DEV_TRUNCATED 0x4u /* device string longer than the inline copy; use dev_off/dev_len       */
#define GPUD_HIT_HAS_RULE 0x8u      /* an NVLink decode rule matched (xid.go:3099-3114); rule_index is valid  */

typedef struct {
  int64_t unit_index;    /* 0-based line (LINES) or record (RAW_KMSG) number                               */
  int64_t unit_offset;   /* byte offset of the line / record start in the scanned buffer                  */
  int64_t dev_off;       /* byte offset and length of the device capture in the buffer                    */
  int32_t dev_len;
  int32_t kind;          /* GPUD_KIND_*                                                                    */
  int32_t code;          /* Xid or SXid                                                                    */
  uint32_t flags;        /* GPUD_HIT_*                                                                     */
  /* extended (NVLink5) fields, zero unless GPUD_HIT_EXTENDED — ExtractedInfo, kmsg.go:84-98               */
  int32_t sub_code;      /* (intrinfo >> 20) & 0x3F                                                        */
  int32_t kmsg_priority; /* RAW_KMSG only: parseLine fields (pkg/kmsg/watcher.go:292-332), else 0                 */
  int64_t kmsg_seq;
  int64_t kmsg_usec;     /* microseconds since boot; event time = boot time + kmsg_usec                           */
  int64_t link;          /* Atoi("-?\\d+"): Go int is 64-bit                                                      */
  uint32_t intrinfo;
  uint32_t error_status;
  uint32_t extra[4];
  int32_t n_extra;
  int32_t severity_fatal; /* log says "Fatal" (1) / "Nonfatal" (0)                                         */
  int32_t xc;             /* 0 / 1 from XC0 / XC1                                                          */
  int64_t unit_name_off;  /* capture 5 (sub-code mnemonic): offset/len in the buffer                       */
  int32_t unit_name_len;
  int64_t pid_off;        /* optional captures 3,4; len 0 when absent                                      */
  int32_t pid_len;
  int64_t pname_off;
  int32_t pname_len;
  int64_t inj_off;        /* capture 8 ("i0")                                                              */
  int32_t inj_len;
  /* classification (Detail of xid.go:12-42 as ids; strings are rendered by gpud_hit_detail_json)          */
  int32_t event_type;     /* GPUD_EVENT_*                                                                  */
  int32_t n_actions;      /* -1 = SuggestedActionsByGPUd nil                                               */
  int32_t actions[4];     /* GPUD_ACT_*, reference order                                                   */
  int32_t rule_index;     /* index into the NVLink rule table, -1 if none                                  */
  int32_t detail_variant; /* 0 base / sub-code table; 1, 2 = the 149.4 / 149.10 operational overrides       */
  char device[40];        /* NUL-terminated device id as Match returns it ("PCI:0000:05:00", "0000:03:00") */
  char unit_name[40];     /* NUL-terminated capture 5, truncated                                           */
} gpud_xid_hit;

/* Scan `len` bytes of host memory.  hits[cap] receives the hits in (unit_index, kind) order; *n_hits is the
 * number found (may exceed cap -> GPUD_E_CAPACITY, first cap are valid); *n_units = number of lines/records. */
int32_t gpud_kmsg_scan(gpud_ctx* ctx, int32_t dev, const uint8_t* buf, int64_t len, int32_t mode,
                       gpud_xid_hit* hits, int64_t cap, int64_t* n_hits, int64_t* n_units);
/* The same scan over every GPU of the ctx (SURVEY.md 8e): the buffer is cut at unit boundaries into one piece per device, the pieces
 * are scanned concurrently and the hits merged in unit order; result identical to gpud_kmsg_scan of the whole buffer. */
int32_t gpud_kmsg_scan_sharded(gpud_ctx* ctx, const uint8_t* buf, int64_t len, int32_t mode,
                               gpud_xid_hit* hits, int64_t cap, int64_t* n_hits, int64_t* n_units);
/* Device-resident variant: dev_buf on `dev`; kernels only, results copied to the caller's host arrays. */
int32_t gpud_kmsg_scan_device(gpud_ctx* ctx, int32_t dev, const uint8_t* dev_buf, int64_t len, int32_t mode,
                              gpud_xid_hit* hits, int64_t cap, int64_t* n_hits, int64_t* n_units, void* cuda_stream);
/* Device time (ms) of the last scan on `dev`.  By default the scan's kernels run as one overlapped chain (programmatic dependent
 * launch, no event between them): ms3[0] = the whole device time, ms3[1] = ms3[2] = 0.  After gpud_kmsg_scan_phase_timing(ctx, dev, 1)
 * the launches are plain and split by events: [0] anchor filter, [1] separator prefix, [2] match (candidate sort + automata + unit
 * numbers) - a profiling aid; the results of a scan do not depend on the setting. */
int32_t gpud_kmsg_scan_kernel_ms(gpud_ctx* ctx, int32_t dev, float* ms3);
int32_t gpud_kmsg_scan_phase_timing(gpud_ctx* ctx, int32_t dev, int32_t on);
/* Counters of the last scan on `dev`: [0] verified anchors, [1] hits, [2] unit separators. */
int32_t gpud_kmsg_scan_stats(gpud_ctx* ctx, int32_t dev, int64_t* out3);
/* Classify already-extracted hits (fills event_type/actions/rule_index/detail_variant) with the device LUT
 * kernel; `hits` is host memory, updated in place.  unit_name[] must hold capture 5 for extended hits. */
int32_t gpud_xid_classify(gpud_ctx* ctx, int32_t dev, gpud_xid_hit* hits, int64_t n);
/* Host-side rendering of the persisted payload (xidErrorEventDetail JSON, xid/health_state.go:284-315 and
 * xid/component.go:503-554) for one hit; `buf_bytes` is the scanned buffer (for long captures) or NULL. */
int32_t gpud_hit_detail_json(const gpud_xid_hit* hit, int64_t unix_seconds, char* out, int32_t cap);
/* Catalog accessors (xid/xid.go:74, sxid/sxid.go:32): description / mnemonic / name strings, "" if unknown. */
const char* gpud_xid_description(int32_t code, int32_t detail_variant);
const char* gpud_xid_mnemonic(int32_t code);
const char* gpud_sxid_name(int32_t code);
const char* gpud_nvlink_rule_hint(int32_t rule_index);
/* Reason string of the sxid component's health state (sxid/health_state.go:93-106); sxid < 0 = healthy. Returns the length. */
int32_t gpud_sxid_reason(int64_t sxid, const char* device, char* out, int32_t cap);
/* getDetailWithSubCodeAndStatus (xid/xid.go:97-107; falls back to the sub-code table, sub-code 0, then GetDetail): 1 = found.
 * event_type GPUD_EVENT_*, n_actions -1 = SuggestedActionsByGPUd nil, actions4[4] GPUD_ACT_*, detail_variant for
 * gpud_xid_description, sub_code_out = the Detail's SubCode.  Any out pointer may be NULL. */
int32_t gpud_xid_get_detail(int32_t xid, int32_t* event_type, int32_t* n_actions, int32_t* actions4);   /* GetDetail (xid/xid.go:74-77) */
int32_t gpud_sxid_get_detail(int32_t sxid, int32_t* event_type, int32_t* n_actions, int32_t* actions4); /* GetDetail (sxid/sxid.go:31-35) */
int32_t gpud_xid_detail(int32_t xid, int32_t sub_code, uint32_t error_status, int32_t* event_type, int32_t* n_actions, int32_t* actions4,
                        int32_t* detail_variant, int32_t* sub_code_out);
/* (*xidErrorEventDetail).buildMessage (xid/health_state.go:130-169): Message of a resolved xid event / Reason of the xid health
 * state, e.g. "XID 149.37 (err status 0x00000000) NVLINK_NETIR_ERROR detected on GPU PCI:0000:04:00 UUID:GPU-..."; gpu_uuid is the
 * NVML UUID convertBusIDToUUID resolved, or NULL.  _hit_ renders it for the payload gpud_hit_detail_json persists.  Return the
 * length, -1 if `out` is too small.  gpud_xid_device_matches_bus_id: the prefix test of convertBusIDToUUID (:171-182). */
int32_t gpud_xid_build_message(uint64_t xid, int32_t sub_code, uint32_t error_status, const char* description, const char* device_uuid,
                               const char* gpu_uuid, char* out, int32_t cap);
int32_t gpud_xid_hit_message(const gpud_xid_hit* hit, const char* gpu_uuid, char* out, int32_t cap);
int32_t gpud_xid_device_matches_bus_id(const char* device_uuid, const char* pci_bus_id);
/* GPU product capabilities from the NVML product name (pkg/nvidia/product/capabilities.go:56-137): memory error management
 * (bit 1 ErrorContainment, 2 DynamicPageOfflining, 4 RowRemapping -- the xid component drops Xid 63/64 when row remapping is
 * supported, xid/component.go:290,484), the on-node fabric manager, NVML fabric-state telemetry. */
int32_t gpud_product_mem_caps(const char* product_name);
int32_t gpud_product_fm_supported(const char* product_name);
int32_t gpud_product_fabric_state_supported(const char* product_name);
/* kmsg.MatchFunc results (eventName, message) of the extra matchers, by hit kind; "" for xid / sxid kinds. */
const char* gpud_kmsg_event_name(int32_t kind);
const char* gpud_kmsg_event_message(int32_t kind);
/* Component name that owns the pattern ("nccl", "peermem", "infiniband", "cpu", "os", "disk"). */
const char* gpud_kmsg_component(int32_t kind);
/* The message `Match` returns for this hit: the pattern's text plus the capture where the reference appends one
 * (cpu/kmsg_matcher.go:54-63, infiniband/kmsg_matcher.go:136-142).  `buf` is the scanned buffer (needed only when the
 * capture is longer than device[]: GPUD_HIT_DEV_TRUNCATED) or NULL.  Returns the length, -1 if `cap` is too small. */
int32_t gpud_kmsg_hit_message(const gpud_xid_hit* hit, const uint8_t* buf, char* out, int32_t cap);

/* The stateful matchers.  One object per kmsg stream (the reference keeps one closure per component:
 * os/kmsg_matcher.go:159, memory/kmsg_matcher.go:29); feed it the hits of every GPUD_SCAN_EXT_MATCHERS scan of that stream in
 * scan order together with the scanned buffer and the scan's n_units.  Events come out exactly where the reference's
 * Match returns them: (component, eventName, message) at unit_index (index inside this scan; a kernel-panic fallback event
 * belongs to the 10th line after the panic start whatever that line holds).  State carries over to the next feed. */
typedef struct gpud_kmsg_stateful gpud_kmsg_stateful;
typedef struct {
  int64_t unit_index;      /* line / record of THIS scan the event is returned for; negative = a line of an earlier scan */
  char component[16];      /* "os" | "memory" */
  char event[32];          /* "kernel_panic" | "OOM" */
  char message[440];
} gpud_kmsg_event;
int32_t gpud_kmsg_stateful_create(gpud_kmsg_stateful** out);
void gpud_kmsg_stateful_destroy(gpud_kmsg_stateful* st);
int32_t gpud_kmsg_stateful_feed(gpud_kmsg_stateful* st, const gpud_xid_hit* hits, int64_t n_hits, const uint8_t* buf, int64_t n_units,
                                gpud_kmsg_event* out, int32_t cap, int32_t* n_out);
/* The kmsg watcher hands a message to the matchers only the first time its (minute, message) key shows up within the cache TTL
 * (pkg/kmsg/watcher.go:281-286, deduper.go:63-125).  gpud_kmsg_dedup_units marks the units of a scanned buffer the watcher would have
 * skipped (dropped[u] = 1); `deduper` is the cache, kept across calls (gpud_kmsg_deduper_create: ttl 0 = the reference's 15 min,
 * truncate 0 = 60 s).  RAW_KMSG units are timed boot_unix + usec, LINES units all carry lines_unix.  gpud_kmsg_stateful_feed_units is
 * gpud_kmsg_stateful_feed without those units: a dropped line neither matches nor counts towards the panic matcher's ten lines. */
void* gpud_kmsg_deduper_create(int64_t ttl_seconds, int32_t truncate_seconds);
void gpud_kmsg_deduper_destroy(void* deduper);
int32_t gpud_kmsg_dedup_units(void* deduper, const uint8_t* buf, int64_t len, int32_t mode, int64_t boot_unix, int64_t lines_unix, int64_t now_unix,
                              uint8_t* dropped, int64_t n_units, int64_t* n_dropped);
int32_t gpud_kmsg_stateful_feed_units(gpud_kmsg_stateful* st, const gpud_xid_hit* hits, int64_t n_hits, const uint8_t* buf, int64_t n_units,
                                      const uint8_t* dropped, gpud_kmsg_event* out, int32_t cap, int32_t* n_out);

/* Write path into the reference's SQLite stores (SURVEY.md 8f.2): the same tables, columns, indexes and statements as
 * pkg/eventstore/database.go:136-143,198-275 and pkg/metrics/store/sqlite.go:87-164, so gpud's /v1/events and /v1/metrics
 * readers work on them unchanged.  SQLite is dlopen'ed (GPUD_E_UNSUPPORTED without libsqlite3.so.0). */
typedef struct gpud_store gpud_store;
typedef struct { int64_t unix_ms; const char* component; const char* name; const char* labels_json; double value; } gpud_metric;
int32_t gpud_store_open(const char* path, gpud_store** out);
void gpud_store_close(gpud_store* st);
int32_t gpud_store_last_error(gpud_store* st, char* out, int32_t cap);
/* Bucket(component): creates "components_<name>_events_v0_5_0" (+ its three indexes) and returns the table name. */
int32_t gpud_store_event_table(gpud_store* st, const char* component, char* table_out, int32_t cap);
int32_t gpud_store_insert_event(gpud_store* st, const char* table, int64_t unix_s, const char* name, const char* type, const char* message,
                                const char* extra_info_json);
/* Bucket.Find (database.go:277-324): *found = 1 when a row of the same (timestamp, name, type[, message if non-empty]) carries an
 * equal ExtraInfo map (compareEvent :459-469; NULL / "" / "null" = no map).  extra_info_json: one JSON object of string values. */
int32_t gpud_store_find_event(gpud_store* st, const char* table, int64_t unix_s, const char* name, const char* type, const char* message,
                              const char* extra_info_json, int32_t* found);
/* The read side of a Bucket (eventstore/types.go:54-66): Get = rows with timestamp > since, newest first (database.go:327-365);
 * Latest (:367-384); Purge = delete rows with timestamp < before (:449-457).  A row's message and extra_info text live in the
 * caller's `text` arena at [off, off+len) (NUL-terminated); a stored extra_info that is not a JSON object of strings fails the call
 * like scanRows does.  GPUD_E_CAPACITY when rows or text do not fit (*n_rows = the rows that did). */
typedef struct { int64_t unix_s; char name[64]; char type[16]; int32_t message_off, message_len, extra_off, extra_len; } gpud_event_row;
int32_t gpud_store_get_events(gpud_store* st, const char* table, int64_t since_unix, gpud_event_row* rows, int32_t cap_rows, char* text, int32_t cap_text,
                              int32_t* n_rows);
int32_t gpud_store_latest_event(gpud_store* st, const char* table, gpud_event_row* row, char* text, int32_t cap_text, int32_t* found);
int32_t gpud_store_purge_events(gpud_store* st, const char* table, int64_t before_unix, int32_t* n_purged);
/* updateCurrentState of the xid / sxid components (xid/component.go:581-611, sxid/component.go:478-507) over the stores: the component's
 * events and the "reboot" events of the os bucket (os_table = gpud_store_event_table(st, "os"), pkg/host/event.go:15-17; NULL = none)
 * since now - lookback_seconds (default eventstore.DefaultRetention = 3 days), cut at the newest SetHealthy, merged newest first and
 * folded by evolveHealthyState (xid/health_state.go:57-128, sxid/health_state.go:38-111).  *health 0 Healthy / 1 Degraded / 2 Unhealthy,
 * *action the first suggested GPUD_ACT_* (0 = none), reason as the reference words it.  devices = "uuid=pci_bus_id;..." for the UUID
 * in the xid reason (NULL = none). */
int32_t gpud_xid_state_from_store(gpud_store* st, const char* xid_table, const char* os_table, int64_t now_unix, int64_t lookback_seconds, int32_t reboot_threshold,
                                  const char* devices, int32_t* health, int32_t* action, char* reason, int32_t cap);
int32_t gpud_sxid_state_from_store(gpud_store* st, const char* sxid_table, const char* os_table, int64_t now_unix, int64_t lookback_seconds, int32_t* health,
                                   int32_t* action, char* reason, int32_t cap);
/* RebootEventStore.RecordReboot (pkg/host/event.go:85-132) into the os bucket: Event{boot time, "reboot", "Warning", "system reboot detected
 * <time>"} unless the boot is older than 3 days, already stored, older than the latest stored event, or within a minute after it. */
int32_t gpud_store_record_reboot(gpud_store* st, const char* os_table, int64_t now_unix, int64_t boot_unix, int32_t* inserted);
/* The xid component's persist loop (xid/component.go:468-577) for the hits of one scan: "error_xid" events, duplicates skipped. */
int32_t gpud_store_insert_xid_hits(gpud_store* st, const char* table, const gpud_xid_hit* hits, int64_t n, int64_t fallback_unix,
                                   int64_t boot_unix, int32_t raw_kmsg, int32_t* n_inserted);
/* The sxid component's persist step (sxid/component.go:433-469) for the SXid hits of one scan: "error_sxid" events with an empty type,
 * extra_info {"data": "<decimal code>", "device_uuid": device}, duplicates skipped.  Resolved on read by resolveSXIDEvent. */
int32_t gpud_store_insert_sxid_hits(gpud_store* st, const char* table, const gpud_xid_hit* hits, int64_t n, int64_t fallback_unix,
                                    int64_t boot_unix, int32_t raw_kmsg, int32_t* n_inserted);
/* hw-slowdown's persist step (hw-slowdown/component.go:294-343): Event{unix_s, "hw_slowdown", "Warning", HWSlowdownEvent message,
 * {"data_source": "nvml", "gpu_uuid": uuid}} unless the reading has no hardware-slowdown reason or the event is already stored. */
int32_t gpud_store_insert_hw_slowdown(gpud_store* st, const char* table, int64_t unix_s, uint64_t bitmask, const char* gpu_uuid, int32_t* inserted);
/* The pkg/kmsg Syncer step (syncer.go:73-143) for the hits of RAW_KMSG + GPUD_SCAN_EXT_MATCHERS scans: `component` names the
 * event table (e.g. "disk" -> components_disk_events_v0_5_0), `kmsg_component` selects the line matchers
 * (gpud_kmsg_component()); per record the component's first firing pattern becomes Event{boot + usec, name, message, "Warning"},
 * goes through the parsed-message dedup (60 s buckets, 15 min TTL against `now_unix`) and the store's duplicate check, and is
 * inserted.  One syncer per (component, kmsg stream); its dedup cache carries over between feeds. */
typedef struct gpud_kmsg_syncer gpud_kmsg_syncer;
/* One clause of a kmsg.EventDedupWindowFunc (pkg/kmsg/deduper.go:26,49-56) as data: an event whose name equals `event` and whose
 * message contains `message_contains` ("" = any) is coalesced over `window_seconds` (bucket width and cache TTL, syncer.go:145-155);
 * the first matching rule decides, window_seconds <= 0 = "not configured" for that event. */
typedef struct { char event[32]; char message_contains[32]; int64_t window_seconds; } gpud_dedup_rule;
int32_t gpud_kmsg_syncer_create(gpud_store* st, const char* component, gpud_kmsg_syncer** out);
void gpud_kmsg_syncer_destroy(gpud_kmsg_syncer* sy);
/* kmsg.WithCacheKeyTruncateSeconds (<= 0 keeps 60), withDisableDedup, WithEventDedupWindowFunc (rules copied). */
int32_t gpud_kmsg_syncer_configure(gpud_kmsg_syncer* sy, int32_t truncate_seconds, int32_t disable_dedup, const gpud_dedup_rule* rules, int32_t n_rules);
/* The options the reference's own component passes to kmsg.NewSyncer: "infiniband" (5 min; access_reg_failed 24 h per PCI device,
 * infiniband/component.go:149-179), "peermem", "disk" (5 min), "nccl", "os", "cpu", "memory" (defaults). */
int32_t gpud_kmsg_syncer_configure_component(gpud_kmsg_syncer* sy, const char* kmsg_component);
/* The loop body of Syncer.sync (syncer.go:84-140) for ONE event a matcher produced -- the entry for the events of the stateful
 * matchers (gpud_kmsg_stateful_feed) and for callers with their own MatchFunc: parsed dedup, Find, Insert as type "Warning". */
int32_t gpud_kmsg_syncer_offer(gpud_kmsg_syncer* sy, int64_t unix_s, const char* name, const char* message, int64_t now_unix, int32_t* inserted);
int32_t gpud_kmsg_syncer_feed(gpud_kmsg_syncer* sy, const char* kmsg_component, const gpud_xid_hit* hits, int64_t n, const uint8_t* buf,
                              int64_t boot_unix, int64_t now_unix, int32_t* n_inserted);
/* table NULL or "" = "gpud_metrics_v0_5" (metrics/store/sqlite.go:36) */
int32_t gpud_store_metrics_table(gpud_store* st, const char* table);
int32_t gpud_store_record_metrics(gpud_store* st, const char* table, const gpud_metric* ms, int64_t n);
/* purge (metrics/store/sqlite.go:258-275): DELETE the rows with unix_milliseconds < before_unix_ms; the reference Syncer runs it on its
 * own ticker (syncer.go:55-71) so that a table fed every tick does not grow without bound. */
int32_t gpud_store_purge_metrics(gpud_store* st, const char* table, int64_t before_unix_ms, int64_t* n_purged);
/* Name of a drained window aggregate: "<field>_window_<op>", op = min | max | mean | ema | p<Q> | n_over (GPUD_OP_*), Q = printf("%g",
 * 100 q_num / q_den) with '.' -> '_' (99/100 -> p99, 999/1000 -> p99_9: Prometheus names have no '.').  Returns the length, -1 if cap
 * is too small. */
int32_t gpud_window_metric_name(const char* field, int32_t op, int32_t q_num, int32_t q_den, char* out, int32_t cap);
/* The Syncer's sync step (syncer.go:76-82) over a ring: gpud_ring_drain, then one metrics row (store/sqlite.go:108-164, INSERT OR
 * REPLACE) per returned window x field whose field_names[f] is not NULL x op of ops_mask (bit GPUD_OP_*; 0 = all six):
 * component_name components[f], metric_name gpud_window_metric_name(field_names[f], ...), metric_labels labels_json (rendered like
 * json.Marshal: sorted keys, no spaces; "" = none), metric_value (n_over as REAL), unix_milliseconds the window's end time.  A window
 * without a time fails the call with GPUD_E_STATE.  A window whose time is not after the previous exported window of this ring is
 * written 1 ms after it (counted in *n_shifted), so that two windows never share a primary key.  Atomic: all rows in one transaction,
 * and the ring's cursor and EMA state advance only after COMMIT; on any failure the store, the cursor and the EMA are as they were and
 * the next call returns the same windows.  *n_rows = rows written. */
int32_t gpud_ring_drain_to_store(gpud_ring* ring, gpud_store* st, const char* table, const char* const* components, const char* const* field_names,
                                 const char* labels_json, uint32_t ops_mask, int64_t max_windows, gpud_drain_info* info, int64_t* n_rows, int64_t* n_shifted);
/* temperature component only: while a store is attached (st = NULL detaches), every Check drains each GPU's ring into `table` right
 * after the poll, with all six ops, labels {"uuid":"<uuid>"} and the reference gauges' names (INTEGRATION.md).  A failed drain leaves
 * the Check result alone, as the reference Syncer only logs; the message goes to gpud_last_error and the windows stay for the next
 * tick.  GPUD_E_INVALID for other components. */
int32_t gpud_component_set_metrics_store(gpud_component* c, gpud_store* st, const char* table);

/* InfiniBand port drop / flap scans (SURVEY.md 8f.4): findDrops / findFlaps of
 * components/accelerator/nvidia/infiniband/store/scan_drops.go:41-116 and scan_flaps.go:47-134 over many (device, port)
 * snapshot series at once.  snaps = the series back to back, each in ascending time; series s is
 * snaps[series_off[s] .. series_off[s+1]).  `down` = (state != "active").  ts and the thresholds share one unit (the
 * store keeps unix seconds; defaults 4 min drop, scan_drops.go:11).  One verdict per series. */
typedef struct { int64_t ts; uint64_t total_link_downed; int32_t down; int32_t pad; } gpud_ib_snapshot;
typedef struct {
  int32_t drop, flap;          /* 1 = the reference returns a drop / flap event for this series                       */
  int64_t drop_down_since;     /* ts of the oldest snapshot of the trailing down run ("... down since %s")             */
  int64_t drop_index;          /* index (in the series) of the snapshot returned with the event: the latest one      */
  int64_t flap_down_since;     /* ts of down1 of the revert that reached the threshold                                 */
  int64_t flap_index;          /* index of that revert-to-active snapshot                                              */
  int64_t n_reverts;           /* persistent-down -> active reverts in the series                                      */
} gpud_ib_verdict;
int32_t gpud_ib_scan(gpud_ctx* ctx, int32_t dev, const gpud_ib_snapshot* snaps, const int64_t* series_off, int64_t n_series,
                     int64_t drop_threshold, int64_t flap_down_interval, int32_t flap_back_to_active_threshold, gpud_ib_verdict* out);
/* "%s port %d down since %s" / "... (and flapped back to active)" with the RFC3339 UTC time (scan_drops.go:112, scan_flaps.go:67). */
int32_t gpud_ib_reason(const char* device, uint32_t port, int64_t down_since_unix_s, int32_t flap, char* out, int32_t cap);


/* ------------------------------------------------------------------------------------------------
 * Whole-box NVLink / fabric view.
 * Replaces: the single-process loops of nvlink.Check (nvlink/component.go:164-311),
 * evaluateHealthStateWithThresholds (nvlink/evaluate_threshold.go:77-188) and collectFabricState /
 * FabricState.GetIssues (fabric-manager/fabric_state.go:67-113, pkg/nvidia/nvml/device/fabric_state.go:115-177)
 * with: per-GPU pack kernel -> allgather of one 128-byte record per GPU over NVLink -> replicated verdict kernel.
 * ---------------------------------------------------------------------------------------------- */
#define GPUD_MAX_LINKS 18 /* NVML_NVLINK_MAX_LINKS, nvml.h:389 */
#define GPUD_MAX_GPUS 16
#define GPUD_P2P_UNPROBED 0xFF

typedef struct { /* what the host poller read from NVML for ONE GPU (nvlink/nvlink.go:93-168, p2p.go:21-50) */
  uint32_t gpu_index;                     /* position in the sorted-UUID order (component.go:185-190)      */
  uint32_t nvlink_supported;              /* NVLink.Supported                                              */
  uint32_t system_expected_nvlink;        /* FabricManagerSupported() || FabricStateSupported()            */
  uint32_t n_links;                       /* len(States)                                                   */
  uint8_t link_feature_enabled[GPUD_MAX_LINKS];
  uint8_t pad0[2];
  uint64_t link_replay_errors[GPUD_MAX_LINKS];
  uint64_t link_recovery_errors[GPUD_MAX_LINKS];
  uint64_t link_crc_errors[GPUD_MAX_LINKS];
  uint8_t p2p_status[GPUD_MAX_GPUS];      /* NVML P2P status vs peer j (0 OK .. 6 UNKNOWN), GPUD_P2P_UNPROBED */
  uint32_t fabric_valid;                  /* fabric info was read                                          */
  uint8_t fabric_state;                   /* nvml.h:3433-3436; 3 = COMPLETED                               */
  uint8_t fabric_summary;                 /* 0 NOT_SUPPORTED 1 HEALTHY 2 UNHEALTHY 3 LIMITED_CAPACITY       */
  uint8_t pad1[2];
  int32_t fabric_status;                  /* nvml.Return, 0 = SUCCESS                                      */
  uint32_t fabric_health_mask;            /* nvml.h:3453-3488                                              */
  uint32_t clique_id;
} gpud_fabric_raw;

typedef struct { /* the 128-byte record each GPU contributes to the allgather */
  uint32_t gpu_index;
  uint32_t flags;              /* bit0 nvlink_supported, bit1 system_expected_nvlink, bit2 fabric_valid,
                                  bit3 all-links-feature-enabled && n_links > 0 ("active", component.go:281) */
  uint32_t n_links;
  uint32_t links_enabled_mask;
  uint64_t replay_errors, recovery_errors, crc_errors; /* NVLinkStates.Total*Errors, nvlink.go:44-68       */
  uint8_t p2p_status[GPUD_MAX_GPUS];
  uint8_t fabric_state, fabric_summary, fabric_issue_bits, pad0;
  int32_t fabric_status;
  uint32_t fabric_health_mask;
  uint32_t clique_id;
  uint8_t pad1[128 - 76];
} gpud_fabric_local;

enum { GPUD_NVLINK_NO_ISSUE = 0, GPUD_NVLINK_P2P_FAILURE = 1, GPUD_NVLINK_NO_ACTIVE_LINKS = 2,
       GPUD_NVLINK_THRESHOLD_SATISFIED = 3, GPUD_NVLINK_THRESHOLD_VIOLATED = 4, GPUD_NVLINK_NO_THRESHOLD = 5,
       GPUD_NVLINK_NO_DATA = 6, GPUD_NVLINK_P2P_INCOMPLETE_NO_THRESHOLD = 7 };
/* fabric_issue_bits: */
#define GPUD_FAB_STATE_NOT_COMPLETED 0x01u
#define GPUD_FAB_STATUS_NOT_SUCCESS 0x02u
#define GPUD_FAB_SUMMARY_UNHEALTHY 0x04u
#define GPUD_FAB_SUMMARY_LIMITED 0x08u
#define GPUD_FAB_BW_DEGRADED 0x10u
#define GPUD_FAB_ROUTE_RECOVERY 0x20u
#define GPUD_FAB_ROUTE_UNHEALTHY 0x40u
#define GPUD_FAB_ACCESS_TIMEOUT 0x80u

/* FabricState.GetIssues (pkg/nvidia/nvml/device/fabric_state.go:115-177) of one GPU's record as text: the sorted issue
 * strings joined with ", " ("" = healthy or no fabric info).  Returns the length, -1 if cap is too small. */
int32_t gpud_fabric_issues(const gpud_fabric_raw* gpu, char* out, int32_t cap);
/* Where the text of an NVML status comes from ("status=<text>" above is nvml.Return.Error()): NULL, the default, gives go-nvml's constant
 * names ("ERROR_UNKNOWN"), which is what the reference prints while libnvidia-ml is not loaded (its unit tests); a daemon that has NVML
 * loaded prints nvmlErrorString's text -- pass that function (or call gpud_nvml_error_strings_from_driver, which installs the dlopen'ed
 * one; GPUD_E_UNSUPPORTED without a driver library). */
typedef const char* (*gpud_nvml_error_string_fn)(int32_t nvml_return);
void gpud_set_nvml_error_string(gpud_nvml_error_string_fn fn);
int32_t gpud_nvml_error_strings_from_driver(void);

typedef struct {
  int32_t n_gpus;
  int32_t nvlink_health;  /* 0 Healthy, 2 Unhealthy (api/v1/types.go:20-25)                                 */
  int32_t nvlink_reason;  /* GPUD_NVLINK_*                                                                  */
  int32_t required, active, inactive, unsupported;
  int32_t p2p_expected_pairs, p2p_probed_pairs, p2p_ok_pairs;
  uint32_t p2p_ok_gpu_mask;       /* PeerNVLinkOKGPUUUIDs as a bit per gpu_index                            */
  uint32_t p2p_observed_status_mask; /* bit s set if status code s was observed                             */
  uint32_t active_mask, inactive_mask, unsupported_mask;
  int32_t fabric_healthy;         /* report.Healthy, fabric_state.go:67-113                                 */
  uint32_t fabric_unhealthy_gpu_mask;
  uint8_t fabric_issue_bits[GPUD_MAX_GPUS];
  uint64_t total_replay, total_recovery, total_crc;
} gpud_fabric_verdict;
/* The host poller's side of the record (SURVEY.md 8a rows A3/A13): GetNVLink (nvlink/nvlink.go:93-168: per-link FEATURE_ENABLED and the
 * DL replay / recovery / CRC-flit counters; NOT_SUPPORTED on link 0 = no NVLink, later = fewer links), the V3 fabric info
 * (pkg/nvidia/nvml/device/fabric_state.go:268-306), SystemExpectedNVLink from the product name, and the NVLink P2P status against
 * each peer (nvlink/p2p.go:21-50; peer_bus_ids[j] = PCI bus id of gpu_index j, NULL / "" entries and j == gpu_index are skipped).
 * GPUD_E_STATE with "GPU lost" / "GPU requires reset" in gpud_last_error mirrors nvmlerrors.ErrGPULost / ErrGPURequiresReset. */
int32_t gpud_poller_fabric_raw(gpud_poller* poller, uint32_t gpu_index, const char* const* peer_bus_ids, int32_t n_peers, gpud_fabric_raw* out);
int32_t gpud_poller_product_name(gpud_poller* poller, char* out, int32_t cap);   /* nvmlDeviceGetName */
/* Does this (unhealthy) verdict carry RepairActionTypeRebootSystem?  setNVLinkSuggestedActions, nvlink/evaluate_threshold.go:37-52:
 * a GPU with inactive links, or complete P2P coverage with no OK pair and a status outside the five "not supported" codes. */
int32_t gpud_fabric_suggest_reboot(const gpud_fabric_verdict* v);
/* The nvlink check result's reason for a verdict, as the reference words it (nvlink/evaluate_threshold.go:11-35,77-188; the
 * no-issue text of component.go:307): gpu_uuids[i] names gpu_index i in the "inactive nvlinks=" / "unsupported nvlinks=" lists
 * (NULL or short: "GPU-<i>").  Returns the length, -1 if it does not fit. */
int32_t gpud_fabric_reason(const gpud_fabric_verdict* v, const char* const* gpu_uuids, int32_t n_uuids, char* out, int32_t cap);
/* collectFabricState's report (fabric-manager/fabric_state.go:67-113) over the box's records: *healthy, and the reason
 * "GPU <uuid>: <issues>" per affected GPU, sorted, joined by "; " ("" when healthy).  Returns the length, -1 if it does not fit. */
int32_t gpud_fabric_report_reason(const gpud_fabric_raw* gpus, const char* const* gpu_uuids, int32_t n, int32_t* healthy, char* out, int32_t cap);

/* Single-rank pieces (one process per GPU; the collective itself is done by the host plumbing, e.g.
 * torch.distributed / ncclAllGather on `dev_send` -> `dev_all`): */
int32_t gpud_fabric_pack(gpud_ctx* ctx, int32_t dev, const gpud_fabric_raw* raw, void* dev_send /*128 B*/, void* cuda_stream);
int32_t gpud_fabric_verdict_device(gpud_ctx* ctx, int32_t dev, const void* dev_all /*[n]x128 B*/, int32_t n,
                                   int32_t at_least_gpus_with_all_links, gpud_fabric_verdict* out, void* cuda_stream);
/* All-in-one for a process that owns the communicator: NCCL is dlopen'ed (libnccl.so.2) on first use. */
int32_t gpud_comm_unique_id(void* out128);
int32_t gpud_comm_init(gpud_ctx* ctx, int32_t dev, int32_t n_ranks, int32_t rank, const void* unique_id128);
int32_t gpud_fabric_gather(gpud_ctx* ctx, int32_t dev, const gpud_fabric_raw* raw, int32_t at_least_gpus_with_all_links,
                           gpud_fabric_local* all_out /*[n_ranks] host*/, gpud_fabric_verdict* out);
/* Single-process multi-GPU (the reference's own deployment shape): every device of the ctx packs its record and
 * writes it straight into every peer's table over NVLink peer stores (no NCCL), then each evaluates the verdict. */
int32_t gpud_fabric_gather_p2p(gpud_ctx* ctx, const gpud_fabric_raw* raws /*[n devs]*/, int32_t at_least_gpus_with_all_links,
                               gpud_fabric_local* all_out /*[n] host*/, gpud_fabric_verdict* verdicts /*[n]*/);

#ifdef __cplusplus
}
#endif
#endif /* GPUD_B200_H */
