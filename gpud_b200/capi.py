"""ctypes binding of include/gpud_b200.h (the same surface a cgo shim binds; see INTEGRATION.md)."""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GPUD_B200_LIB") or os.path.join(_HERE, "libgpud_b200.so")   # override: kernel-variant experiments only

OPS = {"min": 0, "max": 1, "mean": 2, "ema": 3, "p99": 4, "n_over": 5}
EVENT_NAMES = ["Unknown", "Info", "Warning", "Critical", "Fatal"]
ACTION_WIRE = {1: "IGNORE_NO_ACTION_REQUIRED", 2: "REBOOT_SYSTEM", 3: "HARDWARE_INSPECTION", 4: "CHECK_USER_APP_AND_GPU"}
SCAN_LINES, SCAN_RAW_KMSG = 0, 1
SCAN_EXT_MATCHERS = 0x100
DTYPES = {"float64": 0, "uint32": 1, "int32": 2, "float32": 3, "int64": 4, "uint64": 5, "uint16": 6, "int16": 7, "uint8": 8}   # GPUD_DT_*
MAX_LINKS, MAX_GPUS = 18, 16


class GpudError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("gpud_b200 error %d: %s" % (code, msg))
        self.code = code


class RingCfg(C.Structure):
    _fields_ = [("n_fields", C.c_int32), ("window", C.c_int32), ("capacity", C.c_int64), ("ema_alpha", C.c_double),
                ("q_num", C.c_int32), ("q_den", C.c_int32), ("thresholds", C.POINTER(C.c_double))]


class XidHit(C.Structure):
    _fields_ = [("unit_index", C.c_int64), ("unit_offset", C.c_int64), ("dev_off", C.c_int64), ("dev_len", C.c_int32),
                ("kind", C.c_int32), ("code", C.c_int32), ("flags", C.c_uint32), ("sub_code", C.c_int32),
                ("kmsg_priority", C.c_int32), ("kmsg_seq", C.c_int64), ("kmsg_usec", C.c_int64), ("link", C.c_int64),
                ("intrinfo", C.c_uint32), ("error_status", C.c_uint32), ("extra", C.c_uint32 * 4), ("n_extra", C.c_int32),
                ("severity_fatal", C.c_int32), ("xc", C.c_int32), ("unit_name_off", C.c_int64), ("unit_name_len", C.c_int32),
                ("pid_off", C.c_int64), ("pid_len", C.c_int32), ("pname_off", C.c_int64), ("pname_len", C.c_int32),
                ("inj_off", C.c_int64), ("inj_len", C.c_int32), ("event_type", C.c_int32), ("n_actions", C.c_int32),
                ("actions", C.c_int32 * 4), ("rule_index", C.c_int32), ("detail_variant", C.c_int32),
                ("device", C.c_char * 40), ("unit_name", C.c_char * 40)]

    def as_dict(self) -> dict:
        na = self.n_actions
        return {"line": self.unit_index, "offset": self.unit_offset, "kind": self.kind, "code": self.code,
                "device": self.device.decode("latin-1"), "event_type": self.event_type,
                "actions": [self.actions[i] for i in range(max(na, 0))], "actions_nil": na < 0,
                "extended": bool(self.flags & 1), "sub_code": self.sub_code, "unit": self.unit_name.decode("latin-1"),
                "error_status": self.error_status, "intrinfo": self.intrinfo, "link": self.link,
                "rule_index": self.rule_index, "variant": self.detail_variant, "flags": self.flags,
                "extra": [self.extra[i] for i in range(self.n_extra)], "severity_fatal": self.severity_fatal, "xc": self.xc,
                "kmsg": (self.kmsg_priority, self.kmsg_seq, self.kmsg_usec)}


class Metric(C.Structure):
    _fields_ = [("unix_ms", C.c_int64), ("component", C.c_char_p), ("name", C.c_char_p), ("labels_json", C.c_char_p), ("value", C.c_double)]


class DrainInfo(C.Structure):
    _fields_ = [("first_window", C.c_int64), ("n_windows", C.c_int64), ("n_lost", C.c_int64), ("n_pending", C.c_int64)]

    def as_dict(self) -> dict:
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


def window_metric_name(field: str, op: str, q_num: int = 99, q_den: int = 100) -> str:
    """gpud_window_metric_name: "<field>_window_<op>" (op one of OPS; the order statistic is named p<Q>)"""
    out = C.create_string_buffer(512)
    n = lib().gpud_window_metric_name(field.encode(), OPS[op], q_num, q_den, out, 512)
    if n < 0:
        raise GpudError(n, "gpud_window_metric_name")
    return out.value.decode()


def hw_slowdown_event_message(bitmask: int, gpu_uuid: str) -> str:
    buf = C.create_string_buffer(2048)
    n = lib().gpud_hw_slowdown_event_message(bitmask, gpu_uuid.encode(), buf, 2048)
    if n < 0:
        raise GpudError(n, "gpud_hw_slowdown_event_message")
    return buf.value.decode()


def hw_slowdown_check(event_unix, now_unix: int, window_seconds: int = 600, threshold_per_minute: float = 0.6):
    """-> (health 0/2, freq per minute, hardware_inspection, reason)"""
    arr = (C.c_int64 * max(1, len(event_unix)))(*event_unix)
    h, insp, freq = C.c_int32(), C.c_int32(), C.c_double()
    buf = C.create_string_buffer(512)
    rc = lib().gpud_hw_slowdown_check(arr, len(event_unix), now_unix, window_seconds, threshold_per_minute, C.byref(h), C.byref(freq), C.byref(insp), buf, 512)
    if rc:
        raise GpudError(rc, "gpud_hw_slowdown_check")
    return h.value, freq.value, bool(insp.value), buf.value.decode()


def fabric_reason(verdict, gpu_uuids=()) -> str:
    arr = (C.c_char_p * max(1, len(gpu_uuids)))(*[u.encode() for u in gpu_uuids])
    buf = C.create_string_buffer(2048)
    n = lib().gpud_fabric_reason(C.byref(verdict), arr, len(gpu_uuids), buf, 2048)
    if n < 0:
        raise GpudError(n, "gpud_fabric_reason")
    return buf.value.decode()


def fabric_report_reason(raws, gpu_uuids):
    """collectFabricState -> (healthy, reason)"""
    n = len(raws)
    arr = (FabricRaw * max(1, n))(*raws)
    uu = (C.c_char_p * max(1, n))(*[u.encode() for u in gpu_uuids])
    h = C.c_int32()
    buf = C.create_string_buffer(8192)
    rc = lib().gpud_fabric_report_reason(arr, uu, n, C.byref(h), buf, 8192)
    if rc < 0:
        raise GpudError(rc, "gpud_fabric_report_reason")
    return bool(h.value), buf.value.decode()


def xid_detail(xid: int, sub_code: int = 0, error_status: int = 0):
    """getDetailWithSubCodeAndStatus -> None or dict(event_type, actions (None = nil), description, sub_code)"""
    ev, na, var, sc = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
    acts = (C.c_int32 * 4)()
    L = lib()
    if not L.gpud_xid_detail(xid, sub_code, error_status, C.byref(ev), C.byref(na), acts, C.byref(var), C.byref(sc)):
        return None
    return {"event_type": ev.value, "actions": None if na.value < 0 else [acts[i] for i in range(na.value)],
            "description": L.gpud_xid_description(xid, var.value).decode("utf-8"), "sub_code": sc.value}


def xid_build_message(xid: int, sub_code: int = 0, error_status: int = 0, description: str = "", device_uuid: str = "", gpu_uuid: str = "") -> str:
    buf = C.create_string_buffer(1024)
    n = lib().gpud_xid_build_message(xid, sub_code, error_status, description.encode(), device_uuid.encode(), gpu_uuid.encode() if gpu_uuid else None, buf, 1024)
    if n < 0:
        raise GpudError(n, "gpud_xid_build_message")
    return buf.value.decode("utf-8")


def xid_hit_message(hit, gpu_uuid: str = "") -> str:
    buf = C.create_string_buffer(1024)
    n = lib().gpud_xid_hit_message(C.byref(hit), gpu_uuid.encode() if gpu_uuid else None, buf, 1024)
    if n < 0:
        raise GpudError(n, "gpud_xid_hit_message")
    return buf.value.decode("utf-8")


class EventRow(C.Structure):
    _fields_ = [("unix_s", C.c_int64), ("name", C.c_char * 64), ("type", C.c_char * 16), ("message_off", C.c_int32), ("message_len", C.c_int32),
                ("extra_off", C.c_int32), ("extra_len", C.c_int32)]


class DedupRule(C.Structure):
    _fields_ = [("event", C.c_char * 32), ("message_contains", C.c_char * 32), ("window_seconds", C.c_int64)]


class Store:
    """the reference's SQLite event / metrics stores, written by the library (gpud_store_*)"""

    def __init__(self, path: str):
        self._L = lib()
        self._h = C.c_void_p()
        rc = self._L.gpud_store_open(path.encode(), C.byref(self._h))
        if rc:
            raise GpudError(rc, "gpud_store_open")

    def _check(self, rc):
        if rc:
            buf = C.create_string_buffer(512)
            self._L.gpud_store_last_error(self._h, buf, 512)
            raise GpudError(rc, buf.value.decode())

    def event_table(self, component: str) -> str:
        out = C.create_string_buffer(256)
        self._check(self._L.gpud_store_event_table(self._h, component.encode(), out, 256))
        return out.value.decode()

    def insert_event(self, table, unix_s, name, typ, message="", extra_info_json=""):
        self._check(self._L.gpud_store_insert_event(self._h, table.encode(), unix_s, name.encode(), typ.encode(), message.encode(), extra_info_json.encode()))

    def insert_xid_hits(self, table, hits, fallback_unix=0, boot_unix=0, raw_kmsg=False) -> int:
        arr = (XidHit * max(1, len(hits)))(*hits)
        n = C.c_int32()
        self._check(self._L.gpud_store_insert_xid_hits(self._h, table.encode(), arr, len(hits), fallback_unix, boot_unix, 1 if raw_kmsg else 0, C.byref(n)))
        return n.value

    def insert_hw_slowdown(self, table, unix_s: int, bitmask: int, gpu_uuid: str) -> bool:
        f = C.c_int32()
        self._check(self._L.gpud_store_insert_hw_slowdown(self._h, table.encode(), unix_s, bitmask, gpu_uuid.encode(), C.byref(f)))
        return bool(f.value)

    def insert_sxid_hits(self, table, hits, fallback_unix=0, boot_unix=0, raw_kmsg=False) -> int:
        arr = (XidHit * max(1, len(hits)))(*hits)
        n = C.c_int32()
        self._check(self._L.gpud_store_insert_sxid_hits(self._h, table.encode(), arr, len(hits), fallback_unix, boot_unix, 1 if raw_kmsg else 0, C.byref(n)))
        return n.value

    def syncer(self, component: str):
        h = C.c_void_p()
        self._check(self._L.gpud_kmsg_syncer_create(self._h, component.encode(), C.byref(h)))
        return h

    @staticmethod
    def _row(r, text):
        return (r.unix_s, r.name.decode(), r.type.decode(), text[r.message_off:r.message_off + r.message_len].decode("utf-8"),
                text[r.extra_off:r.extra_off + r.extra_len].decode("utf-8"))

    def get_events(self, table, since_unix: int, cap_rows: int = 4096, cap_text: int = 1 << 20):
        """Bucket.Get: (unix_s, name, type, message, extra_info_json) newest first"""
        rows = (EventRow * max(1, cap_rows))()
        text = C.create_string_buffer(cap_text)
        n = C.c_int32()
        self._check(self._L.gpud_store_get_events(self._h, table.encode(), since_unix, rows, cap_rows, text, cap_text, C.byref(n)))
        return [self._row(rows[i], text.raw) for i in range(n.value)]

    def latest_event(self, table):
        row, text, f = EventRow(), C.create_string_buffer(1 << 16), C.c_int32()
        self._check(self._L.gpud_store_latest_event(self._h, table.encode(), C.byref(row), text, 1 << 16, C.byref(f)))
        return self._row(row, text.raw) if f.value else None

    def purge_events(self, table, before_unix: int) -> int:
        n = C.c_int32()
        self._check(self._L.gpud_store_purge_events(self._h, table.encode(), before_unix, C.byref(n)))
        return n.value

    def xid_state(self, xid_table, os_table, now_unix: int, lookback_seconds: int = 3 * 24 * 3600, reboot_threshold: int = 2, devices=None):
        """-> (health 0/1/2, first suggested action id or 0, reason)"""
        h, a, buf = C.c_int32(), C.c_int32(), C.create_string_buffer(2048)
        spec = ";".join("%s=%s" % kv for kv in (devices or {}).items()).encode()
        self._check(self._L.gpud_xid_state_from_store(self._h, xid_table.encode(), os_table.encode() if os_table else None, now_unix, lookback_seconds, reboot_threshold,
                                                      spec, C.byref(h), C.byref(a), buf, 2048))
        return h.value, a.value, buf.value.decode("utf-8")

    def sxid_state(self, sxid_table, os_table, now_unix: int, lookback_seconds: int = 3 * 24 * 3600):
        h, a, buf = C.c_int32(), C.c_int32(), C.create_string_buffer(2048)
        self._check(self._L.gpud_sxid_state_from_store(self._h, sxid_table.encode(), os_table.encode() if os_table else None, now_unix, lookback_seconds,
                                                       C.byref(h), C.byref(a), buf, 2048))
        return h.value, a.value, buf.value.decode("utf-8")

    def record_reboot(self, os_table, now_unix: int, boot_unix: int) -> bool:
        f = C.c_int32()
        self._check(self._L.gpud_store_record_reboot(self._h, os_table.encode(), now_unix, boot_unix, C.byref(f)))
        return bool(f.value)

    def find_event(self, table, unix_s, name, typ, message="", extra_info_json="") -> bool:
        f = C.c_int32()
        self._check(self._L.gpud_store_find_event(self._h, table.encode(), unix_s, name.encode(), typ.encode(), message.encode(), extra_info_json.encode(), C.byref(f)))
        return bool(f.value)

    def syncer_configure(self, sy, truncate_seconds=60, disable_dedup=False, rules=()):
        """rules: (event, message_contains, window_seconds)"""
        arr = (DedupRule * max(1, len(rules)))()
        for i, (ev, sub, win) in enumerate(rules):
            arr[i].event, arr[i].message_contains, arr[i].window_seconds = ev.encode(), sub.encode(), win
        self._check(self._L.gpud_kmsg_syncer_configure(sy, truncate_seconds, 1 if disable_dedup else 0, arr, len(rules)))

    def syncer_configure_component(self, sy, kmsg_component: str):
        self._check(self._L.gpud_kmsg_syncer_configure_component(sy, kmsg_component.encode()))

    def syncer_offer(self, sy, unix_s: int, name: str, message: str, now_unix: int) -> bool:
        f = C.c_int32()
        self._check(self._L.gpud_kmsg_syncer_offer(sy, unix_s, name.encode(), message.encode(), now_unix, C.byref(f)))
        return bool(f.value)

    def syncer_feed(self, sy, kmsg_component: str, hits, buf: bytes, boot_unix: int, now_unix: int) -> int:
        arr = (XidHit * max(1, len(hits)))(*hits)
        n = C.c_int32()
        self._check(self._L.gpud_kmsg_syncer_feed(sy, kmsg_component.encode(), arr, len(hits), C.cast(C.c_char_p(buf), C.c_void_p), boot_unix, now_unix, C.byref(n)))
        return n.value

    def purge_metrics(self, before_unix_ms: int, table: str = "") -> int:
        """purge (metrics/store/sqlite.go:258-275): deletes the rows older than before_unix_ms; returns how many"""
        n = C.c_int64()
        self._check(self._L.gpud_store_purge_metrics(self._h, table.encode(), before_unix_ms, C.byref(n)))
        return n.value

    def metrics_table(self, table: str = ""):
        self._check(self._L.gpud_store_metrics_table(self._h, table.encode()))

    def record_metrics(self, rows, table: str = ""):
        """rows: (unix_ms, component, name, labels_json, value)"""
        arr = (Metric * max(1, len(rows)))()
        keep = []
        for i, (ms, comp, name, labels, val) in enumerate(rows):
            b = (comp.encode(), name.encode(), labels.encode())
            keep.append(b)
            arr[i].unix_ms, arr[i].component, arr[i].name, arr[i].labels_json, arr[i].value = ms, b[0], b[1], b[2], val
        self._check(self._L.gpud_store_record_metrics(self._h, table.encode(), arr, len(rows)))

    def close(self):
        if self._h:
            self._L.gpud_store_close(self._h)
            self._h = None


class IbSnapshot(C.Structure):
    _fields_ = [("ts", C.c_int64), ("total_link_downed", C.c_uint64), ("down", C.c_int32), ("pad", C.c_int32)]


class IbVerdict(C.Structure):
    _fields_ = [("drop", C.c_int32), ("flap", C.c_int32), ("drop_down_since", C.c_int64), ("drop_index", C.c_int64),
                ("flap_down_since", C.c_int64), ("flap_index", C.c_int64), ("n_reverts", C.c_int64)]


def ib_reason(device: str, port: int, down_since: int, flap: bool) -> str:
    out = C.create_string_buffer(256)
    n = lib().gpud_ib_reason(device.encode(), port, down_since, 1 if flap else 0, out, 256)
    if n < 0:
        raise GpudError(n, "gpud_ib_reason")
    return out.value.decode()


POLL_FIELDS = ["temperature_c", "power_mw", "clock_graphics_mhz", "clock_sm_mhz", "clock_mem_mhz", "util_gpu_pct", "util_mem_pct", "memory_used_mib"]


class Temperature(C.Structure):
    _fields_ = [("current_gpu_core_c", C.c_uint32), ("current_hbm_c", C.c_uint32), ("threshold_shutdown_c", C.c_uint32), ("threshold_slowdown_c", C.c_uint32),
                ("threshold_mem_max_c", C.c_uint32), ("threshold_gpu_max_c", C.c_uint32), ("slowdown_margin_c", C.c_int32),
                ("hbm_supported", C.c_uint8), ("margin_supported", C.c_uint8), ("pad", C.c_uint8 * 2)]


class PollCounters(C.Structure):
    _fields_ = [("clock_event_reasons", C.c_uint64), ("ecc_aggregate_corrected", C.c_uint64), ("ecc_aggregate_uncorrected", C.c_uint64),
                ("ecc_volatile_corrected", C.c_uint64), ("ecc_volatile_uncorrected", C.c_uint64), ("clock_events_supported", C.c_uint32),
                ("ecc_read_mask", C.c_uint32)]


def temperature_check(t: "Temperature", margin_threshold_c: int = 0) -> int:
    bits = C.c_int32()
    rc = lib().gpud_temperature_check(C.byref(t), margin_threshold_c, C.byref(bits))
    if rc:
        raise GpudError(rc, "gpud_temperature_check")
    return bits.value


def temperature_reason(readings, gpu_uuids, margin_threshold_c: int = 0):
    """-> (health 0 / 1, reason) of the temperature component over the box's readings"""
    n = len(readings)
    arr = (Temperature * max(1, n))(*readings)
    uu = (C.c_char_p * max(1, n))(*[u.encode() for u in gpu_uuids])
    h = C.c_int32()
    buf = C.create_string_buffer(4096)
    rc = lib().gpud_temperature_reason(arr, uu, n, margin_threshold_c, C.byref(h), buf, 4096)
    if rc < 0:
        raise GpudError(rc, "gpud_temperature_reason")
    return h.value, buf.value.decode("utf-8")


class NvmlDevice(C.Structure):
    _fields_ = [("index", C.c_int32), ("cuda_device", C.c_int32), ("nvml_rc", C.c_int32), ("pad", C.c_int32), ("uuid", C.c_char * 96), ("bus_id", C.c_char * 32),
                ("name", C.c_char * 96)]


class RemappedRows(C.Structure):
    _fields_ = [("remapped_due_to_correctable_errors", C.c_int32), ("remapped_due_to_uncorrectable_errors", C.c_int32), ("remapping_pending", C.c_uint8),
                ("remapping_failed", C.c_uint8), ("supported", C.c_uint8), ("pad", C.c_uint8)]


class EccCounts(C.Structure):
    _fields_ = [("corrected", C.c_uint64), ("uncorrected", C.c_uint64)]


ECC_LOCATIONS = ("total", "l1_cache", "l2_cache", "dram", "sram", "gpu_device_memory", "gpu_texture_memory", "shared_memory", "gpu_register_file")
FIELD_ROW = ("power_instant_mw", "power_average_mw", "memory_temp_c", "total_energy_mj", "ecc_sbe_volatile", "ecc_dbe_volatile", "ecc_sbe_aggregate",
             "ecc_dbe_aggregate", "nvlink_crc_flit_total", "nvlink_crc_data_total", "nvlink_replay_total", "nvlink_recovery_total", "remapped_correctable",
             "remapped_uncorrectable", "remapped_pending", "remapped_failure", "pcie_replay")


class EccErrors(C.Structure):
    _fields_ = [("aggregate", EccCounts * 9), ("volatile_", EccCounts * 9), ("ecc_mode_current", C.c_uint8), ("ecc_mode_pending", C.c_uint8), ("supported", C.c_uint8),
                ("pad", C.c_uint8 * 5)]


GPM_METRICS = ("sm_occupancy", "integer_util", "any_tensor_util", "dfma_tensor_util", "hmma_tensor_util", "imma_tensor_util", "fp64_util", "fp32_util", "fp16_util")
GPM_METRIC_IDS = (3, 4, 5, 6, 7, 9, 11, 12, 13)          # nvml.GPM_METRIC_* of the names above (gpm/component.go:56-64)


class GpmMetrics(C.Structure):
    _fields_ = [("value", C.c_double * 9), ("nvml_rc", C.c_int32 * 9), ("supported", C.c_int32), ("sample_seconds", C.c_double)]

    def as_dict(self):
        return dict(zip(GPM_METRICS, list(self.value)))


def gpm_check(metrics):
    """gpud_gpm_check: (health, reason)"""
    n = len(metrics)
    arr = (GpmMetrics * max(n, 1))(*metrics)
    health = C.c_int32()
    buf = C.create_string_buffer(256)
    k = lib().gpud_gpm_check(arr, n, C.byref(health), buf, 256)
    if k < 0:
        raise GpudError(k, "gpud_gpm_check")
    return health.value, buf.value.decode()


def nvml_devices(cap: int = 16):
    """gpud_nvml_devices: (list of NvmlDevice, driver version)"""
    arr = (NvmlDevice * cap)()
    n = C.c_int32()
    drv = C.create_string_buffer(96)
    rc = lib().gpud_nvml_devices(arr, cap, C.byref(n), drv, 96)
    if rc not in (0, -4):
        raise GpudError(rc, "gpud_nvml_devices")
    return [arr[i] for i in range(min(n.value, cap))], drv.value.decode()


def nvml_devices_arg() -> str:
    buf = C.create_string_buffer(4096)
    rc = lib().gpud_nvml_devices_arg(buf, 4096)
    if rc < 0:
        raise GpudError(rc, "gpud_nvml_devices_arg")
    return buf.value.decode()


def nvml_bus_id(nvml_bus_id_str: str) -> str:
    buf = C.create_string_buffer(64)
    lib().gpud_nvml_bus_id(nvml_bus_id_str.encode(), buf, 64)
    return buf.value.decode()


def remapped_rows_check(rows, bus_ids):
    """gpud_remapped_rows_check: (health, action, reason)"""
    n = len(rows)
    arr = (RemappedRows * max(n, 1))(*rows)
    ids = (C.c_char_p * max(n, 1))(*[b.encode() for b in bus_ids])
    health, action = C.c_int32(), C.c_int32()
    buf = C.create_string_buffer(4096)
    k = lib().gpud_remapped_rows_check(arr, ids, n, C.byref(health), C.byref(action), buf, 4096)
    if k < 0:
        raise GpudError(k, "gpud_remapped_rows_check")
    return health.value, action.value, buf.value.decode()


def poll_row_hold(fresh, nvml_rc, held):
    """gpud_poll_row_hold: the row that goes to the ring when some getters failed; updates `held` in place.  Returns (row, fail_mask)."""
    n = len(fresh)
    f = (C.c_uint32 * n)(*fresh)
    r = (C.c_int32 * n)(*nvml_rc)
    h = (C.c_uint32 * n)(*held)
    out = (C.c_uint32 * n)()
    mask = C.c_uint32()
    rc = lib().gpud_poll_row_hold(f, r, n, h, out, C.byref(mask))
    if rc:
        raise GpudError(rc, "gpud_poll_row_hold")
    held[:] = list(h)
    return list(out), mask.value


class Poller:
    """host NVML poller feeding a ring with raw uint32 poll rows (gpud_poller_*)"""

    def __init__(self, ctx: "Context", ring: "Ring", dev: Optional[int] = None):
        self.ctx, self._L = ctx, ctx._L
        self._h = C.c_void_p()
        dev = ctx.devices[0] if dev is None else dev
        ctx._check(self._L.gpud_poller_create(ctx._h, dev, ring._h, C.byref(self._h)))

    def poll(self, n_polls: int, interval_us: int = 0):
        self.ctx._check(self._L.gpud_poller_poll(self._h, n_polls, interval_us))

    def last_rows(self, cap_rows: int = 1 << 14):
        rows = np.empty((cap_rows, len(POLL_FIELDS)), dtype=np.uint32)
        n, sec = C.c_int64(), C.c_double()
        self.ctx._check(self._L.gpud_poller_last_rows(self._h, C.c_void_p(rows.ctypes.data), cap_rows, C.byref(n), C.byref(sec)))
        return rows[: min(cap_rows, n.value)], sec.value

    def remapped_rows(self) -> "RemappedRows":
        r = RemappedRows()
        self.ctx._check(self._L.gpud_poller_remapped_rows(self._h, C.byref(r)))
        return r

    def ecc_errors(self) -> "EccErrors":
        e = EccErrors()
        self.ctx._check(self._L.gpud_poller_ecc_errors(self._h, C.byref(e)))
        return e

    def gpm_supported(self) -> bool:
        v = C.c_int32()
        self.ctx._check(self._L.gpud_poller_gpm_supported(self._h, C.byref(v)))
        return bool(v.value)

    def gpm_metrics(self, sample_ms: int = 5000) -> "GpmMetrics":
        m = GpmMetrics()
        self.ctx._check(self._L.gpud_poller_gpm_metrics(self._h, sample_ms, C.byref(m)))
        return m

    def poll_gpm(self, ring: "Ring", n_polls: int, sample_ms: int = 5000) -> float:
        sec = C.c_double()
        self.ctx._check(self._L.gpud_poller_poll_gpm(self._h, ring._h, n_polls, sample_ms, C.byref(sec)))
        return sec.value

    def field_row(self):
        """one nvmlDeviceGetFieldValues call: ({name: value}, {name: nvml return code})"""
        v = (C.c_uint64 * len(FIELD_ROW))()
        rc = (C.c_int32 * len(FIELD_ROW))()
        self.ctx._check(self._L.gpud_poller_field_row(self._h, v, rc))
        return dict(zip(FIELD_ROW, list(v))), dict(zip(FIELD_ROW, list(rc)))

    def poll_fields(self, ring: "Ring", n_polls: int, interval_us: int = 0) -> float:
        sec = C.c_double()
        self.ctx._check(self._L.gpud_poller_poll_fields(self._h, ring._h, n_polls, interval_us, C.byref(sec)))
        return sec.value

    def errors(self):
        """(fail_mask, last NVML return code per column, failures per column): getters that failed since create"""
        mask = C.c_uint32()
        rc = (C.c_int32 * len(POLL_FIELDS))()
        nf = (C.c_uint64 * len(POLL_FIELDS))()
        self.ctx._check(self._L.gpud_poller_errors(self._h, C.byref(mask), rc, nf))
        return mask.value, list(rc), list(nf)

    def fabric_raw(self, gpu_index: int = 0, peer_bus_ids=()) -> "FabricRaw":
        """this GPU's NVLink / fabric record read from NVML (GetNVLink, GetFabricState, P2P status against the peers)"""
        raw = FabricRaw()
        arr = (C.c_char_p * max(1, len(peer_bus_ids)))(*[b.encode() if b else None for b in peer_bus_ids])
        self.ctx._check(self._L.gpud_poller_fabric_raw(self._h, gpu_index, arr, len(peer_bus_ids), C.byref(raw)))
        return raw

    def temperature(self) -> "Temperature":
        t = Temperature()
        self.ctx._check(self._L.gpud_poller_temperature(self._h, C.byref(t)))
        return t

    def counters(self) -> "PollCounters":
        c = PollCounters()
        self.ctx._check(self._L.gpud_poller_counters(self._h, C.byref(c)))
        return c

    def product_name(self) -> str:
        buf = C.create_string_buffer(96)
        self.ctx._check(self._L.gpud_poller_product_name(self._h, buf, 96))
        return buf.value.decode()

    def close(self):
        if self._h:
            self._L.gpud_poller_destroy(self._h)
            self._h = None


class KmsgEvent(C.Structure):
    _fields_ = [("unit_index", C.c_int64), ("component", C.c_char * 16), ("event", C.c_char * 32), ("message", C.c_char * 440)]


class KmsgStateful:
    """the reference's two stateful kmsg matchers (os kernel panic, memory OOM) over the primitives of EXT scans"""

    def __init__(self):
        self._L = lib()
        self._h = C.c_void_p()
        if self._L.gpud_kmsg_stateful_create(C.byref(self._h)):
            raise GpudError(-1, "gpud_kmsg_stateful_create")

    def feed(self, hits, buf: bytes, n_units: int, cap: int = 4096):
        arr = (XidHit * max(1, len(hits)))(*hits)
        out = (KmsgEvent * cap)()
        n = C.c_int32()
        rc = self._L.gpud_kmsg_stateful_feed(self._h, arr, len(hits), C.cast(C.c_char_p(buf), C.c_void_p), n_units, out, cap, C.byref(n))
        if rc:
            raise GpudError(rc, "gpud_kmsg_stateful_feed")
        return [(out[i].unit_index, out[i].component.decode(), out[i].event.decode(), out[i].message.decode("latin-1")) for i in range(n.value)]

    def feed_units(self, hits, buf: bytes, n_units: int, dropped: bytes, cap: int = 4096):
        """gpud_kmsg_stateful_feed_units: feed without the units the watcher's dedup dropped (dropped[u] != 0)"""
        arr = (XidHit * max(1, len(hits)))(*hits)
        out = (KmsgEvent * cap)()
        n = C.c_int32()
        rc = self._L.gpud_kmsg_stateful_feed_units(self._h, arr, len(hits), C.cast(C.c_char_p(buf), C.c_void_p), n_units, C.cast(C.c_char_p(dropped), C.c_void_p),
                                                   out, cap, C.byref(n))
        if rc:
            raise GpudError(rc, "gpud_kmsg_stateful_feed_units")
        return [(out[i].unit_index, out[i].component.decode(), out[i].event.decode(), out[i].message.decode("latin-1")) for i in range(n.value)]

    def close(self):
        if self._h:
            self._L.gpud_kmsg_stateful_destroy(self._h)
            self._h = None


class ComponentCfg(C.Structure):
    _fields_ = [("row_remapping_supported", C.c_int32), ("reboot_threshold", C.c_int32), ("margin_threshold_c", C.c_int32), ("nvlink_at_least", C.c_int32)]


class Component:
    """gpud_component_*: the mirror of components.Component (components/types.go:20-66) for the xid / temperature / nvlink paths"""

    def __init__(self, ctx: "Context", name: str, **cfg):
        import json
        self._json = json
        self.ctx, self._L = ctx, ctx._L
        c = ComponentCfg(**cfg)
        self._h = C.c_void_p()
        ctx._check(self._L.gpud_component_create(ctx._h, name.encode(), C.byref(c), C.byref(self._h)))

    def name(self) -> str:
        b = C.create_string_buffer(128)
        self._L.gpud_component_name(self._h, b, 128)
        return b.value.decode()

    def start(self, interval_ms: int):
        self.ctx._check(self._L.gpud_component_start(self._h, interval_ms))

    def check(self):
        health, b = C.c_int32(), C.create_string_buffer(8192)
        self.ctx._check(self._L.gpud_component_check(self._h, C.byref(health), b, 8192))
        return health.value, b.value.decode()

    def last_health_states(self):
        b = C.create_string_buffer(1 << 16)
        n = self._L.gpud_component_last_health_states(self._h, b, 1 << 16)
        if n < 0:
            raise GpudError(n, "gpud_component_last_health_states")
        return self._json.loads(b.value.decode())

    def events(self, since_unix: int = 0):
        b = C.create_string_buffer(1 << 20)
        n = self._L.gpud_component_events(self._h, since_unix, b, 1 << 20)
        if n < 0:
            raise GpudError(n, "gpud_component_events")
        return self._json.loads(b.value.decode())

    def checks(self) -> int:
        return int(self._L.gpud_component_checks(self._h))

    def xid_set_source(self, buf: bytes, raw_kmsg: bool = False, boot_unix: int = 0):
        self.ctx._check(self._L.gpud_component_xid_set_source(self._h, C.cast(C.c_char_p(buf), C.c_void_p), len(buf), int(raw_kmsg), boot_unix))

    def xid_set_healthy(self, now_unix: int):
        self.ctx._check(self._L.gpud_component_xid_set_healthy(self._h, now_unix))

    def xid_add_reboot(self, unix_s: int):
        self.ctx._check(self._L.gpud_component_xid_add_reboot(self._h, unix_s))

    def xid_set_devices(self, devices: str):
        self.ctx._check(self._L.gpud_component_xid_set_devices(self._h, devices.encode()))

    def stop(self):
        """Close(): stops the ticker; the object stays readable"""
        self.ctx._check(self._L.gpud_component_close(self._h))

    def ring_handle(self, slot: int = 0):
        return self._L.gpud_component_ring(self._h, slot)

    def set_metrics_store(self, store: Optional["Store"], table: str = ""):
        """temperature only: drain every GPU's ring into `store` on each Check (None detaches)"""
        self.ctx._check(self._L.gpud_component_set_metrics_store(self._h, store._h if store is not None else None, table.encode()))
        self._store = store                    # the store must outlive the attachment

    def close(self):
        if self._h:
            self._L.gpud_component_close(self._h)
            self._L.gpud_component_destroy(self._h)
            self._h = None


class KmsgDeduper:
    """the kmsg watcher's duplicate drop (pkg/kmsg/watcher.go:281-286) over the units of a scanned buffer"""

    def __init__(self, ttl_seconds: int = 0, truncate_seconds: int = 0):
        self._L = lib()
        self._L.gpud_kmsg_deduper_create.restype = C.c_void_p
        self._h = C.c_void_p(self._L.gpud_kmsg_deduper_create(C.c_int64(ttl_seconds), C.c_int32(truncate_seconds)))

    def units(self, buf: bytes, n_units: int, mode: int = 0, boot_unix: int = 0, lines_unix: int = 0, now_unix: int = 0) -> bytes:
        dropped = C.create_string_buffer(max(1, n_units))
        nd = C.c_int64()
        rc = self._L.gpud_kmsg_dedup_units(self._h, C.cast(C.c_char_p(buf), C.c_void_p), C.c_int64(len(buf)), C.c_int32(mode), C.c_int64(boot_unix), C.c_int64(lines_unix),
                                           C.c_int64(now_unix), dropped, C.c_int64(n_units), C.byref(nd))
        if rc:
            raise GpudError(rc, "gpud_kmsg_dedup_units")
        return dropped.raw[:n_units]

    def close(self):
        if self._h:
            self._L.gpud_kmsg_deduper_destroy(self._h)
            self._h = None


class FabricRaw(C.Structure):
    _fields_ = [("gpu_index", C.c_uint32), ("nvlink_supported", C.c_uint32), ("system_expected_nvlink", C.c_uint32),
                ("n_links", C.c_uint32), ("link_feature_enabled", C.c_uint8 * MAX_LINKS), ("pad0", C.c_uint8 * 2),
                ("link_replay_errors", C.c_uint64 * MAX_LINKS), ("link_recovery_errors", C.c_uint64 * MAX_LINKS),
                ("link_crc_errors", C.c_uint64 * MAX_LINKS), ("p2p_status", C.c_uint8 * MAX_GPUS), ("fabric_valid", C.c_uint32),
                ("fabric_state", C.c_uint8), ("fabric_summary", C.c_uint8), ("pad1", C.c_uint8 * 2), ("fabric_status", C.c_int32),
                ("fabric_health_mask", C.c_uint32), ("clique_id", C.c_uint32)]


class FabricLocal(C.Structure):
    _fields_ = [("gpu_index", C.c_uint32), ("flags", C.c_uint32), ("n_links", C.c_uint32), ("links_enabled_mask", C.c_uint32),
                ("replay_errors", C.c_uint64), ("recovery_errors", C.c_uint64), ("crc_errors", C.c_uint64),
                ("p2p_status", C.c_uint8 * MAX_GPUS), ("fabric_state", C.c_uint8), ("fabric_summary", C.c_uint8),
                ("fabric_issue_bits", C.c_uint8), ("pad0", C.c_uint8), ("fabric_status", C.c_int32),
                ("fabric_health_mask", C.c_uint32), ("clique_id", C.c_uint32), ("pad1", C.c_uint8 * (128 - 76))]


class FabricVerdict(C.Structure):
    _fields_ = [("n_gpus", C.c_int32), ("nvlink_health", C.c_int32), ("nvlink_reason", C.c_int32), ("required", C.c_int32),
                ("active", C.c_int32), ("inactive", C.c_int32), ("unsupported", C.c_int32), ("p2p_expected_pairs", C.c_int32),
                ("p2p_probed_pairs", C.c_int32), ("p2p_ok_pairs", C.c_int32), ("p2p_ok_gpu_mask", C.c_uint32),
                ("p2p_observed_status_mask", C.c_uint32), ("active_mask", C.c_uint32), ("inactive_mask", C.c_uint32),
                ("unsupported_mask", C.c_uint32), ("fabric_healthy", C.c_int32), ("fabric_unhealthy_gpu_mask", C.c_uint32),
                ("fabric_issue_bits", C.c_uint8 * MAX_GPUS), ("total_replay", C.c_uint64), ("total_recovery", C.c_uint64),
                ("total_crc", C.c_uint64)]

    def as_dict(self) -> dict:
        d = {k: getattr(self, k) for k, _ in self._fields_ if k != "fabric_issue_bits"}
        d["fabric_issue_bits"] = list(self.fabric_issue_bits)
        return d


# every symbol include/gpud_b200.h declares (tests check the library exports each one)
SYMBOLS = ["gpud_abi_version", "gpud_sizeof", "gpud_ctx_create", "gpud_ctx_destroy", "gpud_last_error", "gpud_host_alloc",
           "gpud_host_free", "gpud_ring_create", "gpud_ring_destroy", "gpud_ring_set_stream", "gpud_ring_push",
           "gpud_ring_push_device", "gpud_ring_push_raw", "gpud_clock_event_reasons", "gpud_hw_slowdown_event_message", "gpud_hw_slowdown_check", "gpud_store_insert_hw_slowdown", "gpud_store_open", "gpud_store_close", "gpud_store_last_error", "gpud_store_event_table", "gpud_store_insert_event", "gpud_store_insert_xid_hits", "gpud_store_metrics_table", "gpud_store_record_metrics", "gpud_kmsg_syncer_create", "gpud_kmsg_syncer_destroy", "gpud_kmsg_syncer_feed", "gpud_store_find_event", "gpud_store_record_reboot", "gpud_xid_state_from_store", "gpud_sxid_state_from_store", "gpud_store_get_events", "gpud_store_latest_event", "gpud_store_purge_events", "gpud_kmsg_syncer_configure", "gpud_kmsg_syncer_configure_component", "gpud_kmsg_syncer_offer", "gpud_ib_scan", "gpud_ib_reason", "gpud_poller_create", "gpud_poller_destroy", "gpud_poller_poll", "gpud_poller_last_rows", "gpud_poller_errors", "gpud_poll_row_hold", "gpud_nvml_devices", "gpud_nvml_devices_arg", "gpud_nvml_bus_id", "gpud_poller_remapped_rows", "gpud_remapped_rows_check", "gpud_poller_ecc_errors", "gpud_poller_field_row", "gpud_poller_poll_fields", "gpud_poller_gpm_supported", "gpud_poller_gpm_metrics", "gpud_poller_poll_gpm", "gpud_gpm_check", "gpud_poller_fabric_raw", "gpud_poller_product_name", "gpud_poller_temperature", "gpud_temperature_check", "gpud_temperature_reason", "gpud_poller_counters", "gpud_ring_counts", "gpud_ring_reduce", "gpud_ring_sync", "gpud_ring_kernel_ms", "gpud_ring_read",
           "gpud_ring_result_ptr", "gpud_ring_reduce_range", "gpud_ring_range_stats", "gpud_ring_drain", "gpud_ring_push_timed", "gpud_ring_drain_to_store",
           "gpud_store_purge_metrics", "gpud_window_metric_name", "gpud_ring_set_cta_reserve", "gpud_kmsg_scan", "gpud_kmsg_scan_sharded", "gpud_kmsg_scan_device", "gpud_kmsg_scan_kernel_ms", "gpud_kmsg_scan_phase_timing", "gpud_kmsg_scan_stats", "gpud_xid_classify",
           "gpud_hit_detail_json", "gpud_xid_description", "gpud_xid_mnemonic", "gpud_sxid_name", "gpud_nvlink_rule_hint", "gpud_sxid_reason", "gpud_sxid_get_detail", "gpud_store_insert_sxid_hits", "gpud_product_mem_caps", "gpud_product_fm_supported", "gpud_product_fabric_state_supported", "gpud_xid_get_detail", "gpud_xid_detail", "gpud_xid_build_message", "gpud_xid_hit_message", "gpud_xid_device_matches_bus_id", "gpud_kmsg_event_name", "gpud_kmsg_event_message", "gpud_kmsg_component", "gpud_kmsg_hit_message", "gpud_kmsg_stateful_create", "gpud_kmsg_stateful_destroy", "gpud_kmsg_stateful_feed", "gpud_component_create", "gpud_component_destroy", "gpud_component_name", "gpud_component_start", "gpud_component_check", "gpud_component_last_health_states", "gpud_component_events", "gpud_component_close", "gpud_component_checks", "gpud_component_xid_set_source", "gpud_component_xid_set_healthy", "gpud_component_xid_add_reboot", "gpud_component_xid_set_devices", "gpud_component_ring", "gpud_component_set_metrics_store", "gpud_kmsg_stateful_feed_units", "gpud_kmsg_deduper_create", "gpud_kmsg_deduper_destroy", "gpud_kmsg_dedup_units",
           "gpud_fabric_issues", "gpud_fabric_suggest_reboot", "gpud_set_nvml_error_string", "gpud_nvml_error_strings_from_driver", "gpud_fabric_reason", "gpud_fabric_report_reason", "gpud_fabric_pack", "gpud_fabric_verdict_device", "gpud_comm_unique_id", "gpud_comm_init", "gpud_fabric_gather",
           "gpud_fabric_gather_p2p"]

_lib = None


def lib() -> C.CDLL:
    """Load libgpud_b200.so (fails loudly if it has not been built: there is no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GpudError(-2, "%s is missing: build it with `make` (or __graft_entry__.build())" % LIB_PATH)
    L = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    sig = {
        "gpud_abi_version": (i32, []), "gpud_sizeof": (i32, [i32]),
        "gpud_ctx_create": (i32, [C.POINTER(i32), i32, C.POINTER(vp)]), "gpud_ctx_destroy": (i32, [vp]),
        "gpud_last_error": (i32, [vp, C.c_char_p, i32]),
        "gpud_host_alloc": (i32, [i64, C.POINTER(vp)]), "gpud_host_free": (i32, [vp]),
        "gpud_ring_create": (i32, [vp, i32, C.POINTER(RingCfg), C.POINTER(vp)]), "gpud_ring_destroy": (i32, [vp]),
        "gpud_ring_set_stream": (i32, [vp, vp]), "gpud_ring_push": (i32, [vp, vp, i64]), "gpud_ring_push_device": (i32, [vp, vp, i64]), "gpud_ring_push_raw": (i32, [vp, vp, i64, i32]),
        "gpud_clock_event_reasons": (i32, [C.c_uint64, vp, i32, vp, i32, vp]),
        "gpud_store_open": (i32, [C.c_char_p, vp]), "gpud_store_close": (None, [vp]), "gpud_store_last_error": (i32, [vp, vp, i32]),
        "gpud_store_event_table": (i32, [vp, C.c_char_p, vp, i32]),
        "gpud_store_insert_event": (i32, [vp, C.c_char_p, i64, C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p]),
        "gpud_store_insert_xid_hits": (i32, [vp, C.c_char_p, vp, i64, i64, i64, i32, vp]),
        "gpud_kmsg_syncer_create": (i32, [vp, C.c_char_p, vp]), "gpud_kmsg_syncer_destroy": (None, [vp]),
        "gpud_kmsg_syncer_feed": (i32, [vp, C.c_char_p, vp, i64, vp, i64, i64, vp]),
        "gpud_store_get_events": (i32, [vp, C.c_char_p, i64, vp, i32, vp, i32, vp]), "gpud_store_latest_event": (i32, [vp, C.c_char_p, vp, vp, i32, vp]),
        "gpud_store_purge_events": (i32, [vp, C.c_char_p, i64, vp]), "gpud_store_record_reboot": (i32, [vp, C.c_char_p, i64, i64, vp]),
        "gpud_xid_state_from_store": (i32, [vp, C.c_char_p, C.c_char_p, i64, i64, i32, C.c_char_p, vp, vp, vp, i32]),
        "gpud_sxid_state_from_store": (i32, [vp, C.c_char_p, C.c_char_p, i64, i64, vp, vp, vp, i32]),
        "gpud_store_find_event": (i32, [vp, C.c_char_p, i64, C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p, vp]),
        "gpud_kmsg_syncer_configure": (i32, [vp, i32, i32, vp, i32]), "gpud_kmsg_syncer_configure_component": (i32, [vp, C.c_char_p]),
        "gpud_kmsg_syncer_offer": (i32, [vp, i64, C.c_char_p, C.c_char_p, i64, vp]),
        "gpud_store_metrics_table": (i32, [vp, C.c_char_p]), "gpud_store_record_metrics": (i32, [vp, C.c_char_p, vp, i64]),
        "gpud_ib_scan": (i32, [vp, i32, vp, vp, i64, i64, i64, i32, vp]), "gpud_ib_reason": (i32, [C.c_char_p, C.c_uint32, i64, i32, vp, i32]),
        "gpud_poller_create": (i32, [vp, i32, vp, vp]), "gpud_poller_destroy": (None, [vp]), "gpud_poller_poll": (i32, [vp, i64, i64]),
        "gpud_poller_last_rows": (i32, [vp, vp, i64, vp, vp]), "gpud_poller_errors": (i32, [vp, vp, vp, vp]),
        "gpud_poll_row_hold": (i32, [vp, vp, i32, vp, vp, vp]),
        "gpud_nvml_devices": (i32, [vp, i32, vp, vp, i32]), "gpud_nvml_devices_arg": (i32, [vp, i32]), "gpud_nvml_bus_id": (i32, [C.c_char_p, vp, i32]),
        "gpud_poller_remapped_rows": (i32, [vp, vp]), "gpud_remapped_rows_check": (i32, [vp, vp, i32, vp, vp, vp, i32]),
        "gpud_poller_ecc_errors": (i32, [vp, vp]), "gpud_poller_field_row": (i32, [vp, vp, vp]), "gpud_poller_poll_fields": (i32, [vp, vp, i64, i64, vp]),
        "gpud_poller_gpm_supported": (i32, [vp, vp]), "gpud_poller_gpm_metrics": (i32, [vp, i64, vp]), "gpud_poller_poll_gpm": (i32, [vp, vp, i64, i64, vp]),
        "gpud_gpm_check": (i32, [vp, i32, vp, vp, i32]),
        "gpud_poller_temperature": (i32, [vp, C.POINTER(Temperature)]), "gpud_temperature_check": (i32, [C.POINTER(Temperature), i32, vp]),
        "gpud_temperature_reason": (i32, [vp, vp, i32, i32, vp, vp, i32]),
        "gpud_poller_counters": (i32, [vp, C.POINTER(PollCounters)]),
        "gpud_poller_fabric_raw": (i32, [vp, C.c_uint32, vp, i32, C.POINTER(FabricRaw)]), "gpud_poller_product_name": (i32, [vp, vp, i32]),
        "gpud_ring_counts": (i32, [vp, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)]),
        "gpud_ring_reduce": (i32, [vp]), "gpud_ring_sync": (i32, [vp]),
        "gpud_ring_kernel_ms": (i32, [vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]), "gpud_ring_read": (i32, [vp, i32, vp, i64]),
        "gpud_ring_result_ptr": (i32, [vp, i32, C.POINTER(vp)]), "gpud_ring_reduce_range": (i32, [vp, i64, vp, vp]),
        "gpud_ring_set_cta_reserve": (i32, [vp, i32]),
        "gpud_ring_drain": (i32, [vp, i64, vp, vp, vp, C.POINTER(DrainInfo)]), "gpud_ring_push_timed": (i32, [vp, vp, i64, i32, vp]),
        "gpud_ring_drain_to_store": (i32, [vp, vp, C.c_char_p, vp, vp, C.c_char_p, C.c_uint32, i64, C.POINTER(DrainInfo), C.POINTER(i64), C.POINTER(i64)]),
        "gpud_store_purge_metrics": (i32, [vp, C.c_char_p, i64, C.POINTER(i64)]), "gpud_window_metric_name": (i32, [C.c_char_p, i32, i32, i32, vp, i32]),
        "gpud_component_set_metrics_store": (i32, [vp, vp, C.c_char_p]),
        "gpud_ring_range_stats": (i32, [vp, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_int32), vp]),
        "gpud_kmsg_scan": (i32, [vp, i32, vp, i64, i32, C.POINTER(XidHit), i64, C.POINTER(i64), C.POINTER(i64)]),
        "gpud_kmsg_scan_sharded": (i32, [vp, vp, i64, i32, C.POINTER(XidHit), i64, C.POINTER(i64), C.POINTER(i64)]),
        "gpud_kmsg_scan_device": (i32, [vp, i32, vp, i64, i32, C.POINTER(XidHit), i64, C.POINTER(i64), C.POINTER(i64), vp]),
        "gpud_kmsg_scan_kernel_ms": (i32, [vp, i32, C.POINTER(C.c_float)]),
        "gpud_kmsg_scan_phase_timing": (i32, [vp, i32, i32]),
        "gpud_kmsg_scan_stats": (i32, [vp, i32, C.POINTER(i64)]),
        "gpud_xid_classify": (i32, [vp, i32, C.POINTER(XidHit), i64]),
        "gpud_hit_detail_json": (i32, [C.POINTER(XidHit), i64, C.c_char_p, i32]),
        "gpud_xid_description": (C.c_char_p, [i32, i32]), "gpud_xid_mnemonic": (C.c_char_p, [i32]),
        "gpud_sxid_name": (C.c_char_p, [i32]), "gpud_nvlink_rule_hint": (C.c_char_p, [i32]),
        "gpud_sxid_reason": (i32, [i64, C.c_char_p, vp, i32]),
        "gpud_hw_slowdown_event_message": (i32, [C.c_uint64, C.c_char_p, vp, i32]),
        "gpud_hw_slowdown_check": (i32, [vp, i32, i64, i64, C.c_double, vp, vp, vp, vp, i32]),
        "gpud_store_insert_hw_slowdown": (i32, [vp, C.c_char_p, i64, C.c_uint64, C.c_char_p, vp]),
        "gpud_xid_get_detail": (i32, [i32, vp, vp, vp]), "gpud_sxid_get_detail": (i32, [i32, vp, vp, vp]),
        "gpud_store_insert_sxid_hits": (i32, [vp, C.c_char_p, vp, i64, i64, i64, i32, vp]),
        "gpud_product_mem_caps": (i32, [C.c_char_p]), "gpud_product_fm_supported": (i32, [C.c_char_p]), "gpud_product_fabric_state_supported": (i32, [C.c_char_p]),
        "gpud_xid_detail": (i32, [i32, i32, C.c_uint32, vp, vp, vp, vp, vp]),
        "gpud_xid_build_message": (i32, [C.c_uint64, i32, C.c_uint32, C.c_char_p, C.c_char_p, C.c_char_p, vp, i32]),
        "gpud_xid_hit_message": (i32, [C.POINTER(XidHit), C.c_char_p, vp, i32]), "gpud_xid_device_matches_bus_id": (i32, [C.c_char_p, C.c_char_p]), "gpud_kmsg_event_name": (C.c_char_p, [i32]), "gpud_kmsg_event_message": (C.c_char_p, [i32]),
        "gpud_kmsg_component": (C.c_char_p, [i32]), "gpud_kmsg_hit_message": (i32, [vp, vp, vp, i32]),
        "gpud_kmsg_stateful_create": (i32, [vp]), "gpud_kmsg_stateful_destroy": (None, [vp]),
        "gpud_kmsg_stateful_feed": (i32, [vp, vp, i64, vp, i64, vp, i32, vp]),
        "gpud_component_create": (i32, [vp, C.c_char_p, vp, vp]), "gpud_component_destroy": (None, [vp]), "gpud_component_name": (i32, [vp, vp, i32]),
        "gpud_component_start": (i32, [vp, i64]), "gpud_component_check": (i32, [vp, vp, vp, i32]), "gpud_component_last_health_states": (i32, [vp, vp, i32]),
        "gpud_component_events": (i32, [vp, i64, vp, i32]), "gpud_component_close": (i32, [vp]), "gpud_component_checks": (i64, [vp]),
        "gpud_component_xid_set_source": (i32, [vp, vp, i64, i32, i64]), "gpud_component_xid_set_healthy": (i32, [vp, i64]),
        "gpud_component_xid_add_reboot": (i32, [vp, i64]), "gpud_component_xid_set_devices": (i32, [vp, C.c_char_p]), "gpud_component_ring": (vp, [vp, i32]),
        "gpud_kmsg_stateful_feed_units": (i32, [vp, vp, i64, vp, i64, vp, vp, i32, vp]), "gpud_kmsg_deduper_create": (vp, [i64, i32]),
        "gpud_kmsg_deduper_destroy": (None, [vp]), "gpud_kmsg_dedup_units": (i32, [vp, vp, i64, i32, i64, i64, i64, vp, i64, vp]),
        "gpud_fabric_pack": (i32, [vp, i32, C.POINTER(FabricRaw), vp, vp]),
        "gpud_fabric_verdict_device": (i32, [vp, i32, vp, i32, i32, C.POINTER(FabricVerdict), vp]),
        "gpud_comm_unique_id": (i32, [vp]), "gpud_comm_init": (i32, [vp, i32, i32, i32, vp]),
        "gpud_fabric_issues": (i32, [vp, vp, i32]), "gpud_fabric_suggest_reboot": (i32, [vp]), "gpud_fabric_reason": (i32, [vp, vp, i32, vp, i32]), "gpud_set_nvml_error_string": (None, [vp]), "gpud_nvml_error_strings_from_driver": (i32, []), "gpud_fabric_report_reason": (i32, [vp, vp, i32, vp, vp, i32]),
        "gpud_fabric_gather": (i32, [vp, i32, C.POINTER(FabricRaw), i32, C.POINTER(FabricLocal), C.POINTER(FabricVerdict)]),
        "gpud_fabric_gather_p2p": (i32, [vp, C.POINTER(FabricRaw), i32, C.POINTER(FabricLocal), C.POINTER(FabricVerdict)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    for which, st in enumerate((XidHit, FabricRaw, FabricLocal, FabricVerdict, RingCfg, KmsgEvent, IbSnapshot, IbVerdict, Metric, DedupRule, Temperature, PollCounters, EventRow, NvmlDevice, RemappedRows, EccErrors, GpmMetrics, DrainInfo)):
        if L.gpud_sizeof(which) != C.sizeof(st):
            raise GpudError(-1, "ABI layout mismatch for %s: C %d vs ctypes %d" % (st.__name__, L.gpud_sizeof(which), C.sizeof(st)))
    _lib = L
    return L


class Context:
    """gpud_ctx: one per process, naming the CUDA devices it drives."""

    def __init__(self, devices: Sequence[int] = (0,)):
        self._L = lib()
        self.devices = list(devices)
        arr = (C.c_int32 * len(self.devices))(*self.devices)
        h = C.c_void_p()
        rc = self._L.gpud_ctx_create(arr, len(self.devices), C.byref(h))
        if rc:
            raise GpudError(rc, "gpud_ctx_create failed (no CUDA device? this path has no CPU fallback)")
        self._h = h

    def _check(self, rc: int):
        if rc:
            buf = C.create_string_buffer(512)
            self._L.gpud_last_error(self._h, buf, 512)
            raise GpudError(rc, buf.value.decode("utf-8", "replace"))

    def close(self):
        if self._h:
            self._L.gpud_ctx_destroy(self._h)
            self._h = None

    # ---- kmsg scan ----
    def kmsg_scan(self, buf: bytes, mode: int = SCAN_LINES, dev: Optional[int] = None, cap: int = 1 << 16):
        """Scan host bytes; returns (hits: List[XidHit], n_units)."""
        dev = self.devices[0] if dev is None else dev
        n = len(buf)
        src = C.c_char_p(buf)                     # no copy: the library only reads the bytes during the call
        while True:
            hits = (XidHit * cap)()
            nh, nu = C.c_int64(), C.c_int64()
            rc = self._L.gpud_kmsg_scan(self._h, dev, C.cast(src, C.c_void_p), n, mode, hits, cap, C.byref(nh), C.byref(nu))
            if rc == -4 and nh.value > cap:
                cap = int(nh.value)
                continue
            self._check(rc)
            self.last_scan_raw = (hits, nh.value)
            return [hits[i] for i in range(nh.value)], nu.value

    def kmsg_scan_c(self, buf: bytes, hits, cap: int, mode: int = SCAN_LINES, dev: Optional[int] = None):
        """The bare C call (preallocated XidHit array): what a cgo caller pays.  Returns (n_hits, n_units)."""
        dev = self.devices[0] if dev is None else dev
        nh, nu = C.c_int64(), C.c_int64()
        self._check(self._L.gpud_kmsg_scan(self._h, dev, C.cast(C.c_char_p(buf), C.c_void_p), len(buf), mode, hits, cap, C.byref(nh), C.byref(nu)))
        return nh.value, nu.value

    def kmsg_scan_sharded(self, buf: bytes, mode: int = SCAN_LINES, cap: int = 1 << 16):
        """gpud_kmsg_scan_sharded: the buffer split over every GPU of this context.  Returns (hits, n_units)."""
        hits = (XidHit * cap)()
        nh, nu = C.c_int64(), C.c_int64()
        self._check(self._L.gpud_kmsg_scan_sharded(self._h, C.cast(C.c_char_p(buf), C.c_void_p), len(buf), mode, hits, cap, C.byref(nh), C.byref(nu)))
        return [hits[i] for i in range(min(nh.value, cap))], nu.value

    def kmsg_scan_sharded_c(self, buf: bytes, hits, cap: int, mode: int = SCAN_LINES):
        """the bare C call with a preallocated XidHit array.  Returns (n_hits, n_units)."""
        nh, nu = C.c_int64(), C.c_int64()
        self._check(self._L.gpud_kmsg_scan_sharded(self._h, C.cast(C.c_char_p(buf), C.c_void_p), len(buf), mode, hits, cap, C.byref(nh), C.byref(nu)))
        return nh.value, nu.value

    def kmsg_scan_device(self, dev_ptr: int, length: int, mode: int = SCAN_LINES, dev: Optional[int] = None, cap: int = 1 << 16,
                         stream: int = 0):
        dev = self.devices[0] if dev is None else dev
        hits = (XidHit * cap)()
        nh, nu = C.c_int64(), C.c_int64()
        rc = self._L.gpud_kmsg_scan_device(self._h, dev, C.c_void_p(dev_ptr), length, mode, hits, cap, C.byref(nh), C.byref(nu),
                                           C.c_void_p(stream))
        self._check(rc)
        return [hits[i] for i in range(nh.value)], nu.value

    def scan_kernel_ms(self, dev: Optional[int] = None):
        dev = self.devices[0] if dev is None else dev
        ms = (C.c_float * 3)()
        self._check(self._L.gpud_kmsg_scan_kernel_ms(self._h, dev, ms))
        return list(ms)

    def scan_phase_timing(self, on: bool, dev: Optional[int] = None):
        """on: plain launches split by events (scan_kernel_ms -> [filter, prefix, match]); off (default): one overlapped chain
        (scan_kernel_ms -> [whole device time, 0, 0])"""
        dev = self.devices[0] if dev is None else dev
        self._check(self._L.gpud_kmsg_scan_phase_timing(self._h, dev, 1 if on else 0))

    def scan_stats(self, dev: Optional[int] = None):
        dev = self.devices[0] if dev is None else dev
        out = (C.c_int64 * 3)()
        self._check(self._L.gpud_kmsg_scan_stats(self._h, dev, out))
        return {"candidates": out[0], "hits": out[1], "separators": out[2]}

    def classify(self, hits: List[XidHit], dev: Optional[int] = None) -> List[XidHit]:
        dev = self.devices[0] if dev is None else dev
        arr = (XidHit * len(hits))(*hits)
        self._check(self._L.gpud_xid_classify(self._h, dev, arr, len(hits)))
        return [arr[i] for i in range(len(hits))]

    def hit_json(self, hit: XidHit, unix_seconds: int = 0) -> str:
        buf = C.create_string_buffer(4096)
        rc = self._L.gpud_hit_detail_json(C.byref(hit), unix_seconds, buf, 4096)
        if rc:
            raise GpudError(rc, "gpud_hit_detail_json")
        return buf.value.decode("utf-8")

    def hit_message(self, hit: XidHit, gpu_uuid: str = "") -> str:
        return xid_hit_message(hit, gpu_uuid)

    def ib_scan(self, series, drop_threshold: int, flap_down_interval: int, flap_back_threshold: int, dev: Optional[int] = None):
        """series: list of lists of (ts, down, total_link_downed); returns one IbVerdict per series"""
        dev = self.devices[0] if dev is None else dev
        total = sum(len(s) for s in series)
        snaps = (IbSnapshot * max(1, total))()
        offs = (C.c_int64 * (len(series) + 1))()
        k = 0
        for i, s in enumerate(series):
            offs[i] = k
            for ts, down, tld in s:
                snaps[k].ts, snaps[k].down, snaps[k].total_link_downed = ts, 1 if down else 0, tld
                k += 1
        offs[len(series)] = k
        out = (IbVerdict * max(1, len(series)))()
        self._check(self._L.gpud_ib_scan(self._h, dev, snaps, offs, len(series), drop_threshold, flap_down_interval, flap_back_threshold, out))
        return [out[i] for i in range(len(series))]

    def kmsg_message(self, hit: XidHit, buf: bytes = None) -> str:
        """(eventName, message) of an extra-matcher hit exactly as the component's Match returns it"""
        out = C.create_string_buffer(4096)
        n = self._L.gpud_kmsg_hit_message(C.byref(hit), C.cast(C.c_char_p(buf), C.c_void_p) if buf is not None else None, out, 4096)
        if n < 0:
            raise GpudError(n, "gpud_kmsg_hit_message")
        return out.raw[:n].decode("latin-1")

    # ---- fabric ----
    def fabric_pack(self, raw: FabricRaw, dev_send_ptr: int, dev: Optional[int] = None, stream: int = 0):
        dev = self.devices[0] if dev is None else dev
        self._check(self._L.gpud_fabric_pack(self._h, dev, C.byref(raw), C.c_void_p(dev_send_ptr), C.c_void_p(stream)))

    def fabric_verdict(self, dev_all_ptr: int, n: int, at_least: int = 0, dev: Optional[int] = None, stream: int = 0) -> FabricVerdict:
        dev = self.devices[0] if dev is None else dev
        v = FabricVerdict()
        self._check(self._L.gpud_fabric_verdict_device(self._h, dev, C.c_void_p(dev_all_ptr), n, at_least, C.byref(v), C.c_void_p(stream)))
        return v

    def fabric_gather_p2p(self, raws: Sequence[FabricRaw], at_least: int = 0):
        n = len(self.devices)
        arr = (FabricRaw * n)(*raws)
        allrec = (FabricLocal * n)()
        vs = (FabricVerdict * n)()
        self._check(self._L.gpud_fabric_gather_p2p(self._h, arr, at_least, allrec, vs))
        return [allrec[i] for i in range(n)], [vs[i] for i in range(n)]

    def comm_init(self, n_ranks: int, rank: int, unique_id: bytes, dev: Optional[int] = None):
        dev = self.devices[0] if dev is None else dev
        b = C.create_string_buffer(unique_id, 128)
        self._check(self._L.gpud_comm_init(self._h, dev, n_ranks, rank, b))

    def fabric_gather(self, raw: FabricRaw, n_ranks: int, at_least: int = 0, dev: Optional[int] = None):
        dev = self.devices[0] if dev is None else dev
        allrec = (FabricLocal * n_ranks)()
        v = FabricVerdict()
        self._check(self._L.gpud_fabric_gather(self._h, dev, C.byref(raw), at_least, allrec, C.byref(v)))
        return [allrec[i] for i in range(n_ranks)], v


def comm_unique_id() -> bytes:
    b = C.create_string_buffer(128)
    rc = lib().gpud_comm_unique_id(b)
    if rc:
        raise GpudError(rc, "gpud_comm_unique_id (libnccl.so.2 not loadable?)")
    return b.raw


class Ring:
    """gpud_ring: device-resident [F][CAP] sample ring with fused windowed aggregates."""

    def __init__(self, ctx: Context, n_fields: int, capacity: int, window: int, thresholds: Optional[np.ndarray] = None,
                 ema_alpha: float = 0.0, q_num: int = 0, q_den: int = 0, dev: Optional[int] = None):
        self.ctx, self._L = ctx, ctx._L
        self.F, self.cap, self.W = n_fields, capacity, window
        cfg = RingCfg(n_fields, window, capacity, ema_alpha, q_num, q_den, None)
        if thresholds is not None:
            self._thr = np.ascontiguousarray(thresholds, dtype=np.float64)
            assert self._thr.shape == (n_fields,)
            cfg.thresholds = self._thr.ctypes.data_as(C.POINTER(C.c_double))
        h = C.c_void_p()
        ctx._check(self._L.gpud_ring_create(ctx._h, ctx.devices[0] if dev is None else dev, C.byref(cfg), C.byref(h)))
        self._h = h

    def close(self):
        if self._h:
            self._L.gpud_ring_destroy(self._h)
            self._h = None

    def set_cta_reserve(self, n_ctas: int):
        self.ctx._check(self._L.gpud_ring_set_cta_reserve(self._h, n_ctas))

    def set_stream(self, cuda_stream: int):
        self.ctx._check(self._L.gpud_ring_set_stream(self._h, C.c_void_p(cuda_stream)))

    def push(self, rows: np.ndarray):
        rows = np.ascontiguousarray(rows, dtype=np.float64)
        assert rows.ndim == 2 and rows.shape[1] == self.F
        self.ctx._check(self._L.gpud_ring_push(self._h, C.c_void_p(rows.ctypes.data), rows.shape[0]))

    def push_ptr(self, host_ptr: int, n_rows: int):
        self.ctx._check(self._L.gpud_ring_push(self._h, C.c_void_p(host_ptr), n_rows))

    def push_raw(self, rows: np.ndarray):
        """rows [n][F] of raw counter samples in the getter's own type (uint32 / int32 / float32 / int64 / uint64 / float64)"""
        rows = np.ascontiguousarray(rows)
        assert rows.ndim == 2 and rows.shape[1] == self.F
        self.ctx._check(self._L.gpud_ring_push_raw(self._h, C.c_void_p(rows.ctypes.data), rows.shape[0], DTYPES[rows.dtype.name]))

    def push_raw_ptr(self, host_ptr: int, n_rows: int, dtype: int):
        self.ctx._check(self._L.gpud_ring_push_raw(self._h, C.c_void_p(host_ptr), n_rows, dtype))

    def push_device(self, dev_ptr: int, n_rows: int):
        self.ctx._check(self._L.gpud_ring_push_device(self._h, C.c_void_p(dev_ptr), n_rows))

    def counts(self):
        t, c, w = C.c_int64(), C.c_int64(), C.c_int64()
        self.ctx._check(self._L.gpud_ring_counts(self._h, C.byref(t), C.byref(c), C.byref(w)))
        return t.value, c.value, w.value

    def reduce(self):
        self.ctx._check(self._L.gpud_ring_reduce(self._h))

    def sync(self):
        self.ctx._check(self._L.gpud_ring_sync(self._h))

    def kernel_ms(self):
        a, b = C.c_float(), C.c_float()
        self.ctx._check(self._L.gpud_ring_kernel_ms(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def read(self, op: str) -> np.ndarray:
        _, _, nw = self.counts()
        dt = np.uint32 if op == "n_over" else np.float64
        out = np.empty((self.F, nw), dtype=dt)
        self.ctx._check(self._L.gpud_ring_read(self._h, OPS[op], C.c_void_p(out.ctypes.data), out.nbytes))
        return out

    def result_ptr(self, op: str) -> int:
        p = C.c_void_p()
        self.ctx._check(self._L.gpud_ring_result_ptr(self._h, OPS[op], C.byref(p)))
        return p.value

    def reduce_all(self) -> dict:
        self.reduce()
        return {k: self.read(k) for k in OPS}

    def push_timed(self, rows: np.ndarray, unix_ms):
        """push_raw with the unix-ms time of every row (non-decreasing, not before the last timed row)"""
        rows = np.ascontiguousarray(rows)
        assert rows.ndim == 2 and rows.shape[1] == self.F
        ms = np.ascontiguousarray(unix_ms, dtype=np.int64)
        assert ms.shape == (rows.shape[0],)
        self.ctx._check(self._L.gpud_ring_push_timed(self._h, C.c_void_p(rows.ctypes.data), rows.shape[0], DTYPES[rows.dtype.name],
                                                     C.c_void_p(ms.ctypes.data)))

    def drain(self, max_windows: int) -> dict:
        """gpud_ring_drain: the next complete stream-aligned windows, each [F][n] like reduce_all, plus "window_end_unix_ms" [n] and
        "info" {first_window, n_windows, n_lost, n_pending}.  max_windows = 0 only reports the counts."""
        mw = max(0, int(max_windows))
        f64 = np.empty((5, self.F, max(1, mw)), dtype=np.float64)
        nov = np.empty((self.F, max(1, mw)), dtype=np.uint32)
        ms = np.empty((max(1, mw),), dtype=np.int64)
        info = DrainInfo()
        self.ctx._check(self._L.gpud_ring_drain(self._h, mw, C.c_void_p(f64.ctypes.data), C.c_void_p(nov.ctypes.data), C.c_void_p(ms.ctypes.data),
                                                C.byref(info)))
        n = info.n_windows
        out = {k: f64[OPS[k]][:, :n].copy() for k in ("min", "max", "mean", "ema", "p99")}
        out["n_over"] = nov[:, :n].copy()
        out["window_end_unix_ms"] = ms[:n].copy()
        out["info"] = info.as_dict()
        return out

    def drain_to_store(self, store: "Store", components, field_names, labels_json: str = "", ops_mask: int = 0, max_windows: int = 1 << 20,
                       table: str = ""):
        """gpud_ring_drain_to_store: one metrics row per returned window x named field x op; field_names[f] None skips field f.
        Returns (info dict, rows written, windows moved to keep their times increasing)."""
        assert len(components) == self.F and len(field_names) == self.F
        comps = [c.encode() if c is not None else None for c in components]
        names = [f.encode() if f is not None else None for f in field_names]
        ca, na = (C.c_char_p * self.F)(*comps), (C.c_char_p * self.F)(*names)
        info, rows, shifted = DrainInfo(), C.c_int64(), C.c_int64()
        rc = self._L.gpud_ring_drain_to_store(self._h, store._h, table.encode(), ca, na, labels_json.encode(), ops_mask, max_windows, C.byref(info),
                                              C.byref(rows), C.byref(shifted))
        if rc:
            sb, cb = C.create_string_buffer(512), C.create_string_buffer(512)
            self._L.gpud_store_last_error(store._h, sb, 512)
            self._L.gpud_last_error(self.ctx._h, cb, 512)
            raise GpudError(rc, "%s (ring: %s)" % (sb.value.decode("utf-8", "replace"), cb.value.decode("utf-8", "replace")))
        return info.as_dict(), rows.value, shifted.value

    def reduce_range(self, last_n: int = 0) -> dict:
        f64 = np.empty((5, self.F), dtype=np.float64)
        nov = np.empty((self.F,), dtype=np.uint32)
        self.ctx._check(self._L.gpud_ring_reduce_range(self._h, last_n, C.c_void_p(f64.ctypes.data), C.c_void_p(nov.ctypes.data)))
        return {"min": f64[0], "max": f64[1], "mean": f64[2], "ema": f64[3], "p99": f64[4], "n_over": nov}

    def range_stats(self):
        """Device ms of the last single-pass reduce_range (fused pass alone, whole device side) and the number of fields the
        radix select had to redo."""
        a, b, n = C.c_float(), C.c_float(), C.c_int32()
        why = (C.c_int32 * 7)()
        self.ctx._check(self._L.gpud_ring_range_stats(self._h, C.byref(a), C.byref(b), C.byref(n), why))
        self.range_open_reasons = {k: int(why[i]) for i, k in enumerate(("", "short", "nan", "pivots", "above", "below", "overflow")) if i and why[i]}
        return float(a.value), float(b.value), int(n.value)
