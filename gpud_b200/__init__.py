"""gpud_b200 — B200-native telemetry aggregation + Xid scan hot path of gpud behind a C ABI (include/gpud_b200.h).

The product is `libgpud_b200.so` (hand-written sm_100a CUDA, gpud_b200/csrc).  This package is only the Python
binding over that C ABI used by the tests and bench.py; it contains no compute and no CPU fallback: every entry
point raises if the shared library or a CUDA device is missing.
"""
from .capi import (Context, GpudError, Ring, FabricRaw, FabricLocal, FabricVerdict, XidHit, lib, OPS, EVENT_NAMES,
                   ACTION_WIRE, SCAN_LINES, SCAN_RAW_KMSG, SCAN_EXT_MATCHERS, DTYPES, KmsgStateful, KmsgEvent, Poller, POLL_FIELDS, IbSnapshot, IbVerdict, ib_reason, Store, Metric, DedupRule, EventRow, xid_build_message, xid_hit_message, xid_detail, Temperature, PollCounters, temperature_check, fabric_reason, hw_slowdown_event_message, hw_slowdown_check, temperature_reason, fabric_report_reason, DrainInfo, window_metric_name)

__all__ = ["Context", "GpudError", "Ring", "FabricRaw", "FabricLocal", "FabricVerdict", "XidHit", "lib", "OPS",
           "EVENT_NAMES", "ACTION_WIRE", "SCAN_LINES", "SCAN_RAW_KMSG", "SCAN_EXT_MATCHERS", "DTYPES", "KmsgStateful", "KmsgEvent", "Poller", "POLL_FIELDS", "IbSnapshot", "IbVerdict", "ib_reason", "Store", "Metric", "DedupRule", "EventRow", "xid_build_message", "xid_hit_message", "xid_detail", "Temperature", "PollCounters", "temperature_check", "fabric_reason", "hw_slowdown_event_message", "hw_slowdown_check", "temperature_reason", "fabric_report_reason", "DrainInfo", "window_metric_name"]
