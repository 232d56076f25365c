// ring_drain.h — the two halves of a streaming drain (ring.cu), shared with the store writer (store_sqlite.cpp).  Not part of the ABI:
// C++ linkage, no CUDA types, so a host translation unit can include it without the CUDA headers.
#pragma once
#include <stdint.h>

#include "../../include/gpud_b200.h"

// Reduce the complete stream-aligned windows [k0, k0 + n) the cursor points at (n <= max_windows) into the caller's arrays
// (gpud_ring_drain's layout) WITHOUT moving the cursor or the EMA state; *info says which windows they are.  max_windows = 0 only
// fills *info.  Synchronous.  Errors are recorded on the ring's ctx.
int32_t gpud_ring_drain_peek(gpud_ring* r, int64_t max_windows, double* out_f64, uint32_t* out_n_over, int64_t* window_end_unix_ms,
                             gpud_drain_info* info);
// Make a peek final: the cursor moves past the windows it returned (and the lost ones before them) and the EMA state becomes the EMA of
// its last window.  last_export_ms (when not INT64_MIN) is the time the store writer gave the newest exported window.
void gpud_ring_drain_commit(gpud_ring* r, const gpud_drain_info* info, int64_t last_export_ms);
// Time the store writer gave the newest window it exported from this ring (INT64_MIN: none yet).
int64_t gpud_ring_drain_last_export(const gpud_ring* r);
// The ring's field count and order statistic (ring.cu).
int gpud_ring_n_fields(const gpud_ring* r);
void gpud_ring_quantile(gpud_ring* r, int* q_num, int* q_den);
