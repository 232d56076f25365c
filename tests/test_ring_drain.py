"""Streaming windows: gpud_ring_drain / push_timed / drain_to_store / purge_metrics and the temperature component as a metrics source.

The oracle of every drained window is the window aggregate over the WHOLE pushed stream (stream index = sample index since create), sliced
to the windows the drain returned; the EMA chain starts at the first sample of the window where the drain restarted it (the first drain,
or one after a loss).  Selections and n_over are bit-exact, mean and EMA at 1e-6 relative (oracle/SPEC.md)."""
import ctypes as C
import json
import sqlite3
import time

import numpy as np
import pytest

import gpud_b200 as g
from oracle import coracle
from oracle import pyoracle as O
import synth

F64_OPS = ("min", "max", "mean", "ema", "p99")
ALL_OPS = F64_OPS + ("n_over",)
# the temperature component's column map (poll column -> component_name, metric name)
POLL_COMPONENTS = ["accelerator-nvidia-temperature", "accelerator-nvidia-power", "accelerator-nvidia-clock-speed", "accelerator-nvidia-clock-speed",
                   "accelerator-nvidia-clock-speed", "accelerator-nvidia-utilization", "accelerator-nvidia-utilization", "accelerator-nvidia-memory"]
POLL_METRICS = ["accelerator_nvidia_temperature_current_celsius", "accelerator_nvidia_power_current_usage_milli_watts",
                "accelerator_nvidia_clock_speed_graphics_mhz", "accelerator_nvidia_clock_speed_sm_mhz", "accelerator_nvidia_clock_speed_memory_mhz",
                "accelerator_nvidia_utilization_gpu_util_percent", "accelerator_nvidia_utilization_memory_util_percent", "accelerator_nvidia_memory_used_mib"]
# the reference's read query (pkg/metrics/store/sqlite.go:169-256) without Since / component selection
READ_SQL = "SELECT unix_milliseconds, component_name, metric_name, metric_labels, metric_value\nFROM %s\nORDER BY unix_milliseconds ASC;"


class DrainModel:
    """The cursor arithmetic of a push / drain schedule, and where the EMA chain of each drain starts."""

    def __init__(self, W: int, cap: int):
        self.W, self.cap = W, cap
        self.total, self.next, self.ema_window, self.ema_seed = 0, 0, -1, 0

    def push(self, n: int):
        self.total += n

    def drain(self, max_windows: int) -> dict:
        W, count = self.W, min(self.total, self.cap)
        complete = self.total // W
        k0 = max(self.next, -(-(self.total - count) // W))
        avail = complete - k0
        n = min(avail, max_windows)
        info = {"first_window": k0, "n_windows": n, "n_lost": k0 - self.next, "n_pending": avail - n}
        if max_windows > 0:
            if n > 0 and not (k0 > 0 and self.ema_window == k0 - 1):
                self.ema_seed = k0                          # first drain, or one after a loss: the EMA restarts at x[k0 W]
            self.next = k0 + n
            if n > 0:
                self.ema_window = k0 + n - 1
        return info


def _want(stream, W, thr, k0, n, seed, alpha=0.0, qn=0, qd=0):
    """oracle of windows [k0, k0 + n) of the stream [samples][F], EMA chain started at window `seed`"""
    out = coracle.windows_fields(np.ascontiguousarray(stream[seed * W:(k0 + n) * W].T), W, thr, alpha, qn, qd)
    return {k: v[:, k0 - seed:k0 - seed + n] for k, v in out.items()}


def _check(got, want, scale):
    for k in ("min", "max", "p99"):
        assert np.array_equal(got[k].view(np.uint64), want[k].view(np.uint64)), k
    assert np.array_equal(got["n_over"].astype(np.uint64), want["n_over"].astype(np.uint64))
    for k in ("mean", "ema"):
        with np.errstate(invalid="ignore"):
            err = np.abs(got[k] - want[k])
            tol = 1e-6 * np.maximum(np.abs(want[k]), scale)
            same = (got[k] == want[k]) | (np.isnan(got[k]) & np.isnan(want[k]))
        assert np.all((err <= tol) | same), (k, got[k], want[k])


def _scale(x):
    f = np.abs(x[np.isfinite(x)])
    return max(1e-300, float(f.max()) if f.size else 0.0)


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("qn,qd,want", [(99, 100, "p99"), (50, 100, "p50"), (999, 1000, "p99_9"), (1, 3, "p33_3333"), (0, 1, "p0"), (1, 1, "p100")])
def test_window_metric_name_quantiles(qn, qd, want):
    assert g.window_metric_name("gpu_temp", "p99", qn, qd) == "gpu_temp_window_" + want


def test_window_metric_name_ops_and_capacity():
    for op in ("min", "max", "mean", "ema", "n_over"):
        assert g.window_metric_name("f", op) == "f_window_" + op
    L = g.lib()
    buf = C.create_string_buffer(64)
    assert L.gpud_window_metric_name(b"f", 0, 99, 100, buf, 11) == -1          # "f_window_min" needs 13 bytes
    assert L.gpud_window_metric_name(b"f", 0, 99, 100, buf, 13) == 12 and buf.value == b"f_window_min"
    assert L.gpud_window_metric_name(b"f", 6, 99, 100, buf, 64) == -1          # no such op
    assert L.gpud_sizeof(17) == C.sizeof(g.DrainInfo) == 32


def test_purge_metrics(tmp_path):
    try:
        st = g.Store(str(tmp_path / "gpud.state"))
    except g.GpudError as e:
        pytest.skip("no libsqlite3.so.0: %s" % e)
    st.metrics_table()
    rows = [(1000 + 10 * i, "c%d" % (i % 3), "m", '{"uuid":"GPU-0"}', float(i)) for i in range(50)]
    st.record_metrics(rows)
    assert st.purge_metrics(1000) == 0
    assert st.purge_metrics(1200) == 20                                         # unix_milliseconds < 1200: rows 0..19
    assert st.purge_metrics(1200) == 0
    db = sqlite3.connect(str(tmp_path / "gpud.state"))
    left = db.execute(READ_SQL % "gpud_metrics_v0_5").fetchall()
    db.close()
    assert left == [r for r in rows if r[0] >= 1200]
    with pytest.raises(g.GpudError):
        st.purge_metrics(0, table="no such table")
    st.close()


def test_drain_model_cursor_cases():
    m = DrainModel(W=10, cap=30)
    m.push(25)
    assert m.drain(0) == {"first_window": 0, "n_windows": 0, "n_lost": 0, "n_pending": 2}      # a query moves nothing
    assert m.drain(1) == {"first_window": 0, "n_windows": 1, "n_lost": 0, "n_pending": 1}
    assert m.drain(0) == {"first_window": 1, "n_windows": 0, "n_lost": 0, "n_pending": 1}
    m.push(40)                                                                  # total 65: samples 35.. survive, windows 1..3 are gone
    assert m.drain(5) == {"first_window": 4, "n_windows": 2, "n_lost": 3, "n_pending": 0}
    assert m.ema_seed == 4
    m.push(3)
    assert m.drain(5) == {"first_window": 6, "n_windows": 0, "n_lost": 0, "n_pending": 0}
    m.push(7)
    assert m.drain(5) == {"first_window": 6, "n_windows": 1, "n_lost": 0, "n_pending": 0} and m.ema_seed == 4   # the EMA continues
    m2 = DrainModel(W=7, cap=20)
    m2.push(100)                                                                # one push larger than CAP: the skipped rows count
    assert m2.drain(100) == {"first_window": 12, "n_windows": 2, "n_lost": 12, "n_pending": 0}


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def ctx():
    c = g.Context([0])
    yield c
    c.close()


@pytest.fixture
def store(tmp_path):
    try:
        st = g.Store(str(tmp_path / "gpud.state"))
    except g.GpudError as e:
        pytest.skip("no libsqlite3.so.0: %s" % e)
    st.metrics_table()
    yield st, str(tmp_path / "gpud.state")
    st.close()


def _drain_all(ring, chunk):
    parts = []
    while True:
        d = ring.drain(chunk)
        if d["info"]["n_windows"] == 0:
            break
        parts.append(d)
    if not parts:
        return None
    out = {k: np.concatenate([p[k] for p in parts], axis=1) for k in ALL_OPS}
    out["window_end_unix_ms"] = np.concatenate([p["window_end_unix_ms"] for p in parts])
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [1 << 14, 1, 3, 64])
@pytest.mark.parametrize("F,n,W,cap", [(8, 4000, 1000, 4096), (5, 4096, 1000, 4096), (3, 2777, 1024, 4096), (4, 600, 7, 1024),
                                        (2, 100, 1, 128), (6, 3000, 333, 4096), (64, 10000, 1000, 10000)])
def test_drain_before_wrap_equals_reduce(ctx, F, n, W, cap, chunk):
    x = synth.gauge_stream(F, n, seed=F * 1000 + W)
    thr = synth.thresholds_for(x)
    r = g.Ring(ctx, F, cap, W, thresholds=thr)
    r.push(x)
    red = r.reduce_all()
    got = _drain_all(r, chunk)
    nc = n // W
    for k in ("min", "max", "p99"):                             # the same kernel on the same samples
        assert np.array_equal(got[k].view(np.uint64), red[k][:, :nc].view(np.uint64)), k
    assert np.array_equal(got["n_over"], red["n_over"][:, :nc])
    _check(got, {k: red[k][:, :nc] for k in ALL_OPS}, _scale(x))
    _check(got, _want(x, W, thr, 0, nc, 0), _scale(x))
    assert r.drain(0)["info"] == {"first_window": nc, "n_windows": 0, "n_lost": 0, "n_pending": 0}
    assert not got["window_end_unix_ms"].any()                  # untimed pushes
    r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("W,cap", [(1, 64), (7, 100), (333, 1000), (1000, 3500), (1024, 3000)])
@pytest.mark.parametrize("keep_up", [True, False])
def test_drain_random_schedules(ctx, W, cap, keep_up):
    F = 3
    rng = np.random.default_rng(W * 7 + cap + keep_up)
    n_total = 12 * cap + 3 * W
    x = synth.gauge_stream(F, n_total, seed=W + 5)
    thr = synth.thresholds_for(x)
    r = g.Ring(ctx, F, cap, W, thresholds=thr)
    m = DrainModel(W, cap)
    pos, n_checked, scale = 0, 0, _scale(x)
    nw_max = -(-cap // W)
    while pos < n_total:
        hi = cap - W + 1 if keep_up else 2 * cap
        b = int(min(n_total - pos, rng.choice([1, 2, max(1, W - 1), W, W + 1, rng.integers(1, hi + 1), hi])))
        b = max(1, min(b, hi))
        r.push(x[pos:pos + b])
        m.push(b)
        pos += b
        mw = int(rng.choice([0, 1, 2, nw_max, 4 * nw_max])) if not keep_up else nw_max
        want_info = m.drain(mw)
        d = r.drain(mw)
        assert d["info"] == want_info, (pos, mw)
        if keep_up:
            assert want_info["n_lost"] == 0 and want_info["n_pending"] == 0
        n = want_info["n_windows"]
        if n:
            _check(d, _want(x, W, thr, want_info["first_window"], n, m.ema_seed), scale)
            n_checked += n
    assert n_checked > 5
    r.close()


@pytest.mark.gpu
def test_drain_chunks_inside_one_call(ctx):
    """more windows than one launch's scratch holds (2^20 (field, window) pairs): the drain runs several launches, EMA carried across"""
    F, W, cap = 1, 1, 1_500_000
    x = synth.gauge_stream(F, cap + 4, seed=3)
    thr = synth.thresholds_for(x)
    r = g.Ring(ctx, F, cap, W, thresholds=thr)
    r.push(x)
    d = r.drain(cap)
    assert d["info"] == {"first_window": 4, "n_windows": cap, "n_lost": 4, "n_pending": 0}
    _check(d, _want(x, W, thr, 4, cap, 4), _scale(x))
    r.close()


@pytest.mark.gpu
def test_drain_loss_restarts_ema(ctx):
    F, W, cap, alpha = 4, 100, 1050, 5e-4                       # a slow EMA: the restart is visible long after it
    x = synth.gauge_stream(F, 4000, seed=17)
    thr = synth.thresholds_for(x)
    r = g.Ring(ctx, F, cap, W, thresholds=thr, ema_alpha=alpha)
    r.push(x[:450])
    d = r.drain(2)
    assert d["info"] == {"first_window": 0, "n_windows": 2, "n_lost": 0, "n_pending": 2}
    _check(d, _want(x, W, thr, 0, 2, 0, alpha), _scale(x))
    r.push(x[450:2450])                                          # total 2450, count 1050: samples 1400.. survive
    d = r.drain(5)
    assert d["info"] == {"first_window": 14, "n_windows": 5, "n_lost": 12, "n_pending": 5}
    _check(d, _want(x, W, thr, 14, 5, 14, alpha), _scale(x))
    whole = _want(x, W, thr, 14, 5, 0, alpha)["ema"]            # the EMA of the whole stream is a different number
    assert np.abs(d["ema"] - whole).max() > 1e-3 * _scale(x)
    d = r.drain(100)                                             # no loss: the EMA continues from window 18
    assert d["info"] == {"first_window": 19, "n_windows": 5, "n_lost": 0, "n_pending": 0}
    _check(d, _want(x, W, thr, 19, 5, 14, alpha), _scale(x))
    r.close()


@pytest.mark.gpu
def test_drain_leaves_reduce_results_alone(ctx):
    F, W, cap = 6, 333, 4000
    x = synth.gauge_stream(F, 9001, seed=23)
    thr = synth.thresholds_for(x)
    r = g.Ring(ctx, F, cap, W, thresholds=thr)
    r.push(x[:5000])
    r.drain(64)                                                  # the ring has wrapped once; the cursor is in the middle of it
    r.push(x[5000:])
    rng_before = r.reduce_range(3000)
    r.reduce()
    d = r.drain(64)
    assert d["info"]["n_windows"] > 0
    after = {k: r.read(k) for k in ALL_OPS}
    again = r.reduce_all()
    for k in ALL_OPS:
        assert np.array_equal(after[k].view(np.uint8), again[k].view(np.uint8)), k
    rng_after = r.reduce_range(3000)
    for k in ALL_OPS:
        assert np.array_equal(np.asarray(rng_before[k]).view(np.uint8), np.asarray(rng_after[k]).view(np.uint8)), k
    r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [1 << 14, 1])
def test_drain_special_values(ctx, chunk):
    W, cap, n = 1000, 4000, 4000
    rng = np.random.default_rng(3)
    cols = [np.full(n, 65.0), np.arange(n, dtype=np.float64), -np.arange(n, dtype=np.float64),
            rng.integers(60, 64, n).astype(np.float64), np.where(rng.random(n) < 0.5, 0.0, -0.0),
            np.concatenate([np.full(n - 3, 1.0), [np.inf, -np.inf, 5.0]]), rng.standard_normal(n) * 1e300,
            np.where(np.arange(n) % 1000 < 15, 1e6 + np.arange(n), rng.standard_normal(n)),
            rng.integers(0, 2, n).astype(np.float64)]
    x = np.ascontiguousarray(np.stack(cols, axis=1))
    x[1234, 3] = np.nan
    thr = np.zeros(x.shape[1])
    r = g.Ring(ctx, x.shape[1], cap, W, thresholds=thr)
    r.push(x)
    got = _drain_all(r, chunk)
    for f in range(x.shape[1]):
        with np.errstate(invalid="ignore"):                    # inf + -inf in a window's sum is NaN on both sides
            want = O.window_aggregates(x[:, f], W, thr[f])
        _check({k: got[k][f] for k in ALL_OPS}, want, _scale(x[:, f]))
    r.close()


@pytest.mark.gpu
def test_timed_pushes(ctx, store):
    st, path = store
    F, W, cap = 2, 50, 1000
    x = synth.gauge_stream(F, 600, seed=31)
    ms = 1_700_000_000_000 + 3 * np.arange(600, dtype=np.int64)
    r = g.Ring(ctx, F, cap, W)
    r.push_timed(x[:130], ms[:130])
    r.push_timed(x[130:400], ms[130:400])
    d = r.drain(64)
    assert d["info"]["n_windows"] == 8
    assert np.array_equal(d["window_end_unix_ms"], ms[np.arange(1, 9) * W - 1])
    with pytest.raises(g.GpudError) as e:                        # decreasing inside the call: nothing appended
        r.push_timed(x[400:410], ms[400:410][::-1].copy())
    assert e.value.code == -1 and r.counts()[0] == 400
    with pytest.raises(g.GpudError) as e:                        # earlier than the last timed row
        r.push_timed(x[400:410], ms[300:310])
    assert e.value.code == -1 and r.counts()[0] == 400
    r.push(x[400:500])                                           # untimed: windows 8, 9 have no time
    d = r.drain(0)
    assert d["info"] == {"first_window": 8, "n_windows": 0, "n_lost": 0, "n_pending": 2}
    with pytest.raises(g.GpudError) as e:
        r.drain_to_store(st, ["c"] * F, ["f0", "f1"])
    assert e.value.code == -6
    assert r.drain(0)["info"] == {"first_window": 8, "n_windows": 0, "n_lost": 0, "n_pending": 2}   # the cursor did not move
    d = r.drain(64)
    assert not d["window_end_unix_ms"].any()
    r.close()
    # W = 1 and one millisecond for every row: the windows are moved apart so that none replaces another
    r = g.Ring(ctx, 1, 64, 1)
    r.push_timed(np.arange(10, dtype=np.float64)[:, None], np.full(10, 5000, dtype=np.int64))
    info, n_rows, shifted = r.drain_to_store(st, ["c"], ["g"], ops_mask=1 << g.OPS["max"])
    assert (info["n_windows"], n_rows, shifted) == (10, 10, 9)
    db = sqlite3.connect(path)
    got = db.execute(READ_SQL % "gpud_metrics_v0_5").fetchall()
    db.close()
    assert got == [(5000 + i, "c", "g_window_max", "", float(i)) for i in range(10)]
    r.push_timed(np.zeros((1, 1)), np.array([5003], dtype=np.int64))   # after the previous export's last time (5009): 5010
    assert r.drain_to_store(st, ["c"], ["g"], ops_mask=1)[1:] == (1, 1)
    r.close()


@pytest.mark.gpu
def test_drain_to_store_rows_and_retry(ctx, store):
    st, path = store
    F, W, cap = 3, 100, 1000
    x = synth.gauge_stream(F, 950, seed=41)
    thr = synth.thresholds_for(x)
    ms = 1_700_000_000_000 + 7 * np.arange(950, dtype=np.int64)
    r = g.Ring(ctx, F, cap, W, thresholds=thr, q_num=999, q_den=1000)
    r.push_timed(x, ms)
    comps, names, labels = ["comp-a", "comp-b", None], ["field_a", "field_b", None], '{"gpu":"0","uuid":"GPU-x"}'
    with pytest.raises(g.GpudError):
        r.drain_to_store(st, comps, names, labels, table="not_created")
    assert r.drain(0)["info"]["n_pending"] == 9
    info, n_rows, shifted = r.drain_to_store(st, comps, names, labels, max_windows=6)
    assert info == {"first_window": 0, "n_windows": 6, "n_lost": 0, "n_pending": 3} and n_rows == 6 * 2 * 6 and shifted == 0
    info, n_rows, _ = r.drain_to_store(st, comps, names, labels)
    assert info == {"first_window": 6, "n_windows": 3, "n_lost": 0, "n_pending": 0} and n_rows == 3 * 2 * 6
    want = _want(x, W, thr, 0, 9, 0, qn=999, qd=1000)
    op_name = {"min": "min", "max": "max", "mean": "mean", "ema": "ema", "p99": "p99_9", "n_over": "n_over"}
    db = sqlite3.connect(path)
    rows = db.execute(READ_SQL % "gpud_metrics_v0_5").fetchall()
    db.close()
    assert len(rows) == 9 * 2 * 6
    got = {(t, c, nm): v for t, c, nm, lab, v in rows}
    assert all(lab == labels for _, _, _, lab, _ in rows)
    for k in range(9):
        t = int(ms[(k + 1) * W - 1])
        for f in range(2):
            for op in ALL_OPS:
                v = got[(t, comps[f], "%s_window_%s" % (names[f], op_name[op]))]
                w = float(want[op][f, k])
                if op in ("mean", "ema"):
                    assert abs(v - w) <= 1e-6 * max(abs(w), _scale(x)), (k, f, op)
                else:
                    assert v == w, (k, f, op)
    r.close()


@pytest.mark.gpu
def test_poller_windows_into_store(ctx, store):
    st, path = store
    W, cap, n = 1000, 4096, 3000
    thr = np.array([60.0, 200000.0, 1500.0, 1500.0, 3000.0, 50.0, 50.0, 1000.0])
    ring = g.Ring(ctx, len(g.POLL_FIELDS), cap, W, thresholds=thr)
    try:
        poller = g.Poller(ctx, ring)
    except g.GpudError as e:
        ring.close()
        pytest.skip("no NVML on this host: %s" % e)
    t0 = int(time.time() * 1000)
    poller.poll(n)
    t1 = int(time.time() * 1000)
    rows, _ = poller.last_rows()
    info, n_rows, _ = ring.drain_to_store(st, POLL_COMPONENTS, POLL_METRICS, '{"uuid":"GPU-test"}')
    assert info["n_windows"] == 3 and n_rows == 3 * 8 * 6
    db = sqlite3.connect(path)
    got = db.execute(READ_SQL % "gpud_metrics_v0_5").fetchall()
    db.close()
    times = sorted({r[0] for r in got})
    assert len(times) == 3 and all(t0 <= t <= t1 + 2 for t in times), (t0, times, t1)
    x = rows.astype(np.float64)
    want = _want(x, W, thr, 0, 3, 0)
    vals = {(t, nm): v for t, _, nm, _, v in got}
    for k, t in enumerate(times):
        for f, name in enumerate(POLL_METRICS):
            for op in ALL_OPS:
                v, w = vals[(t, g.window_metric_name(name, op))], float(want[op][f, k])
                assert (abs(v - w) <= 1e-6 * max(abs(w), 1.0)) if op in ("mean", "ema") else v == w, (name, op, k)
    poller.close()
    ring.close()


@pytest.mark.gpu
def test_temperature_component_metrics(ctx, store):
    st, path = store
    L = g.lib()
    xid = g.capi.Component(ctx, "accelerator-nvidia-error-xid")
    with pytest.raises(g.GpudError) as e:
        xid.set_metrics_store(st)
    assert e.value.code == -1
    xid.close()
    try:
        comp = g.capi.Component(ctx, "accelerator-nvidia-temperature")
    except g.GpudError as e:
        pytest.skip("temperature component unavailable: %s" % e)
    comp.set_metrics_store(st, "window_metrics")
    for _ in range(2000):
        comp.check()
    h = comp.ring_handle(0)
    assert L.gpud_ring_reduce(h) == 0
    red = {}
    for op in ALL_OPS:
        dt = np.uint32 if op == "n_over" else np.float64
        a = np.empty((8, 2), dtype=dt)
        assert L.gpud_ring_read(h, g.OPS[op], C.c_void_p(a.ctypes.data), a.nbytes) == 0
        red[op] = a
    db = sqlite3.connect(path)
    rows = db.execute(READ_SQL % "window_metrics").fetchall()
    assert len(rows) == 2 * 8 * 6
    times = sorted({r[0] for r in rows})
    assert len(times) == 2 and times[0] < times[1]
    for t, c, nm, lab, v in rows:
        k = times.index(t)
        assert set(json.loads(lab)) == {"uuid"} and lab.startswith('{"uuid":"')
        f = [i for i, m in enumerate(POLL_METRICS) if nm.startswith(m + "_window_")]
        assert len(f) == 1 and c == POLL_COMPONENTS[f[0]], (c, nm)
        op = nm[len(POLL_METRICS[f[0]] + "_window_"):]
        w = float(red[op][f[0], k])
        assert (abs(v - w) <= 1e-6 * max(abs(w), 1.0)) if op in ("mean", "ema") else v == w, (nm, k)
    comp.set_metrics_store(None)                                 # detached: the component writes nothing more
    for _ in range(1000):
        comp.check()
    assert db.execute("SELECT COUNT(*) FROM window_metrics").fetchone()[0] == 2 * 8 * 6
    db.close()
    comp.close()
