"""Streaming drain vs whole-ring reduce on one B200: prints one JSON line (and writes it to --out when given).

  (a) full drain   512 fields x 2^20 samples (the survey stream of tests/synth_device.py), W = 1000: gpud_ring_drain of every complete
                   window (1048 on the first fill) vs gpud_ring_reduce + six gpud_ring_read of the same ring.  Before every repeat the whole
                   stream is pushed again (untimed), so each drain finds 1047 or 1048 new windows (the window that straddles the
                   overwritten edge is lost).
  (b) steady state after each push of 32 768 rows: the drain of the 32 or 33 windows they complete vs reduce + six reads of the ring.
  (c) configs[1] live second: 64 fields x 1 M samples, 10 000 uint32 rows pushed per second: push + drain vs push + reduce + six reads.
Times are host ms around the C call, which ends in a stream synchronise (reads and drain copy into preallocated host arrays); warm-up
repeats are discarded, the spread is over --repeats.  Every drain's windows are checked against the C oracle (coracle.windows_fields) on
the same stream slice for a subset of fields: selections and n_over bit-exact, mean at 1e-6 relative, EMA where the oracle's seed is the
drain's (a drain after a loss restarts the EMA at its first window; (b) and (c) continue it, so their EMA is not compared here)."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

OPS6 = ("min", "max", "mean", "ema", "p99", "n_over")


def card_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                             timeout=30).stdout.strip()
        name, limit = [s.strip() for s in out.split(",")[:2]]
        return name, limit
    except Exception as ex:
        return None, "unknown (%s)" % type(ex).__name__


def spread(ts):
    a = np.asarray(ts) * 1e3
    return {"median_ms": float(np.median(a)), "min_ms": float(a.min()), "max_ms": float(a.max()), "n": int(a.size)}


class Raw:
    """the C calls with preallocated host buffers (what a cgo caller pays, without numpy allocation in the timed region)"""

    def __init__(self, g, ring, F, max_windows, nw_reduce):
        self.L, self.h, self.F, self.mw = g.lib(), ring._h, F, max_windows
        self.f64 = np.empty((5, F, max_windows), dtype=np.float64)
        self.nov = np.empty((F, max_windows), dtype=np.uint32)
        self.ms = np.empty((max_windows,), dtype=np.int64)
        self.info = g.DrainInfo()
        self.red = [np.empty((F, nw_reduce), dtype=np.uint32 if op == "n_over" else np.float64) for op in OPS6]
        for a in (self.f64, self.nov, self.ms, *self.red):
            a.fill(0)                                            # touch the pages outside the timed region

    def drain(self):
        t0 = time.perf_counter()
        rc = self.L.gpud_ring_drain(self.h, self.mw, C.c_void_p(self.f64.ctypes.data), C.c_void_p(self.nov.ctypes.data),
                                    C.c_void_p(self.ms.ctypes.data), C.byref(self.info))
        t = time.perf_counter() - t0
        assert rc == 0, rc
        n = self.info.n_windows
        out = {k: self.f64[i][:, :n] for i, k in enumerate(OPS6[:5])}
        out["n_over"] = self.nov[:, :n]
        return t, self.info.as_dict(), out

    def reduce_read(self):
        t0 = time.perf_counter()
        assert self.L.gpud_ring_reduce(self.h) == 0
        for i, a in enumerate(self.red):
            assert self.L.gpud_ring_read(self.h, i, C.c_void_p(a.ctypes.data), a.nbytes) == 0
        return time.perf_counter() - t0


class Mirror:
    """host copy of the pushed stream for a subset of fields, addressed by stream index (only the newest `keep` samples are kept)"""

    def __init__(self, n_fields, keep):
        self.buf = np.empty((0, n_fields)), 0
        self.keep = keep

    def push(self, rows):
        b, start = self.buf
        b = np.concatenate([b, rows])
        drop = max(0, b.shape[0] - self.keep)
        self.buf = b[drop:], start + drop

    def slice(self, a, b):
        buf, start = self.buf
        assert a >= start, (a, start)
        return buf[a - start:b - start]


def verify(got, info, mirror, sub, W, thr, ema_seeded):
    from oracle import coracle
    k0, n = info["first_window"], info["n_windows"]
    x = mirror.slice(k0 * W, (k0 + n) * W)
    want = coracle.windows_fields(np.ascontiguousarray(x.T), W, thr[sub])
    for k in ("min", "max", "p99"):
        assert np.array_equal(got[k][sub].view(np.uint64), want[k].view(np.uint64)), k
    assert np.array_equal(got["n_over"][sub], want["n_over"])
    keys = ("mean", "ema") if ema_seeded else ("mean",)
    for k in keys:
        err = np.abs(got[k][sub] - want[k])
        assert np.all(err <= 1e-6 * np.maximum(np.abs(want[k]), np.abs(x).max())), k
    return {"windows": n, "fields": len(sub), "ema_compared": ema_seeded}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default="")
    a = ap.parse_args()

    import torch
    import gpud_b200 as g
    import synth_device as sd

    name, limit = card_info()
    dev = torch.device("cuda:0")
    ctx = g.Context([0])
    res = {"tool": "tools/bench_drain.py", "card": name or torch.cuda.get_device_name(0), "power_limit": limit, "repeats": a.repeats,
           "warmup": a.warmup}

    # ---- (a) + (b): 512 x 2^20, W = 1000 ----
    F, CAP, W, SEED = 512, 1 << 20, 1000, 1234
    sub = np.arange(0, F, 16)                                    # 32 fields checked against the oracle (every kind of gauge and the counters)
    thr = sd.thresholds("survey", F, CAP, SEED)
    stream = torch.empty((CAP, F), dtype=torch.float64, device=dev)
    t0 = 0
    for x, n in sd.chunks("survey", F, CAP, 1 << 16, SEED, dev):
        stream[t0:t0 + n] = x
        t0 += n
    torch.cuda.synchronize()
    host_sub = stream[:, torch.as_tensor(sub, device=dev)].cpu().numpy()
    ring = g.Ring(ctx, F, CAP, W, thresholds=thr)
    mirror = Mirror(len(sub), CAP + 4 * W)
    nw_red = -(-CAP // W)
    raw = Raw(g, ring, F, nw_red, nw_red)

    def push_rows(lo, hi):
        ring.push_device(stream[lo:hi].data_ptr(), hi - lo)
        ring.sync()
        mirror.push(host_sub[lo:hi])

    drain_t, red_t, checks, nws = [], [], [], []
    for rep in range(a.warmup + a.repeats):
        push_rows(0, CAP)
        order = (0, 1) if rep % 2 == 0 else (1, 0)
        for which in order:
            if which == 0:
                t, info, got = raw.drain()
                assert info["n_windows"] in (1047, 1048) and info["n_lost"] == (0 if rep == 0 else 1), info
                nws.append(info["n_windows"])
                checks.append(verify(got, info, mirror, sub, W, thr, ema_seeded=True))
                if rep >= a.warmup:
                    drain_t.append(t)
            else:
                t = raw.reduce_read()
                if rep >= a.warmup:
                    red_t.append(t)
    res["a_full_drain"] = {"shape": "512 fields x 2^20 samples, W = 1000, survey stream", "windows_per_drain": sorted(set(nws)),
                           "drain": spread(drain_t), "reduce_plus_six_reads": spread(red_t),
                           "drain_over_reduce": float(np.median(drain_t) / np.median(red_t)), "verified_drains": len(checks)}

    step = 32768
    drain_t, red_t, nws, pos = [], [], [], 0
    for rep in range(a.warmup + a.repeats):
        lo = pos % CAP
        hi = lo + step
        push_rows(lo, hi)
        pos += step
        t, info, got = raw.drain()
        assert info["n_lost"] == 0 and info["n_pending"] == 0 and info["n_windows"] in (32, 33), info
        verify(got, info, mirror, sub, W, thr, ema_seeded=False)
        t2 = raw.reduce_read()
        if rep >= a.warmup:
            drain_t.append(t)
            red_t.append(t2)
            nws.append(info["n_windows"])
    res["b_steady_state"] = {"push_rows": step, "windows_per_drain": sorted(set(nws)), "drain": spread(drain_t), "reduce_plus_six_reads": spread(red_t),
                             "reduce_over_drain": float(np.median(red_t) / np.median(drain_t))}
    ring.close()
    del stream
    torch.cuda.empty_cache()

    # ---- (c): BASELINE configs[1], 64 fields x 1 M samples, one second of 10 kHz polls per step ----
    F1, N1, ROWS = 64, 1000000, 10000
    thr1 = sd.thresholds("survey", F1, N1, SEED)
    r1 = g.Ring(ctx, F1, N1, W, thresholds=thr1)
    sd.fill_ring(r1, "survey", F1, N1, SEED, dev, chunk=1 << 17)
    raw1 = Raw(g, r1, F1, N1 // W, N1 // W)
    raw1.drain()                                                 # the 1000 windows of the fill
    rng = np.random.default_rng(5)
    mirror1 = Mirror(F1, 4 * ROWS)
    push_t, drain_t, red_t = [], [], []
    for rep in range(a.warmup + a.repeats):
        rows = rng.integers(30, 90, (ROWS, F1)).astype(np.uint32)
        t0 = time.perf_counter()
        r1.push_raw(rows)
        tp = time.perf_counter() - t0
        mirror1.push(rows.astype(np.float64))
        t, info, got = raw1.drain()
        assert info["n_windows"] == 10 and info["n_lost"] == 0, info
        verify(got, info, _Offset(mirror1, N1), np.arange(F1), W, thr1, ema_seeded=False)
        t2 = raw1.reduce_read()
        if rep >= a.warmup:
            push_t.append(tp)
            drain_t.append(t)
            red_t.append(t2)
    res["c_live_second"] = {"shape": "64 fields x 1 M samples, W = 1000; 10 000 uint32 rows per step", "push": spread(push_t), "drain": spread(drain_t),
                            "reduce_plus_six_reads": spread(red_t),
                            "push_plus_drain_ms": float(np.median(np.asarray(push_t) + np.asarray(drain_t)) * 1e3)}
    r1.close()
    ctx.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


class _Offset:
    """a Mirror whose first pushed row is stream index `base` (the ring was filled before the mirror started)"""

    def __init__(self, m, base):
        self.m, self.base = m, base

    def slice(self, a, b):
        buf, start = self.m.buf
        return buf[a - self.base - start:b - self.base - start]


if __name__ == "__main__":
    main()
