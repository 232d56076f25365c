#!/usr/bin/env python3
"""bench.py — counter-samples/sec of the telemetry hot path (BASELINE.json metric) on N B200s of one node.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
  N > 1:  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Workload (config.workload, BASELINE configs[3] per GPU): 512 fields x 1 Mi-sample f64 ring (4 GiB, >> the 126 MB L2, so
every step streams from HBM), tumbling W = 1000 windows, all six aggregates fused (min/max/mean/EMA/p99/n_over).  The
stream is the one SURVEY.md 8(d) defines (tests/synth_device.py "survey": gauges base + A sin + sigma N(0,1) with 0.1 %
spikes over the threshold, every 8th field a monotone counter), generated on the device and appended through the real
append kernel.  A "step" = one pass of the hot path over the whole ring: the fused window-reduce kernel + the EMA carry kernel;
at N > 1 every step also packs the GPU's 128-byte NVLink/fabric record, all-gathers it over NCCL and evaluates the box verdict
on a side stream (the exchange has no data dependency on the reduce).  Weak scaling: every GPU owns its own ring.

`value`    whole-job samples/s with the ring already resident in HBM (CUDA events on the launch stream, max over ranks).
`e2e`      same metric through the C ABI from pinned HOST rows: push (H2D + append kernel) + reduce + D2H of every aggregate, all
           inside the timed region; the rows cross PCIe as uint32 ("u32 transport": NVML getters return uint32, the append
           kernel widens to f64); `e2e_f64` is the same with rows already widened on the host.
`roofline` algorithmic bytes (8 B/sample) / the fused kernel's CUDA-event time on the survey stream, against
           MEASURED_PEAKS.json hbm_gbs; `roofline.by_shape` repeats kernel ms + frac for other stream shapes (tie-heavy gauges take
           a slower selection path), `range` is the whole-ring (W = CAP) order statistic of configs[3].
`verify`   the WHOLE 512 x 1 Mi result of the last timed step against the C oracle (bit-exact selections and counts, max relative
           error of mean / EMA), and the W = CAP result the same way.
`--dump-outputs DIR`  the six [512][1049] aggregates of the last timed step (rank 0's ring) as DIR/<op>.npy, float64 (n_over
           widened exactly), 26 MB in all.  The stream is seeded, so two builds run with the same arguments can be compared
           output for output.
`cpu_baseline` / `--impl reference`: the C oracle (oracle/oracle.c, kind "port": the Go reference cannot be built here and has no
           windowed aggregation at all) rebuilt -O3 -march=native on this host, on the CPUs this process may really use
           (affinity and cgroup quota, not `nproc`), bounded sample, rank 0 only.
"""
import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

F, CAP, W = 512, 1 << 20, 1000
SEED = 0x67707564          # "gpud"; + rank per GPU (SURVEY 8d)
METRIC = "counter-samples/sec"
FALLBACK_HBM_GBS = 6650.0
SHAPES = ("survey", "uniform", "mw", "temp", "const", "walk")
SHAPE_NOTE = {"survey": "SURVEY 8(d) mix: gauges + 0.1 % spikes + every 8th field a monotone counter", "uniform": "white noise in [30, 90)",
              "mw": "integer mW readings uniform in [30000, 90000)", "temp": "integer degrees C uniform in [30, 90)", "const": "flat gauge",
              "walk": "integer random walk"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback"


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of one k_window_reduce launch on this workload, from the committed
    `ncu --set full` capture (profiles/window_reduce_traffic.json, written by tools/ncu_summary.py); None if absent.
    A constant of that capture, not measured in this run (ncu cannot run inside a timed bench)."""
    p = os.path.join(ROOT, "profiles", "window_reduce_traffic.json")
    try:
        d = json.load(open(p))
        return float(d["dram_bytes_read"]) + float(d["dram_bytes_write"])
    except Exception:
        return None


class ClockSampler:
    """SM clock and throttle reasons sampled through NVML every 5 ms during the timed region (the recipe's clocks line;
    NVML instead of the nvidia-smi CLI because the timed region lasts tens of milliseconds)."""

    def __init__(self, index):
        self.index, self.sm, self.reasons, self.max_mhz, self._stop, self._t = index, [], set(), None, False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4, "hw_power_brake": 0x80}
        while not self._stop:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        if self.nv is not None:
            self._t = threading.Thread(target=self._loop, daemon=True)
            self._t.start()

    def stop(self):
        self._stop = True
        if self._t:
            self._t.join(timeout=1.0)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.sm), "source": "nvml"}


def cpu_stream(fields):
    """the survey stream for `fields` fields x CAP samples, field-major float64, generated on the host"""
    import torch
    import synth_device as sd
    ring = np.empty((fields, CAP), dtype=np.float64)
    t0 = 0
    for x, n in sd.chunks("survey", fields, CAP, 1 << 16, SEED, torch.device("cpu")):
        ring[:, t0:t0 + n] = x.numpy().T
        t0 += n
    return ring, sd.thresholds("survey", fields, CAP, SEED)


def cpu_leg(steps, warmup, fields, ring=None, thr=None):
    """Times the C oracle on a bounded sample of the same workload: `fields` fields x CAP samples per step."""
    from oracle import coracle
    note = coracle.use_native()
    cpus = coracle.host_cpus()
    if ring is None:
        ring, thr = cpu_stream(fields)
    cores = cpus["threads_used"]
    for _ in range(warmup):
        coracle.windows_fields(ring[: max(1, fields // 8)], W, thr[: max(1, fields // 8)], threads=cores)
    t0 = time.perf_counter()
    for _ in range(steps):
        coracle.windows_fields(ring, W, thr, threads=cores)
    dt = (time.perf_counter() - t0) / steps
    v = fields * CAP / dt
    return {"value": v, "unit": "samples/s", "cores": cores, "kind": "port",
            "sample": "%d of 512 fields x 1Mi samples per step, survey stream (C oracle oracle/oracle.c, pthreads over fields)" % fields,
            "achieved_GBps": v * 8 / 1e9, "build": note, "host_cpus": cpus}, dt


def dump_outputs(d, got):
    """what a caller of the reduce receives, one .npy per aggregate; float64 holds every uint32 n_over exactly"""
    os.makedirs(d, exist_ok=True)
    for k, v in got.items():
        np.save(os.path.join(d, k + ".npy"), v.astype(np.float64))


def verify_windows(got, ring_host, thr, coracle):
    """the whole [F][nw] result against the C oracle on the same samples: exact selections / counts, max relative error of the float ones"""
    want = coracle.windows_fields(ring_host, W, thr)
    out = {"fields": int(ring_host.shape[0]), "windows_per_field": int(want["min"].shape[1]), "samples": int(ring_host.size)}
    exact = True
    for k in ("min", "max", "p99"):
        same = bool(np.array_equal(got[k].view(np.uint64), want[k].view(np.uint64)))
        out[k + "_bit_exact"] = same
        exact &= same
    out["n_over_exact"] = bool(np.array_equal(got["n_over"].astype(np.uint64), want["n_over"].astype(np.uint64)))
    out["n_over_total"] = int(want["n_over"].astype(np.int64).sum())
    exact &= out["n_over_exact"]
    scale = np.abs(ring_host).max(axis=1, keepdims=True)
    for k in ("mean", "ema"):
        err = np.abs(got[k] - want[k])
        out[k + "_max_rel_err"] = float(np.max(err / np.maximum(np.abs(want[k]), 1e-300)))
        out[k + "_max_err_over_field_scale"] = float(np.max(err / np.maximum(scale, 1e-300)))
    out["float_tolerance"] = 1e-6
    out["ok"] = bool(exact and out["mean_max_rel_err"] <= 1e-6 and out["ema_max_rel_err"] <= 1e-6)
    return out


def verify_range(got, ring_host, thr, alpha, coracle):
    """the W = CAP aggregates of every field against the oracle run with one window of CAP samples"""
    want = coracle.windows_fields(ring_host, CAP, thr, alpha=alpha)
    out = {}
    exact = True
    for k in ("min", "max", "p99"):
        same = bool(np.array_equal(got[k].view(np.uint64), want[k][:, 0].view(np.uint64)))
        out[k + "_bit_exact"] = same
        exact &= same
    out["n_over_exact"] = bool(np.array_equal(got["n_over"].astype(np.uint64), want["n_over"][:, 0].astype(np.uint64)))
    exact &= out["n_over_exact"]
    for k in ("mean", "ema"):
        out[k + "_max_rel_err"] = float(np.max(np.abs(got[k] - want[k][:, 0]) / np.maximum(np.abs(want[k][:, 0]), 1e-300)))
    out["ok"] = bool(exact and out["mean_max_rel_err"] <= 1e-6 and out["ema_max_rel_err"] <= 1e-6)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-fields", type=int, default=0, help="fields in the CPU sample (0 = auto, about 10-30 s of CPU work)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-scan", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--no-shapes", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the aggregates of the last timed step to DIR/<op>.npy")
    a = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    warmup = max(a.warmup, 3) if a.impl == "b200" else a.warmup
    config = {"workload": "ring 512 fields x 1Mi f64 samples per GPU (4 GiB), W=1000 tumbling, fused min/max/mean/ema/p99/n_over",
              "samples": "synthetic SURVEY 8(d) stream: gauges base + A sin(2 pi t / P) + sigma N(0,1) (temperature / power / utilisation), 0.1 % spikes over "
                         "the threshold, every 8th field a monotone counter; float64 in the ring",
              "n_fields": F, "capacity": CAP, "window": W, "parallelism": "one ring per GPU, no data-path collective (weak)",
              "l2": "input 4 GiB per GPU >> 126 MB L2; every step re-streams HBM"}

    if a.impl == "reference":
        if a.dump_outputs:
            ap.error("--dump-outputs writes the device result: --impl b200 only")
        # The reference's own CPU path for this metric does not exist (no windowed aggregation in gpud) and Go cannot be
        # built here; the timed arm is the C oracle port with every CPU this process may use.  Rank 0 only.
        if rank != 0:
            return 0
        fields = a.cpu_fields or 128
        cpu, dt = cpu_leg(max(1, a.steps), a.warmup, fields)
        line = {"impl": "reference", "metric": METRIC, "value": cpu["value"], "unit": "samples/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config, "cpu_baseline": cpu,
                "e2e": {"value": cpu["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    import torch
    import gpud_b200 as g
    import synth
    import synth_device as sd

    if world > 1:
        import torch.distributed as dist
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"        # the version banner goes to stdout; this program prints one JSON line there
        # the only collective of the step is a 128-byte-per-rank all-gather on the side stream; the persistent reduce grid leaves it ONE
        # CTA slot (gpud_ring_set_cta_reserve).  Between two GPUs NCCL would otherwise open one channel - one CTA - per NVLink; the
        # surplus CTAs only get a slot when a reduce kernel drains and then delay the next one's last CTA (measured at N = 2:
        # 0.776 ms per step against 0.728 at N = 1).
        os.environ.setdefault("NCCL_MAX_CTAS", "1")
        os.environ.setdefault("NCCL_MIN_CTAS", "1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    ctx = g.Context([local])
    seed = SEED + rank
    thr = sd.thresholds("survey", F, CAP, seed)
    ring = g.Ring(ctx, F, CAP, W, thresholds=thr, dev=local)
    stream = torch.cuda.Stream(device=dev)            # a real (non-NULL) stream: the library launches on it and torch events time it
    side = torch.cuda.Stream(device=dev)              # the fabric exchange of N > 1 runs here, concurrently with the reduce
    torch.cuda.set_stream(stream)
    ring.set_stream(stream.cuda_stream)
    assert stream.cuda_stream != 0
    if world > 1:
        ring.set_cta_reserve(1)                       # one CTA slot for the side stream's kernels (include/gpud_b200.h)
    peak, how = peaks()
    do_verify = rank == 0 and not a.no_verify
    nw = (CAP + W - 1) // W

    # ---- other stream shapes (N = 1 only): kernel ms of the fused reduce and of the W = CAP range call on each ----
    by_shape, range_by_shape = {}, {}
    reps = 10

    def time_shape(ring, shape):
        for _ in range(3):
            ring.reduce()
        ks = []
        for _ in range(reps):
            ring.reduce()
            ks.append(ring.kernel_ms()[0])
        k = float(np.mean(ks))
        by_shape[shape] = {"kernel_ms": k, "GBps": F * CAP * 8 / (k * 1e-3) / 1e9, "frac": F * CAP * 8 / (k * 1e-3) / 1e9 / peak, "stream": SHAPE_NOTE[shape]}
        ring.reduce_range(0)
        rs, hs = [], []
        for _ in range(5):
            t0 = time.perf_counter()
            ring.reduce_range(0)
            hs.append((time.perf_counter() - t0) * 1e3)
            rs.append(ring.range_stats())
        dev_ms = float(np.mean([r[1] for r in rs]))
        range_by_shape[shape] = {"device_ms": dev_ms, "pass_ms": float(np.mean([r[0] for r in rs])), "host_call_ms": float(np.median(hs)),
                                 "frac": F * CAP * 8 / (dev_ms * 1e-3) / 1e9 / peak, "fields_redone_by_radix_select": int(rs[-1][2]),
                                 "why": dict(ring.range_open_reasons)}

    if world == 1 and not a.no_shapes:
        for shape in SHAPES[1:]:
            r2 = g.Ring(ctx, F, CAP, W, thresholds=sd.thresholds(shape, F, CAP, seed), dev=local)
            r2.set_stream(stream.cuda_stream)
            sd.fill_ring(r2, shape, F, CAP, seed, dev)
            time_shape(r2, shape)
            r2.close()

    # ---- the benched stream, resident in HBM (and a host copy on rank 0 for the oracle) ----
    ring_host = np.empty((F, CAP), dtype=np.float64) if do_verify else None
    sd.fill_ring(ring, "survey", F, CAP, seed, dev, host_copy=ring_host)
    if world == 1 and not a.no_shapes:
        time_shape(ring, "survey")

    # fabric leg (N > 1): 128-byte summary per GPU, all-gather over NCCL, verdict kernel - all on the side stream
    fab_send = torch.zeros(128, dtype=torch.uint8, device=dev)
    fab_all = torch.zeros(128 * world, dtype=torch.uint8, device=dev)
    raw = g.FabricRaw()
    raw.gpu_index, raw.nvlink_supported, raw.system_expected_nvlink, raw.n_links = rank, 1, 1, 18
    for i in range(18):
        raw.link_feature_enabled[i] = 1
    for j in range(16):
        raw.p2p_status[j] = 0 if (j < world and j != rank) else 0xFF
    raw.fabric_valid, raw.fabric_state, raw.fabric_summary, raw.fabric_health_mask = 1, 3, 1, 0xAA

    def step():
        ring.reduce()
        if world > 1:
            with torch.cuda.stream(side):
                ctx.fabric_pack(raw, fab_send.data_ptr(), dev=local, stream=side.cuda_stream)
                dist.all_gather_into_tensor(fab_all, fab_send)

    def join_side():
        if world > 1:
            stream.wait_stream(side)                  # every exchange of the timed steps completes inside the timed region

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warmup):
        step()
    join_side()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(a.steps):
        step()
    join_side()
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    # the result of the last timed step, before anything else touches the ring
    do_dump = rank == 0 and a.dump_outputs
    got = {k: ring.read(k) for k in g.OPS} if do_verify or do_dump else None
    if do_dump:
        dump_outputs(a.dump_outputs, got)
    # per-kernel device time of the dominant kernel: the same step K more times, reading the library's own events
    kms = []
    for _ in range(a.steps):
        ring.reduce()
        kms.append(ring.kernel_ms())
    # per-step spread (N > 1): 200 further steps with an event after every step, max over ranks per step
    per_step = None
    if world > 1:
        n_ps = 200
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(n_ps + 1)]
        barrier()
        evs[0].record()
        for i in range(n_ps):
            step()
            evs[i + 1].record()
        join_side()
        barrier()
        d = torch.tensor([evs[i].elapsed_time(evs[i + 1]) for i in range(n_ps)], dtype=torch.float64, device=dev)
        dist.all_reduce(d, op=dist.ReduceOp.MAX)
        d = d.cpu().numpy()
        per_step = {"steps": n_ps, "median_ms": float(np.median(d)), "p95_ms": float(np.percentile(d, 95)), "max_ms": float(d.max()),
                    "note": "reduce + carry on the main stream, max over ranks per step; the fabric exchange overlaps on the side stream"}
        v = ctx.fabric_verdict(fab_all.data_ptr(), world, world, dev=local)
        assert v.nvlink_health == 0 and v.active == world, v.as_dict()
        t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms_step = ms_total / a.steps
    samples_step = F * CAP * world
    value = samples_step / (ms_step * 1e-3)
    k_reduce = float(np.mean([k[0] for k in kms]))
    k_carry = float(np.mean([k[1] for k in kms]))
    achieved = F * CAP * 8 / (k_reduce * 1e-3) / 1e9

    # ---- the W = CAP order statistic (the other half of configs[3]) on the benched stream ----
    ring.reduce_range(0)
    rs, hs = [], []
    for _ in range(5):
        t0 = time.perf_counter()
        rgot = ring.reduce_range(0)
        hs.append((time.perf_counter() - t0) * 1e3)
        rs.append(ring.range_stats())
    r_dev = float(np.mean([r[1] for r in rs]))
    rng_sec = {"workload": "p99 (+ min/max/mean/ema/n_over) over the whole ring, W = CAP = 1 Mi samples x 512 fields", "kernel": "k_range_pivots + k_window_reduce<range> + k_ema_carry + k_range_finish",
               "hbm_passes": 1, "device_ms": r_dev, "pass_ms": float(np.mean([r[0] for r in rs])), "host_call_ms": float(np.median(hs)),
               "achieved": F * CAP * 8 / (r_dev * 1e-3) / 1e9, "unit": "GB/s", "frac": F * CAP * 8 / (r_dev * 1e-3) / 1e9 / peak,
               "fields_redone_by_radix_select": int(rs[-1][2]), "why": dict(ring.range_open_reasons), "by_shape": range_by_shape or None}

    # ---- verification of what was timed: the whole result of the last timed step, and the W = CAP result, against the C oracle ----
    verify = None
    if do_verify:
        from oracle import coracle
        t0 = time.perf_counter()
        verify = verify_windows(got, ring_host, thr, coracle)
        verify["range"] = verify_range(rgot, ring_host, thr, 2.0 / (W + 1.0), coracle)
        verify["oracle_seconds"] = time.perf_counter() - t0
        verify["ok"] = bool(verify["ok"] and verify["range"]["ok"])
        del got

    # ---- e2e: pinned host rows -> push (H2D + append) -> reduce -> D2H of all aggregates, every step ----
    # Headline e2e: the poller hands over RAW NVML samples in the getter's own type (uint32) through gpud_ring_push_raw; the
    # widening to float64 happens in the append kernel.  e2e_f64: the same stream already widened on the host (gpud_ring_push).
    e2e = e2e_f64 = None
    if not a.no_e2e:
        outs = {k: np.empty((F, nw), dtype=np.uint32 if k == "n_over" else np.float64) for k in g.OPS}
        d2h = sum(o.nbytes for o in outs.values())

        def run_e2e(host, rows_chunk, dtype_code, esz, steps):
            def e2e_step():
                for _ in range(CAP // rows_chunk):
                    ring.push_raw_ptr(host.data_ptr(), rows_chunk, dtype_code)
                ring.reduce()
                for k in g.OPS:
                    ctx._check(ring._L.gpud_ring_read(ring._h, g.OPS[k], C.c_void_p(outs[k].ctypes.data), outs[k].nbytes))
            e2e_step()
            barrier()
            t0 = time.perf_counter()
            e0.record()
            for _ in range(steps):
                e2e_step()
            e1.record()
            barrier()
            ms = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3) / steps
            if world > 1:
                t = torch.tensor([ms], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t.item())
            return {"value": samples_step / (ms * 1e-3), "unit": "samples/s", "h2d_bytes_per_step": F * CAP * esz, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms, "steps": steps, "h2d_GBps": F * CAP * esz / (ms * 1e-3) / 1e9}

        e2e_steps = max(2, min(a.steps, 5))
        host = torch.randint(30000, 90000, (1 << 19, F), dtype=torch.int32).pin_memory()        # 1 GiB pinned, pushed 2x per step = the whole ring
        e2e = run_e2e(host, 1 << 19, g.DTYPES["uint32"], 4, e2e_steps)
        e2e["transport"] = "u32"
        e2e["sample_dtype"] = "u32 transport: uint32 raw NVML counters (gpud_ring_push_raw) cross PCIe, widened to f64 on the device; arithmetic is f64"
        del host
        host = torch.randint(30000, 90000, (1 << 18, F), dtype=torch.int32).to(torch.float64).pin_memory()   # 1 GiB pinned, pushed 4x per step
        e2e_f64 = run_e2e(host, 1 << 18, g.DTYPES["float64"], 8, 2)
        e2e_f64["transport"] = "f64"
        e2e_f64["sample_dtype"] = "float64 widened on the host (gpud_ring_push)"
        del host

    cpu = None
    if rank == 0 and world == 1:
        fields = a.cpu_fields or 128
        cpu, _dt = cpu_leg(1, 1, fields, ring=ring_host[:fields] if ring_host is not None else None, thr=thr[:fields] if ring_host is not None else None)
    ring_host = None

    # ---- BASELINE configs[1]: 64 NVML fields x 10 kHz (100 s = 1 M polls), W = 1000, rank 0 at N = 1 only ----
    c1 = None
    if rank == 0 and world == 1 and not a.no_shapes:
        try:
            F1, N1 = 64, 1000000
            r1 = g.Ring(ctx, F1, N1, W, thresholds=sd.thresholds("survey", F1, N1, SEED), dev=local)
            r1.set_stream(stream.cuda_stream)
            sd.fill_ring(r1, "survey", F1, N1, SEED, dev, chunk=1 << 17)
            for _ in range(3):
                r1.reduce()
            ks = []
            for _ in range(20):
                r1.reduce()
                ks.append(r1.kernel_ms())
            k1 = float(np.mean([k[0] for k in ks]))
            rows = torch.randint(30, 90, (10000, F1), dtype=torch.int32).pin_memory()      # one second of polls at 10 kHz
            t0 = time.perf_counter()
            secs = 20
            for _ in range(secs):
                r1.push_raw_ptr(rows.data_ptr(), 10000, g.DTYPES["uint32"])
                r1.reduce()
                r1.sync()
            wall = (time.perf_counter() - t0) / secs
            c1 = {"workload": "64 fields x 10 kHz x 100 s (1 M polls, 512 MB), W = 1000 min/max/mean (all six aggregates computed)", "kernel_ms": k1,
                  "samples_per_s": F1 * N1 / (k1 * 1e-3), "GBps": F1 * N1 * 8 / (k1 * 1e-3) / 1e9, "frac": F1 * N1 * 8 / (k1 * 1e-3) / 1e9 / peak,
                  "live_second_ms": wall * 1e3, "live_headroom": 1.0 / wall,
                  "note": "live_second_ms = push one second of polls (10 000 rows, uint32) + reduce of the whole 100 s ring + sync; headroom = how many such 10 kHz "
                          "streams one GPU keeps up with"}
            r1.close()
        except Exception as ex:
            c1 = {"error": repr(ex)}

    # ---- secondary workload (BASELINE configs[2]): Xid/SXid scan of a 100 MiB synthetic dmesg buffer, rank 0 at N=1 only ----
    scan = None
    if rank == 0 and world == 1 and not a.no_scan:
        try:
            from oracle import coracle
            unit = synth.dmesg_buffer(4 << 20, hit_every=1000)
            buf = unit * 25
            d = torch.frombuffer(bytearray(buf), dtype=torch.uint8).to(dev)
            torch.cuda.synchronize()
            tot = []
            for _ in range(4):                                   # default: the scan's kernels as one overlapped launch chain, whole device time
                hits, n_units = ctx.kmsg_scan_device(d.data_ptr(), len(buf), cap=1 << 17, dev=local)
                tot.append(ctx.scan_kernel_ms(dev=local)[0])
            dev_ms = float(np.mean(tot[1:]))
            ctx.scan_phase_timing(True, dev=local)               # plain launches split by events, for the filter's own time
            ms = []
            for _ in range(4):
                ctx.kmsg_scan_device(d.data_ptr(), len(buf), cap=1 << 17, dev=local)
                ms.append(ctx.scan_kernel_ms(dev=local))
            ctx.scan_phase_timing(False, dev=local)
            filt, pre, mat = np.array(ms[1:]).mean(axis=0)
            harr = (g.XidHit * (1 << 17))()
            ctx.kmsg_scan_c(buf, harr, 1 << 17, dev=local)
            t0 = time.perf_counter()
            nh2, _ = ctx.kmsg_scan_c(buf, harr, 1 << 17, dev=local)
            e2e_s = time.perf_counter() - t0
            t0 = time.perf_counter()
            ch, _nl = coracle.scan_lines(buf)
            cpu_s = time.perf_counter() - t0
            same = [(h.line, h.kind, h.code) for h in ch] == [(h.unit_index, h.kind, h.code) for h in hits]
            scan = {"workload": "100 MiB synthetic dmesg (reference fixtures + noise + injected Xid/SXid lines)", "bytes": len(buf), "lines": n_units,
                    "hits": len(hits), "device_ms": dev_ms, "device_GBps": len(buf) / dev_ms / 1e6,
                    "device_frac_of_hbm_peak": len(buf) / dev_ms / 1e6 / peak, "phases_ms": {"filter": float(filt), "prefix": float(pre), "match": float(mat)},
                    "filter_kernel_ms": float(filt), "filter_frac_of_hbm_peak": len(buf) / float(filt) / 1e6 / peak,
                    "e2e_host_ms": e2e_s * 1e3, "e2e_GBps": len(buf) / e2e_s / 1e9, "cpu_oracle_ms": cpu_s * 1e3, "cpu_oracle_GBps": len(buf) / cpu_s / 1e9,
                    "cpu_threads": coracle.max_threads(), "hits_identical_to_oracle": bool(same and nh2 == len(hits))}
            # same buffer with the nccl / peermem matchers switched on (SURVEY 8f.1): four anchor words instead of two in the filter
            ebuf = synth.ext_buffer(4 << 20, hit_every=1000) * 25
            d2 = torch.frombuffer(bytearray(ebuf), dtype=torch.uint8).to(dev)
            etot = []
            for _ in range(4):
                ehits, _eu = ctx.kmsg_scan_device(d2.data_ptr(), len(ebuf), mode=g.SCAN_LINES | g.SCAN_EXT_MATCHERS, cap=1 << 18, dev=local)
                etot.append(ctx.scan_kernel_ms(dev=local)[0])
            ctx.scan_phase_timing(True, dev=local)
            ems = []
            for _ in range(3):
                ctx.kmsg_scan_device(d2.data_ptr(), len(ebuf), mode=g.SCAN_LINES | g.SCAN_EXT_MATCHERS, cap=1 << 18, dev=local)
                ems.append(ctx.scan_kernel_ms(dev=local))
            ctx.scan_phase_timing(False, dev=local)
            ech, _ = coracle.scan_lines(ebuf, ext=True)
            ef, ep, em = np.array(ems[1:]).mean(axis=0)
            scan["ext_matchers"] = {"bytes": len(ebuf), "hits": len(ehits), "nccl_hits": sum(h.kind == 3 for h in ehits),
                                    "peermem_hits": sum(h.kind == 4 for h in ehits), "device_ms": float(np.mean(etot[1:])), "filter_kernel_ms": float(ef),
                                    "hits_identical_to_oracle": [(h.line, h.kind, h.code) for h in ech] == [(h.unit_index, h.kind, h.code) for h in ehits]}
            del d2
            del d
        except Exception as ex:   # the scan leg must never cost the headline line
            scan = {"error": repr(ex)}

    # ---- real ingest (SURVEY 8f.3, BASELINE configs[1] shape): NVML getters -> pinned uint32 rows -> K1, rank 0 at N=1 only ----
    ingest = None
    if rank == 0 and world == 1 and not a.no_scan:
        try:
            iring = g.Ring(ctx, len(g.POLL_FIELDS), 1 << 16, 1000, thresholds=np.zeros(len(g.POLL_FIELDS)), dev=local)
            poller = g.Poller(ctx, iring, dev=local)
            poller.poll(200)
            poller.poll(5000)
            rows, sec = poller.last_rows()
            iring.reduce()
            iring.sync()
            ingest = {"source": "NVML getters (temperature, power, 3 clocks, 2 utilisations, memory used) via the library's poller",
                      "fields": len(g.POLL_FIELDS), "polls": int(rows.shape[0]), "polls_per_s": rows.shape[0] / sec,
                      "samples_per_s": rows.shape[0] * len(g.POLL_FIELDS) / sec,
                      "last_row": {k: int(v) for k, v in zip(g.POLL_FIELDS, rows[-1])}, "getter_failures": poller.errors()[0]}
            try:                                                 # GPM (gpm/gpm.go:65-149): one 250 ms sample interval under whatever is running
                gm = poller.gpm_metrics(250)
                ingest["gpm"] = {"supported": bool(gm.supported), "sample_s": gm.sample_seconds, "metrics": gm.as_dict() if gm.supported else None}
            except Exception as ex:
                ingest["gpm"] = {"error": repr(ex)}
            poller.close()
            iring.close()
        except Exception as ex:
            ingest = {"error": repr(ex)}

    ring.close()
    ctx.close()
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": a.steps, "warmup": warmup, "ms_per_step": ms_step,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
                "gpu_launches": (3 + (1 if world > 1 else 0)) * a.steps,   # window_reduce (specialised + generic tail) + ema_carry (+ fabric pack)
                "clocks": clocks, "e2e": e2e,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": ncu_traffic(),
                             "traffic_source": "profiles/window_reduce_traffic.json: one `ncu --set full` capture of this kernel on this workload (constant, not this run)",
                             "kernel": "k_window_reduce", "kernel_ms": k_reduce, "carry_kernel_ms": k_carry, "peak_source": how + " (MEASURED_PEAKS.json hbm_gbs, burst copy)"
                             if how == "measured" else "fallback 6650 GB/s (B200_PROFILING.md)", "algorithmic_bytes_per_launch": F * CAP * 8,
                             "stream": "survey", "by_shape": by_shape or None},
                "range": rng_sec, "verify": verify, "per_step": per_step,
                "cpu_baseline": cpu, "e2e_f64": e2e_f64, "configs1": c1, "scan": scan, "ingest": ingest}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
