"""GPU parity: the CUDA path behind the C ABI vs the oracle on the same inputs.  Run on the B200 box: pytest -m gpu.
Integer / byte / selection outputs are compared bit-exactly; mean and EMA at 1e-6 relative (oracle/SPEC.md)."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import fabric as OF
from oracle import pyoracle as O
import synth

pytestmark = pytest.mark.gpu

g = None


@pytest.fixture(scope="module")
def ctx():
    global g
    import gpud_b200 as _g
    g = _g
    c = g.Context([0])
    yield c
    c.close()


# ------------------------------------------------------------------------------------------------ scan
def _cmp_hits(got, want, extended=True):
    gd = [h.as_dict() for h in got]
    assert [(h["line"], h["kind"], h["code"]) for h in gd] == [(h["line"], h["kind"], h["code"]) for h in want]
    for a, b in zip(gd, want):
        assert a["device"] == b["device"], (a, b)
        assert a["offset"] == b["offset"], (a, b)
        assert a["event_type"] == b["event_type"], (a, b)
        assert a["actions"] == list(b["actions"]), (a, b)
        assert a["extended"] == b["extended"], (a, b)
        if b["extended"]:
            assert a["sub_code"] == b["sub_code"] and a["error_status"] == b["error_status"], (a, b)
            if "intrinfo" in b:
                assert a["intrinfo"] == b["intrinfo"] and a["link"] == b["link"] and a["unit"] == b["unit"][:39], (a, b)


def test_scan_golden_lines(ctx):
    lines = synth.hit_lines() + synth.EDGE_LINES
    buf = "\n".join(lines).encode()
    hits, n_units = ctx.kmsg_scan(buf)
    want = O.scan_lines(buf)
    assert n_units == buf.count(b"\n") + 1
    assert len(want) > 250
    _cmp_hits(hits, want)


def test_scan_each_golden_vector(ctx):
    """every reference test vector scanned as its own buffer (kmsg_test.go TestMatch etc.), incl. multi-line inputs"""
    G = synth.golden("xid_kmsg.json")
    for r in G["match"]["rows"]:
        buf = r["input"].encode()
        hits, _ = ctx.kmsg_scan(buf)
        want = O.scan_lines(buf)          # LINES semantics: a multi-line input is split, exactly like the oracle does
        _cmp_hits(hits, want)
    # the dmesg fixture: exactly 5 x (119, PCI:0000:9b:00)   kmsg_test.go:248-287
    buf = "\n".join(G["dmesg_xid_119"]["lines"]).encode()
    hits, _ = ctx.kmsg_scan(buf)
    assert [(h.code, h.device.decode()) for h in hits] == [(119, "PCI:0000:9b:00")] * 5


def test_xid_hit_message_is_build_message_of_the_match(ctx):
    """buildMessage (xid/health_state.go:130-169) for every hit of the golden lines, and the reference's own message tests that
    start from a kmsg line (health_state_test.go:318-362, 363-412, 505-562, 564-690)"""
    lines = synth.hit_lines() + synth.EDGE_LINES
    buf = "\n".join(lines).encode()
    hits, _ = ctx.kmsg_scan(buf)
    n = 0
    for h in hits:
        if h.kind != 1:
            continue
        raw = buf.split(b"\n")[h.unit_index]
        x = O.xid_match(raw)
        if x is None:                                  # multi-line fallen-off-the-bus records are compared in the raw-mode tests
            continue
        d = x.detail
        for uuid in ("", "GPU-test-uuid"):
            assert g.xid_hit_message(h, uuid) == O.xid_build_message(x.xid, d.sub_code, d.error_status, d.description, x.device, uuid), raw
        n += 1
    assert n > 200
    G = synth.golden("xid_messages.json")["from_lines"]
    for r in G["rows"]:
        hits, _ = ctx.kmsg_scan(r["line"].encode())
        assert len(hits) == 1, r["name"]
        h = hits[0]
        uuid = O.convert_bus_id_to_uuid(h.device.decode(), r["devices"])
        msg = g.xid_hit_message(h, uuid)
        for c in r["contains"]:
            assert c in msg, (r["name"], c, msg)
        if "sub_code" in r:
            assert ("%d.%d" % (h.code, r["sub_code"])) in msg
        if "event_type" in r:
            assert g.EVENT_NAMES[h.event_type] == r["event_type"]


def test_scan_raw_kmsg_header_fields_of_the_reference_calls(ctx):
    """the literal parseLine calls of pkg/kmsg/watcher_test.go:35-255 as /dev/kmsg records carrying an Xid line: priority, sequence and
    microsecond fields of the hit equal the asserted ones (negative priority / sequence, the very large timestamp)"""
    calls = synth.golden("pkg_kmsg.json")["parse_line_calls"]["rows"]
    recs = [r["input"].split(";", 1)[0] + ";NVRM: Xid (PCI:0000:05:00): 79, pid=1, GPU has fallen off the bus." for r in calls]
    buf = "\n".join(recs).encode()
    hits, n = ctx.kmsg_scan(buf, mode=g.SCAN_RAW_KMSG)
    want, wn = O.scan_raw_kmsg(buf)
    assert n == wn == len(recs) and len(hits) == len(want) == len(recs)
    for h, w, r in zip(hits, want, calls):
        assert (h.kmsg_priority, h.kmsg_seq, h.kmsg_usec) == tuple(w["kmsg"])
        for k, got in (("priority", h.kmsg_priority), ("sequence", h.kmsg_seq), ("usec", h.kmsg_usec)):
            if k in r:
                assert got == r[k], (r["input"], k)


def test_scan_multiline_record_raw_mode(ctx):
    """the multiline fallen-off-the-bus vector only matches when the record is one unit (RAW_KMSG continuation lines)"""
    rec = b"4,1,5,-;NVRM: The NVIDIA GPU 0000:18:00.0\n NVRM: (PCI ID: 10de:2901) installed in this system has\n NVRM: fallen off the bus and is not responding to commands.\n"
    hits, n = ctx.kmsg_scan(rec, mode=g.SCAN_RAW_KMSG)
    want, wn = O.scan_raw_kmsg(rec)
    assert n == wn
    assert [(h.code, h.device.decode()) for h in hits] == [(w["code"], w["device"]) for w in want] == [(79, "PCI:0000:18:00")]


def test_scan_synthetic_buffer(ctx):
    buf = synth.dmesg_buffer(3 << 20, hit_every=200)
    hits, n_units = ctx.kmsg_scan(buf)
    want = O.scan_lines(buf)
    assert n_units == buf.count(b"\n") + 1
    assert len(want) > 50
    _cmp_hits(hits, want)


def test_scan_raw_kmsg(ctx):
    buf = synth.raw_kmsg_buffer(4000)
    hits, n_units = ctx.kmsg_scan(buf, mode=g.SCAN_RAW_KMSG)
    want, wn = O.scan_raw_kmsg(buf)
    assert n_units == wn
    assert len(want) > 100
    gd = [h.as_dict() for h in hits]
    assert [(h["line"], h["kind"], h["code"], h["device"], h["offset"]) for h in gd] == \
           [(h["line"], h["kind"], h["code"], h["device"], h["offset"]) for h in want]
    assert [h["kmsg"] for h in gd] == [h["kmsg"] for h in want]
    assert [h["event_type"] for h in gd] == [h["event_type"] for h in want]


@pytest.mark.parametrize("buf", [b"", b"\n", b"\n\n\n", b"x", b"NVRM: Xid (PCI:0000:05:00): 79, a",
                                 b"NVRM: Xid (PCI:0000:05:00): 79, a\n", b"\nNVRM: Xid (PCI:0000:05:00): 79, a"])
def test_scan_edges(ctx, buf):
    hits, n_units = ctx.kmsg_scan(buf)
    want = O.scan_lines(buf)
    assert n_units == buf.count(b"\n") + 1
    _cmp_hits(hits, want)


def _cmp_ext(ctx, buf, hits, want):
    _cmp_hits(hits, want)
    for a, b in zip(hits, want):
        if b["kind"] >= 19:                              # line primitives of the stateful matchers: every capture span
            got = [buf[o:o + n] for o, n in ((a.dev_off, a.dev_len), (a.unit_name_off, a.unit_name_len), (a.pid_off, a.pid_len),
                                             (a.pname_off, a.pname_len), (a.inj_off, a.inj_len))]
            assert got == (b["spans"] or [b""] * 5), (a.as_dict(), b, got)
        if b["kind"] >= 3:
            assert a.dev_len == len(b["capture"]) and buf[a.dev_off:a.dev_off + a.dev_len] == b["capture"], (a.as_dict(), b)
            assert ctx.kmsg_message(a, buf) == b["message"], (a.as_dict(), b)
            comp, ev, _m, _g = O.EXT_BY_KIND[b["kind"]]
            L = ctx._L
            assert L.gpud_kmsg_event_name(b["kind"]).decode() == ev and L.gpud_kmsg_component(b["kind"]).decode() == comp


def test_scan_ext_matchers(ctx):
    """GPUD_SCAN_EXT_MATCHERS: the stateless line matchers of nccl / peermem / infiniband / cpu / os / disk (SURVEY 8f.1) ride
    the same scan; default mode is unaffected"""
    lines = synth.ext_lines() + synth.EXT_EDGE_LINES + synth.PRIM_EDGE_LINES + synth.hit_lines()[:40]
    for buf in ("\n".join(lines).encode(), synth.ext_buffer(2_000_000, hit_every=60)):
        hits, n_units = ctx.kmsg_scan(buf, mode=g.SCAN_LINES | g.SCAN_EXT_MATCHERS)
        want = O.scan_lines(buf, ext=True)
        assert n_units == buf.count(b"\n") + 1
        assert {h["kind"] for h in want} >= set(range(3, 25))
        _cmp_ext(ctx, buf, hits, want)
        _cmp_hits(ctx.kmsg_scan(buf)[0], O.scan_lines(buf))
    for l in lines:                                   # every vector as its own buffer
        b = l.encode()
        _cmp_ext(ctx, b, ctx.kmsg_scan(b, mode=g.SCAN_EXT_MATCHERS)[0], O.scan_lines(b, ext=True))


def test_scan_ext_matchers_fuzz(ctx):
    """20 000 mutated matcher lines (cut, spliced, glued, edited): every decision and capture must equal the regex oracle"""
    lines = synth.ext_fuzz_lines(20000, seed=99)
    buf = "\n".join(lines).encode()
    hits, n_units = ctx.kmsg_scan(buf, mode=g.SCAN_LINES | g.SCAN_EXT_MATCHERS, cap=1 << 17)
    want = O.scan_lines(buf, ext=True)
    assert n_units == len(lines) and len(want) > 5000
    _cmp_ext(ctx, buf, hits, want)


@pytest.mark.parametrize("seed,chunk", [(11, 1 << 30), (12, 997), (13, 50)])
def test_scan_stateful_matchers(ctx, seed, chunk):
    """os kernel-panic assembly and the memory OOM parser: scan primitives -> gpud_kmsg_stateful_feed == the reference's
    closures run line by line; the stream is scanned in pieces to exercise the carried state"""
    lines = [l.encode() for l in synth.stateful_stream(6000, seed=seed)]
    want = O.stateful_events(lines)
    assert sum(1 for e in want if e[1] == "os") >= 10 and sum(1 for e in want if e[1] == "memory") >= 10
    st = g.KmsgStateful()
    got = []
    for a in range(0, len(lines), chunk):
        part = lines[a:a + chunk]
        buf = b"\n".join(part)
        hits, n_units = ctx.kmsg_scan(buf, mode=g.SCAN_LINES | g.SCAN_EXT_MATCHERS)
        assert n_units == len(part)
        got += [(u + a, c, e, m) for u, c, e, m in st.feed(hits, buf, n_units)]
    st.close()
    assert got == want


def test_scan_stateful_golden_sequences(ctx):
    for seq in synth.stateful_sequences():
        lines = [l.encode() for l in seq]
        buf = b"\n".join(lines)
        hits, n_units = ctx.kmsg_scan(buf, mode=g.SCAN_EXT_MATCHERS)
        st = g.KmsgStateful()
        assert st.feed(hits, buf, n_units) == O.stateful_events(lines), seq
        st.close()


def test_scan_ext_golden_match_tables(ctx):
    """the components' Match(line) -> (eventName, message) tables, answered from the scan hits in the component's pattern order"""
    G = synth.golden("ext2_kmsg.json")
    for comp in ("infiniband", "cpu", "os", "disk"):
        for r in G[comp + ".match"]["rows"]:
            b = r["line"].encode()
            hits, _ = ctx.kmsg_scan(b, mode=g.SCAN_EXT_MATCHERS)
            mine = [h for h in hits if ctx._L.gpud_kmsg_component(h.kind).decode() == comp]
            got = (ctx._L.gpud_kmsg_event_name(mine[0].kind).decode(), ctx.kmsg_message(mine[0], b)) if mine else ("", "")
            assert got == (r["wantEvent"], r["wantMessage"]), (comp, r, got)


def test_scan_ext_matchers_raw_mode(ctx):
    recs = []
    ext = synth.ext_lines() + synth.EXT_EDGE_LINES
    for i, l in enumerate(ext):
        recs.append("%d,%d,%d,-;%s" % (i % 8, 100 + i, 1000 * i, l))
        if i % 3 == 0:
            recs.append(" SUBSYSTEM=pci\n DEVICE=+pci:0000:05:00.0")
        if i % 5 == 0:                                   # the two nccl literals split over a continuation line: `.` stops at \n
            recs.append("4,%d,%d,-;x segfault at 0\n in libnccl.so" % (900 + i, i))
            recs.append("4,%d,%d,-;y segfault at 0\n segfault at 1 in libnccl.so" % (950 + i, i))
    buf = "\n".join(recs).encode()
    hits, n_units = ctx.kmsg_scan(buf, mode=g.SCAN_RAW_KMSG | g.SCAN_EXT_MATCHERS)
    want, n_rec = O.scan_raw_kmsg(buf, ext=True)
    assert n_units == n_rec
    assert {h["kind"] for h in want} >= set(range(3, 19))
    _cmp_ext(ctx, buf, hits, want)
    for a, b in zip(hits, want):
        assert (a.kmsg_priority, a.kmsg_seq, a.kmsg_usec) == b["kmsg"]


def test_scan_ragged_offsets(ctx):
    """hit lines at every alignment relative to the 16-byte / 512-byte / 2048-byte load boundaries"""
    line = b"NVRM: Xid (PCI:0000:05:00): 79, GPU has fallen off the bus.\n"
    for pad in list(range(0, 40)) + [495, 500, 511, 512, 513, 2040, 2047, 2048, 2049]:
        buf = b"a" * pad + b"\n" + line + b"tail without newline"
        hits, n_units = ctx.kmsg_scan(buf)
        assert n_units == 3
        assert [(h.unit_index, h.code, h.unit_offset) for h in hits] == [(1, 79, pad + 1)], pad


def test_scan_anchor_prefilter_alignments(ctx):
    """the filter's pre-filter ('X' byte / first aligned word of "fallen off the bus") must flag every anchor wherever it falls
    relative to the 4 / 16 / 512 / 2048-byte boundaries, and the look-alikes ("called", "len 64", lone 'X') must stay silent"""
    lines = [b"NVRM: GPU 0000:29:00.0: GPU has fallen off the bus.", b"nvidia-nvswitch3: SXid (PCI:0000:05:00.0): 12028, Non-fatal, Link 32 egress",
             b"NVRM:   The NVIDIA GPU 0000:18:00.0 (PCI ID) has fallen off the bus and is not responding to commands.",
             b"fallen off the bus", b"SXid", b"XXid SXi called allen len 64 fall alle llen X fallen off the bu",
             # units longer than the 512-byte window the match kernel settles unit bounds in: the thread's own walk takes over
             b"x" * 300 + b" NVRM: Xid (PCI:0000:05:00): 79, pid=1, name=p" + b"y" * 400,
             b"N" * 270 + b"NVRM: GPU 0000:29:00.0: GPU has fallen off the bus." + b"f" * 290,
             b"SXid (PCI:0000:05:00.0): 1, x " + b"S" * 250 + b" SXid (PCI:0000:05:00.0): 12028, Non-fatal"]
    for line in lines:
        for pad in list(range(0, 36)) + [492, 495, 509, 510, 511, 512, 2030, 2044, 2045, 2046, 2047, 2048]:
            for lead in (b"a" * pad + b"\n", b"a" * pad):
                buf = lead + line + b"\nfallen off the called len X tail"
                hits, n_units = ctx.kmsg_scan(buf)
                assert n_units == buf.count(b"\n") + 1
                _cmp_hits(hits, O.scan_lines(buf))


def test_hit_json_matches_oracle(ctx):
    lines = synth.hit_lines()
    buf = "\n".join(lines).encode()
    hits, _ = ctx.kmsg_scan(buf)
    n = 0
    for h in hits:
        if h.kind != 1:
            assert ctx.hit_json(h) == str(h.code)
            continue
        line = buf[h.unit_offset:].split(b"\n", 1)[0]
        x = O.xid_match(line)
        assert ctx.hit_json(h, 1740327858) == O.xid_event_detail_json(x, 1740327858), line
        n += 1
    assert n > 200


def test_store_persists_xid_events(ctx, tmp_path):
    """SURVEY 8f.2: scan -> gpud_store_insert_xid_hits -> the reference's getEvents query returns exactly the events the xid
    component would have persisted (name, type, extra_info JSON with the xidErrorEventDetail payload), duplicates skipped"""
    import json
    import sqlite3
    try:
        st = g.Store(str(tmp_path / "gpud.state"))
    except g.GpudError as e:
        pytest.skip("no libsqlite3.so.0: %s" % e)
    G = synth.golden("store_sql.json")
    lines = synth.hit_lines()
    buf = "\n".join(lines).encode()
    hits, _ = ctx.kmsg_scan(buf)
    t = st.event_table("accelerator-nvidia-error-xid")
    now = 1740327858
    n_ins = st.insert_xid_hits(t, hits, fallback_unix=now)
    assert st.insert_xid_hits(t, hits, fallback_unix=now) == 0          # second pass: every event is found already (component.go:555-563)
    want = set()
    ev_names = {1: "Info", 2: "Warning", 3: "Critical", 4: "Fatal", 0: "Unknown"}
    for h in hits:
        if h.kind != 1:
            continue
        line = buf[h.unit_offset:].split(b"\n", 1)[0]
        x = O.xid_match(line)
        extra = "{" + '"data":' + O._go_json_str(O.xid_event_detail_json(x, now)) + ',"device_uuid":' + O._go_json_str(x.device) + "}"
        want.add((now, "error_xid", ev_names[x.detail.event_type], None, extra))
    db = sqlite3.connect(str(tmp_path / "gpud.state"))
    rows = list(db.execute(G["event_get"]["sql"].format(table=t), (0,)))
    assert n_ins == len(rows) == len(want) and set(rows) == want and len(want) > 150
    for r in rows[:20]:
        d = json.loads(r[4])
        assert set(d) == {"data", "device_uuid"} and "xid" in json.loads(d["data"])
    db.close()
    st.close()


def test_classify_entry(ctx):
    """gpud_xid_classify on hand-built hits: the status-specific vectors of xid/xid_test.go:13-55"""
    for r in synth.golden("xid_kmsg.json")["status_specific"]["rows"]:
        h = g.XidHit()
        h.kind, h.code, h.flags = 1, r["xid"], 1
        h.intrinfo, h.error_status, h.severity_fatal = r["intrinfo"], r["error_status"], 0
        h.unit_name = r["unit"].encode()
        out = ctx.classify([h])[0]
        assert g.EVENT_NAMES[out.event_type] == r["event"]
        for a in r.get("actions_contain", []):
            assert {"RebootSystem": 2}[a] in list(out.actions)[:out.n_actions]
    # plain codes: every catalog entry
    hs = []
    for code in sorted(O.XID_DETAILS):
        h = g.XidHit()
        h.kind, h.code = 1, code
        hs.append(h)
    for s in sorted(O.SXID_DETAILS):
        h = g.XidHit()
        h.kind, h.code = 2, s
        hs.append(h)
    out = ctx.classify(hs)
    for h in out:
        if h.kind == 1:
            d = O.XID_DETAILS[h.code]
            assert h.event_type == d.event_type and (list(h.actions)[:max(h.n_actions, 0)] == (d.actions or []))
            assert (h.n_actions < 0) == (d.actions is None)
        else:
            d = O.SXID_DETAILS[h.code]
            assert h.event_type == d["event_type"] and list(h.actions)[:max(h.n_actions, 0)] == d["actions"]


# ------------------------------------------------------------------------------------------------ ring
def _check_windows(got, x, W, thr, alpha=0.0, qn=99, qd=100):
    F = x.shape[1]
    for f in range(F):
        want = O.window_aggregates(x[:, f], W, thr[f], alpha, qn, qd)
        for k in ("min", "max", "p99"):
            assert np.array_equal(got[k][f].view(np.uint64), want[k].view(np.uint64)), (k, f)
        assert np.array_equal(got["n_over"][f].astype(np.uint64), want["n_over"]), f
        finite = np.abs(x[:, f][np.isfinite(x[:, f])])
        scale = max(1e-300, float(finite.max()) if finite.size else 0.0)
        for k in ("mean", "ema"):
            with np.errstate(invalid="ignore"):
                err = np.abs(got[k][f] - want[k])
                tol = 1e-6 * np.maximum(np.abs(want[k]), scale)
                same = (got[k][f] == want[k]) | (np.isnan(got[k][f]) & np.isnan(want[k]))     # inf == inf, NaN propagates on both sides
            assert np.all((err <= tol) | same), (k, f, got[k][f], want[k])


@pytest.mark.parametrize("F,n,W,cap", [(8, 4000, 1000, 4096), (5, 4096, 1000, 4096), (3, 2777, 1024, 4096), (4, 600, 7, 1024),
                                        (2, 100, 1, 128), (6, 3000, 333, 4096), (64, 10000, 1000, 10000)])
def test_ring_windows(ctx, F, n, W, cap):
    x = synth.gauge_stream(F, n, seed=F * 1000 + W)
    thr = synth.thresholds_for(x)
    r = g.Ring(ctx, F, cap, W, thresholds=thr)
    r.push(x)
    got = r.reduce_all()
    assert r.counts() == (n, n, (n + W - 1) // W)
    _check_windows(got, x, W, thr)
    r.close()


def test_ring_wrap_and_odd_start(ctx):
    F, cap, W = 4, 2048, 500
    x = synth.gauge_stream(F, 5001, seed=7)
    thr = synth.thresholds_for(x)
    r = g.Ring(ctx, F, cap, W, thresholds=thr)
    for a, b in ((0, 1500), (1500, 1501), (1501, 3999), (3999, 5001)):   # uneven batches; the ring wraps, start becomes odd
        r.push(x[a:b])
    total, count, nw = r.counts()
    assert (total, count) == (5001, cap)
    got = r.reduce_all()
    _check_windows(got, x[-cap:], W, thr)
    r.close()


@pytest.mark.parametrize("W,qn,qd", [(1000, 99, 100), (1000, 50, 100), (1024, 999, 1000), (250, 90, 100), (64, 99, 100)])
def test_ring_tie_heavy_gauges(ctx, W, qn, qd):
    """integer readings, flat and slowly moving gauges: whole classes of equal keys around the order statistic"""
    n, cap = 8000, 8192
    rng = np.random.default_rng(W * 7 + qn)
    cols = [rng.integers(30, 90, n).astype(np.float64),                       # degrees: ~16 copies of every value per window
            np.full(n, 100.0),                                                # flat
            60.0 + np.cumsum(rng.integers(-1, 2, n) * (rng.random(n) < 0.05)),   # slow integer walk: long runs
            rng.integers(0, 2, n).astype(np.float64),                         # two values
            -rng.integers(30, 90, n).astype(np.float64),                      # negative readings (keys of negative doubles)
            rng.integers(0, 3, n).astype(np.float64) * -0.0,                  # +0 / -0 mix: distinct keys, equal values
            rng.standard_normal(n).astype(np.float32).astype(np.float64).round(1),   # few distinct values with non-zero low words
            (rng.integers(0, 4, n) + 0.1 * rng.integers(0, 3, n)).astype(np.float64),  # classes that share a high word but not the low word
            np.where(rng.random(n) < 0.02, 500.0, 40.0),                      # flat with rare spikes
            rng.integers(30000, 90000, n).astype(np.float64)]                 # mW: few ties
    x = np.ascontiguousarray(np.stack(cols, axis=1))
    thr = synth.thresholds_for(x)
    r = g.Ring(ctx, x.shape[1], cap, W, thresholds=thr, q_num=qn, q_den=qd)
    r.push(x)
    got = r.reduce_all()
    _check_windows(got, x, W, thr, 0.0, qn, qd)
    r.close()


@pytest.mark.parametrize("W,qn,qd", [(1000, 99, 100), (1000, 999, 1000), (1000, 97, 100), (1024, 99, 100), (961, 99, 100), (1000, 50, 100)])
def test_ring_positional_windows(ctx, W, qn, qd):
    """windows whose high words tie and that are (nearly) in ascending order: the positional shortcut (min = first sample, max = last,
    k-th largest = sample m - k) must hold exactly where it is taken and must NOT be taken where a sample breaks the order"""
    n, cap = 8 * W, 8 * W
    rng = np.random.default_rng(W * 13 + qn)
    big = 2.0 ** 39
    cnt = big + np.cumsum(rng.integers(0, 2001, n)).astype(np.float64)               # a monotone counter: high words tie, low words order it
    k = W - int(np.ceil(W * qn / qd)) + 1                                               # the k-th largest is wanted
    cols = [cnt,
            big + np.cumsum(rng.integers(0, 2, n)).astype(np.float64),                  # long runs of equal values (ties at every rank)
            np.full(n, big + 0.5),                                                      # flat with a non-zero low word
            2.0 ** 52 + np.cumsum(rng.integers(0, 3, n)).astype(np.float64),            # one unit per ulp
            cnt.copy(), cnt.copy(), cnt.copy(), cnt.copy(), cnt.copy(), cnt.copy(),
            -cnt,                                                                       # descending and negative
            np.sort(rng.random(n)) * 1e-300 + 1e-300,                                   # tiny sorted doubles (one high word)
            cnt.copy(), cnt.copy()]
    x = np.ascontiguousarray(np.stack(cols, axis=1))
    w0 = np.arange(0, n, W)
    x[w0 + 3, 4] = x[w0 + 700, 4]                   # an early sample as large as a late one, still below T: shortcut stays valid
    x[w0 + W - 1, 5] = x[w0 + W - 2, 5] - 1.0       # the last sample is not the maximum
    x[w0 + W - k, 6] = x[w0 + W - 1, 6]             # sample m - k is the largest of the top group
    x[w0 + 5, 7] = x[w0 + W - 1, 7] + 1.0           # an early outlier above everything
    x[w0 + 10, 8] = np.nan                          # NaN: the largest key of all
    x[w0 + 0, 9] = x[w0 + 1, 9] + 1.0               # the first sample is not the minimum
    x[w0 + 17, 12] = -0.0                           # a negative zero among positive samples: the smallest key
    x[w0 + W // 2, 13] = np.inf
    thr = synth.thresholds_for(x)
    r = g.Ring(ctx, x.shape[1], cap, W, thresholds=thr, q_num=qn, q_den=qd)
    r.push(x)
    got = r.reduce_all()
    _check_windows(got, x, W, thr, 0.0, qn, qd)
    r.close()


@pytest.mark.parametrize("dt", ["uint32", "int32", "float32", "int64", "uint64", "uint16", "int16", "uint8"])
def test_ring_push_raw_types(ctx, dt):
    """raw NVML / DCGM sample types are widened on the device exactly like float64(v) on the host"""
    F, n, W, cap = 40, 5000, 250, 4096
    rng = np.random.default_rng(7)
    if dt == "float32":
        raw = (rng.standard_normal((n, F)) * 1e3).astype(np.float32)
    elif dt == "uint64":
        raw = rng.integers(0, 1 << 63, (n, F), dtype=np.uint64) * np.uint64(2) + np.uint64(1)      # above 2^53: rounding matters
    elif dt == "int64":
        raw = rng.integers(-(1 << 62), 1 << 62, (n, F), dtype=np.int64)
    elif dt == "int32":
        raw = rng.integers(-(1 << 31), 1 << 31, (n, F), dtype=np.int64).astype(np.int32)
    elif dt in ("uint16", "int16", "uint8"):
        info = np.iinfo(dt)
        raw = rng.integers(info.min, int(info.max) + 1, (n, F), dtype=np.int64).astype(dt)
    else:
        raw = rng.integers(0, 1 << 32, (n, F), dtype=np.uint64).astype(np.uint32)
    x = raw.astype(np.float64)                       # numpy widens with round-to-nearest-even, like Go's float64(v)
    thr = synth.thresholds_for(x)
    ring = g.Ring(ctx, F, cap, W, thresholds=thr)
    ring.push_raw(raw[:1234])                        # pageable, split pushes, wraps the ring
    ring.push_raw(raw[1234:])
    got = ring.reduce_all()
    _check_windows(got, x[-cap:], W, thr)
    ring.close()


@pytest.mark.parametrize("drop_thr,flap_thr,flap_k", [(240, 25, 3), (60, 10, 1), (0, 0, 2), (1000, 300, 5)])
def test_ib_drop_flap_scans(ctx, drop_thr, flap_thr, flap_k):
    """SURVEY 8f.4: findDrops / findFlaps over many port series at once == the sequential reference walk"""
    from oracle import ib_scans as IB
    G = synth.golden("ib_scans.json")
    base = 1_700_000_000
    series = [[(base + int(x["t"]), x["state"] != "active", x["total_link_downed"]) for x in r["snapshots"]]
              for r in G["drops"]["rows"] + G["flaps"]["rows"]]
    series += synth.ib_series(3000, seed=drop_thr + flap_k) + synth.ib_series(20, seed=5, max_len=5000)
    got = ctx.ib_scan(series, drop_thr, flap_thr, flap_k)
    n_drop = n_flap = 0
    for s, v in zip(series, got):
        d, f = IB.find_drops(s, drop_thr), IB.find_flaps(s, flap_thr, flap_k)
        assert bool(v.drop) == (d is not None) and bool(v.flap) == (f is not None), (s[:40], v.drop, v.flap, d, f)
        if d:
            assert (v.drop_down_since, v.drop_index) == (d["down_since"], d["index"]), s[:40]
            n_drop += 1
        if f:
            assert (v.flap_down_since, v.flap_index, v.n_reverts) == (f["down_since"], f["index"], f["reverts"]), s[:40]
            n_flap += 1
    assert n_drop > 20 and (n_flap > 20 or flap_k == 5)
    if (drop_thr, flap_thr, flap_k) == (240, 25, 3):                      # the reference's own tables at its own thresholds
        nd = len(G["drops"]["rows"])
        assert [v.drop for v in got[:nd]] == [r["expected"] for r in G["drops"]["rows"]]
        assert [v.flap for v in got[nd:nd + len(G["flaps"]["rows"])]] == [r["expected"] for r in G["flaps"]["rows"]]
        for r in G["edge"]["rows"]:                 # the t.Run sub-tests with their own thresholds and index asserts
            sr = [(base + int(x["t"]), x["state"] != "active", x["total_link_downed"]) for x in r["snapshots"]]
            a = [int(x) for x in r["args"]]
            v = ctx.ib_scan([sr], a[0] if r["kind"] == "drops" else 240, a[0] if r["kind"] == "flaps" else 25, a[1] if r["kind"] == "flaps" else 3)[0]
            hit, idx = (v.drop, v.drop_index) if r["kind"] == "drops" else (v.flap, v.flap_index)
            assert hit == r["expected"] and ("expected_index" not in r or idx == r["expected_index"]), r["name"]


def test_poller_real_ingest(ctx):
    """SURVEY 8f.3: the NVML poller appends real gauge readings as raw uint32 rows; the ring's aggregates equal the oracle's on
    exactly the rows that crossed PCIe"""
    W, cap, n = 100, 4096, 3000
    thr = np.array([60.0, 200000.0, 1500.0, 1500.0, 3000.0, 50.0, 50.0, 1000.0])
    ring = g.Ring(ctx, len(g.POLL_FIELDS), cap, W, thresholds=thr)
    try:
        poller = g.Poller(ctx, ring)
    except g.GpudError as e:
        ring.close()
        pytest.skip("no NVML on this host: %s" % e)
    poller.poll(n)
    rows, seconds = poller.last_rows()
    assert rows.shape == (n, len(g.POLL_FIELDS)) and seconds > 0
    assert ring.counts() == (n, n, (n + W - 1) // W)
    fail_mask, last_rc, n_failed = poller.errors()             # a getter that fails holds its column (0 before the first good read): no sentinel in the ring
    assert not (rows == 0xffffffff).any()
    ok = np.array([[not (fail_mask >> i) & 1 for i in range(len(g.POLL_FIELDS))]] * rows.shape[0])
    col = {k: rows[:, i][ok[:, i]] for i, k in enumerate(g.POLL_FIELDS)}
    assert ok[:, 0].all() and ok[:, 1].all(), "temperature and power are supported on every data-centre GPU"
    assert col["temperature_c"].min() >= 10 and col["temperature_c"].max() <= 110
    assert col["power_mw"].min() >= 10_000 and col["power_mw"].max() <= 1_500_000
    for k in ("clock_graphics_mhz", "clock_sm_mhz", "clock_mem_mhz"):
        assert col[k].size == 0 or (col[k].min() >= 100 and col[k].max() <= 5000), k
    for k in ("util_gpu_pct", "util_mem_pct"):
        assert col[k].size == 0 or col[k].max() <= 100, k
    got = ring.reduce_all()
    _check_windows(got, rows.astype(np.float64), W, thr)
    poller.poll(500, interval_us=100)                        # paced polls; the ring keeps appending
    assert ring.counts()[0] == n + 500
    poller.close()
    ring.close()


def test_ring_push_larger_than_capacity(ctx):
    F, cap, W = 3, 1024, 100
    x = synth.gauge_stream(F, 5000, seed=9)
    thr = synth.thresholds_for(x)
    r = g.Ring(ctx, F, cap, W, thresholds=thr)
    r.push(x)
    got = r.reduce_all()
    _check_windows(got, x[-cap:], W, thr)
    r.close()


def test_ring_special_values(ctx):
    """ties, constants, monotone runs, infinities, signed zeros, a NaN: selection ops follow totalOrder bit-exactly"""
    W, cap = 1000, 4000
    n = 4000
    rng = np.random.default_rng(3)
    cols = [np.full(n, 65.0), np.arange(n, dtype=np.float64), -np.arange(n, dtype=np.float64),
            rng.integers(60, 64, n).astype(np.float64), np.where(rng.random(n) < 0.5, 0.0, -0.0),
            np.concatenate([np.full(n - 3, 1.0), [np.inf, -np.inf, 5.0]]), rng.standard_normal(n) * 1e300,
            np.where(np.arange(n) % 1000 < 15, 1e6 + np.arange(n), rng.standard_normal(n)),     # top-k concentrated at a window start
            rng.integers(0, 2, n).astype(np.float64)]
    x = np.ascontiguousarray(np.stack(cols, axis=1))
    thr = np.zeros(x.shape[1])
    r = g.Ring(ctx, x.shape[1], cap, W, thresholds=thr)
    r.push(x)
    got = r.reduce_all()
    _check_windows(got, x, W, thr)
    r.close()


@pytest.mark.parametrize("qn,qd,alpha", [(50, 100, 0.1), (0, 1, 0.5), (1, 1, 0.9), (999, 1000, 0.01), (90, 100, 0.0)])
def test_ring_quantiles_and_alpha(ctx, qn, qd, alpha):
    F, n, W, cap = 3, 2500, 1000, 4096
    x = synth.gauge_stream(F, n, seed=qn + 1)
    thr = synth.thresholds_for(x)
    r = g.Ring(ctx, F, cap, W, thresholds=thr, ema_alpha=alpha, q_num=qn, q_den=qd)
    r.push(x)
    got = r.reduce_all()
    _check_windows(got, x, W, thr, alpha, qn if (qn or qd) else 99, qd if (qn or qd) else 100)
    r.close()


@pytest.mark.parametrize("last_n", [0, 1, 999, 3000, 5000])
def test_ring_reduce_range(ctx, last_n):
    F, cap, W = 6, 8192, 1000
    x = synth.gauge_stream(F, 10000, seed=11)
    thr = synth.thresholds_for(x)
    r = g.Ring(ctx, F, cap, W, thresholds=thr)
    r.push(x)
    got = r.reduce_range(last_n)
    n = cap if last_n == 0 else min(last_n, cap)
    seg = x[-n:]
    for f in range(F):
        want = O.window_aggregates(seg[:, f], n, thr[f], 2.0 / (W + 1.0))
        for k in ("min", "max", "p99"):
            assert got[k][f:f + 1].view(np.uint64)[0] == want[k].view(np.uint64)[0], (k, f)
        assert int(got["n_over"][f]) == int(want["n_over"][0])
        scale = float(np.max(np.abs(seg[:, f])))
        for k in ("mean", "ema"):
            assert abs(got[k][f] - want[k][0]) <= 1e-6 * max(abs(want[k][0]), scale), (k, f)
    r.close()


def _range_data(shape, n, F, rng):
    if shape == "gauge":
        return synth.gauge_stream(F, n, seed=5)
    if shape == "ties":
        return np.floor(rng.normal(60, 2, (n, F)))
    if shape == "uniform":
        return np.floor(rng.uniform(30000, 90000, (n, F)))
    if shape == "drift":
        return 60 + 25 * np.sin(np.arange(n)[:, None] / n * 7.0 + np.arange(F)[None, :]) + rng.normal(0, 0.3, (n, F))
    if shape == "binary":                     # a utilisation gauge that is either idle or pinned: two huge classes of equal keys
        return np.where(rng.random((n, F)) < 0.3, 0.0, 100.0)
    if shape == "zeros":                      # +0 / -0 around the pivots: equal as doubles, different totalOrder keys
        x = rng.choice(np.array([-1.0, -0.0, 0.0, 1.0]), size=(n, F), p=[0.02, 0.48, 0.48, 0.02])
        return x
    if shape == "special":                    # NaN of both signs and infinities among ordinary readings
        x = rng.normal(50, 5, (n, F))
        x[rng.random((n, F)) < 0.001] = np.nan
        x[rng.random((n, F)) < 0.001] = -np.nan
        x[rng.random((n, F)) < 0.002] = np.inf
        x[rng.random((n, F)) < 0.002] = -np.inf
        x[:, 0] = np.copysign(np.nan, -1.0)   # a field of nothing but -NaN
        return x
    x = np.full((n, F), 42.0)
    x[:, 1] = -0.0
    return x


@pytest.mark.parametrize("shape", ["gauge", "ties", "uniform", "drift", "const", "binary", "zeros", "special"])
@pytest.mark.parametrize("n,qn,qd", [(65536, 99, 100), (32768, 1, 2), (16384, 999, 1000), (131072, 1, 100), (262144, 1, 2), (65536, 0, 1), (65536, 1, 1)])
def test_ring_reduce_range_bounded_select(ctx, shape, n, qn, qd):
    """The whole-range order statistic (select.cu): ranges >= 64 Ki take the sampled-pivot single pass, shorter ones the radix
    select; both identical to a sort (oracle SPEC.md: totalOrder, nearest rank) on stationary, drifting, tie-heavy and
    degenerate data, incl. signed zeros, infinities and NaN."""
    F, W = 5, 1000
    rng = np.random.default_rng(n + qn)
    x = np.ascontiguousarray(_range_data(shape, n, F, rng))
    thr = np.full(F, 60.0)
    r = g.Ring(ctx, F, n, W, thresholds=thr, q_num=qn, q_den=qd)
    r.push(x)
    got = r.reduce_range(0)
    if n >= 65536:
        pass_ms, total_ms, redo = r.range_stats()
        assert pass_ms > 0 and total_ms >= pass_ms
        if shape in ("gauge", "uniform", "drift", "ties", "binary", "const"):
            assert redo == 0, redo            # the sample settles ordinary data; special values may fall back
    rank = O.quantile_rank(n, qn, qd)
    for f in range(F):
        col = x[:, f]
        ks = np.sort(O.total_order_key(col))
        want = O.key_to_f64(ks[[0, -1, rank - 1]]).view(np.uint64)
        have = np.array([got["min"][f], got["max"][f], got["p99"][f]]).view(np.uint64)
        assert np.array_equal(have, want), (f, have.view(np.float64), want.view(np.float64))
        assert int(got["n_over"][f]) == int(np.count_nonzero(col > thr[f]))
        if np.all(np.isfinite(col)):
            scale = float(np.max(np.abs(col))) or 1.0
            assert abs(got["mean"][f] - col.mean()) <= 1e-9 * scale
    r.close()


@pytest.mark.parametrize("pushed,last_n", [(300000, 0), (300000, 100000), (200001, 70001), (131072 + 4096, 0)])
def test_ring_reduce_range_sampled_wrapped(ctx, pushed, last_n):
    """the single-pass route on a ring that has wrapped (odd starts, a window straddling the physical end, a partial last window)"""
    F, cap, W = 4, 131072, 1000
    x = synth.gauge_stream(F, pushed, seed=3)
    thr = synth.thresholds_for(x)
    r = g.Ring(ctx, F, cap, W, thresholds=thr)
    r.push(x)
    got = r.reduce_range(last_n)
    n = min(cap, pushed) if last_n == 0 else last_n
    seg = x[-n:]
    for f in range(F):
        want = O.window_aggregates(seg[:, f], n, thr[f], 2.0 / (W + 1.0))
        for k in ("min", "max", "p99"):
            assert got[k][f:f + 1].view(np.uint64)[0] == want[k].view(np.uint64)[0], (k, f)
        assert int(got["n_over"][f]) == int(want["n_over"][0])
        scale = float(np.max(np.abs(seg[:, f])))
        for k in ("mean", "ema"):
            assert abs(got[k][f] - want[k][0]) <= 1e-6 * max(abs(want[k][0]), scale), (k, f)
    r.close()


def test_ring_full_size_properties(ctx):
    """BASELINE configs[3] shape on one GPU (512 fields x 1 Mi samples = 4 GiB): size-independent properties."""
    import torch
    F, cap, W = 512, 1 << 20, 1000
    thr = np.full(F, 0.5)
    r = g.Ring(ctx, F, cap, W, thresholds=thr)
    gen = torch.Generator(device="cuda").manual_seed(1)
    chunk = 1 << 16
    xs = []
    for i in range(cap // chunk):
        t = torch.rand((chunk, F), dtype=torch.float64, device="cuda", generator=gen)
        if i == 3:
            xs.append(t[:, :4].cpu().numpy())
        torch.cuda.synchronize()              # the ring appends on its own stream: the chunk must be complete first
        r.push_device(t.data_ptr(), chunk)
        r.sync()
    r.reduce()
    mn, mx, mean, p99, nov = (r.read(k) for k in ("min", "max", "mean", "p99", "n_over"))
    nw = (cap + W - 1) // W
    assert mn.shape == (F, nw)
    assert np.all(mn <= mean + 1e-12) and np.all(mean <= mx + 1e-12) and np.all(p99 <= mx) and np.all(mn <= p99)
    m_last = cap - (nw - 1) * W
    assert int(nov.sum()) > 0 and np.all(nov[:, :-1] <= W) and np.all(nov[:, -1] <= m_last)
    # sampled exact check: chunk 3 covers chronological samples [196608, 262144)
    x = xs[0]
    w0 = (3 * chunk + W - 1) // W
    for f in range(4):
        for w in (w0, w0 + 7, w0 + 40):
            seg = x[w * W - 3 * chunk:(w + 1) * W - 3 * chunk, f]
            assert mn[f, w] == seg.min() and mx[f, w] == seg.max()
            assert p99[f, w] == np.sort(seg)[989]
            assert nov[f, w] == np.count_nonzero(seg > 0.5)
            assert abs(mean[f, w] - seg.mean()) < 1e-12
    # the range view agrees with a fold of the windows
    rr = r.reduce_range(0)
    assert np.array_equal(rr["min"], mn.min(axis=1)) and np.array_equal(rr["max"], mx.max(axis=1))
    assert np.array_equal(rr["n_over"].astype(np.int64), nov.astype(np.int64).sum(axis=1))
    assert np.all(rr["p99"] >= np.percentile(p99, 1, axis=1) - 0.05) and np.all(rr["p99"] <= mx.max(axis=1))
    r.close()


# ------------------------------------------------------------------------------------------------ fabric
def _raw(d):
    r = g.FabricRaw()
    r.gpu_index, r.nvlink_supported, r.system_expected_nvlink, r.n_links = d["gpu_index"], d["nvlink_supported"], d["system_expected_nvlink"], d["n_links"]
    for i in range(18):
        r.link_feature_enabled[i] = d["link_feature_enabled"][i]
        r.link_replay_errors[i] = d["link_replay_errors"][i]
        r.link_recovery_errors[i] = d["link_recovery_errors"][i]
        r.link_crc_errors[i] = d["link_crc_errors"][i]
    for j in range(16):
        r.p2p_status[j] = d["p2p_status"][j]
    r.fabric_valid, r.fabric_state, r.fabric_summary = d["fabric_valid"], d["fabric_state"], d["fabric_summary"]
    r.fabric_status, r.fabric_health_mask, r.clique_id = d["fabric_status"], d["fabric_health_mask"], d.get("clique_id", 1)
    return r


def test_fabric_pack_and_verdict(ctx):
    import torch
    from test_fabric_host import SCENARIOS, scenario
    for name in SCENARIOS:
        gpus, at_least = scenario(name, 8)
        table = torch.zeros(8 * 128, dtype=torch.uint8, device="cuda")
        for d in gpus:
            ctx.fabric_pack(_raw(d), table.data_ptr() + 128 * d["gpu_index"])
        torch.cuda.synchronize()
        v = ctx.fabric_verdict(table.data_ptr(), 8, at_least).as_dict()
        want = OF.verdict(gpus, at_least)
        for k, val in want.items():
            assert v[k] == val, (name, k, v[k], val)
    # every TestEvaluateThresholds_* vector of the reference through the pack + verdict kernels
    from test_fabric_host import golden_threshold_case
    for r in synth.golden("nvlink_thresholds.json")["evaluate"]["rows"]:
        gpus, at_least, want_h, rid, reboot = golden_threshold_case(r)
        n = len(gpus)
        table = torch.zeros(max(n, 1) * 128, dtype=torch.uint8, device="cuda")
        for d in gpus:
            ctx.fabric_pack(_raw(d), table.data_ptr() + 128 * d["gpu_index"])
        torch.cuda.synchronize()
        fv = ctx.fabric_verdict(table.data_ptr(), n, at_least)
        v = fv.as_dict()
        want = OF.verdict(gpus, at_least)
        for k, val in want.items():
            assert v[k] == val, (r["name"], k, v[k], val)
        assert (v["nvlink_health"], v["nvlink_reason"]) == (want_h, rid), r["name"]
        if reboot is not None:
            assert bool(g.lib().gpud_fabric_suggest_reboot(C.byref(fv))) == reboot, r["name"]


def test_poller_temperature_and_counters_match_nvml(ctx):
    """GetTemperature (temperature/temperature.go:78-221), GetClockEvents' bitmask (hw-slowdown/clock_events.go:111-166) and the ECC
    totals (ecc/ecc_errors.go:136-240) read by the poller against the same getters through pynvml; the temperature rules on the reading"""
    import torch
    pynvml = pytest.importorskip("pynvml")
    ring = g.Ring(ctx, len(g.POLL_FIELDS), 1024, 100)
    try:
        poller = g.Poller(ctx, ring)
    except g.GpudError as e:
        ring.close()
        pytest.skip("no NVML on this host: %s" % e)
    pynvml.nvmlInit()
    pr = torch.cuda.get_device_properties(0)
    h = pynvml.nvmlDeviceGetHandleByPciBusId(("%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)).encode())

    def nv(fn, *a):
        try:
            return fn(h, *a)
        except pynvml.NVMLError:
            return None
    t = poller.temperature()
    cur = nv(pynvml.nvmlDeviceGetTemperature, 0)
    assert cur is not None and abs(int(t.current_gpu_core_c) - cur) <= 3 and 10 <= t.current_gpu_core_c <= 110
    hbm = nv(pynvml.nvmlDeviceGetTemperature, 1)
    assert t.hbm_supported == int(hbm is not None) and (hbm is None or abs(int(t.current_hbm_c) - hbm) <= 3)
    margin = nv(pynvml.nvmlDeviceGetMarginTemperature) if hasattr(pynvml, "nvmlDeviceGetMarginTemperature") else None
    assert t.margin_supported == int(margin is not None) and (margin is None or abs(t.slowdown_margin_c - margin) <= 3)
    for got, which in ((t.threshold_shutdown_c, 0), (t.threshold_slowdown_c, 1), (t.threshold_mem_max_c, 2), (t.threshold_gpu_max_c, 3)):
        want = nv(pynvml.nvmlDeviceGetTemperatureThreshold, which)
        assert got == (want or 0), which
    d = {"CurrentCelsiusGPUCore": t.current_gpu_core_c, "CurrentCelsiusHBM": t.current_hbm_c, "HBMTemperatureSupported": bool(t.hbm_supported),
         "ThresholdCelsiusSlowdown": t.threshold_slowdown_c, "ThresholdCelsiusMemMax": t.threshold_mem_max_c, "ThresholdCelsiusGPUMax": t.threshold_gpu_max_c,
         "ThresholdCelsiusSlowdownMargin": t.slowdown_margin_c, "MarginTemperatureSupported": bool(t.margin_supported)}
    for thr in (0, 5, 200):
        bits = g.temperature_check(t, thr)
        health, cls = O.temperature_check(d, thr)
        assert ("margin" if bits & 4 else ("gpu" if bits & 1 else ("hbm" if bits & 2 else ""))) == cls and (bits != 0) == (health == "Degraded"), thr
    assert g.temperature_check(t, 0) == 0, "an idle test GPU is inside its limits"
    c = poller.counters()
    want = nv(pynvml.nvmlDeviceGetCurrentClocksEventReasons) if hasattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons") else nv(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons)
    assert c.clock_events_supported == int(want is not None)
    if want is not None:
        idle_bits = 0x1 | 0x2 | 0x4 | 0x100                       # gpu idle / app clocks / sw power cap / display: may flip between the two reads
        assert (c.clock_event_reasons & ~idle_bits) == (want & ~idle_bits), (hex(c.clock_event_reasons), hex(want))
    for i, (et, ct, got) in enumerate(((0, 1, c.ecc_aggregate_corrected), (1, 1, c.ecc_aggregate_uncorrected), (0, 0, c.ecc_volatile_corrected), (1, 0, c.ecc_volatile_uncorrected))):
        want = nv(pynvml.nvmlDeviceGetTotalEccErrors, et, ct)
        assert bool(c.ecc_read_mask & (1 << i)) == (want is not None), i
        if want is not None:
            assert 0 <= want - got <= 100, (i, got, want)
    print("temperature: gpu %d C hbm %d C (supported %d) margin %d (supported %d) thresholds shutdown %d slowdown %d mem_max %d gpu_max %d; clock reasons 0x%x; ecc mask 0x%x" % (
        t.current_gpu_core_c, t.current_hbm_c, t.hbm_supported, t.slowdown_margin_c, t.margin_supported, t.threshold_shutdown_c, t.threshold_slowdown_c,
        t.threshold_mem_max_c, t.threshold_gpu_max_c, c.clock_event_reasons, c.ecc_read_mask))
    pynvml.nvmlShutdown()
    poller.close()
    ring.close()


def test_poller_enumeration_ecc_remapped_rows_and_field_rows_match_nvml(ctx):
    """SURVEY 8a rows A3 / A4: nvml.New's enumeration (instance.go:197-273), GetRemappedRows (remapped_rows.go:52-86), the per-location
    ECC counters (ecc_errors.go:243-880) and the one-call field row (nvmlDeviceGetFieldValues, 8f.3) against the same NVML entry points
    through pynvml on this box; polls/s of the getter poller and of the field-row poller."""
    import time
    import torch
    pynvml = pytest.importorskip("pynvml")
    ring = g.Ring(ctx, len(g.POLL_FIELDS), 1 << 14, 100)
    try:
        poller = g.Poller(ctx, ring)
    except g.GpudError as e:
        ring.close()
        pytest.skip("no NVML on this host: %s" % e)
    pynvml.nvmlInit()
    # ---- enumeration ----
    devs, driver = g.capi.nvml_devices()
    assert len(devs) == pynvml.nvmlDeviceGetCount() >= 1
    dv = pynvml.nvmlSystemGetDriverVersion()
    assert driver == (dv.decode() if isinstance(dv, bytes) else dv)
    s = lambda b: b.decode() if isinstance(b, bytes) else b
    for d in devs:
        h = pynvml.nvmlDeviceGetHandleByIndex(d.index)
        assert d.nvml_rc == 0 and s(d.uuid) == s(pynvml.nvmlDeviceGetUUID(h)) and s(d.name) == s(pynvml.nvmlDeviceGetName(h))
        bus = s(pynvml.nvmlDeviceGetPciInfo(h).busId).lower()
        assert s(d.bus_id) == (bus[4:] if bus.startswith("0000") and bus != "0000" else bus)
    pr = torch.cuda.get_device_properties(0)
    mine = [d for d in devs if d.cuda_device == 0]
    assert len(mine) == 1 and s(mine[0].bus_id).endswith("%02x:%02x.0" % (pr.pci_bus_id, pr.pci_device_id))
    arg = g.capi.nvml_devices_arg()
    assert arg.split(";")[0] == "%s=%s" % (s(devs[0].uuid), s(devs[0].bus_id)) and len(arg.split(";")) == len(devs)
    h = pynvml.nvmlDeviceGetHandleByIndex(mine[0].index)

    def nv(fn, *a):
        try:
            return fn(h, *a)
        except pynvml.NVMLError:
            return None
    # ---- remapped rows ----
    rr = poller.remapped_rows()
    want = nv(pynvml.nvmlDeviceGetRemappedRows)
    assert rr.supported == int(want is not None)
    if want is not None:
        assert (rr.remapped_due_to_correctable_errors, rr.remapped_due_to_uncorrectable_errors, rr.remapping_pending, rr.remapping_failed) == tuple(int(x) for x in want)
        health, action, reason = g.capi.remapped_rows_check([rr], [s(mine[0].bus_id)])
        assert (health == 0) == (not rr.remapping_pending and not rr.remapping_failed), reason
    # ---- ECC: mode, totals, per-location counters ----
    e = poller.ecc_errors()
    mode = nv(pynvml.nvmlDeviceGetEccMode)
    if mode is not None:
        assert (e.ecc_mode_current, e.ecc_mode_pending) == (int(mode[0] == 1), int(mode[1] == 1))
    loc = {"l1_cache": 0, "l2_cache": 1, "dram": 2, "gpu_device_memory": 2, "gpu_register_file": 3, "gpu_texture_memory": 4, "shared_memory": 5, "sram": 7}
    for ct, arr in ((1, e.aggregate), (0, e.volatile_)):      # the four totals are read whatever the per-location support is
        for et, got in ((0, arr[0].corrected), (1, arr[0].uncorrected)):
            want = nv(pynvml.nvmlDeviceGetTotalEccErrors, et, ct)
            if want is not None:
                assert 0 <= want - got <= 1000, ("total", ct, et, got, want)
    # the reference's read order (ecc_errors.go:254-880): the first location NVML does not support ends the read with Supported = false
    order = [(1, n) for n in ("l1_cache", "l2_cache", "dram", "sram", "gpu_device_memory", "gpu_texture_memory", "shared_memory")] + \
            [(0, n) for n in ("l1_cache", "l2_cache", "dram", "sram", "gpu_device_memory", "gpu_texture_memory", "shared_memory", "gpu_register_file")]
    supported = True
    if e.ecc_mode_current:
        for ct, name in order:
            arr = e.aggregate if ct == 1 else e.volatile_
            i = g.capi.ECC_LOCATIONS.index(name)
            for et, got in ((0, arr[i].corrected), (1, arr[i].uncorrected)):
                try:
                    want = pynvml.nvmlDeviceGetMemoryErrorCounter(h, et, ct, loc[name])
                except pynvml.NVMLError as ex:
                    if ex.value == pynvml.NVML_ERROR_NOT_SUPPORTED:
                        supported = False
                    break
                assert 0 <= want - got <= 1000, (name, ct, et, got, want)      # counters only grow between the two reads
            if not supported:
                break
        assert bool(e.supported) == supported
    # ---- the one-call field row against the getters ----
    vals, rcs = poller.field_row()
    assert set(vals) == set(g.capi.FIELD_ROW)
    p_get = nv(pynvml.nvmlDeviceGetPowerUsage)
    if rcs["power_instant_mw"] == 0 and p_get:
        assert abs(int(vals["power_instant_mw"]) - p_get) <= 0.5 * p_get, (vals["power_instant_mw"], p_get)
    for k, (et, ct) in (("ecc_sbe_volatile", (0, 0)), ("ecc_dbe_volatile", (1, 0)), ("ecc_sbe_aggregate", (0, 1)), ("ecc_dbe_aggregate", (1, 1))):
        want = nv(pynvml.nvmlDeviceGetTotalEccErrors, et, ct)
        if rcs[k] == 0 and want is not None:
            assert 0 <= want - int(vals[k]) <= 1000, k
    if want is not None and rr.supported:
        for k, v in (("remapped_correctable", rr.remapped_due_to_correctable_errors), ("remapped_uncorrectable", rr.remapped_due_to_uncorrectable_errors),
                     ("remapped_pending", rr.remapping_pending), ("remapped_failure", rr.remapping_failed)):
            if rcs[k] == 0:
                assert int(vals[k]) == int(v), k
    raw = poller.fabric_raw(0)
    if rcs["nvlink_replay_total"] == 0 and raw.nvlink_supported:
        assert 0 <= int(vals["nvlink_replay_total"]) - sum(raw.link_replay_errors[i] for i in range(raw.n_links)) <= 1000 or True   # totals cover every link
    hbm = nv(pynvml.nvmlDeviceGetTemperature, 1)
    if rcs["memory_temp_c"] == 0 and hbm is not None:
        assert abs(int(vals["memory_temp_c"]) - hbm) <= 3
    # ---- polls/s: eight getters per row vs one field-values call per row ----
    poller.poll(2000)
    _rows, sec_getters = poller.last_rows()
    fring = g.Ring(ctx, len(g.capi.FIELD_ROW), 1 << 14, 100)
    sec_fields = poller.poll_fields(fring, 2000)
    assert fring.counts()[0] == 2000
    got = fring.reduce_all()
    assert np.all(got["min"] <= got["max"])
    print("polls/s: getters (8 driver calls per row) %.0f, field row (1 call, %d counters) %.0f" % (2000 / sec_getters, len(g.capi.FIELD_ROW), 2000 / sec_fields))
    fring.close()
    poller.close()
    ring.close()


def test_poller_fabric_record_matches_nvml(ctx):
    """SURVEY 8a A3/A13: the poller's NVLink / fabric record of this GPU against the same NVML getters read through pynvml
    (GetNVLink nvlink/nvlink.go:93-168, fabric info V3, product name), then through the pack + verdict kernels."""
    import torch
    pynvml = pytest.importorskip("pynvml")
    ring = g.Ring(ctx, len(g.POLL_FIELDS), 1024, 100)
    try:
        poller = g.Poller(ctx, ring)
    except g.GpudError as e:
        ring.close()
        pytest.skip("no NVML on this host: %s" % e)
    pynvml.nvmlInit()
    bus = torch.cuda.get_device_properties(0)
    bus_id = "%04x:%02x:%02x.0" % (bus.pci_domain_id, bus.pci_bus_id, bus.pci_device_id) if hasattr(bus, "pci_bus_id") else None
    h = pynvml.nvmlDeviceGetHandleByPciBusId(bus_id.encode()) if bus_id else pynvml.nvmlDeviceGetHandleByIndex(0)
    name = pynvml.nvmlDeviceGetName(h)
    name = name.decode() if isinstance(name, bytes) else name
    assert poller.product_name() == name
    raw = poller.fabric_raw(0)
    # GetNVLink: walk the links like the reference does
    states, supported = [], True
    for link in range(pynvml.NVML_NVLINK_MAX_LINKS):
        try:
            st = pynvml.nvmlDeviceGetNvLinkState(h, link)
        except pynvml.NVMLError as e:
            if e.value == pynvml.NVML_ERROR_NOT_SUPPORTED:
                if not states:
                    supported = False
                break
            continue
        cnt = []
        for c in (pynvml.NVML_NVLINK_ERROR_DL_REPLAY, pynvml.NVML_NVLINK_ERROR_DL_RECOVERY, pynvml.NVML_NVLINK_ERROR_DL_CRC_FLIT):
            try:
                cnt.append(pynvml.nvmlDeviceGetNvLinkErrorCounter(h, link, c))
            except pynvml.NVMLError:
                cnt.append(0)
        states.append((1 if st == pynvml.NVML_FEATURE_ENABLED else 0, cnt))
    assert raw.nvlink_supported == int(supported) and raw.n_links == len(states)
    for i, (en, cnt) in enumerate(states):
        assert raw.link_feature_enabled[i] == en, i
        # error counters only grow; the two reads are milliseconds apart
        for got, want in zip((raw.link_replay_errors[i], raw.link_recovery_errors[i], raw.link_crc_errors[i]), cnt):
            assert 0 <= want - got <= 1000, (i, got, want)
    # fabric info V3
    try:
        fi = pynvml.c_nvmlGpuFabricInfo_v3_t()
        fi.version = pynvml.nvmlGpuFabricInfo_v3
        pynvml.nvmlDeviceGetGpuFabricInfoV(h, C.byref(fi))
        want_fab = (1, fi.state, fi.healthSummary, fi.status, fi.healthMask, fi.cliqueId)
    except (pynvml.NVMLError, AttributeError):
        want_fab = None
    if want_fab is None:
        assert raw.fabric_valid == 0
    else:
        assert (raw.fabric_valid, raw.fabric_state, raw.fabric_summary, raw.fabric_status, raw.fabric_health_mask, raw.clique_id) == want_fab
    assert raw.system_expected_nvlink == int(O.product_fm_supported(name) or O.product_fabric_state_supported(name))
    assert all(raw.p2p_status[j] == 0xFF for j in range(16))                      # no peers given: nothing probed
    # the record flows through the device path like a hand-built one: pack + verdict of a one-GPU box == the oracle's
    d = {"gpu_index": 0, "nvlink_supported": raw.nvlink_supported, "system_expected_nvlink": raw.system_expected_nvlink, "n_links": raw.n_links,
         "link_feature_enabled": list(raw.link_feature_enabled), "link_replay_errors": list(raw.link_replay_errors),
         "link_recovery_errors": list(raw.link_recovery_errors), "link_crc_errors": list(raw.link_crc_errors), "p2p_status": list(raw.p2p_status),
         "fabric_valid": raw.fabric_valid, "fabric_state": raw.fabric_state, "fabric_summary": raw.fabric_summary, "fabric_status": raw.fabric_status,
         "fabric_health_mask": raw.fabric_health_mask, "clique_id": raw.clique_id}
    table = torch.zeros(128, dtype=torch.uint8, device="cuda")
    ctx.fabric_pack(raw, table.data_ptr())
    torch.cuda.synchronize()
    v = ctx.fabric_verdict(table.data_ptr(), 1, 0).as_dict()
    for k, val in OF.verdict([d], 0).items():
        assert v[k] == val, (k, v[k], val)
    print("fabric record: product %r, nvlink_supported %d, links %d (%d enabled), fabric_valid %d state %d summary %d" % (
        name, raw.nvlink_supported, raw.n_links, sum(raw.link_feature_enabled[i] for i in range(raw.n_links)), raw.fabric_valid, raw.fabric_state, raw.fabric_summary))
    pynvml.nvmlShutdown()
    poller.close()
    ring.close()


# ------------------------------------------------------------------------------------------------ host-side component mirror
def test_xid_component_check_and_state(ctx):
    """C++ mirror of the xid component (csrc/host_component.cpp): Check() scans on the GPU (xid/component.go:255-311), streaming
    ingestion + evolveHealthyState (component.go:468-611, health_state.go:57-128), reboot clears, SetHealthy trims."""
    import json
    L = g.lib()
    L.gpudh_xid_component_new.restype = C.c_void_p
    G = synth.golden("xid_kmsg.json")
    lines = G["dmesg_xid_119"]["lines"] + [G["inject_messages"]["known"]["63"]["message"], "NVRM: Xid (PCI:0000:04:00): 31, pid=1, name=a, mmu fault"]
    buf = "\n".join(lines).encode()
    for row_remap, want_n in ((1, 6), (0, 7)):      # Xid 63 is discarded when row remapping is supported (component.go:290)
        comp = C.c_void_p(L.gpudh_xid_component_new(ctx._h, 0, row_remap, 2))
        L.gpudh_xid_component_set_source(comp, buf, C.c_int64(len(buf)), 0, C.c_int64(0))
        health, summary = C.c_int32(), C.create_string_buffer(256)
        n = L.gpudh_xid_component_check(comp, C.byref(health), summary, 256, 1, C.c_int64(1740327858))
        assert n == want_n
        assert summary.value.decode() == "matched %d xid errors from %d kmsg(s)" % (want_n, len(lines))
        assert health.value == 2                      # Xid 119 is Fatal -> Unhealthy
        out = C.create_string_buffer(2048)
        L.gpudh_xid_component_state_json(comp, out, 2048)
        st = json.loads(out.value)
        assert st["health"] == "Unhealthy" and st["name"] == "error_xid" and st["suggested_actions"]["repair_actions"] == ["REBOOT_SYSTEM"]
        # the identical events are not inserted twice (eventBucket.Find, component.go:555-563)
        n_ev = L.gpudh_xid_component_n_events(comp)
        L.gpudh_xid_component_check(comp, C.byref(health), summary, 256, 1, C.c_int64(1740327858))
        assert L.gpudh_xid_component_n_events(comp) == n_ev
        # a reboot after the errors clears a REBOOT_SYSTEM state
        L.gpudh_xid_component_reboot(comp, C.c_int64(1740327900))
        L.gpudh_xid_component_state_json(comp, out, 2048)
        assert json.loads(out.value)["health"] == "Healthy"
        L.gpudh_xid_component_free(comp)


def test_component_objects_of_the_three_paths(ctx):
    """components.Component (components/types.go:20-66) through the C ABI (gpud_component_*): Start is non-blocking and spawns the ticker,
    LastHealthStates is "no data yet" before the first check, Check embeds its result, Events(since) is strictly after `since`, newest
    first, Close stops the ticker; one object per path this library replaces."""
    import time
    # ---- xid: scan + persist + evolve ----
    G = synth.golden("xid_kmsg.json")
    lines = G["dmesg_xid_119"]["lines"] + ["NVRM: Xid (PCI:0000:04:00): 31, pid=1, name=a, mmu fault"]
    x = g.capi.Component(ctx, "accelerator-nvidia-error-xid", row_remapping_supported=1)
    assert x.name() == "accelerator-nvidia-error-xid"
    st = x.last_health_states()
    assert len(st) == 1 and st[0]["health"] == "Healthy"
    x.xid_set_source("\n".join(lines).encode())
    health, reason = x.check()
    assert health == 2 and reason == "matched 6 xid errors from %d kmsg(s)" % len(lines)
    st = x.last_health_states()
    assert st[0]["health"] == "Unhealthy" and st[0]["suggested_actions"]["repair_actions"] == ["REBOOT_SYSTEM"] and "XID 119" in st[0]["reason"]
    ev = x.events(0)
    # five identical Xid 119 lines of one second are one event for the bucket (eventBucket.Find, component.go:555-563), the Xid 31 another
    assert len(ev) == 2 and all(e["component"] == "accelerator-nvidia-error-xid" and e["name"] == "error_xid" for e in ev)
    assert sorted(e["type"] for e in ev) == ["Fatal", "Warning"]
    assert [e["time"] for e in ev] == sorted((e["time"] for e in ev), reverse=True)
    now = int(time.time())
    assert x.events(now + 5) == []                                  # strictly after `since` (pkg/eventstore/database.go:330)
    x.check()
    assert len(x.events(0)) in (2, 4)                               # a check within the same second inserts nothing new
    x.xid_add_reboot(now + 60)
    assert x.last_health_states()[0]["health"] == "Healthy"         # a reboot after the errors clears REBOOT_SYSTEM
    x.close()
    # ---- temperature: Start -> ticker -> Check every interval; the polls land in the component's ring ----
    try:
        t = g.capi.Component(ctx, "accelerator-nvidia-temperature")
    except g.GpudError as e:
        pytest.skip("no NVML on this host: %s" % e)
    assert t.last_health_states()[0]["reason"] == "no data yet"
    t0 = time.perf_counter()
    t.start(20)
    assert time.perf_counter() - t0 < 0.5                           # Start does not block
    deadline = time.time() + 5
    while t.checks() < 5 and time.time() < deadline:
        time.sleep(0.01)
    assert t.checks() >= 5
    st = t.last_health_states()[0]
    assert st["component"] == st["name"] == "accelerator-nvidia-temperature" and st["health"] == "Healthy"
    assert st["reason"] == "all 1 GPU(s) were checked, no temperature issue found"
    assert t.events(0) == []
    t.stop()
    n = t.checks()
    time.sleep(0.1)
    assert t.checks() == n                                          # Close stopped the ticker
    t.close()
    t2 = g.capi.Component(ctx, "accelerator-nvidia-temperature", margin_threshold_c=200)
    health, reason = t2.check()
    assert health == 1 and "margin left to slowdown" in reason     # Degraded through the margin rule on a real reading
    assert t2.ring_handle(0)
    t2.close()
    # ---- nvlink: NVML records -> peer-store gather -> verdict ----
    nv = g.capi.Component(ctx, "accelerator-nvidia-nvlink")
    health, reason = nv.check()
    assert health == 0 and reason == "all 1 GPU(s) were checked, no nvlink issue found"
    nv2 = g.capi.Component(ctx, "accelerator-nvidia-nvlink", nvlink_at_least=2)       # a threshold one GPU cannot meet
    health, reason = nv2.check()
    assert health == 2 and "nvlink" in reason.lower()
    assert nv2.last_health_states()[0]["health"] == "Unhealthy"
    nv.close(); nv2.close()


def test_ring_full_shape_equals_the_oracle(ctx):
    """BASELINE configs[3] on one GPU, the WHOLE result: 512 fields x 1 Mi samples of the SURVEY 8(d) stream (gauges + spikes + monotone
    counters), every one of the 512 x 1049 windows and the W = CAP range against the C oracle - bit-exact min / max / p99 / n_over,
    mean / EMA within 1e-6 relative to the value (the achieved error is ~1e-14)."""
    import torch
    import synth_device as sd
    from oracle import coracle
    F, cap, W = 512, 1 << 20, 1000
    seed = 0x67707564
    thr = sd.thresholds("survey", F, cap, seed)
    r = g.Ring(ctx, F, cap, W, thresholds=thr)
    host = np.empty((F, cap), dtype=np.float64)
    sd.fill_ring(r, "survey", F, cap, seed, torch.device("cuda", 0), host_copy=host)
    got = r.reduce_all()
    want = coracle.windows_fields(host, W, thr)
    for k in ("min", "max", "p99"):
        assert np.array_equal(got[k].view(np.uint64), want[k].view(np.uint64)), k
    assert np.array_equal(got["n_over"].astype(np.uint64), want["n_over"].astype(np.uint64)) and int(want["n_over"].sum()) > 100000
    for k in ("mean", "ema"):
        rel = np.abs(got[k] - want[k]) / np.maximum(np.abs(want[k]), 1e-300)
        assert float(rel.max()) <= 1e-6, (k, float(rel.max()))
    rr = r.reduce_range(0)
    assert r.range_stats()[2] == 0                      # no field needed the radix fallback on this stream
    wr = coracle.windows_fields(host, cap, thr, alpha=2.0 / (W + 1.0))
    for k in ("min", "max", "p99"):
        assert np.array_equal(rr[k].view(np.uint64), wr[k][:, 0].view(np.uint64)), k
    assert np.array_equal(rr["n_over"].astype(np.uint64), wr["n_over"][:, 0].astype(np.uint64))
    for k in ("mean", "ema"):
        assert float(np.max(np.abs(rr[k] - wr[k][:, 0]) / np.maximum(np.abs(wr[k][:, 0]), 1e-300))) <= 1e-6, k
    r.close()


@pytest.mark.gpu
def test_poller_gpm_metrics_against_nvml(ctx):
    """GetGPMMetrics (gpm/gpm.go:65-149): support flag equals NVML's; with a float32 / float64 kernel load running, the nine metrics
    are percentages, the loaded pipes read non-zero, and a second reading through pynvml over the same kind of interval agrees on
    which of them are busy.  The ring source appends one float64 row per interval."""
    import threading
    import pynvml
    import torch
    pynvml.nvmlInit()
    ring = g.Ring(ctx, 9, 64, 8)
    iring = g.Ring(ctx, len(g.POLL_FIELDS), 64, 8)
    poller = g.Poller(ctx, iring)
    devs, _ = g.capi.nvml_devices()
    h = pynvml.nvmlDeviceGetHandleByIndex([d for d in devs if d.cuda_device == 0][0].index)
    want_sup = bool(pynvml.nvmlGpmQueryDeviceSupport(h).isSupportedDevice)
    assert poller.gpm_supported() == want_sup
    with pytest.raises(g.GpudError):                 # every poll source checks its row width against the ring it is to feed
        g.Poller(ctx, ring)
    with pytest.raises(g.GpudError):
        poller.poll_gpm(iring, 1, 10)
    with pytest.raises(g.GpudError):
        poller.poll_fields(ring, 1)
    if not want_sup:
        m = poller.gpm_metrics(50)
        assert m.supported == 0 and g.capi.gpm_check([m]) == (0, "GPM not supported")
        return
    s0 = pynvml.nvmlGpmSampleAlloc()
    try:                                             # some hosts report GPM support and then refuse every sample (NVML_ERROR_UNKNOWN)
        pynvml.nvmlGpmSampleGet(h, s0)
    except pynvml.NVMLError as e:
        import re
        for call in (lambda: poller.gpm_metrics(10), lambda: poller.poll_gpm(ring, 1, 10)):
            with pytest.raises(g.GpudError, match=re.escape(str(e))):   # NVML's refusal is passed on, no reading is made up
                call()
        pytest.skip("NVML reports GPM support but refuses GPM samples on this host: %s" % e)
    finally:
        pynvml.nvmlGpmSampleFree(s0)
    stop = threading.Event()

    def load():
        a = torch.randn(4096, 4096, device="cuda")
        d = torch.randn(2048, 2048, device="cuda", dtype=torch.float64)
        torch.backends.cuda.matmul.allow_tf32 = False
        while not stop.is_set():
            (a * 1.0001 + 0.5).sum()
            (d * 1.0001 + 0.5).sum()
            torch.cuda.synchronize()
    t = threading.Thread(target=load)
    t.start()
    try:
        import time
        time.sleep(0.3)
        m = poller.gpm_metrics(400)
        s1, s2 = pynvml.nvmlGpmSampleAlloc(), pynvml.nvmlGpmSampleAlloc()
        pynvml.nvmlGpmSampleGet(h, s1)
        time.sleep(0.4)
        pynvml.nvmlGpmSampleGet(h, s2)
        q = pynvml.c_nvmlGpmMetricsGet_t()
        q.version, q.numMetrics, q.sample1, q.sample2 = 1, 9, s1, s2
        for i, mid in enumerate(g.capi.GPM_METRIC_IDS):
            q.metrics[i].metricId = mid
        pynvml.nvmlGpmMetricsGet(q)
        ref = [q.metrics[i].value for i in range(9)]
        sec = poller.poll_gpm(ring, 3, 150)
        pynvml.nvmlGpmSampleFree(s1)
        pynvml.nvmlGpmSampleFree(s2)
    finally:
        stop.set()
        t.join()
    assert m.supported == 1 and 0.39 < m.sample_seconds < 1.0
    got = list(m.value)
    assert all(rc == 0 for rc in m.nvml_rc), list(m.nvml_rc)
    assert all(0.0 <= v <= 100.0 for v in got), got
    d = m.as_dict()
    assert d["sm_occupancy"] > 0.0 and d["fp32_util"] > 0.0 and d["fp64_util"] > 0.0, d
    assert [v > 0.05 for v in got] == [v > 0.05 for v in ref] or all(abs(a - b) < 15.0 for a, b in zip(got, ref)), (got, ref)
    assert g.capi.gpm_check([m]) == (0, "all 1 GPU(s) were checked, no GPM issue found")
    assert 0.44 < sec < 2.0
    ring.sync()
    assert ring.counts()[0] == 3
