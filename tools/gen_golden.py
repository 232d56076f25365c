#!/usr/bin/env python3
"""Extract the reference's own table-driven test vectors and fixtures into tests/golden/*.json.

The reference tests are Go; no Go toolchain exists in this image, so the vectors (inputs and the
expected values the Go tests assert) are lifted *as data* by parsing the struct-literal tables.
Every output record carries `src` = reference file:line of the test function it came from.

Run in the build container (needs /root/reference).  Outputs are committed; the GPU box only
reads tests/golden/.
"""
import json
import os
import re
import sys

REF = os.environ.get("GPUD_REFERENCE", "/root/reference")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests/golden")

TOK = re.compile(r"""
    (?P<ws>\s+|//[^\n]*|/\*.*?\*/)
  | (?P<str>"(?:[^"\\]|\\.)*"|`[^`]*`)
  | (?P<num>-?0[xX][0-9a-fA-F_]+|-?\d[\d_]*(?:\.\d+)?(?:[eE][-+]?\d+)?)
  | (?P<id>[A-Za-z_][\w\.]*)
  | (?P<p>[{}\[\](),:+*&\-<>=!|;/%])
""", re.X | re.S)


def unquote(lit):
    if lit.startswith("`"):
        return lit[1:-1]
    body = lit[1:-1]
    out, i = [], 0
    simple = {"n": "\n", "t": "\t", '"': '"', "\\": "\\", "'": "'", "r": "\r", "a": "\a", "b": "\b", "f": "\f", "v": "\v"}
    while i < len(body):
        c = body[i]
        if c != "\\":
            out.append(c); i += 1; continue
        n = body[i + 1]
        if n in simple:
            out.append(simple[n]); i += 2
        elif n == "x":
            out.append(chr(int(body[i + 2:i + 4], 16))); i += 4
        elif n == "u":
            out.append(chr(int(body[i + 2:i + 6], 16))); i += 6
        elif n in "01234567":
            out.append(chr(int(body[i + 1:i + 4], 8))); i += 4
        else:
            raise ValueError(n)
    return "".join(out)


def tokenize(src):
    pos, toks = 0, []
    while pos < len(src):
        m = TOK.match(src, pos)
        if not m:
            raise ValueError("tokenize at %r" % src[pos:pos + 40])
        pos = m.end()
        k = m.lastgroup
        if k == "ws":
            continue
        toks.append((k, m.group(k)))
    return toks


class P:
    def __init__(self, toks):
        self.t, self.i = toks, 0

    def peek(self, o=0):
        return self.t[self.i + o] if self.i + o < len(self.t) else ("eof", "")

    def next(self):
        x = self.peek(); self.i += 1; return x

    def expect(self, v):
        x = self.next()
        assert x[1] == v, (x, v, self.t[max(0, self.i - 8):self.i + 4])

    def skip_type(self):
        """Skip a type prefix such as []apiv1.RepairActionType, &Foo, map[string]string, *T."""
        while True:
            k, v = self.peek()
            if v in ("&", "*"):
                self.next()
            elif v == "[":
                self.next()
                while self.peek()[1] != "]":
                    self.next()
                self.next()
            elif k == "id" and v == "map":
                self.next(); self.expect("[")
                while self.peek()[1] != "]":
                    self.next()
                self.next()
            elif k == "id" and v == "struct":
                self.next(); self.expect("{")
                d = 1
                while d:
                    x = self.next()[1]
                    d += (x == "{") - (x == "}")
            elif k == "id" and self.peek(1)[1] == "{":
                self.next()
                return
            else:
                return

    def value(self):
        k, v = self.peek()
        if k == "str":
            s = unquote(self.next()[1])
            while self.peek()[1] == "+" and self.peek(1)[0] == "str":
                self.next(); s += unquote(self.next()[1])
            return s
        if k == "num":
            self.next()
            v = v.replace("_", "")
            try:
                return int(v, 0)
            except ValueError:
                return float(v)
        if v == "-" and self.peek(1)[0] == "num":
            self.next()
            return -self.value()
        if v in ("&", "*", "[") or (k == "id" and (self.peek(1)[1] == "{" or v in ("map", "struct"))):
            self.skip_type()
            return self.composite()
        if v == "{":
            return self.composite()
        if k == "id":
            self.next()
            if self.peek()[1] == "(":     # call: keep as opaque text  fn(args)
                depth, parts = 0, [v]
                while True:
                    x = self.next()
                    parts.append(x[1])
                    depth += (x[1] == "(") - (x[1] == ")")
                    if depth == 0:
                        break
                txt = "".join(parts)
                while self.peek()[1] == ".":   # unlikely
                    break
                return {"$call": txt}
            if v == "true":
                return True
            if v == "false":
                return False
            if v == "nil":
                return None
            return {"$id": v}
        raise ValueError("value at %r" % (self.t[self.i:self.i + 6],))

    def composite(self):
        self.expect("{")
        items, keyed = [], None
        while self.peek()[1] != "}":
            if (self.peek()[0] in ("id", "str", "num")) and self.peek(1)[1] == ":":
                kk = self.next()
                key = unquote(kk[1]) if kk[0] == "str" else kk[1]
                self.next()
                items.append((key, self.value()))
                keyed = True
            else:
                items.append(self.value())
            # tolerate binary expressions we do not need (e.g. a * b) by skipping to , or }
            while self.peek()[1] not in (",", "}"):
                self.next()
            if self.peek()[1] == ",":
                self.next()
        self.expect("}")
        if keyed:
            return {k: v for k, v in items}
        return items


def find_func(src, name):
    m = re.search(r"^func %s\(" % re.escape(name), src, re.M)
    assert m, name
    line = src.count("\n", 0, m.start()) + 1
    # function body ends at next "\n}\n"
    end = src.index("\n}\n", m.start())
    return src[m.start():end], line


def table(path, func, var=None):
    """Return rows (list of dict) of the first `[]struct{...}{...}` table in func."""
    src = open(os.path.join(REF, path)).read()
    body, line = find_func(src, func)
    pat = r"(?:%s)\s*:?=\s*\[\]struct\s*\{" % (var or r"\w+")
    m = re.search(pat, body)
    assert m, (path, func)
    decl_end = body.index("}{", m.end())
    fields = []
    for ln in body[m.end():decl_end].split("\n"):
        ln = ln.split("//")[0].strip()
        if not ln:
            continue
        parts = ln.split()
        names = [p.rstrip(",") for p in parts[:-1]] if len(parts) > 1 else [parts[0]]
        # "a, b int" declares two fields
        fields.extend(names if len(parts) > 1 else [])
    toks = tokenize(body[decl_end + 1:])
    rows = P(toks).composite()
    out = []
    for r in rows:
        if isinstance(r, list):
            r = {fields[i]: v for i, v in enumerate(r)}
        out.append(r)
    return out, "%s:%d" % (path, line)


def ident(v):
    """apiv1.EventTypeWarning -> 'Warning' etc."""
    if isinstance(v, dict) and "$id" in v:
        s = v["$id"].split(".")[-1]
        for pre in ("EventType", "RepairActionType", "HealthStateType"):
            if s.startswith(pre):
                return s[len(pre):]
        return s
    if isinstance(v, list):
        return [ident(x) for x in v]
    if isinstance(v, dict):
        return {k: ident(x) for k, x in v.items()}
    return v


def dump(name, obj):
    os.makedirs(OUT, exist_ok=True)
    with open(os.path.join(OUT, name), "w") as f:
        json.dump(obj, f, indent=1, ensure_ascii=False)
        f.write("\n")
    n = sum(len(v["rows"]) if isinstance(v, dict) and "rows" in v else 1 for v in obj.values()) if isinstance(obj, dict) else len(obj)
    print("%-32s %d vectors" % (name, n))


def main():
    X = "components/accelerator/nvidia/xid/"
    S = "components/accelerator/nvidia/sxid/"
    g = {}
    for key, path, fn in [
        ("extract_xid", X + "kmsg_test.go", "TestExtractNVRMXid"),
        ("extract_device", X + "kmsg_test.go", "TestExtractNVRMXidDeviceUUID"),
        ("match", X + "kmsg_test.go", "TestMatch"),
        ("normalize_bdf", X + "kmsg_test.go", "TestNormalizePCIBDF"),
        ("extended", X + "kmsg_extended_test.go", "TestExtractNVRMXidInfoExtended"),
        ("subcode", X + "kmsg_extended_test.go", "TestCalculateSubCode"),
        ("detail_with_subcode", X + "kmsg_extended_test.go", "TestGetDetailWithSubCode"),
        ("match_nvlink_examples", X + "kmsg_extended_test.go", "TestMatchNVLinkExamples"),
        ("nvlink_log_coverage", X + "nvlink_logs_test.go", "Test_NVLinkLogCoverage"),
    ]:
        rows, src = table(path, fn)
        g[key] = {"src": src, "rows": ident(rows)}
    # single-assert tests
    g["short_match"] = {"src": X + "kmsg_extended_test.go:350", "rows": [
        {"line": "NVRM: Xid (PCI:0018:01:00): 149, NETIR Fatal XC0 i0 Link -1 (0x000fe406", "extended_nil": True}]}
    g["unknown_code"] = {"src": X + "kmsg_test.go:289", "rows": [
        {"input": "NVRM: Xid (PCI:0000:05:00): 99999, unknown error", "expectNil": True}]}
    g["status_specific"] = {"src": X + "xid_test.go:13", "rows": [
        {"xid": 144, "unit": "SAW_MVB", "severity": "Nonfatal", "intrinfo": 0x21, "error_status": 0x8, "event": "Warning"},
        {"xid": 144, "unit": "SAW_MVB", "severity": "Nonfatal", "intrinfo": 0x21, "error_status": 0x2, "event": "Fatal",
         "actions_contain": ["RebootSystem"]},
        {"xid": 144, "unit": "SAW_MVB", "severity": "Nonfatal", "intrinfo": 0x21, "error_status": 0xDEADBEEF, "event": "Warning"}]}
    # fixture file: 43 dmesg lines -> exactly 5 x (119, PCI:0000:9b:00)   (kmsg_test.go:248-287)
    lines = open(os.path.join(REF, X, "testdata/dmesg-with-xid-119.log")).read().split("\n")
    g["dmesg_xid_119"] = {"src": X + "kmsg_test.go:248", "lines": lines,
                          "rows": [{"xid": 119, "device": "PCI:0000:9b:00"}] * 5}
    # injectable messages (kmsg.go:278-311): known ones + the generic template
    src = open(os.path.join(REF, X, "kmsg.go")).read()
    msgs = {}
    for m in re.finditer(r"\n\t(\d+): \{\n\t\tPriority: \"(\w+)\",\n\t\tMessage:\s+(\"(?:[^\"\\]|\\.)*\"),", src):
        msgs[int(m.group(1))] = {"priority": m.group(2), "message": unquote(m.group(3))}
    assert sorted(msgs) == [63, 64, 69, 74, 79], sorted(msgs)
    g["inject_messages"] = {"src": X + "kmsg.go:278", "known": {str(k): v for k, v in msgs.items()},
                            "template": "NVRM: Xid (PCI:0000:04:00): %d, unknown", "rows": []}
    dump("xid_kmsg.json", g)

    s = {}
    for key, fn in [("extract_sxid", "TestExtractNVSwitchSXid"), ("extract_device", "TestExtractNVSwitchSXidDeviceUUID"),
                    ("match", "TestMatch")]:
        rows, src = table(S + "kmsg_test.go", fn)
        s[key] = {"src": src, "rows": ident(rows)}
    dump("sxid_kmsg.json", s)

    # pkg/kmsg parseLine + fixtures
    K = "pkg/kmsg/"
    k = {}
    ksrc = open(os.path.join(REF, K, "watcher_test.go")).read()
    for fn in ("Test_parseLineComprehensive",):           # the table test; the others are literal calls, extracted below
        try:
            rows, src = table(K + "watcher_test.go", fn)
            k[fn] = {"src": src, "rows": ident(rows)}
        except Exception as e:  # noqa
            print("  skip", fn, type(e).__name__, e)
    # the non-table parseLine tests: every `input := "..."` / parseLine(bootTime, "...") literal with the equalities asserted after it
    calls = []
    for fn in ("Test_parseLine", "Test_parseLineWithDifferentBootTimes", "Test_parseLineEdgeCases"):
        body, line = find_func(ksrc, fn)
        for seg in (re.split(r"\n\tt\.Run\(", body)[1:] if fn == "Test_parseLineEdgeCases" else [body]):
            m = re.search(r'(?:input := |parseLine\(bootTime, )"((?:[^"\\]|\\.)*)"', seg)
            row = {"func": fn, "line": line, "input": bytes(m.group(1), "utf-8").decode("unicode_escape")}
            for pat, key, conv in ((r'assert\.Equal\(t, msg\.Message, "((?:[^"\\]|\\.)*)"\)', "message", str), (r'assert\.Equal\(t, "((?:[^"\\]|\\.)*)", msg\.Message\)', "message", str),
                                   (r"assert\.Equal\(t, msg\.Priority, (-?\d+)\)", "priority", int), (r"assert\.Equal\(t, (-?\d+), msg\.Priority\)", "priority", int),
                                   (r"assert\.Equal\(t, msg\.SequenceNumber, (-?\d+)\)", "sequence", int), (r"assert\.Equal\(t, (-?\d+), msg\.SequenceNumber\)", "sequence", int),
                                   (r"bootTime\.Add\((\d+)\s*\*\s*time\.Microsecond\)", "usec", int)):
                mm = re.search(pat, seg)
                if mm:
                    row[key] = conv(mm.group(1))
            calls.append(row)
    k["parse_line_calls"] = {"src": K + "watcher_test.go", "rows": calls}
    for fx in ("kmsg.1.log", "kmsg.2.peermem.log"):
        p = os.path.join(REF, K, "testdata", fx)
        if os.path.exists(p):
            k["fixture:" + fx] = {"src": K + "testdata/" + fx, "rows": [],
                                  "records": open(p, encoding="utf-8", errors="surrogateescape").read().split("\n")}
    dump("pkg_kmsg.json", k)

    # SURVEY §8(f).1: the next kmsg matchers that ride the same scanner
    N = "components/accelerator/nvidia/"
    ext = {}
    for key, path, fn in [("nccl_has", N + "nccl/kmsg_matcher_test.go", "TestHasNCCLSegfaultInLibnccl"),
                          ("nccl_match", N + "nccl/kmsg_matcher_test.go", "TestMatch"),
                          ("peermem_has", N + "peermem/kmsg_matcher_test.go", "TestHasPeermemInvalidContext"),
                          ("peermem_match", N + "peermem/kmsg_matcher_test.go", "TestMatch")]:
        rows, src = table(path, fn)
        ext[key] = {"src": src, "rows": ident(rows)}
    ext["constants"] = {"src": N + "nccl/kmsg_matcher.go:11-13 ; " + N + "peermem/kmsg_matcher.go:13-15", "rows": [],
                        "nccl": {"event": "nvidia_nccl_segfault_in_libnccl", "message": "NCCL communication error (segfault in libnccl.so)"},
                        "peermem": {"event": "nvidia_peermem_invalid_context", "message": "peermem error detected (possible GPU communication issue)"}}
    dump("ext_kmsg.json", ext)

    # ---- the stateless line matchers of infiniband / cpu / os / disk (SURVEY 8f.1, second batch) ----
    def consts(path):
        """name -> string for every `name = "..."` / `name = `...`` constant of a Go file (behavioural data only)"""
        out = {}
        for i, ln in enumerate(open(os.path.join(REF, path)).read().split("\n"), 1):
            m = re.match(r'^\s*(?:const\s+)?(\w+)\s*=\s*(?:"((?:[^"\\]|\\.)*)"|`([^`]*)`)\s*$', ln)
            if m:
                out[m.group(1)] = {"value": m.group(3) if m.group(3) is not None else bytes(m.group(2), "utf-8").decode("unicode_escape"), "line": i}
        return out

    def resolve_msgs(path, func, field, rows, cs):
        """re-read `field: <expr>,` of every row as Go source: identifiers -> constants, strings literal, + concatenates"""
        body, _ = find_func(open(os.path.join(REF, path)).read(), func)
        exprs = re.findall(r"\b%s:\s*(.+?),\s*\n" % field, body)
        assert len(exprs) == len(rows), (path, func, field, len(exprs), len(rows))
        for r, e in zip(rows, exprs):
            val = ""
            for tok in re.findall(r'"(?:[^"\\]|\\.)*"|\w+', e):
                val += bytes(tok[1:-1], "utf-8").decode("unicode_escape") if tok.startswith('"') else cs[tok]["value"]
            r[field] = val

    comps = {"infiniband": (N + "infiniband/", [("pci_power_insufficient", "TestHasPCIPowerInsufficient", "regexPCIPowerInsufficient", "eventPCIPowerInsufficient", "messagePCIPowerInsufficient"),
                                                 ("port_module_high_temperature", "TestHasPortModuleHighTemperature", "regexPortModuleHighTemperature", "eventPortModuleHighTemperature", "messagePortModuleHighTemperature"),
                                                 ("access_reg_failed", "TestHasAccessRegFailed", "regexAccessRegFailed", "eventAccessRegFailed", "messageAccessRegFailed")], "wantEvent"),
             "cpu": ("components/cpu/", [("blocked_too_long", "TestHasBlockedTooLong", "regexBlockedTooLong", "eventBlockedTooLong", "messageBlockedTooLong"),
                                         ("soft_lockup", "TestHasSoftLockup", "regexSoftLockup", "eventSoftLockup", "messageSoftLockup")], "wantName"),
             "os": ("components/os/", [("vfs_file_max", "TestHasVFSFileMaxLimitReached", "regexVFSFileMaxLimitReached", "eventNameVFSFileMaxLimitReached", "messageVFSFileMaxLimitReached")], "wantName"),
             "disk": ("components/disk/", [("raid_array_failure", "TestHasRAIDArrayFailure", "regexRAIDArrayFailure", "eventRAIDArrayFailure", "messageRAIDArrayFailure"),
                                           ("filesystem_read_only", "TestHasFilesystemReadOnly", "regexFilesystemReadOnly", "eventFilesystemReadOnly", "messageFilesystemReadOnly"),
                                           ("nvme_path_failure", "TestHasNVMePathFailure", "regexNVMePathFailure", "eventNVMePathFailure", "messageNVMePathFailure"),
                                           ("nvme_timeout", "TestHasNVMeTimeout", "regexNVMeTimeout", "eventNVMeTimeout", "messageNVMeTimeout"),
                                           ("nvme_device_disabled", "TestHasNVMeDeviceDisabled", "regexNVMeDeviceDisabled", "eventNVMeDeviceDisabled", "messageNVMeDeviceDisabled"),
                                           ("beyond_end_of_device", "TestHasBeyondEndOfDevice", "regexBeyondEndOfDevice", "eventBeyondEndOfDevice", "messageBeyondEndOfDevice"),
                                           ("buffer_io_error", "TestHasBufferIOError", "regexBufferIOError", "eventBufferIOError", "messageBufferIOError"),
                                           ("superblock_write_error", "TestHasSuperblockWriteError", "regexSuperblockWriteError", "eventSuperblockWriteError", "messageSuperblockWriteError")], "wantEventName")}
    ext2 = {}
    for comp, (d, pats, ev_field) in comps.items():
        cs = consts(d + "kmsg_matcher.go")
        plist = []
        for key, fn, rx, ev, msg in pats:
            rows, src = table(d + "kmsg_matcher_test.go", fn)
            ext2["%s.%s" % (comp, key)] = {"src": src, "rows": ident(rows)}
            plist.append({"key": key, "regex": cs[rx]["value"], "event": cs[ev]["value"], "message": cs[msg]["value"],
                          "src": "%skmsg_matcher.go:%d" % (d, cs[rx]["line"])})
        rows, src = table(d + "kmsg_matcher_test.go", "TestMatch")
        rows = ident(rows)
        resolve_msgs(d + "kmsg_matcher_test.go", "TestMatch", ev_field, rows, cs)
        resolve_msgs(d + "kmsg_matcher_test.go", "TestMatch", "wantMessage", rows, cs)
        for r in rows:
            r["wantEvent"] = r.pop(ev_field)
        ext2["%s.match" % comp] = {"src": src, "rows": rows}
        ext2["%s.patterns" % comp] = {"src": d + "kmsg_matcher.go", "rows": [], "patterns": plist}
    cs = consts(N + "infiniband/kmsg_matcher.go")
    rows, src = table(N + "infiniband/kmsg_matcher_test.go", "TestAccessRegFailedMessage")
    rows = ident(rows)
    resolve_msgs(N + "infiniband/kmsg_matcher_test.go", "TestAccessRegFailedMessage", "want", rows, cs)
    ext2["infiniband.access_reg_message"] = {"src": src, "rows": rows, "regexPCIDevice": cs["regexPCIDevice"]["value"], "prefix": cs["pciDeviceMessagePrefix"]["value"]}
    dump("ext2_kmsg.json", ext2)

    # ---- the two STATEFUL matchers: os kernel-panic assembly and the memory OOM parser ----
    ext3 = {}
    OSD, MEMD = "components/os/", "components/memory/"
    cs = consts(OSD + "kmsg_matcher.go")
    rows, src = table(OSD + "kmsg_matcher_test.go", "TestKernelPanicDetection")
    rows = ident(rows)
    for r in rows:
        r["wantEventName"] = cs[r["wantEventName"]]["value"] if r["wantEventName"] in cs else r["wantEventName"]
        # the kernel's hung-task hint quotes a shell command that changes a kernel setting; the fixture keeps the line (it comes
        # before the panic and matches no pattern) in plain words, so no file in the repository carries that command
        r["logLines"] = [re.sub(r'"echo 0 [^"]*/hung_task_timeout_secs"', "Setting kernel.hung_task_timeout_secs to 0", l) for l in r["logLines"]]
    ext3["os.panic_detection"] = {"src": src, "rows": rows, "note": "lines fed to Match until the first non-empty event"}
    rows, src = table(OSD + "kmsg_matcher_test.go", "TestKernelPanicStatefulMatcher")
    rows = ident(rows)
    for r in rows:
        r["scenario"] = [[st[0], cs[st[1]]["value"] if st[1] in cs else st[1], st[2]] for st in r["scenario"]]
    ext3["os.panic_stateful"] = {"src": src, "rows": rows, "note": "scenario steps: [line, eventName, message] through one matcher instance"}
    body, line = find_func(open(os.path.join(REF, OSD + "kmsg_matcher_test.go")).read(), "TestKernelPanicHelperFunctions")
    starts = [{"line": bytes(m.group(1), "utf-8").decode("unicode_escape"), "want": m.group(2) == "true"}
              for m in re.finditer(r'\{"((?:[^"\\\\]|\\\\.)*)",\s*(true|false)\}', body)]
    ext3["os.panic_start"] = {"src": OSD + "kmsg_matcher_test.go:%d" % line, "rows": starts}
    cpu = []
    for m in re.finditer(r'\{\s*line:\s*"((?:[^"\\\\]|\\\\.)*)",(?:\s*//[^\n]*)?\s*wantFound:\s*(true|false),((?:\s*want\w+:\s*[^,]+,)*)\s*\}', body):
        r = {"line": bytes(m.group(1), "utf-8").decode("unicode_escape"), "wantFound": m.group(2) == "true"}
        for k, v in re.findall(r'(want\w+):\s*([^,]+),', m.group(3)):
            r[k] = int(v) if v.strip().isdigit() else v.strip().strip('"')
        cpu.append(r)
    ext3["os.panic_cpu_pid"] = {"src": OSD + "kmsg_matcher_test.go:%d" % line, "rows": cpu}
    ext3["os.max_lines"] = {"src": OSD + "kmsg_matcher_test.go:712 ; " + OSD + "kmsg_matcher.go:64", "rows": [],
                            "max_lines_after_start": 10, "fallback_message": "Kernel panic detected (no CPU/PID info found)",
                            "event": cs["eventNameKernelPanic"]["value"]}
    for key, fn in [("memory.match_func", "TestCreateMatchFunc"), ("memory.stream", "TestCreateMatchFuncStreamOOMs"),
                    ("memory.container_name", "TestGetContainerName"), ("memory.process_pid", "TestGetProcessNamePid"),
                    ("memory.oom_start", "TestCheckIfStartOfOomMessages"), ("memory.summary", "TestOomInstanceSummary")]:
        rows, src = table(MEMD + "kmsg_matcher_test.go", fn)
        ext3[key] = {"src": src, "rows": ident(rows)}
    dump("ext3_kmsg.json", ext3)

    # ---- SURVEY 8f.4: InfiniBand port drop / flap scans over snapshot series (infiniband/store/scan_drops.go, scan_flaps.go) ----
    IBD = N + "infiniband/store/"
    DUR = {"time.Second": 1, "time.Minute": 60, "time.Hour": 3600, "time.Millisecond": 0.001}

    def dur_seconds(expr):
        """30*time.Second / 1*time.Minute+30*time.Second / -5 * time.Minute -> seconds (float)"""
        total = 0.0
        for term in re.findall(r"[+-]?[^+-]+", expr.replace(" ", "")):
            sign = -1.0 if term.startswith("-") else 1.0
            term = term.lstrip("+-")
            val = 1.0
            for f in term.split("*"):
                val *= DUR[f] if f in DUR else float(f)
            total += sign * val
        return total

    def snapshot_cases(path, func):
        """cases of a `tests := []struct{ name; snapshots devPortSnapshots; expected int }` table: time offsets relative to baseTime"""
        body, line = find_func(open(os.path.join(REF, path)).read(), func)
        out = []
        for m in re.finditer(r'name:\s*"([^"]+)",\s*snapshots:\s*devPortSnapshots\{(.*?)\},\s*expected:\s*(\d+)', body, re.S):
            snaps = []
            for sm in re.finditer(r'createSnapshot\(baseTime(?:\.Add\(([^)]*)\))?,\s*"(\w+)",\s*(\d+)\)', m.group(2)):
                snaps.append({"t": dur_seconds(sm.group(1)) if sm.group(1) else 0.0, "state": sm.group(2), "total_link_downed": int(sm.group(3))})
            out.append({"name": m.group(1), "snapshots": snaps, "expected": int(m.group(3))})
        return out, "%s:%d" % (path, line)

    ib = {}
    rows, src = snapshot_cases(IBD + "scan_drops_test.go", "TestFindDrops")
    ib["drops"] = {"src": src, "rows": rows, "threshold_s": 240, "note": "threshold := 4 * time.Minute (scan_drops_test.go:27)"}
    rows, src = snapshot_cases(IBD + "scan_flaps_test.go", "TestFindFlaps")
    ib["flaps"] = {"src": src, "rows": rows, "down_interval_threshold_s": 25, "flap_back_to_active_threshold": 3,
                   "note": "downIntervalThreshold := 25 * time.Second, flapBackToActiveThreshold := 3 (scan_flaps_test.go:27-28)"}
    def snapshot_subtests(path, func, kind):
        """the t.Run sub-tests (and a bare body) of `func`: struct-literal snapshots, the call's thresholds, Len / index asserts"""
        body, line = find_func(open(os.path.join(REF, path)).read(), func)
        env = {m.group(1): m.group(2).strip() for m in re.finditer(r"(\w+)\s*:=\s*([^\n]+)", body)}
        blocks = re.split(r't\.Run\("', body)
        out = []
        for blk in blocks:
            name = blk.split('"', 1)[0] if blk is not blocks[0] else func
            snaps = [{"t": dur_seconds(m.group(1)) if m.group(1) else 0.0, "state": m.group(2), "total_link_downed": int(m.group(3))}
                     for m in re.finditer(r'\{ts:\s*baseTime(?:\.Add\(([^)]*)\))?,\s*state:\s*"(\w+)",\s*totalLinkDowned:\s*(\d+)\}', blk)]
            call = re.search(r"\.find(?:Drops|Flaps)\(device,\s*port,\s*([^)]*)\)", blk)
            ln = re.search(r"assert\.Len\(t,\s*result,\s*(\d+)", blk)
            if not call or not ln or "nilSnapshots" in blk:
                continue
            args = [a.strip() for a in call.group(1).split(",")]
            def val(a):
                a = env.get(a, a)
                return int(a) if re.fullmatch(r"\d+", a) else dur_seconds(a)
            row = {"name": name, "snapshots": snaps, "expected": int(ln.group(1)), "args": [val(a) for a in args]}
            ix = re.search(r"assert\.Equal\(t,\s*snapshots\[(\d+)\]\.ts,\s*(?:result\[0\]|flap|drop)\.ts\)", blk)
            if ix:
                row["expected_index"] = int(ix.group(1))
            out.append(row)
        return out, "%s:%d" % (path, line)

    edge = []
    for fn in ("TestFindDrops_EdgeCases", "TestFindDrops_ReasonMessage"):
        rows, src = snapshot_subtests(IBD + "scan_drops_test.go", fn, "drops")
        edge += [dict(r, kind="drops", src=src) for r in rows]
    for fn in ("TestFindFlaps_EdgeCases", "TestFindFlaps_ReasonMessage", "TestFindFlaps_ComplexScenarios"):
        rows, src = snapshot_subtests(IBD + "scan_flaps_test.go", fn, "flaps")
        edge += [dict(r, kind="flaps", src=src) for r in rows]
    ib["edge"] = {"src": IBD + "scan_drops_test.go:174,215 ; " + IBD + "scan_flaps_test.go:216,279,316", "rows": edge,
                  "note": "args = the thresholds of the call: drops [threshold_s], flaps [down_interval_s, flap_back_to_active]"}
    dump("ib_scans.json", ib)

    # ---- SURVEY 8f.2: the SQL of the event store and the metrics store, as the Go sources format it ----
    def go_fmt_sql(path, func, which=0):
        """the `which`-th backquoted or quoted fmt.Sprintf format string of `func`, with its %s arguments substituted"""
        src = open(os.path.join(REF, path)).read()
        body, line = find_func(src, func)
        cs = consts(path)
        cs["tableName"] = cs["table"] = {"value": "{table}"}
        fm = list(re.finditer(r'fmt\.Sprintf\(\s*(`[^`]*`|"(?:[^"\\]|\\.)*")\s*,([^;]*?)\)\s*[,)\n]', body, re.S))[which]
        f = fm.group(1)
        f = f[1:-1] if f.startswith("`") else bytes(f[1:-1], "utf-8").decode("unicode_escape")
        args = [a.strip() for a in re.sub(r"//[^\n]*", "", fm.group(2)).split(",") if a.strip()]
        vals = [cs[a]["value"] if a in cs else "{" + a + "}" for a in args]
        return f % tuple(vals[: f.count("%s")]), "%s:%d" % (path, line)

    sql = {}
    ES, MS = "pkg/eventstore/database.go", "pkg/metrics/store/sqlite.go"
    for key, path, func, which in [("event_create_table", ES, "createTable", 0), ("event_index_0", ES, "createTable", 1), ("event_index_1", ES, "createTable", 2),
                                   ("event_index_2", ES, "createTable", 3), ("event_insert", ES, "insertEvent", 0), ("event_get", ES, "getEvents", 0),
                                   ("event_table_name", ES, "defaultTableName", 0), ("event_latest", ES, "lastEvent", 0), ("event_purge", ES, "purgeEvents", 0), ("event_find", ES, "findEvent", 0), ("metrics_create_table", MS, "CreateTable", 0), ("metrics_insert_prefix", MS, "insert", 0)]:
        text, src = go_fmt_sql(path, func, which)
        sql[key] = {"src": src, "rows": [], "sql": text}
    sql["constants"] = {"src": ES + ":18 ; " + MS + ":22,36", "rows": [], "event_schema_version": consts(ES)["schemaVersion"]["value"],
                        "metrics_schema_version": consts(MS)["schemaVersion"]["value"]}
    body, line = find_func(open(os.path.join(REF, "pkg/eventstore/database_test.go")).read(), "Test_defaultTableName")
    tn = [{"name": m.group(1), "input": m.group(2), "expected": m.group(3) % consts(ES)["schemaVersion"]["value"]}
          for m in re.finditer(r'name:\s*"([^"]*)",\s*input:\s*"([^"]*)",\s*expected:\s*fmt\.Sprintf\("([^"]*)",\s*schemaVersion\)', body)]
    sql["table_names"] = {"src": "pkg/eventstore/database_test.go:%d" % line, "rows": tn}
    dump("store_sql.json", sql)

    # ---- xid buildMessage / health-state reason tests (xid/health_state_test.go:299-942) ----
    HS = N + "xid/health_state_test.go"
    hs_src = open(os.path.join(REF, HS)).read()
    xm = {}
    go_str = lambda lit: bytes(lit, "utf-8").decode("unicode_escape")
    # struct-literal tests: every `v := xidErrorEventDetail{...}`, the `r := v.buildMessage(...)` that follows, and the asserts on r
    lit_rows = []
    for fn in ("Test_buildMessage_SubCode", "Test_buildMessage_Format", "Test_HealthStateReason_UnknownXID", "Test_HealthStateReason_EmptyDescription"):
        body, line = find_func(hs_src, fn)
        for seg in (body.split("t.Run(")[1:] or [body]):
            lits = {}
            for m in re.finditer(r"(\w+) := xidErrorEventDetail\{(.*?)\n\t*\}", seg, re.S):
                f = {}
                for k, v in re.findall(r"(\w+):\s*(\"(?:[^\"\\]|\\.)*\"|0x[0-9a-fA-F]+|\d+),", m.group(2)):
                    f[k] = go_str(v[1:-1]) if v.startswith('"') else int(v, 0)
                lits[m.group(1)] = f
            for rv, lv in re.findall(r"(\w+) := (\w+)\.buildMessage\(nil\)", seg):
                eq = [go_str(x) for x in re.findall(r'assert\.Equal\(t, "((?:[^"\\]|\\.)*)", %s\)' % rv, seg)]
                co = [go_str(x) for x in re.findall(r'assert\.Contains\(t, %s, "((?:[^"\\]|\\.)*)"' % rv, seg)]
                lit_rows.append({"func": fn, "fields": lits[lv], "equal": eq[0] if eq else None, "contains": co})
    xm["literals"] = {"src": HS, "rows": lit_rows}
    rows, src = table(HS, "Test_HealthStateReason_StandardXIDs")
    xm["standard"] = {"src": src, "rows": [{"name": r["name"], "xid": r["xid"], "device_uuid": r["deviceUUID"], "description": r["description"],
                                            "contains": r["expectedContains"]} for r in rows], "bus_id": "0000:9b:00.0", "uuid": "GPU-test-uuid"}
    line_rows = []
    rows, src = table(HS, "Test_HealthStateReason_NVLinkXIDs")
    for r in rows:
        line_rows.append({"func": "Test_HealthStateReason_NVLinkXIDs", "name": r["name"], "line": r["kmsgLine"], "xid": r["expectedXid"], "sub_code": r["expectedSubCode"],
                          "contains": r["expectedContains"] + ["UUID:GPU-test-uuid"], "devices": {"GPU-test-uuid": "0000:04:00.0"}})
    rows, src = table(HS, "Test_StatusAwareMessages")
    for r in rows:
        line_rows.append({"func": "Test_StatusAwareMessages", "name": r["name"], "line": r["line"], "sub_code": r["expectedSub"], "event_type": ident(r["expectedEvent"]),
                          "contains": [r["expectedMnemonic"]], "devices": {}})
    rows, src = table(HS, "Test_MatchToEventMessageFlowFormatsMnemonic")
    for r in rows:
        line_rows.append({"func": "Test_MatchToEventMessageFlowFormatsMnemonic", "name": r["name"], "line": r["kmsgLine"], "contains": ["145.0", "NVLINK_RLW_ERROR", "PCI:0000:04:00"], "devices": {}})
    rows, src = table(HS, "Test_SubCodeDifferentiatesSameUnit")
    for r in rows:
        line_rows.append({"func": "Test_SubCodeDifferentiatesSameUnit", "name": r["name"], "line": r["kmsgLine"], "sub_code": r["subCodeValue"],
                          "contains": ["NVLINK_NETIR_ERROR", "149.%d" % r["subCodeValue"]], "devices": {}})
    rows, src = table(HS, "Test_InvestigatoryHintFiltering")
    for r in rows:
        line_rows.append({"func": "Test_InvestigatoryHintFiltering", "name": r["name"], "line": r["kmsgLine"], "hint": r["expectedVal"], "contains": [], "devices": {}})
    xm["from_lines"] = {"src": HS, "rows": line_rows}
    # evolveHealthyState integration: the events each case builds with createXidEvent / createNVLinkXidEvent (:20-39, :887-905)
    body, line = find_func(hs_src, "Test_HealthStateReason_evolveHealthyState_Integration")
    ev_rows = []
    for m in re.finditer(r'name:\s*"([^"]*)",\s*events:\s*eventstore\.Events\{(.*?)\},\s*expectedHealth:\s*apiv1\.HealthStateType(\w+),\s*expectedContains:\s*\[\]string\{(.*?)\}', body, re.S):
        evs = []
        for em in re.finditer(r'createNVLinkXidEvent\([^,]+(?:\([^)]*\))?, (\d+), (\d+), (0x[0-9a-fA-F]+|\d+), apiv1\.EventType(\w+), apiv1\.RepairActionType(\w+)\)|createXidEvent\((?:[^,()]|\([^)]*\))+, (\d+), apiv1\.EventType(\w+), apiv1\.RepairActionType(\w+)\)|\{Name: "reboot"', m.group(2)):
            if em.group(1):
                evs.append({"name": "error_xid", "type": em.group(4), "xid": int(em.group(1)), "sub_code": int(em.group(2)), "error_status": int(em.group(3), 0),
                            "device_uuid": "PCI:0000:04:00", "description": "NVLINK Error for XID %s" % em.group(1), "action": em.group(5)})
            elif em.group(6):
                evs.append({"name": "error_xid", "type": em.group(7), "xid": int(em.group(6)), "sub_code": 0, "error_status": 0, "device_uuid": "PCI:0000:9b:00",
                            "description": "", "action": em.group(8)})
            else:
                evs.append({"name": "reboot"})
        ev_rows.append({"name": m.group(1), "events": evs, "health": m.group(3), "contains": [go_str(x) for x in re.findall(r'"((?:[^"\\]|\\.)*)"', m.group(4))]})
    xm["evolve"] = {"src": "%s:%d" % (HS, line), "rows": ev_rows, "devices": {"GPU-test-uuid": "0000:04:00.0"}}
    dump("xid_messages.json", xm)

    # ---- NVML error classes (pkg/nvidia/errors/error_test.go): constant tables + the mocked error-string tables ----
    ET = "pkg/nvidia/errors/error_test.go"
    et_src = open(os.path.join(REF, ET)).read()
    NVML_RET = {"SUCCESS": 0, "ERROR_UNINITIALIZED": 1, "ERROR_INVALID_ARGUMENT": 2, "ERROR_NOT_SUPPORTED": 3, "ERROR_NO_PERMISSION": 4, "ERROR_ALREADY_INITIALIZED": 5,
                "ERROR_NOT_FOUND": 6, "ERROR_INSUFFICIENT_SIZE": 7, "ERROR_INSUFFICIENT_POWER": 8, "ERROR_DRIVER_NOT_LOADED": 9, "ERROR_TIMEOUT": 10,
                "ERROR_IRQ_ISSUE": 11, "ERROR_LIBRARY_NOT_FOUND": 12, "ERROR_FUNCTION_NOT_FOUND": 13, "ERROR_CORRUPTED_INFOROM": 14, "ERROR_GPU_IS_LOST": 15,
                "ERROR_RESET_REQUIRED": 16, "ERROR_OPERATING_SYSTEM": 17, "ERROR_LIB_RM_VERSION_MISMATCH": 18, "ERROR_IN_USE": 19, "ERROR_MEMORY": 20,
                "ERROR_NO_DATA": 21, "ERROR_VGPU_ECC_NOT_SUPPORTED": 22, "ERROR_INSUFFICIENT_RESOURCES": 23, "ERROR_FREQ_NOT_SUPPORTED": 24,
                "ERROR_ARGUMENT_VERSION_MISMATCH": 25, "ERROR_DEPRECATED": 26, "ERROR_NOT_READY": 27, "ERROR_GPU_NOT_FOUND": 28, "ERROR_INVALID_STATE": 29,
                "ERROR_UNKNOWN": 999}                     # nvml.h nvmlReturn_t (go-nvml v0.13.0-1 mirrors it)
    ec = {}
    for fn, key in (("TestIsNotSupportError", "not_supported"), ("TestIsGPULostError", "gpu_lost"), ("TestIsGPURequiresReset", "reset_required")):
        body, line = find_func(et_src, fn)
        mock = {int(c): bytes(v, "utf-8").decode("unicode_escape") for c, v in re.findall(r'case nvml\.Return\((\d+)\):\s*return "((?:[^"\\]|\\.)*)"', body)}
        rows = []
        for nm, ret, exp in re.findall(r'name:\s*"((?:[^"\\]|\\.)*)",\s*ret:\s*nvml\.(\w+(?:\(\d+\))?),\s*expected:\s*(true|false)', body):
            m = re.fullmatch(r"Return\((\d+)\)", ret)
            code = int(m.group(1)) if m else NVML_RET[ret]
            rows.append({"name": nm, "ret": code, "error_string": mock.get(code), "expected": exp == "true"})
        ec[key] = {"src": "%s:%d" % (ET, line), "rows": rows}
    dump("nvml_error_classes.json", ec)

    # ---- GPU product capability tables (pkg/nvidia/product/capabilities_test.go) ----
    PC = "pkg/nvidia/product/capabilities_test.go"
    pc = {}
    rows, src = table(PC, "TestSupportedMemoryMgmtCapsByGPUProduct")
    pc["mem_caps"] = {"src": src, "rows": [{"name": r["name"], "product": r["gpuProductName"],
                                            "caps": (1 if isinstance(r["expected"], dict) and r["expected"].get("ErrorContainment") else 0)
                                                    | (2 if isinstance(r["expected"], dict) and r["expected"].get("DynamicPageOfflining") else 0)
                                                    | (4 if isinstance(r["expected"], dict) and r["expected"].get("RowRemapping") else 0)} for r in rows]}
    rows, src = table(PC, "TestSupportedFMByGPUProduct")
    pc["fm_supported"] = {"src": src, "rows": [{"name": r["name"], "product": r["gpuProductName"], "expected": r["expected"]} for r in rows]}
    rows, src = table(PC, "TestSupportFabricStateByGPUProduct")
    pc["fabric_state_supported"] = {"src": src, "rows": [{"name": r["name"], "product": r["gpuProductName"], "expected": r["expected"]} for r in rows]}
    dump("product_caps.json", pc)

    # ---- eventstore compareEvent / unmarshalIfValid tables + infiniband's kmsg dedup-window policy ----
    es = {}
    rows, src = table("pkg/eventstore/database_test.go", "TestCompareEvent")
    mp = lambda v: v if isinstance(v, dict) else {}                # `map[string]string{}` parses as an empty composite
    es["compare_event"] = {"src": src, "rows": [{"name": r["name"], "a": mp(r["eventA"].get("ExtraInfo", {})), "b": mp(r["eventB"].get("ExtraInfo", {})), "expected": r["expected"]} for r in rows]}
    rows, src = table("pkg/eventstore/database_test.go", "TestUnmarshalIfValid")
    es["unmarshal_if_valid"] = {"src": src, "rows": [{"name": r["name"], "valid": r["data"].get("Valid", False), "string": r["data"].get("String", ""),
                                                      "expected_error": r["expectedError"]} for r in rows]}
    IBC = N + "infiniband/component_test.go"
    ib_src = open(os.path.join(REF, IBC)).read()
    cs = consts(N + "infiniband/kmsg_matcher.go")
    durs = {}
    for m in re.finditer(r"^\s*(default\w+DedupWindow)\s*=\s*(\d+)\s*\*\s*time\.(Minute|Hour)\s*$", open(os.path.join(REF, N + "infiniband/component.go")).read(), re.M):
        durs[m.group(1)] = int(m.group(2)) * {"Minute": 60, "Hour": 3600}[m.group(3)]
    dw = []
    for fm in re.finditer(r"^func (TestComponentKmsgEventDedupWindow_\w+)\(", ib_src, re.M):
        body, line = find_func(ib_src, fm.group(1))
        def expr(e):
            val = ""
            for tok in re.findall(r'"(?:[^"\\]|\\.)*"|\w+', e):
                val += bytes(tok[1:-1], "utf-8").decode("unicode_escape") if tok.startswith('"') else cs[tok]["value"]
            return val
        name = expr(re.search(r"Name:\s*(.+?),\s*\n", body).group(1))
        msg = expr(re.search(r"Message:\s*(.+?),\s*\n", body).group(1))
        if "assert.False(t, ok)" in body:
            ok, win = False, 0
        else:
            ok, win = True, durs[re.search(r"assert\.Equal\(t, (default\w+), dedupWindow\)", body).group(1)]
        dw.append({"name": fm.group(1), "event": name, "message": msg, "ok": ok, "window_seconds": win, "line": line})
    es["infiniband_dedup_window"] = {"src": IBC, "rows": dw, "constants": durs}
    dump("eventstore_cases.json", es)

    # ---- fabric GetIssues / getHealthMaskIssues tables (pkg/nvidia/nvml/device/fabric_state_test.go) ----
    # the nvml.* constants are go-nvml's (v0.13.0-1, go.mod:6), i.e. nvml.h's published values
    NV = {"GPU_FABRIC_STATE_NOT_SUPPORTED": 0, "GPU_FABRIC_STATE_NOT_STARTED": 1, "GPU_FABRIC_STATE_IN_PROGRESS": 2, "GPU_FABRIC_STATE_COMPLETED": 3,
          "GPU_FABRIC_HEALTH_SUMMARY_NOT_SUPPORTED": 0, "GPU_FABRIC_HEALTH_SUMMARY_HEALTHY": 1, "GPU_FABRIC_HEALTH_SUMMARY_UNHEALTHY": 2,
          "GPU_FABRIC_HEALTH_SUMMARY_LIMITED_CAPACITY": 3, "SUCCESS": 0, "ERROR_UNKNOWN": 999,
          "GPU_FABRIC_HEALTH_MASK_SHIFT_DEGRADED_BW": 0, "GPU_FABRIC_HEALTH_MASK_SHIFT_ROUTE_RECOVERY": 2,
          "GPU_FABRIC_HEALTH_MASK_SHIFT_ROUTE_UNHEALTHY": 4, "GPU_FABRIC_HEALTH_MASK_SHIFT_ACCESS_TIMEOUT_RECOVERY": 6}
    for f in ("DEGRADED_BW", "ROUTE_RECOVERY", "ROUTE_UNHEALTHY", "ACCESS_TIMEOUT_RECOVERY"):
        NV.update({"GPU_FABRIC_HEALTH_MASK_%s_NOT_SUPPORTED" % f: 0, "GPU_FABRIC_HEALTH_MASK_%s_TRUE" % f: 1, "GPU_FABRIC_HEALTH_MASK_%s_FALSE" % f: 2})

    def nv_eval(expr):
        e = re.sub(r"nvml\.(\w+)", lambda m: str(NV[m.group(1)]), expr)
        e = re.sub(r"uint32\(([^()]*)\)", r"(\1)", e)
        assert re.fullmatch(r"[\d\s()<|]+", e), expr
        return int(eval(" ".join(e.split())))

    FT = "pkg/nvidia/nvml/device/fabric_state_test.go"
    src_txt = open(os.path.join(REF, FT)).read()
    fab = {}
    body, line = find_func(src_txt, "TestFabricState_GetIssues")
    rows = []
    for m in re.finditer(r'name:\s*"([^"]+)",\s*state:\s*FabricState\{(.*?)\n\t\t\t\},\s*expected:\s*\[\]string\{(.*?)\},\n\t\t\}', body, re.S):
        fields = {k: nv_eval(v) for k, v in re.findall(r"(State|Status|HealthMask|HealthSummary):\s*((?:[^,\n]|\n\t\t\t\t\t)+),", m.group(2))}
        rows.append({"name": m.group(1), "state": fields["State"], "status": fields["Status"], "health_mask": fields["HealthMask"],
                     "summary": fields["HealthSummary"], "expected": re.findall(r'"([^"]*)"', m.group(3))})
    fab["get_issues"] = {"src": "%s:%d" % (FT, line), "rows": rows}
    body, line = find_func(src_txt, "TestGetHealthMaskIssues")
    rows = []
    for m in re.finditer(r'name:\s*"([^"]+)",\s*mask:\s*(.*?),\n\s*expected:\s*\[\]string\{(.*?)\},', body, re.S):
        rows.append({"name": m.group(1), "mask": nv_eval(m.group(2)), "expected": re.findall(r'"([^"]*)"', m.group(3))})
    fab["health_mask_issues"] = {"src": "%s:%d" % (FT, line), "rows": rows}
    fab["constants"] = {"src": "go-nvml v0.13.0-1 (go.mod:6) = nvml.h", "rows": [], "nvml": NV}
    dump("fabric_issues.json", fab)

    # ---- nvlink threshold evaluation: every TestEvaluateThresholds_* function as one vector (nvlink/evaluate_threshold_test.go) ----
    NT = N + "nvlink/evaluate_threshold_test.go"
    ntxt = open(os.path.join(REF, NT)).read()
    P2P_CONST = {"p2pStatusOK": 0, "p2pStatusChipsetNotSupported": 1, "p2pStatusGPUNotSupported": 2, "p2pStatusTopologyNotSupported": 3,
                 "p2pStatusDisabledByRegkey": 4, "p2pStatusNotSupported": 5, "p2pStatusUnknown": 6}   # nvlink/p2p.go:12-18,33-49

    def brace_block(text, start):
        d, i = 0, start
        while True:
            if text[i] == "{":
                d += 1
            elif text[i] == "}":
                d -= 1
                if d == 0:
                    return text[start:i + 1]
            i += 1

    nv_rows = []
    for fm in re.finditer(r"func (TestEvaluateThresholds_\w+)\(t \*testing\.T\) \{", ntxt):
        name = fm.group(1)
        body, line = find_func(ntxt, name)
        r = {"name": name, "line": line}
        m = re.search(r"AtLeastGPUsWithAllLinksFeatureEnabled:\s*(-?\d+)", body)
        r["at_least"] = int(m.group(1)) if m else 0
        gpus = []
        m = re.search(r"NVLinks:\s*\[\]NVLink\{", body)
        if m:
            blk = brace_block(body, m.end() - 1)
            i = 1
            while True:
                j = blk.find("{", i)
                if j < 0:
                    break
                ent = brace_block(blk, j)
                i = j + len(ent)
                u = re.search(r'UUID:\s*"([^"]+)"', ent)
                sup = re.search(r"Supported:\s*(true|false)", ent)
                gpus.append({"uuid": u.group(1), "supported": bool(sup and sup.group(1) == "true"),
                             "states": [x == "true" for x in re.findall(r"FeatureEnabled:\s*(true|false)", ent)]})
        r["nvlinks"] = gpus
        for key, field in (("active", "ActiveNVLinkUUIDs"), ("inactive", "InactiveNVLinkUUIDs"), ("unsupported", "UnsupportedNVLinkUUIDs"), ("p2p_ok_gpus", "PeerNVLinkOKGPUUUIDs")):
            m = re.search(field + r":\s*\[\]string\{([^}]*)\}", body)
            r[key] = re.findall(r'"([^"]+)"', m.group(1)) if m else []
        for key, field in (("p2p_probed", "PeerNVLinkProbePairCount"), ("p2p_expected", "PeerNVLinkExpectedPairCount"), ("p2p_ok", "PeerNVLinkOKPairCount")):
            m = re.search(field + r":\s*(\d+)", body)
            r[key] = int(m.group(1)) if m else 0
        m = re.search(r"PeerNVLinkObservedStatusCodes:\s*\[\]string\{([^}]*)\}", body)
        r["p2p_observed"] = [P2P_CONST[c] for c in re.findall(r"\w+", m.group(1))] if m else []
        r["system_expected"] = bool(re.search(r"SystemExpectedNVLink:\s*true", body))
        m = re.search(r"\n\t\thealth:\s*apiv1\.HealthStateType(\w+)", body)
        r["preset_health"] = m.group(1) if m else ""
        m = re.search(r'\n\t\treason:\s*"([^"]*)"', body)
        r["preset_reason"] = m.group(1) if m else ""
        m = re.search(r"assert\.Equal\(t,\s*apiv1\.HealthStateType(\w+),\s*cr\.health\)", body)
        r["want_health"] = m.group(1) if m else ""
        r["want_reason_contains"] = re.findall(r'assert\.Contains\(t,\s*cr\.reason,\s*"([^"]*)"\)', body)
        m = re.search(r'assert\.Equal\(t,\s*("[^"]*"|\w+),\s*cr\.reason\)', body)
        r["want_reason_equal"] = m.group(1).strip('"') if m else ""
        r["want_reboot"] = True if "RepairActionTypeRebootSystem" in body else (False if re.search(r"assert\.Nil\(t,\s*cr\.suggestedActions\)", body) else None)
        nv_rows.append(r)
    # ---- xid / sxid evolveHealthyState scenarios (health_state_test.go: TestStateUpdateBasedOnEvents), events newest first ----
    def health_scenarios(path, ctor):
        body, line = find_func(open(os.path.join(REF, path)).read(), "TestStateUpdateBasedOnEvents")
        out = []
        for blk in re.split(r'\n\tt\.Run\("', body)[1:]:
            name = blk.split('"', 1)[0]
            if "trimEventsAfterSetHealthy" in blk or "invalid json" in blk or "ExtraInfo:" in blk:
                continue                                   # scenarios about merge/trim plumbing or undecodable payloads
            m = re.search(r"eventstore\.Events\{(.*?)\n\t\t\}", blk, re.S)
            evs = []
            if m:
                for em in re.finditer(ctor + r"\([^,]+,\s*(\d+),\s*apiv1\.EventType(\w+),\s*apiv1\.RepairActionType(\w+)\)|" + ctor +
                                      r"WithNilSuggestedActions\([^,]+,\s*(\d+),\s*apiv1\.EventType(\w+)\)|\{Name:\s*\"reboot\"[^}]*\}", m.group(1)):
                    if em.group(1) is not None:
                        evs.append({"k": "err", "code": int(em.group(1)), "type": em.group(2), "actions": [em.group(3)]})
                    elif em.group(4) is not None:
                        evs.append({"k": "err", "code": int(em.group(4)), "type": em.group(5), "actions": None})
                    else:
                        evs.append({"k": "reboot"})
            r = {"name": name, "events": evs}
            hm = re.search(r"assert\.Equal\(t,\s*apiv1\.HealthStateType(\w+),\s*state\.Health[,)]", blk)
            if hm:
                r["health"] = hm.group(1)
            rm = re.search(r'assert\.Equal\(t,\s*"([^"]*)",\s*state\.Reason\)', blk)
            if rm:
                r["reason"] = rm.group(1)
            am = re.search(r"assert\.Equal\(t,\s*apiv1\.RepairActionType(\w+),\s*state\.SuggestedActions\.RepairActions\[0\]\)", blk)
            if am:
                r["action"] = am.group(1)
            if re.search(r"assert\.Nil\(t,\s*state\.SuggestedActions\)", blk):
                r["action"] = None
            out.append(r)
        return out, "%s:%d" % (path, line)

    rows, src = health_scenarios(N + "sxid/health_state_test.go", "createSXidEvent")
    dump("sxid_health.json", {"scenarios": {"src": src, "rows": rows, "note": "rebootThreshold = 2 (sxid/health_state.go:36)"}})
    rows, src = health_scenarios(N + "xid/health_state_test.go", "createXidEvent")
    dump("xid_health_extracted.json", {"scenarios": {"src": src, "rows": rows, "note": "DefaultRebootThreshold = 2; script-extracted twin of xid_health.json"}})

    # ---- temperature thresholds: every TestCheck_* that builds a Temperature literal and asserts a health (temperature/component_test.go) ----
    TT = N + "temperature/component_test.go"
    ttxt = open(os.path.join(REF, TT)).read()
    trows = []
    for fm in re.finditer(r"func (TestCheck_\w+)\(t \*testing\.T\) \{", ttxt):
        body, line = find_func(ttxt, fm.group(1))
        lit = re.search(r"temperature := Temperature\{(.*?)\n\t*\}", body, re.S)
        if not lit:
            continue
        fields = {}
        for k, v in re.findall(r"(\w+):\s*([^,\n]+),", lit.group(1)):
            v = v.strip()
            fields[k] = v == "true" if v in ("true", "false") else (int(v) if re.fullmatch(r"-?\d+", v) else v)
        mthr = re.search(r"SetDefaultMarginThreshold\(Thresholds\{CelsiusSlowdownMargin:\s*(\d+)\}\)", body)
        cases = []
        tbl = re.findall(r'name:\s*"([^"]*)",\s*marginCelsius:\s*(-?\d+),\s*expectHealthy:\s*apiv1\.HealthStateType(\w+),\s*expectReasonContains:\s*"([^"]*)"', body)
        tbl2 = re.findall(r'name:\s*"([^"]*)",\s*hbmTemp:\s*(\d+),\s*memMaxThreshold:\s*(\d+),\s*expectHealthy:\s*apiv1\.HealthStateType(\w+),\s*expectReasonContains:\s*"([^"]*)"', body)
        if tbl:
            for nm, mc, hl, rs in tbl:
                f2 = dict(fields)
                f2["ThresholdCelsiusSlowdownMargin"] = int(mc)
                cases.append((fm.group(1) + "/" + nm, f2, hl, [rs]))
        elif tbl2:
            for nm, ht, mm, hl, rs in tbl2:
                f2 = dict(fields)
                f2["CurrentCelsiusHBM"], f2["ThresholdCelsiusMemMax"] = int(ht), int(mm)
                cases.append((fm.group(1) + "/" + nm, f2, hl, [rs]))
        else:
            hm = re.search(r"assert\.Equal\(t,\s*apiv1\.HealthStateType(\w+),\s*data\.health", body)
            if not hm:
                continue
            cases.append((fm.group(1), fields, hm.group(1), re.findall(r'assert\.Contains\(t,\s*data\.reason,\s*"([^"]*)"\)', body)))
        for nm, f, hl, rs in cases:
            trows.append({"name": nm, "line": line, "margin_threshold": int(mthr.group(1)) if mthr else None, "health": hl, "reason_contains": rs,
                          "temperature": {k: v for k, v in f.items() if isinstance(v, (int, bool))}})
    dthr = re.search(r"CelsiusSlowdownMargin:\s*(\d+)", open(os.path.join(REF, N + "temperature/threshold.go")).read()) if os.path.exists(os.path.join(REF, N + "temperature/threshold.go")) else None
    dump("temperature_checks.json", {"checks": {"src": TT, "rows": trows, "default_margin_threshold": int(dthr.group(1)) if dthr else None}})

    # ---- hw-slowdown: clock-event reason bitmask -> descriptions (hw-slowdown/clock_events.go:168-264, clock_events_test.go:21) ----
    HS = N + "hw-slowdown/"
    ctxt = open(os.path.join(REF, HS + "clock_events.go")).read()
    flags = {m.group(1): int(m.group(2), 16) for m in re.finditer(r"(reason\w+)\s+uint64\s*=\s*(0x[0-9a-fA-F]+)", ctxt)}
    ce_table = []
    for m in re.finditer(r"(reason\w+):\s*\{\s*description:\s*\"((?:[^\"\\]|\\.)*)\",\s*isHWSlowdown:\s*(true|false),", ctxt):
        ce_table.append({"flag": flags[m.group(1)], "name": m.group(1), "description": m.group(2), "hw_slowdown": m.group(3) == "true"})
    body, line = find_func(open(os.path.join(REF, HS + "clock_events_test.go")).read(), "TestGetClockEventReasons")
    crow = []
    for m in re.finditer(r'name:\s*"([^"]+)",\s*reasons:\s*([^,]+),\s*wantHWSlowdown:\s*\[\]string\{(.*?)\},\s*wantOtherReasons:\s*\[\]string\{(.*?)\},\n\t\t\}', body, re.S):
        ex = m.group(2).strip()
        val = 0
        for tok in ex.split("|"):
            tok = tok.strip()
            val |= int(tok, 16) if tok.startswith("0x") else flags[tok]
        crow.append({"name": m.group(1), "reasons": val, "want_hw": re.findall(r'"((?:[^"\\]|\\.)*)"', m.group(3)), "want_other": re.findall(r'"((?:[^"\\]|\\.)*)"', m.group(4))})
    dump("clock_events.json", {"reasons": {"src": HS + "clock_events_test.go:%d" % line, "rows": crow},
                               "table": {"src": HS + "clock_events.go:192-264", "rows": [], "entries": ce_table}})

    dump("nvlink_thresholds.json", {"evaluate": {"src": NT + ":12-490", "rows": nv_rows,
                                                  "note": "one row per TestEvaluateThresholds_* function: the checkResult it builds and what it asserts"}})
    return 0


if __name__ == "__main__":
    sys.exit(main())
