// store_sqlite.cpp — the write path into the reference's SQLite event store and metrics store (SURVEY.md 8f.2), so that
// the /v1/events and /v1/metrics readers of gpud find what this library produced without any change on their side.
//   events   pkg/eventstore/database.go:18-31 (schema version, columns), :136-143 (table name), :198-246 (createTable),
//            :248-275 (insertEvent: NULLIF(?, '') for message / extra_info), :277-324 (findEvent duplicate check)
//   metrics  pkg/metrics/store/sqlite.go:22-36 (schema version, columns, default table), :87-106 (CreateTable),
//            :108-164 (insert: INSERT OR REPLACE, labels as JSON or ''), :258-275 (purge)
//   window rows  what the Syncer (pkg/metrics/syncer/syncer.go:76-82) records on its ticker, from the ring's streaming drain
//   xid events as persisted by xid/component.go:503-554 (name "error_xid", extra_info {"data", "device_uuid"})
// SQLite itself is dlopen'ed (libsqlite3.so.0; the image carries the library but no headers), WAL + busy timeout like
// pkg/sqlite (SURVEY.md §2: `_journal_mode=WAL&_busy_timeout=5000`).
#include <dlfcn.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <time.h>

#include <algorithm>
#include <map>
#include <string>
#include <vector>

#include "../../include/gpud_b200.h"
#include "json_min.h"
#include "ring_drain.h"

namespace {

struct Sq {
  void* so = nullptr;
  int (*open_v2)(const char*, void**, int, const char*) = nullptr;
  int (*close)(void*) = nullptr;
  int (*exec)(void*, const char*, int (*)(void*, int, char**, char**), void*, char**) = nullptr;
  int (*prepare_v2)(void*, const char*, int, void**, const char**) = nullptr;
  int (*bind_int64)(void*, int, long long) = nullptr;
  int (*bind_double)(void*, int, double) = nullptr;
  int (*bind_text)(void*, int, const char*, int, void (*)(void*)) = nullptr;
  int (*step)(void*) = nullptr;
  int (*reset)(void*) = nullptr;
  int (*finalize)(void*) = nullptr;
  const unsigned char* (*column_text)(void*, int) = nullptr;
  long long (*column_int64)(void*, int) = nullptr;
  int (*changes)(void*) = nullptr;
  const char* (*errmsg)(void*) = nullptr;
  int (*busy_timeout)(void*, int) = nullptr;
  void (*free)(void*) = nullptr;
};
constexpr int kOk = 0, kRow = 100, kDone = 101;
void (*const kTransient)(void*) = (void (*)(void*))(intptr_t)-1;

Sq* sq() {
  static Sq s;
  static bool tried = false;
  if (!tried) {
    tried = true;
    s.so = dlopen("libsqlite3.so.0", RTLD_NOW);
    if (s.so) {
#define SYM(f, name) *(void**)&s.f = dlsym(s.so, name)
      SYM(open_v2, "sqlite3_open_v2"); SYM(close, "sqlite3_close"); SYM(exec, "sqlite3_exec"); SYM(prepare_v2, "sqlite3_prepare_v2");
      SYM(bind_int64, "sqlite3_bind_int64"); SYM(bind_double, "sqlite3_bind_double"); SYM(bind_text, "sqlite3_bind_text"); SYM(step, "sqlite3_step");
      SYM(reset, "sqlite3_reset"); SYM(finalize, "sqlite3_finalize"); SYM(column_text, "sqlite3_column_text"); SYM(errmsg, "sqlite3_errmsg");
      SYM(busy_timeout, "sqlite3_busy_timeout"); SYM(free, "sqlite3_free"); SYM(column_int64, "sqlite3_column_int64"); SYM(changes, "sqlite3_changes");
#undef SYM
      if (!s.open_v2 || !s.close || !s.exec || !s.prepare_v2 || !s.bind_int64 || !s.bind_double || !s.bind_text || !s.step || !s.finalize ||
          !s.column_text || !s.errmsg || !s.column_int64 || !s.changes) { dlclose(s.so); s.so = nullptr; }
    }
  }
  return s.so ? &s : nullptr;
}

// Every statement the event side runs, in one place (the text is the reference's: pkg/eventstore/database.go:248-262 insert,
// :278-298 find, :327-336 get, :367-369 latest, :449-450 purge).  tests/test_store_cpu.py compares them with the strings extracted
// from the reference (tests/golden/store_sql.json).
enum { kSqlInsert = 0, kSqlFind = 1, kSqlFindWithMessage = 2, kSqlGet = 3, kSqlLatest = 4, kSqlPurge = 5 };
std::string event_sql(int which, const std::string& t) {
  switch (which) {
    case kSqlInsert: return "INSERT INTO " + t + " (timestamp, name, type, message, extra_info) VALUES (?, ?, ?, NULLIF(?, ''), NULLIF(?, ''))";
    case kSqlFind: return "\nSELECT timestamp, name, type, message, extra_info FROM " + t + " WHERE timestamp = ? AND name = ? AND type = ?";
    case kSqlFindWithMessage: return event_sql(kSqlFind, t) + " AND message = ?";
    case kSqlGet: return "SELECT timestamp, name, type, message, extra_info\nFROM " + t + "\nWHERE timestamp > ?\nORDER BY timestamp DESC";
    case kSqlLatest: return "SELECT timestamp, name, type, message, extra_info FROM " + t + " ORDER BY timestamp DESC LIMIT 1";
    case kSqlPurge: return "DELETE FROM " + t + " WHERE timestamp < ?";
  }
  return "";
}

// encoding/json string escaping (HTML-safe, like json.Marshal)
void jstr(std::string& o, const std::string& s) {
  o.push_back('"');
  for (unsigned char c : s) {
    if (c == '"') o += "\\\"";
    else if (c == '\\') o += "\\\\";
    else if (c == '\n') o += "\\n";
    else if (c == '\r') o += "\\r";
    else if (c == '\t') o += "\\t";
    else if (c < 0x20 || c == '<' || c == '>' || c == '&') { char b[8]; snprintf(b, sizeof b, "\\u%04x", c); o += b; }
    else o.push_back((char)c);
  }
  o.push_back('"');
}

bool ident_ok(const char* t) {          // table names are spliced into SQL (as the reference does with fmt.Sprintf): keep them identifiers
  if (!t || !*t) return false;
  for (const char* p = t; *p; ++p)
    if (!((*p >= 'a' && *p <= 'z') || (*p >= 'A' && *p <= 'Z') || (*p >= '0' && *p <= '9') || *p == '_')) return false;
  return true;
}

const char* event_type_string(int32_t ev) {   // api/v1/types.go:222-244
  switch (ev) {
    case GPUD_EVENT_INFO: return "Info";
    case GPUD_EVENT_WARNING: return "Warning";
    case GPUD_EVENT_CRITICAL: return "Critical";
    case GPUD_EVENT_FATAL: return "Fatal";
  }
  return "Unknown";
}

}  // namespace

struct gpud_store {
  void* db = nullptr;
  std::string err;
};

static int32_t sfail(gpud_store* st, const char* what) {
  Sq* S = sq();
  st->err = std::string(what) + ": " + (S && st->db ? S->errmsg(st->db) : "sqlite unavailable");
  return GPUD_E_STATE;
}

extern "C" int32_t gpud_store_open(const char* path, gpud_store** out) {
  if (!path || !out) return GPUD_E_INVALID;
  Sq* S = sq();
  if (!S) return GPUD_E_UNSUPPORTED;
  gpud_store* st = new gpud_store();
  if (S->open_v2(path, &st->db, 0x2 | 0x4 /* READWRITE | CREATE */, nullptr) != kOk) { if (st->db) S->close(st->db); delete st; return GPUD_E_STATE; }
  if (S->busy_timeout) S->busy_timeout(st->db, 5000);
  S->exec(st->db, "PRAGMA journal_mode=WAL;", nullptr, nullptr, nullptr);
  *out = st;
  return GPUD_OK;
}
extern "C" void gpud_store_close(gpud_store* st) {
  if (!st) return;
  if (Sq* S = sq()) if (st->db) S->close(st->db);
  delete st;
}
extern "C" int32_t gpud_store_last_error(gpud_store* st, char* out, int32_t cap) {
  if (!st || !out || cap <= 0) return GPUD_E_INVALID;
  snprintf(out, (size_t)cap, "%s", st->err.c_str());
  return GPUD_OK;
}

// defaultTableName (database.go:136-143) + createTable (database.go:198-246)
extern "C" int32_t gpud_store_event_table(gpud_store* st, const char* component, char* table_out, int32_t cap) {
  if (!st || !component || !table_out || cap <= 0) return GPUD_E_INVALID;
  Sq* S = sq();
  std::string c;
  // strings.ReplaceAll is one non-overlapping left-to-right pass each: ' ' -> '_', '-' -> '_', "__" -> "_", then ToLower
  {
    std::string src = component, a;
    for (char ch : src) a.push_back((ch == ' ' || ch == '-') ? '_' : ch);
    std::string b;
    for (size_t i = 0; i < a.size();) { if (i + 1 < a.size() && a[i] == '_' && a[i + 1] == '_') { b.push_back('_'); i += 2; } else b.push_back(a[i++]); }
    for (auto& ch : b) if (ch >= 'A' && ch <= 'Z') ch = (char)(ch - 'A' + 'a');
    c = b;
  }
  const std::string t = "components_" + c + "_events_v0_5_0";
  if (!ident_ok(t.c_str()) || (int32_t)t.size() + 1 > cap) return GPUD_E_INVALID;
  const std::string ddl = "\nCREATE TABLE IF NOT EXISTS " + t + " (\n\ttimestamp INTEGER NOT NULL,\n\tname TEXT NOT NULL,\n\ttype TEXT NOT NULL,\n\tmessage TEXT,\n\textra_info TEXT\n);";
  std::string sql = "BEGIN;" + ddl;
  for (const char* col : {"timestamp", "name", "type"})
    sql += "CREATE INDEX IF NOT EXISTS idx_" + t + "_" + col + " ON " + t + "(" + col + ");";
  sql += "COMMIT;";
  if (S->exec(st->db, sql.c_str(), nullptr, nullptr, nullptr) != kOk) { S->exec(st->db, "ROLLBACK;", nullptr, nullptr, nullptr); return sfail(st, "create event table"); }
  memcpy(table_out, t.c_str(), t.size() + 1);
  return GPUD_OK;
}

// ExtraInfo as the reference reads it back (database.go:428-447 scanRows + :471-482 unmarshalIfValid into map[string]string):
// NULL, "" and "null" are no map at all; anything else must be one JSON object of string values (a null value leaves "").
// Returns false where json.Unmarshal would fail -- the reference's findEvent then returns that error.
static bool parse_extra_info(const char* text, std::map<std::string, std::string>* m) {
  m->clear();
  if (!text || !*text || !strcmp(text, "null")) return true;
  if (text[0] != '{') return false;
  const char* p = text + 1;
  jsonmin::ws(p);
  if (*p == '}') { ++p; jsonmin::ws(p); return *p == 0; }
  for (;;) {
    std::string k, v;
    jsonmin::ws(p);
    if (!jsonmin::string(p, &k)) return false;
    jsonmin::ws(p);
    if (*p++ != ':') return false;
    jsonmin::ws(p);
    if (!strncmp(p, "null", 4)) p += 4;
    else if (!jsonmin::string(p, &v)) return false;
    (*m)[k] = v;
    jsonmin::ws(p);
    if (*p == ',') { ++p; continue; }
    if (*p == '}') { ++p; break; }
    return false;
  }
  jsonmin::ws(p);
  return *p == 0;
}

// findEvent (database.go:277-324): rows of the same (timestamp, name, type[, message]) whose ExtraInfo MAP equals the event's
// (compareEvent :459-469 -- same size, same key/value pairs; the JSON text may differ in key order or spacing).
static int32_t find_event(gpud_store* st, const std::string& t, int64_t unix_s, const char* name, const char* type, const char* message,
                          const char* extra_json, bool* found) {
  Sq* S = sq();
  *found = false;
  std::map<std::string, std::string> want, have;
  if (!parse_extra_info(extra_json, &want)) return sfail(st, "extra_info is not a JSON object of strings");
  void* q = nullptr;
  const std::string sel = event_sql(message && *message ? kSqlFindWithMessage : kSqlFind, t);
  if (S->prepare_v2(st->db, sel.c_str(), -1, &q, nullptr) != kOk) return sfail(st, "prepare find");
  S->bind_int64(q, 1, unix_s); S->bind_text(q, 2, name, -1, kTransient); S->bind_text(q, 3, type, -1, kTransient);
  if (message && *message) S->bind_text(q, 4, message, -1, kTransient);
  int32_t rc = GPUD_OK;
  while (S->step(q) == kRow) {
    if (!parse_extra_info((const char*)S->column_text(q, 4), &have)) { rc = sfail(st, "stored extra_info is not a JSON object of strings"); break; }
    if (have == want) { *found = true; break; }
  }
  S->finalize(q);
  return rc;
}

static int32_t insert_event(gpud_store* st, const char* table, int64_t unix_s, const char* name, const char* type, const char* message,
                            const char* extra_json, bool skip_duplicate, bool* inserted) {
  Sq* S = sq();
  if (inserted) *inserted = false;
  const std::string t = table;
  if (skip_duplicate) {
    bool dup = false;
    const int32_t rc = find_event(st, t, unix_s, name, type, message, extra_json, &dup);
    if (rc) return rc;
    if (dup) return GPUD_OK;
  }
  void* q = nullptr;
  const std::string ins = event_sql(kSqlInsert, t);
  if (S->prepare_v2(st->db, ins.c_str(), -1, &q, nullptr) != kOk) return sfail(st, "prepare insert");
  S->bind_int64(q, 1, unix_s); S->bind_text(q, 2, name, -1, kTransient); S->bind_text(q, 3, type, -1, kTransient);
  S->bind_text(q, 4, message ? message : "", -1, kTransient); S->bind_text(q, 5, extra_json ? extra_json : "", -1, kTransient);
  const int rc = S->step(q);
  S->finalize(q);
  if (rc != kDone) return sfail(st, "insert event");
  if (inserted) *inserted = true;
  return GPUD_OK;
}

extern "C" int32_t gpud_store_insert_event(gpud_store* st, const char* table, int64_t unix_s, const char* name, const char* type, const char* message,
                                           const char* extra_info_json) {
  if (!st || !ident_ok(table) || !name || !type) return GPUD_E_INVALID;
  if (!sq()) return GPUD_E_UNSUPPORTED;
  return insert_event(st, table, unix_s, name, type, message, extra_info_json, false, nullptr);
}

// Bucket.Find (eventstore/types.go:44-47, database.go:277-324)
extern "C" int32_t gpud_store_find_event(gpud_store* st, const char* table, int64_t unix_s, const char* name, const char* type, const char* message,
                                         const char* extra_info_json, int32_t* found) {
  if (!st || !ident_ok(table) || !name || !type || !found) return GPUD_E_INVALID;
  if (!sq()) return GPUD_E_UNSUPPORTED;
  bool f = false;
  const int32_t rc = find_event(st, table, unix_s, name, type, message, extra_info_json, &f);
  *found = f ? 1 : 0;
  return rc;
}

// the Insert loop of xid/component.go:468-577 for one scan's hits: one "error_xid" event per Xid hit, time = boot + kmsg usec
// in RAW_KMSG mode else `fallback_unix`, extra_info = {"data": xidErrorEventDetail JSON, "device_uuid": device}; an event that
// is already in the table is skipped (component.go:555-563).
extern "C" int32_t gpud_store_insert_xid_hits(gpud_store* st, const char* table, const gpud_xid_hit* hits, int64_t n, int64_t fallback_unix,
                                              int64_t boot_unix, int32_t raw_kmsg, int32_t* n_inserted) {
  if (!st || !ident_ok(table) || n < 0 || (n && !hits)) return GPUD_E_INVALID;
  Sq* S = sq();
  if (!S) return GPUD_E_UNSUPPORTED;
  int32_t ins = 0;
  if (S->exec(st->db, "BEGIN;", nullptr, nullptr, nullptr) != kOk) return sfail(st, "begin");
  for (int64_t i = 0; i < n; ++i) {
    const gpud_xid_hit& h = hits[i];
    if (h.kind != GPUD_KIND_XID) continue;
    const int64_t t = raw_kmsg ? boot_unix + h.kmsg_usec / 1000000 : fallback_unix;
    char payload[4096];
    if (gpud_hit_detail_json(&h, t, payload, sizeof payload) != GPUD_OK) continue;
    std::string extra = "{\"data\":";                               // json.Marshal(map[string]string): keys sorted
    jstr(extra, payload);
    extra += ",\"device_uuid\":";
    jstr(extra, std::string(h.device, strnlen(h.device, sizeof h.device)));
    extra += "}";
    bool did = false;
    const int32_t rc = insert_event(st, table, t, "error_xid", event_type_string(h.event_type), "", extra.c_str(), true, &did);
    if (rc) { S->exec(st->db, "ROLLBACK;", nullptr, nullptr, nullptr); return rc; }
    ins += did ? 1 : 0;
  }
  if (S->exec(st->db, "COMMIT;", nullptr, nullptr, nullptr) != kOk) return sfail(st, "commit");
  if (n_inserted) *n_inserted = ins;
  return GPUD_OK;
}

// sxid/component.go:433-469: Event{Time, Name: "error_sxid", ExtraInfo: {"data": strconv.FormatInt(sxid), "device_uuid": device}} --
// no Type, no Message; Find, then Insert.
extern "C" int32_t gpud_store_insert_sxid_hits(gpud_store* st, const char* table, const gpud_xid_hit* hits, int64_t n, int64_t fallback_unix,
                                               int64_t boot_unix, int32_t raw_kmsg, int32_t* n_inserted) {
  if (!st || !ident_ok(table) || n < 0 || (n && !hits)) return GPUD_E_INVALID;
  Sq* S = sq();
  if (!S) return GPUD_E_UNSUPPORTED;
  int32_t ins = 0;
  if (S->exec(st->db, "BEGIN;", nullptr, nullptr, nullptr) != kOk) return sfail(st, "begin");
  for (int64_t i = 0; i < n; ++i) {
    const gpud_xid_hit& h = hits[i];
    if (h.kind != GPUD_KIND_SXID) continue;
    const int64_t t = raw_kmsg ? boot_unix + h.kmsg_usec / 1000000 : fallback_unix;
    std::string extra = "{\"data\":\"" + std::to_string(h.code) + "\",\"device_uuid\":";
    jstr(extra, std::string(h.device, strnlen(h.device, sizeof h.device)));
    extra += "}";
    bool did = false;
    const int32_t rc = insert_event(st, table, t, "error_sxid", "", "", extra.c_str(), true, &did);
    if (rc) { S->exec(st->db, "ROLLBACK;", nullptr, nullptr, nullptr); return rc; }
    ins += did ? 1 : 0;
  }
  if (S->exec(st->db, "COMMIT;", nullptr, nullptr, nullptr) != kOk) return sfail(st, "commit");
  if (n_inserted) *n_inserted = ins;
  return GPUD_OK;
}

// hw-slowdown Check's persist step (hw-slowdown/component.go:294-343): the HWSlowdownEvent of one clock-event reading, Find then Insert
extern "C" int32_t gpud_store_insert_hw_slowdown(gpud_store* st, const char* table, int64_t unix_s, uint64_t bitmask, const char* gpu_uuid, int32_t* inserted) {
  if (!st || !ident_ok(table) || !gpu_uuid) return GPUD_E_INVALID;
  if (!sq()) return GPUD_E_UNSUPPORTED;
  if (inserted) *inserted = 0;
  char msg[2048];
  const int32_t n = gpud_hw_slowdown_event_message(bitmask, gpu_uuid, msg, sizeof msg);
  if (n < 0) return GPUD_E_CAPACITY;
  if (n == 0) return GPUD_OK;                                      // no hardware slowdown reason in this reading: no event
  std::string extra = "{\"data_source\":\"nvml\",\"gpu_uuid\":";
  jstr(extra, gpu_uuid);
  extra += "}";
  bool did = false;
  const int32_t rc = insert_event(st, table, unix_s, "hw_slowdown", "Warning", msg, extra.c_str(), true, &did);
  if (rc == GPUD_OK && inserted) *inserted = did ? 1 : 0;
  return rc;
}

// ---- the read side of a Bucket: Get, Latest, Purge (eventstore/types.go:54-66; database.go:327-402, 449-457) ----
// one row into the caller's arrays: strings of the row go into the text arena, the row records their offsets
static int32_t emit_row(gpud_store* st, void* q, gpud_event_row* row, char* text, int32_t cap_text, int32_t* used) {
  Sq* S = sq();
  memset(row, 0, sizeof *row);
  row->unix_s = S->column_int64(q, 0);
  const char* name = (const char*)S->column_text(q, 1);
  const char* type = (const char*)S->column_text(q, 2);
  const char* msg = (const char*)S->column_text(q, 3);
  const char* extra = (const char*)S->column_text(q, 4);
  if (strlen(name ? name : "") >= sizeof row->name || strlen(type ? type : "") >= sizeof row->type) return sfail(st, "event name / type longer than the row holds");
  snprintf(row->name, sizeof row->name, "%s", name ? name : "");
  snprintf(row->type, sizeof row->type, "%s", type ? type : "");
  std::map<std::string, std::string> m;
  if (!parse_extra_info(extra, &m)) return sfail(st, "failed to unmarshal extra info");        // scanRows' error (database.go:441-443)
  const char* parts[2] = {msg ? msg : "", extra ? extra : ""};
  int32_t* off[2] = {&row->message_off, &row->extra_off};
  int32_t* len[2] = {&row->message_len, &row->extra_len};
  for (int k = 0; k < 2; ++k) {
    const int32_t n = (int32_t)strlen(parts[k]);
    if (*used + n + 1 > cap_text) return GPUD_E_CAPACITY;
    memcpy(text + *used, parts[k], (size_t)n + 1);
    *off[k] = *used; *len[k] = n;
    *used += n + 1;
  }
  return GPUD_OK;
}

extern "C" int32_t gpud_store_get_events(gpud_store* st, const char* table, int64_t since_unix, gpud_event_row* rows, int32_t cap_rows, char* text,
                                         int32_t cap_text, int32_t* n_rows) {
  if (!st || !ident_ok(table) || cap_rows < 0 || (cap_rows && !rows) || !text || cap_text <= 0 || !n_rows) return GPUD_E_INVALID;
  Sq* S = sq();
  if (!S) return GPUD_E_UNSUPPORTED;
  *n_rows = 0;
  const std::string sel = event_sql(kSqlGet, table);
  void* q = nullptr;
  if (S->prepare_v2(st->db, sel.c_str(), -1, &q, nullptr) != kOk) return sfail(st, "prepare get");
  S->bind_int64(q, 1, since_unix);
  int32_t rc = GPUD_OK, used = 0, n = 0;
  while (S->step(q) == kRow) {
    if (n >= cap_rows) { rc = GPUD_E_CAPACITY; break; }
    rc = emit_row(st, q, &rows[n], text, cap_text, &used);
    if (rc) break;
    ++n;
  }
  S->finalize(q);
  *n_rows = n;
  return rc;
}

extern "C" int32_t gpud_store_latest_event(gpud_store* st, const char* table, gpud_event_row* row, char* text, int32_t cap_text, int32_t* found) {
  if (!st || !ident_ok(table) || !row || !text || cap_text <= 0 || !found) return GPUD_E_INVALID;
  Sq* S = sq();
  if (!S) return GPUD_E_UNSUPPORTED;
  *found = 0;
  const std::string sel = event_sql(kSqlLatest, table);
  void* q = nullptr;
  if (S->prepare_v2(st->db, sel.c_str(), -1, &q, nullptr) != kOk) return sfail(st, "prepare latest");
  int32_t rc = GPUD_OK, used = 0;
  if (S->step(q) == kRow) {
    rc = emit_row(st, q, row, text, cap_text, &used);
    if (rc == GPUD_OK) *found = 1;
  }
  S->finalize(q);
  return rc;
}

extern "C" int32_t gpud_store_purge_events(gpud_store* st, const char* table, int64_t before_unix, int32_t* n_purged) {
  if (!st || !ident_ok(table)) return GPUD_E_INVALID;
  Sq* S = sq();
  if (!S) return GPUD_E_UNSUPPORTED;
  const std::string del = event_sql(kSqlPurge, table);
  void* q = nullptr;
  if (S->prepare_v2(st->db, del.c_str(), -1, &q, nullptr) != kOk) return sfail(st, "prepare purge");
  S->bind_int64(q, 1, before_unix);
  const int rc = S->step(q);
  S->finalize(q);
  if (rc != kDone) return sfail(st, "purge events");
  if (n_purged) *n_purged = S->changes(st->db);
  return GPUD_OK;
}

// RebootEventStore.RecordReboot (pkg/host/event.go:40-42, 85-132) into the os bucket: nothing when the boot is older than the
// retention (3 days), when the same event is stored, when a later boot is already stored, or when the previous one is less than a
// minute older; else Event{boot time, "reboot", "Warning", "system reboot detected <boot time as Go prints a UTC time.Time>"}.
extern "C" int32_t gpud_store_record_reboot(gpud_store* st, const char* os_table, int64_t now_unix, int64_t boot_unix, int32_t* inserted) {
  if (!st || !ident_ok(os_table)) return GPUD_E_INVALID;
  if (!sq()) return GPUD_E_UNSUPPORTED;
  if (inserted) *inserted = 0;
  if (now_unix - boot_unix >= 3 * 24 * 3600) return GPUD_OK;                 // eventstore.DefaultRetention (types.go:48)
  time_t t = (time_t)boot_unix;
  struct tm tmv;
  gmtime_r(&t, &tmv);
  char when[64];
  strftime(when, sizeof when, "%Y-%m-%d %H:%M:%S +0000 UTC", &tmv);          // fmt %v of time.Unix(sec, 0).UTC()
  const std::string msg = std::string("system reboot detected ") + when;
  bool found = false;
  int32_t rc = find_event(st, os_table, boot_unix, "reboot", "Warning", msg.c_str(), "", &found);
  if (rc || found) return rc;
  gpud_event_row prev;
  char text[4096];
  int32_t have = 0;
  rc = gpud_store_latest_event(st, os_table, &prev, text, sizeof text, &have);      // the latest event of the bucket, whatever its name (:116-119)
  if (rc) return rc;
  if (have) {
    if (prev.unix_s != 0 && prev.unix_s > boot_unix) return GPUD_OK;         // !prev.Time.IsZero() && prev.Time.After(current)
    const int64_t elapsed = boot_unix - prev.unix_s;
    if (elapsed > 0 && elapsed < 60) return GPUD_OK;
  }
  bool did = false;
  rc = insert_event(st, os_table, boot_unix, "reboot", "Warning", msg.c_str(), "", false, &did);
  if (rc == GPUD_OK && inserted) *inserted = did ? 1 : 0;
  return rc;
}

// ---- pkg/kmsg Syncer over the hits of RAW_KMSG scans (syncer.go:73-143) -----------------------------------------------
// For every kmsg record on which the component's Match fires: Event{Time: boot + usec, Name, Message, Type: Warning};
// dropped when the parsed form "name_message" was already seen in the same truncation bucket (deduper.go:63-125: default 60 s
// buckets, 15 min TTL against the wall clock; an event-specific window replaces both, syncer.go:145-155), or when the
// identical event is already in the table (Find), else inserted.
// The watcher's raw-message dedup upstream (watcher.go) drops nothing this step would keep: identical raw lines of one bucket
// parse to identical events.
struct gpud_kmsg_syncer {
  std::string component, table;
  gpud_store* st = nullptr;
  int truncate_seconds = 60;                       // defaultCacheKeyTruncateSeconds (deduper.go:14), WithCacheKeyTruncateSeconds
  bool disable_dedup = false;                      // withDisableDedup
  std::vector<gpud_dedup_rule> rules;              // the EventDedupWindowFunc as data: first rule that matches decides
  struct Entry { int count; int64_t expires; };
  std::map<std::string, Entry> cache;              // go-cache: an item is live while now <= its expiration
};

extern "C" int32_t gpud_kmsg_syncer_create(gpud_store* st, const char* component, gpud_kmsg_syncer** out) {
  if (!st || !component || !out) return GPUD_E_INVALID;
  char t[256];
  const int32_t rc = gpud_store_event_table(st, component, t, sizeof t);
  if (rc) return rc;
  gpud_kmsg_syncer* sy = new gpud_kmsg_syncer();
  sy->component = component; sy->table = t; sy->st = st;
  *out = sy;
  return GPUD_OK;
}
extern "C" void gpud_kmsg_syncer_destroy(gpud_kmsg_syncer* sy) { delete sy; }

extern "C" int32_t gpud_kmsg_syncer_configure(gpud_kmsg_syncer* sy, int32_t truncate_seconds, int32_t disable_dedup, const gpud_dedup_rule* rules,
                                              int32_t n_rules) {
  if (!sy || n_rules < 0 || (n_rules && !rules)) return GPUD_E_INVALID;
  for (int32_t i = 0; i < n_rules; ++i)
    if (!memchr(rules[i].event, 0, sizeof rules[i].event) || !memchr(rules[i].message_contains, 0, sizeof rules[i].message_contains)) return GPUD_E_INVALID;
  sy->truncate_seconds = truncate_seconds > 0 ? truncate_seconds : 60;          // WithCacheKeyTruncateSeconds ignores values <= 0 (deduper.go:35-41)
  sy->disable_dedup = disable_dedup != 0;
  sy->rules.assign(rules, rules + n_rules);
  return GPUD_OK;
}

// The options each reference component passes to kmsg.NewSyncer: infiniband/component.go:149-155 + :166-179 (5 min buckets;
// access_reg_failed: 24 h per PCI device, 5 min without one), peermem/component.go:64-70 and disk/component.go:198-203 (5 min),
// nccl / os / cpu / memory: defaults (nccl/component.go:61, os/component.go:144, cpu/component.go:74, memory/component.go:89).
extern "C" int32_t gpud_kmsg_syncer_configure_component(gpud_kmsg_syncer* sy, const char* kmsg_component) {
  if (!sy || !kmsg_component) return GPUD_E_INVALID;
  const std::string c = kmsg_component;
  if (c == "infiniband") {
    gpud_dedup_rule r[2];
    memset(r, 0, sizeof r);
    snprintf(r[0].event, sizeof r[0].event, "access_reg_failed"); snprintf(r[0].message_contains, sizeof r[0].message_contains, "(PCI device ");
    r[0].window_seconds = 24 * 3600;
    snprintf(r[1].event, sizeof r[1].event, "access_reg_failed"); r[1].window_seconds = 5 * 60;
    return gpud_kmsg_syncer_configure(sy, 300, 0, r, 2);
  }
  if (c == "peermem" || c == "disk") return gpud_kmsg_syncer_configure(sy, 300, 0, nullptr, 0);
  if (c == "nccl" || c == "os" || c == "cpu" || c == "memory") return gpud_kmsg_syncer_configure(sy, 60, 0, nullptr, 0);
  return GPUD_E_INVALID;
}

// One pass of the loop body of Syncer.sync (syncer.go:84-140) for an event the matcher produced.  Caller holds the transaction.
static int32_t syncer_step(gpud_kmsg_syncer* sy, int64_t t, const char* name, const char* msg, int64_t now_unix, bool* inserted) {
  *inserted = false;
  const bool has_deduper = !sy->disable_dedup || !sy->rules.empty();            // syncer.go:54-59
  if (has_deduper) {
    int64_t trunc = sy->disable_dedup ? 60 : sy->truncate_seconds, ttl = 15 * 60;                // dedupParams (syncer.go:145-155)
    for (const gpud_dedup_rule& r : sy->rules) {
      if (strcmp(r.event, name) != 0) continue;
      if (r.message_contains[0] && !strstr(msg, r.message_contains)) continue;
      if (r.window_seconds > 0) { trunc = r.window_seconds; ttl = r.window_seconds; }
      break;
    }
    int64_t rem = t % trunc;                                                   // Go's % truncates toward zero, like C's
    const std::string key = std::to_string(t - rem) + "-" + name + "_" + msg;  // cacheKeyWithTruncateSeconds of Message{name + "_" + message}
    auto it = sy->cache.find(key);
    int freq = 1;
    if (it != sy->cache.end() && it->second.expires >= now_unix) freq = it->second.count + 1;
    sy->cache[key] = gpud_kmsg_syncer::Entry{freq, now_unix + ttl};
    if (freq > 1) return GPUD_OK;
  }
  return insert_event(sy->st, sy->table.c_str(), t, name, "Warning", msg, "", true, inserted);   // Find, then Insert (syncer.go:112-135)
}

extern "C" int32_t gpud_kmsg_syncer_offer(gpud_kmsg_syncer* sy, int64_t unix_s, const char* name, const char* message, int64_t now_unix, int32_t* inserted) {
  if (!sy || !name || !*name) return GPUD_E_INVALID;                            // Match's "" name means no event (syncer.go:85-88)
  if (!sq()) return GPUD_E_UNSUPPORTED;
  bool did = false;
  const int32_t rc = syncer_step(sy, unix_s, name, message ? message : "", now_unix, &did);
  if (inserted) *inserted = did ? 1 : 0;
  return rc;
}

extern "C" int32_t gpud_kmsg_syncer_feed(gpud_kmsg_syncer* sy, const char* kmsg_component, const gpud_xid_hit* hits, int64_t n, const uint8_t* buf,
                                         int64_t boot_unix, int64_t now_unix, int32_t* n_inserted) {
  if (!sy || !kmsg_component || n < 0 || (n && !hits)) return GPUD_E_INVALID;
  Sq* S = sq();
  if (!S) return GPUD_E_UNSUPPORTED;
  int32_t ins = 0;
  if (S->exec(sy->st->db, "BEGIN;", nullptr, nullptr, nullptr) != kOk) return sfail(sy->st, "begin");
  int64_t last_unit = -1;
  for (int64_t i = 0; i < n; ++i) {
    const gpud_xid_hit& h = hits[i];
    if (h.kind < GPUD_KIND_NCCL_SEGFAULT || h.kind >= GPUD_KIND_OS_PANIC_START) continue;       // the stateless line matchers only
    if (strcmp(gpud_kmsg_component(h.kind), kmsg_component) != 0) continue;
    if (h.unit_index == last_unit) continue;                   // Match returns the first pattern of the component that fires (hits are in kind order)
    last_unit = h.unit_index;
    char msg[4096];
    if (gpud_kmsg_hit_message(&h, buf, msg, sizeof msg) < 0) continue;
    bool did = false;
    const int32_t rc = syncer_step(sy, boot_unix + h.kmsg_usec / 1000000, gpud_kmsg_event_name(h.kind), msg, now_unix, &did);
    if (rc) { S->exec(sy->st->db, "ROLLBACK;", nullptr, nullptr, nullptr); return rc; }
    ins += did ? 1 : 0;
  }
  if (S->exec(sy->st->db, "COMMIT;", nullptr, nullptr, nullptr) != kOk) return sfail(sy->st, "commit");
  if (n_inserted) *n_inserted = ins;
  return GPUD_OK;
}

// metrics/store/sqlite.go:87-106
extern "C" int32_t gpud_store_metrics_table(gpud_store* st, const char* table) {
  if (!st) return GPUD_E_INVALID;
  Sq* S = sq();
  if (!S) return GPUD_E_UNSUPPORTED;
  const std::string t = table && *table ? table : "gpud_metrics_v0_5";
  if (!ident_ok(t.c_str())) return GPUD_E_INVALID;
  const std::string ddl = "\nCREATE TABLE IF NOT EXISTS " + t + " (\n\tunix_milliseconds INTEGER NOT NULL,\n\tcomponent_name TEXT NOT NULL,\n\tmetric_name TEXT NOT NULL,\n"
                          "\tmetric_labels TEXT,\n\tmetric_value REAL NOT NULL,\n\tPRIMARY KEY (unix_milliseconds, component_name, metric_name, metric_labels)\n) WITHOUT ROWID;";
  if (S->exec(st->db, ddl.c_str(), nullptr, nullptr, nullptr) != kOk) return sfail(st, "create metrics table");
  return GPUD_OK;
}

// metrics/store/sqlite.go:108-164: INSERT OR REPLACE, one transaction per call
extern "C" int32_t gpud_store_record_metrics(gpud_store* st, const char* table, const gpud_metric* ms, int64_t n) {
  if (!st || n < 0 || (n && !ms)) return GPUD_E_INVALID;
  Sq* S = sq();
  if (!S) return GPUD_E_UNSUPPORTED;
  const std::string t = table && *table ? table : "gpud_metrics_v0_5";
  if (!ident_ok(t.c_str())) return GPUD_E_INVALID;
  for (int64_t i = 0; i < n; ++i)
    if (!ms[i].component || !*ms[i].component || !ms[i].name || !*ms[i].name) return GPUD_E_INVALID;   // ErrEmptyComponentName / ErrEmptyMetricName
  if (n == 0) return GPUD_OK;
  void* q = nullptr;
  const std::string ins = "INSERT OR REPLACE INTO " + t + " (unix_milliseconds, component_name, metric_name, metric_labels, metric_value) VALUES (?, ?, ?, ?, ?)";
  if (S->exec(st->db, "BEGIN;", nullptr, nullptr, nullptr) != kOk) return sfail(st, "begin");
  if (S->prepare_v2(st->db, ins.c_str(), -1, &q, nullptr) != kOk) { S->exec(st->db, "ROLLBACK;", nullptr, nullptr, nullptr); return sfail(st, "prepare metrics insert"); }
  for (int64_t i = 0; i < n; ++i) {
    S->bind_int64(q, 1, ms[i].unix_ms); S->bind_text(q, 2, ms[i].component, -1, kTransient); S->bind_text(q, 3, ms[i].name, -1, kTransient);
    S->bind_text(q, 4, ms[i].labels_json ? ms[i].labels_json : "", -1, kTransient); S->bind_double(q, 5, ms[i].value);
    if (S->step(q) != kDone) { S->finalize(q); S->exec(st->db, "ROLLBACK;", nullptr, nullptr, nullptr); return sfail(st, "insert metric"); }
    S->reset(q);
  }
  S->finalize(q);
  if (S->exec(st->db, "COMMIT;", nullptr, nullptr, nullptr) != kOk) return sfail(st, "commit");
  return GPUD_OK;
}

// metrics/store/sqlite.go:258-275 (purge)
extern "C" int32_t gpud_store_purge_metrics(gpud_store* st, const char* table, int64_t before_unix_ms, int64_t* n_purged) {
  if (!st) return GPUD_E_INVALID;
  Sq* S = sq();
  if (!S) return GPUD_E_UNSUPPORTED;
  const std::string t = table && *table ? table : "gpud_metrics_v0_5";
  if (!ident_ok(t.c_str())) return GPUD_E_INVALID;
  const std::string del = "\nDELETE FROM " + t + " WHERE unix_milliseconds < ?;";
  void* q = nullptr;
  if (S->prepare_v2(st->db, del.c_str(), -1, &q, nullptr) != kOk) return sfail(st, "prepare metrics purge");
  S->bind_int64(q, 1, before_unix_ms);
  const int rc = S->step(q);
  S->finalize(q);
  if (rc != kDone) return sfail(st, "purge metrics");
  if (n_purged) *n_purged = S->changes(st->db);
  return GPUD_OK;
}

extern "C" int32_t gpud_window_metric_name(const char* field, int32_t op, int32_t q_num, int32_t q_den, char* out, int32_t cap) {
  if (!field || !out || op < 0 || op >= GPUD_N_OPS || q_num < 0 || q_den <= 0 || q_num > q_den) return -1;
  static const char* const kOp[GPUD_N_OPS] = {"min", "max", "mean", "ema", nullptr, "n_over"};
  char q[64];
  const char* suffix = kOp[op];
  if (op == GPUD_OP_P99) {
    char g[48];
    snprintf(g, sizeof g, "%g", 100.0 * q_num / q_den);
    for (char* c = g; *c; ++c) if (*c == '.') *c = '_';
    snprintf(q, sizeof q, "p%s", g);
    suffix = q;
  }
  const std::string name = std::string(field) + "_window_" + suffix;
  if ((int32_t)name.size() + 1 > cap) return -1;
  memcpy(out, name.c_str(), name.size() + 1);
  return (int32_t)name.size();
}

// Syncer.sync (syncer.go:76-82) over a ring: peek the next windows, write them in one transaction, and only then move the ring's cursor
extern "C" int32_t gpud_ring_drain_to_store(gpud_ring* ring, gpud_store* st, const char* table, const char* const* components, const char* const* field_names,
                                            const char* labels_json, uint32_t ops_mask, int64_t max_windows, gpud_drain_info* info, int64_t* n_rows,
                                            int64_t* n_shifted) {
  if (!ring || !st || !components || !field_names || max_windows < 0 || ops_mask >= (1u << GPUD_N_OPS)) return GPUD_E_INVALID;
  Sq* S = sq();
  if (!S) return GPUD_E_UNSUPPORTED;
  const std::string t = table && *table ? table : "gpud_metrics_v0_5";
  if (!ident_ok(t.c_str())) return GPUD_E_INVALID;
  const int F = gpud_ring_n_fields(ring);
  for (int f = 0; f < F; ++f)
    if (field_names[f] && (!*field_names[f] || !components[f] || !*components[f])) return GPUD_E_INVALID;   // ErrEmptyComponentName / ErrEmptyMetricName
  if (ops_mask == 0) ops_mask = (1u << GPUD_N_OPS) - 1;
  gpud_drain_info di;
  if (n_rows) *n_rows = 0;
  if (n_shifted) *n_shifted = 0;
  // counts first, so that the host arrays hold the windows that come back rather than max_windows of them
  int32_t rc = gpud_ring_drain_peek(ring, 0, nullptr, nullptr, nullptr, &di);
  const int64_t want = std::min(max_windows, di.n_pending);
  const size_t mw = (size_t)want;
  std::vector<double> f64(5 * (size_t)F * mw + 1);
  std::vector<uint32_t> nov((size_t)F * mw + 1);
  std::vector<int64_t> ms(mw + 1);
  if (rc == GPUD_OK && want > 0) rc = gpud_ring_drain_peek(ring, want, f64.data(), nov.data(), ms.data(), &di);
  if (rc) { st->err = "drain: the ring's reduce failed (see gpud_last_error)"; return rc; }
  if (info) *info = di;
  if (max_windows == 0) return GPUD_OK;                                         // a query
  const int64_t n = di.n_windows;
  for (int64_t j = 0; j < n; ++j)
    if (ms[j] == 0) {
      st->err = "window " + std::to_string(di.first_window + j) + " has no time (its last row was pushed without one)";
      return GPUD_E_STATE;
    }
  // unix_milliseconds leads the primary key: a window that does not come after the previous exported one moves to 1 ms after it
  int64_t prev = gpud_ring_drain_last_export(ring), shifted = 0;
  for (int64_t j = 0; j < n; ++j) {
    if (prev != INT64_MIN && ms[j] <= prev) { ms[j] = prev + 1; ++shifted; }
    prev = ms[j];
  }
  int qn = 99, qd = 100;
  gpud_ring_quantile(ring, &qn, &qd);
  std::vector<std::string> names((size_t)F * GPUD_N_OPS);
  for (int f = 0; f < F; ++f)
    for (int op = 0; op < GPUD_N_OPS; ++op)
      if (field_names[f] && ((ops_mask >> op) & 1u)) {
        char b[512];
        if (gpud_window_metric_name(field_names[f], op, qn, qd, b, sizeof b) < 0) return GPUD_E_INVALID;
        names[(size_t)f * GPUD_N_OPS + op] = b;
      }
  int64_t rows = 0;
  if (n > 0) {
    const std::string ins = "INSERT OR REPLACE INTO " + t + " (unix_milliseconds, component_name, metric_name, metric_labels, metric_value) VALUES (?, ?, ?, ?, ?)";
    void* q = nullptr;
    if (S->exec(st->db, "BEGIN;", nullptr, nullptr, nullptr) != kOk) return sfail(st, "begin");
    if (S->prepare_v2(st->db, ins.c_str(), -1, &q, nullptr) != kOk) { rc = sfail(st, "prepare metrics insert"); S->exec(st->db, "ROLLBACK;", nullptr, nullptr, nullptr); return rc; }
    for (int64_t j = 0; j < n; ++j)
      for (int f = 0; f < F; ++f)
        for (int op = 0; op < GPUD_N_OPS; ++op) {
          const std::string& name = names[(size_t)f * GPUD_N_OPS + op];
          if (name.empty()) continue;
          const double v = op == GPUD_OP_NOVER ? (double)nov[(size_t)f * mw + j] : f64[((size_t)op * F + f) * mw + j];
          S->bind_int64(q, 1, ms[j]); S->bind_text(q, 2, components[f], -1, kTransient); S->bind_text(q, 3, name.c_str(), -1, kTransient);
          S->bind_text(q, 4, labels_json ? labels_json : "", -1, kTransient); S->bind_double(q, 5, v);
          if (S->step(q) != kDone) { rc = sfail(st, "insert metric"); S->finalize(q); S->exec(st->db, "ROLLBACK;", nullptr, nullptr, nullptr); return rc; }
          S->reset(q);
          ++rows;
        }
    S->finalize(q);
    if (S->exec(st->db, "COMMIT;", nullptr, nullptr, nullptr) != kOk) { rc = sfail(st, "commit"); S->exec(st->db, "ROLLBACK;", nullptr, nullptr, nullptr); return rc; }
  }
  gpud_ring_drain_commit(ring, &di, n > 0 ? prev : INT64_MIN);
  if (n_rows) *n_rows = rows;
  if (n_shifted) *n_shifted = shifted;
  return GPUD_OK;
}

// test entry (not in gpud_b200.h): the text of event statement `which` for `table`
extern "C" int32_t gpudh_store_event_sql(int32_t which, const char* table, char* out, int32_t cap) {
  const std::string q = event_sql(which, table ? table : "");
  if (q.empty() || (int32_t)q.size() + 1 > cap) return -1;
  memcpy(out, q.c_str(), q.size() + 1);
  return (int32_t)q.size();
}
