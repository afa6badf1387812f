// Batched decode of the reference's vehicle wire format (host side, C++17, no third-party JSON).
//
// The reference moves one JSON message per vehicle update through its broker and turns each into a
// Vehicle in Python (producer: src/test/vehicle_simulator.py:721-752 `get_vehicle_json`; consumer:
// src/collision/warning_system.py:638-678 `_handle_vehicle_position`, which reads
// data["id"], data["position"|"velocity"|"acceleration"]["x"|"y"|"z"], data["heading"], data["size"],
// data["type"], data["timestamp"] and drops the message on any exception).  This decoder takes a whole
// buffer of such messages and fills fixed 72-byte records (include/rcd.h, rcd_record) that
// rcd_apply_records scatters into the device-resident frame state and trajectory rings:
//   - numbers are converted with std::from_chars (correctly rounded, like Python's float()); NaN / Infinity /
//     -Infinity are accepted like json.loads does;
//   - id and type strings are unescaped to UTF-8 and interned: id -> dense slot (first seen first; slots freed by
//     rcd_ingest_release are handed out again, lowest first, before any fresh slot),
//     type -> small code (only equality of types is ever used, collision_detection.py:498-513);
//   - a message that is not valid JSON, or lacks one of the fields the reference reads, is skipped and
//     counted (the reference logs and drops it, warning_system.py:677-678);
//   - unknown keys are ignored, key order and whitespace are free, duplicate keys: last one wins
//     (json.loads semantics).
#pragma once
#include <charconv>
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <queue>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "../../include/rcd.h"

namespace rcd_ingest_impl {

struct Msg {
    double pos[3], vel[3], acc[3], heading, size, timestamp;
    std::string id, type;
};

struct Cursor {
    const char *p, *end;
    bool at_end() const { return p >= end; }
    void ws() {
        while (p < end && (*p == ' ' || *p == '\t' || *p == '\n' || *p == '\r')) ++p;
    }
    bool eat(char c) {
        ws();
        if (p < end && *p == c) { ++p; return true; }
        return false;
    }
};

inline void put_utf8(std::string &out, uint32_t cp) {
    if (cp < 0x80) out.push_back((char)cp);
    else if (cp < 0x800) { out.push_back((char)(0xC0 | (cp >> 6))); out.push_back((char)(0x80 | (cp & 0x3F))); }
    else if (cp < 0x10000) {
        out.push_back((char)(0xE0 | (cp >> 12))); out.push_back((char)(0x80 | ((cp >> 6) & 0x3F)));
        out.push_back((char)(0x80 | (cp & 0x3F)));
    } else {
        out.push_back((char)(0xF0 | (cp >> 18))); out.push_back((char)(0x80 | ((cp >> 12) & 0x3F)));
        out.push_back((char)(0x80 | ((cp >> 6) & 0x3F))); out.push_back((char)(0x80 | (cp & 0x3F)));
    }
}
inline bool hex4(Cursor &c, uint32_t &v) {
    if (c.end - c.p < 4) return false;
    v = 0;
    for (int k = 0; k < 4; ++k) {
        char ch = c.p[k];
        uint32_t d;
        if (ch >= '0' && ch <= '9') d = ch - '0';
        else if (ch >= 'a' && ch <= 'f') d = ch - 'a' + 10;
        else if (ch >= 'A' && ch <= 'F') d = ch - 'A' + 10;
        else return false;
        v = v * 16 + d;
    }
    c.p += 4;
    return true;
}

// string at the cursor (opening quote already consumed when `opened`); out may be null (skip)
inline bool parse_string(Cursor &c, std::string *out) {
    c.ws();
    if (c.at_end() || *c.p != '"') return false;
    ++c.p;
    if (out) out->clear();
    while (c.p < c.end) {
        unsigned char ch = (unsigned char)*c.p++;
        if (ch == '"') return true;
        if (ch < 0x20) return false;  // json.loads (strict) rejects raw control characters
        if (ch != '\\') {
            if (out) out->push_back((char)ch);
            continue;
        }
        if (c.p >= c.end) return false;
        char e = *c.p++;
        char lit = 0;
        switch (e) {
            case '"': lit = '"'; break;
            case '\\': lit = '\\'; break;
            case '/': lit = '/'; break;
            case 'b': lit = '\b'; break;
            case 'f': lit = '\f'; break;
            case 'n': lit = '\n'; break;
            case 'r': lit = '\r'; break;
            case 't': lit = '\t'; break;
            case 'u': {
                uint32_t cp;
                if (!hex4(c, cp)) return false;
                if (cp >= 0xD800 && cp < 0xDC00 && c.end - c.p >= 6 && c.p[0] == '\\' && c.p[1] == 'u') {
                    Cursor save = c;
                    c.p += 2;
                    uint32_t lo;
                    if (hex4(c, lo) && lo >= 0xDC00 && lo < 0xE000) cp = 0x10000 + ((cp - 0xD800) << 10) + (lo - 0xDC00);
                    else c = save;  // lone surrogate: kept as is (json.loads does the same)
                }
                if (out) put_utf8(*out, cp);
                continue;
            }
            default: return false;
        }
        if (out) out->push_back(lit);
    }
    return false;
}

// JSON number, or NaN / Infinity / -Infinity (json.loads accepts those); bool / null / strings are not numbers
inline bool parse_number(Cursor &c, double &v) {
    c.ws();
    if (c.at_end()) return false;
    const char *s = c.p;
    size_t left = (size_t)(c.end - s);
    if (left >= 3 && !memcmp(s, "NaN", 3)) { v = NAN; c.p += 3; return true; }
    if (left >= 8 && !memcmp(s, "Infinity", 8)) { v = INFINITY; c.p += 8; return true; }
    if (left >= 9 && !memcmp(s, "-Infinity", 9)) { v = -INFINITY; c.p += 9; return true; }
    // validate the JSON grammar: -? (0 | [1-9][0-9]*) (. [0-9]+)? ([eE] [+-]? [0-9]+)?
    const char *q = s;
    if (q < c.end && *q == '-') ++q;
    if (q >= c.end) return false;
    if (*q == '0') ++q;
    else if (*q >= '1' && *q <= '9') { while (q < c.end && *q >= '0' && *q <= '9') ++q; }
    else return false;
    if (q < c.end && *q == '.') {
        ++q;
        if (q >= c.end || *q < '0' || *q > '9') return false;
        while (q < c.end && *q >= '0' && *q <= '9') ++q;
    }
    if (q < c.end && (*q == 'e' || *q == 'E')) {
        ++q;
        if (q < c.end && (*q == '+' || *q == '-')) ++q;
        if (q >= c.end || *q < '0' || *q > '9') return false;
        while (q < c.end && *q >= '0' && *q <= '9') ++q;
    }
    // correctly rounded like Python's float(): libstdc++'s from_chars (Eisel-Lemire with exact fallback)
    auto res = std::from_chars(s, q, v);
    if (res.ec == std::errc::result_out_of_range) {  // json.loads gives +-inf / 0.0 here; so does strtod
        std::string big(s, (size_t)(q - s));
        v = strtod(big.c_str(), nullptr);
    } else if (res.ec != std::errc() || res.ptr != q) {
        return false;
    }
    c.p = q;
    return true;
}

inline bool skip_value(Cursor &c, int depth = 0);
inline bool skip_container(Cursor &c, char close, bool is_object, int depth) {
    if (depth > 64) return false;
    if (c.eat(close)) return true;
    for (;;) {
        if (is_object) {
            if (!parse_string(c, nullptr)) return false;
            if (!c.eat(':')) return false;
        }
        if (!skip_value(c, depth + 1)) return false;
        if (c.eat(',')) continue;
        return c.eat(close);
    }
}
inline bool skip_value(Cursor &c, int depth) {
    c.ws();
    if (c.at_end()) return false;
    char ch = *c.p;
    if (ch == '"') return parse_string(c, nullptr);
    if (ch == '{') { ++c.p; return skip_container(c, '}', true, depth); }
    if (ch == '[') { ++c.p; return skip_container(c, ']', false, depth); }
    size_t left = (size_t)(c.end - c.p);
    if (left >= 4 && !memcmp(c.p, "true", 4)) { c.p += 4; return true; }
    if (left >= 5 && !memcmp(c.p, "false", 5)) { c.p += 5; return true; }
    if (left >= 4 && !memcmp(c.p, "null", 4)) { c.p += 4; return true; }
    double d;
    return parse_number(c, d);
}

enum { F_ID = 1, F_POS = 2, F_VEL = 4, F_ACC = 8, F_HEADING = 16, F_SIZE = 32, F_TYPE = 64, F_TS = 128, F_ALL = 255 };
enum ParseStatus { PARSE_OK = 0, PARSE_INCOMPLETE = 1, PARSE_SYNTAX = 2 };

// {"x": .., "y": .., "z": ..}; returns 1 ok, 0 well-formed but unusable (missing axis / not numbers), -1 syntax error
inline int parse_vec3(Cursor &c, double v[3]) {
    c.ws();
    if (c.at_end()) return -1;
    if (*c.p != '{') return skip_value(c) ? 0 : -1;
    ++c.p;
    int have = 0;
    bool usable = true;
    if (c.eat('}')) return 0;
    std::string key;
    for (;;) {
        if (!parse_string(c, &key)) return -1;
        if (!c.eat(':')) return -1;
        int axis = (key.size() == 1 && key[0] >= 'x' && key[0] <= 'z') ? key[0] - 'x' : -1;
        if (axis >= 0) {
            Cursor save = c;
            if (parse_number(c, v[axis])) have |= 1 << axis;
            else {
                c = save;
                if (!skip_value(c)) return -1;
                have &= ~(1 << axis);
                usable = false;  // present but not a number: the reference would carry a non-number along
            }
        } else if (!skip_value(c)) return -1;
        if (c.eat(',')) continue;
        if (!c.eat('}')) return -1;
        break;
    }
    return (usable && have == 7) ? 1 : 0;
}

// one message object at the cursor
inline ParseStatus parse_message(Cursor &c, Msg &m) {
    if (!c.eat('{')) return PARSE_SYNTAX;
    int have = 0, bad = 0;
    std::string key;
    if (!c.eat('}')) {
        for (;;) {
            if (!parse_string(c, &key)) return PARSE_SYNTAX;
            if (!c.eat(':')) return PARSE_SYNTAX;
            int field = 0;
            int ok = 1;
            if (key == "id") { field = F_ID; c.ws(); if (!c.at_end() && *c.p == '"') ok = parse_string(c, &m.id) ? 1 : -1; else ok = skip_value(c) ? 0 : -1; }
            else if (key == "type") { field = F_TYPE; c.ws(); if (!c.at_end() && *c.p == '"') ok = parse_string(c, &m.type) ? 1 : -1; else ok = skip_value(c) ? 0 : -1; }
            else if (key == "position") { field = F_POS; ok = parse_vec3(c, m.pos); }
            else if (key == "velocity") { field = F_VEL; ok = parse_vec3(c, m.vel); }
            else if (key == "acceleration") { field = F_ACC; ok = parse_vec3(c, m.acc); }
            else if (key == "heading" || key == "size" || key == "timestamp") {
                field = key[0] == 'h' ? F_HEADING : (key[0] == 's' ? F_SIZE : F_TS);
                double *dst = key[0] == 'h' ? &m.heading : (key[0] == 's' ? &m.size : &m.timestamp);
                Cursor save = c;
                if (!parse_number(c, *dst)) { c = save; ok = skip_value(c) ? 0 : -1; }
            } else if (!skip_value(c)) return PARSE_SYNTAX;
            if (ok < 0) return PARSE_SYNTAX;
            if (field) {  // duplicate keys: the last one wins
                if (ok) { have |= field; bad &= ~field; } else { have &= ~field; bad |= field; }
            }
            if (c.eat(',')) continue;
            if (!c.eat('}')) return PARSE_SYNTAX;
            break;
        }
    }
    return (have == F_ALL && !bad) ? PARSE_OK : PARSE_INCOMPLETE;
}

// all messages of [p, end): objects separated by whitespace / newlines / commas, optionally inside [ ]
inline void parse_range(const char *p, const char *end, std::vector<Msg> &out, uint64_t &n_bad) {
    Cursor c{p, end};
    Msg m;
    for (;;) {
        c.ws();
        if (c.at_end()) break;
        if (*c.p == '[' || *c.p == ']' || *c.p == ',') { ++c.p; continue; }
        const char *start = c.p;
        ParseStatus st = parse_message(c, m);
        if (st == PARSE_OK) { out.push_back(m); continue; }
        ++n_bad;
        if (st == PARSE_SYNTAX) {  // resynchronise at the next line
            const char *nl = (const char *)memchr(start, '\n', (size_t)(end - start));
            c.p = nl ? nl + 1 : end;
        }
    }
}

struct Ingest {
    std::unordered_map<std::string, uint32_t> ids, types;
    std::vector<std::string> id_names, type_names;
    std::vector<uint32_t> batch_stamp;  // per slot: batch number of the last message
    std::vector<uint8_t> batch_seq;     // per slot: messages seen in that batch
    std::vector<uint8_t> slot_free;     // per slot: released, no id (rcd_ingest_release)
    std::priority_queue<uint32_t, std::vector<uint32_t>, std::greater<uint32_t>> free_slots;  // lowest first
    uint32_t batch = 0;
    uint64_t max_ids = ~0ull;           // live ids beyond this are rejected (rcd_ingest_set_limit)
    uint64_t n_rejected = 0;            // messages dropped since creation: unknown id with the table full,
                                        // or more than 255 messages of one vehicle in one call
    std::string err;
    uint64_t n_live() const { return id_names.size() - free_slots.size(); }
};
constexpr uint32_t TYPE_CODE_OTHER = 255;  // every type string beyond the first 255 distinct ones

}  // namespace rcd_ingest_impl

struct rcd_ingest_s : rcd_ingest_impl::Ingest {};

extern "C" {

int rcd_ingest_create(rcd_ingest *out) {
    if (!out) return RCD_EINVAL;
    *out = new (std::nothrow) rcd_ingest_s();
    return *out ? RCD_OK : RCD_ENOMEM;
}
int rcd_ingest_destroy(rcd_ingest g) {
    delete g;
    return RCD_OK;
}
const char *rcd_ingest_last_error(rcd_ingest g) { return g ? g->err.c_str() : "null ingest handle"; }

int rcd_ingest_decode_json(rcd_ingest g, const char *buf, uint64_t len, int32_t threads, rcd_record *out, uint64_t cap,
                           uint64_t *n_out, uint64_t *n_bad_out, uint32_t *max_seq_out) {
    using namespace rcd_ingest_impl;
    if (!g || (len && !buf) || (cap && !out) || !n_out) return RCD_EINVAL;
    try {
        // ---- parse (parallel over line-aligned chunks) ----
        int T = threads <= 0 ? (int)std::min<unsigned>(std::max(1u, std::thread::hardware_concurrency()), 16u) : threads;
        if (len < (1u << 20)) T = 1;
        std::vector<const char *> cut(T + 1);
        cut[0] = buf;
        cut[T] = buf + len;
        for (int k = 1; k < T; ++k) {
            const char *guess = buf + len / T * k;
            if (guess < cut[k - 1]) guess = cut[k - 1];
            const char *nl = (const char *)memchr(guess, '\n', (size_t)(buf + len - guess));
            cut[k] = nl ? nl + 1 : buf + len;
        }
        std::vector<std::vector<Msg>> parts(T);
        std::vector<uint64_t> bad(T, 0);
        if (T == 1) {
            parse_range(cut[0], cut[1], parts[0], bad[0]);
        } else {
            std::vector<std::thread> pool;
            for (int k = 0; k < T; ++k)
                pool.emplace_back([&, k] { parse_range(cut[k], cut[k + 1], parts[k], bad[k]); });
            for (auto &t : pool) t.join();
        }
        // ---- capacity is checked before any state changes: a caller that retries with a larger buffer sees the
        // same slots and sequence numbers as if the first call had never happened
        uint64_t n_parsed = 0, n_bad = 0;
        for (int k = 0; k < T; ++k) { n_parsed += parts[k].size(); n_bad += bad[k]; }
        if (n_parsed > cap) {
            *n_out = n_parsed;
            if (n_bad_out) *n_bad_out = n_bad;
            if (max_seq_out) *max_seq_out = 0;
            g->err = "record buffer too small";
            return RCD_ECAPACITY;
        }
        // ---- intern + fill records (serial: slots are assigned in arrival order).  Every message stands on its
        // own, like in the reference's handler (warning_system.py:638-678): one that cannot be taken is dropped
        // and counted, the rest of the batch is applied.
        ++g->batch;
        uint64_t n = 0;
        uint32_t max_seq = 0;
        for (int k = 0; k < T; ++k) {
            for (const Msg &m : parts[k]) {
                auto it = g->ids.find(m.id);
                uint32_t slot;
                if (it == g->ids.end()) {
                    if (g->n_live() >= g->max_ids) {  // table full: known vehicles keep being served
                        ++n_bad;
                        ++g->n_rejected;
                        continue;
                    }
                    if (!g->free_slots.empty()) {  // a released slot, lowest first
                        slot = g->free_slots.top();
                        g->free_slots.pop();
                        g->slot_free[slot] = 0;
                        g->id_names[slot] = m.id;
                        g->batch_stamp[slot] = 0;
                        g->batch_seq[slot] = 0;
                    } else {
                        slot = (uint32_t)g->id_names.size();
                        g->id_names.push_back(m.id);
                        g->batch_stamp.push_back(0);
                        g->batch_seq.push_back(0);
                        g->slot_free.push_back(0);
                    }
                    g->ids.emplace(m.id, slot);
                } else slot = it->second;
                auto tt = g->types.find(m.type);
                uint32_t code;
                if (tt == g->types.end()) {
                    if (g->type_names.size() >= TYPE_CODE_OTHER) {
                        // the record format has 8 bits: the types beyond the first 255 share one code (only equality
                        // of types is ever used, collision_detection.py:498-513; they compare equal to each other)
                        code = TYPE_CODE_OTHER;
                    } else {
                        code = (uint32_t)g->type_names.size();
                        g->types.emplace(m.type, code);
                        g->type_names.push_back(m.type);
                    }
                } else code = tt->second;
                if (g->batch_stamp[slot] != g->batch) { g->batch_stamp[slot] = g->batch; g->batch_seq[slot] = 0; }
                const uint32_t seq = g->batch_seq[slot];
                if (seq >= 255) {  // 8-bit sequence numbers: the 256th message of one vehicle in one call is dropped
                    ++n_bad;
                    ++g->n_rejected;
                    continue;
                }
                g->batch_seq[slot] = (uint8_t)(seq + 1);
                if (seq > max_seq) max_seq = seq;
                if (n < cap) {
                    rcd_record &r = out[n];
                    r.x = m.pos[0]; r.y = m.pos[1]; r.z = m.pos[2];
                    r.timestamp = m.timestamp;
                    r.vx = (float)m.vel[0]; r.vy = (float)m.vel[1]; r.vz = (float)m.vel[2];
                    r.ax = (float)m.acc[0]; r.ay = (float)m.acc[1]; r.az = (float)m.acc[2];
                    r.size = (float)m.size; r.heading = (float)m.heading;
                    r.slot = slot;
                    r.type = (uint8_t)code;
                    r.seq = (uint8_t)seq;
                    r.reserved = 0;
                }
                ++n;
            }
        }
        *n_out = n;
        if (n_bad_out) *n_bad_out = n_bad;
        if (max_seq_out) *max_seq_out = max_seq;
        return RCD_OK;
    } catch (const std::bad_alloc &) {
        g->err = "out of host memory";
        return RCD_ENOMEM;
    } catch (...) {
        g->err = "unexpected failure";
        return RCD_EINVAL;
    }
}

int rcd_ingest_set_limit(rcd_ingest g, uint64_t max_ids) {
    if (!g) return RCD_EINVAL;
    g->max_ids = max_ids;
    return RCD_OK;
}
int rcd_ingest_rejected(rcd_ingest g, uint64_t *n) {
    if (!g || !n) return RCD_EINVAL;
    *n = g->n_rejected;
    return RCD_OK;
}
int rcd_ingest_counts(rcd_ingest g, uint64_t *n_ids, uint64_t *n_types) {
    if (!g) return RCD_EINVAL;
    if (n_ids) *n_ids = g->id_names.size();
    if (n_types) *n_types = g->type_names.size();
    return RCD_OK;
}
int rcd_ingest_id_name(rcd_ingest g, uint32_t slot, const char **name, uint32_t *len) {
    if (!g || !name || !len || slot >= g->id_names.size() || g->slot_free[slot]) return RCD_EINVAL;
    *name = g->id_names[slot].data();
    *len = (uint32_t)g->id_names[slot].size();
    return RCD_OK;
}
int rcd_ingest_type_name(rcd_ingest g, uint32_t code, const char **name, uint32_t *len) {
    if (!g || !name || !len) return RCD_EINVAL;
    if (code == rcd_ingest_impl::TYPE_CODE_OTHER && g->type_names.size() <= code) {
        *name = "";
        *len = 0;
        return RCD_OK;
    }
    if (code >= g->type_names.size()) return RCD_EINVAL;
    *name = g->type_names[code].data();
    *len = (uint32_t)g->type_names[code].size();
    return RCD_OK;
}
int rcd_ingest_lookup(rcd_ingest g, const char *id, uint32_t len, uint32_t *slot) {
    if (!g || !id || !slot) return RCD_EINVAL;
    auto it = g->ids.find(std::string(id, len));
    if (it == g->ids.end()) return RCD_ESTATE;
    *slot = it->second;
    return RCD_OK;
}

int rcd_ingest_release(rcd_ingest g, uint64_t n, const uint32_t *slots, uint64_t *n_live) {
    if (!g || (n && !slots)) return RCD_EINVAL;
    try {
        // every slot is checked before anything changes
        std::vector<uint8_t> seen(n ? g->id_names.size() : 0, 0);
        for (uint64_t k = 0; k < n; ++k) {
            const uint32_t s = slots[k];
            if (s >= g->id_names.size()) { g->err = "rcd_ingest_release: slot " + std::to_string(s) + " was never handed out"; return RCD_EINVAL; }
            if (g->slot_free[s]) { g->err = "rcd_ingest_release: slot " + std::to_string(s) + " is free"; return RCD_EINVAL; }
            if (seen[s]) { g->err = "rcd_ingest_release: slot " + std::to_string(s) + " is listed twice"; return RCD_EINVAL; }
            seen[s] = 1;
        }
        for (uint64_t k = 0; k < n; ++k) {
            const uint32_t s = slots[k];
            g->ids.erase(g->id_names[s]);
            std::string().swap(g->id_names[s]);
            g->slot_free[s] = 1;
            g->free_slots.push(s);
        }
    } catch (const std::bad_alloc &) {
        g->err = "out of host memory";
        return RCD_ENOMEM;
    }
    if (n_live) *n_live = g->n_live();
    return RCD_OK;
}

}  // extern "C"
