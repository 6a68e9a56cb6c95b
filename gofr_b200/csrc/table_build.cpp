// table_build.cpp — host side of the route table: registration → sealed image.
//
// Mirrors the registration half of the reference: Router.Add (pkg/gofr/http/router.go:30-33) appends
// [methodMatcher, pathRegexp] routes in call order; App.Run (pkg/gofr/gofr.go:102-107) appends health, favicon and
// the PathPrefix("/") catch-all; after Run nothing mutates the table.  gofr_table_seal "compiles" every route into a
// response program (table_format.h) so the device never interprets Go semantics at request time: status line, the
// sorted header block net/http 1.21 writes, the envelope of Responder.Respond (pkg/gofr/http/responder.go:19-41) and
// the struct keys of encoding/json are all folded into literals; only per-request values remain as ops.
#include <algorithm>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/gofr_b200.h"
#include "engine_internal.h"
#include "table_format.h"

namespace gofr {

// FNV-1a, 32 bit: integrity of a sealed image in transit (not a security feature)
static uint32_t image_checksum(const uint8_t* p, size_t n) {
    uint32_t h = 2166136261u;
    for (size_t i = 0; i < n; i++) { h ^= p[i]; h *= 16777619u; }
    return h;
}

// ---------------------------------------------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------------------------------------------

// encoding/json string escaping with escapeHTML=true, Go 1.21 (no \b \f short forms).  Driven by a class table so it
// shares no structure with the test oracle.  Returns the escaped contents WITHOUT the surrounding quotes.
static const uint8_t* escape_class_table() {
    // 0 = copy, 1 = \uXXXX, 2 = backslash + char, 3 = \n, 4 = \r, 5 = \t, 6 = multi-byte lead / invalid
    static uint8_t t[256];
    static bool init = false;
    if (!init) {
        for (int c = 0; c < 256; c++) t[c] = c < 0x20 ? 1 : (c >= 0x80 ? 6 : 0);
        t['"'] = 2; t['\\'] = 2; t['\n'] = 3; t['\r'] = 4; t['\t'] = 5;
        t['<'] = 1; t['>'] = 1; t['&'] = 1;
        init = true;
    }
    return t;
}

// length of the well-formed UTF-8 sequence starting at s (Go utf8 acceptance), 0 if ill-formed
static int utf8_seq_len(const uint8_t* s, size_t n) {
    uint8_t a = s[0];
    int len = a >= 0xC2 && a <= 0xDF ? 2 : a >= 0xE0 && a <= 0xEF ? 3 : a >= 0xF0 && a <= 0xF4 ? 4 : 0;
    if (!len || n < (size_t)len) return 0;
    uint8_t lo = a == 0xE0 ? 0xA0 : a == 0xF0 ? 0x90 : 0x80;
    uint8_t hi = a == 0xED ? 0x9F : a == 0xF4 ? 0x8F : 0xBF;
    if (s[1] < lo || s[1] > hi) return 0;
    for (int k = 2; k < len; k++)
        if ((s[k] & 0xC0) != 0x80) return 0;
    return len;
}

std::string json_escape_go(const std::string& in) {
    static const char* hex = "0123456789abcdef";
    const uint8_t* cls = escape_class_table();
    std::string out;
    out.reserve(in.size() + 8);
    const uint8_t* s = (const uint8_t*)in.data();
    size_t n = in.size();
    for (size_t i = 0; i < n;) {
        uint8_t c = s[i];
        switch (cls[c]) {
            case 0: out.push_back((char)c); i++; break;
            case 1: out += "\\u00"; out.push_back(hex[c >> 4]); out.push_back(hex[c & 15]); i++; break;
            case 2: out.push_back('\\'); out.push_back((char)c); i++; break;
            case 3: out += "\\n"; i++; break;
            case 4: out += "\\r"; i++; break;
            case 5: out += "\\t"; i++; break;
            default: {
                int L = utf8_seq_len(s + i, n - i);
                if (L == 0) { out += "\\ufffd"; i++; break; }
                if (L == 3 && s[i] == 0xE2 && s[i + 1] == 0x80 && (s[i + 2] == 0xA8 || s[i + 2] == 0xA9)) {
                    out += s[i + 2] == 0xA8 ? "\\u2028" : "\\u2029";
                } else {
                    out.append((const char*)s + i, (size_t)L);
                }
                i += (size_t)L;
            }
        }
    }
    return out;
}

static bool valid_utf8(const std::string& s) {
    const uint8_t* p = (const uint8_t*)s.data();
    for (size_t i = 0; i < s.size();) {
        if (p[i] < 0x80) { i++; continue; }
        int L = utf8_seq_len(p + i, s.size() - i);
        if (!L) return false;
        i += (size_t)L;
    }
    return true;
}

static const char* status_text(int code) {
    switch (code) {
        case 200: return "OK";
        case 301: return "Moved Permanently";
        case 404: return "Not Found";
        case 405: return "Method Not Allowed";
        case 500: return "Internal Server Error";
    }
    return "";
}

// http.DetectContentType for static file blobs (seal time): net/http's sniffing algorithm (sniff.go, the WHATWG MIME
// Sniffing tables) restated in the order of its sniffSignatures — the first signature that matches the first 512 bytes wins.
static std::string sniff_content_type(const std::string& blob) {
    const std::string d = blob.substr(0, 512);
    const size_t n = d.size();
    const uint8_t* p = (const uint8_t*)d.data();
    size_t ws = 0;  // firstNonWS
    while (ws < n && (p[ws] == '\t' || p[ws] == '\n' || p[ws] == '\x0c' || p[ws] == '\r' || p[ws] == ' ')) ws++;
    // htmlSig: case-insensitive tag name after leading whitespace, followed by a space or '>'
    static const char* const html[] = {"<!DOCTYPE HTML", "<HTML", "<HEAD", "<SCRIPT", "<IFRAME", "<H1", "<DIV", "<FONT", "<TABLE",
                                       "<A", "<STYLE", "<TITLE", "<B", "<BODY", "<BR", "<P", "<!--"};
    for (const char* sig : html) {
        const size_t L = strlen(sig);
        if (n - ws < L + 1) continue;
        bool ok = true;
        for (size_t q = 0; q < L && ok; q++) {
            uint8_t c = p[ws + q];
            const uint8_t t = (uint8_t)sig[q];
            if (t >= 'A' && t <= 'Z') c &= 0xDF;
            ok = c == t;
        }
        if (ok && (p[ws + L] == ' ' || p[ws + L] == '>')) return "text/html; charset=utf-8";
    }
    // exactSig / maskedSig entries: pattern, mask (nullptr = all ones), length, skip leading whitespace, type
    struct Sig { const char* pat; const char* mask; size_t len; bool skip_ws; const char* ct; };
    static const char kLP[37] = "\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0LP";
    static const char kLPm[37] = "\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\0\xFF\xFF";
    static const Sig before_mp4[] = {
        {"<?xml", nullptr, 5, true, "text/xml; charset=utf-8"},
        {"%PDF-", nullptr, 5, false, "application/pdf"},
        {"%!PS-Adobe-", nullptr, 11, false, "application/postscript"},
        {"\xFE\xFF\0\0", "\xFF\xFF\0\0", 4, false, "text/plain; charset=utf-16be"},
        {"\xFF\xFE\0\0", "\xFF\xFF\0\0", 4, false, "text/plain; charset=utf-16le"},
        {"\xEF\xBB\xBF\0", "\xFF\xFF\xFF\0", 4, false, "text/plain; charset=utf-8"},
        {"\0\0\x01\0", nullptr, 4, false, "image/x-icon"},
        {"\0\0\x02\0", nullptr, 4, false, "image/x-icon"},
        {"BM", nullptr, 2, false, "image/bmp"},
        {"GIF87a", nullptr, 6, false, "image/gif"},
        {"GIF89a", nullptr, 6, false, "image/gif"},
        {"RIFF\0\0\0\0WEBPVP", "\xFF\xFF\xFF\xFF\0\0\0\0\xFF\xFF\xFF\xFF\xFF\xFF", 14, false, "image/webp"},
        {"\x89PNG\x0D\x0A\x1A\x0A", nullptr, 8, false, "image/png"},
        {"\xFF\xD8\xFF", nullptr, 3, false, "image/jpeg"},
        {"FORM\0\0\0\0AIFF", "\xFF\xFF\xFF\xFF\0\0\0\0\xFF\xFF\xFF\xFF", 12, false, "audio/aiff"},
        {"ID3", nullptr, 3, false, "audio/mpeg"},
        {"OggS\0", nullptr, 5, false, "application/ogg"},
        {"MThd\0\0\0\x06", nullptr, 8, false, "audio/midi"},
        {"RIFF\0\0\0\0AVI ", "\xFF\xFF\xFF\xFF\0\0\0\0\xFF\xFF\xFF\xFF", 12, false, "video/avi"},
        {"RIFF\0\0\0\0WAVE", "\xFF\xFF\xFF\xFF\0\0\0\0\xFF\xFF\xFF\xFF", 12, false, "audio/wave"},
    };
    static const Sig after_mp4[] = {
        {"\x1A\x45\xDF\xA3", nullptr, 4, false, "video/webm"},
        {kLP, kLPm, 36, false, "application/vnd.ms-fontobject"},
        {"\0\x01\0\0", nullptr, 4, false, "font/ttf"},
        {"OTTO", nullptr, 4, false, "font/otf"},
        {"ttcf", nullptr, 4, false, "font/collection"},
        {"wOFF", nullptr, 4, false, "font/woff"},
        {"wOF2", nullptr, 4, false, "font/woff2"},
        {"\x1F\x8B\x08", nullptr, 3, false, "application/x-gzip"},
        {"PK\x03\x04", nullptr, 4, false, "application/zip"},
        {"Rar!\x1A\x07\0", nullptr, 7, false, "application/x-rar-compressed"},
        {"Rar!\x1A\x07\x01\0", nullptr, 8, false, "application/x-rar-compressed"},
        {"\0\x61\x73\x6D", nullptr, 4, false, "application/wasm"},
    };
    auto match = [&](const Sig& g) {
        const uint8_t* q = p + (g.skip_ws ? ws : 0);
        const size_t avail = n - (g.skip_ws ? ws : 0);
        if (avail < g.len) return false;
        for (size_t k = 0; k < g.len; k++) {
            const uint8_t m = g.mask ? (uint8_t)g.mask[k] : 0xFF;
            if ((q[k] & m) != (uint8_t)g.pat[k]) return false;
        }
        return true;
    };
    for (const Sig& g : before_mp4) if (match(g)) return g.ct;
    // mp4Sig: an "ftyp" box whose size covers it, with a compatible brand starting "mp4" (the major brand's version is skipped)
    if (n >= 12) {
        const size_t box = (size_t)p[0] << 24 | (size_t)p[1] << 16 | (size_t)p[2] << 8 | p[3];
        if (n >= box && box % 4 == 0 && memcmp(p + 4, "ftyp", 4) == 0)
            for (size_t st = 8; st < box; st += 4)
                if (st != 12 && memcmp(p + st, "mp4", 3) == 0) return "video/mp4";
    }
    for (const Sig& g : after_mp4) if (match(g)) return g.ct;
    // textSig: no binary byte from the first non-whitespace byte on
    for (size_t k = ws; k < n; k++) {
        const uint8_t c = p[k];
        if (c <= 0x08 || c == 0x0B || (c >= 0x0E && c <= 0x1A) || (c >= 0x1C && c <= 0x1F)) return "application/octet-stream";
    }
    return "text/plain; charset=utf-8";
}

// ---------------------------------------------------------------------------------------------------------------
// builder state
// ---------------------------------------------------------------------------------------------------------------

struct Piece {
    std::string lit;
    std::string name;  // variable name (mux.Vars key)
    bool has_var = false;
    uint32_t cls[8] = {0};
    int min_rep = 1;
    int max_rep = 0;       // 0 = unbounded
    int var_idx = 0;       // which variable of the template this atom belongs to
    bool var_first = true, var_last = true;  // first / last atom of its variable (a {name:regexp} may be several atoms)
};

struct RouteDef {
    uint32_t method;
    std::string pattern;
    bool prefix = false, dead = false, is_default = false;  // is_default: appended by gofr_table_add_default_routes
    std::vector<Piece> pieces;
    uint32_t hkind = 0, schema_id = 0;
    std::string s[4];
    std::string blob;
};

struct FieldDef {
    std::string go_name, json_name;
    uint8_t kind;
    bool omitempty;
    uint8_t container = GOFR_C_VALUE, flags = 0;
    int elem = -1;  // GOFR_F_STRUCT: index of the struct's schema in gofr_table::schemas (always smaller than this one's)
};
struct SchemaDef {
    uint32_t id;
    std::string go_type;
    std::vector<FieldDef> fields;
    uint32_t fixed_words = 0;  // words of the fixed part of a row (include/gofr_b200.h "Row format")
    int depth = 1;             // struct nesting below this type, this one included
    bool flat = true;          // int / bool / string fields by value only: what the op programs of round 1 take
    bool bindable = true;      // the same plus float64: what Bind takes
    bool bare() const { return fields.size() == 1 && (fields[0].flags & GOFR_FIELD_BARE); }
};
static uint32_t kind_words(uint8_t kind) { return kind == GOFR_F_TIME ? 4u : (kind == GOFR_F_INT64 || kind == GOFR_F_INT || kind == GOFR_F_FLOAT64 || kind == GOFR_F_UINT64) ? 2u : 1u; }
// words a field owns in the fixed part of its struct
static uint32_t field_words(const std::vector<SchemaDef>& all, const FieldDef& f) {
    if (f.container == GOFR_C_SLICE || f.container == GOFR_C_MAP || f.container == GOFR_C_SLICE_PTR) return 1;
    const uint32_t w = f.kind == GOFR_F_STRUCT ? all[(size_t)f.elem].fixed_words : kind_words(f.kind);
    return w + (f.container == GOFR_C_PTR ? 1u : 0u);
}

// symbolic op before literal-pool assignment
struct SOp {
    uint8_t code;
    uint8_t arg = 0, flags = 0, kind = 0;
    uint32_t aux = 0, off = 0;
    std::string lit;  // OP_LIT / OP_KEY
    bool body = false;
    std::vector<uint32_t> date_pos;  // offsets inside `lit` of 29-byte Date placeholders
};

struct Prog {
    int status = 200;
    bool bind = false;
    int row_words = 0;  // see ProgRec::row_words
    int encfail = -1;   // see ProgRec::encfail
    std::vector<SOp> ops;
};

}  // namespace gofr

using namespace gofr;

struct gofr_table {
    uint32_t frame_mode = 0;
    bool sealed = false;
    bool has_catchall = false;
    std::vector<RouteDef> routes;
    std::vector<SchemaDef> schemas;
    std::vector<uint8_t> image;
};

namespace gofr {

static void cls_set(uint32_t* c, int b) { c[b >> 5] |= 1u << (b & 31); }
static void cls_range(uint32_t* c, int a, int b) { for (int x = a; x <= b; x++) cls_set(c, x); }

// {name:regexp}: a CONCATENATION of quantified units — no alternation, no groups, no anchors, no lazy quantifiers:
//   unit   a bracket class, \d, \w, '.', an escaped metacharacter (\. \- ...) or a plain literal character
//   quant  none, + * ? {n} {n,} {n,m}  (n, m <= 250)
// e.g. [0-9]+   \d{4}-\d{2}   v[0-9]+   [a-z]+\.[a-z]{2,4}   .*
// Each unit becomes one atom (class, min, max) matched greedily with backtracking: what Go's regexp (leftmost-first)
// reports for such a pattern.  Classes are sets of BYTES while Go counts runes: a counted quantifier ({n}, {n,m}, ?) on a
// class that contains non-ASCII bytes ('.', negated classes) would count differently for multi-byte characters and is
// refused; + and * do not care.
struct Atom {
    uint32_t cls[8] = {0};
    int min_rep = 1, max_rep = 0;  // max 0 = unbounded
};
static int parse_var_regexp(const std::string& re, std::vector<Atom>& out) {
    const size_t n = re.size();
    size_t i = 0;
    auto add_esc = [&](uint32_t* c, int e) {
        if (e == 'd') cls_range(c, '0', '9');
        else if (e == 'w') { cls_range(c, '0', '9'); cls_range(c, 'a', 'z'); cls_range(c, 'A', 'Z'); cls_set(c, '_'); }
        else cls_set(c, e);
    };
    while (i < n) {
        Atom at;
        bool ascii_only = true;
        const int ch = (uint8_t)re[i];
        if (ch == '[') {
            bool neg = false, first = true;
            i++;
            if (i < n && re[i] == '^') { neg = true; i++; }
            while (i < n && (re[i] != ']' || first)) {
                int a = (uint8_t)re[i];
                if (a == '[' && i + 1 < n && re[i + 1] == ':') return GOFR_ERR_UNSUPPORTED;  // [[:alpha:]]
                if (a == '\\') {
                    if (i + 1 >= n) return GOFR_ERR_UNSUPPORTED;
                    int e = (uint8_t)re[i + 1];
                    if (e == 'd' || e == 'w') { add_esc(at.cls, e); i += 2; first = false; continue; }
                    if ((e >= '0' && e <= '9') || (e >= 'a' && e <= 'z') || (e >= 'A' && e <= 'Z')) return GOFR_ERR_UNSUPPORTED;  // \s \pL \x41 ...
                    a = e;
                    i++;
                }
                if (a >= 0x80) return GOFR_ERR_UNSUPPORTED;
                if (i + 2 < n && re[i + 1] == '-' && re[i + 2] != ']') {
                    int b2 = (uint8_t)re[i + 2];
                    if (b2 == '\\') { if (i + 3 >= n) return GOFR_ERR_UNSUPPORTED; b2 = (uint8_t)re[i + 3]; i++; }
                    if (b2 >= 0x80 || b2 < a) return GOFR_ERR_UNSUPPORTED;
                    cls_range(at.cls, a, b2);
                    i += 3;
                } else { cls_set(at.cls, a); i++; }
                first = false;
            }
            if (i >= n) return GOFR_ERR_UNSUPPORTED;
            i++;  // ']'
            if (neg) { for (auto& w : at.cls) w = ~w; ascii_only = false; }
        } else if (ch == '\\') {
            if (i + 1 >= n) return GOFR_ERR_UNSUPPORTED;
            const int e = (uint8_t)re[i + 1];
            if (e == 'd' || e == 'w') add_esc(at.cls, e);
            else if ((e >= '0' && e <= '9') || (e >= 'a' && e <= 'z') || (e >= 'A' && e <= 'Z') || e >= 0x80) return GOFR_ERR_UNSUPPORTED;
            else cls_set(at.cls, e);  // an escaped punctuation character stands for itself
            i += 2;
        } else if (ch == '.') {
            for (auto& w : at.cls) w = 0xFFFFFFFFu;
            at.cls[0] &= ~(1u << '\n');
            ascii_only = false;
            i++;
        } else if (ch == '(' || ch == ')' || ch == '|' || ch == '^' || ch == '$' || ch == '+' || ch == '*' || ch == '?' || ch == '{' || ch == '}' ||
                   ch == ']') {
            return GOFR_ERR_UNSUPPORTED;  // groups, alternation, anchors; a quantifier without a unit
        } else {
            cls_set(at.cls, ch);  // a literal byte (the bytes of a multi-byte character are consecutive atoms)
            if (ch >= 0x80) ascii_only = false;
            i++;
        }
        // quantifier
        bool counted = false;
        if (i < n && re[i] == '+') { at.min_rep = 1; at.max_rep = 0; i++; }
        else if (i < n && re[i] == '*') { at.min_rep = 0; at.max_rep = 0; i++; }
        else if (i < n && re[i] == '?') { at.min_rep = 0; at.max_rep = 1; i++; counted = true; }
        else if (i < n && re[i] == '{') {
            size_t j = i + 1;
            auto num = [&](int& v) { if (j >= n || re[j] < '0' || re[j] > '9') return false; v = 0; while (j < n && re[j] >= '0' && re[j] <= '9') { v = v * 10 + (re[j] - '0'); if (v > 250) return false; j++; } return true; };
            int lo = 0, hi = 0;
            if (!num(lo)) return GOFR_ERR_UNSUPPORTED;
            if (j < n && re[j] == '}') hi = lo;
            else if (j < n && re[j] == ',') {
                j++;
                if (j < n && re[j] == '}') hi = 0;  // {n,}
                else { if (!num(hi) || hi < lo) return GOFR_ERR_UNSUPPORTED; if (hi == 0) return GOFR_ERR_UNSUPPORTED; }
            } else return GOFR_ERR_UNSUPPORTED;
            if (j >= n || re[j] != '}') return GOFR_ERR_UNSUPPORTED;
            if (hi == 0 && lo == 0 && re[j - 1] != ',') return GOFR_ERR_UNSUPPORTED;  // {0}: matches nothing but the empty string
            at.min_rep = lo; at.max_rep = hi;
            counted = !(hi == 0);  // {n,} only needs "at least n" — still a count of runes when n > 1
            if (hi == 0 && lo > 1) counted = true;
            i = j + 1;
        } else { at.min_rep = 1; at.max_rep = 1; counted = false; }  // exactly one: one rune; for non-ASCII classes see below
        if (i < n && (re[i] == '?' || re[i] == '+' || re[i] == '*' || re[i] == '{')) return GOFR_ERR_UNSUPPORTED;  // lazy / possessive / stacked
        // a byte of a multi-byte literal character: a quantifier after it would apply to the whole character in Go
        if (ch >= 0x80 && !(at.min_rep == 1 && at.max_rep == 1)) return GOFR_ERR_UNSUPPORTED;
        // exactly-one of a class with non-ASCII members matches one RUNE in Go, one byte here
        if (!ascii_only && (counted || (at.min_rep == 1 && at.max_rep == 1 && ch != '\\' && (ch == '.' || ch == '[')))) return GOFR_ERR_UNSUPPORTED;
        out.push_back(at);
        if (out.size() > 12) return GOFR_ERR_UNSUPPORTED;
    }
    return out.empty() ? GOFR_ERR_UNSUPPORTED : GOFR_OK;
}

// mux newRouteRegexp: literal text between top-level {...}; returns GOFR_OK, GOFR_ERR_UNSUPPORTED, or -1 for a
// template mux itself rejects (the route then exists but never matches).
static int parse_template(const std::string& tpl, std::vector<Piece>& out) {
    size_t n = tpl.size(), i = 0;
    int n_vars = 0;
    for (;;) {
        size_t j = i;
        while (j < n && tpl[j] != '{' && tpl[j] != '}') j++;
        if (j < n && tpl[j] == '}') return -1;
        Piece pc;
        pc.lit = tpl.substr(i, j - i);
        if (j >= n) { out.push_back(pc); break; }
        int depth = 0;
        size_t k = j;
        for (; k < n; k++) {
            if (tpl[k] == '{') depth++;
            else if (tpl[k] == '}' && --depth == 0) break;
        }
        if (k >= n) return -1;
        std::string body = tpl.substr(j + 1, k - j - 1);
        size_t colon = body.find(':');
        std::string name = colon == std::string::npos ? body : body.substr(0, colon);
        if (name.empty()) return -1;
        pc.has_var = true;
        pc.name = name;
        for (auto& prev : out) if (prev.has_var && prev.name == name) return -1;  // mux: duplicated route variable
        if (colon == std::string::npos) {
            for (auto& w : pc.cls) w = 0xFFFFFFFFu;
            pc.cls['/' >> 5] &= ~(1u << ('/' & 31));
            pc.min_rep = 1;
        } else {
            std::string re = body.substr(colon + 1);
            if (re.empty()) return -1;
            std::vector<Atom> atoms;
            int rc = parse_var_regexp(re, atoms);
            if (rc != GOFR_OK) return rc;
            // the first atom follows the piece's literal; the others are pieces with an empty literal
            for (size_t ai = 0; ai < atoms.size(); ai++) {
                Piece ap = ai == 0 ? pc : Piece();
                ap.has_var = true;
                ap.name = name;
                memcpy(ap.cls, atoms[ai].cls, sizeof ap.cls);
                ap.min_rep = atoms[ai].min_rep;
                ap.max_rep = atoms[ai].max_rep;
                ap.var_idx = n_vars;
                ap.var_first = ai == 0;
                ap.var_last = ai + 1 == atoms.size();
                out.push_back(ap);
            }
            n_vars++;
            i = k + 1;
            if (n_vars > kMaxVars || (int)out.size() > kMaxPieces) return GOFR_ERR_UNSUPPORTED;
            continue;
        }
        pc.var_idx = n_vars++;
        out.push_back(pc);
        i = k + 1;
        if (n_vars > kMaxVars || (int)out.size() > kMaxPieces) return GOFR_ERR_UNSUPPORTED;
    }
    return GOFR_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// program construction
// ---------------------------------------------------------------------------------------------------------------

struct HeaderKV { std::string k, v; bool hexid = false; };

enum BodyKind { BODY_NONE, BODY_JSON, BODY_FILE, BODY_PLAIN404, BODY_PANIC,
                BODY_JSON_FAILED };  // Respond set its Content-Type, then json.Encoder.Encode failed: no body bytes

static SOp lit(const std::string& s, bool body) { SOp o; o.code = OP_LIT; o.lit = s; o.body = body; return o; }
static SOp op(uint8_t code, bool body) { SOp o; o.code = code; o.body = body; return o; }

// The header block net/http 1.21 writes (chunkWriter.writeHeader + Header.WriteSubset + extraHeader.Write).
//   handler headers sorted by key; then Date, Content-Length, Content-Type (sniffed only if the handler's snapshot has
//   none and the body is non-empty).  `with_mw`: the Tracer/Logging/CORS chain ran (a route matched).
// `chunked`: the body is ONE Write of more than 2048 bytes — it bypasses response.w (a 2 KiB bufio.Writer) and reaches
// chunkWriter.Write while the handler is still running, so writeHeader knows no Content-Length and an HTTP/1.1 response
// becomes "Transfer-Encoding: chunked" (extraHeader order: Date, Content-Length, Content-Type, Connection, Transfer-Encoding).
static void build_header(Prog& p, uint32_t frame_mode, int status, bool with_mw, BodyKind bk, bool head_no_body,
                         const std::string& file_ct_given, const std::string& file_ct_sniffed, bool location, bool chunked = false) {
    if (frame_mode == GOFR_FRAME_BODY) return;
    std::vector<HeaderKV> h;
    if (with_mw) {
        HeaderKV id; id.k = "X-Correlation-Id"; id.hexid = true;  // Header.Set canonicalises X-Correlation-ID
        h.push_back(id);
        h.push_back({"Access-Control-Allow-Origin", "*"});
        h.push_back({"Access-Control-Allow-Methods", "POST, GET, OPTIONS, PUT, DELETE"});
    }
    bool have_type = false;
    if (bk == BODY_PLAIN404) {  // http.Error sets both before WriteHeader
        h.push_back({"Content-Type", "text/plain; charset=utf-8"});
        h.push_back({"X-Content-Type-Options", "nosniff"});
        have_type = true;
    }
    if (frame_mode == GOFR_FRAME_INTENDED) {
        // what the tests read from the live recorder map: the late Header().Set is visible
        if (bk == BODY_JSON || bk == BODY_JSON_FAILED) { h.push_back({"Content-Type", "application/json"}); have_type = true; }
        if (bk == BODY_FILE) { h.push_back({"Content-Type", file_ct_given}); have_type = true; }
    }
    std::sort(h.begin(), h.end(), [](const HeaderKV& a, const HeaderKV& b) { return a.k < b.k; });
    std::string acc = std::string("HTTP/1.1 ") + std::to_string(status) + " " + status_text(status) + "\r\n";
    if (location) {
        // Location sorts among the handler headers; a 301 carries no others
        acc += "Location: ";
        p.ops.push_back(lit(acc, false));
        p.ops.push_back(op(OP_LOCATION, false));
        acc = "\r\n";
    }
    for (auto& kv : h) {
        acc += kv.k + ": ";
        if (kv.hexid) {
            p.ops.push_back(lit(acc, false));
            p.ops.push_back(op(OP_HEXID, false));
            acc.clear();
        } else acc += kv.v;
        acc += "\r\n";
    }
    acc += "Date: ";
    {
        // the batch's Date is patched into the shared-memory copy of the literal pool at kernel start (fixup)
        SOp d = lit(acc + std::string(29, '\0'), false);
        d.date_pos.push_back((uint32_t)acc.size());
        p.ops.push_back(d);
    }
    acc = "\r\n";
    bool body_nonempty = bk != BODY_NONE && bk != BODY_JSON_FAILED;
    if (!head_no_body && !chunked) {
        acc += "Content-Length: ";
        if (body_nonempty) {
            p.ops.push_back(lit(acc, false));
            p.ops.push_back(op(OP_CLEN, false));
            acc = "\r\n";
        } else acc += "0\r\n";
    }
    if (!have_type && body_nonempty) {
        acc += "Content-Type: ";
        acc += bk == BODY_FILE ? file_ct_sniffed : "text/plain; charset=utf-8";  // JSON text never sniffs as anything else
        acc += "\r\n";
    }
    if (chunked) acc += "Transfer-Encoding: chunked\r\n";
    acc += "\r\n";
    p.ops.push_back(lit(acc, false));
}

// struct → JSON object ops.  Levels without omitempty collapse to literals around value ops; plain nested structs of
// such levels are flattened into the same op list (their words are inline in the parent's fixed part and their strings
// follow in field order, so nothing distinguishes them from the parent's own fields).  Everything whose shape depends on
// the row — pointers, slices, maps, nested structs with omitempty members — is ONE OP_VALUE op: the device walks it with the
// generic encoder (serve_device.cuh value_encode).
static bool flattenable(const std::vector<SchemaDef>& all, const SchemaDef& sc) {
    if (sc.bare()) return false;
    for (auto& f : sc.fields) {
        if (f.container != GOFR_C_VALUE || f.omitempty) return false;
        if (f.kind == GOFR_F_STRUCT && !flattenable(all, all[(size_t)f.elem])) return false;
    }
    return true;
}
static SOp value_op(int schema_idx, size_t field_idx, uint16_t word) {
    SOp v;
    v.code = OP_VALUE; v.body = true; v.off = word; v.aux = (uint32_t)schema_idx; v.arg = (uint8_t)field_idx;
    return v;
}
static void struct_level_ops(Prog& p, const std::vector<SchemaDef>& all, int sidx, bool bind_layout, uint16_t& word,
                             uint16_t& str_ord, std::string& acc) {
    const SchemaDef& sc = all[(size_t)sidx];
    if (sc.bare()) {  // the schema IS its one field's type: no braces, no key
        if (!acc.empty()) { p.ops.push_back(lit(acc, true)); acc.clear(); }
        p.ops.push_back(value_op(sidx, 0, word));
        word = (uint16_t)(word + field_words(all, sc.fields[0]));
        return;
    }
    bool dynamic = false;
    for (auto& f : sc.fields) dynamic |= f.omitempty;
    acc += "{";
    bool first = true;
    for (size_t fi = 0; fi < sc.fields.size(); fi++) {
        const FieldDef& f = sc.fields[fi];
        std::string key = "\"" + json_escape_go(f.json_name) + "\":";
        uint16_t w = word;
        if (bind_layout) {  // span row (bind_device.cuh): 8 header words, strings are (offset, length) pairs
            w = (uint16_t)(8 + word);
            word += (f.kind == GOFR_F_INT32 || f.kind == GOFR_F_BOOL) ? 1 : 2;
        } else word = (uint16_t)(word + field_words(all, f));
        const bool plain = f.container == GOFR_C_VALUE;
        const bool is_str = plain && f.kind == GOFR_F_STRING;
        SOp v;
        v.body = true;
        v.off = w;
        bool generic = !plain;
        if (plain) switch (f.kind) {
            case GOFR_F_INT64: case GOFR_F_INT: v.code = OP_I64; break;
            case GOFR_F_INT32: v.code = OP_I32; break;
            case GOFR_F_BOOL: v.code = OP_BOOL; break;
            case GOFR_F_FLOAT64: v.code = OP_F64; break;
            case GOFR_F_STRING: v.code = bind_layout ? OP_BSTR : OP_STR; v.arg = (uint8_t)str_ord++; break;
            default: generic = true; break;  // GOFR_F_STRUCT
        }
        if (!dynamic) {
            if (!first) acc += ",";
            acc += key;
            if (plain && f.kind == GOFR_F_STRUCT && flattenable(all, all[(size_t)f.elem])) {
                uint16_t sub_word = w;
                struct_level_ops(p, all, f.elem, false, sub_word, str_ord, acc);
            } else {
                if (is_str) acc += "\"";
                p.ops.push_back(lit(acc, true));
                p.ops.push_back(generic ? value_op(sidx, fi, w) : v);
                acc = is_str ? "\"" : "";
            }
        } else {
            if (!acc.empty()) { p.ops.push_back(lit(acc, true)); acc.clear(); }
            SOp k;
            k.code = OP_KEY; k.body = true; k.kind = (uint8_t)(f.kind | f.container << 4); k.off = w; k.lit = key;
            k.flags = f.omitempty ? OPF_OMITEMPTY : 0;
            if (is_str) k.lit += "\"";
            p.ops.push_back(k);
            if (generic) v = value_op(sidx, fi, w);
            v.flags |= OPF_VALUE_OF_KEY;
            p.ops.push_back(v);
            if (is_str) { SOp q = lit("\"", true); q.flags |= OPF_VALUE_OF_KEY; p.ops.push_back(q); }
        }
        first = false;
    }
    acc += "}";
}
static void build_struct_ops(Prog& p, const std::vector<SchemaDef>& all, const SchemaDef& sc, bool bind_layout = false,
                             uint16_t word_base = 0) {
    uint16_t word = word_base, str_ord = word_base ? 1 : 0;
    std::string acc;
    struct_level_ops(p, all, (int)(&sc - all.data()), bind_layout, word, str_ord, acc);
    p.ops.push_back(lit(acc, true));
}

struct Builder {
    gofr_table* t;
    std::vector<Prog> progs;
    std::string err;

    std::map<std::string, int> prog_ids;
    // identical programs (e.g. sixteen routes returning the same struct type) are stored once
    int add(Prog p) {
        // a program that can meet a NaN / Inf float gets a companion for "json.Encoder.Encode failed": same status and
        // headers, no body bytes (ProgRec::encfail)
        bool may_fail = false;
        for (auto& o : p.ops) may_fail |= o.code == OP_F64 || o.code == OP_VALUE;
        if (may_fail && p.encfail < 0) {
            Prog q;
            q.status = p.status;
            build_header(q, t->frame_mode, p.status, true, BODY_JSON_FAILED, false, "", "", false);
            p.encfail = add(std::move(q));
        }
        std::string sig = std::to_string(p.status) + (p.bind ? "B" : "R") + std::to_string(p.row_words);
        for (auto& o : p.ops) {
            sig += "|" + std::to_string(o.code) + "," + std::to_string(o.arg) + "," + std::to_string(o.flags) + "," +
                   std::to_string(o.kind) + "," + std::to_string(o.off) + "," + std::to_string(o.aux) + "," +
                   (o.body ? "b" : "h") + std::to_string(o.lit.size()) + ":" + o.lit;
            for (uint32_t d : o.date_pos) sig += "@" + std::to_string(d);
        }
        auto it = prog_ids.find(sig);
        if (it != prog_ids.end()) return it->second;
        progs.push_back(std::move(p));
        prog_ids[sig] = (int)progs.size() - 1;
        return (int)progs.size() - 1;
    }

    // Responder.Respond envelope: {"error":{"message":...},"data":...}\n  (error first; both omitempty)
    int json_prog(int status, const std::vector<SOp>& body_ops, bool bind = false) {
        Prog p;
        p.status = status;
        p.bind = bind;
        // a body that is all literals has its length now: beyond net/http's 2 KiB buffer the one Write of Encoder.Encode makes the
        // response chunked (see build_header) — decided here for static bodies; bodies whose length depends on the request keep
        // Content-Length whatever their size (DESIGN.md §8, a stated deviation)
        size_t static_len = 0;
        bool all_static = true;
        for (auto& o : body_ops) { all_static &= o.code == OP_LIT && !(o.flags & OPF_VALUE_OF_KEY); static_len += o.lit.size(); }
        const bool chunked = all_static && t->frame_mode == GOFR_FRAME_WIRE && static_len > 2048;
        build_header(p, t->frame_mode, status, true, BODY_JSON, false, "", "", false, chunked);
        if (chunked) {
            char hx[32];
            snprintf(hx, sizeof hx, "%zx\r\n", static_len);
            p.ops.push_back(lit(hx, true));
        }
        for (auto o : body_ops) { o.body = true; p.ops.push_back(o); }
        if (chunked) p.ops.push_back(lit("\r\n0\r\n\r\n", true));
        return add(std::move(p));
    }
};

}  // namespace gofr

// ---------------------------------------------------------------------------------------------------------------
// image assembly
// ---------------------------------------------------------------------------------------------------------------

namespace gofr {

struct Pool {
    std::vector<uint8_t>& img;
    std::map<std::string, uint32_t> seen;
    explicit Pool(std::vector<uint8_t>& i) : img(i) {}
    uint32_t put(const std::string& s, bool dated = false) {  // 4-byte aligned, zero padded to a word (+4 slack)
        std::string key = (dated ? "D" : "L") + s;
        auto it = seen.find(key);
        if (it != seen.end()) return it->second;
        while (img.size() % 4) img.push_back(0);
        uint32_t off = (uint32_t)img.size();
        img.insert(img.end(), s.begin(), s.end());
        while (img.size() % 4) img.push_back(0);
        for (int k = 0; k < 4; k++) img.push_back(0);
        seen[key] = off;
        return off;
    }
    // 16-byte aligned, never shared (response templates: read with aligned 128-bit loads)
    uint32_t put16(const std::string& s) {
        while (img.size() % 16) img.push_back(0);
        uint32_t off = (uint32_t)img.size();
        img.insert(img.end(), s.begin(), s.end());
        while (img.size() % 16) img.push_back(0);
        return off;
    }
};

static void merge_literals(std::vector<SOp>& ops) {
    std::vector<SOp> out;
    for (auto& o : ops) {
        if (o.code == OP_LIT && o.lit.empty()) continue;
        if (o.code == OP_LIT && !out.empty() && out.back().code == OP_LIT && out.back().body == o.body &&
            out.back().flags == o.flags) {
            for (uint32_t dp : o.date_pos) out.back().date_pos.push_back(dp + (uint32_t)out.back().lit.size());
            out.back().lit += o.lit;
        } else out.push_back(o);
    }
    ops.swap(out);
}

// A body made of literals only has a Content-Length known at seal time: the digits become part of the header literal, and
// the whole response becomes position-fixed (one template for the slot-layout kernel, table_format.h FastRec).
static void fold_static_clen(std::vector<SOp>& ops) {
    size_t body = 0;
    for (auto& o : ops) {
        if (!o.body) continue;
        if (o.code != OP_LIT || o.flags) return;  // a value, a blob or a governed literal: length not static
        body += o.lit.size();
    }
    for (auto& o : ops)
        if (o.code == OP_CLEN) { o.code = OP_LIT; o.lit = std::to_string(body); }
}

// LIT followed by a value op of the same part (header/body) → the literal becomes the value op's prefix
static bool op_takes_prefix(uint8_t code) {
    return code == OP_HEXID || code == OP_CLEN || code == OP_I64 || code == OP_I32 || code == OP_BOOL || code == OP_STR ||
           code == OP_BSTR || code == OP_PARAM || code == OP_LOCATION || code == OP_ERRMSG || code == OP_F64;
}
static void fold_prefixes(std::vector<SOp>& ops) {
    std::vector<SOp> out;
    for (size_t i = 0; i < ops.size(); i++) {
        if (ops[i].code == OP_LIT && ops[i].flags == 0 && i + 1 < ops.size() && op_takes_prefix(ops[i + 1].code) &&
            ops[i + 1].flags == 0 && ops[i + 1].body == ops[i].body && ops[i + 1].lit.empty()) {
            SOp v = ops[i + 1];
            v.lit = ops[i].lit;            // prefix bytes
            v.date_pos = ops[i].date_pos;
            out.push_back(v);
            i++;
        } else out.push_back(ops[i]);
    }
    ops.swap(out);
}

static const char* go_kind_name(uint8_t k) {
    switch (k) {
        case GOFR_F_INT64: return "int64";
        case GOFR_F_INT32: return "int32";
        case GOFR_F_BOOL: return "bool";
        case GOFR_F_STRING: return "string";
        case 5: return "int";
        case GOFR_F_FLOAT64: return "float64";
        case GOFR_F_STRUCT: return "struct";
        case GOFR_F_UINT64: return "uint64";
        case GOFR_F_BYTES: return "[]uint8";
        case GOFR_F_FLOAT32: return "float32";
        case GOFR_F_TIME: return "time.Time";
    }
    return "?";
}

static std::string fold_lower(const std::string& s) {
    std::string r = s;
    for (auto& c : r) if (c >= 'A' && c <= 'Z') c = (char)(c + 32);
    return r;
}

int seal_table(gofr_table* t) {
    Builder b{t, {}, {}};
    uint32_t fm = t->frame_mode;

    // ---- fixed programs (mux / middleware outcomes that exist for every table) ----
    auto simple = [&](int status, bool with_mw, BodyKind bk, bool head_no_body, bool location, const std::string& body) {
        Prog p;
        p.status = status;
        build_header(p, fm, status, with_mw, bk, head_no_body, "", "", location);
        if (!body.empty()) p.ops.push_back(lit(body, true));
        return b.add(std::move(p));
    };
    int p301 = simple(301, false, BODY_NONE, false, true, "");
    int p301h = simple(301, false, BODY_NONE, true, true, "");
    int p404 = simple(404, false, BODY_PLAIN404, false, false, "404 page not found\n");  // http.NotFoundHandler
    int p405 = simple(405, false, BODY_NONE, false, false, "");                           // mux methodNotAllowedHandler
    int p405h = simple(405, false, BODY_NONE, true, false, "");
    int popt = simple(200, true, BODY_NONE, false, false, "");                            // CORS short-circuit
    int ppanic = simple(500, true, BODY_PANIC, false, false,
                        "{\"code\":500,\"message\":\"Some unexpected error has occurred\",\"status\":\"ERROR\"}\n");

    // ---- per-route programs ----
    std::vector<int> prog_ok(t->routes.size(), 0xFFFF), prog_err(t->routes.size(), 0xFFFF);
    std::vector<int> prog_err404(t->routes.size(), 0xFFFF), prog_nil(t->routes.size(), 0xFFFF), prog_both(t->routes.size(), 0xFFFF),
        prog_str(t->routes.size(), 0xFFFF);
    std::vector<uint16_t> rawprogs(t->routes.size() * 9, 0xFFFF);  // response.Raw outcomes of GOFR_H_RESULT routes
    for (size_t ri = 0; ri < t->routes.size(); ri++) {
        RouteDef& r = t->routes[ri];
        const SchemaDef* sc = nullptr;
        if (r.hkind == GOFR_H_ROW || r.hkind == GOFR_H_BIND_ECHO || r.hkind == GOFR_H_RESULT) {
            for (auto& s : t->schemas) if (s.id == r.schema_id) sc = &s;
            // a closure that only ever returns strings / errors / nil needs no struct schema
            if (!sc && !(r.hkind == GOFR_H_RESULT && r.schema_id == 0)) { set_last_error("route %s: unknown schema %u", r.pattern.c_str(), r.schema_id); return GOFR_ERR_INVALID; }
            if (sc && r.hkind == GOFR_H_BIND_ECHO && !sc->bindable) {
                set_last_error("route %s: Bind takes flat structs of int / float64 / bool / string fields only (schema %u)", r.pattern.c_str(), r.schema_id);
                return GOFR_ERR_UNSUPPORTED;
            }
        }
        switch (r.hkind) {
            case GOFR_H_HOST: break;
            case GOFR_H_STATIC_STRING:
                prog_ok[ri] = b.json_prog(200, {lit("{\"data\":\"" + json_escape_go(r.s[0]) + "\"}\n", true)});
                break;
            case GOFR_H_STATIC_ERROR:
                prog_ok[ri] = b.json_prog(500, {lit("{\"error\":{\"message\":\"" + json_escape_go(r.s[0]) + "\"}}\n", true)});
                break;
            case GOFR_H_NIL: prog_ok[ri] = b.json_prog(200, {lit("{}\n", true)}); break;
            case GOFR_H_HEALTH: prog_ok[ri] = b.json_prog(200, {lit("{\"data\":{}}\n", true)}); break;
            case GOFR_H_MISSING_FILE:
                prog_ok[ri] = b.json_prog(404, {lit("{\"error\":{\"message\":\"http: no such file\"}}\n", true)});
                break;
            case GOFR_H_PANIC: prog_ok[ri] = ppanic; break;
            case GOFR_H_PATHPARAM_FORMAT:
            case GOFR_H_PARAM_FORMAT: {
                if (!valid_utf8(r.s[2]) || !valid_utf8(r.s[3])) {
                    set_last_error("route %s: format prefix/suffix must be valid UTF-8", r.pattern.c_str());
                    return GOFR_ERR_UNSUPPORTED;
                }
                prog_ok[ri] = b.json_prog(200, {lit("{\"data\":\"" + json_escape_go(r.s[2]), true), op(OP_PARAM, true),
                                                lit(json_escape_go(r.s[3]) + "\"}\n", true)});
                break;
            }
            case GOFR_H_ROW:
            case GOFR_H_BIND_ECHO: {
                Prog p;
                p.status = 200;
                build_header(p, fm, 200, true, BODY_JSON, false, "", "", false);
                p.ops.push_back(lit("{\"data\":", true));
                build_struct_ops(p, t->schemas, *sc, r.hkind == GOFR_H_BIND_ECHO);
                p.ops.push_back(lit("}\n", true));
                p.bind = r.hkind == GOFR_H_BIND_ECHO;
                prog_ok[ri] = b.add(std::move(p));
                if (r.hkind == GOFR_H_BIND_ECHO)
                    prog_err[ri] = b.json_prog(500, {lit("{\"error\":{\"message\":\"", true), op(OP_ERRMSG, true),
                                                     lit("\"}}\n", true)}, true);
                break;
            }
            case GOFR_H_RESULT: {
                // Responder.Respond on a (data, err) the host closure produced (responder.go:19-62)
                if (sc) {
                    Prog p;
                    p.status = 200;
                    build_header(p, fm, 200, true, BODY_JSON, false, "", "", false);
                    p.ops.push_back(lit("{\"data\":", true));
                    build_struct_ops(p, t->schemas, *sc, false);
                    p.ops.push_back(lit("}\n", true));
                    prog_ok[ri] = b.add(std::move(p));
                }
                {   // data is a string: {"data":"…"} (encoding/json string escaping, as for struct fields)
                    Prog p;
                    p.status = 200;
                    build_header(p, fm, 200, true, BODY_JSON, false, "", "", false);
                    p.ops.push_back(lit("{\"data\":\"", true));
                    SOp m = op(OP_STR, true);
                    m.off = 0;  // row word 0 = len, the bytes follow
                    p.ops.push_back(m);
                    p.ops.push_back(lit("\"}\n", true));
                    p.row_words = 1;
                    prog_str[ri] = b.add(std::move(p));
                }
                for (int which = 0; which < 2; which++) {  // 500, and 404 for errors.Is(err, http.ErrMissingFile)
                    Prog e;
                    e.status = which ? 404 : 500;
                    build_header(e, fm, e.status, true, BODY_JSON, false, "", "", false);
                    e.ops.push_back(lit("{\"error\":{\"message\":\"", true));
                    SOp m = op(OP_STR, true);
                    m.off = 0;  // row word 0 = len(err.Error()), the bytes follow
                    e.ops.push_back(m);
                    e.ops.push_back(lit("\"}}\n", true));
                    e.row_words = 1;
                    (which ? prog_err404 : prog_err)[ri] = b.add(std::move(e));
                }
                prog_nil[ri] = b.json_prog(200, {lit("{}\n", true)});
                // response.Raw{Data: …}: the data encoded bare (responder.go:24-26); the error only picks the status
                for (int es = 0; es < 3; es++) {
                    const int status = es == 0 ? 200 : es == 1 ? 500 : 404;
                    if (sc) {
                        Prog p;
                        p.status = status;
                        build_header(p, fm, status, true, BODY_JSON, false, "", "", false);
                        build_struct_ops(p, t->schemas, *sc, false);
                        p.ops.push_back(lit("\n", true));
                        rawprogs[ri * 9 + 0 + es] = (uint16_t)b.add(std::move(p));
                    }
                    {
                        Prog p;
                        p.status = status;
                        build_header(p, fm, status, true, BODY_JSON, false, "", "", false);
                        p.ops.push_back(lit("\"", true));
                        SOp m = op(OP_STR, true);
                        m.off = 0;
                        p.ops.push_back(m);
                        p.ops.push_back(lit("\"\n", true));
                        p.row_words = 1;
                        rawprogs[ri * 9 + 3 + es] = (uint16_t)b.add(std::move(p));
                    }
                    rawprogs[ri * 9 + 6 + es] = (uint16_t)b.json_prog(status, {lit("null\n", true)});
                }
                if (sc) {  // (data, err) both non-nil: response{Error, Data} with both members (responder.go:59-62)
                    Prog e;
                    e.status = 500;
                    build_header(e, fm, 500, true, BODY_JSON, false, "", "", false);
                    e.ops.push_back(lit("{\"error\":{\"message\":\"", true));
                    SOp m = op(OP_STR, true);
                    m.off = 0;
                    e.ops.push_back(m);
                    e.ops.push_back(lit("\"},\"data\":", true));
                    build_struct_ops(e, t->schemas, *sc, false, 1);
                    e.ops.push_back(lit("}\n", true));
                    e.row_words = (int)(1 + sc->fixed_words);
                    prog_both[ri] = b.add(std::move(e));
                }
                break;
            }
            case GOFR_H_FILE: {
                Prog p;
                p.status = 200;
                if (r.blob.empty()) {
                    // Write(nil) after WriteHeader: empty body → "Content-Length: 0" and nothing to sniff; the
                    // recorder's live map (INTENDED) still shows the type the handler set.
                    build_header(p, fm, 200, true, fm == GOFR_FRAME_INTENDED ? BODY_FILE : BODY_NONE, false, r.s[0], "", false);
                } else {
                    // w.Write(v.Content) is one Write: beyond net/http's 2 KiB buffer the response is chunked on the wire
                    // (the reference's own favicon, 13 149 bytes, is) — one chunk, then chunkWriter.close's terminator.
                    // (A HEAD request would get neither Content-Length nor Transfer-Encoding there; GoFr registers
                    // GET / PUT / POST / DELETE only, so no File route ever sees one.)
                    const bool chunked = fm == GOFR_FRAME_WIRE && r.blob.size() > 2048;
                    build_header(p, fm, 200, true, BODY_FILE, false, r.s[0], sniff_content_type(r.blob), false, chunked);
                    if (chunked) {
                        char hx[32];
                        snprintf(hx, sizeof hx, "%zx\r\n", r.blob.size());
                        p.ops.push_back(lit(hx, true));
                    }
                    SOp bo = op(OP_BLOB, true);
                    bo.lit = r.blob;
                    p.ops.push_back(bo);
                    if (chunked) p.ops.push_back(lit("\r\n0\r\n\r\n", true));
                }
                prog_ok[ri] = b.add(std::move(p));
                break;
            }
            default: set_last_error("route %s: unknown handler kind %u", r.pattern.c_str(), r.hkind); return GOFR_ERR_INVALID;
        }
    }

    // ---- lay out the image ----
    std::vector<uint8_t>& img = t->image;
    img.clear();
    img.resize(sizeof(ImageHeader), 0);
    ImageHeader H;
    memset(&H, 0, sizeof H);
    H.magic = kMagic; H.version = kImageVersion; H.frame_mode = fm;
    H.n_routes = (uint32_t)t->routes.size();
    H.prog_301 = (uint16_t)p301; H.prog_301_head = (uint16_t)p301h; H.prog_404 = (uint16_t)p404; H.prog_405 = (uint16_t)p405;
    H.prog_405_head = (uint16_t)p405h; H.prog_options = (uint16_t)popt; H.prog_panic = (uint16_t)ppanic;
    H.has_catchall = t->has_catchall;

    auto align16 = [&]() { while (img.size() % 16) img.push_back(0); };
    std::vector<RouteRec> routes(t->routes.size());
    std::vector<PieceRec> pieces;
    // We build sections into separate byte vectors, then concatenate.
    std::vector<uint8_t> lits;
    Pool pool(lits);
    std::vector<uint8_t> cold;

    for (size_t ri = 0; ri < t->routes.size(); ri++) {
        RouteDef& r = t->routes[ri];
        RouteRec& R = routes[ri];
        memset(&R, 0, sizeof R);
        R.method = (uint8_t)r.method;
        R.flags = (r.prefix ? RF_PREFIX : 0) | (r.dead ? RF_DEAD : 0) | (r.is_default ? RF_DEFAULT : 0);
        R.hkind = (uint8_t)r.hkind;
        R.first_piece = (uint16_t)pieces.size();
        R.n_pieces = (uint8_t)r.pieces.size();
        R.prog_ok = (uint16_t)prog_ok[ri];
        R.prog_err = (uint16_t)prog_err[ri];
        if (!r.dead && !r.prefix && r.pieces.size() == 1 && !r.pieces[0].has_var) {
            R.flags |= RF_LITERAL;
            R.lit_off = pool.put(r.pattern);
            R.lit_len = (uint16_t)r.pattern.size();
        }
        for (auto& pc : r.pieces) {
            PieceRec P;
            memset(&P, 0, sizeof P);
            P.lit_off = pool.put(pc.lit);
            P.lit_len = (uint16_t)pc.lit.size();
            P.has_var = pc.has_var;
            P.min_rep = (uint8_t)pc.min_rep;
            P.max_rep = (uint8_t)pc.max_rep;
            P.var_idx = (uint8_t)pc.var_idx;
            P.var_flags = (uint8_t)((pc.var_first ? PV_FIRST : 0) | (pc.var_last ? PV_LAST : 0));
            memcpy(P.cls, pc.cls, sizeof P.cls);
            pieces.push_back(P);
        }
        if (r.hkind == GOFR_H_PATHPARAM_FORMAT) {
            // mux.Vars(r)[s0]: resolved to the index of the variable; an unknown name always yields ""
            R.key_len = 0xFFFF;
            for (size_t k = 0; k < r.pieces.size(); k++)
                if (r.pieces[k].has_var && r.pieces[k].name == r.s[0]) R.key_len = (uint16_t)r.pieces[k].var_idx;
            R.def_off = pool.put("");
            R.def_len = 0;
        }
        if (r.hkind == GOFR_H_PARAM_FORMAT) {
            R.key_off = pool.put(r.s[0]);
            R.key_len = (uint16_t)r.s[0].size();
            std::string d = json_escape_go(r.s[1]);
            R.def_off = pool.put(d);
            R.def_len = (uint16_t)d.size();
        }
        if (r.hkind == GOFR_H_RESULT) {  // the two spare 16-bit fields carry the other outcomes' programs
            R.key_len = (uint16_t)prog_nil[ri];
            R.def_len = (uint16_t)prog_err404[ri];
            R.key_off = (uint32_t)prog_both[ri] | (uint32_t)prog_str[ri] << 16;
        }
        if (r.hkind == GOFR_H_ROW || r.hkind == GOFR_H_BIND_ECHO || r.hkind == GOFR_H_RESULT)
            for (size_t si = 0; si < t->schemas.size(); si++)
                if (t->schemas[si].id == r.schema_id) R.schema = (uint16_t)si;
    }

    // ---- literal-route dispatch structures ----
    uint32_t n_lit = 0;
    for (auto& R : routes) n_lit += (R.flags & RF_LITERAL) ? 1 : 0;
    uint32_t hash_bits = 4;
    while ((1u << hash_bits) < 4 * n_lit && hash_bits < 11) hash_bits++;
    std::vector<uint16_t> hash_tab(1u << hash_bits, 0xFFFF), tmpl_list, last_method(16, 0);
    // templates whose leading literal has at least 8 bytes are keyed by those bytes
    uint32_t n_keyed = 0;
    for (size_t ri = 0; ri < routes.size(); ri++)
        if (!(routes[ri].flags & (RF_DEAD | RF_LITERAL)) && !t->routes[ri].pieces.empty() && t->routes[ri].pieces[0].lit.size() >= 8) n_keyed++;
    uint32_t thash_bits = 4;
    while ((1u << thash_bits) < 4 * n_keyed && thash_bits < 11) thash_bits++;
    std::vector<uint16_t> thash_tab(1u << thash_bits, 0xFFFF);
    {
        std::vector<uint16_t> tail(1u << hash_bits, 0xFFFF), ttail(1u << thash_bits, 0xFFFF);
        for (size_t ri = 0; ri < routes.size(); ri++) {
            RouteRec& R = routes[ri];
            R.next_lit = 0xFFFF;
            if (R.flags & RF_DEAD) continue;
            if (R.method < 16) last_method[R.method] = (uint16_t)(ri + 1);
            if (!(R.flags & RF_LITERAL)) {
                const std::string& l0 = t->routes[ri].pieces.empty() ? std::string() : t->routes[ri].pieces[0].lit;
                if (l0.size() < 8) { tmpl_list.push_back((uint16_t)ri); continue; }
                uint32_t w0 = 0, w1 = 0;
                for (int k = 0; k < 4; k++) { w0 |= (uint32_t)(uint8_t)l0[k] << (8 * k); w1 |= (uint32_t)(uint8_t)l0[4 + k] << (8 * k); }
                uint32_t slot = path_hash_step(path_hash_step(8u, w0), w1) >> (32 - thash_bits);
                if (ttail[slot] == 0xFFFF) thash_tab[slot] = (uint16_t)ri; else routes[ttail[slot]].next_lit = (uint16_t)ri;
                ttail[slot] = (uint16_t)ri;
                continue;
            }
            const std::string& pat = t->routes[ri].pattern;
            uint32_t h = (uint32_t)pat.size();
            for (size_t i = 0; i < pat.size(); i += 4) {
                uint32_t w = 0;
                for (size_t k = 0; k < 4 && i + k < pat.size(); k++) w |= (uint32_t)(uint8_t)pat[i + k] << (8 * k);
                h = path_hash_step(h, w);
            }
            uint32_t slot = h >> (32 - hash_bits);
            if (tail[slot] == 0xFFFF) hash_tab[slot] = (uint16_t)ri; else routes[tail[slot]].next_lit = (uint16_t)ri;
            tail[slot] = (uint16_t)ri;
        }
    }

    std::vector<ProgRec> progs(b.progs.size());
    std::vector<Op> ops;
    std::vector<uint32_t> fixups;
    uint32_t max_fixed = 0;
    for (size_t pi = 0; pi < b.progs.size(); pi++) {
        Prog& p = b.progs[pi];
        fold_static_clen(p.ops);
        merge_literals(p.ops);
        fold_prefixes(p.ops);
        ProgRec& P = progs[pi];
        memset(&P, 0, sizeof P);
        P.first_op = (uint16_t)ops.size();
        P.n_ops = (uint16_t)p.ops.size();
        P.status = (uint16_t)p.status;
        P.row_words = (uint16_t)p.row_words;
        P.encfail = p.encfail >= 0 ? (uint16_t)p.encfail : (uint16_t)0xFFFF;
        if (p.bind) P.flags |= PF_BIND;
        for (auto& so : p.ops) {
            Op o;
            memset(&o, 0, sizeof o);
            o.code = so.code; o.arg = so.arg; o.kind = so.kind;
            o.flags = so.flags | (so.body ? OPF_BODY : 0);
            o.off = so.off; o.aux = so.aux;
            uint32_t fixed = 0;
            switch (so.code) {
                case OP_LIT:
                    o.off = pool.put(so.lit, !so.date_pos.empty());
                    o.len = (uint32_t)so.lit.size();
                    for (uint32_t dp : so.date_pos) fixups.push_back(o.off + dp);
                    if (!(so.flags & OPF_VALUE_OF_KEY)) fixed = o.len; else P.flags |= PF_DYNAMIC;
                    break;
                case OP_KEY:
                    o.aux = so.off;  // row word of the governed field
                    o.off = pool.put(so.lit);
                    o.len = (uint32_t)so.lit.size();
                    P.flags |= PF_DYNAMIC | PF_NEEDS_ROW;
                    if (so.kind > GOFR_F_INT) P.flags |= PF_VALUES;  // emptiness test of the wider kinds
                    break;
                case OP_HEXID: fixed = 32; break;
                case OP_CLEN: P.flags |= PF_HAS_CLEN; break;
                case OP_F64: case OP_VALUE: P.flags |= PF_VALUES;  // fall through
                case OP_I64: case OP_I32: case OP_BOOL: case OP_STR: case OP_BSTR:
                    P.flags |= PF_DYNAMIC | PF_NEEDS_ROW;
                    break;
                case OP_BLOB:
                    while (cold.size() % 16) cold.push_back(0);
                    o.off = (uint32_t)cold.size();
                    o.len = (uint32_t)so.lit.size();
                    cold.insert(cold.end(), so.lit.begin(), so.lit.end());
                    fixed = o.len;
                    break;
                default: P.flags |= PF_DYNAMIC; break;
            }
            if (op_takes_prefix(so.code) && !so.lit.empty()) {  // folded literal prefix
                o.aux = pool.put(so.lit, !so.date_pos.empty());
                o.len = (uint32_t)so.lit.size();
                for (uint32_t dp : so.date_pos) fixups.push_back(o.aux + dp);
                fixed += o.len;
            }
            if (so.body) P.body_fixed += fixed; else P.hdr_fixed += fixed;
            ops.push_back(o);
        }
        max_fixed = std::max(max_fixed, P.hdr_fixed + P.body_fixed);
    }

    // shape classes: same op-code / flag sequence → same control flow in the interpreter
    {
        std::map<std::string, int> classes;
        for (size_t pi = 0; pi < progs.size(); pi++) {
            ProgRec& P = progs[pi];
            std::string sig = std::to_string(P.flags & (PF_BIND | PF_NEEDS_ROW));
            for (uint32_t k = 0; k < P.n_ops; k++) {
                const Op& o = ops[P.first_op + k];
                sig += "|" + std::to_string(o.code) + "," + std::to_string(o.flags) + "," + std::to_string(o.kind) + (o.len ? "p" : "");
            }
            auto it = classes.find(sig);
            int id = it != classes.end() ? it->second : (int)classes.size() + 1;
            if (it == classes.end()) classes[sig] = id;
            P.shape_class = (uint8_t)(id > 30 ? 30 : id);
        }
    }

    // the size pass only needs the ops whose length depends on the request (everything else is pre-summed)
    for (size_t pi = 0; pi < progs.size(); pi++) {
        ProgRec& P = progs[pi];
        P.first_dyn = (uint16_t)ops.size();
        std::vector<Op> dyn;
        for (uint32_t k = 0; k < P.n_ops; k++) {
            const Op& o = ops[P.first_op + k];
            bool fixed_len = (o.code == OP_LIT && !(o.flags & OPF_VALUE_OF_KEY)) || o.code == OP_HEXID || o.code == OP_CLEN || o.code == OP_BLOB;
            if (!fixed_len) dyn.push_back(o);
        }
        P.n_dyn = (uint16_t)dyn.size();
        uint16_t nh = 0;
        while (nh < P.n_ops && !(ops[P.first_op + nh].flags & OPF_BODY)) nh++;
        P.n_hdr_ops = nh;
        ops.insert(ops.end(), dyn.begin(), dyn.end());
    }

    // ---- slot-layout fast path: templates and tail ops (table_format.h FastRec) ----
    std::vector<FastRec> fast(progs.size());
    for (size_t pi = 0; pi < progs.size(); pi++) {
        ProgRec& P = progs[pi];
        FastRec& F = fast[pi];
        memset(&F, 0, sizeof F);
        F.hex_pos = 0xFFFF;
        F.tail_op = P.first_op;
        F.n_tail_ops = P.n_ops;
        if (P.flags & PF_BIND) F.flags |= FR_BIND;
        bool simple_ops = true;
        for (uint32_t k = 0; k < P.n_ops; k++) {
            const Op& o = ops[P.first_op + k];
            const bool ok = o.code == OP_LIT || o.code == OP_HEXID || o.code == OP_CLEN || o.code == OP_I64 || o.code == OP_I32 ||
                            o.code == OP_BOOL || o.code == OP_STR || o.code == OP_BSTR || o.code == OP_PARAM || o.code == OP_KEY;
            if (!ok) simple_ops = false;
            // the lean size pass adds every dynamic length to the body
            const bool dynamic = (o.code != OP_LIT || (o.flags & OPF_VALUE_OF_KEY)) && o.code != OP_HEXID && o.code != OP_CLEN;
            if (ok && dynamic && !(o.flags & OPF_BODY)) simple_ops = false;
        }
        if (!simple_ops) continue;
        P.flags |= PF_FAST;
        // the position-fixed prefix: literal bytes (an op's own literal or its folded prefix) and the trace id placeholder,
        // up to the first value whose length depends on the request
        std::string tmpl;
        std::vector<uint32_t> date_at;  // template offsets of Date placeholders
        struct Span { uint32_t op, lit_start, lit_len; };  // where each op's literal bytes sit in the template
        std::vector<Span> spans;
        uint32_t stop_op = P.n_ops;  // first op with a variable-length value
        for (uint32_t k = 0; k < P.n_ops; k++) {
            const Op& o = ops[P.first_op + k];
            if (o.code == OP_KEY || (o.flags & OPF_VALUE_OF_KEY)) { stop_op = k; break; }  // emitted or not: depends on the row
            const uint32_t loff = o.code == OP_LIT ? o.off : o.aux;
            spans.push_back({k, (uint32_t)tmpl.size(), o.len});
            for (uint32_t fx : fixups)
                if (o.len >= 29 && fx >= loff && fx + 29 <= loff + o.len) date_at.push_back((uint32_t)tmpl.size() + (fx - loff));
            tmpl.append((const char*)lits.data() + loff, o.len);
            if (o.code == OP_LIT) continue;
            if (o.code == OP_HEXID && F.hex_pos == 0xFFFF) { F.hex_pos = (uint16_t)tmpl.size(); tmpl.append(32, '0'); continue; }
            stop_op = k;
            break;
        }
        const bool complete = stop_op == P.n_ops;
        uint32_t covered = complete ? (uint32_t)tmpl.size() : ((uint32_t)tmpl.size() & ~15u);
        if (F.hex_pos != 0xFFFF && covered < (uint32_t)F.hex_pos + 32u) {  // the cut would split the trace id: stop before it
            covered = (uint32_t)F.hex_pos & ~15u;
            F.hex_pos = 0xFFFF;
        }
        if (covered > 255u * 16u) covered = 255u * 16u;
        if (!complete || covered != tmpl.size()) covered &= ~15u;
        if (covered == 0) continue;  // nothing worth a template: the whole program is the tail
        std::sort(date_at.begin(), date_at.end());
        date_at.erase(std::unique(date_at.begin(), date_at.end()), date_at.end());
        tmpl.resize(covered);
        F.tmpl_off = pool.put16(tmpl);
        F.tmpl_windows = (uint8_t)((covered + 15u) / 16u);
        F.tmpl_bytes = covered;
        for (uint32_t d : date_at)
            if (d + 29 <= covered) fixups.push_back(F.tmpl_off + d);
            else if (d < covered) { F.tmpl_off = 0; F.tmpl_windows = 0; F.tmpl_bytes = 0; F.hex_pos = 0xFFFF; break; }  // never: Date is followed by > 16 literal bytes
        if (!F.tmpl_windows) continue;
        if (complete && covered == (uint32_t)P.hdr_fixed + P.body_fixed) {
            F.flags |= FR_COMPLETE;
            F.tail_op = 0;
            F.n_tail_ops = 0;
            continue;
        }
        // tail ops: a private copy of the ops from the one that holds byte `covered` on, its literal cut
        uint32_t first = P.n_ops, cut = 0;
        for (auto& sp : spans) {
            const Op& o = ops[P.first_op + sp.op];
            const bool fixed_value = o.code == OP_LIT || (o.code == OP_HEXID && sp.op != stop_op);
            const uint32_t ext = sp.lit_len + (o.code == OP_HEXID && sp.op != stop_op ? 32u : 0u);
            if (fixed_value && sp.lit_start + ext <= covered) continue;  // literal and value both inside the template
            first = sp.op;
            cut = covered > sp.lit_start ? std::min(covered - sp.lit_start, sp.lit_len) : 0u;
            break;
        }
        if (first == P.n_ops && stop_op < P.n_ops) first = stop_op;  // everything before the first variable op is covered
        if (first == P.n_ops) { F.flags |= FR_COMPLETE; F.tail_op = 0; F.n_tail_ops = 0; continue; }
        F.tail_op = (uint16_t)ops.size();
        F.n_tail_ops = (uint16_t)(P.n_ops - first);
        for (uint32_t k = first; k < P.n_ops; k++) {
            Op o = ops[P.first_op + k];
            if (k == first && cut) {  // cut <= o.len by construction (the cut never falls inside a value)
                if (o.code == OP_LIT) o.off += cut; else o.aux += cut;
                o.len -= cut;
            }
            ops.push_back(o);
        }
    }

    std::vector<uint8_t> schema_bytes;
    std::vector<SchemaRec> srecs(t->schemas.size());
    std::vector<std::vector<FieldRec>> frecs(t->schemas.size());
    for (size_t si = 0; si < t->schemas.size(); si++) {
        SchemaDef& s = t->schemas[si];
        SchemaRec& S = srecs[si];
        memset(&S, 0, sizeof S);
        S.n_fields = (uint16_t)s.fields.size();
        S.type_off = pool.put(s.go_type + std::string(1, '\0'));
        uint16_t word = 0, so = 0;
        for (auto& f : s.fields) {
            FieldRec F;
            memset(&F, 0, sizeof F);
            F.kind = f.kind; F.omitempty = f.omitempty; F.word = word;
            F.container = f.container;
            F.n_words = (uint8_t)field_words(t->schemas, f);
            F.elem = f.elem >= 0 ? (uint16_t)f.elem : (uint16_t)0xFFFF;
            word = (uint16_t)(word + F.n_words);
            F.name_len = (uint16_t)f.json_name.size();
            F.name_off = pool.put(f.json_name);
            F.fold_off = pool.put(fold_lower(f.json_name));
            const std::string key = "\"" + json_escape_go(f.json_name) + "\":";
            F.key_off = pool.put(key);
            F.key_len = (uint16_t)key.size();
            if (f.kind == GOFR_F_STRING && f.container == GOFR_C_VALUE) F.str_ord = so++;
            std::string tn = go_kind_name(f.kind);
            F.type_off = pool.put(tn);
            F.type_len = (uint16_t)tn.size();
            frecs[si].push_back(F);
        }
        S.flags = (uint16_t)((s.flat ? SF_FLAT : 0) | (s.bare() ? SF_BARE : 0) | (s.bindable ? SF_BINDABLE : 0));
        S.fixed_words = word;
        S.n_strings = so;
    }

    H.n_pieces = (uint32_t)pieces.size();
    H.n_progs = (uint32_t)progs.size();
    H.n_ops = (uint32_t)ops.size();
    H.n_schemas = (uint32_t)srecs.size();
    for (size_t ri = 0; ri < t->routes.size(); ri++) {
        if (t->routes[ri].hkind != GOFR_H_BIND_ECHO) continue;
        uint32_t words = 8;
        for (auto& f : t->schemas[routes[ri].schema].fields) words += (f.kind == GOFR_F_INT32 || f.kind == GOFR_F_BOOL) ? 1 : 2;  // bindable: checked at seal
        H.bind_row_words = std::max(H.bind_row_words, words);
    }
    H.max_fixed_len = max_fixed;
    {   // image_data_expand (engine_internal.h): the smallest thing that owns data bytes is a 4-byte word; it can drag along
        // one key literal, a comma and a pair of braces per nesting level, and the longest scalar text (a float64: 25 bytes)
        bool any_values = false;
        for (auto& P : progs) any_values |= (P.flags & PF_VALUES) != 0;
        size_t max_key = 0, depth = 1;
        for (auto& sc : t->schemas) {
            depth = std::max(depth, (size_t)sc.depth);
            for (auto& f : sc.fields) max_key = std::max(max_key, json_escape_go(f.json_name).size() + 3);
        }
        H.reserved3[0] = any_values ? (uint32_t)std::max<size_t>(6, (depth * (max_key + 3) + 28 + 3) / 4) : 6u;
    }

    auto append = [&](const void* p, size_t n) {
        align16();
        uint32_t off = (uint32_t)img.size();
        img.insert(img.end(), (const uint8_t*)p, (const uint8_t*)p + n);
        return off;
    };
    H.routes_off = append(routes.data(), routes.size() * sizeof(RouteRec));
    H.pieces_off = append(pieces.data(), pieces.size() * sizeof(PieceRec));
    H.progs_off = append(progs.data(), progs.size() * sizeof(ProgRec));
    H.ops_off = append(ops.data(), ops.size() * sizeof(Op));
    H.hash_off = append(hash_tab.data(), hash_tab.size() * 2);
    H.hash_bits = hash_bits;
    H.thash_off = append(thash_tab.data(), thash_tab.size() * 2);
    H.thash_bits = thash_bits;
    H.tmpl_off = append(tmpl_list.data(), tmpl_list.size() * 2);
    H.n_tmpl = (uint32_t)tmpl_list.size();
    {
        std::vector<uint32_t> keys(tmpl_list.size() * 4, 0u);
        for (size_t ti = 0; ti < tmpl_list.size(); ti++) {
            const RouteDef& r = t->routes[tmpl_list[ti]];
            const std::string& l0 = r.pieces.empty() ? std::string() : r.pieces[0].lit;
            uint8_t kb[8] = {0}, mb[8] = {0};
            for (size_t k = 0; k < l0.size() && k < 8; k++) { kb[k] = (uint8_t)l0[k]; mb[k] = 0xFF; }
            memcpy(&keys[ti * 4], kb, 8);
            memcpy(&keys[ti * 4 + 2], mb, 8);
        }
        if (keys.empty()) keys.resize(4, 0u);
        H.tmplkey_off = append(keys.data(), keys.size() * 4);
    }
    H.last_method_off = append(last_method.data(), last_method.size() * 2);
    {
        std::vector<uint32_t> ids;
        for (auto& sdef : t->schemas) ids.push_back(sdef.id);
        if (ids.empty()) ids.push_back(0xFFFFFFFFu);
        H.schema_ids_off = append(ids.data(), ids.size() * 4);
    }
    H.fast_off = append(fast.data(), fast.size() * sizeof(FastRec));
    if (rawprogs.empty()) rawprogs.resize(9, 0xFFFF);
    H.rawprog_off = append(rawprogs.data(), rawprogs.size() * 2);
    H.fixups_off = append(fixups.data(), fixups.size() * 4);
    H.n_fixups = (uint32_t)fixups.size();
    // schemas: SchemaRec[n] then each field table
    align16();
    H.schemas_off = (uint32_t)img.size();
    size_t srec_pos = img.size();
    img.resize(img.size() + srecs.size() * sizeof(SchemaRec));
    for (size_t si = 0; si < srecs.size(); si++) {
        srecs[si].fields_off = append(frecs[si].data(), frecs[si].size() * sizeof(FieldRec));
        memcpy(img.data() + srec_pos + si * sizeof(SchemaRec), &srecs[si], sizeof(SchemaRec));
    }
    H.lits_off = append(lits.data(), lits.size());
    align16();
    H.hot_bytes = (uint32_t)img.size();
    H.cold_off = append(cold.data(), cold.size());
    align16();
    H.total_bytes = (uint32_t)img.size();
    H.checksum = 0;
    memcpy(img.data(), &H, sizeof H);
    H.checksum = image_checksum(img.data(), img.size());
    memcpy(img.data(), &H, sizeof H);
    if (H.hot_bytes > kMaxHotBytes) {
        set_last_error("sealed table needs %u bytes of shared memory (limit %u)", H.hot_bytes, kMaxHotBytes);
        return GOFR_ERR_CAPACITY;
    }
    t->sealed = true;
    return GOFR_OK;
}

}  // namespace gofr

// ---------------------------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------------------------

extern "C" {

int gofr_table_create(gofr_table** out, uint32_t frame_mode) {
    if (!out || frame_mode > GOFR_FRAME_BODY) return GOFR_ERR_INVALID;
    *out = new gofr_table();
    (*out)->frame_mode = frame_mode;
    return GOFR_OK;
}

void gofr_table_destroy(gofr_table* t) { delete t; }

int gofr_table_add_schema(gofr_table* t, uint32_t schema_id, const char* go_type_name, const gofr_field_desc* fields,
                          uint32_t n_fields) {
    if (!t || !fields || n_fields == 0 || n_fields > (uint32_t)kMaxFields) return GOFR_ERR_INVALID;
    if (t->sealed) return GOFR_ERR_SEALED;
    SchemaDef s;
    s.id = schema_id;
    s.go_type = go_type_name ? go_type_name : "";
    for (auto& o : t->schemas)
        if (o.id == schema_id) { set_last_error("schema %u added twice", schema_id); return GOFR_ERR_INVALID; }
    for (uint32_t i = 0; i < n_fields; i++) {
        FieldDef f;
        f.go_name = fields[i].go_name ? fields[i].go_name : "";
        f.json_name = fields[i].json_name && fields[i].json_name[0] ? fields[i].json_name : f.go_name;
        f.kind = fields[i].kind;
        f.omitempty = fields[i].omitempty != 0;
        f.container = fields[i].container;
        f.flags = fields[i].flags;
        if (f.kind < GOFR_F_INT64 || f.kind > GOFR_F_TIME || f.container > GOFR_C_SLICE_PTR || (f.flags & ~GOFR_FIELD_BARE)) {
            set_last_error("schema %u: unsupported field kind %u / container %u", schema_id, f.kind, f.container);
            return GOFR_ERR_UNSUPPORTED;
        }
        if ((f.flags & GOFR_FIELD_BARE) && n_fields != 1) { set_last_error("schema %u: a bare schema has exactly one field", schema_id); return GOFR_ERR_INVALID; }
        if (f.kind == GOFR_F_STRUCT) {
            for (size_t k = 0; k < t->schemas.size(); k++) if (t->schemas[k].id == fields[i].elem_schema) f.elem = (int)k;
            // the struct type must exist already: a type cannot contain itself by value, and recursive pointer / slice
            // types (trees) have no bound on the nesting the device walker would have to keep
            if (f.elem < 0) { set_last_error("schema %u: field %s refers to schema %u, which has not been added", schema_id, f.go_name.c_str(), fields[i].elem_schema); return GOFR_ERR_INVALID; }
            if (f.container == GOFR_C_MAP) { set_last_error("schema %u: maps of structs are not supported", schema_id); return GOFR_ERR_UNSUPPORTED; }
            if (t->schemas[(size_t)f.elem].bare()) { set_last_error("schema %u: a bare schema cannot be a struct member", schema_id); return GOFR_ERR_INVALID; }
            s.depth = std::max(s.depth, 1 + t->schemas[(size_t)f.elem].depth);
        }
        if (f.container != GOFR_C_VALUE || f.kind > GOFR_F_INT || f.flags) s.flat = false;
        if (f.container != GOFR_C_VALUE || f.kind > GOFR_F_FLOAT64 || f.flags) s.bindable = false;
        const uint32_t fw = field_words(t->schemas, f);
        if (fw > 255u || s.fixed_words + fw > 4096u) { set_last_error("schema %u: fixed part too wide", schema_id); return GOFR_ERR_UNSUPPORTED; }
        s.fixed_words += fw;
        s.fields.push_back(f);
    }
    if (s.depth > kMaxValueDepth) { set_last_error("schema %u: structs nest deeper than %d levels", schema_id, kMaxValueDepth); return GOFR_ERR_UNSUPPORTED; }
    t->schemas.push_back(s);
    return GOFR_OK;
}

int gofr_table_add_route(gofr_table* t, uint32_t method, const char* pattern, uint32_t pattern_len,
                         const gofr_handler_desc* h, uint32_t* route_id_out) {
    if (!t || !pattern || !h) return GOFR_ERR_INVALID;
    if (t->sealed) return GOFR_ERR_SEALED;
    if (method > GOFR_M_OTHER && method != GOFR_M_ANY) return GOFR_ERR_INVALID;
    RouteDef r;
    r.method = method;
    r.pattern.assign(pattern, pattern_len);
    r.prefix = method == GOFR_M_ANY;
    r.hkind = h->kind;
    r.schema_id = h->schema_id;
    const char* ss[4] = {h->s0, h->s1, h->s2, h->s3};
    uint32_t sl[4] = {h->s0_len, h->s1_len, h->s2_len, h->s3_len};
    for (int k = 0; k < 4; k++) if (ss[k]) r.s[k].assign(ss[k], sl[k]);
    if (h->blob) r.blob.assign((const char*)h->blob, h->blob_len);
    int rc = parse_template(r.pattern, r.pieces);
    if (rc == GOFR_ERR_UNSUPPORTED) { set_last_error("pattern %s: unsupported variable regexp", r.pattern.c_str()); return rc; }
    // mux: "path must start with a slash" / malformed braces → route.err → the route never matches
    if (rc == -1 || r.pattern.empty() || r.pattern[0] != '/') { r.dead = true; r.pieces.clear(); r.pieces.push_back(Piece()); }
    if (route_id_out) *route_id_out = (uint32_t)t->routes.size();
    t->routes.push_back(std::move(r));
    return GOFR_OK;
}

int gofr_table_slot_ctas(const gofr_table* t, int* ctas_per_sm) {
    if (!t || !ctas_per_sm) return GOFR_ERR_INVALID;
    if (!t->sealed) return GOFR_ERR_NOT_SEALED;
    *ctas_per_sm = gofr::kServeCtas;  // the wide instance is opt-in (engine.cu choose_slot_residency)
    return GOFR_OK;
}

int gofr_table_add_default_routes(gofr_table* t, const uint8_t* favicon, uint32_t favicon_len) {
    if (!t) return GOFR_ERR_INVALID;
    if (t->sealed) return GOFR_ERR_SEALED;
    gofr_handler_desc h;
    memset(&h, 0, sizeof h);
    h.kind = GOFR_H_HEALTH;
    int rc = gofr_table_add_route(t, GOFR_M_GET, "/.well-known/health", 19, &h, nullptr);
    if (rc) return rc;
    h.kind = GOFR_H_FILE; h.s0 = "image/x-icon"; h.s0_len = 12; h.blob = favicon; h.blob_len = favicon_len;
    rc = gofr_table_add_route(t, GOFR_M_GET, "/favicon.ico", 12, &h, nullptr);
    if (rc) return rc;
    memset(&h, 0, sizeof h);
    h.kind = GOFR_H_MISSING_FILE;
    rc = gofr_table_add_route(t, GOFR_M_ANY, "/", 1, &h, nullptr);
    for (size_t k = t->routes.size() >= 3 ? t->routes.size() - 3 : 0; k < t->routes.size(); k++) t->routes[k].is_default = true;
    if (rc) return rc;
    t->has_catchall = true;
    return GOFR_OK;
}

int gofr_table_seal(gofr_table* t) {
    if (!t) return GOFR_ERR_INVALID;
    if (t->sealed) return GOFR_ERR_SEALED;
    return seal_table(t);
}

int gofr_table_serialize(const gofr_table* t, uint8_t* buf, uint64_t* len_inout) {
    if (!t || !len_inout) return GOFR_ERR_INVALID;
    if (!t->sealed) return GOFR_ERR_NOT_SEALED;
    uint64_t need = t->image.size();
    if (!buf) { *len_inout = need; return GOFR_OK; }
    if (*len_inout < need) { *len_inout = need; return GOFR_ERR_CAPACITY; }
    memcpy(buf, t->image.data(), need);
    *len_inout = need;
    return GOFR_OK;
}

int gofr_table_deserialize(gofr_table** out, const uint8_t* buf, uint64_t len) {
    if (!out || !buf || len < sizeof(ImageHeader)) return GOFR_ERR_INVALID;
    ImageHeader H;
    memcpy(&H, buf, sizeof H);
    if (H.magic != kMagic || H.version != kImageVersion || H.total_bytes != len || H.hot_bytes > kMaxHotBytes) {
        set_last_error("not a sealed gofr table image (magic/version/length mismatch)");
        return GOFR_ERR_INVALID;
    }
    gofr_table* t = new gofr_table();
    t->frame_mode = H.frame_mode;
    t->has_catchall = H.has_catchall != 0;
    t->image.assign(buf, buf + len);
    {   // the image crossed a process boundary: refuse anything that is not byte for byte what seal produced
        ImageHeader Z = H;
        Z.checksum = 0;
        memcpy(t->image.data(), &Z, sizeof Z);
        const uint32_t sum = gofr::image_checksum(t->image.data(), t->image.size());
        memcpy(t->image.data(), &H, sizeof H);
        if (sum != H.checksum) {
            delete t;
            set_last_error("sealed table image is corrupt (checksum %08x, expected %08x)", sum, H.checksum);
            return GOFR_ERR_INVALID;
        }
    }
    t->sealed = true;
    *out = t;
    return GOFR_OK;
}

uint32_t gofr_table_route_count(const gofr_table* t) {
    if (!t) return 0;
    if (!t->image.empty()) { ImageHeader H; memcpy(&H, t->image.data(), sizeof H); return H.n_routes; }
    return (uint32_t)t->routes.size();
}

uint32_t gofr_table_max_response_bytes(const gofr_table* t, uint32_t max_data_len) {
    if (!t || t->image.empty()) return 0;
    ImageHeader H;
    memcpy(&H, t->image.data(), sizeof H);
    // fixed part + Content-Length digits + every data byte escaped six-fold (\u00XX) + Location (3x path + query)
    const uint64_t b = (uint64_t)H.max_fixed_len + 16 + (uint64_t)gofr::image_data_expand(H) * max_data_len + 3 * 65535 + 65535 + 2;
    return b > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)b;  // saturates like gofr_table_response_bound
}

uint32_t gofr_table_response_bound(const gofr_table* t, uint32_t path_len, uint32_t query_len, uint32_t data_len) {
    if (!t || t->image.empty()) return 0;
    ImageHeader H;
    memcpy(&H, t->image.data(), sizeof H);
    // fixed part + Content-Length digits + every request byte that can reach the response (a path variable, a query value,
    // a data byte; the Location of a redirect is at most 3x path + query) escaped six-fold (\u00XX)
    const uint64_t b = (uint64_t)H.max_fixed_len + 16 + 6ull * ((uint64_t)path_len + query_len) + (uint64_t)gofr::image_data_expand(H) * data_len + 2;
    return b > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)b;
}

}  // extern "C"

const std::vector<uint8_t>& gofr_table_image(const gofr_table* t) { return t->image; }
