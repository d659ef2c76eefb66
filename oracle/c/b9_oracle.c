/*
 * CPU ORACLE in plain C (TEST INFRASTRUCTURE — never linked into or called by the product).
 *
 * A batch-at-a-time restatement of beta9's per-task dispatch loop, same steps and order as
 * oracle/pyoracle/loop.py, used (a) to check the CUDA path bit-for-bit at sizes where the Python
 * oracle is too slow and (b) as bench.py's `cpu_baseline` ("port") on the GPU box's host cores.
 *
 * Reference lines restated (relative to /root/reference):
 *   decode   pkg/abstractions/taskqueue/taskqueue.go:213-214   json.Unmarshal(in.Payload,&TaskPayload)
 *            pkg/types/task.go:13-16                           TaskPayload{Args,Kwargs}
 *   send     pkg/task/dispatch.go:84-105                       TaskMessage fill, Encode
 *   encode   pkg/types/task.go:55-65,79-90                     TaskMessage JSON, nil Args -> []
 *   policy   pkg/abstractions/taskqueue/taskqueue.go:191-196   Expires = now + TTL
 *   fifo     pkg/abstractions/taskqueue/client.go:29-96        RPUSH / LPOP, popped bytes returned
 *   loads    sdk/src/beta9/runner/taskqueue.py:196-201         json.loads(task_msg)
 *   call     sdk/src/beta9/runner/taskqueue.py:349-361         handler(*(args or []), **(kwargs or {}))
 *   result   sdk/src/beta9/runner/taskqueue.py:378             serialize_result(result) if result else None
 *            sdk/src/beta9/runner/common.py:484-489            json.dumps(result).encode("utf-8")
 *
 * Third-party arithmetic restated: Go 1.23 encoding/json + time.Time.MarshalJSON (go.mod:3),
 * CPython json.loads/json.dumps (ensure_ascii, default separators), zlib.crc32, base64.
 *
 * PARITY: the Go encode/decode boundary is UNPINNED (no reference golden bytes, no Go toolchain
 * here — SURVEY.md §8c). This file is pinned only against oracle/pyoracle (whose Python halves
 * are the reference's own stdlib calls) by tests/test_oracle_c_vs_py.py.
 *
 * Restricted domain: numbers that are not integers of magnitude <= 2^53 need shortest-float
 * formatting (Go strconv / CPython repr); this port reports them as B9O_UNSUPPORTED instead of
 * guessing. oracle/pyoracle covers the full domain.
 */
#define _GNU_SOURCE
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

enum { B9O_COMPLETE = 0, B9O_ERROR = 1, B9O_REJECTED = 3, B9O_UNSUPPORTED = 4 };
enum { H_IDENTITY = 0, H_CRC32 = 1, H_VADD_F32 = 2, H_JSON_SUM = 3 };

/* ------------------------------------------------------------------ arena + byte buffer */
typedef struct { uint8_t *base; size_t cap, used; } arena_t;

static void *arena_alloc(arena_t *a, size_t n) {
    n = (n + 15) & ~(size_t)15;
    if (a->used + n > a->cap) {
        size_t nc = a->cap ? a->cap * 2 : (1u << 16);
        while (nc < a->used + n) nc *= 2;
        /* blocks are chained by leaking the old one into a list: keep it simple and never move */
        uint8_t *nb = (uint8_t *)malloc(nc + sizeof(void *));
        *(void **)nb = a->base ? (void *)(a->base - sizeof(void *)) : NULL;
        a->base = nb + sizeof(void *);
        a->cap = nc;
        a->used = 0;
    }
    void *p = a->base + a->used;
    a->used += n;
    return p;
}
static void arena_free_all(arena_t *a) {
    void *p = a->base ? (void *)(a->base - sizeof(void *)) : NULL;
    while (p) { void *nx = *(void **)p; free(p); p = nx; }
    a->base = NULL; a->cap = a->used = 0;
}

typedef struct { uint8_t *p; size_t len, cap; } buf_t;
static void buf_reserve(buf_t *b, size_t extra) {
    if (b->len + extra <= b->cap) return;
    size_t nc = b->cap ? b->cap * 2 : 1024;
    while (nc < b->len + extra) nc *= 2;
    b->p = (uint8_t *)realloc(b->p, nc);
    b->cap = nc;
}
static void buf_put(buf_t *b, const void *s, size_t n) { buf_reserve(b, n); memcpy(b->p + b->len, s, n); b->len += n; }
static void buf_putc(buf_t *b, uint8_t c) { buf_reserve(b, 1); b->p[b->len++] = c; }
static void buf_puts(buf_t *b, const char *s) { buf_put(b, s, strlen(s)); }

/* ------------------------------------------------------------------ value tree */
typedef enum { T_NULL, T_FALSE, T_TRUE, T_NUM, T_STR, T_ARR, T_OBJ } vtype_t;
typedef struct val {
    vtype_t t;
    /* T_NUM */
    double num;
    int is_int;             /* python mode: literal had no frac/exp;  go mode: integer-valued */
    int overflow;           /* go mode: ParseFloat ErrRange */
    const uint8_t *lit; size_t lit_len;   /* literal text */
    /* T_STR: decoded UTF-8 */
    const uint8_t *s; size_t slen;
    /* T_ARR / T_OBJ */
    struct val **items; struct val **keys; size_t n;
} val_t;

typedef struct {
    const uint8_t *d; size_t i, n;
    arena_t *ar;
    int err;
    int depth;
} parser_t;

static int is_ws(uint8_t c) { return c == ' ' || c == '\t' || c == '\r' || c == '\n'; }
static void skip_ws(parser_t *p) { while (p->i < p->n && is_ws(p->d[p->i])) p->i++; }
static val_t *new_val(parser_t *p, vtype_t t) {
    val_t *v = (val_t *)arena_alloc(p->ar, sizeof(val_t));
    memset(v, 0, sizeof(*v)); v->t = t; return v;
}
static int hexv(uint8_t c) {
    if (c >= '0' && c <= '9') return c - '0';
    if (c >= 'a' && c <= 'f') return c - 'a' + 10;
    if (c >= 'A' && c <= 'F') return c - 'A' + 10;
    return -1;
}
/* decode.go getu4 */
static int getu4(const uint8_t *d, size_t at, size_t n) {
    if (at + 6 > n || d[at] != '\\' || d[at + 1] != 'u') return -1;
    int v = 0;
    for (int k = 2; k < 6; k++) { int h = hexv(d[at + k]); if (h < 0) return -1; v = v * 16 + h; }
    return v;
}
static size_t put_utf8(uint8_t *o, uint32_t cp) {
    if (cp < 0x80) { o[0] = (uint8_t)cp; return 1; }
    if (cp < 0x800) { o[0] = 0xC0 | (cp >> 6); o[1] = 0x80 | (cp & 0x3F); return 2; }
    if (cp < 0x10000) { o[0] = 0xE0 | (cp >> 12); o[1] = 0x80 | ((cp >> 6) & 0x3F); o[2] = 0x80 | (cp & 0x3F); return 3; }
    o[0] = 0xF0 | (cp >> 18); o[1] = 0x80 | ((cp >> 12) & 0x3F); o[2] = 0x80 | ((cp >> 6) & 0x3F); o[3] = 0x80 | (cp & 0x3F); return 4;
}
/* Go utf8.DecodeRune: returns width, *cp = rune (0xFFFD, width 1 on invalid) */
static size_t decode_rune(const uint8_t *d, size_t i, size_t n, uint32_t *cp) {
    uint8_t c0 = d[i];
    if (c0 < 0x80) { *cp = c0; return 1; }
    if (c0 >= 0xC2 && c0 <= 0xDF) {
        if (i + 1 < n && (d[i + 1] & 0xC0) == 0x80) { *cp = ((c0 & 0x1Fu) << 6) | (d[i + 1] & 0x3F); return 2; }
    } else if (c0 >= 0xE0 && c0 <= 0xEF) {
        uint8_t lo = 0x80, hi = 0xBF;
        if (c0 == 0xE0) lo = 0xA0; else if (c0 == 0xED) hi = 0x9F;
        if (i + 2 < n && d[i + 1] >= lo && d[i + 1] <= hi && (d[i + 2] & 0xC0) == 0x80) {
            *cp = ((c0 & 0x0Fu) << 12) | ((d[i + 1] & 0x3Fu) << 6) | (d[i + 2] & 0x3F); return 3;
        }
    } else if (c0 >= 0xF0 && c0 <= 0xF4) {
        uint8_t lo = 0x80, hi = 0xBF;
        if (c0 == 0xF0) lo = 0x90; else if (c0 == 0xF4) hi = 0x8F;
        if (i + 3 < n && d[i + 1] >= lo && d[i + 1] <= hi && (d[i + 2] & 0xC0) == 0x80 && (d[i + 3] & 0xC0) == 0x80) {
            *cp = ((c0 & 0x07u) << 18) | ((d[i + 1] & 0x3Fu) << 12) | ((d[i + 2] & 0x3Fu) << 6) | (d[i + 3] & 0x3F); return 4;
        }
    }
    *cp = 0xFFFD; return 1;
}

static val_t *parse_value(parser_t *p);

/* String literal -> decoded UTF-8 following Go's unquote (lone surrogate / bad UTF-8 -> U+FFFD).
 * CPython's json.loads differs only on inputs Go never emits (lone surrogate escapes). */
static val_t *parse_string(parser_t *p) {
    const uint8_t *d = p->d; size_t n = p->n, i = p->i + 1;
    /* worst case growth: 1 invalid byte -> 3 bytes */
    size_t j = i; while (j < n && d[j] != '"') { if (d[j] == '\\') j++; j++; }
    if (j > n) j = n;
    size_t cap = (j > i ? (j - i) : 0) * 3 + 4;
    uint8_t *o = (uint8_t *)arena_alloc(p->ar, cap); size_t ol = 0;
    for (;;) {
        if (i >= n) { p->err = 1; return NULL; }
        uint8_t c = d[i];
        if (c == '"') { i++; break; }
        if (c < 0x20) { p->err = 1; return NULL; }
        if (c == '\\') {
            if (i + 1 >= n) { p->err = 1; return NULL; }
            uint8_t e = d[i + 1];
            switch (e) {
            case '"': o[ol++] = '"'; i += 2; continue;
            case '\\': o[ol++] = '\\'; i += 2; continue;
            case '/': o[ol++] = '/'; i += 2; continue;
            case 'b': o[ol++] = '\b'; i += 2; continue;
            case 'f': o[ol++] = '\f'; i += 2; continue;
            case 'n': o[ol++] = '\n'; i += 2; continue;
            case 'r': o[ol++] = '\r'; i += 2; continue;
            case 't': o[ol++] = '\t'; i += 2; continue;
            case 'u': break;
            default: p->err = 1; return NULL;
            }
            int rr = getu4(d, i, n);
            if (rr < 0) { p->err = 1; return NULL; }
            i += 6;
            uint32_t cp = (uint32_t)rr;
            if (rr >= 0xD800 && rr <= 0xDFFF) {
                int rr1 = getu4(d, i, n);
                if (rr <= 0xDBFF && rr1 >= 0xDC00 && rr1 <= 0xDFFF) {
                    cp = 0x10000u + (((uint32_t)rr - 0xD800u) << 10) + ((uint32_t)rr1 - 0xDC00u);
                    i += 6;
                } else cp = 0xFFFD;
            }
            ol += put_utf8(o + ol, cp);
            continue;
        }
        if (c < 0x80) { o[ol++] = c; i++; continue; }
        uint32_t cp; size_t w = decode_rune(d, i, n, &cp);
        ol += put_utf8(o + ol, cp);
        i += w;
    }
    p->i = i;
    val_t *v = new_val(p, T_STR); v->s = o; v->slen = ol; return v;
}

static val_t *parse_number(parser_t *p) {
    const uint8_t *d = p->d; size_t n = p->n, s = p->i, i = s;
    int isint = 1;
    if (i < n && d[i] == '-') i++;
    if (i >= n) { p->err = 1; return NULL; }
    if (d[i] == '0') i++;
    else if (d[i] >= '1' && d[i] <= '9') { while (i < n && d[i] >= '0' && d[i] <= '9') i++; }
    else { p->err = 1; return NULL; }
    if (i < n && d[i] == '.') {
        isint = 0; i++;
        if (i >= n || d[i] < '0' || d[i] > '9') { p->err = 1; return NULL; }
        while (i < n && d[i] >= '0' && d[i] <= '9') i++;
    }
    if (i < n && (d[i] == 'e' || d[i] == 'E')) {
        isint = 0; i++;
        if (i < n && (d[i] == '+' || d[i] == '-')) i++;
        if (i >= n || d[i] < '0' || d[i] > '9') { p->err = 1; return NULL; }
        while (i < n && d[i] >= '0' && d[i] <= '9') i++;
    }
    p->i = i;
    val_t *v = new_val(p, T_NUM);
    v->lit = d + s; v->lit_len = i - s; v->is_int = isint;
    char tmp[64]; char *t = tmp;
    if (v->lit_len >= sizeof(tmp)) t = (char *)arena_alloc(p->ar, v->lit_len + 1);
    memcpy(t, v->lit, v->lit_len); t[v->lit_len] = 0;
    v->num = strtod(t, NULL);        /* glibc: correctly rounded, like strconv.ParseFloat */
    if (isinf(v->num)) v->overflow = 1;
    return v;
}

static val_t *parse_container(parser_t *p, int is_obj) {
    if (++p->depth > 10000) { p->err = 1; return NULL; }
    p->i++;
    size_t cap = 4, cnt = 0;
    val_t **items = (val_t **)arena_alloc(p->ar, cap * sizeof(val_t *));
    val_t **keys = is_obj ? (val_t **)arena_alloc(p->ar, cap * sizeof(val_t *)) : NULL;
    skip_ws(p);
    uint8_t close = is_obj ? '}' : ']';
    if (p->i < p->n && p->d[p->i] == close) { p->i++; goto done; }
    for (;;) {
        skip_ws(p);
        val_t *k = NULL;
        if (is_obj) {
            if (p->i >= p->n || p->d[p->i] != '"') { p->err = 1; return NULL; }
            k = parse_string(p); if (!k) return NULL;
            skip_ws(p);
            if (p->i >= p->n || p->d[p->i] != ':') { p->err = 1; return NULL; }
            p->i++; skip_ws(p);
        }
        val_t *v = parse_value(p); if (!v) return NULL;
        if (cnt == cap) {
            size_t nc = cap * 2;
            val_t **ni = (val_t **)arena_alloc(p->ar, nc * sizeof(val_t *)); memcpy(ni, items, cnt * sizeof(val_t *)); items = ni;
            if (is_obj) { val_t **nk = (val_t **)arena_alloc(p->ar, nc * sizeof(val_t *)); memcpy(nk, keys, cnt * sizeof(val_t *)); keys = nk; }
            cap = nc;
        }
        items[cnt] = v; if (is_obj) keys[cnt] = k; cnt++;
        skip_ws(p);
        if (p->i >= p->n) { p->err = 1; return NULL; }
        uint8_t c = p->d[p->i++];
        if (c == ',') continue;
        if (c == close) break;
        p->err = 1; return NULL;
    }
done:
    p->depth--;
    val_t *v = new_val(p, is_obj ? T_OBJ : T_ARR);
    v->items = items; v->keys = keys; v->n = cnt;
    return v;
}

static val_t *parse_value(parser_t *p) {
    if (p->i >= p->n) { p->err = 1; return NULL; }
    uint8_t c = p->d[p->i];
    if (c == '{') return parse_container(p, 1);
    if (c == '[') return parse_container(p, 0);
    if (c == '"') return parse_string(p);
    if (c == '-' || (c >= '0' && c <= '9')) return parse_number(p);
    if (p->n - p->i >= 4 && !memcmp(p->d + p->i, "true", 4)) { p->i += 4; return new_val(p, T_TRUE); }
    if (p->n - p->i >= 5 && !memcmp(p->d + p->i, "false", 5)) { p->i += 5; return new_val(p, T_FALSE); }
    if (p->n - p->i >= 4 && !memcmp(p->d + p->i, "null", 4)) { p->i += 4; return new_val(p, T_NULL); }
    p->err = 1; return NULL;
}

static val_t *parse_document(const uint8_t *d, size_t n, arena_t *ar) {
    parser_t p = { d, 0, n, ar, 0, 0 };
    skip_ws(&p);
    val_t *v = parse_value(&p);
    if (!v || p.err) return NULL;
    skip_ws(&p);
    if (p.i != p.n) return NULL;
    return v;
}

/* Map semantics: later duplicate keys win, position of first occurrence is irrelevant for Go
 * (keys get sorted). Returns a deduplicated copy (last value per key). */
static int key_eq(const val_t *a, const val_t *b) { return a->slen == b->slen && !memcmp(a->s, b->s, a->slen); }
static void dedup_obj(val_t *o) {
    size_t w = 0;
    for (size_t i = 0; i < o->n; i++) {
        int later = 0;
        for (size_t j = i + 1; j < o->n; j++) if (key_eq(o->keys[i], o->keys[j])) { later = 1; break; }
        if (!later) { o->keys[w] = o->keys[i]; o->items[w] = o->items[i]; w++; }
    }
    o->n = w;
}
/* python dict semantics for json.loads: later duplicates overwrite the VALUE but keep the FIRST
 * key position. Go never emits duplicates, so the wire never exercises this; kept for exactness. */

static int has_overflow(const val_t *v) {
    if (!v) return 0;
    if (v->t == T_NUM) return v->overflow;
    if (v->t == T_ARR || v->t == T_OBJ) for (size_t i = 0; i < v->n; i++) if (has_overflow(v->items[i])) return 1;
    return 0;
}

/* encoding/json foldName equality against an ASCII lower-case field name */
static int fold_eq(const val_t *k, const char *field) {
    size_t fl = strlen(field), fi = 0, i = 0;
    while (i < k->slen) {
        uint8_t c = k->s[i]; uint8_t f;
        if (c < 0x80) { f = (c >= 'A' && c <= 'Z') ? c + 32 : c; i++; }
        else if (i + 2 < k->slen + 0 && c == 0xE2 && k->s[i + 1] == 0x84 && k->s[i + 2] == 0xAA) { f = 'k'; i += 3; } /* U+212A */
        else if (i + 1 < k->slen && c == 0xC5 && k->s[i + 1] == 0xBF) { f = 's'; i += 2; }                          /* U+017F */
        else return 0;
        if (fi >= fl || f != (uint8_t)field[fi]) return 0;
        fi++;
    }
    return fi == fl;
}

/* ------------------------------------------------------------------ Go marshal */
static const char HEXD[] = "0123456789abcdef";

static void go_quote(buf_t *b, const uint8_t *s, size_t n) {
    buf_putc(b, '"');
    size_t i = 0;
    while (i < n) {
        uint8_t c = s[i];
        if (c < 0x80) {
            switch (c) {
            case '"': buf_puts(b, "\\\""); break;
            case '\\': buf_puts(b, "\\\\"); break;
            case '\b': buf_puts(b, "\\b"); break;
            case '\f': buf_puts(b, "\\f"); break;
            case '\n': buf_puts(b, "\\n"); break;
            case '\r': buf_puts(b, "\\r"); break;
            case '\t': buf_puts(b, "\\t"); break;
            default:
                if (c < 0x20 || c == '<' || c == '>' || c == '&') {
                    char e[6] = { '\\', 'u', '0', '0', HEXD[c >> 4], HEXD[c & 15] }; buf_put(b, e, 6);
                } else buf_putc(b, c);
            }
            i++; continue;
        }
        uint32_t cp; size_t w = decode_rune(s, i, n, &cp);
        if (cp == 0xFFFD && w == 1) { buf_puts(b, "\\ufffd"); i++; continue; }
        if (cp == 0x2028 || cp == 0x2029) { buf_puts(b, cp == 0x2028 ? "\\u2028" : "\\u2029"); i += w; continue; }
        buf_put(b, s + i, w); i += w;
    }
    buf_putc(b, '"');
}

static int cmp_keys(const void *a, const void *b) {
    const val_t *ka = *(val_t *const *)a, *kb = *(val_t *const *)b;
    size_t m = ka->slen < kb->slen ? ka->slen : kb->slen;
    int c = memcmp(ka->s, kb->s, m);
    if (c) return c;
    return (ka->slen > kb->slen) - (ka->slen < kb->slen);
}

/* returns 0 ok, B9O_UNSUPPORTED when a number needs shortest-float formatting */
static int go_marshal(buf_t *b, val_t *v, arena_t *ar) {
    switch (v->t) {
    case T_NULL: buf_puts(b, "null"); return 0;
    case T_TRUE: buf_puts(b, "true"); return 0;
    case T_FALSE: buf_puts(b, "false"); return 0;
    case T_STR: go_quote(b, v->s, v->slen); return 0;
    case T_NUM: {
        double f = v->num;
        if (f != floor(f) || fabs(f) > 9007199254740992.0) return B9O_UNSUPPORTED;
        char t[40];
        if (f == 0 && signbit(f)) { buf_puts(b, "-0"); return 0; }
        snprintf(t, sizeof t, "%.0f", f);
        buf_puts(b, t); return 0;
    }
    case T_ARR:
        buf_putc(b, '[');
        for (size_t i = 0; i < v->n; i++) { if (i) buf_putc(b, ','); int r = go_marshal(b, v->items[i], ar); if (r) return r; }
        buf_putc(b, ']'); return 0;
    case T_OBJ: {
        dedup_obj(v);
        /* sort (key,value) pairs by key bytes */
        val_t **pairs = (val_t **)arena_alloc(ar, (2 * v->n + 1) * sizeof(val_t *));
        /* pack pairs as [key,val] structs for qsort */
        typedef struct { val_t *k, *v; } kv_t;
        kv_t *kv = (kv_t *)pairs;
        for (size_t i = 0; i < v->n; i++) { kv[i].k = v->keys[i]; kv[i].v = v->items[i]; }
        qsort(kv, v->n, sizeof(kv_t), cmp_keys);   /* kv_t begins with the key pointer */
        buf_putc(b, '{');
        for (size_t i = 0; i < v->n; i++) {
            if (i) buf_putc(b, ',');
            go_quote(b, kv[i].k->s, kv[i].k->slen); buf_putc(b, ':');
            int r = go_marshal(b, kv[i].v, ar); if (r) return r;
        }
        buf_putc(b, '}'); return 0;
    }
    }
    return 0;
}

static void civil_from_days(int64_t z, int64_t *y, int *m, int *d) {
    z += 719468;
    int64_t era = (z >= 0 ? z : z - 146096) / 146097;
    int64_t doe = z - era * 146097;
    int64_t yoe = (doe - doe / 1460 + doe / 36524 - doe / 146096) / 365;
    *y = yoe + era * 400;
    int64_t doy = doe - (365 * yoe + yoe / 4 - yoe / 100);
    int64_t mp = (5 * doy + 2) / 153;
    *d = (int)(doy - (153 * mp + 2) / 5 + 1);
    *m = (int)(mp < 10 ? mp + 3 : mp - 9);
    if (*m <= 2) (*y)++;
}
/* time.Time.MarshalJSON at UTC ("Z") */
static void go_time(buf_t *b, int64_t unix_ns) {
    int64_t secs = unix_ns / 1000000000, ns = unix_ns % 1000000000;
    if (ns < 0) { ns += 1000000000; secs--; }
    int64_t days = secs / 86400, sod = secs % 86400;
    if (sod < 0) { sod += 86400; days--; }
    int64_t y; int m, d; civil_from_days(days, &y, &m, &d);
    char t[64];
    int l = snprintf(t, sizeof t, "\"%04lld-%02d-%02dT%02d:%02d:%02d", (long long)y, m, d, (int)(sod / 3600), (int)(sod % 3600 / 60), (int)(sod % 60));
    buf_put(b, t, (size_t)l);
    if (ns) {
        char f[16]; snprintf(f, sizeof f, "%09lld", (long long)ns);
        int e = 9; while (e > 0 && f[e - 1] == '0') e--;
        buf_putc(b, '.'); buf_put(b, f, (size_t)e);
    }
    buf_puts(b, "Z\"");
}

typedef struct {
    const char *workspace_name, *stub_id, *executor;
    uint32_t max_retries; int32_t timeout; uint32_t ttl;
    int64_t now_unix_ns;
} env_t;

static void fmt_uuid(char *o, const uint8_t *id) {
    int k = 0;
    for (int i = 0; i < 16; i++) {
        if (i == 4 || i == 6 || i == 8 || i == 10) o[k++] = '-';
        o[k++] = HEXD[id[i] >> 4]; o[k++] = HEXD[id[i] & 15];
    }
    o[k] = 0;
}

/* TaskMessage.Encode */
static int encode_wire(buf_t *b, const env_t *e, const uint8_t *id, val_t *args, val_t *kwargs, arena_t *ar) {
    char u[40]; fmt_uuid(u, id);
    buf_puts(b, "{\"task_id\":"); go_quote(b, (const uint8_t *)u, 36);
    buf_puts(b, ",\"workspace_name\":"); go_quote(b, (const uint8_t *)e->workspace_name, strlen(e->workspace_name));
    buf_puts(b, ",\"stub_id\":"); go_quote(b, (const uint8_t *)e->stub_id, strlen(e->stub_id));
    buf_puts(b, ",\"executor\":"); go_quote(b, (const uint8_t *)e->executor, strlen(e->executor));
    buf_puts(b, ",\"args\":");
    if (args) { int r = go_marshal(b, args, ar); if (r) return r; } else buf_puts(b, "[]");
    buf_puts(b, ",\"kwargs\":");
    if (kwargs) { int r = go_marshal(b, kwargs, ar); if (r) return r; } else buf_puts(b, "null");
    char t[96];
    int l = snprintf(t, sizeof t, ",\"policy\":{\"max_retries\":%u,\"timeout\":%d,\"expires\":", e->max_retries, e->timeout);
    buf_put(b, t, (size_t)l);
    go_time(b, e->now_unix_ns + (int64_t)e->ttl * 1000000000);
    l = snprintf(t, sizeof t, ",\"ttl\":%u},\"retries\":0,\"timestamp\":%lld}", e->ttl, (long long)(e->now_unix_ns / 1000000000));
    buf_put(b, t, (size_t)l);
    return 0;
}

/* ------------------------------------------------------------------ python side */
static val_t *obj_get_last(val_t *o, const char *key) {
    size_t kl = strlen(key); val_t *r = NULL;
    for (size_t i = 0; i < o->n; i++) if (o->keys[i]->slen == kl && !memcmp(o->keys[i]->s, key, kl)) r = o->items[i];
    return r;
}

/* normalised python int text of an is_int literal: "-0" -> "0" */
static int py_int_is_zero(const val_t *v) {
    for (size_t i = 0; i < v->lit_len; i++) if (v->lit[i] != '-' && v->lit[i] != '0') return 0;
    return 1;
}

static int py_truthy(const val_t *v) {
    switch (v->t) {
    case T_NULL: case T_FALSE: return 0;
    case T_TRUE: return 1;
    case T_NUM: return v->is_int ? !py_int_is_zero(v) : (v->num != 0.0);
    case T_STR: return v->slen != 0;
    default: return v->n != 0;
    }
}

static void py_quote(buf_t *b, const uint8_t *s, size_t n) {   /* json.encoder ESCAPE_ASCII */
    buf_putc(b, '"');
    size_t i = 0;
    while (i < n) {
        uint32_t cp; size_t w = decode_rune(s, i, n, &cp); i += w;
        switch (cp) {
        case '"': buf_puts(b, "\\\""); continue;
        case '\\': buf_puts(b, "\\\\"); continue;
        case '\n': buf_puts(b, "\\n"); continue;
        case '\r': buf_puts(b, "\\r"); continue;
        case '\t': buf_puts(b, "\\t"); continue;
        case '\b': buf_puts(b, "\\b"); continue;
        case '\f': buf_puts(b, "\\f"); continue;
        }
        if (cp >= 0x20 && cp <= 0x7E) { buf_putc(b, (uint8_t)cp); continue; }
        uint32_t u[2]; int nu = 1; u[0] = cp;
        if (cp >= 0x10000) { uint32_t x = cp - 0x10000; u[0] = 0xD800 | (x >> 10); u[1] = 0xDC00 | (x & 0x3FF); nu = 2; }
        for (int k = 0; k < nu; k++) {
            char e[6] = { '\\', 'u', HEXD[(u[k] >> 12) & 15], HEXD[(u[k] >> 8) & 15], HEXD[(u[k] >> 4) & 15], HEXD[u[k] & 15] };
            buf_put(b, e, 6);
        }
    }
    buf_putc(b, '"');
}

static int py_dumps(buf_t *b, const val_t *v) {
    switch (v->t) {
    case T_NULL: buf_puts(b, "null"); return 0;
    case T_TRUE: buf_puts(b, "true"); return 0;
    case T_FALSE: buf_puts(b, "false"); return 0;
    case T_STR: py_quote(b, v->s, v->slen); return 0;
    case T_NUM:
        if (!v->is_int) return B9O_UNSUPPORTED;       /* float repr */
        if (py_int_is_zero(v)) { buf_putc(b, '0'); return 0; }
        buf_put(b, v->lit, v->lit_len); return 0;     /* Go wrote canonical digits already */
    case T_ARR:
        buf_putc(b, '[');
        for (size_t i = 0; i < v->n; i++) { if (i) buf_puts(b, ", "); int r = py_dumps(b, v->items[i]); if (r) return r; }
        buf_putc(b, ']'); return 0;
    case T_OBJ:
        buf_putc(b, '{');
        for (size_t i = 0; i < v->n; i++) {
            if (i) buf_puts(b, ", ");
            py_quote(b, v->keys[i]->s, v->keys[i]->slen); buf_puts(b, ": ");
            int r = py_dumps(b, v->items[i]); if (r) return r;
        }
        buf_putc(b, '}'); return 0;
    }
    return 0;
}

/* ------------------------------------------------------------------ handlers */
static uint32_t crc_table[256]; static int crc_ready;
static void crc_init(void) {
    for (uint32_t i = 0; i < 256; i++) { uint32_t c = i; for (int k = 0; k < 8; k++) c = (c & 1) ? 0xEDB88320u ^ (c >> 1) : c >> 1; crc_table[i] = c; }
    crc_ready = 1;
}
static uint32_t crc32_ieee(const uint8_t *s, size_t n) {
    uint32_t c = 0xFFFFFFFFu;
    for (size_t i = 0; i < n; i++) c = crc_table[(c ^ s[i]) & 0xFF] ^ (c >> 8);
    return c ^ 0xFFFFFFFFu;
}
static int b64v(uint8_t c) {
    if (c >= 'A' && c <= 'Z') return c - 'A';
    if (c >= 'a' && c <= 'z') return c - 'a' + 26;
    if (c >= '0' && c <= '9') return c - '0' + 52;
    if (c == '+') return 62;
    if (c == '/') return 63;
    return -1;
}
static const char B64[] = "ABCDEFGHIJKLMNOPQRSTUVWXYZabcdefghijklmnopqrstuvwxyz0123456789+/";

/* base64.b64decode(s, validate=True) as CPython 3.12 behaves (binascii.a2b_base64 strict_mode):
 * only alphabet characters, then 0..2 '=', total length a multiple of 4, no leading '='.
 * Trailing non-zero bits in the last sextet are accepted and dropped. */
static int b64_decode_strict(const uint8_t *s, size_t n, uint8_t *o, size_t *on) {
    if (n % 4) return -1;
    size_t pad = 0;
    if (n && s[n - 1] == '=') { pad++; if (s[n - 2] == '=') pad++; }
    size_t body = n - pad, k = 0;
    for (size_t i = 0; i < body; i++) if (b64v(s[i]) < 0) return -1;
    for (size_t i = 0; i + 4 <= n; i += 4) {
        int last = (i + 4 == n);
        int a = b64v(s[i]), b = b64v(s[i + 1]);
        int c = (last && pad == 2) ? 0 : b64v(s[i + 2]);
        int d = (last && pad >= 1) ? 0 : b64v(s[i + 3]);
        if (a < 0 || b < 0 || c < 0 || d < 0) return -1;
        uint32_t w = ((uint32_t)a << 18) | ((uint32_t)b << 12) | ((uint32_t)c << 6) | (uint32_t)d;
        o[k++] = (uint8_t)(w >> 16);
        if (!(last && pad == 2)) o[k++] = (uint8_t)(w >> 8);
        if (!(last && pad >= 1)) o[k++] = (uint8_t)w;
    }
    *on = k; return 0;
}

/* Runs handler on python-side (args, kwargs); writes result JSON into out (len 0 + has=0 when the
 * runner sends no result). Returns status. */
static int run_handler(int h, val_t *args, val_t *kwargs, buf_t *out, int *has, arena_t *ar) {
    *has = 0;
    size_t nargs = (args && args->t == T_ARR) ? args->n : 0;          /* task["args"] or []   */
    size_t nkw = (kwargs && kwargs->t == T_OBJ) ? kwargs->n : 0;       /* task["kwargs"] or {} */
    if (nargs != 1 || nkw != 0) return B9O_ERROR;                      /* TypeError            */
    val_t *a = args->items[0];
    switch (h) {
    case H_IDENTITY: {
        if (!py_truthy(a)) return B9O_COMPLETE;
        size_t mark = out->len;
        int r = py_dumps(out, a);
        if (r) { out->len = mark; return r; }
        *has = 1; return B9O_COMPLETE;
    }
    case H_CRC32: {
        if (a->t != T_STR) return B9O_ERROR;                           /* AttributeError       */
        uint32_t c = crc32_ieee(a->s, a->slen);
        if (!c) return B9O_COMPLETE;
        char t[16]; int l = snprintf(t, sizeof t, "%u", c); buf_put(out, t, (size_t)l);
        *has = 1; return B9O_COMPLETE;
    }
    case H_VADD_F32: {
        if (a->t != T_STR) return B9O_ERROR;                           /* TypeError            */
        for (size_t i = 0; i < a->slen; i++) if (a->s[i] >= 0x80) return B9O_ERROR;   /* ValueError: non-ASCII */
        uint8_t *raw = (uint8_t *)arena_alloc(ar, a->slen + 4); size_t rn = 0;
        if (b64_decode_strict(a->s, a->slen, raw, &rn)) return B9O_ERROR;
        if (rn % 8) return B9O_ERROR;
        size_t n = rn / 8;
        if (!n) return B9O_COMPLETE;                                   /* "" is falsy          */
        uint8_t *res = (uint8_t *)arena_alloc(ar, n * 4 + 4);
        for (size_t i = 0; i < n; i++) {
            /* numpy `a + b` on x86-64 (SSE/AVX addps, a = first source): a NaN operand comes back
             * quieted, the first one winning; inf + -inf is the "real indefinite" 0xFFC00000. Written
             * out so that the answer does not depend on the operand order this compiler picks. */
            float x, y; uint32_t xb, yb, zb;
            memcpy(&x, raw + 4 * i, 4); memcpy(&y, raw + 4 * (n + i), 4); memcpy(&xb, &x, 4); memcpy(&yb, &y, 4);
            if ((xb & 0x7FFFFFFFu) > 0x7F800000u) zb = xb | 0x00400000u;
            else if ((yb & 0x7FFFFFFFu) > 0x7F800000u) zb = yb | 0x00400000u;
            else { volatile float z = x + y; float zz = z; memcpy(&zb, &zz, 4); if ((zb & 0x7FFFFFFFu) > 0x7F800000u) zb = 0xFFC00000u; }
            memcpy(res + 4 * i, &zb, 4);
        }
        size_t rl = n * 4;
        buf_putc(out, '"');
        for (size_t i = 0; i < rl; i += 3) {
            uint32_t w = (uint32_t)res[i] << 16; size_t rem = rl - i;
            if (rem > 1) w |= (uint32_t)res[i + 1] << 8;
            if (rem > 2) w |= res[i + 2];
            buf_putc(out, B64[(w >> 18) & 63]); buf_putc(out, B64[(w >> 12) & 63]);
            buf_putc(out, rem > 1 ? B64[(w >> 6) & 63] : '='); buf_putc(out, rem > 2 ? B64[w & 63] : '=');
        }
        buf_putc(out, '"');
        *has = 1; return B9O_COMPLETE;
    }
    case H_JSON_SUM: {
        if (a->t != T_OBJ) return B9O_ERROR;                           /* TypeError            */
        val_t *vals = obj_get_last(a, "values");
        if (!vals) return B9O_ERROR;                                   /* KeyError             */
        if (vals->t == T_STR) return vals->slen ? B9O_ERROR : B9O_COMPLETE;   /* sum("") == 0   */
        if (vals->t == T_OBJ) { dedup_obj(vals); return vals->n ? B9O_ERROR : B9O_COMPLETE; }
        if (vals->t != T_ARR) return B9O_ERROR;
        __int128 acc = 0; int any_float = 0;
        for (size_t i = 0; i < vals->n; i++) {
            val_t *x = vals->items[i];
            if (x->t == T_TRUE) { acc += 1; continue; }
            if (x->t == T_FALSE) continue;
            if (x->t != T_NUM) return B9O_ERROR;                       /* TypeError            */
            if (!x->is_int) { any_float = 1; continue; }
            if (x->lit_len > 17) return B9O_UNSUPPORTED;
            acc += (__int128)strtoll((const char *)x->lit, NULL, 10);  /* literal is followed by , or ] */
        }
        if (any_float) return B9O_UNSUPPORTED;
        /* Python's sum is exact; this prints int64. The device decides nothing outside int64 either. */
        if (acc > (__int128)INT64_MAX || acc < (__int128)INT64_MIN) return B9O_UNSUPPORTED;
        if (acc == 0) return B9O_COMPLETE;
        char t[32]; int l = snprintf(t, sizeof t, "%lld", (long long)acc); buf_put(out, t, (size_t)l);
        *has = 1; return B9O_COMPLETE;
    }
    }
    return B9O_ERROR;
}

/* ------------------------------------------------------------------ one task, end to end */
typedef struct { arena_t ar; buf_t wire, res; } scratch_t;

static int run_one(scratch_t *sc, const env_t *env, const uint8_t *id, const uint8_t *p, size_t plen, int handler, int *has) {
    arena_t *ar = &sc->ar;
    ar->used = 0;                       /* reuse the current block; older chained blocks stay allocated */
    sc->wire.len = 0; sc->res.len = 0; *has = 0;
    /* --- gateway: json.Unmarshal(in.Payload, &TaskPayload) */
    val_t *doc = parse_document(p, plen, ar);
    if (!doc) return B9O_REJECTED;
    val_t *args = NULL, *kwargs = NULL; int type_err = 0;
    if (doc->t == T_NULL) { /* no-op */ }
    else if (doc->t != T_OBJ) return B9O_REJECTED;
    else {
        for (size_t i = 0; i < doc->n; i++) {
            val_t *k = doc->keys[i], *v = doc->items[i];
            /* decode.go converts every number of a DECODED value and keeps the first conversion error (saveError):
             * an overflow inside any occurrence of args / kwargs refuses the payload, whatever a later duplicate
             * of the key does. Values of the wrong kind are skipped after the type error, unknown keys too. */
            if (fold_eq(k, "args")) {
                if (v->t == T_NULL) args = NULL; else if (v->t == T_ARR) { args = v; if (has_overflow(v)) type_err = 1; } else type_err = 1;
            } else if (fold_eq(k, "kwargs")) {
                if (v->t == T_NULL) kwargs = NULL;
                else if (v->t == T_OBJ) {
                    if (has_overflow(v)) type_err = 1;
                    if (!kwargs) kwargs = v;
                    else {  /* decoding into a non-nil map keeps existing entries: merge */
                        val_t *m = (val_t *)arena_alloc(ar, sizeof(val_t)); *m = *kwargs;
                        m->n = kwargs->n + v->n;
                        m->keys = (val_t **)arena_alloc(ar, m->n * sizeof(val_t *));
                        m->items = (val_t **)arena_alloc(ar, m->n * sizeof(val_t *));
                        memcpy(m->keys, kwargs->keys, kwargs->n * sizeof(val_t *)); memcpy(m->items, kwargs->items, kwargs->n * sizeof(val_t *));
                        memcpy(m->keys + kwargs->n, v->keys, v->n * sizeof(val_t *)); memcpy(m->items + kwargs->n, v->items, v->n * sizeof(val_t *));
                        kwargs = m;
                    }
                } else type_err = 1;
            }
        }
    }
    if (type_err || has_overflow(args) || has_overflow(kwargs)) return B9O_REJECTED;
    /* --- dispatcher: TaskMessage fill + Encode; client.Push: RPUSH */
    int r = encode_wire(&sc->wire, env, id, args, kwargs, ar);
    if (r) return r;
    /* --- client.Pop: LPOP returns the same bytes; runner: json.loads */
    val_t *msg = parse_document(sc->wire.p, sc->wire.len, ar);
    if (!msg || msg->t != T_OBJ) return B9O_ERROR;   /* cannot happen */
    val_t *pargs = obj_get_last(msg, "args"), *pkw = obj_get_last(msg, "kwargs");
    /* python ints: is_int marks "literal without frac/exp", which parse_number already set */
    return run_handler(handler, pargs, pkw, &sc->res, has, ar);
}

/* ------------------------------------------------------------------ batch API */
/* Every thread owns a contiguous range of the batch and appends its results (and wire records) to its OWN growing
 * buffer: the batch's result blob is then the threads' buffers back to back, moved by one memcpy per thread, in parallel.
 * (Round 1 malloc'ed every result and gathered serially: 8 threads gave 1.2x of one.) */
typedef struct {
    const uint8_t *ids, *payload; const uint64_t *offsets; uint32_t lo, hi; int handler; env_t env;
    uint8_t *status, *has; uint32_t *out_len;
    buf_t out;                                  /* this thread's results, in task order */
    int keep_wire; uint32_t *wire_len; buf_t wire;
    /* second phase: where this thread's bytes go */
    uint8_t *dst_out, *dst_wire; uint64_t base_out, base_wire; uint64_t *out_offsets, *wire_offsets; int over;
} job_t;

static void *worker(void *arg) {
    job_t *j = (job_t *)arg;
    scratch_t sc; memset(&sc, 0, sizeof sc);
    for (uint32_t i = j->lo; i < j->hi; i++) {
        int has = 0;
        int st = run_one(&sc, &j->env, j->ids + 16 * (size_t)i, j->payload + j->offsets[i], (size_t)(j->offsets[i + 1] - j->offsets[i]), j->handler, &has);
        j->status[i] = (uint8_t)st; j->has[i] = (uint8_t)has;
        j->out_len[i] = has ? (uint32_t)sc.res.len : 0;
        if (has && sc.res.len) buf_put(&j->out, sc.res.p, sc.res.len);
        if (j->keep_wire) {
            if (st != B9O_REJECTED && sc.wire.len) { buf_put(&j->wire, sc.wire.p, sc.wire.len); j->wire_len[i] = (uint32_t)sc.wire.len; }
            else j->wire_len[i] = 0;
        }
    }
    arena_free_all(&sc.ar); free(sc.wire.p); free(sc.res.p);
    return NULL;
}

static void *placer(void *arg) {
    job_t *j = (job_t *)arg;
    if (!j->over && j->out.len) memcpy(j->dst_out + j->base_out, j->out.p, j->out.len);
    uint64_t o = j->base_out;
    for (uint32_t i = j->lo; i < j->hi; i++) { o += j->out_len[i]; j->out_offsets[i + 1] = o; }
    if (j->keep_wire) {
        if (!j->over && j->wire.len) memcpy(j->dst_wire + j->base_wire, j->wire.p, j->wire.len);
        uint64_t w = j->base_wire;
        for (uint32_t i = j->lo; i < j->hi; i++) { w += j->wire_len[i]; j->wire_offsets[i + 1] = w; }
    }
    free(j->out.p); free(j->wire.p);
    return NULL;
}

/*
 * Run the reference loop over a packed batch.
 *   ids[n*16], payload blob, offsets[n+1]  : the TaskQueuePut payloads, in put order
 *   out_status[n], out_has[n]              : per task
 *   out_offsets[n+1], out_payload[cap]     : result bytes, FIFO order, zero-length when !has
 *   wire_offsets[n+1], wire_payload[cap]   : optional (NULL to skip): the Redis list element bytes
 * Returns total result bytes, or -1 if out_cap / wire_cap is too small.
 */
int64_t b9o_run_batch(const uint8_t *ids, const uint8_t *payload, const uint64_t *offsets, uint32_t n, int handler,
                      const char *workspace_name, const char *stub_id, uint32_t max_retries, int32_t timeout, uint32_t ttl, int64_t now_unix_ns,
                      uint8_t *out_status, uint8_t *out_has, uint64_t *out_offsets, uint8_t *out_payload, uint64_t out_cap,
                      uint64_t *wire_offsets, uint8_t *wire_payload, uint64_t wire_cap, int nthreads) {
    if (!crc_ready) crc_init();
    if (nthreads < 1) nthreads = 1;
    if ((uint32_t)nthreads > n && n) nthreads = (int)n;
    uint32_t *out_len = (uint32_t *)calloc((size_t)n + 1, sizeof(uint32_t));
    uint32_t *wire_len = wire_offsets ? (uint32_t *)calloc((size_t)n + 1, sizeof(uint32_t)) : NULL;
    job_t *jobs = (job_t *)calloc((size_t)nthreads, sizeof(job_t));
    pthread_t *th = (pthread_t *)calloc((size_t)nthreads, sizeof(pthread_t));
    for (int t = 0; t < nthreads; t++) {
        job_t *j = &jobs[t];
        j->ids = ids; j->payload = payload; j->offsets = offsets; j->handler = handler;
        j->lo = (uint32_t)((uint64_t)n * (uint64_t)t / (uint64_t)nthreads); j->hi = (uint32_t)((uint64_t)n * (uint64_t)(t + 1) / (uint64_t)nthreads);
        j->env.workspace_name = workspace_name; j->env.stub_id = stub_id; j->env.executor = "taskqueue";
        j->env.max_retries = max_retries; j->env.timeout = timeout; j->env.ttl = ttl; j->env.now_unix_ns = now_unix_ns;
        j->status = out_status; j->has = out_has; j->out_len = out_len;
        j->keep_wire = wire_offsets != NULL; j->wire_len = wire_len;
        if (nthreads == 1) worker(j); else pthread_create(&th[t], NULL, worker, j);
    }
    if (nthreads > 1) for (int t = 0; t < nthreads; t++) pthread_join(th[t], NULL);
    uint64_t total = 0, wtotal = 0; int over = 0;
    for (int t = 0; t < nthreads; t++) {
        jobs[t].base_out = total; jobs[t].base_wire = wtotal;
        total += jobs[t].out.len; wtotal += jobs[t].wire.len;
    }
    if (total > out_cap || (wire_offsets && wtotal > wire_cap)) over = 1;
    out_offsets[0] = 0;
    if (wire_offsets) wire_offsets[0] = 0;
    for (int t = 0; t < nthreads; t++) {
        job_t *j = &jobs[t];
        j->dst_out = out_payload; j->dst_wire = wire_payload; j->out_offsets = out_offsets; j->wire_offsets = wire_offsets; j->over = over;
        if (nthreads == 1) placer(j); else pthread_create(&th[t], NULL, placer, j);
    }
    if (nthreads > 1) for (int t = 0; t < nthreads; t++) pthread_join(th[t], NULL);
    free(out_len); free(wire_len); free(jobs); free(th);
    return over ? -1 : (int64_t)total;
}

/* pkg/abstractions/taskqueue/autoscaler.go:53-79 — returns desired, *valid */
int b9o_task_queue_scale(int64_t queue_length, int64_t tasks_per_container, int64_t max_containers, int64_t max_replicas, int *valid) {
    *valid = 1;
    if (queue_length == 0) return 0;
    if (queue_length == -1) { *valid = 0; return 0; }
    int64_t desired = queue_length / tasks_per_container;
    if (queue_length % tasks_per_container > 0) desired++;
    double mr = fmin((double)max_containers, (double)max_replicas);
    return (int)fmin(mr, (double)desired);
}
