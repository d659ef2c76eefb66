// Device bodies of the GPU "kernel handlers" — the user-function slot of the runner loop
// (sdk/src/beta9/runner/common.py:297-305 `FunctionHandler.__call__`, invoked at
// sdk/src/beta9/runner/taskqueue.py:353). Semantics are those of the Python handlers in
// oracle/pyoracle/handlers.py called as handler(*args, **kwargs); every Python exception maps to
// TaskStatus.ERROR (taskqueue.py:354-361) and a falsy result to "no result bytes" (:378).
//
// v1: each of these runs in ONE thread per task (sizing pass = phase A, writing pass = phase B).
#pragma once
#include <stdint.h>
#include "json_device.cuh"

namespace b9 {

// ---------------------------------------------------------------- crc32 (zlib.crc32(s.encode()))
// IEEE 802.3 reflected polynomial 0xEDB88320, init/xorout 0xFFFFFFFF. `table` is the 256-entry
// byte table in shared memory.
__device__ __forceinline__ uint32_t crc_table_entry(uint32_t i) {
    uint32_t c = i;
    #pragma unroll
    for (int k = 0; k < 8; ++k) c = (c & 1u) ? (0xEDB88320u ^ (c >> 1)) : (c >> 1);
    return c;
}
__device__ __forceinline__ uint32_t crc_byte(uint32_t c, uint32_t b, const uint32_t* __restrict__ table) {
    return table[(c ^ b) & 0xFFu] ^ (c >> 8);
}

// CRC over the UTF-8 encoding of the decoded string token p[s..e) (quotes included, validated).
__device__ inline uint32_t crc32_of_string_token(const uint8_t* __restrict__ p, uint32_t s, uint32_t e, uint32_t flags,
                                                 const uint32_t* __restrict__ table) {
    uint32_t c = 0xFFFFFFFFu;
    uint32_t i = s + 1, end = e - 1;
    if (!(flags & SF_ESC)) {
        if (!(flags & SF_NONPRINT)) {                 // decoded bytes == raw bytes
            for (; i < end; ++i) c = crc_byte(c, p[i], table);
            return ~c;
        }
    }
    while (i < end) {
        uint32_t cp = next_cp(p, i, end);
        if (cp < 0x80) c = crc_byte(c, cp, table);
        else if (cp < 0x800) { c = crc_byte(c, 0xC0 | (cp >> 6), table); c = crc_byte(c, 0x80 | (cp & 0x3F), table); }
        else if (cp < 0x10000) {
            c = crc_byte(c, 0xE0 | (cp >> 12), table); c = crc_byte(c, 0x80 | ((cp >> 6) & 0x3F), table); c = crc_byte(c, 0x80 | (cp & 0x3F), table);
        } else {
            c = crc_byte(c, 0xF0 | (cp >> 18), table); c = crc_byte(c, 0x80 | ((cp >> 12) & 0x3F), table);
            c = crc_byte(c, 0x80 | ((cp >> 6) & 0x3F), table); c = crc_byte(c, 0x80 | (cp & 0x3F), table);
        }
    }
    return ~c;
}

// ---------------------------------------------------------------- json_sum (sum(obj["values"]))
// status: 0 ok (value in *sum), 1 ERROR (KeyError / TypeError), 4 UNSUPPORTED (a float in the list, or a partial
// sum outside int64: Python's int is exact there, and the host's CPU loop answers)
__device__ inline bool key_is_values(const uint8_t* __restrict__ p, uint32_t s, uint32_t e) {
    const char V[] = "values";
    uint32_t k = 0, i = s;
    while (i < e) {
        uint32_t cp = next_cp(p, i, e);
        if (k >= 6 || cp != (uint32_t)V[k]) return false;
        ++k;
    }
    return k == 6;
}

__device__ inline int sum_values_token(const uint8_t* __restrict__ p, uint32_t vs, uint32_t ve, long long* sum) {
    // p[vs..ve) is a validated JSON value: the last "values" entry of the object
    *sum = 0;
    uint8_t c = p[vs];
    if (c == '"') return (ve - vs == 2) ? 0 : 1;                  // sum("") == 0; sum("ab") raises
    if (c == '{') return only_ws(p, vs + 1, ve - 1) ? 0 : 1;      // sum({}) == 0; str keys raise
    if (c != '[') return 1;                                        // not iterable
    uint32_t i = vs + 1;
    long long acc = 0; bool unsupported = false;
    while (i < ve && is_ws(p[i])) ++i;
    if (p[i] == ']') return 0;
    for (;;) {
        uint8_t d = p[i];
        if (d == '-' || is_digit(d)) {
            uint32_t f = 0; bool simple = false;
            int64_t e = scan_number(p, i, ve, f, &simple);
            if (simple) {
                bool neg = d == '-'; long long v = 0;
                for (uint32_t k = i + (neg ? 1 : 0); k < (uint32_t)e; ++k) v = v * 10 + (p[k] - '0');
                const long long s = neg ? -v : v;                   // |s| < 10^15: only the add can leave int64
                if (s > 0 ? acc > INT64_MAX - s : acc < INT64_MIN - s) unsupported = true;
                else acc += s;
            } else unsupported = true;                              // needs float64 arithmetic / repr
            i = (uint32_t)e;
        } else if (d == 't') { if (acc == INT64_MAX) unsupported = true; else acc += 1; i += 4; }   // True + 1 == 2
        else if (d == 'f') { i += 5; }
        else return 1;                                             // None / str / list / dict: TypeError
        while (i < ve && is_ws(p[i])) ++i;
        if (p[i] == ',') { ++i; while (i < ve && is_ws(p[i])) ++i; continue; }
        break;                                                     // ']'
    }
    if (unsupported) return 4;
    *sum = acc;
    return 0;
}

// arg token p[s..e) is a non-empty object (validated). Finds the last "values" key.
__device__ inline int json_sum_object(const uint8_t* __restrict__ p, uint32_t s, uint32_t e, long long* sum) {
    uint32_t i = s + 1;
    bool found = false; uint32_t vs = 0, ve = 0;
    for (;;) {
        while (i < e && is_ws(p[i])) ++i;
        uint32_t f = 0;
        uint32_t ks = i;
        i = (uint32_t)scan_string(p, i, e, f);
        bool is_values = key_is_values(p, ks + 1, i - 1);
        while (i < e && is_ws(p[i])) ++i;
        ++i;                                                       // ':'
        while (i < e && is_ws(p[i])) ++i;
        uint32_t v0 = i, f2 = 0;
        i = (uint32_t)skip_value(p, i, e, f2);
        if (is_values) { found = true; vs = v0; ve = i; }          // later duplicates win (Go map)
        while (i < e && is_ws(p[i])) ++i;
        if (p[i] == ',') { ++i; continue; }
        break;                                                     // '}'
    }
    if (!found) return 1;                                          // KeyError
    return sum_values_token(p, vs, ve, sum);
}

// ---------------------------------------------------------------- vadd_f32
__device__ __forceinline__ int b64_val(uint8_t c) {
    if (c >= 'A' && c <= 'Z') return c - 'A';
    if (c >= 'a' && c <= 'z') return c - 'a' + 26;
    if (c >= '0' && c <= '9') return c - '0' + 52;
    if (c == '+') return 62;
    if (c == '/') return 63;
    return -1;
}
__device__ __forceinline__ uint8_t b64_chr(uint32_t v) {
    return (uint8_t)(v < 26 ? 'A' + v : v < 52 ? 'a' + (v - 26) : v < 62 ? '0' + (v - 52) : (v == 62 ? '+' : '/'));
}

// base64.b64decode(x, validate=True) acceptance for the body p[s..e) (no escapes): returns the
// decoded length or -1 (binascii.Error / ValueError -> ERROR).
__device__ inline int64_t b64_decoded_len(const uint8_t* __restrict__ p, uint32_t s, uint32_t e) {
    uint32_t n = e - s;
    if (n % 4) return -1;
    uint32_t pad = 0;
    if (n && p[e - 1] == '=') { pad = 1; if (p[e - 2] == '=') pad = 2; }
    for (uint32_t i = s; i < e - pad; ++i) if (b64_val(p[i]) < 0) return -1;
    return (int64_t)(n / 4) * 3 - pad;
}
// decoded byte j of the base64 body starting at p[s]
__device__ __forceinline__ uint32_t b64_byte(const uint8_t* __restrict__ p, uint32_t s, uint32_t j) {
    uint32_t q = j / 3, r = j - q * 3;
    const uint8_t* c = p + s + 4 * q;
    uint32_t a = (uint32_t)b64_val(c[r]), b = (uint32_t)b64_val(c[r + 1]);   // pad chars are never needed for a valid j
    switch (r) {
    case 0: return ((a << 2) | (b >> 4)) & 0xFF;
    case 1: return ((a << 4) | (b >> 2)) & 0xFF;
    default: return ((a << 6) | b) & 0xFF;
    }
}
__device__ __forceinline__ float b64_f32(const uint8_t* __restrict__ p, uint32_t s, uint32_t byte_off) {
    uint32_t w = b64_byte(p, s, byte_off) | (b64_byte(p, s, byte_off + 1) << 8) | (b64_byte(p, s, byte_off + 2) << 16) | (b64_byte(p, s, byte_off + 3) << 24);
    return __uint_as_float(w);
}
__device__ __forceinline__ uint32_t b64_encoded_len(uint32_t nbytes) { return ((nbytes + 2) / 3) * 4; }

// IEEE-754 binary32 a+b, round-to-nearest-even, as the reference's runner computes it (numpy on x86-64,
// SSE addss): a NaN operand is propagated quieted (the first operand wins), inf + -inf is the x86
// "real indefinite" 0xFFC00000. The GPU's own NaN (0x7FFFFFFF) never reaches the result.
__device__ __forceinline__ uint32_t vadd_bits(uint32_t xb, uint32_t yb) {
    const uint32_t z = __float_as_uint(__fadd_rn(__uint_as_float(xb), __uint_as_float(yb)));
    const bool xn = (xb & 0x7FFFFFFFu) > 0x7F800000u, yn = (yb & 0x7FFFFFFFu) > 0x7F800000u, zn = (z & 0x7FFFFFFFu) > 0x7F800000u;
    return xn ? (xb | 0x00400000u) : yn ? (yb | 0x00400000u) : zn ? 0xFFC00000u : z;
}

// writes '"' + base64(a+b) + '"' for n floats per vector; body = p[s..)
__device__ inline void vadd_write(const uint8_t* __restrict__ p, uint32_t s, uint32_t n, uint8_t* __restrict__ o) {
    *o++ = '"';
    uint32_t acc = 0, have = 0;
    const uint32_t total = 4 * n;
    for (uint32_t i = 0; i < n; ++i) {
        uint32_t z = vadd_bits(__float_as_uint(b64_f32(p, s, 4 * i)), __float_as_uint(b64_f32(p, s, 4 * (n + i))));
        #pragma unroll
        for (int k = 0; k < 4; ++k) {
            acc = (acc << 8) | ((z >> (8 * k)) & 0xFF); ++have;
            if (have == 3) {
                o[0] = b64_chr((acc >> 18) & 63); o[1] = b64_chr((acc >> 12) & 63); o[2] = b64_chr((acc >> 6) & 63); o[3] = b64_chr(acc & 63);
                o += 4; acc = 0; have = 0;
            }
        }
    }
    (void)total;
    if (have == 1) { acc <<= 16; o[0] = b64_chr((acc >> 18) & 63); o[1] = b64_chr((acc >> 12) & 63); o[2] = '='; o[3] = '='; o += 4; }
    else if (have == 2) { acc <<= 8; o[0] = b64_chr((acc >> 18) & 63); o[1] = b64_chr((acc >> 12) & 63); o[2] = b64_chr((acc >> 6) & 63); o[3] = '='; o += 4; }
    *o = '"';
}

}  // namespace b9
