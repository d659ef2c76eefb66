// drain kernel v2 — the production drain (kernel `drain3_kernel` at the bottom of this file).
//
// Persistent workers, ticket work stealing and ballot compaction as in v1 (drain_kernel.cuh), with
// the data path rebuilt around the B200 memory system and every inter-worker dependency removed:
//
//   * the worker is a WARP: own ticket pipeline, own slice of shared memory, own mbarrier, own
//     cursor add; no block barrier in the loop;
//   * a warp-tile's payload bytes are ONE contiguous range of the ring in the common case; lane 0
//     pulls it into the warp's stage buffer with a single bulk async copy (cp.async.bulk / TMA 1-D,
//     completion on the warp's mbarrier);
//   * thread per task for identity and vadd_f32 (G = 1): 16-byte shared loads, SWAR classification of
//     the string body, 16-byte global stores; the whole warp per task for crc32 and json_sum;
//   * result RECORDS (id, status, has, offset, length) are FIFO-dense: record j belongs to the j-th
//     ready task. When no pending task is cancelled (the host knows) j is plain arithmetic on the
//     tile number; otherwise it is read from a ready-count prefix that two small kernels build from the
//     slot flags ahead of the drain (tile_count_kernel / tile_scan_kernel): no tile ever waits on another;
//   * result BYTES are placed by ONE atomicAdd per warp-tile on a byte cursor: dense, but in
//     completion order (v1 chained the byte prefix through an in-order look-back; ncu showed the
//     whole grid in lockstep behind it, 32 tiles resolved per L2 round trip — profiles/r1_v2a_*);
//   * strings with escapes / non-ASCII (the 1 % "adversarial" share, and most of configs[2]) are
//     NOT walked by one lane: the warp splits the body into 32 chunks, every lane finds its first
//     code-unit boundary by a bounded look-behind and transcodes its chunk (esc_* below);
//   * anything that is not the SDK's canonical frame goes through the sequential validating parser
//     (json_device.cuh) — correctness first, it is rare.
//
// Reference behaviour realised: see drain_kernel.cuh's header (pop, decode, loads, call, result).
#pragma once
#include <stdint.h>
#include <type_traits>
#include "drain_kernel.cuh"
#include "vadd_fast.cuh"

namespace b9 {

// ------------------------------------------------------------------ PTX: mbarrier + bulk copy
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) { while (!mbar_try_wait(bar, parity)) {} }
// global -> shared::cta bulk async copy; dst/src 16-byte aligned, bytes a multiple of 16
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// ------------------------------------------------------------------ SWAR classification
// any byte of the four words outside printable ASCII, or equal to '"' or '\\'?
// Exactness: a false positive can only occur in a group that also holds a byte >= 0x80, which is
// "special" anyway (carries out of a byte need a byte >= 0x80 / 0xA0 below them).
__device__ __forceinline__ bool swar_special16(uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
    const uint32_t K1 = 0x01010101u, K60 = 0x60606060u, K7F = 0x7F7F7F7Fu, Q = 0x22222222u, S = 0x5C5C5C5Cu, H = 0x80808080u;
    uint32_t hi = (x | y | z | w) | ((x + K1) | (y + K1) | (z + K1) | (w + K1));          // >= 0x7F
    uint32_t lo = (x + K60) & (y + K60) & (z + K60) & (w + K60);                          // bit7 clear: < 0x20
    uint32_t eq = ((x ^ Q) + K7F) & ((y ^ Q) + K7F) & ((z ^ Q) + K7F) & ((w ^ Q) + K7F)           // bit7 clear: == '"'
                & ((x ^ S) + K7F) & ((y ^ S) + K7F) & ((z ^ S) + K7F) & ((w ^ S) + K7F);          //            == '\\'
    return ((hi | ~lo | ~eq) & H) != 0;
}
__device__ __forceinline__ bool byte_special(uint32_t c) { return c < 0x20u || c >= 0x7Fu || c == '"' || c == '\\'; }

// per-byte 0xFF where the byte's index (0..15 across the four words) is >= lo and < hi
__device__ __forceinline__ uint32_t byte_range_mask(uint32_t word, uint32_t lo, uint32_t hi) {
    const uint32_t idx = 0x03020100u + 0x04040404u * word;
    return __vcmpgeu4(idx, lo * 0x01010101u) & __vcmpltu4(idx, hi * 0x01010101u);
}

// G threads per task (sub = 0..G-1, adjacent lanes): is the payload exactly
//   {"args": ["<body>"], "kwargs": {}}
// with a body of printable ASCII free of '"' and '\\'?  Returns bit0 = frame matches, bit1 = body
// clean, identical on all G lanes. Must be called by all 32 lanes of the warp (`active` masks the
// loads of lanes whose task does not exist).
template <int G>
__device__ __forceinline__ uint32_t quick_clean_framed(const uint8_t* __restrict__ p, uint32_t len, int sub, bool active) {
    uint32_t bad_frame = 0, special = 0;
    if (active && len >= FRAME_PRE_LEN + FRAME_SUF_LEN) {
        // frame: 11 + 17 bytes compared as 32-bit words ("{\"ar" "gs\":" " [\""  /  "\"], " "\"kwa" "rgs\"" ": {}" "}")
        const uint8_t* q = p + len - FRAME_SUF_LEN;
        if (0 % G == sub) bad_frame |= ld_u32_unaligned(p) != 0x7261227Bu;
        if (1 % G == sub) bad_frame |= ld_u32_unaligned(p + 4) != 0x3A227367u;
        if (2 % G == sub) bad_frame |= (ld_u32_unaligned(p + 8) & 0x00FFFFFFu) != 0x00225B20u;
        if (3 % G == sub) bad_frame |= ld_u32_unaligned(q) != 0x202C5D22u;
        if (4 % G == sub) bad_frame |= ld_u32_unaligned(q + 4) != 0x61776B22u;
        if (5 % G == sub) bad_frame |= ld_u32_unaligned(q + 8) != 0x22736772u;
        if (6 % G == sub) bad_frame |= ld_u32_unaligned(q + 12) != 0x7D7B203Au;
        if (7 % G == sub) bad_frame |= q[16] != '}';
        // body = [b0, b1): aligned 16-byte groups, group i handled by lane i % G; bytes of the first /
        // last group outside the body are replaced by 'a' before the SWAR test. (A garbage frame makes
        // the answer irrelevant, but the loads stay inside the payload: len >= 28.)
        const uint8_t* b0 = p + FRAME_PRE_LEN;
        const uint8_t* b1 = q;
        // (pointer - integer keeps the address space the compiler inferred; an integer round trip loses it)
        const uint8_t* g0 = b0 - ((uintptr_t)b0 & 15u);
        const uint8_t* g1 = b1 + ((16u - ((uintptr_t)b1 & 15u)) & 15u);
        const uint32_t lead = (uint32_t)(b0 - g0);                  // bytes to ignore at the front of the first group
        const uint32_t tail_keep = 16u - (uint32_t)(g1 - b1);       // bytes to keep in the last group
        const uint32_t A = 0x61616161u;
        for (const uint8_t* g = g0 + 16 * sub; g < g1; g += 16 * G) {
            uint4 v = *(const uint4*)g;
            const bool first = g == g0, last = g + 16 == g1;
            if (first | last) {
                const uint32_t lo = first ? lead : 0u, hi = last ? tail_keep : 16u;
                uint32_t m;
                m = byte_range_mask(0, lo, hi); v.x = (v.x & m) | (A & ~m);
                m = byte_range_mask(1, lo, hi); v.y = (v.y & m) | (A & ~m);
                m = byte_range_mask(2, lo, hi); v.z = (v.z & m) | (A & ~m);
                m = byte_range_mask(3, lo, hi); v.w = (v.w & m) | (A & ~m);
            }
            special |= swar_special16(v.x, v.y, v.z, v.w) ? 1u : 0u;
        }
    } else bad_frame = 1;
    uint32_t bits = bad_frame | (special << 1);
    #pragma unroll
    for (int d = 1; d < G; d <<= 1) bits |= __shfl_xor_sync(0xffffffffu, bits, d);
    return (bits & 1u ? 0u : 1u) | (bits & 2u ? 0u : 2u);
}

// up to 15 bytes, destination alignment known to allow the 1/2/4/8-byte ladder used by the callers
__device__ __forceinline__ void copy_small_up(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, uint32_t n) {
    // dst + n is 16-byte aligned (head of a copy): ascending sizes keep every store naturally aligned
    uint32_t i = 0;
    if (n & 1u) { dst[0] = src[0]; i = 1; }
    if (n & 2u) { *(uint16_t*)(dst + i) = (uint16_t)(src[i] | (src[i + 1] << 8)); i += 2; }
    if (n & 4u) { *(uint32_t*)(dst + i) = ld_u32_unaligned(src + i); i += 4; }
    if (n & 8u) { *(uint2*)(dst + i) = make_uint2(ld_u32_unaligned(src + i), ld_u32_unaligned(src + i + 4)); }
}
__device__ __forceinline__ void copy_small_down(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, uint32_t n) {
    // dst is 16-byte aligned (tail of a copy): descending sizes
    uint32_t i = 0;
    if (n & 8u) { *(uint2*)(dst) = make_uint2(ld_u32_unaligned(src), ld_u32_unaligned(src + 4)); i = 8; }
    if (n & 4u) { *(uint32_t*)(dst + i) = ld_u32_unaligned(src + i); i += 4; }
    if (n & 2u) { *(uint16_t*)(dst + i) = (uint16_t)(src[i] | (src[i + 1] << 8)); i += 2; }
    if (n & 1u) dst[i] = src[i];
}

// Copy of n bytes to global memory by the G threads of a task: 16-byte stores on the destination
// (vector v by lane v % G), 4-byte loads + funnel shift on the (arbitrarily aligned) source.
template <int G>
__device__ __forceinline__ void group_copy(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, uint32_t n, int sub) {
    uint32_t head = (uint32_t)((16u - ((uintptr_t)dst & 15u)) & 15u);
    if (head > n) {                                              // tiny copy that never reaches an aligned vector
        if (sub == 0) for (uint32_t i = 0; i < n; ++i) dst[i] = src[i];
        return;
    }
    if (sub == 0) copy_small_up(dst, src, head);
    dst += head; src += head; n -= head;
    const uint32_t nvec = n >> 4;
    const uint32_t sh = (uint32_t)((uintptr_t)src & 3u), bits = sh * 8;
    const uint32_t* sw = (const uint32_t*)(src - sh);
    uint4* dv = (uint4*)dst;
    for (uint32_t v = sub; v < nvec; v += G) {
        const uint32_t* s4 = sw + 4 * v;
        const uint32_t w0 = s4[0], w1 = s4[1], w2 = s4[2], w3 = s4[3], w4 = s4[4];   // w4: <= 3 bytes of over-read, inside the buffers' slack
        uint4 o;
        o.x = __funnelshift_r(w0, w1, bits); o.y = __funnelshift_r(w1, w2, bits);
        o.z = __funnelshift_r(w2, w3, bits); o.w = __funnelshift_r(w3, w4, bits);
        dv[v] = o;
    }
    if (sub == G - 1) { const uint32_t done = nvec << 4; copy_small_down(dst + done, src + done, n - done); }
}

// ------------------------------------------------------------------ chunk-parallel string transcoding
// body = the bytes between the frame's quotes. A "unit" is what Go's unquote consumes at once: a
// plain byte, an escape, a \uXXXX (with its low surrogate partner), a UTF-8 sequence.
// four hex digits -> their value, or -1; all four bytes at once (no per-digit branch: the callers sit in
// code that runs one lane per escape)
__device__ __forceinline__ int hex4(const uint8_t* __restrict__ b) {
    const uint32_t w = (uint32_t)b[0] | ((uint32_t)b[1] << 8) | ((uint32_t)b[2] << 16) | ((uint32_t)b[3] << 24);
    const uint32_t H = 0x80808080u;
    const uint32_t x = w & 0x7F7F7F7Fu, y = x | 0x20202020u;
    const uint32_t isd = ((x + 0x50505050u) & ~(x + 0x46464646u)) & H;    // '0' <= x <= '9'
    const uint32_t isl = ((y + 0x1F1F1F1Fu) & ~(y + 0x19191919u)) & H;    // 'a' <= (x | 0x20) <= 'f'
    if ((isd | isl) != H || (w & H)) return -1;
    const uint32_t nib = (x & 0x0F0F0F0Fu) + (isl >> 7) * 9u;
    return (int)(((nib & 0xFu) << 12) | (((nib >> 8) & 0xFu) << 8) | (((nib >> 16) & 0xFu) << 4) | (nib >> 24));
}
__device__ __forceinline__ uint32_t bs_run_before(const uint8_t* __restrict__ b, uint32_t q) {   // backslashes ending at q-1
    uint32_t r = 0;
    while (r < q && b[q - 1 - r] == '\\') ++r;
    return r;
}
// is there a "\uDC00..\uDFFF" escape text at position q?
__device__ __forceinline__ bool low_surrogate_at(const uint8_t* __restrict__ b, uint32_t q, uint32_t n) {
    if (q + 6 > n || b[q] != '\\' || b[q + 1] != 'u') return false;
    int r = hex4(b + q + 2);
    return r >= 0xDC00 && r <= 0xDFFF;
}
__device__ __forceinline__ bool high_surrogate_escape_at(const uint8_t* __restrict__ b, uint32_t q, uint32_t n) {
    if (q + 6 > n || b[q] != '\\' || b[q + 1] != 'u') return false;
    int r = hex4(b + q + 2);
    return r >= 0xD800 && r <= 0xDBFF;
}
__device__ __forceinline__ uint32_t utf8_valid_len(const uint8_t* __restrict__ b, uint32_t q, uint32_t n) {
    // length of the valid UTF-8 sequence starting at q (Go utf8.DecodeRune), or 0
    uint8_t c = b[q]; uint32_t rem = n - q;
    if (c >= 0xC2 && c <= 0xDF) return (rem >= 2 && (b[q + 1] & 0xC0) == 0x80) ? 2u : 0u;
    if (c >= 0xE0 && c <= 0xEF) {
        uint8_t lo = (c == 0xE0) ? 0xA0 : 0x80, hi = (c == 0xED) ? 0x9F : 0xBF;
        return (rem >= 3 && b[q + 1] >= lo && b[q + 1] <= hi && (b[q + 2] & 0xC0) == 0x80) ? 3u : 0u;
    }
    if (c >= 0xF0 && c <= 0xF4) {
        uint8_t lo = (c == 0xF0) ? 0x90 : 0x80, hi = (c == 0xF4) ? 0x8F : 0xBF;
        return (rem >= 4 && b[q + 1] >= lo && b[q + 1] <= hi && (b[q + 2] & 0xC0) == 0x80 && (b[q + 3] & 0xC0) == 0x80) ? 4u : 0u;
    }
    return 0u;
}

// First unit boundary at or after `lo`, decided from a bounded neighbourhood of lo. Exact for a
// body whose escapes are all well-formed; for a malformed body some lane reports !ok and the
// answer is discarded.
__device__ __noinline__ uint32_t first_unit_start(const uint8_t* __restrict__ b, uint32_t n, uint32_t lo) {
    if (lo == 0 || lo >= n) return lo;
    // (1) lo is the character after an escape's backslash
    if (bs_run_before(b, lo) & 1u) {
        uint32_t next = lo + 1;
        if (b[lo] == 'u') {
            next = lo + 5;
            if (high_surrogate_escape_at(b, lo - 1, n) && low_surrogate_at(b, next, n)) next += 6;
        }
        return next;
    }
    // (2) lo is one of the hex digits of a \uXXXX that began 2..5 bytes earlier
    #pragma unroll
    for (uint32_t k = 2; k <= 5; ++k) {
        if (lo >= k) {
            uint32_t q = lo - k;
            if (b[q] == '\\' && b[q + 1] == 'u' && !(bs_run_before(b, q) & 1u)) {
                uint32_t next = q + 6;
                if (high_surrogate_escape_at(b, q, n) && low_surrogate_at(b, next, n)) next += 6;
                return next;
            }
        }
    }
    // (3) lo starts the low-surrogate escape that the high surrogate 6 bytes earlier consumes
    if (lo >= 6 && low_surrogate_at(b, lo, n) && high_surrogate_escape_at(b, lo - 6, n) && !(bs_run_before(b, lo - 6) & 1u))
        return lo + 6;
    // (4) lo is a continuation byte of a valid UTF-8 sequence that began 1..3 bytes earlier
    if ((b[lo] & 0xC0) == 0x80) {
        for (uint32_t k = 1; k <= 3 && k <= lo; ++k) {
            uint8_t c = b[lo - k];
            if ((c & 0xC0) == 0x80) continue;            // another continuation byte: keep looking back
            if (c >= 0xC2) { uint32_t L = utf8_valid_len(b, lo - k, n); if (L > k) return lo - k + L; }
            break;
        }
    }
    return lo;
}

// One unit at b[i] (i < n): advances i, returns the code point Go's unquote yields; *ok = false on
// anything that is not a well-formed JSON string body byte (bad escape, raw control byte, raw '"').
__device__ __noinline__ uint32_t next_unit(const uint8_t* __restrict__ b, uint32_t& i, uint32_t n, bool* ok) {
    uint8_t c = b[i];
    if (c == '\\') {
        if (i + 1 >= n) { *ok = false; ++i; return 0; }
        uint8_t e = b[i + 1];
        if (e == 'u') {
            int r = (i + 6 <= n) ? hex4(b + i + 2) : -1;
            if (r < 0) { *ok = false; i += 2; return 0; }
            i += 6;
            if (r >= 0xD800 && r <= 0xDFFF) {
                if (r <= 0xDBFF && i + 6 <= n && b[i] == '\\' && b[i + 1] == 'u') {
                    int r1 = hex4(b + i + 2);
                    if (r1 >= 0xDC00 && r1 <= 0xDFFF) { i += 6; return 0x10000u + (((uint32_t)r - 0xD800u) << 10) + ((uint32_t)r1 - 0xDC00u); }
                }
                return 0xFFFDu;
            }
            return (uint32_t)r;
        }
        i += 2;
        switch (e) {
        case '"': case '\\': case '/': return e;
        case 'b': return 8; case 'f': return 12; case 'n': return 10; case 'r': return 13; case 't': return 9;
        default: *ok = false; return 0;
        }
    }
    if (c < 0x20 || c == '"') { *ok = false; ++i; return 0; }
    if (c < 0x80) { ++i; return c; }
    uint32_t L = utf8_valid_len(b, i, n);
    if (!L) { ++i; return 0xFFFDu; }
    uint32_t cp;
    if (L == 2) cp = ((c & 0x1Fu) << 6) | (b[i + 1] & 0x3Fu);
    else if (L == 3) cp = ((c & 0x0Fu) << 12) | ((b[i + 1] & 0x3Fu) << 6) | (b[i + 2] & 0x3Fu);
    else cp = ((c & 0x07u) << 18) | ((b[i + 1] & 0x3Fu) << 12) | ((b[i + 2] & 0x3Fu) << 6) | (b[i + 3] & 0x3Fu);
    i += L;
    return cp;
}

__device__ __forceinline__ uint32_t warp_sum(uint32_t v) {
    #pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    return v;
}
__device__ __forceinline__ uint32_t warp_excl_scan(uint32_t v, int lane) {
    uint32_t inc = v;
    #pragma unroll
    for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t; }
    return inc - v;
}

__device__ __forceinline__ bool plain_byte(uint32_t c) { return c >= 0x20u && c < 0x7Fu && c != '"' && c != '\\'; }
// bit 7 of every byte of w that is NOT a plain byte (same exactness argument as swar_special16)
__device__ __forceinline__ uint32_t special_mask32(uint32_t w) {
    const uint32_t K1 = 0x01010101u, K60 = 0x60606060u, K7F = 0x7F7F7F7Fu, H = 0x80808080u;
    return ((w + K1) | w | ~(w + K60) | ~((w ^ 0x22222222u) + K7F) | ~((w ^ 0x5C5C5C5Cu) + K7F)) & H;
}
// any 'A'..'F' among the four hex digits of a \uXXXX (digits have bit 6 clear, a..f have bit 5 set)
__device__ __forceinline__ bool hex_has_upper(uint32_t w) { return ((w & 0x40404040u) & ~((w & 0x20202020u) << 1)) != 0; }

// What one lane learned about its chunk of an escaped string body.
struct EscLane {
    uint32_t start;        // first unit boundary at or after the chunk start
    uint32_t out_len;      // json.dumps bytes produced by the chunk's units
    uint32_t npatch;       // same-length units whose text must be rewritten (lone surrogate -> �, upper-case hex)
    uint32_t patch_pos[2]; // body offsets of those units
    uint32_t patch_cp[2];
    bool ok;               // chunk is well-formed JSON string text
    bool len_change;       // some unit's json.dumps form has another length than its input text
};

// Warp-cooperative scan of a framed string body: plain bytes are skipped four at a time, only
// escapes / non-ASCII bytes go through the unit decoder. Returns false if the body is not a
// well-formed JSON string ending at the frame's closing quote. *out_len = 2 + sum of units.
// *fast = every unit keeps its length (true for everything json.dumps itself produced): then
// json.dumps(body) is the input text with at most a few same-length patches.
__device__ __noinline__ bool esc_scan(const uint8_t* __restrict__ body, uint32_t n, int lane, EscLane& L, uint32_t* out_len, bool* fast) {
    const uint32_t S = (n + 31u) / 32u;
    const uint32_t lo = min(n, (uint32_t)lane * S), hi = min(n, lo + S);
    L.start = lo; L.out_len = 0; L.npatch = 0; L.ok = true; L.len_change = false;
    L.patch_pos[0] = L.patch_pos[1] = 0; L.patch_cp[0] = L.patch_cp[1] = 0;
    if (lo < hi) {
        uint32_t i = first_unit_start(body, n, lo);
        L.start = i;
        uint32_t mine = 0;
        while (i < hi) {
            // run of plain bytes: four at a time (reading up to 3 bytes past hi is inside the payload: the frame suffix follows)
            bool stop = false;
            while (i < hi) {
                const uint32_t m = special_mask32(ld_u32_unaligned(body + i));
                const uint32_t adv = m ? (uint32_t)(__ffs(m) - 1) >> 3 : 4u;
                const uint32_t take = min(adv, hi - i);
                i += take; mine += take;
                if (adv < 4u || i >= hi) { stop = true; break; }
            }
            (void)stop;
            if (i >= hi) break;
            const uint32_t i0 = i;
            const uint32_t cp = next_unit(body, i, n, &L.ok);
            if (!L.ok) break;
            const uint32_t ol = py_escaped_len(cp), il = i - i0;
            mine += ol;
            if (ol != il) L.len_change = true;
            else if (il >= 6u) {                                      // \uXXXX or a surrogate pair, same length: is the text already canonical?
                bool differs = cp == 0xFFFDu || hex_has_upper(ld_u32_unaligned(body + i0 + 2));
                if (il == 12u) differs |= hex_has_upper(ld_u32_unaligned(body + i0 + 8));
                if (differs) {
                    if (L.npatch < 2u) { L.patch_pos[L.npatch] = i0; L.patch_cp[L.npatch] = cp; }
                    ++L.npatch;
                }
            }
        }
        L.out_len = mine;
    }
    const bool ok = __all_sync(0xffffffffu, L.ok);
    *out_len = 2u + warp_sum(L.out_len);
    *fast = __all_sync(0xffffffffu, !L.len_change && L.npatch <= 2u);
    return ok;
}

// fast emit: the token itself, then the same-length patches
__device__ __forceinline__ void esc_emit_fast(const uint8_t* __restrict__ token, uint32_t tok_len, int lane, uint8_t* __restrict__ dst, const EscLane& L) {
    warp_copy(dst, token, tok_len, lane);
    __syncwarp();
    for (uint32_t q = 0; q < L.npatch && q < 2u; ++q) py_emit(L.patch_cp[q], dst + 1 + L.patch_pos[q]);
}

// general emit (units change length): every lane re-walks its chunk and writes at its scanned offset
__device__ __noinline__ void esc_emit_general(const uint8_t* __restrict__ body, uint32_t n, int lane, uint8_t* __restrict__ dst, const EscLane& L) {
    const uint32_t S = (n + 31u) / 32u;
    const uint32_t lo = min(n, (uint32_t)lane * S), hi = min(n, lo + S);
    bool ok = true;
    const uint32_t at = 1u + warp_excl_scan(L.out_len, lane);
    if (lane == 0) dst[0] = '"';
    if (lane == 31) dst[at + L.out_len] = '"';
    if (lo < hi) {
        uint8_t* o = dst + at;
        uint32_t i = L.start;
        while (i < hi) {
            while (i < hi) { const uint32_t c = body[i]; if (!plain_byte(c)) break; *o++ = (uint8_t)c; ++i; }
            if (i >= hi) break;
            o += py_emit(next_unit(body, i, n, &ok), o);
        }
    }
}

// ------------------------------------------------------------------ warp-cooperative CRC-32 of a framed string
// zlib.crc32(s.encode()) over the DECODED bytes, 32 chunks in parallel. With R(c, b) the reflected
// table step and r_l the register after lane l's decoded bytes (lane 0 starts from 0xFFFFFFFF, the
// others from 0), linearity gives
//   R*(0xFFFFFFFF, B_0 || ... || B_31) = XOR_l Z(r_l, bytes after lane l)
// where Z(c, n) advances the register over n zero bytes. Z for n = 2^k is a fixed linear map, kept as
// 4 x 256-entry byte tables per k (`shift_tabs`, built on the host): a shift costs 4 loads per set bit.
constexpr int CRC_SHIFT_LEVELS = 32;         // any 32-bit byte count (128 KiB of tables, L2-resident)
__device__ __forceinline__ uint32_t crc_zero_shift(uint32_t c, uint32_t nbytes, const uint32_t* __restrict__ shift_tabs) {
    // every lane walks the same levels (up to the warp's highest set bit) and applies its own: no divergence
    const uint32_t levels = 32u - __clz(__reduce_or_sync(0xffffffffu, nbytes));
    for (uint32_t k = 0; k < levels; ++k) {
        const uint32_t* t = shift_tabs + (size_t)k * 1024;
        const uint32_t s = __ldg(t + (c & 0xFFu)) ^ __ldg(t + 256 + ((c >> 8) & 0xFFu)) ^ __ldg(t + 512 + ((c >> 16) & 0xFFu)) ^ __ldg(t + 768 + (c >> 24));
        c = ((nbytes >> k) & 1u) ? s : c;
    }
    return c;
}

// Explicit shared-window loads for the byte loop: 32-bit addresses, no generic-pointer arithmetic per byte.
__device__ __forceinline__ uint32_t lds_u8(uint32_t a) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
struct LdShared  { uint32_t base;   __device__ __forceinline__ uint32_t operator()(uint32_t i) const { return lds_u8(base + i); } };
struct LdGeneric { const uint8_t* p; __device__ __forceinline__ uint32_t operator()(uint32_t i) const { return p[i]; } };
__device__ __forceinline__ uint32_t crc_step(uint32_t r, uint32_t b, uint32_t tab_s) { return lds_u32(tab_s + (((r ^ b) & 0xFFu) << 2)) ^ (r >> 8); }

// returns false when the body is not a well-formed JSON string body (caller falls back to the sequential parser).
// `ld(i)` reads body byte i (shared window or generic); `body` is the same memory as a generic pointer for the
// rare out-of-line helpers; `tab_s` is the shared-window address of the 256-entry CRC table.
template <class LD>
__device__ __forceinline__ bool crc_scan_coop(LD ld, const uint8_t* __restrict__ body, uint32_t n, int lane, uint32_t tab_s,
                                              const uint32_t* __restrict__ shift_tabs, uint32_t* crc_out) {
    const uint32_t S = (n + 31u) / 32u;
    const uint32_t lo = min(n, (uint32_t)lane * S), hi = min(n, lo + S);
    bool ok = true;
    uint32_t r = lane == 0 ? 0xFFFFFFFFu : 0u, dec = 0;                   // lane 0 carries the register's start value
    if (lo < hi) {
        // a chunk that starts on a plain byte with no backslash among the five bytes before it (the reach of
        // a \uXXXX escape) starts on a unit boundary; anything else takes the general look-behind
        uint32_t i = lo;
        if (lo) {
            bool easy = plain_byte(ld(lo));
            #pragma unroll
            for (uint32_t k = 1; k <= 5; ++k) easy = easy && (lo < k || ld(lo - k) != '\\');
            if (!easy) i = first_unit_start(body, n, lo);
        }
        uint32_t c = i < hi ? ld(i) : 0u;
        while (i < hi) {
            // plain byte, or one of the two-byte escapes json.dumps writes for '"' and '\\' (and "\/"): no branch
            const uint32_t e = ld(i + 1u);                                 // i + 1 <= n: the frame suffix follows the body
            const uint32_t bs = c == '\\';
            const uint32_t simple = bs & ((e == '"') | (e == '\\') | (e == '/'));
            const uint32_t plain = (c - 0x20u < 0x5Fu) & (c != '"') & (bs ^ 1u);
            if (plain | simple) {
                const uint32_t e2 = ld(i + 2u);                            // (unconditional: cheaper than a branch; <= n + 1, inside the frame suffix)
                r = crc_step(r, simple ? e : c, tab_s); ++dec;
                c = simple ? e2 : e;                                       // the look-ahead byte is the next byte
                i += 1u + simple;
                continue;
            }
            uint32_t ii = i;                                               // (by reference: keep the loop counter in a register)
            const uint32_t cp = next_unit(body, ii, n, &ok);
            i = ii;
            if (!ok) break;
            if (cp < 0x80) { r = crc_step(r, cp, tab_s); dec += 1; }
            else if (cp < 0x800) { r = crc_step(r, 0xC0 | (cp >> 6), tab_s); r = crc_step(r, 0x80 | (cp & 0x3F), tab_s); dec += 2; }
            else if (cp < 0x10000) {
                r = crc_step(r, 0xE0 | (cp >> 12), tab_s); r = crc_step(r, 0x80 | ((cp >> 6) & 0x3F), tab_s); r = crc_step(r, 0x80 | (cp & 0x3F), tab_s); dec += 3;
            } else {
                r = crc_step(r, 0xF0 | (cp >> 18), tab_s); r = crc_step(r, 0x80 | ((cp >> 12) & 0x3F), tab_s);
                r = crc_step(r, 0x80 | ((cp >> 6) & 0x3F), tab_s); r = crc_step(r, 0x80 | (cp & 0x3F), tab_s); dec += 4;
            }
            c = ld(i);                                                     // i <= n: at worst the closing quote
        }
    }
    if (!__all_sync(0xffffffffu, ok)) return false;
    const uint32_t before = warp_excl_scan(dec, lane);
    const uint32_t total = __shfl_sync(0xffffffffu, before + dec, 31);
    uint32_t v = crc_zero_shift(r, total - before - dec, shift_tabs);
    #pragma unroll
    for (int d = 16; d > 0; d >>= 1) v ^= __shfl_xor_sync(0xffffffffu, v, d);
    *crc_out = ~v;
    return true;
}

template <int HANDLER> __device__ __noinline__ void d2_parse_and_size(const uint8_t* p, uint32_t len, TaskRec& rec, const uint32_t* crc_table, bool http = false);
// one crc32 task with the whole warp; the owner lane keeps the record. `in_smem`: p points into this warp's stage buffer.
__device__ __forceinline__ void crc_task_coop(const uint8_t* __restrict__ p, bool in_smem, uint32_t len, int lane, bool owner, const uint32_t* crc_table,
                                              const uint32_t* __restrict__ shift_tabs, TaskRec& rec) {
    bool framed = len >= FRAME_PRE_LEN + FRAME_SUF_LEN;
    if (framed) {
        bool okb = true;
        if (lane < (int)FRAME_PRE_LEN) okb = p[lane] == FRAME_PRE[lane];
        else if (lane < (int)(FRAME_PRE_LEN + FRAME_SUF_LEN)) okb = p[len - FRAME_SUF_LEN + (lane - FRAME_PRE_LEN)] == FRAME_SUF[lane - FRAME_PRE_LEN];
        framed = __all_sync(0xffffffffu, okb);
    }
    uint32_t crc = 0; bool done = false;
    if (framed) {
        const uint8_t* body = p + FRAME_PRE_LEN;
        const uint32_t n = len - FRAME_PRE_LEN - FRAME_SUF_LEN;
        uint32_t tab_s = smem_u32(crc_table);
        asm volatile("mov.u32 %0, %0;" : "+r"(tab_s));                     // keep the address in a register (ptxas re-derives it per use otherwise)
        if (in_smem) { LdShared ld; ld.base = smem_u32(body); done = crc_scan_coop(ld, body, n, lane, tab_s, shift_tabs, &crc); }
        else         { LdGeneric ld; ld.p = body;             done = crc_scan_coop(ld, body, n, lane, tab_s, shift_tabs, &crc); }
    }
    if (owner) {
        if (done) { if (crc) { rec.value = (long long)crc; rec.out_len = dec_len_u64(crc); rec.mode = OM_U32_DEC; rec.has = 1; } }
        else d2_parse_and_size<1>(p, len, rec, crc_table);
    }
}

// A task of a tile that was not staged as a whole (the tile did not fit, or wraps the ring): pull this one
// task into the warp's stage buffer with 16-byte loads. Returns the task's address there, or nullptr if
// even the single task is larger than the buffer.
__device__ __forceinline__ const uint8_t* stage_one_task(const uint8_t* __restrict__ payload, uint64_t goff, uint32_t len, uint8_t* sbuf, uint32_t in_cap, int lane) {
    const uint32_t mis = (uint32_t)(goff & 15ull);
    if (mis + len + 16u > in_cap) return nullptr;
    const uint4* src = (const uint4*)(payload + goff - mis);
    uint4* dst = (uint4*)sbuf;
    const uint32_t nv = (mis + len + 15u) >> 4;
    __syncwarp();                                                          // everybody is done with the previous task's bytes
    for (uint32_t v = lane; v < nv; v += 32) dst[v] = __ldg(src + v);
    __syncwarp();
    return sbuf + mis;
}

// ------------------------------------------------------------------ json_sum, one task per warp, bit-parallel
// configs[4]: `{"args": [DOC], "kwargs": {}}` with DOC a flat JSON object as json.dumps writes it
// (members `"key": value`, values = non-negative integers, strings without escapes, arrays of integers;
// one optional space after ',' and ':'). Lane r owns bytes [32r, 32r+32) of DOC (DOC <= 1 KiB):
//   1. every byte -> a 4-bit class through a table in shared memory, gathered into four 32-bit planes;
//   2. strings, brackets and separators by prefix-XOR of the class masks (simdjson's stage 1, per warp);
//   3. the grammar as look-behind rules on those masks (each byte against its predecessor token);
//   4. the last "values" key, its array span, and a Horner walk of each lane's own digits.
// Anything the rules do not accept (escapes, non-ASCII, floats, negatives, nesting, literals, > 15 digits,
// other whitespace, no "values" array) is NOT decided here: the caller runs the sequential parser.
enum JsonCls : uint8_t { JC_NONE = 0, JC_QUOTE = 1, JC_DIGIT = 2, JC_COMMA = 3, JC_COLON = 4, JC_SPACE = 5, JC_OB = 6, JC_CB = 7,
                         JC_LB = 8, JC_RB = 9, JC_OTHER = 10, JC_ZERO = 11, JC_BAD = 15 };
__device__ __forceinline__ uint8_t json_cls_of(uint32_t c) {
    if (c < 0x20u || c >= 0x7Fu || c == '\\') return JC_BAD;
    switch (c) {
    case '"': return JC_QUOTE; case ',': return JC_COMMA; case ':': return JC_COLON; case ' ': return JC_SPACE;
    case '[': return JC_OB; case ']': return JC_CB; case '{': return JC_LB; case '}': return JC_RB; case '0': return JC_ZERO;
    default: return (c >= '1' && c <= '9') ? JC_DIGIT : JC_OTHER;
    }
}
__device__ __forceinline__ uint32_t prefix_xor32(uint32_t x) { x ^= x << 1; x ^= x << 2; x ^= x << 4; x ^= x << 8; x ^= x << 16; return x; }
__device__ __forceinline__ uint32_t lane_prev(uint32_t m, int lane) { const uint32_t v = __shfl_up_sync(0xffffffffu, m, 1); return lane ? v : 0u; }
// the mask of the lane below; lane 0 gets `carry` (the last lane's mask of the previous segment). Every lane executes the shuffle.
__device__ __forceinline__ uint32_t lane_prev_carry(uint32_t m, int lane, uint32_t carry) { const uint32_t v = __shfl_up_sync(0xffffffffu, m, 1); return lane ? v : carry; }
// parity of `bit` over the lanes below this one
__device__ __forceinline__ uint32_t parity_below(bool bit, int lane) { return __popc(__ballot_sync(0xffffffffu, bit) & ((1u << lane) - 1u)) & 1u; }

constexpr uint32_t JSON_COOP_MAX_SEG = 4;                              // segments of 32 lanes x 32 bytes
constexpr uint32_t JSON_COOP_MAX_DOC = 1024 * JSON_COOP_MAX_SEG;
constexpr uint32_t JSON_PRE_LEN = FRAME_PRE_LEN - 1, JSON_SUF_LEN = FRAME_SUF_LEN - 1;     // the frame without the string quotes

// 32 bytes at q (any alignment) as eight little-endian words; reads up to 7 bytes past them
__device__ __forceinline__ void json_load32(const uint8_t* __restrict__ q, uint32_t w[8]) {
    const uint32_t mis = (uint32_t)((uintptr_t)q & 3u);
    const uint32_t* qa = (const uint32_t*)(q - mis);
    uint32_t t[9];
    #pragma unroll
    for (int i = 0; i < 9; ++i) t[i] = qa[i];
    #pragma unroll
    for (int i = 0; i < 8; ++i) w[i] = __funnelshift_r(t[i], t[i + 1], 8u * mis);
}
__device__ __forceinline__ uint32_t sel4(uint32_t i, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3) { return i == 0 ? a0 : i == 1 ? a1 : i == 2 ? a2 : a3; }

// 1 = decided (*sum_out valid, task COMPLETE), 0 = not decided. MULTI = false is the instance for documents of
// one segment (<= 1 KiB, the configuration's shape): no carries, and the words stay in registers for the second pass.
template <bool MULTI>
__device__ __forceinline__ int json_sum_coop(const uint8_t* __restrict__ p, uint32_t len, int lane, const uint8_t* cls_tab,
                                             unsigned long long* sum_out) {
    if (len < JSON_PRE_LEN + JSON_SUF_LEN + 2u || len - JSON_PRE_LEN - JSON_SUF_LEN > (MULTI ? JSON_COOP_MAX_DOC : 1024u)) return 0;
    bool okb = true;
    if (lane < (int)JSON_PRE_LEN) okb = p[lane] == FRAME_PRE[lane];
    else if (lane < (int)(JSON_PRE_LEN + JSON_SUF_LEN)) okb = p[len - JSON_SUF_LEN + (lane - JSON_PRE_LEN)] == FRAME_SUF[1 + lane - JSON_PRE_LEN];
    if (!__all_sync(0xffffffffu, okb)) return 0;
    const uint8_t* const D = p + JSON_PRE_LEN;
    const uint32_t n = len - JSON_PRE_LEN - JSON_SUF_LEN;
    const uint32_t nseg = MULTI ? (n + 1023u) >> 10 : 1u;
    const uint32_t last = n - 1u;
    uint32_t wk[8];                                                     // !MULTI: my chunk's words, kept for the second pass
    #pragma unroll
    for (int i = 0; i < 8; ++i) wk[i] = 0;
    #define B9_P1(M, PM) (((M) << 1) | ((PM) >> 31))
    #define B9_P2(M, PM) (((M) << 2) | ((PM) >> 30))

    // state carried from one 1 KiB segment to the next (the same in every lane)
    uint32_t c_quote = 0, c_br = 0, c_sep = 0;                          // parities so far
    uint32_t l_closeq = 0, l_openq = 0, l_dg = 0, l_zr = 0, l_cm = 0, l_cl = 0, l_sp = 0, l_ob = 0, l_cb = 0;   // lane 31's masks of the previous segment
    uint32_t dg0 = 0, dg1 = 0, dg2 = 0, dg3 = 0, cb0 = 0, cb1 = 0, cb2 = 0, cb3 = 0;   // per segment, for the second pass
    uint32_t v = 0;                                                     // violations, any lane, any bit
    int bestJ = -1;

    for (uint32_t seg = 0; seg < nseg; ++seg) {
        const uint32_t base = (seg << 10) + 32u * (uint32_t)lane;       // my chunk's first byte in the document
        const uint32_t cnt = base < n ? min(32u, n - base) : 0u;
        const uint32_t inr = cnt == 32u ? 0xFFFFFFFFu : ((1u << cnt) - 1u);
        // ---- 1. my 32 bytes -> class planes
        uint32_t b0 = 0, b1 = 0, b2 = 0, b3 = 0;
        if (cnt) {
            uint32_t w[8];
            json_load32(D + base, w);                                   // (over-read: frame suffix / stage slack)
            if (!MULTI) {
                #pragma unroll
                for (int i = 0; i < 8; ++i) wk[i] = w[i];
            }
            #pragma unroll
            for (int j = 0; j < 32; ++j) {
                const uint32_t cls = cls_tab[(w[j >> 2] >> (8 * (j & 3))) & 0xFFu];
                b0 = __funnelshift_r(b0, cls, 1); b1 = __funnelshift_r(b1, cls >> 1, 1);
                b2 = __funnelshift_r(b2, cls >> 2, 1); b3 = __funnelshift_r(b3, cls >> 3, 1);
            }
            b0 &= inr; b1 &= inr; b2 &= inr; b3 &= inr;
        }
        const uint32_t Q = ~b3 & ~b2 & ~b1 & b0, DG9 = ~b3 & ~b2 & b1 & ~b0, CM = ~b3 & ~b2 & b1 & b0, CL = ~b3 & b2 & ~b1 & ~b0;
        const uint32_t SP = ~b3 & b2 & ~b1 & b0, OB = ~b3 & b2 & b1 & ~b0, CB = ~b3 & b2 & b1 & b0, LB = b3 & ~b2 & ~b1 & ~b0;
        const uint32_t RB = b3 & ~b2 & ~b1 & b0, OTH = b3 & ~b2 & b1 & ~b0, ZR = b3 & ~b2 & b1 & b0, BAD = b3 & b2;
        v |= BAD;

        // ---- 2. strings / arrays / object-level separators
        const uint32_t qinc = prefix_xor32(Q) ^ ((parity_below(__popc(Q) & 1u, lane) ^ c_quote) ? 0xFFFFFFFFu : 0u);   // quotes in [0, i], parity
        const uint32_t OPENQ = Q & qinc, CLOSEQ = Q & ~qinc;
        const uint32_t out = ~(qinc & ~Q) & inr;                        // not string content
        v |= OTH & out;
        const uint32_t dg = (DG9 | ZR) & out, zr = ZR & out, cm = CM & out, cl = CL & out, sp = SP & out;
        const uint32_t ob = OB & out, cb = CB & out, lb = LB & out, rb = RB & out;
        const uint32_t br = ob | cb;
        const uint32_t binc = prefix_xor32(br) ^ ((parity_below(__popc(br) & 1u, lane) ^ c_br) ? 0xFFFFFFFFu : 0u);
        v |= (ob & ~binc) | (cb & binc);                                // '[' opens at depth 0 only, ']' closes
        const uint32_t arr = binc & ~ob & inr;                          // strictly inside an array
        v |= cl & arr;
        const uint32_t sep = (cm | cl) & ~arr;
        const uint32_t sinc = prefix_xor32(sep) ^ ((parity_below(__popc(sep) & 1u, lane) ^ c_sep) ? 0xFFFFFFFFu : 0u);
        v |= (cl & ~sinc) | (cm & ~arr & sinc);                         // object level: ':' ',' ':' ',' ... ':'
        c_quote ^= __popc(__ballot_sync(0xffffffffu, __popc(Q) & 1u)) & 1u;
        c_br ^= __popc(__ballot_sync(0xffffffffu, __popc(br) & 1u)) & 1u;
        c_sep ^= __popc(__ballot_sync(0xffffffffu, __popc(sep) & 1u)) & 1u;

        // ---- 3. the grammar, each byte against its predecessor (one optional space after ',' ':')
        #define B9_PREV(M, LM) lane_prev_carry((M), lane, (LM))
        const uint32_t p_closeq = B9_PREV(CLOSEQ, l_closeq), p_openq = B9_PREV(OPENQ, l_openq), p_dg = B9_PREV(dg, l_dg), p_zr = B9_PREV(zr, l_zr);
        const uint32_t p_cm = B9_PREV(cm, l_cm), p_cl = B9_PREV(cl, l_cl), p_sp = B9_PREV(sp, l_sp);
        const uint32_t p_ob = B9_PREV(ob, l_ob), p_cb = B9_PREV(cb, l_cb);
        #undef B9_PREV
        const uint32_t a_closeq = B9_P1(CLOSEQ, p_closeq), a_dg = B9_P1(dg, p_dg), a_cm = B9_P1(cm, p_cm), a_cl = B9_P1(cl, p_cl);
        const uint32_t a_sp = B9_P1(sp, p_sp), a_ob = B9_P1(ob, p_ob), a_cb = B9_P1(cb, p_cb), a_zr = B9_P1(zr, p_zr);
        const uint32_t a_lb = (lb << 1);                                // '{' is byte 0 (checked below): never a chunk's last byte
        const uint32_t t_cm = a_cm | (a_sp & B9_P2(cm, p_cm)), t_cl = a_cl | (a_sp & B9_P2(cl, p_cl));   // previous token, through the space
        const uint32_t ds = dg & ~a_dg;                                 // first digit of a number
        v |= sp & ~(a_cm | a_cl);
        v |= a_closeq & inr & ~(cl | cm | rb);
        v |= a_dg & inr & ~dg & ~(cm | cb | rb);
        v |= a_cb & inr & ~(cm | rb);
        v |= dg & a_zr & ~B9_P2(dg, p_dg);                              // a digit after a leading zero
        v |= OPENQ & (arr | ~(a_lb | t_cm | t_cl));
        v |= cl & ~a_closeq;
        v |= cm & ~arr & ~(a_closeq | a_dg | a_cb);
        v |= cm & arr & ~a_dg;
        v |= ob & ~t_cl;
        v |= cb & ~(a_ob | a_dg);
        v |= ds & ((arr & ~(a_ob | t_cm)) | (~arr & ~t_cl));
        v |= lb ^ (base == 0u ? 1u : 0u);                               // exactly one '{', at byte 0
        const uint32_t lastbit = (last >= base && last < base + 32u) ? (1u << (last - base)) : 0u;
        v |= rb ^ lastbit;                                              // exactly one '}', at byte n-1
        v |= rb & ~(a_lb | a_closeq | a_dg | a_cb);
        if (rb && !(rb & a_lb) && !c_sep) v |= 1u;                      // a non-empty object ends after "key": value
        {   // a run of 16 or more digits lies inside some (previous chunk, this chunk) window
            unsigned long long x = ((unsigned long long)dg << 32) | p_dg;
            x &= x >> 1; x &= x >> 2; x &= x >> 4; x &= x >> 8;
            v |= x != 0ull ? 1u : 0u;
        }
        // ---- 4a. the last `"values":` key so far: ':' at J, '"' at J-1 and J-8
        uint32_t cand = cl & a_closeq & ((OPENQ << 8) | (p_openq >> 24));
        while (cand) {
            const int j = 31 - __clz(cand);
            const uint8_t* k = D + base + j - 7;
            if (k[0] == 'v' && k[1] == 'a' && k[2] == 'l' && k[3] == 'u' && k[4] == 'e' && k[5] == 's') { bestJ = max(bestJ, (int)base + j); break; }
            cand &= ~(1u << j);
        }
        if (seg == 0) { dg0 = dg; cb0 = cb; } else if (seg == 1) { dg1 = dg; cb1 = cb; } else if (seg == 2) { dg2 = dg; cb2 = cb; } else { dg3 = dg; cb3 = cb; }
        l_closeq = __shfl_sync(0xffffffffu, CLOSEQ, 31); l_openq = __shfl_sync(0xffffffffu, OPENQ, 31); l_dg = __shfl_sync(0xffffffffu, dg, 31);
        l_zr = __shfl_sync(0xffffffffu, zr, 31); l_cm = __shfl_sync(0xffffffffu, cm, 31); l_cl = __shfl_sync(0xffffffffu, cl, 31);
        l_sp = __shfl_sync(0xffffffffu, sp, 31); l_ob = __shfl_sync(0xffffffffu, ob, 31); l_cb = __shfl_sync(0xffffffffu, cb, 31);
    }
    if (__any_sync(0xffffffffu, v != 0u) || c_quote || c_br) return 0;
    bestJ = __reduce_max_sync(0xffffffffu, bestJ);
    if (bestJ < 0) return 0;                                            // KeyError is the sequential path's to report
    uint32_t vs = (uint32_t)bestJ + 1u;
    if (D[vs] == ' ') ++vs;
    if (D[vs] != '[') return 0;                                         // sum() of a non-list
    uint32_t ve = 0xFFFFFFFFu;
    for (uint32_t seg = 0; seg < nseg; ++seg) {
        const uint32_t base = (seg << 10) + 32u * (uint32_t)lane;
        const uint32_t after = vs >= base + 32u ? 0u : (vs < base ? 0xFFFFFFFFu : (vs - base == 31u ? 0u : (0xFFFFFFFFu << (vs - base + 1u))));
        const uint32_t cb_after = (MULTI ? sel4(seg, cb0, cb1, cb2, cb3) : cb0) & after;
        if (cb_after) ve = min(ve, base + (uint32_t)(__ffs(cb_after) - 1));
    }
    ve = __reduce_min_sync(0xffffffffu, ve);

    // ---- 4b. Horner over the numbers that START in my chunk (a number cut by the chunk end is finished from
    // the next chunk's words); no data-dependent branch: run ends, the span and my head digits are masks.
    // No overflow check: a document of <= JSON_COOP_MAX_DOC = 4096 bytes spends 11 on `{"values":[` and 2 on `]}`; a
    // value of d <= 15 digits (< 10^d) takes d + 1 bytes with its ',', so 15-digit ones add the most per byte; k of them
    // take 16k - 1 <= 4083 bytes, k <= 255: sum < 255 * 10^15 ~ 2.6e17, far below 2^63 ~ 9.2e18 (values are >= 0 here).
    unsigned long long sum = 0;
    for (uint32_t seg = 0; seg < nseg; ++seg) {
        const uint32_t base = (seg << 10) + 32u * (uint32_t)lane;
        const uint32_t dg = MULTI ? sel4(seg, dg0, dg1, dg2, dg3) : dg0;
        // neighbours' digit masks: the previous chunk (last lane of the previous segment for lane 0), the next chunk
        const uint32_t up = __shfl_up_sync(0xffffffffu, dg, 1), dn = __shfl_down_sync(0xffffffffu, dg, 1);
        const uint32_t prev_last = (MULTI && seg) ? __shfl_sync(0xffffffffu, sel4(seg - 1u, dg0, dg1, dg2, dg3), 31) : 0u;
        const uint32_t next_first = (MULTI && seg + 1u < nseg) ? __shfl_sync(0xffffffffu, sel4(seg + 1u, dg0, dg1, dg2, dg3), 0) : 0u;
        const uint32_t p_dg = lane ? up : prev_last, n_dg = lane < 31 ? dn : next_first;
        if (MULTI && !__any_sync(0xffffffffu, dg != 0u)) continue;
        uint32_t w[8];
        if (MULTI && dg) json_load32(D + base, w);
        else {
            #pragma unroll
            for (int i = 0; i < 8; ++i) w[i] = MULTI ? 0u : wk[i];
        }
        const uint32_t head_bits = (p_dg >> 31) ? (dg & ~(dg + 1u)) : 0u;   // my leading digits belong to the previous chunk's number
        const uint32_t lo_in = vs < base ? 0xFFFFFFFFu : (vs - base >= 31u ? 0u : (0xFFFFFFFFu << (vs - base + 1u)));      // pos > vs
        const uint32_t hi_in = ve >= base + 32u ? 0xFFFFFFFFu : (ve <= base ? 0u : ((1u << (ve - base)) - 1u));             // pos < ve
        const uint32_t mine_dg = dg & ~head_bits & lo_in & hi_in;       // digits of numbers that start here and lie in the array
        const uint32_t ends = mine_dg & ~(mine_dg >> 1) & 0x7FFFFFFFu; // last digit of a number, bit 31 excluded (finished below)
        unsigned long long val = 0;
        #pragma unroll
        for (int j = 0; j < 32; ++j) {
            const uint32_t c = (w[j >> 2] >> (8 * (j & 3))) & 0xFu;
            val = ((mine_dg >> j) & 1u) ? val * 10ull + c : 0ull;
            if ((ends >> j) & 1u) sum += val;
        }
        // bit 31 tells whether a number is still open; its remaining digits are the next chunk's leading ones
        const uint32_t open = mine_dg >> 31;
        const uint32_t more = open ? (uint32_t)__ffs((int)~n_dg) - 1u : 0u;     // <= 15 (checked above)
        uint32_t nw[4];
        #pragma unroll
        for (int i = 0; i < 4; ++i) nw[i] = __shfl_down_sync(0xffffffffu, w[i], 1);
        if (MULTI && lane == 31 && open) {                              // the next chunk is the next segment's first one
            const uint8_t* q = D + base + 32u;
            #pragma unroll
            for (int i = 0; i < 4; ++i) nw[i] = (uint32_t)q[4 * i] | ((uint32_t)q[4 * i + 1] << 8) | ((uint32_t)q[4 * i + 2] << 16) | ((uint32_t)q[4 * i + 3] << 24);
        }
        #pragma unroll
        for (int j = 0; j < 15; ++j) {
            const uint32_t c = (nw[j >> 2] >> (8 * (j & 3))) & 0xFu;
            if ((uint32_t)j < more) val = val * 10ull + c;
        }
        if (open) sum += val;
    }
    #pragma unroll
    for (int d = 16; d > 0; d >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, d);
    *sum_out = sum;
    return 1;
    #undef B9_P1
    #undef B9_P2
}

// ================================================================== the kernel: warp-autonomous
// Every WARP is an independent worker with its own ticket pipeline, its own slice of shared memory
// (slot metadata + one stage buffer + one mbarrier) and its own cursor add. There is no block
// barrier anywhere in the loop: while one warp waits for its bulk copy or its atomic, the other
// ~27 warps of the SM are in their compute phases. (The CTA-per-tile versions spent most of their
// time at __syncthreads behind warp 0's staging, the cursor atomic and the escaped-string pass:
// profiles/r1_v2c/v2d/v2e.)
constexpr int D3_WARPS = 2;                  // warps per CTA (a container only)
template <int HANDLER> struct D3Cfg {
    // threads per task. G = 2 doubles the warps per staged byte but also doubles the per-task setup
    // instructions (both lanes execute them); with no barriers to hide, G = 1 wins (r1_v3a vs r1_v3b).
#ifndef B9_IDENTITY_G
#define B9_IDENTITY_G 1
#endif
    static constexpr int G = (HANDLER == 0) ? B9_IDENTITY_G : 1;
    // tasks per warp-tile. crc32 (configs[2]: zipf 32..4096-byte strings, ~1 KB on average) works on a task
    // with the whole warp, so its tiles are small: 4 tasks keep the stage buffer at ~5 KB, which leaves L1 room for the shift tables.
#ifndef B9_JSON_T
#define B9_JSON_T 8
#endif
    static constexpr int T = (HANDLER == 1) ? 4 : (HANDLER == 3) ? B9_JSON_T : 32 / G;
};
constexpr int D2_THREADS = 4;                // host: the smallest warp-tile (sizes the per-tile count arrays)

// Tables of the coalesced tile copy (d3_copy_tile): which copied task does an aligned 16-byte vector of the
// tile's output start in, and where do its bytes sit in the stage buffer. Only thread-per-task handlers copy.
struct D3CopyTab {
    alignas(16) uint4 ent[33];     // per copied task r: {first output byte, end, source offset - output offset, the same of task r+1}
    uint2 bp[32];                  // per block of 32 vectors: {bit v set = some task r >= 1 starts in vector v, tasks started before the block}
};
struct D3NoTab {};
template <int T>
struct D3Warp {
    uint64_t goff[T];              // physical ring offset of each task's payload
    uint32_t soff[T];              // offset inside the stage buffer (when staged)
    uint32_t len[T];
    uint8_t  flg[T];               // slot flags (B9_TF_*)
    alignas(8) uint64_t mbar;
    typename std::conditional<T == 32, D3CopyTab, D3NoTab>::type ct;
};

struct D3MetaRegs { uint64_t off, hdr; uint4 id; };   // (the id rides along: it is only copied to the record, and loading it a tile ahead takes its latency off the record write)
// tt = tasks per tile of this launch (<= T; the compile-time T for every handler but json_sum)
template <int T>
__device__ __forceinline__ void d3_load_meta(const DrainArgs& a, unsigned long long tile, int lane, D3MetaRegs& r, uint32_t tt) {
    const uint32_t t0 = (uint32_t)tile * tt;
    r.off = 0; r.hdr = 0; r.id = make_uint4(0u, 0u, 0u, 0u);
    if ((uint32_t)lane < tt && t0 + lane < a.n_tasks) {
        const uint32_t slot = (uint32_t)((a.first_task + t0 + lane) & a.slot_mask);
        r.hdr = __ldg(a.hdr + slot);
        r.off = __ldg(a.off + slot);
        r.id = __ldg(a.ids + slot);
    }
}

// Windows that hold cancelled slots (TaskQueuePop's skip loop, taskqueue.go:243-271): a task's record index is no
// longer its task index. Two small kernels ahead of the drain turn the slot flags (8 B per task) into the number of
// ready tasks before every warp-tile, so the drain itself stays free of any inter-tile dependency:
//   tile_count_kernel   256 slots per block: ready bits by ballot; per tile of T (= 4, 8 or 32) slots the ready tasks
//                       before it INSIDE the block, and the block's total
//   tile_scan_kernel    one CTA: in-place prefix over the block totals (n / 256 values)
// record index base of a tile = its in-block prefix + its block's prefix (two loads in the drain).
// (An earlier version chained the counts through a decoupled look-back inside the drain: 0.32 ms instead of 0.18 ms
// for 1M tasks as soon as ONE slot of the window was cancelled.)
constexpr uint32_t TC_SLOTS = 256;             // slots per tile_count_kernel block (8 warps x 32)
__global__ void __launch_bounds__(TC_SLOTS) tile_count_kernel(const uint64_t* __restrict__ hdr, uint32_t slot_mask, uint64_t first_task, uint32_t n_tasks,
                                                              uint32_t T, uint32_t* __restrict__ base /* [n_tiles]: ready tasks before the tile, inside its block */,
                                                              uint32_t* __restrict__ block_tot /* [blocks + 1], entry b + 1 = ready tasks of block b */) {
    __shared__ uint32_t s_warp[TC_SLOTS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t t = blockIdx.x * TC_SLOTS + threadIdx.x;
    const bool ready = t < n_tasks && !(hdr_flags(__ldg(hdr + (uint32_t)((first_task + t) & slot_mask))) & 1u);
    const uint32_t m = __ballot_sync(0xffffffffu, ready);
    if (lane == 0) s_warp[warp] = __popc(m);
    __syncthreads();
    uint32_t before = 0, total = 0;                                       // ready tasks of the block's earlier warps / of the block
    #pragma unroll
    for (int w = 0; w < (int)(TC_SLOTS / 32); ++w) { const uint32_t c = s_warp[w]; if (w < warp) before += c; total += c; }
    const uint32_t per = 32u / T;                                         // tiles inside a warp's 32 slots
    if ((uint32_t)lane < per) {
        const uint32_t first_slot = blockIdx.x * TC_SLOTS + (uint32_t)warp * 32u + (uint32_t)lane * T;
        if (first_slot < n_tasks) base[first_slot / T] = before + __popc(m & ((1u << (lane * T)) - 1u));
    }
    if (threadIdx.x == 0) { block_tot[blockIdx.x + 1u] = total; if (blockIdx.x == 0) block_tot[0] = 0; }
}
// one CTA: block_tot[b] = ready tasks before block b (in place; entry `blocks` = the window's total)
__global__ void __launch_bounds__(1024) tile_scan_kernel(uint32_t* __restrict__ block_tot, uint32_t blocks) {
    __shared__ uint32_t s_warp[32];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t per = (blocks + 1023u) / 1024u;
    const uint32_t lo = min(blocks, tid * per), hi = min(blocks, lo + per);
    uint32_t sum = 0;
    for (uint32_t i = lo; i < hi; ++i) sum += block_tot[i + 1u];
    uint32_t inc = sum;
    #pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t v = __shfl_up_sync(0xffffffffu, inc, d); if ((int)lane >= d) inc += v; }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        uint32_t x = s_warp[lane], y = x;
        #pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t v = __shfl_up_sync(0xffffffffu, y, d); if ((int)lane >= d) y += v; }
        s_warp[lane] = y - x;                                             // exclusive over warps
    }
    __syncthreads();
    uint32_t run = s_warp[warp] + inc - sum;                              // ready tasks before my first block
    for (uint32_t i = lo; i < hi; ++i) { run += block_tot[i + 1u]; block_tot[i + 1u] = run; }
}
// ready tasks before warp-tile `tile` (of T slots)
__device__ __forceinline__ uint32_t tile_ready_before(const DrainArgs& a, unsigned long long tile, uint32_t T) {
    return __ldg(a.tile_base + tile) + __ldg(a.block_base + (uint32_t)((tile * T) / TC_SLOTS));
}

// scattered tile (it spans pushes): one bulk copy per task, each widened to 16-byte boundaries
template <int T>
__device__ __noinline__ uint32_t d3_stage_scattered(const uint8_t* __restrict__ payload, uint64_t off, uint32_t len, bool valid, D3Warp<T>& W, uint8_t* buf,
                                                    uint32_t in_cap, int lane) {
    const uint64_t end = off + len;
    const uint32_t asz = (valid && len) ? (uint32_t)(((end + 15ull) & ~15ull) - (off & ~15ull)) : 0u;
    const uint32_t ex = warp_excl_scan(asz, lane);
    const uint32_t total = __shfl_sync(0xffffffffu, ex + asz, 31);
    if (total > in_cap) return 0;
    if (lane == 0) mbar_expect_tx(&W.mbar, total);
    __syncwarp();
    if (valid) { W.soff[lane] = ex + (uint32_t)(off & 15ull); if (asz) bulk_g2s(buf + ex, payload + (off & ~15ull), asz, &W.mbar); }
    return 1;
}

// out-of-line generic-pointer versions for tiles that could not be staged (and other cold paths)
template <int G>
__device__ __noinline__ uint32_t quick_clean_framed_generic(const uint8_t* p, uint32_t len, int sub, bool active) { return quick_clean_framed<G>(p, len, sub, active); }
template <int G>
__device__ __noinline__ void group_copy_staged(uint8_t* dst, const uint8_t* src, uint32_t n, int sub) { group_copy<G>(dst, src, n, sub); }   // (tiles the coalesced copy does not take)
template <int G>
__device__ __noinline__ void group_copy_generic(uint8_t* dst, const uint8_t* src, uint32_t n, int sub) { group_copy<G>(dst, src, n, sub); }

template <int HANDLER>
__device__ __forceinline__ void d2_phase_b_task(const uint8_t* __restrict__ p, const TaskRec& rec, uint8_t* __restrict__ o) { seq_emit(p, rec, o); }

// the sequential validating parser + handler sizing, out of line: rare for identity, and it keeps the
// hot loops' registers and instruction-cache footprint small
template <int HANDLER>
__device__ __noinline__ void d2_parse_and_size(const uint8_t* p, uint32_t len, TaskRec& rec, const uint32_t* crc_table, bool http) {
    Parsed pr = parse_payload(p, len, http);
    handler_phase_a(HANDLER, p, pr, rec, crc_table);
}

// ------------------------------------------------------------------ coalesced tile copy
// The results of a warp-tile are ONE dense byte range of the output (a single cursor add), and when every
// result is a plain copy out of the stage buffer (identity's clean strings, vadd_f32's in-place records) that
// range is written by the warp as a whole: lane l stores the aligned 16-byte vectors l, l + 32, ... of the
// range (a store instruction covers 512 contiguous bytes = 4 lines, where one thread per task at a 258-byte
// stride touched 32 lines: the LSU, not HBM, bounded the round-1 kernel — profiles/r1_final_identity_main_summary.txt).
// A vector starts inside exactly one copied task t (entries are >= 16 bytes, so it ends in t or t + 1):
//   t(v) = #{r >= 1 : first byte of r <= 16 v}  =  prefix-popcount of a bitmap with bit ceil(ex_r / 16) set,
// one bitmap word per block of 32 vectors, word prefixes by one warp scan. The 16 source bytes come from two
// aligned 16-byte shared loads + a byte shift. Vectors that cross into the next task are left to one extra
// pass (lane r: the vector around the end of task r).
__device__ __forceinline__ uint4 lds128(const uint8_t* p) { return *(const uint4*)p; }
// 16 bytes at byte offset `at` (any alignment) of the stage buffer
__device__ __forceinline__ uint4 ld_unaligned16(const uint8_t* __restrict__ sbuf, uint32_t at) {
    const uint32_t s = at & 15u, q = s >> 2, bits = (s & 3u) * 8u;
    const uint4 a = lds128(sbuf + (at - s)), b = lds128(sbuf + (at - s) + 16);
    uint32_t w0 = a.x, w1 = a.y, w2 = a.z, w3 = a.w, w4 = b.x, w5 = b.y, w6 = b.z, w7 = b.w;
    if (q & 2u) { w0 = w2; w1 = w3; w2 = w4; w3 = w5; w4 = w6; w5 = w7; }
    if (q & 1u) { w0 = w1; w1 = w2; w2 = w3; w3 = w4; w4 = w5; }
    uint4 o;
    o.x = __funnelshift_r(w0, w1, bits); o.y = __funnelshift_r(w1, w2, bits);
    o.z = __funnelshift_r(w2, w3, bits); o.w = __funnelshift_r(w3, w4, bits);
    return o;
}
constexpr uint32_t D3_COPY_MAX_BYTES = 16384;      // 32 bitmap words x 32 vectors x 16 bytes

// All 32 lanes. c_len = bytes my task contributes (0: none), ex = their offset in the tile's range, src = their
// offset in the stage buffer; tb = bytes of the range; out = its (16-byte aligned) address. Preconditions,
// checked by the caller: every non-zero c_len >= 16, tb <= D3_COPY_MAX_BYTES, the range is padded to 16 bytes.
__device__ __forceinline__ void d3_copy_tile(D3CopyTab& C, const uint8_t* __restrict__ sbuf, uint8_t* __restrict__ out,
                                             uint32_t c_len, uint32_t ex, uint32_t src, uint32_t tb, int lane) {
    const uint32_t nz = __ballot_sync(0xffffffffu, c_len != 0u);
    const uint32_t lt = (1u << lane) - 1u;
    const uint32_t r = __popc(nz & lt), cnt = __popc(nz);
    const uint32_t nblk = (tb + 511u) >> 9;
    const uint32_t delta = src - ex;
    const uint32_t above = nz & ~lt & ~(1u << lane);
    const uint32_t delta_next = __shfl_sync(0xffffffffu, delta, above ? (__ffs(above) - 1) : lane);
    if ((uint32_t)lane < nblk) C.bp[lane] = make_uint2(0u, 0u);
    __syncwarp();
    if (c_len) {
        C.ent[r] = make_uint4(ex, above ? ex + c_len : 0xFFFFFFFFu, delta, delta_next);   // (the last task owns the padding)
        if (r) { const uint32_t fv = (ex + 15u) >> 4; atomicOr(&C.bp[fv >> 5].x, 1u << (fv & 31u)); }
    }
    __syncwarp();
    {
        const uint32_t mine = (uint32_t)lane < nblk ? (uint32_t)__popc(C.bp[lane].x) : 0u;
        const uint32_t before = warp_excl_scan(mine, lane);
        if ((uint32_t)lane < nblk) C.bp[lane].y = before;
    }
    __syncwarp();
    const uint32_t le = lt | (1u << lane);
    #pragma unroll 2
    for (uint32_t i = 0; i < nblk; ++i) {
        const uint32_t o = (i << 9) + ((uint32_t)lane << 4);
        if (o < tb) {
            const uint2 bp = C.bp[i];
            const uint4 e = C.ent[bp.y + __popc(bp.x & le)];
            if (e.y - o >= 16u) *(uint4*)(out + o) = ld_unaligned16(sbuf, o + e.z);
        }
    }
    if ((uint32_t)lane + 1u < cnt) {                                       // the vector around the end of task `lane` (by rank)
        const uint4 e = C.ent[lane];
        const uint32_t keep = e.y & 15u;                                   // its first `keep` bytes are this task's, the rest the next one's
        if (keep) {
            const uint32_t o = e.y - keep;
            const uint4 a = ld_unaligned16(sbuf, o + e.z), b = ld_unaligned16(sbuf, o + e.w);
            uint4 v; uint32_t m;
            m = byte_range_mask(0, 0, keep); v.x = (a.x & m) | (b.x & ~m);
            m = byte_range_mask(1, 0, keep); v.y = (a.y & m) | (b.y & ~m);
            m = byte_range_mask(2, 0, keep); v.z = (a.z & m) | (b.z & ~m);
            m = byte_range_mask(3, 0, keep); v.w = (a.w & m) | (b.w & ~m);
            *(uint4*)(out + o) = v;
        }
    }
}

// ------------------------------------------------------------------ identity: escaped strings, settled in the main loop
// configs[1]'s 1 % "adversarial" share are strings json.dumps had to escape. Whatever json.dumps wrote comes back
// from identity as the very same text (Go decodes, Python re-encodes), with ONE exception: a lone surrogate escape
// becomes � (Go's decoder, oracle/pyoracle/gojson.py:212-264). So the warp does not transcode such a body, it
// VERIFIES that every escape is one json.dumps writes — and then the task is a plain copy like its clean neighbours:
//   * lane r owns bytes [16r, 16r+16) of a 512-byte pass; backslash and quote positions as 16-bit masks
//     (exact SWAR equality + a multiply that gathers the four byte flags of a word into a nibble);
//   * which backslashes START an escape: the odd-backslash-run rule (simdjson's find_escaped) per lane, the carry
//     ("my first byte is escaped") resolved across lanes with two ballots — a lane's carry-out is constant or its
//     carry-in XOR a constant, so the carry into lane r is a parity over the lanes above the last constant one;
//   * one step per escape start: the two-character escapes json.dumps writes, or \uXXXX with lower-case hex and a
//     value json.dumps would write that way (control characters without a short form, DEL, >= 0x80); surrogate
//     escapes are paired by looking 6 bytes ahead / behind, lone ones are rewritten to � in the stage buffer.
// Anything else (raw non-ASCII, "\/", upper-case hex, malformed text) is NOT decided here: the task goes to
// tail of the kernel (slow_task). The rule set has a Python model fuzzed against the oracle on the CPU
// (tests/esc_verify_model.py, tests/test_esc_verify_model.py).
__device__ __forceinline__ uint32_t eq_mask32(uint32_t w, uint32_t k4) {           // 0x80 in every byte of w equal to the byte of k4 (exact)
    const uint32_t z = w ^ k4;
    return ~(((z & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | z) & 0x80808080u;
}
__device__ __forceinline__ uint32_t gather4(uint32_t m) { return (((m >> 7) * 0x00204081u) >> 21) & 0xFu; }   // byte flags (bit 7) -> 4 bits
__device__ __forceinline__ uint32_t eq_bits16(const uint4& v, uint32_t k4) {
    return gather4(eq_mask32(v.x, k4)) | (gather4(eq_mask32(v.y, k4)) << 4) | (gather4(eq_mask32(v.z, k4)) << 8) | (gather4(eq_mask32(v.w, k4)) << 12);
}
// 16 positions, the first cnt of them real bytes: the escaped ones (they follow an escape-start backslash); *cout = the real
// bytes end on an unmatched escape start
__device__ __forceinline__ uint32_t esc16(uint32_t bs, uint32_t cin, uint32_t cnt, uint32_t* cout) {
    bs &= ~cin;
    const uint32_t follows = ((bs << 1) | cin) & 0xFFFFu;
    const uint32_t odd_starts = bs & 0xAAAAu & ~follows;
    const uint32_t seq_even = odd_starts + bs;                             // 17 bits
    const uint32_t escaped = (0x5555u ^ (seq_even << 1)) & follows;
    *cout = cnt < 16u ? (escaped >> cnt) & 1u : (seq_even >> 16) & 1u;
    return escaped;
}
// four hex digits given as a little-endian word -> their value, or -1 (SWAR, no loads)
__device__ __forceinline__ int hex4w(uint32_t w) {
    const uint32_t H = 0x80808080u;
    const uint32_t x = w & 0x7F7F7F7Fu, y = x | 0x20202020u;
    const uint32_t isd = ((x + 0x50505050u) & ~(x + 0x46464646u)) & H;    // '0' <= x <= '9'
    const uint32_t isl = ((y + 0x1F1F1F1Fu) & ~(y + 0x19191919u)) & H;    // 'a' <= (x | 0x20) <= 'f'
    const uint32_t nib = (x & 0x0F0F0F0Fu) + (isl >> 7) * 9u;
    const int v = (int)(((nib & 0xFu) << 12) | (((nib >> 8) & 0xFu) << 8) | (((nib >> 16) & 0xFu) << 4) | (nib >> 24));
    return ((isd | isl) != H || (w & H)) ? -1 : v;
}

// All 32 lanes; the body is sbuf[at, at + n) (stage buffer), `list` is scratch for 256 16-bit positions. true:
// json.dumps(identity(body)) is the body text as it now stands in the stage buffer (lone surrogates rewritten). false:
// not decided. The escape starts of a pass are first compacted into `list` (prefix sum over the lanes' counts), then
// lane l classifies escapes l, l + 32, ... with straight-line code: the work is balanced over the warp however the
// escapes cluster, and no lane walks a chain of dependent byte loads.
__device__ __noinline__ bool esc_verify_canonical(uint8_t* __restrict__ sbuf, uint32_t at, uint32_t n, int lane, uint16_t* __restrict__ list) {
    uint8_t* const body = sbuf + at;
    const uint32_t lt = (1u << lane) - 1u;
    uint32_t carry = 0;
    for (uint32_t base0 = 0; base0 < n; base0 += 512u) {
        const uint32_t base = base0 + 16u * (uint32_t)lane;
        const uint32_t cnt = base < n ? min(16u, n - base) : 0u;
        const uint32_t A = 0x61616161u;
        uint4 v = make_uint4(A, A, A, A);
        if (cnt) {
            v = ld_unaligned16(sbuf, at + base);
            if (cnt < 16u) {
                uint32_t m;
                m = byte_range_mask(0, 0, cnt); v.x = (v.x & m) | (A & ~m);
                m = byte_range_mask(1, 0, cnt); v.y = (v.y & m) | (A & ~m);
                m = byte_range_mask(2, 0, cnt); v.z = (v.z & m) | (A & ~m);
                m = byte_range_mask(3, 0, cnt); v.w = (v.w & m) | (A & ~m);
            }
        }
        // raw control bytes are not JSON; DEL and non-ASCII are escaped by json.dumps: neither is settled here
        const uint32_t K1 = 0x01010101u, K60 = 0x60606060u;
        const uint32_t hi = (v.x | v.y | v.z | v.w) | ((v.x + K1) | (v.y + K1) | (v.z + K1) | (v.w + K1));
        const uint32_t lo = (v.x + K60) & (v.y + K60) & (v.z + K60) & (v.w + K60);
        bool ok = ((hi | ~lo) & 0x80808080u) == 0u;
        const uint32_t bs = eq_bits16(v, 0x5C5C5C5Cu), qt = eq_bits16(v, 0x22222222u);
        uint32_t o0, o1;
        esc16(bs, 0u, cnt, &o0); esc16(bs, 1u, cnt, &o1);
        const uint32_t Kd = __ballot_sync(0xffffffffu, o0 != o1);           // lanes whose carry-out depends on their carry-in
        const uint32_t V0 = __ballot_sync(0xffffffffu, o0 != 0u);
        const uint32_t below = ~Kd & lt;
        const uint32_t cin = below ? (uint32_t)__popc(V0 & lt & ~((1u << (31 - __clz(below))) - 1u)) & 1u : ((uint32_t)__popc(V0 & lt) & 1u) ^ carry;
        const uint32_t fixed = ~Kd;
        const uint32_t next_carry = fixed ? (uint32_t)__popc(V0 & ~((1u << (31 - __clz(fixed))) - 1u)) & 1u : ((uint32_t)__popc(V0) & 1u) ^ carry;
        uint32_t co;
        const uint32_t escaped = esc16(bs, cin, cnt, &co);
        if (qt & ~escaped) ok = false;                                       // a raw quote inside the body
        uint32_t starts = bs & ~cin & ~escaped;
        // ---- compact the escape starts of the pass
        const uint32_t mine_n = (uint32_t)__popc(starts);
        uint32_t slot = warp_excl_scan(mine_n, lane);
        const uint32_t total = __shfl_sync(0xffffffffu, slot + mine_n, 31);
        while (starts) { list[slot++] = (uint16_t)(base - base0 + (uint32_t)(__ffs(starts) - 1)); starts &= starts - 1u; }
        __syncwarp();
        // ---- one escape per lane and round
        uint32_t patch_rounds = 0;
        for (uint32_t e0 = 0, round = 0; e0 < total; e0 += 32u, ++round) {
            const uint32_t e = e0 + (uint32_t)lane;
            if (e < total) {
                const uint32_t i = base0 + list[e];
                // bytes [i-8, i) and [i, i+12): the frame's 11-byte prefix precedes the body and its 17-byte suffix follows it
                const uint32_t sa = at + i - 8u, mis = sa & 3u;
                const uint32_t* wp = (const uint32_t*)(sbuf + (sa - mis));
                const uint32_t w0 = wp[0], w1 = wp[1], w2 = wp[2], w3 = wp[3], w4 = wp[4], w5 = wp[5];
                const uint32_t sh = mis * 8u;
                const uint32_t P0 = __funnelshift_r(w0, w1, sh), P1 = __funnelshift_r(w1, w2, sh);           // i-8 .. i-1
                const uint32_t F0 = __funnelshift_r(w2, w3, sh), F1 = __funnelshift_r(w3, w4, sh), F2 = __funnelshift_r(w4, w5, sh);   // i .. i+11
                const uint32_t t = (F0 >> 8) & 0xFFu;
                const uint32_t d = t - 0x5Cu;
                const bool simple = t == '"' || (d < 32u && ((0x01440441u >> d) & 1u));   // \\ b f n r t
                const uint32_t hw = (F0 >> 16) | (F1 << 16);                                // i+2 .. i+5
                const int h = hex4w(hw);
                bool good;
                bool lone = false;
                if (t != 'u') good = simple;
                else {
                    good = i + 6u <= n && h >= 0 && !hex_has_upper(hw)
                           && !(h < 0x20 && ((0x3700u >> h) & 1u))                          // \b \t \n \f \r have short forms
                           && !(h >= 0x20 && h < 0x7F);                                     // json.dumps writes the character itself
                    if (h >= 0xD800 && h < 0xDC00) {                                        // high surrogate: paired with a low-surrogate escape right behind it?
                        const int l2 = hex4w(F2);                                           // i+8 .. i+11
                        lone = !(i + 12u <= n && (F1 >> 16) == 0x755Cu && l2 >= 0xDC00 && l2 <= 0xDFFF);
                    } else if (h >= 0xDC00 && h < 0xE000) {                                 // low surrogate: consumed by a high-surrogate escape 6 bytes before?
                        const int h2 = hex4w(P1);                                           // i-4 .. i-1
                        lone = true;
                        if (i >= 6u && (P0 >> 16) == 0x755Cu && h2 >= 0xD800 && h2 <= 0xDBFF) {
                            // ... if the backslash at i-6 starts an escape: an even run of backslashes before it
                            uint32_t run = 0;
                            if (i >= 7u && ((P0 >> 8) & 0xFFu) == '\\') run = bs_run_before(body, i - 6u);
                            lone = (run & 1u) != 0u;
                        }
                    }
                }
                if (!good) ok = false;
                if (lone) patch_rounds |= 1u << round;
            }
        }
        if (!__all_sync(0xffffffffu, ok)) return false;
        carry = next_carry;
        __syncwarp();                                                            // every window of the pass is read before a byte of it is rewritten
        while (patch_rounds) {
            const uint32_t round = (uint32_t)(__ffs(patch_rounds) - 1);
            patch_rounds &= patch_rounds - 1u;
            uint8_t* o = body + base0 + list[round * 32u + (uint32_t)lane] + 2u;
            o[0] = 'f'; o[1] = 'f'; o[2] = 'f'; o[3] = 'd';
        }
        __syncwarp();
    }
    return carry == 0u;
}

// ------------------------------------------------------------------ cloudpickle-framed tasks (the function path)
// `Function.map()` sends cloudpickle.dumps({"args": args, "kwargs": kwargs}) per input (sdk/src/beta9/abstractions/function.py:
// 198-205,246-262); the gateway hands a blob that starts 80 05 95 to the runner as it is (pkg/abstractions/function/task.go:
// 84,104-108), the runner unpickles, calls handler(*args, **kwargs) and cloudpickles the result (runner/function.py:236-283).
// A GPU cannot unpickle objects; what it CAN do bit-exactly is the one shape the configurations' handlers take — a single
// `str` argument, no keyword arguments — whose pickle is a fixed template around the UTF-8 bytes:
//   80 05 | 95 <u64 len-11> | 7d 94 28 8c 04 "args" 94 | 8c <u8 n> or 58 <u32 n> | n bytes | 94 85 94 8c 06 "kwargs" 94 7d 94 75 2e
// and identity's result is cloudpickle.dumps(s): 80 05 95 <u64 hdr+n+2> | the same string opcode + bytes | 94 2e. Anything
// else (other argument types, memo references such as the interned "args", strings >= 64 KiB that the pickler writes outside
// its frames, invalid UTF-8) is reported UNSUPPORTED — the host runs exactly those through the reference's CPU loop.
struct PickleStr { uint32_t hdr, n; bool ok; };
__device__ __forceinline__ PickleStr pickle_str_frame(const uint8_t* __restrict__ p, uint32_t len) {
    PickleStr r; r.hdr = 0; r.n = 0; r.ok = false;
    if (len < 39u) return r;
    bool bad = (ld_u32_unaligned(p) & 0x00FFFFFFu) != 0x00950580u;                              // 80 05 95
    bad |= ld_u32_unaligned(p + 3) != len - 11u || ld_u32_unaligned(p + 7) != 0u;          // FRAME length (u64)
    bad |= ld_u32_unaligned(p + 11) != 0x8C28947Du;                                        // 7d 94 28 8c
    bad |= ld_u32_unaligned(p + 15) != 0x67726104u;                                        // 04 'a' 'r' 'g'
    bad |= (ld_u32_unaligned(p + 19) & 0x0000FFFFu) != 0x00009473u;                        // 's' 94
    const uint32_t op = p[21];
    if (op == 0x8Cu) { r.hdr = 2; r.n = p[22]; }
    else if (op == 0x58u) { r.hdr = 5; r.n = ld_u32_unaligned(p + 22); bad |= r.n < 256u || r.n >= 65536u; }   // (the pickler's own choice of opcode)
    else bad = true;
    if (bad || len != 21u + r.hdr + r.n + 16u) return r;
    const uint8_t* q = p + 21u + r.hdr + r.n;                                              // 94 85 94 8c | 06 6b 77 61 | 72 67 73 94 | 7d 94 75 2e
    r.ok = ld_u32_unaligned(q) == 0x8C948594u && ld_u32_unaligned(q + 4) == 0x61776B06u && ld_u32_unaligned(q + 8) == 0x94736772u && ld_u32_unaligned(q + 12) == 0x2E75947Du;
    return r;
}
// any byte >= 0x80 in p[lo, hi)? (4 bytes at a time; reads at most 3 bytes before lo / after hi, inside the payload's frame)
__device__ __forceinline__ bool range_has_high_bit(const uint8_t* __restrict__ p, uint32_t lo, uint32_t hi) {
    uint32_t acc = 0;
    uint32_t i = lo;
    for (; i + 4u <= hi; i += 4u) acc |= ld_u32_unaligned(p + i);
    for (; i < hi; ++i) acc |= p[i];
    return (acc & 0x80808080u) != 0u;
}
// UTF-8 as Python decodes a pickled str ("surrogatepass": the 3-byte encodings of U+D800..DFFF are accepted)
__device__ __noinline__ bool utf8_valid_surrogatepass(const uint8_t* __restrict__ b, uint32_t n) {
    uint32_t i = 0;
    while (i < n) {
        const uint8_t c = b[i];
        if (c < 0x80) { ++i; continue; }
        if (c >= 0xC2 && c <= 0xDF) { if (i + 2 > n || (b[i + 1] & 0xC0) != 0x80) return false; i += 2; continue; }
        if (c >= 0xE0 && c <= 0xEF) {
            if (i + 3 > n) return false;
            const uint8_t lo = c == 0xE0 ? 0xA0 : 0x80;
            if (b[i + 1] < lo || b[i + 1] > 0xBF || (b[i + 2] & 0xC0) != 0x80) return false;
            i += 3; continue;
        }
        if (c >= 0xF0 && c <= 0xF4) {
            if (i + 4 > n) return false;
            const uint8_t lo = c == 0xF0 ? 0x90 : 0x80, hi = c == 0xF4 ? 0x8F : 0xBF;
            if (b[i + 1] < lo || b[i + 1] > hi || (b[i + 2] & 0xC0) != 0x80 || (b[i + 3] & 0xC0) != 0x80) return false;
            i += 4; continue;
        }
        return false;
    }
    return true;
}
__device__ __forceinline__ void pickle_result_header(uint8_t* __restrict__ o, uint32_t frame_len) {    // 80 05 95 <u64>
    o[0] = 0x80; o[1] = 0x05; o[2] = 0x95;
    o[3] = (uint8_t)frame_len; o[4] = (uint8_t)(frame_len >> 8); o[5] = (uint8_t)(frame_len >> 16); o[6] = (uint8_t)(frame_len >> 24);
    o[7] = 0; o[8] = 0; o[9] = 0; o[10] = 0;
}

// ---------------------------------------------------------------- identity: deferred tasks, in the kernel's tail
// What the main loop could not settle (escapes json.dumps would not have written, raw non-ASCII, foreign framing,
// non-string arguments, HTTP bodies) is put on a work list and processed by the workers once they run out of tiles,
// one warp per task. (Round 1 ran a second kernel for this; with the canonical-escape check in the main loop the list is
// empty for SDK-made payloads, and a second launch cost ~6 us of every drain for nothing — profiles/r2_s4_*.)
// No worker ever waits for another one: a worker takes what is claimable and leaves; every worker publishes its items
// BEFORE it counts itself done, so the worker that counts last sees the final list and drains what is left.
__device__ __noinline__ void slow_task(const DrainArgs& a, uint64_t goff, uint32_t lenw, uint32_t j, bool pickle, uint8_t* __restrict__ stage, uint32_t stage_cap, int lane) {
    const uint32_t len = lenw & 0x3FFFFFFFu;
    const bool http = (lenw & 0x40000000u) != 0;
    const uint8_t* p = a.payload + goff;
    if (len + 32u <= stage_cap) {
        // the walks below are chains of dependent byte loads: run them against shared memory instead of L2/HBM
        const uint32_t mis = (uint32_t)(goff & 15ull);
        const uint4* src = (const uint4*)(p - mis);
        uint4* dst = (uint4*)stage;
        const uint32_t nv = (mis + len + 15u) >> 4;
        __syncwarp();
        for (uint32_t v = lane; v < nv; v += 32) dst[v] = __ldg(src + v);
        __syncwarp();
        p = stage + mis;
    }
    TaskRec rec; rec.ready = 1; rec.status = 0; rec.has = 0; rec.mode = OM_NONE; rec.out_len = 0; rec.src_off = 0; rec.src_len = 0; rec.value = 0;
    bool par = false, fast = false;
    EscLane L; L.start = 0; L.out_len = 0; L.npatch = 0; L.ok = true; L.len_change = false;
    L.patch_pos[0] = L.patch_pos[1] = 0; L.patch_cp[0] = L.patch_cp[1] = 0;
    if (pickle) {
        // cloudpickle-framed: lane 0 checks the template and the UTF-8 (anything else is not decided on the device)
        uint32_t w = 0;
        if (lane == 0) { const PickleStr ps = pickle_str_frame(p, len); if (ps.ok && utf8_valid_surrogatepass(p + 21u + ps.hdr, ps.n)) w = 0x80000000u | (ps.hdr << 24) | ps.n; }
        w = __shfl_sync(0xffffffffu, w, 0);
        const uint32_t hdr = (w >> 24) & 0x7Fu, n = w & 0xFFFFFFu;
        const uint32_t out_len = w ? 11u + hdr + n + 2u : 0u;
        unsigned long long base = 0;
        const uint32_t alloc = (out_len + 15u) & ~15u;
        if (lane == 0 && out_len) base = atomicAdd(&a.ctl->bytes, (unsigned long long)alloc);
        base = __shfl_sync(0xffffffffu, base, 0);
        const bool fits = base + alloc <= a.out_cap;
        if (!fits && lane == 0) a.ctl->overflow = 1u;
        if (w && fits) {
            uint8_t* o = a.out_payload + base;
            if (lane == 0) { pickle_result_header(o, hdr + n + 2u); o[11u + hdr + n + 1u] = 0x2E; }
            warp_copy(o + 11, p + 21, hdr + n + 1u, lane);                 // string opcode + bytes + MEMOIZE
        }
        if (lane == 0) { a.out_off[j] = fits ? base : 0; a.out_len[j] = out_len; a.out_status[j] = w ? 0 : ST_UNSUPPORTED; a.out_has[j] = w ? 1 : 0; }
        __syncwarp();
        return;
    }
    const uint32_t nbody = len - FRAME_PRE_LEN - FRAME_SUF_LEN;
    if (lenw & 0x80000000u) {                                              // canonical frame: the body needs transcoding
        uint32_t ol;
        par = esc_scan(p + FRAME_PRE_LEN, nbody, lane, L, &ol, &fast);
        if (par) { rec.has = 1; rec.mode = OM_STR_PAR; rec.src_off = FRAME_PRE_LEN; rec.src_len = nbody; rec.out_len = ol; }
    }
    if (!par) {                                                            // the sequential validating parser decides
        if (lane == 0) d2_parse_and_size<0>(p, len, rec, nullptr, http);
        rec.src_off = __shfl_sync(0xffffffffu, rec.src_off, 0); rec.src_len = __shfl_sync(0xffffffffu, rec.src_len, 0);
        rec.out_len = __shfl_sync(0xffffffffu, rec.out_len, 0);
        const uint32_t w = __shfl_sync(0xffffffffu, (uint32_t)rec.status | ((uint32_t)rec.has << 8) | ((uint32_t)rec.mode << 16), 0);
        rec.status = (uint8_t)w; rec.has = (uint8_t)(w >> 8); rec.mode = (uint8_t)(w >> 16);
    }
    unsigned long long base = 0;
    const uint32_t alloc = (rec.out_len + 15u) & ~15u;                     // the cursor moves in 16-byte units (the tiles' ranges stay vector-aligned)
    if (lane == 0 && rec.out_len) base = atomicAdd(&a.ctl->bytes, (unsigned long long)alloc);
    base = __shfl_sync(0xffffffffu, base, 0);
    const bool fits = base + alloc <= a.out_cap;
    if (!fits && lane == 0) a.ctl->overflow = 1u;
    if (rec.has && fits) {
        uint8_t* o = a.out_payload + base;
        if (rec.mode == OM_STR_PAR) {
            if (fast) esc_emit_fast(p + FRAME_PRE_LEN - 1, nbody + 2, lane, o, L);
            else      esc_emit_general(p + FRAME_PRE_LEN, nbody, lane, o, L);
        }
        else if (rec.mode == OM_COPY) warp_copy(o, p + rec.src_off, rec.src_len, lane);
        else if (lane == 0) d2_phase_b_task<0>(p, rec, o);
    }
    if (lane == 0) { a.out_off[j] = fits ? base : 0; a.out_len[j] = rec.out_len; a.out_status[j] = rec.status; a.out_has[j] = rec.has; }
    __syncwarp();
}

__device__ __noinline__ void d3_identity_tail(const DrainArgs& a, uint8_t* __restrict__ stage, uint32_t stage_cap, int lane, uint32_t n_workers) {
    __syncwarp();
    if (lane == 0) { __threadfence(); atomicAdd(&a.ctl->workers_done, 1u); __threadfence(); }
    for (;;) {
        uint32_t i = 0xFFFFFFFFu;
        if (lane == 0) {
            const uint32_t n = *(volatile unsigned int*)&a.ctl->n_slow;
            uint32_t h = *(volatile unsigned int*)&a.ctl->slow_head;
            while (h < n) {
                const uint32_t old = atomicCAS(&a.ctl->slow_head, h, h + 1u);
                if (old == h) { i = h; break; }
                h = old;
            }
            if (i == 0xFFFFFFFFu && *(volatile unsigned int*)&a.ctl->workers_done == n_workers) {
                // everybody has published: the list is final — one more look, so that the last worker leaves nothing behind
                const uint32_t n2 = *(volatile unsigned int*)&a.ctl->n_slow;
                h = *(volatile unsigned int*)&a.ctl->slow_head;
                while (h < n2) {
                    const uint32_t old = atomicCAS(&a.ctl->slow_head, h, h + 1u);
                    if (old == h) { i = h; break; }
                    h = old;
                }
            }
        }
        i = __shfl_sync(0xffffffffu, i, 0);
        if (i == 0xFFFFFFFFu) break;
        unsigned long long w0 = 0, w1 = 0;
        if (lane == 0) {
            const volatile unsigned long long* pw0 = &a.slow[i].w0;
            do { w0 = *pw0; } while ((uint32_t)(w0 >> 40) != a.epoch);      // its publisher reserved the slot and is writing it
            __threadfence();
            w1 = *(const volatile unsigned long long*)&a.slow[i].w1;
        }
        w0 = __shfl_sync(0xffffffffu, w0, 0); w1 = __shfl_sync(0xffffffffu, w1, 0);
        slow_task(a, w0 & ((1ull << 40) - 1ull), (uint32_t)w1, (uint32_t)(w1 >> 32) & 0xFFFFFFu, ((w1 >> 56) & 1ull) != 0ull, stage, stage_cap, lane);
    }
}

template <int HANDLER>
// resident CTAs per SM the register allocation aims for. crc32's byte loop waits on its table loads and more warps hide
// them: 2.389 ms per 1M zipf strings with 96 registers / 10 CTAs, 2.249 with 80 / 12, 2.150 with 72 / 14, 2.005 with
// 64 / 16 and a stage buffer that lets 16 fit (profiles/r2_c1_*, r2_c2_*, r2_c3_*). identity is limited to 9 CTAs by its
// stage buffers, not by registers.
#ifndef B9_CRC_MINB
#define B9_CRC_MINB 16
#endif
#ifndef B9_VADD_MINB
#define B9_VADD_MINB 9
#endif
#ifndef B9_JSON_MINB
#define B9_JSON_MINB 9
#endif
__global__ void __launch_bounds__(D3_WARPS * 32, (HANDLER == 1 ? B9_CRC_MINB : HANDLER == 2 ? B9_VADD_MINB : HANDLER == 3 ? B9_JSON_MINB : 9)) drain3_kernel(DrainArgs a, uint32_t in_cap, uint32_t warp_stride) {
    constexpr int G = D3Cfg<HANDLER>::G, T = D3Cfg<HANDLER>::T;
    const uint32_t TT = (HANDLER == 3) ? a.tile_tasks : (uint32_t)T;      // tasks per tile: json_sum's is chosen per launch (<= T)
    extern __shared__ __align__(128) uint8_t d3_smem[];
    __shared__ uint32_t s_crc_table[HANDLER == 1 ? 256 : 1];
    __shared__ __align__(128) uint8_t s_b64[HANDLER == 2 ? 320 : 4];
    __shared__ __align__(128) uint8_t s_jcls[HANDLER == 3 ? 256 : 4];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint8_t* const wbase = d3_smem + (size_t)warp * warp_stride;
    D3Warp<T>& W = *reinterpret_cast<D3Warp<T>*>(wbase);
    uint8_t* const sbuf = wbase + ((sizeof(D3Warp<T>) + 127u) & ~127u);   // stage buffer (+64 bytes of readable slack)
    const int k = lane / G, sub = lane % G;                                // my task inside the warp-tile, my share of it

    if (HANDLER == 1) { for (int i = threadIdx.x; i < 256; i += D3_WARPS * 32) s_crc_table[i] = crc_table_entry(i); __syncthreads(); }
    if (HANDLER == 3) {
        for (int i = threadIdx.x; i < 256; i += D3_WARPS * 32) s_jcls[i] = json_cls_of((uint32_t)i);
        __syncthreads();
    }
    if (HANDLER == 2) {
        for (int i = threadIdx.x; i < 320; i += D3_WARPS * 32) s_b64[i] = i < 256 ? (uint8_t)b64_val((uint8_t)i) : b64_chr((uint32_t)i - 256u);
        __syncthreads();
    }
    if (lane == 0) { mbar_init(&W.mbar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    __syncwarp();

    // two tickets ahead: the slot words of the next tile are in registers when its turn comes, and
    // the ticket after that is in flight; nothing global sits between the end of a tile and the bulk
    // copy of the next one. (Holding tickets is harmless: nobody waits on another worker's tile.)
    // Tile sequence of a worker: its first `static_rounds` tiles are worker + q * workers (no shared
    // counter: one L2 atomic round trip less per tile, measured 4 %); the rest of the window comes from
    // the global ticket counter, so the last rounds are still balanced by work stealing. The host sets
    // static_rounds = 0 whenever tile costs are not uniform (cancelled slots, variable-size handlers).
    const unsigned long long n_workers = (unsigned long long)gridDim.x * D3_WARPS;
    const unsigned long long wid = (unsigned long long)blockIdx.x * D3_WARPS + warp;
    const unsigned long long dyn_base = (unsigned long long)a.static_rounds * n_workers;
    unsigned long long q = 0;                                              // sequence number of the next tile to fetch
    auto fetch = [&]() -> unsigned long long {                             // lane 0's value is the tile
        unsigned long long t = 0;
        if (q < a.static_rounds) t = wid + q * n_workers;
        else if (lane == 0) t = dyn_base + atomicAdd(&a.ctl->ticket, 1ull);
        ++q;
        return t;
    };
    unsigned long long t_cur = fetch(), t_raw = fetch();
    t_cur = __shfl_sync(0xffffffffu, t_cur, 0);
    D3MetaRegs mregs; mregs.off = 0; mregs.hdr = 0; mregs.id = make_uint4(0u, 0u, 0u, 0u);
    if (t_cur < a.n_tiles) d3_load_meta<T>(a, t_cur, lane, mregs, TT);
    uint32_t parity = 0;

    while (t_cur < a.n_tiles) {
        // ---------------- stage: decide how the tile's bytes get to shared memory, fire the copy --------
        const unsigned long long tile = t_cur;
        const uint32_t t0 = (uint32_t)tile * TT;
        const uint32_t nt = min(TT, a.n_tasks - t0);
        const bool valid = lane < (int)nt;
        const uint64_t m_off = mregs.off;
        const uint4 m_id = mregs.id;                                       // (lane == task for G == 1)
        const uint32_t m_len = valid ? hdr_len(mregs.hdr) : 0u;
        const bool m_ready = valid && !(hdr_flags(mregs.hdr) & 1u);
        const uint64_t m_end = m_off + m_len;
        uint64_t prev = __shfl_up_sync(0xffffffffu, m_end, 1);
        if (lane == 0) prev = m_off;
        const bool contig = __all_sync(0xffffffffu, !valid || m_off == prev);
        const uint64_t gs = __shfl_sync(0xffffffffu, m_off, 0);
        const uint64_t ge = __shfl_sync(0xffffffffu, m_end, (int)nt - 1);
        uint32_t staged = 0;
        if (valid) { W.goff[lane] = m_off; W.len[lane] = m_len; W.flg[lane] = (uint8_t)hdr_flags(mregs.hdr); }
        if (contig) {
            const uint64_t as = gs & ~15ull;
            const uint64_t bytes = ((ge + 15ull) & ~15ull) - as;
            if (bytes <= in_cap) {
                staged = 1;
                if (valid) W.soff[lane] = (uint32_t)(m_off - as);
                if (lane == 0) { mbar_expect_tx(&W.mbar, (uint32_t)bytes); if (bytes) bulk_g2s(sbuf, a.payload + as, (uint32_t)bytes, &W.mbar); }
            }
        } else staged = d3_stage_scattered<T>(a.payload, m_off, m_len, valid, W, sbuf, in_cap, lane);
        // record indices: ready counts are known from the slot words alone
        const uint32_t ready_mask_t = __ballot_sync(0xffffffffu, m_ready);       // bit = task index
        const uint32_t rc = __popc(ready_mask_t);
        const uint32_t base_cnt = a.count_mode ? tile_ready_before(a, tile, TT) : t0;   // (count_mode: from the pre-pass kernels)
        if (lane == 0 && tile == a.n_tiles - 1) a.ctl->total_cnt = base_cnt + rc;
        // advance the ticket pipeline (loads/atomics issued here are consumed one iteration later)
        t_cur = __shfl_sync(0xffffffffu, t_raw, 0);
        if (t_cur < a.n_tiles) d3_load_meta<T>(a, t_cur, lane, mregs, TT);
        t_raw = fetch();
        __syncwarp();                                                      // W.* visible to all lanes
        if (staged) { mbar_wait(&W.mbar, parity); parity ^= 1u; }

        // ---------------- phase A: G lanes per task ----------------------------------------------------
        const bool mine = k < (int)nt && ((ready_mask_t >> k) & 1u);
        const uint32_t my_len = mine ? W.len[k] : 0u;
        const uint32_t my_soff = (mine && staged) ? W.soff[k] : 0u;
        const uint64_t my_goff = mine ? W.goff[k] : 0ull;
        const bool my_http = mine && (W.flg[k] & B9_TF_HTTP_BODY_BIT) != 0;
        const bool my_pickle = mine && (W.flg[k] & B9_TF_PICKLE_BIT) != 0;
        TaskRec rec; rec.ready = mine; rec.status = 0; rec.has = 0; rec.mode = OM_NONE; rec.out_len = 0; rec.src_off = 0; rec.src_len = 0; rec.value = 0;
        bool clobbered = false;
        if (HANDLER == 0) {
            // identity: settle the common case here (canonical frame, clean body -> the token is its own
            // json.dumps); everything else is put on the work list of the kernel's tail (d3_identity_tail), so that
            // this loop stays small enough for the instruction cache and no worker stalls on a 1 % case
            uint32_t q;
            if (staged) q = quick_clean_framed<G>(sbuf + my_soff, my_len, sub, mine);
            else        q = quick_clean_framed_generic<G>(a.payload + my_goff, my_len, sub, mine);
            if (mine) {
                if (q == 3u) {
                    const uint32_t tok = my_len - FRAME_PRE_LEN - FRAME_SUF_LEN + 2;
                    if (tok > 2) { rec.has = 1; rec.mode = OM_COPY; rec.src_off = FRAME_PRE_LEN - 1; rec.src_len = tok; rec.out_len = tok; }
                } else { rec.mode = OM_DEFER; rec.value = (long long)(q & 1u); }
                if (my_http) { rec.has = 0; rec.out_len = 0; rec.mode = OM_DEFER; rec.value = 0; }   // an HTTP body: the map rules decide (kernel tail)
                if (my_pickle) {                                           // cloudpickle-framed (the function path): one str argument, settled here when it is ASCII
                    rec.has = 0; rec.out_len = 0; rec.mode = OM_DEFER; rec.value = 2;
                    if (staged) {
                        uint8_t* p = sbuf + my_soff;
                        const PickleStr ps = pickle_str_frame(p, my_len);
                        if (ps.ok && !range_has_high_bit(p, 21u + ps.hdr, 21u + ps.hdr + ps.n)) {
                            // the result is the string opcode run with a new frame header in front and STOP behind: patch the
                            // 11 bytes before it and the byte after its MEMOIZE in the stage buffer; the task is then a copy
                            pickle_result_header(p + 10, ps.hdr + ps.n + 2u);
                            p[21u + ps.hdr + ps.n + 1u] = 0x2E;
                            const uint32_t tok = 11u + ps.hdr + ps.n + 2u;
                            rec.has = 1; rec.mode = OM_COPY; rec.src_off = 10; rec.src_len = tok; rec.out_len = tok; rec.value = 0;
                        }
                    }
                }
            }
            if constexpr (HANDLER == 0 && T == 32) {
                // framed, but the body holds escapes: the warp checks that they are json.dumps's own (then the task is a copy after all)
                uint32_t dirty = staged ? __ballot_sync(0xffffffffu, mine && rec.mode == OM_DEFER && rec.value == 1) : 0u;
                while (dirty) {
                    const int kt = __ffs(dirty) - 1;
                    dirty &= dirty - 1u;
                    const uint32_t ln = W.len[kt];
                    const bool canon = esc_verify_canonical(sbuf, W.soff[kt] + FRAME_PRE_LEN, ln - FRAME_PRE_LEN - FRAME_SUF_LEN, lane, (uint16_t*)W.ct.ent);
                    if (canon && lane == kt) {
                        const uint32_t tok = ln - FRAME_PRE_LEN - FRAME_SUF_LEN + 2;
                        rec.has = 1; rec.mode = OM_COPY; rec.src_off = FRAME_PRE_LEN - 1; rec.src_len = tok; rec.out_len = tok; rec.value = 0;
                    }
                }
            }
        } else if (HANDLER == 1) {
            // crc32: the whole warp works on one task at a time (tasks are long and of very different lengths)
            for (uint32_t kt = 0; kt < nt; ++kt) {
                if (!((ready_mask_t >> kt) & 1u)) continue;
                if (W.flg[kt] & B9_TF_PICKLE_BIT) { if (lane == (int)kt) rec.status = ST_UNSUPPORTED; continue; }   // function path: identity only
                if (W.flg[kt] & B9_TF_HTTP_BODY_BIT) {                      // an HTTP body: the sequential parser with the map rules
                    if (lane == (int)kt) d2_parse_and_size<1>(staged ? (const uint8_t*)(sbuf + W.soff[kt]) : a.payload + W.goff[kt], W.len[kt], rec, s_crc_table, true);
                    continue;
                }
                const uint8_t* tp = staged ? (const uint8_t*)(sbuf + W.soff[kt]) : stage_one_task(a.payload, W.goff[kt], W.len[kt], sbuf, in_cap, lane);
                if (tp) crc_task_coop(tp, true, W.len[kt], lane, lane == (int)kt, s_crc_table, a.crc_shift_tabs, rec);
                else    crc_task_coop(a.payload + W.goff[kt], false, W.len[kt], lane, lane == (int)kt, s_crc_table, a.crc_shift_tabs, rec);
            }
        } else if (HANDLER == 3) {
            // json_sum: the whole warp parses one document at a time
            for (uint32_t kt = 0; kt < nt; ++kt) {
                if (!((ready_mask_t >> kt) & 1u)) continue;
                if (W.flg[kt] & B9_TF_PICKLE_BIT) { if (lane == (int)kt) rec.status = ST_UNSUPPORTED; continue; }
                if (W.flg[kt] & B9_TF_HTTP_BODY_BIT) {
                    if (lane == (int)kt) d2_parse_and_size<3>(staged ? (const uint8_t*)(sbuf + W.soff[kt]) : a.payload + W.goff[kt], W.len[kt], rec, nullptr, true);
                    continue;
                }
                int done = 0; unsigned long long sum = 0;
                const uint8_t* tp = staged ? (const uint8_t*)(sbuf + W.soff[kt]) : stage_one_task(a.payload, W.goff[kt], W.len[kt], sbuf, in_cap, lane);
                if (tp) {                                                  // one 1 KiB segment (configs[4]) or up to four
                    if (W.len[kt] <= 1024u + JSON_PRE_LEN + JSON_SUF_LEN) done = json_sum_coop<false>(tp, W.len[kt], lane, s_jcls, &sum);
                    else done = json_sum_coop<true>(tp, W.len[kt], lane, s_jcls, &sum);
                }
                if (lane == (int)kt) {
                    if (done) { if (sum) { rec.value = (long long)sum; rec.out_len = dec_len_u64(sum); rec.mode = OM_I64_DEC; rec.has = 1; } }
                    else d2_parse_and_size<3>(tp ? tp : a.payload + W.goff[kt], W.len[kt], rec, nullptr);
                }
            }
        } else if (my_pickle) {
            rec.status = ST_UNSUPPORTED;                                   // function path: identity only
        } else if (mine) {
            int fr = 0;
            if (HANDLER == 2 && staged && !my_http) fr = vadd_fast(sbuf + my_soff, my_len, s_b64, rec);
            if (fr != 1) {
                clobbered = fr == 2;                                       // stage bytes overwritten: read the ring instead
                const uint8_t* p = (staged && !clobbered) ? (const uint8_t*)(sbuf + my_soff) : a.payload + my_goff;
                d2_parse_and_size<HANDLER>(p, my_len, rec, s_crc_table, my_http);
            }
        }

        // ---------------- compaction (ballot) + sizes (scan) + ONE cursor add per warp-tile -------------
        const uint32_t my_bytes = (sub == 0) ? rec.out_len : 0u;
        const uint32_t ex_bytes0 = warp_excl_scan(my_bytes, lane);
        const uint32_t tb = __shfl_sync(0xffffffffu, ex_bytes0 + my_bytes, 31);
        const uint32_t ex_bytes = __shfl_sync(0xffffffffu, ex_bytes0, k * G);      // every lane of a task sees the task's offset
        const uint32_t ex_cnt = __popc(ready_mask_t & ((1u << k) - 1u));
        // thread-per-task handlers reserve whole 16-byte units, so that every tile's range starts on a vector
        // boundary (the coalesced copy below); the <= 15 bytes of padding per tile are never referenced by a record
        // (identity only: for vadd_f32, whose kernel is bound by the base64 arithmetic, the warp-wide copy's extra
        // instructions cost more than its coalescing saves — 0.2038 -> 0.2215 ms per 1M tasks, profiles/r2_s1_*)
        constexpr bool COAL = (T == 32 && G == 1 && HANDLER == 0);
        const uint32_t tb_alloc = COAL ? ((tb + 15u) & ~15u) : tb;
        unsigned long long base = 0;
        if (lane == 0 && tb) base = atomicAdd(&a.ctl->bytes, (unsigned long long)tb_alloc);
        base = __shfl_sync(0xffffffffu, base, 0);
        const bool fits = base + tb_alloc <= a.out_cap;
        if (!fits && lane == 0) a.ctl->overflow = 1u;
        bool coal = false;
        if constexpr (COAL) {
            const uint32_t c_len = (mine && rec.has && rec.mode == OM_COPY) ? rec.src_len : 0u;
            const bool ok_me = rec.out_len == c_len && (c_len == 0u || c_len >= 16u);
            coal = staged && fits && tb != 0u && tb <= D3_COPY_MAX_BYTES && __all_sync(0xffffffffu, ok_me);
            if (coal) d3_copy_tile(W.ct, sbuf, a.out_payload + base, c_len, ex_bytes0, my_soff + rec.src_off, tb, lane);
        }

        // ---------------- phase B: G lanes per task ----------------------------------------------------
        if (mine) {
            const uint64_t ob = base + ex_bytes;
            if (sub == 0) {
                const uint32_t slot = (uint32_t)((a.first_task + t0 + k) & a.slot_mask);
                const uint32_t j = base_cnt + ex_cnt;
                a.out_ids[j] = (G == 1) ? m_id : __ldg(a.ids + slot);
                if (HANDLER == 0 && rec.mode == OM_DEFER) {                // the second kernel writes the rest of the record
                    SlowItem* it = a.slow + atomicAdd(&a.ctl->n_slow, 1u);
                    it->w1 = (unsigned long long)(my_len | (rec.value == 1 ? 0x80000000u : 0u) | (my_http ? 0x40000000u : 0u)) | ((unsigned long long)j << 32) | (rec.value == 2 ? (1ull << 56) : 0ull);
                    __threadfence();
                    *(volatile unsigned long long*)&it->w0 = my_goff | ((unsigned long long)a.epoch << 40);
                } else { a.out_off[j] = fits ? ob : 0; a.out_len[j] = rec.out_len; a.out_status[j] = rec.status; a.out_has[j] = rec.has; }
            }
            if (rec.has && fits) {
                if (rec.mode == OM_COPY) {
                    if (coal) {}                                            // written by d3_copy_tile
                    else if (staged) group_copy_staged<G>(a.out_payload + ob, sbuf + my_soff + rec.src_off, rec.src_len, sub);
                    else             group_copy_generic<G>(a.out_payload + ob, a.payload + my_goff + rec.src_off, rec.src_len, sub);
                } else if (sub == 0 && rec.mode != OM_STR_PAR) {
                    const uint8_t* p = (staged && !clobbered) ? (const uint8_t*)(sbuf + my_soff) : a.payload + my_goff;
                    d2_phase_b_task<HANDLER>(p, rec, a.out_payload + ob);
                }
            }
        }
        __syncwarp();                                                      // stage buffer and W.* free again
    }
    if constexpr (HANDLER == 0) {
        // (a COPY of the argument block goes to the out-of-line tail: taking the address of the kernel parameter itself makes
        // the compiler keep the whole block in local memory, and the main loop then reads its arguments with LDL — measured
        // +24 us per 1M-task drain)
        const DrainArgs tail_args = a;
        d3_identity_tail(tail_args, sbuf, in_cap, lane, (uint32_t)n_workers);
    }
}

}  // namespace b9
