// The sequential (one thread per task) half of the drain: what a parsed payload means to each handler
// (phase A: status, result size, how the bytes will be produced) and the byte producers that are not plain
// copies (phase B). No CUDA builtins in here: tests/host_shim/host_parse.cpp compiles this file, the parser
// and the handlers for the host, so that the device's slow path is fuzzed against the oracle on a CPU
// (tests/test_device_parser_on_host.py). The warp-cooperative fast paths live in drain2.cuh.
#pragma once
#include <stdint.h>
#include "json_device.cuh"
#include "handlers_device.cuh"

namespace b9 {

// what phase A leaves for phase B, per task of the tile
enum OutMode : uint8_t { OM_NONE = 0, OM_COPY, OM_STR_ESC /* one thread walks the token */, OM_U32_DEC, OM_I64_DEC, OM_VADD,
                         OM_STR_PAR /* warp transcodes the framed body in 32 chunks (drain2) */,
                         OM_DEFER /* identity main kernel: left to drain_slow_kernel */ };
struct TaskRec {
    uint32_t src_off;    // OM_COPY / OM_STR_ESC / OM_VADD: byte offset inside the payload
    uint32_t src_len;
    uint32_t out_len;
    uint8_t  status, has, mode, ready;
    long long value;     // OM_U32_DEC / OM_I64_DEC
};

// decimal digits of v. (Round 1 divided by ten in 64 bits, one lane per task while 31 idle: 6-9 % of the crc32 and json_sum
// kernels' instructions went into printing ~10 digits — profiles/r1_final_crc32_summary.txt. Now: compares against powers
// of ten and 32-bit multiply-shift division by 10, in at most three 9-digit limbs.)
__device__ __forceinline__ uint32_t dec_len_u32(uint32_t v) {
    return 1u + (v >= 10u) + (v >= 100u) + (v >= 1000u) + (v >= 10000u) + (v >= 100000u) + (v >= 1000000u) + (v >= 10000000u) + (v >= 100000000u) + (v >= 1000000000u);
}
__device__ __forceinline__ uint32_t dec_len_u64(unsigned long long v) {
    if (v < 4294967296ull) return dec_len_u32((uint32_t)v);
    const unsigned long long hi = v / 1000000000ull;                    // >= 4: v has more than 9 digits
    if (hi < 4294967296ull) return 9u + dec_len_u32((uint32_t)hi);
    return 18u + dec_len_u32((uint32_t)(hi / 1000000000ull));
}
// exactly n digits of x (x < 10^n), most significant first, zero-padded on the left
__device__ __forceinline__ void write_dec_u32(uint8_t* o, uint32_t x, uint32_t n) {
    for (uint32_t k = n; k-- > 0;) {
        const uint32_t q = (uint32_t)(((unsigned long long)x * 0xCCCCCCCDull) >> 35);   // x / 10
        o[k] = (uint8_t)('0' + (x - q * 10u));
        x = q;
    }
}
__device__ inline void write_dec(uint8_t* o, unsigned long long v, uint32_t len) {
    if (v < 4294967296ull) { write_dec_u32(o, (uint32_t)v, len); return; }
    const unsigned long long hi = v / 1000000000ull;
    write_dec_u32(o + (len - 9u), (uint32_t)(v - hi * 1000000000ull), 9u);
    if (hi < 4294967296ull) { write_dec_u32(o, (uint32_t)hi, len - 9u); return; }
    const unsigned long long top = hi / 1000000000ull;
    write_dec_u32(o + (len - 18u), (uint32_t)(hi - top * 1000000000ull), 9u);
    write_dec_u32(o, (uint32_t)top, len - 18u);
}

// String token p[s..e) (quotes included, validated): does the Python-escaped form equal a plain
// copy?  Computes the json.dumps length either way. One thread.
__device__ inline uint32_t py_string_len(const uint8_t* __restrict__ p, uint32_t s, uint32_t e) {
    uint32_t i = s + 1, end = e - 1, out = 2;
    while (i < end) out += py_escaped_len(next_cp(p, i, end));
    return out;
}

// Lane 0: classify args[0] for the handler and fill the record. `pr` is the parse of the payload.
__device__ inline void handler_phase_a(int handler, const uint8_t* __restrict__ p, const Parsed& pr, TaskRec& rec,
                                       const uint32_t* __restrict__ crc_table = nullptr) {
    rec.has = 0; rec.mode = OM_NONE; rec.out_len = 0; rec.src_off = 0; rec.src_len = 0; rec.value = 0;
    if (pr.status != ST_OK) { rec.status = pr.status; return; }
    // handler(*args, **kwargs) with a positional-only one-parameter handler
    if (pr.nargs != 1 || pr.kwargs_nonempty) { rec.status = 1 /* ERROR: TypeError */; return; }
    rec.status = 0;
    switch (handler) {
    case 0: {   // identity: result = args[0]; `serialize_result(result) if result else None`
        switch (pr.a0_kind) {
        case AK_STR:
            if (pr.a0_len == 2) return;                                     // "" is falsy
            rec.src_off = pr.a0_off; rec.src_len = pr.a0_len; rec.has = 1;
            if (!(pr.a0_flags & (SF_ESC | SF_NONPRINT))) { rec.mode = OM_COPY; rec.out_len = pr.a0_len; }
            else { rec.mode = OM_STR_ESC; rec.out_len = py_string_len(p, pr.a0_off, pr.a0_off + pr.a0_len); }
            return;
        case AK_NULL: case AK_FALSE: case AK_ARR_EMPTY: case AK_OBJ_EMPTY: return;   // falsy
        case AK_TRUE: rec.src_off = pr.a0_off; rec.src_len = 4; rec.out_len = 4; rec.mode = OM_COPY; rec.has = 1; return;
        case AK_INT: {
            // float64 integer -> Go prints the digits -> Python int -> same digits; "-0"/"0" falsy
            bool zero = true;
            for (uint32_t k = 0; k < pr.a0_len; ++k) { uint8_t c = p[pr.a0_off + k]; if (c != '-' && c != '0') zero = false; }
            if (zero) return;
            rec.src_off = pr.a0_off; rec.src_len = pr.a0_len; rec.out_len = pr.a0_len; rec.mode = OM_COPY; rec.has = 1; return;
        }
        default: rec.status = ST_UNSUPPORTED; return;                       // floats / non-empty containers
        }
    }
    case 1: {   // crc32: zlib.crc32(s.encode()); a non-str has no .encode -> AttributeError
        if (pr.a0_kind != AK_STR) { rec.status = 1; return; }
        uint32_t c = crc32_of_string_token(p, pr.a0_off, pr.a0_off + pr.a0_len, pr.a0_flags, crc_table);
        if (c == 0) return;                                                 // 0 is falsy
        rec.value = (long long)c; rec.out_len = dec_len_u64(c); rec.mode = OM_U32_DEC; rec.has = 1;
        return;
    }
    case 2: {   // vadd_f32: base64 -> fp32 a||b -> a+b -> base64
        if (pr.a0_kind != AK_STR) { rec.status = 1; return; }               // TypeError
        if (pr.a0_flags & SF_NONPRINT) { rec.status = 1; return; }          // non-ASCII / DEL: ValueError / binascii.Error
        if (pr.a0_flags & SF_ESC) {
            // escaped text: any decoded character outside the base64 alphabet is an error for sure;
            // a fully valid escaped base64 string (only "\/" can do that) is not produced by the SDK
            uint32_t i = pr.a0_off + 1, end = pr.a0_off + pr.a0_len - 1;
            while (i < end) { uint32_t cp = next_cp(p, i, end); if (cp >= 0x80 || (b64_val((uint8_t)cp) < 0 && cp != '=')) { rec.status = 1; return; } }
            rec.status = ST_UNSUPPORTED; return;
        }
        int64_t rn = b64_decoded_len(p, pr.a0_off + 1, pr.a0_off + pr.a0_len - 1);
        if (rn < 0 || (rn % 8)) { rec.status = 1; return; }
        uint32_t n = (uint32_t)(rn / 8);
        if (n == 0) return;                                                 // "" is falsy
        rec.src_off = pr.a0_off + 1; rec.src_len = n; rec.out_len = 2 + b64_encoded_len(4 * n); rec.mode = OM_VADD; rec.has = 1;
        return;
    }
    case 3: {   // json_sum: sum(obj["values"])
        if (pr.a0_kind != AK_OBJ) { rec.status = 1; return; }               // TypeError, or KeyError for {}
        long long sum = 0;
        int st = json_sum_object(p, pr.a0_off, pr.a0_off + pr.a0_len, &sum);
        if (st) { rec.status = (uint8_t)st; return; }
        if (sum == 0) return;
        rec.value = sum; rec.mode = OM_I64_DEC; rec.has = 1;
        const unsigned long long mag = sum < 0 ? 0ull - (unsigned long long)sum : (unsigned long long)sum;   // (INT64_MIN too)
        rec.out_len = dec_len_u64(mag) + (sum < 0 ? 1u : 0u);
        return;
    }
    default:
        rec.status = ST_UNSUPPORTED; return;
    }
}

// phase B for the modes that are not plain copies: writes exactly rec.out_len bytes at o
__device__ inline void seq_emit(const uint8_t* __restrict__ p, const TaskRec& rec, uint8_t* __restrict__ o) {
    if (rec.mode == OM_VADD) vadd_write(p, rec.src_off, rec.src_len, o);
    else if (rec.mode == OM_U32_DEC || rec.mode == OM_I64_DEC) {
        unsigned long long v = (unsigned long long)rec.value; uint32_t l = rec.out_len;
        if (rec.value < 0) { *o++ = '-'; --l; v = 0ull - v; }          // magnitude without a signed negation (INT64_MIN)
        write_dec(o, v, l);
    } else if (rec.mode == OM_STR_ESC) {                          // string the sequential parser sized (non-canonical frame)
        uint32_t i = rec.src_off + 1, end = rec.src_off + rec.src_len - 1;
        *o++ = '"';
        while (i < end) o += py_emit(next_cp(p, i, end), o);
        *o = '"';
    }
}

}  // namespace b9
