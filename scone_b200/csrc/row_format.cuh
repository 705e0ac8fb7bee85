// row_format.cuh -- the stored row formats of the cache table, defined once: layout and validation (host), scales,
// chunk reader, decoders and chunk writer (device), and the run-time format -> template dispatch (host).
//
// A stored row is its payload (dim elements in order), then for INT8 / INT4 its scales at scale_offset, then padding up to
// row_stride.  The formulas are those of oracle/py_oracle.py (SURVEY.md section 8c, DESIGN.md section 3):
//   FP32  4 bytes per element                                               no scales
//   FP16  2 bytes per element                                               no scales
//   INT8  1 byte per element (q, int8)                                      one fp32 scale per row, 4-byte aligned
//   INT4  one nibble per element (q + 8, element 0 in the low nibble)       one fp16 scale per group, 2-byte aligned;
//         the group is a power of two >= 8 dividing dim
// The kernels read a row in chunks of 8 consecutive elements (dim is a multiple of 8).
#pragma once
#include "common.cuh"

#include <type_traits>

namespace scone {

// ---------------------------------------------------------------------------------------------
// layout (host): what scone_table_layout produces and check_table accepts
// ---------------------------------------------------------------------------------------------
inline int64_t payload_bytes(int32_t quant, int32_t dim) {
    return quant == SCONE_QUANT_FP32 ? 4ll * dim : quant == SCONE_QUANT_FP16 ? 2ll * dim : quant == SCONE_QUANT_INT8 ? dim : dim / 2;
}
// 0 for the formats without scales; INT4 needs a valid group
inline int64_t scale_bytes(int32_t quant, int32_t dim, int32_t group) {
    return quant == SCONE_QUANT_INT8 ? 4 : quant == SCONE_QUANT_INT4 ? 2ll * (dim / group) : 0;
}
inline int32_t scale_align(int32_t quant) { return quant == SCONE_QUANT_INT8 ? 4 : 2; }
inline bool valid_int4_group(int32_t group) { return group >= 8 && (group & (group - 1)) == 0; }
// log2(group / 8): chunk c of an INT4 row uses scale c >> group_shift (only INT4 reads it)
inline int32_t group_shift(int32_t group) {
    int32_t sh = 0;
    while ((1 << sh) < group / 8) ++sh;
    return sh;
}

// Validates a table descriptor against the layout rule above (table.cu); `who` names the caller in the error message.
int check_table(const scone_table_desc_t *t, const char *who);

// ---------------------------------------------------------------------------------------------
// format dispatch (host): calls f(std::integral_constant<int, V>{}) for the V of Vs equal to `v`, a SCONE_QUANT_* or
// SCONE_OUT_* value the caller has validated
// ---------------------------------------------------------------------------------------------
template <int... Vs, class F>
void with_constant(int32_t v, F &&f) {
    ((v == Vs ? f(std::integral_constant<int, Vs>{}) : void()), ...);
}

#ifdef __CUDACC__

// ---------------------------------------------------------------------------------------------
// scales: store_kernel and the projection fold's epilogue (held bit-identical to it) both use these
// ---------------------------------------------------------------------------------------------
// INT8: one fp32 scale per row, amax / 127; 1 for an all-zero row
__device__ __forceinline__ float int8_row_scale(float amax) {
    const float s = __fdiv_rn(amax, 127.0f);
    return s == 0.0f ? 1.0f : s;
}
// INT4: one fp16 scale per group, amax / 7 (at most the fp16 maximum); 1 for an all-zero group
__device__ __forceinline__ __half int4_group_scale(float amax) {
    const __half s = __float2half_rn(fminf(__fdiv_rn(amax, 7.0f), 65504.0f));
    return __half2float(s) == 0.0f ? __float2half_rn(1.0f) : s;
}

// ---------------------------------------------------------------------------------------------
// decode of 8 consecutive elements to fp32 (exact integer -> float, then ONE fp32 multiply).
// Values travel as four float2 pairs (elements 2k, 2k+1) so that the adds and multiplies issue as the sm_100 packed
// instructions FADD2 / FMUL2 (two IEEE round-to-nearest fp32 operations per instruction -- the same roundings as the
// scalar forms, half the issue slots) and the pairs feed cvt.rn.{bf16x2,f16x2}.f32 directly.
// ---------------------------------------------------------------------------------------------
typedef float2 f32x8[4];

__device__ __forceinline__ void decode_fp16x8(uint4 raw, f32x8 &x) {
    const __half2 *h = reinterpret_cast<const __half2 *>(&raw);
#pragma unroll
    for (int k = 0; k < 4; ++k) x[k] = __half22float2(h[k]);
}
__device__ __forceinline__ void decode_bf16x8(uint4 raw, f32x8 &x) {
    const uint32_t *u = reinterpret_cast<const uint32_t *>(&raw);
#pragma unroll
    for (int k = 0; k < 4; ++k) x[k] = make_float2(__uint_as_float(u[k] << 16), __uint_as_float(u[k] & 0xFFFF0000u));
}
// unquantised rows (SCONE_QUANT_FP32): eight floats = two 16-byte vectors
__device__ __forceinline__ void decode_fp32x8(uint4 a, uint4 b, f32x8 &x) {
    x[0] = make_float2(__uint_as_float(a.x), __uint_as_float(a.y));
    x[1] = make_float2(__uint_as_float(a.z), __uint_as_float(a.w));
    x[2] = make_float2(__uint_as_float(b.x), __uint_as_float(b.y));
    x[3] = make_float2(__uint_as_float(b.z), __uint_as_float(b.w));
}
// int8 -> fp32 without the I2F pipe: place (q ^ 0x80) in the low mantissa byte of 2^23 and
// subtract 2^23 + 128; both steps are exact.
__device__ __forceinline__ void decode_int8x8(uint2 raw, float scale, f32x8 &x) {
    const uint32_t w[2] = {raw.x ^ 0x80808080u, raw.y ^ 0x80808080u};
    const float2 bias = make_float2(-8388736.0f, -8388736.0f), sc = make_float2(scale, scale);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t m0 = __byte_perm(w[k >> 1], 0x4B000000u, 0x7650 + ((2 * k) & 3));  // bytes: [q, 0, 0, 0x4B]
        const uint32_t m1 = __byte_perm(w[k >> 1], 0x4B000000u, 0x7650 + ((2 * k + 1) & 3));
        x[k] = __fmul2_rn(__fadd2_rn(make_float2(__uint_as_float(m0), __uint_as_float(m1)), bias), sc);
    }
}
// eight nibbles (q + 8), element 0 in the lowest nibble: split into even / odd elements (one byte each), then the
// same mantissa placement as int8
__device__ __forceinline__ void decode_int4x8(uint32_t raw, float scale, f32x8 &x) {
    const uint32_t ev = raw & 0x0F0F0F0Fu, od = (raw >> 4) & 0x0F0F0F0Fu;  // elements 0,2,4,6 / 1,3,5,7
    const float2 bias = make_float2(-8388616.0f, -8388616.0f), sc = make_float2(scale, scale);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t m0 = __byte_perm(ev, 0x4B000000u, 0x7650 + k);
        const uint32_t m1 = __byte_perm(od, 0x4B000000u, 0x7650 + k);
        x[k] = __fmul2_rn(__fadd2_rn(make_float2(__uint_as_float(m0), __uint_as_float(m1)), bias), sc);
    }
}
__device__ __forceinline__ void zero8(f32x8 &x) {
#pragma unroll
    for (int k = 0; k < 4; ++k) x[k] = make_float2(0.0f, 0.0f);
}
// x += y, eight fp32 round-to-nearest adds (four FADD2)
__device__ __forceinline__ void add8(f32x8 &x, const f32x8 &y) {
#pragma unroll
    for (int k = 0; k < 4; ++k) x[k] = __fadd2_rn(x[k], y[k]);
}

__device__ __forceinline__ uint4 pack_bf16x8(const f32x8 &x) {
    uint4 r;
    uint32_t *u = reinterpret_cast<uint32_t *>(&r);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        __nv_bfloat162 b = __float22bfloat162_rn(x[k]);
        u[k] = *reinterpret_cast<uint32_t *>(&b);
    }
    return r;
}
__device__ __forceinline__ uint4 pack_fp16x8(const f32x8 &x) {
    uint4 r;
    uint32_t *u = reinterpret_cast<uint32_t *>(&r);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        __half2 b = __float22half2_rn(x[k]);
        u[k] = *reinterpret_cast<uint32_t *>(&b);
    }
    return r;
}

// ---------------------------------------------------------------------------------------------
// where a chunk is read from.  Each kind keeps the caching its readers were measured with; the global kinds read
// scales through ld.global.nc.
// ---------------------------------------------------------------------------------------------
struct GlobalRows {  // streamed global rows: ld.global.nc.L1::no_allocate
    __device__ __forceinline__ uint4 v16(const uint8_t *a) const { return ldg_stream_16(a); }
    __device__ __forceinline__ uint2 v8(const uint8_t *a) const { return ldg_stream_8(a); }
    __device__ __forceinline__ uint32_t v4(const uint8_t *a) const { return ldg_stream_4(a); }
    template <class T>
    __device__ __forceinline__ T scale(const T *a) const { return __ldg(a); }
};
struct GlobalRowsEvictFirst : GlobalRows {  // streamed global rows with the L2 evict-first policy `pol`
    uint64_t pol;
    __device__ __forceinline__ uint4 v16(const uint8_t *a) const { return ldg_stream_16(a, pol); }
    __device__ __forceinline__ uint2 v8(const uint8_t *a) const { return ldg_stream_8(a, pol); }
    __device__ __forceinline__ uint32_t v4(const uint8_t *a) const { return ldg_stream_4(a, pol); }
};
struct GlobalRowsCached : GlobalRows {  // global rows re-read by many positions (position rows): ld.global.nc, L1 allocating
    __device__ __forceinline__ uint4 v16(const uint8_t *a) const { return __ldg(reinterpret_cast<const uint4 *>(a)); }
};
struct SharedRows {  // rows staged in shared memory
    __device__ __forceinline__ uint4 v16(const uint8_t *a) const { return *reinterpret_cast<const uint4 *>(a); }
    __device__ __forceinline__ uint2 v8(const uint8_t *a) const { return *reinterpret_cast<const uint2 *>(a); }
    __device__ __forceinline__ uint32_t v4(const uint8_t *a) const { return *reinterpret_cast<const uint32_t *>(a); }
    template <class T>
    __device__ __forceinline__ T scale(const T *a) const { return *a; }
};

// ---------------------------------------------------------------------------------------------
// chunk reader: the raw bytes of chunk c and their scale (load_chunk), then fp32 (decode_chunk).  Split so that a reader
// can put several chunks' loads in flight before it decodes any of them.  `rs` is the row_scale of the row.
// ---------------------------------------------------------------------------------------------
struct RawChunk {
    uint4 a, b;   // payload: FP32 a and b, FP16 a, INT8 a.x and a.y, INT4 a.x
    float scale;  // INT8 / INT4
};

// INT8 rows have one scale, which a reader loads once per row and hands to load_chunk; 1 for the other formats
template <int QUANT, class Mem>
__device__ __forceinline__ float row_scale(const Mem &m, const uint8_t *row, int scale_off) {
    return QUANT == SCONE_QUANT_INT8 ? m.scale(reinterpret_cast<const float *>(row + scale_off)) : 1.0f;
}

template <int QUANT, class Mem>
__device__ __forceinline__ RawChunk load_chunk(const Mem &m, const uint8_t *row, int c, int scale_off, int group_shift, float rs) {
    RawChunk r;
    r.scale = rs;
    if (QUANT == SCONE_QUANT_FP32) {
        r.a = m.v16(row + c * 32);
        r.b = m.v16(row + c * 32 + 16);
    } else if (QUANT == SCONE_QUANT_FP16) {
        r.a = m.v16(row + c * 16);
    } else if (QUANT == SCONE_QUANT_INT8) {
        const uint2 v = m.v8(row + c * 8);
        r.a.x = v.x;
        r.a.y = v.y;
    } else {
        r.scale = __half2float(m.scale(reinterpret_cast<const __half *>(row + scale_off) + (c >> group_shift)));
        r.a.x = m.v4(row + c * 4);
    }
    return r;
}

template <int QUANT>
__device__ __forceinline__ void decode_chunk(const RawChunk &r, f32x8 &x) {
    if (QUANT == SCONE_QUANT_FP32) decode_fp32x8(r.a, r.b, x);
    else if (QUANT == SCONE_QUANT_FP16) decode_fp16x8(r.a, x);
    else if (QUANT == SCONE_QUANT_INT8) decode_int8x8(make_uint2(r.a.x, r.a.y), r.scale, x);
    else decode_int4x8(r.a.x, r.scale, x);
}

// ---------------------------------------------------------------------------------------------
// chunk writer: 8 fp32 values in the output type OUT, round-to-nearest-even.  FP32 is two 16-byte vectors, BF16 / FP16
// one (v[0]); a pointer to OutChunk<OUT> stores the chunk with 16-byte vector stores.
// ---------------------------------------------------------------------------------------------
template <int OUT>
struct OutChunk {
    uint4 v[OUT == SCONE_OUT_FP32 ? 2 : 1];
};

template <int OUT>
__device__ __forceinline__ OutChunk<OUT> pack_chunk(const f32x8 &x) {
    OutChunk<OUT> o;
    if constexpr (OUT == SCONE_OUT_FP32) {
        o.v[0] = make_uint4(__float_as_uint(x[0].x), __float_as_uint(x[0].y), __float_as_uint(x[1].x), __float_as_uint(x[1].y));
        o.v[1] = make_uint4(__float_as_uint(x[2].x), __float_as_uint(x[2].y), __float_as_uint(x[3].x), __float_as_uint(x[3].y));
    } else {
        o.v[0] = OUT == SCONE_OUT_BF16 ? pack_bf16x8(x) : pack_fp16x8(x);
    }
    return o;
}

#endif  // __CUDACC__

}  // namespace scone
