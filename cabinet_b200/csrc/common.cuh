// Shared device/host helpers for libcabinet_b200.so (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <algorithm>

#include "../../include/cabinet_b200.h"

// ----------------------------------------------------------------------------- error plumbing
void cabinet_set_error(const char* fmt, ...);

#define CAB_REQUIRE(cond, ...)                 \
    do {                                       \
        if (!(cond)) {                         \
            cabinet_set_error(__VA_ARGS__);    \
            return CABINET_ERR_INVALID;        \
        }                                      \
    } while (0)

#define CAB_CUDA(expr)                                                                          \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess) {                                                                \
            cabinet_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                              __LINE__);                                                        \
            return CABINET_ERR_CUDA;                                                            \
        }                                                                                       \
    } while (0)

#define CAB_LAUNCH_CHECK() CAB_CUDA(cudaGetLastError())

// ----------------------------------------------------------------------------- element types
// Every entry point that takes an element type checks it against the set it implements BEFORE any CUDA call, and the
// dispatch macros below decode exactly the three known codes: an unknown or unimplemented type is an error, never a
// silent reinterpretation of the bits as one of the other types.
#define CAB_DT_F32 (1 << CABINET_F32)
#define CAB_DT_BF16 (1 << CABINET_BF16)
#define CAB_DT_F16 (1 << CABINET_F16)
#define CAB_DT_ALL (CAB_DT_F32 | CAB_DT_BF16 | CAB_DT_F16)
static inline bool cab_dtype_ok(int dt, int mask) { return dt >= 0 && dt < 30 && ((mask >> dt) & 1); }
static inline const char* cab_dtype_name(int dt) {
    return dt == CABINET_F32 ? "fp32" : dt == CABINET_BF16 ? "bf16" : dt == CABINET_F16 ? "fp16" : "unknown";
}
#define CAB_REQUIRE_DTYPE(what, dt, mask)                                                                          \
    CAB_REQUIRE(cab_dtype_ok((dt), (mask)), "%s: element type %d (%s) is not implemented by this entry point", what, \
                static_cast<int>(dt), cab_dtype_name(dt))
static inline int cab_dtype_size(int dt) { return dt == CABINET_F32 ? 4 : 2; }
static inline long long cab_ceil_div(long long a, long long b) { return (a + b - 1) / b; }

// ----------------------------------------------------------------------------- device helpers
typedef __nv_bfloat16 bf16;
typedef __half f16;

// Host dispatch on one element type: runs the statement list with `T` = float / bf16 / f16.  The caller has
// validated `dt` (CAB_REQUIRE_DTYPE); anything else is still rejected here.
#define CAB_DISPATCH_DT(dt, T, ...)                                                                   \
    do {                                                                                              \
        if ((dt) == CABINET_F32) { typedef float T; __VA_ARGS__; }                                    \
        else if ((dt) == CABINET_BF16) { typedef bf16 T; __VA_ARGS__; }                               \
        else if ((dt) == CABINET_F16) { typedef f16 T; __VA_ARGS__; }                                 \
        else CAB_REQUIRE(false, "unsupported element type %d", static_cast<int>(dt));                 \
    } while (0)

// The same for the 2-byte types only (kernels that exist for bf16 and fp16 operands alone).
#define CAB_DISPATCH_DT_HALF(dt, T, ...)                                                              \
    do {                                                                                              \
        if ((dt) == CABINET_BF16) { typedef bf16 T; __VA_ARGS__; }                                    \
        else if ((dt) == CABINET_F16) { typedef f16 T; __VA_ARGS__; }                                 \
        else CAB_REQUIRE(false, "unsupported 2-byte element type %d", static_cast<int>(dt));          \
    } while (0)

// Host dispatch on two operands, each fp32 or the call's ONE 2-byte type (bf16 and fp16 never mix in a call):
// M(TA, TB) with the matching C++ types.
#define CAB_DISPATCH_DT_PAIR(da, db, M)                                                                             \
    do {                                                                                                            \
        const int _da = (da), _db = (db), _dh = _da != CABINET_F32 ? _da : _db;                                     \
        CAB_REQUIRE(cab_dtype_ok(_dh, CAB_DT_ALL) && (_da == CABINET_F32 || _da == _dh) &&                          \
                        (_db == CABINET_F32 || _db == _dh),                                                         \
                    "unsupported element type pair %d / %d", _da, _db);                                             \
        if (_dh == CABINET_F32) M(float, float);                                                                    \
        else if (_dh == CABINET_BF16) {                                                                             \
            if (_da == CABINET_F32) M(float, bf16); else if (_db == CABINET_F32) M(bf16, float); else M(bf16, bf16); \
        } else {                                                                                                    \
            if (_da == CABINET_F32) M(float, f16); else if (_db == CABINET_F32) M(f16, float); else M(f16, f16);     \
        }                                                                                                           \
    } while (0)

__device__ __forceinline__ float cab_act(float v, int act) {
    // reference: src/models/mobilenetv3.py:38-65 (relu6(x+3)/6, x*hsig(x)); nn.ReLU; nn.Sigmoid
    switch (act) {
        case CABINET_ACT_RELU: return fmaxf(v, 0.f);
        case CABINET_ACT_HSWISH: return v * (fminf(fmaxf(v + 3.f, 0.f), 6.f) / 6.f);
        case CABINET_ACT_HSIGMOID: return fminf(fmaxf(v + 3.f, 0.f), 6.f) / 6.f;
        case CABINET_ACT_SIGMOID: return 1.f / (1.f + __expf(-v));
        default: return v;
    }
}

// Activation over a small register array: ONE uniform branch per call, straight-line code per case
// (a per-element switch compiles to an indirect branch per element and serialises the whole epilogue).
template <int N> __device__ __forceinline__ void cab_act_vec(float* v, int act) {
    if (act == CABINET_ACT_RELU) {
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = fmaxf(v[i], 0.f);
    } else if (act == CABINET_ACT_HSWISH) {  // relu6(x + 3) / 6 == saturate(x / 6 + 0.5): one FFMA.SAT + one FMUL
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = v[i] * __saturatef(fmaf(v[i], 1.f / 6.f, 0.5f));
    } else if (act == CABINET_ACT_HSIGMOID) {
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = __saturatef(fmaf(v[i], 1.f / 6.f, 0.5f));
    } else if (act == CABINET_ACT_SIGMOID) {
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = 1.f / (1.f + __expf(-v[i]));
    }
}

// Packed fp32 FMA (Blackwell FFMA2): acc.{x,y} += x.{x,y} * w.{x,y} in ONE instruction -- two IEEE fp32 FMAs, bit-identical
// to two fmaf() calls.  The depthwise kernels keep (channel c, channel c+1) pairs in adjacent registers for this.
__device__ __forceinline__ void cab_ffma2(float2& acc, const float2 x, const float2 w) {
    uint64_t a, b, c;
    asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "f"(acc.x), "f"(acc.y));
    asm("mov.b64 %0, {%1, %2};" : "=l"(b) : "f"(x.x), "f"(x.y));
    asm("mov.b64 %0, {%1, %2};" : "=l"(c) : "f"(w.x), "f"(w.y));
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(a) : "l"(b), "l"(c));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(acc.x), "=f"(acc.y) : "l"(a));
}

template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<bf16>(bf16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ bf16 from_f32<bf16>(float v) { return __float2bfloat16_rn(v); }
// fp16: round to nearest, overflow -> inf (never saturating: a loss-scale overflow must reach the gradients as inf)
template <> __device__ __forceinline__ float to_f32<f16>(f16 v) { return __half2float(v); }
template <> __device__ __forceinline__ f16 from_f32<f16>(float v) { return __float2half_rn(v); }

// Two packed 2-byte elements (one 32-bit word: element 0 in the low half) -> fp32
template <typename T> __device__ __forceinline__ float2 cab_unpack2(uint32_t w);
template <> __device__ __forceinline__ float2 cab_unpack2<bf16>(uint32_t w) {  // bf16 -> f32 is a 16-bit shift
    return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
}
template <> __device__ __forceinline__ float2 cab_unpack2<f16>(uint32_t w) {
    __half2 h;
    *reinterpret_cast<uint32_t*>(&h) = w;
    return __half22float2(h);
}
// fp32 pair -> two packed 2-byte elements (round to nearest; fp16 overflow -> inf)
template <typename T> __device__ __forceinline__ uint32_t cab_pack2(float lo, float hi);
template <> __device__ __forceinline__ uint32_t cab_pack2<bf16>(float lo, float hi) {
    __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&h);
}
template <> __device__ __forceinline__ uint32_t cab_pack2<f16>(float lo, float hi) {
    __half2 h = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&h);
}

// 16-byte vector of T: 4 floats or 8 bf16 / fp16
template <typename T> struct Vec16;
template <> struct Vec16<float> {
    static constexpr int N = 4;
    float4 raw;
    __device__ __forceinline__ void load(const float* p) { raw = *reinterpret_cast<const float4*>(p); }
    __device__ __forceinline__ void store(float* p) const { *reinterpret_cast<float4*>(p) = raw; }
    __device__ __forceinline__ void unpack(float* f) const { f[0] = raw.x; f[1] = raw.y; f[2] = raw.z; f[3] = raw.w; }
    __device__ __forceinline__ void pack(const float* f) { raw = make_float4(f[0], f[1], f[2], f[3]); }
};
template <typename T> struct Vec16Half {  // T = bf16 or f16
    static constexpr int N = 8;
    uint4 raw;
    __device__ __forceinline__ void load(const T* p) { raw = *reinterpret_cast<const uint4*>(p); }
    __device__ __forceinline__ void store(T* p) const { *reinterpret_cast<uint4*>(p) = raw; }
    __device__ __forceinline__ void unpack(float* f) const {
        const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float2 v = cab_unpack2<T>(w[i]);
            f[2 * i] = v.x;
            f[2 * i + 1] = v.y;
        }
    }
    __device__ __forceinline__ void pack(const float* f) {
        raw = make_uint4(cab_pack2<T>(f[0], f[1]), cab_pack2<T>(f[2], f[3]), cab_pack2<T>(f[4], f[5]), cab_pack2<T>(f[6], f[7]));
    }
};
template <> struct Vec16<bf16> : Vec16Half<bf16> {};
template <> struct Vec16<f16> : Vec16Half<f16> {};

// Bilinear source taps, align_corners=False (ATen area_pixel_compute_source_index; reference call sites
// src/models/cabinet.py:228-245, src/models/cab.py:70-72). scale = in/out as float.
__device__ __forceinline__ void cab_bilinear_tap(int dst, float scale, int in_size, int& i0, int& i1, float& w1) {
    float src = fmaxf((static_cast<float>(dst) + 0.5f) * scale - 0.5f, 0.f);
    i0 = min(static_cast<int>(src), in_size - 1);
    i1 = min(i0 + 1, in_size - 1);
    w1 = src - static_cast<float>(i0);
}
