// Shared device/host helpers for libspt_b200 (sm_100a).  No torch headers anywhere in csrc/.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>

#include "../../include/spt_b200.h"

namespace spt {

// ---- error plumbing ---------------------------------------------------------------------
extern thread_local char g_last_error[512];
extern std::atomic<uint64_t> g_launch_count;

inline int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_last_error, sizeof(g_last_error), fmt, ap);
    va_end(ap);
    return code;
}

#define SPT_REQUIRE(cond, ...)                                              \
    do {                                                                    \
        if (!(cond)) return ::spt::fail(SPT_ERR_INVALID_ARGUMENT, __VA_ARGS__); \
    } while (0)

// Counts the launch and converts a launch error into an spt_status.
inline int after_launch(const char *what) {
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(SPT_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
    return SPT_OK;
}

#define SPT_LAUNCH_CHECK(what)                   \
    do {                                         \
        int _rc = ::spt::after_launch(what);     \
        if (_rc != SPT_OK) return _rc;           \
    } while (0)

inline cudaStream_t as_stream(spt_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

inline int num_sms() {   // of the CURRENT device (one process may drive several): cached per device index
    static int cache[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && cache[dev] > 0) return cache[dev];
    int n = 0;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
    if (dev >= 0 && dev < 64) cache[dev] = n;   // benign race: every writer stores the same value
    return n;
}

// ---- packed variable-length sequences (varlen.cu) ----------------------------------------------
// Work list: int32 [0] = item count, [4 ..) int4 items {first token, length, 128-row tile, bitmap word offset} in
// descending tile order, then int4 per sequence (scratch of the builder).  sum ceil(S_i / 128) <= ceil(T / 128) + n_seq.
__host__ __device__ inline int64_t varlen_capacity(int n_seq, int T) { return ((int64_t)T + 127) / 128 + n_seq; }
constexpr int VARLEN_MAX_SEQLEN = 65536;
// argument checks shared by every varlen entry point; they come before any CUDA call
inline int check_varlen(const char *what, int n_seq, int T, int max_seqlen, int H) {
    if (n_seq < 1) return fail(SPT_ERR_INVALID_ARGUMENT, "%s: need n_seq >= 1 (got %d)", what, n_seq);
    if (T < 1) return fail(SPT_ERR_INVALID_ARGUMENT, "%s: need T >= 1 tokens (got %d)", what, T);
    if (H < 1) return fail(SPT_ERR_INVALID_ARGUMENT, "%s: need H >= 1 heads (got %d)", what, H);
    if (max_seqlen < 1 || max_seqlen > VARLEN_MAX_SEQLEN)
        return fail(SPT_ERR_INVALID_ARGUMENT, "%s: max_seqlen %d outside [1, %d]", what, max_seqlen, VARLEN_MAX_SEQLEN);
    if (varlen_capacity(n_seq, T) > 65535)
        return fail(SPT_ERR_INVALID_ARGUMENT, "%s: ceil(T / 128) + n_seq = %lld work items exceed the grid limit 65535", what,
                    (long long)varlen_capacity(n_seq, T));
    return SPT_OK;
}

// ---- device helpers -----------------------------------------------------------------------
constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

template <int WIDTH>
__device__ __forceinline__ float group_sum(float v) {  // butterfly inside aligned groups of WIDTH lanes
#pragma unroll
    for (int o = WIDTH / 2; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

// streaming (evict-first) 128-bit accessors for data touched exactly once
__device__ __forceinline__ int4 ld_stream(const int4 *p) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ float4 ld_stream(const float4 *p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream(float4 *p, const float4 &v) {
    asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                 : "memory");
}
__device__ __forceinline__ void st_stream(int4 *p, const int4 &v) {
    asm volatile("st.global.cs.v4.s32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
                 : "memory");
}

// Element loaders: VEC consecutive elements of type T -> fp32.
// f32: VEC = 4 (16 B); bf16: VEC = 8 (16 B).
template <typename T>
struct Vec16;
template <>
struct Vec16<float> {
    static constexpr int N = 4;
    __device__ __forceinline__ static void load(const float *p, float (&o)[4]) {
        float4 v = *reinterpret_cast<const float4 *>(p);
        o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
    }
    __device__ __forceinline__ static void store(float *p, const float (&o)[4]) {
        *reinterpret_cast<float4 *>(p) = make_float4(o[0], o[1], o[2], o[3]);
    }
};
template <>
struct Vec16<__nv_bfloat16> {
    static constexpr int N = 8;
    __device__ __forceinline__ static void load(const __nv_bfloat16 *p, float (&o)[8]) {
        uint4 v = *reinterpret_cast<const uint4 *>(p);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {  // bf16 -> fp32 is a 16-bit shift: exact
            o[2 * i] = __uint_as_float(w[i] << 16);
            o[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
        }
    }
    __device__ __forceinline__ static void store(__nv_bfloat16 *p, const float (&o)[8]) {
        uint32_t w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            __nv_bfloat162 h = __floats2bfloat162_rn(o[2 * i], o[2 * i + 1]);
            w[i] = *reinterpret_cast<uint32_t *>(&h);
        }
        *reinterpret_cast<uint4 *>(p) = make_uint4(w[0], w[1], w[2], w[3]);
    }
};

template <>
struct Vec16<__half> {
    static constexpr int N = 8;
    __device__ __forceinline__ static void load(const __half *p, float (&o)[8]) {
        uint4 v = *reinterpret_cast<const uint4 *>(p);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {  // fp16 -> fp32: exact
            const float2 f = __half22float2(*reinterpret_cast<const __half2 *>(&w[i]));
            o[2 * i] = f.x;
            o[2 * i + 1] = f.y;
        }
    }
    __device__ __forceinline__ static void store(__half *p, const float (&o)[8]) {
        uint32_t w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            __half2 h = __floats2half2_rn(o[2 * i], o[2 * i + 1]);
            w[i] = *reinterpret_cast<uint32_t *>(&h);
        }
        *reinterpret_cast<uint4 *>(p) = make_uint4(w[0], w[1], w[2], w[3]);
    }
};

__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(__nv_bfloat16 v) { return __bfloat162float(v); }
__device__ __forceinline__ float to_f32(__half v) { return __half2float(v); }
template <typename T>
__device__ __forceinline__ T from_f32(float v);
template <>
__device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <>
__device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <>
__device__ __forceinline__ __half from_f32<__half>(float v) { return __float2half_rn(v); }

}  // namespace spt
