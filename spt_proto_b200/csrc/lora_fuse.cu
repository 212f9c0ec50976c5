// Fused elementwise stages of the LoRA-routed FFN (reference naive_gpt/layers/tuning/lora_ffn.py:87-115,201-222),
// which the reference (and the first version here) runs as chains of torch elementwise ops over [R, bs] fp32
// tensors — ~30 small launches per layer and pass, each re-reading 50 MB at the LLaMA-7B shape:
//
//   scale_add : out[r, c] = coeff[r] * a[r, c] + b[r, c]                      (coeff = 2 * router prob of the row)
//               bwd: da = coeff * dout, dcoeff[r] = sum_c dout[r, c] * a[r, c]   (db = dout: no kernel)
//   lora_glu  : h[r, c] = silu(coeff[r] * bg + lg) * (coeff[r] * bs + ls)    -> bf16 / fp16   (LLaMA gate / side)
//               bwd: dg = dh * s * silu'(g), ds = dh * silu(g);
//                    d_bg = coeff * dg, d_lg = dg, d_bs = coeff * ds, d_ls = ds,
//                    dcoeff[r] = sum_c (dg * bg + ds * bs)
// One block per row; 128-bit loads; the row reduction of dcoeff in fixed order (deterministic).
#include <initializer_list>

#include "common.cuh"

namespace spt {
namespace lfuse {

constexpr int THREADS = 256;

template <typename T>
__device__ __forceinline__ void load4(const T *p, float (&v)[4]);
template <>
__device__ __forceinline__ void load4<float>(const float *p, float (&v)[4]) {
    const float4 t = *reinterpret_cast<const float4 *>(p);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
template <>
__device__ __forceinline__ void load4<__nv_bfloat16>(const __nv_bfloat16 *p, float (&v)[4]) {
    const uint2 t = *reinterpret_cast<const uint2 *>(p);
    v[0] = __uint_as_float(t.x << 16); v[1] = __uint_as_float(t.x & 0xffff0000u);
    v[2] = __uint_as_float(t.y << 16); v[3] = __uint_as_float(t.y & 0xffff0000u);
}
template <>
__device__ __forceinline__ void load4<__half>(const __half *p, float (&v)[4]) {
    const uint2 t = *reinterpret_cast<const uint2 *>(p);
    const float2 lo = __half22float2(*reinterpret_cast<const __half2 *>(&t.x));
    const float2 hi = __half22float2(*reinterpret_cast<const __half2 *>(&t.y));
    v[0] = lo.x; v[1] = lo.y; v[2] = hi.x; v[3] = hi.y;
}
template <typename T>
__device__ __forceinline__ void store4(T *p, const float (&v)[4]);
template <>
__device__ __forceinline__ void store4<float>(float *p, const float (&v)[4]) {
    *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]);
}
template <>
__device__ __forceinline__ void store4<__nv_bfloat16>(__nv_bfloat16 *p, const float (&v)[4]) {
    __nv_bfloat162 lo = __floats2bfloat162_rn(v[0], v[1]), hi = __floats2bfloat162_rn(v[2], v[3]);
    uint2 t;
    t.x = *reinterpret_cast<uint32_t *>(&lo);
    t.y = *reinterpret_cast<uint32_t *>(&hi);
    *reinterpret_cast<uint2 *>(p) = t;
}

template <>
__device__ __forceinline__ void store4<__half>(__half *p, const float (&v)[4]) {
    __half2 lo = __floats2half2_rn(v[0], v[1]), hi = __floats2half2_rn(v[2], v[3]);
    uint2 t;
    t.x = *reinterpret_cast<uint32_t *>(&lo);
    t.y = *reinterpret_cast<uint32_t *>(&hi);
    *reinterpret_cast<uint2 *>(p) = t;
}

__device__ __forceinline__ float block_sum(float v) {   // fixed-order block reduction, result in every thread of warp 0
    __shared__ float s_red[THREADS / 32];
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    float t = 0.0f;
    if (threadIdx.x < 32) {
#pragma unroll
        for (int i = 0; i < THREADS / 32; ++i) t += s_red[i];
    }
    return t;
}

template <typename TA, typename TB, typename TO>
__global__ void __launch_bounds__(THREADS)
scale_add_fwd_kernel(const float *__restrict__ coeff, const TA *__restrict__ a, const TB *__restrict__ b,
                     TO *__restrict__ out, int C) {
    const size_t row = blockIdx.x;
    const float cf = coeff[row];
    for (int c = threadIdx.x * 4; c < C; c += THREADS * 4) {
        float av[4], bv[4], o[4];
        load4(a + row * C + c, av);
        load4(b + row * C + c, bv);
#pragma unroll
        for (int i = 0; i < 4; ++i) o[i] = fmaf(cf, av[i], bv[i]);
        store4(out + row * C + c, o);
    }
}

template <typename TA, typename TG>
__global__ void __launch_bounds__(THREADS)
scale_add_bwd_kernel(const float *__restrict__ coeff, const TA *__restrict__ a, const TG *__restrict__ dout,
                     TA *__restrict__ da, float *__restrict__ dcoeff, int C) {
    const size_t row = blockIdx.x;
    const float cf = coeff[row];
    float acc = 0.0f;
    for (int c = threadIdx.x * 4; c < C; c += THREADS * 4) {
        float av[4], gv[4], o[4];
        load4(a + row * C + c, av);
        load4(dout + row * C + c, gv);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            o[i] = cf * gv[i];
            acc = fmaf(gv[i], av[i], acc);
        }
        store4(da + row * C + c, o);
    }
    acc = block_sum(acc);
    if (threadIdx.x == 0) dcoeff[row] = acc;
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + __expf(-x)); }

template <typename TH>   // h: bf16 or fp16
__global__ void __launch_bounds__(THREADS)
lora_glu_fwd_kernel(const float *__restrict__ coeff, const float *__restrict__ bg, const float *__restrict__ lg,
                    const float *__restrict__ bs, const float *__restrict__ ls, TH *__restrict__ h, int C) {
    const size_t row = blockIdx.x;
    const float cf = coeff[row];
    for (int c = threadIdx.x * 4; c < C; c += THREADS * 4) {
        float a[4], b[4], x[4], y[4], o[4];
        load4(bg + row * C + c, a);
        load4(lg + row * C + c, b);
        load4(bs + row * C + c, x);
        load4(ls + row * C + c, y);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float g = fmaf(cf, a[i], b[i]), s = fmaf(cf, x[i], y[i]);
            o[i] = g * sigmoidf_(g) * s;
        }
        store4(h + row * C + c, o);
    }
}

template <typename TH>
__global__ void __launch_bounds__(THREADS)
lora_glu_bwd_kernel(const float *__restrict__ coeff, const float *__restrict__ bg, const float *__restrict__ lg,
                    const float *__restrict__ bs, const float *__restrict__ ls, const TH *__restrict__ dh,
                    float *__restrict__ d_bg, float *__restrict__ d_lg, float *__restrict__ d_bs,
                    float *__restrict__ d_ls, float *__restrict__ dcoeff, int C) {
    const size_t row = blockIdx.x;
    const float cf = coeff[row];
    float acc = 0.0f;
    for (int c = threadIdx.x * 4; c < C; c += THREADS * 4) {
        float a[4], b[4], x[4], y[4], gh[4], o1[4], o2[4], o3[4], o4[4];
        load4(bg + row * C + c, a);
        load4(lg + row * C + c, b);
        load4(bs + row * C + c, x);
        load4(ls + row * C + c, y);
        load4(dh + row * C + c, gh);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float g = fmaf(cf, a[i], b[i]), s = fmaf(cf, x[i], y[i]);
            const float sg = sigmoidf_(g);
            const float act = g * sg;
            const float dact = sg * (1.0f + g * (1.0f - sg));      // d silu / dg
            const float dg = gh[i] * s * dact, ds = gh[i] * act;
            o1[i] = cf * dg;
            o2[i] = dg;
            o3[i] = cf * ds;
            o4[i] = ds;
            acc = fmaf(dg, a[i], fmaf(ds, x[i], acc));
        }
        store4(d_bg + row * C + c, o1);
        store4(d_lg + row * C + c, o2);
        store4(d_bs + row * C + c, o3);
        store4(d_ls + row * C + c, o4);
    }
    acc = block_sum(acc);
    if (threadIdx.x == 0) dcoeff[row] = acc;
}

// plain gated unit of RoutedLLaMaFFN (layers/sparse/feedforward.py:172-176, `act(gate) * side` with act = SiLU): bf16 or
// fp16 in / out, fp32 math, 8 elements (16 bytes) per thread; the backward gives both gradients in one pass
template <typename T>
__global__ void __launch_bounds__(THREADS)
silu_mul_fwd_kernel(const T *__restrict__ g, const T *__restrict__ s, T *__restrict__ h, int64_t n8) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
        float a[8], b[8], o[8];
        Vec16<T>::load(g + 8 * i, a);
        Vec16<T>::load(s + 8 * i, b);
#pragma unroll
        for (int u = 0; u < 8; ++u) o[u] = a[u] * sigmoidf_(a[u]) * b[u];
        Vec16<T>::store(h + 8 * i, o);
    }
}

template <typename T>
__global__ void __launch_bounds__(THREADS)
silu_mul_bwd_kernel(const T *__restrict__ g, const T *__restrict__ s, const T *__restrict__ dh, T *__restrict__ dg,
                    T *__restrict__ ds, int64_t n8) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
        float a[8], b[8], gh[8], o1[8], o2[8];
        Vec16<T>::load(g + 8 * i, a);
        Vec16<T>::load(s + 8 * i, b);
        Vec16<T>::load(dh + 8 * i, gh);
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const float sg = sigmoidf_(a[u]);
            o1[u] = gh[u] * b[u] * sg * (1.0f + a[u] * (1.0f - sg));      // d silu / dg
            o2[u] = gh[u] * a[u] * sg;
        }
        Vec16<T>::store(dg + 8 * i, o1);
        Vec16<T>::store(ds + 8 * i, o2);
    }
}

}  // namespace lfuse
}  // namespace spt

using namespace spt;

static int check_rc(const char *what, int64_t R, int C) {
    if (R < 1 || R > 0x7fffffff || C < 4 || C % 4 != 0)
        return fail(SPT_ERR_INVALID_ARGUMENT, "%s: need 1 <= rows < 2^31 and columns a positive multiple of 4 (R=%lld C=%d)", what,
                    (long long)R, C);
    return SPT_OK;
}

// The 16-bit type of a set of operand dtypes, each SPT_F32 or a 16-bit type: SPT_BF16 / SPT_F16 (SPT_BF16 when all are
// fp32), or -1 when one is unknown or bf16 meets fp16.
static int half_kind(std::initializer_list<int> dtypes) {
    int kind = 0;
    for (int d : dtypes) {
        if (d == SPT_F32) continue;
        if ((d != SPT_BF16 && d != SPT_F16) || (kind && kind != d)) return -1;
        kind = d;
    }
    return kind ? kind : SPT_BF16;
}

// a, b, out: each fp32 or one 16-bit type H (bf16 or fp16); key bit = "is H"
template <typename H>
static void scale_add_fwd_launch(int key, const float *coeff, const void *a, const void *b, void *out, int64_t R, int C,
                                 cudaStream_t st) {
    const unsigned grid = (unsigned)R;
#define SPT_SA(TA, TB, TO) lfuse::scale_add_fwd_kernel<TA, TB, TO><<<grid, lfuse::THREADS, 0, st>>>(coeff, (const TA *)a, (const TB *)b, (TO *)out, C)
    switch (key) {
        case 0: SPT_SA(float, float, float); break;
        case 1: SPT_SA(float, float, H); break;
        case 2: SPT_SA(float, H, float); break;
        case 3: SPT_SA(float, H, H); break;
        case 4: SPT_SA(H, float, float); break;
        case 5: SPT_SA(H, float, H); break;
        case 6: SPT_SA(H, H, float); break;
        default: SPT_SA(H, H, H); break;
    }
#undef SPT_SA
}

extern "C" int spt_scale_add_fwd(const float *coeff, const void *a, int a_dtype, const void *b, int b_dtype, void *out,
                                 int o_dtype, int64_t R, int C, spt_stream_t stream) {
    SPT_REQUIRE(coeff && a && b && out, "scale_add_fwd: null pointer");
    int rc = check_rc("scale_add_fwd", R, C);
    if (rc != SPT_OK) return rc;
    const int kind = half_kind({a_dtype, b_dtype, o_dtype});
    SPT_REQUIRE(kind > 0, "scale_add_fwd: dtypes (a %d, b %d, out %d) not supported: each is fp32 or one 16-bit type "
                "(bf16 and fp16 do not mix)", a_dtype, b_dtype, o_dtype);
    const int key = (a_dtype != SPT_F32) * 4 + (b_dtype != SPT_F32) * 2 + (o_dtype != SPT_F32);
    if (kind == SPT_F16) scale_add_fwd_launch<__half>(key, coeff, a, b, out, R, C, as_stream(stream));
    else scale_add_fwd_launch<__nv_bfloat16>(key, coeff, a, b, out, R, C, as_stream(stream));
    return after_launch("scale_add_fwd_kernel");
}

template <typename H>
static void scale_add_bwd_launch(int key, const float *coeff, const void *a, const void *dout, void *da, float *dcoeff,
                                 int64_t R, int C, cudaStream_t st) {
    const unsigned grid = (unsigned)R;
#define SPT_SB(TA, TG) lfuse::scale_add_bwd_kernel<TA, TG><<<grid, lfuse::THREADS, 0, st>>>(coeff, (const TA *)a, (const TG *)dout, (TA *)da, dcoeff, C)
    switch (key) {
        case 0: SPT_SB(float, float); break;
        case 1: SPT_SB(float, H); break;
        case 2: SPT_SB(H, float); break;
        default: SPT_SB(H, H); break;
    }
#undef SPT_SB
}

// da has a's dtype; a and dout each fp32 or one 16-bit type
extern "C" int spt_scale_add_bwd(const float *coeff, const void *a, int a_dtype, const void *dout, int g_dtype, void *da,
                                 float *dcoeff, int64_t R, int C, spt_stream_t stream) {
    SPT_REQUIRE(coeff && a && dout && da && dcoeff, "scale_add_bwd: null pointer");
    int rc = check_rc("scale_add_bwd", R, C);
    if (rc != SPT_OK) return rc;
    const int kind = half_kind({a_dtype, g_dtype});
    SPT_REQUIRE(kind > 0, "scale_add_bwd: dtypes (a %d, grad %d) not supported: each is fp32 or one 16-bit type "
                "(bf16 and fp16 do not mix)", a_dtype, g_dtype);
    const int key = (a_dtype != SPT_F32) * 2 + (g_dtype != SPT_F32);
    if (kind == SPT_F16) scale_add_bwd_launch<__half>(key, coeff, a, dout, da, dcoeff, R, C, as_stream(stream));
    else scale_add_bwd_launch<__nv_bfloat16>(key, coeff, a, dout, da, dcoeff, R, C, as_stream(stream));
    return after_launch("scale_add_bwd_kernel");
}

static int check_half(const char *what, const char *name, int dtype) {
    if (dtype != SPT_BF16 && dtype != SPT_F16)
        return fail(SPT_ERR_INVALID_ARGUMENT, "%s: dtype %d unknown: %s is SPT_BF16 (1) or SPT_F16 (2)", what, dtype, name);
    return SPT_OK;
}

extern "C" int spt_lora_glu_fwd_ex(const float *coeff, const float *bg, const float *lg, const float *bs, const float *ls,
                                   void *h, int64_t R, int C, int h_dtype, spt_stream_t stream) {
    SPT_REQUIRE(coeff && bg && lg && bs && ls && h, "lora_glu_fwd: null pointer");
    int rc = check_rc("lora_glu_fwd", R, C);
    if (rc == SPT_OK) rc = check_half("lora_glu_fwd", "h", h_dtype);
    if (rc != SPT_OK) return rc;
    if (h_dtype == SPT_F16)
        lfuse::lora_glu_fwd_kernel<__half><<<(unsigned)R, lfuse::THREADS, 0, as_stream(stream)>>>(coeff, bg, lg, bs, ls,
                                                                                                 (__half *)h, C);
    else
        lfuse::lora_glu_fwd_kernel<__nv_bfloat16><<<(unsigned)R, lfuse::THREADS, 0, as_stream(stream)>>>(
            coeff, bg, lg, bs, ls, (__nv_bfloat16 *)h, C);
    return after_launch("lora_glu_fwd_kernel");
}

extern "C" int spt_lora_glu_fwd(const float *coeff, const float *bg, const float *lg, const float *bs, const float *ls,
                                void *h, int64_t R, int C, spt_stream_t stream) {
    return spt_lora_glu_fwd_ex(coeff, bg, lg, bs, ls, h, R, C, SPT_BF16, stream);
}

extern "C" int spt_lora_glu_bwd_ex(const float *coeff, const float *bg, const float *lg, const float *bs, const float *ls,
                                   const void *dh, float *d_bg, float *d_lg, float *d_bs, float *d_ls, float *dcoeff,
                                   int64_t R, int C, int dh_dtype, spt_stream_t stream) {
    SPT_REQUIRE(coeff && bg && lg && bs && ls && dh && d_bg && d_lg && d_bs && d_ls && dcoeff, "lora_glu_bwd: null pointer");
    int rc = check_rc("lora_glu_bwd", R, C);
    if (rc == SPT_OK) rc = check_half("lora_glu_bwd", "grad_h", dh_dtype);
    if (rc != SPT_OK) return rc;
    if (dh_dtype == SPT_F16)
        lfuse::lora_glu_bwd_kernel<__half><<<(unsigned)R, lfuse::THREADS, 0, as_stream(stream)>>>(
            coeff, bg, lg, bs, ls, (const __half *)dh, d_bg, d_lg, d_bs, d_ls, dcoeff, C);
    else
        lfuse::lora_glu_bwd_kernel<__nv_bfloat16><<<(unsigned)R, lfuse::THREADS, 0, as_stream(stream)>>>(
            coeff, bg, lg, bs, ls, (const __nv_bfloat16 *)dh, d_bg, d_lg, d_bs, d_ls, dcoeff, C);
    return after_launch("lora_glu_bwd_kernel");
}

extern "C" int spt_lora_glu_bwd(const float *coeff, const float *bg, const float *lg, const float *bs, const float *ls,
                                const void *dh, float *d_bg, float *d_lg, float *d_bs, float *d_ls, float *dcoeff,
                                int64_t R, int C, spt_stream_t stream) {
    return spt_lora_glu_bwd_ex(coeff, bg, lg, bs, ls, dh, d_bg, d_lg, d_bs, d_ls, dcoeff, R, C, SPT_BF16, stream);
}

static unsigned silu_grid(int64_t n8) {
    const int64_t want = (n8 + spt::lfuse::THREADS - 1) / spt::lfuse::THREADS;
    const int64_t cap = (int64_t)spt::num_sms() * 16;
    return (unsigned)(want < cap ? want : cap);
}

extern "C" int spt_silu_mul_fwd_ex(const void *gate, const void *side, void *h, int64_t n, int dtype, spt_stream_t stream) {
    SPT_REQUIRE(gate && side && h, "silu_mul_fwd: null pointer");
    SPT_REQUIRE(n >= 0 && n % 8 == 0, "silu_mul_fwd: element count must be a multiple of 8 (got %lld)", (long long)n);
    SPT_REQUIRE(((uintptr_t)gate | (uintptr_t)side | (uintptr_t)h) % 16 == 0, "silu_mul_fwd: operands must be 16-byte aligned");
    int rc = check_half("silu_mul_fwd", "every operand", dtype);
    if (rc != SPT_OK) return rc;
    if (n == 0) return SPT_OK;
    if (dtype == SPT_F16) {
        using hf = __half;
        lfuse::silu_mul_fwd_kernel<hf><<<silu_grid(n / 8), lfuse::THREADS, 0, as_stream(stream)>>>(
            (const hf *)gate, (const hf *)side, (hf *)h, n / 8);
    } else {
        using bf = __nv_bfloat16;
        lfuse::silu_mul_fwd_kernel<bf><<<silu_grid(n / 8), lfuse::THREADS, 0, as_stream(stream)>>>(
            (const bf *)gate, (const bf *)side, (bf *)h, n / 8);
    }
    return after_launch("silu_mul_fwd_kernel");
}

extern "C" int spt_silu_mul_fwd(const void *gate, const void *side, void *h, int64_t n, spt_stream_t stream) {
    return spt_silu_mul_fwd_ex(gate, side, h, n, SPT_BF16, stream);
}

extern "C" int spt_silu_mul_bwd_ex(const void *gate, const void *side, const void *grad_h, void *grad_gate, void *grad_side,
                                   int64_t n, int dtype, spt_stream_t stream) {
    SPT_REQUIRE(gate && side && grad_h && grad_gate && grad_side, "silu_mul_bwd: null pointer");
    SPT_REQUIRE(n >= 0 && n % 8 == 0, "silu_mul_bwd: element count must be a multiple of 8 (got %lld)", (long long)n);
    SPT_REQUIRE(((uintptr_t)gate | (uintptr_t)side | (uintptr_t)grad_h | (uintptr_t)grad_gate | (uintptr_t)grad_side) % 16 == 0,
                "silu_mul_bwd: operands must be 16-byte aligned");
    int rc = check_half("silu_mul_bwd", "every operand", dtype);
    if (rc != SPT_OK) return rc;
    if (n == 0) return SPT_OK;
    if (dtype == SPT_F16) {
        using hf = __half;
        lfuse::silu_mul_bwd_kernel<hf><<<silu_grid(n / 8), lfuse::THREADS, 0, as_stream(stream)>>>(
            (const hf *)gate, (const hf *)side, (const hf *)grad_h, (hf *)grad_gate, (hf *)grad_side, n / 8);
    } else {
        using bf = __nv_bfloat16;
        lfuse::silu_mul_bwd_kernel<bf><<<silu_grid(n / 8), lfuse::THREADS, 0, as_stream(stream)>>>(
            (const bf *)gate, (const bf *)side, (const bf *)grad_h, (bf *)grad_gate, (bf *)grad_side, n / 8);
    }
    return after_launch("silu_mul_bwd_kernel");
}

extern "C" int spt_silu_mul_bwd(const void *gate, const void *side, const void *grad_h, void *grad_gate, void *grad_side,
                                int64_t n, spt_stream_t stream) {
    return spt_silu_mul_bwd_ex(gate, side, grad_h, grad_gate, grad_side, n, SPT_BF16, stream);
}
