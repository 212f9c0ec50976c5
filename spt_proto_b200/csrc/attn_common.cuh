// Shared pieces of the fused sparse-attention kernels (attn_tc.cu: 128 x 64 tiles, two CTAs per SM;
// attn_tc128.cu: 128 x 128 tiles, one CTA per SM): tile geometry, TMA helpers, the packed element math,
// optional phase timers.
#pragma once
#include <cstdlib>
#include <cstring>
#include <type_traits>

#include "tc.cuh"

namespace spt {
namespace attn_tc {

using namespace tc;

constexpr int BM = 128;        // owner tile rows  (= TMEM lanes)
constexpr int BN = 64;         // other tile rows per iteration
constexpr int STAGES = 3;
constexpr int N_MATH = 256;      // warps 0-7
constexpr int THREADS = 320;
// Head dim D in {64, 80, 128}.  Operand tiles are stored as NSUB = ceil(D / 64) sub-tiles of [rows][64] bf16 or fp16 (one TMA
// box each, 128-byte swizzled): an owner tile is [NSUB][128 rows][64], an "other" tile [NSUB][64 rows][64].
// D = 80 is padded to DP = 128 in shared memory and TMEM only: the second box starts at column 64 and the TMA fills
// its 48 columns past the row end with zeros, so Q K^T is unchanged and O, dQ, dK, dV get zero columns 80 .. 127,
// which the epilogues never store.  The MMA shapes, TMEM columns and pipeline are those of D = 128.
// D = 64 needs 256 TMEM columns (two CTAs per SM), D = 80 and 128 take the whole TMEM (one CTA per SM).
template <int D>
struct Dim {
    static_assert(D == 64 || D == 80 || D == 128, "head dim must be 64, 80 or 128");
    static constexpr int NSUB = (D + 63) / 64;
    static constexpr int DP = NSUB * 64;                                       // padded width in shared memory / TMEM
    static constexpr int PREP_LANES = D / 8 <= 8 ? 8 : 16;                     // lanes per row of attn_bwd_prep_kernel
    static constexpr int OWN_SUB = BM * 64 * 2, T_SUB = BN * 64 * 2;          // 16 KB, 8 KB
    static constexpr int OWN_BYTES = NSUB * OWN_SUB, T_BYTES = NSUB * T_SUB;
    static constexpr int TMEM_COLS = D == 64 ? 256 : 512;
    static constexpr int CTAS = D == 64 ? 2 : 1;
    static constexpr int FWD_SMEM = OWN_BYTES + 2 * STAGES * T_BYTES + 1024 /*row sums*/ + 1024 /*align*/ + 256 /*barriers*/;
    static constexpr int BWD_SMEM = 2 * OWN_BYTES + 2 * STAGES * T_BYTES + STAGES * ((BN + 4) * 16 + BN * 4 + BN * 4) + 1024 + 256;
};
// descriptor offset (16-byte units) of K16 slice k of a K-major tile whose 64-wide sub-tiles are SUB bytes apart
template <int SUB>
__device__ constexpr uint64_t kslice(int k) { return (uint64_t)((k >> 2) * (SUB >> 4) + (k & 3) * 2); }
// TMA: 128-row owner tile / 64-row other tile of head (hn, hh) starting at sequence row `row0`
template <int D>
__device__ __forceinline__ void tma_owner(uint32_t dst, const CUtensorMap *map, uint32_t bar, int hh, int row0, int hn) {
#pragma unroll
    for (int dh = 0; dh < Dim<D>::NSUB; ++dh) {
        tma_load_4d(dst + dh * Dim<D>::OWN_SUB, map, bar, dh * 64, hh, row0, hn);
        tma_load_4d(dst + dh * Dim<D>::OWN_SUB + Dim<D>::T_SUB, map, bar, dh * 64, hh, row0 + BN, hn);
    }
}
template <int D>
__device__ __forceinline__ void tma_other(uint32_t dst, const CUtensorMap *map, uint32_t bar, int hh, int row0, int hn) {
#pragma unroll
    for (int dh = 0; dh < Dim<D>::NSUB; ++dh) tma_load_4d(dst + dh * Dim<D>::T_SUB, map, bar, dh * 64, hh, row0, hn);
}
constexpr float LOG2E = 1.4426950408889634f;

// Packed variable-length batches (the VARLEN instantiations): q, k, v are [1, T, H, D] and every CTA takes one item of
// the work list built by spt_varlen_worklist, {first token of its sequence, sequence length (a multiple of 32), 128-row
// tile index, word offset of the sequence's key bitmaps}.  Items [0, *count) are in descending tile order; CTAs past
// *count exit.  Mask rows are `mwords` 32-bit words wide; per-row data is head-major [H, T].
struct Varlen {
    const int4 *items;
    const int *count;
    int mwords;
};

__device__ __forceinline__ float ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t *>(&h);
}
// ---- element type ---------------------------------------------------------------------------------
// The operands are bf16 or fp16 (T = __nv_bfloat16 / __half): kind::f16 MMAs take either at the same rate.  fp16 has
// 3 more mantissa bits but a largest value of 65504, so the fp16 kernels scale every score row by a power of two
// 2^-o_r (DESIGN.md section 4.1): the exponent argument becomes  scale s log2(e) - o_r, which cancels exactly in
// y = sum e v / Z, in E / Z and in dO / Z.
template <typename T>
constexpr bool is_f16 = std::is_same<T, __half>::value;
template <typename T>
__device__ __forceinline__ constexpr uint32_t idesc_of(int M, int N, int a_mn_major, int b_mn_major) {
    return is_f16<T> ? idesc_fp16(M, N, a_mn_major, b_mn_major) : idesc_bf16(M, N, a_mn_major, b_mn_major);
}
template <typename T>
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
    if constexpr (is_f16<T>) {
        __half2 h = __floats2half2_rn(lo, hi);
        return *reinterpret_cast<uint32_t *>(&h);
    } else {
        return pack_bf16(lo, hi);
    }
}
// largest clamp the fp16 row scaling covers: the smallest element e^-c of a row scaled by 2^-o_min stays a normal fp16
constexpr float F16_MAX_CLAMP = 10.0f;
// Backward row scale of fp16: o_r = floor(log2 Z_r), so Z_r 2^-o_r is in [1, 2).  Returns -o_r (exact, as a float).
__device__ __forceinline__ float f16_bwd_nofs(float z) { return (float)(127 - (int)((__float_as_uint(z) >> 23) & 0xff)); }
// Z 2^-o in [1, 2): the mantissa of Z (Z >= 1e-9 is a normal float)
__device__ __forceinline__ float f16_bwd_zs(float z) { return __uint_as_float((__float_as_uint(z) & 0x007fffffu) | 0x3f800000u); }
// ---- element math --------------------------------------------------------------------------------
// Per score element the three kernels need  e = w * exp(clamp(scale s, -10, 10))  (and, in the backward,
// ds = e (dp - delta') [|scale s| <= 10]).  The first version spent ~11-15 instructions per element on it and was
// issue-bound; this one spends ~5-7:
//   * fp32 pairs are processed with the packed sm_100 instructions (mul.f32x2 / add.f32x2 / fma.rn.f32x2 = FMUL2 /
//     FADD2 / FFMA2: two elements per issue slot), on the register pairs tcgen05.ld delivers;
//   * the clamp is resolved per warp and 32-column chunk: one FMNMX3 per two elements tracks max |s|; only when some
//     lane of the warp holds a score beyond the clamp (a vote) does the chunk take the exact path with min/max and the
//     zero-gradient indicator.  Otherwise clamp(x) = x and the indicator is 1 — bit-identical results either way;
//   * the selection mask is applied to the PACKED bf16 pair with one LOP3: the mask bits of four columns are moved to
//     the sign bits of the four bytes of a register (one shift per four elements), and PRMT's sign-replicate mode
//     expands two of them into a 0xFFFF / 0x0000 pair mask (one PRMT per two elements).
__device__ __forceinline__ uint64_t pk2(float lo, float hi) {
    uint64_t d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "f"(lo), "f"(hi));
    return d;
}
__device__ __forceinline__ void up2(uint64_t v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("mul.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("add.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}
__device__ __forceinline__ float max3abs(float a, float b, float c) {   // max(a, |b|, |c|): one FMNMX3
    float d;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(fabsf(b)), "f"(fabsf(c)));
    return d;
}

struct MathK {      // arg = s * c (log2 units);  |scale s| <= clamp  <=>  |s| <= thr  <=>  |arg| <= L
    float c, thr, L;
};
__device__ __forceinline__ MathK make_math(float scale_log2, float clamp_log2) {
    return {scale_log2, clamp_log2 / scale_log2, clamp_log2};
}
// does any lane of the warp hold a raw score beyond the clamp among its N values?  (warp-uniform result)
template <int N>
__device__ __forceinline__ bool warp_needs_clamp(const uint32_t (&r)[N], float thr) {
    float mx = 0.0f;
#pragma unroll
    for (int i = 0; i < N; i += 2) mx = max3abs(mx, __uint_as_float(r[i]), __uint_as_float(r[i + 1]));
    return __any_sync(0xffffffffu, mx > thr);
}
// e of one pair of raw scores: exp2(clamp(s c)); CLAMP: exact path, also returns the per-element gradient indicators.
// OFS (fp16): exp2(clamp(s c) + nofs), nofs = -o of the pair's rows (one FFMA2 instead of the FMUL2 when unclamped).
template <bool CLAMP, bool OFS = false>
__device__ __forceinline__ void exp_pair(float s0, float s1, const MathK mk, float &e0, float &e1, bool &in0, bool &in1,
                                         uint64_t nofs = 0) {
    uint64_t a = (OFS && !CLAMP) ? fma2(pk2(s0, s1), pk2(mk.c, mk.c), nofs) : mul2(pk2(s0, s1), pk2(mk.c, mk.c));
    if constexpr (CLAMP) {
        float a0, a1;
        up2(a, a0, a1);
        in0 = fabsf(s0) <= mk.thr;
        in1 = fabsf(s1) <= mk.thr;
        a = pk2(fminf(fmaxf(a0, -mk.L), mk.L), fminf(fmaxf(a1, -mk.L), mk.L));
        if constexpr (OFS) a = add2(a, nofs);
    }
    float a0, a1;
    up2(a, a0, a1);
    e0 = ex2(a0);
    e1 = ex2(a1);
}

// The 32 score columns [32 half, 32 half + 32) of key tile j of one query row: gathers, from the row's four lane-major
// mask words of key group j >> 1, the byte (index 2 (j & 1) + half) that covers them.  Result X: byte t bit n <=> column
// 4 n + t of the chunk.
__device__ __forceinline__ uint32_t chunk_mask_bytes(const uint4 mw, int byte_idx) {
    const uint32_t sel = (uint32_t)(((4 + byte_idx) << 4) | byte_idx);
    return prmt(prmt(mw.x, mw.y, sel), prmt(mw.z, mw.w, sel), 0x5410u);
}
// pair masks of columns (4 n, 4 n + 1) and (4 n + 2, 4 n + 3) of a chunk
__device__ __forceinline__ void pair_masks(uint32_t X, int n, uint32_t &m01, uint32_t &m23) {
    const uint32_t Y = X << (7 - n);
    m01 = prmt(Y, 0u, 0x9988u);
    m23 = prmt(Y, 0u, 0xBBAAu);
}
__device__ __forceinline__ uint64_t unpack_bf16x2(uint32_t p) { return pk2(__uint_as_float(p << 16), __uint_as_float(p & 0xffff0000u)); }
template <typename T>
__device__ __forceinline__ uint64_t unpack2(uint32_t p) {
    if constexpr (is_f16<T>) {
        const float2 f = __half22float2(*reinterpret_cast<const __half2 *>(&p));
        return pk2(f.x, f.y);
    } else {
        return unpack_bf16x2(p);
    }
}

// Forward: 32 score columns of one row -> 16 masked packed bf16 pairs of e = w * exp(clamp(scale s)); the row sum
// accumulates the bf16-rounded values (exactly the weights the P V product uses).  FIRST: column 0 is key 0, which also
// carries the row's zero-padding multiplicity ex0 (mult0 = bit + ex0 when > 0).  fp16: e 2^-o, nofs = -o of the row.
template <bool FIRST, bool CLAMP, typename T = __nv_bfloat16>
__device__ __forceinline__ void fwd_chunk32(const uint32_t (&r)[32], uint32_t X, const MathK mk, float ex0, uint64_t &sum2,
                                            uint32_t (&pk)[16], float nofs = 0.0f) {
    constexpr bool OFS = is_f16<T>;
    const uint64_t no2 = pk2(nofs, nofs);
    float mult0 = 1.0f;
    if (FIRST) {
        mult0 = (float)(X & 1u) + ex0;
        if (mult0 > 0.0f) X |= 1u;
        else mult0 = 1.0f;
    }
#pragma unroll
    for (int n = 0; n < 8; ++n) {
        uint32_t m01, m23;
        pair_masks(X, n, m01, m23);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int i = 4 * n + 2 * h;
            float e0, e1;
            bool in0, in1;
            exp_pair<CLAMP, OFS>(__uint_as_float(r[i]), __uint_as_float(r[i + 1]), mk, e0, e1, in0, in1, no2);
            if (FIRST && i == 0) e0 *= mult0;
            const uint32_t p = pack2<T>(e0, e1) & (h ? m23 : m01);
            sum2 = add2(sum2, unpack2<T>(p));
            pk[i >> 1] = p;
        }
    }
}

// dQ kernel: 32 columns (keys) of one query row -> 16 masked packed pairs of ds = e (dp - delta') [unclamped]; ndelta = -delta'.
// fp16: e 2^-o, nofs = -o of the row.
template <bool FIRST, bool CLAMP, typename T = __nv_bfloat16>
__device__ __forceinline__ void bwdq_chunk32(const uint32_t (&r)[32], const uint32_t (&g)[32], uint32_t X, const MathK mk,
                                             float ndelta, float ex0, uint32_t (&pk)[16], float nofs = 0.0f) {
    constexpr bool OFS = is_f16<T>;
    const uint64_t no2 = pk2(nofs, nofs);
    float mult0 = 1.0f;
    if (FIRST) {
        mult0 = (float)(X & 1u) + ex0;
        if (mult0 > 0.0f) X |= 1u;
        else mult0 = 1.0f;
    }
    const uint64_t nd2 = pk2(ndelta, ndelta);
#pragma unroll
    for (int n = 0; n < 8; ++n) {
        uint32_t m01, m23;
        pair_masks(X, n, m01, m23);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int i = 4 * n + 2 * h;
            float e0, e1;
            bool in0 = true, in1 = true;
            exp_pair<CLAMP, OFS>(__uint_as_float(r[i]), __uint_as_float(r[i + 1]), mk, e0, e1, in0, in1, no2);
            if (FIRST && i == 0) e0 *= mult0;
            float d0, d1;
            up2(mul2(pk2(e0, e1), add2(pk2(__uint_as_float(g[i]), __uint_as_float(g[i + 1])), nd2)), d0, d1);
            if (CLAMP) {
                d0 = in0 ? d0 : 0.0f;
                d1 = in1 ? d1 : 0.0f;
            }
            pk[i >> 1] = pack2<T>(d0, d1) & (h ? m23 : m01);
        }
    }
}

// dK/dV kernel: 16 columns (query rows c0 .. c0+15) of one key.  mrow = this key's lane-major word of every row of the
// stage ([64] in shared memory), shl moves the key's bit to bit 31; s_ndelta = -delta' of the rows.
// KEY0: this thread is key 0 (adds the rows' zero-padding multiplicity s_ex0).
// r / g hold NR values of which [OFF, OFF + 16) are processed; c0 = tile row of r[OFF].
// fp16: s_nofs = -o of the rows (the row scale of each column).
template <bool KEY0, bool CLAMP, int OFF = 0, int NR = 16, typename EX0 = float, typename T = __nv_bfloat16>
__device__ __forceinline__ void bwdkv_chunk16(const uint32_t (&rr)[NR], const uint32_t (&gg)[NR], const uint32_t *mrow,
                                              const float *s_ndelta, const EX0 *s_ex0, int c0, int shl, const MathK mk,
                                              uint32_t (&pe)[8], uint32_t (&pd)[8], const float *s_nofs = nullptr) {
    constexpr bool OFS = is_f16<T>;
    uint32_t r[16], g[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        r[i] = rr[OFF + i];
        g[i] = gg[OFF + i];
    }
#pragma unroll
    for (int q4 = 0; q4 < 16; q4 += 4) {
        const uint4 mw = *reinterpret_cast<const uint4 *>(mrow + c0 + q4);
        const float4 nd = *reinterpret_cast<const float4 *>(s_ndelta + c0 + q4);
        const uint32_t mwv[4] = {mw.x << shl, mw.y << shl, mw.z << shl, mw.w << shl};
        const float ndv[4] = {nd.x, nd.y, nd.z, nd.w};
        float4 no = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if constexpr (OFS) no = *reinterpret_cast<const float4 *>(s_nofs + c0 + q4);
        const uint64_t nov[2] = {pk2(no.x, no.y), pk2(no.z, no.w)};
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int i = q4 + 2 * h;
            float e0, e1;
            bool in0 = true, in1 = true;
            exp_pair<CLAMP, OFS>(__uint_as_float(r[i]), __uint_as_float(r[i + 1]), mk, e0, e1, in0, in1, nov[h]);
            uint32_t ma = mwv[2 * h], mb = mwv[2 * h + 1];
            if (KEY0) {     // key 0: weight = bit + zero-padding multiplicity of the row
                const float w0 = (float)(ma >> 31) + (float)s_ex0[c0 + i], w1 = (float)(mb >> 31) + (float)s_ex0[c0 + i + 1];
                e0 *= w0;
                e1 *= w1;
                ma = w0 > 0.0f ? 0x80000000u : 0u;
                mb = w1 > 0.0f ? 0x80000000u : 0u;
            }
            const uint32_t m = prmt(ma, mb, 0xFFBBu);      // sign of ma -> low half, sign of mb -> high half
            float d0, d1;
            up2(mul2(pk2(e0, e1), add2(pk2(__uint_as_float(g[i]), __uint_as_float(g[i + 1])), pk2(ndv[2 * h], ndv[2 * h + 1]))),
                d0, d1);
            if (CLAMP) {
                d0 = in0 ? d0 : 0.0f;
                d1 = in1 ? d1 : 0.0f;
            }
            pe[i >> 1] = pack2<T>(e0, e1) & m;
            pd[i >> 1] = pack2<T>(d0, d1) & m;
        }
    }
}

// ---- optional in-kernel phase timers (build with -DSPT_ATTN_PROF; read with spt_debug_attn_prof) ----------------------
// One math thread (warp 0, lane 0) and the MMA-issuer lane of every CTA accumulate clock64() deltas per phase and add them
// to g_prof[kernel][slot] at exit.  Slots 0-7: math thread (0 wait scores, 1 tcgen05.ld, 2 element math, 3 tcgen05.st +
// arrive, 4 iterations, 5 whole loop); 8-15: issuer (8 wait operands, 9 wait math, 10 issue, 11 whole loop, 12 iterations).
#ifdef SPT_ATTN_PROF
static __device__ unsigned long long g_prof[3][16];   // one copy per translation unit
struct Prof {
    long long t[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    long long last;
    __device__ __forceinline__ void start() { last = clock64(); }
    __device__ __forceinline__ void lap(int slot) {
        const long long now = clock64();
        t[slot] += now - last;
        last = now;
    }
    __device__ __forceinline__ void flush(int kernel, int base, bool on) {
        if (on)
            for (int i = 0; i < 8; ++i) atomicAdd(&g_prof[kernel][base + i], (unsigned long long)t[i]);
    }
};
#define PROF(...) __VA_ARGS__
#else
#define PROF(...)
#endif

struct Smem {
    uint32_t base;            // 1024-aligned shared address
    unsigned char *ptr;       // generic pointer to the same byte
};
__device__ __forceinline__ Smem align_smem(unsigned char *raw) {
    const uint32_t a = smem_u32(raw);
    const uint32_t base = (a + 1023) & ~1023u;
    return {base, raw + (base - a)};
}
__device__ __forceinline__ void math_warps_sync() { asm volatile("bar.sync 1, %0;" ::"n"(N_MATH) : "memory"); }

// store 32 fp32 accumulator values (scaled) as 32 bf16 / fp16 = 64 contiguous bytes
template <typename T>
__device__ __forceinline__ void store_row32(T *dst, const uint32_t (&r)[32], float s) {
#pragma unroll
    for (int i = 0; i < 32; i += 8) {
        float t[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) t[u] = __uint_as_float(r[i + u]) * s;
        Vec16<T>::store(dst + i, t);
    }
}
// the same for the first W (16 or 32) of the 32 values
template <int W, typename T>
__device__ __forceinline__ void store_row_n(T *dst, const uint32_t (&r)[32], float s) {
    static_assert(W % 8 == 0 && W <= 32, "W must be a multiple of 8, at most 32");
#pragma unroll
    for (int i = 0; i < W; i += 8) {
        float t[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) t[u] = __uint_as_float(r[i + u]) * s;
        Vec16<T>::store(dst + i, t);
    }
}
// one output element (the y^T epilogue)
__device__ __forceinline__ __nv_bfloat16 out_elem(float v, __nv_bfloat16 *) { return __float2bfloat16(v); }
__device__ __forceinline__ __half out_elem(float v, __half *) { return __float2half_rn(v); }
template <int W>
using Width = std::integral_constant<int, W>;
// The epilogues read a row's D output columns from TMEM in 32-column chunks shared by the two warpgroups (`half`):
// f(col, Width<W>) stores columns [col, col + W).  D = 64, 128: warpgroup h takes [h D/2, (h + 1) D/2).  D = 80:
// warpgroup 0 takes [0, 32) and [64, 80), warpgroup 1 [32, 64); the padding columns 80 .. 127 are never stored (in the
// [N, S, H, 80] layout they would overwrite the next head's row).
template <int D, typename F>
__device__ __forceinline__ void out_chunks(int half, F &&f) {
    if constexpr (D % 64 == 0) {
#pragma unroll
        for (int c = 0; c < D / 64; ++c) f(half * (D / 2) + c * 32, Width<32>{});
    } else {
        static_assert(D == 80, "odd head dims other than 80 need their own column split");
        if (half == 0) {
            f(0, Width<32>{});
            f(64, Width<16>{});
        } else {
            f(32, Width<32>{});
        }
    }
}

}  // namespace attn_tc

// 128 x 128-tile kernels (attn_tc128.cu), head dim 64
namespace attn_tc128 {
// T = __nv_bfloat16 or __half; zsum is read by the fp16 kernels only (row scales)
template <typename T>
int launch_bwd_kv128(const CUtensorMap &mq, const CUtensorMap &mk, const CUtensorMap &mv, const CUtensorMap &md,
                     const uint32_t *mask, const int32_t *extra0, const float *ndelta, const float *zsum, T *gk, T *gv,
                     int B, int S, int H, float scale, float clamp, cudaStream_t st);
template <typename T>
int launch_bwd_q128(const CUtensorMap &mq, const CUtensorMap &mk, const CUtensorMap &mv, const CUtensorMap &md,
                    const uint32_t *mask, const int32_t *extra0, const float *ndelta, const float *zsum, T *gq, int B,
                    int S, int H, float scale, float clamp, cudaStream_t st);
int read_prof(unsigned long long *out48, int reset);
}  // namespace attn_tc128
}  // namespace spt
