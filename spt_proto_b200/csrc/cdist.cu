// (1) cdist: L1 distance from PQ sub-vectors to codewords + argmin -> PQ codes.
//
// Replaces cdist_forward_cuda / cdist_backward_cuda (reference extension/cdist.cu:185-333) and
// fuses PQBase.forward(mode='encode') (naive_gpt/layers/basic/quantizer.py:26-77).
//
// Numerics contract (bit-exact codes): distance = sum_i |q_i - t_i| accumulated over i ascending
// in fp32 (no FMA is possible: there is no multiply), running strict-'<' minimum starting at 1e13
// => lowest codeword index wins ties (cdist.cu:29,46-54).  bf16 / fp16 inputs are widened to fp32 first
// (exact).  fp16 is taken by the PQ encode / train entry points only; cdist_fwd / _bwd keep fp32 / bf16.
//
// This is L1, not a GEMM: it stays on the CUDA cores (SURVEY.md section 7, hard part 1).  Per
// (sub-vector, codeword, element) it costs one FADD + one FADD-with-|.| source modifier.
// Bound: issue-bound SIMT (6*n*d*c flop vs 2*n*d*e bytes) — see DESIGN.md section 5.
#include <type_traits>

#include "common.cuh"

namespace spt {

constexpr int CDIST_THREADS = 256;

// ---- forward, reference layout: query [m, n, dc] ---------------------------------------------
// One thread per (subspace, query).  The sub-space's codebook slice lives in shared memory and is
// read as a warp-wide broadcast.  DC > 0: compile-time sub-vector length (query in registers);
// DC == 0: generic path, query element re-read through L1.
template <typename T, int DC>
__global__ void __launch_bounds__(CDIST_THREADS)
cdist_fwd_kernel(const T *__restrict__ query, const float *__restrict__ table, float *__restrict__ distance,
                 int32_t *__restrict__ indices, int64_t n, int c, int dc_rt) {
    extern __shared__ __align__(16) float s_table[];  // [c][dc]
    const int dc = DC > 0 ? DC : dc_rt;
    const int s = blockIdx.y;
    for (int i = threadIdx.x; i < c * dc; i += blockDim.x) s_table[i] = table[(size_t)s * c * dc + i];
    __syncthreads();
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const T *qp = query + ((size_t)s * n + q) * dc;
    float qv[DC > 0 ? DC : 1];
    if constexpr (DC > 0 && DC % Vec16<T>::N == 0) {
        // 16-byte loads (a sub-vector is DC * sizeof(T) contiguous bytes; the vector path needs 16-byte alignment)
        if ((reinterpret_cast<uintptr_t>(query) & 15) == 0) {
#pragma unroll
            for (int i = 0; i < DC; i += Vec16<T>::N) {
                float tmp[Vec16<T>::N];
                Vec16<T>::load(qp + i, tmp);
#pragma unroll
                for (int j = 0; j < Vec16<T>::N; ++j) qv[i + j] = tmp[j];
            }
        } else {
#pragma unroll
            for (int i = 0; i < DC; ++i) qv[i] = to_f32(qp[i]);
        }
    } else if (DC > 0) {
#pragma unroll
        for (int i = 0; i < DC; ++i) qv[i] = to_f32(qp[i]);
    }
    float *dp = distance ? distance + ((size_t)s * n + q) * c : nullptr;
    const bool vec_store = dp && (c % 4 == 0);
    int min_index = 0;
    float min_distance = 1e13f;
    float4 pack;
    if constexpr (DC > 0 && DC % 4 == 0) {
        // c == 16 with a distance output (the reference layout's common case): the 16 distances stay in registers and
        // the warp's 32 x 64-byte block leaves through its shared-memory slice as full 512-byte store instructions
        // (a thread's own 64 bytes written 16 at a time touch every 32-byte sector twice)
        if (vec_store && c == 16 && (blockDim.x & 31) == 0 && ((blockIdx.x + 1) * (int64_t)blockDim.x <= n)) {
            float dist[16];
#pragma unroll
            for (int w = 0; w < 16; ++w) {
                const float *tp = s_table + w * DC;
                float reduced = 0.0f;
#pragma unroll
                for (int i = 0; i < DC; i += 4) {
                    const float4 t4 = *reinterpret_cast<const float4 *>(tp + i);
                    reduced += fabsf(qv[i] - t4.x);
                    reduced += fabsf(qv[i + 1] - t4.y);
                    reduced += fabsf(qv[i + 2] - t4.z);
                    reduced += fabsf(qv[i + 3] - t4.w);
                }
                dist[w] = reduced;
                if (reduced < min_distance) {
                    min_distance = reduced;
                    min_index = w;
                }
            }
            indices[(size_t)s * n + q] = min_index;
            // staging area behind the table: [warps][32 rows][16 + 4 pad] floats (row stride 80 B: conflict-free 16-byte accesses)
            float *stage = s_table + ((c * DC + 3) & ~3) + (threadIdx.x >> 5) * (32 * 20);
            const int lane = threadIdx.x & 31;
#pragma unroll
            for (int u = 0; u < 4; ++u)
                *reinterpret_cast<float4 *>(stage + lane * 20 + 4 * u) = make_float4(dist[4 * u], dist[4 * u + 1], dist[4 * u + 2], dist[4 * u + 3]);
            __syncwarp();
            float *wp = distance + ((size_t)s * n + (q - lane)) * 16;          // the warp's 2 KB block
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int id = lane + 32 * u;                                    // 16-byte chunk of the block
                st_stream(reinterpret_cast<float4 *>(wp) + id, *reinterpret_cast<const float4 *>(stage + (id >> 2) * 20 + 4 * (id & 3)));
            }
            return;
        }
    }
    for (int w = 0; w < c; ++w) {
        const float *tp = s_table + w * dc;
        float reduced = 0.0f;
        if constexpr (DC > 0 && DC % 4 == 0) {          // codeword read as 16-byte broadcasts (same summation order)
#pragma unroll
            for (int i = 0; i < DC; i += 4) {
                const float4 t4 = *reinterpret_cast<const float4 *>(tp + i);
                reduced += fabsf(qv[i] - t4.x);
                reduced += fabsf(qv[i + 1] - t4.y);
                reduced += fabsf(qv[i + 2] - t4.z);
                reduced += fabsf(qv[i + 3] - t4.w);
            }
        } else if (DC > 0) {
#pragma unroll
            for (int i = 0; i < DC; ++i) reduced += fabsf(qv[i] - tp[i]);
        } else {
            for (int i = 0; i < dc; ++i) reduced += fabsf(to_f32(qp[i]) - tp[i]);
        }
        if (reduced < min_distance) {
            min_distance = reduced;
            min_index = w;
        }
        if (vec_store) {
            (&pack.x)[w & 3] = reduced;
            if ((w & 3) == 3) st_stream(reinterpret_cast<float4 *>(dp + w - 3), pack);
        } else if (dp) {
            dp[w] = reduced;
        }
    }
    indices[(size_t)s * n + q] = min_index;
}

// ---- fused encode, layer layout: z [rows, m*dc] -> codes [rows, m] ----------------------------
// Thread g handles (row = g / m, subspace = g % m): consecutive threads read consecutive dc-element
// chunks (fully coalesced 16/32-byte loads) and write consecutive int32 codes.  L1 distance is not a
// GEMM; the kernel is bound by the fp32 add pipe (2 adds per (element, codeword)), so the adds are
// issued as packed FADD2 (sm_100 add.f32x2) over PAIRS OF CODEWORDS: the two halves carry codewords
// w and w+1, the element loop stays sequential in i, hence every distance is still the reference's
// i-ascending fp32 sum and, with the strict `<`, the codes are bit-identical to the reference kernel
// (extension/cdist.cu:42-54).  |x| is a LOP3 on the otherwise idle ALU pipe.  The codebook is staged in
// shared memory as [codeword pair][element][subspace] float2 (lanes of a warp differ in subspace:
// distinct banks, equal-subspace lanes broadcast).  blockIdx.y selects one of up to two tensors (q and
// k of a layer share the codebook and are encoded by one launch).
__device__ __forceinline__ uint64_t sub_f32x2(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("sub.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ uint64_t mul_f32x2(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("mul.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ uint64_t fma_f32x2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ uint64_t pk_f32x2(float lo, float hi) {
    uint64_t d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "f"(lo), "f"(hi));
    return d;
}
__device__ __forceinline__ float lo_f32x2(uint64_t v) {
    float lo;
    asm("{\n\t.reg .b32 t;\n\tmov.b64 {%0, t}, %1;\n\t}" : "=f"(lo) : "l"(v));
    return lo;
}
__device__ __forceinline__ float hi_f32x2(uint64_t v) {
    float hi;
    asm("{\n\t.reg .b32 t;\n\tmov.b64 {t, %0}, %1;\n\t}" : "=f"(hi) : "l"(v));
    return hi;
}
__device__ __forceinline__ uint64_t shfl_xor_f32x2(uint64_t v, int o) {
    return pk_f32x2(__shfl_xor_sync(0xffffffffu, lo_f32x2(v), o), __shfl_xor_sync(0xffffffffu, hi_f32x2(v), o));
}
__device__ __forceinline__ uint64_t add_f32x2(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("add.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}

#ifndef SPT_PQ_ENC_UNROLL
#define SPT_PQ_ENC_UNROLL 2
#endif
constexpr int PQ_ENC_UNROLL = SPT_PQ_ENC_UNROLL;   // codeword pairs in flight per thread (independent accumulation chains)

template <typename T, int DC>
__global__ void __launch_bounds__(CDIST_THREADS)
pq_encode_kernel(const T *__restrict__ z0, const T *__restrict__ z1, const float *__restrict__ table,
                 int32_t *__restrict__ codes0, int32_t *__restrict__ codes1, int64_t total /* rows*m */, int m, int c) {
    extern __shared__ __align__(16) float s_table[];  // [(c+1)/2][DC][m][2]; an odd last codeword is paired with +inf
    const int cp = (c + 1) / 2;
    for (int i = threadIdx.x; i < cp * DC * m * 2; i += blockDim.x) {
        const int h = i & 1, s = (i >> 1) % m, e = ((i >> 1) / m) % DC, wp = (i >> 1) / (m * DC);
        const int w = 2 * wp + h;
        s_table[i] = w < c ? table[((size_t)s * c + w) * DC + e] : __int_as_float(0x7f800000);
    }
    __syncthreads();
    const T *z = blockIdx.y ? z1 : z0;
    int32_t *codes = blockIdx.y ? codes1 : codes0;
    // grid-stride over (row, subspace) items: the codebook is staged once per resident block.  A thread takes TWO items
    // of the same subspace per trip (g and g + stride; the stride is a multiple of m), so that every codebook word it
    // reads from shared memory serves both: per (dimension, codeword pair) 1 LDS.64 + 2 x (packed subtract + two FADD
    // with the |x| operand modifier) = 7 issue slots for 4 distances terms (one item per trip with a 64-bit AND for the
    // absolute values: 5 slots for 2).  Every distance is still the reference's i-ascending fp32 sum => codes bit-exact.
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const bool pair_ok = stride % m == 0;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += pair_ok ? 2 * stride : stride) {
        const int s = (int)(g % m);
        const bool has_b = pair_ok && g + stride < total;
        uint64_t qa[DC], qb[DC];   // (q_i, q_i)
#pragma unroll
        for (int it = 0; it < 2; ++it) {
            float qv[DC];
            const T *zp = z + (size_t)(it && has_b ? g + stride : g) * DC;
            if constexpr (DC % Vec16<T>::N == 0) {
#pragma unroll
                for (int i = 0; i < DC; i += Vec16<T>::N) {
                    float tmp[Vec16<T>::N];
                    Vec16<T>::load(zp + i, tmp);
#pragma unroll
                    for (int j = 0; j < Vec16<T>::N; ++j) qv[i + j] = tmp[j];
                }
            } else {
#pragma unroll
                for (int i = 0; i < DC; ++i) qv[i] = to_f32(zp[i]);
            }
#pragma unroll
            for (int i = 0; i < DC; ++i) {
                const uint64_t v = ((uint64_t)__float_as_uint(qv[i]) << 32) | __float_as_uint(qv[i]);
                if (it) qb[i] = v;
                else qa[i] = v;
            }
        }
        int ia = 0, ib = 0;
        float ma = 1e13f, mb = 1e13f;
        const uint64_t *tp = reinterpret_cast<const uint64_t *>(s_table) + s;
#pragma unroll PQ_ENC_UNROLL
        for (int wp = 0; wp < cp; ++wp, tp += (size_t)DC * m) {
            float a0 = 0.0f, a1 = 0.0f, b0 = 0.0f, b1 = 0.0f;
#pragma unroll
            for (int i = 0; i < DC; ++i) {
                const uint64_t t2 = tp[(size_t)i * m];
                const uint64_t da = sub_f32x2(qa[i], t2), db = sub_f32x2(qb[i], t2);
                a0 += fabsf(__uint_as_float((uint32_t)da));
                a1 += fabsf(__uint_as_float((uint32_t)(da >> 32)));
                b0 += fabsf(__uint_as_float((uint32_t)db));
                b1 += fabsf(__uint_as_float((uint32_t)(db >> 32)));
            }
            if (a0 < ma) { ma = a0; ia = 2 * wp; }
            if (a1 < ma) { ma = a1; ia = 2 * wp + 1; }   // an odd c pairs its last codeword with +inf: never selected
            if (b0 < mb) { mb = b0; ib = 2 * wp; }
            if (b1 < mb) { mb = b1; ib = 2 * wp + 1; }
        }
        codes[g] = ia;
        if (has_b) codes[g + stride] = ib;
    }
}

// ---- backward wrt query: gq[s,n,i] = sum_c sgn(q_i - t_ci) * g[s,n,c]  (cdist.cu:72-131) --------
template <int DC>
__global__ void __launch_bounds__(CDIST_THREADS)
cdist_bwd_query_kernel(const float *__restrict__ query, const float *__restrict__ table,
                       const float *__restrict__ grad, float *__restrict__ grad_query, int64_t n, int c,
                       int dc_rt) {
    extern __shared__ float s_table[];
    const int dc = DC > 0 ? DC : dc_rt;
    const int s = blockIdx.y;
    for (int i = threadIdx.x; i < c * dc; i += blockDim.x) s_table[i] = table[(size_t)s * c * dc + i];
    __syncthreads();
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const float *qp = query + ((size_t)s * n + q) * dc;
    const float *gp = grad + ((size_t)s * n + q) * c;
    float *op = grad_query + ((size_t)s * n + q) * dc;
    if (DC > 0) {
        float qv[DC > 0 ? DC : 1], acc[DC > 0 ? DC : 1];
#pragma unroll
        for (int i = 0; i < DC; ++i) { qv[i] = qp[i]; acc[i] = 0.0f; }
        for (int w = 0; w < c; ++w) {
            const float g = gp[w];
            const float *tp = s_table + w * DC;
#pragma unroll
            for (int i = 0; i < DC; ++i) acc[i] += (qv[i] - tp[i]) > 0.0f ? g : -g;
        }
#pragma unroll
        for (int i = 0; i < DC; ++i) op[i] = acc[i];
    } else {
        for (int i = 0; i < dc; ++i) {
            const float qi = qp[i];
            float acc = 0.0f;
            for (int w = 0; w < c; ++w) acc += (qi - s_table[w * dc + i]) > 0.0f ? gp[w] : -gp[w];
            op[i] = acc;
        }
    }
}

// ---- backward wrt table: gt[s,c,i] = -sum_n sgn(q_ni - t_ci) * g[s,n,c]  (cdist.cu:134-182) -----
// Stage 1: each block reduces a chunk of CHUNK queries for one subspace into a partial [c*dc]
// (the reference runs 16 blocks serially over all n, cdist.cu:320-329).  Stage 2 adds the partials
// in chunk order => deterministic.
constexpr int BWD_T_CHUNK = 512;
constexpr int BWD_T_TILE = 32;

__global__ void __launch_bounds__(CDIST_THREADS)
cdist_bwd_table_stage1(const float *__restrict__ query, const float *__restrict__ table,
                       const float *__restrict__ grad, float *__restrict__ partial, int64_t n, int c, int dc,
                       int n_chunks) {
    extern __shared__ float smem[];
    float *s_q = smem;                      // [TILE][dc]
    float *s_g = smem + BWD_T_TILE * dc;    // [TILE][c]
    const int s = blockIdx.y, chunk = blockIdx.x;
    const int64_t n0 = (int64_t)chunk * BWD_T_CHUNK;
    const int64_t n1 = min(n, n0 + BWD_T_CHUNK);
    const int n_out = c * dc;
    // each thread owns outputs o = tid, tid + blockDim, ... ; keep up to 4 in registers
    constexpr int MAX_OWN = 4;
    float acc[MAX_OWN], tv[MAX_OWN];
    int own = 0;
    for (int o = threadIdx.x; o < n_out && own < MAX_OWN; o += blockDim.x, ++own) {
        acc[own] = 0.0f;
        tv[own] = table[(size_t)s * n_out + o];
    }
    for (int64_t t0 = n0; t0 < n1; t0 += BWD_T_TILE) {
        const int rows = (int)min((int64_t)BWD_T_TILE, n1 - t0);
        for (int i = threadIdx.x; i < rows * dc; i += blockDim.x) s_q[i] = query[((size_t)s * n + t0) * dc + i];
        for (int i = threadIdx.x; i < rows * c; i += blockDim.x) s_g[i] = grad[((size_t)s * n + t0) * c + i];
        __syncthreads();
        int k = 0;
        for (int o = threadIdx.x; o < n_out && k < MAX_OWN; o += blockDim.x, ++k) {
            const int w = o / dc, i = o % dc;
            float a = acc[k];
            const float t = tv[k];
            for (int r = 0; r < rows; ++r) {
                const float g = s_g[r * c + w];
                a -= (s_q[r * dc + i] - t) > 0.0f ? g : -g;
            }
            acc[k] = a;
        }
        __syncthreads();
    }
    int k = 0;
    for (int o = threadIdx.x; o < n_out && k < MAX_OWN; o += blockDim.x, ++k)
        partial[((size_t)s * n_chunks + chunk) * n_out + o] = acc[k];
}

__global__ void cdist_bwd_table_stage2(const float *__restrict__ partial, float *__restrict__ grad_table,
                                       int n_out, int n_chunks) {
    const int s = blockIdx.y;
    const int o = blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= n_out) return;
    float a = 0.0f;
    for (int ch = 0; ch < n_chunks; ++ch) a += partial[((size_t)s * n_chunks + ch) * n_out + o];
    grad_table[(size_t)s * n_out + o] = a;
}

template <typename T>
static int launch_cdist_fwd(const T *query, const float *table, float *distance, int32_t *indices, int m,
                            int64_t n, int c, int dc, cudaStream_t st) {
    dim3 grid((unsigned)((n + CDIST_THREADS - 1) / CDIST_THREADS), m);
    // codebook slice + (c == 16 with distances) the per-warp store staging of cdist_fwd_kernel
    size_t smem = (((size_t)c * dc + 3) & ~(size_t)3) * sizeof(float) + (size_t)(CDIST_THREADS / 32) * 32 * 20 * sizeof(float);
#define SPT_CDIST_CASE(D)                                                                               \
    case D:                                                                                             \
        if (smem > 48 * 1024)                                                                           \
            cudaFuncSetAttribute(cdist_fwd_kernel<T, D>, cudaFuncAttributeMaxDynamicSharedMemorySize,   \
                                 (int)smem);                                                            \
        cdist_fwd_kernel<T, D><<<grid, CDIST_THREADS, smem, st>>>(query, table, distance, indices, n, c, dc); \
        break;
    switch (dc) {
        SPT_CDIST_CASE(4)
        SPT_CDIST_CASE(8)
        SPT_CDIST_CASE(16)
        SPT_CDIST_CASE(32)
        default:
            if (smem > 48 * 1024)
                cudaFuncSetAttribute(cdist_fwd_kernel<T, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)smem);
            cdist_fwd_kernel<T, 0><<<grid, CDIST_THREADS, smem, st>>>(query, table, distance, indices, n, c, dc);
    }
#undef SPT_CDIST_CASE
    return after_launch("cdist_fwd_kernel");
}

template <typename T>
static int launch_pq_encode(const T *z0, const T *z1, const float *table, int32_t *codes0, int32_t *codes1,
                            int64_t rows, int m, int c, int dc, cudaStream_t st) {
    const int64_t total = rows * m;
    const int64_t want = (total + CDIST_THREADS - 1) / CDIST_THREADS;
    const int64_t cap = (int64_t)num_sms() * 8 / (z1 ? 2 : 1);      // resident blocks: one codebook staging each
    dim3 grid((unsigned)(want < cap ? want : cap), z1 ? 2 : 1);
    size_t smem = (size_t)m * ((c + 1) / 2) * 2 * dc * sizeof(float);
#define SPT_ENC_CASE(D)                                                                                 \
    case D:                                                                                             \
        if (smem > 48 * 1024)                                                                           \
            cudaFuncSetAttribute(pq_encode_kernel<T, D>, cudaFuncAttributeMaxDynamicSharedMemorySize,   \
                                 (int)smem);                                                            \
        pq_encode_kernel<T, D><<<grid, CDIST_THREADS, smem, st>>>(z0, z1, table, codes0, codes1, total, m, c); \
        break;
    switch (dc) {
        SPT_ENC_CASE(4)
        SPT_ENC_CASE(8)
        SPT_ENC_CASE(16)
        SPT_ENC_CASE(32)
        default:
            return fail(SPT_ERR_UNSUPPORTED, "pq_encode: d_codeword %d not in {4,8,16,32}", dc);
    }
#undef SPT_ENC_CASE
    return after_launch("pq_encode_kernel");
}

}  // namespace spt

using namespace spt;

extern "C" int spt_cdist_fwd(const void *query, const float *table, float *distance, int32_t *indices, int m,
                             int64_t n, int c, int dc, int dtype, spt_stream_t stream) {
    SPT_REQUIRE(query && table && indices, "cdist_fwd: null pointer");
    SPT_REQUIRE(m >= 1 && n >= 0 && c >= 1 && dc >= 1 && dc <= 64, "cdist_fwd: bad sizes m=%d n=%lld c=%d dc=%d",
                m, (long long)n, c, dc);
    SPT_REQUIRE(m <= 65535, "cdist_fwd: n_subspaces %d exceeds grid limit", m);
    SPT_REQUIRE((size_t)c * dc * 4 <= 200 * 1024, "cdist_fwd: codebook slice %d x %d does not fit shared memory", c, dc);
    if (n == 0) return SPT_OK;
    if (dtype == SPT_F32)
        return launch_cdist_fwd((const float *)query, table, distance, indices, m, n, c, dc, as_stream(stream));
    if (dtype == SPT_BF16)
        return launch_cdist_fwd((const __nv_bfloat16 *)query, table, distance, indices, m, n, c, dc, as_stream(stream));
    return fail(SPT_ERR_INVALID_ARGUMENT, "cdist_fwd: unknown dtype %d", dtype);
}

static int pq_encode_impl(const void *z0, const void *z1, const float *table, int32_t *codes0, int32_t *codes1,
                          int64_t rows, int m, int c, int dc, int dtype, spt_stream_t stream) {
    SPT_REQUIRE(z0 && table && codes0 && (!z1 == !codes1), "pq_encode: null pointer");
    SPT_REQUIRE(m >= 1 && rows >= 0 && c >= 1 && dc >= 1, "pq_encode: bad sizes");
    SPT_REQUIRE((size_t)m * c * dc * 4 <= 200 * 1024, "pq_encode: codebook %d x %d x %d does not fit shared memory", m, c, dc);
    if (rows == 0) return SPT_OK;
    if (dtype == SPT_F32)
        return launch_pq_encode((const float *)z0, (const float *)z1, table, codes0, codes1, rows, m, c, dc, as_stream(stream));
    if (dtype == SPT_BF16)
        return launch_pq_encode((const __nv_bfloat16 *)z0, (const __nv_bfloat16 *)z1, table, codes0, codes1, rows, m, c,
                                dc, as_stream(stream));
    if (dtype == SPT_F16)      // fp16 -> fp32 is exact: the same fp32 sums, the same codes as z.float()
        return launch_pq_encode((const __half *)z0, (const __half *)z1, table, codes0, codes1, rows, m, c, dc,
                                as_stream(stream));
    return fail(SPT_ERR_INVALID_ARGUMENT, "pq_encode: unknown dtype %d", dtype);
}

extern "C" int spt_pq_encode(const void *z, const float *table, int32_t *codes, int64_t rows, int m, int c, int dc,
                             int dtype, spt_stream_t stream) {
    return pq_encode_impl(z, nullptr, table, codes, nullptr, rows, m, c, dc, dtype, stream);
}

extern "C" int spt_pq_encode_pair(const void *z0, const void *z1, const float *table, int32_t *codes0, int32_t *codes1,
                                  int64_t rows, int m, int c, int dc, int dtype, spt_stream_t stream) {
    SPT_REQUIRE(z1 && codes1, "pq_encode_pair: null pointer");
    return pq_encode_impl(z0, z1, table, codes0, codes1, rows, m, c, dc, dtype, stream);
}

extern "C" size_t spt_cdist_bwd_workspace_bytes(int m, int64_t n, int c, int dc) {
    const int64_t n_chunks = (n + BWD_T_CHUNK - 1) / BWD_T_CHUNK;
    return (size_t)m * (size_t)n_chunks * c * dc * sizeof(float);
}

extern "C" int spt_cdist_bwd(const float *query, const float *table, const float *grad_distance, float *grad_query,
                             float *grad_table, void *workspace, int m, int64_t n, int c, int dc,
                             spt_stream_t stream) {
    SPT_REQUIRE(query && table && grad_distance && grad_query && grad_table, "cdist_bwd: null pointer");
    SPT_REQUIRE(m >= 1 && m <= 65535 && n >= 1 && c >= 1 && dc >= 1 && dc <= 64, "cdist_bwd: bad sizes");
    SPT_REQUIRE(c * dc <= 4 * CDIST_THREADS, "cdist_bwd: c*dc = %d exceeds %d", c * dc, 4 * CDIST_THREADS);
    SPT_REQUIRE(workspace, "cdist_bwd: workspace required");
    cudaStream_t st = as_stream(stream);
    {
        dim3 grid((unsigned)((n + CDIST_THREADS - 1) / CDIST_THREADS), m);
        size_t smem = (size_t)c * dc * sizeof(float);
        switch (dc) {
            case 4: cdist_bwd_query_kernel<4><<<grid, CDIST_THREADS, smem, st>>>(query, table, grad_distance, grad_query, n, c, dc); break;
            case 8: cdist_bwd_query_kernel<8><<<grid, CDIST_THREADS, smem, st>>>(query, table, grad_distance, grad_query, n, c, dc); break;
            case 16: cdist_bwd_query_kernel<16><<<grid, CDIST_THREADS, smem, st>>>(query, table, grad_distance, grad_query, n, c, dc); break;
            case 32: cdist_bwd_query_kernel<32><<<grid, CDIST_THREADS, smem, st>>>(query, table, grad_distance, grad_query, n, c, dc); break;
            default: cdist_bwd_query_kernel<0><<<grid, CDIST_THREADS, smem, st>>>(query, table, grad_distance, grad_query, n, c, dc);
        }
        SPT_LAUNCH_CHECK("cdist_bwd_query_kernel");
    }
    {
        const int n_chunks = (int)((n + BWD_T_CHUNK - 1) / BWD_T_CHUNK);
        dim3 grid(n_chunks, m);
        size_t smem = (size_t)BWD_T_TILE * (dc + c) * sizeof(float);
        if (smem > 48 * 1024)
            cudaFuncSetAttribute(cdist_bwd_table_stage1, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cdist_bwd_table_stage1<<<grid, CDIST_THREADS, smem, st>>>(query, table, grad_distance, (float *)workspace, n,
                                                                  c, dc, n_chunks);
        SPT_LAUNCH_CHECK("cdist_bwd_table_stage1");
        dim3 grid2((c * dc + 127) / 128, m);
        cdist_bwd_table_stage2<<<grid2, 128, 0, st>>>((const float *)workspace, grad_table, c * dc, n_chunks);
        SPT_LAUNCH_CHECK("cdist_bwd_table_stage2");
    }
    return SPT_OK;
}

// ---------------------------------------------------------------------------------------------------
// PQ 'train' mode, fused (reference naive_gpt/layers/basic/quantizer.py:81-111, SURVEY.md section 8f-2):
//   d_c  = sum_i |z_i - W_ci|                   (L1 distance to the c codewords of the row's subspace)
//   idx  = argmin_c d_c (first minimum)          zq = W_idx                     (hard centroid)
//   w_c  = softmax(-log(clamp(d_c, 1e-5)))_c = (1 / max(d_c, 1e-5)) / sum_k (1 / max(d_k, 1e-5))
//   zw   = sum_c w_c W_c                          (soft centroid)
//   loss = mean((zw - zq)^2) + mean((z - zq)^2)   (means over all rows * m * dc elements)
// The reference runs ~10 torch ops over the materialised [m, rows, c] distance tensor, and its backward
// scatter-adds rows * m * dc values into 16 codewords per subspace (serialised atomics: 4.8 ms per call
// at the LLaMA-7B shape).  Here one thread owns (row, subspace) items of ONE subspace (grid stride is a
// multiple of m), recomputes everything in registers, and in the backward keeps its subspace's
// [c][dc] codebook gradient in registers across all its rows; threads are combined once per block
// through shared memory and once per launch through per-block partials (summed by the caller).
// sgn(x) = +1 if x > 0 else -1, the convention of the cdist backward (extension/cdist.cu:117,168).
// ---------------------------------------------------------------------------------------------------
namespace spt {

constexpr int PQT_THREADS = 256;

// g_loss = dLoss * 2 / (rows * m * dc).  grad_zq (optional, fp32 [rows, m*dc]) is the gradient that reached the
// hard-centroid output.  grad_z in z's dtype; grad_table partials [gridDim.x][m][C][DC] fp32.
//
// Four threads share one (row, subspace) item, each owning C/4 codewords: its slice of the codebook (32 floats) and
// of the codebook-gradient accumulator (32 floats) live in registers for the whole kernel, so the inner loops
// touch no memory at all; the few per-item scalars and the 8-vectors zw / grad_z are combined with quad shuffles.
// (First version: one thread per item with a 128-register accumulator — 255 registers, spills, one block per SM:
// 285 us per 1 M items.)
constexpr int PQB_SPLIT = 4;

template <typename T>
struct RawRow;   // one 8-element row held as raw 16-byte words (prefetched one iteration ahead)
template <>
struct RawRow<__nv_bfloat16> {
    uint4 v;
    __device__ __forceinline__ void load(const __nv_bfloat16 *p) { v = *reinterpret_cast<const uint4 *>(p); }
    __device__ __forceinline__ void unpack(float (&f)[8]) const {
        const uint32_t u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            f[2 * i] = __uint_as_float(u[i] << 16);
            f[2 * i + 1] = __uint_as_float(u[i] & 0xffff0000u);
        }
    }
};
template <>
struct RawRow<__half> {
    uint4 v;
    __device__ __forceinline__ void load(const __half *p) { v = *reinterpret_cast<const uint4 *>(p); }
    __device__ __forceinline__ void unpack(float (&f)[8]) const {
        const uint32_t u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float2 h = __half22float2(*reinterpret_cast<const __half2 *>(&u[i]));
            f[2 * i] = h.x;
            f[2 * i + 1] = h.y;
        }
    }
};
template <>
struct RawRow<float> {
    float4 a, b;
    __device__ __forceinline__ void load(const float *p) {
        a = *reinterpret_cast<const float4 *>(p);
        b = *reinterpret_cast<const float4 *>(p + 4);
    }
    __device__ __forceinline__ void unpack(float (&f)[8]) const {
        f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
    }
};
template <typename T, int DC, int C>
__global__ void __launch_bounds__(PQT_THREADS, 2)
pq_train_bwd_kernel(const T *__restrict__ z, const float *__restrict__ table, const float *__restrict__ grad_zq,
                    const float *__restrict__ grad_loss, float loss_scale, T *__restrict__ grad_z,
                    float *__restrict__ grad_table_partial, int64_t total, int m) {
    static_assert(DC == 8 && C % PQB_SPLIT == 0, "quad layout assumes 8-wide codewords");
    constexpr int KC = C / PQB_SPLIT;
    extern __shared__ __align__(16) float s_mem[];   // [m][PAD] codebook, then [m][C*DC] block gradient
    constexpr int PAD = C * DC + 4;
    float *s_w = s_mem, *s_g = s_mem + (size_t)m * PAD;
    for (int i = threadIdx.x; i < m * C * DC; i += blockDim.x) {
        s_w[(i / (C * DC)) * PAD + i % (C * DC)] = table[i];
        s_g[i] = 0.0f;
    }
    __syncthreads();
    const float gl = grad_loss[0] * loss_scale;
    const int j = threadIdx.x & (PQB_SPLIT - 1);     // which quarter of the codewords
    const int64_t item0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / PQB_SPLIT;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x / PQB_SPLIT;   // a multiple of m: s is fixed per thread
    const int s = (int)(item0 % m);
    const float *wt = s_w + (size_t)s * PAD;
    // element pairs (2p, 2p+1) are kept packed: the multiply-add parts run as FFMA2 / FADD2 (add.f32x2, fma.rn.f32x2)
    constexpr int NP = DC / 2;
    uint64_t w2[KC][NP], acc2[KC][NP];
#pragma unroll
    for (int k = 0; k < KC; ++k)
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            w2[k][p] = pk_f32x2(wt[(j * KC + k) * DC + 2 * p], wt[(j * KC + k) * DC + 2 * p + 1]);
            acc2[k][p] = 0ull;
        }
    // the shuffles need converged warps: the trip count is block-uniform and the tail is predicated.
    // The row of the NEXT iteration is fetched before this one's math (the loads were the largest stall).
    const uint64_t gl2 = pk_f32x2(gl, gl);
    RawRow<T> nxt;
    nxt.load(z + (size_t)(item0 < total ? item0 : total - 1) * DC);
    const int64_t block_item0 = (int64_t)blockIdx.x * (PQT_THREADS / PQB_SPLIT);
    const int n_iter = block_item0 < total ? (int)((total - block_item0 + stride - 1) / stride) : 0;   // block-uniform
    for (int it = 0; it < n_iter; ++it) {
        const int64_t g = item0 + (int64_t)it * stride;
        const bool on = g < total;
        float zv[DC];
        nxt.unpack(zv);
        {
            const int64_t gn = g + stride;
            nxt.load(z + (size_t)(gn < total ? gn : total - 1) * DC);
        }
        float4 q0 = make_float4(0.f, 0.f, 0.f, 0.f), q1 = q0;          // gradient that reached the hard centroid
        if (grad_zq != nullptr && on) {
            q0 = *reinterpret_cast<const float4 *>(grad_zq + (size_t)g * DC);
            q1 = *reinterpret_cast<const float4 *>(grad_zq + (size_t)g * DC + 4);
        }
        uint64_t zv2[NP];
#pragma unroll
        for (int p = 0; p < NP; ++p) zv2[p] = pk_f32x2(zv[2 * p], zv[2 * p + 1]);
        // distances / soft weights of my codewords; quad-wide argmin (lowest index on ties) and weight sum
        float wgt[KC], a_sum = 0.0f, best = 1e13f;
        int idx = 0;
        uint32_t live = 0;
#pragma unroll
        for (int k = 0; k < KC; ++k) {
            float d = 0.0f;
#pragma unroll
            for (int p = 0; p < NP; ++p) {
                d += fabsf(zv[2 * p] - lo_f32x2(w2[k][p]));
                d += fabsf(zv[2 * p + 1] - hi_f32x2(w2[k][p]));
            }
            if (d < best) {
                best = d;
                idx = j * KC + k;
            }
            live |= (d > 1e-5f ? 1u : 0u) << k;
            wgt[k] = 1.0f / fmaxf(d, 1e-5f);
            a_sum += wgt[k];
        }
#pragma unroll
        for (int o = 1; o < PQB_SPLIT; o <<= 1) {
            a_sum += __shfl_xor_sync(0xffffffffu, a_sum, o);
            const float ob = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
            if (ob < best || (ob == best && oi < idx)) {
                best = ob;
                idx = oi;
            }
        }
        const float inv_a = 1.0f / a_sum;
        uint64_t zw2[NP], wk2[KC];
#pragma unroll
        for (int p = 0; p < NP; ++p) zw2[p] = 0ull;
#pragma unroll
        for (int k = 0; k < KC; ++k) {
            wgt[k] *= inv_a;
            wk2[k] = pk_f32x2(wgt[k], wgt[k]);
#pragma unroll
            for (int p = 0; p < NP; ++p) zw2[p] = fma_f32x2(wk2[k], w2[k][p], zw2[p]);
        }
#pragma unroll
        for (int o = 1; o < PQB_SPLIT; o <<= 1)
#pragma unroll
            for (int p = 0; p < NP; ++p) zw2[p] = add_f32x2(zw2[p], shfl_xor_f32x2(zw2[p], o));
        // e1 = g (zw - zq) (soft-assignment error), e2 = g (z - zq);  grad_z starts from e2 (a quarter per lane:
        // the quad sum below restores it exactly), the hard centroid W_idx receives gzq - e1 - e2 on its owner lane
        uint64_t e12[NP], gz2[NP];
        {
            const float4 c0 = *reinterpret_cast<const float4 *>(wt + idx * DC);
            const float4 c1 = *reinterpret_cast<const float4 *>(wt + idx * DC + 4);
            const uint64_t zq2[NP] = {pk_f32x2(c0.x, c0.y), pk_f32x2(c0.z, c0.w), pk_f32x2(c1.x, c1.y), pk_f32x2(c1.z, c1.w)};
            const uint64_t gin2[NP] = {pk_f32x2(q0.x, q0.y), pk_f32x2(q0.z, q0.w), pk_f32x2(q1.x, q1.y), pk_f32x2(q1.z, q1.w)};
            const uint64_t quarter2 = pk_f32x2(0.25f, 0.25f);
            static_assert(PQB_SPLIT == 4 && NP == 4, "the 0.25 above is 1 / PQB_SPLIT");
#pragma unroll
            for (int p = 0; p < NP; ++p) {
                e12[p] = mul_f32x2(gl2, sub_f32x2(zw2[p], zq2[p]));
                const uint64_t e22 = mul_f32x2(gl2, sub_f32x2(zv2[p], zq2[p]));
                gz2[p] = mul_f32x2(quarter2, e22);
                const uint64_t gq2 = sub_f32x2(sub_f32x2(gin2[p], e12[p]), e22);
#pragma unroll
                for (int k = 0; k < KC; ++k)
                    if (on && idx == j * KC + k) acc2[k][p] = add_f32x2(acc2[k][p], gq2);
            }
        }
        // gw_c = e1 . W_c ;  t = sum_c gw_c w_c ;  dd_c = -(a_c)^2 (gw_c - t) / A  with a_c = w_c A
        float gw[KC], t = 0.0f;
#pragma unroll
        for (int k = 0; k < KC; ++k) {
            uint64_t v2 = 0ull;
#pragma unroll
            for (int p = 0; p < NP; ++p) v2 = fma_f32x2(e12[p], w2[k][p], v2);
            gw[k] = lo_f32x2(v2) + hi_f32x2(v2);
            t = fmaf(gw[k], wgt[k], t);
        }
#pragma unroll
        for (int o = 1; o < PQB_SPLIT; o <<= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
        if (on) {
#pragma unroll
            for (int k = 0; k < KC; ++k) {
                // -sg = -dd * sign(z - w): the sign bit of the difference flips -dd (a zero difference counts as positive)
                const uint32_t ndd = __float_as_uint(((live >> k) & 1u) ? (wgt[k] * wgt[k]) * a_sum * (gw[k] - t) : 0.0f);
#pragma unroll
                for (int p = 0; p < NP; ++p) {
                    const uint64_t diff2 = sub_f32x2(zv2[p], w2[k][p]);
                    const uint32_t n_lo = ndd ^ (__float_as_uint(lo_f32x2(diff2)) & 0x80000000u);
                    const uint32_t n_hi = ndd ^ (__float_as_uint(hi_f32x2(diff2)) & 0x80000000u);
                    const uint64_t nsg2 = pk_f32x2(__uint_as_float(n_lo), __uint_as_float(n_hi));
                    gz2[p] = sub_f32x2(gz2[p], nsg2);
                    acc2[k][p] = add_f32x2(fma_f32x2(wk2[k], e12[p], acc2[k][p]), nsg2);
                }
            }
        }
        // reduce-scatter of grad_z over the quad: lane j ends with the pair (2j, 2j+1)
        uint64_t h[2], out2;
#pragma unroll
        for (int p = 0; p < 2; ++p) {
            const uint64_t keep = (j & 2) ? gz2[2 + p] : gz2[p], send = (j & 2) ? gz2[p] : gz2[2 + p];
            h[p] = add_f32x2(keep, shfl_xor_f32x2(send, 2));
        }
        {
            const uint64_t keep = (j & 1) ? h[1] : h[0], send = (j & 1) ? h[0] : h[1];
            out2 = add_f32x2(keep, shfl_xor_f32x2(send, 1));
        }
        if (on) {
            T *op = grad_z + (size_t)g * DC + 2 * j;
            if constexpr (std::is_same<T, __half>::value) {
                *reinterpret_cast<__half2 *>(op) = __floats2half2_rn(lo_f32x2(out2), hi_f32x2(out2));
            } else if constexpr (sizeof(T) == 2) {
                *reinterpret_cast<__nv_bfloat162 *>(op) = __floats2bfloat162_rn(lo_f32x2(out2), hi_f32x2(out2));
            } else {
                *reinterpret_cast<float2 *>(op) = make_float2(lo_f32x2(out2), hi_f32x2(out2));
            }
        }
    }
#pragma unroll
    for (int k = 0; k < KC; ++k)
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            atomicAdd(&s_g[(s * C + j * KC + k) * DC + 2 * p], lo_f32x2(acc2[k][p]));
            atomicAdd(&s_g[(s * C + j * KC + k) * DC + 2 * p + 1], hi_f32x2(acc2[k][p]));
        }
    __syncthreads();
    for (int i = threadIdx.x; i < m * C * DC; i += blockDim.x)
        grad_table_partial[(size_t)blockIdx.x * m * C * DC + i] = s_g[i];
}

// Forward of the 'train' mode: hard centroids (zq_out, optional) and the per-block partial sums of
// |zw - zq|^2 + |z - zq|^2.  Same quad layout as the backward: four lanes per (row, subspace) item, each with
// C/4 codewords in registers (one thread per item reading the codebook from shared memory took 2x longer).
template <typename T, int DC, int C>
__global__ void __launch_bounds__(PQT_THREADS)
pq_train_fwd_kernel(const T *__restrict__ z, const float *__restrict__ table, float *__restrict__ zq_out,
                    float *__restrict__ partial, int64_t total, int m) {
    static_assert(DC == 8 && C % PQB_SPLIT == 0, "quad layout assumes 8-wide codewords");
    constexpr int KC = C / PQB_SPLIT, NP = DC / 2;
    extern __shared__ __align__(16) float s_w[];   // [m][C*DC + 4] (padded: lanes differ in subspace)
    __shared__ float s_red[PQT_THREADS / 32];
    constexpr int PAD = C * DC + 4;
    for (int i = threadIdx.x; i < m * C * DC; i += blockDim.x) s_w[(i / (C * DC)) * PAD + i % (C * DC)] = table[i];
    __syncthreads();
    const int j = threadIdx.x & (PQB_SPLIT - 1);
    const int64_t item0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / PQB_SPLIT;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x / PQB_SPLIT;   // a multiple of m
    const float *wt = s_w + (size_t)(item0 % m) * PAD;
    uint64_t w2[KC][NP];
#pragma unroll
    for (int k = 0; k < KC; ++k)
#pragma unroll
        for (int p = 0; p < NP; ++p)
            w2[k][p] = pk_f32x2(wt[(j * KC + k) * DC + 2 * p], wt[(j * KC + k) * DC + 2 * p + 1]);
    RawRow<T> nxt;
    nxt.load(z + (size_t)(item0 < total ? item0 : total - 1) * DC);
    const int64_t block_item0 = (int64_t)blockIdx.x * (PQT_THREADS / PQB_SPLIT);
    const int n_iter = block_item0 < total ? (int)((total - block_item0 + stride - 1) / stride) : 0;   // block-uniform
    uint64_t local2 = 0ull;
    for (int it = 0; it < n_iter; ++it) {
        const int64_t g = item0 + (int64_t)it * stride;
        const bool on = g < total;
        float zv[DC];
        nxt.unpack(zv);
        {
            const int64_t gn = g + stride;
            nxt.load(z + (size_t)(gn < total ? gn : total - 1) * DC);
        }
        float wgt[KC], a_sum = 0.0f, best = 1e13f;
        int idx = 0;
#pragma unroll
        for (int k = 0; k < KC; ++k) {
            float d = 0.0f;
#pragma unroll
            for (int p = 0; p < NP; ++p) {
                d += fabsf(zv[2 * p] - lo_f32x2(w2[k][p]));
                d += fabsf(zv[2 * p + 1] - hi_f32x2(w2[k][p]));
            }
            if (d < best) {
                best = d;
                idx = j * KC + k;
            }
            wgt[k] = 1.0f / fmaxf(d, 1e-5f);
            a_sum += wgt[k];
        }
#pragma unroll
        for (int o = 1; o < PQB_SPLIT; o <<= 1) {
            a_sum += __shfl_xor_sync(0xffffffffu, a_sum, o);
            const float ob = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
            if (ob < best || (ob == best && oi < idx)) {
                best = ob;
                idx = oi;
            }
        }
        const float inv_a = 1.0f / a_sum;
        uint64_t zw2[NP];
#pragma unroll
        for (int p = 0; p < NP; ++p) zw2[p] = 0ull;
#pragma unroll
        for (int k = 0; k < KC; ++k) {
            const float wk = wgt[k] * inv_a;
            const uint64_t wk2 = pk_f32x2(wk, wk);
#pragma unroll
            for (int p = 0; p < NP; ++p) zw2[p] = fma_f32x2(wk2, w2[k][p], zw2[p]);
        }
        // reduce-scatter over the quad: lane j ends with the pair (2j, 2j+1) of zw, and handles that pair of the loss
        uint64_t h[2], zwj;
#pragma unroll
        for (int p = 0; p < 2; ++p) {
            const uint64_t keep = (j & 2) ? zw2[2 + p] : zw2[p], send = (j & 2) ? zw2[p] : zw2[2 + p];
            h[p] = add_f32x2(keep, shfl_xor_f32x2(send, 2));
        }
        {
            const uint64_t keep = (j & 1) ? h[1] : h[0], send = (j & 1) ? h[0] : h[1];
            zwj = add_f32x2(keep, shfl_xor_f32x2(send, 1));
        }
        if (on) {
            const float2 zq = *reinterpret_cast<const float2 *>(wt + idx * DC + 2 * j);
            const uint64_t zq2 = pk_f32x2(zq.x, zq.y);
            const float za = (j & 2) ? ((j & 1) ? zv[6] : zv[4]) : ((j & 1) ? zv[2] : zv[0]);
            const float zb = (j & 2) ? ((j & 1) ? zv[7] : zv[5]) : ((j & 1) ? zv[3] : zv[1]);
            const uint64_t e1 = sub_f32x2(zwj, zq2), e2 = sub_f32x2(pk_f32x2(za, zb), zq2);
            local2 = fma_f32x2(e1, e1, fma_f32x2(e2, e2, local2));
            if (zq_out) *reinterpret_cast<float2 *>(zq_out + (size_t)g * DC + 2 * j) = zq;
        }
    }
    float local = lo_f32x2(local2) + hi_f32x2(local2);
    local = warp_sum(local);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = local;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.0f;
        for (int i = 0; i < PQT_THREADS / 32; ++i) t += s_red[i];
        partial[blockIdx.x] = t;
    }
}

static int pq_train_grid(int64_t total, int m) {
    // one grid for both directions (the backward runs PQB_SPLIT threads per item, the forward one)
    constexpr int per_block = PQT_THREADS / PQB_SPLIT;
    int64_t want = (total + per_block - 1) / per_block;
    int64_t cap = (int64_t)num_sms() * 2;
    int64_t g = want < cap ? want : cap;
    // the grid stride in items (g * per_block, g * PQT_THREADS) must be a multiple of m: a thread keeps its subspace
    while ((g * per_block) % m != 0) ++g;
    return (int)g;
}

}  // namespace spt

extern "C" int spt_pq_train_blocks(int64_t rows, int m) { return spt::pq_train_grid(rows * m, m); }

extern "C" int spt_pq_train_fwd(const void *z, const float *table, float *zq_out, float *partial, int64_t rows, int m,
                                int c, int dc, int dtype, spt_stream_t stream) {
    SPT_REQUIRE(z && table && partial, "pq_train_fwd: null pointer");
    SPT_REQUIRE(c == 16 && dc == 8 && m >= 1 && m <= 64, "pq_train_fwd: fused path covers c = 16, dc = 8, m <= 64 (got c=%d dc=%d m=%d)", c, dc, m);
    SPT_REQUIRE(rows >= 1, "pq_train_fwd: no rows");
    const int64_t total = rows * m;
    const int grid = pq_train_grid(total, m);
    const size_t smem = (size_t)m * (16 * 8 + 4) * sizeof(float);
    if (dtype == SPT_F32)
        pq_train_fwd_kernel<float, 8, 16><<<grid, PQT_THREADS, smem, as_stream(stream)>>>((const float *)z, table, zq_out, partial, total, m);
    else if (dtype == SPT_BF16)
        pq_train_fwd_kernel<__nv_bfloat16, 8, 16><<<grid, PQT_THREADS, smem, as_stream(stream)>>>((const __nv_bfloat16 *)z, table, zq_out, partial, total, m);
    else if (dtype == SPT_F16)
        pq_train_fwd_kernel<__half, 8, 16><<<grid, PQT_THREADS, smem, as_stream(stream)>>>((const __half *)z, table, zq_out, partial, total, m);
    else
        return fail(SPT_ERR_INVALID_ARGUMENT, "pq_train_fwd: unknown dtype %d", dtype);
    return after_launch("pq_train_fwd_kernel");
}

extern "C" int spt_pq_train_bwd(const void *z, const float *table, const float *grad_zq, const float *grad_loss,
                                void *grad_z, float *grad_table_partial, int64_t rows, int m, int c, int dc, int dtype,
                                spt_stream_t stream) {
    SPT_REQUIRE(z && table && grad_loss && grad_z && grad_table_partial, "pq_train_bwd: null pointer");
    SPT_REQUIRE(c == 16 && dc == 8 && m >= 1 && m <= 64, "pq_train_bwd: fused path covers c = 16, dc = 8, m <= 64");
    SPT_REQUIRE(rows >= 1, "pq_train_bwd: no rows");
    const int64_t total = rows * m;
    const int grid = pq_train_grid(total, m);
    const float loss_scale = 2.0f / (float)((double)total * dc);
    const size_t smem = (size_t)m * (16 * 8 + 4 + 16 * 8) * sizeof(float);
    if (dtype == SPT_F32) {
        cudaFuncSetAttribute(pq_train_bwd_kernel<float, 8, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        pq_train_bwd_kernel<float, 8, 16><<<grid, PQT_THREADS, smem, as_stream(stream)>>>(
            (const float *)z, table, grad_zq, grad_loss, loss_scale, (float *)grad_z, grad_table_partial, total, m);
    } else if (dtype == SPT_BF16) {
        cudaFuncSetAttribute(pq_train_bwd_kernel<__nv_bfloat16, 8, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        pq_train_bwd_kernel<__nv_bfloat16, 8, 16><<<grid, PQT_THREADS, smem, as_stream(stream)>>>(
            (const __nv_bfloat16 *)z, table, grad_zq, grad_loss, loss_scale, (__nv_bfloat16 *)grad_z, grad_table_partial, total, m);
    } else if (dtype == SPT_F16) {
        cudaFuncSetAttribute(pq_train_bwd_kernel<__half, 8, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        pq_train_bwd_kernel<__half, 8, 16><<<grid, PQT_THREADS, smem, as_stream(stream)>>>(
            (const __half *)z, table, grad_zq, grad_loss, loss_scale, (__half *)grad_z, grad_table_partial, total, m);
    } else {
        return fail(SPT_ERR_INVALID_ARGUMENT, "pq_train_bwd: unknown dtype %d", dtype);
    }
    return after_launch("pq_train_bwd_kernel");
}
