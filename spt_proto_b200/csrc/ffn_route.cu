// Routed-FFN plumbing around the grouped GEMM: token -> block bucketing, row gather, block-ordered
// combine, per-group column sums (bias gradients).
//
// Reference semantics (naive_gpt/layers/sparse/feedforward.py:47-85): prob = sigmoid(router(x));
// topk(prob, k) picks the active blocks of each token (only SET MEMBERSHIP matters: the loop tests
// `any(indices == i)`); block i processes the tokens that picked it, in token order; results are
// accumulated into y in ascending block order.  Ties in topk are broken towards the LOWEST block
// index here (DESIGN.md section 6).
//
// Bucket layout produced by spt_route_bucket (everything stays on the device, no host sync):
//   bucket_ptr [nb+1]   row offsets, every bucket padded to a multiple of 128 rows so that each
//                       128-row GEMM tile belongs to exactly one block
//   tile_group [R/128]  block of every 128-row tile, -1 past the last bucket
//   row_token  [R]      token of every bucket row (ascending inside a bucket), -1 for padding rows
//   row_prob   [R]      prob[token, block] of the row (LoRA variant: coeff = 2 * prob), 0 for padding
//   token_rows [T, k]   bucket rows of the token's active blocks, blocks ascending
// R = round_up(T * k + 128 * nb, 128) is the caller-side upper bound (no sync needed to size it).
#include "common.cuh"

namespace spt {
namespace route {

constexpr int CHUNK = 256;  // tokens per CTA

// Total order on router probabilities, as torch.topk has it: NaN is the greatest value, then +inf ... -inf
// (-0 == +0).  Every comparison with NaN being false would give a NaN entry rank 0 WITHOUT ever outranking
// another entry, so a row with NaNs could mark more than k blocks active (and an all-NaN row all of them).
__device__ __forceinline__ uint32_t order_key(float p) {
    if (p != p) return 0xFFFFFFFFu;
    const uint32_t u = __float_as_uint(p + 0.0f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
// active-block mask of one token: block i is active iff fewer than k blocks beat it
// (key_j > key_i, or key_j == key_i with j < i) — exactly k blocks for any input, NaN / inf included.
__device__ __forceinline__ unsigned long long topk_mask(const float *p, int nb, int k) {
    unsigned long long m = 0;
    for (int i = 0; i < nb; ++i) {
        const uint32_t ki = order_key(p[i]);
        int rank = 0;
        for (int j = 0; j < nb; ++j) {
            const uint32_t kj = order_key(p[j]);
            rank += (kj > ki) || (kj == ki && j < i);
        }
        if (rank < k) m |= 1ull << i;
    }
    return m;
}

__global__ void __launch_bounds__(CHUNK)
mask_kernel(const float *__restrict__ prob, unsigned long long *__restrict__ active, int32_t *__restrict__ chunk_cnt,
            long long T, int nb, int k) {
    const long long t = (long long)blockIdx.x * CHUNK + threadIdx.x;
    unsigned long long m = 0;
    if (t < T) {
        float p[64];
        for (int i = 0; i < nb; ++i) p[i] = prob[t * nb + i];
        m = topk_mask(p, nb, k);
        active[t] = m;
    }
    for (int g = 0; g < nb; ++g) {
        const int c = __syncthreads_count((int)((m >> g) & 1ull));
        if (threadIdx.x == 0) chunk_cnt[(long long)blockIdx.x * nb + g] = c;
    }
}

// one CTA: exclusive scan of the chunk counts per block, padded bucket offsets, tile -> block table
__global__ void __launch_bounds__(256)
scan_kernel(int32_t *__restrict__ chunk_cnt, int32_t *__restrict__ bucket_ptr, int32_t *__restrict__ bucket_rows,
            int32_t *__restrict__ tile_group, int n_chunks, int nb, int n_tiles_max) {
    __shared__ int32_t s_ptr[65];
    if (threadIdx.x < nb) {
        const int g = threadIdx.x;
        int32_t run = 0;
        for (int c = 0; c < n_chunks; ++c) {
            const int32_t v = chunk_cnt[(long long)c * nb + g];
            chunk_cnt[(long long)c * nb + g] = run;
            run += v;
        }
        bucket_rows[g] = run;
        s_ptr[g + 1] = (run + 127) / 128 * 128;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        s_ptr[0] = 0;
        for (int g = 0; g < nb; ++g) s_ptr[g + 1] += s_ptr[g];
        for (int g = 0; g <= nb; ++g) bucket_ptr[g] = s_ptr[g];
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n_tiles_max; i += blockDim.x) {
        const int row = i * 128;
        int g = -1;
        for (int j = 0; j < nb; ++j)
            if (row >= s_ptr[j] && row < s_ptr[j + 1]) g = j;
        tile_group[i] = g;
    }
}

__global__ void __launch_bounds__(CHUNK)
place_kernel(const float *__restrict__ prob, const unsigned long long *__restrict__ active,
             const int32_t *__restrict__ chunk_base, const int32_t *__restrict__ bucket_ptr,
             int32_t *__restrict__ row_token, float *__restrict__ row_prob, int32_t *__restrict__ token_rows,
             long long T, int nb, int k) {
    __shared__ int32_t s_warp[CHUNK / 32];
    const long long t = (long long)blockIdx.x * CHUNK + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned long long m = t < T ? active[t] : 0ull;
    int slot = 0;
    for (int g = 0; g < nb; ++g) {
        const bool on = (m >> g) & 1ull;
        const unsigned bal = __ballot_sync(FULL, on);
        if (lane == 0) s_warp[warp] = __popc(bal);
        __syncthreads();
        int off = 0;
        for (int w = 0; w < warp; ++w) off += s_warp[w];
        __syncthreads();
        if (on && slot < k) {   // slot < k always holds (topk_mask marks exactly k blocks); kept as a guard
            const int row = bucket_ptr[g] + chunk_base[(long long)blockIdx.x * nb + g] + off + __popc(bal & ((1u << lane) - 1u));
            row_token[row] = (int32_t)t;
            row_prob[row] = prob[t * nb + g];
            token_rows[t * k + slot] = row;
            ++slot;
        }
    }
}

// dst[r, :] = src[row_token[r], :] (zeros for padding rows); 16-byte chunks, C % 8 == 0 (any 16-bit type: bf16 or fp16,
// the copy never looks at the values).
// One warp per (row, 2 KB span): every lane moves four 16-byte chunks, all four loads in flight before the stores.
constexpr int GR_UNROLL = 4;
__global__ void __launch_bounds__(256)
gather_rows_kernel(const __nv_bfloat16 *__restrict__ src, const int32_t *__restrict__ row_token,
                   __nv_bfloat16 *__restrict__ dst, long long R, int C, int spans) {
    const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= R * spans) return;
    const long long r = w / spans;
    const int c0 = (int)(w % spans) * (GR_UNROLL * 32) + lane;   // first chunk of this lane
    const int chunks = C / 8;
    const int t = row_token[r];
    const uint4 *sp = reinterpret_cast<const uint4 *>(src + (long long)(t < 0 ? 0 : t) * C);
    uint4 *dp = reinterpret_cast<uint4 *>(dst + r * C);
    uint4 v[GR_UNROLL];
#pragma unroll
    for (int u = 0; u < GR_UNROLL; ++u) {
        v[u] = make_uint4(0, 0, 0, 0);
        if (t >= 0 && c0 + 32 * u < chunks) v[u] = sp[c0 + 32 * u];
    }
#pragma unroll
    for (int u = 0; u < GR_UNROLL; ++u)
        if (c0 + 32 * u < chunks) dp[c0 + 32 * u] = v[u];
}

// y[t, :] = bias + sum_j part[token_rows[t, j], :]  (j ascending = block order), fp32 accumulation.
// The k rows are fetched four at a time (independent loads), then added in ascending j.
template <typename TP, typename TY>
__global__ void __launch_bounds__(256)
combine_kernel(const TP *__restrict__ part, const int32_t *__restrict__ token_rows, const float *__restrict__ bias,
               TY *__restrict__ y, long long T, int C, int k) {
    constexpr int V = Vec16<TP>::N;
    const int chunks = C / V;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= T * chunks) return;
    const long long t = idx / chunks;
    const int c = (int)(idx % chunks) * V;
    float acc[V];
#pragma unroll
    for (int i = 0; i < V; ++i) acc[i] = bias ? bias[c + i] : 0.0f;
    for (int j0 = 0; j0 < k; j0 += 4) {
        int row[4];
        float v[4][V];
#pragma unroll
        for (int u = 0; u < 4; ++u) row[u] = j0 + u < k ? token_rows[t * k + j0 + u] : -1;
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (row[u] >= 0) Vec16<TP>::load(part + (long long)row[u] * C + c, v[u]);
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (row[u] >= 0) {
#pragma unroll
                for (int i = 0; i < V; ++i) acc[i] += v[u][i];
            }
    }
    if constexpr (sizeof(TY) == 2 && V == 8) {
        Vec16<TY>::store(y + t * C + c, acc);
    } else {
#pragma unroll
        for (int i = 0; i < V; ++i) y[t * C + c + i] = from_f32<TY>(acc[i]);
    }
}

// out[g, c] = sum over rows bucket_ptr[g] .. bucket_ptr[g+1] of x[row, c]; two deterministic stages
constexpr int CS_SPLIT = 64;
// block = 8 warps over one 256-column strip of one row part: lane = 8 consecutive columns (one 16-byte load per row, a warp
// reads 512 contiguous bytes), warp w takes rows a + w, a + w + 8, ... four at a time (independent loads in flight: with one
// load per thread and 128 blocks the kernel ran at a quarter of the HBM rate); the eight warps' sums meet in shared memory
// in warp order, so the result is deterministic.
constexpr int CS_WARPS = 8;
template <typename T>   // bf16 or fp16
__global__ void __launch_bounds__(32 * CS_WARPS)
colsum_stage1(const T *__restrict__ x, const int32_t *__restrict__ bucket_ptr, float *__restrict__ partial,
              int C) {
    __shared__ float red[CS_WARPS][256 + 8];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int c = blockIdx.x * 256 + lane * 8;
    const int part = blockIdx.y, g = blockIdx.z;
    const int r0 = bucket_ptr[g], r1 = bucket_ptr[g + 1];
    const int per = (r1 - r0 + CS_SPLIT - 1) / CS_SPLIT;
    const int a = r0 + part * per, b = min(r1, a + per);
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (c + 8 <= C && (C % 8 == 0) && (reinterpret_cast<uintptr_t>(x) % 16 == 0)) {
        const T *px = x + c;
        int r = a + w;
        for (; r + 3 * CS_WARPS < b; r += 4 * CS_WARPS) {
            float v[4][8];
#pragma unroll
            for (int u = 0; u < 4; ++u) Vec16<T>::load(px + (long long)(r + u * CS_WARPS) * C, v[u]);
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int i = 0; i < 8; ++i) acc[i] += v[u][i];
        }
        for (; r < b; r += CS_WARPS) {
            float v[8];
            Vec16<T>::load(px + (long long)r * C, v);
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[i] += v[i];
        }
    } else {
        for (int i = 0; i < 8 && c + i < C; ++i)
            for (int r = a + w; r < b; r += CS_WARPS) acc[i] += to_f32(x[(long long)r * C + c + i]);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) red[w][lane * 8 + i] = acc[i];
    __syncthreads();
    const int cc = blockIdx.x * 256 + threadIdx.x;
    if (cc < C) {
        float t = 0.0f;
#pragma unroll
        for (int u = 0; u < CS_WARPS; ++u) t += red[u][threadIdx.x];
        partial[((long long)g * CS_SPLIT + part) * C + cc] = t;
    }
}
__global__ void __launch_bounds__(128)
colsum_stage2(const float *__restrict__ partial, float *__restrict__ out, int C) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int g = blockIdx.y;
    if (c >= C) return;
    float acc = 0.0f;
    for (int p = 0; p < CS_SPLIT; ++p) acc += partial[((long long)g * CS_SPLIT + p) * C + c];
    out[(long long)g * C + c] = acc;
}

// router gradient of the LoRA-routed FFN: coeff[r] = 2 * prob[token(r), block(r)] (lora_ffn.py:92,206), so
// grad_prob[token(r), block(r)] = 2 * grad_coeff[r]; every (token, block) pair owns at most one bucket row: plain stores
__global__ void __launch_bounds__(256)
row_coeff_bwd_kernel(const float *__restrict__ grad_coeff, const int32_t *__restrict__ row_token,
                     const int32_t *__restrict__ tile_group, float *__restrict__ grad_prob, long long R, int nb) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    const int t = row_token[r], g = tile_group[r >> 7];
    if (t >= 0 && g >= 0) grad_prob[(long long)t * nb + g] = 2.0f * grad_coeff[r];
}

}  // namespace route
}  // namespace spt

using namespace spt;

extern "C" int spt_row_coeff_bwd(const float *grad_coeff, const int32_t *row_token, const int32_t *tile_group,
                                 float *grad_prob, int64_t R, int64_t T, int nb, spt_stream_t stream) {
    SPT_REQUIRE(grad_coeff && row_token && tile_group && grad_prob, "row_coeff_bwd: null pointer");
    SPT_REQUIRE(R >= 128 && R % 128 == 0 && T >= 1 && nb >= 1 && nb <= 64, "row_coeff_bwd: bad sizes");
    cudaStream_t st = as_stream(stream);
    if (cudaMemsetAsync(grad_prob, 0, (size_t)T * nb * sizeof(float), st) != cudaSuccess)
        return fail(SPT_ERR_CUDA, "row_coeff_bwd: memset failed");
    route::row_coeff_bwd_kernel<<<(unsigned)((R + 255) / 256), 256, 0, st>>>(grad_coeff, row_token, tile_group, grad_prob, R, nb);
    return after_launch("row_coeff_bwd_kernel");
}

extern "C" size_t spt_route_bucket_workspace_bytes(int64_t T, int nb) {
    const size_t n_chunks = (size_t)(T + route::CHUNK - 1) / route::CHUNK;
    return (size_t)T * 8 + n_chunks * nb * 4 + 64;
}

extern "C" int spt_route_bucket(const float *prob, int32_t *bucket_ptr, int32_t *bucket_rows, int32_t *tile_group,
                                int32_t *row_token, float *row_prob, int32_t *token_rows, void *workspace, int64_t T,
                                int nb, int k_active, int64_t R, spt_stream_t stream) {
    SPT_REQUIRE(prob && bucket_ptr && bucket_rows && tile_group && row_token && row_prob && token_rows && workspace,
                "route_bucket: null pointer");
    SPT_REQUIRE(T >= 1 && nb >= 1 && nb <= 64 && k_active >= 1 && k_active <= nb, "route_bucket: bad sizes T=%lld nb=%d k=%d",
                (long long)T, nb, k_active);
    SPT_REQUIRE(R % 128 == 0 && R >= T * k_active + 127LL * nb, "route_bucket: R=%lld too small (need >= T*k + 127*nb, multiple of 128)", (long long)R);
    cudaStream_t st = as_stream(stream);
    const int n_chunks = (int)((T + route::CHUNK - 1) / route::CHUNK);
    unsigned long long *active = (unsigned long long *)workspace;
    int32_t *chunk_cnt = (int32_t *)((char *)workspace + (size_t)T * 8);
    cudaMemsetAsync(row_token, 0xFF, (size_t)R * 4, st);
    cudaMemsetAsync(row_prob, 0, (size_t)R * 4, st);
    route::mask_kernel<<<n_chunks, route::CHUNK, 0, st>>>(prob, active, chunk_cnt, T, nb, k_active);
    SPT_LAUNCH_CHECK("route mask_kernel");
    route::scan_kernel<<<1, 256, 0, st>>>(chunk_cnt, bucket_ptr, bucket_rows, tile_group, n_chunks, nb, (int)(R / 128));
    SPT_LAUNCH_CHECK("route scan_kernel");
    route::place_kernel<<<n_chunks, route::CHUNK, 0, st>>>(prob, active, chunk_cnt, bucket_ptr, row_token, row_prob,
                                                           token_rows, T, nb, k_active);
    SPT_LAUNCH_CHECK("route place_kernel");
    return SPT_OK;
}

extern "C" int spt_gather_rows_bf16(const void *src, const int32_t *row_token, void *dst, int64_t R, int C,
                                    spt_stream_t stream) {
    SPT_REQUIRE(src && row_token && dst, "gather_rows: null pointer");
    SPT_REQUIRE(R >= 1 && C >= 8 && C % 8 == 0, "gather_rows: C must be a positive multiple of 8 (got %d)", C);
    const int spans = (C / 8 + route::GR_UNROLL * 32 - 1) / (route::GR_UNROLL * 32);
    const long long n = (long long)R * spans * 32;     // one warp per (row, span)
    SPT_REQUIRE((n + 255) / 256 < (1ll << 31), "gather_rows: too many rows");
    route::gather_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, as_stream(stream)>>>(
        (const __nv_bfloat16 *)src, row_token, (__nv_bfloat16 *)dst, R, C, spans);
    return after_launch("gather_rows_kernel");
}

extern "C" int spt_ffn_combine(const void *partial, const int32_t *token_rows, const float *bias, void *y, int64_t T,
                               int C, int k_active, int partial_dtype, int y_dtype, spt_stream_t stream) {
    SPT_REQUIRE(partial && token_rows && y, "ffn_combine: null pointer");
    SPT_REQUIRE(T >= 1 && C >= 8 && C % 8 == 0 && k_active >= 1, "ffn_combine: bad sizes");
    using bf = __nv_bfloat16;
    using hf = __half;
    cudaStream_t st = as_stream(stream);
    const int V = partial_dtype == SPT_F32 ? 4 : 8;
    const long long n = (long long)T * (C / V);
    const unsigned grid = (unsigned)((n + 255) / 256);
    if (partial_dtype == SPT_BF16 && y_dtype == SPT_BF16)
        route::combine_kernel<bf, bf><<<grid, 256, 0, st>>>((const bf *)partial, token_rows, bias, (bf *)y, T, C, k_active);
    else if (partial_dtype == SPT_BF16 && y_dtype == SPT_F32)
        route::combine_kernel<bf, float><<<grid, 256, 0, st>>>((const bf *)partial, token_rows, bias, (float *)y, T, C, k_active);
    else if (partial_dtype == SPT_F32 && y_dtype == SPT_F32)
        route::combine_kernel<float, float><<<grid, 256, 0, st>>>((const float *)partial, token_rows, bias, (float *)y, T, C, k_active);
    else if (partial_dtype == SPT_F32 && y_dtype == SPT_BF16)
        route::combine_kernel<float, bf><<<grid, 256, 0, st>>>((const float *)partial, token_rows, bias, (bf *)y, T, C, k_active);
    else if (partial_dtype == SPT_F16 && y_dtype == SPT_F16)
        route::combine_kernel<hf, hf><<<grid, 256, 0, st>>>((const hf *)partial, token_rows, bias, (hf *)y, T, C, k_active);
    else if (partial_dtype == SPT_F16 && y_dtype == SPT_F32)
        route::combine_kernel<hf, float><<<grid, 256, 0, st>>>((const hf *)partial, token_rows, bias, (float *)y, T, C, k_active);
    else if (partial_dtype == SPT_F32 && y_dtype == SPT_F16)
        route::combine_kernel<float, hf><<<grid, 256, 0, st>>>((const float *)partial, token_rows, bias, (hf *)y, T, C, k_active);
    else
        return fail(SPT_ERR_INVALID_ARGUMENT,
                    "ffn_combine: dtype pair (partial %d, y %d) not supported: fp32 pairs with fp32, bf16 or fp16, and a "
                    "16-bit type with itself or fp32 (bf16 and fp16 do not mix)", partial_dtype, y_dtype);
    return after_launch("combine_kernel");
}

extern "C" size_t spt_group_colsum_workspace_bytes(int n_groups, int C) {
    return (size_t)n_groups * route::CS_SPLIT * C * sizeof(float);
}

extern "C" int spt_group_colsum(const void *x, const int32_t *bucket_ptr, float *out, void *workspace, int n_groups, int C,
                                int dtype, spt_stream_t stream) {
    SPT_REQUIRE(x && bucket_ptr && out && workspace, "group_colsum: null pointer");
    SPT_REQUIRE(n_groups >= 1 && n_groups <= 65535 && C >= 1, "group_colsum: bad sizes");
    SPT_REQUIRE(dtype == SPT_BF16 || dtype == SPT_F16, "group_colsum: dtype %d unknown: x is SPT_BF16 (1) or SPT_F16 (2)", dtype);
    cudaStream_t st = as_stream(stream);
    dim3 g1((C + 255) / 256, route::CS_SPLIT, n_groups);
    if (dtype == SPT_F16)
        route::colsum_stage1<__half><<<g1, 32 * route::CS_WARPS, 0, st>>>((const __half *)x, bucket_ptr, (float *)workspace, C);
    else
        route::colsum_stage1<__nv_bfloat16><<<g1, 32 * route::CS_WARPS, 0, st>>>((const __nv_bfloat16 *)x, bucket_ptr,
                                                                                 (float *)workspace, C);
    SPT_LAUNCH_CHECK("colsum_stage1");
    route::colsum_stage2<<<dim3((C + 127) / 128, n_groups), 128, 0, st>>>((const float *)workspace, out, C);
    return after_launch("colsum_stage2");
}

extern "C" int spt_group_colsum_bf16(const void *x, const int32_t *bucket_ptr, float *out, void *workspace, int n_groups,
                                     int C, spt_stream_t stream) {
    return spt_group_colsum(x, bucket_ptr, out, workspace, n_groups, C, SPT_BF16, stream);
}
