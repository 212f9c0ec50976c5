// (6) Routed-FFN grouped GEMM on the 5th-generation tensor cores (tcgen05 + TMEM + TMA), bf16 or fp16 in
// (A and B of one type T, a template parameter of both kernels), fp32 accumulate.
//
// The reference ships the routed FFN as a Python loop over weight blocks — boolean mask, gather,
// addmm, activation, matmul, scatter-add per block (naive_gpt/layers/sparse/feedforward.py:47-85);
// its native attempt (legacy/routed.cpp:10-68) was never finished.  Here tokens are bucketed by
// activated block once (ffn_route.cu), every bucket is padded to a multiple of 128 rows, and all
// blocks run in ONE launch per product:
//
//   mode 0 "M-grouped":  C[i, :] = epi( A[i, :] . B_g^T ),  g = group of the 128-row tile of row i
//       fc1 : A = bucketed tokens  [R, d]  (K-major)   B_g = W1[g*bs:(g+1)*bs, :]        (K-major)
//       fc2 : A = bucketed hidden  [R, bs] (K-major)   B_g = W2[:, g*bs:(g+1)*bs]        (K-major, ld F)
//       dH  : A = dY bucketed      [R, d]  (K-major)   B_g = W2[:, g*bs:(g+1)*bs]^T      (MN-major)
//       dX  : A = dU               [R, bs] (K-major)   B_g = W1[g*bs:(g+1)*bs, :]^T      (MN-major)
//   mode 1 "K-grouped":  C_g = A_g^T-style products over the group's rows (weight gradients)
//       dW1_g = dU_g^T X_g : A = dU [R, bs] (MN-major, M = bs), B = X [R, d] (MN-major, N = d)
//       dW2_g = dY_g^T H_g : A = dY [R, d]  (MN-major, M = d),  B = H [R, bs] (MN-major, N = bs)
//   MN-major operands are consumed straight from their row-major home through MN-major UMMA shared
//   memory descriptors — no transposed copies of weights or activations are ever made (the
//   reference materialises a permuted copy of W2 on every call, feedforward.py:94-102).
//
// Two kernels share the operand layout and the epilogue:
//   grouped_gemm_pair_kernel (default): CTA pairs (tcgen05 cta_group::2), 256x256 units, see its header below
//   grouped_gemm_kernel      (SPT_GEMM_CTA_PAIR=0, or more than 1024 m-tiles): one CTA per SM, 128x256 tiles
// Anatomy of both (persistent CTAs, tiles dealt round-robin):
//   warp 0   : TMA producer  — cp.async.bulk.tensor.2d into a ring of 128B-swizzled tiles
//   warp 1   : TMEM allocator + MMA issuer — one elected lane issues tcgen05.mma (kind::f16)
//   warps 2-9: epilogue — tcgen05.ld TMEM -> registers, bias / activation / row scale / gate, staged through
//              shared memory into coalesced global stores
//   smem full/empty mbarriers between TMA and MMA, full/empty mbarriers per TMEM accumulator (two of them)
//   between MMA and epilogue.
#include <algorithm>
#include <cstdlib>
#include <type_traits>

#include "tc.cuh"

namespace spt {
namespace gemm {

// Single-CTA kernel: 128 x 256 output tiles, PERSISTENT CTAs (one per SM): the TMA producer streams k-blocks of
// consecutive tiles through a 3-stage ring without draining between tiles, and two 256-column TMEM accumulators
// let the epilogue of tile i run under the main loop of tile i+1.  An N = 256 MMA of one CTA reads 12 KB of shared
// memory per k-step while TMA writes the next stage: the stream runs at ~2/3 of the MMA floor (171 clk measured
// against 128), which is what the CTA-pair kernel below removes.
//
// Round-1 measurements on the FFN step of bench.py (6 GEMMs, 0.825 TFLOP): first version 1.70 ms; epilogue through
// shared memory + N-fastest tile order 0.91 ms; CTA pairs 0.78 ms; epilogue values kept in registers (a run-time
// loop bound in the ragged-edge path had put the 32-value row buffer in local memory in EVERY path) 0.63 ms
// = 1.30 PFLOP/s.  With the epilogue switched off the pair kernel needs 0.565 ms, the MMA stream alone 0.50 ms
// (1.65 PFLOP/s, the cuBLAS burst figure of MEASURED_PEAKS.json), TMA alone 0.48 ms (12.9 TB/s out of L2).
constexpr int BM = 128, BN = 256, BK = 64, UMMA_K = 16, STAGES = 3;
constexpr int EPI_WARPS = 8;                            // two per TMEM lane quarter, each owning 128 of the 256 columns
constexpr int THREADS = 64 + EPI_WARPS * 32;
constexpr int STG_PITCH = 144;                          // staging row pitch in bytes (32 fp32 + pad; 16-byte aligned, conflict-free)
constexpr int A_TILE_BYTES = BM * BK * 2;               // 16 KB
constexpr int B_TILE_BYTES = BN * BK * 2;               // 32 KB
constexpr int SMEM_BYTES = STAGES * (A_TILE_BYTES + B_TILE_BYTES) + EPI_WARPS * 32 * STG_PITCH + 1024 /*align slack*/ + 256 /*barriers*/;
constexpr int TMEM_COLS = 512;                          // two accumulators of BN columns

struct Params {
    int mode;                      // 0 = M-grouped, 1 = K-grouped
    const int32_t *tile_group;     // mode 0: group of every 128-row tile (-1 = unused tail tile)
    int tiles_m, tiles_n, n_tiles; // tile grid: tile t -> (n = t % tiles_n, m = (t / tiles_n) % tiles_m, z = t / (tiles_n * tiles_m))
    const int32_t *group_ptr;      // mode 1: padded row offsets [G+1] (K range of group g)
    int K;                         // mode 0: reduction extent
    int M, N;                      // mode 1: output tile extents per group; mode 0: N only
    int a_mn_major, b_mn_major;
    // per-group coordinate offsets (elements): *_k along the reduction dim, *_mn along M / N
    int a_k_off, a_mn_off, b_k_off, b_mn_off;
    long long c_row_off, c_col_off;  // mode 1: C_g origin = (g * c_row_off, g * c_col_off)
    void *C;
    long long ldc;
    int c_dtype;                   // SPT_F32 or the operand type
    const float *bias;             // optional, bias[g * bias_stride + n]
    int bias_stride;
    const float *row_scale;        // optional, one factor per C row (mode 0)
    int act;                       // 0 none, 1 relu, 2 silu
    const void *gate;              // optional (mode 0, operand type): zero C where gate <= 0, gate[row * ldg + col]
    long long ldg;
};

using namespace spt::tc;

// Operand tile of one stage -> descriptor of its k-th K16 slice.
//   K-major  : [128 rows][64 k] rows of 128 B, 8-row swizzle atoms: SBO = 1024, slice k = +32 B
//   MN-major : two [64 k][64 mn] halves (8 KB each): SBO = 1024 (8 k-rows), LBO = 8192 (next 64 mn),
//              slice k = +16 rows = +2048 B
__device__ __forceinline__ uint64_t operand_desc(uint32_t tile_addr, int mn_major, int k) {
    return mn_major ? make_desc(tile_addr + k * (UMMA_K * 128), BK * 128, 1024)
                    : make_desc(tile_addr + k * (UMMA_K * 2), 0, 1024);
}

__device__ __forceinline__ float apply_act(float v, int act) {
    if (act == 1) return fmaxf(v, 0.0f);
    if (act == 2) return v / (1.0f + __expf(-v));
    return v;
}

// tile t of the launch -> coordinates, group, k range (identical in every role)
struct Tile {
    int g, m0, n0, k_begin, n_kblk;
    long long c_row0, c_col0;
    bool valid;
};
__device__ __forceinline__ Tile get_tile(const Params &p, int t) {
    Tile ti;
    const int tile_n = t % p.tiles_n, tile_m = (t / p.tiles_n) % p.tiles_m, z = t / (p.tiles_n * p.tiles_m);
    ti.m0 = tile_m * BM;
    ti.n0 = tile_n * BN;
    if (p.mode == 0) {
        ti.g = p.tile_group[tile_m];
        ti.valid = ti.g >= 0;
        ti.k_begin = 0;
        ti.n_kblk = ti.valid ? (p.K + BK - 1) / BK : 0;
        ti.c_row0 = ti.m0;
        ti.c_col0 = ti.n0;
    } else {
        ti.g = z;
        ti.valid = true;
        ti.k_begin = p.group_ptr[z];
        ti.n_kblk = (p.group_ptr[z + 1] - ti.k_begin + BK - 1) / BK;
        ti.c_row0 = (long long)z * p.c_row_off + ti.m0;
        ti.c_col0 = (long long)z * p.c_col_off + ti.n0;
    }
    return ti;
}

// kind::f16 instruction descriptor bits of the operand type: A / B format fields (bits 7-9, 10-12) = 1 for bf16,
// 0 for fp16 (tc.cuh idesc_fp16)
template <typename T>
constexpr uint32_t ab_format_bits() { return std::is_same<T, __half>::value ? 0u : (1u << 7) | (1u << 10); }
template <typename T>
constexpr int c16_dtype() { return std::is_same<T, __half>::value ? SPT_F16 : SPT_BF16; }

template <typename T>
__global__ void __launch_bounds__(THREADS, 1)
grouped_gemm_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                    const Params p) {
    extern __shared__ unsigned char smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023) & ~1023u;                 // 128B swizzle needs 1024-byte alignment
    unsigned char *smem = smem_raw + (base - raw);
    const uint32_t s_a = base, s_b = base + STAGES * A_TILE_BYTES;
    unsigned char *s_stage = smem + STAGES * (A_TILE_BYTES + B_TILE_BYTES);                  // epilogue staging, per warp
    uint64_t *bars = reinterpret_cast<uint64_t *>(s_stage + EPI_WARPS * 32 * STG_PITCH);
    const uint32_t bar0 = smem_u32(bars);
    auto full_bar = [&](int s) { return bar0 + s * 8; };
    auto empty_bar = [&](int s) { return bar0 + (STAGES + s) * 8; };
    auto acc_full = [&](int a) { return bar0 + (2 * STAGES + a) * 8; };
    auto acc_empty = [&](int a) { return bar0 + (2 * STAGES + 2 + a) * 8; };
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * STAGES + 4);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full_bar(s), 1);
            mbar_init(empty_bar(s), 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(acc_full(a), 1);
            mbar_init(acc_empty(a), EPI_WARPS * 32);
        }
        mbar_fence_init();
    }
    if (warp == 1) tmem_alloc<TMEM_COLS>(smem_u32(tmem_slot));
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;

    // Tiles are dealt round-robin: at any moment the resident CTAs work on consecutive tiles = consecutive N
    // tiles of the same M tile, which share the A tile (read from DRAM once) and walk the group's weight panel.
    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            uint32_t it = 0;   // k-blocks issued so far (ring position)
            for (int t = blockIdx.x; t < p.n_tiles; t += gridDim.x) {
                const Tile ti = get_tile(p, t);
                if (!ti.valid) continue;
                const int a_k = ti.g * p.a_k_off, a_mn = (p.mode == 0 ? ti.m0 : ti.g * p.a_mn_off + ti.m0);
                const int b_k = ti.g * p.b_k_off, b_mn = ti.g * p.b_mn_off + ti.n0;
                for (int kb = 0; kb < ti.n_kblk; ++kb, ++it) {
                    const int s = it % STAGES;
                    mbar_wait(empty_bar(s), ((it / STAGES) & 1) ^ 1);
                    mbar_expect_tx(full_bar(s), A_TILE_BYTES + B_TILE_BYTES);
                    const int k0 = ti.k_begin + kb * BK;
                    const uint32_t da = s_a + s * A_TILE_BYTES, db = s_b + s * B_TILE_BYTES;
                    if (p.a_mn_major) {   // tensor map dims: (mn contiguous, k rows); 64-wide chunks of 8 KB
#pragma unroll
                        for (int h = 0; h < BM / 64; ++h) tma_load_2d(da + h * 8192, &map_a, full_bar(s), a_mn + 64 * h, a_k + k0);
                    } else {              // tensor map dims: (k contiguous, mn rows)
                        tma_load_2d(da, &map_a, full_bar(s), a_k + k0, a_mn);
                    }
                    if (p.b_mn_major) {
#pragma unroll
                        for (int h = 0; h < BN / 64; ++h) tma_load_2d(db + h * 8192, &map_b, full_bar(s), b_mn + 64 * h, b_k + k0);
                    } else {              // two boxes of 128 rows
                        tma_load_2d(db, &map_b, full_bar(s), b_k + k0, b_mn);
                        tma_load_2d(db + B_TILE_BYTES / 2, &map_b, full_bar(s), b_k + k0, b_mn + 128);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: the whole warp runs the (uniform) loops, one elected lane issues; descriptors of a
        // stage's k-slices are a base (computed once) plus small adds =====
        // instruction descriptor: D = f32 (bits 4-5 = 1), A / B format (bits 7-9, 10-12: 1 = bf16, 0 = fp16),
        // a_major bit 15, b_major bit 16, N >> 3 at bit 17, M >> 4 at bit 24
        const uint32_t idesc = (1u << 4) | ab_format_bits<T>() | ((uint32_t)p.a_mn_major << 15) |
                               ((uint32_t)p.b_mn_major << 16) | ((uint32_t)((BN / 2) >> 3) << 17) |
                               ((uint32_t)(BM >> 4) << 24);
        const uint64_t da0 = operand_desc(s_a, p.a_mn_major, 0), db0 = operand_desc(s_b, p.b_mn_major, 0);
        const uint64_t a_step = p.a_mn_major ? MNMAJOR_K16 : KMAJOR_K16, b_step = p.b_mn_major ? MNMAJOR_K16 : KMAJOR_K16;
        uint32_t it = 0, n_acc = 0;   // ring position; accumulators handed to the epilogue so far
        for (int t = blockIdx.x; t < p.n_tiles; t += gridDim.x) {
            const Tile ti = get_tile(p, t);
            if (!ti.valid) continue;
            const int acc = n_acc & 1;
            mbar_wait(acc_empty(acc), ((n_acc >> 1) & 1) ^ 1);   // the epilogue has drained this accumulator
            fence_after_sync();
            for (int kb = 0; kb < ti.n_kblk; ++kb, ++it) {
                const int s = it % STAGES;
                mbar_wait(full_bar(s), (it / STAGES) & 1);
                fence_after_sync();
                if (elect_one()) {
                    const uint64_t da = da0 + (uint64_t)(s * (A_TILE_BYTES >> 4)), db = db0 + (uint64_t)(s * (B_TILE_BYTES >> 4));
                    // Back-to-back MMAs into the SAME accumulator are serialised by the accumulate dependency (~93 clk
                    // each in a micro-benchmark, whatever N); the tile is therefore issued as two N = 128 halves whose
                    // k-steps alternate: consecutive instructions are independent and run at the MMA floor.
                    const uint64_t db_hi = db + (uint64_t)((B_TILE_BYTES / 2) >> 4);
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k) {
                        umma_bf16(tmem_base + acc * BN, da + k * a_step, db + k * b_step, idesc, (kb | k) != 0);
                        umma_bf16(tmem_base + acc * BN + BN / 2, da + k * a_step, db_hi + k * b_step, idesc, (kb | k) != 0);
                    }
                    umma_commit(empty_bar(s));                      // frees the smem stage when the MMAs retire
                }
                __syncwarp();
            }
            if (elect_one()) umma_commit(acc_full(acc));            // accumulator complete (also for an empty group)
            __syncwarp();
            ++n_acc;
        }
    } else {
        // ===== epilogue: warps 2..9.  TMEM lane quarter = warp % 4; the two warps of a quarter split the 256 columns.
        // A 32-row x 32-column chunk goes TMEM -> registers (thread = row) -> bias / activation / scale / gate ->
        // a per-warp shared-memory tile -> global memory with consecutive lanes on consecutive 16-byte segments
        // of a row (full sectors).  The first version stored 16 bytes per lane to 32 different rows and did
        // everything per element with run-time branches: it took 185 us per GEMM against 108 us of main loop.
        const int quarter = warp & 3, chalf = (warp - 2) >> 2;
        const int row_in_tile = quarter * 32 + lane;
        unsigned char *stage = s_stage + (warp - 2) * 32 * STG_PITCH;
        const bool out16 = p.c_dtype == c16_dtype<T>();
        const int esz = out16 ? 2 : 4;
        uint32_t n_acc = 0;
        for (int t = blockIdx.x; t < p.n_tiles; t += gridDim.x) {
            const Tile ti = get_tile(p, t);
            const int n_valid = min(BN, p.N - ti.n0);
            if (!ti.valid) {
                // tail tile beyond the bucketed rows: define its output (zeros) so that elementwise
                // consumers of the whole [R, N] buffer never see uninitialised memory
                for (int i = threadIdx.x - 64; i < BM * n_valid; i += EPI_WARPS * 32) {
                    const long long off = ((long long)ti.m0 + i / n_valid) * p.ldc + ti.n0 + i % n_valid;
                    if (out16) reinterpret_cast<T *>(p.C)[off] = from_f32<T>(0.0f);
                    else reinterpret_cast<float *>(p.C)[off] = 0.0f;
                }
                continue;
            }
            const int acc = n_acc & 1;
            mbar_wait(acc_full(acc), (n_acc >> 1) & 1);
            fence_after_sync();
            const int rows_ok = p.mode == 0 ? BM : min(BM, p.M - ti.m0);      // valid rows of the tile
            const long long c_row = ti.c_row0 + row_in_tile;
            const float rs = (p.row_scale && p.mode == 0) ? p.row_scale[c_row] : 1.0f;
            unsigned char *c_base = reinterpret_cast<unsigned char *>(p.C);
            const bool aligned = ((reinterpret_cast<uintptr_t>(p.C) + (size_t)ti.c_col0 * esz) % 16 == 0) && ((p.ldc * esz) % 16 == 0);
#pragma unroll 1
            for (int c0 = chalf * (BN / 2); c0 < (chalf + 1) * (BN / 2); c0 += 32) {
                if (c0 >= n_valid) break;    // (uniform) nothing to store beyond N
                uint32_t r[32];
                __syncwarp();
                tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * BN + c0, r);
                float v[32];
                const bool full = c0 + 32 <= n_valid;
                if (ti.n_kblk == 0) {
#pragma unroll
                    for (int i = 0; i < 32; ++i) r[i] = 0;           // empty group: no MMA ever wrote TMEM
                }
                if (p.bias) {
                    const float *bp = p.bias + (long long)ti.g * p.bias_stride + ti.n0 + c0;
#pragma unroll
                    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]) + ((full || c0 + i < n_valid) ? __ldg(bp + i) : 0.0f);
                } else {
#pragma unroll
                    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
                }
                if (p.act == 1) {
#pragma unroll
                    for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.0f);
                } else if (p.act == 2) {
#pragma unroll
                    for (int i = 0; i < 32; ++i) v[i] = v[i] / (1.0f + __expf(-v[i]));
                }
#pragma unroll
                for (int i = 0; i < 32; ++i) v[i] *= rs;
                if (p.gate && row_in_tile < rows_ok) {   // ReLU backward mask of the tensor this GEMM differentiates through
                    const T *gp = static_cast<const T *>(p.gate) + c_row * p.ldg + ti.c_col0 + c0;
                    if (full && (reinterpret_cast<uintptr_t>(gp) % 16 == 0)) {
#pragma unroll
                        for (int i = 0; i < 32; i += 8) {
                            float gv[8];
                            Vec16<T>::load(gp + i, gv);
#pragma unroll
                            for (int u = 0; u < 8; ++u)
                                if (!(gv[u] > 0.0f)) v[i + u] = 0.0f;
                        }
                    } else {
#pragma unroll
                        for (int i = 0; i < 32; ++i)
                            if (c0 + i < n_valid && !(to_f32(gp[i]) > 0.0f)) v[i] = 0.0f;
                    }
                }
                if (full && aligned) {
                    // registers -> staging tile (thread = row) -> coalesced global stores (lane = 16-byte segment)
                    unsigned char *srow = stage + lane * STG_PITCH;
                    if (out16) {
#pragma unroll
                        for (int i = 0; i < 32; i += 8) {
                            float t8[8] = {v[i], v[i + 1], v[i + 2], v[i + 3], v[i + 4], v[i + 5], v[i + 6], v[i + 7]};
                            Vec16<T>::store(reinterpret_cast<T *>(srow) + i, t8);
                        }
                    } else {
#pragma unroll
                        for (int i = 0; i < 32; i += 4)
                            *reinterpret_cast<float4 *>(srow + i * 4) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
                    }
                    __syncwarp();
                    const int segs = out16 ? 4 : 8;                 // 16-byte segments per row of the chunk
                    const int rows_per = 32 / segs;
                    const int seg = lane % segs, rsub = lane / segs;
                    for (int r0 = 0; r0 < 32; r0 += rows_per) {
                        const int rr = r0 + rsub;
                        if (quarter * 32 + rr < rows_ok) {
                            const uint4 val = *reinterpret_cast<const uint4 *>(stage + rr * STG_PITCH + seg * 16);
                            unsigned char *dst = c_base + ((ti.c_row0 + quarter * 32 + rr) * p.ldc + ti.c_col0 + c0) * esz + seg * 16;
                            *reinterpret_cast<uint4 *>(dst) = val;
                        }
                    }
                } else if (row_in_tile < rows_ok) {
                    if (out16) {
                        T *dst = reinterpret_cast<T *>(p.C) + c_row * p.ldc + ti.c_col0 + c0;
#pragma unroll
                        for (int i = 0; i < 32; ++i)      // static indices: a run-time bound would put v[] in local memory
                            if (c0 + i < n_valid) dst[i] = from_f32<T>(v[i]);
                    } else {
                        float *dst = reinterpret_cast<float *>(p.C) + c_row * p.ldc + ti.c_col0 + c0;
#pragma unroll
                        for (int i = 0; i < 32; ++i)
                            if (c0 + i < n_valid) dst[i] = v[i];
                    }
                }
            }
            fence_before_sync();
            mbar_arrive(acc_empty(acc));     // 256 arrivals: the accumulator may be overwritten
            ++n_acc;
        }
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 1) tmem_dealloc<TMEM_COLS>(tmem_base);
}

// =====================================================================================================
// CTA-pair version (tcgen05 cta_group::2): the two CTAs of a cluster sit on the two SMs of a TPC and run ONE
// M = 256, N = 256 MMA stream.  Each CTA stages its own 128 rows of A and HALF of the B tile (128 of the 256
// columns), so a k-step costs every SM 8 KB of shared-memory reads instead of 12 KB: the single-CTA kernel
// above is bound by exactly that (N = 256 MMAs took 171 clk against a floor of 128).  Stages shrink to 32 KB,
// the ring grows to 5.
//
//   unit          : 256 rows x 256 columns = m-tiles (2i, 2i+1) x one n-tile.  In mode 0 a pair that straddles two
//                   groups is run twice, once per group, with the other CTA's half computed on the wrong weights
//                   and thrown away (at most one such pair per group boundary).
//   leader (rank 0): expects the bytes of both CTAs on its full barrier, issues the MMAs, multicasts the
//                   commits (stage free / accumulator full) to both CTAs
//   both CTAs     : TMA producer warp (loads complete on the leader's barrier), 8 epilogue warps over their own
//                   128 TMEM lanes; one arrive per epilogue warp on the leader's accumulator-empty barrier
constexpr int STAGES2 = 5;
constexpr int HALF_BYTES = 128 * BK * 2;                // 16 KB: A rows of this CTA, or its half of B
constexpr int MAX_LIST = 1024;                          // mode 0: (pair, sub) entries -> up to 1024 m-tiles
constexpr int SMEM2_BYTES = STAGES2 * 2 * HALF_BYTES + EPI_WARPS * 32 * STG_PITCH + MAX_LIST * 2 + 1024 + 256;

struct Unit {
    int g, n0, k_begin, n_kblk;
    int a_mn, b_mn;          // this CTA's TMA coordinates along M / N
    long long c_row0, c_col0;  // this CTA's output origin
    bool mma;                // the unit runs MMAs (false: tail pair without rows -> zero fill only)
    int role;                // this CTA: 0 = idle (its half is discarded), 1 = active, 2 = zero-fill its rows
    int rows_ok;             // valid rows of this CTA's half
};

// mode 0 candidates c = 2 * pair + sub: sub 0 always exists; sub 1 only where the pair's second m-tile belongs to
// another (valid) group.  Shared by the kernel and the host-side plan (spt_grouped_gemm_plan, used by the CPU tests).
__host__ __device__ inline bool unit_exists(const int32_t *tile_group, int tiles_m, int c) {
    if ((c & 1) == 0) return true;
    const int t0 = c & ~1, t1 = t0 + 1;
    if (t1 >= tiles_m) return false;
    const int g1 = tile_group[t1];
    return g1 >= 0 && g1 != tile_group[t0];
}

__host__ __device__ inline Unit get_unit(const Params &p, int u, const uint16_t *list, int rank) {
    Unit un;
    const int tile_n = u % p.tiles_n;
    un.n0 = tile_n * BN;
    un.b_mn = un.n0 + rank * (BN / 2);
    un.c_col0 = un.n0;
    if (p.mode == 0) {
        const int e = list[u / p.tiles_n], pair = e >> 1, sub = e & 1;
        const int t0 = 2 * pair, t1 = 2 * pair + 1;
        const int g0 = p.tile_group[t0], g1 = t1 < p.tiles_m ? p.tile_group[t1] : -2;   // -2: no such tile
        un.g = sub ? g1 : g0;
        un.mma = un.g >= 0;
        const int mine = rank ? g1 : g0;
        un.role = (un.mma && mine == un.g) ? 1 : ((mine == -1 && sub == 0) ? 2 : 0);
        un.k_begin = 0;
        un.n_kblk = un.mma ? (p.K + BK - 1) / BK : 0;
        un.a_mn = (t0 + rank) * BM;
        un.c_row0 = (long long)(t0 + rank) * BM;
        un.rows_ok = BM;
        un.b_mn += un.g * p.b_mn_off;
    } else {
        const int pairs_m = (p.tiles_m + 1) / 2;
        const int pm = (u / p.tiles_n) % pairs_m, z = u / (p.tiles_n * pairs_m);
        const int m0 = (2 * pm + rank) * BM;
        un.g = z;
        un.mma = true;
        un.role = 1;
        un.k_begin = p.group_ptr[z];
        un.n_kblk = (p.group_ptr[z + 1] - un.k_begin + BK - 1) / BK;
        un.a_mn = z * p.a_mn_off + m0;
        un.c_row0 = (long long)z * p.c_row_off + m0;
        un.c_col0 += (long long)z * p.c_col_off;
        un.rows_ok = p.M - m0 < BM ? p.M - m0 : BM;     // <= 0 for the phantom half of an odd tile count
        un.b_mn += z * p.b_mn_off;
    }
    return un;
}

template <typename T>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS, 1)
grouped_gemm_pair_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                         const Params p, const int n_units_mode1) {
    extern __shared__ unsigned char smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023) & ~1023u;
    unsigned char *smem = smem_raw + (base - raw);
    const uint32_t s_a = base, s_b = base + STAGES2 * HALF_BYTES;
    unsigned char *s_stage = smem + STAGES2 * 2 * HALF_BYTES;
    uint16_t *s_list = reinterpret_cast<uint16_t *>(s_stage + EPI_WARPS * 32 * STG_PITCH);
    uint64_t *bars = reinterpret_cast<uint64_t *>(reinterpret_cast<unsigned char *>(s_list) + MAX_LIST * 2);
    const uint32_t bar0 = smem_u32(bars);
    auto full_bar = [&](int s) { return bar0 + s * 8; };
    auto empty_bar = [&](int s) { return bar0 + (STAGES2 + s) * 8; };
    auto acc_full = [&](int a) { return bar0 + (2 * STAGES2 + a) * 8; };
    auto acc_empty = [&](int a) { return bar0 + (2 * STAGES2 + 2 + a) * 8; };
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * STAGES2 + 4);
    int *s_scan = reinterpret_cast<int *>(tmem_slot + 2);       // [THREADS / 32 + 1] warp totals of the list scan

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int rank = (int)cluster_ctarank();
    const int cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES2; ++s) {
            mbar_init(full_bar(s), 1);       // leader's: its producer's arrive.expect_tx (bytes of both CTAs)
            mbar_init(empty_bar(s), 1);      // one multicast commit
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(acc_full(a), 1);
            mbar_init(acc_empty(a), 2 * EPI_WARPS);   // leader's: one arrive per epilogue warp of both CTAs
        }
        mbar_fence_init();
    }
    if (warp == 1) tmem_alloc_pair<TMEM_COLS>(smem_u32(tmem_slot));

    // mode 0: the list of (pair, sub) entries that exist.  sub 0 always; sub 1 only where the pair's second tile
    // belongs to another group.  Both CTAs build the same list.
    int n_units = n_units_mode1;
    if (p.mode == 0) {
        const int n_cand = 2 * ((p.tiles_m + 1) / 2);
        int base_cnt = 0;
        for (int c0 = 0; c0 < n_cand; c0 += THREADS) {
            const int c = c0 + threadIdx.x;
            const bool real = c < n_cand && unit_exists(p.tile_group, p.tiles_m, c);
            const uint32_t bal = __ballot_sync(0xffffffffu, real);
            if (lane == 0) s_scan[warp] = __popc(bal);
            __syncthreads();
            int before = base_cnt, total = base_cnt;
            for (int w = 0; w < THREADS / 32; ++w) {
                const int cnt = s_scan[w];
                if (w < warp) before += cnt;
                total += cnt;
            }
            if (real) s_list[before + __popc(bal & ((1u << lane) - 1))] = (uint16_t)c;
            base_cnt = total;
            __syncthreads();
        }
        n_units = base_cnt * p.tiles_n;
    }
    fence_before_sync();
    cluster_sync_all();          // barriers of both CTAs initialised, TMEM allocated, list visible
    fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===== TMA producer (both CTAs): own A rows + own half of B; bytes are counted on the leader's barrier =====
        if (lane == 0) {
            uint32_t it = 0;
            for (int u = cluster_id; u < n_units; u += n_clusters) {
                const Unit un = get_unit(p, u, s_list, rank);
                if (!un.mma) continue;
                const int a_k = un.g * p.a_k_off, b_k = un.g * p.b_k_off;
                for (int kb = 0; kb < un.n_kblk; ++kb, ++it) {
                    const int s = it % STAGES2;
                    mbar_wait(empty_bar(s), ((it / STAGES2) & 1) ^ 1);
                    if (rank == 0) mbar_expect_tx(full_bar(s), 4 * HALF_BYTES);
                    const int k0 = un.k_begin + kb * BK;
                    const uint32_t da = s_a + s * HALF_BYTES, db = s_b + s * HALF_BYTES;
                    if (p.a_mn_major) {
#pragma unroll
                        for (int h = 0; h < 2; ++h) tma_load_2d_pair(da + h * 8192, &map_a, full_bar(s), un.a_mn + 64 * h, a_k + k0);
                    } else {
                        tma_load_2d_pair(da, &map_a, full_bar(s), a_k + k0, un.a_mn);
                    }
                    if (p.b_mn_major) {
#pragma unroll
                        for (int h = 0; h < 2; ++h) tma_load_2d_pair(db + h * 8192, &map_b, full_bar(s), un.b_mn + 64 * h, b_k + k0);
                    } else {
                        tma_load_2d_pair(db, &map_b, full_bar(s), b_k + k0, un.b_mn);
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (rank == 0) {
            // ===== MMA issuer (leader only): M = 256 over both CTAs, N = 256, K = 16 per instruction =====
            const uint32_t idesc = (1u << 4) | ab_format_bits<T>() | ((uint32_t)p.a_mn_major << 15) |
                                   ((uint32_t)p.b_mn_major << 16) | ((uint32_t)(BN >> 3) << 17) |
                                   ((uint32_t)((2 * BM) >> 4) << 24);
            const uint64_t da0 = operand_desc(s_a, p.a_mn_major, 0), db0 = operand_desc(s_b, p.b_mn_major, 0);
            const uint64_t a_step = p.a_mn_major ? MNMAJOR_K16 : KMAJOR_K16, b_step = p.b_mn_major ? MNMAJOR_K16 : KMAJOR_K16;
            uint32_t it = 0, n_acc = 0;
            for (int u = cluster_id; u < n_units; u += n_clusters) {
                const Unit un = get_unit(p, u, s_list, rank);
                if (!un.mma) continue;
                const int acc = n_acc & 1;
                mbar_wait(acc_empty(acc), ((n_acc >> 1) & 1) ^ 1);   // both CTAs have drained this accumulator
                fence_after_sync();
                for (int kb = 0; kb < un.n_kblk; ++kb, ++it) {
                    const int s = it % STAGES2;
                    mbar_wait(full_bar(s), (it / STAGES2) & 1);
                    fence_after_sync();
                    if (elect_one()) {
                        const uint64_t da = da0 + (uint64_t)(s * (HALF_BYTES >> 4)), db = db0 + (uint64_t)(s * (HALF_BYTES >> 4));
#pragma unroll
                        for (int k = 0; k < BK / UMMA_K; ++k)
                            umma_bf16_pair(tmem_base + acc * BN, da + k * a_step, db + k * b_step, idesc, (kb | k) != 0);
                        umma_commit_pair(empty_bar(s), 0b11);         // frees the stage in both CTAs
                    }
                    __syncwarp();
                }
                if (elect_one()) umma_commit_pair(acc_full(acc), 0b11);
                __syncwarp();
                ++n_acc;
            }
        }
    } else {
        // ===== epilogue (both CTAs): as in the single-CTA kernel, over this CTA's 128 rows of the unit =====
        const int quarter = warp & 3, chalf = (warp - 2) >> 2;
        const int row_in_tile = quarter * 32 + lane;
        unsigned char *stage = s_stage + (warp - 2) * 32 * STG_PITCH;
        const bool out16 = p.c_dtype == c16_dtype<T>();
        const int esz = out16 ? 2 : 4;
        uint32_t n_acc = 0;
        for (int u = cluster_id; u < n_units; u += n_clusters) {
            const Unit un = get_unit(p, u, s_list, rank);
            const int n_valid = min(BN, p.N - un.n0);
            if (un.role == 2) {
                // tail tile beyond the bucketed rows: define its output (zeros)
                for (int i = threadIdx.x - 64; i < BM * n_valid; i += EPI_WARPS * 32) {
                    const long long off = (un.c_row0 + i / n_valid) * p.ldc + un.c_col0 + i % n_valid;
                    if (out16) reinterpret_cast<T *>(p.C)[off] = from_f32<T>(0.0f);
                    else reinterpret_cast<float *>(p.C)[off] = 0.0f;
                }
            }
            if (!un.mma) continue;
            const int acc = n_acc & 1;
            mbar_wait(acc_full(acc), (n_acc >> 1) & 1);
            fence_after_sync();
            if (un.role == 1 && un.rows_ok > 0) {
                const int rows_ok = un.rows_ok;
                const long long c_row = un.c_row0 + row_in_tile;
                const float rs = (p.row_scale && p.mode == 0) ? p.row_scale[c_row] : 1.0f;
                unsigned char *c_base = reinterpret_cast<unsigned char *>(p.C);
                const bool aligned = ((reinterpret_cast<uintptr_t>(p.C) + (size_t)un.c_col0 * esz) % 16 == 0) && ((p.ldc * esz) % 16 == 0);
#pragma unroll 1
                for (int c64 = chalf * (BN / 2); c64 < (chalf + 1) * (BN / 2); c64 += 64) {
                    if (c64 >= n_valid) break;
                    // one 64-column tcgen05.ld per step, processed as two 32-column halves through the staging tile
                    uint32_t r64[64];
                    __syncwarp();
                    tmem_ld64_nowait(tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * BN + c64, r64);
                    tmem_ld_wait();
#pragma unroll
                  for (int hh = 0; hh < 2; ++hh) {
                    const int c0 = c64 + 32 * hh;
                    if (c0 >= n_valid) break;
                    uint32_t r[32];
#pragma unroll
                    for (int i = 0; i < 32; ++i) r[i] = r64[32 * hh + i];
                    __syncwarp();          // the staging tile is reused: everyone has read the previous half
                    float v[32];
                    const bool full = c0 + 32 <= n_valid;
                    if (un.n_kblk == 0) {
#pragma unroll
                        for (int i = 0; i < 32; ++i) r[i] = 0;
                    }
                    if (p.bias) {
                        const float *bp = p.bias + (long long)un.g * p.bias_stride + un.n0 + c0;
#pragma unroll
                        for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]) + ((full || c0 + i < n_valid) ? __ldg(bp + i) : 0.0f);
                    } else {
#pragma unroll
                        for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
                    }
                    if (p.act == 1) {
#pragma unroll
                        for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.0f);
                    } else if (p.act == 2) {
#pragma unroll
                        for (int i = 0; i < 32; ++i) v[i] = v[i] / (1.0f + __expf(-v[i]));
                    }
#pragma unroll
                    for (int i = 0; i < 32; ++i) v[i] *= rs;
                    if (p.gate && row_in_tile < rows_ok) {
                        const T *gp = static_cast<const T *>(p.gate) + c_row * p.ldg + un.c_col0 + c0;
                        if (full && (reinterpret_cast<uintptr_t>(gp) % 16 == 0)) {
#pragma unroll
                            for (int i = 0; i < 32; i += 8) {
                                float gv[8];
                                Vec16<T>::load(gp + i, gv);
#pragma unroll
                                for (int q = 0; q < 8; ++q)
                                    if (!(gv[q] > 0.0f)) v[i + q] = 0.0f;
                            }
                        } else {
#pragma unroll
                            for (int i = 0; i < 32; ++i)
                                if (c0 + i < n_valid && !(to_f32(gp[i]) > 0.0f)) v[i] = 0.0f;
                        }
                    }
                    if (full && aligned) {
                        unsigned char *srow = stage + lane * STG_PITCH;
                        if (out16) {
#pragma unroll
                            for (int i = 0; i < 32; i += 8) {
                                float t8[8] = {v[i], v[i + 1], v[i + 2], v[i + 3], v[i + 4], v[i + 5], v[i + 6], v[i + 7]};
                                Vec16<T>::store(reinterpret_cast<T *>(srow) + i, t8);
                            }
                        } else {
#pragma unroll
                            for (int i = 0; i < 32; i += 4)
                                *reinterpret_cast<float4 *>(srow + i * 4) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
                        }
                        __syncwarp();
                        const int segs = out16 ? 4 : 8;
                        const int rows_per = 32 / segs;
                        const int seg = lane % segs, rsub = lane / segs;
                        for (int r0 = 0; r0 < 32; r0 += rows_per) {
                            const int rr = r0 + rsub;
                            if (quarter * 32 + rr < rows_ok) {
                                const uint4 val = *reinterpret_cast<const uint4 *>(stage + rr * STG_PITCH + seg * 16);
                                unsigned char *dst = c_base + ((un.c_row0 + quarter * 32 + rr) * p.ldc + un.c_col0 + c0) * esz + seg * 16;
                                *reinterpret_cast<uint4 *>(dst) = val;
                            }
                        }
                    } else if (row_in_tile < rows_ok) {
                        if (out16) {
                            T *dst = reinterpret_cast<T *>(p.C) + c_row * p.ldc + un.c_col0 + c0;
    #pragma unroll
                        for (int i = 0; i < 32; ++i)      // static indices: a run-time bound would put v[] in local memory
                            if (c0 + i < n_valid) dst[i] = from_f32<T>(v[i]);
                        } else {
                            float *dst = reinterpret_cast<float *>(p.C) + c_row * p.ldc + un.c_col0 + c0;
    #pragma unroll
                        for (int i = 0; i < 32; ++i)
                            if (c0 + i < n_valid) dst[i] = v[i];
                        }
                    }
                  }
                }
            }
            fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(acc_empty(acc), 0);   // 16 arrivals on the leader: accumulator may be overwritten
            ++n_acc;
        }
    }
    fence_before_sync();
    cluster_sync_all();          // nobody leaves (or frees TMEM) while the partner may still signal or be read
    if (warp == 1) tmem_dealloc_pair<TMEM_COLS>(tmem_base);
}

// ---- host: tensor maps ---------------------------------------------------------------------------
// 2-D 16-bit tensor map (bf16 or fp16): `inner` contiguous elements per row, `outer` rows of `ld` elements;
// box = (64, box_outer)
static int make_map(CUtensorMap *map, const void *base, uint64_t inner, uint64_t outer, uint64_t ld, uint32_t box_outer,
                    CUtensorMapDataType type) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return fail(SPT_ERR_CUDA, "grouped_gemm: cuTensorMapEncodeTiled entry point not available");
    cuuint64_t dims[2] = {inner, outer};
    cuuint64_t strides[1] = {ld * 2};
    cuuint32_t box[2] = {64, box_outer};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, type, 2, const_cast<void *>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(SPT_ERR_CUDA, "grouped_gemm: cuTensorMapEncodeTiled failed (%d)", (int)r);
    return SPT_OK;
}

template <typename T>
static int launch(const CUtensorMap &map_a, const CUtensorMap &map_b, const Params &p, int mode, int n_groups,
                  spt_stream_t stream) {
    static const bool use_pair = [] {
        const char *e = getenv("SPT_GEMM_CTA_PAIR");       // "0": keep the single-CTA kernel (A/B measurements)
        return !(e && e[0] == '0');
    }();
    if (use_pair && (mode == 1 || p.tiles_m <= MAX_LIST)) {
        const int pairs_m = (p.tiles_m + 1) / 2;
        const long long units_cap = (long long)p.tiles_n * (mode == 0 ? 2ll * pairs_m : (long long)pairs_m * n_groups);
        SPT_REQUIRE(units_cap < (1ll << 31), "grouped_gemm: too many tiles");
        const int n_units1 = mode == 1 ? (int)units_cap : 0;    // mode 0 counts its units on the device
        const int n_clusters = (int)std::min<long long>(mode == 1 ? units_cap : (long long)p.tiles_n * pairs_m, num_sms() / 2);
        // the attribute is per DEVICE and ext._on_device lets one process drive several GPUs: set it on every call
        // (cheap, and what attn_tc.cu / lookup.cu do) instead of caching a process-wide flag
        cudaFuncSetAttribute(grouped_gemm_pair_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM2_BYTES);
        grouped_gemm_pair_kernel<T><<<2 * n_clusters, THREADS, SMEM2_BYTES, as_stream(stream)>>>(map_a, map_b, p, n_units1);
        return after_launch("grouped_gemm_pair_kernel");
    }
    const int n_ctas = (int)std::min<long long>(p.n_tiles, num_sms());
    cudaFuncSetAttribute(grouped_gemm_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    grouped_gemm_kernel<T><<<n_ctas, THREADS, SMEM_BYTES, as_stream(stream)>>>(map_a, map_b, p);
    return after_launch("grouped_gemm_kernel");
}

}  // namespace gemm
}  // namespace spt

using namespace spt;

// See include/spt_b200.h.  A: rows x cols as stored (row-major, leading dim lda); for a K-major operand
// the stored matrix is [MN, K], for an MN-major operand it is [K, MN].
extern "C" int spt_grouped_gemm(int mode, const void *A, long long a_rows, long long a_cols, long long lda,
                                int a_mn_major, const void *B, long long b_rows, long long b_cols, long long ldb,
                                int b_mn_major, const int32_t *tile_group, int n_m_tiles,
                                const int32_t *group_ptr, int n_groups, int M, int N, int K, int a_k_off,
                                int a_mn_off, int b_k_off, int b_mn_off, long long c_row_off, long long c_col_off,
                                void *C, long long ldc, int c_dtype, const float *bias, int bias_stride,
                                const float *row_scale, int act, const void *gate, long long ldg, int ab_dtype,
                                spt_stream_t stream) {
    SPT_REQUIRE(A && B && C, "grouped_gemm: null pointer");
    SPT_REQUIRE(mode == 0 || mode == 1, "grouped_gemm: bad mode %d", mode);
    SPT_REQUIRE(mode == 1 || (tile_group && n_m_tiles >= 1 && K >= 1 && !a_mn_major),
                "grouped_gemm: mode 0 needs tile_group, K and a K-major A");
    SPT_REQUIRE(mode == 0 || (group_ptr && n_groups >= 1 && M >= 1), "grouped_gemm: mode 1 needs group_ptr and M");
    SPT_REQUIRE(N >= 1, "grouped_gemm: bad N");
    SPT_REQUIRE(lda % 8 == 0 && ldb % 8 == 0 && ((uintptr_t)A % 16 == 0) && ((uintptr_t)B % 16 == 0),
                "grouped_gemm: operands must be 16-byte aligned with leading dims multiple of 8");
    SPT_REQUIRE(ab_dtype == SPT_BF16 || ab_dtype == SPT_F16,
                "grouped_gemm: ab_dtype %d unknown: the operands A and B are SPT_BF16 (1) or SPT_F16 (2)", ab_dtype);
    SPT_REQUIRE(c_dtype == SPT_F32 || c_dtype == ab_dtype,
                "grouped_gemm: c_dtype %d not allowed: C is SPT_F32 (0) or the operand type ab_dtype (%d)", c_dtype, ab_dtype);
    const CUtensorMapDataType map_type = ab_dtype == SPT_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    CUtensorMap map_a, map_b;
    int rc = gemm::make_map(&map_a, A, (uint64_t)a_cols, (uint64_t)a_rows, (uint64_t)lda, a_mn_major ? 64 : 128, map_type);
    if (rc != SPT_OK) return rc;
    rc = gemm::make_map(&map_b, B, (uint64_t)b_cols, (uint64_t)b_rows, (uint64_t)ldb, b_mn_major ? 64 : 128, map_type);
    if (rc != SPT_OK) return rc;
    gemm::Params p;
    p.mode = mode; p.tile_group = tile_group; p.group_ptr = group_ptr; p.K = K; p.M = M; p.N = N;
    p.a_mn_major = a_mn_major; p.b_mn_major = b_mn_major;
    p.a_k_off = a_k_off; p.a_mn_off = a_mn_off; p.b_k_off = b_k_off; p.b_mn_off = b_mn_off;
    p.c_row_off = c_row_off; p.c_col_off = c_col_off; p.C = C; p.ldc = ldc; p.c_dtype = c_dtype;
    p.bias = bias; p.bias_stride = bias_stride; p.row_scale = row_scale; p.act = act;
    p.gate = gate; p.ldg = ldg;
    SPT_REQUIRE(!gate || mode == 0, "grouped_gemm: gate is a mode-0 epilogue");
    p.tiles_n = (N + gemm::BN - 1) / gemm::BN;
    p.tiles_m = mode == 0 ? n_m_tiles : (M + gemm::BM - 1) / gemm::BM;
    const long long n_tiles = (long long)p.tiles_n * p.tiles_m * (mode == 0 ? 1 : n_groups);
    SPT_REQUIRE(n_tiles < (1ll << 31), "grouped_gemm: too many tiles");
    p.n_tiles = (int)n_tiles;
    return ab_dtype == SPT_F16 ? gemm::launch<__half>(map_a, map_b, p, mode, n_groups, stream)
                               : gemm::launch<__nv_bfloat16>(map_a, map_b, p, mode, n_groups, stream);
}

extern "C" int spt_grouped_gemm_bf16(int mode, const void *A, long long a_rows, long long a_cols, long long lda,
                                     int a_mn_major, const void *B, long long b_rows, long long b_cols, long long ldb,
                                     int b_mn_major, const int32_t *tile_group, int n_m_tiles,
                                     const int32_t *group_ptr, int n_groups, int M, int N, int K, int a_k_off,
                                     int a_mn_off, int b_k_off, int b_mn_off, long long c_row_off, long long c_col_off,
                                     void *C, long long ldc, int c_dtype, const float *bias, int bias_stride,
                                     const float *row_scale, int act, const void *gate, long long ldg,
                                     spt_stream_t stream) {
    return spt_grouped_gemm(mode, A, a_rows, a_cols, lda, a_mn_major, B, b_rows, b_cols, ldb, b_mn_major, tile_group,
                            n_m_tiles, group_ptr, n_groups, M, N, K, a_k_off, a_mn_off, b_k_off, b_mn_off, c_row_off,
                            c_col_off, C, ldc, c_dtype, bias, bias_stride, row_scale, act, gate, ldg, SPT_BF16, stream);
}

// Host-side replay of the CTA-pair kernel's mode-0 schedule (same unit_exists / get_unit code as the device), for
// tests without a GPU.  tile_group is a HOST array.  Writes one record of 6 ints per (unit, CTA rank):
//   unit, rank, group, m_tile, n_tile, role | mma << 4      (role: 0 idle, 1 active, 2 zero-fill)
// and returns the number of records (nothing is written beyond `cap` records), or a negative spt_status.
extern "C" int spt_grouped_gemm_plan(const int32_t *tile_group, int n_m_tiles, int tiles_n, int32_t *out, int cap) {
    if (!tile_group || n_m_tiles < 1 || n_m_tiles > gemm::MAX_LIST || tiles_n < 1 || (!out && cap > 0)) {
        fail(SPT_ERR_INVALID_ARGUMENT, "grouped_gemm_plan: bad arguments");
        return -SPT_ERR_INVALID_ARGUMENT;
    }
    gemm::Params p{};
    p.mode = 0; p.tile_group = tile_group; p.tiles_m = n_m_tiles; p.tiles_n = tiles_n; p.K = gemm::BK;
    uint16_t list[gemm::MAX_LIST];
    int n_list = 0;
    const int n_cand = 2 * ((n_m_tiles + 1) / 2);
    for (int c = 0; c < n_cand; ++c)
        if (gemm::unit_exists(tile_group, n_m_tiles, c)) list[n_list++] = (uint16_t)c;
    int n = 0;
    for (int u = 0; u < n_list * tiles_n; ++u)
        for (int rank = 0; rank < 2; ++rank, ++n) {
            if (n >= cap) continue;
            const gemm::Unit un = gemm::get_unit(p, u, list, rank);
            int32_t *r = out + 6 * (size_t)n;
            r[0] = u; r[1] = rank; r[2] = un.g; r[3] = (int)(un.c_row0 / gemm::BM); r[4] = un.n0 / gemm::BN;
            r[5] = un.role | ((int)un.mma << 4);
        }
    return n;
}
