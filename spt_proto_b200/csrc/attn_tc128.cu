// Backward of the fused PQ-sparse attention on 128 x 128 score tiles, ONE persistent CTA per SM (head dim 64).
//
// Same mathematics, mask format and C ABI as attn_tc.cu (see its header); what changes is the shape of the work:
//   * every tcgen05.mma is M128 x N128 (score products, operands in shared memory: 64 clk = the tensor pipe's peak) or
//     M128 x N64 with the probability tile as a TMEM A-operand (32 clk = peak).  The 128 x 64 kernels issue N = 32 / 64
//     score MMAs whose cost is the shared-memory read of the 128-row A tile (40 - 48 clk whatever N; micro-benchmark
//     scratch/mb/umma_rate2.cu), i.e. a tensor pipe at 1/3 - 1/2 of its rate;
//   * 16 math warps (thread = TMEM lane x 32 score columns) take their scores into registers and release the score
//     columns at once, so the tensor core computes the next tile's scores under this tile's exp / mask math; the
//     bf16 probability / dS tiles have TMEM columns of their own;
//   * the CTA is persistent: it walks a static list of (owner tile, head) items, heaviest first; the producer warp
//     prefetches the next item's owner tiles and the score MMAs of its first tile run under the epilogue of the
//     previous item (with one CTA per SM nothing else would hide the prologue / epilogue).
// 576 threads: warps 0-15 math, 16 TMA / row-data producer, 17 TMEM allocator + MMA issuer.
#include "attn_common.cuh"

namespace spt {
namespace attn_tc128 {

using namespace tc;
using namespace attn_tc;

constexpr int T = 128;                       // tile edge: owner rows (= TMEM lanes) and other rows per iteration
constexpr int MATH_WARPS = 16;
constexpr int THREADS = (MATH_WARPS + 2) * 32;
constexpr int W_TMA = MATH_WARPS, W_MMA = MATH_WARPS + 1;
constexpr int D = 64;
constexpr int TILE = T * D * 2;              // 16 KB: one 128 x 64 bf16 operand tile
constexpr int ST = 3;                        // pipeline stages of the "other" tiles

// Static schedule: items are ordered heaviest first; round w hands items [w G, (w + 1) G) to the G CTAs, in reversed CTA
// order on odd rounds so that no CTA collects the heaviest item of every round (backward 0.393 -> 0.380 ms against plain
// round-robin).  -1 = done.
__device__ __forceinline__ int sched_item(int round, int n_items) {
    const int G = gridDim.x;
    const int item = round * G + ((round & 1) ? G - 1 - (int)blockIdx.x : (int)blockIdx.x);
    return item < n_items ? item : -1;
}

// elected arrive of a whole warp whose lanes have all executed the tcgen05 operation being signalled
__device__ __forceinline__ void warp_arrive(uint32_t bar, int lane) {
    fence_before_sync();
    __syncwarp();
    if (lane == 0) mbar_arrive(bar);
}


// ---------------------------------------------------------------------------------------------------------------------
// Backward, dK / dV.  Owner = 128 keys (K, V; one lane-major mask group), loop over the 128-row query tiles at and below
// the diagonal.  S^T = K Q_j^T and dP'^T = V dO'_j^T (keys on the TMEM lanes), E^T / dS^T written as bf16 A-operands,
//   dV += E^T dO'_j,  dK += dS^T Q_j.
// TMEM columns: S^T 0, dP'^T 128, E^T 256, dS^T 320, dV 384, dK 448.
// Per-row data of the 128 query rows of a stage: this key group's mask words transposed ([4][128 + 4]) by the producer
// lanes, -delta' and extra0 by 1-D bulk copies.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int MT = T + 4;                              // padded row of the transposed mask: the 4 words hit distinct banks
constexpr int ROWQ = MT * 16 + T * 4 + T * 4;          // bytes per stage
constexpr int KV_SMEM = 4 * TILE + 2 * ST * TILE + ST * ROWQ + 256 + 1024;
// fp16 adds the rows' -o (row scale, from zsum) to every stage: T * 4 bytes after extra0
template <typename E>
constexpr int rowq_bytes = ROWQ + (is_f16<E> ? T * 4 : 0);
template <typename E>
constexpr int kv_smem = KV_SMEM + ST * (rowq_bytes<E> - ROWQ);

// E: element type (__nv_bfloat16 or __half); zsum is read by the fp16 instantiation only
template <typename E>
__global__ void __launch_bounds__(THREADS, 1)
attn_bwd_kv128_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                      const __grid_constant__ CUtensorMap map_v, const __grid_constant__ CUtensorMap map_dys,
                      const uint32_t *__restrict__ mask, const int32_t *__restrict__ extra0,
                      const float *__restrict__ ndelta, E *__restrict__ dk, E *__restrict__ dv,
                      int S, int H, int B, float scale, float scale_log2, float clamp_log2, const float *__restrict__ zsum,
                      int G) {
    constexpr int ROWQ = rowq_bytes<E>;
    extern __shared__ unsigned char smem_raw[];
    const Smem sm = align_smem(smem_raw);
    const uint32_t s_k = sm.base, s_v = s_k + 2 * TILE, s_q = s_v + 2 * TILE, s_dy = s_q + ST * TILE;
    unsigned char *rowq = sm.ptr + 4 * TILE + 2 * ST * TILE;
    uint64_t *bars = reinterpret_cast<uint64_t *>(rowq + ST * ROWQ);
    const uint32_t bar0 = smem_u32(bars);
    auto own_full = [&](int i) { return bar0 + i * 8; };
    auto own_empty = [&](int i) { return bar0 + 16 + i * 8; };
    auto qd_full = [&](int s) { return bar0 + 32 + s * 8; };
    auto qd_empty = [&](int s) { return bar0 + 32 + (ST + s) * 8; };
    const uint32_t sc_full = bar0 + 32 + 2 * ST * 8, s_read = sc_full + 8, p_full = sc_full + 16, e_free = sc_full + 24,
                   acc_full = sc_full + 32, acc_empty = sc_full + 40;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 4 + 2 * ST + 6);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_own = S / T;
    const int n_items = n_own * B;
    const int words = S / 32;

    if (threadIdx.x == 0) {
        for (int i = 0; i < 2; ++i) {
            mbar_init(own_full(i), 1);
            mbar_init(own_empty(i), 1);
        }
        for (int s = 0; s < ST; ++s) {
            mbar_init(qd_full(s), 2);                  // expect_tx arrive + the producer warp's row data
            mbar_init(qd_empty(s), 1);
        }
        mbar_init(sc_full, 1);
        mbar_init(s_read, MATH_WARPS);
        mbar_init(p_full, MATH_WARPS);
        mbar_init(e_free, 1);
        mbar_init(acc_full, 1);
        mbar_init(acc_empty, MATH_WARPS);
        mbar_fence_init();
    }
    if (warp == W_MMA) tmem_alloc<512>(smem_u32(tmem_slot));
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    constexpr uint32_t COL_S = 0, COL_DP = 128, COL_E = 256, COL_DS = 320, COL_DV = 384, COL_DK = 448;

    if (warp == W_TMA) {
        // ===== producer: owner tiles of the next item, query-side tiles + row data of every stage =====
        int g = 0, w = 0;
        for (int item; (item = sched_item(w, n_items)) >= 0; ++w) {
            const int kt = item / B, b = item % B;     // key tile 0 is the heaviest: items are ordered by key tile
            const int hn = b / H, hh = b % H, n0 = kt * T, n_tiles = n_own - kt;
            const int hk = hh / G;                     // key / value head of query head hh (G > 1: grouped-query attention)
            const size_t head = (size_t)b * S;
            const int buf = w & 1;
            if (lane == 0) {
                mbar_wait(own_empty(buf), ((w >> 1) & 1) ^ 1);
                mbar_expect_tx(own_full(buf), 2 * TILE);
                tma_owner<D>(s_k + buf * TILE, &map_k, own_full(buf), hk, n0, hn);
                tma_owner<D>(s_v + buf * TILE, &map_v, own_full(buf), hk, n0, hn);
            }
            uint4 mw[4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                mw[u] = __ldg(reinterpret_cast<const uint4 *>(mask + (head + n0 + lane + 32 * u) * words) + kt);
            for (int j = 0; j < n_tiles; ++j, ++g) {
                const int st = g % ST;
                const int r0 = (kt + j) * T;
                unsigned char *slot = rowq + st * ROWQ;
                mbar_wait(qd_empty(st), ((g / ST) & 1) ^ 1);
                if (lane == 0) {
                    mbar_expect_tx(qd_full(st), 2 * TILE + 2 * T * 4);
                    tma_owner<D>(s_q + st * TILE, &map_q, qd_full(st), hh, r0, hn);
                    tma_owner<D>(s_dy + st * TILE, &map_dys, qd_full(st), hh, r0, hn);
                    bulk_load_1d(smem_u32(slot + MT * 16), ndelta + head + r0, T * 4, qd_full(st));
                    bulk_load_1d(smem_u32(slot + MT * 16 + T * 4), extra0 + head + r0, T * 4, qd_full(st));
                }
                uint32_t *mt = reinterpret_cast<uint32_t *>(slot);        // transposed: [word t][row], rows padded to MT
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int rr = lane + 32 * u;
                    mt[rr] = mw[u].x;
                    mt[MT + rr] = mw[u].y;
                    mt[2 * MT + rr] = mw[u].z;
                    mt[3 * MT + rr] = mw[u].w;
                    if constexpr (is_f16<E>) reinterpret_cast<float *>(slot + MT * 16 + 2 * T * 4)[rr] = f16_bwd_nofs(zsum[head + r0 + rr]);
                }
                if (j + 1 < n_tiles) {                                    // the next tile's words travel under this wait
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        mw[u] = __ldg(reinterpret_cast<const uint4 *>(mask + (head + r0 + T + lane + 32 * u) * words) + kt);
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(qd_full(st));
            }
        }
    } else if (warp == W_MMA) {
        // ===== MMA issuer (warp-uniform loop, one elected lane) =====
        constexpr uint32_t id_s = idesc_of<E>(T, T, 0, 0);     // S^T = K Q^T, dP'^T = V dO'^T
        constexpr uint32_t id_a = idesc_of<E>(T, D, 0, 1);     // dV += E^T dO', dK += dS^T Q   (A in TMEM, B MN-major)
        const uint64_t dk0 = desc_kmajor(s_k, 0), dv0 = desc_kmajor(s_v, 0), dq0 = desc_kmajor(s_q, 0),
                       ddy0 = desc_kmajor(s_dy, 0), dqt0 = desc_mnmajor(s_q, 0, TILE), ddyt0 = desc_mnmajor(s_dy, 0, TILE);
        int g = 0, w = 0;
        PROF(Prof pf; pf.start(); const long long t0 = pf.last;)
        for (int item; (item = sched_item(w, n_items)) >= 0; ++w) {
            const int kt = item / B, n_tiles = n_own - kt;
            const int buf = w & 1;
            const uint64_t own_off = (uint64_t)((buf * TILE) >> 4);
            auto issue_scores = [&](int gg) {                  // tile with running index gg (of this item)
                const int st = gg % ST;
                mbar_wait(qd_full(st), (gg / ST) & 1);
                if (gg > 0) mbar_wait(s_read, (gg - 1) & 1);   // the previous tile's scores are in registers
                fence_after_sync();
                if (elect_one()) {
                    const uint64_t off = (uint64_t)((st * TILE) >> 4);
#pragma unroll
                    for (int k = 0; k < D / 16; ++k) {         // two independent accumulators, k-steps alternate
                        umma_bf16(tmem_base + COL_S, dk0 + own_off + k * KMAJOR_K16, dq0 + off + k * KMAJOR_K16, id_s, k != 0);
                        umma_bf16(tmem_base + COL_DP, dv0 + own_off + k * KMAJOR_K16, ddy0 + off + k * KMAJOR_K16, id_s, k != 0);
                    }
                    umma_commit(sc_full);
                }
                __syncwarp();
            };
            mbar_wait(own_full(buf), (w >> 1) & 1);
            issue_scores(g);
            for (int j = 0; j < n_tiles; ++j, ++g) {
                PROF(pf.lap(2);)
                if (j + 1 < n_tiles) issue_scores(g + 1);
                PROF(pf.lap(0);)
                const int st = g % ST;
                mbar_wait(p_full, g & 1);
                if (j == 0 && w > 0) mbar_wait(acc_empty, (w - 1) & 1);     // the previous item's dV / dK have been read
                PROF(pf.lap(1);)
                fence_after_sync();
                if (elect_one()) {
                    const uint64_t off = (uint64_t)((st * TILE) >> 4);
#pragma unroll
                    for (int k = 0; k < T / 16; ++k) {         // query rows 16 k .. 16 k + 15 = columns 8 k .. 8 k + 7 of E^T / dS^T
                        umma_bf16_ts(tmem_base + COL_DV, tmem_base + COL_E + k * 8, ddyt0 + off + k * MNMAJOR_K16, id_a, (j | k) != 0);
                        umma_bf16_ts(tmem_base + COL_DK, tmem_base + COL_DS + k * 8, dqt0 + off + k * MNMAJOR_K16, id_a, (j | k) != 0);
                    }
                    umma_commit(qd_empty(st));
                    umma_commit(e_free);
                    if (j + 1 == n_tiles) {
                        umma_commit(acc_full);
                        umma_commit(own_empty(buf));
                    }
                }
                __syncwarp();
            }
        }
        PROF(pf.t[3] = clock64() - t0; pf.t[4] = g; pf.flush(2, 8, lane == 0);)
    } else {
        // ===== math warps: thread = (key = TMEM lane, 32 query columns) =====
        const int quarter = warp & 3, cg = warp >> 2;
        const int kk = quarter * 32 + lane;
        const int wsel = kk & 3;
        const int shl = 31 - (kk >> 2);                 // moves this key's bit of a lane-major word to the sign bit
        const MathK mk = make_math(scale_log2, clamp_log2);
        const uint32_t lane_base = tmem_base + ((uint32_t)(quarter * 32) << 16);
        const int c0 = cg * 32;                         // query rows c0 .. c0 + 31 of every tile
        int g = 0, w = 0;
        PROF(Prof pf; pf.start(); const long long t0 = pf.last;)
        for (int item; (item = sched_item(w, n_items)) >= 0; ++w) {
            const int kt = item / B, b = item % B;
            const int hn = b / H, hh = b % H, n0 = kt * T, n_tiles = n_own - kt;
            const bool key0 = (n0 + kk) == 0;
            for (int j = 0; j < n_tiles; ++j, ++g) {
                const int st = g % ST;
                const unsigned char *slot = rowq + st * ROWQ;
                const uint32_t *mrow = reinterpret_cast<const uint32_t *>(slot) + wsel * MT;   // this key's word of every row
                const float *s_nd = reinterpret_cast<const float *>(slot + MT * 16);
                const int32_t *s_ex0 = reinterpret_cast<const int32_t *>(slot + MT * 16 + T * 4);
                const float *s_nofs = reinterpret_cast<const float *>(slot + MT * 16 + 2 * T * 4);
                mbar_wait(qd_full(st), (g / ST) & 1);
                mbar_wait(sc_full, g & 1);
                PROF(pf.lap(0);)
                fence_after_sync();
                uint32_t r[32], gr[32];
                tmem_ld32_nowait(lane_base + COL_S + c0, r);
                tmem_ld32_nowait(lane_base + COL_DP + c0, gr);
                tmem_ld_wait();
                warp_arrive(s_read, lane);
                PROF(pf.lap(1);)
                const bool clamp = warp_needs_clamp(r, mk.thr);
                // key 0 carries the rows' zero-padding multiplicity: the (slow, divergent) variant only runs for tiles whose
                // rows have any padding — the first rows of a sequence, and the rare rows a bucket overflow left short
                bool pad = false;
                if (key0) {
#pragma unroll
                    for (int i = 0; i < 32; i += 4) {
                        const int4 e4 = *reinterpret_cast<const int4 *>(s_ex0 + c0 + i);
                        pad |= (e4.x | e4.y | e4.z | e4.w) != 0;
                    }
                }
                uint32_t pe0[8], pd0[8], pe1[8], pd1[8];
#define SPT_KV_HALF(OFF, PE, PD)                                                                                           \
                if (pad) {                                                                                                \
                    if (clamp) bwdkv_chunk16<true, true, OFF, 32, int32_t, E>(r, gr, mrow, s_nd, s_ex0, c0 + OFF, shl, mk, PE, PD, s_nofs);  \
                    else bwdkv_chunk16<true, false, OFF, 32, int32_t, E>(r, gr, mrow, s_nd, s_ex0, c0 + OFF, shl, mk, PE, PD, s_nofs);       \
                } else {                                                                                                   \
                    if (clamp) bwdkv_chunk16<false, true, OFF, 32, int32_t, E>(r, gr, mrow, s_nd, s_ex0, c0 + OFF, shl, mk, PE, PD, s_nofs); \
                    else bwdkv_chunk16<false, false, OFF, 32, int32_t, E>(r, gr, mrow, s_nd, s_ex0, c0 + OFF, shl, mk, PE, PD, s_nofs);      \
                }
                SPT_KV_HALF(0, pe0, pd0)
                SPT_KV_HALF(16, pe1, pd1)
#undef SPT_KV_HALF
                PROF(pf.lap(2);)
                if (g > 0) {                            // E^T / dS^T of the previous tile have been consumed
                    mbar_wait(e_free, (g - 1) & 1);
                    fence_after_sync();
                }
                tmem_st8(lane_base + COL_E + c0 / 2, pe0);
                tmem_st8(lane_base + COL_E + c0 / 2 + 8, pe1);
                tmem_st8(lane_base + COL_DS + c0 / 2, pd0);
                tmem_st8(lane_base + COL_DS + c0 / 2 + 8, pd1);
                tmem_st_wait();
                warp_arrive(p_full, lane);
                PROF(pf.lap(3);)
            }
            // epilogue: column group 0, 1 -> dV halves, 2, 3 -> dK halves (dK follows dV in TMEM)
            mbar_wait(acc_full, w & 1);
            fence_after_sync();
            {
                uint32_t o[32];
                tmem_ld32(lane_base + COL_DV + c0, o);
                warp_arrive(acc_empty, lane);
                const size_t off = (((size_t)hn * S + n0 + kk) * H + hh) * D + (cg & 1) * 32;
                store_row32((cg < 2 ? dv : dk) + off, o, cg < 2 ? 1.0f : scale);
            }
            PROF(pf.lap(5);)
        }
        PROF(pf.t[6] = clock64() - t0; pf.t[4] = g; pf.flush(2, 0, threadIdx.x == 0);)
    }
    fence_before_sync();
    __syncthreads();
    if (warp == W_MMA) tmem_dealloc<512>(tmem_base);
}

template <typename E>
int launch_bwd_kv128(const CUtensorMap &mq, const CUtensorMap &mk, const CUtensorMap &mv, const CUtensorMap &md,
                     const uint32_t *mask, const int32_t *extra0, const float *ndelta, const float *zsum, E *gk, E *gv,
                     int B, int S, int H, int G, float scale, float clamp, cudaStream_t st) {
    cudaFuncSetAttribute(attn_bwd_kv128_kernel<E>, cudaFuncAttributeMaxDynamicSharedMemorySize, kv_smem<E>);
    const int n_items = (S / T) * B;
    const int grid = n_items < num_sms() ? n_items : num_sms();
    attn_bwd_kv128_kernel<E><<<grid, THREADS, kv_smem<E>, st>>>(mq, mk, mv, md, mask, extra0, ndelta, gk, gv, S, H, B, scale,
                                                              scale * LOG2E, clamp * LOG2E, zsum, G);
    return after_launch("attn_bwd_kv128_kernel");
}
template int launch_bwd_kv128<__nv_bfloat16>(const CUtensorMap &, const CUtensorMap &, const CUtensorMap &,
                                             const CUtensorMap &, const uint32_t *, const int32_t *, const float *,
                                             const float *, __nv_bfloat16 *, __nv_bfloat16 *, int, int, int, int, float,
                                             float, cudaStream_t);
template int launch_bwd_kv128<__half>(const CUtensorMap &, const CUtensorMap &, const CUtensorMap &, const CUtensorMap &,
                                      const uint32_t *, const int32_t *, const float *, const float *, __half *, __half *,
                                      int, int, int, int, float, float, cudaStream_t);


// 16 fp32 accumulator values (scaled) -> 16 bf16 / fp16 = 32 contiguous bytes
template <typename E>
__device__ __forceinline__ void store_row16(E *dst, const uint32_t (&r)[16], float s) {
#pragma unroll
    for (int i = 0; i < 16; i += 8) {
        float t[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) t[u] = __uint_as_float(r[i + u]) * s;
        Vec16<E>::store(dst + i, t);
    }
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    tmem_ld16_nowait(taddr, r);
    tmem_ld_wait();
}

// ---------------------------------------------------------------------------------------------------------------------
// Backward, dQ.  Owner = 128 query rows (Q, dO'), loop over the 128-key tiles 0 .. diagonal (K_j, V_j).
//   S = Q K_j^T,  dP' = dO' V_j^T,  dS = e (dP' - delta') as a bf16 TMEM A-operand,  dQ += dS K_j.
// TMEM columns: S 0, dP' 128, dS[2] 256 / 320, dQ 384.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int Q_SMEM = 4 * TILE + 2 * ST * TILE + 256 + 1024;

// E: element type; zsum is read by the fp16 instantiation only (row scales)
template <typename E>
__global__ void __launch_bounds__(THREADS, 1)
attn_bwd_q128_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                     const __grid_constant__ CUtensorMap map_v, const __grid_constant__ CUtensorMap map_dys,
                     const uint32_t *__restrict__ mask, const int32_t *__restrict__ extra0,
                     const float *__restrict__ ndelta, E *__restrict__ dq, int S, int H, int B, float scale,
                     float scale_log2, float clamp_log2, const float *__restrict__ zsum, int G) {
    extern __shared__ unsigned char smem_raw[];
    const Smem sm = align_smem(smem_raw);
    const uint32_t s_q = sm.base, s_dy = s_q + 2 * TILE, s_k = s_dy + 2 * TILE, s_v = s_k + ST * TILE;
    uint64_t *bars = reinterpret_cast<uint64_t *>(sm.ptr + 4 * TILE + 2 * ST * TILE);
    const uint32_t bar0 = smem_u32(bars);
    auto own_full = [&](int i) { return bar0 + i * 8; };
    auto own_empty = [&](int i) { return bar0 + 16 + i * 8; };
    auto kv_full = [&](int s) { return bar0 + 32 + s * 8; };
    auto kv_empty = [&](int s) { return bar0 + 32 + (ST + s) * 8; };
    const uint32_t sc_full = bar0 + 32 + 2 * ST * 8, s_read = sc_full + 8, acc_full = sc_full + 16, acc_empty = sc_full + 24;
    auto p_full = [&](int i) { return sc_full + 32 + i * 8; };
    auto e_free = [&](int i) { return sc_full + 48 + i * 8; };
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 4 + 2 * ST + 8);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_own = S / T;
    const int n_items = n_own * B;

    if (threadIdx.x == 0) {
        for (int i = 0; i < 2; ++i) {
            mbar_init(own_full(i), 1);
            mbar_init(own_empty(i), 1);
            mbar_init(p_full(i), MATH_WARPS);
            mbar_init(e_free(i), 1);
        }
        for (int s = 0; s < ST; ++s) {
            mbar_init(kv_full(s), 1);
            mbar_init(kv_empty(s), 1);
        }
        mbar_init(sc_full, 1);
        mbar_init(s_read, MATH_WARPS);
        mbar_init(acc_full, 1);
        mbar_init(acc_empty, MATH_WARPS);
        mbar_fence_init();
    }
    if (warp == W_MMA) tmem_alloc<512>(smem_u32(tmem_slot));
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    constexpr uint32_t COL_S = 0, COL_DP = 128, COL_DS = 256, COL_DQ = 384;

    if (warp == W_TMA) {
        if (lane == 0) {
            int g = 0, w = 0;
            for (int item; (item = sched_item(w, n_items)) >= 0; ++w) {
                const int qt = n_own - 1 - item / B, b = item % B;       // the last query tile sees the most keys
                const int hn = b / H, hh = b % H, hk = hh / G, n_tiles = qt + 1;
                const int buf = w & 1;
                mbar_wait(own_empty(buf), ((w >> 1) & 1) ^ 1);
                mbar_expect_tx(own_full(buf), 2 * TILE);
                tma_owner<D>(s_q + buf * TILE, &map_q, own_full(buf), hh, qt * T, hn);
                tma_owner<D>(s_dy + buf * TILE, &map_dys, own_full(buf), hh, qt * T, hn);
                for (int j = 0; j < n_tiles; ++j, ++g) {
                    const int st = g % ST;
                    mbar_wait(kv_empty(st), ((g / ST) & 1) ^ 1);
                    mbar_expect_tx(kv_full(st), 2 * TILE);
                    tma_owner<D>(s_k + st * TILE, &map_k, kv_full(st), hk, j * T, hn);
                    tma_owner<D>(s_v + st * TILE, &map_v, kv_full(st), hk, j * T, hn);
                }
            }
        }
    } else if (warp == W_MMA) {
        constexpr uint32_t id_s = idesc_of<E>(T, T, 0, 0);     // S = Q K^T, dP' = dO' V^T
        constexpr uint32_t id_a = idesc_of<E>(T, D, 0, 1);     // dQ += dS K   (A in TMEM, K MN-major)
        const uint64_t dq0 = desc_kmajor(s_q, 0), ddy0 = desc_kmajor(s_dy, 0), dk0 = desc_kmajor(s_k, 0),
                       dv0 = desc_kmajor(s_v, 0), dkt0 = desc_mnmajor(s_k, 0, TILE);
        int g = 0, w = 0;
        PROF(Prof pf; pf.start(); const long long t0 = pf.last;)
        for (int item; (item = sched_item(w, n_items)) >= 0; ++w) {
            const int n_tiles = n_own - item / B;
            const int buf = w & 1;
            const uint64_t own_off = (uint64_t)((buf * TILE) >> 4);
            auto issue_scores = [&](int gg) {
                const int st = gg % ST;
                mbar_wait(kv_full(st), (gg / ST) & 1);
                if (gg > 0) mbar_wait(s_read, (gg - 1) & 1);
                fence_after_sync();
                if (elect_one()) {
                    const uint64_t off = (uint64_t)((st * TILE) >> 4);
#pragma unroll
                    for (int k = 0; k < D / 16; ++k) {
                        umma_bf16(tmem_base + COL_S, dq0 + own_off + k * KMAJOR_K16, dk0 + off + k * KMAJOR_K16, id_s, k != 0);
                        umma_bf16(tmem_base + COL_DP, ddy0 + own_off + k * KMAJOR_K16, dv0 + off + k * KMAJOR_K16, id_s, k != 0);
                    }
                    umma_commit(sc_full);
                }
                __syncwarp();
            };
            mbar_wait(own_full(buf), (w >> 1) & 1);
            issue_scores(g);
            for (int j = 0; j < n_tiles; ++j, ++g) {
                PROF(pf.lap(2);)
                if (j + 1 < n_tiles) issue_scores(g + 1);
                PROF(pf.lap(0);)
                const int st = g % ST;
                mbar_wait(p_full(g & 1), (g >> 1) & 1);
                if (j == 0 && w > 0) mbar_wait(acc_empty, (w - 1) & 1);
                PROF(pf.lap(1);)
                fence_after_sync();
                if (elect_one()) {
                    const uint64_t off = (uint64_t)((st * TILE) >> 4);
#pragma unroll
                    for (int k = 0; k < T / 16; ++k)
                        umma_bf16_ts(tmem_base + COL_DQ, tmem_base + COL_DS + (g & 1) * 64 + k * 8, dkt0 + off + k * MNMAJOR_K16, id_a,
                                     (j | k) != 0);
                    umma_commit(kv_empty(st));
                    umma_commit(e_free(g & 1));
                    if (j + 1 == n_tiles) {
                        umma_commit(acc_full);
                        umma_commit(own_empty(buf));
                    }
                }
                __syncwarp();
            }
        }
        PROF(pf.t[3] = clock64() - t0; pf.t[4] = g; pf.flush(1, 8, lane == 0);)
    } else {
        // ===== math warps: thread = (query row = TMEM lane, 32 key columns) =====
        const int quarter = warp & 3, cg = warp >> 2;
        const int rt = quarter * 32 + lane;
        const MathK mk = make_math(scale_log2, clamp_log2);
        const uint32_t lane_base = tmem_base + ((uint32_t)(quarter * 32) << 16);
        int g = 0, w = 0;
        PROF(Prof pf; pf.start(); const long long t0 = pf.last;)
        for (int item; (item = sched_item(w, n_items)) >= 0; ++w) {
            const int qt = n_own - 1 - item / B, b = item % B;
            const int hn = b / H, hh = b % H, n_tiles = qt + 1;
            const int row = qt * T + rt;
            const size_t grow = (size_t)b * S + row;
            const uint4 *mrow = reinterpret_cast<const uint4 *>(mask + grow * (S / 32));
            const float ex0 = (float)extra0[grow];
            const float nd = ndelta[grow];
            const float nofs = is_f16<E> ? f16_bwd_nofs(zsum[grow]) : 0.0f;
            uint4 mw = __ldg(mrow);
            for (int j = 0; j < n_tiles; ++j, ++g) {
                const uint4 mw_next = (j + 1 < n_tiles) ? __ldg(mrow + j + 1) : mw;
                mbar_wait(sc_full, g & 1);
                PROF(pf.lap(0);)
                fence_after_sync();
                uint32_t r[32], gr[32];
                tmem_ld32_nowait(lane_base + COL_S + cg * 32, r);
                tmem_ld32_nowait(lane_base + COL_DP + cg * 32, gr);
                tmem_ld_wait();
                warp_arrive(s_read, lane);
                PROF(pf.lap(1);)
                const uint32_t X = chunk_mask_bytes(mw, cg);
                uint32_t pk[16];
                const bool first = (j == 0 && cg == 0);
                if (!warp_needs_clamp(r, mk.thr)) {
                    if (first) bwdq_chunk32<true, false, E>(r, gr, X, mk, nd, ex0, pk, nofs);
                    else bwdq_chunk32<false, false, E>(r, gr, X, mk, nd, ex0, pk, nofs);
                } else {
                    if (first) bwdq_chunk32<true, true, E>(r, gr, X, mk, nd, ex0, pk, nofs);
                    else bwdq_chunk32<false, true, E>(r, gr, X, mk, nd, ex0, pk, nofs);
                }
                PROF(pf.lap(2);)
                if (g >= 2) {                           // this dS buffer's previous tile has been consumed
                    mbar_wait(e_free(g & 1), ((g >> 1) - 1) & 1);
                    fence_after_sync();
                }
                tmem_st16(lane_base + COL_DS + (g & 1) * 64 + cg * 16, pk);
                tmem_st_wait();
                warp_arrive(p_full(g & 1), lane);
                PROF(pf.lap(3);)
                mw = mw_next;
            }
            mbar_wait(acc_full, w & 1);
            fence_after_sync();
            {
                uint32_t o[16];
                tmem_ld16(lane_base + COL_DQ + cg * 16, o);
                warp_arrive(acc_empty, lane);
                store_row16(dq + (((size_t)hn * S + row) * H + hh) * D + cg * 16, o, scale);
            }
            PROF(pf.lap(5);)
        }
        PROF(pf.t[6] = clock64() - t0; pf.t[4] = g; pf.flush(1, 0, threadIdx.x == 0);)
    }
    fence_before_sync();
    __syncthreads();
    if (warp == W_MMA) tmem_dealloc<512>(tmem_base);
}

static int grid_for(int n_items) { return n_items < num_sms() ? n_items : num_sms(); }

template <typename E>
int launch_bwd_q128(const CUtensorMap &mq, const CUtensorMap &mk, const CUtensorMap &mv, const CUtensorMap &md,
                    const uint32_t *mask, const int32_t *extra0, const float *ndelta, const float *zsum, E *gq, int B,
                    int S, int H, int G, float scale, float clamp, cudaStream_t st) {
    cudaFuncSetAttribute(attn_bwd_q128_kernel<E>, cudaFuncAttributeMaxDynamicSharedMemorySize, Q_SMEM);
    attn_bwd_q128_kernel<E><<<grid_for((S / T) * B), THREADS, Q_SMEM, st>>>(mq, mk, mv, md, mask, extra0, ndelta, gq, S, H, B,
                                                                           scale, scale * LOG2E, clamp * LOG2E, zsum, G);
    return after_launch("attn_bwd_q128_kernel");
}
template int launch_bwd_q128<__nv_bfloat16>(const CUtensorMap &, const CUtensorMap &, const CUtensorMap &,
                                            const CUtensorMap &, const uint32_t *, const int32_t *, const float *,
                                            const float *, __nv_bfloat16 *, int, int, int, int, float, float, cudaStream_t);
template int launch_bwd_q128<__half>(const CUtensorMap &, const CUtensorMap &, const CUtensorMap &, const CUtensorMap &,
                                     const uint32_t *, const int32_t *, const float *, const float *, __half *, int, int,
                                     int, int, float, float, cudaStream_t);

}  // namespace attn_tc128
}  // namespace spt

int spt::attn_tc128::read_prof(unsigned long long *out48, int reset) {
#ifdef SPT_ATTN_PROF
    if (out48 && cudaMemcpyFromSymbol(out48, attn_tc::g_prof, sizeof(unsigned long long) * 48) != cudaSuccess)
        return fail(SPT_ERR_CUDA, "debug_attn_prof: copy failed");
    if (reset) {
        static unsigned long long zeros[48] = {0};
        if (cudaMemcpyToSymbol(attn_tc::g_prof, zeros, sizeof(zeros)) != cudaSuccess) return fail(SPT_ERR_CUDA, "debug_attn_prof: reset failed");
    }
    return 1;
#else
    (void)reset;
    if (out48) memset(out48, 0, sizeof(unsigned long long) * 48);
    return 0;
#endif
}
