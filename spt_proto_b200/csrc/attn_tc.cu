// Fused PQ-sparse attention, forward + backward, as MASKED DENSE TILES on the 5th-generation tensor
// cores: tcgen05.mma with accumulators in TMEM, operands staged by TMA, the probability tile fed back
// to the second GEMM as a TMEM A-operand (never through shared memory or HBM).
//
// What it replaces: the stage chain  sddmm -> clamp_(scaling * ., -10, 10) -> causal CSR softmax ->
// spmm  of SparseVanillaAttentionV2._get_attn/_apply_attn (reference naive_gpt/layers/sparse/
// attention.py:122-141) and its autograd backward (kernels/spmm.py:23-49, softmax.py:21-30,
// sddmm.py:25-51), including the transposed products dK = dS^T Q, dV = P^T dO.
//
// Why dense tiles: the gathered formulation moves one 128-byte K/V row per selected (query, key)
// pair through L1/shared memory and needs a CSR->CSC transpose for dK/dV; on B200 the dense causal
// tile product is cheaper even though only 1/4 of the causal entries are selected (DESIGN.md).  The
// selection enters as the lookup kernel's lane-major bitmask (S % 128 == 0):
//     mask[b][r][4 g + t] bit i  <=>  key 128 g + 4 i + t is one of row r's lookup candidates
// plus extra0[b][r] = number of zero-padding slots of the row (they alias key 0 and, like in the
// reference, take part in the softmax).
//
//   w[r][j] = mask bit (+ extra0[r] for j == 0)
//   e[r][j] = w * exp(clamp(scale * q_r.k_j, -10, 10)),  Z_r = max(1e-9, sum_j e),  y_r = sum_j e/Z v_j
// No running max is needed (the clamp bounds the exponent), so there is no rescaling pass.
// Backward recomputes e from q, k (flash style); only Z [B,S] is saved.  With dO' = dO / Z and
// delta' = (dO . y) / Z prepared by a small row kernel:
//   dP' = dO' V^T,  dS = e * (dP' - delta') * [|scale s| <= 10],  dQ = scale dS K
//   dV = E^T dO',   dK = scale dS^T Q      (E = w * exp(...), unnormalised)
// Deterministic: no atomics anywhere.
//
// Kernel anatomy (all three kernels): a CTA owns one 128-row "owner" tile (queries for fwd / dQ, keys
// for dK/dV) and loops over 64-row "other" tiles.  320 threads:
//   warps 0-7 : two warpgroups; thread = (owner row = TMEM lane, column half): tcgen05.ld its 32 score
//               columns, mask/exp math, tcgen05.st the bf16 probability columns back to TMEM
//   warp  8   : TMA producer (cp.async.bulk.tensor 4-D straight from the [N, S, H, d] layout)
//   warp  9   : TMEM allocator + tcgen05.mma issuer (one thread)
// Two CTAs per SM (256 TMEM columns each): 16 math warps per SM keep the XU/FMA pipes fed while the
// other CTA's MMAs and barrier round trips are in flight.  Score tiles of the next iteration are
// issued while the current one is still in the math phase (double-buffered S in the forward; in the
// dQ kernel the score columns are released as soon as they are in registers).
#include <mutex>

#include "attn_common.cuh"

namespace spt {
namespace attn_tc {

// ---------------------------------------------------------------------------------------------------
// Forward.  TMEM columns: S[2] 0/64 (fp32 128x64), P[2] 128/160 (bf16 pairs, 32 cols), O 192 (128x64).
// ---------------------------------------------------------------------------------------------------

// fp16 (T = __half): kg is the key tensor itself (the row scale reads key row 0 of the head); unused in bf16.
// VARLEN: packed sequences (S = T, H heads, grid (H, work-list capacity)); rows at or past the sequence end read
// neutral per-row data and store nothing.
template <int D, typename T, bool VARLEN = false>
__global__ void __launch_bounds__(THREADS, Dim<D>::CTAS)
attn_fwd_tc_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                   const __grid_constant__ CUtensorMap map_v, const uint32_t *__restrict__ mask,
                   const int32_t *__restrict__ extra0, T *__restrict__ y, float *__restrict__ zsum, int S,
                   int H, float scale_log2, float clamp_log2, int y_transposed, const T *__restrict__ kg,
                   const Varlen vl = {}) {
    constexpr int OWN_BYTES = Dim<D>::OWN_BYTES, T_BYTES = Dim<D>::T_BYTES, OWN_SUB = Dim<D>::OWN_SUB, T_SUB = Dim<D>::T_SUB,
                  TMEM_COLS = Dim<D>::TMEM_COLS, DP = Dim<D>::DP;
    constexpr int NBUF = 3;                            // score buffers
    extern __shared__ unsigned char smem_raw[];
    const Smem sm = align_smem(smem_raw);
    const uint32_t s_q = sm.base, s_k = s_q + OWN_BYTES, s_v = s_k + STAGES * T_BYTES;
    float *s_part = reinterpret_cast<float *>(sm.ptr + OWN_BYTES + 2 * STAGES * T_BYTES);   // [2][128] partial row sums
    uint64_t *bars = reinterpret_cast<uint64_t *>(sm.ptr + OWN_BYTES + 2 * STAGES * T_BYTES + 1024);
    const uint32_t bar0 = smem_u32(bars);
    const uint32_t q_full = bar0, o_full = bar0 + 8;
    auto k_full = [&](int s) { return bar0 + 16 + s * 8; };
    auto k_empty = [&](int s) { return bar0 + 16 + (STAGES + s) * 8; };
    auto v_full = [&](int s) { return bar0 + 16 + (2 * STAGES + s) * 8; };
    auto v_empty = [&](int s) { return bar0 + 16 + (3 * STAGES + s) * 8; };
    auto s_full = [&](int b) { return bar0 + 16 + (4 * STAGES + b) * 8; };          // b = 0 .. NBUF-1
    auto p_full = [&](int b) { return bar0 + 16 + (4 * STAGES + NBUF + b) * 8; };   // b = warpgroup 0, 1
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 + 4 * STAGES + NBUF + 2);

    PROF(const long long t_entry = clock64(); unsigned long long ns0; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns0));)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // grid (heads, query tiles): blockIdx.x (fastest) = head, so the heaviest (last) query tile of EVERY head is scheduled
    // before any lighter tile — the launch ends on the lightest CTAs
    int tile = gridDim.y - 1 - blockIdx.y, start = 0, len = S;
    if constexpr (VARLEN) {
        if ((int)blockIdx.y >= *vl.count) return;
        const int4 it = vl.items[blockIdx.y];
        start = it.x, len = it.y, tile = it.z;
    }
    const int b = blockIdx.x;
    const int m0 = tile * BM;
    const int n_tiles = VARLEN ? (min(m0 + BM, len) + BN - 1) / BN : (m0 + BM) / BN;   // key tiles 0 .. (causal)
    const int hn = VARLEN ? 0 : b / H, hh = VARLEN ? b : b % H;

    if (threadIdx.x == 0) {
        mbar_init(q_full, 1);
        mbar_init(o_full, 1);
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(k_full(s), 1);
            mbar_init(k_empty(s), 1);
            mbar_init(v_full(s), 1);
            mbar_init(v_empty(s), 1);
        }
        for (int i = 0; i < NBUF; ++i) mbar_init(s_full(i), 1);
        for (int i = 0; i < 2; ++i) mbar_init(p_full(i), N_MATH / 2);          // one arrival per thread of a warpgroup
        mbar_fence_init();
    }
    if (warp == 9) tmem_alloc<TMEM_COLS>(smem_u32(tmem_slot));
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    // TMEM columns: score buffers S[b] at 64 b (fp32 128 x 64); P (bf16 pairs, 32 columns) is written IN PLACE over the
    // first half of its own score buffer; O at 192.  Three buffers for two warpgroups: the scores of a group's next tile
    // are computed while it is still in the element math of its current one.
    constexpr uint32_t COL_S = 0, COL_O = NBUF * BN;

    if (warp == 8) {
        // ===== TMA producer =====
        if (lane == 0) {
            mbar_expect_tx(q_full, OWN_BYTES);
            tma_owner<D>(s_q, &map_q, q_full, hh, start + m0, hn);
            for (int j = 0; j < n_tiles; ++j) {
                const int st = j % STAGES;
                const uint32_t ph = (j / STAGES) & 1;
                mbar_wait(k_empty(st), ph ^ 1);
                mbar_expect_tx(k_full(st), T_BYTES);
                tma_other<D>(s_k + st * T_BYTES, &map_k, k_full(st), hh, start + j * BN, hn);
                mbar_wait(v_empty(st), ph ^ 1);
                mbar_expect_tx(v_full(st), T_BYTES);
                tma_other<D>(s_v + st * T_BYTES, &map_v, v_full(st), hh, start + j * BN, hn);
            }
        }
    } else if (warp == 9) {
        // ===== MMA issuer: the whole warp runs the (uniform) loop, one elected lane issues =====
        constexpr uint32_t id_s = idesc_of<T>(BM, BN, 0, 0);   // S = Q K^T   (both K-major)
        constexpr uint32_t id_o = idesc_of<T>(BM, DP, 0, 1);    // O += P V    (A from TMEM, V MN-major)
        const uint64_t dq0 = desc_kmajor(s_q, 0), dk0 = desc_kmajor(s_k, 0), dv0 = desc_mnmajor(s_v, 0, T_SUB);
        // S = Q K^T runs two tiles ahead of O += P V, into the third (free) buffer, so the k-steps of S(j + 2) and of
        // PV(j) touch different TMEM columns and are interleaved: two accumulator chains in flight (consecutive MMAs into
        // one accumulator are serialised, ~93 clk each).
        // (Running three ahead — S(j + 3) into tile j's own buffer right behind PV(j) — was built and produced NaNs under
        // load even with a full drain between the two, for a reason not understood; not used.)
        auto issue_s = [&](int j) {
            const int st = j % STAGES;
            mbar_wait(k_full(st), (j / STAGES) & 1);
            fence_after_sync();
            if (elect_one()) {
                const uint64_t dk = dk0 + (uint64_t)(st * (T_BYTES >> 4));
#pragma unroll
                for (int k = 0; k < DP / 16; ++k)
                    umma_bf16(tmem_base + COL_S + (j % NBUF) * BN, dq0 + kslice<OWN_SUB>(k), dk + kslice<T_SUB>(k), id_s, k != 0);
                umma_commit(s_full(j % NBUF));
                umma_commit(k_empty(st));
            }
            __syncwarp();
        };
        mbar_wait(q_full, 0);
        issue_s(0);
        if (n_tiles > 1) issue_s(1);
        PROF(Prof pf; pf.start(); const long long t0 = pf.last;)
        for (int j = 0; j < n_tiles; ++j) {
            mbar_wait(p_full(j & 1), (j >> 1) & 1);      // warpgroup j & 1 has written P_j
            PROF(pf.lap(1);)
            const int st = j % STAGES;
            mbar_wait(v_full(st), (j / STAGES) & 1);
            const bool has_next = j + 2 < n_tiles;
            const int stn = (j + 2) % STAGES;
            if (has_next) mbar_wait(k_full(stn), ((j + 2) / STAGES) & 1);
            PROF(pf.lap(0);)
            fence_after_sync();
            if (elect_one()) {
                const uint64_t dv = dv0 + (uint64_t)(st * (T_BYTES >> 4));
                const uint64_t dk = dk0 + (uint64_t)(stn * (T_BYTES >> 4));
                const uint32_t s_next = tmem_base + COL_S + ((j + 2) % NBUF) * BN, p_cur = tmem_base + COL_S + (j % NBUF) * BN;
                constexpr int KS = DP / 16, KP = BN / 16;
#pragma unroll
                for (int k = 0; k < (KS > KP ? KS : KP); ++k) {
                    if (k < KS && has_next) umma_bf16(s_next, dq0 + kslice<OWN_SUB>(k), dk + kslice<T_SUB>(k), id_s, k != 0);
                    if (k < KP) umma_bf16_ts(tmem_base + COL_O, p_cur + k * 8, dv + k * MNMAJOR_K16, id_o, (j | k) != 0);
                }
                if (has_next) {
                    umma_commit(s_full((j + 2) % NBUF));
                    umma_commit(k_empty(stn));
                }
                umma_commit(v_empty(st));
                if (j + 1 == n_tiles) umma_commit(o_full);
            }
            __syncwarp();
            PROF(pf.lap(2);)
        }
        PROF(pf.t[3] = clock64() - t0; pf.t[4] = n_tiles; pf.flush(0, 8, lane == 0);)
    } else {
        // ===== softmax warps: thread = (query row = TMEM lane, column half) =====
        const int quarter = warp & 3, half = warp >> 2;
        const int rt = quarter * 32 + lane;               // row inside the tile
        const int row = m0 + rt;
        const bool live = !VARLEN || row < len;           // warp-uniform (len is a multiple of 32)
        const size_t grow = (size_t)b * S + start + row;
        const uint4 *mrow = reinterpret_cast<const uint4 *>(mask + grow * (VARLEN ? vl.mwords : S / 32));
        const float ex0 = live ? (float)extra0[grow] : 0.0f;
        const uint32_t lane_base = tmem_base + ((uint32_t)(quarter * 32) << 16);
        // Ping-pong: warpgroup `half` (warps 4 half .. 4 half + 3, one per scheduler) owns the key tiles j = half (mod 2) and
        // score buffer `half`; a thread processes ALL 64 columns of its row as two 32-column chunks.  The two groups of a
        // CTA (and the two CTAs of the SM) are then in different phases by construction: while one group is in its
        // element math the other waits for / loads its scores, instead of all eight warps contending for the same
        // issue slots and then idling together (measured: 1640 clk per tile and CTA of which 380 waiting, with every
        // warp of the CTA on every tile).
        uint64_t sum2 = pk2(0.0f, 0.0f);
        const MathK mk = make_math(scale_log2, clamp_log2);
        uint4 mw = live ? __ldg(mrow) : make_uint4(0, 0, 0, 0);
        float nofs = 0.0f;                                // fp16: -o of this row
        if constexpr (is_f16<T>) {
            // o = max(floor(c log2 e) - 15, floor(log2 t0) - 14), t0 = (1 + ex0) exp(clamp(scale q.k_0)) the key-0 term:
            // t0 2^-o < 2^15 and e^c 2^-o < 2^16, so no element can overflow, and a row whose scores are all low keeps
            // normal fp16 values.  q.k_0 in fp32 from the row's Q in shared memory and key row 0 of the head.
            mbar_wait(q_full, 0);
            const T *k0 = VARLEN ? kg + ((size_t)start * H + hh) * D : kg + ((size_t)hn * S * H + hh) * D;   // the sequence's key 0
            float dot = 0.0f;
#pragma unroll
            for (int c = 0; c < D / 8; ++c) {              // 16-byte chunk c: sub-tile c / 8, 128-byte swizzled by the row
                const uint4 qa = *reinterpret_cast<const uint4 *>(sm.ptr + (c / 8) * OWN_SUB + rt * 128 + (((c % 8) ^ (rt & 7)) * 16));
                const uint4 ka = __ldg(reinterpret_cast<const uint4 *>(k0) + c);
                const uint32_t qw[4] = {qa.x, qa.y, qa.z, qa.w}, kw[4] = {ka.x, ka.y, ka.z, ka.w};
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    float q0, q1, k0f, k1f;
                    up2(unpack2<T>(qw[i]), q0, q1);
                    up2(unpack2<T>(kw[i]), k0f, k1f);
                    dot = fmaf(q1, k1f, fmaf(q0, k0f, dot));
                }
            }
            const float l0 = __log2f(1.0f + ex0) + fminf(fmaxf(dot * mk.c, -mk.L), mk.L);
            nofs = -fmaxf(floorf(mk.L) - 15.0f, floorf(l0) - 14.0f);
        }
        PROF(Prof pf; pf.start(); const long long t0 = pf.last; pf.t[6] = t0 - t_entry;)
        for (int j = half, it = 0; j < n_tiles; j += 2, ++it) {
            // tile j = keys 64 j .. 64 j + 63 = bits 16 half .. 16 half + 15 of the lane-major words of key group it = j >> 1
            const uint4 mw_next = (j + 2 < n_tiles && live) ? __ldg(mrow + it + 1) : mw;
            const uint32_t buf = lane_base + COL_S + (uint32_t)(j % NBUF) * BN;
            mbar_wait(s_full(j % NBUF), (j / NBUF) & 1);
            PROF(pf.lap(0);)
            fence_after_sync();
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                uint32_t r[32];
                tmem_ld32(buf + c * 32, r);
                PROF(pf.lap(1);)
                const uint32_t X = chunk_mask_bytes(mw, 2 * half + c);
                uint32_t pk[16];
                const bool first = (j == 0 && c == 0);
                if (!warp_needs_clamp(r, mk.thr)) {
                    if (first) fwd_chunk32<true, false, T>(r, X, mk, ex0, sum2, pk, nofs);
                    else fwd_chunk32<false, false, T>(r, X, mk, ex0, sum2, pk, nofs);
                } else {
                    if (first) fwd_chunk32<true, true, T>(r, X, mk, ex0, sum2, pk, nofs);
                    else fwd_chunk32<false, true, T>(r, X, mk, ex0, sum2, pk, nofs);
                }
                PROF(pf.lap(2);)
                tmem_st16(buf + c * 16, pk);             // in place: these columns were consumed by this thread's chunk 0
            }
            tmem_st_wait();
            fence_before_sync();
            mbar_arrive(p_full(half));
            PROF(pf.lap(3);)
            mw = mw_next;
        }
        PROF(pf.t[5] = clock64() - t0; pf.t[4] = n_tiles / 2; const long long t_loop_end = clock64();)
        float sum;
        {
            float lo, hi;
            up2(sum2, lo, hi);
            sum = lo + hi;
        }
        s_part[half * BM + rt] = sum;
        math_warps_sync();
        float inv;
        if constexpr (is_f16<T>) {                        // sum of e 2^-o; Z = sum 2^o (exact)
            const float rs = __uint_as_float((uint32_t)(127 + (int)nofs) << 23);     // 2^-o
            sum = fmaxf(s_part[rt] + s_part[BM + rt], 1e-9f * rs);
            if (half == 0 && live) zsum[grow] = sum * __uint_as_float((uint32_t)(127 - (int)nofs) << 23);
            inv = 1.0f / sum;
        } else {
            sum = fmaxf(s_part[rt] + s_part[BM + rt], 1e-9f);
            if (half == 0 && live) zsum[grow] = sum;
            inv = 1.0f / sum;
        }
        mbar_wait(o_full, 0);
        fence_after_sync();
        if (!live) {
        } else if (!y_transposed) {
            T *dst = y + (((size_t)hn * S + start + row) * H + hh) * D;
            out_chunks<D>(half, [&](int col, auto w) {
                uint32_t r[32];
                tmem_ld32(lane_base + COL_O + col, r);
                store_row_n<decltype(w)::value>(dst + col, r, inv);
            });
        } else {
            // the shipped reference layer's output layout (attention.py:139-142): y^T [B, D, S] memory; a warp's 32
            // consecutive rows of one feature are 64 contiguous bytes
            // (VARLEN: each sequence's own y^T [H, D, len], at token offset start)
            out_chunks<D>(half, [&](int col, auto w) {
                T *dst = VARLEN ? y + (size_t)start * H * D + ((size_t)b * D + col) * len + row : y + ((size_t)b * D + col) * S + row;
                const size_t stride = VARLEN ? len : S;
                uint32_t r[32];
                tmem_ld32(lane_base + COL_O + col, r);
#pragma unroll
                for (int i = 0; i < decltype(w)::value; ++i) dst[(size_t)i * stride] = out_elem(__uint_as_float(r[i]) * inv, dst);
            });
        }
        PROF(pf.t[7] = clock64() - t_loop_end; pf.flush(0, 0, threadIdx.x == 0);)
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 9) tmem_dealloc<TMEM_COLS>(tmem_base);
    PROF(if (threadIdx.x == 0) {
        unsigned long long ns1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns1));
        atomicAdd(&g_prof[0][15], (unsigned long long)(clock64() - t_entry));
        atomicAdd(&g_prof[0][14], 1ull);
        atomicAdd(&g_prof[0][13], ns1 - ns0);
    })
}

// ---------------------------------------------------------------------------------------------------
// Backward prologue: -delta'_r = -(dO_r . y_r) / Z_r (stored negated)  and  dO'_r = dO_r / Z_r (bf16, same layout as dO).
// D / 8 lanes per row (16 B each) in an aligned group of PREP_LANES lanes (a power of two for the butterfly sum; at
// D = 80, 10 of 16 lanes carry data).  fp16: Z_r 2^-o_r in [1, 2) takes the place of Z_r (the kernels scale e by 2^-o_r),
// so dO' stays within the range of dO.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ float prep_inv(float z, bool f16) { return 1.0f / (f16 ? f16_bwd_zs(z) : z); }

template <int D, typename T>
__global__ void __launch_bounds__(256)
attn_bwd_prep_kernel(const T *__restrict__ dy, const T *__restrict__ y,
                     const float *__restrict__ zsum, float *__restrict__ delta, T *__restrict__ dys,
                     int64_t rows, int S, int H) {
    constexpr int LPR = D / 8, G = Dim<D>::PREP_LANES;                    // data lanes per row, lanes per row
    const int64_t row = (int64_t)blockIdx.x * (256 / G) + (threadIdx.x / G);
    if (row >= rows) return;
    const int sub = threadIdx.x % G;
    const bool active = sub < LPR;
    const int64_t b = row / S, r = row % S;                               // delta, zsum are head-major [B, S]
    const int64_t off = (((b / H) * S + r) * H + (b % H)) * D + sub * 8;
    float a[8], c[8];
    if (active) {
        Vec16<T>::load(dy + off, a);
        Vec16<T>::load(y + off, c);
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) a[i] = c[i] = 0.0f;
    }
    float acc = 0.0f;
#pragma unroll
    for (int i = 0; i < 8; ++i) acc = fmaf(a[i], c[i], acc);
    acc = group_sum<G>(acc);
    const float inv = prep_inv(zsum[row], is_f16<T>);
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] *= inv;
    if (active) Vec16<T>::store(dys + off, a);
    if (sub == 0) delta[row] = -acc * inv;        // stored negated: the kernels add it (dp - delta')
}

// The same for dO and y in the reference layer's output layout (y^T, dO^T: [B, D, S] memory): a block transposes a
// [D] x [64 rows] tile of each through shared memory; dO' is written in the standard [N, S, H, D] layout the TMA maps read.
// VARLEN: block x = one 64-row half of a work-list item; a sequence's y^T / dO^T is [H, D, len] at token offset start.
template <int D, typename T, bool VARLEN = false>
__global__ void __launch_bounds__(256)
attn_bwd_prep_t_kernel(const T *__restrict__ dyt, const T *__restrict__ yt,
                       const float *__restrict__ zsum, float *__restrict__ delta, T *__restrict__ dys, int S,
                       int H, const Varlen vl = {}) {
    constexpr int TR = 64, LD = TR + 8;
    __shared__ __align__(16) T s_dy[D][LD];
    __shared__ __align__(16) T s_y[D][LD];
    int r0 = blockIdx.x * TR, start = 0, len = S;
    if constexpr (VARLEN) {
        if ((int)(blockIdx.x >> 1) >= *vl.count) return;
        const int4 it = vl.items[blockIdx.x >> 1];
        start = it.x, len = it.y, r0 = it.z * 128 + (blockIdx.x & 1) * TR;
        if (r0 >= len) return;
    }
    const int b = blockIdx.y;
    const size_t base = VARLEN ? (size_t)start * H * D + (size_t)b * D * len + r0 : (size_t)b * D * S + r0;
    const size_t ld = VARLEN ? len : S;
    constexpr int EPT = D / 4;                       // features per thread
    // the 16-byte row chunks of feature e sit at chunk index (c / 8) ^ (e / EPT): the four threads of a row read the
    // same column of four features 16 * LD elements apart (the same bank without the swizzle: 4-way conflicts on
    // every one of the 2 * EPT reads)
    for (int id = threadIdx.x; id < D * (TR / 8); id += 256) {
        const int e = id / (TR / 8), c = (id % (TR / 8)) * 8, cs = (((id % (TR / 8)) ^ (e / EPT)) & (TR / 8 - 1)) * 8;
        if (VARLEN && r0 + c >= len) continue;       // rows past the sequence end (the rows of those threads store nothing)
        *reinterpret_cast<uint4 *>(&s_dy[e][cs]) = *reinterpret_cast<const uint4 *>(dyt + base + (size_t)e * ld + c);
        *reinterpret_cast<uint4 *>(&s_y[e][cs]) = *reinterpret_cast<const uint4 *>(yt + base + (size_t)e * ld + c);
    }
    __syncthreads();
    const int r = threadIdx.x >> 2, qd = threadIdx.x & 3;
    const int rs = ((((r >> 3) ^ qd) & (TR / 8 - 1)) << 3) | (r & 7);
    float a[EPT];
    float acc = 0.0f;
#pragma unroll
    for (int i = 0; i < EPT; ++i) {
        a[i] = to_f32(s_dy[qd * EPT + i][rs]);
        acc = fmaf(a[i], to_f32(s_y[qd * EPT + i][rs]), acc);
    }
    acc = group_sum<4>(acc);
    if (VARLEN && r0 + r >= len) return;
    const size_t grow = (size_t)b * S + start + r0 + r;
    const float inv = prep_inv(zsum[grow], is_f16<T>);
    const int hn = VARLEN ? 0 : b / H, hh = VARLEN ? b : b % H;
    T *dst = dys + (((size_t)hn * S + start + r0 + r) * H + hh) * D + qd * EPT;
    if constexpr (EPT % 8 == 0) {
#pragma unroll
        for (int i = 0; i < EPT; i += 8) {
            float t[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) t[u] = a[i + u] * inv;
            Vec16<T>::store(dst + i, t);
        }
    } else {
        // D = 80: a thread's 20 features start 40 bytes apart, so 8-byte stores
        static_assert(EPT % 4 == 0, "features per thread must be a multiple of 4");
#pragma unroll
        for (int i = 0; i < EPT; i += 4)
            *reinterpret_cast<uint2 *>(dst + i) = make_uint2(pack2<T>(a[i] * inv, a[i + 1] * inv), pack2<T>(a[i + 2] * inv, a[i + 3] * inv));
    }
    if (qd == 0) delta[grow] = -acc * inv;
}

// ---------------------------------------------------------------------------------------------------
// Backward, dQ: owner = 128 query rows (Q, dO'), loop over 64-key tiles (K_j, V_j).
// TMEM columns: S 0, dP' 64 (128x64 fp32 each), dS[2] 128/160 (bf16 pairs), dQ 192.
// The score columns are released (s_read) as soon as every math thread holds its 32+32 values in
// registers, so the tensor core computes the next tile's scores under this tile's exp math.
// ---------------------------------------------------------------------------------------------------

// fp16: zsum gives the row scales (read by the fp16 instantiations only).  VARLEN: see the forward.
template <int D, typename T, bool VARLEN = false>
__global__ void __launch_bounds__(THREADS, Dim<D>::CTAS)
attn_bwd_q_tc_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                     const __grid_constant__ CUtensorMap map_v, const __grid_constant__ CUtensorMap map_dys,
                     const uint32_t *__restrict__ mask, const int32_t *__restrict__ extra0,
                     const float *__restrict__ delta, T *__restrict__ dq, int S, int H, float scale,
                     float scale_log2, float clamp_log2, const float *__restrict__ zsum, const Varlen vl = {}) {
    constexpr int OWN_BYTES = Dim<D>::OWN_BYTES, T_BYTES = Dim<D>::T_BYTES, OWN_SUB = Dim<D>::OWN_SUB, T_SUB = Dim<D>::T_SUB,
                  TMEM_COLS = Dim<D>::TMEM_COLS, DP = Dim<D>::DP;
    extern __shared__ unsigned char smem_raw[];
    const Smem sm = align_smem(smem_raw);
    const uint32_t s_q = sm.base, s_dy = s_q + OWN_BYTES, s_k = s_dy + OWN_BYTES, s_v = s_k + STAGES * T_BYTES;
    uint64_t *bars = reinterpret_cast<uint64_t *>(sm.ptr + 2 * OWN_BYTES + 2 * STAGES * T_BYTES);
    const uint32_t bar0 = smem_u32(bars);
    const uint32_t own_full = bar0, acc_full = bar0 + 8, s_read = bar0 + 24;
    // one "scores ready" barrier per warpgroup (tile parity): the two groups may be a phase apart, and a parity wait
    // cannot tell "phase j+1 complete" from "phase j-1 complete"
    auto sc_full = [&](int i) { return i == 0 ? bar0 + 16 : bar0 + 48 + 2 * STAGES * 8; };
    auto p_full = [&](int i) { return bar0 + 32 + i * 8; };
    auto kv_full = [&](int s) { return bar0 + 48 + s * 8; };
    auto kv_empty = [&](int s) { return bar0 + 48 + (STAGES + s) * 8; };
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 7 + 2 * STAGES);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int tile = gridDim.y - 1 - blockIdx.y, start = 0, len = S;   // grid (heads, tiles): every head's heaviest tile first (see the forward)
    if constexpr (VARLEN) {
        if ((int)blockIdx.y >= *vl.count) return;
        const int4 it = vl.items[blockIdx.y];
        start = it.x, len = it.y, tile = it.z;
    }
    const int b = blockIdx.x;
    const int m0 = tile * BM;
    const int n_tiles = VARLEN ? (min(m0 + BM, len) + BN - 1) / BN : (m0 + BM) / BN;
    const int hn = VARLEN ? 0 : b / H, hh = VARLEN ? b : b % H;

    if (threadIdx.x == 0) {
        mbar_init(own_full, 1);
        mbar_init(acc_full, 1);
        mbar_init(sc_full(0), 1);
        mbar_init(sc_full(1), 1);
        mbar_init(s_read, N_MATH / 2);                // one warpgroup per tile
        mbar_init(p_full(0), N_MATH / 2);
        mbar_init(p_full(1), N_MATH / 2);
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(kv_full(s), 1);
            mbar_init(kv_empty(s), 1);
        }
        mbar_fence_init();
    }
    if (warp == 9) tmem_alloc<TMEM_COLS>(smem_u32(tmem_slot));
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    constexpr uint32_t COL_S = 0, COL_DP = 64, COL_DS = 128, COL_DQ = 192;

    if (warp == 8) {
        if (lane == 0) {
            mbar_expect_tx(own_full, 2 * OWN_BYTES);
            tma_owner<D>(s_q, &map_q, own_full, hh, start + m0, hn);
            tma_owner<D>(s_dy, &map_dys, own_full, hh, start + m0, hn);
            for (int j = 0; j < n_tiles; ++j) {
                const int st = j % STAGES;
                mbar_wait(kv_empty(st), ((j / STAGES) & 1) ^ 1);
                mbar_expect_tx(kv_full(st), 2 * T_BYTES);
                tma_other<D>(s_k + st * T_BYTES, &map_k, kv_full(st), hh, start + j * BN, hn);
                tma_other<D>(s_v + st * T_BYTES, &map_v, kv_full(st), hh, start + j * BN, hn);
            }
        }
    } else if (warp == 9) {
        constexpr uint32_t id_s = idesc_of<T>(BM, BN, 0, 0);   // S = Q K^T, dP' = dO' V^T
        constexpr uint32_t id_a = idesc_of<T>(BM, DP, 0, 1);    // dQ += dS K   (A from TMEM, K MN-major)
        const uint64_t dq0 = desc_kmajor(s_q, 0), ddy0 = desc_kmajor(s_dy, 0), dk0 = desc_kmajor(s_k, 0),
                       dv0 = desc_kmajor(s_v, 0), dkt0 = desc_mnmajor(s_k, 0, T_SUB);
        // The score MMAs of tile j are issued as soon as tile j-1's scores are in the math warps' registers (s_read): they are
        // on the critical path (the math warps wait for them), the accumulating MMAs dQ += dS_{j-1} K_{j-1} are not and
        // follow once dS_{j-1} is written.  (Interleaving the three chains in one group was measured slower: 2125 vs 1940
        // clk per tile — it delays the scores behind p_full.)
        auto issue_acc = [&](int j, bool last) {                  // dQ += dS_j K_j
            const int st = j % STAGES;
            mbar_wait(p_full(j & 1), (j >> 1) & 1);
            fence_after_sync();
            if (elect_one()) {
                const uint64_t dkt = dkt0 + (uint64_t)(st * (T_BYTES >> 4));
#pragma unroll
                for (int k = 0; k < BN / 16; ++k)
                    umma_bf16_ts(tmem_base + COL_DQ, tmem_base + COL_DS + (j & 1) * 32 + k * 8, dkt + k * MNMAJOR_K16, id_a,
                                 (j | k) != 0);
                umma_commit(kv_empty(st));
                if (last) umma_commit(acc_full);
            }
            __syncwarp();
        };
        mbar_wait(own_full, 0);
        PROF(Prof pf; pf.start(); const long long t0 = pf.last;)
        for (int j = 0; j < n_tiles; ++j) {
            const int st = j % STAGES;
            mbar_wait(kv_full(st), (j / STAGES) & 1);
            PROF(pf.lap(0);)
            if (j > 0) mbar_wait(s_read, (j - 1) & 1);        // tile j-1's scores are in registers
            PROF(pf.lap(1);)
            fence_after_sync();
            if (elect_one()) {
                const uint64_t off = (uint64_t)(st * (T_BYTES >> 4));
                // S and dP' are independent accumulators: alternating their k-steps keeps consecutive MMAs independent
                // (back-to-back MMAs into one accumulator are serialised by the accumulate dependency, ~93 clk each)
#pragma unroll
                for (int k = 0; k < DP / 16; ++k) {
                    umma_bf16(tmem_base + COL_S, dq0 + kslice<OWN_SUB>(k), dk0 + off + kslice<T_SUB>(k), id_s, k != 0);
                    umma_bf16(tmem_base + COL_DP, ddy0 + kslice<OWN_SUB>(k), dv0 + off + kslice<T_SUB>(k), id_s, k != 0);
                }
                umma_commit(sc_full(j & 1));
            }
            __syncwarp();
            PROF(pf.lap(2);)
            if (j > 0) issue_acc(j - 1, false);
            PROF(pf.lap(5);)
        }
        issue_acc(n_tiles - 1, true);
        PROF(pf.t[3] = clock64() - t0; pf.t[4] = n_tiles; pf.flush(1, 8, lane == 0);)
    } else {
        const int quarter = warp & 3, half = warp >> 2;
        const int row = m0 + quarter * 32 + lane;
        const bool live = !VARLEN || row < len;           // warp-uniform (len is a multiple of 32)
        const size_t grow = (size_t)b * S + start + row;
        const uint4 *mrow = reinterpret_cast<const uint4 *>(mask + grow * (VARLEN ? vl.mwords : S / 32));
        const float ex0 = live ? (float)extra0[grow] : 0.0f;
        const float dl = live ? delta[grow] : 0.0f;
        const float nofs = (is_f16<T> && live) ? f16_bwd_nofs(zsum[grow]) : 0.0f;
        const uint32_t lane_base = tmem_base + ((uint32_t)(quarter * 32) << 16);
        const MathK mk = make_math(scale_log2, clamp_log2);
        uint4 mw = live ? __ldg(mrow) : make_uint4(0, 0, 0, 0);
        PROF(Prof pf; pf.start(); const long long t0 = pf.last;)
        // Ping-pong (see the forward kernel): warpgroup `half` owns the key tiles j = half (mod 2) and dS buffer `half`; a
        // thread processes all 64 columns of its row as two 32-column chunks, and releases the (single) score buffer as
        // soon as the second chunk is in registers.
        for (int j = half, it = 0; j < n_tiles; j += 2, ++it) {
            const uint4 mw_next = (j + 2 < n_tiles && live) ? __ldg(mrow + it + 1) : mw;
            mbar_wait(sc_full(half), it & 1);
            PROF(pf.lap(0);)
            fence_after_sync();
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                uint32_t r[32], g[32];
                tmem_ld32_nowait(lane_base + COL_S + c * 32, r);
                tmem_ld32_nowait(lane_base + COL_DP + c * 32, g);
                tmem_ld_wait();
                if (c == 1) {
                    fence_before_sync();
                    mbar_arrive(s_read);
                }
                PROF(pf.lap(1);)
                const uint32_t X = chunk_mask_bytes(mw, 2 * half + c);
                uint32_t pk[16];
                const bool first = (j == 0 && c == 0);
                if (!warp_needs_clamp(r, mk.thr)) {
                    if (first) bwdq_chunk32<true, false, T>(r, g, X, mk, dl, ex0, pk, nofs);
                    else bwdq_chunk32<false, false, T>(r, g, X, mk, dl, ex0, pk, nofs);
                } else {
                    if (first) bwdq_chunk32<true, true, T>(r, g, X, mk, dl, ex0, pk, nofs);
                    else bwdq_chunk32<false, true, T>(r, g, X, mk, dl, ex0, pk, nofs);
                }
                PROF(pf.lap(2);)
                tmem_st16(lane_base + COL_DS + half * 32 + c * 16, pk);
            }
            tmem_st_wait();
            fence_before_sync();
            mbar_arrive(p_full(half));
            PROF(pf.lap(3);)
            mw = mw_next;
        }
        PROF(pf.t[5] = clock64() - t0; pf.t[4] = n_tiles / 2; pf.flush(1, 0, threadIdx.x == 0);)
        mbar_wait(acc_full, 0);
        fence_after_sync();
        T *dst = dq + (((size_t)hn * S + start + row) * H + hh) * D;
        if (live)
            out_chunks<D>(half, [&](int col, auto w) {
                uint32_t r[32];
                tmem_ld32(lane_base + COL_DQ + col, r);
                store_row_n<decltype(w)::value>(dst + col, r, scale);
            });
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 9) tmem_dealloc<TMEM_COLS>(tmem_base);
}

// ---------------------------------------------------------------------------------------------------
// Backward, dK / dV: owner = 128 keys (K, V) = one lane-major mask group, loop over 64-row query tiles
// (Q_j, dO'_j) at and below the diagonal.  Works on the transposed tiles S^T = K Q^T, dP'^T = V dO'^T
// so that E^T and dS^T come out with keys on the TMEM lanes, ready to be the A operands of
//   dV += E^T dO'_j   and   dK += dS^T Q_j.
// The 64-row tiles are consumed as two 32-row sub-tiles with two score buffers in TMEM (S^T 32 + dP'^T 32
// columns each, then dV, dK): the tensor core computes the next sub-tile's scores under this one's exp math.
// E^T / dS^T (bf16 pairs) are written back over score columns the same thread has already consumed.
// Per-row quantities of the 64 query rows (mask words of this key group, delta', extra0) are staged in
// shared memory by the producer warp, one slot per pipeline stage (fp16: also the rows' -o, from zsum).
// ---------------------------------------------------------------------------------------------------
// VARLEN: see the forward.
template <int D, typename T, bool VARLEN = false>
__global__ void __launch_bounds__(THREADS, Dim<D>::CTAS)
attn_bwd_kv_tc_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                      const __grid_constant__ CUtensorMap map_v, const __grid_constant__ CUtensorMap map_dys,
                      const uint32_t *__restrict__ mask, const int32_t *__restrict__ extra0,
                      const float *__restrict__ delta, T *__restrict__ dk, T *__restrict__ dv,
                      int S, int H, float scale, float scale_log2, float clamp_log2, const float *__restrict__ zsum,
                      const Varlen vl = {}) {
    constexpr int OWN_BYTES = Dim<D>::OWN_BYTES, T_BYTES = Dim<D>::T_BYTES, OWN_SUB = Dim<D>::OWN_SUB, T_SUB = Dim<D>::T_SUB,
                  TMEM_COLS = Dim<D>::TMEM_COLS, DP = Dim<D>::DP;
    extern __shared__ unsigned char smem_raw[];
    const Smem sm = align_smem(smem_raw);
    const uint32_t s_k = sm.base, s_v = s_k + OWN_BYTES, s_q = s_v + OWN_BYTES, s_dy = s_q + STAGES * T_BYTES;
    unsigned char *rowq = sm.ptr + 2 * OWN_BYTES + 2 * STAGES * T_BYTES;   // per stage: mask^T [4][64 + 4], delta[64], ex0[64] (, -o[64])
    constexpr int MT = BN + 4;                         // padded row of the transposed mask: the 4 words hit distinct banks
    constexpr int ROWQ_BYTES = MT * 16 + BN * 4 + BN * 4 + (is_f16<T> ? BN * 4 : 0);
    uint64_t *bars = reinterpret_cast<uint64_t *>(rowq + STAGES * ROWQ_BYTES);
    const uint32_t bar0 = smem_u32(bars);
    const uint32_t own_full = bar0, acc_full = bar0 + 8;
    auto sc_full = [&](int i) { return bar0 + 16 + i * 8; };
    auto p_full = [&](int i) { return bar0 + 32 + i * 8; };
    auto qd_full = [&](int s) { return bar0 + 48 + s * 8; };
    auto qd_empty = [&](int s) { return bar0 + 48 + (STAGES + s) * 8; };
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 6 + 2 * STAGES);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int kt = blockIdx.y, start = 0, len = S;           // key tile (early key tiles are the heaviest); grid (heads, tiles):
    if constexpr (VARLEN) {                            // every head's heaviest tile first (see the forward)
        if ((int)blockIdx.y >= *vl.count) return;
        const int4 it = vl.items[blockIdx.y];
        // the work list puts the query tiles with the most keys first; mirrored inside each sequence, its first items are
        // the key tiles with the most query rows at and below them
        start = it.x, len = it.y, kt = (len + BM - 1) / BM - 1 - it.z;
    }
    const int b = blockIdx.x;
    const int n0 = kt * BM;
    const int j0 = n0 / BN;                            // first query tile that can see these keys
    const int n_tiles = (VARLEN ? (len + BN - 1) / BN : S / BN) - j0;
    const int hn = VARLEN ? 0 : b / H, hh = VARLEN ? b : b % H;
    const size_t head = (size_t)b * S + start;
    const int words = VARLEN ? vl.mwords : S / 32;

    if (threadIdx.x == 0) {
        mbar_init(own_full, 1);
        mbar_init(acc_full, 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(sc_full(i), 1);
            mbar_init(p_full(i), N_MATH / 2);          // one warpgroup per score buffer
        }
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(qd_full(s), 1 + 32);             // expect_tx arrive + the 32 producer lanes' row data
            mbar_init(qd_empty(s), 1);
        }
        mbar_fence_init();
    }
    if (warp == 9) tmem_alloc<TMEM_COLS>(smem_u32(tmem_slot));
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    // score buffers b = 0, 1 (one per 32-row sub-tile in flight): S^T at 64 b, dP'^T at 64 b + 32
    constexpr uint32_t COL_SC = 0, COL_DV = 128, COL_DK = 128 + DP;
    constexpr int SUBN = 32;

    if (warp == 8) {
        if (lane == 0) {
            mbar_expect_tx(own_full, 2 * OWN_BYTES);
            tma_owner<D>(s_k, &map_k, own_full, hh, start + n0, hn);
            tma_owner<D>(s_v, &map_v, own_full, hh, start + n0, hn);
        }
        for (int j = 0; j < n_tiles; ++j) {
            const int st = j % STAGES;
            const int r0 = (j0 + j) * BN;
            mbar_wait(qd_empty(st), ((j / STAGES) & 1) ^ 1);
            if (lane == 0) {
                mbar_expect_tx(qd_full(st), 2 * T_BYTES);
                tma_other<D>(s_q + st * T_BYTES, &map_q, qd_full(st), hh, start + r0, hn);
                tma_other<D>(s_dy + st * T_BYTES, &map_dys, qd_full(st), hh, start + r0, hn);
            }
            unsigned char *slot = rowq + st * ROWQ_BYTES;
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int rr = lane + 32 * u;
                const size_t gr = head + r0 + rr;
                const bool live = !VARLEN || r0 + rr < len;   // rows past the sequence end: no key, neutral row data
                const uint4 mw = live ? __ldg(reinterpret_cast<const uint4 *>(mask + gr * words) + kt) : make_uint4(0, 0, 0, 0);
                uint32_t *mt = reinterpret_cast<uint32_t *>(slot);        // transposed: [word t][row], rows padded to MT
                mt[rr] = mw.x;
                mt[MT + rr] = mw.y;
                mt[2 * MT + rr] = mw.z;
                mt[3 * MT + rr] = mw.w;
                reinterpret_cast<float *>(slot + MT * 16)[rr] = live ? delta[gr] : 0.0f;      // -delta' (the math adds it: dp - delta')
                reinterpret_cast<float *>(slot + MT * 16 + BN * 4)[rr] = live ? (float)extra0[gr] : 0.0f;
                if constexpr (is_f16<T>) reinterpret_cast<float *>(slot + MT * 16 + 2 * BN * 4)[rr] = live ? f16_bwd_nofs(zsum[gr]) : 0.0f;
            }
            mbar_arrive(qd_full(st));
        }
    } else if (warp == 9) {
        // Sub-tiles t = 2 j + h of 32 query rows: scores of sub-tile t+1 are issued before the math warps have
        // finished sub-tile t (two score buffers), the accumulating MMAs of t follow once its E^T / dS^T are written.
        constexpr uint32_t id_s = idesc_of<T>(BM, SUBN, 0, 0); // S^T = K Q^T, dP'^T = V dO'^T   (N = 32 query rows)
        constexpr uint32_t id_a = idesc_of<T>(BM, DP, 0, 1);    // dV += E^T dO', dK += dS^T Q (B MN-major, K = 32)
        const uint64_t dk0 = desc_kmajor(s_k, 0), dv0 = desc_kmajor(s_v, 0), dq0 = desc_kmajor(s_q, 0),
                       ddy0 = desc_kmajor(s_dy, 0), dqt0 = desc_mnmajor(s_q, 0, T_SUB),
                       ddyt0 = desc_mnmajor(s_dy, 0, T_SUB);
        const int n_sub = 2 * n_tiles;
        auto issue_scores = [&](int t) {
            const int j = t >> 1, h = t & 1, st = j % STAGES;
            if (h == 0) mbar_wait(qd_full(st), (j / STAGES) & 1);
            fence_after_sync();
            if (elect_one()) {
                // rows 32 h .. 32 h + 31 of the stage's 64-row tiles: + 32 rows * 128 B inside every 64-wide sub-tile
                const uint64_t off = (uint64_t)((st * T_BYTES + h * SUBN * 128) >> 4);
                const uint32_t col = tmem_base + COL_SC + (t & 1) * 64;
                // S^T and dP'^T are independent accumulators: alternate their k-steps (see the dQ kernel)
#pragma unroll
                for (int k = 0; k < DP / 16; ++k) {
                    umma_bf16(col, dk0 + kslice<OWN_SUB>(k), dq0 + off + kslice<T_SUB>(k), id_s, k != 0);
                    umma_bf16(col + 32, dv0 + kslice<OWN_SUB>(k), ddy0 + off + kslice<T_SUB>(k), id_s, k != 0);
                }
                umma_commit(sc_full(t & 1));
            }
            __syncwarp();
        };
        mbar_wait(own_full, 0);
        issue_scores(0);
        PROF(Prof pf; pf.start(); const long long t0 = pf.last;)
        for (int t = 0; t < n_sub; ++t) {
            if (t + 1 < n_sub) issue_scores(t + 1);   // its buffer was last read by the accumulating MMAs of t - 1 (in order)
            PROF(pf.lap(0);)
            const int j = t >> 1, h = t & 1, st = j % STAGES;
            mbar_wait(p_full(t & 1), (t >> 1) & 1);
            PROF(pf.lap(1);)
            fence_after_sync();
            if (elect_one()) {
                const uint64_t off = (uint64_t)((st * T_BYTES) >> 4);
                const uint32_t col = tmem_base + COL_SC + (t & 1) * 64;
                // query rows 16 k .. 16 k + 15 of the sub-tile sit in columns 8 k .. 8 k + 7 of E^T (over S^T) / dS^T (over dP'^T)
#pragma unroll
                for (int k = 0; k < SUBN / 16; ++k) {   // dV and dK alternate as well
                    umma_bf16_ts(tmem_base + COL_DV, col + k * 8, ddyt0 + off + (2 * h + k) * MNMAJOR_K16, id_a, (t | k) != 0);
                    umma_bf16_ts(tmem_base + COL_DK, col + 32 + k * 8, dqt0 + off + (2 * h + k) * MNMAJOR_K16, id_a, (t | k) != 0);
                }
                if (h == 1) umma_commit(qd_empty(st));
                if (t + 1 == n_sub) umma_commit(acc_full);
            }
            __syncwarp();
            PROF(pf.lap(2);)
        }
        PROF(pf.t[3] = clock64() - t0; pf.t[4] = n_sub; pf.flush(2, 8, lane == 0);)
    } else {
        // thread = (key n0 + kk = TMEM lane kk, column half): lane-major word kk & 3 of the row's group kt, bit kk >> 2
        const int quarter = warp & 3, half = warp >> 2;
        const int kk = quarter * 32 + lane;
        const int wsel = kk & 3;
        const int shl = 31 - (kk >> 2);                 // moves this key's bit of a lane-major word to the sign bit
        const bool key0 = (n0 + kk) == 0;
        const MathK mk = make_math(scale_log2, clamp_log2);
        const uint32_t lane_base = tmem_base + ((uint32_t)(quarter * 32) << 16);
        PROF(Prof pf; pf.start(); const long long t0 = pf.last;)
        // Ping-pong: warpgroup `half` owns the sub-tiles t = 2 j + half (rows 32 half .. 32 half + 31 of every 64-row tile)
        // and score buffer `half`; a thread processes all 32 query rows of its key's sub-tile (see the forward kernel).
        for (int j = 0; j < n_tiles; ++j) {
            const int st = j % STAGES, h = half;
            const unsigned char *slot = rowq + st * ROWQ_BYTES;
            const uint32_t *mrow = reinterpret_cast<const uint32_t *>(slot) + wsel * MT;   // this key's word of every row
            const float *s_ndelta = reinterpret_cast<const float *>(slot + MT * 16);
            const float *s_ex0 = s_ndelta + BN;
            const float *s_nofs = s_ndelta + 2 * BN;
            mbar_wait(qd_full(st), (j / STAGES) & 1);   // the producer lanes' row data of this stage
            mbar_wait(sc_full(h), j & 1);
            PROF(pf.lap(0);)
            fence_after_sync();
            const uint32_t col = lane_base + COL_SC + h * 64;       // S^T at col, dP'^T at col + 32
            const int c0 = h * SUBN;                                 // rows c0 .. c0 + 31 of the tile
            uint32_t r[32], g[32];
            tmem_ld32_nowait(col, r);
            tmem_ld32_nowait(col + 32, g);
            tmem_ld_wait();
            PROF(pf.lap(1);)
            const bool clamp = warp_needs_clamp(r, mk.thr);
            uint32_t pe[8], pd[8];
#define SPT_KV_HALF(OFF)                                                                                                   \
            if (key0) {                                                                                                    \
                if (clamp) bwdkv_chunk16<true, true, OFF, 32, float, T>(r, g, mrow, s_ndelta, s_ex0, c0 + OFF, shl, mk, pe, pd, s_nofs); \
                else bwdkv_chunk16<true, false, OFF, 32, float, T>(r, g, mrow, s_ndelta, s_ex0, c0 + OFF, shl, mk, pe, pd, s_nofs);      \
            } else {                                                                                                       \
                if (clamp) bwdkv_chunk16<false, true, OFF, 32, float, T>(r, g, mrow, s_ndelta, s_ex0, c0 + OFF, shl, mk, pe, pd, s_nofs); \
                else bwdkv_chunk16<false, false, OFF, 32, float, T>(r, g, mrow, s_ndelta, s_ex0, c0 + OFF, shl, mk, pe, pd, s_nofs);     \
            }                                                                                                              \
            tmem_st8(col + (OFF) / 2, pe);      /* E^T over the S^T columns this thread has consumed */                    \
            tmem_st8(col + 32 + (OFF) / 2, pd); /* dS^T over its dP'^T columns */
            SPT_KV_HALF(0)
            SPT_KV_HALF(16)
#undef SPT_KV_HALF
            PROF(pf.lap(2);)
            tmem_st_wait();
            fence_before_sync();
            mbar_arrive(p_full(h));
            PROF(pf.lap(3);)
        }
        PROF(pf.t[5] = clock64() - t0; pf.t[4] = n_tiles; pf.flush(2, 0, threadIdx.x == 0);)
        mbar_wait(acc_full, 0);
        fence_after_sync();
        const size_t off = (((size_t)hn * S + start + n0 + kk) * H + hh) * D;
        if (!VARLEN || n0 + kk < len)                  // warp-uniform
            out_chunks<D>(half, [&](int col, auto w) {
                uint32_t r[32];
                tmem_ld32(lane_base + COL_DV + col, r);
                store_row_n<decltype(w)::value>(dv + off + col, r, 1.0f);
                tmem_ld32(lane_base + COL_DK + col, r);
                store_row_n<decltype(w)::value>(dk + off + col, r, scale);
            });
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 9) tmem_dealloc<TMEM_COLS>(tmem_base);
}

// ---- host -----------------------------------------------------------------------------------------
// 4-D bf16 / fp16 tensor map over a [N, S, H, D] tensor (H = 1: head-major [B, S, D]); box = 64 rows x 64 elements of one
// head.  D = 80: the box at column 64 holds the row's last 16 elements; the 48 out-of-bounds columns are filled with zeros.
static int make_map(CUtensorMap *map, const void *base, int N, int S, int H, int D, bool f16) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return fail(SPT_ERR_CUDA, "sparse_attn: cuTensorMapEncodeTiled entry point not available");
    cuuint64_t dims[4] = {(cuuint64_t)D, (cuuint64_t)H, (cuuint64_t)S, (cuuint64_t)N};
    cuuint64_t strides[3] = {(cuuint64_t)D * 2, (cuuint64_t)H * D * 2, (cuuint64_t)S * H * D * 2};
    cuuint32_t box[4] = {64, 1, (cuuint32_t)BN, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = fn(map, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void *>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(SPT_ERR_CUDA, "sparse_attn: cuTensorMapEncodeTiled failed (%d)", (int)r);
    return SPT_OK;
}

// head dim 64: the backward runs on the 128 x 128-tile kernels of attn_tc128.cu unless SPT_ATTN_TILE=64 (A/B switch); the
// forward stays on the 128 x 64 two-CTAs-per-SM kernel: it is bound by the exp unit, not by the tensor pipe, and a
// 128 x 128 forward measured slower (DESIGN.md section 4.1)
static bool tile128() {
    static const bool on = [] { const char *e = getenv("SPT_ATTN_TILE"); return !(e && atoi(e) == 64); }();
    return on;
}
struct SideStream {
    cudaStream_t stream = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
};
// one side stream + event pair per device, created on first use (never inside a capture: creation is not a stream operation)
static std::mutex g_side_mu;   // held while a fork / launch / join sequence is enqueued: callers on different streams share the side stream
static SideStream *side_stream(cudaStream_t caller) {   // g_side_mu held
    static SideStream table[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    SideStream &s = table[dev];
    if (!s.stream) {
        // never create streams / events while the caller's stream is being captured (an API call that is not a stream
        // operation can invalidate a global-mode capture): that one call runs the two kernels back to back
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(caller, &cap) != cudaSuccess || cap != cudaStreamCaptureStatusNone) return nullptr;
        if (cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
        if (cudaEventCreateWithFlags(&s.fork, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&s.join, cudaEventDisableTiming) != cudaSuccess) {
            s.stream = nullptr;
            return nullptr;
        }
    }
    return &s;
}

// k: the key tensor (read by the fp16 forward only, for its row scales)
template <int D, typename T>
static int launch_fwd(const CUtensorMap &mq, const CUtensorMap &mk, const CUtensorMap &mv, const uint32_t *mask,
                      const int32_t *extra0, T *y, float *zsum, int B, int S, int H, float scale, float clamp,
                      int y_transposed, const T *k, cudaStream_t st) {
    cudaFuncSetAttribute(attn_fwd_tc_kernel<D, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, Dim<D>::FWD_SMEM);
    attn_fwd_tc_kernel<D, T><<<dim3(B, S / BM), THREADS, Dim<D>::FWD_SMEM, st>>>(mq, mk, mv, mask, extra0, y, zsum, S, H,
                                                                                 scale * LOG2E, clamp * LOG2E, y_transposed, k);
    return after_launch("attn_fwd_tc_kernel");
}

template <int D, typename T>
static int launch_prep(const T *y, const T *grad_y, const float *zsum, float *delta, T *dys, int B, int S, int H,
                       int y_transposed, cudaStream_t st) {
    if (y_transposed) {
        attn_bwd_prep_t_kernel<D, T><<<dim3(S / 64, B), 256, 0, st>>>(grad_y, y, zsum, delta, dys, S, H);
        return after_launch("attn_bwd_prep_t_kernel");
    }
    const int64_t rows = (int64_t)B * S;
    constexpr int RPB = 256 / Dim<D>::PREP_LANES;
    attn_bwd_prep_kernel<D, T><<<(unsigned)((rows + RPB - 1) / RPB), 256, 0, st>>>(grad_y, y, zsum, delta, dys, rows, S, H);
    return after_launch("attn_bwd_prep_kernel");
}

template <int D, typename T>
static int launch_bwd(const CUtensorMap &mq, const CUtensorMap &mk, const CUtensorMap &mv, const CUtensorMap &md,
                      const uint32_t *mask, const int32_t *extra0, const float *delta, const float *zsum, T *gq, T *gk,
                      T *gv, int B, int S, int H, float scale, float clamp, cudaStream_t st) {
    if (D == 64 && tile128()) {
        {
            // The dK/dV and the dQ kernel are independent: the dQ kernel goes to a side stream (fork / join with events,
            // which a stream capture records as graph edges), so its CTAs start on each SM as that SM's dK/dV CTA retires
            // instead of after the whole grid has drained (both are one-CTA-per-SM persistent grids: they never share an SM).
            std::lock_guard<std::mutex> lock(g_side_mu);
            SideStream *ss = side_stream(st);
            if (ss) {
                if (cudaEventRecord(ss->fork, st) != cudaSuccess || cudaStreamWaitEvent(ss->stream, ss->fork, 0) != cudaSuccess)
                    return fail(SPT_ERR_CUDA, "sparse_attn_bwd: fork to the side stream failed");
                int rc = attn_tc128::launch_bwd_kv128(mq, mk, mv, md, mask, extra0, delta, zsum, gk, gv, B, S, H, scale, clamp, st);
                if (rc != SPT_OK) return rc;
                rc = attn_tc128::launch_bwd_q128(mq, mk, mv, md, mask, extra0, delta, zsum, gq, B, S, H, scale, clamp, ss->stream);
                if (rc != SPT_OK) return rc;
                if (cudaEventRecord(ss->join, ss->stream) != cudaSuccess || cudaStreamWaitEvent(st, ss->join, 0) != cudaSuccess)
                    return fail(SPT_ERR_CUDA, "sparse_attn_bwd: join of the side stream failed");
                return SPT_OK;
            }
        }
        // no side stream (it is never created during a capture, so a process whose first backward is captured gets
        // here): one kernel after the other on the caller's stream
        const int rc = attn_tc128::launch_bwd_kv128(mq, mk, mv, md, mask, extra0, delta, zsum, gk, gv, B, S, H, scale, clamp, st);
        if (rc != SPT_OK) return rc;
        return attn_tc128::launch_bwd_q128(mq, mk, mv, md, mask, extra0, delta, zsum, gq, B, S, H, scale, clamp, st);
    }
    constexpr int kv_smem = Dim<D>::BWD_SMEM + (is_f16<T> ? STAGES * BN * 4 : 0);      // fp16: the rows' -o per stage
    cudaFuncSetAttribute(attn_bwd_kv_tc_kernel<D, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, kv_smem);
    attn_bwd_kv_tc_kernel<D, T><<<dim3(B, S / BM), THREADS, kv_smem, st>>>(
        mq, mk, mv, md, mask, extra0, delta, gk, gv, S, H, scale, scale * LOG2E, clamp * LOG2E, zsum);
    SPT_LAUNCH_CHECK("attn_bwd_kv_tc_kernel");
    cudaFuncSetAttribute(attn_bwd_q_tc_kernel<D, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, Dim<D>::BWD_SMEM);
    attn_bwd_q_tc_kernel<D, T><<<dim3(B, S / BM), THREADS, Dim<D>::BWD_SMEM, st>>>(
        mq, mk, mv, md, mask, extra0, delta, gq, S, H, scale, scale * LOG2E, clamp * LOG2E, zsum);
    SPT_LAUNCH_CHECK("attn_bwd_q_tc_kernel");
    return SPT_OK;
}

// ---- packed variable-length sequences: q, k, v [1, T, H, D]; grids (H, work-list capacity) -----------------------------
// Every head dim runs the 128 x 64 kernels (the persistent 128 x 128 kernels of attn_tc128.cu have no varlen form).
template <int D, typename T>
static int launch_fwd_varlen(const CUtensorMap &mq, const CUtensorMap &mk, const CUtensorMap &mv, const uint32_t *mask,
                             const int32_t *extra0, T *y, float *zsum, const Varlen &vl, int cap, int S, int H, float scale,
                             float clamp, int y_transposed, const T *k, cudaStream_t st) {
    cudaFuncSetAttribute(attn_fwd_tc_kernel<D, T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Dim<D>::FWD_SMEM);
    attn_fwd_tc_kernel<D, T, true><<<dim3(H, cap), THREADS, Dim<D>::FWD_SMEM, st>>>(
        mq, mk, mv, mask, extra0, y, zsum, S, H, scale * LOG2E, clamp * LOG2E, y_transposed, k, vl);
    return after_launch("attn_fwd_tc_kernel(varlen)");
}

template <int D, typename T>
static int launch_prep_varlen(const T *y, const T *grad_y, const float *zsum, float *delta, T *dys, const Varlen &vl, int cap,
                              int S, int H, int y_transposed, cudaStream_t st) {
    if (!y_transposed) return launch_prep<D, T>(y, grad_y, zsum, delta, dys, H, S, H, 0, st);   // row-wise: N = 1, S = T
    attn_bwd_prep_t_kernel<D, T, true><<<dim3(2 * cap, H), 256, 0, st>>>(grad_y, y, zsum, delta, dys, S, H, vl);
    return after_launch("attn_bwd_prep_t_kernel(varlen)");
}

template <int D, typename T>
static int launch_bwd_varlen(const CUtensorMap &mq, const CUtensorMap &mk, const CUtensorMap &mv, const CUtensorMap &md,
                             const uint32_t *mask, const int32_t *extra0, const float *delta, const float *zsum, T *gq, T *gk,
                             T *gv, const Varlen &vl, int cap, int S, int H, float scale, float clamp, cudaStream_t st) {
    constexpr int kv_smem = Dim<D>::BWD_SMEM + (is_f16<T> ? STAGES * BN * 4 : 0);      // fp16: the rows' -o per stage
    cudaFuncSetAttribute(attn_bwd_kv_tc_kernel<D, T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kv_smem);
    attn_bwd_kv_tc_kernel<D, T, true><<<dim3(H, cap), THREADS, kv_smem, st>>>(
        mq, mk, mv, md, mask, extra0, delta, gk, gv, S, H, scale, scale * LOG2E, clamp * LOG2E, zsum, vl);
    SPT_LAUNCH_CHECK("attn_bwd_kv_tc_kernel(varlen)");
    cudaFuncSetAttribute(attn_bwd_q_tc_kernel<D, T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Dim<D>::BWD_SMEM);
    attn_bwd_q_tc_kernel<D, T, true><<<dim3(H, cap), THREADS, Dim<D>::BWD_SMEM, st>>>(
        mq, mk, mv, md, mask, extra0, delta, gq, S, H, scale, scale * LOG2E, clamp * LOG2E, zsum, vl);
    SPT_LAUNCH_CHECK("attn_bwd_q_tc_kernel(varlen)");
    return SPT_OK;
}

}  // namespace attn_tc
}  // namespace spt

using namespace spt;

static int check_attn_type(const char *what, int d, int dtype, float clamp) {
    if (dtype != SPT_BF16 && dtype != SPT_F16)
        return fail(SPT_ERR_UNSUPPORTED, "%s: only bf16 and fp16 are supported on the fused path", what);
    if (dtype == SPT_F16 && !(clamp >= 0.0f && clamp <= attn_tc::F16_MAX_CLAMP))
        return fail(SPT_ERR_UNSUPPORTED, "%s: fp16 needs 0 <= clamp <= %g (got %g)", what, (double)attn_tc::F16_MAX_CLAMP, (double)clamp);
    if (d != 64 && d != 80 && d != 128)
        return fail(SPT_ERR_UNSUPPORTED, "%s: head dim %d not supported (64, 80 or 128)", what, d);
    return SPT_OK;
}

static int check_attn_args(const char *what, int B, int S, int d, int H, int dtype, float clamp) {
    const int rc = check_attn_type(what, d, dtype, clamp);
    if (rc != SPT_OK) return rc;
    if (B < 1 || B > 65535 || S < 128 || S % 128 != 0)
        return fail(SPT_ERR_INVALID_ARGUMENT, "%s: need 1 <= B <= 65535 and S a positive multiple of 128 (B=%d S=%d)", what, B, S);
    if (H < 1 || B % H != 0)
        return fail(SPT_ERR_INVALID_ARGUMENT, "%s: B=%d must be a multiple of the interleaved head count H=%d", what, B, H);
    return SPT_OK;
}

template <typename T>
static int attn_fwd_typed(const CUtensorMap &mq, const CUtensorMap &mk, const CUtensorMap &mv, const uint32_t *mask,
                          const int32_t *extra0, void *y, float *zsum, int B, int S, int d, int H, float scale, float clamp,
                          int yt, const void *k, cudaStream_t st) {
    T *yy = (T *)y;
    const T *kk = (const T *)k;
    if (d == 64) return attn_tc::launch_fwd<64, T>(mq, mk, mv, mask, extra0, yy, zsum, B, S, H, scale, clamp, yt, kk, st);
    if (d == 80) return attn_tc::launch_fwd<80, T>(mq, mk, mv, mask, extra0, yy, zsum, B, S, H, scale, clamp, yt, kk, st);
    return attn_tc::launch_fwd<128, T>(mq, mk, mv, mask, extra0, yy, zsum, B, S, H, scale, clamp, yt, kk, st);
}

// the backward after the argument checks: row kernel, tensor maps, dK/dV + dQ kernels
template <typename T>
static int attn_bwd_typed(const void *q, const void *k, const void *v, const void *y, const void *grad_y,
                          const uint32_t *mask, const int32_t *extra0, const float *zsum, void *grad_q, void *grad_k,
                          void *grad_v, void *workspace, int B, int S, int d, int H, float scale, float clamp, int yt,
                          cudaStream_t st) {
    constexpr bool f16 = attn_tc::is_f16<T>;
    float *delta = (float *)workspace;
    T *dys = (T *)((char *)workspace + (size_t)B * S * sizeof(float));
    // the row kernel goes first: besides producing dO' and delta' it is a runtime-API launch, which binds the
    // device's primary context to this (autograd worker) thread before the driver-API tensor-map encoder runs
    int rc = d == 64   ? attn_tc::launch_prep<64, T>((const T *)y, (const T *)grad_y, zsum, delta, dys, B, S, H, yt, st)
             : d == 80 ? attn_tc::launch_prep<80, T>((const T *)y, (const T *)grad_y, zsum, delta, dys, B, S, H, yt, st)
                       : attn_tc::launch_prep<128, T>((const T *)y, (const T *)grad_y, zsum, delta, dys, B, S, H, yt, st);
    if (rc != SPT_OK) return rc;
    CUtensorMap mq, mk, mv, md;
    if ((rc = attn_tc::make_map(&mq, q, B / H, S, H, d, f16)) != SPT_OK) return rc;
    if ((rc = attn_tc::make_map(&mk, k, B / H, S, H, d, f16)) != SPT_OK) return rc;
    if ((rc = attn_tc::make_map(&mv, v, B / H, S, H, d, f16)) != SPT_OK) return rc;
    if ((rc = attn_tc::make_map(&md, dys, B / H, S, H, d, f16)) != SPT_OK) return rc;
    T *gq = (T *)grad_q, *gk = (T *)grad_k, *gv = (T *)grad_v;
    if (d == 64)
        return attn_tc::launch_bwd<64, T>(mq, mk, mv, md, mask, extra0, delta, zsum, gq, gk, gv, B, S, H, scale, clamp, st);
    if (d == 80)
        return attn_tc::launch_bwd<80, T>(mq, mk, mv, md, mask, extra0, delta, zsum, gq, gk, gv, B, S, H, scale, clamp, st);
    return attn_tc::launch_bwd<128, T>(mq, mk, mv, md, mask, extra0, delta, zsum, gq, gk, gv, B, S, H, scale, clamp, st);
}

extern "C" int spt_sparse_attn_fwd(const void *q, const void *k, const void *v, const uint32_t *mask,
                                   const int32_t *extra0, void *y, float *zsum, int B, int S, int d, int H,
                                   float scale, float clamp, int dtype, spt_stream_t stream) {
    return spt_sparse_attn_fwd_ex(q, k, v, mask, extra0, y, zsum, B, S, d, H, scale, clamp, dtype, 0, stream);
}

extern "C" int spt_sparse_attn_fwd_ex(const void *q, const void *k, const void *v, const uint32_t *mask,
                                      const int32_t *extra0, void *y, float *zsum, int B, int S, int d, int H,
                                      float scale, float clamp, int dtype, int flags, spt_stream_t stream) {
    SPT_REQUIRE(q && k && v && mask && extra0 && y && zsum, "sparse_attn_fwd: null pointer");
    const int yt = (flags & SPT_ATTN_Y_TRANSPOSED) ? 1 : 0;
    int rc = check_attn_args("sparse_attn_fwd", B, S, d, H, dtype, clamp);
    if (rc != SPT_OK) return rc;
    SPT_REQUIRE(((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)y) % 16 == 0, "sparse_attn_fwd: operands must be 16-byte aligned");
    const bool f16 = dtype == SPT_F16;
    CUtensorMap mq, mk, mv;
    if ((rc = attn_tc::make_map(&mq, q, B / H, S, H, d, f16)) != SPT_OK) return rc;
    if ((rc = attn_tc::make_map(&mk, k, B / H, S, H, d, f16)) != SPT_OK) return rc;
    if ((rc = attn_tc::make_map(&mv, v, B / H, S, H, d, f16)) != SPT_OK) return rc;
    return f16 ? attn_fwd_typed<__half>(mq, mk, mv, mask, extra0, y, zsum, B, S, d, H, scale, clamp, yt, k, as_stream(stream))
               : attn_fwd_typed<__nv_bfloat16>(mq, mk, mv, mask, extra0, y, zsum, B, S, d, H, scale, clamp, yt, k, as_stream(stream));
}

// diagnostics: phase timers of the attention kernels (all zeros unless built with -DSPT_ATTN_PROF); reset != 0 clears them
extern "C" int spt_debug_attn_prof(unsigned long long *out48, int reset) {
    if (reset & 2) return attn_tc128::read_prof(out48, reset & 1);      // bit 1: the 128 x 128-tile kernels' counters
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

// workspace: delta' [B, S] fp32, then dO' (bf16 / fp16, same shape as grad_y; sized for the largest head dim)
extern "C" size_t spt_sparse_attn_bwd_workspace_bytes(int B, int S) {
    return (size_t)B * S * sizeof(float) + (size_t)B * S * 128 * 2;
}

extern "C" int spt_sparse_attn_bwd(const void *q, const void *k, const void *v, const void *y, const void *grad_y,
                                   const uint32_t *mask, const int32_t *extra0, const float *zsum, void *grad_q,
                                   void *grad_k, void *grad_v, void *workspace, int B, int S, int d, int H,
                                   float scale, float clamp, int dtype, spt_stream_t stream) {
    return spt_sparse_attn_bwd_ex(q, k, v, y, grad_y, mask, extra0, zsum, grad_q, grad_k, grad_v, workspace, B, S, d, H,
                                  scale, clamp, dtype, 0, stream);
}

extern "C" int spt_sparse_attn_bwd_ex(const void *q, const void *k, const void *v, const void *y, const void *grad_y,
                                      const uint32_t *mask, const int32_t *extra0, const float *zsum, void *grad_q,
                                      void *grad_k, void *grad_v, void *workspace, int B, int S, int d, int H,
                                      float scale, float clamp, int dtype, int flags, spt_stream_t stream) {
    const int yt = (flags & SPT_ATTN_Y_TRANSPOSED) ? 1 : 0;
    SPT_REQUIRE(q && k && v && y && grad_y && mask && extra0 && zsum && grad_q && grad_k && grad_v && workspace,
                "sparse_attn_bwd: null pointer");
    int rc = check_attn_args("sparse_attn_bwd", B, S, d, H, dtype, clamp);
    if (rc != SPT_OK) return rc;
    SPT_REQUIRE(((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)grad_y | (uintptr_t)workspace) % 16 == 0,
                "sparse_attn_bwd: operands must be 16-byte aligned");
    if (dtype == SPT_F16)
        return attn_bwd_typed<__half>(q, k, v, y, grad_y, mask, extra0, zsum, grad_q, grad_k, grad_v, workspace, B, S, d, H,
                                      scale, clamp, yt, as_stream(stream));
    return attn_bwd_typed<__nv_bfloat16>(q, k, v, y, grad_y, mask, extra0, zsum, grad_q, grad_k, grad_v, workspace, B, S, d,
                                         H, scale, clamp, yt, as_stream(stream));
}

// ---- packed variable-length sequences ----------------------------------------------------------------------------------
static attn_tc::Varlen varlen_of(const void *work, int max_seqlen) {
    const int32_t *w = (const int32_t *)work;
    return {reinterpret_cast<const int4 *>(w + 4), w, 4 * ((max_seqlen + 127) / 128)};
}

template <typename T>
static int attn_varlen_fwd_typed(const CUtensorMap &mq, const CUtensorMap &mk, const CUtensorMap &mv, const uint32_t *mask,
                                 const int32_t *extra0, void *y, float *zsum, const attn_tc::Varlen &vl, int cap, int S, int d,
                                 int H, float scale, float clamp, int yt, const void *k, cudaStream_t st) {
    T *yy = (T *)y;
    const T *kk = (const T *)k;
    if (d == 64) return attn_tc::launch_fwd_varlen<64, T>(mq, mk, mv, mask, extra0, yy, zsum, vl, cap, S, H, scale, clamp, yt, kk, st);
    if (d == 80) return attn_tc::launch_fwd_varlen<80, T>(mq, mk, mv, mask, extra0, yy, zsum, vl, cap, S, H, scale, clamp, yt, kk, st);
    return attn_tc::launch_fwd_varlen<128, T>(mq, mk, mv, mask, extra0, yy, zsum, vl, cap, S, H, scale, clamp, yt, kk, st);
}

extern "C" int spt_sparse_attn_varlen_fwd(const void *q, const void *k, const void *v, const uint32_t *mask,
                                          const int32_t *extra0, void *y, float *zsum, const void *work, int n_seq, int T,
                                          int max_seqlen, int d, int H, float scale, float clamp, int dtype, int flags,
                                          spt_stream_t stream) {
    const char *what = "sparse_attn_varlen_fwd";
    SPT_REQUIRE(q && k && v && mask && extra0 && y && zsum && work, "%s: null pointer", what);
    int rc = check_attn_type(what, d, dtype, clamp);
    if (rc != SPT_OK) return rc;
    if ((rc = check_varlen(what, n_seq, T, max_seqlen, H)) != SPT_OK) return rc;
    SPT_REQUIRE(((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)y | (uintptr_t)mask | (uintptr_t)work) % 16 == 0,
                "%s: operands must be 16-byte aligned", what);
    const int yt = (flags & SPT_ATTN_Y_TRANSPOSED) ? 1 : 0;
    const bool f16 = dtype == SPT_F16;
    CUtensorMap mq, mk, mv;
    if ((rc = attn_tc::make_map(&mq, q, 1, T, H, d, f16)) != SPT_OK) return rc;
    if ((rc = attn_tc::make_map(&mk, k, 1, T, H, d, f16)) != SPT_OK) return rc;
    if ((rc = attn_tc::make_map(&mv, v, 1, T, H, d, f16)) != SPT_OK) return rc;
    const attn_tc::Varlen vl = varlen_of(work, max_seqlen);
    const int cap = (int)varlen_capacity(n_seq, T);
    return f16 ? attn_varlen_fwd_typed<__half>(mq, mk, mv, mask, extra0, y, zsum, vl, cap, T, d, H, scale, clamp, yt, k, as_stream(stream))
               : attn_varlen_fwd_typed<__nv_bfloat16>(mq, mk, mv, mask, extra0, y, zsum, vl, cap, T, d, H, scale, clamp, yt, k,
                                                      as_stream(stream));
}

// workspace: delta' [H, T] fp32, then (16-byte aligned) dO' [T, H, d] (sized for the largest head dim)
static size_t varlen_delta_bytes(int T, int H) { return ((size_t)H * T * sizeof(float) + 15) & ~(size_t)15; }

extern "C" size_t spt_sparse_attn_varlen_bwd_workspace_bytes(int T, int H) {
    if (T < 1 || H < 1) return 16;
    return varlen_delta_bytes(T, H) + (size_t)H * T * 128 * 2;
}

template <typename T>
static int attn_varlen_bwd_typed(const void *q, const void *k, const void *v, const void *y, const void *grad_y,
                                 const uint32_t *mask, const int32_t *extra0, const float *zsum, void *grad_q, void *grad_k,
                                 void *grad_v, void *workspace, const attn_tc::Varlen &vl, int cap, int S, int d, int H,
                                 float scale, float clamp, int yt, cudaStream_t st) {
    constexpr bool f16 = attn_tc::is_f16<T>;
    float *delta = (float *)workspace;
    T *dys = (T *)((char *)workspace + varlen_delta_bytes(S, H));
    const T *yy = (const T *)y, *dy = (const T *)grad_y;
    // the row kernel goes first (it binds the primary context before the tensor-map encoder runs; see attn_bwd_typed)
    int rc = d == 64   ? attn_tc::launch_prep_varlen<64, T>(yy, dy, zsum, delta, dys, vl, cap, S, H, yt, st)
             : d == 80 ? attn_tc::launch_prep_varlen<80, T>(yy, dy, zsum, delta, dys, vl, cap, S, H, yt, st)
                       : attn_tc::launch_prep_varlen<128, T>(yy, dy, zsum, delta, dys, vl, cap, S, H, yt, st);
    if (rc != SPT_OK) return rc;
    CUtensorMap mq, mk, mv, md;
    if ((rc = attn_tc::make_map(&mq, q, 1, S, H, d, f16)) != SPT_OK) return rc;
    if ((rc = attn_tc::make_map(&mk, k, 1, S, H, d, f16)) != SPT_OK) return rc;
    if ((rc = attn_tc::make_map(&mv, v, 1, S, H, d, f16)) != SPT_OK) return rc;
    if ((rc = attn_tc::make_map(&md, dys, 1, S, H, d, f16)) != SPT_OK) return rc;
    T *gq = (T *)grad_q, *gk = (T *)grad_k, *gv = (T *)grad_v;
    if (d == 64)
        return attn_tc::launch_bwd_varlen<64, T>(mq, mk, mv, md, mask, extra0, delta, zsum, gq, gk, gv, vl, cap, S, H, scale, clamp, st);
    if (d == 80)
        return attn_tc::launch_bwd_varlen<80, T>(mq, mk, mv, md, mask, extra0, delta, zsum, gq, gk, gv, vl, cap, S, H, scale, clamp, st);
    return attn_tc::launch_bwd_varlen<128, T>(mq, mk, mv, md, mask, extra0, delta, zsum, gq, gk, gv, vl, cap, S, H, scale, clamp, st);
}

extern "C" int spt_sparse_attn_varlen_bwd(const void *q, const void *k, const void *v, const void *y, const void *grad_y,
                                          const uint32_t *mask, const int32_t *extra0, const float *zsum, void *grad_q,
                                          void *grad_k, void *grad_v, void *workspace, const void *work, int n_seq, int T,
                                          int max_seqlen, int d, int H, float scale, float clamp, int dtype, int flags,
                                          spt_stream_t stream) {
    const char *what = "sparse_attn_varlen_bwd";
    SPT_REQUIRE(q && k && v && y && grad_y && mask && extra0 && zsum && grad_q && grad_k && grad_v && workspace && work,
                "%s: null pointer", what);
    int rc = check_attn_type(what, d, dtype, clamp);
    if (rc != SPT_OK) return rc;
    if ((rc = check_varlen(what, n_seq, T, max_seqlen, H)) != SPT_OK) return rc;
    SPT_REQUIRE(((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)y | (uintptr_t)grad_y | (uintptr_t)mask |
                 (uintptr_t)workspace | (uintptr_t)work | (uintptr_t)grad_q | (uintptr_t)grad_k | (uintptr_t)grad_v) % 16 == 0,
                "%s: operands must be 16-byte aligned", what);
    const int yt = (flags & SPT_ATTN_Y_TRANSPOSED) ? 1 : 0;
    const attn_tc::Varlen vl = varlen_of(work, max_seqlen);
    const int cap = (int)varlen_capacity(n_seq, T);
    if (dtype == SPT_F16)
        return attn_varlen_bwd_typed<__half>(q, k, v, y, grad_y, mask, extra0, zsum, grad_q, grad_k, grad_v, workspace, vl, cap, T, d,
                                             H, scale, clamp, yt, as_stream(stream));
    return attn_varlen_bwd_typed<__nv_bfloat16>(q, k, v, y, grad_y, mask, extra0, zsum, grad_q, grad_k, grad_v, workspace, vl, cap,
                                                T, d, H, scale, clamp, yt, as_stream(stream));
}
