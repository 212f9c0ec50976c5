// (2) lookup: PQ-code match counting + bucketed causal candidate selection -> fixed-stride CSR.
//
// Replaces lookup_forward_cuda (reference extension/lookup.cu:87-174).  The output is bit-exact with
// the reference kernel's semantics (restated in oracle/spt_oracle.py::lookup_spec):
//   row r, lane t in 0..3 owns keys j = t (mod 4), j <= r (ascending); bucket(j) = min(3, matches /
//   (m/4)); lane t fills output positions t, t+4, ... < min(r+1, nnz) with its keys ordered (bucket
//   desc, j asc); a (lane, bucket) list holds cap_t = nnz/4 (t < 2) or nnz/4 - 1 (t >= 2) entries;
//   overflow of lanes 2/3 lands on lane 1/0's last slot of that bucket (latest warp instruction
//   wins, the owner lane wins inside one instruction); unfilled positions are 0.
//
// B200 design (not a port of the reference's 64-thread, serial-per-lane kernel):
//   * Bit-sliced matching.  A pre-pass turns the key codes of a head into bitmaps
//       KB[s][w][v][t] : bit i set  <=>  key j = 128 w + 4 i + t has code v in subspace s,
//     i.e. the keys of one reference "lane" t are contiguous bits.  For query row r the match
//     indicator of subspace s over 32 keys is ONE shared-memory word KB[s][w][code_r(s)][t]; the m
//     words are summed with a carry-save adder tree (LOP3) and compared against the bucket
//     thresholds — about 1 integer instruction per (query, key) pair instead of ~20.
//   * One thread per (row, lane t): pass 1 popcounts bucket sizes, pass 2 walks set bits and writes
//     only the entries that survive (<= nnz/4 per thread) into a shared-memory row image, which is
//     flushed with coalesced 128-bit stores.  Every output element is written (zeros included).
//   * Codes >= 16 (or m without a specialised adder) take a generic compare path with the same
//     selection logic; the choice is made on the device through a flag, no host sync.
//
// Bound: integer-issue (S^2/2 * m bit-ops per head) and the S*nnz*4-byte index write; see DESIGN.md.
#include <cstdlib>

#include "common.cuh"

namespace spt {

constexpr int LK_ROWS = 32;                  // query rows per block
constexpr int LK_THREADS = LK_ROWS * 4;      // one thread per (row, lane t)
constexpr int LK_CV = 16;                    // code values covered by the bitmap path
constexpr int LK_WORD_U32 = LK_CV * 4;       // u32 per (subspace, 128-key word): [v][t]

// Packed variable-length batches (the VARLEN instantiations, spt_lookup_mask_varlen_fwd): codes are [1, T, H, m] (S = T),
// blocks take items of the work list (varlen.cu: {first token, length, 128-row tile, bitmap word offset}) and exit past
// *count.  Keys are relative to the sequence start; a sequence's key bitmaps are words [offset, offset + tiles) of the
// head's bitmap row; mask rows are 4 `groups` words wide; nnz = length / coeff per sequence.
struct LkVarlen {
    const int4 *items;
    const int *count;
    int groups;
    int coeff;
};

// ------------------------------------------------------------------------------------------
// Pre-pass: key codes [B, S, m] -> bitmaps KB[b][s][w][v][t], overflow flag if any code >= 16.
// grid (W, B), block 128: warp = lane t, lane = bit i  (key j = 128 w + 4 i + t).
// ------------------------------------------------------------------------------------------
// VARLEN: grid (work-list capacity, H); item = one 128-key group of one sequence, keys past its end match nothing.
template <bool VARLEN = false>
__global__ void __launch_bounds__(128)
lookup_pack_kernel(const int32_t *__restrict__ key_codes, uint32_t *__restrict__ kb, int *__restrict__ flag,
                   int S, int m, int W, int H, const LkVarlen vl = {}) {
    int w = blockIdx.x, wo = blockIdx.x, start = 0, len = S;      // wo: the group's word in the bitmaps
    if constexpr (VARLEN) {
        if ((int)blockIdx.x >= *vl.count) return;
        const int4 it = vl.items[blockIdx.x];
        start = it.x, len = it.y, w = it.z, wo = it.w + it.z;
    }
    const int b = blockIdx.y;
    const int t = threadIdx.x >> 5, i = threadIdx.x & 31;
    const int j = 128 * w + 4 * i + t;
    // codes are [N, S, H, m] (heads interleaved; H = 1: [B, S, m])
    const int32_t *kp = key_codes + (((size_t)(b / H) * S + start + j) * H + (b % H)) * m;
    bool overflow = false;
    // m = 8 / 16 (the PQ shapes of the layer): the key's codes are fetched with 16-byte loads up front — the loop below
    // would otherwise issue one dependent 4-byte load per subspace between its ballots (a latency chain per block)
    int32_t pre[16];
    const bool fast = (m == 8 || m == 16) && (reinterpret_cast<uintptr_t>(key_codes) % 16 == 0);
    if (fast && j < len) {
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (q * 4 < m) {
                const int4 v = *reinterpret_cast<const int4 *>(kp + q * 4);
                pre[q * 4] = v.x; pre[q * 4 + 1] = v.y; pre[q * 4 + 2] = v.z; pre[q * 4 + 3] = v.w;
            }
    }
#pragma unroll 1
    for (int s0 = 0; s0 < m; s0 += 8) {
#pragma unroll
      for (int ss = 0; ss < 8; ++ss) {
        const int s = s0 + ss;
        if (s >= m) break;
        const unsigned code = (j < len) ? ((unsigned)(fast ? pre[s0 == 0 ? ss : ss + 8] : kp[s]) & 0xffffu) : 0xffffu;
        overflow |= (j < len) && (code >= (unsigned)LK_CV);
        // lane v (< 16) wants the mask of keys whose code is v: four ballots over the code's bits, each lane keeps or
        // complements them according to its own index (16 compare + ballot + select rounds took 770 instructions per warp)
        static_assert(LK_CV == 16, "four code bits");
        unsigned mine = __ballot_sync(FULL, code < (unsigned)LK_CV);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const unsigned bk = __ballot_sync(FULL, (code >> k) & 1u);
            mine &= ((i >> k) & 1) ? bk : ~bk;
        }
        if (i < LK_CV) kb[(((size_t)b * m + s) * W + wo) * LK_WORD_U32 + i * 4 + t] = mine;
      }
    }
    if (__any_sync(FULL, overflow) && i == 0) atomicOr(flag, 1);
}

// ------------------------------------------------------------------------------------------
// Bit-sliced population count of M one-bit inputs (32 keys per word) -> NB count bit-planes.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void full_add(uint32_t a, uint32_t b, uint32_t c, uint32_t &s, uint32_t &cy) {
    s = a ^ b ^ c;
    cy = (a & b) | (c & (a ^ b));
}

template <int M>
struct BitCount {
    static constexpr int NB = (M >= 32) ? 6 : (M >= 16) ? 5 : (M >= 8) ? 4 : (M >= 4) ? 3 : 2;
    // generic ripple-carry accumulate
    __device__ __forceinline__ static void run(const uint32_t (&x)[M], uint32_t (&bits)[NB]) {
#pragma unroll
        for (int b = 0; b < NB; ++b) bits[b] = 0;
#pragma unroll
        for (int i = 0; i < M; ++i) {
            uint32_t carry = x[i];
#pragma unroll
            for (int b = 0; b < NB; ++b) {
                const uint32_t t = bits[b] & carry;
                bits[b] ^= carry;
                carry = t;
            }
        }
    }
};

__device__ __forceinline__ void count8(const uint32_t *x, uint32_t *bits /*4*/) {
    uint32_t s0, c0, s1, c1, s2, c2, s4, c4;
    full_add(x[0], x[1], x[2], s0, c0);
    full_add(x[3], x[4], x[5], s1, c1);
    full_add(x[6], x[7], s0, s2, c2);
    bits[0] = s1 ^ s2;
    const uint32_t c3 = s1 & s2;
    full_add(c0, c1, c2, s4, c4);
    bits[1] = s4 ^ c3;
    const uint32_t c5 = s4 & c3;
    bits[2] = c4 ^ c5;
    bits[3] = c4 & c5;
}

template <>
struct BitCount<8> {
    static constexpr int NB = 4;
    __device__ __forceinline__ static void run(const uint32_t (&x)[8], uint32_t (&bits)[4]) { count8(x, bits); }
};

template <>
struct BitCount<16> {
    static constexpr int NB = 5;
    __device__ __forceinline__ static void run(const uint32_t (&x)[16], uint32_t (&bits)[5]) {
        uint32_t s[7], c[8];
#pragma unroll
        for (int i = 0; i < 5; ++i) full_add(x[3 * i], x[3 * i + 1], x[3 * i + 2], s[i], c[i]);
        full_add(s[0], s[1], s[2], s[5], c[5]);
        full_add(s[3], s[4], x[15], s[6], c[6]);
        bits[0] = s[5] ^ s[6];
        c[7] = s[5] & s[6];
        count8(c, bits + 1);
    }
};

// count >= T (compile-time T) on bit-planes, LSB first.
template <int NB>
__device__ __forceinline__ uint32_t ge_const(const uint32_t (&bits)[NB], int T) {
    uint32_t ge = 0xffffffffu;
#pragma unroll
    for (int b = 0; b < NB; ++b) ge = ((T >> b) & 1) ? (bits[b] & ge) : (bits[b] | ge);
    if (T >> NB) ge = 0;
    return ge;
}

// ------------------------------------------------------------------------------------------
// Bucket providers: masks[s] bit i set <=> own key index 32*w + i (j = 4*(32w+i) + t) is in bucket s.
// ------------------------------------------------------------------------------------------
template <int M>
struct BitmapMatcher {
    const uint32_t *s_kb;  // shared: [M][cw][16][4] for the current chunk
    int cw;                // words in the chunk
    int w0;                // first word of the chunk
    unsigned q[M];         // query codes (mod 2^16)
    int t;
    __device__ __forceinline__ void buckets(int w, uint32_t valid, uint32_t (&mask)[4]) const {
        uint32_t x[M];
#pragma unroll
        for (int s = 0; s < M; ++s)
            x[s] = (q[s] < (unsigned)LK_CV) ? s_kb[((s * cw + (w - w0)) * LK_CV + q[s]) * 4 + t] : 0u;
        uint32_t bits[BitCount<M>::NB];
        BitCount<M>::run(x, bits);
        constexpr int DIV = M / 4;
        const uint32_t g1 = ge_const(bits, DIV), g2 = ge_const(bits, 2 * DIV), g3 = ge_const(bits, 3 * DIV);
        mask[3] = g3 & valid;
        mask[2] = g2 & ~g3 & valid;
        mask[1] = g1 & ~g2 & valid;
        mask[0] = ~g1 & valid;
    }
};

struct GenericMatcher {
    const int32_t *kc;     // key codes of this head, row j at kc + j * kstride
    const uint16_t *s_q;   // shared: this row's query codes [m]
    int m, div, t, kstride;
    __device__ __forceinline__ void buckets(int w, uint32_t valid, uint32_t (&mask)[4]) const {
        mask[0] = mask[1] = mask[2] = mask[3] = 0;
        uint32_t v = valid;
        while (v) {
            const int i = __ffs(v) - 1;
            v &= v - 1;
            const int j = 4 * (32 * w + i) + t;
            const int32_t *kp = kc + (size_t)j * kstride;
            int cnt = 0;
            for (int s = 0; s < m; ++s) cnt += ((unsigned)s_q[s] == ((unsigned)kp[s] & 0xffffu));
            const int bucket = min(3, cnt / div);
            mask[bucket] |= 1u << i;
        }
    }
};

// ------------------------------------------------------------------------------------------
// Selection core shared by both paths.  Thread = (row, t).
// ------------------------------------------------------------------------------------------
struct LaneState {
    int len[4], take[4], start[4], done[4];
    int s_need, track, last_j;
};

// Bitmask output layout ("lane-major", S % 128 == 0): word 4 g + t of a row holds the keys
// 128 g + 4 i + t at bit i — exactly the words the (row, lane t) threads of this kernel work on.
__device__ __forceinline__ int mask_word(int j) { return ((j >> 7) << 2) | (j & 3); }
__device__ __forceinline__ int mask_bit(int j) { return (j & 127) >> 2; }

__device__ __forceinline__ uint32_t valid_mask(int w, int nkeys) {
    const int rem = nkeys - 32 * w;
    return rem >= 32 ? 0xffffffffu : (rem <= 0 ? 0u : ((1u << rem) - 1u));
}

__device__ __forceinline__ void plan_lane(LaneState &st, int t, int n_t, int quarter) {
    const int cap = (t < 2) ? quarter : quarter - 1;
    int rem = n_t, acc = 0;
    st.s_need = -1;
#pragma unroll
    for (int s = 3; s >= 0; --s) {
        const int stored = min(st.len[s], cap);
        st.take[s] = min(stored, rem);
        st.start[s] = acc;
        acc += st.take[s];
        rem -= st.take[s];
        st.done[s] = 0;
        if (t < 2 && st.take[s] == quarter) st.s_need = s;
    }
    // lanes 2/3 learn which bucket (if any) their partner (lane 3 - t == tid ^ 3) reads its clobbered slot from
    const int partner_need = __shfl_xor_sync(FULL, st.s_need, 3);
    st.track = -1;
#pragma unroll
    for (int s = 0; s < 4; ++s)
        if (partner_need == s && st.len[s] >= quarter) st.track = s;
    st.last_j = -1;
}

__device__ __forceinline__ void place_word(LaneState &st, const uint32_t (&mask)[4], int w, int t,
                                           uint16_t *row_img, uint32_t *row_bits) {
#pragma unroll
    for (int s = 3; s >= 0; --s) {
        uint32_t mk = mask[s];
        if (st.track == s && mk) st.last_j = 4 * (32 * w + 31 - __clz(mk)) + t;
        while (mk && st.done[s] < st.take[s]) {
            const int i = __ffs(mk) - 1;
            mk &= mk - 1;
            const int j = 4 * (32 * w + i) + t;
            row_img[t + 4 * (st.start[s] + st.done[s])] = (uint16_t)j;
            if (row_bits) atomicOr(&row_bits[mask_word(j)], 1u << mask_bit(j));
            st.done[s] += 1;
        }
    }
}

__device__ __forceinline__ void fix_clobber(const LaneState &st, int t, int quarter, uint16_t *row_img,
                                            uint32_t *row_bits) {
    const int recv = __shfl_xor_sync(FULL, st.track >= 0 ? st.last_j : -1, 3);
    if (st.s_need >= 0 && recv >= 0) {
        // The partner's overflow store lands after ours only if it belongs to a later warp
        // instruction of the reference kernel (keys 4g..4g+3 are one instruction); inside the same
        // instruction the lower lane (ours) survives — measured on B200, see oracle/spt_oracle_c.c.
        const int p = t + 4 * (quarter - 1);
        const int old = (int)row_img[p];
        if ((recv >> 2) > (old >> 2)) {
            row_img[p] = (uint16_t)recv;
            if (row_bits) {
                atomicAnd(&row_bits[mask_word(old)], ~(1u << mask_bit(old)));
                atomicOr(&row_bits[mask_word(recv)], 1u << mask_bit(recv));
            }
        }
    }
}

// bitmask image [LK_ROWS][S/32] -> mask_out[b][r][:]; extra0[b][r] = nnz - (#filled positions) is the
// number of zero-padding slots of the row, i.e. the extra multiplicity of key 0 in the CSR row.
__device__ __forceinline__ void flush_mask(const uint32_t *s_bits, uint32_t *mask_out, int b, int r0, int S) {
    const int words = S / 32;
    const int rows = min(LK_ROWS, S - r0);
    uint32_t *dst = mask_out + ((size_t)b * S + r0) * words;
    for (int i = threadIdx.x; i < rows * words; i += blockDim.x) dst[i] = s_bits[i];
}

// the same for a packed sequence: `rows` live rows of `words` words from dst on
__device__ __forceinline__ void flush_mask_rows(const uint32_t *s_bits, uint32_t *dst, int rows, int words) {
    for (int i = threadIdx.x; i < rows * words; i += blockDim.x) dst[i] = s_bits[i];
}

__device__ __forceinline__ void store_extra0(const LaneState &st, int32_t *extra0_out, int b, int r, int S, int nnz,
                                             bool live, int t) {
    int filled = st.take[0] + st.take[1] + st.take[2] + st.take[3];
    filled += __shfl_xor_sync(FULL, filled, 1);
    filled += __shfl_xor_sync(FULL, filled, 2);
    if (extra0_out && live && t == 0) extra0_out[(size_t)b * S + r] = nnz - filled;
}

__device__ __forceinline__ void flush_rows(const uint16_t *s_out, int32_t *out, int b, int r0, int S, int nnz) {
    if (!out) return;
    const int per_row = nnz / 4;
    for (int idx = threadIdx.x; idx < LK_ROWS * per_row; idx += blockDim.x) {
        const int rl = idx / per_row, c4 = idx % per_row;
        const int r = r0 + rl;
        if (r >= S) break;
        const uint2 v = *reinterpret_cast<const uint2 *>(s_out + rl * nnz + 4 * c4);
        int4 o;
        o.x = v.x & 0xffff; o.y = v.x >> 16; o.z = v.y & 0xffff; o.w = v.y >> 16;
        st_stream(reinterpret_cast<int4 *>(out + ((size_t)b * S + r) * nnz) + c4, o);
    }
}

// ---- bitmap path ---------------------------------------------------------------------------
// smem: [ out image: LK_ROWS * nnz u16 ][ bitmaps: M * cw * 64 u32 ]
template <int M>
__global__ void __launch_bounds__(LK_THREADS)
lookup_bitmap_kernel(const int32_t *__restrict__ query_codes, const uint32_t *__restrict__ kb,
                     const int *__restrict__ flag, int32_t *__restrict__ out, uint32_t *__restrict__ mask_out,
                     int32_t *__restrict__ extra0_out, int S, int nnz, int W, int chunk_words, int H) {
    if (*flag) return;  // some key code >= 16: the generic kernel handles this call
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint16_t *s_out = reinterpret_cast<uint16_t *>(smem_raw);
    const size_t img_bytes = ((size_t)LK_ROWS * nnz * 2 + 15) & ~(size_t)15;
    const size_t bits_bytes = mask_out ? (size_t)LK_ROWS * (S / 32) * 4 : 0;
    uint32_t *s_bits = mask_out ? reinterpret_cast<uint32_t *>(smem_raw + img_bytes) : nullptr;
    uint32_t *s_kb = reinterpret_cast<uint32_t *>(smem_raw + img_bytes + bits_bytes);
    const int b = blockIdx.x;                      // grid (heads, row groups): every head's heaviest (last) row group first
    const int tile = gridDim.y - 1 - blockIdx.y;
    const int r0 = tile * LK_ROWS;
    const int rl = threadIdx.x >> 2, t = threadIdx.x & 3;
    const int r = r0 + rl;
    const bool live = r < S;
    const int quarter = nnz / 4;
    const int nkeys = (live && r >= t) ? (r - t) / 4 + 1 : 0;
    const int lim = live ? min(r + 1, nnz) : 0;
    const int n_t = lim > t ? (lim - t + 3) / 4 : 0;
    const int tile_words = min(W, (min(S, r0 + LK_ROWS) + 127) / 128);  // words any row of the tile needs

    for (int i = threadIdx.x; i < LK_ROWS * nnz / 2; i += blockDim.x) reinterpret_cast<uint32_t *>(s_out)[i] = 0;
    if (s_bits)
        for (int i = threadIdx.x; i < LK_ROWS * (S / 32); i += blockDim.x) s_bits[i] = 0;
    uint32_t *row_bits = s_bits ? s_bits + rl * (S / 32) : nullptr;

    BitmapMatcher<M> mt;
    mt.s_kb = s_kb;
    mt.t = t;
#pragma unroll
    for (int s = 0; s < M; ++s)
        mt.q[s] = live ? ((unsigned)query_codes[(((size_t)(b / H) * S + r) * H + (b % H)) * M + s] & 0xffffu) : 0xffffu;

    LaneState st;
#pragma unroll
    for (int s = 0; s < 4; ++s) st.len[s] = 0;
    const uint32_t *kb_head = kb + (size_t)b * M * W * LK_WORD_U32;
    const int my_words = (nkeys + 31) / 32;

    for (int pass = 0; pass < 2; ++pass) {
        for (int w0 = 0; w0 < tile_words; w0 += chunk_words) {
            const int cw = min(chunk_words, tile_words - w0);
            if (pass == 0 || tile_words > chunk_words) {  // single-chunk tiles keep the bitmaps for pass 2
                __syncthreads();
                const int per_s = cw * LK_WORD_U32 / 4;  // uint4 per subspace
                for (int i = threadIdx.x; i < M * per_s; i += blockDim.x) {
                    const int s = i / per_s, o = i % per_s;
                    reinterpret_cast<uint4 *>(s_kb)[s * per_s + o] =
                        reinterpret_cast<const uint4 *>(kb_head + ((size_t)s * W + w0) * LK_WORD_U32)[o];
                }
                __syncthreads();
            }
            mt.cw = cw;
            mt.w0 = w0;
            const int w_end = min(w0 + cw, my_words);
            for (int w = w0; w < w_end; ++w) {
                uint32_t mask[4];
                mt.buckets(w, valid_mask(w, nkeys), mask);
                if (pass == 0) {
#pragma unroll
                    for (int s = 0; s < 4; ++s) st.len[s] += __popc(mask[s]);
                } else {
                    place_word(st, mask, w, t, s_out + rl * nnz, row_bits);
                }
            }
        }
        if (pass == 0) plan_lane(st, t, n_t, quarter);
    }
    fix_clobber(st, t, quarter, s_out + rl * nnz, row_bits);
    store_extra0(st, extra0_out, b, r, S, nnz, live, t);
    __syncthreads();
    flush_rows(s_out, out, b, r0, S, nnz);
    if (s_bits) flush_mask(s_bits, mask_out, b, r0, S);
}

// ---- mask-only path (fused attention) -------------------------------------------------------------
// Same selection, but only the SET of selected keys is needed (bitmask + extra0), not their output
// positions.  A block owns one lane-major group of 128 query rows (512 threads, thread = (row, lane
// t)); every row of the group has the same number of 128-key words, so the block is perfectly
// balanced.  Pass 1 evaluates the adder tree ONCE per 32-key word and parks the bucket id of every
// key as two bit-planes in shared memory (bucket = 2 hi + lo) while popcounting the bucket sizes;
// after the plan (sizes -> quotas) pass 2 re-reads the planes and selects whole words: a bucket that
// is taken completely is OR-ed in, only the single partially taken bucket needs a "lowest q bits"
// trim.  The thread's words ARE the lane-major mask words — no per-key loop, no atomics.  Both passes
// are rolled loops (a few hundred instructions in total: the fully unrolled register version of this
// kernel spent 70 % of its issue slots waiting on instruction fetch).
constexpr int LKM_ROWS = 128;
constexpr int LKM_THREADS = LKM_ROWS * 4;

__device__ __forceinline__ uint32_t pick_lowest(uint32_t mask, int &quota) {
    if (quota <= 0 || mask == 0) return 0;
    const int c = __popc(mask);
    if (c <= quota) {
        quota -= c;
        return mask;
    }
    uint32_t r = 0, x = mask;
    for (int k = 0; k < quota; ++k) {
        r |= x & (0u - x);
        x &= x - 1;
    }
    quota = 0;
    return r;
}

template <int M>
__global__ void __launch_bounds__(LKM_THREADS)
lookup_maskonly_kernel(const int32_t *__restrict__ query_codes, const uint32_t *__restrict__ kb,
                       const int *__restrict__ flag, uint32_t *__restrict__ mask_out,
                       int32_t *__restrict__ extra0_out, int S, int nnz, int W, int H) {
    if (*flag) return;  // some key code >= 16: the generic kernel handles this call
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int b = blockIdx.x;                      // grid (heads, row groups): every head's heaviest (last) row group first
    const int tile = gridDim.y - 1 - blockIdx.y;
    const int tw = tile + 1;                       // 128-key words a row of this group can see
    uint32_t *s_kb = reinterpret_cast<uint32_t *>(smem_raw);                 // [M][tw][16][4]
    uint32_t *s_pl = s_kb + (size_t)M * tw * LK_WORD_U32;                    // [2 tw][LKM_THREADS]
    const int tid = threadIdx.x;
    const int rl = tid >> 2, t = tid & 3;
    const int r = tile * LKM_ROWS + rl;            // S % 128 == 0: every row is live
    const int quarter = nnz / 4;
    const int nkeys = r >= t ? (r - t) / 4 + 1 : 0;
    const int lim = min(r + 1, nnz);
    const int n_t = lim > t ? (lim - t + 3) / 4 : 0;

    {
        const uint32_t *kb_head = kb + (size_t)b * M * W * LK_WORD_U32;
        const int per_s = tw * LK_WORD_U32 / 4;  // uint4 per subspace
        for (int i = tid; i < M * per_s; i += LKM_THREADS) {
            const int s = i / per_s, o = i - s * per_s;
            reinterpret_cast<uint4 *>(s_kb)[i] = reinterpret_cast<const uint4 *>(kb_head + (size_t)s * W * LK_WORD_U32)[o];
        }
    }
    // this row's bitmap column of every subspace: s_kb[s][w][q_s][t] = s_kb[koff[s] + 64 w]; a query code the
    // bitmaps do not cover (>= 16) matches no key (qmask[s] = 0)
    uint32_t koff[M], qmask[M];
    {
        const int32_t *qp = query_codes + (((size_t)(b / H) * S + r) * H + (b % H)) * M;
#pragma unroll
        for (int s = 0; s < M; ++s) {
            const unsigned q = (unsigned)qp[s] & 0xffffu;
            qmask[s] = q < (unsigned)LK_CV ? 0xffffffffu : 0u;
            koff[s] = (uint32_t)((s * tw * LK_CV + (q & (LK_CV - 1))) * 4 + t);
        }
    }
    __syncthreads();

    constexpr int DIV = M / 4;
    LaneState st;
    int len1 = 0, len2 = 0, len3 = 0;
#pragma unroll 1
    for (int w = 0; w < tw; ++w) {
        const uint32_t valid = valid_mask(w, nkeys);
        uint32_t x[M];
#pragma unroll
        for (int s = 0; s < M; ++s) x[s] = s_kb[koff[s] + w * LK_WORD_U32] & qmask[s];
        uint32_t bits[BitCount<M>::NB];
        BitCount<M>::run(x, bits);
        const uint32_t g1 = ge_const(bits, DIV), g2 = ge_const(bits, 2 * DIV), g3 = ge_const(bits, 3 * DIV);
        s_pl[(2 * w) * LKM_THREADS + tid] = g1 ^ g2 ^ g3;   // lo (g3 <= g2 <= g1 as sets)
        s_pl[(2 * w + 1) * LKM_THREADS + tid] = g2;         // hi
        len3 += __popc(g3 & valid);
        len2 += __popc(g2 & valid);
        len1 += __popc(g1 & valid);
    }
    st.len[3] = len3;
    st.len[2] = len2 - len3;
    st.len[1] = len1 - len2;
    st.len[0] = nkeys - len1;
    plan_lane(st, t, n_t, quarter);

    int q3 = st.take[3], q2 = st.take[2], q1 = st.take[1], q0 = st.take[0];
    int j_old = -1, last_j = -1;
#pragma unroll 1
    for (int w = 0; w < tw; ++w) {
        const uint32_t valid = valid_mask(w, nkeys);
        const uint32_t lo = s_pl[(2 * w) * LKM_THREADS + tid], hi = s_pl[(2 * w + 1) * LKM_THREADS + tid];
        const uint32_t m3 = hi & lo & valid, m2 = hi & ~lo & valid, m1 = ~hi & lo & valid, m0 = ~hi & ~lo & valid;
        const uint32_t g3 = pick_lowest(m3, q3), g2 = pick_lowest(m2, q2), g1 = pick_lowest(m1, q1), g0 = pick_lowest(m0, q0);
        s_pl[(2 * w) * LKM_THREADS + tid] = g3 | g2 | g1 | g0;
        // own last TAKEN key of the bucket whose last slot the partner lane may clobber (see fix_clobber)
        const uint32_t gn = st.s_need == 3 ? g3 : st.s_need == 2 ? g2 : st.s_need == 1 ? g1 : st.s_need == 0 ? g0 : 0u;
        if (gn) j_old = 4 * (32 * w + 31 - __clz(gn)) + t;
        // own last key (taken or not) of the bucket the partner reads its clobbered slot from
        const uint32_t mt = st.track == 3 ? m3 : st.track == 2 ? m2 : st.track == 1 ? m1 : st.track == 0 ? m0 : 0u;
        if (mt) last_j = 4 * (32 * w + 31 - __clz(mt)) + t;
    }
    // lanes 2/3 report the last key of the tracked bucket; the owner (lane 1/0) swaps its own last taken key
    // of that bucket for it if a later warp instruction of the reference kernel would have overwritten the slot
    const int recv = __shfl_xor_sync(FULL, last_j, 3);
    const int swap_old = (st.s_need >= 0 && recv >= 0 && j_old >= 0 && (recv >> 2) > (j_old >> 2)) ? j_old : -1;
    const int partner_swapped = __shfl_xor_sync(FULL, swap_old >= 0 ? 1 : 0, 3);
    if (swap_old >= 0) s_pl[(2 * (swap_old >> 7)) * LKM_THREADS + tid] &= ~(1u << mask_bit(swap_old));
    if (partner_swapped && last_j >= 0) s_pl[(2 * (last_j >> 7)) * LKM_THREADS + tid] |= 1u << mask_bit(last_j);
    store_extra0(st, extra0_out, b, r, S, nnz, true, t);
    __syncthreads();

    // flush: thread -> (row, word w): 16 B = the four lane words; words the group cannot see are zero
    uint4 *dst = reinterpret_cast<uint4 *>(mask_out + ((size_t)b * S + (size_t)tile * LKM_ROWS) * (S / 32));
    for (int i = tid; i < LKM_ROWS * W; i += LKM_THREADS) {
        const int w = i / LKM_ROWS, row = i - w * LKM_ROWS;
        uint4 v = make_uint4(0, 0, 0, 0);
        if (w < tw) v = *reinterpret_cast<const uint4 *>(s_pl + (size_t)(2 * w) * LKM_THREADS + row * 4);
        dst[(size_t)row * W + w] = v;
    }
}

#ifndef SPT_LKM_UNROLL
#define SPT_LKM_UNROLL 2     // pass 1 of the mask-only kernel: 1 -> 0.1077 ms, 2 -> 0.104, 4 -> 0.105 at the bench shape
#endif
#ifndef SPT_LKM_UNROLL2
#define SPT_LKM_UNROLL2 2    // pass 2
#endif
constexpr int LKM_UNROLL_P1 = SPT_LKM_UNROLL, LKM_UNROLL_P2 = SPT_LKM_UNROLL2;   // loop unroll factors of the two passes (A/B)
// ---- mask-only path, second version ---------------------------------------------------------------
// Same algorithm and shared-memory layout as lookup_maskonly_kernel, written for instruction count (that kernel spends
// ~270 warp instructions per (thread, 32-key word); ncu: integer-issue bound):
//   * both passes handle the only partially valid word (the last one: words below the diagonal word are fully valid
//     for every row of the group) outside their loops — no per-word validity mask;
//   * pass 2 takes every completely selected bucket with three LOP3 (a per-thread all-ones / zero flag per bucket
//     muxed by the two bit-planes) and runs the "lowest q keys" selection only for the bucket that is cut, as a
//     five-step popcount search instead of a bit-by-bit loop (a second cut bucket — possible when a bucket overflows
//     its capacity — goes through the same code once more);
//   * the clobber bookkeeping (which needs the last key of two buckets) only runs in warps that have such a row.
__device__ __forceinline__ uint32_t lowest_bits(uint32_t m, int q) {        // the q lowest set bits of m, 0 < q < popc(m)
    uint32_t lowmask = 0;   // bits below the position reached so far
    int pos = 0;
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
        const uint32_t probe = ((1u << s) - 1u) << pos;
        const int c = __popc(m & probe);
        const bool up = q > c;          // the q-th bit lies above this probe window
        q -= up ? c : 0;
        lowmask |= up ? probe : 0u;
        pos += up ? s : 0;
    }
    // now q == 1 and the wanted bit is at `pos` (if set) — take everything below pos plus bit pos
    return m & (lowmask | (1u << pos));
}

template <int M, bool TRACK>
__device__ __forceinline__ void lkm2_select(uint32_t *s_pl, int tw, int tid, uint32_t last_valid, const int (&take)[4],
                                            const int (&len)[4], int s_need, int track, int t, int &j_old, int &last_j) {
    // per-bucket flags: F = taken completely, P = cut (0 < take < len)
    uint32_t F[4];
    int q[4];
    bool cut[4];
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        F[s] = (take[s] == len[s] && len[s] > 0) ? 0xffffffffu : 0u;
        cut[s] = take[s] > 0 && take[s] < len[s];
        q[s] = take[s];
    }
#pragma unroll LKM_UNROLL_P2
    for (int w = 0; w < tw; ++w) {
        const uint32_t lo = s_pl[(2 * w) * LKM_THREADS + tid], hi = s_pl[(2 * w + 1) * LKM_THREADS + tid];
        const uint32_t valid = (w == tw - 1) ? last_valid : 0xffffffffu;
        // completely taken buckets: bucket = 2 hi + lo
        const uint32_t fa = (lo & F[3]) | (~lo & F[2]), fb = (lo & F[1]) | (~lo & F[0]);
        uint32_t sel = ((hi & fa) | (~hi & fb)) & valid;
#pragma unroll
        for (int s = 3; s >= 0; --s) {
            if (cut[s] && q[s] > 0) {
                const uint32_t ms = ((s & 2) ? hi : ~hi) & ((s & 1) ? lo : ~lo) & valid;
                const int c = __popc(ms);
                if (c <= q[s]) {
                    sel |= ms;
                    q[s] -= c;
                } else {
                    sel |= lowest_bits(ms, q[s]);
                    q[s] = 0;
                }
            }
        }
        s_pl[(2 * w) * LKM_THREADS + tid] = sel;
        if (TRACK) {
            if (s_need >= 0) {
                const uint32_t ms = ((s_need & 2) ? hi : ~hi) & ((s_need & 1) ? lo : ~lo) & sel;
                if (ms) j_old = 4 * (32 * w + 31 - __clz(ms)) + t;
            }
            if (track >= 0) {
                const uint32_t mt = ((track & 2) ? hi : ~hi) & ((track & 1) ? lo : ~lo) & valid;
                if (mt) last_j = 4 * (32 * w + 31 - __clz(mt)) + t;
            }
        }
    }
}

// VARLEN: grid (H, work-list capacity); rows past the sequence end (whole warps: lengths are multiples of 32) select
// nothing and store nothing.
template <int M, bool VARLEN = false>
__global__ void __launch_bounds__(LKM_THREADS)
lookup_maskonly2_kernel(const int32_t *__restrict__ query_codes, const uint32_t *__restrict__ kb,
                        const int *__restrict__ flag, uint32_t *__restrict__ mask_out,
                        int32_t *__restrict__ extra0_out, int S, int nnz, int W, int H, const LkVarlen vl = {}) {
    if (*flag) return;  // some key code >= 16: the generic kernel handles this call
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int b = blockIdx.x;                      // grid (heads, row groups): every head's heaviest (last) row group first
    int tile = gridDim.y - 1 - blockIdx.y, start = 0, len = S, woff = 0, groups = W;
    if constexpr (VARLEN) {
        if ((int)blockIdx.y >= *vl.count) return;
        const int4 it = vl.items[blockIdx.y];
        start = it.x, len = it.y, tile = it.z, woff = it.w, groups = vl.groups, nnz = it.y / vl.coeff;
    }
    const int tw = tile + 1;                       // 128-key words a row of this group can see
    uint32_t *s_kb = reinterpret_cast<uint32_t *>(smem_raw);                 // [M][tw][16][4]
    uint32_t *s_pl = s_kb + (size_t)M * tw * LK_WORD_U32;                    // [2 tw][LKM_THREADS]
    const int tid = threadIdx.x;
    const int rl = tid >> 2, t = tid & 3;
    const int r = tile * LKM_ROWS + rl;
    const bool live = !VARLEN || r < len;          // fixed length: S % 128 == 0, every row is live
    const int quarter = nnz / 4;
    const int nkeys = (live && r >= t) ? (r - t) / 4 + 1 : 0;
    const int lim = live ? min(r + 1, nnz) : 0;
    const int n_t = lim > t ? (lim - t + 3) / 4 : 0;
    const uint32_t last_valid = valid_mask(tw - 1, nkeys);   // words 0 .. tw - 2 are fully valid for every row of the group

    {
        const uint32_t *kb_head = kb + (size_t)b * M * W * LK_WORD_U32;
        const int per_s = tw * LK_WORD_U32 / 4;  // uint4 per subspace
        for (int i = tid; i < M * per_s; i += LKM_THREADS) {
            const int s = i / per_s, o = i - s * per_s;
            reinterpret_cast<uint4 *>(s_kb)[i] = reinterpret_cast<const uint4 *>(kb_head + ((size_t)s * W + woff) * LK_WORD_U32)[o];
        }
    }
    // this row's bitmap column of every subspace: s_kb[s][w][q_s][t] = s_kb[koff[s] + 64 w]; a query code the bitmaps do
    // not cover (>= 16) matches no key: handled by clearing the loaded word (warp-uniformly skipped when no lane has one)
    uint32_t koff[M];
    uint32_t badq = 0;
    {
        const int32_t *qp = query_codes + (((size_t)(b / H) * S + start + r) * H + (b % H)) * M;
#pragma unroll
        for (int s = 0; s < M; ++s) {
            const unsigned qc = live ? (unsigned)qp[s] & 0xffffu : 0xffffu;
            badq |= (qc >= (unsigned)LK_CV) ? (1u << s) : 0u;
            koff[s] = (uint32_t)((s * tw * LK_CV + (qc & (LK_CV - 1))) * 4 + t);
        }
    }
    const bool any_bad = __any_sync(FULL, badq != 0);
    __syncthreads();

    constexpr int DIV = M / 4;
    int len1 = 0, len2 = 0, len3 = 0;
    const uint32_t *pw = s_kb;                      // warp-uniform word base
#pragma unroll LKM_UNROLL_P1
    for (int w = 0; w < tw; ++w, pw += LK_WORD_U32) {
        uint32_t x[M];
#pragma unroll
        for (int s = 0; s < M; ++s) x[s] = pw[koff[s]];
        if (any_bad) {
#pragma unroll
            for (int s = 0; s < M; ++s) x[s] = ((badq >> s) & 1u) ? 0u : x[s];
        }
        uint32_t bits[BitCount<M>::NB];
        BitCount<M>::run(x, bits);
        const uint32_t g1 = ge_const(bits, DIV), g2 = ge_const(bits, 2 * DIV), g3 = ge_const(bits, 3 * DIV);
        s_pl[(2 * w) * LKM_THREADS + tid] = g1 ^ g2 ^ g3;   // lo (g3 <= g2 <= g1 as sets)
        s_pl[(2 * w + 1) * LKM_THREADS + tid] = g2;         // hi
        const uint32_t valid = (w == tw - 1) ? last_valid : 0xffffffffu;
        len3 += __popc(g3 & valid);
        len2 += __popc(g2 & valid);
        len1 += __popc(g1 & valid);
    }
    LaneState st;
    st.len[3] = len3;
    st.len[2] = len2 - len3;
    st.len[1] = len1 - len2;
    st.len[0] = nkeys - len1;
    plan_lane(st, t, n_t, quarter);

    int j_old = -1, last_j = -1;
    if (__any_sync(FULL, st.s_need >= 0 || st.track >= 0))
        lkm2_select<M, true>(s_pl, tw, tid, last_valid, st.take, st.len, st.s_need, st.track, t, j_old, last_j);
    else
        lkm2_select<M, false>(s_pl, tw, tid, last_valid, st.take, st.len, st.s_need, st.track, t, j_old, last_j);
    // lanes 2/3 report the last key of the tracked bucket; the owner (lane 1/0) swaps its own last taken key
    // of that bucket for it if a later warp instruction of the reference kernel would have overwritten the slot
    const int recv = __shfl_xor_sync(FULL, last_j, 3);
    const int swap_old = (st.s_need >= 0 && recv >= 0 && j_old >= 0 && (recv >> 2) > (j_old >> 2)) ? j_old : -1;
    const int partner_swapped = __shfl_xor_sync(FULL, swap_old >= 0 ? 1 : 0, 3);
    if (swap_old >= 0) s_pl[(2 * (swap_old >> 7)) * LKM_THREADS + tid] &= ~(1u << mask_bit(swap_old));
    if (partner_swapped && last_j >= 0) s_pl[(2 * (last_j >> 7)) * LKM_THREADS + tid] |= 1u << mask_bit(last_j);
    store_extra0(st, extra0_out, b, start + r, S, nnz, live, t);
    __syncthreads();

    // flush: thread -> (row, word w): 16 B = the four lane words; words the group cannot see are zero
    uint4 *dst = reinterpret_cast<uint4 *>(mask_out + ((size_t)b * S + start + (size_t)tile * LKM_ROWS) * (VARLEN ? 4 * groups : S / 32));
    for (int i = tid; i < LKM_ROWS * groups; i += LKM_THREADS) {
        const int w = i / LKM_ROWS, row = i - w * LKM_ROWS;
        if (VARLEN && tile * LKM_ROWS + row >= len) continue;
        uint4 v = make_uint4(0, 0, 0, 0);
        if (w < tw) v = *reinterpret_cast<const uint4 *>(s_pl + (size_t)(2 * w) * LKM_THREADS + row * 4);
        dst[(size_t)row * groups + w] = v;
    }
}

// ---- mask-only path for long sequences ---------------------------------------------------------------
// lookup_maskonly2_kernel keeps two bit-planes per (thread, word) between its passes: 4 KB per word and block, i.e. its
// shared memory runs out beyond S 4096 (m 8).  This variant stores NO planes: pass 1 only counts, pass 2 evaluates the
// adder tree again (the bitmaps are in shared memory anyway) and selects; the selected words leave through a 16-word
// staging area.  ~1.7x the instructions per word of the plane kernel, but S 8192 no longer falls back to the
// index-emitting kernel (1.7 - 2.3 ms per 8192 tokens there).
constexpr int LKB_CHUNK = 16;

template <int M>
__device__ __forceinline__ void lkb_planes(const uint32_t *pw, const uint32_t (&koff)[M], bool any_bad, uint32_t badq,
                                           uint32_t &lo, uint32_t &hi, uint32_t &g1o, uint32_t &g3o) {
    constexpr int DIV = M / 4;
    uint32_t x[M];
#pragma unroll
    for (int s = 0; s < M; ++s) x[s] = pw[koff[s]];
    if (any_bad) {
#pragma unroll
        for (int s = 0; s < M; ++s) x[s] = ((badq >> s) & 1u) ? 0u : x[s];
    }
    uint32_t bits[BitCount<M>::NB];
    BitCount<M>::run(x, bits);
    const uint32_t g1 = ge_const(bits, DIV), g2 = ge_const(bits, 2 * DIV), g3 = ge_const(bits, 3 * DIV);
    lo = g1 ^ g2 ^ g3;
    hi = g2;
    g1o = g1;
    g3o = g3;
}

// ---- streaming: no length cap ------------------------------------------------------------------------
// STREAM keeps a head's bitmaps in global memory (L2 serves them: m * 256 B per 128-key word, 2 MiB per head at S 65536,
// m 16) and moves them through two shared-memory buffers of LKB_CHUNK words each, in both passes: chunk k + 1 is copied
// (cp.async) while chunk k is evaluated.  The chunks of pass 1 and pass 2 form one sequence 0 .. 2 nc - 1 (nc chunks per
// pass), chunk i in buffer i & 1.  Shared memory: (2 m LKB_CHUNK 256 + LKB_CHUNK LKM_THREADS 4) B whatever S is.
__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
__device__ __forceinline__ void cp_async_wait1() { asm volatile("cp.async.wait_group 1;\n" ::: "memory"); }

// issue chunk i of the sequence (an empty group past its end, so that wait_group 1 always means "chunk i - 1 landed")
template <int M>
__device__ __forceinline__ void lks_load(uint32_t *s_kb, const uint32_t *kb_head, int i, int nc, int tw, int W, int woff) {
    if (i < 2 * nc) {
        const int c0 = (i % nc) * LKB_CHUNK, cw = min(LKB_CHUNK, tw - c0);
        uint32_t *buf = s_kb + (size_t)(i & 1) * M * LKB_CHUNK * LK_WORD_U32;
        const int per_s = cw * LK_WORD_U32 / 4;  // uint4 per subspace
        for (int k = threadIdx.x; k < M * per_s; k += LKM_THREADS) {
            const int s = k / per_s, o = k - s * per_s;
            cp_async16(reinterpret_cast<uint4 *>(buf + (size_t)s * LKB_CHUNK * LK_WORD_U32) + o,
                       reinterpret_cast<const uint4 *>(kb_head + ((size_t)s * W + woff + c0) * LK_WORD_U32) + o);
        }
    }
    cp_async_commit();
}

// VARLEN: as lookup_maskonly2_kernel.  STREAM: two blocks per SM at m 8 / 10 (96 / 112 KB of shared memory each), one
// at m 16 (160 KB), which then needs more than 64 registers to keep from spilling.
template <int M, bool VARLEN = false, bool STREAM = false>
__global__ void __launch_bounds__(LKM_THREADS, STREAM ? (M == 16 ? 1 : 2) : 0)
lookup_maskonly_big_kernel(const int32_t *__restrict__ query_codes, const uint32_t *__restrict__ kb,
                           const int *__restrict__ flag, uint32_t *__restrict__ mask_out,
                           int32_t *__restrict__ extra0_out, int S, int nnz, int W, int H, const LkVarlen vl = {}) {
    if (*flag) return;  // some key code >= 16: the generic kernel handles this call
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int b = blockIdx.x;                      // grid (heads, row groups): every head's heaviest (last) row group first
    int tile = gridDim.y - 1 - blockIdx.y, start = 0, len = S, woff = 0, groups = W;
    if constexpr (VARLEN) {
        if ((int)blockIdx.y >= *vl.count) return;
        const int4 it = vl.items[blockIdx.y];
        start = it.x, len = it.y, tile = it.z, woff = it.w, groups = vl.groups, nnz = it.y / vl.coeff;
    }
    const int tw = tile + 1;                       // 128-key words a row of this group can see
    const int kw = STREAM ? LKB_CHUNK : tw;        // words per subspace in shared memory
    uint32_t *s_kb = reinterpret_cast<uint32_t *>(smem_raw);                 // [M][kw][16][4] (STREAM: two of them)
    uint32_t *s_out = s_kb + (size_t)(STREAM ? 2 : 1) * M * kw * LK_WORD_U32;  // [LKB_CHUNK][LKM_THREADS]
    const int tid = threadIdx.x;
    const int rl = tid >> 2, t = tid & 3;
    const int r = tile * LKM_ROWS + rl;
    const bool live = !VARLEN || r < len;
    const int live_rows = VARLEN ? min(LKM_ROWS, len - tile * LKM_ROWS) : LKM_ROWS;
    const int quarter = nnz / 4;
    const int nkeys = (live && r >= t) ? (r - t) / 4 + 1 : 0;
    const int lim = live ? min(r + 1, nnz) : 0;
    const int n_t = lim > t ? (lim - t + 3) / 4 : 0;
    const uint32_t last_valid = valid_mask(tw - 1, nkeys);
    const int nc = (tw + LKB_CHUNK - 1) / LKB_CHUNK;   // STREAM: chunks per pass
    if constexpr (STREAM) {
        lks_load<M>(s_kb, kb + (size_t)b * M * W * LK_WORD_U32, 0, nc, tw, W, woff);
    } else {
        const uint32_t *kb_head = kb + (size_t)b * M * W * LK_WORD_U32;
        const int per_s = tw * LK_WORD_U32 / 4;  // uint4 per subspace
        for (int i = tid; i < M * per_s; i += LKM_THREADS) {
            const int s = i / per_s, o = i - s * per_s;
            reinterpret_cast<uint4 *>(s_kb)[i] = reinterpret_cast<const uint4 *>(kb_head + ((size_t)s * W + woff) * LK_WORD_U32)[o];
        }
    }
    uint32_t koff[M];
    uint32_t badq = 0;
    {
        const int32_t *qp = query_codes + (((size_t)(b / H) * S + start + r) * H + (b % H)) * M;
#pragma unroll
        for (int s = 0; s < M; ++s) {
            const unsigned qc = live ? (unsigned)qp[s] & 0xffffu : 0xffffu;
            badq |= (qc >= (unsigned)LK_CV) ? (1u << s) : 0u;
            koff[s] = (uint32_t)((s * kw * LK_CV + (qc & (LK_CV - 1))) * 4 + t);
        }
    }
    const bool any_bad = __any_sync(FULL, badq != 0);
    if constexpr (!STREAM) __syncthreads();

    // pass 1: bucket sizes
    int len1 = 0, len2 = 0, len3 = 0;
    if constexpr (STREAM) {
        for (int c = 0; c < nc; ++c) {
            lks_load<M>(s_kb, kb + (size_t)b * M * W * LK_WORD_U32, c + 1, nc, tw, W, woff);
            cp_async_wait1();
            __syncthreads();
            const uint32_t *pw = s_kb + (size_t)(c & 1) * M * LKB_CHUNK * LK_WORD_U32;
            const int c1 = min(tw, (c + 1) * LKB_CHUNK);
#pragma unroll 1
            for (int w = c * LKB_CHUNK; w < c1; ++w, pw += LK_WORD_U32) {
                uint32_t lo, hi, g1, g3;
                lkb_planes<M>(pw, koff, any_bad, badq, lo, hi, g1, g3);
                const uint32_t valid = (w == tw - 1) ? last_valid : 0xffffffffu;
                len3 += __popc(g3 & valid);
                len2 += __popc(hi & valid);
                len1 += __popc(g1 & valid);
            }
            __syncthreads();   // buffer c & 1 is refilled by the next iteration's copy
        }
    } else {
        const uint32_t *pw = s_kb;
#pragma unroll 1
        for (int w = 0; w < tw; ++w, pw += LK_WORD_U32) {
            uint32_t lo, hi, g1, g3;
            lkb_planes<M>(pw, koff, any_bad, badq, lo, hi, g1, g3);
            const uint32_t valid = (w == tw - 1) ? last_valid : 0xffffffffu;
            len3 += __popc(g3 & valid);
            len2 += __popc(hi & valid);
            len1 += __popc(g1 & valid);
        }
    }
    LaneState st;
    st.len[3] = len3;
    st.len[2] = len2 - len3;
    st.len[1] = len1 - len2;
    st.len[0] = nkeys - len1;
    plan_lane(st, t, n_t, quarter);

    // pass 2: planes again, selection, chunked flush
    uint32_t F[4];
    int q[4];
    bool cut[4];
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        F[s] = (st.take[s] == st.len[s] && st.len[s] > 0) ? 0xffffffffu : 0u;
        cut[s] = st.take[s] > 0 && st.take[s] < st.len[s];
        q[s] = st.take[s];
    }
    const bool track = __any_sync(FULL, st.s_need >= 0 || st.track >= 0);
    int j_old = -1, last_j = -1;
    const int row_words = VARLEN ? 4 * groups : S / 32;
    uint4 *dst = reinterpret_cast<uint4 *>(mask_out + ((size_t)b * S + start + (size_t)tile * LKM_ROWS) * row_words);
    for (int c0 = 0; c0 < tw; c0 += LKB_CHUNK) {
        const int c1 = min(tw, c0 + LKB_CHUNK);
        const uint32_t *pw = s_kb + (size_t)c0 * LK_WORD_U32;
        if constexpr (STREAM) {
            const int i = nc + c0 / LKB_CHUNK;
            lks_load<M>(s_kb, kb + (size_t)b * M * W * LK_WORD_U32, i + 1, nc, tw, W, woff);
            cp_async_wait1();
            __syncthreads();
            pw = s_kb + (size_t)(i & 1) * M * LKB_CHUNK * LK_WORD_U32;
        }
#pragma unroll 1
        for (int w = c0; w < c1; ++w, pw += LK_WORD_U32) {
            uint32_t lo, hi, g1, g3;
            lkb_planes<M>(pw, koff, any_bad, badq, lo, hi, g1, g3);
            const uint32_t valid = (w == tw - 1) ? last_valid : 0xffffffffu;
            const uint32_t fa = (lo & F[3]) | (~lo & F[2]), fb = (lo & F[1]) | (~lo & F[0]);
            uint32_t sel = ((hi & fa) | (~hi & fb)) & valid;
#pragma unroll
            for (int s = 3; s >= 0; --s) {
                if (cut[s] && q[s] > 0) {
                    const uint32_t ms = ((s & 2) ? hi : ~hi) & ((s & 1) ? lo : ~lo) & valid;
                    const int c = __popc(ms);
                    if (c <= q[s]) {
                        sel |= ms;
                        q[s] -= c;
                    } else {
                        sel |= lowest_bits(ms, q[s]);
                        q[s] = 0;
                    }
                }
            }
            s_out[(w - c0) * LKM_THREADS + tid] = sel;
            if (track) {
                if (st.s_need >= 0) {
                    const uint32_t ms = ((st.s_need & 2) ? hi : ~hi) & ((st.s_need & 1) ? lo : ~lo) & sel;
                    if (ms) j_old = 4 * (32 * w + 31 - __clz(ms)) + t;
                }
                if (st.track >= 0) {
                    const uint32_t mt = ((st.track & 2) ? hi : ~hi) & ((st.track & 1) ? lo : ~lo) & valid;
                    if (mt) last_j = 4 * (32 * w + 31 - __clz(mt)) + t;
                }
            }
        }
        __syncthreads();
        for (int i = tid; i < LKM_ROWS * (c1 - c0); i += LKM_THREADS) {
            const int w = i / LKM_ROWS, row = i - w * LKM_ROWS;
            if (!VARLEN || row < live_rows) dst[(size_t)row * groups + c0 + w] = *reinterpret_cast<const uint4 *>(s_out + (size_t)w * LKM_THREADS + row * 4);
        }
        __syncthreads();
    }
    // words the group cannot see are zero
    for (int i = tid; i < LKM_ROWS * (groups - tw); i += LKM_THREADS) {
        const int w = i / LKM_ROWS, row = i - w * LKM_ROWS;
        if (!VARLEN || row < live_rows) dst[(size_t)row * groups + tw + w] = make_uint4(0, 0, 0, 0);
    }
    // clobber fix-up (see lookup_maskonly_kernel) on the flushed words: this thread's word of key j is mask word
    // 4 (j >> 7) + t of its row (every flush above is ordered before by the __syncthreads)
    const int recv = __shfl_xor_sync(FULL, last_j, 3);
    const int swap_old = (st.s_need >= 0 && recv >= 0 && j_old >= 0 && (recv >> 2) > (j_old >> 2)) ? j_old : -1;
    const int partner_swapped = __shfl_xor_sync(FULL, swap_old >= 0 ? 1 : 0, 3);
    uint32_t *my_row = mask_out + ((size_t)b * S + start + r) * row_words;   // (rows past a sequence end change nothing)
    if (swap_old >= 0) my_row[4 * (swap_old >> 7) + t] &= ~(1u << mask_bit(swap_old));
    if (partner_swapped && last_j >= 0) my_row[4 * (last_j >> 7) + t] |= 1u << mask_bit(last_j);
    store_extra0(st, extra0_out, b, start + r, S, nnz, live, t);
}

// ---- generic path ----------------------------------------------------------------------------
// smem: [ out image ][ query codes LK_ROWS * m u16 ]
// VARLEN (mask only): nnz is the largest per-sequence nnz (it sizes the image); items = (head, 32-row quarter of a
// work-list item), in work-list order.
template <bool VARLEN = false>
__global__ void __launch_bounds__(LK_THREADS)
lookup_generic_kernel(const int32_t *__restrict__ query_codes, const int32_t *__restrict__ key_codes,
                      const int *__restrict__ flag, int flag_expect, int32_t *__restrict__ out,
                      uint32_t *__restrict__ mask_out, int32_t *__restrict__ extra0_out, int S, int m, int nnz, int H,
                      int tiles, int nb, const LkVarlen vl = {}) {
    if (flag && (*flag != 0) != (flag_expect != 0)) return;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint16_t *s_out = reinterpret_cast<uint16_t *>(smem_raw);
    const int words = VARLEN ? 4 * vl.groups : S / 32;        // mask words per row
    const size_t img_bytes = ((size_t)LK_ROWS * nnz * 2 + 15) & ~(size_t)15;
    const size_t bits_bytes = mask_out ? (size_t)LK_ROWS * words * 4 : 0;
    uint32_t *s_bits = mask_out ? reinterpret_cast<uint32_t *>(smem_raw + img_bytes) : nullptr;
    uint16_t *s_q = reinterpret_cast<uint16_t *>(smem_raw + img_bytes + bits_bytes);
    if constexpr (VARLEN) tiles = 4 * *vl.count;
    // items = (head, row tile), the block strides over them: as the flag-guarded fallback behind the bitmap kernels it is
    // launched with a few hundred blocks (an early exit of one block per item cost 6 us per lookup at 128 heads)
    for (int item = blockIdx.x; item < tiles * nb; item += gridDim.x) {
    const int b = item / tiles;
    int tile = tiles - 1 - item % tiles, start = 0, len = S;
    if constexpr (VARLEN) {
        const int4 it = vl.items[(item % tiles) >> 2];
        start = it.x, len = it.y, tile = 4 * it.z + (item % tiles & 3), nnz = it.y / vl.coeff;
        if (tile * LK_ROWS >= len) continue;     // block-uniform
    }
    const int r0 = tile * LK_ROWS;
    const int rl = threadIdx.x >> 2, t = threadIdx.x & 3;
    const int r = r0 + rl;
    const bool live = r < len;
    const int quarter = nnz / 4;
    const int nkeys = (live && r >= t) ? (r - t) / 4 + 1 : 0;
    const int lim = live ? min(r + 1, nnz) : 0;
    const int n_t = lim > t ? (lim - t + 3) / 4 : 0;

    for (int i = threadIdx.x; i < LK_ROWS * nnz / 2; i += blockDim.x) reinterpret_cast<uint32_t *>(s_out)[i] = 0;
    if (s_bits)
        for (int i = threadIdx.x; i < LK_ROWS * words; i += blockDim.x) s_bits[i] = 0;
    uint32_t *row_bits = s_bits ? s_bits + rl * words : nullptr;
    for (int i = threadIdx.x; i < LK_ROWS * m; i += blockDim.x) {
        const int rr = r0 + i / m;
        s_q[i] = rr < len ? (uint16_t)((unsigned)query_codes[(((size_t)(b / H) * S + start + rr) * H + (b % H)) * m + i % m] & 0xffffu) : 0;
    }
    __syncthreads();

    GenericMatcher mt;
    mt.kc = key_codes + ((size_t)(b / H) * S * H + (b % H)) * m + (size_t)start * H * m;
    mt.kstride = H * m;
    mt.s_q = s_q + rl * m;
    mt.m = m;
    mt.div = m / 4;
    mt.t = t;
    LaneState st;
#pragma unroll
    for (int s = 0; s < 4; ++s) st.len[s] = 0;
    const int my_words = (nkeys + 31) / 32;
    for (int w = 0; w < my_words; ++w) {
        uint32_t mask[4];
        mt.buckets(w, valid_mask(w, nkeys), mask);
#pragma unroll
        for (int s = 0; s < 4; ++s) st.len[s] += __popc(mask[s]);
    }
    plan_lane(st, t, n_t, quarter);
    for (int w = 0; w < my_words; ++w) {
        uint32_t mask[4];
        mt.buckets(w, valid_mask(w, nkeys), mask);
        place_word(st, mask, w, t, s_out + rl * nnz, row_bits);
    }
    fix_clobber(st, t, quarter, s_out + rl * nnz, row_bits);
    store_extra0(st, extra0_out, b, start + r, S, nnz, live, t);
    __syncthreads();
    if constexpr (VARLEN) {
        flush_mask_rows(s_bits, mask_out + ((size_t)b * S + start + r0) * words, min(LK_ROWS, len - r0), words);
    } else {
        flush_rows(s_out, out, b, r0, S, nnz);
        if (s_bits) flush_mask(s_bits, mask_out, b, r0, S);
    }
    __syncthreads();
    }
}

static bool bitmap_m_supported(int m) { return m == 4 || m == 8 || m == 10 || m == 12 || m == 16 || m == 32; }

constexpr size_t LK_SMEM_BUDGET = 160 * 1024;

static size_t out_image_bytes(int nnz) { return (((size_t)LK_ROWS * nnz * 2) + 15) & ~(size_t)15; }

}  // namespace spt

using namespace spt;

extern "C" size_t spt_lookup_workspace_bytes(int B, int S, int m, int nnz) {
    (void)nnz;
    if (!bitmap_m_supported(m)) return 16;
    const size_t W = (size_t)(S + 127) / 128;
    return 16 + (size_t)B * m * W * LK_WORD_U32 * sizeof(uint32_t);
}

// shared memory of the streaming mask-only kernel (lookup_maskonly_big_kernel<M, VARLEN, true>), independent of S
static size_t lks_smem(int m) { return (size_t)2 * m * LKB_CHUNK * LK_WORD_U32 * 4 + (size_t)LKB_CHUNK * LKM_THREADS * 4; }

template <int M, bool VARLEN>
static void lks_launch(dim3 grid, const int32_t *qc, const uint32_t *kb, const int *flag, uint32_t *mask, int32_t *extra0,
                       int S, int nnz, int W, int H, cudaStream_t st, const LkVarlen &vl = {}) {
    const size_t smem = lks_smem(M);
    cudaFuncSetAttribute(lookup_maskonly_big_kernel<M, VARLEN, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    lookup_maskonly_big_kernel<M, VARLEN, true><<<grid, LKM_THREADS, smem, st>>>(qc, kb, flag, mask, extra0, S, nnz, W, H, vl);
}

// n_codewords: codes are < n_codewords (the _ex entry points), or -1: unknown.  Where the generic kernel's row images do not
// fit, only a promise of n_codewords <= 16 lets a call run: the fallback is skipped and a code >= 16 matches no key.
static int lookup_impl(const int32_t *query_codes, const int32_t *key_codes, int32_t *output, uint32_t *mask_out,
                       int32_t *extra0_out, void *workspace, int B, int S, int m, int nnz, int H, int n_codewords,
                       spt_stream_t stream) {
    SPT_REQUIRE(query_codes && key_codes && (output || mask_out), "lookup_fwd: null pointer");
    SPT_REQUIRE(H >= 1 && B % H == 0, "lookup_fwd: B=%d must be a multiple of the interleaved head count H=%d", B, H);
    SPT_REQUIRE(B >= 1 && S >= 1 && S <= 65536, "lookup_fwd: bad batch/seq (B=%d, S=%d; S must be <= 65536)", B, S);
    SPT_REQUIRE(B <= 65535, "lookup_fwd: batch %d exceeds grid limit", B);
    SPT_REQUIRE(m >= 4, "lookup_fwd: n_subspaces must be >= 4 (got %d)", m);
    SPT_REQUIRE(nnz >= 8 && nnz % 4 == 0 && nnz <= S, "lookup_fwd: nonzeros per row must be a multiple of 4 in [8, S] (got %d)", nnz);
    SPT_REQUIRE(!mask_out || (S % 128 == 0 && extra0_out), "lookup_fwd: bitmask output needs S %% 128 == 0 and extra0");
    const int tiles = (S + LK_ROWS - 1) / LK_ROWS;
    const size_t img = out_image_bytes(nnz) + (mask_out ? (size_t)LK_ROWS * (S / 32) * 4 : 0);
    const size_t gen_smem = img + (size_t)LK_ROWS * m * 2;
    const bool fb_fits = gen_smem <= 200 * 1024;
    // mask-only calls at m 8, 10, 16: the plane kernel, else the plane-free kernel, else the streaming kernel
    const bool mask_only = mask_out && !output && (m == 8 || m == 10 || m == 16);
    if (!fb_fits) {
        SPT_REQUIRE(n_codewords >= 0, "lookup_fwd: nnz=%d / S=%d too large for the shared-memory row images", nnz, S);
        if (n_codewords > LK_CV || !mask_only)
            return fail(SPT_ERR_UNSUPPORTED,
                        "lookup_mask_fwd_ex: S=%d, nnz=%d, m=%d runs only as a mask-only lookup with n_codewords <= %d "
                        "(got %d): the fallback for codes >= %d needs %zu bytes of row images, beyond its limit of %d",
                        S, nnz, m, LK_CV, n_codewords, LK_CV, gen_smem, 200 * 1024);
    }
    const int W = (S + 127) / 128;
    const size_t per_word = (size_t)m * LK_WORD_U32 * 4;   // bitmaps per 128-key word: m * 256 B
    const size_t msmem = (per_word + 2 * LKM_THREADS * 4) * (size_t)W;
    const size_t bsmem = per_word * (size_t)W + (size_t)LKB_CHUNK * LKM_THREADS * 4;
    if (bitmap_m_supported(m) && !mask_only)
        SPT_REQUIRE(img + per_word <= LK_SMEM_BUDGET, "lookup_fwd: nnz=%d / S=%d too large", nnz, S);
    cudaStream_t st = as_stream(stream);
    const unsigned grid = (unsigned)tiles * B;                                            // one block per (head, row tile)
    const unsigned fb_grid = grid < 2u * num_sms() ? grid : 2u * num_sms();               // the flag-guarded fallback
    if (fb_fits && gen_smem > 48 * 1024)
        cudaFuncSetAttribute(lookup_generic_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gen_smem);

    if (!bitmap_m_supported(m)) {
        lookup_generic_kernel<<<grid, LK_THREADS, gen_smem, st>>>(query_codes, key_codes, nullptr, 0, output, mask_out,
                                                                  extra0_out, S, m, nnz, H, tiles, B);
        SPT_LAUNCH_CHECK("lookup_generic_kernel");
        return SPT_OK;
    }
    SPT_REQUIRE(workspace, "lookup_fwd: workspace required");
    int *flag = reinterpret_cast<int *>(workspace);
    uint32_t *kb = reinterpret_cast<uint32_t *>(reinterpret_cast<char *>(workspace) + 16);
    cudaError_t e = cudaMemsetAsync(flag, 0, 16, st);
    if (e != cudaSuccess) return fail(SPT_ERR_CUDA, "lookup_fwd: memset: %s", cudaGetErrorString(e));
    lookup_pack_kernel<<<dim3(W, B), 128, 0, st>>>(key_codes, kb, flag, S, m, W, H);
    SPT_LAUNCH_CHECK("lookup_pack_kernel");
    // without the fallback the kernels read flag + 1, a word of the zeroed 16 bytes that nothing raises
    const int *kflag = fb_fits ? flag : flag + 1;

    // pick the chunk so that images + chunk fit the budget
    int chunk_words = (int)((LK_SMEM_BUDGET - img) / per_word);
    if (chunk_words > W) chunk_words = W;
    const size_t smem = img + per_word * chunk_words;
    if (mask_only) {
        const dim3 mgrid(B, S / LKM_ROWS);
        if (msmem <= 200 * 1024) {
            static const bool v1 = [] { const char *e = getenv("SPT_LOOKUP_MASK_V1"); return e && atoi(e) == 1; }();   // A/B switch
            if (v1 && m != 10) {
                if (m == 8) {
                    cudaFuncSetAttribute(lookup_maskonly_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msmem);
                    lookup_maskonly_kernel<8><<<mgrid, LKM_THREADS, msmem, st>>>(query_codes, kb, kflag, mask_out, extra0_out, S, nnz, W, H);
                } else {
                    cudaFuncSetAttribute(lookup_maskonly_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msmem);
                    lookup_maskonly_kernel<16><<<mgrid, LKM_THREADS, msmem, st>>>(query_codes, kb, kflag, mask_out, extra0_out, S, nnz, W, H);
                }
            } else if (m == 8) {
                cudaFuncSetAttribute(lookup_maskonly2_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msmem);
                lookup_maskonly2_kernel<8><<<mgrid, LKM_THREADS, msmem, st>>>(query_codes, kb, kflag, mask_out, extra0_out, S, nnz, W, H);
            } else if (m == 10) {       // head dim 80 (OPT-2.7B) at d_codeword 8
                cudaFuncSetAttribute(lookup_maskonly2_kernel<10>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msmem);
                lookup_maskonly2_kernel<10><<<mgrid, LKM_THREADS, msmem, st>>>(query_codes, kb, kflag, mask_out, extra0_out, S, nnz, W, H);
            } else {
                cudaFuncSetAttribute(lookup_maskonly2_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msmem);
                lookup_maskonly2_kernel<16><<<mgrid, LKM_THREADS, msmem, st>>>(query_codes, kb, kflag, mask_out, extra0_out, S, nnz, W, H);
            }
            SPT_LAUNCH_CHECK("lookup_maskonly_kernel");
        } else if (bsmem <= 200 * 1024) {
            // long sequences: the plane-free mask-only kernel (S 8192 at m 8)
            if (m == 8) {
                cudaFuncSetAttribute(lookup_maskonly_big_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bsmem);
                lookup_maskonly_big_kernel<8><<<mgrid, LKM_THREADS, bsmem, st>>>(query_codes, kb, kflag, mask_out, extra0_out, S, nnz, W, H);
            } else if (m == 10) {
                cudaFuncSetAttribute(lookup_maskonly_big_kernel<10>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bsmem);
                lookup_maskonly_big_kernel<10><<<mgrid, LKM_THREADS, bsmem, st>>>(query_codes, kb, kflag, mask_out, extra0_out, S, nnz, W, H);
            } else {
                cudaFuncSetAttribute(lookup_maskonly_big_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bsmem);
                lookup_maskonly_big_kernel<16><<<mgrid, LKM_THREADS, bsmem, st>>>(query_codes, kb, kflag, mask_out, extra0_out, S, nnz, W, H);
            }
            SPT_LAUNCH_CHECK("lookup_maskonly_big_kernel");
        } else {
            // longer still: the streaming kernel (its shared memory does not grow with S)
            if (m == 8)
                lks_launch<8, false>(mgrid, query_codes, kb, kflag, mask_out, extra0_out, S, nnz, W, H, st);
            else if (m == 10)
                lks_launch<10, false>(mgrid, query_codes, kb, kflag, mask_out, extra0_out, S, nnz, W, H, st);
            else
                lks_launch<16, false>(mgrid, query_codes, kb, kflag, mask_out, extra0_out, S, nnz, W, H, st);
            SPT_LAUNCH_CHECK("lookup_maskonly_big_kernel(stream)");
        }
        if (!fb_fits) return SPT_OK;
        lookup_generic_kernel<<<fb_grid, LK_THREADS, gen_smem, st>>>(query_codes, key_codes, flag, 1, output, mask_out,
                                                                  extra0_out, S, m, nnz, H, tiles, B);
        SPT_LAUNCH_CHECK("lookup_generic_kernel(fallback)");
        return SPT_OK;
    }
#define SPT_LK_CASE(MM)                                                                                          \
    case MM:                                                                                                     \
        if (smem > 48 * 1024)                                                                                    \
            cudaFuncSetAttribute(lookup_bitmap_kernel<MM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        lookup_bitmap_kernel<MM><<<dim3(B, tiles), LK_THREADS, smem, st>>>(query_codes, kb, flag, output, mask_out, extra0_out, S, \
                                                                 nnz, W, chunk_words, H);                        \
        break;
    switch (m) {
        SPT_LK_CASE(4)
        SPT_LK_CASE(8)
        SPT_LK_CASE(10)
        SPT_LK_CASE(12)
        SPT_LK_CASE(16)
        SPT_LK_CASE(32)
        default:
            return fail(SPT_ERR_UNSUPPORTED, "lookup_fwd: unreachable m=%d", m);
    }
#undef SPT_LK_CASE
    SPT_LAUNCH_CHECK("lookup_bitmap_kernel");
    lookup_generic_kernel<<<fb_grid, LK_THREADS, gen_smem, st>>>(query_codes, key_codes, flag, 1, output, mask_out,
                                                              extra0_out, S, m, nnz, H, tiles, B);
    SPT_LAUNCH_CHECK("lookup_generic_kernel(fallback)");
    return SPT_OK;
}

extern "C" int spt_lookup_fwd(const int32_t *query_codes, const int32_t *key_codes, int32_t *output, void *workspace,
                              int B, int S, int m, int nnz, spt_stream_t stream) {
    SPT_REQUIRE(output, "lookup_fwd: null output");
    return lookup_impl(query_codes, key_codes, output, nullptr, nullptr, workspace, B, S, m, nnz, 1, -1, stream);
}

extern "C" int spt_lookup_mask_fwd(const int32_t *query_codes, const int32_t *key_codes, int32_t *output,
                                   uint32_t *mask, int32_t *extra0, void *workspace, int B, int S, int m, int nnz,
                                   int H, spt_stream_t stream) {
    SPT_REQUIRE(mask && extra0, "lookup_mask_fwd: null mask / extra0");
    return lookup_impl(query_codes, key_codes, output, mask, extra0, workspace, B, S, m, nnz, H, -1, stream);
}

extern "C" int spt_lookup_mask_fwd_ex(const int32_t *query_codes, const int32_t *key_codes, int32_t *output,
                                      uint32_t *mask, int32_t *extra0, void *workspace, int B, int S, int m, int nnz,
                                      int H, int n_codewords, spt_stream_t stream) {
    SPT_REQUIRE(mask && extra0, "lookup_mask_fwd_ex: null mask / extra0");
    SPT_REQUIRE(n_codewords >= 1, "lookup_mask_fwd_ex: n_codewords must be >= 1 (got %d)", n_codewords);
    return lookup_impl(query_codes, key_codes, output, mask, extra0, workspace, B, S, m, nnz, H, n_codewords, stream);
}

// ---- packed variable-length sequences ----------------------------------------------------------------------------------
// shared memory of the varlen kernels at `groups` 128-key groups per row: plane kernel, plane-free kernel, generic fallback
static size_t lkv_plane_smem(int m, int groups) { return ((size_t)m * LK_WORD_U32 * 4 + 2 * LKM_THREADS * 4) * groups; }
static size_t lkv_big_smem(int m, int groups) { return (size_t)m * LK_WORD_U32 * 4 * groups + (size_t)LKB_CHUNK * LKM_THREADS * 4; }
static size_t lkv_generic_smem(int m, int groups, int nnz_max) {
    return out_image_bytes(nnz_max) + (size_t)LK_ROWS * 4 * groups * 4 + (size_t)LK_ROWS * m * 2;
}
constexpr size_t LKV_SMEM_MAX = 200 * 1024;

extern "C" size_t spt_lookup_mask_varlen_workspace_bytes(int n_seq, int T, int H, int m) {
    if (n_seq < 1 || T < 1 || H < 1 || m < 1) return 16;
    return 16 + (size_t)H * m * varlen_capacity(n_seq, T) * LK_WORD_U32 * sizeof(uint32_t);
}

extern "C" int spt_lookup_mask_varlen_max_seqlen(int m) {
    return (m == 8 || m == 10 || m == 16) ? VARLEN_MAX_SEQLEN : 0;    // the streaming kernel has no length cap
}

template <int M>
static int lookup_varlen_launch(const int32_t *qc, const int32_t *kc, const uint32_t *kb, const int *flag, uint32_t *mask,
                                int32_t *extra0, const LkVarlen &vl, int cap, int T, int H, cudaStream_t st) {
    const size_t psmem = lkv_plane_smem(M, vl.groups), bsmem = lkv_big_smem(M, vl.groups);
    if (psmem <= LKV_SMEM_MAX) {
        cudaFuncSetAttribute(lookup_maskonly2_kernel<M, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psmem);
        lookup_maskonly2_kernel<M, true><<<dim3(H, cap), LKM_THREADS, psmem, st>>>(qc, kb, flag, mask, extra0, T, 0, cap, H, vl);
        return after_launch("lookup_maskonly2_kernel(varlen)");
    }
    if (bsmem <= LKV_SMEM_MAX) {
        cudaFuncSetAttribute(lookup_maskonly_big_kernel<M, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bsmem);
        lookup_maskonly_big_kernel<M, true><<<dim3(H, cap), LKM_THREADS, bsmem, st>>>(qc, kb, flag, mask, extra0, T, 0, cap, H, vl);
        return after_launch("lookup_maskonly_big_kernel(varlen)");
    }
    lks_launch<M, true>(dim3(H, cap), qc, kb, flag, mask, extra0, T, 0, cap, H, st, vl);
    return after_launch("lookup_maskonly_big_kernel(stream, varlen)");
}

static int lookup_varlen_impl(const int32_t *query_codes, const int32_t *key_codes, const void *work, uint32_t *mask,
                              int32_t *extra0, void *workspace, int n_seq, int T, int max_seqlen, int H, int m,
                              int sparse_coeff, int n_codewords, spt_stream_t stream) {
    const char *what = n_codewords < 0 ? "lookup_mask_varlen_fwd" : "lookup_mask_varlen_fwd_ex";
    SPT_REQUIRE(query_codes && key_codes && work && mask && extra0 && workspace, "%s: null pointer", what);
    int rc = check_varlen(what, n_seq, T, max_seqlen, H);
    if (rc != SPT_OK) return rc;
    SPT_REQUIRE(m == 8 || m == 10 || m == 16, "%s: n_subspaces must be 8, 10 or 16 (got %d)", what, m);
    SPT_REQUIRE(sparse_coeff >= 1, "%s: sparse_coeff must be >= 1 (got %d)", what, sparse_coeff);
    SPT_REQUIRE(((uintptr_t)work | (uintptr_t)mask | (uintptr_t)workspace) % 16 == 0, "%s: work, mask and workspace must be 16-byte aligned", what);
    const int nnz_max = (max_seqlen / sparse_coeff + 3) & ~3;       // sizes the generic fallback's row images
    const size_t gsmem = lkv_generic_smem(m, (max_seqlen + 127) / 128, nnz_max);
    const bool fb_fits = gsmem <= LKV_SMEM_MAX;
    if (!fb_fits) {
        SPT_REQUIRE(n_codewords >= 0, "%s: max_seqlen %d / sparse_coeff %d too large for the row images", what, max_seqlen, sparse_coeff);
        if (n_codewords > LK_CV)
            return fail(SPT_ERR_UNSUPPORTED,
                        "%s: max_seqlen %d / sparse_coeff %d needs n_codewords <= %d (got %d): the fallback for codes >= %d "
                        "needs %zu bytes of row images, beyond its limit of %zu",
                        what, max_seqlen, sparse_coeff, LK_CV, n_codewords, LK_CV, gsmem, LKV_SMEM_MAX);
    }
    cudaStream_t st = as_stream(stream);
    const int cap = (int)varlen_capacity(n_seq, T);
    const int32_t *w = (const int32_t *)work;
    const LkVarlen vl{reinterpret_cast<const int4 *>(w + 4), w, (max_seqlen + 127) / 128, sparse_coeff};
    int *flag = reinterpret_cast<int *>(workspace);
    uint32_t *kb = reinterpret_cast<uint32_t *>(reinterpret_cast<char *>(workspace) + 16);
    cudaError_t e = cudaMemsetAsync(flag, 0, 16, st);
    if (e != cudaSuccess) return fail(SPT_ERR_CUDA, "%s: memset: %s", what, cudaGetErrorString(e));
    lookup_pack_kernel<true><<<dim3(cap, H), 128, 0, st>>>(key_codes, kb, flag, T, m, cap, H, vl);
    SPT_LAUNCH_CHECK("lookup_pack_kernel(varlen)");
    const int *kflag = fb_fits ? flag : flag + 1;       // as in lookup_impl: flag + 1 is never raised
    rc = m == 8    ? lookup_varlen_launch<8>(query_codes, key_codes, kb, kflag, mask, extra0, vl, cap, T, H, st)
         : m == 10 ? lookup_varlen_launch<10>(query_codes, key_codes, kb, kflag, mask, extra0, vl, cap, T, H, st)
                   : lookup_varlen_launch<16>(query_codes, key_codes, kb, kflag, mask, extra0, vl, cap, T, H, st);
    if (rc != SPT_OK || !fb_fits) return rc;
    // codes >= 16 somewhere: the generic kernel redoes the call (flag-guarded, decided on the device)
    cudaFuncSetAttribute(lookup_generic_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gsmem);
    lookup_generic_kernel<true><<<2 * num_sms(), LK_THREADS, gsmem, st>>>(query_codes, key_codes, flag, 1, nullptr, mask, extra0,
                                                                         T, m, nnz_max, H, 0, H, vl);
    return after_launch("lookup_generic_kernel(varlen fallback)");
}

extern "C" int spt_lookup_mask_varlen_fwd(const int32_t *query_codes, const int32_t *key_codes, const void *work,
                                          uint32_t *mask, int32_t *extra0, void *workspace, int n_seq, int T,
                                          int max_seqlen, int H, int m, int sparse_coeff, spt_stream_t stream) {
    return lookup_varlen_impl(query_codes, key_codes, work, mask, extra0, workspace, n_seq, T, max_seqlen, H, m, sparse_coeff,
                              -1, stream);
}

extern "C" int spt_lookup_mask_varlen_fwd_ex(const int32_t *query_codes, const int32_t *key_codes, const void *work,
                                             uint32_t *mask, int32_t *extra0, void *workspace, int n_seq, int T,
                                             int max_seqlen, int H, int m, int sparse_coeff, int n_codewords,
                                             spt_stream_t stream) {
    SPT_REQUIRE(n_codewords >= 1, "lookup_mask_varlen_fwd_ex: n_codewords must be >= 1 (got %d)", n_codewords);
    return lookup_varlen_impl(query_codes, key_codes, work, mask, extra0, workspace, n_seq, T, max_seqlen, H, m, sparse_coeff,
                              n_codewords, stream);
}
