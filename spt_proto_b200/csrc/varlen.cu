// Work list of a packed variable-length batch: cu_seqlens -> one item per (sequence, 128-row tile), shared by the
// varlen lookup (lookup.cu) and the varlen attention kernels (attn_tc.cu).
//
// The items are ordered by descending tile index over all sequences (a counting sort: one pass per tile index), so the
// CTAs with the most causal work of every sequence are launched first and the launch ends on the lightest ones (the
// heaviest-first order of the fixed-length grids, DESIGN.md section 4.1).  The dK/dV kernel mirrors the tile index
// inside each sequence and gets the same property.  Consumers size their grids from the capacity ceil(T/128) + n_seq
// and exit past the device-side count: nothing synchronises with the host, so the calls can be captured in a graph.
//
// Every sequence is clamped to [0, T], to max_seqlen and down to a multiple of 32, and the word offsets are cut at the
// capacity: a bad device-side cu_seqlens cannot make a consumer read or write outside its tensors.
#include <cub/block/block_scan.cuh>

#include "common.cuh"

namespace spt {

constexpr int WL_THREADS = 1024;

__global__ void __launch_bounds__(WL_THREADS)
varlen_worklist_kernel(const int32_t *__restrict__ cu, int n_seq, int T, int max_seqlen, int32_t *__restrict__ work) {
    using Scan = cub::BlockScan<int, WL_THREADS>;
    __shared__ typename Scan::TempStorage tmp;
    __shared__ int s_levels;                          // the largest tile count of any sequence
    if (threadIdx.x == 0) s_levels = 0;
    const int cap = (int)varlen_capacity(n_seq, T);
    int4 *items = reinterpret_cast<int4 *>(work + 4);
    int4 *seqs = items + cap;                         // {start, len, tiles, word offset} per sequence
    // pass 1: clamped sequences, their tile counts and bitmap word offsets (exclusive prefix sum of the tile counts)
    int carry = 0, levels = 0;
    for (int i0 = 0; i0 < n_seq; i0 += WL_THREADS) {
        const int i = i0 + threadIdx.x;
        int start = 0, len = 0, nt = 0;
        if (i < n_seq) {
            start = min(max(cu[i], 0), T);
            const int end = min(max(cu[i + 1], start), T);
            len = min(end - start, max_seqlen) & ~31;
            nt = (len + 127) / 128;
        }
        int off, total;
        Scan(tmp).ExclusiveSum(nt, off, total);
        off += carry;
        nt = min(nt, max(0, cap - off));
        if (i < n_seq) seqs[i] = make_int4(start, len, nt, off);
        levels = max(levels, nt);
        carry += total;
        __syncthreads();                              // tmp is reused by the next scan
    }
    atomicMax(&s_levels, levels);
    __syncthreads();
    levels = s_levels;
    // pass 2: tile index `level` of every sequence that has one, deepest level first, sequences in order
    int pos = 0;
    for (int level = levels - 1; level >= 0; --level)
        for (int i0 = 0; i0 < n_seq; i0 += WL_THREADS) {
            const int i = i0 + threadIdx.x;
            const int4 s = i < n_seq ? seqs[i] : make_int4(0, 0, 0, 0);
            const int f = s.z > level;
            int rank, total;
            Scan(tmp).ExclusiveSum(f, rank, total);
            if (f) items[pos + rank] = make_int4(s.x, s.y, level, s.w);
            pos += total;
            __syncthreads();
        }
    if (threadIdx.x == 0) work[0] = pos;
}

}  // namespace spt

using namespace spt;

extern "C" size_t spt_varlen_worklist_bytes(int n_seq, int T) {
    if (n_seq < 1 || T < 1) return 16;
    return 16 + (size_t)varlen_capacity(n_seq, T) * 16 + (size_t)n_seq * 16;
}

extern "C" int spt_varlen_worklist(const int32_t *cu_seqlens, int n_seq, int T, int max_seqlen, void *work,
                                   spt_stream_t stream) {
    int rc = check_varlen("varlen_worklist", n_seq, T, max_seqlen, 1);
    if (rc != SPT_OK) return rc;
    SPT_REQUIRE(cu_seqlens && work, "varlen_worklist: null pointer");
    SPT_REQUIRE((uintptr_t)work % 16 == 0, "varlen_worklist: work must be 16-byte aligned");
    varlen_worklist_kernel<<<1, WL_THREADS, 0, as_stream(stream)>>>(cu_seqlens, n_seq, T, max_seqlen, (int32_t *)work);
    return after_launch("varlen_worklist_kernel");
}
