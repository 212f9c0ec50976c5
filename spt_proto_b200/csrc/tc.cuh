// tcgen05 / TMEM / TMA / mbarrier primitives shared by the tensor-core kernels (ffn_gemm.cu,
// attn_tc.cu).  sm_100a inline PTX only.
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace spt {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier ------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {  // try_wait suspends the thread in hardware up to a time limit, so this is not a hot spin
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}" : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    } while (!done);
}

// ---- TMA -----------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap *map, uint32_t bar, int c0, int c1, int c2,
                                            int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}

// 1-D bulk copy global -> shared (bytes and both addresses multiples of 16); completes on the mbarrier like a tensor load
__device__ __forceinline__ void bulk_load_1d(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

// One lane of a converged warp (warp-uniform control flow around it keeps operands in uniform registers).
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}" : "=r"(pred));
    return pred != 0;
}

// ---- clusters --------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {   // every thread of every CTA of the cluster
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// ---- CTA pair (cta_group::2): two CTAs of a cluster on the SMs of one TPC run M = 256 MMAs together ------------
constexpr uint32_t PEER_BIT_MASK = 0xFEFFFFFFu;   // clears the CTA-rank bit of a shared::cluster address -> the even CTA
// TMA load into the executing CTA's shared memory whose complete_tx goes to the LEADER CTA's mbarrier
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap *map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar & PEER_BIT_MASK), "r"(c0), "r"(c1) : "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_alloc_pair(uint32_t slot_smem_addr) {  // one full warp, same warp id in both CTAs
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_smem_addr), "n"(COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t tmem_base) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(COLS));
}
// arrive (when all prior MMAs of the pair retire) on the barrier at this offset in every CTA of `mask`
__device__ __forceinline__ void umma_commit_pair(uint32_t bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"(mask) : "memory");
}
// D[tmem of both CTAs, 128 lanes each] (+)= A[256 x 16: 128 rows from each CTA's smem] * B[16 x N: N/2 from each CTA]
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
// arrive on the barrier at the same offset in CTA `rank` of the cluster.  Relaxed: the only thing ordered through it
// is tensor memory (tcgen05.fence::before_thread_sync precedes it); a release here makes the compiler drain every
// outstanding global store of the warp and invalidate L1 (MEMBAR + ERRBAR + CCTL.IVALL) on each arrive.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar, uint32_t rank) {
    asm volatile(
        "{\n\t"
        ".reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [ra];\n\t"
        "}" ::"r"(bar), "r"(rank) : "memory");
}
// mbar_wait with cluster-scope acquire (the arrivals come from the other CTA)
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}" : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    } while (!done);
}

// TMA load delivered to the same shared-memory offset of every CTA in `mask`; each destination CTA's mbarrier
// (same offset) receives the complete_tx
__device__ __forceinline__ void tma_load_2d_mc(uint32_t dst, const CUtensorMap *map, uint32_t bar, int c0, int c1,
                                               uint16_t mask) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "h"(mask) : "memory");
}

// ---- tcgen05 -------------------------------------------------------------------------------------
template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t slot_smem_addr) {  // one full warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_smem_addr), "n"(COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t tmem_base) {     // the allocating warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(COLS));
}
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// the same arrive delivered to the barrier at this offset in every CTA of `mask`
__device__ __forceinline__ void umma_commit_mc(uint32_t bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"(mask) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
// D[tmem] (+)= A[tmem: lane = row, 2 bf16 per 32-bit column, K-major] * B[smem desc]
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}

// 32 lanes x 32 columns of 32-bit: thread `lane` of the warp gets its lane's 32 consecutive columns
__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
// 32 lanes x 64 columns in one instruction (every tcgen05.ld costs the concurrent MMA stream a fixed bubble: fewer, wider loads)
__device__ __forceinline__ void tmem_ld64_nowait(uint32_t taddr, uint32_t (&r)[64]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x64.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32,%33,%34,%35,%36,%37,%38,%39,%40,%41,%42,%43,%44,%45,%46,%47,%48,%49,%50,%51,%52,%53,%54,%55,%56,%57,%58,%59,%60,%61,%62,%63}, [%64];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31]), "=r"(r[32]), "=r"(r[33]), "=r"(r[34]), "=r"(r[35]), "=r"(r[36]), "=r"(r[37]), "=r"(r[38]), "=r"(r[39]), "=r"(r[40]), "=r"(r[41]), "=r"(r[42]), "=r"(r[43]), "=r"(r[44]), "=r"(r[45]), "=r"(r[46]), "=r"(r[47]), "=r"(r[48]), "=r"(r[49]), "=r"(r[50]), "=r"(r[51]), "=r"(r[52]), "=r"(r[53]), "=r"(r[54]), "=r"(r[55]), "=r"(r[56]), "=r"(r[57]), "=r"(r[58]), "=r"(r[59]), "=r"(r[60]), "=r"(r[61]), "=r"(r[62]), "=r"(r[63])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    tmem_ld32_nowait(taddr, r);
    tmem_ld_wait();
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
          "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- UMMA descriptors ------------------------------------------------------------------------------
// Shared-memory matrix descriptor (sm_100 UMMA): start address, leading / stride byte offsets (all
// >> 4), descriptor version 1, 128-byte swizzle.
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3fff);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3fff) << 32;
    d |= (uint64_t)1 << 46;   // version = 1
    d |= (uint64_t)2 << 61;   // SWIZZLE_128B
    return d;
}
// A bf16 operand tile stored as rows of 64 elements (128 B, 128B-swizzled in 8-row atoms of 1 KB),
// exactly what a TMA box (64, rows) with CU_TENSOR_MAP_SWIZZLE_128B writes.  Descriptor of its k-th
// K16 slice:
//   K-major  (rows = M/N index, the 64 columns = K): SBO = 1024, slice k = +32 B
//   MN-major (rows = K index, the 64 columns = M/N): SBO = 1024 (8 k-rows), LBO = bytes to the next
//             64-wide MN chunk, slice k = +16 rows = +2048 B
// The address field (bits 0-13, 16-byte units) never carries for shared-memory offsets, so a slice /
// stage offset is a plain add on a precomputed descriptor: KMAJOR_K16 per K16 slice of a K-major tile,
// MNMAJOR_K16 per K16 slice of an MN-major tile, bytes >> 4 for a stage offset.
constexpr uint64_t KMAJOR_K16 = 32 >> 4, MNMAJOR_K16 = 2048 >> 4;
__device__ __forceinline__ uint64_t desc_kmajor(uint32_t tile_addr, int k) { return make_desc(tile_addr + k * 32, 0, 1024); }
__device__ __forceinline__ uint64_t desc_mnmajor(uint32_t tile_addr, int k, uint32_t lbo_bytes) {
    return make_desc(tile_addr + k * 2048, lbo_bytes, 1024);
}
// Instruction descriptor, kind::f16: D = f32, A = B = bf16; a_major / b_major: 0 = K-major, 1 = MN-major
__device__ __forceinline__ constexpr uint32_t idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
           ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// The same with A = B = fp16: the A / B format fields (bits 7-9, 10-12) are 0 for fp16
__device__ __forceinline__ constexpr uint32_t idesc_fp16(int M, int N, int a_mn_major, int b_mn_major) {
    return idesc_bf16(M, N, a_mn_major, b_mn_major) & ~((7u << 7) | (7u << 10));
}

// ---- host: tensor maps -----------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_fn() {
    // cuTensorMapEncodeTiled is a driver-API call: it needs the device's primary context bound to the
    // calling thread.  A thread whose first CUDA action is this call (an autograd worker entering a
    // backward pass) has none yet (CUDA_ERROR_INVALID_CONTEXT).
    static thread_local bool bound = false;
    if (!bound) {   // cudaSetDevice binds the primary context and is not a stream operation (safe under graph capture)
        int dev = 0;
        cudaGetDevice(&dev);
        cudaSetDevice(dev);
        bound = true;
    }
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *ptr = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(ptr);
    }
    return fn;
}

}  // namespace tc
}  // namespace spt
