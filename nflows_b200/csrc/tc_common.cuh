// tcgen05 / TMA / mbarrier building blocks shared by the tensor-core kernels of libnfk_sm100.so (inline PTX; the
// CUTLASS headers in this image are only consulted for descriptor bit layouts, nothing is included from them).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>

#include "nfk_common.cuh"

namespace nfk {
namespace tc {

constexpr int BM = 128;            // rows per tile = TMEM lanes
constexpr int BN_MAX = 256;        // columns per tile (runtime BN <= BN_MAX, multiple of 16)
constexpr int BK = 32;             // fp16 elements per K-slab = one 64-byte swizzle row (SWIZZLE_64B) = two UMMA K-steps
constexpr int STAGES = 4;          // 4 x 48 KB slabs: 3 TMA loads in flight while one slab is consumed
constexpr int THREADS = 384;        // warpgroup 0: TMA + MMA warps (2 idle); warpgroups 1-2: accumulate/epilogue
// K-slabs accumulated inside the tensor core before the partial sum is drained to registers (precision vs drain cost):
constexpr int DRAIN_SLABS_LINEAR = 2;   // dense layers: K = 64 (12 MMAs) -- their outputs feed log p directly
constexpr int DRAIN_SLABS_FUSED = 4;    // fused coupling: K = 128 (24 MMAs) -- its outputs are spline logits
constexpr int HALF = BN_MAX / 2;     // columns per epilogue warp
constexpr int A_BYTES = BM * BK * 2;             // 8 KB
constexpr int B_BYTES = BN_MAX * BK * 2;         // 16 KB
constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;   // 48 KB
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*alignment slack*/ + 256 /*barriers*/;

// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(bar),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
// 1-D bulk copy global -> this CTA's shared memory, bytes (multiple of 16, 16-byte aligned both sides) counted on `bar`
__device__ __forceinline__ void bulk_load_1d(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar)
                 : "memory");
}
// ---- thread-block-cluster variants: one TMA box delivered to the same smem offset of every CTA in `mask`, each
// destination CTA's mbarrier (same offset) receives the bytes; tcgen05.commit arriving on the barrier of every CTA in `mask`
__device__ __forceinline__ void tma_load_2d_multicast(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1,
                                                      uint16_t mask) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], "
        "[%2], %5;" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "h"(mask)
        : "memory");
}
// One lane of a converged warp (elect.sync).  Code that issues tcgen05.mma / TMA under `if (elect_one())` is compiled onto the
// UNIFORM datapath: descriptors live in uniform registers and UTCHMMA / UTMALDG issue back to back.  Under `if (lane == 0)` ptxas
// cannot know a single lane is active and wraps EVERY such instruction in an ELECT + five R2UR moves + a lane loop (~190 cycles
// per tcgen05.mma measured, against 96-128 cycles of tensor work: the issuing warp, never idle, was what capped the tensor pipe
// at ~50 % in every tensor-core kernel of this library up to round 2).
// Hands a TMA-filled shared-memory slot back to its producer AFTER this warp's loads from it have returned.  mbarrier.arrive
// is not ordered behind earlier LDS of the same warp (ptxas schedules it two instructions after the last LDS.128 and the barrier
// unit does not wait for the load queue), so the producer's next bulk copy could overwrite the slot under a load still queued:
// measured on hardware (r2) as the last float4 of a warp's bias window holding the bias of column tile n+2.  The guard is a
// true data dependency -- the barrier address is offset by (loaded bits & zero), `zero` a kernel parameter that is always 0,
// which ptxas cannot fold away: the arrive cannot issue before the loaded registers exist, i.e. before shared memory was read.
// (A generic->async proxy fence in front of it as well costs ~1 000 cycles per use: two per column tile and warp.)
__device__ __forceinline__ void mbar_arrive_after_loads(uint32_t bar, uint32_t loaded_bits, uint32_t zero) {
    mbar_arrive(bar + (loaded_bits & zero));
}

__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "elect.sync _|P1, 0xffffffff;\n"
        "selp.u32 %0, 1, 0, P1;\n"
        "}\n"
        : "+r"(pred));
    return pred != 0;
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void umma_commit_multicast(uint32_t bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
                 "h"(mask)
                 : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major swizzled shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
// [0,14) start>>4 | [16,30) LBO>>4 (=1, unused for swizzled K-major) | [32,46) SBO>>4 (8 rows x row bytes)
// | [46,48) version=1 (sm_100) | [61,64) layout: 2 = SWIZZLE_128B (128-byte rows), 4 = SWIZZLE_64B (64-byte rows)
constexpr int ROW_BYTES = BK * 2;
static_assert(ROW_BYTES == 128 || ROW_BYTES == 64, "K-slab rows must be 64 or 128 bytes");
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | (1ull << 16) | ((uint64_t)((8 * ROW_BYTES) >> 4) << 32) | (1ull << 46) |
           ((uint64_t)(ROW_BYTES == 128 ? 2 : 4) << 61);
}
// cute::UMMA::InstrDescriptor: c=F32 (1<<4), a=b=F16 (format 0 at [7,10) and [10,13)), K-major both, N>>3 at [17,23),
// M>>4 at [24,29) (M = BM)
__device__ __forceinline__ uint32_t make_idesc(int bn) {
    return (1u << 4) | ((uint32_t)(bn >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}


// Split of one fp32 value into the fp16 pair the kernels multiply with: v * scale = hi + lo (+ <= 2^-22 relative), hi the
// nearest fp16, lo the nearest fp16 of the exact remainder.  |v * scale| beyond the fp16 range raises NFK_FLAG_F16_RANGE.
__device__ __forceinline__ void split_f16(float v, float scale, __half& hi, __half& lo, int& flag) {
    const float s = v * scale;
    if (!(fabsf(s) <= 65000.0f)) flag |= 4;
    hi = __float2half_rn(s);
    lo = __float2half_rn(s - __half2float(hi));
}

// host helpers (nfk_linear_tc.cu)
int make_map(CUtensorMap* map, const __half* base, int64_t rows, int K, int64_t ld, int box_rows);
int make_out_map(CUtensorMap* map, float* base, int64_t rows, int64_t cols, int64_t ld, int box_cols, int box_rows);
int make_out_map16(CUtensorMap* map, __half* base, int64_t rows, int64_t cols, int64_t ld, int box_cols, int box_rows);
int sm_count();

}  // namespace tc
}  // namespace nfk
