// Dense layer on the 5th-generation tensor cores (tcgen05) with fp32-equivalent operand precision.
//
//   Y = post(A W^T + b) + R           A: [n_rows, K]   W: [N, K] (nn.Linear layout)   fp32 accumulate in TMEM
//
// PyTorch's reference GEMM is true fp32 (allow_tf32=False); one reduced-precision pass misses the 1e-5 parity bar by two
// orders of magnitude (SURVEY.md Appendix C).  So every operand is carried as a split pair of fp16 numbers
//   v * 2^e = v_hi + v_lo,   v_hi = rn_fp16(v * 2^e),   v_lo = rn_fp16(v * 2^e - v_hi)        (22 mantissa bits)
// with a per-tensor power-of-two scale 2^e that keeps v_lo out of the fp16 subnormals (weights: max |w| -> 2^14;
// activations: a fixed exponent, overflow raises NFK_FLAG_F16_RANGE), and each K-step issues three kind::f16 MMAs into
// the same accumulator:  a_lo*w_hi + a_hi*w_lo + a_hi*w_hi  (the dropped a_lo*w_lo term is ~2^-22 relative; fp16 x fp16
// products are exact in the fp32 accumulator).  The epilogue multiplies by 2^-(e_a + e_w), exactly.
// Why fp16 and not TF32 pairs (the first version of this kernel): the GPU runs these kernels AT ITS POWER CAP -- cuBLAS
// sustains 643 TFLOP/s in TF32 but 1417 TFLOP/s in 16-bit on this box (scripts/tf32_peak.py) -- and the 3xTF32 kernels
// already executed 630 TFLOP/s of TF32 MMAs.  fp16 pairs carry the same 22 bits at half the operand bytes (4 B per
// element for the pair = one fp32), twice the K per MMA instruction and ~2.2x the flops per joule.
//
// Accumulation: the tensor core adds into its fp32 accumulator with round-toward-zero, so a long chain of MMAs
// acquires a bias of ~0.5 ulp per instruction (measured: 2e-5 relative after 294 MMAs, the effect Ootomo & Yokota 2022
// report for Ampere).  The accumulator in TMEM therefore only ever holds a PARTIAL sum over DRAIN_SLABS_LINEAR K-slabs
// (12 MMAs); the epilogue warps drain it with tcgen05.ld and keep the running sum in registers with round-to-nearest
// FADDs, while the issuer continues into the other TMEM buffer.
//
// Kernel shape (one persistent CTA per SM, 384 threads; setmaxnreg moves registers from warpgroup 0 to 1-2):
//   warp 0   : TMA producer   -- cp.async.bulk.tensor 2-D boxes {32 k, 128 rows} / {32 k, BN rows} of fp16, SWIZZLE_64B,
//                                out-of-bounds rows/columns zero-filled by the TMA unit (no padding anywhere)
//   warp 1   : TMEM allocator + tcgen05.mma issuer (UMMA 128 x BN x 16, K-major smem descriptors)
//   warps 4-11: accumulate/epilogue -- warp w owns TMEM lanes [32(w%4), +32) and column half (w-4)/4 of the tile:
//                                tcgen05.ld of each partial sum -> 128 running sums per thread in registers; at the end of
//                                a tile scale / relu / residual -> global stores of the fp32 result and/or the fp16 pair
//                                consumed by the next layer
//                                consumed by the next layer.  Outputs leave through shared memory: each warp stages 32-row x
//                                128-byte chunks (SWIZZLE_128B, conflict-free) and one lane issues a TMA store per chunk --
//                                full-line writes instead of the 32-sector scatter of a row-per-thread st.global (ncu, r1:
//                                the epilogue warps spent 43 % of their samples waiting for the LSU to drain those stores)
//   smem: TWO operand rings -- A (activations, streamed from HBM: latency of microseconds under load) LIN_A_STAGES x 16 KB,
//         W (weights, L2-resident) LIN_W_STAGES x 32 KB, each with its own producer thread and barriers, so the A stream runs
//         4 K-slabs ahead of the MMAs while W needs only 2 (round 1 had ONE ring of 3 x 48 KB released in pairs of slabs: one
//         load in flight, the tensor pipe waited a full HBM round trip per pair -- ncu r2: 21 % tensor, 39 % DRAM, 31 % L2);
//         + 8 warps x 2 x 4 KB store staging;
//   TMEM: 2 partial accumulators x 256 columns.
#include <mutex>

#include "tc_common.cuh"

namespace nfk {
namespace tc {

struct Params {
    const float* bias;       // [N] or null
    const float* residual;   // [n_rows, ldr] or null
    float* y;                // fp32 result or null
    __half* y_hi;            // fp16 split pair of pre(y) * out_scale for the next layer, or null
    __half* y_lo;
    int32_t* flags;          // NFK_FLAG_F16_RANGE when a pair output leaves the fp16 range
    float acc_scale;         // 2^(e_a + e_w): the accumulators hold (A W^T) * acc_scale
    float inv_acc_scale;
    float out_scale;         // 2^e of the pair output
    int split_n;             // pair output for columns < split_n only
    int64_t ldr, ldy, lds;
    int64_t n_rows;
    int K, N, BN;
    int relu_out;            // relu applied to (acc + bias) before the residual add / store
    int split_relu;          // relu applied before splitting (the next layer consumes relu(y))
    int num_m_tiles, num_n_tiles;
    int n_inner;             // tile schedule, see tile_of()
    int tma_store;           // outputs are TMA-addressable (16-byte aligned bases and row pitches): staged stores
    int y_first_col;         // the fp32 result is only needed for columns >= y_first_col (32-column chunks below it are skipped)
    int a_stages, w_stages;  // ring depths
    int w_slot_bytes;        // bytes per W ring slot (hi part first, lo part at w_slot_bytes / 2)
    // affine-coupling epilogue (nfk_affine_coupling_final_f16x3): the GEMM result is the conditioner's parameter row --
    // interleaved (shift_j, raw scale_j) pairs when c_mult == 2, shift_j when 1 -- consumed in registers, never stored
    const float* cx;         // coupling input [n_rows, ldcx]; NULL = plain dense layer
    float* cy;               // coupling output [n_rows, ldcy] (transformed columns only; may alias cx)
    const int32_t* c_cols;   // column of transformed feature j, or NULL: c_col0 + j
    float* c_lad;            // running log|det| per row (atomicAdd of this thread's share), may be NULL
    int64_t ldcx, ldcy;
    int c_col0, c_dt, c_mult, c_act, c_inverse;
};

// Operand rings share LIN_RING_BYTES: LIN_W_STAGES weight slots of [W hi | W lo] sized for the launch's column tile (BN rows of
// 64 bytes each, twice), the rest A slots of 16 KB [A hi | A lo] (BN = 208: 3 x 26 KB + 5 x 16 KB; BN = 256: 3 x 32 KB + 4 x 16 KB)
constexpr int LIN_RING_BYTES = 160 * 1024;
constexpr int LIN_A_STAGES_MAX = 8;
constexpr int LIN_W_STAGES_MAX = 8;
constexpr int LIN_A_STAGE_BYTES = 2 * A_BYTES;
constexpr int LIN_BAR_OFF = LIN_RING_BYTES;
constexpr int LIN_STG_OFF = LIN_BAR_OFF + 1024;                         // after the rings and the barrier block, 1024-aligned
constexpr int LIN_STG_BYTES = 4096;                                     // one 32-row x 128-byte chunk
constexpr int LIN_SMEM_BYTES = LIN_STG_OFF + 8 * 2 * LIN_STG_BYTES + 1024 /*alignment slack*/;

__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(map)),
                 "r"(src), "r"(c0), "r"(c1)
                 : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}

// Tile schedule of a persistent CTA.  With at least one 128-row block per CTA ("n_inner") a CTA walks all column tiles of
// its row block back to back, so the A slabs it just streamed are re-read from L2, not from HBM (K = N = 784: 4 column
// tiles -> 4x less HBM traffic for A).  Small batches keep the flat row-fastest order to fill the machine.
// With CL = 2 the two CTAs of a cluster take neighbouring row blocks (2u, 2u+1) of the SAME column tile and multicast
// half of every weight slab to each other; a trailing odd row block is paired with an out-of-range one (all-zero A, no stores).
template <int CL>
__device__ __forceinline__ bool tile_of(const int it, const int n_inner, const int num_m, const int num_n, const int rank,
                                        int& m, int& n) {
    const int units = (num_m + CL - 1) / CL;                  // row-block groups
    const int first = blockIdx.x / CL, step = gridDim.x / CL;
    if (n_inner) {
        const int u = first + (it / num_n) * step;
        m = u * CL + rank;
        n = it % num_n;
        return u < units;
    }
    const int t = first + it * step;
    m = (t % units) * CL + rank;
    n = t / units;
    return t < units * num_n;
}

template <int CL>
__global__ void __launch_bounds__(THREADS, 1)
linear_f16x3_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                     const __grid_constant__ CUtensorMap map_w_hi, const __grid_constant__ CUtensorMap map_w_lo,
                     const __grid_constant__ CUtensorMap map_y, const __grid_constant__ CUtensorMap map_yh,
                     const __grid_constant__ CUtensorMap map_yl, const __grid_constant__ CUtensorMap map_y_tail,
                     const __grid_constant__ CUtensorMap map_yh_tail, const __grid_constant__ CUtensorMap map_yl_tail,
                     const Params p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;      // SWIZZLE_128B needs 1024-byte alignment
    uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
    const int LIN_A_STAGES = p.a_stages, LIN_W_STAGES = p.w_stages;
    const uint32_t LIN_W_STAGE_BYTES = (uint32_t)p.w_slot_bytes, W_LO = LIN_W_STAGE_BYTES / 2;
    const uint32_t ring_w = smem_base + LIN_A_STAGES * LIN_A_STAGE_BYTES;
    const uint32_t bars = smem_base + LIN_BAR_OFF;                         // 8-byte mbarriers
    const uint32_t bar_afull = bars, bar_aempty = bars + 8 * LIN_A_STAGES_MAX;
    const uint32_t bar_wfull = bars + 16 * LIN_A_STAGES_MAX, bar_wempty = bar_wfull + 8 * LIN_W_STAGES_MAX;
    const uint32_t bar_tfull = bar_wempty + 8 * LIN_W_STAGES_MAX, bar_tempty = bar_tfull + 16;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem_gen + LIN_BAR_OFF + 16 * LIN_A_STAGES_MAX + 16 * LIN_W_STAGES_MAX + 32);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int num_k = (p.K + BK - 1) / BK;

    if (threadIdx.x == 0) {
        for (int s = 0; s < LIN_A_STAGES; ++s) { mbar_init(bar_afull + 8 * s, 1); mbar_init(bar_aempty + 8 * s, 1); }
        // both CTAs' MMA threads of a cluster release a weight slot (the peer multicasts into it)
        for (int s = 0; s < LIN_W_STAGES; ++s) { mbar_init(bar_wfull + 8 * s, 1); mbar_init(bar_wempty + 8 * s, CL); }
        for (int a = 0; a < 2; ++a) { mbar_init(bar_tfull + 8 * a, 1); mbar_init(bar_tempty + 8 * a, 8); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        prefetch_tmap(&map_a_hi); prefetch_tmap(&map_a_lo); prefetch_tmap(&map_w_hi); prefetch_tmap(&map_w_lo);
    }
    if (warp == 1) tmem_alloc(smem_u32(tmem_slot), 512);
    tc_fence_before();
    if (CL > 1) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int cta_rank = CL > 1 ? (int)cluster_ctarank() : 0;
    constexpr uint16_t cl_mask = (uint16_t)((1u << CL) - 1);
    const int num_groups = (num_k + DRAIN_SLABS_LINEAR - 1) / DRAIN_SLABS_LINEAR;   // partial sums per tile

    if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;" ::: "memory");     // hand registers to the epilogue warpgroups
    if (warp == 0) {
        // ================================================= TMA producer of the A ring (this CTA's 128 rows of every K-slab); one
        // ELECTED thread, so that ptxas keeps the role on the uniform datapath (tc_common.cuh: elect_one)
        if (elect_one()) {
            int stage = 0; uint32_t phase = 0;
            int tm, tn;
            for (int it = 0; tile_of<CL>(it, p.n_inner, p.num_m_tiles, p.num_n_tiles, cta_rank, tm, tn); ++it) {
                const int m0 = tm * BM;
                for (int ks = 0; ks < num_k; ++ks) {
                    mbar_wait(bar_aempty + 8 * stage, phase ^ 1);
                    const uint32_t full = bar_afull + 8 * stage;
                    const uint32_t sa = smem_base + stage * LIN_A_STAGE_BYTES;
                    mbar_expect_tx(full, 2u * A_BYTES);
                    tma_load_2d(sa, &map_a_hi, full, ks * BK, m0);
                    tma_load_2d(sa + A_BYTES, &map_a_lo, full, ks * BK, m0);
                    if (++stage == LIN_A_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 2) {
        // ================================================= TMA producer of the W ring (each CTA of a cluster fetches half of every
        // weight slab and multicasts it to both)
        if (elect_one()) {
            const uint32_t tx_bytes = 2u * (uint32_t)p.BN * ROW_BYTES;
            int stage = 0; uint32_t phase = 0;
            int tm, tn;
            const int wrows = p.BN / CL;                                   // weight rows this CTA fetches per slab
            for (int it = 0; tile_of<CL>(it, p.n_inner, p.num_m_tiles, p.num_n_tiles, cta_rank, tm, tn); ++it) {
                const int n0 = tn * p.BN;
                for (int ks = 0; ks < num_k; ++ks) {
                    mbar_wait(bar_wempty + 8 * stage, phase ^ 1);          // every CTA of the cluster has released the slot
                    const uint32_t full = bar_wfull + 8 * stage;
                    const uint32_t sw = ring_w + stage * LIN_W_STAGE_BYTES;
                    mbar_expect_tx(full, tx_bytes);
                    if (CL == 1) {
                        tma_load_2d(sw, &map_w_hi, full, ks * BK, n0);
                        tma_load_2d(sw + W_LO, &map_w_lo, full, ks * BK, n0);
                    } else {
                        const uint32_t off = (uint32_t)(cta_rank * wrows) * ROW_BYTES;
                        tma_load_2d_multicast(sw + off, &map_w_hi, full, ks * BK, n0 + cta_rank * wrows, cl_mask);
                        tma_load_2d_multicast(sw + W_LO + off, &map_w_lo, full, ks * BK, n0 + cta_rank * wrows, cl_mask);
                    }
                    if (++stage == LIN_W_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ================================================= MMA issuer: one ELECTED thread (uniform datapath: descriptors in
        // uniform registers, tcgen05.mma back to back -- see tc_common.cuh: elect_one).
        // Per K-slab: the two small cross terms (a_lo w_hi, a_hi w_lo), then the main product, then both ring slots are released;
        // a partial sum (one TMEM buffer, alternating) covers DRAIN_SLABS_LINEAR slabs.
        if (elect_one()) {
            const uint32_t idesc = make_idesc(p.BN);
            int sa_i = 0; uint32_t pa = 0;
            int sw_i = 0; uint32_t pw = 0;
            uint32_t gc = 0;                                              // partial sums so far: buffer gc & 1, use gc >> 1 of it
            int tm, tn;
            for (int it = 0; tile_of<CL>(it, p.n_inner, p.num_m_tiles, p.num_n_tiles, cta_rank, tm, tn); ++it) {
                for (int g = 0; g < num_groups; ++g, ++gc) {
                    const int slabs = min(DRAIN_SLABS_LINEAR, num_k - g * DRAIN_SLABS_LINEAR);
                    const int acc = gc & 1u;
                    const uint32_t acc_phase = (gc >> 1) & 1u;
                    mbar_wait(bar_tempty + 8 * acc, acc_phase ^ 1);       // epilogue has drained this partial accumulator
                    const uint32_t d_tmem = tmem_base + acc * BN_MAX;
                    for (int j = 0; j < slabs; ++j) {
                        mbar_wait(bar_afull + 8 * sa_i, pa);               // TMA bytes have landed
                        mbar_wait(bar_wfull + 8 * sw_i, pw);
                        tc_fence_after();
                        const uint32_t sa = smem_base + sa_i * LIN_A_STAGE_BYTES;
                        const uint32_t sw = ring_w + sw_i * LIN_W_STAGE_BYTES;
                        const uint64_t a_hi = make_smem_desc(sa), a_lo = make_smem_desc(sa + A_BYTES);
                        const uint64_t w_hi = make_smem_desc(sw), w_lo = make_smem_desc(sw + W_LO);
#pragma unroll
                        for (int kk = 0; kk < BK / 16; ++kk) {             // UMMA K = 16 fp16 = 32 bytes = +2 in descriptor units
                            const uint64_t adv = (uint64_t)(kk * 2);
                            umma_f16(d_tmem, a_lo + adv, w_hi + adv, idesc, (j | kk) != 0);
                            umma_f16(d_tmem, a_hi + adv, w_lo + adv, idesc, 1);
                        }
#pragma unroll
                        for (int kk = 0; kk < BK / 16; ++kk) {
                            const uint64_t adv = (uint64_t)(kk * 2);
                            umma_f16(d_tmem, a_hi + adv, w_hi + adv, idesc, 1);
                        }
                        umma_commit(bar_aempty + 8 * sa_i);                             // frees the slots when the MMAs retire
                        if (CL == 1) umma_commit(bar_wempty + 8 * sw_i);
                        else umma_commit_multicast(bar_wempty + 8 * sw_i, cl_mask);     // ... the weight slot in every CTA of the cluster
                        if (++sa_i == LIN_A_STAGES) { sa_i = 0; pa ^= 1; }
                        if (++sw_i == LIN_W_STAGES) { sw_i = 0; pw ^= 1; }
                    }
                    umma_commit(bar_tfull + 8 * acc);                      // partial sum complete -> drain
                }
            }
        }
    }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 232;" ::: "memory");
        // ================================================= accumulate + epilogue: 8 warps
        const int q = warp & 3;                   // TMEM lane quarter this warp may access
        const int half = (warp - 4) >> 2;         // column half of the tile
        int acc = 0; uint32_t acc_phase = 0;
        const bool vec_y = p.y && (p.ldy % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.y) & 15) == 0);
        const bool vec_s = p.y_hi && (p.lds % 8 == 0) && ((reinterpret_cast<uintptr_t>(p.y_hi) & 15) == 0) &&
                           ((reinterpret_cast<uintptr_t>(p.y_lo) & 15) == 0);
        int flag = 0;
        const bool vec_r = p.residual && (p.ldr % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.residual) & 15) == 0);
        const bool vec_b = !p.bias || ((reinterpret_cast<uintptr_t>(p.bias) & 15) == 0);
        uint8_t* stg_gen = smem_gen + LIN_STG_OFF + (warp - 4) * 2 * LIN_STG_BYTES;      // this warp's two store-staging chunks
        const uint32_t stg_u32 = smem_base + LIN_STG_OFF + (warp - 4) * 2 * LIN_STG_BYTES;
        int stg_buf = 0;
        int tm, tn;
        // this lane's float4 of the bias of tile `it` (zeros past the tile / the matrix, or without a bias)
        auto bias_of = [&](int it) -> float4 {
            float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
            int bm, bn;
            if (p.bias && tile_of<CL>(it, p.n_inner, p.num_m_tiles, p.num_n_tiles, cta_rank, bm, bn)) {
                const int c = 4 * lane, col = bn * p.BN + half * HALF + c;
                if (c + half * HALF < p.BN) {
                    if (vec_b && col + 3 < p.N) {
                        b = __ldg(reinterpret_cast<const float4*>(p.bias + col));
                    } else {
                        if (col < p.N) b.x = __ldg(p.bias + col);
                        if (col + 1 < p.N) b.y = __ldg(p.bias + col + 1);
                        if (col + 2 < p.N) b.z = __ldg(p.bias + col + 2);
                        if (col + 3 < p.N) b.w = __ldg(p.bias + col + 3);
                    }
                }
            }
            return b;
        };
        float4 bias_cur = bias_of(0);
        for (int it = 0; tile_of<CL>(it, p.n_inner, p.num_m_tiles, p.num_n_tiles, cta_rank, tm, tn); ++it) {
            const int64_t row = (int64_t)tm * BM + q * 32 + lane;
            const int n0 = tn * p.BN + half * HALF;
            // The running sums start from bias (+ residual when no relu sits between them): the loads are issued here, at the
            // start of the tile, and complete under the first MMAs instead of stalling the tile epilogue (ncu: the serialised
            // DRAM-latency residual reads of the epilogue held up drains -> MMA -> TMA; 15 % tensor activity on 256x256).
            const bool fold_residual = p.residual && !p.relu_out;
            if (p.residual) {      // pull the NEXT tile's residual rows towards L2 while this tile is computed
                int nm, nn;
                if (tile_of<CL>(it + 1, p.n_inner, p.num_m_tiles, p.num_n_tiles, cta_rank, nm, nn)) {
                    const int64_t nrow = (int64_t)nm * BM + q * 32 + lane;
                    const int ncol = nn * p.BN + half * HALF;
                    if (nrow < p.n_rows) {
#pragma unroll
                        for (int c = 0; c < HALF; c += 32)
                            if (ncol + c < p.N && c + half * HALF < p.BN)
                                asm volatile("prefetch.global.L2 [%0];" ::"l"(p.residual + nrow * p.ldr + ncol + c));
                    }
                }
            }
            float sum[HALF];
            // The running sums live in the accumulators' power-of-two scaled domain (exact) and start from the bias: ONE coalesced
            // float4 per thread (lane l: columns 4l..4l+3 of this warp's column half; fetched during the PREVIOUS tile, see
            // bias_of) broadcast by shuffles.  The first form -- 32 broadcast float4 loads, each followed by its adds -- serialised
            // 32 L2 latencies per tile: 8 600 of a tile's 28 000 cycles, the MMA thread waiting for drained accumulators meanwhile
            // (r2 cycle counters, profiles/linear_cycles_r2.txt; L1 keeps little beside 227 KB of shared memory).
            const float4 mine = make_float4(bias_cur.x * p.acc_scale, bias_cur.y * p.acc_scale, bias_cur.z * p.acc_scale,
                                            bias_cur.w * p.acc_scale);
            if (fold_residual) {
                // residual rows straight into the sums, every load issued before anything depends on one (a dependent add between
                // two loads would serialise the DRAM latencies), then scaled and joined with the bias
#pragma unroll
                for (int c = 0; c < HALF; c += 4) {
                    const int col = n0 + c;
                    float4 r4 = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (row < p.n_rows && c + half * HALF < p.BN) {
                        if (vec_r && col + 3 < p.N) {
                            r4 = __ldcs(reinterpret_cast<const float4*>(p.residual + row * p.ldr + col));
                        } else {
                            const float* rp = p.residual + row * p.ldr + col;
                            if (col < p.N) r4.x = rp[0];
                            if (col + 1 < p.N) r4.y = rp[1];
                            if (col + 2 < p.N) r4.z = rp[2];
                            if (col + 3 < p.N) r4.w = rp[3];
                        }
                    }
                    sum[c] = r4.x; sum[c + 1] = r4.y; sum[c + 2] = r4.z; sum[c + 3] = r4.w;
                }
#pragma unroll
                for (int c = 0; c < HALF; c += 4) {
                    sum[c] = fmaf(sum[c], p.acc_scale, __shfl_sync(0xffffffffu, mine.x, c >> 2));
                    sum[c + 1] = fmaf(sum[c + 1], p.acc_scale, __shfl_sync(0xffffffffu, mine.y, c >> 2));
                    sum[c + 2] = fmaf(sum[c + 2], p.acc_scale, __shfl_sync(0xffffffffu, mine.z, c >> 2));
                    sum[c + 3] = fmaf(sum[c + 3], p.acc_scale, __shfl_sync(0xffffffffu, mine.w, c >> 2));
                }
            } else {
#pragma unroll
                for (int c = 0; c < HALF; c += 4) {
                    sum[c] = __shfl_sync(0xffffffffu, mine.x, c >> 2);
                    sum[c + 1] = __shfl_sync(0xffffffffu, mine.y, c >> 2);
                    sum[c + 2] = __shfl_sync(0xffffffffu, mine.z, c >> 2);
                    sum[c + 3] = __shfl_sync(0xffffffffu, mine.w, c >> 2);
                }
            }
            for (int g = 0; g < num_groups; ++g) {
                mbar_wait(bar_tfull + 8 * acc, acc_phase);
                tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * BN_MAX + half * HALF;
#pragma unroll
                for (int c = 0; c < HALF; c += 64) {                       // two 32-column TMEM loads in flight per wait
                    uint32_t raw[2][32];
                    tmem_ld32(taddr + c, raw[0]);
                    tmem_ld32(taddr + c + 32, raw[1]);
                    tmem_ld_wait();
#pragma unroll
                    for (int u = 0; u < 2; ++u) {
#pragma unroll
                        for (int j = 0; j < 32; j += 2) {                  // packed fp32x2 round-to-nearest adds (FADD2)
                            const float2 r2 = __fadd2_rn(make_float2(sum[c + 32 * u + j], sum[c + 32 * u + j + 1]),
                                                         make_float2(__uint_as_float(raw[u][j]), __uint_as_float(raw[u][j + 1])));
                            sum[c + 32 * u + j] = r2.x;
                            sum[c + 32 * u + j + 1] = r2.y;
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_tempty + 8 * acc);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
            const float4 bias_nxt = bias_of(it + 1);      // lands while this tile is written out
            if (p.tma_store) {
                // ---- finish the values in place ...
                const bool row_ok = row < p.n_rows;
#pragma unroll
                for (int c = 0; c < HALF; ++c) {
                    float x = sum[c] * p.inv_acc_scale;
                    if (p.relu_out) x = fmaxf(x, 0.0f);
                    sum[c] = x;
                }
                if (p.residual && !fold_residual) {
#pragma unroll
                    for (int c = 0; c < HALF; c += 4) {
                        const int col = n0 + c;
                        if (!row_ok || c + half * HALF >= p.BN || col >= p.N) continue;
                        const float* rp = p.residual + row * p.ldr + col;
                        if (vec_r && col + 3 < p.N) {
                            const float4 r4 = *reinterpret_cast<const float4*>(rp);
                            sum[c] += r4.x; sum[c + 1] += r4.y; sum[c + 2] += r4.z; sum[c + 3] += r4.w;
                        } else {
#pragma unroll
                            for (int j = 0; j < 4; ++j) if (col + j < p.N) sum[c + j] += rp[j];
                        }
                    }
                }
                // ---- ... and send them out chunk by chunk: [32 rows][128 bytes] per TMA store, 16-byte pieces XOR-swizzled
                // by the row (SWIZZLE_128B) so the row-per-lane st.shared is conflict-free; the TMA unit clips rows/columns
                // beyond the tensor, so ragged tiles need no guards
                const int row0 = tm * BM + q * 32;
                auto stage_begin = [&]() -> uint4* {
                    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");   // the chunk before last has left
                    __syncwarp();
                    return reinterpret_cast<uint4*>(stg_gen + stg_buf * LIN_STG_BYTES) + lane * 8;
                };
                auto stage_end = [&](const CUtensorMap* map, int c0) {
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) tma_store_2d(map, stg_u32 + stg_buf * LIN_STG_BYTES, c0, row0);
                    stg_buf ^= 1;
                };
                if (p.y) {
#pragma unroll
                    for (int ch = 0; ch < HALF / 32; ++ch) {
                        const int col0 = n0 + 32 * ch;
                        if (32 * ch + half * HALF >= p.BN || col0 >= p.N || col0 + 32 <= p.y_first_col) continue;
                        if (32 * ch + 32 + half * HALF > p.BN) {           // chunk straddles the tile's right edge (the columns
                            // beyond it belong to the next tile): a narrower, unswizzled [32][16 floats] chunk through its own map
                            if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                            __syncwarp();
                            uint4* dst = reinterpret_cast<uint4*>(stg_gen) + lane * 4;
#pragma unroll
                            for (int j = 0; j < 4; ++j)
                                dst[j] = make_uint4(__float_as_uint(sum[32 * ch + 4 * j]), __float_as_uint(sum[32 * ch + 4 * j + 1]),
                                                    __float_as_uint(sum[32 * ch + 4 * j + 2]), __float_as_uint(sum[32 * ch + 4 * j + 3]));
                            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                            __syncwarp();
                            if (lane == 0) tma_store_2d(&map_y_tail, stg_u32, col0, row0);
                            stg_buf = 1;
                            continue;
                        }
                        uint4* dst = stage_begin();
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            dst[j ^ (lane & 7)] = make_uint4(__float_as_uint(sum[32 * ch + 4 * j]), __float_as_uint(sum[32 * ch + 4 * j + 1]),
                                                             __float_as_uint(sum[32 * ch + 4 * j + 2]), __float_as_uint(sum[32 * ch + 4 * j + 3]));
                        stage_end(&map_y, col0);
                    }
                }
                if (p.y_hi) {
#pragma unroll
                    for (int ch = 0; ch < HALF / 64; ++ch) {
                        const int col0 = n0 + 64 * ch;
                        if (64 * ch + half * HALF >= p.BN || col0 >= p.N || col0 >= p.split_n) continue;
                        const int tail = p.BN - half * HALF - 64 * ch;     // < 64: chunk straddles the tile's right edge -> narrow chunk
                        const bool is_tail = tail < 64;
                        // both halves of the pair are formed once -- in registers, BEFORE waiting for the staging chunks: the previous
                        // chunk's TMA stores read them out meanwhile (the wait used to sit in front of the conversions and
                        // serialised store latency and arithmetic, twice per tile) -- and staged in the warp's two chunks
                        // full chunk: [32][128 B] swizzled; tail chunk: [32][2 * tail B] plain row-major (tail = 16, 32 or 48 columns)
                        const int pieces = is_tail ? tail >> 3 : 8;         // 16-byte pieces per row
                        uint4* dh = reinterpret_cast<uint4*>(stg_gen) + lane * pieces;
                        uint4* dl = reinterpret_cast<uint4*>(stg_gen + LIN_STG_BYTES) + lane * pieces;
                        float amax = 0.0f;
                        uint4 vh[8], vl[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            __half2 h2[4], l2[4];
#pragma unroll
                            for (int e = 0; e < 4; ++e) {
                                float x0 = sum[64 * ch + 8 * j + 2 * e], x1 = sum[64 * ch + 8 * j + 2 * e + 1];
                                if (p.split_relu) { x0 = fmaxf(x0, 0.0f); x1 = fmaxf(x1, 0.0f); }
                                x0 *= p.out_scale; x1 *= p.out_scale;
                                if (j < pieces) amax = fmaxf(amax, fmaxf(fabsf(x0), fabsf(x1)));
                                h2[e] = __floats2half2_rn(x0, x1);
                                const float2 hf = __half22float2(h2[e]);
                                l2[e] = __floats2half2_rn(x0 - hf.x, x1 - hf.y);
                            }
                            vh[j] = *reinterpret_cast<const uint4*>(h2);
                            vl[j] = *reinterpret_cast<const uint4*>(l2);
                        }
                        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                        __syncwarp();
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            if (j < pieces) {
                                const int slot = is_tail ? j : (j ^ (lane & 7));
                                dh[slot] = vh[j];
                                dl[slot] = vl[j];
                            }
                        }
                        if (row_ok && !(amax <= 65000.0f)) flag |= 4;
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        __syncwarp();
                        if (lane == 0) {
                            tma_store_2d(is_tail ? &map_yh_tail : &map_yh, stg_u32, col0, row0);
                            tma_store_2d(is_tail ? &map_yl_tail : &map_yl, stg_u32 + LIN_STG_BYTES, col0, row0);
                        }
                        stg_buf = 0;
                    }
                }
            } else if (p.cx) {
                // ---- affine / additive coupling (coupling.py:212-269 of the reference) on the parameters held in registers:
                // y_j = x_j * s_j + t_j (inverse: (x_j - t_j) / s_j), log|det| += +-sum_j log s_j
                float lad = 0.0f;
                if (row < p.n_rows) {
#pragma unroll
                    for (int c = 0; c < HALF; c += 2) {
                        const int col = n0 + c;                            // even: tiles and halves start on even columns
                        if (c + half * HALF >= p.BN || col >= p.N) continue;
                        const float a0 = sum[c] * p.inv_acc_scale, a1 = sum[c + 1] * p.inv_acc_scale;
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const int j = p.c_mult == 2 ? (col >> 1) : col + e;
                            if ((p.c_mult == 2 && e == 1) || j >= p.c_dt) continue;
                            const int cf = p.c_cols ? __ldg(p.c_cols + j) : p.c_col0 + j;
                            const float x = p.cx[row * p.ldcx + cf];
                            const float shift = (p.c_mult == 2 || e == 0) ? a0 : a1;
                            float out;
                            if (p.c_mult == 2) {
                                float scale;
                                if (p.c_act == 0) {
                                    scale = 1.0f / (1.0f + expf(-(a1 + 2.0f))) + 1e-3f;
                                } else {
                                    const float sp = a1 > 20.0f ? a1 : log1pf(expf(a1));
                                    scale = fminf(fmaxf(sp + 1e-3f, 0.0f), 3.0f);
                                }
                                lad += logf(scale);
                                out = p.c_inverse ? __fdiv_rn(__fsub_rn(x, shift), scale) : __fadd_rn(__fmul_rn(x, scale), shift);
                            } else {
                                out = p.c_inverse ? (x - shift) : (x + shift);
                            }
                            p.cy[row * p.ldcy + cf] = out;
                        }
                    }
                    if (p.c_lad && p.c_mult == 2) atomicAdd(p.c_lad + row, p.c_inverse ? -lad : lad);
                }
            } else if (row < p.n_rows) {
#pragma unroll
                for (int c = 0; c < HALF; c += 16) {
                    const int col0 = n0 + c;
                    if (c + half * HALF >= p.BN || col0 >= p.N) continue;
                    float v[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        float x = sum[c + j] * p.inv_acc_scale;            // bias (and a foldable residual) already included
                        if (p.relu_out) x = fmaxf(x, 0.0f);
                        v[j] = x;
                    }
                    const bool full16 = col0 + 16 <= p.N;
                    if (p.residual && !fold_residual) {
                        const float* rp = p.residual + row * p.ldr + col0;
                        if (vec_r && full16) {
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                float4 r4 = *reinterpret_cast<const float4*>(rp + 4 * j);
                                v[4 * j] += r4.x; v[4 * j + 1] += r4.y; v[4 * j + 2] += r4.z; v[4 * j + 3] += r4.w;
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < 16; ++j) if (col0 + j < p.N) v[j] += rp[j];
                        }
                    }
                    if (p.y && col0 + 16 > p.y_first_col) {
                        float* yp = p.y + row * p.ldy + col0;
                        if (vec_y && full16) {
#pragma unroll
                            for (int j = 0; j < 4; ++j)
                                *reinterpret_cast<float4*>(yp + 4 * j) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                        } else {
#pragma unroll
                            for (int j = 0; j < 16; ++j) if (col0 + j < p.N) yp[j] = v[j];
                        }
                    }
                    if (p.y_hi && col0 < p.split_n) {
                        __half hi[16], lo[16];
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const float x = p.split_relu ? fmaxf(v[j], 0.0f) : v[j];
                            split_f16(x, p.out_scale, hi[j], lo[j], flag);
                        }
                        __half* hp = p.y_hi + row * p.lds + col0;
                        __half* lp = p.y_lo + row * p.lds + col0;
                        if (vec_s && col0 + 16 <= p.split_n && full16) {
                            const uint4* h4 = reinterpret_cast<const uint4*>(hi);
                            const uint4* l4 = reinterpret_cast<const uint4*>(lo);
                            reinterpret_cast<uint4*>(hp)[0] = h4[0]; reinterpret_cast<uint4*>(hp)[1] = h4[1];
                            reinterpret_cast<uint4*>(lp)[0] = l4[0]; reinterpret_cast<uint4*>(lp)[1] = l4[1];
                        } else {
#pragma unroll
                            for (int j = 0; j < 16; ++j) if (col0 + j < p.N && col0 + j < p.split_n) { hp[j] = hi[j]; lp[j] = lo[j]; }
                        }
                    }
                }
            }
            __syncwarp();
            bias_cur = bias_nxt;
        }
        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // staging must outlive its stores
        if (flag && p.flags) atomicOr(p.flags, flag);
    }

    tc_fence_before();
    if (CL > 1) cluster_sync_all(); else __syncthreads();   // no CTA exits while a peer may still signal its barriers
    if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// ---------------------------------------------------------------- fp32 -> fp16 (hi, lo) split pair, optional relu
// HBM-bound: 4 B read + 4 B written per element.  Used for weights (once per parameter update), for tensors entering a
// tensor-core chain from outside and for the transformed half of a coupling output.
__global__ void __launch_bounds__(256) split_f16_kernel(const float* __restrict__ x, int64_t ldx, int n_cols, int relu,
                                                        float scale, __half* __restrict__ hi, __half* __restrict__ lo,
                                                        int64_t ldo, int64_t n_rows, int vec4, int32_t* flags) {
    int flag = 0;
    if (vec4) {
        const int n4 = n_cols >> 2;
        const int64_t total = n_rows * n4;
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
            const int64_t r = i / n4;
            const int j = (int)(i - r * n4) * 4;
            float4 v = __ldcs(reinterpret_cast<const float4*>(x + r * ldx + j));
            if (relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
            __half h[4], l[4];
            split_f16(v.x, scale, h[0], l[0], flag); split_f16(v.y, scale, h[1], l[1], flag);
            split_f16(v.z, scale, h[2], l[2], flag); split_f16(v.w, scale, h[3], l[3], flag);
            *reinterpret_cast<uint2*>(hi + r * ldo + j) = *reinterpret_cast<const uint2*>(h);
            *reinterpret_cast<uint2*>(lo + r * ldo + j) = *reinterpret_cast<const uint2*>(l);
        }
    } else {
        const int64_t total = n_rows * n_cols;
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
            const int64_t r = i / n_cols;
            const int j = (int)(i - r * n_cols);
            float v = x[r * ldx + j];
            if (relu) v = fmaxf(v, 0.0f);
            __half h, l;
            split_f16(v, scale, h, l, flag);
            hi[r * ldo + j] = h;
            lo[r * ldo + j] = l;
        }
    }
    if (flag && flags) atomicOr(flags, flag);
}

// Context gate of a residual block (nn/nets/resnet.py:50-53): y = skip + t * sigmoid(gate), i.e. F.glu(cat(t, gate)) + inputs,
// in one pass; writes the fp32 result (the next block's skip tensor) and/or the fp16 pair the next dense layer multiplies.
__global__ void __launch_bounds__(256) glu_skip_kernel(const float* __restrict__ t, int64_t ldt, const float* __restrict__ gate,
                                                       int64_t ldg, const float* __restrict__ skip, int64_t ldsk, float* __restrict__ y,
                                                       int64_t ldy, __half* __restrict__ hi, __half* __restrict__ lo, int64_t ldo,
                                                       float scale, int relu, int64_t n_rows, int n_cols, int32_t* flags) {
    int flag = 0;
    const int64_t total = n_rows * n_cols;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / n_cols;
        const int j = (int)(i - r * n_cols);
        const float g = gate[r * ldg + j];
        float v = t[r * ldt + j] * (1.0f / (1.0f + expf(-g)));
        if (skip) v += skip[r * ldsk + j];
        if (y) y[r * ldy + j] = v;
        if (hi) {
            __half h, l;
            split_f16(relu ? fmaxf(v, 0.0f) : v, scale, h, l, flag);
            hi[r * ldo + j] = h;
            lo[r * ldo + j] = l;
        }
    }
    if (flag && flags) atomicOr(flags, flag);
}

// ---------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* sym = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(sym);
    });
    return fn;
}

// 2-D map of an output tensor for the staged TMA stores: boxes of 32 rows x 128 bytes, SWIZZLE_128B
static int make_store_map(CUtensorMap* map, void* base, bool fp16, int64_t rows, int64_t cols, int64_t ld, int box_cols = 0) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return fail(NFK_E_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    const int es = fp16 ? 2 : 4;
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * es};
    cuuint32_t box[2] = {(cuuint32_t)(box_cols ? box_cols : 128 / es), 32};      // box_cols: narrow unswizzled tail chunk
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, fp16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, box_cols ? CU_TENSOR_MAP_SWIZZLE_NONE : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(NFK_E_CUDA, "cuTensorMapEncodeTiled (store map) failed with CUresult %d", (int)r);
    return NFK_OK;
}

// plain (unswizzled) fp32 output map: box of box_cols x box_rows elements
int make_out_map(CUtensorMap* map, float* base, int64_t rows, int64_t cols, int64_t ld, int box_cols, int box_rows) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return fail(NFK_E_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
    cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(NFK_E_CUDA, "cuTensorMapEncodeTiled (output map) failed with CUresult %d", (int)r);
    return NFK_OK;
}

int make_out_map16(CUtensorMap* map, __half* base, int64_t rows, int64_t cols, int64_t ld, int box_cols, int box_rows) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return fail(NFK_E_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
    cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(NFK_E_CUDA, "cuTensorMapEncodeTiled (fp16 output map) failed with CUresult %d", (int)r);
    return NFK_OK;
}

int make_map(CUtensorMap* map, const __half* base, int64_t rows, int K, int64_t ld, int box_rows) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return fail(NFK_E_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
    cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<__half*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, ROW_BYTES == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(NFK_E_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return NFK_OK;
}

int sm_count() {
    static std::atomic<int> counts[64];                      // per device
    int dev = 0;
    cudaGetDevice(&dev);
    int n = counts[dev & 63].load(std::memory_order_relaxed);
    if (!n) {
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
        counts[dev & 63].store(n, std::memory_order_relaxed);
    }
    return n;
}

}  // namespace tc
}  // namespace nfk

using namespace nfk;

static bool pow2_exp_ok(int e) { return e >= -60 && e <= 60; }

extern "C" int nfk_split_f16(const float* x, int64_t ldx, int32_t n_cols, int relu, int32_t scale_exp, void* hi, void* lo,
                             int64_t ldo, int64_t n_rows, int32_t* flags, void* stream) {
    NFK_REQUIRE(n_rows >= 0 && n_cols >= 0 && pow2_exp_ok(scale_exp), "bad sizes");
    if (n_rows == 0 || n_cols == 0) return NFK_OK;
    NFK_REQUIRE(x && hi && lo, "NULL pointer");
    const int vec4 = (n_cols % 4 == 0 && ldx % 4 == 0 && ldo % 4 == 0 && aligned16(x) && (reinterpret_cast<uintptr_t>(hi) & 7) == 0 &&
                      (reinterpret_cast<uintptr_t>(lo) & 7) == 0) ? 1 : 0;
    int64_t blocks = (n_rows * (vec4 ? n_cols / 4 : n_cols) + 255) / 256;
    int grid = (int)(blocks > 148 * 32 ? 148 * 32 : blocks);
    tc::split_f16_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, ldx, n_cols, relu, ldexpf(1.0f, scale_exp), (__half*)hi, (__half*)lo,
                                                                 ldo, n_rows, vec4, flags);
    return check_launch("split_f16_kernel");
}

extern "C" int nfk_glu_skip_rows(const float* t, int64_t ldt, const float* gate, int64_t ldg, const float* skip, int64_t ldsk,
                                 float* y, int64_t ldy, void* y_hi, void* y_lo, int64_t lds, int32_t y_exp, int split_relu,
                                 int64_t n_rows, int32_t n_cols, int32_t* flags, void* stream) {
    NFK_REQUIRE(n_rows >= 0 && n_cols >= 0 && pow2_exp_ok(y_exp), "bad sizes");
    if (n_rows == 0 || n_cols == 0) return NFK_OK;
    NFK_REQUIRE(t && gate, "NULL pointer");
    NFK_REQUIRE(y || (y_hi && y_lo), "no output requested");
    NFK_REQUIRE((y_hi == nullptr) == (y_lo == nullptr), "y_hi and y_lo must be given together");
    int64_t blocks = (n_rows * n_cols + 255) / 256;
    int grid = (int)(blocks > 148 * 32 ? 148 * 32 : blocks);
    tc::glu_skip_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(t, ldt, gate, ldg, skip, ldsk, y, ldy, (__half*)y_hi, (__half*)y_lo, lds,
                                                                ldexpf(1.0f, y_exp), split_relu, n_rows, n_cols, flags);
    return check_launch("glu_skip_kernel");
}

// fp16 rows must start on 16-byte boundaries for TMA: leading dimensions and K multiples of 8
extern "C" int nfk_linear_f16x3_supported(int64_t lda, int64_t ldw, int32_t in_features) {
    return (in_features >= 8 && in_features % 8 == 0 && lda % 8 == 0 && ldw % 8 == 0) ? 1 : 0;
}

namespace {
struct CouplingEpilogue {        // set by nfk_affine_coupling_final_f16x3
    const float* x; int64_t ldx; float* y; int64_t ldy; const int32_t* t_cols; int t_col0, d_t, mult, act, inverse; float* lad;
};
}  // namespace

static int linear_f16x3_launch(const void* a_hi_, const void* a_lo_, int64_t lda, int32_t a_exp, const void* w_hi_,
                               const void* w_lo_, int64_t ldw, int32_t w_exp, const float* bias, const float* R, int64_t ldr,
                               float* Y, int64_t ldy, void* y_hi_, void* y_lo_, int64_t lds, int32_t y_exp, int32_t split_cols,
                               int32_t y_first_col, int relu_out, int split_relu, int64_t n_rows, int32_t in_features,
                               int32_t out_features, int32_t* flags, void* stream, const CouplingEpilogue* ce);

extern "C" int nfk_linear_f16x3(const void* a_hi_, const void* a_lo_, int64_t lda, int32_t a_exp, const void* w_hi_,
                                const void* w_lo_, int64_t ldw, int32_t w_exp, const float* bias, const float* R, int64_t ldr,
                                float* Y, int64_t ldy, void* y_hi_, void* y_lo_, int64_t lds, int32_t y_exp, int32_t split_cols,
                                int32_t y_first_col, int relu_out, int split_relu, int64_t n_rows, int32_t in_features,
                                int32_t out_features, int32_t* flags, void* stream) {
    NFK_REQUIRE(Y || (y_hi_ && y_lo_), "no output requested");
    return linear_f16x3_launch(a_hi_, a_lo_, lda, a_exp, w_hi_, w_lo_, ldw, w_exp, bias, R, ldr, Y, ldy, y_hi_, y_lo_, lds, y_exp,
                               split_cols, y_first_col, relu_out, split_relu, n_rows, in_features, out_features, flags, stream, nullptr);
}

extern "C" int nfk_affine_coupling_final_f16x3(const void* a_hi, const void* a_lo, int64_t lda, int32_t a_exp, const void* w_hi,
                                               const void* w_lo, int64_t ldw, int32_t w_exp, const float* bias, int32_t hidden_features,
                                               const float* x, int64_t ldx, const int32_t* t_cols, int32_t t_col0, int32_t d_t,
                                               int32_t mult, int32_t scale_activation, int inverse, float* y, int64_t ldy,
                                               float* lad_accum, int64_t n_rows, int32_t* flags, void* stream) {
    NFK_REQUIRE(d_t >= 1 && (mult == 1 || mult == 2) && (scale_activation == 0 || scale_activation == 1), "bad coupling description");
    if (n_rows == 0) return NFK_OK;
    NFK_REQUIRE(x && y && (t_cols || t_col0 >= 0), "NULL pointer");
    CouplingEpilogue ce{x, ldx, y, ldy, t_cols, t_col0, d_t, mult, scale_activation, inverse, lad_accum};
    return linear_f16x3_launch(a_hi, a_lo, lda, a_exp, w_hi, w_lo, ldw, w_exp, bias, nullptr, 0, nullptr, 0, nullptr, nullptr, 0, 0, 0, 0,
                               0, 0, n_rows, hidden_features, mult * d_t, flags, stream, &ce);
}

static int linear_f16x3_launch(const void* a_hi_, const void* a_lo_, int64_t lda, int32_t a_exp, const void* w_hi_,
                               const void* w_lo_, int64_t ldw, int32_t w_exp, const float* bias, const float* R, int64_t ldr,
                               float* Y, int64_t ldy, void* y_hi_, void* y_lo_, int64_t lds, int32_t y_exp, int32_t split_cols,
                               int32_t y_first_col, int relu_out, int split_relu, int64_t n_rows, int32_t in_features,
                               int32_t out_features, int32_t* flags, void* stream, const CouplingEpilogue* ce) {
    const __half* a_hi = (const __half*)a_hi_; const __half* a_lo = (const __half*)a_lo_;
    const __half* w_hi = (const __half*)w_hi_; const __half* w_lo = (const __half*)w_lo_;
    __half* y_hi = (__half*)y_hi_; __half* y_lo = (__half*)y_lo_;
    NFK_REQUIRE(n_rows >= 0 && in_features >= 1 && out_features >= 1, "bad sizes");
    if (n_rows == 0) return NFK_OK;
    NFK_REQUIRE(a_hi && a_lo && w_hi && w_lo, "NULL operand pointer");
    NFK_REQUIRE(ce || Y || (y_hi && y_lo), "no output requested");
    NFK_REQUIRE((y_hi == nullptr) == (y_lo == nullptr), "y_hi and y_lo must be given together");
    NFK_REQUIRE(nfk_linear_f16x3_supported(lda, ldw, in_features), "f16x3 path needs in_features, lda, ldw multiples of 8");
    NFK_REQUIRE(aligned16(a_hi) && aligned16(a_lo) && aligned16(w_hi) && aligned16(w_lo), "operands must be 16-byte aligned");
    NFK_REQUIRE(n_rows < (1ll << 31), "n_rows too large for one launch");
    NFK_REQUIRE(pow2_exp_ok(a_exp) && pow2_exp_ok(w_exp) && pow2_exp_ok(y_exp), "scale exponent out of range");

    tc::Params p;
    p.bias = bias; p.residual = R; p.y = Y; p.y_hi = y_hi; p.y_lo = y_lo; p.flags = flags;
    p.acc_scale = ldexpf(1.0f, a_exp + w_exp); p.inv_acc_scale = ldexpf(1.0f, -(a_exp + w_exp)); p.out_scale = ldexpf(1.0f, y_exp);
    p.split_n = split_cols > 0 ? split_cols : out_features;
    p.ldr = ldr; p.ldy = ldy; p.lds = lds; p.n_rows = n_rows; p.K = in_features; p.N = out_features;
    p.relu_out = relu_out; p.split_relu = split_relu;
    p.y_first_col = y_first_col > 0 ? y_first_col : 0;
    p.cx = nullptr; p.cy = nullptr; p.c_cols = nullptr; p.c_lad = nullptr; p.ldcx = p.ldcy = 0;
    p.c_col0 = p.c_dt = p.c_mult = p.c_act = p.c_inverse = 0;
    if (ce) {
        p.cx = ce->x; p.cy = ce->y; p.c_cols = ce->t_cols; p.c_lad = ce->lad; p.ldcx = ce->ldx; p.ldcy = ce->ldy;
        p.c_col0 = ce->t_col0; p.c_dt = ce->d_t; p.c_mult = ce->mult; p.c_act = ce->act; p.c_inverse = ce->inverse;
    }
    p.num_n_tiles = (out_features + tc::BN_MAX - 1) / tc::BN_MAX;
    int bn = (out_features + p.num_n_tiles - 1) / p.num_n_tiles;
    bn = (bn + 15) / 16 * 16;
    p.BN = bn;
    p.num_n_tiles = (out_features + bn - 1) / bn;
    p.num_m_tiles = (int)((n_rows + tc::BM - 1) / tc::BM);

    const int CL = p.num_m_tiles >= 2 ? 2 : 1;
    // ring split: weight slots hold the BN rows of a K-slab, hi part then lo part, each rounded to the 1024-byte swizzle
    // alignment; the rest of the ring holds 16 KB A slots
    p.w_slot_bytes = 2 * ((bn * tc::ROW_BYTES + 1023) / 1024 * 1024);
    p.w_stages = 3;
    p.a_stages = (tc::LIN_RING_BYTES - p.w_stages * p.w_slot_bytes) / tc::LIN_A_STAGE_BYTES;
    if (p.a_stages > tc::LIN_A_STAGES_MAX) p.a_stages = tc::LIN_A_STAGES_MAX;
    CUtensorMap ma_hi, ma_lo, mw_hi, mw_lo;
    int rc;
    if ((rc = tc::make_map(&ma_hi, a_hi, n_rows, in_features, lda, tc::BM))) return rc;
    if ((rc = tc::make_map(&ma_lo, a_lo, n_rows, in_features, lda, tc::BM))) return rc;
    if ((rc = tc::make_map(&mw_hi, w_hi, out_features, in_features, ldw, bn / CL))) return rc;
    if ((rc = tc::make_map(&mw_lo, w_lo, out_features, in_features, ldw, bn / CL))) return rc;
    // staged TMA stores need 16-byte aligned bases and row pitches for every requested output
    CUtensorMap my = mw_hi, myh = mw_hi, myl = mw_hi, myt = mw_hi, myht = mw_hi, mylt = mw_hi;   // placeholders (never dereferenced)
    p.tma_store = (!ce && (!Y || (aligned16(Y) && ldy % 4 == 0)) && (!y_hi || (aligned16(y_hi) && aligned16(y_lo) && lds % 8 == 0))) ? 1 : 0;
    if (p.tma_store) {
        const int64_t pn = p.split_n < out_features ? p.split_n : out_features;
        if (Y && (rc = tc::make_store_map(&my, Y, false, n_rows, out_features, ldy))) return rc;
        if (y_hi && (rc = tc::make_store_map(&myh, y_hi, true, n_rows, pn, lds))) return rc;
        if (y_hi && (rc = tc::make_store_map(&myl, y_lo, true, n_rows, pn, lds))) return rc;
        // the second column half of a tile is bn - 128 wide: what does not fill a 32- (fp32) / 64-column (fp16) chunk leaves
        // through narrow chunks
        const int w1 = bn > 128 ? bn - 128 : bn;
        if (Y && w1 % 32 && (rc = tc::make_store_map(&myt, Y, false, n_rows, out_features, ldy, w1 % 32))) return rc;
        if (y_hi && w1 % 64 && (rc = tc::make_store_map(&myht, y_hi, true, n_rows, pn, lds, w1 % 64))) return rc;
        if (y_hi && w1 % 64 && (rc = tc::make_store_map(&mylt, y_lo, true, n_rows, pn, lds, w1 % 64))) return rc;
    }

    static DeviceOnce attr_once;
    int attr_dev = 0;
    if (attr_once.pending(&attr_dev)) {
        cudaError_t e = cudaFuncSetAttribute(tc::linear_f16x3_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::LIN_SMEM_BYTES);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(tc::linear_f16x3_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::LIN_SMEM_BYTES);
        if (e != cudaSuccess) return fail(NFK_E_CUDA, "cudaFuncSetAttribute(smem=%d): %s", tc::LIN_SMEM_BYTES, cudaGetErrorString(e));
        attr_once.mark(attr_dev);
    }
    const int units = (p.num_m_tiles + CL - 1) / CL;
    const int max_clusters = tc::sm_count() / CL;
    // a CTA walks the column tiles of its row block back to back: the activations are read from HBM once and re-read from L2
    // (r1 measured no gain from this order -- its single 3-stage ring was bound by operand latency, not by DRAM traffic)
    p.n_inner = (p.num_n_tiles > 1 && units >= max_clusters) ? 1 : 0;
    const int work = units * p.num_n_tiles;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(CL * (work < max_clusters ? work : max_clusters)));
    cfg.blockDim = dim3(tc::THREADS);
    cfg.dynamicSmemBytes = tc::LIN_SMEM_BYTES;
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CL; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t le = CL == 2 ? cudaLaunchKernelEx(&cfg, tc::linear_f16x3_kernel<2>, ma_hi, ma_lo, mw_hi, mw_lo, my, myh, myl, myt, myht, mylt, p)
                             : cudaLaunchKernelEx(&cfg, tc::linear_f16x3_kernel<1>, ma_hi, ma_lo, mw_hi, mw_lo, my, myh, myl, myt, myht, mylt, p);
    if (le != cudaSuccess) return fail(NFK_E_CUDA, "cudaLaunchKernelEx(linear_f16x3_kernel, cluster %d): %s", CL, cudaGetErrorString(le));
    return check_launch("linear_f16x3_kernel");
}
