// ONE kernel per PiecewiseRationalQuadraticCouplingTransform step (reference: coupling.py:73-99, 279-293, 549-582 around
// nn/nets/resnet.py:92-100 and splines/rational_quadratic.py:13-181): the WHOLE conditioner -- initial layer, the square
// layers of the residual blocks, the final layer -- on tcgen05 tensor cores, the spline, the scatter of the transformed
// features and the per-row log|det| in the epilogue.  Nothing the conditioner computes is written to global memory:
//
//   * a CTA owns a 128-row tile from the first layer to the spline.  The activation of the tile lives in shared memory as
//     the K-major fp16 (hi, lo) split pair the NEXT layer multiplies ("R": 8 K-slabs x [hi 8 KB | lo 8 KB] = 128 KB, written
//     by the epilogue warps in the SWIZZLE_64B placement the UMMA descriptors read); only weights stream (L2-resident,
//     each CTA of a 2-CTA cluster fetches half of every box and multicasts it to both);
//   * the final layer walks the column tiles of the packed weight (MP rows per transformed feature, nfk_rq_coupling_tc.cu)
//     against the SAME resident operand: the round-1 kernel re-streamed the 128 x 256 pair for each of its 40 column tiles
//     (L2 -> SM 159 KB per row, the chip-wide L2 request bandwidth was what its tensor pipe waited for);
//   * the residual-block skip tensor goes through a per-CTA fp32 scratch (one 128 x H tile per CTA, L2-resident, every thread
//     reads back exactly what it wrote).
//
// Arithmetic is that of nfk_linear_tc.cu / nfk_rq_coupling_tc.cu: fp16 split pairs with power-of-two scales, three
// kind::f16 MMAs per K-step, partial sums of STEP_DRAIN_TRUNK = 4 (trunk) / STEP_DRAIN_FINAL = 8 (final layer) K-slabs
// drained from TMEM and accumulated in registers with round-to-nearest adds.
//
// Shared memory (dynamic, 1024-aligned):
//   [0, 128 KB)        R
//   [128 KB, 208 KB)   weight ring, three geometries (the producer drains the ring before it switches):
//        G0 initial layer : 4 stages x 48 KB [A hi | A lo | W hi | W lo] laid from offset 0 -- over R, which is dead until the
//                           initial layer's epilogue writes it
//        G1 square layers : 5 units  x 16 KB [W hi | W lo] of one K-slab x one column chunk (H/2 columns when H > 128)
//        G2 final layer   : 3 stages x 24 KB [W hi | W lo] of one K-slab x one column tile (BN <= 192)
//   then barriers, log|det| partials, packed-bias double buffer, 3 output staging buffers.
// TMEM: 2 partial accumulators x 256 columns.
#include <string.h>

#include "fused_spline.cuh"

namespace nfk {
namespace tc {

constexpr int STEP_MAX_LAYERS = 9;                                   // initial layer + up to 8 square layers
// K-slabs accumulated inside the tensor core (round-toward-zero adds) before a partial sum is drained to registers.  Draining is
// not free: TMEM reads run at ~64 B/clk per SM, a 128 x 192 fp32 partial sum is 1536 cycles of that against 96 cycles per MMA.
// Final layer (spline logits, insensitive): the whole K = 256 in one partial sum; trunk layers: K = 128 per partial sum.
// Measured (cfg 3, 2^20 rows, parity_check of bench.py against the CPU oracle): final 4 -> 8: 182 -> 175 ms in this kernel,
// rel. error 2.2e-6 -> 2.4e-6; trunk 2 -> 4: -2 ms, unchanged error (profiles/drain_sweep_r2.txt).
constexpr int STEP_DRAIN_FINAL = 8;
constexpr int STEP_DRAIN_TRUNK = 4;
constexpr int STEP_SLAB_BYTES = 2 * A_BYTES;                         // one K-slab of R: hi | lo
constexpr int STEP_R_BYTES = (BN_MAX / BK) * STEP_SLAB_BYTES;        // 128 KB
constexpr int STEP_RING_BYTES = 80 * 1024;
constexpr int STEP_G0_STAGES = 4;                                    // x STAGE_BYTES (48 KB)
constexpr int STEP_G1_UNITS = 5;
constexpr int STEP_G1_UNIT_BYTES = 16384;
constexpr int STEP_G1_LO_OFF = 8192;
constexpr int STEP_G2_STAGES = 3;
constexpr int STEP_G2_STAGE_BYTES = 24576;
constexpr int STEP_G2_LO_OFF = 12288;
constexpr int STEP_BN_MAX = 192;                                     // widest final-layer column tile
constexpr int STEP_NBAR = 6;                                         // ring barriers (max stages of any geometry)
constexpr int STEP_BAR_OFF = STEP_R_BYTES + STEP_RING_BYTES;
constexpr int STEP_BIAS_OFF = STEP_BAR_OFF + 256;                    // [2][192] fp32 packed bias of the current / next column tile
constexpr int STEP_Y_OFF = STEP_BIAS_OFF + 2 * STEP_BN_MAX * 4;      // 3 x 4 KB output staging (128-byte aligned)
constexpr int STEP_Y_BUF_BYTES = 4096;
constexpr int STEP_X_OFF = STEP_Y_OFF + 3 * STEP_Y_BUF_BYTES;        // 4 KB: every epilogue thread's next inputs (cp.async), and
constexpr int STEP_X_BYTES = 4096;                                   // at the end of a row block the log|det| partials
constexpr int STEP_SMEM_BYTES = STEP_X_OFF + STEP_X_BYTES + 1024 /*alignment slack*/;
static_assert(STEP_G0_STAGES * STAGE_BYTES <= STEP_R_BYTES + STEP_RING_BYTES, "G0 ring");
static_assert(STEP_G1_UNITS * STEP_G1_UNIT_BYTES <= STEP_RING_BYTES && STEP_G2_STAGES * STEP_G2_STAGE_BYTES <= STEP_RING_BYTES, "ring");
static_assert(STEP_Y_OFF % 128 == 0, "staging alignment");
static_assert(STEP_SMEM_BYTES <= 232448, "coupling-step kernel shared memory");

// layer_flags bits (include/nfk.h: NfkCouplingStep)
constexpr int SL_RELU_OUT = 1;     // relu on (acc + bias)
constexpr int SL_ADD_SKIP = 2;     // + the saved skip tensor (never combined with SL_RELU_OUT)
constexpr int SL_SAVE_SKIP = 4;    // the fp32 result is the skip tensor of a later layer
constexpr int SL_SPLIT_RELU = 8;   // the consumer of this layer's output applies relu to its input

// Column tile of the final layer: TF features (8, 4 or 2) of MP packed rows each, shared by EWG epilogue warpgroups (FPT
// features per thread).  EWG = 4 puts four warps on every scheduler: the spline epilogue is a long dependent instruction
// stream, two warps per scheduler left 56 % of the issue slots empty (ncu, r2: issue active 44 %, tensor pipe 43 %).
template <int NB, bool TAILS, int EWG = 2>
struct StepCfg {
    static constexpr int M = TAILS ? 3 * NB - 1 : 3 * NB + 1;
    static constexpr int MP = (M + 7) / 8 * 8;
    static constexpr int TF = 8 * MP <= STEP_BN_MAX ? 8 : (4 * MP <= STEP_BN_MAX ? 4 : 2);   // features per column tile
    static constexpr int FPT = TF / EWG;                 // features per epilogue thread
    static constexpr int HC = FPT * MP;                  // accumulator columns per epilogue thread
    static constexpr int BN = TF * MP;                   // MMA N = packed weight rows per tile
    static_assert(FPT >= 1 && FPT * EWG == TF, "too many epilogue warpgroups for this bin count");
    static constexpr int YG = TF >= 4 ? 1 : 4 / TF;      // column tiles per fp32 output store (rows of >= 16 bytes)
    static constexpr int YROW = YG * TF;                 // floats per staged row: 8 or 4
    static constexpr int YG16 = 8 / TF;                  // column tiles per pair output store
    static constexpr int YROW16 = 8;                     // halfs per staged row (hi rows, then lo rows)
    static_assert(BN % 16 == 0 && BN <= STEP_BN_MAX && 2 * MP <= STEP_BN_MAX, "unsupported bin count for the coupling-step kernel");
    static_assert(BM * YROW * 4 <= STEP_Y_BUF_BYTES && 2 * BM * YROW16 * 2 <= STEP_Y_BUF_BYTES, "staging buffer");
    static_assert(128 * EWG * FPT * 4 <= STEP_X_BYTES && (EWG - 1) * 128 * 4 <= STEP_X_BYTES, "x staging");
};

struct StepParams {
    // ---- conditioner trunk
    const float* bias_trunk;      // [num_layers * H]: initial layer, then the square layers
    float4* skip_buf;             // [gridDim.x][H / 4][128] scratch
    int H, K0, num_layers;        // num_layers = 1 + number of square layers
    int layer_flags[STEP_MAX_LAYERS];
    float acc_scale[STEP_MAX_LAYERS], inv_acc_scale[STEP_MAX_LAYERS];
    float act_scale;              // 2^e_act: exponent of every hidden activation pair
    int trunk_only;               // stop after the trunk: its output pair leaves through map_h_hi / map_h_lo
    // ---- final layer + spline (nfk_rq_coupling_tc.cu: FusedParams)
    const float* bias;            // packed [d_t * MP]
    const float* x;
    float* y;
    const int32_t* t_cols;
    int t_col0, tma_y, pair_only;
    uint32_t zero;                // always 0 (mbar_arrive_after_loads)
    int tma_x;                    // inputs of the transformed features arrive as TMA boxes (consecutive columns, 16-byte aligned)
    float out_scale;
    float* lad_accum;
    int32_t* flags;
    int64_t ldx, ldy, n_rows;
    int d_t, num_m_tiles, num_n_tiles, inverse;
    float inv_acc_scale_f;
    SplineParams sp;
};

__device__ __forceinline__ void step_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(map)),
                 "r"(src), "r"(c0), "r"(c1)
                 : "memory");
}

template <int NB, bool TAILS, int CL, int EWG>
__global__ void __launch_bounds__(128 + 128 * EWG, 1)
rq_coupling_step_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                        const __grid_constant__ CUtensorMap map_w0_hi, const __grid_constant__ CUtensorMap map_w0_lo,
                        const __grid_constant__ CUtensorMap map_wt_hi, const __grid_constant__ CUtensorMap map_wt_lo,
                        const __grid_constant__ CUtensorMap map_wf_hi, const __grid_constant__ CUtensorMap map_wf_lo,
                        const __grid_constant__ CUtensorMap map_y, const __grid_constant__ CUtensorMap map_yh,
                        const __grid_constant__ CUtensorMap map_yl, const __grid_constant__ CUtensorMap map_h_hi,
                        const __grid_constant__ CUtensorMap map_h_lo, const __grid_constant__ CUtensorMap map_x,
                        const StepParams p) {
    using Cfg = StepCfg<NB, TAILS, EWG>;
    constexpr int MP = Cfg::MP, FPT = Cfg::FPT, HC = Cfg::HC, BN = Cfg::BN, TF = Cfg::TF;
    constexpr int NEPI = 4 * EWG;                  // epilogue warps
    constexpr int CT = BN_MAX / EWG;               // trunk-layer columns per epilogue thread

    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
    const uint32_t ring = smem_base + STEP_R_BYTES;
    const uint32_t bars = smem_base + STEP_BAR_OFF;
    const uint32_t bar_full = bars, bar_empty = bars + 8 * STEP_NBAR;
    const uint32_t bar_tfull = bars + 16 * STEP_NBAR, bar_tempty = bar_tfull + 16;
    const uint32_t bar_aready = bar_tfull + 32;   // the epilogue warps have written the next layer's operand into R
    const uint32_t bar_outready = bar_tfull + 40; // trunk_only: ... the trunk's output, ready for the TMA stores
    const uint32_t bar_bfull = bar_tfull + 48, bar_bempty = bar_tfull + 64;
    const uint32_t bar_xfull = bar_tfull + 80, bar_xempty = bar_tfull + 96;      // the two TMA-staged input tiles (tma_x)
    static_assert(16 * STEP_NBAR + 112 + 8 <= 248, "barrier block");
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem_gen + STEP_BAR_OFF + 248);
    // [2][128 rows][TF] fp32 input tiles in the tail of the ring region, which the final layer's geometry (G2) leaves unused
    constexpr int X_TILE_OFF = STEP_R_BYTES + STEP_G2_STAGES * STEP_G2_STAGE_BYTES;
    static_assert(X_TILE_OFF + 2 * BM * 8 * 4 <= STEP_R_BYTES + STEP_RING_BYTES, "input tiles must fit behind the G2 stages");
    float* s_bias = reinterpret_cast<float*>(smem_gen + STEP_BIAS_OFF);        // [2][STEP_BN_MAX]
    float* s_lad = reinterpret_cast<float*>(smem_gen + STEP_X_OFF);            // [EWG-1][128], aliases the (then idle) x staging

    uint32_t tid_x;
    asm volatile("mov.u32 %0, %%tid.x;" : "=r"(tid_x));
    const int warp = tid_x >> 5, lane = tid_x & 31;
    const int num_k0 = (p.K0 + BK - 1) / BK;                 // K-slabs of the initial layer
    const int num_kh = p.H / BK;                             // K-slabs of every other layer (H is a multiple of 32)
    constexpr int drain_t = STEP_DRAIN_TRUNK;                // K-slabs per partial sum of a trunk layer
    const int groups0 = (num_k0 + drain_t - 1) / drain_t;
    const int groupsh = (num_kh + drain_t - 1) / drain_t;
    constexpr int drain_f = STEP_DRAIN_FINAL;                // K-slabs per partial sum of the final layer
    const int groupsf = (num_kh + drain_f - 1) / drain_f;
    const int nch = p.H > 128 ? 2 : 1;                       // column chunks of a square layer
    const int ch = p.H / nch;                                // columns per chunk (multiple of 16)

    if (tid_x == 0) {
        for (int s = 0; s < STEP_NBAR; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, CL); }
        for (int a = 0; a < 2; ++a) { mbar_init(bar_tfull + 8 * a, 1); mbar_init(bar_tempty + 8 * a, NEPI); }
        mbar_init(bar_aready, NEPI); mbar_init(bar_outready, NEPI);
        for (int b = 0; b < 2; ++b) { mbar_init(bar_bfull + 8 * b, 1); mbar_init(bar_bempty + 8 * b, NEPI); }
        for (int b = 0; b < 2; ++b) { mbar_init(bar_xfull + 8 * b, 1); mbar_init(bar_xempty + 8 * b, NEPI); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        prefetch_tmap(&map_a_hi); prefetch_tmap(&map_a_lo); prefetch_tmap(&map_w0_hi); prefetch_tmap(&map_w0_lo);
        prefetch_tmap(&map_wt_hi); prefetch_tmap(&map_wt_lo); prefetch_tmap(&map_wf_hi); prefetch_tmap(&map_wf_lo);
    }
    if (warp == 1) tmem_alloc(smem_u32(tmem_slot), 512);
    tc_fence_before();
    if (CL > 1) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int cta_rank = CL > 1 ? (int)cluster_ctarank() : 0;
    constexpr uint16_t cl_mask = (uint16_t)((1u << CL) - 1);
    const int units = (p.num_m_tiles + CL - 1) / CL;         // groups of CL neighbouring 128-row tiles
    const int first = blockIdx.x / CL, step = gridDim.x / CL;

    if (warp < 4) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 40;" ::: "memory");
        if (warp == 0) {
            // ================================================= TMA producer (one elected thread: uniform datapath, see elect_one)
            if (elect_one()) {
                uint32_t uses = 0;                                   // bit s: parity of the number of loads issued into ring slot s
                auto slot_wait = [&](int s) { mbar_wait(bar_empty + 8 * s, ((uses >> s) & 1u) ^ 1u); };   // last use released by every CTA
                auto drain = [&]() {
                    for (int s = 0; s < STEP_NBAR; ++s) slot_wait(s);
                };
                int bslot = 0; uint32_t bphase = 0, out_phase = 0;
                int xslot = 0; uint32_t xphase = 0;
                for (int u = first; u < units; u += step) {
                    const int m0 = (u * CL + cta_rank) * BM;
                    // ---- G0: initial layer, A and W streamed through 48 KB stages laid over R
                    drain();                                         // the previous tile's last MMAs have read R and the ring
                    {
                        const uint32_t tx = 2u * A_BYTES + 2u * (uint32_t)p.H * ROW_BYTES;
                        const int wrows = p.H / CL;
                        int s = 0;
                        for (int ks = 0; ks < num_k0; ++ks) {
                            slot_wait(s);
                            const uint32_t full = bar_full + 8 * s;
                            const uint32_t sa = smem_base + s * STAGE_BYTES;
                            mbar_expect_tx(full, tx);
                            tma_load_2d(sa, &map_a_hi, full, ks * BK, m0);
                            tma_load_2d(sa + A_BYTES, &map_a_lo, full, ks * BK, m0);
                            if (CL == 1) {
                                tma_load_2d(sa + 2 * A_BYTES, &map_w0_hi, full, ks * BK, 0);
                                tma_load_2d(sa + 2 * A_BYTES + B_BYTES, &map_w0_lo, full, ks * BK, 0);
                            } else {
                                const uint32_t off = (uint32_t)(cta_rank * wrows) * ROW_BYTES;
                                tma_load_2d_multicast(sa + 2 * A_BYTES + off, &map_w0_hi, full, ks * BK, cta_rank * wrows, cl_mask);
                                tma_load_2d_multicast(sa + 2 * A_BYTES + B_BYTES + off, &map_w0_lo, full, ks * BK, cta_rank * wrows, cl_mask);
                            }
                            uses ^= 1u << s;
                            if (++s == STEP_G0_STAGES) s = 0;
                        }
                    }
                    // ---- G1: square layers, one unit = one K-slab of one column chunk
                    if (p.num_layers > 1) {
                        drain();                                     // the initial layer's MMAs are done with the stages over the ring
                        const uint32_t tx = 2u * (uint32_t)ch * ROW_BYTES;
                        const int wrows = ch / CL;
                        int s = 0;
                        for (int l = 1; l < p.num_layers; ++l) {
                            for (int g = 0; g < groupsh; ++g) {
                                const int slabs = min(drain_t, num_kh - g * drain_t);
                                for (int c = 0; c < nch; ++c) {
                                    for (int j = 0; j < slabs; ++j) {
                                        const int ks = g * drain_t + j;
                                        const int row0 = (l - 1) * p.H + c * ch;
                                        slot_wait(s);
                                        const uint32_t full = bar_full + 8 * s;
                                        const uint32_t su = ring + s * STEP_G1_UNIT_BYTES;
                                        mbar_expect_tx(full, tx);
                                        if (CL == 1) {
                                            tma_load_2d(su, &map_wt_hi, full, ks * BK, row0);
                                            tma_load_2d(su + STEP_G1_LO_OFF, &map_wt_lo, full, ks * BK, row0);
                                        } else {
                                            const uint32_t off = (uint32_t)(cta_rank * wrows) * ROW_BYTES;
                                            tma_load_2d_multicast(su + off, &map_wt_hi, full, ks * BK, row0 + cta_rank * wrows, cl_mask);
                                            tma_load_2d_multicast(su + STEP_G1_LO_OFF + off, &map_wt_lo, full, ks * BK, row0 + cta_rank * wrows, cl_mask);
                                        }
                                        uses ^= 1u << s;
                                        if (++s == STEP_G1_UNITS) s = 0;
                                    }
                                }
                            }
                        }
                    }
                    if (p.trunk_only) {
                        // the epilogue warps have left the trunk's output pair in R: send it out, and do not load the next tile over
                        // it before the stores have read it
                        mbar_wait(bar_outready, out_phase);
                        out_phase ^= 1;
                        for (int ks = 0; ks < num_kh; ++ks) {
                            step_store_2d(&map_h_hi, smem_base + ks * STEP_SLAB_BYTES, ks * BK, m0);
                            step_store_2d(&map_h_lo, smem_base + ks * STEP_SLAB_BYTES + A_BYTES, ks * BK, m0);
                        }
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                        continue;
                    }
                    // ---- G2: final layer, one stage = one K-slab of one column tile
                    drain();
                    {
                        constexpr uint32_t tx = 2u * (uint32_t)BN * ROW_BYTES;
                        constexpr int wrows = BN / CL;
                        int s = 0;
                        for (int n = 0; n < p.num_n_tiles; ++n) {
                            if (p.tma_x) {   // this tile's inputs: box [128 rows][TF columns] of x (columns past d_t are zero-filled)
                                mbar_wait(bar_xempty + 8 * xslot, xphase ^ 1);
                                mbar_expect_tx(bar_xfull + 8 * xslot, (uint32_t)(BM * TF * 4));
                                tma_load_2d(smem_base + X_TILE_OFF + xslot * (BM * TF * 4), &map_x, bar_xfull + 8 * xslot,
                                            p.t_col0 + n * TF, m0);
                                if (++xslot == 2) { xslot = 0; xphase ^= 1; }
                            }
                            {   // this tile's slice of the packed bias -> s_bias[bslot]
                                const int cols = min(BN, p.d_t * MP - n * BN);
                                mbar_wait(bar_bempty + 8 * bslot, bphase ^ 1);
                                mbar_expect_tx(bar_bfull + 8 * bslot, (uint32_t)cols * 4u);
                                bulk_load_1d(smem_u32(s_bias + bslot * STEP_BN_MAX), p.bias + (int64_t)n * BN, (uint32_t)cols * 4u,
                                             bar_bfull + 8 * bslot);
                                if (++bslot == 2) { bslot = 0; bphase ^= 1; }
                            }
                            for (int ks = 0; ks < num_kh; ++ks) {
                                slot_wait(s);
                                const uint32_t full = bar_full + 8 * s;
                                const uint32_t sw = ring + s * STEP_G2_STAGE_BYTES;
                                mbar_expect_tx(full, tx);
                                if (CL == 1) {
                                    tma_load_2d(sw, &map_wf_hi, full, ks * BK, n * BN);
                                    tma_load_2d(sw + STEP_G2_LO_OFF, &map_wf_lo, full, ks * BK, n * BN);
                                } else {
                                    const uint32_t off = (uint32_t)(cta_rank * wrows) * ROW_BYTES;
                                    tma_load_2d_multicast(sw + off, &map_wf_hi, full, ks * BK, n * BN + cta_rank * wrows, cl_mask);
                                    tma_load_2d_multicast(sw + STEP_G2_LO_OFF + off, &map_wf_lo, full, ks * BK, n * BN + cta_rank * wrows, cl_mask);
                                }
                                uses ^= 1u << s;
                                if (++s == STEP_G2_STAGES) s = 0;
                            }
                        }
                    }
                }
            }
        } else if (warp == 1) {
            // ================================================= MMA issuer (one elected thread: uniform datapath, see elect_one)
            if (elect_one()) {
            uint32_t seen = 0;                                       // bit s: parity of the number of fills of ring slot s consumed
            auto full_wait = [&](int s) { mbar_wait(bar_full + 8 * s, (seen >> s) & 1u); seen ^= 1u << s; };
            auto release = [&](int s) {
                if (CL == 1) umma_commit(bar_empty + 8 * s); else umma_commit_multicast(bar_empty + 8 * s, cl_mask);
            };
            const uint32_t idesc0 = make_idesc(p.H), idesc1 = make_idesc(ch), idescf = make_idesc(BN);
            uint32_t gc = 0;                                         // partial sums so far: buffer gc & 1, use (gc >> 1) of it
            uint32_t aready_phase = 0;
            for (int u = first; u < units; u += step) {
                // ---- initial layer: A and W from the G0 stages
                {
                    int s = 0;
                    for (int g = 0; g < groups0; ++g, ++gc) {
                        const int slabs = min(drain_t, num_k0 - g * drain_t);
                        const int acc = gc & 1u;
                        mbar_wait(bar_tempty + 8 * acc, ((gc >> 1) & 1u) ^ 1u);
                        const uint32_t d_tmem = tmem_base + acc * BN_MAX;
                        for (int j = 0; j < slabs; ++j) {              // per slab: the two small cross terms, the main product, release
                            full_wait(s);
                            tc_fence_after();
                            const uint32_t sa = smem_base + s * STAGE_BYTES;
                            const uint64_t a_hi = make_smem_desc(sa), a_lo = make_smem_desc(sa + A_BYTES);
                            const uint64_t w_hi = make_smem_desc(sa + 2 * A_BYTES), w_lo = make_smem_desc(sa + 2 * A_BYTES + B_BYTES);
#pragma unroll
                            for (int kk = 0; kk < BK / 16; ++kk) {
                                const uint64_t adv = (uint64_t)(kk * 2);
                                umma_f16(d_tmem, a_lo + adv, w_hi + adv, idesc0, (j | kk) != 0);
                                umma_f16(d_tmem, a_hi + adv, w_lo + adv, idesc0, 1);
                            }
#pragma unroll
                            for (int kk = 0; kk < BK / 16; ++kk) {
                                const uint64_t adv = (uint64_t)(kk * 2);
                                umma_f16(d_tmem, a_hi + adv, w_hi + adv, idesc0, 1);
                            }
                            release(s);
                            if (++s == STEP_G0_STAGES) s = 0;
                        }
                        umma_commit(bar_tfull + 8 * acc);
                    }
                }
                // ---- square layers: A from R, W from the G1 units
                {
                    int s = 0;
                    for (int l = 1; l < p.num_layers; ++l) {
                        mbar_wait(bar_aready, aready_phase);
                        aready_phase ^= 1;
                        tc_fence_after();
                        for (int g = 0; g < groupsh; ++g, ++gc) {
                            const int slabs = min(drain_t, num_kh - g * drain_t);
                            const int acc = gc & 1u;
                            mbar_wait(bar_tempty + 8 * acc, ((gc >> 1) & 1u) ^ 1u);
                            for (int c = 0; c < nch; ++c) {
                                const uint32_t d_tmem = tmem_base + acc * BN_MAX + c * ch;
                                for (int j = 0; j < slabs; ++j) {
                                    full_wait(s);
                                    tc_fence_after();
                                    const uint32_t sa = smem_base + (g * drain_t + j) * STEP_SLAB_BYTES;
                                    const uint32_t sw = ring + s * STEP_G1_UNIT_BYTES;
                                    const uint64_t a_hi = make_smem_desc(sa), a_lo = make_smem_desc(sa + A_BYTES);
                                    const uint64_t w_hi = make_smem_desc(sw), w_lo = make_smem_desc(sw + STEP_G1_LO_OFF);
#pragma unroll
                                    for (int kk = 0; kk < BK / 16; ++kk) {
                                        const uint64_t adv = (uint64_t)(kk * 2);
                                        umma_f16(d_tmem, a_lo + adv, w_hi + adv, idesc1, (j | kk) != 0);
                                        umma_f16(d_tmem, a_hi + adv, w_lo + adv, idesc1, 1);
                                    }
#pragma unroll
                                    for (int kk = 0; kk < BK / 16; ++kk) {
                                        const uint64_t adv = (uint64_t)(kk * 2);
                                        umma_f16(d_tmem, a_hi + adv, w_hi + adv, idesc1, 1);
                                    }
                                    release(s);
                                    if (++s == STEP_G1_UNITS) s = 0;
                                }
                            }
                            umma_commit(bar_tfull + 8 * acc);
                        }
                    }
                }
                if (p.trunk_only) continue;
                // ---- final layer: A from R, one G2 stage per K-slab of a column tile.  Per slab: cross terms, then the main
                // product, then the stage is released (3 stages: holding two slabs for a cross-terms-first pair would leave one
                // load in flight)
                {
                    mbar_wait(bar_aready, aready_phase);
                    aready_phase ^= 1;
                    tc_fence_after();
                    int s = 0;
                    for (int n = 0; n < p.num_n_tiles; ++n) {
                        for (int g = 0; g < groupsf; ++g, ++gc) {
                            const int slabs = min(drain_f, num_kh - g * drain_f);
                            const int acc = gc & 1u;
                            mbar_wait(bar_tempty + 8 * acc, ((gc >> 1) & 1u) ^ 1u);
                            const uint32_t d_tmem = tmem_base + acc * BN_MAX;
                            for (int j = 0; j < slabs; ++j) {
                                full_wait(s);
                                tc_fence_after();
                                const uint32_t sa = smem_base + (g * drain_f + j) * STEP_SLAB_BYTES;
                                const uint32_t sw = ring + s * STEP_G2_STAGE_BYTES;
                                const uint64_t a_hi = make_smem_desc(sa), a_lo = make_smem_desc(sa + A_BYTES);
                                const uint64_t w_hi = make_smem_desc(sw), w_lo = make_smem_desc(sw + STEP_G2_LO_OFF);
#pragma unroll
                                for (int kk = 0; kk < BK / 16; ++kk) {
                                    const uint64_t adv = (uint64_t)(kk * 2);
                                    umma_f16(d_tmem, a_lo + adv, w_hi + adv, idescf, (j | kk) != 0);
                                    umma_f16(d_tmem, a_hi + adv, w_lo + adv, idescf, 1);
                                }
#pragma unroll
                                for (int kk = 0; kk < BK / 16; ++kk) {
                                    const uint64_t adv = (uint64_t)(kk * 2);
                                    umma_f16(d_tmem, a_hi + adv, w_hi + adv, idescf, 1);
                                }
                                release(s);
                                if (++s == STEP_G2_STAGES) s = 0;
                            }
                            umma_commit(bar_tfull + 8 * acc);
                        }
                    }
                }
            }
            }
        }
    } else {
        if (EWG == 2) asm volatile("setmaxnreg.inc.sync.aligned.u32 232;" ::: "memory");
        else asm volatile("setmaxnreg.inc.sync.aligned.u32 104;" ::: "memory");   // 640 x 96 at launch; the control warpgroup frees 56 x 128
        // ================================================= accumulate + epilogues: 4 * EWG warps.  Thread = one row of the tile
        // (TMEM lane) x one 1/EWG share of the columns.
        const int q = warp & 3;
        const int wg = (warp - 4) >> 2;
        const int r_tile = q * 32 + lane;
        int acc = 0; uint32_t acc_phase = 0;
        int flag = 0;
        int bslot = 0; uint32_t bphase = 0;
        int xslot = 0; uint32_t xphase = 0;
        int ybuf = 0;
        float4* skip = p.skip_buf + (size_t)blockIdx.x * (size_t)(p.H / 4) * 128 + r_tile;       // [c4 * 128]: coalesced across lanes
        float* s_x = reinterpret_cast<float*>(smem_gen + STEP_X_OFF) + (tid_x - 128) * FPT;     // this thread's staged inputs
        for (int u = first; u < units; u += step) {
            const int m = u * CL + cta_rank;
            const int64_t row = (int64_t)m * BM + r_tile;
            const bool row_ok = row < p.n_rows;
            // Inputs of the FPT features this thread owns in column tile n -> its shared-memory slot, asynchronously (LDGSTS): a
            // register prefetch was spilled by the compiler and the store waited for the load (ncu, r2: 22 % of the epilogue
            // warps' samples).  Issued one tile ahead (tile 0: before the trunk); read back by the same thread.
            auto prefetch_x = [&](int n) {
                const int jn = (n * EWG + wg) * FPT;
#pragma unroll
                for (int f = 0; f < FPT; ++f) {
                    if (row_ok && jn + f < p.d_t) {
                        const int cf = p.t_cols ? __ldg(p.t_cols + jn + f) : p.t_col0 + jn + f;
                        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(s_x + f)), "l"(p.x + row * p.ldx + cf) : "memory");
                    }
                }
                asm volatile("cp.async.commit_group;" ::: "memory");
            };
            if (!p.trunk_only && !p.tma_x) prefetch_x(0);
            // ------------------------------------------------ conditioner trunk: layer l's epilogue writes layer l+1's operand into R
            for (int l = 0; l < p.num_layers; ++l) {
                const int lf = p.layer_flags[l];
                const bool last = l == p.num_layers - 1;
                const int n0 = wg * CT;
                float sum[CT];
#pragma unroll
                for (int c = 0; c < CT; c += 4) {
                    float4 r4 = make_float4(0.f, 0.f, 0.f, 0.f);
                    if ((lf & SL_ADD_SKIP) && n0 + c < p.H) r4 = skip[(size_t)((n0 + c) >> 2) * 128];
                    sum[c] = r4.x; sum[c + 1] = r4.y; sum[c + 2] = r4.z; sum[c + 3] = r4.w;
                }
                {   // bias: ONE coalesced float4 load per thread (lane l: columns 4l..4l+3 of this thread's CT columns), broadcast by
                    // shuffles -- a broadcast load per float4, each followed by its adds, serialises CT/4 L2 latencies per layer
                    // (measured in the dense-layer kernel, r2: 8 600 cycles per tile)
                    float4 mine = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (4 * lane < CT && n0 + 4 * lane < p.H)
                        mine = __ldg(reinterpret_cast<const float4*>(p.bias_trunk + l * p.H + n0 + 4 * lane));
#pragma unroll
                    for (int c = 0; c < CT; c += 4) {
                        sum[c] += __shfl_sync(0xffffffffu, mine.x, c >> 2);
                        sum[c + 1] += __shfl_sync(0xffffffffu, mine.y, c >> 2);
                        sum[c + 2] += __shfl_sync(0xffffffffu, mine.z, c >> 2);
                        sum[c + 3] += __shfl_sync(0xffffffffu, mine.w, c >> 2);
                    }
                }
                const float as = p.acc_scale[l], ias = p.inv_acc_scale[l];
#pragma unroll
                for (int c = 0; c < CT; ++c) sum[c] *= as;
                const int groups = l == 0 ? groups0 : groupsh;
                for (int g = 0; g < groups; ++g) {
                    mbar_wait(bar_tfull + 8 * acc, acc_phase);
                    tc_fence_after();
                    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * BN_MAX + wg * CT;
                    constexpr int LD = EWG == 2 ? 2 : 1;               // 32-column TMEM loads in flight per wait (register budget)
#pragma unroll
                    for (int c = 0; c < CT; c += 32 * LD) {
                        uint32_t raw[LD][32];
#pragma unroll
                        for (int v = 0; v < LD; ++v) tmem_ld32(taddr + c + 32 * v, raw[v]);
                        tmem_ld_wait();
#pragma unroll
                        for (int v = 0; v < LD; ++v) {
#pragma unroll
                            for (int j = 0; j < 32; j += 2) {
                                const float2 r2 = __fadd2_rn(make_float2(sum[c + 32 * v + j], sum[c + 32 * v + j + 1]),
                                                             make_float2(__uint_as_float(raw[v][j]), __uint_as_float(raw[v][j + 1])));
                                sum[c + 32 * v + j] = r2.x;
                                sum[c + 32 * v + j + 1] = r2.y;
                            }
                        }
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_tempty + 8 * acc);
                    if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                }
                // ---- layer epilogue.  Every MMA of this layer has retired (its last partial sum was drained), so R may be
                // overwritten with the next layer's operand.
#pragma unroll
                for (int c = 0; c < CT; ++c) {
                    float x = sum[c] * ias;
                    if (lf & SL_RELU_OUT) x = fmaxf(x, 0.0f);
                    sum[c] = x;
                }
                if (lf & SL_SAVE_SKIP) {
#pragma unroll
                    for (int c = 0; c < CT; c += 4)
                        if (n0 + c < p.H) skip[(size_t)((n0 + c) >> 2) * 128] = make_float4(sum[c], sum[c + 1], sum[c + 2], sum[c + 3]);
                }
                float amax = 0.0f;
#pragma unroll
                for (int s = 0; s < CT / BK; ++s) {                   // CT / 32 K-slabs of 32 columns per thread
                    const int slab = wg * (CT / BK) + s;
                    if (slab < num_kh) {
                        uint8_t* base = smem_gen + slab * STEP_SLAB_BYTES + r_tile * ROW_BYTES;
#pragma unroll
                        for (int c = 0; c < 4; ++c) {                 // 16-byte pieces of the 64-byte row, SWIZZLE_64B placement
                            __half2 h2[4], l2[4];
#pragma unroll
                            for (int e = 0; e < 4; ++e) {
                                float x0 = sum[32 * s + 8 * c + 2 * e], x1 = sum[32 * s + 8 * c + 2 * e + 1];
                                if (lf & SL_SPLIT_RELU) { x0 = fmaxf(x0, 0.0f); x1 = fmaxf(x1, 0.0f); }
                                x0 *= p.act_scale; x1 *= p.act_scale;
                                amax = fmaxf(amax, fmaxf(fabsf(x0), fabsf(x1)));
                                h2[e] = __floats2half2_rn(x0, x1);
                                const float2 hf = __half22float2(h2[e]);
                                l2[e] = __floats2half2_rn(x0 - hf.x, x1 - hf.y);
                            }
                            const int piece = (c ^ ((r_tile >> 1) & 3)) * 16;
                            *reinterpret_cast<uint4*>(base + piece) = *reinterpret_cast<const uint4*>(h2);
                            *reinterpret_cast<uint4*>(base + A_BYTES + piece) = *reinterpret_cast<const uint4*>(l2);
                        }
                    }
                }
                if (row_ok && !(amax <= 65000.0f)) flag |= 4;
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic writes -> tcgen05.mma / TMA store reads
                __syncwarp();
                if (lane == 0) mbar_arrive((last && p.trunk_only) ? bar_outready : bar_aready);
            }
            if (p.trunk_only) continue;
            // ------------------------------------------------ final layer + spline: the column tiles of this row block
            float lad_row = 0.0f;
            for (int n = 0; n < p.num_n_tiles; ++n) {
                const int j0 = (n * EWG + wg) * FPT;                       // first feature this thread owns in this tile
                float sum[HC];
#pragma unroll
                for (int c = 0; c < HC; ++c) sum[c] = 0.0f;
                for (int g = 0; g < groupsf; ++g) {
                    mbar_wait(bar_tfull + 8 * acc, acc_phase);
                    tc_fence_after();
                    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * BN_MAX + wg * HC;
                    constexpr int LDB = HC <= 48 ? 3 : 4;           // TMEM loads in flight per wait
#pragma unroll
                    for (int c = 0; c < HC; c += 8 * LDB) {
                        uint32_t raw[LDB][8];
#pragma unroll
                        for (int v = 0; v < LDB; ++v)
                            if (c + 8 * v < HC) tmem_ld8(taddr + c + 8 * v, raw[v]);
                        tmem_ld_wait();
#pragma unroll
                        for (int v = 0; v < LDB; ++v)
                            if (c + 8 * v < HC) {
#pragma unroll
                                for (int i = 0; i < 8; i += 2) {
                                    const float2 r2 = __fadd2_rn(make_float2(sum[c + 8 * v + i], sum[c + 8 * v + i + 1]),
                                                                 make_float2(__uint_as_float(raw[v][i]), __uint_as_float(raw[v][i + 1])));
                                    sum[c + 8 * v + i] = r2.x;
                                    sum[c + 8 * v + i + 1] = r2.y;
                                }
                            }
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_tempty + 8 * acc);
                    if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                }
                // ---- this tile's inputs out of the staging slot, the next tile's on their way into it
                float xin[FPT];
                if (p.tma_x) {
                    mbar_wait(bar_xfull + 8 * xslot, xphase);
                    const float* xt = reinterpret_cast<const float*>(smem_gen + X_TILE_OFF + xslot * (BM * TF * 4)) + r_tile * TF + wg * FPT;
#pragma unroll
                    for (int f = 0; f < FPT; ++f) xin[f] = (row_ok && j0 + f < p.d_t) ? xt[f] : 0.0f;
                    // the slot goes back to the producer only once the loads have RETURNED (mbar_arrive_after_loads)
                    uint32_t bits = 0;
#pragma unroll
                    for (int f = 0; f < FPT; ++f) bits |= __float_as_uint(xin[f]);
                    __syncwarp();
                    if (lane == 0) mbar_arrive_after_loads(bar_xempty + 8 * xslot, bits, p.zero);
                    if (++xslot == 2) { xslot = 0; xphase ^= 1; }
                } else {
                    asm volatile("cp.async.wait_group 0;" ::: "memory");
#pragma unroll
                    for (int f = 0; f < FPT; ++f) xin[f] = (row_ok && j0 + f < p.d_t) ? s_x[f] : 0.0f;
                    if (n + 1 < p.num_n_tiles) prefetch_x(n + 1);
                }
                // ---- back from the accumulators' power-of-two scaled domain, plus the packed bias staged in shared memory
                {
                    mbar_wait(bar_bfull + 8 * bslot, bphase);
                    const float4* bias4 = reinterpret_cast<const float4*>(s_bias + bslot * STEP_BN_MAX + wg * HC);
#pragma unroll
                    for (int c = 0; c < HC; c += 4) {
                        const float4 b4 = (j0 + c / MP < p.d_t) ? bias4[c >> 2] : make_float4(0.f, 0.f, 0.f, 0.f);
                        sum[c] = fmaf(sum[c], p.inv_acc_scale_f, b4.x); sum[c + 1] = fmaf(sum[c + 1], p.inv_acc_scale_f, b4.y);
                        sum[c + 2] = fmaf(sum[c + 2], p.inv_acc_scale_f, b4.z); sum[c + 3] = fmaf(sum[c + 3], p.inv_acc_scale_f, b4.w);
                    }
                    uint32_t bits = 0;                    // one component of every LDS.128 (mbar_arrive_after_loads)
#pragma unroll
                    for (int c = 0; c < HC; c += 4) bits |= __float_as_uint(sum[c]);
                    __syncwarp();
                    if (lane == 0) mbar_arrive_after_loads(bar_bempty + 8 * bslot, bits, p.zero);
                    if (++bslot == 2) { bslot = 0; bphase ^= 1; }
                }
                // ---- spline on the FPT features held in registers
                float yy[FPT], ll[FPT];
                if (p.inverse) rqs_eval_lean<NB, TAILS, true, FPT, MP>(p.sp, xin, sum, yy, ll, flag);
                else rqs_eval_lean<NB, TAILS, false, FPT, MP>(p.sp, xin, sum, yy, ll, flag);
                const bool issuer = warp == 4 && lane == 0;
                if (p.pair_only || p.tma_y) {
                    // Outputs leave through one of three staging buffers, one TMA store (pair: two) per group of YG column tiles.
                    // ONE barrier per group: the issuer waits, right after it has issued group k, until group k-1's stores have read
                    // their buffer; every thread that passes the barrier of group k+1 therefore knows the buffer of group k-1 ==
                    // the buffer of group k+2 is free.
                    constexpr int YG = Cfg::YG, YROW = Cfg::YROW, YG16 = Cfg::YG16, YROW16 = Cfg::YROW16;
                    const int grp = p.pair_only ? YG16 : YG;
                    uint8_t* buf = smem_gen + STEP_Y_OFF + ybuf * STEP_Y_BUF_BYTES;
                    if (p.pair_only) {
                        __half* sh = reinterpret_cast<__half*>(buf);
                        __half* sl = sh + BM * YROW16;
                        const int off = r_tile * YROW16 + (n % YG16) * TF + wg * FPT;
                        __half hi[FPT], lo[FPT];
#pragma unroll
                        for (int f = 0; f < FPT; ++f) {
                            int f2 = 0;
                            split_f16(yy[f], p.out_scale, hi[f], lo[f], f2);
                            if (row_ok && j0 + f < p.d_t) { lad_row += ll[f]; flag |= f2; }
                        }
                        if (FPT % 2 == 0) {          // two features per 32-bit store (2-byte stores: 4 bank-conflict passes each)
#pragma unroll
                            for (int f = 0; f < FPT; f += 2) {
                                *reinterpret_cast<__half2*>(sh + off + f) = __halves2half2(hi[f], hi[f + 1]);
                                *reinterpret_cast<__half2*>(sl + off + f) = __halves2half2(lo[f], lo[f + 1]);
                            }
                        } else {
#pragma unroll
                            for (int f = 0; f < FPT; ++f) { sh[off + f] = hi[f]; sl[off + f] = lo[f]; }
                        }
                    } else {
                        float* dst = reinterpret_cast<float*>(buf) + r_tile * YROW + (n % YG) * TF + wg * FPT;
#pragma unroll
                        for (int f = 0; f < FPT; ++f) {
                            dst[f] = yy[f];
                            if (row_ok && j0 + f < p.d_t) lad_row += ll[f];
                        }
                    }
                    if (n % grp == grp - 1 || n == p.num_n_tiles - 1) {
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        asm volatile("bar.sync 2, %0;" ::"n"(128 * EWG) : "memory");
                        if (issuer) {
                            const uint32_t src = smem_base + STEP_Y_OFF + ybuf * STEP_Y_BUF_BYTES;
                            if (p.pair_only) {
                                const int c0 = p.t_col0 + (n / YG16) * YROW16;
                                step_store_2d(&map_yh, src, c0, m * BM);
                                step_store_2d(&map_yl, src + BM * YROW16 * 2, c0, m * BM);
                            } else {
                                step_store_2d(&map_y, src, p.t_col0 + (n / YG) * YROW, m * BM);
                            }
                            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                            asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
                        }
                        if (++ybuf == 3) ybuf = 0;
                    }
                } else {
#pragma unroll
                    for (int f = 0; f < FPT; ++f) {
                        if (row_ok && j0 + f < p.d_t) {
                            const int cf = p.t_cols ? __ldg(p.t_cols + j0 + f) : p.t_col0 + j0 + f;
                            p.y[row * p.ldy + cf] = yy[f];
                            lad_row += ll[f];
                        }
                    }
                }
                __syncwarp();
            }
            // ---- finish the row block: lad_accum[row] += the warpgroups' partial sums, fixed order (the x staging is idle here)
            if (p.lad_accum) {
                if (wg > 0) s_lad[(wg - 1) * 128 + r_tile] = lad_row;
                asm volatile("bar.sync 1, %0;" ::"n"(128 * EWG) : "memory");
                if (wg == 0 && row_ok) {
                    float t = lad_row;
#pragma unroll
                    for (int h = 1; h < EWG; ++h) t += s_lad[(h - 1) * 128 + r_tile];
                    p.lad_accum[row] += t;
                }
                asm volatile("bar.sync 1, %0;" ::"n"(128 * EWG) : "memory");
            }
        }
        if (warp == 4 && lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // staging outlives its stores
        if (flag && p.flags) atomicOr(p.flags, flag);
    }

    tc_fence_before();
    if (CL > 1) cluster_sync_all(); else __syncthreads();   // no CTA exits while a peer may still signal its barriers
    if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// Four epilogue warpgroups where a column tile has at least four features, else two (only NB = 16 without tails).
template <int NB, bool TAILS>
static int launch_step(const NfkCouplingStep* d, StepParams& p, cudaStream_t st) {
    constexpr int EWG = StepCfg<NB, TAILS, 2>::TF >= 4 ? 4 : 2;
    using Cfg = StepCfg<NB, TAILS, EWG>;
    const int H = p.H;
    const int nch = H > 128 ? 2 : 1, ch = H / nch;
    // trunk-only launches run single CTAs: their TMA stores read R while a cluster peer could already multicast the next
    // tile's weights over it
    const int CL = (!p.trunk_only && p.num_m_tiles >= 2 && ch % 16 == 0 && (ch / 2) % 8 == 0) ? 2 : 1;
    const int L = p.num_layers - 1;
    CUtensorMap ma_hi, ma_lo, mw0_hi, mw0_lo, mwt_hi, mwt_lo, mwf_hi, mwf_lo;
    int rc;
    if ((rc = make_map(&ma_hi, (const __half*)d->a_hi, p.n_rows, p.K0, d->lda, BM))) return rc;
    if ((rc = make_map(&ma_lo, (const __half*)d->a_lo, p.n_rows, p.K0, d->lda, BM))) return rc;
    if ((rc = make_map(&mw0_hi, (const __half*)d->w0_hi, H, p.K0, d->ldw0, H / CL))) return rc;
    if ((rc = make_map(&mw0_lo, (const __half*)d->w0_lo, H, p.K0, d->ldw0, H / CL))) return rc;
    mwt_hi = mw0_hi; mwt_lo = mw0_lo;                          // placeholders when there is no square layer
    if (L > 0) {
        if ((rc = make_map(&mwt_hi, (const __half*)d->wt_hi, (int64_t)L * H, H, d->ldwt, ch / CL))) return rc;
        if ((rc = make_map(&mwt_lo, (const __half*)d->wt_lo, (int64_t)L * H, H, d->ldwt, ch / CL))) return rc;
    }
    mwf_hi = mw0_hi; mwf_lo = mw0_lo;
    CUtensorMap my = mw0_hi, myh = mw0_hi, myl = mw0_hi, mh_hi = mw0_hi, mh_lo = mw0_hi, mx = mw0_hi;
    if (p.trunk_only) {
        if ((rc = make_map(&mh_hi, (const __half*)d->h_hi, p.n_rows, H, d->ldh, BM))) return rc;
        if ((rc = make_map(&mh_lo, (const __half*)d->h_lo, p.n_rows, H, d->ldh, BM))) return rc;
    } else {
        const int packed_rows = p.d_t * Cfg::MP;
        if ((rc = make_map(&mwf_hi, (const __half*)d->wp_hi, packed_rows, H, d->ldwp, Cfg::BN / CL))) return rc;
        if ((rc = make_map(&mwf_lo, (const __half*)d->wp_lo, packed_rows, H, d->ldwp, Cfg::BN / CL))) return rc;
        p.num_n_tiles = (p.d_t + Cfg::TF - 1) / Cfg::TF;
        p.tma_y = (p.y && !p.t_cols && p.t_col0 % 4 == 0 && p.ldy % 4 == 0 && aligned16(p.y)) ? 1 : 0;
        // inputs as TMA boxes of TF columns: consecutive columns from a 16-byte aligned first column (tiles start at multiples of TF >= 4 floats...
        // TF = 2: 8-byte boxes are below the TMA minimum -> cp.async staging)
        p.tma_x = (!p.t_cols && Cfg::TF >= 4 && p.t_col0 % 4 == 0 && p.ldx % 4 == 0 && aligned16(p.x)) ? 1 : 0;
        if (p.tma_x && (rc = make_out_map(&mx, const_cast<float*>(p.x), p.n_rows, p.t_col0 + p.d_t, p.ldx, Cfg::TF, BM))) return rc;
        if (p.tma_y && (rc = make_out_map(&my, p.y, p.n_rows, p.t_col0 + p.d_t, p.ldy, Cfg::YROW, BM))) return rc;
        if (p.pair_only) {
            NFK_REQUIRE(!p.t_cols && p.t_col0 % 8 == 0 && d->lds % 8 == 0 && aligned16(d->y_hi) && aligned16(d->y_lo),
                        "pair output needs consecutive transformed columns starting at a multiple of 8 and 16-byte aligned rows");
            if ((rc = make_out_map16(&myh, (__half*)d->y_hi, p.n_rows, p.t_col0 + p.d_t, d->lds, Cfg::YROW16, BM))) return rc;
            if ((rc = make_out_map16(&myl, (__half*)d->y_lo, p.n_rows, p.t_col0 + p.d_t, d->lds, Cfg::YROW16, BM))) return rc;
        }
    }
    const int units = (p.num_m_tiles + CL - 1) / CL;
    const int max_clusters = sm_count() / CL;
    const int grid = CL * (units < max_clusters ? units : max_clusters);
    NFK_REQUIRE(d->workspace_bytes >= (size_t)grid * (size_t)H * 128 * 4, "workspace too small: %zu bytes given, %zu needed",
                d->workspace_bytes, (size_t)grid * (size_t)H * 128 * 4);
    auto kern1 = rq_coupling_step_kernel<NB, TAILS, 1, EWG>;
    auto kern2 = rq_coupling_step_kernel<NB, TAILS, 2, EWG>;
    cudaError_t e = cudaSuccess;
    static DeviceOnce attr_once;
    int attr_dev = 0;
    if (attr_once.pending(&attr_dev)) {
        e = cudaFuncSetAttribute(kern1, cudaFuncAttributeMaxDynamicSharedMemorySize, STEP_SMEM_BYTES);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(kern2, cudaFuncAttributeMaxDynamicSharedMemorySize, STEP_SMEM_BYTES);
        if (e != cudaSuccess) return fail(NFK_E_CUDA, "cudaFuncSetAttribute(smem=%d): %s", STEP_SMEM_BYTES, cudaGetErrorString(e));
        attr_once.mark(attr_dev);
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(128 + 128 * EWG);
    cfg.dynamicSmemBytes = STEP_SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CL; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    e = (CL == 2) ? cudaLaunchKernelEx(&cfg, kern2, ma_hi, ma_lo, mw0_hi, mw0_lo, mwt_hi, mwt_lo, mwf_hi, mwf_lo, my, myh, myl, mh_hi, mh_lo, mx, p)
                  : cudaLaunchKernelEx(&cfg, kern1, ma_hi, ma_lo, mw0_hi, mw0_lo, mwt_hi, mwt_lo, mwf_hi, mwf_lo, my, myh, myl, mh_hi, mh_lo, mx, p);
    if (e != cudaSuccess) return fail(NFK_E_CUDA, "cudaLaunchKernelEx(rq_coupling_step_kernel, cluster %d): %s", CL, cudaGetErrorString(e));
    return check_launch("rq_coupling_step_kernel");
}

}  // namespace tc
}  // namespace nfk

using namespace nfk;

extern "C" int nfk_rq_coupling_step_supported(int32_t num_bins, int32_t linear_tails, int32_t hidden_features, int32_t in_features,
                                              int32_t num_square_layers) {
    const bool bins_ok = (num_bins == 8 || num_bins == 10 || num_bins == 4 || num_bins == 16);
    return (bins_ok && hidden_features >= 32 && hidden_features <= tc::BN_MAX && hidden_features % 32 == 0 && in_features >= 8 &&
            in_features % 8 == 0 && num_square_layers >= 0 && num_square_layers < tc::STEP_MAX_LAYERS) ? 1 : 0;
}

extern "C" size_t nfk_rq_coupling_step_workspace_bytes(int32_t hidden_features) {
    return (size_t)tc::sm_count() * (size_t)hidden_features * 128 * 4;
}

extern "C" int nfk_rq_coupling_step_f16x3(const NfkCouplingStep* d, void* stream) {
    NFK_REQUIRE(d, "NULL descriptor");
    NFK_REQUIRE(d->n_rows >= 0 && d->hidden_features >= 1 && d->in_features >= 1, "bad sizes");
    if (d->n_rows == 0) return NFK_OK;
    const bool trunk_only = d->h_hi != nullptr;
    const int nb = trunk_only && !d->spline ? 8 : (d->spline ? d->spline->num_bins : 0);
    const int lt = trunk_only && !d->spline ? 1 : (d->spline ? d->spline->linear_tails : 0);
    NFK_REQUIRE(trunk_only || d->spline, "spline descriptor missing");
    NFK_REQUIRE(nfk_rq_coupling_step_supported(nb, lt, d->hidden_features, d->in_features, d->num_square_layers),
                "coupling-step kernel does not take num_bins=%d hidden=%d in_features=%d square layers=%d", nb, d->hidden_features,
                d->in_features, d->num_square_layers);
    NFK_REQUIRE(d->a_hi && d->a_lo && d->w0_hi && d->w0_lo && d->bias_trunk && d->layer_flags && d->workspace, "NULL pointer");
    NFK_REQUIRE(d->num_square_layers == 0 || (d->wt_hi && d->wt_lo && d->wt_exps), "square-layer weights missing");
    NFK_REQUIRE(d->lda % 8 == 0 && d->ldw0 % 8 == 0 && (d->num_square_layers == 0 || d->ldwt % 8 == 0), "row pitches must be multiples of 8");
    NFK_REQUIRE(aligned16(d->a_hi) && aligned16(d->a_lo) && aligned16(d->w0_hi) && aligned16(d->w0_lo) && aligned16(d->bias_trunk) &&
                    aligned16(d->workspace) && (d->num_square_layers == 0 || (aligned16(d->wt_hi) && aligned16(d->wt_lo))),
                "operands must be 16-byte aligned");
    NFK_REQUIRE(d->n_rows < (1ll << 31), "n_rows too large for one launch");
    tc::StepParams p;
    memset(&p, 0, sizeof(p));
    p.bias_trunk = d->bias_trunk; p.skip_buf = (float4*)d->workspace; p.H = d->hidden_features; p.K0 = d->in_features;
    p.num_layers = 1 + d->num_square_layers; p.act_scale = ldexpf(1.0f, d->act_exp); p.trunk_only = trunk_only ? 1 : 0;
    for (int l = 0; l < p.num_layers; ++l) {
        const int lf = d->layer_flags[l];
        const int e = l == 0 ? d->a_exp + d->w0_exp : d->act_exp + d->wt_exps[l - 1];
        NFK_REQUIRE(!((lf & tc::SL_ADD_SKIP) && (lf & tc::SL_RELU_OUT)), "layer %d: skip add after a relu output is not supported", l);
        NFK_REQUIRE(e >= -60 && e <= 60, "scale exponent out of range");
        p.layer_flags[l] = lf;
        p.acc_scale[l] = ldexpf(1.0f, e);
        p.inv_acc_scale[l] = ldexpf(1.0f, -e);
    }
    p.flags = d->flags; p.n_rows = d->n_rows;
    p.num_m_tiles = (int)((d->n_rows + tc::BM - 1) / tc::BM);
    cudaStream_t st = (cudaStream_t)stream;
    if (trunk_only) {
        NFK_REQUIRE(d->h_lo && d->ldh % 8 == 0 && aligned16(d->h_hi) && aligned16(d->h_lo), "bad trunk output pair");
        return tc::launch_step<8, true>(d, p, st);               // four epilogue warpgroups
    }
    int rc = make_spline_params(d->spline, &p.sp);
    if (rc) return rc;
    NFK_REQUIRE(d->wp_hi && d->wp_lo && d->bias_packed && d->x && d->d_t >= 1, "NULL pointer");
    NFK_REQUIRE((d->y != nullptr) != (d->y_hi != nullptr), "give either y (fp32 outputs) or y_hi / y_lo (their fp16 split pair)");
    NFK_REQUIRE((d->y_hi == nullptr) == (d->y_lo == nullptr) && d->y_exp >= -60 && d->y_exp <= 60, "bad pair output");
    NFK_REQUIRE(d->t_cols || d->t_col0 >= 0, "t_cols is NULL and t_col0 is negative");
    NFK_REQUIRE(aligned16(d->bias_packed) && aligned16(d->wp_hi) && aligned16(d->wp_lo) && d->ldwp % 8 == 0, "packed final layer must be 16-byte aligned");
    NFK_REQUIRE(d->act_exp + d->wp_exp >= -60 && d->act_exp + d->wp_exp <= 60, "scale exponent out of range");
    p.bias = d->bias_packed; p.x = d->x; p.y = d->y; p.t_cols = d->t_cols; p.t_col0 = d->t_col0; p.lad_accum = d->lad_accum;
    p.ldx = d->ldx; p.ldy = d->ldy; p.d_t = d->d_t; p.inverse = d->inverse;
    p.inv_acc_scale_f = ldexpf(1.0f, -(d->act_exp + d->wp_exp));
    p.pair_only = d->y_hi ? 1 : 0; p.out_scale = ldexpf(1.0f, d->y_exp);
    const bool tails = d->spline->linear_tails != 0;
    switch (d->spline->num_bins) {
        case 4: return tails ? tc::launch_step<4, true>(d, p, st) : tc::launch_step<4, false>(d, p, st);
        case 8: return tails ? tc::launch_step<8, true>(d, p, st) : tc::launch_step<8, false>(d, p, st);
        case 10: return tails ? tc::launch_step<10, true>(d, p, st) : tc::launch_step<10, false>(d, p, st);
        case 16: return tails ? tc::launch_step<16, true>(d, p, st) : tc::launch_step<16, false>(d, p, st);
    }
    return fail(NFK_E_UNSUPPORTED, "num_bins=%d has no coupling-step kernel instance", d->spline->num_bins);
}
