// ONE kernel for the dominant step of PiecewiseRationalQuadraticCouplingTransform (coupling.py:279-293, 549-582 +
// splines/rational_quadratic.py:13-181 in the reference): the final conditioner layer (hidden -> d_t * (3K-1)
// spline parameters, 86 % of the flow's FLOPs) on tcgen05 tensor cores, with the rational-quadratic spline, the scatter of
// the transformed features and the per-row log|det| evaluated by the epilogue warps straight from the accumulators.
// The [B, d_t*M] parameter tensor the reference materialises (37.8 GB per layer at B = 2^20) never exists.
//
// Same machinery as nfk_linear_tc.cu (TMA-fed fp16 split-pair operands, partial sums drained from TMEM into registers);
// what differs:
//   * the packed weight has MP = roundup(M, 8) rows per transformed feature (zero padded), so a tile of BN = 2*FPT*MP
//     columns holds whole features and each accumulate/epilogue thread ends a tile owning ALL parameters of FPT features
//     of its row in registers (K = 8 bins, linear tails: MP = 24, FPT = 5, BN = 240);
//   * a CTA walks the N-tiles of one 128-row block consecutively, so every thread keeps the running log|det| of its row
//     in a register and the row is finished (y written, lad_accum updated, deterministically) when the CTA moves on.
#include "fused_spline.cuh"

namespace nfk {
namespace tc {

struct FusedParams {
    const float* bias;      // [d_t * MP] packed like the weight rows, zero padded
    const float* x;         // coupling input [n_rows, ldx]
    float* y;               // coupling output [n_rows, ldy]; identity columns are written by the caller
    const int32_t* t_cols;  // [d_t] column of transformed feature j, or null: feature j lives in column t_col0 + j
    int t_col0;
    int tma_y;              // y goes out through staged TMA stores (consecutive columns, 16-byte aligned)
    int pair_only;          // write the fp16 split pair of the outputs (through map_yh / map_yl) INSTEAD of fp32 y
    float out_scale;        // 2^e of that pair
    float* lad_accum;       // [n_rows] running log|det| (read-modify-write) or null
    int32_t* flags;
    int64_t ldx, ldy, n_rows;
    int K;                  // hidden features (GEMM reduction length)
    int d_t;
    int num_m_tiles, num_n_tiles;
    int inverse;
    float acc_scale;        // 2^(e_a + e_w): the accumulators hold (A Wp^T) * acc_scale (fp16 pairs are power-of-two scaled)
    float inv_acc_scale;
    uint32_t zero;          // always 0 (mbar_arrive_after_loads)
    SplineParams sp;
};

// Epilogue warpgroups of the fused kernel.  Measured on B200, cfg 3 (ms per step spent in this kernel):
// EWG = 2 (5 features per thread, BN = 240, 40 N-tiles): 263;  EWG = 4 (2 features per thread, BN = 192, 49 N-tiles): 274 --
// the epilogue is not what the tensor pipe waits for, and narrower tiles re-stream the activations more often.
constexpr int EWG = 2;
constexpr int FUSED_THREADS = 128 + 128 * EWG;
// registers: the launch allocates floor(64K / threads) per thread; the control warpgroup shrinks to 40 and the epilogue
// warpgroups share what that frees (setmaxnreg needs multiples of 8)
constexpr int FUSED_LAUNCH_REGS = (65536 / FUSED_THREADS) / 8 * 8 > 255 ? 248 : (65536 / FUSED_THREADS) / 8 * 8;
constexpr int FUSED_EPI_REGS = ((FUSED_THREADS * FUSED_LAUNCH_REGS - 128 * 40) / (128 * EWG)) / 8 * 8;

template <int NB, bool TAILS>
struct FusedCfg {
    static constexpr int M = TAILS ? 3 * NB - 1 : 3 * NB + 1;   // parameters per feature
    static constexpr int MP = (M + 7) / 8 * 8;                  // padded
    static constexpr int FPT = BN_MAX / (EWG * MP);             // features per thread per tile
    static constexpr int HALF_COLS = FPT * MP;                  // columns per accumulate/epilogue thread
    static constexpr int TILE_FEATURES = EWG * FPT;
    static constexpr int TILE_COLS = EWG * HALF_COLS;           // packed weight rows per tile
    static constexpr int BN = (TILE_COLS + 15) / 16 * 16;       // MMA N (the pad columns compute the next feature's first rows, unused)
    // outputs leave through shared memory, YG column tiles at a time, so that a staged row (YG * TILE_FEATURES floats) is a
    // multiple of 16 bytes -- what a TMA store needs
    static constexpr int YG = TILE_FEATURES % 4 == 0 ? 1 : (TILE_FEATURES % 2 == 0 ? 2 : 4);
    static constexpr int YROW = YG * TILE_FEATURES;             // floats per staged row
    // pair-only output (fp16 hi / lo instead of fp32 y): groups of YG16 tiles make a staged row a multiple of 16 bytes
    static constexpr int YG16 = TILE_FEATURES % 8 == 0 ? 1 : (TILE_FEATURES % 4 == 0 ? 2 : (TILE_FEATURES % 2 == 0 ? 4 : 8));
    static constexpr int YROW16 = YG16 * TILE_FEATURES;         // halfs per staged row
    static_assert(2 * YROW16 * 2 <= 2 * YROW * 4, "pair staging must fit the y staging area");
    static_assert(FPT >= 1 && BN <= BN_MAX, "unsupported bin count for the fused kernel");
};

// Clusters of two CTAs on neighbouring 128-row blocks walk the same weight tiles in lockstep; each loads HALF of every weight
// slab and multicasts it into both CTAs' shared memory (halves the L2 -> SM weight stream; ncu: L2->SM 8.2 TB/s at 40 %
// tensor-pipe activity with one CTA per row block, 57 % with the cluster).  A trailing odd row block is paired with an
// out-of-range one (all-zero A, no stores).
template <int NB, bool TAILS>
__global__ void __launch_bounds__(FUSED_THREADS, 1)
rq_coupling_final_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                         const __grid_constant__ CUtensorMap map_w_hi, const __grid_constant__ CUtensorMap map_w_lo,
                         const __grid_constant__ CUtensorMap map_y, const __grid_constant__ CUtensorMap map_yh,
                         const __grid_constant__ CUtensorMap map_yl, const FusedParams p) {
    using Cfg = FusedCfg<NB, TAILS>;
    constexpr int MP = Cfg::MP, FPT = Cfg::FPT, HC = Cfg::HALF_COLS, BN = Cfg::BN, TILE = Cfg::TILE_COLS;
    constexpr int CL = 2;                                            // CTAs per cluster

    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
    const uint32_t bars = smem_base + STAGES * STAGE_BYTES;
    const uint32_t bar_full = bars, bar_empty = bars + 8 * STAGES;
    const uint32_t bar_tfull = bars + 16 * STAGES, bar_tempty = bars + 16 * STAGES + 16;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem_gen + STAGES * STAGE_BYTES + 16 * STAGES + 32);   // then bias barriers at +48, +64
    float* s_lad = reinterpret_cast<float*>(smem_gen + STAGES * STAGE_BYTES + 256);       // [EWG-1][128] partial log|det|
    // the packed bias of the current / next column tile, staged by the producer with a bulk copy so the epilogue reads it
    // with ~30-cycle shared loads (ncu, r1: bias + x + column-index loads at the top of every tile, L2 latency each, were
    // 40 % of the epilogue warps' samples)
    float* s_bias = reinterpret_cast<float*>(smem_gen + STAGES * STAGE_BYTES + 256 + 512 * EWG);   // [2][BN_MAX]
    const uint32_t bar_bfull = bars + 16 * STAGES + 48, bar_bempty = bars + 16 * STAGES + 64;
    // transformed outputs of YG consecutive column tiles, [2 buffers][128 rows][YROW] fp32, sent out by one TMA store per
    // group: a row-per-thread st.global of 5 floats per tile touched 32 sectors per instruction with 4 useful bytes each
    constexpr int YG = Cfg::YG, YROW = Cfg::YROW;
    constexpr int Y_OFF = STAGES * STAGE_BYTES + 256 + 512 * EWG + 2 * BN_MAX * 4;
    float* s_y = reinterpret_cast<float*>(smem_gen + Y_OFF);

    uint32_t tid_x;
    asm volatile("mov.u32 %0, %%tid.x;" : "=r"(tid_x));      // volatile: not re-read (S2R) inside the tile loop
    const int warp = tid_x >> 5, lane = tid_x & 31;
    const int num_k = (p.K + BK - 1) / BK;
    const int num_groups = (num_k + DRAIN_SLABS_FUSED - 1) / DRAIN_SLABS_FUSED;     // partial sums per tile

    if (tid_x == 0) {
        for (int b = 0; b < 2; ++b) { mbar_init(bar_bfull + 8 * b, 1); mbar_init(bar_bempty + 8 * b, 4 * EWG); }
        // both CTAs' MMA threads release a slot (the peer multicasts into it)
        for (int s = 0; s < STAGES; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, CL); }
        for (int a = 0; a < 2; ++a) { mbar_init(bar_tfull + 8 * a, 1); mbar_init(bar_tempty + 8 * a, 4 * EWG); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        prefetch_tmap(&map_a_hi); prefetch_tmap(&map_a_lo); prefetch_tmap(&map_w_hi); prefetch_tmap(&map_w_lo);
    }
    if (warp == 1) tmem_alloc(smem_u32(tmem_slot), 512);
    tc_fence_before();
    cluster_sync_all();                                      // peers' barriers are initialised before anyone signals them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int cta_rank = (int)cluster_ctarank();
    const int first_block = blockIdx.x / CL, block_step = gridDim.x / CL;    // a "block" = CL neighbouring 128-row tiles
    const int num_blocks = (p.num_m_tiles + CL - 1) / CL;
    constexpr uint16_t cl_mask = (uint16_t)((1u << CL) - 1);

    if (warp < 4) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 40;" ::: "memory");
        if (warp == 0) {
            // ================================================= TMA producer (one elected thread: uniform datapath, tc_common.cuh)
            if (elect_one()) {
                // bytes counted on the slab's barrier: everything landing in THIS CTA's slab
                constexpr uint32_t tx_bytes = 2u * A_BYTES + 2u * (uint32_t)BN * ROW_BYTES;
                constexpr int WROWS = BN / CL;                                             // weight rows this CTA fetches
                int stage = 0; uint32_t phase = 0;
                int bslot = 0; uint32_t bphase = 0;
                for (int mb = first_block; mb < num_blocks; mb += block_step) {
                    const int m = mb * CL + cta_rank;
                    for (int n = 0; n < p.num_n_tiles; ++n) {
                        {   // this tile's slice of the packed bias -> s_bias[bslot]
                            const int cols = min(TILE, p.d_t * MP - n * TILE);
                            mbar_wait(bar_bempty + 8 * bslot, bphase ^ 1);
                            mbar_expect_tx(bar_bfull + 8 * bslot, (uint32_t)cols * 4u);
                            bulk_load_1d(smem_u32(s_bias + bslot * BN_MAX), p.bias + (int64_t)n * TILE, (uint32_t)cols * 4u,
                                         bar_bfull + 8 * bslot);
                            if (++bslot == 2) { bslot = 0; bphase ^= 1; }
                        }
                        for (int ks = 0; ks < num_k; ++ks) {
                            mbar_wait(bar_empty + 8 * stage, phase ^ 1);      // every CTA of the cluster has released the slot
                            const uint32_t full = bar_full + 8 * stage;
                            const uint32_t sa = smem_base + stage * STAGE_BYTES;   // [A hi | A lo | W hi | W lo]
                            mbar_expect_tx(full, tx_bytes);
                            tma_load_2d(sa, &map_a_hi, full, ks * BK, m * BM);
                            tma_load_2d(sa + A_BYTES, &map_a_lo, full, ks * BK, m * BM);
                            const uint32_t off = (uint32_t)cta_rank * WROWS * ROW_BYTES;
                            tma_load_2d_multicast(sa + 2 * A_BYTES + off, &map_w_hi, full, ks * BK, n * TILE + cta_rank * WROWS, cl_mask);
                            tma_load_2d_multicast(sa + 2 * A_BYTES + B_BYTES + off, &map_w_lo, full, ks * BK,
                                                  n * TILE + cta_rank * WROWS, cl_mask);
                            if (++stage == STAGES) { stage = 0; phase ^= 1; }
                        }
                    }
                }
            }
        } else if (warp == 1) {
            // ================================================= MMA issuer: one partial sum per DRAIN_SLABS_FUSED slabs
            if (elect_one()) {                       // one elected thread runs the role (uniform datapath, tc_common.cuh: elect_one)
                const uint32_t idesc = make_idesc(BN);
                int stage = 0; uint32_t phase = 0;
                int acc = 0; uint32_t acc_phase = 0;
                for (int mb = first_block; mb < num_blocks; mb += block_step) {
                    for (int n = 0; n < p.num_n_tiles; ++n) {
                        for (int g = 0; g < num_groups; ++g) {
                            // one partial sum = DRAIN_SLABS_FUSED resident K-slabs; every small cross term (lo*hi, hi*lo) is
                            // issued before the first main product, so only the main MMAs round at full magnitude
                            const int slabs = min(DRAIN_SLABS_FUSED, num_k - g * DRAIN_SLABS_FUSED);
                            mbar_wait(bar_tempty + 8 * acc, acc_phase ^ 1);
                            const uint32_t d_tmem = tmem_base + acc * BN_MAX;
                            for (int j0 = 0; j0 < slabs; j0 += 2) {           // pairs of resident slabs: cross terms of both, then mains
                                const int pair = min(2, slabs - j0);
                                int st = stage; uint32_t ph = phase;
                                for (int j = 0; j < pair; ++j) {
                                    mbar_wait(bar_full + 8 * st, ph);
                                    if (++st == STAGES) { st = 0; ph ^= 1; }
                                }
                                tc_fence_after();
                                st = stage;
                                for (int j = 0; j < pair; ++j) {
                                    const uint32_t sa = smem_base + st * STAGE_BYTES;
                                    const uint64_t a_hi = make_smem_desc(sa), a_lo = make_smem_desc(sa + A_BYTES);
                                    const uint64_t w_hi = make_smem_desc(sa + 2 * A_BYTES), w_lo = make_smem_desc(sa + 2 * A_BYTES + B_BYTES);
#pragma unroll
                                    for (int kk = 0; kk < BK / 16; ++kk) {
                                        const uint64_t adv = (uint64_t)(kk * 2);
                                        umma_f16(d_tmem, a_lo + adv, w_hi + adv, idesc, (j0 | j | kk) != 0);
                                        umma_f16(d_tmem, a_hi + adv, w_lo + adv, idesc, 1);
                                    }
                                    if (++st == STAGES) st = 0;
                                }
                                for (int j = 0; j < pair; ++j) {
                                    const uint32_t sa = smem_base + stage * STAGE_BYTES;
                                    const uint64_t a_hi = make_smem_desc(sa), w_hi = make_smem_desc(sa + 2 * A_BYTES);
#pragma unroll
                                    for (int kk = 0; kk < BK / 16; ++kk) {
                                        const uint64_t adv = (uint64_t)(kk * 2);
                                        umma_f16(d_tmem, a_hi + adv, w_hi + adv, idesc, 1);
                                    }
                                    umma_commit_multicast(bar_empty + 8 * stage, cl_mask);   // releases the slot in every CTA
                                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                                }
                            }
                            umma_commit(bar_tfull + 8 * acc);
                            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                        }
                    }
                }
            }
        }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(FUSED_EPI_REGS) : "memory");
        // ================================================= accumulate + spline epilogue: 4 * EWG warps
        const int q = warp & 3;                   // TMEM lane quarter
        const int half = (warp - 4) >> 2;         // warpgroup: which FPT features of the tile
        int acc = 0; uint32_t acc_phase = 0;
        int flag = 0;
        int bslot = 0; uint32_t bphase = 0;
        int ybuf = 0;
        for (int mb = first_block; mb < num_blocks; mb += block_step) {
            const int m = mb * CL + cta_rank;
            const int64_t row = (int64_t)m * BM + q * 32 + lane;
            const bool row_ok = row < p.n_rows;
            float lad_row = 0.0f;
            // input values and columns of the FPT features this thread owns in a tile; loaded one tile ahead so their latency
            // hides under the spline of the tile before (y may alias x: the columns of different tiles are disjoint and every
            // element is read, then written, by this thread only)
            float xin[FPT], xin_next[FPT];
            int col[FPT], col_next[FPT];
            auto load_x = [&](int n, float (&xv)[FPT], int (&cv)[FPT]) {
                const int jn = (n * EWG + half) * FPT;
#pragma unroll
                for (int f = 0; f < FPT; ++f) {
                    const bool ok = row_ok && (jn + f < p.d_t);
                    cv[f] = !ok ? 0 : (p.t_cols ? __ldg(p.t_cols + jn + f) : p.t_col0 + jn + f);
                    xv[f] = ok ? p.x[row * p.ldx + cv[f]] : 0.0f;
                }
            };
            load_x(0, xin, col);
            for (int n = 0; n < p.num_n_tiles; ++n) {
                const int j0 = (n * EWG + half) * FPT;                     // first feature this thread owns in this tile
                float sum[HC];
#pragma unroll
                for (int c = 0; c < HC; ++c) sum[c] = 0.0f;
                for (int ks = 0; ks < num_groups; ++ks) {
                    mbar_wait(bar_tfull + 8 * acc, acc_phase);
                    tc_fence_after();
                    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * BN_MAX + half * HC;
                    constexpr int LDB = HC <= 48 ? 3 : 5;           // TMEM loads in flight per wait (register budget)
#pragma unroll
                    for (int c = 0; c < HC; c += 8 * LDB) {
                        uint32_t raw[LDB][8];
#pragma unroll
                        for (int u = 0; u < LDB; ++u)
                            if (c + 8 * u < HC) tmem_ld8(taddr + c + 8 * u, raw[u]);
                        tmem_ld_wait();
#pragma unroll
                        for (int u = 0; u < LDB; ++u)
                            if (c + 8 * u < HC) {
#pragma unroll
                                for (int i = 0; i < 8; i += 2) {       // packed fp32x2 round-to-nearest adds (FADD2)
                                    const float2 r2 = __fadd2_rn(make_float2(sum[c + 8 * u + i], sum[c + 8 * u + i + 1]),
                                                                 make_float2(__uint_as_float(raw[u][i]), __uint_as_float(raw[u][i + 1])));
                                    sum[c + 8 * u + i] = r2.x;
                                    sum[c + 8 * u + i + 1] = r2.y;
                                }
                            }
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_tempty + 8 * acc);
                    if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                }
                if (n + 1 < p.num_n_tiles) load_x(n + 1, xin_next, col_next);
                // ---- back from the accumulators' power-of-two scaled domain, plus the packed bias staged in shared memory
                {
                    mbar_wait(bar_bfull + 8 * bslot, bphase);
                    const float4* bias4 = reinterpret_cast<const float4*>(s_bias + bslot * BN_MAX + half * HC);
#pragma unroll
                    for (int c = 0; c < HC; c += 4) {
                        const float4 b4 = (j0 + c / MP < p.d_t) ? bias4[c >> 2] : make_float4(0.f, 0.f, 0.f, 0.f);
                        sum[c] = fmaf(sum[c], p.inv_acc_scale, b4.x); sum[c + 1] = fmaf(sum[c + 1], p.inv_acc_scale, b4.y);
                        sum[c + 2] = fmaf(sum[c + 2], p.inv_acc_scale, b4.z); sum[c + 3] = fmaf(sum[c + 3], p.inv_acc_scale, b4.w);
                    }
                    uint32_t bits = 0;                    // one component of every LDS.128 (mbar_arrive_after_loads)
#pragma unroll
                    for (int c = 0; c < HC; c += 4) bits |= __float_as_uint(sum[c]);
                    __syncwarp();
                    if (lane == 0) mbar_arrive_after_loads(bar_bempty + 8 * bslot, bits, p.zero);
                    if (++bslot == 2) { bslot = 0; bphase ^= 1; }
                }
                // ---- spline on the FPT features held in registers, all features advanced together (ILP = FPT)
                {
                    float yy[FPT], ll[FPT];
                    if (p.inverse) rqs_eval_lean<NB, TAILS, true, FPT, MP>(p.sp, xin, sum, yy, ll, flag);
                    else rqs_eval_lean<NB, TAILS, false, FPT, MP>(p.sp, xin, sum, yy, ll, flag);
                    if (p.pair_only) {
                        // the consumer of this coupling's output is a tensor-core layer: it reads the fp16 split pair, so that
                        // is all that is written (no fp32 y, no separate split pass).  One staging area (hi rows, then lo
                        // rows), reused per group of YG16 tiles: the issuer makes sure the previous group's stores have
                        // read it before the first write of a group.
                        constexpr int YG16 = Cfg::YG16, YROW16 = Cfg::YROW16;
                        const bool issuer = warp == 4 && lane == 0;
                        if (n % YG16 == 0) {
                            if (issuer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                            asm volatile("bar.sync 2, %0;" ::"n"(128 * EWG) : "memory");
                        }
                        __half* sh = reinterpret_cast<__half*>(s_y);
                        __half* sl = sh + BM * YROW16;
                        const int off = (q * 32 + lane) * YROW16 + (n % YG16) * Cfg::TILE_FEATURES + half * FPT;
#pragma unroll
                        for (int f = 0; f < FPT; ++f) {
                            __half hi, lo;
                            int f2 = 0;
                            split_f16(yy[f], p.out_scale, hi, lo, f2);
                            sh[off + f] = hi;
                            sl[off + f] = lo;
                            if (row_ok && j0 + f < p.d_t) { lad_row += ll[f]; flag |= f2; }
                        }
                        if (n % YG16 == YG16 - 1 || n == p.num_n_tiles - 1) {
                            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                            asm volatile("bar.sync 2, %0;" ::"n"(128 * EWG) : "memory");
                            if (issuer) {
                                const int c0 = p.t_col0 + (n / YG16) * YROW16;
                                asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                                                 reinterpret_cast<uint64_t>(&map_yh)),
                                             "r"(smem_base + Y_OFF), "r"(c0), "r"(m * BM)
                                             : "memory");
                                asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                                                 reinterpret_cast<uint64_t>(&map_yl)),
                                             "r"(smem_base + Y_OFF + BM * YROW16 * 2), "r"(c0), "r"(m * BM)
                                             : "memory");
                                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                            }
                        }
                    } else if (p.tma_y) {
                        float* dst = s_y + ((size_t)ybuf * BM + q * 32 + lane) * YROW + (n % YG) * Cfg::TILE_FEATURES + half * FPT;
#pragma unroll
                        for (int f = 0; f < FPT; ++f) {
                            dst[f] = yy[f];
                            if (row_ok && j0 + f < p.d_t) lad_row += ll[f];
                        }
                        if (n % YG == YG - 1 || n == p.num_n_tiles - 1) {
                            const bool issuer = warp == 4 && lane == 0;
                            if (issuer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the other buffer is free again
                            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                            asm volatile("bar.sync 2, %0;" ::"n"(128 * EWG) : "memory");
                            if (issuer) {
                                asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                                                 reinterpret_cast<uint64_t>(&map_y)),
                                             "r"(smem_base + Y_OFF + ybuf * BM * YROW * 4), "r"(p.t_col0 + (n / YG) * YROW), "r"(m * BM)
                                             : "memory");
                                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                            }
                            ybuf ^= 1;
                        }
                    } else {
#pragma unroll
                        for (int f = 0; f < FPT; ++f) {
                            if (row_ok && j0 + f < p.d_t) {
                                p.y[row * p.ldy + col[f]] = yy[f];
                                lad_row += ll[f];
                            }
                        }
                    }
                }
#pragma unroll
                for (int f = 0; f < FPT; ++f) { xin[f] = xin_next[f]; col[f] = col_next[f]; }
                __syncwarp();
            }
            // ---- finish the row block: lad_accum[row] += the warpgroups' partial sums, fixed order
            if (p.lad_accum) {
                if (half > 0) s_lad[(half - 1) * 128 + q * 32 + lane] = lad_row;
                asm volatile("bar.sync 1, %0;" ::"n"(128 * EWG) : "memory");
                if (half == 0 && row_ok) {
                    float t = lad_row;
#pragma unroll
                    for (int h = 1; h < EWG; ++h) t += s_lad[(h - 1) * 128 + q * 32 + lane];
                    p.lad_accum[row] += t;
                }
                asm volatile("bar.sync 1, %0;" ::"n"(128 * EWG) : "memory");
            }
        }
        if (warp == 4 && lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // staging outlives its stores
        if (flag && p.flags) atomicOr(p.flags, flag);
    }

    tc_fence_before();
    cluster_sync_all();                                      // no CTA exits while a peer may still signal its barriers
    if (warp == 1) tmem_dealloc(tmem_base, 512);
}

template <int NB, bool TAILS>
static int launch_fused(const CUtensorMap& ma_hi, const CUtensorMap& ma_lo, const __half* w_hi, const __half* w_lo, int64_t ldw,
                        FusedParams& p, cudaStream_t st, __half* pair_hi, __half* pair_lo, int64_t pair_lds) {
    using Cfg = FusedCfg<NB, TAILS>;
    constexpr int CL = 2;
    const int packed_rows = p.d_t * Cfg::MP;
    CUtensorMap mw_hi, mw_lo;
    int rc;
    if ((rc = make_map(&mw_hi, w_hi, packed_rows, p.K, ldw, Cfg::BN / CL))) return rc;
    if ((rc = make_map(&mw_lo, w_lo, packed_rows, p.K, ldw, Cfg::BN / CL))) return rc;
    p.num_n_tiles = (p.d_t + Cfg::TILE_FEATURES - 1) / Cfg::TILE_FEATURES;
    constexpr int smem = SMEM_BYTES + 512 * EWG + 2 * BN_MAX * 4 + 2 * BM * Cfg::YROW * 4;
    static_assert(smem <= 232448, "fused kernel shared memory");
    // y through staged TMA stores: consecutive transformed columns and 16-byte aligned rows / first column
    CUtensorMap my = mw_hi;
    p.tma_y = (p.y && !p.t_cols && p.t_col0 % 4 == 0 && p.ldy % 4 == 0 && aligned16(p.y)) ? 1 : 0;
    if (p.tma_y && (rc = make_out_map(&my, p.y, p.n_rows, p.t_col0 + p.d_t, p.ldy, Cfg::YROW, BM))) return rc;
    CUtensorMap myh = mw_hi, myl = mw_hi;
    if (p.pair_only) {
        NFK_REQUIRE(!p.t_cols && p.t_col0 % 8 == 0 && pair_lds % 8 == 0 && aligned16(pair_hi) && aligned16(pair_lo),
                    "pair-only output needs consecutive transformed columns starting at a multiple of 8 and 16-byte aligned rows");
        if ((rc = make_out_map16(&myh, pair_hi, p.n_rows, p.t_col0 + p.d_t, pair_lds, Cfg::YROW16, BM))) return rc;
        if ((rc = make_out_map16(&myl, pair_lo, p.n_rows, p.t_col0 + p.d_t, pair_lds, Cfg::YROW16, BM))) return rc;
    }
    static DeviceOnce attr_once;
    int attr_dev = 0;
    if (attr_once.pending(&attr_dev)) {
        cudaError_t e = cudaFuncSetAttribute(rq_coupling_final_kernel<NB, TAILS>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return fail(NFK_E_CUDA, "cudaFuncSetAttribute(smem=%d): %s", smem, cudaGetErrorString(e));
        attr_once.mark(attr_dev);
    }
    const int blocks = (p.num_m_tiles + CL - 1) / CL;
    const int max_clusters = sm_count() / CL;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(CL * (blocks < max_clusters ? blocks : max_clusters)));
    cfg.blockDim = dim3(FUSED_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CL; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, rq_coupling_final_kernel<NB, TAILS>, ma_hi, ma_lo, mw_hi, mw_lo, my, myh, myl, p);
    if (e != cudaSuccess) return fail(NFK_E_CUDA, "cudaLaunchKernelEx(rq_coupling_final_kernel, cluster %d): %s", CL, cudaGetErrorString(e));
    return check_launch("rq_coupling_final_kernel");
}

}  // namespace tc
}  // namespace nfk

using namespace nfk;

extern "C" int nfk_rq_coupling_final_supported(int32_t num_bins, int32_t linear_tails, int32_t hidden_features, int64_t lda) {
    const bool bins_ok = (num_bins == 8 || num_bins == 10 || num_bins == 4 || num_bins == 16);
    return (bins_ok && hidden_features >= 8 && hidden_features % 8 == 0 && lda % 8 == 0) ? 1 : 0;
}

extern "C" int32_t nfk_rq_coupling_final_padded_params(int32_t num_bins, int32_t linear_tails) {
    const int m = linear_tails ? 3 * num_bins - 1 : 3 * num_bins + 1;
    return (m + 7) / 8 * 8;
}

extern "C" int nfk_rq_coupling_final_f16x3(const NfkSplineDesc* desc, int inverse, const void* a_hi_, const void* a_lo_,
                                          int64_t lda, int32_t a_exp, const void* wp_hi_, const void* wp_lo_, int64_t ldw,
                                          int32_t w_exp, const float* bias_packed, int32_t hidden_features, const float* x,
                                          int64_t ldx, const int32_t* t_cols, int32_t t_col0, int32_t d_t, float* y,
                                          int64_t ldy, void* y_hi, void* y_lo, int64_t lds, int32_t y_exp, float* lad_accum,
                                          int64_t n_rows, int32_t* flags, void* stream) {
    const __half* a_hi = (const __half*)a_hi_; const __half* a_lo = (const __half*)a_lo_;
    const __half* wp_hi = (const __half*)wp_hi_; const __half* wp_lo = (const __half*)wp_lo_;
    tc::FusedParams p;
    p.zero = 0;
    int rc = make_spline_params(desc, &p.sp);
    if (rc) return rc;
    NFK_REQUIRE(n_rows >= 0 && d_t >= 1 && hidden_features >= 1, "bad sizes");
    if (n_rows == 0) return NFK_OK;
    NFK_REQUIRE(a_hi && a_lo && wp_hi && wp_lo && bias_packed && x, "NULL pointer");
    NFK_REQUIRE((y != nullptr) != (y_hi != nullptr), "give either y (fp32 outputs) or y_hi / y_lo (their fp16 split pair)");
    NFK_REQUIRE((y_hi == nullptr) == (y_lo == nullptr) && y_exp >= -60 && y_exp <= 60, "bad pair output");
    NFK_REQUIRE(t_cols || t_col0 >= 0, "t_cols is NULL and t_col0 is negative");
    NFK_REQUIRE(aligned16(bias_packed), "bias_packed must be 16-byte aligned");
    NFK_REQUIRE(nfk_rq_coupling_final_supported(desc->num_bins, desc->linear_tails, hidden_features, lda) && ldw % 8 == 0,
                "fused coupling kernel does not take num_bins=%d hidden=%d", desc->num_bins, hidden_features);
    NFK_REQUIRE(aligned16(a_hi) && aligned16(a_lo) && aligned16(wp_hi) && aligned16(wp_lo), "operands must be 16-byte aligned");
    NFK_REQUIRE(n_rows < (1ll << 31), "n_rows too large for one launch");
    NFK_REQUIRE(a_exp + w_exp >= -60 && a_exp + w_exp <= 60, "scale exponent out of range");
    p.bias = bias_packed; p.x = x; p.y = y; p.t_cols = t_cols; p.t_col0 = t_col0; p.lad_accum = lad_accum; p.flags = flags;
    p.ldx = ldx; p.ldy = ldy; p.n_rows = n_rows; p.K = hidden_features; p.d_t = d_t; p.inverse = inverse;
    p.acc_scale = ldexpf(1.0f, a_exp + w_exp); p.inv_acc_scale = ldexpf(1.0f, -(a_exp + w_exp));
    p.pair_only = y_hi ? 1 : 0; p.out_scale = ldexpf(1.0f, y_exp);
    p.num_m_tiles = (int)((n_rows + tc::BM - 1) / tc::BM);
    CUtensorMap ma_hi, ma_lo;
    if ((rc = tc::make_map(&ma_hi, a_hi, n_rows, hidden_features, lda, tc::BM))) return rc;
    if ((rc = tc::make_map(&ma_lo, a_lo, n_rows, hidden_features, lda, tc::BM))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const bool tails = desc->linear_tails != 0;
#define NFK_FUSED(NB)                                                                                       \
    return tails ? tc::launch_fused<NB, true>(ma_hi, ma_lo, wp_hi, wp_lo, ldw, p, st, (__half*)y_hi, (__half*)y_lo, lds)   \
                 : tc::launch_fused<NB, false>(ma_hi, ma_lo, wp_hi, wp_lo, ldw, p, st, (__half*)y_hi, (__half*)y_lo, lds)
    switch (desc->num_bins) {
        case 4: NFK_FUSED(4);
        case 8: NFK_FUSED(8);
        case 10: NFK_FUSED(10);
        case 16: NFK_FUSED(16);
    }
#undef NFK_FUSED
    return fail(NFK_E_UNSUPPORTED, "num_bins=%d has no fused kernel instance", desc->num_bins);
}
