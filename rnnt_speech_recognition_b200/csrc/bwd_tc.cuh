// bwd_tc.cuh -- the two backward contractions of the joint (SURVEY 8 a19: TF autograd through model.py:162-166,
// triggered at run_rnnt.py:284) as hand-written tcgen05 kernels.  They consume what the forward KEPT: the bf16 softmax
// numerators E[row, v] = 2^(y_v - ref_row) (one reference per lattice row) -- the logit gradient of a row is
//     dl[row, :] = rs_row * E'[row, :],     rs_row = g_b * 2^(ref_row + (alpha + beta - ll - lse) * log2 e)
// where E' is E with the row's two special columns (blank, label) replaced by (final value) / rs_row (row_scale_kernel,
// two 2-byte writes per row).  A scale per ROW commutes with both GEMMs, so neither needs a per-element prologue:
//
//   bwd_dz_kernel   dZ[rows,H] = rs_row * (E'[rows,V] . W^T): both operands straight from TMA (K-major), the row scale,
//                   (1 - tanh^2(enc+pred)) and the tile's sums over u (-> d_enc, accumulated in REGISTERS along a run of
//                   tiles and stored once) and over t (-> one fp32 partial plane of d_pred per t-block) in the epilogue.
//                   Neither dl nor dZ ever exists in HBM.
//   bwd_dw_kernel   dW[H,V] (+)= (rs_row * z)^T . E'  as a split-K GEMM over the lattice rows: the A operand is REGENERATED
//                   from enc/pred by producer warps (tanh, times the row scale, K-major SWIZZLE_128B tiles), the B operand
//                   is E' loaded MN-major by TMA; db = sum_rows dl is one more row of the product (an A block whose row 0
//                   holds the row scales).  Partial tiles go to fp32 planes (deterministic), summed by sum_planes_kernel.
//
// All operands bf16 (E' needs the exponent range: it is relative to a reference that may lie far below the row maximum),
// fp32 accumulation.  Tile geometry: 16 x 8 lattice tiles (TT = 16 time steps, UU = 8 label positions), row r = tl*8 + ul of
// a tile is TMEM lane r; rows of tile `tile` live at row block slot[tile] of the kept arrays.
//
// What round 2 measured on the way here (profiles/r02/README.md): a first version scaled the numerators per 32-column
// group inside shared-memory prologues (fp16 -> fp32 -> bf16, later four HMUL2 per 16 bytes); the role wait counters
// (RNNTB200_PROF) showed both MMA warps waiting on those prologue warps 60-85 % of the time (dW 15 -> 5.5 ms, dZ 4.6 -> 4.1 ms
// after three rounds of tuning) -- the per-row reference removed the prologues altogether.
#pragma once
#include "joint_tc.cuh"

namespace rb {

constexpr int BW_TT = 16, BW_UU = 8;
#ifndef RNNTB200_DZ_EG
#define RNNTB200_DZ_EG 4
#endif
constexpr int DZ_EG = RNNTB200_DZ_EG;                 // epilogue warp groups (one warp per TMEM lane quarter each): chunk c belongs to group c % DZ_EG
constexpr int DZ_EPI_WARPS = 4 * DZ_EG;
constexpr int DZ_MAXJ = (12 + DZ_EG - 1) / DZ_EG;     // 32-column chunks per warp and unit (NCZ <= 384)
constexpr int DZ_TMA2_WARP = 2 + DZ_EPI_WARPS;        // enc / pred TMA for the epilogue
constexpr int DZ_THREADS = 32 * (3 + DZ_EPI_WARPS);   // warp 0 operand TMA | 1 MMA | 2.. epilogue | last: enc/pred TMA for the epilogue
constexpr int DZ_MAX_STAGES = 6;
constexpr int DW_THREADS = 576;      // warp 0 TMA | 1 MMA | 2-17 z producers, then epilogue (16 warps: the tanh chain is latency-bound at 2 warps per scheduler)
constexpr int DW_STAGES = 3;
constexpr int DW_NV = 256;           // vocabulary columns per dW output tile
constexpr int DW_NRS = 8;            // depth of the row-scale ring (K steps): the A producers run ahead of the B loads

struct BwdParams {
    const float* enc; const float* pred;
    const int* xlen; const int* ylen;
    int maxT, maxU, H, V;       // H, V: the padded Hp, Vp (enc / pred / d_enc rows are Hp wide, the kept rows Vp)
    int nTb, nUb, b0, nb;
    const int* slot;            // tile -> row block of the kept arrays (-1: tile outside the valid lattice)
    const int* tile_of_slot;    // inverse map (valid tiles only)
    const int4* slot_meta;      // per compact slot {first enc row, first pred row, #t rows, #u rows} of the tile
    const int* count;           // number of valid tiles (device word)
    const float* rowscale;      // per row of the kept arrays: rs_row (0 for rows outside the lattice)   [row_scale_kernel]
    // ---- dZ kernel
    int NP, NCZ, priv, sh, odd_base;   // passes over H, columns per pass, private / shared accumulator columns
    int dz_stages;                     // operand ring depth
    float* d_enc;               // (B, maxT, H), rows of this launch's utterances are fully written
    float* ppred;               // (nTb, nb, maxU, H) partial planes of d_pred
    // ---- dW kernel
    int nVT, nItems, nHB, S, Hrows;    // v-tiles, h-items per v-tile, 128-row blocks of H, K splits, rows per plane
    float* dWp;                 // (S, Hrows, V) partial planes of dW (zeroed by the host, accumulated over utterance chunks)
    float* dbp;                 // (S, V) partial planes of db
    long long* prof;            // optional (RNNTB200_PROF=1): per-CTA cycle counters of the roles' waits
};

// cycle accounting for bring-up (p.prof != NULL): t += clock64() spent in the bracketed region, by one lane of one warp per role
#define RB_PROF_BEGIN(flag) const long long _t0 = (flag) ? clock64() : 0
#define RB_PROF_END(flag, acc) if (flag) (acc) += clock64() - _t0

// ---------------------------------------------------------------------------------------------------------------
// dZ kernel
// ---------------------------------------------------------------------------------------------------------------
// Work order (identical in every role): runs = (utterance, t-block) assigned round-robin to CTAs; inside a run the
// valid tiles along u; inside a tile NP passes over H.  Accumulators: an even unit uses TMEM columns [0, NCZ), an odd
// unit [priv .. NCZ) (the SHARED zone, drained first by the epilogue) + [odd_base, 512): two units are in flight
// (MMA of unit q+1 over the epilogue of unit q) although 2*NCZ may exceed the 512 columns.
//
// PAIR = true: a thread-block cluster of 2 runs the kernel as ONE M = 256 machine (tcgen05 cta_group::2).  The kernel is bound by
// the L2 -> SM operand stream (1.79 MB per tile at H = 640, V = 1024: 29 GB per launch at C3, at the ~6.3 KB / clk the L2 can
// deliver), two thirds of it the W rows every tile re-reads.  The pair walks a run's u-blocks two at a time (CTA r owns
// u-block 2j + r) and shares ONE copy of every W stage: each CTA loads its own E' rows and HALF of the W rows, all bytes are
// counted on the leader's stage_full, the leader's MMA warp issues for both, the commits are multicast to both CTAs, and the
// epilogues of both CTAs release the accumulators on the leader's barriers.  With an odd number of u-blocks the last step's
// second CTA is padding: it loads the leader's rows again, takes part in every handshake and stores nothing.  The two CTAs'
// partial d_enc rows meet in global memory as two atomic adds onto the zeroed array (two addends: order-independent).
template <bool PROF, bool PAIR>
__global__ void __launch_bounds__(DZ_THREADS, 1) bwd_dz_kernel(const __grid_constant__ CUtensorMap tmap_e,
                                                               const __grid_constant__ CUtensorMap tmap_wp,
                                                               const __grid_constant__ CUtensorMap tmap_ws,
                                                               const __grid_constant__ CUtensorMap tmap_pred,
                                                               const __grid_constant__ CUtensorMap tmap_enc,
                                                               const BwdParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const int NCZ = p.NCZ, NP = p.NP, priv = p.priv, sh = p.sh, KBV = p.V >> 6, DZ_STAGES = p.dz_stages, nch = NCZ >> 5;
    const uint32_t rank = PAIR ? ptx::cluster_ctarank() : 0u;
    const bool leader = rank == 0;
    const int hP = PAIR ? priv >> 1 : priv, hS = PAIR ? sh >> 1 : sh;       // W rows of the private / shared zone THIS CTA loads
    const uint32_t stage_bytes = 16384u + (uint32_t)(hP + hS) * 128u;       // A [128 rows x 64 v] | B [hP + hS rows of W x 64 v]
    const int cta0 = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x, cstep = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    auto arrive_leader = [&](uint64_t* bar) {      // the leader's copy of a barrier collects both CTAs
        if (!PAIR || leader) ptx::mbar_arrive(bar);
        else ptx::mbar_arrive_cluster(ptx::mapa_u32(bar, 0));
    };
    // the unit's enc / pred rows for the epilogue's (1 - tanh^2): per 32-column chunk a pred box [32 fp32 x 8 rows] (1 KB,
    // SWIZZLE_128B) and an enc box [32 fp32 x 16 rows] (2 KB), loaded by warp 10 while the unit's MMAs run (measured before:
    // reading them with LDG put 54 % of the epilogue's stall samples on the L2 latency)
    uint8_t* predb = smem + (size_t)DZ_STAGES * stage_bytes;               // [nch][8 x 128 B]
    uint8_t* encb = predb + (size_t)nch * 1024;                            // [nch][16 x 128 B]
    uint8_t* dpb = encb + (size_t)nch * 2048;                              // [hh][buf][4][8][36] floats
    constexpr int DP_ONE = 4 * 8 * 36;                                     // floats per (hh, buf)
    uint64_t* bars = reinterpret_cast<uint64_t*>(dpb + DZ_EG * 2 * DP_ONE * 4);
    uint64_t* stage_full = bars;                         // [stages] TMA -> MMA
    uint64_t* stage_empty = stage_full + DZ_MAX_STAGES;  // [stages] MMA -> TMA
    uint64_t* acc_full = stage_empty + DZ_MAX_STAGES;    // [2] MMA -> epilogue (unit parity)
    uint64_t* priv_free = acc_full + 2;                  // [2] epilogue -> MMA
    uint64_t* shared_free = priv_free + 2;               // [1]
    uint64_t* epi_full = shared_free + 1;                // enc/pred TMA -> epilogue
    uint64_t* epi_empty = epi_full + 1;                  // epilogue -> enc/pred TMA
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(epi_empty + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int i = 0; i < DZ_MAX_STAGES; ++i) { ptx::mbar_init(&stage_full[i], 1); ptx::mbar_init(&stage_empty[i], 1); }
        ptx::mbar_init(epi_full, 1); ptx::mbar_init(epi_empty, DZ_EPI_WARPS);
        for (int i = 0; i < 2; ++i) { ptx::mbar_init(&acc_full[i], 1); ptx::mbar_init(&priv_free[i], (PAIR ? 2 : 1) * DZ_EPI_WARPS); }
        ptx::mbar_init(shared_free, (PAIR ? 2 : 1) * DZ_EPI_WARPS);
        ptx::fence_barrier_init();
    }
    if (warp == 1) {
        if (PAIR) { ptx::tmem_alloc2(tmem_ptr, TC_TMEM_COLS); ptx::tmem_relinquish2(); }
        else { ptx::tmem_alloc(tmem_ptr, TC_TMEM_COLS); ptx::tmem_relinquish(); }
    }
    if (warp == 0 && lane == 0) { ptx::prefetch_tmap(&tmap_e); ptx::prefetch_tmap(&tmap_wp); ptx::prefetch_tmap(&tmap_ws); }
    if (warp == DZ_TMA2_WARP && lane == 0) { ptx::prefetch_tmap(&tmap_pred); ptx::prefetch_tmap(&tmap_enc); }
    ptx::tc_fence_before();
    __syncthreads();
    if (PAIR) ptx::cluster_sync();       // the peer's barriers exist before anyone arrives on them remotely
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    const int nruns = p.nb * p.nTb;
    const bool pf = PROF && p.prof != nullptr && (lane == 0) && (warp == 0 || warp == 1 || warp == 2);   // PROF = false: all of it folds away
    long long pc[4] = {0, 0, 0, 0};
    const long long t_start = pf ? clock64() : 0;

    if (warp == 0) {
        // ===================== TMA: A = kept numerators [128 rows x 64 v], B = W rows [NCZ h x 64 v] =====================
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int run = cta0; run < nruns; run += cstep) {
                const int bl = run / p.nTb, tb = run - bl * p.nTb, b = p.b0 + bl;
                const int Tn = p.xlen[b], Un = p.ylen[b] + 1;
                if (tb * BW_TT >= Tn) continue;
                const int nub = (Un + BW_UU - 1) / BW_UU, nq = PAIR ? (nub + 1) >> 1 : nub;
                for (int j = 0; j < nq; ++j) {
                    const int ub = PAIR ? min(2 * j + (int)rank, nub - 1) : j;     // a padding CTA loads the leader's rows again
                    const int tile = (bl * p.nTb + tb) * p.nUb + ub;
                    const int sl = p.slot ? p.slot[tile] : tile;
                    for (int pass = 0; pass < NP; ++pass) {
                        const int n0 = pass * NCZ;
                        for (int kb = 0; kb < KBV; ++kb) {
                            { RB_PROF_BEGIN(pf); ptx::mbar_wait(&stage_empty[stage], phase ^ 1); RB_PROF_END(pf, pc[0]); }
                            uint8_t* st = smem + (size_t)stage * stage_bytes;
                            if (PAIR) {
                                // both CTAs' bytes complete on the LEADER's barrier; only the leader posts the expected count
                                if (leader) ptx::mbar_arrive_expect_tx(&stage_full[stage], 2u * stage_bytes);
                                const uint32_t bar = ptx::mapa_u32(&stage_full[stage], 0);
                                ptx::tma_load_2d_2sm(st, &tmap_e, bar, kb * 64, sl * 128);
                                ptx::tma_load_2d_2sm(st + 16384, &tmap_wp, bar, kb * 64, n0 + (int)rank * hP);
                                if (sh) ptx::tma_load_2d_2sm(st + 16384 + (size_t)hP * 128, &tmap_ws, bar, kb * 64, n0 + priv + (int)rank * hS);
                            } else {
                                ptx::mbar_arrive_expect_tx(&stage_full[stage], stage_bytes);
                                ptx::tma_load_2d(st, &tmap_e, &stage_full[stage], kb * 64, sl * 128);
                                ptx::tma_load_2d(st + 16384, &tmap_wp, &stage_full[stage], kb * 64, n0);
                                if (sh) ptx::tma_load_2d(st + 16384 + (size_t)priv * 128, &tmap_ws, &stage_full[stage], kb * 64, n0 + priv);
                            }
                            if (++stage == DZ_STAGES) { stage = 0; phase ^= 1; }
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA: D[128 x NCZ] += A[128 x 64] . B[NCZ x 64]^T, both operands K-major in smem =====================
        const uint32_t idescP = ptx::umma_idesc_bf16(PAIR ? 256 : 128, priv), idescS = ptx::umma_idesc_bf16(PAIR ? 256 : 128, sh ? sh : 16);
        int stage = 0; uint32_t phase = 0, q = 0;
        if (!PAIR || leader)
        for (int run = cta0; run < nruns; run += cstep) {
            const int bl = run / p.nTb, tb = run - bl * p.nTb, b = p.b0 + bl;
            const int Tn = p.xlen[b], Un = p.ylen[b] + 1;
            if (tb * BW_TT >= Tn) continue;
            const int nub = (Un + BW_UU - 1) / BW_UU, nq = PAIR ? (nub + 1) >> 1 : nub;
            for (int j = 0; j < nq; ++j)
                for (int pass = 0; pass < NP; ++pass, ++q) {
                    const uint32_t par = q & 1;
                    { RB_PROF_BEGIN(pf); ptx::mbar_wait(&priv_free[par], ((q >> 1) & 1) ^ 1); RB_PROF_END(pf, pc[0]); }
                    ptx::tc_fence_after();
                    const uint32_t dP = tmem_base + (par ? (uint32_t)p.odd_base : 0u), dS = tmem_base + (uint32_t)priv;
                    for (int kb = 0; kb < KBV; ++kb) {
                        { RB_PROF_BEGIN(pf); ptx::mbar_wait(&stage_full[stage], phase); RB_PROF_END(pf, pc[1]); }
                        const uint32_t sa = ptx::smem_u32(smem + (size_t)stage * stage_bytes);
                        const uint64_t ad = ptx::umma_desc_k_sw128(sa), bp = ptx::umma_desc_k_sw128(sa + 16384u),
                                       bs = ptx::umma_desc_k_sw128(sa + 16384u + (uint32_t)hP * 128u);
                        if (ptx::elect_one()) {
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                if (PAIR) ptx::umma_ss2(dP, ad + (uint64_t)(k * 2), bp + (uint64_t)(k * 2), idescP, (uint32_t)((kb | k) != 0));
                                else ptx::umma_bf16(dP, ad + (uint64_t)(k * 2), bp + (uint64_t)(k * 2), idescP, (uint32_t)((kb | k) != 0));
                            }
                        }
                        __syncwarp();
                        if (sh) {
                            if (kb == 0) {   // the shared zone still holds the previous unit until its epilogue has drained it
                                RB_PROF_BEGIN(pf);
                                ptx::mbar_wait(shared_free, (q & 1) ^ 1);
                                RB_PROF_END(pf, pc[2]);
                                ptx::tc_fence_after();
                            }
                            if (ptx::elect_one()) {
#pragma unroll
                                for (int k = 0; k < 4; ++k) {
                                    if (PAIR) ptx::umma_ss2(dS, ad + (uint64_t)(k * 2), bs + (uint64_t)(k * 2), idescS, (uint32_t)((kb | k) != 0));
                                    else ptx::umma_bf16(dS, ad + (uint64_t)(k * 2), bs + (uint64_t)(k * 2), idescS, (uint32_t)((kb | k) != 0));
                                }
                            }
                            __syncwarp();
                        }
                        if (ptx::elect_one()) {
                            if (PAIR) {
                                ptx::umma_commit2_mc(&stage_empty[stage], 3);
                                if (kb == KBV - 1) ptx::umma_commit2_mc(&acc_full[par], 3);
                            } else {
                                ptx::umma_commit(&stage_empty[stage]);
                                if (kb == KBV - 1) ptx::umma_commit(&acc_full[par]);
                            }
                        }
                        __syncwarp();
                        if (++stage == DZ_STAGES) { stage = 0; phase ^= 1; }
                    }
                }
        }
    } else if (warp == DZ_TMA2_WARP) {
        // ===================== enc / pred TMA for the epilogue: one unit ahead of it =====================
        if (lane == 0) {
            uint32_t uq = 0;
            for (int run = cta0; run < nruns; run += cstep) {
                const int bl = run / p.nTb, tb = run - bl * p.nTb, b = p.b0 + bl;
                const int Tn = p.xlen[b], Un = p.ylen[b] + 1;
                if (tb * BW_TT >= Tn) continue;
                const int nub = (Un + BW_UU - 1) / BW_UU;
                for (int ub = PAIR ? (int)rank : 0; ub < nub; ub += PAIR ? 2 : 1)     // live tiles of this CTA only
                    for (int pass = 0; pass < NP; ++pass, ++uq) {
                        ptx::mbar_wait(epi_empty, (uq & 1) ^ 1);
                        ptx::mbar_arrive_expect_tx(epi_full, (uint32_t)nch * 3072u);
                        for (int c = 0; c < nch; ++c) {
                            ptx::tma_load_2d(predb + c * 1024, &tmap_pred, epi_full, pass * NCZ + 32 * c, b * p.maxU + ub * BW_UU);
                            ptx::tma_load_2d(encb + c * 2048, &tmap_enc, epi_full, pass * NCZ + 32 * c, b * p.maxT + tb * BW_TT);
                        }
                    }
            }
        }
    } else {
        // ===================== epilogue (warps 2-9): g = rs_row * acc * (1 - tanh^2), tile sums =====================
        const int qd = warp & 3, hh = (warp - 2) >> 2, qslot = (warp - 2) & 3;
        const int r = qd * 32 + lane, ul = lane & 7;
        const int npr = priv >> 5, nsh = sh >> 5;                  // 32-column chunks of the private / shared zone
        // The unit's chunks in processing order -- shared zone first, then the private zone -- are dealt round-robin to the
        // DZ_EG groups: group hh takes positions hh, hh + DZ_EG, ...  (at most DZ_MAXJ = ceil(12 / DZ_EG) of them).
        const int nsh_h = (nsh - hh + DZ_EG - 1) / DZ_EG;           // how many of this warp's positions lie in the shared zone
        const int nj = (npr + nsh - hh + DZ_EG - 1) / DZ_EG;
        const uint32_t dp0 = ptx::smem_u32(dpb) + (uint32_t)hh * 2 * DP_ONE * 4;
        const int off4 = (ul & 1) * 16 + ((ul >> 1) & 1) * 8 + ((ul >> 2) & 1) * 4;   // columns this lane keeps after the u butterfly
        const int cbase = ((lane >> 3) & 1) * 16 + ((lane >> 4) & 1) * 8;              // ... after the t butterfly
        const uint32_t enc_a = ptx::smem_u32(encb) + (uint32_t)(r >> 3) * 128u, pred_a = ptx::smem_u32(predb) + (uint32_t)ul * 128u;
        uint32_t q = 0, nchunk = 0, eq = 0;      // q counts the pair's units (accumulator parity), eq this CTA's live units (enc / pred boxes)
        for (int run = cta0; run < nruns; run += cstep) {
            const int bl = run / p.nTb, tb = run - bl * p.nTb, b = p.b0 + bl;
            const int Tn = p.xlen[b], Un = p.ylen[b] + 1;
            if (tb * BW_TT >= Tn) continue;
            const int nub = (Un + BW_UU - 1) / BW_UU;
            const int t = tb * BW_TT + (r >> 3);
            float accE[2][DZ_MAXJ][4];
#pragma unroll
            for (int a = 0; a < 2; ++a)
#pragma unroll
                for (int j = 0; j < DZ_MAXJ; ++j)
#pragma unroll
                    for (int i = 0; i < 4; ++i) accE[a][j][i] = 0.f;
            const int nq = PAIR ? (nub + 1) >> 1 : nub;
            for (int jq = 0; jq < nq; ++jq) {
                const int ub = PAIR ? 2 * jq + (int)rank : jq;
                if (PAIR && ub >= nub) {
                    // padding half of the run's last step: release the accumulators the leader's MMAs wrote here, nothing else
                    for (int pass = 0; pass < NP; ++pass, ++q) {
                        ptx::mbar_wait(&acc_full[q & 1], (q >> 1) & 1);
                        ptx::tc_fence_after();
                        ptx::tc_fence_before();
                        __syncwarp();
                        if (lane == 0) {
                            if (sh) arrive_leader(shared_free);
                            arrive_leader(&priv_free[q & 1]);
                        }
                    }
                    continue;
                }
                const int tile = (bl * p.nTb + tb) * p.nUb + ub;
                const int tslot = p.slot ? p.slot[tile] : tile;              // < 0 only after a broken valid_tile_bound promise
                const float rs = tslot >= 0 ? __ldg(p.rowscale + (size_t)tslot * 128 + r) : 0.f;   // 0 outside the lattice
#pragma unroll
                for (int pass = 0; pass < 2; ++pass) {
                    if (pass >= NP) continue;
                    const uint32_t par = q & 1;
                    { RB_PROF_BEGIN(pf); ptx::mbar_wait(&acc_full[par], (q >> 1) & 1); RB_PROF_END(pf, pc[0]); }
                    ptx::tc_fence_after();
                    { RB_PROF_BEGIN(pf); ptx::mbar_wait(epi_full, eq & 1); RB_PROF_END(pf, pc[2]); }
                    const int n0 = pass * NCZ;
#pragma unroll
                    if ((sh && nsh_h == 0) || nj == 0) {       // no chunk of the shared zone / of the unit falls to this warp (narrow H)
                        __syncwarp();
                        if (lane == 0) {
                            if (sh && nsh_h == 0) arrive_leader(shared_free);
                            if (nj == 0) arrive_leader(&priv_free[par]);
                        }
                    }
#pragma unroll
                    for (int j = 0; j < DZ_MAXJ; ++j) {
                        if (j >= nj) continue;
                        const int pos = hh + DZ_EG * j, c = pos < nsh ? npr + pos : pos - nsh;      // chunk of this pass's NCZ columns
                        const uint32_t col = c < npr ? (par ? (uint32_t)p.odd_base : 0u) + 32u * c : 32u * c;
                        uint32_t v[32];
                        ptx::tmem_ld_32x32(tmem_base + ((uint32_t)(qd * 32) << 16) + col, v);
                        ptx::tmem_ld_wait();
                        if (j == nsh_h - 1 || j == nj - 1) {    // this warp is done with the shared zone / with the whole unit
                            ptx::tc_fence_before();
                            __syncwarp();
                            if (lane == 0) {
                                if (j == nsh_h - 1) arrive_leader(shared_free);
                                if (j == nj - 1) arrive_leader(&priv_free[par]);
                            }
                        }
                        const int h0 = n0 + 32 * c;
                        float g[32];
                        {
#pragma unroll
                            for (int i = 0; i < 8; ++i) {
                                const float4 e = ptx::lds128f(enc_a + (uint32_t)(c * 2048 + i * 16)),
                                             qq = ptx::lds128f(pred_a + (uint32_t)(c * 1024 + ((i ^ (ul & 7)) << 4)));
                                const float z0 = ptx::tanh_approx(e.x + qq.x), z1 = ptx::tanh_approx(e.y + qq.y),
                                            z2 = ptx::tanh_approx(e.z + qq.z), z3 = ptx::tanh_approx(e.w + qq.w);
                                const float d0 = __uint_as_float(v[4 * i]) * rs, d1 = __uint_as_float(v[4 * i + 1]) * rs,
                                            d2 = __uint_as_float(v[4 * i + 2]) * rs, d3 = __uint_as_float(v[4 * i + 3]) * rs;
                                g[4 * i] = fmaf(-d0 * z0, z0, d0); g[4 * i + 1] = fmaf(-d1 * z1, z1, d1);
                                g[4 * i + 2] = fmaf(-d2 * z2, z2, d2); g[4 * i + 3] = fmaf(-d3 * z3, z3, d3);
                            }
                        }
                        // ---- sum over u (8 adjacent lanes): butterfly that halves the register set at every step
                        {
                            float a16[16], a8[8];
                            const bool h1 = lane & 1, h2 = lane & 2, h4 = lane & 4;
#pragma unroll
                            for (int i = 0; i < 16; ++i) {
                                const float send = h1 ? g[i] : g[16 + i], keep = h1 ? g[16 + i] : g[i];
                                a16[i] = keep + __shfl_xor_sync(0xffffffffu, send, 1);
                            }
#pragma unroll
                            for (int i = 0; i < 8; ++i) {
                                const float send = h2 ? a16[i] : a16[8 + i], keep = h2 ? a16[8 + i] : a16[i];
                                a8[i] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
                            }
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const float send = h4 ? a8[i] : a8[4 + i], keep = h4 ? a8[4 + i] : a8[i];
                                accE[pass][j][i] += keep + __shfl_xor_sync(0xffffffffu, send, 4);
                            }
                        }
                        // ---- sum over t: 4 time steps inside the warp (lane bits 3, 4), then across the four quarter warps
                        {
                            float a16[16], a8[8];
                            const bool h8 = lane & 8, h16 = lane & 16;
#pragma unroll
                            for (int i = 0; i < 16; ++i) {
                                const float send = h8 ? g[i] : g[16 + i], keep = h8 ? g[16 + i] : g[i];
                                a16[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
                            }
#pragma unroll
                            for (int i = 0; i < 8; ++i) {
                                const float send = h16 ? a16[i] : a16[8 + i], keep = h16 ? a16[8 + i] : a16[i];
                                a8[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
                            }
                            const uint32_t dp = dp0 + (uint32_t)(nchunk & 1) * (DP_ONE * 4);
                            const uint32_t w = dp + (uint32_t)(((qslot * 8 + ul) * 36 + cbase) * 4);
                            ptx::sts128f(w, make_float4(a8[0], a8[1], a8[2], a8[3]));
                            ptx::sts128f(w + 16, make_float4(a8[4], a8[5], a8[6], a8[7]));
                            { RB_PROF_BEGIN(pf); ptx::named_bar_sync(1 + hh, 128); RB_PROF_END(pf, pc[1]); }
                            const int o = (qslot * 32 + lane) * 2, uo = o >> 5, co = o & 31;
                            float2 s = make_float2(0.f, 0.f);
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                const float2 x = ptx::lds64f(dp + (uint32_t)((((k * 8 + uo) * 36) + co) * 4));
                                s.x += x.x; s.y += x.y;
                            }
                            const int uu = ub * BW_UU + uo;
                            if (uu < p.maxU)
                                *reinterpret_cast<float2*>(p.ppred + (((size_t)tb * p.nb + bl) * p.maxU + uu) * p.H + h0 + co) = s;
                            ++nchunk;
                        }
                    }
                    __syncwarp();
                    if (lane == 0) ptx::mbar_arrive(epi_empty);      // this warp has read the unit's enc / pred rows
                    ++q; ++eq;
                }
            }
            // ---- the run is complete: this lane owns (t, 4 columns per chunk) of d_enc
            if (t < p.maxT) {
                float* drow = p.d_enc + ((size_t)b * p.maxT + t) * p.H;
#pragma unroll
                for (int pass = 0; pass < 2; ++pass) {
                    if (pass >= NP) continue;
#pragma unroll
                    for (int j = 0; j < DZ_MAXJ; ++j) {
                        if (j >= nj) continue;
                        const int pos = hh + DZ_EG * j, c = pos < nsh ? npr + pos : pos - nsh;
                        const float4 v4 = make_float4(accE[pass][j][0], accE[pass][j][1], accE[pass][j][2], accE[pass][j][3]);
                        if (PAIR) atomicAdd(reinterpret_cast<float4*>(drow + pass * NCZ + 32 * c + off4), v4);    // the two CTAs' halves of the run
                        else *reinterpret_cast<float4*>(drow + pass * NCZ + 32 * c + off4) = v4;
                    }
                }
            }
        }
    }
    if (pf) {   // [role 0..2][total, wait0..3]: role = TMA, MMA, epilogue warp 2
        long long* o = p.prof + ((size_t)blockIdx.x * 4 + warp) * 8;
        o[0] = clock64() - t_start; o[1] = pc[0]; o[2] = pc[1]; o[3] = pc[2]; o[4] = pc[3];
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (PAIR) ptx::cluster_sync();       // no CTA leaves while its peer may still arrive on its barriers
    if (warp == 1) {
        if (PAIR) ptx::tmem_dealloc2(tmem_base, TC_TMEM_COLS);
        else ptx::tmem_dealloc(tmem_base, TC_TMEM_COLS);
    }
}

// d_pred[b,u,:] = sum over the t-blocks that intersect the utterance of its partial planes (0 for u >= U_b).  The planes
// are Hp = 4 * H4 wide; d_pred (B, maxU, H) receives the first H columns of each row.
__global__ void __launch_bounds__(256) sum_pred_planes_kernel(const float4* __restrict__ ppred, const int* __restrict__ xlen,
                                                              const int* __restrict__ ylen, int b0, int nb, int maxU, int H4,
                                                              int H, float* __restrict__ d_pred) {
    const size_t n4 = (size_t)nb * maxU * H4;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
        const int bl = (int)(i / ((size_t)maxU * H4)), u = (int)((i / H4) % maxU), b = b0 + bl;
        const int h = (int)(i % H4) * 4;
        if (h >= H) continue;                   // padding columns of the planes
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        if (u < ylen[b] + 1) {
            const int ntb = (xlen[b] + BW_TT - 1) / BW_TT;
#pragma unroll 4
            for (int k = 0; k < ntb; ++k) {
                const float4 v = ppred[(size_t)k * n4 + i];
                acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
            }
        }
        if (H == 4 * H4) {
            reinterpret_cast<float4*>(d_pred)[(size_t)b0 * maxU * H4 + i] = acc;
        } else {
            float* o = d_pred + ((size_t)b0 * maxU + i / H4) * H + h;
            o[0] = acc.x;
            if (h + 1 < H) o[1] = acc.y;
            if (h + 2 < H) o[2] = acc.z;
            if (h + 3 < H) o[3] = acc.w;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// dW kernel
// ---------------------------------------------------------------------------------------------------------------
// CTA = (v-tile of DW_NV columns, h-item, split of the K = lattice-row range).  An h-item owns two block slots of 128 output
// rows; the block list is [h-block 0 .. nHB-1, SCALE]: the SCALE block is an A tile whose row 0 holds the row scales, so that
// row 0 of its product is db = sum_rows dl (H = 640: items (0,1) (2,3) (4,SCALE) -- three equal units of work per v-tile).
// K step = half a tile (64 lattice rows: 8 time steps x 8 label positions).
struct DwWork { int vt, item, split; };
__device__ __forceinline__ DwWork dw_decode(const BwdParams& p, int cta) {
    DwWork w;
    const int per_vt = p.nItems * p.S;
    w.vt = cta / per_vt;
    const int rem = cta - w.vt * per_vt;
    w.item = rem / p.S;
    w.split = rem - w.item * p.S;
    return w;
}
// block slot k2 of an item: index into [h-block 0 .. nHB-1, SCALE]; kind 0 = h-block, 1 = SCALE, 2 = none
__device__ __forceinline__ int dw_kind(const BwdParams& p, int item, int k2) {
    const int blk = 2 * item + k2;
    return blk < p.nHB ? 0 : (blk == p.nHB ? 1 : 2);
}

template <bool PROF>
__global__ void __launch_bounds__(DW_THREADS, 1) bwd_dw_kernel(const __grid_constant__ CUtensorMap tmap_e, const BwdParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    // stage = A: 2 x [128 x 64 k] K-major (32 KB) | B: 4 x [64 k x 64 v] MN-major (32 KB); beside the stages a ring of the
    // K steps' row scales (64 floats each), loaded DW_NRS - DW_STAGES steps ahead of the B tiles so that the A producers
    // only ever wait for the MMA to release a stage, never for a load
    constexpr uint32_t STAGE = 65536u;
    uint8_t* rsring = smem + DW_STAGES * STAGE;                 // [DW_NRS][64] floats
    uint64_t* bars = reinterpret_cast<uint64_t*>(rsring + DW_NRS * 256);
    uint64_t* b_full = bars;                       // [DW_STAGES] TMA -> MMA
    uint64_t* a_ready = b_full + DW_STAGES;        // producers -> MMA
    uint64_t* stage_empty = a_ready + DW_STAGES;   // MMA -> TMA, producers
    uint64_t* rs_full = stage_empty + DW_STAGES;   // [DW_NRS] TMA -> producers
    uint64_t* rs_empty = rs_full + DW_NRS;         // [DW_NRS] producers -> TMA
    uint64_t* acc_full = rs_empty + DW_NRS;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(acc_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const DwWork wk = dw_decode(p, blockIdx.x);
    const int v0 = wk.vt * DW_NV, Nv = min(DW_NV, p.V - v0), nbox = Nv >> 6;
    const int kind0 = dw_kind(p, wk.item, 0), kind1 = dw_kind(p, wk.item, 1);
    const int narr = 8 * ((kind0 == 0) + (kind1 == 0)) + (kind0 == 1) + (kind1 == 1);   // warps that arrive on a_ready per K step
    if (threadIdx.x == 0) {
        for (int i = 0; i < DW_STAGES; ++i) {
            ptx::mbar_init(&b_full[i], 1); ptx::mbar_init(&a_ready[i], narr ? narr : 1); ptx::mbar_init(&stage_empty[i], 1);
        }
        for (int i = 0; i < DW_NRS; ++i) { ptx::mbar_init(&rs_full[i], 1); ptx::mbar_init(&rs_empty[i], narr ? narr : 1); }
        ptx::mbar_init(acc_full, 1);
        ptx::fence_barrier_init();
    }
    // the SCALE block's A tile: rows 1..127 stay zero for the whole kernel, row 0 is rewritten every K step
#pragma unroll
    for (int k2 = 0; k2 < 2; ++k2)
        if ((k2 ? kind1 : kind0) == 1)
            for (int st = 0; st < DW_STAGES; ++st)
                for (int i = threadIdx.x; i < 16384 / 16; i += DW_THREADS)
                    reinterpret_cast<uint4*>(smem + (size_t)st * STAGE + k2 * 16384)[i] = make_uint4(0u, 0u, 0u, 0u);
    ptx::fence_proxy_async_smem();
    if (warp == 1) { ptx::tmem_alloc(tmem_ptr, TC_TMEM_COLS); ptx::tmem_relinquish(); }
    if (warp == 0 && lane == 0) ptx::prefetch_tmap(&tmap_e);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    const long long cnt = *p.count;
    const int s_beg = (int)(cnt * wk.split / p.S), s_end = (int)(cnt * (wk.split + 1) / p.S);
    const int per_utt = p.nTb * p.nUb;
    const bool pf = PROF && p.prof != nullptr && (lane == 0) && (warp == 0 || warp == 1 || warp == 2);   // PROF = false: all of it folds away
    long long pc[4] = {0, 0, 0, 0};
    const long long t_start = pf ? clock64() : 0;

    if (warp == 0) {
        // ===================== TMA: B = kept numerators, boxes [64 rows x 64 v] (rows = K); the rows' scales run ahead =====================
        if (lane == 0) {
            const int nsteps = 2 * (s_end - s_beg);
            auto load_rs = [&](int k) {        // K step k -> ring entry k % DW_NRS
                const int e = k % DW_NRS;
                ptx::mbar_wait(&rs_empty[e], ((k / DW_NRS) & 1) ^ 1);
                ptx::mbar_arrive_expect_tx(&rs_full[e], 256u);
                ptx::bulk_load_1d(rsring + e * 256, p.rowscale + (size_t)(s_beg + (k >> 1)) * 128 + (k & 1) * 64, 256u, &rs_full[e]);
            };
            if (narr)
                for (int k = 0; k < DW_NRS - DW_STAGES && k < nsteps; ++k) load_rs(k);
            int stage = 0; uint32_t phase = 0, it = 0;
            for (int s = s_beg; s < s_end; ++s)
                for (int half = 0; half < 2; ++half, ++it) {
                    if (narr && (int)it + DW_NRS - DW_STAGES < nsteps) load_rs((int)it + DW_NRS - DW_STAGES);
                    { RB_PROF_BEGIN(pf); ptx::mbar_wait(&stage_empty[stage], phase ^ 1); RB_PROF_END(pf, pc[0]); }
                    ptx::mbar_arrive_expect_tx(&b_full[stage], (uint32_t)nbox * 8192u);
                    uint8_t* bs = smem + (size_t)stage * STAGE + 32768;
                    for (int j = 0; j < nbox; ++j)
                        ptx::tma_load_2d(bs + j * 8192, &tmap_e, &b_full[stage], v0 + 64 * j, s * 128 + half * 64);
                    if (++stage == DW_STAGES) { stage = 0; phase ^= 1; }
                }
        }
    } else if (warp == 1) {
        // ===================== MMA: D[slot][128 x Nv] += A[128 x 64 k] . E'[64 k x Nv]  (A K-major, B MN-major) =====================
        const uint32_t idesc = ptx::umma_idesc_bf16(128, Nv, 0, 1);
        int stage = 0; uint32_t phase = 0, it = 0;
        for (int s = s_beg; s < s_end; ++s)
            for (int half = 0; half < 2; ++half, ++it) {
                { RB_PROF_BEGIN(pf); ptx::mbar_wait(&b_full[stage], phase); RB_PROF_END(pf, pc[0]); }
                if (narr) { RB_PROF_BEGIN(pf); ptx::mbar_wait(&a_ready[stage], phase); RB_PROF_END(pf, pc[1]); }
                ptx::tc_fence_after();
                const uint32_t sa = ptx::smem_u32(smem + (size_t)stage * STAGE);
                const uint64_t bd = ptx::umma_desc_mn_sw128(sa + 32768u, 8192u);
                if (ptx::elect_one()) {
#pragma unroll
                    for (int k2 = 0; k2 < 2; ++k2) {
                        if ((k2 ? kind1 : kind0) != 2) {
                            const uint64_t ad = ptx::umma_desc_k_sw128(sa + (uint32_t)k2 * 16384u);
#pragma unroll
                            for (int k = 0; k < 4; ++k)   // K = 16 lattice rows per MMA: 32 B along A's rows, 16 x 128 B of B
                                ptx::umma_bf16(tmem_base + (uint32_t)k2 * DW_NV, ad + (uint64_t)(k * 2), bd + (uint64_t)(k * 128),
                                               idesc, (uint32_t)((it | (uint32_t)k) != 0));
                        }
                    }
                    ptx::umma_commit(&stage_empty[stage]);
                    if (s == s_end - 1 && half == 1) ptx::umma_commit(acc_full);
                }
                __syncwarp();
                if (++stage == DW_STAGES) { stage = 0; phase ^= 1; }
            }
    } else {
        // ===================== A producers (warps 2-17): thread = (column h of the joint, 4 of a K step's 8 time rows), or the SCALE row; then the epilogue =====================
        const int ptid = threadIdx.x - 64, k2 = ptid >> 8, q2 = (ptid >> 7) & 1, hl = ptid & 127;
        const int kind = k2 ? kind1 : kind0, hb = 2 * wk.item + k2;
        const int h = hb * 128 + hl;
        const uint32_t smem_a = ptx::smem_u32(smem);
        if (kind == 0) {
            // Inputs of slot s+1 (its tile's 8 pred rows and this thread's 8 enc rows of column h) are loaded while slot s is
            // computed; the slot's descriptor is read two slots ahead, so no load waits on another load.  No division and no
            // 64-bit multiply per load: the descriptor carries the tile's first rows (measured: with the tile decoded here and
            // the rows addressed one by one, two thirds of the producers' instructions were integer address arithmetic and the
            // kernel was issue-bound).  Rows outside the lattice carry rs = 0, so no length test is needed, only in-bounds reads.
            const int hc = min(h, p.H - 1);     // columns past H (H % 128 != 0) feed output rows nobody reads
            auto meta_at = [&](int s) { return s < s_end ? __ldg(p.slot_meta + s) : make_int4(0, 0, 1, 1); };
            float pv[8], ev[8], npv[8], nev[8];     // ev[half * 4 + j] = enc row t0 + half * 8 + q2 * 4 + j
            auto load = [&](const int4 m, float* pvv, float* evv) {
                const char* pp = reinterpret_cast<const char*>(p.pred + (size_t)m.y * p.H + hc);
                const char* pe = reinterpret_cast<const char*>(p.enc + (size_t)m.x * p.H + hc);
                const uint32_t hb4 = (uint32_t)p.H * 4u;      // unsigned 32-bit byte offsets inside the tile: one IMAD.WIDE.U32 per address
#pragma unroll
                for (int k = 0; k < 8; ++k) pvv[k] = __ldg(reinterpret_cast<const float*>(pp + (uint32_t)min(k, m.w - 1) * hb4));
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    evv[k] = __ldg(reinterpret_cast<const float*>(pe + (uint32_t)min((k >> 2) * 8 + q2 * 4 + (k & 3), m.z - 1) * hb4));
            };
            load(meta_at(s_beg), pv, ev);
            int4 meta_n = meta_at(s_beg + 1);
            int stage = 0; uint32_t phase = 0, it = 0;
            for (int s = s_beg; s < s_end; ++s) {
                const int4 meta_nn = meta_at(s + 2);
                if (s + 1 < s_end) load(meta_n, npv, nev);
                for (int half = 0; half < 2; ++half, ++it) {
                    const int e_rs = it % DW_NRS;
                    { RB_PROF_BEGIN(pf); ptx::mbar_wait(&stage_empty[stage], phase ^ 1); RB_PROF_END(pf, pc[0]); }   // the MMAs that read this A slot retired
                    { RB_PROF_BEGIN(pf); ptx::mbar_wait(&rs_full[e_rs], (it / DW_NRS) & 1); RB_PROF_END(pf, pc[2]); }
                    const uint32_t arow = smem_a + (uint32_t)stage * STAGE + (uint32_t)(k2 * 16384 + hl * 128);
                    const uint32_t rsa = ptx::smem_u32(rsring) + (uint32_t)e_rs * 256u;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int tl = q2 * 4 + j;
                        const float e = half ? ev[4 + j] : ev[j];
                        const float4 r0 = ptx::lds128f(rsa + (uint32_t)(tl * 32)), r1 = ptx::lds128f(rsa + (uint32_t)(tl * 32 + 16));   // rs of rows tl*8 .. +7
                        const float rsv[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
                        float z[8];
#pragma unroll
                        for (int k = 0; k < 8; ++k) z[k] = ptx::tanh_approx(e + pv[k]) * rsv[k];
                        ptx::sts128(arow + (uint32_t)((tl ^ (hl & 7)) << 4),
                                    make_uint4(ptx::pack_bf16x2(z[0], z[1]), ptx::pack_bf16x2(z[2], z[3]), ptx::pack_bf16x2(z[4], z[5]),
                                               ptx::pack_bf16x2(z[6], z[7])));
                    }
                    ptx::fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) { ptx::mbar_arrive(&a_ready[stage]); ptx::mbar_arrive(&rs_empty[e_rs]); }
                    if (++stage == DW_STAGES) { stage = 0; phase ^= 1; }
                }
                meta_n = meta_nn;
#pragma unroll
                for (int k = 0; k < 8; ++k) pv[k] = npv[k];
#pragma unroll
                for (int k = 0; k < 8; ++k) ev[k] = nev[k];
            }
        } else if (kind == 1 && (ptid & 255) < 32) {
            // SCALE block: one warp copies the stage's 64 row scales (bf16) into row 0 of the slot's A tile (row 0: no swizzle)
            int stage = 0; uint32_t phase = 0, it = 0;
            for (int s = s_beg; s < s_end; ++s)
                for (int half = 0; half < 2; ++half, ++it) {
                    const int e_rs = it % DW_NRS;
                    ptx::mbar_wait(&stage_empty[stage], phase ^ 1);
                    ptx::mbar_wait(&rs_full[e_rs], (it / DW_NRS) & 1);
                    const uint32_t st = smem_a + (uint32_t)stage * STAGE;
                    const float2 x = ptx::lds64f(ptx::smem_u32(rsring) + (uint32_t)e_rs * 256u + (uint32_t)lane * 8u);
                    ptx::sts32(st + (uint32_t)(k2 * 16384) + (uint32_t)lane * 4u, ptx::pack_bf16x2(x.x, x.y));
                    ptx::fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) { ptx::mbar_arrive(&a_ready[stage]); ptx::mbar_arrive(&rs_empty[e_rs]); }
                    if (++stage == DW_STAGES) { stage = 0; phase ^= 1; }
                }
        }
        // ---- epilogue: this warp's 32 rows of block slot k2, Nv columns -> accumulated into the split's partial plane
        if (kind != 2 && s_end > s_beg) {
            { RB_PROF_BEGIN(pf); ptx::mbar_wait(acc_full, 0); RB_PROF_END(pf, pc[1]); }
            ptx::tc_fence_after();
            const int qd = warp & 3, hr = hb * 128 + qd * 32 + lane;
            // h-block: row hr of the dW plane; SCALE block: only TMEM lane 0 carries data (db)
            const bool on = kind == 0 ? hr < p.Hrows : (qd == 0 && lane == 0);
            float* dst = kind == 0 ? p.dWp + ((size_t)wk.split * p.Hrows + hr) * p.V + v0 : p.dbp + (size_t)wk.split * p.V + v0;
            if (kind == 0 || qd == 0) {
                for (int j = q2 * (Nv >> 6); j < (q2 + 1) * (Nv >> 6); ++j) {     // the slot's two warps per lane quarter take half the columns each
                    uint32_t v[32];
                    ptx::tmem_ld_32x32(tmem_base + ((uint32_t)(qd * 32) << 16) + (uint32_t)(k2 * DW_NV + j * 32), v);
                    ptx::tmem_ld_wait();
                    if (on) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            float4* d4 = reinterpret_cast<float4*>(dst + j * 32 + i * 4);
                            const float4 x = *d4;
                            *d4 = make_float4(__uint_as_float(v[4 * i]) + x.x, __uint_as_float(v[4 * i + 1]) + x.y,
                                              __uint_as_float(v[4 * i + 2]) + x.z, __uint_as_float(v[4 * i + 3]) + x.w);
                        }
                    }
                }
            }
        }
    }
    if (pf) {   // [role 0..2][total, wait0, wait1]: role = TMA, MMA, producer warp 2
        long long* o = p.prof + ((size_t)blockIdx.x * 4 + warp) * 8;
        o[0] = clock64() - t_start; o[1] = pc[0]; o[2] = pc[1]; o[3] = pc[2]; o[4] = pc[3];
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 1) ptx::tmem_dealloc(tmem_base, TC_TMEM_COLS);
}

// ---------------------------------------------------------------------------------------------------------------
// dW kernel, CTA-pair form (default)
// ---------------------------------------------------------------------------------------------------------------
// The one-CTA kernel above regenerates every z tile once per 256-column v-tile (4 x at V = 1024) and its 16 producer warps,
// not the tensor pipe, set its pace (measured: 1420 cycles of tanh per K step against 1048 cycles of MMA).  A wider output tile
// per z tile needs more accumulator columns than one CTA has for two row blocks, so here a CLUSTER OF 2 owns the two block
// slots of an h-item: CTA r regenerates block 2*item + r ONCE per K step and multiplies it against 512 columns of E'
// (tcgen05 cta_group::2, M = 256: rows 0-127 accumulate in CTA 0's tensor memory, rows 128-255 in CTA 1's, all 512 columns
// each).  Per K step and CTA: 8 k tanh instead of 16 k, the same 32 KB of E' (each CTA loads half of the columns of both
// N = 256 instructions), the same 1024 cycles of tensor pipe -- which now is the bound.  Barriers as in the dZ pair kernel.
constexpr int DW2_STAGES = 4;
constexpr int DW2_NV = 512;
constexpr uint32_t DW2_STAGE = 49152u;      // A [128 x 64 k] K-major (16 KB) | B: 2 instructions x 2 boxes [64 k x 64 v] MN-major (32 KB)

template <bool PROF>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(DW_THREADS, 1) bwd_dw2_kernel(const __grid_constant__ CUtensorMap tmap_e, const BwdParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* rsring = smem + DW2_STAGES * DW2_STAGE;            // [DW_NRS][64] floats
    uint64_t* bars = reinterpret_cast<uint64_t*>(rsring + DW_NRS * 256);
    uint64_t* b_full = bars;                       // [stages] both CTAs' TMA -> leader's MMA
    uint64_t* a_ready = b_full + DW2_STAGES;       // both CTAs' producers -> leader's MMA
    uint64_t* stage_empty = a_ready + DW2_STAGES;  // MMA (multicast commit) -> TMA, producers of both CTAs
    uint64_t* rs_full = stage_empty + DW2_STAGES;  // [DW_NRS] TMA -> producers (local)
    uint64_t* rs_empty = rs_full + DW_NRS;         // [DW_NRS] producers -> TMA (local)
    uint64_t* acc_full = rs_empty + DW_NRS;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(acc_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = ptx::cluster_ctarank();
    const bool leader = rank == 0;
    DwWork wk;
    {
        const int pair = blockIdx.x >> 1, per_vt = p.nItems * p.S;
        wk.vt = pair / per_vt;
        const int rem = pair - wk.vt * per_vt;
        wk.item = rem / p.S;
        wk.split = rem - wk.item * p.S;
    }
    const int v0 = wk.vt * DW2_NV, Nv = min(DW2_NV, p.V - v0);
    // the two N <= 256 instructions of a K step; N is rounded up to whole 64-column boxes per CTA (columns past V are
    // zero-filled by the TMA and never stored)
    const int N0 = min(256, (Nv + 127) & ~127), N1 = Nv > 256 ? (Nv - 256 + 127) & ~127 : 0;
    const int nb0 = N0 >> 7, nb1 = N1 >> 7;        // boxes per CTA and instruction
    const int kind = dw_kind(p, wk.item, (int)rank), kind_peer = dw_kind(p, wk.item, (int)rank ^ 1);
    auto warps_of = [](int k) { return k == 0 ? 16 : (k == 1 ? 1 : 0); };      // producer warps that arrive per K step
    const int narr = warps_of(kind), narr_pair = narr + warps_of(kind_peer);
    if (threadIdx.x == 0) {
        for (int i = 0; i < DW2_STAGES; ++i) {
            ptx::mbar_init(&b_full[i], 1); ptx::mbar_init(&a_ready[i], narr_pair ? narr_pair : 1); ptx::mbar_init(&stage_empty[i], 1);
        }
        for (int i = 0; i < DW_NRS; ++i) { ptx::mbar_init(&rs_full[i], 1); ptx::mbar_init(&rs_empty[i], narr ? narr : 1); }
        ptx::mbar_init(acc_full, 1);
        ptx::fence_barrier_init();
    }
    // A tiles of a SCALE block (rows 1..127 stay zero, row 0 is rewritten every K step) and of an empty slot (all zero)
    if (kind != 0)
        for (int st = 0; st < DW2_STAGES; ++st)
            for (int i = threadIdx.x; i < 16384 / 16; i += DW_THREADS)
                reinterpret_cast<uint4*>(smem + (size_t)st * DW2_STAGE)[i] = make_uint4(0u, 0u, 0u, 0u);
    ptx::fence_proxy_async_smem();
    if (warp == 1) { ptx::tmem_alloc2(tmem_ptr, TC_TMEM_COLS); ptx::tmem_relinquish2(); }
    if (warp == 0 && lane == 0) ptx::prefetch_tmap(&tmap_e);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::cluster_sync();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    const long long cnt = *p.count;
    const int s_beg = (int)(cnt * wk.split / p.S), s_end = (int)(cnt * (wk.split + 1) / p.S);
    const int nsteps = 2 * (s_end - s_beg);
    const bool pf = PROF && p.prof != nullptr && (lane == 0) && (warp == 0 || warp == 1 || warp == 2);
    long long pc[4] = {0, 0, 0, 0};
    const long long t_start = pf ? clock64() : 0;
    auto arrive_leader = [&](uint64_t* bar) {
        if (leader) ptx::mbar_arrive(bar);
        else ptx::mbar_arrive_cluster(ptx::mapa_u32(bar, 0));
    };

    if (warp == 0) {
        // ===================== TMA: this CTA's half of the K step's E' columns; the rows' scales run ahead =====================
        if (lane == 0) {
            auto load_rs = [&](int k) {
                const int e = k % DW_NRS;
                ptx::mbar_wait(&rs_empty[e], ((k / DW_NRS) & 1) ^ 1);
                ptx::mbar_arrive_expect_tx(&rs_full[e], 256u);
                ptx::bulk_load_1d(rsring + e * 256, p.rowscale + (size_t)(s_beg + (k >> 1)) * 128 + (k & 1) * 64, 256u, &rs_full[e]);
            };
            if (narr)
                for (int k = 0; k < DW_NRS - DW2_STAGES && k < nsteps; ++k) load_rs(k);
            const uint32_t tx = (uint32_t)(nb0 + nb1) * 8192u;
            int stage = 0; uint32_t phase = 0, it = 0;
            for (int s = s_beg; s < s_end; ++s)
                for (int half = 0; half < 2; ++half, ++it) {
                    if (narr && (int)it + DW_NRS - DW2_STAGES < nsteps) load_rs((int)it + DW_NRS - DW2_STAGES);
                    { RB_PROF_BEGIN(pf); ptx::mbar_wait(&stage_empty[stage], phase ^ 1); RB_PROF_END(pf, pc[0]); }
                    if (leader) ptx::mbar_arrive_expect_tx(&b_full[stage], 2u * tx);
                    const uint32_t bar = ptx::mapa_u32(&b_full[stage], 0);
                    uint8_t* bs = smem + (size_t)stage * DW2_STAGE + 16384;
                    const int row = s * 128 + half * 64;
                    for (int j = 0; j < nb0; ++j)
                        ptx::tma_load_2d_2sm(bs + j * 8192, &tmap_e, bar, v0 + (int)rank * (N0 >> 1) + 64 * j, row);
                    for (int j = 0; j < nb1; ++j)
                        ptx::tma_load_2d_2sm(bs + 16384 + j * 8192, &tmap_e, bar, v0 + 256 + (int)rank * (N1 >> 1) + 64 * j, row);
                    if (++stage == DW2_STAGES) { stage = 0; phase ^= 1; }
                }
        }
    } else if (warp == 1) {
        // ===================== MMA (leader): D[256 x Nv] += A[256 x 64 k] . E'[64 k x Nv], two N <= 256 instructions per 16 rows =====================
        const uint32_t idesc0 = ptx::umma_idesc_bf16(256, N0, 0, 1), idesc1 = ptx::umma_idesc_bf16(256, N1 ? N1 : 128, 0, 1);
        int stage = 0; uint32_t phase = 0, it = 0;
        if (leader)
        for (int s = s_beg; s < s_end; ++s)
            for (int half = 0; half < 2; ++half, ++it) {
                { RB_PROF_BEGIN(pf); ptx::mbar_wait(&b_full[stage], phase); RB_PROF_END(pf, pc[0]); }
                if (narr_pair) { RB_PROF_BEGIN(pf); ptx::mbar_wait(&a_ready[stage], phase); RB_PROF_END(pf, pc[1]); }
                ptx::tc_fence_after();
                const uint32_t sa = ptx::smem_u32(smem + (size_t)stage * DW2_STAGE);
                const uint64_t ad = ptx::umma_desc_k_sw128(sa), bd0 = ptx::umma_desc_mn_sw128(sa + 16384u, 8192u),
                               bd1 = ptx::umma_desc_mn_sw128(sa + 32768u, 8192u);
                if (ptx::elect_one()) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) {   // K = 16 lattice rows per MMA: 32 B along A's rows, 16 x 128 B of B
                        ptx::umma_ss2(tmem_base, ad + (uint64_t)(k * 2), bd0 + (uint64_t)(k * 128), idesc0, (uint32_t)((it | (uint32_t)k) != 0));
                        if (N1) ptx::umma_ss2(tmem_base + 256u, ad + (uint64_t)(k * 2), bd1 + (uint64_t)(k * 128), idesc1, (uint32_t)((it | (uint32_t)k) != 0));
                    }
                    ptx::umma_commit2_mc(&stage_empty[stage], 3);
                    if (s == s_end - 1 && half == 1) ptx::umma_commit2_mc(acc_full, 3);
                }
                __syncwarp();
                if (++stage == DW2_STAGES) { stage = 0; phase ^= 1; }
            }
    } else {
        // ===================== A producers (warps 2-17): thread = (column h of this CTA's block, 2 of a K step's 8 time rows), or the SCALE row; then the epilogue =====================
        const int ptid = threadIdx.x - 64, q4 = ptid >> 7, hl = ptid & 127;
        const int hb = 2 * wk.item + (int)rank, h = hb * 128 + hl;
        const uint32_t smem_a = ptx::smem_u32(smem);
        if (kind == 0) {
            const int hc = min(h, p.H - 1);
            auto meta_at = [&](int s) { return s < s_end ? __ldg(p.slot_meta + s) : make_int4(0, 0, 1, 1); };
            float pv[8], ev[4], npv[8], nev[4];     // ev[half * 2 + j] = enc row t0 + half * 8 + q4 * 2 + j
            auto load = [&](const int4 m, float* pvv, float* evv) {
                const char* pp = reinterpret_cast<const char*>(p.pred + (size_t)m.y * p.H + hc);
                const char* pe = reinterpret_cast<const char*>(p.enc + (size_t)m.x * p.H + hc);
                const uint32_t hb4 = (uint32_t)p.H * 4u;
#pragma unroll
                for (int k = 0; k < 8; ++k) pvv[k] = __ldg(reinterpret_cast<const float*>(pp + (uint32_t)min(k, m.w - 1) * hb4));
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    evv[k] = __ldg(reinterpret_cast<const float*>(pe + (uint32_t)min((k >> 1) * 8 + q4 * 2 + (k & 1), m.z - 1) * hb4));
            };
            load(meta_at(s_beg), pv, ev);
            int4 meta_n = meta_at(s_beg + 1);
            int stage = 0; uint32_t phase = 0, it = 0;
            for (int s = s_beg; s < s_end; ++s) {
                const int4 meta_nn = meta_at(s + 2);
                if (s + 1 < s_end) load(meta_n, npv, nev);
                for (int half = 0; half < 2; ++half, ++it) {
                    const int e_rs = it % DW_NRS;
                    { RB_PROF_BEGIN(pf); ptx::mbar_wait(&stage_empty[stage], phase ^ 1); RB_PROF_END(pf, pc[0]); }
                    { RB_PROF_BEGIN(pf); ptx::mbar_wait(&rs_full[e_rs], (it / DW_NRS) & 1); RB_PROF_END(pf, pc[2]); }
                    const uint32_t arow = smem_a + (uint32_t)stage * DW2_STAGE + (uint32_t)(hl * 128);
                    const uint32_t rsa = ptx::smem_u32(rsring) + (uint32_t)e_rs * 256u;
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const int tl = q4 * 2 + j;
                        const float e = half ? ev[2 + j] : ev[j];
                        const float4 r0 = ptx::lds128f(rsa + (uint32_t)(tl * 32)), r1 = ptx::lds128f(rsa + (uint32_t)(tl * 32 + 16));
                        const float rsv[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
                        float z[8];
#pragma unroll
                        for (int k = 0; k < 8; ++k) z[k] = ptx::tanh_approx(e + pv[k]) * rsv[k];
                        ptx::sts128(arow + (uint32_t)((tl ^ (hl & 7)) << 4),
                                    make_uint4(ptx::pack_bf16x2(z[0], z[1]), ptx::pack_bf16x2(z[2], z[3]), ptx::pack_bf16x2(z[4], z[5]),
                                               ptx::pack_bf16x2(z[6], z[7])));
                    }
                    ptx::fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) { arrive_leader(&a_ready[stage]); ptx::mbar_arrive(&rs_empty[e_rs]); }
                    if (++stage == DW2_STAGES) { stage = 0; phase ^= 1; }
                }
                meta_n = meta_nn;
#pragma unroll
                for (int k = 0; k < 8; ++k) pv[k] = npv[k];
#pragma unroll
                for (int k = 0; k < 4; ++k) ev[k] = nev[k];
            }
        } else if (kind == 1 && ptid < 32) {
            // SCALE block: one warp copies the K step's 64 row scales (bf16) into row 0 of the A tile (row 0: no swizzle)
            int stage = 0; uint32_t phase = 0, it = 0;
            for (int s = s_beg; s < s_end; ++s)
                for (int half = 0; half < 2; ++half, ++it) {
                    const int e_rs = it % DW_NRS;
                    ptx::mbar_wait(&stage_empty[stage], phase ^ 1);
                    ptx::mbar_wait(&rs_full[e_rs], (it / DW_NRS) & 1);
                    const float2 x = ptx::lds64f(ptx::smem_u32(rsring) + (uint32_t)e_rs * 256u + (uint32_t)lane * 8u);
                    ptx::sts32(smem_a + (uint32_t)stage * DW2_STAGE + (uint32_t)lane * 4u, ptx::pack_bf16x2(x.x, x.y));
                    ptx::fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) { arrive_leader(&a_ready[stage]); ptx::mbar_arrive(&rs_empty[e_rs]); }
                    if (++stage == DW2_STAGES) { stage = 0; phase ^= 1; }
                }
        }
        // ---- epilogue: this CTA's 128 rows x Nv columns -> accumulated into the split's partial plane (4 warps per lane quarter)
        if (s_end > s_beg) {
            { RB_PROF_BEGIN(pf); ptx::mbar_wait(acc_full, 0); RB_PROF_END(pf, pc[1]); }
            ptx::tc_fence_after();
            if (kind != 2) {
                const int qd = warp & 3, hr = hb * 128 + qd * 32 + lane;
                const bool on = kind == 0 ? hr < p.Hrows : (qd == 0 && lane == 0);      // SCALE block: only TMEM lane 0 carries data (db)
                float* dst = kind == 0 ? p.dWp + ((size_t)wk.split * p.Hrows + hr) * p.V + v0 : p.dbp + (size_t)wk.split * p.V + v0;
                if (kind == 0 || qd == 0) {
                    const int nch = Nv >> 5;
                    for (int j = q4; j < nch; j += 4) {
                        uint32_t v[32];
                        ptx::tmem_ld_32x32(tmem_base + ((uint32_t)(qd * 32) << 16) + (uint32_t)(j * 32), v);
                        ptx::tmem_ld_wait();
                        if (on) {
#pragma unroll
                            for (int i = 0; i < 8; ++i) {
                                float4* d4 = reinterpret_cast<float4*>(dst + j * 32 + i * 4);
                                const float4 x = *d4;
                                *d4 = make_float4(__uint_as_float(v[4 * i]) + x.x, __uint_as_float(v[4 * i + 1]) + x.y,
                                                  __uint_as_float(v[4 * i + 2]) + x.z, __uint_as_float(v[4 * i + 3]) + x.w);
                            }
                        }
                    }
                }
            }
        }
    }
    if (pf) {
        long long* o = p.prof + ((size_t)blockIdx.x * 4 + warp) * 8;
        o[0] = clock64() - t_start; o[1] = pc[0]; o[2] = pc[1]; o[3] = pc[2]; o[4] = pc[3];
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::cluster_sync();
    if (warp == 1) ptx::tmem_dealloc2(tmem_base, TC_TMEM_COLS);
}

}  // namespace rb
