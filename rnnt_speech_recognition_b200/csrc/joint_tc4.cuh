// joint_tc4.cuh -- the fused joint forward kernel of joint_tc3.cuh as a CTA-PAIR kernel (thread-block cluster of 2,
// tcgen05 cta_group::2).  Every 128-row tile re-reads all of W^T; with one CTA per tile that stream (22.5 GB of L2 -> SM
// traffic per launch at C3) bounds the kernel.  Here two CTAs own two consecutive tiles and ONE copy of every W^T stage
// between them:
//   * W^T ring: each stage holds THIS CTA's 32 of the chunk's 64 vocabulary rows (4 KB per K block instead of 8); both
//     halves complete on the LEADER's w_full (cp.async.bulk.tensor...cta_group::2, barrier addressed through mapa)
//   * MMA: only the leader's warp 13 issues tcgen05.mma.cta_group::2 with M = 256 (128 TMEM lanes per CTA): A from each
//     CTA's own z columns, B = the two shared-memory halves, D in the same accumulator columns of both CTAs
//   * barriers: z_full (16 arrivals) and acc_empty (8) live in the leader and collect both CTAs (remote arrive through
//     mapa); w_empty / acc_full / z_free are signalled in both CTAs by tcgen05.commit...multicast::cluster
// Everything else -- input ring, producers, epilogues, TMEM budget -- is joint_tc3's code; a CTA whose tile lies outside the
// valid lattice feeds zeros and keeps every handshake.  PTX forms validated by tools/probes/mma2_probe (profiles/r02).
#pragma once
#include "joint_tc3.cuh"

namespace rb {

// W stages are half as large as joint_tc3's: twice as many fit
inline Tc2Geom tc4_geometry(int H, int V) {
    Tc2Geom g = tc3_geometry(H, V);
    if (!g.ok) return g;
    const size_t in_bytes = (size_t)TC3_IN_STAGES * TC3_IN_STAGE;
    const size_t bias_bytes = V <= 4096 ? (size_t)V * 4 : 0;
    const size_t budget = 232448 - 1024 - 1024 - in_bytes - bias_bytes;
    g.stages = (int)(budget / ((size_t)g.ks * 4096));
    if (g.stages > 12) g.stages = 12;
    g.smem_bytes = 1024 + in_bytes + (size_t)g.stages * g.ks * 4096 + 1024 + bias_bytes;
    g.ok = g.stages >= 2;
    return g;
}

#ifndef RNNTB200_TC4_PRE
#define RNNTB200_TC4_PRE 4
#endif
constexpr int TC4_PRE = RNNTB200_TC4_PRE;      // K blocks of the next tile's z produced into registers ahead of z_free
static_assert(TC4_PRE >= 1, "at least the first K block is produced ahead");

template <int MODE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TC3_THREADS, 1) joint_tc4_kernel(const __grid_constant__ CUtensorMap tmap_wt,
                                                                   const __grid_constant__ CUtensorMap tmap_pred,
                                                                   const __grid_constant__ CUtensorMap tmap_enc,
                                                                   const JointTcParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const int KB = p.KB, NCH = p.NCH, stages = p.stages, NBUF = p.nbuf, KS = p.ks;
    const uint32_t stage_bytes = (uint32_t)KS * 4096u;    // THIS CTA's half of a W stage: KS slabs of [32 v x 64 k]
    const uint32_t rank = ptx::cluster_ctarank();
    const bool leader = rank == 0;
    constexpr int NC = TC2_NC;
    uint8_t* insm = smem;                                 // TC3_IN_STAGES x {pred box k-half 0, k-half 1 (1 KB each, SW128), enc box (4 KB)}
    constexpr uint32_t IN_STAGE = TC3_IN_STAGE;
    uint8_t* wsm = smem + TC3_IN_STAGES * IN_STAGE;       // stages x KS x [32 x 64] fp16 (this CTA's vocabulary half), SW128 K-major (TMA)
    uint64_t* bars = reinterpret_cast<uint64_t*>(wsm + (size_t)stages * stage_bytes);
    uint64_t* z_full = bars;                              // [TC_MAX_KB]      producers -> MMA (K block in TMEM)
    uint64_t* z_free = bars + TC_MAX_KB;                  //                  MMA -> producers
    uint64_t* w_full = z_free + 1;                        // [TC2_MAX_STAGES] TMA -> MMA
    uint64_t* w_empty = w_full + TC2_MAX_STAGES;          // [TC2_MAX_STAGES] MMA -> TMA
    uint64_t* acc_full = w_empty + TC2_MAX_STAGES;        // [TC2_MAX_NBUF]   MMA -> epilogue
    uint64_t* acc_empty = acc_full + TC2_MAX_NBUF;        // [TC2_MAX_NBUF]   epilogue -> MMA
    uint64_t* in_full = acc_empty + TC2_MAX_NBUF;         // [TC3_IN_STAGES]  input TMA -> producers
    uint64_t* in_empty = in_full + TC3_IN_STAGES;         // [TC3_IN_STAGES]  producers -> input TMA
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(in_empty + TC3_IN_STAGES);
    float* bias2 = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + 1024);   // bias * log2(e) for Vp <= 4096 (else read from global)
    const bool bias_in_smem = p.Vp <= 4096;
    // a padding column v >= V gets the bias -inf: its numerator 2^(y - ref) is exactly 0 (ref, the maximum of the first 32
    // logits, always includes column 0 and stays finite)
    if (bias_in_smem)
        for (int i = threadIdx.x; i < p.Vp; i += TC3_THREADS) bias2[i] = i < p.V ? __ldg(p.bias + i) * 1.4426950408889634f : -CUDART_INF_F;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int i = 0; i < TC_MAX_KB; ++i) ptx::mbar_init(&z_full[i], 16);      // 8 producer warps of EACH CTA (the leader's copy is used)
        ptx::mbar_init(z_free, 1);
        for (int i = 0; i < TC2_MAX_STAGES; ++i) { ptx::mbar_init(&w_full[i], 1); ptx::mbar_init(&w_empty[i], 1); }
        for (int i = 0; i < TC2_MAX_NBUF; ++i) { ptx::mbar_init(&acc_full[i], 1); ptx::mbar_init(&acc_empty[i], 8); }   // 4 epilogue warps of each CTA (leader's copy)
        for (int i = 0; i < TC3_IN_STAGES; ++i) { ptx::mbar_init(&in_full[i], 1); ptx::mbar_init(&in_empty[i], 8); }
        ptx::fence_barrier_init();
    }
    if (warp == 13) { ptx::tmem_alloc2(tmem_ptr, TC_TMEM_COLS); ptx::tmem_relinquish2(); }   // the same warp of both CTAs
    if (warp == 12 && lane == 0) ptx::prefetch_tmap(&tmap_wt);
    if (warp == 14 && lane == 0) { ptx::prefetch_tmap(&tmap_pred); ptx::prefetch_tmap(&tmap_enc); }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::cluster_sync();                                  // the peer's barriers exist before anyone arrives on them remotely
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    const uint32_t acc0 = tmem_base + (uint32_t)KB * 32;  // accumulator region starts after the z columns
    const int ntiles = p.nb * p.nTb * p.nUb, npairs = (ntiles + 1) >> 1, pstart = blockIdx.x >> 1, pstep = gridDim.x >> 1;
    // The pair walks tile pairs (2q, 2q+1), one tile per CTA.  A CTA whose tile lies outside the valid lattice still takes
    // part in every handshake of a live pair (z = 0, no input loads, no stores); a pair with two such tiles is skipped by all
    // roles alike.
    auto my_tile = [&](int q) { return 2 * q + (int)rank; };
    auto tile_ok = [&](int t) { return t < ntiles && decode_tile(p, t).valid; };
    auto pair_ok = [&](int q) { return tile_ok(2 * q) || tile_ok(2 * q + 1); };
    // arrive on the LEADER's copy of a barrier (its count collects both CTAs)
    auto arrive_leader = [&](uint64_t* bar) {
        if (leader) ptx::mbar_arrive(bar);
        else ptx::mbar_arrive_cluster(ptx::mapa_u32(bar, 0));
    };

    if (warp == 14) {
        // ===================== enc / pred TMA: one K block of the tile's rows per ring stage, runs ahead across tiles
        if (lane == 0 && !(p.dbg & 8)) {
            int st = 0; uint32_t ph = 0;
            const uint32_t tx = 2u * (uint32_t)p.UU * 128u + (uint32_t)p.TT * 256u;
            for (int q = pstart; q < npairs; q += pstep) {
                const int tile = my_tile(q);
                if (!tile_ok(tile)) continue;            // nothing to load for a padding tile (or a dead pair)
                const TileInfo ti = decode_tile(p, tile);
                for (int kb = 0; kb < KB; ++kb) {
                    ptx::mbar_wait(&in_empty[st], ph ^ 1);
                    ptx::mbar_arrive_expect_tx(&in_full[st], tx);
                    uint8_t* base = insm + (size_t)st * IN_STAGE;
                    ptx::tma_load_2d(base, &tmap_pred, &in_full[st], kb * 64, ti.b * p.maxU + ti.u0);
                    ptx::tma_load_2d(base + TC3_PRED_BOX, &tmap_pred, &in_full[st], kb * 64 + 32, ti.b * p.maxU + ti.u0);
                    ptx::tma_load_2d(base + 2 * TC3_PRED_BOX, &tmap_enc, &in_full[st], kb * 64, ti.b * p.maxT + ti.t0);
                    if (++st == TC3_IN_STAGES) { st = 0; ph ^= 1; }
                }
            }
        }
    } else if (warp == 12) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int q = pstart; q < npairs; q += pstep) {
                if (!pair_ok(q)) continue;
                if (p.dbg & 4) continue;
                for (int c = 0; c < NCH; ++c)
                    for (int kb0 = 0; kb0 < KB; kb0 += KS) {   // KB % KS == 0: one 3-D box = KS K-block slabs
                        ptx::mbar_wait(&w_empty[stage], phase ^ 1);
                        // both halves complete on the LEADER's barrier; only the leader posts the expected bytes
                        if (leader) ptx::mbar_arrive_expect_tx(&w_full[stage], 2u * stage_bytes);
                        ptx::tma_load_3d_2sm(wsm + (size_t)stage * stage_bytes, &tmap_wt, ptx::mapa_u32(&w_full[stage], 0), 0,
                                             c * NC + 32 * (int)rank, kb0);
                        if (++stage == stages) { stage = 0; phase ^= 1; }
                    }
            }
        }
    } else if (warp == 13) {
        // ===================== MMA issuer: A from TMEM, B from smem =====================
        // The WHOLE warp runs this loop convergently and one elected lane issues: descriptors, TMEM addresses and
        // barrier addresses then stay in uniform registers.  (Issuing from inside `if (lane == 0)` made every
        // operand a vector register that had to be moved to the uniform datapath per instruction -- measured
        // 117 cycles per N=64 MMA instead of the 32-cycle dispatch floor.)
        const uint32_t idesc = ptx::umma_idesc_f16(256, NC);   // M = 256: 128 lanes in each CTA of the pair
        int stage = 0; uint32_t phase = 0, g = 0, it = 0;
        if (leader)
        for (int q = pstart; q < npairs; q += pstep) {
            if (!pair_ok(q)) continue;
            for (int c = 0; c < NCH; ++c, ++g) {
                const uint32_t buf = g % NBUF, use = g / NBUF;
                if (!(p.dbg & 128)) {
                    ptx::mbar_wait(&acc_empty[buf], (use & 1) ^ 1);
                    ptx::tc_fence_after();
                }
                const uint32_t d_tmem = acc0 + buf * NC;
                for (int kb0 = 0; kb0 < KB; kb0 += KS) {
                    if (!(p.dbg & 4)) ptx::mbar_wait(&w_full[stage], phase);
                    // TMA-written smem is consumed by the same (async) proxy the MMA reads through: the mbarrier wait
                    // alone orders it.  tcgen05.fence::after_thread_sync is only needed where OTHER THREADS' tcgen05
                    // traffic is involved: after acc_empty (epilogue tcgen05.ld) and z_full (producer tcgen05.st).
                    if (p.dbg & 64) ptx::tc_fence_after();
                    const uint64_t bdesc0 = ptx::umma_desc_k_sw128(ptx::smem_u32(wsm + (size_t)stage * stage_bytes));
                    const uint32_t a_st = tmem_base + (uint32_t)kb0 * 32;
                    if (c == 0 && !(p.dbg & 8)) {
                        // first chunk of a tile: each K block of z must have landed in TMEM before it is read
                        for (int i = 0; i < KS; ++i) {
                            ptx::mbar_wait(&z_full[kb0 + i], it & 1);
                            ptx::tc_fence_after();
                            if (ptx::elect_one()) {
#pragma unroll
                                for (int k = 0; k < 4; ++k)
                                    ptx::umma_ts2(d_tmem, a_st + i * 32 + k * 8, bdesc0 + (uint64_t)(i * 256 + k * 2),
                                                      idesc, (uint32_t)((kb0 | i | k) != 0));
                            }
                            __syncwarp();
                        }
                    } else {
                        // steady state: the whole stage (up to 20 MMAs) AND its commits from ONE elected block with
                        // immediate operand offsets.  The single issuing thread is the pace-setter at N=64 (the probe
                        // reaches the 32-cycle floor only with >= 20 MMAs per block), so nothing else goes in between.
                        if (ptx::elect_one()) {
#pragma unroll
                            for (int i = 0; i < 5; ++i) {
                                if (i < KS) {
#pragma unroll
                                    for (int k = 0; k < 4; ++k)
                                        ptx::umma_ts2(d_tmem, a_st + i * 32 + k * 8,
                                                          bdesc0 + (uint64_t)(i * 256 + k * 2), idesc,
                                                          (i | k) ? 1u : (uint32_t)(kb0 != 0));
                                }
                            }
                            if (!(p.dbg & 4)) ptx::umma_commit2_mc(&w_empty[stage], 3);
                            if (kb0 + KS >= KB) ptx::umma_commit2_mc(&acc_full[buf], 3);
                        }
                        __syncwarp();
                        if (++stage == stages) { stage = 0; phase ^= 1; }
                        continue;
                    }
                    if (ptx::elect_one()) {
                        if (!(p.dbg & 4)) ptx::umma_commit2_mc(&w_empty[stage], 3);
                        if (kb0 + KS >= KB) ptx::umma_commit2_mc(&acc_full[buf], 3);
                    }
                    __syncwarp();
                    if (++stage == stages) { stage = 0; phase ^= 1; }
                }
            }
            if (!(p.dbg & 8) && ptx::elect_one()) ptx::umma_commit2_mc(z_free, 3);
            __syncwarp();
            ++it;
        }
    } else if (warp >= 4 && warp < 12) {
        // ===================== producers (warps 4-11): thread = (lattice row r2 = TMEM lane, k-half hh) =====================
        const int pw = warp - 4;
        const int q4 = pw & 3, hh = pw >> 2, r2 = q4 * 32 + lane;
        const bool fast_tanh = (p.dbg & 512) == 0;
        const uint32_t insm_a = ptx::smem_u32(insm);
        uint32_t it = 0; int st = 0; uint32_t ph = 0;
        for (int q = pstart; q < npairs; q += pstep) {
            if (p.dbg & 8) continue;
            if (!pair_ok(q)) continue;
            const int tile = my_tile(q);
            if (!tile_ok(tile)) {
                // the peer's tile is live: feed zeros for this CTA's half of the M = 256 instruction and keep every handshake
                uint32_t zz[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) zz[i] = 0u;
                for (int kb = 0; kb < KB; ++kb) {
                    if (kb == 0) ptx::mbar_wait(z_free, (it & 1) ^ 1);
                    ptx::tmem_st_32x16(tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(kb * 32 + hh * 16), zz);
                    ptx::tmem_st_wait();
                    ptx::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) arrive_leader(&z_full[kb]);
                }
                ++it;
                continue;
            }
            const TileInfo ti = decode_tile(p, tile);
            const int tl = r2 / p.UU, ul = r2 % p.UU;   // row of the enc box / of the pred box
            const bool ok = (ti.t0 + tl) < ti.Tn && (ti.u0 + ul) < ti.Un;
            // one K block of z: this thread's 32 columns (k-half hh) of its lattice row, tanh -> fp16 pairs
            auto produce = [&](uint32_t (&zr)[16]) {
                ptx::mbar_wait(&in_full[st], ph);
                const uint32_t base = insm_a + (uint32_t)st * IN_STAGE;
                const uint32_t prow = base + (uint32_t)hh * TC3_PRED_BOX + (uint32_t)(ul * 128);      // SW128: chunk c at (c ^ (row & 7)) * 16
                const uint32_t erow = base + 2 * TC3_PRED_BOX + (uint32_t)(tl * 256 + hh * 128);       // plain layout
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const float4 q = ptx::lds128f(prow + (uint32_t)((c ^ (ul & 7)) << 4));
                    const float4 e = ptx::lds128f(erow + (uint32_t)(c << 4));
                    if (ok && !fast_tanh) {
                        zr[c * 2 + 0] = ptx::pack_f16x2(ptx::tanh_accurate(e.x + q.x), ptx::tanh_accurate(e.y + q.y));
                        zr[c * 2 + 1] = ptx::pack_f16x2(ptx::tanh_accurate(e.z + q.z), ptx::tanh_accurate(e.w + q.w));
                    } else if (ok) {   // default: tanh.approx (one MUFU op instead of two, 2^-11 relative); RNNTB200_DBG bit 512 selects the accurate form
                        zr[c * 2 + 0] = ptx::pack_f16x2(ptx::tanh_approx(e.x + q.x), ptx::tanh_approx(e.y + q.y));
                        zr[c * 2 + 1] = ptx::pack_f16x2(ptx::tanh_approx(e.z + q.z), ptx::tanh_approx(e.w + q.w));
                    } else {
                        zr[c * 2 + 0] = 0u; zr[c * 2 + 1] = 0u;
                    }
                }
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(&in_empty[st]);                       // this warp is done with the stage
                if (++st == TC3_IN_STAGES) { st = 0; ph ^= 1; }
            };
            auto store = [&](int kb, const uint32_t (&zr)[16]) {      // asynchronous: completed by the next tcgen05.wait::st
                ptx::tmem_st_32x16(tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(kb * 32 + hh * 16), zr);
            };
            auto publish = [&](int kb0, int n) {                      // K blocks [kb0, kb0 + n) of this warp's rows are in tensor memory
                ptx::tmem_st_wait();
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0)
                    for (int i = 0; i < n; ++i) arrive_leader(&z_full[kb0 + i]);
            };
            // z is single-buffered in tensor memory: its columns are free only when the previous tile's MMAs have retired
            // (z_free).  The first TC4_PRE K blocks of the tile are produced into REGISTERS while those MMAs still run, so
            // that after z_free only KB - TC4_PRE blocks remain on the tile's critical path.
            uint32_t zp[TC4_PRE][16];
            const int npre = KB < TC4_PRE ? KB : TC4_PRE;
#pragma unroll
            for (int i = 0; i < TC4_PRE; ++i)
                if (i < npre) produce(zp[i]);
            ptx::mbar_wait(z_free, (it & 1) ^ 1);
#pragma unroll
            for (int i = 0; i < TC4_PRE; ++i)
                if (i < npre) store(i, zp[i]);
            publish(0, npre);
            // (Producing block kb+1 while the tcgen05.st of block kb is still in flight -- i.e. publishing kb one block later --
            //  was measured slower: 2.86 vs 2.73 ms.  The first chunk's MMAs trail the producers block by block, so what counts
            //  is when each block becomes available, not the producers' throughput.)
            for (int kb = npre; kb < KB; ++kb) {
                produce(zp[0]);
                store(kb, zp[0]);
                publish(kb, 1);
            }
            ++it;
        }
    } else if (warp < 4) {
        // ===================== epilogue warps 0-3: thread = lattice cell (TMEM lane) =====================
        // (Eight epilogue warps -- two per lattice row, each taking one 32-column half of every chunk and combining their row
        //  states through shared memory -- were measured: 2.80 vs 2.71 ms in keep mode, 2.54 vs 2.54 without.  The epilogue is
        //  not short of warps; the 0.34 ms it costs comes from sharing the MUFU / issue slots with the producers.)
        constexpr float LOG2E = 1.4426950408889634f, LN2 = 0.6931471805599453f;
        const uint32_t bias_a = ptx::smem_u32(bias2);
        uint32_t g = 0;
        for (int q = pstart; q < npairs; q += pstep) {
            if (!pair_ok(q)) continue;
            const int tile = my_tile(q);
            if (!tile_ok(tile)) {                        // padding half of a live pair: release the accumulators, nothing else
                for (int c = 0; c < NCH; ++c, ++g) {
                    const uint32_t buf = g % NBUF, use = g / NBUF;
                    ptx::mbar_wait(&acc_full[buf], use & 1);
                    ptx::tc_fence_after();
                    ptx::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) arrive_leader(&acc_empty[buf]);
                }
                continue;
            }
            const TileInfo ti = decode_tile(p, tile);
            const int tslot = p.slot ? p.slot[tile] : tile;                        // row block of this tile in the kept arrays
            const bool has_slot = tslot >= 0;       // false only when the caller's valid_tile_bound was too small (flagged by tile_compact_kernel)
            const size_t rowbase = (size_t)(has_slot ? tslot : 0) * 128;
            const int r = warp * 32 + lane;
            const int t = ti.t0 + r / p.UU, u = ti.u0 + r % p.UU;
            const bool rv = t < ti.Tn && u < ti.Un;
            const int lab = (rv && u < ti.Un - 1) ? p.labels[(size_t)ti.b * (p.maxU - 1) + u] : -1;
            const long long cell = ((long long)ti.b * p.maxT + t) * p.maxU + u;
            float m2 = -CUDART_INF_F, s = 0.f, yb = 0.f, yl = 0.f, ref = 0.f;
            const uint32_t lane_addr = acc0 + ((uint32_t)(warp * 32) << 16);
            for (int c = 0; c < NCH; ++c, ++g) {
                const uint32_t buf = g % NBUF, use = g / NBUF;
                ptx::mbar_wait(&acc_full[buf], use & 1);
                ptx::tc_fence_after();
#pragma unroll
                for (int j = 0; j < NC / 32; ++j) {
                    if (p.dbg & 256) continue;
                    uint32_t v[32];
                    ptx::tmem_ld_32x32(lane_addr + buf * NC + j * 32, v);
                    ptx::tmem_ld_wait();
                    if (p.dbg & 1) { s += __uint_as_float(v[0]); continue; }
                    const int col0 = c * NC + j * 32;
                    float y[32];
                    if (bias_in_smem) {
                        // the 32 biases of the group (pre-scaled by log2 e) as 8 broadcast 16-byte shared-memory loads -- one
                        // wavefront each -- instead of one load and 32 shuffles
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const float4 b4 = ptx::lds128f(bias_a + (uint32_t)((col0 + 4 * i) * 4));
                            y[4 * i] = fmaf(__uint_as_float(v[4 * i]), LOG2E, b4.x); y[4 * i + 1] = fmaf(__uint_as_float(v[4 * i + 1]), LOG2E, b4.y);
                            y[4 * i + 2] = fmaf(__uint_as_float(v[4 * i + 2]), LOG2E, b4.z); y[4 * i + 3] = fmaf(__uint_as_float(v[4 * i + 3]), LOG2E, b4.w);
                        }
                    } else {
                        const float bv = col0 + lane < p.V ? __ldg(p.bias + col0 + lane) * LOG2E : -CUDART_INF_F;
#pragma unroll
                        for (int i = 0; i < 32; ++i)
                            y[i] = fmaf(__uint_as_float(v[i]), LOG2E, __shfl_sync(0xffffffffu, bv, i));
                    }
                    {
                        // The row sum is kept as (m2, s): sum = s * 2^m2.  m2 starts as the row's FIXED reference (the maximum of its
                        // first 32 logits) and stays there unless a later logit exceeds ref + 100 (detected on the group's sum, no
                        // running maximum is computed in the common path).  Both modes use the same arithmetic, hence identical costs
                        // whether or not the numerators are kept.  MODE 2 stores the numerators 2^(y - ref) (bf16).
                        if (col0 == 0) {
                            float gm = y[0];
#pragma unroll
                            for (int i = 1; i < 32; ++i) gm = fmaxf(gm, y[i]);
                            ref = gm; m2 = gm;
                        }
                        uint32_t o[16];
                        float accr = 0.f;
#pragma unroll
                        for (int i = 0; i < 32; i += 2) {
                            const float e0 = ptx::ex2_approx(y[i] - ref), e1 = ptx::ex2_approx(y[i + 1] - ref);
                            accr += e0 + e1;
                            if (MODE == 2) o[i >> 1] = ptx::pack_bf16x2(e0, e1);
                        }
                        if (accr < 1.0e30f) {            // every term below 2^100 (NaN / inf fail the test)
                            s += (m2 == ref) ? accr : accr * ptx::ex2_approx(ref - m2);
                        } else {
                            // a logit about 2^100 above the reference (never seen outside adversarial inputs): the group's sum is
                            // taken against its own maximum and the row switches to that frame; stored values are clamped at 2^100
                            float gm = y[0];
#pragma unroll
                            for (int i = 1; i < 32; ++i) gm = fmaxf(gm, y[i]);
                            const float mn = fmaxf(m2, gm);
                            float acc = 0.f;
#pragma unroll
                            for (int i = 0; i < 32; i += 2) {
                                acc += ptx::ex2_approx(y[i] - mn) + ptx::ex2_approx(y[i + 1] - mn);
                                if (MODE == 2)
                                    o[i >> 1] = ptx::pack_bf16x2(ptx::ex2_approx(fminf(y[i] - ref, 100.f)), ptx::ex2_approx(fminf(y[i + 1] - ref, 100.f)));
                            }
                            s = s * ptx::ex2_approx(m2 - mn) + acc;
                            m2 = mn;
                        }
                        if (MODE == 2 && has_slot) {
                            __nv_bfloat16* dst = p.dl + (rowbase + r) * p.Vp + col0;
                            ptx::st_global_256(dst, o);
                            ptx::st_global_256(dst + 16, o + 8);
                        }
                        if (p.blank >= col0 && p.blank < col0 + 32) {
#pragma unroll
                            for (int i = 0; i < 32; ++i)
                                if (col0 + i == p.blank) yb = y[i];
                        }
                        // logit[label_u]: the label differs per thread, so the wanted element sits at a DYNAMIC index of
                        // this thread's 32 registers: a binary select tree on the five index bits (31 selects, registers
                        // only -- the load/store pipe is the scarce unit of this kernel), run only when some lane of the
                        // warp has its label in this column group.
                        const int d = lab - col0;
                        const bool mine = (unsigned)d < 32u;
                        if (__any_sync(0xffffffffu, mine)) {
                            float s16[16], s8[8], s4[4];
#pragma unroll
                            for (int i = 0; i < 16; ++i) s16[i] = (d & 1) ? y[2 * i + 1] : y[2 * i];
#pragma unroll
                            for (int i = 0; i < 8; ++i) s8[i] = (d & 2) ? s16[2 * i + 1] : s16[2 * i];
#pragma unroll
                            for (int i = 0; i < 4; ++i) s4[i] = (d & 4) ? s8[2 * i + 1] : s8[2 * i];
                            const float s2a = (d & 8) ? s4[1] : s4[0], s2b = (d & 8) ? s4[3] : s4[2];
                            if (mine) yl = (d & 16) ? s2b : s2a;
                        }
                    }
                }
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0) arrive_leader(&acc_empty[buf]);
            }
            if (MODE == 2 && has_slot) p.gm[rowbase + r] = ref;   // the row's reference (log2 domain), coalesced
            if (rv && p.lse) {   // (lse == NULL: a backward-time recompute that only wants the kept activations)
                const float lse2 = m2 + log2f(s);
                p.lse[cell] = lse2 * LN2;
                const long long k = sk_index(ti.b, t, u, p.maxU, p.SK);
                p.lpb[k] = (yb - lse2) * LN2;
                if (u < ti.Un - 1) p.lpl[k] = (yl - lse2) * LN2;
            }
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::cluster_sync();                                  // the peer's barriers / tensor memory stay alive until both CTAs are done
    if (warp == 13) ptx::tmem_dealloc2(tmem_base, TC_TMEM_COLS);
}



template <int MODE>
inline rnntStatus_t tc4_launch(const Tc2Geom& g4, const CUtensorMap& tm, const CUtensorMap& tmp, const CUtensorMap& tme,
                               const JointTcParams& p, cudaStream_t s) {
    if (!tc_smem_optin(reinterpret_cast<const void*>(joint_tc4_kernel<MODE>))) return RNNT_STATUS_EXECUTION_FAILED;
    const int ntiles = p.nb * p.nTb * p.nUb, npairs = (ntiles + 1) / 2;
    int grid = 2 * npairs < tc_num_sms() ? 2 * npairs : tc_num_sms();
    grid &= ~1;
    ScopedTimer tmr(MODE == 0 ? "joint_tc4_kernel<fwd>" : "joint_tc4_kernel<fwd+keep>", s);
    joint_tc4_kernel<MODE><<<grid, TC3_THREADS, g4.smem_bytes, s>>>(tm, tmp, tme, p);
    return cudaGetLastError() == cudaSuccess ? RNNT_STATUS_SUCCESS : RNNT_STATUS_EXECUTION_FAILED;
}

}  // namespace rb
