// joint_tc3.cuh -- the fused joint FORWARD kernel (SURVEY 8 a1-a5, a11: model.py:158-166 + the log-softmax and
// gather of gpu_rnnt.h:73-80 / gpu_rnnt_kernel.h:5-9), generation 3: the A operand z = tanh(enc + pred) lives in
// TENSOR MEMORY as fp16, W^T (fp16) streams through a deep TMA ring, whole-stage MMA issue, TMA-fed producers.
//
// A dedicated warp TMA-loads the tile's pred rows (box [32 fp32 x UU rows], SWIZZLE_128B) and enc rows (box [64 x TT])
// K block by K block into a ring, RUNNING AHEAD across tiles; each producer thread reads ITS OWN lattice row straight
// from shared memory (conflict-free), applies tanh, packs to fp16 and writes its TMEM lane with tcgen05.st -- no
// staging pass, no inter-warp barrier, no register prefetch buffers.
//
// Operand format: fp16 (same tcgen05.mma.kind::f16 rate as bf16, 11-bit instead of 8-bit significand): z is in
// [-1, 1] and W ~ 1/sqrt(H), both far inside the fp16 range.  tanh is tanh.approx.f32 (2^-11 relative, one MUFU op);
// the fp32-accurate form (ex2 + rcp, two MUFU ops: +0.45 ms per launch at C3 because z production is exposed once per
// tile) changed neither the cost error (2.3e-5) nor the gradient error (2.9e-3) at C3 -- profiles/r02/accuracy.json.
//
// Roles (480 threads): warps 0-3 epilogue | 4-11 producers | 12 W TMA | 13 MMA | 14 enc/pred TMA
//
// MODE 0  forward: lse + (blank, label) log-probs per cell; nothing else leaves the SM
// MODE 2  forward that KEEPS its activations (rnntb200JointDesc.keep_activations, and the backward's per-chunk
//         recompute): MODE 0 + the softmax numerators E[row, v] = 2^(y_v - ref_row) as bf16, all columns of a row against
//         ONE frame ref_row, and ref_row itself.  ref_row is the maximum of the row's first 32 logits unless a later
//         group reaches 2^64 against it; the row then moves its frame up (here to its running maximum, in joint_tc4 to
//         that group's maximum) and rescales what it has already stored (tc_rescale_kept).  So every kept numerator is below 2^64 (bf16 keeps its 8 significant bits over
//         the whole exponent range), and a row scale flushed to 0 below 1e-30 drops at most 1e-30 * 2^64 ~ 2e-11 of
//         gradient.  The logit gradients are then row_scale * E: the two backward GEMMs take E straight from TMA and apply
//         the row scale in an epilogue (dZ) or to the regenerated A operand (dW) -- no per-element prologue.
#pragma once
#include <cuda_fp16.h>
#include "joint_tc.cuh"

namespace rb {

constexpr int TC3_THREADS = 480;
#ifndef RNNTB200_IN_STAGES
#define RNNTB200_IN_STAGES 3
#endif
constexpr int TC3_IN_STAGES = RNNTB200_IN_STAGES;
constexpr uint32_t TC3_PRED_BOX = 8 * 128, TC3_ENC_BOX = 16 * 256, TC3_IN_STAGE = 2 * TC3_PRED_BOX + TC3_ENC_BOX;   // 16 x 8 tiles
constexpr int TC2_NC = 64;             // vocabulary columns per accumulator buffer / W^T chunk
constexpr int TC2_MAX_STAGES = 24;
constexpr int TC2_MAX_NBUF = 4;

// z occupies H/2 TMEM columns (two fp16 per 32-bit column), the rest holds `nbuf` 64-column fp32 accumulators.
// One W stage = ks K-blocks ([64 v x 64 k] boxes, 8 KB each): the MMA thread pays one mbarrier wait and one commit per
// 4*ks MMAs (with ks = 1 the single issuing thread, not the tensor pipe, set the pace: 123 k cycles per tile measured).
struct Tc2Geom { int nbuf, stages, zcols, ks; size_t smem_bytes; bool ok; };
inline Tc2Geom tc3_geometry(int H, int V) {
    Tc2Geom g{};
    if (H % 64 || V % 64 || H < 64) return g;
    g.zcols = (H / 64) * 32;
    const int acc_cols = TC_TMEM_COLS - g.zcols;
    g.nbuf = acc_cols / TC2_NC;
    if (g.nbuf > TC2_MAX_NBUF) g.nbuf = TC2_MAX_NBUF;
    if (g.nbuf < 2) return g;
    const int KB = H / 64;
    g.ks = 1;
    for (int k = 5; k >= 1; --k)
        if (KB % k == 0) { g.ks = k; break; }   // largest divisor of KB that is <= 5: stages are never partial
    // smem: enc/pred ring (TC3_IN_STAGES x (2 x 1 KB pred boxes [32 fp32 x 8 rows] + 4 KB enc box [64 fp32 x 16 rows])) + W ring
    const size_t in_bytes = (size_t)TC3_IN_STAGES * TC3_IN_STAGE;
    const size_t bias_bytes = V <= 4096 ? (size_t)V * 4 : 0;
    const size_t budget = 232448 - 1024 - 1024 - in_bytes - bias_bytes;
    g.stages = (int)(budget / ((size_t)g.ks * 8192));
    if (g.stages > 8) g.stages = 8;
    g.smem_bytes = 1024 + in_bytes + (size_t)g.stages * g.ks * 8192 + 1024 + bias_bytes;
    g.ok = g.stages >= 2;
    return g;
}

// The row's frame moved up: multiply the n numerators it has already kept (n a multiple of 32, the row 32-byte aligned)
// by f = 2^(old frame - new frame) < 1.  The calling thread stored them itself, so plain loads see them.
__device__ __forceinline__ void tc_rescale_kept(__nv_bfloat16* row, int n, float f) {
    uint4* q = reinterpret_cast<uint4*>(row);
    for (int i = 0; i < n / 8; ++i) {
        uint4 w = q[i];
        uint32_t* x = reinterpret_cast<uint32_t*>(&w);
#pragma unroll
        for (int j = 0; j < 4; ++j)
            x[j] = ptx::pack_bf16x2(__uint_as_float(x[j] << 16) * f, __uint_as_float(x[j] & 0xffff0000u) * f);
        q[i] = w;
    }
}

template <int MODE>
__global__ void __launch_bounds__(TC3_THREADS, 1) joint_tc3_kernel(const __grid_constant__ CUtensorMap tmap_wt,
                                                                   const __grid_constant__ CUtensorMap tmap_pred,
                                                                   const __grid_constant__ CUtensorMap tmap_enc,
                                                                   const JointTcParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const int KB = p.KB, NCH = p.NCH, stages = p.stages, NBUF = p.nbuf, KS = p.ks;
    const uint32_t stage_bytes = (uint32_t)KS * 8192u;
    constexpr int NC = TC2_NC;
    uint8_t* insm = smem;                                 // TC3_IN_STAGES x {pred box k-half 0, k-half 1 (1 KB each, SW128), enc box (4 KB)}
    constexpr uint32_t IN_STAGE = TC3_IN_STAGE;
    uint8_t* wsm = smem + TC3_IN_STAGES * IN_STAGE;       // stages x KS x [64 x 64] bf16, SW128 K-major (TMA)
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
        for (int i = 0; i < TC_MAX_KB; ++i) ptx::mbar_init(&z_full[i], 8);
        ptx::mbar_init(z_free, 1);
        for (int i = 0; i < TC2_MAX_STAGES; ++i) { ptx::mbar_init(&w_full[i], 1); ptx::mbar_init(&w_empty[i], 1); }
        for (int i = 0; i < TC2_MAX_NBUF; ++i) { ptx::mbar_init(&acc_full[i], 1); ptx::mbar_init(&acc_empty[i], 4); }
        for (int i = 0; i < TC3_IN_STAGES; ++i) { ptx::mbar_init(&in_full[i], 1); ptx::mbar_init(&in_empty[i], 8); }
        ptx::fence_barrier_init();
    }
    if (warp == 13) { ptx::tmem_alloc(tmem_ptr, TC_TMEM_COLS); ptx::tmem_relinquish(); }
    if (warp == 12 && lane == 0) ptx::prefetch_tmap(&tmap_wt);
    if (warp == 14 && lane == 0) { ptx::prefetch_tmap(&tmap_pred); ptx::prefetch_tmap(&tmap_enc); }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    const uint32_t acc0 = tmem_base + (uint32_t)KB * 32;  // accumulator region starts after the z columns
    const int ntiles = p.nb * p.nTb * p.nUb;

    if (warp == 14) {
        // ===================== enc / pred TMA: one K block of the tile's rows per ring stage, runs ahead across tiles
        if (lane == 0 && !(p.dbg & 8)) {
            int st = 0; uint32_t ph = 0;
            const uint32_t tx = 2u * (uint32_t)p.UU * 128u + (uint32_t)p.TT * 256u;
            for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
                const TileInfo ti = decode_tile(p, tile);
                if (!ti.valid) continue;
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
            for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
                if (!decode_tile(p, tile).valid) continue;
                if (p.dbg & 4) continue;
                for (int c = 0; c < NCH; ++c)
                    for (int kb0 = 0; kb0 < KB; kb0 += KS) {   // KB % KS == 0: one 3-D box = KS K-block slabs
                        ptx::mbar_wait(&w_empty[stage], phase ^ 1);
                        ptx::mbar_arrive_expect_tx(&w_full[stage], stage_bytes);
                        ptx::tma_load_3d(wsm + (size_t)stage * stage_bytes, &tmap_wt, &w_full[stage], 0, c * NC, kb0);
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
        const uint32_t idesc = ptx::umma_idesc_f16(128, NC);
        int stage = 0; uint32_t phase = 0, g = 0, it = 0;
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            if (!decode_tile(p, tile).valid) continue;
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
                                    ptx::umma_bf16_ts(d_tmem, a_st + i * 32 + k * 8, bdesc0 + (uint64_t)(i * 512 + k * 2),
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
                                        ptx::umma_bf16_ts(d_tmem, a_st + i * 32 + k * 8,
                                                          bdesc0 + (uint64_t)(i * 512 + k * 2), idesc,
                                                          (i | k) ? 1u : (uint32_t)(kb0 != 0));
                                }
                            }
                            if (!(p.dbg & 4)) ptx::umma_commit(&w_empty[stage]);
                            if (kb0 + KS >= KB) ptx::umma_commit(&acc_full[buf]);
                        }
                        __syncwarp();
                        if (++stage == stages) { stage = 0; phase ^= 1; }
                        continue;
                    }
                    if (ptx::elect_one()) {
                        if (!(p.dbg & 4)) ptx::umma_commit(&w_empty[stage]);
                        if (kb0 + KS >= KB) ptx::umma_commit(&acc_full[buf]);
                    }
                    __syncwarp();
                    if (++stage == stages) { stage = 0; phase ^= 1; }
                }
            }
            if (!(p.dbg & 8) && ptx::elect_one()) ptx::umma_commit(z_free);
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
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            const TileInfo ti = decode_tile(p, tile);
            if (p.dbg & 8) continue;
            if (!ti.valid) continue;
            const int tl = r2 / p.UU, ul = r2 % p.UU;   // row of the enc box / of the pred box
            const bool ok = (ti.t0 + tl) < ti.Tn && (ti.u0 + ul) < ti.Un;
            for (int kb = 0; kb < KB; ++kb) {
                ptx::mbar_wait(&in_full[st], ph);
                const uint32_t base = insm_a + (uint32_t)st * IN_STAGE;
                const uint32_t prow = base + (uint32_t)hh * TC3_PRED_BOX + (uint32_t)(ul * 128);      // SW128: chunk c at (c ^ (row & 7)) * 16
                const uint32_t erow = base + 2 * TC3_PRED_BOX + (uint32_t)(tl * 256 + hh * 128);       // plain layout
                uint32_t zr[16];
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
                if (kb == 0) ptx::mbar_wait(z_free, (it & 1) ^ 1);   // previous tile's MMAs have retired: z columns reusable
                ptx::tmem_st_32x16(tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(kb * 32 + hh * 16), zr);
                ptx::tmem_st_wait();
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(&z_full[kb]);
            }
            ++it;
        }
    } else if (warp < 4) {
        // ===================== epilogue warps 0-3: thread = lattice cell (TMEM lane) =====================
        constexpr float LOG2E = 1.4426950408889634f, LN2 = 0.6931471805599453f;
        const uint32_t bias_a = ptx::smem_u32(bias2);
        uint32_t g = 0;
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            const TileInfo ti = decode_tile(p, tile);
            if (!ti.valid) continue;
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
                    const float bv = bias_in_smem ? __uint_as_float(ptx::lds32(bias_a + (uint32_t)((col0 + lane) * 4)))
                                                  : (col0 + lane < p.V ? __ldg(p.bias + col0 + lane) * LOG2E : -CUDART_INF_F);
                    float y[32];
#pragma unroll
                    for (int i = 0; i < 32; ++i)
                        y[i] = fmaf(__uint_as_float(v[i]), LOG2E, __shfl_sync(0xffffffffu, bv, i));
                    {
                        float gm = y[0];
#pragma unroll
                        for (int i = 1; i < 32; ++i) gm = fmaxf(gm, y[i]);
                        const float mn = fmaxf(m2, gm);
                        float acc = 0.f;
                        // Both modes form the group's sum from 2^(y - ref) against the row's frame ref (the maximum of its first 32
                        // logits until a group reaches 2^64 against it), rescaled once per group into the running-maximum frame:
                        // identical arithmetic, hence identical costs, whether or not the numerators are kept.  MODE 2 stores
                        // those numerators (bf16).
                        if (col0 == 0) ref = gm;
                        uint32_t o[16];
                        if (gm - ref <= 64.f) {
                            float accr = 0.f;
#pragma unroll
                            for (int i = 0; i < 32; i += 2) {
                                const float e0 = ptx::ex2_approx(y[i] - ref), e1 = ptx::ex2_approx(y[i + 1] - ref);
                                accr += e0 + e1;
                                if (MODE == 2) o[i >> 1] = ptx::pack_bf16x2(e0, e1);
                            }
                            acc = accr * ptx::ex2_approx(ref - mn);
                        } else {
                            // a logit more than 64 bits above the frame (a confident row whose maximum lies beyond its first 32
                            // columns): the row's frame moves up to the running maximum, which this group's numerators and the sum are
                            // taken against; the numerators kept so far are brought into the new frame
#pragma unroll
                            for (int i = 0; i < 32; i += 2) {
                                const float e0 = ptx::ex2_approx(y[i] - mn), e1 = ptx::ex2_approx(y[i + 1] - mn);
                                acc += e0 + e1;
                                if (MODE == 2) o[i >> 1] = ptx::pack_bf16x2(e0, e1);
                            }
                            if (MODE == 2 && has_slot) tc_rescale_kept(p.dl + (rowbase + r) * p.Vp, col0, ptx::ex2_approx(ref - mn));
                            ref = mn;
                        }
                        if (MODE == 2 && has_slot) {
                            __nv_bfloat16* dst = p.dl + (rowbase + r) * p.Vp + col0;
                            ptx::st_global_256(dst, o);
                            ptx::st_global_256(dst + 16, o + 8);
                        }
                        s = s * ptx::ex2_approx(m2 - mn) + acc;
                        m2 = mn;
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
                if (lane == 0) ptx::mbar_arrive(&acc_empty[buf]);
            }
            if (MODE == 2 && has_slot) p.gm[rowbase + r] = ref;   // the row's final frame (log2 domain), coalesced
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
    if (warp == 13) ptx::tmem_dealloc(tmem_base, TC_TMEM_COLS);
}


template <int MODE>
inline rnntStatus_t tc3_launch(const Tc2Geom& g3, const CUtensorMap& tm, const CUtensorMap& tmp, const CUtensorMap& tme,
                               const JointTcParams& p, cudaStream_t s) {
    if (!tc_smem_optin(reinterpret_cast<const void*>(joint_tc3_kernel<MODE>))) return RNNT_STATUS_EXECUTION_FAILED;
    const int ntiles = p.nb * p.nTb * p.nUb;
    const int grid = ntiles < tc_num_sms() ? ntiles : tc_num_sms();
    ScopedTimer tmr(MODE == 0 ? "joint_tc3_kernel<fwd>" : "joint_tc3_kernel<fwd+keep>", s);
    joint_tc3_kernel<MODE><<<grid, TC3_THREADS, g3.smem_bytes, s>>>(tm, tmp, tme, p);
    return cudaGetLastError() == cudaSuccess ? RNNT_STATUS_SUCCESS : RNNT_STATUS_EXECUTION_FAILED;
}

}  // namespace rb
