// joint_tc.cuh -- tensor-core (tcgen05 / TMEM / TMA) path of the fused joint + loss: shared definitions (tile
// geometry, kernel parameters, tensor maps, workspace layout, small helper kernels) and the host-side orchestration
// (tc_forward / tc_backward).  The kernels themselves: joint_tc3.cuh (forward), bwd_tc.cuh (the two backward
// contractions).  One persistent CTA per SM, each looping over 128-cell lattice tiles (16 time steps x 8 label positions
// of one utterance); the (B,T,U,H) activation tensor of model.py:158-163 and the (B,T,U,V) logits of model.py:165-166
// never exist in HBM.
//
// Any 1 <= H <= 768 and any V >= 1: the kernels always work on the PADDED problem Hp = ceil64(H), Vp = ceil64(V), whose
// padding contributes exactly zero -- W^T / W are converted into zero-padded (Vp, Hp) / (Hp, Vp) operands, a column v >= V
// gets the bias -inf (numerator 0), and when H % 64 != 0 enc / pred are staged into zero-padded (rows, Hp) arrays and d_enc
// is accumulated at width Hp and narrowed once.  Aligned shapes run exactly the launches they always did.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <mutex>
#include <unordered_map>
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdio>
#include <cstdlib>

#include "../../include/rnnt_b200.h"
#include "kernels_simt.cuh"
#include "ptx.cuh"
#include "timing.cuh"

namespace rb {

constexpr int TC_MAX_KB = 16;        // H <= 1024
constexpr int TC_TMEM_COLS = 512;

// the tensor-core kernels' granularity along H and V: every problem is run at (ceil64(H), ceil64(V))
inline int tc_pad64(int x) { return (x + 63) / 64 * 64; }
inline rnntb200JointDesc tc_padded(const rnntb200JointDesc& d) {
    rnntb200JointDesc p = d;
    p.H = tc_pad64(d.H);
    p.V = tc_pad64(d.V);
    return p;
}

struct TcGeom {
    int TT, UU, nTb, nUb;  // tile = TT x UU cells (TT*UU == 128); tiles per utterance
    int KB;
    bool ok;
};

// Tile shape: 16 time steps x 8 label positions.  (Round 1 picked, per problem, the power-of-two shape with the least
// padding; every tile re-reads its TT enc rows and UU pred rows (fp32, H wide) from L2, so a balanced shape also
// minimises that stream: 1 x 128 tiles cost 330 KB per tile, 16 x 8 cost 61 KB.  The backward kernels reduce a tile
// over u and over t in registers, which fixes the lane <-> (t, u) mapping, so the whole path now uses 16 x 8.)
inline TcGeom tc_geometry(int maxT, int maxU, int H, int V) {
    TcGeom g{};
    g.ok = false;
    if (H % 64 || V % 64 || H > 64 * TC_MAX_KB) return g;
    g.UU = 8;
    g.TT = 16;
    g.nTb = (maxT + g.TT - 1) / g.TT;
    g.nUb = (maxU + g.UU - 1) / g.UU;
    g.KB = H / 64;
    g.ok = true;
    return g;
}

// SM count of the CURRENT device (queried per call: the library may be used on several devices of one process)
inline int tc_num_sms() {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
        n = 148;
    return n;
}

// Geometry of the two backward kernels (bwd_tc.cuh), a pure function of (H, V) and the SM count.
//   dZ: NP passes over H of NCZ columns; accumulators of two consecutive passes share `sh` TMEM columns.
//   dW: output tiles of (2 block slots of 128 rows out of [H blocks..., ONES]) x 256 columns of V, split S ways over the
//       lattice rows.
struct BwdGeom {
    int NP, NCZ, priv, sh, odd_base, dz_stages;
    size_t dz_smem, dw_smem;
    int nVT, nHB, nItems, S_max, dw_grid;     // S_max = the split count S
    bool ok;
};
#ifndef RNNTB200_DZ_EG
#define RNNTB200_DZ_EG 4
#endif
constexpr int RB_DZ_EG = RNNTB200_DZ_EG;      // epilogue warp groups of the dZ kernel (bwd_tc.cuh: DZ_EG)
// dZ kernel variant: 2 (default) = CTA pairs (cta_group::2, one copy of each W stage per two tiles), 1 = one CTA per tile
inline int tc_dz_variant() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("RNNTB200_DZ"); v = e ? atoi(e) : 2; if (v != 1 && v != 2) v = 2; }
    return v;
}
// dW kernel variant: 2 (default) = CTA pairs (one z block per CTA against 512 columns), 1 = one CTA per (2 blocks x 256 columns)
inline int tc_dw_variant() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("RNNTB200_DW"); v = e ? atoi(e) : 2; if (v != 1 && v != 2) v = 2; }
    return v;
}
inline BwdGeom bwd_geometry(int H, int V, int sms = 148, bool dz_pair = true, bool dw_pair = true) {
    BwdGeom g{};
    g.ok = false;
    if (H % 64 || V % 64 || H > 768 || H < 64) return g;
    g.NP = H <= 384 ? 1 : 2;
    g.NCZ = H / g.NP;
    g.sh = 2 * g.NCZ > 512 ? 2 * g.NCZ - 512 : 0;
    g.priv = g.NCZ - g.sh;
    g.odd_base = 512 - g.priv;
    // operand stage: the tile's E' block (16 KB) + the W rows this CTA loads (all NCZ of the pass, or half of them in a pair)
    const size_t dz_stage = 16384 + (size_t)(dz_pair ? g.NCZ / 2 : g.NCZ) * 128;
    for (g.dz_stages = dz_pair ? 6 : 3; g.dz_stages >= 2; --g.dz_stages) {
        g.dz_smem = 1024 + (size_t)g.dz_stages * dz_stage + (size_t)(g.NCZ / 32) * 3072 + (size_t)RB_DZ_EG * 2 * 4 * 8 * 36 * 4 + 512;
        if (g.dz_smem <= 232448) break;
    }
    g.nHB = (H + 127) / 128;
    g.nItems = (g.nHB + 2) / 2;               // blocks [0 .. nHB-1, ONES] in pairs
    if (dw_pair) {                            // a cluster of 2 per (512 columns, item, split): bwd_dw2_kernel
        g.dw_smem = 1024 + (size_t)4 * 49152 + 8 * 256 + 512;
        g.nVT = (V + 511) / 512;
        g.S_max = (sms / 2) / (g.nVT * g.nItems);
        if (g.S_max < 1) g.S_max = 1;
        g.dw_grid = 2 * g.nVT * g.nItems * g.S_max;
    } else {
        g.dw_smem = 1024 + (size_t)3 * 65536 + 8 * 256 + 512;
        g.nVT = (V + 255) / 256;
        g.S_max = sms / (g.nVT * g.nItems);
        if (g.S_max < 1) g.S_max = 1;
        g.dw_grid = g.nVT * g.nItems * g.S_max;
    }
    g.ok = g.dz_smem <= 232448 && g.dw_smem <= 232448;
    return g;
}

struct JointTcParams {
    const float* enc; const float* pred; const float* bias;
    const int* labels; const int* xlen; const int* ylen;
    int B, maxT, maxU, H, V, blank;   // H: the padded width Hp (enc / pred rows as the kernel reads them); V: the REAL vocabulary
    int Vp;                           // ceil64(V): columns of W^T, of the kept rows and of the bias table; v >= V is masked (bias -inf)
    int TT, UU, nTb, nUb, NC, NCH, KB, stages;
    long long SK;
    int b0, nb;                 // utterance range of this launch
    const int* slot;            // tile -> compact row block of the kept arrays (valid tiles only); NULL = tile order
    int nbuf, ks, dbg;          // TMEM accumulator buffers; K-blocks per W stage; bring-up switches
    float* lse; float* lpb; float* lpl;              // outputs (NULL: a recompute that only wants the kept activations)
    // MODE 2 (forward that KEEPS its activations): dl receives the softmax numerators 2^(y - gm) as fp16, one row of V
    // per lattice cell, gm the running maximum each 32-column group was taken against.
    __nv_bfloat16* dl;          // (16-bit storage; the numerators are fp16)
    float* gm;
};
struct TileInfo { int b, t0, u0, Tn, Un; bool valid; };
__device__ __forceinline__ TileInfo decode_tile(const JointTcParams& p, int tile) {
    TileInfo ti;
    const int per_utt = p.nTb * p.nUb;
    const int bl = tile / per_utt, rem = tile - bl * per_utt;
    ti.b = p.b0 + bl;
    ti.t0 = (rem / p.nUb) * p.TT;
    ti.u0 = (rem % p.nUb) * p.UU;
    ti.Tn = p.xlen[ti.b];
    ti.Un = p.ylen[ti.b] + 1;
    ti.valid = ti.t0 < ti.Tn && ti.u0 < ti.Un;
    return ti;
}

// W (H,V) fp32 -> Wt (Vp,Hp) fp16 [B operand of the logits GEMM, K=h] and Wb (Hp,Vp) bf16 [B operand of dZ, K=v], zero
// outside (H, V); grid (Vp / 32, Hp / 32)
__global__ void __launch_bounds__(256) convert_w_kernel(const float* __restrict__ W, __nv_bfloat16* __restrict__ Wt,
                                                        __nv_bfloat16* __restrict__ Wb, int H, int V, int Hp, int Vp) {
    __shared__ float tile[32][33];
    const int v0 = blockIdx.x * 32, h0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
    for (int i = ty; i < 32; i += 8) {
        const int h = h0 + i, v = v0 + tx;
        const float w = (h < H && v < V) ? W[(size_t)h * V + v] : 0.f;
        tile[i][tx] = w;
        if (h < Hp && v < Vp) Wb[(size_t)h * Vp + v] = __float2bfloat16(w);
    }
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        const int v = v0 + i, h = h0 + tx;
        if (h < Hp && v < Vp) reinterpret_cast<__half*>(Wt)[(size_t)v * Hp + h] = __float2half_rn(tile[tx][i]);
    }
}

// H % 64 != 0: enc (rows_e, H) and pred (rows_p, H) -> zero-padded (rows, Hp) copies in the workspace, one launch.  The
// caller's rows cannot be read in place: TMA needs 16-byte row strides and the dZ epilogue adds d_enc as float4.
__global__ void __launch_bounds__(256) stage_rows_kernel(const float* __restrict__ enc, const float* __restrict__ pred,
                                                         float* __restrict__ enc_s, float* __restrict__ pred_s,
                                                         long long rows_e, long long rows_p, int H, int Hp) {
    const long long ne = rows_e * Hp, n = (rows_e + rows_p) * Hp;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const bool is_e = i < ne;
        const long long j = is_e ? i : i - ne, r = j / Hp;
        const int h = (int)(j - r * Hp);
        const float x = h < H ? (is_e ? enc : pred)[r * H + h] : 0.f;
        (is_e ? enc_s : pred_s)[j] = x;
    }
}

// out (rows, H) = the first H columns of src (rows, Hp): d_enc accumulated at the padded width
__global__ void __launch_bounds__(256) narrow_rows_kernel(const float* __restrict__ src, long long rows, int Hp, int H,
                                                          float* __restrict__ out) {
    const long long n = rows * H;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long r = i / H;
        out[i] = src[r * Hp + (i - r * H)];
    }
}

// slot[tile] = rank of the tile among the VALID tiles of this launch (-1 if it lies in the padding); *count = #valid.
// One block; a serial-over-chunks block scan is plenty for the <= ~1e5 tiles of a launch.
__global__ void __launch_bounds__(1024) tile_compact_kernel(const int* __restrict__ xlen, const int* __restrict__ ylen,
                                                            int b0, int ntiles, int nTb, int nUb, int TT, int UU,
                                                            int* __restrict__ slot, int* __restrict__ count,
                                                            int* __restrict__ tile_of_slot = nullptr,
                                                            int4* __restrict__ slot_meta = nullptr, int maxT = 0, int maxU = 0,
                                                            int max_slots = 0x7fffffff) {
    __shared__ int warp_sums[32];
    __shared__ int base;
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    const int per_utt = nTb * nUb, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int t0 = 0; t0 < ntiles; t0 += 1024) {
        const int tile = t0 + threadIdx.x;
        int v = 0;
        int4 meta = make_int4(0, 0, 1, 1);
        if (tile < ntiles) {
            const int bl = tile / per_utt, rem = tile - bl * per_utt, b = b0 + bl;
            const int tt = (rem / nUb) * TT, uu = (rem % nUb) * UU;
            v = (tt < xlen[b] && uu < ylen[b] + 1) ? 1 : 0;
            // what the kernels that walk the compact slots need of a tile, so that none of them divides: first enc / pred row
            // (in rows of H floats) and how many of the tile's TT / UU rows exist in the padded arrays
            meta = make_int4(b * maxT + tt, b * maxU + uu, min(TT, maxT - tt), min(UU, maxU - uu));
        }
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int n = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += n; }
        if (lane == 31) warp_sums[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            int w = warp_sums[lane], wi = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int n = __shfl_up_sync(0xffffffffu, wi, o); if (lane >= o) wi += n; }
            warp_sums[lane] = wi - w;   // exclusive prefix of the warp totals
        }
        __syncthreads();
        const int excl = base + warp_sums[warp] + incl - v;
        if (tile < ntiles) {
            // a valid tile beyond the row blocks the workspace holds (the caller's valid_tile_bound was too small) gets no slot:
            // nothing is stored for it, the overflow word is raised and the forward call poisons the costs
            const bool fits = excl < max_slots;
            slot[tile] = (v && fits) ? excl : -1;
            if (v && fits && tile_of_slot) tile_of_slot[excl] = tile;
            if (v && fits && slot_meta) slot_meta[excl] = meta;
        }
        __syncthreads();
        if (threadIdx.x == 1023) base = excl + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        count[0] = min(base, max_slots);
        count[1] = base > max_slots ? base : 0;        // overflow word: the number of valid tiles found
        if (base > max_slots)
            printf("rnnt_b200: %d lattice tiles are valid but rnntb200JointDesc.valid_tile_bound promised at most %d -- results are invalid\n",
                   base, max_slots);
    }
}
// out = sum_k part[k] over `nplanes` planes of `n4` float4 each; a plane is (rows, 4 * cols4) and out receives its
// window (rows_out, cols_out) -- the real (H, V) of a padded (Hp, Vp) plane -- as a dense row-major array
__global__ void __launch_bounds__(256) sum_planes_kernel(const float4* __restrict__ part, int nplanes, size_t n4,
                                                         float* __restrict__ out, int rows_out, int cols4, int cols_out) {
    const bool whole = cols_out == 4 * cols4 && (size_t)rows_out * cols4 == n4;      // aligned: the window is the whole plane
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
        size_t r = 0;
        int c = 0;
        if (!whole) {
            r = i / cols4;
            c = (int)(i - r * cols4) * 4;
            if (r >= (size_t)rows_out || c >= cols_out) continue;
        }
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
        for (int k = 0; k < nplanes; ++k) {
            const float4 v = part[(size_t)k * n4 + i];
            acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
        if (whole) {
            reinterpret_cast<float4*>(out)[i] = acc;
        } else {
            float* o = out + r * cols_out + c;
            o[0] = acc.x;
            if (c + 1 < cols_out) o[1] = acc.y;
            if (c + 2 < cols_out) o[2] = acc.z;
            if (c + 3 < cols_out) o[3] = acc.w;
        }
    }
}
// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline PFN_encodeTiled get_encode_fn() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_encodeTiled>(p);
    }
    return fn;
}
// 2-D row-major bf16 matrix [rows x cols] (cols contiguous), box [box_rows x 64 cols], SWIZZLE_128B
inline bool make_tmap_bf16(CUtensorMap* tm, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows,
                           uint32_t box_cols = 64) {
    PFN_encodeTiled fn = get_encode_fn();
    if (!fn) return false;
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {cols * 2};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    return fn(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// W^T (V,H) bf16 viewed as 3-D (k within a 64-wide K block, v, K block): one request brings `kblocks` K-major
// SWIZZLE_128B slabs [box_rows x 64] that land back to back in shared memory.
inline bool make_tmap_bf16_kblocks(CUtensorMap* tm, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows,
                                   uint32_t kblocks) {
    PFN_encodeTiled fn = get_encode_fn();
    if (!fn) return false;
    cuuint64_t dims[3] = {64, rows, cols / 64};
    cuuint64_t strides[2] = {cols * 2, 128};
    cuuint32_t box[3] = {64, box_rows, kblocks};
    cuuint32_t estr[3] = {1, 1, 1};
    return fn(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// 2-D row-major fp32 matrix [rows x cols], box [box_rows x box_cols]; swizzle128 requires box_cols*4 == 128
inline bool make_tmap_f32(CUtensorMap* tm, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows,
                          uint32_t box_cols, bool swizzle128) {
    PFN_encodeTiled fn = get_encode_fn();
    if (!fn) return false;
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {cols * 4};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    return fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Workspace of the tensor-core path (a pure function of the descriptor).  The kept arrays (numerators + maxima) are
// laid out per 128-row tile; the batch is processed in utterance chunks that keep them under ~16 GiB.  Every size below is
// that of the padded problem (Hp, Vp) = (ceil64(H), ceil64(V)); the three staged arrays at the end exist only when H != Hp,
// so an aligned descriptor has exactly the layout it always had.
struct TcScratch {
    __nv_bfloat16 *Wt, *Wb;                 // W^T (Vp,Hp) fp16 [forward B operand, 16-bit storage] and W (Hp,Vp) bf16 [dZ B operand]
    __nv_bfloat16* dl;                      // (rows_chunk, Vp) bf16 softmax numerators E = 2^(y - ref_row)
    float* gm;                              // (rows_chunk) fp32 reference of each row's numerators (log2 domain)
    int* slot;                              // tile -> compact row block (-1: outside the valid lattice), per chunk
    int* tile_of_slot;                      // compact row block -> tile
    int4* slot_meta;                        // compact row block -> {first enc row, first pred row, #t rows, #u rows} (tile_compact_kernel)
    int* count;                             // number of valid tiles of the chunk
    float* ppl;                             // (nTb, bchunk, maxU, H) fp32 partial planes of d_pred (bwd_dz_kernel)
    float* dWp;                             // (S_max, H, V) fp32 split-K planes of dW (bwd_dw_kernel)
    float* dbp;                             // (S_max, V) planes of db
    float* rowscale;                        // (rows_chunk) per-row scale of the logit gradients (row_scale_kernel)
    float *enc_s, *pred_s;                  // H != Hp only: (B*maxT, Hp) / (B*maxU, Hp) zero-padded copies of enc / pred
    float* denc_s;                          // H != Hp only: (B*maxT, Hp) d_enc at the padded width, narrowed at the end
    int bchunk;                             // utterances per chunk
    size_t rows_chunk;                      // bchunk * tiles_per_utt * 128
    size_t bytes;
};
// bytes of kept activations per utterance chunk: 16 GiB (RNNTB200_CHUNK_MB overrides it for the tests of the
// multi-chunk backward; read once per process, so the workspace size stays a pure function of the descriptor)
inline size_t tc_chunk_budget() {
    static size_t v = 0;
    if (!v) { const char* e = getenv("RNNTB200_CHUNK_MB"); v = e && atoll(e) > 0 ? (size_t)atoll(e) << 20 : (size_t)16 << 30; }
    return v;
}
inline TcScratch tc_scratch_layout(const rnntb200JointDesc& desc, void* base) {
    TcScratch s{};
    const rnntb200JointDesc d = tc_padded(desc);
    const TcGeom g = tc_geometry(d.maxT, d.maxU, d.H, d.V);
    const BwdGeom bg = bwd_geometry(d.H, d.V, 148, tc_dz_variant() == 2, tc_dw_variant() == 2);
    const size_t rows_utt = (size_t)g.nTb * g.nUb * 128;
    const size_t per_row = (size_t)d.V * 2 + 8;
    size_t bc = tc_chunk_budget() / (rows_utt * per_row);
    if (bc < 1) bc = 1;
    if (bc > (size_t)d.B) bc = d.B;
    s.bchunk = (int)bc;
    s.rows_chunk = bc * rows_utt;
    // The kept arrays are indexed by COMPACT slots (valid tiles only), but how many tiles are valid is known to the device
    // alone, so the default sizes them for every tile of the padded (maxT, maxU) lattice and chunks the batch.  A caller
    // that knows its lengths on the host can promise an upper bound: the whole batch is then ONE chunk of that many row
    // blocks (C5: 46 k valid of 160 k padded tiles -- keep mode instead of 11 recomputing chunks).
    if (d.valid_tile_bound > 0 && bc < (size_t)d.B) {
        const size_t tiles = (size_t)d.valid_tile_bound < (size_t)d.B * g.nTb * g.nUb ? (size_t)d.valid_tile_bound : (size_t)d.B * g.nTb * g.nUb;
        if (tiles * 128 * per_row <= ((size_t)160 << 30)) { bc = d.B; s.bchunk = d.B; s.rows_chunk = tiles * 128; }
    }
    char* p = static_cast<char*>(base);
    auto take = [&](size_t n) { char* r = p; p += (n + 255) / 256 * 256; return r; };
    s.Wt = reinterpret_cast<__nv_bfloat16*>(take((size_t)d.V * d.H * 2));
    s.Wb = reinterpret_cast<__nv_bfloat16*>(take((size_t)d.V * d.H * 2));
    s.dl = reinterpret_cast<__nv_bfloat16*>(take(s.rows_chunk * d.V * 2));
    s.gm = reinterpret_cast<float*>(take(s.rows_chunk * 4));
    s.slot = reinterpret_cast<int*>(take((size_t)bc * g.nTb * g.nUb * 4));
    s.tile_of_slot = reinterpret_cast<int*>(take((size_t)bc * g.nTb * g.nUb * 4));
    s.slot_meta = reinterpret_cast<int4*>(take((size_t)bc * g.nTb * g.nUb * 16));
    s.count = reinterpret_cast<int*>(take(256));
    s.ppl = reinterpret_cast<float*>(take((size_t)g.nTb * bc * d.maxU * d.H * 4));
    s.dWp = reinterpret_cast<float*>(take((size_t)bg.S_max * d.H * d.V * 4));
    s.dbp = reinterpret_cast<float*>(take((size_t)bg.S_max * d.V * 4));
    s.rowscale = reinterpret_cast<float*>(take(s.rows_chunk * 4));
    if (desc.H != d.H) {
        s.enc_s = reinterpret_cast<float*>(take((size_t)d.B * d.maxT * d.H * 4));
        s.pred_s = reinterpret_cast<float*>(take((size_t)d.B * d.maxU * d.H * 4));
        s.denc_s = reinterpret_cast<float*>(take((size_t)d.B * d.maxT * d.H * 4));
    }
    s.bytes = (size_t)(p - static_cast<char*>(base));
    return s;
}

inline rnntStatus_t tc_unsupported(const rnntb200JointDesc& d) {
    fprintf(stderr,
            "rnnt_b200: RNNTB200_BF16_TC supports joint widths H <= 768 (got H=%d); use RNNTB200_FP32_EXACT\n", d.H);
    return RNNT_STATUS_INVALID_VALUE;
}

inline bool tc_fill_params(const rnntb200JointDesc& d, const TcGeom& g, JointTcParams& p, const float* enc,
                           const float* pred, const float* bias, const int* labels, const int* ylen,
                           const int* xlen) {
    p = JointTcParams{};
    p.enc = enc; p.pred = pred; p.bias = bias; p.labels = labels; p.xlen = xlen; p.ylen = ylen;
    p.B = d.B; p.maxT = d.maxT; p.maxU = d.maxU; p.H = tc_pad64(d.H); p.V = d.V; p.Vp = tc_pad64(d.V); p.blank = d.blank_label;
    p.TT = g.TT; p.UU = g.UU; p.nTb = g.nTb; p.nUb = g.nUb; p.KB = g.KB;
    p.SK = (long long)(d.maxT + d.maxU - 1) * d.maxU;
    return true;
}

// RNNTB200_DBG=<bits>: switch kernel roles off for timing experiments (results are wrong by design)
inline int tc_dbg() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("RNNTB200_DBG"); v = e ? atoi(e) : 0; }
    return v;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-DEVICE property of a kernel: set it once per (device, kernel),
// thread-safe (the library may be driven from several host threads / several devices of one process).
inline bool tc_smem_optin(const void* func) {
    static std::mutex mu;
    static std::unordered_map<unsigned long long, bool> done;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return false;
    const unsigned long long key = (unsigned long long)reinterpret_cast<uintptr_t>(func) * 64ull + (unsigned long long)dev;
    std::lock_guard<std::mutex> lk(mu);
    auto it = done.find(key);
    if (it != done.end()) return true;
    if (cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448) != cudaSuccess) return false;
    done[key] = true;
    return true;
}

}  // namespace rb

#include "joint_tc3.cuh"
#include "joint_tc4.cuh"
#include "bwd_tc.cuh"

namespace rb {

// RNNTB200_PROF=1 (bring-up): the backward kernels record per-role wait cycles into a managed buffer that
// rnntb200_debug_prof() exposes (tools/role_profile.py); off by default, never touched otherwise.
inline long long* tc_prof_buffer(int which) {
    static long long* buf[2] = {nullptr, nullptr};
    static int on = -1;
    if (on < 0) { const char* e = getenv("RNNTB200_PROF"); on = e ? atoi(e) : 0; }
    if (!on) return nullptr;
    if (!buf[which]) {
        if (cudaMallocManaged(reinterpret_cast<void**>(&buf[which]), sizeof(long long) * 256 * 4 * 8) != cudaSuccess) return nullptr;
        cudaMemset(buf[which], 0, sizeof(long long) * 256 * 4 * 8);
    }
    return buf[which];
}

// 1 <= H <= 768 and V >= 1: the geometries are those of the padded problem
inline bool tc_supported(const rnntb200JointDesc& desc) {
    if (desc.H < 1 || desc.H > 768 || desc.V < 1) return false;
    const rnntb200JointDesc d = tc_padded(desc);
    return tc_geometry(d.maxT, d.maxU, d.H, d.V).ok && tc3_geometry(d.H, d.V).ok && bwd_geometry(d.H, d.V, 148, tc_dz_variant() == 2, tc_dw_variant() == 2).ok;
}
inline size_t tc_scratch_bytes(const rnntb200JointDesc& d) {
    if (!tc_supported(d)) return 0;
    return tc_scratch_layout(d, nullptr).bytes;
}

// keep_activations is honoured when the whole batch is one workspace chunk (RNNTB200_KEEP=0 turns it off for A/B
// measurements); otherwise the backward re-runs the keeping forward chunk by chunk.
inline bool tc_keep(const rnntb200JointDesc& d, const TcScratch& sc) {
    static int env = -1;
    if (env < 0) { const char* e = getenv("RNNTB200_KEEP"); env = e ? atoi(e) : 1; }
    return d.keep_activations && env && sc.bchunk >= d.B;
}

// RNNTB200_FWD=3|4: forward kernel generation (4 = CTA pairs, the default; 3 = one CTA per tile, kept for A/B measurements)
inline int tc_fwd_variant() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("RNNTB200_FWD"); v = e ? atoi(e) : 4; if (v != 3 && v != 4) v = 4; }
    return v;
}

// the forward kernel over utterances [b0, b0+nb); KEEP: rank the chunk's valid tiles on the device (nothing is read
// back) and leave numerators + maxima in the workspace
template <bool KEEP>
inline rnntStatus_t tc_run_forward(const rnntb200JointDesc& d, const TcGeom& g, const TcScratch& sc, const float* enc,
                                   const float* pred, const float* bias, const int* labels, const int* ylen,
                                   const int* xlen, float* lse, float* lpb, float* lpl, int b0, int nb, cudaStream_t s,
                                   unsigned* launches) {
    const bool pair = tc_fwd_variant() == 4;             // CTA-pair kernel (joint_tc4.cuh) or one CTA per tile (joint_tc3.cuh)
    const int Hp = tc_pad64(d.H), Vp = tc_pad64(d.V);    // enc / pred are (rows, Hp) here: the caller's or the staged copies
    const Tc2Geom g3 = pair ? tc4_geometry(Hp, Vp) : tc3_geometry(Hp, Vp);
    JointTcParams p;
    tc_fill_params(d, g, p, enc, pred, bias, labels, ylen, xlen);
    p.b0 = b0; p.nb = nb;
    p.lse = lse; p.lpb = lpb; p.lpl = lpl;
    p.NC = TC2_NC; p.NCH = Vp / TC2_NC; p.stages = g3.stages; p.nbuf = g3.nbuf; p.ks = g3.ks;
    p.dbg = tc_dbg();
    if (KEEP) {
        const int ntiles = nb * g.nTb * g.nUb;
        tile_compact_kernel<<<1, 1024, 0, s>>>(xlen, ylen, b0, ntiles, g.nTb, g.nUb, g.TT, g.UU, sc.slot, sc.count, sc.tile_of_slot, sc.slot_meta,
                                             d.maxT, d.maxU, (int)(sc.rows_chunk / 128));
        *launches += 1;
        p.slot = sc.slot; p.dl = sc.dl; p.gm = sc.gm;
    }
    CUtensorMap tm, tmp, tme;
    if (!make_tmap_bf16_kblocks(&tm, sc.Wt, Vp, Hp, pair ? TC2_NC / 2 : TC2_NC, g3.ks) ||
        !make_tmap_f32(&tmp, pred, (uint64_t)d.B * d.maxU, Hp, g.UU, 32, true) ||
        !make_tmap_f32(&tme, enc, (uint64_t)d.B * d.maxT, Hp, g.TT, 64, false)) {
        fprintf(stderr, "rnnt_b200: cuTensorMapEncodeTiled failed\n");
        return RNNT_STATUS_EXECUTION_FAILED;
    }
    *launches += 1;
    if (pair) return tc4_launch<KEEP ? 2 : 0>(g3, tm, tmp, tme, p, s);
    return tc3_launch<KEEP ? 2 : 0>(g3, tm, tmp, tme, p, s);
}

inline rnntStatus_t tc_forward(const rnntb200JointDesc& d, void* scratch, const float* enc, const float* pred,
                               const float* W, const float* bias, const int* labels, const int* ylen,
                               const int* xlen, float* lse, float* lpb, float* lpl, cudaStream_t s,
                               unsigned* launches) {
    if (!tc_supported(d)) return tc_unsupported(d);
    const rnntb200JointDesc dp = tc_padded(d);
    const TcGeom g = tc_geometry(dp.maxT, dp.maxU, dp.H, dp.V);
    TcScratch sc = tc_scratch_layout(d, scratch);
    convert_w_kernel<<<dim3(dp.V / 32, dp.H / 32), 256, 0, s>>>(W, sc.Wt, sc.Wb, d.H, d.V, dp.H, dp.V);
    *launches += 1;
    if (dp.H != d.H) {      // the backward reads these copies too (it follows the forward with the same workspace)
        const long long re = (long long)d.B * d.maxT, rp = (long long)d.B * d.maxU, n = (re + rp) * dp.H;
        stage_rows_kernel<<<(unsigned)((n + 255) / 256 < 4096 ? (n + 255) / 256 : 4096), 256, 0, s>>>(enc, pred, sc.enc_s, sc.pred_s,
                                                                                                   re, rp, d.H, dp.H);
        *launches += 1;
        enc = sc.enc_s;
        pred = sc.pred_s;
    }
    if (tc_keep(d, sc))
        return tc_run_forward<true>(d, g, sc, enc, pred, bias, labels, ylen, xlen, lse, lpb, lpl, 0, d.B, s, launches);
    return tc_run_forward<false>(d, g, sc, enc, pred, bias, labels, ylen, xlen, lse, lpb, lpl, 0, d.B, s, launches);
}

struct LossPlanes { const float *lse, *lpb, *lpl, *alphas, *betas, *llf; };   // outputs of the forward + alpha/beta (loss workspace)

// Backward (SURVEY 8 a19) with the library's own tcgen05 kernels (bwd_tc.cuh).  Per utterance chunk: (a keeping
// forward of the chunk unless the forward call already kept the whole batch) -> bwd_dz_kernel -> d_pred plane sum ->
// bwd_dw_kernel; after the last chunk the split-K planes of dW / db are summed.  Stream-ordered, no host
// synchronisation, no library calls.
inline rnntStatus_t tc_backward(const rnntb200JointDesc& d, void* scratch, const float* enc, const float* pred,
                                const float* bias, const int* labels, const int* ylen, const int* xlen,
                                const LossPlanes& lp, const float* grad_costs, float* d_enc, float* d_pred, float* dW,
                                float* db, cudaStream_t s, unsigned* launches) {
    if (!tc_supported(d)) return tc_unsupported(d);
    const rnntb200JointDesc dp = tc_padded(d);
    const int Hp = dp.H, Vp = dp.V;
    const TcGeom g = tc_geometry(dp.maxT, dp.maxU, Hp, Vp);
    const bool dz_pair = tc_dz_variant() == 2, dw_pair = tc_dw_variant() == 2;
    const BwdGeom bg = bwd_geometry(Hp, Vp, 148, dz_pair, dw_pair);
    TcScratch sc = tc_scratch_layout(d, scratch);   // Wt / Wb (and for H != Hp the staged enc / pred) were produced by the forward call
    const bool kept = tc_keep(d, sc);
    float* d_enc_out = d_enc;
    if (Hp != d.H) { enc = sc.enc_s; pred = sc.pred_s; d_enc = sc.denc_s; }
    if (!tc_smem_optin(reinterpret_cast<const void*>(bwd_dz_kernel<false, false>)) || !tc_smem_optin(reinterpret_cast<const void*>(bwd_dz_kernel<true, false>)) ||
        !tc_smem_optin(reinterpret_cast<const void*>(bwd_dz_kernel<false, true>)) || !tc_smem_optin(reinterpret_cast<const void*>(bwd_dz_kernel<true, true>)) ||
        !tc_smem_optin(reinterpret_cast<const void*>(bwd_dw_kernel<false>)) || !tc_smem_optin(reinterpret_cast<const void*>(bwd_dw_kernel<true>)) ||
        !tc_smem_optin(reinterpret_cast<const void*>(bwd_dw2_kernel<false>)) || !tc_smem_optin(reinterpret_cast<const void*>(bwd_dw2_kernel<true>)))
        return RNNT_STATUS_EXECUTION_FAILED;
    if (cudaMemsetAsync(sc.dWp, 0, sizeof(float) * (size_t)bg.S_max * Hp * Vp, s) != cudaSuccess ||
        cudaMemsetAsync(sc.dbp, 0, sizeof(float) * (size_t)bg.S_max * Vp, s) != cudaSuccess)
        return RNNT_STATUS_MEMOPS_FAILED;
    CUtensorMap tm_e128, tm_e64, tm_wp, tm_ws, tm_p32, tm_e32;
    if (!make_tmap_f32(&tm_p32, pred, (uint64_t)d.B * d.maxU, Hp, BW_UU, 32, true) ||
        !make_tmap_f32(&tm_e32, enc, (uint64_t)d.B * d.maxT, Hp, BW_TT, 32, false) ||
        !make_tmap_bf16(&tm_e128, sc.dl, sc.rows_chunk, Vp, 128) || !make_tmap_bf16(&tm_e64, sc.dl, sc.rows_chunk, Vp, 64) ||
        !make_tmap_bf16(&tm_wp, sc.Wb, Hp, Vp, dz_pair ? bg.priv / 2 : bg.priv) ||
        !make_tmap_bf16(&tm_ws, sc.Wb, Hp, Vp, bg.sh ? (dz_pair ? bg.sh / 2 : bg.sh) : 8)) {
        fprintf(stderr, "rnnt_b200: cuTensorMapEncodeTiled failed\n");
        return RNNT_STATUS_EXECUTION_FAILED;
    }
    const int sms = tc_num_sms();
    for (int b0 = 0; b0 < d.B; b0 += sc.bchunk) {
        const int nb = (d.B - b0 < sc.bchunk) ? d.B - b0 : sc.bchunk;
        if (!kept) {
            rnntStatus_t st = tc_run_forward<true>(d, g, sc, enc, pred, bias, labels, ylen, xlen, nullptr, nullptr, nullptr, b0, nb, s, launches);
            if (st) return st;
        }
        BwdParams p{};
        p.enc = enc; p.pred = pred; p.xlen = xlen; p.ylen = ylen;
        p.maxT = d.maxT; p.maxU = d.maxU; p.H = Hp; p.V = Vp;
        p.nTb = g.nTb; p.nUb = g.nUb; p.b0 = b0; p.nb = nb;
        {   // per-row scales of this chunk (row order of the kept arrays) + the two special columns of every row
            ScopedTimer tmr("row_scale_kernel", s);
            row_scale_kernel<<<(unsigned)(((size_t)nb * g.nTb * g.nUb * 128 + 255) / 256), 256, 0, s>>>(
                sc.tile_of_slot, sc.count, b0, g.nTb, g.nUb, xlen, ylen, labels, d.blank_label, d.maxT, d.maxU,
                (long long)(d.maxT + d.maxU - 1) * d.maxU, lp.lse, lp.lpb, lp.lpl, lp.alphas, lp.betas, lp.llf, grad_costs, sc.gm,
                Vp, reinterpret_cast<unsigned short*>(sc.dl), sc.rowscale);
            *launches += 1;
        }
        p.slot = sc.slot; p.tile_of_slot = sc.tile_of_slot; p.slot_meta = sc.slot_meta; p.count = sc.count; p.rowscale = sc.rowscale;
        p.NP = bg.NP; p.NCZ = bg.NCZ; p.priv = bg.priv; p.sh = bg.sh; p.odd_base = bg.odd_base; p.dz_stages = bg.dz_stages;
        p.d_enc = d_enc; p.ppred = sc.ppl;
        p.nVT = bg.nVT; p.nItems = bg.nItems; p.nHB = bg.nHB; p.S = bg.S_max; p.Hrows = Hp;
        p.dWp = sc.dWp; p.dbp = sc.dbp;
        long long* prof_dz = tc_prof_buffer(0), *prof_dw = tc_prof_buffer(1);
        // rows of d_enc whose t-block lies outside the utterance are never visited by the dZ kernel
        if (cudaMemsetAsync(d_enc + (size_t)b0 * d.maxT * Hp, 0, sizeof(float) * (size_t)nb * d.maxT * Hp, s) != cudaSuccess)
            return RNNT_STATUS_MEMOPS_FAILED;
        {
            const int nruns = nb * g.nTb;
            ScopedTimer tmr("bwd_dz_kernel", s);
            p.prof = prof_dz;
            if (dz_pair) {
                const int npairs = nruns < sms / 2 ? nruns : sms / 2;
                cudaLaunchConfig_t cfg{};
                cfg.gridDim = dim3(2 * npairs); cfg.blockDim = dim3(DZ_THREADS); cfg.dynamicSmemBytes = bg.dz_smem; cfg.stream = s;
                cudaLaunchAttribute at[1];
                at[0].id = cudaLaunchAttributeClusterDimension;
                at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
                cfg.attrs = at; cfg.numAttrs = 1;
                if (cudaLaunchKernelEx(&cfg, p.prof ? bwd_dz_kernel<true, true> : bwd_dz_kernel<false, true>, tm_e128, tm_wp, tm_ws, tm_p32,
                                       tm_e32, p) != cudaSuccess)
                    return RNNT_STATUS_EXECUTION_FAILED;
            } else if (p.prof) bwd_dz_kernel<true, false><<<nruns < sms ? nruns : sms, DZ_THREADS, bg.dz_smem, s>>>(tm_e128, tm_wp, tm_ws, tm_p32, tm_e32, p);
            else bwd_dz_kernel<false, false><<<nruns < sms ? nruns : sms, DZ_THREADS, bg.dz_smem, s>>>(tm_e128, tm_wp, tm_ws, tm_p32, tm_e32, p);
        }
        {
            const size_t n4 = (size_t)nb * d.maxU * Hp / 4;
            ScopedTimer tmr("sum_pred_planes_kernel", s);
            sum_pred_planes_kernel<<<(unsigned)((n4 + 255) / 256 < 4096 ? (n4 + 255) / 256 : 4096), 256, 0, s>>>(
                reinterpret_cast<const float4*>(sc.ppl), xlen, ylen, b0, nb, d.maxU, Hp / 4, d.H, d_pred);
        }
        {
            ScopedTimer tmr(dw_pair ? "bwd_dw2_kernel" : "bwd_dw_kernel", s);
            p.prof = prof_dw;
            if (dw_pair) {
                if (p.prof) bwd_dw2_kernel<true><<<bg.dw_grid, DW_THREADS, bg.dw_smem, s>>>(tm_e64, p);
                else bwd_dw2_kernel<false><<<bg.dw_grid, DW_THREADS, bg.dw_smem, s>>>(tm_e64, p);
            } else if (p.prof) bwd_dw_kernel<true><<<bg.dw_grid, DW_THREADS, bg.dw_smem, s>>>(tm_e64, p);
            else bwd_dw_kernel<false><<<bg.dw_grid, DW_THREADS, bg.dw_smem, s>>>(tm_e64, p);
        }
        *launches += 3;
        if (cudaGetLastError() != cudaSuccess) return RNNT_STATUS_EXECUTION_FAILED;
    }
    {
        ScopedTimer tmr("sum_planes_kernel", s);
        const size_t nw4 = (size_t)Hp * Vp / 4, nb4 = (size_t)Vp / 4;
        sum_planes_kernel<<<(unsigned)((nw4 + 255) / 256 < 4096 ? (nw4 + 255) / 256 : 4096), 256, 0, s>>>(
            reinterpret_cast<const float4*>(sc.dWp), bg.S_max, nw4, dW, d.H, Vp / 4, d.V);
        sum_planes_kernel<<<(unsigned)((nb4 + 255) / 256), 256, 0, s>>>(reinterpret_cast<const float4*>(sc.dbp), bg.S_max, nb4,
                                                                       db, 1, Vp / 4, d.V);
    }
    *launches += 2;
    if (Hp != d.H) {
        const long long n = (long long)d.B * d.maxT * d.H;
        narrow_rows_kernel<<<(unsigned)((n + 255) / 256 < 4096 ? (n + 255) / 256 : 4096), 256, 0, s>>>(sc.denc_s, (long long)d.B * d.maxT,
                                                                                                    Hp, d.H, d_enc_out);
        *launches += 1;
    }
    return cudaGetLastError() == cudaSuccess ? RNNT_STATUS_SUCCESS : RNNT_STATUS_EXECUTION_FAILED;
}

}  // namespace rb
