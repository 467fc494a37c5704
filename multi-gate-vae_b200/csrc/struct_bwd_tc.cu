// Struct encoder BACKWARD on the 5th-generation tensor cores (the forward is struct_tc.cu): MultiGCNEncoder.forward
// (digae_layer.py:257-277) with AggConv (arch/gcn_conv.py:30-42) differentiated step by step in reverse.  Per half-round
// step k = 2R .. 1 two kernels, 128-node tiles, fp16 hi/lo planes with fp32 accumulation in tensor memory:
//
//   struct_bwd_pw_kernel   (persistent, weights resident, warp-specialised like the forward)
//     tile     [agg | h | x deg 1] operand tile of state_{k-1}: bulk copy of the tile the FORWARD saved (no second gather)
//     gather   d state_k = part + sum of the neighbours' d agg_{k+1}
//     MMA      recompute the GRU pre-activations (identical products to the forward)            -> TMEM columns 0..255
//     epilogue thread = node: gates, LayerNorm backward, GRU backward; d gates (d r, d z, d gi_n, d gh_n) go back into
//              the SAME tensor-memory columns, first as fp32, then -- scaled by the tile's power of two -- as fp16 hi/lo
//              planes (16 gates = 8 + 8 packed columns), which is the A operand of
//     MMA      d agg = d gi Wc,  d part = d gh Whh   (A from tensor memory, B = the forward's weight image read MN-major)
//     epilogue d agg / d part -> HBM for step k-1; d ln_w / d ln_b partial sums live in tensor memory per thread
//     The d-gate planes also go to HBM for
//   struct_bwd_wgrad_kernel (persistent, streaming): d W^T-free weight gradient  d Wcx | d Whh | d b  +=  d gates^T [agg | h | x deg 1]
//     both operands MN-major straight from bulk-copied planes (d gates from the kernel above, operand tiles from the
//     forward), K = nodes, accumulators persistent in tensor memory
//     (2 x 144 columns at a 160-column stride) over all tiles of the CTA, flushed once into the CTA's private partial block.
//
// Shared memory cannot hold weights (112 KB) + operand tile (72 KB) + d-gate planes (128 KB) and tensor memory cannot hold
// recompute (256) + data-gradient (128) + weight-gradient (288) columns, hence the split; the hand-off buffers are
// processed in chunks of tiles so they stay L2-sized.
#include <stdlib.h>
#include "struct_layout.cuh"

long long* mgv_debug_trace();
size_t mgv_struct_image_bytes(int num_enc);
int mgv_struct_build_image(const float* weights, int num_enc, uint8_t* image, int precision, cudaStream_t st);

namespace {
using namespace struct_layout;

constexpr int SGRAD = MGV_STRUCT_GRAD_FLOATS;
constexpr int EPI_WARPS = 8, GATHER_WARPS = 8;              // epilogue: 2 warps per 32 TMEM lanes (32 units each); gather: 4 rows per lane
constexpr int THREADS = (EPI_WARPS + GATHER_WARPS + 1) * 32; // + the MMA / bulk-copy warp: 17 warps, 5 on one scheduler -> 96 registers
constexpr int LDGS = 68;                                   // d state staging row stride (floats)
constexpr uint32_t DG_TILE_BYTES = 131072;                 // [hi | lo][64-node half][8-gate chunk (32)][node row (64)][16 B]: no-swizzle core matrices
constexpr int CHUNK_TILES_DEFAULT = 2048;                  // tiles per encoder per kernel pair (MGV_STRUCT_CHUNK overrides: tuning)

// ---- shared memory of the pointwise kernel (after the weight image and the operand tile, struct_layout.cuh)
constexpr uint32_t S_G = A_X_LO + 4096;                    // d state_k staging, fp32 [128][LDGS]
constexpr uint32_t S_LN = S_G + TM * LDGS * 4;             // ln_w, ln_b
constexpr uint32_t S_AMAX = S_LN + 512;                    // 3 rotating tile-amax words
constexpr uint32_t S_EX = S_AMAX + 16;                     // row sums exchanged between the two epilogue warps of a row: [4][2][128]
constexpr uint32_t S_BAR = S_EX + 4 * 2 * TM * 4;          // 6 mbarriers
constexpr uint32_t S_TMEM = S_BAR + 128;
constexpr uint32_t P_SMEM = S_TMEM + 64 + 1024;            // + alignment slack
static_assert(P_SMEM <= 227 * 1024, "struct backward: shared memory");
static_assert(A_TILE_BYTES + TM * LDGS * 4 >= TM * 132 * 4, "LayerNorm gradient scratch aliases the tile + staging");
// tensor memory columns
constexpr uint32_t T_ACC = 0, T_OUT = 256, T_LNP = 384;

struct BwdTC {
    int N, feat, layernorm, first, last, dir;
    int tile_beg, tile_end;    // this launch's chunk of tiles
    const int* ptr;            // neighbour CSR of this step's direction
    const int* idx;
    const int* order;
    const int* gdesc;
    const unsigned* tile_cost;
    const float* x;
    const uint8_t* image;      // weight image of (enc 0, this dir); encoder stride 2 * IMG_BYTES
    const float* gout;         // [enc][N][64]
    const float* in_part; const float* in_agg;
    float* out_part; float* out_agg;
    const uint8_t* tiles;      // operand tiles saved by the forward for this step, enc 0: [tile][A_TILE_BYTES]
    size_t tiles_enc_stride;   // bytes between encoders
    uint8_t* dgbuf;            // [enc][chunk tiles][DG_TILE_BYTES]
    float* scales;             // [enc][chunk tiles]
    unsigned* smin;            // [enc] min of the chunk's tile scales (float bits)
    float* partial;            // [enc][gxp][2][SGRAD]
    int gxp;
    int chunk_cap;             // tiles per encoder the hand-off buffers are sized for
    long long* trace;
};
#define PTRACE_MAX(slot) do { if (p.trace && it < 16) atomicMax(reinterpret_cast<unsigned long long*>(p.trace) + (((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 16 + it) * 16 + (slot), (unsigned long long)clock64()); } while (0)
#define PTRACE(slot) do { if (p.trace && it < 16) p.trace[(((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 16 + it) * 16 + (slot)] = clock64(); } while (0)

__device__ __forceinline__ float4 lds4(const float* p) { return *reinterpret_cast<const float4*>(p); }
// Power of two s with amax * s in [2^8, 2^9) (amax > 0), else 1.
__device__ __forceinline__ float pow2_scale(float amax) {
    if (!(amax > 0.f) || !isfinite(amax)) return 1.0f;
    const int e = (int)((__float_as_uint(amax) >> 23) & 0xff) - 127;
    int k = 8 - e;
    k = k < -100 ? -100 : (k > 100 ? 100 : k);
    return __uint_as_float((uint32_t)(k + 127) << 23);
}
__device__ __forceinline__ float pow2_scale_keep(float amax, float cur) {
    const float v = amax * cur;
    if (v >= 4.0f && v <= 8192.0f) return cur;
    return (amax > 0.f) ? pow2_scale(amax) : cur;
}

// ======================================================================================= recompute + pointwise + data gradient
// LOWP = bf16 mode: one plane of bf16 operands everywhere (the forward saved only the hi planes of its tiles), single products,
// no tile scale (bf16 has the fp32 exponent range), half the hand-off bytes.
template <bool LOWP>
__global__ void __launch_bounds__(THREADS, 1) struct_bwd_pw_kernel(const BwdTC p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const uint32_t sbase = (tc::smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* sgen = smem_raw + (sbase - tc::smem_u32(smem_raw));
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int enc = blockIdx.y;
    const size_t eoff = (size_t)enc * p.N * D;
    const uint8_t* image = p.image + (size_t)enc * 2 * IMG_BYTES;

    const uint32_t bar_w = sbase + S_BAR, bar_a_full = bar_w + 8, bar_t_full = bar_w + 16, bar_g_empty = bar_w + 24;
    const uint32_t bar_acc_full = bar_w + 32, bar_out_full = bar_w + 40, bar_h_read = bar_w + 48, bar_dg_full = bar_w + 56;
    const uint32_t bar_dg_stored = bar_w + 64;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sgen + S_TMEM);
    float* s_ln = reinterpret_cast<float*>(sgen + S_LN);
    unsigned* s_amax = reinterpret_cast<unsigned*>(sgen + S_AMAX);
    float* s_g = reinterpret_cast<float*>(sgen + S_G);

    if (tid == 0) {
        tc::mbar_init(bar_w, 1);
        tc::mbar_init(bar_a_full, GATHER_WARPS * 32);
        tc::mbar_init(bar_t_full, 1);                  // operand tile (bulk copy of the forward's saved tile) has landed
        tc::mbar_init(bar_g_empty, EPI_WARPS * 32);
        tc::mbar_init(bar_acc_full, 1);
        tc::mbar_init(bar_out_full, 1);
        tc::mbar_init(bar_h_read, EPI_WARPS * 32);      // the epilogue has copied the tile's h rows: the tile may be overwritten
        tc::mbar_init(bar_dg_full, EPI_WARPS * 32);     // d-gate planes are in tensor memory
        tc::mbar_init(bar_dg_stored, EPI_WARPS * 32);   // ... and have been copied to HBM: T_ACC may be overwritten
        tc::fence_barrier_init();
        tc::mbar_expect_tx(bar_w, IMG_W);
#pragma unroll 1
        for (uint32_t o = 0; o < IMG_W; o += 16384u) tc::bulk_g2s(sbase + o, image + o, 16384u, bar_w);
    }
    if (tid < 2 * D) s_ln[tid] = __ldg(reinterpret_cast<const float*>(image + IMG_W) + tid);
    if (tid < 4) s_amax[tid] = 0u;
    if (warp == 0) tc::tmem_alloc(tmem_slot, 512);
    // Equal tile counts per CTA (with the operand tile bulk-copied a tile's time is set by the epilogue: constant per 128
    // nodes), dealt ROUND-ROBIN: rows are in degree order, so the few tiles whose gather of hub rows outlasts the epilogue
    // (fan-out direction) sit next to each other -- a contiguous range put all of them on CTA 0 (measured: 141 us per launch
    // in the fan-out direction against 100 us in the fan-in direction).
    const int tile_beg = p.tile_beg + (int)blockIdx.x, tile_end = p.tile_end, tile_step = (int)gridDim.x;
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem = *tmem_slot;

    if (warp >= EPI_WARPS && warp < EPI_WARPS + GATHER_WARPS) {
        // ===================================================================== gather of d state_k
        // d state_k = d part (or the incoming gradient at the last step) + neighbour sum of d agg_{k+1}, fp32, into the
        // staging rows.  (The [agg | h | x deg 1] operand tile is NOT re-gathered: the forward saved it, thread 0 bulk-copies it.)
        // lane = (row group rg, 16-byte chunk c): 8 lanes cover one 256-byte row; a lane owns 2 rows of the tile.  ONE wave of
        // independent loads (own row, first neighbour, second-neighbour id), then one wave per further neighbour; the next
        // tile's row descriptors are loaded one tile ahead.
        const int gw = warp - EPI_WARPS, rg = lane >> 3, c = lane & 7;
        const int4* gdesc = reinterpret_cast<const int4*>(p.gdesc);
        const float* gsrc = p.last ? p.gout + eoff : p.in_part + eoff;
        const float* asrc = p.in_agg + eoff;
        const bool nbg = !p.last;
        int4 dn[4];
#pragma unroll
        for (int ps = 0; ps < 4; ++ps) {
            const int r = tile_beg * TM + gw * 16 + ps * 4 + rg;
            dn[ps] = (tile_beg < tile_end && r < p.N) ? __ldg(gdesc + r) : make_int4(-1, 0, 0, 0);
        }
        int it = 0;
        for (int tile = tile_beg; tile < tile_end; tile += tile_step, ++it) {
            if (lane == 0) PTRACE_MAX(13);
            int4 dc[4];
#pragma unroll
            for (int ps = 0; ps < 4; ++ps) dc[ps] = dn[ps];
#pragma unroll
            for (int ps = 0; ps < 4; ++ps) {
                const int r = (tile + tile_step) * TM + gw * 16 + ps * 4 + rg;
                dn[ps] = (tile + tile_step < tile_end && r < p.N) ? __ldg(gdesc + r) : make_int4(-1, 0, 0, 0);
            }
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {           // the lane's 4 rows, two at a time
                int node[2], beg[2], cnt[2], jn[2];
                float4 g[2][2], va[2][2];
                int maxc = 0;
                const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const int4 d = dc[2 * hf + q];
                    node[q] = d.x; beg[q] = d.y; cnt[q] = nbg ? d.z : 0; jn[q] = d.w;
                    maxc = max(maxc, cnt[q]);
                    g[q][0] = z4; g[q][1] = z4; va[q][0] = z4; va[q][1] = z4;
                    if (node[q] >= 0) {
                        g[q][0] = mgv_ld4(gsrc + (size_t)node[q] * D + c * 8);
                        g[q][1] = mgv_ld4(gsrc + (size_t)node[q] * D + c * 8 + 4);
                    }
                    if (cnt[q] > 0) {
                        va[q][0] = mgv_ld4(asrc + (size_t)jn[q] * D + c * 8);
                        va[q][1] = mgv_ld4(asrc + (size_t)jn[q] * D + c * 8 + 4);
                    }
                    if (cnt[q] > 1) jn[q] = p.idx[beg[q] + 1] & NODE_MASK;
                }
                float ag[2][8];
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    ag[q][0] = g[q][0].x + va[q][0].x; ag[q][1] = g[q][0].y + va[q][0].y; ag[q][2] = g[q][0].z + va[q][0].z; ag[q][3] = g[q][0].w + va[q][0].w;
                    ag[q][4] = g[q][1].x + va[q][1].x; ag[q][5] = g[q][1].y + va[q][1].y; ag[q][6] = g[q][1].z + va[q][1].z; ag[q][7] = g[q][1].w + va[q][1].w;
                }
                // further neighbours, two per row per trip
                for (int sl = 1; sl < maxc; sl += 2) {
                    int j[2][2];
#pragma unroll
                    for (int q = 0; q < 2; ++q) {
                        j[q][0] = jn[q];
                        j[q][1] = (sl + 1 < cnt[q]) ? (p.idx[beg[q] + sl + 1] & NODE_MASK) : 0;
                        if (sl + 2 < cnt[q]) jn[q] = p.idx[beg[q] + sl + 2] & NODE_MASK;
                    }
                    float4 wa[2][2][2];
#pragma unroll
                    for (int q = 0; q < 2; ++q)
#pragma unroll
                        for (int t = 0; t < 2; ++t) {
                            wa[q][t][0] = z4; wa[q][t][1] = z4;
                            if (sl + t < cnt[q]) {
                                wa[q][t][0] = mgv_ld4(asrc + (size_t)j[q][t] * D + c * 8);
                                wa[q][t][1] = mgv_ld4(asrc + (size_t)j[q][t] * D + c * 8 + 4);
                            }
                        }
#pragma unroll
                    for (int q = 0; q < 2; ++q)
#pragma unroll
                        for (int t = 0; t < 2; ++t) {
                            ag[q][0] += wa[q][t][0].x; ag[q][1] += wa[q][t][0].y; ag[q][2] += wa[q][t][0].z; ag[q][3] += wa[q][t][0].w;
                            ag[q][4] += wa[q][t][1].x; ag[q][5] += wa[q][t][1].y; ag[q][6] += wa[q][t][1].z; ag[q][7] += wa[q][t][1].w;
                        }
                }
                if (hf == 0) {
                    if (lane == 0) PTRACE_MAX(14);
                    tc::mbar_wait_warp(bar_g_empty, (uint32_t)((it & 1) ^ 1), lane, 64);   // previous tile's epilogue has read the staging rows
                }
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    float* dst = s_g + (gw * 16 + (2 * hf + q) * 4 + rg) * LDGS + c * 8;
                    *reinterpret_cast<float4*>(dst) = make_float4(ag[q][0], ag[q][1], ag[q][2], ag[q][3]);
                    *reinterpret_cast<float4*>(dst + 4) = make_float4(ag[q][4], ag[q][5], ag[q][6], ag[q][7]);
                }
            }
            tc::mbar_arrive(bar_a_full);
            if (lane == 0) PTRACE_MAX(15);
        }
    } else if (warp == EPI_WARPS + GATHER_WARPS) {
        // ===================================================================== MMA issue + operand-tile bulk copies (one thread)
        if (lane == 0 && tile_beg < tile_end) {
            auto load_tile = [&](int t) {       // the forward's saved operand tile -> the (idle) tile buffer
                const uint8_t* src = p.tiles + (size_t)enc * p.tiles_enc_stride + (size_t)t * A_TILE_BYTES;
                if (LOWP) {                     // hi planes only: agg 16 KB, h 16 KB, x 4 KB
                    tc::mbar_expect_tx(bar_t_full, 36864u);
#pragma unroll 1
                    for (uint32_t o = 0; o < 16384u; o += 8192u) {
                        tc::bulk_g2s(sbase + A_AGG_HI + o, src + o, 8192u, bar_t_full);
                        tc::bulk_g2s(sbase + A_H_HI + o, src + (A_H_HI - A_AGG_HI) + o, 8192u, bar_t_full);
                    }
                    tc::bulk_g2s(sbase + A_X_HI, src + (A_X_HI - A_AGG_HI), 4096u, bar_t_full);
                } else {
                    tc::mbar_expect_tx(bar_t_full, A_TILE_BYTES);
#pragma unroll 1
                    for (uint32_t o = 0; o < A_TILE_BYTES; o += 8192u) tc::bulk_g2s(sbase + A_AGG_HI + o, src + o, 8192u, bar_t_full);
                }
            };
            auto issue_recompute = [&](uint32_t tph) {     // the 39 recompute MMAs of a tile (bit-identical products to the forward)
                tc::mbar_wait_sleep(bar_t_full, tph, 32);
                tc::fence_after_sync();
                const uint32_t d = tmem + T_ACC;
                tc::mma3p<LOWP>(d, tc::desc_k_plain16(sbase + A_X_HI), tc::desc_k_plain16(sbase + A_X_LO),
                         tc::desc_k_plain16(sbase + WX_HI), tc::desc_k_plain16(sbase + WX_LO), tc::make_idesc(128, 256, false, false, LOWP), 0u);
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    tc::mma3p<LOWP>(d, tc::desc_k_sw128(sbase + A_H_HI + 32 * j), tc::desc_k_sw128(sbase + A_H_LO + 32 * j),
                             tc::desc_k_sw128(sbase + WHH_HI + 32 * j), tc::desc_k_sw128(sbase + WHH_LO + 32 * j),
                             tc::make_idesc(128, 128, false, false, LOWP), 1u);
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    tc::mma3p<LOWP>(d + 192u, tc::desc_k_sw128(sbase + A_H_HI + 32 * j), tc::desc_k_sw128(sbase + A_H_LO + 32 * j),
                             tc::desc_k_sw128(sbase + WHH_HI + 16384 + 32 * j), tc::desc_k_sw128(sbase + WHH_LO + 16384 + 32 * j),
                             tc::make_idesc(128, 64, false, false, LOWP), 1u);
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    tc::mma3p<LOWP>(d, tc::desc_k_sw128(sbase + A_AGG_HI + 32 * j), tc::desc_k_sw128(sbase + A_AGG_LO + 32 * j),
                             tc::desc_k_sw128(sbase + WC_HI + 32 * j), tc::desc_k_sw128(sbase + WC_LO + 32 * j),
                             tc::make_idesc(128, 192, false, false, LOWP), 1u);
                tc::mma_commit(bar_acc_full);
            };
            tc::mbar_wait_sleep(bar_w, 0u);
            load_tile(tile_beg);
            issue_recompute(0u);
            int it = 0;
            for (int tile = tile_beg; tile < tile_end; tile += tile_step, ++it) {
                const uint32_t ph = (uint32_t)(it & 1);
                // the tile buffer is free once the recompute MMAs have read it and the epilogue has copied its h rows
                tc::mbar_wait_sleep(bar_acc_full, ph, 32);
                tc::mbar_wait_sleep(bar_h_read, ph, 32);
                if (tile + tile_step < tile_end) load_tile(tile + tile_step);
                tc::mbar_wait_sleep(bar_dg_full, ph, 32);
                tc::fence_after_sync();
                PTRACE(7);
                if (!p.first) {
                    const uint32_t o = tmem + T_OUT;
                    const uint32_t i128 = tc::make_idesc(128, 128, false, true, LOWP), i64 = tc::make_idesc(128, 64, false, true, LOWP);
#pragma unroll
                    for (int s = 0; s < 8; ++s) {        // d r, d z: [d agg | d part] += d g . [Wc | Whh] rows 16 s ..
                        const uint32_t a = tmem + T_ACC + 16u * s;
                        tc::mma3p_ts<LOWP>(o, a, a + 8u, tc::desc_mn_sw128(sbase + WC_HI + 2048u * s, WHH_HI - WC_HI),
                                            tc::desc_mn_sw128(sbase + WC_LO + 2048u * s, WHH_LO - WC_LO), i128, 1u);
                    }
#pragma unroll
                    for (int s = 8; s < 12; ++s) {       // d gi_n: d agg += . Wc rows 128 ..
                        const uint32_t a = tmem + T_ACC + 16u * s;
                        tc::mma3p_ts<LOWP>(o, a, a + 8u, tc::desc_mn_sw128(sbase + WC_HI + 2048u * s, 0),
                                            tc::desc_mn_sw128(sbase + WC_LO + 2048u * s, 0), i64, 1u);
                    }
#pragma unroll
                    for (int s = 12; s < 16; ++s) {      // d gh_n: d part += . Whh rows 128 ..
                        const uint32_t a = tmem + T_ACC + 16u * s;
                        tc::mma3p_ts<LOWP>(o + 64u, a, a + 8u, tc::desc_mn_sw128(sbase + WHH_HI + 2048u * (s - 4), 0),
                                            tc::desc_mn_sw128(sbase + WHH_LO + 2048u * (s - 4), 0), i64, 1u);
                    }
                    tc::mma_commit(bar_out_full);
                }
                // the next tile's recompute runs behind the data-gradient MMAs (in issue order) while the epilogue stores
                // this tile's outputs: it only writes T_ACC, which the epilogue is done with
                if (tile + tile_step < tile_end) {
                    tc::mbar_wait_sleep(bar_dg_stored, ph, 32);      // the epilogue re-reads the planes for their HBM copy
                    issue_recompute(ph ^ 1u);
                }
                PTRACE(3);
            }
        }
    } else if (warp < EPI_WARPS) {
        // ===================================================================== epilogue: 2 threads per tile row = TMEM lane
        // Warps q and 4 + q own lanes 32 q .. 32 q + 31; warp group wg = warp / 4 handles units 32 wg .. 32 wg + 31 of its
        // row (row sums are exchanged through shared memory).  
        // All per-row arrays live in the thread's tensor-memory lane, so every loop below is ROLLED: a fully unrolled
        // body is > 100 KB of straight-line code that one warp executes once per tile, i.e. pure instruction-cache
        // misses (measured: 8 cycles per instruction).
        //   T_ACC   r | z | gi_n | gh_n pre-activations -> r | z | n | gh_n -> fp32 d gates -> fp16 hi/lo planes
        //   T_OUT   [0, 64) own state row h (later zero = d agg accumulator init), [64, 128) pre-LayerNorm output ->
        //           g z (the direct part of d part), scaled: the data-gradient MMAs accumulate on top of both
        //   T_LNP   d ln_w | d ln_b partial sums of this thread's rows
        const int wg = warp >> 2, row = (warp & 3) * 32 + lane, u0 = 32 * wg;
        const uint32_t tl = tmem + ((uint32_t)((warp & 3) * 32) << 16);
        const uint32_t t_acc = tl + T_ACC, t_out = tl + T_OUT, t_lnp = tl + T_LNP;
        const float* gs = s_g + row * LDGS;
        float* s_ex = reinterpret_cast<float*>(sgen + S_EX);
        constexpr int EPI_T = EPI_WARPS * 32;
#pragma unroll 1
        for (int cc = 0; cc < 32; cc += 4) {
            tc::tmem_st4(t_lnp + u0 + cc, 0.f, 0.f, 0.f, 0.f);
            tc::tmem_st4(t_lnp + 64 + u0 + cc, 0.f, 0.f, 0.f, 0.f);
        }
        tc::tmem_st_wait();
        float run_scale = 1.0f;
        const uint64_t pol_stream = tc::l2_policy_evict_first();      // hand-off buffers: written once, read once by the next kernel
        int it = 0;
        for (int tile = tile_beg; tile < tile_end; tile += tile_step, ++it) {
            const uint32_t ph = (uint32_t)(it & 1);
            const bool valid = tile * TM + row < p.N;
            const int node = valid ? p.order[tile * TM + row] : 0;
            // own state row (this thread's 32 units) -> tensor memory, from the operand tile's h planes (hi + lo is h to
            // 2^-22: no second global read of the row); the tile is overwritten by the next bulk copy after the barrier
            tc::mbar_wait_warp(bar_t_full, ph, lane, 32);
#pragma unroll
            for (int c8 = 0; c8 < 4; ++c8) {
                const uint32_t off = tc::sw128_off(row, 4 * wg + c8);
                const uint4 hi = *reinterpret_cast<const uint4*>(sgen + A_H_HI + off);
                float h[8];
                if (LOWP) {                     // the bf16 operand the forward multiplied (bf16 mode: h to 2^-9)
                    const uint32_t* w = reinterpret_cast<const uint32_t*>(&hi);
#pragma unroll
                    for (int e = 0; e < 4; ++e) { h[2 * e] = __uint_as_float(w[e] << 16); h[2 * e + 1] = __uint_as_float(w[e] & 0xffff0000u); }
                } else {
                    const uint4 lo = *reinterpret_cast<const uint4*>(sgen + A_H_LO + off);
                    const __half2* h2 = reinterpret_cast<const __half2*>(&hi);
                    const __half2* l2 = reinterpret_cast<const __half2*>(&lo);
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const float2 a = __half22float2(h2[e]), bq = __half22float2(l2[e]);
                        h[2 * e] = a.x + bq.x; h[2 * e + 1] = a.y + bq.y;
                    }
                }
                tc::tmem_st8f(t_out + u0 + 8 * c8, h);
            }
            tc::mbar_arrive(bar_h_read);
            tc::mbar_wait_warp(bar_acc_full, ph, lane, 32);
            tc::mbar_wait_warp(bar_a_full, ph, lane, 32);
            tc::fence_after_sync();
            tc::tmem_st_wait();
            if (tid == 0) PTRACE(4);
            // ---- pass 1: gates, pre-LayerNorm output
            float sum = 0.f;
#pragma unroll 1
            for (int c8 = 0; c8 < 4; ++c8) {
                const int u = u0 + 8 * c8;
                float gr[8], gz[8], gi[8], gh[8], h[8];
                tc::tmem_ld8(t_acc + u, gr);
                tc::tmem_ld8(t_acc + 64 + u, gz);
                tc::tmem_ld8(t_acc + 128 + u, gi);
                tc::tmem_ld8(t_acc + 192 + u, gh);
                tc::tmem_ld8(t_out + u, h);
                tc::tmem_ld_wait();
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    float r, z, n, hn;
                    gru_gates(gr[e], gz[e], gi[e], gh[e], r, z, n, hn);
                    gr[e] = r; gz[e] = z; gi[e] = n;
                    h[e] = fmaf(z, h[e] - n, n);
                    sum += h[e];
                }
                tc::tmem_st8f(t_acc + u, gr);
                tc::tmem_st8f(t_acc + 64 + u, gz);
                tc::tmem_st8f(t_acc + 128 + u, gi);
                tc::tmem_st8f(t_out + 64 + u, h);
            }
            tc::tmem_st_wait();
            // ---- LayerNorm statistics (two-pass, like the forward) and the two row sums of its backward
            float mean = 0.f, rstd = 1.0f, c1 = 0.f, c2 = 0.f;
            if (p.layernorm) {
                s_ex[wg * TM + row] = sum;
                tc::named_bar_sync(1, EPI_T);
                mean = (s_ex[row] + s_ex[TM + row]) * (1.0f / D);
                float var = 0.f;
#pragma unroll 1
                for (int c8 = 0; c8 < 4; ++c8) {
                    const int u = u0 + 8 * c8;
                    float xv[8];
                    tc::tmem_ld8(t_out + 64 + u, xv);
                    const float4 ga = lds4(gs + u), gb = lds4(gs + u + 4);
                    const float4 wa = lds4(s_ln + u), wb = lds4(s_ln + u + 4);
                    const float gw[8] = {ga.x * wa.x, ga.y * wa.y, ga.z * wa.z, ga.w * wa.w, gb.x * wb.x, gb.y * wb.y, gb.z * wb.z, gb.w * wb.w};
                    tc::tmem_ld_wait();
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        const float d = xv[e] - mean;
                        var = fmaf(d, d, var);
                        c1 += gw[e];
                        c2 = fmaf(gw[e], d, c2);
                    }
                }
                s_ex[(2 + wg) * TM + row] = var;
                s_ex[(4 + wg) * TM + row] = c1;
                s_ex[(6 + wg) * TM + row] = c2;
                tc::named_bar_sync(1, EPI_T);
                var = s_ex[2 * TM + row] + s_ex[3 * TM + row];
                c1 = s_ex[4 * TM + row] + s_ex[5 * TM + row];
                c2 = s_ex[6 * TM + row] + s_ex[7 * TM + row];
                rstd = rsqrtf(var * (1.0f / D) + LN_EPS);
                c1 *= (1.0f / D);
                c2 *= rstd * (1.0f / D);
            }
            if (tid == 0) PTRACE(5);
            // ---- pass 2: LayerNorm backward + GRU backward -> fp32 d gates in place, g z, LayerNorm parameter gradients
            float amax = 0.f;
#pragma unroll 1
            for (int c4 = 0; c4 < 8; ++c4) {           // 4 units per trip (80 registers per thread)
                const int u = u0 + 4 * c4;
                float r[4], z[4], n[4], hn[4], h[4], xv[4], lw[4], lb[4];
                tc::tmem_ld4(t_acc + u, r);
                tc::tmem_ld4(t_acc + 64 + u, z);
                tc::tmem_ld4(t_acc + 128 + u, n);
                tc::tmem_ld4(t_acc + 192 + u, hn);
                tc::tmem_ld4(t_out + u, h);
                tc::tmem_ld4(t_out + 64 + u, xv);
                if (p.layernorm) { tc::tmem_ld4(t_lnp + u, lw); tc::tmem_ld4(t_lnp + 64 + u, lb); }
                const float4 ga = lds4(gs + u), wa = lds4(s_ln + u);
                const float gv[4] = {ga.x, ga.y, ga.z, ga.w};
                const float wv[4] = {wa.x, wa.y, wa.z, wa.w};
                tc::tmem_ld_wait();
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    float dxh = gv[e];
                    if (p.layernorm) {
                        const float xn = (xv[e] - mean) * rstd;
                        lw[e] = fmaf(gv[e], xn, lw[e]);
                        lb[e] += gv[e];
                        dxh = rstd * (fmaf(gv[e], wv[e], -c1) - xn * c2);
                    }
                    const float dn = dxh * (1.0f - z[e]);
                    const float dzz = dxh * (h[e] - n[e]);
                    const float dni = dn * (1.0f - n[e] * n[e]);
                    const float dr = dni * hn[e] * r[e] * (1.0f - r[e]);
                    const float dz = dzz * z[e] * (1.0f - z[e]);
                    hn[e] = dni * r[e];
                    xv[e] = dxh * z[e];
                    r[e] = dr; z[e] = dz; n[e] = dni;
                    amax = fmaxf(amax, fmaxf(fmaxf(fabsf(dr), fabsf(dz)), fabsf(dni)));
                }
                tc::tmem_st4(t_acc + u, r[0], r[1], r[2], r[3]);
                tc::tmem_st4(t_acc + 64 + u, z[0], z[1], z[2], z[3]);
                tc::tmem_st4(t_acc + 128 + u, n[0], n[1], n[2], n[3]);
                tc::tmem_st4(t_acc + 192 + u, hn[0], hn[1], hn[2], hn[3]);
                tc::tmem_st4(t_out + 64 + u, xv[0], xv[1], xv[2], xv[3]);
                if (p.layernorm) {
                    tc::tmem_st4(t_lnp + u, lw[0], lw[1], lw[2], lw[3]);
                    tc::tmem_st4(t_lnp + 64 + u, lb[0], lb[1], lb[2], lb[3]);
                }
            }
            tc::mbar_arrive(bar_g_empty);
            if (tid == 0) PTRACE(12);
            // ---- tile-wide power-of-two scale (fp16 range), shared with the weight-gradient kernel through HBM
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
            if (lane == 0) atomicMax(s_amax + (it % 3), __float_as_uint(amax));
            tc::named_bar_sync(1, EPI_T);
            const float scale = LOWP ? 1.0f : pow2_scale_keep(__uint_as_float(s_amax[it % 3]), run_scale);
            run_scale = scale;
            if (tid == 0) {
                s_amax[(it + 2) % 3] = 0u;
                p.scales[(size_t)enc * p.chunk_cap + (tile - p.tile_beg)] = scale;
                atomicMin(p.smin + enc, __float_as_uint(scale));
            }
            tc::tmem_st_wait();
            if (tid == 0) PTRACE(6);
            // ---- pass 3: fp32 d gates -> scaled fp16 hi/lo planes, in place (A operand of the data-gradient MMAs).
            //      K step s = gates 16 s .. 16 s + 15; this warp group's units are the K steps with (s & 3) / 2 == wg.
            {
#pragma unroll 2
                for (int k = 0; k < 8; ++k) {
                    const int s = 4 * (k >> 1) + 2 * wg + (k & 1);
                    float v[16];
                    tc::tmem_ld16(t_acc + 16 * s, v);
                    tc::tmem_ld_wait();
                    if (LOWP) {
                        uint32_t pk[8];
#pragma unroll
                        for (int e = 0; e < 8; ++e) pk[e] = tc::pack_bf16x2(v[2 * e], v[2 * e + 1]);
                        tc::tmem_st8(t_acc + 16 * s, pk);
                    } else {
                        uint32_t pk[16];
#pragma unroll
                        for (int e = 0; e < 8; ++e) tc::split2(v[2 * e] * scale, v[2 * e + 1] * scale, pk[e], pk[8 + e]);
                        tc::tmem_st16(t_acc + 16 * s, pk);
                    }
                }
                // accumulator init of the data-gradient MMAs: d agg = 0, d part = scale * g z
                if (!p.first) {
#pragma unroll 2
                    for (int c8 = 0; c8 < 4; ++c8) {
                        const int u = u0 + 8 * c8;
                        float q[8];
                        tc::tmem_ld8(t_out + 64 + u, q);
                        tc::tmem_ld_wait();
#pragma unroll
                        for (int e = 0; e < 8; ++e) q[e] *= scale;
                        tc::tmem_st8f(t_out + 64 + u, q);
#pragma unroll
                        for (int e = 0; e < 8; ++e) q[e] = 0.f;
                        tc::tmem_st8f(t_out + u, q);
                    }
                }
            }
            tc::tmem_st_wait();
            tc::fence_before_sync();
            tc::mbar_arrive(bar_dg_full);
            // ---- pass 3b, while the data-gradient MMAs run: the planes (re-read from tensor memory, which the MMAs only
            //      read) -> HBM [plane][64-node half][8-gate chunk (32)][node row (64)][16 B] for the weight-gradient kernel
            {
                uint8_t* dg = p.dgbuf + ((size_t)enc * p.chunk_cap + (tile - p.tile_beg)) * DG_TILE_BYTES + (row >> 6) * 32768 + (row & 63) * 16;
#pragma unroll 1
                for (int b = 0; b < 4; ++b) {          // gate block b (r, z, gi_n, gh_n): this warp group's two K steps, one wait
                    const int s0 = 4 * b + 2 * wg;
                    float v0[16], v1[16];
                    tc::tmem_ld16(t_acc + 16 * s0, v0);
                    tc::tmem_ld16(t_acc + 16 * (s0 + 1), v1);
                    tc::tmem_ld_wait();
                    const uint32_t* pk = reinterpret_cast<const uint32_t*>(v0);
                    const uint32_t* qk = reinterpret_cast<const uint32_t*>(v1);
                    uint8_t* hb = dg + (size_t)(2 * s0) * 1024;
                    tc::stg_v4_hint(hb, make_uint4(pk[0], pk[1], pk[2], pk[3]), pol_stream);
                    tc::stg_v4_hint(hb + 1024, make_uint4(pk[4], pk[5], pk[6], pk[7]), pol_stream);
                    tc::stg_v4_hint(hb + 2048, make_uint4(qk[0], qk[1], qk[2], qk[3]), pol_stream);
                    tc::stg_v4_hint(hb + 3072, make_uint4(qk[4], qk[5], qk[6], qk[7]), pol_stream);
                    if (!LOWP) {
                        tc::stg_v4_hint(hb + 65536, make_uint4(pk[8], pk[9], pk[10], pk[11]), pol_stream);
                        tc::stg_v4_hint(hb + 65536 + 1024, make_uint4(pk[12], pk[13], pk[14], pk[15]), pol_stream);
                        tc::stg_v4_hint(hb + 65536 + 2048, make_uint4(qk[8], qk[9], qk[10], qk[11]), pol_stream);
                        tc::stg_v4_hint(hb + 65536 + 3072, make_uint4(qk[12], qk[13], qk[14], qk[15]), pol_stream);
                    }
                }
            }
            tc::fence_before_sync();
            tc::mbar_arrive(bar_dg_stored);
            // ---- data gradients of step k-1
            if (!p.first) {
                tc::mbar_wait_warp(bar_out_full, ph, lane, 32);
                tc::fence_after_sync();
                if (tid == 0) PTRACE(8);
                const float inv = 1.0f / scale;
#pragma unroll 2
                for (int c8 = 0; c8 < 4; ++c8) {
                    const int u = u0 + 8 * c8;
                    float a[8], q[8];
                    tc::tmem_ld8(t_out + u, a);
                    tc::tmem_ld8(t_out + 64 + u, q);
                    tc::tmem_ld_wait();
#pragma unroll
                    for (int e = 0; e < 8; ++e) { a[e] *= inv; q[e] *= inv; }
                    if (valid) {
                        stg8(p.out_agg + eoff + (size_t)node * D + u, a);
                        stg8(p.out_part + eoff + (size_t)node * D + u, q);
                    }
                }
            }
            if (tid == 0) PTRACE(9);
        }
    }
    // ---- LayerNorm parameter gradients: per-thread partial sums (tensor memory) -> column sums -> this CTA's partial block
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    float* scratch = reinterpret_cast<float*>(sgen + A_AGG_HI);      // [128][132], the tile and staging buffers are idle now
    if (warp < EPI_WARPS) {
        const int row = (warp & 3) * 32 + lane, u0 = 32 * (warp >> 2);
        const uint32_t t_lnp = tmem + ((uint32_t)((warp & 3) * 32) << 16) + T_LNP;
#pragma unroll 1
        for (int c8 = 0; c8 < 8; ++c8) {
            const int col = (c8 < 4) ? u0 + 8 * c8 : 64 + u0 + 8 * (c8 - 4);
            float v[8];
            tc::tmem_ld8(t_lnp + col, v);
            tc::tmem_ld_wait();
            *reinterpret_cast<float4*>(scratch + row * 132 + col) = make_float4(v[0], v[1], v[2], v[3]);
            *reinterpret_cast<float4*>(scratch + row * 132 + col + 4) = make_float4(v[4], v[5], v[6], v[7]);
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (tid < 2 * D && p.layernorm && tile_beg < tile_end) {
        float s = 0.f;
#pragma unroll 8
        for (int r = 0; r < TM; ++r) s += scratch[r * 132 + tid];
        float* part = p.partial + (((size_t)enc * p.gxp + blockIdx.x) * 2 + p.dir) * SGRAD;
        part[O_LNW + tid] += s;
    }
    if (warp == 0) tc::tmem_dealloc(tmem, 512);
}

// Fire-and-forget vector add to global memory (the block is private to this CTA; a read-modify-write loop would pay one
// memory round trip per element: measured 55 000 cycles for the 113 KB block).
__device__ __forceinline__ void red_add4(float4* dst, const float4& v) {
    asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(dst), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// ======================================================================================= weight gradients (streaming)
constexpr int W_THREADS = 6 * 32;          // warp 0 bulk-copy producer, warp 1 MMA issue, warps 2-5 rescale + flush
// stage = 64 nodes (half a tile): d-gate planes, operand planes
constexpr uint32_t ST_DG_HI = 0, ST_DG_LO = 32768, ST_AGG_HI = 65536, ST_H_HI = 73728, ST_AGG_LO = 81920, ST_H_LO = 90112;
constexpr uint32_t ST_X_HI = 98304, ST_X_LO = 100352, ST_BYTES = 102400;
constexpr uint32_t W_BAR = 2 * ST_BYTES;   // full[2], ready[2], empty[2], done
constexpr uint32_t W_TMEM = W_BAR + 64;
constexpr uint32_t W_SMEM = W_TMEM + 64 + 1024;
static_assert(W_SMEM <= 227 * 1024, "struct weight gradient: shared memory");

struct WgTC {
    int ntiles;                // tiles of this chunk
    int chunk_cap;
    int dir, gxp;
    const uint8_t* tiles;      // the forward's saved operand tiles of this step, enc 0
    size_t tiles_enc_stride;
    int tile_base;             // first tile of this chunk
    const uint8_t* dgbuf;
    const float* scales;
    const unsigned* smin;
    float* partial;
    long long* trace;          // optional [CTA][16 stages][16] clock64 samples (dev tool)
};
#define WTRACE(slot) do { if (p.trace && i < 16) p.trace[(((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 16 + i) * 16 + (slot)] = clock64(); } while (0)

template <bool LOWP>
__global__ void __launch_bounds__(W_THREADS, 1) struct_bwd_wgrad_kernel(const WgTC p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const uint32_t sbase = (tc::smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* sgen = smem_raw + (sbase - tc::smem_u32(smem_raw));
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int enc = blockIdx.y;
    const uint32_t bar_full = sbase + W_BAR, bar_ready = bar_full + 16, bar_empty = bar_full + 32, bar_done = bar_full + 48;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sgen + W_TMEM);
    if (tid == 0) {
        for (int s = 0; s < 2; ++s) {
            tc::mbar_init(bar_full + 8 * s, 1);
            tc::mbar_init(bar_ready + 8 * s, 4 * 32);
            tc::mbar_init(bar_empty + 8 * s, 1);
        }
        tc::mbar_init(bar_done, 1);
        tc::fence_barrier_init();
    }
    if (warp == 0) tc::tmem_alloc(tmem_slot, 512);
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    const int tile_beg = (int)((long long)p.ntiles * blockIdx.x / gridDim.x);
    const int tile_end = (int)((long long)p.ntiles * (blockIdx.x + 1) / gridDim.x);
    const int nhalf = 2 * (tile_end - tile_beg);
    const float smin = __uint_as_float(p.smin[enc]);

    if (warp == 0) {
        if (lane == 0) {
            const uint64_t pol = tc::l2_policy_evict_first();
            for (int i = 0; i < nhalf; ++i) {
                const int s = i & 1, tile = tile_beg + (i >> 1), h = i & 1;
                WTRACE(0);
                tc::mbar_wait_sleep(bar_empty + 8 * s, (uint32_t)(((i >> 1) & 1) ^ 1));
                WTRACE(1);
                tc::mbar_expect_tx(bar_full + 8 * s, LOWP ? 51200u : ST_BYTES);
                const uint8_t* dg = p.dgbuf + ((size_t)enc * p.chunk_cap + tile) * DG_TILE_BYTES + (size_t)h * 32768;
                const uint8_t* at = p.tiles + (size_t)enc * p.tiles_enc_stride + (size_t)(p.tile_base + tile) * A_TILE_BYTES;
                const uint32_t st = sbase + (uint32_t)s * ST_BYTES, bar = bar_full + 8 * s;
                tc::bulk_g2s_hint(st + ST_DG_HI, dg, 16384u, bar, pol);
                tc::bulk_g2s_hint(st + ST_DG_HI + 16384u, dg + 16384, 16384u, bar, pol);
                tc::bulk_g2s_hint(st + ST_AGG_HI, at + 0 + h * 8192, 8192u, bar, pol);
                tc::bulk_g2s_hint(st + ST_H_HI, at + 32768 + h * 8192, 8192u, bar, pol);
                tc::bulk_g2s_hint(st + ST_X_HI, at + 65536 + h * 2048, 2048u, bar, pol);
                if (!LOWP) {
                    tc::bulk_g2s_hint(st + ST_DG_LO, dg + 65536, 16384u, bar, pol);
                    tc::bulk_g2s_hint(st + ST_DG_LO + 16384u, dg + 65536 + 16384, 16384u, bar, pol);
                    tc::bulk_g2s_hint(st + ST_AGG_LO, at + 16384 + h * 8192, 8192u, bar, pol);
                    tc::bulk_g2s_hint(st + ST_H_LO, at + 49152 + h * 8192, 8192u, bar, pol);
                    tc::bulk_g2s_hint(st + ST_X_LO, at + 69632 + h * 2048, 2048u, bar, pol);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t i128 = tc::make_idesc(128, 128, true, true, LOWP), i16 = tc::make_idesc(128, 16, true, true, LOWP);
            for (int i = 0; i < nhalf; ++i) {
                const int s = i & 1;
                WTRACE(4);
                tc::mbar_wait_sleep(bar_ready + 8 * s, (uint32_t)((i >> 1) & 1), 32);
                tc::fence_after_sync();
                WTRACE(5);
                const uint32_t st = sbase + (uint32_t)s * ST_BYTES;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint32_t acc = (i > 0 || j > 0) ? 1u : 0u;
                    const uint64_t b_hi = tc::desc_mn_sw128(st + ST_AGG_HI + 2048u * j, 8192), b_lo = tc::desc_mn_sw128(st + ST_AGG_LO + 2048u * j, 8192);
                    const uint64_t x_hi = tc::desc_mn_plain16(st + ST_X_HI + 512u * j), x_lo = tc::desc_mn_plain16(st + ST_X_LO + 512u * j);
#pragma unroll
                    for (int g = 0; g < 2; ++g) {
                        // d gates^T: 16 chunks of 8 gates 1 KB apart (SBO), 8-node K groups 128 B apart (LBO), no swizzle
                        const uint64_t a_hi = tc::make_desc(st + ST_DG_HI + 16384u * g + 256u * j, 128, 1024, tc::LAYOUT_NONE);
                        const uint64_t a_lo = tc::make_desc(st + ST_DG_LO + 16384u * g + 256u * j, 128, 1024, tc::LAYOUT_NONE);
                        tc::mma3p<LOWP>(tmem + 160u * g, a_hi, a_lo, b_hi, b_lo, i128, acc);
                        tc::mma3p<LOWP>(tmem + 160u * g + 128u, a_hi, a_lo, x_hi, x_lo, i16, acc);
                    }
                }
                tc::mma_commit(bar_empty + 8 * s);
                WTRACE(6);
            }
            tc::mma_commit(bar_done);
        }
    } else {
        // rescale the tile's planes from its own power-of-two scale to the chunk-wide one, then hand the stage to the MMA thread
        const int t128 = tid - 64;
        for (int i = 0; i < nhalf; ++i) {
            const int s = i & 1, tile = tile_beg + (i >> 1);
            tc::mbar_wait_warp(bar_full + 8 * s, (uint32_t)((i >> 1) & 1), lane, 32);
            if (tid == 64) WTRACE(2);
            const float m = smin / p.scales[(size_t)enc * p.chunk_cap + tile];
            if (!LOWP && m != 1.0f) {
                const __half2 m2 = __float2half2_rn(m);
                uint4* st = reinterpret_cast<uint4*>(sgen + (size_t)s * ST_BYTES);
#pragma unroll 4
                for (int q = t128; q < 65536 / 16; q += 128) {
                    uint4 v = st[q];
                    __half2* h = reinterpret_cast<__half2*>(&v);
                    h[0] = __hmul2(h[0], m2); h[1] = __hmul2(h[1], m2); h[2] = __hmul2(h[2], m2); h[3] = __hmul2(h[3], m2);
                    st[q] = v;
                }
            }
            tc::fence_async_smem();
            tc::mbar_arrive(bar_ready + 8 * s);
            if (tid == 64) WTRACE(3);
        }
        // flush: thread = accumulator row = d-gate column
        if (nhalf > 0) {
            const int i = 0;
            if (tid == 64) WTRACE(8);
            tc::mbar_wait_warp(bar_done, 0u, lane, 64);
            tc::fence_after_sync();
            if (tid == 64) WTRACE(9);
            // tensor memory -> shared memory (the stages are idle) -> coalesced vector reductions into the partial block
            const int L = (warp & 3) * 32 + lane;
            const uint32_t tl = tmem + ((uint32_t)((warp & 3) * 32) << 16);
            float* part = p.partial + (((size_t)enc * p.gxp + blockIdx.x) * 2 + p.dir) * SGRAD;
            float* stg = reinterpret_cast<float*>(sgen);                  // [2 groups][128 rows][FLD]
            constexpr int FLD = 148;
            const float un = 1.0f / smin;
#pragma unroll 1
            for (int g = 0; g < 2; ++g)
#pragma unroll 2
                for (int c8 = 0; c8 < 18; ++c8) {
                    float v[8];
                    tc::tmem_ld8(tl + 160u * g + 8 * c8, v);
                    tc::tmem_ld_wait();
                    float* d = stg + (g * 128 + L) * FLD + 8 * c8;
                    *reinterpret_cast<float4*>(d) = make_float4(v[0] * un, v[1] * un, v[2] * un, v[3] * un);
                    *reinterpret_cast<float4*>(d + 4) = make_float4(v[4] * un, v[5] * un, v[6] * un, v[7] * un);
                }
            tc::named_bar_sync(1, 4 * 32);
            float4* part4 = reinterpret_cast<float4*>(part);
            for (int q = t128; q < G3 * 19; q += 128) {                   // d Wcx rows: 64 agg columns, 8 feature columns, 4 pad
                const int o = q / 19, c4 = q % 19;
                if (c4 < 18) {
                    const int g = o >= 128 ? 1 : 0, col = c4 < 16 ? 4 * c4 : 128 + 4 * (c4 - 16);
                    const float4 v = *reinterpret_cast<const float4*>(stg + (g * 128 + o - 128 * g) * FLD + col);
                    red_add4(part4 + (O_WCX + o * LDC) / 4 + c4, v);
                }
            }
            for (int q = t128; q < G3 * 17; q += 128) {                   // d Whh rows (d gh_n rows live in group 1, rows 64..127)
                const int o = q / 17, c4 = q % 17;
                if (c4 < 16) {
                    const int row = o >= 128 ? 128 + o - 64 : o;
                    const float4 v = *reinterpret_cast<const float4*>(stg + row * FLD + 64 + 4 * c4);
                    red_add4(part4 + (O_WHH + o * LDM) / 4 + c4, v);
                }
            }
            for (int o = t128; o < G3; o += 128) {                        // biases: deg column -> d bc, ones column -> d b_ih, d b_hh
                const int rc = o >= 128 ? 128 + o - 128 : o, rh = o >= 128 ? 128 + o - 64 : o;
                atomicAdd(part + O_BC + o, stg[rc * FLD + 136]);
                atomicAdd(part + O_BIH + o, stg[rc * FLD + 137]);
                atomicAdd(part + O_BHH + o, stg[rh * FLD + 137]);
            }
            if (tid == 64) WTRACE(10);
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc(tmem, 512);
}

__global__ void struct_reduce_tc_kernel(const float* __restrict__ partial, int gxp, float* __restrict__ grads, int num_enc) {
    const size_t total = (size_t)num_enc * 2 * SGRAD;
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int enc = (int)(idx / (2 * SGRAD));
    const size_t rem = idx % (2 * (size_t)SGRAD);
    float s = 0.f;
    for (int b = 0; b < gxp; ++b) s += partial[((size_t)enc * gxp + b) * 2 * SGRAD + rem];
    grads[idx] = s;
}

__global__ void fill_u32_kernel(unsigned* p, unsigned v, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

int sm_count(int* sms) {
    int dev = 0;
    MGV_CUDA(cudaGetDevice(&dev));
    MGV_CUDA(cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev));
    return MGV_OK;
}

int chunk_tiles() {
    const char* e = getenv("MGV_STRUCT_CHUNK");
    const int v = e ? atoi(e) : 0;
    return v > 0 ? v : CHUNK_TILES_DEFAULT;
}

}  // namespace

extern "C" size_t mgv_struct_bwd_workspace_bytes(int64_t N, int32_t num_enc) {
    int sms = 148;
    sm_count(&sms);
    const int64_t ntiles = (N + TM - 1) / TM;
    const int CHUNK_TILES = chunk_tiles();
    const int64_t cap = ntiles < CHUNK_TILES ? ntiles : CHUNK_TILES;
    size_t b = mgv_struct_image_bytes(num_enc) + 256;
    b += 4 * mgv_align_up((size_t)num_enc * N * D * 4 + 256, 256);
    b += mgv_align_up((size_t)sms * 2 * SGRAD * 4 + 256, 256);
    b += mgv_align_up((size_t)num_enc * cap * DG_TILE_BYTES + 1024, 1024);
    b += mgv_align_up((size_t)num_enc * cap * 4 + 256, 256);
    const int64_t chunks = (ntiles + CHUNK_TILES - 1) / CHUNK_TILES;
    b += mgv_align_up((size_t)(chunks > 0 ? chunks : 1) * 2 * 4 + 256, 256) + 4096;   // smin words of one step (re-filled per step)
    return b;
}

extern "C" int mgv_struct_encoder_bwd(const mgv_schedule* sch, int32_t num_enc, int32_t rounds, int32_t layernorm,
                                      int32_t feat, const float* x, const float* weights, const void* tiles,
                                      const float* gout, float* grads, void* ws, size_t ws_bytes,
                                      int32_t precision, mgv_stream_t stream) {
    cudaStream_t st = (cudaStream_t)stream;
    MGV_REQUIRE(sch != nullptr, "struct encoder: null schedule");
    MGV_REQUIRE(num_enc >= 1 && num_enc <= 2, "struct encoder: num_enc must be 1 or 2");
    MGV_REQUIRE(rounds >= 1, "struct encoder: rounds must be >= 1");
    MGV_REQUIRE(feat >= 0 && feat <= MGV_MAX_FEAT, "struct encoder: dim_feature %d > %d", feat, MGV_MAX_FEAT);
    const int N = sch->N;
    MGV_CUDA(cudaMemsetAsync(grads, 0, (size_t)num_enc * 2 * SGRAD * sizeof(float), st));
    if (N == 0) return MGV_OK;
    MGV_REQUIRE(sch->deg_order_in && sch->deg_order_out && sch->tile_cost_in && sch->tile_cost_out && sch->gdesc_in && sch->gdesc_out,
                "struct encoder: the schedule carries no degree order (mgv_build_degree_order)");
    MGV_REQUIRE(tiles != nullptr, "mgv_struct_encoder_bwd: the operand tiles saved by mgv_struct_encoder_fwd are required (tiles == NULL)");
    if (ws_bytes < mgv_struct_bwd_workspace_bytes(N, num_enc)) {
        mgv_set_error("mgv_struct_encoder_bwd: workspace %zu < %zu bytes", ws_bytes, mgv_struct_bwd_workspace_bytes(N, num_enc));
        return MGV_ERR_WORKSPACE;
    }
    int sms = 0;
    int rc = sm_count(&sms);
    if (rc != MGV_OK) return rc;
    const int ntiles = (N + TM - 1) / TM;
    const int CHUNK_TILES = chunk_tiles();
    const int cap = ntiles < CHUNK_TILES ? ntiles : CHUNK_TILES;
    const int chunks = (ntiles + CHUNK_TILES - 1) / CHUNK_TILES;
    const int gxp = sms / num_enc > 0 ? sms / num_enc : 1;
    const int steps = 2 * rounds;
    const size_t slot = (size_t)N * D;

    MgvArena a(ws, ws_bytes);
    uint8_t* image = a.take<uint8_t>((size_t)num_enc * 2 * IMG_BYTES);
    float* part[2];
    float* agg[2];
    part[0] = a.take<float>((size_t)num_enc * slot); part[1] = a.take<float>((size_t)num_enc * slot);
    agg[0] = a.take<float>((size_t)num_enc * slot); agg[1] = a.take<float>((size_t)num_enc * slot);
    float* partial = a.take<float>((size_t)num_enc * gxp * 2 * SGRAD);
    a.off = mgv_align_up(a.off, 1024);
    uint8_t* dgbuf = a.take<uint8_t>((size_t)num_enc * cap * DG_TILE_BYTES);
    float* scales = a.take<float>((size_t)num_enc * cap);
    unsigned* smin = a.take<unsigned>((size_t)chunks * 2);
    MGV_REQUIRE(a.ok(), "mgv_struct_encoder_bwd: workspace layout overflow");
    MGV_REQUIRE(precision == 0 || precision == 1, "struct encoder: precision must be 0 (fp32-accurate) or 1 (bf16)");
    rc = mgv_struct_build_image(weights, num_enc, image, precision, st);
    if (rc != MGV_OK) return rc;
    MGV_CUDA(cudaMemsetAsync(partial, 0, (size_t)num_enc * gxp * 2 * SGRAD * sizeof(float), st));
    const bool lowp = precision == 1;
    const void* pw_fn = lowp ? (const void*)struct_bwd_pw_kernel<true> : (const void*)struct_bwd_pw_kernel<false>;
    const void* wg_fn = lowp ? (const void*)struct_bwd_wgrad_kernel<true> : (const void*)struct_bwd_wgrad_kernel<false>;
    MGV_CUDA(cudaFuncSetAttribute(pw_fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P_SMEM));
    MGV_CUDA(cudaFuncSetAttribute(wg_fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)W_SMEM));

    for (int k = steps; k >= 1; --k) {
        const int dir = (k & 1) ? 0 : 1;
        fill_u32_kernel<<<(chunks * 2 + 63) / 64, 64, 0, st>>>(smin, 0x7f000000u, chunks * 2);
        mgv_count_launches(1);
        for (int ch = 0; ch < chunks; ++ch) {
            const int tb = ch * CHUNK_TILES, te = (tb + CHUNK_TILES < ntiles) ? tb + CHUNK_TILES : ntiles;
            int gx = gxp;
            if (gx > te - tb) gx = te - tb;
            BwdTC p{};
            p.N = N; p.feat = feat; p.layernorm = layernorm; p.first = (k == 1); p.last = (k == steps); p.dir = dir;
            p.tile_beg = tb; p.tile_end = te;
            p.ptr = dir == 0 ? sch->in_ptr : sch->out_ptr;
            p.idx = dir == 0 ? sch->in_src : sch->out_pack;
            p.order = dir == 0 ? sch->deg_order_in : sch->deg_order_out;
            p.gdesc = dir == 0 ? sch->gdesc_in : sch->gdesc_out;
            p.tile_cost = dir == 0 ? sch->tile_cost_in : sch->tile_cost_out;
            p.x = x;
            p.image = image + (size_t)dir * IMG_BYTES;
            p.gout = gout;
            p.in_part = part[k & 1]; p.in_agg = agg[k & 1];
            p.out_part = part[(k - 1) & 1]; p.out_agg = agg[(k - 1) & 1];
            p.tiles = (const uint8_t*)tiles + (size_t)(k - 1) * ntiles * A_TILE_BYTES;
            p.tiles_enc_stride = (size_t)steps * ntiles * A_TILE_BYTES;
            p.dgbuf = dgbuf; p.scales = scales; p.smin = smin + 2 * ch;
            p.partial = partial; p.gxp = gxp; p.chunk_cap = cap;
            p.trace = (k == 2 && ch == 0 && !getenv("MGV_TRACE_WGRAD")) ? mgv_debug_trace() : nullptr;
            if (lowp) struct_bwd_pw_kernel<true><<<dim3(gx, num_enc), THREADS, P_SMEM, st>>>(p);
            else struct_bwd_pw_kernel<false><<<dim3(gx, num_enc), THREADS, P_SMEM, st>>>(p);
            WgTC w{};
            w.ntiles = te - tb; w.chunk_cap = cap; w.dir = dir; w.gxp = gxp;
            w.tiles = p.tiles; w.tiles_enc_stride = p.tiles_enc_stride; w.tile_base = tb;
            w.dgbuf = dgbuf; w.scales = scales; w.smin = smin + 2 * ch; w.partial = partial;
            w.trace = (k == 2 && ch == 0 && getenv("MGV_TRACE_WGRAD")) ? mgv_debug_trace() : nullptr;
            if (lowp) struct_bwd_wgrad_kernel<true><<<dim3(gx, num_enc), W_THREADS, W_SMEM, st>>>(w);
            else struct_bwd_wgrad_kernel<false><<<dim3(gx, num_enc), W_THREADS, W_SMEM, st>>>(w);
            mgv_count_launches(2);
        }
    }
    const size_t total = (size_t)num_enc * 2 * SGRAD;
    struct_reduce_tc_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(partial, gxp, grads, num_enc);
    mgv_count_launches(1);
    return mgv_check_cuda(cudaGetLastError(), "mgv_struct_encoder_bwd");
}
