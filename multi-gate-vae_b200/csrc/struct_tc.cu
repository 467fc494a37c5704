// Struct encoder on the 5th-generation tensor cores: MultiGCNEncoder.forward (digae_layer.py:257-277)
// with AggConv (arch/gcn_conv.py:30-42), one fused kernel per half-round step:
//   gather-sum of neighbour states -> GRU_{70->64}([W agg + deg b || x], state) -> LayerNorm
// Step k = 1..2R uses in-neighbours when k is odd (aggr/update) and out-neighbours when k is even
// (aggr_r/update_r); LayerNorm parameters are shared by both directions (digae_layer.py:270,275).
// source_conv and target_conv (digae_layer.py:294-297) run batched: blockIdx.y = encoder.
//
// A step is ONE tile product per 128 nodes (the AggConv linear is pre-composed into the GRU input weights
// on the host, Wc = W_ih[:, :64] W, bc = W_ih[:, :64] b):
//     [agg(64) | h(64) | x(8) deg 1 (16)]  x  [Wc | W_hh | W_ih_x bc b_ih b_hh]^T  ->  r, z, gi_n, gh_n   (256 fp32 columns)
// issued as tcgen05.mma kind::f16 on fp16 hi/lo planes (csrc/mgv_tc.cuh) with the accumulator in tensor
// memory; biases and the degree term ride along as two extra K columns, so the epilogue is gates + LayerNorm.
//
// Persistent CTAs (one per SM, weights resident in shared memory for the whole launch), warp-specialised
// (8 epilogue + 16 gather + 1 MMA warp; the kernel is templated on the split):
//   gather      neighbour sums, own state and [x deg 1] -> fp16 hi/lo -> operand tile (UMMA layout), 2 rows per lane;
//               rows come in descending-degree order (mgv_build_degree_order) so a warp's lanes run equal trip counts;
//               in a training step the same chunks also go to the tile image in HBM that the backward recomputes from
//   MMA warp    one thread issues the MMAs of a tile once the tile is full; completion frees the tile (tcgen05.commit)
//   epilogue    two threads per node = TMEM lane (32 units each): tensor memory -> GRU gates -> LayerNorm -> state_k
//               (two accumulator buffers: the epilogue of tile t overlaps the gather and MMAs of tile t+1)
#include <stdlib.h>
#include "struct_layout.cuh"

namespace {
using namespace struct_layout;

constexpr uint32_t S_LN = A_X_LO + 4096;            // 128 floats
constexpr uint32_t S_EX = S_LN + 512;               // LayerNorm partial sums [2][128][2] floats
constexpr uint32_t S_BAR = S_EX + 2048;             // 7 mbarriers
constexpr uint32_t S_TMEM = S_BAR + 64;
constexpr uint32_t F_SMEM = S_TMEM + 64 + 1024;     // + alignment slack


struct StepTC {
    int N, feat, layernorm;
    const int* ptr;            // neighbour CSR of this step's direction
    const int* idx;
    const int* order;          // degree order of this direction (tile row -> node id)
    const int* gdesc;          // [N][4] row descriptors of the degree order
    const unsigned* tile_cost; // [ntiles + 1] exclusive prefix of the tile cost model
    const float* x;            // [N][feat]
    const uint8_t* image;      // weight image of (enc 0, this dir); encoder stride 2 * IMG_BYTES
    const float* prev;         // state_{k-1}, enc 0
    float* next;               // state_k, enc 0
    size_t enc_stride;         // floats between encoders in the states buffer
    uint8_t* tiles;            // optional: operand tiles of this step, enc 0 ([tile][A_TILE_BYTES]); saved for the backward
    size_t tiles_enc_stride;   // bytes between encoders in the tile buffer
    long long* trace;          // optional [CTA][16 tiles][16] clock64 samples (dev tool), may be null
};
#define TRACE(slot) do { if (p.trace && it < 16) p.trace[(((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 16 + it) * 16 + (slot)] = clock64(); } while (0)


// r, z, gi_n, gh_n of 4 consecutive units: columns c, 64 + c, 128 + c, 192 + c (4 each) of the accumulator
__device__ __forceinline__ void tmem_ld4x4(uint32_t taddr, float (&v)[16]) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
#pragma unroll
    for (int k = 0; k < 4; ++k)
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];"
                     : "=r"(r[4 * k]), "=r"(r[4 * k + 1]), "=r"(r[4 * k + 2]), "=r"(r[4 * k + 3]) : "r"(taddr + 64u * k) : "memory");
}
// `gt` (optional): the same 16-byte chunks also go to the tile image in HBM that the backward recomputes from
// (a row's 8 chunks are one 128-byte line, so a warp's 4 rows write 4 full lines per plane).
template <bool LOWP>
__device__ __forceinline__ void split_store_sw128(uint32_t hi_base, uint32_t lo_base, int row, int c, const float (&v)[8],
                                                  uint8_t* gt = nullptr, uint32_t g_hi = 0, uint32_t g_lo = 0, uint64_t pol = 0) {
    uint4 hi, lo;
    tc::split8p<LOWP>(v, hi, lo);
    const uint32_t off = tc::sw128_off(row, c);
    tc::st_shared_v4(hi_base + off, hi);
    if (!LOWP) tc::st_shared_v4(lo_base + off, lo);
    if (gt) {       // read once, much later, by the backward: do not let it displace the state rows in L2
        tc::stg_v4_hint(gt + g_hi + off, hi, pol);
        if (!LOWP) tc::stg_v4_hint(gt + g_lo + off, lo, pol);
    }
}

// ======================================================================================= weight image
// natural fp32 block -> fp16 hi/lo planes in the UMMA layouts the step kernels consume.
template <bool LOWP>
__global__ void struct_image_kernel(const float* __restrict__ pack, uint8_t* __restrict__ image, int blocks) {
    const int blk = blockIdx.y;
    if (blk >= blocks) return;
    const float* W = pack + (size_t)blk * SPACK;
    uint8_t* img = image + (size_t)blk * IMG_BYTES;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    float v[8];
    uint4 hi, lo;
    if (i < G3 * 8) {                                  // Wc: 192 rows x 8 chunks
        const int o = i >> 3, c = i & 7;
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] = W[O_WCX + o * LDC + c * 8 + e];
        tc::split8p<LOWP>(v, hi, lo);
        const uint32_t off = tc::sw128_off(o, c);
        *reinterpret_cast<uint4*>(img + WC_HI + off) = hi;
        *reinterpret_cast<uint4*>(img + WC_LO + off) = lo;
    } else if (i < 2 * G3 * 8) {                       // Whh
        const int j = i - G3 * 8, o = j >> 3, c = j & 7;
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] = W[O_WHH + o * LDM + c * 8 + e];
        tc::split8p<LOWP>(v, hi, lo);
        const uint32_t off = tc::sw128_off(o, c);
        *reinterpret_cast<uint4*>(img + WHH_HI + off) = hi;
        *reinterpret_cast<uint4*>(img + WHH_LO + off) = lo;
    } else if (i < 2 * G3 * 8 + 256 * 2) {             // [W_ih_x | bc | bias] : 256 accumulator columns x 16
        const int j = i - 2 * G3 * 8, n = j >> 1, c = j & 1;
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] = 0.f;
        if (c == 0) {
            if (n < G3) {
#pragma unroll
                for (int e = 0; e < 8; ++e) v[e] = W[O_WCX + n * LDC + D + e];
            }
        } else {
            if (n < 2 * D) { v[0] = W[O_BC + n]; v[1] = W[O_BIH + n] + W[O_BHH + n]; }     // r, z: merged biases
            else if (n < G3) { v[0] = W[O_BC + n]; v[1] = W[O_BIH + n]; }                   // gi_n
            else { v[1] = W[O_BHH + n - D]; }                                               // gh_n
        }
        tc::split8p<LOWP>(v, hi, lo);
        const uint32_t off = tc::plain16_off(n, c);
        *reinterpret_cast<uint4*>(img + WX_HI + off) = hi;
        *reinterpret_cast<uint4*>(img + WX_LO + off) = lo;
    } else if (i < 2 * G3 * 8 + 256 * 2 + 2 * D) {
        const int j = i - (2 * G3 * 8 + 256 * 2);
        reinterpret_cast<float*>(img + IMG_W)[j] = W[O_LNW + j];      // ln_w then ln_b (contiguous in the block)
    }
}

// ======================================================================================= forward step
// RPL = rows per gather lane (4 -> 8 gather warps, 2 -> 16: twice the loads in flight), EW = epilogue warps (4: one thread
// per node; 8: two threads per node, 32 units each, LayerNorm row sums exchanged through shared memory).
template <bool LOWP, int RPL, int EW>
__global__ void __launch_bounds__((EW + 128 / (4 * RPL) + 1) * 32, 1) struct_fwd_tc_kernel(const StepTC p) {
    constexpr int EPI_WARPS = EW, GATHER_WARPS = 128 / (4 * RPL), UPT = 64 / (EW / 4);     // units per epilogue thread
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const uint32_t sbase = (tc::smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* sgen = smem_raw + (sbase - tc::smem_u32(smem_raw));
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int enc = blockIdx.y;
    const float* prev = p.prev + (size_t)enc * p.enc_stride;
    float* next = p.next + (size_t)enc * p.enc_stride;
    const uint8_t* image = p.image + (size_t)enc * 2 * IMG_BYTES;

    const uint32_t bar_a_full = sbase + S_BAR, bar_a_empty = bar_a_full + 8;
    const uint32_t bar_acc_full = bar_a_full + 16, bar_acc_empty = bar_a_full + 32;      // [2] each
    const uint32_t bar_w = bar_a_full + 48;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sgen + S_TMEM);
    float* s_ln = reinterpret_cast<float*>(sgen + S_LN);

    // ---- one-time setup: barriers, weights -> shared memory (bulk async copy, overlaps the first gather), tensor memory
    if (tid == 0) {
        tc::mbar_init(bar_a_full, GATHER_WARPS * 32);
        tc::mbar_init(bar_a_empty, 1);
        tc::mbar_init(bar_acc_full, 1);
        tc::mbar_init(bar_acc_full + 8, 1);
        tc::mbar_init(bar_acc_empty, EPI_WARPS * 32);
        tc::mbar_init(bar_acc_empty + 8, EPI_WARPS * 32);
        tc::mbar_init(bar_w, 1);
        tc::fence_barrier_init();
        tc::mbar_expect_tx(bar_w, IMG_W);
#pragma unroll 1
        for (uint32_t o = 0; o < IMG_W; o += 16384u) tc::bulk_g2s(sbase + o, image + o, 16384u, bar_w);
    }
    if (tid < 2 * D) s_ln[tid] = __ldg(reinterpret_cast<const float*>(image + IMG_W) + tid);
    if (warp == 0) tc::tmem_alloc(tmem_slot, 512);
    // contiguous tile range of equal modelled cost for this CTA (tiles are in descending-degree order)
    const int ntiles = (p.N + TM - 1) / TM;
    int tile_beg, tile_end;
    {
        const unsigned long long total = p.tile_cost[ntiles];
        const unsigned lo = (unsigned)(total * blockIdx.x / gridDim.x), hi = (unsigned)(total * (blockIdx.x + 1) / gridDim.x);
        tile_beg = tc::warp_lower_bound(p.tile_cost, ntiles, lo, lane);
        tile_end = tc::warp_lower_bound(p.tile_cost, ntiles, hi, lane);
        // the ranges must partition [0, ntiles) whatever the search returns: first CTA starts at 0, last ends at ntiles
        if (blockIdx.x == 0) tile_beg = 0;
        if (blockIdx.x == gridDim.x - 1) tile_end = ntiles;
        tile_beg = min(max(tile_beg, 0), ntiles);
        tile_end = min(max(tile_end, tile_beg), ntiles);
    }
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem = *tmem_slot;

    if (warp >= EPI_WARPS && warp < EPI_WARPS + GATHER_WARPS) {
        // ===================================================================== gather
        // lane = (row group rg, 16-byte chunk c): 8 lanes cover one 256-byte state row; a lane owns RPL rows of the tile.
        const int gw = warp - EPI_WARPS, rg = lane >> 3, c = lane & 7;
        const int4* gdesc = reinterpret_cast<const int4*>(p.gdesc);
        const uint64_t pol_stream = tc::l2_policy_evict_first();
        int4 dn[RPL];                                   // row descriptors of the NEXT tile, loaded one tile ahead
#pragma unroll
        for (int ps = 0; ps < RPL; ++ps) {
            const int r = tile_beg * TM + gw * (4 * RPL) + ps * 4 + rg;
            dn[ps] = (tile_beg < tile_end && r < p.N) ? __ldg(gdesc + r) : make_int4(-1, 0, 0, 0);
        }
        int it = 0;
        for (int tile = tile_beg; tile < tile_end; ++tile, ++it) {
            if (warp == EPI_WARPS && lane == 0) TRACE(0);
            uint8_t* gt = p.tiles ? p.tiles + (size_t)enc * p.tiles_enc_stride + (size_t)tile * A_TILE_BYTES : nullptr;
            // ---- loads into registers (overlap the previous tile's MMAs): own-state rows, the lane's feature element,
            //      first neighbour rows, second neighbour ids, next tile's descriptors
            int node[RPL], beg[RPL], cnt[RPL], jn[RPL];
#pragma unroll
            for (int ps = 0; ps < RPL; ++ps) { node[ps] = dn[ps].x; beg[ps] = dn[ps].y; cnt[ps] = dn[ps].z; jn[ps] = dn[ps].w; }
            float4 ha[RPL], hb[RPL], va[RPL], vb[RPL];
            float xe[RPL];
            int maxc = 0;
#pragma unroll
            for (int ps = 0; ps < RPL; ++ps) {
                ha[ps] = make_float4(0.f, 0.f, 0.f, 0.f); hb[ps] = ha[ps]; va[ps] = ha[ps]; vb[ps] = ha[ps];
                xe[ps] = 0.f;
                maxc = max(maxc, cnt[ps]);
                if (node[ps] >= 0) {
                    ha[ps] = mgv_ld4(prev + (size_t)node[ps] * D + c * 8);
                    hb[ps] = mgv_ld4(prev + (size_t)node[ps] * D + c * 8 + 4);
                    if (c < p.feat) xe[ps] = p.x[(size_t)node[ps] * p.feat + c];
                }
                if (cnt[ps] > 0) {
                    va[ps] = mgv_ld4(prev + (size_t)jn[ps] * D + c * 8);
                    vb[ps] = mgv_ld4(prev + (size_t)jn[ps] * D + c * 8 + 4);
                }
                if (cnt[ps] > 1) jn[ps] = p.idx[beg[ps] + 1] & NODE_MASK;
            }
#pragma unroll
            for (int ps = 0; ps < RPL; ++ps) {
                const int r = (tile + 1) * TM + gw * (4 * RPL) + ps * 4 + rg;
                dn[ps] = (tile + 1 < tile_end && r < p.N) ? __ldg(gdesc + r) : make_int4(-1, 0, 0, 0);
            }
            if (warp == EPI_WARPS && lane == 0) TRACE(1);
            tc::mbar_wait(bar_a_empty, (uint32_t)((it & 1) ^ 1));            // previous tile's MMAs have read the stage
            if (warp == EPI_WARPS && lane == 0) TRACE(2);
            // ---- own state rows and the [x deg 1] block
#pragma unroll
            for (int ps = 0; ps < RPL; ++ps) {
                const int row = gw * (4 * RPL) + ps * 4 + rg;
                const float h8[8] = {ha[ps].x, ha[ps].y, ha[ps].z, ha[ps].w, hb[ps].x, hb[ps].y, hb[ps].z, hb[ps].w};
                split_store_sw128<LOWP>(sbase + A_H_HI, sbase + A_H_LO, row, c, h8, gt, A_H_HI - A_AGG_HI, A_H_LO - A_AGG_HI, pol_stream);
                float xv[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) xv[e] = __shfl_sync(0xffffffffu, xe[ps], (lane & 24) + e);   // features of this row
                if (c == 1) {
#pragma unroll
                    for (int e = 0; e < 8; ++e) xv[e] = 0.f;
                    if (node[ps] >= 0) { xv[0] = (float)cnt[ps]; xv[1] = 1.0f; }
                }
                if (c < 2) {
                    uint4 hi, lo;
                    tc::split8p<LOWP>(xv, hi, lo);
                    const uint32_t off = tc::plain16_off(row, c);
                    tc::st_shared_v4(sbase + A_X_HI + off, hi);
                    if (!LOWP) tc::st_shared_v4(sbase + A_X_LO + off, lo);
                    if (gt) {
                        tc::stg_v4_hint(gt + (A_X_HI - A_AGG_HI) + off, hi, pol_stream);
                        if (!LOWP) tc::stg_v4_hint(gt + (A_X_LO - A_AGG_HI) + off, lo, pol_stream);
                    }
                }
            }
            if (warp == EPI_WARPS && lane == 0) TRACE(3);
            // ---- neighbour sums: one neighbour of each of the lane's 4 rows per trip (8 x 16-byte loads in flight),
            //      next trip's neighbour ids prefetched
            float acc[RPL][8];
#pragma unroll
            for (int ps = 0; ps < RPL; ++ps) {
                acc[ps][0] = va[ps].x; acc[ps][1] = va[ps].y; acc[ps][2] = va[ps].z; acc[ps][3] = va[ps].w;
                acc[ps][4] = vb[ps].x; acc[ps][5] = vb[ps].y; acc[ps][6] = vb[ps].z; acc[ps][7] = vb[ps].w;
            }
            for (int sl = 1; sl < maxc; ++sl) {
                int j[RPL];
#pragma unroll
                for (int ps = 0; ps < RPL; ++ps) {
                    j[ps] = jn[ps];
                    if (sl + 1 < cnt[ps]) jn[ps] = p.idx[beg[ps] + sl + 1] & NODE_MASK;
                }
#pragma unroll
                for (int ps = 0; ps < RPL; ++ps) {
                    va[ps] = make_float4(0.f, 0.f, 0.f, 0.f); vb[ps] = va[ps];
                    if (sl < cnt[ps]) {
                        va[ps] = mgv_ld4(prev + (size_t)j[ps] * D + c * 8);
                        vb[ps] = mgv_ld4(prev + (size_t)j[ps] * D + c * 8 + 4);
                    }
                }
#pragma unroll
                for (int ps = 0; ps < RPL; ++ps) {
                    acc[ps][0] += va[ps].x; acc[ps][1] += va[ps].y; acc[ps][2] += va[ps].z; acc[ps][3] += va[ps].w;
                    acc[ps][4] += vb[ps].x; acc[ps][5] += vb[ps].y; acc[ps][6] += vb[ps].z; acc[ps][7] += vb[ps].w;
                }
            }
#pragma unroll
            for (int ps = 0; ps < RPL; ++ps)
                split_store_sw128<LOWP>(sbase + A_AGG_HI, sbase + A_AGG_LO, gw * (4 * RPL) + ps * 4 + rg, c, acc[ps], gt, 0u, A_AGG_LO - A_AGG_HI, pol_stream);
            if (warp == EPI_WARPS && lane == 0) TRACE(4);
            tc::fence_async_smem();
            tc::mbar_arrive(bar_a_full);
        }
    } else if (warp == EPI_WARPS + GATHER_WARPS) {
        // ===================================================================== MMA issue (one thread)
        if (lane == 0) {
            int it = 0;
            for (int tile = tile_beg; tile < tile_end; ++tile, ++it) {
                const int b = it & 1;
                if (it == 0) tc::mbar_wait(bar_w, 0u);                              // weight image has landed
                TRACE(5);
                tc::mbar_wait(bar_acc_empty + 8 * b, (uint32_t)(((it >> 1) & 1) ^ 1));   // epilogue drained this buffer
                tc::mbar_wait(bar_a_full, (uint32_t)(it & 1));
                tc::fence_after_sync();
                TRACE(6);
                const uint32_t d = tmem + (uint32_t)b * 256u;
                // [x deg 1] block first: initialises all 256 columns (biases, degree term, feature term)
                tc::mma3p<LOWP>(d, tc::desc_k_plain16(sbase + A_X_HI), tc::desc_k_plain16(sbase + A_X_LO),
                         tc::desc_k_plain16(sbase + WX_HI), tc::desc_k_plain16(sbase + WX_LO), tc::make_idesc(128, 256, false, false, LOWP), 0u);
#pragma unroll
                for (int j = 0; j < 4; ++j)      // h . Whh[r, z]^T -> r, z
                    tc::mma3p<LOWP>(d, tc::desc_k_sw128(sbase + A_H_HI + 32 * j), tc::desc_k_sw128(sbase + A_H_LO + 32 * j),
                             tc::desc_k_sw128(sbase + WHH_HI + 32 * j), tc::desc_k_sw128(sbase + WHH_LO + 32 * j),
                             tc::make_idesc(128, 128, false, false, LOWP), 1u);
#pragma unroll
                for (int j = 0; j < 4; ++j)      // h . Whh[n]^T -> gh_n
                    tc::mma3p<LOWP>(d + 192u, tc::desc_k_sw128(sbase + A_H_HI + 32 * j), tc::desc_k_sw128(sbase + A_H_LO + 32 * j),
                             tc::desc_k_sw128(sbase + WHH_HI + 16384 + 32 * j), tc::desc_k_sw128(sbase + WHH_LO + 16384 + 32 * j),
                             tc::make_idesc(128, 64, false, false, LOWP), 1u);
#pragma unroll
                for (int j = 0; j < 4; ++j)      // agg . Wc^T -> r, z, gi_n
                    tc::mma3p<LOWP>(d, tc::desc_k_sw128(sbase + A_AGG_HI + 32 * j), tc::desc_k_sw128(sbase + A_AGG_LO + 32 * j),
                             tc::desc_k_sw128(sbase + WC_HI + 32 * j), tc::desc_k_sw128(sbase + WC_LO + 32 * j),
                             tc::make_idesc(128, 192, false, false, LOWP), 1u);
                tc::mma_commit(bar_a_empty);
                tc::mma_commit(bar_acc_full + 8 * b);
                TRACE(7);
            }
        }
    } else if (warp < EPI_WARPS) {
        // ===================================================================== epilogue: EW / 4 threads per tile row = TMEM lane
        // Warps q, 4 + q, .. own lanes 32 q .. 32 q + 31; warp group wg = warp / 4 handles units UPT wg .. of its row.
        // Gates are read 4 units at a time (r, z, gi_n, gh_n -> 16 registers) with the next chunk's tensor-memory loads
        // in flight while the current chunk is computed.
        const int wg = warp >> 2, row = (warp & 3) * 32 + lane, u0 = UPT * wg;
        float* s_ex = reinterpret_cast<float*>(sgen + S_EX);          // [2 quantities][2 warp groups][128 rows]
        int it = 0;
        for (int tile = tile_beg; tile < tile_end; ++tile, ++it) {
            const int b = it & 1;
            const bool valid = tile * TM + row < p.N;
            const int node = valid ? p.order[tile * TM + row] : 0;
            float h[UPT];
            if (valid) {
#pragma unroll
                for (int ch = 0; ch < UPT / 8; ++ch) ldg8(prev + (size_t)node * D + u0 + 8 * ch, *reinterpret_cast<float(*)[8]>(&h[8 * ch]));
            } else {
#pragma unroll
                for (int e = 0; e < UPT; ++e) h[e] = 0.f;
            }
            if (tid == 0) TRACE(8);
            tc::mbar_wait(bar_acc_full + 8 * b, (uint32_t)((it >> 1) & 1));
            tc::fence_after_sync();
            if (tid == 0) TRACE(9);
            const uint32_t ta = tmem + (uint32_t)b * 256u + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)u0;
            float g0[16], g1[16];
            tmem_ld4x4(ta, g0);
#pragma unroll
            for (int ch = 0; ch < UPT / 4; ch += 2) {
                tc::tmem_ld_wait();
                tmem_ld4x4(ta + 4 * (ch + 1), g1);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    float r, z, n, hnb;
                    gru_gates(g0[e], g0[4 + e], g0[8 + e], g0[12 + e], r, z, n, hnb);
                    h[4 * ch + e] = fmaf(z, h[4 * ch + e] - n, n);          // (1 - z) n + z h
                }
                tc::tmem_ld_wait();
                if (ch + 2 < UPT / 4) tmem_ld4x4(ta + 4 * (ch + 2), g0);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    float r, z, n, hnb;
                    gru_gates(g1[e], g1[4 + e], g1[8 + e], g1[12 + e], r, z, n, hnb);
                    h[4 * (ch + 1) + e] = fmaf(z, h[4 * (ch + 1) + e] - n, n);
                }
            }
            tc::fence_before_sync();
            tc::mbar_arrive(bar_acc_empty + 8 * b);
            if (tid == 0) TRACE(10);
            if (p.layernorm) {
                float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
                for (int e = 0; e < UPT; e += 4) { s0 += h[e]; s1 += h[e + 1]; s2 += h[e + 2]; s3 += h[e + 3]; }
                float tot = (s0 + s1) + (s2 + s3);
                if (EW == 8) {
                    s_ex[wg * TM + row] = tot;
                    tc::named_bar_sync(1, EW * 32);
                    tot = s_ex[row] + s_ex[TM + row];
                }
                const float mean = tot * (1.0f / D);
                s0 = s1 = s2 = s3 = 0.f;
#pragma unroll
                for (int e = 0; e < UPT; e += 4) {
                    h[e] -= mean; h[e + 1] -= mean; h[e + 2] -= mean; h[e + 3] -= mean;
                    s0 = fmaf(h[e], h[e], s0); s1 = fmaf(h[e + 1], h[e + 1], s1);
                    s2 = fmaf(h[e + 2], h[e + 2], s2); s3 = fmaf(h[e + 3], h[e + 3], s3);
                }
                tot = (s0 + s1) + (s2 + s3);
                if (EW == 8) {
                    s_ex[(2 + wg) * TM + row] = tot;
                    tc::named_bar_sync(1, EW * 32);
                    tot = s_ex[2 * TM + row] + s_ex[3 * TM + row];
                }
                const float rstd = rsqrtf(tot * (1.0f / D) + LN_EPS);
#pragma unroll
                for (int e = 0; e < UPT; e += 4) {
                    const float4 w4 = *reinterpret_cast<const float4*>(s_ln + u0 + e), b4 = *reinterpret_cast<const float4*>(s_ln + D + u0 + e);
                    h[e] = fmaf(h[e] * rstd, w4.x, b4.x); h[e + 1] = fmaf(h[e + 1] * rstd, w4.y, b4.y);
                    h[e + 2] = fmaf(h[e + 2] * rstd, w4.z, b4.z); h[e + 3] = fmaf(h[e + 3] * rstd, w4.w, b4.w);
                }
            }
            if (valid) {
#pragma unroll
                for (int ch = 0; ch < UPT / 8; ++ch) stg8(next + (size_t)node * D + u0 + 8 * ch, *reinterpret_cast<float(*)[8]>(&h[8 * ch]));
            }
            if (tid == 0) TRACE(11);
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc(tmem, 512);
}

__global__ void fill_ones_kernel(float* p, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = 1.0f;
}

}  // namespace

static long long* g_trace = nullptr;
extern "C" void mgv_debug_set_trace(void* p) { g_trace = (long long*)p; }
long long* mgv_debug_trace() { return g_trace; }

size_t mgv_struct_image_bytes(int num_enc) { return mgv_align_up((size_t)num_enc * 2 * IMG_BYTES, 256); }

int mgv_struct_build_image(const float* weights, int num_enc, uint8_t* image, int precision, cudaStream_t st) {
    const int items = 2 * G3 * 8 + 256 * 2 + 2 * D;
    if (precision == 1) struct_image_kernel<true><<<dim3((items + 255) / 256, num_enc * 2), 256, 0, st>>>(weights, image, num_enc * 2);
    else struct_image_kernel<false><<<dim3((items + 255) / 256, num_enc * 2), 256, 0, st>>>(weights, image, num_enc * 2);
    mgv_count_launches(1);
    return mgv_check_cuda(cudaGetLastError(), "struct_image_kernel");
}

extern "C" size_t mgv_struct_fwd_workspace_bytes(int64_t N, int32_t num_enc) {
    (void)N;
    return mgv_struct_image_bytes(num_enc) + 1024;
}

extern "C" size_t mgv_struct_tiles_bytes(int64_t N, int32_t num_enc, int32_t rounds) {
    const size_t ntiles = (size_t)((N + TM - 1) / TM);
    return (size_t)num_enc * 2 * rounds * ntiles * A_TILE_BYTES;
}

extern "C" int mgv_struct_encoder_fwd(const mgv_schedule* sch, int32_t num_enc, int32_t rounds, int32_t layernorm,
                                      int32_t feat, const float* x, const float* weights, float* states, void* tiles,
                                      void* ws, size_t ws_bytes, int32_t precision, mgv_stream_t stream) {
    cudaStream_t st = (cudaStream_t)stream;
    MGV_REQUIRE(sch != nullptr, "struct encoder: null schedule");
    MGV_REQUIRE(precision == 0 || precision == 1, "struct encoder: precision must be 0 (fp32-accurate) or 1 (bf16)");
    MGV_REQUIRE(num_enc >= 1 && num_enc <= 2, "struct encoder: num_enc must be 1 or 2");
    MGV_REQUIRE(rounds >= 1, "struct encoder: rounds must be >= 1");
    MGV_REQUIRE(feat >= 0 && feat <= MGV_MAX_FEAT, "struct encoder: dim_feature %d > %d", feat, MGV_MAX_FEAT);
    const int N = sch->N;
    if (N == 0) return MGV_OK;
    MGV_REQUIRE(sch->deg_order_in && sch->deg_order_out && sch->tile_cost_in && sch->tile_cost_out && sch->gdesc_in && sch->gdesc_out,
                "struct encoder: the schedule carries no degree order (mgv_build_degree_order)");
    if (ws_bytes < mgv_struct_fwd_workspace_bytes(N, num_enc)) {
        mgv_set_error("mgv_struct_encoder_fwd: workspace %zu < %zu bytes", ws_bytes, mgv_struct_fwd_workspace_bytes(N, num_enc));
        return MGV_ERR_WORKSPACE;
    }
    MgvArena a(ws, ws_bytes);
    uint8_t* image = a.take<uint8_t>((size_t)num_enc * 2 * IMG_BYTES);
    int rc = mgv_struct_build_image(weights, num_enc, image, precision, st);
    if (rc != MGV_OK) return rc;
    const int steps = 2 * rounds;
    const size_t slot = (size_t)N * D;
    const size_t enc_stride = 2 * slot;
    // launch shape: 16 gather warps x 2 rows per lane + 8 epilogue warps (25 warps, 72 registers)
    MGV_CUDA(cudaFuncSetAttribute((const void*)struct_fwd_tc_kernel<false, 2, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)F_SMEM));
    MGV_CUDA(cudaFuncSetAttribute((const void*)struct_fwd_tc_kernel<true, 2, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)F_SMEM));
    int dev = 0, sms = 0;
    MGV_CUDA(cudaGetDevice(&dev));
    MGV_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int ntiles = (N + TM - 1) / TM;
    int gx = sms / num_enc;
    if (gx > ntiles) gx = ntiles;
    if (gx < 1) gx = 1;
    for (int e = 0; e < num_enc; ++e) {
        fill_ones_kernel<<<(unsigned)((slot + 255) / 256), 256, 0, st>>>(states + e * enc_stride, slot);
        mgv_count_launches(1);
    }
    const char* ts_env = getenv("MGV_TRACE_STEP");          // dev tool: which step's kernel records the phase trace
    const int trace_step = (ts_env && atoi(ts_env) > 0) ? atoi(ts_env) : steps;
    for (int k = 1; k <= steps; ++k) {
        const int dir = (k & 1) ? 0 : 1;
        StepTC p{};
        p.N = N; p.feat = feat; p.layernorm = layernorm;
        p.ptr = dir == 0 ? sch->in_ptr : sch->out_ptr;
        p.idx = dir == 0 ? sch->in_src : sch->out_pack;
        p.order = dir == 0 ? sch->deg_order_in : sch->deg_order_out;
        p.gdesc = dir == 0 ? sch->gdesc_in : sch->gdesc_out;
        p.tile_cost = dir == 0 ? sch->tile_cost_in : sch->tile_cost_out;
        p.x = x;
        p.image = image + (size_t)dir * IMG_BYTES;
        p.prev = states + (size_t)((k - 1) & 1) * slot;      // two slots, ping-pong: the last step (2 * rounds) writes slot 0
        p.next = states + (size_t)(k & 1) * slot;
        p.enc_stride = enc_stride;
        // tile buffer [enc][step][tile][A_TILE_BYTES] (fp16 hi/lo planes; bf16 mode writes its single bf16 plane into the hi slots)
        p.tiles = tiles ? (uint8_t*)tiles + (size_t)(k - 1) * ntiles * A_TILE_BYTES : nullptr;
        p.tiles_enc_stride = (size_t)steps * ntiles * A_TILE_BYTES;
        p.trace = (k == trace_step) ? g_trace : nullptr;
        if (precision == 1) struct_fwd_tc_kernel<true, 2, 8><<<dim3(gx, num_enc), 25 * 32, F_SMEM, st>>>(p);
        else struct_fwd_tc_kernel<false, 2, 8><<<dim3(gx, num_enc), 25 * 32, F_SMEM, st>>>(p);
        mgv_count_launches(1);
    }
    return mgv_check_cuda(cudaGetLastError(), "mgv_struct_encoder_fwd");
}
