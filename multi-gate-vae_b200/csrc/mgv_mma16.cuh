// Warp-level tensor-core tiles on fp16 hi/lo planes: mma.sync m16n8k16 (fp16 x fp16 -> fp32) with the same
// three-product scheme as the tcgen05 path (mgv_tc.cuh): c += a_lo b_hi + a_hi b_lo + a_hi b_hi, both operands
// pre-split into two fp16 planes in shared memory ONCE (when the tile is written), so fragment loads are plain
// ldmatrix with no conversion work.  Used by the kernels whose tiles are too small / too irregular for a
// 128-row UMMA tile (struct encoder backward, level sweep).
//
// Shared-memory tiles are arrays of __half with a row stride (in halves) that is a multiple of 8 and whose byte
// size is 16 mod 32 modulo 128 (72, 88, 264, ...): every ldmatrix row address is 16-byte aligned and the 8 rows
// of a matrix land in distinct bank groups.
//
// Fragment ownership (PTX ISA, mma.m16n8k16 .f16): g = lane / 4, t = lane % 4
//   A (16x16, row): a0 (g, 2t..2t+1)  a1 (g+8, 2t..)  a2 (g, 2t+8..)  a3 (g+8, 2t+8..)
//   B (16x8,  col): b0 (k = 2t..2t+1, n = g)   b1 (k = 2t+8.., n = g)
//   C (16x8)      : c0 (g, 2t)  c1 (g, 2t+1)  c2 (g+8, 2t)  c3 (g+8, 2t+1)
#pragma once
#include <cuda_fp16.h>
#include "mgv_common.cuh"

namespace m16 {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ uint32_t pack_f16x2_sat(float e0, float e1) {
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(e1), "f"(e0));
    return r;
}
// two floats -> packed (hi, hi) and (lo, lo); element 0 in the low half-word
__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
    hi = pack_f16x2_sat(a, b);
    const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hi));
    lo = pack_f16x2_sat(a - hf.x, b - hf.y);
}
// bf16 mode (precision = 1): ONE plane, bf16 operands, fp32 accumulate -- the "stated tolerance" configuration.
__device__ __forceinline__ uint32_t pack_bf16x2(float e0, float e1) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(e1), "f"(e0));
    return r;
}
template <bool LOWP>
__device__ __forceinline__ void split2p(float a, float b, uint32_t& hi, uint32_t& lo) {
    if (LOWP) { hi = pack_bf16x2(a, b); lo = 0u; }
    else split2(a, b, hi, lo);
}
__device__ __forceinline__ float2 join2(uint32_t hi, uint32_t lo) {
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&hi));
    const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&lo));
    return make_float2(a.x + b.x, a.y + b.y);
}

__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t (&r)[4]) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t (&r)[4]) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x2(uint32_t addr, uint32_t (&r)[2]) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x2_t(uint32_t addr, uint32_t (&r)[2]) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(addr));
}
__device__ __forceinline__ void mma(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

__device__ __forceinline__ void mma_bf16(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

// Per-lane byte offset (inside a plane) of the ldmatrix row this lane addresses.
//   A, not transposed: storage S[m][k] (k contiguous)      A(m, k) = S[m0 + m][k0 + k]
//   A, transposed    : storage S[k][m] (m contiguous)      A(m, k) = S[k0 + k][m0 + m]
template <bool TRANS>
__device__ __forceinline__ uint32_t a_lane_off(int ld, int m0, int k0, int lane) {
    const int i = lane >> 3, r = lane & 7;
    return TRANS ? (uint32_t)(((k0 + (i >> 1) * 8 + r) * ld + m0 + (i & 1) * 8) * 2)
                 : (uint32_t)(((m0 + (i & 1) * 8 + r) * ld + k0 + (i >> 1) * 8) * 2);
}
//   B, NK: storage S[n][k] (k contiguous; an nn.Linear weight used as y = x W^T)    B(k, n) = S[n0 + n][k0 + k]
//   B, KN: storage S[k][n] (n contiguous)                                            B(k, n) = S[k0 + k][n0 + n]
// One ldmatrix.x4 fetches the B fragments of TWO consecutive k-steps (k0 .. k0+31) of one 8-column tile.
template <bool KN>
__device__ __forceinline__ uint32_t b_lane_off(int ld, int k0, int n0, int lane) {
    const int i = lane >> 3, r = lane & 7;
    return KN ? (uint32_t)(((k0 + i * 8 + r) * ld + n0) * 2) : (uint32_t)(((n0 + r) * ld + k0 + i * 8) * 2);
}

// c[mt][nt] += A[16 mt .., 16 KSTEPS) * B[.., n0[nt] ..)  for one warp; planes given as shared-memory byte addresses.
// A rows (or storage columns when A_TRANS) start at am0 + 16 mt; its K range starts at ak0; B's K range at bk0.
// The three products go to separate accumulator chains when MT * NT is small (more independent MMAs in flight).
template <int MT, int NT, int KSTEPS, bool A_TRANS, bool B_KN, bool LOWP = false>
__device__ __forceinline__ void warp_gemm(float (&c)[MT][NT][4], uint32_t a_hi, uint32_t a_lo, int lda, int am0, int ak0,
                                          uint32_t b_hi, uint32_t b_lo, int ldb, const int (&n0)[NT], int bk0, int lane) {
    constexpr bool SPLIT = !LOWP && (MT * NT <= 2);
    uint32_t aoff[MT], boff[NT];
#pragma unroll
    for (int mt = 0; mt < MT; ++mt) aoff[mt] = a_lane_off<A_TRANS>(lda, am0 + 16 * mt, ak0, lane);
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) boff[nt] = b_lane_off<B_KN>(ldb, bk0, n0[nt], lane);
    const uint32_t astep = A_TRANS ? (uint32_t)(16 * lda * 2) : 32u;
    const uint32_t bstep = B_KN ? (uint32_t)(16 * ldb * 2) : 32u;
    float c1[SPLIT ? MT : 1][SPLIT ? NT : 1][4], c2[SPLIT ? MT : 1][SPLIT ? NT : 1][4];
    if (SPLIT) {
#pragma unroll
        for (int i = 0; i < MT; ++i)
#pragma unroll
            for (int j = 0; j < NT; ++j)
#pragma unroll
                for (int e = 0; e < 4; ++e) { c1[i][j][e] = 0.f; c2[i][j][e] = 0.f; }
    }
#pragma unroll
    for (int kp = 0; kp < (KSTEPS + 1) / 2; ++kp) {
        uint32_t bhi[NT][4], blo[NT][4];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            if (2 * kp + 1 < KSTEPS) {
                if (B_KN) { ldsm_x4_t(b_hi + boff[nt] + 2 * kp * bstep, bhi[nt]); if (!LOWP) ldsm_x4_t(b_lo + boff[nt] + 2 * kp * bstep, blo[nt]); }
                else { ldsm_x4(b_hi + boff[nt] + 2 * kp * bstep, bhi[nt]); if (!LOWP) ldsm_x4(b_lo + boff[nt] + 2 * kp * bstep, blo[nt]); }
            } else {                                   // odd tail: one k-step (lanes 16..31 re-address rows of the first half)
                uint32_t t2[2];
                const uint32_t o = boff[nt] - (B_KN ? (uint32_t)(((lane >> 4) * 16) * ldb * 2) : (uint32_t)((lane >> 4) * 32));
                blo[nt][0] = blo[nt][1] = 0u;
                if (B_KN) { ldsm_x2_t(b_hi + o + 2 * kp * bstep, t2); bhi[nt][0] = t2[0]; bhi[nt][1] = t2[1]; if (!LOWP) { ldsm_x2_t(b_lo + o + 2 * kp * bstep, t2); blo[nt][0] = t2[0]; blo[nt][1] = t2[1]; } }
                else { ldsm_x2(b_hi + o + 2 * kp * bstep, t2); bhi[nt][0] = t2[0]; bhi[nt][1] = t2[1]; if (!LOWP) { ldsm_x2(b_lo + o + 2 * kp * bstep, t2); blo[nt][0] = t2[0]; blo[nt][1] = t2[1]; } }
                bhi[nt][2] = bhi[nt][3] = blo[nt][2] = blo[nt][3] = 0u;
            }
        }
#pragma unroll
        for (int kk = 0; kk < 2; ++kk) {
            const int ks = 2 * kp + kk;
            if (ks < KSTEPS) {
                uint32_t ahi[MT][4], alo[MT][4];
#pragma unroll
                for (int mt = 0; mt < MT; ++mt) {
                    if (A_TRANS) { ldsm_x4_t(a_hi + aoff[mt] + ks * astep, ahi[mt]); if (!LOWP) ldsm_x4_t(a_lo + aoff[mt] + ks * astep, alo[mt]); }
                    else { ldsm_x4(a_hi + aoff[mt] + ks * astep, ahi[mt]); if (!LOWP) ldsm_x4(a_lo + aoff[mt] + ks * astep, alo[mt]); }
                }
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    const uint32_t bh[2] = {bhi[nt][2 * kk], bhi[nt][2 * kk + 1]}, bl[2] = {blo[nt][2 * kk], blo[nt][2 * kk + 1]};
#pragma unroll
                    for (int mt = 0; mt < MT; ++mt) {
                        if (LOWP) {
                            mma_bf16(c[mt][nt], ahi[mt], bh);
                        } else {
                            if (SPLIT) {
                                mma(c1[mt][nt], alo[mt], bh);
                                mma(c2[mt][nt], ahi[mt], bl);
                            } else {
                                mma(c[mt][nt], alo[mt], bh);
                                mma(c[mt][nt], ahi[mt], bl);
                            }
                            mma(c[mt][nt], ahi[mt], bh);
                        }
                    }
                }
            }
        }
    }
    if (SPLIT) {
#pragma unroll
        for (int i = 0; i < MT; ++i)
#pragma unroll
            for (int j = 0; j < NT; ++j)
#pragma unroll
                for (int e = 0; e < 4; ++e) c[i][j][e] += c1[i][j][e] + c2[i][j][e];
    }
}

template <int MT, int NT>
__device__ __forceinline__ void zero_frag(float (&c)[MT][NT][4]) {
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < NT; ++j) { c[i][j][0] = 0.f; c[i][j][1] = 0.f; c[i][j][2] = 0.f; c[i][j][3] = 0.f; }
}
template <int MT, int NT>
__device__ __forceinline__ void scale_frag(float (&c)[MT][NT][4], float f) {
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < NT; ++j) { c[i][j][0] *= f; c[i][j][1] *= f; c[i][j][2] *= f; c[i][j][3] *= f; }
}

// Power of two s with  amax * s in [2^8, 2^9)  (amax > 0), else 1: gradient tiles are scaled into fp16's range
// before the hi/lo split and un-scaled after the product.
__device__ __forceinline__ float pow2_scale(float amax) {
    if (!(amax > 0.f) || !isfinite(amax)) return 1.0f;
    const int e = (int)((__float_as_uint(amax) >> 23) & 0xff) - 127;      // floor(log2 amax) for normal numbers
    int k = 8 - e;
    k = k < -100 ? -100 : (k > 100 ? 100 : k);
    return __uint_as_float((uint32_t)(k + 127) << 23);
}

__device__ __forceinline__ float pow2_scale_band(float amax, float cur, float lo, float hi) {
    const float v = amax * cur;
    if (v >= lo && v <= hi) return cur;
    return (amax > 0.f) ? pow2_scale(amax) : cur;
}

}  // namespace m16
