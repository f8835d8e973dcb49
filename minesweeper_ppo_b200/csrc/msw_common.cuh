// msw_common.cuh -- device helpers shared by the env kernels (sm_100a).
//
// Board representation: one board = flat bitstring of H*W cells (cell r*W+c at
// bit r*W+c) spread over the lanes of ONE warp, lane w holding bits
// [32w, 32w+32).  H*W <= 1024 and W <= 32, so a 3-word window
// (previous lane, this lane, next lane) reaches every 8-neighbour of every
// cell: all eight neighbour boards are funnel shifts of that window by
// {1, W-1, W, W+1} bits, which costs two warp shuffles per dilation.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace msw {

constexpr unsigned FULL = 0xffffffffu;

struct Geo {               // per-lane geometry words (host-precomputed, see make_geo)
    uint32_t valid;        // bits of this lane's word that are cells of the board
    uint32_t notcol0;      // cells whose column != 0
    uint32_t notlast;      // cells whose column != W-1
};

// ---------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11).  Counter-based: the board drawn for
// (seed, global env id, episode) does not depend on how envs are sharded.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void philox4x32_10(uint32_t k0, uint32_t k1, uint32_t c0, uint32_t c1,
                                              uint32_t c2, uint32_t c3, uint32_t (&out)[4])
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// Dropout2d's draw for (global board gb, 8-channel chunk): channel 8 * chunk + k is dropped when
// dropout2d_u16(w, k) < (uint32_t)(p * 65536).  Keyed by the GLOBAL board, so masks do not depend on sharding;
// call id and the nullable device epoch (added per graph replay) give every forward fresh masks.
__device__ __forceinline__ void dropout2d_draw(uint32_t k0, uint32_t k1, long long gb, uint32_t chunk, uint32_t call_lo,
                                               uint32_t call_hi, const uint32_t *epoch, uint32_t (&w)[4])
{
    philox4x32_10(k0, k1 ^ 0x44524f50u, (uint32_t)gb, (uint32_t)(gb >> 32) ^ chunk, call_lo, call_hi + (epoch ? *epoch : 0u), w);
}
__device__ __forceinline__ uint32_t dropout2d_u16(const uint32_t (&w)[4], int k)
{
    return (w[k >> 1] >> (16 * (k & 1))) & 0xFFFFu;
}

// Window shifts.  win_shl: bit j of the result is flat bit (32*lane + j - s);
// win_shr: flat bit (32*lane + j + s).  0 <= s <= 33; for s == 33 (W == 32 only)
// the one bit that would come from two lanes away belongs to a cell the column
// masks remove anyway.
__device__ __forceinline__ uint32_t win_shl(uint32_t prev, uint32_t cur, int s)
{
    return s <= 32 ? __funnelshift_lc(prev, cur, s) : (prev << (s - 32));
}
__device__ __forceinline__ uint32_t win_shr(uint32_t cur, uint32_t next, int s)
{
    return s <= 32 ? __funnelshift_rc(cur, next, s) : (next >> (s - 32));
}

struct Nbr8 {              // the eight neighbour boards of X
    uint32_t e, w, n, ne, nw, s, se, sw;
};

template <int CW>
__device__ __forceinline__ Nbr8 neighbours(uint32_t X, int lane, int Wrt, const Geo &g)
{
    const int W = CW ? CW : Wrt;
    uint32_t prev = __shfl_up_sync(FULL, X, 1);
    uint32_t next = __shfl_down_sync(FULL, X, 1);
    if (lane == 0) prev = 0;
    if (lane == 31) next = 0;
    Nbr8 o;
    o.e  = win_shl(prev, X, 1) & g.notcol0;        // X[i-1]
    o.w  = win_shr(X, next, 1) & g.notlast;        // X[i+1]
    o.n  = win_shl(prev, X, W) & g.valid;          // X[i-W]
    o.ne = win_shl(prev, X, W + 1) & g.notcol0;    // X[i-W-1]
    o.nw = win_shl(prev, X, W - 1) & g.notlast;    // X[i-W+1]
    o.s  = win_shr(X, next, W) & g.valid;          // X[i+W]
    o.se = win_shr(X, next, W - 1) & g.notcol0;    // X[i+W-1]
    o.sw = win_shr(X, next, W + 1) & g.notlast;    // X[i+W+1]
    return o;
}

template <int CW>
__device__ __forceinline__ uint32_t dilate8(uint32_t X, int lane, int W, const Geo &g)
{
    const Nbr8 o = neighbours<CW>(X, lane, W, g);
    return o.e | o.w | o.n | o.ne | o.nw | o.s | o.se | o.sw;
}

// Bit-sliced population count of the eight neighbour boards -> 4 bit planes
// (adjacent_counts, env.py:314-335, defined for every cell, self excluded).
struct Planes { uint32_t c0, c1, c2, c3; };

__device__ __forceinline__ void full_add(uint32_t a, uint32_t b, uint32_t c, uint32_t &sum, uint32_t &carry)
{
    sum = a ^ b ^ c;
    carry = (a & b) | (c & (a ^ b));
}

template <int CW>
__device__ __forceinline__ Planes count_planes(uint32_t M, int lane, int W, const Geo &g)
{
    const Nbr8 o = neighbours<CW>(M, lane, W, g);
    uint32_t s1, k1, s2, k2, s3, k3, t1, d1;
    full_add(o.e, o.w, o.n, s1, k1);
    full_add(o.ne, o.nw, o.s, s2, k2);
    s3 = o.se ^ o.sw; k3 = o.se & o.sw;
    Planes p;
    uint32_t k4;
    full_add(s1, s2, s3, p.c0, k4);           // ones
    full_add(k1, k2, k3, t1, d1);             // twos (three of the four carries)
    p.c1 = t1 ^ k4;
    const uint32_t d2 = t1 & k4;
    p.c2 = d1 ^ d2;
    p.c3 = d1 & d2;
    return p;
}

__device__ __forceinline__ int warp_popc_sum(uint32_t x)
{
    return (int)__reduce_add_sync(FULL, (unsigned)__popc(x));
}

// {0,1} nibble -> four fp32 {0.0f,1.0f}
__device__ __forceinline__ float4 nib_to_f4(uint32_t nib)
{
    float4 v;
    v.x = (nib & 1u) ? 1.0f : 0.0f;
    v.y = (nib & 2u) ? 1.0f : 0.0f;
    v.z = (nib & 4u) ? 1.0f : 0.0f;
    v.w = (nib & 8u) ? 1.0f : 0.0f;
    return v;
}

// L2 residency control.  The env kernel streams ~690 MB of observations through the 126 MB L2
// every step; without a hint that stream evicts the few MB of persistent board state, and the
// next step's state loads queue in HBM behind the writes (ncu: long-scoreboard stalls even on
// prefetched loads).  State accesses therefore carry an evict_last policy, the observation stream
// is st.global.cs (evict_first).
__device__ __forceinline__ uint64_t l2_keep_policy()
{
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint32_t ld_keep(const uint32_t *p, uint64_t pol)
{
    uint32_t v;
    asm volatile("ld.global.L2::cache_hint.b32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ int4 ld_keep(const int4 *p, uint64_t pol)
{
    int4 v;
    asm volatile("ld.global.L2::cache_hint.v4.s32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ void st_keep(uint32_t *p, uint32_t v, uint64_t pol)
{
    asm volatile("st.global.L2::cache_hint.b32 [%0], %1, %2;" :: "l"(p), "r"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_keep(int4 *p, int4 v, uint64_t pol)
{
    asm volatile("st.global.L2::cache_hint.v4.s32 [%0], {%1,%2,%3,%4}, %5;"
                 :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "l"(pol) : "memory");
}

// {0,1} nibble -> four bool bytes packed in a u32 (byte k = bit k)
__device__ __forceinline__ uint32_t nib_to_b4(uint32_t nib)
{
    return (nib * 0x00204081u) & 0x01010101u;
}

}  // namespace msw
