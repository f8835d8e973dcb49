// msw_gn.cu -- fused GroupNorm + (residual add) + ReLU + Dropout2d for the rollout forward
// (SURVEY.md section 8, row f4).
//
// The reference policy (minesweeper/models/cnn_residual.py:7-27, 50-54) interleaves cuDNN
// convolutions with GroupNorm / ReLU / Dropout2d / residual adds.  Under fp16 autocast
// (train_rl.py:222) each conv output is cast to fp32, normalised, activated, dropped, added and
// cast back to fp16 by ~8 eager ATen kernels per layer; on a B200 those memory-bound kernels take
// 9x longer than the convolutions themselves (profiles/r01_profile_forward.txt; the reference
// hides this behind torch.compile, train_rl.py:391-399, which this project may not use).  This
// kernel does the whole inter-conv step in one pass over the activation:
//     y = relu( GN(x) [+ residual] ) [* dropout2d mask / (1-p)]
// x: fp16 NHWC conv output; statistics and arithmetic in fp32 (as autocast runs GroupNorm);
// outputs: fp16 NHWC (the next conv's input -- the same rounding point as autocast's cast) and,
// optionally, fp32 NHWC (the residual stream, which the reference keeps in fp32).
//
// One CTA per sample: the sample's [HW][C] fp16 tile (48 KB at 16x16x96) is staged in shared
// memory once, so HBM sees exactly one read and one write of the activation.  Thread (j, r) owns
// the 8-channel chunk j of pixels r, r+PPB, ...; 8 | channels-per-group, so a thread's chunk lies
// in one group and its partial sums go to that group with one shared-memory atomic.
#include "../../include/msw_b200.h"
#include "msw_common.cuh"
#include "msw_error.h"
#include "msw_sm100.cuh"

#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

namespace msw {

// Chan et al. update of (count, mean, M2) a <- a (+) b; empty sides pass the other through.
__device__ __forceinline__ void chan_merge(float &na, float &ma, float &qa, float nb, float mb, float qb)
{
    if (nb > 0.0f) {
        const float nn = na + nb, delta = mb - ma, w = __fdividef(nb, nn);
        ma = fmaf(delta, w, ma);
        qa += qb + delta * delta * (na * w);
        na = nn;
    }
}

struct GnParams {
    const __half *x;        // [n][HW][C]
    const float *cbias;     // nullable [C]: bias of the convolution that produced x, added before the norm
    const float *res;       // nullable [n][HW][C]
    const float *gamma, *beta;   // [C]
    __half *y16;            // nullable [n][HW][C]
    float *y32;             // nullable [n][HW][C]
    int HW, C, G, cpg, CB, PPB;
    unsigned tile_bytes;
    float eps, inv_count, drop_p, drop_scale;
    int relu;
    uint32_t k0, k1, call_lo, call_hi;
    const uint32_t *epoch;  // nullable device counter added to call_hi (fresh dropout masks per graph replay)
    // training forward: what msw_gn_act_bwd needs (all nullable)
    float *save_mean, *save_rstd;   // [n][G] statistics of (x + conv_bias)
    uint8_t *save_mask;             // [n][HW][C/8]: bit k of a byte = output channel 8j+k is "on" (ReLU active, not dropped)
    float *pool;                    // nullable [n][C]: mean over HW of the fp32 output (AdaptiveAvgPool2d(1) of the value head)
    long long sample_base;          // global index of sample 0: the Dropout2d stream is keyed by the GLOBAL sample (shard-invariant)
};

__global__ void __launch_bounds__(256, 4) gn_act_kernel(const GnParams p, long long n_samples)
{
    // One CTA per sample, 4 CTAs per SM (48 registers, ~50 KB of shared memory each).  A persistent,
    // double-buffered variant (2 tiles per CTA, next sample prefetched during the current one's
    // compute + store) was measured SLOWER (5.0 vs 4.0 ms per forward): it halves the resident warps,
    // and the latency-bound statistics / normalise phases need them more than the loads need overlap.
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const size_t tile_bytes = p.tile_bytes;       // the fp16 sample, or the pooling scratch if that is larger
    float *s_sum = reinterpret_cast<float *>(smem_raw + tile_bytes);              // [G]
    float *s_sq = s_sum + p.G;
    float *s_part = s_sq + p.G;                                                   // [3][256] per-thread partials

    const int tid = threadIdx.x;
    const int j = tid % p.CB, r0 = tid / p.CB;
    const bool active = r0 < p.PPB;
    const int g = (j * 8) / p.cpg;
    float cb0[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) cb0[k] = (p.cbias && active) ? p.cbias[j * 8 + k] : 0.0f;

    const long long n = blockIdx.x;
    __shared__ __align__(8) unsigned long long s_bar;
    const unsigned sample_bytes = (unsigned)p.HW * (unsigned)p.C * 2u;
    if (n < n_samples) {
        // the sample is one contiguous block of global memory: one bulk copy, completion on an mbarrier
        const unsigned bar = smem_u32(&s_bar);
        if (tid == 0) {
            mbar_init(bar, 1);
            mbar_fence_init();
            mbar_expect_tx(bar, sample_bytes);
            bulk_load(smem_u32(smem_raw), reinterpret_cast<const uint4 *>(p.x) + n * (long long)p.HW * p.CB, sample_bytes, bar);
        }
        __syncthreads();                              // the barrier is initialised before anyone polls it
        mbar_wait(bar, 0);
        uint4 *tile = reinterpret_cast<uint4 *>(smem_raw);
        const long long base = n * (long long)p.HW * p.CB;                       // in uint4 chunks

        // ONE pass for the statistics: per thread, shifted sums S1 = sum (v - c), S2 = sum (v - c)^2 of
        // v = x + conv_bias with c = the thread's first value (no cancellation in S2 - S1^2/m); the
        // per-thread (count, mean, M2) triples of a group are merged with Chan's update in a FIXED order
        // by one thread per group -- no float atomics, bitwise reproducible like the eager GroupNorm.
        float cnt = 0.0f, tmean = 0.0f, tm2 = 0.0f;
        if (active) {
            float c0 = 0.0f, S1 = 0.0f, S2 = 0.0f;
            bool have_shift = false;
            for (int r = r0; r < p.HW; r += p.PPB) {
                const uint4 v = tile[r * p.CB + j];
                const __half2 *h = reinterpret_cast<const __half2 *>(&v);
                if (!have_shift) {
                    c0 = __low2float(h[0]) + cb0[0];
                    have_shift = true;
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const float2 f = __half22float2(h[k]);
                    const float d0 = (f.x + cb0[2 * k]) - c0, d1 = (f.y + cb0[2 * k + 1]) - c0;
                    S1 += d0 + d1;
                    S2 = fmaf(d0, d0, fmaf(d1, d1, S2));
                }
                cnt += 8.0f;
            }
            if (cnt > 0.0f) {
                tmean = c0 + S1 / cnt;
                tm2 = S2 - S1 * S1 / cnt;
            }
        }
        s_part[tid] = cnt;
        s_part[256 + tid] = tmean;
        s_part[512 + tid] = tm2;
        __syncthreads();
        // One warp per group: lane l folds partials l, l+32, ... of the group in index order, then a
        // shuffle tree merges the 32 lanes (a fixed order again, ~10x shorter than one thread walking
        // all PPB * cpg/8 partials while the CTA waits at the barrier).
        {
            const int cpc = p.cpg / 8, per_group = p.PPB * cpc, lane = tid & 31;
            for (int gg = tid >> 5; gg < p.G; gg += 8) {
                float na = 0.0f, ma = 0.0f, qa = 0.0f;
                for (int q = lane; q < per_group; q += 32) {
                    const int t = (q / cpc) * p.CB + gg * cpc + q % cpc;
                    chan_merge(na, ma, qa, s_part[t], s_part[256 + t], s_part[512 + t]);
                }
#pragma unroll
                for (int off = 1; off < 32; off <<= 1) {
                    const float nb = __shfl_down_sync(0xffffffffu, na, off);
                    const float mb = __shfl_down_sync(0xffffffffu, ma, off);
                    const float qb = __shfl_down_sync(0xffffffffu, qa, off);
                    chan_merge(na, ma, qa, nb, mb, qb);
                }
                if (lane == 0) {
                    const float rstd = rsqrtf(qa * p.inv_count + p.eps);   // biased variance, eps as torch
                    s_sum[gg] = ma;                                         // group mean of (x + conv_bias)
                    s_sq[gg] = rstd;
                    if (p.save_mean) {
                        p.save_mean[n * p.G + gg] = ma;
                        p.save_rstd[n * p.G + gg] = rstd;
                    }
                }
            }
        }
        __syncthreads();
        float psum[8];
        if (active) {
            const float mean = s_sum[g], rstd = s_sq[g];
            // per-channel affine folded with the statistics, and the Dropout2d channel mask
            float a[8], b[8];
            uint32_t kept = 0xFFu;                                    // channels that survive Dropout2d
            uint32_t w[4] = {0u, 0u, 0u, 0u};
            if (p.drop_p > 0.0f)
                philox4x32_10(p.k0, p.k1 ^ 0x44524f50u, (uint32_t)(n + p.sample_base),
                              (uint32_t)((n + p.sample_base) >> 32) ^ (uint32_t)j, p.call_lo, p.call_hi + (p.epoch ? *p.epoch : 0u), w);
            const uint32_t thresh = (uint32_t)(p.drop_p * 65536.0f);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const float ga = p.gamma[j * 8 + k] * rstd;
                a[k] = ga;
                b[k] = fmaf(cb0[k] - mean, ga, p.beta[j * 8 + k]);  // beta + (bias_c - mean) * gamma * rstd
                if (p.drop_p > 0.0f) {
                    // relu(z)*s == relu(z*s) for s >= 0, so the mask/scale folds into the affine when no
                    // residual is added (Dropout2d follows ReLU only on that path, cnn_residual.py:20-21)
                    const uint32_t u16 = (w[k >> 1] >> (16 * (k & 1))) & 0xFFFFu;
                    const float sc = (u16 < thresh) ? 0.0f : p.drop_scale;
                    if (u16 < thresh) kept &= ~(1u << k);
                    a[k] *= sc;
                    b[k] *= sc;
                }
            }
            const float4 *__restrict__ res = p.res ? reinterpret_cast<const float4 *>(p.res) + 2 * base : nullptr;
            float4 *__restrict__ y32 = p.y32 ? reinterpret_cast<float4 *>(p.y32) + 2 * base : nullptr;
#pragma unroll
            for (int k = 0; k < 8; ++k) psum[k] = 0.0f;
#pragma unroll 4
            for (int r = r0; r < p.HW; r += p.PPB) {
                const int idx = r * p.CB + j;
                const uint4 v = tile[idx];
                const __half2 *h = reinterpret_cast<const __half2 *>(&v);
                float o[8];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const float2 f = __half22float2(h[k]);
                    o[2 * k] = fmaf(f.x, a[2 * k], b[2 * k]);
                    o[2 * k + 1] = fmaf(f.y, a[2 * k + 1], b[2 * k + 1]);
                }
                if (res) {
                    const float4 q0 = __ldcs(res + 2 * idx), q1 = __ldcs(res + 2 * idx + 1);
                    o[0] += q0.x; o[1] += q0.y; o[2] += q0.z; o[3] += q0.w;
                    o[4] += q1.x; o[5] += q1.y; o[6] += q1.z; o[7] += q1.w;
                }
                if (p.save_mask) {
                    uint32_t on = 0u;
#pragma unroll
                    for (int k = 0; k < 8; ++k) on |= ((!p.relu || o[k] > 0.0f) ? 1u : 0u) << k;
                    p.save_mask[(n * p.HW + r) * (long long)p.CB + j] = (uint8_t)(on & kept);
                }
                if (p.relu) {
#pragma unroll
                    for (int k = 0; k < 8; ++k) o[k] = fmaxf(o[k], 0.0f);
                }
                if (p.pool) {
#pragma unroll
                    for (int k = 0; k < 8; ++k) psum[k] += o[k];
                }
                if (y32) {
                    y32[2 * idx] = make_float4(o[0], o[1], o[2], o[3]);
                    y32[2 * idx + 1] = make_float4(o[4], o[5], o[6], o[7]);
                }
                if (p.y16) {
                    uint4 out;
                    __half2 *oh = reinterpret_cast<__half2 *>(&out);
#pragma unroll
                    for (int k = 0; k < 4; ++k) oh[k] = __floats2half2_rn(o[2 * k], o[2 * k + 1]);
                    tile[idx] = out;                  // in place over the thread's own input chunk
                }
            }
        }
        if (p.y16) {
            fence_proxy_async();                      // generic-proxy writes -> visible to the bulk store
            __syncthreads();
            if (tid == 0) {
                bulk_store(reinterpret_cast<uint4 *>(p.y16) + n * (long long)p.HW * p.CB, smem_u32(smem_raw), sample_bytes);
                bulk_commit();
                bulk_wait_read<0>();
            }
        }
        if (p.pool) {
            // per-channel mean of the output: the thread partials go through the (now dead) tile and are
            // summed over the PPB pixel slots in index order -- fixed order, no float atomics
            __syncthreads();
            float *s_pool = reinterpret_cast<float *>(smem_raw);                      // [PPB][C]
            if (active) {
#pragma unroll
                for (int k = 0; k < 8; ++k) s_pool[r0 * p.C + j * 8 + k] = psum[k];
            }
            __syncthreads();
            for (int c = tid; c < p.C; c += 256) {
                float t = 0.0f;
                for (int r = 0; r < p.PPB; ++r) t += s_pool[r * p.C + c];
                p.pool[n * p.C + c] = t / (float)p.HW;
            }
        }
    }
}

// ---------------------------------------------------------------------------
// Backward of gn_act_kernel for the training forward (the autograd half of SURVEY row f4).
// With z = (x + bias_c - mean_g) * rstd_g, y = on * s * (z * gamma_c + beta_c [+ res]):
//   dy'      = (g16 + g32) * on * s                  (on: saved ReLU/Dropout2d bit, s = 1/(1-p))
//   dgamma_c = sum dy' * z,  dbeta_c = sum dy',  dres = dy'
//   dx       = rstd_g * (dy' * gamma_c - mean_g(dy' gamma) - z * mean_g(dy' gamma z)),  dbias_c = sum dx
// One CTA per sample; per-channel sums leave the CTA as per-sample partials [n][C] that the host
// reduces over n in a fixed order (no float atomics -> reproducible).
// ---------------------------------------------------------------------------
struct GnBwdParams {
    const __half *x;            // [n][HW][C] conv output saved by the forward
    const float *cbias, *gamma; // [C] (cbias nullable)
    const float *mean, *rstd;   // [n][G]
    const uint8_t *mask;        // [n][HW][C/8]
    const __half *g16;          // nullable upstream gradient of y16
    const float *g32;           // nullable upstream gradient of y32
    __half *dx;                 // [n][HW][C]
    float *dres;                // nullable [n][HW][C]
    float *p_dgamma, *p_dbeta, *p_dbias;   // [n][C] per-sample partials (p_dbias nullable)
    int HW, C, G, cpg, CB, PPB;
    float inv_count, scale;
};

__global__ void __launch_bounds__(256) gn_act_bwd_kernel(const GnBwdParams p)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint4 *tile = reinterpret_cast<uint4 *>(smem_raw);                              // x, [HW][CB]
    float *s_g1 = reinterpret_cast<float *>(smem_raw + (size_t)p.HW * p.C * 2);     // [G]
    float *s_g2 = s_g1 + p.G;
    float *s_part = s_g2 + p.G;                                                     // [256]
    float *s_ch = s_part + 256;                                                     // [3][PPB][C]

    const int tid = threadIdx.x;
    const int j = tid % p.CB, r0 = tid / p.CB;
    const bool active = r0 < p.PPB;
    const int g = (j * 8) / p.cpg;
    const long long n = blockIdx.x;
    const long long base = n * (long long)p.HW * p.CB;
    auto group_total = [&](float mine, float *dst) {
        s_part[tid] = active ? mine : 0.0f;
        __syncthreads();
        if (tid < p.G) {
            const int j0 = tid * (p.cpg / 8), j1 = j0 + p.cpg / 8;
            float t = 0.0f;
            for (int r = 0; r < p.PPB; ++r)
                for (int jj = j0; jj < j1; ++jj) t += s_part[r * p.CB + jj];
            dst[tid] = t;
        }
        __syncthreads();
    };

    const float mean = p.mean[n * p.G + g], rstd = p.rstd[n * p.G + g];
    float cb[8], gam[8], dg[8], db[8], dcb[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        cb[k] = ((p.cbias && active) ? p.cbias[j * 8 + k] : 0.0f) - mean;
        gam[k] = active ? p.gamma[j * 8 + k] : 0.0f;
        dg[k] = db[k] = dcb[k] = 0.0f;
    }
    const uint4 *xs = reinterpret_cast<const uint4 *>(p.x) + base;
    const uint4 *g16 = p.g16 ? reinterpret_cast<const uint4 *>(p.g16) + base : nullptr;
    const float4 *g32 = p.g32 ? reinterpret_cast<const float4 *>(p.g32) + 2 * base : nullptr;
    const uint8_t *mk = p.mask + base;

    auto load_dy = [&](int idx, float (&dy)[8]) {
#pragma unroll
        for (int k = 0; k < 8; ++k) dy[k] = 0.0f;
        if (g16) {
            const uint4 v = __ldg(g16 + idx);
            const __half2 *h = reinterpret_cast<const __half2 *>(&v);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float2 f = __half22float2(h[k]);
                dy[2 * k] += f.x; dy[2 * k + 1] += f.y;
            }
        }
        if (g32) {
            const float4 q0 = __ldg(g32 + 2 * idx), q1 = __ldg(g32 + 2 * idx + 1);
            dy[0] += q0.x; dy[1] += q0.y; dy[2] += q0.z; dy[3] += q0.w;
            dy[4] += q1.x; dy[5] += q1.y; dy[6] += q1.z; dy[7] += q1.w;
        }
        const uint32_t on = mk[idx];
#pragma unroll
        for (int k = 0; k < 8; ++k) dy[k] = ((on >> k) & 1u) ? dy[k] * p.scale : 0.0f;
    };

    // pass A: group sums of dy*gamma and dy*gamma*z; per-channel dgamma / dbeta
    float s1 = 0.0f, s2 = 0.0f;
    if (active) {
        // cp.async puts every thread's loads in flight at once (a synchronous copy loop left the forward kernel
        // at half the HBM rate)
        for (int r = r0; r < p.HW; r += p.PPB) {
            const uint4 *src = xs + r * p.CB + j;
            cp_async16(smem_u32(tile + r * p.CB + j), src);
        }
        cp_async_commit();
        cp_async_wait<0>();
#pragma unroll 2
        for (int r = r0; r < p.HW; r += p.PPB) {
            const int idx = r * p.CB + j;
            const uint4 v = tile[idx];
            const __half2 *h = reinterpret_cast<const __half2 *>(&v);
            float dy[8];
            load_dy(idx, dy);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float2 f = __half22float2(h[k]);
                const float z0 = (f.x + cb[2 * k]) * rstd, z1 = (f.y + cb[2 * k + 1]) * rstd;
                const float a0 = dy[2 * k] * gam[2 * k], a1 = dy[2 * k + 1] * gam[2 * k + 1];
                s1 += a0 + a1;
                s2 += a0 * z0 + a1 * z1;
                dg[2 * k] += dy[2 * k] * z0; dg[2 * k + 1] += dy[2 * k + 1] * z1;
                db[2 * k] += dy[2 * k];      db[2 * k + 1] += dy[2 * k + 1];
            }
        }
    }
    group_total(s1, s_g1);
    group_total(s2, s_g2);
    const float m1 = s_g1[g] * p.inv_count, m2 = s_g2[g] * p.inv_count;

    // pass B: dx (and dres), per-channel dbias
    if (active) {
        uint4 *dxo = reinterpret_cast<uint4 *>(p.dx) + base;
        float4 *dro = p.dres ? reinterpret_cast<float4 *>(p.dres) + 2 * base : nullptr;
#pragma unroll 2
        for (int r = r0; r < p.HW; r += p.PPB) {
            const int idx = r * p.CB + j;
            const uint4 v = tile[idx];
            const __half2 *h = reinterpret_cast<const __half2 *>(&v);
            float dy[8], dx[8];
            load_dy(idx, dy);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float2 f = __half22float2(h[k]);
                const float z0 = (f.x + cb[2 * k]) * rstd, z1 = (f.y + cb[2 * k + 1]) * rstd;
                dx[2 * k] = rstd * (dy[2 * k] * gam[2 * k] - m1 - z0 * m2);
                dx[2 * k + 1] = rstd * (dy[2 * k + 1] * gam[2 * k + 1] - m1 - z1 * m2);
                dcb[2 * k] += dx[2 * k]; dcb[2 * k + 1] += dx[2 * k + 1];
            }
            uint4 out;
            __half2 *oh = reinterpret_cast<__half2 *>(&out);
#pragma unroll
            for (int k = 0; k < 4; ++k) oh[k] = __floats2half2_rn(dx[2 * k], dx[2 * k + 1]);
            dxo[idx] = out;
            if (dro) {
                dro[2 * idx] = make_float4(dy[0], dy[1], dy[2], dy[3]);
                dro[2 * idx + 1] = make_float4(dy[4], dy[5], dy[6], dy[7]);
            }
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            s_ch[(0 * p.PPB + r0) * p.C + j * 8 + k] = dg[k];
            s_ch[(1 * p.PPB + r0) * p.C + j * 8 + k] = db[k];
            s_ch[(2 * p.PPB + r0) * p.C + j * 8 + k] = dcb[k];
        }
    }
    __syncthreads();
    for (int c = tid; c < p.C; c += blockDim.x) {
        float t0 = 0.0f, t1 = 0.0f, t2 = 0.0f;
        for (int r = 0; r < p.PPB; ++r) {
            t0 += s_ch[(0 * p.PPB + r) * p.C + c];
            t1 += s_ch[(1 * p.PPB + r) * p.C + c];
            t2 += s_ch[(2 * p.PPB + r) * p.C + c];
        }
        p.p_dgamma[n * p.C + c] = t0;
        p.p_dbeta[n * p.C + c] = t1;
        if (p.p_dbias) p.p_dbias[n * p.C + c] = t2;
    }
}

}  // namespace msw

namespace msw {

// fp32 NCHW observation planes -> fp16 NHWC with the channels padded to 16 (zeros): the stem convolution's input
// in the layout the tensor cores want, in one pass instead of a cast kernel plus cuDNN's own padding kernels.
__global__ void __launch_bounds__(256) pack_obs16_kernel(const float *__restrict__ obs, uint4 *__restrict__ out, long long n,
                                                         int Cin, int HW)
{
    const long long total = n * HW;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long b = i / HW;
        const int px = (int)(i - b * HW);
        const float *src = obs + (b * Cin) * HW + px;           // consecutive threads read consecutive pixels of a plane
        __half2 h[8];
#pragma unroll
        for (int c = 0; c < 16; c += 2) {
            const float v0 = c < Cin ? __ldcs(src + (long long)c * HW) : 0.0f;
            const float v1 = c + 1 < Cin ? __ldcs(src + (long long)(c + 1) * HW) : 0.0f;
            h[c >> 1] = __floats2half2_rn(v0, v1);
        }
        out[2 * i] = *reinterpret_cast<const uint4 *>(&h[0]);
        out[2 * i + 1] = *reinterpret_cast<const uint4 *>(&h[4]);
    }
}

}  // namespace msw

extern "C" int msw_pack_obs16(const float *obs, void *out16, int64_t n, int32_t Cin, int32_t HW, void *stream)
{
    using namespace msw;
    if (!obs || !out16) return fail(MSW_ERR_NULL, "msw_pack_obs16: NULL pointer");
    if (n < 0 || Cin < 1 || Cin > 16 || HW < 1) return fail(MSW_ERR_BAD_SHAPE, "msw_pack_obs16: n=%lld Cin=%d HW=%d", (long long)n, Cin, HW);
    if (((uintptr_t)out16 & 15u) != 0) return fail(MSW_ERR_ALIGN, "msw_pack_obs16: output must be 16-byte aligned");
    if (n == 0) return MSW_OK;
    const long long total = n * HW;
    const long long blocks = (total + 255) / 256;
    pack_obs16_kernel<<<(unsigned)(blocks < 148LL * 16 ? blocks : 148LL * 16), 256, 0, (cudaStream_t)stream>>>(
        obs, (uint4 *)out16, n, Cin, HW);
    MSW_CUDA_TRY(cudaGetLastError());
    return MSW_OK;
}

extern "C" int msw_gn_act(const void *x16, const float *conv_bias, const float *res32, const float *gamma,
                          const float *beta, void *y16,
                          float *y32, int64_t n, int32_t HW, int32_t C, int32_t G, float eps, int32_t relu,
                          float drop_p, uint64_t seed, uint64_t call_id, const uint32_t *epoch, float *save_mean,
                          float *save_rstd, uint8_t *save_mask, float *pool32, int64_t sample_id_base, void *stream)
{
    using namespace msw;
    if (!x16 || !gamma || !beta || (!y16 && !y32 && !pool32)) return fail(MSW_ERR_NULL, "msw_gn_act: NULL pointer");
    if (n < 0 || HW < 1 || C < 8 || G < 1 || C % G != 0 || C % 8 != 0 || (C / G) % 8 != 0 || C / 8 > 256 || 2 * G > 256)
        return fail(MSW_ERR_BAD_SHAPE, "msw_gn_act: need C %% 8 == 0, (C/G) %% 8 == 0 (C=%d G=%d HW=%d)", C, G, HW);
    if (drop_p < 0.0f || drop_p >= 1.0f) return fail(MSW_ERR_ARG, "msw_gn_act: drop_p=%f", drop_p);
    if (drop_p > 0.0f && res32) return fail(MSW_ERR_ARG, "msw_gn_act: dropout is only defined on the no-residual path");
    if ((((uintptr_t)x16 | (uintptr_t)res32 | (uintptr_t)y16 | (uintptr_t)y32) & 15u) != 0)
        return fail(MSW_ERR_ALIGN, "msw_gn_act: tensors must be 16-byte aligned");
    if (n == 0) return MSW_OK;
    size_t tile_bytes = (size_t)HW * C * 2;
    if (pool32 && (size_t)(256 / (C / 8)) * C * sizeof(float) > tile_bytes) tile_bytes = (size_t)(256 / (C / 8)) * C * sizeof(float);
    const size_t smem = tile_bytes + (2 * (size_t)G + 3 * 256) * sizeof(float);
    if (smem > 200 * 1024) return fail(MSW_ERR_BAD_SHAPE, "msw_gn_act: sample of %zu bytes does not fit shared memory", smem);
    if (smem > 48 * 1024) MSW_SET_MAX_SMEM(gn_act_kernel, 200 * 1024);
    GnParams p;
    p.x = (const __half *)x16; p.cbias = conv_bias; p.res = res32; p.gamma = gamma; p.beta = beta;
    p.y16 = (__half *)y16; p.y32 = y32;
    p.HW = HW; p.C = C; p.G = G; p.cpg = C / G; p.CB = C / 8; p.PPB = 256 / p.CB;
    p.eps = eps; p.inv_count = 1.0f / (float)((long long)HW * p.cpg);
    p.drop_p = drop_p; p.drop_scale = drop_p > 0.0f ? 1.0f / (1.0f - drop_p) : 1.0f;
    p.relu = relu;
    p.k0 = (uint32_t)seed; p.k1 = (uint32_t)(seed >> 32);
    p.call_lo = (uint32_t)call_id; p.call_hi = (uint32_t)(call_id >> 32);
    p.epoch = epoch;
    p.pool = pool32;
    p.sample_base = (long long)sample_id_base;
    p.tile_bytes = (unsigned)tile_bytes;
    if ((save_mean != nullptr) != (save_rstd != nullptr) || (save_mean != nullptr) != (save_mask != nullptr))
        return fail(MSW_ERR_ARG, "msw_gn_act: save_mean / save_rstd / save_mask must be given together");
    p.save_mean = save_mean; p.save_rstd = save_rstd; p.save_mask = save_mask;
    if (n > 0x7fffffffLL) return fail(MSW_ERR_BAD_SHAPE, "msw_gn_act: n too large");
    gn_act_kernel<<<(unsigned)n, 256, smem, (cudaStream_t)stream>>>(p, (long long)n);
    MSW_CUDA_TRY(cudaGetLastError());
    return MSW_OK;
}

extern "C" int msw_gn_act_bwd(const void *x16, const float *conv_bias, const float *gamma, const float *mean,
                              const float *rstd, const uint8_t *mask, const void *g16, const float *g32, void *dx16,
                              float *dres32, float *part_dgamma, float *part_dbeta, float *part_dbias, int64_t n,
                              int32_t HW, int32_t C, int32_t G, float drop_p, void *stream)
{
    using namespace msw;
    if (!x16 || !gamma || !mean || !rstd || !mask || !dx16 || !part_dgamma || !part_dbeta || (!g16 && !g32))
        return fail(MSW_ERR_NULL, "msw_gn_act_bwd: NULL pointer");
    if (n < 0 || HW < 1 || C < 8 || G < 1 || C % G != 0 || C % 8 != 0 || (C / G) % 8 != 0 || C / 8 > 256 || 2 * G > 256)
        return fail(MSW_ERR_BAD_SHAPE, "msw_gn_act_bwd: need C %% 8 == 0, (C/G) %% 8 == 0 (C=%d G=%d HW=%d)", C, G, HW);
    if (drop_p < 0.0f || drop_p >= 1.0f) return fail(MSW_ERR_ARG, "msw_gn_act_bwd: drop_p=%f", drop_p);
    if ((((uintptr_t)x16 | (uintptr_t)g16 | (uintptr_t)g32 | (uintptr_t)dx16 | (uintptr_t)dres32) & 15u) != 0)
        return fail(MSW_ERR_ALIGN, "msw_gn_act_bwd: tensors must be 16-byte aligned");
    if (n == 0) return MSW_OK;
    GnBwdParams p;
    p.x = (const __half *)x16; p.cbias = conv_bias; p.gamma = gamma; p.mean = mean; p.rstd = rstd; p.mask = mask;
    p.g16 = (const __half *)g16; p.g32 = g32; p.dx = (__half *)dx16; p.dres = dres32;
    p.p_dgamma = part_dgamma; p.p_dbeta = part_dbeta; p.p_dbias = part_dbias;
    p.HW = HW; p.C = C; p.G = G; p.cpg = C / G; p.CB = C / 8; p.PPB = 256 / p.CB;
    p.inv_count = 1.0f / (float)((long long)HW * p.cpg);
    p.scale = drop_p > 0.0f ? 1.0f / (1.0f - drop_p) : 1.0f;
    const size_t smem = (size_t)HW * C * 2 + (2 * (size_t)G + 256 + 3 * (size_t)p.PPB * C) * sizeof(float);
    if (smem > 200 * 1024) return fail(MSW_ERR_BAD_SHAPE, "msw_gn_act_bwd: sample of %zu bytes does not fit shared memory", smem);
    if (smem > 48 * 1024) MSW_SET_MAX_SMEM(gn_act_bwd_kernel, 200 * 1024);
    if (n > 0x7fffffffLL) return fail(MSW_ERR_BAD_SHAPE, "msw_gn_act_bwd: n too large");
    gn_act_bwd_kernel<<<(unsigned)n, 256, smem, (cudaStream_t)stream>>>(p);
    MSW_CUDA_TRY(cudaGetLastError());
    return MSW_OK;
}
