// HBM/latency-bound kernels of the sampling step: time embeddings + projections, the 8x8/s2 stem convolution on the
// fp32 state, InstanceNorm statistics/apply, the Cout=1 tail convolution, the DDPM posterior update and the DDIM update.
#pragma once
#include <algorithm>
#include <cmath>

#include "common.cuh"

namespace b2d {

// ------------------------------------------------------------------------------------------------ time embeddings
// One CTA per sample.  Computes both reference embeddings and all nine SiLU->Linear projections in one launch:
//   encoder (modules_DANRA_conditional.py:203-211,256): e = [sin(t*inv_j) | cos(t*inv_j)] (+ label_emb[y]), inv_j = 1000^(-2j/256)
//   decoder (modules_DANRA_conditional.py:42-63):       d[2j] = sin(t/div_j), d[2j+1] = cos(t/div_j),   div_j = 10000^(2j/256)
//   out[b][o] = bias[o] + sum_k W[o][k] * silu(emb_sel(o)[k]),  rows o < n_enc use e, the rest use d.
// Family D (unet_ms.py:138-146) uses the [sin|cos] layout with base 10000 for every projection (n_enc = n_out, inv table differs).
constexpr int TEMB_DIM = 256;
constexpr int TEMB_SB = 8;    // samples per CTA (weights are read once per 8 samples)
constexpr int TEMB_OC = 64;   // outputs per CTA
// grid = (ceil(n_out/64), ceil(B/8)), 256 threads.
__global__ void __launch_bounds__(256) temb_project_kernel(const int* __restrict__ t, const int* __restrict__ y,
                                                           const float* __restrict__ label_emb,  // [ncls][256] or null
                                                           const float* __restrict__ enc_inv,    // [128]
                                                           const float* __restrict__ dec_div,    // [128]
                                                           const float* __restrict__ W,          // [n_out][256]
                                                           const float* __restrict__ bias,       // [n_out]
                                                           float* __restrict__ out,              // [B][n_out]
                                                           int n_enc, int n_out, int B, int t_off, int enc_interleaved) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ float se[TEMB_SB][TEMB_DIM];   // silu(embedding) of this CTA's samples (encoder OR decoder flavour)
    const int b0 = blockIdx.y * TEMB_SB;
    const int o0 = blockIdx.x * TEMB_OC;
    // n_enc is a multiple of TEMB_OC (host-checked): a CTA is all-encoder or all-decoder.  enc_interleaved: the Downscaling
    // generation's encoder embeds t with the decoder's interleaved base-10000 SinusoidalEmbedding (modules_DANRA_downscaling.py:190)
    const bool enc = o0 < n_enc && !enc_interleaved;
    {
        const int k = threadIdx.x;  // 256 threads <-> 256 embedding entries
        // inside the reverse loop every sample carries the same t: the sin/cos is evaluated once and reused
        const int t0 = t[min(b0, B - 1)] + t_off;   // t_off = -1: embeddings of the NEXT reverse step
        auto emb = [&](int tt) -> float {
            const float tf = (float)tt;
            if (enc) {
                const float a = tf * enc_inv[k & 127];
                return (k < 128) ? sinf(a) : cosf(a);
            }
            const float a2 = __fdiv_rn(tf, dec_div[k >> 1]);
            return (k & 1) ? cosf(a2) : sinf(a2);
        };
        const float e0 = emb(t0);
        const bool labelled = enc && label_emb != nullptr && y != nullptr;
        const float s0 = silu(e0);
#pragma unroll
        for (int sidx = 0; sidx < TEMB_SB; ++sidx) {
            const int b = min(b0 + sidx, B - 1);
            const int tb = t[b] + t_off;
            float e = (tb == t0) ? e0 : emb(tb);
            float sv = s0;
            if (labelled) sv = silu(e + label_emb[(size_t)y[b] * TEMB_DIM + k]);
            else if (tb != t0) sv = silu(e);
            se[sidx][k] = sv;
        }
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // this lane's slice of the 8 embeddings stays in registers for all outputs of the warp
    float ev[TEMB_SB][8];
#pragma unroll
    for (int sidx = 0; sidx < TEMB_SB; ++sidx)
#pragma unroll
        for (int q = 0; q < 8; ++q) ev[sidx][q] = se[sidx][lane + 32 * q];
#pragma unroll 2
    for (int oi = 0; oi < TEMB_OC / 8; ++oi) {
        const int o = o0 + warp * (TEMB_OC / 8) + oi;
        if (o >= n_out) break;
        const float* w = W + (size_t)o * TEMB_DIM;
        float wv[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) wv[q] = __ldg(w + lane + 32 * q);
        float acc[TEMB_SB];
#pragma unroll
        for (int sidx = 0; sidx < TEMB_SB; ++sidx) {
            float a = 0.f;
#pragma unroll
            for (int q = 0; q < 8; ++q) a = fmaf(wv[q], ev[sidx][q], a);
            acc[sidx] = a;
        }
        // transposed butterfly: 8 per-lane partials -> lane L ends with the total of sample ((L>>4)&1)*4 + ((L>>3)&1)*2 + ((L>>2)&1)
        float r4[4], r2[2], r1;
        {
            const bool up = lane & 16;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float keep = up ? acc[4 + i] : acc[i], give = up ? acc[i] : acc[4 + i];
                r4[i] = keep + __shfl_xor_sync(0xffffffffu, give, 16);
            }
        }
        {
            const bool up = lane & 8;
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const float keep = up ? r4[2 + i] : r4[i], give = up ? r4[i] : r4[2 + i];
                r2[i] = keep + __shfl_xor_sync(0xffffffffu, give, 8);
            }
        }
        {
            const bool up = lane & 4;
            const float keep = up ? r2[1] : r2[0], give = up ? r2[0] : r2[1];
            r1 = keep + __shfl_xor_sync(0xffffffffu, give, 4);
        }
        r1 += __shfl_xor_sync(0xffffffffu, r1, 2);
        r1 += __shfl_xor_sync(0xffffffffu, r1, 1);
        const int sidx = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
        if ((lane & 3) == 0 && b0 + sidx < B) out[(size_t)(b0 + sidx) * n_out + o] = r1 + bias[o];
    }
}

// ------------------------------------------------------------------------------------------------ stem convolution
// Direct KSxKS / stride / pad convolution of an fp32 NCHW tensor with few channels (the diffusion state x, or the
// step-invariant conditioning stack) to 64 channels, NHWC output.  FP32 FMA: K = KS*KS*Cx is tiny and the state must
// not be rounded to f16 before its first use.
//   out[b,ho,wo,co] = sum_{c,r,s} in[b,c,ho*st+r-pad,wo*st+s-pad] * w[co][c][r][s] (+ add[b,ho,wo,co]) (+ vec[b][co])
// Encoder.conv1 (modules_DANRA_conditional.py:178-183, :260) is linear in its input channels, so the conditioning
// channels' contribution is computed once per sampling job (out_f32) and added each step through `add`.
// CTA: 16x16 output pixels x 64 channels, 256 threads; thread = 4 consecutive output pixels of one row x 16 channels
// (64 fp32 accumulators): per filter row the thread loads its 4*STRIDE+KS-STRIDE inputs once and reuses them over the
// KS taps and 4 pixels, so shared-memory traffic is ~1 load per 11 FMAs.
template <int KS, int STRIDE>
__global__ void __launch_bounds__(256) stem_conv_kernel(const float* __restrict__ in, int Cx, int Hi, int Wi,
                                                        const float* __restrict__ w,  // packed [Cin_total][KS*KS][64]
                                                        int w_cstride_total,          // channels in the full weight (unused)
                                                        int w_coffset,                // first weight channel used
                                                        const float* __restrict__ add,  // [B,Ho,Wo,64] fp32 or null
                                                        const float* __restrict__ vec, int vec_stride,  // [B][..] or null
                                                        f16* __restrict__ out_f16, float* __restrict__ out_f32, int Ho,
                                                        int Wo, int pad) {
    pdl_launch_dependents();
    pdl_wait();
    constexpr int PT = 16;                        // output tile side
    constexpr int IT = (PT - 1) * STRIDE + KS;    // input tile side
    constexpr int NX = 3 * STRIDE + KS;           // inputs one thread needs per filter row (4 pixels)
    __shared__ float s_in[IT][IT + 1];
    __shared__ __align__(16) float s_w[KS * KS][64];
    const int b = blockIdx.z;
    const int ho0 = blockIdx.y * PT, wo0 = blockIdx.x * PT;
    const int cg = threadIdx.x >> 6;              // warp-uniform channel group (16 channels)
    const int pg = threadIdx.x & 63;              // pixel group: row py, columns 4*px4 .. 4*px4+3
    const int py = pg >> 2, px4 = pg & 3;
    float acc[4][16];
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int i = 0; i < 16; ++i) acc[j][i] = 0.f;
    for (int c = 0; c < Cx; ++c) {
        __syncthreads();
        const float* ip = in + ((size_t)b * Cx + c) * Hi * Wi;
        for (int i = threadIdx.x; i < IT * IT; i += 256) {
            const int iy = i / IT, ix = i - iy * IT;
            const int gy = ho0 * STRIDE - pad + iy, gx = wo0 * STRIDE - pad + ix;
            s_in[iy][ix] = (gy >= 0 && gy < Hi && gx >= 0 && gx < Wi) ? ip[(size_t)gy * Wi + gx] : 0.f;
        }
        {
            const float4* wsrc = reinterpret_cast<const float4*>(w + (size_t)(w_coffset + c) * (KS * KS * 64));
            float4* wdst = reinterpret_cast<float4*>(&s_w[0][0]);
            for (int i = threadIdx.x; i < KS * KS * 16; i += 256) wdst[i] = __ldg(wsrc + i);
        }
        __syncthreads();
#pragma unroll 1
        for (int r = 0; r < KS; ++r) {
            float xin[NX];
            const float* row = &s_in[py * STRIDE + r][px4 * 4 * STRIDE];
#pragma unroll
            for (int k = 0; k < NX; ++k) xin[k] = row[k];
#pragma unroll
            for (int sx = 0; sx < KS; ++sx) {
                const float4* wv = reinterpret_cast<const float4*>(&s_w[r * KS + sx][cg * 16]);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float4 w4 = wv[q];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float v = xin[j * STRIDE + sx];
                        acc[j][q * 4 + 0] = fmaf(v, w4.x, acc[j][q * 4 + 0]);
                        acc[j][q * 4 + 1] = fmaf(v, w4.y, acc[j][q * 4 + 1]);
                        acc[j][q * 4 + 2] = fmaf(v, w4.z, acc[j][q * 4 + 2]);
                        acc[j][q * 4 + 3] = fmaf(v, w4.w, acc[j][q * 4 + 3]);
                    }
                }
            }
        }
    }
    const int ho = ho0 + py;
    if (ho >= Ho) return;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int wo = wo0 + px4 * 4 + j;
        if (wo >= Wo) continue;
        const size_t o = (((size_t)b * Ho + ho) * Wo + wo) * 64 + cg * 16;
        float a[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) a[i] = acc[j][i];
        if (add) {
#pragma unroll
            for (int i = 0; i < 16; i += 4) {
                const float4 t4 = *reinterpret_cast<const float4*>(add + o + i);
                a[i] += t4.x; a[i + 1] += t4.y; a[i + 2] += t4.z; a[i + 3] += t4.w;
            }
        }
        if (vec) {
#pragma unroll
            for (int i = 0; i < 16; ++i) a[i] += vec[(size_t)b * vec_stride + cg * 16 + i];
        }
        if (out_f32) {
#pragma unroll
            for (int i = 0; i < 16; i += 4)
                *reinterpret_cast<float4*>(out_f32 + o + i) = make_float4(a[i], a[i + 1], a[i + 2], a[i + 3]);
        } else {
            uint4 v0, v1;
            v0.x = pack_h2(a[0], a[1]);   v0.y = pack_h2(a[2], a[3]);
            v0.z = pack_h2(a[4], a[5]);   v0.w = pack_h2(a[6], a[7]);
            v1.x = pack_h2(a[8], a[9]);   v1.y = pack_h2(a[10], a[11]);
            v1.z = pack_h2(a[12], a[13]); v1.w = pack_h2(a[14], a[15]);
            uint4* op = reinterpret_cast<uint4*>(out_f16 + o);
            op[0] = v0;
            op[1] = v1;
        }
    }
}

// Tensor-core version of the per-step 8x8 / stride 2 / pad 3 stem (Encoder.conv1 on the diffusion state), used when the
// output extent is a multiple of 16.  The fp32 state is NOT rounded: x is split into an fp16 (hi, lo) pair and the product is
// formed as x_hi*w + x_lo*w with fp32 accumulation (mma.sync m16n8k16); the weights are fp16 like every other layer's.
// CTA = 16x16 output pixels x 64 channels, 8 warps; warp = 2 output rows (two m16 tiles) x all 64 channels.
// GEMM view per input channel: M = pixel, K = 64 taps (k-tile = two filter rows), N = 64.  The A fragments are plain
// 32-bit shared-memory loads from the (38 x 38) input tile: tap (ky, kx) of output pixel (oy, ox) is tile[2oy+ky][2ox+kx],
// and a fragment register holds two consecutive kx.  Epilogue: + precomputed conditioning part (fp32) + time projection,
// fp16 rows staged per warp in swizzled shared memory and written as full 128-byte lines.
constexpr int STEM_IT = 38, STEM_XP = 40, STEM_WP = 72;
constexpr int STEM_MMA_SMEM = 2 * STEM_IT * STEM_XP * 2 + 64 * STEM_WP * 2 + 8 * 4096 + 64 * 4;
__global__ void __launch_bounds__(256, 2) stem_mma_kernel(const float* __restrict__ in, int Cx, int Hi, int Wi,
                                                          const float* __restrict__ w,    // packed [Cin_total][64 taps][64]
                                                          const float* __restrict__ add,  // [B,Ho,Wo,64] fp32 or null
                                                          const float* __restrict__ vec, int vec_stride,
                                                          f16* __restrict__ out, int Ho, int Wo) {
    pdl_launch_dependents();
    pdl_wait();
    extern __shared__ __align__(16) uint8_t stem_smem[];
    f16* s_xh = reinterpret_cast<f16*>(stem_smem);
    f16* s_xl = s_xh + STEM_IT * STEM_XP;
    f16* s_wh = s_xl + STEM_IT * STEM_XP;
    uint32_t* s_stage = reinterpret_cast<uint32_t*>(s_wh + 64 * STEM_WP);
    float* s_vec = reinterpret_cast<float*>(s_stage + 8 * 1024);
    const int b = blockIdx.z;
    const int ho0 = blockIdx.y * 16, wo0 = blockIdx.x * 16;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, tg = lane & 3;
    if (threadIdx.x < 64) s_vec[threadIdx.x] = vec ? vec[(size_t)b * vec_stride + threadIdx.x] : 0.f;
    float acc[2][8][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[mt][nt][i] = 0.f;
    for (int c = 0; c < Cx; ++c) {
        __syncthreads();
        const float* ip = in + ((size_t)b * Cx + c) * Hi * Wi;
        for (int i = threadIdx.x; i < STEM_IT * STEM_IT; i += 256) {
            const int iy = i / STEM_IT, ix = i - iy * STEM_IT;
            const int gy = ho0 * 2 - 3 + iy, gx = wo0 * 2 - 3 + ix;
            const float v = (gy >= 0 && gy < Hi && gx >= 0 && gx < Wi) ? ip[(size_t)gy * Wi + gx] : 0.f;
            const f16 hi = __float2half_rn(v);
            s_xh[iy * STEM_XP + ix] = hi;
            s_xl[iy * STEM_XP + ix] = __float2half_rn(v - __half2float(hi));
        }
        const float* wsrc = w + (size_t)c * 4096;
        for (int i = threadIdx.x; i < 4096; i += 256) {
            const int tap = i >> 6, n = i & 63;
            const float v = __ldg(wsrc + i);
            s_wh[n * STEM_WP + tap] = __float2half_rn(v);
        }
        __syncthreads();
#pragma unroll 1
        for (int kt = 0; kt < 4; ++kt) {
            uint32_t ah[2][4], al[2][4];
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
                const int base = (2 * (2 * warp + mt) + 2 * kt) * STEM_XP + 2 * g + 2 * tg;
                ah[mt][0] = *reinterpret_cast<const uint32_t*>(s_xh + base);
                ah[mt][1] = *reinterpret_cast<const uint32_t*>(s_xh + base + 16);
                ah[mt][2] = *reinterpret_cast<const uint32_t*>(s_xh + base + STEM_XP);
                ah[mt][3] = *reinterpret_cast<const uint32_t*>(s_xh + base + STEM_XP + 16);
                al[mt][0] = *reinterpret_cast<const uint32_t*>(s_xl + base);
                al[mt][1] = *reinterpret_cast<const uint32_t*>(s_xl + base + 16);
                al[mt][2] = *reinterpret_cast<const uint32_t*>(s_xl + base + STEM_XP);
                al[mt][3] = *reinterpret_cast<const uint32_t*>(s_xl + base + STEM_XP + 16);
            }
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
                const int wb = (nt * 8 + g) * STEM_WP + kt * 16 + 2 * tg;
                const uint32_t bh0 = *reinterpret_cast<const uint32_t*>(s_wh + wb);
                const uint32_t bh1 = *reinterpret_cast<const uint32_t*>(s_wh + wb + 8);
#pragma unroll
                for (int mt = 0; mt < 2; ++mt) {
                    mma_f16_16816(acc[mt][nt], ah[mt], bh0, bh1);
                    mma_f16_16816(acc[mt][nt], al[mt], bh0, bh1);
                }
            }
        }
    }
    uint32_t* stg = s_stage + warp * 1024;          // 32 pixels x 128 B
    float satm = 0.f;
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
        const int ho = ho0 + 2 * warp + mt;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int ox = g + 8 * half;
                const int ch = nt * 8 + 2 * tg;
                float v0 = acc[mt][nt][half * 2], v1 = acc[mt][nt][half * 2 + 1];
                if (add) {
                    const float2 a2 = *reinterpret_cast<const float2*>(add + (((size_t)b * Ho + ho) * Wo + wo0 + ox) * 64 + ch);
                    v0 += a2.x;
                    v1 += a2.y;
                }
                v0 += s_vec[ch];
                v1 += s_vec[ch + 1];
                const int p = mt * 16 + ox;
                stg[p * 32 + ((nt * 4 + tg) ^ ((p & 7) << 2))] = pack_h2_acc(v0, v1, satm);
            }
        }
    }
    sat_flush(satm);
    __syncwarp();
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        const int idx = it * 32 + lane;
        const int p = idx >> 3, chunk = idx & 7;
        const uint4 v = *reinterpret_cast<const uint4*>(stg + p * 32 + ((chunk ^ (p & 7)) << 2));
        const int ho = ho0 + 2 * warp + (p >> 4), wo = wo0 + (p & 15);
        *reinterpret_cast<uint4*>(out + (((size_t)b * Ho + ho) * Wo + wo) * 64 + chunk * 8) = v;
    }
}

// ------------------------------------------------------------------------------------------------ InstanceNorm
// Statistics of an NHWC f16 tensor per (sample, channel) plane -> stats[b][c] = {mean, rstd} (biased variance, eps 1e-5:
// InstanceNorm2d defaults, modules_DANRA_conditional.py:409,417).  Deterministic two-level reduction without float
// atomics: every CTA (8 channel chunks of 16 B x 32 pixel lanes over a slab of pixels) writes its partial {sum, sumsq};
// the last CTA to arrive for a (sample, 64-channel group) adds the partials in slab order and publishes mean/rstd.
__global__ void __launch_bounds__(256) plane_stats_kernel(const f16* __restrict__ x, float* __restrict__ partial,
                                                          unsigned int* __restrict__ counters, float* __restrict__ stats,
                                                          int HW, int C, int pix_per_cta) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ float s_sum[32][65], s_sq[32][65];
    __shared__ bool s_last;
    const int b = blockIdx.z, grp = blockIdx.y, ngrp = gridDim.y, nslab = gridDim.x, slab = blockIdx.x;
    const int c0 = grp * 64;
    const int cg8 = (threadIdx.x & 7) * 8, pl = threadIdx.x >> 3;     // 16-byte channel chunk x 32 pixel lanes
    const int p0 = slab * pix_per_cta;
    const int p1 = min(p0 + pix_per_cta, HW);
    float a[8], q[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { a[j] = 0.f; q[j] = 0.f; }
    const f16* xb = x + (size_t)b * HW * C + c0 + cg8;
#pragma unroll 4
    for (int p = p0 + pl; p < p1; p += 32) {
        const uint4 v = *reinterpret_cast<const uint4*>(xb + (size_t)p * C);
        float2 t;
        t = unpack_h2(v.x); a[0] += t.x; a[1] += t.y; q[0] = fmaf(t.x, t.x, q[0]); q[1] = fmaf(t.y, t.y, q[1]);
        t = unpack_h2(v.y); a[2] += t.x; a[3] += t.y; q[2] = fmaf(t.x, t.x, q[2]); q[3] = fmaf(t.y, t.y, q[3]);
        t = unpack_h2(v.z); a[4] += t.x; a[5] += t.y; q[4] = fmaf(t.x, t.x, q[4]); q[5] = fmaf(t.y, t.y, q[5]);
        t = unpack_h2(v.w); a[6] += t.x; a[7] += t.y; q[6] = fmaf(t.x, t.x, q[6]); q[7] = fmaf(t.y, t.y, q[7]);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) { s_sum[pl][cg8 + j] = a[j]; s_sq[pl][cg8 + j] = q[j]; }
    __syncthreads();
    float* part = partial + ((size_t)(b * ngrp + grp) * nslab) * 128;
    if (threadIdx.x < 64) {
        float s = 0.f, q = 0.f;
#pragma unroll
        for (int i = 0; i < 32; ++i) { s += s_sum[i][threadIdx.x]; q += s_sq[i][threadIdx.x]; }
        part[(size_t)slab * 128 + threadIdx.x] = s;
        part[(size_t)slab * 128 + 64 + threadIdx.x] = q;
        __threadfence();
    }
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(&counters[b * ngrp + grp], 1u) == (unsigned)(nslab - 1));
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    if (threadIdx.x < 64) {
        float s = 0.f, q = 0.f;
        for (int i0 = 0; i0 < nslab; i0 += 16) {       // 32 independent loads in flight, then summed in slab order
            float vs[16], vq[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const bool ok = i0 + j < nslab;
                vs[j] = ok ? __ldcg(part + (size_t)(i0 + j) * 128 + threadIdx.x) : 0.f;
                vq[j] = ok ? __ldcg(part + (size_t)(i0 + j) * 128 + 64 + threadIdx.x) : 0.f;
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) { s += vs[j]; q += vq[j]; }
        }
        const float inv = 1.0f / (float)HW;
        const float mean = s * inv;
        const float var = fmaxf(q * inv - mean * mean, 0.f);
        float* st = stats + ((size_t)b * C + c0 + threadIdx.x) * 2;
        st[0] = mean;
        st[1] = rsqrtf(var + 1e-5f);
    }
    if (threadIdx.x == 0) counters[b * ngrp + grp] = 0u;  // self-resetting: no per-step memset
}

// y = (x - mean) * rstd (+ skip) (+ vec[b][c]); stats[b][c] = {mean, rstd}.  8 channels (16 B) per thread.
__global__ void __launch_bounds__(256) instnorm_apply_kernel(const f16* __restrict__ x, const float* __restrict__ stats,
                                                             const f16* __restrict__ skip, const float* __restrict__ vec,
                                                             int vec_stride, f16* __restrict__ y, int HW, int C,
                                                             size_t total_vec8) {
    pdl_launch_dependents();
    pdl_wait();
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total_vec8; i += (size_t)gridDim.x * blockDim.x) {
        const size_t e = i * 8;
        const int c = (int)(e % C);
        const int b = (int)(e / ((size_t)HW * C));
        const uint4 xv = *reinterpret_cast<const uint4*>(x + e);
        float f[8];
        float2 t;
        t = unpack_h2(xv.x); f[0] = t.x; f[1] = t.y;
        t = unpack_h2(xv.y); f[2] = t.x; f[3] = t.y;
        t = unpack_h2(xv.z); f[4] = t.x; f[5] = t.y;
        t = unpack_h2(xv.w); f[6] = t.x; f[7] = t.y;
        const float* st = stats + ((size_t)b * C + c) * 2;
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] = (f[j] - st[2 * j]) * st[2 * j + 1];
        if (skip) {
            const uint4 sv = *reinterpret_cast<const uint4*>(skip + e);
            t = unpack_h2(sv.x); f[0] += t.x; f[1] += t.y;
            t = unpack_h2(sv.y); f[2] += t.x; f[3] += t.y;
            t = unpack_h2(sv.z); f[4] += t.x; f[5] += t.y;
            t = unpack_h2(sv.w); f[6] += t.x; f[7] += t.y;
        }
        if (vec) {
            const float* vp = vec + (size_t)b * vec_stride + c;
#pragma unroll
            for (int j = 0; j < 8; ++j) f[j] += vp[j];
        }
        uint4 o;
        o.x = pack_h2(f[0], f[1]); o.y = pack_h2(f[2], f[3]);
        o.z = pack_h2(f[4], f[5]); o.w = pack_h2(f[6], f[7]);
        *reinterpret_cast<uint4*>(y + e) = o;
    }
}

// ------------------------------------------------------------------------------------------------ tail convolution
// Decoder.final_layer (modules_DANRA_conditional.py:503-509): InstanceNorm(ConvT out) -> Conv3x3(64 -> c_out) + bias, fp32 NCHW
// result (eps_hat).  Cout is 1 (or a few): a 576-long reduction per pixel, not a GEMM.  The normalisation is applied on
// the fly; zero padding applies to the *normalised* tensor, so out-of-image taps contribute nothing.
// CTA = 8 x 32 output pixels: the (8+2) x (32+2) x 64-channel input tile is staged in shared memory with cp.async (all
// loads in flight at once; out-of-image pixels zero-filled).  Thread = (vertical strip of 8 output pixels) x (8 of the 64
// channels): each normalised input vector (16 B) is read once and used by the up-to-3 output rows it touches, with the 72
// weights of the thread's channels in registers; the 8 channel groups of a pixel sit in adjacent lanes and are combined
// with 3 shuffles.  grid = (ceil(W/32), ceil(H/8), B), 256 threads.
constexpr int TAIL_SMEM = 10 * 34 * 64 * 2;
__global__ void __launch_bounds__(256, 2) tail_conv_kernel(const f16* __restrict__ x,       // [B,H,W,64] (un-normalised)
                                                        const float* __restrict__ stats,  // [B][64] x {mean, rstd}
                                                        const float* __restrict__ w,      // [c_out][64][3][3]
                                                        const float* __restrict__ bias, float* __restrict__ out,  // [B,c_out,H,W]
                                                        int H, int W, int c_out) {
    pdl_launch_dependents();
    pdl_wait();
    extern __shared__ __align__(16) uint8_t tail_smem[];
    f16* tile = reinterpret_cast<f16*>(tail_smem);     // [10][34][64]
    const int b = blockIdx.z;
    const int w0 = blockIdx.x * 32, h0 = blockIdx.y * 8;
    for (int i = threadIdx.x; i < 10 * 34 * 8; i += 256) {
        const int ch8 = i & 7, pix = i >> 3;
        const int iy = pix / 34, ix = pix - iy * 34;
        const int hi = h0 - 1 + iy, wi = w0 - 1 + ix;
        const bool ok = hi >= 0 && hi < H && wi >= 0 && wi < W;
        const f16* src = x + (((size_t)b * H + (ok ? hi : 0)) * W + (ok ? wi : 0)) * 64 + ch8 * 8;
        cp_async16(tile + (size_t)pix * 64 + ch8 * 8, src, ok);
    }
    cp_async_commit();
    const int cgp = threadIdx.x & 7;                    // channels cgp*8 .. +7
    const int lcol = threadIdx.x >> 3;                  // 0..31
    const int wcol = w0 + lcol;
    float mean[8], rstd[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const float2 st = *reinterpret_cast<const float2*>(stats + ((size_t)b * 64 + cgp * 8 + c) * 2);
        mean[c] = st.x;
        rstd[c] = st.y;
    }
    cp_async_wait<0>();
    __syncthreads();
    for (int oc = 0; oc < c_out; ++oc) {
        // (v - mean) * rstd * w  ==  v * (rstd * w) - mean * rstd * w: the normalisation is folded into the 72 weights of this
        // thread's channels, and the mean term becomes one constant per filter tap, subtracted only for in-image taps
        // (zero padding applies to the NORMALISED tensor; out-of-image pixels are zero-filled in the tile and add nothing).
        float wr[9][8], mt[9];
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
            float m = 0.f;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                wr[tap][c] = __ldg(w + ((size_t)oc * 64 + cgp * 8 + c) * 9 + tap) * rstd[c];
                m = fmaf(wr[tap][c], mean[c], m);
            }
            mt[tap] = m;
        }
        float acc[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] = 0.f;
#pragma unroll
        for (int ir = 0; ir < 10; ++ir) {
            const int hi = h0 - 1 + ir;
            const bool rok = hi >= 0 && hi < H;
#pragma unroll
            for (int sx = 0; sx < 3; ++sx) {
                const int wi = wcol + sx - 1;
                const bool ok = rok && wi >= 0 && wi < W;
                const uint4 raw = *reinterpret_cast<const uint4*>(tile + ((size_t)(ir * 34 + lcol + sx)) * 64 + cgp * 8);
                float v[8];
                float2 t2;
                t2 = unpack_h2(raw.x); v[0] = t2.x; v[1] = t2.y;
                t2 = unpack_h2(raw.y); v[2] = t2.x; v[3] = t2.y;
                t2 = unpack_h2(raw.z); v[4] = t2.x; v[5] = t2.y;
                t2 = unpack_h2(raw.w); v[6] = t2.x; v[7] = t2.y;
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    const int orow = ir - r;  // output row (within the strip) that sees this input row through filter row r
                    if (orow < 0 || orow >= 8) continue;
                    float a = acc[orow] - (ok ? mt[r * 3 + sx] : 0.f);
#pragma unroll
                    for (int c = 0; c < 8; ++c) a = fmaf(v[c], wr[r * 3 + sx][c], a);
                    acc[orow] = a;
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float a = acc[i];
            a += __shfl_xor_sync(0xffffffffu, a, 1);
            a += __shfl_xor_sync(0xffffffffu, a, 2);
            a += __shfl_xor_sync(0xffffffffu, a, 4);
            acc[i] = a;
        }
        if (cgp == 0 && wcol < W) {
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (h0 + i < H) out[(((size_t)b * c_out + oc) * H + h0 + i) * W + wcol] = acc[i] + bias[oc];
        }
    }
}

// Tensor-core version of the tail convolution for c_out <= 8.  GEMM view: M = output pixel, K = 9 taps x 64 channels, N = 8
// (c_out real columns).  The InstanceNorm is folded into the weights per sample (w' = w * rstd, rounded to fp16 like every
// other layer's weights) and its mean term becomes one constant per (output channel, tap), subtracted in the epilogue
// for in-image taps only (zero padding applies to the NORMALISED tensor).  A fragments come straight from the cp.async-staged
// (10 x 34 pixel) x 64-channel tile with ldmatrix (pixel pitch 144 B: conflict-free).  CTA = 8 x 32 output pixels, 8 warps,
// warp = one output row = two m16 tiles.
constexpr int TAILM_PP = 72;                 // halves per pixel in the tile (64 + 8 pad)
constexpr int TAILM_WP = 584;                // halves per weight row (576 + 8 pad)
constexpr int TAILM_SMEM = 10 * 34 * TAILM_PP * 2 + 8 * TAILM_WP * 2 + 8 * 9 * 4 + 128 * 4;
__global__ void __launch_bounds__(256, 2) tail_mma_kernel(const f16* __restrict__ x,       // [B,H,W,64] (un-normalised)
                                                          const float* __restrict__ stats,  // [B][64] x {mean, rstd}
                                                          const float* __restrict__ w,      // K-major [c_out][tap * 64 + c]
                                                          const float* __restrict__ bias, float* __restrict__ out,  // [B,c_out,H,W]
                                                          int H, int W, int c_out) {
    pdl_launch_dependents();
    extern __shared__ __align__(16) uint8_t tailm_smem[];
    f16* tile = reinterpret_cast<f16*>(tailm_smem);                 // [10][34][72]
    f16* s_wh = tile + 10 * 34 * TAILM_PP;                          // [8][584]
    float* s_mt = reinterpret_cast<float*>(s_wh + 8 * TAILM_WP);    // [8][9] mean term per (output channel, tap)
    float* s_st = s_mt + 72;                                        // [64] x {mean, rstd}
    const int b = blockIdx.z;
    const int w0 = blockIdx.x * 32, h0 = blockIdx.y * 8;
    pdl_wait();
    {   // tile load: thread = (16-byte channel chunk, column); columns 32/33 of each row by the first 160 threads
        const int ch8 = threadIdx.x & 7, ixl = threadIdx.x >> 3;
        const f16* xb = x + (size_t)b * H * W * 64 + ch8 * 8;
        {
            const int wi = w0 - 1 + ixl;
            const bool cok = wi >= 0 && wi < W;
#pragma unroll
            for (int iy = 0; iy < 10; ++iy) {
                const int hi = h0 - 1 + iy;
                const bool ok = cok && hi >= 0 && hi < H;
                cp_async16(tile + (size_t)(iy * 34 + ixl) * TAILM_PP + ch8 * 8, xb + ((size_t)(ok ? hi : 0) * W + (ok ? wi : 0)) * 64, ok);
            }
        }
        if (threadIdx.x < 160) {
            const int iy = threadIdx.x >> 4, ix = 32 + ((threadIdx.x >> 3) & 1);
            const int hi = h0 - 1 + iy, wi = w0 - 1 + ix;
            const bool ok = hi >= 0 && hi < H && wi >= 0 && wi < W;
            cp_async16(tile + (size_t)(iy * 34 + ix) * TAILM_PP + ch8 * 8, xb + ((size_t)(ok ? hi : 0) * W + (ok ? wi : 0)) * 64, ok);
        }
    }
    cp_async_commit();
    if (threadIdx.x < 128) s_st[threadIdx.x] = stats[(size_t)b * 128 + threadIdx.x];
    {   // rows n >= c_out of the B operand are zero
        uint4* z = reinterpret_cast<uint4*>(s_wh + (size_t)c_out * TAILM_WP);
        const int nz = (8 - c_out) * TAILM_WP / 8;
        for (int i = threadIdx.x; i < nz; i += 256) z[i] = make_uint4(0, 0, 0, 0);
    }
    __syncthreads();
    // folded weights: w is K-major [n][tap * 64 + c]
    const int warp_ = threadIdx.x >> 5, lane_ = threadIdx.x & 31;
    for (int n = 0; n < c_out; ++n) {
        for (int k = threadIdx.x; k < 576; k += 256)
            s_wh[n * TAILM_WP + k] = __float2half_rn(__ldg(w + (size_t)n * 576 + k) * s_st[2 * (k & 63) + 1]);
        for (int tap = warp_; tap < 9; tap += 8) {
            const float* wr = w + (size_t)n * 576 + tap * 64;
            float m = __ldg(wr + lane_) * s_st[2 * lane_ + 1] * s_st[2 * lane_] +
                      __ldg(wr + lane_ + 32) * s_st[2 * (lane_ + 32) + 1] * s_st[2 * (lane_ + 32)];
            m = warp_sum(m);
            if (lane_ == 0) s_mt[n * 9 + tap] = m;
        }
    }
    cp_async_wait<0>();
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, tg = lane & 3;
    float acc[2][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[mt][i] = 0.f;
    // ldmatrix row address of this lane: pixel (lane & 7) + 8 * ((lane >> 3) & 1), channel offset 8 * (lane >> 4)
    const int lpix = (lane & 7) + ((lane >> 3) & 1) * 8, lch = (lane >> 4) * 8;
    const uint32_t tile_u = smem_u32(tile);
#pragma unroll 1
    for (int tap = 0; tap < 9; ++tap) {
        const int ky = tap / 3, kx = tap - ky * 3;
        const uint32_t rowbase = tile_u + (uint32_t)((((warp + ky) * 34) + kx + lpix) * TAILM_PP + lch) * 2;
#pragma unroll
        for (int kc = 0; kc < 4; ++kc) {
            uint32_t a0[4], a1[4];
            ldmatrix_x4(a0, rowbase + kc * 32);
            ldmatrix_x4(a1, rowbase + 16 * TAILM_PP * 2 + kc * 32);
            const int wb = g * TAILM_WP + tap * 64 + kc * 16 + 2 * tg;
            const uint32_t bh0 = *reinterpret_cast<const uint32_t*>(s_wh + wb);
            const uint32_t bh1 = *reinterpret_cast<const uint32_t*>(s_wh + wb + 8);
            mma_f16_16816(acc[0], a0, bh0, bh1);
            mma_f16_16816(acc[1], a1, bh0, bh1);
        }
    }
    const int ho = h0 + warp;
    if (ho >= H) return;
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int wo = w0 + mt * 16 + g + 8 * half;
            if (wo >= W) continue;
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int n = 2 * tg + j;
                if (n >= c_out) continue;
                float corr = 0.f;
#pragma unroll
                for (int tap = 0; tap < 9; ++tap) {
                    const int hi = ho + tap / 3 - 1, wi = wo + tap % 3 - 1;
                    if (hi >= 0 && hi < H && wi >= 0 && wi < W) corr += s_mt[n * 9 + tap];
                }
                out[(((size_t)b * c_out + n) * H + ho) * W + wo] = acc[mt][half * 2 + j] - corr + bias[n];
            }
        }
}

// ------------------------------------------------------------------------------------------------ posterior update
// diffusion_DANRA_conditional.py:135-157:  x <- (1/sqrt(alpha_i)) * (x - ((1-alpha_i)/sqrt(1-alpha_hat_i)) * eps) + sqrt(beta_i) * z
// with coefficients indexed by i itself, z = 0 at i == 1.  Same op order as the reference and no FMA contraction so that
// identical eps/z give bit-identical x.  z is either host-provided (noise[i][...], parity runs) or drawn in-kernel from
// Philox4x32-10 keyed by (seed; global sample index, element, step) so results do not depend on how the batch is sharded.
__device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
    c[0] = hi1 ^ c[1] ^ k0;
    c[1] = lo1;
    c[2] = hi0 ^ c[3] ^ k1;
    c[3] = lo0;
}
__device__ __forceinline__ void philox4x32_10(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        philox_round(c, k0, k1);
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
}
__device__ __forceinline__ float2 box_muller(uint32_t a, uint32_t b) {
    const float u1 = ((float)a + 1.0f) * 2.3283064365386963e-10f;  // (0,1]
    const float u2 = (float)b * 2.3283064365386963e-10f;
    const float r = sqrtf(-2.0f * logf(u1));
    float s, c;
    sincosf(6.283185307179586f * u2, &s, &c);
    return make_float2(r * c, r * s);
}

// Everything a sampling job may change between calls, resident in device memory so that the captured step graphs never
// depend on it (b2d_sample writes the block with set_job_kernel before the first replay).
struct SampleJob {
    const float* noise;                 // host-injected z: [T][noise_stride] indexed by i, or null = in-kernel Philox
    unsigned long long seed, sample_offset;
    unsigned long long noise_stride;    // elements per step of `noise`
    float noise_scale;                  // multiplies z (1.0; 0.005 for data_scaled, src/diffusion_modules.py:173-174)
    int pad;
};
__global__ void set_job_kernel(SampleJob* job, SampleJob v, int* t_arr, int* step_ptr, int i0, int B) {
    pdl_launch_dependents();
    pdl_wait();
    if (threadIdx.x == 0) {
        *job = v;
        step_ptr[0] = i0;
        step_ptr[1] = 0;
    }
    for (int b = threadIdx.x; b < B; b += blockDim.x) t_arr[b] = i0;
}

// step_ptr[0] holds the current i (device-resident so one captured graph is replayed for every step).
// t_arr[b] is rewritten to i-1 for the next evaluation.  4 elements per thread (n % 4 == 0 and per_sample % 4 == 0 are
// checked by the C entry points).
__global__ void __launch_bounds__(256) posterior_update_kernel(float* __restrict__ x, const float* __restrict__ eps,
                                                               const SampleJob* __restrict__ job,
                                                               const float* __restrict__ alphas, const float* __restrict__ betas,
                                                               const float* __restrict__ alpha_hat, int* __restrict__ step_ptr,
                                                               int* __restrict__ t_arr, int B, size_t n, size_t per_sample) {
    pdl_launch_dependents();
    pdl_wait();
    const int i = *step_ptr;
    const float* noise = job->noise;
    const unsigned long long seed = job->seed, sample_offset = job->sample_offset;
    const size_t noise_stride = job->noise_stride;
    const float noise_scale = job->noise_scale;
    const float alpha = alphas[i], beta = betas[i], ahat = alpha_hat[i];
    const float c1 = __fdiv_rn(1.0f, __fsqrt_rn(alpha));
    const float c2 = __fdiv_rn(__fsub_rn(1.0f, alpha), __fsqrt_rn(__fsub_rn(1.0f, ahat)));
    const float c3 = __fsqrt_rn(beta);
    const size_t n4 = n >> 2;
    for (size_t v = blockIdx.x * (size_t)blockDim.x + threadIdx.x; v < n4; v += (size_t)gridDim.x * blockDim.x) {
        float4 xv = reinterpret_cast<float4*>(x)[v];
        const float4 ev = reinterpret_cast<const float4*>(eps)[v];
        float4 zv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i > 1) {
            if (noise) {   // injected z stands in for randn_like's output: the data_scaled factor applies to it too (:173-174)
                zv = reinterpret_cast<const float4*>(noise + (size_t)i * noise_stride)[v];
                zv = make_float4(__fmul_rn(zv.x, noise_scale), __fmul_rn(zv.y, noise_scale), __fmul_rn(zv.z, noise_scale),
                                 __fmul_rn(zv.w, noise_scale));
            } else {
                const size_t e = v * 4;
                const unsigned long long sample = sample_offset + e / per_sample;
                const unsigned long long within = (e % per_sample) >> 2;
                uint32_t c[4] = {(uint32_t)within, (uint32_t)i, (uint32_t)sample, (uint32_t)(sample >> 32)};
                philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
                const float2 g0 = box_muller(c[0], c[1]), g1 = box_muller(c[2], c[3]);
                zv = make_float4(g0.x * noise_scale, g0.y * noise_scale, g1.x * noise_scale, g1.y * noise_scale);
            }
        }
        xv.x = __fadd_rn(__fmul_rn(c1, __fsub_rn(xv.x, __fmul_rn(c2, ev.x))), __fmul_rn(c3, zv.x));
        xv.y = __fadd_rn(__fmul_rn(c1, __fsub_rn(xv.y, __fmul_rn(c2, ev.y))), __fmul_rn(c3, zv.y));
        xv.z = __fadd_rn(__fmul_rn(c1, __fsub_rn(xv.z, __fmul_rn(c2, ev.z))), __fmul_rn(c3, zv.z));
        xv.w = __fadd_rn(__fmul_rn(c1, __fsub_rn(xv.w, __fmul_rn(c2, ev.w))), __fmul_rn(c3, zv.w));
        reinterpret_cast<float4*>(x)[v] = xv;
    }
    // Inside the reverse loop (t_arr != nullptr) the last block to finish advances the device-resident step state for the next
    // UNet evaluation: i <- i-1, t[b] <- i-1.  Every block read *step_ptr before it arrives, so nobody sees the new value early.
    // step_ptr[1] is the (self-resetting) arrival counter.
    if (t_arr != nullptr) {
        __shared__ bool s_last;
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            s_last = atomicAdd(reinterpret_cast<unsigned int*>(step_ptr + 1), 1u) == gridDim.x - 1;
        }
        __syncthreads();
        if (s_last) {
            for (int b = threadIdx.x; b < B; b += blockDim.x) t_arr[b] = i - 1;
            if (threadIdx.x == 0) {
                step_ptr[0] = i - 1;
                step_ptr[1] = 0;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------ DDIM update
// Song, Meng & Ermon 2021, eq. 12, over a strided timestep sequence tau_0 > tau_1 > ... > tau_{S-1} (every tau_k in [1, T-1]).
// Step k goes from t = tau_k to t' = tau_{k+1}; a = alpha_hat[t], a' = alpha_hat[t'] (a' = 1 after the last step: x0_hat):
//   x0_hat = (x - sqrt(1-a) eps) / sqrt(a)
//   sigma  = eta * sqrt((1-a')/(1-a)) * sqrt(1 - a/a')
//   x'     = sqrt(a') x0_hat + sqrt(max(0, 1-a'-sigma^2)) eps + sigma * noise_scale * z
// folded into x' = cx x + ce eps + sigma (noise_scale z) with cx = sqrt(a'/a) and ce = sqrt(max(0, 1-a'-sigma^2)) - cx sqrt(1-a).
// The coefficients are computed here, on the host, in double from the fp32 alpha_hat values: the square roots of differences of
// nearby alpha_hat values lose most of their bits in fp32.  Both the handle's per-step table and b2d_op_ddim_update use this
// function.  No x0_hat clipping (the reference has none); sigma is 0 on the last step and for eta = 0, so no noise is drawn there.
inline float4 ddim_coefficients(float abar, float abar_next, float eta) {
    const double a = abar, an = abar_next;
    const double sigma = (double)eta * std::sqrt((1.0 - an) / (1.0 - a)) * std::sqrt(std::max(0.0, 1.0 - a / an));
    const double cx = std::sqrt(an / a);
    const double ce = std::sqrt(std::max(0.0, 1.0 - an - sigma * sigma)) - cx * std::sqrt(1.0 - a);
    return make_float4((float)cx, (float)ce, (float)sigma, 0.f);
}

// Reverse-loop state of a DDIM job: k = 0, t[b] = tau_0 for the first evaluation, t_next[b] = tau_1 for the time-embedding
// side branch that runs before the first update.  tau is the device table [S + 2] (two trailing zeros).
__global__ void set_job_ddim_kernel(SampleJob* job, SampleJob v, const int* __restrict__ tau, int* t_arr, int* t_next_arr,
                                    int* step_ptr, int B) {
    pdl_launch_dependents();
    pdl_wait();
    if (threadIdx.x == 0) {
        *job = v;
        step_ptr[0] = 0;
        step_ptr[1] = 0;
    }
    const int t0 = tau[0], t1 = tau[1];
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
        t_arr[b] = t0;
        t_next_arr[b] = t1;
    }
}

// State, sequence and coefficients of one stand-alone step (b2d_op_ddim_update), written in stream order.
__global__ void ddim_op_setup_kernel(SampleJob* job, SampleJob v, int* step_ptr, int* tau, float4* coef, int t, float4 c) {
    if (threadIdx.x == 0) {
        *job = v;
        step_ptr[0] = 0;
        step_ptr[1] = 0;
        tau[0] = t;
        coef[0] = c;
    }
}

// step_ptr[0] holds k; tau [S + 2] and coef [S] = {cx, ce, sigma, 0} are device tables written by the host.  z is host-injected
// (noise[k][...]) or drawn from the same Philox stream as posterior_update_kernel with the step slot set to tau_k.  Inside the
// reverse loop (t_arr != nullptr) the last block to arrive writes t[b] = tau_{k+1} (the next evaluation) and
// t_next[b] = tau_{k+2} (the time embeddings the side branch of that evaluation precomputes), then k <- k+1.
__global__ void __launch_bounds__(256) ddim_update_kernel(float* __restrict__ x, const float* __restrict__ eps,
                                                          const SampleJob* __restrict__ job, const int* __restrict__ tau,
                                                          const float4* __restrict__ coef, int* __restrict__ step_ptr,
                                                          int* __restrict__ t_arr, int* __restrict__ t_next_arr, int B, size_t n,
                                                          size_t per_sample) {
    pdl_launch_dependents();
    pdl_wait();
    const int k = *step_ptr;
    const int t = tau[k];
    const float4 c = coef[k];
    const float* noise = job->noise;
    const unsigned long long seed = job->seed, sample_offset = job->sample_offset;
    const size_t noise_stride = job->noise_stride;
    const float noise_scale = job->noise_scale;
    const bool draw = c.z != 0.f;
    const size_t n4 = n >> 2;
    for (size_t v = blockIdx.x * (size_t)blockDim.x + threadIdx.x; v < n4; v += (size_t)gridDim.x * blockDim.x) {
        float4 xv = reinterpret_cast<float4*>(x)[v];
        const float4 ev = reinterpret_cast<const float4*>(eps)[v];
        float4 zv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (draw) {
            if (noise) {
                zv = reinterpret_cast<const float4*>(noise + (size_t)k * noise_stride)[v];
                zv = make_float4(zv.x * noise_scale, zv.y * noise_scale, zv.z * noise_scale, zv.w * noise_scale);
            } else {
                const size_t e = v * 4;
                const unsigned long long sample = sample_offset + e / per_sample;
                const unsigned long long within = (e % per_sample) >> 2;
                uint32_t ctr[4] = {(uint32_t)within, (uint32_t)t, (uint32_t)sample, (uint32_t)(sample >> 32)};
                philox4x32_10(ctr, (uint32_t)seed, (uint32_t)(seed >> 32));
                const float2 g0 = box_muller(ctr[0], ctr[1]), g1 = box_muller(ctr[2], ctr[3]);
                zv = make_float4(g0.x * noise_scale, g0.y * noise_scale, g1.x * noise_scale, g1.y * noise_scale);
            }
        }
        xv.x = fmaf(c.z, zv.x, fmaf(c.y, ev.x, c.x * xv.x));
        xv.y = fmaf(c.z, zv.y, fmaf(c.y, ev.y, c.x * xv.y));
        xv.z = fmaf(c.z, zv.z, fmaf(c.y, ev.z, c.x * xv.z));
        xv.w = fmaf(c.z, zv.w, fmaf(c.y, ev.w, c.x * xv.w));
        reinterpret_cast<float4*>(x)[v] = xv;
    }
    if (t_arr != nullptr) {
        __shared__ bool s_last;
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            s_last = atomicAdd(reinterpret_cast<unsigned int*>(step_ptr + 1), 1u) == gridDim.x - 1;
        }
        __syncthreads();
        if (s_last) {
            const int t1 = tau[k + 1], t2 = tau[k + 2];
            for (int b = threadIdx.x; b < B; b += blockDim.x) {
                t_arr[b] = t1;
                t_next_arr[b] = t2;
            }
            if (threadIdx.x == 0) {
                step_ptr[0] = k + 1;
                step_ptr[1] = 0;
            }
        }
    }
}

// x_T ~ N(0,1) * scale drawn on the device (ensemble driver): same Philox keying as the per-step noise — (seed; global sample
// index, element) — with the step slot set to 0x7FFFFFFF, which no reverse step uses, so members are independent of how the
// ensemble is cut into sub-batches and ranks.
__global__ void __launch_bounds__(256) init_noise_kernel(float* __restrict__ x, size_t n, size_t per_sample, unsigned long long seed,
                                                         unsigned long long sample_offset, float scale) {
    pdl_launch_dependents();
    pdl_wait();
    const size_t n4 = n >> 2;
    for (size_t v = blockIdx.x * (size_t)blockDim.x + threadIdx.x; v < n4; v += (size_t)gridDim.x * blockDim.x) {
        const size_t e = v * 4;
        const unsigned long long sample = sample_offset + e / per_sample;
        const unsigned long long within = (e % per_sample) >> 2;
        uint32_t c[4] = {(uint32_t)within, 0x7FFFFFFFu, (uint32_t)sample, (uint32_t)(sample >> 32)};
        philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
        const float2 g0 = box_muller(c[0], c[1]), g1 = box_muller(c[2], c[3]);
        reinterpret_cast<float4*>(x)[v] = make_float4(g0.x * scale, g0.y * scale, g1.x * scale, g1.y * scale);
    }
}
__global__ void fill_int_kernel(int* p, int v, int n) {
    pdl_launch_dependents();
    pdl_wait();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

}  // namespace b2d
