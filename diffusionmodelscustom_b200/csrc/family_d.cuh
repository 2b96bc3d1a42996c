// Family D — UNet_downscale (DDPM_clean_application/src/unet_ms.py:103-179): kernels that only this family needs, weight
// packing and the per-step program.  Included by b200ddpm.cu after Handle/Builder are defined.
//   DoubleConv (:30-49)  = conv3x3 -> GroupNorm(1,C) -> GELU -> conv3x3 -> GroupNorm(1,C) [-> gelu(x + .) if residual]
//   Down (:52-73)        = MaxPool2d(2) -> DoubleConv(res) -> DoubleConv, + Linear(SiLU(t_emb))
//   Up (:76-100)         = bilinear x2 (align_corners=True) -> cat[skip, x] -> DoubleConv(res) -> DoubleConv(mid=in/2), + emb
//   SelfAttention (:6-27)= LN -> MHA(4 heads) -> +x -> +FF(LN, Linear, GELU, Linear)
// The 3x3 convolutions and all projections run on the tcgen05 implicit-GEMM kernel; GroupNorm(1,C) is a per-sample
// LayerNorm over C*H*W done as a deterministic two-level reduction + one fused apply (affine, residual, GELU, +emb).
#pragma once
namespace b2d {

// ------------------------------------------------------------------------------------------------ bicubic resize (once)
// torch upsample_bicubic2d, align_corners=False, A=-0.75 (F.interpolate(y, size, mode='bicubic'), unet_ms.py:156).
__device__ __forceinline__ float cubic1(float x, float A) { return ((A + 2.f) * x - (A + 3.f)) * x * x + 1.f; }
__device__ __forceinline__ float cubic2(float x, float A) { return ((A * x - 5.f * A) * x + 8.f * A) * x - 4.f * A; }
__global__ void __launch_bounds__(256) bicubic_resize_kernel(const float* __restrict__ in, float* __restrict__ out, int planes,
                                                             int hi, int wi, int Ho, int Wo) {
    pdl_launch_dependents();
    pdl_wait();
    const size_t total = (size_t)planes * Ho * Wo;
    const float A = -0.75f;
    const float sh = (float)hi / (float)Ho, sw = (float)wi / (float)Wo;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int ox = (int)(idx % Wo);
        const int oy = (int)((idx / Wo) % Ho);
        const int pl = (int)(idx / ((size_t)Wo * Ho));
        const float ry = sh * (oy + 0.5f) - 0.5f, rx = sw * (ox + 0.5f) - 0.5f;
        const float fy = floorf(ry), fx = floorf(rx);
        const float ty = ry - fy, tx = rx - fx;
        const int iy = (int)fy, ix = (int)fx;
        const float wy[4] = {cubic2(ty + 1.f, A), cubic1(ty, A), cubic1(1.f - ty, A), cubic2(2.f - ty, A)};
        const float wx[4] = {cubic2(tx + 1.f, A), cubic1(tx, A), cubic1(1.f - tx, A), cubic2(2.f - tx, A)};
        const float* p = in + (size_t)pl * hi * wi;
        float acc = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int yy = min(max(iy - 1 + j, 0), hi - 1);
            float row = 0.f;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int xx = min(max(ix - 1 + i, 0), wi - 1);
                row += p[(size_t)yy * wi + xx] * wx[i];
            }
            acc += row * wy[j];
        }
        out[idx] = acc;
    }
}

// F.interpolate(y, size, mode='bilinear') (align_corners=False: src = scale * (dst + 0.5) - 0.5 clamped at 0) and
// mode='nearest' (src = floor(dst * scale)): the other interp_mode values of UNet_downscale (unet_ms.py:105,156).
__global__ void __launch_bounds__(256) linear_nearest_resize_kernel(const float* __restrict__ in, float* __restrict__ out, int planes,
                                                                    int hi, int wi, int Ho, int Wo, int nearest) {
    pdl_launch_dependents();
    pdl_wait();
    const size_t total = (size_t)planes * Ho * Wo;
    const float sh = (float)hi / (float)Ho, sw = (float)wi / (float)Wo;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int ox = (int)(idx % Wo);
        const int oy = (int)((idx / Wo) % Ho);
        const float* p = in + (size_t)(idx / ((size_t)Wo * Ho)) * hi * wi;
        if (nearest) {
            const int iy = min((int)floorf(oy * sh), hi - 1), ix = min((int)floorf(ox * sw), wi - 1);
            out[idx] = p[(size_t)iy * wi + ix];
            continue;
        }
        const float ry = fmaxf(sh * (oy + 0.5f) - 0.5f, 0.f), rx = fmaxf(sw * (ox + 0.5f) - 0.5f, 0.f);
        const int y0 = (int)ry, x0 = (int)rx;
        const int y1 = y0 + (y0 < hi - 1 ? 1 : 0), x1 = x0 + (x0 < wi - 1 ? 1 : 0);
        const float ly = ry - (float)y0, lx = rx - (float)x0;
        const float hy = 1.f - ly, hx = 1.f - lx;
        // torch's upsample_bilinear2d order: h0 * (w0 * a + w1 * b) + h1 * (w0 * c + w1 * d)
        out[idx] = hy * (hx * p[(size_t)y0 * wi + x0] + lx * p[(size_t)y0 * wi + x1]) +
                   ly * (hx * p[(size_t)y1 * wi + x0] + lx * p[(size_t)y1 * wi + x1]);
    }
}

// ------------------------------------------------------------------------------------------------ GroupNorm(1, C)
// Per-sample {mean, rstd} over all C*H*W elements of an NHWC f16 tensor (biased variance, eps 1e-5).  Deterministic:
// per-slab partials, last-arriving CTA of a sample adds them in slab order.  grid = (nslab, B).
__global__ void __launch_bounds__(256) sample_stats_kernel(const f16* __restrict__ x, float* __restrict__ partial,
                                                           unsigned int* __restrict__ counters, float* __restrict__ stats,
                                                           size_t per_sample, size_t slab_elems) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ float s_s[8], s_q[8];
    __shared__ bool s_last;
    const int b = blockIdx.y, slab = blockIdx.x, nslab = gridDim.x;
    const size_t e0 = (size_t)slab * slab_elems;
    const size_t e1 = min(e0 + slab_elems, per_sample);
    const f16* xb = x + (size_t)b * per_sample;
    float s = 0.f, q = 0.f;
    for (size_t e = e0 + (size_t)threadIdx.x * 8; e < e1; e += 256 * 8) {
        const uint4 v = *reinterpret_cast<const uint4*>(xb + e);
        float2 t;
        t = unpack_h2(v.x); s += t.x + t.y; q = fmaf(t.x, t.x, q); q = fmaf(t.y, t.y, q);
        t = unpack_h2(v.y); s += t.x + t.y; q = fmaf(t.x, t.x, q); q = fmaf(t.y, t.y, q);
        t = unpack_h2(v.z); s += t.x + t.y; q = fmaf(t.x, t.x, q); q = fmaf(t.y, t.y, q);
        t = unpack_h2(v.w); s += t.x + t.y; q = fmaf(t.x, t.x, q); q = fmaf(t.y, t.y, q);
    }
    s = warp_sum(s);
    q = warp_sum(q);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { s_s[warp] = s; s_q[warp] = q; }
    __syncthreads();
    if (threadIdx.x == 0) {
        float ts = 0.f, tq = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) { ts += s_s[i]; tq += s_q[i]; }
        partial[((size_t)b * nslab + slab) * 2] = ts;
        partial[((size_t)b * nslab + slab) * 2 + 1] = tq;
        __threadfence();
        s_last = (atomicAdd(&counters[b], 1u) == (unsigned)(nslab - 1));
    }
    __syncthreads();
    if (!s_last) return;
    if (threadIdx.x < 32) {
        __threadfence();
        double ts = 0.0, tq = 0.0;   // few dozen partials: fp64 here costs nothing and removes the cancellation worry
        for (int i = threadIdx.x; i < nslab; i += 32) {   // lane-parallel loads, fixed reduction tree => deterministic
            ts += (double)__ldcg(partial + ((size_t)b * nslab + i) * 2);
            tq += (double)__ldcg(partial + ((size_t)b * nslab + i) * 2 + 1);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            ts += __shfl_xor_sync(0xffffffffu, ts, o);
            tq += __shfl_xor_sync(0xffffffffu, tq, o);
        }
        if (threadIdx.x == 0) {
            const double mean = ts / (double)per_sample;
            const double var = fmax(tq / (double)per_sample - mean * mean, 0.0);
            stats[b * 2] = (float)mean;
            stats[b * 2 + 1] = (float)(1.0 / sqrt(var + 1e-5));
            counters[b] = 0u;
        }
    }
}

// y = act( (x - mean_b) * rstd_b * gamma_c + beta_c  (+ res) ) (+ vec[b][c]);  act: 0 none, 2 GELU(erf).
// Statistics come either from stats[b] = {mean, rstd} (sample_stats_kernel) or from the per-tile {sum, sumsq} partials the
// producing convolution wrote in its epilogue (gn_partial: [ntiles][mtiles][2], sample b owns m-tiles [b*tps, (b+1)*tps)):
// every CTA of sample b adds them in the same fixed order.  grid = (chunks, B).
constexpr int GNA_ITER = 4;
__global__ void __launch_bounds__(256) groupnorm_apply_kernel(const f16* __restrict__ x, const float* __restrict__ stats,
                                                              const float* __restrict__ gn_partial, int tps, int ntiles, int mtiles,
                                                              const float* __restrict__ gamma, const float* __restrict__ beta,
                                                              const f16* __restrict__ res, int act,
                                                              const float* __restrict__ vec, int vec_stride,
                                                              f16* __restrict__ y, size_t per_sample, int C) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ float s_ms[2];
    const int b = blockIdx.y;
    if (gn_partial != nullptr) {
        if (threadIdx.x < 32) {
            double ts = 0.0, tq = 0.0;
            const int cnt = tps * ntiles;
            for (int i = threadIdx.x; i < cnt; i += 32) {
                const int nb = i / tps, mt = b * tps + (i - nb * tps);
                ts += (double)__ldcg(gn_partial + ((size_t)nb * mtiles + mt) * 2);
                tq += (double)__ldcg(gn_partial + ((size_t)nb * mtiles + mt) * 2 + 1);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                ts += __shfl_xor_sync(0xffffffffu, ts, o);
                tq += __shfl_xor_sync(0xffffffffu, tq, o);
            }
            if (threadIdx.x == 0) {
                const double mean = ts / (double)per_sample;
                const double var = fmax(tq / (double)per_sample - mean * mean, 0.0);
                s_ms[0] = (float)mean;
                s_ms[1] = (float)(1.0 / sqrt(var + 1e-5));
            }
        }
    } else if (threadIdx.x == 0) {
        s_ms[0] = stats[b * 2];
        s_ms[1] = stats[b * 2 + 1];
    }
    __syncthreads();
    const float mean = s_ms[0], rstd = s_ms[1];
    const size_t n8 = per_sample / 8;
    // Every CTA covers GNA_ITER * 256 consecutive 16-byte vectors; 256 * 8 elements are a multiple of C (checked on the host), so
    // a thread's eight channels are the same in every iteration: gamma / beta are folded once into  y = a * x + c,
    // and all of the thread's loads are issued before the (GELU-heavy) arithmetic starts.
    const int c = (int)((threadIdx.x * 8) % C);
    float aa[8], cc[8];
    {
        const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma + c)), g1 = __ldg(reinterpret_cast<const float4*>(gamma + c + 4));
        const float4 b0 = __ldg(reinterpret_cast<const float4*>(beta + c)), b1 = __ldg(reinterpret_cast<const float4*>(beta + c + 4));
        const float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
        const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            aa[j] = rstd * gg[j];
            cc[j] = fmaf(-mean, aa[j], bb[j]);
            if (vec) cc[j] += act == 2 ? 0.f : vec[(size_t)b * vec_stride + c + j];   // the vector is added AFTER the activation
        }
    }
    float vv[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) vv[j] = (vec && act == 2) ? vec[(size_t)b * vec_stride + c + j] : 0.f;
    const size_t i0 = (size_t)blockIdx.x * (GNA_ITER * 256) + threadIdx.x;
    uint4 xv[GNA_ITER], rv[GNA_ITER];
    float satm = 0.f;
#pragma unroll
    for (int it = 0; it < GNA_ITER; ++it) {
        const size_t i = i0 + (size_t)it * 256;
        if (i < n8) {
            const size_t e = (size_t)b * per_sample + i * 8;
            xv[it] = *reinterpret_cast<const uint4*>(x + e);
            if (res) rv[it] = *reinterpret_cast<const uint4*>(res + e);
        }
    }
#pragma unroll
    for (int it = 0; it < GNA_ITER; ++it) {
        const size_t i = i0 + (size_t)it * 256;
        if (i >= n8) break;
        const size_t e = (size_t)b * per_sample + i * 8;
        float f[8];
        float2 t;
        t = unpack_h2(xv[it].x); f[0] = t.x; f[1] = t.y;
        t = unpack_h2(xv[it].y); f[2] = t.x; f[3] = t.y;
        t = unpack_h2(xv[it].z); f[4] = t.x; f[5] = t.y;
        t = unpack_h2(xv[it].w); f[6] = t.x; f[7] = t.y;
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] = fmaf(f[j], aa[j], cc[j]);
        if (res) {
            t = unpack_h2(rv[it].x); f[0] += t.x; f[1] += t.y;
            t = unpack_h2(rv[it].y); f[2] += t.x; f[3] += t.y;
            t = unpack_h2(rv[it].z); f[4] += t.x; f[5] += t.y;
            t = unpack_h2(rv[it].w); f[6] += t.x; f[7] += t.y;
        }
        if (act == 2) {
#pragma unroll
            for (int j = 0; j < 8; ++j) f[j] = gelu_erf(f[j]) + vv[j];
        }
        uint4 o;
        o.x = pack_h2_acc(f[0], f[1], satm); o.y = pack_h2_acc(f[2], f[3], satm);
        o.z = pack_h2_acc(f[4], f[5], satm); o.w = pack_h2_acc(f[6], f[7], satm);
        *reinterpret_cast<uint4*>(y + e) = o;
    }
    sat_flush(satm);
}

// ------------------------------------------------------------------------------------------------ MaxPool2d(2), NHWC
__global__ void __launch_bounds__(256) maxpool2_kernel(const f16* __restrict__ x, f16* __restrict__ y, int B, int Ho, int Wo,
                                                       int C) {
    pdl_launch_dependents();
    pdl_wait();
    const size_t total8 = (size_t)B * Ho * Wo * C / 8;
    const int c8n = C / 8;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total8; i += (size_t)gridDim.x * blockDim.x) {
        const int c8 = (int)(i % c8n);
        size_t pix = i / c8n;
        const int wo = (int)(pix % Wo);
        pix /= Wo;
        const int ho = (int)(pix % Ho);
        const int b = (int)(pix / Ho);
        const f16* p = x + ((((size_t)b * (2 * Ho) + 2 * ho) * (2 * Wo)) + 2 * wo) * C + c8 * 8;
        const uint4 a = *reinterpret_cast<const uint4*>(p);
        const uint4 bq = *reinterpret_cast<const uint4*>(p + C);
        const uint4 c = *reinterpret_cast<const uint4*>(p + (size_t)2 * Wo * C);
        const uint4 d = *reinterpret_cast<const uint4*>(p + (size_t)2 * Wo * C + C);
        uint4 o;
        const f162* pa = reinterpret_cast<const f162*>(&a);
        const f162* pb = reinterpret_cast<const f162*>(&bq);
        const f162* pc = reinterpret_cast<const f162*>(&c);
        const f162* pd = reinterpret_cast<const f162*>(&d);
        f162* po = reinterpret_cast<f162*>(&o);
#pragma unroll
        for (int j = 0; j < 4; ++j) po[j] = __hmax2(__hmax2(pa[j], pb[j]), __hmax2(pc[j], pd[j]));
        *reinterpret_cast<uint4*>(y + i * 8) = o;
    }
}

// ------------------------------------------------------------------------------------------------ Upsample x2 + concat
// out[b,y,x, 0:Cs] = skip[b,y,x,:];  out[b,y,x, Cs:Cs+Cx] = bilinear(xin)[b,y,x,:]  (nn.Upsample(scale_factor=2,
// mode='bilinear', align_corners=True), unet_ms.py:81; concat order [skip_x, x], :97).
__global__ void __launch_bounds__(256) upsample_cat_kernel(const f16* __restrict__ skip, const f16* __restrict__ xin,
                                                           f16* __restrict__ out, int B, int hi, int wi, int Cs, int Cx) {
    pdl_launch_dependents();
    pdl_wait();
    const int Ho = 2 * hi, Wo = 2 * wi, Ct = Cs + Cx, c8n = Ct / 8;
    const size_t total8 = (size_t)B * Ho * Wo * c8n;
    const float sh = Ho > 1 ? (float)(hi - 1) / (float)(Ho - 1) : 0.f;
    const float sw = Wo > 1 ? (float)(wi - 1) / (float)(Wo - 1) : 0.f;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total8; i += (size_t)gridDim.x * blockDim.x) {
        const int c8 = (int)(i % c8n);
        size_t pix = i / c8n;
        const int ox = (int)(pix % Wo);
        const int oy = (int)((pix / Wo) % Ho);
        const int b = (int)(pix / ((size_t)Wo * Ho));
        const int c = c8 * 8;
        uint4 o;
        if (c < Cs) {
            o = *reinterpret_cast<const uint4*>(skip + pix * Cs + c);
        } else {
            const float ry = sh * oy, rx = sw * ox;
            const int y0 = (int)ry, x0 = (int)rx;
            const int y1 = min(y0 + 1, hi - 1), x1 = min(x0 + 1, wi - 1);
            const float ly = ry - y0, lx = rx - x0;
            const float hy = 1.f - ly, hx = 1.f - lx;
            const f16* base = xin + (size_t)b * hi * wi * Cx + (c - Cs);
            const uint4 v00 = *reinterpret_cast<const uint4*>(base + ((size_t)y0 * wi + x0) * Cx);
            const uint4 v01 = *reinterpret_cast<const uint4*>(base + ((size_t)y0 * wi + x1) * Cx);
            const uint4 v10 = *reinterpret_cast<const uint4*>(base + ((size_t)y1 * wi + x0) * Cx);
            const uint4 v11 = *reinterpret_cast<const uint4*>(base + ((size_t)y1 * wi + x1) * Cx);
            const uint32_t* a00 = reinterpret_cast<const uint32_t*>(&v00);
            const uint32_t* a01 = reinterpret_cast<const uint32_t*>(&v01);
            const uint32_t* a10 = reinterpret_cast<const uint32_t*>(&v10);
            const uint32_t* a11 = reinterpret_cast<const uint32_t*>(&v11);
            uint32_t* po = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float2 p00 = unpack_h2(a00[j]), p01 = unpack_h2(a01[j]), p10 = unpack_h2(a10[j]), p11 = unpack_h2(a11[j]);
                const float r0 = hy * (hx * p00.x + lx * p01.x) + ly * (hx * p10.x + lx * p11.x);
                const float r1 = hy * (hx * p00.y + lx * p01.y) + ly * (hx * p10.y + lx * p11.y);
                po[j] = pack_h2(r0, r1);
            }
        }
        *reinterpret_cast<uint4*>(out + i * 8) = o;
    }
}

// ------------------------------------------------------------------------------------------------ outc: 1x1 conv 64 -> c_out
// 8 lanes per pixel (16 B each), 3 shuffles; fp32 NCHW output (eps_hat).  unet_ms.py:136.
__global__ void __launch_bounds__(256) outc_kernel(const f16* __restrict__ x, const float* __restrict__ w,
                                                   const float* __restrict__ bias, float* __restrict__ out, int B, int HW,
                                                   int c_out) {
    pdl_launch_dependents();
    pdl_wait();
    const size_t gid = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    const size_t pix = gid >> 3;
    const int cg = (int)(gid & 7);
    const bool ok = pix < (size_t)B * HW;
    float v[8];
    {
        uint4 raw = make_uint4(0, 0, 0, 0);
        if (ok) raw = *reinterpret_cast<const uint4*>(x + pix * 64 + cg * 8);
        float2 t;
        t = unpack_h2(raw.x); v[0] = t.x; v[1] = t.y;
        t = unpack_h2(raw.y); v[2] = t.x; v[3] = t.y;
        t = unpack_h2(raw.z); v[4] = t.x; v[5] = t.y;
        t = unpack_h2(raw.w); v[6] = t.x; v[7] = t.y;
    }
    for (int oc = 0; oc < c_out; ++oc) {
        float a = 0.f;
#pragma unroll
        for (int c = 0; c < 8; ++c) a = fmaf(v[c], __ldg(w + oc * 64 + cg * 8 + c), a);
        a += __shfl_xor_sync(0xffffffffu, a, 1);
        a += __shfl_xor_sync(0xffffffffu, a, 2);
        a += __shfl_xor_sync(0xffffffffu, a, 4);
        if (ok && cg == 0) {
            const size_t b = pix / HW, p = pix % HW;
            out[(b * c_out + oc) * HW + p] = a + bias[oc];
        }
    }
}

// ------------------------------------------------------------------------------------------------ packing
static const int D_TEMB_OFF[6] = {0, 128, 384, 640, 768, 832};   // down1(128) down2(256) down3(256) up1(128) up2(64) up3(64)
static const int D_TEMB_TOTAL = 896;

static int pack_double_conv(Handle* h, const std::string& role, const std::string& prefix) {
    B2D_TRY(pack_conv(h, role + ".c1", prefix + ".double_conv.0.weight", "", ""));
    B2D_TRY(pack_conv(h, role + ".c2", prefix + ".double_conv.3.weight", "", ""));
    NEED(g1, prefix + ".double_conv.1.weight");
    NEED(b1, prefix + ".double_conv.1.bias");
    NEED(g2, prefix + ".double_conv.4.weight");
    NEED(b2, prefix + ".double_conv.4.bias");
    B2D_TRY(upload_f32(h, role + ".gn1.g", g1->v));
    B2D_TRY(upload_f32(h, role + ".gn1.b", b1->v));
    B2D_TRY(upload_f32(h, role + ".gn2.g", g2->v));
    B2D_TRY(upload_f32(h, role + ".gn2.b", b2->v));
    return 0;
}

static int pack_family_d(Handle* h) {
    const int cin_total = h->cfg.c_hr + h->cfg.cond_channels;
    {   // inc first conv: fp32 [64][cin_total][3][3] -> [cin_total][9][64] for the direct stem kernel
        NEED(w, "inc.double_conv.0.weight");
        if (w->shape[0] != 64 || w->shape[1] != cin_total || w->shape[2] != 3)
            return fail(-3, "inc.double_conv.0.weight does not match c_hr + low-res channels");
        std::vector<float> wt((size_t)cin_total * 9 * 64);
        for (int co = 0; co < 64; ++co)
            for (int ci = 0; ci < cin_total; ++ci)
                for (int tap = 0; tap < 9; ++tap) wt[((size_t)ci * 9 + tap) * 64 + co] = w->v[((size_t)co * cin_total + ci) * 9 + tap];
        B2D_TRY(upload_f32(h, "inc.stem.w", wt));
        B2D_TRY(pack_conv(h, "inc.c2", "inc.double_conv.3.weight", "", ""));
        NEED(g1, "inc.double_conv.1.weight");
        NEED(b1, "inc.double_conv.1.bias");
        NEED(g2, "inc.double_conv.4.weight");
        NEED(b2, "inc.double_conv.4.bias");
        B2D_TRY(upload_f32(h, "inc.gn1.g", g1->v));
        B2D_TRY(upload_f32(h, "inc.gn1.b", b1->v));
        B2D_TRY(upload_f32(h, "inc.gn2.g", g2->v));
        B2D_TRY(upload_f32(h, "inc.gn2.b", b2->v));
    }
    const char* downs[3] = {"down1", "down2", "down3"};
    const char* ups[3] = {"up1", "up2", "up3"};
    std::vector<float> W((size_t)D_TEMB_TOTAL * 256), Bv(D_TEMB_TOTAL);
    for (int i = 0; i < 3; ++i) {
        const std::string d = downs[i], u = ups[i];
        B2D_TRY(pack_double_conv(h, d + ".dc1", d + ".maxpool_conv.1"));
        B2D_TRY(pack_double_conv(h, d + ".dc2", d + ".maxpool_conv.2"));
        B2D_TRY(pack_double_conv(h, u + ".dc1", u + ".conv.0"));
        B2D_TRY(pack_double_conv(h, u + ".dc2", u + ".conv.1"));
        NEED(dw, d + ".emb_layer.1.weight");
        NEED(db, d + ".emb_layer.1.bias");
        NEED(uw, u + ".emb_layer.1.weight");
        NEED(ub, u + ".emb_layer.1.bias");
        memcpy(&W[(size_t)D_TEMB_OFF[i] * 256], dw->v.data(), dw->v.size() * 4);
        memcpy(&Bv[D_TEMB_OFF[i]], db->v.data(), db->v.size() * 4);
        memcpy(&W[(size_t)D_TEMB_OFF[3 + i] * 256], uw->v.data(), uw->v.size() * 4);
        memcpy(&Bv[D_TEMB_OFF[3 + i]], ub->v.data(), ub->v.size() * 4);
    }
    B2D_TRY(upload_f32(h, "temb.w", W));
    B2D_TRY(upload_f32(h, "temb.b", Bv));
    B2D_TRY(pack_double_conv(h, "bot1", "bot1"));
    B2D_TRY(pack_double_conv(h, "bot3", "bot3"));
    for (int i = 1; i <= 6; ++i)
        B2D_TRY(pack_attention(h, "sa" + std::to_string(i), "sa" + std::to_string(i), "ln", "mha"));
    {
        NEED(w, "outc.weight");
        NEED(b, "outc.bias");
        if (w->shape[0] != h->cfg.c_out || w->shape[1] != 64) return fail(-3, "outc.weight shape mismatch");
        B2D_TRY(upload_f32(h, "outc.w", w->v));
        B2D_TRY(upload_f32(h, "outc.b", b->v));
    }
    // UNet_downscale.pos_encoding (:138-146): inv_freq = 1 / 10000^(2j/256), layout [sin | cos]
    std::vector<float> inv(128), dummy(128, 1.0f);
    for (int j = 0; j < 128; ++j)
        inv[j] = (float)(1.0 / (double)(float)std::pow(10000.0, (double)(float)((float)(2 * j) / 256.0f)));
    B2D_TRY(upload_f32(h, "enc_inv", inv));
    B2D_TRY(upload_f32(h, "dec_div", dummy));
    return 0;
}

// ------------------------------------------------------------------------------------------------ program
struct BuilderD : Builder {
    using Builder::Builder;

    void gn_stats(const f16* x, size_t per_sample, float* st) {
        const size_t slab = 32768;   // elements per CTA
        const int nslab = (int)((per_sample + slab - 1) / slab), Bc = B;
        float* partial = nullptr;
        unsigned int* counters = nullptr;
        if (h->alloc(&partial, (size_t)B * nslab * 2) != 0 || h->alloc(&counters, (size_t)B) != 0) { err = -2; return; }
        if (cudaMemset(counters, 0, (size_t)B * sizeof(unsigned int)) != cudaSuccess) err = -2;
        ops.meta("gn_stats", "sample_stats", 0, 2.0 * B * per_sample);
        ops.push_back([=](cudaStream_t s) {
            B2D_CUDA(launch_k(sample_stats_kernel, dim3(nslab, Bc), dim3(256), 0, s, x, partial, counters, st, per_sample, slab));
            return 0;
        });
    }
    void gn_apply(const f16* x, const float* st, const std::string& gnrole, const f16* res, int act, const float* vec,
                  int vec_stride, f16* y, size_t per_sample, int C, const float* partial = nullptr, int tps = 0,
                  int ntiles = 0, int mtiles = 0) {
        const float* g = W<float>(gnrole + ".g");
        const float* b = W<float>(gnrole + ".b");
        const size_t n8 = per_sample / 8;
        const int Bc = B;
        if (2048 % C != 0) { err = -1; fail(-1, "groupnorm_apply: 2048 must be a multiple of the channel count"); return; }
        ops.meta("gn_apply", "groupnorm_apply", 0, 2.0 * B * per_sample * (res ? 3 : 2));
        ops.push_back([=](cudaStream_t s) {
            const int chunks = (int)((n8 + GNA_ITER * 256 - 1) / (GNA_ITER * 256));
            B2D_CUDA(launch_k(groupnorm_apply_kernel, dim3(chunks, Bc), dim3(256), 0, s, x, st, partial, tps, ntiles, mtiles, g, b,
                              res, act, vec, vec_stride, y, per_sample, C));
            return 0;
        });
    }
    // GroupNorm(1,C) statistics + affine (+residual, GELU, +emb) in ONE launch when a sample fits a cluster's shared memory
    bool gn_fused(const f16* x, const std::string& gnrole, const f16* res, int act, const float* vec, int vec_stride, f16* y,
                  size_t per_sample, int C) {
        // measured on B200 (cfg4): the clustered one-pass kernel loses to the two-pass pair (4.28 vs 3.97 ms per step —
        // 8-CTA clusters schedule poorly next to the other kernels of the graph), so it is opt-in for Family D
        static const bool off = getenv("B2D_FUSED_GN") == nullptr;
        const int rows = (int)(per_sample / 64);
        if (off || norm_fused_cluster(rows) == 0) return false;
        NormParams np{};
        np.x = x; np.y = y; np.add = res; np.vec = vec; np.vec_stride = vec_stride; np.act = act; np.C = C; np.rows = rows;
        np.gamma = W<float>(gnrole + ".g");
        np.beta = W<float>(gnrole + ".b");
        np.slab_stride = (long long)per_sample;
        const int Bc = B;
        ops.meta("gn_fused", "norm_fused", 0, 2.0 * B * per_sample * (res ? 3 : 2));
        ops.push_back([=](cudaStream_t s) { return norm_fused_launch<1>(np, Bc, 1, s); });
        return true;
    }
    void gn(const f16* x, const std::string& gnrole, const f16* res, int act, const float* vec, int vec_stride, f16* y,
            size_t per_sample, int C) {
        if (last_gn_partial != nullptr) {   // the convolution that produced x already reduced it per tile
            const float* part = last_gn_partial;
            last_gn_partial = nullptr;
            gn_apply(x, nullptr, gnrole, res, act, vec, vec_stride, y, per_sample, C, part, last_gn_tps, last_gn_ntiles,
                     last_gn_mtiles);
            return;
        }
        if (gn_fused(x, gnrole, res, act, vec, vec_stride, y, per_sample, C)) return;
        float* st = stat2();
        gn_stats(x, per_sample, st);
        gn_apply(x, st, gnrole, res, act, vec, vec_stride, y, per_sample, C);
    }
    float* stat2() {
        float* p = h->d_stats + h->stats_floats;
        h->stats_floats += (size_t)B * 2;
        return p;
    }
    // DoubleConv on `in` [B,hw,hw,Cin] -> [B,hw,hw,Cout]; residual => gelu(in + .); vec = time projection added at the end
    f16* double_conv(const f16* in, int hw, int Cin, int Cmid, int Cout, const std::string& role, bool residual,
                     const float* vec, int vec_stride) {
        const size_t px = (size_t)hw * hw;
        f16* a = act(B * px * Cmid);
        want_gn_partial = true;
        conv(in, hw, hw, Cin, a, Cmid, 3, 1, 1, false, role + ".c1", nullptr, nullptr, 0, 0);
        gn(a, role + ".gn1", nullptr, 2, nullptr, 0, a, px * Cmid, Cmid);
        f16* c = act(B * px * Cout);
        want_gn_partial = true;
        conv(a, hw, hw, Cmid, c, Cout, 3, 1, 1, false, role + ".c2", nullptr, nullptr, 0, 0);
        gn(c, role + ".gn2", residual ? in : nullptr, residual ? 2 : 0, vec, vec_stride, c, px * Cout, Cout);
        return c;
    }
};

static int build_program_d(Handle* h, int B) {
    const b2d_config& c = h->cfg;
    const int H = c.img_size;
    OpList ops;
    BuilderD bd(h, B, ops);
    h->stats_floats = 0;
    const size_t max_rc = (size_t)B * H * H * 64;   // sa6: L = H^2 tokens x 64 channels is the largest attention input
    bd.s_xn = bd.act(max_rc);
    bd.s_qkv = bd.act(max_rc * 3);
    bd.s_ao = bd.act(max_rc);
    bd.s_h1 = bd.act(max_rc);
    bd.s_mid = bd.act(max_rc);
    float* temb = h->d_temb;
    const int TS = D_TEMB_TOTAL;
    Handle* hh = h;
    {
        const float* ei = bd.W<float>("enc_inv");
        const float* dd = bd.W<float>("dec_div");
        const float* tw = bd.W<float>("temb.w");
        const float* tb = bd.W<float>("temb.b");
        ops.meta("temb", "temb_project", 2.0 * B * TS * 256, 4.0 * TS * 256);
        ops.push_back([=](cudaStream_t st) {
            dim3 grid((TS + TEMB_OC - 1) / TEMB_OC, (B + TEMB_SB - 1) / TEMB_SB);
            B2D_CUDA(launch_k(temb_project_kernel, grid, dim3(256), 0, st, hh->temb_t, nullptr, nullptr, ei, dd, tw, tb, temb, TS, TS, B, hh->temb_t_off, 0));
            return 0;
        });
    }
    // ---- inc = DoubleConv(c_in, 64): first conv direct on the fp32 state (+ precomputed low-res part), unet_ms.py:160
    const size_t px0 = (size_t)H * H;
    f16* a0 = bd.act(B * px0 * 64);
    {
        const float* sw = bd.W<float>("inc.stem.w");
        const int chr = c.c_hr, Hh = H, cin_total = c.c_hr + c.cond_channels;
        ops.meta("inc.c1", "stem_conv", 2.0 * B * px0 * 64 * 9 * chr, (double)B * px0 * (4.0 * chr + 64 * (2 + 4)));
        ops.push_back([=](cudaStream_t st) {
            dim3 grid(Hh / 16, Hh / 16, B);
            B2D_CUDA(launch_k(stem_conv_kernel<3, 1>, grid, dim3(256), 0, st, hh->cur_x, chr, Hh, Hh, sw, cin_total, 0,
                              hh->d_cond_pre, nullptr, 0, a0, nullptr, Hh, Hh, 1));
            return 0;
        });
    }
    bd.gn(a0, "inc.gn1", nullptr, 2, nullptr, 0, a0, px0 * 64, 64);
    f16* x1 = bd.act(B * px0 * 64);
    bd.want_gn_partial = true;
    bd.conv(a0, H, H, 64, x1, 64, 3, 1, 1, false, "inc.c2", nullptr, nullptr, 0, 0);
    bd.gn(x1, "inc.gn2", nullptr, 0, nullptr, 0, x1, px0 * 64, 64);
    h->taps["x1"] = {x1, 64, H};

    auto down = [&](const f16* in, int hw_in, int Cin, int Cout, const std::string& role, int temb_off) -> f16* {
        const int hw = hw_in / 2;
        f16* p = bd.act((size_t)B * hw * hw * Cin);
        const int Bc = B;
        ops.meta(role + ".pool", "maxpool", 0, 2.0 * B * hw * hw * Cin * 5);
        ops.push_back([=](cudaStream_t st) {
            const size_t total8 = (size_t)Bc * hw * hw * Cin / 8;
            const int blocks = (int)std::min<size_t>((total8 + 255) / 256, (size_t)148 * 16);
            B2D_CUDA(launch_k(maxpool2_kernel, dim3(blocks), dim3(256), 0, st, in, p, Bc, hw, hw, Cin));
            return 0;
        });
        f16* r = bd.double_conv(p, hw, Cin, Cin, Cin, role + ".dc1", true, nullptr, 0);
        return bd.double_conv(r, hw, Cin, Cout, Cout, role + ".dc2", false, temb + temb_off, TS);
    };
    auto up = [&](const f16* xin, int hw_in, int Cx, const f16* skip, int Cs, int Cout, const std::string& role,
                  int temb_off) -> f16* {
        const int hw = hw_in * 2, Ct = Cs + Cx;
        f16* u = bd.act((size_t)B * hw * hw * Ct);
        const int Bc = B;
        ops.meta(role + ".upcat", "upsample_cat", 0, 2.0 * B * hw * hw * Ct * 2);
        ops.push_back([=](cudaStream_t st) {
            const size_t total8 = (size_t)Bc * hw * hw * Ct / 8;
            const int blocks = (int)std::min<size_t>((total8 + 255) / 256, (size_t)148 * 16);
            B2D_CUDA(launch_k(upsample_cat_kernel, dim3(blocks), dim3(256), 0, st, skip, xin, u, Bc, hw_in, hw_in, Cs, Cx));
            return 0;
        });
        f16* r = bd.double_conv(u, hw, Ct, Ct, Ct, role + ".dc1", true, nullptr, 0);
        return bd.double_conv(r, hw, Ct, Ct / 2, Cout, role + ".dc2", false, temb + temb_off, TS);
    };
    auto sa = [&](const f16* in, int hw, int C, const std::string& role) -> f16* {
        f16* o = bd.act((size_t)B * hw * hw * C);
        bd.attention(in, hw, C, role, o, 0);
        return o;
    };
    f16* x2_pre = down(x1, H, 64, 128, "down1", D_TEMB_OFF[0]);
    f16* x2 = sa(x2_pre, H / 2, 128, "sa1");
    f16* x3_pre = down(x2, H / 2, 128, 256, "down2", D_TEMB_OFF[1]);
    f16* x3 = sa(x3_pre, H / 4, 256, "sa2");
    f16* x4_pre = down(x3, H / 4, 256, 256, "down3", D_TEMB_OFF[2]);
    f16* x4 = sa(x4_pre, H / 8, 256, "sa3");
    h->taps["x2_pre"] = {x2_pre, 128, H / 2};
    h->taps["x3_pre"] = {x3_pre, 256, H / 4};
    h->taps["x4_pre"] = {x4_pre, 256, H / 8};
    h->taps["x2"] = {x2, 128, H / 2};
    h->taps["x3"] = {x3, 256, H / 4};
    h->taps["x4"] = {x4, 256, H / 8};
    x4 = bd.double_conv(x4, H / 8, 256, 256, 256, "bot1", false, nullptr, 0);
    x4 = bd.double_conv(x4, H / 8, 256, 256, 256, "bot3", false, nullptr, 0);
    h->taps["bot"] = {x4, 256, H / 8};
    f16* u1_pre = up(x4, H / 8, 256, x3, 256, 128, "up1", D_TEMB_OFF[3]);
    f16* u1 = sa(u1_pre, H / 4, 128, "sa4");
    f16* u2_pre = up(u1, H / 4, 128, x2, 128, 64, "up2", D_TEMB_OFF[4]);
    f16* u2 = sa(u2_pre, H / 2, 64, "sa5");
    f16* u3_pre = up(u2, H / 2, 64, x1, 64, 64, "up3", D_TEMB_OFF[5]);
    h->temb_free_op = (int)ops.v.size();   // nothing below reads d_temb
    f16* u3 = sa(u3_pre, H, 64, "sa6");
    h->taps["u1_pre"] = {u1_pre, 128, H / 4};
    h->taps["u2_pre"] = {u2_pre, 64, H / 2};
    h->taps["u3_pre"] = {u3_pre, 64, H};
    h->taps["u1"] = {u1, 128, H / 4};
    h->taps["u2"] = {u2, 64, H / 2};
    h->taps["u3"] = {u3, 64, H};
    {
        const float* ow = bd.W<float>("outc.w");
        const float* ob = bd.W<float>("outc.b");
        const int HW = H * H, cout = c.c_out;
        ops.meta("outc", "outc", 2.0 * B * HW * 64 * cout, (double)B * HW * (128 + 4 * cout));
        ops.push_back([=](cudaStream_t st) {
            const size_t threads = (size_t)B * HW * 8;
            B2D_CUDA(launch_k(outc_kernel, dim3((unsigned)((threads + 255) / 256)), dim3(256), 0, st, u3, ow, ob, hh->cur_eps, B, HW,
                              cout));
            return 0;
        });
    }
    if (bd.err) return g_status.code ? g_status.code : fail(-1, "program build failed");
    h->step_ops.swap(ops.v);
    h->prog_B = B;
    return 0;
}

// Low-res field -> bicubic to H x H (once) -> its share of inc's first convolution (once); zeros when absent (:158).
static int set_conditioning_d(Handle* h, const float* cond, int ch, int cw, int B, cudaStream_t st) {
    const b2d_config& c = h->cfg;
    const int H = c.img_size;
    const size_t n_pre = (size_t)B * H * H * 64;
    if (cond == nullptr || c.cond_channels == 0) {
        B2D_CUDA(cudaMemsetAsync(h->d_cond_pre, 0, n_pre * sizeof(float), st));
        return 0;
    }
    B2D_CHECK(ch >= 1 && cw >= 1, "low-resolution field needs its height/width");
    const int planes = B * c.cond_channels;
    const size_t total = (size_t)planes * H * H;
    const int blocks = (int)std::min<size_t>((total + 255) / 256, (size_t)148 * 16);
    if (c.interp_mode == B2D_INTERP_BICUBIC)
        B2D_CUDA(launch_k(bicubic_resize_kernel, dim3(blocks), dim3(256), 0, st, cond, h->d_cond_stack, planes, ch, cw, H, H));
    else
        B2D_CUDA(launch_k(linear_nearest_resize_kernel, dim3(blocks), dim3(256), 0, st, cond, h->d_cond_stack, planes, ch, cw, H, H,
                          c.interp_mode == B2D_INTERP_NEAREST ? 1 : 0));
    dim3 grid(H / 16, H / 16, B);
    B2D_CUDA(launch_k(stem_conv_kernel<3, 1>, grid, dim3(256), 0, st, (const float*)h->d_cond_stack, c.cond_channels, H, H,
                      (const float*)h->dev["inc.stem.w"], c.c_hr + c.cond_channels, c.c_hr, (const float*)nullptr,
                      (const float*)nullptr, 0, (f16*)nullptr, h->d_cond_pre, H, H, 1));
    return 0;
}

}  // namespace b2d
