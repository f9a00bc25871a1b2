// D7 — ZoeDepth-NK, -N and -K: everything around the DPT-BEiT core that the reference's DepthModel / ZoeDepthNK adds
// (dzoedepth/models/depth_model.py:57-152, zoedepth_nk/zoedepth_nk_v1.py:159-243, layers/attractor.py:127-208,
// layers/dist_layers.py:29-121, layers/patch_transformer.py:29-92, base_models/midas.py:175-186).
// The 1x1 convolutions of the head run on the tcgen05 GEMM (NHWC activations = row-major [pixels, channels]); the
// kernels here are the bandwidth-side pieces, fp32 math:
//   zoe_preprocess_patchify  ToTensor -> reflect pad -> (flip) -> bilinear align_corners=True to the net size -> (x-.5)/.5
//                            -> fp16 patch matrix; forward 2b is image b, forward 2b+1 its horizontal flip (TTA)
//   layernorm_post           post-norm transformer layer of the router: x = LN(x) in place (fp32) + fp16 copy
//   attention_small          router self-attention (4 heads x 32 dims, 257 tokens), SIMT
//   select_softplus          seed bin centres of the routed head: softplus(seed[:, head*64 : head*64+64])
//   seed_normed              normed seed bin centres of ZoeDepth-K: widths normalised over 64 bins, cumulative sum, midpoints
//   resize_add_nhwc          x = b_emb + bilinear(prev_b_embedding)            (attractor.py:173-177)
//   attractor                b_new = b + mean_i inv_attractor(A_i - b), b = bilinear(b_prev)   (attractor.py:178-208); templated
//                            on the attractor count and on normed (ZoeDepth-K: + scale, per-pixel sort, clip) / unnormed bins
//   clb_final                ConditionalLogBinomial + sum(p * bin centres) per output pixel of the routed head, with the
//                            1x1 conv on cat(out_conv, bilinear(b_emb)) split by linearity into W_o . out_conv (here) +
//                            bilinear(W_e . b_emb) (a GEMM at a quarter of the pixels)
//   clb_final_single         the same for the single metric head of ZoeDepth-N / -K: 33 + 128 inputs (out_conv + the core's
//                            relative depth + bin embedding), 80 hidden units, no router
//   tta_combine              bicubic (align_corners=False) back to the padded size, crop, average with the un-flipped
//                            flipped prediction
// The router decision is taken per forward on the device (argmax of the two logits): no host synchronisation
// (the reference calls .item(), zoedepth_nk_v1.py:194-195) and no cross-image vote (SURVEY §8e).
#include <cuda_fp16.h>
#include <math.h>

#include "common.cuh"

namespace dm {

__device__ __forceinline__ void cubic_coeffs_z(float x, float *c) {
    const float A = -0.75f;
    c[0] = ((A * (x + 1.f) - 5.f * A) * (x + 1.f) + 8.f * A) * (x + 1.f) - 4.f * A;
    c[1] = ((A + 2.f) * x - (A + 3.f)) * x * x + 1.f;
    c[2] = ((A + 2.f) * (1.f - x) - (A + 3.f)) * (1.f - x) * (1.f - x) + 1.f;
    c[3] = 1.f - c[0] - c[1] - c[2];
}
__device__ __forceinline__ float softplus_f(float x) { return x > 20.f ? x : log1pf(expf(x)); }   // F.softplus defaults
__device__ __forceinline__ int route_of(const float *logits, int ld, int f) { return logits[(size_t)f * ld + 1] > logits[(size_t)f * ld] ? 1 : 0; }

// ---------------------------------------------------------------------------------------------------------------
struct ZoePre {
    const uint8_t *rgb;
    int B, H, W, pad_h, pad_w, nh, nw, patch, gh, gw, kpad;
    __half *out;
};

__global__ void __launch_bounds__(256) zoe_preprocess_patchify_kernel(ZoePre p) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)2 * p.B * p.nh * p.nw;
    if (idx >= total) return;
    const int x = (int)(idx % p.nw);
    const int y = (int)((idx / p.nw) % p.nh);
    const int f = (int)(idx / ((long long)p.nw * p.nh));
    const int b = f >> 1, flip = f & 1;
    const int Hp = p.H + 2 * p.pad_h, Wp = p.W + 2 * p.pad_w;
    const uint8_t *img = p.rgb + (long long)b * p.H * p.W * 3;
    // F.interpolate(bilinear, align_corners=True) over the padded (and flipped) image
    const float sy = p.nh > 1 ? (float)(Hp - 1) / (float)(p.nh - 1) : 0.f;
    const float sx = p.nw > 1 ? (float)(Wp - 1) / (float)(p.nw - 1) : 0.f;
    const float fy = sy * (float)y, fx = sx * (float)x;
    const int y0 = min((int)fy, Hp - 1), x0 = min((int)fx, Wp - 1);
    const int y1 = min(y0 + 1, Hp - 1), x1 = min(x0 + 1, Wp - 1);
    const float ly = fy - (float)y0, lx = fx - (float)x0, hy = 1.f - ly, hx = 1.f - lx;
    auto src = [&](int yy, int xx, float *v) {
        if (flip) xx = Wp - 1 - xx;
        int sy_ = yy - p.pad_h, sx_ = xx - p.pad_w;           // F.pad(mode="reflect"): edge not repeated
        sy_ = sy_ < 0 ? -sy_ : (sy_ >= p.H ? 2 * (p.H - 1) - sy_ : sy_);
        sx_ = sx_ < 0 ? -sx_ : (sx_ >= p.W ? 2 * (p.W - 1) - sx_ : sx_);
        const uint8_t *px = img + ((long long)sy_ * p.W + sx_) * 3;
        v[0] = (float)px[0] / 255.0f; v[1] = (float)px[1] / 255.0f; v[2] = (float)px[2] / 255.0f;   // transforms.ToTensor
    };
    float v00[3], v01[3], v10[3], v11[3];
    src(y0, x0, v00); src(y0, x1, v01); src(y1, x0, v10); src(y1, x1, v11);
    const int py = y / p.patch, ky = y % p.patch, pxi = x / p.patch, kx = x % p.patch;
    __half *row = p.out + ((long long)(f * p.gh + py) * p.gw + pxi) * p.kpad;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float r = hy * (hx * v00[c] + lx * v01[c]) + ly * (hx * v10[c] + lx * v11[c]);
        row[(c * p.patch + ky) * p.patch + kx] = __float2half_rn((r - 0.5f) / 0.5f);
    }
}

// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) layernorm_post_kernel(float *__restrict__ x, long long rows, const float *__restrict__ gamma,
                                                             const float *__restrict__ beta, float eps, __half *__restrict__ out) {
    // C = 128: one warp per row, one float4 per lane
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * 8 + warp;
    if (row >= rows) return;
    float4 v = reinterpret_cast<const float4 *>(x + row * 128)[lane];
    float s = (v.x + v.y) + (v.z + v.w);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float mean = s / 128.f;
    const float a = v.x - mean, b = v.y - mean, c = v.z - mean, d = v.w - mean;
    float q = (a * a + b * b) + (c * c + d * d);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
    const float rstd = rsqrtf(q / 128.f + eps);
    const float4 g = reinterpret_cast<const float4 *>(gamma)[lane], bt = reinterpret_cast<const float4 *>(beta)[lane];
    v = make_float4(a * rstd * g.x + bt.x, b * rstd * g.y + bt.y, c * rstd * g.z + bt.z, d * rstd * g.w + bt.w);
    reinterpret_cast<float4 *>(x + row * 128)[lane] = v;
    const __half2 h0 = __floats2half2_rn(v.x, v.y), h1 = __floats2half2_rn(v.z, v.w);
    uint2 u;
    u.x = *reinterpret_cast<const uint32_t *>(&h0);
    u.y = *reinterpret_cast<const uint32_t *>(&h1);
    reinterpret_cast<uint2 *>(out + row * 128)[lane] = u;
}

// router attention: qkv fp16 [F*S, 3*E] (q | k | v, head h at columns h*32), out fp16 [F*S, E]; grid (F, heads)
constexpr int RA_HD = 32, RA_PITCH = 33;
__global__ void __launch_bounds__(256) attention_small_kernel(const __half *__restrict__ qkv, int S, int E, float scale, __half *__restrict__ out) {
    extern __shared__ float ra_smem[];
    float *sk = ra_smem, *sv = sk + (size_t)S * RA_PITCH, *sp = sv + (size_t)S * RA_PITCH;   // sp: [8 warps][S]
    const int f = blockIdx.x, h = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const __half *base = qkv + (size_t)f * S * 3 * E + h * RA_HD;
    for (int i = threadIdx.x; i < S * RA_HD; i += 256) {
        const int t = i >> 5, d = i & 31;
        sk[t * RA_PITCH + d] = __half2float(base[(size_t)t * 3 * E + E + d]);
        sv[t * RA_PITCH + d] = __half2float(base[(size_t)t * 3 * E + 2 * E + d]);
    }
    __syncthreads();
    float *pw = sp + (size_t)warp * S;
    const int rows_per = (S + gridDim.z - 1) / gridDim.z, t_beg = blockIdx.z * rows_per, t_end = min(S, t_beg + rows_per);
    for (int t = t_beg + warp; t < t_end; t += 8) {
        const float qd = __half2float(base[(size_t)t * 3 * E + lane]) * scale;
        float mx = -INFINITY;
        for (int j0 = 0; j0 < S; j0 += 32) {                 // uniform trip count: the shuffles need every lane
            const int j = j0 + lane;
            const float *kr = sk + (size_t)min(j, S - 1) * RA_PITCH;
            float s = 0.f;
#pragma unroll
            for (int d = 0; d < RA_HD; ++d) s = fmaf(__shfl_sync(0xffffffffu, qd, d), kr[d], s);
            if (j < S) { pw[j] = s; mx = fmaxf(mx, s); }
        }
        __syncwarp();
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        float sum = 0.f;
        for (int j = lane; j < S; j += 32) { const float e = __expf(pw[j] - mx); pw[j] = e; sum += e; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        __syncwarp();
        float acc = 0.f;                                    // lane = output dim
        for (int j = 0; j < S; ++j) acc = fmaf(pw[j], sv[j * RA_PITCH + lane], acc);
        out[((size_t)f * S + t) * E + h * RA_HD + lane] = __float2half_rn(acc / sum);
        __syncwarp();
    }
}

__global__ void __launch_bounds__(256) cast_f32_f16_kernel(const float *__restrict__ x, long long n4, __half *__restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n4) return;
    const float4 v = reinterpret_cast<const float4 *>(x)[i];
    const __half2 h0 = __floats2half2_rn(v.x, v.y), h1 = __floats2half2_rn(v.z, v.w);
    uint2 u;
    u.x = *reinterpret_cast<const uint32_t *>(&h0);
    u.y = *reinterpret_cast<const uint32_t *>(&h1);
    reinterpret_cast<uint2 *>(out)[i] = u;
}

__global__ void __launch_bounds__(256) select_softplus_kernel(const float *__restrict__ seed, int ld, const float *__restrict__ logits, int lld,
                                                              long long rows, int rows_per_fwd, float *__restrict__ out) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * 64) return;
    const long long r = idx >> 6;
    const int k = (int)(idx & 63);
    const int head = route_of(logits, lld, (int)(r / rows_per_fwd));
    out[idx] = softplus_f(seed[r * ld + head * 64 + k]);
}

// out = a + bilinear_align_corners(b), NHWC fp16, 8 channels per thread; grid (ceil(W*C/8/256), H, B)
__global__ void __launch_bounds__(256) resize_add_nhwc_kernel(const __half *__restrict__ a, const __half *__restrict__ bsm, int Hs, int Ws, int C,
                                                              __half *__restrict__ out, int H, int W, float sy, float sx) {
    const int c8 = C >> 3;
    const int t = blockIdx.x * 256 + threadIdx.x;
    if (t >= W * c8) return;
    const int x = t / c8;
    const int c = (t - x * c8) << 3;
    const int y = blockIdx.y, b = blockIdx.z;
    const float fy = sy * (float)y, fx = sx * (float)x;
    const int y0 = min((int)fy, Hs - 1), x0 = min((int)fx, Ws - 1);
    const int y1 = min(y0 + 1, Hs - 1), x1 = min(x0 + 1, Ws - 1);
    const float ly = fy - (float)y0, lx = fx - (float)x0, hy = 1.f - ly, hx = 1.f - lx;
    const __half *base = bsm + (size_t)b * Hs * Ws * C + c;
    const uint4 u00 = __ldg(reinterpret_cast<const uint4 *>(base + (size_t)(y0 * Ws + x0) * C));
    const uint4 u01 = __ldg(reinterpret_cast<const uint4 *>(base + (size_t)(y0 * Ws + x1) * C));
    const uint4 u10 = __ldg(reinterpret_cast<const uint4 *>(base + (size_t)(y1 * Ws + x0) * C));
    const uint4 u11 = __ldg(reinterpret_cast<const uint4 *>(base + (size_t)(y1 * Ws + x1) * C));
    const size_t o_off = ((size_t)(b * H + y) * W + x) * C + c;
    const uint4 ua = __ldg(reinterpret_cast<const uint4 *>(a + o_off));
    const __half2 *p00 = reinterpret_cast<const __half2 *>(&u00), *p01 = reinterpret_cast<const __half2 *>(&u01);
    const __half2 *p10 = reinterpret_cast<const __half2 *>(&u10), *p11 = reinterpret_cast<const __half2 *>(&u11);
    const __half2 *pa = reinterpret_cast<const __half2 *>(&ua);
    uint4 o;
    __half2 *oh = reinterpret_cast<__half2 *>(&o);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float2 f00 = __half22float2(p00[k]), f01 = __half22float2(p01[k]), f10 = __half22float2(p10[k]), f11 = __half22float2(p11[k]);
        const float2 fa = __half22float2(pa[k]);
        oh[k] = __floats2half2_rn(fa.x + (hy * (hx * f00.x + lx * f01.x) + ly * (hx * f10.x + lx * f11.x)),
                                  fa.y + (hy * (hx * f00.y + lx * f01.y) + ly * (hx * f10.y + lx * f11.y)));
    }
    *reinterpret_cast<uint4 *>(out + o_off) = o;
}

// b_new[f, y, x, k] = b + (1/NA) * sum_i dx_i / (1 + 300 dx_i^2), dx_i = a_i - b, b = bilinear_align_corners(b_prev)[k], where the
// NA attractor points a_i of the pixel are
//   ROUTED (ZoeDepth-NK, NA = 16):  softplus(A[f, y, x, head*32 + i]), head picked per forward by the router logits
//   unnormed (ZoeDepth-N):          softplus(A[f, y, x, i])                      (AttractorLayerUnnormed, attractor.py:139-208)
//   NORMED (ZoeDepth-K):            relu(A[f, y, x, 2i]) + 1e-3                   (AttractorLayer, attractor.py:60-136: the
//                                   normalisation of A is overwritten by the next line, so channel 0 of each pair is used as is)
// NORMED with Bsort: also B = clip(sort_ascending((max - min) * b_new + min), min, max) over the 64 bins of the pixel.
// One thread per (pixel, bin); the attractors of a pixel are broadcast by shuffle.
template <int NA, bool NORMED, bool ROUTED>
__global__ void __launch_bounds__(256) attractor_kernel(const float *__restrict__ A, int lda, const float *__restrict__ logits, int lld,
                                                        const float *__restrict__ bprev, int Hp, int Wp, int H, int W, float sy, float sx,
                                                        float *__restrict__ bout, float min_d, float max_d, float range, float *__restrict__ Bsort) {
    static_assert(NA == 1 || NA == 2 || NA == 4 || NA == 8 || NA == 16, "attractor counts are powers of two up to 16");
    static_assert(!(ROUTED && NORMED), "the routed head has unnormed bin centres");
    const int y = blockIdx.y, f = blockIdx.z;
    const int t = blockIdx.x * 256 + threadIdx.x;       // (x, bin): 64 bins per pixel -> half a warp per pixel
    const int x = t >> 6, k = t & 63;
    const int lane = threadIdx.x & 31;
    const bool ok = x < W;
    const int xc = ok ? x : W - 1;
    const int head = ROUTED ? route_of(logits, lld, f) : 0;
    const float fy = sy * (float)y, fx = sx * (float)xc;
    const int y0 = min((int)fy, Hp - 1), x0 = min((int)fx, Wp - 1);
    const int y1 = min(y0 + 1, Hp - 1), x1 = min(x0 + 1, Wp - 1);
    const float ly = fy - (float)y0, lx = fx - (float)x0, hy = 1.f - ly, hx = 1.f - lx;
    const float *bp = bprev + (size_t)f * Hp * Wp * 64 + k;
    const float b = hy * (hx * bp[(size_t)(y0 * Wp + x0) * 64] + lx * bp[(size_t)(y0 * Wp + x1) * 64]) +
                    ly * (hx * bp[(size_t)(y1 * Wp + x0) * 64] + lx * bp[(size_t)(y1 * Wp + x1) * 64]);
    // lanes 0..NA-1 of the warp fetch the attractor points of this warp's pixel (a warp covers 32 bins of ONE pixel)
    const float *arow = A + ((size_t)(f * H + y) * W + xc) * lda + head * 32;
    const float a_mine = NORMED ? fmaxf(arow[2 * (lane & (NA - 1))], 0.f) + 1e-3f : softplus_f(arow[lane & (NA - 1)]);
    float delta = 0.f;
#pragma unroll
    for (int i = 0; i < NA; ++i) {
        const float dx = __shfl_sync(0xffffffffu, a_mine, i) - b;
        delta += __fdividef(dx, 1.f + 300.f * (dx * dx));      // 2 ulp; the head's bar is a tolerance, and this is NA divisions per thread
    }
    const float bn = b + delta / (float)NA;
    const size_t pix = (size_t)(f * H + y) * W + x;
    if (ok) bout[pix * 64 + k] = bn;
    if (NORMED && Bsort != nullptr) {                   // uniform over the grid: every thread reaches the barrier
        // rank sort of the pixel's 64 scaled centres in shared memory (4 pixels per block); equal values get consecutive ranks
        // in bin order, and clipping after sorting equals sorting after clipping (clip is monotone)
        __shared__ float s_B[256];
        const float v = range * bn + min_d;
        s_B[threadIdx.x] = v;
        __syncthreads();
        const float *row = s_B + (threadIdx.x & ~63);
        int rank = 0;
#pragma unroll 16
        for (int j = 0; j < 64; ++j) {
            const float u = row[j];
            rank += (u < v || (u == v && j < k)) ? 1 : 0;
        }
        if (ok) Bsort[pix * 64 + rank] = fminf(fmaxf(v, min_d), max_d);
    }
}

// SeedBinRegressor (normed bin centres, localbins_layers.py:29-68) and ZoeDepth.forward's normalisation of its output
// (zoedepth_v1.py:148-150), per pixel r: w_k = relu(seed[r, k]) + 1e-3, w_k = range * w_k / sum_j w_j, edges e_0 = min,
// e_{k+1} = e_k + w_k, out[r, k] = ((e_k + e_{k+1}) / 2 - min) / range.  One thread per pixel: the cumulative sum runs in bin
// order, as torch.cumsum does.
__global__ void __launch_bounds__(256) seed_normed_kernel(const float *__restrict__ seed, int ld, long long rows, float min_d, float range,
                                                          float *__restrict__ out) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    const float4 *s4 = reinterpret_cast<const float4 *>(seed + r * ld);
    float w[64];
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        const float4 v = __ldg(s4 + q);
        w[4 * q + 0] = fmaxf(v.x, 0.f) + 1e-3f; w[4 * q + 1] = fmaxf(v.y, 0.f) + 1e-3f;
        w[4 * q + 2] = fmaxf(v.z, 0.f) + 1e-3f; w[4 * q + 3] = fmaxf(v.w, 0.f) + 1e-3f;
    }
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < 64; ++j) sum += w[j];
    float e = min_d;
    float4 *o4 = reinterpret_cast<float4 *>(out + r * 64);
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        float c[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float e1 = e + range * (w[4 * q + j] / sum);
            c[j] = (0.5f * (e + e1) - min_d) / range;
            e = e1;
        }
        o4[q] = make_float4(c[0], c[1], c[2], c[3]);
    }
}

// ---------------------------------------------------------------------------------------------------------------
struct ClbParams {
    const __half *o32; int ldo;          // [F, nh, nw, ldo] relu'd out_conv activation, channels 0..31
    const float *ze; int ldz;            // [F, h3, w3, ldz]: W_e . b_emb, nyu at columns 0..39, kitti at 64..103
    const float *bc;                     // [F, h3, w3, 64] bin centres of the routed head
    const float *logits; int lld;
    const float *wo;                     // [2][32][40]  (input channel major)
    const float *b0;                     // [2][40]
    const float *w2;                     // [2][4][40]
    const float *b2;                     // [2][4]
    int F, nh, nw, h3, w3;
    float sy, sx, min_temp, max_temp;
    float *out;                          // [F, nh, nw]
};

__device__ __forceinline__ float log_binom_f(float n, float k) {   // dist_layers.py:29-33 (eps = 1e-7 added to n and k)
    n += 1e-7f; k += 1e-7f;
    return n * logf(n) - k * logf(k) - (n - k) * logf(n - k + 1e-7f);
}

// LogBinomial (dist_layers.py:36-121) on the MLP output pt (pre-softplus) and the expectation of the bilinearly up-sampled bin
// centres bc at the neighbours i00..i11 with weights (hy, hx, ly, lx): softmax over the 64 bins of y_k / temp.
__device__ __forceinline__ float log_binomial_expectation(const float *pt, const float *s_lb, float min_temp, float max_temp, const float *bc,
                                                          size_t i00, size_t i01, size_t i10, size_t i11, float hy, float hx, float ly, float lx) {
    const float pa = softplus_f(pt[0]) + 1e-4f, pb = softplus_f(pt[1]) + 1e-4f, ta = softplus_f(pt[2]) + 1e-4f, tb = softplus_f(pt[3]) + 1e-4f;
    const float prob = pa / (pa + pb);
    const float temp = (max_temp - min_temp) * (ta / (ta + tb)) + min_temp;
    const float lp = logf(fminf(fmaxf(prob, 1e-4f), 1.f)), lq = logf(fminf(fmaxf(1.f - prob, 1e-4f), 1.f));
    // softmax over the 64 bins of y_k / temp and the expectation of the (bilinearly up-sampled) bin centres; y_k is concave in k,
    // its maximum is found in a first pass without touching memory
    const float inv_t = 1.f / temp;
    float mx = -INFINITY;
#pragma unroll 8
    for (int k = 0; k < 64; ++k) mx = fmaxf(mx, (s_lb[k] + (float)k * lp + (float)(63 - k) * lq) * inv_t);
    const float4 *c00 = reinterpret_cast<const float4 *>(bc + i00 * 64), *c01 = reinterpret_cast<const float4 *>(bc + i01 * 64);
    const float4 *c10 = reinterpret_cast<const float4 *>(bc + i10 * 64), *c11 = reinterpret_cast<const float4 *>(bc + i11 * 64);
    float den = 0.f, num = 0.f;
#pragma unroll 4
    for (int k4 = 0; k4 < 16; ++k4) {
        const float4 a = __ldg(c00 + k4), b = __ldg(c01 + k4), c = __ldg(c10 + k4), d = __ldg(c11 + k4);
        const float bcv[4] = {hy * (hx * a.x + lx * b.x) + ly * (hx * c.x + lx * d.x), hy * (hx * a.y + lx * b.y) + ly * (hx * c.y + lx * d.y),
                              hy * (hx * a.z + lx * b.z) + ly * (hx * c.z + lx * d.z), hy * (hx * a.w + lx * b.w) + ly * (hx * c.w + lx * d.w)};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int k = 4 * k4 + e;
            const float ek = expf((s_lb[k] + (float)k * lp + (float)(63 - k) * lq) * inv_t - mx);
            den += ek;
            num = fmaf(ek, bcv[e], num);
        }
    }
    return num / den;
}

// One THREAD per output pixel (the first version spent a warp per pixel: ~900 warp-instructions per pixel in shuffles, reductions
// and scalar work replicated 32 times; this form needs ~110).  The weights sit in shared memory and are read as broadcasts; a
// thread's loads are whole contiguous vectors (64 B of out_conv, 160 B per neighbour of ze, 256 B per neighbour of the bin centres)
// and neighbouring threads share their bilinear neighbours in L1.
__global__ void __launch_bounds__(128) clb_final_kernel(ClbParams p) {
    __shared__ float s_wo[32 * 40], s_b0[40], s_w2[4 * 40], s_b2[4], s_lb[64];
    const int f = blockIdx.z;
    const int head = route_of(p.logits, p.lld, f);
    for (int i = threadIdx.x; i < 32 * 40; i += 128) s_wo[i] = p.wo[head * 32 * 40 + i];
    for (int i = threadIdx.x; i < 4 * 40; i += 128) s_w2[i] = p.w2[head * 4 * 40 + i];
    if (threadIdx.x < 40) s_b0[threadIdx.x] = p.b0[head * 40 + threadIdx.x];
    if (threadIdx.x < 4) s_b2[threadIdx.x] = p.b2[head * 4 + threadIdx.x];
    if (threadIdx.x < 64) s_lb[threadIdx.x] = log_binom_f(63.f, (float)threadIdx.x);
    __syncthreads();
    const int y = blockIdx.y, x = blockIdx.x * 128 + threadIdx.x;
    if (x >= p.nw) return;
    const float fy = p.sy * (float)y, fx = p.sx * (float)x;
    const int y0 = min((int)fy, p.h3 - 1), y1 = min(y0 + 1, p.h3 - 1), x0 = min((int)fx, p.w3 - 1), x1 = min(x0 + 1, p.w3 - 1);
    const float ly = fy - (float)y0, hy = 1.f - ly, lx = fx - (float)x0, hx = 1.f - lx;
    const size_t i00 = ((size_t)f * p.h3 + y0) * p.w3 + x0, i01 = ((size_t)f * p.h3 + y0) * p.w3 + x1;
    const size_t i10 = ((size_t)f * p.h3 + y1) * p.w3 + x0, i11 = ((size_t)f * p.h3 + y1) * p.w3 + x1;
    // pre-activation of mlp.0 = b0 + W_o . out_conv + bilinear(W_e . b_emb)
    float pre[40];
    {
        const float4 *z00 = reinterpret_cast<const float4 *>(p.ze + i00 * p.ldz + head * 64), *z01 = reinterpret_cast<const float4 *>(p.ze + i01 * p.ldz + head * 64);
        const float4 *z10 = reinterpret_cast<const float4 *>(p.ze + i10 * p.ldz + head * 64), *z11 = reinterpret_cast<const float4 *>(p.ze + i11 * p.ldz + head * 64);
#pragma unroll
        for (int k = 0; k < 10; ++k) {
            const float4 a = __ldg(z00 + k), b = __ldg(z01 + k), c = __ldg(z10 + k), d = __ldg(z11 + k);
            pre[4 * k + 0] = s_b0[4 * k + 0] + (hy * (hx * a.x + lx * b.x) + ly * (hx * c.x + lx * d.x));
            pre[4 * k + 1] = s_b0[4 * k + 1] + (hy * (hx * a.y + lx * b.y) + ly * (hx * c.y + lx * d.y));
            pre[4 * k + 2] = s_b0[4 * k + 2] + (hy * (hx * a.z + lx * b.z) + ly * (hx * c.z + lx * d.z));
            pre[4 * k + 3] = s_b0[4 * k + 3] + (hy * (hx * a.w + lx * b.w) + ly * (hx * c.w + lx * d.w));
        }
    }
    {
        const uint4 *op = reinterpret_cast<const uint4 *>(p.o32 + (((size_t)f * p.nh + y) * p.nw + x) * p.ldo);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const uint4 u = __ldg(op + q);
            const __half2 *h2 = reinterpret_cast<const __half2 *>(&u);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float2 o2 = __half22float2(h2[e]);
                const float *w0 = s_wo + (q * 8 + 2 * e) * 40, *w1 = w0 + 40;
#pragma unroll
                for (int k = 0; k < 40; ++k) pre[k] = fmaf(w1[k], o2.y, fmaf(w0[k], o2.x, pre[k]));
            }
        }
    }
    float pt[4] = {s_b2[0], s_b2[1], s_b2[2], s_b2[3]};
#pragma unroll
    for (int k = 0; k < 40; ++k) {
        const float g = 0.5f * pre[k] * (1.f + erff(pre[k] * 0.70710678118654752f));                 // nn.GELU (erf form)
#pragma unroll
        for (int j = 0; j < 4; ++j) pt[j] = fmaf(s_w2[j * 40 + k], g, pt[j]);
    }
    p.out[((size_t)f * p.nh + y) * p.nw + x] = log_binomial_expectation(pt, s_lb, p.min_temp, p.max_temp, p.bc, i00, i01, i10, i11, hy, hx, ly, lx);
}

struct ClbSingleParams {
    const __half *o32; int ldo;          // [F, nh, nw, ldo] relu'd out_conv activation, channels 0..31
    const float *ze; int ldz;            // [F, h3, w3, ldz]: W_e . b_emb at columns 0..79
    const float *bc;                     // [F, h3, w3, 64] bin centres
    const float *wo;                     // [32][80] mlp.0 weights of the out_conv inputs (input channel major)
    const float *wr;                     // [80]     mlp.0 weights of the relative-depth input
    const float *b0;                     // [80]
    const float *w2;                     // [4][80]
    const float *b2;                     // [4]
    const float *w_rel; float b_rel;     // [32] + bias: the core's last 1x1 conv (MiDaS output_conv.4), out_conv -> relative depth
    int F, nh, nw, h3, w3;
    float sy, sx, min_temp, max_temp;
    float *out;                          // [F, nh, nw]
};

// The single-head form of clb_final (ZoeDepth-N / -K, zoedepth_v1.py:166-186): the log-binomial MLP sees cat(out_conv, rel_depth,
// bilinear(b_emb)), 161 inputs and (33 + 128) // 2 = 80 hidden units, where rel_depth = relu(w_rel . out_conv + b_rel) is the
// MiDaS core's own output at out_conv's size (its resize is the identity).  The 32 out_conv channels stay in registers and the
// hidden layer is evaluated in two halves of 40, so a thread holds 32 inputs + 40 pre-activations + 4 outputs at a time.
__global__ void __launch_bounds__(128) clb_final_single_kernel(ClbSingleParams p) {
    constexpr int NH = 80;
    __shared__ float s_wo[32 * NH], s_wr[NH], s_b0[NH], s_w2[4 * NH], s_b2[4], s_lb[64], s_wrel[32];
    for (int i = threadIdx.x; i < 32 * NH; i += 128) s_wo[i] = p.wo[i];
    for (int i = threadIdx.x; i < 4 * NH; i += 128) s_w2[i] = p.w2[i];
    if (threadIdx.x < NH) { s_b0[threadIdx.x] = p.b0[threadIdx.x]; s_wr[threadIdx.x] = p.wr[threadIdx.x]; }
    if (threadIdx.x < 4) s_b2[threadIdx.x] = p.b2[threadIdx.x];
    if (threadIdx.x < 32) s_wrel[threadIdx.x] = p.w_rel[threadIdx.x];
    if (threadIdx.x < 64) s_lb[threadIdx.x] = log_binom_f(63.f, (float)threadIdx.x);
    __syncthreads();
    const int f = blockIdx.z, y = blockIdx.y, x = blockIdx.x * 128 + threadIdx.x;
    if (x >= p.nw) return;
    const float fy = p.sy * (float)y, fx = p.sx * (float)x;
    const int y0 = min((int)fy, p.h3 - 1), y1 = min(y0 + 1, p.h3 - 1), x0 = min((int)fx, p.w3 - 1), x1 = min(x0 + 1, p.w3 - 1);
    const float ly = fy - (float)y0, hy = 1.f - ly, lx = fx - (float)x0, hx = 1.f - lx;
    const size_t i00 = ((size_t)f * p.h3 + y0) * p.w3 + x0, i01 = ((size_t)f * p.h3 + y0) * p.w3 + x1;
    const size_t i10 = ((size_t)f * p.h3 + y1) * p.w3 + x0, i11 = ((size_t)f * p.h3 + y1) * p.w3 + x1;
    float o[32];
    {
        const uint4 *op = reinterpret_cast<const uint4 *>(p.o32 + (((size_t)f * p.nh + y) * p.nw + x) * p.ldo);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const uint4 u = __ldg(op + q);
            const __half2 *h2 = reinterpret_cast<const __half2 *>(&u);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float2 o2 = __half22float2(h2[e]);
                o[q * 8 + 2 * e] = o2.x;
                o[q * 8 + 2 * e + 1] = o2.y;
            }
        }
    }
    float rel = p.b_rel;
#pragma unroll
    for (int c = 0; c < 32; ++c) rel = fmaf(s_wrel[c], o[c], rel);
    rel = fmaxf(rel, 0.f);                                                     // MiDaS non_negative head: final ReLU
    float pt[4] = {s_b2[0], s_b2[1], s_b2[2], s_b2[3]};
#pragma unroll 1
    for (int half = 0; half < 2; ++half) {
        const int h0 = half * 40;
        // pre-activation of mlp.0 = b0 + w_r rel + W_o . out_conv + bilinear(W_e . b_emb), hidden units h0 .. h0+39
        float pre[40];
        const float4 *z00 = reinterpret_cast<const float4 *>(p.ze + i00 * p.ldz + h0), *z01 = reinterpret_cast<const float4 *>(p.ze + i01 * p.ldz + h0);
        const float4 *z10 = reinterpret_cast<const float4 *>(p.ze + i10 * p.ldz + h0), *z11 = reinterpret_cast<const float4 *>(p.ze + i11 * p.ldz + h0);
#pragma unroll
        for (int k = 0; k < 10; ++k) {
            const float4 a = __ldg(z00 + k), b = __ldg(z01 + k), c = __ldg(z10 + k), d = __ldg(z11 + k);
            pre[4 * k + 0] = fmaf(s_wr[h0 + 4 * k + 0], rel, s_b0[h0 + 4 * k + 0]) + (hy * (hx * a.x + lx * b.x) + ly * (hx * c.x + lx * d.x));
            pre[4 * k + 1] = fmaf(s_wr[h0 + 4 * k + 1], rel, s_b0[h0 + 4 * k + 1]) + (hy * (hx * a.y + lx * b.y) + ly * (hx * c.y + lx * d.y));
            pre[4 * k + 2] = fmaf(s_wr[h0 + 4 * k + 2], rel, s_b0[h0 + 4 * k + 2]) + (hy * (hx * a.z + lx * b.z) + ly * (hx * c.z + lx * d.z));
            pre[4 * k + 3] = fmaf(s_wr[h0 + 4 * k + 3], rel, s_b0[h0 + 4 * k + 3]) + (hy * (hx * a.w + lx * b.w) + ly * (hx * c.w + lx * d.w));
        }
#pragma unroll
        for (int c = 0; c < 32; ++c) {
            const float *w = s_wo + c * NH + h0;
#pragma unroll
            for (int k = 0; k < 40; ++k) pre[k] = fmaf(w[k], o[c], pre[k]);
        }
#pragma unroll
        for (int k = 0; k < 40; ++k) {
            const float g = 0.5f * pre[k] * (1.f + erff(pre[k] * 0.70710678118654752f));             // nn.GELU (erf form)
#pragma unroll
            for (int j = 0; j < 4; ++j) pt[j] = fmaf(s_w2[j * NH + h0 + k], g, pt[j]);
        }
    }
    p.out[((size_t)f * p.nh + y) * p.nw + x] = log_binomial_expectation(pt, s_lb, p.min_temp, p.max_temp, p.bc, i00, i01, i10, i11, hy, hx, ly, lx);
}

// out[b, y, x] = 0.5 * (up(d[2b])[y + pad_h, x + pad_w] + up(d[2b+1])[y + pad_h, Wp - 1 - (x + pad_w)]), up = bicubic
// align_corners=False from (nh, nw) to the padded size (Hp, Wp); identity when the sizes agree (depth_model.py:88-89)
__global__ void __launch_bounds__(256) tta_combine_kernel(const float *__restrict__ d, int B, int nh, int nw, int Hp, int Wp, int pad_h, int pad_w,
                                                          int H, int W, float *__restrict__ out) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)B * H * W;
    if (idx >= total) return;
    const int x = (int)(idx % W);
    const int y = (int)((idx / W) % H);
    const int b = (int)(idx / ((long long)W * H));
    const bool same = (nh == Hp && nw == Wp);
    const float sy = (float)nh / (float)Hp, sx = (float)nw / (float)Wp;
    auto sample = [&](const float *img, int yy, int xx) {
        if (same) return img[(long long)yy * nw + xx];
        float fy = sy * ((float)yy + 0.5f) - 0.5f, fx = sx * ((float)xx + 0.5f) - 0.5f;
        const int iy = (int)floorf(fy), ix = (int)floorf(fx);
        fy -= (float)iy; fx -= (float)ix;
        float cx[4], cy[4];
        cubic_coeffs_z(fx, cx);
        cubic_coeffs_z(fy, cy);
        float acc = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int yr = min(max(iy - 1 + j, 0), nh - 1);
            float r = 0.f;
#pragma unroll
            for (int i = 0; i < 4; ++i) r += cx[i] * img[(long long)yr * nw + min(max(ix - 1 + i, 0), nw - 1)];
            acc += cy[j] * r;
        }
        return acc;
    };
    const float a = sample(d + (long long)(2 * b) * nh * nw, y + pad_h, x + pad_w);
    const float c = sample(d + (long long)(2 * b + 1) * nh * nw, y + pad_h, Wp - 1 - (x + pad_w));
    out[idx] = (a + c) / 2.f;
}

}  // namespace dm

#define DM_EXPORT extern "C" __attribute__((visibility("default")))

DM_EXPORT int dm_zoe_preprocess_patchify(const uint8_t *rgb, int B, int H, int W, int pad_h, int pad_w, int net_h, int net_w, int patch,
                                         void *out, int kpad, void *stream_) {
    using namespace dm;
    if (!rgb || !out || net_h % patch || net_w % patch || kpad != 3 * patch * patch || pad_h >= H || pad_w >= W || pad_h < 0 || pad_w < 0) {
        set_error("dm_zoe_preprocess_patchify: bad arguments (reflect padding must be smaller than the image; kpad = 3*patch^2)");
        return DM_E_INVALID;
    }
    ZoePre p;
    p.rgb = rgb; p.B = B; p.H = H; p.W = W; p.pad_h = pad_h; p.pad_w = pad_w; p.nh = net_h; p.nw = net_w; p.patch = patch;
    p.gh = net_h / patch; p.gw = net_w / patch; p.kpad = kpad; p.out = (__half *)out;
    const long long total = (long long)2 * B * net_h * net_w;
    zoe_preprocess_patchify_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream_>>>(p);
    DM_LAUNCH_CHECK("zoe_preprocess_patchify_kernel");
    return DM_OK;
}

DM_EXPORT int dm_layernorm_post_f16(float *x, long long rows, int C, const float *gamma, const float *beta, float eps, void *out, void *stream_) {
    using namespace dm;
    if (C != 128) { set_error("dm_layernorm_post_f16: width must be 128 (router embedding)"); return DM_E_UNSUPPORTED; }
    layernorm_post_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, (cudaStream_t)stream_>>>(x, rows, gamma, beta, eps, (__half *)out);
    DM_LAUNCH_CHECK("layernorm_post_kernel");
    return DM_OK;
}

DM_EXPORT int dm_attention_small_f16(const void *qkv, int F, int S, int heads, float scale, void *out, void *stream_) {
    using namespace dm;
    const size_t smem = ((size_t)2 * S * RA_PITCH + (size_t)8 * S) * sizeof(float);
    if (smem > 200 * 1024) { set_error("dm_attention_small_f16: %d tokens do not fit in shared memory", S); return DM_E_UNSUPPORTED; }
    if (smem > 48 * 1024) {
        static PerDeviceFlag configured;
        if (!configured.test_and_set())
            DM_CUDA_CHECK(cudaFuncSetAttribute(attention_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    }
    attention_small_kernel<<<dim3(F, heads, 4), 256, smem, (cudaStream_t)stream_>>>((const __half *)qkv, S, heads * RA_HD, scale, (__half *)out);   // 4 query-row blocks per (forward, head)
    DM_LAUNCH_CHECK("attention_small_kernel");
    return DM_OK;
}

DM_EXPORT int dm_cast_f32_f16(const float *x, long long n, void *out, void *stream_) {
    using namespace dm;
    if (n % 4) { set_error("dm_cast_f32_f16: element count must be a multiple of 4"); return DM_E_INVALID; }
    cast_f32_f16_kernel<<<(unsigned)((n / 4 + 255) / 256), 256, 0, (cudaStream_t)stream_>>>(x, n / 4, (__half *)out);
    DM_LAUNCH_CHECK("cast_f32_f16_kernel");
    return DM_OK;
}

DM_EXPORT int dm_zoe_select_softplus(const float *seed, int ld, const float *logits, int lld, int F, int rows_per_fwd, float *out, void *stream_) {
    using namespace dm;
    const long long rows = (long long)F * rows_per_fwd;
    select_softplus_kernel<<<(unsigned)((rows * 64 + 255) / 256), 256, 0, (cudaStream_t)stream_>>>(seed, ld, logits, lld, rows, rows_per_fwd, out);
    DM_LAUNCH_CHECK("select_softplus_kernel");
    return DM_OK;
}

DM_EXPORT int dm_resize_add_nhwc_f16(const void *a, const void *b_small, int B, int Hs, int Ws, int C, void *out, int H, int W, void *stream_) {
    using namespace dm;
    if (C % 8 || H > 65535 || B > 65535) { set_error("dm_resize_add_nhwc_f16: bad shape"); return DM_E_INVALID; }
    const float sy = H > 1 ? (float)(Hs - 1) / (float)(H - 1) : 0.f;
    const float sx = W > 1 ? (float)(Ws - 1) / (float)(W - 1) : 0.f;
    const dim3 grid((unsigned)((W * (C / 8) + 255) / 256), (unsigned)H, (unsigned)B);
    resize_add_nhwc_kernel<<<grid, 256, 0, (cudaStream_t)stream_>>>((const __half *)a, (const __half *)b_small, Hs, Ws, C, (__half *)out, H, W, sy, sx);
    DM_LAUNCH_CHECK("resize_add_nhwc_kernel");
    return DM_OK;
}

DM_EXPORT int dm_zoe_attractor(const float *A, int lda, const float *logits, int lld, const float *b_prev, int F, int Hp, int Wp, int H, int W,
                               float *b_out, void *stream_) {
    using namespace dm;
    if (H > 65535 || F > 65535) { set_error("dm_zoe_attractor: bad shape"); return DM_E_INVALID; }
    const float sy = H > 1 ? (float)(Hp - 1) / (float)(H - 1) : 0.f;
    const float sx = W > 1 ? (float)(Wp - 1) / (float)(W - 1) : 0.f;
    const dim3 grid((unsigned)((W * 64 + 255) / 256), (unsigned)H, (unsigned)F);
    attractor_kernel<16, false, true><<<grid, 256, 0, (cudaStream_t)stream_>>>(A, lda, logits, lld, b_prev, Hp, Wp, H, W, sy, sx, b_out, 0.f, 0.f, 0.f,
                                                                             nullptr);
    DM_LAUNCH_CHECK("attractor_kernel");
    return DM_OK;
}

DM_EXPORT int dm_zoe_attractor_single(const float *A, int lda, int n_attractors, int normed, const float *b_prev, int F, int Hp, int Wp, int H,
                                      int W, float min_depth, float max_depth, float *b_out, float *B_sorted, void *stream_) {
    using namespace dm;
    if (H > 65535 || F > 65535 || (B_sorted && !normed) || lda < (normed ? 2 : 1) * n_attractors) {
        set_error("dm_zoe_attractor_single: bad shape (lda must hold the attractor columns; B_sorted needs normed bin centres)");
        return DM_E_INVALID;
    }
    const float sy = H > 1 ? (float)(Hp - 1) / (float)(H - 1) : 0.f;
    const float sx = W > 1 ? (float)(Wp - 1) / (float)(W - 1) : 0.f;
    const float range = (float)((double)max_depth - (double)min_depth);
    const dim3 grid((unsigned)((W * 64 + 255) / 256), (unsigned)H, (unsigned)F);
    cudaStream_t st = (cudaStream_t)stream_;
#define DM_ATTR(NA, NORMED) attractor_kernel<NA, NORMED, false><<<grid, 256, 0, st>>>(A, lda, nullptr, 0, b_prev, Hp, Wp, H, W, sy, sx, b_out, \
                                                                                   min_depth, max_depth, range, B_sorted)
    switch (n_attractors * 2 + (normed ? 1 : 0)) {
        case 32: DM_ATTR(16, false); break;
        case 33: DM_ATTR(16, true); break;
        case 16: DM_ATTR(8, false); break;
        case 17: DM_ATTR(8, true); break;
        case 8: DM_ATTR(4, false); break;
        case 9: DM_ATTR(4, true); break;
        case 2: DM_ATTR(1, false); break;
        case 3: DM_ATTR(1, true); break;
        default: set_error("dm_zoe_attractor_single: %d attractors (built for 16, 8, 4, 1)", n_attractors); return DM_E_UNSUPPORTED;
    }
#undef DM_ATTR
    DM_LAUNCH_CHECK("attractor_kernel");
    return DM_OK;
}

DM_EXPORT int dm_zoe_seed_normed(const float *seed, int ld, long long rows, float min_depth, float max_depth, float *out, void *stream_) {
    using namespace dm;
    if (ld % 4 || ld < 64) { set_error("dm_zoe_seed_normed: ld must be a multiple of 4 and at least 64"); return DM_E_INVALID; }
    const float range = (float)((double)max_depth - (double)min_depth);
    seed_normed_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, (cudaStream_t)stream_>>>(seed, ld, rows, min_depth, range, out);
    DM_LAUNCH_CHECK("seed_normed_kernel");
    return DM_OK;
}

DM_EXPORT int dm_zoe_clb_final(const void *o32, int ldo, const float *ze, int ldz, const float *bc, const float *logits, int lld, const float *wo,
                               const float *b0, const float *w2, const float *b2, int F, int nh, int nw, int h3, int w3, float min_temp,
                               float max_temp, float *out, void *stream_) {
    using namespace dm;
    if (nh > 65535 || F > 65535) { set_error("dm_zoe_clb_final: bad shape"); return DM_E_INVALID; }
    ClbParams p;
    p.o32 = (const __half *)o32; p.ldo = ldo; p.ze = ze; p.ldz = ldz; p.bc = bc; p.logits = logits; p.lld = lld;
    p.wo = wo; p.b0 = b0; p.w2 = w2; p.b2 = b2; p.F = F; p.nh = nh; p.nw = nw; p.h3 = h3; p.w3 = w3;
    p.sy = nh > 1 ? (float)(h3 - 1) / (float)(nh - 1) : 0.f;
    p.sx = nw > 1 ? (float)(w3 - 1) / (float)(nw - 1) : 0.f;
    p.min_temp = min_temp; p.max_temp = max_temp; p.out = out;
    if (ldo % 8 || ldz % 4) { set_error("dm_zoe_clb_final: ldo must be a multiple of 8 and ldz of 4"); return DM_E_INVALID; }
    clb_final_kernel<<<dim3((unsigned)((nw + 127) / 128), (unsigned)nh, (unsigned)F), 128, 0, (cudaStream_t)stream_>>>(p);
    DM_LAUNCH_CHECK("clb_final_kernel");
    return DM_OK;
}

DM_EXPORT int dm_zoe_clb_final_single(const void *o32, int ldo, const float *ze, int ldz, const float *bc, const float *wo, const float *wr,
                                      const float *b0, const float *w2, const float *b2, const float *w_rel, float b_rel, int F, int nh, int nw,
                                      int h3, int w3, float min_temp, float max_temp, float *out, void *stream_) {
    using namespace dm;
    if (nh > 65535 || F > 65535) { set_error("dm_zoe_clb_final_single: bad shape"); return DM_E_INVALID; }
    if (ldo % 8 || ldz % 4 || ldz < 80) { set_error("dm_zoe_clb_final_single: ldo must be a multiple of 8 and ldz of 4, at least 80"); return DM_E_INVALID; }
    ClbSingleParams p;
    p.o32 = (const __half *)o32; p.ldo = ldo; p.ze = ze; p.ldz = ldz; p.bc = bc;
    p.wo = wo; p.wr = wr; p.b0 = b0; p.w2 = w2; p.b2 = b2; p.w_rel = w_rel; p.b_rel = b_rel; p.F = F; p.nh = nh; p.nw = nw; p.h3 = h3; p.w3 = w3;
    p.sy = nh > 1 ? (float)(h3 - 1) / (float)(nh - 1) : 0.f;
    p.sx = nw > 1 ? (float)(w3 - 1) / (float)(nw - 1) : 0.f;
    p.min_temp = min_temp; p.max_temp = max_temp; p.out = out;
    clb_final_single_kernel<<<dim3((unsigned)((nw + 127) / 128), (unsigned)nh, (unsigned)F), 128, 0, (cudaStream_t)stream_>>>(p);
    DM_LAUNCH_CHECK("clb_final_single_kernel");
    return DM_OK;
}

DM_EXPORT int dm_zoe_tta_combine(const float *d, int B, int nh, int nw, int pad_h, int pad_w, int H, int W, float *out, void *stream_) {
    using namespace dm;
    const long long total = (long long)B * H * W;
    tta_combine_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream_>>>(d, B, nh, nw, H + 2 * pad_h, W + 2 * pad_w, pad_h, pad_w, H, W, out);
    DM_LAUNCH_CHECK("tta_combine_kernel");
    return DM_OK;
}
