// Backward kernels of the hot path (training, SURVEY K12 / §8 row a13).
//
//  * input gradient of a conv  = the forward conv kernel run on the output gradient with the weights packed
//    transposed + flipped (vsrb_conv_geom.transpose = 1) - no new kernel;
//  * weight / bias gradient     = dW[co][ci][ky][kx] = sum_pixels dz[p][co] * x[p + tap][ci] on the tcgen05 kernels of
//    wgrad_tc.cu / wgrad_taps.cu, or the FFMA fallback conv_wgrad_kernel below (vsrb_conv2d_wgrad picks one per input
//    segment; reference: autograd's ConvolutionBackward0 of every nn.Conv2d on the path);
//  * flow_warp backward         = flow_warp_bwd_kernel: scatter of the output gradient through the four bilinear
//    taps (grad wrt the warped features) and the derivative of the taps wrt the sample position (grad wrt the
//    flow, needed when train_flow=True) - reference: GridSampler2DBackward0 behind spynet.py:95-106.
#include <algorithm>
#include <vector>

#include "common.cuh"
#include "warp_modes.cuh"

namespace vsrb {

template <typename T> struct Ld8;
template <> struct Ld8<__nv_bfloat16> {
    __device__ static void load(const __nv_bfloat16* p, float (&v)[8]) {
        uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
        float2 a = unpack_bf16(u.x), b = unpack_bf16(u.y), c = unpack_bf16(u.z), d = unpack_bf16(u.w);
        v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; v[4] = c.x; v[5] = c.y; v[6] = d.x; v[7] = d.y;
    }
};
template <> struct Ld8<float> {
    __device__ static void load(const float* p, float (&v)[8]) {
        float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    }
};

// ---------------------------------------------------------------------------------------
// weight gradient (FFMA fallback for the segments neither tcgen05 kernel takes: fp32 data, bf16 non-square filters).
// One CTA = one filter ROW ky x one 64(co) x 64(ci) tile x a run of 32-pixel row chunks.  Per chunk it stages dz
// [32 px][64 co] and ONE extended activation strip [32 + kw - 1 px][64 ci] of image row y + ky - pad, and updates the kw
// taps of the row from it (kw x 4x4 fp32 accumulators per thread), so dz is read kh times instead of kh*kw times.
// Results are added to the OIHW fp32 gradient with atomics.
// ---------------------------------------------------------------------------------------
struct WgradParams {
    const void* in[2];
    int in_c[2], seg_c[2], seg_off[2];
    const void* dz;
    int dz_c;
    int kh, kw, H, W;
    int cout, cin_total;
    int chunks_per_row, units, units_per_cta;     // unit = (image, row y, 32-pixel chunk)
    int n_co_blk, n_ci_blk;                       // 64-wide blocks
    int ci_blk_seg[8], ci_blk_c0[8];
    float* dw;
};

// A thread owns a 4x4 (co, ci) patch of the 64 x 64 tile; the 256 threads are one pixel group walking the 32 pixels of a
// chunk.
template <typename T, int KW>
__global__ void __launch_bounds__(256) conv_wgrad_kernel(WgradParams P) {
    __shared__ __align__(16) float zs[32][64];
    __shared__ __align__(16) float xs[32 + KW - 1][64];
    const int tid = threadIdx.x;
    const int tx = tid % 16, ty = tid / 16;             // 4 ci per tx, 4 co per ty
    const int ky = blockIdx.y;
    const int cib = blockIdx.z % P.n_ci_blk, cob = blockIdx.z / P.n_ci_blk;
    const int s = P.ci_blk_seg[cib], c0 = P.ci_blk_c0[cib];
    const int co0 = cob * 64;
    const int hw = P.H * P.W;
    const int u_begin = blockIdx.x * P.units_per_cta;
    const int u_end = min(u_begin + P.units_per_cta, P.units);
    const T* zin = reinterpret_cast<const T*>(P.dz);
    const T* xin = reinterpret_cast<const T*>(P.in[s]);
    const int dy = ky - P.kh / 2, pad = KW / 2;

    float acc[KW][4][4];
#pragma unroll
    for (int k = 0; k < KW; ++k)
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[k][i][j] = 0.f;

    for (int u = u_begin; u < u_end; ++u) {
        const int xc = u % P.chunks_per_row;
        const int rowi = u / P.chunks_per_row;
        const int y = rowi % P.H;
        const long long img = rowi / P.H;
        const int x0 = xc * 32;
        const int yy = y + dy;
        __syncthreads();
        for (int i = tid; i < 32 * 8; i += 256) {           // dz chunk [32 px][64 co]
            const int lp = i / 8, lc = (i % 8) * 8;
            float zv[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) zv[e] = 0.f;
            if (x0 + lp < P.W && co0 + lc < P.dz_c) {
                Ld8<T>::load(zin + (img * hw + (long long)y * P.W + x0 + lp) * P.dz_c + co0 + lc, zv);
#pragma unroll
                for (int e = 0; e < 8; ++e)
                    if (co0 + lc + e >= P.cout) zv[e] = 0.f;
            }
            *reinterpret_cast<float4*>(&zs[lp][lc]) = make_float4(zv[0], zv[1], zv[2], zv[3]);
            *reinterpret_cast<float4*>(&zs[lp][lc + 4]) = make_float4(zv[4], zv[5], zv[6], zv[7]);
        }
        for (int i = tid; i < (32 + KW - 1) * 8; i += 256) {   // extended strip: image columns x0 - pad + e
            const int ep = i / 8, lc = (i % 8) * 8;
            float xv[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) xv[e] = 0.f;
            const int xx = x0 - pad + ep;
            if (yy >= 0 && yy < P.H && xx >= 0 && xx < P.W && c0 + lc < P.in_c[s]) {
                Ld8<T>::load(xin + (img * hw + (long long)yy * P.W + xx) * P.in_c[s] + c0 + lc, xv);
#pragma unroll
                for (int e = 0; e < 8; ++e)
                    if (c0 + lc + e >= P.seg_c[s]) xv[e] = 0.f;
            }
            *reinterpret_cast<float4*>(&xs[ep][lc]) = make_float4(xv[0], xv[1], xv[2], xv[3]);
            *reinterpret_cast<float4*>(&xs[ep][lc + 4]) = make_float4(xv[4], xv[5], xv[6], xv[7]);
        }
        __syncthreads();
#pragma unroll 2
        for (int q = 0; q < 32; ++q) {
            const float4 a = *reinterpret_cast<const float4*>(&zs[q][ty * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
            for (int k = 0; k < KW; ++k) {
                const float4 b = *reinterpret_cast<const float4*>(&xs[q + k][tx * 4]);
                const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[k][i][j] = fmaf(av[i], bv[j], acc[k][i][j]);
            }
        }
    }
    const int taps = P.kh * KW;
#pragma unroll
    for (int k = 0; k < KW; ++k)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int co = co0 + ty * 4 + i;
            if (co >= P.cout) continue;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int ci = c0 + tx * 4 + j;
                if (ci < P.seg_c[s])
                    atomicAdd(P.dw + ((size_t)co * P.cin_total + P.seg_off[s] + ci) * taps + ky * KW + k, acc[k][i][j]);
            }
        }
}

// ---------------------------------------------------------------------------------------
// flow_warp backward.  C/8 (bf16) or C/4 (fp32) threads per pixel as in the forward kernel; dx is an fp32
// buffer (zeroed by the caller) updated with atomics; dflow gets the channel-reduced tap derivative.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void sample_pos_b(float px, float py, int w, int h, float& ix, float& iy) {
    float nx = 2.0f * px / (float)max(w - 1, 1) - 1.0f;
    float ny = 2.0f * py / (float)max(h - 1, 1) - 1.0f;
    ix = (nx + 1.0f) / 2.0f * (float)(w - 1);
    iy = (ny + 1.0f) / 2.0f * (float)(h - 1);
}

template <typename T, int TPP>
__global__ void __launch_bounds__(256) flow_warp_bwd_kernel(const T* __restrict__ x, const float2* __restrict__ flow,
                                                            const T* __restrict__ dout, float* __restrict__ dx,
                                                            float2* __restrict__ dflow, int n, int h, int w, int border,
                                                            int tpp_rt) {
    constexpr int VEC = 16 / sizeof(T);
    const int tpp = TPP > 0 ? TPP : tpp_rt;            // TPP == 0: any channel count; dflow must then be zeroed (atomics)
    const int C = tpp * VEC;
    const int hw = h * w;
    const long long total = (long long)n * hw * tpp;
    const long long total_up = (total + 31) / 32 * 32;          // whole warps iterate together (shuffles below)
    for (long long i0 = (long long)blockIdx.x * 256 + threadIdx.x; i0 < total_up; i0 += (long long)gridDim.x * 256) {
        const bool live = i0 < total;
        const long long i = live ? i0 : total - 1;              // dead lanes shadow the last item, write nothing
        const int part = (int)(i % tpp);
        const long long pix = i / tpp;
        const int img = (int)(pix / hw), r = (int)(pix - (long long)img * hw);
        const int yy = r / w, xx = r - yy * w;
        const float2 f = __ldg(flow + pix);
        float ix, iy;
        sample_pos_b((float)xx + f.x, (float)yy + f.y, w, h, ix, iy);
        float gmx = 1.f, gmy = 1.f;                    // derivative of the border clamp
        if (border) {
            if (ix < 0.f || ix > (float)(w - 1)) gmx = 0.f;
            if (iy < 0.f || iy > (float)(h - 1)) gmy = 0.f;
            ix = fminf(fmaxf(ix, 0.f), (float)(w - 1));
            iy = fminf(fmaxf(iy, 0.f), (float)(h - 1));
        }
        float fx = floorf(ix), fy = floorf(iy);
        const float wx1 = ix - fx, wy1 = iy - fy, wx0 = 1.f - wx1, wy0 = 1.f - wy1;
        fx = fminf(fmaxf(fx, -2.f), (float)w);
        fy = fminf(fmaxf(fy, -2.f), (float)h);
        const int x0 = (int)fx, y0 = (int)fy;
        float go[VEC];
        {
            float tmp[8];
            if (VEC == 8) {
                Ld8<T>::load(dout + pix * C + part * VEC, tmp);
#pragma unroll
                for (int j = 0; j < VEC; ++j) go[j] = tmp[j];
            } else {
                const float4 q = __ldg(reinterpret_cast<const float4*>(dout + pix * C + part * VEC));
                go[0] = q.x; go[1] = q.y; go[2] = q.z; go[3] = q.w;
            }
        }
        float gx = 0.f, gy = 0.f;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int xi = x0 + (k & 1), yi = y0 + (k >> 1);
            if (xi < 0 || xi >= w || yi < 0 || yi >= h) continue;
            const float wgt = ((k & 1) ? wx1 : wx0) * ((k >> 1) ? wy1 : wy0);
            const float dwx = ((k & 1) ? 1.f : -1.f) * ((k >> 1) ? wy1 : wy0);   // d wgt / d ix
            const float dwy = ((k >> 1) ? 1.f : -1.f) * ((k & 1) ? wx1 : wx0);   // d wgt / d iy
            const long long tp = ((long long)img * hw + (long long)yi * w + xi) * C + part * VEC;
            float xv[VEC];
            if (dflow) {
                if (VEC == 8) {
                    float tmp[8];
                    Ld8<T>::load(x + tp, tmp);
#pragma unroll
                    for (int j = 0; j < VEC; ++j) xv[j] = tmp[j];
                } else {
                    const float4 q = __ldg(reinterpret_cast<const float4*>(x + tp));
                    xv[0] = q.x; xv[1] = q.y; xv[2] = q.z; xv[3] = q.w;
                }
            }
#pragma unroll
            for (int j = 0; j < VEC; ++j) {
                if (dx && live) atomicAdd(dx + tp + j, go[j] * wgt);
                if (dflow) {
                    gx = fmaf(go[j] * xv[j], dwx, gx);
                    gy = fmaf(go[j] * xv[j], dwy, gy);
                }
            }
        }
        if (dflow) {
            if (TPP > 0) {
                // reduce over the TPP lanes of this pixel (TPP is a power of two <= 32, lanes are consecutive)
#pragma unroll
                for (int o = TPP / 2; o > 0; o >>= 1) {
                    gx += __shfl_xor_sync(0xffffffffu, gx, o);
                    gy += __shfl_xor_sync(0xffffffffu, gy, o);
                }
                if (part == 0 && live) dflow[pix] = make_float2(gx * gmx, gy * gmy);
            } else if (live) {
                atomicAdd(&dflow[pix].x, gx * gmx);
                atomicAdd(&dflow[pix].y, gy * gmy);
            }
        }
    }
}

template <typename T>
static int launch_warp_bwd(const T* x, const float2* flow, const T* dout, float* dx, float2* dflow, int n, int h, int w, int c,
                           int border, cudaStream_t s) {
    constexpr int VEC = 16 / sizeof(T);
    const int tpp = c / VEC;
    const long long total = (long long)n * h * w * tpp;
    long long b = (total + 255) / 256;
    // whole warps must stay inside the loop together for the shuffles: total is a multiple of tpp and
    // 256 % tpp == 0, and a grid-stride of gridDim*256 keeps a pixel's lanes in one warp
    if (b > 148 * 16) b = 148 * 16;
    const int blocks = (int)b;
    switch (tpp) {
        case 1: flow_warp_bwd_kernel<T, 1><<<blocks, 256, 0, s>>>(x, flow, dout, dx, dflow, n, h, w, border, tpp); break;
        case 2: flow_warp_bwd_kernel<T, 2><<<blocks, 256, 0, s>>>(x, flow, dout, dx, dflow, n, h, w, border, tpp); break;
        case 4: flow_warp_bwd_kernel<T, 4><<<blocks, 256, 0, s>>>(x, flow, dout, dx, dflow, n, h, w, border, tpp); break;
        case 8: flow_warp_bwd_kernel<T, 8><<<blocks, 256, 0, s>>>(x, flow, dout, dx, dflow, n, h, w, border, tpp); break;
        case 16: flow_warp_bwd_kernel<T, 16><<<blocks, 256, 0, s>>>(x, flow, dout, dx, dflow, n, h, w, border, tpp); break;
        case 32: flow_warp_bwd_kernel<T, 32><<<blocks, 256, 0, s>>>(x, flow, dout, dx, dflow, n, h, w, border, tpp); break;
        default:
            if (dflow) cudaMemsetAsync(dflow, 0, sizeof(float2) * (size_t)n * h * w, s);
            flow_warp_bwd_kernel<T, 0><<<blocks, 256, 0, s>>>(x, flow, dout, dx, dflow, n, h, w, border, tpp);
            break;
    }
    return VSRB_OK;
}

// ---------------------------------------------------------------------------------------
// flow_warp_ex backward (nearest / bicubic, reflection, align_corners=False): flow_warp_bwd_kernel's work split, taps
// from warp_modes.cuh.  dx: the output gradient scattered through the taps (fp32 atomics; reflected / clipped taps may
// coincide).  dflow: sum over taps and channels of dout * x * d weight / d coordinate, times the derivative of the
// coordinate wrt the flow (un-normalisation, and for nearest / bilinear the padding).  nearest: 0.
// ---------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ void ld_vec(const T* p, float (&v)[16 / sizeof(T)]) {
    if constexpr (sizeof(T) == 2) {
        Ld8<T>::load(p, v);
    } else {
        const float4 q = __ldg(reinterpret_cast<const float4*>(p));
        v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
    }
}

template <typename T, int TPP, int kInterp>
__global__ void __launch_bounds__(256) flow_warp_ex_bwd_kernel(const T* __restrict__ x, const float2* __restrict__ flow,
                                                               const T* __restrict__ dout, float* __restrict__ dx,
                                                               float2* __restrict__ dflow, int n, int h, int w, int pad, int align,
                                                               int tpp_rt) {
    constexpr int VEC = 16 / sizeof(T);
    const int tpp = TPP > 0 ? TPP : tpp_rt;            // TPP == 0: any channel count; dflow must then be zeroed (atomics)
    const int C = tpp * VEC;
    const int hw = h * w;
    const long long total = (long long)n * hw * tpp;
    const long long total_up = (total + 31) / 32 * 32;          // whole warps iterate together (shuffles below)
    for (long long i0 = (long long)blockIdx.x * 256 + threadIdx.x; i0 < total_up; i0 += (long long)gridDim.x * 256) {
        const bool live = i0 < total;
        const long long i = live ? i0 : total - 1;              // dead lanes shadow the last item, write nothing
        const int part = (int)(i % tpp);
        const long long pix = i / tpp;
        const int img = (int)(pix / hw), r = (int)(pix - (long long)img * hw);
        const int yy = r / w, xx = r - yy * w;
        const float2 f = __ldg(flow + pix);
        float ix = ex_unnormalize((float)xx + f.x, w, align), iy = ex_unnormalize((float)yy + f.y, h, align);
        float gmx = ex_unnormalize_grad(w, align), gmy = ex_unnormalize_grad(h, align);
        const T* xb = x + (long long)img * hw * C + part * VEC;
        float* dxb = dx + (long long)img * hw * C + part * VEC;
        float go[VEC];
        ld_vec<T>(dout + pix * C + part * VEC, go);
        float gx = 0.f, gy = 0.f;
        if constexpr (kInterp == VSRB_INTERP_NEAREST) {
            float g;
            const int xi = ex_index(nearbyintf(ex_pad_coord(ix, w, pad, align, g)), w);
            const int yi = ex_index(nearbyintf(ex_pad_coord(iy, h, pad, align, g)), h);
            if (dx && live && xi >= 0 && yi >= 0) {
#pragma unroll
                for (int j = 0; j < VEC; ++j) atomicAdd(dxb + ((long long)yi * w + xi) * C + j, go[j]);
            }
            gmx = gmy = 0.f;                           // piecewise constant in the flow
        } else if constexpr (kInterp == VSRB_INTERP_BILINEAR) {
            float px, py;
            ix = ex_pad_coord(ix, w, pad, align, px);
            iy = ex_pad_coord(iy, h, pad, align, py);
            gmx *= px;
            gmy *= py;
            float fx = floorf(ix), fy = floorf(iy);
            const float wx1 = ix - fx, wy1 = iy - fy, wx0 = 1.f - wx1, wy0 = 1.f - wy1;
            fx = fminf(fmaxf(fx, -2.f), (float)w);
            fy = fminf(fmaxf(fy, -2.f), (float)h);
            const int x0 = (int)fx, y0 = (int)fy;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int xi = x0 + (k & 1), yi = y0 + (k >> 1);
                if (xi < 0 || xi >= w || yi < 0 || yi >= h) continue;
                const long long tp = ((long long)yi * w + xi) * C;
                if (dx && live) {
                    const float wgt = ((k & 1) ? wx1 : wx0) * ((k >> 1) ? wy1 : wy0);
#pragma unroll
                    for (int j = 0; j < VEC; ++j) atomicAdd(dxb + tp + j, go[j] * wgt);
                }
                if (dflow) {
                    float xv[VEC];
                    ld_vec<T>(xb + tp, xv);
                    float dot = 0.f;
#pragma unroll
                    for (int j = 0; j < VEC; ++j) dot = fmaf(go[j], xv[j], dot);
                    gx = fmaf(dot, ((k & 1) ? 1.f : -1.f) * ((k >> 1) ? wy1 : wy0), gx);
                    gy = fmaf(dot, ((k >> 1) ? 1.f : -1.f) * ((k & 1) ? wx1 : wx0), gy);
                }
            }
        } else {
            const float fx = floorf(ix), fy = floorf(iy);
            float wx[4], wy[4], dwx[4], dwy[4];
            cubic_weights(ix - fx, wx);
            cubic_weights(iy - fy, wy);
            cubic_weights_grad(ix - fx, dwx);
            cubic_weights_grad(iy - fy, dwy);
            int xo[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) xo[q] = ex_bicubic_tap(fx + (float)(q - 1), w, pad, align);
#pragma unroll
            for (int rr = 0; rr < 4; ++rr) {
                const int yi = ex_bicubic_tap(fy + (float)(rr - 1), h, pad, align);
                if (yi < 0) continue;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    if (xo[q] < 0) continue;
                    const long long tp = ((long long)yi * w + xo[q]) * C;
                    if (dx && live) {
                        const float wgt = wx[q] * wy[rr];
#pragma unroll
                        for (int j = 0; j < VEC; ++j) atomicAdd(dxb + tp + j, go[j] * wgt);
                    }
                    if (dflow) {
                        float xv[VEC];
                        ld_vec<T>(xb + tp, xv);
                        float dot = 0.f;
#pragma unroll
                        for (int j = 0; j < VEC; ++j) dot = fmaf(go[j], xv[j], dot);
                        gx = fmaf(dot, dwx[q] * wy[rr], gx);
                        gy = fmaf(dot, wx[q] * dwy[rr], gy);
                    }
                }
            }
        }
        if (dflow) {
            if (TPP > 0) {
#pragma unroll
                for (int o = TPP / 2; o > 0; o >>= 1) {
                    gx += __shfl_xor_sync(0xffffffffu, gx, o);
                    gy += __shfl_xor_sync(0xffffffffu, gy, o);
                }
                if (part == 0 && live) dflow[pix] = make_float2(gx * gmx, gy * gmy);
            } else if (live && kInterp != VSRB_INTERP_NEAREST) {
                atomicAdd(&dflow[pix].x, gx * gmx);
                atomicAdd(&dflow[pix].y, gy * gmy);
            }
        }
    }
}

template <typename T, int kInterp>
static void launch_warp_ex_bwd_t(const T* x, const float2* flow, const T* dout, float* dx, float2* dflow, int n, int h, int w,
                                 int c, int pad, int align, cudaStream_t s) {
    constexpr int VEC = 16 / sizeof(T);
    const int tpp = c / VEC;
    const long long total = (long long)n * h * w * tpp;
    long long b = (total + 255) / 256;
    if (b > 148 * 16) b = 148 * 16;                    // grid-stride: a pixel's lanes stay in one warp (see launch_warp_bwd)
    const int blocks = (int)b;
#define VSRB_WARP_EX_BWD(TPP) \
    flow_warp_ex_bwd_kernel<T, TPP, kInterp><<<blocks, 256, 0, s>>>(x, flow, dout, dx, dflow, n, h, w, pad, align, tpp)
    switch (tpp) {
        case 1: VSRB_WARP_EX_BWD(1); break;
        case 2: VSRB_WARP_EX_BWD(2); break;
        case 4: VSRB_WARP_EX_BWD(4); break;
        case 8: VSRB_WARP_EX_BWD(8); break;
        case 16: VSRB_WARP_EX_BWD(16); break;
        case 32: VSRB_WARP_EX_BWD(32); break;
        default:
            if (dflow) cudaMemsetAsync(dflow, 0, sizeof(float2) * (size_t)n * h * w, s);
            VSRB_WARP_EX_BWD(0);
            break;
    }
#undef VSRB_WARP_EX_BWD
}

template <typename T>
static void launch_warp_ex_bwd(const T* x, const float2* flow, const T* dout, float* dx, float2* dflow, int n, int h, int w, int c,
                               int interp, int pad, int align, cudaStream_t s) {
    if (interp == VSRB_INTERP_NEAREST) launch_warp_ex_bwd_t<T, VSRB_INTERP_NEAREST>(x, flow, dout, dx, dflow, n, h, w, c, pad, align, s);
    else if (interp == VSRB_INTERP_BICUBIC) launch_warp_ex_bwd_t<T, VSRB_INTERP_BICUBIC>(x, flow, dout, dx, dflow, n, h, w, c, pad, align, s);
    else launch_warp_ex_bwd_t<T, VSRB_INTERP_BILINEAR>(x, flow, dout, dx, dflow, n, h, w, c, pad, align, s);
}

int launch_bias_grad(const void* dz, int dz_c, long long pixels, int cout, int dtype, float* db, cudaStream_t s, WgradDet* det);
int launch_wgrad_tc_multi(const void* const* xs, int x_c, int c0, int ci_off, const void* const* dzs, int dz_c, int n_chunks,
                          int batch, int h, int w, int cout, int cin_total, float* dw, cudaStream_t stream, float* db, WgradDet* det);
int launch_wgrad_taps(const void* x, int x_c, int x_c0, int ci_n, int ci_off, const void* dz, int dz_c, int z_c0, int co_n, int K,
                      int batch, int h, int w, int cin_total, float* dw, cudaStream_t stream, WgradDet* det);

// The kernel that computes the weight gradient of input segment s.  3x3 layers whose segment has a multiple of 64 channels
// (the resblock, upsampling and HR convs: > 85 % of the FLOPs) run on wgrad_tc_kernel - except thin outputs: the 64 -> 3
// image convs would zero-fill 61 of its 64 dz columns.  Every other bf16 segment of an odd square filter up to 7x7
// (SPyNet's 7x7 stacks, 3-channel image segments, 1x1, thin outputs) runs on the tap-stacking kernel of wgrad_taps.cu,
// and the rest (fp32 data, non-square filters) on the FFMA kernel conv_wgrad_kernel.
enum WgradPath { kWgradTc, kWgradTaps, kWgradFfma };
static WgradPath wgrad_path(const vsrb_conv_geom* g, int s) {
    if (g->dtype != VSRB_BF16) return kWgradFfma;
    if (g->kh == 3 && g->kw == 3 && g->seg_c[s] % 64 == 0 && g->cout > 16) return kWgradTc;
    if (g->kh == g->kw && (g->kw & 1) && g->kw <= 7) return kWgradTaps;
    return kWgradFfma;
}

// Every 64-channel block of input segment s on wgrad_tc_kernel, summed over n_chunks (x, dz) pairs.  The bias gradient
// rides on the first launch if *db is set (the kernel's idle epilogue warps add up the dz tiles it streams anyway); *db is
// then cleared.
static int wgrad_tc_segment(const vsrb_conv_geom* g, int s, const void* const* xs, int x_c, const void* const* dzs, int dz_c,
                            int n_chunks, int batch, int h, int w, int cin_total, float* dw, float** db, cudaStream_t st,
                            WgradDet* det) {
    for (int c0 = 0; c0 < g->seg_c[s]; c0 += 64) {
        int rc = launch_wgrad_tc_multi(xs, x_c, c0, g->seg_off[s] + c0, dzs, dz_c, n_chunks, batch, h, w, g->cout, cin_total, dw, st,
                                       *db, det);
        if (rc != VSRB_OK) return rc;
        *db = nullptr;
    }
    return VSRB_OK;
}

// ---------------------------------------------------------------------------------------
// Deterministic dx of flow_warp_bwd (vsrb_flow_warp_bwd_det).  The output gradient is scattered through the four bilinear
// taps as 64-bit fixed-point integers: integer addition is associative, so the order in which the atomics land does not
// change the sum.  The scale is a power of two derived from max|dout|, itself found with an atomicMax of the bit patterns
// (order-independent), such that no target can overflow: a target receives at most h*w contributions (one per source
// pixel of its image: a pixel's four taps are distinct) of at most max|dout| each.  The quantum is then at most
// max|dout| * h*w * 2^-60, far below fp32 rounding of any entry that is not ~2^-30 times smaller than max|dout|.
// ---------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) abs_max_kernel(const T* __restrict__ v, long long n, unsigned* __restrict__ out) {
    unsigned m = 0;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256)
        m = max(m, __float_as_uint(fabsf((float)v[i])));           // non-negative floats order like their bit patterns
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}

// 2^(62 - e - e_hw) with max|dout| < 2^e and h*w < 2^e_hw
__device__ __forceinline__ double fixed_scale(unsigned amax_bits, int hw) {
    int e;
    frexpf(__uint_as_float(amax_bits), &e);
    const int e_hw = 32 - __clz(hw);
    return ldexp(1.0, 62 - e - e_hw);
}

template <typename T>
__global__ void __launch_bounds__(256) flow_warp_bwd_dx_fixed_kernel(const float2* __restrict__ flow, const T* __restrict__ dout,
                                                                     unsigned long long* __restrict__ acc, const unsigned* __restrict__ amax,
                                                                     int n, int h, int w, int tpp, int border) {
    constexpr int VEC = 16 / sizeof(T);
    const unsigned mbits = *amax;
    if (mbits >= 0x7f800000u) return;                               // inf / NaN in dout: the conversion reports it
    const double scale = fixed_scale(mbits, h * w);
    const int C = tpp * VEC;
    const int hw = h * w;
    const long long total = (long long)n * hw * tpp;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
        const int part = (int)(i % tpp);
        const long long pix = i / tpp;
        const int img = (int)(pix / hw), r = (int)(pix - (long long)img * hw);
        const int yy = r / w, xx = r - yy * w;
        const float2 f = __ldg(flow + pix);
        float ix, iy;                                               // the forward's / flow_warp_bwd_kernel's fp32 arithmetic
        sample_pos_b((float)xx + f.x, (float)yy + f.y, w, h, ix, iy);
        if (border) {
            ix = fminf(fmaxf(ix, 0.f), (float)(w - 1));
            iy = fminf(fmaxf(iy, 0.f), (float)(h - 1));
        }
        float fx = floorf(ix), fy = floorf(iy);
        const float wx1 = ix - fx, wy1 = iy - fy, wx0 = 1.f - wx1, wy0 = 1.f - wy1;
        fx = fminf(fmaxf(fx, -2.f), (float)w);
        fy = fminf(fmaxf(fy, -2.f), (float)h);
        const int x0 = (int)fx, y0 = (int)fy;
        float go[VEC];
        ld_vec<T>(dout + pix * C + part * VEC, go);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int xi = x0 + (k & 1), yi = y0 + (k >> 1);
            if (xi < 0 || xi >= w || yi < 0 || yi >= h) continue;
            const double wgt = (double)(((k & 1) ? wx1 : wx0) * ((k >> 1) ? wy1 : wy0)) * scale;
            unsigned long long* dst = acc + ((long long)img * hw + (long long)yi * w + xi) * C + part * VEC;
#pragma unroll
            for (int j = 0; j < VEC; ++j)
                if (go[j] != 0.f) atomicAdd(dst + j, (unsigned long long)__double2ll_rn((double)go[j] * wgt));
        }
    }
}

// dx = acc / scale, one store per element (targets nothing reached get 0); a non-finite max|dout| gives NaN everywhere
__global__ void __launch_bounds__(256) fixed_to_float_kernel(const long long* __restrict__ acc, const unsigned* __restrict__ amax,
                                                             long long n, int hw, float* __restrict__ dx) {
    const unsigned mbits = *amax;
    const bool finite = mbits < 0x7f800000u;
    const double inv = finite ? 1.0 / fixed_scale(mbits, hw) : 0.0;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256)
        dx[i] = finite ? (float)((double)acc[i] * inv) : __int_as_float(0x7fffffff);
}

template <typename T>
static int launch_warp_bwd_dx_det(const float2* flow, const T* dout, float* dx, int n, int h, int w, int c, int border, void* ws,
                                  cudaStream_t s) {
    constexpr int VEC = 16 / sizeof(T);
    const long long elems = (long long)n * h * w * c;
    unsigned* amax = reinterpret_cast<unsigned*>(ws);
    long long* acc = reinterpret_cast<long long*>(reinterpret_cast<char*>(ws) + 16);
    VSRB_CUDA(cudaMemsetAsync(ws, 0, 16 + (size_t)elems * 8, s));
    auto grid = [](long long items) { long long b = (items + 255) / 256; return (int)(b > 148 * 16 ? 148 * 16 : b); };
    abs_max_kernel<T><<<grid(elems), 256, 0, s>>>(dout, elems, amax);
    flow_warp_bwd_dx_fixed_kernel<T><<<grid(elems / VEC), 256, 0, s>>>(flow, dout, reinterpret_cast<unsigned long long*>(acc), amax, n,
                                                                       h, w, c / VEC, border);
    fixed_to_float_kernel<<<grid(elems), 256, 0, s>>>(acc, amax, elems, h * w, dx);
    VSRB_LAUNCH_CHECK();
    return VSRB_OK;
}

static size_t warp_bwd_det_bytes(int n, int h, int w, int c) { return 16 + (size_t)n * h * w * c * 8; }

// The launches of vsrb_conv2d_wgrad_multi after its argument checks (det: deterministic mode, see WgradDet)
static int wgrad_multi_run(const vsrb_conv_geom* g, int n_chunks, const void* const* in, const int32_t* in_c, const void* const* dz,
                           int dz_c, int batch, int h, int w, int cin_total, float* dw, float* db, cudaStream_t st, WgradDet* det) {
    for (int k0 = 0; k0 < n_chunks; k0 += 16) {
        const int nk = n_chunks - k0 < 16 ? n_chunks - k0 : 16;
        float* bias = db;                                   // once per group of chunks
        for (int s = 0; s < g->n_seg; ++s) {
            const void* xs[16];
            for (int k = 0; k < nk; ++k) xs[k] = in[(size_t)(k0 + k) * g->n_seg + s];
            int rc = wgrad_tc_segment(g, s, xs, in_c[s], dz + k0, dz_c, nk, batch, h, w, cin_total, dw, &bias, st, det);
            if (rc != VSRB_OK) return rc;
        }
    }
    return VSRB_OK;
}

static int check_wgrad_multi(const vsrb_conv_geom* g, int32_t n_chunks, const void* const* in, const int32_t* in_c,
                             const void* const* dz, int32_t dz_c, int32_t cin_total, float* dw) {
    VSRB_CHECK_ARG(g && in && in_c && dz && dw && n_chunks >= 1, "wgrad_multi: null argument");
    VSRB_CHECK_ARG(g->dtype == VSRB_BF16 && g->kh == 3 && g->kw == 3 && g->groups == 1 && !g->pixshuf && !g->transpose &&
                       g->n_seg >= 1 && g->n_seg <= 2 && dz_c >= g->cout && dz_c % 8 == 0,
                   "wgrad_multi: bf16 3x3 ungrouped convs only (tensor-core path)");
    for (int s = 0; s < g->n_seg; ++s)
        VSRB_CHECK_ARG(g->seg_c[s] % 64 == 0 && in_c[s] % 8 == 0 && in_c[s] >= g->seg_c[s] && g->seg_off[s] + g->seg_c[s] <= cin_total,
                       "wgrad_multi: segment %d must have a multiple of 64 channels", s);
    return VSRB_OK;
}

static int wgrad_impl(const vsrb_conv_geom* g, const void* const* in, const int32_t* in_c, const void* dz, int32_t dz_c,
                      int32_t batch, int32_t h, int32_t w, int32_t imgs_per_group, int32_t cin_total, float* dw, float* db,
                      void* stream, WgradDet* det);

// Runs `run` once in planning mode, checks the caller's workspace against what it needs, then runs it for real.
template <typename Run>
static int det_run(void* workspace, size_t workspace_bytes, const char* what, Run run) {
    WgradDet det = {nullptr, 0, true};
    int rc = run(&det);
    if (rc != VSRB_OK) return rc;
    VSRB_CHECK_ARG(det.need * 4 <= workspace_bytes && (det.need == 0 || workspace) && (reinterpret_cast<uintptr_t>(workspace) & 15) == 0,
                   "%s: the workspace must be 16-byte aligned and hold %zu bytes (got %zu)", what, det.need * 4, workspace_bytes);
    det.ws = reinterpret_cast<float*>(workspace);
    det.plan = false;
    return run(&det);
}

}  // namespace vsrb

using namespace vsrb;

extern "C" {

int vsrb_conv2d_wgrad_multi(const vsrb_conv_geom* g, int32_t n_chunks, const void* const* in, const int32_t* in_c,
                            const void* const* dz, int32_t dz_c, int32_t batch, int32_t h, int32_t w, int32_t cin_total,
                            float* dw, float* db, void* stream) {
    const int rc = check_wgrad_multi(g, n_chunks, in, in_c, dz, dz_c, cin_total, dw);
    if (rc != VSRB_OK) return rc;
    return wgrad_multi_run(g, n_chunks, in, in_c, dz, dz_c, batch, h, w, cin_total, dw, db, (cudaStream_t)stream, nullptr);
}

int vsrb_conv2d_wgrad_multi_det(const vsrb_conv_geom* g, int32_t n_chunks, const void* const* in, const int32_t* in_c,
                                const void* const* dz, int32_t dz_c, int32_t batch, int32_t h, int32_t w, int32_t cin_total,
                                float* dw, float* db, void* workspace, size_t workspace_bytes, void* stream) {
    const int rc = check_wgrad_multi(g, n_chunks, in, in_c, dz, dz_c, cin_total, dw);
    if (rc != VSRB_OK) return rc;
    return det_run(workspace, workspace_bytes, "wgrad_multi_det", [&](WgradDet* det) {
        return wgrad_multi_run(g, n_chunks, in, in_c, dz, dz_c, batch, h, w, cin_total, dw, db, (cudaStream_t)stream, det);
    });
}

int vsrb_conv2d_wgrad(const vsrb_conv_geom* g, const void* const* in, const int32_t* in_c, const void* dz, int32_t dz_c,
                      int32_t batch, int32_t h, int32_t w, int32_t imgs_per_group, int32_t cin_total, float* dw, float* db,
                      void* stream) {
    return wgrad_impl(g, in, in_c, dz, dz_c, batch, h, w, imgs_per_group, cin_total, dw, db, stream, nullptr);
}

int vsrb_conv2d_wgrad_det(const vsrb_conv_geom* g, const void* const* in, const int32_t* in_c, const void* dz, int32_t dz_c,
                          int32_t batch, int32_t h, int32_t w, int32_t imgs_per_group, int32_t cin_total, float* dw, float* db,
                          void* workspace, size_t workspace_bytes, void* stream) {
    return det_run(workspace, workspace_bytes, "wgrad_det", [&](WgradDet* det) {
        return wgrad_impl(g, in, in_c, dz, dz_c, batch, h, w, imgs_per_group, cin_total, dw, db, stream, det);
    });
}

size_t vsrb_conv2d_wgrad_det_workspace_bytes(const vsrb_conv_geom* g, int32_t n_chunks, int32_t batch, int32_t h, int32_t w,
                                             int32_t with_bias) {
    // the planning pass of the entry point on placeholder tensors (16-byte aligned, never dereferenced: nothing is launched)
    if (!g || n_chunks < 1 || n_chunks > 4096 || g->n_seg < 1 || g->n_seg > 2) {
        set_error("wgrad_det_workspace_bytes: bad geometry or chunk count");
        return 0;
    }
    const void* fake = reinterpret_cast<const void*>(uintptr_t(1) << 20);
    std::vector<const void*> ins((size_t)n_chunks * g->n_seg, fake), dzs((size_t)n_chunks, fake);
    int32_t in_c[2] = {(g->seg_c[0] + 7) / 8 * 8, g->n_seg > 1 ? (g->seg_c[1] + 7) / 8 * 8 : 0};
    const int cin_total = g->n_seg > 1 ? std::max(g->seg_off[0] + g->seg_c[0], g->seg_off[1] + g->seg_c[1]) : g->seg_off[0] + g->seg_c[0];
    float* dw = reinterpret_cast<float*>(uintptr_t(1) << 20);
    float* db = with_bias ? dw : nullptr;
    const int dz_c = (g->cout + 7) / 8 * 8;
    WgradDet det = {nullptr, 0, true};
    const int rc = n_chunks == 1
        ? wgrad_impl(g, ins.data(), in_c, fake, dz_c, batch, h, w, batch, cin_total, dw, db, nullptr, &det)
        : (check_wgrad_multi(g, n_chunks, ins.data(), in_c, dzs.data(), dz_c, cin_total, dw) != VSRB_OK
               ? VSRB_E_ARG
               : wgrad_multi_run(g, n_chunks, ins.data(), in_c, dzs.data(), dz_c, batch, h, w, cin_total, dw, db, nullptr, &det));
    return rc == VSRB_OK ? std::max<size_t>(det.need * 4, 16) : 0;
}

}  // extern "C"

namespace vsrb {
static int wgrad_impl(const vsrb_conv_geom* g, const void* const* in, const int32_t* in_c, const void* dz, int32_t dz_c,
                      int32_t batch, int32_t h, int32_t w, int32_t imgs_per_group, int32_t cin_total, float* dw, float* db,
                      void* stream, WgradDet* det) {
    VSRB_CHECK_ARG(g && in && in_c && dz && dw, "wgrad: null argument");
    VSRB_CHECK_ARG(g->n_seg == 1 || g->n_seg == 2, "wgrad: n_seg must be 1 or 2");
    VSRB_CHECK_ARG(!g->pixshuf && !g->transpose, "wgrad: pass the plain forward geometry (un-shuffle the gradient first)");
    VSRB_CHECK_ARG(g->groups == 1 && imgs_per_group == batch, "wgrad: grouped weight gradients are not supported (groups %d, "
                   "imgs_per_group %d, batch %d): call once per group", g->groups, imgs_per_group, batch);
    VSRB_CHECK_ARG(batch >= 1 && h >= 1 && w >= 1 && (long long)batch * h * w < (1LL << 31), "wgrad: 1 .. 2^31 - 1 pixels");
    VSRB_CHECK_ARG(g->dtype == VSRB_BF16 || g->dtype == VSRB_F32, "wgrad: dtype must be bf16 or fp32");
    VSRB_CHECK_ARG(g->kh >= 1 && g->kh <= 7 && (g->kh & 1) && g->kw >= 1 && g->kw <= 7 && (g->kw & 1),
                   "wgrad: kernel %dx%d unsupported (odd sizes 1..7)", g->kh, g->kw);
    VSRB_CHECK_ARG(dz_c % 8 == 0 && dz_c >= g->cout, "wgrad: dz channel stride %d must be a multiple of 8 and >= cout %d", dz_c,
                   g->cout);
    VSRB_CHECK_ARG((reinterpret_cast<uintptr_t>(dz) & 15) == 0, "wgrad: dz must be 16-byte aligned");
    WgradParams P;
    memset(&P, 0, sizeof(P));
    for (int s = 0; s < g->n_seg; ++s) {
        VSRB_CHECK_ARG(in[s] && (reinterpret_cast<uintptr_t>(in[s]) & 15) == 0, "wgrad: input segment %d must be 16-byte aligned", s);
        VSRB_CHECK_ARG(in_c[s] % 8 == 0 && in_c[s] >= g->seg_c[s],
                       "wgrad: input segment %d: channel stride %d must be a multiple of 8 and >= its %d channels", s, in_c[s], g->seg_c[s]);
        VSRB_CHECK_ARG(g->seg_off[s] + g->seg_c[s] <= cin_total, "wgrad: segment %d exceeds cin_total", s);
        P.in[s] = in[s]; P.in_c[s] = in_c[s]; P.seg_c[s] = g->seg_c[s]; P.seg_off[s] = g->seg_off[s];
        if (wgrad_path(g, s) != kWgradFfma) continue;
        VSRB_CHECK_ARG(!det, "wgrad_det: no deterministic kernel for a %dx%d %s filter (its FFMA fallback adds with atomics)", g->kh,
                       g->kw, g->dtype == VSRB_BF16 ? "bf16" : "fp32");
        VSRB_CHECK_ARG(g->kw == 1 || g->kw == 3 || g->kw == 7, "wgrad: no kernel for a %dx%d %s filter (the FFMA fallback takes "
                       "widths 1, 3 and 7)", g->kh, g->kw, g->dtype == VSRB_BF16 ? "bf16" : "fp32");
        for (int c0 = 0; c0 < g->seg_c[s]; c0 += 64) {
            VSRB_CHECK_ARG(P.n_ci_blk < 8, "wgrad: more than 512 input channels on the FFMA fallback");
            P.ci_blk_seg[P.n_ci_blk] = s;
            P.ci_blk_c0[P.n_ci_blk] = c0;
            ++P.n_ci_blk;
        }
    }
    cudaStream_t st = (cudaStream_t)stream;
    float* bias = db;
    for (int s = 0; s < g->n_seg; ++s) {
        const WgradPath path = wgrad_path(g, s);
        if (path == kWgradTc) {
            int rc = wgrad_tc_segment(g, s, &in[s], in_c[s], &dz, dz_c, 1, batch, h, w, cin_total, dw, &bias, st, det);
            if (rc != VSRB_OK) return rc;
        } else if (path == kWgradTaps) {
            for (int c0 = 0; c0 < g->seg_c[s]; c0 += 64)
                for (int n0 = 0; n0 < g->cout; n0 += 64) {
                    const int ci_n = g->seg_c[s] - c0 < 64 ? g->seg_c[s] - c0 : 64, co_n = g->cout - n0 < 64 ? g->cout - n0 : 64;
                    int rc = launch_wgrad_taps(in[s], in_c[s], c0, ci_n, g->seg_off[s] + c0, dz, dz_c, n0, co_n, g->kw, batch, h, w, cin_total,
                                               dw, st, det);
                    if (rc != VSRB_OK) return rc;
                }
        }
    }
    if (bias) {
        int rc = launch_bias_grad(dz, dz_c, (long long)batch * h * w, g->cout, g->dtype, bias, st, det);
        if (rc != VSRB_OK) return rc;
    }
    if (P.n_ci_blk == 0) return VSRB_OK;
    // every FFMA segment in one launch
    P.dz = dz; P.dz_c = dz_c;
    P.kh = g->kh; P.kw = g->kw; P.H = h; P.W = w;
    P.cout = g->cout; P.cin_total = cin_total;
    P.n_co_blk = ceil_div(g->cout, 64);
    P.dw = dw;
    P.chunks_per_row = ceil_div(w, 32);
    P.units = batch * h * P.chunks_per_row;
    // ~6 waves of the 148 SMs, at least 16 chunks (512 pixels) per CTA to amortise the final atomics
    const int other = g->kh * P.n_co_blk * P.n_ci_blk;
    const int ctas = (148 * 6 + other - 1) / other;
    int per = (P.units + ctas - 1) / ctas;
    if (per < 16) per = 16;
    P.units_per_cta = per;
    const dim3 grid((unsigned)ceil_div(P.units, per), g->kh, P.n_co_blk * P.n_ci_blk);
    using Kern = void (*)(WgradParams);
    const Kern kern = g->dtype == VSRB_BF16
        ? (g->kw == 1 ? conv_wgrad_kernel<__nv_bfloat16, 1> : g->kw == 3 ? conv_wgrad_kernel<__nv_bfloat16, 3> : conv_wgrad_kernel<__nv_bfloat16, 7>)
        : (g->kw == 1 ? conv_wgrad_kernel<float, 1> : g->kw == 3 ? conv_wgrad_kernel<float, 3> : conv_wgrad_kernel<float, 7>);
    kern<<<grid, 256, 0, st>>>(P);
    VSRB_LAUNCH_CHECK();
    return VSRB_OK;
}
}  // namespace vsrb

extern "C" {

int vsrb_flow_warp_bwd(const void* x, const float* flow, const void* dout, float* dx, float* dflow, int32_t n, int32_t h,
                       int32_t w, int32_t c, int32_t dtype, int32_t padding_mode, void* stream) {
    VSRB_CHECK_ARG(flow && dout && (dx || dflow) && n >= 1 && h >= 1 && w >= 1, "flow_warp_bwd: bad arguments");
    VSRB_CHECK_ARG(!dflow || x, "flow_warp_bwd: the flow gradient needs the forward input x");
    VSRB_CHECK_ARG((long long)n * h * w * c < (1LL << 40), "flow_warp_bwd: tensor too large");
    cudaStream_t s = (cudaStream_t)stream;
    int rc;
    if (dtype == VSRB_BF16) {
        VSRB_CHECK_ARG(c % 8 == 0, "flow_warp_bwd: bf16 needs c %% 8 == 0");
        rc = launch_warp_bwd<__nv_bfloat16>(reinterpret_cast<const __nv_bfloat16*>(x), reinterpret_cast<const float2*>(flow),
                                            reinterpret_cast<const __nv_bfloat16*>(dout), dx, reinterpret_cast<float2*>(dflow), n, h,
                                            w, c, padding_mode, s);
    } else {
        VSRB_CHECK_ARG(c % 4 == 0, "flow_warp_bwd: fp32 needs c %% 4 == 0");
        rc = launch_warp_bwd<float>(reinterpret_cast<const float*>(x), reinterpret_cast<const float2*>(flow),
                                    reinterpret_cast<const float*>(dout), dx, reinterpret_cast<float2*>(dflow), n, h, w, c,
                                    padding_mode, s);
    }
    if (rc != VSRB_OK) return rc;
    VSRB_LAUNCH_CHECK();
    return VSRB_OK;
}

size_t vsrb_flow_warp_bwd_det_workspace_bytes(int32_t n, int32_t h, int32_t w, int32_t c) {
    if (n < 1 || h < 1 || w < 1 || c < 1 || (long long)n * h * w * c >= (1LL << 40)) {
        set_error("flow_warp_bwd_det_workspace_bytes: bad shape");
        return 0;
    }
    return warp_bwd_det_bytes(n, h, w, c);
}

int vsrb_flow_warp_bwd_det(const void* x, const float* flow, const void* dout, float* dx, float* dflow, int32_t n, int32_t h,
                           int32_t w, int32_t c, int32_t dtype, int32_t padding_mode, void* workspace, size_t workspace_bytes,
                           void* stream) {
    VSRB_CHECK_ARG(flow && dout && (dx || dflow) && n >= 1 && h >= 1 && w >= 1 && c >= 1, "flow_warp_bwd_det: bad arguments");
    VSRB_CHECK_ARG(!dflow || x, "flow_warp_bwd_det: the flow gradient needs the forward input x");
    VSRB_CHECK_ARG((long long)n * h * w * c < (1LL << 40) && (long long)h * w < (1LL << 30), "flow_warp_bwd_det: tensor too large");
    VSRB_CHECK_ARG(dtype == VSRB_BF16 || dtype == VSRB_F32, "flow_warp_bwd_det: dtype must be bf16 or fp32 (got %d)", dtype);
    VSRB_CHECK_ARG(padding_mode == VSRB_PAD_ZEROS || padding_mode == VSRB_PAD_BORDER,
                   "flow_warp_bwd_det: padding_mode must be zeros (0) or border (1), got %d", padding_mode);
    const int vec = dtype == VSRB_BF16 ? 8 : 4, tpp = c / vec;
    VSRB_CHECK_ARG(c % vec == 0, "flow_warp_bwd_det: %s needs c %% %d == 0 (got %d)", dtype == VSRB_BF16 ? "bf16" : "fp32", vec, c);
    // the flow gradient is single-writer when a pixel's lanes form a power-of-two group inside a warp (see launch_warp_bwd)
    VSRB_CHECK_ARG(!dflow || (tpp <= 32 && (tpp & (tpp - 1)) == 0),
                   "flow_warp_bwd_det: the flow gradient needs c / %d to be a power of two <= 32 (got c = %d)", vec, c);
    VSRB_CHECK_ARG(!dx || (workspace && (reinterpret_cast<uintptr_t>(workspace) & 15) == 0 &&
                           workspace_bytes >= warp_bwd_det_bytes(n, h, w, c)),
                   "flow_warp_bwd_det: dx needs a 16-byte aligned workspace of %zu bytes (got %zu)", warp_bwd_det_bytes(n, h, w, c),
                   workspace_bytes);
    cudaStream_t s = (cudaStream_t)stream;
    const float2* fl = reinterpret_cast<const float2*>(flow);
    int rc = VSRB_OK;
    if (dtype == VSRB_BF16) {
        const __nv_bfloat16 *xb = reinterpret_cast<const __nv_bfloat16*>(x), *db = reinterpret_cast<const __nv_bfloat16*>(dout);
        if (dflow) rc = launch_warp_bwd<__nv_bfloat16>(xb, fl, db, nullptr, reinterpret_cast<float2*>(dflow), n, h, w, c, padding_mode, s);
        if (rc == VSRB_OK && dx) rc = launch_warp_bwd_dx_det<__nv_bfloat16>(fl, db, dx, n, h, w, c, padding_mode, workspace, s);
    } else {
        const float *xf = reinterpret_cast<const float*>(x), *df = reinterpret_cast<const float*>(dout);
        if (dflow) rc = launch_warp_bwd<float>(xf, fl, df, nullptr, reinterpret_cast<float2*>(dflow), n, h, w, c, padding_mode, s);
        if (rc == VSRB_OK && dx) rc = launch_warp_bwd_dx_det<float>(fl, df, dx, n, h, w, c, padding_mode, workspace, s);
    }
    if (rc != VSRB_OK) return rc;
    VSRB_LAUNCH_CHECK();
    return VSRB_OK;
}

int vsrb_flow_warp_ex_bwd(const void* x, const float* flow, const void* dout, float* dx, float* dflow, int32_t n, int32_t h,
                          int32_t w, int32_t c, int32_t dtype, int32_t interp, int32_t padding_mode, int32_t align_corners,
                          void* stream) {
    VSRB_CHECK_ARG(flow && dout && (dx || dflow) && n >= 1 && h >= 1 && w >= 1, "flow_warp_ex_bwd: bad arguments");
    VSRB_CHECK_ARG(!dflow || x, "flow_warp_ex_bwd: the flow gradient needs the forward input x");
    VSRB_CHECK_ARG(interp == VSRB_INTERP_BILINEAR || interp == VSRB_INTERP_NEAREST || interp == VSRB_INTERP_BICUBIC,
                   "flow_warp_ex_bwd: bad interpolation mode %d (bilinear 0, nearest 1, bicubic 2)", interp);
    VSRB_CHECK_ARG(padding_mode == VSRB_PAD_ZEROS || padding_mode == VSRB_PAD_BORDER || padding_mode == VSRB_PAD_REFLECTION,
                   "flow_warp_ex_bwd: bad padding mode %d (zeros 0, border 1, reflection 2)", padding_mode);
    VSRB_CHECK_ARG(align_corners == 0 || align_corners == 1, "flow_warp_ex_bwd: align_corners must be 0 or 1 (got %d)", align_corners);
    VSRB_CHECK_ARG(dtype == VSRB_BF16 || dtype == VSRB_F32, "flow_warp_ex_bwd: dtype must be bf16 or fp32 (got %d)", dtype);
    if (interp == VSRB_INTERP_BILINEAR && align_corners && padding_mode != VSRB_PAD_REFLECTION)
        return vsrb_flow_warp_bwd(x, flow, dout, dx, dflow, n, h, w, c, dtype, padding_mode, stream);
    VSRB_CHECK_ARG((long long)h * w < (1LL << 31) && (long long)n * h * w * c < (1LL << 40), "flow_warp_ex_bwd: tensor too large");
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == VSRB_BF16) {
        VSRB_CHECK_ARG(c >= 8 && c % 8 == 0, "flow_warp_ex_bwd: bf16 needs c %% 8 == 0 (got %d)", c);
        launch_warp_ex_bwd<__nv_bfloat16>(reinterpret_cast<const __nv_bfloat16*>(x), reinterpret_cast<const float2*>(flow),
                                          reinterpret_cast<const __nv_bfloat16*>(dout), dx, reinterpret_cast<float2*>(dflow), n, h, w,
                                          c, interp, padding_mode, align_corners, s);
    } else {
        VSRB_CHECK_ARG(c >= 4 && c % 4 == 0, "flow_warp_ex_bwd: fp32 needs c %% 4 == 0 (got %d)", c);
        launch_warp_ex_bwd<float>(reinterpret_cast<const float*>(x), reinterpret_cast<const float2*>(flow),
                                  reinterpret_cast<const float*>(dout), dx, reinterpret_cast<float2*>(dflow), n, h, w, c, interp,
                                  padding_mode, align_corners, s);
    }
    VSRB_LAUNCH_CHECK();
    return VSRB_OK;
}

}  // extern "C"
