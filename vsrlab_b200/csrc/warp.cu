// Memory-bound resampling kernels: backward warp (flow_warp), layout changes, SPyNet glue.
// All activations NHWC; every gather is a 16-byte vector of consecutive channels.
#include "common.cuh"
#include "warp_modes.cuh"

namespace vsrb {

// ---------------------------------------------------------------------------------------
// flow_warp  (reference spynet.py:95-106)
//
// A CTA owns 256 consecutive pixels.  Phase 1: the 256 flow vectors are read with one
// coalesced float2 load per thread and turned, ONCE per pixel, into four tap offsets and
// four bilinear weights that are staged in shared memory.  Phase 2: C/VEC threads per pixel
// each gather four 16-byte channel vectors (coalesced: the C/VEC threads of a pixel read one
// contiguous C*sizeof(T) run per tap), blend in fp32 and store one 16-byte vector.
// Algorithmic traffic: C*sizeof(T) read + 8 B flow + C*sizeof(T) written per pixel.
// ---------------------------------------------------------------------------------------
struct TapSet {
    int off[4];     // pixel index of the tap inside the image, or -1 when it contributes zero
    float wgt[4];
};

__device__ __forceinline__ void sample_pos(float px, float py, int w, int h, float& ix, float& iy) {
    // the reference normalises to [-1,1] and grid_sample(align_corners=True) maps back
    float nx = 2.0f * px / (float)max(w - 1, 1) - 1.0f;
    float ny = 2.0f * py / (float)max(h - 1, 1) - 1.0f;
    ix = (nx + 1.0f) / 2.0f * (float)(w - 1);
    iy = (ny + 1.0f) / 2.0f * (float)(h - 1);
}

__device__ __forceinline__ void make_taps(float ix, float iy, int w, int h, int border, TapSet& t) {
    if (border) {
        ix = fminf(fmaxf(ix, 0.f), (float)(w - 1));
        iy = fminf(fmaxf(iy, 0.f), (float)(h - 1));
    }
    float fx = floorf(ix), fy = floorf(iy);
    float wx1 = ix - fx, wy1 = iy - fy, wx0 = 1.f - wx1, wy0 = 1.f - wy1;
    // guard the float->int conversion for wild flows
    fx = fminf(fmaxf(fx, -2.f), (float)w);
    fy = fminf(fmaxf(fy, -2.f), (float)h);
    int x0 = (int)fx, y0 = (int)fy;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        int xi = x0 + (k & 1), yi = y0 + (k >> 1);
        bool ok = xi >= 0 && xi < w && yi >= 0 && yi < h;
        t.off[k] = ok ? yi * w + xi : -1;
        t.wgt[k] = ((k & 1) ? wx1 : wx0) * ((k >> 1) ? wy1 : wy0);
    }
}

template <typename T> struct Vec16;
template <> struct Vec16<__nv_bfloat16> {
    static constexpr int N = 8;
    __device__ static void load(const __nv_bfloat16* p, float (&v)[8]) {
        uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
        float2 a = unpack_bf16(u.x), b = unpack_bf16(u.y), c = unpack_bf16(u.z), d = unpack_bf16(u.w);
        v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; v[4] = c.x; v[5] = c.y; v[6] = d.x; v[7] = d.y;
    }
    __device__ static void store(__nv_bfloat16* p, const float (&v)[8]) {
        uint4 u;
        u.x = pack_bf16(v[0], v[1]); u.y = pack_bf16(v[2], v[3]);
        u.z = pack_bf16(v[4], v[5]); u.w = pack_bf16(v[6], v[7]);
        *reinterpret_cast<uint4*>(p) = u;
    }
};
template <> struct Vec16<float> {
    static constexpr int N = 4;
    __device__ static void load(const float* p, float (&v)[4]) {
        float4 f = __ldg(reinterpret_cast<const float4*>(p));
        v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
    }
    __device__ static void store(float* p, const float (&v)[4]) {
        *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    }
};

static constexpr int kWarpPix = 256;

struct WarpTap {
    long long base;   // element offset of the pixel's image inside x
    TapSet t;
};

// TPP = 16-byte vectors per pixel (C / VEC); a power of two here so the work split is shifts only
// kSplit (bf16 only): the tensor is split-bf16 [hi C | lo C] per pixel (value = hi + lo); taps are blended on
// the fp32 sum and the result is split again, so the warp keeps fp32-level accuracy.  tpp counts C / 8.
template <typename T, int TPP, bool kSplit = false>
__global__ void __launch_bounds__(256) flow_warp_kernel(const T* __restrict__ x, long long x_stride,
                                                        const float2* __restrict__ flow, long long f_stride,
                                                        T* __restrict__ out, int n, int h, int w, int border, int tpp_rt,
                                                        int ipg = 0x7fffffff, long long x_gstride = 0, long long f_gstride = 0) {
    __shared__ WarpTap taps[kWarpPix];
    constexpr int VEC = Vec16<T>::N;
    const int tpp = TPP > 0 ? TPP : tpp_rt;            // TPP == 0: any channel count (runtime divisions)
    const int half = tpp * VEC;                        // channels of one half when kSplit
    const int C = kSplit ? 2 * half : half;
    const int hw = h * w;
    const int total = n * hw;                          // launcher guarantees < 2^31
    const int pix0 = blockIdx.x * kWarpPix;
    {
        const int pix = pix0 + threadIdx.x;
        if (pix < total) {
            const int img = pix / hw, r = pix - img * hw;
            const int yy = r / w, xx = r - yy * w;
            // images come in groups of `ipg` (the two propagation directions read different frames of the feature bank
            // and different flow fields): image = group * ipg + li
            const int grp = img / ipg, li = img - grp * ipg;
            const float2 f = __ldg(flow + (long long)grp * f_gstride + (long long)li * f_stride + r);
            float ix, iy;
            sample_pos((float)xx + f.x, (float)yy + f.y, w, h, ix, iy);
            make_taps(ix, iy, w, h, border, taps[threadIdx.x].t);
            taps[threadIdx.x].base = (long long)grp * x_gstride + (long long)li * x_stride;
        }
    }
    __syncthreads();
    const int npix = min(kWarpPix, total - pix0);
    const int work = npix * tpp;
#pragma unroll 4
    for (int i = threadIdx.x; i < work; i += 256) {
        const int lp = i / tpp, part = i % tpp;          // compile-time power of two: shift / mask
        const WarpTap wt = taps[lp];
        const T* img = x + wt.base + part * VEC;
        float acc[VEC];
#pragma unroll
        for (int j = 0; j < VEC; ++j) acc[j] = 0.f;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (wt.t.off[k] >= 0) {
                float v[VEC];
                Vec16<T>::load(img + (long long)wt.t.off[k] * C, v);
                if (kSplit) {
                    float lo[VEC];
                    Vec16<T>::load(img + (long long)wt.t.off[k] * C + half, lo);
#pragma unroll
                    for (int j = 0; j < VEC; ++j) v[j] += lo[j];
                }
#pragma unroll
                for (int j = 0; j < VEC; ++j) acc[j] = fmaf(v[j], wt.t.wgt[k], acc[j]);
            }
        }
        if (kSplit) {
            float hi[VEC], lo[VEC];
#pragma unroll
            for (int j = 0; j < VEC; ++j) {
                hi[j] = (float)(T)acc[j];
                lo[j] = acc[j] - hi[j];
            }
            Vec16<T>::store(out + (long long)(pix0 + lp) * C + part * VEC, hi);
            Vec16<T>::store(out + (long long)(pix0 + lp) * C + half + part * VEC, lo);
        } else {
            Vec16<T>::store(out + (long long)(pix0 + lp) * C + part * VEC, acc);
        }
    }
}

template <typename T>
static int launch_flow_warp(const T* x, long long xs, const float2* flow, long long fs, T* out, int n, int h, int w, int c,
                            int border, cudaStream_t s, int ipg = 0x7fffffff, long long xg = 0, long long fg = 0) {
    constexpr int VEC = Vec16<T>::N;
    const int tpp = c / VEC;
    const int blocks = (int)(((long long)n * h * w + kWarpPix - 1) / kWarpPix);
    switch (tpp) {
        case 1: flow_warp_kernel<T, 1><<<blocks, 256, 0, s>>>(x, xs, flow, fs, out, n, h, w, border, tpp, ipg, xg, fg); break;
        case 2: flow_warp_kernel<T, 2><<<blocks, 256, 0, s>>>(x, xs, flow, fs, out, n, h, w, border, tpp, ipg, xg, fg); break;
        case 4: flow_warp_kernel<T, 4><<<blocks, 256, 0, s>>>(x, xs, flow, fs, out, n, h, w, border, tpp, ipg, xg, fg); break;
        case 8: flow_warp_kernel<T, 8><<<blocks, 256, 0, s>>>(x, xs, flow, fs, out, n, h, w, border, tpp, ipg, xg, fg); break;
        case 16: flow_warp_kernel<T, 16><<<blocks, 256, 0, s>>>(x, xs, flow, fs, out, n, h, w, border, tpp, ipg, xg, fg); break;
        case 32: flow_warp_kernel<T, 32><<<blocks, 256, 0, s>>>(x, xs, flow, fs, out, n, h, w, border, tpp, ipg, xg, fg); break;
        default: flow_warp_kernel<T, 0><<<blocks, 256, 0, s>>>(x, xs, flow, fs, out, n, h, w, border, tpp, ipg, xg, fg); break;
    }
    return VSRB_OK;
}

// ---------------------------------------------------------------------------------------
// flow_warp_ex: the other F.grid_sample modes (nearest / bicubic, reflection padding, align_corners=False).
// The structure of flow_warp_kernel: taps built once per pixel into shared memory, then C/VEC threads per pixel gather
// 16-byte channel vectors and blend in fp32.  nearest keeps one tap, bilinear four (a TapSet), bicubic a separable
// 4 + 4 table (column indices, row offsets, weights; -1 = reads zero) instead of 16 offsets.
// ---------------------------------------------------------------------------------------
struct NearestTap {
    int off;        // pixel index of the tap, or -1
};
struct BicubicTaps {
    int xo[4];      // column of tap floor(ix) - 1 + i after padding, or -1
    int yo[4];      // row offset (row * w) of tap floor(iy) - 1 + j after padding, or -1
    float wx[4], wy[4];
};
template <int kInterp> struct ExTapsOf { using type = TapSet; };
template <> struct ExTapsOf<VSRB_INTERP_NEAREST> { using type = NearestTap; };
template <> struct ExTapsOf<VSRB_INTERP_BICUBIC> { using type = BicubicTaps; };

__device__ __forceinline__ void make_taps_ex(float ix, float iy, int w, int h, int pad, int align, NearestTap& t) {
    float g;
    const int xi = ex_index(nearbyintf(ex_pad_coord(ix, w, pad, align, g)), w);     // round half to even
    const int yi = ex_index(nearbyintf(ex_pad_coord(iy, h, pad, align, g)), h);
    t.off = (xi >= 0 && yi >= 0) ? yi * w + xi : -1;
}
__device__ __forceinline__ void make_taps_ex(float ix, float iy, int w, int h, int pad, int align, TapSet& t) {
    float g;
    make_taps(ex_pad_coord(ix, w, pad, align, g), ex_pad_coord(iy, h, pad, align, g), w, h, 0, t);
}
__device__ __forceinline__ void make_taps_ex(float ix, float iy, int w, int h, int pad, int align, BicubicTaps& t) {
    const float fx = floorf(ix), fy = floorf(iy);
    cubic_weights(ix - fx, t.wx);
    cubic_weights(iy - fy, t.wy);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        t.xo[i] = ex_bicubic_tap(fx + (float)(i - 1), w, pad, align);
        const int yi = ex_bicubic_tap(fy + (float)(i - 1), h, pad, align);
        t.yo[i] = yi >= 0 ? yi * w : -1;
    }
}

template <typename T, int VEC>
__device__ __forceinline__ void gather_ex(const T* img, int C, const NearestTap& t, float (&acc)[VEC]) {
    if (t.off >= 0) Vec16<T>::load(img + (long long)t.off * C, acc);
}
template <typename T, int VEC>
__device__ __forceinline__ void gather_ex(const T* img, int C, const TapSet& t, float (&acc)[VEC]) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (t.off[k] >= 0) {
            float v[VEC];
            Vec16<T>::load(img + (long long)t.off[k] * C, v);
#pragma unroll
            for (int j = 0; j < VEC; ++j) acc[j] = fmaf(v[j], t.wgt[k], acc[j]);
        }
    }
}
template <typename T, int VEC>
__device__ __forceinline__ void gather_ex(const T* img, int C, const BicubicTaps& t, float (&acc)[VEC]) {
    // along x within each row, then across the rows (ATen's cubic_interp1d order)
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        if (t.yo[r] < 0) continue;
        float row[VEC];
#pragma unroll
        for (int j = 0; j < VEC; ++j) row[j] = 0.f;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            if (t.xo[q] < 0) continue;
            float v[VEC];
            Vec16<T>::load(img + (long long)(t.yo[r] + t.xo[q]) * C, v);
#pragma unroll
            for (int j = 0; j < VEC; ++j) row[j] = fmaf(v[j], t.wx[q], row[j]);
        }
#pragma unroll
        for (int j = 0; j < VEC; ++j) acc[j] = fmaf(row[j], t.wy[r], acc[j]);
    }
}

// (256, 1): under the plain (256) bound ptxas held the bf16 bicubic variants to 40 - 48 registers and spilled
template <typename T, int TPP, int kInterp>
__global__ void __launch_bounds__(256, 1) flow_warp_ex_kernel(const T* __restrict__ x, long long x_stride,
                                                           const float2* __restrict__ flow, long long f_stride,
                                                           T* __restrict__ out, int n, int h, int w, int pad, int align,
                                                           int tpp_rt) {
    using Taps = typename ExTapsOf<kInterp>::type;
    __shared__ Taps taps[kWarpPix];
    __shared__ long long bases[kWarpPix];
    constexpr int VEC = Vec16<T>::N;
    const int tpp = TPP > 0 ? TPP : tpp_rt;            // TPP == 0: any channel count (runtime divisions)
    const int C = tpp * VEC;
    const int hw = h * w;
    const int total = n * hw;                          // launcher guarantees < 2^31
    const int pix0 = blockIdx.x * kWarpPix;
    {
        const int pix = pix0 + threadIdx.x;
        if (pix < total) {
            const int img = pix / hw, r = pix - img * hw;
            const int yy = r / w, xx = r - yy * w;
            const float2 f = __ldg(flow + (long long)img * f_stride + r);
            make_taps_ex(ex_unnormalize((float)xx + f.x, w, align), ex_unnormalize((float)yy + f.y, h, align), w, h, pad, align,
                         taps[threadIdx.x]);
            bases[threadIdx.x] = (long long)img * x_stride;
        }
    }
    __syncthreads();
    const int npix = min(kWarpPix, total - pix0);
    const int work = npix * tpp;
    constexpr int kUnroll = kInterp == VSRB_INTERP_BICUBIC ? 1 : 4;     // bicubic: 16 loads in flight per item already
#pragma unroll kUnroll
    for (int i = threadIdx.x; i < work; i += 256) {
        const int lp = i / tpp, part = i % tpp;          // compile-time power of two: shift / mask
        float acc[VEC];
#pragma unroll
        for (int j = 0; j < VEC; ++j) acc[j] = 0.f;
        gather_ex<T, VEC>(x + bases[lp] + part * VEC, C, taps[lp], acc);       // the table is read from shared memory
        Vec16<T>::store(out + (long long)(pix0 + lp) * C + part * VEC, acc);
    }
}

template <typename T, int kInterp>
static void launch_flow_warp_ex_t(const T* x, long long xs, const float2* flow, long long fs, T* out, int n, int h, int w, int c,
                                  int pad, int align, cudaStream_t s) {
    constexpr int VEC = Vec16<T>::N;
    const int tpp = c / VEC;
    const int blocks = (int)(((long long)n * h * w + kWarpPix - 1) / kWarpPix);
#define VSRB_WARP_EX(TPP) flow_warp_ex_kernel<T, TPP, kInterp><<<blocks, 256, 0, s>>>(x, xs, flow, fs, out, n, h, w, pad, align, tpp)
    switch (tpp) {
        case 1: VSRB_WARP_EX(1); break;
        case 2: VSRB_WARP_EX(2); break;
        case 4: VSRB_WARP_EX(4); break;
        case 8: VSRB_WARP_EX(8); break;
        case 16: VSRB_WARP_EX(16); break;
        case 32: VSRB_WARP_EX(32); break;
        default: VSRB_WARP_EX(0); break;
    }
#undef VSRB_WARP_EX
}

template <typename T>
static void launch_flow_warp_ex(const T* x, long long xs, const float2* flow, long long fs, T* out, int n, int h, int w, int c,
                                int interp, int pad, int align, cudaStream_t s) {
    if (interp == VSRB_INTERP_NEAREST) launch_flow_warp_ex_t<T, VSRB_INTERP_NEAREST>(x, xs, flow, fs, out, n, h, w, c, pad, align, s);
    else if (interp == VSRB_INTERP_BICUBIC) launch_flow_warp_ex_t<T, VSRB_INTERP_BICUBIC>(x, xs, flow, fs, out, n, h, w, c, pad, align, s);
    else launch_flow_warp_ex_t<T, VSRB_INTERP_BILINEAR>(x, xs, flow, fs, out, n, h, w, c, pad, align, s);
}

// ---------------------------------------------------------------------------------------
// layout
// ---------------------------------------------------------------------------------------
template <typename T>
__global__ void nchw_to_nhwc_kernel(const float* __restrict__ src, T* __restrict__ dst, int n, int c, int h, int w, int c_dst) {
    const long long plane = (long long)h * w;
    const long long total = (long long)n * plane;
    for (long long pix = (long long)blockIdx.x * blockDim.x + threadIdx.x; pix < total;
         pix += (long long)gridDim.x * blockDim.x) {
        const long long img = pix / plane, r = pix - img * plane;
        const float* sp = src + img * c * plane + r;
        T* dp = dst + pix * c_dst;
        for (int k = 0; k < c_dst; ++k) {
            float v = k < c ? __ldg(sp + k * plane) : 0.f;
            dp[k] = (T)v;
        }
    }
}

// the model's entry layout (3-channel frames -> 16-channel bf16 pixels): two 16-byte stores per pixel instead of sixteen
// 2-byte ones (0.27 ms -> ~0.04 ms for 60 frames of 180 x 320)
__global__ void nchw_to_nhwc16_bf16_kernel(const float* __restrict__ src, uint4* __restrict__ dst, int n, int c, int h, int w) {
    const long long plane = (long long)h * w;
    const long long total = (long long)n * plane;
    for (long long pix = (long long)blockIdx.x * blockDim.x + threadIdx.x; pix < total;
         pix += (long long)gridDim.x * blockDim.x) {
        const long long img = pix / plane, r = pix - img * plane;
        const float* sp = src + img * c * plane + r;
        float v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = k < c ? __ldg(sp + k * plane) : 0.f;
        dst[2 * pix] = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
        dst[2 * pix + 1] = make_uint4(0u, 0u, 0u, 0u);
    }
}

// split-bf16: channels [0, c_dst/2) hold hi = bf16(v), channels [c_dst/2, c_dst) hold lo = bf16(v - hi)
__global__ void nchw_to_nhwc_split_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int n, int c, int h, int w,
                                          int c_dst) {
    const long long plane = (long long)h * w;
    const long long total = (long long)n * plane;
    const int half = c_dst / 2;
    for (long long pix = (long long)blockIdx.x * blockDim.x + threadIdx.x; pix < total;
         pix += (long long)gridDim.x * blockDim.x) {
        const long long img = pix / plane, r = pix - img * plane;
        const float* sp = src + img * c * plane + r;
        __nv_bfloat16* dp = dst + pix * c_dst;
        for (int k = 0; k < half; ++k) {
            const float v = k < c ? __ldg(sp + k * plane) : 0.f;
            const __nv_bfloat16 hi = __float2bfloat16_rn(v);
            dp[k] = hi;
            dp[half + k] = __float2bfloat16_rn(v - __bfloat162float(hi));
        }
    }
}

__global__ void nhwc_split_to_nchw_kernel(const __nv_bfloat16* __restrict__ src, float* __restrict__ dst, int n, int c, int h, int w,
                                          int c_src) {
    const long long plane = (long long)h * w;
    const long long total = (long long)n * c * plane;
    const int half = c_src / 2;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long r = i % plane;
        const long long nc = i / plane;
        const int k = (int)(nc % c);
        const long long img = nc / c;
        const __nv_bfloat16* p = src + (img * plane + r) * c_src;
        dst[i] = __bfloat162float(p[k]) + __bfloat162float(p[half + k]);
    }
}

template <typename T>
__global__ void nhwc_to_nchw_kernel(const T* __restrict__ src, float* __restrict__ dst, int n, int c, int h, int w, int c_src) {
    const long long plane = (long long)h * w;
    const long long total = (long long)n * c * plane;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long r = i % plane;
        const long long nc = i / plane;
        const int k = (int)(nc % c);
        const long long img = nc / c;
        dst[i] = (float)src[(img * plane + r) * c_src + k];
    }
}

// ---------------------------------------------------------------------------------------
// SPyNet glue
// ---------------------------------------------------------------------------------------
__global__ void pyramid_base_kernel(const float* __restrict__ frames, float4* __restrict__ lvl, int F, int h, int w, int Hp,
                                    int Wp, float m0, float m1, float m2, float s0, float s1, float s2) {
    const long long total = (long long)F * Hp * Wp;
    const float sy = (float)h / (float)Hp, sx = (float)w / (float)Wp;
    const long long plane = (long long)h * w;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int X = (int)(i % Wp), Y = (int)((i / Wp) % Hp);
        const long long f = i / ((long long)Wp * Hp);
        int y0, y1, x0, x1;
        float ly, lx;
        up_tap(Y, sy, h, y0, y1, ly);
        up_tap(X, sx, w, x0, x1, lx);
        const float hy = 1.f - ly, hx = 1.f - lx;
        float v[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float* p = frames + (f * 3 + c) * plane;
            float a00 = __ldg(p + y0 * w + x0), a01 = __ldg(p + y0 * w + x1);
            float a10 = __ldg(p + y1 * w + x0), a11 = __ldg(p + y1 * w + x1);
            v[c] = hy * (hx * a00 + lx * a01) + ly * (hx * a10 + lx * a11);
        }
        lvl[i] = make_float4((v[0] - m0) / s0, (v[1] - m1) / s1, (v[2] - m2) / s2, 0.f);
    }
}

__global__ void avgpool2_c4_kernel(const float4* __restrict__ in, float4* __restrict__ out, int F, int H, int W) {
    const int Ho = H / 2, Wo = W / 2;
    const long long total = (long long)F * Ho * Wo;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int X = (int)(i % Wo), Y = (int)((i / Wo) % Ho);
        const long long f = i / ((long long)Wo * Ho);
        const float4* p = in + (f * H + 2 * Y) * W + 2 * X;
        float4 a = __ldg(p), b = __ldg(p + 1), c = __ldg(p + W), d = __ldg(p + W + 1);
        out[i] = make_float4((((a.x + b.x) + c.x) + d.x) * 0.25f, (((a.y + b.y) + c.y) + d.y) * 0.25f,
                             (((a.z + b.z) + c.z) + d.z) * 0.25f, 0.f);
    }
}

// ATen upsample_bilinear2d(align_corners=True) source tap for one axis
__device__ __forceinline__ void up_tap_ac(int dst, int in_size, int out_size, int& i0, int& i1, float& l1) {
    const float scale = out_size > 1 ? (float)(in_size - 1) / (float)(out_size - 1) : 0.f;
    const float src = scale * (float)dst;
    i0 = (int)src;
    if (i0 > in_size - 1) i0 = in_size - 1;
    i1 = i0 + (i0 < in_size - 1 ? 1 : 0);
    l1 = src - (float)i0;
}

template <typename T>
__global__ void level_input_kernel(const float4* __restrict__ lvl, const int* __restrict__ ref_idx,
                                   const int* __restrict__ supp_idx, const float2* __restrict__ flow_prev,
                                   float2* __restrict__ flow_up, T* __restrict__ conv_in, int P, int Hl, int Wl, int c_in,
                                   int split) {
    const long long plane = (long long)Hl * Wl;
    const long long total = (long long)P * plane;
    const int Hi = Hl / 2, Wi = Wl / 2;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int X = (int)(i % Wl), Y = (int)((i / Wl) % Hl);
        const int p = (int)(i / plane);
        float2 fu = make_float2(0.f, 0.f);
        if (flow_prev) {
            int y0, y1, x0, x1;
            float ly, lx;
            up_tap_ac(Y, Hi, Hl, y0, y1, ly);
            up_tap_ac(X, Wi, Wl, x0, x1, lx);
            const float hy = 1.f - ly, hx = 1.f - lx;
            const float2* fp = flow_prev + (long long)p * Hi * Wi;
            float2 a00 = __ldg(fp + y0 * Wi + x0), a01 = __ldg(fp + y0 * Wi + x1);
            float2 a10 = __ldg(fp + y1 * Wi + x0), a11 = __ldg(fp + y1 * Wi + x1);
            fu.x = (hy * (hx * a00.x + lx * a01.x) + ly * (hx * a10.x + lx * a11.x)) * 2.0f;
            fu.y = (hy * (hx * a00.y + lx * a01.y) + ly * (hx * a10.y + lx * a11.y)) * 2.0f;
        }
        flow_up[i] = fu;
        float ix, iy;
        sample_pos((float)X + fu.x, (float)Y + fu.y, Wl, Hl, ix, iy);
        TapSet t;
        make_taps(ix, iy, Wl, Hl, 1, t);
        const float4* sp = lvl + (long long)__ldg(supp_idx + p) * plane;
        float wr = 0.f, wg = 0.f, wb = 0.f;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (t.off[k] >= 0) {
                float4 v = __ldg(sp + t.off[k]);
                wr = fmaf(v.x, t.wgt[k], wr);
                wg = fmaf(v.y, t.wgt[k], wg);
                wb = fmaf(v.z, t.wgt[k], wb);
            }
        }
        const float4 r = __ldg(lvl + (long long)__ldg(ref_idx + p) * plane + (long long)Y * Wl + X);
        float v[16] = {r.x, r.y, r.z, wr, wg, wb, fu.x, fu.y, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        T* op = conv_in + i * c_in;
        if (split) {                                   // [hi 16 | lo 16]
            float hi[16], lo[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                hi[k] = (float)(T)v[k];
                lo[k] = v[k] - hi[k];
            }
            Act<T>::store16(op, hi);
            Act<T>::store16(op + 16, lo);
        } else if (c_in == 16) Act<T>::store16(op, v);
        else {
            for (int k = 0; k < c_in; ++k) op[k] = (T)(k < 8 ? v[k] : 0.f);
        }
    }
}

__global__ void flow_resize_kernel(const float2* __restrict__ fin, float2* __restrict__ fout, int P, int Hp, int Wp, int h,
                                   int w) {
    const long long total = (long long)P * h * w;
    const float sy = (float)Hp / (float)h, sx = (float)Wp / (float)w;
    const float rx = (float)((double)w / (double)Wp), ry = (float)((double)h / (double)Hp);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int X = (int)(i % w), Y = (int)((i / w) % h);
        const long long p = i / ((long long)w * h);
        int y0, y1, x0, x1;
        float ly, lx;
        up_tap(Y, sy, Hp, y0, y1, ly);
        up_tap(X, sx, Wp, x0, x1, lx);
        const float hy = 1.f - ly, hx = 1.f - lx;
        const float2* fp = fin + p * Hp * Wp;
        float2 a00 = __ldg(fp + y0 * Wp + x0), a01 = __ldg(fp + y0 * Wp + x1);
        float2 a10 = __ldg(fp + y1 * Wp + x0), a11 = __ldg(fp + y1 * Wp + x1);
        float vx = hy * (hx * a00.x + lx * a01.x) + ly * (hx * a10.x + lx * a11.x);
        float vy = hy * (hx * a00.y + lx * a01.y) + ly * (hx * a10.y + lx * a11.y);
        fout[i] = make_float2(vx * rx, vy * ry);
    }
}

static inline int grid_for(long long total, int block) {
    long long b = (total + block - 1) / block;
    if (b > 148 * 32) b = 148 * 32;
    if (b < 1) b = 1;
    return (int)b;
}

}  // namespace vsrb

using namespace vsrb;

// Inverse of PixelShuffle(2) on bf16 NHWC (training: the gradient of an upsampling conv arrives in the shuffled layout):
// dst[b][y][x][4c + 2i + j] = src[b][2y + i][2x + j][c].  A thread owns 8 consecutive source channels of one LR pixel:
// four 16-byte loads (the 2 x 2 HR pixels), four 16-byte stores (32 consecutive destination channels).  HBM-bound.
__global__ void pixel_unshuffle2_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, long long lr_pixels, int w, int c) {
    const int groups = c / 8;
    const long long total = lr_pixels * groups;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int g = (int)(i % groups);
        const long long p = i / groups;                       // b * h * w + y * w + x
        const int x = (int)(p % w);
        const long long by = p / w;                           // b * h + y
        uint32_t q[4][4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {                         // k = 2i + j
            const long long sp = (2 * by + (k >> 1)) * (2LL * w) + 2 * x + (k & 1);
            const uint4 v = __ldg(src + sp * groups + g);
            q[k][0] = v.x; q[k][1] = v.y; q[k][2] = v.z; q[k][3] = v.w;
        }
        // source channel e (0..7) of sub-pixel k goes to destination channel 4 * (8g + e) + k
        uint32_t o[16];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const uint32_t sh = (e & 1) * 16;
            const uint32_t v0 = (q[0][e >> 1] >> sh) & 0xFFFFu, v1 = (q[1][e >> 1] >> sh) & 0xFFFFu;
            const uint32_t v2 = (q[2][e >> 1] >> sh) & 0xFFFFu, v3 = (q[3][e >> 1] >> sh) & 0xFFFFu;
            o[2 * e] = v0 | (v1 << 16);
            o[2 * e + 1] = v2 | (v3 << 16);
        }
        uint4* d = dst + (p * (4LL * groups) + 4LL * g);
#pragma unroll
        for (int k = 0; k < 4; ++k) d[k] = make_uint4(o[4 * k], o[4 * k + 1], o[4 * k + 2], o[4 * k + 3]);
    }
}

namespace vsrb {
// 3x3 im2col of 3-channel frames: one thread per (pixel, 16-byte quarter of its 64-byte patch row): eight of the 27
// neighbourhood values (+ 5 zeros at the end), so a warp's stores are 512 consecutive bytes.  blockIdx.x = image row
// (img * h + y), threads run along the row: 32-bit index arithmetic, no divisions by w / h per element (the first version
// spent most of its 235 us per 60 frames on three 64-bit div / mod per thread), neighbouring pixels' loads hit in L1.
__global__ void __launch_bounds__(256) im2col3x3_c3_kernel(const float* __restrict__ src, uint4* __restrict__ dst, int h, int w) {
    const int row = blockIdx.x;                         // img * h + y
    const int img = row / h, y = row - img * h;
    const int plane = h * w;
    const float* fp = src + (size_t)img * 3 * plane;
    uint4* out = dst + (size_t)row * w * 4;
    for (int i = blockIdx.y * blockDim.x + threadIdx.x; i < 4 * w; i += gridDim.y * blockDim.x) {
        const int j = i & 3, x = i >> 2;
        float v[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int k = 8 * j + e, tap = k / 3, c = k - tap * 3;          // (j and e are small: constant-folded per j)
            const int yy = y + tap / 3 - 1, xx = x + tap % 3 - 1;
            v[e] = (k < 27 && yy >= 0 && yy < h && xx >= 0 && xx < w) ? __ldg(fp + c * plane + yy * w + xx) : 0.f;
        }
        out[i] = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
    }
}
// The same through shared memory: a block stages the three input rows of its image row (3 channels x 3 rows x (w + 2)
// floats, zero padded, coalesced loads) and builds the patches from there - the direct kernel's eight scattered 4-byte
// loads per thread kept it at 1.4 TB/s; this one is bound by its 64 bytes of output per pixel.
__global__ void __launch_bounds__(256) im2col3x3_c3_smem_kernel(const float* __restrict__ src, uint4* __restrict__ dst, int h, int w) {
    extern __shared__ float rows_s[];                   // [c * 3 + dy][w + 2]
    const int row = blockIdx.x;
    const int img = row / h, y = row - img * h;
    const int plane = h * w, pitch = w + 2;
    const float* fp = src + (size_t)img * 3 * plane;
#pragma unroll
    for (int r = 0; r < 9; ++r) {                       // (no division per element: the first version of this kernel was instruction bound)
        const int c = r / 3, yy = y + (r - c * 3) - 1;
        const bool row_ok = yy >= 0 && yy < h;
        const float* rp = fp + c * plane + yy * w;
        for (int xs = threadIdx.x; xs < pitch; xs += blockDim.x) {
            const int xx = xs - 1;
            rows_s[r * pitch + xs] = (row_ok && xx >= 0 && xx < w) ? __ldg(rp + xx) : 0.f;
        }
    }
    __syncthreads();
    uint4* out = dst + (size_t)row * w * 4;
    // one thread per pixel: its 27 values sit at compile-time offsets, the 64-byte patch row leaves as four 16-byte stores
    for (int x = threadIdx.x; x < w; x += blockDim.x) {
        float v[32];
#pragma unroll
        for (int k = 0; k < 32; ++k) {
            const int tap = k / 3, c = k - tap * 3;
            v[k] = k < 27 ? rows_s[(c * 3 + tap / 3) * pitch + x + tap % 3] : 0.f;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)
            out[x * 4 + j] = make_uint4(pack_bf16(v[8 * j], v[8 * j + 1]), pack_bf16(v[8 * j + 2], v[8 * j + 3]),
                                        pack_bf16(v[8 * j + 4], v[8 * j + 5]), pack_bf16(v[8 * j + 6], v[8 * j + 7]));
    }
}
}  // namespace vsrb

extern "C" {

int vsrb_im2col3x3_c3(const float* frames, void* patches, int32_t n, int32_t h, int32_t w, void* stream) {
    VSRB_CHECK_ARG(frames && patches && n >= 1 && h >= 1 && w >= 1, "im2col3x3_c3: bad arguments");
    VSRB_CHECK_ARG((reinterpret_cast<uintptr_t>(patches) & 15) == 0, "im2col3x3_c3: output must be 16-byte aligned");
    const long long rows = (long long)n * h;
    VSRB_CHECK_ARG((long long)h * w * 3 < (1LL << 31) && rows <= 0x7fffffffLL && w <= (1 << 22), "im2col3x3_c3: image too large");
    const size_t smem = (size_t)9 * (w + 2) * sizeof(float);
    if (smem <= 48 * 1024) {                            // rows up to 1 363 pixels: no opt-in needed
        vsrb::im2col3x3_c3_smem_kernel<<<(unsigned)rows, 256, smem, (cudaStream_t)stream>>>(frames, reinterpret_cast<uint4*>(patches), h, w);
    } else {
        unsigned gy = (unsigned)((4 * w + 255) / 256);
        if (gy > 65535u) gy = 65535u;
        dim3 grid((unsigned)rows, gy);
        vsrb::im2col3x3_c3_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(frames, reinterpret_cast<uint4*>(patches), h, w);
    }
    VSRB_LAUNCH_CHECK();
    return VSRB_OK;
}

int vsrb_flow_warp(const void* x, int64_t x_img_stride, const float* flow, int64_t flow_img_stride, void* out, int32_t n,
                   int32_t h, int32_t w, int32_t c, int32_t dtype, int32_t padding_mode, void* stream) {
    const long long xs = x_img_stride ? x_img_stride : (long long)h * w * c;
    const long long fs = flow_img_stride ? flow_img_stride : (long long)h * w;
    VSRB_CHECK_ARG(x && flow && out && n >= 1 && h >= 1 && w >= 1, "flow_warp: bad arguments");
    VSRB_CHECK_ARG(padding_mode == VSRB_PAD_ZEROS || padding_mode == VSRB_PAD_BORDER, "flow_warp: bad padding mode");
    VSRB_CHECK_ARG((long long)h * w < (1LL << 31), "flow_warp: image too large");
    VSRB_CHECK_ARG((long long)n * h * w < (1LL << 31), "flow_warp: more than 2^31 pixels in one call");
    cudaStream_t s = (cudaStream_t)stream;
    int rc = VSRB_OK;
    if (dtype == VSRB_BF16) {
        VSRB_CHECK_ARG(c % 8 == 0, "flow_warp: bf16 needs c %% 8 == 0 (got %d)", c);
        rc = launch_flow_warp<__nv_bfloat16>(reinterpret_cast<const __nv_bfloat16*>(x), xs, reinterpret_cast<const float2*>(flow), fs,
                                             reinterpret_cast<__nv_bfloat16*>(out), n, h, w, c, padding_mode, s);
    } else if (dtype == VSRB_BF16X2) {
        VSRB_CHECK_ARG(c % 16 == 0, "flow_warp: split-bf16 needs c %% 16 == 0 (got %d)", c);
        const int blocks = (int)(((long long)n * h * w + kWarpPix - 1) / kWarpPix);
        flow_warp_kernel<__nv_bfloat16, 0, true><<<blocks, 256, 0, s>>>(
            reinterpret_cast<const __nv_bfloat16*>(x), xs, reinterpret_cast<const float2*>(flow), fs,
            reinterpret_cast<__nv_bfloat16*>(out), n, h, w, padding_mode, c / 16);
    } else if (dtype == VSRB_F32) {
        VSRB_CHECK_ARG(c % 4 == 0, "flow_warp: fp32 needs c %% 4 == 0 (got %d)", c);
        rc = launch_flow_warp<float>(reinterpret_cast<const float*>(x), xs, reinterpret_cast<const float2*>(flow), fs,
                                     reinterpret_cast<float*>(out), n, h, w, c, padding_mode, s);
    } else {
        VSRB_CHECK_ARG(false, "flow_warp: bad dtype");
    }
    if (rc != VSRB_OK) return rc;
    VSRB_LAUNCH_CHECK();
    return VSRB_OK;
}

int vsrb_flow_warp_groups(const void* x, int64_t x_img_stride, int64_t x_group_stride, const float* flow, int64_t flow_img_stride,
                          int64_t flow_group_stride, void* out, int32_t imgs_per_group, int32_t groups, int32_t h, int32_t w, int32_t c,
                          int32_t dtype, int32_t padding_mode, void* stream) {
    VSRB_CHECK_ARG(x && flow && out && imgs_per_group >= 1 && groups >= 1 && h >= 1 && w >= 1, "flow_warp_groups: bad arguments");
    VSRB_CHECK_ARG(padding_mode == VSRB_PAD_ZEROS || padding_mode == VSRB_PAD_BORDER, "flow_warp_groups: bad padding mode");
    VSRB_CHECK_ARG(dtype == VSRB_BF16 && c % 8 == 0, "flow_warp_groups: bf16 NHWC with c %% 8 == 0 only");
    VSRB_CHECK_ARG((long long)imgs_per_group * groups * h * w < (1LL << 31), "flow_warp_groups: more than 2^31 pixels in one call");
    const long long xs = x_img_stride ? x_img_stride : (long long)h * w * c;
    const long long fs = flow_img_stride ? flow_img_stride : (long long)h * w;
    int rc = launch_flow_warp<__nv_bfloat16>(reinterpret_cast<const __nv_bfloat16*>(x), xs, reinterpret_cast<const float2*>(flow), fs,
                                             reinterpret_cast<__nv_bfloat16*>(out), imgs_per_group * groups, h, w, c, padding_mode,
                                             (cudaStream_t)stream, imgs_per_group, x_group_stride, flow_group_stride);
    if (rc != VSRB_OK) return rc;
    VSRB_LAUNCH_CHECK();
    return VSRB_OK;
}

int vsrb_flow_warp_ex(const void* x, int64_t x_img_stride, const float* flow, int64_t flow_img_stride, void* out, int32_t n,
                      int32_t h, int32_t w, int32_t c, int32_t dtype, int32_t interp, int32_t padding_mode, int32_t align_corners,
                      void* stream) {
    VSRB_CHECK_ARG(x && flow && out && n >= 1 && h >= 1 && w >= 1, "flow_warp_ex: bad arguments");
    VSRB_CHECK_ARG(interp == VSRB_INTERP_BILINEAR || interp == VSRB_INTERP_NEAREST || interp == VSRB_INTERP_BICUBIC,
                   "flow_warp_ex: bad interpolation mode %d (bilinear 0, nearest 1, bicubic 2)", interp);
    VSRB_CHECK_ARG(padding_mode == VSRB_PAD_ZEROS || padding_mode == VSRB_PAD_BORDER || padding_mode == VSRB_PAD_REFLECTION,
                   "flow_warp_ex: bad padding mode %d (zeros 0, border 1, reflection 2)", padding_mode);
    VSRB_CHECK_ARG(align_corners == 0 || align_corners == 1, "flow_warp_ex: align_corners must be 0 or 1 (got %d)", align_corners);
    // the propagation warp's mode: the existing kernel, so these results are the ones vsrb_flow_warp gives
    if (interp == VSRB_INTERP_BILINEAR && align_corners && padding_mode != VSRB_PAD_REFLECTION)
        return vsrb_flow_warp(x, x_img_stride, flow, flow_img_stride, out, n, h, w, c, dtype, padding_mode, stream);
    VSRB_CHECK_ARG((long long)n * h * w < (1LL << 31), "flow_warp_ex: more than 2^31 pixels in one call");
    const long long xs = x_img_stride ? x_img_stride : (long long)h * w * c;
    const long long fs = flow_img_stride ? flow_img_stride : (long long)h * w;
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == VSRB_BF16) {
        VSRB_CHECK_ARG(c >= 8 && c % 8 == 0, "flow_warp_ex: bf16 needs c %% 8 == 0 (got %d)", c);
        launch_flow_warp_ex<__nv_bfloat16>(reinterpret_cast<const __nv_bfloat16*>(x), xs, reinterpret_cast<const float2*>(flow), fs,
                                           reinterpret_cast<__nv_bfloat16*>(out), n, h, w, c, interp, padding_mode, align_corners, s);
    } else if (dtype == VSRB_F32) {
        VSRB_CHECK_ARG(c >= 4 && c % 4 == 0, "flow_warp_ex: fp32 needs c %% 4 == 0 (got %d)", c);
        launch_flow_warp_ex<float>(reinterpret_cast<const float*>(x), xs, reinterpret_cast<const float2*>(flow), fs,
                                   reinterpret_cast<float*>(out), n, h, w, c, interp, padding_mode, align_corners, s);
    } else {
        VSRB_CHECK_ARG(false, "flow_warp_ex: this mode needs dtype bf16 or fp32 (got %d)", dtype);
    }
    VSRB_LAUNCH_CHECK();
    return VSRB_OK;
}

int vsrb_nchw_to_nhwc(const float* src, void* dst, int32_t n, int32_t c, int32_t h, int32_t w, int32_t c_dst, int32_t dtype,
                      void* stream) {
    VSRB_CHECK_ARG(src && dst && n >= 1 && c >= 1 && c_dst >= c, "nchw_to_nhwc: bad arguments");
    const long long total = (long long)n * h * w;
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == VSRB_BF16X2) {
        VSRB_CHECK_ARG(c_dst % 2 == 0 && c_dst / 2 >= c, "nchw_to_nhwc: split layout needs c_dst = 2 * padded channels");
        nchw_to_nhwc_split_kernel<<<grid_for(total, 256), 256, 0, s>>>(src, reinterpret_cast<__nv_bfloat16*>(dst), n, c, h, w, c_dst);
    } else if (dtype == VSRB_BF16 && c <= 8 && c_dst == 16 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0)
        nchw_to_nhwc16_bf16_kernel<<<grid_for(total, 256), 256, 0, s>>>(src, reinterpret_cast<uint4*>(dst), n, c, h, w);
    else if (dtype == VSRB_BF16)
        nchw_to_nhwc_kernel<__nv_bfloat16><<<grid_for(total, 256), 256, 0, s>>>(src, reinterpret_cast<__nv_bfloat16*>(dst), n, c, h,
                                                                                 w, c_dst);
    else
        nchw_to_nhwc_kernel<float><<<grid_for(total, 256), 256, 0, s>>>(src, reinterpret_cast<float*>(dst), n, c, h, w, c_dst);
    VSRB_LAUNCH_CHECK();
    return VSRB_OK;
}

int vsrb_nhwc_to_nchw(const void* src, float* dst, int32_t n, int32_t c, int32_t h, int32_t w, int32_t c_src, int32_t dtype,
                      void* stream) {
    VSRB_CHECK_ARG(src && dst && n >= 1 && c >= 1 && c_src >= c, "nhwc_to_nchw: bad arguments");
    const long long total = (long long)n * c * h * w;
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == VSRB_BF16X2) {
        VSRB_CHECK_ARG(c_src % 2 == 0 && c_src / 2 >= c, "nhwc_to_nchw: split layout needs c_src = 2 * padded channels");
        nhwc_split_to_nchw_kernel<<<grid_for(total, 256), 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(src), dst, n, c, h, w,
                                                                        c_src);
    } else if (dtype == VSRB_BF16)
        nhwc_to_nchw_kernel<__nv_bfloat16><<<grid_for(total, 256), 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(src), dst, n,
                                                                                 c, h, w, c_src);
    else
        nhwc_to_nchw_kernel<float><<<grid_for(total, 256), 256, 0, s>>>(reinterpret_cast<const float*>(src), dst, n, c, h, w, c_src);
    VSRB_LAUNCH_CHECK();
    return VSRB_OK;
}

int vsrb_spynet_pyramid_base(const float* frames, float* lvl, int32_t F, int32_t h, int32_t w, int32_t Hp, int32_t Wp,
                             const float* mean3, const float* std3, void* stream) {
    VSRB_CHECK_ARG(frames && lvl && mean3 && std3 && F >= 1 && Hp % 32 == 0 && Wp % 32 == 0 && Hp >= h && Wp >= w,
                   "pyramid_base: bad arguments");
    const long long total = (long long)F * Hp * Wp;
    pyramid_base_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(frames, reinterpret_cast<float4*>(lvl), F, h, w, Hp,
                                                                                 Wp, mean3[0], mean3[1], mean3[2], std3[0], std3[1],
                                                                                 std3[2]);
    VSRB_LAUNCH_CHECK();
    return VSRB_OK;
}

int vsrb_avgpool2_c4(const float* in, float* out, int32_t F, int32_t H, int32_t W, void* stream) {
    VSRB_CHECK_ARG(in && out && F >= 1 && H % 2 == 0 && W % 2 == 0, "avgpool2: bad arguments");
    const long long total = (long long)F * (H / 2) * (W / 2);
    avgpool2_c4_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(in),
                                                                                reinterpret_cast<float4*>(out), F, H, W);
    VSRB_LAUNCH_CHECK();
    return VSRB_OK;
}

int vsrb_spynet_level_input(const float* lvl, const int32_t* ref_idx, const int32_t* supp_idx, const float* flow_prev,
                            float* flow_up, void* conv_in, int32_t P, int32_t Hl, int32_t Wl, int32_t c_in, int32_t dtype,
                            void* stream) {
    VSRB_CHECK_ARG(lvl && ref_idx && supp_idx && flow_up && conv_in && P >= 1 && c_in >= 8, "level_input: bad arguments");
    VSRB_CHECK_ARG(!flow_prev || (Hl % 2 == 0 && Wl % 2 == 0), "level_input: level extent must be even");
    const long long total = (long long)P * Hl * Wl;
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == VSRB_BF16) {
        VSRB_CHECK_ARG(c_in == 16, "level_input: bf16 path expects 16 allocated channels");
        level_input_kernel<__nv_bfloat16><<<grid_for(total, 256), 256, 0, s>>>(
            reinterpret_cast<const float4*>(lvl), ref_idx, supp_idx, reinterpret_cast<const float2*>(flow_prev),
            reinterpret_cast<float2*>(flow_up), reinterpret_cast<__nv_bfloat16*>(conv_in), P, Hl, Wl, c_in, 0);
    } else if (dtype == VSRB_BF16X2) {
        VSRB_CHECK_ARG(c_in == 32, "level_input: split-bf16 path expects 2 x 16 allocated channels");
        level_input_kernel<__nv_bfloat16><<<grid_for(total, 256), 256, 0, s>>>(
            reinterpret_cast<const float4*>(lvl), ref_idx, supp_idx, reinterpret_cast<const float2*>(flow_prev),
            reinterpret_cast<float2*>(flow_up), reinterpret_cast<__nv_bfloat16*>(conv_in), P, Hl, Wl, c_in, 1);
    } else {
        VSRB_CHECK_ARG(c_in % 4 == 0, "level_input: fp32 channel stride must be %% 4");
        level_input_kernel<float><<<grid_for(total, 256), 256, 0, s>>>(
            reinterpret_cast<const float4*>(lvl), ref_idx, supp_idx, reinterpret_cast<const float2*>(flow_prev),
            reinterpret_cast<float2*>(flow_up), reinterpret_cast<float*>(conv_in), P, Hl, Wl, c_in, 0);
    }
    VSRB_LAUNCH_CHECK();
    return VSRB_OK;
}

int vsrb_flow_resize(const float* flow_in, float* flow_out, int32_t P, int32_t Hp, int32_t Wp, int32_t h, int32_t w, void* stream) {
    VSRB_CHECK_ARG(flow_in && flow_out && P >= 1, "flow_resize: bad arguments");
    const long long total = (long long)P * h * w;
    flow_resize_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float2*>(flow_in), reinterpret_cast<float2*>(flow_out), P, Hp, Wp, h, w);
    VSRB_LAUNCH_CHECK();
    return VSRB_OK;
}

int vsrb_pixel_unshuffle2(const void* src, void* dst, int32_t n, int32_t h, int32_t w, int32_t c, void* stream) {
    VSRB_CHECK_ARG(src && dst && n >= 1 && h >= 1 && w >= 1 && c >= 8 && c % 8 == 0, "pixel_unshuffle2: bad arguments (c %% 8 == 0)");
    VSRB_CHECK_ARG(((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0, "pixel_unshuffle2: 16-byte alignment");
    const long long lr_pixels = (long long)n * h * w;
    pixel_unshuffle2_kernel<<<grid_for(lr_pixels * (c / 8), 256), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const uint4*>(src), reinterpret_cast<uint4*>(dst), lr_pixels, w, c);
    VSRB_LAUNCH_CHECK();
    return VSRB_OK;
}

}  // extern "C"
