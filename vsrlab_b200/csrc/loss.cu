// Training objective and evaluation metrics of the reference's loops, fused (SURVEY §8f row 2).  All HBM-bound: every
// operand is read once, reductions end in one atomic per block, nothing is synchronised and no scalar goes to the host.
// The *_det entry points store each block's sum to a slot of the caller's workspace instead and add the slots up in block
// order (ordered_sums_kernel): bit-reproducible sums for torch.use_deterministic_algorithms.
//
//  * vsrb_charbonnier          mean(sqrt((x-y)^2 + eps)) and its gradient in one pass      (core/losses.py:10-18)
//  * vsrb_charbonnier_resized  the same against `resize(hr, (h, w))` computed on the fly   (core/utils.py:238-239;
//                              kornia resize = bilinear, align_corners=False, no antialias)
//  * vsrb_psnr_sums            per-image sum of squared errors of clamp(x,0,1) vs y         (core/utils.py:242-247, piqa.PSNR)
//  * vsrb_ssim_sums            per-image sum of the SSIM map (11x11 Gaussian window, sigma 1.5, 'valid' borders,
//                              k1 = 0.01, k2 = 0.03, value range 1: piqa.SSIM's defaults)
#include <math.h>

#include "common.cuh"

namespace vsrb {

__device__ __forceinline__ double block_sum(double v) {
    __shared__ double part[32];
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __syncthreads();                     // `part` may still be read by a previous call in this block
    if (lane == 0) part[warp] = v;
    __syncthreads();
    v = (threadIdx.x < (blockDim.x >> 5)) ? part[threadIdx.x] : 0.0;
    if (warp == 0) {
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    }
    return v;                            // valid in thread 0
}

// thread 0's block sum: to the block's slot (deterministic mode) or atomically into *dst
__device__ __forceinline__ void block_out(double v, double* parts, long long slot, double* dst) {
    if (threadIdx.x == 0) {
        if (parts) parts[slot] = v;
        else atomicAdd(dst, v);
    }
}

// sums[j] += parts[j * run] + parts[j * run + 1] + ... + parts[j * run + run - 1], in that order
__global__ void ordered_sums_kernel(const double* __restrict__ parts, int run, int outs, double* sums) {
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < outs; j += gridDim.x * blockDim.x) {
        double acc = 0.0;
        for (int k = 0; k < run; ++k) acc += parts[(long long)j * run + k];
        sums[j] += acc;
    }
}

// sum += sum_i sqrt((x_i - y_i)^2 + eps);  grad_i = gscale * (x_i - y_i) / sqrt(...)   (gscale = upstream / n)
__global__ void charbonnier_kernel(const float* __restrict__ x, const float* __restrict__ y, long long n, float eps, double* sum,
                                   float* __restrict__ grad, const float* gscale_dev, float gscale, double* parts) {
    const float gs = gscale_dev ? *gscale_dev * gscale : gscale;
    double acc = 0.0;
    const long long n4 = n >> 2;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(x) + i), b = __ldg(reinterpret_cast<const float4*>(y) + i);
        const float d[4] = {a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w};
        float r[4], g[4];
        float part = 0.f;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            r[k] = sqrtf(d[k] * d[k] + eps);
            part += r[k];
            g[k] = gs * d[k] / r[k];
        }
        acc += (double)part;
        if (grad) reinterpret_cast<float4*>(grad)[i] = make_float4(g[0], g[1], g[2], g[3]);
    }
    for (long long i = (n4 << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float d = x[i] - y[i], r = sqrtf(d * d + eps);
        acc += (double)r;
        if (grad) grad[i] = gs * d / r;
    }
    acc = block_sum(acc);
    block_out(acc, parts, blockIdx.x, sum);
}

// lq [B,C,h,w] against the bilinear (align_corners=False) resize of hr [B,C,H,W] to (h,w)
__global__ void charbonnier_resized_kernel(const float* __restrict__ lq, const float* __restrict__ hr, int planes, int h, int w, int H,
                                           int W, float eps, double* sum, float* __restrict__ grad, const float* gscale_dev,
                                           float gscale, double* parts) {
    const float gs = gscale_dev ? *gscale_dev * gscale : gscale;
    const float sy = (float)H / (float)h, sx = (float)W / (float)w;
    const long long n = (long long)planes * h * w;
    double acc = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int xo = (int)(i % w);
        const long long t = i / w;
        const int yo = (int)(t % h);
        const long long p = t / h;
        int y0, y1, x0, x1;
        float ly, lx;
        up_tap(yo, sy, H, y0, y1, ly);
        up_tap(xo, sx, W, x0, x1, lx);
        const float* hp = hr + p * (long long)H * W;
        const float a00 = __ldg(hp + (long long)y0 * W + x0), a01 = __ldg(hp + (long long)y0 * W + x1);
        const float a10 = __ldg(hp + (long long)y1 * W + x0), a11 = __ldg(hp + (long long)y1 * W + x1);
        const float ref = (1.f - ly) * ((1.f - lx) * a00 + lx * a01) + ly * ((1.f - lx) * a10 + lx * a11);
        const float d = lq[i] - ref, r = sqrtf(d * d + eps);
        acc += (double)r;
        if (grad) grad[i] = gs * d / r;
    }
    acc = block_sum(acc);
    block_out(acc, parts, blockIdx.x, sum);
}

// sums[img] += sum over the image of (clamp(x,0,1) - y)^2
__global__ void psnr_sums_kernel(const float* __restrict__ x, const float* __restrict__ y, long long per_img, double* sums,
                                 double* parts) {
    const int img = blockIdx.y;
    const float* xp = x + (long long)img * per_img;
    const float* yp = y + (long long)img * per_img;
    double acc = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < per_img; i += (long long)gridDim.x * blockDim.x) {
        const float d = fminf(fmaxf(xp[i], 0.f), 1.f) - yp[i];
        acc += (double)(d * d);
    }
    acc = block_sum(acc);
    block_out(acc, parts, (long long)img * gridDim.x + blockIdx.x, sums + img);
}

// SSIM map of one 16x16 output tile of one (image, channel) plane: the 26x26 input patches of x and y are staged in shared
// memory, the five Gaussian moments are filtered separably (rows, then columns), the map is summed into sums[img].
static constexpr int kSsimT = 16, kSsimK = 11, kSsimP = kSsimT + kSsimK - 1;
struct SsimWin { float w[kSsimK]; };
__global__ void __launch_bounds__(256) ssim_sums_kernel(const float* __restrict__ x, const float* __restrict__ y, int C, int H, int W,
                                                       int clamp_x, SsimWin win, double* sums, double* parts) {
    __shared__ float sx[kSsimP][kSsimP + 1], sy_[kSsimP][kSsimP + 1];
    __shared__ float hm[5][kSsimP][kSsimT + 1];        // moments after the horizontal pass
    const int plane = blockIdx.z, img = plane / C;
    const int oy0 = blockIdx.y * kSsimT, ox0 = blockIdx.x * kSsimT;
    const int OH = H - kSsimK + 1, OW = W - kSsimK + 1;
    const float* xp = x + (long long)plane * H * W;
    const float* yp = y + (long long)plane * H * W;
    for (int i = threadIdx.x; i < kSsimP * kSsimP; i += 256) {
        const int r = i / kSsimP, c = i - r * kSsimP;
        const int gy = oy0 + r, gx = ox0 + c;
        float a = 0.f, b = 0.f;
        if (gy < H && gx < W) {
            a = xp[(long long)gy * W + gx];
            b = yp[(long long)gy * W + gx];
            if (clamp_x) a = fminf(fmaxf(a, 0.f), 1.f);
        }
        sx[r][c] = a;
        sy_[r][c] = b;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kSsimP * kSsimT; i += 256) {
        const int r = i / kSsimT, c = i - r * kSsimT;
        float m[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int k = 0; k < kSsimK; ++k) {
            const float a = sx[r][c + k], b = sy_[r][c + k], wk = win.w[k];
            m[0] += wk * a; m[1] += wk * b; m[2] += wk * a * a; m[3] += wk * b * b; m[4] += wk * a * b;
        }
#pragma unroll
        for (int j = 0; j < 5; ++j) hm[j][r][c] = m[j];
    }
    __syncthreads();
    const int r = threadIdx.x / kSsimT, c = threadIdx.x - r * kSsimT;
    double acc = 0.0;
    if (oy0 + r < OH && ox0 + c < OW) {
        float m[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int k = 0; k < kSsimK; ++k) {
            const float wk = win.w[k];
#pragma unroll
            for (int j = 0; j < 5; ++j) m[j] += wk * hm[j][r + k][c];
        }
        const float c1 = 0.01f * 0.01f, c2 = 0.03f * 0.03f;
        const float mxx = m[0] * m[0], myy = m[1] * m[1], mxy = m[0] * m[1];
        const float sxx = m[2] - mxx, syy = m[3] - myy, sxy = m[4] - mxy;
        const float cs = (2.f * sxy + c2) / (sxx + syy + c2);
        acc = (double)((2.f * mxy + c1) / (mxx + myy + c1) * cs);
    }
    acc = block_sum(acc);
    // blocks of one image are consecutive in (z, y, x) order: planes img*C .. img*C + C-1
    block_out(acc, parts, ((long long)plane * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x, sums + img);
}

}  // namespace vsrb

using namespace vsrb;

static int grid_for_n(long long n, int threads, int max_blocks = 148 * 8) {
    long long b = (n + threads - 1) / threads;
    if (b > max_blocks) b = max_blocks;
    return b < 1 ? 1 : (int)b;
}

// The launches of the entry points below; parts = null: atomics, else the deterministic slots (see ordered_sums_kernel).
// Each returns the number of blocks (= slots) it uses per output, or < 0 on a refused argument.
static long long charbonnier_blocks(long long n) { return grid_for_n(n / 4 + 1, 256); }
static long long charbonnier_resized_blocks(int planes, int h, int w) { return grid_for_n((long long)planes * h * w, 256); }
static long long psnr_blocks(long long per_image) { return grid_for_n(per_image, 256, 64); }
static long long ssim_blocks(int channels, int h, int w) {
    return (long long)ceil_div(w - kSsimK + 1, kSsimT) * ceil_div(h - kSsimK + 1, kSsimT) * channels;
}

static int check_workspace(const char* what, void* ws, size_t bytes, long long slots) {
    VSRB_CHECK_ARG(ws && (reinterpret_cast<uintptr_t>(ws) & 15) == 0 && bytes >= (size_t)slots * 8,
                   "%s: the workspace must be 16-byte aligned and hold %lld bytes (got %zu)", what, slots * 8, bytes);
    return VSRB_OK;
}

static int finish_ordered(double* parts, long long run, int outs, double* sums, cudaStream_t s) {
    VSRB_LAUNCH_CHECK();
    if (!parts) return VSRB_OK;
    ordered_sums_kernel<<<ceil_div(outs, 128), 128, 0, s>>>(parts, (int)run, outs, sums);
    VSRB_LAUNCH_CHECK();
    return VSRB_OK;
}

static int charbonnier_impl(const float* x, const float* y, int64_t n, float eps, double* sum, float* grad, const float* grad_scale_dev,
                            float grad_scale, double* parts, void* stream) {
    VSRB_CHECK_ARG(x && y && sum && n >= 1, "charbonnier: bad arguments");
    VSRB_CHECK_ARG(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(grad)) & 15) == 0,
                   "charbonnier: pointers must be 16-byte aligned");
    const int blocks = (int)charbonnier_blocks(n);
    charbonnier_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(x, y, n, eps, sum, grad, grad_scale_dev, grad_scale, parts);
    return finish_ordered(parts, blocks, 1, sum, (cudaStream_t)stream);
}

static int charbonnier_resized_impl(const float* lq, const float* hr, int32_t planes, int32_t h, int32_t w, int32_t H, int32_t W,
                                    float eps, double* sum, float* grad, const float* grad_scale_dev, float grad_scale, double* parts,
                                    void* stream) {
    VSRB_CHECK_ARG(lq && hr && sum && planes >= 1 && h >= 1 && w >= 1 && H >= 1 && W >= 1, "charbonnier_resized: bad arguments");
    const int blocks = (int)charbonnier_resized_blocks(planes, h, w);
    charbonnier_resized_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(lq, hr, planes, h, w, H, W, eps, sum, grad, grad_scale_dev,
                                                                         grad_scale, parts);
    return finish_ordered(parts, blocks, 1, sum, (cudaStream_t)stream);
}

static int psnr_sums_impl(const float* x, const float* y, int32_t images, int64_t per_image, double* sums, double* parts, void* stream) {
    VSRB_CHECK_ARG(x && y && sums && images >= 1 && images <= 65535 && per_image >= 1, "psnr_sums: bad arguments");
    dim3 grid((unsigned)psnr_blocks(per_image), images);
    psnr_sums_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, y, per_image, sums, parts);
    return finish_ordered(parts, grid.x, images, sums, (cudaStream_t)stream);
}

static int ssim_sums_impl(const float* x, const float* y, int32_t images, int32_t channels, int32_t h, int32_t w, int32_t clamp_x,
                          double* sums, double* parts, void* stream) {
    VSRB_CHECK_ARG(x && y && sums && images >= 1 && channels >= 1 && h >= kSsimK && w >= kSsimK, "ssim_sums: images must be at least 11x11");
    VSRB_CHECK_ARG((long long)images * channels <= 65535, "ssim_sums: too many planes in one call");
    SsimWin win;
    double tot = 0.0;
    for (int k = 0; k < kSsimK; ++k) {                 // piqa.utils.functional.gaussian_kernel(11, sigma=1.5), normalised
        const double d = k - (kSsimK - 1) / 2.0;
        win.w[k] = (float)exp(-d * d / (2.0 * 1.5 * 1.5));
        tot += win.w[k];
    }
    for (int k = 0; k < kSsimK; ++k) win.w[k] = (float)(win.w[k] / tot);
    dim3 grid(ceil_div(w - kSsimK + 1, kSsimT), ceil_div(h - kSsimK + 1, kSsimT), images * channels);
    ssim_sums_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, y, channels, h, w, clamp_x, win, sums, parts);
    return finish_ordered(parts, ssim_blocks(channels, h, w), images, sums, (cudaStream_t)stream);
}

extern "C" {

int vsrb_charbonnier(const float* x, const float* y, int64_t n, float eps, double* sum, float* grad, const float* grad_scale_dev,
                     float grad_scale, void* stream) {
    return charbonnier_impl(x, y, n, eps, sum, grad, grad_scale_dev, grad_scale, nullptr, stream);
}

int vsrb_charbonnier_resized(const float* lq, const float* hr, int32_t planes, int32_t h, int32_t w, int32_t H, int32_t W, float eps,
                             double* sum, float* grad, const float* grad_scale_dev, float grad_scale, void* stream) {
    return charbonnier_resized_impl(lq, hr, planes, h, w, H, W, eps, sum, grad, grad_scale_dev, grad_scale, nullptr, stream);
}

int vsrb_psnr_sums(const float* x, const float* y, int32_t images, int64_t per_image, double* sums, void* stream) {
    return psnr_sums_impl(x, y, images, per_image, sums, nullptr, stream);
}

int vsrb_ssim_sums(const float* x, const float* y, int32_t images, int32_t channels, int32_t h, int32_t w, int32_t clamp_x,
                   double* sums, void* stream) {
    return ssim_sums_impl(x, y, images, channels, h, w, clamp_x, sums, nullptr, stream);
}

size_t vsrb_charbonnier_det_workspace_bytes(int64_t n) { return n >= 1 ? (size_t)charbonnier_blocks(n) * 8 : 0; }
size_t vsrb_charbonnier_resized_det_workspace_bytes(int32_t planes, int32_t h, int32_t w) {
    return planes >= 1 && h >= 1 && w >= 1 ? (size_t)charbonnier_resized_blocks(planes, h, w) * 8 : 0;
}
size_t vsrb_psnr_sums_det_workspace_bytes(int32_t images, int64_t per_image) {
    return images >= 1 && per_image >= 1 ? (size_t)psnr_blocks(per_image) * images * 8 : 0;
}
size_t vsrb_ssim_sums_det_workspace_bytes(int32_t images, int32_t channels, int32_t h, int32_t w) {
    return images >= 1 && channels >= 1 && h >= kSsimK && w >= kSsimK ? (size_t)ssim_blocks(channels, h, w) * images * 8 : 0;
}

int vsrb_charbonnier_det(const float* x, const float* y, int64_t n, float eps, double* sum, float* grad, const float* grad_scale_dev,
                         float grad_scale, void* workspace, size_t workspace_bytes, void* stream) {
    int rc = check_workspace("charbonnier_det", workspace, workspace_bytes, n >= 1 ? charbonnier_blocks(n) : 0);
    if (rc != VSRB_OK) return rc;
    return charbonnier_impl(x, y, n, eps, sum, grad, grad_scale_dev, grad_scale, reinterpret_cast<double*>(workspace), stream);
}

int vsrb_charbonnier_resized_det(const float* lq, const float* hr, int32_t planes, int32_t h, int32_t w, int32_t H, int32_t W,
                                 float eps, double* sum, float* grad, const float* grad_scale_dev, float grad_scale, void* workspace,
                                 size_t workspace_bytes, void* stream) {
    int rc = check_workspace("charbonnier_resized_det", workspace, workspace_bytes,
                             planes >= 1 && h >= 1 && w >= 1 ? charbonnier_resized_blocks(planes, h, w) : 0);
    if (rc != VSRB_OK) return rc;
    return charbonnier_resized_impl(lq, hr, planes, h, w, H, W, eps, sum, grad, grad_scale_dev, grad_scale,
                                    reinterpret_cast<double*>(workspace), stream);
}

int vsrb_psnr_sums_det(const float* x, const float* y, int32_t images, int64_t per_image, double* sums, void* workspace,
                       size_t workspace_bytes, void* stream) {
    int rc = check_workspace("psnr_sums_det", workspace, workspace_bytes,
                             images >= 1 && per_image >= 1 ? psnr_blocks(per_image) * images : 0);
    if (rc != VSRB_OK) return rc;
    return psnr_sums_impl(x, y, images, per_image, sums, reinterpret_cast<double*>(workspace), stream);
}

int vsrb_ssim_sums_det(const float* x, const float* y, int32_t images, int32_t channels, int32_t h, int32_t w, int32_t clamp_x,
                       double* sums, void* workspace, size_t workspace_bytes, void* stream) {
    int rc = check_workspace("ssim_sums_det", workspace, workspace_bytes,
                             images >= 1 && channels >= 1 && h >= kSsimK && w >= kSsimK ? ssim_blocks(channels, h, w) * images : 0);
    if (rc != VSRB_OK) return rc;
    return ssim_sums_impl(x, y, images, channels, h, w, clamp_x, sums, reinterpret_cast<double*>(workspace), stream);
}

}  // extern "C"
