// Backward kernels of the hot path (training, SURVEY K12 / §8 row a13).
//
//  * input gradient of a conv  = the forward conv kernel run on the output gradient with the weights packed
//    transposed + flipped (vsrb_conv_geom.transpose = 1) - no new kernel;
//  * weight / bias gradient     = conv_wgrad_kernel below: dW[co][ci][ky][kx] = sum_pixels dz[p][co] * x[p + tap][ci]
//    (reference: autograd's ConvolutionBackward0 of every nn.Conv2d on the path);
//  * flow_warp backward         = flow_warp_bwd_kernel: scatter of the output gradient through the four bilinear
//    taps (grad wrt the warped features) and the derivative of the taps wrt the sample position (grad wrt the
//    flow, needed when train_flow=True) - reference: GridSampler2DBackward0 behind spynet.py:95-106.
#include <stdlib.h>

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
// weight gradient (FFMA fallback for the shapes the tensor-core kernel does not take: 7x7, 1x1, 3-channel
// segments).  One CTA = one filter ROW ky x one 64(co) x 64(ci) tile x a run of 32-pixel row chunks.  Per chunk it
// stages dz [32 px][64 co] and ONE extended activation strip [32 + kw - 1 px][64 ci] of image row y + ky - pad, and
// updates the kw taps of the row from it (kw x 4x4 fp32 accumulators per thread), so dz is read kh times instead
// of kh*kw times.  Results are added to the OIHW fp32 gradient with atomics.
// ---------------------------------------------------------------------------------------
struct WgradParams {
    const void* in[2];
    int in_c[2], seg_c[2], seg_off[2];
    int n_seg;
    const void* dz;
    int dz_c;
    int kh, kw, H, W, imgs_per_group, groups;
    int cout, cin_total;
    int chunks_per_row, units_g, units_per_cta;   // unit = (image of the group, row y, 32-pixel chunk)
    int n_co_blk, n_ci_blk;                       // 64-wide blocks
    int ci_blk_seg[8], ci_blk_c0[8];
    float* dw;
};

// CO_T x CI_T = the (co, ci) tile of one CTA (16, 32 or 64 each).  A thread owns a 4x4 patch of it; the 256 threads
// form 256 / (CO_T/4 * CI_T/4) pixel groups that split the 32 pixels of a chunk between them, so narrow layers
// (SPyNet's 8->32, 32->16, 16->2 ...) do not pay for a full 64x64 tile.
template <typename T, int KW, int CO_T, int CI_T>
__global__ void __launch_bounds__(256) conv_wgrad_kernel(WgradParams P) {
    constexpr int TY = CO_T / 4, TX = CI_T / 4, TPG = TY * TX, PG = 256 / TPG;
    __shared__ __align__(16) float zs[32][CO_T];
    __shared__ __align__(16) float xs[32 + KW - 1][CI_T];
    const int tid = threadIdx.x;
    const int pg = tid / TPG, rr = tid % TPG;
    const int tx = rr % TX, ty = rr / TX;               // 4 ci per tx, 4 co per ty
    const int ky = blockIdx.y;
    int z = blockIdx.z;
    const int cib = z % P.n_ci_blk; z /= P.n_ci_blk;
    const int cob = z % P.n_co_blk;
    const int g = z / P.n_co_blk;
    const int s = P.ci_blk_seg[cib], c0 = P.ci_blk_c0[cib];
    const int co0 = cob * CO_T;
    const int hw = P.H * P.W;
    const int u_begin = blockIdx.x * P.units_per_cta;
    const int u_end = min(u_begin + P.units_per_cta, P.units_g);
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
        const long long img = (long long)g * P.imgs_per_group + rowi / P.H;
        const int x0 = xc * 32;
        const int yy = y + dy;
        __syncthreads();
        for (int i = tid; i < 32 * (CO_T / 8); i += 256) {          // dz chunk [32 px][CO_T]
            const int lp = i / (CO_T / 8), lc = (i % (CO_T / 8)) * 8;
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
        for (int i = tid; i < (32 + KW - 1) * (CI_T / 8); i += 256) {   // extended strip: image columns x0 - pad + e
            const int ep = i / (CI_T / 8), lc = (i % (CI_T / 8)) * 8;
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
        for (int q = pg; q < 32; q += PG) {
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
                    atomicAdd(P.dw + (((size_t)g * P.cout + co) * P.cin_total + P.seg_off[s] + ci) * taps + ky * KW + k, acc[k][i][j]);
            }
        }
}

// ---------------------------------------------------------------------------------------
// bf16 weight gradient on the warp-level tensor-core path (mma.sync m16n8k16) for the shapes wgrad_tc_kernel does not
// take (SPyNet's 7x7 layers, 1x1, 3-channel segments).  Same decomposition as conv_wgrad_kernel - one filter row ky and
// one CO_T x CI_T tile per CTA, 32-pixel row chunks - but the chunk is staged as bf16 and each filter column kx is the
// GEMM  D_kx[co][ci] += sum_q dz[q][co] * x[q + kx][ci]  (K = 32 pixels = two k16 steps).  Both operands sit pixel-major
// in shared memory, i.e. transposed for the MMA, and are fetched with ldmatrix.trans; the kx shift is just a row offset
// of the B fetch, so dz fragments are loaded once per k-step and reused by all kw columns.  (tcgen05 needs the pixel
// shift in whole swizzle atoms - wgrad_tc.cu pays three halo copies for kw = 3; seven would not fit.)
// Rows are padded by 16 bytes so the eight 16-byte rows of an ldmatrix land in different banks.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t (&r)[4]) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(addr));
}
__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// keeps the first `valid` (0..8) bf16 of a 16-byte vector, zeroes the rest
__device__ __forceinline__ uint4 keep_bf16(uint4 u, int valid) {
    uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int left = valid - 2 * i;
        w[i] = left >= 2 ? w[i] : (left == 1 ? (w[i] & 0xFFFFu) : 0u);
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

static constexpr int kMmaPx = 64;      // pixels of a chunk: four k16 steps amortise the per-chunk address math and barriers

template <int KW, int CO_T, int CI_T>
__global__ void __launch_bounds__(256) conv_wgrad_mma_kernel(WgradParams P) {
    constexpr int PX = kMmaPx, NKS = PX / 16;
    constexpr int ZP = CO_T * 2 + 16, XP = CI_T * 2 + 16;             // padded row pitch in bytes
    constexpr int WT = (CO_T / 16) * (CI_T / 16);                     // 16 x 16 warp tiles of the CTA tile
    constexpr int TPW = WT >= 8 ? WT / 8 : 1;                         // tiles per warp
    constexpr int KS = WT >= 8 ? 1 : (8 / WT > NKS ? NKS : 8 / WT);   // warps sharing a tile split the k16 steps
    __shared__ __align__(16) uint8_t zs[PX * ZP];
    __shared__ __align__(16) uint8_t xs[(PX + KW - 1) * XP];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int ky = blockIdx.y;
    int z = blockIdx.z;
    const int cib = z % P.n_ci_blk; z /= P.n_ci_blk;
    const int cob = z % P.n_co_blk;
    const int g = z / P.n_co_blk;
    const int s = P.ci_blk_seg[cib], c0 = P.ci_blk_c0[cib];
    const int co0 = cob * CO_T;
    const int hw = P.H * P.W;
    const int u_begin = blockIdx.x * P.units_per_cta;
    const int u_end = min(u_begin + P.units_per_cta, P.units_g);
    const __nv_bfloat16* zin = reinterpret_cast<const __nv_bfloat16*>(P.dz);
    const __nv_bfloat16* xin = reinterpret_cast<const __nv_bfloat16*>(P.in[s]);
    const int dy = ky - P.kh / 2, pad = KW / 2;

    // this warp's tiles and k-steps
    const int t_first = WT >= 8 ? warp * TPW : warp % WT;
    const int ks_own = WT >= 8 ? -1 : warp / WT;                       // -1: all k16 steps; else steps ks_own, ks_own + KS, ...
    const bool active = WT >= 8 || ks_own < KS;
    float acc[TPW][KW][2][4];
#pragma unroll
    for (int t = 0; t < TPW; ++t)
#pragma unroll
        for (int k = 0; k < KW; ++k)
#pragma unroll
            for (int n = 0; n < 2; ++n)
#pragma unroll
                for (int i = 0; i < 4; ++i) acc[t][k][n][i] = 0.f;
    const uint32_t zs0 = (uint32_t)__cvta_generic_to_shared(zs), xs0 = (uint32_t)__cvta_generic_to_shared(xs);
    const int lj = lane >> 3, lr = lane & 7;                            // ldmatrix: matrix index and row of this lane's address

    // Register double buffering: the next chunk's 16-byte global loads are issued before the current chunk's MMAs and only
    // written to shared memory after them, so the global-memory latency hides behind the tensor-core work.
    constexpr int ZI = PX * (CO_T / 8), XI = (PX + KW - 1) * (CI_T / 8);   // 16-byte items per chunk
    constexpr int ZJ = (ZI + 255) / 256, XJ = (XI + 255) / 256;
    uint4 zr[ZJ], xr[XJ];
    auto fetch = [&](int u) {
        const int xc = u % P.chunks_per_row;
        const int rowi = u / P.chunks_per_row;
        const int y = rowi % P.H;
        const long long img = (long long)g * P.imgs_per_group + rowi / P.H;
        const int x0 = xc * PX;
        const int yy = y + dy;
#pragma unroll
        for (int j = 0; j < ZJ; ++j) {                              // dz chunk [PX px][CO_T] bf16
            const int i = tid + j * 256;
            zr[j] = make_uint4(0u, 0u, 0u, 0u);
            if (i < ZI) {
                const int lp = i / (CO_T / 8), lc = (i % (CO_T / 8)) * 8;
                if (x0 + lp < P.W && co0 + lc < P.dz_c) {
                    zr[j] = __ldg(reinterpret_cast<const uint4*>(zin + (img * hw + (long long)y * P.W + x0 + lp) * P.dz_c + co0 + lc));
                    zr[j] = keep_bf16(zr[j], P.cout - (co0 + lc));
                }
            }
        }
#pragma unroll
        for (int j = 0; j < XJ; ++j) {                              // extended strip: image columns x0 - pad + e
            const int i = tid + j * 256;
            xr[j] = make_uint4(0u, 0u, 0u, 0u);
            if (i < XI) {
                const int ep = i / (CI_T / 8), lc = (i % (CI_T / 8)) * 8;
                const int xx = x0 - pad + ep;
                if (yy >= 0 && yy < P.H && xx >= 0 && xx < P.W && c0 + lc < P.in_c[s]) {
                    xr[j] = __ldg(reinterpret_cast<const uint4*>(xin + (img * hw + (long long)yy * P.W + xx) * P.in_c[s] + c0 + lc));
                    xr[j] = keep_bf16(xr[j], P.seg_c[s] - (c0 + lc));
                }
            }
        }
    };
    if (u_begin < u_end) fetch(u_begin);
    for (int u = u_begin; u < u_end; ++u) {
        __syncthreads();                                            // the previous chunk's fragments have been read
#pragma unroll
        for (int j = 0; j < ZJ; ++j) {
            const int i = tid + j * 256;
            if (i < ZI) *reinterpret_cast<uint4*>(zs + (i / (CO_T / 8)) * ZP + (i % (CO_T / 8)) * 16) = zr[j];
        }
#pragma unroll
        for (int j = 0; j < XJ; ++j) {
            const int i = tid + j * 256;
            if (i < XI) *reinterpret_cast<uint4*>(xs + (i / (CI_T / 8)) * XP + (i % (CI_T / 8)) * 16) = xr[j];
        }
        __syncthreads();
        if (u + 1 < u_end) fetch(u + 1);
        if (active) {
#pragma unroll
            for (int ks = 0; ks < NKS; ++ks) {
                if (ks_own >= 0 && (ks % KS) != ks_own) continue;
                const int q0 = ks * 16;
#pragma unroll
                for (int t = 0; t < TPW; ++t) {
                    const int tile = t_first + t;
                    const int co_off = (tile / (CI_T / 16)) * 16, ci_off = (tile % (CI_T / 16)) * 16;
                    uint32_t a[4];
                    ldsm_x4_t(zs0 + (uint32_t)((q0 + (lj >> 1) * 8 + lr) * ZP + (co_off + (lj & 1) * 8) * 2), a);
#pragma unroll
                    for (int k = 0; k < KW; ++k) {
                        uint32_t b[4];
                        ldsm_x4_t(xs0 + (uint32_t)((q0 + k + (lj & 1) * 8 + lr) * XP + (ci_off + (lj >> 1) * 8) * 2), b);
                        mma_bf16_16816(acc[t][k][0], a, b[0], b[1]);
                        mma_bf16_16816(acc[t][k][1], a, b[2], b[3]);
                    }
                }
            }
        }
    }
    if (!active) return;
    const int taps = P.kh * KW;
    const int gq = lane >> 2, tq = lane & 3;
#pragma unroll
    for (int t = 0; t < TPW; ++t) {
        const int tile = t_first + t;
        const int co_off = (tile / (CI_T / 16)) * 16, ci_off = (tile % (CI_T / 16)) * 16;
#pragma unroll
        for (int k = 0; k < KW; ++k)
#pragma unroll
            for (int n = 0; n < 2; ++n)
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int co = co0 + co_off + gq + (i >> 1) * 8;
                    const int ci = c0 + ci_off + n * 8 + tq * 2 + (i & 1);
                    if (co < P.cout && ci < P.seg_c[s])
                        atomicAdd(P.dw + (((size_t)g * P.cout + co) * P.cin_total + P.seg_off[s] + ci) * taps + ky * KW + k,
                                  acc[t][k][n][i]);
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

int launch_wgrad_tc(const void* x, int x_c, int c0, int ci_off, const void* dz, int dz_c, int batch, int h, int w, int cout,
                    int cin_total, float* dw, cudaStream_t stream, float* db = nullptr);
int launch_bias_grad(const void* dz, int dz_c, long long pixels, int cout, int dtype, float* db, cudaStream_t s);
int launch_bias_grad_multi(const void* const* dzs, int n_chunks, int dz_c, long long pixels, int cout, int dtype, float* db,
                           cudaStream_t s);
int launch_wgrad_tc_multi(const void* const* xs, int x_c, int c0, int ci_off, const void* const* dzs, int dz_c, int n_chunks,
                          int batch, int h, int w, int cout, int cin_total, float* dw, cudaStream_t stream, float* db = nullptr);
int launch_wgrad_taps(const void* x, int x_c, int x_c0, int ci_n, int ci_off, const void* dz, int dz_c, int z_c0, int co_n, int K,
                      int batch, int h, int w, int cin_total, float* dw, cudaStream_t stream);

}  // namespace vsrb

using namespace vsrb;

extern "C" {

int vsrb_conv2d_wgrad_multi(const vsrb_conv_geom* g, int32_t n_chunks, const void* const* in, const int32_t* in_c,
                            const void* const* dz, int32_t dz_c, int32_t batch, int32_t h, int32_t w, int32_t cin_total,
                            float* dw, float* db, void* stream) {
    VSRB_CHECK_ARG(g && in && in_c && dz && dw && n_chunks >= 1, "wgrad_multi: null argument");
    VSRB_CHECK_ARG(g->dtype == VSRB_BF16 && g->kh == 3 && g->kw == 3 && g->groups == 1 && !g->pixshuf && !g->transpose &&
                       g->n_seg >= 1 && g->n_seg <= 2 && dz_c >= g->cout && dz_c % 8 == 0,
                   "wgrad_multi: bf16 3x3 ungrouped convs only (tensor-core path)");
    for (int s = 0; s < g->n_seg; ++s)
        VSRB_CHECK_ARG(g->seg_c[s] % 64 == 0 && in_c[s] % 8 == 0 && in_c[s] >= g->seg_c[s] && g->seg_off[s] + g->seg_c[s] <= cin_total,
                       "wgrad_multi: segment %d must have a multiple of 64 channels", s);
    cudaStream_t st = (cudaStream_t)stream;
    // the bias gradient rides along with the first input-channel block of every group of chunks (the kernel's idle epilogue
    // warps add up the dz tiles it streams anyway); VSRB_WGRAD_SEPARATE_BIAS=1 keeps the separate reduction kernel
    const bool fuse_bias = db && !getenv("VSRB_WGRAD_SEPARATE_BIAS");
    for (int k0 = 0; k0 < n_chunks; k0 += 16) {
        const int nk = n_chunks - k0 < 16 ? n_chunks - k0 : 16;
        bool first = true;
        for (int s = 0; s < g->n_seg; ++s) {
            const void* xs[16];
            for (int k = 0; k < nk; ++k) xs[k] = in[(size_t)(k0 + k) * g->n_seg + s];
            for (int c0 = 0; c0 < g->seg_c[s]; c0 += 64) {
                int rc = launch_wgrad_tc_multi(xs, in_c[s], c0, g->seg_off[s] + c0, dz + k0, dz_c, nk, batch, h, w, g->cout, cin_total, dw, st,
                                               (fuse_bias && first) ? db : nullptr);
                if (rc != VSRB_OK) return rc;
                first = false;
            }
        }
    }
    if (db && !fuse_bias) {
        int rc = launch_bias_grad_multi(dz, n_chunks, dz_c, (long long)batch * h * w, g->cout, g->dtype, db, st);
        if (rc != VSRB_OK) return rc;
    }
    return VSRB_OK;
}

int vsrb_conv2d_wgrad(const vsrb_conv_geom* g, const void* const* in, const int32_t* in_c, const void* dz, int32_t dz_c,
                      int32_t batch, int32_t h, int32_t w, int32_t imgs_per_group, int32_t cin_total, float* dw, float* db,
                      void* stream) {
    VSRB_CHECK_ARG(g && in && in_c && dz && dw, "wgrad: null argument");
    VSRB_CHECK_ARG(g->n_seg == 1 || g->n_seg == 2, "wgrad: n_seg must be 1 or 2");
    VSRB_CHECK_ARG(!g->pixshuf && !g->transpose, "wgrad: pass the plain forward geometry (un-shuffle the gradient first)");
    VSRB_CHECK_ARG(imgs_per_group >= 1 && imgs_per_group * g->groups == batch, "wgrad: batch/groups mismatch");
    VSRB_CHECK_ARG((long long)imgs_per_group * h * w < (1LL << 31), "wgrad: too many pixels per group");
    const int vec = g->dtype == VSRB_BF16 ? 8 : 8;
    VSRB_CHECK_ARG(dz_c % vec == 0, "wgrad: dz channel stride must be a multiple of 8");
    WgradParams P;
    memset(&P, 0, sizeof(P));
    P.n_seg = g->n_seg;
    P.n_ci_blk = 0;
    // 3x3 layers whose segment has a multiple of 64 channels (the resblock, upsampling and HR convs: > 85 % of
    // the FLOPs; a cout below 64 is zero-filled by the TMA box) run on the tensor cores; everything else on the
    // FFMA kernel
    const bool tc_ok = g->dtype == VSRB_BF16 && g->kh == 3 && g->kw == 3 && g->groups == 1 && dz_c >= g->cout &&
                       (reinterpret_cast<uintptr_t>(dz) & 15) == 0 && !getenv("VSRB_WGRAD_SIMT");
    // ... except that every other bf16 segment of an odd square filter up to 7x7 (SPyNet's 7x7 stacks, 3-channel image
    // segments, 1x1) takes the tap-stacking tcgen05 kernel of wgrad_taps.cu; VSRB_WGRAD_MMA=1 keeps the mma.sync kernel
    const bool taps_ok = g->dtype == VSRB_BF16 && g->kh == g->kw && (g->kw & 1) && g->kw <= 7 && g->groups == 1 && dz_c % 8 == 0 &&
                         (reinterpret_cast<uintptr_t>(dz) & 15) == 0 && !getenv("VSRB_WGRAD_SIMT") && !getenv("VSRB_WGRAD_FFMA") &&
                         !getenv("VSRB_WGRAD_MMA");
    bool on_tc[4] = {false, false, false, false};
    bool db_done = false;
    // (co, ci) tile of the mma.sync kernel: as narrow as its segments allow (the FFMA kernels keep 64 x 64)
    int co_t = 64, ci_t = 64, cmax = 0;
    for (int s = 0; s < g->n_seg; ++s) {
        // (a thin output - the 64 -> 3 image convs - would zero-fill 61 of wgrad_tc's 64 dz columns: the tap kernel takes dz as
        // its narrow operand instead; VSRB_WGRAD_TAPS_ALL=1 sends every segment there, for A/B measurements)
        on_tc[s] = tc_ok && g->seg_c[s] % 64 == 0 && (reinterpret_cast<uintptr_t>(in[s]) & 15) == 0 &&
                   !(taps_ok && (g->cout <= 16 || getenv("VSRB_WGRAD_TAPS_ALL")));
        if (!on_tc[s] && g->seg_c[s] > cmax) cmax = g->seg_c[s];
    }
    if (g->dtype == VSRB_BF16 && !getenv("VSRB_WGRAD_FFMA")) {
        co_t = g->cout <= 16 ? 16 : (g->cout <= 32 ? 32 : 64);
        ci_t = cmax <= 16 ? 16 : (cmax <= 32 ? 32 : 64);
    }
    for (int s = 0; s < g->n_seg; ++s) {
        VSRB_CHECK_ARG(in[s] && in_c[s] % 8 == 0 && in_c[s] >= g->seg_c[s], "wgrad: bad input segment %d", s);
        VSRB_CHECK_ARG(g->seg_off[s] + g->seg_c[s] <= cin_total, "wgrad: segment %d exceeds cin_total", s);
        P.in[s] = in[s]; P.in_c[s] = in_c[s]; P.seg_c[s] = g->seg_c[s]; P.seg_off[s] = g->seg_off[s];
        if (on_tc[s]) {
            for (int c0 = 0; c0 < g->seg_c[s]; c0 += 64) {
                const bool ride = db && !db_done && !getenv("VSRB_WGRAD_SEPARATE_BIAS");      // bias gradient from the same pass over dz
                int rc = launch_wgrad_tc(in[s], in_c[s], c0, g->seg_off[s] + c0, dz, dz_c, batch, h, w, g->cout, cin_total, dw,
                                         (cudaStream_t)stream, ride ? db : nullptr);
                if (rc != VSRB_OK) return rc;
                db_done = db_done || ride;
            }
            continue;
        }
        if (taps_ok && (reinterpret_cast<uintptr_t>(in[s]) & 15) == 0) {
            for (int c0 = 0; c0 < g->seg_c[s]; c0 += 64)
                for (int n0 = 0; n0 < g->cout; n0 += 64) {
                    const int ci_n = g->seg_c[s] - c0 < 64 ? g->seg_c[s] - c0 : 64, co_n = g->cout - n0 < 64 ? g->cout - n0 : 64;
                    int rc = launch_wgrad_taps(in[s], in_c[s], c0, ci_n, g->seg_off[s] + c0, dz, dz_c, n0, co_n, g->kw, batch, h, w, cin_total,
                                               dw, (cudaStream_t)stream);
                    if (rc != VSRB_OK) return rc;
                }
            continue;
        }
        for (int c0 = 0; c0 < g->seg_c[s]; c0 += ci_t) {
            VSRB_CHECK_ARG(P.n_ci_blk < 8, "wgrad: too many input-channel blocks");
            P.ci_blk_seg[P.n_ci_blk] = s;
            P.ci_blk_c0[P.n_ci_blk] = c0;
            ++P.n_ci_blk;
        }
    }
    if (db && !db_done) {
        int rc = launch_bias_grad(dz, dz_c, (long long)batch * h * w, g->cout * g->groups == g->cout ? g->cout : g->cout, g->dtype, db,
                                  (cudaStream_t)stream);
        if (rc != VSRB_OK) return rc;
    }
    if (P.n_ci_blk == 0) return VSRB_OK;
    P.dz = dz; P.dz_c = dz_c;
    P.kh = g->kh; P.kw = g->kw; P.H = h; P.W = w; P.imgs_per_group = imgs_per_group; P.groups = g->groups;
    P.cout = g->cout; P.cin_total = cin_total;
    P.n_co_blk = ceil_div(g->cout, co_t);
    P.dw = dw;
    const bool mma_path = g->dtype == VSRB_BF16 && !getenv("VSRB_WGRAD_FFMA");
    P.chunks_per_row = ceil_div(w, mma_path ? kMmaPx : 32);
    const long long units_g = (long long)imgs_per_group * h * P.chunks_per_row;
    VSRB_CHECK_ARG(units_g < (1LL << 31), "wgrad: too many pixels per group");
    P.units_g = (int)units_g;
    // ~6 waves of the 148 SMs, at least 16 chunks (512 pixels) per CTA to amortise the final atomics
    const long long other = (long long)g->kh * P.n_co_blk * P.n_ci_blk * g->groups;
    long long ctas = (148LL * 6 + other - 1) / other;
    long long per = (units_g + ctas - 1) / ctas;
    if (per < 16) per = 16;
    P.units_per_cta = (int)per;
    dim3 grid((unsigned)((units_g + per - 1) / per), g->kh, P.n_co_blk * P.n_ci_blk * g->groups);
    cudaStream_t st = (cudaStream_t)stream;
#define VSRB_WG_KW(KERN, CO, CI)                                                       \
    do {                                                                                \
        if (g->kw == 1) KERN(1, CO, CI)<<<grid, 256, 0, st>>>(P);                       \
        else if (g->kw == 3) KERN(3, CO, CI)<<<grid, 256, 0, st>>>(P);                  \
        else if (g->kw == 7) KERN(7, CO, CI)<<<grid, 256, 0, st>>>(P);                  \
        else {                                                                          \
            set_error("wgrad: kernel width %d unsupported", g->kw);                     \
            return VSRB_E_ARG;                                                          \
        }                                                                               \
    } while (0)
#define VSRB_WG_CI(KERN, CO)                               \
    do {                                                    \
        if (ci_t == 16) VSRB_WG_KW(KERN, CO, 16);           \
        else if (ci_t == 32) VSRB_WG_KW(KERN, CO, 32);      \
        else VSRB_WG_KW(KERN, CO, 64);                      \
    } while (0)
#define VSRB_K_MMA(KW, CO, CI) conv_wgrad_mma_kernel<KW, CO, CI>
#define VSRB_K_F32(KW, CO, CI) conv_wgrad_kernel<float, KW, CO, CI>
#define VSRB_K_FFMA16(KW, CO, CI) conv_wgrad_kernel<__nv_bfloat16, KW, CO, CI>
    if (g->dtype == VSRB_BF16 && !getenv("VSRB_WGRAD_FFMA")) {
        if (co_t == 16) VSRB_WG_CI(VSRB_K_MMA, 16);
        else if (co_t == 32) VSRB_WG_CI(VSRB_K_MMA, 32);
        else VSRB_WG_CI(VSRB_K_MMA, 64);
    } else if (g->dtype == VSRB_BF16) {                    // cross-check path: the FFMA kernel on bf16 data, 64 x 64 tiles
        VSRB_WG_KW(VSRB_K_FFMA16, 64, 64);
    } else {
        VSRB_WG_KW(VSRB_K_F32, 64, 64);
    }
#undef VSRB_K_FFMA16
#undef VSRB_K_F32
#undef VSRB_K_MMA
#undef VSRB_WG_CI
#undef VSRB_WG_KW
    VSRB_LAUNCH_CHECK();
    return VSRB_OK;
}

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
