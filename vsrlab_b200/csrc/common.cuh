// Internal helpers shared by every translation unit of libvsrb200.so.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <functional>

#include "../../include/vsrb200.h"

namespace vsrb {

// ---------------------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
void count_launch();
int* debug_flag();   // device flag raised by kernels on a pipeline time-out

#define VSRB_CHECK_ARG(cond, ...)                      \
    do {                                               \
        if (!(cond)) {                                 \
            vsrb::set_error(__VA_ARGS__);              \
            return VSRB_E_ARG;                         \
        }                                              \
    } while (0)

#define VSRB_CUDA(call)                                                                   \
    do {                                                                                  \
        cudaError_t e__ = (call);                                                         \
        if (e__ != cudaSuccess) {                                                         \
            vsrb::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__),      \
                            __FILE__, __LINE__);                                          \
            return VSRB_E_CUDA;                                                           \
        }                                                                                 \
    } while (0)

#define VSRB_LAUNCH_CHECK()                                                               \
    do {                                                                                  \
        vsrb::count_launch();                                                             \
        cudaError_t e__ = cudaGetLastError();                                             \
        if (e__ != cudaSuccess) {                                                         \
            vsrb::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(e__),  \
                            __FILE__, __LINE__);                                          \
            return VSRB_E_CUDA;                                                           \
        }                                                                                 \
    } while (0)

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline size_t round_up(size_t a, size_t b) { return (a + b - 1) / b * b; }

// ---------------------------------------------------------------------------------------
// host plumbing of the tcgen05 launchers
// ---------------------------------------------------------------------------------------
int env_int(const char* name);   // integer debug switch from the environment, 0 when unset

constexpr int kMaxDevices = 64;
// The current device and its SM count (read once per device).  `setup` is the caller's one-time set-up for that device
// (function attributes, constant tables); it runs under the library's initialisation lock until it returns VSRB_OK,
// which the caller's `done` records.
int device_setup(int* dev, int* sms, bool (&done)[kMaxDevices], const std::function<int(int dev)>& setup);

// Deterministic weight / bias gradients (the *_det entry points of train.cu): the launchers store every CTA's partial block
// in a slot of the caller's workspace `ws` and sum the slots in slot order (launch_slot_reduce) instead of adding with
// atomics.  With `plan` set they launch nothing and only raise `need` (floats) to what they would use.
struct WgradDet {
    float* ws;
    size_t need;
    bool plan;
};
int launch_slot_reduce(const float* parts, int slots, int rows, int row_len, long long dst_stride, float* dst, cudaStream_t s);
// a launcher about to use `floats` of the workspace: true = planning only, launch nothing
static inline bool det_take(WgradDet* det, size_t floats) {
    if (floats > det->need) det->need = floats;
    return det->plan;
}

// Swizzle of a K-major shared-memory tile whose rows hold `channels` bf16 (64: 128 B, 32: 64 B, 16: 32 B)
static inline CUtensorMapSwizzle swizzle_for(int channels) {
    return channels == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : (channels == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
}
// A bf16 tensor map of rank 4 or 5 (unit element strides, no interleave, 128-byte L2 promotion, zero fill out of bounds).
// `strides` are the byte strides of dims 1..rank-1.  On failure the error names the map (`what`), its extents and strides.
int encode_map(CUtensorMap* map, const char* what, const void* base, int rank, const cuuint64_t* dims,
               const cuuint64_t* strides, const cuuint32_t* box, CUtensorMapSwizzle swz);
// The dense NHWC map: dims {c, w, h, n}, box {box_c, box_w, box_h, 1}, swizzle_for(box_c)
int encode_nhwc(CUtensorMap* map, const char* what, const void* base, int c, int w, int h, int n, int box_c, int box_w,
                int box_h);

// cudaLaunchKernelEx with programmatic stream serialization (`pdl`) and clusters of `cluster_x` CTAs along x
template <typename Params>
int launch_ex(void (*kernel)(Params), const Params& args, dim3 grid, dim3 block, int smem, cudaStream_t stream, bool pdl,
              int cluster_x) {
    cudaLaunchAttribute attr[2];
    int na = 0;
    if (pdl) {
        attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[na].val.programmaticStreamSerializationAllowed = 1;
        ++na;
    }
    if (cluster_x > 1) {
        attr[na].id = cudaLaunchAttributeClusterDimension;
        attr[na].val.clusterDim.x = cluster_x;
        attr[na].val.clusterDim.y = 1;
        attr[na].val.clusterDim.z = 1;
        ++na;
    }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cfg.attrs = attr;
    cfg.numAttrs = na;
    VSRB_CUDA(cudaLaunchKernelEx(&cfg, kernel, args));
    VSRB_LAUNCH_CHECK();
    return VSRB_OK;
}

// ---------------------------------------------------------------------------------------
// conv geometry shared by packer and launchers
// ---------------------------------------------------------------------------------------
struct SegPlan {
    int c;         // real channels
    int cpad;      // padded to 16
    int ck;        // channels per K chunk: 16, 32 or 64   (tensor-core path)
    int chunks;    // cpad / ck
    int rowbytes;  // ck * 2: the shared-memory row of one pixel / one filter row
    int swz_mask;  // 1, 3, 7  (bits of addr>>7 XORed into addr>>4)
    int layout;    // UMMA layout_type: 6 (32B), 4 (64B), 2 (128B)
    int off;       // offset on the OIHW input-channel axis
};

struct ConvPlan {
    int kh, kw, n_seg, groups, pixshuf, dtype;
    SegPlan seg[4];
    int cin_packed;        // sum of real segment channels (fp32 path K extent per tap)
    int cout, cout_pad;    // cout_pad = round_up(cout, 16)
    int n_tile, n_blocks;  // tensor-core path: output channels per CTA, CTAs along N
    int stacked, ns;       // stacked layout: kw filter columns side by side along the MMA N (ns = kw*n_tile)
    int stages_per_tile;   // sum over segments of chunks*kw
    int b_stage_bytes[4];  // kh * n_tile * rowbytes
    size_t wblock_bytes;   // packed weights of one (group, n_block)
    size_t bias_bytes;     // groups*cout_pad floats rounded to 1 KiB
    size_t total_bytes;
    int ring;              // 3x3 bf16 conv to 64 channels that conv_ring_kernel can run: a second weight image follows the
                           // classic one.  Bit 1: a 64-channel segment (main operand), bit 2: a 3-channel segment (patch operand)
    int ring_main_seg, ring_patch_seg;
    size_t ring_off;       // byte offset of the ring image: [group][cta rank]{ [kx][96 rows][128 B] | patch [32 rows][64 B] }
};

// conv_ring.cu: per (group, CTA rank) three filter-column tiles of 96 rows x 64 channels (see pack_ring_kernel), then
// the K = 32 im2col tile of a 3-channel segment (32 rows x 64 B)
#define VSRB_RING_W_MAIN (3 * 96 * 128)
#define VSRB_RING_W_PATCH (32 * 64)
#define VSRB_RING_W_BYTES (VSRB_RING_W_MAIN + VSRB_RING_W_PATCH)

int make_plan(const vsrb_conv_geom* g, ConvPlan* p);   // returns VSRB_OK or error

// ---------------------------------------------------------------------------------------
// epilogue shared by the tensor-core and the fp32 conv kernels
// ---------------------------------------------------------------------------------------
struct EpiParams {
    int mode, act;
    float slope;
    float act_k;          // act(v) = max(v, v*act_k): 1 = none, 0 = ReLU, slope = LeakyReLU
    int H, W;             // conv extent
    int cout_pad, cq;     // cq = cout/4 when pixshuf
    int pixshuf;
    void* out;
    int out_c;
    long long out_img_stride, out_group_stride;   // elements
    int imgs_per_group;
    int split;            // out / residual are split-bf16 [hi | lo]; half = out_c / 2 (res_c / 2)
    const void* res;
    int res_c;
    float* f32_io;
    const float* f32_in;
    int aux_h, aux_w;
    int sr_kind;          // EPI_SR output element: 0 fp32, 1 fp16, 2 uint8 = floor(clamp(v,0,1)*255 + 0.5) (VSRB_CONV_SR_*)
    const float* bias;    // [groups][cout_pad], packed channel order
};

#ifdef __CUDACC__

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
    __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ float2 unpack_bf16(uint32_t u) {
    __nv_bfloat162 t = *reinterpret_cast<__nv_bfloat162*>(&u);
    return __bfloat1622float2(t);
}

template <typename T> struct Act;   // activation storage helpers
template <> struct Act<__nv_bfloat16> {
    static constexpr int kDtype = VSRB_BF16;
    __device__ static void load16(const void* p, float (&v)[16]) {
        const uint4* q = reinterpret_cast<const uint4*>(p);
        uint4 a = __ldg(q), b = __ldg(q + 1);
        uint32_t u[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float2 f = unpack_bf16(u[i]);
            v[2 * i] = f.x;
            v[2 * i + 1] = f.y;
        }
    }
    __device__ static void store16(void* p, const float (&v)[16]) {
        uint4 a, b;
        a.x = pack_bf16(v[0], v[1]);   a.y = pack_bf16(v[2], v[3]);
        a.z = pack_bf16(v[4], v[5]);   a.w = pack_bf16(v[6], v[7]);
        b.x = pack_bf16(v[8], v[9]);   b.y = pack_bf16(v[10], v[11]);
        b.z = pack_bf16(v[12], v[13]); b.w = pack_bf16(v[14], v[15]);
        uint4* q = reinterpret_cast<uint4*>(p);
        q[0] = a;
        q[1] = b;
    }
    __device__ static void store_n(void* p, const float* v, int n) {   // n <= 16, generic
        __nv_bfloat16* q = reinterpret_cast<__nv_bfloat16*>(p);
        for (int i = 0; i < n; ++i) q[i] = __float2bfloat16_rn(v[i]);
    }
};
template <> struct Act<float> {
    static constexpr int kDtype = VSRB_F32;
    __device__ static void load16(const void* p, float (&v)[16]) {
        const float4* q = reinterpret_cast<const float4*>(p);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            float4 f = __ldg(q + i);
            v[4 * i] = f.x; v[4 * i + 1] = f.y; v[4 * i + 2] = f.z; v[4 * i + 3] = f.w;
        }
    }
    __device__ static void store16(void* p, const float (&v)[16]) {
        float4* q = reinterpret_cast<float4*>(p);
#pragma unroll
        for (int i = 0; i < 4; ++i) q[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
    }
    __device__ static void store_n(void* p, const float* v, int n) {
        float* q = reinterpret_cast<float*>(p);
        for (int i = 0; i < n; ++i) q[i] = v[i];
    }
};

// ATen upsample_bilinear2d(align_corners=False) source tap for one axis
__device__ __forceinline__ void up_tap(int dst, float scale, int in_size, int& i0, int& i1, float& l1) {
    float src = (dst + 0.5f) * scale - 0.5f;
    src = src < 0.f ? 0.f : src;
    i0 = (int)src;
    if (i0 > in_size - 1) i0 = in_size - 1;
    i1 = i0 + (i0 < in_size - 1 ? 1 : 0);
    l1 = src - (float)i0;
}

// bias of 16 consecutive packed channels (global memory copy of the packed bias)
__device__ __forceinline__ void epi_bias16(const EpiParams& e, int g, int n0, float (&v)[16]) {
    const float4* bp = reinterpret_cast<const float4*>(e.bias + (size_t)g * e.cout_pad + n0);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float4 f = __ldg(bp + i);
        v[4 * i] += f.x; v[4 * i + 1] += f.y; v[4 * i + 2] += f.z; v[4 * i + 3] += f.w;
    }
}

// Branch-free activation: act(v) = max(v, v * k) with k = 1 (none), 0 (ReLU), slope (LeakyReLU, slope <= 1)
__device__ __forceinline__ void epi_act16(const EpiParams& e, float (&v)[16]) {
    const float k = e.act_k;
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i], v[i] * k);
}

// EPI_SR in two halves so a caller can fetch the skip term before its accumulator is ready: the bilinear x(H/aux_h)
// upsample of the fp32 NCHW LR frame at HR pixel (y, x) (ATen align_corners=False taps) ...
__device__ __forceinline__ void epi_sr_up(const EpiParams& e, int b, int y, int x, float (&up)[3]) {
    const int ih = e.aux_h, iw = e.aux_w;
    const float sy = (float)ih / (float)e.H, sx = (float)iw / (float)e.W;
    int y0, y1, x0, x1;
    float ly, lx;
    up_tap(y, sy, ih, y0, y1, ly);
    up_tap(x, sx, iw, x0, x1, lx);
    const float hy = 1.f - ly, hx = 1.f - lx;
    const size_t iplane = (size_t)ih * iw;
    const float* lp = e.f32_in + (size_t)b * 3 * iplane;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float* cp = lp + c * iplane;
        const float a00 = __ldg(cp + y0 * iw + x0), a01 = __ldg(cp + y0 * iw + x1);
        const float a10 = __ldg(cp + y1 * iw + x0), a11 = __ldg(cp + y1 * iw + x1);
        up[c] = hy * (hx * a00 + lx * a01) + ly * (hx * a10 + lx * a11);
    }
}
// ... and the fp32 NCHW store of conv + skip
template <int N>
__device__ __forceinline__ void epi_sr_store(const EpiParams& e, int b, int y, int x, const float (&v)[N], const float (&up)[3]) {
    const size_t oplane = (size_t)e.H * e.W;
    const size_t o = (size_t)b * 3 * oplane + (size_t)y * e.W + x;
    if (e.sr_kind == 0) {
        float* op = e.f32_io + o;
#pragma unroll
        for (int c = 0; c < 3; ++c) op[c * oplane] = v[c] + up[c];
    } else if (e.sr_kind == 1) {
        __half* op = reinterpret_cast<__half*>(e.f32_io) + o;
#pragma unroll
        for (int c = 0; c < 3; ++c) op[c * oplane] = __float2half_rn(v[c] + up[c]);
    } else {   // what torchvision.utils.save_image stores (test.py:138-141): mul(255).add(0.5).clamp(0,255).to(uint8)
        uint8_t* op = reinterpret_cast<uint8_t*>(e.f32_io) + o;
#pragma unroll
        for (int c = 0; c < 3; ++c) op[c * oplane] = (uint8_t)fminf(fmaxf(__fadd_rn(__fmul_rn(v[c] + up[c], 255.f), 0.5f), 0.f), 255.f);   // two roundings, like torch
    }
}

// EPI_CLEAN / EPI_FLOW in two halves as well: the fp32 value the conv result is added to ...
__device__ __forceinline__ void epi_clean_fetch(const EpiParams& e, int b, int y, int x, float (&pre)[3]) {
    const size_t plane = (size_t)e.H * e.W;
    const float* xp = e.f32_io + (size_t)b * 3 * plane + (size_t)y * e.W + x;
#pragma unroll
    for (int c = 0; c < 3; ++c) pre[c] = xp[c * plane];
}
__device__ __forceinline__ void epi_flow_fetch(const EpiParams& e, int b, int y, int x, float (&pre)[3]) {
    const float2 f = __ldg(reinterpret_cast<const float2*>(e.f32_in) + ((size_t)b * e.H + y) * e.W + x);
    pre[0] = f.x; pre[1] = f.y; pre[2] = 0.f;
}
// ... and the stores (EPI_CLEAN: fp32 NCHW frame in place + its bf16 NHWC-16 shadow; EPI_FLOW: flow_up + relu(conv))
template <typename T>
__device__ __forceinline__ void epi_clean_store(const EpiParams& e, int b, int y, int x, const float (&v)[4], const float (&pre)[3]) {
    const size_t plane = (size_t)e.H * e.W;
    float* xp = e.f32_io + (size_t)b * 3 * plane + (size_t)y * e.W + x;
    float nv[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) nv[i] = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        nv[c] = pre[c] + v[c];
        xp[c * plane] = nv[c];
    }
    T* op = reinterpret_cast<T*>(e.out) + (((size_t)b * e.H + y) * e.W + x) * e.out_c;
    Act<T>::store16(op, nv);
}
__device__ __forceinline__ void epi_flow_store(const EpiParams& e, int b, int y, int x, const float (&v)[4], const float (&pre)[3]) {
    reinterpret_cast<float2*>(e.f32_io)[((size_t)b * e.H + y) * e.W + x] = make_float2(pre[0] + v[0], pre[1] + v[1]);
}

// One pixel (b,y,x), 16 consecutive packed output channels starting at n0 (multiple of 16);
// v = act(acc + bias) already applied by the caller.  `g` = weight group of image b.
// kResDone: the caller has already added the residual.
template <typename T, bool kResDone = false>
__device__ __forceinline__ void epi_store16(const EpiParams& e, int g, int b, int y, int x, int n0, float (&v)[16]) {
    if (e.mode == VSRB_EPI_NHWC) {
        int Y = y, X = x, OH = e.H, OW = e.W, c0 = n0;
        if (e.pixshuf) {
            int q = n0 / e.cq;
            c0 = n0 - q * e.cq;
            Y = 2 * y + (q >> 1);
            X = 2 * x + (q & 1);
            OH = 2 * e.H;
            OW = 2 * e.W;
        }
        if (!kResDone && e.res) {
            float r[16];
            size_t pix = ((size_t)b * OH + Y) * OW + X;
            Act<T>::load16(reinterpret_cast<const T*>(e.res) + pix * e.res_c + c0, r);
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] += r[i];
            if (e.split) {                       // split-bf16 residual: value = hi + lo
                Act<T>::load16(reinterpret_cast<const T*>(e.res) + pix * e.res_c + e.res_c / 2 + c0, r);
#pragma unroll
                for (int i = 0; i < 16; ++i) v[i] += r[i];
            }
        }
        long long o = (long long)g * e.out_group_stride + (long long)(b - g * e.imgs_per_group) * e.out_img_stride +
                      ((long long)Y * OW + X) * e.out_c + c0;
        if (e.split) {                           // split-bf16 output: hi = bf16(v), lo = bf16(v - hi)
            float hi[16], lo[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                hi[i] = __bfloat162float(__float2bfloat16_rn(v[i]));
                lo[i] = v[i] - hi[i];
            }
            Act<T>::store16(reinterpret_cast<T*>(e.out) + o, hi);
            Act<T>::store16(reinterpret_cast<T*>(e.out) + o + e.out_c / 2, lo);
            return;
        }
        Act<T>::store16(reinterpret_cast<T*>(e.out) + o, v);
    } else if (e.mode == VSRB_EPI_CLEAN) {
        if (n0 != 0) return;
        float nv[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) nv[i] = 0.f;
        size_t plane = (size_t)e.H * e.W;
        float* xp = e.f32_io + (size_t)b * 3 * plane + (size_t)y * e.W + x;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            float t = xp[c * plane] + v[c];
            xp[c * plane] = t;
            nv[c] = t;
        }
        size_t pix = ((size_t)b * e.H + y) * e.W + x;
        T* op = reinterpret_cast<T*>(e.out) + pix * e.out_c;
        if (e.split) {                           // refreshed frame as [hi 16 | lo 16]
            float hi[16], lo[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                hi[i] = __bfloat162float(__float2bfloat16_rn(nv[i]));
                lo[i] = nv[i] - hi[i];
            }
            Act<T>::store16(op, hi);
            Act<T>::store16(op + e.out_c / 2, lo);
        } else if (e.out_c >= 16) Act<T>::store16(op, nv);
        else Act<T>::store_n(op, nv, e.out_c);
    } else if (e.mode == VSRB_EPI_FLOW) {
        if (n0 != 0) return;
        size_t pix = ((size_t)b * e.H + y) * e.W + x;
        float2 f = __ldg(reinterpret_cast<const float2*>(e.f32_in) + pix);
        reinterpret_cast<float2*>(e.f32_io)[pix] = make_float2(f.x + v[0], f.y + v[1]);
    } else {   // VSRB_EPI_SR
        if (n0 != 0) return;
        float up[3];
        epi_sr_up(e, b, y, x, up);
        epi_sr_store(e, b, y, x, v, up);
    }
}
#endif  // __CUDACC__

// launchers implemented in the kernel translation units
int launch_conv_tc(const vsrb_conv_args* a, const ConvPlan& p, cudaStream_t s);
int launch_conv_f32(const vsrb_conv_args* a, const ConvPlan& p, cudaStream_t s);
bool ring_eligible(const vsrb_conv_args* a, const ConvPlan& p);
int launch_conv_ring(const vsrb_conv_args* a, const ConvPlan& p, cudaStream_t s);
int launch_pack(const vsrb_conv_geom* g, const ConvPlan& p, const float* w, int cin_total, const float* bias,
                void* packed, cudaStream_t s);
void fill_epi(const vsrb_conv_args* a, const ConvPlan& p, EpiParams* e);

}  // namespace vsrb
