/*
 * vsrb200.h — C-ABI of libvsrb200.so: the B200 (sm_100a) kernels behind the
 * Real-BasicVSR / BasicVSR hot path of santurini/vsrlab.
 *
 * The reference has no FFI of its own (it is pure PyTorch); every entry point
 * below replaces the stock torch library call(s) named in its comment, cited as
 * reference file:line relative to the reference repo root.  INTEGRATION.md shows
 * the ctypes stub a maintainer of the reference would add.
 *
 * Conventions
 *  - every function returns 0 on success, a negative VSRB_E_* code on failure;
 *    vsrb_last_error() returns a human-readable reason (thread-local).
 *  - all pointers are DEVICE pointers owned by the caller unless stated; the
 *    library never allocates, frees or synchronises; kernels are enqueued on the
 *    `stream` argument (a cudaStream_t passed as void*).
 *  - activations are NHWC ("channels-last"); `dtype` selects the activation
 *    element type AND the arithmetic path: VSRB_BF16 = bf16 operands, fp32
 *    accumulate, tcgen05/TMEM tensor-core implicit GEMM fed by TMA;
 *    VSRB_F32 = fp32 operands and accumulate on the FFMA pipes ("fp32 mode").
 *  - flows are fp32 channels-last [N,h,w,2] (x then y displacement, pixels),
 *    which is what the reference hands to flow_warp (basicvsr.py:54,69).
 */
#ifndef VSRB200_H
#define VSRB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VSRB_VERSION 101

/* error codes */
#define VSRB_OK            0
#define VSRB_E_ARG        -1   /* invalid argument / unsupported shape            */
#define VSRB_E_CUDA       -2   /* CUDA runtime / driver error                      */
#define VSRB_E_NODEVICE   -3   /* no sm_100 device / driver entry point missing    */
#define VSRB_E_SMEM       -4   /* tile does not fit shared memory / TMEM           */

/* dtypes */
#define VSRB_BF16 0
#define VSRB_F32  1
#define VSRB_BF16X2 2      /* layout kernels only: split-bf16, per pixel [hi C | lo C], value = hi + lo   */

/* activations fused in the conv epilogue */
#define VSRB_ACT_NONE  0
#define VSRB_ACT_RELU  1       /* reference conv.py:19,87 ; spynet.py:16-18        */
#define VSRB_ACT_LRELU 2       /* LeakyReLU(slope); reference conv.py:98           */

/* padding modes of the backward warp (reference spynet.py:95; F.grid_sample padding_mode) */
#define VSRB_PAD_ZEROS      0
#define VSRB_PAD_BORDER     1
#define VSRB_PAD_REFLECTION 2   /* vsrb_flow_warp_ex / _ex_bwd only */

/* interpolation modes of vsrb_flow_warp_ex (F.grid_sample mode) */
#define VSRB_INTERP_BILINEAR 0
#define VSRB_INTERP_NEAREST  1
#define VSRB_INTERP_BICUBIC  2

/* conv epilogues (what happens to acc + bias) */
#define VSRB_EPI_NHWC   0  /* act(acc+bias) [+ residual] -> NHWC `out`; with geom.pixshuf=2 the store
                              is the PixelShuffle(2) of the result (upsampling.py:10-12)                */
#define VSRB_EPI_CLEAN  1  /* 3-channel residue: x_nchw_f32 += acc+bias in place, and the refreshed
                              frame is also written NHWC for the next stem (realbasicvsr.py:28-29)      */
#define VSRB_EPI_FLOW   2  /* flow = flow_up + relu(acc+bias), fp32 [B,h,w,2] (spynet.py:56-65)         */
#define VSRB_EPI_SR     3  /* sr_nchw_f32 = acc+bias + bilinear_x4(lq) (basicvsr.py:81-82; ac=False)   */

/* vsrb_conv_args.flags */
#define VSRB_CONV_PDL 1    /* launch with programmatic dependent launch: the kernel's prologue (TMEM
                              allocation, barrier set-up, weight fetch) may overlap the tail of the previous
                              kernel on the stream; only legal when `packed` was complete before that
                              previous kernel was enqueued                                                */
#define VSRB_CONV_SR_F16 4 /* EPI_SR only: `f32_io` points to an fp16 [B,3,4h,4w] tensor (opt-in narrow output)   */
#define VSRB_CONV_SR_U8  2 /* EPI_SR only: `f32_io` points to a uint8 [B,3,4h,4w] tensor holding
                              floor(clamp(sr,0,1)*255 + 0.5): the bytes torchvision.utils.save_image writes
                              for the reference's PNG dump (test.py:138-141)                               */

/* Geometry of one convolution's weights: everything the packer and the launcher
 * must agree on.  Stride 1, 'same' padding (kh//2, kw//2), dilation 1. */
typedef struct vsrb_conv_geom {
    int32_t kh, kw;         /* 1, 3 or 7                                                        */
    int32_t n_seg;          /* 1..4 weight segments (a fused torch.cat along channels)          */
    int32_t seg_c[4];       /* real channels of each segment                                    */
    int32_t seg_off[4];     /* where the segment sits on the OIHW input-channel axis            */
    int32_t cout;           /* real output channels                                             */
    int32_t pixshuf;        /* 0, or 2 = output channel 4c+2i+j is stored at pixel (2y+i,2x+j)  */
    int32_t groups;         /* independent weight sets applied to consecutive image groups      */
    int32_t dtype;          /* VSRB_BF16 or VSRB_F32                                            */
    int32_t transpose;      /* 1 = pack the input-gradient conv of `w`: channels swapped, filter
                               flipped; then seg_c[0] = forward cout, cout = forward cin and
                               cin_total passed to the packer = forward cout                      */
} vsrb_conv_geom;

typedef struct vsrb_conv_args {
    vsrb_conv_geom geom;
    int32_t      n_in;        /* 0: in[s] is the input of weight segment s.  Otherwise the number of
                                 input OPERANDS (<= 6): operand i multiplies weight segment in_wseg[i]
                                 and reads geom.seg_c[in_wseg[i]] channels of in[i] starting at channel
                                 in_c0[i].  Several operands may share one weight segment - the
                                 split-bf16 fp32 mode feeds (hi, W_hi), (lo, W_hi), (hi, W_lo).       */
    const void*  in[6];       /* NHWC inputs                                                     */
    int32_t      in_c[6];     /* channels allocated per pixel in in[i]                           */
    int32_t      in_c0[6];    /* first channel of operand i inside in[i] (n_in > 0)              */
    int32_t      in_wseg[6];  /* weight segment of operand i (n_in > 0)                          */
    int32_t      batch, h, w; /* input (== pre-shuffle output) extent                            */
    int32_t      imgs_per_group; /* images per weight group (batch = groups*imgs_per_group)      */
    const void*  packed;      /* buffer written by vsrb_pack_conv_weight                         */
    int32_t      act;         /* VSRB_ACT_*                                                      */
    float        slope;       /* LeakyReLU slope                                                 */
    int32_t      epilogue;    /* VSRB_EPI_*                                                      */
    void*        out;         /* EPI_NHWC: NHWC output (dtype); EPI_CLEAN: NHWC refreshed frame  */
    int32_t      out_c;       /* channels allocated per pixel in `out`.  EPI_NHWC: a multiple of 8
                                 (of 16 with `split`).  EPI_CLEAN: 3..16, or exactly 32 with
                                 `split`; `out` must be 16-byte aligned when out_c == 16 or split */
    int64_t      out_img_stride;   /* EPI_NHWC: elements between consecutive images of a group in
                                      `out` (0 = dense); lets a step write straight into frame t
                                      of a [N,T,h,w,C] feature bank                               */
    int64_t      out_group_stride; /* EPI_NHWC: elements between the first images of two groups   */
    const void*  residual;    /* EPI_NHWC: optional NHWC tensor added after act (same extent)    */
    int32_t      res_c;
    float*       f32_io;      /* EPI_CLEAN: x [B,3,h,w] updated in place; EPI_FLOW: flow out
                                 [B,h,w,2]; EPI_SR: sr [B,3,4h,4w]                               */
    const float* f32_in;      /* EPI_FLOW: flow_up [B,h,w,2]; EPI_SR: lq [B,3,aux_h,aux_w]       */
    int32_t      aux_h, aux_w;/* EPI_SR: extent of the low-resolution skip frame                 */
    int32_t      max_ctas;    /* 0 = one persistent CTA per SM                                   */
    int32_t      flags;       /* VSRB_CONV_* bits                                                */
    int32_t      split;       /* 1: `out`, `residual` (and the EPI_CLEAN frame) are split-bf16: per pixel
                                 [hi C | lo C] with C = out_c/2, value = hi + lo.  The stores move
                                 16 channels at a time, so out_c and res_c must be multiples of 16;
                                 the EPI_CLEAN frame is [hi 16 | lo 16] (out_c = 32).  Anything
                                 else returns VSRB_E_ARG                                          */
    /* Optional fast operand for a 3-channel 3x3 segment (the image stems 3 -> 64 and 64+3 -> 64: conv.py:97-98 behind
     * realbasicvsr.py:21 and basicvsr.py:56,71): the frames as 3x3 im2col patches, bf16 [.,h,w,32] written by
     * vsrb_im2col3x3_c3.  When given (and the launch is large enough) the ring-walk kernel multiplies the whole
     * 27-tap neighbourhood as ONE K = 32 chunk instead of nine K = 16 chunks of mostly padding.  Image li of weight
     * group g starts at patch + g * patch_group_stride + li * patch_img_stride (elements; strides may be negative:
     * the two propagation directions walk the clip in opposite orders; both 0 = dense).  in[] of that segment must
     * still be valid (launches the ring-walk kernel does not take use it).                                        */
    const void*  patch;
    int64_t      patch_img_stride, patch_group_stride;
} vsrb_conv_args;

/* ---- library ------------------------------------------------------------------------- */
int         vsrb_version(void);
const char* vsrb_last_error(void);
/* sm count / compute capability of the current device */
int         vsrb_device_info(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor);
/* number of kernels this library has launched since load (bench.py's gpu_launches) */
int64_t     vsrb_launch_count(void);
/* 0 if no kernel reported a pipeline time-out since the last call (debug aid) */
int         vsrb_debug_status(void* stream);
/* debug aid: with VSRB_TC_DEBUG bit 64 set, every CTA of a tensor-core conv records %globaltimer stamps (ns) of its
 * pipeline milestones (8 per CTA: entry, prologue done, weights resident, first tile loaded, first accumulator ready,
 * last tile stored, stores drained, exit); copies the first `n_ctas` CTAs' stamps of the last launch to `out[n_ctas*8]` */
int         vsrb_debug_trace(uint64_t* out, int32_t n_ctas);

/* debug aid: with VSRB_RING_DEBUG bit 64 set, CTA (0,0) of every ring-walk conv adds up clock cycles: out[0] MMA issuer waiting
 * for a free accumulator slot, [1] waiting for operand rows, [2] steps issued, [3] epilogue warp waiting for finished rows,
 * [4] epilogue work                                                                                                    */
int         vsrb_ring_debug_stats(uint64_t* out, int32_t reset);

/* ---- convolution: replaces nn.Conv2d -> F.conv2d (+ the pointwise op that follows it) --
 * reference: conv.py:89-92,101-103 (ResidualConv/ResidualBlock), conv.py:21 (ConvReLU),
 * upsampling.py:10-12 (PixelShufflePack), basicvsr.py:75-82 (point_conv, conv_last, skip),
 * realbasicvsr.py:28-29 (cleaner residue), spynet.py:56-65 (SpynetModule + flow add).   */
size_t vsrb_packed_weight_bytes(const vsrb_conv_geom* g);
/* w: fp32 OIHW [groups][cout][cin_total][kh][kw] on device (cin_total = the conv's real
 * in_channels; segments index into it), bias: fp32 [groups][cout] or NULL.             */
int    vsrb_pack_conv_weight(const vsrb_conv_geom* g, const float* w, int32_t cin_total,
                             const float* bias, void* packed, void* stream);
int    vsrb_conv2d_fwd(const vsrb_conv_args* a, void* stream);
/* How the library will tile this geometry (diagnostics / tests): info = {stacked, n_tile, n_blocks,
 * mma_n, k_chunk of segment 0, k_chunk of segment 1, pipeline stages per tile, weight KiB per block} */
int    vsrb_conv_plan_info(const vsrb_conv_geom* g, int32_t info[8]);

/* ---- training (backward of the path; reference: autograd through the same modules) -------
 * input gradient of a conv: vsrb_conv2d_fwd on the output gradient with weights packed with
 * geom.transpose = 1.  Weight/bias gradient: dw [cout][cin_total][kh][kw] and db [cout] (or
 * NULL) are fp32, ACCUMULATED into (zero them first); `g` is the forward geometry (groups = 1,
 * imgs_per_group = batch), in[]/in_c[] the forward inputs, dz the gradient wrt the conv output
 * before the activation, NHWC with dz_c >= cout channels per pixel.  in[] and dz 16-byte
 * aligned, in_c[] and dz_c multiples of 8.  Kernels: bf16 3x3 segments of a multiple of 64
 * channels (cout > 16) and bf16 odd square filters up to 7x7 on the tensor cores; fp32 data
 * and bf16 non-square filters of width 1, 3 or 7 on the FFMA kernel.  Anything else is
 * refused with VSRB_E_ARG before any work is enqueued.                                    */
int vsrb_conv2d_wgrad(const vsrb_conv_geom* g, const void* const* in, const int32_t* in_c, const void* dz,
                      int32_t dz_c, int32_t batch, int32_t h, int32_t w, int32_t imgs_per_group,
                      int32_t cin_total, float* dw, float* db, void* stream);
/* the same gradient summed over n_chunks (x, dz) pairs of one shape - the uses of a recurrent conv at different time
 * steps (basicvsr.py:46-73 applies the same resblocks at every frame) - in one launch per 64-channel block:
 * in[k * n_seg + s] = input segment s of chunk k, dz[k] = its output gradient, `batch` images per chunk.
 * bf16, 3x3, ungrouped, segments of a multiple of 64 channels (the tensor-core path); other shapes: concatenate. */
int vsrb_conv2d_wgrad_multi(const vsrb_conv_geom* g, int32_t n_chunks, const void* const* in, const int32_t* in_c,
                            const void* const* dz, int32_t dz_c, int32_t batch, int32_t h, int32_t w,
                            int32_t cin_total, float* dw, float* db, void* stream);
/* backward of vsrb_flow_warp: dx (fp32 [n,h,w,c], accumulated with atomics, zero it first; or
 * NULL) and dflow (fp32 [n,h,w,2], overwritten; or NULL; needs the forward input x).        */
int vsrb_flow_warp_bwd(const void* x, const float* flow, const void* dout, float* dx, float* dflow,
                       int32_t n, int32_t h, int32_t w, int32_t c, int32_t dtype, int32_t padding_mode,
                       void* stream);

/* ---- deterministic gradients (torch.use_deterministic_algorithms) ----------------------
 * The same gradients with a fixed order of every floating-point addition: two calls on the same inputs, on a GPU with the
 * same SM count, give bit-identical results.  The library allocates nothing: the caller passes a device workspace of at
 * least the bytes its *_workspace_bytes query returns (16-byte aligned; 0 from a query = refused arguments, see
 * vsrb_last_error).  Nothing synchronises the host, so the calls can be captured in CUDA graphs.  Arguments, including a
 * workspace that is too small, are refused with VSRB_E_ARG before any work is enqueued.
 * vsrb_conv2d_wgrad(_multi)_det: the contract of vsrb_conv2d_wgrad(_multi) (dw, db accumulated); every CTA stores its
 * partial block to its own workspace slot and one kernel adds the slots in slot order.  Refused: the geometries of the
 * FFMA fallback (fp32 data, non-square filters).  The query takes the forward geometry, the chunk count (1 = the plan of
 * vsrb_conv2d_wgrad_det) and whether db is computed.                                                                  */
size_t vsrb_conv2d_wgrad_det_workspace_bytes(const vsrb_conv_geom* g, int32_t n_chunks, int32_t batch, int32_t h, int32_t w,
                                             int32_t with_bias);
int vsrb_conv2d_wgrad_det(const vsrb_conv_geom* g, const void* const* in, const int32_t* in_c, const void* dz,
                          int32_t dz_c, int32_t batch, int32_t h, int32_t w, int32_t imgs_per_group,
                          int32_t cin_total, float* dw, float* db, void* workspace, size_t workspace_bytes, void* stream);
int vsrb_conv2d_wgrad_multi_det(const vsrb_conv_geom* g, int32_t n_chunks, const void* const* in, const int32_t* in_c,
                                const void* const* dz, int32_t dz_c, int32_t batch, int32_t h, int32_t w,
                                int32_t cin_total, float* dw, float* db, void* workspace, size_t workspace_bytes,
                                void* stream);
/* vsrb_flow_warp_bwd with dx OVERWRITTEN (fp32 [n,h,w,c], or NULL): the taps' contributions are summed as 64-bit
 * fixed-point integers scaled from max|dout|; a non-finite dout makes all of dx NaN.  dflow (or NULL) is the output of
 * vsrb_flow_warp_bwd itself (single writer per pixel); it needs c / (8 bf16 | 4 fp32) to be a power of two <= 32.
 * padding_mode zeros or border.  The workspace is needed for dx only.                                                 */
size_t vsrb_flow_warp_bwd_det_workspace_bytes(int32_t n, int32_t h, int32_t w, int32_t c);
int vsrb_flow_warp_bwd_det(const void* x, const float* flow, const void* dout, float* dx, float* dflow,
                           int32_t n, int32_t h, int32_t w, int32_t c, int32_t dtype, int32_t padding_mode,
                           void* workspace, size_t workspace_bytes, void* stream);

/* ---- backward warp: replaces flow_warp = meshgrid + normalise + F.grid_sample ---------
 * reference: spynet.py:95-106; callers basicvsr.py:54,69.
 * x,out: NHWC [n,h,w,c] of `dtype`, c % 8 == 0; flow fp32 [n,h,w,2].                    */
int vsrb_flow_warp(const void* x, int64_t x_img_stride /* elements, 0 = dense */, const float* flow,
                   int64_t flow_img_stride /* float2 elements, 0 = dense */, void* out, int32_t n,
                   int32_t h, int32_t w, int32_t c, int32_t dtype, int32_t padding_mode, void* stream);

/* the same for `groups` x `imgs_per_group` images in ONE launch: image li of group g reads x + g * x_group_stride + li *
 * x_img_stride (elements) and flow + g * flow_group_stride + li * flow_img_stride (float2 elements; group strides may be
 * negative), out is dense [groups * imgs_per_group, h, w, c].  The two propagation directions of a time step
 * (basicvsr.py:52-54 and :66-69) warp different frames of the feature bank with different flow fields.  bf16 only.     */
int vsrb_flow_warp_groups(const void* x, int64_t x_img_stride, int64_t x_group_stride, const float* flow,
                          int64_t flow_img_stride, int64_t flow_group_stride, void* out, int32_t imgs_per_group,
                          int32_t groups, int32_t h, int32_t w, int32_t c, int32_t dtype, int32_t padding_mode, void* stream);

/* vsrb_flow_warp with every F.grid_sample mode the reference flow_warp accepts (spynet.py:95-106 passes them through):
 * interp VSRB_INTERP_*, padding_mode VSRB_PAD_* (reflection included), align_corners 0 / 1.  The pixel position
 * (x + fx, y + fy) is normalised with max(size-1, 1) whatever align_corners is, as the reference does, and
 * grid_sample's un-normalisation is applied to that.  dtype VSRB_BF16 (c % 8 == 0) or VSRB_F32 (c % 4 == 0);
 * (bilinear, zeros | border, align_corners = 1) runs vsrb_flow_warp itself, and then VSRB_BF16X2 is accepted too.   */
int vsrb_flow_warp_ex(const void* x, int64_t x_img_stride, const float* flow, int64_t flow_img_stride, void* out,
                      int32_t n, int32_t h, int32_t w, int32_t c, int32_t dtype, int32_t interp,
                      int32_t padding_mode, int32_t align_corners, void* stream);
/* backward of vsrb_flow_warp_ex; the contract of vsrb_flow_warp_bwd (dx accumulated, dflow overwritten).  nearest:
 * dflow = 0, as grid_sample's.  (bilinear, zeros | border, align_corners = 1) runs vsrb_flow_warp_bwd itself.      */
int vsrb_flow_warp_ex_bwd(const void* x, const float* flow, const void* dout, float* dx, float* dflow,
                          int32_t n, int32_t h, int32_t w, int32_t c, int32_t dtype, int32_t interp,
                          int32_t padding_mode, int32_t align_corners, void* stream);

/* ---- layout: module-boundary NCHW fp32 <-> internal NHWC ------------------------------
 * (the reference keeps NCHW throughout; these sit at the nn.Module boundary)            */
int vsrb_nchw_to_nhwc(const float* src, void* dst, int32_t n, int32_t c, int32_t h, int32_t w,
                      int32_t c_dst, int32_t dtype, void* stream);   /* channels >= c are zeroed */
int vsrb_nhwc_to_nchw(const void* src, float* dst, int32_t n, int32_t c, int32_t h, int32_t w,
                      int32_t c_src, int32_t dtype, void* stream);
/* 3x3 im2col of 3-channel fp32 NCHW frames [n,3,h,w] -> bf16 [n,h,w,32]: element (ky*3+kx)*3 + c of pixel (y,x) is
 * frame[c, y+ky-1, x+kx-1] (zero outside the image), elements 27..31 are zero.  Feeds vsrb_conv_args.patch.        */
int vsrb_im2col3x3_c3(const float* frames, void* patches, int32_t n, int32_t h, int32_t w, void* stream);
/* inverse of nn.PixelShuffle(2) (upsampling.py:10-12) on bf16 NHWC, for the backward pass of the upsampling convs:
 * src [n, 2h, 2w, c] -> dst [n, h, w, 4c] with dst channel 4*cc + 2*i + j = src pixel (2y+i, 2x+j), channel cc */
int vsrb_pixel_unshuffle2(const void* src, void* dst, int32_t n, int32_t h, int32_t w, int32_t c, void* stream);

/* ---- SPyNet glue ------------------------------------------------------------------------
 * reference spynet.py:38-48 (normalise + 5x avg_pool2d), :71-80 (resize to /32),
 * :54-61 (x2 flow upsample, border warp, concat), :83-91 (resize back + rescale).       */
/* frames [F,3,h,w] fp32 NCHW -> finest pyramid level [F,Hp,Wp,4] fp32 (r,g,b,0), normalised
 * by mean/std (host floats), resized bilinear align_corners=False when (Hp,Wp)!=(h,w). */
int vsrb_spynet_pyramid_base(const float* frames, float* lvl, int32_t F, int32_t h, int32_t w,
                             int32_t Hp, int32_t Wp, const float* mean3, const float* std3, void* stream);
/* 2x2 average pool of an [F,H,W,4] fp32 level into [F,H/2,W/2,4] */
int vsrb_avgpool2_c4(const float* in, float* out, int32_t F, int32_t H, int32_t W, void* stream);
/* One pyramid level's network input.  pair p uses frames ref_idx[p], supp_idx[p] (device
 * int32 arrays).  flow_prev [P,Hl/2,Wl/2,2] or NULL (level 0: zero flow).  Writes
 * flow_up [P,Hl,Wl,2] fp32 = 2*up2(flow_prev) (align_corners=True) and the 8-channel
 * input (ref rgb, border-warped supp rgb, flow_up xy) into conv_in [P,Hl,Wl,c_in], padded
 * with zeros to c_in channels.                                                          */
int vsrb_spynet_level_input(const float* lvl, const int32_t* ref_idx, const int32_t* supp_idx,
                            const float* flow_prev, float* flow_up, void* conv_in,
                            int32_t P, int32_t Hl, int32_t Wl, int32_t c_in, int32_t dtype, void* stream);
/* flow [P,Hp,Wp,2] -> [P,h,w,2], bilinear align_corners=False, x*=w/Wp, y*=h/Hp */
int vsrb_flow_resize(const float* flow_in, float* flow_out, int32_t P, int32_t Hp, int32_t Wp,
                     int32_t h, int32_t w, void* stream);

/* ---- training objective and evaluation metrics of the callers (next rows of the path) -------
 * reference: CharbonnierLoss (core/losses.py:10-18), compute_loss (core/utils.py:235-240: the second term compares
 * lq with kornia `resize(hr, (h, w))` = bilinear, align_corners=False), compute_metric (core/utils.py:242-247) with
 * piqa.PSNR / piqa.SSIM (conf/train/default.yaml:9-15).  Reductions ACCUMULATE into device doubles the caller zeroes;
 * nothing is synchronised, no scalar travels to the host.                                                         */
/* *sum += sum_i sqrt((x_i-y_i)^2 + eps); if grad: grad_i = s * (x_i-y_i)/sqrt(...), s = grad_scale * (*grad_scale_dev
 * if not NULL): the backward pass passes the upstream gradient as a device scalar and 1/n as grad_scale.          */
int vsrb_charbonnier(const float* x, const float* y, int64_t n, float eps, double* sum, float* grad,
                     const float* grad_scale_dev, float grad_scale, void* stream);
/* the same for lq [planes,h,w] against hr [planes,H,W] resized to (h,w) on the fly; grad is d/d lq                */
int vsrb_charbonnier_resized(const float* lq, const float* hr, int32_t planes, int32_t h, int32_t w, int32_t H,
                             int32_t W, float eps, double* sum, float* grad, const float* grad_scale_dev,
                             float grad_scale, void* stream);
/* sums[i] += sum over image i of (clamp(x,0,1) - y)^2 (piqa.PSNR on core/utils.py:244's clamped frames)           */
int vsrb_psnr_sums(const float* x, const float* y, int32_t images, int64_t per_image, double* sums, void* stream);
/* sums[i] += sum of the SSIM map of image i (x,y [images,channels,h,w]; 11x11 Gaussian window sigma 1.5, 'valid'
 * borders, k1 0.01, k2 0.03, value range 1 = piqa.SSIM defaults); the map has channels*(h-10)*(w-10) entries      */
int vsrb_ssim_sums(const float* x, const float* y, int32_t images, int32_t channels, int32_t h, int32_t w,
                   int32_t clamp_x, double* sums, void* stream);
/* the same four with each block's sum stored to a workspace slot and the slots added in block order (deterministic
 * sums, see "deterministic gradients" above); the queries take the shape arguments of their entry point           */
size_t vsrb_charbonnier_det_workspace_bytes(int64_t n);
size_t vsrb_charbonnier_resized_det_workspace_bytes(int32_t planes, int32_t h, int32_t w);
size_t vsrb_psnr_sums_det_workspace_bytes(int32_t images, int64_t per_image);
size_t vsrb_ssim_sums_det_workspace_bytes(int32_t images, int32_t channels, int32_t h, int32_t w);
int vsrb_charbonnier_det(const float* x, const float* y, int64_t n, float eps, double* sum, float* grad,
                         const float* grad_scale_dev, float grad_scale, void* workspace, size_t workspace_bytes,
                         void* stream);
int vsrb_charbonnier_resized_det(const float* lq, const float* hr, int32_t planes, int32_t h, int32_t w, int32_t H,
                                 int32_t W, float eps, double* sum, float* grad, const float* grad_scale_dev,
                                 float grad_scale, void* workspace, size_t workspace_bytes, void* stream);
int vsrb_psnr_sums_det(const float* x, const float* y, int32_t images, int64_t per_image, double* sums,
                       void* workspace, size_t workspace_bytes, void* stream);
int vsrb_ssim_sums_det(const float* x, const float* y, int32_t images, int32_t channels, int32_t h, int32_t w,
                       int32_t clamp_x, double* sums, void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VSRB200_H */
