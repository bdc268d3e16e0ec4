// Sample coordinates of the F.grid_sample modes behind vsrb_flow_warp_ex (forward, warp.cu) and vsrb_flow_warp_ex_bwd
// (train.cu): fp32 restatements of ATen's grid_sampler_unnormalize, grid_sampler_compute_source_index (nearest,
// bilinear: padding applied to the sample coordinate) and get_value_bounded (bicubic: padding applied to every tap),
// with the gradient multipliers of their _set_grad variants.
#pragma once
#include "common.cuh"

namespace vsrb {

// pixel position p (x + fx) -> the coordinate grid_sample samples at.  The reference normalises with max(size-1, 1)
// whatever align_corners is; grid_sample un-normalises with (size-1) (align_corners) or size (not).  With
// align_corners this is sample_pos() of warp.cu operation for operation.
__device__ __forceinline__ float ex_unnormalize(float p, int size, int align) {
    const float g = 2.0f * p / (float)max(size - 1, 1) - 1.0f;
    return align ? (g + 1.0f) / 2.0f * (float)(size - 1) : ((g + 1.0f) * (float)size - 1.0f) / 2.0f;
}

// d ex_unnormalize / d p: 1 (align_corners, size > 1), 0 (align_corners, size 1), size / max(size-1, 1) (not)
__device__ __forceinline__ float ex_unnormalize_grad(int size, int align) {
    return (float)(align ? size - 1 : size) / (float)max(size - 1, 1);
}

// clip to [0, size-1]; g = 0 where clipped (the bounds included, as ATen's clip_coordinates_set_grad)
__device__ __forceinline__ float ex_clip(float c, int size, float& g) {
    const float hi = (float)(size - 1);
    if (c <= 0.f) { g = 0.f; return 0.f; }
    if (c >= hi) { g = 0.f; return hi; }
    g = 1.f;
    return c;
}

// reflect over [twice_low / 2, twice_high / 2] as often as needed; g = +-1
__device__ __forceinline__ float ex_reflect(float c, int twice_low, int twice_high, float& g) {
    if (twice_low == twice_high) { g = 0.f; return 0.f; }
    const float lo = (float)twice_low / 2.f, span = (float)(twice_high - twice_low) / 2.f;
    c -= lo;
    float s = 1.f;
    if (c < 0.f) { s = -1.f; c = -c; }
    const float extra = fmodf(c, span);
    const float flips = floorf(c / span);           // parity taken in float: no int conversion of a wild value
    if (fmodf(flips, 2.f) == 0.f) { g = s; return extra + lo; }
    g = -s;
    return span - extra + lo;
}

// padding of a sample coordinate (grid_sampler_compute_source_index_set_grad without the un-normalisation); g is its
// derivative.  Non-finite and out-of-int-range results become -100 (ATen's safe_downgrade_to_int_range): they read zero.
__device__ __forceinline__ float ex_pad_coord(float c, int size, int pad, int align, float& g) {
    g = 1.f;
    if (pad == VSRB_PAD_BORDER) {
        c = ex_clip(c, size, g);
    } else if (pad == VSRB_PAD_REFLECTION) {
        float gr, gc;
        c = align ? ex_reflect(c, 0, 2 * (size - 1), gr) : ex_reflect(c, -1, 2 * size - 1, gr);
        c = ex_clip(c, size, gc);
        g = gr * gc;
    }
    if (!(fabsf(c) <= 2.0e9f)) c = -100.f;
    return c;
}

// integer index of a padded coordinate (truncated as ATen's int64 cast), or -1 when it lies outside [0, size)
__device__ __forceinline__ int ex_index(float c, int size) {
    return (c > -1.f && c < (float)size) ? (int)c : -1;
}

// one bicubic tap at integer coordinate c, padded on its own (get_value_bounded): index or -1
__device__ __forceinline__ int ex_bicubic_tap(float c, int size, int pad, int align) {
    float g;
    return ex_index(ex_pad_coord(c, size, pad, align, g), size);
}

// cubic convolution weights (A = -0.75) of the taps at floor - 1 .. floor + 2 for the fraction t, and their d / dt
static constexpr float kCubicA = -0.75f;
__device__ __forceinline__ float cubic_conv1(float x) { return ((kCubicA + 2.f) * x - (kCubicA + 3.f)) * x * x + 1.f; }
__device__ __forceinline__ float cubic_conv2(float x) { return ((kCubicA * x - 5.f * kCubicA) * x + 8.f * kCubicA) * x - 4.f * kCubicA; }
__device__ __forceinline__ float cubic_conv1_d(float x) { return (3.f * (kCubicA + 2.f) * x - 2.f * (kCubicA + 3.f)) * x; }
__device__ __forceinline__ float cubic_conv2_d(float x) { return (3.f * kCubicA * x - 10.f * kCubicA) * x + 8.f * kCubicA; }

__device__ __forceinline__ void cubic_weights(float t, float (&c)[4]) {
    c[0] = cubic_conv2(t + 1.f);
    c[1] = cubic_conv1(t);
    c[2] = cubic_conv1(1.f - t);
    c[3] = cubic_conv2(2.f - t);
}
__device__ __forceinline__ void cubic_weights_grad(float t, float (&d)[4]) {
    d[0] = cubic_conv2_d(t + 1.f);
    d[1] = cubic_conv1_d(t);
    d[2] = -cubic_conv1_d(1.f - t);
    d[3] = -cubic_conv2_d(2.f - t);
}

}  // namespace vsrb
