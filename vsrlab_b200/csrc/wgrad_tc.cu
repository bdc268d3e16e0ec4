// Weight gradient of the 3x3, 64-input-channel convolutions on the tensor cores (tcgen05 + TMEM, TMA fed).
//
//   dW[tap][ci][co] = sum over pixels p of  x[p + tap][ci] * dz[p][co]
//
// is a GEMM whose K dimension is the pixel index.  Both operands are "MN-major" for UMMA: a TMA box of
// pixels x 64 channels lands in shared memory as rows of 128 bytes (128B swizzle) = K rows of 64
// contiguous M (resp. N) elements, which is exactly the canonical MN-major layout, so no transpose is needed:
//   A (M side) = the activation x, shifted by the filter tap.  ONE halo box of (4 + 2) rows x (16 + 2) pixels per tile:
//                an MN-major SW128 operand may start at any 128-byte K row of its tile (tools/umma_mn_offset_test.cu: the
//                hardware swizzles on absolute address bits), so tap (ky, kx) of K step ks is simply the 16 consecutive
//                pixels that start at pixel ((ky + ks) * 18 + kx) of the box.  (Round 1 loaded three kx-shifted copies, 2.7x
//                the unique bytes.  Measured after the change: same 85 us for 120 x 64x64 images - VSRB_WG_DEBUG shows the
//                kernel is MMA-ISSUE bound, not load bound: twenty N = 64 MMAs of ~96 cycles per 64-pixel tile = 1.1 us,
//                57 us with the final atomics skipped and no MMAs at all.)  Two taps are issued as ONE M=128 MMA:
//                the descriptor's leading-dimension byte offset (the distance between consecutive 64-element M blocks)
//                points from the first tap's window to the second tap's window (one pixel, or one box row).
//   B (N side) = the output gradient dz (N = 64 output channels).
//   D          = five accumulators of 128 x 64 fp32 in TMEM (9 taps = 4 pairs + 1 single), kept for the whole
//                persistent CTA; K advances 16 pixels (2048 bytes) per MMA.
// Every pixel tile is read once; at the end each CTA adds its partial dW into the fp32 OIHW gradient with atomics, or, for
// deterministic gradients, stores it to its own slot of a workspace that slot_reduce_kernel then sums in slot order.
// Replaces the wgrad half of autograd's ConvolutionBackward0 for the hot 64->64 / 64->256 3x3 layers.
#include "common.cuh"
#include "tc_ptx.cuh"

namespace vsrb {

static constexpr int kWgThreads = 256;
static constexpr int kWgTW = 16, kWgRows = 4;                               // 64-pixel tiles: four K=16 steps
static constexpr int kWgXW = kWgTW + 2;                                     // halo box width in pixels
static constexpr int kWgXBytes = (kWgRows + 2) * kWgXW * 128;               // the halo box: 13.5 KiB
static constexpr int kWgCopyBytes = 14 * 1024;                              // ... padded so that the dz tile stays 1 KiB aligned
static constexpr int kWgZBytes = kWgRows * kWgTW * 128;                     // dz tile: 8 KiB
static constexpr int kWgStageBytes = kWgCopyBytes + kWgZBytes;              // 22 KiB
static constexpr int kWgStages = 8;
static constexpr int kWgSmem = 1024 + 1024 + kWgStages * kWgStageBytes;

static constexpr int kWgMaxChunks = 16;
struct WgTcParams {
    // One launch may sum over up to 16 (x, dz) tensor pairs of one shape ("chunks": the uses of a recurrent conv at
    // different time steps), so their weight gradient needs neither a launch per use nor a concatenation.
    CUtensorMap xmap[kWgMaxChunks], zmap[kWgMaxChunks];
    int tiles_per_chunk;
    int H, W, batch;
    int tiles_x, tiles_per_img, total_tiles;
    int c0, n0;                 // channel offsets inside x / dz
    int cout, cin_total, ci_off;   // OIHW geometry of dw; ci_off = first input channel of this block on the OIHW axis
    float* dw;
    float* db;                  // bias gradient (sum of dz over the pixels), or null: the epilogue warps, idle while the tiles stream
                                // through, add up the dz tiles in shared memory - no second pass over dz
    float* slots;               // deterministic mode: CTA x stores its [cout][64][9] block at slots + x * cout * 576 (else null)
    float* bslots;              // ... and its bias sums at bslots + x * cout
    int* dbg;
    int debug;                  // VSRB_WG_DEBUG: 1 / 2 / 4 = skip the final atomics / the MMAs / the loads (timing decomposition only)
};

// MN-major, 128B-swizzled operand descriptor: start>>4 | LBO>>4 @16 | SBO>>4 @32 (8 K-rows = 1024 B) | version 1 @46 | layout 2 @61
__device__ __forceinline__ uint64_t mn_desc(uint32_t saddr, uint32_t lbo_bytes) {
    const uint32_t lo = ((saddr >> 4) & 0x3FFFu) | (((lbo_bytes >> 4) & 0x3FFFu) << 16);
    const uint32_t hi = (1024u >> 4) | (1u << 14) | (2u << 29);
    return ((uint64_t)hi << 32) | lo;
}

__global__ void __launch_bounds__(kWgThreads, 1) wgrad_tc_kernel(const __grid_constant__ WgTcParams P) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    uint8_t* base_ptr = smem_raw + (base - raw);
    const uint32_t full0 = base, empty0 = base + 64, done = base + 128;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(base_ptr + 192);
    const uint32_t stage0 = base + 1024;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n0 = P.n0 + (int)blockIdx.y * 64;         // this CTA's 64-wide block of output channels

    if (warp == 1 && lane == 0) {
        for (int i = 0; i < kWgStages; ++i) {
            mbar_init(full0 + 8 * i, 1);
            mbar_init(empty0 + 8 * i, P.db ? 5 : 1);          // the MMAs' commit (+ the four bias warps)
        }
        mbar_init(done, 1);
        fence_barrier_init();
    }
    if (warp == 2) tmem_alloc(smem_u32(tmem_slot), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
    bool dead = false;
    const int my_tiles = (P.total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    float bs0 = 0.f, bs1 = 0.f;                                // bias warps: this lane's channels 2*lane, 2*lane + 1

    if (warp == 0) {
        // ---- producer: one halo box of x and the dz tile per pixel tile ----
        int slot = 0;
        uint32_t phase = 0;
        for (int tile = blockIdx.x; tile < P.total_tiles; tile += gridDim.x) {
            const int chunk = tile / P.tiles_per_chunk;
            const int tc = tile - chunk * P.tiles_per_chunk;
            const int img = tc / P.tiles_per_img;                 // image inside its chunk
            const int t = tc - img * P.tiles_per_img;
            const int ty = t / P.tiles_x, tx = t - ty * P.tiles_x;
            const uint32_t sa = stage0 + slot * kWgStageBytes;
            mbar_wait(empty0 + 8 * slot, phase ^ 1, P.dbg, 11, dead);
            if (elect_one() && (P.debug & 4)) {
                mbar_arrive(full0 + 8 * slot);                // timing decomposition: no loads
            } else if (elect_one()) {
                mbar_expect_tx(full0 + 8 * slot, kWgXBytes + kWgZBytes);
                tma_load_4d(&P.xmap[chunk], full0 + 8 * slot, sa, P.c0, tx * kWgTW - 1, ty * kWgRows - 1, img);
                tma_load_4d(&P.zmap[chunk], full0 + 8 * slot, sa + kWgCopyBytes, n0, tx * kWgTW, ty * kWgRows, img);
            }
            __syncwarp();
            if (++slot == kWgStages) { slot = 0; phase ^= 1; }
        }
    } else if (warp == 1) {
        // ---- MMA issuer: D_pair[128 x 64] += X_pair^T[128 x 16] * dZ[16 x 64] for kWgRows K steps x 5 tap pairs ----
        // instruction descriptor: D=f32, A=B=bf16, A and B MN-major (bits 15, 16), N=64, M=128
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(64 >> 3) << 17) | (8u << 24);
        const bool leader = elect_one();
        const uint32_t tm0 = __shfl_sync(0xffffffffu, tmem_base, 0);
        int slot = 0;
        uint32_t phase = 0;
        bool first = true;
        for (int it = 0; it < my_tiles; ++it) {
            const uint32_t sa = stage0 + slot * kWgStageBytes;
            mbar_wait(full0 + 8 * slot, phase, P.dbg, 12, dead);
            tc_fence_after();
            if (!(P.debug & 2)) {     // warp-uniform arithmetic, only the instruction is predicated on the elected lane (no R2UR)
                // descriptor low words advance by adds (the issuing thread has ~49 cycles per N = 64 MMA): the high word and the
                // LBO fields are constants, every window start below is the stage address plus an immediate
                constexpr uint32_t kRow16 = (kWgXW * 128u) >> 4;    // one box row of 18 pixels, in 16-byte units
                constexpr uint32_t kHi = (1024u >> 4) | (1u << 14) | (2u << 29);
                constexpr uint32_t kLboPx = (128u >> 4) << 16, kLboRow = kRow16 << 16;
                const uint32_t x0 = (sa >> 4) & 0x3FFFu, z0 = ((sa + kWgCopyBytes) >> 4) & 0x3FFFu;
#pragma unroll
                for (int ks = 0; ks < kWgRows; ++ks) {
                    const uint32_t bd = z0 + ks * (2048u >> 4);
                    const uint32_t acc = (first && ks == 0) ? 0u : 1u;
                    // pairs (ky,0)&(ky,1): the second tap's window starts one pixel further
#pragma unroll
                    for (int ky = 0; ky < 3; ++ky)
                        if (leader) umma_bf16_words(tm0 + ky * 64, (x0 + (ky + ks) * kRow16) | kLboPx, kHi, bd, kHi, idesc, acc);
                    // pair (0,2)&(1,2): two pixels in, the second tap one box row further down
                    if (leader) umma_bf16_words(tm0 + 3 * 64, (x0 + ks * kRow16 + (256u >> 4)) | kLboRow, kHi, bd, kHi, idesc, acc);
                    // (2,2) & a don't-care second half
                    if (leader) umma_bf16_words(tm0 + 4 * 64, (x0 + (2 + ks) * kRow16 + (256u >> 4)) | kLboPx, kHi, bd, kHi, idesc, acc);
                }
            }
            if (leader) umma_commit(empty0 + 8 * slot);
            __syncwarp();
            first = false;
            if (++slot == kWgStages) { slot = 0; phase ^= 1; }
        }
        if (leader) umma_commit(done);
        __syncwarp();
    } else if (warp >= 4) {
        // ---- epilogue (once), part 1: TMEM -> shared memory in the OIHW order of the 64(co) x 64(ci) x 9 block.  Lanes
        // differ in ci, i.e. by 9 floats: conflict-free.  The pipeline stages are free once `done` has fired. ----
        const int wq = warp - 4;
        if (P.db) {
            // ---- bias gradient: every warp adds 16 of the 64 pixel rows of each dz tile; a row is 128 swizzled bytes, the
            // lane's two channels sit in 16-byte chunk (lane / 4) ^ (row & 7): one conflict-free 4-byte load per row ----
            int slot = 0;
            uint32_t phase = 0;
            for (int it = 0; it < my_tiles; ++it) {
                const uint32_t zb = stage0 + slot * kWgStageBytes + kWgCopyBytes;
                mbar_wait(full0 + 8 * slot, phase, P.dbg, 14, dead);
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const uint32_t r = (uint32_t)(wq * 16 + i);
                    uint32_t v;
                    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(zb + r * 128u + ((((uint32_t)lane >> 2) ^ (r & 7u)) << 4) + ((uint32_t)lane & 3u) * 4u));
                    const float2 f = unpack_bf16(v);
                    bs0 += f.x;
                    bs1 += f.y;
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(empty0 + 8 * slot);
                if (++slot == kWgStages) { slot = 0; phase ^= 1; }
            }
        }
        mbar_wait(done, 0, P.dbg, 13, dead);
        tc_fence_after();
        if (my_tiles > 0) {
            const int half = wq >> 1;                       // rows 0..63 = first tap of the pair, 64..127 = second
            const int ci = (wq & 1) * 32 + lane;
            // tap = ky*3 + kx of (pair, half)
            const int tapA[5] = {0, 3, 6, 2, 8}, tapB[5] = {1, 4, 7, 5, -1};
            float* stg = reinterpret_cast<float*>(base_ptr + 1024);
            for (int pr = 0; pr < 5; ++pr) {
                const int tap = half ? tapB[pr] : tapA[pr];
                for (int c0 = 0; c0 < 64; c0 += 16) {
                    uint32_t r[16];
                    tmem_ld16_nowait(tmem_base + ((uint32_t)(wq * 32) << 16) + pr * 64 + c0, r);
                    tmem_ld_wait();
                    if (tap >= 0) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) stg[((c0 + j) * 64 + ci) * 9 + tap] = __uint_as_float(r[j]);
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    // ---- epilogue part 2 (all warps): the block leaves with coalesced atomics - consecutive lanes add consecutive floats
    // of dw[co][ci_off .. ci_off+63][0..8], 8x fewer L2 sector operations than one scattered atomic per (ci, tap) ----
    if (P.slots) {
        const float* stg = reinterpret_cast<const float*>(base_ptr + 1024);
        float* slot = P.slots + (size_t)blockIdx.x * P.cout * 576;
        for (int co = 0; co < 64 && n0 + co < P.cout; ++co)
            for (int i = threadIdx.x; i < 576; i += kWgThreads) slot[(size_t)(n0 + co) * 576 + i] = my_tiles > 0 ? stg[co * 576 + i] : 0.f;
    } else if (my_tiles > 0 && !(P.debug & 1)) {
        const float* stg = reinterpret_cast<const float*>(base_ptr + 1024);
        for (int co = 0; co < 64 && n0 + co < P.cout; ++co) {
            float* dst = P.dw + ((size_t)(n0 + co) * P.cin_total + P.ci_off) * 9;
            for (int i = threadIdx.x; i < 576; i += kWgThreads) atomicAdd(dst + i, stg[co * 576 + i]);
        }
    }
    if (P.db) {                                                // the four bias warps' partial sums -> one atomic per channel and CTA
        float* bsum = reinterpret_cast<float*>(base_ptr + 256);
        if (warp >= 4) {
            bsum[(warp - 4) * 64 + 2 * lane] = bs0;
            bsum[(warp - 4) * 64 + 2 * lane + 1] = bs1;
        }
        __syncthreads();
        if (P.bslots && threadIdx.x < 64 && n0 + (int)threadIdx.x < P.cout)
            P.bslots[(size_t)blockIdx.x * P.cout + n0 + threadIdx.x] =
                my_tiles > 0 ? bsum[threadIdx.x] + bsum[64 + threadIdx.x] + bsum[128 + threadIdx.x] + bsum[192 + threadIdx.x] : 0.f;
        else if (threadIdx.x < 64 && my_tiles > 0 && n0 + (int)threadIdx.x < P.cout && !(P.debug & 1))
            atomicAdd(P.db + n0 + threadIdx.x, bsum[threadIdx.x] + bsum[64 + threadIdx.x] + bsum[128 + threadIdx.x] + bsum[192 + threadIdx.x]);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// bias gradient: db[co] += sum over pixels of dz[p][co]
__device__ __forceinline__ void bias_ld8(const __nv_bfloat16* p, float (&v)[8]) {
    const uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
    const float2 a = unpack_bf16(u.x), b = unpack_bf16(u.y), c = unpack_bf16(u.z), d = unpack_bf16(u.w);
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; v[4] = c.x; v[5] = c.y; v[6] = d.x; v[7] = d.y;
}
__device__ __forceinline__ void bias_ld8(const float* p, float (&v)[8]) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

// db[c] += sum over pixels of dz[p][c].  HBM-bound (reads dz once): every thread owns 8 consecutive channels (one 16-byte
// load per pixel for bf16) and a strided set of pixels; the pixel lanes of a CTA are reduced in shared memory, then one
// atomic per channel and CTA (or, deterministic, a store to the CTA's slot: slots + blockIdx.x * cout).
// blockDim = 256 = G channel groups (G = 8 for 64 channels) x 256/G pixel lanes.
template <typename T>
__global__ void __launch_bounds__(256) bias_grad_kernel(const T* __restrict__ dz, int dz_c, long long pixels, int cout, int G,
                                                        float* __restrict__ db, float* __restrict__ slots) {
    __shared__ float red[256][9];                                  // [thread][8 channels] (+1: no bank conflicts)
    const int grp = threadIdx.x % G, lane = threadIdx.x / G, lanes = 256 / G;
    const int c0 = (blockIdx.y * G + grp) * 8;
    float s[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) s[i] = 0.f;
    if (c0 < dz_c) {
        for (long long p = (long long)blockIdx.x * lanes + lane; p < pixels; p += (long long)gridDim.x * lanes) {
            float v[8];
            bias_ld8(dz + p * dz_c + c0, v);
#pragma unroll
            for (int i = 0; i < 8; ++i) s[i] += v[i];
        }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) red[threadIdx.x][i] = s[i];
    __syncthreads();
    if (threadIdx.x < G * 8) {                                     // thread = (group, channel of the group)
        const int g2 = threadIdx.x / 8, ch = threadIdx.x % 8;
        float t = 0.f;
        for (int l = 0; l < lanes; ++l) t += red[l * G + g2][ch];
        const int c = (blockIdx.y * G + g2) * 8 + ch;
        if (c < cout) {
            if (slots) slots[(size_t)blockIdx.x * cout + c] = t;
            else atomicAdd(db + c, t);
        }
    }
}

// dst[r * dst_stride + e] += sum over s = 0, 1, ..., slots - 1 of parts[s][r][e]  (parts: `slots` blocks of rows x row_len).
// One writer per element and a fixed order of the additions: the deterministic end of every weight / bias gradient.
__global__ void __launch_bounds__(256) slot_reduce_kernel(const float* __restrict__ parts, int slots, int rows, int row_len,
                                                          long long dst_stride, float* __restrict__ dst) {
    const long long n = (long long)rows * row_len;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
        float acc = 0.f;
        for (int s = 0; s < slots; ++s) acc += __ldg(parts + (long long)s * n + i);
        const long long r = i / row_len;
        dst[r * dst_stride + (i - r * row_len)] += acc;
    }
}

int launch_slot_reduce(const float* parts, int slots, int rows, int row_len, long long dst_stride, float* dst, cudaStream_t s) {
    const long long n = (long long)rows * row_len;
    long long b = (n + 255) / 256;
    if (b > 148 * 8) b = 148 * 8;
    slot_reduce_kernel<<<(int)b, 256, 0, s>>>(parts, slots, rows, row_len, dst_stride, dst);
    VSRB_LAUNCH_CHECK();
    return VSRB_OK;
}

int launch_bias_grad(const void* dz, int dz_c, long long pixels, int cout, int dtype, float* db, cudaStream_t s, WgradDet* det) {
    const int groups = ceil_div(cout, 8);
    int G = 1;
    while (G < groups && G < 32) G *= 2;                            // channel groups per CTA: power of two <= 32
    long long want = (pixels + 256 / G * 8 - 1) / (256 / G * 8);   // >= 8 pixels per thread
    int gx = (int)(want < 1 ? 1 : (want > 148 * 4 ? 148 * 4 : want));
    dim3 grid(gx, ceil_div(groups, G));
    float* slots = nullptr;
    if (det) {
        if (det_take(det, (size_t)gx * cout)) return VSRB_OK;
        slots = det->ws;
    }
    if (dtype == VSRB_BF16)
        bias_grad_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(dz), dz_c, pixels, cout, G, db, slots);
    else
        bias_grad_kernel<float><<<grid, 256, 0, s>>>(reinterpret_cast<const float*>(dz), dz_c, pixels, cout, G, db, slots);
    VSRB_LAUNCH_CHECK();
    return slots ? launch_slot_reduce(slots, gx, 1, cout, 0, db, s) : VSRB_OK;
}

// one 64-input-channel block (x channels [c0, c0+64), OIHW offset ci_off) against all 64-wide output blocks, summed over
// `n_chunks` (x, dz) pairs of `batch` images each
int launch_wgrad_tc_multi(const void* const* xs, int x_c, int c0, int ci_off, const void* const* dzs, int dz_c, int n_chunks,
                          int batch, int h, int w, int cout, int cin_total, float* dw, cudaStream_t stream, float* db, WgradDet* det) {
    static bool ready[kMaxDevices] = {false};
    VSRB_CHECK_ARG(n_chunks >= 1 && n_chunks <= kWgMaxChunks, "wgrad: 1..%d chunks per launch", kWgMaxChunks);
    int dev = 0, sms = 0;
    int rc = device_setup(&dev, &sms, ready, [](int) {
        VSRB_CUDA(cudaFuncSetAttribute(wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kWgSmem));
        return VSRB_OK;
    });
    if (rc != VSRB_OK) return rc;
    WgTcParams P;
    memset(&P, 0, sizeof(P));
    P.H = h; P.W = w; P.batch = batch;
    P.tiles_x = ceil_div(w, kWgTW);
    P.tiles_per_img = P.tiles_x * ceil_div(h, kWgRows);
    P.tiles_per_chunk = P.tiles_per_img * batch;
    P.total_tiles = P.tiles_per_chunk * n_chunks;
    P.c0 = c0; P.cout = cout; P.cin_total = cin_total; P.ci_off = ci_off; P.dw = dw; P.db = db;
    P.dbg = debug_flag();
    const int n_blocks = ceil_div(cout, 64);
    // every CTA ends with 9*64*64 atomics, so small problems use fewer CTAs (>= 32 pixel tiles each)
    int ctas = sms / n_blocks;
    if (ctas > P.total_tiles / 32) ctas = P.total_tiles / 32;
    if (ctas < 1) ctas = 1;
    for (int k = 0; k < n_chunks; ++k) {
        VSRB_CHECK_ARG(xs[k] && dzs[k] && ((reinterpret_cast<uintptr_t>(xs[k]) | reinterpret_cast<uintptr_t>(dzs[k])) & 15) == 0,
                       "wgrad: chunk %d: null or unaligned tensor", k);
        rc = encode_nhwc(&P.xmap[k], "wgrad x", xs[k], x_c, w, h, batch, 64, kWgXW, kWgRows + 2);
        if (rc != VSRB_OK) return rc;
        rc = encode_nhwc(&P.zmap[k], "wgrad dz", dzs[k], dz_c, w, h, batch, 64, kWgTW, kWgRows);
        if (rc != VSRB_OK) return rc;
    }
    // deterministic mode: the planning pass stops here, after every argument check of the launch
    if (det) {
        if (det_take(det, (size_t)ctas * cout * (576 + (db ? 1 : 0)))) return VSRB_OK;
        P.slots = det->ws;
        P.bslots = db ? det->ws + (size_t)ctas * cout * 576 : nullptr;
    }
    P.debug = env_int("VSRB_WG_DEBUG");
    // blockIdx.y = 64-wide output block: all blocks of a wide layer (64 -> 256) share ONE launch.  (A launch per block on
    // sms / n_blocks CTAs each ran them one after the other - same stream - on a quarter of the GPU: 560 -> 230 us.)
    P.n0 = 0;
    wgrad_tc_kernel<<<dim3(ctas, n_blocks), kWgThreads, kWgSmem, stream>>>(P);
    VSRB_LAUNCH_CHECK();
    if (det) {
        rc = launch_slot_reduce(P.slots, ctas, cout, 576, (long long)cin_total * 9, dw + (size_t)ci_off * 9, stream);
        if (rc == VSRB_OK && db) rc = launch_slot_reduce(P.bslots, ctas, 1, cout, 0, db, stream);
        return rc;
    }
    return VSRB_OK;
}

}  // namespace vsrb
