// Weight gradient of K x K convolutions (K = 1, 3, 5, 7) over 16-, 32- or 64-channel blocks on the tensor cores: the
// layers wgrad_tc.cu does not take - SPyNet's 7x7 stacks (8->32->64->32->16->2), 3-channel image segments, 1x1 fusion.
//
//   Out[ty][tx][s][u] = sum over pixels (y, x) of  S[y][x + tx - K/2][s] * U[y - ty + K/2][x][u]
//
// is a GEMM over the pixel index with both operands MN-major (a TMA box of pixels x C channels is K rows of C contiguous
// elements), and BOTH filter axes are folded into ONE instruction per 16 pixels:
//   * S, the NARROWER of (x, dz), carries the horizontal shift: its 128/Cs windows of consecutive tx fill the M = 128 rows
//     (the descriptor's leading-dimension offset is one pixel; an MN-major operand may start at any pixel row of its tile in
//     the 32B, 64B and 128B swizzle modes alike - tools/umma_mn_modes_test.cu);
//   * U, the wider tensor, carries the vertical shift: the N columns are the Cu channels of up to 256/Cu box rows one below
//     the other (leading-dimension offset = one box row).
// 7x7, 8 -> 32 channels: ONE MMA of N = 224 per 16 pixels instead of 49 x 2 mma.sync tiles.  The point of the stacking is
// the tensor pipe's cost of 40 / 41 / 49 / 65 / 129 cycles at N = 16 / 32 / 64 / 128 / 256 (same tool): seven N = 32 MMAs
// cost 287 cycles, one N = 224 MMA 112, and the issuing thread has to feed 7x fewer instructions.
// With S = x the taps are the filter's (ky, kx) = (ty, tx); with S = dz the sum runs over the mirrored taps
// (K-1-ty, K-1-tx) - zero padding outside the image is the TMA's out-of-bounds fill either way.  When G * K * Cu
// accumulator columns exceed the 512 of TMEM (or K * Cu > 256), blockIdx.y splits the ty range; each pass loads only the
// U rows it needs.  One box of S (R rows, 16 + K-1 pixels) and one of U (R + nj-1 rows, 16 pixels) per 16 x R pixel tile,
// mbarrier ring.  Epilogue: per 16 U channels the accumulators go through shared memory in OIHW order, then leave as runs
// of nj*K consecutive floats with coalesced atomics (deterministic mode: stores to the CTA's slot, summed in slot order).
#include "common.cuh"
#include "tc_ptx.cuh"

namespace vsrb {

static constexpr int kTpThreads = 256;
static constexpr int kTpTW = 16;                    // tile width = one K = 16 step per tile row
static constexpr int kTpMaxStages = 8;

struct WgTapsParams {
    CUtensorMap smap, umap;
    int K, pad;                 // filter size, K / 2
    int cs, cu;                 // channel block of S / U: 16, 32 or 64
    int rows;                   // tile rows R
    int nj_max, G, tpg;         // U rows (ty values) per pass; MMAs per 16 pixels; tx per MMA (128 / cs)
    int s_bytes, u_bytes, u_off, stage_bytes, stages;   // u_off: where the U box sits inside a stage
    int tiles_x, tiles_per_img, total_tiles;
    int s_c0, u_c0;             // first channel of the block inside its tensor
    int s_is_x;                 // 1: S = x (rows of Out are input channels), 0: S = dz
    int co0, ci0;               // OIHW origin of this block (ci0 includes the segment offset)
    int co_valid, ci_valid;     // channels of the block that exist
    int cin_total;
    float* dw;
    float* slots;               // deterministic mode: CTA x stores its [co_valid][ci_valid][K*K] block at slots + x * that size
    int* dbg;
    int debug;                  // VSRB_WG_DEBUG: 1 / 2 / 4 = skip the final atomics / the MMAs / the loads
};

// MN-major operand descriptor in the swizzle mode of its row pitch (32, 64 or 128 bytes): start>>4 | LBO>>4 @16 |
// SBO>>4 @32 (8 K rows) | version 1 @46 | layout @61 (2 = 128B, 4 = 64B, 6 = 32B)
__device__ __forceinline__ uint64_t mn_desc_pitch(uint32_t saddr, uint32_t lbo_bytes, uint32_t pitch) {
    const uint32_t layout = pitch == 128u ? 2u : (pitch == 64u ? 4u : 6u);
    const uint32_t lo = ((saddr >> 4) & 0x3FFFu) | (((lbo_bytes >> 4) & 0x3FFFu) << 16);
    const uint32_t hi = ((8u * pitch) >> 4) | (1u << 14) | (layout << 29);
    return ((uint64_t)hi << 32) | lo;
}

__global__ void __launch_bounds__(kTpThreads, 1) wgrad_taps_kernel(const __grid_constant__ WgTapsParams P) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    uint8_t* base_ptr = smem_raw + (base - raw);
    const uint32_t full0 = base, empty0 = base + 64, done = base + 128;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(base_ptr + 192);
    const uint32_t stage0 = base + 1024;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // this pass owns the U rows (N blocks) j0 .. j0 + nj - 1; block j holds ty = K-1-j
    const int j0 = blockIdx.y * P.nj_max;
    const int nj = (P.K - j0) < P.nj_max ? (P.K - j0) : P.nj_max;
    const int box_w = kTpTW + P.K - 1;
    const uint32_t pitch_s = 2u * P.cs, pitch_u = 2u * P.cu;
    const uint32_t acc_cols = (uint32_t)(P.nj_max * P.cu);            // TMEM columns per accumulator (one per tx group)

    if (warp == 1 && lane == 0) {
        for (int i = 0; i < P.stages; ++i) {
            mbar_init(full0 + 8 * i, 1);
            mbar_init(empty0 + 8 * i, 1);
        }
        mbar_init(done, 1);
        fence_barrier_init();
    }
    if (warp == 2) tmem_alloc(smem_u32(tmem_slot), 512);
    if (warp == 0 && lane == 0) {
        prefetch_tensormap(&P.smap);
        prefetch_tensormap(&P.umap);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
    bool dead = false;
    const int my_tiles = (P.total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

    if (warp == 0) {
        // ---- producer: the halo box of S (rows this pass needs) and the tile of U ----
        int slot = 0;
        uint32_t phase = 0;
        for (int tile = blockIdx.x; tile < P.total_tiles; tile += gridDim.x) {
            const int img = tile / P.tiles_per_img;
            const int t = tile - img * P.tiles_per_img;
            const int ty = t / P.tiles_x, tx = t - ty * P.tiles_x;
            const uint32_t sa = stage0 + slot * P.stage_bytes;
            mbar_wait(empty0 + 8 * slot, phase ^ 1, P.dbg, 21, dead);
            if (elect_one()) {
                if (P.debug & 4) {
                    mbar_arrive(full0 + 8 * slot);
                } else {
                    mbar_expect_tx(full0 + 8 * slot, P.s_bytes + P.u_bytes);
                    tma_load_4d(&P.smap, full0 + 8 * slot, sa, P.s_c0, tx * kTpTW - P.pad, ty * P.rows, img);
                    tma_load_4d(&P.umap, full0 + 8 * slot, sa + P.u_off, P.u_c0, tx * kTpTW, ty * P.rows - P.pad + j0, img);
                }
            }
            __syncwarp();
            if (++slot == P.stages) { slot = 0; phase ^= 1; }
        }
    } else if (warp == 1) {
        // ---- MMA issuer: per tile row (K = 16 pixels) and tx group: Out_g[128 x nj*Cu] += S_windows^T[128 x 16] * U_rows[16 x nj*Cu].
        // The loops run warp-uniformly and only the instruction is predicated on the elected lane, so the operand words live in
        // uniform registers; descriptor high words are constants, the low words (start >> 4 | LBO >> 4 @16) advance by adds.
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)((nj * P.cu) >> 3) << 17) | (8u << 24);
        const uint32_t a_hi = (uint32_t)(mn_desc_pitch(0u, 0u, pitch_s) >> 32), b_hi = (uint32_t)(mn_desc_pitch(0u, 0u, pitch_u) >> 32);
        const uint32_t a_lbo = (pitch_s >> 4) << 16, b_lbo = ((kTpTW * pitch_u) >> 4) << 16;
        const uint32_t row_step = ((uint32_t)box_w * pitch_s) >> 4, g_step = ((uint32_t)P.tpg * pitch_s) >> 4, b_step = (kTpTW * pitch_u) >> 4;
        const int G = P.G, rows = (P.debug & 2) ? 0 : P.rows;
        const bool leader = elect_one();
        const uint32_t tm0 = __shfl_sync(0xffffffffu, tmem_base, 0);
        int slot = 0;
        uint32_t phase = 0;
        uint32_t acc = 0u;
        for (int it = 0; it < my_tiles; ++it) {
            const uint32_t sa = stage0 + slot * P.stage_bytes;
            const uint32_t ub = sa + P.u_off;
            mbar_wait(full0 + 8 * slot, phase, P.dbg, 22, dead);
            tc_fence_after();
            uint32_t a_row = ((sa >> 4) & 0x3FFFu) | a_lbo, b_lo = ((ub >> 4) & 0x3FFFu) | b_lbo;
            for (int ks = 0; ks < rows; ++ks) {
                uint32_t a_lo = a_row, tm = tm0;
                for (int g = 0; g < G; ++g) {
                    if (leader) umma_bf16_words(tm, a_lo, a_hi, b_lo, b_hi, idesc, acc);
                    tm += acc_cols;
                    a_lo += g_step;
                }
                acc = 1u;
                a_row += row_step;
                b_lo += b_step;
            }
            if (leader) umma_commit(empty0 + 8 * slot);
            __syncwarp();
            acc = 1u;
            if (++slot == P.stages) { slot = 0; phase ^= 1; }
        }
        if (leader) umma_commit(done);
        __syncwarp();
    } else if (warp >= 4) {
        mbar_wait(done, 0, P.dbg, 23, dead);
        tc_fence_after();
    }
    // ---- epilogue: 16 U channels at a time.  stg[co_local][ci_local][r], r = the run of nj*K taps this pass owns ----
    const int run = nj * P.K;
    const int A = P.s_is_x ? 16 : P.cs, B = P.s_is_x ? P.cs : 16;      // extents of (co_local, ci_local) in the staging block
    // S = x: block j is ky = K-1-j, the pass owns ky in [K-j0-nj, K-j0);  S = dz: block j is ky = j
    const int r_base = P.s_is_x ? (P.K - j0 - nj) * P.K : j0 * P.K;
    float* stg = reinterpret_cast<float*>(base_ptr + 1024);
    const int KK = P.K * P.K;
    for (int n0 = 0; n0 < P.cu; n0 += 16) {
        __syncthreads();                                                // staging block free (first pass: the roles are done)
        if (warp >= 4 && my_tiles > 0) {
            const int wq = warp - 4;
            const int m = wq * 32 + lane;
            const int t = m / P.cs, c = m - t * P.cs;
            for (int g = 0; g < P.G; ++g)
                for (int jl = 0; jl < nj; ++jl) {
                    uint32_t r[16];
                    tmem_ld16_nowait(tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)g * acc_cols + (uint32_t)(jl * P.cu + n0), r);
                    tmem_ld_wait();
                    const int tx = g * P.tpg + t;
                    if (tx < P.K) {
                        const int rr = P.s_is_x ? (nj - 1 - jl) * P.K + tx : jl * P.K + (P.K - 1 - tx);
#pragma unroll
                        for (int q = 0; q < 16; ++q) {
                            const int a = P.s_is_x ? q : c, b = P.s_is_x ? c : q;
                            stg[(a * B + b) * run + rr] = __uint_as_float(r[q]);
                        }
                    }
                }
        }
        tc_fence_before();
        __syncthreads();
        if (P.slots) {
            const int co_rel = P.s_is_x ? n0 : 0, ci_rel = P.s_is_x ? 0 : n0;
            const int co_lim = P.co_valid - co_rel, ci_lim = P.ci_valid - ci_rel;
            float* slot = P.slots + (size_t)blockIdx.x * P.co_valid * P.ci_valid * KK;
            for (int i = threadIdx.x; i < A * B * run; i += kTpThreads) {
                const int ab = i / run, rr = i - ab * run;
                const int a = ab / B, b = ab - a * B;
                if (a < co_lim && b < ci_lim)
                    slot[((size_t)(co_rel + a) * P.ci_valid + ci_rel + b) * KK + r_base + rr] = my_tiles > 0 ? stg[i] : 0.f;
            }
        } else if (my_tiles > 0 && !(P.debug & 1)) {
            const int co_base = P.co0 + (P.s_is_x ? n0 : 0), ci_base = P.ci0 + (P.s_is_x ? 0 : n0);
            const int co_lim = P.co_valid - (P.s_is_x ? n0 : 0), ci_lim = P.ci_valid - (P.s_is_x ? 0 : n0);
            const int total = A * B * run;
            for (int i = threadIdx.x; i < total; i += kTpThreads) {
                const int ab = i / run, rr = i - ab * run;
                const int a = ab / B, b = ab - a * B;
                if (a < co_lim && b < ci_lim)
                    atomicAdd(P.dw + ((size_t)(co_base + a) * P.cin_total + ci_base + b) * KK + r_base + rr, stg[i]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

static int pow2_block(int c) { return c <= 16 ? 16 : (c <= 32 ? 32 : 64); }

// One (input-channel block, output-channel block) pair: x channels [x_c0, x_c0 + ci_n), dz channels [z_c0, z_c0 + co_n),
// ci_n, co_n <= 64.  `ci_off` = OIHW position of x channel x_c0.
int launch_wgrad_taps(const void* x, int x_c, int x_c0, int ci_n, int ci_off, const void* dz, int dz_c, int z_c0, int co_n, int K,
                      int batch, int h, int w, int cin_total, float* dw, cudaStream_t stream, WgradDet* det) {
    static bool ready[kMaxDevices] = {false};
    VSRB_CHECK_ARG(K >= 1 && K <= 7 && (K & 1) && ci_n >= 1 && ci_n <= 64 && co_n >= 1 && co_n <= 64, "wgrad_taps: bad block");
    constexpr int kSmemMax = 200 * 1024;
    int dev = 0, sms = 0;
    int rc = device_setup(&dev, &sms, ready, [](int) {
        VSRB_CUDA(cudaFuncSetAttribute(wgrad_taps_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemMax + 2048));
        return VSRB_OK;
    });
    if (rc != VSRB_OK) return rc;
    WgTapsParams P;
    memset(&P, 0, sizeof(P));
    const int bx = pow2_block(ci_n), bz = pow2_block(co_n);
    P.s_is_x = bx <= bz;
    P.cs = P.s_is_x ? bx : bz;
    P.cu = P.s_is_x ? bz : bx;
    P.K = K; P.pad = K / 2;
    P.tpg = 128 / P.cs;
    P.G = ceil_div(K, P.tpg);
    P.nj_max = 512 / (P.G * P.cu);                  // TMEM: G accumulators of nj * cu columns
    if (P.nj_max > 256 / P.cu) P.nj_max = 256 / P.cu;   // N <= 256 per instruction
    if (P.nj_max > K) P.nj_max = K;
    const int passes = ceil_div(K, P.nj_max);
    P.rows = K >= 5 ? 8 : 4;
    if (h <= 4) P.rows = 4;
    const int box_w = kTpTW + K - 1, u_rows = P.rows + P.nj_max - 1;
    P.s_bytes = box_w * P.rows * P.cs * 2;
    P.u_bytes = kTpTW * u_rows * P.cu * 2;
    // the S box at the start of a stage, the U box behind it (1 KiB aligned); the windows of the junk taps beyond tx = K-1
    // read at most 16 pixels past the S box, i.e. into the gap: finite or not, those accumulator rows are never used
    // (u_bytes is a multiple of 512 B; the stage size is rounded so that both boxes start 1 KiB aligned)
    P.u_off = (P.s_bytes + 16 * P.cs * 2 + 1023) & ~1023;
    P.stage_bytes = P.u_off + ((P.u_bytes + 1023) & ~1023);
    P.stages = kSmemMax / P.stage_bytes;
    if (P.stages > kTpMaxStages) P.stages = kTpMaxStages;
    VSRB_CHECK_ARG(P.stages >= 2, "wgrad_taps: stage of %d bytes does not fit", P.stage_bytes);
    const int stg_bytes = 16 * P.cs * P.nj_max * K * 4;
    VSRB_CHECK_ARG(stg_bytes <= P.stages * P.stage_bytes, "wgrad_taps: staging block of %d bytes does not fit", stg_bytes);
    P.tiles_x = ceil_div(w, kTpTW);
    P.tiles_per_img = P.tiles_x * ceil_div(h, P.rows);
    const long long total = (long long)P.tiles_per_img * batch;
    VSRB_CHECK_ARG(total < (1LL << 31), "wgrad_taps: too many tiles");
    P.total_tiles = (int)total;
    const void* s_ptr = P.s_is_x ? x : dz;
    const void* u_ptr = P.s_is_x ? dz : x;
    const int s_c = P.s_is_x ? x_c : dz_c, u_c = P.s_is_x ? dz_c : x_c;
    P.s_c0 = P.s_is_x ? x_c0 : z_c0;
    P.u_c0 = P.s_is_x ? z_c0 : x_c0;
    P.co0 = z_c0; P.ci0 = ci_off;
    P.co_valid = co_n; P.ci_valid = ci_n;
    P.cin_total = cin_total;
    P.dw = dw;
    P.dbg = debug_flag();
    // every CTA ends with K*K*cs*cu/passes atomics: small problems use fewer CTAs (>= 8 tiles each)
    int ctas = sms / passes;
    if (ctas > P.total_tiles / 8) ctas = P.total_tiles / 8;
    if (ctas < 1) ctas = 1;
    VSRB_CHECK_ARG(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dz)) & 15) == 0 && x_c % 8 == 0 && dz_c % 8 == 0,
                   "wgrad_taps: tensors must be 16-byte aligned with channel strides that are multiples of 8");
    rc = encode_nhwc(&P.smap, "wgrad_taps S", s_ptr, s_c, w, h, batch, P.cs, box_w, P.rows);
    if (rc != VSRB_OK) return rc;
    rc = encode_nhwc(&P.umap, "wgrad_taps U", u_ptr, u_c, w, h, batch, P.cu, kTpTW, u_rows);
    if (rc != VSRB_OK) return rc;
    // deterministic mode: the planning pass stops here, after every argument check of the launch
    if (det) {
        if (det_take(det, (size_t)ctas * co_n * ci_n * K * K)) return VSRB_OK;
        P.slots = det->ws;
    }
    P.debug = env_int("VSRB_WG_DEBUG");
    const int smem = 1024 + 1024 + P.stages * P.stage_bytes;
    wgrad_taps_kernel<<<dim3(ctas, passes), kTpThreads, smem, stream>>>(P);
    VSRB_LAUNCH_CHECK();
    if (det)
        return launch_slot_reduce(P.slots, ctas, co_n, ci_n * K * K, (long long)cin_total * K * K,
                                  dw + ((size_t)z_c0 * cin_total + ci_off) * K * K, stream);
    return VSRB_OK;
}

}  // namespace vsrb
