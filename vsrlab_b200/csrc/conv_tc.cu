// Implicit-GEMM convolution on the 5th-generation tensor cores (tcgen05 + TMEM), fed by TMA.
//
//   D[pixel, cout] = sum over (segment, channel chunk, kx, ky) A[pixel shifted by (ky,kx), ck] * W[cout, ck]
//
// * A is never materialised as im2col.  For every (segment, chunk, kx) the producer issues ONE
//   TMA box load of (rows + kh - 1) x TW pixels x ck channels from the NHWC activation, shifted by
//   kx - kw/2 in x; out-of-image elements are zero-filled by TMA, which IS the conv's zero padding.
//   Inside the box, the A operand of filter row ky is the contiguous run of 128 pixels that starts
//   ky*TW pixels further down, so the kh filter rows reuse the same shared-memory bytes through
//   nothing but a different UMMA descriptor start address (always a whole number of 8-row swizzle
//   atoms because TW % 8 == 0).
// * W is pre-packed by vsrb_pack_conv_weight into the exact swizzled K-major shared-memory image
//   of each stage and copied with cp.async.bulk; when one (group, n_block) worth of weights fits,
//   it is loaded once per persistent CTA and stays resident.
// * A residual input (`x + conv(...)`, act none) is folded into the accumulation as one more K=64
//   stage: the residual tile is the A operand and a 64x64 identity matrix the B operand, so the
//   tensor core adds it exactly (bf16 * 1.0 into the fp32 accumulator) and the epilogue never
//   touches it.
// * One CTA per SM, persistent over output tiles.  Warp 0 = TMA producer, warp 1 = MMA issuer
//   (one elected lane issues tcgen05.mma, accumulators live in TMEM, double buffered), warp 2 =
//   TMEM allocator, warp 3 = bias loader, warps 4..7 = epilogue: tcgen05.ld -> bias/act -> bf16 ->
//   swizzled shared-memory staging -> one TMA store per warp (full 128-byte lines, asynchronous,
//   clipped at the image border by the tensor map; the PixelShuffle(2) store is just a strided
//   tensor map per sub-pixel).  Special epilogues (3-channel fp32 outputs) store directly.
//
// Replaces: F.conv2d behind nn.Conv2d at reference conv.py:89-92,101-103; upsampling.py:10-12;
// basicvsr.py:75-82; realbasicvsr.py:28-29; spynet.py:16-21 (see include/vsrb200.h).
#include <stdlib.h>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace vsrb {

static constexpr int kMaxSlots = 8;
static constexpr int kEpiPerQ = 2;     // epilogue warps per TMEM lane quarter (they split the channels)
static constexpr int kThreads = 128 + 128 * kEpiPerQ;   // 4 control warps + 4*kEpiPerQ epilogue warps
static constexpr int kSmemMax = 232448;   // 227 KiB opt-in maximum per CTA on sm_100
static constexpr int kCtrlBytes = 1024;
static constexpr int kIdentBytes = 8192;  // 64 x 64 bf16 identity, swizzle-128B K-major image

struct TcParams {
    CUtensorMap tmap[6];   // one per input operand
    CUtensorMap rmap;      // residual (MMA-identity path)
    CUtensorMap smap[4];   // output maps for the staged TMA store (one per pixel-shuffle sub-position)
    const uint8_t* w;      // packed weights (after the bias header)
    const uint8_t* ident;  // identity image in global memory
    EpiParams epi;
    int n_seg;
    int seg_chunks[4], seg_ck[4], seg_rowbytes[4], seg_layout[4], seg_bstage[4], seg_abytes[4], seg_stages[4];   // per weight segment
    uint32_t seg_woff[4];  // byte offset of the segment's first stage inside a packed weight block
    int n_ops;             // input operands; operand o multiplies weight segment op_wseg[o], starts at channel op_c0[o]
    int op_wseg[6], op_c0[6];
    int kh, kw;
    int H, W;
    int TW, rows_sub, MT, box_rows;
    int UW;                // output columns per tile: TW (classic) or TW - (kw-1) (stacked)
    int kxs;               // pipeline stages per channel chunk: kw (classic) or 1 (stacked)
    int ns;                // accumulator columns per sub-tile: n_tile (classic) or kw*n_tile (stacked)
    int res_xoff;          // x offset of the residual box relative to the tile's first output column
    int tiles_x, tiles_per_img;
    int imgs_per_group, groups;
    int n_tile, n_blocks;
    int num_slots, slot_bytes;
    int resident;
    uint32_t wblock_bytes, wres_bytes;
    int acc_cols;
    int res_mma;           // 1: residual added by the tensor core (identity stage)
    uint32_t res_abytes;
    int n_store;           // channels per store block (<= 64)
    int stg_bytes;         // bytes of one staging buffer (two are allocated)
    int epi_alt;           // narrow direct-store epilogues: the two warps of a lane quarter take alternate tiles
    int pdl;               // launched with programmatic stream serialization (weights already stable)
    int* dbg;
    int debug;             // VSRB_TC_DEBUG bits (timing experiments only): 1 = no loads, 2 = no stores, 4 = no MMA
};

// K-major, swizzled shared-memory operand descriptor (sm_100 "version 1"):
//  [0,14) start>>4 | [16,30) LBO>>4 (unused for swizzled K-major, 1) | [32,46) SBO>>4 = 8 rows |
//  [46,48) version=1 | [61,64) layout type (2 = 128B, 4 = 64B, 6 = 32B swizzle)
// All MMAs of one pipeline stage: MT sub-tiles x KH filter rows x ksteps K=16 steps.  Descriptors
// differ only in their 14-bit start-address field, so each MMA costs one add per operand.
template <int KH, bool kPair = false>
__device__ __forceinline__ void issue_stage(uint32_t d0, uint32_t a_lo, uint32_t b_lo, uint32_t desc_hi, uint32_t idesc,
                                            int MT, int d_m, uint32_t a_m, uint32_t a_ky, uint32_t b_ky, int ksteps,
                                            bool first) {
    for (int m = 0; m < MT; ++m) {
#pragma unroll
        for (int ky = 0; ky < KH; ++ky) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (k < ksteps) {
                    const uint64_t ad = ((uint64_t)desc_hi << 32) | (a_lo + m * a_m + ky * a_ky + k * 2);
                    const uint64_t bd = ((uint64_t)desc_hi << 32) | (b_lo + ky * b_ky + k * 2);
                    if constexpr (kPair) umma_bf16_pair(d0 + m * d_m, ad, bd, idesc, (first && ky == 0 && k == 0) ? 0u : 1u);
                    else umma_bf16(d0 + m * d_m, ad, bd, idesc, (first && ky == 0 && k == 0) ? 0u : 1u);
                }
            }
        }
    }
}

// bias + activation + bf16 pack of 16 accumulator columns into one swizzled staging row
__device__ __forceinline__ void stage_chunk(const EpiParams& e, const uint32_t (&r)[16], const float* bias16, uint32_t row_base,
                                            uint32_t col_bytes, uint32_t msk) {
    float v[16];
    const float4* bp = reinterpret_cast<const float4*>(bias16);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float4 f = bp[i];
        v[4 * i] = __uint_as_float(r[4 * i]) + f.x;
        v[4 * i + 1] = __uint_as_float(r[4 * i + 1]) + f.y;
        v[4 * i + 2] = __uint_as_float(r[4 * i + 2]) + f.z;
        v[4 * i + 3] = __uint_as_float(r[4 * i + 3]) + f.w;
    }
    epi_act16(e, v);
    uint32_t o0 = row_base + col_bytes, o1 = o0 + 16u;      // the XOR only touches address bits 4..6
    o0 ^= ((o0 >> 7) & msk) << 4;
    o1 ^= ((o1 >> 7) & msk) << 4;
    st_shared_v4(o0, pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
    st_shared_v4(o1, pack_bf16(v[8], v[9]), pack_bf16(v[10], v[11]), pack_bf16(v[12], v[13]), pack_bf16(v[14], v[15]));
}

// VSRB_TC_DEBUG bit 64: per-CTA %globaltimer stamps of the pipeline milestones (vsrb_debug_trace)
static constexpr int kTraceCtas = 512;
__device__ unsigned long long g_trace[kTraceCtas * 8];
__device__ __forceinline__ void trace_stamp(int debug, int slot) {
    if (debug & 64) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        const int cta = blockIdx.y * gridDim.x + blockIdx.x;
        if (cta < kTraceCtas) g_trace[cta * 8 + slot] = t;
    }
}

// Walks the tiles blockIdx.x, blockIdx.x + gridDim.x, ... of one group as (image, tile row, tile column) with
// carries instead of two integer divisions per tile (the divisions were ~15 % of the epilogue's instructions).
struct TileWalk {
    int li, ty, tx, d_li, d_ty, d_tx, tiles_x, tiles_y;
    __device__ __forceinline__ TileWalk(int first, int stride, int tiles_x_, int tiles_per_img) {
        tiles_x = tiles_x_;
        tiles_y = tiles_per_img / tiles_x_;
        li = first / tiles_per_img;
        int t = first - li * tiles_per_img;
        ty = t / tiles_x;
        tx = t - ty * tiles_x;
        d_li = stride / tiles_per_img;
        t = stride - d_li * tiles_per_img;
        d_ty = t / tiles_x;
        d_tx = t - d_ty * tiles_x;
    }
    __device__ __forceinline__ void next() {
        tx += d_tx;
        int c = tx >= tiles_x;
        tx -= c ? tiles_x : 0;
        ty += d_ty + c;
        c = ty >= tiles_y;
        ty -= c ? tiles_y : 0;
        li += d_li + c;
    }
};

// Stacked layout, NCH (16 or 4) output channels of one pixel row segment: gathers the kKW partial sums of every
// channel from the neighbouring lanes, adds the bias, applies the activation (kAct: 0 none, 1 ReLU, 2 max(v, v*act_k)).
template <int kKW, int kAct, int NCH = 16>
__device__ __forceinline__ void stacked_chunk16(uint32_t taddr, int n_tile, const float* bias16, float act_k, int lane,
                                                float (&v)[NCH]) {
    constexpr int PAD = kKW / 2;
    constexpr int CH = NCH < 16 ? NCH : (kKW == 3 ? 16 : 8);        // channels gathered per TMEM round trip
#pragma unroll
    for (int hh = 0; hh < NCH / CH; ++hh) {
        uint32_t r[kKW][CH];
#pragma unroll
        for (int kx = 0; kx < kKW; ++kx) tmem_ld_n<CH>(taddr + kx * n_tile + hh * CH, r[kx]);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < CH; ++i) {
            float sacc = __uint_as_float(r[PAD][i]) + bias16[hh * CH + i];
#pragma unroll
            for (int kx = 0; kx < kKW; ++kx)
                if (kx != PAD) sacc += __shfl_sync(0xffffffffu, __uint_as_float(r[kx][i]), (lane + kx - PAD) & 31);
            v[hh * CH + i] = kAct == 0 ? sacc : (kAct == 1 ? fmaxf(sacc, 0.f) : fmaxf(sacc, sacc * act_k));
        }
    }
}

// 3-wide stacked layout, hot shape (a warp owns 32 channels = two 16-channel chunks): the second chunk's TMEM loads
// are in flight while the first chunk is gathered, activated and written to the staging row.
__device__ __forceinline__ void ld_taps3(uint32_t taddr, int n_tile, uint32_t (&r)[3][16]) {
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) tmem_ld16_nowait(taddr + kx * n_tile, r[kx]);
}
template <int kAct>
__device__ __forceinline__ void combine3_store(const uint32_t (&r)[3][16], const float* bias16, float act_k, int lane, bool lane_ok,
                                               uint32_t row_addr, uint32_t msk) {
    float v[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        float sacc = __uint_as_float(r[1][i]) + bias16[i];
        sacc += __shfl_sync(0xffffffffu, __uint_as_float(r[0][i]), (lane - 1) & 31);
        sacc += __shfl_sync(0xffffffffu, __uint_as_float(r[2][i]), (lane + 1) & 31);
        v[i] = kAct == 0 ? sacc : (kAct == 1 ? fmaxf(sacc, 0.f) : fmaxf(sacc, sacc * act_k));
    }
    if (lane_ok) {
        uint32_t o0 = row_addr, o1 = o0 + 16u;
        o0 ^= ((o0 >> 7) & msk) << 4;
        o1 ^= ((o1 >> 7) & msk) << 4;
        st_shared_v4(o0, pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
        st_shared_v4(o1, pack_bf16(v[8], v[9]), pack_bf16(v[10], v[11]), pack_bf16(v[12], v[13]), pack_bf16(v[14], v[15]));
    }
}
template <int kAct>
__device__ __forceinline__ void stacked3_two_chunks(uint32_t (&ra)[3][16], uint32_t taddr, int n_tile, const float* bias32, float act_k,
                                                    int lane, bool lane_ok, uint32_t row_addr, uint32_t msk) {
    uint32_t rb[3][16];
    tmem_ld_wait();                                   // chunk 0 (issued by the caller before its barrier) has landed
    ld_taps3(taddr + 16, n_tile, rb);
    combine3_store<kAct>(ra, bias32, act_k, lane, lane_ok, row_addr, msk);
    tmem_ld_wait();
    combine3_store<kAct>(rb, bias32 + 16, act_k, lane, lane_ok, row_addr + 32u, msk);
}

// ---------------------------------------------------------------------------------------
// kStaged = true : EPI_NHWC through swizzled staging + per-warp TMA stores (the hot path)
// kStaged = false: every other epilogue, direct per-thread stores (3-channel fp32 outputs etc.)
// kKW = 0: classic layout (one stage per filter column); 3 / 7: stacked layout (see api.cu make_plan)
// kPair: two CTAs of a cluster (adjacent blockIdx.x) run each MMA together as one M = 256 instruction (cta_group::2):
// every CTA keeps its own pixel tile (A) and accumulator, but only HALF of the weight rows (B) - the tensor cores
// exchange the halves - so the shared-memory operand fetch per MMA drops from 128 + N to 128 + N/2 rows.  The leader
// (cluster rank 0) issues the MMAs; full/accumulator-empty barriers live in the leader, slot-empty/accumulator-full
// barriers are signalled in both CTAs by multicast commits.  Only the hot resblock shape uses it (launch_conv_tc).
template <bool kStaged, int kKW, bool kPair = false>
__global__ void __launch_bounds__(kThreads, 1) conv_tc_kernel(const __grid_constant__ TcParams P) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;                // swizzle atoms need 1 KiB alignment
    uint8_t* base_ptr = smem_raw + (base - raw);
    // control block: barriers, TMEM base, bias of this (group, n_block)
    const uint32_t full0 = base, empty0 = base + 8 * kMaxSlots, tfull0 = base + 16 * kMaxSlots,
                   tempty0 = tfull0 + 16, wbar = tempty0 + 16, wready = wbar + 8;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(base_ptr + 16 * kMaxSlots + 48);
    float* bias_s = reinterpret_cast<float*>(base_ptr + 256);   // up to 128 floats
    const uint32_t wres = base + kCtrlBytes;
    const uint32_t wid = wres + P.wres_bytes;                    // identity image (residual path)
    const uint32_t slots0 = wid + (P.res_mma ? kIdentBytes : 0);
    const uint32_t stg0 = slots0 + P.num_slots * P.slot_bytes;   // two staging buffers for the TMA store

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) trace_stamp(P.debug, 0);
    const int g = blockIdx.y / P.n_blocks, qb = blockIdx.y - g * P.n_blocks;
    const int tiles_g = P.imgs_per_group * P.tiles_per_img;
    const int rows_tile = P.rows_sub * P.MT;
    uint32_t crank = 0;                                         // rank in the CTA pair (0 = leader)
    if constexpr (kPair) crank = cluster_ctarank();

    // Prologue in two steps so the first loads leave as early as possible: (1) barriers exist (CTA- or pair-wide sync),
    // after which the producer warp starts; (2) the other eleven warps meet once more for the TMEM address and the bias.
    if (warp == 0 && lane == 0) {
        for (int o = 0; o < P.n_ops; ++o) prefetch_tensormap(&P.tmap[o]);
        if (P.res_mma) prefetch_tensormap(&P.rmap);
        if (kStaged) prefetch_tensormap(&P.smap[0]);
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < P.num_slots; ++i) {
            mbar_init(full0 + 8 * i, 1);
            mbar_init(empty0 + 8 * i, 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(tfull0 + 8 * i, 1);
            mbar_init(tempty0 + 8 * i, (P.epi_alt ? 4 : 4 * kEpiPerQ) * (kPair ? 2 : 1));
        }
        mbar_init(wbar, 1);
        mbar_init(wready, 2);
        fence_barrier_init();
    }
    if constexpr (kPair) cluster_sync_all();       // the peer's barriers must exist before anything is signalled across
    else __syncthreads();
    griddep_launch();      // the next kernel on the stream may start its own prologue as SMs free up
    uint32_t tmem_base = 0;
    if (warp >= 1) {
        if (warp == 2) {
            if constexpr (kPair) tmem_alloc_pair(smem_u32(tmem_slot), 512);
            else tmem_alloc(smem_u32(tmem_slot), 512);
        }
        if (warp == 3)
            for (int i = lane; i < P.n_tile; i += 32) bias_s[i] = __ldg(P.epi.bias + (size_t)g * P.epi.cout_pad + qb * P.n_tile + i);
        tc_fence_before();
        asm volatile("bar.sync 5, %0;" ::"n"(kThreads - 32) : "memory");
        tc_fence_after();
        tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
    }
    if (threadIdx.x == 32) trace_stamp(P.debug, 1);
    const uint8_t* wsrc = P.w + ((size_t)g * P.n_blocks + qb) * P.wblock_bytes;
    bool dead = false;

    if (warp < 4) {
    // pair kernel: registers move from the control warps to the epilogue warps (two chunks of accumulators in flight);
    // 4*32*72 + 8*32*216 = the 384*168 registers the CTA was launched with
    if constexpr (kPair) asm volatile("setmaxnreg.dec.sync.aligned.u32 72;");
    if (warp == 0) {
        // =============================== TMA producer ===============================
        // the warp stays converged; one elected lane arms the barrier and issues the copies
        if (kPair && elect_one()) {
            // this CTA's half of every weight block: rows [crank * ns/2, +ns/2) of each filter row's N = ns rows
            mbar_expect_tx(wbar, P.wblock_bytes / 2 + (P.res_mma ? (uint32_t)kIdentBytes / 2 : 0u));
            uint32_t off = 0;
            for (int s = 0; s < P.n_seg; ++s) {
                const uint32_t hb = P.seg_bstage[s] / (2u * (uint32_t)P.kh);
                for (int i = 0; i < P.seg_stages[s]; ++i) {
                    for (int ky = 0; ky < P.kh; ++ky)
                        bulk_load(wres + off / 2 + ky * hb, wsrc + off + (2 * ky + crank) * hb, hb, wbar);
                    off += P.seg_bstage[s];
                }
            }
            if (P.res_mma) bulk_load(wid, P.ident + crank * (kIdentBytes / 2), kIdentBytes / 2, wbar);
        } else if (!kPair && (P.resident || P.res_mma) && elect_one()) {
            mbar_expect_tx(wbar, (P.resident ? P.wblock_bytes : 0u) + (P.res_mma ? (uint32_t)kIdentBytes : 0u));
            if (P.resident) {
                uint32_t off = 0;
                for (int s = 0; s < P.n_seg; ++s)
                    for (int i = 0; i < P.seg_stages[s]; ++i) {
                        bulk_load(wres + off, wsrc + off, P.seg_bstage[s], wbar);
                        off += P.seg_bstage[s];
                    }
            }
            if (P.res_mma) bulk_load(wid, P.ident, kIdentBytes, wbar);
        }
        __syncwarp();
        griddep_wait();        // activations (and the residual) come from the previous kernel(s)
        int slot = 0;
        uint32_t phase = 0;
        TileWalk tw(blockIdx.x, gridDim.x, P.tiles_x, P.tiles_per_img);
        const bool stat = (P.debug & 32) && blockIdx.x == 0 && blockIdx.y == 0;      // VSRB_TC_DEBUG bit 32: wait-cycle accounting of CTA 0
        long long st_t0 = stat ? clock64() : 0, st_wait = 0;
        // pair: the loop runs while the LEADER's tile exists; an odd tile count leaves the peer one dummy tile whose
        // loads fall outside the tensor (zero fill) and whose result is never stored
        for (int tile = blockIdx.x; tile - (int)crank < tiles_g; tile += gridDim.x, tw.next()) {
            const int img = g * P.imgs_per_group + tw.li;
            const int ty = tw.ty, tx = tw.tx;
            const int y0 = ty * rows_tile - P.kh / 2, x0 = tx * P.UW - P.kw / 2;
            for (int o = 0; o < P.n_ops; ++o) {
                const int s = P.op_wseg[o];
                const uint32_t abytes = P.seg_abytes[s], bbytes = P.seg_bstage[s];
                uint32_t boff = P.seg_woff[s];
                int chunk = 0, kx = 0;
                for (int local = 0; local < P.seg_stages[s]; ++local) {
                    const uint32_t sa = slots0 + slot * P.slot_bytes;
                    const long long w0 = stat ? clock64() : 0;
                    mbar_wait(empty0 + 8 * slot, phase ^ 1, P.dbg, 1, dead);
                    if (stat) st_wait += clock64() - w0;
                    if (elect_one()) {
                        if constexpr (kPair) {                 // both tiles' bytes are counted on the leader's barrier
                            if (P.debug & 1) {
                                if (crank == 0) mbar_arrive(full0 + 8 * slot);
                            } else {
                                if (crank == 0) mbar_expect_tx(full0 + 8 * slot, 2 * abytes);
                                tma_load_4d_pair(&P.tmap[o], mapa_rank(full0 + 8 * slot, 0), sa, P.op_c0[o] + chunk * P.seg_ck[s], x0 + kx,
                                                 y0, img);
                            }
                        } else if (P.debug & 1) {
                            mbar_arrive(full0 + 8 * slot);
                        } else {
                            mbar_expect_tx(full0 + 8 * slot, abytes + (P.resident ? 0 : bbytes));
                            tma_load_4d(&P.tmap[o], full0 + 8 * slot, sa, P.op_c0[o] + chunk * P.seg_ck[s], x0 + kx, y0, img);
                            if (!P.resident) bulk_load(sa + abytes, wsrc + boff, bbytes, full0 + 8 * slot);
                        }
                    }
                    __syncwarp();
                    boff += bbytes;
                    if (++kx == P.kxs) { kx = 0; ++chunk; }
                    if (++slot == P.num_slots) { slot = 0; phase ^= 1; }
                }
            }
            if (P.res_mma) {                                   // residual tile: A operand of the identity stage
                const uint32_t sa = slots0 + slot * P.slot_bytes;
                mbar_wait(empty0 + 8 * slot, phase ^ 1, P.dbg, 6, dead);
                if (elect_one()) {
                    if constexpr (kPair) {
                        if (P.debug & 1) {
                            if (crank == 0) mbar_arrive(full0 + 8 * slot);
                        } else {
                            if (crank == 0) mbar_expect_tx(full0 + 8 * slot, 2 * P.res_abytes);
                            tma_load_4d_pair(&P.rmap, mapa_rank(full0 + 8 * slot, 0), sa, qb * P.n_tile, tx * P.UW - P.res_xoff,
                                             ty * rows_tile, img);
                        }
                    } else if (P.debug & 1) {
                        mbar_arrive(full0 + 8 * slot);
                    } else {
                        mbar_expect_tx(full0 + 8 * slot, P.res_abytes);
                        tma_load_4d(&P.rmap, full0 + 8 * slot, sa, qb * P.n_tile, tx * P.UW - P.res_xoff, ty * rows_tile, img);
                    }
                }
                __syncwarp();
                if (++slot == P.num_slots) { slot = 0; phase ^= 1; }
            }
        }
        if (stat && lane == 0) { g_trace[300 * 8 + 0] = clock64() - st_t0; g_trace[300 * 8 + 1] = st_wait; }
    } else if (warp == 1) {
        // =============================== MMA issuer =================================
        // instruction descriptor: D=f32, A=B=bf16, K-major both, N>>3 @17, M>>4 @24
        constexpr uint32_t kM = kPair ? 16u : 8u;               // M = 256 across the pair, 128 alone
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(P.ns >> 3) << 17) | (kM << 24);
        const uint32_t idesc_res = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(64 >> 3) << 17) | (kM << 24);
        if (kPair || P.resident || P.res_mma) mbar_wait(wbar, 0, P.dbg, 2, dead);
        if constexpr (kPair) {                                  // both halves of the weights must be resident
            if (elect_one()) mbar_arrive_cluster(mapa_rank(wready, 0));
            __syncwarp();
            if (crank == 0) mbar_wait(wready, 0, P.dbg, 8, dead);
        }
        if (lane == 0) trace_stamp(P.debug, 2);
        int slot = 0, acc = 0;
        uint32_t phase = 0, acc_phase = 0;
        bool first_stage = true;
        const bool stat = (P.debug & 32) && blockIdx.x == 0 && blockIdx.y == 0;
        long long st_t0 = stat ? clock64() : 0, st_we = 0, st_wf = 0;
        // One operand, one stage per tile, no residual stage (the thin image / flow convs, whose MMA warp is the bound): every
        // per-op value is loop invariant and the tile body is two waits, the MMAs and two commits.
        const bool simple = P.n_ops == 1 && P.seg_stages[P.op_wseg[0]] == 1 && !P.res_mma && kKW > 0 && !(P.debug & (4 | 128));     // (bit 128: A/B switch)
        if (simple) {
            const int s = P.op_wseg[0];
            const uint32_t rb = P.seg_rowbytes[s];
            const uint32_t desc_hi = ((rb * 8u) >> 4) | (1u << 14) | ((uint32_t)P.seg_layout[s] << 29);
            const uint32_t a_ky = (P.TW * rb) >> 4, b_ky = ((kPair ? P.ns / 2 : P.ns) * rb) >> 4, a_m = (P.rows_sub * P.TW * rb) >> 4;
            const int ksteps = P.seg_ck[s] >> 4, MT = P.MT, ns = P.ns;
            const uint32_t sb_res = kPair ? (wres + P.seg_woff[s] / 2) : (wres + P.seg_woff[s]);
            const uint32_t b_off = P.seg_abytes[s], slot_bytes = P.slot_bytes, acc_cols = P.acc_cols;
            const bool resident = kPair || P.resident;
            const int num_slots = P.num_slots;
            for (int tile = blockIdx.x; tile < tiles_g && crank == 0; tile += gridDim.x) {
                const long long w0 = stat ? clock64() : 0;
                mbar_wait(tempty0 + 8 * acc, acc_phase ^ 1, P.dbg, 3, dead);
                const long long w1 = stat ? clock64() : 0;
                mbar_wait(full0 + 8 * slot, phase, P.dbg, 4, dead);
                if (stat) { st_we += w1 - w0; st_wf += clock64() - w1; }
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t sa = slots0 + slot * slot_bytes;
                    const uint32_t sb = resident ? sb_res : (sa + b_off);
                    const uint32_t d0 = tmem_base + acc * acc_cols;
                    const uint32_t a_lo = ((sa >> 4) & 0x3FFFu) | (1u << 16), b_lo = ((sb >> 4) & 0x3FFFu) | (1u << 16);
                    issue_stage<kKW == 0 ? 1 : kKW, kPair>(d0, a_lo, b_lo, desc_hi, idesc, MT, ns, a_m, a_ky, b_ky, ksteps, true);
                    if constexpr (kPair) {
                        umma_commit_pair(empty0 + 8 * slot);
                        umma_commit_pair(tfull0 + 8 * acc);
                    } else {
                        umma_commit(empty0 + 8 * slot);
                        umma_commit(tfull0 + 8 * acc);
                    }
                }
                __syncwarp();
                if (++slot == num_slots) { slot = 0; phase ^= 1; }
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        } else
        for (int tile = blockIdx.x; tile < tiles_g && crank == 0; tile += gridDim.x) {
            const long long w0 = stat ? clock64() : 0;
            mbar_wait(tempty0 + 8 * acc, acc_phase ^ 1, P.dbg, 3, dead);
            if (stat) st_we += clock64() - w0;
            tc_fence_after();
            const uint32_t d0 = tmem_base + acc * P.acc_cols;
            bool first = true;
            for (int o = 0; o < P.n_ops; ++o) {
                const int s = P.op_wseg[o];
                uint32_t boff = P.seg_woff[s];
                const uint32_t rb = P.seg_rowbytes[s];
                const uint32_t desc_hi = ((rb * 8u) >> 4) | (1u << 14) | ((uint32_t)P.seg_layout[s] << 29);
                const uint32_t a_ky = (P.TW * rb) >> 4, b_ky = ((kPair ? P.ns / 2 : P.ns) * rb) >> 4,
                               a_m = (P.rows_sub * P.TW * rb) >> 4;
                const int ksteps = P.seg_ck[s] >> 4;
                for (int local = 0; local < P.seg_stages[s]; ++local) {
                    const uint32_t sa = slots0 + slot * P.slot_bytes;
                    const uint32_t sb = kPair ? (wres + boff / 2) : (P.resident ? (wres + boff) : (sa + P.seg_abytes[s]));
                    const long long w1 = stat ? clock64() : 0;
                    mbar_wait(full0 + 8 * slot, phase, P.dbg, 4, dead);
                    if (stat) st_wf += clock64() - w1;
                    tc_fence_after();
                    if (first_stage && lane == 0) trace_stamp(P.debug, 3);
                    first_stage = false;
                    if (elect_one()) {
                        const uint32_t a_lo = ((sa >> 4) & 0x3FFFu) | (1u << 16), b_lo = ((sb >> 4) & 0x3FFFu) | (1u << 16);
                        if (P.debug & 4) {
                        } else if (P.kh == 3) issue_stage<3, kPair>(d0, a_lo, b_lo, desc_hi, idesc, P.MT, P.ns, a_m, a_ky, b_ky, ksteps, first);
                        else if (P.kh == 7) issue_stage<7, kPair>(d0, a_lo, b_lo, desc_hi, idesc, P.MT, P.ns, a_m, a_ky, b_ky, ksteps, first);
                        else if (kPair) {
                        } else if (P.kh == 1) issue_stage<1>(d0, a_lo, b_lo, desc_hi, idesc, P.MT, P.ns, a_m, a_ky, b_ky, ksteps, first);
                        else issue_stage<5>(d0, a_lo, b_lo, desc_hi, idesc, P.MT, P.ns, a_m, a_ky, b_ky, ksteps, first);
                        // frees the slot (in both CTAs of a pair) when these MMAs retire
                        if constexpr (kPair) umma_commit_pair(empty0 + 8 * slot);
                        else umma_commit(empty0 + 8 * slot);
                    }
                    __syncwarp();
                    first = false;
                    boff += P.seg_bstage[s];
                    if (++slot == P.num_slots) { slot = 0; phase ^= 1; }
                }
            }
            if (P.res_mma) {                                   // D += residual * I
                const uint32_t sa = slots0 + slot * P.slot_bytes;
                mbar_wait(full0 + 8 * slot, phase, P.dbg, 7, dead);
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t a_lo = ((sa >> 4) & 0x3FFFu) | (1u << 16), b_lo = ((wid >> 4) & 0x3FFFu) | (1u << 16);
                    const uint32_t desc_hi = ((128u * 8u) >> 4) | (1u << 14) | (2u << 29);
                    if (!(P.debug & 4))
                        issue_stage<1, kPair>(d0 + (kKW / 2) * P.n_tile, a_lo, b_lo, desc_hi, idesc_res, P.MT, P.ns,
                                              (P.rows_sub * P.TW * 128u) >> 4, 0, 0, 4, false);
                    if constexpr (kPair) umma_commit_pair(empty0 + 8 * slot);
                    else umma_commit(empty0 + 8 * slot);
                }
                __syncwarp();
                if (++slot == P.num_slots) { slot = 0; phase ^= 1; }
            }
            if (elect_one()) {                                 // accumulator complete -> epilogue (of both CTAs)
                if constexpr (kPair) umma_commit_pair(tfull0 + 8 * acc);
                else umma_commit(tfull0 + 8 * acc);
            }
            __syncwarp();
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        if (stat && lane == 0) { g_trace[301 * 8 + 0] = clock64() - st_t0; g_trace[301 * 8 + 1] = st_we; g_trace[301 * 8 + 2] = st_wf; }
    }
    } else {
        if constexpr (kPair) asm volatile("setmaxnreg.inc.sync.aligned.u32 216;");
        // =============================== epilogue ===================================
        // kEpiPerQ warps per TMEM lane quarter (hardware rule: a warp reads lanes 32*(warp%4)..+31): the warps
        // (wq, eh=0..kEpiPerQ-1) share the 32 pixels of quarter wq and split their channels.
        const int wq = (warp - 4) & 3;
        const int eh = (warp - 4) >> 2;
        const int p = wq * 32 + lane;
        const int py = p / P.TW, px = p - py * P.TW;
        int acc = 0, sbuf = 0;
        uint32_t acc_phase = 0;
        // staged path: the pair owns rows [32*wq, 32*wq+32) of each staging buffer (a 1 KiB-aligned region
        // of whole swizzle atoms) and stores them with its own TMA store - no CTA-wide barrier
        const uint32_t rowb = (uint32_t)P.n_store * 2u;
        const uint32_t msk = rowb == 128u ? 7u : (rowb == 64u ? 3u : 1u);
        const int rows_warp = 32 / P.TW;                  // image rows covered by one quarter's 32 pixels
        // a store block of n_store channels is split in 16-channel chunks over the kEpiPerQ warps of the quarter
        const int nsplit = min(kEpiPerQ, P.n_store / 16);
        const int cpw = P.n_store / nsplit;               // channels of a store block per working warp (16 or 32)
        // 16-channel direct-store epilogues (conv_last, the cleaner's image conv, SPyNet's flow conv) leave the second
        // warp of a quarter without channels: there the two warps own one accumulator buffer each (alternate tiles)
        const bool alt = kKW > 0 && !kStaged && P.epi_alt;
        const bool works = alt || eh < nsplit;
        const int cbeg = (works && !alt) ? eh * cpw : 0;
        // stacked layout (n_tile <= 64, one store block): this warp's bias values live in registers
        float bias_r[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) bias_r[i] = (kKW > 0 && i < cpw) ? bias_s[cbeg + i] : 0.f;
        const float act_k = P.epi.act_k;
        griddep_wait();        // this role reads/writes global memory other kernels on the stream own
        const int actm = act_k == 1.f ? 0 : (act_k == 0.f ? 1 : 2);
        const uint32_t tempty_lead = kPair ? mapa_rank(tempty0, 0) : 0u;
        TileWalk tw(blockIdx.x, gridDim.x, P.tiles_x, P.tiles_per_img);
        const bool estat = (P.debug & 32) && blockIdx.x == 0 && blockIdx.y == 0 && warp == 4;
        long long est_t0 = estat ? clock64() : 0, est_w = 0;
        for (int tile = blockIdx.x; tile - (int)crank < tiles_g; tile += gridDim.x, tw.next()) {
            const bool dummy = kPair && tile >= tiles_g;       // the pair's odd tile out: handshakes only
            if (alt && eh != acc) {                            // the twin warp's tile
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                continue;
            }
            const int li = tw.li, ty = tw.ty, tx = tw.tx;
            const int img = g * P.imgs_per_group + li;
            const int x = tx * P.TW + px;
            // image epilogues (<= 3 real channels) of the stacked layout take a 4-channel path; EPI_SR fetches its
            // bilinear skip term while the tile's MMAs are still running
            const bool narrow = kKW > 0 && !kStaged && P.epi.mode != VSRB_EPI_NHWC;
            // (EPI_CLEAN / EPI_FLOW likewise fetch the fp32 value they add to; plain layouts only - the split-bf16 mode
            // keeps the generic store)
            float upv[2][3];
            const bool prefetch = narrow && !dummy && !P.epi.split && (P.epi.mode != VSRB_EPI_CLEAN || P.epi.out_c >= 16);
            if (prefetch) {
#pragma unroll
                for (int m = 0; m < 2; ++m) {
                    const int y = ty * rows_tile + m * P.rows_sub + wq, xo = tx * P.UW + lane - kKW / 2;
                    upv[m][0] = upv[m][1] = upv[m][2] = 0.f;
                    if (m < P.MT && lane >= kKW / 2 && lane < 32 - kKW / 2 && y < P.H && xo < P.W) {
                        if (P.epi.mode == VSRB_EPI_SR) epi_sr_up(P.epi, img, y, xo, upv[m]);
                        else if (P.epi.mode == VSRB_EPI_CLEAN) epi_clean_fetch(P.epi, img, y, xo, upv[m]);
                        else epi_flow_fetch(P.epi, img, y, xo, upv[m]);
                    }
                }
            }
            const long long w2 = estat ? clock64() : 0;
            mbar_wait(tfull0 + 8 * acc, acc_phase, P.dbg, 5, dead);
            if (estat) est_w += clock64() - w2;
            tc_fence_after();
            if (tile == (int)blockIdx.x && warp == 4 && lane == 0) trace_stamp(P.debug, 4);
            for (int m = 0; m < (((P.debug & 8) || dummy) ? 0 : P.MT); ++m) {
                const uint32_t t0 = tmem_base + ((uint32_t)(wq * 32) << 16) + acc * P.acc_cols + m * P.ns;
                if constexpr (kKW > 0) {
                    // ---- stacked layout: the quarter is one image row, lane = box column; filter column kx
                    // sits in accumulator columns [kx*n_tile, (kx+1)*n_tile) and belongs to the output pixel
                    // kx - pad lanes to the left, so out[lane] = sum_kx D_kx[lane + kx - pad] (warp shuffles)
                    constexpr int PAD = kKW / 2;
                    const int y = ty * rows_tile + m * P.rows_sub + wq;
                    const bool lane_ok = lane >= PAD && lane < 32 - PAD;
                    const int xo = tx * P.UW + lane - PAD;
                    if (narrow) {
                        if (works) {
                            float v4[4];
                            stacked_chunk16<kKW, 2, 4>(t0, P.n_tile, bias_r, act_k, lane, v4);
                            if (lane_ok && y < P.H && xo < P.W && !(P.debug & 2)) {
                                if (prefetch) {
                                    const float up[3] = {m ? upv[1][0] : upv[0][0], m ? upv[1][1] : upv[0][1], m ? upv[1][2] : upv[0][2]};
                                    if (P.epi.mode == VSRB_EPI_SR) epi_sr_store(P.epi, img, y, xo, v4, up);
                                    else if (P.epi.mode == VSRB_EPI_CLEAN) epi_clean_store<__nv_bfloat16>(P.epi, img, y, xo, v4, up);
                                    else epi_flow_store(P.epi, img, y, xo, v4, up);
                                } else {
                                    float v[16];
#pragma unroll
                                    for (int i = 0; i < 16; ++i) v[i] = i < 4 ? v4[i] : 0.f;
                                    epi_store16<__nv_bfloat16, false>(P.epi, g, img, y, xo, 0, v);
                                }
                            }
                        }
                        continue;
                    }
                    for (int b0 = 0; b0 < P.n_tile; b0 += P.n_store) {
                        const uint32_t row_base = stg0 + sbuf * P.stg_bytes + (uint32_t)(wq * 32 + lane - PAD) * rowb;
                        if constexpr (kStaged && kKW == 3 && kPair) {
                            if (cpw == 32) {                                   // hot shape: pipelined TMEM reads
                                uint32_t ra[3][16];
                                const uint32_t ta = t0 + b0 + cbeg;
                                ld_taps3(ta, P.n_tile, ra);
                                if (eh == 0 && lane == 0) bulk_wait_read<1>();
                                pair_sync(wq, 32 * kEpiPerQ);
                                const uint32_t ro = row_base + (uint32_t)cbeg * 2u;
                                if (actm == 0) stacked3_two_chunks<0>(ra, ta, P.n_tile, bias_r, act_k, lane, lane_ok, ro, msk);
                                else if (actm == 1) stacked3_two_chunks<1>(ra, ta, P.n_tile, bias_r, act_k, lane, lane_ok, ro, msk);
                                else stacked3_two_chunks<2>(ra, ta, P.n_tile, bias_r, act_k, lane, lane_ok, ro, msk);
                                fence_proxy_async();
                                pair_sync(wq, 32 * kEpiPerQ);
                                if (eh == 0 && lane == 0 && !(P.debug & 2)) {
                                    const int n0 = qb * P.n_tile + b0;         // PixelShuffle: one output map per sub-pixel
                                    const int q = P.epi.pixshuf ? n0 / P.epi.cq : 0;
                                    tma_store_5d(&P.smap[q], stg0 + sbuf * P.stg_bytes + (uint32_t)(wq * 32) * rowb, n0 - q * P.epi.cq,
                                                 tx * P.UW, y, li, g);
                                    bulk_commit();
                                }
                                sbuf ^= 1;
                                continue;
                            }
                        }
                        if (kStaged) {
                            if (eh == 0 && lane == 0) bulk_wait_read<1>();
                            pair_sync(wq, 32 * kEpiPerQ);
                        }
                        if (works) {
#pragma unroll
                            for (int cc = 0; cc < 2; ++cc) {
                                const int c0 = cbeg + cc * 16;
                                if (cc * 16 < cpw) {
                                    float v[16];
                                    const uint32_t ta = t0 + b0 + c0;
                                    if (actm == 0) stacked_chunk16<kKW, 0>(ta, P.n_tile, bias_r + cc * 16, act_k, lane, v);
                                    else if (actm == 1) stacked_chunk16<kKW, 1>(ta, P.n_tile, bias_r + cc * 16, act_k, lane, v);
                                    else stacked_chunk16<kKW, 2>(ta, P.n_tile, bias_r + cc * 16, act_k, lane, v);
                                    if (kStaged) {
                                        if (lane_ok) {
                                            uint32_t o0 = row_base + (uint32_t)c0 * 2u, o1 = o0 + 16u;
                                            o0 ^= ((o0 >> 7) & msk) << 4;
                                            o1 ^= ((o1 >> 7) & msk) << 4;
                                            st_shared_v4(o0, pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]),
                                                         pack_bf16(v[6], v[7]));
                                            st_shared_v4(o1, pack_bf16(v[8], v[9]), pack_bf16(v[10], v[11]), pack_bf16(v[12], v[13]),
                                                         pack_bf16(v[14], v[15]));
                                        }
                                    } else if (lane_ok && y < P.H && xo < P.W && !(P.debug & 2)) {
                                        epi_store16<__nv_bfloat16, false>(P.epi, g, img, y, xo, qb * P.n_tile + b0 + c0, v);
                                    }
                                }
                            }
                        }
                        if (kStaged) {
                            fence_proxy_async();
                            pair_sync(wq, 32 * kEpiPerQ);
                            if (eh == 0 && lane == 0 && !(P.debug & 2)) {
                                const int n0 = qb * P.n_tile + b0;
                                const int q = P.epi.pixshuf ? n0 / P.epi.cq : 0;
                                tma_store_5d(&P.smap[q], stg0 + sbuf * P.stg_bytes + (uint32_t)(wq * 32) * rowb, n0 - q * P.epi.cq,
                                             tx * P.UW, y, li, g);
                                bulk_commit();
                            }
                            sbuf ^= 1;
                        }
                    }
                } else if (kStaged) {
                    for (int b0 = 0; b0 < P.n_tile; b0 += P.n_store) {
                        uint32_t r[2][16];
#pragma unroll
                        for (int j = 0; j < 2; ++j)
                            if (works && j * 16 < cpw) tmem_ld16_nowait(t0 + b0 + cbeg + j * 16, r[j]);
                        if (eh == 0 && lane == 0) bulk_wait_read<1>();      // the buffer used two stores ago is free again
                        pair_sync(wq, 32 * kEpiPerQ);
                        tmem_ld_wait();
                        const uint32_t row_base = stg0 + sbuf * P.stg_bytes + (uint32_t)p * rowb;
#pragma unroll
                        for (int j = 0; j < 2; ++j)
                            if (works && j * 16 < cpw)
                                stage_chunk(P.epi, r[j], bias_s + b0 + cbeg + j * 16, row_base, (uint32_t)(cbeg + j * 16) * 2u, msk);
                        fence_proxy_async();
                        pair_sync(wq, 32 * kEpiPerQ);
                        if (eh == 0 && lane == 0 && !(P.debug & 2)) {
                            const int n0 = qb * P.n_tile + b0;
                            const int q = P.epi.pixshuf ? n0 / P.epi.cq : 0;
                            const int ch = P.epi.pixshuf ? n0 - q * P.epi.cq : n0;
                            tma_store_5d(&P.smap[q], stg0 + sbuf * P.stg_bytes + (uint32_t)(wq * 32) * rowb, ch, tx * P.TW,
                                         ty * rows_tile + m * P.rows_sub + wq * rows_warp, li, g);
                            bulk_commit();
                        }
                        sbuf ^= 1;
                    }
                } else {
                    const int y = ty * rows_tile + m * P.rows_sub + py;
                    const bool valid = (y < P.H) && (x < P.W) && !(P.debug & 2);
                    for (int c0 = eh * 16; c0 < P.n_tile; c0 += 16 * kEpiPerQ) {     // the quarter's warps interleave 16-channel chunks
                        uint32_t r[16];
                        tmem_ld16_nowait(t0 + c0, r);
                        tmem_ld_wait();
                        float v[16];
#pragma unroll
                        for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]) + bias_s[c0 + i];
                        epi_act16(P.epi, v);
                        if (valid) epi_store16<__nv_bfloat16, false>(P.epi, g, img, y, x, qb * P.n_tile + c0, v);
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if constexpr (kPair) mbar_arrive_cluster(tempty_lead + 8 * acc);
                else mbar_arrive(tempty0 + 8 * acc);
            }
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        if (estat && lane == 0) { g_trace[302 * 8 + 0] = clock64() - est_t0; g_trace[302 * 8 + 1] = est_w; }
        if (warp == 4 && lane == 0) trace_stamp(P.debug, 5);
        if (kStaged && eh == 0 && lane == 0) bulk_wait_all();   // staged tiles must be read out before shared memory goes away
        if (warp == 4 && lane == 0) trace_stamp(P.debug, 6);
        tc_fence_before();
        if constexpr (kPair) cluster_sync_all();               // neither CTA may leave while its peer still signals it
        else asm volatile("bar.sync 0;" ::: "memory");
        return;
    }
    tc_fence_before();
    if constexpr (kPair) cluster_sync_all();
    else asm volatile("bar.sync 0;" ::: "memory");
    if (warp == 2) {
        tc_fence_after();
        if constexpr (kPair) tmem_dealloc_pair(tmem_base, 512);
        else tmem_dealloc(tmem_base, 512);
        if (lane == 0) trace_stamp(P.debug, 7);
    }
}

// 64 x 64 bf16 identity in the swizzle-128B K-major layout (row n, 16-byte chunk j at j ^ (n & 7))
__device__ __align__(1024) uint8_t g_identity[kIdentBytes];
__global__ void fill_identity_kernel() {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;   // element index, 64 x 64
    if (i >= 64 * 64) return;
    const int n = i >> 6, k = i & 63;
    uint32_t off = (uint32_t)n * 128u + (uint32_t)k * 2u;
    off ^= ((off >> 7) & 7u) << 4;
    *reinterpret_cast<__nv_bfloat16*>(g_identity + off) = __float2bfloat16_rn(n == k ? 1.f : 0.f);
}

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
// conv_tc_kernel<staged, kw, pair> by [staged][pair][kw: 0, 3, 7] (kw 0: classic layout, 3 / 7: stacked)
static void (*const kConvTcKernels[2][2][3])(TcParams) = {
    {{conv_tc_kernel<false, 0>, conv_tc_kernel<false, 3>, conv_tc_kernel<false, 7>},
     {conv_tc_kernel<false, 0, true>, conv_tc_kernel<false, 3, true>, conv_tc_kernel<false, 7, true>}},
    {{conv_tc_kernel<true, 0>, conv_tc_kernel<true, 3>, conv_tc_kernel<true, 7>},
     {conv_tc_kernel<true, 0, true>, conv_tc_kernel<true, 3, true>, conv_tc_kernel<true, 7, true>}}};

static bool g_dev_ready[kMaxDevices] = {false};
static const uint8_t* g_ident_ptr[kMaxDevices] = {nullptr};

int launch_conv_tc(const vsrb_conv_args* a, const ConvPlan& p, cudaStream_t stream) {
    int dev = 0, sms = 0;
    int rc = device_setup(&dev, &sms, g_dev_ready, [&](int d) {
        for (auto& by_pair : kConvTcKernels)
            for (auto& by_kw : by_pair)
                for (auto kern : by_kw) VSRB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemMax));
        void* ip = nullptr;
        VSRB_CUDA(cudaGetSymbolAddress(&ip, g_identity));
        g_ident_ptr[d] = reinterpret_cast<const uint8_t*>(ip);
        // one-time: finish before any other stream of this process can launch a conv that reads it
        fill_identity_kernel<<<16, 256, 0, stream>>>();
        VSRB_LAUNCH_CHECK();
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        cudaStreamIsCapturing(stream, &cap);
        if (cap == cudaStreamCaptureStatusNone) VSRB_CUDA(cudaStreamSynchronize(stream));
        return VSRB_OK;
    });
    if (rc != VSRB_OK) return rc;
    TcParams P;
    memset(&P, 0, sizeof(P));
    P.n_seg = p.n_seg; P.kh = p.kh; P.kw = p.kw; P.H = a->h; P.W = a->w;
    P.groups = p.groups; P.imgs_per_group = a->imgs_per_group;
    P.n_tile = p.n_tile; P.n_blocks = p.n_blocks;
    P.wblock_bytes = (uint32_t)p.wblock_bytes;
    P.w = reinterpret_cast<const uint8_t*>(a->packed) + p.bias_bytes;
    P.ident = g_ident_ptr[dev];
    P.dbg = debug_flag();
    P.debug = env_int("VSRB_TC_DEBUG");
    fill_epi(a, p, &P.epi);

    P.TW = p.stacked ? 32 : (a->w <= 8 ? 8 : 16);
    P.rows_sub = 128 / P.TW;
    P.UW = p.stacked ? P.TW - (p.kw - 1) : P.TW;
    P.kxs = p.stacked ? 1 : p.kw;
    P.ns = p.ns;
    P.res_xoff = p.stacked ? p.kw / 2 : 0;
    const int units = p.groups * p.n_blocks;
    const int ctas_budget = (a->max_ctas > 0 ? a->max_ctas : sms);

    // EPI_NHWC tiles leave through two swizzled staging buffers and TMA stores (full-line, asynchronous
    // writes); needs positive 16-byte-multiple strides.
    const long long oimg = P.epi.out_img_stride, ogrp = P.epi.out_group_stride;
    bool staged = a->epilogue == VSRB_EPI_NHWC && oimg > 0 && ogrp > 0 && oimg % 8 == 0 && ogrp % 8 == 0 && !a->split &&
                  (reinterpret_cast<uintptr_t>(a->out) & 15) == 0;
    P.n_store = (p.n_tile % 64 == 0) ? 64 : ((p.n_tile % 32 == 0) ? 32 : 16);   // store block must divide n_tile
    if (p.pixshuf && p.cout / 4 < P.n_store) P.n_store = p.cout / 4;
    if (P.n_store != 16 && P.n_store != 32 && P.n_store != 64) staged = false;
    P.stg_bytes = (int)round_up((size_t)128 * P.n_store * 2, 4096);
    const int stg_total = staged ? 2 * P.stg_bytes : 0;

    // residual: folded into the accumulation by an identity-matrix MMA stage when it has the plain
    // resblock shape; otherwise the direct-store epilogue adds it
    P.res_mma = staged && a->residual && a->act == VSRB_ACT_NONE && p.n_tile == 64 && p.n_blocks == 1 && a->res_c % 8 == 0 &&
                (reinterpret_cast<uintptr_t>(a->residual) & 15) == 0;
    if (a->residual && !P.res_mma) staged = false;
    P.epi_alt = (!staged && p.stacked && P.n_store == 16 && kEpiPerQ == 2) ? 1 : 0;
    if (P.res_mma) P.epi.res = nullptr;
    const int ident_total = P.res_mma ? kIdentBytes : 0;

    const int avail = kSmemMax - kCtrlBytes - 1024 - (staged ? stg_total : 0) - ident_total;
    // CTA pairs (cta_group::2) for staged NHWC stacked 3x3 / 7x7 convs whose half weight block stays resident (every CTA
    // holds ns/2 rows of each filter row: whole 8-row swizzle atoms; N of an M=256 MMA is a multiple of 16)
    // (narrow tiles, N < 96, are bound by the A fetch and the per-tile handshake, which is longer across two CTAs: no pairs)
    // Classic-layout convs with wide tiles (the 64->256 upsampling conv, N = 128) pair the same way.
    bool pair = ((p.stacked && (p.kw == 3 || p.kw == 7) && p.kh == p.kw) || (!p.stacked && p.kh == 3 && p.n_tile >= 128)) &&
                (p.ns / 2) % 8 == 0 && p.ns % 16 == 0 && p.ns >= 96 && !getenv("VSRB_TC_NO_PAIR");
    for (int attempt = 0; attempt < 2; ++attempt) {
    int MT = (2 * 2 * p.ns <= 512) ? 2 : 1;
    if (MT == 2) {
        long tiles2 = (long)a->imgs_per_group * ceil_div(a->h, 2 * P.rows_sub) * ceil_div(a->w, P.UW) * units;
        if (a->h <= P.rows_sub || tiles2 < 2L * ctas_budget) MT = 1;
    }
    for (;; MT = 1) {
        P.MT = MT;
        P.box_rows = P.rows_sub * MT + p.kh - 1;
        int amax = 0, abmax = 0;
        for (int s = 0; s < p.n_seg; ++s) {
            P.seg_abytes[s] = P.box_rows * P.TW * p.seg[s].rowbytes;
            amax = amax > P.seg_abytes[s] ? amax : P.seg_abytes[s];
            int ab = P.seg_abytes[s] + p.b_stage_bytes[s];
            abmax = abmax > ab ? abmax : ab;
        }
        P.res_abytes = (uint32_t)(P.rows_sub * MT * P.TW * 128);
        if (P.res_mma) {
            amax = amax > (int)P.res_abytes ? amax : (int)P.res_abytes;
            abmax = abmax > (int)P.res_abytes ? abmax : (int)P.res_abytes;
        }
        const int slot_res = (int)round_up(amax, 1024), slot_str = (int)round_up(abmax, 1024);
        const int wres = (int)round_up(pair ? p.wblock_bytes / 2 : p.wblock_bytes, 1024);
        if (P.box_rows <= 256 && wres + (pair ? 2 : 3) * slot_res <= avail) {
            P.resident = 1; P.wres_bytes = wres; P.slot_bytes = slot_res;
            P.num_slots = (avail - wres) / slot_res;
        } else {
            P.resident = 0; P.wres_bytes = 0; P.slot_bytes = slot_str;
            P.num_slots = avail / slot_str;
        }
        if (P.num_slots > kMaxSlots) P.num_slots = kMaxSlots;
        if (P.num_slots >= 2 && P.box_rows <= 256) break;
        if (MT == 1) {
            set_error("conv tile does not fit shared memory (kh=%d n_tile=%d)", p.kh, p.n_tile);
            return VSRB_E_SMEM;
        }
    }
    if (!pair || P.resident) break;
    pair = false;                                   // the pair kernel only exists for resident weights
    }
    P.acc_cols = P.MT * p.ns;
    P.tiles_x = ceil_div(a->w, P.UW);
    P.tiles_per_img = P.tiles_x * ceil_div(a->h, P.rows_sub * P.MT);
    {
        uint32_t woff = 0;
        for (int s = 0; s < p.n_seg; ++s) {
            const SegPlan& sp = p.seg[s];
            P.seg_chunks[s] = sp.chunks; P.seg_ck[s] = sp.ck; P.seg_rowbytes[s] = sp.rowbytes;
            P.seg_layout[s] = sp.layout; P.seg_bstage[s] = p.b_stage_bytes[s]; P.seg_stages[s] = sp.chunks * P.kxs;
            P.seg_woff[s] = woff;
            woff += (uint32_t)P.seg_stages[s] * (uint32_t)p.b_stage_bytes[s];
        }
    }
    P.n_ops = a->n_in ? a->n_in : p.n_seg;
    for (int s = 0; s < P.n_ops; ++s) {            // s = operand index
        P.op_wseg[s] = a->n_in ? a->in_wseg[s] : s;
        P.op_c0[s] = a->n_in ? a->in_c0[s] : 0;
        const SegPlan& sp = p.seg[P.op_wseg[s]];
        VSRB_CHECK_ARG(a->in_c[s] % 8 == 0, "segment %d: channel stride %d must be a multiple of 8", s, a->in_c[s]);
        VSRB_CHECK_ARG((reinterpret_cast<uintptr_t>(a->in[s]) & 15) == 0, "segment %d: pointer not 16-byte aligned", s);
        rc = encode_nhwc(&P.tmap[s], "input", a->in[s], a->in_c[s], a->w, a->h, a->batch, sp.ck, P.TW, P.box_rows);
        if (rc != VSRB_OK) return rc;
    }
    if (P.res_mma) {
        rc = encode_nhwc(&P.rmap, "residual", a->residual, a->res_c, a->w, a->h, a->batch, 64, P.TW, P.rows_sub * P.MT);
        if (rc != VSRB_OK) return rc;
    }
    if (staged) {
        const int nq = p.pixshuf ? 4 : 1, sx = p.pixshuf ? 2 : 1;
        const long long OW = (long long)sx * a->w;
        for (int q = 0; q < nq; ++q) {
            char* obase = reinterpret_cast<char*>(a->out) + (((long long)(q >> 1) * OW + (q & 1)) * a->out_c) * 2;
            cuuint64_t dims[5] = {(cuuint64_t)a->out_c, (cuuint64_t)a->w, (cuuint64_t)a->h, (cuuint64_t)a->imgs_per_group,
                                  (cuuint64_t)p.groups};
            cuuint64_t strides[4] = {(cuuint64_t)sx * a->out_c * 2, (cuuint64_t)sx * OW * a->out_c * 2, (cuuint64_t)oimg * 2,
                                     (cuuint64_t)ogrp * 2};
            cuuint32_t box[5] = {(cuuint32_t)P.n_store, (cuuint32_t)P.UW, (cuuint32_t)(p.stacked ? 1 : 32 / P.TW), 1, 1};
            rc = encode_map(&P.smap[q], "store", obase, 5, dims, strides, box, swizzle_for(P.n_store));
            if (rc != VSRB_OK) return rc;
        }
    }
    const int tiles_g = a->imgs_per_group * P.tiles_per_img;
    int ctas_x = ctas_budget / units;
    if (ctas_x < 1) ctas_x = 1;
    if (ctas_x > tiles_g) ctas_x = tiles_g;
    if (pair) {                                     // whole pairs; an odd tile count leaves one dummy tile
        const int want = (int)round_up((size_t)tiles_g, 2);
        ctas_x = (ctas_budget / units) & ~1;
        if (ctas_x < 2) ctas_x = 2;
        if (ctas_x > want) ctas_x = want;
    }
    const int smem = kCtrlBytes + 1024 + (int)P.wres_bytes + ident_total + P.num_slots * P.slot_bytes + (staged ? stg_total : 0);
    P.pdl = (a->flags & VSRB_CONV_PDL) ? 1 : 0;
    const int kkw = p.stacked ? p.kw : 0;
    return launch_ex(kConvTcKernels[staged][pair][kkw == 3 ? 1 : (kkw == 7 ? 2 : 0)], P, dim3(ctas_x, units), dim3(kThreads), smem,
                     stream, P.pdl, pair ? 2 : 1);
}

}  // namespace vsrb

extern "C" int vsrb_debug_trace(uint64_t* out, int32_t n_ctas) {
    using namespace vsrb;
    VSRB_CHECK_ARG(out && n_ctas >= 1 && n_ctas <= kTraceCtas, "debug_trace: 1..%d CTAs", kTraceCtas);
    VSRB_CUDA(cudaDeviceSynchronize());
    VSRB_CUDA(cudaMemcpyFromSymbol(out, g_trace, sizeof(unsigned long long) * 8 * (size_t)n_ctas));
    return VSRB_OK;
}
