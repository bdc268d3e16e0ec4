// 3x3 64->64 convolution as a "ring walk": the hot layer of Real-BasicVSR (every ResidualConv of the cleaner, of the two
// propagation trunks and conv_last.0 at 720p; reference conv.py:89-92, basicvsr.py:20,81) on tcgen05/TMEM/TMA.
//
// conv_tc.cu's stacked layout puts the three filter COLUMNS side by side along the MMA N dimension, which leaves the
// epilogue three partial sums per output to fetch from TMEM (192 accumulator columns per 128 pixels at 64 B/clk/SM: the
// bound of that kernel) and to recombine with warp shuffles.  Here the three filter ROWS are stacked along N instead and
// the column shift kx is a start-address offset of the A operand (a K-major SW128 operand may start at any 128-byte row
// of its tile: tools/umma_offset_test.cu).  A CTA walks DOWN the image one input row per step:
//
//   * M = 128 lanes = 4 lane quarters x 32 pixels.  Every quarter walks its own range of rows of a 30-pixel-wide column
//     strip (32-pixel boxes with a one-pixel halo left and right; lanes 30,31 of a quarter compute garbage, dropped).
//   * step t loads input row t of each quarter (four 4 KiB TMA boxes) and issues, per kx and per K=16 step, ONE MMA with
//     N = 192 = [W(ky=2) | W(ky=1) | W(ky=0)]: input row t contributes to output rows t-1, t, t+1.  Output rows live in
//     six accumulator slots, slot = (row + 1) mod 6; the MMA of step t writes the three consecutive 64-column blocks
//     starting at block t mod 6 of the 8 blocks TMEM has.  Blocks 6 and 7 are overflow aliases of slots 0 and 1: when the
//     triple starts at block 4 or 5 the contributions for slot 0 / 1 land there, and the epilogue of those two slots adds
//     the alias block to the main one - so the MMA never has to be split where the ring wraps.
//   * after step t output row t-1 is complete: ONE epilogue warp (the two warps of a lane quarter take alternate rows)
//     reads its 64-column block (3x fewer TMEM reads than the stacked layout, no shuffles), re-initialises it with the
//     bias (tcgen05.st: every MMA accumulates, the bias costs nothing), applies the activation, adds the residual - TMA-
//     loaded into the warp's staging row beforehand - and stores the bf16 row with one TMA store.
//   * CTA pairs (cta_group::2): the leader issues M = 256 MMAs for both CTAs' walks; each CTA holds half of the rows of
//     every B tile (rank 0: [ky2 | ky1 lower half], rank 1: [ky1 upper half | ky0]).
//
// The propagation stem's flow_warp is not folded in here: epilogue warps that also sample the operand rows through the
// flow were measured slower than the separate warp kernel plus this stem (DESIGN §4.1c).
//
// Work split: the rows of all column strips of a weight group are cut into 4 * gridDim.x ranges, either as one linear
// index space (large launches: a range that starts mid-strip loads one halo row above and below, a range that crosses
// into the next strip pays two zero rows - TMA out-of-bounds fill is the conv's zero padding) or, for small launches,
// as an equal number of ranges per strip (no crossings).  The launcher picks whichever needs fewer steps.
#include <stdlib.h>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace vsrb {

static constexpr int kRingThreads = 384;              // 4 control warps + 8 epilogue warps
static constexpr int kRingSlots = 8;                  // activation rows in flight (6 when a patch operand rides along)
static constexpr int kRingSlotBytes = 17 * 1024;      // 4 quarters x 32 pixels x 128 B + the two rows a kx shift runs over
static constexpr int kRingPatchBytes = 8 * 1024;      // 4 quarters x 32 pixels x 64 B of 3x3 im2col patches
static constexpr int kRingSlotsPatch = 6;
static constexpr int kRingUW = 30;                    // useful output columns of a 32-pixel quarter
static constexpr int kRingStageBytes = 8 * 4096;      // one staging row (32 pixels x 128 B) per epilogue warp
static constexpr int kRingCtrl = 1024;
static constexpr int kRingSlotArea = kRingSlotsPatch * (kRingSlotBytes + kRingPatchBytes) > kRingSlots * kRingSlotBytes
                                         ? kRingSlotsPatch * (kRingSlotBytes + kRingPatchBytes) : kRingSlots * kRingSlotBytes;
static constexpr int kRingSmem = kRingCtrl + 1024 + VSRB_RING_W_BYTES + kRingSlotArea + kRingStageBytes;
static constexpr int kRingAcc = 6;                    // accumulator slots (output rows in flight)

struct RingParams {
    CUtensorMap in_map;    // [C, W, H, B] box {64, 32, 1, 1}
    CUtensorMap res_map;   // residual, same geometry
    CUtensorMap out_map;   // [out_c, W, H, imgs_per_group, groups] box {64, 30, 1, 1, 1}
    CUtensorMap patch_map[2];   // per weight group: 3x3 im2col patches [32, W, H, imgs_per_group] box {32, 32, 1, 1} (SW64)
    int has_main, has_patch;    // operands: the 64-channel segment (N = 192 ring MMAs) / the 3-channel segment as K = 32 patches
    int num_slots, slot_bytes;
    const uint8_t* w;      // ring image: [group][rank]{[kx][96 rows][128 B] | patch [32 rows][64 B]}
    const float* bias;     // [group][64]
    int has_res;
    int H, strips, ipg;
    int cols;              // ipg * strips column strips per weight group
    int rpc;               // ranges per column strip (aligned split), 0 = linear split of all rows
    uint32_t rows_g;       // cols * H
    float act_k;
    int* dbg;
    int debug;             // VSRB_RING_DEBUG bits (timing experiments only): 1 no loads, 2 no stores, 4 no MMA, 8 no epilogue math
};

// One lane quarter's share of the rows: the linear range [lo, hi) of (column strip, row) pairs, visited as items
// (column, input row y): for every stretch of output rows [ya, yb) inside one column the input rows ya-1 .. yb.
// An item's own row is an output row of this quarter iff ya <= y < yb.
struct RingWalk {
    uint32_t lo, hi;
    int H, col, ya, yb, y;
    bool done;
    __device__ __forceinline__ void init(uint32_t lo_, uint32_t hi_, int H_) {
        lo = lo_; hi = hi_; H = H_;
        done = lo >= hi;
        if (!done) {
            col = (int)(lo / (uint32_t)H);
            ya = (int)(lo - (uint32_t)col * H);
            const uint32_t rest = hi - lo;
            yb = (rest < (uint32_t)(H - ya)) ? ya + (int)rest : H;
            y = ya - 1;
        }
    }
    __device__ __forceinline__ bool valid() const { return !done && y >= ya && y < yb; }
    __device__ __forceinline__ void next() {
        if (done) return;
        if (++y > yb) {
            lo += yb - ya;
            if (lo >= hi) { done = true; return; }
            ++col;
            ya = 0;
            const uint32_t rest = hi - lo;
            yb = rest < (uint32_t)H ? (int)rest : H;
            y = -1;
        }
    }
};

// rows [lo, hi) of range r (linear index = column * H + row).  32-bit arithmetic: the launcher only takes this kernel
// when rows_g * n_ranges < 2^31 (a 64-bit division costs ~100 cycles and every role computes eight of these up front).
__host__ __device__ __forceinline__ void ring_range(uint32_t rows_g, int H, int cols, int rpc, int n_ranges, int r, uint32_t& lo,
                                                    uint32_t& hi) {
    if (rpc > 0) {
        const int col = r / rpc, part = r - col * rpc;
        if (col >= cols) { lo = hi = 0; return; }
        lo = (uint32_t)col * H + (uint32_t)(H * part) / (uint32_t)rpc;
        hi = (uint32_t)col * H + (uint32_t)(H * (part + 1)) / (uint32_t)rpc;
    } else {
        lo = rows_g * (uint32_t)r / (uint32_t)n_ranges;
        hi = rows_g * (uint32_t)(r + 1) / (uint32_t)n_ranges;
    }
}
// number of items (= steps) of range [lo, hi)
__host__ __device__ __forceinline__ int ring_items(uint32_t lo, uint32_t hi, int H) {
    if (hi <= lo) return 0;
    const uint32_t c0 = lo / (uint32_t)H, c1 = (hi - 1) / (uint32_t)H;
    return (int)(hi - lo) + 2 * (int)(c1 - c0 + 1);
}

__device__ __forceinline__ void tmem_st32(uint32_t taddr, const float (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]), "f"(v[8]), "f"(v[9]),
          "f"(v[10]), "f"(v[11]), "f"(v[12]), "f"(v[13]), "f"(v[14]), "f"(v[15]), "f"(v[16]), "f"(v[17]), "f"(v[18]), "f"(v[19]),
          "f"(v[20]), "f"(v[21]), "f"(v[22]), "f"(v[23]), "f"(v[24]), "f"(v[25]), "f"(v[26]), "f"(v[27]), "f"(v[28]), "f"(v[29]),
          "f"(v[30]), "f"(v[31])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ uint4 ld_shared_v4(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
    return v;
}
// bias (or zeros) into the 64 columns of one accumulator block, this warp's 32 lanes
__device__ __forceinline__ void ring_fill_block(uint32_t taddr, const float* bias64) {
    float b[32];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float4 f = bias64 ? reinterpret_cast<const float4*>(bias64)[h * 8 + i] : make_float4(0.f, 0.f, 0.f, 0.f);
            b[4 * i] = f.x; b[4 * i + 1] = f.y; b[4 * i + 2] = f.z; b[4 * i + 3] = f.w;
        }
        tmem_st32(taddr + h * 32, b);
    }
}

// VSRB_RING_DEBUG bit 64: cycle counters of CTA (0,0): [0] issuer waiting for a free accumulator slot, [1] issuer waiting for
// operand rows, [2] steps, [3] epilogue warp 4 waiting for finished rows, [4] its epilogue time (vsrb_ring_debug_stats)
__device__ unsigned long long g_ring_stat[8];
__device__ __forceinline__ long long ring_clock() { return clock64(); }

__global__ void __launch_bounds__(kRingThreads, 1) conv_ring_kernel(const __grid_constant__ RingParams P) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    uint8_t* base_ptr = smem_raw + (base - raw);
    // control block: barriers, TMEM base, bias
    const uint32_t full0 = base, empty0 = base + 64, tfull0 = base + 128, tempty0 = base + 176, rbar0 = base + 224, wbar = base + 288,
                   wready = base + 296;
    const int kSlots = P.num_slots;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(base_ptr + 304);
    float* bias_s = reinterpret_cast<float*>(base_ptr + 512);
    // then the weights, the operand slots (wres + VSRB_RING_W_BYTES) and one staging row per epilogue warp.  Each role
    // computes the addresses it needs from wres: a slot base held from here on is spilled by ptxas.
    const uint32_t wres = base + kRingCtrl;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.y;
    const uint32_t crank = cluster_ctarank();
    const int n_ranges = 4 * (int)gridDim.x;
    const int pair0 = ((int)blockIdx.x & ~1) * 4;                // first range of this CTA pair
    // steps of the pair: the longest of its eight walks
    int S = 0;
    {
        uint32_t lo, hi;
        ring_range(P.rows_g, P.H, P.cols, P.rpc, n_ranges, pair0 + (lane & 7), lo, hi);       // lane r of 8 takes range r
        S = ring_items(lo, hi, P.H);
#pragma unroll
        for (int o = 4; o >= 1; o >>= 1) S = max(S, __shfl_xor_sync(0xffffffffu, S, o));
    }

    if (warp == 0 && lane == 0) {
        if (P.has_main) prefetch_tensormap(&P.in_map);
        if (P.has_patch) prefetch_tensormap(&P.patch_map[g]);
        prefetch_tensormap(&P.out_map);
        if (P.has_res) prefetch_tensormap(&P.res_map);
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < kSlots; ++i) {
            mbar_init(full0 + 8 * i, 1);                          // the TMA bytes have landed (expect_tx of the leader's producer)
            mbar_init(empty0 + 8 * i, 1);
        }
        for (int i = 0; i < kRingAcc; ++i) {
            mbar_init(tfull0 + 8 * i, 1);
            mbar_init(tempty0 + 8 * i, 8);                        // one epilogue warp per lane quarter and CTA of the pair
        }
        for (int i = 0; i < 8; ++i) mbar_init(rbar0 + 8 * i, 1);
        mbar_init(wbar, 1);
        mbar_init(wready, 2);
        fence_barrier_init();
    }
    if (warp == 3)
        for (int i = lane; i < 64; i += 32) bias_s[i] = __ldg(P.bias + (size_t)g * 64 + i);
    cluster_sync_all();        // the peer's barriers must exist before anything is signalled across (also publishes bias_s)
    griddep_launch();
    uint32_t tmem_base = 0;
    if (warp >= 1) {
        if (warp == 2) tmem_alloc_pair(smem_u32(tmem_slot), 512);
        tc_fence_before();
        asm volatile("bar.sync 5, %0;" ::"n"(kRingThreads - 32) : "memory");
        tc_fence_after();
        tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
    }
    bool dead = false;

    if (warp < 4) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 72;");
        if (warp == 0) {
            // =============================== TMA producer ===============================
            if (lane == 0) {                                      // this CTA's half of every filter column's B tile
                const uint8_t* wsrc = P.w + ((size_t)g * 2 + crank) * VSRB_RING_W_BYTES;
                mbar_expect_tx(wbar, VSRB_RING_W_BYTES);
                bulk_load(wres, wsrc, VSRB_RING_W_BYTES, wbar);
            }
            __syncwarp();
            griddep_wait();        // activations come from the previous kernel(s)
            // lane q < 4 walks quarter q of this CTA; every lane knows how many of the pair's quarters are active at step t
            int items[8];
            RingWalk wk;
            {
                uint32_t lo, hi;
                ring_range(P.rows_g, P.H, P.cols, P.rpc, n_ranges, pair0 + (lane & 7), lo, hi);
                const int mine = ring_items(lo, hi, P.H);
#pragma unroll
                for (int r = 0; r < 8; ++r) items[r] = __shfl_sync(0xffffffffu, mine, r);
                const int src = (int)crank * 4 + (lane & 3);                                   // lane q < 4 walks this CTA's quarter q
                wk.init(__shfl_sync(0xffffffffu, lo, src), __shfl_sync(0xffffffffu, hi, src), P.H);
            }
            const uint32_t full_lead = mapa_rank(full0, 0);
            int slot = 0;
            uint32_t phase = 0;
            for (int t = 0; t < S; ++t) {
                if ((P.debug & 1) && crank != 0) break;            // (timing experiment without loads: nothing paces this warp)
                mbar_wait(empty0 + 8 * slot, phase ^ 1, P.dbg, 11, dead);
                if (P.debug & 1) {
                    if (lane == 0 && crank == 0) mbar_arrive(full0 + 8 * slot);
                } else if (lane == 0 && crank == 0) {
                    int act = 0;
#pragma unroll
                    for (int r = 0; r < 8; ++r) act += t < items[r] ? 1 : 0;
                    mbar_expect_tx(full0 + 8 * slot, (uint32_t)act * ((P.has_main ? 4096u : 0u) + (P.has_patch ? 2048u : 0u)));
                }
                if (lane < 4 && !wk.done && !(P.debug & 1)) {
                    const int li = wk.col / P.strips, strip = wk.col - li * P.strips;
                    const uint32_t sa = wres + VSRB_RING_W_BYTES + slot * P.slot_bytes;
                    if (P.has_main)
                        tma_load_4d_pair(&P.in_map, full_lead + 8 * slot, sa + lane * 4096, 0, strip * kRingUW - 1, wk.y, g * P.ipg + li);
                    if (P.has_patch)      // the im2col row of this item's own pixels: no halo column, no kx shift
                        tma_load_4d_pair(&P.patch_map[g], full_lead + 8 * slot, sa + kRingSlotBytes + lane * 2048, 0, strip * kRingUW, wk.y, li);
                }
                wk.next();
                __syncwarp();
                if (++slot == kSlots) { slot = 0; phase ^= 1; }
            }
        } else if (warp == 1) {
            // =============================== MMA issuer (leader CTA) ====================
            mbar_wait(wbar, 0, P.dbg, 12, dead);
            if (elect_one()) mbar_arrive_cluster(mapa_rank(wready, 0));
            __syncwarp();
            if (crank == 0) {
                mbar_wait(wready, 0, P.dbg, 13, dead);             // both CTAs' weights are resident
                // instruction descriptor: D=f32, A=B=bf16, K-major both, N = 192 (>>3 @17), M = 256 (>>4 @24) across the pair
                const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((192u >> 3) << 17) | (16u << 24);
                const uint32_t idesc_p = (1u << 4) | (1u << 7) | (1u << 10) | ((64u >> 3) << 17) | (16u << 24);
                const uint32_t desc_hi = ((128u * 8u) >> 4) | (1u << 14) | (2u << 29);       // SBO = 8 rows, SW128
                const uint32_t desc_hi_p = ((64u * 8u) >> 4) | (1u << 14) | (4u << 29);      // 64-byte rows, SW64
                const uint32_t w_lo = ((wres >> 4) & 0x3FFFu) | (1u << 16);
                const uint32_t wp_lo = (((wres + VSRB_RING_W_MAIN) >> 4) & 0x3FFFu) | (1u << 16);
                int slot = 0, b0 = 0, nb = 2;                       // b0 = t mod 6, nb = (t + 2) mod 6
                uint32_t phase = 0, nb_phase = 0;                   // nb_phase = ((t + 2) / 6) & 1
                mbar_wait(tempty0 + 0, 0, P.dbg, 14, dead);         // step 0 also touches slots 0 and 1 for the first time
                mbar_wait(tempty0 + 8, 0, P.dbg, 14, dead);
                for (int t = 0; t < S; ++t) {
                    // the slot of output row t+1 is touched for the first time at this step: its previous tenant
                    // (row t-5) must have been read out and the block(s) re-initialised
                    const bool stat = (P.debug & 64) && blockIdx.x == 0 && blockIdx.y == 0 && lane == 0;
                    const long long c0 = stat ? ring_clock() : 0;
                    mbar_wait(tempty0 + 8 * nb, nb_phase, P.dbg, 15, dead);
                    const long long c1 = stat ? ring_clock() : 0;
                    mbar_wait(full0 + 8 * slot, phase, P.dbg, 16, dead);
                    if (stat) {
                        const long long c2 = ring_clock();
                        atomicAdd(&g_ring_stat[0], (unsigned long long)(c1 - c0));
                        atomicAdd(&g_ring_stat[1], (unsigned long long)(c2 - c1));
                        atomicAdd(&g_ring_stat[2], 1ull);
                    }
                    tc_fence_after();
                    if (elect_one()) {
                        const uint32_t sa = wres + VSRB_RING_W_BYTES + slot * P.slot_bytes;
                        const uint32_t a_lo = ((sa >> 4) & 0x3FFFu) | (1u << 16);
                        const uint32_t d0 = tmem_base + (uint32_t)b0 * 64u;
                        if (P.has_patch && !(P.debug & 4)) {
                            // the 27-tap neighbourhood of this row's own pixels: straight into the block of output row t
                            const uint32_t ap_lo = (((sa + kRingSlotBytes) >> 4) & 0x3FFFu) | (1u << 16);
#pragma unroll
                            for (int k = 0; k < 2; ++k)
                                umma_bf16_pair(d0 + 64u, ((uint64_t)desc_hi_p << 32) | (ap_lo + k * 2), ((uint64_t)desc_hi_p << 32) | (wp_lo + k * 2),
                                               idesc_p, 1u);
                        }
#pragma unroll
                        for (int kx = 0; kx < 3; ++kx) {
                            if ((P.debug & 4) || !P.has_main) break;
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                const uint64_t ad = ((uint64_t)desc_hi << 32) | (a_lo + kx * 8 + k * 2);       // + kx rows of 128 B
                                const uint64_t bd = ((uint64_t)desc_hi << 32) | (w_lo + kx * (96 * 8) + k * 2);
                                umma_bf16_pair(d0, ad, bd, idesc, 1u);
                            }
                        }
                        umma_commit_pair(empty0 + 8 * slot);       // the slot is free (both CTAs) when these MMAs retire
                        umma_commit_pair(tfull0 + 8 * b0);         // ... and output row t-1 is complete
                    }
                    __syncwarp();
                    if (++slot == kSlots) { slot = 0; phase ^= 1; }
                    if (++b0 == kRingAcc) b0 = 0;
                    if (++nb == kRingAcc) { nb = 0; nb_phase ^= 1; }
                }
            }
        }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 216;");
        // =============================== epilogue ===================================
        const int q = warp & 3;                   // TMEM lane quarter (hardware: warp % 4) = walk of this warp
        const int eh = (warp - 4) >> 2;           // this warp takes the output rows p with (p & 1) == eh
        const uint32_t t_q = tmem_base + ((uint32_t)(q * 32) << 16);
        const uint32_t tempty_lead = mapa_rank(tempty0, 0);
        // every slot starts out holding the bias (alias blocks: zero); "empty" phase 0 of a slot = this initialisation,
        // done by the warp that will own the slot's tenants: row p = s - 1 (mod 6) has parity (s + 1) & 1
        for (int s = 0; s < kRingAcc; ++s) {
            if (((s + 1) & 1) != eh) continue;
            ring_fill_block(t_q + s * 64, bias_s);
            if (s < 2) ring_fill_block(t_q + (6 + s) * 64, nullptr);
        }
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0)
            for (int s = 0; s < kRingAcc; ++s)
                if (((s + 1) & 1) == eh) mbar_arrive_cluster(tempty_lead + 8 * s);
        RingWalk wk;
        {
            uint32_t lo, hi;
            ring_range(P.rows_g, P.H, P.cols, P.rpc, n_ranges, pair0 + (int)crank * 4 + q, lo, hi);
            wk.init(lo, hi, P.H);
        }
        // this warp's staging row
        const uint32_t stg = wres + VSRB_RING_W_BYTES + (uint32_t)P.num_slots * (uint32_t)P.slot_bytes + (uint32_t)(eh * 4 + q) * 4096u;
        const float act_k = P.act_k;
        const uint32_t rbar = rbar0 + 8 * (eh * 4 + q);
        uint32_t rphase = 0;
        griddep_wait();        // this role reads / writes global memory other kernels on the stream own
        // output row p (p = -1 is the ring's dummy first tenant) is complete after step p + 1; slot = (p + 1) mod 6
        int slot = 0;
        uint32_t sphase = 0;                      // ((p + 1) / 6) & 1
        for (int p = -1; p <= S - 2; ++p) {
            const bool mine = (p & 1) == eh;
            const bool valid = mine && p >= 0 && wk.valid();
            int li = 0, x0 = 0, y = 0;
            if (valid) {
                li = wk.col / P.strips;
                x0 = (wk.col - li * P.strips) * kRingUW;
                y = wk.y;
            }
            if (p >= 0) wk.next();
            const int s = slot;
            const uint32_t sp = sphase;
            if (++slot == kRingAcc) { slot = 0; sphase ^= 1; }
            if (!mine) continue;
            if (valid && !(P.debug & 8)) {
                // the staging row is free once the previous store has read it; the residual row is fetched into it
                if (lane == 0) {
                    bulk_wait_read<0>();
                    if (P.has_res) {
                        mbar_expect_tx(rbar, 4096u);
                        tma_load_4d(&P.res_map, rbar, stg, 0, x0, y, g * P.ipg + li);
                    }
                }
                __syncwarp();
            }
            const bool estat = (P.debug & 64) && blockIdx.x == 0 && blockIdx.y == 0 && warp == 4 && lane == 0;
            const long long e0 = estat ? ring_clock() : 0;
            mbar_wait(tfull0 + 8 * s, sp, P.dbg, 17, dead);
            const long long e1 = estat ? ring_clock() : 0;
            if (estat) atomicAdd(&g_ring_stat[3], (unsigned long long)(e1 - e0));
            tc_fence_after();
            float v[64];
            if (valid) {
                uint32_t r[4][16];
#pragma unroll
                for (int i = 0; i < 4; ++i) tmem_ld16_nowait(t_q + s * 64 + i * 16, r[i]);
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 64; ++i) v[i] = __uint_as_float(r[i >> 4][i & 15]);
                if (s < 2) {                                       // slots 0 / 1: part of the sum sits in alias block 6 / 7
#pragma unroll
                    for (int i = 0; i < 4; ++i) tmem_ld16_nowait(t_q + (6 + s) * 64 + i * 16, r[i]);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 64; ++i) v[i] += __uint_as_float(r[i >> 4][i & 15]);
                }
            }
            ring_fill_block(t_q + s * 64, bias_s);                 // the next tenant (row p + 6) starts from the bias
            if (s < 2) ring_fill_block(t_q + (6 + s) * 64, nullptr);
            if (valid && !(P.debug & 8)) {
#pragma unroll
                for (int i = 0; i < 64; ++i) v[i] = fmaxf(v[i], v[i] * act_k);
                const uint32_t row = stg + (uint32_t)lane * 128u;
                if (P.has_res) {
                    mbar_wait(rbar, rphase, P.dbg, 18, dead);
                    rphase ^= 1;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const uint4 rv = ld_shared_v4(row + (((uint32_t)j ^ ((uint32_t)lane & 7u)) << 4));
                        const uint32_t u[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            const float2 f = unpack_bf16(u[k]);
                            v[8 * j + 2 * k] += f.x;
                            v[8 * j + 2 * k + 1] += f.y;
                        }
                    }
                }
                // staging row `lane`: 128 B per pixel, 16-byte chunk j stored at j ^ (row & 7) (SW128)
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    st_shared_v4(row + (((uint32_t)j ^ ((uint32_t)lane & 7u)) << 4), pack_bf16(v[8 * j], v[8 * j + 1]),
                                 pack_bf16(v[8 * j + 2], v[8 * j + 3]), pack_bf16(v[8 * j + 4], v[8 * j + 5]),
                                 pack_bf16(v[8 * j + 6], v[8 * j + 7]));
                fence_proxy_async();
            }
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                mbar_arrive_cluster(tempty_lead + 8 * s);
                if (valid && !(P.debug & 10)) {
                    tma_store_5d(&P.out_map, stg, 0, x0, y, li, g);
                    bulk_commit();
                }
            }
            if (estat) atomicAdd(&g_ring_stat[4], (unsigned long long)(ring_clock() - e1));
        }
        if (lane == 0) bulk_wait_all();                            // staged rows must be read out before shared memory goes away
        tc_fence_before();
        cluster_sync_all();
        return;
    }
    tc_fence_before();
    cluster_sync_all();                                            // neither CTA may leave while its peer still signals it
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc_pair(tmem_base, 512);
    }
}

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
static bool g_ring_ready[kMaxDevices] = {false};

// Does this launch take the ring kernel?  (geometry: make_plan's p.ring; arguments: plain bf16 NHWC in / out)
bool ring_eligible(const vsrb_conv_args* a, const ConvPlan& p) {
    if (!p.ring || getenv("VSRB_TC_NO_RING")) return false;
    if (a->epilogue != VSRB_EPI_NHWC || a->split || a->n_in != 0 || a->max_ctas != 0) return false;
    if ((p.ring & 2) && (!a->patch || p.groups > 2 || (reinterpret_cast<uintptr_t>(a->patch) & 15) != 0 || a->patch_img_stride % 8 != 0 ||
                         a->patch_img_stride < 0 || a->patch_group_stride % 8 != 0))
        return false;
    if (p.ring & 1) {
        const int ms = p.ring_main_seg;
        if (a->in_c[ms] % 8 != 0 || (reinterpret_cast<uintptr_t>(a->in[ms]) & 15) != 0) return false;
    }
    if (a->out_c % 8 != 0 || (reinterpret_cast<uintptr_t>(a->out) & 15) != 0) return false;
    if (a->out_img_stride % 8 != 0 || a->out_group_stride % 8 != 0 || a->out_img_stride < 0 || a->out_group_stride < 0) return false;
    if (a->residual && (a->res_c % 8 != 0 || (reinterpret_cast<uintptr_t>(a->residual) & 15) != 0)) return false;
    // small launches do not amortise the two halo rows per range
    int min_rows = 6;
    if (const char* e = getenv("VSRB_RING_MIN_ROWS")) min_rows = atoi(e);
    const long long rows_g = (long long)a->imgs_per_group * ceil_div(a->w, kRingUW) * a->h;
    if (rows_g * 4 * 148 >= (1LL << 31)) return false;      // the kernel's range arithmetic is 32-bit
    return rows_g >= (long long)min_rows * 4 * 148 / p.groups;
}

// steps of the slowest CTA pair for a given split (what the kernel's pairs compute for themselves)
static int ring_steps(uint32_t rows_g, int H, int cols, int rpc, int n_ranges) {
    int worst = 0;
    for (int r = 0; r < n_ranges; ++r) {
        uint32_t lo, hi;
        ring_range(rows_g, H, cols, rpc, n_ranges, r, lo, hi);
        const int it = ring_items(lo, hi, H);
        worst = it > worst ? it : worst;
    }
    return worst;
}

int launch_conv_ring(const vsrb_conv_args* a, const ConvPlan& p, cudaStream_t stream) {
    int dev = 0, sms = 0;
    int rc = device_setup(&dev, &sms, g_ring_ready, [](int) {
        VSRB_CUDA(cudaFuncSetAttribute(conv_ring_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kRingSmem));
        return VSRB_OK;
    });
    if (rc != VSRB_OK) return rc;
    RingParams P;
    memset(&P, 0, sizeof(P));
    EpiParams e;
    fill_epi(a, p, &e);
    P.w = reinterpret_cast<const uint8_t*>(a->packed) + p.ring_off;
    P.bias = reinterpret_cast<const float*>(a->packed);
    P.has_res = a->residual != nullptr;
    P.has_main = (p.ring & 1) ? 1 : 0;
    P.has_patch = (p.ring & 2) ? 1 : 0;
    P.num_slots = P.has_patch ? kRingSlotsPatch : kRingSlots;
    P.slot_bytes = kRingSlotBytes + (P.has_patch ? kRingPatchBytes : 0);
    P.H = a->h; P.strips = ceil_div(a->w, kRingUW); P.ipg = a->imgs_per_group;
    P.cols = P.ipg * P.strips;
    P.rows_g = (uint32_t)P.cols * (uint32_t)P.H;
    P.act_k = e.act_k;
    P.dbg = debug_flag();
    P.debug = env_int("VSRB_RING_DEBUG");
    if (P.has_main) {
        const int ms = p.ring_main_seg;
        rc = encode_nhwc(&P.in_map, "ring input", a->in[ms], a->in_c[ms], a->w, a->h, a->batch, 64, 32, 1);
        if (rc != VSRB_OK) return rc;
    }
    for (int gi = 0; gi < (P.has_patch ? p.groups : 0); ++gi) {
        // both strides 0 = dense [groups][imgs_per_group]; with an explicit image stride the group stride is taken literally
        // (0 is then a real value: both propagation directions read the same frame at the middle time step)
        const long long istr = a->patch_img_stride ? a->patch_img_stride : (long long)a->h * a->w * 32;
        const long long gstr = (a->patch_img_stride || a->patch_group_stride) ? a->patch_group_stride : istr * a->imgs_per_group;
        const char* base = reinterpret_cast<const char*>(a->patch) + (long long)gi * gstr * 2;
        cuuint64_t dims[4] = {32, (cuuint64_t)a->w, (cuuint64_t)a->h, (cuuint64_t)a->imgs_per_group};
        cuuint64_t strides[3] = {64, (cuuint64_t)a->w * 64, (cuuint64_t)istr * 2};
        cuuint32_t box[4] = {32, 32, 1, 1};
        rc = encode_map(&P.patch_map[gi], "ring patches", base, 4, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_64B);
        if (rc != VSRB_OK) return rc;
    }
    if (P.has_res) {
        rc = encode_nhwc(&P.res_map, "ring residual", a->residual, a->res_c, a->w, a->h, a->batch, 64, 32, 1);
        if (rc != VSRB_OK) return rc;
    }
    {
        cuuint64_t dims[5] = {(cuuint64_t)a->out_c, (cuuint64_t)a->w, (cuuint64_t)a->h, (cuuint64_t)a->imgs_per_group, (cuuint64_t)p.groups};
        cuuint64_t strides[4] = {(cuuint64_t)a->out_c * 2, (cuuint64_t)a->w * a->out_c * 2, (cuuint64_t)e.out_img_stride * 2,
                                 (cuuint64_t)e.out_group_stride * 2};
        cuuint32_t box[5] = {64, (cuuint32_t)kRingUW, 1, 1, 1};
        rc = encode_map(&P.out_map, "ring output", a->out, 5, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
        if (rc != VSRB_OK) return rc;
    }
    int ctas_x = (sms / p.groups) & ~1;
    if (ctas_x < 2) ctas_x = 2;
    {   // never more ranges than rows: empty walks are legal but pointless
        long long want = ((long long)P.rows_g + 3) / 4;
        want = (want + 1) & ~1LL;
        if (want < 2) want = 2;
        if ((long long)ctas_x > want) ctas_x = (int)want;
    }
    {   // linear split of all rows, or the same number of ranges for every column strip: whichever needs fewer steps
        const int n_ranges = 4 * ctas_x;
        P.rpc = 0;
        const int rpc = n_ranges / P.cols;
        if (rpc >= 1 && P.rows_g <= (1u << 20) &&
            ring_steps(P.rows_g, P.H, P.cols, rpc, n_ranges) < ring_steps(P.rows_g, P.H, P.cols, 0, n_ranges))
            P.rpc = rpc;
    }
    const int smem = kRingCtrl + 1024 + VSRB_RING_W_BYTES + P.num_slots * P.slot_bytes + kRingStageBytes;
    return launch_ex(conv_ring_kernel, P, dim3(ctas_x, p.groups), dim3(kRingThreads), smem, stream, a->flags & VSRB_CONV_PDL, 2);
}

}  // namespace vsrb

extern "C" int vsrb_ring_debug_stats(uint64_t* out, int32_t reset) {
    using namespace vsrb;
    VSRB_CHECK_ARG(out, "ring_debug_stats: null output");
    VSRB_CUDA(cudaDeviceSynchronize());
    VSRB_CUDA(cudaMemcpyFromSymbol(out, g_ring_stat, sizeof(unsigned long long) * 8));
    if (reset) {
        unsigned long long z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        VSRB_CUDA(cudaMemcpyToSymbol(g_ring_stat, z, sizeof(z)));
    }
    return VSRB_OK;
}
