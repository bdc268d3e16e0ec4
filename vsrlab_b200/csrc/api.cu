// C-ABI plumbing: errors, device info, conv geometry, weight packing, conv dispatch; the per-device set-up and tensor
// maps of the tcgen05 launchers.
#include <stdarg.h>
#include <stdlib.h>

#include <atomic>
#include <mutex>

#include "common.cuh"

namespace vsrb {

static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};
__device__ int g_debug_flag = 0;

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

int* debug_flag() {
    int* p = nullptr;
    cudaGetSymbolAddress(reinterpret_cast<void**>(&p), g_debug_flag);
    return p;
}

int env_int(const char* name) {
    const char* e = getenv(name);
    return e ? atoi(e) : 0;
}

static std::mutex g_init_mutex;            // one-time per-process / per-device initialisation (callers may be threads)
static int g_sm_count[kMaxDevices] = {0};

int device_setup(int* dev, int* sms, bool (&done)[kMaxDevices], const std::function<int(int dev)>& setup) {
    VSRB_CUDA(cudaGetDevice(dev));
    VSRB_CHECK_ARG(*dev >= 0 && *dev < kMaxDevices, "device ordinal %d out of range", *dev);
    std::lock_guard<std::mutex> lock(g_init_mutex);
    if (!g_sm_count[*dev]) VSRB_CUDA(cudaDeviceGetAttribute(&g_sm_count[*dev], cudaDevAttrMultiProcessorCount, *dev));
    if (!done[*dev]) {
        const int rc = setup(*dev);
        if (rc != VSRB_OK) return rc;
        done[*dev] = true;
    }
    *sms = g_sm_count[*dev];
    return VSRB_OK;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int encode_map(CUtensorMap* map, const char* what, const void* base, int rank, const cuuint64_t* dims,
               const cuuint64_t* strides, const cuuint32_t* box, CUtensorMapSwizzle swz) {
    static const EncodeTiledFn encode = [] {      // looked up once per process; a failed lookup stays failed
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        const bool ok = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
                        q == cudaDriverEntryPointSuccess;
        return ok ? reinterpret_cast<EncodeTiledFn>(p) : nullptr;
    }();
    if (!encode) {
        set_error("cuTensorMapEncodeTiled not available from the driver");
        return VSRB_E_NODEVICE;
    }
    const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    const CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, const_cast<void*>(base), dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r == CUDA_SUCCESS) return VSRB_OK;
    char msg[400];
    int n = snprintf(msg, sizeof(msg), "cuTensorMapEncodeTiled (%.40s) failed with %d: dims", what, (int)r);
    for (int i = 0; i < rank; ++i) n += snprintf(msg + n, sizeof(msg) - n, " %llu", (unsigned long long)dims[i]);
    n += snprintf(msg + n, sizeof(msg) - n, ", byte strides");
    for (int i = 0; i + 1 < rank; ++i) n += snprintf(msg + n, sizeof(msg) - n, " %llu", (unsigned long long)strides[i]);
    n += snprintf(msg + n, sizeof(msg) - n, ", box");
    for (int i = 0; i < rank; ++i) n += snprintf(msg + n, sizeof(msg) - n, " %u", (unsigned)box[i]);
    set_error("%s", msg);
    return VSRB_E_CUDA;
}

int encode_nhwc(CUtensorMap* map, const char* what, const void* base, int c, int w, int h, int n, int box_c, int box_w,
                int box_h) {
    const cuuint64_t dims[4] = {(cuuint64_t)c, (cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)n};
    const cuuint64_t strides[3] = {(cuuint64_t)c * 2, (cuuint64_t)w * c * 2, (cuuint64_t)h * w * c * 2};
    const cuuint32_t box[4] = {(cuuint32_t)box_c, (cuuint32_t)box_w, (cuuint32_t)box_h, 1};
    return encode_map(map, what, base, 4, dims, strides, box, swizzle_for(box_c));
}

// ---------------------------------------------------------------------------------------
int make_plan(const vsrb_conv_geom* g, ConvPlan* p) {
    VSRB_CHECK_ARG(g && p, "null geometry");
    VSRB_CHECK_ARG(g->kh >= 1 && g->kh <= 7 && (g->kh & 1) && g->kw >= 1 && g->kw <= 7 && (g->kw & 1),
                   "kernel %dx%d unsupported (odd sizes 1..7)", g->kh, g->kw);
    VSRB_CHECK_ARG(g->n_seg >= 1 && g->n_seg <= 4, "n_seg must be 1..4, got %d", g->n_seg);
    VSRB_CHECK_ARG(g->cout >= 1 && g->cout <= 1024, "cout %d unsupported", g->cout);
    VSRB_CHECK_ARG(g->groups >= 1, "groups must be >= 1");
    VSRB_CHECK_ARG(g->dtype == VSRB_BF16 || g->dtype == VSRB_F32, "bad dtype %d", g->dtype);
    VSRB_CHECK_ARG(g->pixshuf == 0 || (g->pixshuf == 2 && g->cout % 64 == 0),
                   "pixshuf needs factor 2 and cout %% 64 == 0");
    VSRB_CHECK_ARG(g->transpose == 0 || (g->transpose == 1 && !g->pixshuf), "transpose packing excludes pixshuf");
    memset(p, 0, sizeof(*p));
    p->kh = g->kh; p->kw = g->kw; p->n_seg = g->n_seg; p->groups = g->groups;
    p->pixshuf = g->pixshuf; p->dtype = g->dtype;
    p->cout = g->cout;
    p->cout_pad = (int)round_up(g->cout, 16);
    if (p->cout_pad <= 128) { p->n_tile = p->cout_pad; p->n_blocks = 1; }
    else if (p->cout_pad % 128 == 0) { p->n_tile = 128; p->n_blocks = p->cout_pad / 128; }
    else if (p->cout_pad % 64 == 0) { p->n_tile = 64; p->n_blocks = p->cout_pad / 64; }
    else { p->n_tile = 16; p->n_blocks = p->cout_pad / 16; }
    // "stacked" tensor-core layout: the kw filter columns sit side by side along the MMA N dimension
    // (N = kw * n_tile <= 256), so one un-shifted activation tile feeds all of them and the x-shift
    // is undone in the epilogue.  Cuts the A-operand shared-memory traffic per FLOP by kw.
    p->stacked = 0;
    p->ns = p->n_tile;
    int ck_cap = 64;                                   // largest K chunk (channels) a stage may carry
    if (p->dtype == VSRB_BF16 && !p->pixshuf && (p->kw == 3 || p->kw == 7) && !getenv("VSRB_TC_NO_STACK")) {
        // Pick classic vs stacked (and the stacked tile) with the operand-fetch model measured on B200
        // (DESIGN.md "tensor-core cost model"): one K=16 MMA costs (128 + N) shared-memory row fetches, two
        // per cycle for 64/128-byte rows and one per cycle for 32-byte rows; the stacked epilogue costs
        // n_tile*(4*(kw-1)+24) cycles per 128 pixels; a stacked tile only yields (33-kw)/32 useful columns.
        auto rows_cost = [](int ck) { return ck >= 32 ? 0.5 : 1.0; };
        auto mma_cost = [&](int n_tile, int n, int cap, int stages_kx, bool pair = false) {
            double c = 0;
            for (int s = 0; s < g->n_seg; ++s) {
                const int cpad = (int)round_up(g->seg_c[s], 16);
                int ck = (cpad % 64 == 0) ? 64 : (cpad % 32 == 0 ? 32 : 16);
                if (ck > cap) ck = cap;
                c += (double)(cpad / 16) * p->kh * stages_kx * (128 + (pair ? n / 2 : n)) * rows_cost(ck);
            }
            return c * (p->cout_pad / n_tile);
        };
        // CTA pairs (conv_tc.cu, cta_group::2): every CTA holds half of the weight rows, resident.  A stacked plan whose
        // stages are too large to stream (7x7 with 32/64-channel chunks) is still fine when half of the whole weight block
        // plus two activation slots fit next to the staging buffers; launch_conv_tc then always runs it in pairs.
        auto pair_fits = [&](int n_tile, int cap) {
            if (p->kh != p->kw || (p->kw * n_tile / 2) % 8 != 0 || (p->kw * n_tile) % 16 != 0) return false;
            size_t total = 0, amax = 0;
            for (int s = 0; s < g->n_seg; ++s) {
                const size_t cpad = round_up(g->seg_c[s], 16);
                size_t ck = (cpad % 64 == 0) ? 64 : (cpad % 32 == 0 ? 32 : 16);
                if (ck > (size_t)cap) ck = cap;
                total += (size_t)p->kh * p->kw * n_tile * cpad * 2;
                const size_t ab = (size_t)(4 + p->kh - 1) * 32 * ck * 2;
                amax = amax > ab ? amax : ab;
            }
            return round_up(total / 2, 1024) + 3 * round_up(amax, 1024) <= (size_t)160 * 1024;
        };
        double best = mma_cost(p->n_tile, p->n_tile, 64, p->kw);
        const double classic_epi = 10.0 * p->cout_pad;
        if (best < classic_epi) best = classic_epi;
        const int cands[3] = {64, 32, 16};
        for (int i = 0; i < 3; ++i) {
            if (p->cout_pad % cands[i] != 0 || p->kw * cands[i] > 256) continue;
            for (int j = 0; j < 3; ++j) {
                const bool pf = pair_fits(cands[i], cands[j]);
                if (p->kh * p->kw * cands[i] * cands[j] * 2 > 76 * 1024 && !pf) continue;
                double c = mma_cost(cands[i], p->kw * cands[i], cands[j], 1, pf);
                const double epi = (double)p->cout_pad * (4 * (p->kw - 1) + 24);
                if (c < epi) c = epi;
                c *= 32.0 / (33 - p->kw);
                if (c < best) {
                    best = c;
                    p->stacked = 1;
                    p->n_tile = cands[i];
                    p->n_blocks = p->cout_pad / cands[i];
                    p->ns = p->kw * cands[i];
                    ck_cap = cands[j];
                }
                break;   // smaller chunks of the same tile are never cheaper
            }
        }
    }
    const int kx_stages = p->stacked ? 1 : p->kw;      // pipeline stages per channel chunk
    const int kx_rows = p->stacked ? p->kw : 1;        // filter columns inside one stage's B tile
    p->stages_per_tile = 0;
    p->wblock_bytes = 0;
    for (int s = 0; s < g->n_seg; ++s) {
        SegPlan& sp = p->seg[s];
        VSRB_CHECK_ARG(g->seg_c[s] >= 1 && g->seg_off[s] >= 0, "bad segment %d", s);
        sp.c = g->seg_c[s];
        sp.off = g->seg_off[s];
        sp.cpad = (int)round_up(sp.c, 16);
        sp.ck = (sp.cpad % 64 == 0) ? 64 : (sp.cpad % 32 == 0 ? 32 : 16);
        if (sp.ck > ck_cap) sp.ck = ck_cap;
        sp.chunks = sp.cpad / sp.ck;
        sp.rowbytes = sp.ck * 2;
        sp.swz_mask = sp.ck == 64 ? 7 : (sp.ck == 32 ? 3 : 1);
        sp.layout = sp.ck == 64 ? 2 : (sp.ck == 32 ? 4 : 6);
        p->cin_packed += sp.c;
        p->b_stage_bytes[s] = p->kh * kx_rows * p->n_tile * sp.rowbytes;
        p->stages_per_tile += sp.chunks * kx_stages;
        p->wblock_bytes += (size_t)sp.chunks * kx_stages * p->b_stage_bytes[s];
    }
    p->bias_bytes = round_up((size_t)p->groups * p->cout_pad * sizeof(float), 1024);
    p->ring = 0;
    p->ring_main_seg = p->ring_patch_seg = -1;
    if (p->dtype == VSRB_BF16 && p->kh == 3 && p->kw == 3 && p->cout == 64 && !p->pixshuf && p->n_seg <= 2 && !(g->transpose && p->n_seg > 1)) {
        bool ok = true;
        for (int s = 0; s < p->n_seg; ++s) {
            if (g->seg_c[s] == 64 && p->ring_main_seg < 0) p->ring_main_seg = s;
            else if (g->seg_c[s] == 3 && p->ring_patch_seg < 0 && !g->transpose) p->ring_patch_seg = s;
            else ok = false;
        }
        if (ok) p->ring = (p->ring_main_seg >= 0 ? 1 : 0) | (p->ring_patch_seg >= 0 ? 2 : 0);
    }
    if (p->dtype == VSRB_BF16) {
        p->total_bytes = p->bias_bytes + (size_t)p->groups * p->n_blocks * p->wblock_bytes;
        if (p->ring) {
            p->ring_off = round_up(p->total_bytes, 1024);
            p->total_bytes = p->ring_off + (size_t)p->groups * 2 * VSRB_RING_W_BYTES;
        }
    } else
        p->total_bytes = p->bias_bytes +
                         (size_t)p->groups * p->kh * p->kw * p->cin_packed * p->cout_pad * sizeof(float);
    return VSRB_OK;
}

// packed output channel n' -> original output channel (PixelShuffle(2) groups sub-pixels together)
__host__ __device__ static inline int orig_cout(int np, int cout, int pixshuf) {
    if (!pixshuf) return np;
    int cq = cout / 4;
    int q = np / cq, c = np - q * cq;
    return 4 * c + q;
}

// element of the OIHW source: forward layout w[g][o][c][ky][kx]; transposed (input-gradient conv): the
// packed conv maps the forward OUTPUT channels (its input, index c) to the forward INPUT channels (its
// output, index o) with the filter flipped: w_t[o][c][ky][kx] = w[c][o][kh-1-ky][kw-1-kx]
#define VSRB_W_SRC(pp, g, o, c, ky, kx)                                                                              \
    ((pp).transpose                                                                                                 \
         ? w[((((size_t)(g) * (pp).cin_total + (c)) * (pp).cout + (o)) * (pp).kh + ((pp).kh - 1 - (ky))) * (pp).kw + \
             ((pp).kw - 1 - (kx))]                                                                                  \
         : w[((((size_t)(g) * (pp).cout + (o)) * (pp).cin_total + (c)) * (pp).kh + (ky)) * (pp).kw + (kx)])

struct PackParams {
    int kh, kw, n_seg, groups, pixshuf;
    int seg_c[4], seg_off[4], seg_ck[4], seg_chunks[4], seg_rowbytes[4], seg_mask[4], seg_bstage[4];
    int cin_total, cin_packed, cout, cout_pad, n_tile, n_blocks, stacked, transpose, ring_main_seg, ring_patch_seg;
    size_t wblock_bytes, bias_bytes;
};

__global__ void pack_bias_kernel(PackParams pp, const float* __restrict__ bias, float* __restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    int total = pp.groups * pp.cout_pad;
    if (i >= total) return;
    int g = i / pp.cout_pad, np = i - g * pp.cout_pad;
    float v = 0.f;
    if (bias && np < pp.cout) v = bias[(size_t)g * pp.cout + orig_cout(np, pp.cout, pp.pixshuf)];
    out[i] = v;
}

// Tensor-core image: [group][n_block][stage (seg, chunk, kx)][ky][n][ck] bf16 (classic) or
// [group][n_block][stage (seg, chunk)][ky][kx][n][ck] (stacked), each stage region stored exactly as
// it must sit in shared memory (swizzled K-major rows).
__global__ void pack_tc_kernel(PackParams pp, const float* __restrict__ w, uint8_t* __restrict__ out) {
    size_t elems_per_block = pp.wblock_bytes / 2;
    size_t total = (size_t)pp.groups * pp.n_blocks * elems_per_block;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        size_t blk = i / elems_per_block;
        size_t r = i - blk * elems_per_block;
        int g = (int)(blk / pp.n_blocks), qb = (int)(blk % pp.n_blocks);
        // locate segment / stage
        int s = 0;
        const int kxs = pp.stacked ? 1 : pp.kw;        // stages per channel chunk
        size_t base_bytes = 0;
        for (; s < pp.n_seg - 1; ++s) {
            const size_t seg_elems = (size_t)pp.seg_chunks[s] * kxs * pp.seg_bstage[s] / 2;
            if (r < seg_elems) break;
            r -= seg_elems;
            base_bytes += seg_elems * 2;
        }
        size_t st_elems = (size_t)pp.seg_bstage[s] / 2;
        int local = (int)(r / st_elems);
        size_t e = r - (size_t)local * st_elems;
        int chunk = local / kxs, kx = local - chunk * kxs;
        int ck = pp.seg_ck[s];
        int row = (int)(e / ck), kk = (int)(e - (size_t)row * ck);
        int ky, n;
        if (pp.stacked) {
            ky = row / (pp.kw * pp.n_tile);
            const int rem = row - ky * pp.kw * pp.n_tile;
            kx = rem / pp.n_tile;
            n = rem - kx * pp.n_tile;
        } else {
            ky = row / pp.n_tile;
            n = row - ky * pp.n_tile;
        }
        int np = qb * pp.n_tile + n;
        int ci = chunk * ck + kk;
        float v = 0.f;
        if (np < pp.cout && ci < pp.seg_c[s]) {
            int o = orig_cout(np, pp.cout, pp.pixshuf);
            v = VSRB_W_SRC(pp, g, o, pp.seg_off[s] + ci, ky, kx);
        }
        uint32_t off = (uint32_t)row * pp.seg_rowbytes[s] + (uint32_t)kk * 2;
        off ^= ((off >> 7) & pp.seg_mask[s]) << 4;
        size_t dst = blk * pp.wblock_bytes + base_bytes + (size_t)local * pp.seg_bstage[s] + off;
        *reinterpret_cast<__nv_bfloat16*>(out + dst) = __float2bfloat16_rn(v);
    }
}

// Ring image (conv_ring.cu): [group][cta rank][kx][96 rows][64 ch] bf16, rows swizzled like every K-major SW128 tile.
// The B operand of the ring walk's MMA is N = 192 = [W(ky=2) | W(ky=1) | W(ky=0)] x 64 output channels; the CTA pair
// splits it in halves of 96 rows: rank 0 holds [ky2 0-63 | ky1 0-31], rank 1 holds [ky1 32-63 | ky0 0-63].
__global__ void pack_ring_kernel(PackParams pp, const float* __restrict__ w, uint8_t* __restrict__ out) {
    const size_t per_rank = VSRB_RING_W_BYTES / 2;        // elements
    const size_t total = (size_t)pp.groups * 2 * per_rank;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int g = (int)(i / (2 * per_rank));
        size_t r = i - (size_t)g * 2 * per_rank;
        const int rank = (int)(r / per_rank);
        r -= (size_t)rank * per_rank;
        const size_t base = (size_t)(g * 2 + rank) * VSRB_RING_W_BYTES;
        if (r < VSRB_RING_W_MAIN / 2) {
            const int kx = (int)(r / (96 * 64));
            r -= (size_t)kx * 96 * 64;
            const int row = (int)(r / 64), k = (int)(r - (size_t)row * 64);
            const int nrow = rank * 96 + row;                  // row of the N = 192 operand
            const int ky = 2 - nrow / 64, n = nrow & 63;
            const float v = pp.ring_main_seg >= 0 ? VSRB_W_SRC(pp, g, n, pp.seg_off[pp.ring_main_seg] + k, ky, kx) : 0.f;
            uint32_t off = (uint32_t)row * 128u + (uint32_t)k * 2u;
            off ^= ((off >> 7) & 7u) << 4;
            *reinterpret_cast<__nv_bfloat16*>(out + base + (size_t)kx * (96 * 128) + off) = __float2bfloat16_rn(v);
        } else {
            // patch tile: row = output channel (this rank's 32), k = (ky*3 + kx)*3 + c of the 3x3x3 neighbourhood (27 used of 32);
            // 64-byte rows, SW64: 16-byte chunk index ^= (row >> 1) & 3
            r -= VSRB_RING_W_MAIN / 2;
            const int row = (int)(r / 32), k = (int)(r - (size_t)row * 32);
            float v = 0.f;
            if (pp.ring_patch_seg >= 0 && k < 27) {
                const int tap = k / 3, c = k - tap * 3;
                v = VSRB_W_SRC(pp, g, rank * 32 + row, pp.seg_off[pp.ring_patch_seg] + c, tap / 3, tap % 3);
            }
            uint32_t off = (uint32_t)row * 64u + (uint32_t)k * 2u;
            off ^= ((off >> 7) & 3u) << 4;
            *reinterpret_cast<__nv_bfloat16*>(out + base + VSRB_RING_W_MAIN + off) = __float2bfloat16_rn(v);
        }
    }
}

// fp32 image: [group][tap][cin_packed][cout_pad]
__global__ void pack_f32_kernel(PackParams pp, const float* __restrict__ w, float* __restrict__ out) {
    size_t per_g = (size_t)pp.kh * pp.kw * pp.cin_packed * pp.cout_pad;
    size_t total = per_g * pp.groups;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        int g = (int)(i / per_g);
        size_t r = i - (size_t)g * per_g;
        int np = (int)(r % pp.cout_pad);
        r /= pp.cout_pad;
        int cp = (int)(r % pp.cin_packed);
        int tap = (int)(r / pp.cin_packed);
        int ky = tap / pp.kw, kx = tap - ky * pp.kw;
        int s = 0, ci = cp;
        while (s < pp.n_seg - 1 && ci >= pp.seg_c[s]) { ci -= pp.seg_c[s]; ++s; }
        float v = 0.f;
        if (np < pp.cout) {
            int o = orig_cout(np, pp.cout, pp.pixshuf);
            v = VSRB_W_SRC(pp, g, o, pp.seg_off[s] + ci, ky, kx);
        }
        out[i] = v;
    }
}

int launch_pack(const vsrb_conv_geom* g, const ConvPlan& p, const float* w, int cin_total, const float* bias,
                void* packed, cudaStream_t s) {
    PackParams pp;
    memset(&pp, 0, sizeof(pp));
    pp.kh = p.kh; pp.kw = p.kw; pp.n_seg = p.n_seg; pp.groups = p.groups; pp.pixshuf = p.pixshuf;
    for (int i = 0; i < p.n_seg; ++i) {
        pp.seg_c[i] = p.seg[i].c; pp.seg_off[i] = p.seg[i].off; pp.seg_ck[i] = p.seg[i].ck;
        pp.seg_chunks[i] = p.seg[i].chunks; pp.seg_rowbytes[i] = p.seg[i].rowbytes;
        pp.seg_mask[i] = p.seg[i].swz_mask; pp.seg_bstage[i] = p.b_stage_bytes[i];
        VSRB_CHECK_ARG(p.seg[i].off + p.seg[i].c <= cin_total, "segment %d exceeds cin_total %d", i, cin_total);
    }
    pp.cin_total = cin_total; pp.cin_packed = p.cin_packed; pp.cout = p.cout; pp.cout_pad = p.cout_pad;
    pp.ring_main_seg = p.ring_main_seg; pp.ring_patch_seg = p.ring_patch_seg;
    pp.n_tile = p.n_tile; pp.n_blocks = p.n_blocks; pp.stacked = p.stacked; pp.transpose = g->transpose; pp.wblock_bytes = p.wblock_bytes; pp.bias_bytes = p.bias_bytes;
    int nb = p.groups * p.cout_pad;
    pack_bias_kernel<<<ceil_div(nb, 256), 256, 0, s>>>(pp, bias, reinterpret_cast<float*>(packed));
    VSRB_LAUNCH_CHECK();
    uint8_t* wp = reinterpret_cast<uint8_t*>(packed) + p.bias_bytes;
    if (p.dtype == VSRB_BF16) {
        size_t total = (size_t)p.groups * p.n_blocks * p.wblock_bytes / 2;
        int blocks = (int)((total + 255) / 256);
        if (blocks > 4096) blocks = 4096;
        pack_tc_kernel<<<blocks, 256, 0, s>>>(pp, w, wp);
        if (p.ring) {
            VSRB_LAUNCH_CHECK();
            pack_ring_kernel<<<256, 256, 0, s>>>(pp, w, reinterpret_cast<uint8_t*>(packed) + p.ring_off);
        }
    } else {
        size_t total = (size_t)p.groups * p.kh * p.kw * p.cin_packed * p.cout_pad;
        int blocks = (int)((total + 255) / 256);
        if (blocks > 4096) blocks = 4096;
        pack_f32_kernel<<<blocks, 256, 0, s>>>(pp, w, reinterpret_cast<float*>(wp));
    }
    VSRB_LAUNCH_CHECK();
    return VSRB_OK;
}

void fill_epi(const vsrb_conv_args* a, const ConvPlan& p, EpiParams* e) {
    e->mode = a->epilogue; e->act = a->act; e->slope = a->slope;
    e->act_k = a->act == VSRB_ACT_NONE ? 1.f : (a->act == VSRB_ACT_RELU ? 0.f : a->slope);
    e->H = a->h; e->W = a->w;
    e->cout_pad = p.cout_pad; e->cq = p.pixshuf ? p.cout / 4 : 0; e->pixshuf = p.pixshuf;
    e->out = a->out; e->out_c = a->out_c; e->res = a->residual; e->res_c = a->res_c;
    {
        long long oh = p.pixshuf ? 2LL * a->h : a->h, ow = p.pixshuf ? 2LL * a->w : a->w;
        e->out_img_stride = a->out_img_stride ? a->out_img_stride : oh * ow * a->out_c;
        e->out_group_stride = a->out_group_stride ? a->out_group_stride : e->out_img_stride * a->imgs_per_group;
        e->imgs_per_group = a->imgs_per_group;
        e->split = a->split;
    }
    e->f32_io = a->f32_io; e->f32_in = a->f32_in; e->aux_h = a->aux_h; e->aux_w = a->aux_w;
    e->sr_kind = (a->flags & VSRB_CONV_SR_U8) ? 2 : ((a->flags & VSRB_CONV_SR_F16) ? 1 : 0);
    e->bias = reinterpret_cast<const float*>(a->packed);
}

}  // namespace vsrb

using namespace vsrb;

extern "C" {

int vsrb_version(void) { return VSRB_VERSION; }
const char* vsrb_last_error(void) { return g_err; }
int64_t vsrb_launch_count(void) { return g_launches.load(); }

int vsrb_device_info(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor) {
    int dev = 0;
    VSRB_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    VSRB_CUDA(cudaGetDeviceProperties(&prop, dev));
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    return VSRB_OK;
}

int vsrb_debug_status(void* stream) {
    int v = 0;
    int* p = debug_flag();
    VSRB_CUDA(cudaMemcpyAsync(&v, p, sizeof(int), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    VSRB_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    if (v) {
        int z = 0;
        VSRB_CUDA(cudaMemcpyAsync(p, &z, sizeof(int), cudaMemcpyHostToDevice, (cudaStream_t)stream));
        VSRB_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    }
    return v;
}

size_t vsrb_packed_weight_bytes(const vsrb_conv_geom* g) {
    ConvPlan p;
    if (make_plan(g, &p) != VSRB_OK) return 0;
    return p.total_bytes;
}

int vsrb_pack_conv_weight(const vsrb_conv_geom* g, const float* w, int32_t cin_total, const float* bias,
                          void* packed, void* stream) {
    ConvPlan p;
    int rc = make_plan(g, &p);
    if (rc != VSRB_OK) return rc;
    VSRB_CHECK_ARG(w && packed, "null weight / packed pointer");
    return launch_pack(g, p, w, cin_total, bias, packed, (cudaStream_t)stream);
}

int vsrb_conv_plan_info(const vsrb_conv_geom* g, int32_t info[8]) {
    ConvPlan p;
    int rc = make_plan(g, &p);
    if (rc != VSRB_OK) return rc;
    VSRB_CHECK_ARG(info, "null info");
    info[0] = p.stacked; info[1] = p.n_tile; info[2] = p.n_blocks; info[3] = p.ns;
    info[4] = p.seg[0].ck; info[5] = p.n_seg > 1 ? p.seg[1].ck : 0;
    info[6] = p.stages_per_tile; info[7] = (int32_t)(p.wblock_bytes / 1024);
    return VSRB_OK;
}

int vsrb_conv2d_fwd(const vsrb_conv_args* a, void* stream) {
    VSRB_CHECK_ARG(a, "null args");
    ConvPlan p;
    int rc = make_plan(&a->geom, &p);
    if (rc != VSRB_OK) return rc;
    VSRB_CHECK_ARG(a->batch >= 1 && a->h >= 1 && a->w >= 1, "bad extent %dx%dx%d", a->batch, a->h, a->w);
    VSRB_CHECK_ARG(a->imgs_per_group >= 1 && a->imgs_per_group * p.groups == a->batch,
                   "batch %d != groups %d * imgs_per_group %d", a->batch, p.groups, a->imgs_per_group);
    VSRB_CHECK_ARG(a->packed, "null packed weights");
    VSRB_CHECK_ARG(a->act != VSRB_ACT_LRELU || (a->slope >= 0.f && a->slope <= 1.f), "LeakyReLU slope must be in [0,1]");
    VSRB_CHECK_ARG(a->n_in >= 0 && a->n_in <= 6, "n_in must be 0..6");
    VSRB_CHECK_ARG(a->n_in == 0 || p.dtype == VSRB_BF16, "operand lists (n_in > 0) exist for the tensor-core path only");
    const int n_ops = a->n_in ? a->n_in : p.n_seg;
    for (int i = 0; i < n_ops; ++i) {
        const int s = a->n_in ? a->in_wseg[i] : i, c0 = a->n_in ? a->in_c0[i] : 0;
        VSRB_CHECK_ARG(s >= 0 && s < p.n_seg && c0 >= 0, "operand %d: bad weight segment / channel offset", i);
        VSRB_CHECK_ARG(a->in[i], "null input operand %d", i);
        int need = p.dtype == VSRB_BF16 ? p.seg[s].cpad : p.seg[s].c;
        VSRB_CHECK_ARG(a->in_c[i] >= c0 + need, "operand %d: %d channels allocated, need %d", i, a->in_c[i], c0 + need);
    }
    VSRB_CHECK_ARG(!a->split || (p.dtype == VSRB_BF16 && (a->epilogue == VSRB_EPI_NHWC || a->epilogue == VSRB_EPI_CLEAN)),
                   "split outputs exist for bf16 EPI_NHWC / EPI_CLEAN only");
    switch (a->epilogue) {
        case VSRB_EPI_NHWC:
            VSRB_CHECK_ARG(a->out && (a->split ? a->out_c / 2 : a->out_c) >= (p.pixshuf ? p.cout / 4 : p.cout_pad),
                           "EPI_NHWC: out_c %d too small", a->out_c);
            VSRB_CHECK_ARG(!a->residual || (!p.pixshuf && (a->split ? a->res_c / 2 : a->res_c) >= p.cout_pad), "bad residual");
            VSRB_CHECK_ARG(a->out_c % 8 == 0 && (!a->residual || a->res_c % 8 == 0), "channel strides must be %% 8");
            // split stores and loads move 16 channels (two 16-byte vectors) at channel c0 and at c0 + out_c/2
            VSRB_CHECK_ARG(!a->split || (a->out_c % 16 == 0 && (!a->residual || a->res_c % 16 == 0)),
                           "EPI_NHWC split: out_c %d and res_c %d must be multiples of 16 (the lo half starts at C/2)", a->out_c,
                           a->res_c);
            break;
        case VSRB_EPI_CLEAN:
            VSRB_CHECK_ARG(p.cout == 3 && a->f32_io && a->out && !p.pixshuf, "EPI_CLEAN needs cout==3, f32_io, out");
            // the split store writes the frame as [hi 16 | lo 16]: exactly 32 channels per pixel
            if (a->split) VSRB_CHECK_ARG(a->out_c == 32, "EPI_CLEAN split: out_c must be 32 ([hi 16 | lo 16]), got %d", a->out_c);
            else VSRB_CHECK_ARG(a->out_c >= 3 && a->out_c <= 16, "EPI_CLEAN needs out with 3..16 channels, got %d", a->out_c);
            // 16-channel and split stores are 16-byte vectors
            VSRB_CHECK_ARG((a->out_c != 16 && !a->split) || (reinterpret_cast<uintptr_t>(a->out) & 15) == 0,
                           "EPI_CLEAN: out must be 16-byte aligned for a %d-channel store", a->out_c);
            break;
        case VSRB_EPI_FLOW:
            VSRB_CHECK_ARG(p.cout == 2 && a->f32_io && a->f32_in && !p.pixshuf, "EPI_FLOW needs cout==2, f32_io, f32_in");
            break;
        case VSRB_EPI_SR:
            VSRB_CHECK_ARG(p.cout == 3 && a->f32_io && a->f32_in && a->aux_h >= 1 && a->aux_w >= 1 && !p.pixshuf,
                           "EPI_SR needs cout==3, f32_io, f32_in, aux_h/w");
            break;
        default:
            VSRB_CHECK_ARG(false, "unknown epilogue %d", a->epilogue);
    }
    if (p.dtype == VSRB_BF16 && ring_eligible(a, p)) return launch_conv_ring(a, p, (cudaStream_t)stream);
    if (p.dtype == VSRB_BF16) return launch_conv_tc(a, p, (cudaStream_t)stream);
    return launch_conv_f32(a, p, (cudaStream_t)stream);
}

}  // extern "C"
