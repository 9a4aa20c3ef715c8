// conv_tc.cu -- the tensor-core layers of UNetDC as one persistent, warp-specialised
// implicit-GEMM kernel for sm_100a (tcgen05.mma, accumulators in TMEM, operands fed by TMA).
//
// Replaces, layer by layer (reference models/model_2.py):
//   nn.Conv2d(k=3, padding=d, dilation=d) + BatchNorm2d(eval) + ReLU        :40-54
//   F.max_pool2d(x, 2)                       (fused: DC_EPI_STORE_POOL)      :59-61,64
//   nn.ConvTranspose2d(k=2, stride=2)        (DC_KIND_UPCONV2/UPSCATTER)     :20,23,26,29
//   torch.cat([up, enc], 1)                  (never copied: both producers write straight into
//                                             channel slices of one NHWC buffer)  :68,71,74,77
//   out_conv 1x1 + sigmoid, and the `> prob_thresh` of quantify_droplets_batch.py:56
//                                            (fused: DC_EPI_HEAD)            :32,79-80
//
// GEMM view.  M = 128 output pixels (an 8 x 16 patch of one image), N = BN output channels,
// K = taps x Cin walked in chunks of 64 channels (64 bf16 = 128 B = one swizzle row).
//   A chunk = TMA box (64 ch, 16 w, 8 h, 1 img) of the NHWC activation tensor at the signed offset
//             ((ky-1)*d, (kx-1)*d): TMA's out-of-bounds zero fill IS the conv padding.  Lands in
//             shared memory as 128 rows x 128 B, 128B-swizzled = the canonical K-major UMMA layout.
//   B chunk = TMA box (64 k, BN rows) of the packed weights [rows][K], same layout.
//   D       = 128 lanes x BN fp32 columns in TMEM, double buffered (2*BN columns) so the epilogue
//             of tile i overlaps the MMAs of tile i+1.
// Taps whose shifted patch is wholly outside the image (large dilation on small maps) are skipped.
//
// Kernels (they share the roles and the epilogue; DESIGN.md 3.1 has the measurements):
//   conv_tc_kernel     generic: one TMA box per (tap, 64-channel chunk), A re-fetched per tap from L2.
//                      Used for dilation 8 / 16 (enc4, bottleneck) and the transposed convs.
//   conv_halo_kernel   single CTA: ONE haloed activation region (16+2d) x (16+2d) pixels x 64 ch per tile and
//                      chunk; the nine taps are nine UMMA descriptors into that region (start = base +
//                      (ky*d*RW + kx*d) rows, stride between 8-pixel groups = RW rows).  Cout = 64 layers with
//                      long K at dilation <= 4, weights streamed (the pair kernel does not stream at N = 64).
//   conv_halo2_kernel  the same on a CTA pair (cta_group::2): M = 256 MMAs over two SMs, each SM holds half of the
//                      weight rows and its own pixel tile.  Runs every 3x3 layer with dilation <= 4.
//   stem_tc_kernel     first layer (Cin = 3): im2col tile built by producer warps, K = 9 -> 16 or 27 -> 32.
//   conv_tc_split_kernel  the generic kernel on fp32 values held as three bf16 planes (UNetDC.precision = "fp32"):
//                      six plane products per (tap, chunk), every layer of that forward.
//
// Warp roles (384 threads, 1 CTA / SM, persistent over tiles):
//   warp 0 : TMA producer           warp 1 : tcgen05.mma issuer       (warp-uniform loops, one elected lane issues)
//   warp 2 : TMEM alloc / dealloc   warps 4..11 : two epilogue groups (TMEM -> regs -> smem transpose -> global)
#include "common.cuh"

#include <cuda.h>
#include <stdlib.h>
#include <string.h>

namespace dc {

namespace {

constexpr int TILE_H = 8, TILE_W = 16, TILE_M = TILE_H * TILE_W;
constexpr int KCHUNK = 64;
constexpr int A_STAGE_BYTES = TILE_M * KCHUNK * 2;   // 16 KB
constexpr int NUM_THREADS = 384;      // 4 role warps + 2 epilogue groups x 4 warps
constexpr int EPI_WARP0 = 4;

// Kernel-family override for the tests (dc_debug_set_conv_family): the product path never changes it.
int g_kernel_family = DC_CONV_FAMILY_AUTO;

// cudaFuncAttributeMaxDynamicSharedMemorySize is per (function, device): set once per device, not per launch.
template <class K>
int set_max_smem_once(K kernel, int bytes, unsigned long long* done_mask) {
    int dev = 0;
    DC_CUDA(cudaGetDevice(&dev));
    const unsigned long long bit = 1ull << (dev & 63);
    if (!(__atomic_load_n(done_mask, __ATOMIC_ACQUIRE) & bit)) {
        DC_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
        __atomic_fetch_or(done_mask, bit, __ATOMIC_RELEASE);
    }
    return DC_OK;
}

// floor(n / d) for 0 <= n < 2^31 as one widening multiply and a shift (Granlund-Montgomery round-up magic number):
// s = ceil(log2 d), m = floor(2^(31+s) / d) + 1 < 2^32.
struct FastDiv {
    uint32_t mul, shift;
};
inline FastDiv make_fastdiv(int d) {
    FastDiv f;
    uint32_t s = 0;
    while ((1ll << s) < d) ++s;
    f.shift = 31 + s;
    f.mul = (uint32_t)(((1ull << f.shift) / (uint32_t)d) + 1ull);
    return f;
}
__device__ __forceinline__ int fast_div(int n, const FastDiv& f) {
    return (int)(((unsigned long long)(uint32_t)n * f.mul) >> f.shift);
}

struct alignas(64) ConvParams {
    CUtensorMap tmA;
    CUtensorMap tmB;
    CUtensorMap tmS;                // parity-class kernels only: the skip tensor as two column-parity planes
    CUtensorMap tmB2;               // conv_upfused_wide_kernel only: the skip half of the 3x3 weights
    int B, H, W, Cin, Cout;
    int dil, ntaps, kchunks;
    int tiles_w, tiles_h, n_tiles, total_tiles, m_tiles;      // m_tiles = pixel tiles = total_tiles / n_tiles
    FastDiv fd_ntiles, fd_per_img, fd_tiles_w;      // exact division of tile indices (< 2^31) without the ~20-instruction IDIV
    int epilogue, relu;
    const float* bias;
    int bias_const;                 // Cout == 64 and the host knows the values: bias_c[] below, read as c[0][..] operands
    float bias_c[64];
    __nv_bfloat16* out;
    int out_stride, out_offset;
    __nv_bfloat16* pool_out;
    int pool_stride;
    const float* head_w;
    float head_b, thresh;
    float* prob_out;
    uint8_t* mask_out;
    // conv_halo_kernel only
    int region_w, region_h, region_stride, nstages, nbstages;
    // parity-class kernels: 1 = p.bias is row 4 of a [9][Cout] border-class table (upconv folded in)
    int border_bias;
    int real_ntiles;                // conv_upfused_wide_kernel: n-tiles of Cout (p.n_tiles also counts the class groups)
    // conv_tc_split_kernel only: channel distance between the bf16 planes of the input, output and pooled output
    int in_plane_stride, out_plane_stride, pool_plane_stride;
};

struct TileCoord {
    int img, h0, w0, n0;
};

template <int TH = TILE_H, int TW = TILE_W>
__device__ __forceinline__ TileCoord decode_tile(const ConvParams& p, int tile, int BN) {
    TileCoord t;
    int m = fast_div(tile, p.fd_ntiles);
    int nt = tile - m * p.n_tiles;
    int per_img = p.tiles_h * p.tiles_w;
    t.img = fast_div(m, p.fd_per_img);
    int r = m - t.img * per_img;
    int th = fast_div(r, p.fd_tiles_w);
    t.h0 = th * TH;
    t.w0 = (r - th * p.tiles_w) * TW;
    t.n0 = nt * BN;
    return t;
}

// Offset of tap `tap`; false when the shifted 8x16 patch has no pixel inside the image.
template <int TH = TILE_H, int TW = TILE_W>
__device__ __forceinline__ bool tap_offset(const ConvParams& p, const TileCoord& t, int tap, int& dy, int& dx) {
    if (p.ntaps == 1) { dy = 0; dx = 0; return true; }
    int ky = tap / 3, kx = tap - ky * 3;
    dy = (ky - 1) * p.dil;
    dx = (kx - 1) * p.dil;
    return (t.h0 + dy + TH > 0) && (t.h0 + dy < p.H) && (t.w0 + dx + TW > 0) && (t.w0 + dx < p.W);
}

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t max_bf16x2(uint32_t a, uint32_t b) {
    __nv_bfloat162 r = __hmax2(*reinterpret_cast<__nv_bfloat162*>(&a), *reinterpret_cast<__nv_bfloat162*>(&b));
    return *reinterpret_cast<uint32_t*>(&r);
}

// CTA pairs: the two CTAs of a pair work on two different pixel tiles of the SAME n-tile (they share B).
// pair index -> (m-tile pair, n-tile); tile of CTA `rank` = (2 * mpair + rank) * n_tiles + nt.  An odd m-tile
// count makes the last peer redo the last m-tile (identical stores).
__device__ __forceinline__ int pair_count(const ConvParams& p) {
    return ((p.m_tiles + 1) >> 1) * p.n_tiles;
}
__device__ __forceinline__ int pair_to_tile(const ConvParams& p, int pair, int rank) {
    const int m_tiles = p.m_tiles;
    const int mpair = fast_div(pair, p.fd_ntiles), nt = pair - mpair * p.n_tiles;
    int m = 2 * mpair + rank;
    if (m >= m_tiles) m = m_tiles - 1;
    return m * p.n_tiles + nt;
}

// tcgen05.wait::ld that also names the registers an earlier tcgen05.ld fills: the compiler must not touch
// them before this point (the loads are asynchronous; a plain wait carries no data dependency).
__device__ __forceinline__ void tmem_ld_wait_on(uint32_t* v) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]),
                   "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]),
                   "+r"(v[16]), "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]),
                   "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
                 :
                 : "memory");
}

// Epilogue: EPI_GROUPS groups of 4 warps work on the SAME tile (both wait for the accumulator stage the MMA warp
// just committed).  Within a group the 4 x 32 threads are the 128 TMEM lanes: thread L owns pixel (L / TW, L % TW).
// The groups split the tile's columns: group g drains the 32-column chunks c = g (mod 2) of every half (for the
// HEAD epilogue, whose per-pixel dot product needs all 64 channels in one thread, group g takes the halves
// g (mod 2)).  Draining a stage with all eight warps halves the time the MMA warp waits for it; the stage is
// handed back as soon as a warp's last tcgen05.ld has landed, before that chunk is processed.
// TMEM -> registers (next chunk in flight while this one is processed) -> +bias (staged in smem) -> bf16 with the
// ReLU folded into the conversion -> a warp-private smem tile -> NHWC stores of 8 pixels x 64 B per instruction
// (measured: a thread writing its own pixel's 64 B directly, even as two st.global.v8.b32 sectors, is slower --
// 32 lines per instruction instead of 8).  STORE_POOL also writes the 2x2 max from the staged tile; UPSCATTER
// sends each chunk to its output parity.
// NHALF > 1: the tile is NHALF side-by-side TW-wide patches, each with its own BN-column accumulator.
constexpr int EPI_GROUPS = 2;
constexpr int EPI_STAGE_BYTES = 32 * 64;                    // per warp: 32 pixels x 32 channels bf16
constexpr int EPI_STAGE_TOTAL = EPI_GROUPS * 4 * EPI_STAGE_BYTES;

// Staging slot of 16-byte chunk q (0..3) of pixel row r in a warp's 32 x 64 B buffer: rows 2k, 2k+1 share a
// 128-byte line, (r ^ r>>1) & 1 picks the half and the chunk is rotated by k, so the per-pixel writes (32 rows,
// one q) and the pooled reads (rows r, r+1, r+TW, r+TW+1 for even r; 4 lanes per row) are both conflict-free.
__device__ __forceinline__ uint32_t stg_off(int r, int q) {
    return (uint32_t)(((r >> 1) << 7) | (((r ^ (r >> 1)) & 1) << 6) | ((q ^ ((r >> 1) & 3)) << 4));
}

__device__ __forceinline__ uint32_t pack_bf16_relu(float a, float b) {      // max(., 0) folded into the conversion
    uint32_t r;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
    return r;
}
template <bool PAIR>
__device__ __forceinline__ void release_accumulator(uint64_t* bar, int lane) {
    tc_fence_before();
    __syncwarp();
    if (lane == 0) {
        if (PAIR) mbar_arrive_leader(bar);      // the leader's MMA warp waits for both CTAs
        else mbar_arrive(bar);
    }
}

// fp32 precision (dc_conv_args.planes == 3): the value is stored as three bf16 planes hi + mid + lo, each the
// round-to-nearest bf16 of what the planes before it leave (exact residuals in fp32).  Term t of the six products
// a_i * b_j (i + j <= 2) of a split layer takes activation plane SPLIT_PLANE_A(t) and weight plane SPLIT_PLANE_B(t):
// (0,0) (0,1) (0,2) (1,0) (1,1) (2,0); a1 b2, a2 b1 and a2 b2 are below one fp32 rounding of the product.
__host__ __device__ constexpr int split_plane_a(int t) { return (0x940 >> (2 * t)) & 3; }
__host__ __device__ constexpr int split_plane_b(int t) { return (0x124 >> (2 * t)) & 3; }
constexpr int SPLIT_TERMS = 6;
static_assert(split_plane_a(3) == 1 && split_plane_b(2) == 2 && split_plane_a(5) == 2 && split_plane_b(4) == 1, "terms");

__device__ __forceinline__ float bf16_lo_f(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16_hi_f(uint32_t v) { return __uint_as_float(v & 0xFFFF0000u); }

// UPF (conv_upfused2_kernel): the tile is TH x TW pixels of the HALF-resolution grid and the NHALF = 4 accumulators are
// the four output parities (py, px) = (half / 2, half % 2): pixel (h, w) of accumulator `half` is output pixel
// (2h + py, 2w + px); p.H, p.W are the half-resolution shape and the bias depends on the border class of the pixel.
// SPLIT (conv_tc_split_kernel only): fp32 values stored as three bf16 planes, see split_plane_a.
template <int BN, int TH, int TW, int NHALF = 1, bool PAIR = false, bool COOP = true, bool UPF = false, bool SPLIT = false>
__device__ __forceinline__ void run_epilogue(const ConvParams& p, const int e, const int lane, const int group,
                                             const uint32_t tmem_base, uint64_t* tfull_bar, uint64_t* tempty_bar,
                                             const float* bias_s, uint8_t* stg_all) {
    static_assert(!SPLIT || (TH == 8 && TW == 16 && NHALF == 1 && !PAIR && COOP && !UPF), "split epilogue: generic tiles only");
    const int L = e * 32 + lane;                               // e == warp % 4: TMEM lanes [32e, 32e+32)
    const int lh = L / TW, lw = L % TW;
    const float* head_s = bias_s + p.Cout;                     // out_conv weights follow the bias (HEAD only)
    uint8_t* stg = stg_all + (group * 4 + e) * EPI_STAGE_BYTES;
    const int sq = lane & 3;                                   // the 16-byte chunk this lane handles of a pooled pixel
    // first of the four warp-local pixels (index = row * TW + col) of the pooled pixel this lane stores
    const int pool_r0 = (TW == 16) ? 2 * (lane >> 2) : (16 * (lane >> 4) + 2 * ((lane >> 2) & 3));
    // COOP = false (the stem, whose MMA is a single instruction per tile): the groups take alternate tiles instead,
    // group g owning accumulator stage g, so that a warp always has a second chunk to prefetch.
    constexpr int CPG = COOP ? BN / 64 : BN / 32;              // chunks per half per group
    constexpr int CSTEP = COOP ? 64 : 32;                      // column distance between a group's chunks
    constexpr int NI = NHALF * CPG;                            // chunks per tile per group
    const int cgrp = COOP ? group * 32 : 0;                    // first column of this group's first chunk
    // Output addressing, split into a per-lane part fixed for the whole kernel and warp-uniform parts per tile /
    // half / chunk (the address arithmetic used to cost more instructions than the arithmetic on the data).
    // After the transpose this lane stores chunk sq of pixels pL0 + 8 r (r = 0..3) of its warp's 32.
    const bool up = !UPF && p.epilogue == DC_EPI_UPSCATTER;
    const bool up_geo = UPF || up;                             // output pixels are 2 apart in a [B,2H,2W,*] tensor
    const int pL0 = e * 32 + (lane >> 2);
    const int row0 = pL0 / TW, col0 = pL0 % TW;
    const long long cs = (long long)p.out_stride * (up_geo ? 2 : 1);             // elements per tile column
    const long long rs = (long long)p.out_stride * (up_geo ? 4 : 1) * p.W;       // elements per tile row
    __nv_bfloat16* const lane_ptr = p.out + (row0 * rs + col0 * cs + p.out_offset + sq * 8);
    // pooled pixel of this lane: lane / 4 of the 8 the warp's 32 pixels pool into
    const int prow = (TW == 16) ? e : 2 * e + (lane >> 4);
    const int pcol = (TW == 16) ? (lane >> 2) : ((lane >> 2) & 3);
    // UPF: the pooled tensor has the tile's own (half-resolution) geometry; this lane stores chunk sq of pixels pL0 + 8 r
    __nv_bfloat16* const pool_lane_ptr =
        UPF ? p.pool_out + (((long long)row0 * p.W + col0) * p.pool_stride + sq * 8)
            : p.pool_out + (((long long)prow * (p.W >> 1) + pcol) * p.pool_stride + sq * 8);
    for (int it = COOP ? 0 : group;; it += COOP ? 1 : EPI_GROUPS) {
        int tile;
        if (PAIR) {                     // CTA pair: pair = cluster + it * clusters
            const int pair = (int)(blockIdx.x >> 1) + it * (int)(gridDim.x >> 1);
            if (pair >= pair_count(p)) break;
            tile = pair_to_tile(p, pair, (int)(blockIdx.x & 1));
        } else {
            tile = blockIdx.x + it * gridDim.x;
            if (tile >= p.total_tiles) break;
        }
        TileCoord t = decode_tile<TH, UPF ? TW : TW * NHALF>(p, tile, BN);
        // UPF with fewer than four classes per pass (conv_upfused_wide_kernel): the n-tile index also carries the class
        // group; accumulator `half` is parity class cls_base + half.  With all four classes in one pass (NHALF == 4) the
        // accumulators sit in Gray order 0, 1, 3, 2 (class = half ^ (half >> 1)): three of the four class pairings are
        // then adjacent TMEM ranges and run as one N = 128 MMA (tools/gen_upf_schedule.py)
        int cls_base = 0;
        if (UPF) {
            const int cg = t.n0 / p.Cout;
            t.n0 -= cg * p.Cout;
            cls_base = cg * NHALF;
        }
        const int as = it & 1;
        const uint32_t aphase = (uint32_t)(it >> 1) & 1u;
        mbar_wait(&tfull_bar[as], aphase);
        tc_fence_after();
        const uint32_t tstage = tmem_base + ((uint32_t)(e * 32) << 16) + (uint32_t)(as * NHALF * BN);

        if (p.epilogue == DC_EPI_HEAD) {
#pragma unroll 1
            for (int half = COOP ? group : 0; half < NHALF; half += COOP ? EPI_GROUPS : 1) {
                // UPF: accumulator `half` = parity class (half / 2, half % 2) of half-resolution pixel (t.h0 + lh, t.w0 + lw)
                const int cls = NHALF == 4 ? (half ^ (half >> 1)) : cls_base + half;
                const int h = UPF ? 2 * (t.h0 + lh) + (cls >> 1) : t.h0 + lh;
                const int w = UPF ? 2 * (t.w0 + lw) + (cls & 1) : t.w0 + half * TW + lw;
                const int H_out = UPF ? 2 * p.H : p.H, W_out = UPF ? 2 * p.W : p.W;
                float head_acc = p.head_b;
                const uint32_t taddr = tstage + (uint32_t)(half * BN);
                uint32_t vbuf[2][32];
                tmem_ld32(taddr, vbuf[0]);
#pragma unroll
                for (int c = 0; c < BN / 32; ++c) {
                    uint32_t* v = vbuf[c & 1];
                    tmem_ld_wait_on(v);
                    if (c + 1 < BN / 32) tmem_ld32(taddr + (uint32_t)(c * 32 + 32), vbuf[(c + 1) & 1]);
                    else if (half + (COOP ? EPI_GROUPS : 1) >= NHALF) release_accumulator<PAIR>(&tempty_bar[as], lane);
                    const float4* b4 = reinterpret_cast<const float4*>(bias_s + t.n0 + c * 32);
                    const float4* w4 = reinterpret_cast<const float4*>(head_s + c * 32);
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float4 b = b4[j], hw = w4[j];
                        float x0 = __uint_as_float(v[4 * j + 0]) + b.x, x1 = __uint_as_float(v[4 * j + 1]) + b.y;
                        float x2 = __uint_as_float(v[4 * j + 2]) + b.z, x3 = __uint_as_float(v[4 * j + 3]) + b.w;
                        if (p.relu) { x0 = fmaxf(x0, 0.f); x1 = fmaxf(x1, 0.f); x2 = fmaxf(x2, 0.f); x3 = fmaxf(x3, 0.f); }
                        head_acc = fmaf(x0, hw.x, head_acc);
                        head_acc = fmaf(x1, hw.y, head_acc);
                        head_acc = fmaf(x2, hw.z, head_acc);
                        head_acc = fmaf(x3, hw.w, head_acc);
                    }
                }
                if ((h < H_out) && (w < W_out)) {
                    const float prob = 1.0f / (1.0f + expf(-head_acc));              // torch.sigmoid, fp32
                    const size_t opix = ((size_t)t.img * H_out + h) * (size_t)W_out + w;
                    if (p.prob_out) p.prob_out[opix] = prob;
                    if (p.mask_out) p.mask_out[opix] = prob > p.thresh ? 1 : 0;      // qdb:56
                }
            }
            if (COOP && group >= NHALF) release_accumulator<PAIR>(&tempty_bar[as], lane);     // a group with no half of its own
            continue;
        }

        const uint32_t tbase = tstage + (uint32_t)cgrp;
        uint32_t vbuf[2][32];
        tmem_ld32(tbase, vbuf[0]);
        // warp-uniform offsets of this tile
        const long long tile_off = up_geo ? (((long long)t.img * (2 * p.H) + 2 * t.h0) * (2 * p.W) + 2 * t.w0) * p.out_stride + (UPF ? t.n0 : 0)
                                          : (((long long)t.img * p.H + t.h0) * p.W + t.w0) * p.out_stride + t.n0;
        const long long ptile_off = UPF ? (((long long)t.img * p.H + t.h0) * p.W + t.w0) * p.pool_stride + t.n0
                                        : (((long long)t.img * (p.H >> 1) + (t.h0 >> 1)) * (p.W >> 1) + (t.w0 >> 1)) * p.pool_stride + t.n0;
        uint32_t pmax[16];                                     // UPF + STORE_POOL: running 2x2 max over the four classes
        const int hmax = p.H - t.h0;
        int q0 = 0, rem0 = 0;                                  // UPSCATTER: n0 = q0 * Cout + rem0
        if (up) { q0 = t.n0 / p.Cout; rem0 = t.n0 - q0 * p.Cout; }
        uint32_t vmask = 0;                                    // bit r: pixel pL0 + 8 r of this half is inside the image
        bool pval = false;
        long long half_off = 0, phalf_off = 0;
#pragma unroll
        for (int j = 0; j < NI; ++j) {
            const int half = j / CPG, cc = j % CPG;            // compile-time
            const int c0 = cc * CSTEP + cgrp;                  // first GEMM column of this chunk within the n-tile
            uint32_t* v = vbuf[j & 1];
            tmem_ld_wait_on(v);
            if (j + 1 < NI) tmem_ld32(tbase + (uint32_t)(((j + 1) / CPG) * BN + ((j + 1) % CPG) * CSTEP), vbuf[(j + 1) & 1]);
            else release_accumulator<PAIR>(&tempty_bar[as], lane);            // this warp has read all it will
            if (cc == 0) {
                const int wmax = p.W - t.w0 - (UPF ? 0 : half * TW);
                vmask = 0;
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const int row = row0 + (TW == 16 ? (r >> 1) : r), col = col0 + (TW == 16 ? (r & 1) * 8 : 0);
                    vmask |= (uint32_t)((row < hmax) && (col < wmax)) << r;
                }
                pval = (2 * prow < hmax) && (2 * pcol < wmax);
                const int cls = NHALF == 4 ? (half ^ (half >> 1)) : cls_base + half;
                half_off = UPF ? ((long long)(cls >> 1) * (2 * p.W) + (cls & 1)) * p.out_stride : half * TW * cs;
                phalf_off = (long long)(half * (TW / 2)) * p.pool_stride;
            }
            int bias_at = t.n0 + c0;
            long long chunk_off = c0;
            if (up) {
                // GEMM column n = (a*2 + b)*Cout + co  ->  output pixel (2h + a, 2w + b), channel co
                int co = rem0 + c0, q = q0;
                while (co >= p.Cout) { co -= p.Cout; ++q; }
                bias_at = co;
                chunk_off = ((long long)(q >> 1) * (2 * p.W) + (q & 1)) * p.out_stride + co;
            }
            __nv_bfloat16* const dst = lane_ptr + (tile_off + half_off + chunk_off);
            float x[32];
            if (p.bias_const) {
                // Cout == 64: this chunk's 32 biases are kernel parameters at a compile-time offset, i.e. constant-bank
                // operands of the FADDs (the smem path below costs 16 of a chunk's ~64 LSU wavefronts, and the
                // store-heavy layers run at 85 % of the LSU data pipe)
                if ((COOP ? group : (cc & 1)) == 0) {
#pragma unroll
                    for (int k = 0; k < 32; ++k) x[k] = __uint_as_float(v[k]) + p.bias_c[k];
                } else {
#pragma unroll
                    for (int k = 0; k < 32; ++k) x[k] = __uint_as_float(v[k]) + p.bias_c[32 + k];
                }
            } else {
                const float4* b4 = reinterpret_cast<const float4*>(bias_s + bias_at);
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const float4 b = b4[k];
                    x[4 * k + 0] = __uint_as_float(v[4 * k + 0]) + b.x;
                    x[4 * k + 1] = __uint_as_float(v[4 * k + 1]) + b.y;
                    x[4 * k + 2] = __uint_as_float(v[4 * k + 2]) + b.z;
                    x[4 * k + 3] = __uint_as_float(v[4 * k + 3]) + b.w;
                }
            }
            if (UPF && p.border_bias) {
                // taps of the 3x3 that fall outside the (upsampled) image carry no transposed-conv bias: only the
                // pixels of the first / last output row and column differ from the interior constant
                const int hh = t.h0 + lh, ww = t.w0 + lw;
                const int cls = NHALF == 4 ? (half ^ (half >> 1)) : cls_base + half;
                const int py = cls >> 1, px = cls & 1;
                const int rc = (py == 0 && hh == 0) ? 0 : ((py == 1 && hh == p.H - 1) ? 2 : 1);
                const int cc9 = (px == 0 && ww == 0) ? 0 : ((px == 1 && ww == p.W - 1) ? 2 : 1);
                if (rc * 3 + cc9 != 4) {               // p.bias = the interior row (4) of the fp32 [9][Cout] class table
                    const float* b4 = p.bias + t.n0 + c0;
                    const float* bc = b4 + (rc * 3 + cc9 - 4) * p.Cout;
#pragma unroll
                    for (int k = 0; k < 32; ++k) x[k] += __ldg(bc + k) - __ldg(b4 + k);
                }
            }
            if constexpr (SPLIT) {
                if (p.relu) {
#pragma unroll
                    for (int k = 0; k < 32; ++k) x[k] = fmaxf(x[k], 0.f);
                }
                if (p.epilogue == DC_EPI_STORE_POOL) {
                    // 2x2 max of the fp32 values, then split: a max per plane is not the max of the sums.  Pixel
                    // (row, col) of this warp's two rows is lane row * 16 + col, so the window of pooled pixel (e, pc)
                    // is lanes 2 pc, 2 pc + 1, 2 pc + 16, 2 pc + 17 and lane 2 pc stores it.
                    const int pc = (lane >> 1) & 7;
                    const bool pown = (lane & 17) == 0 && (2 * e < hmax) && (2 * pc < p.W - t.w0);
                    __nv_bfloat16* const pdst = p.pool_out + (ptile_off + ((long long)e * (p.W >> 1) + pc) * p.pool_stride + c0);
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        float m[8];
#pragma unroll
                        for (int k = 0; k < 8; ++k) {
                            const float a = fmaxf(x[8 * g + k], __shfl_xor_sync(0xffffffffu, x[8 * g + k], 1));
                            m[k] = fmaxf(a, __shfl_xor_sync(0xffffffffu, a, 16));
                        }
#pragma unroll
                        for (int pl = 0; pl < 3; ++pl) {
                            uint32_t q[4];
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                q[k] = pack_bf16(m[2 * k], m[2 * k + 1]);
                                m[2 * k] -= bf16_lo_f(q[k]);
                                m[2 * k + 1] -= bf16_hi_f(q[k]);
                            }
                            if (pown)
                                *reinterpret_cast<uint4*>(pdst + (8 * g + (long long)pl * p.pool_plane_stride)) =
                                    make_uint4(q[0], q[1], q[2], q[3]);
                        }
                    }
                }
                // plane pl = round-to-nearest bf16 of what planes 0..pl-1 leave of x; each through the staged transpose
#pragma unroll 1
                for (int pl = 0; pl < 3; ++pl) {
                    uint32_t pk[16];
#pragma unroll
                    for (int k = 0; k < 16; ++k) {
                        pk[k] = pack_bf16(x[2 * k], x[2 * k + 1]);
                        x[2 * k] -= bf16_lo_f(pk[k]);
                        x[2 * k + 1] -= bf16_hi_f(pk[k]);
                    }
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        *reinterpret_cast<uint4*>(stg + stg_off(lane, q)) = make_uint4(pk[4 * q], pk[4 * q + 1], pk[4 * q + 2], pk[4 * q + 3]);
                    __syncwarp();
                    __nv_bfloat16* const pdst = dst + (long long)pl * p.out_plane_stride;
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
                        const uint4 val = *reinterpret_cast<const uint4*>(stg + stg_off(8 * r + (lane >> 2), sq));
                        const long long d = (r & 1) * 8 * cs + (r >> 1) * rs;
                        if (vmask & (1u << r)) *reinterpret_cast<uint4*>(pdst + d) = val;
                    }
                    __syncwarp();
                }
                continue;
            }
            uint32_t pk[16];
            if (p.relu) {
#pragma unroll
                for (int k = 0; k < 16; ++k) pk[k] = pack_bf16_relu(x[2 * k], x[2 * k + 1]);
            } else {
#pragma unroll
                for (int k = 0; k < 16; ++k) pk[k] = pack_bf16(x[2 * k], x[2 * k + 1]);
            }
            // Stores go out transposed: a thread holds 32 channels of ONE pixel (64 B); written directly, every store
            // instruction would touch 32 different lines.  The chunk is staged in a warp-private smem tile and stored
            // as 8 pixels x 64 contiguous bytes per instruction (4 lanes per pixel).
#pragma unroll
            for (int q = 0; q < 4; ++q)
                *reinterpret_cast<uint4*>(stg + stg_off(lane, q)) = make_uint4(pk[4 * q], pk[4 * q + 1], pk[4 * q + 2], pk[4 * q + 3]);
            __syncwarp();
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const uint4 val = *reinterpret_cast<const uint4*>(stg + stg_off(8 * r + (lane >> 2), sq));
                const long long d = (TW == 16) ? (r & 1) * 8 * cs + (r >> 1) * rs : r * rs;      // pixel pL0 + 8 r
                if (vmask & (1u << r)) *reinterpret_cast<uint4*>(dst + d) = val;
            }
            if (UPF && p.epilogue == DC_EPI_STORE_POOL) {
                // the four classes of this lane's pixel are the 2x2 window (max of bf16-rounded values = bf16 rounding
                // of the max): keep the running max in registers, store after the fourth class through the same
                // staging transpose as the full-resolution stores
#pragma unroll
                for (int k = 0; k < 16; ++k) pmax[k] = half == 0 ? pk[k] : max_bf16x2(pmax[k], pk[k]);
                if (half == NHALF - 1) {
                    __syncwarp();
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        *reinterpret_cast<uint4*>(stg + stg_off(lane, q)) = make_uint4(pmax[4 * q], pmax[4 * q + 1], pmax[4 * q + 2], pmax[4 * q + 3]);
                    __syncwarp();
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
                        const uint4 val = *reinterpret_cast<const uint4*>(stg + stg_off(8 * r + (lane >> 2), sq));
                        if (vmask & (1u << r))
                            *reinterpret_cast<uint4*>(pool_lane_ptr + (ptile_off + (long long)r * p.W * p.pool_stride + c0)) = val;
                    }
                }
            } else if (p.epilogue == DC_EPI_STORE_POOL) {
                // 2x2 max straight from the staged tile: lane (pp, sq) reads chunk sq of the four pixels of pooled
                // pixel pp (the max of bf16-rounded values = the bf16 rounding of the max)
                const uint4 a0 = *reinterpret_cast<const uint4*>(stg + stg_off(pool_r0, sq));
                const uint4 a1 = *reinterpret_cast<const uint4*>(stg + stg_off(pool_r0 + 1, sq));
                const uint4 a2 = *reinterpret_cast<const uint4*>(stg + stg_off(pool_r0 + TW, sq));
                const uint4 a3 = *reinterpret_cast<const uint4*>(stg + stg_off(pool_r0 + TW + 1, sq));
                uint4 m;
                m.x = max_bf16x2(max_bf16x2(a0.x, a1.x), max_bf16x2(a2.x, a3.x));
                m.y = max_bf16x2(max_bf16x2(a0.y, a1.y), max_bf16x2(a2.y, a3.y));
                m.z = max_bf16x2(max_bf16x2(a0.z, a1.z), max_bf16x2(a2.z, a3.z));
                m.w = max_bf16x2(max_bf16x2(a0.w, a1.w), max_bf16x2(a2.w, a3.w));
                if (pval) *reinterpret_cast<uint4*>(pool_lane_ptr + (ptile_off + phalf_off + c0)) = m;
            }
            __syncwarp();
        }
    }
}

// bias (+ out_conv weights for the HEAD epilogue) -> shared memory, by every thread, before the role split
__device__ __forceinline__ void stage_bias(const ConvParams& p, float* bias_s) {
    for (int i = threadIdx.x; i < p.Cout; i += blockDim.x) bias_s[i] = p.bias[i];
    if (p.epilogue == DC_EPI_HEAD)
        for (int i = threadIdx.x; i < p.Cout; i += blockDim.x) bias_s[p.Cout + i] = p.head_w[i];
}

// The body of conv_tc_kernel (bf16) and conv_tc_split_kernel (fp32 precision: the K walk of every tap is (term,
// 64-channel chunk) over the six terms of split_plane_a, and the epilogue stores three planes).
template <int BN, int NSTAGES, bool SPLIT>
__device__ __forceinline__ void conv_tc_body(const ConvParams& p) {
    constexpr int B_STAGE_BYTES = BN * KCHUNK * 2;
    constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
    constexpr int TMEM_COLS = 2 * BN;   // 128 / 256 / 512: a power of two >= 32

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // SWIZZLE_128B wants 1024 B
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + NSTAGES * STAGE_BYTES);
    uint64_t* empty_bar = full_bar + NSTAGES;
    uint64_t* tfull_bar = empty_bar + NSTAGES;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
    float* bias_s = reinterpret_cast<float*>(smem + NSTAGES * STAGE_BYTES + 256);
    uint8_t* stg_s = smem + NSTAGES * STAGE_BYTES + 256 + 4096 + 256;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    stage_bias(p, bias_s);
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&p.tmA);
        tma_prefetch_desc(&p.tmB);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < NSTAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(&tfull_bar[s], 1); mbar_init(&tempty_bar[s], 4 * EPI_GROUPS); }
        fence_barrier_init();
    }
    if (warp == 2) {
        tmem_alloc(tmem_slot, TMEM_COLS);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer (warp-uniform loop)
        int stage = 0;
        uint32_t phase = 0;
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
            const TileCoord t = decode_tile(p, tile, BN);
            for (int tap = 0; tap < p.ntaps; ++tap) {
                int dy, dx;
                if (!tap_offset(p, t, tap, dy, dx)) continue;
                for (int kc = 0; kc < (SPLIT ? SPLIT_TERMS * p.kchunks : p.kchunks); ++kc) {
                    mbar_wait(&empty_bar[stage], phase ^ 1u);
                    if (elect_one()) {
                        uint8_t* sa = smem + stage * STAGE_BYTES;
                        mbar_expect_tx(&full_bar[stage], STAGE_BYTES);
                        if constexpr (SPLIT) {
                            // weights [Cout][9 taps][3 planes][Cin]: column tap * 3 Cin + plane * Cin + channel
                            const int term = kc / p.kchunks, ch = (kc - term * p.kchunks) * KCHUNK;
                            tma_load_4d(sa, &p.tmA, &full_bar[stage], split_plane_a(term) * p.in_plane_stride + ch, t.w0 + dx,
                                        t.h0 + dy, t.img);
                            tma_load_2d(sa + A_STAGE_BYTES, &p.tmB, &full_bar[stage], (3 * tap + split_plane_b(term)) * p.Cin + ch,
                                        t.n0);
                        } else {
                            tma_load_4d(sa, &p.tmA, &full_bar[stage], kc * KCHUNK, t.w0 + dx, t.h0 + dy, t.img);
                            tma_load_2d(sa + A_STAGE_BYTES, &p.tmB, &full_bar[stage], tap * p.Cin + kc * KCHUNK, t.n0);
                        }
                    }
                    __syncwarp();
                    if (++stage == NSTAGES) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer (warp-uniform loop)
        const uint32_t idesc = umma_idesc_bf16(TILE_M, BN);
        int stage = 0;
        uint32_t phase = 0;
        int it = 0;
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
            const TileCoord t = decode_tile(p, tile, BN);
            const int as = it & 1;
            const uint32_t aphase = (uint32_t)(it >> 1) & 1u;
            mbar_wait(&tempty_bar[as], aphase ^ 1u);      // epilogue has drained this accumulator
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)(as * BN);
            uint32_t accumulate = 0;
            for (int tap = 0; tap < p.ntaps; ++tap) {
                int dy, dx;
                if (!tap_offset(p, t, tap, dy, dx)) continue;
                for (int kc = 0; kc < (SPLIT ? SPLIT_TERMS * p.kchunks : p.kchunks); ++kc) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    const uint32_t sa = smem_u32(smem + stage * STAGE_BYTES);
                    const uint64_t adesc = umma_desc_sw128(sa);
                    const uint64_t bdesc = umma_desc_sw128(sa + A_STAGE_BYTES);
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < KCHUNK / 16; ++k) {
                            // +32 B per K=16 step inside the 128 B swizzle row (address field is >>4)
                            umma_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc,
                                      (k == 0) ? accumulate : 1u);
                        }
                        umma_commit(&empty_bar[stage]);        // frees the stage once these MMAs retire
                    }
                    __syncwarp();
                    accumulate = 1;
                    if (++stage == NSTAGES) { stage = 0; phase ^= 1u; }
                }
            }
            if (elect_one()) umma_commit(&tfull_bar[as]);       // accumulator complete -> epilogue
            __syncwarp();
        }
    } else if (warp >= EPI_WARP0) {
        // ------------------------------------------------------------------ epilogue
        run_epilogue<BN, TILE_H, TILE_W, 1, false, true, false, SPLIT>(p, warp & 3, lane, (warp - EPI_WARP0) >> 2, tmem_base,
                                                                       tfull_bar, tempty_bar, bias_s, stg_s);
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

template <int BN, int NSTAGES>
__global__ void __launch_bounds__(NUM_THREADS, 1) conv_tc_kernel(const __grid_constant__ ConvParams p) {
    conv_tc_body<BN, NSTAGES, false>(p);
}

template <int BN, int NSTAGES>
__global__ void __launch_bounds__(NUM_THREADS, 1) conv_tc_split_kernel(const __grid_constant__ ConvParams p) {
    conv_tc_body<BN, NSTAGES, true>(p);
}

// ---------------------------------------------------------------------------- halo variant
constexpr int HT_H = 16, HT_W = 8;      // 16 x 8 output patch: each 8-pixel row is one UMMA 8-row group
// NHALF = 2: two patches side by side (16 x 16 pixels) share one haloed region and accumulate into separate
// TMEM tiles -- two independent MMA chains hide the latency of back-to-back accumulating MMAs at N = 64 / 128.
constexpr int HALO_MAX_STAGES = 8;
constexpr int HALO_BAR_BYTES = 512;     // 4 x 8 stage barriers + TMEM / weight barriers + TMEM slot
constexpr int HALO_BIAS_BYTES = 4096 + 256;   // bias (<= 1024 channels) + out_conv weights

// K-major SWIZZLE_128B descriptor whose 8-row groups are `sbo_bytes` apart and whose start may sit on any
// 128 B row of a 1024 B-aligned region.  Measured on B200 (tests/test_gpu_conv.py halo cases): the MMA unit
// derives the swizzle phase from the absolute shared-memory address bits [7,10), exactly as TMA does when it
// writes the region, so base_offset stays 0 and a window may start on any row.
__device__ __forceinline__ uint64_t umma_desc_sw128_strided(uint32_t smem_addr, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

// Cout = 64 layers with long K at dilation <= 4, whose weights do not fit next to the pair kernel's regions (and the
// pair kernel does not stream weights at N = 64): two 8-wide halves per tile, the weights streamed through a ring of
// p.nbstages 64 x 64 (tap, chunk) slices.  Each slice still feeds 2 x 4 MMAs and the activations are still loaded
// once per chunk instead of once per tap, which is what keeps these layers off the L2 roofline.
constexpr int HALO_BN = 64, HALO_NHALF = 2;
constexpr int HALO_W_TILE_BYTES = HALO_BN * KCHUNK * 2;      // one (tap, chunk) slice of the weights

__global__ void __launch_bounds__(NUM_THREADS, 1) conv_halo_kernel(const __grid_constant__ ConvParams p) {
    constexpr int BN = HALO_BN;
    constexpr int HT_TW = HT_W * HALO_NHALF;
    constexpr int W_TILE_BYTES = HALO_W_TILE_BYTES;
    constexpr int TMEM_COLS = 2 * HALO_NHALF * BN;

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* w_ring = smem;                                            // the weight ring
    uint8_t* a_ring = smem + p.nbstages * W_TILE_BYTES;                // haloed activation regions
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(a_ring + p.nstages * p.region_stride);
    uint64_t* empty_bar = full_bar + HALO_MAX_STAGES;
    uint64_t* bfull_bar = empty_bar + HALO_MAX_STAGES;
    uint64_t* bempty_bar = bfull_bar + HALO_MAX_STAGES;
    uint64_t* tfull_bar = bempty_bar + HALO_MAX_STAGES;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
    float* bias_s = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full_bar) + HALO_BAR_BYTES);
    uint8_t* stg_s = reinterpret_cast<uint8_t*>(full_bar) + HALO_BAR_BYTES + HALO_BIAS_BYTES;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int NST = p.nstages;
    const int NBS = p.nbstages;

    stage_bias(p, bias_s);
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&p.tmA);
        tma_prefetch_desc(&p.tmB);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < HALO_MAX_STAGES; ++s) {
            mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1);
            mbar_init(&bfull_bar[s], 1); mbar_init(&bempty_bar[s], 1);
        }
        for (int s = 0; s < 2; ++s) { mbar_init(&tfull_bar[s], 1); mbar_init(&tempty_bar[s], 4 * EPI_GROUPS); }
        fence_barrier_init();
    }
    if (warp == 2) {
        tmem_alloc(tmem_slot, TMEM_COLS);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t region_bytes = (uint32_t)(p.region_w * p.region_h * KCHUNK * 2);

    // taps whose window lies wholly in the zero padding contribute nothing: both roles skip them
    auto tile_tap_mask = [&](const TileCoord& t) {
        uint32_t m = 0;
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
            int dy, dx;
            if (tap_offset<HT_H, HT_TW>(p, t, tap, dy, dx)) m |= 1u << tap;
        }
        return m;
    };

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer (warp-uniform loop)
        int stage = 0, bstage = 0;
        uint32_t phase = 0, bphase = 0;
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
            const TileCoord t = decode_tile<HT_H, HT_TW>(p, tile, BN);
            const uint32_t tap_mask = tile_tap_mask(t);
            for (int kc = 0; kc < p.kchunks; ++kc) {
                mbar_wait(&empty_bar[stage], phase ^ 1u);
                if (elect_one()) {
                    mbar_expect_tx(&full_bar[stage], region_bytes);
                    tma_load_4d(a_ring + stage * p.region_stride, &p.tmA, &full_bar[stage], kc * KCHUNK, t.w0 - p.dil,
                                t.h0 - p.dil, t.img);
                }
                __syncwarp();
                if (++stage == NST) { stage = 0; phase ^= 1u; }
                for (int tap = 0; tap < 9; ++tap) {
                    if (!((tap_mask >> tap) & 1u)) continue;
                    mbar_wait(&bempty_bar[bstage], bphase ^ 1u);
                    if (elect_one()) {
                        mbar_expect_tx(&bfull_bar[bstage], W_TILE_BYTES);
                        tma_load_2d(w_ring + bstage * W_TILE_BYTES, &p.tmB, &bfull_bar[bstage],
                                    (tap * p.kchunks + kc) * KCHUNK, 0);
                    }
                    __syncwarp();
                    if (++bstage == NBS) { bstage = 0; bphase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer (warp-uniform loop)
        const uint32_t idesc = umma_idesc_bf16(TILE_M, BN);
        const uint32_t sbo = (uint32_t)p.region_w * 128u;
        const uint32_t w_addr = smem_u32(w_ring);
        const uint32_t tap_dy_bytes = (uint32_t)(p.dil * p.region_w) * 128u;     // one tap row down
        const uint32_t tap_dx_bytes = (uint32_t)p.dil * 128u;                    // one tap column right
        int stage = 0, bstage = 0;
        uint32_t phase = 0, bphase = 0;
        int it = 0;
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
            const TileCoord t = decode_tile<HT_H, HT_TW>(p, tile, BN);
            const int as = it & 1;
            const uint32_t aphase = (uint32_t)(it >> 1) & 1u;
            const uint32_t tap_mask = tile_tap_mask(t);
            mbar_wait(&tempty_bar[as], aphase ^ 1u);
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)(as * HALO_NHALF * BN);
            uint32_t accumulate = 0;
            for (int kc = 0; kc < p.kchunks; ++kc) {
                mbar_wait(&full_bar[stage], phase);
                tc_fence_after();
                const uint32_t region = smem_u32(a_ring + stage * p.region_stride);
#pragma unroll 1
                for (int tap = 0; tap < 9; ++tap) {
                    if (!((tap_mask >> tap) & 1u)) continue;
                    mbar_wait(&bfull_bar[bstage], bphase);
                    tc_fence_after();
                    const uint32_t a_addr = region + (uint32_t)(tap / 3) * tap_dy_bytes + (uint32_t)(tap % 3) * tap_dx_bytes;
                    const uint64_t adesc = umma_desc_sw128_strided(a_addr, sbo);
                    const uint64_t bdesc = umma_desc_sw128(w_addr + (uint32_t)(bstage * W_TILE_BYTES));
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < KCHUNK / 16; ++k) {
#pragma unroll
                            for (int half = 0; half < HALO_NHALF; ++half)   // right patch = 8 region rows (1024 B) further
                                umma_bf16(d_tmem + (uint32_t)(half * BN), adesc + (uint64_t)(2 * k + 64 * half),
                                          bdesc + (uint64_t)(2 * k), idesc, (k == 0) ? accumulate : 1u);
                        }
                        umma_commit(&bempty_bar[bstage]);
                    }
                    __syncwarp();
                    accumulate = 1;
                    if (++bstage == NBS) { bstage = 0; bphase ^= 1u; }
                }
                if (elect_one()) umma_commit(&empty_bar[stage]);
                __syncwarp();
                if (++stage == NST) { stage = 0; phase ^= 1u; }
            }
            if (elect_one()) umma_commit(&tfull_bar[as]);
            __syncwarp();
        }
    } else if (warp >= EPI_WARP0) {
        run_epilogue<BN, HT_H, HT_W, HALO_NHALF>(p, warp & 3, lane, (warp - EPI_WARP0) >> 2, tmem_base, tfull_bar, tempty_bar, bias_s, stg_s);
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

// ---------------------------------------------------------------------------- halo variant on CTA pairs
// cta_group::2: the two SMs of a pair run ONE M = 256 MMA stream.  Each CTA owns its own 16 x 16 pixel tile
// (rows [0,128) / [128,256) of the MMA come from the leader's / the peer's haloed region at the same smem offset)
// and HALF of the weight rows (N/2), so the weights of a layer need half the shared memory per SM -- dec1.0's
// 144 KB become 72 KB and leave room for two-half regions -- and the B-operand smem reads per SM halve
// (A 4 KB + B N/2 x 32 B per MMA), which is what bounds the N = 64 layers.
// Leader = even CTA: it alone issues the MMAs; both CTAs run a TMA producer (bytes credited to the leader's
// barriers), both run epilogues on their own TMEM half, commits are multicast to both CTAs' barriers.
template <int BN, int NH, bool WRES>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
conv_halo2_kernel(const __grid_constant__ ConvParams p) {
    constexpr int HT_TW = HT_W * NH;
    constexpr int W_TILE_BYTES = (BN / 2) * KCHUNK * 2;     // this CTA's half of one (tap, chunk) weight slice
    constexpr int TMEM_USED = 2 * NH * BN;
    constexpr int TMEM_COLS = TMEM_USED <= 128 ? 128 : (TMEM_USED <= 256 ? 256 : 512);   // power of two
    static_assert(TMEM_USED <= 512, "accumulators exceed TMEM");

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const int n_wtiles = WRES ? 9 * p.kchunks : p.nbstages;
    uint8_t* w_res = smem;                                          // resident half-weights, or the weight ring
    uint8_t* a_ring = smem + n_wtiles * W_TILE_BYTES;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(a_ring + p.nstages * p.region_stride);
    uint64_t* empty_bar = full_bar + HALO_MAX_STAGES;
    uint64_t* bfull_bar = empty_bar + HALO_MAX_STAGES;
    uint64_t* bempty_bar = bfull_bar + HALO_MAX_STAGES;
    uint64_t* tfull_bar = bempty_bar + HALO_MAX_STAGES;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint64_t* w_bar = tempty_bar + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(w_bar + 1);
    float* bias_s = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full_bar) + HALO_BAR_BYTES);
    uint8_t* stg_s = reinterpret_cast<uint8_t*>(full_bar) + HALO_BAR_BYTES + HALO_BIAS_BYTES;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int NST = p.nstages;
    const int NBS = p.nbstages;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;
    const int cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;
    const int n_pairs = pair_count(p);

    stage_bias(p, bias_s);
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&p.tmA);
        tma_prefetch_desc(&p.tmB);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < HALO_MAX_STAGES; ++s) {
            mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1);
            mbar_init(&bfull_bar[s], 1); mbar_init(&bempty_bar[s], 1);
        }
        for (int s = 0; s < 2; ++s) { mbar_init(&tfull_bar[s], 1); mbar_init(&tempty_bar[s], 8 * EPI_GROUPS); }   // 4 x EPI_GROUPS warps x 2 CTAs
        mbar_init(w_bar, 1);
        fence_barrier_init();
    }
    if (warp == 2) {
        tmem_alloc_2sm(tmem_slot, TMEM_COLS);
        tmem_relinquish_2sm();
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                 // the peer's barriers exist before anything is signalled across the pair
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t region_bytes = (uint32_t)(p.region_w * p.region_h * KCHUNK * 2);

    auto pair_tile = [&](int pair) { return pair_to_tile(p, pair, (int)rank); };

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer (one per CTA)
        if (WRES) {
            if (elect_one()) {
                if (leader) mbar_expect_tx(w_bar, (uint32_t)(2 * n_wtiles * W_TILE_BYTES));
                for (int j = 0; j < n_wtiles; ++j)
                    tma_load_2d_2sm(w_res + j * W_TILE_BYTES, &p.tmB, w_bar, j * KCHUNK, (int)rank * (BN / 2));   // n_tiles == 1
            }
            __syncwarp();
        }
        int stage = 0, bstage = 0;
        uint32_t phase = 0, bphase = 0;
        for (int pair = cluster_id; pair < n_pairs; pair += n_clusters) {
            const TileCoord t = decode_tile<HT_H, HT_TW>(p, pair_tile(pair), BN);
            for (int kc = 0; kc < p.kchunks; ++kc) {
                mbar_wait(&empty_bar[stage], phase ^ 1u);
                if (elect_one()) {
                    if (leader) mbar_expect_tx(&full_bar[stage], 2 * region_bytes);
                    tma_load_4d_2sm(a_ring + stage * p.region_stride, &p.tmA, &full_bar[stage], kc * KCHUNK, t.w0 - p.dil,
                                    t.h0 - p.dil, t.img);
                }
                __syncwarp();
                if (++stage == NST) { stage = 0; phase ^= 1u; }
                if (!WRES) {
                    for (int tap = 0; tap < 9; ++tap) {           // this CTA's half of every (tap, chunk) weight slice
                        mbar_wait(&bempty_bar[bstage], bphase ^ 1u);
                        if (elect_one()) {
                            if (leader) mbar_expect_tx(&bfull_bar[bstage], 2 * W_TILE_BYTES);
                            tma_load_2d_2sm(w_res + bstage * W_TILE_BYTES, &p.tmB, &bfull_bar[bstage],
                                            (tap * p.kchunks + kc) * KCHUNK, t.n0 + (int)rank * (BN / 2));
                        }
                        __syncwarp();
                        if (++bstage == NBS) { bstage = 0; bphase ^= 1u; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer (leader CTA only)
        if (leader) {
            const uint32_t idesc = umma_idesc_bf16(2 * TILE_M, BN);
            const uint32_t sbo = (uint32_t)p.region_w * 128u;
            const uint32_t w_addr = smem_u32(w_res);
            const uint32_t tap_dy_bytes = (uint32_t)(p.dil * p.region_w) * 128u;
            const uint32_t tap_dx_bytes = (uint32_t)p.dil * 128u;
            int stage = 0, bstage = 0;
            uint32_t phase = 0, bphase = 0;
            int it = 0;
            if (WRES) mbar_wait(w_bar, 0);
            for (int pair = cluster_id; pair < n_pairs; pair += n_clusters, ++it) {
                const int as = it & 1;
                const uint32_t aphase = (uint32_t)(it >> 1) & 1u;
                mbar_wait(&tempty_bar[as], aphase ^ 1u);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(as * NH * BN);
                uint32_t accumulate = 0;
                for (int kc = 0; kc < p.kchunks; ++kc) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    const uint32_t region = smem_u32(a_ring + stage * p.region_stride);
                    if (WRES) {
                        const uint32_t w_chunk = w_addr + (uint32_t)(kc * W_TILE_BYTES);
                        const uint32_t w_tap_stride = (uint32_t)(p.kchunks * W_TILE_BYTES);
                        if (elect_one()) {
                            // (no tap skipping here: the two tiles of a pair may sit at different image borders;
                            //  windows in the padding read TMA's zero fill)
#pragma unroll
                            for (int tap = 0; tap < 9; ++tap) {
                                const uint32_t a_addr = region + (uint32_t)(tap / 3) * tap_dy_bytes + (uint32_t)(tap % 3) * tap_dx_bytes;
                                const uint64_t adesc = umma_desc_sw128_strided(a_addr, sbo);
                                const uint64_t bdesc = umma_desc_sw128(w_chunk + (uint32_t)tap * w_tap_stride);
#pragma unroll
                                for (int k = 0; k < KCHUNK / 16; ++k) {
#pragma unroll
                                    for (int half = 0; half < NH; ++half)
                                        umma_bf16_2sm(d_tmem + (uint32_t)(half * BN), adesc + (uint64_t)(2 * k + 64 * half),
                                                      bdesc + (uint64_t)(2 * k), idesc, accumulate);
                                    accumulate = 1;
                                }
                            }
                            umma_commit_2sm(&empty_bar[stage]);
                        }
                        __syncwarp();
                        accumulate = 1;
                    } else {
#pragma unroll 1
                        for (int tap = 0; tap < 9; ++tap) {
                            mbar_wait(&bfull_bar[bstage], bphase);
                            tc_fence_after();
                            const uint32_t a_addr = region + (uint32_t)(tap / 3) * tap_dy_bytes + (uint32_t)(tap % 3) * tap_dx_bytes;
                            const uint64_t adesc = umma_desc_sw128_strided(a_addr, sbo);
                            const uint64_t bdesc = umma_desc_sw128(w_addr + (uint32_t)(bstage * W_TILE_BYTES));
                            if (elect_one()) {
#pragma unroll
                                for (int k = 0; k < KCHUNK / 16; ++k) {
#pragma unroll
                                    for (int half = 0; half < NH; ++half)
                                        umma_bf16_2sm(d_tmem + (uint32_t)(half * BN), adesc + (uint64_t)(2 * k + 64 * half),
                                                      bdesc + (uint64_t)(2 * k), idesc, (k == 0) ? accumulate : 1u);
                                }
                                umma_commit_2sm(&bempty_bar[bstage]);
                            }
                            __syncwarp();
                            accumulate = 1;
                            if (++bstage == NBS) { bstage = 0; bphase ^= 1u; }
                        }
                        if (elect_one()) umma_commit_2sm(&empty_bar[stage]);
                        __syncwarp();
                    }
                    if (++stage == NST) { stage = 0; phase ^= 1u; }
                }
                if (elect_one()) umma_commit_2sm(&tfull_bar[as]);
                __syncwarp();
            }
        }
    } else if (warp >= EPI_WARP0) {
        run_epilogue<BN, HT_H, HT_W, NH, true>(p, warp & 3, lane, (warp - EPI_WARP0) >> 2, tmem_base, tfull_bar, tempty_bar,
                                               bias_s, stg_s);
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                 // neither CTA leaves (or frees TMEM) while the other may still signal it
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc_2sm(tmem_base, TMEM_COLS);
    }
}

// ---------------------------------------------------------------------------- upconv1 folded into dec1.0
// ConvTranspose2d(128, 64, 2, stride 2) -> cat([up, skip]) -> Conv2d(128, 64, 3, padding 1) + BN + ReLU
// (reference models/model_2.py:29, :76-77) as ONE kernel that never materialises `up`.  A 2x2/stride-2 transposed
// conv followed by a 3x3 conv is, for the output pixels of one parity class (py, px) = (y & 1, x & 1), a 2x2-tap conv
// over the HALF-resolution tensor x with composed weights (the host composes Wu with Wd in fp64 and rounds the result
// to bf16 once: model.py compose_upconv)
// -- K = 4 x 128 instead of 9 x 64 -- plus the ordinary 3x3 over the skip half sampled at stride 2.  Taps of the 3x3
// that fall outside the upsampled image contribute nothing, bias of the transposed conv included: TMA's zero fill does
// that for the data, the border-class bias of the epilogue for the bias.
//
// Tile = 16 x 8 pixels of the half-resolution grid per CTA = a 32 x 16 output patch; its four parity classes are the
// four accumulators (4 x 64 TMEM columns, double buffered = 512).  K is walked as three "chunks", each with its own
// region and barrier pair (stage == chunk):
//   chunk 0, 1: x channels [0,64) / [64,128): region (16+2) x (8+2) half-res pixels; class (py, px), tap (a, b) reads
//               the window starting at row py + a, column px + b.
//   chunk 2   : the skip tensor's 34 x 18 full-resolution pixels around the patch, loaded as two column-parity planes
//               (a 5-D tensor map splits W into (W/2, 2)) of 34 x 9 pixels: class (py, px), tap (ky, kx) reads the
//               window starting at row py + ky with 8-row groups TWO region rows apart (SBO), in plane (px + kx) & 1,
//               column (px + kx) >> 1.
// Shared windows.  An N = 64 MMA reads A 4 KB + B 1 KB of shared memory per 32 tensor cycles (160 B/cycle against the
// 128 the MMA unit gets): that bounds the ordinary N = 64 layers at 74 % tensor.  Here the window only depends on
// (py + a, px + b) resp. (py + ky, px + kx), so several classes read the SAME window -- with different weights into
// ADJACENT accumulators -- and run as one MMA of N = 128 (classes 0,1 or 2,3) or N = 256 (all four) whose B operand is
// the classes' weight tiles stacked; the accumulators sit in Gray order (slot s = class s ^ (s >> 1)) so that three of
// the four class pairings are adjacent: 10 MMAs instead of 16 per K = 16 step of an x chunk, 18 instead of 36 for the
// skip chunk, same tensor cycles, A reads 40 / 72 KB instead of 64 / 144 KB.  The schedule is the table below; the
// host packs the weights in exactly this order (dc_debug_upfuse_schedule), per CTA of the pair (a pair MMA takes rows
// [0, N/2) of B from the leader and [N/2, N) from the peer), and they stream through a ring of 16 KB groups (= 512
// tensor cycles each; within a group the MMAs go to different accumulators, so no chain waits for itself).
// Roles as conv_halo2_kernel plus warp 3 = producer of the weight ring (region loads never queue behind weights).
constexpr int UPF_U_W = HT_W + 2, UPF_U_H = HT_H + 2;
constexpr int UPF_U_BYTES = UPF_U_W * UPF_U_H * 128;                 // 23,040
constexpr int UPF_S_W = HT_W + 1, UPF_S_H = 2 * HT_H + 2;
constexpr int UPF_PLANE_BYTES = UPF_S_W * UPF_S_H * 128;             // 39,168
constexpr int UPF_GROUP_ROWS = 128;                                  // weight rows per CTA and ring slot (16 KB)
constexpr int UPF_GROUP_BYTES = UPF_GROUP_ROWS * 128;
constexpr int UPF_RING = 5;
constexpr int UPF_BIAS_BYTES = 256;
constexpr size_t UPF_SMEM = UPF_RING * UPF_GROUP_BYTES + 2 * UPF_U_BYTES + 2 * UPF_PLANE_BYTES + 1024 + HALO_BAR_BYTES +
                            UPF_BIAS_BYTES + EPI_STAGE_TOTAL;
static_assert(UPF_SMEM <= 227 * 1024, "conv_upfused2_kernel: shared memory");

// upf_schedule.inc defines, host side, upf_u_op(i) / upf_s_op(i) = MMA i of one K = 16 step of an x chunk / the skip
// chunk and upf_u_count() / upf_s_count(); device side, the specialisations of upf_issue_group below.
// upf_issue_group<KIND, G> issues the 4 x (MMAs of group G) of chunk kind KIND (0 = x, 1 = skip); d = accumulator base,
// a = descriptor of the region's first row, b = descriptor of the group's ring slot; fresh = overwrite at the tile's
// first K step
template <int KIND, int G>
__device__ __forceinline__ void upf_issue_group(uint32_t d, uint64_t a, uint64_t b, bool fresh);
#include "upf_schedule.inc"
constexpr int UPF_GROUPS_PER_TILE = 2 * 4 + 9;
constexpr int UPF_ROWS_PER_RANK = UPF_GROUPS_PER_TILE * UPF_GROUP_ROWS;      // 2176 weight rows per CTA of the pair

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
conv_upfused2_kernel(const __grid_constant__ ConvParams p) {
    constexpr int BN = 64;
    constexpr int TMEM_COLS = 512;

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* w_ring = smem;                                          // UPF_RING groups of 128 weight rows
    uint8_t* u_reg = w_ring + UPF_RING * UPF_GROUP_BYTES;            // x regions of chunk 0, 1
    uint8_t* s_reg = u_reg + 2 * UPF_U_BYTES;                        // skip planes: [0] odd columns (from 2 w0 - 1), [1] even
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(s_reg + 2 * UPF_PLANE_BYTES);
    uint64_t* empty_bar = full_bar + HALO_MAX_STAGES;
    uint64_t* bfull_bar = empty_bar + HALO_MAX_STAGES;
    uint64_t* bempty_bar = bfull_bar + HALO_MAX_STAGES;
    uint64_t* tfull_bar = bempty_bar + HALO_MAX_STAGES;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
    float* bias_s = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full_bar) + HALO_BAR_BYTES);
    uint8_t* stg_s = reinterpret_cast<uint8_t*>(full_bar) + HALO_BAR_BYTES + UPF_BIAS_BYTES;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;
    const int cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;
    const int n_pairs = pair_count(p);

    stage_bias(p, bias_s);
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&p.tmA);
        tma_prefetch_desc(&p.tmB);
        tma_prefetch_desc(&p.tmS);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < HALO_MAX_STAGES; ++s) {
            mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1);
            mbar_init(&bfull_bar[s], 1); mbar_init(&bempty_bar[s], 1);
        }
        for (int s = 0; s < 2; ++s) { mbar_init(&tfull_bar[s], 1); mbar_init(&tempty_bar[s], 8 * EPI_GROUPS); }
        fence_barrier_init();
    }
    if (warp == 2) {
        tmem_alloc_2sm(tmem_slot, TMEM_COLS);
        tmem_relinquish_2sm();
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ------------------------------------------------------------------ region producer (one per CTA)
        int it = 0;
        for (int pair = cluster_id; pair < n_pairs; pair += n_clusters, ++it) {
            const TileCoord t = decode_tile<HT_H, HT_W>(p, pair_to_tile(p, pair, (int)rank), BN);
            const uint32_t ph = (uint32_t)it & 1u;
            for (int kc = 0; kc < 2; ++kc) {
                mbar_wait(&empty_bar[kc], ph ^ 1u);
                if (elect_one()) {
                    if (leader) mbar_expect_tx(&full_bar[kc], 2u * UPF_U_BYTES);
                    tma_load_4d_2sm(u_reg + kc * UPF_U_BYTES, &p.tmA, &full_bar[kc], kc * KCHUNK, t.w0 - 1, t.h0 - 1, t.img);
                }
                __syncwarp();
            }
            mbar_wait(&empty_bar[2], ph ^ 1u);
            if (elect_one()) {
                if (leader) mbar_expect_tx(&full_bar[2], 4u * UPF_PLANE_BYTES);
                // W is split into (W/2, parity): odd columns 2 w0 - 1, 2 w0 + 1, ... = (parity 1, from w0 - 1)
                tma_load_5d_2sm(s_reg, &p.tmS, &full_bar[2], 0, 1, t.w0 - 1, 2 * t.h0 - 1, t.img);
                tma_load_5d_2sm(s_reg + UPF_PLANE_BYTES, &p.tmS, &full_bar[2], 0, 0, t.w0, 2 * t.h0 - 1, t.img);
            }
            __syncwarp();
        }
    } else if (warp == 3) {
        // ------------------------------------------------------------------ weight producer (one per CTA)
        int bg = 0;
        uint32_t bphase = 0;
        for (int pair = cluster_id; pair < n_pairs; pair += n_clusters) {
            for (int g = 0; g < UPF_GROUPS_PER_TILE; ++g) {
                mbar_wait(&bempty_bar[bg], bphase ^ 1u);
                if (elect_one()) {
                    if (leader) mbar_expect_tx(&bfull_bar[bg], 2u * UPF_GROUP_BYTES);
                    tma_load_2d_2sm(w_ring + bg * UPF_GROUP_BYTES, &p.tmB, &bfull_bar[bg], 0,
                                    (int)rank * UPF_ROWS_PER_RANK + g * UPF_GROUP_ROWS);
                }
                __syncwarp();
                if (++bg == UPF_RING) { bg = 0; bphase ^= 1u; }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer (leader CTA only)
        if (leader) {
            // Descriptors are base + constant: the address field is (addr & 0x3FFFF) >> 4 and every operand lies below
            // 256 KB, so desc(addr + off) == desc(addr) + (off >> 4) and each MMA costs two 64-bit adds, not a rebuild
            // (with the mask in the way the compiler rebuilt every descriptor: 38 uniform-datapath instructions per
            // MMA, and the issuing warp -- not the tensor pipe -- set the pace).
            const uint64_t adesc_u = umma_desc_sw128_strided(smem_u32(u_reg), UPF_U_W * 128u);
            const uint64_t adesc_s = umma_desc_sw128_strided(smem_u32(s_reg), 2u * UPF_S_W * 128u);
            const uint64_t bdesc_ring = umma_desc_sw128(smem_u32(w_ring));
            int bg = 0;
            uint32_t bphase = 0;
            int it = 0;
            for (int pair = cluster_id; pair < n_pairs; pair += n_clusters, ++it) {
                const int as = it & 1;
                const uint32_t aphase = (uint32_t)(it >> 1) & 1u;
                const uint32_t ph = (uint32_t)it & 1u;
                mbar_wait(&tempty_bar[as], aphase ^ 1u);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(as * 4 * BN);
#define DC_UPF_GROUP(KIND, G, ADESC, FRESH)                                                                         \
    {                                                                                                               \
        mbar_wait(&bfull_bar[bg], bphase);                                                                          \
        tc_fence_after();                                                                                           \
        if (elect_one()) {                                                                                          \
            upf_issue_group<KIND, G>(d_tmem, ADESC, bdesc_ring + (uint64_t)(bg * (UPF_GROUP_BYTES >> 4)), FRESH);       \
            umma_commit_2sm(&bempty_bar[bg]);                                                                       \
        }                                                                                                           \
        __syncwarp();                                                                                               \
        if (++bg == UPF_RING) { bg = 0; bphase ^= 1u; }                                                             \
    }
#pragma unroll 1
                for (int kc = 0; kc < 2; ++kc) {
                    mbar_wait(&full_bar[kc], ph);
                    tc_fence_after();
                    const uint64_t areg = adesc_u + (uint64_t)(kc * (UPF_U_BYTES >> 4));
                    DC_UPF_GROUP(0, 0, areg, kc == 0) DC_UPF_GROUP(0, 1, areg, kc == 0)
                    DC_UPF_GROUP(0, 2, areg, kc == 0) DC_UPF_GROUP(0, 3, areg, kc == 0)
                    if (elect_one()) umma_commit_2sm(&empty_bar[kc]);
                    __syncwarp();
                }
                mbar_wait(&full_bar[2], ph);
                tc_fence_after();
                DC_UPF_GROUP(1, 0, adesc_s, false) DC_UPF_GROUP(1, 1, adesc_s, false) DC_UPF_GROUP(1, 2, adesc_s, false)
                DC_UPF_GROUP(1, 3, adesc_s, false) DC_UPF_GROUP(1, 4, adesc_s, false) DC_UPF_GROUP(1, 5, adesc_s, false)
                DC_UPF_GROUP(1, 6, adesc_s, false) DC_UPF_GROUP(1, 7, adesc_s, false) DC_UPF_GROUP(1, 8, adesc_s, false)
#undef DC_UPF_GROUP
                if (elect_one()) {
                    umma_commit_2sm(&empty_bar[2]);
                    umma_commit_2sm(&tfull_bar[as]);
                }
                __syncwarp();
            }
        }
    } else if (warp >= EPI_WARP0) {
        run_epilogue<BN, HT_H, HT_W, 4, true, true, true>(p, warp & 3, lane, (warp - EPI_WARP0) >> 2, tmem_base, tfull_bar, tempty_bar,
                                                          bias_s, stg_s);
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc_2sm(tmem_base, TMEM_COLS);
    }
}

// ---------------------------------------------------------------------------- upconv{2,3,4} folded into dec{2,3,4}.0
// The composition of conv_upfused2_kernel for Cout = 128 / 256 / 512, where the four parity classes of a tile no longer
// fit TMEM at once (4 x BN x 2 stages): a tile is walked in PASSES of NCLS = 256 / BN classes (BN = 128: the two
// classes of one output-row parity; BN = 256: one class), each pass a full K loop into NCLS accumulators, and the pass
// index rides in the n-tile index (p.n_tiles = class groups x real n-tiles), so the tile / pair / epilogue machinery
// is the ordinary one.  These layers are tensor-bound at N >= 128, so no window sharing: one MMA per (class, tap).
// K order per pass: [x chunk, x chunk, skip chunk] x (C / 64) -- Cx = 2 C, so the two x chunks between consecutive
// skip chunks (4096 tensor cycles) cover the load of the single 78 KB skip slot; x chunks rotate through three 23 KB
// slots.  Weights stream through a ring of three 16 KB slots, each worth 512 tensor cycles: an x slot holds the
// (chunk, tap) tiles of the pass's NCLS classes (NCLS x BN/2 rows per CTA), a skip slot one (chunk, tap) tile shared by
// the classes (BN/2 rows).
constexpr int UPW_XSLOTS = 2;
constexpr int UPW_RING = 5;
constexpr int UPW_BIAS_BYTES = 2048;
constexpr size_t UPW_SMEM = UPW_RING * UPF_GROUP_BYTES + UPW_XSLOTS * UPF_U_BYTES + 2 * UPF_PLANE_BYTES + 1024 + HALO_BAR_BYTES +
                            UPW_BIAS_BYTES + EPI_STAGE_TOTAL;
static_assert(UPW_SMEM <= 227 * 1024, "conv_upfused_wide_kernel: shared memory");

template <int BN>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
conv_upfused_wide_kernel(const __grid_constant__ ConvParams p) {
    constexpr int NCLS = 256 / BN;                       // classes per pass
    constexpr int TMEM_COLS = 512;
    constexpr int SKIP_TILE_BYTES = (BN / 2) * 128;      // one (chunk, tap) skip tile per CTA

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* w_ring = smem;
    uint8_t* x_reg = w_ring + UPW_RING * UPF_GROUP_BYTES;
    uint8_t* s_reg = x_reg + UPW_XSLOTS * UPF_U_BYTES;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(s_reg + 2 * UPF_PLANE_BYTES);      // [0..2] x slots, [3] the skip slot
    uint64_t* empty_bar = full_bar + HALO_MAX_STAGES;
    uint64_t* bfull_bar = empty_bar + HALO_MAX_STAGES;
    uint64_t* bempty_bar = bfull_bar + HALO_MAX_STAGES;
    uint64_t* tfull_bar = bempty_bar + HALO_MAX_STAGES;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
    float* bias_s = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full_bar) + HALO_BAR_BYTES);
    uint8_t* stg_s = reinterpret_cast<uint8_t*>(full_bar) + HALO_BAR_BYTES + UPW_BIAS_BYTES;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;
    const int cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;
    const int n_pairs = pair_count(p);
    const int SC = p.kchunks;                            // skip chunks; x chunks = 2 * SC

    stage_bias(p, bias_s);
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&p.tmA);
        tma_prefetch_desc(&p.tmB);
        tma_prefetch_desc(&p.tmB2);
        tma_prefetch_desc(&p.tmS);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < HALO_MAX_STAGES; ++s) {
            mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1);
            mbar_init(&bfull_bar[s], 1); mbar_init(&bempty_bar[s], 1);
        }
        for (int s = 0; s < 2; ++s) { mbar_init(&tfull_bar[s], 1); mbar_init(&tempty_bar[s], 8 * EPI_GROUPS); }
        fence_barrier_init();
    }
    if (warp == 2) {
        tmem_alloc_2sm(tmem_slot, TMEM_COLS);
        tmem_relinquish_2sm();
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ------------------------------------------------------------------ region producer (one per CTA)
        int xs = 0;
        uint32_t xph = 0, sph = 0;
        for (int pair = cluster_id; pair < n_pairs; pair += n_clusters) {
            const TileCoord t = decode_tile<HT_H, HT_W>(p, pair_to_tile(p, pair, (int)rank), BN);
            for (int g = 0; g < SC; ++g) {
                for (int r = 0; r < 2; ++r) {
                    mbar_wait(&empty_bar[xs], xph ^ 1u);
                    if (elect_one()) {
                        if (leader) mbar_expect_tx(&full_bar[xs], 2u * UPF_U_BYTES);
                        tma_load_4d_2sm(x_reg + xs * UPF_U_BYTES, &p.tmA, &full_bar[xs], (2 * g + r) * KCHUNK, t.w0 - 1, t.h0 - 1, t.img);
                    }
                    __syncwarp();
                    if (++xs == UPW_XSLOTS) { xs = 0; xph ^= 1u; }
                }
                mbar_wait(&empty_bar[3], sph ^ 1u);
                if (elect_one()) {
                    if (leader) mbar_expect_tx(&full_bar[3], 4u * UPF_PLANE_BYTES);
                    tma_load_5d_2sm(s_reg, &p.tmS, &full_bar[3], g * KCHUNK, 1, t.w0 - 1, 2 * t.h0 - 1, t.img);
                    tma_load_5d_2sm(s_reg + UPF_PLANE_BYTES, &p.tmS, &full_bar[3], g * KCHUNK, 0, t.w0, 2 * t.h0 - 1, t.img);
                }
                __syncwarp();
                sph ^= 1u;
            }
        }
    } else if (warp == 3) {
        // ------------------------------------------------------------------ weight producer (one per CTA)
        // x tiles: [class group][n-tile][CTA][x chunk][tap][NCLS x BN/2 rows]; skip tiles: [n-tile][CTA][chunk][tap][BN/2 rows]
        int bg = 0;
        uint32_t bphase = 0;
        for (int pair = cluster_id; pair < n_pairs; pair += n_clusters) {
            const int nt_eff = pair - fast_div(pair, p.fd_ntiles) * p.n_tiles;       // class group * real n-tiles + n-tile
            const int nt = nt_eff % p.real_ntiles;
            const int xrow0 = ((nt_eff * 2 + (int)rank) * 2 * SC) * 4 * UPF_GROUP_ROWS;
            const int srow0 = ((nt * 2 + (int)rank) * SC) * 9 * (BN / 2);
            for (int g = 0; g < SC; ++g) {
                for (int j = 0; j < 8; ++j) {                     // x chunk 2 g + (j >> 2), tap j & 3
                    mbar_wait(&bempty_bar[bg], bphase ^ 1u);
                    if (elect_one()) {
                        if (leader) mbar_expect_tx(&bfull_bar[bg], 2u * UPF_GROUP_BYTES);
                        tma_load_2d_2sm(w_ring + bg * UPF_GROUP_BYTES, &p.tmB, &bfull_bar[bg], 0, xrow0 + (g * 8 + j) * UPF_GROUP_ROWS);
                    }
                    __syncwarp();
                    if (++bg == UPW_RING) { bg = 0; bphase ^= 1u; }
                }
                for (int tap = 0; tap < 9; ++tap) {
                    mbar_wait(&bempty_bar[bg], bphase ^ 1u);
                    if (elect_one()) {
                        if (leader) mbar_expect_tx(&bfull_bar[bg], 2u * SKIP_TILE_BYTES);
                        tma_load_2d_2sm(w_ring + bg * UPF_GROUP_BYTES, &p.tmB2, &bfull_bar[bg], 0, srow0 + (g * 9 + tap) * (BN / 2));
                    }
                    __syncwarp();
                    if (++bg == UPW_RING) { bg = 0; bphase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer (leader CTA only)
        if (leader) {
            const uint32_t idesc = umma_idesc_bf16(2 * TILE_M, BN);
            const uint64_t adesc_x = umma_desc_sw128_strided(smem_u32(x_reg), UPF_U_W * 128u);
            const uint64_t adesc_s = umma_desc_sw128_strided(smem_u32(s_reg), 2u * UPF_S_W * 128u);
            const uint64_t bdesc_ring = umma_desc_sw128(smem_u32(w_ring));
            int bg = 0, xs = 0;
            uint32_t bphase = 0, xph = 0, sph = 0;
            int it = 0;
            for (int pair = cluster_id; pair < n_pairs; pair += n_clusters, ++it) {
                const int as = it & 1;
                const uint32_t aphase = (uint32_t)(it >> 1) & 1u;
                const int nt_eff = pair - fast_div(pair, p.fd_ntiles) * p.n_tiles;
                const int cls_base = (nt_eff / p.real_ntiles) * NCLS;
                // descriptor offsets (16-byte units) of class `half`'s windows relative to tap (0, 0)
                uint32_t xoff[NCLS], soff_row[NCLS];
                int spx[NCLS];
#pragma unroll
                for (int half = 0; half < NCLS; ++half) {
                    const int py = (cls_base + half) >> 1, px = (cls_base + half) & 1;
                    xoff[half] = (uint32_t)((py * UPF_U_W + px) * 8);
                    soff_row[half] = (uint32_t)(py * UPF_S_W * 8);
                    spx[half] = px;
                }
                mbar_wait(&tempty_bar[as], aphase ^ 1u);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(as * NCLS * BN);
                uint32_t accumulate = 0;
#pragma unroll 1
                for (int g = 0; g < SC; ++g) {
#pragma unroll 1
                    for (int r = 0; r < 2; ++r) {
                        mbar_wait(&full_bar[xs], xph);
                        tc_fence_after();
                        const uint64_t areg = adesc_x + (uint64_t)(xs * (UPF_U_BYTES >> 4));
#pragma unroll
                        for (int tap = 0; tap < 4; ++tap) {
                            mbar_wait(&bfull_bar[bg], bphase);
                            tc_fence_after();
                            const uint64_t wg = bdesc_ring + (uint64_t)(bg * (UPF_GROUP_BYTES >> 4));
                            if (elect_one()) {
#pragma unroll
                                for (int k = 0; k < KCHUNK / 16; ++k) {
#pragma unroll
                                    for (int half = 0; half < NCLS; ++half)
                                        umma_bf16_2sm(d_tmem + (uint32_t)(half * BN),
                                                      areg + (uint64_t)(xoff[half] + (uint32_t)(((tap >> 1) * UPF_U_W + (tap & 1)) * 8 + 2 * k)),
                                                      wg + (uint64_t)(half * (BN / 2) * 8 + 2 * k), idesc, (k == 0) ? accumulate : 1u);
                                }
                                umma_commit_2sm(&bempty_bar[bg]);
                            }
                            __syncwarp();
                            accumulate = 1;
                            if (++bg == UPW_RING) { bg = 0; bphase ^= 1u; }
                        }
                        if (elect_one()) umma_commit_2sm(&empty_bar[xs]);
                        __syncwarp();
                        if (++xs == UPW_XSLOTS) { xs = 0; xph ^= 1u; }
                    }
                    mbar_wait(&full_bar[3], sph);
                    tc_fence_after();
#pragma unroll
                    for (int tap = 0; tap < 9; ++tap) {
                        mbar_wait(&bfull_bar[bg], bphase);
                        tc_fence_after();
                        const uint64_t wg = bdesc_ring + (uint64_t)(bg * (UPF_GROUP_BYTES >> 4));
                        if (elect_one()) {
#pragma unroll
                            for (int k = 0; k < KCHUNK / 16; ++k) {
#pragma unroll
                                for (int half = 0; half < NCLS; ++half) {
                                    const int cx = spx[half] + tap % 3;
                                    const uint32_t off = (uint32_t)((cx & 1) * (UPF_PLANE_BYTES >> 4) + ((tap / 3) * UPF_S_W + (cx >> 1)) * 8) + soff_row[half];
                                    umma_bf16_2sm(d_tmem + (uint32_t)(half * BN), adesc_s + (uint64_t)(off + (uint32_t)(2 * k)), wg + (uint64_t)(2 * k), idesc, 1u);
                                }
                            }
                            umma_commit_2sm(&bempty_bar[bg]);
                        }
                        __syncwarp();
                        if (++bg == UPW_RING) { bg = 0; bphase ^= 1u; }
                    }
                    if (elect_one()) umma_commit_2sm(&empty_bar[3]);
                    __syncwarp();
                    sph ^= 1u;
                }
                if (elect_one()) umma_commit_2sm(&tfull_bar[as]);
                __syncwarp();
            }
        }
    } else if (warp >= EPI_WARP0) {
        run_epilogue<BN, HT_H, HT_W, NCLS, true, true, true>(p, warp & 3, lane, (warp - EPI_WARP0) >> 2, tmem_base, tfull_bar, tempty_bar,
                                                             bias_s, stg_s);
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc_2sm(tmem_base, TMEM_COLS);
    }
}

// ---------------------------------------------------------------------------- 64 -> 64 channel 3x3 layers by parity class
// The skip chunk of conv_upfused2_kernel on its own is a plain Conv2d(64, 64, 3, padding 1) computed per output parity
// class: enc1.3 and dec1.3 (models/model_2.py:10, :30) run through it.  Same windows, same shared-window MMA schedule
// (chunk kind 2 of upf_schedule.inc), i.e. A reads 80 KB instead of 144 KB per K = 16 step -- these layers sat at
// 74 % tensor with the MMA unit's shared-memory reads at 90 % in the 4-strip kernel (conv_halo2_kernel<64, 4>).
// Two region stages (the next tile's planes load during this tile's MMAs), weights through a ring of 3 groups.
// Epilogues: STORE, STORE_POOL (the four classes of a lane ARE the 2x2 pooling window: the max is taken in registers)
// and HEAD.
constexpr int PAR_RING = 3;
constexpr int PAR_STAGES = 2;
constexpr int PAR_BIAS_BYTES = 1024;                                  // bias + out_conv weights (HEAD)
constexpr int PAR_ROWS_PER_RANK = 9 * UPF_GROUP_ROWS;                 // 1152 weight rows per CTA of the pair
constexpr size_t PAR_SMEM = PAR_RING * UPF_GROUP_BYTES + PAR_STAGES * 2 * UPF_PLANE_BYTES + 1024 + HALO_BAR_BYTES +
                            PAR_BIAS_BYTES + EPI_STAGE_TOTAL;
static_assert(PAR_SMEM <= 227 * 1024, "conv_par2_kernel: shared memory");

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
conv_par2_kernel(const __grid_constant__ ConvParams p) {
    constexpr int BN = 64;
    constexpr int TMEM_COLS = 512;
    constexpr int STAGE_BYTES = 2 * UPF_PLANE_BYTES;

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* w_ring = smem;
    uint8_t* s_reg = w_ring + PAR_RING * UPF_GROUP_BYTES;            // PAR_STAGES x {odd-column plane, even-column plane}
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(s_reg + PAR_STAGES * STAGE_BYTES);
    uint64_t* empty_bar = full_bar + HALO_MAX_STAGES;
    uint64_t* bfull_bar = empty_bar + HALO_MAX_STAGES;
    uint64_t* bempty_bar = bfull_bar + HALO_MAX_STAGES;
    uint64_t* tfull_bar = bempty_bar + HALO_MAX_STAGES;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
    float* bias_s = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full_bar) + HALO_BAR_BYTES);
    uint8_t* stg_s = reinterpret_cast<uint8_t*>(full_bar) + HALO_BAR_BYTES + PAR_BIAS_BYTES;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;
    const int cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;
    const int n_pairs = pair_count(p);

    stage_bias(p, bias_s);
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&p.tmB);
        tma_prefetch_desc(&p.tmS);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < HALO_MAX_STAGES; ++s) {
            mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1);
            mbar_init(&bfull_bar[s], 1); mbar_init(&bempty_bar[s], 1);
        }
        for (int s = 0; s < 2; ++s) { mbar_init(&tfull_bar[s], 1); mbar_init(&tempty_bar[s], 8 * EPI_GROUPS); }
        fence_barrier_init();
    }
    if (warp == 2) {
        tmem_alloc_2sm(tmem_slot, TMEM_COLS);
        tmem_relinquish_2sm();
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ------------------------------------------------------------------ region producer (one per CTA)
        int it = 0;
        for (int pair = cluster_id; pair < n_pairs; pair += n_clusters, ++it) {
            const TileCoord t = decode_tile<HT_H, HT_W>(p, pair_to_tile(p, pair, (int)rank), BN);
            const int st = it & 1;
            mbar_wait(&empty_bar[st], (((uint32_t)it >> 1) & 1u) ^ 1u);
            if (elect_one()) {
                if (leader) mbar_expect_tx(&full_bar[st], 2u * STAGE_BYTES);
                tma_load_5d_2sm(s_reg + st * STAGE_BYTES, &p.tmS, &full_bar[st], 0, 1, t.w0 - 1, 2 * t.h0 - 1, t.img);
                tma_load_5d_2sm(s_reg + st * STAGE_BYTES + UPF_PLANE_BYTES, &p.tmS, &full_bar[st], 0, 0, t.w0, 2 * t.h0 - 1, t.img);
            }
            __syncwarp();
        }
    } else if (warp == 3) {
        // ------------------------------------------------------------------ weight producer (one per CTA)
        int bg = 0;
        uint32_t bphase = 0;
        for (int pair = cluster_id; pair < n_pairs; pair += n_clusters) {
            for (int g = 0; g < 9; ++g) {
                mbar_wait(&bempty_bar[bg], bphase ^ 1u);
                if (elect_one()) {
                    if (leader) mbar_expect_tx(&bfull_bar[bg], 2u * UPF_GROUP_BYTES);
                    tma_load_2d_2sm(w_ring + bg * UPF_GROUP_BYTES, &p.tmB, &bfull_bar[bg], 0,
                                    (int)rank * PAR_ROWS_PER_RANK + g * UPF_GROUP_ROWS);
                }
                __syncwarp();
                if (++bg == PAR_RING) { bg = 0; bphase ^= 1u; }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer (leader CTA only)
        if (leader) {
            const uint64_t adesc_s = umma_desc_sw128_strided(smem_u32(s_reg), 2u * UPF_S_W * 128u);
            const uint64_t bdesc_ring = umma_desc_sw128(smem_u32(w_ring));
            int bg = 0;
            uint32_t bphase = 0;
            int it = 0;
            for (int pair = cluster_id; pair < n_pairs; pair += n_clusters, ++it) {
                const int as = it & 1;
                const uint32_t aphase = (uint32_t)(it >> 1) & 1u;
                mbar_wait(&tempty_bar[as], aphase ^ 1u);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(as * 4 * BN);
                mbar_wait(&full_bar[as], aphase);                 // region stage == accumulator stage == it & 1
                tc_fence_after();
                const uint64_t areg = adesc_s + (uint64_t)(as * (STAGE_BYTES >> 4));
#define DC_PAR_GROUP(G)                                                                                             \
    {                                                                                                               \
        mbar_wait(&bfull_bar[bg], bphase);                                                                          \
        tc_fence_after();                                                                                           \
        if (elect_one()) {                                                                                          \
            upf_issue_group<2, G>(d_tmem, areg, bdesc_ring + (uint64_t)(bg * (UPF_GROUP_BYTES >> 4)), true);        \
            umma_commit_2sm(&bempty_bar[bg]);                                                                       \
        }                                                                                                           \
        __syncwarp();                                                                                               \
        if (++bg == PAR_RING) { bg = 0; bphase ^= 1u; }                                                             \
    }
                DC_PAR_GROUP(0) DC_PAR_GROUP(1) DC_PAR_GROUP(2) DC_PAR_GROUP(3) DC_PAR_GROUP(4)
                DC_PAR_GROUP(5) DC_PAR_GROUP(6) DC_PAR_GROUP(7) DC_PAR_GROUP(8)
#undef DC_PAR_GROUP
                if (elect_one()) {
                    umma_commit_2sm(&empty_bar[as]);
                    umma_commit_2sm(&tfull_bar[as]);
                }
                __syncwarp();
            }
        }
    } else if (warp >= EPI_WARP0) {
        run_epilogue<BN, HT_H, HT_W, 4, true, true, true>(p, warp & 3, lane, (warp - EPI_WARP0) >> 2, tmem_base, tfull_bar, tempty_bar,
                                                          bias_s, stg_s);
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc_2sm(tmem_base, TMEM_COLS);
    }
}

// ---------------------------------------------------------------------------- stem on tensor cores
// First layer, Conv2d(3, 64, 3, padding=d, dilation=d) + BN + ReLU (reference models/model_2.py:10, :41-46),
// fused with the input conversion of quantify_droplets_batch.py:45-46 (u8 -> /255 -> NCHW float).
// K = 27 is far too thin for TMA boxes, so four producer warps build the im2col tile themselves, straight
// into the 128B-swizzled K-major layout the MMA reads:
//   u8 inputs are exact in bf16 (0..255) and the 1/255 is folded into the bf16 weights;
//   grayscale input (the reference replicates it to 3 identical channels, qdb:41) folds the three channel
//   weights into one, K = 9 -> one K=16 MMA per 128-pixel tile; RGB / float input: K = 27 -> two MMAs.
// Roles (416 threads): warps 0-7 two epilogue groups, warps 8-11 im2col producers, warp 12 MMA + TMEM.
constexpr int STEM_THREADS = 416;
constexpr int STEM_PROD0 = 256;          // first producer thread
constexpr int STEM_STAGES = 4;

struct alignas(64) StemParams {
    ConvParams c;            // epilogue fields (bias, out, strides, tiles); c.tmA = tensor map of the OUTPUT (TMA stores)
    const void* in;
    const float* weight;     // fp32 [64][27] = (co, ci*9 + ky*3 + kx), BatchNorm folded
    int in_kind;
};

// Raw tap value (u8 as an integer, or the float's bits): converted only when the tile is packed, so the
// prefetched loads of the next tile stay in flight instead of stalling on an early int->float conversion.
template <int IN_KIND>
__device__ __forceinline__ uint32_t stem_px_raw(const void* in, int img, int c, int y, int x, int H, int W) {
    if (y < 0 || y >= H || x < 0 || x >= W) return 0u;                        // zero padding (0 and 0.0f)
    if (IN_KIND == 0) return __float_as_uint(reinterpret_cast<const float*>(in)[(((size_t)img * 3 + c) * H + y) * W + x]);
    if (IN_KIND == 1) return reinterpret_cast<const uint8_t*>(in)[((size_t)img * H + y) * W + x];
    return reinterpret_cast<const uint8_t*>(in)[(((size_t)img * H + y) * W + x) * 3 + c];
}
template <int IN_KIND>
__device__ __forceinline__ float stem_val(uint32_t raw) {
    return IN_KIND == 0 ? __uint_as_float(raw) : (float)raw;
}

// Epilogue of the stem: the layer is nothing but stores (K = 16 of arithmetic per 64 output channels), and the
// register -> shared -> register -> st.global transpose of run_epilogue kept the LSU pipe at 68 % with DRAM at 51 %.
// Here a warp writes its 32 pixels x 32 channels chunk ONCE into a 64B-swizzled shared tile (conflict-free 16-byte
// stores) and one lane hands it to the TMA engine (cp.async.bulk.tensor store, out-of-image pixels clipped by the
// hardware); four tiles per warp are in flight, so the next chunk never waits for the previous store to drain.
constexpr int STEM_STORE_DEPTH = 4;
constexpr int STEM_STG_BYTES = 8 * STEM_STORE_DEPTH * EPI_STAGE_BYTES;       // 8 epilogue warps

__device__ __forceinline__ void tma_store_4d(const void* tmap, const void* src, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ void stem_epilogue_tma(const ConvParams& p, const int e, const int lane, const int group,
                                                  const uint32_t tmem_base, uint64_t* tfull_bar, uint64_t* tempty_bar,
                                                  const float* bias_s, uint8_t* stg_all) {
    constexpr int BN = 64;
    uint8_t* ring = stg_all + (group * 4 + e) * (STEM_STORE_DEPTH * EPI_STAGE_BYTES);
    // this lane's pixel is row `lane` of the warp's [2 rows][16 px][32 ch] box: 64-byte rows, 16-byte chunk q of row r
    // sits at chunk q ^ ((r >> 1) & 3) (CU_TENSOR_MAP_SWIZZLE_64B: address bits [4,6) ^= bits [7,9))
    const uint32_t row_off = (uint32_t)lane * 64u, sw = ((uint32_t)lane >> 1) & 3u;
    int n = 0;                                               // chunks this warp has stored
    for (int it = group;; it += EPI_GROUPS) {                // groups take alternate tiles, group g owns TMEM stage g
        const int tile = blockIdx.x + it * gridDim.x;
        if (tile >= p.total_tiles) break;
        const TileCoord t = decode_tile(p, tile, BN);
        const int as = it & 1;
        const uint32_t aphase = (uint32_t)(it >> 1) & 1u;
        mbar_wait(&tfull_bar[as], aphase);
        tc_fence_after();
        const uint32_t tstage = tmem_base + ((uint32_t)(e * 32) << 16) + (uint32_t)(as * BN);
        uint32_t vbuf[2][32];
        tmem_ld32(tstage, vbuf[0]);
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            uint32_t* v = vbuf[c];
            tmem_ld_wait_on(v);
            if (c == 0) tmem_ld32(tstage + 32u, vbuf[1]);
            else release_accumulator<false>(&tempty_bar[as], lane);
            uint32_t pk[16];
            if (p.bias_const) {
                if (c == 0) {
#pragma unroll
                    for (int k = 0; k < 16; ++k)
                        pk[k] = pack_bf16_relu(__uint_as_float(v[2 * k]) + p.bias_c[2 * k], __uint_as_float(v[2 * k + 1]) + p.bias_c[2 * k + 1]);
                } else {
#pragma unroll
                    for (int k = 0; k < 16; ++k)
                        pk[k] = pack_bf16_relu(__uint_as_float(v[2 * k]) + p.bias_c[32 + 2 * k], __uint_as_float(v[2 * k + 1]) + p.bias_c[32 + 2 * k + 1]);
                }
            } else {
#pragma unroll
                for (int k = 0; k < 16; ++k)
                    pk[k] = pack_bf16_relu(__uint_as_float(v[2 * k]) + bias_s[c * 32 + 2 * k], __uint_as_float(v[2 * k + 1]) + bias_s[c * 32 + 2 * k + 1]);
            }
            uint8_t* buf = ring + (n % STEM_STORE_DEPTH) * EPI_STAGE_BYTES;
            if (n >= STEM_STORE_DEPTH) {                      // the store that last used this tile has read it
                if (lane == 0) bulk_wait_read<STEM_STORE_DEPTH - 1>();
                __syncwarp();
            }
#pragma unroll
            for (int q = 0; q < 4; ++q)
                *reinterpret_cast<uint4*>(buf + row_off + ((q ^ sw) << 4)) = make_uint4(pk[4 * q], pk[4 * q + 1], pk[4 * q + 2], pk[4 * q + 3]);
            fence_proxy_async();                              // generic-proxy writes -> visible to the TMA engine
            __syncwarp();
            if (lane == 0) {
                tma_store_4d(&p.tmA, buf, p.out_offset + c * 32, t.w0, t.h0 + 2 * e, t.img);
                bulk_commit();
            }
            ++n;
        }
    }
    if (lane == 0) bulk_wait_all();                           // shared memory must outlive the stores
}

template <int IN_KIND>
__global__ void __launch_bounds__(STEM_THREADS, 1) stem_tc_kernel(const __grid_constant__ StemParams sp) {
    constexpr int BN = 64;
    constexpr int NK = IN_KIND == 1 ? 1 : 2;          // K = 16 * NK
    constexpr int KREAL = IN_KIND == 1 ? 9 : 27;
    constexpr int TMEM_COLS = 2 * BN;
    const ConvParams& p = sp.c;

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* b_tile = smem;                                        // 64 rows x 128 B
    uint8_t* a_ring = smem + BN * 128;                             // STEM_STAGES x (128 rows x 128 B)
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(a_ring + STEM_STAGES * A_STAGE_BYTES);
    uint64_t* empty_bar = full_bar + STEM_STAGES;
    uint64_t* tfull_bar = empty_bar + STEM_STAGES;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
    float* bias_s = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full_bar) + 256);
    uint8_t* stg_s = reinterpret_cast<uint8_t*>(full_bar) + 1024;          // 1024 B aligned: swizzled TMA-store tiles

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    stage_bias(p, bias_s);
    if (threadIdx.x == 0) {
        tma_prefetch_desc(&p.tmA);
        for (int s = 0; s < STEM_STAGES; ++s) { mbar_init(&full_bar[s], 128); mbar_init(&empty_bar[s], 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(&tfull_bar[s], 1); mbar_init(&tempty_bar[s], 4); }          // groups take alternate tiles
        fence_barrier_init();
    }
    if (warp == 12) {
        tmem_alloc(tmem_slot, TMEM_COLS);
        tmem_relinquish();
    }
    if (warp >= 8 && warp < 12) {
        // weights -> bf16 B tile (row = co, 16-byte chunk c of row r sits at chunk c ^ (r & 7))
        const float scale = IN_KIND == 0 ? 1.0f : 1.0f / 255.0f;
        for (int i = threadIdx.x - STEM_PROD0; i < BN * NK * 2; i += 128) {
            const int co = i / (NK * 2), chunk = i % (NK * 2);
            uint32_t pk[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float v[2];
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int kk = chunk * 8 + j * 2 + u;
                    float w = 0.f;
                    if (kk < KREAL) {
                        const float* wr = sp.weight + co * 27;
                        w = IN_KIND == 1 ? (wr[kk] + wr[9 + kk] + wr[18 + kk]) : wr[kk];
                    }
                    v[u] = w * scale;
                }
                pk[j] = pack_bf16(v[0], v[1]);
            }
            *reinterpret_cast<uint4*>(b_tile + co * 128 + ((chunk ^ (co & 7)) << 4)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
        fence_proxy_async();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp < 8) {
        stem_epilogue_tma(p, warp & 3, lane, warp >> 2, tmem_base, tfull_bar, tempty_bar, bias_s, stg_s);
    } else if (warp < 12) {
        // ------------------------------------------------------------------ im2col producers: one tile row each
        // The taps of tile i+1 are requested before tile i is converted and stored, so the global-load latency
        // overlaps a whole tile of work instead of stalling every tile.
        const int r = threadIdx.x - STEM_PROD0;
        const int lh = r / TILE_W, lw = r % TILE_W;
        int stage = 0;
        uint32_t phase = 0;
        uint32_t buf[3][KREAL];                 // taps of tiles i, i+1, i+2 (loads two tiles ahead of their use)
        auto fetch = [&](int tile, uint32_t* dst) {
            const TileCoord t = decode_tile(p, tile, BN);
            const int y = t.h0 + lh, x = t.w0 + lw;
#pragma unroll
            for (int kk = 0; kk < KREAL; ++kk) {
                const int c = kk / 9, tap = kk % 9;
                dst[kk] = stem_px_raw<IN_KIND>(sp.in, t.img, c, y + (tap / 3 - 1) * p.dil, x + (tap % 3 - 1) * p.dil, p.H, p.W);
            }
        };
        const int G = gridDim.x;
        if ((int)blockIdx.x < p.total_tiles) fetch(blockIdx.x, buf[0]);
        if ((int)blockIdx.x + G < p.total_tiles) fetch(blockIdx.x + G, buf[1]);
        for (int base = blockIdx.x; base < p.total_tiles; base += 3 * G) {
#pragma unroll
            for (int u = 0; u < 3; ++u) {
                const int tile = base + u * G;
                if (tile >= p.total_tiles) break;
                if (tile + 2 * G < p.total_tiles) fetch(tile + 2 * G, buf[(u + 2) % 3]);
                const uint32_t* cur = buf[u];
                uint32_t pk[NK * 8];
#pragma unroll
                for (int j = 0; j < NK * 8; ++j)
                    pk[j] = pack_bf16(2 * j < KREAL ? stem_val<IN_KIND>(cur[2 * j]) : 0.f,
                                      2 * j + 1 < KREAL ? stem_val<IN_KIND>(cur[2 * j + 1]) : 0.f);
                mbar_wait(&empty_bar[stage], phase ^ 1u);
                uint8_t* row = a_ring + stage * A_STAGE_BYTES + r * 128;
#pragma unroll
                for (int chunk = 0; chunk < NK * 2; ++chunk)
                    *reinterpret_cast<uint4*>(row + ((chunk ^ (r & 7)) << 4)) =
                        make_uint4(pk[4 * chunk], pk[4 * chunk + 1], pk[4 * chunk + 2], pk[4 * chunk + 3]);
                fence_proxy_async();                // generic-proxy stores -> visible to the tensor core (async proxy)
                mbar_arrive(&full_bar[stage]);
                if (++stage == STEM_STAGES) { stage = 0; phase ^= 1u; }
            }
        }
    } else {
        // ------------------------------------------------------------------ MMA issuer (warp-uniform loop)
        const uint32_t idesc = umma_idesc_bf16(TILE_M, BN);
        const uint64_t bdesc = umma_desc_sw128(smem_u32(b_tile));
        int stage = 0;
        uint32_t phase = 0;
        int it = 0;
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
            const int as = it & 1;
            const uint32_t aphase = (uint32_t)(it >> 1) & 1u;
            mbar_wait(&tempty_bar[as], aphase ^ 1u);
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after();
            const uint64_t adesc = umma_desc_sw128(smem_u32(a_ring + stage * A_STAGE_BYTES));
            if (elect_one()) {
#pragma unroll
                for (int k = 0; k < NK; ++k)
                    umma_bf16(tmem_base + (uint32_t)(as * BN), adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc,
                              k ? 1u : 0u);
                umma_commit(&empty_bar[stage]);
                umma_commit(&tfull_bar[as]);
            }
            __syncwarp();
            if (++stage == STEM_STAGES) { stage = 0; phase ^= 1u; }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 12) {
        tc_fence_after();
        tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

// ---------------------------------------------------------------------------- host side

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(ptr);
    }
    return fn;
}

int encode_map(CUtensorMap* m, const void* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes,
               const cuuint32_t* box, CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B) {
    EncodeTiledFn fn = encode_fn();
    DC_REQUIRE(fn, DC_ECUDA, "cuTensorMapEncodeTiled entry point not available");
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), dims, strides_bytes,
                    box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    DC_REQUIRE(r == CUDA_SUCCESS, DC_ECUDA, "cuTensorMapEncodeTiled failed (CUresult %d)", (int)r);
    return DC_OK;
}

template <int BN, int NSTAGES, bool SPLIT = false>
int launch_variant(const ConvParams& p, cudaStream_t stream) {
    constexpr int STAGE_BYTES = A_STAGE_BYTES + BN * KCHUNK * 2;
    constexpr size_t SMEM = (size_t)NSTAGES * STAGE_BYTES + 1024 /* alignment slack */ + 256 /* barriers */ +
                            4096 + 256 /* bias (<= 1024 ch) + out_conv weights */ + EPI_STAGE_TOTAL;
    static_assert(SMEM <= 227 * 1024, "stage ring exceeds shared memory");
    static unsigned long long attr_done = 0;
    void (*kernel)(ConvParams) = SPLIT ? conv_tc_split_kernel<BN, NSTAGES> : conv_tc_kernel<BN, NSTAGES>;
    { int rc = set_max_smem_once(kernel, (int)SMEM, &attr_done); if (rc != DC_OK) return rc; }
    int grid = p.total_tiles < num_sms() ? p.total_tiles : num_sms();
    kernel<<<grid, NUM_THREADS, SMEM, stream>>>(p);
    DC_CUDA(cudaGetLastError());
    return DC_OK;
}

}  // namespace

// 64 -> 64 channel 3x3 layer, dilation 1, even H and W, by output parity class (conv_par2_kernel); arguments already
// validated by launch_conv_tc.
static int launch_conv_par(const dc_conv_args_t* a, cudaStream_t stream, const float* bias_host) {
    DC_REQUIRE(((uintptr_t)a->weight_par & 15) == 0, DC_EINVAL, "dc_conv_tc: weight_par must be 16-byte aligned");
    ConvParams p;
    memset(&p, 0, sizeof(p));
    const int Hh = a->H / 2, Wh = a->W / 2;          // the tile grid is the half-resolution one
    {   // in: [B, H, W, 64 of in_stride] seen as [B, H, W/2, parity, 64]: a box is one column-parity plane
        const cuuint64_t ps = (cuuint64_t)a->in_stride * 2;
        cuuint64_t dims[5] = {64, 2, (cuuint64_t)Wh, (cuuint64_t)a->H, (cuuint64_t)a->B};
        cuuint64_t str[4] = {ps, 2 * ps, (cuuint64_t)a->W * ps, (cuuint64_t)a->H * a->W * ps};
        cuuint32_t box[5] = {KCHUNK, 1, UPF_S_W, UPF_S_H, 1};
        int rc = encode_map(&p.tmS, a->in, 5, dims, str, box);
        if (rc != DC_OK) return rc;
    }
    {   // weights: [2 CTAs of a pair][PAR_ROWS_PER_RANK rows in schedule order][64]
        cuuint64_t dims[2] = {KCHUNK, (cuuint64_t)2 * PAR_ROWS_PER_RANK};
        cuuint64_t str[1] = {KCHUNK * 2};
        cuuint32_t box[2] = {KCHUNK, UPF_GROUP_ROWS};
        int rc = encode_map(&p.tmB, a->weight_par, 2, dims, str, box);
        if (rc != DC_OK) return rc;
    }
    p.B = a->B; p.H = Hh; p.W = Wh; p.Cin = 64; p.Cout = 64;
    p.dil = 1; p.ntaps = 9; p.kchunks = 1;
    p.tiles_w = ceil_div(Wh, HT_W);
    p.tiles_h = ceil_div(Hh, HT_H);
    p.n_tiles = 1;
    const long long total = (long long)a->B * p.tiles_w * p.tiles_h;
    DC_REQUIRE(total < (1ll << 31), DC_EINVAL, "dc_conv_tc: too many tiles");
    p.total_tiles = p.m_tiles = (int)total;
    p.fd_ntiles = make_fastdiv(1); p.fd_per_img = make_fastdiv(p.tiles_h * p.tiles_w); p.fd_tiles_w = make_fastdiv(p.tiles_w);
    p.epilogue = a->epilogue;
    p.relu = a->relu != 0;
    p.bias = a->bias;
    if (bias_host && a->epilogue != DC_EPI_HEAD) {
        p.bias_const = 1;
        memcpy(p.bias_c, bias_host, sizeof(p.bias_c));
    }
    p.out = reinterpret_cast<__nv_bfloat16*>(a->out);
    p.out_stride = a->out_stride; p.out_offset = a->out_offset;
    p.pool_out = reinterpret_cast<__nv_bfloat16*>(a->pool_out);
    p.pool_stride = a->pool_stride;
    p.head_w = a->head_w; p.head_b = a->head_b; p.thresh = a->thresh;
    p.prob_out = a->prob_out; p.mask_out = a->mask_out;

    const int n_pairs = (p.m_tiles + 1) / 2;
    const int max_clusters = num_sms() / 2;
    const int grid = 2 * (n_pairs < max_clusters ? n_pairs : max_clusters);
    static unsigned long long attr_done = 0;
    int rc = set_max_smem_once(conv_par2_kernel, (int)PAR_SMEM, &attr_done);
    if (rc != DC_OK) return rc;
    conv_par2_kernel<<<grid, NUM_THREADS, PAR_SMEM, stream>>>(p);
    DC_CUDA(cudaGetLastError());
    return DC_OK;
}

int launch_conv_tc(const dc_conv_args_t* a, cudaStream_t stream, const float* bias_host) {
    DC_REQUIRE(a && a->in && a->weight && a->bias, DC_EINVAL, "dc_conv_tc: null pointer argument");
    DC_REQUIRE(a->kind == DC_KIND_CONV3X3 || a->kind == DC_KIND_UPCONV2, DC_EINVAL, "dc_conv_tc: kind %d", a->kind);
    DC_REQUIRE(a->B > 0 && a->H > 0 && a->W > 0, DC_EINVAL, "dc_conv_tc: bad shape %d x %d x %d", a->B, a->H, a->W);
    DC_REQUIRE(a->Cin > 0 && a->Cin % KCHUNK == 0, DC_EINVAL, "dc_conv_tc: Cin %d must be a multiple of 64", a->Cin);
    DC_REQUIRE(a->Cout > 0 && a->Cout % 64 == 0 && a->Cout <= 1024, DC_EINVAL,
               "dc_conv_tc: Cout %d must be a multiple of 64 and at most 1024", a->Cout);
    DC_REQUIRE(a->in_stride >= a->Cin && a->in_stride % 8 == 0, DC_EINVAL, "dc_conv_tc: in_stride %d", a->in_stride);
    DC_REQUIRE(((uintptr_t)a->in & 15) == 0 && ((uintptr_t)a->weight & 15) == 0, DC_EINVAL,
               "dc_conv_tc: in / weight must be 16-byte aligned");
    const bool up = a->kind == DC_KIND_UPCONV2;
    DC_REQUIRE(up == (a->epilogue == DC_EPI_UPSCATTER), DC_EINVAL, "dc_conv_tc: kind %d with epilogue %d", a->kind,
               a->epilogue);
    DC_REQUIRE(a->epilogue >= DC_EPI_STORE && a->epilogue <= DC_EPI_UPSCATTER, DC_EINVAL, "dc_conv_tc: epilogue %d",
               a->epilogue);
    DC_REQUIRE(up || a->dilation >= 1, DC_EINVAL, "dc_conv_tc: dilation %d", a->dilation);
    if (a->epilogue == DC_EPI_HEAD) {
        DC_REQUIRE(a->Cout == 64 && a->head_w && (a->prob_out || a->mask_out), DC_EINVAL,
                   "dc_conv_tc: HEAD epilogue needs Cout == 64, head_w and prob_out or mask_out");
    } else {
        DC_REQUIRE(a->out && ((uintptr_t)a->out & 15) == 0, DC_EINVAL, "dc_conv_tc: out must be 16-byte aligned");
        DC_REQUIRE(a->out_stride % 8 == 0 && a->out_offset % 8 == 0 && a->out_offset >= 0 &&
                       a->out_stride >= a->out_offset + a->Cout,
                   DC_EINVAL, "dc_conv_tc: out_stride %d / out_offset %d", a->out_stride, a->out_offset);
    }
    if (a->epilogue == DC_EPI_STORE_POOL) {
        DC_REQUIRE(a->pool_out && ((uintptr_t)a->pool_out & 15) == 0 && a->pool_stride % 8 == 0 &&
                       a->pool_stride >= a->Cout,
                   DC_EINVAL, "dc_conv_tc: pool_out / pool_stride");
        DC_REQUIRE(a->H % 2 == 0 && a->W % 2 == 0, DC_EINVAL, "dc_conv_tc: pooled layer needs even H, W");
    }
    // fp32 precision: three bf16 planes per tensor, `*_plane_stride` channels apart within a pixel; always the per-tap
    // kernel (conv_tc_split_kernel)
    DC_REQUIRE(a->planes == 0 || a->planes == 1 || a->planes == 3, DC_EINVAL, "dc_conv_tc: planes %d (1 or 3)", a->planes);
    const bool split = a->planes == 3;
    if (split) {
        DC_REQUIRE(a->in_plane_stride >= a->Cin && a->in_plane_stride % 8 == 0 && a->in_stride >= 2 * a->in_plane_stride + a->Cin,
                   DC_EINVAL, "dc_conv_tc: in_plane_stride %d with in_stride %d", a->in_plane_stride, a->in_stride);
        if (a->epilogue != DC_EPI_HEAD)
            DC_REQUIRE(a->out_plane_stride >= a->Cout && a->out_plane_stride % 8 == 0 &&
                           a->out_stride >= a->out_offset + 2 * a->out_plane_stride + a->Cout,
                       DC_EINVAL, "dc_conv_tc: out_plane_stride %d with out_stride %d / out_offset %d", a->out_plane_stride,
                       a->out_stride, a->out_offset);
        if (a->epilogue == DC_EPI_STORE_POOL)
            DC_REQUIRE(a->pool_plane_stride >= a->Cout && a->pool_plane_stride % 8 == 0 &&
                           a->pool_stride >= 2 * a->pool_plane_stride + a->Cout,
                       DC_EINVAL, "dc_conv_tc: pool_plane_stride %d with pool_stride %d", a->pool_plane_stride, a->pool_stride);
    }
    if (!split && !up && a->weight_par && a->Cin == 64 && a->Cout == 64 && a->dilation == 1 && a->H % 2 == 0 &&
        a->W % 2 == 0 && g_kernel_family == DC_CONV_FAMILY_AUTO)
        return launch_conv_par(a, stream, bias_host);
    const int gemm_n = up ? 4 * a->Cout : a->Cout;      // upconv: the four output parities are one wide GEMM N
    const int BN = gemm_n % 256 == 0 ? 256 : (gemm_n % 128 == 0 ? 128 : 64);

    ConvParams p;
    memset(&p, 0, sizeof(p));

    // Thin layers (Cout = 64 / 128): one haloed region per tile and chunk; weights resident in shared memory when
    // the whole layer fits, else streamed through a ring of (tap, chunk) slices.
    bool halo = false, halo_wres = true, halo_pair = false;
    int halo_nhalf = 1;
    size_t halo_smem = 0;
    if (!split && !up && a->dilation <= 4 && g_kernel_family == DC_CONV_FAMILY_AUTO) {
        // CTA pair (cta_group::2): half of the weight rows per SM.  BN <= 128: two 8-wide halves per tile (two MMA
        // chains); BN = 256: one half (a 128-cycle MMA hides its own latency, and 2 x 2 x 256 columns would not fit
        // TMEM).  Weights resident when Cout == BN and the layer's half fits next to two regions, else streamed
        // (not at BN = 64: a 4 KB slice is too little work to cover the L2 latency with the ring that fits).
        // Halves per tile = independent accumulator chains.  Back-to-back MMAs into one accumulator issue ~130 cycles
        // apart, so a chain needs >= 128 cycles of other work between its MMAs: N = 128 -> 2 halves (64-cycle MMAs),
        // N = 64 -> 4 halves (32-cycle MMAs; 3 or 2 when the regions would not fit), N = 256 -> 1.
        const size_t w_tile = (size_t)(BN / 2) * KCHUNK * 2;
        const size_t w_half = (size_t)9 * (a->Cin / KCHUNK) * w_tile;
        const size_t budget = 227 * 1024 - 1024 - HALO_BAR_BYTES - HALO_BIAS_BYTES - EPI_STAGE_TOTAL;
        const int nh_max = BN == 256 ? 1 : (BN == 128 ? 2 : 4);
        for (int nh = nh_max; nh >= (BN == 64 ? 2 : nh_max) && !halo; --nh) {
        const int rw = HT_W * nh + 2 * a->dilation, rh = HT_H + 2 * a->dilation;
        const size_t region_stride = (size_t)rw * rh * KCHUNK * 2;
        for (int pass = 0; pass < 2 && !halo; ++pass) {
            size_t wsm = w_half;
            int nb = 0;
            if (pass == 0 && (a->Cout != BN || BN == 256)) continue;   // resident: single n-tile, BN <= 128 kernels
            if (pass == 1) {
                if (BN == 64 || budget < 2 * region_stride + 4 * w_tile) break;
                nb = (int)((budget - 2 * region_stride) / w_tile);
                if (nb > HALO_MAX_STAGES) nb = HALO_MAX_STAGES;
                wsm = (size_t)nb * w_tile;
            }
            const long long nst = wsm < budget ? (long long)((budget - wsm) / region_stride) : 0;
            if (nst >= 2) {
                halo = halo_pair = true;
                halo_wres = pass == 0;
                halo_nhalf = nh;
                p.region_w = rw; p.region_h = rh; p.region_stride = (int)region_stride;
                p.nstages = nst > HALO_MAX_STAGES ? HALO_MAX_STAGES : (int)nst;
                p.nbstages = nb;
                halo_smem = wsm + (size_t)p.nstages * region_stride + 1024 + HALO_BAR_BYTES + HALO_BIAS_BYTES + EPI_STAGE_TOTAL;
            }
        }
        }
    }
    if (!split && !halo && !up && a->Cout == HALO_BN && a->dilation <= 4) {
        // Cout = 64 layers whose weights do not fit next to the pair kernel's regions: conv_halo_kernel streams them.
        // TMA and the MMA unit both take the swizzle phase from absolute address bits, so a region only needs
        // TMA's 128 B alignment, not a 1024 B one: regions are packed back to back
        constexpr size_t budget = 227 * 1024 - 1024 /* alignment slack */ - HALO_BAR_BYTES - HALO_BIAS_BYTES -
                                  EPI_STAGE_TOTAL /* epilogue transpose buffers */;
        constexpr size_t max_region = (size_t)(HT_W * HALO_NHALF + 2 * 4) * (HT_H + 2 * 4) * KCHUNK * 2;    // dilation 4
        static_assert(budget >= 2 * max_region + 4 * HALO_W_TILE_BYTES, "conv_halo_kernel: two regions and a 4-slice ring");
        const int rw = HT_W * HALO_NHALF + 2 * a->dilation, rh = HT_H + 2 * a->dilation;
        const size_t region_stride = (size_t)rw * rh * KCHUNK * 2;
        int nb = (int)((budget - 2 * region_stride) / HALO_W_TILE_BYTES);
        if (nb > HALO_MAX_STAGES) nb = HALO_MAX_STAGES;
        const size_t wsm = (size_t)nb * HALO_W_TILE_BYTES;
        const int nst = (int)((budget - wsm) / region_stride);
        halo = true;
        halo_nhalf = HALO_NHALF;
        p.region_w = rw; p.region_h = rh; p.region_stride = (int)region_stride;
        p.nstages = nst > HALO_MAX_STAGES ? HALO_MAX_STAGES : nst;
        p.nbstages = nb;
        halo_smem = wsm + (size_t)p.nstages * region_stride + 1024 + HALO_BAR_BYTES + HALO_BIAS_BYTES + EPI_STAGE_TOTAL;
    }
    if (g_kernel_family == DC_CONV_FAMILY_GENERIC) halo = halo_pair = false;      // test-only override (dc_debug_set_conv_family)
    {
        const int cin_span = split ? 2 * a->in_plane_stride + a->Cin : a->Cin;      // channels the boxes may read
        cuuint64_t dims[4] = {(cuuint64_t)cin_span, (cuuint64_t)a->W, (cuuint64_t)a->H, (cuuint64_t)a->B};
        cuuint64_t str[3] = {(cuuint64_t)a->in_stride * 2, (cuuint64_t)a->W * a->in_stride * 2,
                             (cuuint64_t)a->H * a->W * a->in_stride * 2};
        cuuint32_t box[4] = {KCHUNK, TILE_W, TILE_H, 1};
        if (halo) { box[1] = (cuuint32_t)p.region_w; box[2] = (cuuint32_t)p.region_h; }
        int rc = encode_map(&p.tmA, a->in, 4, dims, str, box);
        if (rc != DC_OK) return rc;
    }
    {
        const int ktot = (up ? a->Cin : 9 * a->Cin) * (split ? 3 : 1);
        const int rows = up ? 4 * a->Cout : a->Cout;
        cuuint64_t dims[2] = {(cuuint64_t)ktot, (cuuint64_t)rows};
        cuuint64_t str[1] = {(cuuint64_t)ktot * 2};
        cuuint32_t box[2] = {KCHUNK, (cuuint32_t)(halo_pair ? BN / 2 : BN)};
        int rc = encode_map(&p.tmB, a->weight, 2, dims, str, box);
        if (rc != DC_OK) return rc;
    }
    p.B = a->B; p.H = a->H; p.W = a->W; p.Cin = a->Cin; p.Cout = a->Cout;
    p.dil = up ? 1 : a->dilation;
    p.ntaps = up ? 1 : 9;
    p.kchunks = a->Cin / KCHUNK;
    p.tiles_w = ceil_div(a->W, halo ? HT_W * halo_nhalf : TILE_W);
    p.tiles_h = ceil_div(a->H, halo ? HT_H : TILE_H);
    p.n_tiles = (up ? 4 * a->Cout : a->Cout) / BN;
    const long long total = (long long)a->B * p.tiles_w * p.tiles_h * p.n_tiles;
    DC_REQUIRE(total < (1ll << 31), DC_EINVAL, "dc_conv_tc: too many tiles");
    p.total_tiles = (int)total;
    p.m_tiles = p.total_tiles / p.n_tiles;
    p.fd_ntiles = make_fastdiv(p.n_tiles); p.fd_per_img = make_fastdiv(p.tiles_h * p.tiles_w); p.fd_tiles_w = make_fastdiv(p.tiles_w);
    p.epilogue = a->epilogue;
    p.relu = up ? 0 : (a->relu != 0);
    p.bias = a->bias;
    if (bias_host && a->Cout == 64 && a->epilogue != DC_EPI_HEAD) {
        p.bias_const = 1;
        memcpy(p.bias_c, bias_host, sizeof(p.bias_c));
    }
    p.out = reinterpret_cast<__nv_bfloat16*>(a->out);
    p.out_stride = a->out_stride; p.out_offset = a->out_offset;
    p.pool_out = reinterpret_cast<__nv_bfloat16*>(a->pool_out);
    p.pool_stride = a->pool_stride;
    p.head_w = a->head_w; p.head_b = a->head_b; p.thresh = a->thresh;
    p.prob_out = a->prob_out; p.mask_out = a->mask_out;
    p.in_plane_stride = a->in_plane_stride; p.out_plane_stride = a->out_plane_stride; p.pool_plane_stride = a->pool_plane_stride;

    if (split) {
        switch (BN) {
            case 256: return launch_variant<256, 4, true>(p, stream);
            case 128: return launch_variant<128, 6, true>(p, stream);
            default:  return launch_variant<64, 8, true>(p, stream);
        }
    }
    if (halo_pair) {
        const int m_tiles = p.total_tiles / p.n_tiles;
        const int n_pairs = ((m_tiles + 1) / 2) * p.n_tiles;
        const int max_clusters = num_sms() / 2;
        const int grid = 2 * (n_pairs < max_clusters ? n_pairs : max_clusters);
#define DC_PAIR_CASE(bn, nh, wr)                                                                                      \
        if (BN == bn && halo_nhalf == nh && halo_wres == wr) {                                                        \
            static unsigned long long attr_done = 0;                                                                  \
            int rc_ = set_max_smem_once(conv_halo2_kernel<bn, nh, wr>, 227 * 1024, &attr_done);                       \
            if (rc_ != DC_OK) return rc_;                                                                             \
            conv_halo2_kernel<bn, nh, wr><<<grid, NUM_THREADS, halo_smem, stream>>>(p);                               \
        }
        DC_PAIR_CASE(64, 4, true) DC_PAIR_CASE(64, 3, true) DC_PAIR_CASE(64, 2, true)
        DC_PAIR_CASE(128, 2, true) DC_PAIR_CASE(128, 2, false) DC_PAIR_CASE(256, 1, false)
#undef DC_PAIR_CASE
        DC_CUDA(cudaGetLastError());
        return DC_OK;
    }
    if (halo) {
        const int grid = p.total_tiles < num_sms() ? p.total_tiles : num_sms();
        static unsigned long long attr_done = 0;
        int rc = set_max_smem_once(conv_halo_kernel, 227 * 1024, &attr_done);
        if (rc != DC_OK) return rc;
        conv_halo_kernel<<<grid, NUM_THREADS, halo_smem, stream>>>(p);
        DC_CUDA(cudaGetLastError());
        return DC_OK;
    }
    switch (BN) {
        case 256: return launch_variant<256, 4>(p, stream);
        case 128: return launch_variant<128, 6>(p, stream);
        default:  return launch_variant<64, 8>(p, stream);
    }
}

// C = 128 / 256 / 512: conv_upfused_wide_kernel (arguments validated by launch_conv_upfused)
static int launch_conv_upfused_wide(const dc_upfuse_args_t* a, cudaStream_t stream) {
    const int C = a->channels;
    const int BN = C == 128 ? 128 : 256;
    const int ncls = 256 / BN, groups = 4 / ncls, real_ntiles = C / BN, SC = C / KCHUNK;
    DC_REQUIRE(a->weight_skip && ((uintptr_t)a->weight_skip & 15) == 0, DC_EINVAL, "dc_conv_upfused: weight_skip");
    ConvParams p;
    memset(&p, 0, sizeof(p));
    {
        cuuint64_t dims[4] = {(cuuint64_t)2 * C, (cuuint64_t)a->W, (cuuint64_t)a->H, (cuuint64_t)a->B};
        cuuint64_t str[3] = {(cuuint64_t)a->x_stride * 2, (cuuint64_t)a->W * a->x_stride * 2,
                             (cuuint64_t)a->H * a->W * a->x_stride * 2};
        cuuint32_t box[4] = {KCHUNK, UPF_U_W, UPF_U_H, 1};
        int rc = encode_map(&p.tmA, a->x, 4, dims, str, box);
        if (rc != DC_OK) return rc;
    }
    {
        const cuuint64_t ps = (cuuint64_t)a->skip_stride * 2;
        cuuint64_t dims[5] = {(cuuint64_t)C, 2, (cuuint64_t)a->W, (cuuint64_t)(2 * a->H), (cuuint64_t)a->B};
        cuuint64_t str[4] = {ps, 2 * ps, 2 * (cuuint64_t)a->W * ps, 4 * (cuuint64_t)a->H * a->W * ps};
        cuuint32_t box[5] = {KCHUNK, 1, UPF_S_W, UPF_S_H, 1};
        int rc = encode_map(&p.tmS, a->skip, 5, dims, str, box);
        if (rc != DC_OK) return rc;
    }
    {   // composed weights: [class group][n-tile][CTA][x chunk][tap][ncls x BN/2 rows][64]
        cuuint64_t dims[2] = {KCHUNK, (cuuint64_t)groups * real_ntiles * 2 * (2 * SC) * 4 * UPF_GROUP_ROWS};
        cuuint64_t str[1] = {KCHUNK * 2};
        cuuint32_t box[2] = {KCHUNK, UPF_GROUP_ROWS};
        int rc = encode_map(&p.tmB, a->weight, 2, dims, str, box);
        if (rc != DC_OK) return rc;
    }
    {   // skip weights: [n-tile][CTA][chunk][tap][BN/2 rows][64]
        cuuint64_t dims[2] = {KCHUNK, (cuuint64_t)real_ntiles * 2 * SC * 9 * (BN / 2)};
        cuuint64_t str[1] = {KCHUNK * 2};
        cuuint32_t box[2] = {KCHUNK, (cuuint32_t)(BN / 2)};
        int rc = encode_map(&p.tmB2, a->weight_skip, 2, dims, str, box);
        if (rc != DC_OK) return rc;
    }
    p.B = a->B; p.H = a->H; p.W = a->W; p.Cin = 3 * C; p.Cout = C;
    p.dil = 1; p.ntaps = 9; p.kchunks = SC;
    p.tiles_w = ceil_div(a->W, HT_W);
    p.tiles_h = ceil_div(a->H, HT_H);
    p.n_tiles = groups * real_ntiles;
    p.real_ntiles = real_ntiles;
    const long long total = (long long)a->B * p.tiles_w * p.tiles_h * p.n_tiles;
    DC_REQUIRE(total < (1ll << 31), DC_EINVAL, "dc_conv_upfused: too many tiles");
    p.total_tiles = (int)total;
    p.m_tiles = p.total_tiles / p.n_tiles;
    p.fd_ntiles = make_fastdiv(p.n_tiles); p.fd_per_img = make_fastdiv(p.tiles_h * p.tiles_w); p.fd_tiles_w = make_fastdiv(p.tiles_w);
    p.epilogue = DC_EPI_STORE;
    p.relu = a->relu != 0;
    p.bias = a->bias9 + 4 * C;
    p.border_bias = 1;
    p.out = reinterpret_cast<__nv_bfloat16*>(a->out);
    p.out_stride = a->out_stride; p.out_offset = a->out_offset;

    const int n_pairs = ((p.m_tiles + 1) / 2) * p.n_tiles;
    const int max_clusters = num_sms() / 2;
    const int grid = 2 * (n_pairs < max_clusters ? n_pairs : max_clusters);
#define DC_UPW_CASE(bn)                                                                                      \
    if (BN == bn) {                                                                                          \
        static unsigned long long attr_done = 0;                                                             \
        int rc = set_max_smem_once(conv_upfused_wide_kernel<bn>, (int)UPW_SMEM, &attr_done);                 \
        if (rc != DC_OK) return rc;                                                                          \
        conv_upfused_wide_kernel<bn><<<grid, NUM_THREADS, UPW_SMEM, stream>>>(p);                            \
    }
    DC_UPW_CASE(128) DC_UPW_CASE(256)
#undef DC_UPW_CASE
    DC_CUDA(cudaGetLastError());
    return DC_OK;
}

int launch_conv_upfused(const dc_upfuse_args_t* a, cudaStream_t stream, const float* bias9_host) {
    DC_REQUIRE(a && a->x && a->skip && a->weight && a->bias9 && a->out, DC_EINVAL,
               "dc_conv_upfused: null pointer argument");
    const int C = a->channels ? a->channels : 64;
    DC_REQUIRE(C == 64 || C == 128 || C == 256 || C == 512, DC_EINVAL, "dc_conv_upfused: channels %d (64, 128, 256 or 512)", C);
    DC_REQUIRE(C != 64 || bias9_host, DC_EINVAL, "dc_conv_upfused: null pointer argument");
    DC_REQUIRE(a->B > 0 && a->H > 0 && a->W > 0, DC_EINVAL, "dc_conv_upfused: bad shape %d x %d x %d", a->B, a->H, a->W);
    DC_REQUIRE(a->x_stride >= 2 * C && a->x_stride % 8 == 0 && a->skip_stride >= C && a->skip_stride % 8 == 0, DC_EINVAL,
               "dc_conv_upfused: x_stride %d / skip_stride %d", a->x_stride, a->skip_stride);
    DC_REQUIRE(((uintptr_t)a->x & 15) == 0 && ((uintptr_t)a->skip & 15) == 0 && ((uintptr_t)a->weight & 15) == 0 &&
                   ((uintptr_t)a->out & 15) == 0,
               DC_EINVAL, "dc_conv_upfused: x / skip / weight / out must be 16-byte aligned");
    DC_REQUIRE(a->out_stride % 8 == 0 && a->out_offset % 8 == 0 && a->out_offset >= 0 && a->out_stride >= a->out_offset + C,
               DC_EINVAL, "dc_conv_upfused: out_stride %d / out_offset %d", a->out_stride, a->out_offset);
    if (C != 64) {
        dc_upfuse_args_t b = *a;
        b.channels = C;
        return launch_conv_upfused_wide(&b, stream);
    }
    ConvParams p;
    memset(&p, 0, sizeof(p));
    {   // x: [B, H, W, 128 of x_stride], one haloed region per 64-channel chunk
        cuuint64_t dims[4] = {128, (cuuint64_t)a->W, (cuuint64_t)a->H, (cuuint64_t)a->B};
        cuuint64_t str[3] = {(cuuint64_t)a->x_stride * 2, (cuuint64_t)a->W * a->x_stride * 2,
                             (cuuint64_t)a->H * a->W * a->x_stride * 2};
        cuuint32_t box[4] = {KCHUNK, UPF_U_W, UPF_U_H, 1};
        int rc = encode_map(&p.tmA, a->x, 4, dims, str, box);
        if (rc != DC_OK) return rc;
    }
    {   // skip: [B, 2H, 2W, 64 of skip_stride] seen as [B, 2H, W, parity, 64]: a box is one column-parity plane
        const cuuint64_t ps = (cuuint64_t)a->skip_stride * 2;
        cuuint64_t dims[5] = {64, 2, (cuuint64_t)a->W, (cuuint64_t)(2 * a->H), (cuuint64_t)a->B};
        cuuint64_t str[4] = {ps, 2 * ps, 2 * (cuuint64_t)a->W * ps, 4 * (cuuint64_t)a->H * a->W * ps};
        cuuint32_t box[5] = {KCHUNK, 1, UPF_S_W, UPF_S_H, 1};
        int rc = encode_map(&p.tmS, a->skip, 5, dims, str, box);
        if (rc != DC_OK) return rc;
    }
    {   // weights: [2 CTAs of a pair][UPF_ROWS_PER_RANK rows in the order the MMA schedule consumes them][64]
        cuuint64_t dims[2] = {KCHUNK, (cuuint64_t)2 * UPF_ROWS_PER_RANK};
        cuuint64_t str[1] = {KCHUNK * 2};
        cuuint32_t box[2] = {KCHUNK, UPF_GROUP_ROWS};
        int rc = encode_map(&p.tmB, a->weight, 2, dims, str, box);
        if (rc != DC_OK) return rc;
    }
    p.B = a->B; p.H = a->H; p.W = a->W; p.Cin = 192; p.Cout = 64;
    p.dil = 1; p.ntaps = 9; p.kchunks = 3;
    p.tiles_w = ceil_div(a->W, HT_W);
    p.tiles_h = ceil_div(a->H, HT_H);
    p.n_tiles = 1;
    const long long total = (long long)a->B * p.tiles_w * p.tiles_h;
    DC_REQUIRE(total < (1ll << 31), DC_EINVAL, "dc_conv_upfused: too many tiles");
    p.total_tiles = p.m_tiles = (int)total;
    p.fd_ntiles = make_fastdiv(1); p.fd_per_img = make_fastdiv(p.tiles_h * p.tiles_w); p.fd_tiles_w = make_fastdiv(p.tiles_w);
    p.epilogue = DC_EPI_STORE;
    p.relu = a->relu != 0;
    p.bias = a->bias9 + 4 * 64;                       // interior class
    p.border_bias = 1;
    p.bias_const = 1;
    memcpy(p.bias_c, bias9_host + 4 * 64, sizeof(p.bias_c));
    p.out = reinterpret_cast<__nv_bfloat16*>(a->out);
    p.out_stride = a->out_stride; p.out_offset = a->out_offset;

    const int n_pairs = (p.m_tiles + 1) / 2;
    const int max_clusters = num_sms() / 2;
    const int grid = 2 * (n_pairs < max_clusters ? n_pairs : max_clusters);
    static unsigned long long attr_done = 0;
    int rc = set_max_smem_once(conv_upfused2_kernel, (int)UPF_SMEM, &attr_done);
    if (rc != DC_OK) return rc;
    conv_upfused2_kernel<<<grid, NUM_THREADS, UPF_SMEM, stream>>>(p);
    DC_CUDA(cudaGetLastError());
    return DC_OK;
}

// The MMA schedule of conv_upfused2_kernel for the host-side weight packer: one row {chunk (0, 1 = x channels,
// 2 = skip), window row, window column, first class, classes} per MMA, in issue order.
int upfuse_schedule(int* out, int cap) {
    const int nu = upf_u_count(), ns = upf_s_count();
    const int n = 2 * nu + ns;
    DC_REQUIRE(out && cap >= 5 * n, DC_EINVAL, "dc_debug_upfuse_schedule: need room for %d ints", 5 * n);
    int* o = out;
    for (int kc = 0; kc < 2; ++kc)
        for (int i = 0; i < nu; ++i) {
            const UpfOp op = upf_u_op(i);
            *o++ = kc; *o++ = op.r; *o++ = op.c; *o++ = op.cls0; *o++ = op.ncls;
        }
    for (int i = 0; i < ns; ++i) {
        const UpfOp op = upf_s_op(i);
        *o++ = 2; *o++ = op.r; *o++ = op.c; *o++ = op.cls0; *o++ = op.ncls;
    }
    return n;
}

int set_conv_family(int family) {
    DC_REQUIRE(family == DC_CONV_FAMILY_AUTO || family == DC_CONV_FAMILY_GENERIC, DC_EINVAL, "dc_debug_set_conv_family: %d", family);
    g_kernel_family = family;
    return DC_OK;
}

int launch_stem(const dc_stem_args_t* a, cudaStream_t stream, const float* bias_host) {
    DC_REQUIRE(a && a->in && a->weight && a->bias && a->out, DC_EINVAL, "dc_stem: null pointer argument");
    DC_REQUIRE(a->Cout == 64, DC_EINVAL, "dc_stem: Cout must be 64 (got %d)", a->Cout);
    DC_REQUIRE(a->B > 0 && a->H > 0 && a->W > 0 && a->dilation >= 1, DC_EINVAL, "dc_stem: bad shape");
    DC_REQUIRE(a->out_stride % 8 == 0 && a->out_offset % 8 == 0 && a->out_stride >= a->out_offset + 64, DC_EINVAL,
               "dc_stem: output stride/offset must be multiples of 8 channels");
    DC_REQUIRE(((uintptr_t)a->out & 15) == 0, DC_EINVAL, "dc_stem: out must be 16-byte aligned");
    DC_REQUIRE(a->in_kind >= 0 && a->in_kind <= 2, DC_EINVAL, "dc_stem: in_kind %d", a->in_kind);
    StemParams sp;
    memset(&sp, 0, sizeof(sp));
    ConvParams& p = sp.c;
    p.B = a->B; p.H = a->H; p.W = a->W; p.Cin = 3; p.Cout = 64;
    p.dil = a->dilation; p.ntaps = 9; p.kchunks = 1;
    p.tiles_w = ceil_div(a->W, TILE_W);
    p.tiles_h = ceil_div(a->H, TILE_H);
    p.n_tiles = 1;
    const long long total = (long long)a->B * p.tiles_w * p.tiles_h;
    DC_REQUIRE(total < (1ll << 31), DC_EINVAL, "dc_stem: too many tiles");
    p.total_tiles = (int)total;
    p.m_tiles = p.total_tiles / p.n_tiles;
    p.fd_ntiles = make_fastdiv(p.n_tiles); p.fd_per_img = make_fastdiv(p.tiles_h * p.tiles_w); p.fd_tiles_w = make_fastdiv(p.tiles_w);
    p.epilogue = DC_EPI_STORE; p.relu = 1;
    p.bias = a->bias;
    if (bias_host) {
        p.bias_const = 1;
        memcpy(p.bias_c, bias_host, sizeof(p.bias_c));
    }
    p.out = reinterpret_cast<__nv_bfloat16*>(a->out);
    p.out_stride = a->out_stride; p.out_offset = a->out_offset;
    sp.in = a->in; sp.weight = a->weight; sp.in_kind = a->in_kind;
    {
        // output as a 4D tensor (channel, x, y, image) for the TMA stores: boxes of 32 channels x 16 x 2 pixels
        cuuint64_t dims[4] = {(cuuint64_t)a->out_stride, (cuuint64_t)a->W, (cuuint64_t)a->H, (cuuint64_t)a->B};
        cuuint64_t str[3] = {(cuuint64_t)a->out_stride * 2, (cuuint64_t)a->W * a->out_stride * 2,
                             (cuuint64_t)a->H * a->W * a->out_stride * 2};
        cuuint32_t box[4] = {32, TILE_W, 2, 1};
        int rc = encode_map(&p.tmA, a->out, 4, dims, str, box, CU_TENSOR_MAP_SWIZZLE_64B);
        if (rc != DC_OK) return rc;
    }
    constexpr size_t SMEM = 64 * 128 + (size_t)STEM_STAGES * A_STAGE_BYTES + 1024 /* alignment slack */ +
                            1024 /* barriers + bias */ + STEM_STG_BYTES;
    static unsigned long long attr_done[3] = {0, 0, 0};
    {
        int rc = set_max_smem_once(stem_tc_kernel<0>, (int)SMEM, &attr_done[0]);
        if (rc == DC_OK) rc = set_max_smem_once(stem_tc_kernel<1>, (int)SMEM, &attr_done[1]);
        if (rc == DC_OK) rc = set_max_smem_once(stem_tc_kernel<2>, (int)SMEM, &attr_done[2]);
        if (rc != DC_OK) return rc;
    }
    const int grid = p.total_tiles < num_sms() ? p.total_tiles : num_sms();
    switch (a->in_kind) {
        case 0: stem_tc_kernel<0><<<grid, STEM_THREADS, SMEM, stream>>>(sp); break;
        case 1: stem_tc_kernel<1><<<grid, STEM_THREADS, SMEM, stream>>>(sp); break;
        default: stem_tc_kernel<2><<<grid, STEM_THREADS, SMEM, stream>>>(sp); break;
    }
    DC_CUDA(cudaGetLastError());
    return DC_OK;
}

}  // namespace dc
