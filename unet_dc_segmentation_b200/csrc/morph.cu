// morph.cu -- "rolling ball" background correction on the GPU.
//
// Replaces rolling_ball_correction_rgb (reference utils/data_loader.py:11-24), per plane:
//   kernel  = cv2.getStructuringElement(MORPH_ELLIPSE, (radius, radius))        :17
//   bg      = cv2.morphologyEx(channel, MORPH_OPEN, kernel)   erode, then dilate  :19
//   corr    = cv2.subtract(channel, bg)                       saturating u8       :20
//   out     = cv2.normalize(corr, None, 0, 255, NORM_MINMAX)                      :21
//
// The element is a radius x radius flat ellipse (NOT separable, not symmetric for even sizes): row i covers the
// columns [j1[i], j2[i]).  erode(y,x) = min_i min_{j in row i} src[y+i-an, x+j-an], dilate uses max over the SAME
// offsets, taps outside the image are ignored (OpenCV semantics).
//
// Kernel plan (chord tables, after Urbach & Wilkinson 2008, with centred chords).  The rows of the ellipse are
// NESTED intervals [lo_m, hi_m] (M distinct ones: 16 at radius 50), so the horizontal range-min over the m-th chord,
//   H_m[r][x] = min(H_{m-1}[r][x], min over [lo_m, lo_{m-1}) , min over (hi_{m-1}, hi_m]),
// is one step away from the previous chord's: two side windows of 1..12 pixels, each read from a power-of-two
// range table of the staged tile (2 fetches, tables of 1/2/4/8 pixels only).  Each chord table is then consumed at
// the SAME x by every element row of that width:  out[y][x] = min_m min_{dy in rows(m)} H_m[y+dy][x] -- aligned
// 4-pixel words, no shifts.  Per output word that is ~32 unaligned fetches (x 1.4 for the row halo) + 50 aligned
// ones, against 100 unaligned fetches for the row-by-row form, and only 3 small range tables instead of 6.
// A block owns a 64 x 128 tile; chord tables are double-buffered in shared memory with one barrier per chord.
// All arithmetic is u8 (as 16-bit lanes for the DPX min/max), so the result is bit-exact.
//
// Radii past the tiled kernel's limit (the haloed tile stops fitting shared memory at 171) run the banded pass
// (morph_band_kernel, below).  cv2's ellipse is the union of K rectangles Y_m x X_m: X_m are the distinct row
// intervals (nested), Y_m the rows whose interval contains X_m (a contiguous band holding the anchor row).  So
//   erode(y,x) = min_m min_{x' in x+X_m} V_m(y,x'),   V_m(y,x') = min_{y' in y+Y_m} src(y',x'),
// walked from the widest chord (shortest band) to the narrowest (tallest band): V_m is V_{m-1} plus the rows the band
// newly covers, and the horizontal range-min over the shrinking X_m is van Herk / Gil-Werman (prefix / suffix extrema
// over blocks of |X_m| pixels, two lookups per pixel) on full rows in shared memory, which needs no horizontal halo.
// Every rectangle contains the anchor, so taps outside the image are the identity (255 erode, 0 dilate).
#include "common.cuh"
#include <math.h>
#include <string.h>
#include <algorithm>

namespace dc {

namespace {

constexpr int TW = 64;            // tile width: 16 words of 4 pixels (a half-warp per tile row)
constexpr int TH_MAX = 128;       // tile height
constexpr int NT = 512;           // threads per block: 16 warps, each handling tile rows w and w + 16 of a 32-row group
constexpr int MAX_CHORDS = 64;    // distinct row widths (radius 150 has 45)
constexpr int MAX_ROWS = 256;     // element rows
constexpr int MAX_TABLES = 5;     // range tables of 1, 2, 4, 8, 16 pixels
constexpr int HP = 17;            // chord-table pitch in words: rows r and r + 16 land 16 banks apart
constexpr int A_ITS = 8;         // 32-row groups of the haloed region: tile rows + element rows - 1 <= 256

struct Fetch {
    int woff;                     // word offset of the window inside the range tables (table base + column)
    unsigned sel_e, sel_o;        // PRMT selectors: shift of the window inside the word pair + split into even / odd pixels
};
struct Chord {
    Fetch f[4];                   // left window (1-2 fetches) then right window (0-2 fetches); unused slots repeat
    int nf;
    int row_begin, row_end;       // element rows of this width: indices into SEPlan::rowoff
};
struct SEPlan {
    int k, an, pad, pitch, RH, level_words, ntables, nchords, th;
    Chord chord[MAX_CHORDS];
    int rowoff[MAX_ROWS + MAX_CHORDS];   // byte offset (dy + an) * HP * 4 of the rows inside a chord table, grouped by
                                         // chord, each chord's list padded to an even length (last row repeated)
};

template <bool IS_MAX>
__device__ __forceinline__ unsigned vop(unsigned a, unsigned b) {
    return IS_MAX ? __vmaxu4(a, b) : __vminu4(a, b);
}
// sm_100a has no byte-lane SIMD min/max, but it has the DPX three-operand 16-bit-lane form.  Pixels travel as
// 16-bit lanes holding the byte TWICE (v * 257: order-preserving), which one PRMT produces from any byte of a word
// pair -- so the unaligned window fetch (funnel shift) and the split into even / odd pixels are a single instruction.
template <bool IS_MAX>
__device__ __forceinline__ unsigned vop3_16(unsigned acc, unsigned a, unsigned b) {
    return IS_MAX ? __vimax3_u16x2(acc, a, b) : __vimin3_u16x2(acc, a, b);
}
__device__ __forceinline__ unsigned pack_lanes(unsigned e, unsigned o) { return __byte_perm(e, o, 0x6240); }   // e0 o1 e2 o3
// prmt with a selector whose nibbles are all <= 7 (no masking of the selector needed, unlike __byte_perm)
__device__ __forceinline__ unsigned prmt(unsigned a, unsigned b, unsigned sel) {
    unsigned d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}
// shared-memory accesses by 32-bit address (+ immediate): one address add per window instead of index arithmetic
template <int IMM>
__device__ __forceinline__ unsigned lds(unsigned addr) {
    unsigned v;
    asm volatile("ld.shared.u32 %0, [%1+%2];" : "=r"(v) : "r"(addr), "n"(IMM) : "memory");
    return v;
}
__device__ __forceinline__ unsigned lds_dyn(unsigned addr) {
    unsigned v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void sts_dyn(unsigned addr, unsigned v) {
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// One morphology pass over planes addressed as in[((p/C)*H*W + y*W + x)*C + p%C] (in_c = C) and
// written planar.  SUBTRACT: out = saturate(orig - result), plus a per-plane min/max reduction.
// NB = tile rows / 32; NA = 32-row groups of the haloed region this instantiation covers (RH <= 32 NA).
// PITCH / NTAB > 0: the region pitch and the number of range tables are compile-time (the instantiation for the
// reference's default radius 50: every shared-memory offset of the chord loop becomes an immediate).
template <bool IS_MAX, bool SUBTRACT, int NB, int NA, int PITCH, int NTAB>
__global__ void __launch_bounds__(NT, 2) morph_chord_kernel(const uint8_t* __restrict__ in, int in_c,
                                                            uint8_t* __restrict__ out, const uint8_t* __restrict__ orig,
                                                            int orig_c, int H, int W, int* __restrict__ minmax,
                                                            const __grid_constant__ SEPlan se) {
    extern __shared__ unsigned smem[];
    constexpr int TH = NB * 32;
    const int an = se.an, pad = se.pad, pitch = PITCH ? PITCH : se.pitch, RH = se.RH, level_words = pitch * RH;
    const unsigned ident = IS_MAX ? 0u : 0xffffffffu;
    unsigned* hbuf = smem + se.ntables * level_words;          // two chord tables of (32 NA) x HP words
    constexpr int hwords = NA * 32 * HP;

    const int plane = blockIdx.z;
    const int b = plane / in_c, c = plane % in_c;
    const int x0 = blockIdx.x * TW - an - pad, y0 = blockIdx.y * TH - an;   // region origin in the image (x0 % 4 == 0)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (!SUBTRACT && minmax && blockIdx.x == 0 && blockIdx.y == 0 && tid == 0) {
        minmax[2 * plane] = 255;                 // the dilate pass (a later launch) reduces into these
        minmax[2 * plane + 1] = 0;
    }

    // ---- stage the tile + halo (range table 0) and build the range tables, one warp per region row ----
    // T_l[x] = op(T_{l-1}[x], T_{l-1}[x + 2^(l-1)]), identity outside the image / beyond the row.
    const uint8_t* src = in + (size_t)b * H * W * in_c + c;
    const int ntables = NTAB ? NTAB : se.ntables;
    if (in_c == 1 && (W & 3) == 0 && (reinterpret_cast<uintptr_t>(in) & 3) == 0 && pitch <= 32) {
        // planar input with 4-pixel-aligned rows and a region row of at most 32 words: a lane holds one word of the
        // row (x0 % 4 == 0 and W % 4 == 0, so a word lies wholly inside or wholly outside the image) and the tables
        // are built in registers -- the neighbour words come from shuffles, nothing is read back from shared memory
        const int gx = x0 + 4 * lane;
        const bool colok = lane < pitch && gx >= 0 && gx < W;
        const uint8_t* colp = src + gx;                                // this lane's column (dereferenced only when colok)
        const unsigned sbase = smem_u32(smem) + (unsigned)(lane * 4);
        const unsigned lw4 = (unsigned)level_words * 4u;
#pragma unroll 4
        for (int ry = warp; ry < RH; ry += NT / 32) {
            const int gy = y0 + ry;
            unsigned v = ident;
            if (colok && (unsigned)gy < (unsigned)H) v = __ldg(reinterpret_cast<const unsigned*>(colp + (size_t)gy * W));
            const unsigned row = sbase + (unsigned)(ry * pitch * 4);
            if (lane < pitch) sts_dyn(row, v);
#pragma unroll
            for (int l = 1; l < MAX_TABLES; ++l) {
                if (l < ntables) {
                    const int step = 1 << (l - 1);                         // bytes (compile time)
                    const int ws = step < 4 ? 1 : (step >> 2);             // words to the partner
                    unsigned nxt = __shfl_down_sync(0xffffffffu, v, ws);
                    if (lane + ws >= pitch) nxt = ident;
                    const unsigned bb = step < 4 ? __funnelshift_r(v, nxt, step * 8) : nxt;
                    // op on the four bytes through the 16-bit lanes of the DPX instruction
                    const unsigned be = prmt(bb, 0u, 0x2200u), bo = prmt(bb, 0u, 0x3311u);
                    const unsigned e = vop3_16<IS_MAX>(prmt(v, 0u, 0x2200u), be, be);
                    const unsigned o = vop3_16<IS_MAX>(prmt(v, 0u, 0x3311u), bo, bo);
                    v = pack_lanes(e, o);
                    if (lane < pitch) sts_dyn(row + l * lw4, v);
                }
            }
        }
    } else {
        if (in_c == 1 && (W & 3) == 0 && (reinterpret_cast<uintptr_t>(in) & 3) == 0) {
            for (int ry = warp; ry < RH; ry += NT / 32) {
                const int gy = y0 + ry;
                const bool rowok = gy >= 0 && gy < H;
                for (int rxw = lane; rxw < pitch; rxw += 32) {
                    const int gx = x0 + 4 * rxw;
                    unsigned v = ident;
                    if (rowok && gx >= 0 && gx < W) v = __ldg(reinterpret_cast<const unsigned*>(src + (size_t)gy * W + gx));
                    smem[ry * pitch + rxw] = v;
                }
            }
        } else {
            uint8_t* s8 = reinterpret_cast<uint8_t*>(smem);
            for (int ry = warp; ry < RH; ry += NT / 32) {
                const int gy = y0 + ry;
                const bool rowok = gy >= 0 && gy < H;
                for (int rx = lane; rx < pitch * 4; rx += 32) {
                    const int gx = x0 + rx;
                    uint8_t v = IS_MAX ? 0 : 255;
                    if (rowok && gx >= 0 && gx < W) v = src[((size_t)gy * W + gx) * in_c];
                    s8[ry * pitch * 4 + rx] = v;
                }
            }
        }
        __syncthreads();
        for (int ry = warp; ry < RH; ry += NT / 32) {          // a row is built by the warp that owns it
            unsigned* row = smem + ry * pitch;
            for (int l = 1; l < ntables; ++l) {
                const unsigned* prev = row + (l - 1) * level_words;
                unsigned* cur = row + l * level_words;
                const int step = 1 << (l - 1);           // bytes
                for (int rxw = lane; rxw < pitch; rxw += 32) {
                    const unsigned a = prev[rxw];
                    unsigned bb;
                    if (step < 4) {
                        const unsigned nxt = (rxw + 1 < pitch) ? prev[rxw + 1] : ident;
                        bb = __funnelshift_r(a, nxt, step * 8);
                    } else {
                        const int ws = step >> 2;
                        bb = (rxw + ws < pitch) ? prev[rxw + ws] : ident;
                    }
                    cur[rxw] = vop<IS_MAX>(a, bb);
                }
                __syncwarp();
            }
        }
    }
    __syncthreads();

    // ---- chords ----
    // lane -> (row within a 32-row group, word of the row): half-warps work on rows 16 apart, which an odd table
    // pitch and the chord-table pitch of 17 words put on disjoint banks.  Rows >= RH of the last group compute on
    // whatever follows the tables in shared memory and land in chord-table rows nobody reads.
    const int xw = lane & 15;
    const int row0 = warp + 16 * (lane >> 4);
    unsigned he[NA], ho[NA];                      // running chord minimum of this thread's region rows (16-bit lanes)
    unsigned ae[NB], ao[NB];                      // result of this thread's output rows
#pragma unroll
    for (int it = 0; it < NA; ++it) he[it] = ho[it] = ident;
#pragma unroll
    for (int it = 0; it < NB; ++it) ae[it] = ao[it] = ident;
    const unsigned abase = smem_u32(smem) + (unsigned)((row0 * pitch + xw) * 4);
    const unsigned astep = (unsigned)(32 * pitch * 4);          // bytes between a thread's rows in a range table (an
                                                                // immediate when PITCH is a template constant)
    const unsigned hbase = smem_u32(hbuf) + (unsigned)((row0 * HP + xw) * 4);
    constexpr int HSTEP = 32 * HP * 4;            // bytes between a thread's rows in a chord table
    const int nchords = se.nchords;
    for (int m = 0; m < nchords; ++m) {
        const Chord& ch = se.chord[m];
        const unsigned hb = hbase + (unsigned)((m & 1) * hwords * 4);
        const unsigned w0 = abase + (unsigned)ch.f[0].woff * 4u, w1 = abase + (unsigned)ch.f[1].woff * 4u;
        const unsigned e0 = ch.f[0].sel_e, o0 = ch.f[0].sel_o, e1 = ch.f[1].sel_e, o1 = ch.f[1].sel_o;
        if (ch.nf <= 2) {
            // loads of a group of rows first, arithmetic after: one shared-memory latency per group, not per row
            constexpr int G = 3;
#pragma unroll
            for (int g0 = 0; g0 < NA; g0 += G) {
                unsigned a0[G], a1[G], b0[G], b1[G];
#pragma unroll
                for (int u = 0; u < G; ++u) {
                    if (g0 + u < NA) {
                        const unsigned pa = w0 + (g0 + u) * astep, pb = w1 + (g0 + u) * astep;
                        a0[u] = lds<0>(pa); a1[u] = lds<4>(pa); b0[u] = lds<0>(pb); b1[u] = lds<4>(pb);
                    }
                }
#pragma unroll
                for (int u = 0; u < G; ++u) {
                    if (g0 + u < NA) {
                        const int it = g0 + u;
                        he[it] = vop3_16<IS_MAX>(he[it], prmt(a0[u], a1[u], e0), prmt(b0[u], b1[u], e1));
                        ho[it] = vop3_16<IS_MAX>(ho[it], prmt(a0[u], a1[u], o0), prmt(b0[u], b1[u], o1));
                        sts_dyn(hb + it * HSTEP, pack_lanes(he[it], ho[it]));
                    }
                }
            }
        } else {
            const unsigned w2 = abase + (unsigned)ch.f[2].woff * 4u, w3 = abase + (unsigned)ch.f[3].woff * 4u;
            const unsigned e2 = ch.f[2].sel_e, o2 = ch.f[2].sel_o, e3 = ch.f[3].sel_e, o3 = ch.f[3].sel_o;
#pragma unroll
            for (int it = 0; it < NA; ++it) {
                const unsigned pa = w0 + it * astep, pb = w1 + it * astep, pc = w2 + it * astep, pd = w3 + it * astep;
                const unsigned a0 = lds<0>(pa), a1 = lds<4>(pa), b0 = lds<0>(pb), b1 = lds<4>(pb);
                const unsigned c0 = lds<0>(pc), c1 = lds<4>(pc), d0 = lds<0>(pd), d1 = lds<4>(pd);
                he[it] = vop3_16<IS_MAX>(he[it], prmt(a0, a1, e0), prmt(b0, b1, e1));
                ho[it] = vop3_16<IS_MAX>(ho[it], prmt(a0, a1, o0), prmt(b0, b1, o1));
                he[it] = vop3_16<IS_MAX>(he[it], prmt(c0, c1, e2), prmt(d0, d1, e3));
                ho[it] = vop3_16<IS_MAX>(ho[it], prmt(c0, c1, o2), prmt(d0, d1, o3));
                sts_dyn(hb + it * HSTEP, pack_lanes(he[it], ho[it]));
            }
        }
        __syncthreads();
        // every element row of this width, at the same x: aligned words of the chord table, two rows per step (the
        // plan pads an odd count by repeating its last row: min / max do not care)
        const int jend = ch.row_end;
        for (int j = ch.row_begin; j < jend; j += 2) {
            const unsigned q0 = hb + (unsigned)se.rowoff[j];
            const unsigned q1 = hb + (unsigned)se.rowoff[j + 1];
            unsigned v0[NB], v1[NB];
#pragma unroll
            for (int it = 0; it < NB; ++it) { v0[it] = lds_dyn(q0 + it * HSTEP); v1[it] = lds_dyn(q1 + it * HSTEP); }
#pragma unroll
            for (int it = 0; it < NB; ++it) {
                ae[it] = vop3_16<IS_MAX>(ae[it], prmt(v0[it], 0u, 0x2200u), prmt(v1[it], 0u, 0x2200u));
                ao[it] = vop3_16<IS_MAX>(ao[it], prmt(v0[it], 0u, 0x3311u), prmt(v1[it], 0u, 0x3311u));
            }
        }
        // (no second barrier: the next chord writes the other buffer, and the one after that is behind the
        //  next chord's barrier)
    }

    // ---- write (and, for the second pass, subtract + reduce) ----
    int mn = 255, mx = 0;
    const int gx = blockIdx.x * TW + 4 * xw;
#pragma unroll
    for (int it = 0; it < NB; ++it) {
        const int ly = it * 32 + row0;
        const int gy = blockIdx.y * TH + ly;
        if (gy < H && gx < W) {
            const unsigned acc = pack_lanes(ae[it], ao[it]);
            uint8_t* dst = out + ((size_t)plane * H + gy) * W + gx;
            unsigned res = acc;
            if (SUBTRACT) {
                const int ob = plane / orig_c, oc = plane % orig_c;
                const uint8_t* o = orig + ((size_t)ob * H * W + (size_t)gy * W + gx) * orig_c + oc;
                unsigned ov = 0;
                if (orig_c == 1 && gx + 3 < W && ((reinterpret_cast<uintptr_t>(o) & 3) == 0)) {
                    ov = __ldg(reinterpret_cast<const unsigned*>(o));
                } else {
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        if (gx + q < W) ov |= (unsigned)o[(size_t)q * orig_c] << (8 * q);
                }
                res = __vsubus4(ov, acc);            // cv2.subtract saturates at 0
            }
            if (gx + 3 < W && ((reinterpret_cast<uintptr_t>(dst) & 3) == 0)) {
                *reinterpret_cast<unsigned*>(dst) = res;
                if (SUBTRACT) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int v = (res >> (8 * q)) & 0xff;
                        mn = min(mn, v); mx = max(mx, v);
                    }
                }
            } else {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    if (gx + q < W) {
                        const int v = (res >> (8 * q)) & 0xff;
                        dst[q] = (uint8_t)v;
                        mn = min(mn, v); mx = max(mx, v);
                    }
                }
            }
        }
    }
    if (SUBTRACT) {
        mn = __reduce_min_sync(0xffffffffu, mn);
        mx = __reduce_max_sync(0xffffffffu, mx);
        if (lane == 0) {
            atomicMin(&minmax[2 * plane], mn);
            atomicMax(&minmax[2 * plane + 1], mx);
        }
    }
}

// cv2.normalize(NORM_MINMAX, 0..255) on u8: scale = 255 * (1/(max-min)) and shift = -min*scale in
// double, then fp32 fma(v, scale, shift) rounded half-to-even (matches cv2 4.13 on every input).
__global__ void __launch_bounds__(256) stretch_kernel(const uint8_t* __restrict__ corr, uint8_t* __restrict__ out,
                                                      int out_c, int H, int W, const int* __restrict__ minmax) {
    __shared__ uint8_t lut[256];
    const int plane = blockIdx.y;
    const int b = plane / out_c, c = plane % out_c;
    {
        int mn = minmax[2 * plane], mx = minmax[2 * plane + 1];
        double scale = (mx - mn) > 0 ? __dmul_rn(255.0, __ddiv_rn(1.0, (double)(mx - mn))) : 0.0;
        double shift = __dsub_rn(0.0, __dmul_rn((double)mn, scale));
        float a = (float)scale, sh = (float)shift;
        int q = __float2int_rn(__fmaf_rn((float)threadIdx.x, a, sh));
        lut[threadIdx.x] = (uint8_t)min(255, max(0, q));
    }
    __syncthreads();
    const size_t HW = (size_t)H * W;
    const uint8_t* src = corr + (size_t)plane * HW;
    uint8_t* dst = out + (size_t)b * HW * out_c + c;
    if (out_c == 1 && (HW & 15) == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0) {
        // planar: 16 pixels per thread and iteration
        const size_t n16 = HW >> 4;
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) {
            const uint4 v = __ldg(reinterpret_cast<const uint4*>(src) + i);
            const unsigned in4[4] = {v.x, v.y, v.z, v.w};
            unsigned o4[4];
#pragma unroll
            for (int q = 0; q < 4; ++q)
                o4[q] = (unsigned)lut[in4[q] & 0xff] | ((unsigned)lut[(in4[q] >> 8) & 0xff] << 8) |
                        ((unsigned)lut[(in4[q] >> 16) & 0xff] << 16) | ((unsigned)lut[in4[q] >> 24] << 24);
            reinterpret_cast<uint4*>(dst)[i] = make_uint4(o4[0], o4[1], o4[2], o4[3]);
        }
        return;
    }
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < HW; i += (size_t)gridDim.x * blockDim.x)
        dst[i * out_c] = lut[src[i]];
}

// ---------------------------------------------------------------- banded pass (any radius up to RB_MAX_K)
constexpr int RB_NT = 512;             // threads per block
constexpr int RB_PIECE = 31;           // pixels of a van Herk block one thread scans (odd: the byte streams of
                                       // neighbouring threads fall on different banks)
constexpr int RB_MAX_K = 2047;         // largest element: covers frames up to 4096^2
constexpr int RB_MAX_BANDS = 1024;     // rectangles of the element (600 at k = 2047)
constexpr int RB_TMAX = 16;            // output rows per block

struct Band { short ya, yb, xa, xb; };  // rows [ya, yb] x columns [xa, xb] relative to the output pixel
struct BandPlan {
    int k, nbands;
    Band band[RB_MAX_BANDS];           // walk order: widest chord (shortest band) first
};

template <bool IS_MAX>
__device__ __forceinline__ uint8_t op8(uint8_t a, uint8_t b) { return IS_MAX ? (a > b ? a : b) : (a < b ? a : b); }

// One morphology pass over T output rows x the full width of one plane (blockIdx.x: row band, blockIdx.y: plane).
// Planes are addressed as in the tiled kernel; SUBTRACT as there.  Shared memory, per output row:
//   V  vp bytes  vertical extremum over the current band Y_m        (word per 4 pixels)
//   A  vp bytes  result so far
//   P  lp bytes  block prefix extrema over u = x' - xa_m in [0, W + |X_m| - 1), blocks [j |X_m|, (j + 1) |X_m|)
//   S  lp bytes  block suffix extrema
//   PC cp bytes  per piece of RB_PIECE pixels: extremum of the earlier pieces of its block (blocks wider than a piece)
//   SC cp bytes  ... of the later pieces
// Output x then takes op(S[x], P[x + |X_m| - 1]): the window [x + xa, x + xb] is the suffix of one block and the
// prefix of the next (or all of one block).
template <bool IS_MAX, bool SUBTRACT>
__global__ void __launch_bounds__(RB_NT) morph_band_kernel(const uint8_t* __restrict__ in, int in_c,
                                                           uint8_t* __restrict__ out, const uint8_t* __restrict__ orig,
                                                           int orig_c, int H, int W, int T, int vp, int lp, int cp,
                                                           int* __restrict__ minmax, const __grid_constant__ BandPlan bp) {
    extern __shared__ __align__(16) uint8_t bsm[];
    uint8_t* V = bsm;
    uint8_t* A = V + T * vp;
    uint8_t* P = A + T * vp;
    uint8_t* S = P + T * lp;
    uint8_t* PC = S + T * lp;
    uint8_t* SC = PC + T * cp;
    unsigned* V32 = reinterpret_cast<unsigned*>(V);
    unsigned* A32 = reinterpret_cast<unsigned*>(A);
    const unsigned* P32 = reinterpret_cast<const unsigned*>(P);
    const unsigned* S32 = reinterpret_cast<const unsigned*>(S);
    const int vpw = vp >> 2, lpw = lp >> 2;

    const unsigned ident = IS_MAX ? 0u : 0xffffffffu;
    const uint8_t id8 = IS_MAX ? 0 : 255;
    const int tid = threadIdx.x, plane = blockIdx.y, y0 = blockIdx.x * T;
    const int b = plane / in_c, c = plane % in_c;
    if (!SUBTRACT && minmax && blockIdx.x == 0 && tid == 0) {
        minmax[2 * plane] = 255;                 // the dilate pass (a later launch) reduces into these
        minmax[2 * plane + 1] = 0;
    }
    const uint8_t* src = in + (size_t)b * H * W * in_c + c;
    const bool vec = in_c == 1 && (W & 3) == 0 && (reinterpret_cast<uintptr_t>(in) & 3) == 0;
    const int ww = (W + 3) >> 2, nw = T * ww;    // words per row, words of the band

    // op of source row yy into the word xw of a V row (identity outside the image)
    auto fold = [&](unsigned v, int yy, int xw) -> unsigned {
        if ((unsigned)yy >= (unsigned)H) return v;
        unsigned w;
        if (vec) {
            w = __ldg(reinterpret_cast<const unsigned*>(src + (size_t)yy * W) + xw);
        } else {
            w = 0;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int x = 4 * xw + q;
                const unsigned p = x < W ? src[((size_t)yy * W + x) * in_c] : id8;
                w |= p << (8 * q);
            }
        }
        return vop<IS_MAX>(v, w);
    };

    const int K = bp.nbands;
    int pya = bp.band[0].ya, pyb = bp.band[0].yb;          // band folded into V
    for (int i = tid; i < nw; i += RB_NT) {
        const int t = i / ww, xw = i - t * ww, y = y0 + t;
        unsigned v = ident;
        for (int dy = pya; dy <= pyb; ++dy) v = fold(v, y + dy, xw);
        V32[t * vpw + xw] = v;
        A32[t * vpw + xw] = ident;
    }
    __syncthreads();

    for (int m = 0; m < K; ++m) {
        const int xa = bp.band[m].xa, w = bp.band[m].xb - xa + 1, L = W + w - 1;
        const int nb = (L + w - 1) / w, np = (w + RB_PIECE - 1) / RB_PIECE, npr = nb * np;
        // 1. prefix and suffix extrema of every piece (u outside the image's columns is the identity)
        for (int i = tid; i < T * npr; i += RB_NT) {
            const int t = i / npr, r = i - t * npr, blk = r / np, pc = r - blk * np;
            const int bs = blk * w, u0 = bs + pc * RB_PIECE;
            if (u0 >= L) continue;
            const int u1 = min(min(u0 + RB_PIECE, bs + w), L);
            const uint8_t* vr = V + t * vp;
            uint8_t* pr = P + t * lp;
            uint8_t* sr = S + t * lp;
            uint8_t run = id8;
            for (int u = u0; u < u1; ++u) {
                const int x = u + xa;
                run = op8<IS_MAX>(run, (unsigned)x < (unsigned)W ? vr[x] : id8);
                pr[u] = run;
            }
            run = id8;
            for (int u = u1 - 1; u >= u0; --u) {
                const int x = u + xa;
                run = op8<IS_MAX>(run, (unsigned)x < (unsigned)W ? vr[x] : id8);
                sr[u] = run;
            }
        }
        __syncthreads();
        if (np > 1) {
            // 2. blocks of several pieces: carry the extrema of the other pieces of the block into P and S
            for (int i = tid; i < T * nb; i += RB_NT) {
                const int t = i / nb, blk = i - t * nb, bs = blk * w;
                const int npb = min(np, (L - bs + RB_PIECE - 1) / RB_PIECE);     // pieces of this block inside [0, L)
                const uint8_t* pr = P + t * lp;
                const uint8_t* sr = S + t * lp;
                uint8_t* pcr = PC + t * cp + blk * np;
                uint8_t* scr = SC + t * cp + blk * np;
                uint8_t run = id8;
                for (int q = 0; q < npb; ++q) {
                    pcr[q] = run;
                    run = op8<IS_MAX>(run, pr[min(min(bs + (q + 1) * RB_PIECE, bs + w), L) - 1]);
                }
                run = id8;
                for (int q = npb - 1; q >= 0; --q) {
                    scr[q] = run;
                    run = op8<IS_MAX>(run, sr[bs + q * RB_PIECE]);
                }
            }
            __syncthreads();
            for (int i = tid; i < T * npr; i += RB_NT) {
                const int t = i / npr, r = i - t * npr, blk = r / np, pc = r - blk * np;
                const int bs = blk * w, u0 = bs + pc * RB_PIECE;
                if (u0 >= L) continue;
                const int u1 = min(min(u0 + RB_PIECE, bs + w), L);
                uint8_t* pr = P + t * lp;
                uint8_t* sr = S + t * lp;
                const uint8_t pcv = PC[t * cp + r], scv = SC[t * cp + r];
                for (int u = u0; u < u1; ++u) {
                    pr[u] = op8<IS_MAX>(pr[u], pcv);
                    sr[u] = op8<IS_MAX>(sr[u], scv);
                }
            }
            __syncthreads();
        }
        // 3. fold this rectangle into the result, and grow V to the next rectangle's band
        const bool more = m + 1 < K;
        const int nya = more ? bp.band[m + 1].ya : pya, nyb = more ? bp.band[m + 1].yb : pyb;
        for (int i = tid; i < nw; i += RB_NT) {
            const int t = i / ww, xw = i - t * ww;
            const int e = 4 * xw + w - 1;
            const unsigned sv = S32[t * lpw + xw];
            const unsigned pv = __funnelshift_r(P32[t * lpw + (e >> 2)], P32[t * lpw + (e >> 2) + 1], (e & 3) * 8);
            A32[t * vpw + xw] = vop<IS_MAX>(A32[t * vpw + xw], vop<IS_MAX>(sv, pv));
            if (more) {
                const int y = y0 + t;
                unsigned v = V32[t * vpw + xw];
                for (int dy = nya; dy < pya; ++dy) v = fold(v, y + dy, xw);
                for (int dy = pyb + 1; dy <= nyb; ++dy) v = fold(v, y + dy, xw);
                V32[t * vpw + xw] = v;
            }
        }
        pya = nya;
        pyb = nyb;
        __syncthreads();
    }

    // ---- write (and, for the second pass, subtract + reduce) ----
    int mn = 255, mx = 0;
    for (int i = tid; i < nw; i += RB_NT) {
        const int t = i / ww, xw = i - t * ww, gy = y0 + t, gx = 4 * xw;
        if (gy >= H) continue;
        const unsigned acc = A32[t * vpw + xw];
        uint8_t* dst = out + ((size_t)plane * H + gy) * W + gx;
        unsigned res = acc;
        if (SUBTRACT) {
            const int ob = plane / orig_c, oc = plane % orig_c;
            const uint8_t* o = orig + ((size_t)ob * H * W + (size_t)gy * W + gx) * orig_c + oc;
            unsigned ov = 0;
            if (orig_c == 1 && gx + 3 < W && ((reinterpret_cast<uintptr_t>(o) & 3) == 0)) {
                ov = __ldg(reinterpret_cast<const unsigned*>(o));
            } else {
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (gx + q < W) ov |= (unsigned)o[(size_t)q * orig_c] << (8 * q);
            }
            res = __vsubus4(ov, acc);            // cv2.subtract saturates at 0
        }
        if (gx + 3 < W && ((reinterpret_cast<uintptr_t>(dst) & 3) == 0)) {
            *reinterpret_cast<unsigned*>(dst) = res;
            if (SUBTRACT) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int v = (res >> (8 * q)) & 0xff;
                    mn = min(mn, v); mx = max(mx, v);
                }
            }
        } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (gx + q < W) {
                    const int v = (res >> (8 * q)) & 0xff;
                    dst[q] = (uint8_t)v;
                    mn = min(mn, v); mx = max(mx, v);
                }
            }
        }
    }
    if (SUBTRACT) {
        mn = __reduce_min_sync(0xffffffffu, mn);
        mx = __reduce_max_sync(0xffffffffu, mx);
        if ((tid & 31) == 0) {
            atomicMin(&minmax[2 * plane], mn);
            atomicMax(&minmax[2 * plane + 1], mx);
        }
    }
}

// Element rows of cv2.getStructuringElement(MORPH_ELLIPSE, (k, k)) (OpenCV: dx = cvRound(c * sqrt((r^2 - dy^2) / r^2)),
// j1 = max(c - dx, 0), j2 = min(c + dx + 1, k)) turned into the chord plan of morph_chord_kernel.
int build_plan(int k, int th, SEPlan* se) {
    memset(se, 0, sizeof(*se));
    const int r = k / 2, c = k / 2;
    const double inv_r2 = r ? 1.0 / ((double)r * r) : 0.0;
    int lo[MAX_ROWS], hi[MAX_ROWS];
    if (k > MAX_ROWS) return -1;
    for (int i = 0; i < k; ++i) {
        const int dy = i - r;
        const int dx = (int)nearbyint(c * sqrt(((double)r * r - (double)dy * dy) * inv_r2));   // cvRound
        const int j1 = c - dx < 0 ? 0 : c - dx;
        const int j2 = c + dx + 1 > k ? k : c + dx + 1;
        if (j2 - j1 <= 0) return -1;
        lo[i] = j1 - c;                   // columns [lo, hi] relative to the output pixel
        hi[i] = j2 - 1 - c;
    }
    se->k = k;
    se->an = c;
    se->pad = (4 - (c & 3)) & 3;          // extra columns on the left: the region starts on a 4-pixel boundary
    se->th = th;
    se->RH = th + k - 1;
    const int RW = TW + k - 1 + se->pad;
    se->pitch = ((RW - 1) >> 2) + 2;      // words per region row (+1 so that the two-word window fetch stays in-row)
    if ((se->pitch & 1) == 0) ++se->pitch;   // odd: rows 16 apart fall on disjoint banks
    se->level_words = se->pitch * se->RH;

    // distinct chords, narrowest first; they must be nested
    bool used[MAX_ROWS] = {false};
    int nrows = 0, maxtab = 0;
    int plo = 0, phi = -1;                // previous chord (empty)
    for (int m = 0;; ++m) {
        int best = -1;
        for (int i = 0; i < k; ++i)
            if (!used[i] && (best < 0 || hi[i] - lo[i] < hi[best] - lo[best])) best = i;
        if (best < 0) break;
        if (m >= MAX_CHORDS) return -1;
        const int clo = lo[best], chi = hi[best];
        if (m > 0 && (clo > plo || chi < phi)) return -1;          // not nested: cannot happen for cv2's ellipse
        Chord& ch = se->chord[m];
        ch.nf = 0;
        auto window = [&](int a, int b) {          // min over columns [a, b]: one or two power-of-two tables
            const int w = b - a + 1;
            if (w <= 0) return;
            int l = 0;
            while ((2 << l) <= w) ++l;             // 2^l <= w < 2^(l+1)
            if (l > maxtab) maxtab = l;
            const int starts[2] = {a, b - (1 << l) + 1};
            for (int q = 0; q < ((1 << l) == w ? 1 : 2); ++q) {
                const int bx = starts[q] + c + se->pad;            // byte column inside the region row
                Fetch f;
                const unsigned sb = (unsigned)(bx & 3);             // first byte of the window inside the word pair
                f.woff = l * se->level_words + (bx >> 2);
                f.sel_e = sb | (sb << 4) | ((sb + 2) << 8) | ((sb + 2) << 12);          // bytes s, s, s+2, s+2
                f.sel_o = (sb + 1) | ((sb + 1) << 4) | ((sb + 3) << 8) | ((sb + 3) << 12);
                ch.f[ch.nf++] = f;
            }
        };
        if (m == 0) {
            window(clo, chi);
        } else {
            window(clo, plo - 1);
            const int nleft = ch.nf;
            window(phi + 1, chi);
            if (nleft == 1 && ch.nf > 1) {         // keep pairs together: slots (0,1) and (2,3) are consumed as pairs
                // 1 left + 1 right -> one pair; 1 left + 2 right -> left, left | right, right
                if (ch.nf == 3) { ch.f[3] = ch.f[2]; ch.f[2] = ch.f[1]; ch.f[1] = ch.f[0]; ch.nf = 4; }
            }
        }
        if (ch.nf == 0) return -1;
        if (ch.nf == 1) { ch.f[1] = ch.f[0]; }
        if (ch.nf == 3) { ch.f[3] = ch.f[2]; }
        if (ch.nf <= 2) { ch.f[2] = ch.f[0]; ch.f[3] = ch.f[0]; }
        ch.row_begin = nrows;
        for (int i = 0; i < k; ++i)
            if (!used[i] && lo[i] == clo && hi[i] == chi) {
                used[i] = true;
                se->rowoff[nrows++] = i * HP * 4;                  // (dy + an) * HP words, in bytes (dy = i - an)
            }
        if ((nrows - ch.row_begin) & 1) { se->rowoff[nrows] = se->rowoff[nrows - 1]; ++nrows; }
        ch.row_end = nrows;
        plo = clo; phi = chi;
        se->nchords = m + 1;
    }
    se->ntables = maxtab + 1;
    if (se->ntables > MAX_TABLES) return -1;
    // the window fetches address the tables relative to a lane's own word: woff is used as p[woff], p = table 0 + row + xw
    return 0;
}

// The rectangles Y_m x X_m of the k x k ellipse (same cvRound rows as build_plan), widest chord first.  Fails (-1)
// unless the rows are nested intervals and each Y_m is one contiguous band through the anchor row.
int build_bands(int k, BandPlan* bp) {
    if (k < 1 || k > RB_MAX_K) return -1;
    const int r = k / 2, c = k / 2;
    const double inv_r2 = r ? 1.0 / ((double)r * r) : 0.0;
    int lo[RB_MAX_K], hi[RB_MAX_K], order[RB_MAX_K];
    for (int i = 0; i < k; ++i) {
        const int dy = i - r;
        const int dx = (int)nearbyint(c * sqrt(((double)r * r - (double)dy * dy) * inv_r2));   // cvRound
        const int j1 = c - dx < 0 ? 0 : c - dx;
        const int j2 = c + dx + 1 > k ? k : c + dx + 1;
        if (j2 - j1 <= 0) return -1;
        lo[i] = j1 - c;
        hi[i] = j2 - 1 - c;
        order[i] = i;
    }
    std::sort(order, order + k, [&](int a, int b) {
        const int wa = hi[a] - lo[a], wb = hi[b] - lo[b];
        return wa != wb ? wa > wb : (lo[a] != lo[b] ? lo[a] < lo[b] : a < b);
    });
    bp->k = k;
    bp->nbands = 0;
    int ya = 1 << 30, yb = -(1 << 30), rows = 0;
    for (int j = 0; j < k;) {
        const int a = lo[order[j]], b = hi[order[j]];
        if (bp->nbands > 0) {
            const Band& p = bp->band[bp->nbands - 1];
            if (a < p.xa || b > p.xb) return -1;                       // not nested
        }
        for (; j < k && lo[order[j]] == a && hi[order[j]] == b; ++j) {   // rows of exactly this interval
            ya = std::min(ya, order[j] - c);
            yb = std::max(yb, order[j] - c);
            ++rows;
        }
        // the rows containing [a, b] are those of this and every wider interval: one band through the anchor
        if (yb - ya + 1 != rows || ya > 0 || yb < 0 || bp->nbands >= RB_MAX_BANDS) return -1;
        bp->band[bp->nbands++] = Band{(short)ya, (short)yb, (short)a, (short)b};
    }
    return 0;
}

int plan_groups(const SEPlan& se) { return (se.th == 128 && se.RH <= 192) ? 6 : 8; }     // NA of the instantiation used
size_t plan_smem_bytes(const SEPlan& se) {
    return ((size_t)se.ntables * se.level_words + 2 * (size_t)(plan_groups(se) * 32) * HP) * 4;
}

size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

}  // namespace

size_t rolling_ball_workspace_bytes(int planes, int H, int W) {
    return 2 * align256((size_t)planes * H * W) + align256(sizeof(int) * 2 * (size_t)planes);
}

// Largest radius the tiled kernel can run: the haloed region of the smallest tile must fit in shared memory and the
// per-thread row state covers 256 region rows.
int rolling_ball_tiled_max_radius() {
    static int cached = 0;
    if (!cached) {
        int best = 1;
        for (int k = 1; k <= MAX_ROWS; ++k) {
            SEPlan se;
            if (32 + k - 1 <= 32 * A_ITS && build_plan(k, 32, &se) == 0 && plan_smem_bytes(se) <= 226 * 1024) best = k;
            else break;
        }
        cached = best;
    }
    return cached;
}

// Host-only dump of the chord plan (tests pin the plan builder on the CPU with a numpy model of the kernel):
// [k, an, pad, pitch, RH, level_words, ntables, nchords, th, HP], then per chord {nf, woff0, shift0, .., woff3, shift3,
// row_begin, row_end}, then rowoff[row_end of the last chord].
int rolling_ball_plan_dump(int radius, int th, int* out, int cap) {
    SEPlan se;
    DC_REQUIRE(out && radius >= 1 && th >= 1 && th <= TH_MAX, DC_EINVAL, "dc_debug_rolling_ball_plan: bad argument");
    DC_REQUIRE(build_plan(radius, th, &se) == 0, DC_EINVAL, "dc_debug_rolling_ball_plan: no plan for radius %d", radius);
    const int nrows = se.chord[se.nchords - 1].row_end;          // (includes the pair padding)
    const int need = 10 + 11 * se.nchords + nrows;
    DC_REQUIRE(cap >= need, DC_EINVAL, "dc_debug_rolling_ball_plan: need %d ints", need);
    int n = 0;
    const int head[10] = {se.k, se.an, se.pad, se.pitch, se.RH, se.level_words, se.ntables, se.nchords, se.th, HP};
    for (int v : head) out[n++] = v;
    for (int m = 0; m < se.nchords; ++m) {
        const Chord& ch = se.chord[m];
        out[n++] = ch.nf;
        for (int q = 0; q < 4; ++q) { out[n++] = ch.f[q].woff; out[n++] = (int)(ch.f[q].sel_e & 3u) * 8; }
        out[n++] = ch.row_begin;
        out[n++] = ch.row_end;
    }
    for (int j = 0; j < nrows; ++j) out[n++] = se.rowoff[j] / 4;
    return n;
}

int rolling_ball_max_radius() { return RB_MAX_K; }

// Host-only dump of the banded pass's rectangles: [k, K, RB_PIECE], then {ya, yb, xa, xb} per rectangle in walk order.
int rolling_ball_bands_dump(int radius, int* out, int cap) {
    static BandPlan bp;                       // 8 KB: off the stack (host-only test aid)
    DC_REQUIRE(out && radius >= 1 && radius <= RB_MAX_K, DC_EINVAL, "dc_debug_rolling_ball_bands: radius %d outside [1,%d]",
               radius, RB_MAX_K);
    DC_REQUIRE(build_bands(radius, &bp) == 0, DC_EINVAL, "dc_debug_rolling_ball_bands: no rectangle cover for radius %d", radius);
    const int need = 3 + 4 * bp.nbands;
    DC_REQUIRE(cap >= need, DC_EINVAL, "dc_debug_rolling_ball_bands: need %d ints", need);
    int n = 0;
    out[n++] = bp.k; out[n++] = bp.nbands; out[n++] = RB_PIECE;
    for (int m = 0; m < bp.nbands; ++m) {
        const Band& r = bp.band[m];
        out[n++] = r.ya; out[n++] = r.yb; out[n++] = r.xa; out[n++] = r.xb;
    }
    return n;
}

static int check_rolling_ball_args(const dc_rolling_ball_args_t* a, const char* who, int max_radius) {
    DC_REQUIRE(a && a->in && a->out, DC_EINVAL, "%s: null pointer argument", who);
    DC_REQUIRE(a->B > 0 && a->H > 0 && a->W > 0 && a->C > 0, DC_EINVAL, "%s: bad shape", who);
    DC_REQUIRE(a->radius >= 1 && a->radius <= max_radius, DC_EINVAL, "%s: radius %d outside [1,%d]", who, a->radius, max_radius);
    DC_REQUIRE((long long)a->B * a->C <= 65535, DC_EINVAL, "%s: more than 65535 planes in one call", who);
    DC_REQUIRE((long long)a->H * a->W < (1ll << 31), DC_EINVAL, "%s: image too large for int32 indices", who);
    DC_REQUIRE(a->workspace && a->workspace_bytes >= rolling_ball_workspace_bytes(a->B * a->C, a->H, a->W), DC_EWORKSPACE,
               "%s: workspace too small", who);
    return DC_OK;
}

// blocks per plane of the stretch pass: one per 16 K pixels, 1..1024 (the pixel count is up to 2^31 - 1)
static int stretch_blocks(int H, int W) {
    const long long n = ((long long)H * W + 256 * 64 - 1) / (256 * 64);
    return (int)std::min(std::max(n, 1ll), 1024ll);
}

// erode in -> er, dilate er -> corr with the subtract and the per-plane min / max, stretch corr -> out: the banded
// pass in place of the tiled one, same workspace.
int launch_rolling_ball_banded(const dc_rolling_ball_args_t* a, cudaStream_t stream, const char* who) {
    int rc = check_rolling_ball_args(a, who, RB_MAX_K);
    if (rc != DC_OK) return rc;
    const int planes = a->B * a->C, H = a->H, W = a->W;
    DC_REQUIRE(W <= DC_ROLLING_BALL_BANDED_MAX_WIDTH, DC_EINVAL,
               "%s: rows of %d pixels are wider than the %d the banded pass (radius > %d) keeps in shared memory",
               who, W, DC_ROLLING_BALL_BANDED_MAX_WIDTH, rolling_ball_tiled_max_radius());
    thread_local BandPlan bp;
    DC_REQUIRE(build_bands(a->radius, &bp) == 0, DC_EINVAL, "%s: no rectangle cover for radius %d", who, a->radius);

    // shared memory per output row (morph_band_kernel): V, A, P, S and the piece carries
    const int ww = (W + 3) >> 2;
    const int vp = 4 * ww;
    int wmax = 0, cmax = 0;
    for (int m = 0; m < bp.nbands; ++m) {
        const int w = bp.band[m].xb - bp.band[m].xa + 1, L = W + w - 1;
        const int np = (w + RB_PIECE - 1) / RB_PIECE;
        wmax = std::max(wmax, w);
        if (np > 1) cmax = std::max(cmax, ((L + w - 1) / w) * np);
    }
    const int lp = (vp + wmax + 8 + 15) & ~15;
    const int cp = (cmax + 15) & ~15;
    auto smem_of = [&](int T) { return (size_t)T * (2 * (size_t)vp + 2 * (size_t)lp + 2 * (size_t)cp); };
    // band height: at most RB_TMAX rows, no taller than the image, two blocks per SM where they fit, and enough
    // blocks for two per SM where the batch allows
    int T = RB_TMAX;
    while (T > 1 && T / 2 >= H) T >>= 1;
    while (T > 1 && (smem_of(T) > 112 * 1024 || (long long)ceil_div(H, T) * planes < 2LL * num_sms())) T >>= 1;
    const size_t smem = smem_of(T);
    DC_REQUIRE(smem <= 226 * 1024, DC_EINVAL, "%s: a %d-pixel row does not fit shared memory", who, W);

    char* p = (char*)a->workspace;
    uint8_t* er = (uint8_t*)p;   p += align256((size_t)planes * H * W);
    uint8_t* corr = (uint8_t*)p; p += align256((size_t)planes * H * W);
    int* minmax = (int*)p;

    static unsigned long long attr_done = 0;
    {
        int dev = 0;
        DC_CUDA(cudaGetDevice(&dev));
        const unsigned long long bit = 1ull << (dev & 63);
        if (!(__atomic_load_n(&attr_done, __ATOMIC_ACQUIRE) & bit)) {      // per (function, device), once
            DC_CUDA(cudaFuncSetAttribute(morph_band_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
            DC_CUDA(cudaFuncSetAttribute(morph_band_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
            __atomic_fetch_or(&attr_done, bit, __ATOMIC_RELEASE);
        }
    }
    const dim3 grid(ceil_div(H, T), planes);
    morph_band_kernel<false, false><<<grid, RB_NT, smem, stream>>>(a->in, a->C, er, nullptr, 0, H, W, T, vp, lp, cp, minmax, bp);
    morph_band_kernel<true, true><<<grid, RB_NT, smem, stream>>>(er, 1, corr, a->in, a->C, H, W, T, vp, lp, cp, minmax, bp);
    const int sblocks = stretch_blocks(H, W);
    stretch_kernel<<<dim3(sblocks, planes), 256, 0, stream>>>(corr, a->out, a->C, H, W, minmax);
    DC_CUDA(cudaGetLastError());
    return DC_OK;
}

// tiled_only: dc_rolling_ball_tiled, which refuses what the tiled kernel cannot run instead of handing it to the
// banded pass (radius > rolling_ball_tiled_max_radius(), more than 65535 rows of tiles)
int launch_rolling_ball(const dc_rolling_ball_args_t* a, cudaStream_t stream, bool tiled_only) {
    const char* who = tiled_only ? "dc_rolling_ball_tiled" : "dc_rolling_ball";
    int rc = check_rolling_ball_args(a, who, tiled_only ? rolling_ball_tiled_max_radius() : RB_MAX_K);
    if (rc != DC_OK) return rc;
    if (a->radius > rolling_ball_tiled_max_radius()) return launch_rolling_ball_banded(a, stream, who);
    const int planes = a->B * a->C, H = a->H, W = a->W;
    // tile height: the tallest whose haloed region fits twice per SM (else once), within the per-thread row state
    SEPlan se;
    int th = 0;
    for (int pass = 0; pass < 2 && !th; ++pass)
        for (int cand = TH_MAX; cand >= 32 && !th; cand >>= 1) {
            if (cand + a->radius - 1 > 32 * A_ITS) continue;
            if (build_plan(a->radius, cand, &se) != 0) continue;
            if (plan_smem_bytes(se) <= (pass == 0 ? 112 * 1024 : 226 * 1024)) th = cand;
            if (cand > 32 && cand / 2 >= H) th = 0;            // a shorter tile already covers the whole image
        }
    DC_REQUIRE(th > 0 && build_plan(a->radius, th, &se) == 0, DC_EINVAL, "%s: no tile fits radius %d", who, a->radius);
    // rows of tiles go in gridDim.y (at most 65535).  A taller frame runs the banded pass, which gives the same
    // result bit for bit and keeps its row bands in gridDim.x; such a frame has H * W < 2^31 and H > 65535 * 32, so
    // its rows are narrower than the banded pass's width limit.
    if (ceil_div(H, th) > 65535) {
        DC_REQUIRE(!tiled_only, DC_EINVAL, "%s: image too tall (%d rows of %d-row tiles at radius %d; at most 65535)", who,
                   ceil_div(H, th), th, a->radius);
        return launch_rolling_ball_banded(a, stream, who);
    }
    const size_t smem = plan_smem_bytes(se);

    char* p = (char*)a->workspace;
    uint8_t* er = (uint8_t*)p;   p += align256((size_t)planes * H * W);
    uint8_t* corr = (uint8_t*)p; p += align256((size_t)planes * H * W);
    int* minmax = (int*)p;

    static unsigned long long attr_done = 0;
    {
        int dev = 0;
        DC_CUDA(cudaGetDevice(&dev));
        const unsigned long long bit = 1ull << (dev & 63);
        if (!(__atomic_load_n(&attr_done, __ATOMIC_ACQUIRE) & bit)) {      // per (function, device), once
#define DC_MORPH_ATTR(nb, na, pi, nt)                                                                                           \
            DC_CUDA(cudaFuncSetAttribute(morph_chord_kernel<false, false, nb, na, pi, nt>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024)); \
            DC_CUDA(cudaFuncSetAttribute(morph_chord_kernel<true, true, nb, na, pi, nt>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
            DC_MORPH_ATTR(4, 6, 31, 3) DC_MORPH_ATTR(4, 6, 0, 0) DC_MORPH_ATTR(4, 8, 0, 0) DC_MORPH_ATTR(2, 8, 0, 0) DC_MORPH_ATTR(1, 8, 0, 0)
#undef DC_MORPH_ATTR
            __atomic_fetch_or(&attr_done, bit, __ATOMIC_RELEASE);
        }
    }
    dim3 grid(ceil_div(W, TW), ceil_div(H, th), planes);
    const int na = plan_groups(se);                            // 32-row groups the instantiation covers
    // the reference's default radius (50; also its neighbours with the same region pitch and table count) runs the
    // instantiation with compile-time shared-memory offsets
    const bool special = th == 128 && na == 6 && se.pitch == 31 && se.ntables == 3;
#define DC_MORPH_LAUNCH(nb, nax, pi, nt, cond)                                                                                    \
    if (th == 32 * nb && na == nax && (cond)) {                                                                                   \
        morph_chord_kernel<false, false, nb, nax, pi, nt><<<grid, NT, smem, stream>>>(a->in, a->C, er, nullptr, 0, H, W, minmax, se); \
        morph_chord_kernel<true, true, nb, nax, pi, nt><<<grid, NT, smem, stream>>>(er, 1, corr, a->in, a->C, H, W, minmax, se);      \
    }
    DC_MORPH_LAUNCH(4, 6, 31, 3, special) DC_MORPH_LAUNCH(4, 6, 0, 0, !special) DC_MORPH_LAUNCH(4, 8, 0, 0, true)
    DC_MORPH_LAUNCH(2, 8, 0, 0, true) DC_MORPH_LAUNCH(1, 8, 0, 0, true)
#undef DC_MORPH_LAUNCH
    const int sblocks = stretch_blocks(H, W);
    stretch_kernel<<<dim3(sblocks, planes), 256, 0, stream>>>(corr, a->out, a->C, H, W, minmax);
    DC_CUDA(cudaGetLastError());
    return DC_OK;
}

}  // namespace dc
