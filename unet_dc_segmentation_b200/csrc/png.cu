// png.cu -- u8 frames -> PNG files on the device (dc_png_encode), byte for byte what cv2.imwrite / cv2.imencode
// write with their default parameters: the mask PNG of quantify_droplets_batch.py:58 and the overlay of :78.
//
// What OpenCV's writer (libpng 1.6 + zlib 1.3) produces, and so what this file reproduces:
//   signature, IHDR (bit depth 8, colour type 0 for [H,W] / 2 for BGR [H,W,3] stored as RGB, no interlace), IDAT chunks
//   of exactly 8192 bytes with a shorter last one, IEND; every row filtered with SUB (None for 1-pixel-wide images, where
//   libpng drops SUB); the zlib stream of deflate level 1, strategy Z_RLE, memLevel 8, whose CMF/FLG libpng rewrites to
//   the smallest window that fits when the filtered data is at most 16384 bytes (optimize_cmf).
//
// Z_RLE makes the encoder parallel.  zlib's deflate_rle only ever matches at distance 1, so its greedy parse is a pure
// function of the maximal runs of equal bytes: a run of R bytes emits one literal, (R-1)/258 matches of 258, then one
// match of r = (R-1) % 258 when r >= 3, else r literals.  memLevel 8 gives lit_bufsize 16384, and zlib flushes a block
// after every 16383 symbols (the final block holds the rest and is empty when 16383 divides the symbol count).  Every
// block then picks stored / fixed / dynamic codes exactly as _tr_flush_block does; the tree code below (build_tree,
// gen_bitlen with its overflow fix-up, scan_tree / send_tree, build_bl_tree) is zlib's trees.c restated as
// __host__ __device__ code, and dc_debug_png_host runs it on the host.
//
// Stored blocks and zlib's `block_start >= 0`: _tr_flush_block only stores a block whose start is still in the window.
// That condition never decides anything here.  A stored block is chosen only when stored_len + 4 <= the fixed-code size
// in bytes, and fixed codes spend at most 9 bits on a literal and 8 + 5 + 5 bits on a match of >= 3 bytes: with at most
// 16383 symbols the block then covers at most 21064 bytes.  block_start goes negative only when the window slides
// (strstart >= 2 * 32768 - 262) past a block that began 32768 bytes earlier, i.e. for blocks longer than 32506 bytes.
// The layout checks the bound anyway: a frame with a stored block over 21064 bytes would get no file written.
//
// Device stages (grid.y = frame; all frames of a batch have one shape): filter + run edges + Adler partials per 4096-byte
// tile; per-frame scans; symbol counts per tile; histograms per deflate block; one thread per block builds its trees;
// per-frame bit layout (64-bit bit offsets); headers and symbols OR'ed into a zeroed per-frame zlib buffer; IDAT chunks
// copied out with one CRC-32 per chunk.  No synchronisation and no allocation: the call can sit in a CUDA graph.
#include "common.cuh"

namespace dc {
namespace {

constexpr int kLCodes = 286, kDCodes = 30, kBLCodes = 19, kHeapSize = 2 * kLCodes + 1;
constexpr int kMaxBits = 15, kMaxBLBits = 7, kEndBlock = 256;
constexpr int kBlockSyms = 16383;          // lit_bufsize - 1 symbols per block (memLevel 8)
constexpr int kMaxStored = 21064;          // see the header comment
constexpr int kChunk = 8192;               // libpng's IDAT size (PNG_ZBUF_SIZE)
constexpr int kTile = 4096, kTileThreads = 256, kPerThread = kTile / kTileThreads;
constexpr int kScanThreads = 1024;

__host__ __device__ __forceinline__ int extra_lbits(int c) {    // length code c - 257
    return c < 8 ? 0 : c == 28 ? 0 : (c - 4) >> 2;
}
__host__ __device__ __forceinline__ int base_length(int c) {    // length - 3 of the code's first length
    if (c == 28) return 255;
    if (c < 8) return c;
    return (4 + (c & 3)) << ((c - 4) >> 2);
}
__host__ __device__ __forceinline__ int length_code(int lc) {   // lc = length - 3 in [0, 255] -> code - 257
    if (lc == 255) return 28;
    int c = 27;
    while (base_length(c) > lc) --c;
    return c;
}
__host__ __device__ __forceinline__ int extra_blbits(int n) { return n == 16 ? 2 : n == 17 ? 3 : n == 18 ? 7 : 0; }
__host__ __device__ __forceinline__ int bl_order(int i) {
    const uint8_t o[kBLCodes] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    return o[i];
}
__host__ __device__ __forceinline__ int static_llen(int n) { return n < 144 ? 8 : n < 256 ? 9 : n < 280 ? 7 : 8; }
// zlib's static_ltree codes (defined over 288 symbols, so 9-bit codes start at 400, not at 396)
__host__ __device__ __forceinline__ uint32_t static_lcode_raw(int n) {
    return n < 144 ? 0x30 + n : n < 256 ? 0x190 + (n - 144) : n < 280 ? n - 256 : 0xC0 + (n - 280);
}
__host__ __device__ __forceinline__ uint32_t bi_reverse(uint32_t code, int len) {
    uint32_t r = 0;
    for (int i = 0; i < len; ++i) {
        r = (r << 1) | (code & 1);
        code >>= 1;
    }
    return r;
}

// ---------------------------------------------------------------- filter (stage 1)
struct Shape {
    int H, W, C;
    int64_t row;     // 1 + W*C filtered bytes per row
    int64_t N;       // H * row
};
__host__ __device__ __forceinline__ Shape make_shape(int H, int W, int C) {
    Shape s{H, W, C, 1 + (int64_t)W * C, 0};
    s.N = s.row * H;
    return s;
}
// byte i of the filtered stream of one frame (img: u8 [H,W] or BGR [H,W,3])
__host__ __device__ __forceinline__ uint8_t filtered_byte(const uint8_t* img, const Shape& s, int64_t i) {
    const int64_t y = i / s.row, col = i - y * s.row;
    const int ft = s.W == 1 ? 0 : 1;
    if (col == 0) return (uint8_t)ft;
    const int64_t k = col - 1;
    const int64_t x = k / s.C;
    const int ch = (int)(k - x * s.C);
    const int src = s.C == 3 ? 2 - ch : 0;            // BGR in, RGB out
    const uint8_t* r = img + y * (int64_t)s.W * s.C;
    const uint8_t v = r[x * s.C + src];
    return ft && x > 0 ? (uint8_t)(v - r[(x - 1) * s.C + src]) : v;
}

// ---------------------------------------------------------------- the RLE parse (stage 2)
// Position j (0-based) of a run of R equal bytes: 0 = no symbol starts here, 1 = literal, 2 = match of *len bytes.
__host__ __device__ __forceinline__ int run_symbol(int64_t j, int64_t R, int* len) {
    if (j == 0) return 1;
    const int64_t jj = j - 1, k = jj / 258, t = jj - k * 258, m = (R - 1) / 258;
    const int r = (int)((R - 1) - m * 258);
    if (k < m) {
        *len = 258;
        return t == 0 ? 2 : 0;
    }
    if (r >= 3) {
        *len = r;
        return t == 0 ? 2 : 0;
    }
    return 1;
}

// ---------------------------------------------------------------- Huffman trees (stage 4): zlib's trees.c
struct TreeWork {
    uint16_t freq[kHeapSize];   // ct_data.fc.freq (the code is kept apart)
    uint16_t dl[kHeapSize];     // ct_data.dl: dad, then len
    int heap[kHeapSize];
    uint8_t depth[kHeapSize];
    uint16_t bl_count[kMaxBits + 1];
    int heap_len, heap_max;
    uint64_t opt_len, static_len;
    uint32_t lf[kLCodes], df[kDCodes], blf[kBLCodes];   // plan_block's frequencies
};

__host__ __device__ __forceinline__ bool smaller(const TreeWork& w, int n, int m) {
    return w.freq[n] < w.freq[m] || (w.freq[n] == w.freq[m] && w.depth[n] <= w.depth[m]);
}
__host__ __device__ inline void pqdownheap(TreeWork& w, int k) {
    const int v = w.heap[k];
    int j = k << 1;
    while (j <= w.heap_len) {
        if (j < w.heap_len && smaller(w, w.heap[j + 1], w.heap[j])) j++;
        if (smaller(w, v, w.heap[j])) break;
        w.heap[k] = w.heap[j];
        k = j;
        j <<= 1;
    }
    w.heap[k] = v;
}

// kind: 0 literal/length, 1 distance, 2 bit length.  freq_in[elems] -> len[elems]; returns max_code; *overflow set when
// gen_bitlen had to limit the code lengths.
__host__ __device__ inline int build_tree(TreeWork& w, int kind, const uint32_t* freq_in, uint8_t* len, bool* overflowed) {
    const int elems = kind == 0 ? kLCodes : kind == 1 ? kDCodes : kBLCodes;
    const int max_length = kind == 2 ? kMaxBLBits : kMaxBits;
    int max_code = -1;
    w.heap_len = 0;
    w.heap_max = kHeapSize;
    for (int n = 0; n < elems; n++) {
        w.freq[n] = (uint16_t)freq_in[n];
        if (freq_in[n] != 0) {
            w.heap[++w.heap_len] = max_code = n;
            w.depth[n] = 0;
        } else {
            w.dl[n] = 0;
        }
    }
    while (w.heap_len < 2) {                          // force at least two codes of non-zero frequency
        const int node = w.heap[++w.heap_len] = (max_code < 2 ? ++max_code : 0);
        w.freq[node] = 1;
        w.depth[node] = 0;
        w.opt_len--;
        if (kind == 0) w.static_len -= static_llen(node);
        else if (kind == 1) w.static_len -= 5;
    }
    for (int n = w.heap_len / 2; n >= 1; n--) pqdownheap(w, n);
    int node = elems;
    do {
        const int n = w.heap[1];                      // pqremove
        w.heap[1] = w.heap[w.heap_len--];
        pqdownheap(w, 1);
        const int m = w.heap[1];
        w.heap[--w.heap_max] = n;
        w.heap[--w.heap_max] = m;
        w.freq[node] = (uint16_t)(w.freq[n] + w.freq[m]);
        w.depth[node] = (uint8_t)((w.depth[n] >= w.depth[m] ? w.depth[n] : w.depth[m]) + 1);
        w.dl[n] = w.dl[m] = (uint16_t)node;
        w.heap[1] = node++;
        pqdownheap(w, 1);
    } while (w.heap_len >= 2);
    w.heap[--w.heap_max] = w.heap[1];

    // gen_bitlen
    for (int b = 0; b <= kMaxBits; b++) w.bl_count[b] = 0;
    w.dl[w.heap[w.heap_max]] = 0;
    int overflow = 0, h;
    for (h = w.heap_max + 1; h < kHeapSize; h++) {
        const int n = w.heap[h];
        int bits = w.dl[w.dl[n]] + 1;
        if (bits > max_length) bits = max_length, overflow++;
        w.dl[n] = (uint16_t)bits;
        if (n > max_code) continue;
        w.bl_count[bits]++;
        int xbits = 0;
        if (kind == 0 && n >= 257) xbits = extra_lbits(n - 257);
        else if (kind == 1 && n >= 4) xbits = (n - 2) >> 1;
        else if (kind == 2) xbits = extra_blbits(n);
        const uint64_t f = w.freq[n];
        w.opt_len += f * (uint64_t)(bits + xbits);
        if (kind == 0) w.static_len += f * (uint64_t)(static_llen(n) + xbits);
        else if (kind == 1) w.static_len += f * (uint64_t)(5 + xbits);
    }
    *overflowed = overflow != 0;
    if (overflow) {
        do {
            int bits = max_length - 1;
            while (w.bl_count[bits] == 0) bits--;
            w.bl_count[bits]--;
            w.bl_count[bits + 1] += 2;
            w.bl_count[max_length]--;
            overflow -= 2;
        } while (overflow > 0);
        h = kHeapSize;
        for (int bits = max_length; bits != 0; bits--) {
            int n = w.bl_count[bits];
            while (n != 0) {
                const int m = w.heap[--h];
                if (m > max_code) continue;
                if (w.dl[m] != (unsigned)bits) {
                    w.opt_len += ((uint64_t)bits - w.dl[m]) * w.freq[m];
                    w.dl[m] = (uint16_t)bits;
                }
                n--;
            }
        }
    }
    for (int n = 0; n < elems; n++) len[n] = (uint8_t)w.dl[n];
    return max_code;
}

// canonical codes (gen_codes), bit-reversed for LSB-first output
__host__ __device__ inline void gen_codes(const uint8_t* len, int max_code, uint16_t* code) {
    uint16_t count[kMaxBits + 1] = {0};
    uint16_t next[kMaxBits + 1];
    for (int n = 0; n <= max_code; n++) count[len[n]]++;
    count[0] = 0;
    uint32_t c = 0;
    for (int b = 1; b <= kMaxBits; b++) {
        c = (c + count[b - 1]) << 1;
        next[b] = (uint16_t)c;
    }
    for (int n = 0; n <= max_code; n++)
        if (len[n]) code[n] = (uint16_t)bi_reverse(next[len[n]]++, len[n]);
}

// scan_tree (bl_freq != NULL) and send_tree (put != NULL) over len[0..max_code] with the guard len[max_code+1] = 0xff..
template <class Put>
__host__ __device__ inline void walk_tree(const uint8_t* len, int max_code, uint32_t* bl_freq, const uint8_t* bl_len,
                                          const uint16_t* bl_code, Put put) {
    int prevlen = -1, count = 0, max_count = 7, min_count = 4;
    int nextlen = len[0];
    if (nextlen == 0) max_count = 138, min_count = 3;
    auto code = [&](int c) {
        if (bl_freq) bl_freq[c]++;
        else put(bl_code[c], bl_len[c]);
    };
    for (int n = 0; n <= max_code; n++) {
        const int curlen = nextlen;
        nextlen = n + 1 <= max_code ? len[n + 1] : 0xffff;
        if (++count < max_count && curlen == nextlen) {
            continue;
        } else if (count < min_count) {
            if (bl_freq) bl_freq[curlen] += count;
            else
                do put(bl_code[curlen], bl_len[curlen]); while (--count != 0);
        } else if (curlen != 0) {
            if (curlen != prevlen) {
                code(curlen);
                count--;
            }
            code(16);
            if (!bl_freq) put(count - 3, 2);
        } else if (count <= 10) {
            code(17);
            if (!bl_freq) put(count - 3, 3);
        } else {
            code(18);
            if (!bl_freq) put(count - 11, 7);
        }
        count = 0;
        prevlen = curlen;
        if (nextlen == 0) max_count = 138, min_count = 3;
        else if (curlen == nextlen) max_count = 6, min_count = 3;
        else max_count = 7, min_count = 4;
    }
}

enum BlockType { kStored = 0, kFixed = 1, kDynamic = 2 };

// One deflate block's codes and sizes, what _tr_flush_block decides.
struct BlockPlan {
    int type;
    int lmax, dmax, blmax_index;
    int overflow;                 // bit 0: literal/length or distance lengths limited to 15, bit 1: bit lengths to 7
    uint8_t llen[kLCodes], dlen[kDCodes], bllen[kBLCodes];
    uint16_t lcode[kLCodes], dcode[kDCodes], blcode[kBLCodes];
    int64_t header_bits;          // compressed blocks: type bits + trees
    int64_t data_bits;            // compressed blocks: symbols, END_BLOCK excluded
};

// hist: literal/length frequencies without END_BLOCK; nmatch: the distance-1 matches; stored_len: the block's bytes
__host__ __device__ inline void plan_block(const uint32_t* hist, uint32_t nmatch, int64_t stored_len, BlockPlan& p,
                                           TreeWork& w) {
    uint32_t* lf = w.lf;
    uint32_t* df = w.df;
    uint32_t* blf = w.blf;
    for (int n = 0; n < kLCodes; n++) lf[n] = hist[n];
    lf[kEndBlock] = 1;
    for (int n = 0; n < kDCodes; n++) df[n] = 0;
    df[0] = nmatch;
    for (int n = 0; n < kBLCodes; n++) blf[n] = 0;
    w.opt_len = w.static_len = 0;
    bool o1, o2, o3;
    p.lmax = build_tree(w, 0, lf, p.llen, &o1);
    p.dmax = build_tree(w, 1, df, p.dlen, &o2);
    walk_tree(p.llen, p.lmax, blf, nullptr, nullptr, [](uint32_t, int) {});
    walk_tree(p.dlen, p.dmax, blf, nullptr, nullptr, [](uint32_t, int) {});
    build_tree(w, 2, blf, p.bllen, &o3);
    int mb;
    for (mb = kBLCodes - 1; mb >= 3; mb--)
        if (p.bllen[bl_order(mb)] != 0) break;
    p.blmax_index = mb;
    w.opt_len += 3 * ((uint64_t)mb + 1) + 5 + 5 + 4;
    p.overflow = (o1 || o2 ? 1 : 0) | (o3 ? 2 : 0);

    uint64_t opt_lenb = (w.opt_len + 3 + 7) >> 3;
    const uint64_t static_lenb = (w.static_len + 3 + 7) >> 3;
    if (static_lenb <= opt_lenb) opt_lenb = static_lenb;
    if ((uint64_t)stored_len + 4 <= opt_lenb) p.type = kStored;
    else if (static_lenb == opt_lenb) p.type = kFixed;
    else p.type = kDynamic;

    if (p.type == kFixed) {
        for (int n = 0; n < kLCodes; n++) p.llen[n] = (uint8_t)static_llen(n);
        for (int n = 0; n < kDCodes; n++) p.dlen[n] = 5;
        p.lmax = kLCodes - 1;
        p.dmax = kDCodes - 1;
    }
    if (p.type == kFixed) {
        for (int n = 0; n < kLCodes; n++) p.lcode[n] = (uint16_t)bi_reverse(static_lcode_raw(n), p.llen[n]);
        for (int n = 0; n < kDCodes; n++) p.dcode[n] = (uint16_t)bi_reverse((uint32_t)n, 5);
    } else {
        gen_codes(p.llen, p.lmax, p.lcode);
        gen_codes(p.dlen, p.dmax, p.dcode);
    }
    gen_codes(p.bllen, kBLCodes - 1, p.blcode);
    if (p.type == kStored) {
        p.header_bits = p.data_bits = 0;
        return;
    }
    int64_t hb = 3;
    if (p.type == kDynamic) {
        hb += 5 + 5 + 4 + 3 * (int64_t)(mb + 1);
        auto count = [&](uint32_t, int n) { hb += n; };
        walk_tree(p.llen, p.lmax, nullptr, p.bllen, p.blcode, count);
        walk_tree(p.dlen, p.dmax, nullptr, p.bllen, p.blcode, count);
    }
    p.header_bits = hb;
    int64_t db = 0;
    for (int n = 0; n < kLCodes; n++)
        if (hist[n]) db += (int64_t)hist[n] * (p.llen[n] + (n >= 257 ? extra_lbits(n - 257) : 0));
    db += (int64_t)nmatch * p.dlen[0];
    p.data_bits = db;
}

// the block's type bits and trees (compressed blocks); put(value, nbits) writes LSB first
template <class Put>
__host__ __device__ inline void put_block_header(const BlockPlan& p, bool last, Put put) {
    put((uint32_t)((p.type == kFixed ? 2 : 4) + (last ? 1 : 0)), 3);
    if (p.type != kDynamic) return;
    put((uint32_t)(p.lmax + 1 - 257), 5);
    put((uint32_t)p.dmax, 5);
    put((uint32_t)(p.blmax_index + 1 - 4), 4);
    for (int r = 0; r <= p.blmax_index; r++) put(p.bllen[bl_order(r)], 3);
    walk_tree(p.llen, p.lmax, nullptr, p.bllen, p.blcode, put);
    walk_tree(p.dlen, p.dmax, nullptr, p.bllen, p.blcode, put);
}

// the bits of one symbol: literal v (kind 1) or match of len bytes (kind 2); returns the bit count, *bits the value
__host__ __device__ __forceinline__ int symbol_bits(const uint16_t* lcode, const uint8_t* llen, uint16_t dcode0,
                                                    int dlen0, int kind, int v, uint64_t* bits) {
    if (kind == 1) {
        *bits = lcode[v];
        return llen[v];
    }
    const int lc = v - 3, c = length_code(lc), sym = 257 + c, e = extra_lbits(c), n = llen[sym];
    *bits = (uint64_t)lcode[sym] | ((uint64_t)(lc - base_length(c)) << n) | ((uint64_t)dcode0 << (n + e));
    return n + e + dlen0;
}

// The code bits of a symbol of a block: none in a stored block, whose bytes are copied as they are.
__host__ __device__ __forceinline__ int block_code_bits(const BlockPlan& p, int kind, int v, uint64_t* bits) {
    if (p.type == kStored) {
        *bits = 0;
        return 0;
    }
    return symbol_bits(p.lcode, p.llen, p.dcode[0], p.dlen[0], kind, v, bits);
}

// ---------------------------------------------------------------- container (stage 6)
__host__ __device__ __forceinline__ uint32_t crc_step(const uint32_t* table, uint32_t c, uint8_t b) {
    return table[(c ^ b) & 0xff] ^ (c >> 8);
}
__host__ __device__ inline void crc_table_fill(uint32_t* t, int i) {
    uint32_t c = (uint32_t)i;
    for (int k = 0; k < 8; k++) c = c & 1 ? 0xEDB88320u ^ (c >> 1) : c >> 1;
    t[i] = c;
}
__host__ __device__ __forceinline__ void put_be32(uint8_t* p, uint32_t v) {
    p[0] = (uint8_t)(v >> 24); p[1] = (uint8_t)(v >> 16); p[2] = (uint8_t)(v >> 8); p[3] = (uint8_t)v;
}
// zlib's CMF/FLG for windowBits 15, level 1, as libpng's optimize_cmf leaves them for `data` filtered bytes
__host__ __device__ inline void zlib_header(int64_t data, uint8_t* h) {
    unsigned cmf = 0x78, flg = 0x01;
    if (data <= 16384) {
        unsigned cinfo = cmf >> 4, half = 1u << (cinfo + 7);
        if (data <= (int64_t)half) {
            do {
                half >>= 1;
                --cinfo;
            } while (cinfo > 0 && data <= (int64_t)half);
            cmf = (cmf & 0x0f) | (cinfo << 4);
            const unsigned t = flg & 0xe0;
            flg = t + 0x1f - ((cmf << 8) + t) % 0x1f;
        }
    }
    h[0] = (uint8_t)cmf;
    h[1] = (uint8_t)flg;
}
__host__ __device__ __forceinline__ int64_t png_bytes_for(int64_t zbytes) {
    return 8 + 25 + zbytes + 12 * ((zbytes + kChunk - 1) / kChunk) + 12;
}
// signature + IHDR (33 bytes)
__host__ __device__ inline void write_png_head(uint8_t* o, const Shape& s, const uint32_t* crc_t) {
    const uint8_t sig[8] = {0x89, 'P', 'N', 'G', '\r', '\n', 0x1a, '\n'};
    for (int i = 0; i < 8; i++) o[i] = sig[i];
    put_be32(o + 8, 13);
    o[12] = 'I'; o[13] = 'H'; o[14] = 'D'; o[15] = 'R';
    put_be32(o + 16, (uint32_t)s.W);
    put_be32(o + 20, (uint32_t)s.H);
    o[24] = 8; o[25] = s.C == 3 ? 2 : 0; o[26] = 0; o[27] = 0; o[28] = 0;
    uint32_t c = 0xffffffffu;
    for (int i = 12; i < 29; i++) c = crc_step(crc_t, c, o[i]);
    put_be32(o + 29, ~c);
}
__host__ __device__ inline void write_png_tail(uint8_t* o) {
    const uint8_t iend[12] = {0, 0, 0, 0, 'I', 'E', 'N', 'D', 0xAE, 0x42, 0x60, 0x82};
    for (int i = 0; i < 12; i++) o[i] = iend[i];
}
// IDAT chunk c of a zlib stream of zbytes bytes: length, tag, data, CRC (o: the chunk's first byte)
__host__ __device__ inline void write_idat(uint8_t* o, const uint8_t* z, int64_t zbytes, int64_t c, const uint32_t* crc_t) {
    const int64_t beg = c * kChunk;
    const int n = (int)(zbytes - beg < kChunk ? zbytes - beg : kChunk);
    put_be32(o, (uint32_t)n);
    o[4] = 'I'; o[5] = 'D'; o[6] = 'A'; o[7] = 'T';
    uint32_t crc = 0xffffffffu;
    for (int i = 4; i < 8; i++) crc = crc_step(crc_t, crc, o[i]);
    for (int i = 0; i < n; i++) {
        const uint8_t b = z[beg + i];
        o[8 + i] = b;
        crc = crc_step(crc_t, crc, b);
    }
    put_be32(o + 8 + n, ~crc);
}

// ---------------------------------------------------------------- bounds and workspace layout
__host__ __device__ __forceinline__ int64_t max_blocks(int64_t N) { return N / kBlockSyms + 2; }
// a block never costs more than its stored form (3 + 7 + 32 bits + its bytes), see zlib's deflateBound
__host__ __device__ __forceinline__ int64_t zlib_bound(int64_t N) { return 2 + N + 6 * max_blocks(N) + 1 + 4; }

size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

struct TileInfo {
    int32_t first, last;          // first / last run start in the tile (N / -1 when none)
    int32_t carry, next;          // last run start before the tile, first run start after it
    int32_t nsym, symbase;        // symbols starting in the tile, symbols before it
    int64_t bits, bitbase;        // code bits of those symbols (stored blocks: 0), bits before it
    uint64_t ad_s, ad_w;          // Adler-32 partial sums: sum d, sum (len - k) d
};

struct BlockInfo {
    int32_t pos;                  // filtered byte of its first symbol (N for an empty final block)
    int32_t nmatch;
    int64_t start_bit;            // first bit of the block in the zlib stream
    int64_t data_bit;             // first symbol bit (stored: the first data BYTE * 8)
    int64_t cbase;                // code bits of the frame's symbols before the block
    uint32_t hist[kLCodes];
    BlockPlan plan;               // trees, codes and sizes (png_trees_kernel)
};

struct FrameInfo {
    int64_t nsym;
    int64_t nblocks;
    int64_t total_bits;
    int64_t zbytes;
    int64_t png_bytes;
    uint32_t adler;
    int32_t error;
};

struct Layout {
    Shape s;
    int B;
    int64_t nt, nbmax, zcap;      // tiles, blocks, zlib buffer bytes per frame (multiple of 4)
    size_t off_filt, off_tile, off_block, off_frame, off_z, total;
    int64_t filt_stride;
};

inline Layout make_layout(int B, int H, int W, int C) {
    Layout L;
    L.s = make_shape(H, W, C);
    L.B = B;
    L.nt = (L.s.N + kTile - 1) / kTile;
    L.nbmax = max_blocks(L.s.N);
    L.zcap = (zlib_bound(L.s.N) + 8) & ~(int64_t)3;
    L.filt_stride = (L.s.N + 255) & ~(int64_t)255;
    size_t o = 0;
    L.off_filt = o;  o += align256((size_t)B * L.filt_stride);
    L.off_tile = o;  o += align256((size_t)B * L.nt * sizeof(TileInfo));
    L.off_block = o; o += align256((size_t)B * L.nbmax * sizeof(BlockInfo));
    L.off_frame = o; o += align256((size_t)B * sizeof(FrameInfo));
    L.off_z = o;     o += align256((size_t)B * L.zcap);
    L.total = o;
    return L;
}

struct Ptrs {
    Layout L;
    const uint8_t* img;
    uint8_t* filt;
    TileInfo* tile;
    BlockInfo* blk;
    FrameInfo* frame;
    uint32_t* z;                  // zlib streams, zeroed, OR'ed into
    uint8_t* out;
    int64_t out_bytes;
    int64_t* offsets;
};

// ---------------------------------------------------------------- device helpers
__device__ __forceinline__ void or_bits(uint32_t* z, int64_t pos, uint64_t v, int n) {   // n <= 32
    if (n == 0) return;
    const int64_t w = pos >> 5;
    const int sh = (int)(pos & 31);
    const uint64_t x = v << sh;
    if ((uint32_t)x) atomicOr(z + w, (uint32_t)x);
    if (sh + n > 32 && (uint32_t)(x >> 32)) atomicOr(z + w + 1, (uint32_t)(x >> 32));
}
__device__ __forceinline__ void or_byte(uint32_t* z, int64_t byte, uint8_t v) {
    if (v) atomicOr(z + (byte >> 2), (uint32_t)v << (8 * (byte & 3)));
}

// block-wide inclusive scan in shared memory (Hillis-Steele), op: 0 sum, 1 max, 2 min
// (the inclusive results stay in sh[0..NT) until the caller's next write; slot: this thread's place in the order)
template <int NT>
__device__ int64_t block_scan(int64_t v, int op, int64_t* sh, int slot = -1) {
    const int t = slot < 0 ? (int)threadIdx.x : slot;
    sh[t] = v;
    __syncthreads();
    for (int o = 1; o < NT; o <<= 1) {
        const int64_t y = t >= o ? sh[t - o] : 0;
        __syncthreads();
        if (t >= o) {
            const int64_t x = sh[t];
            sh[t] = op == 0 ? x + y : op == 1 ? (x > y ? x : y) : (x < y ? x : y);
        }
        __syncthreads();
    }
    const int64_t r = sh[t];
    __syncthreads();
    return r;
}

// The symbols of the kPerThread positions of one thread in tile t of frame b.  kind[q]: 0 / 1 literal / 2 match,
// val[q]: the literal byte or the match length.  Needs TileInfo.carry / next.
struct ThreadSyms {
    int64_t p0;
    int n;                        // positions of this thread inside the frame
    uint8_t kind[kPerThread];
    int16_t val[kPerThread];
};
__device__ void thread_symbols(const Ptrs& P, int b, int64_t t, ThreadSyms& ts, int64_t* sh) {
    const int64_t N = P.L.s.N;
    const uint8_t* f = P.filt + (int64_t)b * P.L.filt_stride;
    const TileInfo& ti = P.tile[(int64_t)b * P.L.nt + t];
    ts.p0 = t * kTile + (int64_t)threadIdx.x * kPerThread;
    ts.n = (int)(N - ts.p0 < 0 ? 0 : N - ts.p0 < kPerThread ? N - ts.p0 : kPerThread);
    uint8_t v[kPerThread];
    uint32_t starts = 0;
    for (int q = 0; q < ts.n; q++) {
        v[q] = f[ts.p0 + q];
        const int64_t i = ts.p0 + q;
        const bool st = i == 0 || v[q] != (q ? v[q - 1] : f[i - 1]);
        starts |= (uint32_t)st << q;
    }
    const int64_t mylast = starts ? ts.p0 + 31 - __clz((int)starts) : -1;
    const int64_t myfirst = starts ? ts.p0 + __ffs((int)starts) - 1 : INT64_MAX;
    // the run start before my positions: max over earlier threads and the tile's carry
    block_scan<kTileThreads>(mylast, 1, sh);
    int64_t excl_s = threadIdx.x ? sh[threadIdx.x - 1] : -1;
    if (excl_s < ti.carry) excl_s = ti.carry;
    __syncthreads();
    // the run start after my positions: min over later threads (a scan in reverse order) and the tile's next
    const int rslot = kTileThreads - 1 - threadIdx.x;
    block_scan<kTileThreads>(myfirst, 2, sh, rslot);
    int64_t excl_e = rslot ? sh[rslot - 1] : INT64_MAX;
    if (excl_e > ti.next) excl_e = ti.next;
    __syncthreads();
    // walk: next start after each position
    int64_t nexts[kPerThread];
    int64_t e = excl_e;
    for (int q = ts.n - 1; q >= 0; q--) {
        nexts[q] = e;
        if (starts >> q & 1) e = ts.p0 + q;
    }
    int64_t cur = excl_s;
    for (int q = 0; q < kPerThread; q++) {
        ts.kind[q] = 0;
        if (q >= ts.n) continue;
        if (starts >> q & 1) cur = ts.p0 + q;
        int len = 0;
        const int k = run_symbol(ts.p0 + q - cur, nexts[q] - cur, &len);
        ts.kind[q] = (uint8_t)k;
        ts.val[q] = (int16_t)(k == 1 ? v[q] : len);
    }
}

// ---------------------------------------------------------------- kernels
// stage 1: filter, run edges and Adler partial sums per tile
__global__ void __launch_bounds__(kTileThreads) png_filter_kernel(Ptrs P) {
    const int b = blockIdx.y;
    const int64_t t = blockIdx.x, N = P.L.s.N;
    const uint8_t* img = P.img + (int64_t)b * P.L.s.H * P.L.s.W * P.L.s.C;
    uint8_t* f = P.filt + (int64_t)b * P.L.filt_stride;
    const int64_t t0 = t * kTile, tl = N - t0 < kTile ? N - t0 : kTile;
    const int64_t p0 = t0 + (int64_t)threadIdx.x * kPerThread;
    int64_t first = INT64_MAX, last = -1;
    uint64_t as = 0, aw = 0;
    uint8_t prev = p0 > 0 && p0 < N ? filtered_byte(img, P.L.s, p0 - 1) : 0;
    for (int q = 0; q < kPerThread; q++) {
        const int64_t i = p0 + q;
        if (i >= N) break;
        const uint8_t v = filtered_byte(img, P.L.s, i);
        f[i] = v;
        if (i == 0 || v != prev) {
            if (first == INT64_MAX) first = i;
            last = i;
        }
        prev = v;
        as += v;
        aw += (uint64_t)(tl - (i - t0)) * v;
    }
    __shared__ int64_t sh[kTileThreads];
    const int64_t mn = block_scan<kTileThreads>(first, 2, sh);
    const int64_t mx = block_scan<kTileThreads>(last, 1, sh);
    const int64_t ss = block_scan<kTileThreads>((int64_t)as, 0, sh);
    const int64_t sw = block_scan<kTileThreads>((int64_t)aw, 0, sh);
    if (threadIdx.x == kTileThreads - 1) {
        TileInfo& ti = P.tile[(int64_t)b * P.L.nt + t];
        ti.first = (int32_t)(mn == INT64_MAX ? N : mn);
        ti.last = (int32_t)mx;
        ti.ad_s = (uint64_t)ss;
        ti.ad_w = (uint64_t)sw;
    }
}

// exclusive scan over the frame's tiles of one TileInfo field, carried through 1024-thread passes
template <class Get, class Set>
__device__ int64_t frame_scan(int64_t n, int op, int64_t ident, Get get, Set set, int64_t* sh) {
    const int64_t per = (n + kScanThreads - 1) / kScanThreads;
    const int64_t lo = (int64_t)threadIdx.x * per, hi = lo + per < n ? lo + per : n;
    auto comb = [&](int64_t a, int64_t c) { return op == 0 ? a + c : op == 1 ? (a > c ? a : c) : (a < c ? a : c); };
    int64_t agg = ident;
    for (int64_t i = lo; i < hi; i++) agg = comb(agg, get(i));
    const int64_t incl = block_scan<kScanThreads>(agg, op, sh);
    // exclusive prefix of this thread
    sh[threadIdx.x] = incl;
    __syncthreads();
    int64_t run = threadIdx.x ? sh[threadIdx.x - 1] : ident;
    const int64_t total = sh[kScanThreads - 1];
    __syncthreads();
    for (int64_t i = lo; i < hi; i++) {
        const int64_t x = get(i);
        set(i, run);
        run = comb(run, x);
    }
    return total;
}

// per frame: run start before / after every tile, Adler-32
__global__ void __launch_bounds__(kScanThreads) png_scan_runs_kernel(Ptrs P) {
    __shared__ int64_t sh[kScanThreads];
    const int b = blockIdx.x;
    const int64_t nt = P.L.nt, N = P.L.s.N;
    TileInfo* T = P.tile + (int64_t)b * nt;
    frame_scan(nt, 1, -1, [&](int64_t i) { return (int64_t)T[i].last; }, [&](int64_t i, int64_t v) { T[i].carry = (int32_t)v; }, sh);
    // reverse min scan: tile nt-1-i
    frame_scan(nt, 2, N, [&](int64_t i) { return (int64_t)T[nt - 1 - i].first; },
               [&](int64_t i, int64_t v) { T[nt - 1 - i].next = (int32_t)v; }, sh);
    // Adler-32: a = 1 + sum d, b = N + sum over tiles (W_t + (N - end_t) S_t), mod 65521
    uint64_t a = 0, bb = 0;
    for (int64_t i = threadIdx.x; i < nt; i += kScanThreads) {
        const int64_t end = (i + 1) * kTile < N ? (i + 1) * kTile : N;
        a += T[i].ad_s % 65521;
        bb += (T[i].ad_w % 65521 + ((uint64_t)(N - end) % 65521) * (T[i].ad_s % 65521)) % 65521;
    }
    a = (uint64_t)block_scan<kScanThreads>((int64_t)(a % 65521), 0, sh);
    bb = (uint64_t)block_scan<kScanThreads>((int64_t)(bb % 65521), 0, sh);
    if (threadIdx.x == kScanThreads - 1) {
        const uint32_t A = (uint32_t)((1 + a) % 65521), Bv = (uint32_t)((bb + (uint64_t)N % 65521) % 65521);
        P.frame[b].adler = (Bv << 16) | A;
        P.frame[b].error = 0;
    }
}

// stage 2: symbols per tile
__global__ void __launch_bounds__(kTileThreads) png_count_kernel(Ptrs P) {
    __shared__ int64_t sh[kTileThreads];
    ThreadSyms ts;
    thread_symbols(P, blockIdx.y, blockIdx.x, ts, sh);
    int c = 0;
    for (int q = 0; q < kPerThread; q++) c += ts.kind[q] != 0;
    const int64_t tot = block_scan<kTileThreads>(c, 0, sh);
    if (threadIdx.x == kTileThreads - 1) P.tile[(int64_t)blockIdx.y * P.L.nt + blockIdx.x].nsym = (int32_t)tot;
}

__global__ void __launch_bounds__(kScanThreads) png_scan_syms_kernel(Ptrs P) {
    __shared__ int64_t sh[kScanThreads];
    const int b = blockIdx.x;
    TileInfo* T = P.tile + (int64_t)b * P.L.nt;
    const int64_t total = frame_scan(P.L.nt, 0, 0, [&](int64_t i) { return (int64_t)T[i].nsym; },
                                     [&](int64_t i, int64_t v) { T[i].symbase = (int32_t)v; }, sh);
    if (threadIdx.x == 0) {
        const int64_t nb = total / kBlockSyms + 1;
        P.frame[b].nsym = total;
        P.frame[b].nblocks = nb;
        if (total % kBlockSyms == 0) P.blk[(int64_t)b * P.L.nbmax + nb - 1].pos = (int32_t)P.L.s.N;   // empty final block
    }
}

// stage 3: histograms per block, block start positions
__global__ void __launch_bounds__(kTileThreads) png_hist_kernel(Ptrs P) {
    __shared__ int64_t sh[kTileThreads];
    __shared__ uint32_t hist[2][kLCodes];
    __shared__ uint32_t nm[2];
    const int b = blockIdx.y;
    ThreadSyms ts;
    thread_symbols(P, b, blockIdx.x, ts, sh);
    for (int i = threadIdx.x; i < 2 * kLCodes; i += kTileThreads) hist[i / kLCodes][i % kLCodes] = 0;
    if (threadIdx.x < 2) nm[threadIdx.x] = 0;
    int c = 0;
    for (int q = 0; q < kPerThread; q++) c += ts.kind[q] != 0;
    const TileInfo& ti = P.tile[(int64_t)b * P.L.nt + blockIdx.x];
    int64_t idx = ti.symbase + block_scan<kTileThreads>(c, 0, sh) - c;
    const int64_t blk0 = ti.symbase / kBlockSyms;
    BlockInfo* B = P.blk + (int64_t)b * P.L.nbmax;
    for (int q = 0; q < kPerThread; q++) {
        if (!ts.kind[q]) continue;
        const int64_t blk = idx / kBlockSyms;
        if (idx % kBlockSyms == 0) B[blk].pos = (int32_t)(ts.p0 + q);
        const int slot = (int)(blk - blk0);
        if (ts.kind[q] == 1) atomicAdd(&hist[slot][ts.val[q]], 1u);
        else {
            atomicAdd(&hist[slot][257 + length_code(ts.val[q] - 3)], 1u);
            atomicAdd(&nm[slot], 1u);
        }
        idx++;
    }
    __syncthreads();
    const int64_t nb = P.frame[b].nblocks;
    for (int i = threadIdx.x; i < 2 * kLCodes; i += kTileThreads) {
        const int slot = i / kLCodes;
        const uint32_t h = hist[slot][i % kLCodes];
        if (h && blk0 + slot < nb) atomicAdd(&B[blk0 + slot].hist[i % kLCodes], h);
    }
    if (threadIdx.x < 2 && nm[threadIdx.x] && blk0 + threadIdx.x < nb)
        atomicAdd((uint32_t*)&B[blk0 + threadIdx.x].nmatch, nm[threadIdx.x]);
}

// stage 4: one thread per block builds its trees, its heap and scratch in shared memory (a per-thread stack of ~7 KB
// would make the driver reserve that much local memory for every thread the GPU can hold)
__global__ void __launch_bounds__(32) png_trees_kernel(Ptrs P) {
    __shared__ TreeWork w;
    const int b = blockIdx.y;
    const int64_t k = blockIdx.x;
    if (threadIdx.x != 0 || k >= P.frame[b].nblocks) return;
    BlockInfo* B = P.blk + (int64_t)b * P.L.nbmax;
    BlockInfo& bi = B[k];
    const int64_t end = k + 1 < P.frame[b].nblocks ? B[k + 1].pos : P.L.s.N;
    plan_block(bi.hist, (uint32_t)bi.nmatch, end - bi.pos, bi.plan, w);
}

// code bits per tile
__global__ void __launch_bounds__(kTileThreads) png_tile_bits_kernel(Ptrs P) {
    __shared__ int64_t sh[kTileThreads];
    const int b = blockIdx.y;
    ThreadSyms ts;
    thread_symbols(P, b, blockIdx.x, ts, sh);
    int c = 0;
    for (int q = 0; q < kPerThread; q++) c += ts.kind[q] != 0;
    TileInfo& ti = P.tile[(int64_t)b * P.L.nt + blockIdx.x];
    int64_t idx = ti.symbase + block_scan<kTileThreads>(c, 0, sh) - c;
    const BlockInfo* B = P.blk + (int64_t)b * P.L.nbmax;
    int64_t bits = 0;
    for (int q = 0; q < kPerThread; q++) {
        if (!ts.kind[q]) continue;
        uint64_t v;
        bits += block_code_bits(B[idx / kBlockSyms].plan, ts.kind[q], ts.val[q], &v);
        idx++;
    }
    const int64_t tot = block_scan<kTileThreads>(bits, 0, sh);
    if (threadIdx.x == kTileThreads - 1) ti.bits = tot;
}

// stage 5: bit layout of every block, the frame's sizes
__global__ void __launch_bounds__(kScanThreads) png_layout_kernel(Ptrs P) {
    __shared__ int64_t sh[kScanThreads];
    const int b = blockIdx.x;
    TileInfo* T = P.tile + (int64_t)b * P.L.nt;
    frame_scan(P.L.nt, 0, 0, [&](int64_t i) { return T[i].bits; }, [&](int64_t i, int64_t v) { T[i].bitbase = v; }, sh);
    if (threadIdx.x != 0) return;
    FrameInfo& fr = P.frame[b];
    BlockInfo* B = P.blk + (int64_t)b * P.L.nbmax;
    int64_t pos = 16, cb = 0;
    int err = 0;
    for (int64_t k = 0; k < fr.nblocks; k++) {
        BlockInfo& bi = B[k];
        bi.start_bit = pos;
        bi.cbase = cb;
        if (bi.plan.type == kStored) {
            const int64_t len = (k + 1 < fr.nblocks ? B[k + 1].pos : P.L.s.N) - bi.pos;
            if (len > kMaxStored) err = 1;
            const int64_t aligned = (pos + 3 + 7) & ~(int64_t)7;
            bi.data_bit = aligned + 32;
            pos = aligned + 32 + 8 * len;
        } else {
            bi.data_bit = pos + bi.plan.header_bits;
            cb += bi.plan.data_bits;
            pos = bi.data_bit + bi.plan.data_bits + bi.plan.llen[kEndBlock];
        }
    }
    fr.total_bits = pos;
    fr.zbytes = (pos + 7) / 8 + 4;
    fr.png_bytes = png_bytes_for(fr.zbytes);
    fr.error = err;
}

__global__ void __launch_bounds__(kScanThreads) png_offsets_kernel(Ptrs P) {
    __shared__ int64_t sh[kScanThreads];
    const int64_t total = frame_scan(P.L.B, 0, 0, [&](int64_t i) { return P.frame[i].png_bytes; },
                                     [&](int64_t i, int64_t v) { P.offsets[i] = v; }, sh);
    if (threadIdx.x == 0) P.offsets[P.L.B] = total;
}

// block headers, stored-block lengths, END_BLOCK codes, the zlib header and trailer
__global__ void __launch_bounds__(64) png_headers_kernel(Ptrs P) {
    const int b = blockIdx.y;
    const int64_t k = (int64_t)blockIdx.x * 64 + threadIdx.x;
    const FrameInfo& fr = P.frame[b];
    if (k >= fr.nblocks) return;
    uint32_t* z = P.z + (int64_t)b * (P.L.zcap / 4);
    const BlockInfo& bi = P.blk[(int64_t)b * P.L.nbmax + k];
    const bool last = k == fr.nblocks - 1;
    if (k == 0) {
        uint8_t h[2];
        zlib_header(P.L.s.N, h);
        or_byte(z, 0, h[0]);
        or_byte(z, 1, h[1]);
    }
    if (last) {
        const int64_t at = (fr.total_bits + 7) / 8;
        for (int i = 0; i < 4; i++) or_byte(z, at + i, (uint8_t)(fr.adler >> (24 - 8 * i)));
    }
    if (bi.plan.type == kStored) {
        or_bits(z, bi.start_bit, last ? 1 : 0, 3);
        const int64_t len = (last ? P.L.s.N : P.blk[(int64_t)b * P.L.nbmax + k + 1].pos) - bi.pos;
        const uint32_t ln = (uint32_t)len | ((uint32_t)(~len & 0xffff) << 16);
        or_bits(z, bi.data_bit - 32, ln, 32);
        return;
    }
    int64_t pos = bi.start_bit;
    put_block_header(bi.plan, last, [&](uint32_t v, int n) {
        or_bits(z, pos, v, n);
        pos += n;
    });
    or_bits(z, bi.data_bit + bi.plan.data_bits, bi.plan.lcode[kEndBlock], bi.plan.llen[kEndBlock]);
}

// symbols and stored bytes
__global__ void __launch_bounds__(kTileThreads) png_emit_kernel(Ptrs P) {
    __shared__ int64_t sh[kTileThreads];
    const int b = blockIdx.y;
    ThreadSyms ts;
    thread_symbols(P, b, blockIdx.x, ts, sh);
    int c = 0;
    int64_t bits = 0;
    const TileInfo& ti = P.tile[(int64_t)b * P.L.nt + blockIdx.x];
    const BlockInfo* B = P.blk + (int64_t)b * P.L.nbmax;
    // pass 1: my symbol count and bits (for the in-tile offsets)
    {
        int64_t idx0 = 0;
        for (int q = 0; q < kPerThread; q++) c += ts.kind[q] != 0;
        idx0 = ti.symbase + block_scan<kTileThreads>(c, 0, sh) - c;
        int64_t idx = idx0;
        for (int q = 0; q < kPerThread; q++) {
            if (!ts.kind[q]) continue;
            uint64_t v;
            bits += block_code_bits(B[idx / kBlockSyms].plan, ts.kind[q], ts.val[q], &v);
            idx++;
        }
        int64_t cbit = ti.bitbase + block_scan<kTileThreads>(bits, 0, sh) - bits;
        uint32_t* z = P.z + (int64_t)b * (P.L.zcap / 4);
        idx = idx0;
        for (int q = 0; q < kPerThread; q++) {
            if (!ts.kind[q]) continue;
            const BlockInfo& bi = B[idx / kBlockSyms];
            uint64_t v;
            const int n = block_code_bits(bi.plan, ts.kind[q], ts.val[q], &v);
            if (bi.plan.type != kStored) {
                const int64_t at = bi.data_bit + (cbit - bi.cbase);
                if (n > 32) {
                    or_bits(z, at, v & 0xffffffffu, 32);
                    or_bits(z, at + 32, v >> 32, n - 32);
                } else {
                    or_bits(z, at, v, n);
                }
            } else {
                // the raw bytes of this symbol: one for a literal, the match length for a match
                const int64_t p = ts.p0 + q;
                const int cnt = ts.kind[q] == 1 ? 1 : ts.val[q];
                const uint8_t* f = P.filt + (int64_t)b * P.L.filt_stride;
                for (int r = 0; r < cnt; r++) or_byte(z, bi.data_bit / 8 + (p + r - bi.pos), f[p + r]);
            }
            cbit += n;
            idx++;
        }
    }
}

// PNG container: one thread per IDAT chunk (copy + CRC), chunk 0's thread also writes the signature, IHDR and IEND
__global__ void __launch_bounds__(128) png_container_kernel(Ptrs P) {
    __shared__ uint32_t crc_t[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) crc_table_fill(crc_t, i);
    __syncthreads();
    const int b = blockIdx.y;
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const FrameInfo& fr = P.frame[b];
    const int64_t nch = (fr.zbytes + kChunk - 1) / kChunk;
    if (c >= nch) return;
    const int64_t start = P.offsets[b], end = P.offsets[b + 1];
    if (fr.error || end > P.out_bytes || end - start != fr.png_bytes) return;     // never write past out_bytes
    uint8_t* o = P.out + start;
    const uint8_t* z = (const uint8_t*)(P.z + (int64_t)b * (P.L.zcap / 4));
    write_idat(o + 33 + c * (kChunk + 12), z, fr.zbytes, c, crc_t);
    if (c == 0) {
        write_png_head(o, P.L.s, crc_t);
        write_png_tail(o + fr.png_bytes - 12);
    }
}

int check_shape(int B, int H, int W, int C, const char* who) {
    DC_REQUIRE(B >= 1 && B <= 65535 && H >= 1 && W >= 1 && (C == 1 || C == 3), DC_EINVAL,
               "%s: B %d, H %d, W %d, C %d out of range (1 <= B <= 65535, C 1 or 3)", who, B, H, W, C);
    const Shape s = make_shape(H, W, C);
    DC_REQUIRE(s.N <= ((int64_t)1 << 31) - ((int64_t)1 << 20), DC_EINVAL,
               "%s: %lld filtered bytes per frame; at most 2^31 - 2^20", who, (long long)s.N);
    const Layout L = make_layout(B, H, W, C);
    DC_REQUIRE(L.nt < 0x7fffffff && (int64_t)B * L.nbmax < ((int64_t)1 << 40), DC_EINVAL, "%s: shape too large", who);
    return DC_OK;
}

// ---------------------------------------------------------------- host encoder (dc_debug_png_host)
struct HostSink;
struct SinkRef {
    HostSink* s;
    __host__ __device__ void operator()(uint32_t v, int n) const;
};
struct HostSink {
    uint32_t* z;
    int64_t pos;
    __host__ __device__ void operator()(uint32_t v, int n) {
        for (int i = 0; i < n; i++, pos++)
            if (v >> i & 1) z[pos >> 5] |= 1u << (pos & 31);
    }
};

__host__ __device__ void SinkRef::operator()(uint32_t v, int n) const { (*s)(v, n); }

}  // namespace

int launch_png_encode(const dc_png_args_t* a, cudaStream_t stream) {
    DC_REQUIRE(a, DC_EINVAL, "dc_png_encode: null argument");
    int rc = check_shape(a->B, a->H, a->W, a->C, "dc_png_encode");
    if (rc != DC_OK) return rc;
    DC_REQUIRE(a->images && a->out && a->offsets, DC_EINVAL, "dc_png_encode: null pointer");
    int64_t need = 0;
    size_t ws = 0;
    rc = dc_png_bounds(a->B, a->H, a->W, a->C, &need, &ws);
    if (rc != DC_OK) return rc;
    DC_REQUIRE(a->out_bytes >= need, DC_EINVAL, "dc_png_encode: out_bytes %lld < bound %lld", (long long)a->out_bytes,
               (long long)need);
    DC_REQUIRE(a->workspace && a->workspace_bytes >= ws, DC_EWORKSPACE, "dc_png_encode: workspace too small (%zu < %zu)",
               a->workspace_bytes, ws);
    DC_REQUIRE(((uintptr_t)a->workspace & 255) == 0, DC_EINVAL, "dc_png_encode: workspace must be 256-byte aligned");
    Ptrs P;
    P.L = make_layout(a->B, a->H, a->W, a->C);
    char* w = (char*)a->workspace;
    P.img = a->images;
    P.filt = (uint8_t*)(w + P.L.off_filt);
    P.tile = (TileInfo*)(w + P.L.off_tile);
    P.blk = (BlockInfo*)(w + P.L.off_block);
    P.frame = (FrameInfo*)(w + P.L.off_frame);
    P.z = (uint32_t*)(w + P.L.off_z);
    P.out = a->out;
    P.out_bytes = a->out_bytes;
    P.offsets = a->offsets;
    const int B = a->B;
    DC_CUDA(cudaMemsetAsync(P.blk, 0, P.L.off_frame - P.L.off_block, stream));
    DC_CUDA(cudaMemsetAsync(P.z, 0, P.L.total - P.L.off_z, stream));
    const dim3 tiles((unsigned)P.L.nt, (unsigned)B);
    png_filter_kernel<<<tiles, kTileThreads, 0, stream>>>(P);
    png_scan_runs_kernel<<<B, kScanThreads, 0, stream>>>(P);
    png_count_kernel<<<tiles, kTileThreads, 0, stream>>>(P);
    png_scan_syms_kernel<<<B, kScanThreads, 0, stream>>>(P);
    png_hist_kernel<<<tiles, kTileThreads, 0, stream>>>(P);
    png_trees_kernel<<<dim3((unsigned)P.L.nbmax, (unsigned)B), 32, 0, stream>>>(P);
    png_tile_bits_kernel<<<tiles, kTileThreads, 0, stream>>>(P);
    png_layout_kernel<<<B, kScanThreads, 0, stream>>>(P);
    png_offsets_kernel<<<1, kScanThreads, 0, stream>>>(P);
    png_headers_kernel<<<dim3((unsigned)((P.L.nbmax + 63) / 64), (unsigned)B), 64, 0, stream>>>(P);
    png_emit_kernel<<<tiles, kTileThreads, 0, stream>>>(P);
    const int64_t max_chunks = (P.L.zcap + kChunk - 1) / kChunk;
    png_container_kernel<<<dim3((unsigned)((max_chunks + 127) / 128), (unsigned)B), 128, 0, stream>>>(P);
    DC_CUDA(cudaGetLastError());
    return DC_OK;
}

int png_encode_host(const uint8_t* img, int H, int W, int C, uint8_t* out, int64_t out_bytes, int64_t* png_bytes,
                    int32_t* block_stats, int64_t stats_cap, int64_t* nblocks_out) {
    DC_REQUIRE(img && out && png_bytes, DC_EINVAL, "dc_debug_png_host: null pointer");
    int rc = check_shape(1, H, W, C, "dc_debug_png_host");
    if (rc != DC_OK) return rc;
    int64_t need = 0;
    size_t ws = 0;
    rc = dc_png_bounds(1, H, W, C, &need, &ws);
    if (rc != DC_OK) return rc;
    DC_REQUIRE(out_bytes >= need, DC_EINVAL, "dc_debug_png_host: out_bytes %lld < bound %lld", (long long)out_bytes,
               (long long)need);
    const Shape s = make_shape(H, W, C);
    const int64_t N = s.N;
    uint8_t* f = new uint8_t[N];
    for (int64_t i = 0; i < N; i++) f[i] = filtered_byte(img, s, i);
    // the parse: symbols in order (kind, value, position)
    struct Sym { int32_t pos; int16_t val; uint8_t kind; };
    Sym* sy = new Sym[N];
    int64_t ns = 0;
    for (int64_t i = 0; i < N;) {
        int64_t e = i + 1;
        while (e < N && f[e] == f[i]) e++;
        for (int64_t j = 0; j < e - i; j++) {
            int len = 0;
            const int k = run_symbol(j, e - i, &len);
            if (k) sy[ns++] = Sym{(int32_t)(i + j), (int16_t)(k == 1 ? f[i + j] : len), (uint8_t)k};
        }
        i = e;
    }
    const int64_t nb = ns / kBlockSyms + 1;
    const int64_t zcap = (zlib_bound(N) + 8) & ~(int64_t)3;
    uint32_t* z = new uint32_t[zcap / 4]();
    HostSink sink{z, 0};
    uint8_t h[2];
    zlib_header(N, h);
    sink(h[0], 8);
    sink(h[1], 8);
    TreeWork* w = new TreeWork;
    BlockPlan* p = new BlockPlan;
    uint32_t hist[kLCodes];
    rc = DC_OK;
    for (int64_t k = 0; k < nb; k++) {
        const int64_t s0 = k * kBlockSyms, s1 = s0 + kBlockSyms < ns ? s0 + kBlockSyms : ns;
        const int64_t p0 = s0 < ns ? sy[s0].pos : N, p1 = s1 < ns ? sy[s1].pos : N;
        uint32_t nmatch = 0;
        for (int n = 0; n < kLCodes; n++) hist[n] = 0;
        for (int64_t i = s0; i < s1; i++) {
            if (sy[i].kind == 1) hist[sy[i].val]++;
            else {
                hist[257 + length_code(sy[i].val - 3)]++;
                nmatch++;
            }
        }
        plan_block(hist, nmatch, p1 - p0, *p, *w);
        const bool last = k == nb - 1;
        if (block_stats && k < stats_cap) block_stats[k] = p->type | (p->overflow << 2);
        if (p->type == kStored) {
            if (p1 - p0 > kMaxStored) rc = DC_EINVAL;
            sink(last ? 1 : 0, 3);
            sink.pos = (sink.pos + 7) & ~(int64_t)7;
            sink((uint32_t)(p1 - p0), 16);
            sink((uint32_t)(~(p1 - p0) & 0xffff), 16);
            for (int64_t i = p0; i < p1; i++) sink(f[i], 8);
            continue;
        }
        put_block_header(*p, last, SinkRef{&sink});
        for (int64_t i = s0; i < s1; i++) {
            uint64_t v;
            const int n = block_code_bits(*p, sy[i].kind, sy[i].val, &v);
            sink((uint32_t)(v & 0xffffffffu), n > 32 ? 32 : n);
            if (n > 32) sink((uint32_t)(v >> 32), n - 32);
        }
        sink(p->lcode[kEndBlock], p->llen[kEndBlock]);
    }
    sink.pos = (sink.pos + 7) & ~(int64_t)7;
    uint32_t a = 1, bb = 0;
    for (int64_t i = 0; i < N; i++) {
        a = (a + f[i]) % 65521;
        bb = (bb + a) % 65521;
    }
    const uint32_t adler = (bb << 16) | a;
    for (int i = 0; i < 4; i++) sink((adler >> (24 - 8 * i)) & 0xff, 8);
    const int64_t zbytes = sink.pos / 8;
    uint32_t crc_t[256];
    for (int i = 0; i < 256; i++) crc_table_fill(crc_t, i);
    write_png_head(out, s, crc_t);
    const int64_t nch = (zbytes + kChunk - 1) / kChunk;
    for (int64_t c = 0; c < nch; c++) write_idat(out + 33 + c * (kChunk + 12), (const uint8_t*)z, zbytes, c, crc_t);
    *png_bytes = png_bytes_for(zbytes);
    write_png_tail(out + *png_bytes - 12);
    if (nblocks_out) *nblocks_out = nb;
    delete[] f;
    delete[] sy;
    delete[] z;
    delete w;
    delete p;
    if (rc != DC_OK) set_error("dc_debug_png_host: a stored block longer than %d bytes", kMaxStored);
    return rc;
}

}  // namespace dc

extern "C" int dc_png_bounds(int B, int H, int W, int C, int64_t* out_bytes, size_t* workspace_bytes) {
    DC_REQUIRE(out_bytes && workspace_bytes, DC_EINVAL, "dc_png_bounds: null pointer");
    const int rc = dc::check_shape(B, H, W, C, "dc_png_bounds");
    if (rc != DC_OK) return rc;
    const dc::Layout L = dc::make_layout(B, H, W, C);
    *out_bytes = (int64_t)B * dc::png_bytes_for(dc::zlib_bound(L.s.N));
    *workspace_bytes = L.total;
    return DC_OK;
}
