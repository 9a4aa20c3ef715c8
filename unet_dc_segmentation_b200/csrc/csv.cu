// csv.cu -- droplet table -> CSV text on the device (dc_table_csv), byte for byte what pandas' to_csv writes for the
// per-image DataFrames of quantify_droplets_batch.py:62-63.
//
// One source for the device and the host: every formatting routine is __host__ __device__, and the Ryu tables exist
// as a __device__ copy and a host copy expanded from the same generated initialiser (csv_tables.inc), so the host-only
// test entry points (dc_debug_format_values, dc_debug_table_csv_host) run exactly the code the kernels run.
//
// float64 -> text is Ryu (Ulf Adams, PLDI 2018): the shortest decimal that rounds back to the same double, the closest
// to it when several qualify, ties by round-half-even on the removed digits -- the digits of Python's repr and of
// numpy's str (David Gay's shortest mode), which is what pandas writes.  The layout is repr's: positional when the
// leading digit's exponent is in [-4, 16), with ".0" when no fraction is left, else d[.ddd]e+XX.
#include "common.cuh"
#include "csv_tables.inc"

#include <string.h>

namespace dc {
namespace {

__device__ const uint64_t kPow5InvDev[DC_POW5_INV_SIZE][2] = DC_POW5_INV_SPLIT_INIT;
__device__ const uint64_t kPow5Dev[DC_POW5_SIZE][2] = DC_POW5_SPLIT_INIT;
#ifndef __CUDA_ARCH__
const uint64_t kPow5InvHost[DC_POW5_INV_SIZE][2] = DC_POW5_INV_SPLIT_INIT;
const uint64_t kPow5Host[DC_POW5_SIZE][2] = DC_POW5_SPLIT_INIT;
#endif

constexpr int kPow5InvBits = 125;
constexpr int kPow5Bits = 125;
constexpr int kMaxF64Chars = 24;     // "-1.2345678901234567e-308"
constexpr int kMaxI64Chars = 20;     // "-9223372036854775808"
constexpr int kMaxLabelChars = 10;   // label = row + 1 <= capacity < 2^31

__host__ __device__ __forceinline__ const uint64_t* pow5_inv(uint32_t q) {
#ifdef __CUDA_ARCH__
    return kPow5InvDev[q];
#else
    return kPow5InvHost[q];
#endif
}
__host__ __device__ __forceinline__ const uint64_t* pow5(uint32_t i) {
#ifdef __CUDA_ARCH__
    return kPow5Dev[i];
#else
    return kPow5Host[i];
#endif
}
__host__ __device__ __forceinline__ uint64_t umulh(uint64_t a, uint64_t b) {
#ifdef __CUDA_ARCH__
    return __umul64hi(a, b);
#else
    return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}
__host__ __device__ __forceinline__ uint64_t f64_bits(double x) {
#ifdef __CUDA_ARCH__
    return (uint64_t)__double_as_longlong(x);
#else
    uint64_t u;
    memcpy(&u, &x, sizeof(u));
    return u;
#endif
}

// ---------------------------------------------------------------- Ryu (d2s.c of the reference implementation)
__host__ __device__ __forceinline__ int32_t pow5bits(int32_t e) { return ((e * 1217359) >> 19) + 1; }   // ceil(log2 5^e), e >= 1
__host__ __device__ __forceinline__ uint32_t log10_pow2(int32_t e) { return (uint32_t)((e * 78913) >> 18); }
__host__ __device__ __forceinline__ uint32_t log10_pow5(int32_t e) { return (uint32_t)((e * 732923) >> 20); }

__host__ __device__ inline uint32_t pow5_factor(uint64_t v) {
    uint32_t n = 0;
    while (v % 5 == 0) {
        v /= 5;
        ++n;
    }
    return n;
}
__host__ __device__ __forceinline__ bool multiple_of_pow5(uint64_t v, uint32_t p) { return pow5_factor(v) >= p; }
__host__ __device__ __forceinline__ bool multiple_of_pow2(uint64_t v, uint32_t p) { return (v & ((1ull << p) - 1)) == 0; }

// (m * mul) >> j for the 128-bit multiplier {mul[0] low, mul[1] high}; 64 <= j < 128 for every call below
__host__ __device__ __forceinline__ uint64_t mul_shift64(uint64_t m, const uint64_t* mul, int32_t j) {
    const uint64_t b0_hi = umulh(m, mul[0]);
    const uint64_t b2_lo = m * mul[1];
    const uint64_t b2_hi = umulh(m, mul[1]);
    const uint64_t lo = b0_hi + b2_lo;
    const uint64_t hi = b2_hi + (lo < b0_hi);
    const int s = j - 64;
    return s == 0 ? lo : (lo >> s) | (hi << (64 - s));
}

// Finite, non-zero x = (ieee_m, ieee_e) -> digits * 10^e10 with the fewest digits.
__host__ __device__ inline void ryu_d2d(uint64_t ieee_m, uint32_t ieee_e, uint64_t* digits, int32_t* e10_out) {
    int32_t e2;
    uint64_t m2;
    if (ieee_e == 0) {
        e2 = 1 - 1023 - 52 - 2;
        m2 = ieee_m;
    } else {
        e2 = (int32_t)ieee_e - 1023 - 52 - 2;
        m2 = (1ull << 52) | ieee_m;
    }
    const bool accept_bounds = (m2 & 1) == 0;      // round-half-even on input: the interval ends belong to x
    const uint64_t mv = 4 * m2;
    const uint32_t mm_shift = ieee_m != 0 || ieee_e <= 1;
    uint64_t vr, vp, vm;
    int32_t e10;
    bool vm_tz = false, vr_tz = false;
    if (e2 >= 0) {
        const uint32_t q = log10_pow2(e2) - (e2 > 3);
        e10 = (int32_t)q;
        const int32_t k = kPow5InvBits + pow5bits((int32_t)q) - 1;
        const int32_t i = -e2 + (int32_t)q + k;
        const uint64_t* mul = pow5_inv(q);
        vr = mul_shift64(4 * m2, mul, i);
        vp = mul_shift64(4 * m2 + 2, mul, i);
        vm = mul_shift64(4 * m2 - 1 - mm_shift, mul, i);
        if (q <= 21) {
            if (mv % 5 == 0) vr_tz = multiple_of_pow5(mv, q);
            else if (accept_bounds) vm_tz = multiple_of_pow5(mv - 1 - mm_shift, q);
            else vp -= multiple_of_pow5(mv + 2, q);
        }
    } else {
        const uint32_t q = log10_pow5(-e2) - (-e2 > 1);
        e10 = (int32_t)q + e2;
        const int32_t i = -e2 - (int32_t)q;
        const int32_t k = pow5bits(i) - kPow5Bits;
        const int32_t j = (int32_t)q - k;
        const uint64_t* mul = pow5(i);
        vr = mul_shift64(4 * m2, mul, j);
        vp = mul_shift64(4 * m2 + 2, mul, j);
        vm = mul_shift64(4 * m2 - 1 - mm_shift, mul, j);
        if (q <= 1) {
            vr_tz = true;
            if (accept_bounds) vm_tz = mm_shift == 1;
            else --vp;
        } else if (q < 63) {
            vr_tz = multiple_of_pow2(mv, q);
        }
    }
    int32_t removed = 0;
    uint32_t last = 0;
    uint64_t out;
    if (vm_tz || vr_tz) {                           // rare general case: track exact trailing zeros
        while (vp / 10 > vm / 10) {
            vm_tz &= vm % 10 == 0;
            vr_tz &= last == 0;
            last = (uint32_t)(vr % 10);
            vr /= 10;
            vp /= 10;
            vm /= 10;
            ++removed;
        }
        if (vm_tz) {
            while (vm % 10 == 0) {
                vr_tz &= last == 0;
                last = (uint32_t)(vr % 10);
                vr /= 10;
                vp /= 10;
                vm /= 10;
                ++removed;
            }
        }
        if (vr_tz && last == 5 && vr % 2 == 0) last = 4;   // exactly ...50..0: round half to even
        out = vr + ((vr == vm && (!accept_bounds || !vm_tz)) || last >= 5);
    } else {
        bool round_up = false;
        if (vp / 100 > vm / 100) {
            round_up = vr % 100 >= 50;
            vr /= 100;
            vp /= 100;
            vm /= 100;
            removed += 2;
        }
        while (vp / 10 > vm / 10) {
            round_up = vr % 10 >= 5;
            vr /= 10;
            vp /= 10;
            vm /= 10;
            ++removed;
        }
        out = vr + (vr == vm || round_up);
    }
    *digits = out;
    *e10_out = e10 + removed;
}

__host__ __device__ __forceinline__ int decimal_length(uint64_t v) {
    int n = 1;
    uint64_t p = 10;
    while (v >= p) {
        if (++n == 20) break;
        p *= 10;
    }
    return n;
}
__host__ __device__ __forceinline__ void put_digits(char* d, uint64_t v, int n) {
    for (int i = n - 1; i >= 0; --i) {
        d[i] = (char)('0' + v % 10);
        v /= 10;
    }
}

// ---------------------------------------------------------------- one value -> text (out: >= kMaxF64Chars bytes)
__host__ __device__ inline int format_i64(char* out, int64_t v) {
    int n = 0;
    uint64_t u = (uint64_t)v;
    if (v < 0) {
        out[n++] = '-';
        u = 0 - u;
    }
    const int len = decimal_length(u);
    put_digits(out + n, u, len);
    return n + len;
}

__host__ __device__ inline int format_f64(char* out, double x) {
    const uint64_t bits = f64_bits(x);
    const uint64_t ieee_m = bits & ((1ull << 52) - 1);
    const uint32_t ieee_e = (uint32_t)(bits >> 52) & 0x7FF;
    if (ieee_e == 0x7FF && ieee_m != 0) return 0;   // NaN: pandas' na_rep, the empty field
    int n = 0;
    if (bits >> 63) out[n++] = '-';
    if (ieee_e == 0x7FF) {
        out[n] = 'i'; out[n + 1] = 'n'; out[n + 2] = 'f';
        return n + 3;
    }
    if (ieee_e == 0 && ieee_m == 0) {
        out[n] = '0'; out[n + 1] = '.'; out[n + 2] = '0';
        return n + 3;
    }
    uint64_t digits;
    int32_t e10;
    ryu_d2d(ieee_m, ieee_e, &digits, &e10);
    char d[17];
    const int len = decimal_length(digits);
    put_digits(d, digits, len);
    const int E = e10 + len - 1;                    // decimal exponent of the leading digit
    if (E >= -4 && E < 16) {
        if (E < 0) {                                // 0.000ddd
            out[n++] = '0';
            out[n++] = '.';
            for (int i = 0; i < -E - 1; ++i) out[n++] = '0';
            for (int i = 0; i < len; ++i) out[n++] = d[i];
        } else if (len <= E + 1) {                  // ddd000.0
            for (int i = 0; i < len; ++i) out[n++] = d[i];
            for (int i = len; i <= E; ++i) out[n++] = '0';
            out[n++] = '.';
            out[n++] = '0';
        } else {                                    // ddd.ddd
            for (int i = 0; i <= E; ++i) out[n++] = d[i];
            out[n++] = '.';
            for (int i = E + 1; i < len; ++i) out[n++] = d[i];
        }
    } else {                                        // d.ddde+XX
        out[n++] = d[0];
        if (len > 1) {
            out[n++] = '.';
            for (int i = 1; i < len; ++i) out[n++] = d[i];
        }
        out[n++] = 'e';
        out[n++] = E < 0 ? '-' : '+';
        const int ae = E < 0 ? -E : E;
        if (ae >= 100) out[n++] = (char)('0' + ae / 100);
        out[n++] = (char)('0' + ae / 10 % 10);
        out[n++] = (char)('0' + ae % 10);
    }
    return n;
}

// ---------------------------------------------------------------- rows and frames
__host__ __device__ __forceinline__ const char* csv_header(bool micron) {
    return micron ? "filename,label,area,equivalent_diameter,centroid-0,centroid-1,area_sqmicron,eq_diam_micron\n"
                  : "filename,label,area,equivalent_diameter,centroid-0,centroid-1\n";
}
__host__ __device__ __forceinline__ int64_t cstr_len(const char* s) {
    int64_t n = 0;
    while (s[n]) ++n;
    return n;
}
constexpr int64_t kEmptyFrameChars = 9;             // "filename\n": DataFrame() + insert + to_csv

__host__ __device__ __forceinline__ bool has_micron(const dc_table_csv_args_t& a) { return a.area_um2 != nullptr; }

// rows of frame b, or -1 when its count exceeds the capacity (the table is incomplete)
__host__ __device__ __forceinline__ int frame_rows(const dc_table_csv_args_t& a, int b) {
    const int n = a.counts[b];
    return n > a.capacity ? -1 : (n < 0 ? 0 : n);
}

__host__ __device__ __forceinline__ int64_t frame_head_len(const dc_table_csv_args_t& a, int n) {
    return n > 0 ? cstr_len(csv_header(has_micron(a))) : kEmptyFrameChars;
}

// Row r of frame b -> dst (NULL: length only).  Returns the row's length, newline included.
__host__ __device__ inline int64_t table_row(const dc_table_csv_args_t& a, int b, int r, char* dst) {
    const int64_t i = (int64_t)b * a.capacity + r;
    const int64_t n0 = a.name_offsets[b], n1 = a.name_offsets[b + 1];
    char tmp[kMaxF64Chars];
    int64_t n = 0;
    auto put = [&](const char* s, int64_t len) {
        if (dst)
            for (int64_t k = 0; k < len; ++k) dst[n + k] = s[k];
        n += len;
    };
    put(a.names + n0, n1 - n0);
    put(",", 1);
    put(tmp, format_i64(tmp, (int64_t)r + 1));
    put(",", 1);
    put(tmp, format_i64(tmp, a.area[i]));
    const double* cols[5] = {a.eq_diam, a.centroid0, a.centroid1, a.area_um2, a.diam_um};
    const int nf = has_micron(a) ? 5 : 3;
    for (int c = 0; c < nf; ++c) {
        put(",", 1);
        put(tmp, format_f64(tmp, cols[c][i]));
    }
    put("\n", 1);
    return n;
}

__host__ __device__ inline void write_frame_head(const dc_table_csv_args_t& a, int n, char* dst) {
    const char* h = n > 0 ? csv_header(has_micron(a)) : "filename\n";
    for (int64_t k = 0; h[k]; ++k) dst[k] = h[k];
}

int64_t row_bound_fixed(bool micron) {            // widest row without its filename field
    const int nf = micron ? 5 : 3;
    return kMaxLabelChars + kMaxI64Chars + (int64_t)nf * kMaxF64Chars + (nf + 2) + 1;
}

size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// ---------------------------------------------------------------- kernels
constexpr int kScanThreads = 1024;
constexpr int kRowThreads = 256;

__device__ int64_t block_exclusive_scan(int64_t v, int64_t* total) {
    __shared__ int64_t warp_sums[kScanThreads / 32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int64_t x = v;
    for (int o = 1; o < 32; o <<= 1) {
        const int64_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) warp_sums[wid] = x;
    __syncthreads();
    if (wid == 0) {
        int64_t s = warp_sums[lane];
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t y = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += y;
        }
        warp_sums[lane] = s;
    }
    __syncthreads();
    const int64_t before = (wid ? warp_sums[wid - 1] : 0) + x - v;
    *total = warp_sums[31];
    __syncthreads();                                // warp_sums is reused by the next call
    return before;
}

// pass 1: the length of every row
__global__ void __launch_bounds__(kRowThreads) csv_row_len_kernel(dc_table_csv_args_t a, int64_t* row_off) {
    const int b = blockIdx.y;
    const int r = blockIdx.x * kRowThreads + threadIdx.x;
    if (r < frame_rows(a, b)) row_off[(int64_t)b * a.capacity + r] = table_row(a, b, r, nullptr);
}

// per frame: row lengths -> offsets inside the frame (after its header), frame length, area sum
__global__ void __launch_bounds__(kScanThreads) csv_frame_scan_kernel(dc_table_csv_args_t a, int64_t* row_off,
                                                                      int64_t* frame_len) {
    const int b = blockIdx.x;
    const int n = frame_rows(a, b);
    if (n < 0) {
        if (threadIdx.x == 0) {
            frame_len[b] = 0;
            a.area_sum[b] = -1;
        }
        return;
    }
    int64_t* off = row_off + (int64_t)b * a.capacity;
    const int64_t* area = a.area + (int64_t)b * a.capacity;
    int64_t carry = 0, asum = 0;
    for (int base = 0; base < n; base += kScanThreads) {
        const int r = base + threadIdx.x;
        int64_t tot;
        const int64_t ex = block_exclusive_scan(r < n ? off[r] : 0, &tot);
        if (r < n) {
            off[r] = carry + ex;
            asum += area[r];
        }
        carry += tot;
    }
    int64_t area_total;
    block_exclusive_scan(asum, &area_total);
    if (threadIdx.x == 0) {
        frame_len[b] = frame_head_len(a, n) + carry;
        a.area_sum[b] = area_total;
    }
}

// one block: frame lengths -> frame_offsets[0..B]
__global__ void __launch_bounds__(kScanThreads) csv_batch_scan_kernel(dc_table_csv_args_t a, const int64_t* frame_len) {
    int64_t carry = 0;
    for (int base = 0; base < a.B; base += kScanThreads) {
        const int b = base + threadIdx.x;
        int64_t tot;
        const int64_t ex = block_exclusive_scan(b < a.B ? frame_len[b] : 0, &tot);
        if (b < a.B) a.frame_offsets[b] = carry + ex;
        carry += tot;
    }
    if (threadIdx.x == 0) a.frame_offsets[a.B] = carry;
}

// pass 2: every row (and the header, by row 0's thread) at its place
__global__ void __launch_bounds__(kRowThreads) csv_write_kernel(dc_table_csv_args_t a, const int64_t* row_off) {
    const int b = blockIdx.y;
    const int r = blockIdx.x * kRowThreads + threadIdx.x;
    const int n = frame_rows(a, b);
    if (n < 0 || (r >= n && r != 0)) return;
    const int64_t start = a.frame_offsets[b], end = a.frame_offsets[b + 1];
    if (end > a.out_bytes || end < start) return;   // cannot happen with out_bytes >= the bound; never write past it
    if (r == 0) write_frame_head(a, n, a.out + start);
    if (r < n) table_row(a, b, r, a.out + start + frame_head_len(a, n) + row_off[(int64_t)b * a.capacity + r]);
}

int check_args(const dc_table_csv_args_t* a, bool device, const char* who) {
    DC_REQUIRE(a, DC_EINVAL, "%s: null argument", who);
    DC_REQUIRE(a->B >= 1 && a->B <= 65535 && a->capacity >= 1 && a->capacity < 0x7fffffff, DC_EINVAL,
               "%s: B %d / capacity %d out of range", who, a->B, a->capacity);
    DC_REQUIRE(a->counts && a->area && a->eq_diam && a->centroid0 && a->centroid1 && a->names && a->name_offsets &&
               a->out && a->frame_offsets && a->area_sum, DC_EINVAL, "%s: null pointer", who);
    DC_REQUIRE((a->area_um2 == nullptr) == (a->diam_um == nullptr), DC_EINVAL,
               "%s: area_um2 and diam_um must both be given or both be NULL", who);
    int64_t need = 0;
    size_t ws = 0;
    int rc = dc_table_csv_bounds(a->B, a->capacity, a->area_um2 != nullptr, a->names_bytes, &need, &ws);
    if (rc != DC_OK) return rc;
    DC_REQUIRE(a->out_bytes >= need, DC_EINVAL, "%s: out_bytes %lld < bound %lld", who, (long long)a->out_bytes,
               (long long)need);
    if (device) {
        DC_REQUIRE(a->workspace && a->workspace_bytes >= ws, DC_EWORKSPACE, "%s: workspace too small (%zu < %zu)", who,
                   a->workspace_bytes, ws);
        DC_REQUIRE(((uintptr_t)a->workspace & 255) == 0, DC_EINVAL, "%s: workspace must be 256-byte aligned", who);
    }
    return DC_OK;
}

}  // namespace

int launch_table_csv(const dc_table_csv_args_t* args, cudaStream_t stream) {
    int rc = check_args(args, true, "dc_table_csv");
    if (rc != DC_OK) return rc;
    const dc_table_csv_args_t a = *args;
    int64_t* row_off = (int64_t*)a.workspace;
    int64_t* frame_len = (int64_t*)((char*)a.workspace + align256((size_t)a.B * a.capacity * sizeof(int64_t)));
    const dim3 rows_grid((unsigned)ceil_div(a.capacity, kRowThreads), (unsigned)a.B);
    csv_row_len_kernel<<<rows_grid, kRowThreads, 0, stream>>>(a, row_off);
    csv_frame_scan_kernel<<<a.B, kScanThreads, 0, stream>>>(a, row_off, frame_len);
    csv_batch_scan_kernel<<<1, kScanThreads, 0, stream>>>(a, frame_len);
    csv_write_kernel<<<rows_grid, kRowThreads, 0, stream>>>(a, row_off);
    DC_CUDA(cudaGetLastError());
    return DC_OK;
}

int table_csv_host(const dc_table_csv_args_t* args) {
    int rc = check_args(args, false, "dc_debug_table_csv_host");
    if (rc != DC_OK) return rc;
    const dc_table_csv_args_t& a = *args;
    int64_t pos = 0;
    for (int b = 0; b < a.B; ++b) {
        a.frame_offsets[b] = pos;
        const int n = frame_rows(a, b);
        if (n < 0) {
            a.area_sum[b] = -1;
            continue;
        }
        write_frame_head(a, n, a.out + pos);
        pos += frame_head_len(a, n);
        int64_t asum = 0;
        for (int r = 0; r < n; ++r) {
            pos += table_row(a, b, r, a.out + pos);
            asum += a.area[(int64_t)b * a.capacity + r];
        }
        a.area_sum[b] = asum;
    }
    a.frame_offsets[a.B] = pos;
    return DC_OK;
}

int format_values_host(const void* values, int is_double, int64_t n, char* out, int64_t cap, int64_t* offsets) {
    DC_REQUIRE(values && out && offsets && n >= 0 && cap >= 0, DC_EINVAL, "dc_debug_format_values: bad argument");
    char tmp[kMaxF64Chars];
    int64_t pos = 0;
    for (int64_t i = 0; i < n; ++i) {
        offsets[i] = pos;
        const int len = is_double ? format_f64(tmp, ((const double*)values)[i]) : format_i64(tmp, ((const int64_t*)values)[i]);
        DC_REQUIRE(pos + len <= cap, DC_EINVAL, "dc_debug_format_values: %lld bytes are not enough", (long long)cap);
        memcpy(out + pos, tmp, len);
        pos += len;
    }
    offsets[n] = pos;
    return DC_OK;
}

}  // namespace dc

extern "C" int dc_table_csv_bounds(int B, int capacity, int micron, int64_t names_bytes, int64_t* out_bytes,
                                   size_t* workspace_bytes) {
    DC_REQUIRE(out_bytes && workspace_bytes && B >= 1 && B <= 65535 && capacity >= 1 && capacity < 0x7fffffff &&
               names_bytes >= 0 && names_bytes < ((int64_t)1 << 40), DC_EINVAL, "dc_table_csv_bounds: bad argument");
    // per frame: its header (at least the 9 bytes of an empty frame) + capacity rows of the widest kind
    const int64_t head = dc::cstr_len(dc::csv_header(micron != 0));
    const double need = (double)B * head + (double)capacity * ((double)names_bytes + (double)B * dc::row_bound_fixed(micron != 0));
    DC_REQUIRE(need < 9.0e18, DC_EINVAL, "dc_table_csv_bounds: %g bytes do not fit in int64", need);
    *out_bytes = (int64_t)B * head + (int64_t)capacity * (names_bytes + (int64_t)B * dc::row_bound_fixed(micron != 0));
    *workspace_bytes = dc::align256((size_t)B * capacity * sizeof(int64_t)) + dc::align256((size_t)B * sizeof(int64_t));
    return DC_OK;
}
