// api.cu -- the extern "C" surface of libunetdc_b200.so (include/unetdc_b200.h): argument checks,
// error plumbing, and the layer schedule of one UNetDC forward (reference models/model_2.py:56-80).
#include "common.cuh"

#include <new>
#include <stdarg.h>
#include <string.h>

namespace dc {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
    set_error("CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
    return DC_ECUDA;
}

// Device gate: every entry point that launches work refuses anything that is not sm_100.
static int check_current_device(int* sms_out) {
    static thread_local int cached_dev = -1, cached_sms = 0, cached_rc = DC_OK;
    int dev = -1;
    DC_CUDA(cudaGetDevice(&dev));
    if (dev != cached_dev) {
        cudaDeviceProp prop;
        DC_CUDA(cudaGetDeviceProperties(&prop, dev));
        cached_dev = dev;
        cached_sms = prop.multiProcessorCount;
        cached_rc = (prop.major == 10) ? DC_OK : DC_EDEVICE;
        if (cached_rc != DC_OK)
            set_error("device %d (%s) is compute capability %d.%d; this library is sm_100a only and has no fallback",
                      dev, prop.name, prop.major, prop.minor);
    } else if (cached_rc != DC_OK) {
        set_error("current device is not compute capability 10.x; this library is sm_100a only and has no fallback");
    }
    if (sms_out) *sms_out = cached_sms;
    return cached_rc;
}

int num_sms() {
    int sms = 0;
    check_current_device(&sms);
    return sms > 0 ? sms : 148;
}

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

}  // namespace dc

using namespace dc;

struct dc_model {
    int device;
    dc_model_desc_t desc;
    int cin, cout;           // UNetDC(in_channels, out_channels); (3, 1) is the fused path
    float head_b;
    // host copies of the biases of the 64-channel layers (enc1.0, enc1.3, upconv1, dec1.0): their kernels take the
    // bias as kernel parameters (constant-bank operands) instead of staging it in shared memory
    float bias64[DC_NUM_LAYERS][64];
    bool has_bias64[DC_NUM_LAYERS];
    bool fused1;             // upconv1 + dec1.0 as one launch (desc.fused_weight1)
    bool fused[4];           // [l]: upconv{l+1} + dec{l+1}.0 as one launch ([0] == fused1)
    float fused_bias9[9 * 64];
};

namespace {

// Activation buffers of one forward, carved out of the caller's workspace (all bf16 NHWC).
struct ForwardBuffers {
    char* a[5];      // first-conv output of enc1..enc4 / bottleneck
    char* ad[4];     // dec{l}.0 output
    char* cat[4];    // [B,Hl,Wl,2*Cl]: channels [0,Cl) <- upconv, [Cl,2Cl) <- encoder skip (torch.cat order)
    char* pool[4];   // 2x2 max-pooled encoder output
    char* bott;      // bottleneck.3 output
    char* db[4];     // dec{l}.3 output for l = 1..3 (index l); dec1.3 goes straight to the head
    char* xin;       // in_channels != 3: the input as bf16 NHWC padded to 64 channels
    char* feat;      // out_channels != 1: dec1.3 output for the 1x1 head kernel
    size_t total;
};

// Buffers are placed by lifetime: [t0, t1] = first launch that writes .. last launch that reads (launch numbers of
// forward_impl below); two buffers may share memory when their lifetimes do not intersect.  Largest first, each at
// the lowest offset that is free for its whole lifetime.  At 32 x 1024^2 this is 15.6 GB (the skip halves of cat[0..3]
// have to survive the whole bottom of the U) instead of the 30.5 GB of one private buffer per tensor.
// fused[l] (upconv{l+1} + dec{l+1}.0 as one launch, at the number of the dec launch): cat[l] holds only the skip half,
// and the transposed conv's input is read by the launch that writes ad[l], so it has to live one launch longer.
ForwardBuffers carve(char* base, int B, int H, int W, bool generic_in = false, bool generic_out = false,
                     const bool* fused = nullptr) {
    const bool none[4] = {false, false, false, false};
    if (!fused) fused = none;
    ForwardBuffers f;
    memset(&f, 0, sizeof(f));
    struct Item { size_t bytes; int t0, t1; char** slot; size_t off; };
    Item items[24];
    int n = 0;
    auto add = [&](char** slot, size_t elems, int t0, int t1) {
        Item it = {align256(elems * 2), t0, t1, slot, 0};
        items[n++] = it;
    };
    if (generic_in) add(&f.xin, (size_t)B * H * W * 64, -1, 0);
    if (generic_out) add(&f.feat, (size_t)B * H * W * 64, 21, 22);
    for (int l = 0; l < 5; ++l) {
        const size_t px = (size_t)B * (H >> l) * (W >> l);
        const size_t C = (size_t)64 << l;
        add(&f.a[l], px * C, 2 * l, 2 * l + 1);
        if (l < 4) {
            add(&f.cat[l], px * (fused[l] ? 1 : 2) * C, 2 * l + 1, 20 - 3 * l);
            add(&f.pool[l], px / 4 * C, 2 * l + 1, 2 * l + 2);
            add(&f.ad[l], px * C, 20 - 3 * l, 21 - 3 * l);
            if (l > 0) add(&f.db[l], px * C, 21 - 3 * l, 22 - 3 * l + (fused[l - 1] ? 1 : 0));
        } else {
            add(&f.bott, px * C, 9, 10 + (fused[3] ? 1 : 0));
        }
    }
    int order[24];
    for (int i = 0; i < n; ++i) order[i] = i;
    for (int i = 1; i < n; ++i)                              // insertion sort, bytes descending (stable)
        for (int j = i; j > 0 && items[order[j]].bytes > items[order[j - 1]].bytes; --j) {
            int t = order[j]; order[j] = order[j - 1]; order[j - 1] = t;
        }
    size_t total = 0;
    for (int oi = 0; oi < n; ++oi) {
        Item& it = items[order[oi]];
        size_t best = 0;
        bool moved = true;
        while (moved) {                                       // lowest offset with no live neighbour overlapping it
            moved = false;
            for (int oj = 0; oj < oi; ++oj) {
                const Item& o = items[order[oj]];
                if (o.t1 < it.t0 || it.t1 < o.t0) continue;   // never alive together
                if (best < o.off + o.bytes && o.off < best + it.bytes) { best = o.off + o.bytes; moved = true; }
            }
        }
        it.off = best;
        if (best + it.bytes > total) total = best + it.bytes;
    }
    for (int i = 0; i < n; ++i) *items[i].slot = base ? base + items[i].off : nullptr;
    f.total = total;
    return f;
}

}  // namespace

extern "C" {

const char* dc_last_error(void) { return g_err; }

int dc_version(void) { return DC_ABI_VERSION; }

int dc_debug_set_conv_family(int family) { return set_conv_family(family); }

int dc_debug_upfuse_schedule(int* out, int cap) { return upfuse_schedule(out, cap); }

int dc_debug_set_upfuse_mode(int mode) { return set_upfuse_mode(mode); }

int dc_device_check(int device, int* sm_count) {
    cudaDeviceProp prop;
    DC_CUDA(cudaGetDeviceProperties(&prop, device));
    if (sm_count) *sm_count = prop.multiProcessorCount;
    DC_REQUIRE(prop.major == 10, DC_EDEVICE, "device %d (%s) is compute capability %d.%d, need 10.x", device, prop.name,
               prop.major, prop.minor);
    return DC_OK;
}

int dc_conv_tc(const dc_conv_args_t* args, void* stream) {
    int rc = check_current_device(nullptr);
    if (rc != DC_OK) return rc;
    return launch_conv_tc(args, (cudaStream_t)stream);
}

int dc_conv_upfused(const dc_upfuse_args_t* args, void* stream) {
    int rc = check_current_device(nullptr);
    if (rc != DC_OK) return rc;
    DC_REQUIRE(args && args->bias9, DC_EINVAL, "dc_conv_upfused: null argument");
    float bias9[9 * 64];        // single-layer entry (tests): level 1's interior row travels as kernel parameters
    if (args->channels == 0 || args->channels == 64)
        DC_CUDA(cudaMemcpy(bias9, args->bias9, sizeof(bias9), cudaMemcpyDeviceToHost));
    return launch_conv_upfused(args, (cudaStream_t)stream, bias9);
}

int dc_stem(const dc_stem_args_t* args, void* stream) {
    int rc = check_current_device(nullptr);
    if (rc != DC_OK) return rc;
    return launch_stem(args, (cudaStream_t)stream);
}

int dc_rolling_ball_workspace_bytes(int B, int H, int W, int C, size_t* bytes) {
    DC_REQUIRE(bytes && B > 0 && H > 0 && W > 0 && C > 0, DC_EINVAL, "dc_rolling_ball_workspace_bytes: bad argument");
    *bytes = rolling_ball_workspace_bytes(B * C, H, W);
    return DC_OK;
}

int dc_rolling_ball_max_radius(void) { return rolling_ball_max_radius(); }

int dc_rolling_ball_tiled_max_radius(void) { return rolling_ball_tiled_max_radius(); }

int dc_debug_rolling_ball_plan(int radius, int tile_h, int* out, int cap) { return rolling_ball_plan_dump(radius, tile_h, out, cap); }

int dc_debug_rolling_ball_bands(int radius, int* out, int cap) { return rolling_ball_bands_dump(radius, out, cap); }

int dc_rolling_ball(const dc_rolling_ball_args_t* args, void* stream) {
    int rc = check_current_device(nullptr);
    if (rc != DC_OK) return rc;
    return launch_rolling_ball(args, (cudaStream_t)stream, false);
}

int dc_rolling_ball_tiled(const dc_rolling_ball_args_t* args, void* stream) {
    int rc = check_current_device(nullptr);
    if (rc != DC_OK) return rc;
    return launch_rolling_ball(args, (cudaStream_t)stream, true);
}

int dc_rolling_ball_banded(const dc_rolling_ball_args_t* args, void* stream) {
    int rc = check_current_device(nullptr);
    if (rc != DC_OK) return rc;
    return launch_rolling_ball_banded(args, (cudaStream_t)stream, "dc_rolling_ball_banded");
}

int dc_resize_linear_u8(const dc_resize_args_t* args, void* stream) {
    int rc = check_current_device(nullptr);
    if (rc != DC_OK) return rc;
    return launch_resize_linear_u8(args, (cudaStream_t)stream);
}

int dc_label_workspace_bytes(int B, int H, int W, size_t* bytes) {
    DC_REQUIRE(bytes && B > 0 && H > 0 && W > 0, DC_EINVAL, "dc_label_workspace_bytes: bad argument");
    *bytes = label_workspace_bytes(B, H, W);
    return DC_OK;
}

int dc_label_stats(const dc_label_args_t* args, void* stream) {
    int rc = check_current_device(nullptr);
    if (rc != DC_OK) return rc;
    return launch_label_stats(args, (cudaStream_t)stream);
}

int dc_overlay_workspace_bytes(int B, int H, int W, size_t* bytes) {
    DC_REQUIRE(bytes && B > 0 && H > 0 && W > 0, DC_EINVAL, "dc_overlay_workspace_bytes: bad argument");
    *bytes = overlay_workspace_bytes(B, H, W);
    return DC_OK;
}

int dc_overlay_stencil(const dc_overlay_args_t* args, void* stream) {
    int rc = check_current_device(nullptr);
    if (rc != DC_OK) return rc;
    return launch_overlay_stencil(args, (cudaStream_t)stream);
}

int dc_roi_workspace_bytes(int B, int H, int W, size_t* bytes) {
    DC_REQUIRE(bytes && B > 0 && H > 0 && W > 0, DC_EINVAL, "dc_roi_workspace_bytes: bad argument");
    *bytes = roi_workspace_bytes(B, H, W);
    return DC_OK;
}

int dc_roi_mask(const dc_roi_args_t* args, void* stream) {
    int rc = check_current_device(nullptr);
    if (rc != DC_OK) return rc;
    return launch_roi_mask(args, (cudaStream_t)stream);
}

int dc_radial_workspace_bytes(int B, size_t* bytes) {
    DC_REQUIRE(bytes && B > 0, DC_EINVAL, "dc_radial_workspace_bytes: bad argument");
    *bytes = radial_workspace_bytes(B);
    return DC_OK;
}

int dc_radial_density(const dc_radial_args_t* args, void* stream) {
    int rc = check_current_device(nullptr);
    if (rc != DC_OK) return rc;
    return launch_radial_density(args, (cudaStream_t)stream);
}

int dc_spatial_workspace_bytes(int B, int H, int W, size_t* bytes) {
    DC_REQUIRE(bytes && B > 0 && H > 0 && W > 0, DC_EINVAL, "dc_spatial_workspace_bytes: bad argument");
    *bytes = spatial_workspace_bytes(B, H, W);
    return DC_OK;
}

int dc_spatial_density(const dc_spatial_args_t* args, void* stream) {
    int rc = check_current_device(nullptr);
    if (rc != DC_OK) return rc;
    return launch_spatial_density(args, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------ whole network

int dc_model_create(dc_model_t** out, int device, const dc_model_desc_t* desc) {
    DC_REQUIRE(out && desc, DC_EINVAL, "dc_model_create: null argument");
    *out = nullptr;
    int rc = dc_device_check(device, nullptr);
    if (rc != DC_OK) return rc;
    DC_REQUIRE(desc->base_channels == 64, DC_EINVAL, "dc_model_create: base_channels must be 64 (got %d)",
               desc->base_channels);
    for (int i = 0; i < DC_NUM_LAYERS; ++i)
        DC_REQUIRE(desc->weight[i] && desc->bias[i], DC_EINVAL, "dc_model_create: layer %d has a null blob", i);
    for (int i = 0; i < 5; ++i)
        DC_REQUIRE(desc->dilations[i] >= 1 && desc->dilations[i] <= 64, DC_EINVAL, "dc_model_create: dilation[%d] = %d", i,
                   desc->dilations[i]);
    const int cin = desc->in_channels > 0 ? desc->in_channels : 3, cout = desc->out_channels > 0 ? desc->out_channels : 1;
    DC_REQUIRE(cin <= 64 && cout <= 64, DC_EINVAL, "dc_model_create: in_channels %d / out_channels %d (at most 64)", cin, cout);
    dc_model* m = new (std::nothrow) dc_model;
    DC_REQUIRE(m, DC_EINVAL, "dc_model_create: out of host memory");
    m->device = device;
    m->desc = *desc;
    m->cin = cin;
    m->cout = cout;
    cudaError_t e = cudaMemcpy(&m->head_b, desc->bias[22], sizeof(float), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) {
        delete m;
        return cuda_fail(e, "cudaMemcpy(out_conv.bias)");
    }
    memset(m->has_bias64, 0, sizeof(m->has_bias64));
    for (int layer : {0, 1, 19, 20}) {
        if (layer == 0 && cin != 3) continue;          // enc1.0 then runs as an ordinary conv layer
        e = cudaMemcpy(m->bias64[layer], desc->bias[layer], 64 * sizeof(float), cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) {
            delete m;
            return cuda_fail(e, "cudaMemcpy(bias of a 64-channel layer)");
        }
        m->has_bias64[layer] = true;
    }
    m->fused1 = desc->fused_weight1 != nullptr;
    m->fused[0] = m->fused1;
    for (int l = 1; l < 4; ++l) {
        m->fused[l] = desc->fused_wide_x[l - 1] != nullptr;
        if (m->fused[l] && !(desc->fused_wide_s[l - 1] && desc->fused_wide_b[l - 1])) {
            delete m;
            set_error("dc_model_create: fused_wide_x[%d] without fused_wide_s / fused_wide_b", l - 1);
            return DC_EINVAL;
        }
    }
    if (m->fused1) {
        e = desc->fused_bias1 ? cudaMemcpy(m->fused_bias9, desc->fused_bias1, sizeof(m->fused_bias9), cudaMemcpyDeviceToHost)
                              : cudaErrorInvalidValue;
        if (e != cudaSuccess) {
            delete m;
            return cuda_fail(e, "cudaMemcpy(fused_bias1)");
        }
    }
    *out = m;
    return DC_OK;
}

int dc_model_destroy(dc_model_t* m) {
    delete m;
    return DC_OK;
}

int dc_forward_workspace_bytes(const dc_model_t* m, int B, int H, int W, size_t* bytes) {
    DC_REQUIRE(m && bytes, DC_EINVAL, "dc_forward_workspace_bytes: null argument");
    DC_REQUIRE(B > 0 && H > 0 && W > 0 && H % 16 == 0 && W % 16 == 0, DC_EINVAL,
               "dc_forward: H and W must be positive multiples of 16 (got %d x %d x %d)", B, H, W);
    *bytes = carve(nullptr, B, H, W, m->cin != 3, m->cout != 1, m->fused).total;
    return DC_OK;
}

int dc_forward_num_launches(const dc_model_t* m) {
    // stem + 17 conv3x3 + 4 upconv (+ the input conversion / the 1x1 head kernel for other channel counts), minus one per
    // decoder level whose upconv is composed into the following conv
    int n = 22 + (m && m->cin != 3 ? 1 : 0) + (m && m->cout != 1 ? 1 : 0);
    for (int l = 0; m && l < 4; ++l) n -= m->fused[l] ? 1 : 0;
    return n;
}

}  // extern "C"

// One forward; when `ev` is non-NULL it receives DC_FORWARD_LAUNCHES + 1 events recorded around the launches.
static int forward_impl(dc_model_t* m, int in_kind, const void* in, int B, int H, int W, float thresh, float* prob_out,
                        uint8_t* mask_out, void* workspace, size_t workspace_bytes, void* stream_, cudaEvent_t* ev) {
    DC_REQUIRE(m && in && workspace, DC_EINVAL, "dc_forward: null argument");
    DC_REQUIRE(prob_out || mask_out, DC_EINVAL, "dc_forward: prob_out and mask_out are both NULL");
    DC_REQUIRE(B > 0 && H > 0 && W > 0 && H % 16 == 0 && W % 16 == 0, DC_EINVAL,
               "dc_forward: H and W must be positive multiples of 16 (got %d x %d x %d)", B, H, W);
    int rc = check_current_device(nullptr);
    if (rc != DC_OK) return rc;
    int dev = -1;
    DC_CUDA(cudaGetDevice(&dev));
    DC_REQUIRE(dev == m->device, DC_EINVAL, "dc_forward: model lives on device %d, current device is %d", m->device, dev);
    const bool gen_in = m->cin != 3, gen_out = m->cout != 1;
    DC_REQUIRE(!gen_in || in_kind == 0, DC_EINVAL, "dc_forward: u8 inputs need in_channels == 3 (model has %d)", m->cin);
    ForwardBuffers f = carve((char*)workspace, B, H, W, gen_in, gen_out, m->fused);
    DC_REQUIRE(workspace_bytes >= f.total, DC_EWORKSPACE, "dc_forward: workspace too small (%zu < %zu)", workspace_bytes,
               f.total);
    DC_REQUIRE(((uintptr_t)workspace & 255) == 0, DC_EINVAL, "dc_forward: workspace must be 256-byte aligned");
    cudaStream_t stream = (cudaStream_t)stream_;
    const dc_model_desc_t& d = m->desc;

    auto conv = [&](int layer, int kind, int epi, int relu, int h, int w, int cin, int cout, int dil, const void* src,
                    int src_stride, void* dst, int dst_stride, int dst_off, void* pool) -> int {
        dc_conv_args_t a;
        memset(&a, 0, sizeof(a));
        a.kind = kind; a.epilogue = epi; a.relu = relu;
        a.B = B; a.H = h; a.W = w; a.Cin = cin; a.Cout = cout; a.dilation = dil;
        a.in = src; a.in_stride = src_stride;
        a.weight = d.weight[layer]; a.bias = d.bias[layer];
        a.out = dst; a.out_stride = dst_stride; a.out_offset = dst_off;
        a.pool_out = pool; a.pool_stride = cout;
        if (layer == 1) a.weight_par = d.par_weight[0];        // launch_conv_tc takes it only when dilation == 1
        if (layer == 21) a.weight_par = d.par_weight[1];
        if (epi == DC_EPI_HEAD) {
            a.head_w = (const float*)d.weight[22];
            a.head_b = m->head_b;
            a.thresh = thresh;
            a.prob_out = prob_out;
            a.mask_out = mask_out;
        }
        return launch_conv_tc(&a, stream, m->has_bias64[layer] ? m->bias64[layer] : nullptr);
    };
    int launch_no = 0;
#define DC_TRY(x)                                                        \
    do {                                                                 \
        if (ev && launch_no == 0) DC_CUDA(cudaEventRecord(ev[0], stream)); \
        int _rc = (x);                                                   \
        if (_rc != DC_OK) return _rc;                                    \
        ++launch_no;                                                     \
        if (ev) DC_CUDA(cudaEventRecord(ev[launch_no], stream));         \
    } while (0)

    // encoder (model_2.py:58-61) -- layer ids per include/unetdc_b200.h
    if (gen_in) {
        DC_TRY(launch_pad_input((const float*)in, f.xin, B, m->cin, H, W, stream));
        DC_TRY(conv(0, DC_KIND_CONV3X3, DC_EPI_STORE, 1, H, W, 64, 64, d.dilations[0], f.xin, 64, f.a[0], 64, 0, nullptr));
    } else {
        dc_stem_args_t s;
        memset(&s, 0, sizeof(s));
        s.in_kind = in_kind; s.B = B; s.H = H; s.W = W; s.Cout = 64; s.dilation = d.dilations[0];
        s.in = in; s.weight = (const float*)d.weight[0]; s.bias = d.bias[0];
        s.out = f.a[0]; s.out_stride = 64; s.out_offset = 0;
        DC_TRY(launch_stem(&s, stream, m->has_bias64[0] ? m->bias64[0] : nullptr));
    }
    DC_TRY(conv(1, DC_KIND_CONV3X3, DC_EPI_STORE_POOL, 1, H, W, 64, 64, d.dilations[0], f.a[0], 64, f.cat[0],
                m->fused1 ? 64 : 128, m->fused1 ? 0 : 64, f.pool[0]));
    for (int l = 1; l < 4; ++l) {
        const int h = H >> l, w = W >> l, c = 64 << l;
        DC_TRY(conv(2 * l, DC_KIND_CONV3X3, DC_EPI_STORE, 1, h, w, c / 2, c, d.dilations[l], f.pool[l - 1], c / 2, f.a[l], c,
                    0, nullptr));
        DC_TRY(conv(2 * l + 1, DC_KIND_CONV3X3, DC_EPI_STORE_POOL, 1, h, w, c, c, d.dilations[l], f.a[l], c, f.cat[l],
                    m->fused[l] ? c : 2 * c, m->fused[l] ? 0 : c, f.pool[l]));
    }
    // bottleneck (model_2.py:64)
    DC_TRY(conv(8, DC_KIND_CONV3X3, DC_EPI_STORE, 1, H >> 4, W >> 4, 512, 1024, d.dilations[4], f.pool[3], 512, f.a[4], 1024,
                0, nullptr));
    DC_TRY(conv(9, DC_KIND_CONV3X3, DC_EPI_STORE, 1, H >> 4, W >> 4, 1024, 1024, d.dilations[4], f.a[4], 1024, f.bott, 1024,
                0, nullptr));
    // decoder (model_2.py:67-77): upconv -> [up | skip] -> double conv, dilation 1
    const void* src = f.bott;
    for (int l = 3; l >= 0; --l) {
        const int h = H >> l, w = W >> l, c = 64 << l;
        const int base = 10 + 3 * (3 - l);
        if (m->fused[l]) {
            // upconv + dec.0 in one launch: `up` (channels [0,c) of cat[l]) is never written, cat[l] is the skip alone
            dc_upfuse_args_t u;
            memset(&u, 0, sizeof(u));
            u.B = B; u.H = h / 2; u.W = w / 2; u.channels = c;
            u.x = src; u.x_stride = 2 * c;
            u.skip = f.cat[l]; u.skip_stride = c;
            u.weight = l == 0 ? d.fused_weight1 : d.fused_wide_x[l - 1];
            u.weight_skip = l == 0 ? nullptr : d.fused_wide_s[l - 1];
            u.bias9 = l == 0 ? d.fused_bias1 : d.fused_wide_b[l - 1];
            u.relu = 1;
            u.out = f.ad[l]; u.out_stride = c; u.out_offset = 0;
            DC_TRY(launch_conv_upfused(&u, stream, m->fused_bias9));
        } else {
        DC_TRY(conv(base, DC_KIND_UPCONV2, DC_EPI_UPSCATTER, 0, h / 2, w / 2, 2 * c, c, 1, src, 2 * c, f.cat[l], 2 * c, 0,
                    nullptr));
        DC_TRY(conv(base + 1, DC_KIND_CONV3X3, DC_EPI_STORE, 1, h, w, 2 * c, c, 1, f.cat[l], 2 * c, f.ad[l], c, 0, nullptr));
        }
        if (l > 0) {
            DC_TRY(conv(base + 2, DC_KIND_CONV3X3, DC_EPI_STORE, 1, h, w, c, c, 1, f.ad[l], c, f.db[l], c, 0, nullptr));
            src = f.db[l];
        } else if (!gen_out) {
            // dec1.3 + out_conv + sigmoid + threshold (model_2.py:79-80, qdb:56)
            DC_TRY(conv(base + 2, DC_KIND_CONV3X3, DC_EPI_HEAD, 1, h, w, c, c, 1, f.ad[l], c, nullptr, 0, 0, nullptr));
        } else {
            DC_TRY(conv(base + 2, DC_KIND_CONV3X3, DC_EPI_STORE, 1, h, w, c, c, 1, f.ad[l], c, f.feat, c, 0, nullptr));
            DC_TRY(launch_head1x1(f.feat, (const float*)d.weight[22], d.bias[22], prob_out, mask_out, thresh, B, m->cout, H, W,
                                  stream));
        }
    }
#undef DC_TRY
    return DC_OK;
}

extern "C" {

int dc_forward(dc_model_t* m, int in_kind, const void* in, int B, int H, int W, float thresh, float* prob_out,
               uint8_t* mask_out, void* workspace, size_t workspace_bytes, void* stream) {
    return forward_impl(m, in_kind, in, B, H, W, thresh, prob_out, mask_out, workspace, workspace_bytes, stream, nullptr);
}

int dc_forward_profile(dc_model_t* m, int in_kind, const void* in, int B, int H, int W, float thresh, float* prob_out,
                       uint8_t* mask_out, void* workspace, size_t workspace_bytes, void* stream, float* launch_ms) {
    DC_REQUIRE(launch_ms, DC_EINVAL, "dc_forward_profile: launch_ms is NULL");
    const int n = dc_forward_num_launches(m);
    cudaEvent_t ev[64];
    for (int i = 0; i <= n; ++i) DC_CUDA(cudaEventCreate(&ev[i]));
    int rc = forward_impl(m, in_kind, in, B, H, W, thresh, prob_out, mask_out, workspace, workspace_bytes, stream, ev);
    if (rc == DC_OK) {
        cudaError_t e = cudaStreamSynchronize((cudaStream_t)stream);
        if (e != cudaSuccess) rc = cuda_fail(e, "cudaStreamSynchronize");
    }
    for (int i = 0; i < n && rc == DC_OK; ++i) {
        cudaError_t e = cudaEventElapsedTime(&launch_ms[i], ev[i], ev[i + 1]);
        if (e != cudaSuccess) rc = cuda_fail(e, "cudaEventElapsedTime");
    }
    for (int i = 0; i <= n; ++i) cudaEventDestroy(ev[i]);
    return rc;
}

}  // extern "C"
