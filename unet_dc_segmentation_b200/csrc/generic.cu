// generic.cu -- the two plain kernels that let UNetDC(in_channels, out_channels) (reference models/model_2.py:6,10,32)
// take channel counts other than the (3, 1) the inference script builds (quantify_droplets_batch.py:35).  They wrap
// the tensor-core layers; the bf16 (3, 1) network never launches them.  The fp32-precision forward (DC_PRECISION_FP32)
// always starts with split_input_kernel and, for out_channels != 1, ends with the three-plane head1x1_kernel.
#include "common.cuh"

#include <algorithm>

namespace dc {

namespace {

// fp32 NCHW [B,C,H,W] -> bf16 NHWC [B,H,W,64], channels >= C zero: enc1.0 then runs as an ordinary 64-channel layer
// (images b = blockIdx.y, blockIdx.y + gridDim.y, ...: gridDim.y stops at 65535, the batch does not)
__global__ void pad_nchw_to_nhwc64_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out, int B, int C,
                                          long long HW) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;       // pixel within the image
    if (p >= HW) return;
    for (int img = blockIdx.y; img < B; img += gridDim.y) {
        const float* src = in + (size_t)img * C * HW + p;
        uint4* dst = reinterpret_cast<uint4*>(out + ((size_t)img * HW + p) * 64);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            unsigned w[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int c0 = q * 8 + j * 2;
                const float a = c0 < C ? src[(size_t)c0 * HW] : 0.f;
                const float b = c0 + 1 < C ? src[(size_t)(c0 + 1) * HW] : 0.f;
                __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
                w[j] = *reinterpret_cast<unsigned*>(&h);
            }
            dst[q] = make_uint4(w[0], w[1], w[2], w[3]);
        }
    }
}

// x -> (hi, mid, lo) with hi + (mid + lo) == x exactly in fp32 (the three planes of DC_PRECISION_FP32).  hi rounds to
// nearest, except where that would overflow bf16 (|x| within half a bf16 ulp of FLT_MAX): then the largest finite bf16.
__device__ __forceinline__ void split3(float x, __nv_bfloat16& hi, __nv_bfloat16& mid, __nv_bfloat16& lo) {
    hi = __float2bfloat16_rn(x);
    if (isinf(__bfloat162float(hi)) && !isinf(x)) hi = __float2bfloat16_rz(x);
    const float r = x - __bfloat162float(hi);
    mid = __float2bfloat16_rn(r);
    lo = __float2bfloat16_rn(r - __bfloat162float(mid));
}

// DC_PRECISION_FP32 input: fp32 NCHW [B,C,H,W] (in_kind 0), u8 grey [B,H,W] replicated to 3 channels (1) or u8 HWC
// [B,H,W,3] (2) -> three bf16 planes [B,H,W][3][64], channels >= C zero.  u8 values become u8 / 255 as an IEEE fp32
// division, as the reference's preprocessing computes them (quantify_droplets_batch.py:45).
__global__ void split_input_kernel(const void* __restrict__ in, int in_kind, __nv_bfloat16* __restrict__ out, int B, int C,
                                   long long HW) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= HW) return;
    for (int img = blockIdx.y; img < B; img += gridDim.y) {
        uint4* dst = reinterpret_cast<uint4*>(out + ((size_t)img * HW + p) * 192);
        for (int q = 0; q < 8; ++q) {                          // channels [8q, 8q + 8) of the three planes
            __align__(16) __nv_bfloat16 pl[3][8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int c = 8 * q + j;
                float v = 0.f;
                if (c < C) {
                    if (in_kind == 0) v = static_cast<const float*>(in)[((size_t)img * C + c) * HW + p];
                    else {
                        const uint8_t* u = static_cast<const uint8_t*>(in);
                        v = __fdiv_rn((float)(in_kind == 1 ? u[(size_t)img * HW + p] : u[((size_t)img * HW + p) * 3 + c]), 255.f);
                    }
                }
                split3(v, pl[0][j], pl[1][j], pl[2][j]);
            }
#pragma unroll
            for (int k = 0; k < 3; ++k) dst[8 * k + q] = *reinterpret_cast<const uint4*>(pl[k]);
        }
    }
}

// out_conv (1x1, 64 -> OC) + sigmoid (+ threshold of channel 0) on the bf16 NHWC feature map of dec1.3
// (models/model_2.py:79-80, quantify_droplets_batch.py:56).  PLANES == 3: the map is [B,H,W][3][64] (DC_PRECISION_FP32)
// and the features are the fp32 values hi + (mid + lo).
template <int PLANES>
__global__ void head1x1_kernel(const __nv_bfloat16* __restrict__ feat, const float* __restrict__ w, const float* __restrict__ b,
                               float* __restrict__ prob, uint8_t* __restrict__ mask, float thresh, int B, int OC,
                               long long HW) {
    extern __shared__ float ws[];                  // [OC][64] weights, then [OC] biases
    for (int i = threadIdx.x; i < OC * 64; i += blockDim.x) ws[i] = w[i];
    for (int i = threadIdx.x; i < OC; i += blockDim.x) ws[OC * 64 + i] = b[i];
    __syncthreads();
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= HW) return;
    for (int b = blockIdx.y; b < B; b += gridDim.y) {          // as in pad_nchw_to_nhwc64_kernel
        float x[64];
#pragma unroll
        for (int pl = PLANES - 1; pl >= 0; --pl) {             // lo, mid, hi: x = hi + (mid + lo)
            const uint4* src = reinterpret_cast<const uint4*>(feat + ((size_t)b * HW + p) * 64 * PLANES + 64 * pl);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const uint4 v = src[q];
                const unsigned u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&u[j]);
                    const float a = __low2float(h), c = __high2float(h);
                    x[q * 8 + 2 * j] = pl == PLANES - 1 ? a : a + x[q * 8 + 2 * j];
                    x[q * 8 + 2 * j + 1] = pl == PLANES - 1 ? c : c + x[q * 8 + 2 * j + 1];
                }
            }
        }
        for (int o = 0; o < OC; ++o) {
            float acc = ws[OC * 64 + o];
#pragma unroll
            for (int c = 0; c < 64; ++c) acc = fmaf(x[c], ws[o * 64 + c], acc);
            const float pr = 1.0f / (1.0f + expf(-acc));
            if (prob) prob[((size_t)b * OC + o) * HW + p] = pr;
            if (o == 0 && mask) mask[(size_t)b * HW + p] = pr > thresh ? 1 : 0;
        }
    }
}

}  // namespace

int launch_pad_input(const float* in, void* out_nhwc64, int B, int C, int H, int W, cudaStream_t stream) {
    DC_REQUIRE(in && out_nhwc64 && C >= 1 && C <= 64, DC_EINVAL, "dc_forward: in_channels %d outside [1,64]", C);
    const long long HW = (long long)H * W;
    pad_nchw_to_nhwc64_kernel<<<dim3((unsigned)((HW + 255) / 256), std::min(B, 65535)), 256, 0, stream>>>(
        in, reinterpret_cast<__nv_bfloat16*>(out_nhwc64), B, C, HW);
    DC_CUDA(cudaGetLastError());
    return DC_OK;
}

int launch_split_input(const void* in, int in_kind, int C, void* out_planes, int B, int H, int W, cudaStream_t stream) {
    DC_REQUIRE(in && out_planes && C >= 1 && C <= 64, DC_EINVAL, "dc_forward: in_channels %d outside [1,64]", C);
    DC_REQUIRE(in_kind == 0 || ((in_kind == 1 || in_kind == 2) && C == 3), DC_EINVAL,
               "dc_forward: in_kind %d (u8 inputs need in_channels == 3, model has %d)", in_kind, C);
    const long long HW = (long long)H * W;
    split_input_kernel<<<dim3((unsigned)((HW + 127) / 128), std::min(B, 65535)), 128, 0, stream>>>(
        in, in_kind, reinterpret_cast<__nv_bfloat16*>(out_planes), B, C, HW);
    DC_CUDA(cudaGetLastError());
    return DC_OK;
}

int launch_head1x1(const void* feat_nhwc64, const float* w, const float* b, float* prob, uint8_t* mask, float thresh, int B,
                   int OC, int H, int W, cudaStream_t stream, int planes) {
    DC_REQUIRE(feat_nhwc64 && w && b && OC >= 1 && OC <= 64, DC_EINVAL, "dc_forward: out_channels %d outside [1,64]", OC);
    const long long HW = (long long)H * W;
    const dim3 grid((unsigned)((HW + 127) / 128), std::min(B, 65535));
    const size_t smem = (size_t)(OC * 65) * sizeof(float);
    if (planes == 3)
        head1x1_kernel<3><<<grid, 128, smem, stream>>>(reinterpret_cast<const __nv_bfloat16*>(feat_nhwc64), w, b, prob, mask,
                                                       thresh, B, OC, HW);
    else
        head1x1_kernel<1><<<grid, 128, smem, stream>>>(reinterpret_cast<const __nv_bfloat16*>(feat_nhwc64), w, b, prob, mask,
                                                       thresh, B, OC, HW);
    DC_CUDA(cudaGetLastError());
    return DC_OK;
}

}  // namespace dc
