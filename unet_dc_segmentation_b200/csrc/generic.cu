// generic.cu -- the two plain kernels that let UNetDC(in_channels, out_channels) (reference models/model_2.py:6,10,32)
// take channel counts other than the (3, 1) the inference script builds (quantify_droplets_batch.py:35).  They wrap
// the tensor-core layers; the (3, 1) network never launches them.
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

// out_conv (1x1, 64 -> OC) + sigmoid (+ threshold of channel 0) on the bf16 NHWC feature map of dec1.3
// (models/model_2.py:79-80, quantify_droplets_batch.py:56)
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
        const uint4* src = reinterpret_cast<const uint4*>(feat + ((size_t)b * HW + p) * 64);
        float x[64];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const uint4 v = src[q];
            const unsigned u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&u[j]);
                x[q * 8 + 2 * j] = __low2float(h);
                x[q * 8 + 2 * j + 1] = __high2float(h);
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

int launch_head1x1(const void* feat_nhwc64, const float* w, const float* b, float* prob, uint8_t* mask, float thresh, int B,
                   int OC, int H, int W, cudaStream_t stream) {
    DC_REQUIRE(feat_nhwc64 && w && b && OC >= 1 && OC <= 64, DC_EINVAL, "dc_forward: out_channels %d outside [1,64]", OC);
    const long long HW = (long long)H * W;
    head1x1_kernel<<<dim3((unsigned)((HW + 127) / 128), std::min(B, 65535)), 128, (size_t)(OC * 65) * sizeof(float), stream>>>(
        reinterpret_cast<const __nv_bfloat16*>(feat_nhwc64), w, b, prob, mask, thresh, B, OC, HW);
    DC_CUDA(cudaGetLastError());
    return DC_OK;
}

}  // namespace dc
