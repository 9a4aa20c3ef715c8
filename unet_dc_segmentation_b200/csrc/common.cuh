// common.cuh -- shared helpers for the sm_100a kernels of the droplet-quantification path.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/unetdc_b200.h"

namespace dc {

// ---------------------------------------------------------------- error plumbing (api.cu)
void set_error(const char* fmt, ...);
int  cuda_fail(cudaError_t e, const char* what);

#define DC_CUDA(call)                                                         \
    do {                                                                      \
        cudaError_t _e = (call);                                              \
        if (_e != cudaSuccess) return dc::cuda_fail(_e, #call);               \
    } while (0)

#define DC_REQUIRE(cond, code, ...)                                           \
    do {                                                                      \
        if (!(cond)) { dc::set_error(__VA_ARGS__); return (code); }           \
    } while (0)

static inline int ceil_div(int a, int b) { return a / b + (a % b != 0); }   // a >= 0, b > 0; no overflow near INT_MAX

// ---------------------------------------------------------------- launchers implemented per .cu
// bias_host: optional HOST copy of a->bias (dc_model_create keeps one); layers with Cout == 64 then take their bias
// from the kernel parameters (constant-bank operands) instead of shared memory.
int launch_conv_tc(const dc_conv_args_t* a, cudaStream_t stream, const float* bias_host = nullptr);
int launch_stem(const dc_stem_args_t* a, cudaStream_t stream, const float* bias_host = nullptr);
// bias9_host: HOST copy of a->bias9 (the interior class becomes kernel parameters); required.
int launch_conv_upfused(const dc_upfuse_args_t* a, cudaStream_t stream, const float* bias9_host);
int set_conv_family(int family);
int upfuse_schedule(int* out, int cap);
int set_upfuse_mode(int mode);
int launch_label_stats(const dc_label_args_t* a, cudaStream_t stream);
int launch_rolling_ball(const dc_rolling_ball_args_t* a, cudaStream_t stream, bool tiled_only);
int launch_rolling_ball_banded(const dc_rolling_ball_args_t* a, cudaStream_t stream, const char* who);
int launch_resize_linear_u8(const dc_resize_args_t* a, cudaStream_t stream);
size_t label_workspace_bytes(int B, int H, int W);
int launch_overlay_stencil(const dc_overlay_args_t* a, cudaStream_t stream);
size_t overlay_workspace_bytes(int B, int H, int W);
int launch_roi_mask(const dc_roi_args_t* a, cudaStream_t stream);
size_t roi_workspace_bytes(int B, int H, int W);
int launch_radial_density(const dc_radial_args_t* a, cudaStream_t stream);
size_t radial_workspace_bytes(int B);
int launch_spatial_density(const dc_spatial_args_t* a, cudaStream_t stream);
size_t spatial_workspace_bytes(int B, int H, int W);
size_t rolling_ball_workspace_bytes(int planes, int H, int W);
int rolling_ball_max_radius();
int rolling_ball_tiled_max_radius();
int rolling_ball_plan_dump(int radius, int th, int* out, int cap);
int rolling_ball_bands_dump(int radius, int* out, int cap);
int num_sms();
int launch_pad_input(const float* in, void* out_nhwc64, int B, int C, int H, int W, cudaStream_t stream);
int launch_head1x1(const void* feat_nhwc64, const float* w, const float* b, float* prob, uint8_t* mask, float thresh, int B,
                   int OC, int H, int W, cudaStream_t stream);

#ifdef __CUDACC__
// ---------------------------------------------------------------- PTX wrappers (sm_100a)
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a pipeline bug must fail the launch (trap), never hang the GPU box.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000ll) {   // ~2 s at 2 GHz: no legitimate wait is this long
            printf("dc: mbarrier timeout block %d thread %d bar %u parity %u\n", (int)blockIdx.x,
                   (int)threadIdx.x, smem_u32(bar), parity);
            __trap();
        }
    }
}

// One lane of a converged warp.  Role loops run warp-uniform and only the issuing instructions sit under this
// predicate: ptxas then keeps descriptors / coordinates in uniform registers and emits UTCHMMA / UTMALDG
// back to back (a role body under `if (lane == 0)` gets an ELECT + branch waterfall around every one).
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(pred));
    return pred != 0;
}

// TMA tiled loads (global -> shared, completion on an mbarrier)
__device__ __forceinline__ void tma_load_2d(void* dst, const void* tmap, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const void* tmap, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
        "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}

// tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {   // one full warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
                 "r"(ncols)
                 : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {      // same warp as alloc
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]; bf16 inputs, fp32 accumulate; issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// mbarrier arrives when every MMA issued so far by this thread has completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread t of the warp gets lane (base_lane + t).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}


// ---------------------------------------------------------------- CTA pairs (cta_group::2)
// Shared-memory addresses of the two CTAs of a pair differ only in this bit of the shared::cluster window;
// clearing it turns "my barrier" into "the leader's (even CTA's) barrier at the same offset".
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA loads issued by either CTA of a pair; the bytes are credited to the LEADER's mbarrier.
__device__ __forceinline__ void tma_load_2d_2sm(void* dst, const void* tmap, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d_2sm(void* dst, const void* tmap, uint64_t* bar, int c0, int c1, int c2,
                                                int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1),
        "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_load_5d_2sm(void* dst, const void* tmap, uint64_t* bar, int c0, int c1, int c2,
                                                int c3, int c4) {
    asm volatile(
        "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1),
        "r"(c2), "r"(c3), "r"(c4)
        : "memory");
}
// arrive on the leader CTA's copy of `bar` (from either CTA of the pair).  Relaxed: what it orders is TMEM reads
// (tcgen05.wait::ld + fence::before_thread_sync), not memory; a release at cluster scope costs MEMBAR.GPU + ERRBAR,
// i.e. a wait for every global store the warp has in flight (13 % of enc1.3's samples).
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
    asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPeerBitMask) : "memory");
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t* dst_smem, uint32_t ncols) {   // one full warp in EACH CTA
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
                 : "memory");
}
__device__ __forceinline__ void tmem_relinquish_2sm() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// M = 256 across the pair: rows [0,128) from the leader's smem, [128,256) from the peer's, same descriptors;
// each CTA supplies N/2 rows of B.  Issued by ONE thread of the leader CTA.
__device__ __forceinline__ void umma_bf16_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                              uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives (once the pair's MMAs issued so far retire) on `bar` in BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)3)
                 : "memory");
}

// K-major, 128-byte-swizzled shared-memory operand descriptor (UMMA "SmemDescriptor"):
// start address >> 4 in [0,14), LBO (unused for swizzled K-major) in [16,30), SBO = 1024 B
// (8 rows x 128 B) >> 4 in [32,46), descriptor version 1 in [46,48), SWIZZLE_128B (2) in [61,64).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// Instruction descriptor for kind::f16: D fp32 (1<<4), A bf16 (1<<7), B bf16 (1<<10),
// both operands K-major, N>>3 in [17,23), M>>4 in [24,29).
__device__ __forceinline__ uint32_t umma_idesc_bf16(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
#endif  // __CUDACC__

}  // namespace dc
