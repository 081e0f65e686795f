// Shared helpers for the sm_100a SMPLify fitting kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <mutex>
#include <nvtx3/nvToolsExt.h>
#include "../../include/bodyfit_b200.h"

#define BF_MAXJ 55          // SMPL-X kinematic tree
#define BF_MAXNS 20         // 10 betas + 10 expression coefficients
#define BF_MAXNP 100        // theta entries without the face block (86 / 98)
#define BF_THETA_SMEM 112   // per-frame theta storage: a face-parameter row adds 3 + NE <= 23 entries (at most 111)
#define BF_GMM_D 69

void bf_set_error(const char* fmt, ...);

// ---- per-device host state ------------------------------------------------------------------------------------
// Kernel attributes (opt-in shared memory) and the SM count belong to a DEVICE, not to the process: every cache below is
// indexed by the current device, and the slow paths (first use on a device, side-stream / tensor-map tables) take one
// process-wide mutex, so two host threads driving two GPUs (or the same one) do not race.
#define BF_MAXDEV 32
static std::mutex g_bf_mu;
static inline int bf_cur_dev() { int d = 0; cudaGetDevice(&d); return (d >= 0 && d < BF_MAXDEV) ? d : 0; }
static inline int bf_num_sms() {
    static int sms[BF_MAXDEV] = {0};
    const int d = bf_cur_dev();
    if (!sms[d]) {
        std::lock_guard<std::mutex> lk(g_bf_mu);
        int n = 0;
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, d);
        sms[d] = n > 0 ? n : 1;
    }
    return sms[d];
}
// opt a kernel into `smem` bytes of dynamic shared memory on the current device (once per device and size)
template <typename F>
static inline int bf_ensure_smem(F* fn, size_t smem, size_t* cache /* [BF_MAXDEV] */, const char* what) {
    const int d = bf_cur_dev();
    if (cache[d] >= smem) return BF_OK;
    std::lock_guard<std::mutex> lk(g_bf_mu);
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { bf_set_error("cudaFuncSetAttribute(%s, %zu): %s", what, smem, cudaGetErrorString(e)); return BF_ECUDA; }
    cache[d] = smem;
    return BF_OK;
}
// NVTX range around every C-ABI entry point (visible in nsys / ncu --nvtx; a no-op without an attached tool)
struct BfRange {
    explicit BfRange(const char* name) { nvtxRangePushA(name); }
    ~BfRange() { nvtxRangePop(); }
};
#define BF_NVTX() BfRange bf_nvtx_range_(__func__)

#define BF_REQUIRE(cond, msg)                                   \
    do { if (!(cond)) { bf_set_error("%s: %s", __func__, msg); return BF_EINVAL; } } while (0)

// a failed runtime call: report it AND clear the runtime's last-error slot, so that the next launch check of an unrelated
// call does not trip over it
#define BF_CUDA_FAIL(msg)                                                              \
    do { cudaError_t e_ = cudaGetLastError(); bf_set_error("%s: %s (%s)", __func__, msg, cudaGetErrorString(e_)); return BF_ECUDA; } while (0)

#define BF_LAUNCH_CHECK()                                                              \
    do { cudaError_t e_ = cudaGetLastError();                                          \
         if (e_ != cudaSuccess) { bf_set_error("%s: launch failed: %s", __func__,      \
                                               cudaGetErrorString(e_)); return BF_ECUDA; } } while (0)

// theta layout (see include/bodyfit_b200.h)
struct ThetaLayout {
    int nbody, off_betas, off_leye, off_reye, off_lh, off_rh, off_jaw, off_expr, np;
};
// nbetas: 10, or 11 for the SMPL kid model (age='kid': the SMIL template difference is an extra shape direction)
// face (SMPL-X only): the row ends with [jaw 3 | expression nexpr]; without it off_jaw = off_expr = np
__host__ __device__ __forceinline__ ThetaLayout theta_layout(int is_smplx, int nbetas = 10, int face = 0, int nexpr = 0) {
    ThetaLayout t;
    t.nbody = is_smplx ? 63 : 69;
    t.off_betas = 7 + t.nbody;
    t.off_leye = t.off_betas + nbetas;
    t.off_reye = t.off_leye + 3;
    t.off_lh = t.off_reye + 3;
    t.off_rh = t.off_lh + 6;
    t.off_jaw = is_smplx ? t.off_rh + 6 : t.off_betas + nbetas;
    t.off_expr = t.off_jaw + ((is_smplx && face) ? 3 : 0);
    t.np = t.off_expr + ((is_smplx && face) ? nexpr : 0);
    return t;
}
__host__ __device__ __forceinline__ ThetaLayout theta_layout(const BfModel& m) {
    return theta_layout(m.is_smplx, m.NB, m.face, m.NS - m.NB);
}

// round-to-nearest TF32 (10-bit mantissa, low 13 bits zero) and the exact fp32 remainder: x = hi + lo
__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    hi = __uint_as_float(r);
    lo = x - hi;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// R = I + sin(a) K + (1 - cos(a)) K^2 with a = ||r + 1e-8||, K = skew(r / a)
// (smplx.lbs.batch_rodrigues as restated in oracle/smplx_port.py).  Row-major R[9].
__device__ __forceinline__ void rodrigues_fwd(float rx, float ry, float rz, float* R) {
    const float ex = rx + 1e-8f, ey = ry + 1e-8f, ez = rz + 1e-8f;
    const float a = sqrtf(ex * ex + ey * ey + ez * ez);
    const float dx = rx / a, dy = ry / a, dz = rz / a;
    float s, c;
    sincosf(a, &s, &c);
    const float oc = 1.0f - c;
    R[0] = 1.0f + oc * (-(dy * dy + dz * dz));
    R[1] = -s * dz + oc * (dx * dy);
    R[2] = s * dy + oc * (dx * dz);
    R[3] = s * dz + oc * (dx * dy);
    R[4] = 1.0f + oc * (-(dx * dx + dz * dz));
    R[5] = -s * dx + oc * (dy * dz);
    R[6] = -s * dy + oc * (dx * dz);
    R[7] = s * dx + oc * (dy * dz);
    R[8] = 1.0f + oc * (-(dx * dx + dy * dy));
}

// Backward of exactly the composite above (matches autograd of the restatement,
// including the epsilon placement).  G = dL/dR (row-major), out = dL/dr.
__device__ __forceinline__ void rodrigues_bwd(float rx, float ry, float rz, const float* G, float* out) {
    const float ex = rx + 1e-8f, ey = ry + 1e-8f, ez = rz + 1e-8f;
    const float a = sqrtf(ex * ex + ey * ey + ez * ez);
    const float ia = 1.0f / a;
    const float dx = rx * ia, dy = ry * ia, dz = rz * ia;
    float s, c;
    sincosf(a, &s, &c);
    const float oc = 1.0f - c;
    // K and K^2
    const float K[9] = {0.f, -dz, dy, dz, 0.f, -dx, -dy, dx, 0.f};
    const float K2[9] = {-(dy * dy + dz * dz), dx * dy, dx * dz,
                         dx * dy, -(dx * dx + dz * dz), dy * dz,
                         dx * dz, dy * dz, -(dx * dx + dy * dy)};
    float dLds = 0.f, dLdoc = 0.f;
#pragma unroll
    for (int i = 0; i < 9; ++i) { dLds += G[i] * K[i]; dLdoc += G[i] * K2[i]; }
    // dL/dK = s G + oc (G K^T + K^T G)
    float dK[9];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            float h = 0.f;
#pragma unroll
            for (int k = 0; k < 3; ++k) h += G[i * 3 + k] * K[j * 3 + k] + K[k * 3 + i] * G[k * 3 + j];
            dK[i * 3 + j] = s * G[i * 3 + j] + oc * h;
        }
    const float ddx = dK[7] - dK[5];
    const float ddy = dK[2] - dK[6];
    const float ddz = dK[3] - dK[1];
    float dLda = dLds * c + dLdoc * s;
    dLda -= (ddx * rx + ddy * ry + ddz * rz) * ia * ia;
    out[0] = ddx * ia + dLda * ex * ia;
    out[1] = ddy * ia + dLda * ey * ia;
    out[2] = ddz * ia + dLda * ez * ia;
}

__device__ __forceinline__ void mat3_mul(const float* A, const float* B, float* C) {   // C = A B
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c)
            C[r * 3 + c] = A[r * 3 + 0] * B[0 * 3 + c] + A[r * 3 + 1] * B[1 * 3 + c] + A[r * 3 + 2] * B[2 * 3 + c];
}

// mbarrier + bulk-copy (TMA) primitives shared by the tcgen05 GEMMs (bf_blend_tc.cuh) and the per-frame kernel (bf_frame.cuh)
namespace tc {
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// bounded wait: a pipeline bug must trap (-> CUDA error at the caller), never hang the GPU
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const long long t0 = clock64();
    while (!mbar_try(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) { printf("bodyfit: mbarrier wait timed out (block %d,%d thread %d)\n", blockIdx.x, blockIdx.y, threadIdx.x); __trap(); }
    }
}
// 1-D bulk copy global -> shared through the TMA unit: src / dst 16-byte aligned, bytes a multiple of 16; completion is
// signalled on `bar` as transaction bytes
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
}  // namespace tc
