// Input packing of a fit (so that no torch arithmetic sits on the product path) and the NVLink halo of the temporal term.
//
//   k_pack_keypoints : detections [B,Nv,K,3] (x, y, conf) in the caller's layout -> the kernels' joint-major layout
//                      [B,K,Nv,3] (x, y, effective weight).  Body joints weigh conf^2; the reference passes hand / face
//                      confidences as [N,1], which broadcasts against the [N] residuals, so every joint of such a group
//                      weighs sum_i conf_i^2 of that group and view (smplify/loss.py:134 with :168,:173,:179).
//   k_init_theta     : network output (betas [B,10], poses [B,>=3+nbody]) -> theta rows: transl 0, scale 1, global
//                      orient / body pose / betas from the network, eyes / hands 0 (smplify/smplify.py:103-128).  A model
//                      with more than 10 betas (the kid model) starts the others at 0; one with fewer takes the first NB.
//   halo             : the temporal term couples frame f with f-1 / f+1; across shards the boundary rows live on the
//                      neighbouring GPUs.  Each rank owns one small cudaMalloc'ed buffer (exported by CUDA IPC, mapped by
//                      its neighbours); a rank WRITES its boundary theta rows straight into the neighbours' buffers over
//                      NVLink from the optimiser kernel (k_pose_bwd, right after the Adam step) and raises a flag with
//                      a system-scope release store; the consumer (k_temporal, two warps of the next iteration) spins on
//                      its local flag with acquire loads.  No host involvement per iteration -> the whole fit is one
//                      CUDA graph.  Slots are double-buffered by the parity of a global tick (= epoch base + iteration):
//                      tick T+2 can only be written after the peer has consumed tick T (it needs our tick T+1 first).
#pragma once
#include "bf_common.cuh"

#define BF_HALO_ROW 128                      // floats per boundary row slot (NP <= 111)
#define BF_HALO_PREV 0                       // [2][128] rows written by rank-1 (its LAST frame)
#define BF_HALO_NEXT (2 * BF_HALO_ROW)       // [2][128] rows written by rank+1 (its FIRST frame)
#define BF_HALO_FLAGS (4 * BF_HALO_ROW)      // uint32: flag_prev[2], flag_next[2]
#define BF_HALO_EPOCH (4 * BF_HALO_ROW + 4)  // uint32: tick of iteration 0 of the current run (local)
#define BF_HALO_FLOATS (4 * BF_HALO_ROW + 8)

__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// bounded spin (a dead peer must surface as a CUDA error, never hang the GPU): ~20 s at 2 GHz -- ranks may reach their
// first run seconds apart (model preparation on the host); in steady state the wait is a few microseconds
__device__ __forceinline__ void halo_wait(const uint32_t* flag, uint32_t tick) {
    const long long t0 = clock64();
    while ((int32_t)(ld_acquire_sys(flag) - tick) < 0) {
        if (clock64() - t0 > 40000000000LL) { printf("bodyfit: halo wait timed out (tick %u, flag %u)\n", tick, *(volatile const uint32_t*)flag); __trap(); }
        __nanosleep(64);
    }
}
// all 32 lanes: copy one theta row into a peer's slot, then publish `tick` on the peer's flag
__device__ __forceinline__ void halo_push_row(const float* row, int NP, float* peer_buf, int region, uint32_t tick, int lane) {
    float* dst = peer_buf + region + (tick & 1u) * BF_HALO_ROW;
    for (int i = lane; i < NP; i += 32) dst[i] = row[i];
    __threadfence_system();
    __syncwarp();
    if (lane == 0) {
        uint32_t* flags = reinterpret_cast<uint32_t*>(peer_buf + BF_HALO_FLAGS);
        st_release_sys(flags + (region == BF_HALO_PREV ? 0 : 2) + (tick & 1u), tick);
    }
}

// start of a run: advance the epoch by the number of iterations of the previous run and publish the initial boundary rows
// (tick = base + 0).  One CTA of 64 threads: warp 0 -> previous rank, warp 1 -> next rank.
__global__ void __launch_bounds__(64) k_halo_begin(BfFrames f, int NP, int n_iters) {
    __shared__ uint32_t base_s;
    uint32_t* epoch = reinterpret_cast<uint32_t*>(f.halo_buf + BF_HALO_EPOCH);
    if (threadIdx.x == 0) { base_s = epoch[0] + (uint32_t)n_iters; epoch[0] = base_s; }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0 && f.halo_peer_prev) halo_push_row(f.theta, NP, f.halo_peer_prev, BF_HALO_NEXT, base_s, lane);
    if (warp == 1 && f.halo_peer_next) halo_push_row(f.theta + (size_t)(f.B - 1) * NP, NP, f.halo_peer_next, BF_HALO_PREV, base_s, lane);
}

#define PK_MAXG 4
// src_index (optional): output frame b is input frame src_index[b] (frames sorted by contour row, engine.FitSession)
__global__ void __launch_bounds__(256) k_pack_keypoints(const float* __restrict__ src, float* __restrict__ dst, int B, int Nv, int K,
                                                        int hand_face, const int32_t* __restrict__ src_index) {
    extern __shared__ float pk_sm[];                      // [Nv*K*3] the frame's detections + [Nv*PK_MAXG] group weights
    const int b = blockIdx.x, n = Nv * K * 3;
    float* raw = pk_sm;
    float* gw = pk_sm + ((n + 3) & ~3);
    const float* s = src + (size_t)(src_index ? src_index[b] : b) * n;
    for (int i = threadIdx.x; i < n; i += blockDim.x) raw[i] = s[i];
    __syncthreads();
    // hand / face groups of the SMPL-X joint order (models/utils.py:74-94): [25,46) left hand, [46,67) right hand, [67,K) face
    const int g_lo[3] = {25, 46, 67}, g_hi[3] = {46, 67, K};
    if (hand_face) {
        for (int i = threadIdx.x; i < Nv * 3; i += blockDim.x) {
            const int v = i / 3, g = i % 3;
            float acc = 0.f;
            for (int k = g_lo[g]; k < g_hi[g]; ++k) { const float c = raw[(v * K + k) * 3 + 2]; acc += c * c; }
            gw[v * PK_MAXG + g] = acc;
        }
    }
    __syncthreads();
    float* d = dst + (size_t)b * n;
    for (int i = threadIdx.x; i < Nv * K; i += blockDim.x) {
        const int k = i / Nv, v = i % Nv;                 // destination order: joint-major
        const float* r = raw + (v * K + k) * 3;
        float w = r[2] * r[2];
        if (hand_face && k >= 25) w = gw[v * PK_MAXG + (k < 46 ? 0 : k < 67 ? 1 : 2)];
        d[i * 3] = r[0]; d[i * 3 + 1] = r[1]; d[i * 3 + 2] = w;
    }
}

__global__ void __launch_bounds__(256) k_init_theta(const float* __restrict__ poses, int ldp, const float* __restrict__ betas,
                                                    float* __restrict__ theta, int B, int NP, int nbody, int nbeta_in,
                                                    const int32_t* __restrict__ src_index) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)B * NP) return;
    const int c = (int)(i % NP);
    const int b = src_index ? src_index[i / NP] : (int)(i / NP);
    float v = 0.f;
    if (c == 3) v = 1.0f;                                                      // body_scale
    else if (c >= 4 && c < 7 + nbody) v = poses[(size_t)b * ldp + (c - 4)];    // global_orient | body_pose
    else if (c >= 7 + nbody && c < 7 + nbody + nbeta_in) v = betas[(size_t)b * 10 + (c - 7 - nbody)];
    theta[i] = v;
}

// dst[index[r], :] = src[r, :] (index == NULL: plain copy): results of a row-sorted batch back into the caller's frame order
__global__ void __launch_bounds__(256) k_scatter_rows(const float* __restrict__ src, const int32_t* __restrict__ index,
                                                      float* __restrict__ dst, int rows, int cols) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)rows * cols) return;
    const int r = (int)(i / cols), c = (int)(i % cols);
    dst[(size_t)(index ? index[r] : r) * cols + c] = src[i];
}
