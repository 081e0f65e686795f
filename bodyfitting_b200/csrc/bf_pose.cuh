// Pose kernels: one warp per frame.
//   k_pose_fwd : theta -> full_pose, Rodrigues, pose-feature row (GEMM A operand),
//                rest joints from betas, kinematic chain by tree level, A = rest-pose-removed
//                transforms, posed joints, dynamic-landmark yaw row.
//   k_pose_bwd : recompute the above in shared memory, reverse chain traversal,
//                Rodrigues backward, PCA-hand backward, GMM / angle / shape priors and the
//                Adam update, fused per frame.
// A face-parameter SMPL-X model (BfModel.face) also carries the jaw pose and the expression coefficients in theta: the forward
// takes them into the full pose / shape row, the backward produces their gradients (+ the expression L2 prior) and Adam steps them.
// Hands: n_hand parameters per hand, expanded by the [n_hand,45] component tables (the identity for axis-angle hands).
// Both kernels are instantiated for two theta capacities per frame: BF_THETA_SMEM (every row of at most 112 entries, the
// default launch shape) and BF_THETA_SMEM_WIDE (longer rows: wider hands); the launcher picks one from BfModel.NP.
// Replaces smplx batch_rodrigues + batch_rigid_transform (restated in oracle/smplx_port.py),
// smplify/prior.py:181-196, smplify/loss.py:54-61,206-217 and torch.optim.Adam
// (smplify/smplify.py:167-174,211-213).
#pragma once
#include "bf_common.cuh"
#include "bf_pack.cuh"

// fp | R | Jr | GR are contiguous and 16-byte aligned (in PoseSmemBwd), in the order of a saved forward-state row ([fp 3J |
// R 9J | Jr 3J | GR 9J], pose_write_outputs): for J == BF_MAXJ the backward fetches the row with ONE bulk copy.  No tail
// padding: PoseSmemBwd packs its scratch right behind it (see the size check there).
template <int TH>
struct PoseSmemT {
    float th[TH];
    float sh[BF_MAXNS];
    float fp[BF_MAXJ * 3];
    float R[BF_MAXJ * 9];
    float Jr[BF_MAXJ * 3];
    float GR[BF_MAXJ * 9];
    float Gt[BF_MAXJ * 3];
};
typedef PoseSmemT<BF_THETA_SMEM> PoseSmem;
typedef PoseSmemT<BF_THETA_SMEM_WIDE> PoseSmemWide;
static_assert((BF_THETA_SMEM + BF_MAXNS) % 4 == 0 && offsetof(PoseSmem, fp) % 16 == 0, "PoseSmem::fp must be 16-byte aligned");
static_assert((BF_THETA_SMEM_WIDE + BF_MAXNS) % 4 == 0 && offsetof(PoseSmemWide, fp) % 16 == 0, "PoseSmemWide::fp must be 16-byte aligned");
static_assert(BF_THETA_SMEM >= BF_MAXNP - 9 + BF_MAXNS, "PoseSmem::th must hold the longest face-parameter row with 6 hand components");
static_assert(BF_THETA_SMEM_WIDE >= BF_MAXNP - 9 + BF_MAXNS + 2 * (BF_MAXHAND - 6), "PoseSmemWide::th must hold the longest row");
// Backward scratch.  Everything else the backward needs lives in forward slots that are dead by then (smaller footprint ->
// six CTAs of four frames per SM): d(posed joints) and later d(rel) in f.Gt (the backward never reads the posed joints),
// d(full pose) in f.fp (each lane overwrites exactly the three angles it has just consumed), the updated theta in f.th, and --
// once the reverse chain traversal is done with the local rotations -- the gradient row in f.R[0:NP] and d(rest joints) in
// f.R[dJr_off:dJr_off+3J] (until then each lane keeps the d(rest joints) of its own joints in registers).
template <int TH>
struct __align__(16) PoseSmemBwdT {
    PoseSmemT<TH> f;
    float dGR[BF_MAXJ * 9];
    uint64_t bar;                 // mbarrier of the forward-state bulk copy
    static constexpr int dJr_off = TH <= 128 ? 128 : TH;   // d(rest joints) in f.R, right behind the gradient row
};
typedef PoseSmemBwdT<BF_THETA_SMEM> PoseSmemBwd;
typedef PoseSmemBwdT<BF_THETA_SMEM_WIDE> PoseSmemBwdWide;
// 13 CTAs of the default two frames fit into an SM's 228 KB (+ 1 KB per CTA): 2 * 8464 + 1024 = 17952 bytes per CTA.  The
// face-parameter theta storage (BF_THETA_SMEM) fits into what the 16-byte tail padding of PoseSmem used to take.
static_assert(sizeof(PoseSmemBwd) <= 8464, "k_pose_bwd: 13 CTAs of 2 frames per SM need <= 8464 bytes per frame");
static_assert(PoseSmemBwd::dJr_off == 128 && PoseSmemBwdWide::dJr_off + BF_MAXJ * 3 <= BF_MAXJ * 9,
              "gradient row / d(rest joints) must fit into PoseSmem::R");

// Fills S for frame b (all lanes of one warp participate).
template <int TH>
__device__ __forceinline__ void pose_forward_from_smem(const BfModel& m, PoseSmemT<TH>& S, int lane);

template <int TH>
__device__ __forceinline__ void pose_forward_warp(const BfModel& m, const float* __restrict__ theta_row,
                                                  PoseSmemT<TH>& S, int lane) {
    const int np = theta_layout(m).np;
    for (int i = lane; i < np; i += 32) S.th[i] = theta_row[i];
    __syncwarp();
    pose_forward_from_smem(m, S, lane);
}

// theta already in S.th
template <int TH>
__device__ __forceinline__ void pose_forward_from_smem(const BfModel& m, PoseSmemT<TH>& S, int lane) {
    const ThetaLayout L = theta_layout(m);
    const int J = m.J;
    // full pose
    for (int i = lane; i < 3 * J; i += 32) {
        float v = 0.f;
        if (i < 3) v = S.th[4 + i];
        else if (i < 3 + L.nbody) v = S.th[7 + (i - 3)];
        else if (m.is_smplx) {
            if (i < 69) v = m.face ? S.th[L.off_jaw + (i - 66)] : 0.f;   // jaw: 0 unless the model carries face parameters
            else if (i < 72) v = S.th[L.off_leye + (i - 69)];
            else if (i < 75) v = S.th[L.off_reye + (i - 72)];
            else if (i < 120) {
                const int c0 = i - 75;
                for (int c = 0; c < m.n_hand; ++c) v += S.th[L.off_lh + c] * __ldg(m.hand_l + c * 45 + c0);
            } else {
                const int c0 = i - 120;
                for (int c = 0; c < m.n_hand; ++c) v += S.th[L.off_rh + c] * __ldg(m.hand_r + c * 45 + c0);
            }
        }
        S.fp[i] = v + __ldg(m.pose_mean + i);
    }
    for (int l = lane; l < m.NS; l += 32) S.sh[l] = (l < m.NB) ? S.th[L.off_betas + l] : m.face ? S.th[L.off_expr + (l - m.NB)] : 0.f;
    __syncwarp();
    // rotations and rest joints
    for (int j = lane; j < J; j += 32) {
        float R[9];
        rodrigues_fwd(S.fp[3 * j], S.fp[3 * j + 1], S.fp[3 * j + 2], R);
#pragma unroll
        for (int e = 0; e < 9; ++e) S.R[j * 9 + e] = R[e];
        if (m.NB == 10 && (m.NS & 3) == 0) {          // the usual 10 betas: three vector loads per regressor row
            float sh[10];
#pragma unroll
            for (int l = 0; l < 10; ++l) sh[l] = S.sh[l];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float* jd = m.Jd + (j * 3 + c) * m.NS;
                const float4 a = __ldg(reinterpret_cast<const float4*>(jd)), q = __ldg(reinterpret_cast<const float4*>(jd) + 1);
                const float2 r = __ldg(reinterpret_cast<const float2*>(jd) + 4);
                float acc = 0.f;                       // same order as the scalar loop below
                acc += a.x * sh[0]; acc += a.y * sh[1]; acc += a.z * sh[2]; acc += a.w * sh[3];
                acc += q.x * sh[4]; acc += q.y * sh[5]; acc += q.z * sh[6]; acc += q.w * sh[7];
                acc += r.x * sh[8]; acc += r.y * sh[9];
                if (m.face)                            // expression columns after the betas, in the order of the scalar loop
                    for (int l = 10; l < m.NS; ++l) acc += __ldg(jd + l) * S.sh[l];
                S.Jr[j * 3 + c] = __ldg(m.Jt + j * 3 + c) + acc;
            }
        } else {
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                float acc = 0.f;
                const float* jd = m.Jd + (j * 3 + c) * m.NS;
                // sh[l] = 0 for l >= NB (expression) unless the model carries face parameters
                const int nl = m.face ? m.NS : m.NB;
                for (int l = 0; l < nl; ++l) acc += __ldg(jd + l) * S.sh[l];
                S.Jr[j * 3 + c] = __ldg(m.Jt + j * 3 + c) + acc;
            }
        }
    }
    __syncwarp();
    // kinematic chain, level by level (parents[j] < j, depth[parent] = depth[j] - 1)
    for (int lev = 0; lev <= m.max_depth; ++lev) {
        for (int idx = __ldg(m.lvl_ptr + lev) + lane; idx < __ldg(m.lvl_ptr + lev + 1); idx += 32) {
            const int j = __ldg(m.lvl_j + idx);
            if (lev == 0) {
#pragma unroll
                for (int e = 0; e < 9; ++e) S.GR[j * 9 + e] = S.R[j * 9 + e];
#pragma unroll
                for (int c = 0; c < 3; ++c) S.Gt[j * 3 + c] = S.Jr[j * 3 + c];
            } else {
                const int p = __ldg(m.parents + j);
                float rel[3], G[9];
#pragma unroll
                for (int c = 0; c < 3; ++c) rel[c] = S.Jr[j * 3 + c] - S.Jr[p * 3 + c];
                mat3_mul(&S.GR[p * 9], &S.R[j * 9], G);
#pragma unroll
                for (int e = 0; e < 9; ++e) S.GR[j * 9 + e] = G[e];
#pragma unroll
                for (int r = 0; r < 3; ++r)
                    S.Gt[j * 3 + r] = S.GR[p * 9 + r * 3 + 0] * rel[0] + S.GR[p * 9 + r * 3 + 1] * rel[1] +
                                      S.GR[p * 9 + r * 3 + 2] * rel[2] + S.Gt[p * 3 + r];
            }
        }
        __syncwarp();
    }
}

// forward outputs of frame b from the state in S: GEMM A operand (+ 3xTF32 split), joint transforms,
// posed joints, full pose, contour-landmark row
// mask_par: parity of the iteration that will consume these outputs (selects the block-mask buffer, BfFrames.blk_mask)
template <int TH>
__device__ __forceinline__ void pose_write_outputs(const BfModel& m, const BfFrames& f, PoseSmemT<TH>& S, int b, int lane, int mask_par) {
    const int J = m.J;
    if (f.fwd_state) {                       // [fp 3J | R 9J | Jr 3J | GR 9J] for the backward pass
        float* st = f.fwd_state + (size_t)b * 24 * J;
        for (int i = lane; i < 3 * J; i += 32) { st[i] = S.fp[i]; st[12 * J + i] = S.Jr[i]; }
        for (int i = lane; i < 9 * J; i += 32) { st[3 * J + i] = S.R[i]; st[15 * J + i] = S.GR[i]; }
    }
    // GEMM A operand row: [R_1..R_{J-1} - I | shape | 1 | 0...]
    float* pf = f.pf + (size_t)b * m.Kp;
    const bool tc_only = (f.flags & BF_F_TC) && f.pf_hi && f.pf_lo;
    for (int i = lane; i < m.Kp; i += 32) {
        float v = 0.f;
        if (i < m.P) {
            const int e = i % 9;
            v = S.R[9 + i] - ((e == 0 || e == 4 || e == 8) ? 1.0f : 0.0f);
        } else if (i < m.P + m.NS) v = S.sh[i - m.P];
        else if (i == m.P + m.NS) v = 1.0f;
        if (!tc_only) pf[i] = v;                     // the unsplit row is read by the FFMA contraction only
        if (f.pf_hi) {
            float hi, lo;
            split_tf32(v, hi, lo);
            f.pf_hi[(size_t)b * m.Kp + i] = hi;
            f.pf_lo[(size_t)b * m.Kp + i] = lo;
        }
    }
    // A_j = [GR_j | Gt_j - GR_j Jr_j],  posed joints = Gt
    for (int j = lane; j < J; j += 32) {
        float4* Aj = reinterpret_cast<float4*>(f.A + ((size_t)b * J + j) * 12);
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const float g0 = S.GR[j * 9 + r * 3], g1 = S.GR[j * 9 + r * 3 + 1], g2 = S.GR[j * 9 + r * 3 + 2];
            const float4 row = make_float4(g0, g1, g2, S.Gt[j * 3 + r] - (g0 * S.Jr[j * 3] + g1 * S.Jr[j * 3 + 1] + g2 * S.Jr[j * 3 + 2]));
            Aj[r] = row;
            f.Jtr[((size_t)b * J + j) * 3 + r] = S.Gt[j * 3 + r];
        }
    }
    if (f.full_pose)
        for (int i = lane; i < 3 * J; i += 32) f.full_pose[(size_t)b * 3 * J + i] = S.fp[i];
    // dynamic landmark row from the head yaw (smplx find_dynamic_lmk_idx_and_bcoords):
    // rel = R0 (R3 (R6 (R9 R12))), yaw = atan2(-rel[2][0], sqrt(rel00^2 + rel10^2))
    if (lane == 0 && f.yaw) {
        int row = 0;
        if (m.is_smplx) {
            float rel[9], t[9];
#pragma unroll
            for (int e = 0; e < 9; ++e) rel[e] = S.R[12 * 9 + e];
            const int chain[4] = {9, 6, 3, 0};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                mat3_mul(&S.R[chain[q] * 9], rel, t);
#pragma unroll
                for (int e = 0; e < 9; ++e) rel[e] = t[e];
            }
            const float sy = sqrtf(rel[0] * rel[0] + rel[3] * rel[3]);
            const float ang = atan2f(-rel[6], sy);
            float y = rintf(fminf((-ang * 180.0f) / 3.14159265358979323846f, 39.0f));
            int yi = (int)y;
            if (yi < 0) yi = (yi < -39) ? 78 : (39 - yi);
            row = yi;
        }
        f.yaw[b] = row;
        // the 16-vertex blocks of the active set this frame needs, OR-ed into its 128-frame tile's mask (order-independent)
        if (f.blk_mask && m.act.lv_blk)
            atomicOr(f.blk_mask + (size_t)mask_par * ((f.B + 127) >> 7) + (b >> 7), __ldg(m.act.lv_blk + (m.act.n_rows > 1 ? row : 0)));
    }
}

template <int TH>
__global__ void __launch_bounds__(128) k_pose_fwd(BfModel m, BfFrames f) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    PoseSmemT<TH>* all = reinterpret_cast<PoseSmemT<TH>*>(smem_raw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * (blockDim.x >> 5) + warp;
    if (b >= f.B) return;
    PoseSmemT<TH>& S = all[warp];
    pose_forward_warp(m, f.theta + (size_t)b * m.NP, S, lane);
    pose_write_outputs(m, f, S, b, lane, f.iter & 1);
}

// flags: 1 = priors, 2 = Adam, 4 = keep grad[0:4] written by the loss kernel (else zero them),
//        8 = after the Adam step also run the NEXT iteration's pose forward (saves a launch + a theta round trip),
//        16 = NVLink halo: the first / last frame of the shard store their updated theta row into the neighbouring
//             ranks' halo buffers and raise the flag of the next iteration's tick (bf_pack.cuh)
struct AdamArgs { float step_ts, step_lr, bc2_sqrt, beta2, om_beta1, om_beta2, eps; };

// (128, 7): at most 72 registers, so that the default launch shape (2 warps per CTA) keeps 13 CTAs per SM, the shared-memory
// bound; without the cap the face-parameter code paths let ptxas take 96 registers, which would cut it to 10
// TH: theta capacity per frame.  Up to 128 entries the Adam moments are prefetched into registers at kernel entry (4 per
// lane); the wide instantiation reads them at the step instead, so that it needs no more registers.
template <int TH>
__global__ void __launch_bounds__(128, 7) k_pose_bwd(BfModel m, BfFrames f, int flags, AdamArgs ad) {
    constexpr bool kPrefetchAdam = TH <= 128;
    constexpr int kSlots = (TH + 31) / 32;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    PoseSmemBwdT<TH>* all = reinterpret_cast<PoseSmemBwdT<TH>*>(smem_raw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * (blockDim.x >> 5) + warp;
    if (b >= f.B) return;
    PoseSmemBwdT<TH>& W = all[warp];
    PoseSmemT<TH>& S = W.f;
    float* const drel = S.Gt;
    float* const dfp = S.fp;
    const int J = m.J;
    const ThetaLayout L = theta_layout(m);
    // ---- everything this frame reads from HBM is requested up front: the saved forward state by bulk copy (TMA), the
    // loss kernel's dA / dJtr rows, the Adam moments and the GMM gradient into registers; nothing below waits on HBM again
    // (J == BF_MAXJ: the row is one contiguous block of PoseSmem; smaller skeletons take the plain loops below)
    const bool use_bulk = f.fwd_state && J == BF_MAXJ && ((uintptr_t)f.fwd_state & 15) == 0;
    if (use_bulk) {
        if (lane == 0) {
            tc::mbar_init(&W.bar, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            const float* st = f.fwd_state + (size_t)b * 24 * J;
            tc::mbar_expect_tx(&W.bar, (uint32_t)(96 * J));
            tc::bulk_g2s(S.fp, st, (uint32_t)(96 * J), &W.bar);
        }
    }
    float4 dA_r[2][3];
    float dJ_r[2][3];
#pragma unroll
    for (int s = 0; s < 2; ++s) {
        const int j = lane + 32 * s;
        if (j < J) {
            const float4* dAj = reinterpret_cast<const float4*>(f.dA + ((size_t)b * J + j) * 12);
            const float* dJj = f.dJtr + ((size_t)b * J + j) * 3;
            dA_r[s][0] = dAj[0]; dA_r[s][1] = dAj[1]; dA_r[s][2] = dAj[2];
            dJ_r[s][0] = dJj[0]; dJ_r[s][1] = dJj[1]; dJ_r[s][2] = dJj[2];
        }
    }
    float am_r[4], av_r[4], gg_r[3];
    if (kPrefetchAdam && (flags & 2)) {
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            const int i = lane + 32 * s;
            if (i < m.NP) { am_r[s] = f.adam_m[(size_t)b * m.NP + i]; av_r[s] = f.adam_v[(size_t)b * m.NP + i]; }
        }
    }
    if (flags & 1) {
#pragma unroll
        for (int s = 0; s < 3; ++s) {
            const int i = lane + 32 * s;
            gg_r[s] = i < L.nbody ? f.gmm_grad[(size_t)b * BF_GMM_D + i] : 0.f;
        }
    }
    float* const g = S.R;                    // gradient row: live from the betas phase on (S.R is dead by then)
    float* const dJr_s = S.R + PoseSmemBwdT<TH>::dJr_off;   // d(rest joints), same
    const float g_ts = (lane < 4 && (flags & 4)) ? f.grad[(size_t)b * m.NP + lane] : 0.f;     // d/d(transl, scale) from the loss kernel
    if (f.fwd_state) {                       // forward state saved by the pose forward of this iteration
        for (int i = lane; i < L.np; i += 32) S.th[i] = f.theta[(size_t)b * m.NP + i];
        if (use_bulk) {
            __syncwarp();                    // the barrier init (lane 0) is visible to the whole warp
            int spins = 0;
            while (!tc::mbar_try(&W.bar, 0)) { if (++spins > (1 << 26)) __trap(); }
        } else {
            const float* st = f.fwd_state + (size_t)b * 24 * J;
            for (int i = lane; i < 3 * J; i += 32) { S.fp[i] = st[i]; S.Jr[i] = st[12 * J + i]; }
            for (int i = lane; i < 9 * J; i += 32) { S.R[i] = st[3 * J + i]; S.GR[i] = st[15 * J + i]; }
        }
        __syncwarp();
    } else {
        pose_forward_warp(m, f.theta + (size_t)b * m.NP, S, lane);
    }

    // direct terms
    float dJr_r[2][3];
#pragma unroll
    for (int s = 0; s < 2; ++s) {
        const int j = lane + 32 * s;
        if (j >= J) break;
        const float dAj[12] = {dA_r[s][0].x, dA_r[s][0].y, dA_r[s][0].z, dA_r[s][0].w, dA_r[s][1].x, dA_r[s][1].y, dA_r[s][1].z, dA_r[s][1].w,
                               dA_r[s][2].x, dA_r[s][2].y, dA_r[s][2].z, dA_r[s][2].w};
        float dAt[3];
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            dAt[r] = dAj[r * 4 + 3];
            S.Gt[j * 3 + r] = dJ_r[s][r] + dAt[r];
#pragma unroll
            for (int c = 0; c < 3; ++c) W.dGR[j * 9 + r * 3 + c] = dAj[r * 4 + c] - dAt[r] * S.Jr[j * 3 + c];
        }
#pragma unroll
        for (int c = 0; c < 3; ++c)
            dJr_r[s][c] = -(S.GR[j * 9 + 0 * 3 + c] * dAt[0] + S.GR[j * 9 + 1 * 3 + c] * dAt[1] +
                            S.GR[j * 9 + 2 * 3 + c] * dAt[2]);
    }
    __syncwarp();
    // reverse traversal: a joint gathers from its children (one level deeper, already final)
    for (int lev = m.max_depth - 1; lev >= 0; --lev) {
        for (int idx = __ldg(m.lvl_ptr + lev) + lane; idx < __ldg(m.lvl_ptr + lev + 1); idx += 32) {
            const int j = __ldg(m.lvl_j + idx);
            const int c0 = __ldg(m.child_ptr + j), c1 = __ldg(m.child_ptr + j + 1);
            if (c0 == c1) continue;
            float aR[9], aT[3], pj[3];                 // the parent's sums stay in registers across its children
#pragma unroll
            for (int e = 0; e < 9; ++e) aR[e] = W.dGR[j * 9 + e];
#pragma unroll
            for (int c = 0; c < 3; ++c) { aT[c] = S.Gt[j * 3 + c]; pj[c] = S.Jr[j * 3 + c]; }
            for (int q = c0; q < c1; ++q) {
                const int ch = __ldg(m.child_idx + q);
                float rel[3], Rc[9];
#pragma unroll
                for (int c = 0; c < 3; ++c) rel[c] = S.Jr[ch * 3 + c] - pj[c];
#pragma unroll
                for (int e = 0; e < 9; ++e) Rc[e] = S.R[ch * 9 + e];
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    const float g0 = W.dGR[ch * 9 + r * 3], g1 = W.dGR[ch * 9 + r * 3 + 1], g2 = W.dGR[ch * 9 + r * 3 + 2];
                    const float gt = S.Gt[ch * 3 + r];
#pragma unroll
                    for (int c = 0; c < 3; ++c)   // dGR_p += dGR_c R_c^T + dGt_c (x) rel_c
                        aR[r * 3 + c] += g0 * Rc[c * 3] + g1 * Rc[c * 3 + 1] + g2 * Rc[c * 3 + 2] + gt * rel[c];
                    aT[r] += gt;
                }
            }
#pragma unroll
            for (int e = 0; e < 9; ++e) W.dGR[j * 9 + e] = aR[e];
#pragma unroll
            for (int c = 0; c < 3; ++c) S.Gt[j * 3 + c] = aT[c];
        }
        __syncwarp();
    }
    // local rotation / offset gradients
    for (int j = lane; j < J; j += 32) {
        float dR[9], dr[3];
        if (j == 0) {
#pragma unroll
            for (int e = 0; e < 9; ++e) dR[e] = W.dGR[e];
#pragma unroll
            for (int c = 0; c < 3; ++c) dr[c] = S.Gt[c];
        } else {
            const int p = __ldg(m.parents + j);
#pragma unroll
            for (int r = 0; r < 3; ++r) {
#pragma unroll
                for (int c = 0; c < 3; ++c)       // dR = GR_p^T dGR_j
                    dR[r * 3 + c] = S.GR[p * 9 + 0 * 3 + r] * W.dGR[j * 9 + 0 * 3 + c] +
                                    S.GR[p * 9 + 1 * 3 + r] * W.dGR[j * 9 + 1 * 3 + c] +
                                    S.GR[p * 9 + 2 * 3 + r] * W.dGR[j * 9 + 2 * 3 + c];
                dr[r] = S.GR[p * 9 + 0 * 3 + r] * S.Gt[j * 3 + 0] + S.GR[p * 9 + 1 * 3 + r] * S.Gt[j * 3 + 1] +
                        S.GR[p * 9 + 2 * 3 + r] * S.Gt[j * 3 + 2];
            }
            const float* dpf = f.dpf + (size_t)b * m.Kp + (j - 1) * 9;
            if (f.dpf2) {                                  // two half-reductions of the masked blend backward GEMM
                const float* dq = f.dpf2 + (size_t)b * m.Kp + (j - 1) * 9;
#pragma unroll
                for (int e = 0; e < 9; ++e) dR[e] += dpf[e] + dq[e];
            } else {
#pragma unroll
                for (int e = 0; e < 9; ++e) dR[e] += dpf[e];
            }
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) drel[j * 3 + c] = dr[c];
        float g[3];
        rodrigues_bwd(S.fp[3 * j], S.fp[3 * j + 1], S.fp[3 * j + 2], dR, g);
#pragma unroll
        for (int c = 0; c < 3; ++c) dfp[j * 3 + c] = g[c];
    }
    __syncwarp();
#pragma unroll
    for (int s = 0; s < 2; ++s) {
        const int j = lane + 32 * s;
        if (j >= J) break;
        float acc[3] = {drel[j * 3], drel[j * 3 + 1], drel[j * 3 + 2]};
        const int c0 = __ldg(m.child_ptr + j), c1 = __ldg(m.child_ptr + j + 1);
        for (int q = c0; q < c1; ++q) {
            const int ch = __ldg(m.child_idx + q);
#pragma unroll
            for (int c = 0; c < 3; ++c) acc[c] -= drel[ch * 3 + c];
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) dJr_s[j * 3 + c] = dJr_r[s][c] + acc[c];
    }
    if (lane < 4) g[lane] = g_ts;
    __syncwarp();

    // betas: rest-joint path + shape rows of the blend GEMM
    {
        // lanes (l, part): the 3J rest-joint coordinates are split into as many parts as fit into the warp -- 3 up to 10
        // betas, 2 up to 16 (the kid model), 1 above -- and combined in a fixed order.  Lane l + NB * part must stay below
        // 32: a part beyond that would wrap around the shuffles below and add another beta's partial sum.
        const int l = lane % m.NB, part = lane / m.NB;
        const int nparts = 3 * m.NB <= 32 ? 3 : 2 * m.NB <= 32 ? 2 : 1;
        const int nq = 3 * J, per = (nq + nparts - 1) / nparts;
        float acc = 0.f;
        if (part < nparts) {
            const int q1 = min(nq, (part + 1) * per);
#pragma unroll 11
            for (int q = part * per; q < q1; ++q) acc += __ldg(m.Jd + q * m.NS + l) * dJr_s[q];
        }
        const float a1s = __shfl_sync(0xffffffffu, acc, (lane + m.NB) & 31);
        const float a2s = __shfl_sync(0xffffffffu, acc, (lane + 2 * m.NB) & 31);
        const float a1 = nparts > 1 ? a1s : 0.f;
        const float a2 = nparts > 2 ? a2s : 0.f;
        if (lane < m.NB) {
            float dsh = f.dpf[(size_t)b * m.Kp + m.P + lane];
            if (f.dpf2) dsh += f.dpf2[(size_t)b * m.Kp + m.P + lane];
            g[L.off_betas + lane] = dsh + ((acc + a1) + a2);
        }
    }
    if (m.face) {
        // expression coefficients: the same rest-joint + blend-row sum as the betas above, in a lane pass of its own (so that
        // the betas' lanes and summation order do not depend on the flag); lanes (e, part), NE = NS - NB
        const int ne = m.NS - m.NB;
        if (ne > 0) {
            const int e = lane % ne, part = lane / ne;
            const int nparts = 3 * ne <= 32 ? 3 : 2 * ne <= 32 ? 2 : 1;
            const int nq = 3 * J, per = (nq + nparts - 1) / nparts;
            float acc = 0.f;
            if (part < nparts) {
                const int q1 = min(nq, (part + 1) * per);
                for (int q = part * per; q < q1; ++q) acc += __ldg(m.Jd + q * m.NS + m.NB + e) * dJr_s[q];
            }
            const float a1s = __shfl_sync(0xffffffffu, acc, (lane + ne) & 31);
            const float a2s = __shfl_sync(0xffffffffu, acc, (lane + 2 * ne) & 31);
            const float a1 = nparts > 1 ? a1s : 0.f;
            const float a2 = nparts > 2 ? a2s : 0.f;
            if (lane < ne) {
                float dsh = f.dpf[(size_t)b * m.Kp + m.P + m.NB + lane];
                if (f.dpf2) dsh += f.dpf2[(size_t)b * m.Kp + m.P + m.NB + lane];
                g[L.off_expr + lane] = dsh + ((acc + a1) + a2);
            }
        }
        if (lane < 3) g[L.off_jaw + lane] = dfp[66 + lane];                 // jaw: full-pose entries 66..68
    }
    for (int i = lane; i < 3 + L.nbody; i += 32) g[4 + i] = dfp[i];      // global_orient + body_pose
    if (m.is_smplx) {
        if (lane < 3) { g[L.off_leye + lane] = dfp[69 + lane]; g[L.off_reye + lane] = dfp[72 + lane]; }
        // hand parameters: lanes (side, component), 2 n_hand outputs (one pass for up to 16 components per hand)
        const int nh = m.n_hand;
        for (int q = lane; q < 2 * nh; q += 32) {
            const bool left = q < nh;
            const int c = left ? q : q - nh;
            const float* comp = (left ? m.hand_l : m.hand_r) + c * 45;
            const float* d = dfp + (left ? 75 : 120);
            float acc = 0.f;
#pragma unroll 15
            for (int i = 0; i < 45; ++i) acc += __ldg(comp + i) * d[i];
            g[(left ? L.off_lh : L.off_rh) + c] = acc;
        }
    }
    __syncwarp();

    float total = (flags & 4) ? f.loss[b] : 0.f;
    if (flags & 1) {
        // ---- GMM pose prior: value and gradient come from k_gmm_prior (bf_gmm.cuh) ----
#pragma unroll
        for (int s = 0; s < 3; ++s) {
            const int i = lane + 32 * s;
            if (i < L.nbody) g[7 + i] += gg_r[s];
        }
        const float pose_l = f.gmm_loss[b];
        __syncwarp();
        // ---- temporal smoothness (optional, bf_temporal_prior) ----
        float temp_l = 0.f;
        if (f.tgrad) {
            for (int i = lane; i < m.NP; i += 32) g[i] += f.tgrad[(size_t)b * m.NP + i];
            temp_l = f.tloss[b];
            __syncwarp();
        }
        // ---- angle prior: exp(sign * pose[idx])^2 on elbows / knees ----
        float ang = 0.f;
        if (lane < 4) {
            const int idx = (lane == 0) ? 52 : (lane == 1) ? 55 : (lane == 2) ? 9 : 12;
            const float sg = (lane == 0) ? 1.0f : -1.0f;
            const float e = expf(S.th[7 + idx] * sg);
            ang = e * e;
            g[7 + idx] += f.w_angle * f.w_angle * 2.0f * ang * sg;
        }
        const float angle_l = f.w_angle * f.w_angle * warp_sum(ang);
        // ---- shape prior ----
        float sq = 0.f;
        if (lane < m.NB) {
            const float be = S.th[L.off_betas + lane];
            sq = be * be;
            g[L.off_betas + lane] += f.w_shape * f.w_shape * 2.0f * be;
        }
        float shape_l = f.w_shape * f.w_shape * warp_sum(sq);
        if (m.face) {
            // expression prior w_expr^2 sum psi^2 (this project's choice; the reference optimises no expression).  It is
            // reported with the shape prior.  No jaw prior: the reference defines none, so the jaw is held by the data alone.
            float eq = 0.f;
            if (lane < m.NS - m.NB) {
                const float ps = S.th[L.off_expr + lane];
                eq = ps * ps;
                g[L.off_expr + lane] += f.w_expr * f.w_expr * 2.0f * ps;
            }
            shape_l += f.w_expr * f.w_expr * warp_sum(eq);
        }
        if (lane == 0 && f.loss_terms) {
            f.loss_terms[b * 4 + 0] = total;
            f.loss_terms[b * 4 + 1] = pose_l;
            f.loss_terms[b * 4 + 2] = angle_l;
            f.loss_terms[b * 4 + 3] = shape_l;
        }
        total += pose_l + angle_l + shape_l + temp_l;
    }
    if (lane == 0) {
        f.loss[b] = total;
        if (f.trace) f.trace[(size_t)f.iter * f.B + b] = total;
    }
    __syncwarp();
    for (int i = lane; i < m.NP; i += 32) f.grad[(size_t)b * m.NP + i] = g[i];
    if (flags & 2) {
        // torch.optim.Adam (torch 2.x single-tensor path): m.lerp_(g, 1-b1); v = v*b2 + (1-b2) g g;
        // denom = sqrt(v)/sqrt(bc2) + eps; p -= (lr/bc1) * m / denom
        float* th = f.theta + (size_t)b * m.NP;
        float* am = f.adam_m + (size_t)b * m.NP;
        float* av = f.adam_v + (size_t)b * m.NP;
#pragma unroll
        for (int s = 0; s < kSlots; ++s) {
            const int i = lane + 32 * s;
            if (i >= m.NP) break;
            const float gi = g[i];
            float mi, vi;
            if (kPrefetchAdam) { mi = am_r[s & 3]; vi = av_r[s & 3]; }    // loaded at kernel entry
            else { mi = am[i]; vi = av[i]; }
            mi = mi + (gi - mi) * ad.om_beta1;
            vi = vi * ad.beta2 + ad.om_beta2 * gi * gi;
            const float denom = sqrtf(vi) / ad.bc2_sqrt + ad.eps;
            const float step = (i < 4) ? ad.step_ts : ad.step_lr;
            const float tn = S.th[i] + (-step) * mi / denom;
            th[i] = tn;
            am[i] = mi; av[i] = vi;
            S.th[i] = tn;
        }
        if ((flags & 16) && f.halo_buf && (b == 0 || b + 1 == f.B)) {
            __syncwarp();
            const uint32_t tick = *reinterpret_cast<const uint32_t*>(f.halo_buf + BF_HALO_EPOCH) + (uint32_t)f.iter + 1u;
            const int nrow = min(m.NP, BF_HALO_ROW);      // the temporal term reads entries below 7 + nbody only
            if (b == 0 && f.halo_peer_prev) halo_push_row(S.th, nrow, f.halo_peer_prev, BF_HALO_NEXT, tick, lane);
            if (b + 1 == f.B && f.halo_peer_next) halo_push_row(S.th, nrow, f.halo_peer_next, BF_HALO_PREV, tick, lane);
        }
        if (flags & 8) {
            __syncwarp();
            pose_forward_from_smem(m, S, lane);
            pose_write_outputs(m, f, S, b, lane, (f.iter + 1) & 1);
        }
    }
}
