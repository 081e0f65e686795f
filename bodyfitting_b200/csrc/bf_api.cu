// C ABI of the B200 SMPLify fitting core (see include/bodyfit_b200.h).
// Plain launchers: validate, launch on the caller's stream, report errors by return code.
#include <math.h>
#include <stdarg.h>
#include <string.h>
#include <stddef.h>
#include <stdlib.h>

#include "bf_common.cuh"
#include "bf_pose.cuh"
#include "bf_skin.cuh"
#include "bf_loss.cuh"
#include "bf_gmm.cuh"
#include "bf_frame.cuh"
#include "bf_ops.cuh"
#include "bf_grid.cuh"
#include "bf_mask.cuh"
#include "../../include/bodyfit_b200_ops.h"
#include "bf_blend_tc.cuh"
#include "bf_blend_tc2.cuh"
#include "bf_pack.cuh"
#include "bf_model_build.cuh"

static thread_local char g_err[512] = "";

void bf_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

static int check_model(const BfModel* m, const BfFrames* f) {
    BF_REQUIRE(m && f, "null model / frames");
    BF_REQUIRE(m->J > 0 && m->J <= BF_MAXJ, "J out of range");
    BF_REQUIRE(m->NS > 0 && m->NS <= BF_MAXNS && m->NB <= m->NS, "NS/NB out of range");
    BF_REQUIRE(m->face == 0 || (m->face == 1 && m->is_smplx), "face parameters apply to SMPL-X only");
    BF_REQUIRE(m->NP == theta_layout(*m).np && theta_layout(m->is_smplx, m->NB).np <= BF_MAXNP && m->NP <= BF_THETA_SMEM,
               "NP does not match theta layout");
    BF_REQUIRE(m->Kp % 16 == 0 && m->Kp >= m->P + m->NS + 1, "Kp must be a multiple of 16 covering P+NS+1");
    BF_REQUIRE(m->P == (m->J - 1) * 9, "P != 9(J-1)");
    BF_REQUIRE(m->parents && m->lvl_ptr && m->lvl_j && m->child_ptr && m->child_idx, "kinematic tree tables missing");
    BF_REQUIRE(f->B > 0, "B <= 0");
    BF_REQUIRE(f->theta, "theta is null");
    return BF_OK;
}

static int check_vset(const BfVSet* vs, const BfFrames* f) {
    BF_REQUIRE(vs->Bm && vs->ell_j && vs->ell_w, "vertex set tables missing");
    BF_REQUIRE(vs->n > 0 && vs->n_pad % 32 == 0 && vs->n_pad >= vs->n && vs->ldn == 3 * vs->n_pad, "bad vertex set padding");
    BF_REQUIRE(f->ld_v >= 3 * vs->n, "ld_v < 3n");
    BF_REQUIRE(vs->K_out <= BF_MAXK, "too many output joints");
    return BF_OK;
}

extern "C" {

int bf_abi_version(void) { return BF_ABI_VERSION; }
int bf_sizeof(int which) {
    switch (which) {
        case 0: return (int)sizeof(BfVSet);
        case 1: return (int)sizeof(BfModel);
        case 2: return (int)sizeof(BfFrames);
        case 3: return (int)sizeof(BfGrid);
        case 4: return (int)sizeof(BfSmpld);
        case 5: return (int)sizeof(BfMask);
        default: return -1;
    }
}
const char* bf_last_error(void) { return g_err; }

int bf_check_device(void) {
    int dev = 0;
    cudaDeviceProp p;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaGetDeviceProperties(&p, dev) != cudaSuccess) {
        bf_set_error("bf_check_device: no CUDA device");
        return BF_ECUDA;
    }
    if (p.major != 10) {
        bf_set_error("bf_check_device: device %s is sm_%d%d; this library is sm_100a only (no fallback)", p.name, p.major, p.minor);
        return BF_EARCH;
    }
    return BF_OK;
}

int bf_pose_forward(const BfModel* m, const BfFrames* f, void* stream) {
    BF_NVTX();
    int rc = check_model(m, f); if (rc) return rc;
    BF_REQUIRE(f->pf && f->A && f->Jtr, "pf/A/Jtr is null");
    const int wpb = 4;
    const dim3 grid((f->B + wpb - 1) / wpb), block(32 * wpb);
    k_pose_fwd<<<grid, block, wpb * sizeof(PoseSmem), (cudaStream_t)stream>>>(*m, *f);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

int bf_skin_forward(const BfModel* m, const BfFrames* f, int use_full, void* stream) {
    BF_NVTX();
    int rc = check_model(m, f); if (rc) return rc;
    const BfVSet* vs = use_full ? &m->full : &m->act;
    rc = check_vset(vs, f); if (rc) return rc;
    BF_REQUIRE(f->pf && f->A && f->verts, "pf/A/verts is null");
    if (bf_tc_ready_fwd(vs, f)) {
        // tensor cores blend (v_posed), then the row kernel skins with the joint transforms resident in shared memory;
        // without a v_posed buffer (inference) the blend goes to f->verts and is skinned in place
        float* vp = f->vposed ? f->vposed : f->verts;
        rc = bf_blend_forward_tc(m, vs, f, vp, (cudaStream_t)stream); if (rc) return rc;
        rc = bf_launch_skin_frame(0, m, vs, f, vp, f->verts, nullptr, nullptr, 0, (f->flags & BF_F_WORLD) ? 1 : 0, 0, (cudaStream_t)stream);
        if (rc != 1) return rc;
        return bf_launch_skin_rows(0, vs, m->J, f->A, vp, f->verts, nullptr, nullptr, f->B, f->ld_v, 0,
                                   (f->flags & BF_F_WORLD) ? f->theta : nullptr, m->NP, f->constant_scale, (cudaStream_t)stream);
    }
    const dim3 grid(vs->n_pad / SK_TV, (f->B + SK_TB - 1) / SK_TB), block(256);
    k_skin_fwd<<<grid, block, 0, (cudaStream_t)stream>>>(*vs, m->J, m->Kp, f->pf, f->A, f->verts, f->vposed, f->B, f->ld_v,
                                                           (f->flags & BF_F_WORLD) ? f->theta : nullptr, m->NP, f->constant_scale);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

int bf_blend_forward(const BfModel* m, const BfFrames* f, int use_full, void* stream) {
    BF_NVTX();
    int rc = check_model(m, f); if (rc) return rc;
    const BfVSet* vs = use_full ? &m->full : &m->act;
    rc = check_vset(vs, f); if (rc) return rc;
    BF_REQUIRE(f->vposed, "vposed is null");
    BF_REQUIRE((f->flags & BF_F_TC) && vs->Bt_hi && vs->Bt_lo && f->pf_hi && f->pf_lo, "bf_blend_forward needs the tensor-core operands (BF_F_TC)");
    return bf_blend_forward_tc(m, vs, f, f->vposed, (cudaStream_t)stream);
}

int bf_joints_forward(const BfModel* m, const BfFrames* f, int use_full, void* stream) {
    BF_NVTX();
    int rc = check_model(m, f); if (rc) return rc;
    const BfVSet* vs = use_full ? &m->full : &m->act;
    rc = check_vset(vs, f); if (rc) return rc;
    BF_REQUIRE(f->joints && f->Jtr && f->verts, "joints/Jtr/verts is null");
    k_joints_fwd<<<f->B, 160, 0, (cudaStream_t)stream>>>(*m, *vs, *f);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

int bf_joints_backward(const BfModel* m, const BfFrames* f, int use_full, int accumulate_dverts, void* stream) {
    BF_NVTX();
    int rc = check_model(m, f); if (rc) return rc;
    const BfVSet* vs = use_full ? &m->full : &m->act;
    rc = check_vset(vs, f); if (rc) return rc;
    BF_REQUIRE(f->dJtr && f->dverts, "dJtr/dverts is null");
    k_joints_bwd<<<f->B, 256, 0, (cudaStream_t)stream>>>(*m, *vs, *f, accumulate_dverts);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

int bf_keypoint_loss(const BfModel* m, const BfFrames* f, int use_full, void* stream) {
    BF_NVTX();
    int rc = check_model(m, f); if (rc) return rc;
    const BfVSet* vs = use_full ? &m->full : &m->act;
    rc = check_vset(vs, f); if (rc) return rc;
    BF_REQUIRE(f->kp && f->cams && f->loss && f->grad && f->dJtr && f->dverts && f->verts && f->Jtr, "loss buffers missing");
    BF_REQUIRE(f->Nv > 0 && f->Nv <= BF_MAXVIEWS, "Nv out of range");
    BF_REQUIRE(m->K_used <= vs->K_out, "K_used > K_out");
    const int threads = use_full ? 256 : 160;
    k_keypoint_loss<<<f->B, threads, 0, (cudaStream_t)stream>>>(*m, *vs, *f);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

// Side streams (+ fork / join events) per (device, caller stream, slot), created on first use.
//   slot 0: the GMM prior of a fit iteration only needs theta, so it runs next to the blend / loss kernels (fork after the
//           parameters are final, join before the pose backward);
//   slot 1: in the all-vertex backward, dA (gathers per joint, no shared memory) runs next to dvp (row kernel) -- both
//           only read d(verts).
struct SideStream { cudaStream_t main = nullptr; cudaStream_t s = nullptr; cudaEvent_t fork = nullptr, join = nullptr; int dev = -1, slot = 0; };
static SideStream* side_stream(cudaStream_t main_s, int slot = 0) {
    static SideStream table[512];
    static int used = 0;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
    std::lock_guard<std::mutex> lk(g_bf_mu);
    for (int i = 0; i < used; ++i)
        if (table[i].dev == dev && table[i].main == main_s && table[i].slot == slot) return &table[i];
    if (used >= 512) return nullptr;
    SideStream* ss = &table[used];
    if (cudaStreamCreateWithFlags(&ss->s, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&ss->fork, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&ss->join, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    ss->dev = dev; ss->main = main_s; ss->slot = slot;
    ++used;
    return ss;
}

// parts: bit0 dvp, bit1 dA, bit2 blend backward GEMM (bf_skin_backward = all three)
int bf_skin_backward_parts(const BfModel* m, const BfFrames* f, int use_full, int parts, void* stream) {
    BF_NVTX();
    int rc = check_model(m, f); if (rc) return rc;
    const BfVSet* vs = use_full ? &m->full : &m->act;
    rc = check_vset(vs, f); if (rc) return rc;
    BF_REQUIRE(f->dverts && f->dvp && f->vposed && f->dA && f->dpf && f->A, "backward buffers missing");
    BF_REQUIRE(vs->jv_ptr && vs->jv_vid && vs->jv_w, "joint->vertex lists missing");
    cudaStream_t s = (cudaStream_t)stream;
    SideStream* s2 = ((parts & 3) == 3) ? side_stream(s, 1) : nullptr;
    if (s2) {                                              // dA next to dvp: both only read d(verts)
        cudaEventRecord(s2->fork, s);
        cudaStreamWaitEvent(s2->s, s2->fork, 0);
        k_skin_bwd_dA<<<f->B, 256, 0, s2->s>>>(*vs, m->J, f->dverts, f->vposed, f->dA, f->B, f->ld_v);
        BF_LAUNCH_CHECK();
        cudaEventRecord(s2->join, s2->s);
    }
    if ((parts & 1) && bf_tc_ready_bwd(vs, f)) {
        // tensor-core mode: only the 3xTF32 split of dvp is consumed (by the blend backward GEMM)
        rc = bf_launch_skin_frame(1, m, vs, f, f->dverts, nullptr, f->dvp_hi, f->dvp_lo, vs->ldn, 0, 0, s);
        if (rc == 1)
            rc = bf_launch_skin_rows(1, vs, m->J, f->A, f->dverts, nullptr, f->dvp_hi, f->dvp_lo, f->B, f->ld_v, vs->ldn,
                                     nullptr, m->NP, 0.f, s);
        if (rc) return rc;
    } else if (parts & 1) {
        const dim3 grid((vs->n + 255) / 256, (f->B + DV_FB - 1) / DV_FB);
        const bool tcb = false;
        k_skin_bwd_dvp<<<grid, 256, 0, s>>>(*vs, m->J, f->A, f->dverts, f->dvp, f->B, f->ld_v,
                                           tcb ? f->dvp_hi : nullptr, tcb ? f->dvp_lo : nullptr);
        BF_LAUNCH_CHECK();
    }
    if ((parts & 2) && !s2) {
        k_skin_bwd_dA<<<f->B, 256, 0, s>>>(*vs, m->J, f->dverts, f->vposed, f->dA, f->B, f->ld_v);
        BF_LAUNCH_CHECK();
    }
    int tc_rc = 1;
    if ((parts & 4) && bf_tc_ready_bwd(vs, f)) {
        tc_rc = bf_blend_backward_tc(m, vs, f, s);
        if (tc_rc < 0) return tc_rc;
    }
    if ((parts & 4) && tc_rc == 1) {                       // FP32 FFMA contraction (no tensor cores / no workspace)
        const dim3 grid((m->Kp + GB_T - 1) / GB_T, (f->B + GB_T - 1) / GB_T);
        k_blend_bwd<<<grid, 256, 0, s>>>(*vs, m->Kp, f->dvp, f->dpf, f->B, f->ld_v);
        BF_LAUNCH_CHECK();
    }
    if (s2) cudaStreamWaitEvent(s, s2->join, 0);
    return BF_OK;
}

int bf_skin_backward(const BfModel* m, const BfFrames* f, int use_full, void* stream) {
    return bf_skin_backward_parts(m, f, use_full, 7, stream);
}

static int launch_gmm(const BfModel* m, const float* pose, int ld, int nvalid, int B, float wp, float* grad, float* loss,
                      cudaStream_t s) {
    BF_REQUIRE(m->gmm_mean && m->gmm_psym && m->gmm_logw && m->n_gmm > 0, "GMM tables missing");
    BF_REQUIRE(pose && grad && loss && B > 0, "gmm buffers missing");
    static size_t attr[BF_MAXDEV] = {0};
    { const int rc = bf_ensure_smem(k_gmm_prior, sizeof(GmmSmem), attr, "k_gmm_prior"); if (rc) return rc; }
    k_gmm_prior<<<(B + GM_F - 1) / GM_F, GM_F * GM_PARTS, sizeof(GmmSmem), s>>>(*m, pose, ld, nvalid, B, wp, grad, loss);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

// temporal smoothness: one warp per frame.  The shard's outer neighbours come either from halo_prev / halo_next (rows the
// host exchanged before the launch) or, with the NVLink halo (f.halo_buf, bf_pack.cuh), from the local slots the neighbouring
// ranks' optimiser kernels wrote: the two boundary warps wait for the tick of this iteration.
__global__ void __launch_bounds__(128) k_temporal(BfModel m, BfFrames f) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * 4 + warp;
    if (b >= f.B) return;
    const int nb = theta_layout(m.is_smplx).nbody;
    const float* cur = f.theta + (size_t)b * m.NP;
    const float* prev = b > 0 ? cur - m.NP : f.halo_prev;
    const float* next = b + 1 < f.B ? cur + m.NP : f.halo_next;
    if (f.halo_buf && (b == 0 || b + 1 == f.B)) {
        const uint32_t tick = *reinterpret_cast<const uint32_t*>(f.halo_buf + BF_HALO_EPOCH) + (uint32_t)f.iter;
        const uint32_t* flags = reinterpret_cast<const uint32_t*>(f.halo_buf + BF_HALO_FLAGS);
        if (b == 0 && f.halo_peer_prev) {
            halo_wait(flags + (tick & 1u), tick);
            prev = f.halo_buf + BF_HALO_PREV + (tick & 1u) * BF_HALO_ROW;
        }
        if (b + 1 == f.B && f.halo_peer_next) {
            halo_wait(flags + 2 + (tick & 1u), tick);
            next = f.halo_buf + BF_HALO_NEXT + (tick & 1u) * BF_HALO_ROW;
        }
    }
    const float w = f.w_temporal;
    float acc = 0.f;
    for (int i = lane; i < m.NP; i += 32) {
        const bool used = i < 3 || (i >= 4 && i < 7 + nb);           // transl, global_orient, body_pose
        float g = 0.f;
        if (used) {
            const float x = cur[i];
            if (prev) { const float d = x - __ldcv(prev + i); acc += d * d; g += 2.0f * w * d; }
            if (next) g += 2.0f * w * (x - __ldcv(next + i));
        }
        f.tgrad[(size_t)b * m.NP + i] = g;
    }
    acc = warp_sum(acc);
    if (lane == 0) f.tloss[b] = w * acc;
}

int bf_temporal_prior(const BfModel* m, const BfFrames* f, void* stream) {
    BF_NVTX();
    int rc = check_model(m, f); if (rc) return rc;
    BF_REQUIRE(f->tgrad && f->tloss, "tgrad / tloss is null");
    k_temporal<<<(f->B + 3) / 4, 128, 0, (cudaStream_t)stream>>>(*m, *f);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

int bf_gmm_prior(const BfModel* m, const BfFrames* f, void* stream) {
    BF_NVTX();
    int rc = check_model(m, f); if (rc) return rc;
    BF_REQUIRE(f->gmm_grad && f->gmm_loss, "gmm_grad / gmm_loss is null");
    if ((f->flags & BF_F_TC) && m->gmm_bt_hi && m->gmm_bt_lo && f->gmm_ws && (m->n_gmm * GM_LD) % TC_BN1 == 0 && GM_KG % TC_BK == 0) {
        // tensor-core form: pack [pose | 1] -> one 3xTF32 GEMM against [P_sym,m | -P_sym,m mu_m] -> per-frame select
        BF_REQUIRE(m->gmm_mean && m->gmm_logw && m->n_gmm > 0, "GMM tables missing");
        cudaStream_t s = (cudaStream_t)stream;
        const int ny = m->n_gmm * GM_LD, nb = theta_layout(m->is_smplx).nbody;
        float* Y = f->gmm_ws;
        float* x_hi = f->gmm_ws + (size_t)f->B * ny;
        float* x_lo = x_hi + (size_t)f->B * GM_KG;
        const float wp = f->w_pose * f->w_pose;
        k_gmm_pack<<<(unsigned)(((size_t)f->B * GM_KG + 255) / 256), 256, 0, s>>>(f->theta + 7, m->NP, nb, f->B, x_hi, x_lo);
        BF_LAUNCH_CHECK();
        rc = bf_gemm_forward_tc(x_hi, x_lo, m->gmm_bt_hi, m->gmm_bt_lo, f->B, GM_KG, ny, ny / 3, Y, ny, s); if (rc) return rc;
        k_gmm_select<<<(f->B + 3) / 4, 128, 0, s>>>(*m, f->theta + 7, m->NP, nb, f->B, Y, ny, wp, f->gmm_grad, f->gmm_loss);
        BF_LAUNCH_CHECK();
        return BF_OK;
    }
    return launch_gmm(m, f->theta + 7, m->NP, theta_layout(m->is_smplx).nbody, f->B, f->w_pose * f->w_pose,
                      f->gmm_grad, f->gmm_loss, (cudaStream_t)stream);
}

// ---- stand-alone loss / prior operators (include/bodyfit_b200_ops.h) ------------------------------
int bf_op_project(const float* pts, const float* R, const float* t, const float* K, float* uv, int B, int N, int nb, void* stream) {
    BF_REQUIRE(pts && R && t && K && uv && B > 0 && N > 0 && (nb == 1 || nb == B), "bad arguments");
    k_project_fwd<<<(B * N + 255) / 256, 256, 0, (cudaStream_t)stream>>>(pts, R, t, K, uv, B, N, nb);
    BF_LAUNCH_CHECK();
    return BF_OK;
}
int bf_op_project_backward(const float* pts, const float* R, const float* t, const float* K, const float* duv, float* dpts,
                           int B, int N, int nb, void* stream) {
    BF_REQUIRE(pts && R && t && K && duv && dpts && B > 0 && N > 0 && (nb == 1 || nb == B), "bad arguments");
    k_project_bwd<<<(B * N + 255) / 256, 256, 0, (cudaStream_t)stream>>>(pts, R, t, K, duv, dpts, B, N, nb);
    BF_LAUNCH_CHECK();
    return BF_OK;
}
int bf_op_gmof(const float* x, float* y, float sigma, int64_t n, void* stream) {
    BF_REQUIRE(x && y && n > 0, "bad arguments");
    k_gmof_fwd<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, y, sigma, (size_t)n);
    BF_LAUNCH_CHECK();
    return BF_OK;
}
int bf_op_gmof_backward(const float* x, const float* dy, float* dx, float sigma, int64_t n, void* stream) {
    BF_REQUIRE(x && dy && dx && n > 0, "bad arguments");
    k_gmof_bwd<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, dy, dx, sigma, (size_t)n);
    BF_LAUNCH_CHECK();
    return BF_OK;
}
int bf_op_reprojection(const float* cord, const float* gt, const float* w, float coef, float sigma, int N, float* out,
                       float* dcord, void* stream) {
    BF_REQUIRE(cord && gt && w && out && dcord && N > 0, "bad arguments");
    k_reproj<<<1, 256, 0, (cudaStream_t)stream>>>(cord, gt, w, coef, sigma, N, out, dcord);
    BF_LAUNCH_CHECK();
    return BF_OK;
}
int bf_op_keypoints_world(const float* joints, const float* kp, const float* cams, int B, int K, int Nv, float coef,
                          float sigma, float* loss_bk, float* dJ, void* stream) {
    BF_REQUIRE(joints && kp && cams && loss_bk && dJ && B > 0 && K > 0 && Nv > 0, "bad arguments");
    k_kp_world<<<(B * K + 127) / 128, 128, 0, (cudaStream_t)stream>>>(joints, kp, cams, B, K, Nv, coef, sigma, loss_bk, dJ);
    BF_LAUNCH_CHECK();
    return BF_OK;
}
int bf_op_angle_prior(const float* pose, int B, int D, float* out, float* dout, void* stream) {
    BF_REQUIRE(pose && out && dout && B > 0 && D >= 56, "bad arguments (pose needs >= 56 columns)");
    k_angle_prior<<<(B * 4 + 127) / 128, 128, 0, (cudaStream_t)stream>>>(pose, B, D, out, dout);
    BF_LAUNCH_CHECK();
    return BF_OK;
}
int bf_op_gmm_pose(const BfModel* m, const float* pose, int ld, int nvalid, int B, float weight, float* grad, float* loss,
                   void* stream) {
    BF_REQUIRE(m && nvalid > 0 && nvalid <= 69 && ld >= nvalid, "bad arguments");
    return launch_gmm(m, pose, ld, nvalid, B, weight, grad, loss, (cudaStream_t)stream);
}

int bf_pose_backward(const BfModel* m, const BfFrames* f, int flags, void* stream) {
    BF_NVTX();
    int rc = check_model(m, f); if (rc) return rc;
    BF_REQUIRE(f->dA && f->dJtr && f->dpf && f->grad && f->loss, "pose backward buffers missing");
    if (flags & 1) BF_REQUIRE(f->gmm_grad && f->gmm_loss, "gmm_grad / gmm_loss missing (run bf_gmm_prior first)");
    if (flags & 8) BF_REQUIRE((flags & 2) && f->pf && f->A && f->Jtr, "flag 8 needs the Adam step and the forward buffers");
    if (flags & 2) BF_REQUIRE(f->adam_m && f->adam_v, "Adam state missing");
    // bias corrections in double on the host, exactly as torch.optim.Adam does for python-float steps
    const double t = (double)(f->iter + 1);
    const double bc1 = 1.0 - pow(f->beta1, t);
    const double bc2 = 1.0 - pow(f->beta2, t);
    AdamArgs ad;
    ad.step_ts = (float)(f->lr_ts / bc1);
    ad.step_lr = (float)(f->lr / bc1);
    ad.bc2_sqrt = (float)sqrt(bc2);
    ad.beta2 = (float)f->beta2;
    ad.om_beta1 = (float)(1.0 - f->beta1);
    ad.om_beta2 = (float)(1.0 - f->beta2);
    ad.eps = (float)f->eps;
    // frames (warps) per CTA: shared memory bounds the residency (8.4 KB per frame + 1 KB per CTA): 4 -> 24, 2 -> 26 warps / SM
    static int wpb = 0;
    if (!wpb) { const char* e = getenv("BODYFIT_POSE_WPB"); wpb = e ? atoi(e) : 2; if (wpb < 1 || wpb > 4) wpb = 2; }
    const dim3 grid((f->B + wpb - 1) / wpb), block(32 * wpb);
    BfFrames g = *f;
    if (!bf_bwd_two_cta(m, f)) g.dpf2 = nullptr;         // the backward GEMM added its two half-reductions itself
    k_pose_bwd<<<grid, block, wpb * sizeof(PoseSmemBwd), (cudaStream_t)stream>>>(*m, g, flags, ad);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

int bf_lbs_forward(const BfModel* m, const BfFrames* f, void* stream) {
    BF_NVTX();
    int rc = bf_pose_forward(m, f, stream); if (rc) return rc;
    const BfVSet* vs = &m->full;
    if (f->joints && bf_tc_ready_fwd(vs, f) && f->verts && f->Jtr) {
        // blend GEMM, then ONE per-frame kernel: skinning (+ world transform) and the output joints of the frame
        rc = check_vset(vs, f); if (rc) return rc;
        float* vp = f->vposed ? f->vposed : f->verts;
        rc = bf_blend_forward_tc(m, vs, f, vp, (cudaStream_t)stream); if (rc) return rc;
        rc = bf_launch_skin_frame(0, m, vs, f, vp, f->verts, nullptr, nullptr, 0, (f->flags & BF_F_WORLD) ? 1 : 0, 1, (cudaStream_t)stream);
        if (rc == 2) return BF_OK;                         // joints done
        if (rc == BF_OK) return bf_joints_forward(m, f, 1, stream);
        if (rc != 1) return rc;
        rc = bf_launch_skin_rows(0, vs, m->J, f->A, vp, f->verts, nullptr, nullptr, f->B, f->ld_v, 0,
                                 (f->flags & BF_F_WORLD) ? f->theta : nullptr, m->NP, f->constant_scale, (cudaStream_t)stream);
        if (rc) return rc;
        return bf_joints_forward(m, f, 1, stream);
    }
    rc = bf_skin_forward(m, f, 1, stream); if (rc) return rc;
    if (f->joints) rc = bf_joints_forward(m, f, 1, stream);
    return rc;
}

int bf_lbs_backward(const BfModel* m, const BfFrames* f, void* stream) {
    BF_NVTX();
    // f->dverts holds the incoming d(vertices) (dense); f->djoints the incoming d(joints) or NULL
    int rc = bf_joints_backward(m, f, 1, 1, stream); if (rc) return rc;
    rc = bf_skin_backward(m, f, 1, stream); if (rc) return rc;
    return bf_pose_backward(m, f, 0, stream);
}

// shared memory of k_frame_loss_bwd: joint gradients + positions, cameras, reduction scratch, the frame's transforms,
// skinned vertices / d(verts), v_posed, and the live vertices' outer products
static size_t bf_frame_smem(const BfModel* m, const BfVSet* vs, int Nv, int tma) {
    return sizeof(float) * (size_t)frame_smem_layout(m->K_used, Nv, m->J, vs->ldn, vs->lmax, tma).total;
}
// The bulk-copy (TMA) staging of the per-frame kernel needs 16-byte aligned, 16-byte granular keypoint rows and room for
// them in shared memory; otherwise the plain-load variant runs.  BODYFIT_FRAME_TMA=0 forces the latter (A/B timing).
static bool bf_frame_use_tma(const BfModel* m, const BfVSet* vs, const BfFrames* f) {
    static int env = -1;
    if (env < 0) { const char* e = getenv("BODYFIT_FRAME_TMA"); env = e ? atoi(e) : 1; }
    return env != 0 && (m->K_used * f->Nv) % 4 == 0 && ((uintptr_t)f->kp & 15) == 0 && ((uintptr_t)f->A & 15) == 0 &&
           ((uintptr_t)f->vposed & 15) == 0 && bf_frame_smem(m, vs, f->Nv, 1) <= 48 * 1024;
}

int bf_frame_loss_backward(const BfModel* m, const BfFrames* f, void* stream) {
    BF_NVTX();
    int rc = check_model(m, f); if (rc) return rc;
    const BfVSet* vs = &m->act;
    rc = check_vset(vs, f); if (rc) return rc;
    const int skin_here = (f->flags & BF_F_SKIN_FUSED) ? 1 : 0;
    BF_REQUIRE(f->kp && f->cams && f->loss && f->grad && f->dJtr && (skin_here || f->verts) && f->vposed && f->Jtr && f->A && f->dA,
               "fused loss/backward buffers missing");
    BF_REQUIRE(vs->lv_n && vs->lv_vid && vs->lt_ptr && vs->lt_k && vs->lt_w && vs->lj_ptr && vs->lj_vid && vs->lj_w && vs->lmax > 0 &&
               vs->n_rows > 0, "live-vertex lists of the active set missing");
    BF_REQUIRE(f->ld_v % 4 == 0 && vs->ldn % 4 == 0, "ld_v / ldn must be multiples of 4 floats");
    BF_REQUIRE(f->dvp_hi || f->dvp, "dvp (or its 3xTF32 split) missing");
    BF_REQUIRE(f->Nv > 0 && f->Nv <= BF_MAXVIEWS, "Nv out of range");
    BF_REQUIRE(vs->jv_ptr && vs->jv_vid && vs->jv_w && vs->jv_nz, "joint->vertex lists missing");
    const bool tma = bf_frame_use_tma(m, vs, f);
    const size_t smem = bf_frame_smem(m, vs, f->Nv, tma);
    BF_REQUIRE(smem <= 48 * 1024, "active vertex set too large for the fused per-frame kernel");
    BfFrames g = *f;
    if (!bf_tc_ready_bwd(vs, f)) { g.dvp_hi = nullptr; g.dvp_lo = nullptr; }
    // Launch shape (bf_frame.cuh): eight resident frames of 160 threads win once the batch covers their 8 x SMs slots about twice
    // (10,000 frames: 189 -> 181 us); a 1,250-frame shard is ONE wave of the 224-thread shape's slots plus a half, but one wave of
    // the 160-thread shape plus 66 frames (37.8 vs 32.0 us), so small batches keep 224 x 5.  Both shapes run the same per-frame
    // arithmetic in the same order (bit-identical; tests/test_gpu_parity.py::test_full_size_batch_properties crosses them).
    static int nt_env = -1;
    if (nt_env < 0) { const char* e = getenv("BODYFIT_FRAME_THREADS"); const int v = e ? atoi(e) : 0; nt_env = (v == 256 || v == 224 || v == 160) ? v : 0; }
    const int nt = nt_env ? nt_env : (f->B >= 2048 ? 160 : 224);
    const cudaStream_t s_ = (cudaStream_t)stream;
    if (tma && nt == 160) {
        // keypoints from global memory: 27 KB of shared memory per frame; the full carve-out makes room for eight CTAs per SM
        const size_t smem2 = bf_frame_smem(m, vs, f->Nv, 2);
        static bool carve[BF_MAXDEV] = {false};
        const int dev = bf_cur_dev();
        {
            std::lock_guard<std::mutex> lk(g_bf_mu);
            if (!carve[dev]) {
                cudaFuncSetAttribute(k_frame_loss_bwd<2, 160>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
                cudaGetLastError();
                carve[dev] = true;
            }
        }
        k_frame_loss_bwd<2, 160><<<f->B, 160, smem2, s_>>>(*m, *vs, g, skin_here);
    } else if (tma) {
        if (nt == 256) k_frame_loss_bwd<1, 256><<<f->B, 256, smem, s_>>>(*m, *vs, g, skin_here);
        else k_frame_loss_bwd<1, 224><<<f->B, 224, smem, s_>>>(*m, *vs, g, skin_here);
    } else {
        if (nt == 256) k_frame_loss_bwd<0, 256><<<f->B, 256, smem, s_>>>(*m, *vs, g, skin_here);
        else k_frame_loss_bwd<0, 224><<<f->B, 224, smem, s_>>>(*m, *vs, g, skin_here);
    }
    BF_LAUNCH_CHECK();
    return BF_OK;
}

static int fit_iteration(const BfModel* m, const BfFrames* f, bool with_forward, bool fuse_next, void* stream) {
    int rc;
    cudaStream_t main_s = (cudaStream_t)stream;
    SideStream* ss = side_stream(main_s);
    if (ss) {                                                     // theta of this iteration is final here
        cudaEventRecord(ss->fork, main_s);
        cudaStreamWaitEvent(ss->s, ss->fork, 0);
        rc = bf_gmm_prior(m, f, ss->s); if (rc) return rc;
        cudaEventRecord(ss->join, ss->s);
    }
    if (f->tgrad && f->w_temporal > 0.f) { rc = bf_temporal_prior(m, f, stream); if (rc) return rc; }
    if (with_forward) { rc = bf_pose_forward(m, f, stream); if (rc) return rc; }
    const size_t fused_smem = bf_frame_smem(m, &m->act, f->Nv, 0);
    const bool fused = fused_smem <= 48 * 1024 && m->act.lv_n;
    // tensor-core path of the fused loop: the GEMM only blends (v_posed); the per-frame kernel skins its live vertices
    const bool blend_only = fused && bf_tc_ready_fwd(&m->act, f) && f->vposed && !(f->flags & BF_F_WORLD);
    if (blend_only) { rc = bf_blend_forward(m, f, 0, stream); if (rc) return rc; }
    else { rc = bf_skin_forward(m, f, 0, stream); if (rc) return rc; }
    if (fused) {
        BfFrames g = *f;
        if (blend_only) g.flags |= BF_F_SKIN_FUSED;
        rc = bf_frame_loss_backward(m, &g, stream); if (rc) return rc;          // skin + loss + dverts (on chip) + dvp + dA
        if (!ss) { rc = bf_gmm_prior(m, f, stream); if (rc) return rc; }
        rc = bf_skin_backward_parts(m, f, 0, 4, stream); if (rc) return rc;    // dpf = dvp @ Bm^T
    } else {
        rc = bf_keypoint_loss(m, f, 0, stream); if (rc) return rc;
        if (!ss) { rc = bf_gmm_prior(m, f, stream); if (rc) return rc; }
        rc = bf_skin_backward(m, f, 0, stream); if (rc) return rc;
    }
    if (ss) cudaStreamWaitEvent(main_s, ss->join, 0);
    const int push = (f->halo_buf && f->tgrad && f->w_temporal > 0.f && f->iter + 1 < f->halo_iters) ? 16 : 0;
    return bf_pose_backward(m, f, 1 | 2 | 4 | (fuse_next ? 8 : 0) | push, stream);
}

int bf_fit_step(const BfModel* m, const BfFrames* f, void* stream) {
    BF_NVTX();
    return fit_iteration(m, f, true, false, stream);
}

int bf_fit_iteration(const BfModel* m, const BfFrames* f, int with_forward, int fuse_next, void* stream) {
    BF_NVTX();
    BF_REQUIRE(m && f, "bad arguments");
    return fit_iteration(m, f, with_forward != 0, fuse_next != 0, stream);
}

int bf_fit_run(const BfModel* m, const BfFrames* f, int n_iters, void* stream) {
    BF_NVTX();
    BF_REQUIRE(m && f && n_iters >= 0, "bad arguments");
    BfFrames g = *f;
    for (int i = 0; i < n_iters; ++i) {
        // the pose-backward kernel of iteration i also runs the pose forward of iteration i+1
        int rc = fit_iteration(m, &g, i == 0, i + 1 < n_iters, stream); if (rc) return rc;
        g.iter++;
    }
    return BF_OK;
}

// ---- model / frame-buffer construction for hosts that do not run Python ---------------------------------------------
// A model blob is written once by bodyfitting_b200.model.PreparedModel.save_blob (the table building stays in one place);
// loading = one file read, one cudaMalloc, one upload, pointer patching.
struct BfModelOwned { BfModel m; void* dev; uint64_t magic; };
#define BF_OWNED_MAGIC 0xB200F17B200F17ULL

static void patch_ptrs(void** fields, int n, char* dev_base, int64_t total, int* bad) {
    for (int i = 0; i < n; ++i) {
        const uintptr_t v = (uintptr_t)fields[i];
        if (v == 0) continue;
        if ((int64_t)(v - 1) >= total) { *bad = 1; fields[i] = nullptr; continue; }
        fields[i] = dev_base + (v - 1);
    }
}

int bf_model_load_memory(const void* blob, int64_t nbytes, BfModel** out) {
    BF_REQUIRE(blob && out && nbytes > 16 + (int64_t)sizeof(BfModel) + 8, "blob too small");
    const char* p = (const char*)blob;
    BF_REQUIRE(memcmp(p, "BFMODEL1", 8) == 0, "not a bodyfit model blob");
    int32_t abi, sz;
    memcpy(&abi, p + 8, 4); memcpy(&sz, p + 12, 4);
    BF_REQUIRE(abi == BF_ABI_VERSION && sz == (int32_t)sizeof(BfModel), "model blob was written for another ABI version");
    int64_t total;
    memcpy(&total, p + 16 + sizeof(BfModel), 8);
    BF_REQUIRE(total >= 0 && 16 + (int64_t)sizeof(BfModel) + 8 + total <= nbytes, "truncated model blob");
    BfModelOwned* o = (BfModelOwned*)calloc(1, sizeof(BfModelOwned));
    BF_REQUIRE(o, "out of host memory");
    memcpy(&o->m, p + 16, sizeof(BfModel));
    if (cudaMalloc(&o->dev, (size_t)(total > 0 ? total : 16)) != cudaSuccess) { free(o); bf_set_error("bf_model_load: cudaMalloc(%lld) failed", (long long)total); return BF_ECUDA; }
    if (cudaMemcpy(o->dev, p + 16 + sizeof(BfModel) + 8, (size_t)total, cudaMemcpyHostToDevice) != cudaSuccess) {
        cudaFree(o->dev); free(o); bf_set_error("bf_model_load: upload failed"); return BF_ECUDA;
    }
    int bad = 0;
    // pointer fields: the leading block of BfModel, and of each BfVSet (layout checked against the header by static_assert)
    patch_ptrs((void**)&o->m, (int)(offsetof(BfModel, full) / sizeof(void*)), (char*)o->dev, total, &bad);
    patch_ptrs((void**)&o->m.full, (int)(offsetof(BfVSet, n) / sizeof(void*)), (char*)o->dev, total, &bad);
    patch_ptrs((void**)&o->m.act, (int)(offsetof(BfVSet, n) / sizeof(void*)), (char*)o->dev, total, &bad);
    if (bad) { cudaFree(o->dev); free(o); bf_set_error("bf_model_load: corrupt offsets"); return BF_EINVAL; }
    o->magic = BF_OWNED_MAGIC;
    *out = &o->m;
    return BF_OK;
}

int bf_model_build_blob(const BfModelDesc* desc, void** blob, int64_t* nbytes) {
    BF_REQUIRE(desc && blob && nbytes, "bad arguments");
    bfb::Builder b(*desc);
    BfModel img;
    if (!b.run(&img)) { bf_set_error("bf_model_create: %s", b.err ? b.err : "invalid model description"); return BF_EINVAL; }
    const int64_t total = (int64_t)b.arr.bytes.size();
    const int64_t n = 16 + (int64_t)sizeof(BfModel) + 8 + total;
    char* p = (char*)malloc((size_t)n);
    BF_REQUIRE(p, "out of host memory");
    memcpy(p, "BFMODEL1", 8);
    const int32_t abi = BF_ABI_VERSION, sz = (int32_t)sizeof(BfModel);
    memcpy(p + 8, &abi, 4); memcpy(p + 12, &sz, 4);
    memcpy(p + 16, &img, sizeof(BfModel));
    memcpy(p + 16 + sizeof(BfModel), &total, 8);
    memcpy(p + 16 + sizeof(BfModel) + 8, b.arr.bytes.data(), (size_t)total);
    *blob = p; *nbytes = n;
    return BF_OK;
}
void bf_blob_free(void* blob) { free(blob); }
int bf_model_create(const BfModelDesc* desc, BfModel** out) {
    BF_REQUIRE(desc && out, "bad arguments");
    void* blob = nullptr; int64_t n = 0;
    int rc = bf_model_build_blob(desc, &blob, &n);
    if (rc) return rc;
    rc = bf_model_load_memory(blob, n, out);
    free(blob);
    return rc;
}
int bf_model_load(const char* path, BfModel** out) {
    BF_REQUIRE(path && out, "bad arguments");
    FILE* fp = fopen(path, "rb");
    if (!fp) { bf_set_error("bf_model_load: cannot open %s", path); return BF_EINVAL; }
    fseek(fp, 0, SEEK_END);
    const long n = ftell(fp);
    fseek(fp, 0, SEEK_SET);
    void* buf = n > 0 ? malloc((size_t)n) : nullptr;
    if (!buf || fread(buf, 1, (size_t)n, fp) != (size_t)n) { fclose(fp); free(buf); bf_set_error("bf_model_load: cannot read %s", path); return BF_EINVAL; }
    fclose(fp);
    const int rc = bf_model_load_memory(buf, n, out);
    free(buf);
    return rc;
}

int bf_model_destroy(BfModel* m) {
    if (!m) return BF_OK;
    BfModelOwned* o = (BfModelOwned*)m;                        // BfModel is the first member
    BF_REQUIRE(o->magic == BF_OWNED_MAGIC, "model was not created by bf_model_load");
    o->magic = 0;
    cudaFree(o->dev);
    free(o);
    return BF_OK;
}

// frame buffers: one caller-owned device workspace carved into the BfFrames fields (what engine.FrameBuffers does with
// torch tensors).  opts: 1 = all-vertex set, 2 = buffers of the backward / optimiser, 8 = temporal term.
struct FrameCarver {
    char* base; size_t off; bool dry;
    void* take(size_t bytes) { const size_t o = off; off += (bytes + 255) & ~(size_t)255; return dry ? nullptr : (void*)(base + o); }
};
static void carve_frames(const BfModel* m, int B, int Nv, int opts, int n_trace, FrameCarver& c, BfFrames* f) {
    const bool full = opts & 1, bwd = opts & 2, temporal = opts & 8;
    const BfVSet* vs = full ? &m->full : &m->act;
    const bool tc = vs->Bt_hi && vs->Bt_lo;
    const size_t ld_v = full ? (size_t)3 * vs->n : (size_t)vs->ldn, F4 = sizeof(float);
    memset(f, 0, sizeof(*f));
    f->theta = (float*)c.take(F4 * B * m->NP);
    f->pf = (float*)c.take(F4 * B * m->Kp);
    if (tc) { f->pf_hi = (float*)c.take(F4 * B * m->Kp); f->pf_lo = (float*)c.take(F4 * B * m->Kp); }
    f->A = (float*)c.take(F4 * B * m->J * 12);
    f->Jtr = (float*)c.take(F4 * B * m->J * 3);
    f->full_pose = (float*)c.take(F4 * B * m->J * 3);
    f->yaw = (int32_t*)c.take(sizeof(int32_t) * B);
    f->verts = (float*)c.take(F4 * B * ld_v);
    f->joints = (float*)c.take(F4 * B * vs->K_out * 3);
    f->loss = (float*)c.take(F4 * B);
    if (Nv > 0) { f->kp = (const float*)c.take(F4 * B * m->K_used * Nv * 3); f->cams = (const float*)c.take(F4 * Nv * 12); }
    if (bwd) {
        f->grad = (float*)c.take(F4 * B * m->NP);
        f->adam_m = (float*)c.take(F4 * B * m->NP);
        f->adam_v = (float*)c.take(F4 * B * m->NP);
        f->dpf = (float*)c.take(F4 * B * m->Kp);
        f->dA = (float*)c.take(F4 * B * m->J * 12);
        f->dJtr = (float*)c.take(F4 * B * m->J * 3);
        f->vposed = (float*)c.take(F4 * B * ld_v);
        f->dverts = (float*)c.take(F4 * B * ld_v);
        f->dvp = (float*)c.take(F4 * B * ld_v);
        if (tc) {
            f->dvp_hi = (float*)c.take(F4 * B * vs->ldn);
            f->dvp_lo = (float*)c.take(F4 * B * vs->ldn);
            const int nsplit = (vs->ldn / TC_BK + 2048 / TC_BK - 1) / (2048 / TC_BK);
            if (nsplit > 1) { f->ws_floats = (int64_t)nsplit * B * m->Kp; f->ws = (float*)c.take(F4 * (size_t)f->ws_floats); }
        }
        f->loss_terms = (float*)c.take(F4 * B * 4);
        if (tc && m->n_gmm > 0 && (m->n_gmm * GM_LD) % TC_BN1 == 0) f->gmm_ws = (float*)c.take(F4 * B * ((size_t)m->n_gmm * GM_LD + 2 * GM_KG));
        f->gmm_grad = (float*)c.take(F4 * B * BF_GMM_D);
        f->gmm_loss = (float*)c.take(F4 * B);
        f->fwd_state = (float*)c.take(F4 * B * 24 * m->J);
        if (tc && !full && vs->lv_blk && vs->n_pad <= 512) {
            f->blk_mask = (uint32_t*)c.take(sizeof(uint32_t) * 2 * ((B + 127) / 128));
            f->dpf2 = (float*)c.take(F4 * B * m->Kp);
        }
        if (temporal) { f->tgrad = (float*)c.take(F4 * B * m->NP); f->tloss = (float*)c.take(F4 * B); }
    }
    if (n_trace > 0) f->trace = (float*)c.take(F4 * (size_t)n_trace * B);
    f->B = B; f->Nv = Nv; f->ld_v = (int)ld_v; f->iter = 0;
    f->flags = tc ? BF_F_TC : 0;
    // the reference's hard-coded hyper-parameters: smplify.py:160,167-174 (lr 0.1 for transl / scale, 1e-2 otherwise, Adam
    // defaults), loss.py:139-141 (sigma 100, prior weights 4.78 / 15.2 / 5)
    f->lr_ts = 0.1; f->lr = 1e-2; f->beta1 = 0.9; f->beta2 = 0.999; f->eps = 1e-8;
    f->imsize = 512.f; f->constant_scale = 0.3f; f->sigma = 100.f; f->w_pose = 4.78f; f->w_angle = 15.2f; f->w_shape = 5.f;
    f->w_expr = 5.f;                                  // expression prior of face models (this project's default)
}

int64_t bf_workspace_bytes(const BfModel* m, int B, int Nv, int opts, int n_trace) {
    if (!m || B <= 0 || Nv < 0 || n_trace < 0) { bf_set_error("bf_workspace_bytes: bad arguments"); return BF_EINVAL; }
    FrameCarver c{nullptr, 0, true};
    BfFrames f;
    carve_frames(m, B, Nv, opts, n_trace, c, &f);
    return (int64_t)c.off;
}

int bf_frames_bind(const BfModel* m, int B, int Nv, int opts, int n_trace, void* workspace, int64_t bytes, BfFrames* out, void* stream) {
    BF_REQUIRE(m && out && workspace && B > 0 && Nv >= 0 && n_trace >= 0, "bad arguments");
    BF_REQUIRE(((uintptr_t)workspace & 255) == 0, "workspace must be 256-byte aligned");
    const int64_t need = bf_workspace_bytes(m, B, Nv, opts, n_trace);
    BF_REQUIRE(bytes >= need, "workspace smaller than bf_workspace_bytes()");
    if (cudaMemsetAsync(workspace, 0, (size_t)need, (cudaStream_t)stream) != cudaSuccess) BF_CUDA_FAIL("memset failed");
    FrameCarver c{(char*)workspace, 0, false};
    carve_frames(m, B, Nv, opts, n_trace, c, out);
    return BF_OK;
}

// Kernel nodes of a captured CUDA graph do not inherit the priority of the stream the graph is later launched on (measured:
// four concurrently replayed part graphs all finished together whatever the priority of their streams), so the priority is
// written into every kernel node before instantiation.  `graph` = cudaGraph_t; returns the number of kernel nodes changed.
int bf_graph_set_kernel_priority(void* graph, int priority) {
    BF_REQUIRE(graph, "graph is null");
    cudaGraph_t g = (cudaGraph_t)graph;
    size_t n = 0;
    if (cudaGraphGetNodes(g, nullptr, &n) != cudaSuccess) { bf_set_error("cudaGraphGetNodes failed"); return BF_ECUDA; }
    if (n == 0) return 0;
    cudaGraphNode_t* nodes = (cudaGraphNode_t*)malloc(n * sizeof(cudaGraphNode_t));
    BF_REQUIRE(nodes, "out of host memory");
    int changed = 0;
    if (cudaGraphGetNodes(g, nodes, &n) != cudaSuccess) { free(nodes); bf_set_error("cudaGraphGetNodes failed"); return BF_ECUDA; }
    for (size_t i = 0; i < n; ++i) {
        cudaGraphNodeType t;
        if (cudaGraphNodeGetType(nodes[i], &t) != cudaSuccess || t != cudaGraphNodeTypeKernel) continue;
        cudaLaunchAttributeValue v;
        memset(&v, 0, sizeof(v));
        v.priority = priority;
        if (cudaGraphKernelNodeSetAttribute(nodes[i], cudaLaunchAttributePriority, &v) == cudaSuccess) ++changed;
    }
    free(nodes);
    cudaGetLastError();
    return changed;
}

// ---- input packing ------------------------------------------------------------------------------------------
int bf_pack_keypoints(const float* kp_raw, float* kp_packed, int B, int Nv, int K, int hand_face, const int32_t* src_index,
                      void* stream) {
    BF_NVTX();
    BF_REQUIRE(kp_raw && kp_packed && B > 0 && Nv > 0 && K > 0, "bad arguments");
    BF_REQUIRE(!hand_face || K > 67, "hand / face groups need the SMPL-X joint layout (K > 67)");
    const size_t smem = sizeof(float) * (((size_t)Nv * K * 3 + 3) / 4 * 4 + (size_t)Nv * PK_MAXG);
    BF_REQUIRE(smem <= 48 * 1024, "Nv * K too large for one frame per CTA");
    k_pack_keypoints<<<B, 256, smem, (cudaStream_t)stream>>>(kp_raw, kp_packed, B, Nv, K, hand_face, src_index);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

int bf_init_theta(const BfModel* m, const float* poses, int ld_poses, const float* betas, float* theta, int B,
                  const int32_t* src_index, void* stream) {
    BF_NVTX();
    BF_REQUIRE(m && poses && betas && theta && B > 0, "bad arguments");
    const int nb = theta_layout(m->is_smplx).nbody;
    BF_REQUIRE(ld_poses >= 3 + nb, "poses need global_orient + body_pose columns");
    const size_t n = (size_t)B * m->NP;
    k_init_theta<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(poses, ld_poses, betas, theta, B, m->NP, nb,
                                                                                 m->NB < 10 ? m->NB : 10, src_index);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

int bf_scatter_rows(const float* src, const int32_t* index, float* dst, int rows, int cols, void* stream) {
    BF_NVTX();
    BF_REQUIRE(src && dst && rows > 0 && cols > 0, "bad arguments");
    const size_t n = (size_t)rows * cols;
    k_scatter_rows<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(src, index, dst, rows, cols);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

// ---- NVLink halo of the temporal term (bf_pack.cuh) --------------------------------------------------------------
int bf_halo_bytes(void) { return (int)(BF_HALO_FLOATS * sizeof(float)); }
int bf_halo_handle_bytes(void) { return (int)sizeof(cudaIpcMemHandle_t); }

int bf_halo_alloc(void** buf, void* ipc_handle_out) {
    BF_REQUIRE(buf, "buf is null");
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, BF_HALO_FLOATS * sizeof(float));
    if (e != cudaSuccess) { bf_set_error("bf_halo_alloc: cudaMalloc: %s", cudaGetErrorString(e)); return BF_ECUDA; }
    cudaMemset(p, 0, BF_HALO_FLOATS * sizeof(float));
    cudaDeviceSynchronize();
    if (ipc_handle_out) {
        cudaIpcMemHandle_t h;
        e = cudaIpcGetMemHandle(&h, p);
        if (e != cudaSuccess) { cudaFree(p); bf_set_error("bf_halo_alloc: cudaIpcGetMemHandle: %s", cudaGetErrorString(e)); return BF_ECUDA; }
        memcpy(ipc_handle_out, &h, sizeof(h));
    }
    *buf = p;
    return BF_OK;
}
int bf_halo_open(const void* ipc_handle, void** peer_buf) {
    BF_REQUIRE(ipc_handle && peer_buf, "bad arguments");
    cudaIpcMemHandle_t h;
    memcpy(&h, ipc_handle, sizeof(h));
    cudaError_t e = cudaIpcOpenMemHandle(peer_buf, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) { bf_set_error("bf_halo_open: cudaIpcOpenMemHandle: %s", cudaGetErrorString(e)); return BF_ECUDA; }
    return BF_OK;
}
int bf_halo_close(void* peer_buf) {
    if (peer_buf && cudaIpcCloseMemHandle(peer_buf) != cudaSuccess) { bf_set_error("bf_halo_close failed"); return BF_ECUDA; }
    return BF_OK;
}
int bf_halo_free(void* buf) {
    if (buf && cudaFree(buf) != cudaSuccess) { bf_set_error("bf_halo_free failed"); return BF_ECUDA; }
    return BF_OK;
}
int bf_halo_begin(const BfModel* m, const BfFrames* f, int n_iters, void* stream) {
    BF_NVTX();
    int rc = check_model(m, f); if (rc) return rc;
    BF_REQUIRE(f->halo_buf && n_iters > 0, "halo buffer missing");
    k_halo_begin<<<1, 64, 0, (cudaStream_t)stream>>>(*f, m->NP, n_iters);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

// ---- uniform grid / closest point / SMPL+D (include/bodyfit_b200_grid.h) ------------------------------
static int check_grid(const BfGrid* g) {
    BF_REQUIRE(g && g->verts && g->faces && g->cell_start, "grid tables missing");
    BF_REQUIRE(g->step > 0.f && g->dim[0] > 0 && g->dim[1] > 0 && g->dim[2] > 0, "bad grid geometry");
    BF_REQUIRE((long long)g->dim[0] * g->dim[1] * g->dim[2] == g->ncell, "ncell != dim product");
    BF_REQUIRE(g->Fs > 0 && g->Ns > 0, "empty mesh");
    return BF_OK;
}

int bf_grid_count(const BfGrid* g, int32_t* counts, void* stream) {
    BF_NVTX();
    int rc = check_grid(g); if (rc) return rc;
    BF_REQUIRE(counts, "counts is null");
    cudaStream_t s = (cudaStream_t)stream;
    if (cudaMemsetAsync(counts, 0, sizeof(int32_t) * g->ncell, s) != cudaSuccess) BF_CUDA_FAIL("memset failed");
    k_grid_insert<<<(g->Fs + 255) / 256, 256, 0, s>>>(*g, counts, nullptr, nullptr);
    BF_LAUNCH_CHECK();
    k_grid_scan<<<1, 1024, 0, s>>>(counts, g->cell_start, g->ncell);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

int bf_grid_fill(const BfGrid* g, int32_t* cursor, void* stream) {
    BF_NVTX();
    int rc = check_grid(g); if (rc) return rc;
    BF_REQUIRE(cursor && g->cell_tris, "cursor / cell_tris is null");
    cudaStream_t s = (cudaStream_t)stream;
    if (cudaMemsetAsync(cursor, 0, sizeof(int32_t) * g->ncell, s) != cudaSuccess) BF_CUDA_FAIL("memset failed");
    k_grid_insert<<<(g->Fs + 255) / 256, 256, 0, s>>>(*g, cursor, g->cell_start, g->cell_tris);
    BF_LAUNCH_CHECK();
    k_grid_sort<<<(g->ncell + 255) / 256, 256, 0, s>>>(g->cell_start, g->cell_tris, g->ncell);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

int bf_grid_nearest(const BfGrid* g, const float* points, int Q, float* near_pts, int32_t* near_faces, float* dist2, void* stream) {
    BF_NVTX();
    int rc = check_grid(g); if (rc) return rc;
    BF_REQUIRE(g->cell_tris && points && near_pts && near_faces && Q > 0, "bad arguments");
    k_grid_nearest<<<(Q + 7) / 8, 256, 0, (cudaStream_t)stream>>>(*g, points, Q, near_pts, near_faces, dist2);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

int bf_grid_barycentric(const BfGrid* g, const float* points, const int32_t* near_faces, int Q, float* coeff, void* stream) {
    BF_NVTX();
    BF_REQUIRE(g && g->verts && g->faces && points && near_faces && coeff && Q > 0, "bad arguments");
    k_grid_bary<<<(Q + 255) / 256, 256, 0, (cudaStream_t)stream>>>(*g, points, near_faces, Q, coeff);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

int bf_grid_nearest_backward(const BfGrid* g, const float* points, const int32_t* near_faces, int Q, float* grad, void* stream) {
    BF_NVTX();
    BF_REQUIRE(g && g->verts && g->faces && points && near_faces && grad && Q > 0, "bad arguments");
    k_grid_nearest_bwd<<<(Q + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*g, points, near_faces, Q, grad);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

int bf_grid_inside(const BfGrid* g, const float* points, int Q, float* signs, void* stream) {
    BF_NVTX();
    int rc = check_grid(g); if (rc) return rc;
    BF_REQUIRE(g->cell_tris && points && signs && Q > 0, "bad arguments");
    k_grid_inside<<<(Q + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*g, points, Q, signs);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

int bf_grid_intersects_any(const BfGrid* g, const float* origins, const float* directions, int Q, uint8_t* hit, void* stream) {
    BF_NVTX();
    int rc = check_grid(g); if (rc) return rc;
    BF_REQUIRE(g->cell_tris && origins && directions && hit && Q > 0, "bad arguments");
    k_grid_ray_any<<<(Q + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*g, origins, directions, Q, hit);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

int bf_smpld_step(const BfGrid* g, const BfSmpld* p, void* stream) {
    BF_NVTX();
    int rc = check_grid(g); if (rc) return rc;
    BF_REQUIRE(p && p->base && p->disp && p->adam_m && p->adam_v && p->faces && p->vf_ptr && p->vf_face && p->scan_fn &&
               p->P && p->C && p->near_faces && p->nhat && p->nlen && p->m && p->Nlen && p->dN && p->dcorner &&
               p->partial && p->totals && p->V > 0 && p->F > 0, "SMPL+D buffers missing");
    cudaStream_t s = (cudaStream_t)stream;
    const int V = p->V, F = p->F, nb = 64;
    k_add3<<<(3 * V + 255) / 256, 256, 0, s>>>(p->base, p->disp, p->P, 3 * V);
    BF_LAUNCH_CHECK();
    k_face_normals<<<(F + 255) / 256, 256, 0, s>>>(p->P, p->faces, F, p->nhat, p->nlen);
    BF_LAUNCH_CHECK();
    k_vertex_normals<<<(V + 255) / 256, 256, 0, s>>>(p->nhat, p->vf_ptr, p->vf_face, V, p->m, p->Nlen);
    BF_LAUNCH_CHECK();
    k_grid_nearest<<<(V + 7) / 8, 256, 0, s>>>(*g, p->P, V, p->C, p->near_faces, nullptr);
    BF_LAUNCH_CHECK();
    k_smpld_partials<<<nb, 256, 0, s>>>(p->P, p->C, p->near_faces, p->scan_fn, p->m, p->faces, V, F, p->partial);
    BF_LAUNCH_CHECK();
    k_smpld_finish<<<1, 32, 0, s>>>(p->partial, nb, V, F, p->reg_scale, p->totals);
    BF_LAUNCH_CHECK();
    k_smpld_dm<<<(V + 255) / 256, 256, 0, s>>>(p->near_faces, p->scan_fn, p->m, p->faces, p->vf_ptr, p->vf_face, V, F,
                                               p->reg_scale, p->Nlen, p->dN);
    BF_LAUNCH_CHECK();
    k_smpld_dface<<<(F + 255) / 256, 256, 0, s>>>(p->P, p->faces, p->nhat, p->nlen, p->dN, F, p->dcorner);
    BF_LAUNCH_CHECK();
    const double t = (double)(p->iter + 1);
    const double bc1 = 1.0 - pow(p->beta1, t), bc2 = 1.0 - pow(p->beta2, t);
    k_smpld_step<<<(V + 255) / 256, 256, 0, s>>>(p->P, p->C, p->totals, p->dcorner, p->faces, p->vf_ptr, p->vf_face, V,
                                                 p->disp, p->adam_m, p->adam_v, p->grad, (float)(p->lr / bc1), (float)sqrt(bc2),
                                                 (float)p->beta2, (float)(1.0 - p->beta1), (float)(1.0 - p->beta2), (float)p->eps);
    BF_LAUNCH_CHECK();
    if (p->trace) {
        if (cudaMemcpyAsync(p->trace + 4 * (size_t)p->iter, p->totals, 4 * sizeof(float), cudaMemcpyDeviceToDevice, s) != cudaSuccess) {
            BF_CUDA_FAIL("trace copy failed");
        }
    }
    return BF_OK;
}

int bf_smpld_run(const BfGrid* g, const BfSmpld* p, int n_iters, void* stream) {
    BF_NVTX();
    BF_REQUIRE(g && p && n_iters >= 0, "bad arguments");
    BfSmpld q = *p;
    for (int i = 0; i < n_iters; ++i) {
        int rc = bf_smpld_step(g, &q, stream); if (rc) return rc;
        q.iter++;
    }
    return BF_OK;
}

// world-space copy of the skinned vertices: Pw = (v + transl) * scale * cs  (smplify/smplify.py:190)
__global__ void k_world_points(const float* __restrict__ verts, const float* __restrict__ theta, int NP, int V, int ld_v,
                               float cs, float* __restrict__ Pw, int B) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)B * V) return;
    const int b = (int)(i / V), v = (int)(i % V);
    const float* th = theta + (size_t)b * NP;
    const float* p = verts + (size_t)b * ld_v + 3 * v;
    const float sc = th[3];
    Pw[3 * i] = (p[0] + th[0]) * sc * cs; Pw[3 * i + 1] = (p[1] + th[1]) * sc * cs; Pw[3 * i + 2] = (p[2] + th[2]) * sc * cs;
}

// per frame: n = |Pw - C|_F ; loss[b] += weight*scale*n ; g = weight*scale*(Pw - C)/n is d/dPw, chained to the
// model-space vertices (x s cs), transl (sum g s cs) and scale (sum g.(v+t) cs)
__global__ void __launch_bounds__(256) k_pc_world_bwd(const float* __restrict__ verts, const float* __restrict__ Pw,
                                                      const float* __restrict__ C, const float* __restrict__ theta, int NP,
                                                      int V, int ld_v, float cs, float scale, float weight,
                                                      float* __restrict__ loss, float* __restrict__ pc_loss,
                                                      float* __restrict__ dverts, float* __restrict__ grad) {
    __shared__ float red[4][8];
    __shared__ float nrm;
    const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float* P = Pw + (size_t)b * V * 3;
    const float* Cb = C + (size_t)b * V * 3;
    float acc = 0.f;
    for (int i = threadIdx.x; i < 3 * V; i += 256) { const float d = P[i] - Cb[i]; acc += d * d; }
    acc = warp_sum(acc);
    if (lane == 0) red[0][warp] = acc;
    __syncthreads();
    if (threadIdx.x == 0) { float s = 0.f; for (int w = 0; w < 8; ++w) s += red[0][w]; nrm = sqrtf(s); }
    __syncthreads();
    const float* th = theta + (size_t)b * NP;
    const float sc = th[3];
    const float k = weight * scale / nrm;
    float g0 = 0.f, g1 = 0.f, g2 = 0.f, gs = 0.f;
    float* dv = dverts + (size_t)b * ld_v;
    const float* vb = verts + (size_t)b * ld_v;
    for (int v = threadIdx.x; v < V; v += 256) {
        float gw[3];
#pragma unroll
        for (int d = 0; d < 3; ++d) gw[d] = k * (P[3 * v + d] - Cb[3 * v + d]);
#pragma unroll
        for (int d = 0; d < 3; ++d) dv[3 * v + d] += gw[d] * sc * cs;
        g0 += gw[0] * sc * cs; g1 += gw[1] * sc * cs; g2 += gw[2] * sc * cs;
        gs += (gw[0] * (vb[3 * v] + th[0]) + gw[1] * (vb[3 * v + 1] + th[1]) + gw[2] * (vb[3 * v + 2] + th[2])) * cs;
    }
    g0 = warp_sum(g0); g1 = warp_sum(g1); g2 = warp_sum(g2); gs = warp_sum(gs);
    __syncthreads();
    if (lane == 0) { red[0][warp] = g0; red[1][warp] = g1; red[2][warp] = g2; red[3][warp] = gs; }
    __syncthreads();
    if (threadIdx.x < 4) {
        float s = 0.f;
        for (int w = 0; w < 8; ++w) s += red[threadIdx.x][w];
        grad[(size_t)b * NP + threadIdx.x] += s;
    }
    if (threadIdx.x == 0) { loss[b] += weight * scale * nrm; if (pc_loss) pc_loss[b] = scale * nrm; }
}

int bf_mask_loss(const BfModel* m, const BfFrames* f, const BfMask* k, float weight, void* stream) {
    BF_NVTX();
    int rc = check_model(m, f); if (rc) return rc;
    const int V = m->full.n;
    BF_REQUIRE(k && k->masks && k->cams && k->contour && k->cptr && k->cown && k->uv && k->near_q && k->cdist && k->cw && k->dPw &&
               k->part, "mask buffers missing");
    BF_REQUIRE(k->Nm > 0 && k->H > 0 && k->W > 0 && k->stride > 0 && k->Nq == (V + k->stride - 1) / k->stride && k->total >= 0 &&
               k->imsize > 0.f, "bad mask geometry");
    BF_REQUIRE(f->verts && f->dverts && f->grad && f->loss && f->ld_v >= 3 * V, "all-vertex frame buffers missing");
    cudaStream_t s = (cudaStream_t)stream;
    const size_t n = (size_t)f->B * k->Nm * k->Nq;
    k_mask_project<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(*f, *k, m->NP);
    BF_LAUNCH_CHECK();
    if (k->total > 0) {
        k_mask_nearest<<<(k->total + 7) / 8, 256, 0, s>>>(*k, k->total);
        BF_LAUNCH_CHECK();
    }
    k_mask_vertex<<<(unsigned)(((size_t)f->B * k->Nq + 127) / 128), 128, 0, s>>>(*f, *k, m->NP);
    BF_LAUNCH_CHECK();
    k_mask_finish<<<f->B, 256, 0, s>>>(*f, *k, m->NP, weight);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

int bf_pc_loss(const BfGrid* g, const BfModel* m, const BfFrames* f, float scale, float weight, float* Pw,
               float* near_pts, int32_t* near_faces, float* pc_loss, void* stream) {
    BF_NVTX();
    int rc = check_grid(g); if (rc) return rc;
    rc = check_model(m, f); if (rc) return rc;
    const int V = m->full.n;
    BF_REQUIRE(f->verts && f->dverts && f->grad && f->loss && Pw && near_pts && near_faces && f->ld_v >= 3 * V, "bad arguments");
    cudaStream_t s = (cudaStream_t)stream;
    const size_t n = (size_t)f->B * V;
    k_world_points<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(f->verts, f->theta, m->NP, V, f->ld_v, f->constant_scale, Pw, f->B);
    BF_LAUNCH_CHECK();
    k_grid_nearest<<<(unsigned)((n + 7) / 8), 256, 0, s>>>(*g, Pw, (int)n, near_pts, near_faces, nullptr);
    BF_LAUNCH_CHECK();
    k_pc_world_bwd<<<f->B, 256, 0, s>>>(f->verts, Pw, near_pts, f->theta, m->NP, V, f->ld_v, f->constant_scale, scale, weight,
                                        f->loss, pc_loss, f->dverts, f->grad);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

// ---- scan / normal / silhouette terms as stand-alone operators (include/bodyfit_b200_ops.h) ---------------------------
int bf_op_pc_loss(const float* points, const float* closest, int64_t n, float* out, float* dpoints, void* stream) {
    BF_NVTX();
    BF_REQUIRE(points && closest && out && dpoints && n > 0 && n < (1LL << 31), "bad arguments");
    k_op_pc_loss<<<1, 1024, 0, (cudaStream_t)stream>>>(points, closest, (int)n, out, dpoints);
    BF_LAUNCH_CHECK();
    return BF_OK;
}
int bf_op_normal_loss(const int32_t* near_faces, const float* face_norm, const float* point_norm, int V, float* out,
                      float* dpoint_norm, void* stream) {
    BF_NVTX();
    BF_REQUIRE(near_faces && face_norm && point_norm && out && dpoint_norm && V > 0, "bad arguments");
    k_op_normal_loss<<<1, 1024, 0, (cudaStream_t)stream>>>(near_faces, face_norm, point_norm, V, out, dpoint_norm);
    BF_LAUNCH_CHECK();
    return BF_OK;
}
int bf_op_laplacian(const float* norms, const int32_t* faces, const int32_t* vf_ptr, const int32_t* vf_face, int V, int F,
                    float* out, float* dnorms, void* stream) {
    BF_NVTX();
    BF_REQUIRE(norms && faces && vf_ptr && vf_face && out && dnorms && V > 0 && F > 0, "bad arguments");
    k_op_laplacian_value<<<1, 1024, 0, (cudaStream_t)stream>>>(norms, faces, F, out);
    BF_LAUNCH_CHECK();
    k_op_laplacian_grad<<<(V + 255) / 256, 256, 0, (cudaStream_t)stream>>>(norms, faces, vf_ptr, vf_face, V, F, dnorms);
    BF_LAUNCH_CHECK();
    return BF_OK;
}
int bf_op_vertex_normals(const float* verts, const int32_t* faces, const int32_t* vf_ptr, const int32_t* vf_face, int V, int F,
                         float* nhat, float* nlen, float* normals, float* Nlen, void* stream) {
    BF_NVTX();
    BF_REQUIRE(verts && faces && vf_ptr && vf_face && nhat && nlen && normals && Nlen && V > 0 && F > 0, "bad arguments");
    k_face_normals<<<(F + 255) / 256, 256, 0, (cudaStream_t)stream>>>(verts, faces, F, nhat, nlen);
    BF_LAUNCH_CHECK();
    k_vertex_normals<<<(V + 255) / 256, 256, 0, (cudaStream_t)stream>>>(nhat, vf_ptr, vf_face, V, normals, Nlen);
    BF_LAUNCH_CHECK();
    return BF_OK;
}
int bf_op_vertex_normals_backward(const float* verts, const int32_t* faces, const int32_t* vf_ptr, const int32_t* vf_face, int V,
                                  int F, const float* nhat, const float* nlen, const float* normals, const float* Nlen,
                                  const float* dnormals, float* dm_scratch, float* dcorner_scratch, float* dverts, void* stream) {
    BF_NVTX();
    BF_REQUIRE(verts && faces && vf_ptr && vf_face && nhat && nlen && normals && Nlen && dnormals && dm_scratch &&
               dcorner_scratch && dverts && V > 0 && F > 0, "bad arguments");
    cudaStream_t s = (cudaStream_t)stream;
    k_op_vnormal_bwd<<<(V + 255) / 256, 256, 0, s>>>(dnormals, normals, Nlen, V, dm_scratch);
    BF_LAUNCH_CHECK();
    k_smpld_dface<<<(F + 255) / 256, 256, 0, s>>>(verts, faces, nhat, nlen, dm_scratch, F, dcorner_scratch);
    BF_LAUNCH_CHECK();
    k_op_corner_gather<<<(V + 255) / 256, 256, 0, s>>>(dcorner_scratch, faces, vf_ptr, vf_face, V, dverts);
    BF_LAUNCH_CHECK();
    return BF_OK;
}
int bf_op_regress_joints(const float* points, const int32_t* ptr, const int32_t* idx, const float* w, int B, int N, int R,
                         float* out, void* stream) {
    BF_NVTX();
    BF_REQUIRE(points && ptr && idx && w && out && B > 0 && N > 0 && R > 0, "bad arguments");
    const size_t warps = (size_t)B * R;
    k_op_spmm3<<<(unsigned)((warps + 7) / 8), 256, 0, (cudaStream_t)stream>>>(points, ptr, idx, w, B, N, R, out);
    BF_LAUNCH_CHECK();
    return BF_OK;
}
int bf_op_mask_loss(const float* verts_world, int B, int V, const BfMask* k, float* scratch, float* loss, float* dverts,
                    void* stream) {
    BF_NVTX();
    BF_REQUIRE(verts_world && k && scratch && loss && dverts && B > 0 && V > 0, "bad arguments");
    BF_REQUIRE(k->masks && k->cams && k->contour && k->cptr && k->cown && k->uv && k->near_q && k->cdist && k->cw && k->dPw && k->part,
               "mask buffers missing");
    BF_REQUIRE(k->Nm > 0 && k->H > 0 && k->W > 0 && k->stride > 0 && k->Nq == (V + k->stride - 1) / k->stride && k->total >= 0 &&
               k->imsize > 0.f, "bad mask geometry");
    cudaStream_t s = (cudaStream_t)stream;
    // world-space vertices in, world-space gradient out: identity (transl 0, scale 1, constant_scale 1) frames of NP = 4
    BfFrames f;
    memset(&f, 0, sizeof(f));
    f.theta = scratch; f.grad = scratch + 4 * (size_t)B;
    f.verts = const_cast<float*>(verts_world); f.dverts = dverts; f.loss = loss;
    f.B = B; f.ld_v = 3 * V; f.constant_scale = 1.0f;
    k_op_identity_theta<<<(B + 127) / 128, 128, 0, s>>>(scratch, B);
    BF_LAUNCH_CHECK();
    if (cudaMemsetAsync(f.grad, 0, sizeof(float) * 4 * (size_t)B, s) != cudaSuccess || cudaMemsetAsync(loss, 0, sizeof(float) * B, s) != cudaSuccess ||
        cudaMemsetAsync(dverts, 0, sizeof(float) * 3 * (size_t)V * B, s) != cudaSuccess) BF_CUDA_FAIL("memset failed");
    const size_t n = (size_t)B * k->Nm * k->Nq;
    k_mask_project<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(f, *k, 4);
    BF_LAUNCH_CHECK();
    if (k->total > 0) {
        k_mask_nearest<<<(k->total + 7) / 8, 256, 0, s>>>(*k, k->total);
        BF_LAUNCH_CHECK();
    }
    k_mask_vertex<<<(unsigned)(((size_t)B * k->Nq + 127) / 128), 128, 0, s>>>(f, *k, 4);
    BF_LAUNCH_CHECK();
    k_mask_finish<<<B, 256, 0, s>>>(f, *k, 4, 1.0f);
    BF_LAUNCH_CHECK();
    return BF_OK;
}

}  // extern "C"
