/*
 * bodyfit_b200.h -- C ABI of the B200 (sm_100a) SMPLify fitting core.
 *
 * Every entry point is `extern "C"`, takes plain device pointers + sizes and a
 * cudaStream_t (passed as void*), launches on that stream, never allocates and never
 * synchronises.  Return value: 0 on success, a negative BF_E* code otherwise;
 * bf_last_error() gives the text.  There is no CPU fallback: a device that is not
 * compute capability 10.x is an error (BF_EARCH).
 *
 * Reference interfaces replaced (file:line relative to the reference repo):
 *   bf_lbs_forward / bf_lbs_backward
 *       models/smpl.py:69-83 SMPL.forward, smplx.SMPL/SMPLX.forward + smplx.lbs.lbs
 *       (un-vendored, call sites models/smpl.py:71, smplify/smplify.py:179-187) and
 *       their autograd backward.
 *   bf_fit_step / bf_fit_run
 *       smplify/smplify.py:177-213 (one / n iterations of the SMPLify loop:
 *       model forward, smplify/loss.py:139-230 multiview_keypoint_loss incl.
 *       :22-51,:132-136 projection + GMoF, smplify/prior.py:181-196 GMM prior,
 *       loss.py:54-61 angle prior, shape L2, loss.backward(), torch.optim.Adam.step()
 *       as configured at smplify.py:167-174).
 *   bf_grid_* (declared in bodyfit_b200_grid.h)
 *       thirdparty/mesh_grid/mesh_grid.cpp:129-136.
 *
 * All floating point data is fp32, row-major, contiguous unless a leading dimension
 * is given.  "theta" is the per-frame optimisation vector:
 *   [transl 3 | scale 1 | global_orient 3 | body_pose 69(smpl) or 63(smplx) | betas 10 |
 *    (smplx only) leye 3 | reye 3 | left_hand nh | right_hand nh |
 *    (face-parameter smplx model only, BfModel.face) jaw 3 | expression NE]   NP = 86 / 98 / 86 + 2 nh (+ 3 + NE)
 * with 10 betas (num_betas in general; 11 for the kid model).  nh = BfModel.n_hand: the number of hand PCA components
 * (6 by default, BfModelDesc.num_pca_comps), or 45 axis-angle entries per hand without PCA (BfModelDesc.hand_axis_angle).
 * The face block of a face-parameter model (BfModelDesc.face_params) follows every other entry, so all other offsets are
 * the same with and without it; every offset before left_hand is the same for every hand configuration.  The longest row
 * (axis-angle hands and face parameters) has 7 + 63 + 10 + 6 + 90 + 3 + 10 = 189 entries.
 */
#ifndef BODYFIT_B200_H
#define BODYFIT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BF_OK        0
#define BF_EINVAL   -1   /* bad argument (null pointer, bad size)          */
#define BF_ECUDA    -2   /* a CUDA runtime call / launch failed            */
#define BF_EARCH    -3   /* device is not sm_100 (no fallback exists)      */

#define BF_ABI_VERSION 21
#define BF_F_WORLD 1   /* forward outputs in world space: (x + transl) * scale * constant_scale */
#define BF_F_TC    2   /* run the blend-shape contractions on tcgen05 tensor cores (3xTF32) */
#define BF_F_SKIN_FUSED 4  /* bf_frame_loss_backward skins the frame's live vertices itself from vposed (after bf_blend_forward) */

/* A vertex set: either all V vertices of the model or the compacted "active" subset
 * that the keypoint loss can touch.  All index tables refer to positions in this set. */
typedef struct BfVSet {
    const float*   Bm;        /* [Kp, ldn] blend matrix: rows 0..P-1 posedirs, P..P+NS-1 shapedirs^T, P+NS v_template, rest 0 */
    const int32_t* ell_j;     /* [n_pad, nnz] skinning joint ids (ELL, padded with j=0,w=0) */
    const float*   ell_w;     /* [n_pad, nnz] skinning weights */
    const int32_t* jv_ptr;    /* [J+1] CSR by joint over (vertex, weight), for dA */
    const int32_t* jv_vid;    /* [jv_ptr[J]] */
    const float*   jv_w;      /* [jv_ptr[J]] */
    const int32_t* kj_kind;   /* [K_out] 0 chain joint, 1 vertex combination, 2 dynamic landmark slot, 3 regressed extra row */
    const int32_t* kj_src;    /* [K_out,3] chain joint id | vertex ids | slot | row */
    const float*   kj_w;      /* [K_out,3] barycentric weights (kind 1) */
    const int32_t* dyn_src;   /* [79,n_dyn,3] vertex ids per yaw row (or NULL) */
    const float*   dyn_w;     /* [79,n_dyn,3] */
    const int32_t* tg_ptr;    /* [J+n+1] CSR by target (J chain joints, then n vertices) over output joints */
    const int32_t* tg_k;      /* output joint index */
    const int32_t* tg_a;      /* yaw row the entry is valid for, or -1 = always */
    const float*   tg_w;      /* weight */
    const int32_t* xr_ptr;    /* [n_extra+1] CSR of the extra joint regressor (models/smpl.py:62-65,72) or NULL */
    const int32_t* xr_vid;
    const float*   xr_w;
    const float*   Bt_hi;     /* [ldn, Kp] Bm^T split for 3xTF32: tf32-rounded part ... */
    const float*   Bt_lo;     /* ... and the fp32 remainder (forward GEMM B operand, K-major) */
    const float*   Bm_hi;     /* [Kp, ldn] the same split of Bm (backward GEMM B operand, K-major) */
    const float*   Bm_lo;
    const int32_t* dyn_k;     /* [n_dyn] output joint index of each contour-landmark slot */
    const int32_t* jv_nz;     /* [n_nz] joints with a non-empty jv list */
    /* "live" lists of the active set, one row per contour (yaw) row -- n_rows = 79 for SMPL-X, 1 otherwise; NULL for the
     * full set.  A frame on row a has non-zero keypoint gradients only on lv_vid[a][0..lv_n[a]) */
    const int32_t* lv_n;      /* [n_rows] */
    const int32_t* lv_vid;    /* [n_rows, lmax] positions in this set, ascending */
    const int32_t* lt_ptr;    /* [n_rows, lmax+1] absolute offsets into lt_k / lt_w: gradient gather list of live vertex i */
    const int32_t* lt_k;      /* output joint index */
    const float*   lt_w;      /* weight (static entries first, then contour entries in slot order) */
    const int32_t* lj_ptr;    /* [n_rows, n_nz+1] absolute offsets: skinning list of joint jv_nz[jn] restricted to live vertices */
    const int32_t* lj_vid;    /* index into the row's live list (lv_vid[a][.]) */
    const float*   lj_w;
    const uint32_t* lv_blk;   /* [n_rows] bit i set = a frame on this row has live vertices in the 16-vertex block i of the set
                                 (the set is ordered static vertices first, then contour candidates by first row; NULL = full set) */
    int32_t n, n_pad, ldn, nnz, K_out, n_dyn, n_extra, n_nz, lmax, n_rows;
} BfVSet;

typedef struct BfModel {
    const int32_t* parents;   /* [J] */
    const int32_t* depth;     /* [J] */
    const int32_t* lvl_ptr;   /* [max_depth+2] CSR over lvl_j: joints of tree level d are lvl_j[lvl_ptr[d] .. lvl_ptr[d+1]) */
    const int32_t* lvl_j;     /* [J] joints sorted by depth (stable) */
    const int32_t* child_ptr; /* [J+1] */
    const int32_t* child_idx; /* [J-1] */
    const float*   Jt;        /* [J,3]     J_regressor @ v_template */
    const float*   Jd;        /* [J,3,NS]  J_regressor @ shapedirs  */
    const float*   pose_mean; /* [3J] */
    const float*   hand_l;    /* [n_hand,45] hand components (the identity for axis-angle hands) or NULL */
    const float*   hand_r;    /* [n_hand,45] or NULL */
    const float*   gmm_mean;  /* [8,69] */
    const float*   gmm_psym;  /* [8,69,72] (P + P^T)/2 of each component, rows padded with zeros to 72 */
    const float*   gmm_logw;  /* [8] log(nll_weights) */
    const float*   gmm_bt_hi; /* [n_gmm*72, 80] K-major [P_sym,m | -P_sym,m mu_m | 0], 3xTF32 split: the prior as one tcgen05 GEMM (or NULL) */
    const float*   gmm_bt_lo;
    BfVSet full;
    BfVSet act;
    int32_t J, P, NS, NB, Kp, NP, is_smplx, max_depth, K_used, n_gmm;
    int32_t face;             /* 1 = face-parameter SMPL-X model: theta carries jaw pose + the NS - NB expression coefficients */
    int32_t n_hand;           /* SMPL-X: hand parameters per hand in theta (num_pca_comps, or 45 for axis-angle hands); 0 for SMPL */
} BfModel;

/* Per-call frame buffers (all device memory, B frames). */
typedef struct BfFrames {
    float*       theta;      /* [B,NP] in/out */
    float*       grad;       /* [B,NP] out */
    float*       adam_m;     /* [B,NP] */
    float*       adam_v;     /* [B,NP] */
    float*       pf;         /* [B,Kp]   GEMM A operand: pose feature | shape | 1 */
    float*       dpf;        /* [B,Kp] */
    float*       A;          /* [B,J,12] rest-pose-removed joint transforms */
    float*       dA;         /* [B,J,12] */
    float*       Jtr;        /* [B,J,3]  posed joints */
    float*       dJtr;       /* [B,J,3] */
    float*       full_pose;  /* [B,3J] */
    int32_t*     yaw;        /* [B] dynamic-landmark row */
    float*       verts;      /* [B,ld_v] skinned vertices of the vertex set in use */
    float*       vposed;     /* [B,ld_v] blended (unskinned) vertices, saved for backward */
    float*       dverts;     /* [B,ld_v] */
    float*       dvp;        /* [B,ld_v] */
    float*       joints;     /* [B,K_out,3] model-space output joints (optional, may be NULL) */
    float*       djoints;    /* [B,K_out,3] incoming joint gradient (operator backward) or NULL */
    const float* kp;         /* [B,K_used,Nv,3] (x, y, effective weight), joint-major: the views of a joint are contiguous */
    const float* cams;       /* [Nv,12] row-major 3x4  K @ [R|t] (world -> pixel, homogeneous) */
    float*       loss;       /* [B] per-frame total loss of this iteration */
    float*       loss_terms; /* [B,4] data, pose prior, angle prior, shape prior (+ expression prior, face models) (optional) */
    float*       trace;      /* [n_iters,B] optional per-iteration loss trace */
    float*       pf_hi;      /* [B,Kp]  3xTF32 split of pf (BF_F_TC) */
    float*       pf_lo;
    float*       dvp_hi;     /* [B,ldn] 3xTF32 split of dvp, row stride = ldn of the vertex set, pad columns 0 */
    float*       dvp_lo;
    float*       gmm_grad;   /* [B,69] w_pose^2 * gradient of the GMM prior (k_gmm_prior -> k_pose_bwd) */
    float*       gmm_loss;   /* [B]    w_pose^2 * min_m ll_m */
    float*       tgrad;      /* [B,NP] gradient of the temporal smoothness term (bf_temporal_prior -> k_pose_bwd), or NULL */
    float*       tloss;      /* [B]    its per-frame value */
    const float* halo_prev;  /* [NP] theta of the frame before this shard's first frame (previous rank), NULL at the sequence start */
    const float* halo_next;  /* [NP] theta of the frame after this shard's last frame (next rank), NULL at the sequence end */
    float*       halo_buf;       /* NVLink halo (bf_halo_*): this rank's own halo buffer, or NULL = host-exchanged rows above */
    float*       halo_peer_prev; /* the previous rank's halo buffer mapped into this process (NULL on the first rank) */
    float*       halo_peer_next; /* the next rank's halo buffer (NULL on the last rank) */
    float*       fwd_state;  /* [B,24J] optional: full_pose, R, rest joints, chain rotations saved by the pose forward so the
                                pose backward does not recompute them */
    float*       gmm_ws;     /* [B, n_gmm*72 + 160] workspace of the tensor-core GMM prior (y of every component | [pose|1] hi | lo), or NULL */
    float*       ws;         /* split-K workspace of the tensor-core backward GEMM (>= ceil(ldn/2048) * B * Kp floats) or NULL */
    uint32_t*    blk_mask;   /* [2, ceil(B/128)] (or NULL): per 128-frame tile the OR of lv_blk over its frames' yaw rows -- the
                                16-vertex blocks of the active set the blend GEMMs have to touch for that tile.  Written by the pose
                                forward (buffer = iteration parity), cleared by the per-frame kernel; zero before the first iteration */
    float*       dpf2;       /* [B,Kp] (or NULL): second half-reduction of the masked blend backward GEMM; when set (together with
                                blk_mask) the GEMM cuts every tile's reduction in two runs, dpf and dpf2, and bf_pose_backward adds
                                them (dpf + dpf2, fixed order) */
    const int32_t* frame_index; /* [B] (or NULL = identity): row of `kp` that belongs to frame b.  The host may process the frames
                                   of a batch in any order (and re-order them between iterations: only theta / adam_m / adam_v rows
                                   move); the 13 KB keypoint rows stay where they are behind this index */
    int64_t      ws_floats;
    double lr_ts, lr, beta1, beta2, eps;   /* Adam hyper-parameters (python floats in the reference: smplify.py:167-174) */
    int32_t B, Nv, ld_v, iter; /* Nv: camera views, 1 to 64 */
    int32_t flags;             /* BF_F_WORLD: skin/joints forward write (x + transl) * scale * constant_scale (smplify.py:189-190) */
    int32_t halo_iters;        /* NVLink halo: iterations of the run; iteration `iter` publishes its updated boundary rows iff iter + 1 < halo_iters */
    float imsize, constant_scale, sigma, w_pose, w_angle, w_shape;
    float w_temporal;          /* weight of the temporal term (0 = off; not part of the reference) */
    float w_expr;              /* face models: expression prior w_expr^2 sum psi^2 (this project's term, the reference has none;
                                  bf_frames_bind sets 5).  Face-off models ignore it.  There is no jaw prior. */
} BfFrames;

int         bf_abi_version(void);
int         bf_sizeof(int which);                        /* 0 BfVSet, 1 BfModel, 2 BfFrames, 3 BfGrid, 4 BfSmpld, 5 BfMask: layout check for FFI bindings */
const char* bf_last_error(void);
int         bf_check_device(void);                       /* BF_OK iff current device is sm_100 */

/* theta -> pf, A, Jtr, full_pose, yaw */
int bf_pose_forward(const BfModel* m, const BfFrames* f, void* stream);
/* blend shapes only (tensor-core path): pf @ Bm -> vposed; the fused per-frame kernel of the fit skins the live vertices itself */
int bf_blend_forward(const BfModel* m, const BfFrames* f, int use_full, void* stream);
/* blend shapes + skinning over a vertex set (use_full != 0: all vertices) -> verts, vposed */
int bf_skin_forward(const BfModel* m, const BfFrames* f, int use_full, void* stream);
/* model-space output joints [B,K_out,3] from Jtr / verts */
int bf_joints_forward(const BfModel* m, const BfFrames* f, int use_full, void* stream);
/* joints gradient + optional dense dverts -> dJtr, dverts (gather by target) */
int bf_joints_backward(const BfModel* m, const BfFrames* f, int use_full, int accumulate_dverts, void* stream);
/* keypoint data term: loss, d/d(theta[0:4]), dJtr, dverts */
int bf_keypoint_loss(const BfModel* m, const BfFrames* f, int use_full, void* stream);
/* active set only: keypoint term + its backward down to dvp, dA, dJtr, grad[0:4] in one kernel per frame
 * (= bf_keypoint_loss + parts 1|2 of bf_skin_backward without the d(verts) round trip through HBM) */
int bf_frame_loss_backward(const BfModel* m, const BfFrames* f, void* stream);
/* dverts -> dvp, dA, dpf */
int bf_skin_backward(const BfModel* m, const BfFrames* f, int use_full, void* stream);
/* the same, one kernel at a time (profiling): parts bit0 dvp, bit1 dA, bit2 blend-backward GEMM */
int bf_skin_backward_parts(const BfModel* m, const BfFrames* f, int use_full, int parts, void* stream);
/* temporal smoothness between consecutive frames of a sequence (NOT in the reference; BASELINE config 4):
 *   L = w_temporal * sum_f |p_f - p_{f-1}|^2,  p = (transl, global_orient, body_pose);
 * frame f is charged the edge (f-1, f); tgrad[f] = 2 w (2 p_f - p_{f-1} - p_{f+1}) with the shard's outer
 * neighbours taken from halo_prev / halo_next (exchanged between ranks before every iteration) */
int bf_temporal_prior(const BfModel* m, const BfFrames* f, void* stream);
/* one fit iteration with explicit control: with_forward = run the pose forward first, fuse_next = let the pose
 * backward also run the next iteration's pose forward (bf_fit_step = (1, 0)) */
int bf_fit_iteration(const BfModel* m, const BfFrames* f, int with_forward, int fuse_next, void* stream);
/* GMM pose prior of every frame -> gmm_grad, gmm_loss */
int bf_gmm_prior(const BfModel* m, const BfFrames* f, void* stream);
/* dA, dJtr, dpf -> grad (theta[4:]); flags: 1 = add priors (value + grad; needs bf_gmm_prior first), 2 = Adam step,
 * 4 = keep grad[0:4] from the loss kernel, 8 = also run the next iteration's pose forward on the updated theta */
int bf_pose_backward(const BfModel* m, const BfFrames* f, int flags, void* stream);

/* LBS operator: pose_forward + skin_forward(full) + joints_forward */
int bf_lbs_forward(const BfModel* m, const BfFrames* f, void* stream);
/* LBS operator backward: (dverts, djoints) -> grad wrt theta */
int bf_lbs_backward(const BfModel* m, const BfFrames* f, void* stream);
/* one SMPLify iteration on the active vertex set; f->iter is the 0-based iteration */
int bf_fit_step(const BfModel* m, const BfFrames* f, void* stream);
/* n iterations starting at f->iter; if dense_last != 0 the last iteration's forward also
 * materialises all vertices into f_full->verts (the reference returns the vertices of the
 * last forward pass, smplify/smplify.py:217) */
int bf_fit_run(const BfModel* m, const BfFrames* f, int n_iters, void* stream);


/* ---- model and frame buffers for hosts that do not run Python ---------------------------------------------------------
 * The body-model tables (BfModel: ~60 device arrays derived from v_template / shapedirs / posedirs / J_regressor / weights /
 * landmark tables / the GMM prior; reference: models/smpl.py:56-66, smplify/smplify.py:46-80, smplify/prior.py:127-174) are
 * built from the raw model arrays by bf_model_create (C++, no Python), or prepared once by the Python tool
 * (bodyfitting_b200.model.PreparedModel(...).save_blob(path)) and loaded by bf_model_load with one upload; bf_model_destroy
 * frees them.  bf_workspace_bytes / bf_frames_bind size and carve ONE caller-owned, 256-byte aligned
 * device workspace into the BfFrames buffers of a B-frame batch (opts: 1 = all-vertex set, 2 = backward / optimiser buffers,
 * 8 = temporal term; n_trace = rows of the optional per-iteration loss trace), zero it and fill in the reference's
 * hyper-parameters.  These are the only calls besides bf_halo_* that allocate or synchronise. */
/* Raw model arrays, exactly as the reference's model files hold them (SMPL_*.pkl / SMPLX_*.npz keys of the same names; dense,
 * row-major, float32 / int32).  Optional members may be NULL / 0.  bf_model_create builds every derived table on the host (C++,
 * bodyfitting_b200/csrc/bf_model_build.cuh -- the same algorithm as the Python builder, compared table by table in
 * tests/test_host.py) and uploads it; bf_model_build_blob stops before the upload and hands back the image bf_model_load_memory
 * accepts (free it with bf_blob_free).  Reference: models/smpl.py:56-66, smplify/smplify.py:46-80, smplify/prior.py:127-174. */
typedef struct BfModelDesc {
    const float*   v_template;              /* [V,3] */
    const float*   shapedirs;               /* [V,3,n_shape_dirs]; official SMPL-X files: 300 shape + 100 expression directions */
    const float*   posedirs;                /* [V,3,(J-1)*9] */
    const float*   J_regressor;             /* [J,V] dense */
    const float*   weights;                 /* [V,J] skinning weights */
    const int32_t* parents;                 /* [J] kintree_table[0]; parents[0] is ignored */
    const int32_t* faces;                   /* [F,3] (SMPL-X: needed for the landmark tables) */
    const float*   hands_meanl;             /* [45]   SMPL-X */
    const float*   hands_meanr;             /* [45] */
    const float*   hands_componentsl;       /* [>=num_pca_comps,45]: the first num_pca_comps PCA rows are used (unused for
                                               axis-angle hands) */
    const float*   hands_componentsr;
    const int32_t* lmk_faces_idx;           /* [n_lmk]   SMPL-X static face landmarks */
    const float*   lmk_bary_coords;         /* [n_lmk,3] */
    const int32_t* dynamic_lmk_faces_idx;   /* [n_dyn_rows,n_dyn]   SMPL-X contour landmarks per yaw row (79 x 17) */
    const float*   dynamic_lmk_bary_coords; /* [n_dyn_rows,n_dyn,3] */
    const int32_t* extra_vids;              /* [n_extra_vids] vertex-picked joints, or NULL = smplx.vertex_ids (SURVEY Appendix B) */
    const float*   J_regressor_extra;       /* [n_regressor_extra,V] SMPL wrapper's extra joints (models/smpl.py:62-65), or NULL */
    const float*   kid_template;            /* [V,3] SMIL template (age='kid', SMPL only), or NULL */
    const float*   gmm_means;               /* [n_gmm,69]   pose prior (smplify/prior.py:127), or NULL */
    const float*   gmm_covars;              /* [n_gmm,69,69] */
    const float*   gmm_weights;             /* [n_gmm] */
    /* num_betas >= 1 (the kid template adds one more); num_expression >= 0 (SMPL-X only; 0 = no expression directions).
     * The model is rejected when betas + expression exceed 20 or its theta row without the face block exceeds 100 entries
     * (NP above).  face_params != 0 (SMPL-X only): theta also carries the jaw pose and the expression coefficients, which the
     * fit then optimises; 0 keeps them at zero, as the reference does.
     * Hands (SMPL-X only, smplx.create's options): num_pca_comps = hand PCA components per hand, 1..45 (0 means 6, the
     * reference's configuration); the 100-entry limit above is computed with 6.  hand_axis_angle != 0 (smplx use_pca=False):
     * theta carries 45 axis-angle entries per hand and num_pca_comps is only range-checked.  flat_hand_mean != 0: the hand
     * mean is not added to the full pose.  Both flags follow the 16 int32 members of ABI 20, so a host that zero-initialises
     * the struct and fills those keeps its meaning. */
    int32_t is_smplx, V, J, F, n_shape_dirs, num_betas, num_expression, n_lmk, n_dyn_rows, n_dyn, n_extra_vids, n_regressor_extra,
            n_gmm, tensor_cores, face_params, num_pca_comps;
    uint32_t hand_axis_angle, flat_hand_mean;
} BfModelDesc;
int     bf_model_create(const BfModelDesc* desc, BfModel** out);
int     bf_model_build_blob(const BfModelDesc* desc, void** blob, int64_t* nbytes);
void    bf_blob_free(void* blob);
int     bf_model_load(const char* path, BfModel** out);
int     bf_model_load_memory(const void* blob, int64_t nbytes, BfModel** out);
int     bf_model_destroy(BfModel* m);
int64_t bf_workspace_bytes(const BfModel* m, int B, int Nv, int opts, int n_trace);
int     bf_frames_bind(const BfModel* m, int B, int Nv, int opts, int n_trace, void* workspace, int64_t bytes, BfFrames* out,
                       void* stream);

/* every kernel node of a captured cudaGraph_t gets launch priority `priority` (stream priority scale); returns the number of
 * nodes changed or a negative code.  For hosts that replay several part graphs concurrently and want them to finish in order. */
int bf_graph_set_kernel_priority(void* cuda_graph, int priority);

/* ---- input packing (so that no host-framework arithmetic sits on the path) ---------------------------------
 * detections [B,Nv,K,3] (x, y, conf) in the caller's layout -> kp [B,K,Nv,3] (x, y, effective weight): conf^2 for the body,
 * the group's sum of conf^2 for SMPL-X hands / face (smplify/loss.py:134 with :168,:173,:179).  Nv: 1 to 64 views
 * (BfFrames.Nv); one frame's K * Nv detections are staged in shared memory (at most 104,704 bytes: SMPL-X, 64 views) */
int bf_pack_keypoints(const float* kp_raw, float* kp_packed, int B, int Nv, int K, int hand_face, const int32_t* src_index,
                      void* stream);
/* network output -> initial theta rows (smplify/smplify.py:103-128): transl 0, scale 1, global_orient / body_pose from
 * poses[b, 0:3+nbody] (row stride ld_poses), betas[b, 0:10], eye / hand (and face) parameters 0.  betas always has 10 columns: a model
 * with more betas (num_betas > 10, the kid model) starts the betas beyond the 10th at 0, one with fewer takes the first
 * num_betas columns.  To start them elsewhere, write the theta rows directly (layout at the top of this file). */
int bf_init_theta(const BfModel* m, const float* poses, int ld_poses, const float* betas, float* theta, int B,
                  const int32_t* src_index, void* stream);
/* src_index (both calls above, optional): packed frame b is the caller's frame src_index[b] -- a batch whose frames are
 * independent fits may be processed in any order (the host sorts it by contour row so that a 128-frame tile of the blend
 * GEMMs touches few 16-vertex blocks, BfFrames.blk_mask); bf_scatter_rows puts result rows back: dst[index[r]] = src[r] */
int bf_scatter_rows(const float* src, const int32_t* index, float* dst, int rows, int cols, void* stream);

/* ---- NVLink halo of the temporal term (BASELINE config 4; the reference has no multi-GPU path) -----------------
 * One buffer per rank (bf_halo_bytes() bytes of cudaMalloc'ed memory, exported as a CUDA IPC handle of
 * bf_halo_handle_bytes() bytes); neighbours map it with bf_halo_open and the optimiser kernel stores its boundary rows
 * straight into it.  BfFrames.halo_buf / halo_peer_prev / halo_peer_next / halo_iters switch it on; bf_halo_begin starts
 * a run (publishes the initial boundary rows).  The only calls of this library that allocate / synchronise. */
int bf_halo_bytes(void);
int bf_halo_handle_bytes(void);
int bf_halo_alloc(void** buf, void* ipc_handle_out);
int bf_halo_open(const void* ipc_handle, void** peer_buf);
int bf_halo_close(void* peer_buf);
int bf_halo_free(void* buf);
int bf_halo_begin(const BfModel* m, const BfFrames* f, int n_iters, void* stream);

#ifdef __cplusplus
}
#endif
#endif
