"""ctypes binding of the C-ABI shared library ``libbodyfit_b200.so``.

The library holds every kernel of the product path.  There is no CPU fallback and no
alternative backend: if the shared object is missing, or the current device is not
sm_100, importing / calling fails loudly.  Struct layouts mirror
``include/bodyfit_b200.h`` field by field.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('BODYFIT_LIB') or os.path.join(_HERE, 'libbodyfit_b200.so')   # BODYFIT_LIB: A/B builds of the same ABI
ABI_VERSION = 21
F_WORLD = 1
F_TC = 2
F_SKIN_FUSED = 4

_fp = C.c_void_p
_i32 = C.c_int32


class BfVSet(C.Structure):
    _fields_ = [(n, _fp) for n in (
        'Bm', 'ell_j', 'ell_w', 'jv_ptr', 'jv_vid', 'jv_w', 'kj_kind', 'kj_src', 'kj_w',
        'dyn_src', 'dyn_w', 'tg_ptr', 'tg_k', 'tg_a', 'tg_w', 'xr_ptr', 'xr_vid', 'xr_w', 'Bt_hi', 'Bt_lo', 'Bm_hi', 'Bm_lo', 'dyn_k', 'jv_nz',
        'lv_n', 'lv_vid', 'lt_ptr', 'lt_k', 'lt_w', 'lj_ptr', 'lj_vid', 'lj_w', 'lv_blk')] + \
        [(n, _i32) for n in ('n', 'n_pad', 'ldn', 'nnz', 'K_out', 'n_dyn', 'n_extra', 'n_nz', 'lmax', 'n_rows')]


class BfModelDesc(C.Structure):
    """Raw model arrays for bf_model_create / bf_model_build_blob (include/bodyfit_b200.h)."""
    _fields_ = [(n, _fp) for n in (
        'v_template', 'shapedirs', 'posedirs', 'J_regressor', 'weights', 'parents', 'faces', 'hands_meanl', 'hands_meanr',
        'hands_componentsl', 'hands_componentsr', 'lmk_faces_idx', 'lmk_bary_coords', 'dynamic_lmk_faces_idx',
        'dynamic_lmk_bary_coords', 'extra_vids', 'J_regressor_extra', 'kid_template', 'gmm_means', 'gmm_covars', 'gmm_weights')] + \
        [(n, _i32) for n in ('is_smplx', 'V', 'J', 'F', 'n_shape_dirs', 'num_betas', 'num_expression', 'n_lmk', 'n_dyn_rows', 'n_dyn',
                             'n_extra_vids', 'n_regressor_extra', 'n_gmm', 'tensor_cores', 'face_params', 'num_pca_comps')] + \
        [(n, C.c_uint32) for n in ('hand_axis_angle', 'flat_hand_mean')]


class BfModel(C.Structure):
    _fields_ = [(n, _fp) for n in (
        'parents', 'depth', 'lvl_ptr', 'lvl_j', 'child_ptr', 'child_idx', 'Jt', 'Jd', 'pose_mean', 'hand_l', 'hand_r',
        'gmm_mean', 'gmm_psym', 'gmm_logw', 'gmm_bt_hi', 'gmm_bt_lo')] + \
        [('full', BfVSet), ('act', BfVSet)] + \
        [(n, _i32) for n in ('J', 'P', 'NS', 'NB', 'Kp', 'NP', 'is_smplx', 'max_depth', 'K_used',
                             'n_gmm', 'face', 'n_hand')]


class BfFrames(C.Structure):
    _fields_ = [(n, _fp) for n in (
        'theta', 'grad', 'adam_m', 'adam_v', 'pf', 'dpf', 'A', 'dA', 'Jtr', 'dJtr', 'full_pose', 'yaw',
        'verts', 'vposed', 'dverts', 'dvp', 'joints', 'djoints', 'kp', 'cams', 'loss', 'loss_terms', 'trace',
        'pf_hi', 'pf_lo', 'dvp_hi', 'dvp_lo', 'gmm_grad', 'gmm_loss', 'tgrad', 'tloss', 'halo_prev', 'halo_next', 'halo_buf', 'halo_peer_prev', 'halo_peer_next', 'fwd_state', 'gmm_ws', 'ws', 'blk_mask', 'dpf2', 'frame_index')] + [('ws_floats', C.c_int64)] + \
        [(n, C.c_double) for n in ('lr_ts', 'lr', 'beta1', 'beta2', 'eps')] + \
        [(n, _i32) for n in ('B', 'Nv', 'ld_v', 'iter', 'flags', 'halo_iters')] + \
        [(n, C.c_float) for n in ('imsize', 'constant_scale', 'sigma', 'w_pose', 'w_angle', 'w_shape', 'w_temporal', 'w_expr')]


class BfGrid(C.Structure):
    _fields_ = [(n, _fp) for n in ('verts', 'faces', 'cell_start', 'cell_tris')] + \
        [('min', C.c_float * 3), ('step', C.c_float), ('dim', _i32 * 3), ('ncell', _i32), ('Ns', _i32), ('Fs', _i32)]


class BfSmpld(C.Structure):
    _fields_ = [(n, _fp) for n in ('base', 'disp', 'adam_m', 'adam_v', 'faces', 'vf_ptr', 'vf_face', 'scan_fn', 'P', 'C',
                                   'near_faces', 'nhat', 'nlen', 'm', 'Nlen', 'dN', 'dcorner', 'partial', 'totals', 'grad',
                                   'trace')] + \
        [(n, C.c_double) for n in ('lr', 'beta1', 'beta2', 'eps')] + \
        [('reg_scale', C.c_float), ('V', _i32), ('F', _i32), ('iter', _i32)]


class BfMask(C.Structure):
    _fields_ = [(n, _fp) for n in ('masks', 'cams', 'contour', 'cptr', 'cown', 'uv', 'near_q', 'cdist', 'cw', 'dPw', 'part',
                                   'mask_loss')] + \
        [(n, _i32) for n in ('Nm', 'H', 'W', 'Nq', 'stride', 'total')] + [('imsize', C.c_float), ('epsilon', C.c_float)]


class BodyfitError(RuntimeError):
    pass


_lib = None


def lib():
    """Load (once) and return the shared library; raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BodyfitError(
            'CUDA extension %s is missing: run `python -c "import __graft_entry__ as g; g.build()"` '
            '(there is no CPU fallback)' % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    L.bf_abi_version.restype = C.c_int
    L.bf_last_error.restype = C.c_char_p
    L.bf_check_device.restype = C.c_int
    L.bf_sizeof.restype = C.c_int
    L.bf_sizeof.argtypes = [C.c_int]
    if L.bf_abi_version() != ABI_VERSION:
        raise BodyfitError('ABI mismatch: library %d, binding %d -- rebuild' % (L.bf_abi_version(), ABI_VERSION))
    for i, st in enumerate((BfVSet, BfModel, BfFrames, BfGrid, BfSmpld, BfMask)):
        if L.bf_sizeof(i) != C.sizeof(st):
            raise BodyfitError('struct layout mismatch for %s: C %d, ctypes %d' % (st.__name__, L.bf_sizeof(i), C.sizeof(st)))
    pm, pf, vp, ci = C.POINTER(BfModel), C.POINTER(BfFrames), C.c_void_p, C.c_int
    for name, extra in (('bf_pose_forward', []), ('bf_skin_forward', [ci]), ('bf_blend_forward', [ci]), ('bf_joints_forward', [ci]),
                        ('bf_joints_backward', [ci, ci]), ('bf_keypoint_loss', [ci]), ('bf_skin_backward', [ci]), ('bf_skin_backward_parts', [ci, ci]),
                        ('bf_pose_backward', [ci]), ('bf_gmm_prior', []), ('bf_temporal_prior', []), ('bf_fit_iteration', [ci, ci]), ('bf_frame_loss_backward', []), ('bf_lbs_forward', []), ('bf_lbs_backward', []),
                        ('bf_fit_step', []), ('bf_fit_run', [ci]), ('bf_halo_begin', [ci])):
        fn = getattr(L, name)
        fn.restype = C.c_int
        fn.argtypes = [pm, pf] + extra + [vp]
    fp, i32, i64, fl = C.c_void_p, C.c_int, C.c_int64, C.c_float
    ops = {
        'bf_op_project': [fp, fp, fp, fp, fp, i32, i32, i32, vp],
        'bf_op_project_backward': [fp, fp, fp, fp, fp, fp, i32, i32, i32, vp],
        'bf_op_gmof': [fp, fp, fl, i64, vp],
        'bf_op_gmof_backward': [fp, fp, fp, fl, i64, vp],
        'bf_op_reprojection': [fp, fp, fp, fl, fl, i32, fp, fp, vp],
        'bf_op_keypoints_world': [fp, fp, fp, i32, i32, i32, fl, fl, fp, fp, vp],
        'bf_op_angle_prior': [fp, i32, i32, fp, fp, vp],
        'bf_op_gmm_pose': [pm, fp, i32, i32, i32, fl, fp, fp, vp],
    }
    ops.update({
        'bf_pack_keypoints': [fp, fp, i32, i32, i32, i32, fp, vp],
        'bf_init_theta': [pm, fp, i32, fp, fp, i32, fp, vp],
        'bf_scatter_rows': [fp, fp, fp, i32, i32, vp],
        'bf_halo_alloc': [C.POINTER(C.c_void_p), fp], 'bf_halo_open': [fp, C.POINTER(C.c_void_p)],
        'bf_halo_close': [fp], 'bf_halo_free': [fp],
    })
    L.bf_model_load.restype = C.c_int
    L.bf_model_load.argtypes = [C.c_char_p, C.POINTER(pm)]
    L.bf_model_load_memory.restype = C.c_int
    L.bf_model_load_memory.argtypes = [C.c_void_p, C.c_int64, C.POINTER(pm)]
    L.bf_model_destroy.restype = C.c_int
    L.bf_model_destroy.argtypes = [pm]
    L.bf_model_create.restype = C.c_int
    L.bf_model_create.argtypes = [C.POINTER(BfModelDesc), C.POINTER(pm)]
    L.bf_model_build_blob.restype = C.c_int
    L.bf_model_build_blob.argtypes = [C.POINTER(BfModelDesc), C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]
    L.bf_blob_free.restype = None
    L.bf_blob_free.argtypes = [C.c_void_p]
    L.bf_workspace_bytes.restype = C.c_int64
    L.bf_workspace_bytes.argtypes = [pm, i32, i32, i32, i32]
    L.bf_frames_bind.restype = C.c_int
    L.bf_frames_bind.argtypes = [pm, i32, i32, i32, i32, C.c_void_p, C.c_int64, pf, vp]
    L.bf_graph_set_kernel_priority.restype = C.c_int
    L.bf_graph_set_kernel_priority.argtypes = [C.c_void_p, C.c_int]
    for name in ('bf_halo_bytes', 'bf_halo_handle_bytes'):
        getattr(L, name).restype = C.c_int
        getattr(L, name).argtypes = []
    pg, ps = C.POINTER(BfGrid), C.POINTER(BfSmpld)
    ops.update({
        'bf_grid_count': [pg, fp, vp], 'bf_grid_fill': [pg, fp, vp],
        'bf_grid_nearest': [pg, fp, i32, fp, fp, fp, vp],
        'bf_grid_barycentric': [pg, fp, fp, i32, fp, vp], 'bf_grid_nearest_backward': [pg, fp, fp, i32, fp, vp],
        'bf_grid_inside': [pg, fp, i32, fp, vp], 'bf_grid_intersects_any': [pg, fp, fp, i32, fp, vp],
        'bf_smpld_step': [pg, ps, vp], 'bf_smpld_run': [pg, ps, i32, vp],
        'bf_pc_loss': [pg, pm, pf, fl, fl, fp, fp, fp, fp, vp],
        'bf_mask_loss': [pm, pf, C.POINTER(BfMask), fl, vp],
        'bf_op_pc_loss': [fp, fp, i64, fp, fp, vp],
        'bf_op_regress_joints': [fp, fp, fp, fp, i32, i32, i32, fp, vp],
        'bf_op_normal_loss': [fp, fp, fp, i32, fp, fp, vp],
        'bf_op_laplacian': [fp, fp, fp, fp, i32, i32, fp, fp, vp],
        'bf_op_vertex_normals': [fp, fp, fp, fp, i32, i32, fp, fp, fp, fp, vp],
        'bf_op_vertex_normals_backward': [fp, fp, fp, fp, i32, i32, fp, fp, fp, fp, fp, fp, fp, fp, vp],
        'bf_op_mask_loss': [fp, i32, i32, C.POINTER(BfMask), fp, fp, fp, vp],
    })
    for name, at in ops.items():
        fn = getattr(L, name)
        fn.restype = C.c_int
        fn.argtypes = at
    _lib = L
    return L


EXPORTED = ['bf_abi_version', 'bf_sizeof', 'bf_last_error', 'bf_check_device', 'bf_pose_forward', 'bf_skin_forward', 'bf_blend_forward',
            'bf_joints_forward', 'bf_joints_backward', 'bf_keypoint_loss', 'bf_skin_backward', 'bf_skin_backward_parts',
            'bf_pose_backward', 'bf_gmm_prior', 'bf_temporal_prior', 'bf_fit_iteration', 'bf_frame_loss_backward', 'bf_lbs_forward', 'bf_lbs_backward', 'bf_fit_step', 'bf_fit_run',
            'bf_pack_keypoints', 'bf_init_theta', 'bf_scatter_rows', 'bf_halo_bytes', 'bf_halo_handle_bytes', 'bf_halo_alloc', 'bf_halo_open',
            'bf_halo_close', 'bf_halo_free', 'bf_halo_begin', 'bf_model_load', 'bf_model_load_memory', 'bf_model_destroy',
            'bf_model_create', 'bf_model_build_blob', 'bf_blob_free',
            'bf_workspace_bytes', 'bf_frames_bind', 'bf_graph_set_kernel_priority']


EXPORTED_GRID = ['bf_grid_count', 'bf_grid_fill', 'bf_grid_nearest', 'bf_grid_barycentric', 'bf_grid_nearest_backward', 'bf_grid_inside', 'bf_grid_intersects_any', 'bf_smpld_step', 'bf_smpld_run', 'bf_pc_loss']
EXPORTED_MASK = ['bf_mask_loss']
EXPORTED_OPS = ['bf_op_project', 'bf_op_project_backward', 'bf_op_gmof', 'bf_op_gmof_backward', 'bf_op_reprojection',
                'bf_op_keypoints_world', 'bf_op_angle_prior', 'bf_op_gmm_pose', 'bf_op_pc_loss', 'bf_op_normal_loss',
                'bf_op_laplacian', 'bf_op_vertex_normals', 'bf_op_vertex_normals_backward', 'bf_op_mask_loss', 'bf_op_regress_joints']


def last_error():
    msg = lib().bf_last_error()
    return msg.decode() if msg else ''


def check(rc, what=''):
    if rc != 0:
        msg = lib().bf_last_error()
        raise BodyfitError('%s failed (%d): %s' % (what, rc, msg.decode() if msg else ''))


def require_device():
    """Raise unless the current CUDA device is a B200-class (sm_100) GPU."""
    import torch
    if not torch.cuda.is_available():
        raise BodyfitError('no CUDA device: bodyfitting_b200 has no CPU path')
    check(lib().bf_check_device(), 'bf_check_device')
