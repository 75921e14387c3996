"""ctypes binding of libmgconv.so -- the C ABI declared in include/mgconv.h.

This is the Python twin of lua/mgconv_ffi.lua (LuaJIT `ffi.cdef` + `ffi.load`): the same
entry points with the same plain-C signatures.  There is NO fallback: if the shared library is
missing the import raises, and every non-zero mg_status becomes an exception carrying
mg_last_error() -- the same behaviour as a Torch7 module raising a Lua error().
"""
import ctypes as C
import os

MG_MAX_SEG = 6
MG_MAX_SRC = 8
MG_F32, MG_BF16 = 0, 1
MG_SEG_SAME, MG_SEG_POOL, MG_SEG_UP, MG_SRC_POOL3 = 0, 1, 2, 3
MG_IMPL_AUTO, MG_IMPL_SIMT, MG_IMPL_TCGEN05 = 0, 1, 2
MG_TUNE_HALO_SUBTILES, MG_TUNE_PERSISTENT, MG_TUNE_STEM_FUSED_STATS = 0, 1, 2
MG_ALGO_AUTO, MG_ALGO_TILE128, MG_ALGO_TILE256, MG_ALGO_RESIDENT, MG_ALGO_TILE128_DEEP, MG_ALGO_TILE256_DEEP, MG_ALGO_TILE128_MID = 0, 1, 2, 3, 4, 5, 6
MG_ALGO_PAIR128, MG_ALGO_PAIR256, MG_ALGO_RESIDENT_PAIR = 7, 8, 9

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MGCONV_LIB", os.path.join(_HERE, "libmgconv.so"))


class MGError(RuntimeError):
    pass


class mg_grid(C.Structure):
    _fields_ = [("data", C.c_void_p), ("scale", C.c_void_p), ("shift", C.c_void_p), ("relu", C.c_int32),
                ("N", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("C", C.c_int32), ("Cp", C.c_int32)]


class mg_conv_desc(C.Structure):
    _fields_ = [("n_seg", C.c_int32), ("seg", mg_grid * MG_MAX_SEG), ("seg_mode", C.c_int32 * MG_MAX_SEG),
                ("ksize", C.c_int32), ("stride", C.c_int32), ("pad", C.c_int32), ("Cout", C.c_int32),
                ("H", C.c_int32), ("W", C.c_int32), ("algo_fwd", C.c_int32), ("algo_bwd_data", C.c_int32)]


class mg_grad_src(C.Structure):
    _fields_ = [("g", mg_grid), ("c_offset", C.c_int32), ("mode", C.c_int32), ("aux", C.c_void_p)]


MG_STAGE_MAX_GRIDS = 4


class mg_stage_desc(C.Structure):
    _fields_ = [("n_scales", C.c_int32), ("C_in", C.c_int32 * MG_STAGE_MAX_GRIDS), ("C_out", C.c_int32 * MG_STAGE_MAX_GRIDS),
                ("H", C.c_int32 * MG_STAGE_MAX_GRIDS), ("W", C.c_int32 * MG_STAGE_MAX_GRIDS), ("ksize", C.c_int32 * MG_STAGE_MAX_GRIDS),
                ("residual", C.c_int32), ("no_final_relu", C.c_int32), ("eps", C.c_float), ("momentum", C.c_float)]


class mg_stage_params(C.Structure):
    _fields_ = [(name, C.c_void_p * (2 * MG_STAGE_MAX_GRIDS)) for name in
                ("conv_w", "conv_b", "bn_g", "bn_b", "bn_rm", "bn_rv", "conv_gw", "conv_gb", "bn_gg", "bn_gb")]


class mg_bn_fused(C.Structure):
    _fields_ = [("sums", C.c_void_p), ("count", C.c_int64), ("gamma", C.c_void_p), ("beta", C.c_void_p),
                ("running_mean", C.c_void_p), ("running_var", C.c_void_p), ("eps", C.c_float), ("momentum", C.c_float),
                ("training", C.c_int32), ("save_mean", C.c_void_p), ("save_invstd", C.c_void_p)]


class mg_dropout(C.Structure):
    _fields_ = [("p", C.c_float), ("op", C.c_uint32), ("rank", C.c_uint32), ("seed", C.c_uint64), ("step", C.c_void_p)]


def _load():
    if not os.path.exists(LIB_PATH):
        raise MGError(
            f"{LIB_PATH} not found: build it with `make -C multigrid-neural-architectures_b200/csrc` "
            "(or __graft_entry__.build()); there is no CPU / PyTorch fallback for the multigrid hot path")
    return C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)


lib = _load()

_P, _I, _I64, _F, _SZ = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_size_t
_G = C.POINTER(mg_grid)
_D = C.POINTER(mg_conv_desc)

# name -> (restype, argtypes); mirrors include/mgconv.h declaration by declaration
SIGNATURES = {
    "mg_ctx_create": (_I, [_I, _P, _I, C.POINTER(_P)]),
    "mg_ctx_destroy": (_I, [_P]),
    "mg_ctx_set_stream": (_I, [_P, _P]),
    "mg_ctx_set_impl": (_I, [_P, _I]),
    "mg_ctx_sync": (_I, [_P]),
    "mg_ctx_lane": (_I, [_P, _I]),
    "mg_ctx_event_record": (_I, [_P, _I]),
    "mg_ctx_event_wait": (_I, [_P, _I]),
    "mg_ctx_set_tuning": (_I, [_P, _I, _I]),
    "mg_last_error": (C.c_char_p, [_P]),
    "mg_version": (_I, []),
    "mg_ctx_launch_count": (_I, [_P, C.POINTER(_I64)]),
    "mg_ctx_tc_launch_count": (_I, [_P, C.POINTER(_I64)]),
    "mg_ctx_profile": (_I, [_P, _I]),
    "mg_ctx_profile_read": (_I, [_P, C.POINTER(C.c_double), C.POINTER(_I64)]),
    "mg_import_nchw": (_I, [_P, _P, _G]),
    "mg_export_nchw": (_I, [_P, _G, _P]),
    "mg_crop_flip_normalize": (_I, [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P]),
    "mg_conv_packed_bytes": (_SZ, [_D, _I]),
    "mg_conv_pack_weights": (_I, [_P, _D, _P, _P, _I]),
    "mg_conv_forward": (_I, [_P, _D, _P, _P, _P, _G, _P]),
    "mg_bn_finalize": (_I, [_P, _P, _I64, C.c_int32, C.c_int32, _P, _P, _P, _P, _F, _F, _I, _P, _P, _P, _P]),
    "mg_residual_forward": (_I, [_P, _G, _G, _I, _G, _G]),
    "mg_bn_residual_forward": (_I, [_P, _G, C.POINTER(mg_bn_fused), _G, _I, _G, _G]),
    "mg_conv_pack_weights_batched": (_I, [_P, C.c_int32, C.POINTER(_D), C.POINTER(_P), C.POINTER(_P), C.POINTER(C.c_int32)]),
    "mg_bn_stats": (_I, [_P, _G, _P]),
    "mg_memset_zero": (_I, [_P, _P, _SZ]),
    "mg_pool_forward": (_I, [_P, _G, _G, C.c_int32, _P]),
    "mg_copy_channels": (_I, [_P, _G, _G, C.c_int32]),
    "mg_avgpool_forward": (_I, [_P, _G, C.c_int32, _G]),
    "mg_im2col": (_I, [_P, _G, C.c_int32, C.c_int32, C.c_int32, _G]),
    "mg_pool3s2_forward": (_I, [_P, _G, _G, _P]),
    "mg_bn_relu_pool3_forward": (_I, [_P, _G, C.POINTER(mg_bn_fused), _G, _P]),
    "mg_global_avgpool_forward": (_I, [_P, _G, _G]),
    "mg_global_avgpool_backward": (_I, [_P, _G, _G]),
    "mg_upconv2x2_forward": (_I, [_P, _G, _P, _P, _G, _P]),
    "mg_upconv2x2_backward": (_I, [_P, _G, _P, _G, _G, _P, _P, _F]),
    "mg_dropout_forward": (_I, [_P, C.POINTER(mg_dropout), C.c_int32, _G, C.POINTER(C.c_int32), _G]),
    "mg_dropout_backward": (_I, [_P, C.POINTER(mg_dropout), _G]),
    "mg_dropout_advance": (_I, [_P, _P]),
    "mg_grad_combine": (_I, [_P, _G, _I, _G, C.c_int32, C.POINTER(mg_grad_src), _G, _P]),
    "mg_bn_backward": (_I, [_P, _G, _G, _G, _P, _I64, _P, _P, _P, _P, _P, _F, _P, _P]),
    "mg_conv_backward_data": (_I, [_P, _D, _P, _P, _G, _G]),
    "mg_conv_backward_weight": (_I, [_P, _D, _G, _P, _P, _F]),
    "mg_nll_forward_backward": (_I, [_P, _G, _P, _P, _P, _G, _F]),
    "mg_logsoftmax_forward": (_I, [_P, _G, _P]),
    "mg_logsoftmax_backward": (_I, [_P, _P, _P, _G]),
    "mg_bce_forward_backward": (_I, [_P, _G, _P, _P, _P, _G, _F]),
    "mg_sigmoid_forward": (_I, [_P, _G, _P]),
    "mg_sigmoid_backward": (_I, [_P, _P, _P, _G]),
    "mg_nll_criterion": (_I, [_P, _P, _P, C.c_int32, C.c_int32, _P, _P, _F]),
    "mg_bce_criterion": (_I, [_P, _P, _P, _I64, _P, _P, _F]),
    "mg_sgd_step": (_I, [_P, _P, _P, _P, _I64, _F, _F, _F, _I]),
    "mg_plan_create": (_I, [_P, C.POINTER(mg_stage_desc), C.c_int32, C.POINTER(_P)]),
    "mg_plan_workspace_bytes": (_SZ, [_P]),
    "mg_plan_destroy": (_I, [_P]),
    "mg_stage_forward": (_I, [_P, _P, C.POINTER(_P), C.POINTER(mg_stage_params), C.POINTER(_P), _I]),
    "mg_stage_backward": (_I, [_P, _P, C.POINTER(_P), C.POINTER(mg_stage_params), C.POINTER(_P), _F]),
    "mg_comm_unique_id": (_I, [_P]),
    "mg_comm_init": (_I, [_P, _I, _I, _P]),
    "mg_comm_destroy": (_I, [_P]),
    "mg_comm_share": (_I, [_P, _P]),
    "mg_allreduce_launch": (_I, [_P, _P, _I64, _I]),
    "mg_allreduce_wait": (_I, [_P]),
    "mg_allreduce_inline": (_I, [_P, _P, _I64, _I]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)  # AttributeError here = the library does not export what the header declares
    _fn.restype = _res
    _fn.argtypes = _args


class Context:
    """mg_ctx wrapper: one per (device, thread) like the reference's per-GPU Lua states
    (multigpu.lua:94-98).  call('mg_xxx', ...) raises MGError on a non-zero status."""

    def __init__(self, device=0, stream=0, dtype=MG_BF16):
        h = _P()
        rc = lib.mg_ctx_create(int(device), _P(stream), int(dtype), C.byref(h))
        if rc != 0:
            raise MGError(f"mg_ctx_create(device={device}) failed with status {rc} "
                          "(3 = no CUDA device, 5 = not an sm_100 GPU); the multigrid hot path has no CPU fallback")
        self.h = h
        self.dtype = dtype
        self.device = device

    def call(self, name, *args):
        rc = getattr(lib, name)(self.h, *args)
        if rc != 0:
            raise MGError(f"{name}: status {rc}: {lib.mg_last_error(self.h).decode()}")

    def set_stream(self, stream):
        self.call("mg_ctx_set_stream", _P(stream))

    def set_impl(self, impl):
        self.call("mg_ctx_set_impl", int(impl))

    def set_tuning(self, knob, value):
        self.call("mg_ctx_set_tuning", int(knob), int(value))

    def sync(self):
        self.call("mg_ctx_sync")

    def launches(self):
        n = _I64(0)
        self.call("mg_ctx_launch_count", C.byref(n))
        return n.value

    def tc_launches(self):
        n = _I64(0)
        self.call("mg_ctx_tc_launch_count", C.byref(n))
        return n.value

    def profile_read(self):
        ms, n = C.c_double(0), _I64(0)
        self.call("mg_ctx_profile_read", C.byref(ms), C.byref(n))
        return {"conv_ms": ms.value, "conv_launches": n.value}

    def close(self):
        if self.h:
            lib.mg_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def ptr(t):
    """raw device pointer of a torch tensor (or None)"""
    return _P(None) if t is None else _P(t.data_ptr())
