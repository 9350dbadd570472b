"""ctypes binding of libpnce.so (include/pnce.h).  Fails loudly: no CPU or eager fallback."""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# PNCE_EXPERIMENTS=1 selects the experiment build (pnce_debug_* hooks, scratch/ scripts only), see build.py
LIB_PATH = os.path.join(HERE, "libpnce_exp.so" if os.environ.get("PNCE_EXPERIMENTS", "") not in ("", "0") else "libpnce.so")

PNCE_F32, PNCE_F16, PNCE_BF16 = 0, 1, 2
MATH_SIMT_F32, MATH_TC_BF16X3, MATH_TC_BF16 = 0, 1, 2
MAX_LAYERS = 8
MAX_PATCHES = 4096
MAX_CHANNELS = 1024
ABI_VERSION = 10
LAYOUT_NCHW, LAYOUT_NHWC = 0, 1

EXPORTS = [
    "pnce_abi_version", "pnce_status_string", "pnce_last_cuda_error", "pnce_workspace_bytes",
    "pnce_fwd", "pnce_bwd", "pnce_fwd_ex", "pnce_bwd_ex", "pnce_fwd_draw", "pnce_plan_ids_draw", "pnce_draw_ids", "pnce_plan_bytes", "pnce_plan_ids", "pnce_fwd_planned", "pnce_bwd_planned", "pnce_sample_fwd", "pnce_sample_bwd_workspace_bytes",
    "pnce_sample_bwd", "pnce_sample_multi_fwd", "pnce_sample_multi_bwd_workspace_bytes", "pnce_sample_multi_bwd",
    "pnce_rows_loss_workspace_bytes", "pnce_rows_loss_fwd_bwd", "pnce_rows_loss_multi_workspace_bytes", "pnce_rows_loss_multi_fwd_bwd",
    "pnce_selftest_umma", "pnce_comp_supported", "pnce_comp_alloc", "pnce_comp_free", "pnce_comp_is_compressed",
    "pnce_multi_chunk_elems", "pnce_multi_axpby", "pnce_amp_adam_scratch_floats", "pnce_amp_adam_step",
    "pnce_diffaug_scratch_floats", "pnce_diffaug", "pnce_hinge_fwd", "pnce_hinge_bwd",
    "pnce_netf_workspace_bytes", "pnce_netf_fwd", "pnce_netf_bwd",
    "pnce_head_fwd_ex", "pnce_head_bwd_ex", "pnce_head_workspace_bytes", "pnce_head_fwd", "pnce_head_bwd", "pnce_head_bwd_params", "pnce_head_bwd_dense",
    "pnce_mb_workspace_bytes", "pnce_mb_fwd", "pnce_rows_mb_workspace_bytes", "pnce_rows_mb_fwd_bwd",
    "pnce_mb_shard_workspace_bytes", "pnce_mb_shard_keys", "pnce_mb_shard_loss",
    "pnce_head_mb_workspace_bytes", "pnce_head_mb_fwd",
    "pnce_head_mb_shard_workspace_bytes", "pnce_head_mb_shard_keys", "pnce_head_mb_shard_loss",
    "pnce_rows_mb_shard_workspace_bytes", "pnce_rows_mb_shard_keys", "pnce_rows_mb_shard_loss",
]


class PnceLayer(ctypes.Structure):
    """struct pnce_layer (include/pnce.h)."""
    _fields_ = [
        ("src", ctypes.c_void_p), ("tgt", ctypes.c_void_p), ("dtgt", ctypes.c_void_p),
        ("ids", ctypes.c_void_p),
        ("C", ctypes.c_int32), ("H", ctypes.c_int32), ("W", ctypes.c_int32), ("P", ctypes.c_int32),
    ]


class PnceSample(ctypes.Structure):
    """struct pnce_sample (include/pnce.h)."""
    _fields_ = [("feat", ctypes.c_void_p), ("ids", ctypes.c_void_p), ("rows", ctypes.c_void_p),
                ("inv", ctypes.c_void_p), ("drows", ctypes.c_void_p), ("dfeat", ctypes.c_void_p),
                ("C", ctypes.c_int32), ("H", ctypes.c_int32), ("W", ctypes.c_int32), ("P", ctypes.c_int32)]


class PnceRows(ctypes.Structure):
    """struct pnce_rows (include/pnce.h)."""
    _fields_ = [("q", ctypes.c_void_p), ("k", ctypes.c_void_p), ("dq", ctypes.c_void_p),
                ("P", ctypes.c_int32), ("D", ctypes.c_int32)]


class PnceHead(ctypes.Structure):
    """struct pnce_head (include/pnce.h)."""
    _fields_ = [(n, ctypes.c_void_p) for n in ("w1", "b1", "w2", "b2", "dw1", "db1", "dw2", "db2")]


class PnceError(RuntimeError):
    pass


_lib = None


def load():
    """dlopen libpnce.so; building it first if the in-tree copy is missing or stale."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        from . import build as _build
        _build.build()
    lib = ctypes.CDLL(LIB_PATH)
    vp, i32, f32, sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_size_t
    lib.pnce_abi_version.restype = i32
    lib.pnce_status_string.restype = ctypes.c_char_p
    lib.pnce_status_string.argtypes = [i32]
    lib.pnce_last_cuda_error.restype = ctypes.c_char_p
    lib.pnce_workspace_bytes.argtypes = [ctypes.POINTER(PnceLayer), i32, i32, ctypes.POINTER(sz)]
    lib.pnce_fwd.argtypes = [ctypes.POINTER(PnceLayer), i32, i32, i32, f32, i32, vp, sz, vp, vp, vp]
    u64 = ctypes.c_ulonglong
    lib.pnce_fwd_draw.argtypes = [ctypes.POINTER(PnceLayer), i32, i32, i32, f32, i32, vp, sz, u64, u64, vp, vp, vp]
    lib.pnce_plan_ids_draw.argtypes = [ctypes.POINTER(PnceLayer), i32, u64, u64, vp, sz, vp]
    lib.pnce_draw_ids.argtypes = [ctypes.POINTER(PnceLayer), i32, u64, u64, vp]
    lib.pnce_bwd.argtypes = [ctypes.POINTER(PnceLayer), i32, i32, i32, i32, vp, sz, vp, vp]
    lib.pnce_fwd_ex.argtypes = [ctypes.POINTER(PnceLayer), i32, i32, i32, i32, f32, i32, vp, sz, vp, sz,
                                ctypes.POINTER(u64), vp, vp, vp]
    lib.pnce_bwd_ex.argtypes = [ctypes.POINTER(PnceLayer), i32, i32, i32, i32, i32, vp, sz, vp, sz, vp, vp]
    lib.pnce_plan_bytes.argtypes = [ctypes.POINTER(PnceLayer), i32, ctypes.POINTER(sz)]
    lib.pnce_plan_ids.argtypes = [ctypes.POINTER(PnceLayer), i32, vp, sz, vp]
    lib.pnce_fwd_planned.argtypes = [ctypes.POINTER(PnceLayer), i32, i32, i32, f32, i32, vp, sz, vp, sz, vp, vp, vp]
    lib.pnce_bwd_planned.argtypes = [ctypes.POINTER(PnceLayer), i32, i32, i32, i32, vp, sz, vp, sz, vp, vp]
    lib.pnce_sample_fwd.argtypes = [vp, i32, i32, i32, i32, i32, vp, i32, vp, vp, vp]
    lib.pnce_sample_bwd_workspace_bytes.argtypes = [i32, i32, i32, i32, i32, ctypes.POINTER(sz)]
    lib.pnce_sample_bwd.argtypes = [vp, vp, vp, i32, i32, i32, i32, i32, vp, i32, vp, sz, vp, vp]
    lib.pnce_sample_multi_fwd.argtypes = [ctypes.POINTER(PnceSample), i32, i32, i32, vp]
    lib.pnce_sample_multi_bwd_workspace_bytes.argtypes = [ctypes.POINTER(PnceSample), i32, i32, ctypes.POINTER(sz)]
    lib.pnce_sample_multi_bwd.argtypes = [ctypes.POINTER(PnceSample), i32, i32, i32, vp, sz, vp]
    lib.pnce_rows_loss_workspace_bytes.argtypes = [i32, i32, i32, ctypes.POINTER(sz)]
    lib.pnce_rows_loss_fwd_bwd.argtypes = [vp, vp, i32, i32, i32, f32, i32, vp, sz, vp, vp, vp, vp, vp]
    lib.pnce_rows_loss_multi_workspace_bytes.argtypes = [ctypes.POINTER(PnceRows), i32, i32, ctypes.POINTER(sz)]
    lib.pnce_rows_loss_multi_fwd_bwd.argtypes = [ctypes.POINTER(PnceRows), i32, i32, f32, i32, vp, sz, vp, vp, vp]
    lib.pnce_mb_workspace_bytes.argtypes = [ctypes.POINTER(PnceLayer), i32, i32, ctypes.POINTER(sz)]
    lib.pnce_mb_fwd.argtypes = lib.pnce_fwd_ex.argtypes
    lib.pnce_rows_mb_workspace_bytes.argtypes = lib.pnce_rows_loss_multi_workspace_bytes.argtypes
    lib.pnce_rows_mb_fwd_bwd.argtypes = lib.pnce_rows_loss_multi_fwd_bwd.argtypes
    lib.pnce_rows_mb_shard_workspace_bytes.argtypes = [ctypes.POINTER(PnceRows), i32, i32, i32, ctypes.POINTER(sz),
                                                       ctypes.POINTER(sz), ctypes.POINTER(sz)]
    lib.pnce_rows_mb_shard_keys.argtypes = [ctypes.POINTER(PnceRows), i32, i32, i32, i32, i32, vp, sz, vp]
    lib.pnce_rows_mb_shard_loss.argtypes = [ctypes.POINTER(PnceRows), i32, i32, i32, i32, f32, i32, vp, sz, vp, vp, vp]
    lib.pnce_mb_shard_workspace_bytes.argtypes = [ctypes.POINTER(PnceLayer), i32, i32, i32, ctypes.POINTER(sz),
                                                  ctypes.POINTER(sz), ctypes.POINTER(sz)]
    lib.pnce_mb_shard_keys.argtypes = [ctypes.POINTER(PnceLayer), i32, i32, i32, i32, i32, i32, i32, vp, sz, vp, sz,
                                       ctypes.POINTER(u64), vp]
    lib.pnce_mb_shard_loss.argtypes = [ctypes.POINTER(PnceLayer), i32, i32, i32, i32, i32, i32, f32, i32, vp, sz, vp, sz,
                                       vp, vp, vp]
    lib.pnce_head_workspace_bytes.argtypes = [ctypes.POINTER(PnceLayer), i32, i32, i32, ctypes.POINTER(sz)]
    lib.pnce_head_fwd.argtypes = [ctypes.POINTER(PnceLayer), ctypes.POINTER(PnceHead), i32, i32, i32, i32, f32, i32,
                                  vp, sz, vp, vp, vp]
    lib.pnce_head_fwd_ex.argtypes = [ctypes.POINTER(PnceLayer), ctypes.POINTER(PnceHead), i32, i32, i32, i32, i32, f32, i32,
                                     vp, sz, vp, vp, vp]
    lib.pnce_head_bwd_ex.argtypes = [ctypes.POINTER(PnceLayer), ctypes.POINTER(PnceHead), i32, i32, i32, i32, i32, i32, i32,
                                     vp, sz, vp, vp]
    lib.pnce_head_mb_workspace_bytes.argtypes = lib.pnce_head_workspace_bytes.argtypes
    lib.pnce_head_mb_fwd.argtypes = lib.pnce_head_fwd_ex.argtypes
    lib.pnce_head_mb_shard_workspace_bytes.argtypes = [ctypes.POINTER(PnceLayer), i32, i32, i32, i32, ctypes.POINTER(sz),
                                                       ctypes.POINTER(sz), ctypes.POINTER(sz)]
    lib.pnce_head_mb_shard_keys.argtypes = [ctypes.POINTER(PnceLayer), ctypes.POINTER(PnceHead), i32, i32, i32, i32, i32,
                                            i32, i32, i32, vp, sz, vp, vp]
    lib.pnce_head_mb_shard_loss.argtypes = [ctypes.POINTER(PnceLayer), ctypes.POINTER(PnceHead), i32, i32, i32, i32, i32,
                                            i32, i32, f32, i32, vp, sz, vp, vp, vp]
    for fn in (lib.pnce_head_bwd, lib.pnce_head_bwd_params, lib.pnce_head_bwd_dense):
        fn.argtypes = [ctypes.POINTER(PnceLayer), ctypes.POINTER(PnceHead), i32, i32, i32, i32, i32, vp, sz, vp, vp]
    lib.pnce_netf_workspace_bytes.argtypes = [ctypes.POINTER(PnceSample), i32, i32, i32, ctypes.POINTER(sz)]
    for fn in (lib.pnce_netf_fwd, lib.pnce_netf_bwd):
        fn.argtypes = [ctypes.POINTER(PnceSample), ctypes.POINTER(PnceHead), i32, i32, i32, i32, i32, i32, vp, sz, vp, vp]
    lib.pnce_multi_axpby.argtypes = [vp, vp, vp, vp, vp, i32, f32, f32, i32, vp]
    f64 = ctypes.c_double
    lib.pnce_amp_adam_scratch_floats.argtypes = [i32]
    lib.pnce_amp_adam_step.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, vp, vp, f32, f32, i32, f32,
                                       f64, f64, f64, f64, f64, vp, vp]
    lib.pnce_diffaug_scratch_floats.argtypes = [i32, i32, i32]
    lib.pnce_diffaug.argtypes = [vp, vp, i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, i32, i32, vp, i32, vp]
    lib.pnce_hinge_fwd.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp]
    lib.pnce_hinge_bwd.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, vp, vp]
    u32 = ctypes.c_uint
    lib.pnce_selftest_umma.argtypes = [vp, sz, vp, sz, u32, u32, u32, u32, u32, u32, i32, i32, i32, vp, vp, vp]
    lib.pnce_comp_supported.argtypes = [i32]
    lib.pnce_comp_alloc.argtypes = [ctypes.c_ssize_t, i32, vp]
    lib.pnce_comp_alloc.restype = vp
    lib.pnce_comp_free.argtypes = [vp, ctypes.c_ssize_t, i32, vp]
    lib.pnce_comp_free.restype = None
    lib.pnce_comp_is_compressed.argtypes = [vp]
    for name in EXPORTS:
        if name not in ("pnce_status_string", "pnce_last_cuda_error", "pnce_amp_adam_scratch_floats",
                        "pnce_diffaug_scratch_floats", "pnce_comp_alloc", "pnce_comp_free"):
            getattr(lib, name).restype = i32
    lib.pnce_amp_adam_scratch_floats.restype = sz
    lib.pnce_diffaug_scratch_floats.restype = sz
    if lib.pnce_abi_version() != ABI_VERSION:
        raise PnceError("libpnce.so ABI version mismatch")
    _lib = lib
    return lib


def check(status, what):
    if status != 0:
        lib = load()
        msg = lib.pnce_status_string(status).decode()
        extra = lib.pnce_last_cuda_error().decode()
        raise PnceError(f"{what}: {msg}" + (f" ({extra})" if status == -4 and extra else ""))
