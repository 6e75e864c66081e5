"""ctypes binding of libdvq_sm100.so (C ABI declared in include/dvq.h).

There is deliberately no fallback: if the shared library has not been built
(``python d-vqvae_b200/build.py``) importing this module raises, and every
compute call on a machine without an sm_100 GPU raises ``RuntimeError`` with the
library's own message.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# DVQ_LIB selects an instrumented build of the same library (DVQ_TC_STATS=1 python d-vqvae_b200/build.py); default: the in-tree release build
LIB_PATH = os.environ.get("DVQ_LIB") or os.path.join(_HERE, "libdvq_sm100.so")

ABI_VERSION = 1
DVQ_TRAIN = 0x1
DVQ_WRITE_ONEHOT = 0x2
DVQ_CODEBOOK_CACHED = 0x200
DVQ_PATH_MASK = 0x30
DVQ_PATH_AUTO = 0x00
DVQ_PATH_SIMT = 0x10
DVQ_PATH_TC = 0x20
DVQ_HOST_COPY_ONLY = 0x100
DVQ_Z_BF16 = 0x400          # z / z_q (g_zq / dz) are bf16 rows; the codebook stays fp32

STATUS_NAMES = {0: "DVQ_OK", -1: "DVQ_ERR_BAD_SHAPE", -2: "DVQ_ERR_BAD_ALIGN", -3: "DVQ_ERR_UNSUPPORTED_ARCH",
                -4: "DVQ_ERR_WORKSPACE", -5: "DVQ_ERR_CUDA", -6: "DVQ_ERR_NCCL", -7: "DVQ_ERR_BAD_ARG"}

# every symbol include/dvq.h declares: name -> (restype, argtypes)
_vp, _i, _i64, _f, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_size_t
SYMBOLS = {
    "dvq_abi_version": (_i, []),
    "dvq_last_error": (C.c_char_p, []),
    "dvq_launch_count": (C.c_longlong, []),
    "dvq_profile_enable": (_i, [_i]),
    "dvq_vq_set_refine": (_i, [_i, C.c_longlong]),
    "dvq_debug_tc_layout": (_i, [_i, _i, C.POINTER(_i)]),
    "dvq_debug_tc_pair_layout": (_i, [C.c_longlong, _i, _i, C.POINTER(_i)]),
    "dvq_debug_tc_layout_ex": (_i, [C.c_longlong, _i, _i, _i, C.POINTER(_i)]),
    "dvq_debug_tc_image_offset": (C.c_longlong, [_i, _i, _i, _i, _i, C.POINTER(C.c_longlong)]),
    "dvq_profile_mean": (_i, [C.POINTER(_f), C.POINTER(_i), _i]),
    "dvq_debug_umma": (_i, [_vp, C.c_uint32, _vp, C.c_uint32, _i, C.POINTER(C.c_uint32), C.c_uint32, _i, _vp, _vp, _vp]),
    "dvq_device_info": (_i, [C.POINTER(_i), C.POINTER(_i), C.POINTER(_i)]),
    "dvq_vq_workspace_bytes": (_i, [_i64, _i, _i, _i, C.POINTER(_sz)]),
    "dvq_vq_forward": (_i, [_vp, _vp, _i64, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dvq_vq_read_counters": (_i, [_vp, _i64, _i, _i, _i, C.POINTER(_i)]),
    "dvq_vq_finalize": (_i, [_vp, _vp, _i64, _i, _i, _f, _f, _vp, _vp, _vp]),
    "dvq_vq_backward": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _f, _f, _vp, _vp, _vp]),
    "dvq_vq_code_sums": (_i, [_vp, _vp, _i64, _i, _i, _vp, _vp]),
    "dvq_vq_backward_ex": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _f, _f, _i, _vp, _vp, _vp]),
    "dvq_vq_code_sums_ex": (_i, [_vp, _vp, _i64, _i, _i, _i, _vp, _vp]),
    "dvq_pcnn_gemm": (_i, [_vp, _vp]),
    "dvq_pcnn_embed": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _i, _vp, _vp, _vp]),
    "dvq_pcnn_rows_to_image": (_i, [_vp, _i, _i, _vp, _i, _i, _vp, _vp]),
    "dvq_gather": (_i, [_vp, _vp, _i64, _i, _i, _vp, _vp, _vp]),
    "dvq_gather_multi": (_i, [_vp, _i, _vp, _i64, _i, _i, _vp, _i64, _vp, _vp]),
    "dvq_onehot": (_i, [_vp, _i64, _i, _vp, _vp]),
    "dvq_host_ctx_create": (_i, [_i64, _i, _i, C.POINTER(_vp)]),
    "dvq_host_ctx_destroy": (_i, [_vp]),
    "dvq_vq_forward_host": (_i, [_vp, _vp, _vp, _i64, _i, _i, _i, _f, _f, _vp, _vp, C.POINTER(_f), C.POINTER(_f)]),
    "dvq_pointnet_workspace_bytes": (_i, [_i, _i, _i, C.POINTER(_sz)]),
    "dvq_pointnet_forward": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "dvq_pointnet_workspace_bytes_ex": (_i, [_i, _i, _i, _i, C.POINTER(_sz)]),
    "dvq_pointnet_forward_ex": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "dvq_allreduce_stats": (_i, [_vp, _vp, _vp, _i, _vp]),
    "dvq_mano_forward": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp]),
}


class ManoModel(C.Structure):
    """Mirror of ``DvqManoModel`` (include/dvq.h): device pointers to the fp32 tables of a MANO hand model."""
    _fields_ = [(n, C.c_void_p) for n in ("v_template", "shapedirs", "posedirs", "j_regressor", "weights", "hands_components",
                                          "pose_mean", "parents")] + [("ncomps", C.c_int)]


class PointNetWeights(C.Structure):
    """Mirror of ``DvqPointNetWeights`` (include/dvq.h): device pointers to BN-folded fp32 weights."""
    _fields_ = [(n, C.c_void_p) for n in (
        "stn_w1", "stn_b1", "stn_w2", "stn_b2", "stn_w3", "stn_b3",
        "stn_fc1_w", "stn_fc1_b", "stn_fc2_w", "stn_fc2_b", "stn_fc3_w", "stn_fc3_b",
        "w1", "b1", "w2", "b2", "w3", "b3")]


if not os.path.exists(LIB_PATH):
    raise ImportError(
        "dvq: %s is missing — build it with `python d-vqvae_b200/build.py` "
        "(nvcc, sm_100a).  There is no CPU or PyTorch fallback for this path." % LIB_PATH)

lib = C.CDLL(LIB_PATH)
for _name, (_res, _args) in SYMBOLS.items():
    _fn = getattr(lib, _name)  # AttributeError here == header and library disagree
    _fn.restype = _res
    _fn.argtypes = _args

if lib.dvq_abi_version() != ABI_VERSION:
    raise ImportError("dvq: ABI mismatch: library %d, binding %d" % (lib.dvq_abi_version(), ABI_VERSION))


def last_error() -> str:
    msg = lib.dvq_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc: int, what: str = "") -> None:
    """Raise ``RuntimeError(dvq_last_error())`` on any non-zero return (SURVEY §8b error convention)."""
    if rc != 0:
        raise RuntimeError("%s%s: %s" % (what + ": " if what else "", STATUS_NAMES.get(rc, str(rc)), last_error()))


def device_info():
    sm, maj, mnr = C.c_int(), C.c_int(), C.c_int()
    check(lib.dvq_device_info(C.byref(sm), C.byref(maj), C.byref(mnr)), "dvq_device_info")
    return sm.value, maj.value, mnr.value


def vq_workspace_bytes(n: int, k: int, d: int, flags: int) -> int:
    out = C.c_size_t()
    check(lib.dvq_vq_workspace_bytes(n, k, d, flags, C.byref(out)), "dvq_vq_workspace_bytes")
    return out.value


DVQ_PN_FP16_TC = 0x1


def pointnet_workspace_bytes(b: int, c: int, p: int, flags: int = 0) -> int:
    out = C.c_size_t()
    check(lib.dvq_pointnet_workspace_bytes_ex(b, c, p, flags, C.byref(out)), "dvq_pointnet_workspace_bytes_ex")
    return out.value


def launch_count() -> int:
    return int(lib.dvq_launch_count())


def profile_mean():
    """Mean CUDA-event time (ms) per stage of the dvq_vq_forward calls since dvq_profile_enable(1):
    ((code_norms, main_kernel, refine, onehot), calls_averaged)."""
    buf = (C.c_float * 4)()
    cnt = (C.c_int * 4)()
    check(lib.dvq_profile_mean(buf, cnt, 4), "dvq_profile_mean")
    return tuple(float(v) for v in buf), tuple(int(v) for v in cnt)
