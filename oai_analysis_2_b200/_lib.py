"""ctypes binding of liboai_b200.so -- the only route from Python to the CUDA kernels.

There is deliberately no fallback: if the shared object is missing or fails to load, importing this module raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liboai_b200.so")


class OaiError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        from . import build as _build

        _build.build()
    try:
        return ctypes.CDLL(LIB_PATH)
    except OSError as e:  # pragma: no cover
        raise OaiError(f"cannot load {LIB_PATH}: {e}. Run `python -m oai_analysis_2_b200.build`.") from e


lib = _load()
lib.oai_last_error.restype = ctypes.c_char_p
lib.oai_launch_count.restype = ctypes.c_longlong
lib.oai_intensity_window_workspace.restype = ctypes.c_size_t
lib.oai_reg_convt4_mma_workspace.restype = ctypes.c_size_t
lib.oai_reg_conv3_workspace.restype = ctypes.c_size_t
lib.oai_seg_workspace_bytes.restype = ctypes.c_size_t
lib.oai_reg_workspace_bytes.restype = ctypes.c_size_t
lib.oai_reg_loss_workspace_bytes.restype = ctypes.c_size_t
lib.oai_seg_quality_workspace_bytes.restype = ctypes.c_size_t
lib.oai_components_workspace_bytes.restype = ctypes.c_size_t
lib.oai_components_max.restype = ctypes.c_longlong
lib.oai_reg_convt4_umma_wbytes.restype = ctypes.c_size_t
lib.oai_reg_conv3_umma_wbytes.restype = ctypes.c_size_t
lib.oai_reg_conv3_umma_workspace.restype = ctypes.c_size_t
lib.oai_mc_workspace_bytes.restype = ctypes.c_size_t
lib.oai_mesh_regions_workspace_bytes.restype = ctypes.c_size_t
lib.oai_mesh_smooth_workspace_bytes.restype = ctypes.c_size_t
lib.oai_kmeans2_workspace_bytes.restype = ctypes.c_size_t
lib.oai_mesh_project_workspace_bytes.restype = ctypes.c_size_t

c_int, c_ll, c_size, c_void, c_float, c_double = (ctypes.c_int, ctypes.c_longlong, ctypes.c_size_t, ctypes.c_void_p,
                                                   ctypes.c_float, ctypes.c_double)


def check(status, what=""):
    if status != 0:
        raise OaiError(f"{what}: {lib.oai_last_error().decode()}")


def ptr(t):
    """Device/host pointer of a torch tensor or numpy array (None -> NULL)."""
    if t is None:
        return c_void(0)
    if hasattr(t, "data_ptr"):
        return c_void(t.data_ptr())
    return t.ctypes.data_as(c_void)  # keeps a reference to the array alive for the duration of the call


def stream_ptr():
    import torch

    return c_void(torch.cuda.current_stream().cuda_stream)


def launch_count():
    return int(lib.oai_launch_count())
