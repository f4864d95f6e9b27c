"""ctypes binding of libpysp_b200.so (include/pysp_b200.h).  Thin: structs, prototypes, error mapping.

There is no CPU path: if the shared library is missing the import of any compute entry point raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# PYSP_B200_LIB: developer hook to load an A/B build of the same library (tools/kbench.py)
LIB_PATH = os.environ.get("PYSP_B200_LIB") or os.path.join(_HERE, "libpysp_b200.so")

OK, ERR_INVALID, ERR_UNSUPPORTED, ERR_CUDA = 0, -1, -2, -3
CFA = {"RGGB": 1, "BGGR": 2, "GRBG": 3, "GBRG": 4}
IN_U16, IN_F32 = 0, 1
OUT_CAM_F32, OUT_LIN_F32, OUT_LIN_F16, OUT_SRGB_U8, OUT_SRGB_U16, OUT_YCC420_U8 = 0, 1, 2, 3, 4, 5
QUALITY_BEST, QUALITY_FAST = 0, 1
JPEG_444, JPEG_422, JPEG_420 = 0, 1, 2
MAX_BRACKETS = 16


class DevelopArgs(C.Structure):
    """struct pysp_develop_args"""
    _fields_ = [
        ("height", C.c_int32), ("width", C.c_int32),
        ("cfa_pattern", C.c_int32), ("in_kind", C.c_int32),
        ("in_", C.c_void_p), ("in_pitch_bytes", C.c_int64),
        ("in_row0", C.c_int32), ("in_rows", C.c_int32),
        ("black", C.c_float * 4), ("white", C.c_float * 4), ("wb", C.c_float * 3),
        ("cam_to_srgb", C.c_double * 9),
        ("stages", C.c_int32), ("is_hdr", C.c_int32), ("apply_gamma", C.c_int32), ("out_kind", C.c_int32),
        ("out", C.c_void_p), ("out_pitch_bytes", C.c_int64), ("out_row0", C.c_int32),
        ("row_begin", C.c_int32), ("row_end", C.c_int32),
        ("scratch", C.c_void_p), ("scratch_bytes", C.c_int64),
        ("lab_lut", C.c_void_p),
        ("quality", C.c_int32),
        ("dir_map", C.c_void_p), ("dir_map_pitch_bytes", C.c_int64),
        ("out_cb", C.c_void_p), ("out_cr", C.c_void_p), ("out_chroma_pitch_bytes", C.c_int64),
    ]


_lib = None


def lib():
    """Load the CUDA library (built by `__graft_entry__.build()` / `pysp_b200.build`)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "pysp_b200: %s is missing -- build it with `python -m pysp_b200.build` "
            "(nvcc, sm_100a).  There is no CPU fallback." % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    L.pysp_develop.argtypes = [C.POINTER(DevelopArgs), C.c_void_p]
    L.pysp_develop.restype = C.c_int
    L.pysp_develop_scratch_bytes.argtypes = [C.c_int32, C.c_int32, C.c_int32]
    L.pysp_develop_scratch_bytes.restype = C.c_int64
    L.pysp_develop_halo_rows.argtypes = [C.c_int32]
    L.pysp_develop_halo_rows.restype = C.c_int32
    L.pysp_lab_lut_bytes.argtypes = []
    L.pysp_lab_lut_bytes.restype = C.c_int64
    L.pysp_lab_lut_pack_host.argtypes = [C.c_void_p, C.c_void_p]
    L.pysp_lab_lut_pack_host.restype = C.c_int
    L.pysp_normalize_u16.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int32, C.c_int32,
                                     C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_void_p]
    L.pysp_normalize_u16.restype = C.c_int
    L.pysp_cam_to_lin_srgb.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_double), C.c_int32,
                                       C.c_int32, C.c_int32, C.c_void_p]
    L.pysp_cam_to_lin_srgb.restype = C.c_int
    L.pysp_wb_scale.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_double), C.c_double, C.c_int32, C.c_int32,
                                C.c_int32, C.c_int32, C.c_void_p]
    L.pysp_wb_scale.restype = C.c_int
    L.pysp_rgb_to_lab_cv2.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    L.pysp_rgb_to_lab_cv2.restype = C.c_int
    L.pysp_lin_srgb_to_srgb.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    L.pysp_lin_srgb_to_srgb.restype = C.c_int
    L.pysp_fuse_exposures.argtypes = [C.POINTER(C.c_void_p), C.c_int32, C.c_int64, C.c_int32, C.c_int32,
                                      C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int32, C.c_void_p,
                                      C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]
    L.pysp_fuse_exposures.restype = C.c_int
    L.pysp_flat_workspace_bytes.argtypes = [C.c_int32, C.c_int32]
    L.pysp_flat_workspace_bytes.restype = C.c_int64
    L.pysp_bayer_plane_means.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64,
                                         C.c_void_p]
    L.pysp_bayer_plane_means.restype = C.c_int
    L.pysp_flat_frame_correction.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int32,
                                             C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]
    L.pysp_flat_frame_correction.restype = C.c_int
    L.pysp_find_hot_pixels_threshold.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_float, C.c_int32,
                                                 C.c_void_p, C.c_void_p]
    L.pysp_find_hot_pixels_threshold.restype = C.c_int
    L.pysp_fuse_exposures_from_debayer.argtypes = [C.POINTER(C.c_void_p), C.c_int32, C.c_int64, C.POINTER(C.c_float),
                                                   C.c_float, C.POINTER(C.c_int32), C.POINTER(C.c_float),
                                                   C.POINTER(C.c_float), C.c_int32, C.c_double, C.POINTER(C.c_double),
                                                   C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
    L.pysp_fuse_exposures_from_debayer.restype = C.c_int
    L.pysp_warp_rectilinear_table.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.POINTER(C.c_float), C.c_float,
                                              C.c_float, C.c_float, C.c_void_p, C.c_int64, C.c_void_p]
    L.pysp_warp_rectilinear_table.restype = C.c_int
    L.pysp_remap_lanczos4.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32,
                                      C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    L.pysp_remap_lanczos4.restype = C.c_int
    L.pysp_warp_rectilinear_apply.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_float),
                                              C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]
    L.pysp_warp_rectilinear_apply.restype = C.c_int
    L.pysp_jpeg_max_bytes.argtypes = [C.c_int32, C.c_int32]
    L.pysp_jpeg_max_bytes.restype = C.c_int64
    L.pysp_jpeg_workspace_bytes.argtypes = [C.c_int32, C.c_int32]
    L.pysp_jpeg_workspace_bytes.restype = C.c_int64
    L.pysp_jpeg_encode_ycc420.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32,
                                          C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    L.pysp_jpeg_encode_ycc420.restype = C.c_int
    L.pysp_jpeg_rgb_max_bytes.argtypes = [C.c_int32, C.c_int32, C.c_int32]
    L.pysp_jpeg_rgb_max_bytes.restype = C.c_int64
    L.pysp_jpeg_rgb_workspace_bytes.argtypes = [C.c_int32, C.c_int32, C.c_int32]
    L.pysp_jpeg_rgb_workspace_bytes.restype = C.c_int64
    L.pysp_jpeg_encode_rgb.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int64,
                                       C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    L.pysp_jpeg_encode_rgb.restype = C.c_int
    L.pysp_timing_enable.argtypes = [C.c_int32]
    L.pysp_timing_enable.restype = None
    L.pysp_timing_collect.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_int64)]
    L.pysp_timing_collect.restype = C.c_int
    L.pysp_last_error.restype = C.c_char_p
    L.pysp_version.restype = C.c_char_p
    L.pysp_kernel_launches.restype = C.c_int64
    _lib = L
    return L


def check(rc, last_error=None):
    """Map a status code to the exception type the reference raises in the same situation."""
    if rc == OK:
        return
    msg = (last_error or lib().pysp_last_error)().decode("utf-8", "replace")
    if rc == ERR_INVALID:
        raise ValueError(msg)
    if rc == ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise RuntimeError(msg)


def fill_develop_args(height, width, pattern, in_kind, in_ptr, in_pitch, in_row0, in_rows, black, white, wb,
                      cam_to_srgb, stages, is_hdr, gamma, out_kind, out_ptr, out_pitch, out_row0, row_begin,
                      row_end, scratch_ptr, scratch_bytes, lut_ptr, quality=0, dir_map_ptr=None, dir_map_pitch=0,
                      out_cb_ptr=None, out_cr_ptr=None, out_chroma_pitch=0):
    a = DevelopArgs()
    a.height, a.width = int(height), int(width)
    if isinstance(pattern, str):
        if pattern.upper() not in CFA:
            raise NotImplementedError("%s not implemented!" % pattern)      # image.py:152
        pattern = CFA[pattern.upper()]
    a.cfa_pattern = int(pattern)
    a.in_kind = in_kind
    a.in_ = in_ptr
    a.in_pitch_bytes = int(in_pitch)
    a.in_row0, a.in_rows = int(in_row0), int(in_rows)
    for i in range(4):
        a.black[i] = float(black[i]) if black is not None else 0.0
        a.white[i] = float(white[i]) if white is not None else 1.0
    for i in range(3):
        a.wb[i] = float(wb[i])
    m = [float(v) for row in cam_to_srgb for v in row]
    for i in range(9):
        a.cam_to_srgb[i] = m[i]
    a.stages = int(stages)
    a.is_hdr = int(bool(is_hdr))
    a.apply_gamma = int(bool(gamma))
    a.out_kind = out_kind
    a.out = out_ptr
    a.out_pitch_bytes = int(out_pitch)
    a.out_row0 = int(out_row0)
    a.row_begin, a.row_end = int(row_begin), int(row_end)
    a.scratch = scratch_ptr
    a.scratch_bytes = int(scratch_bytes)
    a.lab_lut = lut_ptr
    a.quality = int(quality)
    a.dir_map = dir_map_ptr
    a.dir_map_pitch_bytes = int(dir_map_pitch)
    a.out_cb, a.out_cr = out_cb_ptr, out_cr_ptr
    a.out_chroma_pitch_bytes = int(out_chroma_pitch)
    return a
