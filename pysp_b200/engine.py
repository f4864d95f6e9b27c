"""Device plumbing between the Python drop-in layer and the C ABI (libpysp_b200.so).

PyTorch is used only for device memory, streams and (elsewhere) torch.distributed; every computation on
the develop path happens in the CUDA kernels behind the C ABI.  There is no CPU path: calling into this
module without a CUDA device raises.
"""
import contextlib
import ctypes as C
import os
import threading

import numpy as np
import torch

from . import _capi

_DATA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data", "lab_lut33_i16.npy")
_lock = threading.Lock()
_lut_dev = {}       # device index -> packed Lab table (uint8 tensor)
_scratch = {}       # (device index, stream handle) -> uint8 tensor, grow-only


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("pysp_b200 needs a CUDA device (sm_100a); there is no CPU fallback")


def _stream_ptr(stream=None):
    s = stream if stream is not None else torch.cuda.current_stream()
    return s.cuda_stream


@contextlib.contextmanager
def _on(device, stream):
    """Make `device` current and `stream` torch's current stream for the body of an entry point.  Every temporary and
    output is then allocated by the caching allocator ON the stream the kernels are launched on, so a block that is
    freed while kernels are still queued can only be handed out again behind them (the allocator orders re-use against
    the allocation stream only)."""
    with torch.cuda.device(device):
        if stream is None:
            yield
        else:
            with torch.cuda.stream(stream):
                yield


def lab_lut(device):
    """Device copy of the cv2 RGB->Lab interpolation table (see tools/harvest_lab_lut.py)."""
    idx = torch.device(device).index
    if idx is None:
        idx = torch.cuda.current_device()
    with _lock:
        t = _lut_dev.get(idx)
        if t is None:
            lut = np.ascontiguousarray(np.load(_DATA).astype(np.int16))
            packed = np.empty(int(_capi.lib().pysp_lab_lut_bytes()), dtype=np.uint8)
            _capi.check(_capi.lib().pysp_lab_lut_pack_host(lut.ctypes.data, packed.ctypes.data))
            t = torch.from_numpy(packed).to("cuda:%d" % idx)
            _lut_dev[idx] = t
    return t


def _get_scratch(device, nbytes, stream):
    if nbytes <= 0:
        return None
    key = (torch.device(device).index, _stream_ptr(stream))
    with _lock:
        t = _scratch.get(key)
        if t is None or t.numel() < nbytes:
            t = torch.empty(int(nbytes), dtype=torch.uint8, device=device)
            _scratch[key] = t
    return t


def release_scratch():
    with _lock:
        _scratch.clear()


def padded_pitch_elems(width, elem_size):
    """Row length in elements whose byte pitch is a multiple of 128: TMA needs 16-byte aligned rows (6000 x 2 B is, 11548 x 2 B
    is not), 128 keeps box rows on whole L2 lines."""
    q = 128 // elem_size
    return (int(width) + q - 1) // q * q


def alloc_rows(rows, width, dtype, device):
    """[rows, width] CUDA view over a buffer whose row pitch is padded (see padded_pitch_elems): `develop` can then move a
    frame of ANY even width with TMA."""
    buf = torch.empty((int(rows), padded_pitch_elems(width, torch.empty((), dtype=dtype).element_size())), dtype=dtype, device=device)
    return buf[:, :int(width)]


def to_device(a, device=None, dtype=None, pad_pitch=False):
    """NumPy / CPU tensor / CUDA tensor -> CUDA tensor with unit column stride (no copy if already there).  pad_pitch: 2-D inputs
    are uploaded into a buffer with a padded row pitch (alloc_rows), so that frames whose width is not a multiple of 16 bytes
    still take the TMA path."""
    require_cuda()
    if isinstance(a, np.ndarray):
        if a.dtype == np.uint16:
            a = a.view(np.int16)                     # same bits; uint16 tensors have no CPU kernels
        t = torch.from_numpy(np.ascontiguousarray(a))
    else:
        t = a
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    if pad_pitch and t.dim() == 2 and (t.shape[1] * t.element_size()) % 16 != 0:
        dst = alloc_rows(t.shape[0], t.shape[1], t.dtype, device if device is not None else (t.device if t.is_cuda else "cuda"))
        dst.copy_(t, non_blocking=True)
        return dst
    if not t.is_cuda:
        t = t.to(device if device is not None else "cuda", non_blocking=True)
    if t.dim() == 2 and t.stride(1) == 1 and t.stride(0) >= t.shape[1]:
        return t                                     # a row-padded 2-D view stays as it is (every 2-D entry point takes a pitch)
    return t.contiguous()


_OUT_KINDS = {"cam": _capi.OUT_CAM_F32, "lin": _capi.OUT_LIN_F32, "lin_f16": _capi.OUT_LIN_F16,
              "srgb_u8": _capi.OUT_SRGB_U8, "srgb_u16": _capi.OUT_SRGB_U16, "ycc420": _capi.OUT_YCC420_U8}
_OUT_DTYPES = {_capi.OUT_CAM_F32: torch.float32, _capi.OUT_LIN_F32: torch.float32, _capi.OUT_LIN_F16: torch.float16,
               _capi.OUT_SRGB_U8: torch.uint8, _capi.OUT_SRGB_U16: torch.uint16, _capi.OUT_YCC420_U8: torch.uint8}


def i420_bytes(rows, width):
    """bytes of one I420 buffer (Y [rows, W], then Cb and Cr [rows/2, W/2]) of an even-sized image"""
    return int(rows) * int(width) * 3 // 2


def i420_planes(buf, rows, width):
    """(y, cb, cr): uint8 views [rows, W], [rows/2, W/2], [rows/2, W/2] over the first i420_bytes(rows, W) bytes of the flat
    uint8 tensor `buf`, Y first, then Cb, then Cr -- the layout a JPEG encoder's raw-data input takes, moved by one copy."""
    rows, width = int(rows), int(width)
    if rows % 2 or width % 2 or buf.dtype != torch.uint8 or buf.dim() != 1 or buf.numel() < i420_bytes(rows, width):
        raise ValueError("i420_planes: a flat uint8 buffer of >= %d bytes and an even size are needed" % i420_bytes(rows, width))
    ny, nc = rows * width, (rows // 2) * (width // 2)
    return (buf[:ny].view(rows, width), buf[ny:ny + nc].view(rows // 2, width // 2),
            buf[ny + nc:ny + 2 * nc].view(rows // 2, width // 2))


def _check_ycc_planes(planes, rows, W):
    ok = isinstance(planes, (tuple, list)) and len(planes) == 3
    if ok:
        y, cb, cr = planes
        ok = all(t.is_cuda and t.dtype == torch.uint8 and t.dim() == 2 and t.stride(1) == 1 for t in planes) and \
            y.shape[1] == W and y.shape[0] >= rows and cb.stride(0) == cr.stride(0) and \
            all(t.shape[1] == W // 2 and t.shape[0] >= rows // 2 for t in (cb, cr))
    if not ok:
        raise ValueError("engine.develop: out_tensor for out='ycc420' must be (y, cb, cr) uint8 CUDA views [rows, W], "
                         "[rows/2, W/2], [rows/2, W/2] with unit column stride and one chroma pitch")
    return planes


def develop(mosaic, wb, cam_to_srgb, stages=1, pattern="RGGB", black=None, white=None, hdr=False, gamma=False,
            out="lin", out_tensor=None, rows=None, frame_height=None, in_row0=0, out_row0=None, stream=None,
            quality="best", dir_map=None):
    """Run the fused develop chain on one frame (or one row band of it) that is resident on the GPU.

    mosaic      CUDA tensor [rows_held, W]: uint16/int16 sensor counts (normalisation fused, needs
                black/white in the reference order [TL,TR,BR,BL]) or float32 `sensor_scaled`.
    rows        (row_begin, row_end) of the stored frame to produce; default the whole frame.
    frame_height / in_row0   when `mosaic` holds only rows [in_row0, in_row0+rows_held) of a taller frame.
    quality     "best" = AHD (debayer_ahd), "fast" = edge-assisted Gaussian (debayer_eag; stages/hdr ignored).
    dir_map     optional CUDA uint8 tensor [>= row_end-out_row0, W]: receives the AHD direction choice (1 = horizontal).
    out         "cam" (camera RGB), "lin" (linear sRGB, float32), "lin_f16", or the wire formats "srgb_u8" / "srgb_u16"
                (lin_srgb_to_srgb, then rounded into 8 / 16 bits) and "ycc420": the srgb_u8 result as libjpeg converts and
                subsamples it for a 4:2:0 JPEG (full-range YCbCr; include/pysp_b200.h, PYSP_OUT_YCC420_U8).
    Returns a CUDA tensor [row_end-row_begin, W, 3] of the matching dtype; for "ycc420" the uint8 planes (y, cb, cr) of
    shapes [n, W], [n/2, W/2], [n/2, W/2] (n = row_end - out_row0) over ONE contiguous I420 buffer (i420_planes), or
    `out_tensor` itself, which is then such a triple with any row pitches (Cb and Cr sharing one).
    """
    if quality not in ("best", "fast"):
        raise NotImplementedError("Quality mode not implemented: %s" % str(quality))
    if quality == "fast":
        stages = 0
    require_cuda()
    L = _capi.lib()
    if not mosaic.is_cuda:
        raise ValueError("engine.develop: mosaic must be a CUDA tensor (use engine.to_device)")
    if mosaic.dim() != 2:
        raise ValueError("engine.develop: mosaic must be 2-D")
    held, W = mosaic.shape
    H = int(frame_height) if frame_height is not None else held
    if mosaic.dtype in (torch.uint16, torch.int16):
        in_kind = _capi.IN_U16
        if black is None or white is None:
            raise ValueError("engine.develop: black/white levels are required for integer mosaics")
    elif mosaic.dtype == torch.float32:
        in_kind = _capi.IN_F32
    else:
        raise ValueError("engine.develop: unsupported mosaic dtype %s" % mosaic.dtype)
    rb, re = (0, H) if rows is None else (int(rows[0]), int(rows[1]))
    kind = _OUT_KINDS[out]
    odt = _OUT_DTYPES[kind]
    if out_row0 is None:
        out_row0 = rb
    dev = mosaic.device
    if dir_map is not None and (not dir_map.is_cuda or dir_map.dtype != torch.uint8 or dir_map.dim() != 2
                                or dir_map.shape[1] != W or dir_map.stride(1) != 1 or dir_map.shape[0] < re - out_row0):
        raise ValueError("engine.develop: dir_map must be a CUDA uint8 tensor [rows, W]")
    ycc = kind == _capi.OUT_YCC420_U8
    with _on(dev, stream):
        if mosaic.stride(1) != 1:
            mosaic = mosaic.contiguous()
        if ycc:
            if out_tensor is None:
                n = re - out_row0
                out_tensor = i420_planes(torch.empty(i420_bytes(n, W), dtype=torch.uint8, device=dev), n, W)
            else:
                out_tensor = _check_ycc_planes(out_tensor, re - out_row0, W)
        elif out_tensor is None:
            out_tensor = torch.empty((re - out_row0, W, 3), dtype=odt, device=dev)
        elif (not out_tensor.is_cuda or out_tensor.dtype != odt or out_tensor.dim() != 3
              or out_tensor.shape[1] != W or out_tensor.shape[2] != 3 or out_tensor.stride(2) != 1
              or out_tensor.stride(1) != 3 or out_tensor.shape[0] < re - out_row0):
            raise ValueError("engine.develop: out_tensor has the wrong shape/dtype/layout")
        nscr = int(L.pysp_develop_scratch_bytes(W, re - rb, int(stages)))
        scratch = _get_scratch(dev, nscr, stream)
        lut = lab_lut(dev)
        dst = out_tensor[0] if ycc else out_tensor
        a = _capi.fill_develop_args(
            H, W, pattern, in_kind, mosaic.data_ptr(), mosaic.stride(0) * mosaic.element_size(), in_row0, held,
            black, white, wb, cam_to_srgb, stages, hdr, gamma, kind, dst.data_ptr(),
            dst.stride(0) * dst.element_size(), out_row0, rb, re,
            scratch.data_ptr() if scratch is not None else None, nscr, lut.data_ptr(),
            quality=_capi.QUALITY_FAST if quality == "fast" else _capi.QUALITY_BEST,
            dir_map_ptr=dir_map.data_ptr() if dir_map is not None else None,
            dir_map_pitch=dir_map.stride(0) if dir_map is not None else 0,
            out_cb_ptr=out_tensor[1].data_ptr() if ycc else None, out_cr_ptr=out_tensor[2].data_ptr() if ycc else None,
            out_chroma_pitch=out_tensor[1].stride(0) if ycc else 0)
        _capi.check(L.pysp_develop(C.byref(a), _stream_ptr(stream)))
    return out_tensor


def jpeg_max_bytes(height, width):
    """pysp_jpeg_max_bytes: the largest file encode_jpeg can write for an even-sized frame"""
    n = int(_capi.lib().pysp_jpeg_max_bytes(int(height), int(width)))
    if n <= 0:
        raise ValueError("jpeg_max_bytes: height and width must be even, 2..65535 (got %dx%d)" % (height, width))
    return n


def encode_jpeg(planes, quality=75, out_tensor=None, stream=None):
    """Baseline JPEG of YCbCr 4:2:0 planes on the device (include/pysp_b200.h, pysp_jpeg_encode_ycc420): byte-identical to
    libjpeg's encode of the planes (Pillow: Image.merge("YCbCr", [Y, Cb, Cr upsampled 2x2]).save(f, "JPEG", quality=quality,
    subsampling=2)); when W is a multiple of 16, to libjpeg's JPEG of the srgb_u8 image the planes were developed from.

    planes      (y, cb, cr): uint8 CUDA views [H, W], [H/2, W/2], [H/2, W/2] with unit column stride, any row pitches (Cb and
                Cr sharing one), e.g. what develop(out="ycc420") returns.
    out_tensor  optional flat uint8 CUDA tensor of >= jpeg_max_bytes(H, W) bytes.
    Returns (buf, n): `buf` the uint8 CUDA tensor holding the file in its first n bytes, `n` a 0-d int64 CUDA tensor.  Nothing
    is synchronised: read n (e.g. n.item()) after the stream has reached it.
    """
    require_cuda()
    L = _capi.lib()
    ok = isinstance(planes, (tuple, list)) and len(planes) == 3
    if ok:
        y, cb, cr = planes
        ok = all(isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.uint8 and t.dim() == 2 and t.stride(1) == 1
                 for t in planes)
    if ok:
        H, W = y.shape
        ok = H % 2 == 0 and W % 2 == 0 and cb.shape == cr.shape == (H // 2, W // 2) and cb.stride(0) == cr.stride(0) and \
            cb.device == y.device and cr.device == y.device
    if not ok:
        raise ValueError("encode_jpeg: planes must be (y, cb, cr) uint8 CUDA views [H, W], [H/2, W/2], [H/2, W/2] of even H, W "
                         "on one device, with unit column stride and one chroma pitch")
    dev = y.device
    cap = jpeg_max_bytes(H, W)
    with _on(dev, stream):
        if out_tensor is None:
            out_tensor = torch.empty(cap, dtype=torch.uint8, device=dev)
        elif (not out_tensor.is_cuda or out_tensor.dtype != torch.uint8 or out_tensor.dim() != 1 or not out_tensor.is_contiguous()
              or out_tensor.device != dev):
            raise ValueError("encode_jpeg: out_tensor must be a flat contiguous uint8 CUDA tensor on the planes' device")
        nws = int(L.pysp_jpeg_workspace_bytes(H, W))
        ws = torch.empty(nws, dtype=torch.uint8, device=dev)
        n = torch.empty((), dtype=torch.int64, device=dev)
        _capi.check(L.pysp_jpeg_encode_ycc420(y.data_ptr(), y.stride(0), cb.data_ptr(), cr.data_ptr(), cb.stride(0), H, W,
                                              int(quality), out_tensor.data_ptr(), out_tensor.numel(), n.data_ptr(),
                                              ws.data_ptr(), nws, _stream_ptr(stream)))
    return out_tensor, n


_SUBSAMPLINGS = {"4:4:4": _capi.JPEG_444, "4:2:2": _capi.JPEG_422, "4:2:0": _capi.JPEG_420,
                 0: _capi.JPEG_444, 1: _capi.JPEG_422, 2: _capi.JPEG_420}


def jpeg_subsampling(subsampling):
    """PYSP_JPEG_444 / 422 / 420 of "4:4:4" / "4:2:2" / "4:2:0" or Pillow's integers 0 / 1 / 2"""
    s = _SUBSAMPLINGS.get(subsampling) if isinstance(subsampling, (str, int)) and not isinstance(subsampling, bool) else None
    if s is None:
        raise ValueError('JPEG subsampling must be "4:4:4", "4:2:2", "4:2:0" or 0, 1, 2 (got %r)' % (subsampling,))
    return s


def jpeg_rgb_max_bytes(height, width, subsampling="4:2:0"):
    """pysp_jpeg_rgb_max_bytes: the largest file encode_jpeg_rgb can write for an H x W image"""
    n = int(_capi.lib().pysp_jpeg_rgb_max_bytes(int(height), int(width), jpeg_subsampling(subsampling)))
    if n <= 0:
        raise ValueError("jpeg_rgb_max_bytes: height and width must be 1..65535 (got %dx%d)" % (height, width))
    return n


def encode_jpeg_rgb(rgb, quality=75, subsampling="4:2:0", out_tensor=None, stream=None):
    """Baseline JPEG of an 8-bit RGB image on the device (include/pysp_b200.h, pysp_jpeg_encode_rgb): byte-identical to
    libjpeg's encode of the image at any size (Pillow: Image.fromarray(S, "RGB").save(f, "JPEG", quality=quality,
    subsampling=subsampling)).

    rgb          uint8 CUDA tensor [H, W, 3] with strides (pitch, 3, 1), any pitch >= 3W, e.g. what develop(out="srgb_u8")
                 returns; H and W 1..65535.
    subsampling  "4:4:4" / "4:2:2" / "4:2:0", or Pillow's 0 / 1 / 2.
    out_tensor   optional flat uint8 CUDA tensor of >= jpeg_rgb_max_bytes(H, W, subsampling) bytes.
    Returns (buf, n) as encode_jpeg does: the file is the first n bytes of `buf`, `n` a 0-d int64 CUDA tensor, nothing is
    synchronised.
    """
    require_cuda()
    L = _capi.lib()
    s = jpeg_subsampling(subsampling)
    if not 1 <= int(quality) <= 100:
        raise ValueError("encode_jpeg_rgb: quality %d outside 1..100" % int(quality))
    if not (isinstance(rgb, torch.Tensor) and rgb.is_cuda and rgb.dtype == torch.uint8 and rgb.dim() == 3 and rgb.shape[2] == 3
            and rgb.stride(2) == 1 and rgb.stride(1) == 3 and rgb.stride(0) >= 3 * rgb.shape[1]):
        raise ValueError("encode_jpeg_rgb: rgb must be a uint8 CUDA tensor [H, W, 3] with strides (pitch >= 3W, 3, 1)")
    H, W = int(rgb.shape[0]), int(rgb.shape[1])
    dev = rgb.device
    cap = jpeg_rgb_max_bytes(H, W, s)
    with _on(dev, stream):
        if out_tensor is None:
            out_tensor = torch.empty(cap, dtype=torch.uint8, device=dev)
        elif (not isinstance(out_tensor, torch.Tensor) or not out_tensor.is_cuda or out_tensor.dtype != torch.uint8
              or out_tensor.dim() != 1 or not out_tensor.is_contiguous() or out_tensor.device != dev or out_tensor.numel() < cap):
            raise ValueError("encode_jpeg_rgb: out_tensor must be a flat contiguous uint8 CUDA tensor of >= %d bytes on the "
                             "image's device" % cap)
        nws = int(L.pysp_jpeg_rgb_workspace_bytes(H, W, s))
        ws = torch.empty(nws, dtype=torch.uint8, device=dev)
        n = torch.empty((), dtype=torch.int64, device=dev)
        _capi.check(L.pysp_jpeg_encode_rgb(rgb.data_ptr(), rgb.stride(0), H, W, int(quality), s, out_tensor.data_ptr(),
                                           out_tensor.numel(), n.data_ptr(), ws.data_ptr(), nws, _stream_ptr(stream)))
    return out_tensor, n


def normalize(raw, black, white, stream=None):
    """bayer_normalize on the device: uint16 [H,W] -> float32 [H,W]."""
    require_cuda()
    L = _capi.lib()
    H, W = raw.shape
    b = (C.c_float * 4)(*[float(v) for v in black[:4]])
    w = (C.c_float * 4)(*[float(v) for v in white[:4]])
    with _on(raw.device, stream):
        out = torch.empty((H, W), dtype=torch.float32, device=raw.device)
        _capi.check(L.pysp_normalize_u16(raw.data_ptr(), raw.stride(0) * 2, out.data_ptr(), out.stride(0) * 4, H, W,
                                         b, w, _stream_ptr(stream)))
    return out


def cam_to_rgb(rgb, matrix, clip=True, gamma=False, half=False, stream=None):
    """float32 [...,3] camera RGB -> float64 3x3 -> float32 (colorize/transform.py:37-53)."""
    require_cuda()
    L = _capi.lib()
    m = (C.c_double * 9)(*[float(v) for row in np.asarray(matrix, dtype=np.float64) for v in row])
    with _on(rgb.device, stream):
        rgb = rgb.contiguous()
        out = torch.empty(rgb.shape, dtype=torch.float16 if half else torch.float32, device=rgb.device)
        _capi.check(L.pysp_cam_to_lin_srgb(rgb.data_ptr(), out.data_ptr(), rgb.numel() // 3, m, int(bool(clip)),
                                           int(bool(gamma)), int(bool(half)), _stream_ptr(stream)))
    return out


WB_APPLY, WB_UNDO, CLIP01 = 0, 1, 2


def wb_dtype_flags(wb):
    """(wb_is_f64, max_is_f64) for a white-balance coefficient object, by NumPy's promotion rules (NEP 50) as they act in
    base_types/image_base.py:45-60: a float32 ndarray keeps everything in float32; a float64 ndarray promotes products and
    `max(wb)` (a NumPy float64 scalar) to float64; a Python list / tuple becomes a float64 array in products while its
    `max()` is a Python float (weak: the image stays float32)."""
    if isinstance(wb, np.ndarray):
        f64 = wb.dtype != np.float32
        return f64, f64
    if isinstance(wb, torch.Tensor):
        f64 = wb.dtype != torch.float32
        return f64, f64
    return True, False


def wb_scale(rgb, wb, mode, normalized=False, max_wb=1.0, stream=None):
    """wb_apply / wb_undo / clip_rgb on a float32 [...,3] CUDA tensor (base_types/image_base.py:45-60, transform.py:6-19).
    `wb` keeps its dtype: see wb_dtype_flags."""
    require_cuda()
    L = _capi.lib()
    if rgb.dtype != torch.float32 or rgb.shape[-1] != 3:
        raise ValueError("wb_scale: float32 [...,3] tensor expected")
    wb3 = (C.c_double * 3)(*[float(v) for v in (wb[:3] if wb is not None else (1.0, 1.0, 1.0))])
    wb_f64, max_f64 = wb_dtype_flags(wb) if wb is not None else (False, False)
    with _on(rgb.device, stream):
        rgb = rgb.contiguous()
        out = torch.empty_like(rgb)
        _capi.check(L.pysp_wb_scale(rgb.data_ptr(), out.data_ptr(), rgb.numel() // 3, wb3, float(max_wb), int(mode),
                                    int(bool(normalized)), int(wb_f64), int(max_f64), _stream_ptr(stream)))
    return out


def rgb_to_lab_cv2(rgb, stream=None):
    """cv2.cvtColor(float32 RGB, COLOR_RGB2LAB) on the device (the homogeneity metric's Lab; for stage tests)."""
    require_cuda()
    L = _capi.lib()
    with _on(rgb.device, stream):
        rgb = rgb.contiguous()
        out = torch.empty_like(rgb)
        _capi.check(L.pysp_rgb_to_lab_cv2(rgb.data_ptr(), out.data_ptr(), rgb.numel() // 3, lab_lut(rgb.device).data_ptr(),
                                          _stream_ptr(stream)))
    return out


def srgb_gamma(rgb, stream=None):
    require_cuda()
    L = _capi.lib()
    with _on(rgb.device, stream):
        rgb = rgb.contiguous()
        out = torch.empty_like(rgb)
        _capi.check(L.pysp_lin_srgb_to_srgb(rgb.data_ptr(), out.data_ptr(), rgb.numel(), _stream_ptr(stream)))
    return out


def fuse_exposures(brackets, ev_offsets, bias, brightest, want_count=True, stream=None):
    """raw_hdr.py:135-148 on the device.  brackets: list of float32 CUDA tensors [H,W] with equal strides."""
    require_cuda()
    L = _capi.lib()
    n = len(brackets)
    H, W = brackets[0].shape
    dev = brackets[0].device
    with _on(dev, stream):
        brackets = [b if b.stride(1) == 1 else b.contiguous() for b in brackets]
    pitch = brackets[0].stride(0) * 4
    for b in brackets:
        if b.shape != (H, W) or b.dtype != torch.float32 or b.device != dev:
            raise ValueError("fuse_exposures: brackets must be float32 [H,W] on one device")
        if b.stride(0) * 4 != pitch:
            raise ValueError("fuse_exposures: brackets must share one row pitch")
    ptrs = (C.c_void_p * n)(*[b.data_ptr() for b in brackets])
    evo = (C.c_float * n)(*[float(v) for v in ev_offsets])
    bia = (C.c_float * (3 * n))(*[float(v) for v in np.asarray(bias, dtype=np.float32).reshape(-1)])
    with _on(dev, stream):
        out = torch.empty((H, W), dtype=torch.float32, device=dev)
        cnt = torch.empty((H, W), dtype=torch.int32, device=dev) if want_count else None
        _capi.check(L.pysp_fuse_exposures(ptrs, n, pitch, H, W, evo, bia, int(brightest), out.data_ptr(),
                                          out.stride(0) * 4, cnt.data_ptr() if cnt is not None else None,
                                          (cnt.stride(0) * 4) if cnt is not None else 0, _stream_ptr(stream)))
    return out, cnt


def _f32_2d(t, what):
    if not t.is_cuda or t.dtype != torch.float32 or t.dim() != 2:
        raise ValueError("%s: float32 CUDA tensor [H,W] expected" % what)
    if t.shape[0] % 2 or t.shape[1] % 2:
        raise ValueError("%s: mosaic must have even dimensions" % what)
    return t if t.stride(1) == 1 else t.contiguous()


def bayer_plane_means(mosaic, stream=None):
    """np.mean of the R, G1, B, G2 planes of a float32 mosaic, bit-identical to NumPy (4 floats on the device)."""
    require_cuda()
    L = _capi.lib()
    H, W = mosaic.shape
    with _on(mosaic.device, stream):
        mosaic = _f32_2d(mosaic, "bayer_plane_means")
        nws = int(L.pysp_flat_workspace_bytes(H, W))
        ws = torch.empty(nws, dtype=torch.uint8, device=mosaic.device)
        out = torch.empty(4, dtype=torch.float32, device=mosaic.device)
        _capi.check(L.pysp_bayer_plane_means(mosaic.data_ptr(), mosaic.stride(0) * 4, H, W, out.data_ptr(), ws.data_ptr(), nws,
                                             _stream_ptr(stream)))
    return out


def flat_frame_correction(sensor, flat, clamp_high=False, stream=None):
    """raw_correction.py:25-63 on the device; returns the corrected float32 mosaic."""
    require_cuda()
    L = _capi.lib()
    if flat.shape != sensor.shape or flat.device != sensor.device:
        raise ValueError("flat_frame_correction: image and flat field must have the same shape and device")
    H, W = sensor.shape
    with _on(sensor.device, stream):
        sensor = _f32_2d(sensor, "flat_frame_correction")
        flat = _f32_2d(flat, "flat_frame_correction")
        nws = int(L.pysp_flat_workspace_bytes(H, W))
        ws = torch.empty(nws, dtype=torch.uint8, device=sensor.device)
        out = torch.empty_like(sensor)
        _capi.check(L.pysp_flat_frame_correction(sensor.data_ptr(), sensor.stride(0) * 4, flat.data_ptr(), flat.stride(0) * 4,
                                                 out.data_ptr(), out.stride(0) * 4, H, W, int(bool(clamp_high)), ws.data_ptr(),
                                                 nws, _stream_ptr(stream)))
    return out


def find_hot_pixels_threshold(sensor, min_delta, min_neighbour_count, stream=None):
    """raw_bad_pixel_corr.py:30-65 on the device; returns a bool tensor [4, H/2, W/2] (planes R, G1, B, G2)."""
    require_cuda()
    L = _capi.lib()
    H, W = sensor.shape
    with _on(sensor.device, stream):
        sensor = _f32_2d(sensor, "find_hot_pixels_threshold")
        masks = torch.empty((4, H // 2, W // 2), dtype=torch.uint8, device=sensor.device)
        _capi.check(L.pysp_find_hot_pixels_threshold(sensor.data_ptr(), sensor.stride(0) * 4, H, W, float(min_delta),
                                                     int(min_neighbour_count), masks.data_ptr(), _stream_ptr(stream)))
    return masks.view(torch.bool)


def fuse_exposures_from_debayer(images, wb, max_wb, normalized, ev_offsets, bias, brightest, offset_max, matrix,
                                write_back=True, want_count=True, stream=None):
    """raw_hdr.py:47-81 on the device.  images: float32 CUDA tensors [H,W,3] (contiguous; rewritten when write_back)."""
    require_cuda()
    L = _capi.lib()
    n = len(images)
    dev = images[0].device
    for t in images:
        if not t.is_cuda or t.dtype != torch.float32 or t.dim() != 3 or t.shape != images[0].shape or t.shape[2] != 3 \
                or not t.is_contiguous() or t.device != dev:
            raise ValueError("fuse_exposures_from_debayer: contiguous float32 CUDA tensors [H,W,3] of one shape expected")
    npx = images[0].shape[0] * images[0].shape[1]
    ptrs = (C.c_void_p * n)(*[t.data_ptr() for t in images])
    wb3 = (C.c_float * 3)(*[float(v) for v in wb[:3]])
    norm = (C.c_int32 * n)(*[int(bool(v)) for v in normalized])
    evo = (C.c_float * n)(*[float(v) for v in ev_offsets])
    bia = (C.c_float * n)(*[float(v) for v in bias])
    m = (C.c_double * 9)(*[float(v) for row in np.asarray(matrix, dtype=np.float64) for v in row])
    with _on(dev, stream):
        out = torch.empty_like(images[0])
        cnt = torch.empty(images[0].shape, dtype=torch.int32, device=dev) if want_count else None
        _capi.check(L.pysp_fuse_exposures_from_debayer(ptrs, n, npx, wb3, float(max_wb), norm, evo, bia, int(brightest),
                                                       float(offset_max), m, out.data_ptr(),
                                                       cnt.data_ptr() if cnt is not None else None, int(bool(write_back)),
                                                       _stream_ptr(stream)))
    return out, cnt


def kernel_launches():
    return int(_capi.lib().pysp_kernel_launches())


# ---- DNG WarpRectilinear (include/pysp_b200.h: post-demosaic lens correction) ---------------------------------------
_LANCZOS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data", "lanczos4_tab_f32.npy")
_lanczos_dev = {}


def lanczos_tab(device):
    """Device copy of OpenCV's float32 [32][8] Lanczos-4 table (see tools/harvest_lanczos4.py)."""
    idx = torch.device(device).index
    if idx is None:
        idx = torch.cuda.current_device()
    with _lock:
        t = _lanczos_dev.get(idx)
        if t is None:
            t = torch.from_numpy(np.ascontiguousarray(np.load(_LANCZOS), dtype=np.float32)).to("cuda:%d" % idx)
            _lanczos_dev[idx] = t
    return t


def warp_table(height, width, coeffs, cam_center_norm, scale=1.0, seed=None, device=None, stream=None):
    """compute_remapping_table / compute_offset_remapping_table (dng_warp_rectilinear_coords.pyx:67-95) on the device:
    float32 CUDA tensor [H, W, 2]."""
    require_cuda()
    L = _capi.lib()
    dev = seed.device if seed is not None else torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
    k = (C.c_float * 6)(*[float(v) for v in coeffs])
    with _on(dev, stream):
        if seed is not None:
            if not seed.is_cuda or seed.dtype != torch.float32 or tuple(seed.shape) != (height, width, 2):
                raise ValueError("warp_table: seed must be a float32 CUDA tensor [H, W, 2]")
            seed = seed.contiguous()
        table = torch.empty((height, width, 2), dtype=torch.float32, device=dev)
        _capi.check(L.pysp_warp_rectilinear_table(table.data_ptr(), width * 8, height, width, k, float(cam_center_norm[0]),
                                                  float(cam_center_norm[1]), float(scale),
                                                  seed.data_ptr() if seed is not None else None, width * 8, _stream_ptr(stream)))
    return table


def remap_lanczos4(image, plane, table, stream=None):
    """cv2.remap(image[:, :, plane], clip(table[..., 0]), clip(table[..., 1]), INTER_LANCZOS4): float32 CUDA tensor [H, W]."""
    require_cuda()
    L = _capi.lib()
    if not image.is_cuda or image.dtype != torch.float32 or image.dim() != 3 or not image.is_contiguous():
        raise ValueError("remap_lanczos4: contiguous float32 CUDA tensor [H, W, C] expected")
    H, W, Cn = image.shape
    with _on(image.device, stream):
        table = table.contiguous()
        out = torch.empty((H, W), dtype=torch.float32, device=image.device)
        _capi.check(L.pysp_remap_lanczos4(image.data_ptr() + 4 * int(plane), W * Cn * 4, Cn, out.data_ptr(), W * 4, 1, H, W,
                                          table.data_ptr(), W * 8, lanczos_tab(image.device).data_ptr(), _stream_ptr(stream)))
    return out


def warp_rectilinear(image, coeffs, cam_center_norm, scale=1.0, prior=None, stream=None):
    """opcode_warp_rectilinear (chan_distortion_corr.py:53-98) for all planes in one kernel.  image: contiguous float32 CUDA
    tensor [H, W, C]; coeffs [C][6]; prior optional float32 [H, W, C, 2].  Returns a new tensor."""
    require_cuda()
    L = _capi.lib()
    if not image.is_cuda or image.dtype != torch.float32 or image.dim() != 3:
        raise ValueError("warp_rectilinear: float32 CUDA tensor [H, W, C] expected")
    H, W, Cn = image.shape
    flat = [float(v) for row in coeffs for v in row]
    if len(flat) != 6 * Cn:
        raise ValueError("warp_rectilinear: one coefficient set of 6 per plane")
    k = (C.c_float * len(flat))(*flat)
    with _on(image.device, stream):
        image = image.contiguous()
        if prior is not None:
            if not prior.is_cuda or prior.dtype != torch.float32 or tuple(prior.shape) != (H, W, Cn, 2):
                raise ValueError("warp_rectilinear: prior must be a float32 CUDA tensor [H, W, C, 2]")
            prior = prior.contiguous()
        out = torch.empty_like(image)
        _capi.check(L.pysp_warp_rectilinear_apply(image.data_ptr(), out.data_ptr(), H, W, Cn, k, float(cam_center_norm[0]),
                                                  float(cam_center_norm[1]), float(scale),
                                                  prior.data_ptr() if prior is not None else None,
                                                  lanczos_tab(image.device).data_ptr(), _stream_ptr(stream)))
    return out
