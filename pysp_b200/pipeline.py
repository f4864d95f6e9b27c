"""Host-resident batches: stream frames through one GPU with copies overlapped with the kernels.

`FramePipeline` is the public batch API: frames start and end in (pinned) HOST memory.  Each of `depth`
slots owns a CUDA stream, a device mosaic buffer and a device output buffer; frame i uses slot i % depth:
H2D copy -> fused develop chain -> D2H copy, all asynchronous on the slot's stream, so the upload of frame
i+1 and the download of frame i-1 overlap the kernels of frame i (the two copy engines run concurrently
with the SMs).  No CPU computation is involved.

With out="ycc420" each output is one flat I420 buffer of H*W*3/2 bytes (Y, then Cb, then Cr; engine.i420_planes gives the
three planes of it), so one copy moves a frame.

With out="jpeg" each frame is developed into device ycc420 planes and encoded on the device (engine.encode_jpeg, quality
`jpeg_quality`); its length goes to pinned host memory, and once that has landed exactly that many bytes are copied into the
frame's output.  The host waits for frame i's length only after frame i + depth - 1 has been queued, so the later frames' work
keeps the GPU busy while it waits.  `run` returns the lengths.  `jpeg_subsampling` "4:4:4" or "4:2:2" (or Pillow's 0 / 1)
develops srgb_u8 into the slot's device buffer instead and encodes that with engine.encode_jpeg_rgb; the default "4:2:0"
keeps the ycc420 planes route.
"""
import torch

from . import engine


class FramePipeline:
    def __init__(self, height, width, wb, cam_to_srgb, stages=1, pattern="RGGB", black=None, white=None,
                 hdr=False, gamma=False, out="lin", device=None, depth=3, jpeg_quality=75, jpeg_subsampling="4:2:0"):
        engine.require_cuda()
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self.h, self.w = int(height), int(width)
        self.jpeg = out == "jpeg"
        self.jpeg_quality = int(jpeg_quality)
        self.jpeg_subsampling = engine.jpeg_subsampling(jpeg_subsampling)
        self.jpeg_rgb = self.jpeg and self.jpeg_subsampling != engine._capi.JPEG_420     # 4:4:4 / 4:2:2 from srgb_u8
        planes = out == "ycc420" or (self.jpeg and not self.jpeg_rgb)
        self.kw = dict(wb=wb, cam_to_srgb=cam_to_srgb, stages=stages, pattern=pattern, black=black, white=white,
                       hdr=hdr, gamma=gamma, out=("srgb_u8" if self.jpeg_rgb else "ycc420") if self.jpeg else out)
        self.out_dtype = engine._OUT_DTYPES[engine._OUT_KINDS[self.kw["out"]]]
        self.out_shape = (engine.i420_bytes(self.h, self.w),) if planes else (self.h, self.w, 3)
        self.depth = depth
        with torch.cuda.device(self.device):
            self.streams = [torch.cuda.Stream() for _ in range(depth)]
            self.d_in = [torch.empty((self.h, self.w), dtype=torch.int16, device=self.device) for _ in range(depth)]
            self.d_out = [torch.empty(self.out_shape, dtype=self.out_dtype, device=self.device) for _ in range(depth)]
        # what develop writes into: the output tensor itself, or the three planes over the flat I420 buffer
        self.d_dst = [engine.i420_planes(d, self.h, self.w) if planes else d for d in self.d_out]
        if self.jpeg:
            self.jpeg_bytes = (engine.jpeg_rgb_max_bytes(self.h, self.w, self.jpeg_subsampling) if self.jpeg_rgb
                               else engine.jpeg_max_bytes(self.h, self.w))
            with torch.cuda.device(self.device):
                self.d_jpeg = [torch.empty(self.jpeg_bytes, dtype=torch.uint8, device=self.device) for _ in range(depth)]

    def pinned_input(self):
        return torch.empty((self.h, self.w), dtype=torch.int16).pin_memory()

    def pinned_output(self):
        """a host buffer for one output; for out="jpeg" sized to the largest file (engine.jpeg_max_bytes, or
        engine.jpeg_rgb_max_bytes for 4:4:4 / 4:2:2)"""
        if self.jpeg:
            return torch.empty(self.jpeg_bytes, dtype=torch.uint8).pin_memory()
        return torch.empty(self.out_shape, dtype=self.out_dtype).pin_memory()

    def h2d_bytes(self):
        return self.h * self.w * 2

    def d2h_bytes(self):
        return self.d_out[0].numel() * self.d_out[0].element_size()

    def run(self, host_frames, host_outputs):
        """host_frames[i] (int16/uint16 bits, ideally pinned) -> host_outputs[i] (pinned).  Returns after
        every output has landed in host memory; for out="jpeg" the list of file lengths (host_outputs[i][:n[i]])."""
        assert len(host_frames) == len(host_outputs)
        if self.jpeg:
            return self._run_jpeg(host_frames, host_outputs)
        with torch.cuda.device(self.device):
            for i, (src, dst) in enumerate(zip(host_frames, host_outputs)):
                k = i % self.depth
                s = self.streams[k]
                with torch.cuda.stream(s):
                    self.d_in[k].copy_(src, non_blocking=True)
                    engine.develop(self.d_in[k], out_tensor=self.d_dst[k], stream=s, **self.kw)
                    dst.copy_(self.d_out[k], non_blocking=True)
            for s in self.streams:
                s.synchronize()

    def _run_jpeg(self, host_frames, host_outputs):
        lens = [torch.empty((), dtype=torch.int64).pin_memory() for _ in host_frames]
        landed = [None] * len(host_frames)
        out = [0] * len(host_frames)

        def download(i):                   # frame i's length has been copied: copy exactly that many bytes
            landed[i].synchronize()
            n = out[i] = int(lens[i])
            k = i % self.depth
            with torch.cuda.stream(self.streams[k]):
                host_outputs[i][:n].copy_(self.d_jpeg[k][:n], non_blocking=True)

        with torch.cuda.device(self.device):
            for i, src in enumerate(host_frames):
                k = i % self.depth
                s = self.streams[k]
                with torch.cuda.stream(s):
                    self.d_in[k].copy_(src, non_blocking=True)
                    engine.develop(self.d_in[k], out_tensor=self.d_dst[k], stream=s, **self.kw)
                    if self.jpeg_rgb:
                        _, n = engine.encode_jpeg_rgb(self.d_dst[k], self.jpeg_quality, self.jpeg_subsampling,
                                                      out_tensor=self.d_jpeg[k], stream=s)
                    else:
                        _, n = engine.encode_jpeg(self.d_dst[k], self.jpeg_quality, out_tensor=self.d_jpeg[k], stream=s)
                    lens[i].copy_(n, non_blocking=True)
                    landed[i] = torch.cuda.Event()
                    landed[i].record(s)
                if i - (self.depth - 1) >= 0:
                    download(i - (self.depth - 1))
            for i in range(max(0, len(host_frames) - (self.depth - 1)), len(host_frames)):
                download(i)
            for s in self.streams:
                s.synchronize()
        return out

    def run_copies_only(self, host_frames, host_outputs, nbytes=None):
        """The copies of `run` without the kernels: the same pinned buffers, byte counts, streams and order, one
        cudaMemcpyAsync per copy (what `Tensor.copy_(non_blocking=True)` issues between pinned host and device memory).
        Its rate is the ceiling the host <-> device path of this box puts on `run`.  For out="jpeg", `nbytes[i]` is the
        length of frame i's file (what `run` returned): that many bytes are copied down."""
        assert len(host_frames) == len(host_outputs)
        with torch.cuda.device(self.device):
            for i, (src, dst) in enumerate(zip(host_frames, host_outputs)):
                k = i % self.depth
                with torch.cuda.stream(self.streams[k]):
                    self.d_in[k].copy_(src, non_blocking=True)
                    if self.jpeg:
                        dst[:nbytes[i]].copy_(self.d_jpeg[k][:nbytes[i]], non_blocking=True)
                    else:
                        dst.copy_(self.d_out[k], non_blocking=True)
            for s in self.streams:
                s.synchronize()
