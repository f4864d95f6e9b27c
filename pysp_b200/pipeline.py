"""Host-resident batches: stream frames through one GPU with copies overlapped with the kernels.

`FramePipeline` is the public batch API: frames start and end in (pinned) HOST memory.  Each of `depth`
slots owns a CUDA stream, a device mosaic buffer and a device output buffer; frame i uses slot i % depth:
H2D copy -> fused develop chain -> D2H copy, all asynchronous on the slot's stream, so the upload of frame
i+1 and the download of frame i-1 overlap the kernels of frame i (the two copy engines run concurrently
with the SMs).  No CPU computation is involved.

With out="ycc420" each output is one flat I420 buffer of H*W*3/2 bytes (Y, then Cb, then Cr; engine.i420_planes gives the
three planes of it), so one copy moves a frame.
"""
import torch

from . import engine


class FramePipeline:
    def __init__(self, height, width, wb, cam_to_srgb, stages=1, pattern="RGGB", black=None, white=None,
                 hdr=False, gamma=False, out="lin", device=None, depth=3):
        engine.require_cuda()
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self.h, self.w = int(height), int(width)
        self.kw = dict(wb=wb, cam_to_srgb=cam_to_srgb, stages=stages, pattern=pattern, black=black, white=white,
                       hdr=hdr, gamma=gamma, out=out)
        self.out_dtype = engine._OUT_DTYPES[engine._OUT_KINDS[out]]
        self.out_shape = (engine.i420_bytes(self.h, self.w),) if out == "ycc420" else (self.h, self.w, 3)
        self.depth = depth
        with torch.cuda.device(self.device):
            self.streams = [torch.cuda.Stream() for _ in range(depth)]
            self.d_in = [torch.empty((self.h, self.w), dtype=torch.int16, device=self.device) for _ in range(depth)]
            self.d_out = [torch.empty(self.out_shape, dtype=self.out_dtype, device=self.device) for _ in range(depth)]
        # what develop writes into: the output tensor itself, or the three planes over the flat I420 buffer
        self.d_dst = [engine.i420_planes(d, self.h, self.w) if out == "ycc420" else d for d in self.d_out]

    def pinned_input(self):
        return torch.empty((self.h, self.w), dtype=torch.int16).pin_memory()

    def pinned_output(self):
        return torch.empty(self.out_shape, dtype=self.out_dtype).pin_memory()

    def h2d_bytes(self):
        return self.h * self.w * 2

    def d2h_bytes(self):
        return self.d_out[0].numel() * self.d_out[0].element_size()

    def run(self, host_frames, host_outputs):
        """host_frames[i] (int16/uint16 bits, ideally pinned) -> host_outputs[i] (pinned).  Returns after
        every output has landed in host memory."""
        assert len(host_frames) == len(host_outputs)
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

    def run_copies_only(self, host_frames, host_outputs):
        """The copies of `run` without the kernels: the same pinned buffers, byte counts, streams and order, one
        cudaMemcpyAsync per copy (what `Tensor.copy_(non_blocking=True)` issues between pinned host and device memory).
        Its rate is the ceiling the host <-> device path of this box puts on `run`."""
        assert len(host_frames) == len(host_outputs)
        with torch.cuda.device(self.device):
            for i, (src, dst) in enumerate(zip(host_frames, host_outputs)):
                k = i % self.depth
                with torch.cuda.stream(self.streams[k]):
                    self.d_in[k].copy_(src, non_blocking=True)
                    dst.copy_(self.d_out[k], non_blocking=True)
            for s in self.streams:
                s.synchronize()
