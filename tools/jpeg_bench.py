"""Raw -> JPEG on one GPU, against the host encode it replaces, in one process with the arms alternating round by round:
  device    ms per frame on device-resident frames (CUDA events): develop(out="ycc420") alone, and develop + encode_jpeg at
            qualities 75 / 90 / 95; the encoded bytes per pixel;
  kernels   device time per frame of each kernel of the chain (torch.profiler, in a pass of its own after the timed rounds);
  e2e       FramePipeline.run from pinned host frames to pinned host outputs (3 streams) for out = "jpeg" (quality 90),
            "ycc420" and "srgb_u8", each next to its copies-only ceiling (FramePipeline.run_copies_only);
  pillow    Pillow's (libjpeg-turbo) encode of the same frames' srgb_u8 images, 4:2:0, on 1 thread and on all host threads;
  checked   each frame's device file equals Pillow's JPEG of its srgb_u8 image (W = 6000 is a multiple of 16) at every
            quality, and every pipeline output equals the engine's file.
Workload: bench.py's 8 distinct synthetic 6000x4000 14-bit RGGB frames, QualityDemosaic.Best, postprocess_stages = 1.  The
GPU's name and power limit are read in the same process.
    python tools/jpeg_bench.py [--rounds 5] [--out result.json]      # one JSON object on stdout
"""
import argparse
import concurrent.futures as cf
import io
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")]
from pysp_b200 import engine, parallel, synthetic as syn  # noqa: E402
from pysp_b200.colour import cam_to_rgb_matrix  # noqa: E402
from pysp_b200.pipeline import FramePipeline  # noqa: E402
from pysp_b200.wb_cct import CameraWhiteBalance  # noqa: E402
from ycc_bench import gpu_identity  # noqa: E402

H, W, FRAMES, STAGES = 4000, 6000, 8, 1
QUALITIES = (75, 90, 95)
PIPE_Q = 90
KINDS = ("jpeg", "ycc420", "srgb_u8")


def pillow_jpeg(s8, q):
    from PIL import Image
    b = io.BytesIO()
    Image.fromarray(s8).save(b, format="JPEG", quality=q, subsampling=2)
    return b.getvalue()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=5, help="passes over the frames per device-resident timing")
    ap.add_argument("--steps", type=int, default=5, help="passes over the frames per e2e timing")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "tools/jpeg_bench.py needs a GPU"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    numa = parallel.bind_to_gpu_numa_node(0)
    cam_wb = CameraWhiteBalance(syn.MAT_XYZ_TO_CAM, syn.WHITE_XYZ)
    kw = dict(wb=cam_wb.get_reciprocal_multipliers(), cam_to_srgb=cam_to_rgb_matrix(cam_wb.get_matrix()), stages=STAGES,
              black=syn.BLACK, white=syn.WHITE)
    base = syn.scene_base(H, W)
    host = [torch.from_numpy(syn.scene(H, W, seed=i, base=base).view(np.int16)) for i in range(FRAMES)]
    frames = [h.to(dev) for h in host]
    planes = [engine.i420_planes(torch.empty(engine.i420_bytes(H, W), dtype=torch.uint8, device=dev), H, W) for _ in range(2)]
    jbuf = [torch.empty(engine.jpeg_max_bytes(H, W), dtype=torch.uint8, device=dev) for _ in range(2)]
    lens = {}

    def one_pass(q):                     # q None: the develop alone
        for i, f in enumerate(frames):
            engine.develop(f, out="ycc420", out_tensor=planes[i & 1], **kw)
            if q is not None:
                lens[(q, i)] = engine.encode_jpeg(planes[i & 1], q, out_tensor=jbuf[i & 1])[1]

    def device_ms_per_frame(q):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(args.reps):
            one_pass(q)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / (args.reps * FRAMES)

    arms = (None,) + QUALITIES
    pin_in = [h.pin_memory() for h in host]
    pipes = {k: FramePipeline(H, W, out=k, device=dev, jpeg_quality=PIPE_Q, **kw) for k in KINDS}
    pin_out = {k: [pipes[k].pinned_output() for _ in range(FRAMES)] for k in KINDS}
    for q in arms:                                   # warm-up of every timed shape
        one_pass(q)
    jlens = pipes["jpeg"].run(pin_in, pin_out["jpeg"])
    for k in KINDS:
        pipes[k].run(pin_in, pin_out[k])
        pipes[k].run_copies_only(pin_in, pin_out[k], jlens if k == "jpeg" else None)
    torch.cuda.synchronize()

    def timed_s(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    dev_ms = {str(q): [] for q in arms}
    e2e = {k: {"e2e_s": [], "copies_s": []} for k in KINDS}
    for r in range(args.rounds):
        for q in (arms if r % 2 == 0 else arms[::-1]):
            dev_ms[str(q)].append(device_ms_per_frame(q))
        for k in (KINDS if r % 2 == 0 else KINDS[::-1]):
            p, o = pipes[k], pin_out[k]
            e2e[k]["e2e_s"].append(timed_s(lambda: p.run(pin_in, o)))
            e2e[k]["copies_s"].append(timed_s(lambda: p.run_copies_only(pin_in, o, jlens if k == "jpeg" else None)))

    # encoded sizes, and the check against Pillow's encode of srgb_u8 (which is also the host encode timed below)
    s8 = [engine.develop(f, out="srgb_u8", **kw).cpu().numpy() for f in frames]
    checked, bpp = {}, {}
    for q in QUALITIES:
        one_pass(q)
        torch.cuda.synchronize()
        sizes = [int(lens[(q, i)].item()) for i in range(FRAMES)]
        bpp[str(q)] = round(float(np.mean(sizes)) / (H * W), 4)
        ok = True
        for i, f in enumerate(frames):
            buf, n = engine.encode_jpeg(engine.develop(f, out="ycc420", **kw), q)
            ok = ok and bytes(buf[:int(n.item())].cpu().numpy()) == pillow_jpeg(s8[i], q)
        checked["device_file_equals_pillow_of_srgb_u8_q%d" % q] = bool(ok)
    jlens = pipes["jpeg"].run(pin_in, pin_out["jpeg"])
    ok = all(bytes(pin_out["jpeg"][i][:jlens[i]].numpy()) == pillow_jpeg(s8[i], PIPE_Q) for i in range(FRAMES))
    checked["pipeline_jpeg_equals_pillow_of_srgb_u8"] = bool(ok)

    # Pillow on the host: 1 thread, then all threads, same frames
    threads = os.cpu_count() or 1
    pil = {}
    for q in QUALITIES:
        t0 = time.perf_counter()
        for s in s8:
            pillow_jpeg(s, q)
        one = time.perf_counter() - t0
        with cf.ThreadPoolExecutor(threads) as ex:
            list(ex.map(lambda s: pillow_jpeg(s, q), s8))           # warm the pool
            t0 = time.perf_counter()
            list(ex.map(lambda s: pillow_jpeg(s, q), s8 * 2))
            allt = (time.perf_counter() - t0) / 2
        pil[str(q)] = {"ms_per_frame_1_thread": round(1e3 * one / FRAMES, 2),
                       "gpix_s_1_thread": round(FRAMES * H * W / one / 1e9, 4),
                       "ms_per_frame_all_threads": round(1e3 * allt / FRAMES, 2),
                       "gpix_s_all_threads": round(FRAMES * H * W / allt / 1e9, 4)}

    # per-kernel device time: a profiled pass of its own (the profiler slows the host; the timed numbers above are without it)
    from torch.profiler import ProfilerActivity, profile
    kernels = {}
    for q in QUALITIES:
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            one_pass(q)
            torch.cuda.synchronize()
        per = {}
        for e in prof.key_averages():
            if e.device_type.name == "CUDA" and ("kernel" in e.key):
                name = e.key.split("(")[0].split("<")[0].replace("void ", "").replace("pysp::", "")
                per[name] = per.get(name, 0.0) + e.self_device_time_total / 1e3 / FRAMES
        kernels[str(q)] = {k: round(v, 4) for k, v in sorted(per.items(), key=lambda kv: -kv[1])}

    med = {q: float(np.median(v)) for q, v in dev_ms.items()}
    px = H * W
    res = {"gpu": gpu_identity(), "torch": torch.__version__, "cuda": torch.version.cuda, "numa_node": numa,
           "host_threads": threads,
           "workload": "8 distinct synthetic 6000x4000 14-bit RGGB frames (bench.py's), QualityDemosaic.Best, postprocess_stages=1",
           "rounds": args.rounds, "device_reps": args.reps, "e2e_steps": args.steps, "checked": checked,
           "device_ms_per_frame": {("ycc420_develop" if q == "None" else "develop_plus_encode_q" + q): round(v, 4)
                                   for q, v in med.items()},
           "encode_ms_per_frame": {"q" + q: round(med[q] - med["None"], 4) for q in map(str, QUALITIES)},
           "encoded_bytes_per_pixel": bpp, "kernel_ms_per_frame": kernels, "pillow_host_encode": pil,
           "device_samples_ms": {k: [round(x, 4) for x in v] for k, v in dev_ms.items()}, "e2e": {}}
    for k in KINDS:
        m = {n: float(np.median(v)) for n, v in e2e[k].items()}
        nfr = args.steps * FRAMES
        res["e2e"][k] = {"e2e_gpix_s": round(nfr * px / m["e2e_s"] / 1e9, 2),
                         "copies_only_ceiling_gpix_s": round(nfr * px / m["copies_s"] / 1e9, 2),
                         "d2h_bytes_per_frame": (int(np.mean(jlens)) if k == "jpeg" else pipes[k].d2h_bytes()),
                         "samples_s": {n: [round(x, 4) for x in v] for n, v in e2e[k].items()}}
    res["e2e"]["jpeg"]["quality"] = PIPE_Q
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
