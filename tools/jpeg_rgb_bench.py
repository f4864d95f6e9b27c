"""RGB -> JPEG at 4:4:4, 4:2:2 and 4:2:0 on one GPU (engine.encode_jpeg_rgb), against the host encode it replaces, in one
process with the arms alternating round by round:
  encode    ms per frame of encode_jpeg_rgb on device-resident srgb_u8 frames (CUDA events), per subsampling and quality 75 /
            90 / 95, next to the existing encode_jpeg of the same frames' ycc420 planes (4:2:0); encoded bytes per pixel;
  chain     ms per frame of develop(out="srgb_u8") + encode_jpeg_rgb, and of develop alone;
  kernels   device time per frame of each encode kernel (torch.profiler, in a pass of its own after the timed rounds);
  e2e       FramePipeline(out="jpeg", jpeg_subsampling=...) from pinned raw frames to pinned host files (3 streams, quality 90),
            next to its copies-only ceiling (FramePipeline.run_copies_only);
  pillow    Pillow's (libjpeg-turbo) encode of the same srgb_u8 images at the same subsampling, on 1 thread and on all threads;
  checked   every device file equals Pillow's, every pipeline output equals the engine's file.
Workload: bench.py's 8 distinct synthetic 6000x4000 14-bit RGGB frames, QualityDemosaic.Best, postprocess_stages = 1.  The
GPU's name and power limit are read in the same process.
    python tools/jpeg_rgb_bench.py [--rounds 3] [--out result.json]      # one JSON object on stdout
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
SUBS = ("4:4:4", "4:2:2", "4:2:0")
PIPE_Q = 90


def pillow_jpeg(s8, q, s):
    from PIL import Image
    b = io.BytesIO()
    Image.fromarray(s8).save(b, format="JPEG", quality=q, subsampling=SUBS.index(s))
    return b.getvalue()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5, help="passes over the frames per device-resident timing")
    ap.add_argument("--steps", type=int, default=3, help="passes over the frames per e2e timing")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "tools/jpeg_rgb_bench.py needs a GPU"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    numa = parallel.bind_to_gpu_numa_node(0)
    cam_wb = CameraWhiteBalance(syn.MAT_XYZ_TO_CAM, syn.WHITE_XYZ)
    kw = dict(wb=cam_wb.get_reciprocal_multipliers(), cam_to_srgb=cam_to_rgb_matrix(cam_wb.get_matrix()), stages=STAGES,
              black=syn.BLACK, white=syn.WHITE)
    base = syn.scene_base(H, W)
    host = [torch.from_numpy(syn.scene(H, W, seed=i, base=base).view(np.int16)) for i in range(FRAMES)]
    frames = [h.to(dev) for h in host]
    s8 = [engine.develop(f, out="srgb_u8", **kw) for f in frames]           # resident inputs of the encode-only timings
    ycc = [engine.develop(f, out="ycc420", **kw) for f in frames]
    sbuf = [torch.empty((H, W, 3), dtype=torch.uint8, device=dev) for _ in range(2)]
    jbuf = [torch.empty(engine.jpeg_rgb_max_bytes(H, W, "4:4:4"), dtype=torch.uint8, device=dev) for _ in range(2)]
    lens = {}

    # arms: ("develop", None, None), ("chain", s, q), ("rgb", s, q), ("planes", "4:2:0", q)
    def one_pass(arm):
        what, s, q = arm
        for i in range(FRAMES):
            if what in ("develop", "chain"):
                engine.develop(frames[i], out="srgb_u8", out_tensor=sbuf[i & 1], **kw)
                if what == "chain":
                    engine.encode_jpeg_rgb(sbuf[i & 1], q, s, out_tensor=jbuf[i & 1])
            elif what == "rgb":
                lens[(s, q, i)] = engine.encode_jpeg_rgb(s8[i], q, s, out_tensor=jbuf[i & 1])[1]
            else:
                lens[("planes", q, i)] = engine.encode_jpeg(ycc[i], q, out_tensor=jbuf[i & 1])[1]

    def device_ms_per_frame(arm):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(args.reps):
            one_pass(arm)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / (args.reps * FRAMES)

    arms = [("develop", None, None)] + [(w, s, q) for w in ("rgb", "chain") for s in SUBS for q in QUALITIES] + \
        [("planes", "4:2:0", q) for q in QUALITIES]
    key = lambda arm: "_".join(str(x) for x in arm if x is not None)      # noqa: E731
    pin_in = [h.pin_memory() for h in host]
    pipes = {s: FramePipeline(H, W, out="jpeg", device=dev, jpeg_quality=PIPE_Q, jpeg_subsampling=s, **kw) for s in SUBS}
    pin_out = {s: [pipes[s].pinned_output() for _ in range(FRAMES)] for s in SUBS}
    for arm in arms:                                 # warm-up of every timed shape
        one_pass(arm)
    plens = {}
    for s in SUBS:
        plens[s] = pipes[s].run(pin_in, pin_out[s])
        pipes[s].run_copies_only(pin_in, pin_out[s], plens[s])
    torch.cuda.synchronize()

    def timed_s(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    dev_ms = {key(a): [] for a in arms}
    e2e = {s: {"e2e_s": [], "copies_s": []} for s in SUBS}
    for r in range(args.rounds):
        for arm in (arms if r % 2 == 0 else arms[::-1]):
            dev_ms[key(arm)].append(device_ms_per_frame(arm))
        for s in (SUBS if r % 2 == 0 else SUBS[::-1]):
            p, o = pipes[s], pin_out[s]
            e2e[s]["e2e_s"].append(timed_s(lambda: p.run(pin_in, o)))
            e2e[s]["copies_s"].append(timed_s(lambda: p.run_copies_only(pin_in, o, plens[s])))

    # the files: sizes, and the check against Pillow (whose encode of the same images is timed below)
    host_s8 = [t.cpu().numpy() for t in s8]
    checked, bpp = {}, {}
    for s in SUBS:
        for q in QUALITIES:
            one_pass(("rgb", s, q))
            torch.cuda.synchronize()
            sizes, ok = [], True
            for i in range(FRAMES):
                buf, n = engine.encode_jpeg_rgb(s8[i], q, s)
                data = bytes(buf[:int(n.item())].cpu().numpy())
                sizes.append(len(data))
                ok = ok and len(data) == int(lens[(s, q, i)].item()) and data == pillow_jpeg(host_s8[i], q, s)
            bpp["%s_q%d" % (s, q)] = round(float(np.mean(sizes)) / (H * W), 4)
            checked["device_file_equals_pillow_%s_q%d" % (s, q)] = bool(ok)
        ln = pipes[s].run(pin_in, pin_out[s])
        checked["pipeline_equals_pillow_%s" % s] = all(bytes(pin_out[s][i][:ln[i]].numpy()) == pillow_jpeg(host_s8[i], PIPE_Q, s)
                                                       for i in range(FRAMES))

    threads = os.cpu_count() or 1
    pil = {}
    for s in SUBS:
        for q in QUALITIES:
            t0 = time.perf_counter()
            for x in host_s8:
                pillow_jpeg(x, q, s)
            one = time.perf_counter() - t0
            with cf.ThreadPoolExecutor(threads) as ex:
                list(ex.map(lambda x: pillow_jpeg(x, q, s), host_s8))         # warm the pool
                t0 = time.perf_counter()
                list(ex.map(lambda x: pillow_jpeg(x, q, s), host_s8 * 2))
                allt = (time.perf_counter() - t0) / 2
            pil["%s_q%d" % (s, q)] = {"ms_per_frame_1_thread": round(1e3 * one / FRAMES, 2),
                                      "ms_per_frame_all_threads": round(1e3 * allt / FRAMES, 2)}

    # per-kernel device time of the encode alone: a profiled pass of its own
    from torch.profiler import ProfilerActivity, profile
    kernels = {}
    for arm in [a for a in arms if a[0] in ("rgb", "planes")]:
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            one_pass(arm)
            torch.cuda.synchronize()
        per = {}
        for e in prof.key_averages():
            if e.device_type.name == "CUDA" and "jpeg_" in e.key:
                name = e.key.split("(")[0].split("<")[0].replace("void ", "").replace("pysp::", "")
                per[name] = per.get(name, 0.0) + e.self_device_time_total / 1e3 / FRAMES
        kernels[key(arm)] = {k: round(v, 4) for k, v in sorted(per.items(), key=lambda kv: -kv[1])}

    med = {k: float(np.median(v)) for k, v in dev_ms.items()}
    px = H * W
    res = {"gpu": gpu_identity(), "torch": torch.__version__, "cuda": torch.version.cuda, "numa_node": numa,
           "host_threads": threads,
           "workload": "8 distinct synthetic 6000x4000 14-bit RGGB frames (bench.py's), QualityDemosaic.Best, postprocess_stages=1",
           "rounds": args.rounds, "device_reps": args.reps, "e2e_steps": args.steps, "checked": checked,
           "encode_ms_per_frame": {k: round(v, 4) for k, v in med.items() if k.startswith(("rgb", "planes"))},
           "chain_ms_per_frame": {k: round(v, 4) for k, v in med.items() if k.startswith(("chain", "develop"))},
           "encoded_bytes_per_pixel": bpp, "kernel_ms_per_frame": kernels, "pillow_host_encode": pil,
           "device_samples_ms": {k: [round(x, 4) for x in v] for k, v in dev_ms.items()}, "e2e": {}}
    for s in SUBS:
        m = {n: float(np.median(v)) for n, v in e2e[s].items()}
        nfr = args.steps * FRAMES
        res["e2e"][s] = {"e2e_gpix_s": round(nfr * px / m["e2e_s"] / 1e9, 2),
                         "copies_only_ceiling_gpix_s": round(nfr * px / m["copies_s"] / 1e9, 2),
                         "d2h_bytes_per_frame": int(np.mean(plens[s])), "quality": PIPE_Q,
                         "samples_s": {n: [round(x, 4) for x in v] for n, v in e2e[s].items()}}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
