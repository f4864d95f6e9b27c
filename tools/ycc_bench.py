"""8-bit sRGB against JPEG-ready YCbCr 4:2:0 output (out="srgb_u8" vs out="ycc420") on one GPU, in one process, the two kinds
alternating round by round:
  device    ms per frame of the develop chain on device-resident frames (CUDA events);
  e2e       FramePipeline.run from pinned host frames to pinned host outputs (3 streams), next to its copies-only ceiling
            (FramePipeline.run_copies_only) and to the host-to-device and device-to-host copies alone, as bench.py's e2e leg
            measures them;
  checked   every pipeline output equals engine.develop of the same frame, and the planes of two frames equal the NumPy
            restatement (tests/ycc420_ref.py) of srgb_u8.
Workload: bench.py's 8 distinct synthetic 6000x4000 14-bit RGGB frames (8 x 48 MB of mosaic, larger than the 126 MB L2),
QualityDemosaic.Best, postprocess_stages = 1.  The GPU's name and power limit are read in the same process.
    python tools/ycc_bench.py [--rounds 5] [--out result.json]      # one JSON object on stdout
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from pysp_b200 import engine, parallel, synthetic as syn  # noqa: E402
from pysp_b200.colour import cam_to_rgb_matrix  # noqa: E402
from pysp_b200.pipeline import FramePipeline  # noqa: E402
from pysp_b200.wb_cct import CameraWhiteBalance  # noqa: E402
from ycc420_ref import ycc420  # noqa: E402

H, W, FRAMES, STAGES = 4000, 6000, 8, 1
KINDS = ("srgb_u8", "ycc420")


def gpu_identity():
    q = "name,power.limit,power.max_limit,clocks.max.sm"
    try:
        line = subprocess.run(["nvidia-smi", "--id=%d" % torch.cuda.current_device(), "--query-gpu=" + q,
                               "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), [v.strip() for v in line.split(",")]))
    except Exception as e:                       # the name from the runtime at least
        return {"name": torch.cuda.get_device_name(), "power.limit": "unavailable (%s)" % type(e).__name__}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=10, help="passes over the frames per device-resident timing")
    ap.add_argument("--steps", type=int, default=10, help="passes over the frames per e2e timing")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "tools/ycc_bench.py needs a GPU"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    numa = parallel.bind_to_gpu_numa_node(0)
    cam_wb = CameraWhiteBalance(syn.MAT_XYZ_TO_CAM, syn.WHITE_XYZ)
    kw = dict(wb=cam_wb.get_reciprocal_multipliers(), cam_to_srgb=cam_to_rgb_matrix(cam_wb.get_matrix()), stages=STAGES,
              black=syn.BLACK, white=syn.WHITE)
    base = syn.scene_base(H, W)
    host = [torch.from_numpy(syn.scene(H, W, seed=i, base=base).view(np.int16)) for i in range(FRAMES)]
    frames = [h.to(dev) for h in host]
    outs = {"srgb_u8": [torch.empty((H, W, 3), dtype=torch.uint8, device=dev) for _ in range(2)],
            "ycc420": [engine.i420_planes(torch.empty(engine.i420_bytes(H, W), dtype=torch.uint8, device=dev), H, W)
                       for _ in range(2)]}

    def one_pass(kind):
        for i, f in enumerate(frames):
            engine.develop(f, out=kind, out_tensor=outs[kind][i & 1], **kw)

    def device_ms_per_frame(kind):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(args.reps):
            one_pass(kind)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / (args.reps * FRAMES)

    pin_in = [h.pin_memory() for h in host]
    pipes = {k: FramePipeline(H, W, out=k, device=dev, **kw) for k in KINDS}
    pin_out = {k: [pipes[k].pinned_output() for _ in range(FRAMES)] for k in KINDS}

    def timed_s(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    def one_way(pipe, outs_, h2d):
        """only the uploads (h2d) or only the downloads of pipe.run_copies_only, same streams and buffers"""
        with torch.cuda.device(dev):
            for i, (src, dst) in enumerate(zip(pin_in, outs_)):
                k = i % pipe.depth
                with torch.cuda.stream(pipe.streams[k]):
                    if h2d:
                        pipe.d_in[k].copy_(src, non_blocking=True)
                    else:
                        dst.copy_(pipe.d_out[k], non_blocking=True)
            for s in pipe.streams:
                s.synchronize()

    for k in KINDS:                                   # warm-up of every timed shape
        for _ in range(3):
            one_pass(k)
        pipes[k].run(pin_in, pin_out[k])
        pipes[k].run_copies_only(pin_in, pin_out[k])
    torch.cuda.synchronize()

    samples = {k: {"device_ms": [], "e2e_s": [], "copies_s": [], "h2d_s": [], "d2h_s": []} for k in KINDS}
    for r in range(args.rounds):
        order = KINDS if r % 2 == 0 else KINDS[::-1]
        for k in order:
            samples[k]["device_ms"].append(device_ms_per_frame(k))
        for k in order:
            p, o = pipes[k], pin_out[k]
            samples[k]["e2e_s"].append(timed_s(lambda: p.run(pin_in, o)))
            samples[k]["copies_s"].append(timed_s(lambda: p.run_copies_only(pin_in, o)))
            samples[k]["h2d_s"].append(timed_s(lambda: one_way(p, o, True)))
            samples[k]["d2h_s"].append(timed_s(lambda: one_way(p, o, False)))

    # outputs: the pipeline delivered engine.develop's bytes; the planes are the restatement of srgb_u8
    checked = {}
    for k in KINDS:
        pipes[k].run(pin_in, pin_out[k])
        ok = True
        for i, f in enumerate(frames):
            want = engine.develop(f, out=k, **kw)
            if k == "ycc420":
                want = torch.cat([p.reshape(-1) for p in want])
            ok = ok and torch.equal(pin_out[k][i].to(dev).reshape(-1), want.reshape(-1))
        checked["pipeline_equals_develop_" + k] = bool(ok)
    ok = True
    for i in (0, FRAMES - 1):
        s8 = engine.develop(frames[i], out="srgb_u8", **kw).cpu().numpy()
        got = [p.cpu().numpy() for p in engine.develop(frames[i], out="ycc420", **kw)]
        ok = ok and all(np.array_equal(a, b) for a, b in zip(got, ycc420(s8)))
    checked["ycc420_equals_restatement_of_srgb_u8_frames_0_and_7"] = bool(ok)

    px = H * W
    res = {"gpu": gpu_identity(), "torch": torch.__version__, "cuda": torch.version.cuda, "numa_node": numa,
           "workload": "8 distinct synthetic 6000x4000 14-bit RGGB frames (bench.py's), QualityDemosaic.Best, "
                       "postprocess_stages=1; FramePipeline: pinned host in/out, 3 streams",
           "rounds": args.rounds, "device_reps": args.reps, "e2e_steps": args.steps, "checked": checked, "kinds": {}}
    for k in KINDS:
        s = samples[k]
        med = {n: float(np.median(v)) for n, v in s.items()}
        nfr = args.steps * FRAMES
        out_b = pipes[k].d2h_bytes()
        r = {"d2h_bytes_per_frame": out_b, "h2d_bytes_per_frame": pipes[k].h2d_bytes(),
             "device_ms_per_frame": round(med["device_ms"], 4), "device_ms_per_frame_min": round(min(s["device_ms"]), 4),
             "device_gpix_s": round(px / med["device_ms"] / 1e6, 2),
             "e2e_gpix_s": round(nfr * px / med["e2e_s"] / 1e9, 2),
             "copies_only_ceiling_gpix_s": round(nfr * px / med["copies_s"] / 1e9, 2),
             "h2d_only_gpix_s": round(nfr * px / med["h2d_s"] / 1e9, 2),
             "d2h_only_gpix_s": round(nfr * px / med["d2h_s"] / 1e9, 2),
             "h2d_GBps": round(nfr * pipes[k].h2d_bytes() / med["h2d_s"] / 1e9, 1),
             "d2h_GBps": round(nfr * out_b / med["d2h_s"] / 1e9, 1),
             "samples": {n: [round(x, 5) for x in v] for n, v in s.items()}}
        r["frac_of_ceiling"] = round(r["e2e_gpix_s"] / r["copies_only_ceiling_gpix_s"], 3)
        # what bounds e2e: the slowest of the kernels, the uploads and the downloads when each runs alone
        alone = {"kernels": r["device_gpix_s"], "host_to_device": r["h2d_only_gpix_s"], "device_to_host": r["d2h_only_gpix_s"]}
        r["slowest_alone"] = min(alone, key=alone.get)
        res["kinds"][k] = r
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
