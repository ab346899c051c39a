#!/usr/bin/env python
"""bench.py — composited frames/sec of the fused hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N ...            # the CPU path (oracle port) on host cores

One "step" = one pass of the hot path (pre-proc -> CNN -> decision/IIR -> mask upsample +
5x5 blur + alpha blend + YUYV) over `streams x batch` synthetic frames per GPU.  Streams
are independent (one context each, own CUDA stream, own IIR state), sharded over GPUs with
no data-path collective (weak scaling); NCCL is used only for the barrier and the max-over-
ranks of the timed region.  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[3]: the configuration the 720p metric / 50k-fps target is quoted on
    "meet720": dict(model="segm_full_v679.tflite", W=1280, H=720, desc="segm_full_v679 (Meet 144x256), 1280x720 streams"),
    # configs[1]
    "mlkit480": dict(model="selfiesegmentation_mlkit-256x256-2021_01_19-v1215.f16.tflite", W=640, H=480, desc="MLKit-256, 640x480 stream"),
    # configs[2]
    "deeplab720": dict(model="deeplabv3_257_mv_gpu.tflite", W=1280, H=720, desc="deeplabv3_257_mv_gpu, 1280x720 stream"),
    # configs[4]: 4k camera frames over an animated (video) background — one decoded background image per camera frame
    "bodypix4k": dict(model="body-pix-float-050-8.tflite", W=3840, H=2160, animated="rotating_earth.webm", streams=4, batch=8,
                      desc="body-pix-float-050-8, 3840x2160 stream, animated 960x540 webm background"),
    "mlkit720": dict(model="selfiesegmentation_mlkit-256x256-2021_01_19-v1215.f16.tflite", W=1280, H=720, desc="MLKit-256, 1280x720 stream"),
}
METRIC = "composited frames/sec"
UNIT = "frames/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="meet720", choices=list(WORKLOADS))
    ap.add_argument("--streams", type=int, default=None, help="independent streams (contexts) per GPU (default 8; 4 at 4k)")
    ap.add_argument("--batch", type=int, default=None, help="consecutive frames per stream per step (default 32; 8 at 4k)")
    ap.add_argument("--bgblur", type=int, default=0, help="`-p bgblur:k` of the reference: Gaussian-blur the background (odd k)")
    ap.add_argument("--camera-blur", action="store_true", help="with --bgblur: no background source, blur the camera frame itself")
    ap.add_argument("--tensor-cores", action="store_true", help="tcgen05 3xTF32 1x1 convs for any model (default only for DeepLab / BodyPix)")
    ap.add_argument("--exact", action="store_true", help="fp32 FFMA 1x1 convs everywhere (BSB_FLAG_EXACT: bit-identical to the oracle)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-hugepages", action="store_true", help="end-to-end staging buffers on 2 MB transparent huge pages + cudaHostRegister instead of cudaHostAlloc")
    ap.add_argument("--no-configs", action="store_true", help="skip the short runs of the other BASELINE configs (parsed.configs)")
    ap.add_argument("--frames", default="person", choices=["person", "noise", "const"], help="synthetic stream kind (SURVEY 8d)")
    ap.add_argument("--launches-per-step", type=int, default=20, help="graph launches per stream per timed step (lengthens the timed window)")
    ap.add_argument("--tune", action="append", default=[], metavar="NAME=VALUE", help="bsb_set_tuning switch (A/B runs): pw_variant, dw_plane, post_tma, ...")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step (a seeded sample of pixels) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs records the outputs of the b200 path only")
    return args


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


RING_FRAMES = 16


def background_ring(wl):
    """Decoded frames of the animated background (cv2/FFmpeg on the host, like app/background.cc:126-176);
    a rolled still image if the container's cv2 cannot decode VP9."""
    from tests import synth
    path = os.path.join(ROOT, "backgrounds", wl["animated"])
    frames = []
    try:
        import cv2
        cap = cv2.VideoCapture(path)
        while len(frames) < RING_FRAMES:
            ok, f = cap.read()
            if not ok:
                break
            frames.append(f)
    except Exception:
        frames = []
    if len(frames) == RING_FRAMES:
        return np.stack(frames), f"{wl['animated']} (first {RING_FRAMES} decoded frames, one per camera frame)"
    still = synth.background()
    return np.stack([np.roll(still, 16 * i, axis=1) for i in range(RING_FRAMES)]), "synthetic ring (video decode unavailable)"


def synthetic_frames(W, H, n, stream, kind="person"):
    from tests import synth
    return np.stack([synth.frame(W, H, t=t, stream=stream, kind=kind) for t in range(n)])


def synthetic_yuyv(W, H, n, stream, kind="person"):
    from tests import synth
    return np.stack([synth.yuyv_frame(W, H, t=t, stream=stream, kind=kind) for t in range(n)])


# ----------------------------------------------------------------------------------------
# CPU path: the oracle port of the reference's TFLite+OpenCV pipeline, frame-parallel over
# host threads (the reference itself cannot be built offline — SURVEY.md §8c).
# ----------------------------------------------------------------------------------------
def cpu_path_fps(wl, threads, frames_per_thread, warm=1, bgblur=0, camera_blur=False):
    from oracle import pyoracle as po
    from tests import synth
    model = os.path.join(ROOT, "models", wl["model"])
    W, H = wl["W"], wl["H"]
    ring = background_ring(wl)[0] if wl.get("animated") else synth.background()[None]
    gens = [po.MaskGen(model, W, H) for _ in range(threads)]
    frames = [synthetic_frames(W, H, frames_per_thread + warm, s) for s in range(min(threads, 4))]

    # camera frames arrive as YUYV (the reference lets cv::VideoCapture convert them, app/deepseg.cc:553)
    frames = [np.stack([po.convert_rgb_to_yuyv(f) for f in fr]) for fr in frames]

    def work(i, lo, hi):
        g, fr = gens[i], frames[i % len(frames)]
        for t in range(lo, hi):
            g.composite_ex(po.yuyv_to_bgr(fr[t]), None if camera_blur else ring[t % len(ring)], bgblur=bgblur, want_yuyv=True, reuse=True)

    def run(lo, hi):
        th = [threading.Thread(target=work, args=(i, lo, hi)) for i in range(threads)]
        t0 = time.perf_counter()
        for t in th: t.start()
        for t in th: t.join()
        return time.perf_counter() - t0

    run(0, warm)
    dt = run(warm, warm + frames_per_thread)
    return threads * frames_per_thread / dt, dt


def cnn_calibration(wl):
    """How far the scalar oracle port is from optimised CPU inference kernels, on the CNN alone and on one thread:
    the port, a torch fp32 (oneDNN) evaluation of the same .tflite graph, and — where its importer accepts the
    graph — OpenCV dnn.  Informative only: the reference's own TFLite-XNNPACK build is not available offline."""
    out = {}
    try:
        import torch
        from oracle import pyoracle as po
        from tests import torch_graph
        model = os.path.join(ROOT, "models", wl["model"])
        m = po.Model(model)
        h, w, c = m.shape(m.input)[1:]
        x = np.random.default_rng(0).random((h, w, c), dtype=np.float32)

        def best(fn, n=3):
            fn()
            ts = []
            for _ in range(n):
                t0 = time.perf_counter(); fn(); ts.append(time.perf_counter() - t0)
            return min(ts) * 1e3
        out["port_cnn_ms"] = best(lambda: m.invoke(x))
        nt = torch.get_num_threads()
        torch.set_num_threads(1)
        out["torch_fp32_cnn_ms"] = best(lambda: torch_graph.run(model, x, dtype=torch.float32))
        torch.set_num_threads(nt)
        try:
            if "selfie" not in wl["model"]:
                raise RuntimeError("OpenCV's TFLite importer rejects the Meet graphs and drops the dilation of DeepLab / BodyPix")
            import cv2
            net = cv2.dnn.readNetFromTFLite(model)
            cv2.setNumThreads(1)
            blob = np.ascontiguousarray(x.transpose(2, 0, 1)[None])

            def f():
                net.setInput(blob); net.forward()
            out["opencv_dnn_cnn_ms"] = best(f)
            cv2.setNumThreads(-1)
        except Exception:
            out["opencv_dnn_cnn_ms"] = None            # importer rejects this graph (Meet) or ignores dilation (DeepLab / BodyPix)
        out["note"] = "single thread, CNN only; the model card quotes ~120 frames/s (8 ms) for Meet on TFLite-XNNPACK"
    except Exception as e:  # calibration is optional
        out["error"] = str(e)[:120]
    return out


def tflite_probe():
    """BASELINE.md section 3 step 1: is a real TFLite runtime importable on this box?  (It is not in this image; when one
    is, cpu_path_fps should be pointed at it — recorded so the reader knows which CPU arm ran.)"""
    found = []
    for mod in ("tflite_runtime.interpreter", "ai_edge_litert.interpreter", "tensorflow.lite"):
        try:
            __import__(mod)
            found.append(mod)
        except Exception:
            pass
    return {"importable": found, "used": "oracle port" if not found else "oracle port (runtime found but the XNNPACK arm is not wired up)"}


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_reference(args, wl):
    rank, world, _ = dist_env()
    if rank != 0:
        return
    cores = host_cores()
    threads = max(1, min(cores, 64))
    # calibrate one frame, then size each step to ~ (120 s / (steps + warmup)) of wall time at most
    kw = dict(bgblur=args.bgblur, camera_blur=args.camera_blur)
    fps1, _ = cpu_path_fps(wl, 1, 1, warm=1, **kw)
    budget = 100.0 / max(1, args.steps + args.warmup)
    fpt = max(1, int(min(4, budget * fps1)))
    vals = []
    for s in range(args.warmup + args.steps):
        fps, dt = cpu_path_fps(wl, threads, fpt, warm=0, **kw)
        if s >= args.warmup:
            vals.append((fps, dt))
    total_frames = threads * fpt * len(vals)
    total_time = sum(dt for _, dt in vals)
    value = total_frames / total_time
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total_time / len(vals), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32+u8", "data": "synthetic",
        "config": workload_config(wl, args, 0, 0, 0, 1, {"frames_per_step": threads * fpt}),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{threads} threads x {fpt} frame(s) per step, oracle port of TFLite-reference kernels + OpenCV ops",
                         "tflite_probe": tflite_probe()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(gpu)],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if not self.p:
            return None
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill(); return None
        sm, mx, reasons = [], [], set()
        for ln in out.strip().splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return None
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


def bind_near_gpu(torch, dev):
    """Pin this rank (and the pinned buffers it is about to allocate) to the CPUs NVML reports as local to
    its GPU, so host<->device copies do not cross the socket interconnect.  Returns the previous affinity."""
    old = os.sched_getaffinity(0)
    try:
        import pynvml
        pynvml.nvmlInit()
        uuid = "GPU-" + str(torch.cuda.get_device_properties(dev).uuid)
        try:
            h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(dev)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (max(old) + 64) // 64)
        cpus = {i * 64 + b for i, m in enumerate(words) for b in range(64) if (m >> b) & 1} & old
        if cpus:
            os.sched_setaffinity(0, cpus)
    except Exception:
        pass
    return old


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def post_bytes(W, H, ow, oh, B, yuyv_in, bg_per_frame, bg_cache):
    """Algorithmic HBM bytes of ONE launch of the fused blur+composite kernel over B frames (SURVEY 8d; `bg_cache` is
    accepted for the record only):
    per frame: camera frame in (3WH as BGR, 2WH when the kernel reads the camera YUYV itself) + RGB composite out (3WH) +
    YUYV out (2WH) + full-resolution mask out (WH) + the small mask (ow*oh);
    background: 3WH per frame for an animated / per-frame background, but ONCE per launch for a still image (every frame
    of the launch blends the same L2-resident image; round 1 counted it per frame, which overstated the fraction)."""
    npx = W * H
    per_frame = (2 if yuyv_in else 3) * npx + 3 * npx + 2 * npx + npx + ow * oh
    bg = 3 * npx          # the cached YUYV copy of the background is this implementation's own extra traffic: not counted
    return B * per_frame + (B * bg if bg_per_frame else bg)


DUMP_PIXELS = 1 << 20        # sampled pixels of --dump-outputs: 6 float32 values + 1 float64 index each, 32 MB in all


def dump_outputs(path, slots, B, H, W):
    """--dump-outputs: what one step returned to its caller (RGB composite, YUYV frame and mask of every stream's batch),
    `slots` holding one ring slot per stream, written as float32 for a fixed, seeded sample of DUMP_PIXELS pixels (all
    pixels if there are fewer).  pixel_index.npy holds each sample's flat index into [stream, frame, y, x]."""
    import torch
    os.makedirs(path, exist_ok=True)
    per = B * H * W
    total = len(slots) * per
    idx = np.arange(total) if total <= DUMP_PIXELS else np.unique(np.random.default_rng(0).integers(0, total, DUMP_PIXELS))
    parts = {"composite": [], "yuyv": [], "mask": []}
    for s, sl in enumerate(slots):
        sel = torch.from_numpy(idx[(idx >= s * per) & (idx < (s + 1) * per)] - s * per).to(sl["d_out"].device)
        parts["composite"].append(sl["d_out"].view(per, 3)[sel])
        parts["yuyv"].append(sl["d_yuyv"].view(per, 2)[sel])
        parts["mask"].append(sl["d_mask"].view(per)[sel])
    for name, p in parts.items():
        np.save(os.path.join(path, name + ".npy"), torch.cat(p).cpu().numpy().astype(np.float32))
    np.save(os.path.join(path, "pixel_index.npy"), idx.astype(np.float64))


def measure(args, wl, key, dev, rank, world, S, B, steps, warmup, lps, with_e2e, with_clocks, kind="person", dump_dir=None):
    """One workload on this rank's GPU: device-resident throughput, optional end-to-end, per-stage times, rooflines."""
    import torch

    import backscrub_b200 as bs
    from backscrub_b200 import sharding
    from tests import synth

    W, H = wl["W"], wl["H"]
    model = os.path.join(ROOT, "models", wl["model"])
    fb, npx = W * H * 3, W * H
    R = 2                                     # ring slots per stream: S*R*B frames in + out exceed the 126 MB L2
    bg = synth.background()
    bg_desc = "still 1280x720 PNG (resized once; read from L2)"
    ring_frames = None
    if wl.get("animated"):
        ring_frames, bg_desc = background_ring(wl)
    if args.camera_blur:
        bg_desc = "none: the Gaussian-blurred camera frame (app/deepseg.cc:652-658)"
    my_streams = sharding.streams_for_rank(world * S, rank, world)      # stream ids served by this GPU
    ctxs, rings = [], []
    for s in range(S):
        c = bs.bs_maskgen_new(model, 2, W, H, device=dev, max_batch=B, flags=(4 if args.tensor_cores else 0) | (16 if args.exact else 0))
        if ring_frames is not None and not args.camera_blur:
            c.set_background_ring(ring_frames, advance=1)
        elif not args.camera_blur:
            c.set_background(bg)
        if args.bgblur:
            c.set_bgblur(args.bgblur)
        ctxs.append(c)
        host = synthetic_yuyv(W, H, B, stream=my_streams[s], kind=kind)     # camera-format input frames (plain numpy)
        slots = []
        for r in range(R):
            d_in = torch.from_numpy(host).to(f"cuda:{dev}")
            slots.append(dict(d_in=d_in, d_out=torch.empty((B, H, W, 3), dtype=torch.uint8, device=f"cuda:{dev}"),
                              d_yuyv=torch.empty((B, H, W, 2), dtype=torch.uint8, device=f"cuda:{dev}"),
                              d_mask=torch.empty((B, H, W), dtype=torch.uint8, device=f"cuda:{dev}")))
        rings.append(dict(host=host, slots=slots))
    ext = [torch.cuda.ExternalStream(c.stream, device=dev) for c in ctxs]

    def step(i):
        for l in range(lps):
            r = (i * lps + l) % R
            for s, c in enumerate(ctxs):
                sl = rings[s]["slots"][r]
                c.composite_yuyv_device(B, sl["d_in"].data_ptr(), sl["d_out"].data_ptr(), sl["d_yuyv"].data_ptr(), sl["d_mask"].data_ptr())

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
            torch.cuda.synchronize()

    # ---- device-resident throughput (`value`) ----
    sampler = ClockSampler(dev) if (with_clocks and rank == 0) else None      # samples through the value + e2e regions
    for i in range(warmup):
        step(i)
    barrier()
    ev0 = torch.cuda.Event(enable_timing=True)
    ev1 = [torch.cuda.Event(enable_timing=True) for _ in ctxs]
    ev0.record(ext[0])
    for e in ext[1:]:
        e.wait_event(ev0)
    for i in range(steps):
        step(warmup + i)
    for e, s in zip(ev1, ext):
        e.record(s)
    barrier()
    ms = max(ev0.elapsed_time(e) for e in ev1)
    if dump_dir:
        last = ((warmup + steps) * lps - 1) % R            # ring slot written by the last launch of the last timed step
        dump_outputs(dump_dir, [rg["slots"][last] for rg in rings], B, H, W)
    frames_total, secs, value = sharding.reduce_throughput(S * B * lps * steps, ms * 1e-3,
                                                            torch.distributed if world > 1 else None, f"cuda:{dev}")
    ms = secs * 1e3

    # ---- end to end through the host-buffer C-ABI call (H2D + graph + D2H every step) ----
    e2e = None
    if with_e2e:
        keep = []

        def pin(shape):
            """page-locked staging buffer allocated (first-touched) on this rank's NUMA node"""
            if not args.e2e_hugepages:
                t = torch.empty(shape, dtype=torch.uint8).pin_memory()
                keep.append(t)
                return t.numpy()
            import ctypes
            import mmap
            n = int(np.prod(shape))
            size = (n + (2 << 20) - 1) // (2 << 20) * (2 << 20)
            mm = mmap.mmap(-1, size, flags=mmap.MAP_PRIVATE | mmap.MAP_ANONYMOUS)
            try:
                mm.madvise(mmap.MADV_HUGEPAGE)
            except Exception:
                pass
            arr = np.frombuffer(mm, dtype=np.uint8, count=n).reshape(shape)
            arr[...] = 0
            rt = ctypes.CDLL("libcudart.so.12")
            rt.cudaHostRegister.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint]
            rc = rt.cudaHostRegister(arr.ctypes.data, size, 0)
            if rc != 0:
                raise RuntimeError(f"cudaHostRegister failed: {rc}")
            keep.append((mm, rt))
            return arr
        hb = []
        for s in range(S):
            h_in = pin((B, H, W, 2)); h_in[:] = rings[s]["host"]
            hb.append(dict(inp=h_in, yuyv=pin((B, H, W, 2))))
        e_steps = max(3, steps * lps // 2)

        def worker(s, n):
            for _ in range(n):
                # the frame deepseg.cc hands to the loopback device is the YUYV one (app/deepseg.cc:681-690)
                ctxs[s].composite_yuyv_into(hb[s]["inp"], yuyv=hb[s]["yuyv"])

        def run_threads(n):
            th = [threading.Thread(target=worker, args=(s, n)) for s in range(S)]
            for t in th: t.start()
            for t in th: t.join()

        run_threads(2)
        barrier()
        t0 = time.perf_counter()
        run_threads(e_steps)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device=f"cuda:{dev}")
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            dt = float(t.item())
        e2e = {"value": world * S * B * e_steps / dt, "unit": UNIT, "h2d_bytes_per_step": S * B * npx * 2,
               "d2h_bytes_per_step": S * B * npx * 2, "steps": e_steps, "frames_per_step": world * S * B,
               "pcie_gbs_each_direction": world * S * B * e_steps * npx * 2 / dt / 1e9 / world,
               "host_buffers": "2 MB huge pages + cudaHostRegister" if args.e2e_hugepages else "cudaHostAlloc (torch pin_memory)",
               "input": "camera YUYV frame in pinned host memory (read in place by the GPU kernels; app/deepseg.cc:553 converts it on the CPU)",
               "result": "YUYV frame (what app/deepseg.cc:681-690 writes to the v4l2 loopback device)"}

    if sampler:
        # keep the GPU under the same load until nvidia-smi has delivered a few samples (it needs ~0.3 s to start)
        t_end = time.perf_counter() + 1.0
        i = 0
        while time.perf_counter() < t_end:
            step(warmup + steps + i); i += 1
            if i % 4 == 0:
                torch.cuda.synchronize()
        torch.cuda.synchronize()
    clocks = sampler.stop() if sampler else None

    # ---- per-stage device times + rooflines ----
    stages = {}
    c0 = ctxs[0]
    # bsb_time_stage replays the kernels on the context-owned buffers: fill them with a real batch first (the
    # device-pointer steps above never touch them), so the stage times are those of real frames and real masks
    c0.composite_yuyv_into(rings[0]["host"], yuyv=np.empty((B, H, W, 2), np.uint8))
    for name, st in [("pre", 0), ("cnn", 1), ("decision", 2), ("post", 3), ("all", 4)]:
        stages[name + "_ms_per_frame"] = c0.time_stage(st, B, 5) / B
    peaks = load_peaks()
    peak = float(peaks.get("hbm_gbs", 6650.0))
    oh, ow = c0.out_hwc[0], c0.out_hwc[1]
    yuyv_native = bool(c0.yuyv_native)
    bg_per_frame = bool(wl.get("animated")) or args.camera_blur
    bytes_launch = post_bytes(W, H, ow, oh, B, yuyv_native, bg_per_frame, bg_cache=yuyv_native and not args.camera_blur)
    t_post = c0.time_stage(3, B, 10) * 1e-3                    # seconds per launch (B frames), CUDA events on the context's stream
    achieved = bytes_launch / t_post / 1e9
    traffic = None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "post_traffic.json")))
        traffic = tr.get(key, {}).get(f"{B}:{kind}")
    except Exception:
        pass
    if args.bgblur:
        traffic = None                                          # captured for the un-blurred configurations only
    roi = c0.roidim
    # whole-pipeline algorithmic HBM bytes per frame: camera frame read by the pre-processing stage (ROI, in its wire format)
    # + the post stage; a BGR materialisation (2WH in + 3WH out) is added when the frames cannot stay in YUYV
    pipeline_bytes = (2 if yuyv_native else 3) * roi[2] * roi[3] + bytes_launch / B + (0 if yuyv_native else 5 * npx)
    flops = c0.flops
    t_cnn = stages["cnn_ms_per_frame"] * 1e-3
    roofline = {"bound": "hbm", "kernel": "k_post_tma" if yuyv_native else "k_post_fast",
                "what": "mask upsample + 5x5 blur + alpha blend + RGB->YUYV + mask (one launch = %d frames)" % B,
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": "profiles/post_traffic.json (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch)" if traffic else None,
                "traffic_frac_of_peak": (traffic / t_post / 1e9 / peak) if traffic else None,
                "bytes_per_launch": bytes_launch, "ms_per_launch": t_post * 1e3,
                "bytes_formula": "B*(%s frame + 3WH out + 2WH yuyv + WH mask + ow*oh) + background %s" %
                                 ("2WH" if yuyv_native else "3WH", "per frame" if bg_per_frame else "ONCE per launch (still image)"),
                "frames": kind,
                "pipeline_bytes_per_frame": pipeline_bytes, "pipeline_hbm_frac": value * pipeline_bytes / 1e9 / (peak * world),
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s",
                # the CNN is not HBM-bound: report it against the FFMA pipe (148 SMs x 128 lanes x 2 x SM clock)
                "cnn": {"mflop_per_frame": flops / 1e6, "us_per_frame_one_stream": t_cnn * 1e6,
                        "achieved_tflops_one_stream": flops / t_cnn / 1e12,
                        "achieved_tflops_pipeline": flops * value / world / 1e12,
                        "ffma_peak_tflops": 148 * 128 * 2 * float(peaks.get("sm_max_mhz", 1965.0)) * 1e6 / 1e12,
                        "launches_per_call": c0.launches_per_call}}

    roofline["cnn"]["pointwise_convs"] = "tcgen05 3xTF32 (decisions identical to the exact path on the committed fixtures)" if c0.uses_tensor_cores else "fp32 FFMA (bit-exact vs oracle)"
    roofline["cnn"]["tensor_dense_tf32_peak_tflops"] = 1100.0
    res = dict(value=value, ms=ms, e2e=e2e, clocks=clocks, stages=stages, roofline=roofline, S=S, B=B, lps=lps, tc=bool(c0.uses_tensor_cores),
               launches=c0.launches_per_call, bg_desc=bg_desc, flops=flops, yuyv_native=yuyv_native, steps=steps)
    for c in ctxs:
        bs.bs_maskgen_delete(c)
    del rings, ctxs
    torch.cuda.empty_cache()
    return res


def workload_config(wl, args, S, B, lps, world, extra=None):
    """config keys shared by both arms (the driver compares them)"""
    cfg = {"workload": wl["desc"], "frames": args.frames, "input": "camera YUYV frames", "outputs": "RGB composite + YUYV + mask",
           "background": "blurred camera frame" if args.camera_blur else ("animated (one decoded image per frame)" if wl.get("animated") else "still image"),
           "bgblur": args.bgblur or None}
    if extra:
        cfg.update(extra)
    return cfg


def gpu_for_local_rank(torch, local, world):
    """Which GPU a local rank drives.  The end-to-end path is bound by each socket's host-memory / PCIe root complex, so
    for world < #GPUs the ranks are spread round-robin over the sockets (GPU NUMA groups from NVML's CPU affinity:
    local ranks 0,1,2,3 -> GPUs 0,4,1,5 on a 2 x 4 box) instead of filling socket 0 first.  Every rank computes the same
    order; with all GPUs in use it is a permutation and changes nothing."""
    n = torch.cuda.device_count()
    order = list(range(n))
    try:
        import pynvml
        pynvml.nvmlInit()
        groups = {}
        for d in range(n):
            uuid = "GPU-" + str(torch.cuda.get_device_properties(d).uuid)
            try:
                h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(d)
            key = tuple(pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64))
            groups.setdefault(key, []).append(d)
        lists = [groups[k] for k in sorted(groups, key=lambda k: groups[k][0])]
        order = []
        i = 0
        while len(order) < n:
            for g in lists:
                if i < len(g):
                    order.append(g[i])
            i += 1
    except Exception:
        order = list(range(n))
    return order[local % n] if world <= n else local % n


def run_b200(args, wl):
    import torch

    import backscrub_b200 as bs

    rank, world, local = dist_env()
    dev = gpu_for_local_rank(torch, local, world) if world > 1 else 0
    if world > 1:
        import torch.distributed as dist
        # NCCL writes its version banner / debug lines to stdout while the communicator comes up; rank 0's stdout must
        # carry exactly one JSON line, so point fd 1 at stderr for the duration of the initialisation
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", dev))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    torch.cuda.set_device(dev)
    full_affinity = bind_near_gpu(torch, dev)
    bound_cpus = len(os.sched_getaffinity(0))
    if bs.device_count() <= 0:
        raise SystemExit("bench.py needs a CUDA device: backscrub_b200 has no CPU path")
    if args.camera_blur and not args.bgblur:
        raise SystemExit("--camera-blur needs --bgblur K")
    for t in args.tune:
        name, _, val = t.partition("=")
        bs.set_tuning(name, int(val))
    S, B = args.streams or wl.get("streams", 8), args.batch or wl.get("batch", 32)
    lps = max(1, args.launches_per_step)
    m = measure(args, wl, args.workload, dev, rank, world, S, B, args.steps, args.warmup, lps, not args.no_e2e, True, kind=args.frames,
                dump_dir=args.dump_outputs if rank == 0 else None)

    # ---- the other BASELINE configs, short runs on one GPU (N = 1 only): parsed.configs ----
    configs = None
    if rank == 0 and world == 1 and not args.no_configs and args.workload == "meet720" and not args.bgblur:
        configs = {}
        for key in ("mlkit480", "deeplab720", "bodypix4k"):
            w2 = WORKLOADS[key]
            S2, B2 = w2.get("streams", 8), w2.get("batch", 32)
            try:
                r = measure(args, w2, key, dev, 0, 1, S2, B2, max(2, args.steps // 5), 2, 1, not args.no_e2e, False)
                configs[key] = {"workload": w2["desc"], "value": r["value"], "unit": UNIT, "streams_per_gpu": S2, "batch": B2,
                                "ms_per_step": r["ms"] / r["steps"], "e2e": r["e2e"], "roofline": r["roofline"], "stages": r["stages"],
                                "gpu_launches_per_call": r["launches"]}
            except Exception as e:                   # a side config must never cost the headline line
                configs[key] = {"workload": w2["desc"], "error": str(e)[:200]}

    # ---- CPU baseline (rank 0, N = 1 only; bounded sample) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        os.sched_setaffinity(0, full_affinity)          # the CPU baseline may use every host core
        cores = host_cores()
        threads = max(1, min(cores, 64))
        kw = dict(bgblur=args.bgblur, camera_blur=args.camera_blur)
        fps1, _ = cpu_path_fps(wl, 1, 1, warm=1, **kw)
        fpt = max(1, int(min(8, 12.0 * fps1)))             # ~12 s of wall time
        v, dt = cpu_path_fps(wl, threads, fpt, warm=0, **kw)
        cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"{threads} threads x {fpt} frames of the same workload ({dt:.1f} s), oracle port (TFLite-reference kernels + OpenCV ops restated)",
               "single_thread_value": fps1, "calibration": cnn_calibration(wl), "tflite_probe": tflite_probe()}

    if rank == 0:
        fb, npx = wl["W"] * wl["H"] * 3, wl["W"] * wl["H"]
        line = {
            "metric": METRIC, "value": m["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": m["ms"] / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32+u8", "data": "synthetic",
            "config": workload_config(wl, args, S, B, lps, world, {
                "streams_per_gpu": S, "batch": B, "graph_launches_per_stream_per_step": lps, "frames_per_step": world * S * B * lps,
                "pointwise_convs": "tcgen05 3xTF32" if m["tc"] else "fp32 FFMA (bit-exact vs oracle)",
                "parallelism": f"streams sharded over {world} GPU(s), no data-path collective",
                "gpu_of_rank0": dev,
                "background_detail": m["bg_desc"], "host_affinity_cpus": bound_cpus,
                "camera_frames": "read in place as YUYV by the GPU kernels" if m["yuyv_native"] else "YUYV -> BGR on the GPU, then BGR pipeline",
                "tuning": args.tune or None,
                "l2_policy": f"inputs+outputs of one launch round ({S * 2 * B} frames ring, {S * B * (fb + 5 * npx) / 1e6:.0f} MB per round) exceed the 126 MB L2"}),
            "gpu_launches": args.steps * lps * S * m["launches"],
            "e2e": m["e2e"], "roofline": m["roofline"], "cpu_baseline": cpu, "clocks": m["clocks"], "stages": m["stages"],
            "cnn_mflop_per_frame": m["flops"] / 1e6, "configs": configs,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


def main():
    args = parse()
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_b200(args, wl)


if __name__ == "__main__":
    main()
