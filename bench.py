#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's configs.

metric   Mpixels/s (INPUT pixels) through the per-frame hot path
           scale -> compose -> median-cut -> FS dither -> sixel emit          (-p sixel: C2, C4, C5)
           scale -> compose -> half/quarter-block pick -> ANSI emit           (-p half / -p quarter: C1, C3)
workload --config C2 (default, the configuration the metric is quoted on): 3840x2160 RGBA frames -> "-p sixel"
         on a 300x100-cell terminal (cell 9x18 px, src/timg.cc:760-761) -> CalcScaleToFitDisplay -> 2700x1519
         -> padded to 1524 rows (round_to_sixel, src/sixel-canvas.cc:91-94).  A "step" is one pass of the hot
         path over one batch of --frames distinct synthetic frames; the batch is far larger than L2, so nothing
         is cache-resident between steps.  C1/C3/C4/C5 are the other BASELINE.json configs (SURVEY.md 8d).

  python bench.py [--config C1..C5] [--gpus N] [--steps K] [--warmup W] [--frames F] [--impl b200|reference]
                  [--dump-outputs DIR]

Launched under torchrun for N>1 (one rank per GPU): frames are independent units, each rank runs the same
per-GPU batch (weak scaling) and the encoded byte buffers are gathered to rank 0 over NCCL inside the timed
region.  Prints ONE JSON line on rank 0.

--impl reference times the reference's own CPU path for the same config on this box's host cores with native
threads (oracle/cpu_pipeline.c; oracle/_ref = the reference's unmodified translation units).  That arm imports
neither torch nor timg_b200 and touches no GPU.
"""
import argparse
import ctypes as C
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BG = (0, 0, 0)
SEED = 1234
METRIC = "Mpixels/s scale+dither+sixel-encode @4K→cell"     # BASELINE.json "metric", first clause
QUARTER, FAST_SCALE = 1, 8

# name: source size, CalcScaleToFitDisplay arguments (width px, height px, cell_x, cell_y, width_stretch), canvas
CONFIGS = {
    "C1": dict(iw=640, ih=480, fit=(80, 50, 1, 2, 1.0), canvas="half", flags=0, animation=0, kind="alpha", frames=4096,
               text="C1: 640x480 RGBA -> -p half, 80x25 cells -> 67x50 -> half-block pick + ANSI emit"),
    "C2": dict(iw=3840, ih=2160, fit=(2700, 1800, 9, 18, 1.0), canvas="sixel", flags=0, animation=0, kind="photo", frames=148,
               text="C2: 3840x2160 RGBA -> -p sixel, 300x100 cells of 9x18px -> 2700x1519 (+pad 1524) Mitchell scale + compose + "
                    "256-colour median cut + FS dither + sixel"),
    "C3": dict(iw=1920, ih=1080, fit=(320, 100, 2, 2, 2.0), canvas="quarter", flags=QUARTER, animation=1, kind="video", frames=300,
               text="C3: 1920x1080 video frames (photo base + moving 64x64 noise sprite) -> -p quarter, 160x50 cells -> 320x90, "
                    "first frame full, the rest delta-encoded against the previous frame"),
    "C4": dict(iw=3840, ih=2160, fit=(337, 225, 9, 18, 1.0), canvas="sixel", flags=0, animation=0, kind="photo", frames=128,
               text="C4: --grid=8x8 pages of 4K RGBA frames -> -p sixel, 337x225 px per image -> 337x190 (+pad 192)"),
    "C5": dict(iw=1280, ih=720, fit=(2700, 1800, 9, 18, 1.0), canvas="sixel", flags=0, animation=0, kind="photo", frames=1250,
               text="C5: 1280x720 animation frames shown unscaled -> -p sixel (1280x720, already a multiple of 6 rows)"),
}
CPU_JOBS_PER_THREAD = {"C1": 400, "C2": 2, "C3": 60, "C4": 2, "C5": 8}     # bounded CPU samples (tens of seconds)


def load_synth():
    """timg_b200/synth.py by path: the frame generator is plain numpy and is shared by both arms without
    importing the timg_b200 package (the reference arm must not load the product)."""
    spec = importlib.util.spec_from_file_location("b200_synth", os.path.join(ROOT, "timg_b200", "synth.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def config_dict(name, cfg, ow, oh, frames):
    hp = (oh + 5) // 6 * 6 if cfg["canvas"] == "sixel" else oh
    return {"workload": cfg["text"], "config": name, "frames_per_gpu_per_step": frames, "scaled": [ow, oh, hp],
            "synthetic": cfg["kind"], "l2": "inputs larger than L2 (batch of distinct frames)"}


def frames_numpy(synth, cfg, n, seed0=SEED):
    """n distinct frames of the config as numpy (CPU arm).  C3: one photo base, a noise sprite moving 8 px/frame."""
    iw, ih = cfg["iw"], cfg["ih"]
    if cfg["kind"] != "video":
        return np.stack([synth.frame_np(seed0 + i, iw, ih, cfg["kind"]) for i in range(n)])
    base = synth.frame_np(seed0, iw, ih, "photo")
    out = np.repeat(base[None], n, 0)
    for k in range(n):
        x, y = (37 + 8 * k) % (iw - 64), (91 + 5 * k) % (ih - 64)
        out[k, y:y + 64, x:x + 64] = synth.frame_np(seed0 + 1000 + k, 64, 64, "noise")
    return out


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (profiling recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# --------------------------------------------------------------------------- CPU reference arm
def run_cpu(name, cfg, threads, jobs_per_thread, synth):
    """The reference's CPU path for `cfg` on `threads` native threads over threads*jobs_per_thread frames.
    Returns (Mpx/s, seconds, mean encoded bytes or None, kind, description)."""
    import oracle
    iw, ih = cfg["iw"], cfg["ih"]
    w, h, cx, cy, st = cfg["fit"]
    _, ow, oh = oracle.calc_fit(iw, ih, w, h, cx, cy, st)
    bg = oracle.rgba_u32(*BG)
    n_jobs = max(1, threads * jobs_per_thread)
    pool = frames_numpy(synth, cfg, min(n_jobs, 8 if cfg["canvas"] == "sixel" else 64))
    if cfg["canvas"] == "sixel":
        dt, sizes, what = oracle.cpu_sixel_jobs(pool, n_jobs, ow, oh, bg, threads, mode=0)
        enc, kind = int(sizes.mean()), "port"           # scaler + compose are the reference's own code; libsixel is a restatement
    else:
        dt, what = oracle.cpu_blocks_jobs(pool, n_jobs, ow, oh, bg, threads, flags=cfg["flags"], animation=bool(cfg["animation"]))
        enc, kind = None, "reference"
    return n_jobs * iw * ih / 1e6 / dt, dt, enc, kind, f"{n_jobs} frames on {threads} native threads ({dt:.1f} s); {what}"


def cpu_baseline(name, cfg, threads, synth):
    """All-cores line + 1-thread line (how UnicodeBlockCanvas actually runs), bounded to tens of seconds."""
    per = CPU_JOBS_PER_THREAD[name]
    v, dt, enc, kind, what = run_cpu(name, cfg, threads, per, synth)
    v1, dt1, _, _, _ = run_cpu(name, cfg, 1, per, synth)
    return {"value": v, "unit": "Mpx/s", "cores": threads, "kind": kind, "sample": what,
            "one_thread": {"value": v1, "unit": "Mpx/s", "seconds": dt1}, "encoded_bytes_per_frame": enc}


def reference_arm(args, name, cfg):
    import oracle
    threads = args.cpu_threads or (os.cpu_count() or 1)
    iw, ih = cfg["iw"], cfg["ih"]
    w, h, cx, cy, st = cfg["fit"]
    _, ow, oh = oracle.calc_fit(iw, ih, w, h, cx, cy, st)
    frames = args.frames or cfg["frames"]
    synth = load_synth()
    per = CPU_JOBS_PER_THREAD[name]
    vals, secs, enc, kind, what = [], 0.0, None, "port", ""
    for _ in range(max(0, min(args.warmup, 1))):
        run_cpu(name, cfg, threads, 1, synth)
    for _ in range(max(1, args.steps)):
        v, dt, enc, kind, what = run_cpu(name, cfg, threads, per, synth)
        vals.append(v)
        secs += dt
    value = float(np.mean(vals))
    v1, dt1, _, _, _ = run_cpu(name, cfg, 1, per, synth)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "Mpx/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": secs / max(1, args.steps) * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8/f32", "data": "synthetic", "config": config_dict(name, cfg, ow, oh, frames),
            "cpu_baseline": {"value": value, "unit": "Mpx/s", "cores": threads, "kind": kind, "sample": what,
                             "one_thread": {"value": v1, "unit": "Mpx/s", "seconds": dt1}},
            "e2e": {"value": value, "unit": "Mpx/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "encoded_bytes_per_frame": enc}
    print(json.dumps(line))


# --------------------------------------------------------------------------- helpers of the GPU arm
def pin_to_gpu_numa(local_rank):
    """Bind this process to the CPUs next to its GPU before any pinned allocation (2 NUMA domains per box)."""
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(local_rank)],
                           capture_output=True, text=True, timeout=20).stdout.strip().lower()
        bus = q[4:] if len(q) > 12 else q                     # nvidia-smi prints an 8-digit PCI domain, sysfs uses 4
        cpus = set()
        for part in open(f"/sys/bus/pci/devices/{bus}/local_cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"cpus": len(cpus), "node": open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip()}
    except Exception as ex:
        return {"error": str(ex)[:80]}
    return None


def frames_torch(synth, cfg, n, seed0, dev):
    import torch
    iw, ih = cfg["iw"], cfg["ih"]
    frames = torch.empty((n, ih, iw, 4), dtype=torch.uint8, device=dev)
    if cfg["kind"] != "video":
        for i in range(n):
            frames[i] = synth.frame_torch(seed0 + i, iw, ih, cfg["kind"], dev)
        return frames
    frames[:] = synth.frame_torch(seed0, iw, ih, "photo", dev)
    for k in range(n):
        x, y = (37 + 8 * k) % (iw - 64), (91 + 5 * k) % (ih - 64)
        frames[k, y:y + 64, x:x + 64] = synth.frame_torch(seed0 + 1000 + k, 64, 64, "noise", dev)
    return frames


DUMP_MAX_BYTES = 15 << 20        # encoded bytes dumped at most: 60 MiB as float32


def dump_outputs(out_dir, out, offs):
    """What a caller of the batch call receives: the per-frame byte offsets into the output buffer
    (offsets.npy, float64, all frames) and the encoded bytes (encoded.npy, float32, one value per byte).
    When all frames' bytes exceed DUMP_MAX_BYTES, encoded.npy holds whole frames taken in a fixed seeded
    order until the next would not fit (the first frame is cut at the limit if it alone exceeds it), and
    encoded_frames.npy lists those frames in the order their bytes appear."""
    os.makedirs(out_dir, exist_ok=True)
    offs = offs.cpu().numpy().astype(np.int64)
    np.save(os.path.join(out_dir, "offsets.npy"), offs.astype(np.float64))
    if offs[-1] <= DUMP_MAX_BYTES:
        np.save(os.path.join(out_dir, "encoded.npy"), out[:offs[-1]].cpu().numpy().astype(np.float32))
        return
    picked, parts, size = [], [], 0
    for f in np.random.default_rng(SEED).permutation(len(offs) - 1):
        n = min(int(offs[f + 1] - offs[f]), DUMP_MAX_BYTES - size)
        if n < offs[f + 1] - offs[f] and picked:
            break
        picked.append(int(f))
        parts.append(out[offs[f]:offs[f] + n].cpu().numpy())
        size += n
        if size == DUMP_MAX_BYTES:
            break
    np.save(os.path.join(out_dir, "encoded.npy"), np.concatenate(parts).astype(np.float32))
    np.save(os.path.join(out_dir, "encoded_frames.npy"), np.array(picked, np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="C2", choices=sorted(CONFIGS))
    ap.add_argument("--frames", type=int, default=0, help="frames per GPU per step (one batch); 0 = the config's default")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-threads", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--kernels-only", action="store_true", help="print just the per-kernel table (tuning runs)")
    ap.add_argument("--yuv", action="store_true",
                    help="feed decoder-style I420 frames (1.5 B/px) through the fused colour-conversion + bilinear scaler "
                         "(the video source's sws_scale, src/video-source.cc:352-354) instead of RGBA through ImageScaler")
    ap.add_argument("--py-gather", action="store_true",
                    help="N>1: gather through torch.distributed point-to-point (round 1) instead of the C-ABI b200timg_gather")
    ap.add_argument("--exact-scale", action="store_true",
                    help="bit-exact scaler arithmetic on the sixel path instead of the <= 1 LSB fused-multiply-add mode")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (rank 0's encoded bytes and frame offsets) as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the GPU path's outputs (--impl b200)")
    name, cfg = args.config, CONFIGS[args.config]
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if rank == 0:                      # the reference's own CPU implementation of the path; rank 0 only
            reference_arm(args, name, cfg)
        return

    numa = pin_to_gpu_numa(local_rank)
    # (NCCL's defaults are left alone: routing the point-to-point gather through the copy engines with
    # NCCL_P2P_USE_CUDA_MEMCPY=1 measured 18.1 ms per step on 2 GPUs against 14.25 ms with NCCL's own NVLink kernels, run r2n3)
    import torch
    import torch.distributed as dist
    import timg_b200
    from timg_b200 import shard, synth

    iw, ih, F = cfg["iw"], cfg["ih"], args.frames or cfg["frames"]
    fw, fh, cx, cy, st = cfg["fit"]
    _, ow, oh = timg_b200.calc_fit(iw, ih, fw, fh, cx, cy, st)
    sixel = cfg["canvas"] == "sixel"
    hp = (oh + 5) // 6 * 6 if sixel else oh
    config = config_dict(name, cfg, ow, oh, F)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    stream = torch.cuda.Stream(dev)            # a real (non-default) stream shared by torch and the library,
    torch.cuda.set_stream(stream)              # so torch's CUDA events time the library's launches
    ctx = timg_b200.Context(local_rank, stream.cuda_stream)
    assert stream.cuda_stream != 0
    L = timg_b200.lib()
    frames = frames_torch(synth, cfg, F, SEED + rank * F, dev)
    src_fmt, frame_bytes = 0, iw * ih * 4
    if args.yuv:                                   # BT.601 limited-range I420 of the same frames (2x2 box chroma)
        def to_i420(fr):
            c = fr[..., :3].to(torch.float32)
            r, g, bl = c[..., 0], c[..., 1], c[..., 2]
            y = 16 + 0.256788 * r + 0.504129 * g + 0.097906 * bl
            u = 128 - 0.148223 * r - 0.290993 * g + 0.439216 * bl
            v = 128 + 0.439216 * r - 0.367788 * g - 0.071427 * bl
            box = lambda p: p.reshape(ih // 2, 2, iw // 2, 2).mean((1, 3))
            q = lambda p: p.round().clamp(0, 255).to(torch.uint8).reshape(-1)
            return torch.cat([q(y), q(box(u)), q(box(v))])
        yuv = torch.empty((F, iw * ih * 3 // 2), dtype=torch.uint8, device=dev)
        for i in range(F):
            yuv[i] = to_i420(frames[i])
        frames, src_fmt, frame_bytes = yuv, timg_b200.FMT_I420, iw * ih * 3 // 2
        config["source"] = "I420 (BT.601 limited range), colour conversion fused into the bilinear scaler"
    torch.cuda.synchronize(dev)
    # the sixel path's scaler runs in the <= 1 LSB mode unless --exact-scale; block modes are always bit-exact
    flags = cfg["flags"] | (FAST_SCALE if sixel and not args.exact_scale else 0)
    b = timg_b200.Batch(n_frames=F, src_w=iw, src_h=ih, src_fmt=src_fmt, out_w=ow, out_h=oh, has_bg=1,
                        bg=timg_b200.rgba_u32(*BG), pattern=0, pattern_w=0, pattern_h=0, flags=flags, x_indent_cells=0,
                        animation=cfg["animation"])
    dev_call = L.b200timg_sixel_batch_dev if sixel else L.b200timg_blocks_batch_dev
    host_call = L.b200timg_sixel_batch if sixel else L.b200timg_blocks_batch
    cap = F * max(1 << 16, 2 * ow * hp) if sixel else int(L.b200timg_blocks_bound(ow, oh)) * F + 64
    # two output buffers: with N > 1 the gather of batch k (NCCL, its own stream) runs while batch k+1 is
    # being encoded into the other buffer -- the way a stream of pages / video windows would be served
    nbuf = 2 if world > 1 else 1
    outs = [torch.empty(cap, dtype=torch.uint8, device=dev) for _ in range(nbuf)]
    offss = [torch.zeros(F + 1, dtype=torch.int64, device=dev) for _ in range(nbuf)]
    pending = [None] * nbuf
    step_no = [0]

    def drain():
        for i in range(nbuf):
            if pending[i] is not None:
                pending[i].wait()
                pending[i] = None

    def step(gather=True):
        i = step_no[0] % nbuf
        step_no[0] += 1
        if pending[i] is not None:              # that buffer's previous batch must have left
            pending[i].wait()
            pending[i] = None
        rc = dev_call(ctx.h, C.byref(b), frames.data_ptr(), outs[i].data_ptr(), cap, offss[i].data_ptr())
        if rc != 0:
            raise RuntimeError(L.b200timg_last_error(ctx.h).decode())
        if world > 1 and gather:
            pending[i] = abi_gather.start(outs[i], offss[i]) if abi_gather else shard.gather_encoded_async(outs[i], offss[i], dst=0)

    # first call sizes the output; grow the buffers if the guess was too small (nothing is written past cap)
    abi_gather = None
    step(gather=False)
    torch.cuda.synchronize(dev)
    total = int(offss[0][-1].item())
    slot = 0
    if world > 1:          # one slot size for all ranks: the largest batch + 2 %
        tmax = torch.tensor([total], dtype=torch.int64, device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        slot = (int(tmax.item()) * 102 // 100 + 4095) // 4096 * 4096
    if total > cap or slot > cap:
        cap = max(int(total * 1.05), slot)
        outs = [torch.empty(cap, dtype=torch.uint8, device=dev) for _ in range(nbuf)]
    if world > 1 and not args.py_gather:
        abi_gather = shard.AbiGather(ctx, F, slot, root=0, buffers=nbuf)
    for _ in range(args.warmup):
        step()
    drain()
    torch.cuda.synchronize(dev)
    launches0 = ctx.launches
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()              # after the sampler start-up, so no rank times another rank's sleep
    torch.cuda.synchronize(dev)
    e0.record(stream)
    for _ in range(args.steps):
        step()
    drain()                                    # every batch has arrived on rank 0 inside the timed region
    e1.record(stream)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    ms_total = e0.elapsed_time(e1)
    launches = ctx.launches - launches0
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    total_bytes = int(offss[0][-1].item())
    if rank == 0 and args.dump_outputs:        # before the passes below overwrite the output buffers
        last = (step_no[0] - 1) % nbuf
        dump_outputs(args.dump_outputs, outs[last], offss[last])
    value = world * F * args.steps * iw * ih / 1e6 / (ms_total / 1e3)

    # ---- per-kernel timing (separate pass, profiling on) -> roofline of the dominant kernel
    roofline, kernels = None, None
    if rank == 0:
        ctx.profile(True)
        for _ in range(2):
            step(gather=False)
        rep = ctx.profile_report()
        ctx.profile(False)
        kernels = {k: {"launches": n, "ms_per_launch": ms / n} for k, (n, ms) in rep.items()}
        chain_ms = sum(ms for _, ms in rep.values()) / 2
        dom = max(rep, key=lambda k: rep[k][1])
        n, ms = rep[dom]
        # SURVEY 8(d): read every source pixel once + write every encoded byte once (+ previous scaled frame for deltas)
        alg_bytes = F * frame_bytes + total_bytes + (4 * ow * oh * (F - 1) if cfg["animation"] else 0)
        peak, how = peak_hbm()
        achieved = alg_bytes / (ms / n / 1e3) / 1e9
        traffic = None       # dram__bytes_read+write of that kernel per launch, from the committed ncu capture
        tp = os.path.join(ROOT, "profiles", "r2_traffic.json")
        if os.path.exists(tp):
            k = json.load(open(tp)).get(name, {}).get(dom)
            if k:
                traffic = k["dram_bytes_per_frame"] * F
        roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": traffic, "peak_source": how,
                    "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms_per_launch": ms / n,
                    "kernel_share_of_chain": (ms / 2) / chain_ms,
                    "chain": {"ms_per_step": chain_ms, "achieved": alg_bytes / (chain_ms / 1e3) / 1e9,
                              "frac": alg_bytes / (chain_ms / 1e3) / 1e9 / peak}}

    # ---- single-frame latency (BASELINE configs[1] is literally one frame): device-resident, batch of 1
    latency = None
    if rank == 0 and not cfg["animation"]:
        b1 = timg_b200.Batch.from_buffer_copy(b)
        b1.n_frames = 1
        for _ in range(3):
            dev_call(ctx.h, C.byref(b1), frames.data_ptr(), outs[0].data_ptr(), cap, offss[0].data_ptr())
        torch.cuda.synchronize(dev)
        l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0.record(stream)
        for _ in range(5):
            dev_call(ctx.h, C.byref(b1), frames.data_ptr(), outs[0].data_ptr(), cap, offss[0].data_ptr())
        l1.record(stream)
        torch.cuda.synchronize(dev)
        latency = {"ms": l0.elapsed_time(l1) / 5, "mpx_s": iw * ih / 1e6 / (l0.elapsed_time(l1) / 5 / 1e3),
                   "note": "one frame through the whole chain (FS wavefront split over several CTAs for small batches)"}

    # ---- end to end through the host-buffer ABI call: pinned host frames in, host bytes out
    e2e = None
    if not args.no_e2e:
        Fe = F
        try:
            h_in = torch.empty((Fe,) + tuple(frames.shape[1:]), dtype=torch.uint8, pin_memory=True)
        except RuntimeError:
            Fe = max(1, F // 8)
            h_in = torch.empty((Fe,) + tuple(frames.shape[1:]), dtype=torch.uint8, pin_memory=True)
        h_in.copy_(frames[:Fe])
        h_out = torch.empty(int(total_bytes * Fe / F * 1.1) + 4096, dtype=torch.uint8, pin_memory=True)
        h_offs = np.zeros(Fe + 1, np.uint64)
        be = timg_b200.Batch.from_buffer_copy(b)
        be.n_frames = Fe

        def e2e_step():
            rc = host_call(ctx.h, C.byref(be), h_in.data_ptr(), h_out.data_ptr(), h_out.numel(), h_offs.ctypes.data)
            if rc != 0:
                raise RuntimeError(L.b200timg_last_error(ctx.h).decode())

        e2e_step()
        # raw pinned H2D rate of this box, for context: the e2e number cannot exceed it
        torch.cuda.synchronize(dev)
        nprobe = max(1, min(Fe, (1 << 30) // frame_bytes))
        t0 = time.perf_counter()
        frames[:nprobe].copy_(h_in[:nprobe], non_blocking=True)
        torch.cuda.synchronize(dev)
        h2d_gbs = nprobe * frame_bytes / (time.perf_counter() - t0) / 1e9
        if world > 1:
            dist.barrier()
        ke = max(1, min(args.steps, 5))
        t0 = time.perf_counter()
        for _ in range(ke):
            e2e_step()
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        e2e = {"value": world * Fe * ke * iw * ih / 1e6 / dt, "unit": "Mpx/s",
               "h2d_bytes_per_step": int(Fe * frame_bytes), "d2h_bytes_per_step": int(h_offs[Fe]) + 8 * (Fe + 1),
               "frames_per_step": Fe, "steps": ke,
               "api": ("b200timg_sixel_batch" if sixel else "b200timg_blocks_batch") + " (host buffers, pinned)",
               "pcie_h2d_gbs_measured": h2d_gbs, "pcie_bound_mpx_s": h2d_gbs * 1e9 / (frame_bytes / (iw * ih)) / 1e6, "numa": numa}
        del h_in, h_out

    # ---- the reference's CPU path beside it (rank 0, N=1 only): a bounded sample on native threads
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = args.cpu_threads or (os.cpu_count() or 1)
        try:
            cpu = cpu_baseline(name, cfg, threads, synth)
        except Exception as ex:            # the baseline is reported, never required for the GPU number
            cpu = {"value": None, "unit": "Mpx/s", "cores": threads, "kind": "port", "sample": f"failed: {ex}"}

    if rank == 0 and args.kernels_only:
        print(f"{name} value {value:.0f} Mpx/s  ms/step {ms_total / args.steps:.3f}  " +
              "  ".join(f"{k.replace('sixel_', '').replace('_kernel', '')}={v['ms_per_launch']:.3f}" for k, v in kernels.items()))
    elif rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "Mpx/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/f32", "data": "synthetic",
                "config": dict(config, parallelism=f"frames sharded x{world}, NCCL gather of encoded bytes to rank 0 "
                               f"({'torch.distributed p2p' if args.py_gather else 'b200timg_gather, fixed slots, no host sync'}); "
                               "double-buffered output: the gather of batch k overlaps the kernels of batch k+1"
                               if world > 1 else "1 GPU",
                               scaler="exact" if (args.exact_scale or not sixel) else "fast (<= 1 LSB, B200TIMG_FAST_SCALE)"),
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
                "cpu_baseline": cpu, "kernels": kernels, "encoded_bytes_per_frame": total_bytes // F,
                "single_frame_latency": latency}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
