"""Throughput and size of the kitty / iTerm2 PNG encode at timg's --compress levels 0 and 1, with host zlib -1 as the
yardstick (libdeflate, which the reference links, is not available to run; zlib is the stand-in and is labelled so).

    python tools/png_bench.py [--frames 64] [--repeats 5] [--out FILE]

One JSON line per (geometry, content, level, rgb24):
  batch_ms           device-resident batch of --frames frames (b200timg_png_batch_level_dev), host clock around
                     --repeats warmed runs ending in a device synchronise; the batch input is larger than L2
  gbps_filtered_in   filtered scanline bytes of the batch / batch time;  mpx_s: pixels / batch time
  single_frame_ms    one frame through b200timg_png_encode_level from host buffers (H2D and D2H included)
  ratio              PNG bytes / filtered bytes;  vs_zlib1: our PNG / len(zlib.compress(filtered, 1))
  zlib1_1thread_ms   zlib -1 of one frame on one thread (timg compresses each frame on one pool thread)
  zlib1_allcores_gbps  zlib -1 over a thread per core (zlib releases the GIL)
plus the GPU name and power limit read in the same run, and one line with the per-kernel split (profile_report).
"""
import argparse
import json
import os
import subprocess
import sys
import time
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import timg_b200  # noqa: E402
from timg_b200 import synth  # noqa: E402


def flat_graphic(w, h, seed):
    """Palette blocks with dark one-pixel 'text' lines (UI screenshots, diagrams)."""
    rng = np.random.default_rng(seed)
    pal = rng.integers(0, 256, (12, 4), dtype=np.uint8)
    pal[:, 3] = 255
    bw, bh = 90, 60
    idx = rng.integers(0, len(pal), ((h + bh - 1) // bh, (w + bw - 1) // bw))
    fb = pal[np.repeat(np.repeat(idx, bh, 0), bw, 1)[:h, :w]].copy()
    for y in range(8, h, 17):
        x0 = int(rng.integers(0, max(1, w // 2)))
        fb[y, x0:x0 + int(rng.integers(20, max(21, w // 3))), :3] = 20
    return fb


def filtered(fb, rgb24):
    px = fb[..., :3] if rgb24 else fb
    h, w, bpp = px.shape
    d = px.astype(np.int16)
    d[:, 1:] -= px[:, :-1]
    return np.concatenate([np.ones((h, 1), np.uint8), (d & 255).astype(np.uint8).reshape(h, w * bpp)], axis=1).tobytes()


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (r.stdout.strip().splitlines() or ["?, ?"])[0].split(", ")
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("png_bench: no CUDA device (this benchmark only measures on the GPU)")
    name, power = gpu_info()
    L = timg_b200.lib()
    ctx = timg_b200.Context(0)
    cores = os.cpu_count() or 1
    lines = []

    def emit(d):
        s = json.dumps(d)
        print(s, flush=True)
        lines.append(s)

    for (w, h) in ((2700, 1519), (1920, 1080)):
        for content in ("photo", "flat"):
            distinct = [synth.frame_np(100 + k, w, h, "photo") if content == "photo" else flat_graphic(w, h, 100 + k)
                        for k in range(4)]
            frames = np.stack([distinct[k % 4] for k in range(a.frames)])
            d_frames = torch.from_numpy(frames).cuda()
            for rgb24 in (False, True):
                filt = [filtered(fb, rgb24) for fb in distinct]
                raw = len(filt[0])
                t0 = time.perf_counter()
                z1 = zlib.compress(filt[0], 1)
                z1_ms = (time.perf_counter() - t0) * 1e3
                jobs = [filt[k % 4] for k in range(2 * cores)]
                with ThreadPoolExecutor(cores) as ex:
                    t0 = time.perf_counter()
                    list(ex.map(lambda b: zlib.compress(b, 1), jobs))
                    z_all = time.perf_counter() - t0
                for level in (0, 1):
                    bound = L.b200timg_png_bound(w, h, int(rgb24), level)
                    nb = L.b200timg_base64_size(bound)
                    d_png = torch.empty(a.frames * bound, dtype=torch.uint8, device="cuda")
                    d_b64 = torch.empty(a.frames * nb, dtype=torch.uint8, device="cuda")
                    d_off = torch.zeros(a.frames + 1, dtype=torch.int64, device="cuda")
                    d_boff = torch.zeros(a.frames + 1, dtype=torch.int64, device="cuda")

                    def run():
                        rc = L.b200timg_png_batch_level_dev(ctx.h, d_frames.data_ptr(), w, h, a.frames, int(rgb24), level,
                                                            d_png.data_ptr(), d_png.numel(), d_off.data_ptr(),
                                                            d_b64.data_ptr(), d_b64.numel(), d_boff.data_ptr())
                        assert rc == timg_b200.OK, L.b200timg_last_error(ctx.h)
                    run()
                    run()
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()                                      # the library runs on its own stream:
                    for _ in range(a.repeats):                                    # host clock around a device-wide sync
                        run()
                    torch.cuda.synchronize()
                    batch_ms = (time.perf_counter() - t0) * 1e3 / a.repeats
                    off = d_off.cpu().numpy()
                    png0 = d_png[:int(off[1])].cpu().numpy().tobytes()
                    fb0 = np.ascontiguousarray(frames[0])
                    ctx.png_encode(fb0, rgb24, level=level)                       # warm the one-frame path
                    t0 = time.perf_counter()
                    for _ in range(a.repeats):
                        data, _ = ctx.png_encode(fb0, rgb24, level=level)
                    single_ms = (time.perf_counter() - t0) * 1e3 / a.repeats
                    assert data == png0
                    mean_png = float(off[-1]) / a.frames
                    emit(dict(geometry=f"{w}x{h}", content=content, level=level, rgb24=rgb24, frames=a.frames,
                              batch_ms=round(batch_ms, 3), gbps_filtered_in=round(raw * a.frames / batch_ms / 1e6, 2),
                              mpx_s=round(w * h * a.frames / batch_ms / 1e3, 1), single_frame_ms=round(single_ms, 3),
                              png_bytes_mean=round(mean_png), filtered_bytes=raw, ratio=round(mean_png / raw, 4),
                              vs_zlib1=round(len(data) / len(z1), 4), zlib1_ratio=round(len(z1) / raw, 4),
                              zlib1_1thread_ms=round(z1_ms, 2),
                              zlib1_allcores_gbps=round(raw * len(jobs) / z_all / 1e9, 3), host_cores=cores,
                              gpu=name, power_limit=power))
                    if (w, h, content, rgb24, level) == (2700, 1519, "photo", False, 1) or \
                            (w, h, content, rgb24, level) == (2700, 1519, "flat", False, 1):
                        ctx.profile(True)
                        run()
                        torch.cuda.synchronize()
                        rep = ctx.profile_report()
                        ctx.profile(False)
                        emit(dict(profile=f"{w}x{h} {content} level {level} batch of {a.frames}",
                                  kernels={k: dict(launches=v[0], ms=round(v[1], 3)) for k, v in rep.items()},
                                  gpu=name, power_limit=power))
                    del d_png, d_b64
            del d_frames
            torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write("\n".join(lines) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
