#!/usr/bin/env python3
"""Decode rate of single huge frames: 1 x 1 GiB, 4 x 512 MiB and 1 x (2^31 - 1) B of synthetic text (libzstd level 1,
windowLog 27 with long-distance matching), each shape one batch through device pointers.  Every frame is verified by its
XXH64 (device hash against the trailer).  Prints one JSON line per shape: device-timed GB/s of decoded output (CUDA events
around the decode call, the second of two runs), per-kernel-class ms of that run, and the GPU it ran on.
usage: python scripts/large_frames.py [--out FILE]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import numpy as np
import torch

import largeframes as LF
import cairo_zstd_b200 as czb
from cairo_zstd_b200 import api

SHAPES = [("1x1GiB", 1, 1 << 30), ("4x512MiB", 4, 512 << 20), ("1x(2^31-1)B", 1, LF.MAX_OUT)]


def run(ctx, frames, size):
    dev = torch.device("cuda", 0)
    n = len(frames)
    flens = np.array([len(f) for f in frames], dtype=np.int64)
    soff = np.concatenate([[0], np.cumsum((flens + 15) & ~15)])
    src_h = np.zeros(int(soff[-1]), dtype=np.uint8)
    for i, f in enumerate(frames):
        src_h[soff[i]:soff[i] + len(f)] = np.frombuffer(f, dtype=np.uint8)
    src = torch.from_numpy(src_h).to(dev)
    dst = torch.empty(n * ((size + 15) & ~15), dtype=torch.uint8, device=dev)
    d = np.zeros((n, 4), dtype=np.uint64)
    d[:, 0] = src.data_ptr() + soff[:-1]
    d[:, 1] = flens
    d[:, 2] = dst.data_ptr() + np.arange(n, dtype=np.uint64) * ((size + 15) & ~15)
    d[:, 3] = size
    descs = torch.from_numpy(d.view(np.uint8).reshape(-1)).to(dev)
    results = torch.zeros(n * C.sizeof(api.FrameResult), dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream()
    out = None
    for rep in range(2):  # the first run loads modules and sizes the context's scratch
        ctx.profile_collect()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        ctx.decode_batch_device(descs.data_ptr(), results.data_ptr(), n, api.FLAG_VERIFY_CHECKSUM, stream.cuda_stream)
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        res = (api.FrameResult * n).from_buffer_copy(results.cpu().numpy().tobytes())
        for r in res:
            assert r.status == 0 and r.bytes_written == size, czb.status_name(r.status)
            assert r.checksum_calculated == r.checksum_from_data, "XXH64 mismatch"
        out = dict(ms=round(ms, 2), gb_per_s=round(n * size / ms / 1e6, 3),
                   kernel_ms={k: round(v[0], 2) for k, v in ctx.profile_collect().items()})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    ctx = czb.Context(0)
    ctx.profile_enable(True)
    lines = []
    for name, count, size in SHAPES:
        frames = []
        for k in range(count):
            data = LF.text(size, seed=100 + k)
            frames.append(LF.compress(data, 27, ldm=True))
            del data
        rec = dict(shape=name, frames=count, frame_bytes=size, compressed_bytes=sum(len(f) for f in frames), gpu=gpu)
        rec.update(run(ctx, frames, size))
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    ctx.close()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(lines, f, indent=1)


if __name__ == "__main__":
    main()
