"""Device-timed rate of czb_verify_batch_device against czb_decode_batch_device + XXH64 (CZB_FLAG_VERIFY_CHECKSUM), in GB/s of
decoded output, on config 2 (64 KiB text frames) and config 5 (mixed 1 KiB..4 MiB frames); then one verify call over a batch
whose decoded total exceeds the card's memory (4 Mi x 64 KiB text frames, 256 GiB), checking that every frame verifies with
checksum_calculated == checksum_from_data.  Distinct frames are few and repeated by pointer, so the compressed input is small.

    python scripts/verify_rate.py --out profiles/verify_rate.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cairo_zstd_b200 as czb  # noqa: E402
from cairo_zstd_b200 import api  # noqa: E402
from cairo_zstd_b200 import workloads as W  # noqa: E402


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.returncode == 0 else None}


class Batch:
    """n frames cycling over the distinct `frames` (device copy of each distinct frame once)."""

    def __init__(self, frames, sizes, n):
        import torch
        dev = torch.device("cuda", 0)
        flens = np.array([len(f) for f in frames], dtype=np.int64)
        soff = np.concatenate([[0], np.cumsum((flens + 15) & ~15)])
        src_h = np.zeros(int(soff[-1]) + 16, dtype=np.uint8)
        for i, f in enumerate(frames):
            src_h[soff[i]:soff[i] + len(f)] = np.frombuffer(f, dtype=np.uint8)
        self.src = torch.from_numpy(src_h).to(dev)
        pick = np.arange(n) % len(frames)
        self.n, self.sizes = n, np.asarray(sizes, dtype=np.uint64)[pick]
        self.out_bytes = int(self.sizes.sum())
        self.d = np.zeros((n, 4), dtype=np.uint64)
        self.d[:, 0] = self.src.data_ptr() + soff[:-1][pick]
        self.d[:, 1] = flens[pick]
        self.results = torch.zeros((n * C.sizeof(api.FrameResult),), dtype=torch.uint8, device=dev)
        self.vdescs = torch.from_numpy(self.d.view(np.uint8).reshape(-1).copy()).to(dev)
        self.dst = self.ddescs = None

    def with_dst(self):
        import torch
        doff = np.concatenate([[0], np.cumsum((self.sizes + 15) & ~np.uint64(15))]).astype(np.uint64)
        self.dst = torch.empty((int(doff[-1]) + 16,), dtype=torch.uint8, device=self.src.device)
        d = self.d.copy()
        d[:, 2] = self.dst.data_ptr() + doff[:-1]
        d[:, 3] = self.sizes
        self.ddescs = torch.from_numpy(d.view(np.uint8).reshape(-1)).to(self.src.device)

    def fetch(self):
        return (api.FrameResult * self.n).from_buffer_copy(self.results.cpu().numpy().tobytes())


def timed(fn, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return ms


def check(res, n, want_checksum=True):
    bad = [i for i in range(n) if res[i].status != 0 or (want_checksum and (not res[i].has_checksum or
                                                                          res[i].checksum_calculated != res[i].checksum_from_data))]
    return len(bad), bad[:8]


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--config2-frames", type=int, default=262144)
    ap.add_argument("--config5-frames", type=int, default=4096)
    ap.add_argument("--huge-frames", type=int, default=4 << 20)
    a = ap.parse_args()
    ctx = czb.Context(0)
    stream = torch.cuda.current_stream().cuda_stream
    out = {"card": card(), "reps": a.reps, "unit": "GB/s of decoded output (1e9 bytes / device-timed call)", "rows": []}

    f2, o2 = W.config2_text_frames(512, 65536)
    f5, o5 = W.config5_mixed_sizes(256)
    for name, frames, origs, n in (("config2", f2, o2, a.config2_frames), ("config5", f5, o5, a.config5_frames)):
        b = Batch(frames, [len(o) for o in origs], n)
        b.with_dst()
        ms_v = timed(lambda: ctx.verify_batch_device(b.vdescs.data_ptr(), b.results.data_ptr(), n, stream), a.reps)
        nbad_v, _ = check(b.fetch(), n)
        ms_d = timed(lambda: ctx.decode_batch_device(b.ddescs.data_ptr(), b.results.data_ptr(), n, api.FLAG_VERIFY_CHECKSUM, stream), a.reps)
        nbad_d, _ = check(b.fetch(), n)
        row = {"workload": name, "frames": n, "decoded_bytes": b.out_bytes,
               "verify_ms": ms_v, "decode_xxh64_ms": ms_d,
               "verify_gbps_median": b.out_bytes / 1e6 / float(np.median(ms_v)),
               "decode_xxh64_gbps_median": b.out_bytes / 1e6 / float(np.median(ms_d)),
               "failed_frames": {"verify": nbad_v, "decode": nbad_d}}
        print(json.dumps(row), flush=True)
        out["rows"].append(row)
        del b
        torch.cuda.empty_cache()

    free, total = torch.cuda.mem_get_info()
    b = Batch(f2, [len(o) for o in o2], a.huge_frames)
    t0 = time.time()
    ms = timed(lambda: ctx.verify_batch_device(b.vdescs.data_ptr(), b.results.data_ptr(), b.n, stream), 1)
    nbad, first_bad = check(b.fetch(), b.n)
    row = {"workload": "config2 frames, decoded total above device memory", "frames": b.n, "decoded_bytes": b.out_bytes,
           "device_memory_bytes": total, "verify_ms": ms, "verify_gbps": b.out_bytes / 1e6 / ms[-1],
           "frames_not_verified": nbad, "first_not_verified": first_bad, "wall_s": time.time() - t0}
    print(json.dumps(row), flush=True)
    out["rows"].append(row)
    assert b.out_bytes > total and nbad == 0
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        json.dump(out, open(a.out, "w"), indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
