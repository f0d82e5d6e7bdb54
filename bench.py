#!/usr/bin/env python3
"""bench.py -- decompressed GB/s of the batch decode path (BASELINE.json config 2).

One step = decode the whole batch once: 1 Mi independent 64 KiB frames of synthetic text
(zstd level 3, checksum flag on) per GPU.  N distinct frames are generated with the host's
libzstd and physically replicated in HBM (different addresses, so no L2 reuse of the input).

Arms
  default            this repo's CUDA path through the C ABI (czb_decode_batch_device); `value` is
                     device-timed with inputs resident in HBM; `e2e` goes through
                     czb_decode_batch_host_packed with pinned HOST buffers (H2D + decode + D2H timed).
  --impl reference   the reference's algorithm on the host cores: the C restatement in oracle/
                     (kind "port": the Cairo itself cannot run here, SURVEY.md section 8c), all host threads,
                     each step a bounded sample of the same workload.

Prints ONE JSON line on rank 0.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

FRAME_SIZE = 65536
METRIC = "decompressed GB/s (device-timed, whole box) at 1/2/4/8 B200; % of HBM roofline"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames", type=int, default=1 << 20, help="frames per GPU (config 2: 1 Mi)")
    ap.add_argument("--distinct", type=int, default=2048, help="distinct frames generated on the host, then replicated")
    ap.add_argument("--e2e-frames", type=int, default=0, help="frames in the host-buffer e2e run (0 = choose by host RAM)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-sample-frames", type=int, default=131072)
    ap.add_argument("--verify-checksum", action="store_true", help="include the XXH64 kernel in the timed region")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the config3/4/5 and config5_sharded keys")
    ap.add_argument("--no-link-ceiling", action="store_true", help="skip the raw H2D+D2H ceiling of the e2e record")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last step returned (a fixed, seeded "
                    "sample of the frames: decoded bytes and result fields; rank 0) as DIR/<name>.npy")
    return ap.parse_args()


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        d = json.load(open(path))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clock / throttle-reason sampling during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_workload(distinct, seed=1234):
    from cairo_zstd_b200 import workloads as W
    frames, origs = W.config2_text_frames(distinct, FRAME_SIZE, seed=seed)
    return frames, origs


DUMP_FRAMES = 128  # frames --dump-outputs keeps: their decoded bytes as float32 come to 128 x 64 KiB x 4 B = 32 MiB


def dump_pick(n):
    """The frames --dump-outputs writes: a sample that depends on the batch size only, so two builds dump the same frames."""
    return np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_FRAMES), replace=False))


def dump_outputs(out_dir, pick, decoded, results):
    """Write the sampled frames' outputs: frame_index.npy (which frames of the batch), decoded.npy (one row of decoded bytes per
    frame, float32) and result_<field>.npy (each field of the frames' results, float64; RES_DT names the fields)."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "frame_index.npy"), pick.astype(np.float64))
    np.save(os.path.join(out_dir, "decoded.npy"), decoded.astype(np.float32))
    for name in results.dtype.names:
        np.save(os.path.join(out_dir, f"result_{name}.npy"), results[name].astype(np.float64))


# --------------------------------------------------------------------------------------------
# reference arm: the oracle port on the host cores
# --------------------------------------------------------------------------------------------
def cpu_oracle_throughput(frames, origs, sample_frames, threads):
    """Decode `sample_frames` frames (the distinct set cycled) with the oracle on `threads` threads.
    Returns (GB/s of decompressed bytes, seconds, decoded bytes, per-frame results)."""
    import oracle_lib as O
    L = O.lib()
    n = sample_frames
    d = len(frames)
    src_bufs = [C.create_string_buffer(f, len(f)) for f in frames]
    srcs = (C.c_void_p * n)(*[C.addressof(src_bufs[i % d]) for i in range(n)])
    lens = (C.c_size_t * n)(*[len(frames[i % d]) for i in range(n)])
    out = np.empty(n * FRAME_SIZE, dtype=np.uint8)
    base = out.ctypes.data
    dsts = (C.c_void_p * n)(*[base + i * FRAME_SIZE for i in range(n)])
    caps = (C.c_size_t * n)(*([FRAME_SIZE] * n))
    results = (O.OracleResult * n)()
    t0 = time.perf_counter()
    fails = L.oracle_decode_batch(n, srcs, lens, dsts, caps, 0, results, threads)
    dt = time.perf_counter() - t0
    assert fails == 0
    k = n - 1
    assert out[k * FRAME_SIZE:(k + 1) * FRAME_SIZE].tobytes() == origs[k % d]
    return n * FRAME_SIZE / dt / 1e9, dt, out, results


def run_reference(args, rank, world):
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    frames, origs = make_workload(min(args.distinct, 512))
    sample = args.cpu_sample_frames
    for _ in range(args.warmup):
        cpu_oracle_throughput(frames, origs, min(sample, 2048), threads)
    vals, times = [], []
    for _ in range(args.steps):
        v, dt, out, results = cpu_oracle_throughput(frames, origs, sample, threads)
        vals.append(v); times.append(dt)
    if args.dump_outputs:
        pick = dump_pick(sample)
        dump_outputs(args.dump_outputs, pick, out.reshape(sample, FRAME_SIZE)[pick], np.frombuffer(results, dtype=RES_DT)[pick])
    total_t = sum(times)
    value = args.steps * sample * FRAME_SIZE / total_t / 1e9
    desc = f"{sample} frames x 64 KiB per step ({len(frames)} distinct, cycled), oracle C port, {threads} threads"
    line = {
        "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total_t / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic", "impl": "reference",
        "config": {"workload": "config2: independent 64 KiB frames of synthetic text, zstd level 3, checksum flag on",
                   "frames_per_step": sample, "note": "bounded sample of the 1 Mi-frame workload; host cores only"},
        "cpu_baseline": {"value": value, "unit": "GB/s", "cores": threads, "kind": "port", "sample": desc},
        "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------------------------
def run_b200(args, rank, world, local_rank):
    import torch
    import cairo_zstd_b200 as czb
    from cairo_zstd_b200 import api

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this arm has no CPU fallback (use --impl reference)")
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    peak, peak_src = measured_peak()

    # ---- workload: `distinct` frames, replicated to `frames` per GPU ----
    t_gen = time.perf_counter()
    frames, origs = make_workload(args.distinct, seed=1234 + 7919 * rank)
    n = args.frames
    d = len(frames)
    reps = (n + d - 1) // d
    flens = np.array([len(f) for f in frames], dtype=np.int64)
    fpad = (flens + 15) & ~15
    foff = np.concatenate([[0], np.cumsum(fpad)])
    set_bytes = int(foff[-1])
    host_set = np.zeros(set_bytes, dtype=np.uint8)
    for i, f in enumerate(frames):
        host_set[foff[i]:foff[i] + len(f)] = np.frombuffer(f, dtype=np.uint8)
    t_gen = time.perf_counter() - t_gen

    src_set = torch.from_numpy(host_set).to(dev)
    src_all = src_set.repeat(reps)                     # physical replication in HBM
    dst_all = torch.empty(n * FRAME_SIZE, dtype=torch.uint8, device=dev)
    idx = np.arange(n, dtype=np.int64)
    descs_np = np.zeros((n, 4), dtype=np.uint64)
    descs_np[:, 0] = src_all.data_ptr() + (idx // d) * set_bytes + foff[idx % d]
    descs_np[:, 1] = flens[idx % d]
    descs_np[:, 2] = dst_all.data_ptr() + idx * FRAME_SIZE
    descs_np[:, 3] = FRAME_SIZE
    descs = torch.from_numpy(descs_np.view(np.uint8).reshape(-1)).to(dev)
    results = torch.zeros(n * C.sizeof(api.FrameResult), dtype=torch.uint8, device=dev)
    comp_bytes = int(flens[idx % d].sum())
    out_bytes = n * FRAME_SIZE

    ctx = czb.Context(local_rank)
    stream = torch.cuda.current_stream(dev)
    flags = api.FLAG_VERIFY_CHECKSUM if args.verify_checksum else 0

    def step():
        ctx.decode_batch_device(descs.data_ptr(), results.data_ptr(), n, flags, stream.cuda_stream)

    def barrier():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        step()
    barrier()
    ctx.profile_enable(True)
    ctx.profile_collect()
    launches0 = ctx.kernel_launches()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for _ in range(args.steps):
        step()
    ev1.record(stream)
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    clocks = sampler.stop()
    launches = ctx.kernel_launches() - launches0
    prof = ctx.profile_collect()
    ctx.profile_enable(False)

    # ---- correctness of what was timed: every frame OK, sampled outputs byte-identical, checksums ----
    res_np = results.cpu().numpy().view(np.dtype([("status", "<i4"), ("blocks", "<u4"), ("bytes_read", "<u8"), ("bytes_written", "<u8"),
                                                  ("content_size", "<u8"), ("window", "<u8"), ("chk_data", "<u4"), ("chk_calc", "<u4"),
                                                  ("has_chk", "<i4"), ("finished", "<i4")]))
    if args.dump_outputs and rank == 0:
        pick = dump_pick(n)
        decoded = dst_all.view(n, FRAME_SIZE)[torch.from_numpy(pick).to(dev)].cpu().numpy()
        dump_outputs(args.dump_outputs, pick, decoded, res_np[pick])
    assert (res_np["status"] == 0).all(), f"{int((res_np['status'] != 0).sum())} frames failed"
    assert (res_np["bytes_written"] == FRAME_SIZE).all() and (res_np["finished"] == 1).all()
    for k in list(range(0, min(n, d))) + [n - 1, n // 2]:
        got = dst_all[k * FRAME_SIZE:(k + 1) * FRAME_SIZE].cpu().numpy().tobytes()
        assert got == origs[k % d], f"frame {k}: output differs from the original"
    # one more pass with the XXH64 kernel on (SURVEY 8 row f1), device-timed the same way: reported beside the headline
    evc0, evc1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        ctx.decode_batch_device(descs.data_ptr(), results.data_ptr(), n, api.FLAG_VERIFY_CHECKSUM, stream.cuda_stream)  # warm-up of k_xxh64
        evc0.record(stream)
        ctx.decode_batch_device(descs.data_ptr(), results.data_ptr(), n, api.FLAG_VERIFY_CHECKSUM, stream.cuda_stream)
        evc1.record(stream)
    torch.cuda.synchronize(dev)
    ms_with_checksum = evc0.elapsed_time(evc1)
    res_np = results.cpu().numpy().view(res_np.dtype)
    assert (res_np["chk_calc"] == res_np["chk_data"]).all(), "XXH64 of the output != frame trailer"

    # ---- aggregate over ranks: max time, sum bytes ----
    t_ms = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    tot = torch.tensor([float(out_bytes), float(comp_bytes)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms_total_max = float(t_ms.item())
    out_all_ranks, comp_all_ranks = float(tot[0].item()), float(tot[1].item())
    ms_per_step = ms_total_max / args.steps
    value = out_all_ranks / (ms_per_step * 1e-3) / 1e9

    # ---- roofline of the dominant kernel (live CUDA-event times over the timed region) ----
    dom = max(prof.items(), key=lambda kv: kv[1][0]) if prof else ("none", (0.0, 0))
    kernel_ms_total = sum(v[0] for v in prof.values())
    dom_name, (dom_ms, dom_launches) = dom
    alg_bytes_step = out_bytes + comp_bytes                   # C_i + D_i summed over this GPU's frames (SURVEY 8d)
    alg_bytes_per_launch = alg_bytes_step * args.steps / max(dom_launches, 1)
    dom_avg_ms = dom_ms / max(dom_launches, 1)
    achieved = alg_bytes_per_launch / (dom_avg_ms * 1e-3) / 1e9 if dom_avg_ms else 0.0
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                "kernel": "k_" + dom_name, "kernel_avg_ms": dom_avg_ms, "kernel_launches": dom_launches,
                "peak_source": peak_src,
                "whole_path": {"achieved": alg_bytes_step / (ms_per_step * 1e-3) / 1e9,
                               "frac": alg_bytes_step / (ms_per_step * 1e-3) / 1e9 / peak},
                "kernel_share_of_step": {k: v[0] / kernel_ms_total for k, v in prof.items()} if kernel_ms_total else {},
                "kernel_ms_per_step": {k: v[0] / args.steps for k, v in prof.items()}}
    # DRAM traffic of the dominant kernel from the committed ncu --set full capture (bytes per frame x frames per launch)
    traffic_path = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(traffic_path):
        try:
            tj = json.load(open(traffic_path))
            tk = tj["kernels"].get("k_" + dom_name)
            frames_per_launch = n * args.steps / max(dom_launches, 1)
            if tk:
                roofline["traffic"] = tk["bytes_per_frame"] * frames_per_launch
                roofline["traffic_source"] = ("profiles/r02_traffic.json: dram__bytes_read.sum + dram__bytes_write.sum per frame from this round's "
                                              "ncu --set full capture of the same kernels (scripts/r02b_final.sh, scripts/ncu_traffic.py), x frames per launch")
                roofline["algorithmic_bytes_per_launch"] = alg_bytes_per_launch
                # issue-slot fraction next to the HBM fraction: warp instructions the kernel executes (same capture) against what
                # the SMs can issue in the kernel's live average launch time (4 schedulers per SM, one warp instruction per cycle)
                import torch as _t
                sms = _t.cuda.get_device_properties(dev).multi_processor_count
                clk = (clocks.get("sm_mhz") or 1965.0) * 1e6
                roofline["issue_slots"] = {"warp_inst_per_launch": tk["warp_inst_per_frame"] * frames_per_launch,
                                           "frac": tk["warp_inst_per_frame"] * frames_per_launch / (dom_avg_ms * 1e-3 * sms * 4 * clk),
                                           "note": "fraction of the SMs' issue slots the dominant kernel uses; the kernel is latency / issue bound, not HBM bound"}
            wp = sum(k["warp_inst_per_frame"] for kn, k in tj["kernels"].items())
            roofline["whole_path"]["issue_slot_frac"] = wp * n / (ms_per_step * 1e-3 * sms * 4 * clk)
            # DRAM bytes of all decode kernels per frame (same capture) over the algorithmic C + D per frame of THIS run
            roofline["whole_path"]["dram_traffic_over_algorithmic"] = sum(k["bytes_per_frame"] for k in tj["kernels"].values()) / (alg_bytes_step / n)
        except Exception as e:
            sys.stderr.write(f"traffic/issue-slot annotation skipped: {e}\n")

    # ---- e2e: host buffers through czb_decode_batch_host_packed ----
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, ctx, frames, origs, flens, n, dev, dist, torch)

    # ---- the other BASELINE configs (extra keys; config 2 above is the bench line) ----
    del src_all, dst_all, descs, results
    torch.cuda.empty_cache()
    others, sharded = {}, None
    if not args.no_other_configs:
        if world == 1:
            others = other_configs(args, ctx, torch, dev, peak)
        sharded = config5_sharded(args, ctx, torch, dev, dist, rank, world)

    # ---- CPU baseline beside it (rank 0, N=1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        v, dt, _, _ = cpu_oracle_throughput(frames[:512], origs[:512], args.cpu_sample_frames, threads)
        cpu = {"value": v, "unit": "GB/s", "cores": threads, "kind": "port",
               "sample": f"{args.cpu_sample_frames} of the same frames ({dt:.1f} s wall), oracle C port, one frame per task"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic",
            "config": {"workload": "config2: 1 Mi independent 64 KiB frames of synthetic text, zstd level 3, checksum flag on"
                       if n == (1 << 20) else f"config2 shape at {n} frames per GPU",
                       "frames_per_gpu": n, "frame_bytes": FRAME_SIZE, "distinct_frames": d, "replication": "physical copies in HBM",
                       "compression_ratio": out_bytes / comp_bytes, "parallelism": f"frames sharded over {world} GPU(s), no collective",
                       "l2": "inputs (>= 20 GB) and outputs (>= 60 GB) far exceed the 126 MB L2; no flush needed",
                       "checksum_in_timed_region": bool(args.verify_checksum), "gen_seconds": t_gen},
            "roofline": roofline, "clocks": clocks, "gpu_launches": int(launches),
            "with_checksum": {"value": out_bytes / (ms_with_checksum * 1e-3) / 1e9, "unit": "GB/s", "ms_per_step": ms_with_checksum,
                              "note": "rank 0, one pass (after one warm-up pass) with CZB_FLAG_VERIFY_CHECKSUM (XXH64 of every output on the device, "
                                      "compared with the frame trailer); SURVEY 8 row f1, outside the headline's timed region"},
        }
        line.update(others)
        if sharded is not None:
            line["config5_sharded"] = sharded
        if e2e is not None:
            line["e2e"] = e2e
        if cpu is not None:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


# --------------------------------------------------------------------------------------------
# the other BASELINE configs as extra keys of the bench line (parity-test configs, device-timed, every frame verified)
# --------------------------------------------------------------------------------------------
RES_DT = np.dtype([("status", "<i4"), ("blocks", "<u4"), ("bytes_read", "<u8"), ("bytes_written", "<u8"), ("content_size", "<u8"),
                   ("window", "<u8"), ("chk_data", "<u4"), ("chk_calc", "<u4"), ("has_chk", "<i4"), ("finished", "<i4")])


def device_time_frames(ctx, torch, dev, frames, origs, pick, reps_of, steps=3):
    """Device-timed decode of the frames `pick` (indices into the replicated batch: index i = rep * n0 + distinct) on this GPU.
    The distinct set is uploaded once per replica (physical copies, different addresses).  Every output is verified: status,
    size, and XXH64 computed on the device against the frame trailer (one extra, untimed pass).  Returns (ms, out_bytes, comp_bytes)."""
    from cairo_zstd_b200 import api
    n0 = len(frames)
    flens = np.array([len(f) for f in frames], dtype=np.int64)
    olens = np.array([len(o) for o in origs], dtype=np.int64)
    foff = np.concatenate([[0], np.cumsum((flens + 15) & ~15)])
    host = np.zeros(int(foff[-1]), dtype=np.uint8)
    for i, f in enumerate(frames):
        host[foff[i]:foff[i] + len(f)] = np.frombuffer(f, dtype=np.uint8)
    pick = np.asarray(pick, dtype=np.int64)
    n = int(pick.size)
    if n == 0:
        return 0.0, 0, 0
    src = torch.from_numpy(host).to(dev).repeat(reps_of)
    dl = olens[pick % n0]
    doff = np.concatenate([[0], np.cumsum((dl + 15) & ~15)])
    dst = torch.empty(int(doff[-1]) + 64, dtype=torch.uint8, device=dev)
    d = np.zeros((n, 4), dtype=np.uint64)
    d[:, 0] = src.data_ptr() + (pick // n0) * int(foff[-1]) + foff[pick % n0]
    d[:, 1] = flens[pick % n0]
    d[:, 2] = dst.data_ptr() + doff[:-1]
    d[:, 3] = dl
    descs = torch.from_numpy(d.view(np.uint8).reshape(-1)).to(dev)
    results = torch.zeros(n * C.sizeof(api.FrameResult), dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream(dev)
    for _ in range(2):
        ctx.decode_batch_device(descs.data_ptr(), results.data_ptr(), n, 0, st.cuda_stream)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(steps):
        ctx.decode_batch_device(descs.data_ptr(), results.data_ptr(), n, 0, st.cuda_stream)
    e1.record(st)
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    ctx.decode_batch_device(descs.data_ptr(), results.data_ptr(), n, api.FLAG_VERIFY_CHECKSUM, st.cuda_stream)
    torch.cuda.synchronize(dev)
    res = results.cpu().numpy().view(RES_DT)
    assert (res["status"] == 0).all(), f"{int((res['status'] != 0).sum())} frames failed"
    assert (res["bytes_written"] == dl.astype(np.uint64)).all() and (res["finished"] == 1).all()
    assert (res["chk_calc"] == res["chk_data"]).all(), "XXH64 of an output != its frame trailer"
    k = n - 1
    o = int(doff[k])
    assert dst[o:o + int(dl[k])].cpu().numpy().tobytes() == origs[int(pick[k]) % n0]
    return ms, int(dl.sum()), int(flens[pick % n0].sum())


def other_configs(args, ctx, torch, dev, peak):
    """config3/4/5 on one GPU (rank 0, N=1): device-timed, all outputs verified by XXH64."""
    from cairo_zstd_b200 import workloads as W
    out = {}
    specs = [
        ("config3", "literal-heavy: 1024 frames of 1 MiB (16 distinct x 64), 128 KiB blocks, 4-stream Huffman with treeless tables, raw and RLE blocks",
         lambda: W.config3_literal_heavy(16), 64),
        ("config4", "long window: 64 frames of 17 MiB (2 distinct x 32), windowLog 23, matches ~6 MiB back",
         lambda: W.config4_long_window(2, total=17 << 20), 32),
        ("config4_512", "the same long-window frames as a batch that fills the machine: 512 frames of 17 MiB (2 distinct x 256)",
         lambda: W.config4_long_window(2, total=17 << 20), 256),
        ("config5", "mixed sizes: 8192 frames of 1 KiB..4 MiB log-uniform (512 distinct x 16), level 3",
         lambda: W.config5_mixed_sizes(512, hi=4 << 20), 16),
    ]
    cache = {}
    for key, desc, gen, reps in specs:
        if key == "config4_512" and "config4" in cache:
            frames, origs = cache["config4"]  # same generator, same seed
        else:
            frames, origs = gen()
        cache[key] = (frames, origs)
        n0 = len(frames)
        ms, ob, cb = device_time_frames(ctx, torch, dev, frames, origs, np.arange(n0 * reps), reps)
        out[key] = {"value": ob / ms / 1e6, "unit": "GB/s", "ms": ms, "frames": n0 * reps, "out_bytes": ob, "ratio": ob / cb,
                    "frac_of_hbm_peak": (ob + cb) / ms / 1e6 / peak, "workload": desc,
                    "verified": "status, size and device XXH64 == trailer for every frame"}
        torch.cuda.empty_cache()
    return out


def config5_sharded(args, ctx, torch, dev, dist, rank, world):
    """BASELINE config 5 as north_star states it: ONE mixed-size batch, the same at every N, sharded over the ranks by the host
    (czb_partition_frames: largest first by compressed + decoded bytes), no collective on the data path.  Strong scaling:
    value = whole-batch decoded bytes / max-over-ranks device time."""
    import cairo_zstd_b200 as czb
    from cairo_zstd_b200 import workloads as W
    frames, origs = W.config5_mixed_sizes(512, hi=4 << 20)   # seeded: identical on every rank
    # 131 072 frames (73 GB decoded): large enough that at N = 8 a rank's share is still many times its largest frame -- a frame is
    # one sequential stream (a 4 MiB frame takes ~10 ms however few others there are), so a batch of a few GB cannot scale
    # (65 536 frames: 174.6 GB/s on one GPU, 1134 on eight = 0.81; 8192 frames: 155 -> 188 on two)
    n0, reps = len(frames), 256
    n = n0 * reps
    cost = np.array([len(f) + len(o) for f, o in zip(frames, origs)], dtype=np.int64)
    cost_all = cost[np.arange(n) % n0]
    shard_of, load = czb.partition_frames([int(x) for x in cost_all], world)
    pick = np.nonzero(np.asarray(shard_of) == rank)[0]
    ms, ob, cb = device_time_frames(ctx, torch, dev, frames, origs, pick, reps)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    per_rank = [torch.zeros_like(t) for _ in range(world)] if dist is not None else [t]
    if dist is not None:
        dist.all_gather(per_rank, t)
    ms_ranks = [float(x.item()) for x in per_rank]
    total_out = int(np.array([len(o) for o in origs], dtype=np.int64).sum()) * reps
    return {"value": total_out / max(ms_ranks) / 1e6, "unit": "GB/s", "scaling": "strong", "frames": n, "out_bytes": total_out,
            "ms_max_over_ranks": max(ms_ranks), "ms_per_rank": ms_ranks,
            "shard_cost_bytes": [int(x) for x in load],
            "imbalance": max(load) / (sum(load) / world) - 1.0,
            "partition": "czb_partition_frames (C ABI): largest first by compressed + decoded bytes",
            "workload": "mixed sizes: 131072 frames of 1 KiB..4 MiB log-uniform (512 distinct x 256), the same batch at every N",
            "verified": "status, size and device XXH64 == trailer for every frame of every shard"}


def link_ceiling(torch, dev, dist, h2d_bytes, d2h_bytes, h_src, h_dst):
    """Raw concurrent H2D + D2H of the same byte counts as one e2e step, no decode: what the host link gives this rank while
    every other rank does the same.  Returns seconds (max over ranks)."""
    cudart = torch.cuda.cudart()
    s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    chunk = 1 << 30
    d_in = torch.empty(min(h2d_bytes, chunk), dtype=torch.uint8, device=dev)
    d_out = torch.empty(min(d2h_bytes, chunk), dtype=torch.uint8, device=dev)
    hs = torch.from_numpy(h_src)
    hd = torch.from_numpy(h_dst)

    def one():
        with torch.cuda.stream(s_in):
            for o in range(0, h2d_bytes, chunk):
                m = min(chunk, h2d_bytes - o)
                d_in[:m].copy_(hs[o:o + m], non_blocking=True)
        with torch.cuda.stream(s_out):
            for o in range(0, d2h_bytes, chunk):
                m = min(chunk, d2h_bytes - o)
                hd[o:o + m].copy_(d_out[:m], non_blocking=True)
        s_in.synchronize(); s_out.synchronize()

    one()
    if dist is not None:
        dist.barrier()
    t0 = time.perf_counter()
    one()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    del cudart
    return float(t.item())



def run_e2e(args, ctx, frames, origs, flens, n_dev_frames, dev, dist, torch):
    """Same metric through the host-pointer C-ABI call: pinned host input and output buffers,
    H2D of the compressed frames + decode + D2H of the decoded bytes, all inside the timed region."""
    from cairo_zstd_b200 import api
    d = len(frames)
    n = args.e2e_frames
    if n <= 0:
        # as much of the workload as host RAM allows with margin (pinned in+out ~ 93 KB per frame)
        try:
            avail = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE")
        except Exception:
            avail = 32 << 30
        world = dist.get_world_size() if dist is not None else 1
        per_rank = avail * 0.55 / world
        n = int(min(n_dev_frames, per_rank // (FRAME_SIZE + int(flens.mean()) + 128)))
        n = max(d, (n // d) * d)
    idx = np.arange(n, dtype=np.int64)
    lens = flens[idx % d]
    src_off = np.concatenate([[0], np.cumsum((lens + 15) & ~15)]).astype(np.uint64)
    src_off_true_end = src_off[:-1] + lens.astype(np.uint64)
    dst_off = (np.arange(n + 1, dtype=np.uint64) * FRAME_SIZE)
    t0 = time.perf_counter()
    # exact-size host buffers, page-locked with cudaHostRegister (torch's pinned allocator rounds sizes up to a power of two)
    cudart = torch.cuda.cudart()

    def pinned(nbytes):
        a = np.zeros(nbytes, dtype=np.uint8)
        rc = cudart.cudaHostRegister(a.ctypes.data, nbytes, 0)
        assert int(rc) == 0, f"cudaHostRegister failed: {rc}"
        return a

    h_src = pinned(int(src_off[-1]))
    h_dst = pinned(n * FRAME_SIZE)
    h_res = pinned(n * C.sizeof(api.FrameResult))
    pin_s = time.perf_counter() - t0
    # fill the pinned input: one padded copy of the distinct set, tiled
    set_np = np.zeros(int(((flens + 15) & ~15).sum()), dtype=np.uint8)
    o = 0
    for f in frames:
        set_np[o:o + len(f)] = np.frombuffer(f, dtype=np.uint8)
        o += (len(f) + 15) & ~15
    hs = h_src
    reps = n // d
    for r in range(reps):
        hs[r * set_np.size:(r + 1) * set_np.size] = set_np
    # frames are padded to 16 B in the packed buffer; the decoder takes src_len up to the next frame, which is allowed
    # ("src_len may extend past the frame"): the padding bytes are never consumed.
    del src_off_true_end

    def step():
        ctx.decode_batch_packed(h_src.ctypes.data, src_off, h_dst.ctypes.data, dst_off, n, h_res.ctypes.data, 0)

    step()  # warm-up (also sizes the staging buffers)
    if dist is not None:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        step()
    dt = time.perf_counter() - t0
    res_np = h_res.view(np.dtype([("status", "<i4"), ("blocks", "<u4"), ("bytes_read", "<u8"), ("bytes_written", "<u8"),
                                  ("content_size", "<u8"), ("window", "<u8"), ("chk_data", "<u4"), ("chk_calc", "<u4"),
                                  ("has_chk", "<i4"), ("finished", "<i4")]))
    assert (res_np["status"] == 0).all() and (res_np["bytes_written"] == FRAME_SIZE).all()
    hd = h_dst
    for k in (0, n // 3, n - 1):
        assert hd[k * FRAME_SIZE:(k + 1) * FRAME_SIZE].tobytes() == origs[k % d], f"e2e frame {k} differs"
    t = torch.tensor([dt], dtype=torch.float64, device=dev)
    b = torch.tensor([float(n * FRAME_SIZE)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(b, op=dist.ReduceOp.SUM)
    dt_max = float(t.item())
    value = float(b.item()) * args.e2e_steps / dt_max / 1e9
    ceiling = None
    if not args.no_link_ceiling:
        try:
            # torch sees the registered numpy memory as pinned only through its own allocator; non_blocking copies from
            # cudaHostRegister'ed memory still run at full link rate (the driver recognises the registration)
            sec = link_ceiling(torch, dev, dist, int(src_off[-1]), int(n * FRAME_SIZE), h_src, h_dst)
            ceiling = float(b.item()) / sec / 1e9
        except Exception as e:  # the ceiling is context, never a reason to lose the bench line
            ceiling = None
            sys.stderr.write(f"link ceiling skipped: {e}\n")
    for a in (h_src, h_dst, h_res):
        cudart.cudaHostUnregister(a.ctypes.data)
    world = dist.get_world_size() if dist is not None else 1
    return {"value": value, "link_ceiling": ceiling, "frac_of_link": (value / ceiling) if ceiling else None,
            "link_ceiling_note": "decoded GB/s if the step were only its concurrent H2D (compressed bytes) + D2H (decoded bytes) copies, "
                                 "all ranks at once, no decode; max over ranks", "unit": "GB/s", "h2d_bytes_per_step": int(src_off[-1]) * world, "d2h_bytes_per_step": int(n * FRAME_SIZE) * world,
            "frames_per_step": int(n) * world, "steps": args.e2e_steps, "ms_per_step": 1e3 * dt_max / args.e2e_steps,
            "timing": "host wall clock around czb_decode_batch_host_packed (it returns when outputs are in host memory)",
            "pin_seconds": pin_s,
            "note": "pinned host buffers; frame count bounded by host RAM" if n < n_dev_frames else "pinned host buffers; full workload"}


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
