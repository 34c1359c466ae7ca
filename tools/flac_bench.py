#!/usr/bin/env python3
"""FLAC to PCM on one B200: the restoration followed by the host interleave that decode_flac used to run, against the restoration
with the output stage on the device (symgpu_flac_decode_*) in S16 and S32.  One JSON line (--out FILE also writes it there):

  batch   DESIGN §3's FLAC size, 2048 frames x 4096 samples of 16-bit stereo (64 generated frames repeated; every copy has its own
          samples, 67 MB of int32 input, inside the 126 MB L2 once resident).
            kernel_ms  CUDA events on the engine's stream around symgpu_flac_restore_dev (predict + finish) and symgpu_flac_decode_dev
                       (predict + finish_pack); the input planes are restored from a pristine copy before the start event
            wall_ms    host clock around flac_restore_host + decode.flac_interleave (the old path, int32 out) and around
                       flac_decode_host (S16 / S32 out), each of which ends in a device synchronise
            pcie_bytes what each path copies: descriptors + samples in, restored planes or packed samples out
  files   32 FLAC files (4 distinct, 16-bit stereo, 40 frames of 4096): today's decode_flac per file as it was (plan, restore_host,
          flac_interleave) against decode.decode_files in S16 and S32 (one symgpu_flac_decode_host call for all 32).
The three variants of each workload alternate, three rounds; the best round is reported.  The card's name and power limit are read
in the same run.  Not part of bench.py; numbers go to DESIGN §9c."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from symphonia_b200 import _native as nat  # noqa: E402
from symphonia_b200 import decode, workloads  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def design_batch(times=32):
    frames, subs, samples = workloads.flac_batch(64, 4096, seed=4242, bps=16, channels=2)
    F, S, N = len(frames), len(subs), len(samples)
    fr = np.concatenate([frames] * times)
    fr["first_subframe"] += np.repeat(np.arange(times, dtype=np.uint32) * S, F)
    sb = np.concatenate([subs] * times)
    sb["offset"] += np.repeat(np.arange(times, dtype=np.uint64) * N, S)
    plan = dict(frames=fr, subframes=sb, samples=np.tile(samples, times), channels=2,
                total_frames=int(sb["n"][fr["first_subframe"]].astype(np.int64).sum()))
    return plan


def timed(torch, stream, fn, before, iters=20, warmup=3):
    """Median / min milliseconds of fn() between CUDA events on `stream`; before() runs outside the window."""
    times = []
    for k in range(warmup + iters):
        before()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fn()
        b.record(stream)
        b.synchronize()
        if k >= warmup:
            times.append(a.elapsed_time(b))
    return float(np.median(times)), float(np.min(times))


def wall(fn, iters=5):
    best = 1e9
    for _ in range(iters):
        t0 = time.perf_counter()
        fn()
        best = min(best, time.perf_counter() - t0)
    return best * 1e3


def bench_batch(torch, eng):
    plan = design_batch()
    fr, sb, smp = plan["frames"], plan["subframes"], plan["samples"]
    dst = decode.flac_dst(plan)
    total = plan["total_frames"] * 2
    # the paths must agree before they are timed
    ref = decode.flac_interleave(plan, eng.flac_restore_host(fr, sb, smp.copy()))
    assert (eng.flac_decode_host(fr, sb, smp, dst, nat.FMT_S32, total).reshape(-1, 2) == ref).all()
    assert (eng.flac_decode_host(fr, sb, smp, dst, nat.FMT_S16, total).reshape(-1, 2) == (ref >> 16).astype(np.int16)).all()
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    fr_t, sb_t, dst_t = dev(fr.view(np.uint8)), dev(sb.view(np.uint8)), dev(dst.view(np.int64))
    pristine, work = dev(smp), dev(smp)
    outs = {fmt: torch.empty(total * np.dtype(nat.FMT_NUMPY[fmt]).itemsize, dtype=torch.uint8, device="cuda") for fmt in (nat.FMT_S16, nat.FMT_S32)}
    st = torch.cuda.ExternalStream(eng.cuda_stream)
    restore = lambda: work.copy_(pristine)  # noqa: E731
    kern = {"restore": [], "decode_s16": [], "decode_s32": []}
    walls = {"restore_then_interleave": [], "decode_s16": [], "decode_s32": []}
    for _ in range(3):
        kern["restore"].append(timed(torch, st, lambda: eng.flac_restore_dev(fr_t, len(fr), sb_t, len(sb), work), restore))
        for fmt, key in ((nat.FMT_S16, "decode_s16"), (nat.FMT_S32, "decode_s32")):
            kern[key].append(timed(torch, st, lambda: eng.flac_decode_dev(fr_t, len(fr), sb_t, len(sb), work, dst_t, fmt, outs[fmt]), restore))
        walls["restore_then_interleave"].append(wall(lambda: decode.flac_interleave(plan, eng.flac_restore_host(fr, sb, smp.copy())), iters=2))
        walls["decode_s16"].append(wall(lambda: eng.flac_decode_host(fr, sb, smp, dst, nat.FMT_S16, total)))
        walls["decode_s32"].append(wall(lambda: eng.flac_decode_host(fr, sb, smp, dst, nat.FMT_S32, total)))
    desc = fr.nbytes + sb.nbytes
    pcie = {"restore_then_interleave": dict(h2d=desc + smp.nbytes, d2h=smp.nbytes),
            "decode_s16": dict(h2d=desc + dst.nbytes + smp.nbytes, d2h=total * 2),
            "decode_s32": dict(h2d=desc + dst.nbytes + smp.nbytes, d2h=total * 4)}
    return {"batch": dict(frames=len(fr), samples_per_channel=plan["total_frames"],
                          kernel_ms={k: dict(median=min(m for m, _ in v), min=min(b for _, b in v)) for k, v in kern.items()},
                          wall_ms={k: min(v) for k, v in walls.items()}, pcie_bytes=pcie)}


def bench_files(eng, n_files):
    from tests import test_flac_frontend as tf
    distinct = [tf._flac_file(950 + k, 16, 2, 4096, n_frames=40)[0] for k in range(4)]
    files = [distinct[k % 4] for k in range(n_files)]

    def old_path():                 # decode_flac as it was: planar int32 back, interleaved per frame and channel in Python
        for data in files:
            p = decode.flac_plan(data)
            decode.flac_interleave(p, eng.flac_restore_host(p["frames"], p["subframes"], p["samples"].copy()))
    got = decode.decode_files(eng, files, nat.FMT_S32)
    p = decode.flac_plan(distinct[0])
    assert (got[0][0] == decode.flac_interleave(p, eng.flac_restore_host(p["frames"], p["subframes"], p["samples"].copy()))).all()
    res = {"per_file_restore_then_interleave": [], "decode_files_s16": [], "decode_files_s32": []}
    for _ in range(3):
        res["per_file_restore_then_interleave"].append(wall(old_path, iters=1))
        res["decode_files_s16"].append(wall(lambda: decode.decode_files(eng, files, nat.FMT_S16), iters=1))
        res["decode_files_s32"].append(wall(lambda: decode.decode_files(eng, files, nat.FMT_S32), iters=1))
    t0 = time.perf_counter()
    plans, _ = decode.plan_files(files)
    plan_ms = (time.perf_counter() - t0) * 1e3
    audio = sum(q["total_frames"] / q["sample_rate"] for q in plans)
    return {"files": dict(files=n_files, audio_s=audio, plan_files_ms=plan_ms, wall_ms={k: min(v) for k, v in res.items()})}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--files", type=int, default=32)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import symphonia_b200 as sb
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: these numbers are only measured on the GPU")
    res = {"card": card(), "host_cores": os.cpu_count()}
    with sb.Engine(0) as eng:
        res.update(bench_batch(torch, eng))
        res.update(bench_files(eng, args.files))
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
