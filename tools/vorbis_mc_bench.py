#!/usr/bin/env python3
"""Multichannel Vorbis on one B200, three numbers and the card they were taken on (one JSON line; --out FILE also writes it there):

  synth     symgpu_vorbis_mc_synth_dev on 8192 packets at C = 6 (64 streams x 128 packets, 5.1 coupling steps), device-resident
            inputs, CUDA events around every call, two input sets rotated (each 6 x 8192 x 1024 floats = 201 MB, past the 126 MB L2);
            the call decouples the residue in place, so the set is restored from a pristine copy before the start event.
            symgpu_vorbis_synth_dev on a stereo batch of the same packet count beside it, for scale.
  pack      symgpu_pcm_pack_mapped_dev (the 5.1 channel map) against symgpu_pcm_pack_dev on the same C = 6 PCM, S16, alternated.
  files     decode.decode_files wall clock (host clock around the call, which ends in a device synchronise) on a corpus of 5.1 files
            against the same corpus written with two channels; the plan (CPU) share on its own.

Not part of bench.py; numbers go to DESIGN 9."""
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


def timed(torch, stream, fn, before=None, iters=20, warmup=3):
    """Median / min milliseconds of fn() between CUDA events on `stream` (the engine's: its kernels run there, not on torch's
    current stream); before(k) runs outside the window."""
    times = []
    for k in range(warmup + iters):
        if before:
            before(k)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fn(k)
        b.record(stream)
        b.synchronize()
        if k >= warmup:
            times.append(a.elapsed_time(b))
    return float(np.median(times)), float(np.min(times))


def bench_synth(torch, eng):
    out = {}
    st = torch.cuda.ExternalStream(eng.cuda_stream)
    wl = workloads.vorbis_mc_batch(n_streams=64, packets_per_stream=128, channels=6)
    P, C, slot = len(wl["units"]), int(wl["channels"]), int(wl["slot"])
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    units, fy = dev(wl["units"].view(np.uint8)), dev(wl["floor_y"])
    pristine = dev(wl["residue"])
    res = [torch.empty_like(pristine) for _ in range(2)]
    pcm = [torch.empty((P, C, slot), dtype=torch.float32, device="cuda") for _ in range(2)]
    eng.vorbis_mc_streams_set(wl["streams"])
    eng.vorbis_floors_set(wl["floors"])
    med, best = timed(torch, st, lambda k: eng.vorbis_mc_synth_dev(units, fy, res[k % 2], wl["runs"], C, slot, pcm[k % 2]),
                      before=lambda k: res[k % 2].copy_(pristine))
    out["mc_synth_c6_8192_ms"] = dict(median=med, min=best, packets=P, channels=C)
    sw = workloads.vorbis_batch(64, 128)
    su, sf, sr = dev(sw["units"].view(np.uint8)), dev(sw["floor_y"]), dev(sw["residue"])
    sp = [torch.empty((len(sw["units"]), 2, sw["slot"]), dtype=torch.float32, device="cuda") for _ in range(2)]
    eng.vorbis_streams_set(sw["streams"])
    eng.vorbis_floors_set(sw["floors"])
    med, best = timed(torch, st, lambda k: eng.vorbis_synth_dev(su, sf, sr, sw["runs"], sw["slot"], sp[k % 2]))
    out["stereo_synth_8192_ms"] = dict(median=med, min=best, packets=len(sw["units"]))
    return out


def bench_pack(torch, eng):
    P, C, slot = 8192, 6, 1024
    rng = np.random.default_rng(5)
    pcm = torch.from_numpy((rng.standard_normal((P, C, slot)) * 0.5).astype(np.float32)).cuda()
    spans = np.zeros(P, dtype=nat.PCM_SPAN_DTYPE)
    spans["src"] = np.arange(P, dtype=np.uint64) * C * slot
    spans["plane_stride"], spans["frames"] = slot, 640
    spans["dst_frame"] = np.arange(P, dtype=np.uint64) * 640
    sp = torch.from_numpy(spans.view(np.uint8)).cuda()
    out = [torch.empty(P * 640 * C, dtype=torch.int16, device="cuda") for _ in range(2)]
    m = decode.vorbis_pack_map(C)
    st = torch.cuda.ExternalStream(eng.cuda_stream)
    res = {}
    for rnd in range(2):   # alternated: plain, mapped, plain, mapped
        res.setdefault("plain", []).append(timed(torch, st, lambda k: eng.pcm_pack_dev(pcm, sp, P, C, nat.FMT_S16, out[k % 2]))[0])
        res.setdefault("mapped", []).append(timed(torch, st, lambda k: eng.pcm_pack_dev_mapped(pcm, sp, P, C, m, nat.FMT_S16, out[k % 2]))[0])
    moved = P * 640 * C * (4 + 2)
    return {"pack_c6_s16_ms": {k: min(v) for k, v in res.items()}, "pack_bytes_moved": moved}


def bench_files(eng, n_files, packets):
    from tests import test_vorbis_multichannel as tmc
    out = {}
    for C, couplings in ((6, [(0, 2), (3, 4), (1, 0)]), (2, [(0, 1)])):
        distinct = [tmc.mc_file(900 + k, C, n_packets=packets, couplings=couplings)[0] for k in range(4)]
        files = [distinct[k % 4] for k in range(n_files)]
        t0 = time.perf_counter()
        plans, _ = decode.plan_files(files)
        plan_s = time.perf_counter() - t0
        decode.decode_files(eng, files, nat.FMT_S16)   # warm-up
        best = 1e9
        for _ in range(3):
            t0 = time.perf_counter()
            decode.decode_files(eng, files, nat.FMT_S16)
            best = min(best, time.perf_counter() - t0)
        audio = sum(p["total_frames"] / p["sample_rate"] for p in plans)
        out[f"decode_files_c{C}"] = dict(files=n_files, packets_per_file=packets, audio_s=audio, wall_s=best, plan_s=plan_s,
                                         audio_s_per_s=audio / best, batch=sorted({p["kind"] for p in plans}))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--files", type=int, default=32)
    ap.add_argument("--packets", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import symphonia_b200 as sb
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: these numbers are only measured on the GPU")
    res = {"card": card(), "host_cores": os.cpu_count()}
    with sb.Engine(0) as eng:
        res.update(bench_synth(torch, eng))
        res.update(bench_pack(torch, eng))
        res.update(bench_files(eng, args.files, args.packets))
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
