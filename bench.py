#!/usr/bin/env python
"""bench.py -- decoded audio-seconds/sec of the synthesis back-end, every BASELINE.json config in ONE line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Headline (`value`, `roofline`, `e2e`, `cpu_baseline`): BASELINE config 2 -- MP3 MPEG-1 44.1 kHz stereo, 8192 frames
(64 streams x 128 consecutive frames) per GPU.  `value` is measured with inputs resident in HBM; `e2e` goes through the
reference-facing host entry point (symgpu_mp3_synth_host) with pinned host buffers, H2D + D2H inside the timed region.
`configs` carries the other four: `plumbing` (config 1: one stream, one host call per packet), `aac` (config 3),
`vorbis` (config 4) and `mixed` (config 5: the 65 536-stream MP3 + AAC + Vorbis corpus, stream i on GPU i mod 8 --
every rank decodes 8192 streams, so N = 8 is the whole corpus), each with kernel time, roofline, e2e and its own CPU
baseline.  N > 1 (torchrun): streams shard over ranks, no data-path collective; the one NCCL collective is the
table-blob broadcast at init (weak scaling); every rank checks a sample of its PCM against the oracle.

`--impl reference` times the CPU restatement of the reference's own scalar path (oracle/, built with -march=native on
this box) on all host threads -- the Rust toolchain does not exist here, see DESIGN.md.  Its inputs come from the
oracle's own tables: that arm never maps the product library.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: a benchmark run leaves it as it found it

N_STREAMS = 64
FRAMES_PER_STREAM = 128
N_FRAMES = N_STREAMS * FRAMES_PER_STREAM
N_BUFFER_SETS = 4  # rotating input/output sets: 4 x ~150 MB > 126 MB L2
WORKLOAD = "MP3 MPEG-1 Layer III 44.1kHz stereo, batch=8192 frames (64 streams x 128 frames), synthetic spectra"
# config 5: 65 536 streams over 8 GPUs = 8192 per GPU; 50 % MP3 / 30 % AAC-LC / 20 % Vorbis, MIXED_FRAMES units per stream
MIXED_STREAMS_PER_GPU = 8192
MIXED_SPLIT = (4096, 2458, 1638)
MIXED_FRAMES = 8
METRIC = "decoded audio-seconds/sec (44.1kHz stereo)"


def _dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 6:
                    self.samples.append(parts)
            except Exception:
                pass
            self.stop_flag.wait(0.1)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(float(s[0]) for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(s[2 + k].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.samples[0][1]), "reasons": reasons,
                "samples": len(sm)}


# ---- CPU arm: the oracle (C++ restatement of the reference's scalar path), built for THIS box ---------------------------

def _load_oracle_native():
    """Builds oracle/ with -march=native ON THIS BOX (the CPU baseline must use this host's ISA), into a temporary
    directory: the source tree may be read-only."""
    from tests import _oracle
    try:
        with tempfile.TemporaryDirectory(prefix="symgpu-oracle-") as tmp:
            out = os.path.join(tmp, "liboracle_native.so")
            _oracle.build(arch="-march=native", out=out)
            return _oracle.load(out), "-march=native"
    except Exception:
        return _oracle.load(), "-march=x86-64-v3"


def _oracle_pow43(orc):
    """The POW43 table from the ORACLE's own libm call, so that the reference arm's inputs need nothing of the product."""
    orc.oracle_mp3_pow43.restype = ctypes.c_float
    return np.array([orc.oracle_mp3_pow43(i) for i in range(8207)], dtype=np.float32)


def _repeat(fn, min_seconds):
    """Calls fn() until min_seconds have passed (at least once); (calls, seconds)."""
    fn()  # warm-up: page faults, tables
    n, t0 = 0, time.perf_counter()
    while True:
        fn()
        n += 1
        dt = time.perf_counter() - t0
        if dt >= min_seconds:
            return n, dt


def _cpu_mp3(orc, units, spectra, runs, n_threads, min_seconds):
    from tests import _oracle
    n_streams = int(runs["stream"].max()) + 1
    states = (_oracle.Mp3State * n_streams)()
    pcm = np.zeros((spectra.shape[0], 2, 1152), dtype=np.float32)
    args = (ctypes.byref(states), _oracle.ptr(units), _oracle.ptr(spectra), _oracle.ptr(runs), ctypes.c_uint32(len(runs)),
            _oracle.ptr(pcm), ctypes.c_int(n_threads))
    return _repeat(lambda: orc.oracle_mp3_batch_mt(*args), min_seconds)


def _cpu_aac(orc, units, tns, coeffs, runs, n_threads, min_seconds):
    from tests import _oracle
    n_streams = int(runs["stream"].max()) + 1
    return _repeat(lambda: _oracle.aac_batch(orc, units, tns, coeffs, runs, n_streams, n_threads), min_seconds)


def _cpu_vorbis(orc, wl, n_threads, min_seconds):
    from tests import _oracle
    return _repeat(lambda: _oracle.vorbis_batch(orc, wl, n_threads), min_seconds)


def dump_outputs(out_dir, pcm):
    """Writes the PCM of the last timed headline step as out_dir/mp3_pcm.npy: float32 (frames, 2, 1152) for a fixed
    sample of half the batch's frames (seed 0, in frame order), 38 MB of its 75 MB.  The inputs and the number of steps
    before it follow from the arguments alone, so two builds run with the same arguments can be compared word for word."""
    import torch
    frames = np.sort(np.random.default_rng(0).choice(pcm.shape[0], pcm.shape[0] // 2, replace=False))
    sample = pcm[torch.from_numpy(frames).to(pcm.device)].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "mp3_pcm.npy"), sample)


def _vorbis_algo_bytes(wl):
    n2 = np.where(wl["units"]["block_flag"] == 1, 1 << (int(wl["streams"]["bs1_exp"][0]) - 1), 1 << (int(wl["streams"]["bs0_exp"][0]) - 1))
    return int((n2 * 4 * 2 + 2 * 65 * 2 + 16 + wl["out_len"] * 4 * 2).sum())


def _subset_streams(runs, first_key, count_key, n_keep):
    """The first n_keep runs of a batch whose runs are laid out in order (a bounded sample of whole streams)."""
    r = runs[:n_keep].copy()
    return r, int(r[first_key][-1] + r[count_key][-1])


def cpu_configs(orc, arch, threads, wls, seconds):
    """CPU baselines of every config on `threads` host threads; each a bounded sample (`seconds` of work at least)."""
    from symphonia_b200 import workloads
    out = {}
    label = f"C++ restatement of Symphonia's scalar path, {arch}, {threads} threads (one stream shard per thread)"
    # config 1: one stream, one frame per call, one thread
    u, s, r = wls["plumbing"]
    one = r.copy()
    one["n_frames"] = 1

    def per_packet():
        from tests import _oracle
        states = (_oracle.Mp3State * 1)()
        pcm = np.zeros((1, 2, 1152), dtype=np.float32)
        for f in range(len(u)):
            orc.oracle_mp3_batch_mt(ctypes.byref(states), _oracle.ptr(u[f:f + 1]), _oracle.ptr(s[f:f + 1]), _oracle.ptr(one),
                                    ctypes.c_uint32(1), _oracle.ptr(pcm), ctypes.c_int(1))
    n, dt = _repeat(per_packet, seconds / 3)
    out["plumbing"] = {"value": workloads.mp3_audio_seconds(len(u)) * n / dt, "unit": "audio-s/s", "cores": 1, "kind": "port",
                       "us_per_packet": 1e6 * dt / (n * len(u)),
                       "sample": f"{n} passes over the {len(u)}-frame stream, one call per frame, one thread"}
    au, at, ac, ar = wls["aac"]
    n, dt = _cpu_aac(orc, au, at, ac, ar, threads, seconds)
    out["aac"] = {"value": len(au) * 1024 / 48000.0 * n / dt, "unit": "audio-s/s", "cores": threads, "kind": "port",
                  "sample": f"{n} passes of the same {len(au)}-frame batch ({dt:.1f} s); {label}"}
    wl = wls["vorbis"]
    n, dt = _cpu_vorbis(orc, wl, threads, seconds)
    out["vorbis"] = {"value": float(wl["out_len"].sum()) / 44100.0 * n / dt, "unit": "audio-s/s", "cores": threads, "kind": "port",
                     "sample": f"{n} passes of the same {len(wl['units'])}-packet batch ({dt:.1f} s); {label}"}
    # config 5: a sample of whole streams of each codec (1/8 of this rank's shard), same mix
    (mu, ms, mr), (xu, xt, xc, xr), mwl = wls["mixed"]
    k_mp3, k_aac, k_vor = len(mr) // 8, len(xr) // 8, len(mwl["runs"]) // 8
    r1, f1 = _subset_streams(mr, "first_frame", "n_frames", k_mp3)
    r2, f2 = _subset_streams(xr, "first_frame", "n_frames", k_aac)
    sub = dict(mwl)
    sub["runs"], p3 = _subset_streams(mwl["runs"], "first_packet", "n_packets", k_vor)
    sub["streams"] = mwl["streams"][:k_vor]
    for key in ("units", "floor_y", "residue", "out_len"):
        sub[key] = mwl[key][:p3]
    xt2 = xt[:int(xu[:f2]["tns_first"].max()) + 64] if len(xt) else xt

    def mixed_pass():
        from tests import _oracle
        n_streams = k_mp3
        states = (_oracle.Mp3State * n_streams)()
        pcm = np.zeros((f1, 2, 1152), dtype=np.float32)
        orc.oracle_mp3_batch_mt(ctypes.byref(states), _oracle.ptr(mu[:f1]), _oracle.ptr(ms[:f1]), _oracle.ptr(r1), ctypes.c_uint32(len(r1)),
                                _oracle.ptr(pcm), ctypes.c_int(threads))
        _oracle.aac_batch(orc, xu[:f2], xt2, xc[:f2], r2, k_aac, threads)
        _oracle.vorbis_batch(orc, sub, threads)
    n, dt = _repeat(mixed_pass, seconds)
    audio = workloads.mp3_audio_seconds(f1) + f2 * 1024 / 48000.0 + float(sub["out_len"].sum()) / 44100.0
    out["mixed"] = {"value": audio * n / dt, "unit": "audio-s/s", "cores": threads, "kind": "port",
                    "sample": f"{n} passes over 1/8 of one GPU's shard ({k_mp3} MP3 + {k_aac} AAC + {k_vor} Vorbis streams x "
                              f"{MIXED_FRAMES} frames, {dt:.1f} s); {label}"}
    return out


def make_workloads(rank, pow43=None, mixed=True):
    """Seeded synthetic inputs of every config for one rank (the MP3 headline batch is made by the caller)."""
    from symphonia_b200 import workloads
    base = workloads.SEED_BASE + 1000 * rank
    wls = {}
    wls["plumbing"] = workloads.mp3_batch(1, 128, seed=base + 7, joint=False, pow43=pow43)  # one CBR stereo stream
    wls["aac"] = workloads.aac_batch(N_STREAMS, FRAMES_PER_STREAM, seed=base + 2)
    wls["vorbis"] = workloads.vorbis_batch(N_STREAMS, FRAMES_PER_STREAM, seed=base + 3)
    if mixed:
        n_mp3, n_aac, n_vor = MIXED_SPLIT
        wls["mixed"] = (workloads.mp3_batch(n_mp3, MIXED_FRAMES, seed=base + 51, pow43=pow43),
                        workloads.aac_batch(n_aac, MIXED_FRAMES, seed=base + 52),
                        workloads.vorbis_batch(n_vor, MIXED_FRAMES, seed=base + 53))
    return wls


def run_reference(args):
    """Reference arm: the CPU path on all host threads, same metric / config / unit."""
    rank, _, world = _dist_env()
    if rank != 0:
        return
    from symphonia_b200 import workloads
    orc, arch = _load_oracle_native()
    pow43 = _oracle_pow43(orc)
    threads = min(os.cpu_count() or 1, N_STREAMS)
    units, spectra, runs = workloads.mp3_batch(N_STREAMS, FRAMES_PER_STREAM, seed=workloads.SEED_BASE + 1, pow43=pow43)
    audio_per_pass = workloads.mp3_audio_seconds(N_FRAMES)
    for _ in range(max(args.warmup, 1)):
        _cpu_mp3(orc, units, spectra, runs, threads, 0.0)
    t_total, passes_total = 0.0, 0
    for _ in range(args.steps):
        p, dt = _cpu_mp3(orc, units, spectra, runs, threads, 0.25)  # bounded sample per step
        passes_total += p
        t_total += dt
    value = audio_per_pass * passes_total / t_total
    sample = f"{passes_total} passes of the full 8192-frame batch over {args.steps} steps ({t_total:.2f} s wall)"
    line = {
        "impl": "reference", "metric": METRIC, "value": value,
        "unit": "audio-s/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t_total / passes_total, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "what": "C++ restatement of Symphonia's scalar synthesis path (oracle/), "
                   f"{arch}, one stream shard per thread; the Rust reference cannot be built here"},
        "cpu_baseline": {"value": value, "unit": "audio-s/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if not args.no_configs:
        line["configs"] = cpu_configs(orc, arch, threads, make_workloads(0, pow43=pow43), 1.5)
    print(json.dumps(line), flush=True)


# ---- GPU arm -------------------------------------------------------------------------------------------------------------

def run_ours(args):
    import torch
    import symphonia_b200 as sb
    from symphonia_b200 import workloads
    rank, local_rank, world = _dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    cpus_before = os.sched_getaffinity(0)  # symgpu_ctx_create binds this thread to the GPU's NUMA node
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG_FILE", os.devnull)  # keep NCCL's version banner off stdout (one JSON line)
        dist.init_process_group("nccl", device_id=dev)
    eng = sb.Engine(local_rank)

    # The one collective of this path: broadcast the host-built table blob from rank 0 so that every
    # GPU decodes with byte-identical tables even if host libm builds differ between nodes.
    if world > 1:
        from symphonia_b200 import sharding
        eng.upload_tables(sharding.broadcast_tables(dist, dev, src=0))

    ext = torch.cuda.ExternalStream(eng.cuda_stream, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()

    def pin(a):
        return torch.from_numpy(np.ascontiguousarray(a)).pin_memory()

    def to_dev(a):
        a = np.ascontiguousarray(a)
        return torch.from_numpy(a.view(np.uint8).reshape(-1) if a.dtype.fields else a).to(dev)

    def time_device(step, steps, warmup):
        """(mean per-step ms from per-step events, total ms first-to-last) on the context's stream."""
        for i in range(warmup):
            step(i)
        eng.sync()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        torch.cuda.synchronize()
        with torch.cuda.stream(ext):
            e_first = torch.cuda.Event(enable_timing=True)
            e_last = torch.cuda.Event(enable_timing=True)
            e_first.record()
            for i in range(steps):
                evs[i][0].record()
                step(warmup + i)
                evs[i][1].record()
            e_last.record()
        eng.sync()
        torch.cuda.synchronize()
        barrier()
        return float(np.mean([a.elapsed_time(b) for a, b in evs])), e_first.elapsed_time(e_last)

    def time_host(call, n):
        """2 warm-up calls, then n calls timed one by one on the host clock (each returns after the result is back in
        host memory).  (total seconds, median seconds)"""
        for _ in range(2):
            call()
        barrier()
        per = []
        for _ in range(n):
            t = time.perf_counter()
            call()
            per.append(time.perf_counter() - t)
        return float(np.sum(per)), float(np.median(per))

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"

    def roofline(algo_bytes, kernel_ms, traffic_key=None):
        ach = algo_bytes / (kernel_ms * 1e-3) / 1e9
        traffic = None
        summary = os.path.join(ROOT, "profiles", "r02_ncu_dram_traffic.json")  # per-launch dram bytes of the committed ncu captures
        if traffic_key and os.path.exists(summary):
            traffic = json.load(open(summary)).get(traffic_key)
        return {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                "peak_source": peak_src, "algorithmic_bytes_per_launch": algo_bytes, "kernel_ms": kernel_ms}

    # ---- headline: MP3 config 2 -----------------------------------------------------------------
    units, spectra, runs = workloads.mp3_batch(N_STREAMS, FRAMES_PER_STREAM, seed=workloads.SEED_BASE + 1 + 1000 * rank)
    eng.mp3_streams_alloc(N_STREAMS)
    audio_per_step = workloads.mp3_audio_seconds(N_FRAMES)
    algo_bytes = N_FRAMES * workloads.MP3_ALGO_BYTES_PER_FRAME
    u_pin, s_pin = pin(units.view(np.uint8).reshape(-1)), pin(spectra)
    p_pin = torch.empty((N_FRAMES, 2, 1152), dtype=torch.float32).pin_memory()
    q_pin = torch.empty((N_FRAMES * 1152, 2), dtype=torch.int16).pin_memory()
    g_pin = pin(workloads.mp3_quantize(spectra))
    u_np = u_pin.numpy().view(sb._native.MP3_GC_DTYPE).reshape(N_FRAMES, 2, 2)
    s_np, p_np, q_np, g_np = s_pin.numpy(), p_pin.numpy(), q_pin.numpy(), g_pin.numpy()
    sets = [(to_dev(units), to_dev(spectra), torch.empty((N_FRAMES, 2, 1152), dtype=torch.float32, device=dev))
            for _ in range(N_BUFFER_SETS)]
    torch.cuda.synchronize()

    def step(i):
        u_t, s_t, p_t = sets[i % N_BUFFER_SETS]
        eng.mp3_synth_dev(u_t, s_t, runs, p_t)

    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = eng.launch_count
    t0 = time.perf_counter()
    avg_kernel_ms, total_ms = time_device(step, args.steps, args.warmup)
    wall = time.perf_counter() - t0
    if args.dump_outputs and rank == 0:  # before the untimed launches below overwrite every buffer set
        dump_outputs(args.dump_outputs, sets[(args.warmup + args.steps - 1) % N_BUFFER_SETS][2])
    launches = eng.launch_count - launches0 - args.warmup
    # The clock sampler polls nvidia-smi (a few hundred ms per query, and its driver calls stall CUDA API calls for tens of
    # ms): it covers the device-timed region above and is stopped before the host-timed regions below.  A short timed
    # region may end before three queries have returned: the same launches are then kept going, untimed, until they have.
    t_tail = time.perf_counter()
    tail_launches = 0
    while len(sampler.samples) < 3 and time.perf_counter() - t_tail < 4.0:
        for i in range(50):
            step(i)
        eng.sync()
        tail_launches += 50
    sampler.stop_flag.set()
    sampler.join(timeout=6)

    e2e_steps = max(3, min(args.steps, 20))
    e2e_s, e2e_med = time_host(lambda: eng.mp3_synth_host(u_np, s_np, runs, out=p_np), e2e_steps)
    checksum = float(np.abs(p_np[::512]).sum())
    # every rank checks the PCM of its first two streams (256 frames) against the oracle, bit for bit
    parity_ok = 1.0
    try:
        from tests import _oracle
        orc_chk = _oracle.load()
        two = runs[:2]
        nf2 = int(two["first_frame"][-1] + two["n_frames"][-1])
        rc, want, _ = _oracle.mp3_batch(orc_chk, units[:nf2], spectra[:nf2], two, 2)
        # the e2e calls above ran the same batch e2e_steps + 2 times on streams whose state carried over: compare a fresh run
        eng.mp3_streams_alloc(N_STREAMS)
        got = eng.mp3_synth_host(u_np, s_np, runs)
        parity_ok = float(rc == 0 and bool((got[:nf2].view(np.uint32) == want.view(np.uint32)).all()))
    except Exception as exc:  # the checker is test infrastructure: its absence is reported, not fatal
        parity_ok = -1.0
        sys.stderr.write(f"bench.py: parity check unavailable: {exc}\n")
    e2e16_s, e2e16_med = time_host(lambda: eng.mp3_synth_host_packed(u_np, s_np, runs, sb._native.FMT_S16, out=q_np), e2e_steps)
    e2ec_s, e2ec_med = time_host(lambda: eng.mp3_synth_host_quantized(u_np, g_np, runs, sb._native.FMT_S16, out=q_np), e2e_steps)
    del sets

    # ---- the other configs ------------------------------------------------------------------------
    N_CFG_E2E = 12  # host calls timed for the AAC / Vorbis end-to-end numbers (2.6 ms each): one scheduling hiccup of the host must not
                    # dominate the mean (a 5-call mean once read 9.8 ms with a single ~38 ms outlier)
    cfg_times = {}  # name -> [kernel_ms, total_ms, e2e_s]
    cfg_static = {}
    wls = None
    c_steps = max(3, min(args.steps, 50))
    if not args.no_configs:
        wls = make_workloads(rank)
        # config 1: one stream, one host call per packet (what AudioDecoder::decode does with a batch of one)
        pu, ps, pr = wls["plumbing"]
        eng.mp3_streams_alloc(1)
        pu_pin, ps_pin = pin(pu.view(np.uint8).reshape(-1)), pin(ps)
        pp_pin = torch.empty((1, 2, 1152), dtype=torch.float32).pin_memory()
        pu_np = pu_pin.numpy().view(sb._native.MP3_GC_DTYPE).reshape(len(pu), 2, 2)
        ps_np, pp_np = ps_pin.numpy(), pp_pin.numpy()
        one = pr.copy()
        one["n_frames"] = 1

        def per_packet():
            for f in range(len(pu)):
                eng.mp3_synth_host(pu_np[f:f + 1], ps_np[f:f + 1], one, out=pp_np)
        tot, _ = time_host(per_packet, 5)
        cfg_times["plumbing"] = [0.0, 0.0, tot / 5]
        cfg_static["plumbing"] = {
            "workload": "MP3 CBR 320 kbit/s-class 44.1kHz stereo, 1 stream x 128 frames, ONE host call per packet "
                        "(symgpu_mp3_synth_host with a batch of one: H2D + kernel + D2H inside every call)",
            "audio_s_per_step": workloads.mp3_audio_seconds(len(pu)), "packets_per_step": len(pu),
            "h2d": len(pu) * (256 + 9216), "d2h": len(pu) * 9216}

        # config 3: AAC-LC
        au, at, ac, ar = wls["aac"]
        eng.aac_streams_alloc(N_STREAMS)
        a_sets = [(to_dev(au), to_dev(at) if len(at) else torch.zeros(8, device=dev), to_dev(ac),
                   torch.empty((len(au), 2, 1024), dtype=torch.float32, device=dev)) for _ in range(N_BUFFER_SETS)]
        k_ms, t_ms = time_device(lambda i: eng.aac_synth_dev(a_sets[i % N_BUFFER_SETS][0], a_sets[i % N_BUFFER_SETS][1], len(at),
                                                             a_sets[i % N_BUFFER_SETS][2], ar, a_sets[i % N_BUFFER_SETS][3]), c_steps, 3)
        del a_sets
        au_pin, at_pin, ac_pin = pin(au.view(np.uint8).reshape(-1)), pin(at.view(np.uint8).reshape(-1)), pin(ac)
        ap_pin = torch.empty((len(au), 2, 1024), dtype=torch.float32).pin_memory()
        au_np = au_pin.numpy().view(sb._native.AAC_UNIT_DTYPE).reshape(len(au), 2)
        at_np = at_pin.numpy().view(sb._native.AAC_TNS_DTYPE)
        tot, _ = time_host(lambda: eng.aac_synth_host(au_np, at_np, ac_pin.numpy(), ar, out=ap_pin.numpy()), N_CFG_E2E)
        cfg_times["aac"] = [k_ms, t_ms / c_steps, tot / N_CFG_E2E]
        cfg_static["aac"] = {"workload": f"AAC-LC 48kHz stereo, batch={len(au)} frames (64 streams x 128), TNS in 20% of channel-frames "
                                         f"({len(at)} filters), all four window sequences",
                             "audio_s_per_step": len(au) * 1024 / 48000.0, "algo": len(au) * workloads.AAC_ALGO_BYTES_PER_FRAME,
                             "h2d": au.nbytes + at.nbytes + ac.nbytes, "d2h": len(au) * 8192, "traffic_key": "aac"}

        # config 4: Vorbis
        wl = wls["vorbis"]
        eng.vorbis_streams_set(wl["streams"])
        eng.vorbis_floors_set(wl["floors"])
        slot = wl["slot"]
        v_sets = [(to_dev(wl["units"]), to_dev(wl["floor_y"].view(np.int16)), to_dev(wl["residue"]),
                   torch.zeros((len(wl["units"]), 2, slot), dtype=torch.float32, device=dev)) for _ in range(N_BUFFER_SETS)]
        k_ms, t_ms = time_device(lambda i: eng.vorbis_synth_dev(v_sets[i % N_BUFFER_SETS][0], v_sets[i % N_BUFFER_SETS][1],
                                                                v_sets[i % N_BUFFER_SETS][2], wl["runs"], slot,
                                                                v_sets[i % N_BUFFER_SETS][3]), c_steps, 3)
        del v_sets
        vr_pin, vy_pin = pin(wl["residue"]), pin(wl["floor_y"])
        vp_pin = torch.empty((len(wl["units"]), 2, slot), dtype=torch.float32).pin_memory()
        tot, _ = time_host(lambda: eng.vorbis_synth_host(wl["units"], vy_pin.numpy(), vr_pin.numpy(), wl["runs"], slot, out=vp_pin.numpy()), N_CFG_E2E)
        cfg_times["vorbis"] = [k_ms, t_ms / c_steps, tot / N_CFG_E2E]
        long_share = float((wl["units"]["block_flag"] == 1).mean())
        cfg_static["vorbis"] = {"workload": f"Vorbis 44.1kHz stereo coupled, blocksizes 256/2048, batch={len(wl['units'])} packets "
                                            f"(64 streams x 128, {100 * long_share:.0f}% long)",
                                "audio_s_per_step": float(wl["out_len"].sum()) / 44100.0, "algo": _vorbis_algo_bytes(wl),
                                "h2d": wl["units"].nbytes + wl["floor_y"].nbytes + wl["residue"].nbytes,
                                "d2h": len(wl["units"]) * 2 * slot * 4, "traffic_key": "vorbis"}

        # config 5: this rank's 8192 streams of the 65 536-stream corpus (stream i -> GPU i mod 8), three launches per step
        (mu, ms_, mr), (xu, xt, xc, xr), mwl = wls["mixed"]
        eng.mp3_streams_alloc(len(mr))
        eng.aac_streams_alloc(len(xr))
        eng.vorbis_streams_set(mwl["streams"])
        eng.vorbis_floors_set(mwl["floors"])
        d_mu, d_ms, d_mp = to_dev(mu), to_dev(ms_), torch.empty((len(mu), 2, 1152), dtype=torch.float32, device=dev)
        d_xu, d_xt, d_xc = to_dev(xu), to_dev(xt) if len(xt) else torch.zeros(8, device=dev), to_dev(xc)
        d_xp = torch.empty((len(xu), 2, 1024), dtype=torch.float32, device=dev)
        d_vu, d_vy, d_vr = to_dev(mwl["units"]), to_dev(mwl["floor_y"].view(np.int16)), to_dev(mwl["residue"])
        d_vp = torch.zeros((len(mwl["units"]), 2, mwl["slot"]), dtype=torch.float32, device=dev)

        def mixed_step(i):
            eng.mp3_synth_dev(d_mu, d_ms, mr, d_mp)
            eng.aac_synth_dev(d_xu, d_xt, len(xt), d_xc, xr, d_xp)
            eng.vorbis_synth_dev(d_vu, d_vy, d_vr, mwl["runs"], mwl["slot"], d_vp)
        k_ms, t_ms = time_device(mixed_step, min(c_steps, 20), 3)
        del d_mu, d_ms, d_mp, d_xu, d_xt, d_xc, d_xp, d_vu, d_vy, d_vr, d_vp
        m_pins = [pin(mu.view(np.uint8).reshape(-1)), pin(ms_), torch.empty((len(mu), 2, 1152), dtype=torch.float32).pin_memory(),
                  pin(xc), torch.empty((len(xu), 2, 1024), dtype=torch.float32).pin_memory(),
                  pin(mwl["residue"]), torch.empty((len(mwl["units"]), 2, mwl["slot"]), dtype=torch.float32).pin_memory()]
        mu_np = m_pins[0].numpy().view(sb._native.MP3_GC_DTYPE).reshape(len(mu), 2, 2)

        def mixed_host():
            eng.mp3_synth_host(mu_np, m_pins[1].numpy(), mr, out=m_pins[2].numpy())
            eng.aac_synth_host(xu, xt, m_pins[3].numpy(), xr, out=m_pins[4].numpy())
            eng.vorbis_synth_host(mwl["units"], mwl["floor_y"], m_pins[5].numpy(), mwl["runs"], mwl["slot"], out=m_pins[6].numpy())
        tot, _ = time_host(mixed_host, 3)
        cfg_times["mixed"] = [k_ms, t_ms / min(c_steps, 20), tot / 3]
        audio = workloads.mp3_audio_seconds(len(mu)) + len(xu) * 1024 / 48000.0 + float(mwl["out_len"].sum()) / 44100.0
        algo = len(mu) * workloads.MP3_ALGO_BYTES_PER_FRAME + len(xu) * workloads.AAC_ALGO_BYTES_PER_FRAME + _vorbis_algo_bytes(mwl)
        cfg_static["mixed"] = {
            "workload": f"mixed corpus, 65 536 streams over 8 GPUs (stream i on GPU i mod 8): this GPU's {MIXED_STREAMS_PER_GPU} streams = "
                        f"{len(mr)} MP3 + {len(xr)} AAC-LC + {len(mwl['runs'])} Vorbis x {MIXED_FRAMES} frames, one launch per codec per step, "
                        "state of every stream through HBM",
            "audio_s_per_step": audio, "algo": algo, "streams_this_job": MIXED_STREAMS_PER_GPU * world,
            "h2d": mu.nbytes + ms_.nbytes + xu.nbytes + xt.nbytes + xc.nbytes + mwl["units"].nbytes + mwl["floor_y"].nbytes + mwl["residue"].nbytes,
            "d2h": len(mu) * 9216 + len(xu) * 8192 + len(mwl["units"]) * 2 * mwl["slot"] * 4}
        del m_pins

    # ---- max over ranks ------------------------------------------------------------------------
    names = list(cfg_times)
    flat = [total_ms, e2e_s, avg_kernel_ms, e2e16_s, e2ec_s] + [x for n in names for x in cfg_times[n]]
    tt = torch.tensor(flat, dtype=torch.float64, device=dev)
    ok = torch.tensor([parity_ok], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    vals = [float(x) for x in tt.cpu()]
    total_ms, e2e_s, avg_kernel_ms, e2e16_s, e2ec_s = vals[:5]
    for k, n in enumerate(names):
        cfg_times[n] = vals[5 + 3 * k: 8 + 3 * k]

    if rank == 0:
        line = {
            "metric": METRIC,
            "value": world * audio_per_step * args.steps / (total_ms * 1e-3),
            "unit": "audio-s/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "frames_per_gpu": N_FRAMES, "parallelism": f"streams sharded over {world} GPU(s)",
                       "l2": f"rotating {N_BUFFER_SETS} input/output buffer sets ({N_BUFFER_SETS * 151} MB) > 126 MB L2",
                       "fma": "disabled (bit-exact parity with the reference)",
                       "kernel": os.environ.get("SYMGPU_MP3_KERNEL", "auto (per launch plan; this batch of 256-granule runs: mp3_synth_kernel<16,16,0,1>, "
                                                                     "the first-generation kernel with the packed window phase)")},
            "roofline": dict(roofline(algo_bytes, avg_kernel_ms, "mp3"),
                             note="FMA is off for parity, so the kernel is FP32-pipe bound, not HBM bound: the no-FMA floor for this "
                                  "batch is ~31 us (1.1e9 f32 lane-ops at the measured 35.9e12/s) vs 23 us at the HBM peak; traffic "
                                  "(when not null) is dram bytes per launch from the ncu capture committed in profiles/"),
            "e2e": {"value": world * audio_per_step * e2e_steps / e2e_s, "unit": "audio-s/s",
                    "h2d_bytes_per_step": N_FRAMES * (256 + 9216), "d2h_bytes_per_step": N_FRAMES * 9216,
                    "ms_per_step": 1e3 * e2e_s / e2e_steps, "ms_per_step_median": 1e3 * e2e_med, "checksum": checksum},
            "e2e_s16": {"value": world * audio_per_step * e2e_steps / e2e16_s, "unit": "audio-s/s",
                        "h2d_bytes_per_step": N_FRAMES * (256 + 9216), "d2h_bytes_per_step": N_FRAMES * 4608,
                        "ms_per_step": 1e3 * e2e16_s / e2e_steps, "ms_per_step_median": 1e3 * e2e16_med,
                        "note": "symgpu_mp3_synth_host_packed: output stage (interleave + f32->i16, SURVEY 8f N3) on the "
                                "device, so half the bytes come back; not the headline (the decoder trait returns f32)"},
            "e2e_compact": {"value": world * audio_per_step * e2e_steps / e2ec_s, "unit": "audio-s/s",
                            "h2d_bytes_per_step": N_FRAMES * (256 + 4608), "d2h_bytes_per_step": N_FRAMES * 4608,
                            "ms_per_step": 1e3 * e2ec_s / e2e_steps, "ms_per_step_median": 1e3 * e2ec_med,
                            "note": "symgpu_mp3_synth_host_quantized: the Huffman stage's i16 values in (POW43 lookup on the "
                                    "device), interleaved i16 out -- what a CPU front-end + sound card pair would exchange"},
            "gpu_launches": launches,
            "parity": {"ranks_bit_exact_vs_oracle": world if float(ok.cpu()[0]) == 1.0 else 0,
                       "what": "first two streams (256 frames) of every rank's batch through symgpu_mp3_synth_host, uint32 equality; "
                               "-1 = checker unavailable" if float(ok.cpu()[0]) < 0 else
                               "first two streams (256 frames) of every rank's batch through symgpu_mp3_synth_host, uint32 equality"},
            "clocks": dict(sampler.summary(), window=f"device-timed region + {tail_launches} untimed launches of the same step"),
            "numa": {"node_rank0": eng.numa_node, "cpus_rank0": len(os.sched_getaffinity(0)), "cpus_before": len(cpus_before),
                     "what": "symgpu_ctx_create binds the rank's thread (and its first-touched pinned buffers) to the GPU's NUMA node"},
            "wall_s": wall,
        }
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            os.sched_setaffinity(0, cpus_before)  # the CPU arm may use every core of the box
            orc, arch = _load_oracle_native()
            threads = min(os.cpu_count() or 1, N_STREAMS)
            p1, d1 = _cpu_mp3(orc, units, spectra, runs, 1, 3.0)
            pn, dn = _cpu_mp3(orc, units, spectra, runs, threads, 3.0)
            line["cpu_baseline"] = {
                "value": audio_per_step * pn / dn, "unit": "audio-s/s", "cores": threads, "kind": "port",
                "single_thread_value": audio_per_step * p1 / d1,
                "sample": f"{pn} passes of the same 8192-frame batch on {threads} threads ({dn:.1f} s) and {p1} passes on "
                          f"1 thread ({d1:.1f} s); C++ restatement of Symphonia's scalar path, {arch}"}
            if wls is not None:
                cpu = cpu_configs(orc, arch, threads, wls, 1.5)
        if cfg_times:
            configs = {}
            for n in names:
                k_ms, step_ms, e2e_sec = cfg_times[n]
                st = cfg_static[n]
                audio = st["audio_s_per_step"]
                c = {"workload": st["workload"],
                     "e2e": {"value": world * audio / e2e_sec, "unit": "audio-s/s", "ms_per_step": 1e3 * e2e_sec,
                             "h2d_bytes_per_step": st["h2d"], "d2h_bytes_per_step": st["d2h"]}}
                if n == "plumbing":
                    c["value"] = c["e2e"]["value"]
                    c["us_per_packet"] = 1e6 * e2e_sec / st["packets_per_step"]
                    c["note"] = ("there is no device-resident variant of a one-packet decode() call: value is the end-to-end number; "
                                 "a stream needs 26 ms of audio per packet, so real time = 26 122 us per packet")
                else:
                    c["value"] = world * audio / (step_ms * 1e-3)
                    c["kernel_ms"] = k_ms
                    c["roofline"] = roofline(st["algo"], k_ms, st.get("traffic_key"))
                if "streams_this_job" in st:
                    c["streams"] = st["streams_this_job"]
                c["unit"] = "audio-s/s"
                if cpu and n in cpu:
                    c["cpu_baseline"] = cpu[n]
                configs[n] = c
            line["configs"] = configs
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="only the MP3 headline (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the PCM of the last timed headline step (rank 0) as DIR/mp3_pcm.npy, a seeded half of its frames")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed: it needs --impl ours")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
