"""Every Layer III kernel selection on mixed batches, against the oracle bit for bit and the float64 model.

Which kernel runs depends on the batch: `build_plan` takes the second generation (v2) when runs average fewer than 16
granules and the first generation with the packed window (v1p) otherwise; the v2 launch switches to its compact
instantiation when a plan has at least two run segments per share; the host entry point cuts batches of 512 frames
or more into a slice pipeline, and batches whose runs are out of order go to one launch.  The mixed corpus of
tests/test_mp3_f64_model.py (every sample rate, mono and stereo, MPEG-1 and MPEG-2 runs side by side) goes through each
of those paths here, and then again in a child process for every selection the environment can force.
"""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from symphonia_b200._native import FMT_S16, MP3_RUN_DTYPE
from tests import _mp3_f64_model as model
from tests import _oracle
from tests import test_mp3_f64_model as f64

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# The selections the environment can force (read once per process, when a context is created):
# SYMGPU_MP3_KERNEL, and SYMGPU_MP3_V2_VARIANT=<warps>:<mode> for every entry of kV2Variants (mp3_kernel_v2.cu).
KERNELS = ("v1", "v1p", "v2")
V2_VARIANTS = ("12:33", "12:0", "12:1", "12:5", "12:17", "12:81", "12:64", "14:33", "14:97", "10:33", "12:129", "12:193")
# Layer I / II: kernel (bit-identical to the oracle) vs the model's polyphase bank, max |pcm - model| / RMS(model) per
# frame-channel: measured 1.0e-06 on the case below.
MPA12_BOUND = 4e-6


def test_every_listed_v2_variant_is_built():
    """V2_VARIANTS is exactly the list the library builds: each entry is accepted, and kV2Variants has no other."""
    import symphonia_b200 as sb
    src = open(os.path.join(ROOT, "symphonia_b200", "csrc", "mp3_kernel_v2.cu")).read()
    table = re.search(r"const V2Variant kV2Variants\[\] = \{(.*?)\};", src, re.S).group(1)
    warps = re.search(r"#define SYMGPU_MP3_V2_NW (\d+)", open(os.path.join(ROOT, "symphonia_b200", "csrc", "mp3_kernel.h")).read()).group(1)
    built = [f"{nw.replace('kMp3V2Warps', warps)}:{mode}" for nw, mode in re.findall(r"V2_VARIANT\((\w+), (\d+)\)", table)]
    assert built == list(V2_VARIANTS)
    lib = sb.lib()
    try:
        for v in V2_VARIANTS:
            assert lib.symgpu_debug_mp3_v2_variant(*map(int, v.split(":"))) == 1, v
        assert lib.symgpu_debug_mp3_v2_variant(12, 2) == 0
    finally:
        lib.symgpu_debug_mp3_v2_variant(*map(int, V2_VARIANTS[0].split(":")))  # the selection is process-wide


# ---- mixed batches in this process ---------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def engine():
    import symphonia_b200 as sb
    eng = sb.Engine(0)
    yield eng
    eng.close()


@pytest.fixture(scope="module")
def cases(oracle):
    """small: the corpus (< 512 frames: one launch); big: two copies of it on distinct streams (>= 512 frames: the slice
    pipeline).  Each with the oracle's PCM and the model's."""
    out = {}
    small = f64.build_corpus()
    for name, (units, spectra, runs) in (("small", small), ("big", f64.concat([small, small]))):
        n_streams = int(runs["stream"].max()) + 1
        rc, want, _ = _oracle.mp3_batch(oracle, units, spectra, runs, n_streams)
        assert rc == 0
        out[name] = (units, spectra, runs, n_streams, want, model.mp3_batch(units, spectra, runs))
    assert len(out["small"][0]) < 512 <= len(out["big"][0])
    return out


def _compare(got, want, ref, units, runs, what):
    g, w = np.ascontiguousarray(got, dtype=np.float32).view(np.uint32), want.view(np.uint32)
    bad = np.nonzero(g != w)
    if len(bad[0]):
        f, c, i = (int(a[0]) for a in bad)
        owner = [int(r["stream"]) for r in runs if r["first_frame"] <= f < r["first_frame"] + r["n_frames"]]
        raise AssertionError(f"{what}: {len(bad[0])} of {g.size} PCM words differ from the oracle; first at frame {f} (stream "
                             f"{owner}) ch {c} sample {i}: gpu {got[f, c, i]!r} oracle {want[f, c, i]!r}")
    err = f64.rel_error(got, ref, units, runs).max()
    assert err < f64.BOUND, f"{what}: {err:.3g} of the granule RMS from the float64 model"


def _host(engine, case, runs=None, n_streams=None):
    units, spectra, runs0, n0, want, ref = case
    runs = runs0 if runs is None else runs
    engine.mp3_streams_alloc(n_streams or n0)
    return engine.mp3_synth_host(units, spectra, runs), units, runs, want, ref


def _with_empty_runs(runs, n_streams, sorted_runs):
    """Zero-frame runs at the front, between runs and at the end, on streams that also have frames elsewhere."""
    out = []
    for k, r in enumerate(runs):
        if k % 5 == 0:
            e = r.copy()
            e["n_frames"], e["stream"] = 0, (int(r["stream"]) + 7) % n_streams
            if not sorted_runs:
                e["first_frame"] = int(runs["first_frame"].max())
            out.append(e)
        out.append(r)
    tail = runs[-1].copy()
    tail["first_frame"], tail["n_frames"] = int(runs["first_frame"][-1] + runs["n_frames"][-1]), 0
    out.append(tail)
    return np.array(out, dtype=MP3_RUN_DTYPE)


@pytest.mark.gpu
def test_mixed_single_launch(engine, cases):
    got, units, runs, want, ref = _host(engine, cases["small"])
    _compare(got, want, ref, units, runs, "mixed corpus, one launch")


@pytest.mark.gpu
def test_mixed_slice_pipeline(engine, cases):
    """>= 512 frames with sorted runs: the slice pipeline, whose memset defines the slots mono and MPEG-2 runs leave."""
    got, units, runs, want, ref = _host(engine, cases["big"])
    _compare(got, want, ref, units, runs, "mixed corpus, slice pipeline")
    engine.mp3_streams_alloc(cases["big"][3])
    again = engine.mp3_synth_host(units, cases["big"][1], runs, out=np.full_like(got, np.nan))
    _compare(again, want, ref, units, runs, "mixed corpus, slice pipeline, into a NaN-filled output buffer")


@pytest.mark.gpu
def test_mixed_unsorted_runs(engine, cases):
    runs = cases["big"][2]
    shuffled = runs[np.random.default_rng(5).permutation(len(runs))]
    got, units, runs, want, ref = _host(engine, cases["big"], shuffled)
    _compare(got, want, ref, units, runs, "mixed corpus, runs in shuffled order")


@pytest.mark.gpu
def test_mixed_permuted_streams(engine, cases):
    for name in ("small", "big"):
        runs = cases[name][2].copy()
        runs["stream"] = np.random.default_rng(6).permutation(len(runs))[runs["stream"]]
        got, units, runs, want, ref = _host(engine, cases[name], runs)
        _compare(got, want, ref, units, runs, f"mixed corpus ({name}), stream indices permuted against the runs")


@pytest.mark.gpu
def test_mixed_with_empty_runs(engine, cases):
    for name in ("small", "big"):
        runs, n = cases[name][2], cases[name][3]
        for sorted_runs in (True, False):
            r = _with_empty_runs(runs, n, sorted_runs)
            got, units, r, want, ref = _host(engine, cases[name], r)
            _compare(got, want, ref, units, r, f"mixed corpus ({name}), zero-frame runs, sorted={sorted_runs}")


@pytest.mark.gpu
def test_mixed_device_entry_point(engine, cases):
    import torch
    dev = torch.device("cuda", 0)
    for name in ("small", "big"):
        units, spectra, runs, n, want, ref = cases[name]
        engine.mp3_streams_alloc(n)
        u_t = torch.from_numpy(np.ascontiguousarray(units).view(np.uint8).reshape(-1)).to(dev)
        s_t = torch.from_numpy(spectra).to(dev)
        p_t = torch.zeros((len(units), 2, 1152), dtype=torch.float32, device=dev)
        torch.cuda.synchronize()
        engine.mp3_synth_dev(u_t, s_t, runs, p_t)
        engine.sync()
        _compare(p_t.cpu().numpy(), want, ref, units, runs, f"mixed corpus ({name}), device entry point")


@pytest.mark.gpu
def test_mixed_refused_in_packed_mode(engine, cases):
    """The packed output stage has no slot for what mono and MPEG-2 runs leave undefined: the call is refused."""
    from symphonia_b200.engine import SymgpuError
    units, spectra, runs, n, _, _ = cases["small"]
    engine.mp3_streams_alloc(n)
    with pytest.raises(SymgpuError) as e:
        engine.mp3_synth_host_packed(units, spectra, runs, FMT_S16)
    assert e.value.status == 2  # SYMGPU_ERR_UNSUPPORTED


@pytest.mark.gpu
def test_layer12_against_the_model_polyphase(engine):
    """Layer I / II synthesis shares the polyphase phases with Layer III: its output against the model's ISO bank."""
    from symphonia_b200 import workloads
    for layer, channels in ((1, 2), (2, 1), (2, 2)):
        x, runs = workloads.mpa12_batch(3, 8, layer=layer, seed=700 + layer, channels=channels)
        n = x.shape[-1]
        engine.mp3_streams_alloc(3)
        got = engine.mpa12_synth_host(x, runs)[..., :32 * n].astype(np.float64)
        ref = np.zeros_like(got)
        for r in runs:
            f = np.arange(int(r["first_frame"]), int(r["first_frame"] + r["n_frames"]))
            for c in range(int(r["channels"]) or 2):
                ref[f, c] = model.polyphase(x[f, c].transpose(0, 2, 1).reshape(-1, 32)).reshape(len(f), 32 * n)
        ch = slice(0, channels)
        rms = np.sqrt((ref[:, ch] ** 2).mean(axis=-1))
        err = np.abs(got[:, ch] - ref[:, ch]).max(axis=-1) / rms
        assert rms.min() > 0 and err.max() < MPA12_BOUND, (layer, channels, err.max())


# ---- every selection, in a child process -----------------------------------------------------------------------------
SELECTIONS = [{"SYMGPU_MP3_KERNEL": k} for k in KERNELS] + \
             [{"SYMGPU_MP3_KERNEL": "v2", "SYMGPU_MP3_V2_VARIANT": v} for v in V2_VARIANTS]


@pytest.mark.gpu
@pytest.mark.parametrize("selection", SELECTIONS, ids=lambda s: "-".join(s.values()))
def test_kernel_selection_in_a_child_process(selection):
    """The mixed cases above and the uniform cases of test_mp3_parity_gpu.py (the zero-copy modes included), with one
    kernel forced.  A variant runs under SYMGPU_MP3_KERNEL=v2 so that long runs reach it too; the 8192-frame case runs
    for the v2 selections, the first generation's home ground being covered by the default selection."""
    k = "mixed_ or test_mp3_parity_gpu"
    if selection["SYMGPU_MP3_KERNEL"] != "v2":
        k = "mixed_ or (test_mp3_parity_gpu and not full_size)"
    env = dict(os.environ, **selection)
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), os.path.join(ROOT, "tests", "test_mp3_parity_gpu.py"),
                        "-m", "gpu", "-x", "-q", "-p", "no:cacheprovider", "-k", k],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert " passed" in r.stdout and "failed" not in r.stdout
    print(selection, r.stdout.strip().splitlines()[-1])
