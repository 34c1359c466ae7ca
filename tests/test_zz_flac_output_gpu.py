"""FLAC from file bytes to any sample format on the device: `symgpu_flac_decode_host` / `_dev` (restoration + FromSample<i32> +
interleaving in one call) against the restoration oracle followed by the restated conversion and placement of test_flac_output.py,
`decode.decode_flac` in every format, FLAC in `decode_files`, and the C++ plug-in decoder `GpuFlacDecoder`."""
import subprocess

import numpy as np
import pytest

from symphonia_b200 import _native as nat
from symphonia_b200 import decode, workloads
from tests import test_flac_output as tfo
from tests import test_oracle_kat_flac as kat

pytestmark = [pytest.mark.gpu]


@pytest.fixture(scope="module")
def engine():
    import symphonia_b200 as sb
    with sb.Engine(0) as eng:
        yield eng


def _batch(n_frames, block, seed, bps, channels, gaps=True):
    """workloads.flac_batch (sub-frame planes with gaps between them: short blocks keep their full-size slot) with output positions
    that leave a few unused samples between frames when `gaps`."""
    frames, subs, samples = workloads.flac_batch(n_frames, block, seed=seed, bps=bps, channels=channels)
    n = subs["n"][frames["first_subframe"]].astype(np.int64) * channels
    pad = np.random.default_rng(seed).integers(0, 5, n_frames) if gaps else np.zeros(n_frames, dtype=np.int64)
    dst = np.concatenate([[0], np.cumsum(n + pad)[:-1]]).astype(np.uint64)
    return frames, subs, samples, dst, int((n + pad).sum())


def _expected(frames, subs, restored, dst, total, fmt):
    """The oracle's planes placed and converted; samples no frame writes are zero (also in U8, where a converted 0 is 128)."""
    want = tfo.from_s32(tfo.place(frames, subs, restored, dst, total), fmt)
    covered = np.zeros(total, dtype=bool)
    for f, fr in enumerate(frames):
        n = int(subs[int(fr["first_subframe"])]["n"]) * int(fr["channels"])
        covered[int(dst[f]):int(dst[f]) + n] = True
    want[~covered] = 0
    return want


def _tiled(times):
    """DESIGN §3's FLAC size (2048 frames x 4096 samples, 16-bit stereo) as 64 generated frames repeated: each copy its own samples."""
    frames, subs, samples = workloads.flac_batch(64, 4096, seed=4242, bps=16, channels=2)
    F, S, N = len(frames), len(subs), len(samples)
    fr = np.concatenate([frames] * times)
    fr["first_subframe"] += np.repeat(np.arange(times, dtype=np.uint32) * S, F)
    sb = np.concatenate([subs] * times)
    sb["offset"] += np.repeat(np.arange(times, dtype=np.uint64) * N, S)
    n = sb["n"][fr["first_subframe"]].astype(np.int64) * 2
    dst = np.concatenate([[0], np.cumsum(n)[:-1]]).astype(np.uint64)
    return fr, sb, np.tile(samples, times), dst, int(n.sum())


SPECS = [(8, 1, 64), (12, 2, 97), (16, 2, 576), (20, 6, 300), (24, 8, 256), (32, 1, 512), (32, 2, 128), (16, 2, 4096)]


@pytest.mark.parametrize("bps,channels,block", SPECS)
def test_decode_host_equals_oracle_in_every_format(engine, oracle, bps, channels, block):
    frames, subs, samples, dst, total = _batch(24, block, 1000 + bps * 10 + channels, bps, channels)
    if channels == 2:
        assert set(frames["assignment"].tolist()) == {0, 1, 2, 3}
    rc, restored = kat._restore(oracle, frames, subs, samples)
    assert rc == 0
    kept = samples.copy()
    for fmt in tfo.FORMATS:
        got = engine.flac_decode_host(frames, subs, samples, dst, fmt, total)
        want = _expected(frames, subs, restored, dst, total, fmt)
        assert got.dtype == want.dtype and got.view(np.uint8).tobytes() == want.view(np.uint8).tobytes(), fmt
    assert (samples == kept).all()          # the host variant leaves its input alone


def test_decode_host_at_design_size(engine, oracle):
    frames, subs, samples, dst, total = _tiled(32)
    assert len(frames) == 2048 and int(subs["n"].max()) == 4096
    rc, restored = kat._restore(oracle, frames, subs, samples)
    assert rc == 0
    placed = tfo.place(frames, subs, restored, dst, total)
    for fmt in tfo.FORMATS:
        got = engine.flac_decode_host(frames, subs, samples, dst, fmt, total)
        assert got.view(np.uint8).tobytes() == tfo.from_s32(placed, fmt).view(np.uint8).tobytes(), fmt


def test_decode_dev_equals_host(engine):
    import torch
    for bps, channels, block in ((16, 2, 576), (24, 8, 256), (8, 1, 64)):
        frames, subs, samples, dst, total = _batch(16, block, 77 + channels, bps, channels)
        for fmt in tfo.FORMATS:
            want = engine.flac_decode_host(frames, subs, samples, dst, fmt, total)
            itemsize = np.dtype(nat.FMT_NUMPY[fmt]).itemsize
            out_t = torch.zeros(total * itemsize, dtype=torch.uint8, device="cuda")
            engine.flac_decode_dev(torch.from_numpy(frames.view(np.uint8)).cuda(), len(frames), torch.from_numpy(subs.view(np.uint8)).cuda(),
                                   len(subs), torch.from_numpy(samples.copy()).cuda(), torch.from_numpy(dst.view(np.int64)).cuda(), fmt, out_t)
            engine.sync()
            assert out_t.cpu().numpy().tobytes() == want.view(np.uint8).tobytes(), (bps, channels, fmt)


def test_malformed_input_is_refused_before_the_device(engine, oracle):
    import symphonia_b200 as sb
    frames, subs, samples, dst, total = _batch(4, 64, 7, 16, 2)
    sentinel = np.full(total, 0x5A5A, dtype=np.int16)
    bad = subs.copy()
    bad[0]["type"], bad[0]["order"] = nat.FLAC_LPC, 40          # LPC order above 32: a decode error, as restore_host refuses it
    cases = [(frames, bad, dst, nat.FMT_S16, 1)]
    over = dst.copy()
    over[-1] = total - 1                                        # the last frame's samples would leave `out`
    cases.append((frames, subs, over, nat.FMT_S16, 3))
    cases.append((frames, subs, dst, 9, 6))                      # no such format
    for fr, sf, d, fmt, status in cases:
        out = sentinel.copy()
        with pytest.raises(sb.SymgpuError) as e:
            engine.flac_decode_host(fr, sf, samples, d, fmt, out=out)
        assert e.value.status == status
        assert (out == sentinel).all()
    good = engine.flac_decode_host(frames, subs, samples, dst, nat.FMT_S16, total)   # still healthy
    rc, restored = kat._restore(oracle, frames, subs, samples)
    assert rc == 0 and (good == _expected(frames, subs, restored, dst, total, nat.FMT_S16)).all()


def test_decode_flac_every_format(engine):
    for k, (bps, channels, block) in enumerate(tfo.FLAC_SPECS):
        data, want = tfo.tf._flac_file(900 + k, bps, channels, block)
        base, rate = decode.decode_flac(engine, data)
        assert rate == 44100 and base.dtype == np.int32 and base.shape == want.shape and (base == want).all()
        for fmt in tfo.FORMATS:
            got, _ = decode.decode_flac(engine, data, fmt)
            assert got.shape == want.shape and got.tobytes() == tfo.from_s32(base, fmt).tobytes(), (k, fmt)


def test_decode_files_mixed_corpus(engine):
    files, is_flac, truth = tfo.mixed_corpus()
    rest = [i for i in range(len(files)) if not is_flac[i]]
    for fmt in (nat.FMT_S16, nat.FMT_F32, nat.FMT_S32):
        got = decode.decode_files(engine, files, fmt, threads=4)
        base = decode.decode_files(engine, [files[i] for i in rest], fmt, threads=4)
        for i, data in enumerate(files):
            if data == tfo.BROKEN_FLAC:
                assert got[i][0].shape[0] == 0
            elif is_flac[i]:
                alone, rate = decode.decode_flac(engine, data, fmt)
                assert got[i][1] == rate and got[i][0].shape == alone.shape and got[i][0].tobytes() == alone.tobytes(), i
                assert got[i][0].tobytes() == tfo.from_s32(truth[i], fmt).tobytes(), i
        for j, i in enumerate(rest):
            assert got[i][1] == base[j][1] and got[i][0].shape == base[j][0].shape, i
            assert got[i][0].tobytes() == base[j][0].tobytes(), i


def test_cpp_flac_decoder(tmp_path, engine):
    """registry -> GpuFlacDecoder, one decode() per frame: planar S32 = decode_flac; and its refusals."""
    exe, _ = tfo.build_driver(tmp_path)
    corpus = tfo.flac_corpus()
    for k in (0, 3, 4, 7):                                       # stereo, 6 and 8 channels, the file with a frame that fails its CRC
        data = corpus[k][0]
        want, _ = decode.decode_flac(engine, data)
        inp, outp = tmp_path / f"in{k}.flac", tmp_path / f"out{k}.bin"
        inp.write_bytes(data)
        res = subprocess.run([exe, "file", str(inp), str(outp)], capture_output=True, text=True, timeout=300)
        assert res.returncode == 0, res.stdout + res.stderr
        got = np.frombuffer(outp.read_bytes(), dtype=np.int32)
        assert got.size == want.size and (got.reshape(want.shape) == want).all(), k
    res = subprocess.run([exe, "errors", str(tmp_path / "in0.flac")], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0 and "flac errors: ok" in res.stdout, res.stdout + res.stderr
