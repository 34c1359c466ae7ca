"""Ogg Vorbis with 3 to 8 channels on the device: `decode.decode_ogg_vorbis` and `decode_files` against the synthesis / output oracles
(planes put in the reference's order by the table restated in test_vorbis_multichannel.py), the mapped output stage
(`symgpu_pcm_pack_mapped_*`) against the conversion oracle, and the C++ plug-in decoder on a 5.1 file."""
import subprocess

import numpy as np
import pytest

from symphonia_b200 import _native as nat
from symphonia_b200 import decode
from tests import _oracle
from tests import test_vorbis_multichannel as tmc

FORMATS = (nat.FMT_F32, nat.FMT_S16, nat.FMT_S24, nat.FMT_S32, nat.FMT_U8)


@pytest.fixture(scope="module")
def oracle():
    return _oracle.load()


@pytest.fixture(scope="module")
def engine():
    import symphonia_b200 as sb
    with sb.Engine(0) as eng:
        yield eng


@pytest.mark.gpu
@pytest.mark.parametrize("C", [3, 6, 8])
def test_decode_ogg_vorbis_multichannel(engine, oracle, C):
    for k, pad in enumerate([37, 0, 300]):
        data, s, _, end = tmc.mc_file(600 + 10 * C + k, C, pad=pad)
        plan = decode.ogg_vorbis_plan(data)
        for fmt in (nat.FMT_S16, nat.FMT_F32):
            want = tmc.render_mc(oracle, plan, fmt)
            got, rate = decode.decode_ogg_vorbis(engine, data, fmt)
            assert rate == 44100 and got.shape == want.shape == (end, C)
            assert (got.view(np.uint8) == want.view(np.uint8)).all(), (C, k, fmt)
    # the same context goes back to two-plane streams
    from tests import test_zz_ogg_vorbis_to_pcm as tv
    data = tv._file(300)[0]
    got, _ = decode.decode_ogg_vorbis(engine, data, nat.FMT_S16)
    assert (got == tv._render(oracle, decode.ogg_vorbis_plan(data), nat.FMT_S16)).all()


@pytest.mark.gpu
def test_decode_files_mixed_corpus(engine, oracle):
    from tests import test_zz_many_files as tz
    files, _, extra = tmc.mixed_files()
    allf = files + extra
    for fmt in (nat.FMT_S16, nat.FMT_F32):
        got = decode.decode_files(engine, allf, fmt, threads=4)
        for i, data in enumerate(allf):
            if i >= len(files):
                try:
                    p = decode.ogg_vorbis_plan(data)
                except Exception:   # floor 0 / nine channels: an empty result, the others unaffected
                    assert got[i][0].shape[0] == 0
                    continue
                want = tmc.render_mc(oracle, p, fmt) if p.get("mc") else tz._alone(oracle, data, fmt)
            else:
                want = tz._alone(oracle, data, fmt)
            assert got[i][0].shape == want.shape, i
            assert (got[i][0].view(np.uint8) == want.view(np.uint8)).all(), i


def _spans(rng, n, C, stride):
    sp = np.zeros(n, dtype=nat.PCM_SPAN_DTYPE)
    sp["src"] = np.arange(n, dtype=np.uint64) * (C * stride)
    sp["plane_stride"] = stride
    sp["frames"] = rng.integers(1, stride + 1, n)
    sp["trim_start"] = rng.integers(0, 40, n)
    sp["trim_end"] = rng.integers(0, 40, n)
    left = np.maximum(sp["frames"].astype(np.int64) - sp["trim_end"], 0)                     # symgpu_pcm_span_kept
    kept = np.maximum(left - sp["trim_start"], 0)
    sp["dst_frame"] = np.concatenate([[0], np.cumsum(kept)[:-1]]).astype(np.uint64)
    return sp, int(kept.sum())


@pytest.mark.gpu
@pytest.mark.parametrize("C", range(1, 9))
def test_pack_mapped_equals_the_conversion_oracle(engine, oracle, C):
    import torch
    rng = np.random.default_rng(40 + C)
    n, stride = 37, 1028
    pcm = (rng.standard_normal((n, C, stride)) * 0.7).astype(np.float32)
    pcm.reshape(-1)[rng.integers(0, pcm.size, 64)] = np.float32(np.nan)
    pcm.reshape(-1)[rng.integers(0, pcm.size, 64)] = np.float32(3.5)
    sp, total = _spans(rng, n, C, stride)
    for trial in range(3):
        perm = rng.permutation(C).astype(np.uint8) if trial else np.arange(C, dtype=np.uint8)
        permuted = np.ascontiguousarray(pcm[:, perm])
        for fmt in FORMATS:
            want = _oracle.pcm_pack(oracle, permuted, sp, C, fmt, total)
            got = engine.pcm_pack_host_mapped(pcm, sp, C, perm, fmt, total)
            assert (got.view(np.uint8) == want.view(np.uint8)).all(), (C, trial, fmt)
            if trial == 0:
                plain = engine.pcm_pack_host(pcm, sp, C, fmt, total)
                assert plain.tobytes() == got.tobytes()
            # device variant, and uniform packets (no spans)
            out_t = torch.zeros(total * C * np.dtype(nat.FMT_NUMPY[fmt]).itemsize, dtype=torch.uint8, device="cuda")
            engine.pcm_pack_dev_mapped(torch.from_numpy(pcm).cuda(), torch.from_numpy(sp.view(np.uint8)).cuda(), n, C, perm, fmt, out_t)
            engine.sync()
            assert out_t.cpu().numpy().tobytes() == want.tobytes(), (C, trial, fmt, "dev")
            wu = _oracle.pcm_pack(oracle, permuted, None, C, fmt, n * 300, plane_stride=stride, frames=300, n_spans=n)
            gu = engine.pcm_pack_host_mapped(pcm, None, C, perm, fmt, n * 300, plane_stride=stride, frames=300, n_spans=n)
            assert gu.tobytes() == wu.tobytes(), (C, trial, fmt, "uniform")


@pytest.mark.gpu
def test_cpp_vorbis_decoder_on_a_5_1_file(tmp_path, oracle):
    """registry -> GpuVorbisDecoder (multichannel path), one decode() per packet; planes in the reference's order."""
    from tests.test_cpp_host import _build
    data, s, _, _ = tmc.mc_file(650, 6)
    plan = decode.ogg_vorbis_plan(data)
    want = tmc.render_mc(oracle, plan, nat.FMT_F32)
    inp, outp = tmp_path / "in.ogg", tmp_path / "out.bin"
    inp.write_bytes(data)
    res = subprocess.run([_build(), "file", "vorbis", str(inp), str(outp)], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stdout + res.stderr
    flat = np.frombuffer(outp.read_bytes(), dtype=np.float32)
    sp = plan["spans"]
    left = sp["frames"].astype(np.int64) - sp["trim_start"] - sp["trim_end"]
    rows, at = [], 0
    for n in left:
        rows.append(flat[at:at + n * 6].reshape(6, n).T)
        at += n * 6
    assert at == flat.size
    got = np.concatenate(rows)
    assert got.shape == want.shape and (np.ascontiguousarray(got).view(np.uint32) == np.ascontiguousarray(want).view(np.uint32)).all()
