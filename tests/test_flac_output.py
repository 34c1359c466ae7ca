"""FLAC's output stage and FLAC in `plan_files` (CPU).

`from_s32` restates FromSample<i32> (symphonia-core/src/audio/conv.rs:514-532) for the formats of symgpu_flac_decode_*, pinned to the
reference's own assertions for i32::MIN / MID / MAX.  `place` restates where that call stores a frame: out[dst[f] + i * channels + c].
On a mixed corpus (MP3, Layer I / II, AAC, stereo and 3 to 8 channel Vorbis, FLAC of every channel assignment, 1 / 2 / 6 / 8 channels,
8 to 32 bits, blocks of 64 to 4096 samples, one file with a frame that fails its CRC, a broken "fLaC" file) the 'flac' batch of
`plan_files`, restored by the oracle, placed by its dst and converted, gives every file what its own plan gives and what the encoder
started from; the other files' plans and batches are those of the corpus without the FLAC files."""
import os
import subprocess

import numpy as np

from symphonia_b200 import _native as nat
from symphonia_b200 import decode, packetizer
from tests import test_flac_frontend as tf
from tests import test_oracle_kat_flac as kat

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FORMATS = (nat.FMT_F32, nat.FMT_S16, nat.FMT_S24, nat.FMT_S32, nat.FMT_U8)
I32_MIN, I32_MAX = -(1 << 31), (1 << 31) - 1


def from_s32(x, fmt):
    """FromSample<i32> of conv.rs:514-532, element-wise over int32 `x`."""
    x = np.asarray(x, dtype=np.int32)
    if fmt == nat.FMT_S32:
        return x.copy()
    if fmt == nat.FMT_S24:
        return x >> 8                                                   # i24::from(s >> 8), 4-byte container
    if fmt == nat.FMT_S16:
        return (x >> 16).astype(np.int16)
    if fmt == nat.FMT_U8:
        return ((x.view(np.uint32) + np.uint32(0x8000_0000)) >> np.uint32(24)).astype(np.uint8)
    if fmt == nat.FMT_F32:
        return (x.astype(np.float64) / 2147483648.0).astype(np.float32)
    raise ValueError(fmt)


def place(frames, subs, restored, dst, out_samples):
    """The store of symgpu_flac_decode_*: frame f's sample i of channel c at out[dst[f] + i * channels + c] (int32; zero elsewhere)."""
    out = np.zeros(out_samples, dtype=np.int32)
    for f, fr in enumerate(frames):
        ch, first = int(fr["channels"]), int(fr["first_subframe"])
        n = int(subs[first]["n"])
        region = out[int(dst[f]):int(dst[f]) + n * ch].reshape(n, ch)
        for c in range(ch):
            off = int(subs[first + c]["offset"])
            region[:, c] = restored[off:off + n]
    return out


def test_from_sample_rules_pinned_to_the_reference():
    mn, mid, mx = np.array([I32_MIN]), np.array([0]), np.array([I32_MAX])
    # verify_u8 / i16 / i24 / i32 / f32_from_sample (conv.rs tests): i32::MAX / MID / MIN
    assert [int(from_s32(v, nat.FMT_U8)[0]) for v in (mx, mid, mn)] == [255, 128, 0]
    assert [int(from_s32(v, nat.FMT_S16)[0]) for v in (mx, mid, mn)] == [32767, 0, -32768]
    assert [int(from_s32(v, nat.FMT_S24)[0]) for v in (mx, mid, mn)] == [8388607, 0, -8388608]
    assert [int(from_s32(v, nat.FMT_S32)[0]) for v in (mx, mid, mn)] == [I32_MAX, 0, I32_MIN]
    assert from_s32(mx, nat.FMT_F32)[0] == np.float32(2147483647.0) / np.float32(2147483648.0)
    assert from_s32(mid, nat.FMT_F32)[0] == 0.0 and from_s32(mn, nat.FMT_F32)[0] == -1.0
    # hand cases: arithmetic shifts, the wrapping offset of the unsigned format, exact scaling of f32
    assert int(from_s32(np.array([-1]), nat.FMT_S16)[0]) == -1 and int(from_s32(np.array([-1]), nat.FMT_S24)[0]) == -1
    assert int(from_s32(np.array([-1]), nat.FMT_U8)[0]) == 127 and int(from_s32(np.array([1 << 24]), nat.FMT_U8)[0]) == 129
    assert int(from_s32(np.array([65535]), nat.FMT_S16)[0]) == 0 and int(from_s32(np.array([-65536]), nat.FMT_S16)[0]) == -1
    x = np.random.default_rng(5).integers(I32_MIN, I32_MAX, 4096, endpoint=True).astype(np.int32)
    f = from_s32(x, nat.FMT_F32)
    assert (f == (x.astype(np.float32) * np.float32(2.0 ** -31))).all()   # a power-of-two scale commutes with the rounding
    # 16-bit PCM scaled to 32 bits by the decoder comes back as itself
    s16 = np.arange(-32768, 32768, dtype=np.int32)
    assert (from_s32(s16 << 16, nat.FMT_S16) == s16).all()


# ---- FLAC in plan_files ---------------------------------------------------------------------------------------------------------

FLAC_SPECS = ((16, 2, 1152), (24, 2, 4096), (8, 1, 64), (12, 6, 576), (20, 8, 256), (32, 1, 512), (16, 2, 333))


def flac_corpus():
    """[(bytes, truth [frames, channels] int32 scaled to 32 bits)]: the FLAC_SPECS files, then a copy of the first whose fourth frame
    fails its CRC-16 (the splitter drops it, and so its samples)."""
    out = []
    for k, (bps, channels, block) in enumerate(FLAC_SPECS):
        out.append(tf._flac_file(900 + k, bps, channels, block))
    data, want = out[0]
    _, packets = packetizer.flac_index(data)
    hurt = bytearray(data)
    victim = packets[3]
    hurt[int(victim["offset"]) + int(victim["size"]) // 2] ^= 0x10
    keep = np.ones(len(want), dtype=bool)
    keep[int(victim["ts"]):int(victim["ts"]) + int(victim["dur"])] = False
    out.append((bytes(hurt), want[keep]))
    return out


BROKEN_FLAC = b"fLaC" + bytes(200)


def mixed_corpus():
    """(files, is_flac, truth per FLAC file index): the multichannel Vorbis test's mixed corpus with the FLAC files and the broken
    "fLaC" file spread through it."""
    from tests import test_vorbis_multichannel as tmc
    files, _, extra = tmc.mixed_files()
    others = files + extra
    flacs = flac_corpus()
    every = len(others) // (len(flacs) + 1)
    merged, truth = [], {}
    for k, data in enumerate(others):
        merged.append(data)
        if k % every == every - 1 and flacs:
            data_f, want = flacs.pop(0)
            truth[len(merged)] = want
            merged.append(data_f)
    for data_f, want in flacs:
        truth[len(merged)] = want
        merged.append(data_f)
    merged.insert(3, BROKEN_FLAC)
    truth = {(i + 1 if i >= 3 else i): w for i, w in truth.items()}
    is_flac = [decode.sniff(f) == "flac" for f in merged]
    return merged, is_flac, truth


def _same(a, b):
    if isinstance(a, dict):
        return a.keys() == b.keys() and all(_same(a[k], b[k]) for k in a)
    if isinstance(a, (list, tuple)):
        return len(a) == len(b) and all(_same(x, y) for x, y in zip(a, b))
    if isinstance(a, np.ndarray):
        return isinstance(b, np.ndarray) and a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()
    return a == b


def test_plan_files_with_flac(oracle):
    files, is_flac, truth = mixed_corpus()
    plans, batches = decode.plan_files(files, threads=4)
    broken = files.index(BROKEN_FLAC)
    assert plans[broken]["kind"] == "error" and plans[broken]["error"]
    flac = [i for i in range(len(files)) if is_flac[i] and i != broken]
    assert sorted(truth) == flac and all(plans[i]["kind"] == "flac" for i in flac)
    b = batches["flac"]
    assert b["members"] == flac
    # the corpus covers what the batch must handle
    assert {plans[i]["channels"] for i in flac} == {1, 2, 6, 8} and {plans[i]["bits_per_sample"] for i in flac} == {8, 12, 16, 20, 24, 32}
    assert set(b["frames"]["assignment"].tolist()) == {0, 1, 2, 3}
    blocks = b["subframes"]["n"]
    assert blocks.min() <= 64 and blocks.max() == 4096
    # restored by the oracle, placed by dst, converted: every file's region = its own plan through the same steps = the encoder's truth
    rc, restored = kat._restore(oracle, b["frames"], b["subframes"], b["samples"].copy())
    assert rc == 0
    placed = place(b["frames"], b["subframes"], restored, b["dst"], b["out_samples"])
    assert b["out_samples"] == sum(plans[i]["total_frames"] * plans[i]["channels"] for i in flac)
    for k, i in enumerate(flac):
        p = plans[i]
        n, ch = p["total_frames"], p["channels"]
        region = placed[b["out_first"][k]:b["out_first"][k] + n * ch].reshape(n, ch)
        alone = decode.flac_plan(files[i])
        rc, r = kat._restore(oracle, alone["frames"], alone["subframes"], alone["samples"].copy())
        assert rc == 0
        own = place(alone["frames"], alone["subframes"], r, decode.flac_dst(alone), n * ch).reshape(n, ch)
        assert (own == decode.flac_interleave(alone, r)).all()
        assert region.shape == truth[i].shape and (region == own).all() and (region == truth[i]).all(), i
        for fmt in FORMATS:
            assert from_s32(region, fmt).tobytes() == from_s32(truth[i], fmt).tobytes()
    # every other file: the plans and batches of the corpus without the FLAC files
    rest = [i for i in range(len(files)) if not is_flac[i]]
    base_plans, base_batches = decode.plan_files([files[i] for i in rest], threads=4)
    for j, i in enumerate(rest):
        assert _same(base_plans[j], plans[i]), i
    assert set(batches) == set(base_batches) | {"flac"}
    for kind, bb in base_batches.items():
        assert [rest[m] for m in bb["members"]] == batches[kind]["members"], kind
        for key in bb:
            if key != "members":
                assert _same(bb[key], batches[kind][key]), (kind, key)
    # pack_files leaves FLAC alone and packs the others as before
    pcm = {kind: np.zeros((1 << 16, 1), dtype=np.float32) for kind in batches if kind != "flac"}   # (only the slicing is compared)

    def pack(sl, sp, ch, fmt, total, *_):
        return (sl.size, sp.tobytes(), ch, fmt, total)
    got = decode.pack_files(plans, batches, pcm, pack, nat.FMT_S16, lambda sl, sp, ch, m, fmt, total: pack(sl, sp, ch, fmt, total, m))
    base = decode.pack_files(base_plans, base_batches, pcm, pack, nat.FMT_S16,
                             lambda sl, sp, ch, m, fmt, total: pack(sl, sp, ch, fmt, total, m))
    for i in flac:
        assert got[i] is None
    for j, i in enumerate(rest):
        assert _same(got[i], base[j]), i


def build_driver(out_dir):
    """tests/cpp/flac_decoder_host.cpp against the in-tree library, with -Wall: the warnings (there must be none) and the binary."""
    exe = os.path.join(str(out_dir), "flac_decoder_host")
    lib = os.path.join(ROOT, "symphonia_b200")
    res = subprocess.run(["g++", "-std=c++17", "-O2", "-Wall", "-pthread", "-o", exe, os.path.join(ROOT, "tests", "cpp", "flac_decoder_host.cpp"),
                          "-L" + lib, "-lsymgpu", "-Wl,-rpath," + lib], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    return exe, res.stderr


def test_cpp_flac_driver_compiles_without_warnings(tmp_path):
    _, warnings = build_driver(tmp_path)
    assert "warning" not in warnings, warnings
