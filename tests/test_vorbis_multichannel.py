"""Ogg Vorbis with 3 to 8 channels and any coupling list, CPU half: the multichannel entropy front-end (`symgpu_vorbis_fe_*_mc`)
against the front-end oracle and the stream writer's ground truth, what `symgpu_vorbis_fe_create` / `_create_mc` refuse, the jobs
form against the serial one, the reference's channel order, and Ogg file bytes -> plan -> synthesis / output oracles for single
files and mixed batches (`decode.plan_files`).  The sanitizer run drives the multichannel entry points with mutated streams."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import symphonia_b200 as sb  # noqa: F401  (builds / loads the library)
from oracle import packetizer_oracle as po
from symphonia_b200 import _native as nat
from symphonia_b200 import decode, frontend
from symphonia_b200.engine import SymgpuError
from tests import _oracle
from tests import _streams as st
from tests import _vorbis_mc_bitstream as vb
from tests import _vorbis_mc_oracle as vo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# map_vorbis_channel (symphonia-codec-vorbis/src/lib.rs:771-788, Vorbis I 4.3.9): output plane of Vorbis channel i, restated here
REFERENCE_CHANNEL_MAP = {1: [0], 2: [0, 1], 3: [0, 2, 1], 4: [0, 1, 2, 3], 5: [0, 2, 1, 3, 4], 6: [0, 2, 1, 4, 5, 3],
                         7: [0, 2, 1, 5, 6, 4, 3], 8: [0, 2, 1, 6, 7, 4, 5, 3]}


@pytest.fixture(scope="module")
def oracle():
    return _oracle.load()


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _couplings(rng, C, chained=True):
    """1 to 4 steps over C channels; with `chained` one channel takes part in two steps."""
    steps = []
    for _ in range(int(rng.integers(1, 5))):
        m, a = (int(x) for x in rng.choice(C, size=2, replace=False))
        steps.append((m, a))
    if chained:
        m = steps[0][0]
        a = int(rng.choice([c for c in range(C) if c != m]))
        steps.append((a, m))
    return steps


def _stream(seed, C, **kw):
    rng = np.random.default_rng(seed)
    kw.setdefault("couplings", _couplings(rng, C, chained=bool(seed % 2)))
    kw.setdefault("max_submaps", 1 + seed % 4)
    return vb.Stream(rng, channels=C, **kw)


def _same(a, b, what, C):
    assert bool(a["block_flag"]) == bool(b["block_flag"]) and bool(a["prev_block_flag"]) == bool(b["prev_block_flag"]), what
    assert [bool(x) for x in a["do_not_decode"][:C]] == [bool(x) for x in b["do_not_decode"][:C]], what
    assert list(a["floor"][:C]) == list(b["floor"][:C]), what
    assert np.array_equal(a["floor_y"][:C], b["floor_y"][:C]), what
    assert np.array_equal(bits(a["residue"][:C]), bits(b["residue"][:C])), what


def _as_dict(unit, floor_y, residue):
    fl = [None if int(v) == 0xFFFF else int(v) for v in unit["floor"]]
    return dict(block_flag=int(unit["block_flag"]), prev_block_flag=int(unit["prev_block_flag"]),
                do_not_decode=[int(v) for v in unit["do_not_decode"]], floor=fl, floor_y=floor_y, residue=residue)


# ---- oracle = writer truth, front-end = oracle -----------------------------------------------------------------------------

@pytest.mark.parametrize("residue_type", [0, 1, 2])
def test_oracle_equals_writer_truth(residue_type):
    seen_long, seen_short, seen_unused = set(), set(), 0
    for C in range(3, 9):
        for seed in range(4):
            s = _stream(100 * C + 10 * residue_type + seed, C, residue_type=residue_type, per_word=1)
            o = vo.VorbisFrontend(s.ident, s.setup)
            slot = (1 << s.bs_exp[1]) >> 1
            for k in range(8):
                pkt, truth = s.packet(unused_prob=0.3)
                got = o.decode(pkt, slot)
                _same(got, truth, (C, residue_type, seed, k), C)
                (seen_long if truth["block_flag"] else seen_short).add(C)
                seen_unused += sum(1 for f in truth["floor"][:C] if f is None)
    assert seen_long == seen_short == set(range(3, 9)) and seen_unused > 50


def test_frontend_equals_oracle_and_writer_truth():
    n_cut = n_flip = n_sub = 0
    for C in range(3, 9):
        for seed in range(6):
            rtype = seed % 3
            s = _stream(7000 + 10 * C + seed, C, residue_type=rtype, per_word=1 if seed < 3 else None)
            n_sub += max(len(m["submaps"]) for m in s.mappings) > 1
            fe, o = frontend.VorbisFrontend(s.ident, s.setup, mc=True), vo.VorbisFrontend(s.ident, s.setup)
            fe8 = frontend.VorbisFrontend(s.ident, s.setup, mc=True)
            assert fe.channels == C and int(fe.stream["n_couplings"]) == len(s.couplings)
            assert [(int(m), int(a)) for m, a in zip(fe.stream["magnitude_ch"], fe.stream["angle_ch"])][:len(s.couplings)] == s.couplings
            rng = np.random.default_rng(seed)
            for k in range(9):
                pkt, truth = s.packet(unused_prob=0.25)
                mode = k % 3
                if mode == 1 and len(pkt) > 1:
                    pkt, n_cut = pkt[:int(rng.integers(0, len(pkt)))], n_cut + 1
                elif mode == 2:
                    b = bytearray(pkt)
                    for _ in range(int(rng.integers(1, 4))):
                        b[int(rng.integers(len(b)))] ^= 1 << int(rng.integers(8))
                    pkt, n_flip = bytes(b), n_flip + 1
                what = (C, seed, k, mode)
                try:
                    want = o.decode(pkt, fe.slot)
                except po.ReaderError:
                    for f, planes in ((fe, None), (fe8, 8)):
                        with pytest.raises(SymgpuError) as e:
                            f.decode(pkt, planes=planes)
                        assert e.value.status == 1, what
                    continue
                got = _as_dict(*fe.decode(pkt))
                _same(got, want, what, C)
                if mode == 0 and s.per_word == 1:
                    _same(got, truth, what + ("truth",), C)
                u8, fy8, r8 = fe8.decode(pkt, planes=8)      # more planes than channels: the extra ones are empty
                _same(_as_dict(u8, fy8, r8), want, what + (8,), C)
                assert not fy8[C:].any() and not r8[C:].any() and all(u8["do_not_decode"][C:]) and (u8["floor"][C:] == 0xFFFF).all()
            fe.close(), fe8.close()
    assert n_cut > 40 and n_flip > 40 and n_sub > 10


def test_create_refusals():
    # every multichannel writer stream: the two-plane create still refuses it (as at the parent commit), create_mc takes it
    for C in range(3, 9):
        s = _stream(300 + C, C)
        with pytest.raises(SymgpuError) as e:
            frontend.VorbisFrontend(s.ident, s.setup)
        assert e.value.status == 2
        frontend.VorbisFrontend(s.ident, s.setup, mc=True).close()
    # stereo streams the two-plane create refuses: a step (1, 0), two steps -- create_mc takes them at C = 2
    for steps in ([(1, 0)], [(0, 1), (1, 0)]):
        s = vb.Stream(np.random.default_rng(11), channels=2, couplings=steps)
        with pytest.raises(SymgpuError) as e:
            frontend.VorbisFrontend(s.ident, s.setup)
        assert e.value.status == 2
        fe = frontend.VorbisFrontend(s.ident, s.setup, mc=True)
        assert fe.channels == 2 and int(fe.stream["n_couplings"]) == len(steps)
        fe.close()
    # 0 channels: DECODE (the identification reader); 9 channels: UNSUPPORTED
    s = _stream(20, 3)
    zero = bytearray(s.ident)
    zero[11] = 0
    for mc in (False, True):
        with pytest.raises(SymgpuError) as e:
            frontend.VorbisFrontend(bytes(zero), s.setup, mc=mc)
        assert e.value.status == 1
    s9 = vb.Stream(np.random.default_rng(21), channels=9, couplings=[(0, 8)])
    o = vo.VorbisFrontend(s9.ident, s9.setup)          # (a valid stream: only the channel map is missing)
    assert o.ident["n_channels"] == 9
    for mc in (False, True):
        with pytest.raises(SymgpuError) as e:
            frontend.VorbisFrontend(s9.ident, s9.setup, mc=mc)
        assert e.value.status == 2
    # more than SYMGPU_VORBIS_MAX_COUPLINGS steps
    many = [(k % 8, (k + 1) % 8) for k in range(17)]
    s = vb.Stream(np.random.default_rng(22), channels=8, couplings=many)
    with pytest.raises(SymgpuError) as e:
        frontend.VorbisFrontend(s.ident, s.setup, mc=True)
    assert e.value.status == 2
    frontend.VorbisFrontend(vb.Stream(np.random.default_rng(22), channels=8, couplings=many[:16]).ident,
                            vb.Stream(np.random.default_rng(22), channels=8, couplings=many[:16]).setup, mc=True).close()
    # modes whose mappings have different coupling lists (the stream record holds one list); equal step counts are not enough
    n_diff = 0
    for seed in range(40):
        s = vb.Stream(np.random.default_rng(500 + seed), channels=4, mapping_couplings=[[(0, 1)], [(2, 3)]])
        used = {mp for _, mp in s.modes}
        with pytest.raises(SymgpuError) if len(used) > 1 else _no_error():
            frontend.VorbisFrontend(s.ident, s.setup, mc=True).close()
        n_diff += len(used) > 1
    assert n_diff >= 5
    # floor type 0
    for seed in range(6):
        s = _stream(30 + seed, 6, extra_floor0=True)
        o = vo.VorbisFrontend(s.ident, s.setup)          # the reference reads it
        assert 0 in [f.get("type", 1) for f in o.setup["floors"]] or len(o.setup["floors"]) == len(s.floors) + 1
        for mc in (False, True):
            with pytest.raises(SymgpuError) as e:
                frontend.VorbisFrontend(s.ident, s.setup, mc=mc)
            assert e.value.status == 2


class _no_error:
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


def test_two_plane_entry_points_refuse_a_multichannel_front_end():
    s = _stream(40, 5)
    fe = frontend.VorbisFrontend(s.ident, s.setup, mc=True)
    pkt, _ = s.packet()
    L = nat.lib()
    unit = np.zeros(1, dtype=nat.VORBIS_UNIT_DTYPE)
    fy, res = np.zeros((2, 65), np.uint16), np.zeros((2, fe.slot), np.float32)
    a = np.frombuffer(pkt, np.uint8)
    vp = ctypes.c_void_p
    assert L.symgpu_vorbis_fe_decode(fe._h, vp(a.ctypes.data), a.size, fe.slot, 0, vp(unit.ctypes.data), vp(fy.ctypes.data), vp(res.ctypes.data)) == 6
    # fewer planes than channels
    with pytest.raises(SymgpuError) as e:
        fe.decode(pkt, planes=4)
    assert e.value.status == 6
    fe.close()


# ---- jobs = serial ----------------------------------------------------------------------------------------------------------

def _long_stream(seed, C, rtype):
    """(writer, 64 packets -- some cut, damaged or not audio -- and whether the oracle's partition-class vector grew after packet 0)."""
    s = _stream(seed, C, residue_type=rtype, bs_exp=(7, 10))
    o = vo.VorbisFrontend(s.ident, s.setup)
    rng = np.random.default_rng(seed)
    pk, sizes = [], []
    for j in range(64):
        p, _ = s.packet()
        if j % 9 == 4 and len(p) > 2:
            p = p[:int(rng.integers(1, len(p)))]
        elif j % 9 == 7:
            b = bytearray(p)
            b[int(rng.integers(len(b)))] ^= 1 << int(rng.integers(8))
            p = bytes(b)
        elif j == 20:
            p = b"\x01" + p
        pk.append(p)
        try:
            o.decode(p, (1 << s.bs_exp[1]) >> 1)
        except po.ReaderError:
            pass
        sizes.append(len(o.part_classes))
    return s, pk, len(set(sizes)) > 1


def test_jobs_equal_the_serial_front_end_on_long_streams():
    """Streams whose partition-class vector grows across packets (short -> long blocks, sub-maps of different channel counts, type-2
    residues over 3+ channels): the jobs form must still equal the serial front-end byte for byte, refused packets included."""
    for k, C in enumerate((3, 4, 5, 6, 7, 8)):
        seed = 9000 + 100 * k
        while True:
            s, pk, grew = _long_stream(seed, C, k % 3)
            seed += 1
            if grew:
                break
        blob = b"".join(pk)
        table = np.zeros(len(pk), dtype=nat.PIECE_DTYPE)
        table["len"] = [len(p) for p in pk]
        table["offset"] = np.concatenate([[0], np.cumsum(table["len"][:-1], dtype=np.uint64)])
        fe = frontend.VorbisFrontend(s.ident, s.setup, mc=True)
        for planes in (C, 8):
            units, fy, res, keep = fe.decode_packets(blob, table, planes=planes)
            fe.reset()
            for threads in (1, 3, 8):
                ju, jf, jr, acc = frontend.vorbis_decode_packets_jobs(s.ident, s.setup, blob, table, fe.slot, threads=threads, mc=True, planes=planes)
                assert acc.tolist() == keep.tolist(), (C, threads)
                assert ju[acc].tobytes() == units.tobytes() and jf[acc].tobytes() == fy.tobytes(), (C, threads)
                assert jr[acc].tobytes() == res.tobytes(), (C, threads)
                gone = np.setdiff1d(np.arange(len(pk)), acc)
                assert len(gone) >= 1 and not ju[gone].tobytes().strip(b"\0")
        fe.close()


# ---- channel map --------------------------------------------------------------------------------------------------------------

def test_channel_map_is_the_reference_table():
    for C in range(1, 9):
        assert frontend.vorbis_channel_map(C).tolist() == REFERENCE_CHANNEL_MAP[C]
    for C in (0, 9):
        with pytest.raises(SymgpuError):
            frontend.vorbis_channel_map(C)


# ---- Ogg file bytes -> plan -> oracles ------------------------------------------------------------------------------------------

def mc_file(seed, C, n_packets=20, pad=37, couplings=None, bs_exp=(8, 11)):
    """(ogg bytes, stream writer, truth per packet, end granule) of a C-channel Vorbis file."""
    rng = np.random.default_rng(seed)
    couplings = _couplings(rng, C) if couplings is None else couplings
    s = vb.Stream(rng, channels=C, bs_exp=bs_exp, per_word=1, couplings=couplings, max_submaps=3)
    pk, truth = [], []
    for _ in range(n_packets):
        b, t = s.packet()
        pk.append(b), truth.append(t)
    bs = {False: 1 << bs_exp[0], True: 1 << bs_exp[1]}
    g, gran = 0, []
    for k, t in enumerate(truth):
        if k:
            g += (bs[bool(t["prev_block_flag"])] + bs[bool(t["block_flag"])]) // 4
        gran.append(g)
    end = max(g - pad, gran[-2] if n_packets > 1 else 0)
    gran[-1] = end
    headers = [s.ident, b"\x03vorbis" + bytes(20), s.setup]
    pages = st.ogg_paginate(78, headers[:1], rng, eos=False) + st.ogg_paginate(78, headers[1:], rng, first_sequence=1, bos=False, eos=False)
    pages += st.ogg_paginate(78, pk, rng, max_segments=255, first_sequence=len(pages), bos=False, granule_of=gran)
    return b"".join(pages), s, truth, end


def _reference_order(pcm, C):
    """Planes in Vorbis order -> planes in the reference's order, by the restated table."""
    out = np.zeros_like(pcm[:, :C])
    for i, plane in enumerate(REFERENCE_CHANNEL_MAP[C]):
        out[:, plane] = pcm[:, i]
    return out


def render_mc(oracle, plan, fmt):
    """A multichannel plan through oracle_vorbis_mc_batch and the conversion oracle, planes put in the reference's order first."""
    C, P = plan["channels"], plan["planes"]
    wl = dict(streams=plan["stream"], floors=plan["floors"], units=plan["units"], floor_y=plan["floor_y"], residue=plan["residue"],
              runs=plan["runs"], slot=plan["slot"], channels=P)
    rc, pcm = _oracle.vorbis_mc_batch(oracle, wl)
    assert rc == 0
    ordered = np.zeros_like(pcm)
    ordered[:, :C] = _reference_order(pcm, C)
    return _oracle.pcm_pack(oracle, ordered, plan["spans"], C, fmt, plan["total_frames"])


def _expect_from_truth(oracle, s, truth, end, plan):
    C, n = s.channels, len(truth)
    units = np.zeros(n, dtype=nat.VORBIS_UNIT_MC_DTYPE)
    for k, t in enumerate(truth):
        units[k]["block_flag"], units[k]["prev_block_flag"] = int(t["block_flag"]), int(t["prev_block_flag"])
        units[k]["do_not_decode"][:C] = [int(x) for x in t["do_not_decode"][:C]]
        units[k]["do_not_decode"][C:] = 1
        units[k]["floor"][:C] = [0xFFFF if f is None else f for f in t["floor"][:C]]
        units[k]["floor"][C:] = 0xFFFF
    wl = dict(streams=plan["stream"], floors=plan["floors"], units=units, floor_y=np.stack([t["floor_y"][:C] for t in truth]),
              residue=np.stack([t["residue"][:C] for t in truth]), runs=plan["runs"], slot=plan["slot"], channels=C)
    rc, pcm = _oracle.vorbis_mc_batch(oracle, wl)
    assert rc == 0
    bs = {0: 1 << s.bs_exp[0], 1: 1 << s.bs_exp[1]}
    rows = []
    for k in range(1, n):
        frames = (bs[int(units[k]["prev_block_flag"])] + bs[int(units[k]["block_flag"])]) // 4
        rows.append(_reference_order(pcm[k:k + 1, :C, :frames], C)[0].T)
    return np.concatenate(rows)[:end]


@pytest.mark.parametrize("C", [3, 6, 8])
def test_plan_up_to_the_launch(oracle, C):
    for k, pad in enumerate([37, 0, 300, 1]):
        data, s, truth, end = mc_file(600 + 10 * C + k, C, pad=pad)
        plan = decode.ogg_vorbis_plan(data)
        assert plan["mc"] and plan["planes"] == C and plan["channels"] == C and len(plan["units"]) == len(truth)
        assert plan["total_frames"] == end and plan["floor_y"].shape[1:] == (C, 65) and plan["residue"].shape[1:] == (C, plan["slot"])
        assert plan["plane_of_channel"].tolist() == np.argsort(REFERENCE_CHANNEL_MAP[C]).tolist()
        sp = plan["spans"]
        left = sp["frames"].astype(np.int64) - sp["trim_start"] - sp["trim_end"]
        assert left[0] == 0 and (left >= 0).all() and int(left.sum()) == end
        got = render_mc(oracle, plan, nat.FMT_F32)
        want = _expect_from_truth(oracle, s, truth, end, plan)
        assert got.shape == want.shape == (end, C)
        assert (got.view(np.uint32) == np.ascontiguousarray(want).view(np.uint32)).all()
        assert np.isfinite(got).all() and np.abs(got).max() > 0
        assert decode.plan_file(data)["kind"] == "vorbis_mc"


def test_long_multichannel_stream_as_jobs_gives_the_same_plan():
    data, _, _, _ = mc_file(700, 6, n_packets=48, pad=11)
    a, b = decode.ogg_vorbis_plan(data), decode.ogg_vorbis_plan(data, threads=4)
    assert len(a["units"]) == 48 and a["mc"] and b["mc"]
    for key in ("units", "floor_y", "residue", "runs", "spans", "floors", "stream", "plane_of_channel"):
        assert a[key].tobytes() == b[key].tobytes(), key


def mixed_files():
    """The many-files corpus (MP3, Layer I / II, AAC, mono / stereo Vorbis) + 3 / 6 / 8-channel Vorbis, a stereo file with a (1, 0)
    coupling step, a floor-0 file and a 9-channel file."""
    from tests import test_zz_many_files as tz
    files = tz._files()
    n_plain = len(files)
    extra = [mc_file(800, 3)[0], mc_file(801, 6, bs_exp=(7, 10))[0], mc_file(802, 8, n_packets=9)[0],
             mc_file(803, 2, couplings=[(1, 0)])[0]]
    rng = np.random.default_rng(804)
    s0 = _stream(804, 6, extra_floor0=True)
    s9 = vb.Stream(np.random.default_rng(805), channels=9, couplings=[(0, 8)])
    for ident, setup_b in ((s0.ident, s0.setup), (s9.ident, s9.setup)):
        pages = st.ogg_paginate(79, [ident], rng, eos=False) + st.ogg_paginate(79, [b"\x03vorbis" + bytes(9), setup_b], rng, first_sequence=1, bos=False)
        extra.append(b"".join(pages))
    return files, n_plain, extra


def test_mixed_batches(oracle):
    from tests import test_zz_many_files as tz
    files, n_plain, extra = mixed_files()
    base_plans, base_batches = decode.plan_files(files, threads=4)
    allf = files + extra
    plans, batches = decode.plan_files(allf, threads=4)
    assert set(batches) == {"mp3", "mpa1", "mpa2", "aac", "vorbis", "vorbis_mc"}
    assert batches["vorbis_mc"]["members"] == [n_plain, n_plain + 1, n_plain + 2, n_plain + 3]
    assert batches["vorbis_mc"]["planes"] == 8
    assert [plans[n_plain + k]["kind"] for k in (4, 5)] == ["error", "error"]
    # the stereo-compatible Vorbis batch is the one built without the multichannel files
    for key in ("units", "floor_y", "residue", "streams", "floors", "runs", "slot", "members", "first"):
        a, b = base_batches["vorbis"][key], batches["vorbis"][key]
        assert (a.tobytes() == b.tobytes()) if isinstance(a, np.ndarray) else a == b, key
    pcm = tz._render_batches(oracle, {k: v for k, v in batches.items() if k != "vorbis_mc"})
    b = batches["vorbis_mc"]
    rc, pcm["vorbis_mc"] = _oracle.vorbis_mc_batch(oracle, dict(streams=b["streams"], floors=b["floors"], units=b["units"], floor_y=b["floor_y"],
                                                                residue=b["residue"], runs=b["runs"], slot=b["slot"], channels=b["planes"]))
    assert rc == 0

    def pack(p, sp, ch, f, total):
        return _oracle.pcm_pack(oracle, p, sp, ch, f, total)

    def pack_mapped(p, sp, ch, plane_of_channel, f, total):        # the restated map, not the product's
        assert list(plane_of_channel) == np.argsort(REFERENCE_CHANNEL_MAP[ch]).tolist()
        planes = p.reshape(len(sp), -1, int(sp["plane_stride"][0]))
        ordered = planes.copy()
        ordered[:, :ch] = _reference_order(planes, ch)
        return _oracle.pcm_pack(oracle, ordered, sp, ch, f, total)

    for fmt in (nat.FMT_S16, nat.FMT_F32):
        got = decode.pack_files(plans, batches, pcm, pack, fmt, pack_mapped)
        for i, data in enumerate(allf):
            if plans[i]["kind"] == "error":
                assert got[i][0].shape == (0, 0)
                continue
            p = decode.ogg_vorbis_plan(data) if decode.sniff(data) == "vorbis" else None
            want = render_mc(oracle, p, fmt) if p is not None and p.get("mc") else tz._alone(oracle, data, fmt)
            assert got[i][0].shape == want.shape, (i, plans[i]["kind"])
            assert (got[i][0].view(np.uint8) == want.view(np.uint8)).all(), (i, plans[i]["kind"])


# ---- sanitizers -----------------------------------------------------------------------------------------------------------------

def test_multichannel_front_end_under_address_and_ub_sanitizers(tmp_path):
    exe = str(tmp_path / "fuzz_vorbis_mc")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-g", "-pthread", "-fsanitize=address,undefined", "-fno-sanitize-recover=all", "-ffp-contract=off",
                           "-I/usr/local/cuda/include", "-o", exe, os.path.join(ROOT, "tests", "cpp", "fuzz_vorbis_mc.cpp"),
                           os.path.join(ROOT, "symphonia_b200", "csrc", "vorbis_frontend.cpp"), os.path.join(ROOT, "symphonia_b200", "csrc", "packetizer.cpp"),
                           os.path.join(ROOT, "symphonia_b200", "csrc", "tables.cpp")])
    paths = []
    for k, C in enumerate((3, 4, 5, 6, 7, 8, 2)):
        s = _stream(60 + k, C, residue_type=k % 3)
        parts = [s.ident, s.setup] + [s.packet()[0] for _ in range(10)]
        path = str(tmp_path / f"vfm{C}.bin")
        with open(path, "wb") as f:
            f.write(b"".join(len(q).to_bytes(2, "little") + q for q in parts))
        paths.append(path)
    env = dict(os.environ, FUZZ_ITERS="300", ASAN_OPTIONS="detect_leaks=1:abort_on_error=1")
    res = subprocess.run([exe] + paths, capture_output=True, text=True, timeout=900, env=env)
    assert res.returncode == 0, (res.stdout + res.stderr)[-3000:]
    assert "no sanitizer report" in res.stdout and "2107 inputs" in res.stdout
