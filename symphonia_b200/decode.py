"""File bytes in, gapless interleaved samples out: the public call for MPEG audio files (what a user of the reference does with
`MpaReader` + `MpaDecoder` + `copy_to_slice_interleaved`).  Packetiser and entropy front-end on the CPU (SURVEY §8f N2 / N1),
synthesis and the output stage (N3) on the GPU.  Every device entry point used here is part of the round-1 GPU parity suite."""
import numpy as np

from . import _native as nat
from . import frontend, packetizer
from .engine import SymgpuError


def mpeg_audio_plan(data):
    """CPU half: (kind, payload, runs, spans, sample_rate, channels, total_frames).  kind 3: payload = (units, quant); kind 1 / 2:
    payload = sub-band samples.  spans carry the packetiser's trims (encoder delay / padding from a LAME tag, or the end trim of
    an extrapolated length) and where every packet's surviving frames go in the output."""
    track, packets = packetizer.mpa_index(data)
    layer = int(track["layer"])
    if layer == 3:
        units, quant, frame_of, info = frontend.Mp3Frontend().decode_packets(data, packets)
        payload = (units.reshape(-1), quant)
        n, per = len(units), 1152 if int(info["granules"]) == 2 else 576
        runs = np.zeros(1, dtype=nat.MP3_RUN_DTYPE)
        runs[0] = (0, 0, n, int(info["granules"]), int(info["channels"]), 0)
    else:
        sub, frame_of, info = frontend.mpa12_decode_packets(data, packets, layer)
        payload = sub
        n, per = len(sub), 32 * sub.shape[-1]
        runs = np.zeros(1, dtype=nat.MPA12_RUN_DTYPE)
        runs[0] = (0, 0, n, int(info["channels"]), (0, 0, 0))
    kept = packets[frame_of]
    spans = np.zeros(n, dtype=nat.PCM_SPAN_DTYPE)
    spans["src"] = np.arange(n, dtype=np.uint64) * 2304          # every frame slot holds 2 planes of 1152 floats
    spans["plane_stride"], spans["frames"] = 1152, per
    spans["trim_start"] = np.minimum(kept["trim_start"], per)
    spans["trim_end"] = np.minimum(kept["trim_end"], per - spans["trim_start"])
    left = per - spans["trim_start"].astype(np.int64) - spans["trim_end"].astype(np.int64)
    spans["dst_frame"] = np.concatenate([[0], np.cumsum(left)[:-1]]).astype(np.uint64) if n else 0
    return layer, payload, runs, spans, int(info["sample_rate"]) if n else int(track["sample_rate"]), int(info["channels"]) if n else int(track["channels"]), int(left.sum())


def decode_mpeg_audio(engine, data, fmt=nat.FMT_S16, stream=0):
    """(samples [frames, channels] of `fmt`, sample_rate).  Layers I-III; one stream slot of `engine` is used and reset first."""
    layer, payload, runs, spans, rate, channels, total = mpeg_audio_plan(data)
    runs["stream"] = stream
    if len(spans) == 0:
        return np.zeros((0, channels), dtype=nat.FMT_NUMPY[fmt]), rate
    engine.mp3_stream_reset(stream)
    pcm = engine.mp3_synth_host_quantized(payload[0], payload[1], runs) if layer == 3 else engine.mpa12_synth_host(payload, runs)
    return engine.pcm_pack_host(pcm, spans, channels, fmt, total), rate


def ogg_vorbis_index(data, serial=None):
    """Everything about a Vorbis-in-Ogg file short of decoding its audio packets: pages -> packets (symgpu_ogg_index), the logical
    stream gathered back to back, identification / setup headers, the front-end object (codebooks, floors, ...), per audio packet its
    place, duration, leading discard (mappings/vorbis.rs:45-107) and end trim against the page granule positions
    (symphonia-format-ogg/src/logical.rs:164-302)."""
    packets, pieces = packetizer.ogg_index(data)
    if len(packets) == 0:
        raise ValueError("no Ogg packets")
    serial = int(packets["serial"][0]) if serial is None else serial
    mine = packets[packets["serial"] == serial]
    blob, table = packetizer.ogg_gather(data, mine, pieces)       # the logical stream, packets back to back
    off, ln = table["offset"].astype(np.int64), table["len"].astype(np.int64)
    padded = np.concatenate([blob, np.zeros(8, dtype=np.uint8)])
    b0, b1 = padded[off], padded[off + 1]                           # (bytes beyond a short packet are masked by `ln` below)
    ident_b = blob[off[0]:off[0] + ln[0]].tobytes()
    ident = packetizer.vorbis_ident(ident_b)
    is_setup = (ln >= 7) & (b0 == 5)
    for k, c in enumerate(b"vorbis"):
        is_setup &= padded[off + 1 + k] == c
    is_setup[0] = False
    if not is_setup.any():
        raise ValueError("no Vorbis setup header")
    at = int(np.argmax(is_setup))
    setup_b = blob[off[at]:off[at] + ln[at]].tobytes()
    n_modes, mask = packetizer.vorbis_setup_modes(setup_b, ident)
    audio = np.nonzero((np.arange(len(mine)) > at) & (ln > 0) & ((b0 & 1) == 0))[0]
    heads = b0[audio].astype(np.uint16) | (np.where(ln[audio] > 1, b1[audio], 0).astype(np.uint16) << 8)
    dur, discard, _ = packetizer.vorbis_packet_durations(ident, n_modes, mask, None, heads=heads, lens=np.minimum(ln[audio], 2))
    dur, discard = dur.astype(np.int64), discard.astype(np.int64)
    trim_end = packetizer.ogg_page_end_trims(mine["page_sequence"][audio], mine["page_absgp"][audio], dur, discard).astype(np.int64)
    fe = open_vorbis_frontend(ident_b, setup_b)
    return dict(blob=blob, table=table[audio], ident=ident, fe=fe, discard=discard, trim_end=trim_end, headers=(ident_b, setup_b))


def open_vorbis_frontend(ident_packet, setup_packet):
    """The stream's entropy front-end: the two-plane one (symgpu_vorbis_fe_create) for the streams it takes -- at most two channels,
    every mapping uncoupled or coupled by the one step (0, 1) -- else the multichannel one (up to 8 channels, any coupling list)."""
    try:
        return frontend.VorbisFrontend(ident_packet, setup_packet)
    except SymgpuError as e:
        if e.status != 2:   # (SYMGPU_ERR_UNSUPPORTED: what the two-plane record cannot hold)
            raise
    return frontend.VorbisFrontend(ident_packet, setup_packet, mc=True)


def vorbis_pack_map(channels):
    """plane_of_channel for symgpu_pcm_pack_mapped_*: output channel c (the reference's order) reads Vorbis channel plane k where
    map_vorbis_channel(channels, k) = c."""
    return np.argsort(frontend.vorbis_channel_map(channels)).astype(np.uint8)


def ogg_vorbis_plan(data, serial=None, index=None, out=None, slot=None, floor_base=0, threads=1, planes=None):
    """CPU half for a Vorbis-in-Ogg file: ogg_vorbis_index, then the entropy front-end (symgpu_vorbis_fe_*) over the audio packets
    -> the synthesis stage's batch and the output spans with the reader's trims.  Returns dict(stream, floors, units, floor_y, residue,
    runs, slot, spans, channels, sample_rate, total_frames, mc).  Packets the front-end refuses are dropped, as a caller of the reference
    drops a DecodeError.  index / out / slot / floor_base: for `plan_files` (decode into slices of a batch whose residue rows are
    `slot` long and whose floor tables start at `floor_base`).
    A stream the two-plane front-end does not take (more than two channels, other couplings) gives a multichannel plan (mc=True): stream
    is a VORBIS_STREAM_MC_DTYPE record, units VORBIS_UNIT_MC_DTYPE, floor_y / residue carry `planes` planes (default: the stream's
    channels), and plane_of_channel is the channel map of the output stage (symgpu_pcm_pack_mapped_*: the reference's plane order)."""
    ix = ogg_vorbis_index(data, serial) if index is None else index
    fe, ident, discard, trim_end = ix["fe"], ix["ident"], ix["discard"], ix["trim_end"]
    slot = fe.slot if slot is None else slot
    P = 2 if not fe.mc else (fe.channels if planes is None else int(planes))
    if threads > 1 and out is None and len(ix["table"]) >= 32:   # one long stream: its packets as independent jobs (identical output, DESIGN 10.9)
        ju, jf, jr, keep = frontend.vorbis_decode_packets_jobs(ix["headers"][0], ix["headers"][1], ix["blob"], ix["table"], slot, floor_base, threads,
                                                                mc=fe.mc, planes=P)
        units, fy, res = ju[keep], jf[keep], jr[keep]
    else:
        units, fy, res, keep = fe.decode_packets(ix["blob"], ix["table"], slot=slot, floor_base=floor_base, out=out, planes=P if fe.mc else None)
    n = len(units)
    mc = fe.mc
    stream, floors = np.array([fe.stream], dtype=nat.VORBIS_STREAM_MC_DTYPE if mc else nat.VORBIS_STREAM_DTYPE), fe.floors.copy()
    fe.close()
    bs0, bs1 = 1 << int(ident["bs0_exp"]), 1 << int(ident["bs1_exp"])
    frames = (np.where(units["prev_block_flag"] != 0, bs1, bs0) + np.where(units["block_flag"] != 0, bs1, bs0)).astype(np.int64) // 4
    ts = np.minimum(discard[keep], frames)
    te = np.minimum(trim_end[keep], frames - ts)
    if n:
        ts[0], te[0] = frames[0], 0   # the first packet after a reset is silenced in gapless mode (codec-vorbis lib.rs:318-322)
    left = frames - ts - te
    spans = np.zeros(n, dtype=nat.PCM_SPAN_DTYPE)
    spans["src"] = np.arange(n, dtype=np.uint64) * (P * slot)
    spans["plane_stride"], spans["frames"], spans["trim_start"], spans["trim_end"] = slot, frames, ts, te
    spans["dst_frame"] = np.concatenate([[0], np.cumsum(left)[:-1]]).astype(np.uint64) if n else 0
    total = int(left.sum())
    runs = np.zeros(1, dtype=nat.VORBIS_RUN_DTYPE)
    runs["n_packets"] = n
    plan = dict(stream=stream, floors=floors, units=units, floor_y=fy, residue=res, runs=runs, slot=slot, spans=spans,
                channels=int(ident["channels"]), sample_rate=int(ident["sample_rate"]), total_frames=total)
    if mc:
        plan.update(mc=True, planes=P, plane_of_channel=vorbis_pack_map(int(ident["channels"])))
    return plan


def decode_ogg_vorbis(engine, data, fmt=nat.FMT_S16, serial=None, threads=1):
    """(samples [frames, channels] of `fmt`, sample_rate) of one Vorbis logical stream (1 to 8 channels, floor 1), channels in the
    reference's order.  Registers the stream as slot 0 of `engine` with its floors from index 0."""
    plan = ogg_vorbis_plan(data, serial, threads=threads)
    if len(plan["units"]) == 0:
        return np.zeros((0, plan["channels"]), dtype=nat.FMT_NUMPY[fmt]), plan["sample_rate"]
    if plan.get("mc"):
        engine.vorbis_mc_streams_set(plan["stream"])
        engine.vorbis_floors_set(plan["floors"])
        pcm = engine.vorbis_mc_synth_host(plan["units"], plan["floor_y"], plan["residue"], plan["runs"], plan["planes"], plan["slot"])
        return (engine.pcm_pack_host_mapped(pcm, plan["spans"], plan["channels"], plan["plane_of_channel"], fmt, plan["total_frames"]),
                plan["sample_rate"])
    engine.vorbis_streams_set(plan["stream"])
    engine.vorbis_floors_set(plan["floors"])
    pcm = engine.vorbis_synth_host(plan["units"], plan["floor_y"], plan["residue"], plan["runs"], plan["slot"])
    return engine.pcm_pack_host(pcm, plan["spans"], plan["channels"], fmt, plan["total_frames"]), plan["sample_rate"]


def adts_aac_index(data):
    """(packets, sample_rate, channels): the ADTS frame index and the stream's parameters (the first frame's, AdtsReader::try_new)."""
    packets, _ = packetizer.adts_index(data)
    if len(packets) == 0:
        raise ValueError("no ADTS frames")
    rate, channels = int(packets[0]["sample_rate"]), int(packets[0]["channels"])
    if channels not in (1, 2):
        raise ValueError("channel configuration outside AAC-LC mono / stereo")
    return packets, rate, channels


def adts_aac_plan(data, index=None, out=None, threads=1):
    """CPU half for an ADTS file: frames (symgpu_adts_index: header rules of adts.rs:130-309) -> raw_data_block payloads -> AAC-LC
    entropy front-end (symgpu_aac_fe_*) -> the synthesis stage's batch.  The reader gives every frame 1024 samples and trims
    nothing.  Returns dict(units [n,2], tns, coeffs [n,2,1024], runs, spans, channels, sample_rate, total_frames).  Packets the
    front-end refuses are dropped, as a caller of the reference drops a DecodeError.  index: the result of adts_aac_index (else
    computed here); out: (units, coeffs) staging slices with room for every packet; threads > 1: a stream of 32 blocks or more is
    decoded as independent jobs when it allows that."""
    packets, rate, channels = adts_aac_index(data) if index is None else index
    table = np.zeros(len(packets), dtype=nat.PIECE_DTYPE)
    table["offset"], table["len"] = packets["offset"], packets["size"]
    jobs = frontend.aac_decode_packets_jobs(rate, channels, data, table, threads=threads) if (threads > 1 and out is None and len(packets) >= 32) else None
    if jobs is not None:            # one long stream: its blocks as independent jobs on host threads (identical output, DESIGN 10.9)
        units, tns, coeffs = jobs
    else:                           # (or the stream needs the serial path: a refused block, a changed layout, ...)
        fe = frontend.AacFrontend(rate, channels)
        units, tns, coeffs, _ = fe.decode_packets(data, table, out=out)
        fe.close()
    n = len(units)
    runs = np.zeros(1, dtype=nat.AAC_RUN_DTYPE)
    runs[0]["n_frames"], runs[0]["channels"] = n, channels
    spans = np.zeros(n, dtype=nat.PCM_SPAN_DTYPE)
    spans["src"] = np.arange(n, dtype=np.uint64) * 2048
    spans["plane_stride"], spans["frames"] = 1024, 1024
    spans["dst_frame"] = np.arange(n, dtype=np.uint64) * 1024
    return dict(units=units, tns=tns, coeffs=coeffs, runs=runs, spans=spans, channels=channels, sample_rate=rate,
                total_frames=1024 * n)


class Arena:
    """Reusable staging memory for `plan_files`: take(name, shape, dtype) hands out a view of a buffer that persists across calls (and
    grows when too small), so that a serving loop's front-ends write into pages that are already mapped instead of paying the first
    touch of fresh allocations on every batch (DESIGN 5g).  Contents are whatever the last user left."""

    def __init__(self):
        self._buf = {}

    def take(self, name, shape, dtype):
        need = int(np.prod(shape, dtype=np.int64)) * np.dtype(dtype).itemsize
        b = self._buf.get(name)
        if b is None or b.size < need:
            b = np.zeros(max(need + need // 4, 1), dtype=np.uint8)
            b[::4096] = 0          # touch every page once, here
            self._buf[name] = b
        return b[:need].view(dtype).reshape(shape)


def decode_adts_aac(engine, data, fmt=nat.FMT_S16, stream=0, threads=1):
    """(samples [frames, channels] of `fmt`, sample_rate) of an ADTS AAC-LC file; stream slot `stream` of `engine` is reset first."""
    plan = adts_aac_plan(data, threads=threads)
    if len(plan["units"]) == 0:
        return np.zeros((0, plan["channels"]), dtype=nat.FMT_NUMPY[fmt]), plan["sample_rate"]
    plan["runs"]["stream"] = stream
    engine.aac_stream_reset(stream)
    pcm = engine.aac_synth_host(plan["units"], plan["tns"], plan["coeffs"], plan["runs"])
    return engine.pcm_pack_host(pcm, plan["spans"], plan["channels"], fmt, plan["total_frames"]), plan["sample_rate"]


# ---- many files at once: one synthesis launch per codec --------------------------------------------------------------------

def sniff(data):
    """'vorbis' (Ogg capture pattern), 'flac' (native FLAC marker), 'aac' (ADTS: 12 sync bits, layer field 00) or 'mpa' (anything else:
    the MPEG audio indexer looks for a frame, skipping tags and junk)."""
    head = bytes(data[:4])
    if head == b"OggS":
        return "vorbis"
    if head == b"fLaC":
        return "flac"  # the integer path: restoration + FromSample<i32> on the device, not the f32 synthesis batches
    if len(head) >= 2 and head[0] == 0xFF and (head[1] & 0xF6) == 0xF0:
        return "aac"
    return "mpa"


def plan_file(data):
    """CPU half of one file: dict(kind, ...) -- kind 'mp3' / 'mpa1' / 'mpa2' / 'aac' / 'vorbis' / 'vorbis_mc' / 'flac' (flac_plan)."""
    kind = sniff(data)
    if kind == "vorbis":
        p = ogg_vorbis_plan(data)
        return dict(p, kind="vorbis_mc" if p.get("mc") else "vorbis")
    if kind == "aac":
        return dict(adts_aac_plan(data), kind="aac")
    if kind == "flac":
        return dict(flac_plan(data), kind="flac")
    layer, payload, runs, spans, rate, channels, total = mpeg_audio_plan(data)
    return dict(kind={1: "mpa1", 2: "mpa2", 3: "mp3"}[layer], payload=payload, runs=runs, spans=spans, sample_rate=rate, channels=channels, total_frames=total)


def plan_files(files, threads=None, arena=None):
    """Plans every file (front-ends on `threads` host threads: the native calls release the interpreter lock) and merges the plans
    into one batch per codec, every file a stream of its own.  Returns (plans, batches): batches[kind] = dict(members = indices into
    `files`, first = each member's first unit in the batch, + the arrays of that codec's synthesis entry point).  AAC files are indexed
    first and then decoded straight into their slices of the batch arrays (taken from `arena` when given: reusable staging memory);
    a file whose front-end refuses packets leaves the tail of its slice unused -- runs name what is valid.
    Vorbis files the two-plane synthesis takes form the batch 'vorbis'; the others (3 to 8 channels, other couplings) the batch
    'vorbis_mc', whose arrays carry `planes` = the largest channel count among its members and whose members keep their own channel
    maps (plane_of_channel) for the output stage.
    Native FLAC files are planned by flac_plan (kind 'flac') and form the batch 'flac', the input of ONE symgpu_flac_decode_host call:
    frames, subframes and samples concatenated (first_subframe and the sub-frame offsets re-based), dst placing every file's output in
    its own [total_frames, channels] region of one flat buffer of out_samples samples, out_first[k] = where member k's region starts.
    FLAC plans have no spans: pack_files leaves them alone and decode_files fills them in from that call.
    A file that cannot be indexed or planned at all (an Ogg stream that is not Vorbis, more than eight channels, floor 0, an ADTS channel
    configuration outside 1 / 2, a FLAC file without a valid STREAMINFO, ...) does not take the others down: its plan is
    dict(kind="error", error=<message>) with no spans, it is in no batch, and pack_files returns an empty result for it."""
    import concurrent.futures
    import os
    kinds = [sniff(f) for f in files]
    errors = {}

    def guarded(fn):
        def run(i):
            try:
                return fn(i)
            except Exception as e:  # noqa: BLE001 -- one bad file must not abort the batch; the message is kept in its plan
                errors[i] = f"{type(e).__name__}: {e}"
                return None
        return run

    def error_plan(i):
        return dict(kind="error", error=errors[i], spans=np.zeros(0, dtype=nat.PCM_SPAN_DTYPE), channels=0, sample_rate=0, total_frames=0)
    aac = [i for i, k in enumerate(kinds) if k == "aac"]
    with concurrent.futures.ThreadPoolExecutor(max_workers=threads or os.cpu_count()) as pool:
        index = dict(zip(aac, pool.map(guarded(lambda i: adts_aac_index(files[i])), aac)))
        aac = [i for i in aac if i not in errors]
        starts, total = {}, 0
        for i in aac:
            starts[i] = total
            total += len(index[i][0])
        take = arena.take if arena is not None else (lambda name, shape, dtype: np.zeros(shape, dtype=dtype))
        aac_units, aac_coeffs = take("aac_units", (total, 2), nat.AAC_UNIT_DTYPE), take("aac_coeffs", (total, 2, 1024), np.float32)
        vor = [i for i, k in enumerate(kinds) if k == "vorbis"]
        vindex = dict(zip(vor, pool.map(guarded(lambda i: ogg_vorbis_index(files[i])), vor)))
        vmc = [i for i in vor if i not in errors and vindex[i]["fe"].mc]       # the multichannel batch
        vor = [i for i in vor if i not in errors and not vindex[i]["fe"].mc]
        vstarts, vfloor, vtotal, nfl = {}, {}, 0, 0
        for i in vor:
            vstarts[i], vfloor[i] = vtotal, nfl
            vtotal += len(vindex[i]["table"])
            nfl += len(vindex[i]["fe"].floors)
        vslot = max([vindex[i]["fe"].slot for i in vor], default=0)
        v_units, v_fy = take("vorbis_units", (vtotal,), nat.VORBIS_UNIT_DTYPE), take("vorbis_floor_y", (vtotal, 2, 65), np.uint16)
        v_res = take("vorbis_residue", (vtotal, 2, vslot), np.float32)
        mstarts, mfloor, mtotal, nfl = {}, {}, 0, 0
        for i in vmc:
            mstarts[i], mfloor[i] = mtotal, nfl
            mtotal += len(vindex[i]["table"])
            nfl += len(vindex[i]["fe"].floors)
        mslot = max([vindex[i]["fe"].slot for i in vmc], default=0)
        mplanes = max([vindex[i]["fe"].channels for i in vmc], default=1)
        m_units = take("vorbis_mc_units", (mtotal,), nat.VORBIS_UNIT_MC_DTYPE)
        m_fy, m_res = take("vorbis_mc_floor_y", (mtotal, mplanes, 65), np.uint16), take("vorbis_mc_residue", (mtotal, mplanes, mslot), np.float32)

        def plan(i):
            if i in errors:
                return error_plan(i)
            if kinds[i] == "vorbis" and i in mstarts:
                a, n = mstarts[i], len(vindex[i]["table"])
                p = ogg_vorbis_plan(files[i], index=vindex[i], out=(m_units[a:a + n], m_fy[a:a + n], m_res[a:a + n]), slot=mslot, floor_base=mfloor[i],
                                    planes=mplanes)
                m_units[a + len(p["units"]):a + n].view(np.uint8)[...] = 0
                return dict(p, kind="vorbis_mc", slice_start=a)
            if kinds[i] == "vorbis":
                a, n = vstarts[i], len(vindex[i]["table"])
                p = ogg_vorbis_plan(files[i], index=vindex[i], out=(v_units[a:a + n], v_fy[a:a + n], v_res[a:a + n]), slot=vslot, floor_base=vfloor[i])
                tail = v_units[a + len(p["units"]):a + n].view(np.uint8)
                tail[...] = 0
                return dict(p, kind="vorbis", slice_start=a)
            if kinds[i] == "flac":
                return dict(flac_plan(files[i]), kind="flac")
            if kinds[i] != "aac":
                return plan_file(files[i])
            a, n = starts[i], len(index[i][0])
            p = adts_aac_plan(files[i], index[i], out=(aac_units[a:a + n], aac_coeffs[a:a + n]))
            aac_units[a + len(p["units"]):a + n].view(np.uint8)[...] = 0   # refused packets: the unused tail holds valid (empty) records
            return dict(p, kind="aac", slice_start=a)
        plans = list(pool.map(guarded(plan), range(len(files))))
    for i, p in enumerate(plans):
        if p is None:  # failed in the plan stage: its slice of the batch arrays stays empty records, its front-end is released now
            plans[i] = error_plan(i)
            if kinds[i] == "vorbis" and i in vindex and vindex[i] is not None and hasattr(vindex[i].get("fe"), "close"):
                vindex[i]["fe"].close()
            if kinds[i] == "vorbis" and i in vstarts:
                a, n = vstarts[i], len(vindex[i]["table"])
                v_units[a:a + n].view(np.uint8)[...] = 0
            if kinds[i] == "vorbis" and i in mstarts:
                a, n = mstarts[i], len(vindex[i]["table"])
                m_units[a:a + n].view(np.uint8)[...] = 0
            if kinds[i] == "aac" and i in starts:
                a, n = starts[i], len(index[i][0])
                aac_units[a:a + n].view(np.uint8)[...] = 0
    batches = {}
    for kind in ("mp3", "mpa1", "mpa2", "aac", "vorbis", "vorbis_mc"):
        members = [i for i, p in enumerate(plans) if p["kind"] == kind and len(p["spans"])]
        if not members:
            continue
        first, at = [], 0
        for i in members:
            first.append(at)
            at += len(plans[i]["spans"])
        b = dict(members=members, first=first)
        if kind == "mp3":
            b["units"] = np.concatenate([plans[i]["payload"][0] for i in members])
            b["quant"] = np.concatenate([plans[i]["payload"][1] for i in members])
            runs = np.concatenate([plans[i]["runs"] for i in members])
        elif kind in ("mpa1", "mpa2"):
            b["subbands"] = np.concatenate([plans[i]["payload"] for i in members])
            runs = np.concatenate([plans[i]["runs"] for i in members])
        elif kind == "aac":
            base = 0
            for i in members:                                  # the units already lie in the batch array: re-base their TNS references
                u = plans[i]["units"]
                u["tns_first"] = np.where(u["n_tns"] > 0, u["tns_first"] + base, 0)
                base += len(plans[i]["tns"])
            b["first"] = first = [plans[i]["slice_start"] for i in members]
            b["units"], b["coeffs"] = aac_units, aac_coeffs
            b["tns"] = np.concatenate([plans[i]["tns"] for i in members])
            runs = np.concatenate([plans[i]["runs"] for i in members])
        elif kind == "vorbis":
            b["first"] = first = [plans[i]["slice_start"] for i in members]
            b["streams"] = np.concatenate([plans[i]["stream"] for i in members])
            b["floors"] = np.concatenate([vindex[i]["fe"].floors for i in vor])      # every Vorbis file's tables, in file order (floor_base)
            b["units"], b["floor_y"], b["residue"], b["slot"] = v_units, v_fy, v_res, vslot
            runs = np.concatenate([plans[i]["runs"] for i in members])
        else:
            b["first"] = first = [plans[i]["slice_start"] for i in members]
            b["streams"] = np.concatenate([plans[i]["stream"] for i in members])
            b["floors"] = np.concatenate([vindex[i]["fe"].floors for i in vmc])
            b["units"], b["floor_y"], b["residue"], b["slot"], b["planes"] = m_units, m_fy, m_res, mslot, mplanes
            runs = np.concatenate([plans[i]["runs"] for i in members])
        runs = runs.copy()
        runs["stream"] = np.arange(len(members))
        runs["first_packet" if kind in ("vorbis", "vorbis_mc") else "first_frame"] = first
        b["runs"] = runs
        batches[kind] = b
    members = [i for i, p in enumerate(plans) if p["kind"] == "flac" and len(p["frames"])]
    if members:
        frames, subs, dst, out_first = [], [], [], []
        n_sub = n_smp = out_at = 0
        for i in members:
            p = plans[i]
            f, s = p["frames"].copy(), p["subframes"].copy()
            f["first_subframe"] += n_sub
            s["offset"] += np.uint64(n_smp)
            frames.append(f), subs.append(s), dst.append(flac_dst(p, out_at)), out_first.append(out_at)
            n_sub, n_smp, out_at = n_sub + len(s), n_smp + len(p["samples"]), out_at + p["total_frames"] * p["channels"]
        batches["flac"] = dict(members=members, out_first=out_first, out_samples=out_at, frames=np.concatenate(frames),
                               subframes=np.concatenate(subs), samples=np.concatenate([plans[i]["samples"] for i in members]),
                               dst=np.concatenate(dst))
    return plans, batches


def _file_spans(plan, batch, k, unit_floats, plane_stride=None):
    """The file's spans, re-based onto its slice of the batch's PCM (unit_floats per unit)."""
    sp = plan["spans"].copy()
    sp["src"] = np.arange(len(sp), dtype=np.uint64) * unit_floats
    if plane_stride is not None:
        sp["plane_stride"] = plane_stride
    return sp


def pack_files(plans, batches, pcm, pack, fmt, pack_mapped=None):
    """Output stage per file: pcm[kind] = the batch's planar output, pack(pcm_slice, spans, channels, fmt, total_frames) the packer,
    pack_mapped(pcm_slice, spans, channels, plane_of_channel, fmt, total_frames) the one for files with a channel map ('vorbis_mc').
    FLAC plans and the 'flac' batch are not packed here (their output stage is part of symgpu_flac_decode_*): their entries stay None."""
    out = [None] * len(plans)
    for i, p in enumerate(plans):
        if p["kind"] != "flac" and not len(p["spans"]):
            out[i] = (np.zeros((0, p["channels"]), dtype=nat.FMT_NUMPY[fmt]), p["sample_rate"])
    for kind, b in batches.items():
        if kind == "flac":
            continue
        flat = np.ascontiguousarray(pcm[kind]).reshape(-1)
        per = flat.size // len(pcm[kind])          # floats per unit: two planes (b["planes"] in the multichannel batch)
        for k, i in enumerate(b["members"]):
            p = plans[i]
            n = len(p["spans"])
            sl = flat[b["first"][k] * per:(b["first"][k] + n) * per]
            sp = _file_spans(p, b, k, per, per // b.get("planes", 2))
            if "plane_of_channel" in p:
                out[i] = (pack_mapped(sl, sp, p["channels"], p["plane_of_channel"], fmt, p["total_frames"]), p["sample_rate"])
            else:
                out[i] = (pack(sl, sp, p["channels"], fmt, p["total_frames"]), p["sample_rate"])
    return out


def decode_files(engine, files, fmt=nat.FMT_S16, threads=None):
    """[(samples [frames, channels], sample_rate)] for a list of MPEG audio / ADTS AAC-LC / Ogg Vorbis / native FLAC files: front-ends on
    host threads, ONE synthesis call per codec over all files (every file a stream; multichannel Vorbis files a second one), output stage
    per file.  All FLAC files share one symgpu_flac_decode_host call (restoration, FromSample<i32> into `fmt`, interleaving), whose
    output is cut per file.  (Re)allocates the engine's stream slots."""
    plans, batches = plan_files(files, threads)
    pcm, flac = {}, None
    for kind, b in batches.items():
        n_streams = len(b["members"])
        if kind == "flac":
            flac = engine.flac_decode_host(b["frames"], b["subframes"], b["samples"], b["dst"], fmt, b["out_samples"])
        elif kind == "mp3":
            engine.mp3_streams_alloc(n_streams)
            pcm[kind] = engine.mp3_synth_host_quantized(b["units"], b["quant"], b["runs"])
        elif kind in ("mpa1", "mpa2"):
            engine.mp3_streams_alloc(n_streams)
            pcm[kind] = engine.mpa12_synth_host(b["subbands"], b["runs"])
        elif kind == "aac":
            engine.aac_streams_alloc(n_streams)
            pcm[kind] = engine.aac_synth_host(b["units"], b["tns"], b["coeffs"], b["runs"])
        elif kind == "vorbis":
            engine.vorbis_streams_set(b["streams"])
            engine.vorbis_floors_set(b["floors"])
            pcm[kind] = engine.vorbis_synth_host(b["units"], b["floor_y"], b["residue"], b["runs"], b["slot"])
        else:   # (a context holds classic or multichannel Vorbis streams at a time: this batch runs after 'vorbis')
            engine.vorbis_mc_streams_set(b["streams"])
            engine.vorbis_floors_set(b["floors"])
            pcm[kind] = engine.vorbis_mc_synth_host(b["units"], b["floor_y"], b["residue"], b["runs"], b["planes"], b["slot"])
    out = pack_files(plans, batches, pcm, engine.pcm_pack_host, fmt, engine.pcm_pack_host_mapped)
    at = dict(zip(batches["flac"]["members"], batches["flac"]["out_first"])) if flac is not None else {}
    for i, p in enumerate(plans):
        if p["kind"] == "flac":
            n, ch = (p["total_frames"], p["channels"]) if i in at else (0, p["channels"])
            region = flac[at[i]:at[i] + n * ch] if i in at else np.zeros(0, dtype=nat.FMT_NUMPY[fmt])
            out[i] = (region.reshape(n, ch), p["sample_rate"])
    return out


# ---- FLAC (integer path: restoration on the GPU, samples stay int32 as in the reference's AudioBuffer<i32>) ----------------------

def flac_plan(data):
    """CPU half for a native FLAC file: marker + STREAMINFO + checksum-validated frame split (symgpu_flac_index), frame / sub-frame / Rice
    reader (symgpu_flac_fe_decode_packets) -> dict(frames, subframes, samples (int32: warm-up samples + residuals), info, channels,
    sample_rate, bits_per_sample, total_frames): the input of Engine.flac_restore_host."""
    info, packets = packetizer.flac_index(data)
    table = np.zeros(len(packets), dtype=nat.PIECE_DTYPE)
    table["offset"], table["len"] = packets["offset"], packets["size"]
    frames, infos, frame_of, subs, samples = frontend.flac_decode_packets(data, table, int(info["bits_per_sample"]), int(info["channels"]), int(info["block_max"]))
    total = int(sum(int(subs[int(f["first_subframe"])]["n"]) for f in frames))
    return dict(frames=frames, subframes=subs, samples=samples, info=info, channels=int(info["channels"]), sample_rate=int(info["sample_rate"]),
                bits_per_sample=int(info["bits_per_sample"]), total_frames=total)


def flac_interleave(plan, restored):
    """[total_frames, channels] int32 from the restored planes (each sub-frame's n samples at its offset), frames in stream order."""
    out = np.zeros((plan["total_frames"], plan["channels"]), dtype=np.int32)
    at = 0
    for f in plan["frames"]:
        first = int(f["first_subframe"])
        n = int(plan["subframes"][first]["n"])
        for c in range(int(f["channels"])):
            sf = plan["subframes"][first + c]
            out[at:at + n, c] = restored[int(sf["offset"]):int(sf["offset"]) + n]
        at += n
    return out


def flac_dst(plan, base=0):
    """Output position (in samples) of every frame of a FLAC plan for symgpu_flac_decode_*: the frames back to back from `base`, each
    n * channels samples, so that the plan's output is one [total_frames, channels] region."""
    frames = plan["frames"]
    n = plan["subframes"]["n"][frames["first_subframe"]].astype(np.uint64) * frames["channels"].astype(np.uint64)
    return (np.uint64(base) + np.concatenate([[0], np.cumsum(n)[:-1]])).astype(np.uint64) if len(frames) else np.zeros(0, dtype=np.uint64)


def decode_flac(engine, data, fmt=None):
    """(samples [frames, channels], sample_rate) of a native FLAC file.  fmt None: int32 scaled to 32 bits as the reference's FLAC
    decoder leaves them (AudioBuffer<i32>); else samples of that FMT_* by FromSample<i32> (conv.rs:514-532).  Restoration, conversion and
    interleaving run in one device call (symgpu_flac_decode_host; None is its identity conversion FMT_S32)."""
    plan = flac_plan(data)
    code = nat.FMT_S32 if fmt is None else fmt
    out = np.zeros((plan["total_frames"], plan["channels"]), dtype=nat.FMT_NUMPY[code])
    if len(plan["frames"]) == 0:
        return out, plan["sample_rate"]
    engine.flac_decode_host(plan["frames"], plan["subframes"], plan["samples"], flac_dst(plan), code, out=out)
    return out, plan["sample_rate"]
