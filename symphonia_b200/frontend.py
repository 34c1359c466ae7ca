"""MP3 entropy front-end (SURVEY §8f N1) through the C ABI (`symgpu_mp3_fe_*`, include/symgpu.h): MPEG frame bytes ->
`symgpu_mp3_gc` units + int16 quantised spectra, the input of `Engine.mp3_synth_host_quantized`.  CPU only; mirrors
`MpaDecoder::decode_inner` + `Layer3::decode` up to the synthesis seam (symphonia-bundle-mp3/src/decoder.rs:84-131,
layer3/mod.rs:373-418)."""
import ctypes

import numpy as np

from . import _native as nat
from .engine import SymgpuError

_vp = ctypes.c_void_p


class Mp3Frontend:
    """One stream's front-end state (the bit reservoir and the signal specification of its first frame)."""

    def __init__(self):
        self._L = nat.lib()
        h = _vp()
        rc = self._L.symgpu_mp3_fe_create(ctypes.byref(h))
        if rc != 0:
            raise SymgpuError(rc, "symgpu_mp3_fe_create")
        self._h = h

    def close(self):
        if self._h:
            self._L.symgpu_mp3_fe_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()

    def reset(self):
        self._L.symgpu_mp3_fe_reset(self._h)

    def decode(self, frame):
        """(units[2][2], quant[2][2][576] int16, info) of one packet; SymgpuError(status 1 / 2) where the reference errors."""
        a = np.frombuffer(bytes(frame), dtype=np.uint8)
        units = np.zeros((2, 2), dtype=nat.MP3_GC_DTYPE)
        quant = np.zeros((2, 2, 576), dtype=np.int16)
        info = np.zeros(1, dtype=nat.MP3_FRAME_INFO_DTYPE)
        rc = self._L.symgpu_mp3_fe_decode(self._h, _vp(a.ctypes.data) if a.size else None, a.size, _vp(units.ctypes.data), _vp(quant.ctypes.data),
                                          _vp(info.ctypes.data))
        if rc != 0:
            raise SymgpuError(rc, "symgpu_mp3_fe_decode")
        return units, quant, info[0]

    def decode_packets(self, data, packets):
        """A whole stream: (units[n_good][2][2], quant[n_good][2][2][576], frame_of[n_good], info of the first good frame)."""
        a = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data
        packets = np.ascontiguousarray(packets, dtype=nat.MPA_PACKET_DTYPE)
        n = len(packets)
        units = np.zeros((n, 2, 2), dtype=nat.MP3_GC_DTYPE)
        quant = np.zeros((n, 2, 2, 576), dtype=np.int16)
        frame_of = np.zeros(n, dtype=np.uint32)
        info = np.zeros(1, dtype=nat.MP3_FRAME_INFO_DTYPE)
        good = ctypes.c_size_t(0)
        rc = self._L.symgpu_mp3_fe_decode_packets(self._h, _vp(a.ctypes.data), a.size, _vp(packets.ctypes.data), n, _vp(units.ctypes.data),
                                                  _vp(quant.ctypes.data), _vp(frame_of.ctypes.data), ctypes.byref(good), _vp(info.ctypes.data))
        if rc != 0:
            raise SymgpuError(rc, "symgpu_mp3_fe_decode_packets")
        g = good.value
        return units[:g], quant[:g], frame_of[:g], info[0]


def _u8(data):
    return np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else np.ascontiguousarray(data, dtype=np.uint8)


def entropy_plan(data, packets, bad=None):
    """The side-information pass: (md bytes, jobs [n_good*4] of 64 opaque bytes, frame_of, info).  No Huffman data is read."""
    L = nat.lib()
    a = _u8(data)
    packets = np.ascontiguousarray(packets, dtype=nat.MPA_PACKET_DTYPE)
    n = len(packets)
    md = np.zeros(int(packets["size"].sum()) + 8, dtype=np.uint8)
    jobs = np.zeros((n * 4, 8), dtype=np.uint64)
    frame_of = np.zeros(n, dtype=np.uint32)
    info = np.zeros(1, dtype=nat.MP3_FRAME_INFO_DTYPE)
    md_len, good = ctypes.c_size_t(0), ctypes.c_size_t(0)
    badp = None if bad is None else _vp(np.ascontiguousarray(bad, dtype=np.uint8).ctypes.data)
    rc = L.symgpu_mp3_entropy_plan(_vp(a.ctypes.data), a.size, _vp(packets.ctypes.data), n, badp, _vp(md.ctypes.data), md.size, ctypes.byref(md_len),
                                   _vp(jobs.ctypes.data), _vp(frame_of.ctypes.data), ctypes.byref(good), _vp(info.ctypes.data))
    if rc != 0:
        raise SymgpuError(rc, "symgpu_mp3_entropy_plan")
    return md[:md_len.value], jobs[:good.value * 4], frame_of[:good.value], info[0]


def entropy_run_cpu(md, jobs, threads=1):
    """The kernel body on the host: (units[F][2][2], quant[F][2][2][576], failed[F]); threads > 1 (0 = all cores) splits the jobs."""
    L = nat.lib()
    md = np.ascontiguousarray(md, dtype=np.uint8)
    jobs = np.ascontiguousarray(jobs, dtype=np.uint64)
    n_frames = (len(jobs) + 3) // 4  # slots are relative to the first job's frame
    units = np.zeros((n_frames, 2, 2), dtype=nat.MP3_GC_DTYPE)
    quant = np.zeros((n_frames, 2, 2, 576), dtype=np.int16)
    failed = np.zeros(n_frames, dtype=np.uint8)
    if threads == 1:
        rc = L.symgpu_mp3_entropy_run_cpu(_vp(md.ctypes.data) if md.size else None, md.size, _vp(jobs.ctypes.data), len(jobs), _vp(units.ctypes.data),
                                          _vp(quant.ctypes.data), _vp(failed.ctypes.data))
    else:
        rc = L.symgpu_mp3_entropy_run_cpu_mt(_vp(md.ctypes.data) if md.size else None, md.size, _vp(jobs.ctypes.data), len(jobs), _vp(units.ctypes.data),
                                             _vp(quant.ctypes.data), _vp(failed.ctypes.data), threads)
    if rc != 0:
        raise SymgpuError(rc, "symgpu_mp3_entropy_run_cpu")
    return units, quant, failed


def entropy_decode_cpu(data, packets):
    """plan -> jobs -> re-plan until nothing fails: (units, quant, frame_of, info, rounds), equal to Mp3Frontend.decode_packets on a fresh stream."""
    L = nat.lib()
    a = _u8(data)
    packets = np.ascontiguousarray(packets, dtype=nat.MPA_PACKET_DTYPE)
    n = len(packets)
    units = np.zeros((n, 2, 2), dtype=nat.MP3_GC_DTYPE)
    quant = np.zeros((n, 2, 2, 576), dtype=np.int16)
    frame_of = np.zeros(n, dtype=np.uint32)
    info = np.zeros(1, dtype=nat.MP3_FRAME_INFO_DTYPE)
    good, rounds = ctypes.c_size_t(0), ctypes.c_uint32(0)
    rc = L.symgpu_mp3_entropy_decode_cpu(_vp(a.ctypes.data), a.size, _vp(packets.ctypes.data), n, _vp(units.ctypes.data), _vp(quant.ctypes.data),
                                         _vp(frame_of.ctypes.data), ctypes.byref(good), _vp(info.ctypes.data), ctypes.byref(rounds))
    if rc != 0:
        raise SymgpuError(rc, "symgpu_mp3_entropy_decode_cpu")
    g = good.value
    return units[:g], quant[:g], frame_of[:g], info[0], rounds.value


def mpa12_decode(frame, layer):
    """One Layer I / II packet -> (subbands [2][32][n_slots] f32, info); SymgpuError where the reference errors."""
    a = _u8(bytes(frame))
    n_slots = 12 if layer == 1 else 36
    out = np.zeros((2, 32, n_slots), dtype=np.float32)
    info = np.zeros(1, dtype=nat.MP3_FRAME_INFO_DTYPE)
    rc = nat.lib().symgpu_mpa12_fe_decode(_vp(a.ctypes.data) if a.size else None, a.size, layer, _vp(out.ctypes.data), _vp(info.ctypes.data))
    if rc != 0:
        raise SymgpuError(rc, "symgpu_mpa12_fe_decode")
    return out, info[0]


def mpa12_decode_packets(data, packets, layer):
    """A Layer I / II stream -> (subbands [n_good][2][32][n_slots], frame_of, info): the input of Engine.mpa12_synth_host."""
    a = _u8(data)
    packets = np.ascontiguousarray(packets, dtype=nat.MPA_PACKET_DTYPE)
    n, n_slots = len(packets), 12 if layer == 1 else 36
    out = np.zeros((n, 2, 32, n_slots), dtype=np.float32)
    frame_of = np.zeros(n, dtype=np.uint32)
    info = np.zeros(1, dtype=nat.MP3_FRAME_INFO_DTYPE)
    good = ctypes.c_size_t(0)
    rc = nat.lib().symgpu_mpa12_fe_decode_packets(_vp(a.ctypes.data), a.size, _vp(packets.ctypes.data), n, layer, _vp(out.ctypes.data), _vp(frame_of.ctypes.data),
                                                  ctypes.byref(good), _vp(info.ctypes.data))
    if rc != 0:
        raise SymgpuError(rc, "symgpu_mpa12_fe_decode_packets")
    return out[:good.value], frame_of[:good.value], info[0]


def mpa12_constants():
    out = np.zeros(98, dtype=np.float32)
    nat.lib().symgpu_mpa12_constants(_vp(out.ctypes.data), 98)
    return out[:64], out[64:81], out[81:]


def flac_decode_packets(data, packets, stream_bps=0, stream_channels=0, max_block=0):
    """FLAC packets (PIECE_DTYPE offset / len table over `data`) -> (frames, infos, frame_of, subframes, samples): the input of
    Engine.flac_restore_host.  Packets the reference refuses are left out."""
    a = _u8(data)
    packets = np.ascontiguousarray(packets, dtype=nat.PIECE_DTYPE)
    n = len(packets)
    frames = np.zeros(n, dtype=nat.FLAC_FRAME_DTYPE)
    infos = np.zeros(n, dtype=nat.FLAC_FRAME_INFO_DTYPE)
    frame_of = np.zeros(n, dtype=np.uint32)
    subs = np.zeros(n * 8, dtype=nat.FLAC_SUBFRAME_DTYPE)
    cap = 1 << 16
    while True:
        samples = np.zeros(cap, dtype=np.int32)
        good, n_subs, n_smp = ctypes.c_size_t(0), ctypes.c_size_t(0), ctypes.c_size_t(0)
        rc = nat.lib().symgpu_flac_fe_decode_packets(_vp(a.ctypes.data), a.size, _vp(packets.ctypes.data), n, stream_bps, stream_channels, max_block,
                                                     _vp(frames.ctypes.data), _vp(infos.ctypes.data), _vp(frame_of.ctypes.data), _vp(subs.ctypes.data), len(subs),
                                                     _vp(samples.ctypes.data), cap, ctypes.byref(good), ctypes.byref(n_subs), ctypes.byref(n_smp))
        if rc == 3 and cap < (1 << 31):
            cap *= 4
            continue
        if rc != 0:
            raise SymgpuError(rc, "symgpu_flac_fe_decode_packets")
        g = good.value
        return frames[:g], infos[:g], frame_of[:g], subs[:n_subs.value], samples[:n_smp.value]


class VorbisFrontend:
    """One Vorbis stream's entropy front-end (codebooks, setup, previous block): identification + setup packets in, then audio
    packets -> (unit, floor_y [2][65], residue [2][slot]), the input of Engine.vorbis_synth_host.  mc=True opens the stream with
    symgpu_vorbis_fe_create_mc (1-8 channels, any coupling list): then `stream` is a VORBIS_STREAM_MC_DTYPE record and packets come
    out as (unit VORBIS_UNIT_MC_DTYPE, floor_y [planes][65], residue [planes][slot]), the input of Engine.vorbis_mc_synth_host;
    `planes` (default: the stream's channel count) may be larger, so that streams of different channel counts share a batch."""

    def __init__(self, ident_packet, setup_packet, mc=False):
        self._h = None
        self._L = nat.lib()
        self.mc = bool(mc)
        a, b = _u8(bytes(ident_packet)), _u8(bytes(setup_packet))
        h = _vp()
        create = self._L.symgpu_vorbis_fe_create_mc if self.mc else self._L.symgpu_vorbis_fe_create
        rc = create(_vp(a.ctypes.data), a.size, _vp(b.ctypes.data), b.size, ctypes.byref(h))
        if rc != 0:
            raise SymgpuError(rc, "symgpu_vorbis_fe_create_mc" if self.mc else "symgpu_vorbis_fe_create")
        self._h = h
        stream = np.zeros(1, dtype=nat.VORBIS_STREAM_MC_DTYPE if self.mc else nat.VORBIS_STREAM_DTYPE)
        floors = np.zeros(64, dtype=nat.VORBIS_FLOOR1_DTYPE)
        n = ctypes.c_uint32(0)
        config = self._L.symgpu_vorbis_fe_config_mc if self.mc else self._L.symgpu_vorbis_fe_config
        config(self._h, _vp(stream.ctypes.data), _vp(floors.ctypes.data), ctypes.byref(n))
        self.stream, self.floors = stream[0], floors[:n.value]
        self.slot = (1 << int(self.stream["bs1_exp"])) >> 1
        self.channels = int(self.stream["channels"])

    def close(self):
        if self._h:
            self._L.symgpu_vorbis_fe_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()

    def reset(self):
        self._L.symgpu_vorbis_fe_reset(self._h)

    def _layout(self, planes):
        if not self.mc:
            return nat.VORBIS_UNIT_DTYPE, 2
        return nat.VORBIS_UNIT_MC_DTYPE, self.channels if planes is None else int(planes)

    def decode(self, packet, slot=None, floor_base=0, planes=None):
        slot = self.slot if slot is None else slot
        udt, P = self._layout(planes)
        a = _u8(bytes(packet))
        unit = np.zeros(1, dtype=udt)
        floor_y = np.zeros((P, 65), dtype=np.uint16)
        residue = np.zeros((P, slot), dtype=np.float32)
        pk = (_vp(a.ctypes.data) if a.size else None, a.size, slot, floor_base)
        outs = (_vp(unit.ctypes.data), _vp(floor_y.ctypes.data), _vp(residue.ctypes.data))
        if self.mc:
            rc = self._L.symgpu_vorbis_fe_decode_mc(self._h, *pk, P, *outs)
        else:
            rc = self._L.symgpu_vorbis_fe_decode(self._h, *pk, *outs)
        if rc != 0:
            raise SymgpuError(rc, "symgpu_vorbis_fe_decode_mc" if self.mc else "symgpu_vorbis_fe_decode")
        return unit[0], floor_y, residue

    def decode_packets(self, data, packets, slot=None, floor_base=0, out=None, planes=None):
        """All audio packets of the stream in one call (PIECE_DTYPE table over `data`): (units [g], floor_y [g,P,65], residue [g,P,slot],
        packet_of [g]) with P = 2 (P = planes in mc mode); refused packets are left out.  out = (units [>= n], floor_y [>= n,P,65],
        residue [>= n,P,slot]): contiguous staging memory to decode into."""
        slot = self.slot if slot is None else slot
        udt, P = self._layout(planes)
        a = _u8(data)
        packets = np.ascontiguousarray(packets, dtype=nat.PIECE_DTYPE)
        n = len(packets)
        if out is None:
            units = np.zeros(n, dtype=udt)
            floor_y = np.zeros((n, P, 65), dtype=np.uint16)
            residue = np.zeros((n, P, slot), dtype=np.float32)
        else:
            units, floor_y, residue = out
            assert all(x.flags.c_contiguous and len(x) >= n for x in out) and residue.shape[1:] == (P, slot) and residue.dtype == np.float32
            assert units.dtype == udt and floor_y.dtype == np.uint16 and floor_y.shape[1:] == (P, 65)
        packet_of = np.zeros(n, dtype=np.uint32)
        good = ctypes.c_size_t(0)
        head = (self._h, _vp(a.ctypes.data) if a.size else None, a.size, _vp(packets.ctypes.data), n, slot, floor_base)
        tail = (_vp(units.ctypes.data), _vp(floor_y.ctypes.data), _vp(residue.ctypes.data), _vp(packet_of.ctypes.data), ctypes.byref(good))
        if self.mc:
            rc = self._L.symgpu_vorbis_fe_decode_packets_mc(*head, P, *tail)
        else:
            rc = self._L.symgpu_vorbis_fe_decode_packets(*head, *tail)
        if rc != 0:
            raise SymgpuError(rc, "symgpu_vorbis_fe_decode_packets_mc" if self.mc else "symgpu_vorbis_fe_decode_packets")
        g = good.value
        return units[:g], floor_y[:g], residue[:g], packet_of[:g]


def vorbis_channel_map(channels):
    """The reference's channel order (lib.rs:771-788): out[i] = output plane of Vorbis channel i, channels 1..8."""
    out = np.zeros(8, dtype=np.uint8)
    rc = nat.lib().symgpu_vorbis_channel_map(int(channels), _vp(out.ctypes.data))
    if rc != 0:
        raise SymgpuError(rc, "symgpu_vorbis_channel_map")
    return out[:channels]


class AacFrontend:
    """One AAC-LC stream's entropy front-end (window history, element layout, noise generator): raw_data_block packets ->
    (units [2], tns [n], coeffs [2][1024]), the input of Engine.aac_synth_host."""

    def __init__(self, sample_rate=0, channels=0, extra_data=None):
        """Stream parameters (the ADTS case), or `extra_data` = an AudioSpecificConfig (MP4 / Matroska)."""
        self._h = None
        self._L = nat.lib()
        h = _vp()
        if extra_data is not None:
            a = _u8(bytes(extra_data))
            asc = np.zeros(1, dtype=nat.AAC_ASC_DTYPE)
            rc = self._L.symgpu_aac_fe_create_asc(_vp(a.ctypes.data) if a.size else None, a.size, ctypes.byref(h), _vp(asc.ctypes.data))
            if rc != 0:
                raise SymgpuError(rc, "symgpu_aac_fe_create_asc")
            self.asc = asc[0]
            sample_rate, channels = int(asc[0]["sample_rate"]), int(asc[0]["channels"])
        else:
            rc = self._L.symgpu_aac_fe_create(int(sample_rate), int(channels), ctypes.byref(h))
            if rc != 0:
                raise SymgpuError(rc, "symgpu_aac_fe_create")
        self._h, self.channels, self.sample_rate = h, int(channels), int(sample_rate)

    def close(self):
        if self._h:
            self._L.symgpu_aac_fe_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()

    def reset(self):
        self._L.symgpu_aac_fe_reset(self._h)

    def decode(self, packet, tns_base=0):
        a = _u8(bytes(packet))
        units = np.zeros(2, dtype=nat.AAC_UNIT_DTYPE)
        tns = np.zeros(16, dtype=nat.AAC_TNS_DTYPE)
        coeffs = np.zeros((2, 1024), dtype=np.float32)
        n = ctypes.c_uint32(0)
        rc = self._L.symgpu_aac_fe_decode(self._h, _vp(a.ctypes.data) if a.size else None, a.size, int(tns_base), _vp(units.ctypes.data),
                                          _vp(tns.ctypes.data), ctypes.byref(n), _vp(coeffs.ctypes.data))
        if rc != 0:
            raise SymgpuError(rc, "symgpu_aac_fe_decode")
        return units, tns[:n.value], coeffs

    def decode_packets(self, data, packets, tns_base=0, out=None):
        """All packets of the stream in one call (PIECE_DTYPE table over `data`): (units [g,2], tns [t], coeffs [g,2,1024], frame_of [g]);
        refused packets are left out.  out = (units [>= n, 2], coeffs [>= n, 2, 1024]): contiguous staging memory to decode into."""
        a = _u8(data)
        packets = np.ascontiguousarray(packets, dtype=nat.PIECE_DTYPE)
        n = len(packets)
        tns = np.zeros(16 * n, dtype=nat.AAC_TNS_DTYPE)
        if out is None:
            units = np.zeros((n, 2), dtype=nat.AAC_UNIT_DTYPE)
            coeffs = np.zeros((n, 2, 1024), dtype=np.float32)
        else:
            units, coeffs = out
            assert units.flags.c_contiguous and coeffs.flags.c_contiguous and len(units) >= n and len(coeffs) >= n
            assert units.dtype == nat.AAC_UNIT_DTYPE and coeffs.dtype == np.float32
        frame_of = np.zeros(n, dtype=np.uint32)
        good, n_tns = ctypes.c_size_t(0), ctypes.c_size_t(0)
        rc = self._L.symgpu_aac_fe_decode_packets(self._h, _vp(a.ctypes.data) if a.size else None, a.size, _vp(packets.ctypes.data), n, int(tns_base),
                                                  _vp(units.ctypes.data), _vp(tns.ctypes.data), len(tns), _vp(coeffs.ctypes.data), _vp(frame_of.ctypes.data),
                                                  ctypes.byref(good), ctypes.byref(n_tns))
        if rc != 0:
            raise SymgpuError(rc, "symgpu_aac_fe_decode_packets")
        g = good.value
        return units[:g], tns[:n_tns.value], coeffs[:g], frame_of[:g]


def aac_tables():
    """(x^(4/3) [8192], normal scale factors [256], intensity scale factors [256]) as the front-end holds them."""
    p43, a, b = np.zeros(8192, dtype=np.float32), np.zeros(256, dtype=np.float32), np.zeros(256, dtype=np.float32)
    nat.lib().symgpu_aac_fe_tables(_vp(p43.ctypes.data), _vp(a.ctypes.data), _vp(b.ctypes.data))
    return p43, a, b


def aac_asc_parse(extra_data):
    """The AudioSpecificConfig as the reference reads it (AAC_ASC_DTYPE record); SymgpuError(1 / 2) where it refuses."""
    a = _u8(bytes(extra_data))
    out = np.zeros(1, dtype=nat.AAC_ASC_DTYPE)
    rc = nat.lib().symgpu_aac_asc_parse(_vp(a.ctypes.data) if a.size else None, a.size, _vp(out.ctypes.data))
    if rc != 0:
        raise SymgpuError(rc, "symgpu_aac_asc_parse")
    return out[0]


def aac_decode_packets_jobs(sample_rate, channels, data, packets, tns_base=0, threads=4):
    """The blocks of one AAC-LC stream as independent jobs on host threads (symgpu_aac_fe_decode_packets_jobs): (units [n,2], tns,
    coeffs [n,2,1024]) identical to AacFrontend.decode_packets, or None when the stream needs the serial path."""
    a = _u8(data)
    packets = np.ascontiguousarray(packets, dtype=nat.PIECE_DTYPE)
    n = len(packets)
    units = np.zeros((n, 2), dtype=nat.AAC_UNIT_DTYPE)
    tns = np.zeros(16 * n, dtype=nat.AAC_TNS_DTYPE)
    coeffs = np.zeros((n, 2, 1024), dtype=np.float32)
    n_tns = ctypes.c_size_t(0)
    rc = nat.lib().symgpu_aac_fe_decode_packets_jobs(int(sample_rate), int(channels), _vp(a.ctypes.data) if a.size else None, a.size, _vp(packets.ctypes.data), n,
                                                     int(tns_base), _vp(units.ctypes.data), _vp(tns.ctypes.data), len(tns), _vp(coeffs.ctypes.data),
                                                     ctypes.byref(n_tns), int(threads))
    if rc == 4:
        return None
    if rc != 0:
        raise SymgpuError(rc, "symgpu_aac_fe_decode_packets_jobs")
    return units, tns[:n_tns.value], coeffs


def vorbis_decode_packets_jobs(ident_packet, setup_packet, data, packets, slot, floor_base=0, threads=4, mc=False, planes=None):
    """One Vorbis stream's audio packets as independent jobs on host threads: (units [n], floor_y [n,P,65], residue [n,P,slot], accepted)
    with outputs at their packet's index; units[accepted] etc. equal VorbisFrontend(..., mc).decode_packets (P = 2, or `planes` in mc
    mode, default the stream's channel count)."""
    a, i_, s_ = _u8(data), _u8(bytes(ident_packet)), _u8(bytes(setup_packet))
    packets = np.ascontiguousarray(packets, dtype=nat.PIECE_DTYPE)
    n = len(packets)
    P = 2 if not mc else int(planes if planes is not None else (i_[11] if i_.size > 11 else 0))   # (ident byte 11: the channel count)
    units = np.zeros(n, dtype=nat.VORBIS_UNIT_MC_DTYPE if mc else nat.VORBIS_UNIT_DTYPE)
    floor_y = np.zeros((n, P, 65), dtype=np.uint16)
    residue = np.zeros((n, P, slot), dtype=np.float32)
    accepted = np.zeros(n, dtype=np.uint32)
    good = ctypes.c_size_t(0)
    head = (_vp(i_.ctypes.data), i_.size, _vp(s_.ctypes.data), s_.size, _vp(a.ctypes.data) if a.size else None, a.size, _vp(packets.ctypes.data), n,
            int(slot), int(floor_base))
    tail = (_vp(units.ctypes.data), _vp(floor_y.ctypes.data), _vp(residue.ctypes.data), _vp(accepted.ctypes.data), ctypes.byref(good), int(threads))
    if mc:
        rc = nat.lib().symgpu_vorbis_fe_decode_packets_jobs_mc(*head, P, *tail)
    else:
        rc = nat.lib().symgpu_vorbis_fe_decode_packets_jobs(*head, *tail)
    if rc != 0:
        raise SymgpuError(rc, "symgpu_vorbis_fe_decode_packets_jobs_mc" if mc else "symgpu_vorbis_fe_decode_packets_jobs")
    return units, floor_y, residue, accepted[:good.value]

