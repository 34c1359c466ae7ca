"""Engine: one symgpu context (one CUDA device, one stream) driven from Python.

Host entry points take numpy arrays (ideally backed by pinned memory); device entry points take
torch CUDA tensors that already live in HBM.  torch is plumbing only (allocation / pointers).
"""
import ctypes

import numpy as np

from . import _native
from ._native import (AAC_RUN_DTYPE, AAC_TNS_DTYPE, AAC_UNIT_DTYPE, FMT_NUMPY, MP3_GC_DTYPE, MP3_RUN_DTYPE, MPA12_RUN_DTYPE,
                      PCM_SPAN_DTYPE, VORBIS_FLOOR1_DTYPE, VORBIS_RUN_DTYPE, VORBIS_STREAM_DTYPE, VORBIS_STREAM_MC_DTYPE, VORBIS_UNIT_DTYPE,
                      VORBIS_UNIT_MC_DTYPE)


class SymgpuError(RuntimeError):
    def __init__(self, status, detail=""):
        self.status = status
        msg = _native.lib().symgpu_strerror(status).decode()
        super().__init__(f"{msg} [{status}] {detail}".strip())


def _np_ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


class Engine:
    def __init__(self, device=0):
        self._lib = _native.lib()
        self._ctx = ctypes.c_void_p()
        st = self._lib.symgpu_ctx_create(int(device), ctypes.byref(self._ctx))
        if st != 0:
            self._ctx = None
            raise SymgpuError(st, "symgpu_ctx_create failed: a B200-class CUDA device is required; "
                                  "there is no CPU fallback")
        self.device = int(device)

    # -- lifetime ---------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_ctx", None):
            self._lib.symgpu_ctx_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, st):
        if st != 0:
            raise SymgpuError(st, self._lib.symgpu_last_cuda_error(self._ctx).decode())

    # -- misc -------------------------------------------------------------------------------
    def sync(self):
        self._check(self._lib.symgpu_sync(self._ctx))

    @property
    def cuda_stream(self):
        return self._lib.symgpu_cuda_stream(self._ctx)

    @property
    def numa_node(self):
        """NUMA node the creating thread was bound to by symgpu_ctx_create (-1: unknown, -2: SYMGPU_NUMA_BIND=0)."""
        self._lib.symgpu_ctx_numa_node.restype = ctypes.c_int
        self._lib.symgpu_ctx_numa_node.argtypes = [ctypes.c_void_p]
        return int(self._lib.symgpu_ctx_numa_node(self._ctx))

    @property
    def launch_count(self):
        return int(self._lib.symgpu_launch_count(self._ctx))

    def upload_tables(self, blob):
        blob = np.ascontiguousarray(blob, dtype=np.uint8)
        self._check(self._lib.symgpu_tables_upload(self._ctx, _np_ptr(blob), blob.nbytes))

    # -- MP3 --------------------------------------------------------------------------------
    def mp3_streams_alloc(self, n_streams):
        self._check(self._lib.symgpu_mp3_streams_alloc(self._ctx, int(n_streams)))

    def mp3_stream_reset(self, stream):
        self._check(self._lib.symgpu_mp3_stream_reset(self._ctx, int(stream)))

    @staticmethod
    def _mp3_args(units, spectra, runs):
        units = np.ascontiguousarray(units, dtype=MP3_GC_DTYPE)
        runs = np.ascontiguousarray(runs, dtype=MP3_RUN_DTYPE)
        n_frames = units.size // 4
        if units.size != n_frames * 4:
            raise ValueError("units must hold 4 granule-channels per frame")
        return units, runs, n_frames

    def mp3_synth_host(self, units, spectra, runs, out=None):
        """units [F,2,2] MP3_GC_DTYPE, spectra [F,2,2,576] f32, runs [R] MP3_RUN_DTYPE -> pcm [F,2,1152]."""
        units, runs, n_frames = self._mp3_args(units, spectra, runs)
        spectra = np.ascontiguousarray(spectra, dtype=np.float32)
        if spectra.size != n_frames * 2304:
            raise ValueError("spectra must be [n_frames, 2, 2, 576]")
        if out is None:
            out = np.empty((n_frames, 2, 1152), dtype=np.float32)
        self._check(self._lib.symgpu_mp3_synth_host(self._ctx, _np_ptr(units), _np_ptr(spectra), _np_ptr(runs),
                                                    len(runs), n_frames, _np_ptr(out)))
        return out

    def mp3_synth_dev(self, units_t, spectra_t, runs, pcm_t):
        """Device-resident variant: torch CUDA tensors (uint8 [F*256], f32 [F,2,2,576], f32 [F,2,1152])."""
        runs = np.ascontiguousarray(runs, dtype=MP3_RUN_DTYPE)
        n_frames = spectra_t.numel() // 2304
        assert units_t.is_cuda and spectra_t.is_cuda and pcm_t.is_cuda
        assert units_t.numel() * units_t.element_size() == n_frames * 256
        assert pcm_t.numel() == n_frames * 2304 and spectra_t.is_contiguous() and pcm_t.is_contiguous()
        self._check(self._lib.symgpu_mp3_synth_dev(self._ctx, ctypes.c_void_p(units_t.data_ptr()),
                                                   ctypes.c_void_p(spectra_t.data_ptr()), _np_ptr(runs), len(runs),
                                                   n_frames, ctypes.c_void_p(pcm_t.data_ptr())))

    def mp3_synth_host_packed(self, units, spectra, runs, fmt, out=None):
        """Like mp3_synth_host, but the output stage runs on the device: returns [F*1152, 2] interleaved
        samples of `fmt` (FMT_*); only those cross PCIe on the way back."""
        units, runs, n_frames = self._mp3_args(units, spectra, runs)
        spectra = np.ascontiguousarray(spectra, dtype=np.float32)
        if spectra.size != n_frames * 2304:
            raise ValueError("spectra must be [n_frames, 2, 2, 576]")
        if out is None:
            out = np.empty((n_frames * 1152, 2), dtype=FMT_NUMPY[fmt])
        self._check(self._lib.symgpu_mp3_synth_host_packed(self._ctx, _np_ptr(units), _np_ptr(spectra), _np_ptr(runs),
                                                           len(runs), n_frames, int(fmt), _np_ptr(out)))
        return out

    def mp3_synth_host_quantized(self, units, quant, runs, fmt=None, out=None):
        """Like mp3_synth_host / mp3_synth_host_packed, fed with the quantised spectra [F,2,2,576] int16 (value =
        sign(q) * |q|^(4/3), looked up on the device).  fmt None: planar f32 [F,2,1152]; else interleaved [F*1152,2]."""
        units, runs, n_frames = self._mp3_args(units, quant, runs)
        quant = np.ascontiguousarray(quant, dtype=np.int16)
        if quant.size != n_frames * 2304:
            raise ValueError("quant must be [n_frames, 2, 2, 576]")
        if out is None:
            out = (np.empty((n_frames, 2, 1152), dtype=np.float32) if fmt is None
                   else np.empty((n_frames * 1152, 2), dtype=FMT_NUMPY[fmt]))
        self._check(self._lib.symgpu_mp3_synth_host_quantized(self._ctx, _np_ptr(units), _np_ptr(quant), _np_ptr(runs),
                                                              len(runs), n_frames, -1 if fmt is None else int(fmt),
                                                              _np_ptr(out)))
        return out

    def mp3_decode_files_host(self, files):
        """EXPERIMENTAL device front-end: files = [(bytes, packets (MPA_PACKET_DTYPE), stream slot)] -> (pcm [F,2,1152],
        good_per_file, frame_of, rounds); only the side-information pass runs on the CPU."""
        from ._native import MP3_FILE_DTYPE, MPA_PACKET_DTYPE
        keep, recs = [], np.zeros(len(files), dtype=MP3_FILE_DTYPE)
        for k, (data, packets, stream) in enumerate(files):
            a = np.frombuffer(data, dtype=np.uint8)
            p = np.ascontiguousarray(packets, dtype=MPA_PACKET_DTYPE)
            keep += [a, p]
            recs[k] = (a.ctypes.data, a.size, p.ctypes.data, len(p), stream, 0)
        total = int(recs["n_packets"].sum())
        pcm = np.zeros((total, 2, 1152), dtype=np.float32)
        good = np.zeros(len(files), dtype=np.uint32)
        frame_of = np.zeros(max(total, 1), dtype=np.uint32)
        rounds = ctypes.c_uint32(0)
        self._check(self._lib.symgpu_mp3_decode_files_host(self._ctx, _np_ptr(recs), len(files), _np_ptr(pcm), total, _np_ptr(good), _np_ptr(frame_of),
                                                           ctypes.byref(rounds)))
        n = int(good.sum())
        return pcm[:n], good, frame_of[:n], rounds.value

    # -- MPEG Layer I / II ---------------------------------------------------------------------
    def mpa12_synth_host(self, subbands, runs, out=None):
        """subbands [F,2,32,n_slots] f32 (n_slots 12: Layer I, 36: Layer II), runs MPA12_RUN_DTYPE -> pcm [F,2,1152]
        (the first 32*n_slots samples of a plane are the frame's PCM).  Uses the MP3 stream state slots."""
        subbands = np.ascontiguousarray(subbands, dtype=np.float32)
        runs = np.ascontiguousarray(runs, dtype=MPA12_RUN_DTYPE)
        n_frames, n_slots = subbands.shape[0], subbands.shape[-1]
        if subbands.shape[1:3] != (2, 32):
            raise ValueError("subbands must be [n_frames, 2, 32, n_slots]")
        if out is None:
            out = np.empty((n_frames, 2, 1152), dtype=np.float32)
        self._check(self._lib.symgpu_mpa12_synth_host(self._ctx, _np_ptr(subbands), _np_ptr(runs), len(runs), n_frames,
                                                      n_slots, _np_ptr(out)))
        return out

    def mpa12_synth_dev(self, subbands_t, runs, n_slots, pcm_t):
        runs = np.ascontiguousarray(runs, dtype=MPA12_RUN_DTYPE)
        n_frames = subbands_t.numel() // (64 * n_slots)
        assert subbands_t.is_cuda and pcm_t.is_cuda and pcm_t.numel() == n_frames * 2304
        self._check(self._lib.symgpu_mpa12_synth_dev(self._ctx, ctypes.c_void_p(subbands_t.data_ptr()), _np_ptr(runs), len(runs),
                                                     n_frames, n_slots, ctypes.c_void_p(pcm_t.data_ptr())))

    # -- FLAC ---------------------------------------------------------------------------------
    def flac_restore_host(self, frames, subframes, samples):
        """In place on `samples` (int32): prediction, wasted-bits shift, channel decorrelation, scaling to 32 bits."""
        from ._native import FLAC_FRAME_DTYPE, FLAC_SUBFRAME_DTYPE
        frames = np.ascontiguousarray(frames, dtype=FLAC_FRAME_DTYPE)
        subframes = np.ascontiguousarray(subframes, dtype=FLAC_SUBFRAME_DTYPE)
        assert samples.dtype == np.int32 and samples.flags.c_contiguous
        self._check(self._lib.symgpu_flac_restore_host(self._ctx, _np_ptr(frames), len(frames), _np_ptr(subframes), len(subframes),
                                                       _np_ptr(samples), samples.size))
        return samples

    def flac_restore_dev(self, frames_t, n_frames, subframes_t, n_subframes, samples_t):
        assert frames_t.is_cuda and subframes_t.is_cuda and samples_t.is_cuda
        self._check(self._lib.symgpu_flac_restore_dev(self._ctx, ctypes.c_void_p(frames_t.data_ptr()), n_frames,
                                                      ctypes.c_void_p(subframes_t.data_ptr()), n_subframes,
                                                      ctypes.c_void_p(samples_t.data_ptr()), samples_t.numel()))

    def flac_decode_host(self, frames, subframes, samples, dst, fmt, out_samples=None, out=None):
        """Restoration + FromSample<i32> into `fmt` (FMT_*), interleaved: frame f's n * channels samples at flat index dst[f] of
        the result, a 1-D array of out_samples samples of `fmt` (or `out`, any shape).  `samples` (int32) is left as it is."""
        from ._native import FLAC_FRAME_DTYPE, FLAC_SUBFRAME_DTYPE
        frames = np.ascontiguousarray(frames, dtype=FLAC_FRAME_DTYPE)
        subframes = np.ascontiguousarray(subframes, dtype=FLAC_SUBFRAME_DTYPE)
        samples = np.ascontiguousarray(samples, dtype=np.int32)
        dst = np.ascontiguousarray(dst, dtype=np.uint64)
        if len(dst) != len(frames):
            raise ValueError("dst must hold one output position per frame")
        if out is None:
            out = np.empty(int(out_samples), dtype=FMT_NUMPY[fmt])
        assert out.flags.c_contiguous
        self._check(self._lib.symgpu_flac_decode_host(self._ctx, _np_ptr(frames), len(frames), _np_ptr(subframes), len(subframes),
                                                      _np_ptr(samples), samples.size, _np_ptr(dst), int(fmt), _np_ptr(out), out.nbytes))
        return out

    def flac_decode_dev(self, frames_t, n_frames, subframes_t, n_subframes, samples_t, dst_t, fmt, out_t, out_samples=None):
        """Device-resident flac_decode_host (torch CUDA tensors; dst_t int64 / uint64 per frame).  Runs the predictors in place on
        samples_t; out_samples defaults to what out_t holds in samples of `fmt`."""
        assert frames_t.is_cuda and subframes_t.is_cuda and samples_t.is_cuda and dst_t.is_cuda and out_t.is_cuda
        if out_samples is None:
            out_samples = out_t.numel() * out_t.element_size() // np.dtype(FMT_NUMPY[fmt]).itemsize
        self._check(self._lib.symgpu_flac_decode_dev(self._ctx, ctypes.c_void_p(frames_t.data_ptr()), n_frames,
                                                     ctypes.c_void_p(subframes_t.data_ptr()), n_subframes,
                                                     ctypes.c_void_p(samples_t.data_ptr()), samples_t.numel(),
                                                     ctypes.c_void_p(dst_t.data_ptr()), int(fmt),
                                                     ctypes.c_void_p(out_t.data_ptr()), int(out_samples)))

    # -- output stage -------------------------------------------------------------------------
    def pcm_pack_host(self, pcm, spans, channels, fmt, out_frames, plane_stride=0, frames=0, n_spans=None, out=None):
        """Trim + interleave + convert planar f32 `pcm` (any shape, flat indexing) into [out_frames, channels]
        samples.  spans: PCM_SPAN_DTYPE array, or None for uniform packets (plane_stride, frames, n_spans)."""
        pcm = np.ascontiguousarray(pcm, dtype=np.float32)
        if spans is not None:
            spans = np.ascontiguousarray(spans, dtype=PCM_SPAN_DTYPE)
            n_spans = len(spans)
        if out is None:
            out = np.zeros((out_frames, channels), dtype=FMT_NUMPY[fmt])
        self._check(self._lib.symgpu_pcm_pack_host(self._ctx, _np_ptr(pcm), pcm.size,
                                                   _np_ptr(spans) if spans is not None else None, n_spans, channels,
                                                   plane_stride, frames, int(fmt), _np_ptr(out), out.nbytes))
        return out

    def pcm_pack_dev(self, pcm_t, spans_t, n_spans, channels, fmt, out_t, plane_stride=0, frames=0):
        """Device-resident variant (torch CUDA tensors; spans_t may be None for uniform packets)."""
        assert pcm_t.is_cuda and out_t.is_cuda
        self._check(self._lib.symgpu_pcm_pack_dev(self._ctx, ctypes.c_void_p(pcm_t.data_ptr()),
                                                  ctypes.c_void_p(spans_t.data_ptr()) if spans_t is not None else None,
                                                  n_spans, channels, plane_stride, frames, int(fmt),
                                                  ctypes.c_void_p(out_t.data_ptr())))

    def pcm_pack_host_mapped(self, pcm, spans, channels, plane_of_channel, fmt, out_frames, plane_stride=0, frames=0, n_spans=None, out=None):
        """pcm_pack_host with a channel map: output channel c reads plane plane_of_channel[c]."""
        pcm = np.ascontiguousarray(pcm, dtype=np.float32)
        m = np.ascontiguousarray(plane_of_channel, dtype=np.uint8)
        if m.size != channels:
            raise ValueError("plane_of_channel must name one plane per output channel")
        if spans is not None:
            spans = np.ascontiguousarray(spans, dtype=PCM_SPAN_DTYPE)
            n_spans = len(spans)
        if out is None:
            out = np.zeros((out_frames, channels), dtype=FMT_NUMPY[fmt])
        self._check(self._lib.symgpu_pcm_pack_mapped_host(self._ctx, _np_ptr(pcm), pcm.size, _np_ptr(spans) if spans is not None else None, n_spans,
                                                          channels, plane_stride, frames, _np_ptr(m), int(fmt), _np_ptr(out), out.nbytes))
        return out

    def pcm_pack_dev_mapped(self, pcm_t, spans_t, n_spans, channels, plane_of_channel, fmt, out_t, plane_stride=0, frames=0):
        """Device-resident pcm_pack_host_mapped (torch CUDA tensors; the map is host memory)."""
        assert pcm_t.is_cuda and out_t.is_cuda
        m = np.ascontiguousarray(plane_of_channel, dtype=np.uint8)
        if m.size != channels:
            raise ValueError("plane_of_channel must name one plane per output channel")
        self._check(self._lib.symgpu_pcm_pack_mapped_dev(self._ctx, ctypes.c_void_p(pcm_t.data_ptr()),
                                                         ctypes.c_void_p(spans_t.data_ptr()) if spans_t is not None else None,
                                                         n_spans, channels, plane_stride, frames, _np_ptr(m), int(fmt),
                                                         ctypes.c_void_p(out_t.data_ptr())))

    # -- AAC --------------------------------------------------------------------------------
    def aac_streams_alloc(self, n_streams):
        self._check(self._lib.symgpu_aac_streams_alloc(self._ctx, int(n_streams)))

    def aac_stream_reset(self, stream):
        self._check(self._lib.symgpu_aac_stream_reset(self._ctx, int(stream)))

    def aac_synth_host(self, units, tns, coeffs, runs, out=None):
        """units [F,2] AAC_UNIT_DTYPE, tns [T] AAC_TNS_DTYPE, coeffs [F,2,1024] f32 -> pcm [F,2,1024]."""
        units = np.ascontiguousarray(units, dtype=AAC_UNIT_DTYPE)
        tns = np.ascontiguousarray(tns, dtype=AAC_TNS_DTYPE)
        runs = np.ascontiguousarray(runs, dtype=AAC_RUN_DTYPE)
        coeffs = np.ascontiguousarray(coeffs, dtype=np.float32)
        n_frames = units.size // 2
        if coeffs.size != n_frames * 2048:
            raise ValueError("coeffs must be [n_frames, 2, 1024]")
        if out is None:
            out = np.empty((n_frames, 2, 1024), dtype=np.float32)
        self._check(self._lib.symgpu_aac_synth_host(self._ctx, _np_ptr(units), _np_ptr(tns) if len(tns) else None, len(tns),
                                                    _np_ptr(coeffs), _np_ptr(runs), len(runs), n_frames, _np_ptr(out)))
        return out

    def aac_synth_dev(self, units_t, tns_t, n_tns, coeffs_t, runs, pcm_t):
        runs = np.ascontiguousarray(runs, dtype=AAC_RUN_DTYPE)
        n_frames = coeffs_t.numel() // 2048
        self._check(self._lib.symgpu_aac_synth_dev(
            self._ctx, ctypes.c_void_p(units_t.data_ptr()), ctypes.c_void_p(tns_t.data_ptr()) if n_tns else None, int(n_tns),
            ctypes.c_void_p(coeffs_t.data_ptr()), _np_ptr(runs), len(runs), n_frames, ctypes.c_void_p(pcm_t.data_ptr())))

    # -- Vorbis -----------------------------------------------------------------------------
    def vorbis_streams_set(self, streams):
        streams = np.ascontiguousarray(streams, dtype=VORBIS_STREAM_DTYPE)
        self._check(self._lib.symgpu_vorbis_streams_set(self._ctx, _np_ptr(streams), len(streams)))

    def vorbis_floors_set(self, floors):
        floors = np.ascontiguousarray(floors, dtype=VORBIS_FLOOR1_DTYPE)
        self._check(self._lib.symgpu_vorbis_floors_set(self._ctx, _np_ptr(floors), len(floors)))

    def vorbis_stream_reset(self, stream):
        self._check(self._lib.symgpu_vorbis_stream_reset(self._ctx, int(stream)))

    def vorbis_synth_host(self, units, floor_y, residue, runs, slot, out=None):
        """units [P] VORBIS_UNIT_DTYPE, floor_y [P,2,65] u16, residue [P,2,slot] f32 -> pcm [P,2,slot]."""
        units = np.ascontiguousarray(units, dtype=VORBIS_UNIT_DTYPE)
        floor_y = np.ascontiguousarray(floor_y, dtype=np.uint16)
        residue = np.ascontiguousarray(residue, dtype=np.float32)
        runs = np.ascontiguousarray(runs, dtype=VORBIS_RUN_DTYPE)
        n = len(units)
        if residue.size != n * 2 * slot or floor_y.size != n * 130:
            raise ValueError("residue must be [n, 2, slot] and floor_y [n, 2, 65]")
        if out is None:
            out = np.empty((n, 2, slot), dtype=np.float32)
        self._check(self._lib.symgpu_vorbis_synth_host(self._ctx, _np_ptr(units), _np_ptr(floor_y), _np_ptr(residue),
                                                       _np_ptr(runs), len(runs), n, int(slot), _np_ptr(out)))
        return out

    def vorbis_mc_streams_set(self, streams):
        """Multichannel Vorbis streams (up to 8 channels, every coupling step of the mapping): VORBIS_STREAM_MC_DTYPE records."""
        streams = np.ascontiguousarray(streams, dtype=VORBIS_STREAM_MC_DTYPE)
        self._check(self._lib.symgpu_vorbis_mc_streams_set(self._ctx, _np_ptr(streams), len(streams)))

    def vorbis_mc_synth_host(self, units, floor_y, residue, runs, channels, slot, out=None):
        """units [P] VORBIS_UNIT_MC_DTYPE, floor_y [P,C,65] u16, residue [P,C,slot] f32 -> pcm [P,C,slot]."""
        units = np.ascontiguousarray(units, dtype=VORBIS_UNIT_MC_DTYPE)
        floor_y = np.ascontiguousarray(floor_y, dtype=np.uint16)
        residue = np.ascontiguousarray(residue, dtype=np.float32)
        runs = np.ascontiguousarray(runs, dtype=VORBIS_RUN_DTYPE)
        n, C = len(units), int(channels)
        if residue.size != n * C * slot or floor_y.size != n * C * 65:
            raise ValueError("residue must be [n, channels, slot] and floor_y [n, channels, 65]")
        if out is None:
            out = np.empty((n, C, slot), dtype=np.float32)
        self._check(self._lib.symgpu_vorbis_mc_synth_host(self._ctx, _np_ptr(units), _np_ptr(floor_y), _np_ptr(residue), _np_ptr(runs), len(runs), n,
                                                          C, int(slot), _np_ptr(out)))
        return out

    def vorbis_mc_synth_dev(self, units_t, floor_y_t, residue_t, runs, channels, slot, pcm_t):
        """Device-resident vorbis_mc_synth_host (torch CUDA tensors); decouples residue_t in place."""
        runs = np.ascontiguousarray(runs, dtype=VORBIS_RUN_DTYPE)
        n = units_t.numel() * units_t.element_size() // 32
        self._check(self._lib.symgpu_vorbis_mc_synth_dev(
            self._ctx, ctypes.c_void_p(units_t.data_ptr()), ctypes.c_void_p(floor_y_t.data_ptr()), ctypes.c_void_p(residue_t.data_ptr()),
            _np_ptr(runs), len(runs), n, int(channels), int(slot), ctypes.c_void_p(pcm_t.data_ptr())))

    def vorbis_synth_dev(self, units_t, floor_y_t, residue_t, runs, slot, pcm_t):
        runs = np.ascontiguousarray(runs, dtype=VORBIS_RUN_DTYPE)
        n = units_t.numel() * units_t.element_size() // 16
        self._check(self._lib.symgpu_vorbis_synth_dev(
            self._ctx, ctypes.c_void_p(units_t.data_ptr()), ctypes.c_void_p(floor_y_t.data_ptr()),
            ctypes.c_void_p(residue_t.data_ptr()), _np_ptr(runs), len(runs), n, int(slot), ctypes.c_void_p(pcm_t.data_ptr())))
